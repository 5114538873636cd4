"""Drop-in surface of the reference's student (``StudentCandidateV1``, /root/reference/src/models/model.py:50-187) for its
DECODER half -- the part ``src/inference.py:51`` and ``src/real_time_inference.py:58`` spend their decode loop in.

Same constructor arguments, attribute / state-dict names (``decoder.layers.N.*``, ``embed``, ``linear``, ``pos_enc``) and
method contracts (``forward_decoder(y, memory)`` :135, ``greedy_decode(src, max_len)`` :156, ``forward_image_enc`` :116),
but the decoder arithmetic runs in libgitb200.so (csrc/student.cu): tcgen05 / weight-streaming GEMMs, small attention /
LayerNorm / argmax kernels, and a K/V cache in place of the reference's full re-decode of the growing sequence every step.
The nn.Module tree only holds parameters; there is no torch forward and no CPU path.

The TinyViT image encoder (timm ``features_only`` model, :35-48) is not rebuilt: pass ``image_encoder=`` (any module that
returns the list of stage feature maps like timm's) or call ``greedy_decode_from_memory`` / ``forward_decoder`` with the
``memory`` tensor [B, F, d_model] directly.  ``enable_training`` / ``distillation_step`` / ``DistillationTrainer`` run the
reference's distillation step (model.py:880-983) for the decoder on the same library (csrc/student_train.cu), with the
reference's train-mode dropout when a ``dropout_seed`` is given.
"""
from __future__ import annotations

import ctypes
import math
from typing import Optional

import torch
import torch.nn as nn

from . import _lib
from ._lib import GitB200Error, StudentConfig


def _check(code: int, lib, h, what: str) -> None:
    if code != 0:
        msg = lib.gitb200_student_last_error(h)
        raise GitB200Error(f"{what} failed ({code}): {msg.decode() if msg else ''}")


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


class PositionalEncoding(nn.Module):
    """model.py:320-340: the sinusoidal table as a buffer ``pe`` [1, max_len, d_model]."""

    def __init__(self, d_model: int, max_len: int = 500):
        super().__init__()
        pe = torch.zeros(max_len, d_model)
        position = torch.arange(0, max_len).unsqueeze(1)
        div_term = torch.exp(torch.arange(0, d_model, 2) * -(torch.log(torch.tensor(10000.0)) / d_model))
        pe[:, 0::2] = torch.sin(position * div_term)
        pe[:, 1::2] = torch.cos(position * div_term)
        self.register_buffer("pe", pe.unsqueeze(0))

    def forward(self, x):  # pragma: no cover - guard
        raise RuntimeError("parameter container only: the student decoder runs on the CUDA library")


class _Params(nn.Module):
    def forward(self, *a, **k):  # pragma: no cover - guard
        raise RuntimeError("parameter container only: the student decoder runs on the CUDA library")


class _MHAParams(_Params):
    def __init__(self, d):
        super().__init__()
        self.in_proj_weight = nn.Parameter(torch.empty(3 * d, d))
        self.in_proj_bias = nn.Parameter(torch.zeros(3 * d))
        self.out_proj = nn.Linear(d, d)
        nn.init.xavier_uniform_(self.in_proj_weight)


class _DecoderLayerParams(_Params):
    """Parameter names of nn.TransformerDecoderLayer (model.py:73-75)."""

    def __init__(self, d, f):
        super().__init__()
        self.self_attn, self.multihead_attn = _MHAParams(d), _MHAParams(d)
        self.linear1, self.linear2 = nn.Linear(d, f), nn.Linear(f, d)
        self.norm1, self.norm2, self.norm3 = nn.LayerNorm(d), nn.LayerNorm(d), nn.LayerNorm(d)


class _DecoderParams(_Params):
    def __init__(self, d, f, n):
        super().__init__()
        self.layers = nn.ModuleList([_DecoderLayerParams(d, f) for _ in range(n)])
        self.num_layers = n


class StudentCandidateV1(nn.Module):
    """model.py:50-187 (decoder half on the GPU library)."""

    def __init__(self, image_enc_name: Optional[str], d_model: int, n_head: int, d_ffn: int, dropout: float, num_decoder_layers: int,
                 vocab_length: int, cls_token_id: int, sep_token_id: int, *, image_encoder: Optional[nn.Module] = None):
        super().__init__()
        self.image_enc_name = image_enc_name
        self.image_encoder = image_encoder            # model.py:72 builds TinyVIT(image_enc_name) through timm
        self.n_head, self.d_model, self.d_ffn, self.dropout = n_head, d_model, d_ffn, dropout
        self.ln_eps = 1e-5                            # LayerNorm eps: nn.TransformerDecoderLayer's default layer_norm_eps
        self.decoder = _DecoderParams(d_model, d_ffn, num_decoder_layers)
        self.embed = nn.Embedding(vocab_length, d_model)
        self.linear = nn.Linear(d_model, vocab_length)
        self.cls_token_id, self.sep_token_id = cls_token_id, sep_token_id
        self.pos_enc = PositionalEncoding(d_model=d_model)
        self._h = None
        self._lib = None
        self._stale = True
        self._dev = None
        self._train_cfg = None      # (lr, beta1, beta2, eps) once enable_training() was called
        self._grads = None          # flat fp32 gradient vector (torch owns it so that torch.distributed can reduce it in place)
        self._head_floats = 0
        self._params_dirty = False  # the optimizer has moved the library's master weights past the nn.Parameters
        self._dropout_seed = None   # Philox seed of the training step's dropout masks; None: no dropout
        self._dropout_step = 0      # the library's dropout step as of the last call that read or set it

    # ---- engine plumbing
    def load_state_dict(self, state_dict, strict: bool = False, **kw):
        # the reference's checkpoints also hold the TinyViT, the lazy projector heads and the template decoder_layer
        sd = {k: v for k, v in state_dict.items() if k.startswith(("decoder.layers.", "embed.", "linear.", "pos_enc."))}
        out = super().load_state_dict(sd, strict=False, **kw)
        self._stale = True
        return out

    def _apply(self, fn, *a, **k):
        if getattr(self, "_params_dirty", False):
            self.sync_parameters()  # the trained master weights must not be lost when the module is moved / cast
        self._stale = True
        return super()._apply(fn, *a, **k)

    def _engine(self):
        p = self.embed.weight
        if not p.is_cuda:
            raise RuntimeError("StudentCandidateV1 runs only on a CUDA device (B200): call .to('cuda') first; there is no CPU path")
        if self._h is not None and not self._stale and self._dev == p.device:
            return self._h
        self.close()
        lib = _lib.load()
        cfg = StudentConfig(self.d_model, self.n_head, self.d_ffn, self.decoder.num_layers, self.embed.num_embeddings,
                            self.pos_enc.pe.shape[1], self.cls_token_id, self.sep_token_id, 0, self.ln_eps)
        h = ctypes.c_void_p()
        _check(lib.gitb200_student_create(ctypes.byref(cfg), p.device.index or 0, ctypes.byref(h)), lib, None, "gitb200_student_create")
        if self._train_cfg is not None:
            _check(lib.gitb200_student_set_training(h, 1), lib, h, "gitb200_student_set_training")
        weights = {k: v for k, v in self.state_dict().items() if k.startswith(("decoder.layers.", "embed.", "linear."))}
        weights["pos_enc.pe"] = self.pos_enc.pe[0]
        for name, t in weights.items():
            t = t.detach().to(torch.float32).contiguous()
            shape = (ctypes.c_int64 * max(1, t.dim()))(*t.shape)
            _check(lib.gitb200_student_load_weight(h, name.encode(), _ptr(t), t.dim(), shape), lib, h, f"load_weight({name})")
        _check(lib.gitb200_student_finalize(h), lib, h, "gitb200_student_finalize")
        self._h, self._lib, self._stale, self._dev = h, lib, False, p.device
        self._ld = lib.gitb200_student_logits_ld(h)
        if self._train_cfg is not None:
            n = int(lib.gitb200_student_train_begin(h, *[ctypes.c_float(v) for v in self._train_cfg]))
            if n <= 0:
                raise GitB200Error("gitb200_student_train_begin: " + lib.gitb200_student_last_error(h).decode())
            self._grads = torch.zeros(n, dtype=torch.float32, device=p.device)
            self._head_floats = int(lib.gitb200_student_train_head_floats(h))
            self._params_dirty = False
            if self._dropout_seed is not None:
                _check(lib.gitb200_student_train_set_dropout(h, ctypes.c_float(self.dropout), self._dropout_seed, self._dropout_step),
                       lib, h, "gitb200_student_train_set_dropout")
        return h

    def close(self):
        if self._h is not None:
            self._lib.gitb200_student_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self._dev).cuda_stream)

    # ---- reference methods
    def forward_image_enc(self, x):
        """model.py:116-133: [B, F, C, H, W] -> (stage feature maps, memory [B, F, De]) through the supplied image encoder."""
        if self.image_encoder is None:
            raise RuntimeError("no image encoder: the reference builds a timm TinyViT (model.py:35-48), which this library does "
                               "not contain; pass image_encoder= or call greedy_decode_from_memory / forward_decoder with memory")
        shape = x.shape
        fmaps = self.image_encoder(x.view(shape[0] * shape[1], *shape[2:]))
        memory = torch.mean(fmaps[-1], dim=[2, 3]).view(shape[0], shape[1], -1)
        return fmaps, memory

    @torch.no_grad()
    def forward_decoder(self, y: torch.Tensor, memory: torch.Tensor) -> torch.Tensor:
        """model.py:135-154: y int [B, L], memory [B, F, d_model] -> logits fp32 [B, L, vocab]."""
        h = self._engine()
        tok = y.to(device=self._dev, dtype=torch.int32).contiguous()
        mem = memory.to(device=self._dev, dtype=torch.float32).contiguous()
        B, L = tok.shape
        if mem.shape[0] != B or mem.shape[2] != self.d_model:
            raise ValueError("memory must be [B, F, d_model]")
        logits = torch.empty(B * L, self._ld, dtype=torch.float32, device=self._dev)
        _check(self._lib.gitb200_student_forward_decoder(h, _ptr(tok), _ptr(mem), B, L, mem.shape[1], _ptr(logits), self._stream()),
               self._lib, h, "gitb200_student_forward_decoder")
        return logits.view(B, L, self._ld)[:, :, : self.embed.num_embeddings]

    @torch.no_grad()
    def greedy_decode_from_memory(self, memory: torch.Tensor, max_len: int = 10) -> torch.Tensor:
        """model.py:165-187 after the image encoder: LongTensor [B, <= max_len + 1] starting with CLS; decoding stops only
        when every row emits SEP in the same step (:184)."""
        h = self._engine()
        mem = memory.to(device=self._dev, dtype=torch.float32).contiguous()
        B = mem.shape[0]
        tokens = torch.empty(B, max_len + 1, dtype=torch.int32, device=self._dev)
        out_len = torch.zeros(1, dtype=torch.int32, device=self._dev)
        _check(self._lib.gitb200_student_greedy_decode(h, _ptr(mem), B, mem.shape[1], max_len, _ptr(tokens), _ptr(out_len), self._stream()),
               self._lib, h, "gitb200_student_greedy_decode")
        return tokens[:, : int(out_len.item())].long()

    @torch.no_grad()
    def beam_search_from_memory(self, memory: torch.Tensor, max_len: int = 10, k: int = 3, forward_decoder=None) -> torch.Tensor:
        """model.py:189-316 after the image encoder: the reference's k x k beam search (no end-of-sequence handling, the
        result always has ``max_len`` tokens).  All k beams of all clips are decoded in ONE forward_decoder call per
        step instead of k calls; candidate ranking / beam bookkeeping stay on the device as tensor ops."""
        fd = forward_decoder or self.forward_decoder
        B = memory.size(0)
        dev = memory.device
        tgt = torch.full((B, 1), self.cls_token_id, dtype=torch.long, device=dev)
        logp = torch.log_softmax(fd(tgt, memory)[:, -1, :].float(), dim=-1)
        scores, first = logp.topk(k, dim=-1)                                          # [B, k]
        sequences = torch.cat([tgt.unsqueeze(1).expand(-1, k, -1), first.unsqueeze(-1)], dim=-1)   # [B, k, 2]
        mem_k = memory.repeat_interleave(k, dim=0)                                    # row b*k + i = beam i of clip b
        for step in range(2, max_len):
            logp = torch.log_softmax(fd(sequences.reshape(B * k, -1), mem_k)[:, -1, :].float(), dim=-1)
            top_scores, top_tokens = logp.topk(k, dim=-1)                             # [B*k, k]
            cand = (scores.unsqueeze(-1) + top_scores.view(B, k, k)).view(B, k * k)   # candidate i*k + j = beam i, its j-th word
            _, order = cand.sort(dim=1, descending=True)
            pick = order[:, :k]                                                       # [B, k]
            beam = pick // k
            scores = torch.gather(cand, 1, pick)
            words = torch.gather(top_tokens.view(B, k * k), 1, pick)
            sequences = torch.cat([torch.gather(sequences, 1, beam.unsqueeze(-1).expand(-1, -1, sequences.shape[-1])),
                                   words.unsqueeze(-1)], dim=-1)
        return sequences[torch.arange(B, device=dev), scores.argmax(dim=-1)]

    @torch.no_grad()
    def beam_search(self, src: torch.Tensor, max_len: int = 10, k: int = 3) -> torch.Tensor:
        """model.py:189-316."""
        _, memory = self.forward_image_enc(src)
        return self.beam_search_from_memory(memory.to(self._dev or memory.device), max_len, k)

    @torch.no_grad()
    def greedy_decode(self, src: torch.Tensor, max_len: int = 10) -> torch.Tensor:
        """model.py:156-187."""
        _, memory = self.forward_image_enc(src)
        return self.greedy_decode_from_memory(memory, max_len)

    # ---- distillation training of the decoder half (DistillationTrainer.training_step, model.py:880-983)
    def enable_training(self, lr: float = 1e-4, betas=(0.9, 0.999), eps: float = 1e-8, dropout_seed: Optional[int] = None) -> None:
        """Switch the library context to training mode: fp32 master weights + torch.optim.Adam state (model.py:1105:
        ``Adam(student.parameters(), lr)``) next to the bf16 operand copies.

        Without ``dropout_seed`` the step applies no dropout.  With it, ``distillation_step`` applies the reference's
        train-mode dropout with p = ``self.dropout`` at nn.TransformerDecoderLayer's six sites per layer, from the library's
        Philox masks (include/gitb200.h, gitb200_student_train_set_dropout): a pure function of (seed, ``dropout_step``, site,
        element), so a step can be replayed.  ``dropout_step`` starts at 0.  p = 0 gives the step without dropout, bit for bit."""
        if dropout_seed is not None:
            if not 0.0 <= float(self.dropout) < 1.0:
                raise ValueError(f"dropout p = {self.dropout} is outside [0, 1)")
            if not 0 <= int(dropout_seed) < 2 ** 64:
                raise ValueError("dropout_seed must be an integer in [0, 2**64)")
            dropout_seed = int(dropout_seed)
        self._train_cfg = (float(lr), float(betas[0]), float(betas[1]), float(eps))
        self._dropout_seed, self._dropout_step = dropout_seed, 0
        self._stale = True

    @property
    def dropout_step(self) -> int:
        """Number of dropout forwards since the seed was set: the step whose masks the next ``distillation_step`` uses.
        Set it to resume a run or to replay a step (``dropout_step -= 1`` replays the previous one)."""
        if self._h is not None and not self._stale and self._train_cfg is not None:
            step = ctypes.c_longlong()
            _check(self._lib.gitb200_student_train_get_dropout(self._h, None, None, ctypes.byref(step)), self._lib, self._h,
                   "gitb200_student_train_get_dropout")
            self._dropout_step = step.value
        return self._dropout_step

    @dropout_step.setter
    def dropout_step(self, step: int) -> None:
        if self._dropout_seed is None:
            raise RuntimeError("dropout is off: call enable_training(..., dropout_seed=...) first")
        if int(step) < 0:
            raise ValueError("dropout_step must be >= 0")
        self._dropout_step = int(step)
        if self._h is not None and not self._stale:
            _check(self._lib.gitb200_student_train_set_dropout(self._h, ctypes.c_float(self.dropout), self._dropout_seed, self._dropout_step),
                   self._lib, self._h, "gitb200_student_train_set_dropout")

    def distillation_step(self, y: torch.Tensor, memory: torch.Tensor, teacher_logits: torch.Tensor, temperature: float = 1.0,
                          apply: bool = True, group=None, want_memory_grad: bool = False):
        """One training step on this rank's micro-batch: forward_decoder(y, memory) -> KL(batchmean) * T^2 + CE(ignore 0)
        (model.py:922-935, :983) -> backward -> gradient all-reduce over ``group`` (DDP average; the vocabulary-head bucket is
        reduced while the decoder layers are still in their backward pass) -> Adam.  Returns {'loss','kl','ce'} (device
        scalars, this rank's micro-batch) and, on request, d loss / d memory [B, M, d_model] for an external image encoder.
        With ``enable_training(dropout_seed=...)`` the forward applies dropout with the masks of ``dropout_step``, the backward
        replays them, and ``dropout_step`` advances by one."""
        if self._train_cfg is None:
            raise RuntimeError("call enable_training() first")
        from .dist import all_reduce_bucket, finish_all_reduce
        h = self._engine()
        lib = self._lib
        tok = y.to(device=self._dev, dtype=torch.int32).contiguous()
        mem = memory.to(device=self._dev, dtype=torch.float32).contiguous()
        tl = teacher_logits.to(device=self._dev, dtype=torch.float32)
        B, L = tok.shape
        tl = tl.reshape(B * L, tl.shape[-1])
        if tl.stride(-1) != 1 or tl.stride(0) % 4 != 0:
            tl = tl.contiguous()
        if mem.shape[0] != B or mem.shape[2] != self.d_model:
            raise ValueError("memory must be [B, F, d_model]")
        if tl.shape[-1] < self.embed.num_embeddings:
            raise ValueError("teacher logits must cover the student's vocabulary")
        loss = torch.empty(3, dtype=torch.float32, device=self._dev)
        dmem = torch.empty_like(mem) if want_memory_grad else None
        s = self._stream()
        _check(lib.gitb200_student_train_forward(h, _ptr(tok), _ptr(mem), _ptr(tl), tl.stride(0), B, L, mem.shape[1],
                                                 ctypes.c_float(temperature), _ptr(loss), s), lib, h, "gitb200_student_train_forward")
        if self._dropout_seed is not None:
            _ = self.dropout_step   # refreshes the host-side copy that an engine rebuild restores
        g = self._grads
        _check(lib.gitb200_student_train_backward(h, 0, _ptr(g), None, s), lib, h, "gitb200_student_train_backward(head)")
        w0 = all_reduce_bucket(g, 0, self._head_floats, group)            # overlaps phase 1
        _check(lib.gitb200_student_train_backward(h, 1, _ptr(g), _ptr(dmem), s), lib, h, "gitb200_student_train_backward(layers)")
        w1 = all_reduce_bucket(g, self._head_floats, g.numel(), group)
        scale = finish_all_reduce([w0, w1], group)
        if apply:
            _check(lib.gitb200_student_train_apply(h, _ptr(g), ctypes.c_float(scale), s), lib, h, "gitb200_student_train_apply")
            self._params_dirty = True
        out = {"loss": loss[0], "kl": loss[1], "ce": loss[2]}
        if want_memory_grad:
            out["d_memory"] = dmem
        return out

    def _export(self, name: str, which: int) -> torch.Tensor:
        p = dict(self.named_parameters())[name]
        out = torch.empty(p.shape, dtype=torch.float32, device=self._dev)
        _check(self._lib.gitb200_student_train_export(self._h, name.encode(), which, _ptr(self._grads), _ptr(out), self._stream()),
               self._lib, self._h, f"gitb200_student_train_export({name})")
        return out

    def gradients(self):
        """Gradients of the last distillation_step (after the all-reduce, before the 1/world scaling) under the reference's
        state-dict keys."""
        self._engine()
        return {k: self._export(k, 1) for k, _ in self.named_parameters() if k.startswith(("decoder.layers.", "embed.", "linear."))}

    def sync_parameters(self) -> None:
        """Copy the optimizer's fp32 master weights back into the nn.Parameters (``state_dict()`` does this on its own)."""
        if self._h is None or not self._params_dirty:
            return
        with torch.no_grad():
            for k, p in self.named_parameters():
                if k.startswith(("decoder.layers.", "embed.", "linear.")):
                    p.copy_(self._export(k, 0))
        self._params_dirty = False
        self._stale = False  # the copy above went through Parameter.copy_, not through _apply

    def state_dict(self, *a, **k):
        self.sync_parameters()
        return super().state_dict(*a, **k)

    def forward(self, x, y):
        """model.py:107-114: feature maps of the image encoder + the decoder logits."""
        fmaps, memory = self.forward_image_enc(x)
        return list(fmaps) + [self.forward_decoder(y, memory)]


class DistillationTrainer:
    """DistillationTrainer.training_step (model.py:880-983) for what this library holds of the student: the frozen GIT teacher
    gives the teacher-forced logits (``forward_output_logits``, :896), the student's DECODER is trained on KL + CE (:983) with
    Adam (:1105) and a DDP gradient all-reduce (train.py:217-221).  The student's TinyViT image encoder is not part of the
    library: ``batch['memory']`` ([B, F, d_model], what ``forward_image_enc`` returns at :128) is supplied by the caller, and
    ``d_memory`` comes back for it.  No Lightning: call ``training_step`` from your own loop.

    ``dropout_seed``: None trains without dropout.  An integer applies the reference's train-mode dropout (p = the student's
    ``dropout``) from the library's Philox masks.  The masks do not depend on the rank: for independent masks per rank pass
    ``dropout_seed = seed + rank``."""

    def __init__(self, teacher, student: StudentCandidateV1, lr: float = 1e-4, temperature: float = 1.0, group=None,
                 dropout_seed: Optional[int] = None):
        self.teacher, self.student, self.temperature, self.group = teacher, student, temperature, group
        student.enable_training(lr=lr, dropout_seed=dropout_seed)

    @torch.no_grad()
    def teacher_logits(self, x: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
        out_teacher, _, _ = self.teacher.forward_output_logits(x, y)      # model.py:896
        return torch.cat(out_teacher, dim=0)                               # :919  [B, L, V]

    def training_step(self, batch, batch_idx: int = 0):
        x, y, memory = batch["frames"], batch["caption"], batch["memory"]
        t_logits = self.teacher_logits(x, y)
        out = self.student.distillation_step(y, memory, t_logits, temperature=self.temperature, group=self.group,
                                             want_memory_grad=True)
        self.last = out
        return out["loss"]
