"""Drop-in Python surface of the reference's GIT captioning path (/root/reference/src/models/model.py).

Same names, constructor arguments, return structures and error behaviour as the reference classes
(`get_git_model` :681, `GenerativeImageTextModel` :343, `GeneratorWithBeamSearchV2` :465,
`GenerativeImageTextTeacher` :721), but every tensor operation of the path runs in libgitb200.so
(hand-written sm_100a kernels) through the C ABI of include/gitb200.h.  The nn.Module tree below only
*holds* the parameters under the upstream state-dict key names so that ``load_state_dict``,
``.parameters()``, ``.eval()`` and ``.to()`` behave as callers expect; none of these modules has a torch
forward, and there is no CPU path: without a B200 and the built library every forward raises.

Differences from the reference, all deliberate (DESIGN.md):
  * clips are batched: one call encodes and captions every clip of ``x`` (the reference loops clip by clip,
    model.py:752-759, :765-770);
  * the decoder keeps a true K/V cache (the upstream cache stores layer inputs and re-projects K,V every
    step) and visual K/V are shared by all beams of a clip;
  * the search loop and its bookkeeping run on the device; ``logits_dict`` is materialised on the host only
    when it is read.
"""
from __future__ import annotations

import dataclasses
import functools
from typing import Callable, Dict, List, Optional, Sequence

import numpy as np
import torch
import torch.nn as nn

from .engine import VIT_CONFIGS, Engine, SampleConfig, SearchConfig, make_config

VOCAB_SIZE = 30522  # model.py:689


# ----------------------------------------------------------------------------------------------
# parameter containers (upstream module tree; no torch forward on purpose)
# ----------------------------------------------------------------------------------------------
class _Holder(nn.Module):
    def forward(self, *a, **k):  # pragma: no cover - guard
        raise RuntimeError("gitb200 parameter containers have no torch forward; call the model, it runs on the "
                           "CUDA library")


class _Affine(_Holder):
    """weight (+bias) container: Linear [out,in], LayerNorm [n], Conv2d [out,in,k,k]."""

    def __init__(self, w_shape: Sequence[int], bias: bool = True, ln: bool = False, std: float = 0.02):
        super().__init__()
        w = torch.ones(*w_shape) if ln else torch.randn(*w_shape) * std
        self.weight = nn.Parameter(w)
        if bias:
            self.bias = nn.Parameter(torch.zeros(w_shape[0]))


class _MHA(_Holder):
    def __init__(self, width: int):
        super().__init__()
        self.in_proj_weight = nn.Parameter(torch.randn(3 * width, width) * width ** -0.5)
        self.in_proj_bias = nn.Parameter(torch.zeros(3 * width))
        self.out_proj = _Affine((width, width), std=width ** -0.5)


class _MLP(_Holder):
    def __init__(self, width: int):
        super().__init__()
        self.c_fc = _Affine((4 * width, width), std=width ** -0.5)
        self.c_proj = _Affine((width, 4 * width), std=(4 * width) ** -0.5)


class ResidualAttentionBlock(_Holder):
    """image_encoder.transformer.resblocks[i] (attested at model.py:847)."""

    def __init__(self, width: int):
        super().__init__()
        self.ln_1 = _Affine((width,), ln=True)
        self.attn = _MHA(width)
        self.ln_2 = _Affine((width,), ln=True)
        self.mlp = _MLP(width)


class _Transformer(_Holder):
    def __init__(self, width: int, layers: int):
        super().__init__()
        self.resblocks = nn.ModuleList([ResidualAttentionBlock(width) for _ in range(layers)])


class CLIPVisionTower(_Holder):
    """Parameters of upstream get_image_encoder(image_encoder_type, input_resolution) (model.py:682-685)."""

    def __init__(self, image_encoder_type: str = "CLIPViT_B_16", input_resolution: int = 224):
        super().__init__()
        v = VIT_CONFIGS[image_encoder_type]
        w, p = v["width"], v["patch"]
        self.image_encoder_type, self.input_resolution = image_encoder_type, input_resolution
        self.conv1 = _Affine((w, 3, p, p), bias=False, std=(3 * p * p) ** -0.5)
        self.class_embedding = nn.Parameter(torch.randn(w) * w ** -0.5)
        self.positional_embedding = nn.Parameter(torch.randn((input_resolution // p) ** 2 + 1, w) * w ** -0.5)
        self.ln_pre = _Affine((w,), ln=True)
        self.transformer = _Transformer(w, v["layers"])
        self.ln_post = _Affine((w,), ln=True)


class _SelfAttention(_Holder):
    def __init__(self, h):
        super().__init__()
        self.query, self.key, self.value = _Affine((h, h)), _Affine((h, h)), _Affine((h, h))


class _AttnOutput(_Holder):
    def __init__(self, h_in, h):
        super().__init__()
        self.dense = _Affine((h, h_in))
        self.LayerNorm = _Affine((h,), ln=True)


class _Attention(_Holder):
    def __init__(self, h):
        super().__init__()
        self.self = _SelfAttention(h)
        self.output = _AttnOutput(h, h)


class _Intermediate(_Holder):
    def __init__(self, h, f):
        super().__init__()
        self.dense = _Affine((f, h))


class BertLayer(_Holder):
    """textual.transformer.encoder.layer[i] (``.output`` attested at model.py:857)."""

    def __init__(self, h, f):
        super().__init__()
        self.attention = _Attention(h)
        self.intermediate = _Intermediate(h, f)
        self.output = _AttnOutput(f, h)


class _BertEncoder(_Holder):
    def __init__(self, h, f, layers):
        super().__init__()
        self.layer = nn.ModuleList([BertLayer(h, f) for _ in range(layers)])


class _BertEncoderAsDecoder(_Holder):
    def __init__(self, h, f, layers):
        super().__init__()
        self.encoder = _BertEncoder(h, f, layers)


class _Embedding(_Holder):
    def __init__(self, vocab, h, max_len):
        super().__init__()
        self.words = _Affine((vocab, h), bias=False)
        self.positions = _Affine((max_len, h), bias=False)
        self.layer_norm = _Affine((h,), ln=True)


class TransformerDecoderTextualHead(_Holder):
    """Parameters of the upstream text head built at model.py:687-700 (argument names kept)."""

    def __init__(self, visual_feature_size=768, vocab_size=VOCAB_SIZE, hidden_size=768, num_layers=6, attention_heads=12,
                 feedforward_size=3072, max_caption_length=1024, mask_future_positions=True, padding_idx=0,
                 decoder_type="bert_en", output_hidden_states=True, visual_projection_type="linearLn"):
        super().__init__()
        if decoder_type != "bert_en" or visual_projection_type != "linearLn" or not mask_future_positions:
            raise NotImplementedError("only decoder_type='bert_en', visual_projection_type='linearLn', causal text")
        self.visual_feature_size, self.vocab_size, self.hidden_size = visual_feature_size, vocab_size, hidden_size
        self.num_layers, self.attention_heads, self.feedforward_size = num_layers, attention_heads, feedforward_size
        self.max_caption_length, self.output_hidden_states = max_caption_length, output_hidden_states
        self.visual_projection = nn.ModuleList([_Affine((hidden_size, visual_feature_size), std=visual_feature_size ** -0.5),
                                                _Affine((hidden_size,), ln=True)])
        self.embedding = _Embedding(vocab_size, hidden_size, max_caption_length)
        self.transformer = _BertEncoderAsDecoder(hidden_size, feedforward_size, num_layers)
        self.output = _Affine((vocab_size, hidden_size))
        self.output.weight = self.embedding.words.weight  # upstream ties the vocabulary head to the word embedding


# ----------------------------------------------------------------------------------------------
# search
# ----------------------------------------------------------------------------------------------
class BeamHypotheses:
    """Upstream BeamHypotheses (constructed at model.py:503): n-best list with length-normalised scores."""

    def __init__(self, n_hyp, max_length, length_penalty, early_stopping):
        self.max_length = max_length - 1
        self.length_penalty, self.early_stopping, self.n_hyp = length_penalty, early_stopping, n_hyp
        self.hyp, self.worst_score = [], 1e9

    def __len__(self):
        return len(self.hyp)

    def add(self, hyp, sum_logprobs):
        score = sum_logprobs / len(hyp) ** self.length_penalty
        if len(self) < self.n_hyp or score > self.worst_score:
            self.hyp.append((score, hyp))
            if len(self) > self.n_hyp:
                ranked = sorted((s, i) for i, (s, _) in enumerate(self.hyp))
                del self.hyp[ranked[0][1]]
                self.worst_score = ranked[1][0]
            else:
                self.worst_score = min(score, self.worst_score)

    def is_done(self, best_sum_logprobs):
        if len(self) < self.n_hyp:
            return False
        if self.early_stopping:
            return True
        return self.worst_score >= best_sum_logprobs / self.max_length ** self.length_penalty


def top_k_top_p_filtering(logits, top_k=0, top_p=1.0, filter_value=-float("Inf"), min_tokens_to_keep=1):
    """Upstream sampling filter called at model.py:537: in-place top-k and nucleus (top-p) truncation of a batch of
    logits [rows, V].  ``None`` arguments fail on the comparisons exactly like upstream (TypeError)."""
    if top_k > 0:
        k = min(max(top_k, min_tokens_to_keep), logits.size(-1))
        threshold = torch.topk(logits, k)[0][..., -1, None]
        logits[logits < threshold] = filter_value
    if top_p < 1.0:
        ordered, order = torch.sort(logits, descending=True)
        drop = torch.cumsum(torch.softmax(ordered, dim=-1), dim=-1) > top_p
        if min_tokens_to_keep > 1:
            drop[..., :min_tokens_to_keep] = False
        drop[..., 1:] = drop[..., :-1].clone()  # the token that crosses top_p stays
        drop[..., 0] = False
        logits[drop.scatter(1, order, drop)] = filter_value
    return logits


class LazyLogits(Sequence):
    """``logits_dict`` of the reference (model.py:521: a list over steps of a list over beam rows of
    np.ndarray[V]) backed by the device buffer the decode kernels wrote; copied to the host on first read."""

    def __init__(self, dev: torch.Tensor, vocab: int):
        self._dev, self._vocab, self._host = dev, vocab, None

    def device_tensor(self) -> torch.Tensor:
        """[steps, rows, V] view on the device (no copy)."""
        return self._dev[:, :, : self._vocab]

    def _materialise(self):
        if self._host is None:
            self._host = self.device_tensor().cpu().numpy()
        return self._host

    def __len__(self):
        return self._dev.shape[0]

    def __getitem__(self, i):
        h = self._materialise()
        if isinstance(i, slice):
            return [list(step) for step in h[i]]
        return list(h[i])


class GeneratorWithBeamSearchV2:
    """model.py:465-678.  ``search`` keeps the reference's generic contract -- any ``step`` callable mapping
    input_ids [B*beams, len] to scores [B*beams, V] -- with the control flow on the host; when the model
    recognises its own decoder it bypasses this loop for the fused device-side search (same semantics)."""

    def __init__(self, eos_index, max_steps, beam_size, length_penalty, per_node_beam_size=2, repetition_penalty=1.0,
                 temperature=1.0):
        self._eos_index, self.max_steps, self.beam_size = eos_index, max_steps, beam_size
        self.length_penalty, self.per_node_beam_size = length_penalty, per_node_beam_size
        self.repetition_penalty, self.temperature = repetition_penalty, temperature

    def search_config(self, num_keep_best=1, reorder_cache=False) -> SearchConfig:
        return SearchConfig(self.beam_size, self.max_steps, self.length_penalty, self.per_node_beam_size, num_keep_best,
                            reorder_cache)

    def search(self, input_ids, step: Callable, num_keep_best=1, do_sample=False, top_k=None, top_p=None,
               num_return_sequences=1, on_reorder: Optional[Callable] = None):
        """``on_reorder(beam_idx, pos)`` (not in the reference, whose cache re-ordering is commented out at
        model.py:623-634) is called after every step with the parents chosen for the next rows and the text position
        just decoded, so that a K/V cache behind ``step`` can follow the beams (``cache_reorder='correct'``)."""
        if num_return_sequences != 1:
            input_ids = input_ids[:, None, :].expand(input_ids.shape[0], num_return_sequences, input_ids.shape[1])
            input_ids = input_ids.reshape(-1, input_ids.shape[-1])
        batch_size, cur_len = input_ids.shape
        nb, eos, max_length = self.beam_size, self._eos_index, self.max_steps
        input_ids = input_ids.unsqueeze(1).expand(batch_size, nb, cur_len).contiguous().view(batch_size * nb, cur_len)
        hyps = [BeamHypotheses(num_keep_best, max_length, self.length_penalty, early_stopping=False) for _ in range(batch_size)]
        beam_scores = torch.zeros((batch_size, nb), dtype=torch.float, device=input_ids.device)
        beam_scores[:, 1:] = -1e9
        beam_scores = beam_scores.view(-1)
        done = [False] * batch_size
        saved_logits = []
        while cur_len < max_length:
            scores = step(input_ids)
            vocab = scores.shape[-1]
            saved_logits.append([r.detach().cpu().numpy() for r in scores])
            if self.repetition_penalty != 1.0:
                for i in range(batch_size * nb):
                    for tok in set(input_ids[i].tolist()):
                        scores[i, tok] = scores[i, tok] * self.repetition_penalty if scores[i, tok] < 0 else scores[i, tok] / self.repetition_penalty
            if do_sample:  # model.py:532-554: temperature, top-k / top-p filter, per_node_beam_size samples per beam
                if self.temperature != 1.0:
                    scores = scores / self.temperature
                scores = top_k_top_p_filtering(scores, top_k=top_k, top_p=top_p, min_tokens_to_keep=2)
                words = torch.multinomial(torch.softmax(scores, dim=-1), num_samples=self.per_node_beam_size)
                picked = torch.gather(torch.log_softmax(scores, dim=-1), -1, words) + beam_scores[:, None]
                offsets = (torch.arange(nb, device=words.device) * vocab).repeat(batch_size, self.per_node_beam_size)
                next_words = words.view(batch_size, self.per_node_beam_size * nb) + offsets
                next_scores = picked.view(batch_size, self.per_node_beam_size * nb)
            else:
                lp = torch.log_softmax(scores, dim=-1) + beam_scores[:, None]
                next_scores, next_words = torch.topk(lp.view(batch_size, nb * vocab), self.per_node_beam_size * nb, dim=1,
                                                     largest=True, sorted=True)
            ns_host, nw_host = next_scores.tolist(), next_words.tolist()  # one transfer per step, not one per candidate
            nxt = []
            for b in range(batch_size):
                done[b] = done[b] or hyps[b].is_done(max(ns_host[b]))
                if done[b]:
                    nxt.extend([(0, eos, 0)] * nb)
                    continue
                beam = []
                for idx, score in zip(nw_host[b], ns_host[b]):
                    beam_id, word = idx // vocab, idx % vocab
                    if word == eos or cur_len + 1 == max_length:
                        hyps[b].add(input_ids[b * nb + beam_id, :cur_len].clone(), score)
                    else:
                        beam.append((score, word, b * nb + beam_id))
                    if len(beam) == nb:
                        break
                assert len(beam) == (0 if cur_len + 1 == max_length else nb)
                nxt.extend(beam if beam else [(0, eos, 0)] * nb)
            beam_scores = beam_scores.new_tensor([x[0] for x in nxt])
            beam_words = input_ids.new_tensor([x[1] for x in nxt])
            beam_idx = input_ids.new_tensor([x[2] for x in nxt])
            input_ids = torch.cat([input_ids[beam_idx, :], beam_words.unsqueeze(1)], dim=-1)
            if on_reorder is not None:
                on_reorder(beam_idx, cur_len - 1)
            cur_len += 1
            if all(done):
                break
        tgt_len = torch.ones(batch_size, num_keep_best, dtype=torch.long)
        logprobs = torch.full((batch_size, num_keep_best), -1e5, dtype=torch.float, device=input_ids.device)
        decoded = input_ids.new_full((batch_size, num_keep_best, max_length), eos)
        for i, h in enumerate(hyps):
            order = torch.topk(torch.tensor([x[0] for x in h.hyp]), min(num_keep_best, len(h.hyp)), largest=True)[1]
            for j, hi in enumerate(order.tolist()):
                conf, best = h.hyp[hi]
                logprobs[i, j] = conf
                tgt_len[i, j] = len(best) + 1
                decoded[i, j, : len(best)] = best
                decoded[i, j, len(best)] = eos
        if num_keep_best == 1:
            decoded = decoded.squeeze(dim=1)
        return decoded, logprobs, saved_logits


# ----------------------------------------------------------------------------------------------
# the model
# ----------------------------------------------------------------------------------------------
class GenerativeImageTextModel(nn.Module):
    """model.py:343-462 (subclass of upstream CaptioningModel), executing on a gitb200 Engine."""

    def __init__(self, image_encoder, text_decoder, decoder, tokenizer, param):
        super().__init__()
        self.image_encoder = image_encoder
        self.textual = text_decoder
        self.decoder = decoder
        self.tokenizer = tokenizer
        self.param = dict(param)
        self.sos_index = tokenizer.cls_token_id      # model.py:363
        self.eos_index = tokenizer.sep_token_id      # model.py:364
        self.use_history_for_infer = True            # model.py:366
        self.num_image_with_embedding = param.get("num_image_with_embedding")  # model.py:368
        self.pooling_images = None
        self.prev_encoded_layers = None
        width = VIT_CONFIGS[image_encoder.image_encoder_type]["width"]
        self.img_temperal_embedding = nn.ParameterList(
            [nn.Parameter(torch.zeros(1, 1, width)) for _ in range(self.num_image_with_embedding or 0)])
        self._engine: Optional[Engine] = None
        self._engine_stale = True
        self._vf_token = None          # visual-feature tensor currently resident in the engine
        self._step_pos = 0
        self.cache_reorder = "reference"  # or "correct" (SURVEY Appendix B.1)
        self._force_host_search = False   # tests: take the generic host `search` loop even where the fused one applies

    # ---- engine plumbing
    def load_state_dict(self, state_dict, strict: bool = True, **kw):
        sd = dict(state_dict)
        if "textual.output.weight" not in sd and "textual.embedding.words.weight" in sd:
            sd["textual.output.weight"] = sd["textual.embedding.words.weight"]
        if "textual.output.weight" in sd and "textual.embedding.words.weight" in sd and \
                sd["textual.output.weight"] is not sd["textual.embedding.words.weight"] and \
                not torch.equal(sd["textual.output.weight"], sd["textual.embedding.words.weight"]):
            # untied head (not produced by upstream, used by the parity tests): break the tie before copying
            self.textual.output.weight = nn.Parameter(torch.empty_like(self.textual.embedding.words.weight))
        sd.pop("image_encoder.proj", None)  # present in CLIP checkpoints, unused with output_grid=True
        out = super().load_state_dict(sd, strict=strict, **kw)
        self._engine_stale = True
        return out

    def _apply(self, fn, *a, **k):
        self._engine_stale = True
        return super()._apply(fn, *a, **k)

    def engine(self) -> Engine:
        if self._engine is None or self._engine_stale:
            p = next(self.parameters())
            if not p.is_cuda:
                raise RuntimeError("GenerativeImageTextModel runs only on a CUDA device (B200): call .to('cuda') first; "
                                   "there is no CPU path")
            if self._engine is None or self._engine.device != p.device:
                cfg = make_config(self.param, self.sos_index, self.eos_index, vocab=self.textual.vocab_size,
                                  hidden=self.textual.hidden_size, layers=self.textual.num_layers,
                                  heads=self.textual.attention_heads, ffn=self.textual.feedforward_size,
                                  max_positions=self.textual.max_caption_length)
                self._engine = Engine(cfg, p.device.index or 0)
            else:
                cfg = self._engine.cfg
                self._engine.close()
                self._engine = Engine(cfg, p.device.index or 0)
            self._engine.load_state_dict(self.state_dict())
            self._engine_stale = False
            self._vf_token = None
        return self._engine

    # ---- forward hooks (the reference's DistillationTrainer registers them at model.py:847 and :857)
    def _hooked_resblocks(self):
        return [i for i, blk in enumerate(self.image_encoder.transformer.resblocks) if len(blk._forward_hooks) > 0]

    def _arm_vit_taps(self, eng: Engine, n_clips: int, n_frames: int):
        layers = self._hooked_resblocks()
        return (layers, eng.set_vit_taps(layers, n_clips, n_frames)) if layers else (layers, None)

    def _fire_vit_hooks(self, eng: Engine, layers, taps) -> None:
        """Call the registered forward hooks the way the reference's per-clip loop would have: once per clip, with the
        resblock output in the upstream [T, F, Dv] (sequence-first) layout (read as ``[:, 0]`` at model.py:912)."""
        if not layers:
            return
        eng.set_vit_taps([])
        for c in range(taps.shape[1]):
            for j, li in enumerate(layers):
                blk = self.image_encoder.transformer.resblocks[li]
                out = taps[j, c].permute(1, 0, 2)
                for hook in list(blk._forward_hooks.values()):
                    hook(blk, (None,), out)

    def _fire_decoder_hooks(self, hidden: torch.Tensor) -> None:
        """``textual.transformer.encoder.layer[i].output`` hooks (model.py:857): the module's output is the layer's
        output hidden state = hidden_states[i + 1]; fired per clip with the reference's [1, Nv+L, H] shape."""
        layers = self.textual.transformer.encoder.layer
        if not any(len(l.output._forward_hooks) for l in layers):
            return
        for c in range(hidden.shape[0]):
            for i, l in enumerate(layers):
                for hook in list(l.output._forward_hooks.values()):
                    hook(l.output, (None, None), hidden[c:c + 1, i + 1])

    @staticmethod
    def _stack_frames(images) -> torch.Tensor:
        """batch['image']: list of F tensors [B,3,H,W] (the reference passes B == 1) -> [B,F,3,H,W]."""
        return torch.stack([im if im.dim() == 4 else im.unsqueeze(0) for im in images], dim=1).float()

    # ---- forward paths
    @torch.no_grad()
    def forward_one_custom(self, batch, return_info=False):
        """model.py:371-424: (logits [B,L,V], visual_features [B,Nv,Dv], hidden_states [7,Nv+L,H] for B == 1)."""
        if "context" in batch:
            raise NotImplementedError("'context' inputs are not used by the reference path")
        has_image = "image" in batch
        assert has_image, "text-only forward is not part of the captioning path"
        if self.pooling_images is not None:
            raise NotImplementedError
        eng = self.engine()
        tokens = batch["caption_tokens"]
        if not isinstance(batch["image"], (list, tuple)):  # single image per sample: no temporal embedding (:387-388)
            vf = eng.encode_images(batch["image"].float().to(eng.device))
            logits, _, hidden = eng.forward_logits(None, tokens, want_hidden=True, want_features=False)
            self._vf_token = None
            return logits, vf, (hidden[0] if hidden.shape[0] == 1 else hidden)
        frames = self._stack_frames(batch["image"]).to(eng.device)
        layers, taps = self._arm_vit_taps(eng, frames.shape[0], frames.shape[1])
        logits, vf, hidden = eng.forward_logits(frames, tokens, want_hidden=True, want_features=True)
        self._fire_vit_hooks(eng, layers, taps)
        self._fire_decoder_hooks(hidden)
        self._vf_token = None
        hidden_states = hidden[0] if hidden.shape[0] == 1 else hidden  # reference squeezes the batch dim (B == 1)
        return logits, vf, hidden_states

    def forward(self, batch):
        """Eval-mode CaptioningModel.forward (model.py:768): encode the clip(s), then ``infer``."""
        if self.training:
            raise NotImplementedError("the GIT teacher is frozen (model.py:741-745); training forward is out of scope")
        with torch.no_grad():
            eng = self.engine()
            if not isinstance(batch["image"], (list, tuple)):  # single image per sample (model.py:387-388)
                vf = eng.encode_images(batch["image"].float().to(eng.device))
                self._vf_token = vf
                return self.infer(batch, vf, None)
            frames = self._stack_frames(batch["image"]).to(eng.device)
            layers, taps = self._arm_vit_taps(eng, frames.shape[0], frames.shape[1])
            vf = eng.encode(frames, want_features=True)
            self._fire_vit_hooks(eng, layers, taps)
            self._vf_token = vf
            return self.infer(batch, vf, None)

    @torch.no_grad()
    def forward_host_frames(self, frames_host: torch.Tensor, chunk_clips: int = 64):
        """``forward`` for a batch of clips that still lives on the HOST (fp32 [B, F, 3, R, R]): same result dict, but the
        frames cross PCIe in chunks whose copies overlap the ViT of the previous chunk (gitb200_caption_from_host)
        instead of one blocking ``.to(device)`` in front of everything."""
        if self.training:
            raise NotImplementedError("the GIT teacher is frozen (model.py:741-745); training forward is out of scope")
        eng = self.engine()
        sc = self.decoder.search_config(1, self.cache_reorder == "correct")
        tokens, logprobs, logits, vf = eng.caption_from_host(frames_host, sc, chunk_clips=chunk_clips, save_logits=True,
                                                             want_features=True)
        self.prev_encoded_layers = None
        self._vf_token = vf
        return {"predictions": tokens.long().squeeze(1), "logprobs": logprobs, "logits_dict": LazyLogits(logits, eng.cfg.vocab),
                "visual_features": vf}

    def decoding_step(self, visual_features, visual_features_valid, bi_valid_mask_caption, partial_captions):
        """Upstream CaptioningModel.decoding_step with use_history_for_infer: scores of the last position."""
        eng = self.engine()
        B = visual_features.shape[0]
        rows = partial_captions.shape[0]
        if self.prev_encoded_layers is None:
            if self._vf_token is not visual_features:
                eng.set_visual_features(visual_features.to(eng.device))
                self._vf_token = visual_features
            if rows % B != 0:
                raise ValueError(f"decoding_step: {rows} caption rows for {B} clips")
            eng.decode_begin(rows // B)
            for p in range(partial_captions.shape[1] - 1):  # prefix tokens fill the cache
                eng.decode_step(partial_captions[:, p], p)
            self.prev_encoded_layers = ("gitb200-kv-cache", rows)
        pos = partial_captions.shape[1] - 1
        return eng.decode_step(partial_captions[:, pos], pos).float()

    def infer(self, batch, visual_features, visual_features_valid, search_param=None):
        """model.py:426-462.

        ``search_param['seed']`` (not a reference key) opts into the device's counter-based RNG: sampling, repetition
        penalty and num_return_sequences then run in the fused device search, reproducible for a given seed but not
        token-identical to torch's RNG.  Without it those settings take the generic host loop, as the reference does.

        ``search_param['device_prefix'] = True`` (not a reference key) lets ``batch['prefix']`` (int [1 or B, P]) take the
        fused device search too: one decoder pass over the prompt, then the search from cur_len = P.  The prompt's K/V come
        from a differently shaped GEMM than the host loop's per-token steps, so results agree with it within the parity
        tolerances, not bit for bit.  Without it a prefix takes the host loop, as before."""
        batch_size = visual_features.size(0)
        search_param = dict(search_param or {})
        seed = search_param.pop("seed", None)
        device_prefix = bool(search_param.pop("device_prefix", False))
        eng = self.engine()
        fused = (isinstance(self.decoder, GeneratorWithBeamSearchV2) and ("prefix" not in batch or device_prefix)
                 and visual_features_valid is None and not self._force_host_search)
        fast = (fused and not search_param.get("do_sample", False) and search_param.get("num_return_sequences", 1) == 1
                and self.decoder.repetition_penalty == 1.0)
        sample = None
        if fused and seed is not None:
            do_sample = bool(search_param.get("do_sample", False))
            top_k, top_p = search_param.get("top_k"), search_param.get("top_p")
            if do_sample and (top_k is None or top_p is None):  # upstream top_k_top_p_filtering compares them with numbers
                raise TypeError(f"sampling needs top_k and top_p (got top_k={top_k!r}, top_p={top_p!r})")
            sample = SampleConfig(do_sample, int(top_k or 0), 1.0 if top_p is None else float(top_p), self.decoder.temperature,
                                  self.decoder.repetition_penalty, search_param.get("num_return_sequences", 1), int(seed))
            fast = True
        self.prev_encoded_layers = None
        if fast:
            if self._vf_token is not visual_features:
                eng.set_visual_features(visual_features.to(eng.device))
                self._vf_token = visual_features
            sc = self.decoder.search_config(search_param.get("num_keep_best", 1), self.cache_reorder == "correct")
            if "prefix" in batch:
                tokens, logprobs, logits = eng.decode(batch_size, sc, save_logits=True, sample=sample, prefix=batch["prefix"])
            elif sample is None:
                tokens, logprobs, logits = eng.decode(batch_size, sc, save_logits=True)
            else:
                tokens, logprobs, logits = eng.decode(batch_size, sc, save_logits=True, sample=sample)
            predicted = tokens.long()
            if sc.num_keep_best == 1:
                predicted = predicted.squeeze(1)
            if "prefix" in batch:  # the reference's strip, on whatever shape the search returned (keep > 1: the keep dimension)
                predicted = predicted[:, batch["prefix"].shape[1]:]
            logits_dict = LazyLogits(logits, eng.cfg.vocab)
        else:
            if "prefix" not in batch:
                start = torch.full((batch_size, 1), self.sos_index, dtype=torch.long, device=eng.device)
            else:
                assert len(batch["prefix"]) == 1, "not supported"
                start = batch["prefix"].long().to(eng.device)
            step = functools.partial(self.decoding_step, visual_features, visual_features_valid,
                                     batch.get("bi_valid_mask_caption"))
            if self.cache_reorder == "correct" and isinstance(self.decoder, GeneratorWithBeamSearchV2):
                # the K/V cache follows the beams exactly like the fused device search does under the same setting
                search_param = dict(search_param, on_reorder=lambda beam_idx, pos: eng.decode_reorder(beam_idx, pos))
            predicted, logprobs, logits_dict = self.decoder.search(start, step, **search_param)
            if "prefix" in batch:
                predicted = predicted[:, start.shape[1]:]
        return {"predictions": predicted, "logprobs": logprobs, "logits_dict": logits_dict,
                "visual_features": visual_features}


def get_git_model(tokenizer, param):
    """model.py:681-718 (random-initialised parameters; load a checkpoint with load_state_dict)."""
    image_encoder = CLIPVisionTower(param.get("image_encoder_type", "CLIPViT_B_16"),
                                    input_resolution=param.get("test_crop_size", 224))
    text_decoder = TransformerDecoderTextualHead(
        visual_feature_size=param.get("visual_feature_size", 768), vocab_size=VOCAB_SIZE, hidden_size=768, num_layers=6,
        attention_heads=12, feedforward_size=768 * 4, max_caption_length=1024, mask_future_positions=True, padding_idx=0,
        decoder_type="bert_en", output_hidden_states=True, visual_projection_type="linearLn")
    decoder = GeneratorWithBeamSearchV2(eos_index=tokenizer.sep_token_id, max_steps=15, beam_size=4, length_penalty=0.6)
    return GenerativeImageTextModel(image_encoder, text_decoder, decoder=decoder, tokenizer=tokenizer, param=param)


# ----------------------------------------------------------------------------------------------
# teacher wrapper
# ----------------------------------------------------------------------------------------------
class SyntheticTokenizer:
    """Stand-in for BertTokenizer('bert-base-uncased') when its vocabulary file is not available (offline):
    same special ids (CLS 101, SEP 102, PAD 0), ``decode`` renders token ids as words ``t<id>``."""
    cls_token_id, sep_token_id, pad_token_id = 101, 102, 0
    vocab_size = VOCAB_SIZE

    def decode(self, ids, skip_special_tokens=True):
        special = {self.cls_token_id, self.sep_token_id, self.pad_token_id}
        return " ".join(f"t{int(i)}" for i in ids if not (skip_special_tokens and int(i) in special))


def _load_tokenizer():
    try:
        from transformers import BertTokenizer
        tok = BertTokenizer.from_pretrained("bert-base-uncased", do_lower_case=True)
        if tok.cls_token_id == 101 and tok.sep_token_id == 102 and len(tok) >= VOCAB_SIZE:
            return tok
    except Exception:
        pass
    return SyntheticTokenizer()  # offline images return a 5-token stub vocabulary (SURVEY Appendix C)


class GenerativeImageTextTeacher(nn.Module):
    """model.py:721-793.  ``forward`` / ``forward_output_logits`` keep the reference's per-clip return
    structures but run all clips of ``x`` as one batch on the GPU."""

    def __init__(self, param_path: Optional[str] = None, pretrained_weights: Optional[str] = None, *, param: Optional[dict] = None,
                 tokenizer=None, state_dict=None, device="cuda"):
        super().__init__()
        self.tokenizer = tokenizer or _load_tokenizer()
        if param is None:
            import yaml
            with open(param_path) as fh:
                param = yaml.safe_load(fh)
        self.param = param
        self.model = get_git_model(self.tokenizer, self.param)
        if pretrained_weights is not None:
            ckpt = torch.load(pretrained_weights, map_location="cpu")["model"]      # model.py:736-737
            self._load_checked(ckpt)
        elif state_dict is not None:
            self._load_checked(state_dict)
        for p in self.model.parameters():                                            # model.py:741-742
            p.requires_grad = False
        self.model.eval()                                                            # model.py:745
        self.model.to(device)

    def _load_checked(self, sd) -> None:
        """The upstream loader (model.py:738) is tolerant; a silently half-loaded teacher would caption garbage, so every
        parameter of the path must be present (``image_encoder.proj`` and a tied ``textual.output.weight`` are the only
        benign differences, both handled by the model's load_state_dict) and unknown keys are reported."""
        res = self.model.load_state_dict(sd, strict=False)
        if res.missing_keys:
            raise KeyError(f"checkpoint lacks {len(res.missing_keys)} parameter(s) of the GIT path, e.g. {res.missing_keys[:5]}: "
                           "they would stay at their random initialisation")
        if res.unexpected_keys:
            import warnings
            warnings.warn(f"checkpoint holds {len(res.unexpected_keys)} key(s) the GIT path does not use, e.g. "
                          f"{res.unexpected_keys[:5]}")

    @classmethod
    def from_random_init(cls, param: dict, state_dict=None, device="cuda", tokenizer=None):
        """Benchmark / parity constructor: no checkpoint file, no YAML (SURVEY 8b)."""
        return cls(param=param, state_dict=state_dict, device=device, tokenizer=tokenizer or SyntheticTokenizer())

    @torch.no_grad()
    def forward_output_logits(self, x, y):
        """model.py:747-760: lists (one entry per clip) of logits [1,L,V], visual features [1,Nv,Dv],
        hidden states [7,Nv+L,H]."""
        m = self.model
        eng = m.engine()
        frames = x.to(eng.device).float()
        layers, taps = m._arm_vit_taps(eng, frames.shape[0], frames.shape[1])
        logits, vf, hidden = eng.forward_logits(frames, y, want_hidden=True, want_features=True)
        m._vf_token = None  # the engine now holds these clips' features, not the tensor a previous infer() was given
        m._fire_vit_hooks(eng, layers, taps)
        m._fire_decoder_hooks(hidden)
        n = frames.shape[0]
        return [logits[i:i + 1] for i in range(n)], [vf[i:i + 1] for i in range(n)], [hidden[i] for i in range(n)]

    @torch.no_grad()
    def forward(self, x):
        """model.py:762-793: one result dict per clip with predictions / logprobs / logits_dict / visual_features /
        output / cap.  The reference's per-clip post-processing (:771-789) runs batched: ONE device->host copy of the
        token matrix, one gather + argmax + gather over all clips and steps; the per-clip entries are views."""
        m = self.model
        eng = m.engine()
        n = x.shape[0]
        nb = m.decoder.beam_size
        fast = (isinstance(m.decoder, GeneratorWithBeamSearchV2) and m.decoder.repetition_penalty == 1.0
                and not m._force_host_search and not m._hooked_resblocks())
        if not x.is_cuda and x.dtype == torch.float32 and fast:
            res = m.forward_host_frames(x)          # host batch: chunked copies overlapped with the ViT
        else:
            frames = x.to(eng.device).float()
            res = m({"image": [frames[:, f] for f in range(frames.shape[1])]})
        ld = res["logits_dict"]
        all_logits = ld.device_tensor()                                   # [steps, n*nb, V] (view of the padded buffer)
        steps, V = all_logits.shape[0], all_logits.shape[-1]
        pred = res["predictions"]                                         # [n, max_steps] int64 on the device
        pred_host = pred.cpu()                                            # the only synchronising copy of the call
        caps = [self.tokenizer.decode(row, skip_special_tokens=True) for row in pred_host.tolist()]          # :771
        ks = [min(len(c.split(" ")), steps) for c in caps]                                                   # :772
        K = max(ks) if ks else 0
        # [n, K, nb, V]: distribution of every beam row for each of the first K predicted words of every clip       # :776
        dist = all_logits[:K].view(K, n, nb, V).permute(1, 0, 2, 3)
        words = pred[:, 1:K + 1]                                                                              # :780
        if words.shape[1] < K:  # max_steps - 1 scored steps, max_steps - 1 words after SOS: cannot happen; guard anyway
            K = words.shape[1]
            dist = dist[:, :K]
        at_word = torch.gather(dist, 3, words[:, :, None, None].expand(n, K, nb, 1)).squeeze(3)              # [n, K, nb]
        idx = at_word.argmax(dim=2)                                                                           # :784
        picked = torch.gather(dist, 2, idx[:, :, None, None].expand(n, K, 1, V)).squeeze(2)                  # :787  [n, K, V]
        dev_logits = ld._dev.view(steps, n, nb, -1)
        out = []
        for i in range(n):
            out.append({"predictions": pred[i:i + 1], "logprobs": res["logprobs"][i:i + 1],
                        "logits_dict": LazyLogits(dev_logits[:, i], eng.cfg.vocab),
                        "visual_features": res["visual_features"][i:i + 1], "output": picked[i:i + 1, :ks[i]], "cap": caps[i]})
        return out

    # ---- the generate facade the reference's scripts call on their model (inference.py:51, real_time_inference.py:58)
    @torch.no_grad()
    def greedy_decode(self, src, max_len: int):
        """[B,F,3,H,W] -> LongTensor [B, <= max_len+1] starting with CLS (StudentCandidateV1.greedy_decode contract,
        model.py:156-187): beam 1 over the GIT decoder."""
        return self._generate(src, max_len, 1)

    @torch.no_grad()
    def beam_search(self, src, max_len: int, k: int = 4):
        return self._generate(src, max_len, k)

    def _generate(self, src, max_len, k):
        eng = self.model.engine()
        frames = src.to(eng.device).float()
        eng.encode(frames, want_features=False)
        self.model._vf_token = None
        sc = SearchConfig(beam_size=k, max_steps=max_len + 1, length_penalty=self.model.decoder.length_penalty,
                          per_node_beam_size=self.model.decoder.per_node_beam_size, num_keep_best=1,
                          reorder_cache=self.model.cache_reorder == "correct")
        tokens, _, _ = eng.decode(frames.shape[0], sc, save_logits=False)
        return tokens[:, 0].long()


_M64 = 2 ** 64 - 1
_SAMPLE_KEYS = ("do_sample", "top_k", "top_p", "temperature", "repetition_penalty", "num_return_sequences", "seed")


def _splitmix64(x: int) -> int:
    """splitmix64 (Steele, Lea, Flood 2014): a bijection of 64-bit words with full avalanche."""
    z = (x + 0x9E3779B97F4A7C15) & _M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M64
    return z ^ (z >> 31)


def stream_key(seed: int, stream_id: int, n: int) -> int:
    """The Philox key of camera ``stream_id``'s ``n``-th sampled caption (n = 0, 1, ...) under ``seed``:
    splitmix64(splitmix64(seed) ^ ((stream_id + 1) << 32 | n)).  splitmix64 is a bijection, so under one seed two different
    (stream_id, n) pairs never share a key (stream_id < 2^31 - 1, n < 2^32)."""
    stream_id, n = int(stream_id), int(n)
    if not (0 <= stream_id < 2 ** 31 - 1 and 0 <= n < 2 ** 32):
        raise ValueError(f"stream_key: stream_id {stream_id} or caption count {n} out of range")
    return _splitmix64(_splitmix64(int(seed) & _M64) ^ ((stream_id + 1) << 32 | n))


def _sample_config(sample: Optional[dict]):
    """The captioners' ``sample`` dict (search_param names) -> (SampleConfig, seed), or (None, None)."""
    if sample is None:
        return None, None
    unknown = set(sample) - set(_SAMPLE_KEYS)
    if unknown:
        raise ValueError(f"unknown sample keys {sorted(unknown)} (expected some of {list(_SAMPLE_KEYS)})")
    top_k, top_p = sample.get("top_k"), sample.get("top_p")
    cfg = SampleConfig(bool(sample.get("do_sample", False)), int(top_k or 0), 1.0 if top_p is None else float(top_p),
                       float(sample.get("temperature", 1.0)), float(sample.get("repetition_penalty", 1.0)),
                       int(sample.get("num_return_sequences", 1)))
    return cfg, int(sample.get("seed", 0))


def _prompt_ids(prompt, vocab: int, max_steps: int):
    """A camera's prompt (token ids starting with SOS, as one row of batch['prefix']: a list, a 1-D tensor or a [1, P] tensor)
    -> a tuple of ints, or None for None.  Rejects an empty prompt, a token outside [0, vocab) and a prompt that leaves the
    search no step (P >= max_steps = max_len + 1)."""
    if prompt is None:
        return None
    if isinstance(prompt, torch.Tensor):
        if prompt.dtype.is_floating_point or prompt.dtype.is_complex or prompt.dtype == torch.bool:
            raise ValueError(f"prompt must hold integer token ids (got {prompt.dtype})")
        if prompt.dim() == 2 and prompt.shape[0] == 1:
            prompt = prompt[0]
        if prompt.dim() != 1:
            raise ValueError(f"prompt must be one row of token ids (got shape {tuple(prompt.shape)})")
        ids = tuple(int(t) for t in prompt.tolist())
    else:
        ids = tuple(prompt)
        if not all(isinstance(t, int) and not isinstance(t, bool) for t in ids):
            raise ValueError(f"prompt must hold integer token ids (got {prompt!r})")
    if not ids:
        raise ValueError("prompt must hold at least one token (start it with SOS)")
    bad = [t for t in ids if not 0 <= t < vocab]
    if bad:
        raise ValueError(f"prompt token {bad[0]} lies outside the vocabulary [0, {vocab})")
    if len(ids) >= max_steps:
        raise ValueError(f"a prompt of {len(ids)} tokens leaves no caption token within max_len {max_steps - 1}")
    return ids


def _decode_rows(tokenizer, rows, nrs: int):
    """Token rows [k*nrs, max_steps] -> k captions: a string each, or with nrs > 1 a list of nrs strings each."""
    texts = [tokenizer.decode(r, skip_special_tokens=True) for r in rows]
    return texts if nrs == 1 else [texts[i:i + nrs] for i in range(0, len(texts), nrs)]


class StreamingCaptioner:
    """The webcam loop of src/real_time_inference.py:38-61 on the GPU: every `stride`-th frame is preprocessed
    (image_transform, :16-28) and its ViT features are computed as it arrives; once `window` frames are held the caption
    is decoded -- only ONE frame's ViT stands between the last frame and its caption.  ``sliding=False`` reproduces the
    reference (``frames.clear()`` after each caption, :61); ``sliding=True`` re-captions on every new frame with
    per-frame feature reuse.

    ``sample`` (a dict with search_param's names: do_sample, top_k, top_p, temperature, repetition_penalty,
    num_return_sequences, seed) samples / penalises in the fused device search; the n-th caption draws with the key
    ``stream_key(seed, 0, n)``, so every window gets fresh uniforms.  With num_return_sequences > 1 a caption is a list of
    strings.

    ``prompt`` (token ids starting with SOS, as one row of batch['prefix']) starts every caption's search from that prompt,
    e.g. a question; the caption is the text after it (the reference's strip, ``predicted[:, P:]``).  ``set_prompt``
    changes or clears it."""

    def __init__(self, teacher: GenerativeImageTextTeacher, stride: int = 3, max_len: int = 25, beam_size: int = 1,
                 sliding: bool = False, sample: Optional[dict] = None, prompt=None):
        from .engine import preprocess_frames
        self._pre = preprocess_frames
        self.teacher, self.stride, self.sliding = teacher, stride, sliding
        self.engine = teacher.model.engine()
        self.window = teacher.model.num_image_with_embedding or 6
        d = teacher.model.decoder
        self.search = SearchConfig(beam_size=beam_size, max_steps=max_len + 1, length_penalty=d.length_penalty,
                                   per_node_beam_size=d.per_node_beam_size, num_keep_best=1)
        self._counter = 0
        self.sample, self.seed = _sample_config(sample)
        self._n_captions = 0
        self._raw, self._raw_key = None, None
        self.latest_caption = ""
        self.set_prompt(prompt)
        self.engine.stream_reset()

    def set_prompt(self, prompt) -> None:
        """The prompt of the following captions (None: none); checked here, before any frame is captioned."""
        self.prompt = _prompt_ids(prompt, self.engine.cfg.vocab, self.search.max_steps) if prompt is not None else None

    @torch.no_grad()
    def push(self, frame_bgr_u8: torch.Tensor) -> Optional[str]:
        """frame: uint8 [H, W, 3] BGR (what cv2.VideoCapture.read returns).  Returns a new caption or None."""
        self._counter += 1
        if self._counter < self.stride:
            return None
        self._counter = 0
        # one persistent device buffer per frame size: the same pointer on every push lets the library replay its CUDA
        # graph of (fused image_transform + patch embed + ViT) instead of launching the ~90 kernels one by one
        key = tuple(frame_bgr_u8.shape)
        if self._raw is None or self._raw_key != key:
            self._raw = torch.empty(key, dtype=torch.uint8, device=self.engine.device)
            self._raw_key = key
        self._raw.copy_(frame_bgr_u8, non_blocking=True)
        self.teacher.model._vf_token = None  # the window's features replace whatever an earlier infer() left resident
        held = self.engine.stream_push_u8(self._raw)
        if held < self.window:
            return None
        P = len(self.prompt) if self.prompt is not None else 0
        kw = {"prefix": torch.tensor([self.prompt], dtype=torch.int32)} if self.prompt is not None else {}
        if self.sample is None:
            tokens, _ = self.engine.stream_caption(self.search, **kw)
            self.latest_caption = self.teacher.tokenizer.decode(tokens[0, 0, P:].tolist(), skip_special_tokens=True)
        else:
            x = dataclasses.replace(self.sample, seed=stream_key(self.seed, 0, self._n_captions))
            self._n_captions += 1
            tokens, _, _ = self.engine.stream_caption(self.search, sample=x, **kw)
            self.latest_caption = _decode_rows(self.teacher.tokenizer, tokens[:, 0, P:].tolist(), x.num_return_sequences)[0]
        if not self.sliding:
            self.engine.stream_reset()
        return self.latest_caption


class MultiStreamCaptioner:
    """The webcam loop of src/real_time_inference.py:38-61 for many cameras on ONE engine: every camera (stream id
    0 .. n_streams-1) has its own stride counter and its own window of per-frame ViT features in the engine's stream pool.
    ``push({id: frame})`` takes the frames that arrived this tick; the frames due (every `stride`-th of each camera) are
    encoded as one ViT batch per frame size, and the windows that completed are captioned as one decode batch per
    held-frame count.  ``sliding=False`` reproduces the reference (``frames.clear()`` after each caption, :61);
    ``sliding=True`` re-captions a camera on every frame it pushes, reusing the other frames' features.
    The constructor (re)configures the engine's pool: one captioner per engine.

    ``sample`` (a dict with search_param's names: do_sample, top_k, top_p, temperature, repetition_penalty,
    num_return_sequences, seed) samples / penalises in the pool's fused device search.  Each camera counts the captions it
    has received since the captioner was built (``reset`` keeps the count), and camera i's n-th caption draws with the key
    ``stream_key(seed, i, n)``: its samples depend neither on which cameras share a call nor on earlier windows' uniforms.
    With num_return_sequences > 1 a camera's caption is a list of strings.

    ``prompt`` (token ids starting with SOS, as one row of batch['prefix']) is every camera's default prompt, e.g. a
    question; ``set_prompt(id, prompt)`` gives one camera its own (None: none).  A prompted caption is the text after the
    prompt (the reference's strip, ``predicted[:, P:]``).  The windows due are captioned as one pool call per (held frames,
    prompt length), with the group's prompts as a [k, P] prefix; cameras without a prompt make exactly the calls they make
    without this option."""

    def __init__(self, teacher: GenerativeImageTextTeacher, n_streams: int, stride: int = 3, max_len: int = 25, beam_size: int = 1,
                 sliding: bool = False, sample: Optional[dict] = None, prompt=None):
        if n_streams < 1 or stride < 1:
            raise ValueError("n_streams and stride must be >= 1")
        self.teacher, self.n_streams, self.stride, self.sliding = teacher, n_streams, stride, sliding
        self.engine = teacher.model.engine()
        self.window = teacher.model.num_image_with_embedding or 6
        d = teacher.model.decoder
        self.search = SearchConfig(beam_size=beam_size, max_steps=max_len + 1, length_penalty=d.length_penalty,
                                   per_node_beam_size=d.per_node_beam_size, num_keep_best=1)
        self._counter = [0] * n_streams
        self.sample, self.seed = _sample_config(sample)
        self._n_captions = [0] * n_streams
        self._raw = {}  # (k, H, W) -> persistent device buffer: repeated shapes replay the library's CUDA graphs
        self.latest_caption = [""] * n_streams
        prompt = _prompt_ids(prompt, self.engine.cfg.vocab, self.search.max_steps) if prompt is not None else None
        self._prompts = [prompt] * n_streams
        self.engine.streams_configure(n_streams)

    def set_prompt(self, stream_id: int, prompt) -> None:
        """Camera ``stream_id``'s prompt for its following captions (None: none); checked here, before any frame is captioned."""
        if not 0 <= stream_id < self.n_streams:
            raise KeyError(f"unknown stream id {stream_id} (this captioner has ids 0..{self.n_streams - 1})")
        self._prompts[stream_id] = (_prompt_ids(prompt, self.engine.cfg.vocab, self.search.max_steps)
                                    if prompt is not None else None)

    def reset(self, stream_ids) -> None:
        """Empty the windows (and stride counters) of these cameras, e.g. after a scene cut or a reconnect."""
        ids = list(stream_ids)
        for sid in ids:
            self._counter[sid] = 0
        self.engine.streams_reset(ids)

    @torch.no_grad()
    def push(self, frames: Dict[int, torch.Tensor]) -> Dict[int, str]:
        """frames: {stream id: uint8 [H, W, 3] BGR frame} for the cameras that delivered one this tick (host or device).
        Returns {stream id: new caption} for the cameras whose window produced a caption."""
        due = []
        for sid, frame in frames.items():
            if not 0 <= sid < self.n_streams:
                raise KeyError(f"unknown stream id {sid} (this captioner has ids 0..{self.n_streams - 1})")
            self._counter[sid] += 1
            if self._counter[sid] < self.stride:
                continue
            self._counter[sid] = 0
            due.append((sid, frame))
        if not due:
            return {}
        self.teacher.model._vf_token = None  # the pool's windows replace whatever an earlier infer() left resident
        for (h, w), group in _group_by(due, lambda it: tuple(it[1].shape[:2])).items():
            ids = [sid for sid, _ in group]
            key = (len(ids), h, w)
            if key not in self._raw:
                self._raw[key] = torch.empty(len(ids), h, w, 3, dtype=torch.uint8, device=self.engine.device)
            buf = self._raw[key]
            torch.stack([f.to(buf.device, non_blocking=True) for _, f in group], out=buf)
            self.engine.streams_push_u8(ids, buf)
        ready = [sid for sid, _ in due if self.engine.streams_frames(sid) >= self.window]
        out = {}
        def group(sid):
            p = self._prompts[sid]
            return self.engine.streams_frames(sid), len(p) if p is not None else 0

        for (_, P), ids in _group_by(ready, group).items():
            kw = {"prefix": torch.tensor([self._prompts[sid] for sid in ids], dtype=torch.int32)} if P else {}
            if self.sample is None:
                tokens, _ = self.engine.streams_caption(ids, self.search, **kw)
                captions = [self.teacher.tokenizer.decode(row, skip_special_tokens=True) for row in tokens[:, 0, P:].tolist()]
            else:
                keys = [stream_key(self.seed, sid, self._n_captions[sid]) for sid in ids]
                for sid in ids:
                    self._n_captions[sid] += 1
                tokens, _, _ = self.engine.streams_caption(ids, self.search, sample=self.sample, keys=keys, **kw)
                captions = _decode_rows(self.teacher.tokenizer, tokens[:, 0, P:].tolist(), self.sample.num_return_sequences)
            for sid, caption in zip(ids, captions):
                out[sid] = self.latest_caption[sid] = caption
            if not self.sliding:
                self.engine.streams_reset(ids)
        return out


def _group_by(items, key):
    """Stable grouping: {key: [items in their original order]} with the keys in order of first appearance."""
    groups = {}
    for it in items:
        groups.setdefault(key(it), []).append(it)
    return groups
