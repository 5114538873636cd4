"""Thin Python owner of one gitb200 context (one per GPU).  torch is used only for device memory,
streams and dtype plumbing; every FLOP of the path runs inside libgitb200.so."""
from __future__ import annotations

import ctypes
from dataclasses import dataclass
from typing import Dict, Optional

import torch

from . import _lib
from ._lib import Config, GitB200Error, SampleParams, SearchParams, check

VIT_CONFIGS = {
    # get_image_encoder(param['image_encoder_type']) of the reference (model.py:682-685)
    "CLIPViT_B_16": dict(width=768, layers=12, heads=12, patch=16),
    "CLIPViT_L_14": dict(width=1024, layers=24, heads=16, patch=14),
}


@dataclass
class SearchConfig:
    """GeneratorWithBeamSearchV2 arguments (model.py:702-708) + search() keyword arguments (model.py:479)."""
    beam_size: int = 4
    max_steps: int = 15
    length_penalty: float = 0.6
    per_node_beam_size: int = 2
    num_keep_best: int = 1
    reorder_cache: bool = False  # False = reference behaviour (model.py:623-634 commented out)

    def to_c(self) -> SearchParams:
        return SearchParams(self.beam_size, self.max_steps, self.per_node_beam_size, self.num_keep_best,
                            float(self.length_penalty), 1 if self.reorder_cache else 0)


@dataclass
class SampleConfig:
    """search() sampling keyword arguments (model.py:479-480) and the decoder's repetition_penalty / temperature
    (model.py:524-535), plus the seed of the device's counter-based RNG: a clip's sample depends only on (seed, its index
    in the call, its scores).  The stream pool ignores the seed and takes one key per camera (``Engine.streams_caption``).
    top_k = 0 and top_p = 1.0 disable the filters."""
    do_sample: bool = False
    top_k: int = 0
    top_p: float = 1.0
    temperature: float = 1.0
    repetition_penalty: float = 1.0
    num_return_sequences: int = 1
    seed: int = 0

    def to_c(self) -> SampleParams:
        return SampleParams(1 if self.do_sample else 0, int(self.top_k), float(self.top_p), float(self.temperature),
                            float(self.repetition_penalty), int(self.num_return_sequences), int(self.seed) & (2 ** 64 - 1))


def make_config(param: dict, sos: int, eos: int, *, vocab: int = 30522, hidden: int = 768, layers: int = 6,
                heads: int = 12, ffn: int = 3072, max_positions: int = 1024, embed_ln_eps: float = 1e-8) -> Config:
    """`param` is the reference's parameter.yaml dict (model.py:683-688, :368)."""
    v = VIT_CONFIGS[param.get("image_encoder_type", "CLIPViT_B_16")]
    vfs = param.get("visual_feature_size", 768)
    if vfs != v["width"]:
        raise ValueError(f"visual_feature_size {vfs} does not match the {v['width']}-wide vision tower")
    return Config(v["width"], v["layers"], v["heads"], v["patch"], param.get("test_crop_size", 224),
                  hidden, layers, heads, ffn, vocab, max_positions,
                  int(param.get("num_image_with_embedding") or 0),
                  1e-5, 1e-5, embed_ln_eps, 1e-12, sos, eos)


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _prefix_host(prefix) -> torch.Tensor:
    """batch['prefix'] (model.py:432-437) as the C side takes it: int32 [1 or B, P] on the host, contiguous.  The token values
    are checked by the library (before anything is enqueued)."""
    if not isinstance(prefix, torch.Tensor) or prefix.dim() != 2 or prefix.shape[1] < 1:
        raise GitB200Error(f"prefix must be an int tensor [1 or B, P] with P >= 1 (got {getattr(prefix, 'shape', type(prefix))})")
    if prefix.dtype.is_floating_point or prefix.dtype.is_complex or prefix.dtype == torch.bool:
        raise GitB200Error(f"prefix must hold integer token ids (got {prefix.dtype})")
    return prefix.detach().to(device="cpu", dtype=torch.int32).contiguous()


class Engine:
    """One C context bound to one CUDA device."""

    def __init__(self, cfg: Config, device: int = 0):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise GitB200Error("no CUDA device: gitb200 has no CPU fallback")
        self.cfg = cfg
        self.device = torch.device("cuda", device)
        h = ctypes.c_void_p()
        check(self.lib.gitb200_create(ctypes.byref(cfg), device, ctypes.byref(h)), None, "gitb200_create")
        self.h = h
        self.T = self.lib.gitb200_tokens_per_frame(h)
        self.ld = self.lib.gitb200_logits_ld(h)
        self.finalized = False
        self._cur_nv = 0
        self._cur_clips = 0      # clips whose visual features the context holds
        self._step_rows = 0      # rows per clip of the step-wise decoding state (decode_begin)

    def close(self):
        if getattr(self, "h", None):
            self.lib.gitb200_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- weights
    def load_state_dict(self, sd: Dict[str, torch.Tensor]) -> None:
        for name, t in sd.items():
            t = t.detach().to(torch.float32).contiguous()
            shape = (ctypes.c_int64 * max(1, t.dim()))(*t.shape)
            check(self.lib.gitb200_load_weight(self.h, name.encode(), _ptr(t), t.dim(), shape), self.h,
                  f"gitb200_load_weight({name})")
        check(self.lib.gitb200_finalize_weights(self.h), self.h, "gitb200_finalize_weights")
        self.finalized = True

    def reserve(self, max_clips: int, max_frames: int, rows_per_clip: int, max_text_len: int) -> None:
        check(self.lib.gitb200_reserve(self.h, max_clips, max_frames, rows_per_clip, max_text_len), self.h, "gitb200_reserve")

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ---- hot path
    def encode(self, frames: torch.Tensor, want_features: bool = True) -> Optional[torch.Tensor]:
        """frames fp32 [B, F, 3, R, R] on this device -> visual features fp32 [B, F'*T, Dv]."""
        assert frames.is_cuda and frames.dtype == torch.float32 and frames.dim() == 5
        frames = frames.contiguous()
        B, F = frames.shape[:2]
        n = self.cfg.num_image_with_embedding
        Fe = min(F, n) if n > 0 else F
        out = torch.empty(B, Fe * self.T, self.cfg.vit_width, dtype=torch.float32, device=self.device) if want_features else None
        check(self.lib.gitb200_encode(self.h, _ptr(frames), B, F, _ptr(out), self._stream()), self.h, "gitb200_encode")
        self._cur_nv, self._cur_clips, self._step_rows = Fe * self.T, B, 0
        return out

    def encode_images(self, images: torch.Tensor, want_features: bool = True) -> Optional[torch.Tensor]:
        """Single-image branch (model.py:387-388): images fp32 [B, 3, R, R] -> [B, T, Dv], no temporal embedding."""
        assert images.is_cuda and images.dtype == torch.float32 and images.dim() == 4
        images = images.contiguous()
        B = images.shape[0]
        out = torch.empty(B, self.T, self.cfg.vit_width, dtype=torch.float32, device=self.device) if want_features else None
        check(self.lib.gitb200_encode_images(self.h, _ptr(images), B, _ptr(out), self._stream()), self.h, "gitb200_encode_images")
        self._cur_nv, self._cur_clips, self._step_rows = self.T, B, 0
        return out

    def set_vit_taps(self, layers, n_clips: int = 0, n_frames: int = 0) -> Optional[torch.Tensor]:
        """Forward-hook taps on image_encoder.transformer.resblocks[i] (model.py:847).  ``layers`` = resblock indices;
        returns the fp32 buffer [len(layers), n_clips, F', T, Dv] the next encodes fill.  ``layers`` empty: remove."""
        layers = list(layers)
        if not layers:
            check(self.lib.gitb200_set_vit_taps(self.h, None, 0, None), self.h, "gitb200_set_vit_taps")
            self._tap_buf = None
            return None
        n = self.cfg.num_image_with_embedding
        Fe = min(n_frames, n) if n > 0 else n_frames
        buf = torch.empty(len(layers), n_clips, Fe, self.T, self.cfg.vit_width, dtype=torch.float32, device=self.device)
        arr = (ctypes.c_int32 * len(layers))(*layers)
        check(self.lib.gitb200_set_vit_taps(self.h, arr, len(layers), _ptr(buf)), self.h, "gitb200_set_vit_taps")
        self._tap_buf = buf  # keeps the device memory alive while the taps are set
        return buf

    def set_visual_features(self, vf: torch.Tensor) -> None:
        assert vf.is_cuda and vf.dim() == 3
        vf = vf.to(torch.float32).contiguous()
        check(self.lib.gitb200_set_visual_features(self.h, _ptr(vf), vf.shape[0], vf.shape[1], self._stream()), self.h,
              "gitb200_set_visual_features")
        self._cur_nv, self._cur_clips, self._step_rows = vf.shape[1], vf.shape[0], 0

    def _search_outputs(self, n_clips: int, sp: SearchConfig, sample: Optional[SampleConfig], save_logits: bool, P: int = 1):
        n = n_clips * (sample.num_return_sequences if sample is not None else 1)
        tokens = torch.empty(n, sp.num_keep_best, sp.max_steps, dtype=torch.int32, device=self.device)
        logprobs = torch.empty(n, sp.num_keep_best, dtype=torch.float32, device=self.device)
        logits = torch.empty(max(0, sp.max_steps - P), n * sp.beam_size, self.ld, dtype=torch.float32,
                             device=self.device) if save_logits else None
        return tokens, logprobs, logits

    def decode(self, n_clips: int, sp: SearchConfig, save_logits: bool = False, sample: Optional[SampleConfig] = None,
               prefix: Optional[torch.Tensor] = None):
        """Search on the current visual features: (tokens int32 [B, keep, max_steps], logprobs [B, keep],
        logits fp32 [max_steps-1, B*beam, ld] or None).  With ``sample``, B becomes B * num_return_sequences (row
        i * nrs + j = sequence j of clip i) and the logits are the scores before penalty and temperature.
        ``prefix`` (batch['prefix'], int [1 or B, P], host or device): the search starts from that prompt; the tokens then
        include it (the reference's infer strips it) and the logits hold max_steps - P steps."""
        if prefix is not None:
            pre = _prefix_host(prefix)
            tokens, logprobs, logits = self._search_outputs(n_clips, sp, sample, save_logits, pre.shape[1])
            c, x = sp.to_c(), sample.to_c() if sample is not None else None
            check(self.lib.gitb200_decode_prefix(self.h, ctypes.byref(c), ctypes.byref(x) if x is not None else None, _ptr(pre),
                                                 pre.shape[0], pre.shape[1], _ptr(tokens), _ptr(logprobs), _ptr(logits),
                                                 self._stream()), self.h, "gitb200_decode_prefix")
            if logits is not None:
                logits = logits[: self.last_decode_steps()]
            return tokens, logprobs, logits
        tokens, logprobs, logits = self._search_outputs(n_clips, sp, sample, save_logits)
        c = sp.to_c()
        if sample is None:
            check(self.lib.gitb200_decode(self.h, ctypes.byref(c), _ptr(tokens), _ptr(logprobs), _ptr(logits), self._stream()),
                  self.h, "gitb200_decode")
        else:
            x = sample.to_c()
            check(self.lib.gitb200_decode_ext(self.h, ctypes.byref(c), ctypes.byref(x), _ptr(tokens), _ptr(logprobs), _ptr(logits),
                                              self._stream()), self.h, "gitb200_decode_ext")
        if logits is not None:  # the step loop may have stopped early (`if all(done): break`, model.py:640)
            logits = logits[: self.last_decode_steps()]
        return tokens, logprobs, logits

    def caption(self, frames: torch.Tensor, sp: SearchConfig, save_logits: bool = False, sample: Optional[SampleConfig] = None,
                prefix: Optional[torch.Tensor] = None):
        """encode + decode of frames fp32 [B, F, 3, R, R]; ``sample`` and ``prefix`` as in ``decode``."""
        assert frames.is_cuda and frames.dtype == torch.float32 and frames.dim() == 5
        frames = frames.contiguous()
        B, F = frames.shape[:2]
        pre = _prefix_host(prefix) if prefix is not None else None
        tokens, logprobs, logits = self._search_outputs(B, sp, sample, save_logits, pre.shape[1] if pre is not None else 1)
        c = sp.to_c()
        if pre is not None:
            x = sample.to_c() if sample is not None else None
            check(self.lib.gitb200_caption_prefix(self.h, _ptr(frames), B, F, ctypes.byref(c), ctypes.byref(x) if x is not None else None,
                                                  _ptr(pre), pre.shape[0], pre.shape[1], _ptr(tokens), _ptr(logprobs), _ptr(logits),
                                                  self._stream()), self.h, "gitb200_caption_prefix")
        elif sample is None:
            check(self.lib.gitb200_caption(self.h, _ptr(frames), B, F, ctypes.byref(c), _ptr(tokens), _ptr(logprobs),
                                           _ptr(logits), self._stream()), self.h, "gitb200_caption")
        else:
            x = sample.to_c()
            check(self.lib.gitb200_caption_ext(self.h, _ptr(frames), B, F, ctypes.byref(c), ctypes.byref(x), _ptr(tokens),
                                               _ptr(logprobs), _ptr(logits), self._stream()), self.h, "gitb200_caption_ext")
        n = self.cfg.num_image_with_embedding
        self._cur_nv, self._cur_clips, self._step_rows = (min(F, n) if n > 0 else F) * self.T, B, 0
        if logits is not None:
            logits = logits[: self.last_decode_steps()]
        return tokens, logprobs, logits

    def caption_host(self, frames_host: torch.Tensor, sp: SearchConfig, chunk_clips: int = 32):
        """HOST frames fp32 [N, F, 3, R, R] (pinned recommended) -> HOST tokens int32 [N, keep, max_steps], logprobs.
        Synchronous; host->device copies of chunk i+1 overlap the compute of chunk i."""
        assert not frames_host.is_cuda and frames_host.dtype == torch.float32 and frames_host.dim() == 5
        frames_host = frames_host.contiguous()
        N, F = frames_host.shape[:2]
        tokens = torch.empty(N, sp.num_keep_best, sp.max_steps, dtype=torch.int32).pin_memory()
        logprobs = torch.empty(N, sp.num_keep_best, dtype=torch.float32).pin_memory()
        c = sp.to_c()
        with torch.cuda.device(self.device):
            check(self.lib.gitb200_caption_host(self.h, _ptr(frames_host), N, F, chunk_clips, ctypes.byref(c),
                                                _ptr(tokens), _ptr(logprobs)), self.h, "gitb200_caption_host")
        n = self.cfg.num_image_with_embedding
        self._cur_nv, self._cur_clips, self._step_rows = (min(F, n) if n > 0 else F) * self.T, N, 0
        return tokens, logprobs

    def caption_from_host(self, frames_host: torch.Tensor, sp: SearchConfig, chunk_clips: int = 64, save_logits: bool = False,
                          want_features: bool = False):
        """HOST frames fp32 [N, F, 3, R, R] -> DEVICE (tokens, logprobs, logits | None, visual features | None): the host->device
        copy of chunk i+1 overlaps the ViT of chunk i; nothing is copied back.  Asynchronous on the current stream; the caller
        must keep ``frames_host`` alive until that stream has caught up (any read of the results does that)."""
        assert not frames_host.is_cuda and frames_host.dtype == torch.float32 and frames_host.dim() == 5
        frames_host = frames_host.contiguous()
        N, F = frames_host.shape[:2]
        n = self.cfg.num_image_with_embedding
        nv = (min(F, n) if n > 0 else F) * self.T
        tokens = torch.empty(N, sp.num_keep_best, sp.max_steps, dtype=torch.int32, device=self.device)
        logprobs = torch.empty(N, sp.num_keep_best, dtype=torch.float32, device=self.device)
        logits = torch.empty(sp.max_steps - 1, N * sp.beam_size, self.ld, dtype=torch.float32,
                             device=self.device) if save_logits else None
        vf = torch.empty(N, nv, self.cfg.vit_width, dtype=torch.float32, device=self.device) if want_features else None
        c = sp.to_c()
        with torch.cuda.device(self.device):
            check(self.lib.gitb200_caption_from_host(self.h, _ptr(frames_host), N, F, chunk_clips, ctypes.byref(c), _ptr(tokens),
                                                     _ptr(logprobs), _ptr(logits), _ptr(vf), self._stream()), self.h,
                  "gitb200_caption_from_host")
        self._cur_nv, self._cur_clips, self._step_rows = nv, N, 0
        self._host_frames_in_flight = frames_host  # keeps the source alive while the copies are in flight
        if logits is not None:
            logits = logits[: self.last_decode_steps()]
        return tokens, logprobs, logits, vf

    def caption_host_u8(self, frames_host: torch.Tensor, sp: SearchConfig, chunk_clips: int = 32):
        """HOST raw video frames uint8 [N, F, H, W, 3] (OpenCV BGR, pinned recommended) -> HOST tokens, logprobs.
        image_transform() (dataloader.py:18-32) runs on the device between the byte copy and the ViT; synchronous."""
        assert not frames_host.is_cuda and frames_host.dtype == torch.uint8 and frames_host.dim() == 5 and frames_host.shape[-1] == 3
        frames_host = frames_host.contiguous()
        N, F, H, W = frames_host.shape[:4]
        tokens = torch.empty(N, sp.num_keep_best, sp.max_steps, dtype=torch.int32).pin_memory()
        logprobs = torch.empty(N, sp.num_keep_best, dtype=torch.float32).pin_memory()
        c = sp.to_c()
        with torch.cuda.device(self.device):
            check(self.lib.gitb200_caption_host_u8(self.h, _ptr(frames_host), N, F, H, W, chunk_clips, ctypes.byref(c),
                                                   _ptr(tokens), _ptr(logprobs)), self.h, "gitb200_caption_host_u8")
        n = self.cfg.num_image_with_embedding
        self._cur_nv, self._cur_clips, self._step_rows = (min(F, n) if n > 0 else F) * self.T, N, 0
        return tokens, logprobs

    def forward_logits(self, frames: Optional[torch.Tensor], tokens: torch.Tensor, want_hidden: bool = True,
                       want_features: bool = True):
        """Teacher-forced forward (forward_one_custom, model.py:371-424), batched over clips.
        tokens int [B, L] -> (logits fp32 [B, L, vocab], visual_features [B, Nv, Dv] | None,
        hidden_states [B, layers+1, Nv+L, hidden] | None)."""
        tok = tokens.to(device=self.device, dtype=torch.int32).contiguous()
        B, L = tok.shape
        if frames is not None:
            assert frames.is_cuda and frames.dtype == torch.float32 and frames.dim() == 5 and frames.shape[0] == B
            frames = frames.contiguous()
            F = frames.shape[1]
            n = self.cfg.num_image_with_embedding
            nv = (min(F, n) if n > 0 else F) * self.T
        else:
            F = 0
            nv = self._cur_nv
        if frames is None and B != self._cur_clips:
            raise GitB200Error(f"forward_logits: {B} token rows for the {self._cur_clips} clips whose features are resident")
        self._cur_nv, self._cur_clips, self._step_rows = nv, B, 0
        logits = torch.empty(B * L, self.ld, dtype=torch.float32, device=self.device)
        hidden = torch.empty(B, self.cfg.dec_layers + 1, nv + L, self.cfg.hidden, dtype=torch.float32,
                             device=self.device) if want_hidden else None
        vf = torch.empty(B, nv, self.cfg.vit_width, dtype=torch.float32, device=self.device) if want_features else None
        check(self.lib.gitb200_forward_logits(self.h, _ptr(frames), B, F, _ptr(tok), L, _ptr(logits), _ptr(hidden), _ptr(vf),
                                              self._stream()), self.h, "gitb200_forward_logits")
        return logits.view(B, L, self.ld)[:, :, : self.cfg.vocab], vf, hidden

    # ---- step-wise decoding for a generic search loop
    def decode_begin(self, rows_per_clip: int) -> None:
        check(self.lib.gitb200_decode_begin(self.h, rows_per_clip, self._stream()), self.h, "gitb200_decode_begin")
        self._step_rows = rows_per_clip

    def decode_step(self, tokens: torch.Tensor, pos: int) -> torch.Tensor:
        tok = tokens.to(device=self.device, dtype=torch.int32).contiguous()
        # the C side indexes cur_clips * rows_per_clip rows of `tokens` / `logits`: a mismatch would read out of bounds
        if self._step_rows < 1 or tok.numel() != self._cur_clips * self._step_rows:
            raise GitB200Error(f"decode_step: {tok.numel()} token rows, but decode_begin set up {self._cur_clips} clips x "
                               f"{self._step_rows} rows")
        logits = torch.empty(tok.numel(), self.ld, dtype=torch.float32, device=self.device)
        check(self.lib.gitb200_decode_step(self.h, _ptr(tok), pos, _ptr(logits), self._stream()), self.h, "gitb200_decode_step")
        return logits[:, : self.cfg.vocab]

    def decode_reorder(self, beam_idx: torch.Tensor, pos: int) -> None:
        idx = beam_idx.to(device=self.device, dtype=torch.int32).contiguous()
        if idx.numel() != self._cur_clips * self._step_rows:
            raise GitB200Error("decode_reorder: beam_idx must have one entry per decode row")
        check(self.lib.gitb200_decode_reorder(self.h, _ptr(idx), pos, self._stream()), self.h, "gitb200_decode_reorder")

    # ---- streaming window (real_time_inference.py:38-61)
    def stream_reset(self) -> None:
        check(self.lib.gitb200_stream_reset(self.h), self.h, "gitb200_stream_reset")

    def stream_push(self, frame: torch.Tensor) -> int:
        """Encode one preprocessed frame fp32 [3, R, R] (or [1, 3, R, R]) into the window; returns the frames held."""
        assert frame.is_cuda and frame.dtype == torch.float32 and frame.numel() == 3 * self.cfg.resolution ** 2
        frame = frame.contiguous()
        check(self.lib.gitb200_stream_push(self.h, _ptr(frame), self._stream()), self.h, "gitb200_stream_push")
        return int(self.lib.gitb200_stream_frames(self.h))

    def stream_push_u8(self, frame_u8: torch.Tensor) -> int:
        """Encode one RAW frame uint8 [H, W, 3] (OpenCV BGR, on this device) into the window: image_transform() runs fused
        into the patch-embed loader.  Keep pushing from the same buffer and the library replays a CUDA graph."""
        assert frame_u8.is_cuda and frame_u8.dtype == torch.uint8 and frame_u8.dim() == 3 and frame_u8.shape[-1] == 3
        assert frame_u8.is_contiguous()
        h, w = frame_u8.shape[:2]
        check(self.lib.gitb200_stream_push_u8(self.h, _ptr(frame_u8), h, w, self._stream()), self.h, "gitb200_stream_push_u8")
        return int(self.lib.gitb200_stream_frames(self.h))

    def _window_outputs(self, attr: str, k: int, sp: SearchConfig, sample: Optional[SampleConfig]):
        # persistent output buffers: identical call signatures let the library replay its captured CUDA graph
        n = k * (sample.num_return_sequences if sample is not None else 1)
        key = (n, sp.num_keep_best, sp.max_steps)
        bufs = self.__dict__.setdefault(attr, {})
        if key not in bufs:
            bufs[key] = (torch.empty(n, sp.num_keep_best, sp.max_steps, dtype=torch.int32, device=self.device),
                         torch.empty(n, sp.num_keep_best, dtype=torch.float32, device=self.device))
        return bufs[key]

    def _saved_logits(self, n_rows: int, sp: SearchConfig, save_logits: bool, sample: Optional[SampleConfig], P: int = 1):
        if save_logits and sample is None:
            raise GitB200Error("save_logits needs sample (a SampleConfig; SampleConfig() for plain beam search)")
        return torch.empty(max(0, sp.max_steps - P), n_rows * sp.beam_size, self.ld, dtype=torch.float32,
                           device=self.device) if save_logits else None

    def stream_caption(self, sp: SearchConfig, sample: Optional[SampleConfig] = None, save_logits: bool = False,
                       prefix: Optional[torch.Tensor] = None):
        """Caption the single streaming window: (tokens int32 [1, keep, max_steps], logprobs [1, keep]).  With ``sample``
        (its seed is the Philox key) the result equals ``decode(1, sp, sample=sample)`` on the window's features and the
        call returns (tokens [nrs, keep, max_steps], logprobs [nrs, keep], logits or None) as ``decode`` does.
        ``prefix`` (batch['prefix'], int [1, P], host or device): the result equals ``decode(1, sp, prefix=prefix)`` on the
        window's features (the tokens include the prompt, the logits hold max_steps - P steps); the return form is the same."""
        tokens, logprobs = self._window_outputs("_stream_out", 1, sp, sample)
        c = sp.to_c()
        if prefix is not None:
            pre = _prefix_host(prefix)
            if pre.shape[0] != 1:
                raise GitB200Error(f"stream_caption: prefix must have one row (got {pre.shape[0]})")
            logits = self._saved_logits(tokens.shape[0], sp, save_logits, sample, pre.shape[1])
            x = sample.to_c() if sample is not None else None
            check(self.lib.gitb200_stream_caption_prefix(self.h, ctypes.byref(c), ctypes.byref(x) if x is not None else None,
                                                         _ptr(pre), pre.shape[1], _ptr(tokens), _ptr(logprobs), _ptr(logits),
                                                         self._stream()), self.h, "gitb200_stream_caption_prefix")
        elif sample is None:
            check(self.lib.gitb200_stream_caption(self.h, ctypes.byref(c), _ptr(tokens), _ptr(logprobs), self._stream()), self.h,
                  "gitb200_stream_caption")
        else:
            logits = self._saved_logits(tokens.shape[0], sp, save_logits, sample)
            x = sample.to_c()
            check(self.lib.gitb200_stream_caption_ext(self.h, ctypes.byref(c), ctypes.byref(x), _ptr(tokens), _ptr(logprobs),
                                                      _ptr(logits), self._stream()), self.h, "gitb200_stream_caption_ext")
        self._cur_clips, self._cur_nv, self._step_rows = 1, int(self.lib.gitb200_stream_frames(self.h)) * self.T, 0
        if sample is None:
            return tokens.clone(), logprobs.clone()
        return tokens.clone(), logprobs.clone(), logits[: self.last_decode_steps()] if logits is not None else None

    # ---- multi-stream pool: one window per camera, pushes and captions batched over cameras
    @staticmethod
    def _ids(ids):
        ids = [int(i) for i in ids]
        return (ctypes.c_int32 * max(1, len(ids)))(*ids), len(ids)

    def streams_configure(self, n_streams: int) -> None:
        """A pool of ``n_streams`` windows (ids 0 .. n_streams-1), all empty."""
        check(self.lib.gitb200_streams_configure(self.h, n_streams), self.h, "gitb200_streams_configure")

    def streams_push(self, ids, frames: torch.Tensor) -> None:
        """One preprocessed frame per stream: frames fp32 [k, 3, R, R], frame j into the window of stream ids[j]; one ViT batch."""
        R = self.cfg.resolution
        assert frames.is_cuda and frames.dtype == torch.float32 and frames.shape == (len(ids), 3, R, R)
        frames = frames.contiguous()
        arr, k = self._ids(ids)
        check(self.lib.gitb200_streams_push(self.h, arr, k, _ptr(frames), self._stream()), self.h, "gitb200_streams_push")

    def streams_push_u8(self, ids, frames_u8: torch.Tensor) -> None:
        """One RAW frame per stream: uint8 [k, H, W, 3] (OpenCV BGR, on this device), image_transform() fused into the
        patch-embed loader.  Keep pushing from the same buffer and the library replays a CUDA graph."""
        assert frames_u8.is_cuda and frames_u8.dtype == torch.uint8 and frames_u8.dim() == 4 and frames_u8.shape[-1] == 3
        assert frames_u8.is_contiguous() and frames_u8.shape[0] == len(ids)
        h, w = frames_u8.shape[1:3]
        arr, k = self._ids(ids)
        check(self.lib.gitb200_streams_push_u8(self.h, arr, k, _ptr(frames_u8), h, w, self._stream()), self.h,
              "gitb200_streams_push_u8")

    @staticmethod
    def _keys(keys, k: int):
        if keys is None:
            return None
        keys = [int(x) & (2 ** 64 - 1) for x in keys]
        if len(keys) != k:
            raise GitB200Error(f"streams_caption: {len(keys)} keys for {k} stream ids")
        return (ctypes.c_uint64 * k)(*keys)

    def streams_caption(self, ids, sp: SearchConfig, sample: Optional[SampleConfig] = None, keys=None,
                        save_logits: bool = False, prefix: Optional[torch.Tensor] = None):
        """Caption the windows of the streams ``ids`` (all holding the same number of frames) as one decode batch:
        (tokens int32 [k, keep, max_steps], logprobs [k, keep]), row j = stream ids[j].

        With ``sample`` (its seed is ignored), ``keys`` gives the Philox key of each stream (one int per id, required when
        sampling; see model.stream_key) and the call returns (tokens [k*nrs, keep, max_steps], logprobs [k*nrs, keep],
        logits or None): row j*nrs + r is sequence r of stream ids[j].  A stream's result depends on its window, its key,
        the parameters and the number of rows in the call, not on the other streams or their order.

        ``prefix`` (batch['prefix'], int [1 or k, P], host or device; row j is the prompt of stream ids[j]): the result
        equals ``decode(k, sp, sample=..., prefix=prefix)`` on the windows' features, each stream drawing with its key;
        the tokens include the prompt and the logits hold max_steps - P steps.  The return form is the same as without it."""
        arr, k = self._ids(ids)
        tokens, logprobs = self._window_outputs("_streams_out", k, sp, sample)
        c = sp.to_c()
        if prefix is not None:
            pre = _prefix_host(prefix)
            logits = self._saved_logits(tokens.shape[0], sp, save_logits, sample, pre.shape[1])
            x = sample.to_c() if sample is not None else None
            check(self.lib.gitb200_streams_caption_prefix(self.h, arr, k, ctypes.byref(c), ctypes.byref(x) if x is not None else None,
                                                          self._keys(keys, k), _ptr(pre), pre.shape[0], pre.shape[1], _ptr(tokens),
                                                          _ptr(logprobs), _ptr(logits), self._stream()), self.h,
                  "gitb200_streams_caption_prefix")
        elif sample is None:
            check(self.lib.gitb200_streams_caption(self.h, arr, k, ctypes.byref(c), _ptr(tokens), _ptr(logprobs),
                                                   self._stream()), self.h, "gitb200_streams_caption")
        else:
            logits = self._saved_logits(tokens.shape[0], sp, save_logits, sample)
            key_arr = self._keys(keys, k)
            x = sample.to_c()
            check(self.lib.gitb200_streams_caption_ext(self.h, arr, k, ctypes.byref(c), ctypes.byref(x), key_arr, _ptr(tokens),
                                                       _ptr(logprobs), _ptr(logits), self._stream()), self.h,
                  "gitb200_streams_caption_ext")
        self._cur_clips, self._cur_nv, self._step_rows = k, self.streams_frames(int(ids[0])) * self.T, 0
        if sample is None:
            return tokens.clone(), logprobs.clone()
        return tokens.clone(), logprobs.clone(), logits[: self.last_decode_steps()] if logits is not None else None

    def streams_reset(self, ids) -> None:
        arr, k = self._ids(ids)
        check(self.lib.gitb200_streams_reset(self.h, arr, k), self.h, "gitb200_streams_reset")

    def streams_frames(self, stream_id: int) -> int:
        n = int(self.lib.gitb200_streams_frames(self.h, stream_id))
        if n < 0:
            raise GitB200Error(f"gitb200_streams_frames: unknown stream id {stream_id}")
        return n

    def streams_window(self, stream_id: int) -> torch.Tensor:
        """The window of one stream as the decoder sees it (temporal embeddings added, bf16 values): fp32 [n*T, Dv]."""
        n = self.streams_frames(stream_id)
        out = torch.empty(max(1, n) * self.T, self.cfg.vit_width, dtype=torch.float32, device=self.device)
        check(self.lib.gitb200_streams_window(self.h, stream_id, _ptr(out), self._stream()), self.h, "gitb200_streams_window")
        return out

    def set_fold_layernorm(self, enable: bool) -> None:
        """Opt-in (default off, DESIGN.md dead ends): ViT ln_1/ln_2 folded into the QKV/fc1 GEMM epilogues instead of separate LayerNorm kernels."""
        check(self.lib.gitb200_set_fold_layernorm(self.h, 1 if enable else 0), self.h, "gitb200_set_fold_layernorm")

    def set_sweep_rows(self, rows: int) -> None:
        """Token rows per sub-batch of the ViT / visual-pass sweeps of a large batch (0 = one sweep; results are identical)."""
        check(self.lib.gitb200_set_sweep_rows(self.h, rows), self.h, "gitb200_set_sweep_rows")

    def set_early_exit(self, every_steps: int) -> None:
        """Poll the device's finished-clip count every N decode steps and stop early (`if all(done): break`, model.py:640);
        0 = never (fully asynchronous decode)."""
        check(self.lib.gitb200_set_early_exit(self.h, every_steps), self.h, "gitb200_set_early_exit")

    def set_persistent_decode(self, enable: bool) -> None:
        """Single-clip searches as one persistent cooperative kernel (default on; bit-identical to the launch sequence)."""
        check(self.lib.gitb200_set_persistent_decode(self.h, 1 if enable else 0), self.h, "gitb200_set_persistent_decode")

    def last_decode_steps(self) -> int:
        return int(self.lib.gitb200_last_decode_steps(self.h))

    def set_graph_max_clips(self, max_clips: int) -> None:
        check(self.lib.gitb200_set_graph_max_clips(self.h, max_clips), self.h, "gitb200_set_graph_max_clips")

    def set_fuse_layernorm(self, enable: bool) -> None:
        """Opt-in (default off, measured slower): LayerNorms that follow a residual GEMM written by that GEMM as a second output (sweeps of >= 1024 rows)."""
        check(self.lib.gitb200_set_fuse_layernorm(self.h, 1 if enable else 0), self.h, "gitb200_set_fuse_layernorm")

    def set_graph_segments(self, enable: bool) -> None:
        """Large batches replay CUDA graphs of encode / visual pass / decode-step segments (default on); False = eager launches."""
        check(self.lib.gitb200_set_graph_segments(self.h, 1 if enable else 0), self.h, "gitb200_set_graph_segments")

    def set_pipeline(self, chunk_clips: int) -> None:
        """Clips per chunk of the two-stream encode/decode pipeline (0 = off, -1 = automatic)."""
        check(self.lib.gitb200_set_pipeline(self.h, chunk_clips), self.h, "gitb200_set_pipeline")

    def launch_count(self, reset: bool = False) -> int:
        return int(self.lib.gitb200_launch_count(1 if reset else 0))


# ---- single operators (parity tests) -------------------------------------------------------------
def op_gemm(a: torch.Tensor, w: torch.Tensor, bias=None, residual=None, act: int = 0, out_f32: bool = False, tile_n: int = 0):
    lib = _lib.load()
    assert a.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and a.is_cuda
    a, w = a.contiguous(), w.contiguous()
    M, K = a.shape
    N = w.shape[0]
    out = torch.empty(M, N, dtype=torch.bfloat16, device=a.device)
    o32 = torch.empty(M, N, dtype=torch.float32, device=a.device) if out_f32 else None
    if residual is not None:
        residual = residual.contiguous()
    s = ctypes.c_void_p(torch.cuda.current_stream(a.device).cuda_stream)
    check(lib.gitb200_op_gemm(_ptr(a), _ptr(w), M, N, K, _ptr(bias), _ptr(residual), act, _ptr(out), _ptr(o32), tile_n, s),
          None, "gitb200_op_gemm")
    return (out, o32) if out_f32 else out


def op_gemm_ln(a: torch.Tensor, w: torch.Tensor, bias, residual, gamma: torch.Tensor, beta: torch.Tensor, eps: float):
    """(A W^T + bias + residual, LayerNorm of that) from one launch of the CTA-pair GEMM (M >= 1024, N % 256 == 0, N <= 1024)."""
    lib = _lib.load()
    a, w = a.contiguous(), w.contiguous()
    M, K = a.shape
    N = w.shape[0]
    out = torch.empty(M, N, dtype=torch.bfloat16, device=a.device)
    ln = torch.empty(M, N, dtype=torch.bfloat16, device=a.device)
    if residual is not None:
        residual = residual.contiguous()
    s = ctypes.c_void_p(torch.cuda.current_stream(a.device).cuda_stream)
    check(lib.gitb200_op_gemm_ln(_ptr(a), _ptr(w), M, N, K, _ptr(bias), _ptr(residual), _ptr(gamma), _ptr(beta), eps, _ptr(out), _ptr(ln), s),
          None, "gitb200_op_gemm_ln")
    return out, ln


def op_layernorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float):
    lib = _lib.load()
    x = x.contiguous()
    out = torch.empty_like(x)
    s = ctypes.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)
    check(lib.gitb200_op_layernorm(_ptr(x), x.shape[0], x.shape[1], _ptr(gamma), _ptr(beta), eps, _ptr(out), s), None,
          "gitb200_op_layernorm")
    return out


def op_attention_groups(qkv: torch.Tensor, n_groups: int, group_len: int, heads: int, scale: float, legacy_mma: bool = False,
                        out=None):
    """out: None (a new tensor of qkv's rows), or a contiguous bf16 [n_groups * group_len, heads * 64] tensor to write into,
    such as a row range of a larger buffer."""
    lib = _lib.load()
    qkv = qkv.contiguous()
    if out is None:
        out = torch.empty(qkv.shape[0], heads * 64, dtype=torch.bfloat16, device=qkv.device)
    elif not (out.dtype == torch.bfloat16 and out.is_contiguous() and out.shape == (n_groups * group_len, heads * 64)):
        raise ValueError("op_attention_groups: out must be a contiguous bf16 [n_groups * group_len, heads * 64] tensor")
    s = ctypes.c_void_p(torch.cuda.current_stream(qkv.device).cuda_stream)
    fn = lib.gitb200_op_attention_groups_mma if legacy_mma else lib.gitb200_op_attention_groups
    check(fn(_ptr(qkv), _ptr(out), n_groups, group_len, heads, scale, s), None, "gitb200_op_attention_groups")
    return out


def op_text_attention(q: torch.Tensor, vis_kv: torch.Tensor, txt_kv, anc, n_clips: int, rows_per_clip: int, heads: int, scale: float,
                      splits: int = 1):
    """q bf16 [rows, H]; vis_kv bf16 [n_clips, n_vis, 2H]; txt_kv bf16 [n_text, rows, 2H] or None; anc int32 [rows, n_text] or None."""
    lib = _lib.load()
    q, vis_kv = q.contiguous(), vis_kv.contiguous()
    n_text = 0 if txt_kv is None else txt_kv.shape[0]
    if txt_kv is not None:
        txt_kv = txt_kv.contiguous()
    if anc is not None:
        anc = anc.contiguous()
    out = torch.empty(q.shape[0], heads * 64, dtype=torch.bfloat16, device=q.device)
    s = ctypes.c_void_p(torch.cuda.current_stream(q.device).cuda_stream)
    check(lib.gitb200_op_text_attention(_ptr(q), _ptr(vis_kv), _ptr(txt_kv) if txt_kv is not None else None,
                                        _ptr(anc) if anc is not None else None, n_clips, rows_per_clip, heads, vis_kv.shape[1], n_text,
                                        splits, scale, _ptr(out), s), None, "gitb200_op_text_attention")
    return out


def op_search(logits: torch.Tensor, vocab: int, n_clips: int, sos: int, eos: int, sp: SearchConfig,
              sample: Optional[SampleConfig] = None, prefix: Optional[torch.Tensor] = None):
    """logits fp32 [max_steps-1, n_clips*beam, ld] (device) -> tokens [n_clips, keep, max_steps], logprobs.
    With ``sample``: logits [max_steps-1, n_clips*nrs*beam, ld] -> tokens [n_clips*nrs, keep, max_steps].
    With ``prefix`` (int [1 or n_clips, P]): the search starts from that prompt (``sos`` unused), logits [max_steps-P, ...]."""
    lib = _lib.load()
    logits = logits.contiguous()
    n = n_clips * (sample.num_return_sequences if sample is not None else 1)
    tokens = torch.empty(n, sp.num_keep_best, sp.max_steps, dtype=torch.int32, device=logits.device)
    logprobs = torch.empty(n, sp.num_keep_best, dtype=torch.float32, device=logits.device)
    c = sp.to_c()
    s = ctypes.c_void_p(torch.cuda.current_stream(logits.device).cuda_stream)
    if prefix is not None:
        pre = _prefix_host(prefix)
        x = sample.to_c() if sample is not None else None
        check(lib.gitb200_op_search_prefix(_ptr(logits) if logits.numel() else None, logits.shape[-1], vocab, n_clips, eos,
                                           ctypes.byref(c), ctypes.byref(x) if x is not None else None, _ptr(pre), pre.shape[0],
                                           pre.shape[1], _ptr(tokens), _ptr(logprobs), s), None, "gitb200_op_search_prefix")
    elif sample is None:
        check(lib.gitb200_op_search(_ptr(logits), logits.shape[-1], vocab, n_clips, sos, eos, ctypes.byref(c), _ptr(tokens),
                                    _ptr(logprobs), s), None, "gitb200_op_search")
    else:
        x = sample.to_c()
        check(lib.gitb200_op_search_ext(_ptr(logits), logits.shape[-1], vocab, n_clips, sos, eos, ctypes.byref(c),
                                        ctypes.byref(x), _ptr(tokens), _ptr(logprobs), s), None, "gitb200_op_search_ext")
    return tokens, logprobs


def preprocess_frames(frames_u8: torch.Tensor, size: int = 224) -> torch.Tensor:
    """OpenCV frames uint8 [N, H, W, 3] (BGR, on the GPU) -> fp32 [N, 3, size, size] (RGB, CLIP-normalised): the
    reference's image_transform() (src/utils/dataloader.py:18-32) as one CUDA kernel."""
    lib = _lib.load()
    assert frames_u8.is_cuda and frames_u8.dtype == torch.uint8 and frames_u8.dim() == 4 and frames_u8.shape[-1] == 3
    frames_u8 = frames_u8.contiguous()
    n, h, w, _ = frames_u8.shape
    out = torch.empty(n, 3, size, size, dtype=torch.float32, device=frames_u8.device)
    s = ctypes.c_void_p(torch.cuda.current_stream(frames_u8.device).cuda_stream)
    check(lib.gitb200_preprocess(_ptr(frames_u8), n, h, w, size, _ptr(out), s), None, "gitb200_preprocess")
    return out
