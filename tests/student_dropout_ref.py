"""Host-side references for dropout in the student's distillation step: a numpy restatement of the library's Philox masks
(include/gitb200.h, gitb200_student_train_set_dropout) and the step of the stock torch modules in train mode with those masks
injected at torch's own dropout call sites.

nn.TransformerDecoderLayer in train() calls, per layer and in this order (site = 6 * layer + k):
  k = 0  F.scaled_dot_product_attention(..., dropout_p=p)  self-attention probabilities  [B, H, L, L]
  k = 1  F.dropout (dropout1)                              self-attention output          [B, L, d]
  k = 2  F.scaled_dot_product_attention(..., dropout_p=p)  cross-attention probabilities [B, H, L, M]
  k = 3  F.dropout (dropout2)                              cross-attention output         [B, L, d]
  k = 4  F.dropout (the feed-forward's inner dropout)      relu(linear1(x))               [B, L, d_ffn]
  k = 5  F.dropout (dropout3)                              linear2 output                 [B, L, d]
The patches below replace those two functions for the duration of one step, consume the masks in call order and check each
call's site, shape and p; everything else is PyTorch's own layer code.  A mask is the scale tensor D (0 or 1 / (1 - p), built
as torch builds its dropout noise: keep.div_(1 - p)), applied as torch applies its noise: input * D."""
from __future__ import annotations

import contextlib
import math

import numpy as np
import torch
import torch.nn.functional as F

from oracle import student_oracle as st
from sampling_ref import philox4x32_10, uniform

TAG = 0x44524F50  # "DROP", the fourth counter word
SITES = ("sdpa", "dropout", "sdpa", "dropout", "dropout", "dropout")


def keep(seed, step, site, n, p):
    """bool[n]: element idx is kept iff uniform(word idx % 4 of Philox(counter (idx / 4, step, site, TAG), key = seed)) >= p,
    p compared as the fp32 value the library receives, in float64."""
    g = np.arange((n + 3) // 4, dtype=np.uint64)
    w = philox4x32_10(g, step & 0xFFFFFFFF, site, TAG, seed & 0xFFFFFFFF, seed >> 32)
    return uniform(np.stack(w, axis=1).reshape(-1)[:n]) >= float(np.float32(p))


def site_shapes(cfg: st.StudentConfig, B, L, M):
    """The six (kind, shape) per layer, in torch's call order."""
    d, H, f = cfg.d_model, cfg.n_head, cfg.d_ffn
    return [("sdpa", (B, H, L, L)), ("dropout", (B, L, d)), ("sdpa", (B, H, L, M)), ("dropout", (B, L, d)), ("dropout", (B, L, f)),
            ("dropout", (B, L, d))]


def scale_of(k: np.ndarray, p: float, shape) -> torch.Tensor:
    """Keep pattern -> torch's dropout noise: keep.div_(1 - p) in fp32."""
    return torch.from_numpy(k.reshape(shape)).to(torch.float32).div_(1 - p)


def masks(seed: int, step: int, cfg: st.StudentConfig, B: int, L: int, M: int, p=None):
    """[(kind, D)] for every layer's six sites in call order; D [shape] fp32, element index = the row-major index of the
    logical tensor (probabilities ((b H + h) L + i) n_keys + j, activations r * cols + c with r = b L + i)."""
    p = cfg.dropout if p is None else p
    out = []
    for layer in range(cfg.num_decoder_layers):
        for k, (kind, shape) in enumerate(site_shapes(cfg, B, L, M)):
            out.append((kind, scale_of(keep(seed, step, 6 * layer + k, math.prod(shape), p), p, shape)))
    return out


def ones_masks(cfg: st.StudentConfig, B, L, M):
    return [(kind, torch.ones(shape)) for _ in range(cfg.num_decoder_layers) for kind, shape in site_shapes(cfg, B, L, M)]


def attention(q, k, v, attn_mask, D, variant=None):
    """torch's math attention (scaled_dot_product_attention's reference form) with the mask D applied to the probabilities.
    variant 'before_norm': D applied to the unnormalised exponentials (renormalised over the kept keys); 'dv_uses_p': the
    forward is the same but dV = P^T dO (the undropped probabilities) in the backward pass."""
    s = (q @ k.transpose(-2, -1)) * (1.0 / math.sqrt(q.shape[-1]))
    if attn_mask is not None:
        s = s.masked_fill(~attn_mask, float("-inf")) if attn_mask.dtype == torch.bool else s + attn_mask
    if variant == "before_norm":
        e = torch.exp(s - s.amax(-1, keepdim=True)) * D
        return (e / e.sum(-1, keepdim=True).clamp_min(1e-30)) @ v
    P = torch.softmax(s, dim=-1)
    if variant == "dv_uses_p":
        return (P * D) @ v.detach() + P.detach() @ v - (P.detach() @ v).detach()
    return (P * D) @ v


@contextlib.contextmanager
def injected(m_masks, p, variant=None, calls=None):
    """Replace F.dropout / F.scaled_dot_product_attention: each call takes the next mask, whose kind and shape must match, and
    asserts torch asked for dropout with probability p.  variant 'no_scale' applies the keep pattern without 1 / (1 - p)."""
    it = iter(m_masks)
    orig_do, orig_sdpa = F.dropout, F.scaled_dot_product_attention

    def take(kind, shape, got_p):
        want_kind, D = next(it)
        assert want_kind == kind and tuple(D.shape) == tuple(shape), (kind, tuple(shape), want_kind, tuple(D.shape))
        assert got_p == p, (kind, got_p, p)
        if calls is not None:
            calls.append((kind, tuple(shape)))
        if variant == "no_scale":
            D = (D != 0).to(D.dtype)
        return D

    def dropout(x, p=0.5, training=True, inplace=False):
        assert training and not inplace
        return x * take("dropout", x.shape, p)

    def sdpa(q, k, v, attn_mask=None, dropout_p=0.0, is_causal=False, **kw):
        assert not is_causal and not kw.get("enable_gqa", False)
        D = take("sdpa", (*q.shape[:-1], k.shape[-2]), dropout_p)
        return attention(q, k, v, attn_mask, D, variant if variant in ("before_norm", "dv_uses_p") else None)

    F.dropout, F.scaled_dot_product_attention = dropout, sdpa
    try:
        yield
    finally:
        F.dropout, F.scaled_dot_product_attention = orig_do, orig_sdpa
    assert next(it, None) is None, "fewer dropout calls than masks"


def stock_step_with_masks(m: st.StudentDecoderOracle, y, memory, teacher, temperature, m_masks, variant=None, calls=None):
    """student_oracle.distillation_step with the stock modules in train() (p = cfg.dropout) and the masks injected.
    variant: None, 'no_scale', 'before_norm', 'dv_uses_p' (see attention / injected) or 'dropout3_after_add', which applies
    site 5's mask to x + linear2(...) instead of linear2(...) alone."""
    p = m.cfg.dropout
    layers = list(m.decoder.layers)
    if variant == "dropout3_after_add":
        for layer in layers:
            def ff_block(x, layer=layer):
                z = layer.linear2(layer.dropout(layer.activation(layer.linear1(x))))
                return layer.dropout3(x + z) - x   # the layer adds x back: norm3(D o (x + z))
            layer._ff_block = ff_block
    m.train()
    try:
        with injected(m_masks, p, variant, calls):
            out = st.distillation_step(m, y, memory, teacher, temperature)
    finally:
        m.eval()
        for layer in layers:
            layer.__dict__.pop("_ff_block", None)
    return out
