"""Dropout in the student's distillation step, host side: the restated Philox masks (tests/student_dropout_ref.py) and the
injection of those masks into the stock torch modules, which the GPU tests (test_gpu_student_dropout.py) use as their oracle."""
import importlib
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import student_dropout_ref as dr
from oracle import student_oracle as st

g = importlib.import_module("real-time-video-captioning_b200")


def _small_cfg():
    return st.StudentConfig(d_model=64, n_head=4, d_ffn=128, num_decoder_layers=2, vocab_length=50, cls_token_id=1, sep_token_id=2)


def _inputs(cfg, B, L, M, seed):
    gen = torch.Generator().manual_seed(seed)
    y = torch.randint(3, cfg.vocab_length, (B, L), generator=gen)
    y[:, 0] = cfg.cls_token_id
    y[0, L - 2:] = 0
    return y, torch.randn(B, M, cfg.d_model, generator=gen), torch.randn(B, L, cfg.vocab_length, generator=gen) * 1.5


def test_keep_rate_and_independence_of_the_mask():
    n, p = 1 << 20, 0.3
    k = dr.keep(12345, 0, 0, n, p)
    sigma = math.sqrt(p * (1 - p) / n)
    assert abs(k.mean() - (1 - p)) < 5 * sigma, k.mean()
    for other in (dr.keep(12345, 0, 1, n, p), dr.keep(12345, 1, 0, n, p), dr.keep(12346, 0, 0, n, p), dr.keep(12345 + (1 << 32), 0, 0, n, p)):
        assert abs((k == other).mean() - (p * p + (1 - p) ** 2)) < 5 * math.sqrt(0.5 / n)   # independent patterns agree at p^2 + (1-p)^2
    assert not dr.keep(7, 3, 2, 4096, 0.0).__invert__().any()   # p = 0 keeps everything
    # the four words of one Philox call serve four consecutive elements: element 4 g + w is word w of counter g
    w = dr.philox4x32_10(np.arange(3, dtype=np.uint64), 5, 9, dr.TAG, 77, 0)
    u = dr.uniform(np.stack(w, axis=1).reshape(-1))
    assert np.array_equal(dr.keep(77, 5, 9, 12, 0.45), u >= float(np.float32(0.45)))


def test_masks_follow_the_site_layout():
    cfg = _small_cfg()
    B, L, M = 3, 5, 2
    ms = dr.masks(9, 4, cfg, B, L, M)
    assert [k for k, _ in ms] == list(dr.SITES) * cfg.num_decoder_layers
    assert [tuple(D.shape) for _, D in ms[:6]] == [(B, 4, L, L), (B, L, 64), (B, 4, L, M), (B, L, 64), (B, L, 128), (B, L, 64)]
    scale = torch.tensor(1.0).div_(1 - cfg.dropout)
    for layer in range(2):
        for k in range(6):
            D = ms[6 * layer + k][1]
            assert set(D.unique().tolist()) <= {0.0, scale.item()}
            flat = dr.keep(9, 4, 6 * layer + k, D.numel(), cfg.dropout)
            assert torch.equal(D.reshape(-1) != 0, torch.from_numpy(flat))


def test_stock_step_with_all_ones_masks_is_the_step_without_dropout():
    cfg = _small_cfg()
    m = st.init_student(cfg, seed=3)
    y, mem, teacher = _inputs(cfg, 3, 6, 2, seed=4)
    info, grads, dmem = st.distillation_step(m, y, mem, teacher, 1.5)
    calls = []
    info2, grads2, dmem2 = dr.stock_step_with_masks(m, y, mem, teacher, 1.5, dr.ones_masks(cfg, 3, 6, 2), calls=calls)
    assert not m.training
    for k in ("loss", "kl", "ce"):
        assert abs(info2[k] - info[k]) <= 1e-6 * abs(info[k]), k
    assert set(grads2) == set(grads)
    for k, ref in grads.items():
        assert (grads2[k] - ref).norm() <= 1e-6 * ref.norm() + 1e-12, k
    assert (dmem2 - dmem).norm() <= 1e-6 * dmem.norm()
    # exactly six calls per layer, in nn.TransformerDecoderLayer's order
    assert calls == [(k, s) for _ in range(2) for k, s in dr.site_shapes(cfg, 3, 6, 2)]


def test_masks_change_the_step_and_are_consumed_in_full():
    cfg = _small_cfg()
    m = st.init_student(cfg, seed=3)
    y, mem, teacher = _inputs(cfg, 2, 5, 3, seed=5)
    ones, _, _ = dr.stock_step_with_masks(m, y, mem, teacher, 1.0, dr.ones_masks(cfg, 2, 5, 3))
    a, ga, _ = dr.stock_step_with_masks(m, y, mem, teacher, 1.0, dr.masks(1, 0, cfg, 2, 5, 3))
    b, gb, _ = dr.stock_step_with_masks(m, y, mem, teacher, 1.0, dr.masks(1, 0, cfg, 2, 5, 3))
    assert a["loss"] == b["loss"] and all(torch.equal(ga[k], gb[k]) for k in ga)
    assert a["loss"] != ones["loss"]
    with pytest.raises(AssertionError):   # one mask too many: a layer's six calls did not all happen
        dr.stock_step_with_masks(m, y, mem, teacher, 1.0, dr.masks(1, 0, cfg, 2, 5, 3) + [("dropout", torch.ones(1))])
    with pytest.raises(AssertionError):   # a mask of the wrong shape at a site
        ms = dr.masks(1, 0, cfg, 2, 5, 3)
        ms[2], ms[3] = ms[3], ms[2]
        dr.stock_step_with_masks(m, y, mem, teacher, 1.0, ms)


def test_patch_applies_torch_own_dropout_arithmetic():
    """torch's train-mode F.dropout returns 0 or input / (1 - p); the injected call returns input * D with D built from the
    same keep pattern the way torch builds its noise, bit for bit."""
    torch.manual_seed(0)
    p = 0.3
    x = torch.randn(4, 7, 33) + 0.01
    out = F.dropout(x, p, training=True)
    kept = out != 0
    D = kept.to(torch.float32).div_(1 - p)
    with dr.injected([("dropout", D)], p):
        got = F.dropout(x, p, training=True)
    assert torch.equal(got, out)
    assert torch.allclose(out[kept], x[kept] / (1 - p), rtol=1e-6, atol=0)


@pytest.mark.parametrize("mask_kind", ["bool", "float"])
def test_patched_attention_with_ones_is_torch_attention(mask_kind):
    gen = torch.Generator().manual_seed(1)
    q, k, v = torch.randn(2, 3, 5, 8, generator=gen), torch.randn(2, 3, 6, 8, generator=gen), torch.randn(2, 3, 6, 8, generator=gen)
    allowed = torch.rand(2, 3, 5, 6, generator=gen) > 0.3
    allowed[..., 0] = True
    mask = allowed if mask_kind == "bool" else torch.zeros(2, 3, 5, 6).masked_fill(~allowed, float("-inf"))
    ref = F.scaled_dot_product_attention(q, k, v, attn_mask=mask, dropout_p=0.0)
    orig = F.scaled_dot_product_attention
    with dr.injected([("sdpa", torch.ones(2, 3, 5, 6))], 0.3):
        got = F.scaled_dot_product_attention(q, k, v, attn_mask=mask, dropout_p=0.3)
    assert torch.allclose(got, ref, atol=1e-6, rtol=1e-5)
    assert F.scaled_dot_product_attention is orig   # restored


def test_python_rejects_p_outside_the_unit_interval():
    for p in (1.0, -0.1, 1.5, float("nan")):
        s = g.StudentCandidateV1(None, 64, 4, 128, p, 2, 50, 1, 2)
        with pytest.raises(ValueError, match="outside"):
            s.enable_training(dropout_seed=1)
        s.enable_training()   # no seed: p is never used
    s = g.StudentCandidateV1(None, 64, 4, 128, 0.3, 2, 50, 1, 2)
    with pytest.raises(ValueError):
        s.enable_training(dropout_seed=-1)
    with pytest.raises(RuntimeError, match="dropout is off"):
        s.dropout_step = 3
    s.enable_training(dropout_seed=5)
    assert s.dropout_step == 0
    s.dropout_step = 3
    assert s.dropout_step == 3
    with pytest.raises(ValueError):
        s.dropout_step = -1
