"""Dropout in the student's distillation step on the GPU (csrc/student_train.cu, opt-in through
enable_training(dropout_seed=...)).

Oracle: torch.autograd on the stock nn.TransformerDecoderLayer modules in train() with the library's Philox masks injected at
torch's own dropout call sites (tests/student_dropout_ref.py).  Bounds are those of the step without dropout
(test_student.py::test_distillation_step_gradients_match_autograd); negative controls with one plausible mistake each must
fail them.  The operator tests check each new kernel against float64 on its own operands with the bounds of
test_gpu_student_ops.py, and the mask bit for bit against the numpy restatement."""
import ctypes
import importlib
import math
import os
from ctypes import c_float, c_int, c_longlong, c_uint64, c_void_p as V

import pytest
import torch

import op_modes_shim
import student_dropout_ref as dr
from oracle import student_oracle as st
from test_gpu_gemm_shapes import _check_bound, _control_bound
from test_gpu_parity import record
from test_gpu_student_ops import (BF, SAFE, SENT, SENT32, U, Student, _bf, _gen, _ln_rows, _p, _self_allowed, _stream, _tokens, attn_ref,
                                  fwd_bound, ln_stats)

pytestmark = pytest.mark.gpu

g = importlib.import_module("real-time-video-captioning_b200")
SEED = 0x1234_5678_9ABC
P = 0.3


def _gpu_student(cfg, seed):
    m = st.init_student(cfg, seed=seed)
    s = g.StudentCandidateV1(None, cfg.d_model, cfg.n_head, cfg.d_ffn, cfg.dropout, cfg.num_decoder_layers, cfg.vocab_length,
                             cfg.cls_token_id, cfg.sep_token_id)
    s.load_state_dict(st.state_dict_of(m))
    return m, s.to("cuda")


def _train_inputs(cfg, B, L, F, seed):
    gen = torch.Generator().manual_seed(seed)
    y = torch.randint(1000, cfg.vocab_length, (B, L), generator=gen)
    y[:, 0] = cfg.cls_token_id
    if L > 4:   # padded tails
        y[0, L - 3:] = 0
        y[B - 1, L - 1:] = 0
    mem = torch.randn(B, F, cfg.d_model, generator=gen)
    teacher = torch.randn(B, L, cfg.vocab_length, generator=gen) * 1.5
    return y, mem, teacher


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def _step(s, y, mem, teacher, T):
    out = s.distillation_step(y, mem, teacher, temperature=T, apply=False, want_memory_grad=True)
    torch.cuda.synchronize()
    return ({k: out[k].item() for k in ("loss", "kl", "ce")}, {k: v.cpu() for k, v in s.gradients().items()}, out["d_memory"].cpu())


def _violations(got, ref):
    """The bounds of the step without dropout: KL / CE 2 %, all gradients 3e-2 and each 8e-2 relative Frobenius, d memory 6e-2."""
    (info, grads, dmem), (rinfo, rgrads, rdmem) = got, ref
    bad, num, den, per = [], 0.0, 0.0, {}
    for k in ("kl", "ce"):
        if not abs(info[k] - rinfo[k]) < 2e-2 * abs(rinfo[k]):
            bad.append((k, info[k], rinfo[k]))
    for k, r in rgrads.items():
        per[k] = _rel(grads[k], r)
        num += (grads[k].double() - r.double()).pow(2).sum().item()
        den += r.double().pow(2).sum().item()
        if not per[k] < 8e-2:
            bad.append((k, per[k]))
    total, e_mem = (num / den) ** 0.5, _rel(dmem, rdmem)
    if not total < 3e-2:
        bad.append(("all", total))
    if not e_mem < 6e-2:
        bad.append(("d_memory", e_mem))
    return bad, total, e_mem, per


# ---------------------------------------------------------------------------------------------------------- parity
@pytest.mark.parametrize("B,L,F,T", [(8, 20, 6, 1.0), (3, 7, 2, 2.0)])
def test_dropout_step_matches_autograd_with_the_same_masks(B, L, F, T):
    cfg = st.StudentConfig()
    m, s = _gpu_student(cfg, seed=31)
    y, mem, teacher = _train_inputs(cfg, B, L, F, seed=B * 10 + L)
    s.enable_training(lr=1e-4, dropout_seed=SEED)
    s.dropout_step = 5
    got = _step(s, y, mem, teacher, T)
    assert s.dropout_step == 6
    assert abs(got[0]["loss"] - (got[0]["kl"] + got[0]["ce"])) < 1e-5 * abs(got[0]["loss"])
    masks = dr.masks(SEED, 5, cfg, B, L, F)
    ref = dr.stock_step_with_masks(m, y, mem, teacher, T, masks)
    bad, total, e_mem, per = _violations(got, ref)
    worst = max(per.items(), key=lambda kv: kv[1])
    record("distillation_dropout_step_grads", B=B, L=L, temperature=T, p=P, loss=got[0]["loss"], ref_loss=ref[0]["loss"],
           all_params_rel_fro=total, worst_tensor=worst[0], worst_rel_fro=worst[1], d_memory_rel_fro=e_mem, per_tensor_rel_fro=per)
    assert not bad, bad
    unused = torch.ones(cfg.vocab_length, dtype=torch.bool)
    unused[y.flatten()] = False
    assert (got[1]["embed.weight"][unused] == 0).all()
    if (B, L) != (8, 20):
        return
    # negative controls: each plausible mistake must fail the bounds
    shifted = list(masks)
    kind, D = shifted[7]   # layer 1, dropout1
    shifted[7] = (kind, D.reshape(-1).roll(1).reshape(D.shape))
    controls = {
        "one site's mask shifted by one element": dict(m_masks=shifted),
        "step off by one": dict(m_masks=dr.masks(SEED, 6, cfg, B, L, F)),
        "no 1 / (1 - p) scale": dict(m_masks=masks, variant="no_scale"),
        "attention dropout before the softmax normalisation": dict(m_masks=masks, variant="before_norm"),
        "dropout3 after the residual add": dict(m_masks=masks, variant="dropout3_after_add"),
        "dV from P instead of D o P": dict(m_masks=masks, variant="dv_uses_p"),
    }
    for what, kw in controls.items():
        wrong = dr.stock_step_with_masks(m, y, mem, teacher, T, **kw)
        cbad = _violations(got, wrong)[0]
        record("distillation_dropout_control", control=what, violations=str(cbad[:4]))
        assert cbad, f"negative control passed: the bounds cannot see {what}"


# ---------------------------------------------------------------------------------------------------------- bit identity
def _bits_equal(a, b):
    return a[0] == b[0] and all(torch.equal(a[1][k], b[1][k]) for k in a[1]) and torch.equal(a[2], b[2])


def test_dropout_is_bit_identical_off_replayable_and_seeded():
    cfg = st.StudentConfig()
    y, mem, teacher = _train_inputs(cfg, 8, 20, 6, seed=77)
    _, plain = _gpu_student(cfg, seed=32)
    plain.enable_training()
    base = _step(plain, y, mem, teacher, 1.0)
    _, zero = _gpu_student(cfg, seed=32)
    zero.dropout = 0.0
    zero.enable_training(dropout_seed=SEED)
    assert _bits_equal(_step(zero, y, mem, teacher, 1.0), base), "seed with p = 0 differs from the step without dropout"
    _, s = _gpu_student(cfg, seed=32)
    s.enable_training(dropout_seed=SEED)
    s0 = _step(s, y, mem, teacher, 1.0)
    s1 = _step(s, y, mem, teacher, 1.0)
    assert s.dropout_step == 2
    assert not _bits_equal(s0, s1) and not _bits_equal(s0, base)
    s.dropout_step -= 1
    assert _bits_equal(_step(s, y, mem, teacher, 1.0), s1), "dropout_step set back by one does not replay the step"
    s.dropout_step = 0
    assert _bits_equal(_step(s, y, mem, teacher, 1.0), s0)
    _, again = _gpu_student(cfg, seed=32)
    again.enable_training(dropout_seed=SEED)
    assert _bits_equal(_step(again, y, mem, teacher, 1.0), s0), "same (seed, step) not run-to-run identical"
    _, other = _gpu_student(cfg, seed=32)
    other.enable_training(dropout_seed=SEED + 1)
    assert not _bits_equal(_step(other, y, mem, teacher, 1.0), s0)
    # the step survives an engine rebuild (e.g. a move between devices or a reload of the weights)
    s.dropout_step = 1
    s._stale = True
    assert _bits_equal(_step(s, y, mem, teacher, 1.0), s1) and s.dropout_step == 2


def test_inference_is_untouched_by_a_dropout_step():
    cfg = st.StudentConfig()
    y, mem, teacher = _train_inputs(cfg, 4, 12, 6, seed=78)
    outs = []
    for seed in (None, SEED):
        _, s = _gpu_student(cfg, seed=33)
        s.enable_training(dropout_seed=seed)
        _step(s, y, mem, teacher, 1.0)
        outs.append((s.forward_decoder(y, mem).cpu(), s.greedy_decode_from_memory(mem, 8).cpu()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


def test_set_dropout_rejects_p_outside_the_unit_interval():
    cfg = st.StudentConfig(num_decoder_layers=1)
    _, s = _gpu_student(cfg, seed=34)
    s.enable_training(dropout_seed=SEED)
    h, lib = s._engine(), s._lib
    s.dropout_step = 4
    for p in (1.0, -0.25, 1.5, float("nan"), float("inf")):
        assert lib.gitb200_student_train_set_dropout(h, ctypes.c_float(p), 9, 0) == -1   # GITB200_ERR_INVALID
    assert lib.gitb200_student_train_set_dropout(h, ctypes.c_float(0.2), 9, -1) == -1
    pv, sv, stv = ctypes.c_float(), ctypes.c_uint64(), ctypes.c_longlong()
    assert lib.gitb200_student_train_get_dropout(h, ctypes.byref(pv), ctypes.byref(sv), ctypes.byref(stv)) == 0
    assert (abs(pv.value - P) < 1e-7, sv.value, stv.value) == (True, SEED, 4), "a rejected call changed the state"
    s.dropout = 1.0
    with pytest.raises(ValueError):
        s.enable_training(dropout_seed=SEED)


# ---------------------------------------------------------------------------------------------------------- training runs
def test_adam_with_dropout_lowers_the_loss():
    cfg = st.StudentConfig()
    _, s = _gpu_student(cfg, seed=35)
    y, mem, teacher = _train_inputs(cfg, 8, 20, 6, seed=5)
    s.enable_training(lr=1e-4, dropout_seed=SEED)
    losses = [s.distillation_step(y, mem, teacher)["loss"].item() for _ in range(13)]
    record("distillation_dropout_adam", losses=losses)
    assert all(math.isfinite(v) for v in losses)
    assert sum(losses[-3:]) / 3 < losses[0] - 0.05, losses
    assert s.dropout_step == 13


def test_distillation_trainer_with_dropout_and_the_git_teacher():
    teacher = g.GenerativeImageTextTeacher.from_random_init({"num_image_with_embedding": 2})
    cfg = st.StudentConfig()
    m, s = _gpu_student(cfg, seed=36)
    trainer = g.DistillationTrainer(teacher, s, lr=1e-4, dropout_seed=SEED + 3)
    gen = torch.Generator().manual_seed(3)
    x = torch.randn(2, 2, 3, 224, 224, generator=gen)
    y = torch.randint(1000, 30000, (2, 6), generator=gen)
    y[:, 0] = 101
    mem = torch.randn(2, 2, cfg.d_model, generator=gen)
    t_logits = trainer.teacher_logits(x, y)
    info, _, _ = dr.stock_step_with_masks(m, y, mem, t_logits.cpu().float(), 1.0, dr.masks(SEED + 3, 0, cfg, 2, 6, 2))
    loss = trainer.training_step({"frames": x, "caption": y, "memory": mem})
    assert torch.isfinite(loss) and abs(loss.item() - info["loss"]) < 2e-2 * abs(info["loss"]), (loss.item(), info["loss"])
    assert s.dropout_step == 1 and trainer.last["d_memory"].shape == mem.shape


# ---------------------------------------------------------------------------------------------------------- operators
@pytest.fixture(scope="module")
def lib():
    import gitb200  # noqa: F401  (loads libgitb200.so before the shim that links against it)
    importlib.import_module("real-time-video-captioning_b200._lib").load()
    return op_modes_shim.load(os.path.join(op_modes_shim.ROOT, "tests", "cuda", "student_dropout_ops.cpp"), op_modes_shim.STUDENT_HEADERS,
                              SIGNATURES)


_D = [c_uint64, c_longlong, c_int, c_float]
SIGNATURES = {
    "sdo_attn": (c_int, [V, V, c_int, c_int, V, c_int, c_int, c_int, c_int, c_int, c_int, V, c_int, c_int, V, c_int, *_D, V]),
    "sdo_attn_bwd": (c_int, [V, V, c_int, c_int, V, c_int, c_int, c_int, c_int, c_int, c_int, V, c_int, c_int, V, V, c_int, V, c_int, c_int,
                             c_int, *_D, V]),
    "sdo_add_ln": (c_int, [V, V, V, c_int, V, V, V, V, *_D, V]),
    "sdo_inplace": (c_int, [V, V, c_int, c_int, c_int, *_D, V]),
    "sdo_ln_bwd": (c_int, [V, V, V, c_int, V, V, V, V, V, V, *_D, V]),
    "sdo_relu_bwd": (c_int, [V, V, V, c_longlong, c_float, V]),
}

_students = {}


@pytest.fixture(scope="module")
def students(lib):
    yield lambda name: _students.setdefault(name, Student(name))
    for s in _students.values():
        s.m.close()
    _students.clear()


def _mask(seed, step, site, shape, p=P):
    """D (0 or 1 / (1 - p) in fp32) as float64 on the device, element index = row-major index of `shape`."""
    return dr.scale_of(dr.keep(seed, step, site, math.prod(shape), p), p, shape).double().cuda()


def _drop_attn_ref(Q, K, Vv, allowed, D, before_norm=False):
    """(D o P) V and its bound: the error of D P is D dP plus one rounding of the product."""
    P_, out, dP = attn_ref(Q, K, Vv, allowed)
    if before_norm:
        e = P_ * D
        PD = e / e.sum(-1, keepdim=True).clamp_min(1e-300)
    else:
        PD = P_ * D
    ref = torch.einsum("bhij,bjhc->bihc", PD, Vv)
    return ref, fwd_bound(PD, dP * D + U * PD, Vv, ref)


@pytest.mark.parametrize("cfg", ["prod", "small", "hd128"])
@pytest.mark.parametrize("B,L,M", [(8, 20, 6), (3, 7, 2), (3, 64, 64)])
def test_attention_forward_with_dropout(lib, students, cfg, B, L, M):
    """Self-attention (causal + padding mask, training layout) and cross-attention with dropout on the probabilities.
    Controls: dropout before the softmax normalisation; the mask of another site."""
    s = students(cfg)
    gen = _gen(700 + L)
    H, hd, dp, d = s.H, s.hd, s.dp, s.d
    qkv = torch.zeros(B * L, 3 * dp, device="cuda", dtype=torch.bfloat16)
    for t in range(3):
        qkv[:, t * dp:t * dp + d] = _bf((B * L, d), gen, 1.5 if t == 0 else 1.0)
    tok = _tokens(B, L, s.V, gen, [(0, L - 1), (B - 1, L // 2)])
    out = torch.full((B * L, dp), SENT, device="cuda", dtype=torch.bfloat16)
    assert lib.sdo_attn(s.h, _p(qkv), 3 * dp, L, _p(qkv), L, 3 * dp, dp, 2 * dp, L, 1, _p(tok), L, B * L, _p(out), dp, SEED, 3, 6, P,
                        _stream()) == 0
    q2 = torch.zeros(B * L, dp, device="cuda", dtype=torch.bfloat16)
    q2[:, :d] = _bf((B * L, d), gen, 1.5)
    kv = torch.zeros(B * M, 2 * dp, device="cuda", dtype=torch.bfloat16)
    kv[:, :d] = _bf((B * M, d), gen)
    kv[:, dp:dp + d] = _bf((B * M, d), gen)
    out2 = torch.full((B * L, dp), SENT, device="cuda", dtype=torch.bfloat16)
    assert lib.sdo_attn(s.h, _p(q2), dp, L, _p(kv), M, 2 * dp, 0, dp, M, 0, None, 0, B * L, _p(out2), dp, SEED, 3, 8, P, _stream()) == 0
    torch.cuda.synchronize()
    meta = dict(cfg=cfg, B=B, L=L, M=M)
    view = qkv.double().view(B, L, 3, dp)[..., :d].reshape(B, L, 3, H, hd)
    allowed = _self_allowed(tok, L, 0, L)
    D = _mask(SEED, 3, 6, (B, H, L, L))
    ref, bound = _drop_attn_ref(view[:, :, 0], view[:, :, 1], view[:, :, 2], allowed, D)
    _check_bound("student_dropout_attn_self", out[:, :d], ref.reshape(B * L, d), bound.reshape(B * L, d), **meta)
    assert (out[:, d:] == SENT).all()
    wrong, _ = _drop_attn_ref(view[:, :, 0], view[:, :, 1], view[:, :, 2], allowed, D, before_norm=True)
    _control_bound(out[:, :d], wrong.reshape(B * L, d), bound.reshape(B * L, d), "dropout before the softmax normalisation")
    wrong, _ = _drop_attn_ref(view[:, :, 0], view[:, :, 1], view[:, :, 2], allowed, _mask(SEED, 3, 7, (B, H, L, L)))
    _control_bound(out[:, :d], wrong.reshape(B * L, d), bound.reshape(B * L, d), "the mask of another site")
    Q2 = q2.double()[:, :d].reshape(B, L, H, hd)
    K2, V2 = kv.double()[:, :d].reshape(B, M, H, hd), kv.double()[:, dp:dp + d].reshape(B, M, H, hd)
    D2 = _mask(SEED, 3, 8, (B, H, L, M))
    ones = torch.ones(B, L, M, dtype=torch.bool, device="cuda")
    ref2, bound2 = _drop_attn_ref(Q2, K2, V2, ones, D2)
    _check_bound("student_dropout_attn_cross", out2[:, :d], ref2.reshape(B * L, d), bound2.reshape(B * L, d), **meta)
    wrong2, _ = _drop_attn_ref(Q2, K2, V2, ones, torch.ones_like(D2))
    _control_bound(out2[:, :d], wrong2.reshape(B * L, d), bound2.reshape(B * L, d), "no dropout")


def _drop_attn_bwd_ref(Q, K, Vv, dO, allowed, D, dv_from_p=False):
    """test_gpu_student_ops.attn_bwd_ref for out = (D o P) V: dP = D o (dO V^T), dS = P (dP - rowsum(P dP)), dV = (D o P)^T dO."""
    hd, Lq, nk = Q.shape[-1], Q.shape[1], K.shape[1]
    scale = 1 / math.sqrt(hd)
    P_, _, dPe = attn_ref(Q, K, Vv, allowed)
    Pg = D * torch.einsum("bihc,bjhc->bhij", dO, Vv)
    dPg = D * hd * U * torch.einsum("bihc,bjhc->bhij", dO.abs(), Vv.abs()) + U * Pg.abs()
    dsum = (P_ * Pg).sum(-1, keepdim=True)
    ddsum = (dPe * Pg.abs() + P_ * dPg).sum(-1, keepdim=True) + nk * U * (P_ * Pg.abs()).sum(-1, keepdim=True)
    dS = P_ * (Pg - dsum)
    ddS = dPe * (Pg - dsum).abs() + P_ * (dPg + ddsum + U * (Pg.abs() + dsum.abs())) + U * dS.abs()
    dQ = scale * torch.einsum("bhij,bjhc->bihc", dS, K)
    eQ = scale * (torch.einsum("bhij,bjhc->bihc", ddS, K.abs()) + (nk + 3) * U * torch.einsum("bhij,bjhc->bihc", dS.abs(), K.abs()))
    dK = scale * torch.einsum("bhij,bihc->bjhc", dS, Q)
    eK = scale * (torch.einsum("bhij,bihc->bjhc", ddS, Q.abs()) + (Lq + 3) * U * torch.einsum("bhij,bihc->bjhc", dS.abs(), Q.abs()))
    PD = P_ if dv_from_p else P_ * D
    dV = torch.einsum("bhij,bihc->bjhc", PD, dO)
    eV = torch.einsum("bhij,bihc->bjhc", dPe * D + U * P_ * D, dO.abs()) + (Lq + 1) * U * torch.einsum("bhij,bihc->bjhc", P_ * D, dO.abs())
    return [(dQ, BF * dQ.abs() + SAFE * eQ), (dK, BF * dK.abs() + SAFE * eK), (dV, BF * dV.abs() + SAFE * eV)]


@pytest.mark.parametrize("cfg", ["prod", "small", "hd128"])
@pytest.mark.parametrize("B,L,M", [(8, 20, 6), (3, 7, 2), (3, 64, 64)])
def test_attention_backward_with_dropout(lib, students, cfg, B, L, M):
    """attn_bwd_kernel<true> as the step runs it (self with causal + padding mask into dqkv in place; cross into [B M, 2 dp]).
    Masked keys get exactly zero dK / dV.  Controls: dV from P instead of D o P; dP without the mask."""
    s = students(cfg)
    gen = _gen(B * 1000 + L * 10 + M + 7)
    H, hd, dp, d = s.H, s.hd, s.dp, s.d
    R, Rm = B * L, B * M
    tok = _tokens(B, L, s.V, gen, [(0, L - 1)] + ([(B - 1, L // 2), (0, L - 2)] if L > 3 else []))
    qkv = torch.zeros(R, 3 * dp, device="cuda", dtype=torch.bfloat16)
    for t in range(3):
        qkv[:, t * dp:t * dp + d] = _bf((R, d), gen, 1.5 if t == 0 else 1.0)
    dO = torch.zeros(R, dp, device="cuda", dtype=torch.bfloat16)
    dO[:, :d] = _bf((R, d), gen)
    dqkv = torch.full((R, 3 * dp), SENT, device="cuda", dtype=torch.bfloat16)
    assert lib.sdo_attn_bwd(s.h, _p(qkv), 3 * dp, L, _p(qkv), L, 3 * dp, dp, 2 * dp, L, 1, _p(tok), L, B, _p(dO), _p(dqkv), 3 * dp, _p(dqkv),
                            3 * dp, dp, 2 * dp, SEED, 11, 0, P, _stream()) == 0
    q2 = torch.zeros(R, dp, device="cuda", dtype=torch.bfloat16)
    q2[:, :d] = _bf((R, d), gen, 1.5)
    kv = torch.zeros(Rm, 2 * dp, device="cuda", dtype=torch.bfloat16)
    kv[:, :d] = _bf((Rm, d), gen)
    kv[:, dp:dp + d] = _bf((Rm, d), gen)
    dq2 = torch.full((R, dp), SENT, device="cuda", dtype=torch.bfloat16)
    dkv = torch.full((Rm, 2 * dp), SENT, device="cuda", dtype=torch.bfloat16)
    assert lib.sdo_attn_bwd(s.h, _p(q2), dp, L, _p(kv), M, 2 * dp, 0, dp, M, 0, None, 0, B, _p(dO), _p(dq2), dp, _p(dkv), 2 * dp, 0, dp,
                            SEED, 11, 2, P, _stream()) == 0
    torch.cuda.synchronize()
    meta = dict(cfg=cfg, B=B, L=L, M=M)
    v = qkv.double().view(B, L, 3, dp)[..., :d].reshape(B, L, 3, H, hd)
    G = dO.double()[:, :d].reshape(B, L, H, hd)
    got = dqkv.view(B, L, 3, dp)
    D = _mask(SEED, 11, 0, (B, H, L, L))
    allowed = _self_allowed(tok, L, 0, L)
    res = _drop_attn_bwd_ref(v[:, :, 0], v[:, :, 1], v[:, :, 2], G, allowed, D)
    for t, (name, (ref, bound)) in enumerate(zip(("dq", "dk", "dv"), res)):
        _check_bound(f"student_dropout_attn_bwd_self_{name}", got[:, :, t, :d], ref.reshape(B, L, d), bound.reshape(B, L, d), **meta)
    assert (got[..., d:] == SENT).all()
    assert (got[:, :, 1:, :d][tok == 0] == 0).all(), "padded keys received gradient"
    wrong = _drop_attn_bwd_ref(v[:, :, 0], v[:, :, 1], v[:, :, 2], G, allowed, D, dv_from_p=True)[2][0]
    _control_bound(got[:, :, 2, :d], wrong.reshape(B, L, d), res[2][1].reshape(B, L, d), "dV from P instead of D o P")
    wrong = _drop_attn_bwd_ref(v[:, :, 0], v[:, :, 1], v[:, :, 2], G, allowed, torch.ones_like(D))[0][0]
    _control_bound(got[:, :, 0, :d], wrong.reshape(B, L, d), res[0][1].reshape(B, L, d), "dP without the mask")
    Q2 = q2.double()[:, :d].reshape(B, L, H, hd)
    K2, V2 = kv.double()[:, :d].reshape(B, M, H, hd), kv.double()[:, dp:dp + d].reshape(B, M, H, hd)
    D2 = _mask(SEED, 11, 2, (B, H, L, M))
    (rq, bq), (rk, bk), (rv, bv) = _drop_attn_bwd_ref(Q2, K2, V2, G, torch.ones(B, L, M, dtype=torch.bool, device="cuda"), D2)
    _check_bound("student_dropout_attn_bwd_cross_dq", dq2[:, :d], rq.reshape(R, d), bq.reshape(R, d), **meta)
    _check_bound("student_dropout_attn_bwd_cross_dk", dkv[:, :d], rk.reshape(Rm, d), bk.reshape(Rm, d), **meta)
    _check_bound("student_dropout_attn_bwd_cross_dv", dkv[:, dp:dp + d], rv.reshape(Rm, d), bv.reshape(Rm, d), **meta)


@pytest.mark.parametrize("cfg", ["prod", "small", "hd128"])
@pytest.mark.parametrize("rows", [21, 160])
def test_dropout_add_layernorm(lib, students, cfg, rows):
    """y = bf16(x + D z) (one fp32 product and sum), out = LN(y) gamma + beta with the bound of test_layernorm on the stored y.
    Controls: the mask applied after the add; no 1 / (1 - p) scale."""
    s = students(cfg)
    gen = _gen(800 + rows)
    d, dp = s.d, s.dp
    x = torch.full((rows, dp), SENT, device="cuda", dtype=torch.bfloat16)
    x[:, :d] = _ln_rows(rows, d, gen)
    z = torch.full((rows, dp), SENT, device="cuda", dtype=torch.bfloat16)
    z[:, :d] = _bf((rows, d), gen, 3.0)
    gamma = torch.randn(d, device="cuda", generator=gen) * 0.5 + 1
    beta = torch.randn(d, device="cuda", generator=gen) * 0.3
    y = torch.full((rows, dp), SENT, device="cuda", dtype=torch.bfloat16)
    out = torch.full((rows, dp), SENT, device="cuda", dtype=torch.bfloat16)
    assert lib.sdo_add_ln(s.h, _p(x), _p(z), rows, _p(gamma), _p(beta), _p(y), _p(out), SEED, 2, 5, P, _stream()) == 0
    torch.cuda.synchronize()
    D = _mask(SEED, 2, 5, (rows, d))
    xd, zd = x[:, :d].double(), z[:, :d].double()
    ref_y = xd + D * zd
    b_y = BF * ref_y.abs() + SAFE * 2 * U * (xd.abs() + (D * zd).abs())
    meta = dict(cfg=cfg, rows=rows)
    _check_bound("student_dropout_add_ln_y", y[:, :d], ref_y, b_y, **meta)
    assert (y[:, d:] == SENT).all() and (out[:, d:] == SENT).all()
    _control_bound(y[:, :d], D * (xd + zd), b_y, "the mask applied after the residual add")
    _control_bound(y[:, :d], xd + (D != 0) * zd, b_y, "no 1 / (1 - p) scale")
    yd = y[:, :d].double()
    m, r, dm, er = ln_stats(yd, s.m.ln_eps)
    gd, bd = gamma.double(), beta.double()
    xh = (yd - m) * r
    ref = xh * gd + bd
    dxh = (yd - m).abs() * r * (er + 2 * U) + dm * r
    bound = BF * ref.abs() + SAFE * (gd.abs() * dxh + 2 * U * ((gd * xh).abs() + bd.abs()))
    _check_bound("student_dropout_add_ln_out", out[:, :d], ref, bound, **meta)


def test_dropout_in_place_and_relu_backward_are_exact(lib, students):
    """h' = bf16(h D) over the logical columns (padding untouched); dh = h' > 0 ? bf16(dh / (1 - p)) : 0.  Bit for bit.
    Controls: the mask of the next step; the backward without the scale."""
    s = students("prod")
    gen = _gen(12)
    rows, cols, ld = 160, 1024, 1152
    h = torch.relu(_bf((rows, ld), gen))
    h[:, cols:] = SENT
    h0 = h.clone()
    assert lib.sdo_inplace(s.h, _p(h), ld, rows, cols, SEED, 9, 4, P, _stream()) == 0
    torch.cuda.synchronize()
    D = _mask(SEED, 9, 4, (rows, cols)).float()
    want = (h0[:, :cols].float() * D).bfloat16()
    assert torch.equal(h[:, :cols].view(torch.int16), want.view(torch.int16))
    assert (h[:, cols:] == SENT).all()
    assert not torch.equal(h[:, :cols], (h0[:, :cols].float() * _mask(SEED, 10, 4, (rows, cols)).float()).bfloat16())
    n = rows * ld
    hp = h.clone()
    hp[:, cols:] = 0
    dh = _bf((rows, ld), gen)
    dh0 = dh.clone()
    inv = torch.tensor(1.0, dtype=torch.float32).div_(torch.tensor(1.0, dtype=torch.float32) - torch.tensor(P, dtype=torch.float32))
    assert lib.sdo_relu_bwd(s.h, _p(hp), _p(dh), n, P, _stream()) == 0
    torch.cuda.synchronize()
    want = torch.where(hp.float() > 0, (dh0.float() * inv.cuda()).bfloat16(), torch.zeros_like(dh0))
    assert torch.equal(dh.view(torch.int16), want.view(torch.int16))
    assert not torch.equal(dh, torch.where(hp.float() > 0, dh0, torch.zeros_like(dh0)))


@pytest.mark.parametrize("cfg", ["prod", "small"])
def test_layernorm_backward_with_dropout(lib, students, cfg):
    """dy equals t_ln_bwd's bit for bit (same kernel body) and dz = bf16(dy D) exactly; dgamma / dbeta as t_ln_bwd.
    Control: dz from the mask of another site."""
    s = students(cfg)
    plain = op_modes_shim.load_student()
    gen = _gen(321)
    rows, d, dp = 160, s.d, s.dp
    y = torch.zeros(rows, dp, device="cuda", dtype=torch.bfloat16)
    y[:, :d] = _ln_rows(rows, d, gen)
    dx = torch.zeros(rows, dp, device="cuda", dtype=torch.bfloat16)
    dx[:, :d] = _bf((rows, d), gen) + 0.2
    gamma = torch.randn(d, device="cuda", generator=gen) * 0.5 + 1
    outs = []
    for drop in (False, True):
        dy = torch.full((rows, dp), SENT, device="cuda", dtype=torch.bfloat16)
        dz = torch.full((rows, dp), SENT, device="cuda", dtype=torch.bfloat16)
        dg, db, stats = (torch.full((d,), SENT32, device="cuda"), torch.full((d,), SENT32, device="cuda"),
                         torch.full((2 * rows,), SENT32, device="cuda"))
        if drop:
            assert lib.sdo_ln_bwd(s.h, _p(y), _p(dx), rows, _p(gamma), _p(dy), _p(dz), _p(dg), _p(db), _p(stats), SEED, 1, 3, P, _stream()) == 0
        else:
            assert plain.sto_ln_bwd(s.h, _p(y), _p(dx), rows, _p(gamma), _p(dy), _p(dg), _p(db), _p(stats), _stream()) == 0
        outs.append((dy, dz, dg, db))
    torch.cuda.synchronize()
    (dy0, _, dg0, db0), (dy1, dz1, dg1, db1) = outs
    assert torch.equal(dy0, dy1) and torch.equal(dg0, dg1) and torch.equal(db0, db1)
    D = _mask(SEED, 1, 3, (rows, d)).float()
    want = (dy1[:, :d].float() * D).bfloat16()
    assert torch.equal(dz1[:, :d].view(torch.int16), want.view(torch.int16)) and (dz1[:, d:] == SENT).all()
    assert not torch.equal(dz1[:, :d], (dy1[:, :d].float() * _mask(SEED, 1, 4, (rows, d)).float()).bfloat16())
