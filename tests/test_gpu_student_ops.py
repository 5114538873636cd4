"""Operator tests of the student decoder's kernels (csrc/student.cu: inference, csrc/student_train.cu: the distillation step),
reached through tests/cuda/student_ops.cpp (op_modes_shim.load_student) on the handle of a StudentCandidateV1 in training mode.

Every case feeds the kernel random bf16 / fp32 inputs.  The reference is float64 on the kernel's own operands, so the bf16
rounding of an input is not error.  Each output is checked element by element against a bound derived from the kernel's
arithmetic (u = 2^-24, the fp32 unit roundoff):
  * a bf16 output adds its own rounding, 2^-8 |ref|;
  * an fp32 sum adds n u sum|terms|, where n is the number of roundings a term goes through in the kernel's summation order:
    the terms one thread adds in sequence plus log2(32) shuffle levels (plus the partials of the other warps for a CTA-wide
    sum).  For the warp-per-row LayerNorm over d columns that is d/32 + 5, far below d, which is what lets the bound see a
    one-pass variance on rows with a large mean;
  * __expf(x) adds (2 + 1.173 |x|) 2^-23 relative (CUDA C Programming Guide, intrinsic functions), logf 2^-23 relative,
    rsqrtf 2 ulp;
  * a softmax probability whose logit is off by e is off by p (|e| + sum_k p_k |e_k|) (shift invariance);
  * where the output is a difference (LayerNorm backward, d loss / d logits, dS of the attention backward) the bound is
    absolute on the sum of the terms' magnitudes, not relative to the result.
Errors of errors are covered by a factor 1.01 on the fp32 part.  The measured max error / bound of every case goes to
test_gpu_parity.record().  Each kernel also has negative controls: references with a plausible bug (a dropped term, a mask
off by one, a missing scale, a loss row too many) that the kernel's output must FAIL, so each bound is shown to see them.

Configurations: production (d 576, 8 heads of 72, ffn 1024, vocab 30522 -> 30720), small (64 / 4 heads of 16, vocab 1000) and
the largest head (1024 / 8 heads of 128).  Shapes run up to the limits the code enforces: 64 tokens and 64 memory rows for
training (where the attention backward needs more than 48 KB of shared memory), 128 keys for inference."""
import importlib
import math

import pytest
import torch

import op_modes_shim
from test_gpu_gemm_shapes import _check_bound, _control_bound, f32_bound
from test_gpu_parity import record

pytestmark = pytest.mark.gpu

U = 2.0 ** -24        # fp32 unit roundoff
BF = 2.0 ** -8        # bf16 round to nearest: |bf16(v) - v| <= 2^-8 |v|
SAFE = 1.01           # second-order terms of the fp32 error
SENT = -77.0          # bf16 sentinel
SENT32 = 12345.0      # fp32 sentinel

CONFIGS = {  # name: (d_model, heads, d_ffn, vocab)
    "prod": (576, 8, 1024, 30522),
    "small": (64, 4, 128, 1000),
    "hd128": (1024, 8, 1024, 1000),
}


def _ru(v, m):
    return (v + m - 1) // m * m


class Student:
    def __init__(self, name):
        g = importlib.import_module("real-time-video-captioning_b200")
        d, nh, f, V = CONFIGS[name]
        torch.manual_seed(5)
        self.m = g.StudentCandidateV1(None, d, nh, f, 0.3, 1, V, 101, 102).to("cuda")
        self.m.enable_training()
        self.h = self.m._engine()
        self.name, self.d, self.H, self.hd, self.V = name, d, nh, d // nh, V
        self.dp, self.vp = _ru(d, 128), _ru(V, 256)


@pytest.fixture(scope="module")
def lib():
    import gitb200  # noqa: F401  (loads libgitb200.so before the shim that links against it)
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    importlib.import_module("real-time-video-captioning_b200._lib").load()
    return op_modes_shim.load_student()


_students = {}


@pytest.fixture(scope="module")
def students(lib):
    yield lambda name: _students.setdefault(name, Student(name))
    for s in _students.values():
        s.m.close()
    _students.clear()


def _p(t):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _bf(shape, gen, scale=1.0):
    return (torch.randn(*shape, device="cuda", generator=gen) * scale).bfloat16()


def _expf_err(x):
    """relative error of __expf(x) plus the rounding of its fp32 argument"""
    return (2 + 1.173 * x.abs()) * 2.0 ** -23 + U * x.abs()


def _tokens(B, L, V, gen, pads=()):
    t = torch.randint(1, V, (B, L), device="cuda", generator=gen, dtype=torch.int32)
    t[:, 0] = 101 % V
    for b, j in pads:
        t[b, j] = 0
    return t


# ---------------------------------------------------------------------------------------------------------- embedding
@pytest.mark.parametrize("cfg", ["prod", "small"])
@pytest.mark.parametrize("L,pos0", [(20, 0), (1, 37), (5, 3)])
def test_embed(lib, students, cfg, L, pos0):
    """out[r] = (embed[clamp(tok)] + pe[pos0 + r % L]) / sqrt(d): two fp32 roundings of the sum and product plus the rounding
    of 1/sqrtf(d), then bf16.  Tokens outside [0, vocab) clamp.  Control: the scaling applied before adding pe."""
    s = students(cfg)
    gen = _gen(1)
    B, tok_ld = 3, pos0 + L + 2
    tok = _tokens(B, tok_ld, s.V, gen)
    tok[0, pos0] = -3
    tok[1, pos0 + L - 1] = s.V + 5
    out = torch.full((B * L, s.dp), SENT, device="cuda", dtype=torch.bfloat16)
    assert lib.sto_embed(s.h, _p(tok), tok_ld, L, pos0, B * L, _p(out), _stream()) == 0
    torch.cuda.synchronize()
    emb = s.m._export("embed.weight", 0).double()
    pe = s.m.pos_enc.pe[0].to("cuda").double()
    ids = tok[:, pos0:pos0 + L].long().clamp(0, s.V - 1).reshape(-1)
    e, p = emb[ids], pe[pos0:pos0 + L].repeat(B, 1)
    ref = (e + p) / math.sqrt(s.d)
    bound = BF * ref.abs() + SAFE * 3 * U * (e.abs() + p.abs()) / math.sqrt(s.d)
    _check_bound("student_ops_embed", out[:, :s.d], ref, bound, cfg=cfg, L=L, pos0=pos0)
    assert (out[:, s.d:] == SENT).all()
    _control_bound(out[:, :s.d], e / math.sqrt(s.d) + p, bound, "the scaling applied before adding pe")


# ---------------------------------------------------------------------------------------------------------- LayerNorm
def ln_stats(x, eps):
    """float64 mean / rstd of the rows of x and the kernel's error in them: mean err dm, relative rstd err er."""
    n = x.shape[1]
    depth = math.ceil(n / 32) + 5
    m = x.mean(1, keepdim=True)
    var = ((x - m) ** 2).mean(1, keepdim=True)
    r = (var + eps).rsqrt()
    dm = depth * U * x.abs().sum(1, keepdim=True) / n + U * m.abs()
    dv = dm ** 2 + (depth + 5) * U * (var + dm ** 2 + eps)
    er = SAFE * (0.5 * dv / (var + eps) + 3 * 2.0 ** -23)
    return m, r, dm, er


def _ln_rows(rows, d, gen):
    """random rows, rows with mean 100, and rows that are 2^15 but for a few bumps (mean / sigma ~ 3000: a one-pass
    variance cancels to nothing there)"""
    x = torch.randn(rows, d, device="cuda", generator=gen) * 2
    x[rows // 3:2 * rows // 3] = x[rows // 3:2 * rows // 3] * 2 + 100
    big = torch.full((rows - 2 * rows // 3, d), 32768.0, device="cuda")
    for k in range(big.shape[0]):
        big[k, torch.randint(0, d, (1 + k % 3,), device="cuda", generator=gen)] += 256.0 * (1 + k % 2)
    x[2 * rows // 3:] = big
    return x.bfloat16()


def _one_pass_fp32(x, eps):
    """the kernel with var = E[x^2] - mean^2 in fp32: lane-wise sequential sums, then the 32 lanes"""
    xf = x.float()
    n = xf.shape[1]
    s1 = torch.zeros(xf.shape[0], 32, device="cuda")
    s2 = torch.zeros_like(s1)
    for j in range(0, n, 32):
        c = xf[:, j:j + 32]
        s1[:, :c.shape[1]] += c
        s2[:, :c.shape[1]] += c * c
    m = s1.sum(1, keepdim=True) / n
    var = s2.sum(1, keepdim=True) / n - m * m
    return m.double(), (var.clamp_min(0) + eps).rsqrt().double()


@pytest.mark.parametrize("cfg", ["prod", "small", "hd128"])
def test_layernorm(lib, students, cfg):
    """out = (x - mean) rstd gamma + beta over d columns (eps from the configuration), one warp per row, two-pass variance.  Bound: the mean
    and variance sums as in the module docstring, rsqrtf, then (x - m) rstd gamma + beta and bf16.  Rows with a large mean
    included.  Control: a one-pass variance."""
    s = students(cfg)
    gen = _gen(2)
    rows, d, dp = 150, s.d, s.dp
    x = torch.full((rows, dp), SENT, device="cuda", dtype=torch.bfloat16)
    x[:, :d] = _ln_rows(rows, d, gen)
    gamma = torch.randn(d, device="cuda", generator=gen) * 0.5 + 1
    beta = torch.randn(d, device="cuda", generator=gen) * 0.3
    out = torch.full((rows, dp), SENT, device="cuda", dtype=torch.bfloat16)
    assert lib.sto_ln(s.h, _p(x), dp, rows, _p(gamma), _p(beta), _p(out), dp, _stream()) == 0
    torch.cuda.synchronize()
    xd = x[:, :d].double()
    m, r, dm, er = ln_stats(xd, s.m.ln_eps)
    g, b = gamma.double(), beta.double()
    xh = (xd - m) * r
    ref = xh * g + b
    dxh = (xd - m).abs() * r * (er + 2 * U) + dm * r
    bound = BF * ref.abs() + SAFE * (g.abs() * dxh + 2 * U * ((g * xh).abs() + b.abs()))
    _check_bound("student_ops_layernorm", out[:, :d], ref, bound, cfg=cfg)
    assert (out[:, d:] == SENT).all()
    m1, r1 = _one_pass_fp32(x[:, :d], s.m.ln_eps)
    _control_bound(out[:, :d], (xd - m1) * r1 * g + b, bound, "a one-pass fp32 variance")


# ---------------------------------------------------------------------------------------------------------- attention
def attn_ref(Q, K, Vv, allowed, fwd=True):
    """Q [B, Lq, H, hd], K / V [B, nk, H, hd] (float64 of the bf16 operands), allowed [B, Lq, nk] ->
    (P [B, H, Lq, nk], out [B, Lq, H, hd], dP_bound [B, H, Lq, nk] = the kernel's error in P).
    Score error (hd + 3) u sum|q k| scale (q * scale or s * scale, the fma chain, the fp32 scale); __expf; the normaliser's
    sum (nk + 3 roundings)."""
    hd, nk = Q.shape[-1], K.shape[1]
    scale = 1 / math.sqrt(hd)
    S = torch.einsum("bihc,bjhc->bhij", Q, K) * scale
    Sabs = torch.einsum("bihc,bjhc->bhij", Q.abs(), K.abs()) * scale
    mask = allowed[:, None]
    S = S.masked_fill(~mask, float("-inf"))
    P = torch.softmax(S, -1)
    x = (S - S.amax(-1, keepdim=True)).masked_fill(~mask, 0)
    eta = ((hd + 3) * U * Sabs + _expf_err(x)).masked_fill(~mask, 0)
    dP = P * (eta + (P * eta).sum(-1, keepdim=True) + (nk + 3) * U)
    out = torch.einsum("bhij,bjhc->bihc", P, Vv)
    return P, out, dP


def fwd_bound(P, dP, Vv, out):
    nk = P.shape[-1]
    err = torch.einsum("bhij,bjhc->bihc", dP, Vv.abs()) + (nk + 3) * U * torch.einsum("bhij,bjhc->bihc", P, Vv.abs())
    return BF * out.abs() + SAFE * err


def _self_allowed(tok, Lq, pos0, nk, causal=True, off=0, pads=True):
    B = tok.shape[0]
    i = torch.arange(Lq, device="cuda")[:, None] + pos0
    j = torch.arange(nk, device="cuda")[None, :]
    a = (j <= i + off) if causal else torch.ones(Lq, nk, dtype=torch.bool, device="cuda")
    a = a[None].expand(B, Lq, nk)
    if pads:
        a = a & (tok[:, None, :nk] != 0)
    return a


@pytest.mark.parametrize("cfg", ["prod", "small", "hd128"])
@pytest.mark.parametrize("B,L", [(8, 20), (3, 7), (2, 33), (3, 64), (2, 128)])
def test_self_attention(lib, students, cfg, B, L):
    """Teacher-forced self-attention in the training layout (q | k | v blocks of dp columns in one [B * L, 3 dp] buffer),
    causal + padding mask, pads at the tail and in the middle.  33, 64 and 128 keys: more keys than lanes.  Controls: a
    causal mask that admits j = i + 1; pads ignored."""
    s = students(cfg)
    gen = _gen(3 + L)
    H, hd, dp, d = s.H, s.hd, s.dp, s.d
    qkv = torch.zeros(B * L, 3 * dp, device="cuda", dtype=torch.bfloat16)
    for t in range(3):
        qkv[:, t * dp:t * dp + d] = _bf((B * L, d), gen, 1.5 if t == 0 else 1.0)
    pads = [(0, L - 1), (B - 1, L // 2)] + ([(0, L - 2)] if L > 3 else [])
    tok = _tokens(B, L, s.V, gen, pads)
    out = torch.full((B * L, dp), SENT, device="cuda", dtype=torch.bfloat16)
    assert lib.sto_attn(s.h, _p(qkv), 3 * dp, L, 0, _p(qkv), L, 3 * dp, dp, 2 * dp, L, 1, _p(tok), L, B * L, _p(out), dp, _stream()) == 0
    torch.cuda.synchronize()
    view = qkv.double().view(B, L, 3, dp)[..., :d].reshape(B, L, 3, H, hd)
    Q, K, Vv = view[:, :, 0], view[:, :, 1], view[:, :, 2]
    P, ref, dP = attn_ref(Q, K, Vv, _self_allowed(tok, L, 0, L))
    bound = fwd_bound(P, dP, Vv, ref).reshape(B * L, d)
    got = out[:, :d]
    _check_bound("student_ops_self_attn", got, ref.reshape(B * L, d), bound, cfg=cfg, B=B, L=L)
    assert (out[:, d:] == SENT).all()
    _, wrong, _ = attn_ref(Q, K, Vv, _self_allowed(tok, L, 0, L, off=1))
    _control_bound(got, wrong.reshape(B * L, d), bound, "a causal mask that admits j = i + 1")
    _, wrong, _ = attn_ref(Q, K, Vv, _self_allowed(tok, L, 0, L, pads=False))
    _control_bound(got, wrong.reshape(B * L, d), bound, "padded keys attended to")


@pytest.mark.parametrize("cfg", ["prod", "hd128"])
@pytest.mark.parametrize("Lmax,pos0", [(26, 0), (26, 9), (26, 25), (128, 127)])
def test_cached_decode_attention(lib, students, cfg, Lmax, pos0):
    """The greedy loop's self-attention (run_layers with L = 1): the query of position pos0 sits in the per-layer cache
    [B][Lmax][3 dp] (leading dimension Lmax * 3 dp, offset pos0 * 3 dp) and attends to keys 0 .. pos0 of its own sequence
    with the padding mask.  Keys beyond pos0 hold garbage that must not be read."""
    s = students(cfg)
    gen = _gen(40 + pos0)
    B, H, hd, dp, d = 5, s.H, s.hd, s.dp, s.d
    cache = torch.zeros(B, Lmax, 3 * dp, device="cuda", dtype=torch.bfloat16)
    for t in range(3):
        cache[:, :, t * dp:t * dp + d] = _bf((B, Lmax, d), gen, 1.5 if t == 0 else 1.0)
    cache[:, pos0 + 1:] = 1e4
    tok = _tokens(B, Lmax, s.V, gen, [(1, pos0 // 2)] if pos0 > 1 else [])
    out = torch.full((B, dp), SENT, device="cuda", dtype=torch.bfloat16)
    q = cache[:, pos0]
    assert lib.sto_attn(s.h, _p(q), Lmax * 3 * dp, 1, pos0, _p(cache), Lmax, 3 * dp, dp, 2 * dp, pos0 + 1, 1, _p(tok), Lmax, B, _p(out), dp,
                        _stream()) == 0
    torch.cuda.synchronize()
    view = cache.double()[:, :pos0 + 1].reshape(B, pos0 + 1, 3, dp)[..., :d].reshape(B, pos0 + 1, 3, H, hd)
    Q = view[:, pos0:pos0 + 1, 0]
    K, Vv = view[:, :, 1], view[:, :, 2]
    allowed = _self_allowed(tok, 1, pos0, pos0 + 1)
    P, ref, dP = attn_ref(Q, K, Vv, allowed)
    bound = fwd_bound(P, dP, Vv, ref).reshape(B, d)
    _check_bound("student_ops_cached_attn", out[:, :d], ref.reshape(B, d), bound, cfg=cfg, Lmax=Lmax, pos0=pos0)
    assert (out[:, d:] == SENT).all()
    if pos0 > 2:
        _, wrong, _ = attn_ref(Q, K, Vv, _self_allowed(tok, 1, pos0, pos0 + 1, pads=False))
        _control_bound(out[:, :d], wrong.reshape(B, d), bound, "padded keys attended to")


@pytest.mark.parametrize("cfg", ["prod", "small", "hd128"])
@pytest.mark.parametrize("M", [1, 6, 64, 128])
def test_cross_attention(lib, students, cfg, M):
    """Cross-attention of L = 20 text rows to M memory rows (K | V in one [B * M, 2 dp] buffer), no mask."""
    s = students(cfg)
    gen = _gen(60 + M)
    B, L, H, hd, dp, d = 3, 20, s.H, s.hd, s.dp, s.d
    q = torch.zeros(B * L, dp, device="cuda", dtype=torch.bfloat16)
    q[:, :d] = _bf((B * L, d), gen, 1.5)
    kv = torch.zeros(B * M, 2 * dp, device="cuda", dtype=torch.bfloat16)
    kv[:, :d] = _bf((B * M, d), gen)
    kv[:, dp:dp + d] = _bf((B * M, d), gen)
    out = torch.full((B * L, dp), SENT, device="cuda", dtype=torch.bfloat16)
    assert lib.sto_attn(s.h, _p(q), dp, L, 0, _p(kv), M, 2 * dp, 0, dp, M, 0, None, 0, B * L, _p(out), dp, _stream()) == 0
    torch.cuda.synchronize()
    Q = q.double()[:, :d].reshape(B, L, H, hd)
    K = kv.double()[:, :d].reshape(B, M, H, hd)
    Vv = kv.double()[:, dp:dp + d].reshape(B, M, H, hd)
    P, ref, dP = attn_ref(Q, K, Vv, torch.ones(B, L, M, dtype=torch.bool, device="cuda"))
    _check_bound("student_ops_cross_attn", out[:, :d], ref.reshape(B * L, d), fwd_bound(P, dP, Vv, ref).reshape(B * L, d), cfg=cfg, M=M)
    assert (out[:, d:] == SENT).all()


def test_attention_rejects_more_keys_than_the_kernel_holds(lib, students):
    s = students("small")
    q = torch.zeros(4, 3 * s.dp, device="cuda", dtype=torch.bfloat16)
    out = torch.zeros(4, s.dp, device="cuda", dtype=torch.bfloat16)
    for nk in (0, 129):
        assert lib.sto_attn(s.h, _p(q), 3 * s.dp, 1, 0, _p(q), 4, 3 * s.dp, s.dp, 2 * s.dp, nk, 0, None, 0, 1, _p(out), s.dp, _stream()) != 0


# ---------------------------------------------------------------------------------------------------------- loss
def loss_ref(sl, tl, tok, V, T, ce_rows):
    """float64 loss pieces and d loss / d logits, with the kernel's error bound.  sl, tl [R, >= V] fp32; ce_rows [R] bool,
    tgt [R] the CE targets."""
    R = sl.shape[0]
    B, L = tok.shape
    s, t = sl[:, :V].double(), tl[:, :V].double()
    tgt = torch.zeros(R, dtype=torch.long, device="cuda")
    flat = tok.reshape(-1).long()
    tgt[:-1] = flat[1:]
    nv = int(ce_rows.sum())
    w_kl, w_ce = T / B, (1.0 / nv if nv else 0.0)
    depth = math.ceil(V / 256) + 13

    def lsm(x):
        xs = (x - x.amax(1, keepdim=True))
        lp = torch.log_softmax(xs, 1)
        p = lp.exp()
        ls = torch.logsumexp(xs, 1, keepdim=True)
        dls = (p * (_expf_err(xs) + 2 * U * xs.abs())).sum(1, keepdim=True) + (depth + 1) * U + 2.0 ** -23 * ls.abs()
        dlp = 3 * U * xs.abs() + dls + U * lp.abs()
        return lp, p, dlp, dlp + _expf_err(lp)

    lps, ps, dlps, eps_s = lsm(s / T)
    lpt, pt, dlpt, eps_t = lsm(t / T)
    lp1, p1, _, eps_1 = lsm(s)
    onehot = torch.zeros_like(s)
    onehot[torch.arange(R, device="cuda"), tgt.clamp(0, V - 1)] = 1.0
    ce = ce_rows[:, None].double()
    g = w_kl * (ps - pt) + w_ce * ce * (p1 - onehot)
    gerr = w_kl * (ps * eps_s + pt * eps_t) + w_ce * ce * p1 * eps_1 + 4 * U * (w_kl * (ps + pt) + w_ce * ce * (p1 + onehot))
    gbound = BF * g.abs() + SAFE * gerr
    k = pt * (lpt - lps)
    kl_rows = k.sum(1)
    kl = kl_rows.sum().item() * T * T / B
    kl_err = (T * T / B) * ((pt * (eps_t * (lpt - lps).abs() + dlpt + dlps)).sum() + (depth + 3) * U * k.abs().sum()
                            + (R / 32 + 6) * U * kl_rows.abs().sum()).item() + 3 * U * abs(kl)
    ce_row = -lp1[torch.arange(R, device="cuda"), tgt.clamp(0, V - 1)] * w_ce * ce[:, 0]
    ce_val = ce_row.sum().item()
    ce_err = (w_ce * ce[:, 0] * (3 * U * (s - s.amax(1, keepdim=True)).abs().amax(1) + (p1 * (_expf_err(s - s.amax(1, keepdim=True)))).sum(1)
                                 + (depth + 2) * U + 2.0 ** -23 * lp1.abs().amax(1))).sum().item() + (R / 32 + 7) * U * ce_row.abs().sum().item()
    return g, gbound, kl, SAFE * kl_err, ce_val, SAFE * ce_err


def _run_loss(lib, s, sl, tl, tok, T):
    B, L = tok.shape
    R = B * L
    nvalid = torch.full((1,), -1, device="cuda", dtype=torch.int32)
    dlog = torch.full((R, s.vp), SENT, device="cuda", dtype=torch.bfloat16)
    loss = torch.full((2 * R,), SENT32, device="cuda")
    out = torch.full((3,), SENT32, device="cuda")
    assert lib.sto_distill_loss(s.h, _p(sl), sl.stride(0), _p(tl), tl.stride(0), _p(tok), B, L, T, _p(nvalid), _p(dlog), _p(loss), _p(out),
                                _stream()) == 0
    torch.cuda.synchronize()
    return dlog, out, int(nvalid.item())


@pytest.mark.parametrize("cfg", ["prod", "small"])
@pytest.mark.parametrize("T", [1.0, 2.0, 0.5])
@pytest.mark.parametrize("B,L", [(8, 20), (3, 7), (2, 2)])
def test_distill_loss(lib, students, cfg, T, B, L):
    """KL(batchmean)(log_softmax(s / T), softmax(t / T)) T^2 and CE(ignore 0)(s[:, :-1], y[:, 1:]) over B x L rows, and
    d loss / d logits = T (p_s - p_t) / B + [CE row] (softmax(s) - onehot) / n_valid.  KL and CE are checked separately;
    the last position of a sequence has no CE target; padding columns vocab .. vp of d logits are exactly 0; the student
    logits' own padding columns (set to 1e4 here) are not read; the teacher rows are wider than the vocabulary.  Controls:
    a CE row at position L - 1 (targeting the next sequence's first token); KL without the T^2 factor (T != 1)."""
    s = students(cfg)
    gen = _gen(int(T * 10) + B * L)
    R, V, vp = B * L, s.V, s.vp
    pads = [(0, L - 1)] + ([(B - 1, L - 2), (B - 1, L - 1)] if L > 3 else [])
    tok = _tokens(B, L, V, gen, pads)
    sl = torch.randn(R, vp, device="cuda", generator=gen) * 2
    sl[:, V:] = 1e4
    tl = torch.randn(R, _ru(V, 8) + 8, device="cuda", generator=gen) * 3
    dlog, out, nv = _run_loss(lib, s, sl, tl, tok, T)
    ce_rows = torch.zeros(B, L, dtype=torch.bool, device="cuda")
    ce_rows[:, :-1] = tok[:, 1:] != 0
    ce_rows = ce_rows.reshape(-1)
    assert nv == int(ce_rows.sum())
    g, gb, kl, kl_b, ce, ce_b = loss_ref(sl, tl, tok, V, T, ce_rows)
    _check_bound("student_ops_dlogits", dlog[:, :V], g, gb, cfg=cfg, T=T, B=B, L=L)
    assert (dlog[:, V:] == 0).all()
    kl_got, ce_got = out[1].item(), out[2].item()
    record("student_ops_loss", cfg=cfg, T=T, B=B, L=L, kl_err_over_bound=abs(kl_got - kl) / kl_b, ce_err_over_bound=abs(ce_got - ce) / ce_b)
    assert abs(kl_got - kl) <= kl_b, (kl_got, kl, kl_b)
    assert abs(ce_got - ce) <= ce_b, (ce_got, ce, ce_b)
    assert out[0].item() == (out[1] + out[2]).item()   # loss_total: the fp32 sum of the two parts
    # control: the flat-shifted target gives position L - 1 a CE row (its target: the next sequence's CLS)
    wrong_rows = ce_rows.clone()
    wrong_rows[L - 1::L] = True
    wrong_rows[-1] = False
    gw, _, _, _, ce_w, _ = loss_ref(sl, tl, tok, V, T, wrong_rows)
    _control_bound(dlog[:, :V], gw, gb, "a CE row at position L - 1")
    assert abs(ce_got - ce_w) > ce_b
    if T != 1.0:
        assert abs(kl_got - kl / (T * T)) > kl_b, "negative control passed: the bound cannot see KL without T^2"


@pytest.mark.parametrize("cfg", ["prod", "small"])
def test_distill_loss_with_every_target_ignored(lib, students, cfg):
    """n_valid = 0 (every target is the pad id): the library's choice is CE = 0 with no CE gradient, so the step is the KL
    term alone.  torch's CrossEntropyLoss(ignore_index) returns nan there (mean over no element)."""
    s = students(cfg)
    gen = _gen(77)
    B, L, V, vp = 3, 6, s.V, s.vp
    tok = _tokens(B, L, V, gen)
    tok[:, 1:] = 0
    sl = torch.randn(B * L, vp, device="cuda", generator=gen) * 2
    tl = torch.randn(B * L, _ru(V, 8), device="cuda", generator=gen) * 3
    dlog, out, nv = _run_loss(lib, s, sl, tl, tok, 2.0)
    assert nv == 0 and out[2].item() == 0.0 and out[0].item() == out[1].item()
    g, gb, kl, kl_b, _, _ = loss_ref(sl, tl, tok, V, 2.0, torch.zeros(B * L, dtype=torch.bool, device="cuda"))
    _check_bound("student_ops_dlogits_no_target", dlog[:, :V], g, gb, cfg=cfg)
    assert abs(out[1].item() - kl) <= kl_b
    assert (dlog[:, V:] == 0).all()


# ---------------------------------------------------------------------------------------------------------- LayerNorm backward
@pytest.mark.parametrize("cfg", ["prod", "small", "hd128"])
@pytest.mark.parametrize("rows", [21, 160])
def test_layernorm_backward(lib, students, cfg, rows):
    """dy = rstd (g - mean(g) - xhat mean(g xhat)), g = dx gamma; dgamma = sum_r dx xhat, dbeta = sum_r dx (rows in order);
    stats = (mean, rstd).  dy is a difference: its bound is absolute on |g| + |mean g| + |xhat mean(g xhat)|.  Rows with a
    large mean included.  Controls: the mean(g) (c1) term dropped; the xhat mean(g xhat) (c2) term dropped."""
    s = students(cfg)
    gen = _gen(90 + rows)
    d, dp = s.d, s.dp
    n = d
    depth = math.ceil(n / 32) + 5
    y = torch.full((rows, dp), SENT, device="cuda", dtype=torch.bfloat16)
    y[:, :d] = _ln_rows(rows, d, gen)
    dx = torch.full((rows, dp), SENT, device="cuda", dtype=torch.bfloat16)
    dx[:, :d] = _bf((rows, d), gen) + 0.2
    gamma = torch.randn(d, device="cuda", generator=gen) * 0.5 + 1
    dy = torch.full((rows, dp), SENT, device="cuda", dtype=torch.bfloat16)
    dgamma = torch.full((d,), SENT32, device="cuda")
    dbeta = torch.full((d,), SENT32, device="cuda")
    stats = torch.full((2 * rows,), SENT32, device="cuda")
    assert lib.sto_ln_bwd(s.h, _p(y), _p(dx), rows, _p(gamma), _p(dy), _p(dgamma), _p(dbeta), _p(stats), _stream()) == 0
    torch.cuda.synchronize()
    yd, dxd, gd = y[:, :d].double(), dx[:, :d].double(), gamma.double()
    m, r, dm, er = ln_stats(yd, s.m.ln_eps)
    xh = (yd - m) * r
    g = dxd * gd
    c1 = g.mean(1, keepdim=True)
    c2 = (g * xh).mean(1, keepdim=True)
    inner = g - c1 - xh * c2
    ref = r * inner
    dxh = (yd - m).abs() * r * (er + 2 * U) + dm * r
    dg = U * g.abs()
    dc1 = (depth * U * g.abs().sum(1, keepdim=True) + dg.sum(1, keepdim=True)) / n + U * c1.abs()
    dc2 = ((dg * xh.abs() + g.abs() * dxh).sum(1, keepdim=True) + (depth + 1) * U * (g * xh).abs().sum(1, keepdim=True)) / n + U * c2.abs()
    dinner = dg + dc1 + dxh * c2.abs() + xh.abs() * dc2 + 3 * U * (g.abs() + c1.abs() + (xh * c2).abs())
    bound = BF * ref.abs() + SAFE * (r * dinner + (er + U) * r * inner.abs())
    _check_bound("student_ops_ln_bwd_dy", dy[:, :d], ref, bound, cfg=cfg, rows=rows)
    assert (dy[:, d:] == SENT).all()
    _control_bound(dy[:, :d], r * (g - xh * c2), bound, "the mean(g) term dropped")
    _control_bound(dy[:, :d], r * (g - c1), bound, "the xhat mean(g xhat) term dropped")
    st = stats.view(rows, 2).double()
    _check_bound("student_ops_ln_bwd_stats", st, torch.cat([m, r], 1), torch.cat([dm, er * r], 1) * SAFE, cfg=cfg, rows=rows)
    ref_dg = (dxd * xh).sum(0)
    b_dg = SAFE * ((dxd.abs() * (dxh + 2 * U * xh.abs())).sum(0) + rows * U * (dxd * xh).abs().sum(0))
    _check_bound("student_ops_ln_bwd_dgamma", dgamma, ref_dg, b_dg, cfg=cfg, rows=rows)
    _check_bound("student_ops_ln_bwd_dbeta", dbeta, dxd.sum(0), SAFE * rows * U * dxd.abs().sum(0), cfg=cfg, rows=rows)


# ---------------------------------------------------------------------------------------------------------- attention backward
def attn_bwd_ref(Q, K, Vv, dO, allowed):
    """float64 dQ, dK, dV and their bounds (see the module docstring; dS = P (dP - rowsum(P dP)) is a difference)."""
    hd, Lq, nk = Q.shape[-1], Q.shape[1], K.shape[1]
    scale = 1 / math.sqrt(hd)
    P, _, dPe = attn_ref(Q, K, Vv, allowed)
    Pg = torch.einsum("bihc,bjhc->bhij", dO, Vv)
    dPg = hd * U * torch.einsum("bihc,bjhc->bhij", dO.abs(), Vv.abs())
    dsum = (P * Pg).sum(-1, keepdim=True)
    ddsum = (dPe * Pg.abs() + P * dPg).sum(-1, keepdim=True) + nk * U * (P * Pg.abs()).sum(-1, keepdim=True)
    dS = P * (Pg - dsum)
    ddS = dPe * (Pg - dsum).abs() + P * (dPg + ddsum + U * (Pg.abs() + dsum.abs())) + U * dS.abs()
    dQ = scale * torch.einsum("bhij,bjhc->bihc", dS, K)
    eQ = scale * (torch.einsum("bhij,bjhc->bihc", ddS, K.abs()) + (nk + 3) * U * torch.einsum("bhij,bjhc->bihc", dS.abs(), K.abs()))
    dK = scale * torch.einsum("bhij,bihc->bjhc", dS, Q)
    eK = scale * (torch.einsum("bhij,bihc->bjhc", ddS, Q.abs()) + (Lq + 3) * U * torch.einsum("bhij,bihc->bjhc", dS.abs(), Q.abs()))
    dV = torch.einsum("bhij,bihc->bjhc", P, dO)
    eV = torch.einsum("bhij,bihc->bjhc", dPe, dO.abs()) + (Lq + 1) * U * torch.einsum("bhij,bihc->bjhc", P, dO.abs())
    return [(dQ, BF * dQ.abs() + SAFE * eQ), (dK, BF * dK.abs() + SAFE * eK), (dV, BF * dV.abs() + SAFE * eV)]


@pytest.mark.parametrize("cfg", ["prod", "small", "hd128"])
@pytest.mark.parametrize("B,L,M", [(8, 20, 6), (3, 7, 2), (4, 2, 1), (3, 64, 64)])
def test_attention_backward(lib, students, cfg, B, L, M):
    """attn_bwd_kernel as the distillation step runs it: self-attention with causal + padding mask, q | k | v read from one
    [B L, 3 dp] buffer and dq | dk | dv written in place into one such buffer (the training step's dqkv); cross-attention
    with K | V of the memory rows and d K | d V into [B M, 2 dp].  At L = M = 64 with head dim 128 the kernel runs with
    165 KB of dynamic shared memory.  Masked (padded) keys get exactly zero dK and dV.  Control: dK without the scale."""
    s = students(cfg)
    gen = _gen(B * 1000 + L * 10 + M)
    H, hd, dp, d = s.H, s.hd, s.dp, s.d
    R, Rm = B * L, B * M
    pads = [(0, L - 1)] + ([(B - 1, L // 2), (0, L - 2)] if L > 3 else [])
    tok = _tokens(B, L, s.V, gen, pads)
    qkv = torch.zeros(R, 3 * dp, device="cuda", dtype=torch.bfloat16)
    for t in range(3):
        qkv[:, t * dp:t * dp + d] = _bf((R, d), gen, 1.5 if t == 0 else 1.0)
    dO = torch.zeros(R, dp, device="cuda", dtype=torch.bfloat16)
    dO[:, :d] = _bf((R, d), gen)
    dqkv = torch.full((R, 3 * dp), SENT, device="cuda", dtype=torch.bfloat16)
    assert lib.sto_attn_bwd(s.h, _p(qkv), 3 * dp, L, _p(qkv), L, 3 * dp, dp, 2 * dp, L, 1, _p(tok), L, B, _p(dO), _p(dqkv), 3 * dp, _p(dqkv),
                            3 * dp, dp, 2 * dp, _stream()) == 0
    q2 = torch.zeros(R, dp, device="cuda", dtype=torch.bfloat16)
    q2[:, :d] = _bf((R, d), gen, 1.5)
    kv = torch.zeros(Rm, 2 * dp, device="cuda", dtype=torch.bfloat16)
    kv[:, :d] = _bf((Rm, d), gen)
    kv[:, dp:dp + d] = _bf((Rm, d), gen)
    dq2 = torch.full((R, dp), SENT, device="cuda", dtype=torch.bfloat16)
    dkv = torch.full((Rm, 2 * dp), SENT, device="cuda", dtype=torch.bfloat16)
    assert lib.sto_attn_bwd(s.h, _p(q2), dp, L, _p(kv), M, 2 * dp, 0, dp, M, 0, None, 0, B, _p(dO), _p(dq2), dp, _p(dkv), 2 * dp, 0, dp,
                            _stream()) == 0
    torch.cuda.synchronize()
    meta = dict(cfg=cfg, B=B, L=L, M=M)
    v = qkv.double().view(B, L, 3, dp)[..., :d].reshape(B, L, 3, H, hd)
    G = dO.double()[:, :d].reshape(B, L, H, hd)
    got = dqkv.view(B, L, 3, dp)
    res = attn_bwd_ref(v[:, :, 0], v[:, :, 1], v[:, :, 2], G, _self_allowed(tok, L, 0, L))
    for t, (name, (ref, bound)) in enumerate(zip(("dq", "dk", "dv"), res)):
        _check_bound(f"student_ops_attn_bwd_self_{name}", got[:, :, t, :d], ref.reshape(B, L, d), bound.reshape(B, L, d), **meta)
    assert (got[..., d:] == SENT).all()
    masked = tok == 0
    assert (got[:, :, 1:, :d][masked] == 0).all(), "padded keys received gradient"
    dK, bK = res[1]
    _control_bound(got[:, :, 1, :d], dK.reshape(B, L, d) / s.hd ** -0.5, bK.reshape(B, L, d), "dK without the scale")
    Q2 = q2.double()[:, :d].reshape(B, L, H, hd)
    K2 = kv.double()[:, :d].reshape(B, M, H, hd)
    V2 = kv.double()[:, dp:dp + d].reshape(B, M, H, hd)
    (rq, bq), (rk, bk), (rv, bv) = attn_bwd_ref(Q2, K2, V2, G, torch.ones(B, L, M, dtype=torch.bool, device="cuda"))
    _check_bound("student_ops_attn_bwd_cross_dq", dq2[:, :d], rq.reshape(R, d), bq.reshape(R, d), **meta)
    _check_bound("student_ops_attn_bwd_cross_dk", dkv[:, :d], rk.reshape(Rm, d), bk.reshape(Rm, d), **meta)
    _check_bound("student_ops_attn_bwd_cross_dv", dkv[:, dp:dp + d], rv.reshape(Rm, d), bv.reshape(Rm, d), **meta)
    assert (dq2[:, d:] == SENT).all() and (dkv[:, d:dp] == SENT).all() and (dkv[:, dp + d:] == SENT).all()


def test_attention_backward_rejects_sequences_beyond_the_training_limit(lib, students):
    s = students("small")
    buf = torch.zeros(65, 3 * s.dp, device="cuda", dtype=torch.bfloat16)
    for Lq, nk in ((65, 8), (8, 65), (0, 8)):
        assert lib.sto_attn_bwd(s.h, _p(buf), 3 * s.dp, Lq, _p(buf), nk, 3 * s.dp, s.dp, 2 * s.dp, nk, 0, None, 0, 1, _p(buf), _p(buf),
                                3 * s.dp, _p(buf), 3 * s.dp, s.dp, 2 * s.dp, _stream()) != 0


# ---------------------------------------------------------------------------------------------------------- small kernels
def test_relu_backward(lib, students):
    """dh = 0 wherever the stored activation is not > 0: zero, negative zero and negative values; bit for bit elsewhere."""
    s = students("small")
    gen = _gen(11)
    n = 100_003
    h = _bf((n,), gen)
    h[:1000] = 0.0
    h[1000:2000] = -0.0
    h[2000:2100] = 1e-38
    dh = _bf((n,), gen)
    want = torch.where(h.float() > 0, dh, torch.zeros_like(dh))
    assert lib.sto_relu_bwd(s.h, _p(h), _p(dh), n, _stream()) == 0
    torch.cuda.synchronize()
    assert torch.equal(dh.view(torch.int16), want.view(torch.int16))
    assert (dh[:2000].view(torch.int16) == 0).all()   # +0, not the incoming sign


@pytest.mark.parametrize("R,C", [(21, 640), (160, 1920), (100, 30720), (192, 1024)])
def test_colsum_and_transpose(lib, students, R, C):
    """colsum: fp32 sum over the rows in order -- bit-identical to that sequential fp32 sum, and within R u sum|x| of float64.
    transpose: dst[c, r] = src[r, c], zero in the padding rows R .. round_up(R, 64) and columns C .. C + 64."""
    s = students("prod")
    gen = _gen(R + C)
    ld = C + 64
    x = torch.full((R, ld), SENT, device="cuda", dtype=torch.bfloat16)
    x[:, :C] = _bf((R, C), gen)
    out = torch.full((C + 1,), SENT32, device="cuda")
    assert lib.sto_colsum(s.h, _p(x), ld, R, C, _p(out), _stream()) == 0
    Rp, Cp = _ru(R, 64), C + 64
    t = torch.full((Cp, Rp), SENT, device="cuda", dtype=torch.bfloat16)
    assert lib.sto_transpose(s.h, _p(x), ld, R, C, _p(t), Rp, Cp, _stream()) == 0
    torch.cuda.synchronize()
    seq = torch.zeros(C, device="cuda")
    for r in range(R):
        seq = seq + x[r, :C].float()
    assert torch.equal(out[:C], seq) and out[C].item() == SENT32
    xd = x[:, :C].double()
    _check_bound("student_ops_colsum", out[:C], xd.sum(0), R * U * xd.abs().sum(0), R=R, C=C)
    want = torch.zeros(Cp, Rp, device="cuda", dtype=torch.bfloat16)
    want[:C, :R] = x[:, :C].t()
    assert torch.equal(t, want)


@pytest.mark.parametrize("cfg", ["prod", "small"])
@pytest.mark.parametrize("R", [21, 160, 192])
@pytest.mark.parametrize("which", ["square", "ffn", "memkv"])
def test_weight_grad(lib, students, cfg, R, which):
    """dW [n_pad, k_pad] fp32 = dY^T X over R rows (R not a multiple of 64: the transposes zero-pad the K tail of the GEMM),
    X with x_cols < k_pad (the memory rows: d columns, dp wide) leaves zero columns.  Bound: the fp32 GEMM bound of
    test_gpu_gemm_shapes (f32_bound) at K = round_up(R, 64).  Control: the last row dropped."""
    s = students(cfg)
    gen = _gen(R + len(which))
    d, dp, fp = s.d, s.dp, _ru(CONFIGS[cfg][2], 128)
    n_pad, k_pad, x_cols, ldx = {"square": (dp, dp, dp, dp), "ffn": (fp, dp, dp, dp), "memkv": (2 * dp, dp, d, d)}[which]
    dY = _bf((R, n_pad), gen)
    X = _bf((R, ldx), gen)
    Rp = _ru(R, 64)
    tA = torch.full((n_pad, Rp), SENT, device="cuda", dtype=torch.bfloat16)
    tB = torch.full((k_pad, Rp), SENT, device="cuda", dtype=torch.bfloat16)
    dW = torch.full((n_pad, k_pad), SENT32, device="cuda")
    assert lib.sto_weight_grad(s.h, _p(dY), n_pad, n_pad, _p(X), ldx, x_cols, k_pad, R, _p(dW), _p(tA), _p(tB), _stream()) == 0
    torch.cuda.synchronize()
    Xp = torch.zeros(R, k_pad, device="cuda", dtype=torch.float64)
    Xp[:, :x_cols] = X[:, :x_cols].double()
    ref = dY.double().t() @ Xp
    S = dY.double().abs().t() @ Xp.abs()
    bound = f32_bound(Rp, S, ref, 0)
    _check_bound("student_ops_weight_grad", dW, ref, bound, cfg=cfg, R=R, which=which)
    assert (dW[:, x_cols:] == 0).all()
    wrong = dY[:-1].double().t() @ Xp[:-1]
    _control_bound(dW, wrong, bound, "the last row dropped")


@pytest.mark.parametrize("cfg", ["prod", "small"])
@pytest.mark.parametrize("B,L", [(8, 20), (3, 64)])
def test_embed_backward(lib, students, cfg, B, L):
    """dembed[tok] = sum over the rows of that token, in row order, of fl(dx / sqrt(d)): bit-identical to that ordered fp32
    sum (so run-to-run identical), within R u sum|terms| of the float64 sum.  Repeated tokens (CLS at every sequence start,
    a few words many times), the pad id 0 and ids outside the vocabulary (clamped).  Rows of tokens that do not occur are not
    written (the training step zeroes the block first)."""
    s = students(cfg)
    gen = _gen(B * L)
    d, dp, V = s.d, s.dp, s.V
    R = B * L
    tok = _tokens(B, L, V, gen, [(0, L - 1), (B - 1, 3)])
    tok.view(-1)[5:R:7] = 7
    tok.view(-1)[3] = V + 4
    tok.view(-1)[4] = V - 1
    tok.view(-1)[6] = -2
    dx = torch.full((R, dp), SENT, device="cuda", dtype=torch.bfloat16)
    dx[:, :d] = _bf((R, d), gen)
    runs = []
    for _ in range(2):
        de = torch.full((V, d), SENT32, device="cuda")
        assert lib.sto_embed_bwd(s.h, _p(tok.view(-1)), R, _p(dx), dp, _p(de), _stream()) == 0
        runs.append(de)
    torch.cuda.synchronize()
    de = runs[0]
    assert torch.equal(runs[0], runs[1])
    ids = tok.view(-1).long().clamp(0, V - 1)
    inv = torch.tensor(1.0, dtype=torch.float32) / torch.sqrt(torch.tensor(float(d), dtype=torch.float32))
    seq = torch.zeros(V, d, device="cuda")
    ref = torch.zeros(V, d, device="cuda", dtype=torch.float64)
    absum = torch.zeros_like(ref)
    for r, i in enumerate(ids.tolist()):
        seq[i] = seq[i] + dx[r, :d].float() * inv.item()
        ref[i] += dx[r, :d].double() / math.sqrt(d)
        absum[i] += dx[r, :d].double().abs() / math.sqrt(d)
    used = torch.zeros(V, dtype=torch.bool, device="cuda")
    used[ids] = True
    assert torch.equal(de[used], seq[used]), "not the row-ordered fp32 sum"
    _check_bound("student_ops_embed_bwd", de[used], ref[used], SAFE * (R + 2) * U * absum[used], cfg=cfg, B=B, L=L)
    assert (de[~used] == SENT32).all()
    assert used[0] and used[V - 1] and used[7]


# ---------------------------------------------------------------------------------------------------------- the whole step
def _step_inputs(V, B=8, L=20, M=6, d=576, seed=3):
    gen = torch.Generator().manual_seed(seed)
    y = torch.randint(min(1000, V // 2), V, (B, L), generator=gen)
    y[:, 0] = 101
    y[0, L - 3:] = 0
    y[1, 4:6] = 7
    mem = torch.randn(B, M, d, generator=gen)
    teacher = torch.randn(B, L, V, generator=gen) * 1.5
    return y, mem, teacher


def test_distillation_step_is_bit_reproducible(students):
    """Two distillation_step(apply=False) calls on the same inputs give bit-identical gradients, d loss / d memory and loss
    (the embedding gradient sums each token's rows in row order, and the loss sums its rows' parts in a fixed order, instead
    of with atomics), and so does a third after another batch ran in between."""
    s = students("prod").m
    y, mem, teacher = _step_inputs(30522)
    outs = []
    for k in range(3):
        if k == 2:
            y2, m2, t2 = _step_inputs(30522, B=3, L=7, M=2, seed=9)
            s.distillation_step(y2, m2, t2, apply=False)
        o = s.distillation_step(y, mem, teacher, apply=False, want_memory_grad=True)
        torch.cuda.synchronize()
        outs.append((s._grads.clone(), o["d_memory"].clone(), torch.stack([o["loss"], o["kl"], o["ce"]])))
    for g, dm, loss in outs[1:]:
        assert torch.equal(g, outs[0][0]) and torch.equal(dm, outs[0][1]) and torch.equal(loss, outs[0][2])


def test_padding_of_the_flat_vectors_stays_zero(students):
    """The flat gradient vector's padding (rows / columns beyond the reference shapes, alignment gaps) stays exactly zero:
    its nonzero count equals the nonzero counts of the exported gradients, before and after three Adam steps (the padding of
    the master weights would otherwise leak into the gradients through the padded operands)."""
    s = students("small").m
    y, mem, teacher = _step_inputs(1000, B=4, L=9, M=3, d=64, seed=4)

    def counts():
        torch.cuda.synchronize()
        flat = int((s._grads != 0).sum())
        exported = sum(int((v != 0).sum()) for v in s.gradients().values())
        return flat, exported

    s.distillation_step(y, mem, teacher, apply=False)
    before = counts()
    for _ in range(3):
        s.distillation_step(y, mem, teacher, apply=True)
    after = counts()
    record("student_padding_nonzeros", before_flat=before[0], before_exported=before[1], after_flat=after[0], after_exported=after[1])
    assert before[0] == before[1] and after[0] == after[1], (before, after)
    assert before[1] > 0 and after[1] > 0
