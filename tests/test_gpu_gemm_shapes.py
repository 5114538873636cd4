"""Operator tests of gemm_bf16 at the shapes and epilogues the engine's launch sequences give it (api.cu run_encode /
run_visual_pass / run_text_pass, student.cu, student_train.cu), on every kernel that can run each problem: the skinny
weight-streaming kernel, the 1-CTA tcgen05 kernel with 128- and 256-wide tiles and the CTA-pair kernel.  Reached through
tests/cuda/op_modes.cpp (op_modes_shim.py) with the helpers, sentinels and negative-control style of test_gpu_op_modes.py.

References are float64 torch on the exact bf16 operands.  bf16 outputs use the suite's 0.02 + 0.01 |ref|.  fp32 outputs use
a bound scaled by the size of the sum rather than of its result (f32_bound): 2 units of 2^-23 per 16-deep MMA step (+ 2 for
the epilogue's adds) times S = (|A| |W|^T)_ij + |bias_j| + |res_ij|, times the activation's slope (< 1.13), plus the
activation's own bound (act_bound, from the claims in common.cuh).  At K = 768 that is ~1.2e-5 S, about 40x tighter than
the suite's flat 3e-3 + 2e-3 |ref|.

Bit identity asserted: all tcgen05 kernels (128, 256, pair) give the same bf16 output, and 128 / 256 the same fp32 output,
for every shape (same K order into the fp32 accumulator, same epilogue expression); for m > 8, rows [0, m) do not depend on
how many rows the call has, although the kernel choice does (what the sub-batch sweeps rely on); a bf16 output written
together with an fp32 one is that fp32 output rounded to nearest even; the pair kernel is run-to-run identical.  The skinny
kernel sums in another order and is checked against the reference only: at m <= 8 the engine's call runs it, so the rows of
a decode step of a few rows are NOT bit-identical to the same rows inside a larger call.  Measured errors go through
test_gpu_parity.record()."""
import importlib
import math

import pytest
import torch

import op_modes_shim
from test_gpu_op_modes import (ACT_NONE, ACT_RELU, BF16_TOL, INVALID, SENT, SENT32, _bf, _check, _control, _gen, _p,
                               _stream, gemm)
from test_gpu_parity import record

pytestmark = pytest.mark.gpu

ACT_QUICK, ACT_ERF = 1, 2
SKINNY, TILE128, TILE256, PAIR = 1, 128, 256, 2          # force_bn values
KNAME = {0: "auto", SKINNY: "skinny", TILE128: "tile128", TILE256: "tile256", PAIR: "pair"}
# the GEMM kernels as the profiler names them
KERNEL_TAGS = {"gemv_skinny_kernel": SKINNY, "gemm_tcgen05_kernel<128>": TILE128, "gemm_tcgen05_kernel<256>": TILE256,
               "gemm2_kernel": PAIR}
TANH_REL = 2.0 ** -10.987   # tanh.approx.f32: maximum relative error stated by the PTX ISA
FIT_ERR = 8.7e-5            # erf-GELU: error of the odd-polynomial fit with an exact tanh (common.cuh; 8.68e-5 at |x| = 1.325)
BF16_U = 2.0 ** -8          # bf16 round to nearest: |bf16(v) - v| <= 2^-8 |v|


@pytest.fixture(scope="module")
def lib():
    import gitb200  # noqa: F401  (loads libgitb200.so before the shim that links against it)
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    importlib.import_module("real-time-video-captioning_b200._lib").load()
    return op_modes_shim.load()


def kernels(M, N, f32_only):
    """force_bn values that really run this problem.  gemm_bf16 quietly hands a problem that a forced kernel declines to
    another kernel, so each is requested only where its preconditions hold (test_dispatch pins the rule):
      * skinny (1): M <= 8;
      * 1-CTA 128-wide tiles (128): every shape;
      * 1-CTA 256-wide tiles (256): N % 256 == 0, else the 128-wide kernel runs;
      * CTA pair (2): N % 256 == 0, a bf16 output and no fp32 output (and no row remap), else the 256-wide kernel runs."""
    ks = [TILE128]
    if M <= 8:
        ks.append(SKINNY)
    if N % 256 == 0:
        ks.append(TILE256)
        if not f32_only:
            ks.append(PAIR)
    return ks


def act_ref(x, act):
    if act == ACT_QUICK:
        return x * torch.sigmoid(1.702 * x)
    if act == ACT_ERF:
        return 0.5 * x * (1 + torch.erf(x / math.sqrt(2)))
    if act == ACT_RELU:
        return x.clamp_min(0)
    return x


def act_bound(x, act):
    """|device activation - exact activation| at the float64 input x, from common.cuh's claims: QuickGELU is
    0.5x (1 + tanh.approx(0.851x)); erf-GELU is 0.5x (1 + tanh.approx(g(x))) with g fitted so that the GELU is off by at most
    8.7e-5 with an exact tanh (and tanh(g) within 1.4e-4 of erf).  tanh.approx adds 2^-10.987 relative to |tanh|, times |x| / 2;
    2^-20 |x| / 2 covers the fp32 roundings of the argument and the fma (a few units of 2^-24)."""
    hx = 0.5 * x.abs()
    if act == ACT_QUICK:
        return hx * (TANH_REL * torch.tanh(0.851 * x).abs() + 2.0 ** -20)
    if act == ACT_ERF:
        return FIT_ERR + hx * (TANH_REL * (torch.erf(x.abs() / math.sqrt(2)) + 2e-4).clamp_max(1) + 2.0 ** -20)
    return torch.zeros_like(x)


def reference(A, W, bias, res, act):
    """(ref, pre-activation, S) in float64; S = |A| |W|^T + |bias| + |res|, the size of the sum the kernel forms."""
    pre = A.double() @ W.double().t()
    S = A.double().abs() @ W.double().abs().t()
    if bias is not None:
        pre += bias.double()
        S += bias.double().abs()
    ref = act_ref(pre, act)
    if res is not None:
        ref += res.double()
        S += res.double().abs()
    return ref, pre, S


def f32_bound(K, S, pre, act):
    return 1.13 * (math.ceil(K / 16) + 2) * 2.0 ** -22 * S + act_bound(pre, act)


def _check_bound(name, x, ref, bound, **meta):
    err = (x.double() - ref).abs()
    ratio = (err / bound.clamp_min(1e-300)).max().item()   # (the bound is 0 only where the activation's input is 0)
    record(name, max_err=err.max().item(), max_err_over_bound=ratio, **meta)
    bad = err > bound
    assert not bad.any(), f"{name} {meta}: {int(bad.sum())} elements outside the bound, max err / bound {ratio:.4g}"


def _control_bound(x, wrong, bound, what):
    """Negative control at an fp32 bound: the kernel's output must fail it against a reference with a plausible bug."""
    assert ((x.double() - wrong).abs() > bound).any(), f"negative control passed: the bound cannot see {what}"


def _gemm_kernels(fn):
    """The GEMM kernels fn() launches, in launch order, as force_bn values (torch.profiler's CUDA activity)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    evs = sorted((e for e in prof.events() if any(t in e.name for t in KERNEL_TAGS)), key=lambda e: e.time_range.start)
    return [next(v for t, v in KERNEL_TAGS.items() if t in e.name) for e in evs]


# ------------------------------------------------------------------------------------------ shape table
def _cases():
    """Every GEMM of the launch sequences.  res: None, "sep" (residual != out) or "inplace" (out == residual, x += f(x));
    out: "bf16" or "f32" (fp32 only: the vocabulary heads and the student's weight gradients); lda > K where the engine's
    A rows are wider than K; kv_only: the decoder's last layer, W and bias offset by H rows of the [3H, H] QKV weight and the
    output written into columns [H, 3H) of the [M, 3H] K|V rows (ldo 3H)."""
    cases = []

    def add(path, Ms, N, K, act=ACT_NONE, bias=True, res=None, out="bf16", lda=None, kv_only=False):
        for M in Ms:
            c = dict(path=path, M=M, N=N, K=K, act=act, bias=bias, res=res, out=out, lda=lda or K, kv_only=kv_only)
            cases.append(pytest.param(c, id=f"{path}-M{M}"))

    # ViT-B/16 (api.cu run_encode): 197 tokens per frame, 4 / 6 / 12 / 36 frames
    vit_b = [788, 1182, 2364, 7092]
    add("vitb_qkv", vit_b, 2304, 768)
    add("vitb_out", vit_b, 768, 768, res="inplace")
    add("vitb_fc1", vit_b, 3072, 768, act=ACT_QUICK)
    add("vitb_fc2", vit_b, 768, 3072, res="inplace")
    # ViT-L/14: 257 tokens per frame, 6 / 12 frames
    vit_l = [1542, 3084]
    add("vitl_qkv", vit_l, 3072, 1024)
    add("vitl_out", vit_l, 1024, 1024, res="inplace")
    add("vitl_fc1", vit_l, 4096, 1024, act=ACT_QUICK)
    add("vitl_fc2", vit_l, 1024, 4096, res="inplace")
    # decoder over the visual tokens (run_visual_pass): 1 / 2 clips of 1182
    vis = [1182, 2364]
    add("dec_vis_proj", vis, 768, 768)
    add("dec_vis_proj_vitl", vis, 768, 1024)
    add("dec_vis_qkv", vis, 2304, 768)
    add("dec_vis_kv_only", vis, 1536, 768, kv_only=True)
    add("dec_vis_out", vis, 768, 768, res="sep")
    add("dec_vis_fc1", vis, 3072, 768, act=ACT_ERF)
    add("dec_vis_fc2", vis, 768, 3072, res="sep")
    # decoder text rows (run_text_pass): a beam-4 step of one clip, teacher forcing and decode steps of many clips
    txt = [4, 9, 300, 1023, 1024, 2048]
    add("dec_txt_qkv", txt, 2304, 768)
    add("dec_txt_out", txt, 768, 768, res="sep")
    add("dec_txt_fc1", txt, 3072, 768, act=ACT_ERF)
    add("dec_txt_fc2", txt, 768, 3072, res="sep")
    add("dec_txt_vocab", txt, 30720, 768, out="f32")
    # student decoder forward (student.cu run_layers / prepare, student_train.cu): d 576 in rows of dp = 640, ffn 1024
    st = [48, 160]
    add("stu_qkv", st, 1920, 576, lda=640)
    add("stu_ca_kv", st, 1280, 576)
    add("stu_out", st, 640, 576, res="sep", lda=640)
    add("stu_ff1", st, 1024, 576, act=ACT_RELU, lda=640)
    add("stu_ff2", st, 640, 1024, res="sep")
    add("stu_vocab", st, 30720, 576, out="f32", lda=640)
    # student backward (student_train.cu): dX = dY W^T through the vocabulary head, ff1 and the self-attention input
    add("stu_dx_vocab", [160], 640, 30720, bias=False)
    add("stu_dx_ff1", [160], 640, 1024, bias=False, res="sep")
    add("stu_dx_sa_in", [160], 640, 1920, bias=False, res="sep")
    # weight gradients dW = dY^T X (t_weight_grad): K = round_up(B * L, 64), one to three k-blocks per tile, fp32 output
    for N, K in [(640, 64), (640, 192), (1024, 192)]:
        add(f"stu_dw_{N}x{K}", [640, 1024, 1280, 1920, 30720], N, K, bias=False, out="f32")
    return cases


@pytest.mark.parametrize("case", _cases())
def test_engine_gemm_shapes(lib, case):
    """The engine's call (force_bn 0, its own output mode, in place where the engine works in place) and every kernel that
    can run the problem; the 1-CTA and skinny kernels write both outputs.  Against the fp64 reference, bit identity across
    the tcgen05 kernels and with the engine's call, dual outputs, sentinels, and negative controls."""
    M, N, K, act, path = case["M"], case["N"], case["K"], case["act"], case["path"]
    f32_only, kv_only, res_mode = case["out"] == "f32", case["kv_only"], case["res"]
    gen = _gen(M * 131 + N * 7 + K)
    A = _bf((M, case["lda"]), gen)[:, :K]          # gap columns (lda > K) hold values a wrong lda would read
    if kv_only:
        H = K
        Wq = _bf((3 * H, K), gen, K ** -0.5)
        bq = torch.randn(3 * H, device="cuda", generator=gen)
        W, bias = Wq[H:], bq[H:]
    else:
        W = _bf((N, K), gen, K ** -0.5)
        bias = torch.randn(N, device="cuda", generator=gen) if case["bias"] else None
    res = _bf((M, N), gen, 2.0) if res_mode else None
    ref, pre, S = reference(A, W, bias, res, act)
    bnd32 = f32_bound(K, S, pre, act)
    ldo, c0 = (3 * K, K) if kv_only else (N, 0)
    meta = dict(path=path, M=M, N=N, K=K)

    def run(force_bn, bf16, f32, inplace=False):
        ob = torch.full((M + 1, ldo), SENT, device="cuda", dtype=torch.bfloat16) if bf16 else None
        o32b = torch.full((M + 1, N), SENT32, device="cuda") if f32 else None
        out = ob[:M, c0:c0 + N] if bf16 else None
        o32 = o32b[:M] if f32 else None
        r = res
        if inplace:
            out.copy_(res)
            r = out
        assert gemm(lib, A, W, bias=bias, res=r, act=act, out=out, o32=o32, force_bn=force_bn) == 0
        if bf16:
            assert (ob[M] == SENT).all(), f"{KNAME[force_bn]}: a bf16 row past M was written"
            assert (ob[:, :c0] == SENT).all(), f"{KNAME[force_bn]}: the Q columns of the K|V-only output were written"
        if f32:
            assert (o32b[M] == SENT32).all(), f"{KNAME[force_bn]}: an fp32 row past M was written"
        return out, o32

    prod, prod32 = run(0, not f32_only, f32_only, inplace=res_mode == "inplace")
    got = {}
    for k in kernels(M, N, f32_only):
        got[k] = run(k, True, k != PAIR)
        out, o32 = got[k]
        _check("gemm_shapes_bf16", out, ref, BF16_TOL, kernel=KNAME[k], **meta)
        if o32 is not None:
            _check_bound("gemm_shapes_f32", o32, ref, bnd32, kernel=KNAME[k], **meta)
            assert torch.equal(out, o32.bfloat16()), f"{KNAME[k]}: bf16 output != fp32 output rounded to nearest even"
    base, base32 = got[TILE128]
    for k in (TILE256, PAIR):
        if k in got:
            assert torch.equal(got[k][0], base), f"{KNAME[k]} and tile128 bf16 outputs differ"
    if TILE256 in got:
        assert torch.equal(got[TILE256][1], base32), "tile256 and tile128 fp32 outputs differ"
    if PAIR in got and path.startswith("vit"):
        again, _ = run(PAIR, True, False)
        assert torch.equal(again, got[PAIR][0]), "CTA-pair kernel not run-to-run identical"
    # the engine's call equals the kernel it dispatches to (the skinny kernel for M <= 8, otherwise any tcgen05 kernel)
    same, same32 = got[SKINNY] if M <= 8 else got[TILE128]
    if f32_only:
        assert torch.equal(prod32, same32)
        _check_bound("gemm_shapes_engine_f32", prod32, ref, bnd32, **meta)
    else:
        assert torch.equal(prod, same)
        _check("gemm_shapes_engine_bf16", prod, ref, BF16_TOL, **meta)

    # negative controls on the engine's output (bf16 tolerance or fp32 bound) and on the fp32 output (activations)
    x, tol_ok = (prod32, None) if f32_only else (prod, BF16_TOL)

    def control(wrong, what):
        if tol_ok is None:
            _control_bound(x, wrong, bnd32, what)
        else:
            _control(x, wrong, tol_ok, what)

    rr = res.double() if res is not None else 0
    if bias is not None:
        control(act_ref(pre - bias.double() + bias.double().roll(128), act) + rr, "bias from the neighbouring 128-column tile")
    if res is not None and M > 1:
        control(act_ref(pre, act) + res.double().roll(1, 0), "the residual row off by one")
    if act in (ACT_QUICK, ACT_ERF):
        _control_bound(base32, act_ref(pre, ACT_ERF + ACT_QUICK - act) + rr, bnd32, "the other GELU")
    if act == ACT_RELU:
        _control_bound(base32, pre + rr, bnd32, "a missing ReLU")
    if bias is None:  # the backward GEMMs (no bias, no activation): a tile whose last k-block never reached the accumulator
        k0 = (K - 1) // 64 * 64
        control(A[:, :k0].double() @ W[:, :k0].double().t() + rr, "the last K block dropped")


# ------------------------------------------------------------------------------------------ dispatch
HEURISTIC_SMS = 148  # force_bn 0 weighs tiles against gemm_sm_count(): the expected choices below are those of a B200


def _heuristic_as_on_b200():
    return torch.cuda.get_device_properties(0).multi_processor_count == HEURISTIC_SMS


DISPATCH = [  # (M, N, outputs, force_bn, kernel that runs)
    (4, 2304, "bf16", 0, SKINNY), (4, 30720, "f32", 0, SKINNY), (9, 2304, "bf16", 0, TILE128),
    (788, 2304, "bf16", 0, TILE128), (1024, 2304, "bf16", 0, TILE128), (1182, 2304, "bf16", 0, PAIR),
    (2048, 2304, "bf16", 0, PAIR), (7092, 3072, "bf16", 0, PAIR), (2048, 30720, "f32", 0, TILE256),
    (4, 2304, "bf16", SKINNY, SKINNY), (300, 768, "bf16", TILE128, TILE128), (300, 768, "bf16", TILE256, TILE256),
    (300, 768, "bf16", PAIR, PAIR), (4, 768, "bf16", PAIR, PAIR),
    # a forced kernel that declines the problem hands it on without an error
    (9, 2304, "bf16", SKINNY, TILE256), (300, 640, "bf16", TILE256, TILE128), (2364, 768, "both", PAIR, TILE256),
    (2364, 640, "bf16", PAIR, TILE128), (2364, 768, "f32", PAIR, TILE256),
]


def test_dispatch(lib):
    """The kernel gemm_bf16 runs for each forced kernel (the rule kernels() relies on) and, on a device with the B200's 148
    SMs, for the engine's heuristic (force_bn 0), read from the profiler."""
    table = [d for d in DISPATCH if d[3] != 0 or _heuristic_as_on_b200()]
    probs = []
    for M, N, outs, fbn, _ in table:
        gen = _gen(M + N)
        A, W = _bf((M, 768), gen), _bf((N, 768), gen, 768 ** -0.5)
        out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16) if outs in ("bf16", "both") else None
        o32 = torch.empty(M, N, device="cuda") if outs in ("f32", "both") else None
        probs.append((A, W, out, o32, fbn))

    def launch_all():
        for A, W, out, o32, fbn in probs:
            assert gemm(lib, A, W, out=out, o32=o32, force_bn=fbn) == 0

    launch_all()   # module loads and tensor maps outside the profiled window
    ran = _gemm_kernels(launch_all)
    want = [k for *_, k in table]
    assert ran == want, [(d[:4], KNAME[r]) for d, r, w in zip(table, ran, want) if r != w] or ran


# ------------------------------------------------------------------------------------------ row invariance
@pytest.mark.parametrize("m,M,N,K,act,res", [
    (788, 7092, 2304, 768, ACT_NONE, False), (788, 7092, 3072, 768, ACT_QUICK, False), (788, 7092, 768, 768, ACT_NONE, True),
    (788, 7092, 768, 3072, ACT_NONE, True), (788, 1182, 3072, 768, ACT_ERF, False), (1024, 2048, 2304, 768, ACT_NONE, False),
    (300, 4728, 768, 3072, ACT_NONE, True), (9, 2048, 3072, 768, ACT_ERF, False)])
def test_rows_do_not_depend_on_the_call(lib, m, M, N, K, act, res):
    """Rows [0, m) of a call with m rows == the same rows inside a call with M rows, bit for bit, although the engine's
    heuristic sends the two calls to different kernels (checked on a 148-SM device, where the pairs were chosen so): the
    property the sub-batch sweeps (gitb200_set_sweep_rows) and batch invariance rest on."""
    gen = _gen(m + M + N + K)
    A = _bf((M, K), gen)
    W = _bf((N, K), gen, K ** -0.5)
    bias = torch.randn(N, device="cuda", generator=gen)
    r = _bf((M, N), gen, 2.0) if res else None
    small = torch.full((m + 1, N), SENT, device="cuda", dtype=torch.bfloat16)
    big = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)

    def both():
        assert gemm(lib, A[:m], W, bias=bias, res=None if r is None else r[:m], act=act, out=small[:m]) == 0
        assert gemm(lib, A, W, bias=bias, res=r, act=act, out=big) == 0

    ran = _gemm_kernels(both)
    assert len(ran) == 2, [KNAME[k] for k in ran]
    if _heuristic_as_on_b200():
        assert ran[0] != ran[1], [KNAME[k] for k in ran]
    assert (small[m] == SENT).all()
    assert torch.equal(small[:m], big[:m]), f"rows differ between {KNAME[ran[0]]} (M = {m}) and {KNAME[ran[1]]} (M = {M})"
    ref, _, _ = reference(A[:m], W, bias, None if r is None else r[:m], act)
    _check("gemm_shapes_row_invariance", small[:m], ref, BF16_TOL, m=m, M=M, N=N, K=K)


# ------------------------------------------------------------------------------------------ CTA-pair row tails
@pytest.mark.parametrize("M", [1, 127, 128, 129, 255, 1025, 1151, 1152, 1153, 1279])
def test_pair_row_tails(lib, M):
    """M % 256 in {1, 127, 128, 129, 255}: for M % 256 <= 128 the rank-1 CTA of the last pair has no rows (its A box lies wholly
    past M, its epilogue stores nothing).  The row past M keeps its sentinel; output == the 128-wide kernel's bit for bit."""
    N, K = 768, 768
    gen = _gen(M)
    A = _bf((M, K), gen)
    W = _bf((N, K), gen, K ** -0.5)
    bias = torch.randn(N, device="cuda", generator=gen)
    res = _bf((M, N), gen, 2.0)
    outs = {}
    for k in (PAIR, TILE128):
        buf = torch.full((M + 1, N), SENT, device="cuda", dtype=torch.bfloat16)
        assert gemm(lib, A, W, bias=bias, res=res, act=ACT_ERF, out=buf[:M], force_bn=k) == 0
        assert (buf[M] == SENT).all(), f"{KNAME[k]}: the row past M was written"
        outs[k] = buf[:M]
    assert torch.equal(outs[PAIR], outs[TILE128])
    ref, pre, _ = reference(A, W, bias, res, ACT_ERF)
    _check("gemm_shapes_pair_tail", outs[PAIR], ref, BF16_TOL, M=M)
    if M > 1:
        _control(outs[PAIR], act_ref(pre, ACT_ERF) + res.double().roll(1, 0), BF16_TOL, "the residual row off by one")


# ------------------------------------------------------------------------------------------ K edges
@pytest.mark.parametrize("K", [8, 56, 64, 72, 136, 192, 256, 320, 384, 448])
def test_k_edges_many_tiles(lib, K):
    """gemm_bf16 takes any K % 8 == 0 (the TMA box zero-fills the K tail); the engine only uses multiples of 64.  M 30720 x N 1024:
    13 tiles per CTA on the 128-wide kernel, 480 pair tiles.  k-blocks: 1 (K <= 64), 2-3, and around the stage counts (6 on the
    128-wide and pair kernels: K 384 = 6, 448 = 7; 4 on the 256-wide kernel: K 256 = 4, 320 = 5)."""
    M, N = 30720, 1024
    gen = _gen(K)
    A = _bf((M, K), gen)
    W = _bf((N, K), gen, K ** -0.5)
    bias = torch.randn(N, device="cuda", generator=gen)
    res = _bf((M, N), gen, 2.0)
    ref, pre, S = reference(A, W, bias, res, ACT_NONE)
    bnd32 = f32_bound(K, S, pre, ACT_NONE)
    got = {}
    for k in (TILE128, TILE256, PAIR):
        out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
        o32 = torch.empty(M, N, device="cuda") if k != PAIR else None
        assert gemm(lib, A, W, bias=bias, res=res, out=out, o32=o32, force_bn=k) == 0
        _check("gemm_shapes_k_edge_bf16", out, ref, BF16_TOL, K=K, kernel=KNAME[k])
        if o32 is not None:
            _check_bound("gemm_shapes_k_edge_f32", o32, ref, bnd32, K=K, kernel=KNAME[k])
            assert torch.equal(out, o32.bfloat16())
        got[k] = (out, o32)
    assert torch.equal(got[TILE256][0], got[TILE128][0]) and torch.equal(got[PAIR][0], got[TILE128][0])
    assert torch.equal(got[TILE256][1], got[TILE128][1])
    if K % 64:
        k0 = K // 64 * 64
        dropped = A[:, :k0].double() @ W[:, :k0].double().t() + bias.double() + res.double()
        for k in (TILE128, TILE256, PAIR):
            _control(got[k][0], dropped, BF16_TOL, f"the last K block dropped ({KNAME[k]})")


# ------------------------------------------------------------------------------------------ activations
def _sweep_points():
    """65536 fp32 inputs: 65524 evenly over [-12, 12] plus +-0, +-1e-30, +-1e4, +-8 and its neighbours (erf-GELU's clamp edge)."""
    e = torch.tensor([8.0])
    edge = torch.cat([e, torch.nextafter(e, torch.tensor([0.0])), torch.nextafter(e, torch.tensor([math.inf]))])
    special = torch.cat([torch.tensor([0.0, 1e-30, 1e4]), edge])
    special = torch.cat([special, -special])
    x = torch.linspace(-12, 12, 65536 - special.numel(), dtype=torch.float32)
    return torch.cat([x, special]).cuda()


@pytest.mark.parametrize("act", [ACT_QUICK, ACT_ERF])
def test_activation_contract(lib, act):
    """A bias-only GEMM (A = 0, W = 0: the accumulator is exactly 0, so column n holds act(bias[n])) on every kernel, against
    float64 within act_bound: the device computes what common.cuh claims.  All kernels share the epilogue expression, so
    their outputs are identical.  Control: the other GELU (up to 0.02 away) fails the bound."""
    x = _sweep_points()
    N, K, M = x.numel(), 64, 1
    A = torch.zeros(M, K, device="cuda", dtype=torch.bfloat16)
    W = torch.zeros(N, K, device="cuda", dtype=torch.bfloat16)
    x64 = x.double()[None]
    ref = act_ref(x64, act)
    bnd = act_bound(x64, act)
    bnd16 = bnd + BF16_U * (ref.abs() + bnd)
    wrong = act_ref(x64, ACT_ERF + ACT_QUICK - act)
    name = {ACT_QUICK: "quick_gelu", ACT_ERF: "gelu_erf"}[act]
    outs = {}
    for k in (SKINNY, TILE128, TILE256, PAIR):
        out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
        o32 = torch.empty(M, N, device="cuda") if k != PAIR else None
        assert gemm(lib, A, W, bias=x, act=act, out=out, o32=o32, force_bn=k) == 0
        _check_bound(f"gemm_shapes_act_{name}_bf16", out, ref, bnd16, kernel=KNAME[k])
        _control_bound(out, wrong, bnd16, f"the other GELU ({KNAME[k]}, bf16)")
        if o32 is not None:
            _check_bound(f"gemm_shapes_act_{name}_f32", o32, ref, bnd, kernel=KNAME[k])
            _control_bound(o32, wrong, bnd, f"the other GELU ({KNAME[k]}, fp32)")
            assert torch.equal(out, o32.bfloat16())
        outs[k] = (out, o32)
    for k in (SKINNY, TILE256, PAIR):
        assert torch.equal(outs[k][0], outs[TILE128][0]), KNAME[k]
        if outs[k][1] is not None:
            assert torch.equal(outs[k][1], outs[TILE128][1]), KNAME[k]


# ------------------------------------------------------------------------------------------ rejections
def gemm_raw(lib, A, lda, W, ldw, M, N, K, *, res=None, ldr=0, out=None, ldo=0, o32=None, ldo32=0, force_bn=0):
    """opm_gemm with explicit sizes and leading dimensions (the tensors only provide the memory)."""
    return lib.opm_gemm(_p(A), lda, _p(W), ldw, M, N, K, None, _p(res), ldr, 0, ACT_NONE, _p(out), ldo, _p(o32), ldo32, 0, 0, 0,
                        None, None, 0.0, None, 0, None, 0, 0, None, 0, 1, 0, force_bn, _stream())


REJECT = {  # what breaks the base contract of gemm_bf16 (kernels.h GemmArgs)
    "N_not_multiple_of_128": dict(N=192),
    "K_not_multiple_of_8": dict(K=60),
    "K_zero": dict(K=0),
    "K_negative": dict(K=-64),
    "lda_not_multiple_of_8": dict(lda=68),
    "ldw_not_multiple_of_8": dict(ldw=68),
    "ldo_not_multiple_of_8": dict(ldo=260),
    "ldr_not_multiple_of_8": dict(ldr=260),
    "ldo32_not_multiple_of_4": dict(ldo32=258),
    "no_output": dict(no_out=True),
}


def _reject_buffers(M):
    gen = _gen(M + 3)
    A, W = _bf((16, 80), gen), _bf((256, 80), gen)
    res = _bf((16, 264), gen)
    out = torch.full((16, 264), SENT, device="cuda", dtype=torch.bfloat16)
    o32 = torch.full((16, 264), SENT32, device="cuda")
    return A, W, res, out, o32


@pytest.mark.parametrize("force_bn", [0, SKINNY, TILE128, TILE256, PAIR])
@pytest.mark.parametrize("case", list(REJECT))
def test_rejects_broken_contract(lib, case, force_bn):
    """Each returns cudaErrorInvalidValue whichever kernel is asked for, and writes nothing."""
    p = dict(M=16, N=256, K=64, lda=64, ldw=64, ldo=256, ldr=256, ldo32=256, no_out=False)
    p.update(REJECT[case])
    A, W, res, out, o32 = _reject_buffers(p["M"])
    no = p["no_out"]
    rc = gemm_raw(lib, A, p["lda"], W, p["ldw"], p["M"], p["N"], p["K"], res=res, ldr=p["ldr"], out=None if no else out,
                  ldo=p["ldo"], o32=None if no else o32, ldo32=p["ldo32"], force_bn=force_bn)
    assert rc == INVALID, (case, rc)
    torch.cuda.synchronize()
    assert (out == SENT).all() and (o32 == SENT32).all(), case


@pytest.mark.parametrize("force_bn", [0, SKINNY, TILE128, TILE256, PAIR])
@pytest.mark.parametrize("M", [0, -1])
def test_no_rows_is_a_no_op(lib, M, force_bn):
    A, W, res, out, o32 = _reject_buffers(M)
    assert gemm_raw(lib, A, 64, W, 64, M, 256, 64, res=res, ldr=256, out=out, ldo=256, o32=o32, ldo32=256, force_bn=force_bn) == 0
    torch.cuda.synchronize()
    assert (out == SENT).all() and (o32 == SENT32).all()
