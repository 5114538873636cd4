"""Operator tests of the launcher modes the engine's launch sequences use beyond the plain gitb200_op_* subset: the GEMM's row
remap + periodic residual (patch embedding), fp32-only output (vocabulary head), in-place residual, wide leading dimensions,
ReLU, and the skinny kernel's LayerNorm-on-load and K/V scatter (single-clip decode step); the LayerNorm's addend (temporal
embedding), output-row table (multi-stream push), row statistics and grid-stride rows; the decode attention in the layouts of
teacher forcing and of a beam decode step.  The launchers are reached through tests/cuda/op_modes.cpp (op_modes_shim.py).

Every reference is float64 torch on the exact bf16 inputs the kernel read, at the suite's operator tolerances (bf16 output
0.02 + 0.01 |ref|, fp32 output 3e-3 + 2e-3 |ref|, decode attention 0.01 + 0.008 |ref|); where the code promises bit identity
the test asserts torch.equal.  Buffers a kernel writes into only in part are filled with a sentinel first.  Each mode also has
a negative control: a reference with a plausible bug (an off-by-one row, a dropped term, a mask that admits one key too many)
that the kernel's output must FAIL, so the tolerance is shown to see that kind of error.  Measured errors are logged through
test_gpu_parity.record(), with those of the parity tests."""
import importlib
import math

import pytest
import torch

import op_modes_shim
from test_gpu_parity import record

pytestmark = pytest.mark.gpu

BF16_TOL = (0.02, 0.01)
F32_TOL = (3e-3, 2e-3)
TA_TOL = (0.01, 0.008)
SENT = -77.0        # bf16 sentinel (exactly representable)
SENT32 = 12345.0    # fp32 sentinel
INVALID = 1         # cudaErrorInvalidValue
ACT_NONE, ACT_RELU = 0, 3


@pytest.fixture(scope="module")
def lib():
    import gitb200  # noqa: F401  (loads libgitb200.so before the shim that links against it)
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    importlib.import_module("real-time-video-captioning_b200._lib").load()
    return op_modes_shim.load()


def _p(t):
    return None if t is None else t.data_ptr()


def _ld(t):
    return 0 if t is None else t.stride(0)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _bf(shape, gen, scale=1.0, shift=0.0):
    return (torch.randn(*shape, device="cuda", generator=gen) * scale + shift).bfloat16()


def _within(x, ref, tol):
    return bool(((x.double() - ref).abs() <= tol[0] + tol[1] * ref.abs()).all())


def _check(name, x, ref, tol, **meta):
    err = (x.double() - ref).abs()
    record(name, max_err=err.max().item(), **meta)
    bad = err > tol[0] + tol[1] * ref.abs()
    assert not bad.any(), f"{name} {meta}: {int(bad.sum())} elements outside tolerance, max err {err.max().item():.4g}"


def _control(x, wrong, tol, what):
    """Negative control: the kernel's output must fail the tolerance against a reference with a plausible bug."""
    assert not _within(x, wrong, tol), f"negative control passed: the tolerance cannot see {what}"


def gemm(lib, A, W, *, bias=None, res=None, periodic=0, act=ACT_NONE, out=None, o32=None, remap=(0, 0, 0), lnl=None, sc=None,
         force_bn=0):
    """gemm_bf16 on torch tensors: leading dimensions are the tensors' row strides.  lnl = (gamma, beta, eps, lnl_out or None),
    sc = (kv, q_width, kv_width, pos or None, pos_const, slot_div, n_slots)."""
    g, b, eps, lo = lnl if lnl is not None else (None, None, 0.0, None)
    kv, qw, kvw, pos, pc, sd, ns = sc if sc is not None else (None, 0, 0, None, 0, 1, 0)
    return lib.opm_gemm(_p(A), _ld(A), _p(W), _ld(W), A.shape[0], W.shape[0], A.shape[1], _p(bias), _p(res), _ld(res), periodic, act,
                        _p(out), _ld(out), _p(o32), _ld(o32), *remap, _p(g), _p(b), eps, _p(lo), _ld(lo), _p(kv), qw, kvw, _p(pos), pc,
                        sd, ns, force_bn, _stream())


def layernorm(lib, x, gamma, beta, eps, *, out=None, o32=None, addend=None, add_group=1, add_period=1, stats=None, stats_slots=1,
              row_base=None, out_group=0, cols=None):
    return lib.opm_layernorm(_p(x), _ld(x), x.shape[0], x.shape[1] if cols is None else cols, _p(gamma), _p(beta), eps, _p(addend),
                             add_group, add_period, _p(out), _ld(out), _p(o32), _ld(o32), _p(stats), stats_slots, _p(row_base),
                             out_group, _stream())


def ref_gemm(A, W, bias=None, res=None, act=ACT_NONE):
    r = A.double() @ W.double().t()
    if bias is not None:
        r = r + bias.double()
    if act == ACT_RELU:
        r = r.clamp_min(0)
    if res is not None:
        r = r + res.double()
    return r


def ref_layernorm(x, gamma, beta, eps):
    x = x.double()
    mean = x.mean(-1, keepdim=True)
    var = ((x - mean) ** 2).mean(-1, keepdim=True)
    return (x - mean) / torch.sqrt(var + eps) * gamma.double() + beta.double()


def _weights(gen, N, K, with_bias=True):
    w = _bf((N, K), gen, K ** -0.5)
    bias = torch.randn(N, device="cuda", generator=gen) if with_bias else None
    return w, bias


# ------------------------------------------------------------------------------------------ GEMM
@pytest.mark.parametrize("force_bn", [128, 256])
@pytest.mark.parametrize("n_frames", [1, 6, 7])
@pytest.mark.parametrize("K,kreal,gin,gout,N", [(768, 768, 196, 197, 768), (640, 588, 256, 257, 1024)])
def test_patch_embedding_remap_and_periodic_residual(lib, K, kreal, gin, gout, N, n_frames, force_bn):
    """ViT patch embedding (api.cu encode): patch row r lands in output row (r / gin) * gout + r % gin + 1 and adds positional
    row r % gin + 1; the CLS row of every frame is not written.  ViT-L's K 588 is zero-padded to 640 in A and W."""
    gen = _gen(K + n_frames + force_bn)
    A = _bf((n_frames * gin, K), gen, 0.5)
    w, _ = _weights(gen, N, K, with_bias=False)
    A[:, kreal:] = 0
    w[:, kreal:] = 0
    pos = _bf((gout, N), gen, 0.5)
    out = torch.full((n_frames * gout, N), SENT, device="cuda", dtype=torch.bfloat16)
    assert gemm(lib, A, w, res=pos, periodic=1, out=out, remap=(gin, gout, 1), force_bn=force_bn) == 0
    core = ref_gemm(A, w).view(n_frames, gin, N)
    ref = core + pos[1:].double()
    got = out.view(n_frames, gout, N)
    assert (got[:, 0] == SENT).all(), "a CLS row was written"
    _check("op_modes_patch_embed", got[:, 1:], ref, BF16_TOL, K=K, frames=n_frames, bn=force_bn)
    _control(got[:, 1:], core + pos[:gin].double(), BF16_TOL, "a positional row off by one")


@pytest.mark.parametrize("M", [1, 4, 8, 9, 127, 129, 1023])
def test_fp32_only_output_vocabulary_head(lib, M):
    """Vocabulary head (out == nullptr, out_f32 only), N 30720 K 768: skinny kernel for M <= 8, 1-CTA kernel above.  The row
    after the last one keeps its sentinel."""
    N, K = 30720, 768
    gen = _gen(M)
    A = _bf((M, K), gen, 1.0)
    w, bias = _weights(gen, N, K)
    buf = torch.full((M + 1, N), SENT32, device="cuda")
    assert gemm(lib, A, w, bias=bias, o32=buf[:M]) == 0
    ref = ref_gemm(A, w, bias)
    assert (buf[M] == SENT32).all(), "a row past M was written"
    _check("op_modes_f32_only", buf[:M], ref, F32_TOL, M=M)
    _control(buf[:M], ref - bias.double(), F32_TOL, "a dropped bias")


@pytest.mark.parametrize("M,K,force_bn,kernel", [(4, 768, 0, "skinny"), (4, 3072, 0, "skinny split-K"), (300, 768, 0, "1-CTA"),
                                                 (2364, 768, 2, "CTA pair"), (2364, 3072, 2, "CTA pair")])
def test_in_place_residual_is_bit_identical(lib, M, K, force_bn, kernel):
    """out == residual (every residual GEMM of the ViT and the decoder) equals the same GEMM with a separate residual copy,
    bit for bit, on each kernel."""
    N = 768
    gen = _gen(M + K)
    A = _bf((M, K), gen, 0.5)
    w, bias = _weights(gen, N, K)
    x = _bf((M, N), gen, 2.0)
    sep = torch.empty_like(x)
    assert gemm(lib, A, w, bias=bias, res=x.clone(), out=sep, force_bn=force_bn) == 0
    ref = ref_gemm(A, w, bias, x)
    x0 = x.clone()
    assert gemm(lib, A, w, bias=bias, res=x, out=x, force_bn=force_bn) == 0
    assert torch.equal(x, sep), kernel
    _check("op_modes_in_place", x, ref, BF16_TOL, M=M, K=K, kernel=kernel)
    _control(x, ref - x0.double(), BF16_TOL, "a dropped residual")


@pytest.mark.parametrize("M,force_bn,kernel", [(3, 0, "skinny"), (300, 0, "1-CTA"), (2364, 2, "CTA pair")])
def test_wide_leading_dimensions(lib, M, force_bn, kernel):
    """lda > K, ldo > N, ldr > N (and ldo32 > N where the kernel has an fp32 output): the gap columns keep their sentinel."""
    N, K = 768, 768
    gen = _gen(M + 5)
    Abuf = _bf((M, K + 64), gen, 0.5)  # random gap: a kernel that read it as contiguous rows would see other values
    A = Abuf[:, :K]
    w, bias = _weights(gen, N, K)
    rbuf = _bf((M, N + 64), gen, 1.0)
    res = rbuf[:, :N]
    obuf = torch.full((M, N + 128), SENT, device="cuda", dtype=torch.bfloat16)
    o32buf = torch.full((M, N + 4), SENT32, device="cuda") if kernel != "CTA pair" else None
    o32 = o32buf[:, :N] if o32buf is not None else None
    assert gemm(lib, A, w, bias=bias, res=res, out=obuf[:, :N], o32=o32, force_bn=force_bn) == 0
    ref = ref_gemm(A, w, bias, res)
    assert (obuf[:, N:] == SENT).all(), "bf16 gap columns written"
    _check("op_modes_strides", obuf[:, :N], ref, BF16_TOL, M=M, kernel=kernel)
    if o32 is not None:
        assert (o32buf[:, N:] == SENT32).all(), "fp32 gap columns written"
        _check("op_modes_strides_f32", o32, ref, F32_TOL, M=M, kernel=kernel)
    wrong = ref_gemm(Abuf.flatten()[:M * K].view(M, K), w, bias, res)
    _control(obuf[:, :N], wrong, BF16_TOL, "A read with lda = K")


@pytest.mark.parametrize("M,N,K,force_bn,kernel", [(4, 640, 256, 0, "skinny"), (300, 640, 256, 0, "1-CTA"), (2364, 640, 256, 0, "1-CTA"),
                                                   (2364, 768, 768, 2, "CTA pair")])
def test_relu_epilogue(lib, M, N, K, force_bn, kernel):
    """ACT_RELU (student FFN, N = 576 padded to 640) on every kernel."""
    gen = _gen(M + N)
    A = _bf((M, K), gen, 1.0)
    w, bias = _weights(gen, N, K)
    out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    assert gemm(lib, A, w, bias=bias, act=ACT_RELU, out=out, force_bn=force_bn) == 0
    _check("op_modes_relu", out, ref_gemm(A, w, bias, act=ACT_RELU), BF16_TOL, M=M, N=N, kernel=kernel)
    _control(out, ref_gemm(A, w, bias), BF16_TOL, "a missing ReLU")


def _ln_params(gen, cols):
    return 1 + 0.1 * torch.randn(cols, device="cuda", generator=gen), 0.1 * torch.randn(cols, device="cuda", generator=gen)


@pytest.mark.parametrize("N", [2304, 3072, 30720])
@pytest.mark.parametrize("M", [1, 2, 3, 4])
def test_skinny_layernorm_on_load(lib, M, N):
    """The decode step's LayerNorm inside the skinny GEMM (K 768): lnl_out == layernorm_bf16 of the same rows bit for bit (the
    kernel's stated contract), the output == the plain skinny GEMM on those normalised rows bit for bit, and both within
    tolerance of fp64 LayerNorm -> GEMM.  N 30720 is the vocabulary head: fp32 output only, no lnl_out."""
    K, eps = 768, 1e-12
    gen = _gen(M * 7 + N)
    x = _bf((M, K), gen, 3.0, 1.0)
    gamma, beta = _ln_params(gen, K)
    w, bias = _weights(gen, N, K)
    vocab = N == 30720
    lnl_out = None if vocab else torch.full((M + 1, K), SENT, device="cuda", dtype=torch.bfloat16)
    out = None if vocab else torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    o32 = torch.empty(M, N, device="cuda")
    lo = None if vocab else lnl_out[:M]
    assert gemm(lib, x, w, bias=bias, out=out, o32=o32, lnl=(gamma, beta, eps, lo)) == 0
    xn = torch.empty(M, K, device="cuda", dtype=torch.bfloat16)
    assert layernorm(lib, x, gamma, beta, eps, out=xn) == 0
    plain = None if vocab else torch.empty_like(out)
    plain32 = torch.empty_like(o32)
    assert gemm(lib, xn, w, bias=bias, out=plain, o32=plain32) == 0
    ref_ln = ref_layernorm(x, gamma, beta, eps)
    ref = ref_gemm(ref_ln.bfloat16(), w, bias)   # the kernel rounds the normalised rows to bf16 before its dot products
    if not vocab:
        assert (lnl_out[M] == SENT).all(), "lnl_out row past M written"
        assert torch.equal(lnl_out[:M], xn), "LayerNorm-on-load rows differ from layernorm_bf16"
        _check("op_modes_lnl_rows", lnl_out[:M], ref_ln, BF16_TOL, M=M)
        assert torch.equal(out, plain)
        _check("op_modes_lnl_gemm", out, ref, BF16_TOL, M=M, N=N)
    assert torch.equal(o32, plain32)
    _check("op_modes_lnl_gemm_f32", o32, ref, F32_TOL, M=M, N=N)
    _control(o32, ref_gemm(ref_layernorm(x, gamma, torch.zeros_like(beta), eps).bfloat16(), w, bias), F32_TOL, "a dropped beta")


@pytest.mark.parametrize("with_lnl", [False, True])
@pytest.mark.parametrize("pos_array", [False, True])
@pytest.mark.parametrize("M", [1, 2, 3, 4])
def test_skinny_kv_scatter(lib, M, pos_array, with_lnl):
    """The QKV projection of a decode step also scatters its K|V columns into the text K/V plane (store_text_kv fused):
    the plane equals store_text_kv of the GEMM's own output bit for bit, every other slot keeps its sentinel."""
    K, N, qw, kvw, max_pos = 768, 2304, 768, 1536, 8
    gen = _gen(M * 3 + pos_array + 2 * with_lnl)
    x = _bf((M, K), gen, 3.0 if with_lnl else 0.5, 1.0 if with_lnl else 0.0)
    gamma, beta = _ln_params(gen, K)
    w, bias = _weights(gen, N, K)
    pos = torch.tensor([3, 0, 7, 2][:M], device="cuda", dtype=torch.int32) if pos_array else None
    plane = torch.full((max_pos, M, kvw), SENT, device="cuda", dtype=torch.bfloat16)
    out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    lnl = (gamma, beta, 1e-12, torch.empty(M, K, device="cuda", dtype=torch.bfloat16)) if with_lnl else None
    assert gemm(lib, x, w, bias=bias, out=out, lnl=lnl, sc=(plane, qw, kvw, pos, 5, 1, M)) == 0
    expect = torch.full_like(plane, SENT)
    assert lib.opm_store_text_kv(_p(out), N, M, kvw, qw, _p(pos), 5, 1, M, _p(expect), _stream()) == 0
    assert torch.equal(plane, expect)
    assert int((plane != SENT).sum()) > 0.99 * M * kvw
    xin = ref_layernorm(x, gamma, beta, 1e-12).bfloat16() if with_lnl else x
    _check("op_modes_kv_scatter", out, ref_gemm(xin, w, bias), BF16_TOL, M=M, lnl=with_lnl)
    shifted = torch.full_like(plane, SENT)
    pos1 = (pos + 1) % max_pos if pos is not None else None
    assert lib.opm_store_text_kv(_p(out), N, M, kvw, qw, _p(pos1), 6, 1, M, _p(shifted), _stream()) == 0
    assert not torch.equal(plane, shifted), "negative control: a position off by one leaves the same plane"


@pytest.mark.parametrize("case", ["lnl_M9", "sc_M9", "lnl_M9_skinny_forced", "sc_M9_skinny_forced", "lnl_tile128", "sc_tile256",
                                  "lnl_K1024", "lnl_M5", "lnl_M8"])
def test_skinny_fusions_reject_unsupported_shapes(lib, case):
    """LayerNorm-on-load / K-V scatter exist only in the skinny kernel (M <= 8; the LayerNorm also needs K == 768, M <= 4): every
    other request returns cudaErrorInvalidValue and writes nothing -- never a tensor-core GEMM without the fusion."""
    M = int(case.split("_M")[1].split("_")[0]) if "_M" in case else 4
    K = 1024 if case == "lnl_K1024" else 768
    force_bn = {"tile128": 128, "tile256": 256, "forced": 1}.get(case.split("_")[-1], 0)
    N = 2304
    gen = _gen(len(case))
    x = _bf((M, K), gen)
    w, bias = _weights(gen, N, K)
    gamma, beta = _ln_params(gen, K)
    out = torch.full((M, N), SENT, device="cuda", dtype=torch.bfloat16)
    lnl_out = torch.full((M, K), SENT, device="cuda", dtype=torch.bfloat16)
    plane = torch.full((4, M, 1536), SENT, device="cuda", dtype=torch.bfloat16)
    lnl = (gamma, beta, 1e-12, lnl_out) if case.startswith("lnl") else None
    sc = (plane, 768, 1536, None, 0, 1, M) if case.startswith("sc") else None
    assert gemm(lib, x, w, bias=bias, out=out, lnl=lnl, sc=sc, force_bn=force_bn) == INVALID, case
    torch.cuda.synchronize()
    assert (out == SENT).all() and (lnl_out == SENT).all() and (plane == SENT).all(), case


# ------------------------------------------------------------------------------------------ LayerNorm
@pytest.mark.parametrize("cols", [768, 1024])
@pytest.mark.parametrize("rows", [3551, 3552, 3553, 7105, 9456])
def test_layernorm_grid_stride_rows(lib, rows, cols):
    """More rows than the persistent grid's 444 CTAs x 8 warps = 3552: the grid-stride loop and its next-row prefetch."""
    gen = _gen(rows + cols)
    x = _bf((rows, cols), gen, 3.0, 1.0)
    gamma, beta = _ln_params(gen, cols)
    eps = 1e-5 if cols == 1024 else 1e-12
    buf = torch.full((rows + 1, cols), SENT, device="cuda", dtype=torch.bfloat16)
    assert layernorm(lib, x, gamma, beta, eps, out=buf[:rows]) == 0
    ref = ref_layernorm(x, gamma, beta, eps)
    assert (buf[rows] == SENT).all()
    _check("op_modes_ln_rows", buf[:rows], ref, BF16_TOL, rows=rows, cols=cols)
    if rows > 3552:  # a prefetch bug: the second pass re-normalises the first pass's row
        wrong = ref.clone()
        wrong[3552:] = ref[torch.arange(3552, rows, device="cuda") % 3552]
        _control(buf[:rows], wrong, BF16_TOL, "a grid-stride row taken from the previous pass")


@pytest.mark.parametrize("cols", [768, 1024])
def test_layernorm_wide_leading_dimensions(lib, cols):
    rows = 1000
    gen = _gen(cols + 1)
    xbuf = _bf((rows, cols + 64), gen, 3.0, 1.0)
    gamma, beta = _ln_params(gen, cols)
    obuf = torch.full((rows, cols + 128), SENT, device="cuda", dtype=torch.bfloat16)
    assert layernorm(lib, xbuf[:, :cols], gamma, beta, 1e-5, out=obuf[:, :cols]) == 0
    assert (obuf[:, cols:] == SENT).all()
    _check("op_modes_ln_strides", obuf[:, :cols], ref_layernorm(xbuf[:, :cols], gamma, beta, 1e-5), BF16_TOL, cols=cols)
    wrong = ref_layernorm(xbuf.flatten()[:rows * cols].view(rows, cols), gamma, beta, 1e-5)
    _control(obuf[:, :cols], wrong, BF16_TOL, "x read with ldx = cols")


@pytest.mark.parametrize("F", [1, 2, 6])
@pytest.mark.parametrize("T,cols", [(197, 768), (257, 1024)])
def test_layernorm_temporal_addend(lib, T, cols, F):
    """ln_post + temporal embedding over 2 clips of F frames: row r adds addend[(r / T) % F] (the period wraps at the clip
    boundary); bf16 and fp32 outputs."""
    rows = 2 * F * T
    gen = _gen(T + F)
    x = _bf((rows, cols), gen, 3.0, 1.0)
    gamma, beta = _ln_params(gen, cols)
    temporal = 0.5 * torch.randn(F, cols, device="cuda", generator=gen)
    out = torch.empty(rows, cols, device="cuda", dtype=torch.bfloat16)
    o32 = torch.empty(rows, cols, device="cuda")
    assert layernorm(lib, x, gamma, beta, 1e-5, out=out, o32=o32, addend=temporal, add_group=T, add_period=F) == 0
    ln = ref_layernorm(x, gamma, beta, 1e-5)
    r = torch.arange(rows, device="cuda")
    ref = ln + temporal.double()[(r // T) % F]
    _check("op_modes_ln_addend", out, ref, BF16_TOL, T=T, F=F)
    _check("op_modes_ln_addend_f32", o32, ref, F32_TOL, T=T, F=F)
    if F > 1:
        _control(o32, ln + temporal.double()[r % F], F32_TOL, "the temporal row taken from row % F")
    else:
        _control(o32, ln, F32_TOL, "a dropped addend")


@pytest.mark.parametrize("T,cols", [(197, 768), (257, 1024)])
def test_layernorm_output_row_table(lib, T, cols):
    """Multi-stream push: frame g's T rows go to output rows out_row_base[g] + 0.. (non-contiguous ring slots); mapped rows equal
    the plain kernel's rows bit for bit and every other ring row keeps its sentinel."""
    slots = [7, 2, 9, 4]
    k, cap = len(slots), 10
    gen = _gen(T)
    x = _bf((k * T, cols), gen, 3.0, 1.0)
    gamma, beta = _ln_params(gen, cols)
    base = torch.tensor(slots, device="cuda", dtype=torch.int32) * T
    ring = torch.full((cap * T, cols), SENT, device="cuda", dtype=torch.bfloat16)
    assert layernorm(lib, x, gamma, beta, 1e-5, out=ring, row_base=base, out_group=T) == 0
    plain = torch.empty(k * T, cols, device="cuda", dtype=torch.bfloat16)
    assert layernorm(lib, x, gamma, beta, 1e-5, out=plain) == 0
    ring_v = ring.view(cap, T, cols)
    assert torch.equal(ring_v[slots], plain.view(k, T, cols))
    free = [s for s in range(cap) if s not in slots]
    assert (ring_v[free] == SENT).all()
    _check("op_modes_ln_row_table", ring_v[slots], ref_layernorm(x, gamma, beta, 1e-5).view(k, T, cols), BF16_TOL, cols=cols)
    assert layernorm(lib, x, gamma, beta, 1e-5, out=ring, row_base=base, out_group=0) == INVALID
    rotated = plain.view(k, T, cols)[[1, 2, 3, 0]]
    assert not torch.equal(ring_v[slots], rotated), "negative control: frames written to rotated slots look the same"


@pytest.mark.parametrize("cols", [768, 1024])
def test_layernorm_row_statistics(lib, cols):
    """stats_out: slot 0 holds (sum, sum of squares) of the bf16-rounded output row, the other slots exactly 0."""
    rows, n_slots = 4000, 2 * cols // 256
    gen = _gen(cols + 3)
    x = _bf((rows, cols), gen, 3.0, 1.0)
    gamma, beta = _ln_params(gen, cols)
    out = torch.empty(rows, cols, device="cuda", dtype=torch.bfloat16)
    stats = torch.full((rows, n_slots, 2), SENT32, device="cuda")
    assert layernorm(lib, x, gamma, beta, 1e-5, out=out, stats=stats, stats_slots=n_slots) == 0
    o = out.double()
    ref = torch.stack([o.sum(-1), (o * o).sum(-1)], -1)
    scale = torch.stack([o.abs().sum(-1), (o * o).sum(-1)], -1)
    err = (stats[:, 0].double() - ref).abs()
    record("op_modes_ln_stats", cols=cols, max_rel_err=(err / scale).max().item())
    assert (err <= 2e-5 * scale + 1e-6).all(), (err / scale).max()
    assert (stats[:, 1:] == 0).all()
    ln = ref_layernorm(x, gamma, beta, 1e-5)
    unrounded = torch.stack([ln.sum(-1), (ln * ln).sum(-1)], -1)
    assert ((stats[:, 0].double() - unrounded).abs() > 2e-5 * scale + 1e-6).any(), \
        "negative control: statistics of the unrounded row pass as well"


@pytest.mark.parametrize("cols", [576, 512])
def test_layernorm_rejects_other_widths(lib, cols):
    gen = _gen(cols)
    x = _bf((8, cols), gen)
    gamma, beta = _ln_params(gen, cols)
    out = torch.full((8, cols), SENT, device="cuda", dtype=torch.bfloat16)
    assert layernorm(lib, x, gamma, beta, 1e-5, out=out) == INVALID
    torch.cuda.synchronize()
    assert (out == SENT).all()


# ------------------------------------------------------------------------------------------ decode attention
def ref_text_attention(q, vis_k, vis_v, txt_k, txt_v, mask, n_clips, rpc, heads, scale):
    """fp64 masked softmax: row r attends to the Nv visual keys of clip r / rpc and to its own text keys txt_k[r, s] where
    mask[r, s].  q [rows, W]; vis_k / vis_v [n_clips, Nv, W]; txt_k / txt_v [rows, S, W]; mask [rows, S] bool."""
    rows, W = q.shape
    Nv, S = vis_k.shape[1], txt_k.shape[1]
    qh = q.double().view(rows, heads, 64)
    s_vis = torch.einsum("crhd,cnhd->crhn", qh.view(n_clips, rpc, heads, 64), vis_k.double().view(n_clips, Nv, heads, 64))
    s_txt = torch.einsum("rhd,rshd->rhs", qh, txt_k.double().view(rows, S, heads, 64))
    s_txt = s_txt.masked_fill(~mask[:, None, :], -math.inf)
    p = torch.softmax(torch.cat([s_vis.reshape(rows, heads, Nv), s_txt], -1) * scale, -1)
    o = torch.einsum("crhn,cnhd->crhd", p[..., :Nv].reshape(n_clips, rpc, heads, Nv), vis_v.double().view(n_clips, Nv, heads, 64))
    o = o.reshape(rows, heads, 64) + torch.einsum("rhs,rshd->rhd", p[..., Nv:], txt_v.double().view(rows, S, heads, 64))
    return o.reshape(rows, W)


def _text_attention(lib, q, vis, Nv, n_clips, rpc, heads, txt, txt_slots, slot_is_clip, anc, anc_ld, n_text, n_text_const,
                    max_text, splits):
    W, rows = heads * 64, n_clips * rpc
    out = torch.empty(rows, W, device="cuda", dtype=torch.bfloat16)
    partial = None
    if splits > 1:
        partial = torch.empty(lib.opm_text_attention_workspace_floats(rows, heads, splits), device="cuda")
    rc = lib.opm_text_attention(_p(q), _ld(q), n_clips, rpc, heads, _p(vis), _ld(vis), W, 2 * W, Nv, _p(txt), txt_slots, slot_is_clip,
                                _p(anc), anc_ld, _p(n_text), n_text_const, max_text, 0.125, _p(out), W, _p(partial), splits, _stream())
    assert rc == 0
    return out


@pytest.mark.parametrize("splits", [1, 3])
@pytest.mark.parametrize("Nv", [197, 1182])
@pytest.mark.parametrize("L", [1, 3, 7, 20, 33])
def test_teacher_forced_text_attention(lib, L, Nv, splits):
    """gitb200_forward_logits' layout: visual K|V inside the [B * Nv, 3W] QKV rows (k_off W, v_off 2W, ld 3W), queries in the
    [B * L, 3W] rows, text plane [L][B][2W] with one slot per clip, per-row n_text = p + 1.  The text keys are scaled so they
    carry a real share of the softmax mass: a mask that admitted key p + 1 would move the output far outside the tolerance."""
    B, heads = 2, 12
    W, rows = heads * 64, B * L
    gen = _gen(L * 100 + Nv + splits)
    vis = _bf((B * Nv, 3 * W), gen)
    q = _bf((rows, 3 * W), gen, 1.0)
    txt = torch.randn(L, B, 2 * W, device="cuda", generator=gen)
    txt[..., :W] *= 4
    txt = txt.bfloat16()
    p = torch.arange(rows, device="cuda") % L
    n_text = (p + 1).int()
    out = _text_attention(lib, q, vis, Nv, B, L, heads, txt, B, 1, None, L, n_text, 0, L, splits)
    vk, vv = vis.view(B, Nv, 3 * W)[..., W:2 * W], vis.view(B, Nv, 3 * W)[..., 2 * W:]
    per_row = txt.permute(1, 0, 2)[torch.arange(rows, device="cuda") // L]   # [rows, L, 2W]: the row's clip slot
    s = torch.arange(L, device="cuda")[None, :]
    args = (q[:, :W], vk, vv, per_row[..., :W], per_row[..., W:])
    ref = ref_text_attention(*args, s <= p[:, None], B, L, heads, 0.125)
    _check("op_modes_text_attn_teacher", out, ref, TA_TOL, L=L, Nv=Nv, splits=splits)
    if L > 1:
        _control(out, ref_text_attention(*args, s <= p[:, None] + 1, B, L, heads, 0.125), TA_TOL, "a causal mask admitting p + 1")
    _control(out, ref_text_attention(*args, s < p[:, None], B, L, heads, 0.125), TA_TOL, "a row missing its own text key")


@pytest.mark.parametrize("rpc", [1, 2, 3, 4, 8])
def test_decode_step_text_attention(lib, rpc):
    """run_text_pass' beam step: anc_ld = max_text = max_len (20) > n_text_const (6), ancestor table with the row's own slot at
    the last position, one plane slot per row; the plane positions >= n_text and the unused ancestor entries hold values
    that would show if they were read."""
    n_clips, heads, Nv, max_len, nt = 3, 12, 1182, 20, 6
    W, rows = heads * 64, n_clips * rpc
    chunks = (rpc + 3) // 4
    splits = min(16, -(-2 * 148 // (n_clips * chunks * heads)))
    while splits > 1 and Nv // splits < 64:
        splits -= 1
    gen = _gen(rpc + 1000)
    vis = _bf((n_clips * Nv, 3 * W), gen)
    q = _bf((rows, 3 * W), gen, 1.0)
    txt = torch.randn(max_len, rows, 2 * W, device="cuda", generator=gen)
    txt[..., :W] *= 4
    txt = txt.bfloat16()
    r = torch.arange(rows, device="cuda")
    base = (r // rpc) * rpc
    anc = (base[:, None] + torch.randint(0, rpc, (rows, max_len), device="cuda", generator=gen)).int()
    anc[:, nt - 1:] = ((r + 1) % rows).int()[:, None]   # never read: a valid but wrong slot
    out = _text_attention(lib, q, vis, Nv, n_clips, rpc, heads, txt, rows, 0, anc, max_len, None, nt, max_len, splits)
    vk, vv = vis.view(n_clips, Nv, 3 * W)[..., W:2 * W], vis.view(n_clips, Nv, 3 * W)[..., 2 * W:]

    def ref_with(slots, n):
        kv = txt[torch.arange(n, device="cuda")[None, :], slots[:, :n].long()]   # [rows, n, 2W]
        return ref_text_attention(q[:, :W], vk, vv, kv[..., :W], kv[..., W:], torch.ones(rows, n, dtype=torch.bool, device="cuda"),
                                  n_clips, rpc, heads, 0.125)
    slots = anc.clone()
    slots[:, nt - 1] = r.int()
    ref = ref_with(slots, nt)
    _check("op_modes_text_attn_step", out, ref, TA_TOL, rpc=rpc, splits=splits)
    own = r.int()[:, None].expand(rows, max_len)
    _control(out, ref_with(torch.cat([slots[:, :nt], own[:, nt:]], 1), nt + 1), TA_TOL, "one text position past n_text")
    if rpc > 1:
        _control(out, ref_with(own, nt), TA_TOL, "the ancestor table ignored")
