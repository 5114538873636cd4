"""Operator tests of the group attention (op_attention_groups: attention_groups_tc, the tcgen05 kernel; legacy_mma=True:
the mma.sync kernel of attention.cu) against the float64 reference and per-element error bound of attention_groups_ref.py.
Both kernels must meet the bound; they are not expected to agree bit for bit.

  * every geometry the engine launches (api.cu: the ViT's attention over frames of T tokens, one group per frame; the
    decoder's visual block over a clip's Nv = frames x T visual rows, one group per clip) at the bench's 512 clips, with the
    sub-batch sizes sweep_clips() gives, plus the test configs' one- and two-frame clips;
  * every residue of len mod 16 on both templates of the tcgen05 kernel (193-208 and 1537-1552 keys) with poisoned-neighbour
    inputs, where a key leaked from the next group or from the zero fill past the last row dominates its row;
  * lengths with no tail block (multiples of 64), the LONG_GROUP boundary, a one-key group, and the single-item last pair
    that only an odd number of items reaches;
  * bit identity: run to run, and a group alone against the same group inside the batch (start, middle, end);
  * reads and writes: qkv as a row range of a larger buffer whose other rows hold NaN, output into a row range of a buffer
    holding a sentinel;
  * ramped key norms, so that the tcgen05 kernel's running max moves (and O is rescaled in tensor memory) on most blocks.

Every test on poisoned inputs also checks that the kernel's output fails the bound against the reference of a mask off by
one key either way (attention_groups_ref.attention(extra=+1 / -1)).  Max error / bound per case goes through
test_gpu_parity.record()."""
import importlib
import zlib

import pytest
import torch

import attention_groups_ref as ar
from test_gpu_parity import record

pytestmark = pytest.mark.gpu

KERNELS = {False: "tcgen05", True: "mma_sync"}
SWEEP_ROWS = 151296   # gitb200_ctx::sweep_rows default (api.cu)
BENCH_CLIPS = 512
SENTINEL = -768.0     # exact in bf16, far from any attention output here


def sweep_clips(sweep_rows, rows_per_clip, n_clips):
    """api.cu sweep_clips: clips per sub-batch of a sweep, at most sweep_rows rows, sub-batches balanced."""
    if sweep_rows <= 0 or n_clips <= 1:
        return n_clips
    sub = max(1, sweep_rows // rows_per_clip)
    if sub >= n_clips:
        return n_clips
    n_sub = -(-n_clips // sub)
    return -(-n_clips // n_sub)


def engine_geometry():
    """(n_groups, group_len, heads) of every attention_groups_tc launch of a 512-clip batch: the ViT (api.cu run_encode,
    n_clips * F groups of T rows, vit_heads) and the decoder's visual block (run_visual_pass, B groups of Nv rows, dec_heads),
    for each sub-batch size of run_encode_sweeps / run_visual_pass (both sweep over F * T rows per clip)."""
    models = {"base": (197, 12, 12), "large": (257, 16, 12)}   # T, vit_heads, dec_heads: ViT-B/16 and ViT-L/14 at 224^2
    cases = {(3, 197, 12), (3, 394, 12)}                      # the test configs' one- and two-frame clips
    for model, frames, sweep_rows in (("base", 6, SWEEP_ROWS), ("base", 6, 0), ("large", 6, SWEEP_ROWS), ("large", 24, SWEEP_ROWS)):
        T, vit_heads, dec_heads = models[model]
        sub = sweep_clips(sweep_rows, frames * T, BENCH_CLIPS)
        for clips in {min(sub, BENCH_CLIPS - d) for d in range(0, BENCH_CLIPS, sub)}:
            cases.add((clips * frames, T, vit_heads))
            cases.add((clips, frames * T, dec_heads))
    return sorted(cases, key=lambda c: (c[1], c[0]))


@pytest.fixture(scope="module")
def eng():
    import gitb200  # noqa: F401  (builds / loads the library)
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return importlib.import_module("real-time-video-captioning_b200.engine")


def _gen(*key):
    return torch.Generator(device="cuda").manual_seed(zlib.crc32(repr(key).encode()))


def _run(eng, qkv, n_groups, group_len, heads, legacy=False, out=None):
    return eng.op_attention_groups(qkv, n_groups, group_len, heads, ar.SCALE, legacy_mma=legacy, out=out)


def _check(test, out, ref, bound, legacy, **meta):
    ratio = ar.max_ratio(out, ref, bound)
    bad = ar.violations(out, ref, bound)
    record("attention_groups_" + test, kernel=KERNELS[legacy], max_err_over_bound=ratio,
           max_err=(out.double() - ref).abs().max().item(), **meta)
    assert bad == 0, f"{KERNELS[legacy]} {meta}: {bad} elements outside the bound, max err / bound {ratio:.4g}"


def _mask_controls(out, qkv, n_groups, group_len, heads, bound):
    """The kernel's output against the references of a mask that lets in the next key / drops the last one: both must fail
    the bound, or the poisoned inputs could not have shown such a bug."""
    for extra in (1, -1) if group_len > 1 else (1,):
        wrong, _ = ar.attention(qkv, n_groups, group_len, heads, extra=extra, with_bound=False)
        assert ar.violations(out, wrong, bound) > 0, f"negative control passed: the bound cannot see a mask off by {extra:+d}"


def _batch_invariant(eng, qkv, out, n_groups, group_len, heads):
    """Groups from the start, the middle and the end of the batch, run alone, give the batch's bits."""
    for gi in sorted({0, n_groups // 2, n_groups - 1}):
        rows = slice(gi * group_len, (gi + 1) * group_len)
        alone = _run(eng, qkv[rows], 1, group_len, heads)
        assert torch.equal(alone, out[rows]), f"group {gi} of {n_groups} differs from the same group run alone"


def _straddling_pairs(n_groups, group_len, heads):
    """Pairs of work items (item = (group, head, 128-query tile)) whose two items belong to different (group, head): the
    tcgen05 kernel loads separate K / V tiles for them while the other pairs of long groups share theirs."""
    n_qt = -(-group_len // 128)
    n_items = n_qt * heads * n_groups
    return sum(1 for p in range(n_items // 2) if (2 * p) // n_qt != (2 * p + 1) // n_qt)


# ------------------------------------------------------------------------------------------ engine geometry
@pytest.mark.parametrize("n_groups,group_len,heads", engine_geometry())
def test_engine_geometry(eng, n_groups, group_len, heads):
    """Both kernels within the bound at the engine's launch geometry; the tcgen05 kernel bit-identical run to run and across
    batch positions.  At 1542 and 6168 keys the tile count per head is odd (13, 49), so pairs straddle head boundaries and
    every CTA walks 8 to 24 pairs that alternate between shared and separate K / V tiles."""
    qkv = ar.randn_qkv(n_groups, group_len, heads, _gen(n_groups, group_len, heads), "cuda")
    ref, bound = ar.attention(qkv, n_groups, group_len, heads)
    for legacy in (False, True):
        out = _run(eng, qkv, n_groups, group_len, heads, legacy)
        _check("engine_geometry", out, ref, bound, legacy, n_groups=n_groups, group_len=group_len, heads=heads)
    del ref, bound
    out = _run(eng, qkv, n_groups, group_len, heads)
    assert torch.equal(out, _run(eng, qkv, n_groups, group_len, heads))
    if group_len in (1542, 6168):
        assert _straddling_pairs(1, group_len, heads) > 0
    _batch_invariant(eng, qkv, out, n_groups, group_len, heads)


# ------------------------------------------------------------------------------------------ masks and edges
@pytest.mark.parametrize("legacy", [False, True], ids=["tcgen05", "mma_sync"])
@pytest.mark.parametrize("group_len", list(range(193, 209)) + list(range(1537, 1553)))
def test_mask_width(eng, group_len, legacy):
    """Every residue of len mod 16 (the tcgen05 tail block issues only the 16-key steps holding valid keys) on the short and
    the long template: three poisoned groups, so the middle one has neighbours on both sides and the last one's tail is the
    TMA zero fill."""
    n_groups, heads = 3, 12
    qkv = ar.poisoned_qkv(n_groups, group_len, heads, _gen("mask", group_len), "cuda")
    ref, bound = ar.attention(qkv, n_groups, group_len, heads)
    out = _run(eng, qkv, n_groups, group_len, heads, legacy)
    _check("mask_width", out, ref, bound, legacy, group_len=group_len)
    _mask_controls(out, qkv, n_groups, group_len, heads, bound)


@pytest.mark.parametrize("legacy", [False, True], ids=["tcgen05", "mma_sync"])
@pytest.mark.parametrize("n_groups,group_len,heads", [
    (5, 1, 12), (3, 40, 12), (2, 64, 12), (2, 65, 12), (37, 70, 12), (2, 128, 12), (3, 129, 12), (2, 200, 12),
    (3, 511, 12), (3, 512, 12), (3, 513, 12), (2, 4097, 16)])
def test_edge_lengths(eng, n_groups, group_len, heads, legacy):
    """No tail block (64, 128, 512), one key past a block (65, 129, 513, 4097: a 16-key step with one valid key), the
    LONG_GROUP switch (511 / 512), a one-key group, and 37 groups of 70 (batch positions); poisoned inputs."""
    qkv = ar.poisoned_qkv(n_groups, group_len, heads, _gen("edge", n_groups, group_len, heads), "cuda")
    ref, bound = ar.attention(qkv, n_groups, group_len, heads)
    out = _run(eng, qkv, n_groups, group_len, heads, legacy)
    _check("edge_lengths", out, ref, bound, legacy, n_groups=n_groups, group_len=group_len, heads=heads)
    _mask_controls(out, qkv, n_groups, group_len, heads, bound)
    if not legacy:
        assert torch.equal(out, _run(eng, qkv, n_groups, group_len, heads))
        _batch_invariant(eng, qkv, out, n_groups, group_len, heads)


@pytest.mark.parametrize("legacy", [False, True], ids=["tcgen05", "mma_sync"])
@pytest.mark.parametrize("n_groups,group_len,heads", [(1, 300, 3), (1, 600, 1), (3, 1542, 3)])
def test_single_item_last_pair(eng, n_groups, group_len, heads, legacy):
    """An odd number of work items: the grid's last pair holds one item, whose issuer is the sole reader of its K / V tiles
    (the `single` arrivals).  The engine never gets there (its head counts are multiples of 4).  With 3 heads of 1542 keys
    the groups also start at odd items, so pairs straddle group boundaries: batch invariance is checked across them."""
    assert (-(-group_len // 128) * heads * n_groups) % 2 == 1
    qkv = ar.poisoned_qkv(n_groups, group_len, heads, _gen("single", n_groups, group_len, heads), "cuda")
    ref, bound = ar.attention(qkv, n_groups, group_len, heads)
    out = _run(eng, qkv, n_groups, group_len, heads, legacy)
    _check("single_item_last_pair", out, ref, bound, legacy, n_groups=n_groups, group_len=group_len, heads=heads)
    _mask_controls(out, qkv, n_groups, group_len, heads, bound)
    if not legacy:
        _batch_invariant(eng, qkv, out, n_groups, group_len, heads)


# ------------------------------------------------------------------------------------------ where it reads and writes
@pytest.mark.parametrize("legacy", [False, True], ids=["tcgen05", "mma_sync"])
@pytest.mark.parametrize("n_groups,group_len,heads", [(4, 197, 12), (3, 1542, 12)])
def test_row_ranges_of_larger_buffers(eng, n_groups, group_len, heads, legacy):
    """As the decoder's visual block calls it (a sub-batch's rows at an offset of the K/V cache): qkv is a row range of a
    buffer whose rows before and after hold NaN, and the output a row range of a buffer holding a sentinel.  The result is
    the standalone call's, bit for bit, and no row outside the output range is written."""
    rows, W = n_groups * group_len, heads * 64
    qkv = ar.poisoned_qkv(n_groups, group_len, heads, _gen("rows", group_len), "cuda")
    alone = _run(eng, qkv, n_groups, group_len, heads, legacy)
    ref, bound = ar.attention(qkv, n_groups, group_len, heads)
    _check("row_ranges", alone, ref, bound, legacy, group_len=group_len)
    _mask_controls(alone, qkv, n_groups, group_len, heads, bound)
    before, after = group_len + 5, 2 * group_len + 3
    big = torch.full((before + rows + after, 3 * W), float("nan"), dtype=torch.bfloat16, device="cuda")
    big[before:before + rows] = qkv
    assert torch.equal(_run(eng, big[before:before + rows], n_groups, group_len, heads, legacy), alone)
    obuf = torch.full((before + rows + after, W), SENTINEL, dtype=torch.bfloat16, device="cuda")
    _run(eng, qkv, n_groups, group_len, heads, legacy, out=obuf[before:before + rows])
    assert (obuf[:before] == SENTINEL).all() and (obuf[before + rows:] == SENTINEL).all()
    assert torch.equal(obuf[before:before + rows], alone)


# ------------------------------------------------------------------------------------------ rescale path
@pytest.mark.parametrize("legacy", [False, True], ids=["tcgen05", "mma_sync"])
@pytest.mark.parametrize("n_groups,group_len,heads,gain", [(2, 197, 12, 16.0), (1, 1182, 12, 12.0), (2, 257, 16, 24.0), (3, 40, 12, 16.0)])
def test_ramped_keys(eng, n_groups, group_len, heads, gain, legacy):
    """Key norms growing along the group: the running max moves by many powers of two per key block, so the tcgen05 kernel
    rescales its TMEM accumulator on most blocks; the scores reach |q| |k| ~ 10^3, where the score term of eps matters."""
    qkv = ar.ramped_qkv(n_groups, group_len, heads, gain, _gen("ramp", group_len), "cuda")
    ref, bound = ar.attention(qkv, n_groups, group_len, heads)
    out = _run(eng, qkv, n_groups, group_len, heads, legacy)
    _check("ramped_keys", out, ref, bound, legacy, group_len=group_len, gain=gain)
