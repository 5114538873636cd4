"""float64 reference, error bound, test inputs and a CPU emulation for attention_groups_tc (csrc/attention_tc.cu) and the
mma.sync kernel it replaced (attention_groups, csrc/attention.cu).  Used by test_attention_groups_host.py (no GPU) and
test_gpu_attention_groups.py.

Layout: qkv bf16 [n_groups * L, 3 * heads * 64] (q | k | v, head h at columns h * 64 of each third); output [n_groups * L,
heads * 64].  Group g's queries attend to its own L keys, scale 1/8 (head dim 64).

The bound, per output element (i, d) of one (group, head), with p the float64 softmax, ref = p v, A = p |v| and
D = p |v - ref|:

  bound = 2^-8 |ref| + 2^-8 A + (ceil(L / 16) + 2) 2^-23 A + 2 eps D

  * 2^-8 |ref|: the output is rounded to bf16 (round to nearest, 8 significant bits: relative error <= 2^-8).
  * 2^-8 A: P is rounded to bf16 before the P V product, while the row sum l adds the unrounded fp32 P (attention_tc.cu
    pack_bf16 next to __fadd2_rn; attention.cu pack_bf16 next to ls += p0 + p1).  Each term P_k v_k is then off by at most
    2^-8 P_k |v_k|; divided by l that is 2^-8 A.
  * (ceil(L / 16) + 2) 2^-23 A: fp32 accumulation of P V and of l.  One rounding of at most 2^-23 per 16-key MMA step into
    the fp32 accumulator (the model test_gpu_gemm_shapes.f32_bound uses for 16-deep steps, truncation allowed), + 2 for
    1 / l and the product O * (1 / l).  l adds the same P in chains no longer than the P V steps (8 fadd2 per block, then
    one fmaf per block), so its relative error is covered by the same count.  The rescales O *= alpha add one rounding per
    64-key block, less than the 4 MMA steps of that block already count.
  * 2 eps D: eps bounds the relative error of every key's weight 2^(s c - m) against the exact exp(s / 8), where c is
    scale * log2(e) in fp32.  A weight vector w (1 + eta), |eta| <= eps, moves sum w v / sum w by at most
    eps D / (1 - eps) <= 2 eps D.  eps per query row is the sum of
      - ln 2 * max over keys of the error of the exponent x = s c - m:
          c 4 2^-22 (|q| |k|^T): the score s, an fp32 sum of 64 products in 4 MMA steps of 16 (the same model);
          c 2^-23 |s|: c is fp32(scale * fp32(log2 e)) (relative error 2^-24, scale = 1/8 is exact) and the mma.sync kernel
            rounds s * c before it subtracts m (one more 2^-24);
          2^-24 (c (max_k s - s) + 8): the rounding of x itself; |x| <= c (max_k s - s) + 8 since the lazy running max of
            the tcgen05 kernel trails the true maximum by at most RESCALE_THRESHOLD = 8 (log2 units).
      - 2^-22 per exponential: ex2.approx.ftz.f32 and exp2f are within 2 ulp; a key's weight takes one exp2 of its own and
        one per rescale of the running max after it (alpha = exp2(m_old - m_new), at most one per 64-key block, applied to
        O and l alike), so ceil(L / 64) 2^-22;
      - ln 2 2^-24 c (max_k s - min_k s): the roundings of m_old - m_new, whose magnitudes add up to at most the score range;
      - 7.5e-5 for L >= LONG_GROUP: the tcgen05 kernel computes one pair of every eight keys with ex2_poly2, whose stated
        maximum relative error is 7.5e-5.
    D is replaced by the upper bound p |v - vbar| + |ref - vbar| (triangle inequality, vbar = the column mean of the
    group's v), which is one matrix product instead of an L x L x 64 tensor and still sees a common offset of v cancel.
The same terms cover the mma.sync kernel: its running max is exact (|x| <= c (max_k s - s)), it uses exp2f and no polynomial.

Poisoned-neighbour inputs (poisoned_qkv) make a mask error visible: one dimension of q is (-1)^g b and the same dimension
of k is -(-1)^g b in group g.  Inside a group that adds -b^2 to every score, which the softmax ignores; a key read from
group g + 1 scores +2 b^2 above the group's own keys and a zero-filled key read past the last row (TMA fill) +b^2.  With
b = 16 and scale 1/8 that is 64 resp. 32 nats, far more than the ln(6168) + a few nats the valid keys add up to, so a leaked
key outweighs all valid keys together (test_attention_groups_host checks it).  The V rows of each group's first 16 keys
carry an offset of -3, the others +1: a leaked key moves the output by O(1) whichever neighbour it comes from.
"""
import math

import torch

SCALE = 0.125
HD = 64
BKV = 64                 # keys per block of both kernels
LONG_GROUP = 512         # attention_tc.cu: from here on the EXP_FIRST / SHARE_KV template, one exp2 pair in four on the polynomial
RESCALE_THRESHOLD = 8.0  # attention_tc.cu: the running max moves only when a block exceeds it by more than 2^8
BF16_U = 2.0 ** -8
F32_U = 2.0 ** -24
EX2_REL = 2.0 ** -22     # ex2.approx.ftz.f32 / exp2f: 2 ulp
POLY_REL = 7.5e-5        # ex2_poly2's stated maximum relative error
LN2 = math.log(2.0)
LOG2E_F32 = float(torch.tensor(1.4426950408889634, dtype=torch.float32))

POISON_DIM = 63
POISON_B = 16.0
V_REST, V_FIRST16 = 1.0, -3.0


def scale_log2(scale):
    """c as both kernels form it: fp32(scale * fp32(log2 e))."""
    return float(torch.tensor(scale, dtype=torch.float32) * torch.tensor(LOG2E_F32, dtype=torch.float32))


def _operands(qkv, n_groups, group_len, heads, gh, extra=0, v_head_shift=0, dtype=torch.float64):
    """q [n, L, 64] and k, v [n, L + extra, 64] for the (group, head) pairs gh = (g [n], h [n]).  Keys run on past the
    group into the next group's rows; rows past the end of qkv read as zero (what the TMA tensor map fills in)."""
    g, h = gh
    rows = n_groups * group_len
    x = qkv[:rows].view(rows, 3, heads, HD)
    q = x.view(n_groups, group_len, 3, heads, HD)[g, :, 0, h].to(dtype)
    lk = group_len + extra
    pad = max(0, (n_groups - 1) * group_len + lk - rows)
    if pad:
        x = torch.cat([x, torch.zeros(pad, 3, heads, HD, dtype=x.dtype, device=x.device)])
    idx = g[:, None] * group_len + torch.arange(lk, device=g.device)[None]
    k = x[idx, 1, h[:, None]].to(dtype)
    v = x[idx, 2, ((h + v_head_shift) % heads)[:, None]].to(dtype)
    return q, k, v


def _pairs(n_groups, heads, device, budget_pairs):
    f = torch.arange(n_groups * heads, device=device)
    for i in range(0, f.numel(), budget_pairs):
        c = f[i:i + budget_pairs]
        yield c, (c // heads, c % heads)


def _scatter(out, c, val, group_len, heads):
    """val [n, L, 64] of flat (group, head) indices c -> out [n_groups * L, heads * 64]."""
    o = out.view(-1, group_len, heads, HD)
    o[c // heads, :, c % heads] = val


def attention(qkv, n_groups, group_len, heads, scale=SCALE, extra=0, v_head_shift=0, with_bound=True, budget=1 << 27):
    """float64 attention on the exact bf16 operands, chunked over (group, head) so that 6168-key groups fit in memory; runs
    on qkv's device.  Returns (ref, bound), bound None unless with_bound.  extra = +1 attends one key past each group (the
    next group's first row, or a zero row after the last group), -1 drops each group's last key; v_head_shift = 1 reads V
    of the next head: the references of the negative controls."""
    dev = qkv.device
    rows = n_groups * group_len
    ref = torch.empty(rows, heads * HD, dtype=torch.float64, device=dev)
    bound = torch.empty_like(ref) if with_bound else None
    lk = group_len + extra
    c2 = scale_log2(scale)
    n_blocks = math.ceil(group_len / BKV)
    acc = BF16_U + (math.ceil(group_len / 16) + 2) * 2 * F32_U
    for c, gh in _pairs(n_groups, heads, dev, max(1, budget // (group_len * lk))):
        q, k, v = _operands(qkv, n_groups, group_len, heads, gh, extra, v_head_shift)
        s = q @ k.transpose(1, 2)
        p = torch.softmax(s * scale, dim=-1)
        r = p @ v
        _scatter(ref, c, r, group_len, heads)
        if not with_bound:
            continue
        A = p @ v.abs()
        vbar = v.mean(1, keepdim=True)
        D = p @ (v - vbar).abs() + (r - vbar).abs()
        smax = s.amax(-1, keepdim=True)
        smin = s.amin(-1, keepdim=True)
        dx = c2 * (4 * 2.0 ** -22 * (q.abs() @ k.abs().transpose(1, 2)) + 2 * F32_U * s.abs()) + F32_U * (c2 * (smax - s) + RESCALE_THRESHOLD)
        eps = LN2 * dx.amax(-1, keepdim=True) + n_blocks * EX2_REL + LN2 * F32_U * c2 * (smax - smin)
        if group_len >= LONG_GROUP:
            eps = eps + POLY_REL
        del s, p, dx
        _scatter(bound, c, BF16_U * r.abs() + acc * A + 2 * eps * D, group_len, heads)
    return ref, bound


def max_ratio(out, ref, bound):
    return ((out.double() - ref).abs() / bound).max().item()


def violations(out, ref, bound):
    """Elements of out outside the bound (NaN counts as outside)."""
    return int((~((out.double() - ref).abs() <= bound)).sum())


# ------------------------------------------------------------------------------------------ inputs
def randn_qkv(n_groups, group_len, heads, gen, device="cpu"):
    return torch.randn(n_groups * group_len, 3 * heads * HD, generator=gen, device=device).bfloat16()


def poisoned_qkv(n_groups, group_len, heads, gen, device="cpu", b=POISON_B):
    """See the module docstring: neighbours' keys dominate any row that reads them, first-16 V rows offset from the rest."""
    x = torch.randn(n_groups, group_len, 3, heads, HD, generator=gen, device=device)
    sign = (1.0 - 2.0 * (torch.arange(n_groups, device=device) % 2)).view(n_groups, 1, 1)
    x[:, :, 0, :, POISON_DIM] = sign * b
    x[:, :, 1, :, POISON_DIM] = -sign * b
    x[:, :, 2] += V_REST
    x[:, :16, 2] += V_FIRST16 - V_REST
    return x.reshape(n_groups * group_len, 3 * heads * HD).bfloat16()


def ramped_qkv(n_groups, group_len, heads, gain, gen, device="cpu"):
    """Key norms growing along the group from 0.05 to `gain`: every key block raises the row maximum by many powers of two,
    so the tcgen05 kernel's lazy running max moves (and O is rescaled in tensor memory) on most blocks."""
    x = torch.randn(n_groups, group_len, 3, heads, HD, generator=gen, device=device)
    x[:, :, 1] *= torch.linspace(0.05, gain, group_len, device=device).view(1, group_len, 1, 1)
    return x.reshape(n_groups * group_len, 3 * heads * HD).bfloat16()


# ------------------------------------------------------------------------------------------ emulation
EMULATION_BUGS = (None, "leak", "drop", "no_rescale", "tail_unmasked")


def emulate_tc(qkv, n_groups, group_len, heads, scale=SCALE, bug=None):
    """fp32 CPU emulation of attention_tc_kernel's arithmetic: 64-key blocks, masking at the tail block, the lazy running
    max (moves when a block's maximum exceeds it by more than 2^8; O and l then take alpha = 2^(m_old - m_new)), P = 2^(s c
    - m) rounded to bf16 for P V while l adds the fp32 P, output O * (1 / l) rounded to bf16.  (exp2 is torch's, not
    ex2.approx or the polynomial: their errors are in the bound's eps and too small to matter here.)

    bug: None, or the kernel with a bug in it, for the negative controls:
      "leak"          the tail mask lets in one key more (i > nk instead of i >= nk): the next group's first key / zero fill;
      "drop"          the tail mask drops the group's last valid key;
      "no_rescale"    O is not rescaled when the running max moves (l still is);
      "tail_unmasked" the tail block's P V runs over all 64 keys with P from the unmasked scores (l from the masked ones)."""
    assert bug in EMULATION_BUGS
    n_blocks = math.ceil(group_len / BKV)
    c = torch.tensor(scale_log2(scale), dtype=torch.float32)
    out = torch.empty(n_groups * group_len, heads * HD, dtype=torch.bfloat16)
    gh_all = torch.arange(n_groups * heads)
    cidx, gh = gh_all, (gh_all // heads, gh_all % heads)
    q, k, v = _operands(qkv.cpu(), n_groups, group_len, heads, gh, extra=n_blocks * BKV - group_len, dtype=torch.float32)
    n = q.shape[0]
    m = torch.full((n, group_len, 1), -math.inf)
    l = torch.zeros(n, group_len, 1)
    O = torch.zeros(n, group_len, HD)
    ar = torch.arange(BKV)
    for j in range(n_blocks):
        kb, vb = k[:, j * BKV:(j + 1) * BKV], v[:, j * BKV:(j + 1) * BKV]
        s = q @ kb.transpose(1, 2)
        nk = min(BKV, group_len - j * BKV)
        tail = j + 1 == n_blocks and group_len % BKV != 0
        valid = nk + (1 if (bug == "leak" and tail) else 0) - (1 if (bug == "drop" and j + 1 == n_blocks) else 0)
        sm = torch.where(ar < valid, s, torch.tensor(-math.inf))
        mblk = sm.amax(-1, keepdim=True) * c
        need = mblk > m + RESCALE_THRESHOLD
        alpha = torch.where(need & (j > 0), torch.exp2(m - mblk), torch.ones(()))
        m = torch.where(need, mblk, m)
        P = torch.exp2(sm * c - m)
        Pv = torch.exp2(s * c - m) if (bug == "tail_unmasked" and tail) else P
        l = l * alpha + P.sum(-1, keepdim=True)
        O = (O if bug == "no_rescale" else O * alpha) + Pv.bfloat16().float() @ vb
    _scatter(out, cidx, (O * (1.0 / l)).bfloat16(), group_len, heads)
    return out
