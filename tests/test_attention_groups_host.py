"""The attention bound of attention_groups_ref.py pinned from both sides without a GPU: an fp32 emulation of the tcgen05
kernel's arithmetic stays inside it on small members of the GPU test's case table (random, poisoned-neighbour and
ramped-key inputs), and the same computation with a plausible bug in it -- as an emulation or as a reference -- falls
outside it."""
import pytest
import torch

import attention_groups_ref as ar


def _inputs(kind, n_groups, group_len, heads, gain=16.0):
    gen = torch.Generator().manual_seed(1000 * group_len + n_groups)
    if kind == "randn":
        return ar.randn_qkv(n_groups, group_len, heads, gen)
    if kind == "poisoned":
        return ar.poisoned_qkv(n_groups, group_len, heads, gen)
    return ar.ramped_qkv(n_groups, group_len, heads, gain, gen)


@pytest.mark.parametrize("kind,n_groups,group_len,heads,gain", [
    ("randn", 2, 197, 2, 0), ("randn", 2, 257, 2, 0), ("randn", 1, 1182, 1, 0), ("randn", 2, 70, 3, 0),
    ("poisoned", 3, 193, 2, 0), ("poisoned", 3, 201, 2, 0), ("poisoned", 3, 208, 2, 0), ("poisoned", 3, 1537, 1, 0),
    ("poisoned", 3, 1552, 1, 0), ("poisoned", 3, 512, 2, 0), ("poisoned", 3, 513, 1, 0), ("poisoned", 5, 1, 2, 0),
    ("poisoned", 2, 64, 2, 0), ("poisoned", 3, 129, 2, 0),
    ("ramped", 2, 197, 2, 16.0), ("ramped", 1, 1182, 1, 12.0), ("ramped", 2, 257, 2, 24.0), ("ramped", 3, 40, 2, 16.0)])
def test_emulation_within_bound(kind, n_groups, group_len, heads, gain):
    qkv = _inputs(kind, n_groups, group_len, heads, gain)
    ref, bound = ar.attention(qkv, n_groups, group_len, heads)
    out = ar.emulate_tc(qkv, n_groups, group_len, heads)
    assert ar.violations(out, ref, bound) == 0, ar.max_ratio(out, ref, bound)


@pytest.mark.parametrize("group_len", [197, 1542, 6168])
def test_poisoned_neighbour_outweighs_the_group(group_len):
    """The premise of the mask tests: in every row, a key leaked from the next group, and a zero-filled key leaked past the
    last group, weighs more than all the group's valid keys together -- by a margin far beyond the bound's score error."""
    n_groups = 2
    qkv = _inputs("poisoned", n_groups, group_len, 1)
    x = qkv.double().view(n_groups, group_len, 3, ar.HD)
    for g in range(n_groups):
        q, k = x[g, :, 0], x[g, :, 1]
        lse = torch.logsumexp(q @ k.t() * ar.SCALE, dim=-1)          # log of the valid keys' total weight
        leak = q @ x[g + 1, 0, 1] * ar.SCALE if g + 1 < n_groups else torch.zeros(group_len, dtype=torch.float64)
        assert (leak - lse).min().item() > 10.0, (g, (leak - lse).min().item())


CONTROLS = {
    # name: (how the wrong result is computed, the inputs that expose it)
    "next_group_key_attended": (lambda qkv, G, L, H: ar.emulate_tc(qkv, G, L, H, bug="leak"), ("poisoned", 3, 197, 2)),
    "next_group_key_attended_long": (lambda qkv, G, L, H: ar.emulate_tc(qkv, G, L, H, bug="leak"), ("poisoned", 3, 1542, 1)),
    "zero_fill_attended": (lambda qkv, G, L, H: ar.emulate_tc(qkv, G, L, H, bug="leak"), ("poisoned", 1, 1537, 1)),
    "last_key_dropped": (lambda qkv, G, L, H: ar.emulate_tc(qkv, G, L, H, bug="drop"), ("poisoned", 3, 197, 2)),
    "last_key_dropped_long": (lambda qkv, G, L, H: ar.emulate_tc(qkv, G, L, H, bug="drop"), ("poisoned", 3, 1542, 1)),
    "neighbour_head_v": (lambda qkv, G, L, H: ar.attention(qkv, G, L, H, v_head_shift=1, with_bound=False)[0], ("randn", 2, 197, 2)),
    "scale_applied_twice": (lambda qkv, G, L, H: ar.attention(qkv, G, L, H, scale=ar.SCALE ** 2, with_bound=False)[0], ("randn", 2, 197, 2)),
    "o_not_rescaled": (lambda qkv, G, L, H: ar.emulate_tc(qkv, G, L, H, bug="no_rescale"), ("ramped", 2, 257, 2)),
    "tail_pv_unmasked": (lambda qkv, G, L, H: ar.emulate_tc(qkv, G, L, H, bug="tail_unmasked"), ("poisoned", 3, 197, 2)),
    "tail_pv_unmasked_long": (lambda qkv, G, L, H: ar.emulate_tc(qkv, G, L, H, bug="tail_unmasked"), ("poisoned", 3, 1542, 1)),
}


@pytest.mark.parametrize("control", list(CONTROLS))
def test_negative_control_violates_bound(control):
    wrong_fn, (kind, G, L, H) = CONTROLS[control]
    qkv = _inputs(kind, G, L, H, gain=24.0)
    ref, bound = ar.attention(qkv, G, L, H)
    wrong = wrong_fn(qkv, G, L, H)
    n_bad = ar.violations(wrong, ref, bound)
    print(f"{control}: {n_bad} of {wrong.numel()} elements outside the bound, max err / bound {ar.max_ratio(wrong, ref, bound):.3g}")
    assert n_bad > 0, f"the bound cannot see {control}"


def test_leak_reference_matches_leaking_emulation():
    """The GPU tests run the mask controls as references (attention(extra=+1 / -1)); they describe the same bug as the
    emulation's mask off by one, to within the bound."""
    qkv = _inputs("poisoned", 3, 200, 2)
    for extra, bug in ((1, "leak"), (-1, "drop")):
        wrong_ref, wrong_bound = ar.attention(qkv, 3, 200, 2, extra=extra)
        assert ar.violations(ar.emulate_tc(qkv, 3, 200, 2, bug=bug), wrong_ref, wrong_bound) == 0

