"""GPU tests of the device sampling search (gitb200_op_search_ext / _decode_ext / _caption_ext): repetition penalty,
temperature, top-k / top-p, draws without replacement by the exponential race on Philox uniforms, num_return_sequences.
The oracle is oracle/search_oracle.search with torch.multinomial replaced, inside the test only, by the same race on the
same uniforms (tests/sampling_ref.py).  Sampling decisions closer than 1e-4 (relative) can go either way under fp32
rounding: their search entries are counted, reported and left out of the token comparison.  Deviations go to the
parity-metrics file through test_gpu_parity.record()."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import git_oracle as go
from oracle import search_oracle as so
from sampling_ref import broken_search, oracle_search
from test_gpu_parity import record

pytestmark = pytest.mark.gpu

SOS, EOS = 101, 102


@pytest.fixture(scope="module")
def g():
    import gitb200
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return gitb200


def make_logits(seed, steps, rows, V, ld, *, scale=3.0, hot=0, hot_boost=4.0, eos_boost=0.0):
    """[steps, rows, ld] fp32; columns >= V hold +1e4 (must be ignored).  `hot` tokens get +4 on every row and step, so that
    histories repeat them and the repetition penalty matters; eos_boost raises EOS so that captions end."""
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(steps, rows, ld, generator=gen) * scale
    x[..., V:] = 1e4
    if hot:
        x[..., 200:200 + hot] += hot_boost
    x[..., EOS] += eos_boost
    return x


def run_device(g, logits, n_clips, V, *, nb, pnb, keep, max_steps, lp=0.6, **smp):
    sp = g.SearchConfig(beam_size=nb, max_steps=max_steps, length_penalty=lp, per_node_beam_size=pnb, num_keep_best=keep)
    tok, lps = g.engine.op_search(logits.cuda(), V, n_clips, SOS, EOS, sp, sample=g.SampleConfig(**smp))
    return tok.long().cpu(), lps.cpu()


SAMPLE_CASES = [
    # V, ld, nb, pnb, keep, top_k, top_p, temperature, rp, nrs, eos_boost
    (1000, 1024, 1, 2, 1, 50, 1.0, 1.0, 1.0, 1, 0.0),
    (1000, 1024, 3, 2, 2, 0, 0.9, 1.0, 1.2, 2, 0.0),
    (1000, 1024, 4, 2, 1, 20, 0.8, 0.7, 1.0, 3, 6.0),
    (1000, 1024, 1, 3, 2, 0, 0.6, 1.5, 1.2, 2, 3.0),
    (30522, 30720, 1, 2, 1, 0, 0.9, 1.3, 1.2, 2, 0.0),
    (30522, 30720, 4, 2, 2, 40, 0.95, 1.0, 1.0, 1, 6.0),
    (30522, 30720, 3, 2, 1, 10, 0.7, 0.8, 1.2, 3, 2.0),
]


@pytest.mark.parametrize("case", SAMPLE_CASES)
def test_sampling_matches_oracle_on_identical_scores(g, case):
    V, ld, nb, pnb, keep, top_k, top_p, temp, rp, nrs, eos_boost = case
    n_clips, max_steps, seed = 6, 8, 1234 + V + nb
    rows = n_clips * nrs * nb
    logits = make_logits(seed, max_steps - 1, rows, V, ld, hot=6, eos_boost=eos_boost)
    kw = dict(nb=nb, pnb=pnb, keep=keep, max_steps=max_steps)
    tok, lps = run_device(g, logits, n_clips, V, do_sample=True, top_k=top_k, top_p=top_p, temperature=temp,
                          repetition_penalty=rp, num_return_sequences=nrs, seed=seed, **kw)
    ref_tok, ref_lp, smp = oracle_search(logits, n_clips, V=V, eos=EOS, sos=SOS, max_steps=max_steps, nb=nb, pnb=pnb,
                                         keep=keep, lp=0.6, do_sample=True, top_k=top_k, top_p=top_p, temperature=temp,
                                         rp=rp, nrs=nrs, seed=seed)
    unsure = smp.unsure()
    sure = [e for e in range(n_clips * nrs) if e not in unsure]
    record("sampling_op", case=str(case), entries=n_clips * nrs, excluded=len(unsure),
           max_lp_diff=max([(lps[e] - ref_lp[e]).abs().max().item() for e in sure] or [0.0]))
    assert len(sure) >= (n_clips * nrs) // 2, f"{len(unsure)} of {n_clips * nrs} entries had a near-tie"
    for e in sure:
        assert torch.equal(tok[e], ref_tok[e]), (e, tok[e], ref_tok[e])
        assert torch.allclose(lps[e], ref_lp[e], atol=2e-5, rtol=0), (e, lps[e], ref_lp[e])


DET_CASES = [
    # V, ld, nb, pnb, keep, rp, nrs
    (1000, 1024, 3, 2, 2, 1.2, 2),
    (30522, 30720, 4, 2, 1, 1.3, 1),
    (30522, 30720, 1, 2, 1, 1.2, 3),
    (1000, 1024, 2, 3, 3, 0.8, 2),
]


@pytest.mark.parametrize("case", DET_CASES)
def test_beam_with_penalty_and_return_sequences_is_token_exact(g, case):
    V, ld, nb, pnb, keep, rp, nrs = case
    n_clips, max_steps = 5, 9
    logits = make_logits(77 + nb, max_steps - 1, n_clips * nrs * nb, V, ld, hot=5, hot_boost=10.0, eos_boost=2.0)
    tok, lps = run_device(g, logits, n_clips, V, nb=nb, pnb=pnb, keep=keep, max_steps=max_steps, repetition_penalty=rp,
                          num_return_sequences=nrs, seed=5)
    ref_tok, ref_lp, _ = oracle_search(logits, n_clips, V=V, eos=EOS, sos=SOS, max_steps=max_steps, nb=nb, pnb=pnb, keep=keep,
                                       lp=0.6, do_sample=False, top_k=None, top_p=None, temperature=1.0, rp=rp, nrs=nrs,
                                       seed=5)
    record("penalty_beam_op", case=str(case), max_lp_diff=(lps - ref_lp).abs().max().item())
    assert torch.equal(tok, ref_tok)
    assert torch.allclose(lps, ref_lp, atol=2e-5, rtol=0)
    # the penalty changed something: the same search without it differs
    plain, _ = run_device(g, logits, n_clips, V, nb=nb, pnb=pnb, keep=keep, max_steps=max_steps, num_return_sequences=nrs)
    assert not torch.equal(plain, tok)


def test_return_sequences_without_sampling_are_identical_copies(g):
    V, nrs, nb, n_clips = 1000, 3, 2, 4
    logits = make_logits(5, 7, n_clips * nb, V, 1024, hot=4)
    rep = logits.view(7, n_clips, 1, nb, 1024).expand(7, n_clips, nrs, nb, 1024).reshape(7, n_clips * nrs * nb, 1024)
    tok, lps = run_device(g, rep.contiguous(), n_clips, V, nb=nb, pnb=2, keep=1, max_steps=8, repetition_penalty=1.2,
                          num_return_sequences=nrs)
    tok = tok.view(n_clips, nrs, -1)
    for j in range(1, nrs):
        assert torch.equal(tok[:, j], tok[:, 0])


@pytest.mark.parametrize("rule", ["offsets_j_div_pnb", "no_shift", "penalty_per_occurrence", "penalty_after_filter",
                                  "done_on_first"])
def test_negative_controls_each_broken_rule_is_detected(g, rule):
    """The restated sampling branch equals the device; breaking one rule of it makes it differ."""
    V, ld, nb, pnb, keep, n_clips, max_steps, nrs = 1000, 1024, 3, 2, 2, 48, 8, 1
    args = dict(top_k=0, top_p=0.5, temperature=1.0, rp=1.6, seed=99)
    logits = make_logits(4242, max_steps - 1, n_clips * nrs * nb, V, ld, scale=2.0, hot=3, eos_boost=3.0)
    # a few very repetitive rows: histories repeat the hot tokens
    tok, lps = run_device(g, logits, n_clips, V, nb=nb, pnb=pnb, keep=keep, max_steps=max_steps, do_sample=True,
                          top_k=args["top_k"], top_p=args["top_p"], temperature=args["temperature"],
                          repetition_penalty=args["rp"], num_return_sequences=nrs, seed=args["seed"])
    kw = dict(V=V, eos=EOS, sos=SOS, max_steps=max_steps, nb=nb, pnb=pnb, keep=keep, lp=0.6, nrs=nrs, **args)
    good_tok, good_lp = broken_search(logits, n_clips, **kw)
    ref_tok, _, smp = oracle_search(logits, n_clips, do_sample=True, **{k: v for k, v in kw.items() if k != "rp"},
                                    rp=args["rp"])
    sure = [e for e in range(n_clips) if e not in smp.unsure()]
    assert all(torch.equal(good_tok[e], ref_tok[e]) and torch.equal(tok[e], good_tok[e]) for e in sure)
    bad_tok, bad_lp = broken_search(logits, n_clips, break_rule=rule, **kw)
    differs = sum(not (torch.equal(tok[e], bad_tok[e]) and torch.allclose(lps[e], bad_lp[e], atol=2e-5)) for e in sure)
    record("sampling_negative_control", rule=rule, entries=len(sure), differing=differs)
    assert differs > 0, f"breaking {rule} went unnoticed"


def test_draw_distribution(g):
    """8192 clips over one fixed row: first draws follow the filtered softmax, unordered pairs of draws the law of two
    draws without replacement; nothing outside the kept set is ever drawn."""
    from scipy.stats import chisquare
    V, ld, n = 1000, 1024, 8192
    row = torch.randn(ld, generator=torch.Generator().manual_seed(3)) * 1.5
    row[V:] = 1e4
    row[EOS] = -50.0
    top_k, top_p, temp = 12, 0.9, 1.0
    filt = so.top_k_top_p_filtering(row[None, :V].clone(), top_k=top_k, top_p=top_p, min_tokens_to_keep=2)[0]
    p = torch.softmax(filt.double(), -1).numpy()
    kept = np.flatnonzero(p > 0)
    smp = dict(do_sample=True, top_k=top_k, top_p=top_p, temperature=temp, seed=2024)
    # first draw: nb = 1, the beam continues with candidate 0
    tok, _ = run_device(g, row.expand(2, n, ld).contiguous(), n, V, nb=1, pnb=2, keep=1, max_steps=3, **smp)
    first = tok[:, 0, 1].numpy()
    assert np.isin(first, kept).all()
    obs = np.array([(first == k).sum() for k in kept])
    chi1 = chisquare(obs, p[kept] * n)
    # unordered pairs: nb = 2, candidates 0 and 1 are row 0's two draws (beam ids 0 and 1); all four final hypotheses kept
    tok, _ = run_device(g, row.expand(2, 2 * n, ld).contiguous(), n, V, nb=2, pnb=2, keep=4, max_steps=3, **smp)
    pairs = [tuple(sorted(set(tok[i, :, 1].tolist()))) for i in range(n)]
    assert all(len(q) == 2 and set(q) <= set(kept.tolist()) for q in pairs)
    cats = [(a, b) for ai, a in enumerate(kept) for b in kept[ai + 1:]]
    exp = np.array([p[a] * p[b] / (1 - p[a]) + p[b] * p[a] / (1 - p[b]) for a, b in cats]) * n
    got = np.array([sum(1 for q in pairs if q == (a, b)) for a, b in cats])
    big = exp >= 5  # the chi-square approximation needs expected counts >= 5; the rest are pooled
    if (~big).any():
        got, exp = np.append(got[big], got[~big].sum()), np.append(exp[big], exp[~big].sum())
    chi2 = chisquare(got, exp * (got.sum() / exp.sum()))
    record("sampling_distribution", kept=len(kept), p_first=chi1.pvalue, p_pairs=chi2.pvalue)
    assert chi1.pvalue > 1e-3 and chi2.pvalue > 1e-3, (chi1, chi2)


def test_seeds_and_batch_position(g):
    V, n_clips = 1000, 16
    logits = make_logits(8, 7, n_clips * 2, V, 1024, hot=4)
    kw = dict(nb=2, pnb=2, keep=1, max_steps=8, do_sample=True, top_k=0, top_p=0.95, temperature=1.2, repetition_penalty=1.2)
    a, la = run_device(g, logits, n_clips, V, seed=7, **kw)
    b, lb = run_device(g, logits, n_clips, V, seed=7, **kw)
    c, _ = run_device(g, logits, n_clips, V, seed=8, **kw)
    assert torch.equal(a, b) and torch.equal(la, lb)
    assert not torch.equal(a, c)
    # the first 4 clips alone (their rows are the first 4 * nb of every step): same captions as inside the batch of 16
    d, ld_ = run_device(g, logits[:, :8].contiguous(), 4, V, seed=7, **kw)
    assert torch.equal(d, a[:4]) and torch.equal(ld_, la[:4])


# ------------------------------------------------------------------ model level
@pytest.fixture(scope="module")
def model(g):
    cfg = go.GitConfig(num_image_with_embedding=2, tie_output=False)
    sd = go.init_state_dict(cfg, seed=42, temporal_std=0.02, perturb=True)
    eng = g.Engine(g.make_config({"num_image_with_embedding": 2}, cfg.sos_index, cfg.eos_index), 0)
    eng.load_state_dict(sd)
    frames = torch.randn(4, 2, 3, 224, 224, generator=torch.Generator().manual_seed(9)).cuda()
    return cfg, eng, frames


def test_caption_saved_logits_reproduce_tokens_and_are_pre_penalty(g, model):
    cfg, eng, frames = model
    nb, nrs, ms = 2, 2, 10
    sp = g.SearchConfig(beam_size=nb, max_steps=ms)
    smp = g.SampleConfig(do_sample=True, top_k=30, top_p=0.9, temperature=0.8, repetition_penalty=1.2,
                         num_return_sequences=nrs, seed=31)
    tok, lps, logits = eng.caption(frames[:2], sp, save_logits=True, sample=smp)
    steps = logits.shape[0]
    assert steps == eng.last_decode_steps() and tok.shape == (2 * nrs, 1, ms)
    full = torch.cat([logits.cpu(), logits[-1:].cpu().expand(ms - 1 - steps, -1, -1)]) if steps < ms - 1 else logits.cpu()
    ref_tok, ref_lp, s = oracle_search(full, 2, V=cfg.vocab_size, eos=cfg.eos_index, sos=cfg.sos_index, max_steps=ms, nb=nb,
                                       pnb=2, keep=1, lp=0.6, do_sample=True, top_k=30, top_p=0.9, temperature=0.8, rp=1.2,
                                       nrs=nrs, seed=31)
    sure = [e for e in range(2 * nrs) if e not in s.unsure()]
    record("sampling_model", entries=2 * nrs, excluded=2 * nrs - len(sure), steps=steps)
    assert sure
    for e in sure:
        assert torch.equal(tok[e].long().cpu(), ref_tok[e]), (e, tok[e], ref_tok[e])
        assert torch.allclose(lps[e].cpu(), ref_lp[e], atol=2e-5, rtol=0)
    # pre-penalty: the first step (history = SOS) of the same call without penalty and temperature saves the same scores
    plain = g.SampleConfig(do_sample=True, top_k=30, top_p=0.9, num_return_sequences=nrs, seed=31)
    _, _, logits0 = eng.caption(frames[:2], sp, save_logits=True, sample=plain)
    assert torch.equal(logits0[0], logits[0])


def test_caption_invariants_and_graph_replay(g, model):
    cfg, eng, frames = model
    sp = g.SearchConfig(beam_size=1, max_steps=8)
    # all-default sample parameters: bit-identical to gitb200_caption
    t0, l0, _ = eng.caption(frames[:2], sp)
    t1, l1, _ = eng.caption(frames[:2], sp, sample=g.SampleConfig(seed=123))
    assert torch.equal(t0, t1) and torch.equal(l0, l1)
    smp = dict(do_sample=True, top_k=0, top_p=0.9, temperature=1.0, repetition_penalty=1.2, num_return_sequences=2)
    # graph replay with new seeds (second call captures, later calls replay) equals eager runs with those seeds; the graph
    # key holds the output pointers, so the calls reuse one pair of buffers
    st = torch.cuda.Stream()
    outs = {}
    clips = frames[:2].contiguous()
    tok = torch.empty(4, 1, 8, dtype=torch.int32, device="cuda")
    lpb = torch.empty(4, 1, device="cuda")
    c = sp.to_c()
    with torch.cuda.stream(st):
        n0 = eng.lib.gitb200_graph_launches(eng.h)
        for seed in (1, 1, 2, 3):
            x = g.SampleConfig(seed=seed, **smp).to_c()
            rc = eng.lib.gitb200_caption_ext(eng.h, ctypes.c_void_p(clips.data_ptr()), 2, 2, ctypes.byref(c), ctypes.byref(x),
                                             ctypes.c_void_p(tok.data_ptr()), ctypes.c_void_p(lpb.data_ptr()), None,
                                             ctypes.c_void_p(st.cuda_stream))
            assert rc == 0
            outs[seed] = (tok.clone(), lpb.clone())
        st.synchronize()
        assert eng.lib.gitb200_graph_launches(eng.h) == n0 + 3
    eng.set_graph_max_clips(0)
    eng.set_graph_segments(False)
    try:
        for seed in (2, 3):
            t, l, _ = eng.caption(frames[:2], sp, sample=g.SampleConfig(seed=seed, **smp))
            assert torch.equal(t, outs[seed][0]) and torch.equal(l, outs[seed][1])
    finally:
        eng.set_graph_max_clips(8)
        eng.set_graph_segments(True)
    assert not torch.equal(outs[2][0], outs[3][0])


@pytest.mark.parametrize("field,value,named", [
    ("temperature", 0.0, "temperature"), ("temperature", -1.0, "temperature"), ("top_p", 0.0, "top_p"),
    ("top_p", 1.5, "top_p"), ("repetition_penalty", 0.0, "repetition_penalty"),
    ("num_return_sequences", 0, "num_return_sequences"), ("num_return_sequences", 40000, "rows per clip"),
])
def test_invalid_sample_parameters_are_rejected(g, model, field, value, named):
    cfg, eng, frames = model
    eng.encode(frames[:2], want_features=False)  # decode_ext needs visual features to reach its parameter checks
    sp = g.SearchConfig(beam_size=4, max_steps=8)
    bad = g.SampleConfig(do_sample=True, top_k=5, top_p=0.9, seed=1)
    setattr(bad, field, value)
    n0 = eng.launch_count()
    for call in (lambda: eng.caption(frames[:2], sp, sample=bad), lambda: eng.decode(2, sp, sample=bad),
                 lambda: g.engine.op_search(torch.zeros(7, 8 * max(1, bad.num_return_sequences), 1024, device="cuda")
                                            if value != 40000 else torch.zeros(1, 1, 1024, device="cuda"),
                                            1000, 2, SOS, EOS, sp, sample=bad)):
        with pytest.raises(g.GitB200Error, match=named):
            call()
    assert eng.launch_count() == n0  # nothing was enqueued


@pytest.mark.parametrize("sp_kw,named", [(dict(beam_size=9), "beam"), (dict(beam_size=4, per_node_beam_size=5), "per-node"),
                                         (dict(num_keep_best=16), "keep"), (dict(max_steps=1), "max_steps")])
def test_beam_limits_are_rejected_before_encoding(g, model, sp_kw, named):
    cfg, eng, frames = model
    sp = g.SearchConfig(**{**dict(beam_size=2, max_steps=8), **sp_kw})
    n0 = eng.launch_count()
    with pytest.raises(g.GitB200Error, match=named):
        eng.caption(frames[:2], sp, sample=g.SampleConfig(do_sample=True, top_k=5, top_p=0.9, seed=1))
    assert eng.launch_count() == n0


def test_top_k_below_the_draws_and_the_row_chunk_grid_are_rejected(g, model):
    cfg, eng, frames = model
    eng.encode(frames[:2], want_features=False)
    n0 = eng.launch_count()
    # torch.multinomial without replacement cannot draw 3 words from the 2 that top_k = 2 keeps
    sp3 = g.SearchConfig(beam_size=2, max_steps=8, per_node_beam_size=3)
    with pytest.raises(g.GitB200Error, match="top_k 2 keeps fewer tokens than the 3 draws"):
        eng.decode(2, sp3, sample=g.SampleConfig(do_sample=True, top_k=2, top_p=0.9, seed=1))
    # 3 rows per clip run in 2-row chunks of the decoder's attention grid: 32768 clips need 65536 blocks (> 65535); the check
    # comes before the frames are read, so a one-clip buffer stands in for them
    sp = g.SearchConfig(beam_size=3, max_steps=8)
    x = g.SampleConfig(do_sample=True, top_k=5, top_p=0.9, seed=1).to_c()
    c = sp.to_c()
    tok = torch.empty(1, dtype=torch.int32, device="cuda")
    lp = torch.empty(1, device="cuda")
    rc = eng.lib.gitb200_caption_ext(eng.h, ctypes.c_void_p(frames.data_ptr()), 32768, 2, ctypes.byref(c), ctypes.byref(x),
                                     ctypes.c_void_p(tok.data_ptr()), ctypes.c_void_p(lp.data_ptr()), None, None)
    assert rc != 0 and b"rows per clip" in eng.lib.gitb200_last_error(eng.h)
    assert eng.launch_count() == n0
