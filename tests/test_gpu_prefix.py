"""GPU tests of the prompted device search (batch['prefix'], model.py:432-437): gitb200_op_search_prefix, _decode_prefix and
_caption_prefix.  The oracle is oracle/search_oracle.search with the prompt as input_ids and oracle/git_oracle.DecodingState
(whose first call runs the whole prompt, as upstream's first decoding_step does).  Deviations go to the parity-metrics file
through test_gpu_parity.record()."""
import ctypes
import functools
import re

import numpy as np
import pytest
import torch

from oracle import git_oracle as go
from oracle import search_oracle as so
from sampling_ref import RaceSampler
from test_gpu_parity import record

pytestmark = pytest.mark.gpu

SOS, EOS = 101, 102
ROBUST = 0.3  # sigma(logits) units: twice the stated max logit tolerance (test_gpu_baseline_geometry.py)


@pytest.fixture(scope="module")
def g():
    import gitb200
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return gitb200


def make_logits(seed, steps, rows, V, ld, *, hot=0, eos_boost=0.0):
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(max(steps, 0), rows, ld, generator=gen) * 3.0
    x[..., V:] = 1e4
    if hot:
        x[..., 200:200 + hot] += 4.0
    x[..., EOS] += eos_boost
    return x


def make_prompt(seed, rows, P, V, hot=0):
    gen = torch.Generator().manual_seed(seed)
    p = torch.randint(1, V, (rows, P), generator=gen) if not hot else 200 + torch.randint(0, hot, (rows, P), generator=gen)
    p[:, 0] = SOS
    return p


def oracle(logits, prompt, n_clips, *, V, max_steps, nb, pnb, keep, lp, rp=1.0, nrs=1, sample=None, hyp_cls=None, step_fn=None):
    """so.search over fixed per-step scores with input_ids = the prompt ([1 or n_clips, P]); decoded [n*nrs, keep, max_steps]."""
    steps = iter(range(10 ** 6))
    P = prompt.shape[1]

    def step(ids):
        x = logits[next(steps), :, :V].clone()
        return step_fn(ids, x) if step_fn else x

    start = prompt.long().expand(n_clips, P)
    kw = {}
    if sample is not None:
        kw = dict(do_sample=True, top_k=sample["top_k"], top_p=sample["top_p"], temperature=sample["temperature"])
    with pytest.MonkeyPatch.context() as mp:
        smp = None
        if sample is not None:
            smp = RaceSampler(nb, nrs, sample["seed"], sample["top_p"])
            smp.step = P - 1  # the device's Philox step word is the text position t = cur_len - 1
            mp.setattr(torch, "multinomial", smp.multinomial)
            mp.setattr(so, "top_k_top_p_filtering", smp.filtering)
        if hyp_cls is not None:
            mp.setattr(so, "BeamHypotheses", hyp_cls)
        dec, lps, _ = so.search(start, step, eos_index=EOS, max_steps=max_steps, beam_size=nb, length_penalty=lp,
                                per_node_beam_size=pnb, num_keep_best=keep, save_logits=False, repetition_penalty=rp,
                                num_return_sequences=nrs, **kw)
    if keep == 1:
        dec = dec.unsqueeze(1)
    return dec, lps, smp


def device(g, logits, prompt, n_clips, V, *, max_steps, nb, pnb, keep, lp, reorder=False, sample=None):
    sp = g.SearchConfig(beam_size=nb, max_steps=max_steps, length_penalty=lp, per_node_beam_size=pnb, num_keep_best=keep,
                        reorder_cache=reorder)
    tok, lps = g.engine.op_search(logits.cuda(), V, n_clips, SOS, EOS, sp, sample=sample, prefix=prompt)
    return tok.long().cpu(), lps.cpu()


# ------------------------------------------------------------------ operator search
MS = 8
OP_CASES = []
for P in (1, 2, 5, MS - 1, MS, MS + 2):
    OP_CASES += [(1000, 1024, 1, 2, 1, 0.0, 0.6, P, False), (1000, 1024, 4, 2, 2, 6.0, 0.6, P, True),
                 (1000, 1024, 3, 2, 3, 3.0, 0.6, P, False)]
OP_CASES += [(30522, 30720, 4, 2, 1, 6.0, 0.6, 3, False), (30522, 30720, 1, 2, 1, 0.0, 0.6, 2, True),
             (30522, 30720, 3, 2, 2, 3.0, 0.0, 4, True), (1000, 1024, 4, 3, 1, 6.0, 0.0, 4, False)]


@pytest.mark.parametrize("case", OP_CASES, ids=lambda c: "V{}_nb{}_pnb{}_k{}_eos{}_lp{}_P{}_{}".format(c[0], *c[2:8], "ro" if c[8] else "ref"))
def test_op_search_matches_oracle(g, case):
    V, ld, nb, pnb, keep, eos_boost, lp, P, reorder = case
    n_clips = 5
    logits = make_logits(1000 + P + nb, MS - P, n_clips * nb, V, ld, eos_boost=eos_boost)
    for shared in (False, True):
        prompt = make_prompt(7 + P, 1 if shared else n_clips, P, V)
        kw = dict(max_steps=MS, nb=nb, pnb=pnb, keep=keep, lp=lp)
        tok, lps = device(g, logits, prompt, n_clips, V, reorder=reorder, **kw)
        ref_tok, ref_lp, _ = oracle(logits, prompt, n_clips, V=V, **kw)
        record("prefix_op_search", case=str(case), shared=shared, max_lp_diff=(lps - ref_lp).abs().max().item())
        assert torch.equal(tok, ref_tok), (tok, ref_tok)
        assert torch.allclose(lps, ref_lp, atol=2e-5, rtol=0)
        if P >= MS:
            assert (tok == EOS).all() and (lps == -1e5).all()


@pytest.mark.parametrize("nb,nrs,keep", [(4, 1, 1), (2, 3, 2), (1, 2, 1)])
def test_op_search_penalty_history_includes_the_prompt(g, nb, nrs, keep):
    V, ld, n_clips, P = 1000, 1024, 4, 3
    logits = make_logits(55 + nb, MS - P, n_clips * nrs * nb, V, ld, hot=6, eos_boost=1.0)
    prompt = make_prompt(3, n_clips, P, V, hot=6)  # prompt tokens among the boosted ones: the penalty decides
    kw = dict(max_steps=MS, nb=nb, pnb=2, keep=keep, lp=0.6)
    tok, lps = device(g, logits, prompt, n_clips, V, sample=g.SampleConfig(repetition_penalty=1.6, num_return_sequences=nrs), **kw)
    ref_tok, ref_lp, _ = oracle(logits, prompt, n_clips, V=V, rp=1.6, nrs=nrs, **kw)
    assert torch.equal(tok, ref_tok) and torch.allclose(lps, ref_lp, atol=2e-5, rtol=0)

    def penalise_generated_only(ids, x):  # negative control: the penalty's history omits the prompt
        for i in range(ids.shape[0]):
            for t in set(ids[i, P:].tolist()):
                x[i, t] = x[i, t] * 1.6 if x[i, t] < 0 else x[i, t] / 1.6
        return x
    bad_tok, bad_lp, _ = oracle(logits, prompt, n_clips, V=V, nrs=nrs, step_fn=penalise_generated_only, **kw)
    assert not (torch.equal(tok, bad_tok) and torch.allclose(lps, bad_lp, atol=2e-5, rtol=0))


@pytest.mark.parametrize("P,nb,nrs", [(2, 1, 2), (3, 3, 2), (4, 4, 1)])
def test_op_search_sampling_with_a_prompt(g, P, nb, nrs):
    V, ld, n_clips = 1000, 1024, 6
    smp = dict(top_k=30, top_p=0.9, temperature=0.8, seed=77 + P)
    logits = make_logits(91 + P, MS - P, n_clips * nrs * nb, V, ld, hot=6, eos_boost=2.0)
    prompt = make_prompt(5, 1, P, V, hot=6)
    kw = dict(max_steps=MS, nb=nb, pnb=2, keep=1, lp=0.6)
    tok, lps = device(g, logits, prompt, n_clips, V, sample=g.SampleConfig(do_sample=True, repetition_penalty=1.2,
                                                                           num_return_sequences=nrs, **smp), **kw)
    ref_tok, ref_lp, s = oracle(logits, prompt, n_clips, V=V, rp=1.2, nrs=nrs, sample=smp, **kw)
    unsure = s.unsure()
    sure = [e for e in range(n_clips * nrs) if e not in unsure]
    record("prefix_op_sampling", P=P, nb=nb, nrs=nrs, entries=n_clips * nrs, excluded=len(unsure))
    assert len(sure) >= (n_clips * nrs) // 2
    for e in sure:
        assert torch.equal(tok[e], ref_tok[e]) and torch.allclose(lps[e], ref_lp[e], atol=2e-5, rtol=0), e


def test_op_search_length_penalty_counts_the_prompt(g):
    V, ld, n_clips, P, nb = 1000, 1024, 8, 4, 4
    logits = make_logits(13, MS - P, n_clips * nb, V, ld, eos_boost=5.0)
    prompt = make_prompt(9, n_clips, P, V)
    kw = dict(max_steps=MS, nb=nb, pnb=2, keep=2, lp=1.0)
    tok, lps = device(g, logits, prompt, n_clips, V, **kw)
    ref_tok, ref_lp, _ = oracle(logits, prompt, n_clips, V=V, **kw)
    assert torch.equal(tok, ref_tok) and torch.allclose(lps, ref_lp, atol=2e-5, rtol=0)

    class GeneratedOnly(so.BeamHypotheses):  # negative control: the length penalty over the generated tokens only
        def add(self, hyp, sum_logprobs):
            super().add(hyp[P - 1:], sum_logprobs)
    bad_tok, bad_lp, _ = oracle(logits, prompt, n_clips, V=V, hyp_cls=GeneratedOnly, **kw)
    assert not torch.allclose(lps, bad_lp, atol=2e-5, rtol=0)


@pytest.mark.parametrize("nb,keep,lp", [(1, 1, 0.6), (4, 2, 0.6), (3, 1, 0.0)])
def test_op_search_p1_equals_the_search_without_a_prompt(g, nb, keep, lp):
    V, ld, n_clips = 30522, 30720, 4
    logits = make_logits(3 + nb, MS - 1, n_clips * nb, V, ld, eos_boost=4.0)
    sp = g.SearchConfig(beam_size=nb, max_steps=MS, length_penalty=lp, num_keep_best=keep)
    a = g.engine.op_search(logits.cuda(), V, n_clips, SOS, EOS, sp)
    b = g.engine.op_search(logits.cuda(), V, n_clips, SOS, EOS, sp, prefix=torch.tensor([[SOS]]))
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


# ------------------------------------------------------------------ model level
@pytest.fixture(scope="module")
def models(g):
    """GIT-base, 2-frame clips, seeded and perturbed weights: tied (upstream) and untied vocabulary head."""
    out = {}
    frames = torch.randn(6, 2, 3, 224, 224, generator=torch.Generator().manual_seed(9)).cuda()
    for tied in (True, False):
        cfg = go.GitConfig(num_image_with_embedding=2, tie_output=tied)
        sd = go.init_state_dict(cfg, seed=41 if tied else 42, temporal_std=0.02, perturb=True)
        teacher = g.GenerativeImageTextTeacher.from_random_init({"num_image_with_embedding": 2}, state_dict=sd)
        eng = teacher.model.engine()
        vf = eng.encode(frames[:4])
        out[tied] = (cfg, sd, teacher.model, eng, frames, vf)
    return out


def sconf(g, nb, ms, reorder=False):
    return g.SearchConfig(beam_size=nb, max_steps=ms, reorder_cache=reorder)


def oracle_model(sd, cfg, vf, prompt, nb, ms):
    B = vf.shape[0]
    state = go.DecodingState(sd, cfg, vf.cpu(), reorder_cache=False)
    with torch.no_grad():
        dec, lps, saved = so.search(prompt.long().expand(B, prompt.shape[1]), state, eos_index=cfg.eos_index, max_steps=ms,
                                    beam_size=nb, length_penalty=cfg.length_penalty, per_node_beam_size=2, save_logits=True)
    return dec, lps, torch.from_numpy(np.array(saved))


PROMPTS = [(2, False), (4, True), (9, False), (9, True)]


@pytest.mark.parametrize("P,shared", PROMPTS)
@pytest.mark.parametrize("nb", [1, 4])
def test_model_parity_tied_head(g, models, P, shared, nb):
    cfg, sd, m, eng, frames, vf = models[True]
    ms = P + 6
    prompt = make_prompt(P + 17, 1 if shared else 4, P, cfg.vocab_size)
    eng.set_visual_features(vf)
    tok, lps, logits = eng.decode(4, sconf(g, nb, ms), save_logits=True, prefix=prompt)
    ref_tok, ref_lp, ref_logits = oracle_model(sd, cfg, vf, prompt, nb, ms)
    d0 = (logits[0, :, :cfg.vocab_size].cpu() - ref_logits[0]).abs()
    sigma = ref_logits[0].std().item()
    record("prefix_model_tied", P=P, shared=shared, nb=nb, step0_max_over_sigma=d0.max().item() / sigma,
           step0_mean_over_sigma=d0.mean().item() / sigma)
    assert d0.max().item() < 0.15 * sigma and d0.mean().item() < 0.03 * sigma
    assert torch.equal(tok[:, 0].long().cpu(), ref_tok)
    assert torch.allclose(lps.cpu(), ref_lp, atol=2e-2, rtol=0)


def _greedy_margin_check(tok, ref_tok, ref_logits, P, sigma):
    """Tokens equal while the decoders agree; a disagreement only where the oracle's top-2 margin is below ROBUST sigma."""
    top2 = ref_logits.topk(2, dim=-1).values
    margin = (top2[..., 0] - top2[..., 1]) / sigma  # [steps, rows]
    robust_pos = 0
    for b in range(tok.shape[0]):
        for t in range(P, tok.shape[1]):
            s = t - P
            if s >= margin.shape[0]:
                break
            if tok[b, t] != ref_tok[b, t]:
                assert margin[s, b].item() < ROBUST, (b, t, margin[s, b].item())
                break
            robust_pos += int(margin[s, b].item() >= ROBUST)
            if ref_tok[b, t] == EOS:
                break
    return robust_pos


@pytest.mark.parametrize("P,shared", PROMPTS)
def test_model_parity_untied_head_margin_rule(g, models, P, shared):
    cfg, sd, m, eng, frames, vf = models[False]
    ms = P + 6
    prompt = make_prompt(P + 29, 1 if shared else 4, P, cfg.vocab_size)
    eng.set_visual_features(vf)
    tok, lps, logits = eng.decode(4, sconf(g, 1, ms), save_logits=True, prefix=prompt)
    ref_tok, ref_lp, ref_logits = oracle_model(sd, cfg, vf, prompt, 1, ms)
    sigma = ref_logits[0].std().item()
    d0 = (logits[0, :, :cfg.vocab_size].cpu() - ref_logits[0]).abs()
    assert d0.max().item() < 0.15 * sigma and d0.mean().item() < 0.03 * sigma
    n = _greedy_margin_check(tok[:, 0].long().cpu(), ref_tok, ref_logits, P, sigma)
    record("prefix_model_untied", P=P, shared=shared, robust_positions=n, step0_max_over_sigma=d0.max().item() / sigma)


@pytest.mark.parametrize("tied", [True, False])
def test_model_parity_against_the_package_host_loop(g, models, tied):
    """The package's own generic host search over gitb200_decode_step (one token per step through the prompt)."""
    cfg, sd, m, eng, frames, vf = models[tied]
    P, ms = 4, 10
    prompt = make_prompt(5, 4, P, cfg.vocab_size)
    m.decoder.max_steps, m.decoder.beam_size = ms, 1
    m.prev_encoded_layers = None
    m._vf_token = None
    step = functools.partial(m.decoding_step, vf, None, None)
    host_tok, host_lp, host_logits = m.decoder.search(prompt.long().cuda(), step)
    host_logits = torch.from_numpy(np.array(host_logits))
    eng.set_visual_features(vf)
    tok, lps, logits = eng.decode(4, sconf(g, 1, ms), save_logits=True, prefix=prompt)
    sigma = host_logits[0].std().item()
    d0 = (logits[0, :, :cfg.vocab_size].cpu() - host_logits[0]).abs()
    record("prefix_vs_host_loop", tied=tied, step0_max_over_sigma=d0.max().item() / sigma)
    assert d0.max().item() < 0.15 * sigma and d0.mean().item() < 0.03 * sigma
    _greedy_margin_check(tok[:, 0].long().cpu(), host_tok.long().cpu(), host_logits, P, sigma)


def test_infer_device_prefix_matches_the_oracle(g, models):
    cfg, sd, m, eng, frames, vf = models[True]
    m.decoder.max_steps, m.decoder.beam_size = 10, 4
    prompt = make_prompt(8, 4, 3, cfg.vocab_size)
    out = m.infer({"prefix": prompt}, vf, None, {"device_prefix": True})
    ref_tok, ref_lp, _ = oracle_model(sd, cfg, vf, prompt, 4, 10)
    assert torch.equal(out["predictions"].cpu(), ref_tok[:, 3:]) and len(out["logits_dict"]) <= 10 - 3


def test_structure_shared_prompt_and_permutation(g, models):
    cfg, sd, m, eng, frames, vf = models[False]
    P, ms = 5, 12
    one = make_prompt(3, 1, P, cfg.vocab_size)
    eng.set_visual_features(vf)
    sp = sconf(g, 4, ms)
    a = eng.decode(4, sp, save_logits=True, prefix=one)
    b = eng.decode(4, sp, save_logits=True, prefix=one.expand(4, P).contiguous())
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    per = make_prompt(4, 4, P, cfg.vocab_size)
    c = eng.decode(4, sp, prefix=per)
    perm = torch.tensor([2, 0, 3, 1])
    eng.set_visual_features(vf[perm.cuda()])
    d = eng.decode(4, sp, prefix=per[perm])
    assert torch.equal(d[0], c[0][perm.cuda()]) and torch.equal(d[1], c[1][perm.cuda()])


@pytest.mark.parametrize("n_clips,P", [(1, 2), (1, 5), (2, 3), (1, 6), (4, 9)])
def test_prefill_skinny_and_tensor_core_rows(g, models, n_clips, P):
    """Prefills of <= 4 rows run the fused skinny path, larger ones the tensor-core GEMMs; both match the oracle."""
    cfg, sd, m, eng, frames, vf = models[True]
    ms = P + 4
    prompt = make_prompt(P, n_clips, P, cfg.vocab_size)
    eng.set_visual_features(vf[:n_clips])
    tok, lps, logits = eng.decode(n_clips, sconf(g, 2, ms), save_logits=True, prefix=prompt)
    ref_tok, _, ref_logits = oracle_model(sd, cfg, vf[:n_clips], prompt, 2, ms)
    sigma = ref_logits[0].std().item()
    d0 = (logits[0, :, :cfg.vocab_size].cpu() - ref_logits[0]).abs()
    record("prefix_prefill_rows", rows=n_clips * (P - 1), step0_max_over_sigma=d0.max().item() / sigma)
    assert d0.max().item() < 0.15 * sigma and torch.equal(tok[:, 0].long().cpu(), ref_tok)


def test_kv_only_prefill_writes_no_logits(g, models):
    """The saved-logits buffer gets exactly max_steps - P steps; a canary step behind them stays untouched."""
    cfg, sd, m, eng, frames, vf = models[True]
    P, ms, nb = 4, 9, 2
    eng.set_visual_features(vf[:2])
    eng.set_early_exit(0)
    try:
        buf = torch.full((ms - P + 1, 2 * nb, eng.ld), float("nan"), device="cuda")
        tok = torch.empty(2, 1, ms, dtype=torch.int32, device="cuda")
        lp = torch.empty(2, 1, device="cuda")
        pre = make_prompt(1, 2, P, cfg.vocab_size).int().contiguous()
        c = sconf(g, nb, ms).to_c()
        rc = eng.lib.gitb200_decode_prefix(eng.h, ctypes.byref(c), None, ctypes.c_void_p(pre.data_ptr()), 2, P,
                                           ctypes.c_void_p(tok.data_ptr()), ctypes.c_void_p(lp.data_ptr()),
                                           ctypes.c_void_p(buf.data_ptr()), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0
        torch.cuda.synchronize()
        assert eng.last_decode_steps() == ms - P
        assert torch.isfinite(buf[: ms - P]).all() and torch.isnan(buf[ms - P]).all()
    finally:
        eng.set_early_exit(4)


@pytest.mark.parametrize("nb", [1, 2, 3, 4])
@pytest.mark.parametrize("reorder", [False, True])
@pytest.mark.parametrize("P", [2, 3])
def test_persistent_kernel_with_a_prompt(g, models, nb, reorder, P):
    cfg, sd, m, eng, frames, vf = models[False]
    prompt = make_prompt(P * 11 + nb, 1, P, cfg.vocab_size)
    eng.set_visual_features(vf[:1])
    sp = sconf(g, nb, 12, reorder)
    a = eng.decode(1, sp, prefix=prompt)
    eng.set_persistent_decode(False)
    try:
        b = eng.decode(1, sp, prefix=prompt)
    finally:
        eng.set_persistent_decode(True)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_p1_is_the_existing_path_bit_for_bit(g, models):
    cfg, sd, m, eng, frames, vf = models[True]
    sos = torch.tensor([[cfg.sos_index]])
    for nb, n, save in ((4, 4, True), (1, 1, False), (4, 1, False), (2, 3, True)):
        sp = sconf(g, nb, 10)
        eng.set_visual_features(vf[:n])
        a = eng.decode(n, sp, save_logits=save)
        b = eng.decode(n, sp, save_logits=save, prefix=sos)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and (not save or torch.equal(a[2], b[2]))
        x = eng.caption(frames[:n], sp, save_logits=save)
        y = eng.caption(frames[:n], sp, save_logits=save, prefix=sos)
        assert torch.equal(x[0], y[0]) and torch.equal(x[1], y[1]) and (not save or torch.equal(x[2], y[2]))
    smp = g.SampleConfig(do_sample=True, top_k=20, top_p=0.9, repetition_penalty=1.2, num_return_sequences=2, seed=5)
    sp = sconf(g, 2, 10)
    x = eng.caption(frames[:2], sp, save_logits=True, sample=smp)
    y = eng.caption(frames[:2], sp, save_logits=True, sample=smp, prefix=sos)
    assert all(torch.equal(u, v) for u, v in zip(x, y))


def _caption_prefix_raw(g, eng, clips, sp, prompt, tok, lp, stream):
    c = sp.to_c()
    pre = prompt.int().contiguous()
    return eng.lib.gitb200_caption_prefix(eng.h, ctypes.c_void_p(clips.data_ptr()), clips.shape[0], clips.shape[1], ctypes.byref(c),
                                          None, ctypes.c_void_p(pre.data_ptr()), pre.shape[0], pre.shape[1],
                                          ctypes.c_void_p(tok.data_ptr()), ctypes.c_void_p(lp.data_ptr()), None,
                                          ctypes.c_void_p(stream.cuda_stream))


def test_graph_replay_latency_mode_caption(g, models):
    cfg, sd, m, eng, frames, vf = models[True]
    sp = sconf(g, 4, 10)
    clips = frames[:2].contiguous()
    tok = torch.empty(2, 1, 10, dtype=torch.int32, device="cuda")
    lp = torch.empty(2, 1, device="cuda")
    prompts = [make_prompt(s, 2, 3, cfg.vocab_size) for s in (1, 1, 2, 3)]
    st = torch.cuda.Stream()
    outs = []
    with torch.cuda.stream(st):
        n0 = eng.lib.gitb200_graph_launches(eng.h)
        for p in prompts:
            assert _caption_prefix_raw(g, eng, clips, sp, p, tok, lp, st) == 0
            outs.append((tok.clone(), lp.clone()))
        st.synchronize()
        assert eng.lib.gitb200_graph_launches(eng.h) >= n0 + 2
    eng.set_graph_max_clips(0)
    eng.set_graph_segments(False)
    try:
        for p, (t, l) in zip(prompts[2:], outs[2:]):
            e = eng.caption(clips, sp, prefix=p)
            assert torch.equal(e[0], t) and torch.equal(e[1], l)
    finally:
        eng.set_graph_max_clips(8)
        eng.set_graph_segments(True)
    assert not torch.equal(outs[2][0], outs[3][0])


def test_graph_replay_segmented_batch(g, models):
    cfg, sd, m, eng, frames, vf = models[False]
    sp = sconf(g, 2, 10)
    eng.set_graph_max_clips(2)
    st = torch.cuda.Stream()
    try:
        outs = []
        with torch.cuda.stream(st):
            n0 = eng.lib.gitb200_graph_launches(eng.h)
            for s in (1, 2, 3):
                eng.set_visual_features(vf)
                outs.append(eng.decode(4, sp, prefix=make_prompt(s, 4, 5, cfg.vocab_size)))
            st.synchronize()
            assert eng.lib.gitb200_graph_launches(eng.h) > n0
        eng.set_graph_segments(False)
        for s, o in zip((2, 3), outs[1:]):
            eng.set_visual_features(vf)
            e = eng.decode(4, sp, prefix=make_prompt(s, 4, 5, cfg.vocab_size))
            assert torch.equal(e[0], o[0]) and torch.equal(e[1], o[1])
    finally:
        eng.set_graph_max_clips(8)
        eng.set_graph_segments(True)


def test_sampling_penalty_and_nrs_with_a_prompt_model_level(g, models):
    cfg, sd, m, eng, frames, vf = models[False]
    P, nb, nrs, ms = 3, 2, 2, 10
    smp = dict(top_k=30, top_p=0.9, temperature=0.8, seed=31)
    prompt = make_prompt(6, 1, P, cfg.vocab_size)
    eng.set_visual_features(vf[:2])
    eng.set_early_exit(0)
    try:
        tok, lps, logits = eng.decode(2, sconf(g, nb, ms), save_logits=True, prefix=prompt,
                                      sample=g.SampleConfig(do_sample=True, repetition_penalty=1.2, num_return_sequences=nrs, **smp))
    finally:
        eng.set_early_exit(4)
    assert logits.shape[0] == ms - P
    ref_tok, ref_lp, s = oracle(logits.cpu(), prompt, 2, V=cfg.vocab_size, max_steps=ms, nb=nb, pnb=2, keep=1, lp=0.6, rp=1.2,
                                nrs=nrs, sample=smp)
    sure = [e for e in range(2 * nrs) if e not in s.unsure()]
    record("prefix_sampling_model", entries=2 * nrs, excluded=2 * nrs - len(sure))
    assert sure
    for e in sure:
        assert torch.equal(tok[e].long().cpu(), ref_tok[e]) and torch.allclose(lps[e].cpu(), ref_lp[e], atol=2e-5, rtol=0)


# ------------------------------------------------------------------ negative controls on the decoder side
def _first_step_logits(sd, cfg, vf, prompt, *, shift=0, prompt_kv_rows=None):
    """The oracle's first-step logits [B, V] for one row per clip, with a plausible bug: prefill positions shifted by `shift`,
    or no prompt K/V at all (what the rows other than beam 0 would see if only beam 0 got them)."""
    P = prompt.shape[1]
    vfc = vf.cpu()
    with torch.no_grad():
        nv = go.project_visual(sd, cfg, vfc).shape[1]
        if shift:
            text = go.embed_text(sd, cfg, torch.cat([prompt[:, :1]] * shift + [prompt], 1).long())[:, shift:shift + P - 1]
            x = torch.cat([go.project_visual(sd, cfg, vfc), text], 1)
            mask = go.prefix_lm_mask(nv, P - 1, x.dtype)
            hist = [x]
            for i in range(cfg.num_layers):
                x = go.bert_layer(x, x, mask, sd, f"textual.transformer.encoder.layer.{i}.", cfg.attention_heads, cfg.bert_ln_eps)
                hist.append(x)
        else:
            _, hist = go.textual_forward(sd, cfg, vfc, prompt[:, :P - 1].long())
            if prompt_kv_rows == 0:
                hist = [h[:, :nv] for h in hist]
        logits, _ = go.textual_forward(sd, cfg, vfc, prompt.long(), hist)
    return logits[:, -1].float()


def test_negative_controls_shifted_positions_and_beam0_only_kv(g, models):
    """Over 394 visual keys the prompt's keys hold too little attention for a wrong prompt K/V to move the logits past the
    tolerance (oracle: 0.010 sigma for shifted positions, 0.017 sigma without prompt K/V).  Over the first 8 visual tokens
    they hold about a third: 0.30 / 0.65 sigma, so there the device must match the right reference and miss both wrong ones."""
    cfg, sd, m, eng, frames, vf = models[False]
    P, nb = 5, 4
    prompt = make_prompt(12, 4, P, cfg.vocab_size)
    vf = vf[:, :8].contiguous()
    eng.set_visual_features(vf)
    _, _, logits = eng.decode(4, sconf(g, nb, P + 3), save_logits=True, prefix=prompt)
    dev = logits[0, :, :cfg.vocab_size].cpu().view(4, nb, -1)
    good = _first_step_logits(sd, cfg, vf, prompt)
    sigma = good.std().item()
    for b in range(nb):  # every beam row saw the prompt
        assert (dev[:, b] - good).abs().max().item() < 0.15 * sigma
    shifted = _first_step_logits(sd, cfg, vf, prompt, shift=1)
    no_kv = _first_step_logits(sd, cfg, vf, prompt, prompt_kv_rows=0)
    record("prefix_negative_controls", shifted_max_over_sigma=(dev[:, 0] - shifted).abs().max().item() / sigma,
           beam0_only_max_over_sigma=(dev[:, 1] - no_kv).abs().max().item() / sigma)
    assert (dev[:, 0] - shifted).abs().max().item() > 0.15 * sigma
    assert (dev[:, 1] - no_kv).abs().max().item() > 0.15 * sigma


# ------------------------------------------------------------------ rejections
def test_rejections_leave_the_outputs_untouched(g, models):
    cfg, sd, m, eng, frames, vf = models[True]
    eng.set_visual_features(vf[:2])
    sp = sconf(g, 2, 8)
    c = sp.to_c()
    good = make_prompt(1, 2, 3, cfg.vocab_size).int()
    bad_tok = good.clone()
    bad_tok[1, 2] = cfg.vocab_size
    neg_tok = good.clone()
    neg_tok[0, 1] = -1
    long_p = torch.full((1, 1025), SOS, dtype=torch.int32)
    cases = [(good, 2, 0, "P must be >= 1"), (None, 2, 3, "NULL"), (good, 3, 3, "prefix_rows"), (bad_tok, 2, 3, "outside"),
             (neg_tok, 2, 3, "outside"), (long_p, 1, 1025, "text positions")]
    tok = torch.full((2, 1, 8), -7, dtype=torch.int32, device="cuda")
    lp = torch.full((2, 1), -7.0, device="cuda")
    lg = torch.full((8, 4, eng.ld), -7.0, device="cuda")
    ops = torch.zeros(7, 4, 1024, device="cuda")
    n0 = eng.launch_count()
    for pre, rows, P, named in cases:
        ptr = ctypes.c_void_p(pre.data_ptr()) if pre is not None else None
        rc = eng.lib.gitb200_decode_prefix(eng.h, ctypes.byref(c), None, ptr, rows, P, ctypes.c_void_p(tok.data_ptr()),
                                           ctypes.c_void_p(lp.data_ptr()), ctypes.c_void_p(lg.data_ptr()), None)
        assert rc != 0 and named.encode() in eng.lib.gitb200_last_error(eng.h), named
        rc = eng.lib.gitb200_caption_prefix(eng.h, ctypes.c_void_p(frames.data_ptr()), 2, 2, ctypes.byref(c), None, ptr, rows, P,
                                            ctypes.c_void_p(tok.data_ptr()), ctypes.c_void_p(lp.data_ptr()), None, None)
        assert rc != 0 and named.encode() in eng.lib.gitb200_last_error(eng.h), named
        if named != "text positions":  # the operator search has no position table
            with pytest.raises(g.GitB200Error, match=re.escape(named)):
                rc = g.engine._lib.load().gitb200_op_search_prefix(
                    ctypes.c_void_p(ops.data_ptr()), 1024, 1000, 2, EOS, ctypes.byref(c),
                    None, ptr, rows, P, ctypes.c_void_p(tok.data_ptr()), ctypes.c_void_p(lp.data_ptr()), None)
                g.engine._lib.check(rc, None, "op_search_prefix")
    bad = g.SampleConfig(do_sample=True, top_k=5, top_p=0.9, temperature=0.0, seed=1)
    with pytest.raises(g.GitB200Error, match="temperature"):
        eng.decode(2, sp, sample=bad, prefix=good)
    with pytest.raises(g.GitB200Error, match="temperature"):
        eng.caption(frames[:2], sp, sample=bad, prefix=good)
    torch.cuda.synchronize()
    assert eng.launch_count() == n0
    assert (tok == -7).all() and (lp == -7).all() and (lg == -7).all()
