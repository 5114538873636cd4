"""GPU tests of prompted captions in the multi-stream pool and the single streaming window (gitb200_streams_caption_prefix,
gitb200_stream_caption_prefix, MultiStreamCaptioner / StreamingCaptioner prompts): a prompted caption of k windows is
gitb200_decode_prefix (batch['prefix'], model.py:432-437) on those windows' features, each camera drawing with its own key at
Philox step P - 1.  The oracles are test_gpu_prefix's: oracle/git_oracle.DecodingState with the whole prompt in its first call,
and oracle/search_oracle.search over the device's saved scores with the race sampler.  GIT-base, 2-frame windows, 16 cameras,
tied and untied heads.  Deviations go to the parity-metrics file through record()."""
import ctypes

import pytest
import torch

from oracle import git_oracle as go
from test_gpu_parity import record
from test_gpu_prefix import _greedy_margin_check, make_prompt, oracle, oracle_model

pytestmark = pytest.mark.gpu

N_FRAMES, S = 2, 16
SMP = dict(do_sample=True, top_k=30, top_p=0.9, temperature=0.8, repetition_penalty=1.2)


@pytest.fixture(scope="module")
def g():
    import gitb200
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return gitb200


@pytest.fixture(scope="module")
def models(g):
    """GIT-base geometry, 2-frame windows, tied (upstream) and untied head; a pool of 16 cameras, each holding 2 frames."""
    frames = torch.randn(N_FRAMES, S, 3, 224, 224, generator=torch.Generator().manual_seed(19)).cuda()
    out = {}
    for tied in (True, False):
        cfg = go.GitConfig(num_image_with_embedding=N_FRAMES, tie_output=tied)
        sd = go.init_state_dict(cfg, seed=41 if tied else 42, temporal_std=0.02, perturb=True)
        eng = g.Engine(g.make_config({"num_image_with_embedding": N_FRAMES}, cfg.sos_index, cfg.eos_index), 0)
        eng.load_state_dict(sd)
        eng.streams_configure(S)
        for r in range(N_FRAMES):
            eng.streams_push(list(range(S)), frames[r].contiguous())
        out[tied] = (cfg, sd, eng, frames)
    return out


def keys_of(*v):
    return [0x9E3779B97F4A7C15 * (x + 1) % 2 ** 64 for x in v]


def windows(eng, ids):
    return torch.stack([eng.streams_window(i) for i in ids])


def pad_steps(logits, n):
    """Saved logits of a search that stopped early, padded to n steps (the padding is never read: every entry is done)."""
    steps = logits.shape[0]
    return torch.cat([logits, logits[-1:].expand(n - steps, -1, -1)]) if steps < n else logits


def same(a, b):
    return len(a) == len(b) and all((x is None and y is None) or torch.equal(x, y) for x, y in zip(a, b))


# ------------------------------------------------------------------ 1. oracle parity
@pytest.mark.parametrize("tied,nb", [(True, 1), (True, 4), (False, 1)])
@pytest.mark.parametrize("P,shared", [(3, False), (5, True)])
def test_oracle_parity(g, models, tied, nb, P, shared):
    cfg, sd, eng, _ = models[tied]
    ids = [5, 0, 11, 3]
    ms = P + 6
    prompt = make_prompt(P + 31, 1 if shared else len(ids), P, cfg.vocab_size)
    tok, lps, logits = eng.streams_caption(ids, g.SearchConfig(beam_size=nb, max_steps=ms), sample=g.SampleConfig(),
                                           save_logits=True, prefix=prompt)
    assert tok.shape == (4, 1, ms) and logits.shape[1:] == (4 * nb, eng.ld) and logits.shape[0] <= ms - P
    assert torch.equal(tok[:, 0, :P].long().cpu(), prompt.long().expand(4, P))  # the tokens include the prompt
    vf = windows(eng, ids)
    ref_tok, ref_lp, ref_logits = oracle_model(sd, cfg, vf, prompt, nb, ms)
    sigma = ref_logits[0].std().item()
    d0 = (logits[0, :, :cfg.vocab_size].cpu() - ref_logits[0]).abs()
    record("multistream_prefix_oracle", tied=tied, nb=nb, P=P, shared=shared, step0_max_over_sigma=d0.max().item() / sigma,
           step0_mean_over_sigma=d0.mean().item() / sigma)
    assert d0.max().item() < 0.15 * sigma and d0.mean().item() < 0.03 * sigma
    if tied:
        exact = [j for j in range(4) if torch.equal(tok[j, 0].long().cpu(), ref_tok[j])]
        record("multistream_prefix_oracle_tied", nb=nb, P=P, shared=shared, cameras=4, exact_sequences=len(exact))
        assert torch.allclose(lps[exact].cpu(), ref_lp[exact], atol=2e-2, rtol=0)
        # greedy: every sequence.  Beam 4 keeps four hypotheses of this random model's repeated-token captions whose scores
        # differ by little, and the bf16 device and the fp32 oracle may keep different ones early (measured on one B200:
        # 4 of 4 cameras exact at P = 3 per camera, 2 of 4 at P = 5 shared).  Whatever the search does there, the pool
        # does exactly what gitb200_decode_prefix does on the same windows.
        if nb == 1:
            assert len(exact) == 4, exact
        eng.set_visual_features(vf.cuda())
        assert same((tok, lps, logits), eng.decode(4, g.SearchConfig(beam_size=nb, max_steps=ms), save_logits=True, prefix=prompt))
    else:
        n = _greedy_margin_check(tok[:, 0].long().cpu(), ref_tok, ref_logits, P, sigma)
        record("multistream_prefix_oracle_untied", P=P, shared=shared, robust_positions=n)
    if tied and nb == 1 and not shared:
        # negative control: the prompts rolled by one camera
        bad_tok, _, _ = oracle_model(sd, cfg, vf, prompt.roll(1, 0), nb, ms)
        differing = sum(not torch.equal(tok[j, 0].long().cpu(), bad_tok[j]) for j in range(4))
        record("multistream_prefix_negative_control", control="rolled_prompts", cameras=4, differing=differing)
        assert differing == 4, differing


# ------------------------------------------------------------------ 2. the pool is decode_prefix on the windows
@pytest.mark.parametrize("nb,P,shared", [(1, 3, False), (4, 5, True), (2, 4, False)])
def test_pool_equals_decode_prefix(g, models, nb, P, shared):
    cfg, _, eng, _ = models[False]
    ids = [(7 * j + 2) % S for j in range(12)]
    ms = 12
    sp = g.SearchConfig(beam_size=nb, max_steps=ms)
    prompt = make_prompt(P, 1 if shared else 12, P, cfg.vocab_size)
    a = eng.streams_caption(ids, sp, sample=g.SampleConfig(), save_logits=True, prefix=prompt)
    eng.set_visual_features(windows(eng, ids))
    b = eng.decode(12, sp, save_logits=True, prefix=prompt)
    assert a[2].shape[0] >= 1 and same(a, b), (a[2].shape, b[2].shape)
    c = eng.streams_caption(ids, sp, prefix=prompt)  # without saved logits: the graphed path
    assert same(c, a[:2])


# ------------------------------------------------------------------ 3. k = 1: pool, single window, decode, persistent kernel
def _single(eng, frames, sid):
    """Camera sid's frames pushed one at a time into its pool window and into the single window (one frame per ViT batch)."""
    eng.streams_reset([sid])
    eng.stream_reset()
    for r in range(N_FRAMES):
        eng.streams_push([sid], frames[r, sid][None].contiguous())
        eng.stream_push(frames[r, sid])


@pytest.mark.parametrize("nb", [1, 2, 3, 4])
@pytest.mark.parametrize("P", [2, 3])
def test_k1_pool_single_window_decode_and_persistent_kernel(g, models, nb, P):
    cfg, _, eng, frames = models[False]
    sid = 6
    _single(eng, frames, sid)
    prompt = make_prompt(P * 13 + nb, 1, P, cfg.vocab_size)
    sp = g.SearchConfig(beam_size=nb, max_steps=12)
    a = eng.streams_caption([sid], sp, prefix=prompt)
    b = eng.stream_caption(sp, prefix=prompt)
    eng.set_visual_features(eng.streams_window(sid)[None])
    c = eng.decode(1, sp, prefix=prompt)[:2]
    # the persistent kernel runs the whole search in a few launches; the launch sequence takes dozens per step
    eng.set_graph_max_clips(0)
    eng.set_graph_segments(False)
    try:
        eng.launch_count(reset=True)
        d = eng.streams_caption([sid], sp, prefix=prompt)
        on = eng.launch_count(reset=True)
        eng.set_persistent_decode(False)
        e = eng.streams_caption([sid], sp, prefix=prompt)
        off = eng.launch_count(reset=True)
        f = eng.stream_caption(sp, prefix=prompt)
    finally:
        eng.set_persistent_decode(True)
        eng.set_graph_max_clips(8)
        eng.set_graph_segments(True)
    record("multistream_prefix_persistent", nb=nb, P=P, launches_persistent=on, launches_sequence=off)
    assert off - on >= 10 * (12 - P), (on, off)  # dozens of launches for each of the max_steps - P steps
    for name, x in (("stream_caption", b), ("decode", c), ("eager", d), ("no_persistent", e), ("single_no_persistent", f)):
        assert same(a, x), (name, a, x)


def test_k1_saved_logits_pool_single_window_decode(g, models):
    cfg, _, eng, frames = models[False]
    sid = 9
    _single(eng, frames, sid)
    prompt = make_prompt(4, 1, 4, cfg.vocab_size)
    sp = g.SearchConfig(beam_size=3, max_steps=12)
    a = eng.streams_caption([sid], sp, sample=g.SampleConfig(), save_logits=True, prefix=prompt)
    b = eng.stream_caption(sp, sample=g.SampleConfig(), save_logits=True, prefix=prompt)
    eng.set_visual_features(eng.streams_window(sid)[None])
    c = eng.decode(1, sp, sample=g.SampleConfig(), save_logits=True, prefix=prompt)
    assert same(a, b) and same(a, c)


# ------------------------------------------------------------------ 4. sampling with a prompt
def test_sampling_with_a_prompt_matches_the_oracle_per_camera(g, models):
    cfg, _, eng, _ = models[False]
    k, nb, nrs, P, ms = 12, 2, 2, 3, 11
    ids = [(5 * j + 3) % S for j in range(k)]
    keys = keys_of(*range(300, 300 + k))
    prompt = make_prompt(77, k, P, cfg.vocab_size)
    sp = g.SearchConfig(beam_size=nb, max_steps=ms)
    smp = g.SampleConfig(num_return_sequences=nrs, **SMP)
    tok, lps, logits = eng.streams_caption(ids, sp, sample=smp, keys=keys, save_logits=True, prefix=prompt)
    tok, lps, full = tok.long().cpu(), lps.cpu(), pad_steps(logits.cpu(), ms - P)
    assert tok.shape == (k * nrs, 1, ms) and full.shape[1] == k * nrs * nb
    kw = dict(V=cfg.vocab_size, max_steps=ms, nb=nb, pnb=2, keep=1, lp=0.6, rp=1.2, nrs=nrs)
    rows = nrs * nb
    sure, other_key = [], 0
    for j in range(k):
        smp_j = dict(top_k=30, top_p=0.9, temperature=0.8, seed=keys[j])
        ref_tok, ref_lp, s = oracle(full[:, j * rows:(j + 1) * rows], prompt[j:j + 1], 1, sample=smp_j, **kw)
        bad_tok, _, _ = oracle(full[:, j * rows:(j + 1) * rows], prompt[j:j + 1], 1, sample=dict(smp_j, seed=keys[(j + 1) % k]), **kw)
        for r in range(nrs):
            if r in s.unsure():
                continue
            e = j * nrs + r
            sure.append(e)
            assert torch.equal(tok[e], ref_tok[r]), (j, r, tok[e], ref_tok[r])
            assert torch.allclose(lps[e], ref_lp[r], atol=2e-5, rtol=0), (j, r, lps[e], ref_lp[r])
            other_key += not torch.equal(tok[e], bad_tok[r])
    record("multistream_prefix_sampling_oracle", entries=k * nrs, sure=len(sure), other_key_differs=other_key)
    assert len(sure) >= k * nrs // 2
    assert other_key > len(sure) // 2  # negative control: the neighbour's key

    # k = 1 equals decode_prefix with seed = the key
    sid, x = ids[0], keys[0]
    a = eng.streams_caption([sid], sp, sample=smp, keys=[x], save_logits=True, prefix=prompt[:1])
    eng.set_visual_features(eng.streams_window(sid)[None])
    b = eng.decode(1, sp, sample=g.SampleConfig(seed=x, num_return_sequences=nrs, **SMP), save_logits=True, prefix=prompt[:1])
    assert same(a, b)


# ------------------------------------------------------------------ 5. invariance
def test_invariance_to_order_company_and_p1(g, models):
    cfg, _, eng, _ = models[False]
    sp = g.SearchConfig(beam_size=2, max_steps=10)
    smp = g.SampleConfig(num_return_sequences=2, **SMP)
    ids, keys = [0, 1, 2, 3, 4, 5], keys_of(10, 11, 12, 13, 14, 15)
    prompt = make_prompt(21, 6, 3, cfg.vocab_size)

    def run(i, k, p):
        t, l, _ = eng.streams_caption(i, sp, sample=smp, keys=k, prefix=p)
        return t.view(len(i), 2, -1), l.view(len(i), 2, -1)

    ta, la = run(ids, keys, prompt)
    perm = [4, 0, 5, 2, 1, 3]
    tp, lp_ = run([ids[p] for p in perm], [keys[p] for p in perm], prompt[perm])
    assert torch.equal(tp, ta[perm]) and torch.equal(lp_, la[perm])
    # camera 3 replaced by camera 9 (another window, prompt and key): every other camera unchanged
    other = prompt.clone()
    other[3] = make_prompt(99, 1, 3, cfg.vocab_size)[0]
    tr, lr = run([0, 1, 2, 9, 4, 5], keys[:3] + keys_of(99) + keys[4:], other)
    keep = [0, 1, 2, 4, 5]
    assert torch.equal(tr[keep], ta[keep]) and torch.equal(lr[keep], la[keep])
    assert not torch.equal(tr[3], ta[3])
    assert same(run(ids, keys, prompt), (ta, la))

    # P = 1 with SOS is the existing entry points, bit for bit
    sos = torch.tensor([[cfg.sos_index]])
    for i in ([7], ids, list(range(12))):
        k = keys_of(*range(len(i)))
        for nb in (1, 4):
            spn = g.SearchConfig(beam_size=nb, max_steps=9)
            assert same(eng.streams_caption(i, spn), eng.streams_caption(i, spn, prefix=sos))
            assert same(eng.streams_caption(i, spn, sample=smp, keys=k, save_logits=True),
                        eng.streams_caption(i, spn, sample=smp, keys=k, save_logits=True, prefix=sos))
    eng.stream_reset()
    for r in range(N_FRAMES):
        eng.stream_push(models[False][3][r, 4])
    assert same(eng.stream_caption(sp), eng.stream_caption(sp, prefix=sos))
    x = g.SampleConfig(seed=keys[0], num_return_sequences=2, **SMP)
    assert same(eng.stream_caption(sp, sample=x, save_logits=True), eng.stream_caption(sp, sample=x, save_logits=True, prefix=sos))


# ------------------------------------------------------------------ 6. graph replay
def _replays_equal_eager(g, eng, calls, sp, smp, max_clips):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    outs = []
    eng.set_graph_max_clips(max_clips)
    try:
        before = eng.lib.gitb200_graph_launches(eng.h)
        with torch.cuda.stream(side):
            for ids, keys, prompt in calls:
                outs.append(eng.streams_caption(ids, sp, sample=smp, keys=keys, prefix=prompt)[:2])
            side.synchronize()
        launched = eng.lib.gitb200_graph_launches(eng.h) - before
    finally:
        eng.set_graph_max_clips(8)
    eng.set_graph_max_clips(0)
    eng.set_graph_segments(False)
    try:
        for (ids, keys, prompt), o in zip(calls, outs):
            assert same(eng.streams_caption(ids, sp, sample=smp, keys=keys, prefix=prompt)[:2], o), (ids, prompt)
    finally:
        eng.set_graph_max_clips(8)
        eng.set_graph_segments(True)
    return outs, launched


@pytest.mark.parametrize("k,max_clips", [(1, 8), (3, 8), (12, 4)])
@pytest.mark.parametrize("sampled", [False, True])
def test_graph_replay_equals_eager_for_new_prompts_ids_and_keys(g, models, k, max_clips, sampled):
    cfg, _, eng, _ = models[False]
    sp = g.SearchConfig(beam_size=2, max_steps=9)
    smp = g.SampleConfig(num_return_sequences=2, **SMP) if sampled else None
    P = 3
    calls = [(list(range(k)) if i % 2 == 0 else list(range(S - k, S))[::-1], keys_of(*range(40 * i, 40 * i + k)),
              make_prompt(50 + i, k if i % 3 else 1, P, cfg.vocab_size)) for i in range(5)]
    outs, launched = _replays_equal_eager(g, eng, calls, sp, smp, max_clips)
    record("multistream_prefix_graphs", k=k, sampled=sampled, graph_launches=launched)
    assert launched >= 2, launched
    assert not torch.equal(outs[0][0], outs[2][0])  # same ids, new prompts (and keys)


def test_graph_replay_after_the_prompt_buffer_grows(g, models):
    """A prompt table larger than any before reallocates the prompt buffer: the graphs captured before it are dropped, not
    replayed into freed memory.  (The long prompts are sized above every earlier call of this module: 12 x (2 * 5 - 1).)"""
    cfg, _, eng, _ = models[False]
    for k, max_clips, big in ((3, 8, 30), (12, 4, 10)):  # prompt tables of 3 x 59, then 12 x 19 ints
        sp = g.SearchConfig(beam_size=2, max_steps=big + 4)
        short = [(list(range(k)), None, make_prompt(60 + i, k, 3, cfg.vocab_size)) for i in range(3)]
        long = [(list(range(S - k, S)), None, make_prompt(80 + i, k, big, cfg.vocab_size)) for i in range(3)]
        _, launched = _replays_equal_eager(g, eng, short + long + short, sp, None, max_clips)
        assert launched >= 4, (k, launched)


def test_replayed_call_reports_its_decode_steps(g, models):
    cfg, _, eng, _ = models[False]
    sp = g.SearchConfig(beam_size=2, max_steps=10)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for P in (1, 4, 4, 4):
            n0 = eng.lib.gitb200_graph_launches(eng.h)
            eng.streams_caption([1, 2, 3], sp, prefix=make_prompt(P, 3, P, cfg.vocab_size))
            replayed = eng.lib.gitb200_graph_launches(eng.h) > n0
        side.synchronize()
    assert replayed and eng.last_decode_steps() == 10 - 4


# ------------------------------------------------------------------ 7. rejections
def test_rejections_enqueue_nothing_and_change_nothing(g, models):
    cfg, _, eng, _ = models[False]
    lib, h = eng.lib, eng.h
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    sp = g.SearchConfig(beam_size=2, max_steps=8)
    spc = sp.to_c()
    smp = g.SampleConfig(**SMP)
    ids, keys = [0, 1, 2], keys_of(1, 2, 3)
    good = make_prompt(3, 3, 3, cfg.vocab_size)
    ref = eng.streams_caption(ids, sp, sample=smp, keys=keys, prefix=good)
    eng.streams_reset([14])
    eng.streams_push([14], torch.randn(1, 3, 224, 224, generator=torch.Generator().manual_seed(3)).cuda())
    frames = [eng.streams_frames(i) for i in range(S)]
    before = {i: eng.streams_window(i).clone() for i in (0, 1, 2, 14)}
    tok = torch.full((8, 1, 8), -7, dtype=torch.int32, device="cuda")
    lp = torch.full((8, 1), -7.0, device="cuda")
    logits = torch.full((8, 8, eng.ld), -7.0, device="cuda")
    eng.stream_reset()
    eng.stream_push(models[False][3][0, 0])
    torch.cuda.synchronize()

    def call(ids=ids, smp=smp, keys="auto", prefix=good, rows=None, P=None):
        arr = (ctypes.c_int32 * len(ids))(*ids)
        if keys == "auto":
            keys = (ctypes.c_uint64 * len(ids))(*keys_of(*range(len(ids))))
        pre = prefix.int().contiguous() if prefix is not None else None
        return lib.gitb200_streams_caption_prefix(
            h, arr, len(ids), ctypes.byref(spc), ctypes.byref(smp.to_c()) if smp is not None else None, keys,
            ctypes.c_void_p(pre.data_ptr()) if pre is not None else None, pre.shape[0] if rows is None else rows,
            pre.shape[1] if P is None else P, ctypes.c_void_p(tok.data_ptr()), ctypes.c_void_p(lp.data_ptr()),
            ctypes.c_void_p(logits.data_ptr()), s)

    def single(prefix=good[:1], P=None, smp=None):
        pre = prefix.int().contiguous() if prefix is not None else None
        return lib.gitb200_stream_caption_prefix(
            h, ctypes.byref(spc), ctypes.byref(smp.to_c()) if smp is not None else None,
            ctypes.c_void_p(pre.data_ptr()) if pre is not None else None, pre.shape[1] if P is None else P,
            ctypes.c_void_p(tok.data_ptr()), ctypes.c_void_p(lp.data_ptr()), ctypes.c_void_p(logits.data_ptr()), s)

    def err():
        return lib.gitb200_last_error(h).decode()

    out_of_vocab, negative = good.clone(), good.clone()
    out_of_vocab[1, 2] = cfg.vocab_size
    negative[2, 1] = -1
    too_long = make_prompt(5, 1, 1025, cfg.vocab_size)
    n0 = eng.launch_count()
    rejected = [
        (lambda: call(P=0), "P must be >= 1"), (lambda: call(prefix=None, rows=1, P=3), "NULL"),
        (lambda: call(rows=2), "prefix_rows"), (lambda: call(prefix=good[:2]), "prefix_rows"),
        (lambda: call(prefix=out_of_vocab), f"{cfg.vocab_size} at [1, 2]"), (lambda: call(prefix=negative), "-1 at [2, 1]"),
        (lambda: call(prefix=too_long), "exceeds"), (lambda: call(keys=None), "keys_host"),
        (lambda: call(smp=g.SampleConfig(**dict(SMP, temperature=0.0))), "temperature"),
        (lambda: call(ids=[0, 17]), "unknown"), (lambda: call(ids=[1, 1]), "twice"),
        (lambda: call(ids=[0, 14, 1]), "different lengths"),
        (lambda: single(P=0), "P must be >= 1"), (lambda: single(prefix=None, P=2), "NULL"),
        (lambda: single(prefix=out_of_vocab[1:2]), "outside"), (lambda: single(prefix=too_long), "exceeds"),
        (lambda: single(smp=g.SampleConfig(**dict(SMP, top_p=1.5))), "top_p"),
    ]
    for i, (fn, named) in enumerate(rejected):
        assert fn() == -1, i  # GITB200_ERR_INVALID
        assert named in err(), (i, named, err())
    assert eng.launch_count() == n0  # nothing was enqueued
    torch.cuda.synchronize()
    assert (tok == -7).all() and (lp == -7).all() and (logits == -7).all()
    assert [eng.streams_frames(i) for i in range(S)] == frames and eng.lib.gitb200_stream_frames(h) == 1
    for i, w in before.items():
        assert torch.equal(eng.streams_window(i), w), i
    assert same(eng.streams_caption(ids, sp, sample=smp, keys=keys, prefix=good), ref)
    with pytest.raises(g.GitB200Error, match="one row"):
        eng.stream_caption(sp, prefix=good)


# ------------------------------------------------------------------ 8. the captioner at the benchmark geometry
def test_captioner_groups_at_the_benchmark_geometry(g):
    """MultiStreamCaptioner with 6-frame sliding windows and 24 cameras in three groups (no prompt, P = 3, P = 5): each
    caption equals the engine's call for its group, and its text is what follows the prompt."""
    F6, n = 6, 24
    cfg = go.GitConfig(num_image_with_embedding=F6, tie_output=False)
    sd = go.init_state_dict(cfg, seed=23, temporal_std=0.02, perturb=True)
    teacher = g.GenerativeImageTextTeacher.from_random_init({"num_image_with_embedding": F6}, state_dict=sd)
    raw = torch.randint(0, 256, (F6, n, 96, 128, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(8)).cuda()
    q3, q5 = [cfg.sos_index, 2054, 2003], [cfg.sos_index, 2054, 2003, 1996, 2158]
    cap = g.MultiStreamCaptioner(teacher, n, stride=1, max_len=12, sliding=True, prompt=q5)
    groups = {0: list(range(0, n, 3)), 3: list(range(1, n, 3)), 5: list(range(2, n, 3))}
    for sid in groups[0]:
        cap.set_prompt(sid, None)
    for sid in groups[3]:
        cap.set_prompt(sid, q3)
    outs = [cap.push({s: raw[t, s] for s in range(n)}) for t in range(F6)]
    assert all(o == {} for o in outs[:-1]) and sorted(outs[-1]) == list(range(n))
    eng, tk = teacher.model.engine(), teacher.tokenizer
    for P, ids in groups.items():
        if P == 0:
            tok, _ = eng.streams_caption(ids, cap.search)
        else:
            prompt = torch.tensor([q3 if P == 3 else q5] * len(ids))
            tok, _ = eng.streams_caption(ids, cap.search, prefix=prompt)
            assert torch.equal(tok[:, 0, :P].cpu().long(), prompt)
        for j, sid in enumerate(ids):
            assert outs[-1][sid] == tk.decode(tok[j, 0, P:].tolist(), skip_special_tokens=True), (P, sid)
            if P:
                assert outs[-1][sid] != tk.decode(tok[j, 0].tolist(), skip_special_tokens=True), (P, sid)
    record("multistream_prefix_captioner", cameras=n, groups=len(groups))
