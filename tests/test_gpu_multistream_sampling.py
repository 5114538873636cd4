"""GPU tests of sampled captions in the multi-stream pool (gitb200_streams_caption_ext, gitb200_stream_caption_ext,
MultiStreamCaptioner(sample=...)): every camera draws with its own Philox key, so its caption depends on its window, its key,
the parameters and the call's row count only.  The oracle is test_gpu_sampling's: oracle/search_oracle.search on the
device's saved scores with the race sampler of tests/sampling_ref.py, one camera at a time (n_clips = 1, seed = its key:
clip word 0 is then exactly the pool's counter).  Untied GIT-base head with 2-frame windows (a tied head copies its input
with a wide margin, so its samples would prove little).  Deviations go to the parity-metrics file through record()."""
import ctypes

import pytest
import torch

from oracle import git_oracle as go
from sampling_ref import oracle_search
from test_gpu_parity import record

pytestmark = pytest.mark.gpu

N_FRAMES = 2
SMP = dict(do_sample=True, top_k=30, top_p=0.9, temperature=0.8, repetition_penalty=1.2)


@pytest.fixture(scope="module")
def g():
    import gitb200
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return gitb200


@pytest.fixture(scope="module")
def setup(g):
    """GIT-base geometry, untied head, 2-frame windows; a pool of 16 cameras, each holding 2 frames."""
    cfg = go.GitConfig(num_image_with_embedding=N_FRAMES, tie_output=False)
    sd = go.init_state_dict(cfg, seed=42, temporal_std=0.02, perturb=True)
    eng = g.Engine(g.make_config({"num_image_with_embedding": N_FRAMES}, cfg.sos_index, cfg.eos_index), 0)
    eng.load_state_dict(sd)
    frames = torch.randn(N_FRAMES, 16, 3, 224, 224, generator=torch.Generator().manual_seed(19)).cuda()
    fill(eng, frames)
    return cfg, sd, eng, frames


def fill(eng, frames):
    eng.streams_configure(frames.shape[1])
    for r in range(N_FRAMES):
        eng.streams_push(list(range(frames.shape[1])), frames[r].contiguous())


def keys_of(*v):
    return [0x9E3779B97F4A7C15 * (x + 1) % 2 ** 64 for x in v]


def full_steps(logits, ms):
    """Saved logits of a search that stopped early, padded to max_steps - 1 steps (the padding is never read: every entry is
    done by then)."""
    steps = logits.shape[0]
    return torch.cat([logits, logits[-1:].expand(ms - 1 - steps, -1, -1)]) if steps < ms - 1 else logits


def test_each_camera_matches_the_oracle_with_its_own_key(g, setup):
    cfg, _, eng, _ = setup
    k, nb, nrs, ms = 12, 2, 2, 10
    ids = [(5 * j + 3) % 16 for j in range(k)]
    keys = keys_of(*range(100, 100 + k))
    sp = g.SearchConfig(beam_size=nb, max_steps=ms)
    smp = g.SampleConfig(num_return_sequences=nrs, **SMP)
    tok, lps, logits = eng.streams_caption(ids, sp, sample=smp, keys=keys, save_logits=True)
    tok, lps, full = tok.long().cpu(), lps.cpu(), full_steps(logits.cpu(), ms)
    assert tok.shape == (k * nrs, 1, ms) and full.shape[1] == k * nrs * nb
    kw = dict(V=cfg.vocab_size, eos=cfg.eos_index, sos=cfg.sos_index, max_steps=ms, nb=nb, pnb=2, keep=1, lp=0.6,
              do_sample=True, top_k=30, top_p=0.9, temperature=0.8, rp=1.2, nrs=nrs)
    rows = nrs * nb
    sure = []
    for j in range(k):
        ref_tok, ref_lp, s = oracle_search(full[:, j * rows:(j + 1) * rows], 1, seed=keys[j], **kw)
        for r in range(nrs):
            if r in s.unsure():
                continue
            e = j * nrs + r
            sure.append(e)
            assert torch.equal(tok[e], ref_tok[r]), (j, r, tok[e], ref_tok[r])
            assert torch.allclose(lps[e], ref_lp[r], atol=2e-5, rtol=0), (j, r, lps[e], ref_lp[r])
    record("multistream_sampling_oracle", entries=k * nrs, sure=len(sure), steps=logits.shape[0])
    assert sure, "every entry had a near-tie"

    # negative controls: the clip path's counter (word 3 = the camera's position, one key for the call), and one key for
    # every camera, each disagree with the device on most entries
    clip_tok, _, _ = oracle_search(full, k, seed=keys[0], **kw)
    one_key = torch.cat([oracle_search(full[:, j * rows:(j + 1) * rows], 1, seed=keys[0], **kw)[0] for j in range(k)])
    for name, bad in (("clip_counter", clip_tok), ("one_key", one_key)):
        differs = sum(not torch.equal(tok[e], bad[e]) for e in sure)
        record("multistream_sampling_negative_control", control=name, entries=len(sure), differing=differs)
        assert differs > len(sure) // 2, (name, differs, len(sure))

    # without sampling: beam 4 with repetition penalty 1.2, token-exact per camera
    sp4 = g.SearchConfig(beam_size=4, max_steps=ms)
    tok4, lps4, logits4 = eng.streams_caption(ids, sp4, sample=g.SampleConfig(repetition_penalty=1.2), keys=keys,
                                              save_logits=True)
    full4 = full_steps(logits4.cpu(), ms)
    kw4 = dict(kw, nb=4, nrs=1, do_sample=False, top_k=None, top_p=None, temperature=1.0)
    for j in range(k):
        ref_tok, ref_lp, _ = oracle_search(full4[:, j * 4:(j + 1) * 4], 1, seed=0, **kw4)
        assert torch.equal(tok4[j].long().cpu(), ref_tok[0]), (j, tok4[j], ref_tok[0])
        assert torch.allclose(lps4[j].cpu(), ref_lp[0], atol=2e-5, rtol=0)


def test_k1_equals_single_window_and_decode_ext(g, setup):
    _, _, eng, frames = setup
    sp = g.SearchConfig(beam_size=2, max_steps=10)
    sid, x = 7, keys_of(555)[0]
    smp = dict(num_return_sequences=2, **SMP)
    # the camera's frames pushed one at a time, as the single window encodes them (one frame per ViT batch)
    eng.streams_reset([sid])
    eng.stream_reset()
    for r in range(N_FRAMES):
        eng.streams_push([sid], frames[r, sid][None].contiguous())
        eng.stream_push(frames[r, sid])
    t1, l1, g1 = eng.streams_caption([sid], sp, sample=g.SampleConfig(**smp), keys=[x], save_logits=True)
    t2, l2, g2 = eng.stream_caption(sp, sample=g.SampleConfig(seed=x, **smp), save_logits=True)
    eng.set_visual_features(eng.streams_window(sid)[None])
    t3, l3, g3 = eng.decode(1, sp, sample=g.SampleConfig(seed=x, **smp), save_logits=True)
    for name, (t, l, lg) in (("stream_caption_ext", (t2, l2, g2)), ("decode_ext", (t3, l3, g3))):
        assert lg.shape == g1.shape, (name, lg.shape, g1.shape)
        assert torch.equal(g1, lg), (name, (g1 - lg).abs().max().item())
        assert torch.equal(t1, t) and torch.equal(l1, l), (name, t1, t, l1, l)


def test_invariance_to_order_and_company_and_keys(g, setup):
    _, _, eng, _ = setup
    sp = g.SearchConfig(beam_size=2, max_steps=10)
    smp = g.SampleConfig(num_return_sequences=2, **SMP)
    ids, keys = [0, 1, 2, 3, 4, 5], keys_of(10, 11, 12, 13, 14, 15)

    def run(i, k):
        t, l, _ = eng.streams_caption(i, sp, sample=smp, keys=k)
        return t.view(len(i), 2, -1), l.view(len(i), 2, -1)

    ta, la = run(ids, keys)
    perm = [4, 0, 5, 2, 1, 3]
    tp, lp_ = run([ids[p] for p in perm], [keys[p] for p in perm])
    assert torch.equal(tp, ta[perm]) and torch.equal(lp_, la[perm])
    # camera 3 replaced by camera 9 (another window, another key): every other camera unchanged
    tr, lr = run([0, 1, 2, 9, 4, 5], keys[:3] + keys_of(99) + keys[4:])
    keep = [0, 1, 2, 4, 5]
    assert torch.equal(tr[keep], ta[keep]) and torch.equal(lr[keep], la[keep])
    tb, lb = run(ids, keys)
    assert torch.equal(tb, ta) and torch.equal(lb, la)
    tc, _ = run(ids, keys_of(20, 21, 22, 23, 24, 25))
    assert not torch.equal(tc, ta)
    record("multistream_sampling_other_keys", cameras_differing=sum(not torch.equal(tc[j], ta[j]) for j in range(6)))


def test_defaults_and_return_sequences_without_sampling(g, setup):
    _, _, eng, _ = setup
    ids = [2, 9, 4]
    for nb in (1, 4):
        sp = g.SearchConfig(beam_size=nb, max_steps=8)
        t0, l0 = eng.streams_caption(ids, sp)
        t1, l1, _ = eng.streams_caption(ids, sp, sample=g.SampleConfig(seed=5), keys=keys_of(1, 2, 3))
        assert torch.equal(t0, t1) and torch.equal(l0, l1)
    sp = g.SearchConfig(beam_size=2, max_steps=8)
    t, _, _ = eng.streams_caption(ids, sp, sample=g.SampleConfig(num_return_sequences=3))  # keys ignored without sampling
    t = t.view(3, 3, -1)
    for r in (1, 2):
        assert torch.equal(t[:, r], t[:, 0])


def test_graph_replay_equals_eager_for_new_ids_and_keys(g, setup):
    _, _, eng, _ = setup
    sp = g.SearchConfig(beam_size=2, max_steps=8)
    smp = g.SampleConfig(num_return_sequences=2, **SMP)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    for k in (3, 12):  # 3: the whole call as one graph; 12: graphed assembly + visual pass and decode segments
        calls = [(list(range(k)) if i % 2 == 0 else list(range(16 - k, 16))[::-1], keys_of(*range(40 * i, 40 * i + k)))
                 for i in range(4)]
        outs = []
        before = eng.lib.gitb200_graph_launches(eng.h)
        with torch.cuda.stream(side):
            for ids, keys in calls:
                t, l, _ = eng.streams_caption(ids, sp, sample=smp, keys=keys)
                outs.append((t, l))
            side.synchronize()
        launched = eng.lib.gitb200_graph_launches(eng.h) - before
        record("multistream_sampling_graphs", k=k, graph_launches=launched)
        assert launched >= 2, launched
        eng.set_graph_max_clips(0)
        eng.set_graph_segments(False)
        try:
            for (ids, keys), (t, l) in zip(calls, outs):
                te, le, _ = eng.streams_caption(ids, sp, sample=smp, keys=keys)
                assert torch.equal(te, t) and torch.equal(le, l), (k, ids)
        finally:
            eng.set_graph_max_clips(8)
            eng.set_graph_segments(True)
        assert not torch.equal(outs[0][0], outs[2][0])  # same ids, new keys


def test_rejections_name_the_value_and_change_no_window(g, setup):
    _, _, eng, _ = setup
    lib, h = eng.lib, eng.h
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    tok = torch.empty(64, 1, 8, dtype=torch.int32, device="cuda")
    lp = torch.empty(64, 1, device="cuda")
    sp = g.SearchConfig(beam_size=2, max_steps=8).to_c()
    eng.streams_reset([14])
    eng.streams_push([14], torch.randn(1, 3, 224, 224, generator=torch.Generator().manual_seed(3)).cuda())
    frames = [eng.streams_frames(i) for i in range(16)]
    before = {i: eng.streams_window(i).clone() for i in (0, 1, 14)}
    torch.cuda.synchronize()

    def call(ids, smp, keys="auto"):
        arr = (ctypes.c_int32 * len(ids))(*ids)
        if keys == "auto":
            keys = (ctypes.c_uint64 * len(ids))(*keys_of(*range(len(ids))))
        return lib.gitb200_streams_caption_ext(h, arr, len(ids), ctypes.byref(sp), ctypes.byref(smp.to_c()), keys,
                                               ctypes.c_void_p(tok.data_ptr()), ctypes.c_void_p(lp.data_ptr()), None, s)

    def err():
        return lib.gitb200_last_error(h).decode()

    good = dict(SMP)
    n0 = eng.launch_count()
    assert call([0, 1], g.SampleConfig(**good), keys=None) != 0 and "keys_host" in err()
    for field, value, named in (("temperature", 0.0, "temperature"), ("top_p", 1.5, "top_p"), ("top_p", 0.0, "top_p"),
                                ("repetition_penalty", 0.0, "repetition_penalty"), ("num_return_sequences", 0, "num_return_sequences"),
                                ("top_k", 1, "top_k")):
        x = g.SampleConfig(**good)
        setattr(x, field, value)
        if field == "top_k":
            x.top_k, sp.per_node_beam_size = 2, 3  # two kept tokens for three draws
        assert call([0, 1], x) != 0 and named in err(), (field, err())
        sp.per_node_beam_size = 2
    assert call([0, 17], g.SampleConfig(**good)) != 0 and "17" in err() and "unknown" in err()
    assert call([1, 1], g.SampleConfig(**good)) != 0 and "twice" in err()
    assert call([0, 14], g.SampleConfig(**good)) != 0 and "different lengths" in err() and "14" in err()
    assert lib.gitb200_stream_caption_ext(h, ctypes.byref(sp), None, ctypes.c_void_p(tok.data_ptr()),
                                          ctypes.c_void_p(lp.data_ptr()), None, s) != 0
    assert eng.launch_count() == n0  # nothing was enqueued
    assert [eng.streams_frames(i) for i in range(16)] == frames
    for i, w in before.items():
        assert torch.equal(eng.streams_window(i), w), i
    with pytest.raises(g.GitB200Error, match="keys"):
        eng.streams_caption([0, 1], g.SearchConfig(beam_size=2, max_steps=8), sample=g.SampleConfig(**good))


def test_captioner_at_the_benchmark_geometry(g):
    """MultiStreamCaptioner(sample=...) with 6-frame windows, 64 cameras, 3 return sequences: the same seed twice gives the
    same captions, another seed other captions, every caption is a list of 3 strings."""
    F6, S = 6, 64
    cfg = go.GitConfig(num_image_with_embedding=F6, tie_output=False)
    sd = go.init_state_dict(cfg, seed=23, temporal_std=0.02, perturb=True)
    teacher = g.GenerativeImageTextTeacher.from_random_init({"num_image_with_embedding": F6}, state_dict=sd)
    raw = torch.randint(0, 256, (F6, S, 96, 128, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(8)).cuda()

    def run(seed):
        cap = g.MultiStreamCaptioner(teacher, S, stride=1, max_len=12,
                                     sample=dict(do_sample=True, top_k=0, top_p=0.9, num_return_sequences=3, seed=seed))
        outs = [cap.push({s: raw[t, s] for s in range(S)}) for t in range(F6)]
        assert all(o == {} for o in outs[:-1]) and sorted(outs[-1]) == list(range(S))
        return outs[-1]

    a, b, c = run(1), run(1), run(2)
    assert a == b
    assert all(isinstance(v, list) and len(v) == 3 and all(isinstance(x, str) for x in v) for v in a.values())
    differing = sum(a[s] != c[s] for s in range(S))
    record("multistream_sampling_captioner", cameras=S, differing_other_seed=differing)
    assert differing > 0
