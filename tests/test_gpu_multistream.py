"""GPU tests of the multi-stream pool (gitb200_streams_*, Engine.streams_*, MultiStreamCaptioner): one window of per-frame
ViT features per camera, pushes batched over cameras, captions batched over windows.  Same GIT-base 2-frame setup and
tolerances as test_gpu_parity.py; measured deviations go to the same parity-metrics file, through its record()."""
import ctypes

import pytest
import torch

from oracle import git_oracle as go
from oracle import search_oracle as so
from test_gpu_parity import record, rel_fro

pytestmark = pytest.mark.gpu

N_FRAMES = 2


@pytest.fixture(scope="module")
def g():
    import gitb200
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return gitb200


@pytest.fixture(scope="module")
def setup(g):
    """GIT-base geometry (ViT-B/16 + 6-layer decoder), tied head, 2-frame windows."""
    cfg = go.GitConfig(num_image_with_embedding=N_FRAMES, tie_output=True)
    sd = go.init_state_dict(cfg, seed=11, temporal_std=0.02, perturb=True)
    eng = g.Engine(g.make_config({"num_image_with_embedding": N_FRAMES}, cfg.sos_index, cfg.eos_index), 0)
    eng.load_state_dict(sd)
    return cfg, sd, eng


def frames_of(seed, *shape):
    return torch.randn(*shape, 3, 224, 224, generator=torch.Generator().manual_seed(seed))


def temporal(sd, n):
    return [sd[f"img_temperal_embedding.{i}"].reshape(-1).cuda() for i in range(n)]


def oracle_caption(sd, cfg, clip, nb, max_steps):
    with torch.no_grad():
        return so.infer(sd, cfg, go.encode_clip(sd, cfg, clip), beam_size=nb, max_steps=max_steps, save_logits=False)


def test_push_equals_encode_images_bit_for_bit(g, setup):
    """A push of k frames is gitb200_encode_images on those frames with ln_post writing into the ring slots: every window equals
    bf16(encode_images + temporal[position]) exactly, also after the ring wrapped and with the ids in another order per push."""
    cfg, sd, eng = setup
    k = 5
    eng.streams_configure(k)
    temb = temporal(sd, N_FRAMES)
    frames = frames_of(31, 4, k)
    hist = {s: [] for s in range(k)}
    for r in range(4):  # 4 pushes into windows of 2 frames: the ring wraps twice
        ids = [(j * 2 + r) % k for j in range(k)]
        dev = frames[r].cuda()
        eng.streams_push(ids, dev)
        enc = eng.encode_images(dev)
        for j, sid in enumerate(ids):
            hist[sid].append(enc[j])
        for sid in range(k):
            n = min(r + 1, N_FRAMES)
            assert eng.streams_frames(sid) == n
            want = torch.cat([(f + temb[i]).bfloat16().float() for i, f in enumerate(hist[sid][-n:])])
            got = eng.streams_window(sid)
            assert got.shape == (n * eng.T, 768)
            assert torch.equal(got, want), (r, sid, (got - want).abs().max().item())


def test_windows_and_captions_match_oracle_and_clip_caption(g, setup):
    cfg, sd, eng = setup
    k = 3
    frames = frames_of(32, N_FRAMES, k)
    eng.streams_configure(k)
    for r in range(N_FRAMES):
        eng.streams_push(list(range(k)), frames[r].cuda())
    for nb in (1, 4):
        sp = g.SearchConfig(beam_size=nb, max_steps=8)
        tok, lp = eng.streams_caption(list(range(k)), sp)
        for sid in range(k):
            clip = frames[:, sid]
            if nb == 1:
                with torch.no_grad():
                    ref_vf = go.encode_clip(sd, cfg, clip)[0]
                err = rel_fro(eng.streams_window(sid).cpu(), ref_vf)
                record("multistream_window", stream=sid, rel_fro=err)
                assert err < 2e-2, err
            ref = oracle_caption(sd, cfg, clip, nb, 8)
            record("multistream_caption", nb=nb, stream=sid, lp=lp[sid, 0].item(), ref_lp=ref["logprobs"][0, 0].item())
            assert torch.equal(tok[sid, 0].cpu().long(), ref["predictions"][0]), (nb, sid, tok[sid], ref["predictions"])
            assert torch.allclose(lp[sid].cpu(), ref["logprobs"][0], atol=0.02, rtol=0.02), (lp[sid], ref["logprobs"])
            t2, l2, _ = eng.caption(clip[None].cuda().contiguous(), sp)
            assert torch.equal(tok[sid], t2[0]) and torch.allclose(lp[sid], l2[0], atol=0.01), (nb, sid)


def test_caption_is_batch_invariant_and_k1_equals_single_stream(g, setup):
    cfg, sd, eng = setup
    k = 6
    frames = frames_of(33, N_FRAMES, k)
    eng.streams_configure(k)
    for r in range(N_FRAMES):
        eng.streams_push(list(range(k)), frames[r].cuda())
    perm = [3, 0, 5, 1, 4, 2]
    for nb in (1, 4):
        sp = g.SearchConfig(beam_size=nb, max_steps=8)
        ta, la = eng.streams_caption(list(range(k)), sp)
        tb, lb = eng.streams_caption(perm, sp)
        for j, sid in enumerate(perm):
            assert torch.equal(tb[j], ta[sid]) and torch.equal(lb[j], la[sid]), (nb, sid)
        # k = 1 through the pool == the single-stream window on the same frames
        t1, l1 = eng.streams_caption([2], sp)
        eng.stream_reset()
        for r in range(N_FRAMES):
            eng.stream_push(frames[r, 2].cuda())
        ts, ls = eng.stream_caption(sp)
        assert torch.equal(t1, ts) and torch.allclose(l1, ls, atol=0.01), (nb, t1, ts, l1, ls)
        assert torch.equal(t1[0], ta[2])


def test_ragged_arrival_resets_and_split_by_held_count(g, setup):
    """Cameras start at different ticks and one is reset mid-run; a caption set is split by held-frame count into separate
    calls.  Every caption equals the oracle caption of that camera's own last n frames in arrival order."""
    cfg, sd, eng = setup
    pool = frames_of(34, 12)
    nxt = iter(range(12))
    held = {s: [] for s in range(4)}
    eng.streams_configure(4)
    sp = g.SearchConfig(beam_size=1, max_steps=6)

    def push(ids):
        idx = [next(nxt) for _ in ids]
        eng.streams_push(ids, pool[idx].cuda())
        for sid, i in zip(ids, idx):
            held[sid] = (held[sid] + [i])[-N_FRAMES:]

    def caption(ids):
        by_n = {}
        for sid in ids:
            by_n.setdefault(eng.streams_frames(sid), []).append(sid)
        assert len(by_n) > 1  # the set really is ragged
        n_checked = 0
        for n, part in by_n.items():
            tok, lp = eng.streams_caption(part, sp)
            for j, sid in enumerate(part):
                assert len(held[sid]) == n
                ref = oracle_caption(sd, cfg, pool[held[sid]], 1, 6)
                assert torch.equal(tok[j, 0].cpu().long(), ref["predictions"][0]), (sid, held[sid], tok[j], ref["predictions"])
                assert torch.allclose(lp[j].cpu(), ref["logprobs"][0], atol=0.02, rtol=0.02)
                n_checked += 1
        return n_checked

    push([0, 1])
    push([3, 1])
    assert caption([0, 1, 3]) == 3          # stream 1 holds 2 frames, streams 0 and 3 hold 1
    eng.streams_reset([1])
    held[1] = []
    push([1, 0, 2])
    assert [eng.streams_frames(s) for s in range(4)] == [2, 1, 1, 1]
    assert caption([2, 3, 1, 0]) == 4


def test_raw_frame_push_and_two_frame_sizes_in_one_captioner_push(g, setup):
    cfg, sd, eng = setup
    gen = torch.Generator().manual_seed(35)
    raw = torch.randint(0, 256, (2, 4, 120, 160, 3), dtype=torch.uint8, generator=gen)
    ids = [2, 0, 3, 1]
    eng.streams_configure(4)
    buf = torch.empty(4, 120, 160, 3, dtype=torch.uint8, device="cuda")
    for r in range(2):
        buf.copy_(raw[r])
        eng.streams_push_u8(ids, buf)
    w_u8 = [eng.streams_window(s).clone() for s in range(4)]
    eng.streams_configure(4)
    for r in range(2):
        eng.streams_push(ids, g.preprocess_frames(raw[r].cuda()))
    for s in range(4):
        assert torch.equal(eng.streams_window(s), w_u8[s]), s
    # MultiStreamCaptioner: two frame sizes arrive in the same tick -> one raw push per size, one batched caption
    teacher = g.GenerativeImageTextTeacher.from_random_init({"num_image_with_embedding": N_FRAMES}, state_dict=sd)
    cap = g.MultiStreamCaptioner(teacher, 3, stride=1, max_len=5)
    big = torch.randint(0, 256, (2, 2, 120, 160, 3), dtype=torch.uint8, generator=gen)
    small = torch.randint(0, 256, (2, 100, 180, 3), dtype=torch.uint8, generator=gen)
    ticks = [{0: big[t, 0], 1: big[t, 1], 2: small[t]} for t in range(2)]
    assert cap.push(ticks[0]) == {}
    te = teacher.model.engine()
    first = [te.streams_window(s).clone() for s in range(3)]
    out = cap.push(ticks[1])
    eng.streams_configure(3)
    sp = g.SearchConfig(beam_size=1, max_steps=6, length_penalty=teacher.model.decoder.length_penalty,
                        per_node_beam_size=teacher.model.decoder.per_node_beam_size)
    for t in range(2):
        eng.streams_push([0, 1], g.preprocess_frames(big[t].cuda()))
        eng.streams_push([2], g.preprocess_frames(small[t][None].cuda()))
        if t == 0:
            for s in range(3):
                assert torch.equal(eng.streams_window(s), first[s]), s
    tok, _ = eng.streams_caption([0, 1, 2], sp)
    assert sorted(out) == [0, 1, 2]
    for s in range(3):
        assert out[s] == teacher.tokenizer.decode(tok[s, 0].tolist(), skip_special_tokens=True), s
    assert all(te.streams_frames(s) == 0 for s in range(3))  # cleared after the caption (sliding=False)


def test_graph_replay_equals_eager_with_new_stream_sets(g, setup):
    """Repeated same-shape pushes and captions on a side stream replay CUDA graphs; results equal the eager launches bit for bit,
    also for another set of stream ids of the same k (the graph reads the per-call tables at their fixed address)."""
    cfg, sd, eng = setup
    x = [frames_of(36 + r, 12).cuda() for r in range(N_FRAMES)]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())

    def run(ids, xs, sp):
        for r in range(N_FRAMES):
            eng.streams_push(ids, xs[r])  # the same frame buffers on every call: the push graphs' keys match
        return eng.streams_caption(ids, sp)

    for k in (3, 12):  # 3: one graph per call (latency mode); 12: graphed encode, visual pass and decode segments
        xs = [t[:k].contiguous() for t in x]
        sp = g.SearchConfig(beam_size=1, max_steps=6)
        eng.streams_configure(16)
        ref_t, ref_l = run(list(range(k)), xs, sp)  # legacy default stream: eager
        torch.cuda.synchronize()
        before = eng.lib.gitb200_graph_launches(eng.h)
        with torch.cuda.stream(side):
            for i in range(4):
                ids = list(range(k)) if i % 2 == 0 else list(range(16 - k, 16))[::-1]
                eng.streams_reset(list(range(16)))
                t, l = run(ids, xs, sp)
                side.synchronize()
                assert torch.equal(t, ref_t) and torch.equal(l, ref_l), (k, i)
            launched = eng.lib.gitb200_graph_launches(eng.h) - before
            assert launched >= 3, launched
            if k == 12:  # graph segments off: the same calls run eagerly on the side stream
                eng.set_graph_segments(False)
                try:
                    eng.streams_reset(list(range(16)))
                    t, l = run(list(range(k)), xs, sp)
                    side.synchronize()
                finally:
                    eng.set_graph_segments(True)
                assert torch.equal(t, ref_t) and torch.equal(l, ref_l)
        record("multistream_graphs", k=k, graph_launches=launched)


def test_pool_windows_are_isolated_from_other_calls(g, setup):
    cfg, sd, eng = setup
    eng.streams_configure(3)
    fr = frames_of(37, N_FRAMES, 3)
    for r in range(N_FRAMES):
        eng.streams_push([0, 1, 2], fr[r].cuda())
    sp = g.SearchConfig(beam_size=1, max_steps=6)
    before = [eng.streams_window(s).clone() for s in range(3)]
    t0, l0 = eng.streams_caption([0, 1, 2], sp)
    eng.stream_reset()
    for f in frames_of(38, 3):
        eng.stream_push(f.cuda())
        eng.stream_caption(sp)
    eng.caption(frames_of(39, 4, N_FRAMES).cuda(), sp)
    eng.encode_images(frames_of(40, 5).cuda())
    for s in range(3):
        assert torch.equal(eng.streams_window(s), before[s]), s
    t1, l1 = eng.streams_caption([0, 1, 2], sp)
    assert torch.equal(t0, t1) and torch.equal(l0, l1)


def test_rejections_name_the_id_and_change_no_window(g, setup):
    cfg, sd, _ = setup
    eng = g.Engine(g.make_config({"num_image_with_embedding": N_FRAMES}, cfg.sos_index, cfg.eos_index), 0)
    eng.load_state_dict(sd)
    lib, h = eng.lib, eng.h
    INVALID, STATE = -1, -3
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    x = frames_of(41, 4).cuda()
    tok = torch.empty(4, 1, 6, dtype=torch.int32, device="cuda")
    lp = torch.empty(4, 1, device="cuda")
    c = g.SearchConfig(beam_size=1, max_steps=6).to_c()

    def ids(*v):
        return (ctypes.c_int32 * max(1, len(v)))(*v)

    def err():
        return lib.gitb200_last_error(h).decode()

    assert lib.gitb200_streams_push(h, ids(0), 1, ctypes.c_void_p(x.data_ptr()), s) == STATE and "configure" in err()
    assert lib.gitb200_streams_caption(h, ids(0), 1, ctypes.byref(c), ctypes.c_void_p(tok.data_ptr()),
                                       ctypes.c_void_p(lp.data_ptr()), s) == STATE
    assert lib.gitb200_streams_configure(h, 0) == INVALID
    eng.streams_configure(4)
    eng.streams_push([0, 1], x[:2])
    eng.streams_push([0], x[2:3])
    before = {sid: eng.streams_window(sid).clone() for sid in (0, 1)}

    def push(*v):
        return lib.gitb200_streams_push(h, ids(*v), len(v), ctypes.c_void_p(x.data_ptr()), s)

    def caption(*v):
        return lib.gitb200_streams_caption(h, ids(*v), len(v), ctypes.byref(c), ctypes.c_void_p(tok.data_ptr()),
                                           ctypes.c_void_p(lp.data_ptr()), s)

    assert push(0, 7) == INVALID and "7" in err() and "unknown" in err()
    assert push(2, 2) == INVALID and "2" in err() and "twice" in err()
    assert push(-1) == INVALID and "-1" in err()
    assert lib.gitb200_streams_push(h, ids(), 0, ctypes.c_void_p(x.data_ptr()), s) == INVALID and "k" in err()
    assert lib.gitb200_streams_push_u8(h, ids(0), 1, None, 8, 8, s) == INVALID
    assert caption(3) == STATE and "3" in err()
    assert caption(1, 2) == STATE and "2" in err()
    assert caption(0, 1) == INVALID and "0" in err() and "1" in err()
    assert caption(1, 1) == INVALID and "twice" in err()
    assert caption(9) == INVALID and "9" in err()
    assert lib.gitb200_streams_reset(h, ids(1, 4), 2) == INVALID and "4" in err()
    assert lib.gitb200_streams_window(h, 5, ctypes.c_void_p(lp.data_ptr()), s) == INVALID and "5" in err()
    assert lib.gitb200_streams_window(h, 3, ctypes.c_void_p(lp.data_ptr()), s) == STATE and "3" in err()
    assert lib.gitb200_streams_frames(h, 4) == INVALID and lib.gitb200_streams_frames(h, 0) == 2
    torch.cuda.synchronize()
    assert [eng.streams_frames(sid) for sid in range(4)] == [2, 1, 0, 0]
    for sid in (0, 1):
        assert torch.equal(eng.streams_window(sid), before[sid]), sid
    with pytest.raises(g.GitB200Error, match="different lengths"):
        eng.streams_caption([0, 1], g.SearchConfig(beam_size=1, max_steps=6))
    eng.close()


def test_256_streams_at_the_baseline_geometry(g):
    """GIT-base, 6-frame windows, greedy max_steps 15, tied head: 256 cameras filled by 6 batched pushes (a different id
    order per push), captioned in one call; a sample of 8 cameras equals Engine.caption on their clips."""
    F6, S = 6, 256
    cfg = go.GitConfig(num_image_with_embedding=F6, tie_output=True)
    sd = go.init_state_dict(cfg, seed=21, temporal_std=0.02, perturb=True)
    eng = g.Engine(g.make_config({"num_image_with_embedding": F6}, cfg.sos_index, cfg.eos_index), 0)
    eng.load_state_dict(sd)
    eng.streams_configure(S)
    gen = torch.Generator(device="cuda").manual_seed(6)
    clips = torch.empty(S, F6, 3, 224, 224, device="cuda")
    for p in range(F6):
        perm = torch.randperm(S, generator=torch.Generator().manual_seed(100 + p)).tolist()
        x = torch.randn(S, 3, 224, 224, device="cuda", generator=gen)
        eng.streams_push(perm, x)
        clips[perm, p] = x
    assert all(eng.streams_frames(s) == F6 for s in range(S))
    sp = g.SearchConfig(beam_size=1, max_steps=15)
    tok, lp = eng.streams_caption(list(range(S)), sp)
    sample = list(range(3, S, S // 8))[:8]
    t_ref, l_ref, _ = eng.caption(clips[sample].contiguous(), sp)
    record("multistream_256", max_lp_diff=(lp[sample] - l_ref).abs().max().item())
    assert torch.equal(tok[sample], t_ref), (tok[sample], t_ref)
    assert torch.allclose(lp[sample], l_ref, atol=0.01)
    eng.close()
