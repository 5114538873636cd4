"""Host logic of MultiStreamCaptioner (no GPU): per-camera stride counters, one batched push per frame size, one batched
caption per held-frame count, clear-after-caption versus sliding windows.  A fake engine stands in for the stream pool:
it keeps each stream's window of frame markers, and its "caption" of a window is the list of markers in arrival order, so
the captioner's output can be compared with the same loop run for every camera on its own."""
import importlib
import os
import sys
from collections import deque
from types import SimpleNamespace

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
model = importlib.import_module("real-time-video-captioning_b200.model")

SOS, EOS = 1000, 1001  # outside the byte range of the frame markers


class FakeEngine:
    def __init__(self, window):
        self.window, self.device, self.calls = window, torch.device("cpu"), []

    def streams_configure(self, n):
        self.win = [deque(maxlen=self.window) for _ in range(n)]

    def streams_push_u8(self, ids, buf):
        assert buf.dtype == torch.uint8 and buf.shape[0] == len(ids) and len(set(ids)) == len(ids)
        self.calls.append(("push", list(ids), tuple(buf.shape[1:3])))
        for j, sid in enumerate(ids):
            self.win[sid].append(int(buf[j, 0, 0, 0]))

    def streams_frames(self, sid):
        return len(self.win[sid])

    def streams_caption(self, ids, sp):
        counts = {len(self.win[sid]) for sid in ids}
        assert len(counts) == 1 and len(set(ids)) == len(ids)
        self.calls.append(("caption", list(ids), counts.pop()))
        tok = torch.full((len(ids), 1, sp.max_steps), EOS, dtype=torch.int32)
        for j, sid in enumerate(ids):
            row = [SOS] + list(self.win[sid])
            tok[j, 0, : len(row)] = torch.tensor(row, dtype=torch.int32)
        return tok, torch.zeros(len(ids), 1)

    def streams_reset(self, ids):
        self.calls.append(("reset", list(ids)))
        for sid in ids:
            self.win[sid].clear()


class FakeTokenizer:
    def decode(self, ids, skip_special_tokens=True):
        return " ".join(str(t) for t in ids if t not in (SOS, EOS))


def make_captioner(n_streams, stride, window, sliding):
    eng = FakeEngine(window)
    m = SimpleNamespace(engine=lambda: eng, num_image_with_embedding=window, _vf_token=None,
                        decoder=SimpleNamespace(length_penalty=0.6, per_node_beam_size=2))
    cap = model.MultiStreamCaptioner(SimpleNamespace(model=m, tokenizer=FakeTokenizer()), n_streams, stride=stride, max_len=8,
                                     sliding=sliding)
    return cap, eng


def one_camera(frames, stride, window, sliding):
    """StreamingCaptioner's loop for one camera: {tick: caption}."""
    counter, win, out = 0, [], {}
    for tick, marker in frames:
        counter += 1
        if counter < stride:
            continue
        counter = 0
        win = (win + [marker])[-window:]
        if len(win) >= window:
            out[tick] = " ".join(map(str, win))
            if not sliding:
                win = []
    return out


def schedule(n_streams, ticks):
    """Irregular arrivals: camera s delivers on tick t unless (t + s) % (s + 2) == 0; two frame sizes; marker = unique byte."""
    sched = []
    for t in range(ticks):
        tick = {}
        for s in range(n_streams):
            if (t + s) % (s + 2) == 0:
                continue
            h, w = (4, 6) if s % 2 == 0 else (5, 3)
            tick[s] = torch.full((h, w, 3), s * 40 + t + 1, dtype=torch.uint8)
        sched.append(tick)
    return sched


@pytest.mark.parametrize("sliding", [False, True])
@pytest.mark.parametrize("stride,window", [(1, 3), (3, 2), (2, 4)])
def test_multistream_captions_equal_one_loop_per_camera(sliding, stride, window):
    n, ticks = 5, 30
    sched = schedule(n, ticks)
    cap, eng = make_captioner(n, stride, window, sliding)
    got = {s: {} for s in range(n)}
    for t, frames in enumerate(sched):
        for sid, c in cap.push(frames).items():
            got[sid][t] = c
    for s in range(n):
        want = one_camera([(t, int(f[s][0, 0, 0])) for t, f in enumerate(sched) if s in f], stride, window, sliding)
        assert got[s] == want, s
        assert want, "every camera captions at least once in this schedule"
        assert cap.latest_caption[s] == want[max(want)]


def test_one_push_per_frame_size_and_one_caption_per_held_count():
    n, stride, window = 6, 2, 3
    sched = schedule(n, 24)
    cap, eng = make_captioner(n, stride, window, sliding=True)
    for frames in sched:
        before = len(eng.calls)
        cap.push(frames)
        calls = eng.calls[before:]
        pushes = [c for c in calls if c[0] == "push"]
        shapes = [c[2] for c in pushes]
        assert len(shapes) == len(set(shapes))  # one push call per (H, W) in a tick
        for _, ids, hw in pushes:
            assert all(tuple(frames[sid].shape[:2]) == hw for sid in ids)
        captions = [c for c in calls if c[0] == "caption"]
        assert len({c[2] for c in captions}) == len(captions)  # one caption call per held-frame count
        pushed = [sid for c in pushes for sid in c[1]]
        assert sorted(sid for c in captions for sid in c[1]) == sorted(s for s in pushed if len(eng.win[s]) >= window)
    assert any(len(c[1]) > 1 for c in eng.calls if c[0] == "caption")  # windows really were batched
    assert not any(c[0] == "reset" for c in eng.calls)  # sliding: windows are never cleared


def test_clear_after_caption_and_stride_counters_are_per_camera():
    cap, eng = make_captioner(3, stride=2, window=2, sliding=False)
    f = lambda v: torch.full((2, 2, 3), v, dtype=torch.uint8)  # noqa: E731
    assert cap.push({0: f(1), 1: f(2)}) == {}              # first frame of each camera: skipped by the stride
    assert eng.calls == []
    assert cap.push({0: f(3)}) == {}                       # camera 0's 2nd frame is pushed, camera 1 still waits
    assert eng.calls == [("push", [0], (2, 2))]
    assert cap.push({0: f(5), 1: f(6)}) == {}              # camera 0 skips, camera 1's 2nd frame is pushed
    assert cap.push({0: f(7), 1: f(8)}) == {0: "3 7"}      # camera 0's window is full: caption, then clear
    assert eng.calls[-2:] == [("caption", [0], 2), ("reset", [0])] and eng.win[0] == deque()
    assert cap.push({0: f(9), 1: f(10)}) == {1: "6 10"}
    assert cap.push({2: f(12)}) == {} and cap.push({0: f(11), 2: f(14)}) == {} and cap.push({0: f(13), 2: f(16)}) == {}
    assert cap.push({0: f(15), 2: f(18)}) == {0: "11 15", 2: "14 18"}  # two cameras complete together: one batched caption
    assert eng.calls[-3:] == [("push", [0, 2], (2, 2)), ("caption", [0, 2], 2), ("reset", [0, 2])]
    with pytest.raises(KeyError):
        cap.push({3: f(1)})
    cap.reset([0])
    assert eng.calls[-1] == ("reset", [0])
