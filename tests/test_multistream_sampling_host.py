"""Host logic of sampled live captions (no GPU): the per-camera Philox keys MultiStreamCaptioner and StreamingCaptioner pass to
the engine, the lists of strings of num_return_sequences > 1, unchanged engine calls without ``sample``, and stream_key."""
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

SOS, EOS = 1000, 1001
SAMPLE = dict(do_sample=True, top_k=0, top_p=0.9, temperature=1.0, repetition_penalty=1.0, num_return_sequences=1, seed=77)


class RecordingEngine:
    """A stream pool whose caption of a window is its frame markers, followed by 500 + r when sampled (so that every return
    sequence r differs).  Records every call with its arguments."""

    def __init__(self, window):
        self.window, self.device, self.calls = window, torch.device("cpu"), []

    def streams_configure(self, n):
        self.win = [deque(maxlen=self.window) for _ in range(n)]

    def streams_push_u8(self, ids, buf):
        self.calls.append(("push", list(ids)))
        for j, sid in enumerate(ids):
            self.win[sid].append(int(buf[j, 0, 0, 0]))

    def streams_frames(self, sid):
        return len(self.win[sid])

    def streams_reset(self, ids):
        self.calls.append(("reset", list(ids)))
        for sid in ids:
            self.win[sid].clear()

    def _rows(self, windows, sp, nrs, sampled):
        tok = torch.full((len(windows) * nrs, 1, sp.max_steps), EOS, dtype=torch.int32)
        for j, w in enumerate(windows):
            for r in range(nrs):
                row = [SOS] + list(w) + ([500 + r] if sampled else [])
                tok[j * nrs + r, 0, : len(row)] = torch.tensor(row, dtype=torch.int32)
        return tok

    def streams_caption(self, ids, sp, *args, **kw):
        self.calls.append(("caption", list(ids), args, kw))
        nrs = kw["sample"].num_return_sequences if "sample" in kw else 1
        tok = self._rows([self.win[s] for s in ids], sp, nrs, "sample" in kw)
        if "sample" not in kw:
            return tok, torch.zeros(len(ids), 1)
        return tok, torch.zeros(tok.shape[0], 1), None

    # single-stream window
    def stream_reset(self):
        self.calls.append(("stream_reset",))
        self.ring = deque(maxlen=self.window)

    def stream_push_u8(self, buf):
        self.ring.append(int(buf[0, 0, 0]))
        return len(self.ring)

    def stream_caption(self, sp, *args, **kw):
        self.calls.append(("stream_caption", args, kw))
        nrs = kw["sample"].num_return_sequences if "sample" in kw else 1
        tok = self._rows([self.ring], sp, nrs, "sample" in kw)
        if "sample" not in kw:
            return tok, torch.zeros(1, 1)
        return tok, torch.zeros(nrs, 1), None


class FakeTokenizer:
    def decode(self, ids, skip_special_tokens=True):
        return " ".join(str(t) for t in ids if t not in (SOS, EOS))


def teacher(eng, window):
    m = SimpleNamespace(engine=lambda: eng, num_image_with_embedding=window, _vf_token=None,
                        decoder=SimpleNamespace(length_penalty=0.6, per_node_beam_size=2))
    return SimpleNamespace(model=m, tokenizer=FakeTokenizer())


def frame(v):
    return torch.full((2, 2, 3), v, dtype=torch.uint8)


def test_pool_keys_count_captions_per_camera_across_reset():
    eng = RecordingEngine(2)
    cap = model.MultiStreamCaptioner(teacher(eng, 2), 3, stride=1, max_len=8, sample=SAMPLE)
    n = [0, 0, 0]
    ticks = [{0: 1, 1: 2}, {0: 3, 1: 4, 2: 5}, {0: 6, 2: 7}, {1: 8, 2: 9}, {0: 10, 1: 11, 2: 12}, {0: 13, 1: 14, 2: 15}]
    for t, tick in enumerate(ticks):
        if t == 3:
            cap.reset([0, 1])  # empties the windows and stride counters, not the caption counts
        before = len(eng.calls)
        out = cap.push({sid: frame(v) for sid, v in tick.items()})
        for call in eng.calls[before:]:
            if call[0] != "caption":
                continue
            _, ids, args, kw = call
            assert args == () and kw["sample"].do_sample and kw["sample"].top_p == 0.9
            assert kw["keys"] == [model.stream_key(77, sid, n[sid]) for sid in ids], (t, ids)
            for sid in ids:
                n[sid] += 1
        assert all(isinstance(c, str) for c in out.values())
    assert n == [2, 2, 2]  # camera 0 and 1 captioned once before and once after the reset
    assert len({k for c in eng.calls if c[0] == "caption" for k in c[3]["keys"]}) == sum(n)  # no key used twice


def test_streaming_captioner_keys_and_return_sequences():
    eng = RecordingEngine(2)
    cap = model.StreamingCaptioner(teacher(eng, 2), stride=1, max_len=8, sample=dict(SAMPLE, num_return_sequences=3))
    got = []
    for v in range(1, 8):
        c = cap.push(frame(v))
        if c is not None:
            got.append(c)
    calls = [c for c in eng.calls if c[0] == "stream_caption"]
    assert len(calls) == len(got) == 3
    for n, (_, args, kw) in enumerate(calls):
        assert args == () and kw["sample"].seed == model.stream_key(77, 0, n) and kw["sample"].num_return_sequences == 3
    assert got[0] == ["1 2 500", "1 2 501", "1 2 502"] and cap.latest_caption == got[-1]


def test_pool_return_sequences_are_lists_of_strings():
    eng = RecordingEngine(2)
    cap = model.MultiStreamCaptioner(teacher(eng, 2), 2, stride=1, max_len=8, sample=dict(SAMPLE, num_return_sequences=2),
                                     sliding=True)
    cap.push({0: frame(1), 1: frame(2)})
    out = cap.push({0: frame(3), 1: frame(4)})
    assert out == {0: ["1 3 500", "1 3 501"], 1: ["2 4 500", "2 4 501"]}
    assert cap.latest_caption[1] == ["2 4 500", "2 4 501"]


def test_without_sample_the_engine_calls_are_unchanged():
    eng = RecordingEngine(2)
    cap = model.MultiStreamCaptioner(teacher(eng, 2), 2, stride=1, max_len=8)
    cap.push({0: frame(1), 1: frame(2)})
    assert cap.push({0: frame(3), 1: frame(4)}) == {0: "1 3", 1: "2 4"}
    assert [c for c in eng.calls if c[0] == "caption"] == [("caption", [0, 1], (), {})]
    eng = RecordingEngine(2)
    sc = model.StreamingCaptioner(teacher(eng, 2), stride=1, max_len=8)
    sc.push(frame(1))
    assert sc.push(frame(2)) == "1 2"
    assert [c for c in eng.calls if c[0] == "stream_caption"] == [("stream_caption", (), {})]


def test_stream_key_is_deterministic_and_collision_free():
    keys = {model.stream_key(5, i, n) for i in range(512) for n in range(1000)}
    assert len(keys) == 512 * 1000
    assert all(0 <= k < 2 ** 64 for k in keys)
    assert model.stream_key(5, 3, 7) == model.stream_key(5, 3, 7)
    assert model.stream_key(5, 3, 7) != model.stream_key(6, 3, 7)
    assert model.stream_key(-1, 0, 0) == model.stream_key(2 ** 64 - 1, 0, 0)  # the seed is taken modulo 2^64
    # the documented mix, restated
    M = 2 ** 64 - 1

    def sm(x):
        z = (x + 0x9E3779B97F4A7C15) & M
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M
        return z ^ (z >> 31)

    assert model.stream_key(123, 4, 9) == sm(sm(123) ^ (5 << 32 | 9))
    with pytest.raises(ValueError):
        model.stream_key(1, -1, 0)
    with pytest.raises(ValueError):
        model.stream_key(1, 0, 2 ** 32)


def test_unknown_sample_names_are_rejected():
    with pytest.raises(ValueError, match="topk"):
        model.MultiStreamCaptioner(teacher(RecordingEngine(2), 2), 2, sample={"topk": 5})
