"""Host logic of prompted live captions (no GPU): the calls MultiStreamCaptioner and StreamingCaptioner make with prompts --
one pool call per (held frames, prompt length) with the group's [k, P] prefix in the order of its ids, the caption text after
the prompt, set_prompt's checks, prompts together with sampling keys, and unchanged calls for cameras without a prompt."""
import importlib
import os
import sys
from types import SimpleNamespace

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
model = importlib.import_module("real-time-video-captioning_b200.model")
from test_multistream_sampling_host import EOS, SAMPLE, SOS, RecordingEngine, frame, teacher  # noqa: E402

VOCAB = 2000
Q3, Q3B, Q2 = [SOS, 900, 901], [SOS, 910, 911], [SOS, 920]


class PromptEngine(RecordingEngine):
    """RecordingEngine whose caption of a prompted window is the prompt, then the window's frame markers (then 500 + r when
    sampled), as the device search returns it: the tokens include the prompt."""

    cfg = SimpleNamespace(vocab=VOCAB)

    def _answer(self, windows, sp, kw):
        nrs = kw["sample"].num_return_sequences if "sample" in kw else 1
        pre = kw.get("prefix")
        tok = torch.full((len(windows) * nrs, 1, sp.max_steps), EOS, dtype=torch.int32)
        for j, w in enumerate(windows):
            head = pre[j if pre.shape[0] > 1 else 0].tolist() if pre is not None else [SOS]
            for r in range(nrs):
                row = head + list(w) + ([500 + r] if "sample" in kw else [])
                tok[j * nrs + r, 0, : len(row)] = torch.tensor(row, dtype=torch.int32)
        if "sample" not in kw:
            return tok, torch.zeros(tok.shape[0], 1)
        return tok, torch.zeros(tok.shape[0], 1), None

    def streams_caption(self, ids, sp, *args, **kw):
        self.calls.append(("caption", list(ids), args, kw))
        return self._answer([self.win[s] for s in ids], sp, kw)

    def stream_caption(self, sp, *args, **kw):
        self.calls.append(("stream_caption", args, kw))
        return self._answer([self.ring], sp, kw)


def captions(eng):
    return [c for c in eng.calls if c[0] == "caption"]


def pool(n=4, **kw):
    eng = PromptEngine(2)
    return eng, model.MultiStreamCaptioner(teacher(eng, 2), n, stride=1, max_len=8, sliding=True, **kw)


def test_one_call_per_prompt_length_with_the_prefix_in_id_order():
    eng, cap = pool(5)
    cap.set_prompt(1, Q3)
    cap.set_prompt(3, Q3B)
    cap.set_prompt(4, Q2)
    order = [3, 0, 4, 1, 2]  # arrival order of the frames: the calls keep it
    cap.push({s: frame(10 + s) for s in order})
    out = cap.push({s: frame(20 + s) for s in order})
    calls = captions(eng)
    assert [(c[1], c[2]) for c in calls] == [([3, 1], ()), ([0, 2], ()), ([4], ())]
    assert torch.equal(calls[0][3]["prefix"], torch.tensor([Q3B, Q3], dtype=torch.int32))
    assert calls[0][3]["prefix"].dtype == torch.int32 and set(calls[0][3]) == {"prefix"}
    assert calls[1][3] == {}  # the cameras without a prompt: exactly the call they make without this feature
    assert torch.equal(calls[2][3]["prefix"], torch.tensor([Q2], dtype=torch.int32))
    # the caption is the text after the prompt
    assert out == {s: f"{10 + s} {20 + s}" for s in order}
    assert cap.latest_caption[3] == "13 23"


def test_held_frames_split_groups_of_one_prompt_length():
    eng = PromptEngine(3)  # windows of up to 3 frames, captioned from 2 on: ready cameras may hold 2 or 3
    cap = model.MultiStreamCaptioner(teacher(eng, 2), 3, stride=1, max_len=8, sliding=True, prompt=Q3)
    cap.push({1: frame(1), 2: frame(1)})
    cap.push({0: frame(2), 1: frame(2), 2: frame(2)})
    n = len(captions(eng))
    cap.push({0: frame(3), 1: frame(3), 2: frame(3)})
    calls = captions(eng)[n:]
    assert [c[1] for c in calls] == [[0], [1, 2]]
    assert all(torch.equal(c[3]["prefix"], torch.tensor([Q3] * len(c[1]), dtype=torch.int32)) for c in calls)


def test_default_prompt_and_per_camera_override_and_clearing():
    eng, cap = pool(3, prompt=Q2)
    cap.set_prompt(1, Q3)
    cap.push({0: frame(1), 1: frame(2), 2: frame(3)})
    cap.push({0: frame(4), 1: frame(5), 2: frame(6)})
    a, b = captions(eng)
    assert a[1] == [0, 2] and torch.equal(a[3]["prefix"], torch.tensor([Q2, Q2], dtype=torch.int32))
    assert b[1] == [1] and torch.equal(b[3]["prefix"], torch.tensor([Q3], dtype=torch.int32))
    cap.set_prompt(0, None)
    cap.set_prompt(1, torch.tensor([Q2]))  # a [1, P] tensor, as a row of batch['prefix']
    out = cap.push({0: frame(7), 1: frame(8), 2: frame(9)})
    c, d = captions(eng)[2:]
    assert c[1:] == ([0], (), {})
    assert d[1] == [1, 2] and torch.equal(d[3]["prefix"], torch.tensor([Q2, Q2], dtype=torch.int32))
    assert out == {0: "4 7", 1: "5 8", 2: "6 9"}


@pytest.mark.parametrize("bad,match", [([], "at least one"), ([SOS, VOCAB], "outside"), ([SOS, -1], "outside"),
                                       ([SOS] + [5] * 8, "max_len"), (torch.tensor([1.0, 2.0]), "integer"),
                                       (torch.tensor([[SOS, 3], [SOS, 4]]), "one row"), ([SOS, 2.0], "integer"),
                                       ([SOS, True], "integer")])
def test_set_prompt_rejects_bad_prompts_and_keeps_the_old_one(bad, match):
    eng, cap = pool(2)
    cap.set_prompt(0, Q3)
    with pytest.raises(ValueError, match=match):
        cap.set_prompt(0, bad)
    with pytest.raises(ValueError, match=match):
        model.MultiStreamCaptioner(teacher(PromptEngine(2), 2), 2, stride=1, max_len=8, prompt=bad)
    with pytest.raises(ValueError, match=match):
        model.StreamingCaptioner(teacher(PromptEngine(2), 2), stride=1, max_len=8, prompt=bad)
    cap.push({0: frame(1)})
    cap.push({0: frame(2)})
    assert torch.equal(captions(eng)[0][3]["prefix"], torch.tensor([Q3], dtype=torch.int32))


def test_set_prompt_limits():
    eng, cap = pool(2)
    with pytest.raises(KeyError):
        cap.set_prompt(2, Q3)
    cap.set_prompt(0, [SOS] + [5] * 7)  # P = max_len: one caption token left
    cap.set_prompt(1, torch.tensor([VOCAB - 1], dtype=torch.int16))
    assert cap._prompts == [tuple([SOS] + [5] * 7), (VOCAB - 1,)]


def test_prompts_with_sampling_keys():
    eng, cap = pool(3, sample=dict(SAMPLE, num_return_sequences=2))
    cap.set_prompt(0, Q3)
    cap.set_prompt(2, Q3B)
    n = [0, 0, 0]
    for t in range(4):
        before = len(eng.calls)
        out = cap.push({s: frame(10 * t + s) for s in range(3)})
        for _, ids, args, kw in [c for c in eng.calls[before:] if c[0] == "caption"]:
            assert kw["keys"] == [model.stream_key(77, s, n[s]) for s in ids]
            assert kw["sample"].num_return_sequences == 2
            if ids == [0, 2]:
                assert torch.equal(kw["prefix"], torch.tensor([Q3, Q3B], dtype=torch.int32))
            else:
                assert ids == [1] and "prefix" not in kw
            for s in ids:
                n[s] += 1
        if t:
            assert out[0] == [f"{10 * t - 10} {10 * t} 500", f"{10 * t - 10} {10 * t} 501"]
    assert n == [3, 3, 3]


def test_streaming_captioner_with_a_prompt():
    eng = PromptEngine(2)
    cap = model.StreamingCaptioner(teacher(eng, 2), stride=1, max_len=8, prompt=Q3)
    got = [cap.push(frame(v)) for v in range(1, 4)]
    assert got == [None, "1 2", None]  # the prompt is stripped; the window is emptied after a caption
    calls = [c for c in eng.calls if c[0] == "stream_caption"]
    assert torch.equal(calls[0][2]["prefix"], torch.tensor([Q3], dtype=torch.int32)) and calls[0][1] == ()
    cap.set_prompt(None)
    cap.push(frame(4))
    cap.push(frame(5))
    assert [c for c in eng.calls if c[0] == "stream_caption"][-1] == ("stream_caption", (), {})
    eng = PromptEngine(2)
    cap = model.StreamingCaptioner(teacher(eng, 2), stride=1, max_len=8, prompt=Q2, sample=dict(SAMPLE, num_return_sequences=2))
    cap.push(frame(1))
    assert cap.push(frame(2)) == ["1 2 500", "1 2 501"]
    (_, args, kw), = [c for c in eng.calls if c[0] == "stream_caption"]
    assert kw["sample"].seed == model.stream_key(77, 0, 0) and torch.equal(kw["prefix"], torch.tensor([Q2], dtype=torch.int32))
