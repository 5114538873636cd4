"""CPU tests of the prompted search's host side (batch['prefix'] on the device): infer's routing with search_param
['device_prefix'], the reference's predicted[:, P:] strip (the keep > 1 quirk included), the saved-logits length, the
prompt checks of Engine and the new C entry points' bindings."""
import importlib
import os
import re

import pytest
import torch

from oracle import search_oracle as so

g = importlib.import_module("real-time-video-captioning_b200")
eng_mod = importlib.import_module("real-time-video-captioning_b200.engine")
lib_mod = importlib.import_module("real-time-video-captioning_b200._lib")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EOS = 102


class FakeEngine:
    """Records the entry points infer reaches.  Its decode returns what the device returns: the oracle's search over fixed
    seeded scores with the prompt as input_ids (prompt included in the tokens), and max_steps - P steps of saved logits."""

    def __init__(self, vocab):
        self.cfg = type("Cfg", (), {"vocab": vocab})()
        self.device = torch.device("cpu")
        self.calls = []

    def set_visual_features(self, vf):
        self.calls.append("set_visual_features")

    def decode(self, n_clips, sp, save_logits=False, sample=None, prefix=None):
        self.calls.append(("decode", sample, None if prefix is None else prefix.clone()))
        P = 1 if prefix is None else prefix.shape[1]
        start = torch.full((n_clips, 1), 101) if prefix is None else prefix.long().expand(n_clips, P)
        gen = torch.Generator().manual_seed(5)
        steps = iter(range(10 ** 6))
        table = torch.randn(64, n_clips * sp.beam_size, self.cfg.vocab, generator=gen)

        def step(ids):
            return table[next(steps)].clone()

        dec, lps, _ = so.search(start, step, eos_index=EOS, max_steps=sp.max_steps, beam_size=sp.beam_size,
                                length_penalty=sp.length_penalty, per_node_beam_size=sp.per_node_beam_size,
                                num_keep_best=sp.num_keep_best, save_logits=False)
        if sp.num_keep_best == 1:
            dec = dec.unsqueeze(1)
        self.last = dec
        n = max(0, sp.max_steps - P)
        return dec.int(), lps, torch.zeros(n, n_clips * sp.beam_size, self.cfg.vocab + 6)

    def decode_begin(self, rows_per_clip):
        self.calls.append("decode_begin")

    def decode_step(self, tokens, pos):
        self.calls.append("decode_step")
        return torch.randn(tokens.shape[0], self.cfg.vocab)

    def decode_reorder(self, beam_idx, pos):
        pass


@pytest.fixture
def model():
    m = g.get_git_model(g.SyntheticTokenizer(), {"num_image_with_embedding": 2})
    m.decoder.max_steps = 7
    fake = FakeEngine(m.textual.vocab_size)
    m._engine, m._engine_stale = fake, False
    m.engine = lambda: fake
    return m, fake


def _kinds(fake):
    return [c[0] if isinstance(c, tuple) else c for c in fake.calls]


@pytest.mark.parametrize("seed", [None, 4])
def test_device_prefix_routes_to_the_device_search_with_and_without_seed(model, seed):
    m, fake = model
    prefix = torch.tensor([[101, 7, 9], [101, 8, 3]])
    sp = {"device_prefix": True} if seed is None else {"device_prefix": True, "seed": seed}
    out = m.infer({"prefix": prefix}, torch.zeros(2, 5, 768), None, sp)
    assert "decode" in _kinds(fake) and "decode_step" not in _kinds(fake)
    call = [c for c in fake.calls if isinstance(c, tuple)][0]
    assert torch.equal(call[2], prefix)
    assert (call[1] is None) == (seed is None)
    assert out["predictions"].shape == (2, 7 - 3) and out["logprobs"].shape == (2, 1)
    assert len(out["logits_dict"]) == 7 - 3 and len(out["logits_dict"][0]) == 2 * 4
    assert len(out["logits_dict"][0][0]) == m.textual.vocab_size


def test_without_device_prefix_the_host_loop_runs_as_before(model):
    m, fake = model
    m.infer({"prefix": torch.tensor([[101, 7]])}, torch.zeros(1, 5, 768), None, {"seed": 3})
    assert "decode_step" in fake.calls and "decode" not in _kinds(fake)
    with pytest.raises(AssertionError):  # the host loop still takes one prompt row only
        m.infer({"prefix": torch.tensor([[101, 7], [101, 8]])}, torch.zeros(2, 5, 768), None, {})


@pytest.mark.parametrize("keep,P", [(1, 1), (1, 2), (1, 4), (2, 3), (3, 2), (1, 7), (1, 9)])
def test_infer_strips_the_prompt_like_the_reference(model, keep, P):
    """predictions = the search's output with the reference's predicted[:, P:] applied (keep > 1: the keep dimension)."""
    m, fake = model
    prefix = torch.tensor([[101] + [11 + i for i in range(P - 1)]])
    out = m.infer({"prefix": prefix}, torch.zeros(2, 5, 768), None, {"device_prefix": True, "num_keep_best": keep})
    ref = fake.last.long()
    if keep == 1:
        ref = ref.squeeze(1)
    ref = ref[:, P:]
    assert torch.equal(out["predictions"], ref)
    assert len(out["logits_dict"]) == max(0, 7 - P)
    if P < 7 and keep == 1:  # the search's rows start with the prompt
        assert torch.equal(fake.last[:, 0, :P].long(), prefix.expand(2, P))


@pytest.mark.parametrize("bad", [torch.tensor([101, 7]), torch.zeros(1, 0, dtype=torch.long), torch.tensor([[101.0, 7.0]]),
                                 torch.tensor([[True, False]]), [[101, 7]]])
def test_engine_rejects_malformed_prompts(bad):
    with pytest.raises(g.GitB200Error, match="prefix"):
        eng_mod._prefix_host(bad)


def test_engine_prompt_goes_to_the_host_as_int32():
    p = eng_mod._prefix_host(torch.tensor([[101, 5, 6]], dtype=torch.int64).t().contiguous().t())
    assert p.dtype == torch.int32 and p.device.type == "cpu" and p.is_contiguous() and p.tolist() == [[101, 5, 6]]


def _header_params(name):
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "gitb200.h")).read(), flags=re.S)
    decl = re.search(r"\bint\s+" + name + r"\s*\(([^;]*)\)\s*;", text)
    assert decl, name
    return [p.strip() for p in decl.group(1).split(",")]


@pytest.mark.parametrize("name", ["gitb200_decode_prefix", "gitb200_caption_prefix", "gitb200_op_search_prefix"])
def test_prefix_bindings_match_the_header(name):
    params = _header_params(name)
    res, args = lib_mod.SIGNATURES[name]
    assert res is lib_mod.c_int and len(args) == len(params), (params, args)
    for p, a in zip(params, args):
        if p.startswith("int ") or p.startswith("const int "):
            assert a is lib_mod.c_int, (p, a)
        elif "gitb200_search_params" in p:
            assert a == lib_mod.POINTER(lib_mod.SearchParams)
        elif "gitb200_sample_params" in p:
            assert a == lib_mod.POINTER(lib_mod.SampleParams)
        else:
            assert "*" in p and a is lib_mod.c_void_p, (p, a)
    assert hasattr(lib_mod.load(), name)
