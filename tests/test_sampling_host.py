"""CPU tests of the sampling search's host side: the Philox4x32-10 reference, SampleConfig packing and infer's routing."""
import ctypes
import importlib
import os

import numpy as np
import pytest
import torch

from sampling_ref import gumbel, philox4x32_10, uniform, uniforms

g = importlib.import_module("real-time-video-captioning_b200")
eng_mod = importlib.import_module("real-time-video-captioning_b200.engine")
lib_mod = importlib.import_module("real-time-video-captioning_b200._lib")
CSRC = os.path.join(os.path.dirname(lib_mod.__file__), "csrc")


@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_reproduces_random123_known_answers(ctr, key, want):
    got = philox4x32_10(*ctr, *key)
    assert tuple(int(x) for x in got) == want


def test_uniforms_lie_in_the_open_interval_and_follow_the_counter_layout():
    u = uniforms(1001, 3, 5, 7, 0x123456789ABCDEF0)
    assert u.dtype == np.float64 and u.shape == (1001,) and u.min() > 0 and u.max() < 1
    w = philox4x32_10(250, 3, 5, 7, 0x9ABCDEF0, 0x12345678)  # index 1000 = word 0 of counter 250
    assert u[1000] == ((int(w[0]) >> 8) + 0.5) * 2.0 ** -24
    assert not np.array_equal(u, uniforms(1001, 4, 5, 7, 0x123456789ABCDEF0))


@pytest.mark.parametrize("word", [0x00000000, 0x000000FF, 0xFFFFFF00, 0xFFFFFFFF])
def test_extreme_words_give_an_open_interval_uniform_and_a_finite_race_key(word):
    """(2^24 - 1) + 0.5 is a rounding tie in fp32 (it would give u = 1 and key +inf); the uniform is formed in double."""
    u = uniform(word)
    assert 0.0 < u < 1.0
    assert np.isfinite(gumbel(u)) and -2.86 < gumbel(u) < 17.34


def test_header_philox_uniform_and_gumbel_on_the_host(tmp_path):
    """philox.cuh compiled for the host: the known-answer vector and the extreme words of the uniform."""
    import shutil
    import subprocess
    cxx = shutil.which("c++") or shutil.which("g++")
    if cxx is None:
        pytest.skip("no host C++ compiler")
    src = tmp_path / "t.cpp"
    src.write_text(
        '#include <cstdio>\n#include <initializer_list>\n#include "' + os.path.join(CSRC, "philox.cuh") + '"\n'
        "int main() { Philox4 r = philox4x32_10(0, 0, 0, 0, 0, 0);\n"
        '  std::printf("%08x %08x %08x %08x\\n", r.x[0], r.x[1], r.x[2], r.x[3]);\n'
        "  for (unsigned w : {0x0u, 0xFFu, 0xFFFFFF00u, 0xFFFFFFFFu})\n"
        '    std::printf("%.17g %.9g\\n", philox_uniform(w), (double)philox_gumbel(w));\n}\n')
    exe = tmp_path / "t"
    subprocess.run([cxx, "-O2", "-std=c++17", "-o", str(exe), str(src)], check=True)
    lines = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split("\n")
    assert lines[0] == "6627e8d5 e169c58d bc57ac4c 9b00dbd8"
    for line, w in zip(lines[1:5], (0x0, 0xFF, 0xFFFFFF00, 0xFFFFFFFF)):
        u, gk = (float(v) for v in line.split())
        assert 0.0 < u < 1.0 and u == uniform(w)
        assert np.isfinite(gk) and np.float32(gk) == gumbel(uniform(w))  # %.9g round-trips a float


def test_sample_config_packs_into_the_c_struct():
    assert ctypes.sizeof(lib_mod.SampleParams) == 32
    c = g.SampleConfig(do_sample=True, top_k=7, top_p=0.9, temperature=0.5, repetition_penalty=1.2, num_return_sequences=3,
                       seed=2 ** 64 - 5).to_c()
    assert (c.do_sample, c.top_k, c.num_return_sequences, c.seed) == (1, 7, 3, 2 ** 64 - 5)
    assert (c.top_p, c.temperature, c.repetition_penalty) == pytest.approx((0.9, 0.5, 1.2))
    d = g.SampleConfig().to_c()
    assert (d.do_sample, d.top_k, d.top_p, d.temperature, d.repetition_penalty, d.num_return_sequences, d.seed) == (0, 0, 1.0, 1.0, 1.0, 1, 0)


class FakeEngine:
    """Records which entry points infer reaches; returns well-formed outputs."""

    def __init__(self, vocab):
        self.cfg = type("Cfg", (), {"vocab": vocab})()
        self.device = torch.device("cpu")
        self.calls = []

    def set_visual_features(self, vf):
        self.calls.append("set_visual_features")

    def decode(self, n_clips, sp, save_logits=False, sample=None):
        self.calls.append(("decode", sample))
        n = n_clips * (sample.num_return_sequences if sample else 1)
        return (torch.full((n, sp.num_keep_best, sp.max_steps), 102, dtype=torch.int32), torch.zeros(n, sp.num_keep_best),
                torch.zeros(sp.max_steps - 1, n * sp.beam_size, self.cfg.vocab + 6))

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
    m.decoder.max_steps = 4
    m.decoder.repetition_penalty = 1.2
    m.decoder.temperature = 0.7
    fake = FakeEngine(m.textual.vocab_size)
    m._engine, m._engine_stale = fake, False
    m.engine = lambda: fake
    return m, fake


def test_seed_routes_to_the_device_search_with_every_parameter(model):
    m, fake = model
    vf = torch.zeros(2, 5, 768)
    out = m.infer({}, vf, None, {"do_sample": True, "top_k": 5, "top_p": 0.8, "num_return_sequences": 3, "seed": 11})
    kinds = [c[0] if isinstance(c, tuple) else c for c in fake.calls]
    assert "decode" in kinds and "decode_step" not in kinds
    sample = [c for c in fake.calls if isinstance(c, tuple)][0][1]
    assert sample == g.SampleConfig(True, 5, 0.8, 0.7, 1.2, 3, 11)
    assert out["predictions"].shape == (6, 4) and out["logprobs"].shape == (6, 1)
    assert len(out["logits_dict"]) == 3 and len(out["logits_dict"][0]) == 6 * 4
    assert len(out["logits_dict"][0][0]) == m.textual.vocab_size


def test_without_seed_the_host_loop_runs_as_before(model):
    m, fake = model
    torch.manual_seed(0)
    out = m.infer({}, torch.zeros(2, 5, 768), None, {"do_sample": True, "top_k": 5, "top_p": 0.8})
    kinds = [c[0] if isinstance(c, tuple) else c for c in fake.calls]
    assert "decode" not in kinds and "decode_step" in kinds
    assert out["predictions"].shape[0] == 2


def test_seed_with_a_prefix_takes_the_host_loop(model):
    m, fake = model
    m.infer({"prefix": torch.tensor([[101, 7]])}, torch.zeros(1, 5, 768), None, {"seed": 3})
    assert "decode_step" in fake.calls and not any(isinstance(c, tuple) for c in fake.calls)


@pytest.mark.parametrize("top_k,top_p", [(None, 0.9), (5, None)])
def test_none_filters_raise_type_error_on_both_paths(model, top_k, top_p):
    m, fake = model
    for sp in ({"seed": 1}, {}):
        with pytest.raises(TypeError):
            m.infer({}, torch.zeros(1, 5, 768), None, dict(sp, do_sample=True, top_k=top_k, top_p=top_p))


def test_deterministic_penalty_with_seed_needs_no_filters(model):
    m, fake = model
    m.infer({}, torch.zeros(1, 5, 768), None, {"seed": 5})
    sample = [c for c in fake.calls if isinstance(c, tuple)][0][1]
    assert sample == g.SampleConfig(False, 0, 1.0, 0.7, 1.2, 1, 5)
