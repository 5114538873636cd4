"""bench.py on the GPU: --steps sets the timed steps, and --dump-outputs writes what the timed path returned in its LAST
timed step, on the seeded weights and clips the benchmark builds."""
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def test_bench_dump_outputs_hold_the_last_timed_step(tmp_path):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    B, steps = 2, 3   # the timed steps alternate between two frame batches: the last one reads batch (steps - 1) % 2 = 0
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--quick", "--batch", str(B), "--steps", str(steps),
                        "--warmup", "0", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    assert json.loads(r.stdout)["steps"] == steps
    tok, lp = np.load(tmp_path / "tokens.npy"), np.load(tmp_path / "logprobs.npy")
    assert tok.dtype == np.float64 and tok.shape == (B, 1, 15) and lp.dtype == np.float32 and lp.shape == (B, 1)

    # the benchmark's engine and frame batches, built the way bench.main() builds them, captioned directly
    g = importlib.import_module("real-time-video-captioning_b200")
    gm = importlib.import_module("real-time-video-captioning_b200.model")
    eng, _ = bench.build_engine(g, gm, torch, {"num_image_with_embedding": 6}, 0)
    eng.set_pipeline(0)
    eng.reserve(B, 6, 1, 15)
    gen = torch.Generator(device="cuda").manual_seed(100)
    frames = [torch.randn(B, 6, 3, 224, 224, device="cuda", generator=gen) for _ in range(2)]
    sp = g.SearchConfig(beam_size=1, max_steps=15, length_penalty=0.6, per_node_beam_size=2, num_keep_best=1)
    want = [eng.caption(f, sp)[:2] for f in frames]
    eng.close()
    last, other = want[(steps - 1) % 2], want[steps % 2]
    assert np.array_equal(tok, last[0].cpu().numpy().astype(np.float64))
    assert np.array_equal(lp, last[1].cpu().numpy())
    assert not np.array_equal(lp, other[1].cpu().numpy())   # the two batches are told apart: the dump is the LAST step's
