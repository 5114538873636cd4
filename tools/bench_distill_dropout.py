"""Cost of dropout in the student's distillation step (enable_training(dropout_seed=...)): student.distillation_step (forward,
backward, Adam; one rank, no all-reduce) with fixed teacher logits, with and without dropout.

Student decoder of config.py:76-84 (d_model 576, 8 heads, d_ffn 1024, 2 layers, vocabulary 30522) from seeded random weights,
20 caption tokens and 6 memory tokens per clip, 8 clips (BASELINE.json configs[4]) and 64 clips.  Each arm is a separate
student with the same weights.  Both arms are warmed up, then timed with CUDA events in `--windows` windows of `--iters`
steps each, the two arms alternated window by window.  Reports the median and the spread of the windows' ms per step.
Reads the card's name, power limit and max SM clock in the same run.  Writes one JSON file to --out.

    python tools/bench_distill_dropout.py --out FILE [--clips 8,64] [--iters 50] [--windows 5] [--warmup 10]
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

L, F = 20, 6


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else f"nvidia-smi failed: {r.stderr.strip()}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--clips", default="8,64")
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=10)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: the distillation step runs only on the GPU")
    g = importlib.import_module("real-time-video-captioning_b200")
    dev = torch.device("cuda")
    out = {"gpu": gpu_info(), "what": "student.distillation_step ms (forward + backward + Adam, fixed teacher logits), 1 GPU",
           "tokens_per_clip": L, "memory_tokens": F, "p": 0.3, "iters": a.iters, "windows": a.windows, "warmup": a.warmup, "rows": []}
    for B in [int(v) for v in a.clips.split(",")]:
        gen = torch.Generator(device=dev).manual_seed(B)
        y = torch.randint(1000, 30000, (B, L), device=dev, generator=gen)
        y[:, 0] = 101
        mem = torch.randn(B, F, 576, device=dev, generator=gen)
        teacher = torch.randn(B, L, 30522, device=dev, generator=gen)
        arms = {}
        for name, seed in (("no_dropout", None), ("dropout", 1234)):
            torch.manual_seed(0)
            s = g.StudentCandidateV1(None, 576, 8, 1024, 0.3, 2, 30522, 101, 102).to(dev)
            s.enable_training(lr=1e-4, dropout_seed=seed)
            for _ in range(a.warmup):
                s.distillation_step(y, mem, teacher)
            arms[name] = s
        torch.cuda.synchronize()
        times = {k: [] for k in arms}
        e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for _ in range(a.windows):
            for name, s in arms.items():
                e[0].record()
                for _ in range(a.iters):
                    s.distillation_step(y, mem, teacher)
                e[1].record()
                torch.cuda.synchronize()
                times[name].append(e[0].elapsed_time(e[1]) / a.iters)
        row = {"clips": B, "rows": B * L}
        for name, t in times.items():
            row[f"{name}_ms_median"] = statistics.median(t)
            row[f"{name}_ms_windows"] = t
        row["overhead_ms"] = row["dropout_ms_median"] - row["no_dropout_ms_median"]
        row["overhead_rel"] = row["overhead_ms"] / row["no_dropout_ms_median"]
        out["rows"].append(row)
        print(json.dumps(row), flush=True)
        for s in arms.values():
            s.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps({"gpu": out["gpu"]}))


if __name__ == "__main__":
    main()
