"""Many cameras on one B200 context: the multi-stream pool (gitb200_streams_*) against re-assembled clips through Engine.caption
and, for up to 16 cameras, against one Engine per camera (gitb200_stream_*).

GIT-base, 6-frame windows, greedy search of at most 15 tokens, seeded random weights (tied head), random preprocessed fp32
frames.  Every camera delivers one frame per tick (stride 1 at the push level).  Two modes:
  (a) nonoverlap: the reference's loop (real_time_inference.py:38-61): a window is captioned once it holds 6 frames and then
      cleared; camera phases are staggered so that about 1/6 of the cameras caption on each tick;
  (b) sliding: every camera is captioned on every tick over its last 6 frames.
Per tick, CUDA events on the launching stream give the push and caption time; the latency of a caption is from the start of
the tick (its newest frame arrives) to the end of the work that produced it.  All work runs on one non-default stream, so
every implementation can replay its CUDA graphs; every shape is warmed up for two full phase periods before the timed ticks.
Writes one JSON file to --out.

    python tools/bench_streams.py --out OUTDIR [--streams 1,16,64,256,512] [--ticks 12] [--warmup 12]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

F = 6          # frames per window (num_image_with_embedding)
MAX_STEPS = 15 + 1  # greedy, at most 15 tokens after SOS
# Algorithmic tensor work per caption, BASELINE.md section 3 conventions (GFLOP): one frame's ViT, the 6-frame clip's ViT,
# projection + prefill of the decoder over the 6 x 197 visual tokens.
GFLOP_FRAME, GFLOP_CLIP_VIT, GFLOP_PREFILL = 35.13, 210.76, 127.66


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else f"nvidia-smi failed: {r.stderr.strip()}"


class Ticker:
    """CUDA events on the launching stream: per tick start, after push, after caption (and per camera for the per-camera arm)."""

    def __init__(self):
        self.ticks = []

    def event(self):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def summary(self, n_streams):
        torch.cuda.current_stream().synchronize()
        push, cap, lat, caps = [], [], [], 0
        for t in self.ticks:
            push.append(t["start"].elapsed_time(t["pushed"]))
            cap.append(t["pushed"].elapsed_time(t["end"]))
            for e, n in t["done"]:
                lat += [t["start"].elapsed_time(e)] * n
                caps += n
        total = self.ticks[0]["start"].elapsed_time(self.ticks[-1]["end"]) / 1e3
        lat = np.array(lat) if lat else np.array([float("nan")])
        return {"ticks": len(self.ticks), "push_ms": float(np.mean(push)), "caption_ms": float(np.mean(cap)),
                "tick_ms": 1e3 * total / len(self.ticks), "frames_per_s": n_streams * len(self.ticks) / total,
                "captions_per_s": caps / total, "captions": caps,
                "latency_p50_ms": float(np.percentile(lat, 50)), "latency_p99_ms": float(np.percentile(lat, 99))}


def schedule(mode, S, t):
    """Cameras that push on tick t: in the non-overlapping mode camera s starts at tick s % 6, which staggers the phases."""
    return [s for s in range(S) if mode == "sliding" or s % F <= t]


def run_pool(g, eng, mode, S, frames, n_warm, n_timed, sp):
    """frames: [7, S, 3, R, R] device pool; tick t pushes frames[t % 7]."""
    eng.streams_configure(S)
    bufs = {}
    tk = Ticker()
    tokens = {}
    for t in range(n_warm + n_timed):
        ids = schedule(mode, S, t)
        key = len(ids)
        if key not in bufs:
            bufs[key] = torch.empty(key, *frames.shape[2:], device="cuda")
        x = bufs[key]
        x.copy_(frames[t % 7, ids] if key < S else frames[t % 7])
        rec = {"start": tk.event()}
        eng.streams_push(ids, x)
        rec["pushed"] = tk.event()
        ready = [s for s in ids if eng.streams_frames(s) == F]
        if ready:
            tok, _ = eng.streams_caption(ready, sp)
            if t == n_warm + n_timed - 1:
                tokens = dict(zip(ready, tok[:, 0]))
            del tok
            if mode == "nonoverlap":
                eng.streams_reset(ready)
        rec["end"] = tk.event()
        rec["done"] = [(rec["end"], len(ready))] if ready else []
        if t >= n_warm:
            tk.ticks.append(rec)
    return tk.summary(S), tokens


def window_clip(frames, t, ids):
    """The clips re-assembled from the raw frames: the 6 frames each camera pushed on ticks t-5 .. t, oldest first."""
    return torch.stack([frames[(t - F + 1 + i) % 7, ids] for i in range(F)], dim=1)


def run_clip_baseline(g, eng, mode, S, frames, n_warm, n_timed, sp):
    """The same captions through Engine.caption on clips re-assembled from the raw frames (every frame of a window re-encoded)."""
    count = [0] * S
    tk = Ticker()
    bufs, tokens = {}, {}
    for t in range(n_warm + n_timed):
        ids = schedule(mode, S, t)
        for s in ids:
            count[s] = min(count[s] + 1, F)
        ready = [s for s in ids if count[s] == F]
        if ready:
            if len(ready) not in bufs:
                bufs[len(ready)] = torch.empty(len(ready), F, *frames.shape[2:], device="cuda")
            clip = bufs[len(ready)]
            clip.copy_(window_clip(frames, t, ready))  # host-side re-assembly: not part of the timed work
        rec = {"start": tk.event()}
        rec["pushed"] = rec["start"]
        if ready:
            tok, _, _ = eng.caption(clip, sp)
            if t == n_warm + n_timed - 1:
                tokens = dict(zip(ready, tok[:, 0]))
            del tok
            if mode == "nonoverlap":
                for s in ready:
                    count[s] = 0
        rec["end"] = tk.event()
        rec["done"] = [(rec["end"], len(ready))] if ready else []
        if t >= n_warm:
            tk.ticks.append(rec)
    return tk.summary(S), tokens


def run_per_camera(g, engines, mode, S, frames, n_warm, n_timed, sp):
    """One Engine (context, weights, workspaces) per camera: a single-frame push per camera, one single-clip caption per window."""
    bufs = [torch.empty(*frames.shape[2:], device="cuda") for _ in range(S)]
    for e in engines:
        e.stream_reset()
    tk = Ticker()
    for t in range(n_warm + n_timed):
        ids = schedule(mode, S, t)
        for s in ids:
            bufs[s].copy_(frames[t % 7, s])
        rec = {"start": tk.event()}
        for s in ids:
            engines[s].stream_push(bufs[s])
        rec["pushed"] = tk.event()
        rec["done"] = []
        for s in ids:
            if engines[s].lib.gitb200_stream_frames(engines[s].h) == F:
                engines[s].stream_caption(sp)
                if mode == "nonoverlap":
                    engines[s].stream_reset()
                rec["done"].append((tk.event(), 1))
        rec["end"] = tk.event()
        if t >= n_warm:
            tk.ticks.append(rec)
    return tk.summary(S)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True, help="directory for bench_streams.json")
    ap.add_argument("--streams", default="1,16,64,256,512")
    ap.add_argument("--ticks", type=int, default=12, help="timed ticks per run (two phase periods)")
    ap.add_argument("--warmup", type=int, default=12, help="untimed ticks before them (>= 12 warms every shape twice)")
    ap.add_argument("--per-camera-max", type=int, default=16, help="largest camera count of the one-Engine-per-camera arm")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_streams.py needs a CUDA device: gitb200 has no CPU fallback")
    g = importlib.import_module("real-time-video-captioning_b200")
    gm = importlib.import_module("real-time-video-captioning_b200.model")
    # random-init weights through the package's reference-shaped constructor (as bench.py's build_engine): biases, LayerNorm
    # affines and temporal embeddings randomised so that no term of the path is trivially zero
    param = {"num_image_with_embedding": F}
    tok = gm.SyntheticTokenizer()
    torch.manual_seed(0)
    model = gm.get_git_model(tok, param)
    gen_w = torch.Generator().manual_seed(1)
    with torch.no_grad():
        for name, p_ in model.named_parameters():
            if name.endswith("bias") or "img_temperal_embedding" in name:
                p_.add_(torch.randn(p_.shape, generator=gen_w) * 0.02)
            elif p_.dim() == 1 and name.endswith("weight"):
                p_.add_(torch.randn(p_.shape, generator=gen_w) * 0.1)
    sd = model.state_dict()
    ccfg = g.make_config(param, tok.cls_token_id, tok.sep_token_id)
    sp = g.SearchConfig(beam_size=1, max_steps=MAX_STEPS)
    out = {"gpu": gpu_info(), "model": "GIT-base (ViT-B/16, 6-layer decoder), tied head, seeded random weights (bench.py build_engine recipe)",
           "window_frames": F, "search": "greedy, max_steps 16 (15 tokens after SOS)", "ticks": args.ticks, "warmup": args.warmup,
           "work_gflop_per_caption": {"sliding_pool": GFLOP_FRAME + GFLOP_PREFILL, "clip_baseline": GFLOP_CLIP_VIT + GFLOP_PREFILL},
           "results": []}
    side = torch.cuda.Stream()
    gen = torch.Generator(device="cuda").manual_seed(7)
    for S in [int(s) for s in args.streams.split(",")]:
        frames = torch.randn(7, S, 3, 224, 224, device="cuda", generator=gen)
        eng = g.Engine(ccfg, 0)
        eng.load_state_dict(sd)
        engines = []
        if S <= args.per_camera_max:
            for _ in range(S):
                e = g.Engine(ccfg, 0)
                e.load_state_dict(sd)
                engines.append(e)
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            for mode in ("nonoverlap", "sliding"):
                t0 = time.time()
                pool, tok_a = run_pool(g, eng, mode, S, frames, args.warmup, args.ticks, sp)
                base, tok_b = run_clip_baseline(g, eng, mode, S, frames, args.warmup, args.ticks, sp)
                same = [bool(torch.equal(tok_a[s], tok_b[s])) for s in tok_a if s in tok_b]
                rows = [("pool", pool), ("clip_baseline", base)]
                if engines:
                    rows.append(("per_camera_engines", run_per_camera(g, engines, mode, S, frames, args.warmup, args.ticks, sp)))
                for impl, r in rows:
                    r.update(streams=S, mode=mode, impl=impl)
                    out["results"].append(r)
                    print(json.dumps(r), flush=True)
                out["results"][-len(rows)]["last_tick_captions_equal_clip_baseline"] = f"{sum(same)}/{len(same)}"
                print(f"S={S} {mode}: {time.time() - t0:.1f} s wall, last-tick captions equal to the clip baseline: "
                      f"{sum(same)}/{len(same)}", flush=True)
        side.synchronize()
        for e in [eng] + engines:
            e.close()
        del frames
        torch.cuda.empty_cache()
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "bench_streams.json")
    with open(path, "w") as fh:
        json.dump(out, fh, indent=1)
    print(f"wrote {path}; {out['gpu']}")


if __name__ == "__main__":
    main()
