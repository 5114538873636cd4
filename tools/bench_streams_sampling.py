"""Sampled live captions: the multi-stream pool with per-camera Philox keys (gitb200_streams_caption_ext) against the route
sampled live captions had before it, Engine.caption(..., sample=) on windows re-assembled as clips (every frame of a window
re-encoded).

GIT-base, 6-frame sliding windows (every camera pushes one frame and is captioned on every tick, over its last 6 frames),
captions of at most 15 tokens (max_steps 16), seeded random weights with an untied vocabulary head (bench.py's build_engine
recipe plus a random head, as tools/bench_sampling.py: sampled captions then run their full length instead of copying the
input), random preprocessed fp32 frames.  All work runs on one non-default stream so that every arm replays its CUDA graphs;
each arm runs --warmup untimed ticks, then --ticks timed ticks with CUDA events as in tools/bench_streams.py (the latency
of a caption is from the start of its tick to the end of the work that produced it; the clip arm's re-assembly of the
windows is a device copy before the tick starts).  The pool arms compute each camera's key with model.stream_key on the
host inside the tick, as MultiStreamCaptioner does.  Arms: pool greedy (gitb200_streams_caption), pool top-p 0.9, pool
top-p 0.9 with 5 return sequences, pool beam 4 with repetition penalty 1.2, and the clip route with each of the three
sampled / penalised settings.  Writes one JSON file to --out.

    python tools/bench_streams_sampling.py --out FILE [--streams 1,16,64,256,512] [--ticks 12] [--warmup 12]
"""
import argparse
import dataclasses
import importlib
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.dirname(os.path.abspath(__file__))):
    if p not in sys.path:
        sys.path.insert(0, p)
from bench_streams import F, Ticker, gpu_info, window_clip  # noqa: E402

MAX_STEPS = 15 + 1  # at most 15 tokens after SOS


def run_pool(eng, gm, S, frames, n_warm, n_timed, sp, sample, seed=1):
    """Sliding windows: every tick pushes frames[t % 7] for all S cameras and captions every full window."""
    eng.streams_configure(S)
    ids = list(range(S))
    tk = Ticker()
    n = 0  # captions each camera has received
    for t in range(n_warm + n_timed):
        rec = {"start": tk.event()}
        eng.streams_push(ids, frames[t % 7])
        rec["pushed"] = tk.event()
        rec["done"] = []
        if t >= F - 1:
            if sample is None:
                eng.streams_caption(ids, sp)
            else:
                eng.streams_caption(ids, sp, sample=sample, keys=[gm.stream_key(seed, s, n) for s in ids])
                n += 1
            rec["done"] = [(None, S * (sample.num_return_sequences if sample else 1))]
        rec["end"] = tk.event()
        rec["done"] = [(rec["end"], c) for _, c in rec["done"]]
        if t >= n_warm:
            tk.ticks.append(rec)
    return tk.summary(S)


def run_clips(eng, S, frames, n_warm, n_timed, sp, sample):
    """The same captions through Engine.caption on the windows re-assembled as clips (one seed per call)."""
    tk = Ticker()
    clip = torch.empty(S, F, *frames.shape[2:], device="cuda")
    for t in range(n_warm + n_timed):
        full = t >= F - 1
        if full:
            clip.copy_(window_clip(frames, t, list(range(S))))
        rec = {"start": tk.event()}
        rec["pushed"] = rec["start"]
        rec["done"] = []
        if full:
            eng.caption(clip, sp, sample=dataclasses.replace(sample, seed=t))
        rec["end"] = tk.event()
        if full:
            rec["done"] = [(rec["end"], S * sample.num_return_sequences)]
        if t >= n_warm:
            tk.ticks.append(rec)
    return tk.summary(S)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True, help="JSON file to write")
    ap.add_argument("--streams", default="1,16,64,256,512")
    ap.add_argument("--ticks", type=int, default=12)
    ap.add_argument("--warmup", type=int, default=12)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_streams_sampling.py needs a CUDA device: gitb200 has no CPU fallback")
    g = importlib.import_module("real-time-video-captioning_b200")
    gm = importlib.import_module("real-time-video-captioning_b200.model")
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
    sd = dict(model.state_dict())
    sd["textual.output.weight"] = torch.randn(sd["textual.output.weight"].shape, generator=gen_w) * 0.02
    del model
    ccfg = g.make_config(param, tok.cls_token_id, tok.sep_token_id)
    greedy = g.SearchConfig(beam_size=1, max_steps=MAX_STEPS)
    beam4 = g.SearchConfig(beam_size=4, max_steps=MAX_STEPS)
    settings = {
        "topp0.9": (greedy, g.SampleConfig(do_sample=True, top_k=0, top_p=0.9)),
        "topp0.9_nrs5": (greedy, g.SampleConfig(do_sample=True, top_k=0, top_p=0.9, num_return_sequences=5)),
        "beam4_rp1.2": (beam4, g.SampleConfig(repetition_penalty=1.2)),
    }
    out = {"gpu": gpu_info(),
           "model": "GIT-base (ViT-B/16, 6-layer decoder), untied head, seeded random weights (bench.py build_engine recipe + random head)",
           "window_frames": F, "mode": "sliding (every camera captioned on every tick over its last 6 frames)",
           "search": "max_steps 16 (15 tokens after SOS)",
           "captions": "every return sequence counts as a caption", "ticks": args.ticks, "warmup": args.warmup,
           "timing": "CUDA events on one non-default stream, per tick (tools/bench_streams.py method)", "results": []}
    side = torch.cuda.Stream()
    gen = torch.Generator(device="cuda").manual_seed(7)
    for S in [int(s) for s in args.streams.split(",")]:
        frames = torch.randn(7, S, 3, 224, 224, device="cuda", generator=gen)
        eng = g.Engine(ccfg, 0)
        eng.load_state_dict(sd)
        torch.cuda.synchronize()
        arms = [("pool_greedy", lambda: run_pool(eng, gm, S, frames, args.warmup, args.ticks, greedy, None))]
        for name, (sp, smp) in settings.items():
            arms.append((f"pool_{name}", lambda sp=sp, smp=smp: run_pool(eng, gm, S, frames, args.warmup, args.ticks, sp, smp)))
        for name, (sp, smp) in settings.items():
            arms.append((f"clip_{name}", lambda sp=sp, smp=smp: run_clips(eng, S, frames, args.warmup, args.ticks, sp, smp)))
        with torch.cuda.stream(side):
            for arm, fn in arms:
                r = fn()
                r.update(streams=S, arm=arm)
                out["results"].append(r)
                print(json.dumps(r), flush=True)
        side.synchronize()
        eng.close()
        del frames
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print(f"wrote {args.out}; {out['gpu']}")


if __name__ == "__main__":
    main()
