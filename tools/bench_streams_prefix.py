"""Prompted live captions: the multi-stream pool with a prompt (gitb200_streams_caption_prefix) against the pool without one and
against the route prompted live captions had before it, Engine.caption(..., prefix=) on windows re-assembled as clips (every
frame of a window re-encoded).

GIT-base, 6-frame sliding windows (every camera pushes one frame and is captioned on every tick, over its last 6 frames),
captions of at most 15 tokens (max_steps 16), seeded random weights with an untied vocabulary head (bench.py's build_engine
recipe plus a random head, as tools/bench_streams_sampling.py: captions then run their full length instead of copying the
input), random preprocessed fp32 frames.  Prompts of P = 5 tokens (SOS + 4 random tokens): one shared by every camera
([1, 5]), or one per camera ([k, 5]).  All work runs on one non-default stream so that every arm replays its CUDA graphs;
each arm runs --warmup untimed ticks, then --ticks timed ticks with CUDA events as in tools/bench_streams.py (the latency of
a caption is from the start of its tick to the end of the work that produced it; the clip arm's re-assembly of the windows
is a device copy before the tick starts).  Arms, greedy and beam 4 each: pool without a prompt, pool with the shared prompt,
pool with per-camera prompts, and the clip route with each of the two prompts.  The last tick's tokens of every prompted pool
arm are compared with the clip route's for the same prompts.  Reads the card's name, power limit and max SM clock in the same
run.  Writes one JSON file to --out.

    python tools/bench_streams_prefix.py --out FILE [--streams 1,16,64,256,512] [--ticks 12] [--warmup 12]
"""
import argparse
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
P = 5


def run_pool(eng, S, frames, n_warm, n_timed, sp, prefix):
    """Sliding windows: every tick pushes frames[t % 7] for all S cameras and captions every full window."""
    eng.streams_configure(S)
    ids = list(range(S))
    kw = {"prefix": prefix} if prefix is not None else {}
    tk = Ticker()
    tokens = None
    for t in range(n_warm + n_timed):
        rec = {"start": tk.event()}
        eng.streams_push(ids, frames[t % 7])
        rec["pushed"] = tk.event()
        rec["done"] = []
        if t >= F - 1:
            tokens, _ = eng.streams_caption(ids, sp, **kw)
            rec["done"] = [(None, S)]
        rec["end"] = tk.event()
        rec["done"] = [(rec["end"], c) for _, c in rec["done"]]
        if t >= n_warm:
            tk.ticks.append(rec)
    return tk.summary(S), tokens


def run_clips(eng, S, frames, n_warm, n_timed, sp, prefix):
    """The same captions through Engine.caption(..., prefix=) on the windows re-assembled as clips."""
    tk = Ticker()
    clip = torch.empty(S, F, *frames.shape[2:], device="cuda")
    tokens = None
    for t in range(n_warm + n_timed):
        full = t >= F - 1
        if full:
            clip.copy_(window_clip(frames, t, list(range(S))))
        rec = {"start": tk.event()}
        rec["pushed"] = rec["start"]
        rec["done"] = []
        if full:
            tokens, _, _ = eng.caption(clip, sp, prefix=prefix)
        rec["end"] = tk.event()
        if full:
            rec["done"] = [(rec["end"], S)]
        if t >= n_warm:
            tk.ticks.append(rec)
    return tk.summary(S), tokens


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True, help="JSON file to write")
    ap.add_argument("--streams", default="1,16,64,256,512")
    ap.add_argument("--ticks", type=int, default=12)
    ap.add_argument("--warmup", type=int, default=12)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_streams_prefix.py needs a CUDA device: gitb200 has no CPU fallback")
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
    searches = {"greedy": g.SearchConfig(beam_size=1, max_steps=MAX_STEPS), "beam4": g.SearchConfig(beam_size=4, max_steps=MAX_STEPS)}
    gen_p = torch.Generator().manual_seed(5)
    out = {"gpu": gpu_info(),
           "model": "GIT-base (ViT-B/16, 6-layer decoder), untied head, seeded random weights (bench.py build_engine recipe + random head)",
           "window_frames": F, "mode": "sliding (every camera captioned on every tick over its last 6 frames)",
           "search": "max_steps 16 (15 tokens after SOS); prompted arms run max_steps - P = 11 steps after the prompt's prefill",
           "prompt": f"P = {P}: SOS + {P - 1} random tokens, shared ([1, P]) or one per camera ([k, P])",
           "ticks": args.ticks, "warmup": args.warmup,
           "timing": "CUDA events on one non-default stream, per tick (tools/bench_streams.py method)", "results": []}
    side = torch.cuda.Stream()
    gen = torch.Generator(device="cuda").manual_seed(7)
    for S in [int(s) for s in args.streams.split(",")]:
        frames = torch.randn(7, S, 3, 224, 224, device="cuda", generator=gen)
        per_camera = torch.randint(1000, ccfg.vocab, (S, P), generator=gen_p, dtype=torch.int32)
        per_camera[:, 0] = tok.cls_token_id
        prompts = {"shared": per_camera[:1].clone(), "per_camera": per_camera}
        eng = g.Engine(ccfg, 0)
        eng.load_state_dict(sd)
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            for sname, sp in searches.items():
                runs = [(f"pool_{sname}_no_prompt", lambda sp=sp: run_pool(eng, S, frames, args.warmup, args.ticks, sp, None))]
                for pname, pre in prompts.items():
                    runs.append((f"pool_{sname}_{pname}",
                                 lambda sp=sp, pre=pre: run_pool(eng, S, frames, args.warmup, args.ticks, sp, pre)))
                    runs.append((f"clip_{sname}_{pname}",
                                 lambda sp=sp, pre=pre: run_clips(eng, S, frames, args.warmup, args.ticks, sp, pre)))
                last = {}
                for arm, fn in runs:
                    r, tokens = fn()
                    last[arm] = tokens
                    r.update(streams=S, arm=arm)
                    if arm.startswith("clip_"):
                        pool_tok = last[arm.replace("clip_", "pool_", 1)]
                        equal = int((pool_tok[:, 0] == tokens[:, 0]).all(dim=1).sum().item())
                        r["last_tick_captions_equal_pool"] = f"{equal}/{S}"
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
