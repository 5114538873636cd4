"""Cost of the search settings a captioning user reaches for to get diverse or less repetitive captions: the fused device
search (gitb200_decode_ext) against today's greedy device search and against the generic host loop those settings took
before (GeneratorWithBeamSearchV2.search over gitb200_decode_step, one D2H copy per beam row and step for the saved logits,
Python repetition penalty, torch.sort top-p, a Python candidate walk).

GIT-base, 6-frame clips, captions of at most 15 tokens (max_steps 15), seeded random weights (untied head, so the searches
run their full length rather than stopping at an early EOS), clips resident in HBM: every clip is encoded once, and the
timed calls are the search over the resident visual features (visual pass included on the first call only, as for any
repeated decode; the host-loop arm too finds the features and their visual K/V resident).  Device arms are timed with CUDA
events over `--iters` calls after `--warmup` calls; the host-loop arm is timed with the host clock over one call after one
warm-up call per batch size, and stops growing the batch once a call exceeds `--host-cap` seconds.
Arms: greedy (nb 1), sampling nb 1 top-p 0.9, sampling nb 1 top-p 0.9 with 5 return sequences, beam 4 with repetition
penalty 1.2, host-loop sampling nb 1 top-p 0.9.  Writes one JSON file to --out.

    python tools/bench_sampling.py --out FILE [--clips 1,64,512] [--iters 5] [--warmup 2] [--host-clips 1,64]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

F = 6
MAX_STEPS = 15


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else f"nvidia-smi failed: {r.stderr.strip()}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--clips", default="1,64,512")
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--host-clips", default="1,64")
    ap.add_argument("--host-cap", type=float, default=120.0)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sampling needs a CUDA device (B200): there is no CPU measurement")
    g = importlib.import_module("real-time-video-captioning_b200")
    # bench.py's build_engine recipe (affines and temporal embeddings randomised so that no term of the path is trivially
    # zero) plus an untied vocabulary head
    torch.manual_seed(0)
    model = g.get_git_model(g.SyntheticTokenizer(), {"num_image_with_embedding": F})
    gen_w = torch.Generator().manual_seed(1)
    with torch.no_grad():
        for name, p_ in model.named_parameters():
            if name.endswith("bias") or "img_temperal_embedding" in name:
                p_.add_(torch.randn(p_.shape, generator=gen_w) * 0.02)
            elif p_.dim() == 1 and name.endswith("weight"):
                p_.add_(torch.randn(p_.shape, generator=gen_w) * 0.1)
    sd = model.state_dict()
    sd["textual.output.weight"] = torch.randn(sd["textual.output.weight"].shape, generator=gen_w) * 0.02
    model.load_state_dict(sd)
    model = model.cuda().eval()
    model.decoder.beam_size = 1  # the host-loop arm samples with one beam, like the device sampling arm
    eng = model.engine()

    sp = {"greedy": g.SearchConfig(beam_size=1, max_steps=MAX_STEPS),
          "beam4": g.SearchConfig(beam_size=4, max_steps=MAX_STEPS)}
    arms = {
        "device_greedy": (sp["greedy"], None),
        "device_sample_topp0.9": (sp["greedy"], g.SampleConfig(do_sample=True, top_k=0, top_p=0.9, seed=1)),
        "device_sample_topp0.9_nrs5": (sp["greedy"], g.SampleConfig(do_sample=True, top_k=0, top_p=0.9, num_return_sequences=5,
                                                                    seed=1)),
        "device_beam4_rp1.2": (sp["beam4"], g.SampleConfig(repetition_penalty=1.2, seed=1)),
    }
    out = {"gpu": gpu_info(), "model": "GIT-base, 6 frames, max_steps 15, untied head, seeded random weights (bench.py recipe)",
           "timing": f"CUDA events, {a.iters} calls after {a.warmup} warm-up calls; search over resident visual features",
           "results": []}
    gen = torch.Generator().manual_seed(0)
    for n in [int(x) for x in a.clips.split(",")]:
        frames = torch.randn(n, F, 3, 224, 224, generator=gen).cuda()
        vf = eng.encode(frames, want_features=True)
        del frames
        for name, (s, smp) in arms.items():
            eng.set_visual_features(vf)
            for _ in range(a.warmup):
                eng.decode(n, s, sample=smp)
            torch.cuda.synchronize()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for _ in range(a.iters):
                tok, _, _ = eng.decode(n, s, sample=smp)
            t1.record()
            torch.cuda.synchronize()
            ms = t0.elapsed_time(t1) / a.iters
            rows = n * (smp.num_return_sequences if smp else 1)
            r = {"arm": name, "clips": n, "captions": rows, "ms_per_call": ms, "captions_per_s": rows / ms * 1e3,
                 "steps": eng.last_decode_steps()}
            out["results"].append(r)
            print(json.dumps(r), flush=True)
        if n in [int(x) for x in a.host_clips.split(",")]:
            torch.manual_seed(0)
            for _ in range(2):  # warm-up call, then the timed one
                model._vf_token = vf  # the engine holds vf and its visual K/V since the device arms' calls: no re-upload
                torch.cuda.synchronize()
                t = time.perf_counter()
                model.infer({}, vf, None, {"do_sample": True, "top_k": 0, "top_p": 0.9})
                torch.cuda.synchronize()
                ms = (time.perf_counter() - t) * 1e3
            r = {"arm": "host_loop_sample_topp0.9", "clips": n, "captions": n, "ms_per_call": ms, "captions_per_s": n / ms * 1e3,
                 "calls": 1}
            out["results"].append(r)
            print(json.dumps(r), flush=True)
            if ms / 1e3 > a.host_cap:
                a.host_clips = ",".join(x for x in a.host_clips.split(",") if int(x) <= n)
        model._vf_token = None
        del vf
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps({"gpu": out["gpu"]}))


if __name__ == "__main__":
    main()
