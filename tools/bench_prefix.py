"""Cost of prompted captions (batch['prefix'], GIT's prompted captioning / question answering): the fused device search with
a prompt (gitb200_decode_prefix: one teacher-forced decoder pass over the prompt, then the device search from cur_len = P)
against the generic host loop a prompt took before (GeneratorWithBeamSearchV2.search over gitb200_decode_step: the prompt
fed one token per step, every step's logits copied to the host, a Python candidate walk).

GIT-base, 6-frame clips, max_steps 20, seeded random weights (untied head, so that searches run their full length), clips
resident in HBM: every clip is encoded once and the timed calls are the search over the resident visual features.  Grid: prompt
length P in {1, 5, 10} (SOS plus random tokens, one prompt shared by every clip), greedy and beam 4, 1 / 64 / 512 clips.  Device
arms are timed with CUDA events over `--iters` calls after `--warmup` calls.  Host-loop arm: at 1 clip `infer` as it is without
search_param['device_prefix']; above 1 clip the same generic `search` with a [clips, P] start (infer takes one prompt row only);
one call after one warm-up call, host clock around a device synchronise, skipped above `--host-max-clips`.
Reads the card's name, power limit and max SM clock in the same run.  Writes one JSON file to --out.

    python tools/bench_prefix.py --out FILE [--clips 1,64,512] [--prompts 1,5,10] [--iters 5] [--warmup 2] [--host-max-clips 64]
"""
import argparse
import functools
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
MAX_STEPS = 20


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else f"nvidia-smi failed: {r.stderr.strip()}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--clips", default="1,64,512")
    ap.add_argument("--prompts", default="1,5,10")
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--host-max-clips", type=int, default=64)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_prefix needs a CUDA device (B200): there is no CPU measurement")
    g = importlib.import_module("real-time-video-captioning_b200")
    # bench.py's build_engine recipe (affines and temporal embeddings randomised) plus an untied vocabulary head
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
    model.decoder.max_steps = MAX_STEPS
    eng = model.engine()
    sos = model.sos_index

    out = {"gpu": gpu_info(), "model": f"GIT-base, {F} frames, max_steps {MAX_STEPS}, untied head, seeded random weights (bench.py recipe)",
           "timing": f"device: CUDA events, {a.iters} calls after {a.warmup} warm-up calls; host loop: one call after one warm-up, "
                     "host clock around a device synchronise; search over resident visual features",
           "results": []}
    gen = torch.Generator().manual_seed(0)
    prompts = {P: torch.cat([torch.tensor([[sos]]), torch.randint(1000, 30000, (1, P - 1), generator=gen)], 1)
               for P in [int(x) for x in a.prompts.split(",")]}
    for n in [int(x) for x in a.clips.split(",")]:
        frames = torch.randn(n, F, 3, 224, 224, generator=gen).cuda()
        vf = eng.encode(frames, want_features=True)
        del frames
        for P, prompt in prompts.items():
            for nb in (1, 4):
                sp = g.SearchConfig(beam_size=nb, max_steps=MAX_STEPS)
                eng.set_visual_features(vf)
                for _ in range(a.warmup):
                    ref = eng.decode(n, sp, prefix=prompt)
                torch.cuda.synchronize()
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record()
                for _ in range(a.iters):
                    eng.decode(n, sp, prefix=prompt)
                t1.record()
                torch.cuda.synchronize()
                ms = t0.elapsed_time(t1) / a.iters
                r = {"arm": "device_prefix", "P": P, "beam": nb, "clips": n, "ms_per_call": ms, "captions_per_s": n / ms * 1e3,
                     "steps": eng.last_decode_steps()}
                if n <= a.host_max_clips:
                    model.decoder.beam_size = nb
                    for _ in range(2):  # warm-up call, then the timed one
                        model._vf_token = vf  # the engine holds vf and its visual K/V: no re-upload in the host arm either
                        model.prev_encoded_layers = None
                        torch.cuda.synchronize()
                        t = time.perf_counter()
                        if n == 1:
                            host = model.infer({"prefix": prompt}, vf, None, {})["predictions"]
                        else:
                            step = functools.partial(model.decoding_step, vf, None, None)
                            host = model.decoder.search(prompt.expand(n, P).long().cuda(), step)[0][:, P:]
                        torch.cuda.synchronize()
                        host_ms = (time.perf_counter() - t) * 1e3
                    dev = ref[0][:, 0, P:].long().cpu()
                    r.update({"host_loop_ms_per_call": host_ms, "speedup_vs_host_loop": host_ms / ms,
                              "captions_equal_to_host_loop": float((dev == host.cpu()).all(dim=1).float().mean())})
                out["results"].append(r)
                print(json.dumps(r), flush=True)
        model._vf_token = None
        del vf
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps({"gpu": out["gpu"]}))


if __name__ == "__main__":
    main()
