#!/usr/bin/env python
"""Benchmark of the GIT captioning hot path (BASELINE.json metric: captions/sec on 6-frame clips).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # reference CPU implementation (oracle port)
    python bench.py ... --dump-outputs DIR                    # + the last timed step's tokens / log-probabilities as .npy

One "step" = one batch of synthetic 6 x 224 x 224 clips through the whole path: CLIP ViT-B/16 encode with temporal
embeddings, decoder pass over the visual tokens (K/V cache fill), 14 greedy decode steps (beam_size=1, max_steps=15,
the reference's search defaults with beam 1) and the device-side search.  Workload = BASELINE.json configs[1]
("GIT-base batched greedy decode, 6-frame MSR-VTT-shaped synthetic clips, bf16, 1 B200"); weights are random-init
(seeded), inputs are seeded randn clips.  Prints ONE JSON line (rank 0).

Timing: W warm-up steps, then K steps bracketed by barrier + cuda synchronize, timed with CUDA events on the launching
stream, max over ranks.  Each step reads a different resident batch of frames and streams > 4 GB of activations, far
beyond the 126 MB L2, so no explicit L2 flush is needed between iterations (config.l2 states this).

N > 1: every rank captions its own shard through the product's dist.caption_sharded; the token gather (the path's only
collective) is enqueued asynchronously behind each step and all gathers are waited for once, inside the timed region.

Besides the headline workload the default run times short legs of the other BASELINE.json configurations (key
"configs": beam 4 / max 20, GIT-large 6- and 24-frame) and the drop-in GenerativeImageTextTeacher.forward end to end.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "captions_per_sec_6frame_clips"
UNIT = "clips/s"
FRAMES, RES = 6, 224
# SURVEY.md 8(d) / BASELINE.md section 3: algorithmic tensor-core work per GIT-base 6-frame clip
GFLOP_PER_CLIP = 338.42


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            p = json.load(fh)
        return float(p["bf16_tflops_sustained"]), float(p["bf16_tflops"]), float(p["hbm_gbs"]), "measured"
    except Exception:
        return 1400.0, 1590.0, 6650.0, "fallback"  # B200_PROFILING.md fallback figures


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=self.tmp, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.tmp.flush()
        rows = [l.strip().split(", ") for l in open(self.tmp.name) if l.strip()]
        os.unlink(self.tmp.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for nm, v in zip(names, r[3:7]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        busy = [s for s in sm if s > 500] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ reference arm
def run_reference_cpu(steps: int, warmup: int, clips_per_step: int = 1):
    """Reference CPU implementation of the path = the oracle port in reference-faithful mode (per-frame ViT calls,
    hidden-state history with per-step K/V re-projection, Python search loop, per-step logits -> numpy), fp32, all host
    threads (BASELINE.md section 4; the reference itself cannot be imported: SURVEY.md 8c).  The result's "outputs" are
    the last step's (tokens [clips, 1, 15], logprobs [clips, 1])."""
    import torch
    from oracle import git_oracle as go
    from oracle import search_oracle as so

    torch.set_num_threads(os.cpu_count() or 1)
    cfg = go.GitConfig(num_image_with_embedding=FRAMES)
    sd = go.init_state_dict(cfg, seed=0, temporal_std=0.02, perturb=True)
    g = torch.Generator().manual_seed(1)
    clips = torch.randn(clips_per_step, FRAMES, 3, RES, RES, generator=g)
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            # the reference captions one clip at a time (model.py:765-770)
            res = [so.caption_clip(sd, cfg, c, per_frame_calls=True, beam_size=1, max_steps=15) for c in clips]
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    total = sum(times)
    outputs = (torch.cat([r["predictions"] for r in res])[:, None], torch.cat([r["logprobs"] for r in res]))
    return {"value": clips_per_step * len(times) / total, "ms_per_step": 1e3 * total / len(times), "outputs": outputs,
            "cores": torch.get_num_threads(), "p50_ms": 1e3 * statistics.median(times) / clips_per_step,
            "sample": f"{len(times)} steps x {clips_per_step} clip(s), greedy (beam 1, max_steps 15), fp32, after {warmup} warm-up"}


_JSON_FD = None


def claim_stdout():
    """The contract is ONE JSON line on stdout, but libraries chat there too (NCCL prints its version line to stdout under
    NCCL_DEBUG=VERSION/WARN): from here on file descriptor 1 points at stderr and emit() writes to the real stdout."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict) -> None:
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        os.write(1, data)
    else:
        os.write(_JSON_FD, data)


def dump_outputs(out_dir: str, tokens, logprobs) -> None:
    """tokens [clips, keep, max_steps] (integer ids) -> tokens.npy (float64: every int32 id exactly); logprobs [clips, keep] ->
    logprobs.npy (float32).  At the default geometry that is 512 x 15 tokens and 512 scores per GPU, well under 1 MB."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "tokens.npy"), tokens.cpu().numpy().astype(np.float64))
    np.save(os.path.join(out_dir, "logprobs.npy"), logprobs.cpu().numpy().astype(np.float32))


def pin_rank_to_cores(local_rank: int, world: int):
    """Give every rank of a node its own slice of the host cores (launch threads, pinned-copy staging and the Python
    post-processing of eight ranks otherwise share whatever cores the scheduler picks)."""
    try:
        cores = sorted(os.sched_getaffinity(0))
        per = len(cores) // max(world, 1)
        if world > 1 and per >= 2:
            mine = cores[local_rank * per:(local_rank + 1) * per]
            os.sched_setaffinity(0, mine)
            return len(mine)
        return len(cores)
    except Exception:
        return None


def roofline_model_clips_per_s(gflop_per_clip, kv_mb_per_clip, batch, max_steps, tc_tflops, hbm_gbs):
    """BASELINE.md section 3: 1 / (TC_FLOP / P_tc + (max_steps - 2) cached steps x (W_bytes / batch + KV_bytes) / BW)."""
    t = gflop_per_clip * 1e9 / (tc_tflops * 1e12) + (max_steps - 2) * (131.8e6 / batch + kv_mb_per_clip * 1e6) / (hbm_gbs * 1e9)
    return 1.0 / t


def build_engine(g, gm, torch, param, local_rank, seed=0):
    """Random-init weights through the package's own reference-shaped constructor (get_git_model, model.py:681-718); biases,
    LayerNorm affines and temporal embeddings (zeros upstream) randomised so that no term of the path is trivially zero."""
    tok = gm.SyntheticTokenizer()
    torch.manual_seed(seed)
    model = gm.get_git_model(tok, param)
    gen_w = torch.Generator().manual_seed(1)
    with torch.no_grad():
        for name, p_ in model.named_parameters():
            if name.endswith("bias") or "img_temperal_embedding" in name:
                p_.add_(torch.randn(p_.shape, generator=gen_w) * 0.02)
            elif p_.dim() == 1 and name.endswith("weight"):  # LayerNorm gains
                p_.add_(torch.randn(p_.shape, generator=gen_w) * 0.1)
    eng = g.Engine(g.make_config(param, tok.cls_token_id, tok.sep_token_id), local_rank)
    eng.load_state_dict(model.state_dict())
    return eng, model


def timed_leg(torch, dist, eng, frames_sets, sp, steps, warmup, world, dev, caption_sharded):
    """K steps of eng.caption over resident frame batches (+ the asynchronous token gather when world > 1): ms total,
    max over ranks."""
    B = frames_sets[0].shape[0]
    stream = torch.cuda.current_stream(dev)

    def step(i):
        fr = frames_sets[i % len(frames_sets)]
        return caption_sharded(lambda b, e: eng.caption(fr, sp)[:2], world * B, async_op=True, tail=(sp.num_keep_best, sp.max_steps))

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for h in [step(i) for i in range(warmup)]:
        h.wait()
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    handles = [step(i) for i in range(steps)]
    for h in handles:
        h.wait()
    e1.record(stream)
    sync_all()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.item(), handles


def config_leg(g, gm, torch, dist, name, param, B, frames_n, sp, steps, warmup, world, rank, local_rank, dev, gflop, kv_mb, peaks):
    """One short leg of another BASELINE.json configuration on its own engine."""
    eng, model = build_engine(g, gm, torch, param, local_rank)
    del model
    eng.reserve(B, frames_n, sp.beam_size, sp.max_steps)
    gen = torch.Generator(device=dev).manual_seed(300 + rank)
    sets = [torch.randn(B, frames_n, 3, RES, RES, device=dev, generator=gen) for _ in range(2)]
    caption_sharded = importlib.import_module("real-time-video-captioning_b200.dist").caption_sharded
    ms, _ = timed_leg(torch, dist, eng, sets, sp, steps, warmup, world, dev, caption_sharded)
    out = {"clips_per_gpu_per_step": B, "frames": frames_n, "beam_size": sp.beam_size, "max_steps": sp.max_steps, "steps": steps,
           "warmup": warmup, "ms_per_step": ms / steps, "value": world * B * steps / (ms * 1e-3), "unit": UNIT,
           "algorithmic_gflop_per_clip": gflop, "path_tflops_algorithmic": gflop * 1e9 * B * steps / (ms * 1e-3) / 1e12}
    sustained, burst, hbm, _ = peaks
    out["path_frac"] = out["path_tflops_algorithmic"] / sustained
    out["model_frac"] = (B * steps / (ms * 1e-3)) / roofline_model_clips_per_s(gflop, kv_mb, B, sp.max_steps, sustained, hbm)
    if sp.beam_size > 1:
        # roofline of the leg's HBM-bound kernel (decode-step attention, several beam rows per clip: the warp-level tensor body):
        # one more step with per-launch CUDA events on the launching stream (eager launches), as in the headline's profiled pass
        import ctypes
        eng.lib.gitb200_profile_gemm(1)
        eng.caption(sets[0], sp)
        torch.cuda.synchronize(dev)
        a_ms, a_by, a_n = ctypes.c_double(), ctypes.c_double(), ctypes.c_longlong()
        eng.lib.gitb200_profile_decode_attention_read(ctypes.byref(a_ms), ctypes.byref(a_by), ctypes.byref(a_n))
        eng.lib.gitb200_profile_gemm(0)
        if a_n.value > 0 and a_ms.value > 0:
            gbs = a_by.value / (a_ms.value * 1e-3) / 1e9
            out["roofline_decode"] = {"bound": "hbm", "kernel": "text_attention_kernel<4, 2> (decode-step attention, mma.sync body: the clip's beams share every K/V byte)",
                                      "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm, "launches_timed": int(a_n.value),
                                      "algorithmic_bytes_per_launch": a_by.value / a_n.value, "us_per_launch": 1e3 * a_ms.value / a_n.value,
                                      "share_of_step": a_ms.value / (ms / steps),
                                      "traffic": 962918400.0,
                                      "traffic_note": "dram read+write bytes of one launch at 256 clips x 4 beams, ncu --set full of the kernel alone (profiles/r02_text_attention_mma_raw.csv: 955.1 MB read + 7.8 MB written for 961 MB algorithmic)"}
    if name.startswith("large") and sp.max_steps > 2:
        # BASELINE.json configs[3] is an encode-heavy PREFILL sweep: encode + projection + the first decode step only
        sp2 = g.SearchConfig(beam_size=1, max_steps=2, length_penalty=0.6, per_node_beam_size=2, num_keep_best=1)
        ms2, _ = timed_leg(torch, dist, eng, sets, sp2, steps, 1, world, dev, caption_sharded)
        out["prefill_only"] = {"max_steps": 2, "ms_per_step": ms2 / steps, "value": world * B * steps / (ms2 * 1e-3), "unit": UNIT,
                               "path_tflops_algorithmic": gflop * 1e9 * B * steps / (ms2 * 1e-3) / 1e12}
    del sets
    eng.close()
    torch.cuda.empty_cache()
    return out


def teacher_forward_leg(g, gm, torch, dist, param, B, world, rank, dev, steps=3):
    """The drop-in itself: GenerativeImageTextTeacher.forward(x) (model.py:762-793) on a pinned HOST batch -- encode, beam-4 /
    max_steps-15 search (the reference's own settings, model.py:702-708), saved logits, per-clip result dicts with `output`
    and `cap` -- timed end to end by the wall clock, beside Engine.caption_host with the same search settings."""
    teacher = gm.GenerativeImageTextTeacher.from_random_init(param, device=dev)
    eng = teacher.model.engine()
    d = teacher.model.decoder
    sp = g.SearchConfig(beam_size=d.beam_size, max_steps=d.max_steps, length_penalty=d.length_penalty,
                        per_node_beam_size=d.per_node_beam_size, num_keep_best=1)
    eng.reserve(B, FRAMES, sp.beam_size, sp.max_steps)
    x = torch.randn(B, FRAMES, 3, RES, RES, generator=torch.Generator().manual_seed(70 + rank)).pin_memory()

    def wall(fn):
        for _ in range(3):  # warm-up: sizing call, CUDA-graph capture call, first replay
            r = fn()
            del r
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        r = None
        for _ in range(steps):
            del r  # a caller that keeps the previous batch's 3 GB of results alive makes every call cudaMalloc a new set
            r = fn()
        torch.cuda.synchronize(dev)
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item(), r

    t_engine, _ = wall(lambda: eng.caption_host(x, sp, chunk_clips=64))
    t_teacher, res = wall(lambda: teacher(x))
    out = {"api": "GenerativeImageTextTeacher.forward(x): pinned host frames -> list of per-clip dicts (predictions, logprobs, logits_dict, visual_features, output, cap)",
           "clips_per_gpu_per_step": B, "beam_size": sp.beam_size, "max_steps": sp.max_steps, "steps": steps,
           "value": world * B * steps / t_teacher, "unit": UNIT, "h2d_bytes_per_step": x.numel() * 4,
           "d2h_bytes_per_step": B * sp.max_steps * 8,
           "engine_caption_host_same_search": world * B * steps / t_engine,
           "teacher_over_engine": t_engine / t_teacher, "result_clips": len(res), "result_keys": sorted(res[0].keys())}
    del teacher, x, res
    eng.close()
    torch.cuda.empty_cache()
    return out


def distill_leg(g, gm, torch, dist, world, rank, local_rank, dev, steps=10, warmup=3):
    """BASELINE.json configs[4]: one distillation training step per GPU -- the frozen GIT-large teacher (shipped config: ViT-L/14, 6
    frames) gives teacher-forced logits for 8 clips x 20 caption tokens (forward_output_logits, model.py:896), the student
    DECODER (config.py:76-84) runs forward + KL/CE loss + backward + Adam on the library, gradients are all-reduced over the
    ranks (DDP average; the vocabulary-head bucket overlaps the layers' backward).  The student's TinyViT encoder is not part
    of the library: `memory` is synthetic."""
    sm = importlib.import_module("real-time-video-captioning_b200.student")
    param = {"image_encoder_type": "CLIPViT_L_14", "visual_feature_size": 1024, "num_image_with_embedding": 6}
    teacher = gm.GenerativeImageTextTeacher.from_random_init(param, device=dev)
    torch.manual_seed(0)
    student = sm.StudentCandidateV1(None, 576, 8, 1024, 0.3, 2, 30522, 101, 102).to(dev)
    trainer = sm.DistillationTrainer(teacher, student, lr=1e-4)
    B, L = 8, 20
    gen = torch.Generator(device=dev).manual_seed(500 + rank)
    x = torch.randn(B, 6, 3, RES, RES, device=dev, generator=gen)
    y = torch.randint(1000, 30000, (B, L), device=dev, generator=gen)
    y[:, 0] = 101
    mem = torch.randn(B, 6, 576, device=dev, generator=gen)
    batch = {"frames": x, "caption": y, "memory": mem}
    stream = torch.cuda.current_stream(dev)
    losses = []
    for _ in range(warmup):
        losses.append(trainer.training_step(batch))
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    e[0].record(stream)
    for _ in range(steps):
        losses.append(trainer.training_step(batch))
    e[1].record(stream)
    torch.cuda.synchronize(dev)
    t = torch.tensor([e[0].elapsed_time(e[1])], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = t.item() / steps
    # the student's share, timed on its own with fixed teacher logits; and the bare gradient all-reduce
    t_logits = trainer.teacher_logits(x, y)
    torch.cuda.synchronize(dev)
    e[0].record(stream)
    for _ in range(steps):
        student.distillation_step(y, mem, t_logits)
    e[1].record(stream)
    torch.cuda.synchronize(dev)
    student_ms = e[0].elapsed_time(e[1]) / steps
    ar_ms = None
    if world > 1:
        gbuf = student._grads
        dist.barrier()
        e[0].record(stream)
        for _ in range(steps):
            dist.all_reduce(gbuf)
        e[1].record(stream)
        torch.cuda.synchronize(dev)
        ar_ms = e[0].elapsed_time(e[1]) / steps
    out = {"workload": "BASELINE.json configs[4]: distillation step, GIT-large (6-frame) teacher logits + student decoder fwd/bwd/Adam, DDP gradient all-reduce",
           "clips_per_gpu_per_step": B, "caption_tokens": L, "steps": steps, "warmup": warmup, "ms_per_step": ms,
           "value": world * B / (ms * 1e-3), "unit": "clips/s (training)", "student_fwd_bwd_adam_allreduce_ms": student_ms,
           "teacher_share": 1.0 - student_ms / ms, "gradient_floats": int(student._grads.numel()),
           "allreduce_bytes_per_step": int(student._grads.numel()) * 4 if world > 1 else 0, "bare_allreduce_ms": ar_ms,
           "loss_first": float(losses[0]), "loss_last": float(losses[-1]), "dropout": "not applied (DESIGN.md)"}
    del trainer, teacher, student
    torch.cuda.empty_cache()
    return out


def _count(least: int):
    """argparse type: an integer >= least."""
    def parse(text: str) -> int:
        v = int(text)
        if v < least:
            raise argparse.ArgumentTypeError(f"must be >= {least}, got {v}")
        return v
    return parse


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=_count(1), default=6, help="timed steps (>= 1)")
    ap.add_argument("--warmup", type=_count(0), default=3, help="warm-up steps before the timed ones (the CUDA arm runs at least 4: "
                    "each of its two frame buffers is captured into CUDA graphs on its second use)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=512, help="clips per GPU per step (512: +3.5 %% over 256, the decode-step weights amortise over more rows)")
    ap.add_argument("--beam", type=int, default=1)
    ap.add_argument("--max-steps", type=int, default=15)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-clips", type=int, default=3, help="clips timed for the cpu_baseline leg")
    ap.add_argument("--chunk", type=int, default=64, help="clips per host->device chunk on the e2e path")
    ap.add_argument("--model", default="base", choices=["base", "large"], help="base = CLIPViT_B_16 (the metric's config); large = CLIPViT_L_14 (BASELINE.json configs[3], extra measurement)")
    ap.add_argument("--frames", type=int, default=6)
    ap.add_argument("--pipeline", type=int, default=0, help="clips per chunk of the two-stream encode/decode pipeline (0 off, -1 auto)")
    ap.add_argument("--fold-ln", action="store_true", help="opt-in: ViT LayerNorms folded into the QKV / fc1 GEMM epilogues (DESIGN.md dead ends)")
    ap.add_argument("--sweep-rows", type=int, default=-1, help="token rows per ViT / visual-pass sub-batch (-1: library default 151296 = 128 clips; 0: one sweep)")
    ap.add_argument("--quick", action="store_true", help="timed region only (no e2e / latency / cpu legs): for ncu captures")
    ap.add_argument("--no-config-legs", action="store_true", help="skip the short legs of the other BASELINE.json configurations and the teacher-forward leg")
    ap.add_argument("--early-exit", type=int, default=-1, help="poll the device's finished-clip count every N decode steps (-1: library default 4; 0: never)")
    ap.add_argument("--fuse-ln", action="store_true", help="opt-in: LayerNorms written by the residual GEMMs as a second output (DESIGN.md dead ends)")
    ap.add_argument("--no-graphs", action="store_true", help="A/B: eager launches instead of the CUDA graphs of encode / visual pass / decode segments")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's result to DIR/tokens.npy and "
                    "DIR/logprobs.npy, so that two builds can be compared output for output on the same seeded weights and clips: "
                    "all ranks' caption tokens and log-probabilities as the token gather returns them (with --impl reference: the "
                    "oracle's caption of its one clip, whose weights and clip are seeded apart from the CUDA arm's)")
    args = ap.parse_args()
    claim_stdout()

    global FRAMES, GFLOP_PER_CLIP
    FRAMES = args.frames
    param = {"num_image_with_embedding": FRAMES}
    if args.model == "large":
        param.update({"image_encoder_type": "CLIPViT_L_14", "visual_feature_size": 1024})
    if args.model == "large" or FRAMES != 6:  # algorithmic tensor work of the other BASELINE.md rows
        GFLOP_PER_CLIP = {("large", 6): 1149.51, ("large", 24): 5123.70}.get((args.model, FRAMES), float("nan"))
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    config = {"workload": ("GIT-base (CLIP ViT-B/16" if args.model == "base" else "GIT-large (CLIP ViT-L/14") + f" + 6-layer prefix-LM decoder) batched {'greedy' if args.beam == 1 else 'beam-' + str(args.beam)} caption, {FRAMES}x224x224 synthetic clips",
              "clips_per_gpu_per_step": args.batch, "frames": FRAMES, "beam_size": args.beam, "max_steps": args.max_steps,
              "weights": "random-init (seeded)", "parallelism": f"clip-sharded dp{world}",
              "pipeline": "two-stream chunk pipeline, auto chunk (batch/4 in [32,128])" if args.pipeline < 0 else (f"chunks of {args.pipeline}" if args.pipeline else "off"),
              "l2": f"no flush: every step streams >{args.batch * 60 // 1000} GB of activations and a {args.batch * 3.6128:.0f} MB frame batch (L2 = 126 MB)"}

    if args.impl == "reference":
        if rank != 0:
            return 0
        r = run_reference_cpu(args.steps, args.warmup, 1)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, *r["outputs"])
        line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "fp32", "data": "synthetic", "config": dict(config, clips_per_gpu_per_step=1, parallelism="cpu"),
                "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"]},
                "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "latency_ms_p50": r["p50_ms"]}
        emit(line)
        return 0

    import torch
    import torch.distributed as dist

    g = importlib.import_module("real-time-video-captioning_b200")
    gm = importlib.import_module("real-time-video-captioning_b200.model")
    caption_sharded = importlib.import_module("real-time-video-captioning_b200.dist").caption_sharded
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: gitb200 has no CPU fallback (use --impl reference for the CPU arm)")
    cores_mine = pin_rank_to_cores(local_rank, world)
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    config["host_cores_per_rank"] = cores_mine
    config["token_gather"] = "one packed all_gather_into_tensor per step, enqueued asynchronously (dist.caption_sharded), all waited for at the end of the timed region" if world > 1 else "none (1 rank)"

    # identical random-init weights on every rank (same seed); nothing under oracle/ is touched by this arm
    eng, model = build_engine(g, gm, torch, param, local_rank)
    del model
    sp = g.SearchConfig(beam_size=args.beam, max_steps=args.max_steps, length_penalty=0.6, per_node_beam_size=2, num_keep_best=1)
    B = args.batch
    eng.set_pipeline(args.pipeline)
    if args.sweep_rows >= 0:
        eng.set_sweep_rows(args.sweep_rows)
    if args.fold_ln:
        eng.set_fold_layernorm(True)
    if args.early_exit >= 0:
        eng.set_early_exit(args.early_exit)
    if args.pipeline == 0:
        eng.reserve(B, FRAMES, args.beam, args.max_steps)
    if args.fuse_ln:
        eng.set_fuse_layernorm(True)
    if args.no_graphs:
        eng.set_graph_segments(False)
    config["cuda_graphs"] = "off (eager launches)" if args.no_graphs else "encode + visual pass per frame buffer, decode loop per 4-step segment (finished-clip poll between segments)"

    gen = torch.Generator(device=dev).manual_seed(100 + rank)
    n_sets = 2  # alternate between resident frame batches
    frames = [torch.randn(B, FRAMES, 3, RES, RES, device=dev, generator=gen) for _ in range(n_sets)]
    stream = torch.cuda.current_stream(dev)

    def caption_local(i):
        return eng.caption(frames[i % n_sets], sp)[:2]

    def step(i):
        # C2: the caption tokens of all ranks are gathered (the path's only collective) -- asynchronously, one packed buffer
        return caption_sharded(lambda b, e: caption_local(i), world * B, async_op=True, tail=(1, args.max_steps))

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    eng.launch_count(reset=True)
    per_step_launches = 0
    for i in range(max(args.warmup, 2 * n_sets)):  # every frame buffer's graphs are captured on its second use
        step(i).wait()
        if i == 0:
            per_step_launches = eng.launch_count()  # an eager step: what a graph replay re-issues without passing the counter
    sync_all()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    graph0 = int(eng.lib.gitb200_graph_launches(eng.h))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    handles = [step(i) for i in range(args.steps)]
    for h in handles:
        h.wait()
    e1.record(stream)
    sync_all()
    ms = e0.elapsed_time(e1)
    graph_replays_timed = int(eng.lib.gitb200_graph_launches(eng.h)) - graph0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *handles[-1].wait())
    # every kernel of the step is this library's: a step issues `per_step_launches` of them (counted on the first, eager warm-up
    # step), whether they reach the GPU one by one or inside graph replays
    launches = per_step_launches * args.steps
    # ---- second, PROFILED pass of the same K steps for the roofline numbers: per-launch CUDA events around every GEMM and every
    # decode-step attention launch on the launching stream (the events keep those steps out of the CUDA graphs)
    import ctypes
    eng.lib.gitb200_profile_gemm(1)
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record(stream)
    for i in range(args.steps):
        caption_local(i)
    p1.record(stream)
    sync_all()
    ms_prof = p0.elapsed_time(p1)
    g_ms, g_fl, g_n = ctypes.c_double(), ctypes.c_double(), ctypes.c_longlong()
    eng.lib.gitb200_profile_gemm_read(ctypes.byref(g_ms), ctypes.byref(g_fl), ctypes.byref(g_n))
    a_ms, a_by, a_n = ctypes.c_double(), ctypes.c_double(), ctypes.c_longlong()
    eng.lib.gitb200_profile_decode_attention_read(ctypes.byref(a_ms), ctypes.byref(a_by), ctypes.byref(a_n))
    eng.lib.gitb200_profile_gemm(0)
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = t.item()
    value = world * B * args.steps / (ms * 1e-3)
    # the gathered matrix must hold this rank's own result at this rank's shard (clip order preserved)
    gathered_ok = None
    if world > 1:
        all_tok, all_lp = handles[-1].wait()
        mine_tok, _ = caption_local(args.steps - 1)
        gathered_ok = bool(all_tok.shape[0] == world * B and torch.equal(all_tok[rank * B:(rank + 1) * B], mine_tok.to(torch.int32)))
        assert gathered_ok, "gathered tokens differ from the local shard"

    if args.quick:
        if rank == 0:
            emit({"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                  "ms_per_step": ms / args.steps, "gpu_launches": launches, "quick": True, "graph_replays": graph_replays_timed,
                  "ms_per_step_profiled_pass": ms_prof / args.steps,
                  "gemm_ms": g_ms.value, "gemm_tflops": g_fl.value / max(g_ms.value, 1e-9) / 1e9})
        if world > 1:
            dist.destroy_process_group()
        return 0

    def wall_leg(fn, n):
        fn()  # warm-up (allocates staging buffers)
        sync_all()
        t0 = time.perf_counter()
        for _ in range(n):
            r = fn()
        sync_all()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return world * B * n / t.item(), r

    e2e_steps = max(2, min(args.steps, 6))
    # ---- e2e: the same metric through the public host-buffer API, from RAW video frames (uint8 BGR 240x320, MSR-VTT's frame
    # size, what cv2.VideoCapture delivers: dataloader.py:61-75): bytes over PCIe, image_transform() on the GPU, host tokens out
    raw_frames = torch.randint(0, 256, (B, FRAMES, 240, 320, 3), dtype=torch.uint8,
                               generator=torch.Generator().manual_seed(17 + rank)).pin_memory()
    e2e_value, (tok_h, lp_h) = wall_leg(lambda: eng.caption_host_u8(raw_frames, sp, chunk_clips=args.chunk), e2e_steps)
    d2h = tok_h.numel() * 4 + lp_h.numel() * 4
    e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": raw_frames.numel(), "d2h_bytes_per_step": d2h, "steps": e2e_steps,
           "api": "Engine.caption_host_u8 (gitb200_caption_host_u8): pinned host uint8 BGR 240x320 frames -> GPU image_transform -> host tokens"}
    del raw_frames
    # ---- the same from frames the host has already preprocessed (fp32 224x224: 4x the bytes over PCIe)
    host_frames = torch.randn(B, FRAMES, 3, RES, RES, generator=torch.Generator().manual_seed(7 + rank)).pin_memory()
    e2e_f32_value, _ = wall_leg(lambda: eng.caption_host(host_frames, sp, chunk_clips=args.chunk), e2e_steps)
    e2e_f32 = {"value": e2e_f32_value, "unit": UNIT, "h2d_bytes_per_step": host_frames.numel() * 4, "d2h_bytes_per_step": d2h,
               "steps": e2e_steps, "api": "Engine.caption_host (gitb200_caption_host): pinned host fp32 frames -> host tokens"}
    del host_frames

    # ---- single-clip latency (p50) on rank 0: same buffers every call on a side stream, as a real-time caller would
    # do (the library replays a CUDA graph of the ~850 launches from the third identical call on)
    p50 = p50_stream = graph_replays = None
    if rank == 0:
        one = frames[0][:1].contiguous()
        lat = []
        side = torch.cuda.Stream(dev)
        import ctypes as _ct
        tok1 = torch.empty(1, 1, args.max_steps, dtype=torch.int32, device=dev)
        lp1 = torch.empty(1, 1, dtype=torch.float32, device=dev)
        csp = sp.to_c()
        torch.cuda.synchronize(dev)
        with torch.cuda.stream(side):
            for i in range(30):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(side)
                rc = eng.lib.gitb200_caption(eng.h, _ct.c_void_p(one.data_ptr()), 1, FRAMES, _ct.byref(csp), _ct.c_void_p(tok1.data_ptr()),
                                             _ct.c_void_p(lp1.data_ptr()), None, _ct.c_void_p(side.cuda_stream))
                assert rc == 0, eng.lib.gitb200_last_error(eng.h)
                b.record(side)
                b.synchronize()
                if i >= 8:
                    lat.append(a.elapsed_time(b))
        p50 = statistics.median(lat)
        graph_replays = int(eng.lib.gitb200_graph_launches(eng.h))
        # streaming caller (real_time_inference.py loop): the 6-frame window is already encoded frame by frame; what stands
        # between a new frame and its caption is ONE frame's ViT + the decoder
        lat_s = []
        with torch.cuda.stream(side):
            eng.stream_reset()
            for f in range(FRAMES):
                eng.stream_push(one[0, f])
            for i in range(40):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(side)
                eng.stream_push(one[0, i % FRAMES])
                eng.stream_caption(sp)
                b.record(side)
                b.synchronize()
                if i >= 18:  # every (frame slot, window start) signature has been captured by then
                    lat_s.append(a.elapsed_time(b))
        p50_stream = statistics.median(lat_s)
    del frames
    eng.close()
    torch.cuda.empty_cache()

    # ---- the other BASELINE.json configurations (short legs, every rank) and the drop-in teacher wrapper
    peaks = measured_peaks()
    sustained, burst, hbm, src = peaks
    legs = {}
    if not args.no_config_legs and args.model == "base" and FRAMES == 6:
        base_param = {"num_image_with_embedding": 6}
        large6 = {"image_encoder_type": "CLIPViT_L_14", "visual_feature_size": 1024, "num_image_with_embedding": 6}
        large24 = {"image_encoder_type": "CLIPViT_L_14", "visual_feature_size": 1024, "num_image_with_embedding": 24}
        greedy = g.SearchConfig(beam_size=1, max_steps=15, length_penalty=0.6, per_node_beam_size=2, num_keep_best=1)
        beam4 = g.SearchConfig(beam_size=4, max_steps=20, length_penalty=0.6, per_node_beam_size=2, num_keep_best=1)
        legs["beam4_max20"] = dict(config_leg(g, gm, torch, dist, "beam4_max20", base_param, 256, 6, beam4, 3, 2, world, rank, local_rank, dev,
                                              338.42, 21.8, peaks), workload="BASELINE.json configs[2]: GIT-base beam 4 / max 20 tokens, visual K/V shared by a clip's beams, clip-sharded")
        legs["large_f6"] = dict(config_leg(g, gm, torch, dist, "large_f6", large6, 128, 6, greedy, 3, 2, world, rank, local_rank, dev,
                                           1149.51, 28.4, peaks), workload="GIT-large (ViT-L/14) 6-frame clips: the shipped teacher config (parameter.yaml), greedy max 15")
        legs["large_f24"] = dict(config_leg(g, gm, torch, dist, "large_f24", large24, 32, 24, greedy, 3, 2, world, rank, local_rank, dev,
                                            5123.70, 113.7, peaks), workload="BASELINE.json configs[3]: GIT-large (ViT-L/14) 24-frame clips, greedy max 15 + prefill-only sweep")
        legs["e2e_teacher_forward"] = teacher_forward_leg(g, gm, torch, dist, base_param, 256, world, rank, dev)
        legs["distill_step"] = distill_leg(g, gm, torch, dist, world, rank, local_rank, dev)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    gemm_tflops = (g_fl.value / (g_ms.value * 1e-3) / 1e12) if g_ms.value > 0 else None
    traffic = None
    try:  # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture
        with open(os.path.join(ROOT, "profiles", "r02_gemm2_traffic.json")) as fh:
            traffic = json.load(fh)["traffic_bytes_per_launch_avg"]
    except Exception:
        pass
    path_tflops = GFLOP_PER_CLIP * 1e9 * B * args.steps / (ms * 1e-3) / 1e12
    kv_mb = {("base", 6): 21.8, ("large", 6): 28.4, ("large", 24): 113.7}.get((args.model, FRAMES), float("nan"))
    model_clips = roofline_model_clips_per_s(GFLOP_PER_CLIP, kv_mb, B, args.max_steps, sustained, hbm)
    roofline = {"bound": "tensor", "kernel": "gemm2_kernel (2-CTA tcgen05) + gemm_tcgen05_kernel<128> (decode rows)",
                "achieved": gemm_tflops, "peak": sustained,
                "unit": "TFLOP/s", "frac": (gemm_tflops / sustained) if gemm_tflops else None, "traffic": traffic,
                "traffic_note": "avg DRAM read+write bytes per launch of the 4 ViT-layer GEMMs at M=151296 (one 128-clip sub-batch of the 512-clip step; algorithmic average 1.049 GB; profiles/r02_gemm2_traffic.json)",
                "peak_source": f"{src} bf16_tflops_sustained (kernel timed inside a long step)",
                "launches_timed": g_n.value, "gemm_share_of_step": g_ms.value / ms_prof if ms_prof > 0 else None,
                "timed_in": "a second pass of the same K steps with per-launch CUDA events on the launching stream (eager launches)",
                "ms_per_step_profiled_pass": ms_prof / args.steps,
                "algorithmic_gflop_per_clip": GFLOP_PER_CLIP,
                "path_tflops_algorithmic": path_tflops,
                # whole path against the tensor peak alone, and against BASELINE.md section 3's tensor + HBM model
                "path_frac": path_tflops / sustained,
                "model_clips_per_s_per_gpu": model_clips,
                "model_frac": (B * args.steps / (ms * 1e-3)) / model_clips}

    # second roofline: the HBM-bound kernel of the path (decode-step attention over the visual + text K/V cache)
    dec_gbs = (a_by.value / (a_ms.value * 1e-3) / 1e9) if a_ms.value > 0 else None
    dec_traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "r02_text_attention_traffic.json")) as fh:
            dec_traffic = json.load(fh)["traffic_bytes_per_launch_avg"]
    except Exception:
        pass
    roofline_decode = {"bound": "hbm", "kernel": "text_attention_kernel (decode-step attention, visual K/V shared by a clip's beams)",
                       "achieved": dec_gbs, "peak": hbm, "unit": "GB/s", "frac": (dec_gbs / hbm) if (dec_gbs and hbm) else None,
                       "traffic": dec_traffic,
                       "traffic_note": "dram read+write bytes per launch, ncu capture of the first decode step's 6 launches at 512 clips (profiles/r02_text_attention_traffic.json)",
                       "peak_source": f"{src} hbm_gbs (copy bandwidth)", "launches_timed": a_n.value,
                       "algorithmic_bytes_per_launch": (a_by.value / a_n.value) if a_n.value else None,
                       "share_of_step": (a_ms.value / ms_prof) if ms_prof > 0 else None}

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        r = run_reference_cpu(args.cpu_clips, 1, 1)
        cpu_baseline = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"],
                        "p50_ms": r["p50_ms"]}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "config": config, "clocks": clocks, "gpu_launches": launches, "graph_replays_in_timed_region": graph_replays_timed,
            "e2e": e2e, "e2e_fp32_frames": e2e_f32, "gathered_tokens_match_local_shard": gathered_ok,
            "roofline": roofline, "roofline_decode": roofline_decode, "cpu_baseline": cpu_baseline, "latency_ms_p50_single_clip": p50,
            "latency_cuda_graph_replays": graph_replays, "latency_ms_p50_streaming_new_frame_to_caption": p50_stream,
            "configs": legs}
    emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
