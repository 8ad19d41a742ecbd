#!/usr/bin/env python
"""Benchmark of the WCT inference hot path (BASELINE.json metric: 512x512 five-level
stylised frames/sec), one process per GPU.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl reference] [--dump-outputs DIR]

A "step" = one pass of the hot path (WCT.predict semantics: encode style, then
[encode -> WCT -> decode] x relu5_1..relu1_1, wct_tf semantics, alpha=0.8) over one batch
of B synthetic 512x512 RGB frames, EACH WITH ITS OWN 512x512 STYLE (so the style is
re-encoded and re-decomposed per frame exactly as the reference does per predict call --
no work is shared or cached between frames).

  value   frames/s, inputs (uint8 frames) already resident in HBM, CUDA-event timed
  e2e     frames/s through the public API (WCT.predict_batch) with PINNED HOST uint8
          buffers: H2D of contents+styles and D2H of the uint8 results inside the timed region
  roofline  the dominant kernel = conv_tc2_kernel (tcgen05 implicit-GEMM conv): EXECUTED algorithmic conv
          FLOPs (2*taps*Cin*Cout per output pixel; 4 taps for the convs that absorbed an UpSampling2D) /
          CUDA-event time of those launches, vs the measured bf16 peak; per-level tensor-pipe fractions and
          covariance-only HBM GB/s beside it (north_star)
  cpu_baseline  the oracle (CPU restatement of the reference, torch-CPU convs + NumPy/LAPACK
          transform) timed on the host cores on ONE frame of the same workload

--impl reference: TensorFlow 1.x / Keras 2.0.9 are not installable offline, so the
reference arm is the oracle port run on all host threads (kind "port").

--dump-outputs DIR: after the timed steps, rank 0 writes the uint8 frames its last timed resident step
returned as DIR/output.npy (float32, B x 512 x 512 x 3).  Inputs and weights are seeded, so two builds run
with the same arguments can be compared output for output.  A batch above 64 MB in float32 is cut to a
seeded sample of whole frames; DIR/output_frames.npy (float64) then lists which frames of the batch they are.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

TARGETS = ["relu5_1", "relu4_1", "relu3_1", "relu2_1", "relu1_1"]
SIZE = 512
ALPHA = 0.8
SEMANTICS = "tf"   # what stylize.py actually executes (model.py:154,158)
DUMP_BYTES = 64 * 10 ** 6

WORKLOAD = ("configs[1]: 5-level relu5_1->relu1_1, 512x512 content, 512x512 style per frame, alpha=0.8, "
            "wct_tf semantics")

# algorithmic FLOPs per frame, style re-encoded per frame (BASELINE.md section 3)
GFLOP_PER_FRAME = 1050.10


def frames(n, seed):
    rng = np.random.default_rng(seed)
    return rng.integers(0, 256, (n, SIZE, SIZE, 3), dtype=np.uint8)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d.get("hbm_gbs", 6650.0), tf=d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0)),
                    source="MEASURED_PEAKS.json (bf16_tflops_sustained)")
    return dict(hbm_gbs=6650.0, tf=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.t.start()
            # wait for the first sample: NVML start-up of the freshly spawned nvidia-smi takes 0.3-1 s and touches the
            # driver; it must be over before the warm-up / timed steps begin (it then samples every 100 ms during them)
            t0 = time.time()
            while not self.lines and time.time() - t0 < 15.0 and self.proc.poll() is None:
                time.sleep(0.05)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), power_w_max=float(max(pw)),
                    samples=len(sm), reasons=sorted(reasons))


def cpu_frame_seconds(weights, n_frames=1, threads=None):
    """Time the oracle port on the host: full 5-level 512x512 frame(s), fp32, all threads."""
    import torch
    from oracle import nets
    if threads:
        torch.set_num_threads(threads)
    c, s = frames(n_frames, 1000), frames(n_frames, 7)
    t0 = time.time()
    for i in range(n_frames):
        nets.pipeline(c[i], s[i], weights, TARGETS, alpha=ALPHA, semantics=SEMANTICS, dtype=np.float32)
    return (time.time() - t0) / n_frames


def make_config(world, B, adain, groups, scaling, global_batch):
    """The `config` object of the JSON line -- identical for the GPU arm and the --impl reference arm."""
    cfg = {"workload": WORKLOAD if not adain else WORKLOAD.replace("wct_tf semantics", "AdaIN (configs[4])"),
           "frames_per_gpu_per_step": B, "global_batch": global_batch, "parallelism": "frame-sharded dp%d" % world,
           "style": "one distinct style per frame, re-encoded every step (no caching)",
           "l2": "two input sets alternate; per-step activation working set (>5 GB) >> 126 MB L2",
           "precision": "fp32-class: split-fp16 pairs (22-23 bits, power-of-two scaled weights) x3 products on tcgen05, "
                        "fp32 accumulate (TMEM chunks of 4 k-iterations summed in registers)",
           "transform": "whitening / colouring matrices per frame and level from the frame's own covariances: coupled Newton-Schulz "
                        "on tcgen05 where the 1e-5 threshold provably keeps every eigenvalue (all matrices of this synthetic "
                        "workload: k = C), Jacobi eigendecomposition otherwise",
           "streams": "%d sub-batch group(s) per step, each a (content, style) stream pair" % groups}
    if scaling == "strong":
        cfg["workload"] = ("configs[2]: batch of %d 512x512 frames, ONE shared 512x512 style, 5 levels, alpha=0.8, wct_tf "
                           "semantics, contiguous shards of B/G frames per GPU (parallel.stylize_sharded)" % global_batch)
        cfg["style"] = "one shared style, re-encoded on every GPU every step"
    return cfg


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port) on this box's host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import torch
    from wct_tf_b200.weights import make_synthetic_weights
    from oracle import nets
    host_cores = os.cpu_count() or 1
    threads = min(host_cores, 32)            # torch-CPU convs of this size get slower beyond ~32 threads
    torch.set_num_threads(threads)
    weights = make_synthetic_weights(42)
    c, s = frames(1, 1000), frames(1, 7)
    times = []
    for i in range(args.warmup + args.steps):
        t0 = time.time()
        nets.pipeline(c[0], s[0], weights, TARGETS, alpha=ALPHA, semantics=SEMANTICS, dtype=np.float32)
        if i >= args.warmup:
            times.append(time.time() - t0)
    ms = 1000.0 * float(np.mean(times))
    value = 1000.0 / ms
    world = max(1, args.gpus)
    gb = args.global_batch if args.scaling == "strong" else world * args.batch
    line = {
        "impl": "reference", "metric": "512x512 5-level WCT stylised frames/sec", "value": value, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": len(times), "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": make_config(world, args.batch if args.scaling == "weak" else gb // world, args.adain, max(1, args.groups),
                              args.scaling, gb),
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": host_cores, "threads": threads, "kind": "port",
                         "sample": "%d timed step(s) of ONE full frame each (a bounded sample of the workload: per-frame "
                                   "work is identical, the CPU arm does not batch); TensorFlow/Keras not installable "
                                   "offline -> oracle port (torch-CPU convs + NumPy/LAPACK wct_tf)" % len(times)},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


def dump_outputs(d, frames_u8):
    """Write the frames (uint8, B x H x W x 3) as float32 .npy files under d, at most DUMP_BYTES in all."""
    os.makedirs(d, exist_ok=True)
    frames_u8 = np.asarray(frames_u8)
    per_frame = frames_u8[0].size * 4
    fit = (DUMP_BYTES - 4096) // per_frame                         # 4 KB for the .npy headers and output_frames.npy
    if frames_u8.shape[0] > fit:
        idx = np.sort(np.random.default_rng(0).choice(frames_u8.shape[0], fit, replace=False))
        np.save(os.path.join(d, "output_frames.npy"), idx.astype(np.float64))
        frames_u8 = frames_u8[idx]
    np.save(os.path.join(d, "output.npy"), frames_u8.astype(np.float32))


def level_of_key(key):
    return key.split(":", 1)[0] if ":" in key else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=30, help="frames per GPU per step (30 = two sub-batches of 15: at most 15 eigensolver clusters of 8 CTAs are co-resident on a B200)")
    ap.add_argument("--impl", type=str, default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--adain", action="store_true", help="config 5: AdaIN instead of WCT")
    ap.add_argument("--scaling", choices=["weak", "strong"], default="weak",
                    help="weak: --batch frames per GPU, one style per frame (configs[1]); strong: configs[2], --global-batch "
                         "frames with ONE shared style sharded over the GPUs through parallel.stylize_sharded")
    ap.add_argument("--global-batch", type=int, default=64)
    ap.add_argument("--oversub", type=int, default=0, help="tuning: conv CTAs per SM (0 = library default)")
    ap.add_argument("--no-overlap", action="store_true", help="tuning: run the style side on the main stream")
    ap.add_argument("--groups", type=int, default=2, help="sub-batches per step run as independent stream pairs")
    ap.add_argument("--no-prio", action="store_true", help="tuning: all streams at the same priority")
    ap.add_argument("--no-fuse-upsample", action="store_true", help="tuning: separate upsample2 kernels + 9-tap convs")
    ap.add_argument("--no-fuse-pool", action="store_true", help="tuning: separate maxpool2 kernels after conv1_2/2_2/3_4/4_4")
    ap.add_argument("--no-roofline", action="store_true", help="skip the per-kernel profiling steps")
    ap.add_argument("--jacobi-tolq", type=float, default=0.0, help="tuning: eigensolver predicted-convergence level (0 = library default)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the frames of the last timed step to DIR/output.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the frames of the GPU path; it does not apply to --impl reference")
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from wct_tf_b200 import _capi, parallel
    from wct_tf_b200.engine import Engine
    from wct_tf_b200.weights import make_synthetic_weights
    from wct_tf_b200.wct import WCT

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert args.warmup >= 3, "timing rules: >= 3 warm-up steps"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    strong = args.scaling == "strong"
    GB = args.global_batch if strong else world * args.batch
    lo, hi = parallel.shard_range(GB, world, rank) if strong else (rank * args.batch, (rank + 1) * args.batch)
    B = hi - lo                                          # frames this rank processes per step
    weights = make_synthetic_weights(42)
    wct = WCT(relu_targets=TARGETS, device="cuda:%d" % local, weights=weights, semantics=SEMANTICS)
    if args.no_fuse_upsample or args.no_fuse_pool:
        wct.engine = Engine(weights, TARGETS, device="cuda:%d" % local, semantics=SEMANTICS, fuse_upsample=not args.no_fuse_upsample,
                            fuse_pool=not args.no_fuse_pool)
    eng = wct.engine
    if args.oversub:
        eng.lib.wctb200_debug_set_conv_oversub(args.oversub)
    if args.jacobi_tolq > 0:
        eng.lib.wctb200_debug_set_jacobi_tolq(args.jacobi_tolq)
    if args.no_overlap:
        eng.overlap_style = False
    eng.groups = max(1, args.groups)
    eng.group_priorities = not args.no_prio

    # two input sets rotated between steps.  weak: distinct frames AND styles per rank; strong: the global batch is the same
    # on every rank (frame i -> rank floor(i*G/B), parallel.shard_range), one shared style.
    sets = []
    for j in range(2):
        if strong:
            c = frames(GB, 1000 + 1000 * j)[lo:hi]
            s = frames(1, 7 + 1000 * j)
        else:
            c = frames(B, 1000 + 17 * rank + 1000 * j)
            s = frames(B, 7 + 31 * rank + 1000 * j)
        sets.append((c, s))
    dev_sets = [(torch.from_numpy(c).to(dev), torch.from_numpy(s).to(dev)) for c, s in sets]
    pin_sets = [(torch.from_numpy(c).pin_memory(), torch.from_numpy(s).pin_memory()) for c, s in sets]
    out_pin = torch.empty((B, SIZE, SIZE, 3), dtype=torch.uint8).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def step_resident(i):
        c, s = dev_sets[i % 2]
        out = eng.stylize(c, s, alpha=ALPHA, adain=args.adain)
        return eng.to_u8(out)

    def step_e2e(i):
        # the public API call a user makes: host (pinned) uint8 in, host (pinned) uint8 out, synchronous
        c, s = pin_sets[i % 2]
        return wct.predict_batch(c, s, alpha=ALPHA, adain=args.adain, out=out_pin)

    def timed(fn, steps, warmup):
        for i in range(warmup):
            fn(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = eng.launches
        e0.record()
        for i in range(steps):
            last = fn(i)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        launches = eng.launches - n0
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, launches, last

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_total, launches, last_out = timed(step_resident, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    ms_e2e, _, _ = timed(step_e2e, args.steps, max(3, args.warmup // 2))
    eng.check_device()

    pk = peaks()
    roofline, breakdown, hbm, by_level, cov_hbm = None, None, None, None, None
    if not args.no_roofline:
        # ---- roofline of the dominant kernel: per-call CUDA events on the launching stream.  Stream overlap is switched
        # off for these steps so that an event-bracketed duration is the kernel's own time, not its time while sharing
        # SMs with the Jacobi clusters of another stream.  The new configuration gets its own warm-up (new workspace
        # keys, scratch growth) before anything is recorded.
        PROF_WARM, PROF_STEPS = 2, 5
        eng.groups = 1
        eng.overlap_style = False
        for i in range(PROF_WARM):
            step_resident(i)
        torch.cuda.synchronize(dev)
        eng.profile = {}
        for i in range(PROF_STEPS):
            step_resident(i)
        torch.cuda.synchronize(dev)
        prof = {}
        for key, rec in eng.profile.items():
            ms = sum(a.elapsed_time(b) for a, b in rec["events"])
            prof[key] = dict(ms=ms / PROF_STEPS, flops=rec["flops"] / PROF_STEPS, bytes=rec["bytes"] / PROF_STEPS,
                             calls=len(rec["events"]) // PROF_STEPS)
        eng.profile = None
        eng.overlap_style = not args.no_overlap
        eng.groups = max(1, args.groups)

        def base(k):
            return k.split(":", 1)[1] if ":" in k else k
        conv = {k: v for k, v in prof.items() if base(k).startswith("conv3x3_")}
        conv_ms = sum(v["ms"] for v in conv.values())
        conv_fl = sum(v["flops"] for v in conv.values())
        step_prof_ms = sum(v["ms"] for v in prof.values())
        achieved_tf = conv_fl / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0
        traffic, traffic_of = None, ("not captured for this build: needs one `ncu --set full` launch of conv_tc2_kernel at the "
                                     "bench batch (profiles/r02_conv_traffic.json)")
        tp = os.path.join(ROOT, "profiles", "r02_conv_traffic.json")
        if os.path.exists(tp):
            tj = json.load(open(tp))
            traffic, traffic_of = tj.get("dram_bytes_per_launch"), tj.get("of")
        roofline = {"bound": "tensor", "achieved": achieved_tf, "peak": pk["tf"], "unit": "TFLOP/s",
                    "frac": achieved_tf / pk["tf"], "traffic": traffic, "traffic_of": traffic_of,
                    "kernel": "conv_tc2_kernel (tcgen05 kind::f16, split-fp16 x3: 3 MMAs per algorithmic MAC -> ceiling 1/3 of the "
                              "bf16 peak); flops counted = EXECUTED 2*taps*Cin*Cout per output pixel (taps = 4 in the UP2 convs)",
                    "tensor_pipe_frac": 3.0 * achieved_tf / pk["tf"],
                    "peak_source": pk["source"] + " of measured",
                    "share_of_step": conv_ms / step_prof_ms if step_prof_ms else None,
                    "launches_per_step": sum(v["calls"] for v in conv.values()),
                    "timed": "%d profiled steps after %d warm-up steps in the profiling configuration" % (PROF_STEPS, PROF_WARM)}
        # per-level conv tensor-pipe fraction (north_star): all conv launches of a level's encoder + decoder
        by_level = {}
        for k, v in conv.items():
            lv = level_of_key(k) or "?"
            d = by_level.setdefault(lv, dict(ms=0.0, flops=0.0))
            d["ms"] += v["ms"]
            d["flops"] += v["flops"]
        for lv, d in by_level.items():
            tf = d["flops"] / (d["ms"] * 1e-3) / 1e12 if d["ms"] > 0 else 0.0
            by_level[lv] = {"conv_ms": round(d["ms"], 3), "tflops": round(tf, 1), "tensor_pipe_frac": round(3.0 * tf / pk["tf"], 3)}
        merged = {}
        for k, v in prof.items():
            m = merged.setdefault(base(k), dict(ms=0.0, bytes=0.0))
            m["ms"] += v["ms"]
            m["bytes"] += v["bytes"]
        breakdown = {k: round(v["ms"], 3) for k, v in sorted(merged.items(), key=lambda kv: -kv[1]["ms"])[:16]}
        hbm = {}
        for k, v in merged.items():
            if (k.startswith("wct_") or k in ("upsample2", "maxpool2", "conv_tail", "conv_head")) and v["ms"] > 0:
                hbm[k] = round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1)

        # ---- covariance-only HBM rate (north_star): means + C x HW . HW x C covariance of one level's feature batch
        # through wctb200_covariance (no eigensolver in the bracket); bytes = the compulsory 4*C*HW per frame
        cov_hbm = {}
        nb = min(B, 16)
        for C, hw in ((64, 512), (128, 256), (256, 128), (512, 64)):
            feat = torch.rand((nb, hw, hw, C), dtype=torch.float32, device=dev)
            act = eng.act_from_f32(feat)
            mean = torch.empty((nb, C), dtype=torch.float32, device=dev)
            cov = torch.empty((nb, C, C), dtype=torch.float32, device=dev)
            st = torch.cuda.current_stream(dev).cuda_stream

            def run():
                _capi.check(eng.lib.wctb200_covariance(act.ptr, nb, hw, hw, C, 1e-8, mean.data_ptr(), cov.data_ptr(), st))
            for _ in range(3):
                run()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                run()
            e1.record()
            torch.cuda.synchronize(dev)
            ms = e0.elapsed_time(e1) / 5
            gbs = 4.0 * C * hw * hw * nb / (ms * 1e-3) / 1e9
            cov_hbm["C%d@%d" % (C, hw)] = {"ms": round(ms, 3), "gbs": round(gbs, 1), "frac": round(gbs / pk["hbm_gbs"], 3),
                                           "flops_tf": round(2.0 * C * C * hw * hw * nb / (ms * 1e-3) / 1e12, 1)}
            del feat, act
        eng.check_device()

    gather_ms = None
    sharded_ms = None
    if world > 1:
        out = step_resident(0)
        bufs = [torch.empty_like(out) for _ in range(world)] if not strong else None
        if strong:
            def sharded_step(i):
                c_all, s_one = sharded_inputs[i % 2]
                return parallel.stylize_sharded(lambda cc, ss: eng.to_u8(eng.stylize(cc, ss, alpha=ALPHA, adain=args.adain)),
                                                c_all, s_one)
            sharded_inputs = [(torch.from_numpy(frames(GB, 1000 + 1000 * j)).to(dev), torch.from_numpy(frames(1, 7 + 1000 * j)).to(dev))
                              for j in range(2)]
            sharded_ms, _, _ = timed(sharded_step, max(3, args.steps // 2), 3)     # sharded compute + NCCL gather, event timed, max over ranks
            sharded_ms /= max(3, args.steps // 2)
        else:
            for _ in range(3):
                dist.all_gather(bufs, out)          # warm NCCL (lazy channel setup)
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                dist.all_gather(bufs, out)          # NCCL over NVLink, off the hot path (SURVEY 8e)
            e1.record()
            torch.cuda.synchronize(dev)
            t = torch.tensor([e0.elapsed_time(e1) / 5], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            gather_ms = float(t.item())

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline and world == 1:          # reported at N = 1 only (the other ranks would just wait)
            host_cores = os.cpu_count() or 1
            threads = min(host_cores, 32)
            sec = cpu_frame_seconds(weights, 1, threads)
            cpu = {"value": 1.0 / sec, "unit": "frames/s", "cores": host_cores, "threads": threads, "kind": "port",
                   "sample": "1 full 512x512 5-level frame on the host (oracle port: torch-CPU convs + NumPy/LAPACK wct_tf; "
                             "TensorFlow not installable offline)"}
        total_frames = GB * args.steps
        value = total_frames / (ms_total * 1e-3)
        e2e = total_frames / (ms_e2e * 1e-3)
        line = {
            "metric": "512x512 5-level WCT stylised frames/sec", "value": value, "unit": "frames/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": make_config(world, B, args.adain, eng.groups, args.scaling, GB),
            "e2e": {"value": e2e, "unit": "frames/s", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": int((B + (1 if strong else B)) * SIZE * SIZE * 3), "d2h_bytes_per_step": int(B * SIZE * SIZE * 3)},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "algorithmic_tflops_whole_step": value * GFLOP_PER_FRAME / 1e3 if not (args.adain or strong) else None,
            "conv_by_level": by_level,
            "covariance_hbm": cov_hbm,
            "kernel_ms_per_step": breakdown,
            "hbm_gbs_by_stage": hbm,
            "gather_ms": gather_ms,
            "sharded_step_with_gather_ms": sharded_ms,
        }
        print(json.dumps(line))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last_out.cpu().numpy())
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
