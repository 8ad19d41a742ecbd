"""Cost of spatial control (label masks, one style per region) on the flagship workload.

30 frames of 512x512, five levels relu5_1..relu1_1, wct_tf semantics, alpha 0.8, styles shared by the batch, two
sub-batch groups as in bench.py.  Variants, timed in alternation after a warm-up of each:
  (a) no mask, one style (the unmasked path);   (b) all-zero mask, R = 1;
  (c) left / right halves, R = 2;               (d) three blobs plus a keep region, R = 3.
Prints frames/s per variant (median of the rounds) and, from one CUDA-event-profiled step per variant, the time of each
level's transform call.  usage: python tools/regions_bench.py [rounds] [steps_per_round]"""
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from wct_tf_b200.engine import Engine  # noqa: E402
from wct_tf_b200.weights import make_synthetic_weights  # noqa: E402

ROUNDS = int(sys.argv[1]) if len(sys.argv) > 1 else 5
STEPS = int(sys.argv[2]) if len(sys.argv) > 2 else 3
B, S = 30, 512
T = ["relu5_1", "relu4_1", "relu3_1", "relu2_1", "relu1_1"]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=30).stdout.decode().strip()
    except Exception as e:  # the measurement stands without it, but say so
        q = "nvidia-smi unavailable (%s)" % e
    return "%s | %s" % (torch.cuda.get_device_name(0), q)


def masks():
    y, x = np.mgrid[0:S, 0:S]
    zero = np.zeros((S, S), np.uint8)
    halves = (x >= S // 2).astype(np.uint8)
    blobs = np.full((S, S), 3, np.uint8)                     # keep region: label 3 (>= R)
    for r, (cy, cx, rad) in enumerate([(150, 140, 120), (330, 380, 150), (420, 120, 90)]):
        blobs[(y - cy) ** 2 + (x - cx) ** 2 <= rad ** 2] = r
    return zero, halves, blobs


def main():
    rng = np.random.default_rng(0)
    eng = Engine(make_synthetic_weights(42), T, semantics="tf")
    eng.groups, eng.group_priorities = 2, True
    c = torch.from_numpy(rng.integers(0, 256, (B, S, S, 3), dtype=np.uint8)).cuda()
    styles = [torch.from_numpy(rng.integers(0, 256, (1, S, S, 3), dtype=np.uint8)).cuda() for _ in range(3)]
    zero, halves, blobs = (torch.from_numpy(m[None]).cuda() for m in masks())
    variants = {
        "a_no_mask": lambda: eng.stylize(c, styles[0], alpha=0.8),
        "b_zero_mask_R1": lambda: eng.stylize(c, styles[:1], alpha=0.8, labels=zero),
        "c_halves_R2": lambda: eng.stylize(c, styles[:2], alpha=0.8, labels=halves),
        "d_blobs_keep_R3": lambda: eng.stylize(c, styles[:3], alpha=0.8, labels=blobs),
    }
    print("card: %s" % card())
    print("workload: %d frames %dx%d, 5 levels, wct_tf, alpha 0.8, shared styles, 2 groups; %d rounds x %d steps per variant"
          % (B, S, S, ROUNDS, STEPS))
    for name, fn in variants.items():                        # warm-up: every shape and workspace
        for _ in range(2):
            eng.to_u8(fn())
    torch.cuda.synchronize()
    eng.check_device()
    fps = {k: [] for k in variants}
    for _ in range(ROUNDS):
        for name, fn in variants.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(STEPS):
                eng.to_u8(fn())
            torch.cuda.synchronize()
            fps[name].append(B * STEPS / (time.perf_counter() - t0))
    eng.check_device()
    base = np.median(fps["a_no_mask"])
    for name in variants:
        v = np.array(fps[name])
        print("%-16s %7.1f frames/s (median; min %.1f max %.1f)  %+.1f %% vs (a)"
              % (name, np.median(v), v.min(), v.max(), 100 * (np.median(v) / base - 1)))
    # per-level transform time: one profiled step per variant (CUDA events around each call, on its group stream)
    print("\nper-level transform calls, one profiled step (ms summed over the 2 groups; events bracket each call on its stream)")
    print("%-16s" % "variant" + "".join("%12s" % t for t in T))
    for name, fn in variants.items():
        eng.profile = {}
        eng.to_u8(fn())
        torch.cuda.synchronize()
        row = []
        for t in T:
            ms = sum(a.elapsed_time(b) for k, rec in eng.profile.items()
                     if k.startswith(t + ":") and ("wct_level" in k or "wct_regions" in k) for a, b in rec["events"])
            row.append(ms)
        eng.profile = None
        print("%-16s" % name + "".join("%12.2f" % v for v in row))
    print("card: %s" % card())


if __name__ == "__main__":
    main()
