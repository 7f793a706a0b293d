"""Throughput of all-pairs Sinkhorn for 64..256 cell types (CUDA events after warm-up):
    python profiles/prof_sinkhorn_wide.py [seconds]
For each K, times ops.sinkhorn_pairs on synth.make_pairs problems with algo = 0 (K <= 64: DMMA panels; 65..256:
the cluster-split panels of sinkhorn_wide.cu) and algo = 1 (reference form), for a window of at least `seconds`
(default 1).  Reports problems/s, TFLOP/s as sum(iters * 4 K^2) / time and its fraction of the DMMA pipe peak
measured in the same run (ops.pipe_peak(2)), and checks per K that algo 0 and 1 agree within 1e-9 with identical
iteration and absorption counts on every timed problem."""
import math
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from pilot_b200 import _lib, ops, synth

WINDOW = float(sys.argv[1]) if len(sys.argv) > 1 else 1.0
SHAPES = [(64, 0.1), (65, 0.1), (96, 0.1), (100, 0.1), (128, 0.1), (150, 0.1), (192, 0.1), (200, 0.1),
          (256, 0.1), (128, 0.01)]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3


def measure(Pd, Md, K, reg, algo):
    """(seconds per call, problems per call, costs, iterations, absorptions) over a window of >= WINDOW seconds"""
    S = Pd.shape[0]
    rng = ops.make_range(S * S, _lib.PAIRS_FULL)
    out = torch.empty((S * S,), dtype=torch.float64, device="cuda")
    res, iters, absn, _ = ops.sinkhorn_pairs(Pd, Md, reg, rng, algo=algo, want_info=True)  # warm-up, and the work
    t1 = timed(lambda: ops.sinkhorn_pairs(Pd, Md, reg, rng, algo=algo, out=out))
    reps = max(1, math.ceil(WINDOW / max(t1, 1e-6)))
    t = timed(lambda: [ops.sinkhorn_pairs(Pd, Md, reg, rng, algo=algo, out=out) for _ in range(reps)])
    return t / reps, S * S, res.cpu().numpy(), iters.cpu().numpy(), absn.cpu().numpy()


def main():
    name, pl = card()
    peak = ops.pipe_peak(2)
    print(f"# {name}, power limit {pl}; DMMA (mma.sync m8n8k4 f64) pipe peak measured now: {peak:.1f} TFLOP/s")
    print(f"# window >= {WINDOW:.1f} s per row; TFLOP/s = sum(iters * 4 K^2) / time")
    print(f"{'K':>4} {'reg':>5} {'algo':>4} {'S':>5} {'problems/s':>12} {'TFLOP/s':>8} {'of DMMA':>8} {'ms/call':>9}")
    for K, reg in SHAPES:
        # 65 536 problems per call (many waves of panels at every K: most problems go to refilled slots),
        # repeated to fill the window; the parity check below is on these same batches
        S = 256
        P, M = synth.make_pairs(S, K, seed=5)
        Pd, Md = torch.from_numpy(P).cuda(), torch.from_numpy(M).cuda()
        runs = {}
        for algo in (0, 1):
            t, n, res, iters, absn = measure(Pd, Md, K, reg, algo)
            runs[algo] = (res, iters, absn)
            tf = 4.0 * K * K * float(iters.sum()) / t / 1e12
            print(f"{K:4d} {reg:5.2f} {algo:4d} {S:5d} {n / t:12.4g} {tf:8.3f} {tf / peak:8.3f} {t * 1e3:9.3f}")
            sys.stdout.flush()
        (a, ia, aa), (b, ib, ab) = runs[0], runs[1]
        rel = float(np.max(np.abs(a - b) / np.abs(b)))
        same = bool(np.array_equal(ia, ib) and np.array_equal(aa, ab))
        ok = rel <= 1e-9 and same
        print(f"# K={K} reg={reg}, all {S * S} problems: algo 0 vs 1 max rel diff {rel:.2e}, identical iteration and "
              f"absorption counts: {same}{'' if ok else '  MISMATCH'}")


if __name__ == "__main__":
    main()
