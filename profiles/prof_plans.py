"""Transport plans against the pair solvers on the same pairs (CUDA events, device-resident):
    python profiles/prof_plans.py [out.txt]            (default: profiles/plans_r5.txt)
For K = 16, 64, 128 and 256: synth.make_pairs(256, K, seed = K), symmetric cosine cost, and the list of all
256 x 256 = 65 536 ordered pairs in FULL order, so that the plan calls and the pair calls solve the same problems.
  EMD:      ops.emd_plans (zero-fill and scatter of every plan) vs ops.emd_pairs (costs only), FULL range;
  Sinkhorn: ops.sinkhorn_plans (reference-form kernel writing Gamma) vs ops.sinkhorn_pairs algo 1 (the same kernel
            without the plan) and algo 0 (the default solvers), reg 0.1.
Every call is timed 3 times after a warm-up; the table gives the fastest.  The plans (up to 34 GB at K = 256) stay
on the device.  The last columns check that the plan costs equal the pair costs (EMD, Sinkhorn algo 1: bit for bit;
algo 0: largest relative difference)."""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from pilot_b200 import _lib, ops, synth

OUT = sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(os.path.abspath(__file__)), "plans_r5.txt")
S, REG, REPS = 256, 0.1, 3
LINES = []


def emit(s=""):
    print(s, flush=True)
    LINES.append(s)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def timed(fn):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    r = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3, r


def best(fn):
    t_min, r = float("inf"), None
    for _ in range(REPS):
        r = None  # one call's plans at a time (34 GB at K = 256)
        t, r = timed(fn)
        t_min = min(t_min, t)
    return t_min, r


def main():
    name, pl = card()
    emit(f"# {name}, power limit {pl}")
    emit(f"# {S * S} problems per call (all ordered pairs of {S} samples), fastest of {REPS} calls after a warm-up")
    emit(f"{'K':>4} {'solver':>8} {'call':>16} {'s/call':>9} {'problems/s':>11} {'plans / pairs':>13}  costs")
    rng = ops.make_range(S * S, _lib.PAIRS_FULL)
    ii, jj = np.divmod(np.arange(S * S), S)
    for K in (16, 64, 128, 256):
        P, M = synth.make_pairs(S, K, seed=K)
        Pd, Md = torch.from_numpy(P).cuda(), torch.from_numpy(M).cuda()
        pa, pb = torch.from_numpy(ii).cuda(), torch.from_numpy(jj).cuda()
        # warm-up: every kernel of the timed calls, on a few problems
        ops.emd_plans(Pd, Md, pa[:64], pb[:64])
        ops.emd_pairs(Pd, Md, ops.make_range(64, _lib.PAIRS_FULL))
        ops.sinkhorn_plans(Pd, Md, REG, pa[:64], pb[:64])
        for algo in (0, 1):
            ops.sinkhorn_pairs(Pd, Md, REG, ops.make_range(64, _lib.PAIRS_FULL), algo=algo)

        t_plan, (g, c_plan) = best(lambda: ops.emd_plans(Pd, Md, pa, pb))
        del g
        t_pair, c_pair = best(lambda: ops.emd_pairs(Pd, Md, rng))
        same = torch.equal(c_plan.view(torch.int64), c_pair.view(torch.int64))
        emit(f"{K:4d} {'EMD':>8} {'emd_plans':>16} {t_plan:9.4f} {S * S / t_plan:11.4g} {t_pair / t_plan:13.3f}  "
             f"{'identical' if same else 'DIFFER'}")
        emit(f"{K:4d} {'EMD':>8} {'emd_pairs':>16} {t_pair:9.4f} {S * S / t_pair:11.4g}")
        torch.cuda.empty_cache()

        t_plan, (g, c_plan) = best(lambda: ops.sinkhorn_plans(Pd, Md, REG, pa, pb))
        del g
        torch.cuda.empty_cache()
        t_ref, c_ref = best(lambda: ops.sinkhorn_pairs(Pd, Md, REG, rng, algo=1))
        t_def, c_def = best(lambda: ops.sinkhorn_pairs(Pd, Md, REG, rng, algo=0))
        same = torch.equal(c_plan.view(torch.int64), c_ref.view(torch.int64))
        rel = float(((c_plan - c_def).abs() / c_def.abs()).max())
        emit(f"{K:4d} {'Sinkhorn':>8} {'sinkhorn_plans':>16} {t_plan:9.4f} {S * S / t_plan:11.4g} {'':>13}  "
             f"vs algo 1: {'identical' if same else 'DIFFER'}, vs algo 0: max rel {rel:.2e}")
        emit(f"{K:4d} {'Sinkhorn':>8} {'pairs algo 1':>16} {t_ref:9.4f} {S * S / t_ref:11.4g} {t_ref / t_plan:13.3f}")
        emit(f"{K:4d} {'Sinkhorn':>8} {'pairs algo 0':>16} {t_def:9.4f} {S * S / t_def:11.4g} {t_def / t_plan:13.3f}")
        del Pd, Md, pa, pb, c_plan, c_pair, c_ref, c_def
        torch.cuda.empty_cache()
    emit("# plans / pairs: the pair call's time over the plan call's (below 1: the plans cost that share extra)")
    with open(OUT, "w") as f:
        f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
