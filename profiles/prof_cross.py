"""Extending a C5-sized matrix with new samples against recomputing the square (CUDA events, device-resident):
    python profiles/prof_cross.py [out.txt]            (default: profiles/cross_r4.txt)
C5 shape: synth.make_pairs(22 000, K = 64, seed = 5), reg 0.1, symmetric cosine cost.  The first 20 000 samples are
the old cohort; 200 and 2 000 of the rest join it.  For both solvers it times pairs.extend_pairs (the device part of
tl.wasserstein_d_extend: the RECT old x new block and the window of the new rows, EMD mirrored) and pairs.all_pairs
on the union (the full recompute), and checks that the extension's entries are byte-identical to the square's.
A second part answers whether the Sinkhorn warp form (algo 0 on a small cohort) and the DMMA panels (algo 3) give
the same bits for K <= 32 (pilot_sinkhorn_pairs picks between them from the cohort size for K <= 16)."""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from pilot_b200 import _lib, ops, pairs, synth

OUT = sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(os.path.abspath(__file__)), "cross_r4.txt")
S_OLD, K, REG = 20_000, 64, 0.1
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


def extension_vs_square():
    P, M = synth.make_pairs(S_OLD + 2_000, K, seed=5)
    Pd, Md = torch.from_numpy(P).cuda(), torch.from_numpy(M).cuda()
    emit(f"{'solver':>9} {'S_old':>6} {'S_new':>6} {'problems':>11} {'extend s':>9} {'problems':>11} {'square s':>9} "
         f"{'speed-up':>8}  identical")
    for regularized, name in (("unreg", "EMD"), ("reg", "Sinkhorn")):
        exact = regularized == "unreg"
        # warm-up: every kernel, every shape of the timed calls, on a small cohort
        pairs.extend_pairs(Pd[:300], Pd[300:340], Md, regularized, REG, symmetric=True)
        pairs.all_pairs(Pd[:340], Md, regularized, REG, symmetric=True)
        for S_new in (200, 2_000):
            S = S_OLD + S_new
            mode = _lib.PAIRS_UPPER if exact else _lib.PAIRS_FULL
            n_ext = S_OLD * S_new + (ops.n_pairs(S_new, mode) if exact else S_new * S)
            runs = [timed(lambda: pairs.extend_pairs(Pd[:S_OLD], Pd[S_OLD:S], Md, regularized, REG, symmetric=True))
                    for _ in range(3)]
            t_ext = [t for t, _ in runs]
            old_new, new_rows = runs[-1][1]
            del runs
            t_sq, sq = timed(lambda: pairs.all_pairs(Pd[:S], Md, regularized, REG, symmetric=True))
            same = bool(torch.equal(old_new, sq[:S_OLD, S_OLD:]) and torch.equal(new_rows, sq[S_OLD:]))
            ext_s = min(t_ext)
            emit(f"{name:>9} {S_OLD:6d} {S_new:6d} {n_ext:11d} {ext_s:9.3f} {ops.n_pairs(S, mode):11d} {t_sq:9.3f} "
                 f"{t_sq / ext_s:7.1f}x  {same}{'' if same else '  MISMATCH'}")
            emit(f"#   extend, 3 runs: {', '.join(f'{t:.3f}' for t in t_ext)} s")
            del old_new, new_rows, sq
            torch.cuda.empty_cache()


def warp_form_vs_panels():
    emit(f"{'K':>3} {'reg':>5} {'problems':>9} {'differing':>9} {'max rel diff':>12}")
    for K_ in list(range(2, 17)) + [24, 32]:
        for reg in (0.1, 0.01):
            S = 60  # S*S < 200 000: algo 0 takes the warp form
            P, M = synth.make_pairs(S, K_, seed=K_)
            Pd, Md = torch.from_numpy(P).cuda(), torch.from_numpy(M).cuda()
            rng = ops.make_range(S * S, _lib.PAIRS_FULL)
            a = ops.sinkhorn_pairs(Pd, Md, reg, rng, algo=0).cpu().numpy()
            b = ops.sinkhorn_pairs(Pd, Md, reg, rng, algo=3).cpu().numpy()
            ne = int((a.view(np.int64) != b.view(np.int64)).sum())
            rel = float(np.max(np.abs(a - b) / np.abs(b)))
            emit(f"{K_:3d} {reg:5.2f} {S * S:9d} {ne:9d} {rel:12.2e}")


def main():
    name, pl = card()
    emit(f"# {name}, power limit {pl}")
    emit(f"# extension of a {S_OLD}-sample matrix (K = {K}, reg {REG}) vs the square over the union; CUDA events "
         "around the device calls (inputs resident in HBM, result left on the device); 'identical': every entry of "
         "the extension equals the square's, byte for byte")
    extension_vs_square()
    emit()
    emit("# Sinkhorn warp form (algo 0) vs DMMA panels (algo 3), same problems, symmetric cost: entries whose bits differ")
    warp_form_vs_panels()
    with open(OUT, "w") as f:
        f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
