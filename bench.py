#!/usr/bin/env python
"""bench.py -- pairwise OT distances / second on the PILOT patient-distance hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c5] [--rows R]
                    [--dump-outputs DIR]

Default workload = the configuration BASELINE.json's metric is quoted on, configs[4] ("c5", the scaling
sweep): 20 000 samples x 64 cell types, ALL pairs with BOTH solvers -- exact EMD (199 990 000 unordered
pairs, mirrored) and stabilised Sinkhorn reg 0.1 (400 000 000 ordered problems) -- i.e. the two dense
20 000 x 20 000 FP64 matrices the reference's wasserstein_d would fill
(/root/reference/pilotpy/tools/Trajectory.py:505-515).  One "step" = both matrices.  Prints ONE JSON line.

  value     -- matrix entries produced per second ("OT problems/s": EMD unordered pairs + Sinkhorn ordered
               problems) with the inputs resident in HBM, CUDA-event timed, max over ranks
  e2e       -- the same through the public API pilot_b200.tl.wasserstein_d with HOST containers in
               (dict of proportion vectors, cost ndarray) and out (ndarray + labelled DataFrame)
  roofline  -- the dominant kernel (the Sinkhorn DMMA panels) against the measured FP64 tensor-pipe peak
  cpu_baseline -- the oracle's C port of the two POT calls (or POT itself if importable) on the host cores
  checks    -- entries against the CPU oracle; N > 1: the all-gathered matrices against a single-rank solve

N > 1 (torchrun, one rank per GPU): STRONG scaling -- the same two matrices, pair space dealt in blocks over
the ranks, one NCCL all-gather per matrix inside the timed region, dense result on every rank.
--rows R restricts a step to the first R rows of both matrices (a band of the same workload) for quick runs.
--workload c1..c4 runs the cells path (histogram -> medians -> cdist -> pairs) of the other BASELINE configs.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "pairwise OT distances/sec (exact EMD & Sinkhorn) at 1/2/4/8 B200"
UNIT = "OT problems/s"
C5_S, C5_K, C5_REG = 20_000, 64, 0.1
C5_WORKLOAD = ("c5 (BASELINE configs[4], the scaling sweep): 20000 synthetic samples x 64 cell types, all pairs with "
               "both solvers: exact EMD (199990000 unordered pairs, mirrored) + stabilised Sinkhorn reg=0.1 "
               "(400000000 ordered problems) = the two dense 20000 x 20000 f64 matrices")


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                               f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": float(max(pw))}


def init_dist():
    """(world, rank, local_rank); brings NCCL up quietly when launched under torchrun."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        # NCCL announces its version on stdout when the first communicator comes up; the contract is
        # ONE JSON line on stdout, so stdout points at stderr until the communicator exists
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            warm = torch.zeros(1, device="cuda")
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    return world, rank, local_rank


# ---------------------------------------------------------------------------------------------
# the reference's CPU path for stage 3 (oracle port of the two POT calls, or POT itself)
# ---------------------------------------------------------------------------------------------
def cpu_pairs_sample(P, M, reg, n_cols, threads, rows_per_thread=1):
    """Every thread solves `rows_per_thread` row slices (row i x the first n_cols samples) of the ordered EMD
    matrix and of the ordered Sinkhorn matrix -- what the reference's double loop does per (i, j),
    Trajectory.py:508-515 -- with the C port of ot.emd2 / ot.sinkhorn2 (ctypes releases the GIL, so the
    threads run in parallel), or with POT itself when it is importable (then one thread: POT's Python entry
    points hold the GIL).  Returns per-solver wall times and the number of ordered problems of each."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import pilot_oracle as po
    ot = po.pot()
    Psub = np.ascontiguousarray(P[:n_cols])
    if ot is not None:
        rows = max(1, rows_per_thread)
        t0 = time.perf_counter()
        for i in range(rows):
            for j in range(n_cols):
                ot.emd2(Psub[i], Psub[j], M)
        t1 = time.perf_counter()
        for i in range(rows):
            for j in range(n_cols):
                ot.sinkhorn2(Psub[i], Psub[j], M, reg, method="sinkhorn_stabilized")
        t2 = time.perf_counter()
        return dict(t_emd=t1 - t0, t_sk=t2 - t1, n=rows * n_cols, cores=1, kind=f"pot {po.pot_version()}")
    rows = threads * rows_per_thread
    rows = min(rows, n_cols)
    with ThreadPoolExecutor(threads) as ex:
        t0 = time.perf_counter()
        list(ex.map(lambda i: po.emd_rows(Psub, M, i, i + 1), range(rows)))
        t1 = time.perf_counter()
        list(ex.map(lambda i: po.sinkhorn_rows(Psub, M, reg, i, i + 1), range(rows)))
        t2 = time.perf_counter()
    return dict(t_emd=t1 - t0, t_sk=t2 - t1, n=rows * n_cols, cores=threads, kind="port")


def c5_units(S, rows=None):
    """(EMD unordered pairs, Sinkhorn ordered problems) of the first `rows` rows of the two matrices."""
    rows = S if rows is None else rows
    return rows * (2 * S - rows - 1) // 2, rows * S


DUMP_BYTES = 60_000_000


def dump_outputs(out_dir, arrays, rows=None):
    """--dump-outputs: write each device array the timed path returned in its last step as out_dir/<name>.npy.
    Together they take at most DUMP_BYTES: an array larger than its share is written as a fixed, seeded sample of
    its rows (of its first `rows` rows, the band a --rows step computes), in increasing order, so that the files of
    two builds run with the same arguments hold the same entries."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, a in arrays.items():
        n = a.shape[0] if rows is None else rows
        row_bytes = a[0].numel() * a.element_size()
        if n * row_bytes > share:
            idx = np.sort(np.random.default_rng(0).choice(n, share // row_bytes, replace=False))
            a = a[torch.from_numpy(idx).to(a.device)]
        else:
            a = a[:n]
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())


def run_reference_c5(args):
    """Reference arm: the reference's CPU path for the same job on the host cores, every step a bounded sample
    (n ordered EMD problems + n ordered Sinkhorn problems = the fraction n / S^2 of the job: the reference
    solves all S^2 ordered pairs with either solver, it does not use the symmetry of the exact EMD)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from pilot_b200 import synth
    S, K, reg = C5_S, C5_K, C5_REG
    P, M = synth.make_pairs(S, K, seed=5)
    threads = os.cpu_count() or 1
    n_cols = 1000
    for _ in range(args.warmup):
        cpu_pairs_sample(P, M, reg, 100, threads)
    res = []
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res.append(cpu_pairs_sample(P, M, reg, n_cols, threads, rows_per_thread=4))
    wall = (time.perf_counter() - t0) / args.steps
    n_emd, n_sk = c5_units(S)
    n = res[0]["n"]
    units = (n_emd + n_sk) * (n / (S * S))          # job units covered by one step's sample
    value = units / wall
    t_e = float(np.mean([r["t_emd"] for r in res])) / n
    t_s = float(np.mean([r["t_sk"] for r in res])) / n
    sample = (f"per step {n} ordered exact-EMD problems + {n} ordered Sinkhorn problems (rows x the first {n_cols} "
              f"samples; = {n / (S * S):.3e} of the job's S^2 ordered pairs per solver) on {res[0]['cores']} host "
              f"thread(s); all-core rates {1 / t_e:.0f} emd2/s, {1 / t_s:.0f} sinkhorn2/s; the reference itself runs "
              f"this loop on ONE core (Python double loop, POT numThreads=1)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": wall * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": C5_WORKLOAD},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": res[0]["cores"], "kind": res[0]["kind"],
                             "sample": sample, "host_cpus": os.cpu_count()},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# B200 arm, default workload: C5
# ---------------------------------------------------------------------------------------------
def run_c5(args):
    import torch
    import torch.distributed as dist
    from oracle import pilot_oracle as po          # checker only: spot checks and the cpu_baseline leg
    from pilot_b200 import _lib, ops, pairs, synth, tl

    world, rank, local_rank = init_dist()
    S, K, reg = C5_S, C5_K, C5_REG
    rows = S if args.rows is None else max(2, min(S, args.rows))
    P, M = synth.make_pairs(S, K, seed=5)
    Pd, Md = torch.from_numpy(P).cuda(), torch.from_numpy(M).cuda()
    n_emd, n_sk = c5_units(S, rows)
    dense_e = torch.empty((S, S), dtype=torch.float64, device="cuda")
    dense_s = torch.empty((S, S), dtype=torch.float64, device="cuda")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(marks_e=None, marks_s=None, want_info=False):
        """One pass of the hot path: both matrices (their first `rows` rows), dense on every rank."""
        pairs._solve_window(Pd, Md, True, reg, _lib.PAIRS_UPPER, 0, n_emd, world, rank, None, 0, "f64", dense_e,
                            marks=marks_e)
        return pairs._solve_window(Pd, Md, False, reg, _lib.PAIRS_FULL, 0, n_sk, world, rank, None, 0, "f64",
                                   dense_s, want_info=want_info, marks=marks_s)

    # ---------------- warm-up (the first one also yields the iteration counts for the roofline) -------------
    flops_rank = mean_iters = None
    for w in range(max(1, args.warmup)):
        info = step(want_info=(w == 0))
        if w == 0:
            it = info[0]
            flops_rank = float(it.sum(dtype=torch.int64).item()) * 4.0 * K * K
            mean_iters = float(it.float().mean().item())
            del info, it
            torch.cuda.empty_cache()
    barrier()

    # ---------------- timed region: exactly args.steps steps ----------------
    launches0 = _lib.launch_count()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    marks_e, marks_s = [], []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step(marks_e, marks_s)
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    launches = _lib.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"emd": dense_e, "sinkhorn": dense_s}, rows)
    t = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = t.item() / args.steps
    value = (n_emd + n_sk) / (ms_step * 1e-3)

    def phase_ms(marks):
        out = {}
        per = 4  # start, solve, gather, unpack
        for i in range(0, len(marks), per):
            for (n0, ev0), (n1, ev1) in zip(marks[i:i + per - 1], marks[i + 1:i + per]):
                out.setdefault(n1, []).append(ev0.elapsed_time(ev1))
        return {k: float(np.mean(v)) for k, v in out.items()}

    ph_e, ph_s = phase_ms(marks_e), phase_ms(marks_s)

    # ---------------- checks (untimed) ----------------
    checks = {}
    sub = torch.arange(0, rows, max(1, rows // 48), device="cuda")[:48]
    Psub = Pd[sub].contiguous()
    one_e = pairs.all_pairs(Psub, Md, "unreg", single_rank=True)
    one_s = pairs.all_pairs(Psub, Md, "reg", reg, single_rank=True)
    got_e = dense_e[sub][:, sub]
    got_s = dense_s[sub][:, sub]
    emd_identical = bool(torch.equal(one_e, got_e))
    sk_identical = bool(torch.equal(one_s, got_s))
    sk_rel = float(((one_s - got_s).abs() / one_s.abs()).max().item())
    flags = torch.tensor([0.0 if emd_identical else 1.0, sk_rel, 0.0 if sk_identical else 1.0], dtype=torch.float64,
                         device="cuda")
    if world > 1:
        dist.all_reduce(flags, op=dist.ReduceOp.MAX)
    checks["partition_vs_single_rank"] = {
        "what": f"{sub.numel()} x {sub.numel()} sub-matrix of the {world}-rank all-gathered result vs the same "
                "sub-cohort solved on one rank, on every rank",
        "emd_bit_identical": bool(flags[0].item() == 0.0), "sinkhorn_bit_identical": bool(flags[2].item() == 0.0),
        "sinkhorn_max_rel_diff": float(flags[1].item())}

    if rank == 0:
        rs = np.random.default_rng(0)
        n_chk = 200
        ii, jj = rs.integers(0, rows, n_chk), rs.integers(0, S, n_chk)
        iu, ju = np.minimum(ii, jj), np.maximum(ii, jj)
        keep = iu != ju
        iu, ju = iu[keep], ju[keep]
        got_e = dense_e[torch.from_numpy(iu).cuda(), torch.from_numpy(ju).cuda()].cpu().numpy()
        got_et = dense_e[torch.from_numpy(ju).cuda(), torch.from_numpy(iu).cuda()].cpu().numpy()
        got_s = dense_s[torch.from_numpy(ii).cuda(), torch.from_numpy(jj).cuda()].cpu().numpy()
        want_e = np.array([po.emd2(P[i], P[j], M) for i, j in zip(iu, ju)])
        want_s = np.array([po.sinkhorn2(P[i], P[j], M, reg) for i, j in zip(ii, jj)])
        rel = lambda a, b: float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))
        checks["vs_cpu_oracle"] = {"sampled_entries": int(n_chk), "emd_max_rel_err": rel(got_e, want_e),
                                   "sinkhorn_max_rel_err": rel(got_s, want_s),
                                   "emd_mirror_identical": bool(np.array_equal(got_e, got_et)),
                                   "emd_diag_abs_max": float(dense_e.diagonal()[:rows].abs().max().item()),
                                   "tolerance": "1e-9 relative (BASELINE.json, FP64 mode)"}
        # EMD <= Sinkhorn transport cost on the sampled upper entries
        got_su = dense_s[torch.from_numpy(iu).cuda(), torch.from_numpy(ju).cuda()].cpu().numpy()
        checks["emd_le_sinkhorn"] = bool((got_e <= got_su * (1 + 1e-9)).all())

    # ---------------- end to end through the public API (host containers in and out) ----------------
    ids = [f"s{i:05d}" for i in range(S)]
    clu = {ids[i]: P[i] for i in range(S)}

    def api_step():
        E, Edf = tl.wasserstein_d(clu, M, regularized="unreg")
        del Edf
        R, Rdf = tl.wasserstein_d(clu, M, regularized="reg", reg=reg)
        return float(E[0, 1]) + float(R[0, 1])

    e2e_warm, e2e_steps = 1, 1 if rows == S else max(1, min(args.steps, 2))  # a full-size call takes ~22 s on one GPU
    for _ in range(e2e_warm):
        api_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        api_step()
    torch.cuda.synchronize()
    t_e2e = (time.perf_counter() - t0) / e2e_steps
    te = torch.tensor([t_e2e], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    t_e2e = te.item()
    fe, fs = c5_units(S)
    h2d = 2 * (P.nbytes + M.nbytes)
    d2h = 2 * 2 * S * S * 8  # per solver: the ndarray and the transposed copy the labelled DataFrame owns

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {"fp64_fma_tflops": ops.pipe_peak(0), "fp32_fma_tflops": ops.pipe_peak(1),
             "fp64_dmma_tflops": ops.pipe_peak(2)}
    sk_ms = ph_s["solve"]
    ach = flops_rank / (sk_ms * 1e-3) / 1e12
    roofline = {"kernel": "sinkhorn_batched_kernel (+ setup, tail and reference-form launches of pilot_sinkhorn_pairs)",
                "bound": "tensor", "pipe": "FP64 mma.sync (DMMA m8n8k4); tcgen05 has no FP64 kind",
                "achieved": ach, "peak": peaks["fp64_dmma_tflops"], "unit": "TFLOP/s",
                "frac": ach / peaks["fp64_dmma_tflops"], "traffic": None,
                "peak_source": "FP64 DMMA peak measured in this run by pilot_pipe_peak (MEASURED_PEAKS.json holds "
                               "only the HBM and bf16 peaks); nominal 148 SM x 64 FMA/clk x 2 x 1.965 GHz = 37.2",
                "algorithmic_flops_per_launch": flops_rank, "flops_per_problem": "iters x 4 K^2 (SURVEY 8d)",
                "mean_iters": mean_iters, "ms_per_launch": sk_ms, "timed": "CUDA events around the call, every timed step",
                "share_of_step": sk_ms / ms_step}
    # exact EMD: SURVEY 8d convention -- FP64 operations of the REFERENCE algorithm (3A + 2U + 2C of the oracle's
    # block-search network simplex on the same kind of input) per problem against the FP64 FMA peak
    _, _, st = po.emd_rows(P[:16], M, 0, 16, return_stats=True)
    ops_pp = (3 * st["arcs_priced"] + 2 * st["pot_updates"] + 2 * st["cycle_steps"]) / (16 * 16)
    emd_ms = ph_e["solve"]
    n_emd_rank = pairs.range_count(n_emd, pairs.choose_block(n_emd, world), world, 0)
    n_sk_rank = pairs.range_count(n_sk, pairs.choose_block(n_sk, world), world, 0)
    kernels = {
        "emd_pairs_kernel": {"problems_per_launch": n_emd_rank, "ms_per_launch": emd_ms,
                             "pairs_per_s_per_gpu": n_emd_rank / (emd_ms * 1e-3),
                             "reference_algorithm_fp64_ops_per_problem": ops_pp,
                             "frac_of_fp64_fma_peak": ops_pp * n_emd_rank / (emd_ms * 1e-3) / 1e12 / peaks["fp64_fma_tflops"],
                             "note": "issue-bound integer/shared-memory work (profiles/emd_r2.txt); the FP64 figure "
                                     "is SURVEY 8d's convention", "share_of_step": emd_ms / ms_step},
        "sinkhorn": {"problems_per_launch": n_sk_rank, "ms_per_launch": sk_ms,
                     "problems_per_s_per_gpu": n_sk_rank / (sk_ms * 1e-3)},
        "gather_ms": {"emd": ph_e["gather"], "sinkhorn": ph_s["gather"]},
        "unpack_ms": {"emd": ph_e["unpack"], "sinkhorn": ph_s["unpack"]}}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(1, args.warmup), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": C5_WORKLOAD,
                       "rows_per_step": rows, "units_per_step": {"emd_pairs": n_emd, "sinkhorn_problems": n_sk},
                       "l2": "inputs are 10 MB of proportions + a 32 KB cost matrix (L2/shared-memory resident by "
                             "design); every step streams 1.6 + 3.2 GB of packed results and 6.4 GB of dense output "
                             "through HBM, far more than the 126 MB L2; no flush",
                       "multi_gpu": "strong scaling: pair space dealt in 4096-problem blocks round-robin over the "
                                    "ranks, one NCCL all-gather per matrix, dense result on every rank"},
            "clocks": clocks,
            "e2e": {"value": (fe + fs) / t_e2e, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": t_e2e * 1e3, "steps": e2e_steps,
                    "api": "pilot_b200.tl.wasserstein_d(proportions dict, cost ndarray) x2 (exact, then Sinkhorn): "
                           "host containers in, ndarray + labelled DataFrame out, full 20000 x 20000 matrices; "
                           "rows cross PCIe band by band while later bands are solved"},
            "gpu_launches": int(launches),
            "roofline": roofline, "kernels": kernels, "pipe_peaks": peaks, "checks": checks}
    if world == 1:
        threads = os.cpu_count() or 1
        cb = cpu_pairs_sample(P, M, reg, 1000, threads, rows_per_thread=20)  # ~10 s of wall time
        n = cb["n"]
        t_e, t_s = cb["t_emd"] / n, cb["t_sk"] / n
        line["cpu_baseline"] = {
            "value": (fe + fs) / (S * S * (t_e + t_s)), "unit": UNIT, "cores": cb["cores"], "kind": cb["kind"],
            "host_cpus": os.cpu_count(),
            "sample": f"{n} ordered exact-EMD problems ({cb['t_emd']:.1f}s) + {n} ordered Sinkhorn problems "
                      f"({cb['t_sk']:.1f}s), rows x the first 1000 samples, on {cb['cores']} thread(s): "
                      f"{1 / t_e:.0f} emd2/s, {1 / t_s:.0f} sinkhorn2/s; the job needs S^2 = 4e8 of each on the CPU "
                      "(the reference does not use the EMD's symmetry); the reference itself uses ONE core"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------
# cells path: BASELINE configs[0..3]
# ---------------------------------------------------------------------------------------------
REG = {"c1": None, "c2": 0.1, "c3": 0.1, "c4": 0.01}
CELLS_CONFIG_ID = {"c1": 0, "c2": 1, "c3": 2, "c4": 3}


def workload_shape(name: str, n_gpus: int):
    from pilot_b200 import synth
    n, d, k, s, seed = synth.CONFIGS[name]
    return n, d, k, s, seed


def make_workload(name: str, n_gpus: int):
    from pilot_b200 import synth
    n, d, k, s, seed = workload_shape(name, n_gpus)
    X, obs = synth.make_cells(n, d, k, s, seed, labels="categorical")
    return X, obs, (n, d, k, s)


def cells_workload_string(name, n, d, k, s, reg):
    return (f"{name} (BASELINE configs[{CELLS_CONFIG_ID[name]}]): {n} cells x {d}-dim float32 embedding, {k} cell types, "
            f"{s} samples, cosine cost, " + (f"stabilised Sinkhorn reg={reg}, all {s * s} ordered pairs"
                                            if reg is not None else f"exact EMD, {s * (s - 1) // 2} unordered pairs"))


def cpu_reference_step(X, obs, reg, rows):
    """One bounded pass of the reference's CPU path on the cells workloads (oracle port; the reference's own
    Cluster_Representations / cost_matrix are exec'd verbatim when /root/reference is mounted): stages 1-2 in
    full, stage 3 on the first `rows` rows of the ordered pair matrix (C port of the POT call, one core)."""
    import pandas as pd
    from oracle import pilot_oracle as po
    from oracle import ref_exec
    annot = obs[["cell_types", "sampleID", "status"]].copy()
    annot.columns = ["cell_type", "sampleID", "status"]
    data = pd.DataFrame(X)
    t0 = time.perf_counter()
    if ref_exec.available():
        ref = ref_exec.load()
        props = ref.Cluster_Representations(annot)
        t1 = time.perf_counter()
        dis, _ = ref.cost_matrix(annot, data, "cosine")
    else:
        props = po.cluster_representations(annot)
        t1 = time.perf_counter()
        dis, _ = po.cost_matrix(annot, data, "cosine")
    t2 = time.perf_counter()
    ids = list(props.keys())
    S = len(ids)
    M = dis / dis.max()
    Pm = np.stack([props[i] for i in ids])
    rows = min(rows, S)
    if reg is None:
        po.emd_rows(Pm, M, 0, rows)
    else:
        po.sinkhorn_rows(Pm, M, reg, 0, rows)
    t3 = time.perf_counter()
    return dict(t_props=t1 - t0, t_cost=t2 - t1, t_pairs_sample=t3 - t2, rows=rows, S=S,
                kind="reference+port" if ref_exec.available() else "port")


def run_reference_cells(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    X, obs, (n, d, k, s) = make_workload(args.workload, 1)
    reg = REG[args.workload]
    rows = max(1, min(s, 2000 // s + 1))
    with tempfile.TemporaryDirectory() as tmp:
        cwd = os.getcwd(); os.chdir(tmp)
        try:
            for _ in range(args.warmup):
                cpu_reference_step(X, obs, reg, 1)
            t0 = time.perf_counter()
            res = [cpu_reference_step(X, obs, reg, rows) for _ in range(args.steps)]
            wall = (time.perf_counter() - t0) / args.steps
        finally:
            os.chdir(cwd)
    units_job = s * s if reg is not None else s * (s - 1) // 2
    # job time on the CPU: stages 1-2 once + all S rows of stage 3
    t12 = float(np.mean([r["t_props"] + r["t_cost"] for r in res]))
    t3 = float(np.mean([r["t_pairs_sample"] for r in res])) * s / rows
    frac = wall / (t12 + t3)                        # the share of the job one step's sample covers
    value = units_job * frac / wall
    sample = (f"stages 1-2 in full ({n} cells, {t12:.2f}s) + stage 3 on the first {rows} of {s} rows (C port of the POT "
              f"call, 1 core); one step covers {frac:.3f} of the job")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": wall * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": cells_workload_string(args.workload, n, d, k, s, reg)},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": res[0]["kind"], "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


class DeviceStep:
    """The cells path with device-resident inputs, stage by stage (what tl.wasserstein_distance runs)."""

    def __init__(self, X, obs, reg):
        import torch
        from pilot_b200 import tl
        self.torch = torch
        self.reg = reg
        annot = obs[["cell_types", "sampleID", "status"]].copy()
        annot.columns = ["cell_type", "sampleID", "status"]
        self.lab = tl._Labels(annot, "cell_type", "sampleID")      # codes on device + perms
        self.X = tl._embedding_ready(tl._embedding_to_device(X))

    def run(self, timers=None):
        from pilot_b200 import ops, pairs
        torch = self.torch
        lab = self.lab

        def mark(name):
            if timers is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                timers.append((name, ev))

        mark("start")
        counts_raw, first_ct, first_smp = ops.hist(lab.ct_dev, lab.sm_dev, lab.K_raw, lab.S_raw)
        mark("hist")
        props, counts = ops.props_finalize(counts_raw, lab.perm_k_dev, lab.perm_s_dev, lab.n, 0.2, True)
        mark("props")
        _, cent64_raw = ops.centroid_median(self.X, lab.ct_dev, lab.K_raw)
        mark("median")
        cent64 = cent64_raw.index_select(0, lab.perm_k_dev.long()).contiguous()
        cost, cost_norm, _ = ops.cdist(cent64, "cosine")
        mark("cdist")
        dense = pairs.all_pairs(props, cost_norm, "unreg" if self.reg is None else "reg",
                                self.reg if self.reg is not None else 0.1, symmetric=True)
        mark("pairs")
        return dense, props, cost


def run_cells(args):
    import torch
    import torch.distributed as dist
    from pilot_b200 import _lib, ops, synth, tl

    world, rank, local_rank = init_dist()
    X, obs, (n, d, k, s) = make_workload(args.workload, world)
    reg = REG[args.workload]
    hbm_peak, peak_kind = load_peaks()
    tmp = tempfile.mkdtemp()
    os.chdir(tmp)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    step = DeviceStep(X, obs, reg)
    for _ in range(max(1, args.warmup)):
        step.run()
    barrier()
    launches0 = _lib.launch_count()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        dense, props, cost = step.run()
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    launches = _lib.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"pairs": dense, "proportions": props, "cost": cost})
    t = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = t.item() / args.steps
    units = s * s if reg is not None else s * (s - 1) // 2
    value = units / (ms_step * 1e-3)

    stage_ms = {}
    for _ in range(3):
        timers = []
        step.run(timers)
        torch.cuda.synchronize()
        for (n0, ev0), (n1, ev1) in zip(timers[:-1], timers[1:]):
            stage_ms.setdefault(n1, []).append(ev0.elapsed_time(ev1))
    stage_ms = {kname: float(np.mean(v)) for kname, v in stage_ms.items()}
    elt = X.dtype.itemsize
    alg_bytes = {"hist": n * 8 + s * k * 8, "median": n * d * elt + n * 4 + k * d * elt}
    dominant = max(stage_ms, key=stage_ms.get)
    peaks = {"fp64_fma_tflops": ops.pipe_peak(0), "fp32_fma_tflops": ops.pipe_peak(1),
             "fp64_dmma_tflops": ops.pipe_peak(2)}
    if dominant in alg_bytes:
        ach = alg_bytes[dominant] / (stage_ms[dominant] * 1e-3) / 1e9
        roofline = {"kernel": dominant, "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                    "frac": ach / hbm_peak, "traffic": None,
                    "peak_source": peak_kind + " (MEASURED_PEAKS.json hbm_gbs)",
                    "algorithmic_bytes": alg_bytes[dominant], "ms": stage_ms[dominant]}
    elif reg is not None:
        from pilot_b200 import pairs as _pairs
        total = s * s
        rng = _lib.PairRange(total=total, block=_pairs.choose_block(total, world), nranks=world, rank=rank,
                             mode=_lib.PAIRS_FULL, reserved=0)
        _, it, _, _ = ops.sinkhorn_pairs(props, cost / cost.max(), reg, rng, want_info=True)
        flops = float(it.sum().item()) * 4.0 * k * k
        ach = flops / (stage_ms[dominant] * 1e-3) / 1e12
        warp = k <= 32
        # K <= 32: one warp per problem, scalar DFMA chains (FP64 FMA pipe); above: DMMA panels (FP64 tensor pipe)
        peak = peaks["fp64_fma_tflops"] if warp else peaks["fp64_dmma_tflops"]
        roofline = {"kernel": ("sinkhorn_warp_kernel" if warp else "sinkhorn_batched_kernel") +
                              " (all-pairs stage incl. setup/unpack)",
                    "bound": "fp64" if warp else "tensor", "pipe": "FP64 FMA (DFMA)" if warp else "FP64 mma.sync (DMMA)",
                    "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": None,
                    "peak_source": "measured in this run by pilot_pipe_peak",
                    "algorithmic_flops": flops, "mean_iters": float(it.float().mean().item()),
                    "max_iters": int(it.max().item()), "ms": stage_ms[dominant]}
    else:
        roofline = {"kernel": "emd_pairs_kernel", "bound": "fp64", "achieved": None, "peak": peaks["fp64_fma_tflops"],
                    "unit": "TFLOP/s", "frac": None, "traffic": None, "ms": stage_ms[dominant],
                    "note": "issue-bound integer/shared-memory kernel; see --workload c5 for its throughput"}

    # ---------------- end to end through the public API ----------------
    pinned = torch.empty(X.shape, dtype=torch.float32 if X.dtype == np.float32 else torch.float64, pin_memory=True)
    Xp = pinned.numpy()
    Xp[...] = X
    kw = dict(emb_matrix="X_PCA", clusters_col="cell_types", sample_col="sampleID", status="status",
              regularized="unreg" if reg is None else "reg", reg=reg if reg is not None else 0.1)

    def api_step(emb, o):
        adata = synth.FakeAnnData(o, obsm={"X_PCA": emb})
        tl.wasserstein_distance(adata, **kw)
        return adata

    def time_api(emb, o, steps):
        for _ in range(2):
            api_step(emb, o)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            api_step(emb, o)
        torch.cuda.synchronize()
        te = torch.tensor([(time.perf_counter() - t0) / steps], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        return te.item()

    e2e_steps = max(1, min(args.steps, 10))
    t_e2e = time_api(Xp, obs, e2e_steps)
    # what a user has by default: a pageable ndarray and str label columns (Trajectory.py:255-263)
    obs_str = obs.copy()
    for c in obs_str.columns:
        obs_str[c] = obs_str[c].astype(str).astype(object)
    X_pageable = np.array(X, copy=True)
    tl._factor_cache.clear()
    torch.cuda.synchronize()
    t0c = time.perf_counter()
    api_step(X_pageable, obs_str)            # first call on these label objects: pays the string factorisation
    torch.cuda.synchronize()
    t_e2e_default_first = time.perf_counter() - t0c
    t_e2e_default = time_api(X_pageable, obs_str, max(1, min(args.steps, 3)))
    code_bytes = sum(1 if c < 128 else (2 if c < 32768 else 4) for c in (k, s))
    h2d = n * code_bytes + X.nbytes + (k + s) * 4
    d2h = s * s * 8 + s * k * 8 + k * k * 8 + (k + s) * 8

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(1, args.warmup), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": cells_workload_string(args.workload, n, d, k, s, reg),
                       "l2": "inputs (embedding %.0f MB) larger than the 126 MB L2; no flush" % (X.nbytes / 1e6),
                       "multi_gpu": "pair space block-partitioned over ranks, one NCCL all-gather per step; "
                                    "stages 1-2 replicated"},
            "clocks": clocks,
            "e2e": {"value": units / t_e2e, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": t_e2e * 1e3,
                    "api": "pilot_b200.tl.wasserstein_distance(adata) with categorical obs and a pinned host embedding",
                    "default_inputs": {"value": units / t_e2e_default, "ms_per_step": t_e2e_default * 1e3,
                                       "first_call_ms": t_e2e_default_first * 1e3,
                                       "what": "pageable ndarray embedding and str label columns, every cell its own "
                                               "str object (the reference's default user input, Trajectory.py:255-263); "
                                               "ms_per_step: repeated calls on the same label objects (validated "
                                               "factorisation cache), first_call_ms: the call that factorises them"}},
            "gpu_launches": int(launches), "stage_ms": stage_ms, "roofline": roofline, "pipe_peaks": peaks,
            # the two HBM-bound stages against the measured copy bandwidth (whole stage, all its kernels)
            "stage_hbm": {kn: {"algorithmic_bytes": int(alg_bytes[kn]),
                               "achieved_gbs": alg_bytes[kn] / (stage_ms[kn] * 1e-3) / 1e9,
                               "frac": alg_bytes[kn] / (stage_ms[kn] * 1e-3) / 1e9 / hbm_peak}
                          for kn in ("hist", "median") if kn in stage_ms}}
    if world == 1:
        rows = max(1, min(s, 2000 // s + 1))
        cb = cpu_reference_step(X, obs, reg, rows)
        full = cb["t_props"] + cb["t_cost"] + cb["t_pairs_sample"] * cb["S"] / cb["rows"]
        line["cpu_baseline"] = {
            "value": units / full, "unit": UNIT, "cores": 1, "kind": cb["kind"],
            "sample": f"stages 1-2 in full ({cb['t_props']:.2f}s + {cb['t_cost']:.2f}s); stage 3 on the first "
                      f"{cb['rows']} of {cb['S']} rows ({cb['t_pairs_sample']:.2f}s, C port of the POT call), "
                      f"extrapolated x{cb['S']}/{cb['rows']}"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c5", choices=["c1", "c2", "c3", "c4", "c5"])
    ap.add_argument("--rows", type=int, default=None,
                    help="c5 only: restrict a step to the first R rows of both matrices (default: all 20000)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the matrices the last timed step computed to DIR/<name>.npy (float64, at most 60 MB "
                         "in all: a larger matrix as a fixed, seeded sample of its rows)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the B200 path computes; it does not apply to --impl reference")
    if args.impl == "reference":
        (run_reference_c5 if args.workload == "c5" else run_reference_cells)(args)
    elif args.workload == "c5":
        run_c5(args)
    else:
        run_cells(args)


if __name__ == "__main__":
    main()
