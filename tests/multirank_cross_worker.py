"""Worker of tests/test_gpu_multirank_cross.py (launched under torchrun, one rank per GPU, NCCL): blocks between two
sample sets and extended matrices assembled from the ranks' shares with the NCCL all-gather must equal a single-rank
solve BIT FOR BIT, for both solvers and for a symmetric and an asymmetric cost -- pairs.cross_pairs,
pairs.cross_pairs_host, pairs.extend_pairs and the public tl.wasserstein_d_cross / tl.wasserstein_d_extend."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pilot_b200 import pairs, synth, tl  # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
    for S_old, S_new, K in ((211, 37, 64), (150, 1, 30), (90, 41, 100)):
        S = S_old + S_new
        P, M = synth.make_pairs(S, K, seed=80 + K)
        A = M + 0.3 * np.triu(np.random.default_rng(K).random(M.shape), 1)
        for cost in (M, A / A.max()):
            Pd, Cd = torch.from_numpy(P).cuda(), torch.from_numpy(cost).cuda()
            old = {f"s{i}": P[i] for i in range(S_old)}
            new = {f"s{i}": P[i] for i in range(S_old, S)}
            for regularized in ("unreg", "reg"):
                single = pairs.all_pairs(Pd, Cd, regularized, 0.1, single_rank=True)
                blk = pairs.cross_pairs(Pd[:S_old], Pd[S_old:], Cd, regularized, 0.1)
                assert torch.equal(blk, single[:S_old, S_old:]), f"cross_pairs, {world} ranks, S={S}, K={K}"
                host = pairs.cross_pairs_host(Pd[:S_old], Pd[S_old:], Cd, regularized, 0.1, n_bands=4)
                assert np.array_equal(host, blk.cpu().numpy())
                old_new, new_rows = pairs.extend_pairs(Pd[:S_old], Pd[S_old:], Cd, regularized, 0.1)
                assert torch.equal(old_new, single[:S_old, S_old:]) and torch.equal(new_rows, single[S_old:])
                EMD_old, _ = tl.wasserstein_d(old, cost, regularized, 0.1)
                EMD, df = tl.wasserstein_d_extend(old, EMD_old, new, cost, regularized, 0.1)
                assert np.array_equal(EMD, single.cpu().numpy()), \
                    f"wasserstein_d_extend {regularized}: {world} ranks and 1 rank differ (S={S}, K={K})"
                assert np.array_equal(df.to_numpy(), EMD.T)
                D, _ = tl.wasserstein_d_cross(old, new, cost, regularized, 0.1)
                assert np.array_equal(D, EMD[:S_old, S_old:])
                ref = torch.from_numpy(EMD).cuda()
                dist.broadcast(ref, 0)
                assert np.array_equal(ref.cpu().numpy(), EMD), "ranks disagree after the all-gather"
    dist.barrier()
    if rank == 0:
        print(f"MULTIRANK CROSS OK world={world}", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
