// C-ABI entry of kernel (3): dispatch between the batched shared-Gibbs-kernel solvers and
// the reference-form kernel (reference call site: pilotpy/tools/Trajectory.py:513-515).
#include <stdint.h>
#include <stdlib.h>
#include <algorithm>
#include "sinkhorn.cuh"

namespace pilot {

// the device counters in the workspace's 256-byte header, zeroed at the start of every call
struct SkCounters {
    unsigned long long fast;    // next problem of the warp-form, panel and FP32 kernels
    unsigned long long n_redo;  // problems queued for the reference-form kernel
    unsigned long long slow;    // next work item of the reference-form kernel
    unsigned long long n_tail;  // problems the panels handed over
    unsigned long long tail;    // next handed-over problem of the tail kernel
};

// the regions of a call's workspace
struct SkWorkspace {
    SkCounters *ctr;
    double *setup, *scratch;
    long long *redo;
    SkTailRec *tail_rec;
    double *tail_uv;
    double *gibbs;  // the reference-form kernel's Gibbs matrices when they do not fit shared memory
    size_t bytes;   // end of the last region
};

// carves the workspace at `base` (nullptr: only its size).  Up to 64 types every region is what the panel kernels
// need; above, the setup buffer has the extent roundup(K, 8), and the scratch also holds the wide kernel's rea / reb.
static SkWorkspace sk_workspace(void *base, int K)
{
    const int KP = skb_pad(K <= 64 ? K : 64);
    const size_t tail_slots = (size_t)sm_count() * skb_slots_per_cta();  // every panel slot could be handed over
    uintptr_t p = (uintptr_t)base;
    const auto take = [&p](size_t bytes) { const uintptr_t r = p; p += bytes; return r; };
    SkWorkspace ws;
    ws.ctr = (SkCounters *)take(256);
    ws.setup = (double *)take(skb_setup_bytes(sk_setup_extent(K)));
    const size_t wide_scratch = K > 64 ? skw_scratch_bytes(sm_count()) : 0;
    ws.scratch = (double *)take(std::max(skb_scratch_bytes(KP, sm_count()), wide_scratch));
    ws.redo = (long long *)take((size_t)SK_REDO_CAP * sizeof(long long));
    ws.tail_rec = (SkTailRec *)take((tail_slots * sizeof(SkTailRec) + 255) / 256 * 256);
    ws.tail_uv = (double *)take(tail_slots * 2 * KP * sizeof(double));
    const size_t gibbs = sinkhorn_ref_gibbs_bytes(K);
    ws.gibbs = gibbs ? (double *)take(gibbs) : nullptr;
    ws.bytes = p - (uintptr_t)base;
    return ws;
}

size_t sinkhorn_ws_bytes(int K) { return sk_workspace(nullptr, K).bytes; }

}  // namespace pilot

extern "C" int pilot_sinkhorn_pairs(const double *props, int S, int K, const double *cost, double reg,
                                    int num_iter_max, double stop_thr, double tau, int check_every,
                                    const pilot_pair_range *range, int algo, int precision, double *out,
                                    int32_t *iters,
                                    int32_t *absorptions, int32_t *status, void *workspace,
                                    size_t workspace_bytes, void *stream)
{
    using namespace pilot;
    PILOT_CHECK_ARG(props && cost && out && workspace, "pilot_sinkhorn_pairs: NULL pointer");
    PILOT_CHECK_ARG(S >= 1, "pilot_sinkhorn_pairs: S=%d", S);
    PILOT_CHECK_ARG(K >= 1 && K <= 256, "pilot_sinkhorn_pairs: K=%d outside the supported range [1, 256]", K);
    PILOT_CHECK_ARG(reg > 0.0, "pilot_sinkhorn_pairs: reg must be > 0");
    PILOT_CHECK_ARG(num_iter_max >= 1 && check_every >= 1, "pilot_sinkhorn_pairs: bad iteration parameters");
    PILOT_CHECK_ARG(algo == 0 || algo == 1 || algo == 3, "pilot_sinkhorn_pairs: algo %d", algo);
    PILOT_CHECK_ARG(precision == PILOT_F64 || precision == PILOT_F32, "pilot_sinkhorn_pairs: precision=%d", precision);
    const SkWorkspace ws = sk_workspace(workspace, K);
    PILOT_CHECK_ARG(workspace_bytes >= ws.bytes, "pilot_sinkhorn_pairs: workspace %zu < %zu bytes", workspace_bytes,
                    ws.bytes);
    PairMap pm;
    int rc = make_pair_map(range, S, &pm);
    if (rc) return rc;
    if (pm.n_local == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    SkParams prm{reg, stop_thr, tau, num_iter_max, check_every};
    const SkOut res{out, iters, absorptions, status, ws.redo, &ws.ctr->n_redo};

    PILOT_CUDA(cudaMemsetAsync(ws.ctr, 0, sizeof(SkCounters), st));
    if (algo == 1)
        return sinkhorn_ref_launch(props, K, cost, prm, pm, res, SK_SOLVE_ALL, &ws.ctr->slow, ws.gibbs, st);
    long long redo_cap = SK_REDO_CAP;
    // (PILOT_SK_REDO_CAP, tests only: a smaller list capacity, to exercise the overflow scan)
    if (const char *e = getenv("PILOT_SK_REDO_CAP")) {
        const long long v = atoll(e);
        if (v >= 0 && v < redo_cap) redo_cap = v;
    }
    if (K > 64) {
        // 65..256 types, FP64 whatever the precision: DMMA panels with K0 split over a cluster (both variants are
        // enqueued, the setup kernel's asymmetry flag picks one on the device), then the reference form for
        // the problems the scaled form cannot carry
        rc = skb_setup(cost, K, prm, ws.setup, st);
        if (rc) return rc;
        for (int sym = 1; sym >= 0; --sym) {
            rc = skw_launch(props, K, prm, pm, ws.setup, ws.scratch, sym != 0, res, &ws.ctr->fast, st);
            if (rc) return rc;
        }
        return sinkhorn_ref_launch(props, K, cost, prm, pm, res, redo_cap, &ws.ctr->slow, ws.gibbs, st);
    }
    if (precision == PILOT_F32) {
        // single precision: per-problem kernel in registers (sinkhorn_f32.cu); what it cannot carry (NaN/Inf,
        // zero masses) goes to the FP64 reference-form kernel like in the FP64 mode
        rc = skf_launch(props, K, cost, prm, pm, res, &ws.ctr->fast, st);
        if (rc) return rc;
        return sinkhorn_ref_launch(props, K, cost, prm, pm, res, redo_cap, &ws.ctr->slow, ws.gibbs, st);
    }
    // evict_max measured: 0 (no hand-over) 2.23 ms, 2: 1.45 ms, 4: 1.44 ms, 7: 1.56 ms for 10^4 problems at K = 64
    const SkTail tail{ws.tail_rec, ws.tail_uv, &ws.ctr->n_tail, 2};
    rc = skb_setup(cost, K, prm, ws.setup, st);
    if (rc) return rc;
    // The cost is symmetric in PILOT (a pdist matrix) but the API takes any matrix.  Whether it is is known
    // only on the device (setup kernel), so the symmetric and the general variant of each solver are both
    // enqueued and the one that does not apply returns at once: no host read-back, the call is fully
    // asynchronous on `stream`.
    // persistent grid: one CTA per SM.  With little work (latency-, not throughput-bound) spread it
    // over all SMs and run only as many warps / slot sets per CTA as there are slot-loads of
    // problems: fewer of them share the FP64 tensor pipe, so every iteration returns sooner.
    const int slot_cap = 2;
    // few cell types: one warp per problem with K0 in registers (lowest latency per iteration, and
    // for 17..32 types also the higher throughput).  With <= 16 types half of its lanes idle, so a
    // large batch goes to the DMMA panels instead (measured: 400 K problems, K = 12: 5.6 vs 6.9 ms).
    // The choice depends on the COHORT size only (not on this rank's share or on the window), so that a problem is
    // solved by the same arithmetic however the pair space is partitioned: results are partition-invariant bit for bit.
    // In RECT mode S is the concatenation of the two sets, so a block takes the choice of the square over them.
    const bool warp_form = algo == 0 && K <= swk_max_k() && (K > 16 || (long long)S * S < 200000);
    if (warp_form) {  // symmetric cost only; an asymmetric one falls through to the general panels below
        rc = swk_launch(props, K, prm, pm, ws.setup, res, &ws.ctr->fast, st);
        if (rc) return rc;
    }
    const long long spw = skb_slots_per_warp();
    long long ctas = (pm.n_local + spw - 1) / spw;
    if (ctas > sm_count()) ctas = sm_count();
    long long warp_cap = (pm.n_local + spw * ctas - 1) / (spw * ctas);
    if (warp_cap > skb_warps()) warp_cap = skb_warps();
    if (warp_cap < 1) warp_cap = 1;
    for (int sym = warp_form ? 0 : 1; sym >= 0; --sym) {
        rc = skb_launch(props, K, prm, pm, ws.setup, ws.scratch, (int)ctas, slot_cap, (int)warp_cap, sym != 0,
                        tail, res, &ws.ctr->fast, st);
        if (rc) return rc;
    }
    // the stragglers the panels handed over continue in warp form
    for (int sym = warp_form ? 0 : 1; sym >= 0; --sym) {
        rc = skt_launch(props, K, prm, pm, ws.setup, ws.scratch, sym != 0, tail, &ws.ctr->tail, res, st);
        if (rc) return rc;
    }
    // problems the scaled form could not represent (normally none): reference-form kernel
    return sinkhorn_ref_launch(props, K, cost, prm, pm, res, redo_cap, &ws.ctr->slow, ws.gibbs, st);
}

extern "C" int pilot_sinkhorn_plans(const double *props, int S, int K, const double *cost, double reg,
                                    int num_iter_max, double stop_thr, double tau, int check_every,
                                    const int32_t *pair_a, const int32_t *pair_b, int64_t n, double *plans,
                                    double *out, int32_t *iters, int32_t *absorptions, int32_t *status,
                                    void *workspace, size_t workspace_bytes, void *stream)
{
    using namespace pilot;
    PILOT_CHECK_ARG(props && cost && pair_a && pair_b && plans && out && workspace,
                    "pilot_sinkhorn_plans: NULL pointer");
    PILOT_CHECK_ARG(S >= 1, "pilot_sinkhorn_plans: S=%d", S);
    PILOT_CHECK_ARG(K >= 1 && K <= 256, "pilot_sinkhorn_plans: K=%d outside the supported range [1, 256]", K);
    PILOT_CHECK_ARG(n >= 0, "pilot_sinkhorn_plans: n=%lld", (long long)n);
    PILOT_CHECK_ARG(reg > 0.0, "pilot_sinkhorn_plans: reg must be > 0");
    PILOT_CHECK_ARG(num_iter_max >= 1 && check_every >= 1, "pilot_sinkhorn_plans: bad iteration parameters");
    const SkWorkspace ws = sk_workspace(workspace, K);
    PILOT_CHECK_ARG(workspace_bytes >= ws.bytes, "pilot_sinkhorn_plans: workspace %zu < %zu bytes", workspace_bytes,
                    ws.bytes);
    if (n == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const SkParams prm{reg, stop_thr, tau, num_iter_max, check_every};
    const SkOut res{out, iters, absorptions, status, ws.redo, &ws.ctr->n_redo};
    PILOT_CUDA(cudaMemsetAsync(ws.ctr, 0, sizeof(SkCounters), st));
    // the reference form: POT's own statement of Gamma, for every K <= 256 (bit-identical costs to algo = 1)
    return sinkhorn_ref_plans_launch(props, K, cost, prm, plan_pair_map(n, S), res,
                                     PlanArgs<true>{pair_a, pair_b, S, plans}, &ws.ctr->slow, ws.gibbs, st);
}
