// Shared declarations and device helpers of the Sinkhorn kernels (sinkhorn_ref.cu, sinkhorn_batched.cu,
// sinkhorn_tail.cu, sinkhorn_warp.cu, sinkhorn_f32.cu, sinkhorn_wide.cu).
#pragma once
#include "common.cuh"

namespace pilot {

struct SkParams {
    double reg, stop_thr, tau;
    int num_iter_max, check_every;
};

constexpr long long SK_REDO_CAP = 1LL << 20;
// out[] of a problem queued for the reference-form kernel: a NaN with this payload.  When more than
// SK_REDO_CAP problems are queued the list overflows and the reference-form kernel finds the rest by
// scanning out[] for the marker (sinkhorn_ref.cu, mode 2), so no problem is ever left unsolved.
constexpr long long SK_REDO_MARK = 0x7ff8b200b200b200LL;

// where the solvers leave their results (iters, absn, status may be nullptr), and the list of problems queued for
// the reference-form kernel.  The kernels take the six pointers as __restrict__ parameters and assemble it
// themselves: inside a struct argument the pointers lose __restrict__, which cost the panel and tail kernels
// registers and spills.
struct SkOut {
    double *out;
    int *iters, *absn, *status;
    long long *redo;
    unsigned long long *n_redo;
};

// the setup buffer skb_setup fills (sk_setup_view): K0, K0^T, M o K0 (KP x KP each, zero padded, KP =
// sk_setup_extent(K)), c0 = K0^T (1/K), and a flag that is != 0 when M differs from its transpose; the solver kernels read the flag themselves
struct SkSetup {
    const double *K0, *K0T, *MK, *c0;
    const int *asym;
};

// hand-over of straggler problems from the DMMA-panel kernel to the warp-form tail kernel
struct SkTailRec {
    long long prob;  // local problem index
    int ii, nabs, hasabs;
    int sslot;       // index of the problem's rea / reb block in the panel kernel's scratch
};
struct SkTail {
    SkTailRec *rec;  // nullptr: no hand-over
    double *uv;      // [slot][ut | vt][KP]
    unsigned long long *n_tail;
    int evict_max;   // a warp hands its problems over when the pool is empty and <= this many are left
};

// branch-free x / y for finite positive y: 20-bit seed r, e = 1 - y r, q = x r (1 + e + e^2): relative error
// e^3 ~ 2^-60 before the final rounding.  MUFU + 3 FP64-pipe instructions in a dependent chain of 3: the FP64 pipe
// is what the panels' element-wise phases pay for (it queues behind the DMMAs), the chain what a lone warp pays for.
__device__ __forceinline__ double sk_div(double x, double y)
{
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(y));
    const double e = fma(-y, r, 1.0);
    const double q0 = x * r;
    return fma(q0, fma(e, e, e), q0);
}

// |x| as an ordered integer: for non-NaN doubles the bit pattern orders like the value, NaN / Inf
// sort above every finite value -- max / threshold tests as integer compares
__device__ __forceinline__ long long sk_abs_bits(double x) { return __double_as_longlong(x) & 0x7fffffffffffffffLL; }
constexpr long long SK_NONFINITE_BITS = 0x7ff0000000000000LL;  // sk_abs_bits of +-Inf: NaN and Inf are >= this

// an absorption at ut = u or vt = v outside 1e-250 .. 1e250 would take e^{+-alpha/reg} too close to the edge of
// the FP64 range: the problem goes to the reference form instead
__device__ __forceinline__ bool sk_out_of_range(double u, double v)
{
    return !(u > 1e-250 && u < 1e250 && v > 1e-250 && v < 1e250);
}

// What the next round of a one-problem-per-warp solver (warp form, tail) resolves before it iterates again:
// a pending marginal check (every check_every iterations, counted down in until_check), the iteration cap,
// a problem the scaled form cannot carry.
enum { SK_PEND = 1, SK_FORCE = 2, SK_BAD = 4 };
__device__ __forceinline__ int sk_step(const SkParams &prm, int &until_check, int &ii)
{
    int ctl = (until_check == 0) ? SK_PEND : 0;
    until_check = (until_check == 0 ? prm.check_every : until_check) - 1;
    ++ii;
    if (ii >= prm.num_iter_max) ctl |= SK_FORCE;
    return ctl;
}

// Writes the result of problem w, or (status < 0) queues it for the reference-form kernel and leaves the marker
// in out[w].  One lane per problem calls it.
__device__ __forceinline__ void sk_store(const SkOut &res, long long w, int status, double cost, int ii, int nabs)
{
    if (status >= 0) {
        res.out[w] = cost;
        if (res.iters) res.iters[w] = ii;
        if (res.absn) res.absn[w] = nabs;
        if (res.status) res.status[w] = status;
    } else {
        const unsigned long long slot = atomicAdd(res.n_redo, 1ULL);
        if ((long long)slot < SK_REDO_CAP) res.redo[slot] = w;
        res.out[w] = __longlong_as_double(SK_REDO_MARK);
        if (res.status) res.status[w] = -1;
    }
}

size_t sinkhorn_ref_smem(int K);
// workspace the reference-form kernel needs for its Gibbs matrices: 0 while they fit shared memory
size_t sinkhorn_ref_gibbs_bytes(int K);
// redo_cap: SK_SOLVE_ALL, or solve the problems queued in res.redo (at most redo_cap of them are listed; the rest is
// found by their marker).  gibbs: sinkhorn_ref_gibbs_bytes(K) bytes of workspace (nullptr when that is 0).
constexpr long long SK_SOLVE_ALL = -1;
int sinkhorn_ref_launch(const double *props, int K, const double *cost, const SkParams &prm, const PairMap &pm,
                        const SkOut &res, long long redo_cap, unsigned long long *counter, double *gibbs,
                        cudaStream_t st);
// plan variant (pilot_sinkhorn_plans): mode 0 over the pair list of `plan`, pm = plan_pair_map(n, S)
int sinkhorn_ref_plans_launch(const double *props, int K, const double *cost, const SkParams &prm,
                              const PairMap &pm, const SkOut &res, const PlanArgs<true> &plan,
                              unsigned long long *counter, double *gibbs, cudaStream_t st);

int skb_pad(int K);
// storage extent of the setup buffer: skb_pad(K) up to 64 types, roundup(K, 8) above
int sk_setup_extent(int K);
size_t skb_setup_bytes(int KP);
SkSetup sk_setup_view(const double *setup, int KP);
size_t skb_smem_bytes(int KP);
size_t skb_scratch_bytes(int KP, int ctas);
int skb_slots_per_cta();
int skb_slots_per_warp();
int skb_warps();
int skb_setup(const double *cost, int K, const SkParams &prm, double *setup, cudaStream_t st);
int skb_launch(const double *props, int K, const SkParams &prm, const PairMap &pm, const double *setup,
               double *scratch, int ctas, int slot_cap, int warp_cap, bool symmetric, const SkTail &tail,
               const SkOut &res, unsigned long long *counter, cudaStream_t st);

// warp-form continuation of the handed-over problems (sinkhorn_tail.cu)
int skt_launch(const double *props, int K, const SkParams &prm, const PairMap &pm, const double *setup,
               const double *scratch, bool symmetric, const SkTail &tail, unsigned long long *tail_counter,
               const SkOut &res, cudaStream_t st);

// one warp per problem, K0 in registers (sinkhorn_warp.cu): K <= swk_max_k(), symmetric cost
int swk_max_k();
int swk_launch(const double *props, int K, const SkParams &prm, const PairMap &pm, const double *setup,
               const SkOut &res, unsigned long long *counter, cudaStream_t st);

// 65 <= K <= 256: DMMA panels with K0 split in row stripes over a thread-block cluster (sinkhorn_wide.cu);
// scratch: skw_scratch_bytes(sm_count()) bytes
size_t skw_scratch_bytes(int ctas);
int skw_launch(const double *props, int K, const SkParams &prm, const PairMap &pm, const double *setup,
               double *scratch, bool symmetric, const SkOut &res, unsigned long long *counter, cudaStream_t st);

// FP32 mode: one warp per problem, per-problem kernel in registers (sinkhorn_f32.cu), K <= 64
int skf_launch(const double *props, int K, const double *cost, const SkParams &prm, const PairMap &pm,
               const SkOut &res, unsigned long long *counter, cudaStream_t st);

}  // namespace pilot
