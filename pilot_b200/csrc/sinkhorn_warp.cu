// Kernel (3), small-K form of the shared-Gibbs-kernel Sinkhorn solver: one warp per problem, the
// Gibbs kernel K0 = exp(-M / reg) in REGISTERS (reference call site pilotpy/tools/Trajectory.py:513-515,
// POT sinkhorn_stabilized schedule; same scaled formulation as sinkhorn_batched.cu).
//
// For K <= 32 cell types and a symmetric cost (PILOT's cost is a pdist matrix) lane j owns row j of
// every vector and keeps column j of K0 -- which is also row j -- in 2 * KP registers.  A matvec is
// KP DFMAs per lane against the other vector broadcast from a 256-byte shared buffer, so an
// iteration is two short dependent chains (measured 0.35 us for a lone warp) instead of two
// 8-problem DMMA panels (2.8 us): the stragglers that run the full 1000 iterations no longer set the time of a small
// batch, and with the FP64 DFMA peak equal to the DMMA peak on B200 nothing is lost on a large
// one.  Problems the scaled form cannot represent go to the redo list (reference-form kernel).
#include "sinkhorn.cuh"

namespace pilot {

constexpr int SWK_WARPS = 8;

// sum_i k0[i] * buf[i]; buf is read as 128-bit broadcasts; 8 independent chains of KP / 8 FMAs and a
// 3-level tree (16 chains would save one more dependent op but spill at KP = 32)
template <int KP>
__device__ __forceinline__ double swk_matvec(const double (&k0)[KP], const double *buf)
{
    double s[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) s[c] = 0.0;
#pragma unroll
    for (int i = 0; i < KP; i += 2) {
        const double2 x = *reinterpret_cast<const double2 *>(buf + i);
        s[i & 7] = fma(k0[i], x.x, s[i & 7]);
        s[(i + 1) & 7] = fma(k0[i + 1], x.y, s[(i + 1) & 7]);
    }
    return ((s[0] + s[1]) + (s[2] + s[3])) + ((s[4] + s[5]) + (s[6] + s[7]));
}

template <int KP>
__global__ void __launch_bounds__(SWK_WARPS * 32, 2)
sinkhorn_warp_kernel(const double *__restrict__ props, int K, SkParams prm, PairMap pm, SkSetup s,
                     unsigned long long *__restrict__ counter, double *__restrict__ out, int *__restrict__ iters_out,
                     int *__restrict__ abs_out, int *__restrict__ status_out, long long *__restrict__ redo_list,
                     unsigned long long *__restrict__ n_redo)
{
    const SkOut res{out, iters_out, abs_out, status_out, redo_list, n_redo};
    __shared__ double sMK[KP * KP];                             // M o K0, for the final cost
    __shared__ __align__(16) double sbuf[SWK_WARPS][2][KP];    // per warp: broadcast copies of ut, vt
    if (*s.asym != 0) return;  // asymmetric cost: the panel kernel enqueued behind this one runs instead
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int e = threadIdx.x; e < KP * KP; e += blockDim.x) sMK[e] = s.MK[e];
    __syncthreads();

    const int j = lane;
    const bool in_pad = j < KP, row_ok = j < K;
    const int jc = in_pad ? j : 0;
    double k0[KP];  // column j of K0 (== row j: the cost is symmetric)
#pragma unroll
    for (int i = 0; i < KP; ++i) k0[i] = in_pad ? s.K0[i * KP + jc] : 0.0;
    double *ub = sbuf[warp][0], *vb = sbuf[warp][1];
    const long long tau_bits = __double_as_longlong(prm.tau);
    const double invK = 1.0 / K;

    for (;;) {
        unsigned long long w = 0;
        if (lane == 0) w = atomicAdd(counter, 1ULL);
        w = __shfl_sync(0xffffffffu, w, 0);
        if ((long long)w >= pm.n_local) break;
        int si, sj;
        global_to_ij(pm, local_to_global(pm, (long long)w), si, sj);
        const double a = row_ok ? __ldg(props + (long long)si * K + j) : 0.0;
        const double b = row_ok ? __ldg(props + (long long)sj * K + j) : 0.0;
        // ut, vt >= 0 always; rea = 1 / ut, reb = 1 / vt at the last absorption (1 before the first)
        double u = row_ok ? invK : 0.0, v = u, rea = 1.0, reb = 1.0;
        int ii = 0, nabs = 0, status = PILOT_ST_MAXITER;
        int ctl = 0;               // what the next round has to resolve: SK_PEND | SK_FORCE | SK_BAD
        int until_check = 0;       // iterations until the next convergence check (ii % check_every == 0)
        for (;;) {
            // ---- T = K0^T ut, then resolve the check / cap of the previous iteration ----
            if (in_pad) ub[j] = u;
            __syncwarp();
            const double T = swk_matvec<KP>(k0, ub);
            if (ctl) {
                if (ctl & SK_BAD) { status = -1; break; }
                bool conv = false;
                if (ctl & SK_PEND) {
                    const double d = row_ok ? fma(v, T, -b) : 0.0;
                    conv = sqrt(warp_sum_d(d * d)) <= prm.stop_thr;
                }
                if (conv) { status = PILOT_ST_CONVERGED; break; }
                if (ctl & SK_FORCE) { status = PILOT_ST_MAXITER; break; }
            }
            // ---- vt = b / T ----
            v = row_ok ? sk_div(b, T) : 0.0;
            if (in_pad) vb[j] = v;
            __syncwarp();
            // ---- ut = a / (K0 vt) ----
            const double S = swk_matvec<KP>(k0, vb);
            u = row_ok ? sk_div(a, S) : 0.0;
            // u, v of the reference = ut * rea, vt * reb: absorb when one exceeds tau
            const long long mx = max(sk_abs_bits(u * rea), sk_abs_bits(v * reb));
            ctl = sk_step(prm, until_check, ii);
            if (__any_sync(0xffffffffu, mx > tau_bits)) {
                if (__any_sync(0xffffffffu, mx >= SK_NONFINITE_BITS)) {
                    ctl |= SK_BAD;  // NaN or Inf somewhere in u, v
                } else {
                    // absorption: u = v = 1/K in POT == divide the scaled iterates by K; remember 1/ut, 1/vt
                    bool r = false;
                    if (row_ok) {
                        rea = 1.0 / u;
                        reb = 1.0 / v;
                        r = sk_out_of_range(u, v);
                        u *= invK;
                        v *= invK;
                    }
                    ++nabs;
                    if (__any_sync(0xffffffffu, r)) ctl |= SK_BAD;
                }
            }
        }
        double cost = 0.0;
        if (status >= 0) {
            // cost = sum_j vt_j * sum_i (M o K0)_ij ut_i   (ub holds the current ut)
            double c0 = 0.0, c1 = 0.0;
            if (in_pad) {
#pragma unroll 4
                for (int i = 0; i < KP; i += 2) {
                    c0 = fma(sMK[i * KP + j], ub[i], c0);
                    c1 = fma(sMK[(i + 1) * KP + j], ub[i + 1], c1);
                }
            }
            cost = warp_sum_d(v * (c0 + c1));
        }
        if (lane == 0) sk_store(res, (long long)w, status, cost, ii, nabs);
        __syncwarp();
    }
}

int swk_max_k() { return 32; }

// `setup` must already hold the output of skb_setup (symmetric cost only)
int swk_launch(const double *props, int K, const SkParams &prm, const PairMap &pm, const double *setup,
               const SkOut &res, unsigned long long *counter, cudaStream_t st)
{
    const int KP = skb_pad(K);
    const SkSetup s = sk_setup_view(setup, KP);
    long long ctas = pm.n_local;  // spread a small batch over all SMs, one problem per warp at a time
    if (ctas > 2LL * sm_count()) ctas = 2LL * sm_count();
    if (KP == 16)
        sinkhorn_warp_kernel<16><<<(int)ctas, SWK_WARPS * 32, 0, st>>>(props, K, prm, pm, s, counter, res.out, res.iters,
                                                                       res.absn, res.status, res.redo, res.n_redo);
    else
        sinkhorn_warp_kernel<32><<<(int)ctas, SWK_WARPS * 32, 0, st>>>(props, K, prm, pm, s, counter, res.out, res.iters,
                                                                       res.absn, res.status, res.redo, res.n_redo);
    PILOT_LAUNCH_CHECK();
    return 0;
}

}  // namespace pilot
