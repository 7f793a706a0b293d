// Kernel (3), tail of the DMMA-panel Sinkhorn solver: one warp per handed-over problem, continuing
// from the exported scaled iterates (reference call site pilotpy/tools/Trajectory.py:513-515, POT
// sinkhorn_stabilized schedule; K0 in shared memory because 2 x 64 rows per lane do not fit the
// register file).
//
// BIT-IDENTICAL to the panels.  Which problems are handed over depends on timing, so the result of a
// problem must not depend on where it finishes.  mma.sync.m8n8k4.f64 accumulates its four products as a
// chain of FMAs in ascending k (measured: tools/dmma_order.cu, 0 mismatches in 128 000 entries), so a
// panel matvec row is the sequential chain s = fma(K0[i][row], x[i], s), i = 0, 1, 2, ...; the matvecs here
// run exactly that chain (two rows per lane), the marginal error is summed in the panels' order (rows
// 8m + g ascending in m, then the g-butterfly 1, 2, 4) and the final cost uses the panels' code.  Two runs,
// and runs on 1, 2, 4 or 8 GPUs, therefore give bit-identical Sinkhorn matrices.
//
// A panel of 8 problems costs ~6 us per iteration however few of its slots are still in use; the
// stragglers of a batch (the problems that run to the 1000-iteration cap while the mean is ~55)
// would keep whole SMs busy at 1/8 occupancy for milliseconds.  Here lane j owns rows 2j and 2j + 1,
// a matvec is 2 x KP DFMAs per lane against K0 columns read conflict-free from shared memory (128-bit
// loads), and an iteration takes 1.2 us at K = 64 -- bound by the ~45 B/clk one warp gets out of its SM
// sub-partition's shared-memory port, not by the arithmetic.
#include "sinkhorn.cuh"

namespace pilot {

constexpr int SKT_WARPS = 16;

// res[rr] = sum_i mat[i][row0 + rr] * buf[i] as ONE fma chain in ascending i per row -- the order in which the
// DMMA panels accumulate (see the header) -- (mat is [KP][KP], i-major; the lane's R rows are adjacent, so
// R = 2 reads them with one 128-bit load; buf is broadcast as 128-bit loads)
template <int KP, int R>
__device__ __forceinline__ void skt_matvec(const double *__restrict__ mat, int row0, const double *buf,
                                           double (&res)[R])
{
    double s[R];
#pragma unroll
    for (int rr = 0; rr < R; ++rr) s[rr] = 0.0;
    const double *m = mat + row0;
#pragma unroll 4
    for (int i = 0; i < KP; i += 2) {
        const double2 x = *reinterpret_cast<const double2 *>(buf + i);
        if (R == 2) {
            const double2 k0 = *reinterpret_cast<const double2 *>(m + i * KP);
            const double2 k1 = *reinterpret_cast<const double2 *>(m + (i + 1) * KP);
            s[0] = fma(k0.x, x.x, s[0]);
            s[R - 1] = fma(k0.y, x.x, s[R - 1]);
            s[0] = fma(k1.x, x.y, s[0]);
            s[R - 1] = fma(k1.y, x.y, s[R - 1]);
        } else {
            s[0] = fma(m[i * KP], x.x, s[0]);
            s[0] = fma(m[(i + 1) * KP], x.y, s[0]);
        }
    }
#pragma unroll
    for (int rr = 0; rr < R; ++rr) res[rr] = s[rr];
}

template <int KP, bool SYM>
__global__ void __launch_bounds__(SKT_WARPS * 32, 1)
sinkhorn_tail_kernel(const double *__restrict__ props, int K, SkParams prm, PairMap pm, SkSetup s,
                     const double *__restrict__ scratch, SkTail tail, unsigned long long *__restrict__ tail_counter,
                     double *__restrict__ out, int *__restrict__ iters_out, int *__restrict__ abs_out,
                     int *__restrict__ status_out, long long *__restrict__ redo_list,
                     unsigned long long *__restrict__ n_redo)
{
    const SkOut res{out, iters_out, abs_out, status_out, redo_list, n_redo};
    constexpr int R = (KP + 31) / 32;  // rows per lane
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *sK0 = reinterpret_cast<double *>(smem_raw);  // [i][j]: column access for T = K0^T ut
    double *sMK = sK0 + KP * KP;                         // M o K0
    double *sK0T = SYM ? sK0 : sMK + KP * KP;            // [j][i]: column access for S = K0 vt
    double *sbuf = (SYM ? sMK : sK0T) + KP * KP;         // per warp: broadcast copies of ut, vt
    const unsigned long long n_tail = *tail.n_tail;
    if (n_tail == 0 || (*s.asym != 0) == SYM) return;
    for (int e = threadIdx.x; e < KP * KP; e += blockDim.x) {
        sK0[e] = s.K0[e];
        sMK[e] = s.MK[e];
        if (!SYM) sK0T[e] = s.K0T[e];
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double *ub = sbuf + (size_t)warp * 3 * KP, *vb = ub + KP, *db = vb + KP;
    const int kc = (K + 7) & ~7;  // the panels' compute extent
    int row[R];
    bool in_pad[R], row_ok[R];
#pragma unroll
    for (int rr = 0; rr < R; ++rr) {
        const int r = R * lane + rr;  // adjacent rows per lane
        in_pad[rr] = r < KP;
        row_ok[rr] = r < K;
        row[rr] = in_pad[rr] ? r : 0;
    }
    const long long tau_bits = __double_as_longlong(prm.tau);
    const double invK = 1.0 / K;

    for (;;) {
        unsigned long long idx = 0;
        if (lane == 0) idx = atomicAdd(tail_counter, 1ULL);
        idx = __shfl_sync(0xffffffffu, idx, 0);
        if (idx >= n_tail) break;
        const SkTailRec rec = tail.rec[idx];
        const long long w = rec.prob;
        int si, sj;
        global_to_ij(pm, local_to_global(pm, w), si, sj);
        double a[R], b[R], u[R], v[R], rea[R], reb[R];
#pragma unroll
        for (int rr = 0; rr < R; ++rr) {
            const int r = row[rr];
            a[rr] = row_ok[rr] ? __ldg(props + (long long)si * K + r) : 0.0;
            b[rr] = row_ok[rr] ? __ldg(props + (long long)sj * K + r) : 0.0;
            u[rr] = row_ok[rr] ? tail.uv[idx * 2 * KP + r] : 0.0;
            v[rr] = row_ok[rr] ? tail.uv[idx * 2 * KP + KP + r] : 0.0;
            const bool ha = rec.hasabs && row_ok[rr];
            rea[rr] = ha ? scratch[(size_t)rec.sslot * 2 * KP + r] : 1.0;
            reb[rr] = ha ? scratch[(size_t)rec.sslot * 2 * KP + KP + r] : 1.0;
        }
        int ii = rec.ii, nabs = rec.nabs, status = PILOT_ST_MAXITER;
        int ctl = 0;  // the hand-over happens right after a resolve: nothing pending
        int until_check = (prm.check_every - ii % prm.check_every) % prm.check_every;
        for (;;) {
            // ---- T = K0^T ut, then resolve the check / cap of the previous iteration ----
#pragma unroll
            for (int rr = 0; rr < R; ++rr)
                if (in_pad[rr]) ub[row[rr]] = u[rr];
            __syncwarp();
            double T[R];
            skt_matvec<KP, R>(sK0, row[0], ub, T);
            if (ii == 0) {
                // a slot can be handed over right after it was refilled: the panels take the first product
                // K0^T (1/K) from the setup kernel's c0 (summed in another order), and so must we
#pragma unroll
                for (int rr = 0; rr < R; ++rr) T[rr] = __ldg(s.c0 + row[rr]);
            }
            if (ctl) {
                if (ctl & SK_BAD) { status = -1; break; }
                bool conv = false;
                if (ctl & SK_PEND) {
                    // || vt o T - b ||^2 summed like the panels do: lane g takes rows g, 8 + g, ... in ascending
                    // order, then the butterfly over g
#pragma unroll
                    for (int rr = 0; rr < R; ++rr)
                        if (in_pad[rr]) db[row[rr]] = row_ok[rr] ? fma(v[rr], T[rr], -b[rr]) : 0.0;
                    __syncwarp();
                    double e2 = 0.0;
                    for (int r8 = lane & 7; r8 < kc; r8 += 8)
                        if (r8 < K) { const double d = db[r8]; e2 = fma(d, d, e2); }
                    e2 += __shfl_xor_sync(0xffffffffu, e2, 1);
                    e2 += __shfl_xor_sync(0xffffffffu, e2, 2);
                    e2 += __shfl_xor_sync(0xffffffffu, e2, 4);
                    conv = sqrt(e2) <= prm.stop_thr;
                    __syncwarp();
                }
                if (conv) { status = PILOT_ST_CONVERGED; break; }
                if (ctl & SK_FORCE) { status = PILOT_ST_MAXITER; break; }
            }
            // ---- vt = b / T ----
#pragma unroll
            for (int rr = 0; rr < R; ++rr) {
                v[rr] = row_ok[rr] ? sk_div(b[rr], T[rr]) : 0.0;
                if (in_pad[rr]) vb[row[rr]] = v[rr];
            }
            __syncwarp();
            // ---- ut = a / (K0 vt) ----
            double S[R];
            skt_matvec<KP, R>(sK0T, row[0], vb, S);
            long long mx = 0;
#pragma unroll
            for (int rr = 0; rr < R; ++rr) {
                u[rr] = row_ok[rr] ? sk_div(a[rr], S[rr]) : 0.0;
                // u, v of the reference = ut * rea, vt * reb
                mx = max(mx, max(sk_abs_bits(u[rr] * rea[rr]), sk_abs_bits(v[rr] * reb[rr])));
            }
            ctl = sk_step(prm, until_check, ii);
            if (__any_sync(0xffffffffu, mx > tau_bits)) {
                if (__any_sync(0xffffffffu, mx >= SK_NONFINITE_BITS)) {
                    ctl |= SK_BAD;
                } else {
                    // absorption: u = v = 1/K in POT == divide the scaled iterates by K; remember 1/ut, 1/vt
                    bool r = false;
#pragma unroll
                    for (int rr = 0; rr < R; ++rr)
                        if (row_ok[rr]) {
                            rea[rr] = 1.0 / u[rr];
                            reb[rr] = 1.0 / v[rr];
                            r |= sk_out_of_range(u[rr], v[rr]);
                            u[rr] *= invK;
                            v[rr] *= invK;
                        }
                    ++nabs;
                    if (__any_sync(0xffffffffu, r)) ctl |= SK_BAD;
                }
            }
        }
        if (status >= 0) {
            // cost = sum_j vt_j * sum_i (M o K0)_ij ut_i in the panels' order: lane = column j, even / odd rows in
            // two chains (ub holds the current ut; vt may have been rescaled by an absorption since vb was written)
            __syncwarp();
#pragma unroll
            for (int rr = 0; rr < R; ++rr)
                if (in_pad[rr]) vb[row[rr]] = v[rr];
            __syncwarp();
            double c = 0.0;
            for (int j = lane; j < kc; j += 32) {
                double w0 = 0.0, w1 = 0.0;
                for (int i = 0; i + 1 < K; i += 2) {
                    w0 = fma(sMK[i * KP + j], ub[i], w0);
                    w1 = fma(sMK[(i + 1) * KP + j], ub[i + 1], w1);
                }
                if (K & 1) w0 = fma(sMK[(K - 1) * KP + j], ub[K - 1], w0);
                c = fma(vb[j], w0 + w1, c);
            }
            const double cost = warp_sum_d(c);
            if (lane == 0) sk_store(res, w, status, cost, ii, nabs);
        } else if (lane == 0) {
            sk_store(res, w, status, 0.0, ii, nabs);
        }
        __syncwarp();
    }
}

template <int KP, bool SYM>
static int skt_launch_t(const double *props, int K, const SkParams &prm, const PairMap &pm, const SkSetup &s,
                        const double *scratch, const SkTail &tail, unsigned long long *tail_counter, const SkOut &res,
                        cudaStream_t st)
{
    const size_t smem = sizeof(double) * ((size_t)(SYM ? 2 : 3) * KP * KP + (size_t)SKT_WARPS * 3 * KP);
    PILOT_CUDA(cudaFuncSetAttribute(sinkhorn_tail_kernel<KP, SYM>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)smem));
    sinkhorn_tail_kernel<KP, SYM><<<sm_count(), SKT_WARPS * 32, smem, st>>>(
        props, K, prm, pm, s, scratch, tail, tail_counter, res.out, res.iters, res.absn, res.status, res.redo,
        res.n_redo);
    PILOT_LAUNCH_CHECK();
    return 0;
}

// continues the problems the panel kernel handed over (none: the CTAs return at once)
int skt_launch(const double *props, int K, const SkParams &prm, const PairMap &pm, const double *setup,
               const double *scratch, bool symmetric, const SkTail &tail, unsigned long long *tail_counter,
               const SkOut &res, cudaStream_t st)
{
    const int KP = skb_pad(K);
    const SkSetup s = sk_setup_view(setup, KP);
#define SKT_GO(KPV) \
    return (symmetric ? skt_launch_t<KPV, true> : skt_launch_t<KPV, false>)(props, K, prm, pm, s, scratch, tail, \
                                                                            tail_counter, res, st)
    if (KP == 16) SKT_GO(16);
    if (KP == 32) SKT_GO(32);
    if (KP == 48) SKT_GO(48);
    SKT_GO(64);
#undef SKT_GO
}

}  // namespace pilot
