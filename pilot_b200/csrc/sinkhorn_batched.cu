// Kernel (3), batched variant: all-pairs stabilised Sinkhorn with ONE shared Gibbs kernel
// K0 = exp(-M/reg) resident in shared memory for every problem of the CTA.
// Replaces the loop over ot.sinkhorn2(a_i, a_j, cost, reg, method="sinkhorn_stabilized")
// (reference pilotpy/tools/Trajectory.py:513-515; schedule: SURVEY.md Appendix A.2).
//
// Formulation.  POT keeps K = diag(e^{alpha/reg}) K0 diag(e^{beta/reg}) per problem and
// iterates v = b/(K^T u), u = a/(K v).  With ut = e^{alpha/reg} o u and vt = e^{beta/reg} o v
// the same iteration is vt = b/(K0^T ut), ut = a/(K0 vt) on the SHARED K0; alpha/beta only
// matter for (i) the absorption trigger max|u|,|v| > tau, u = ut * rea with rea = e^{-alpha/reg}
// (= 1/ut at the last absorption), and (ii) the reset u = v = 1/K at an absorption, which
// in scaled variables is ut /= K, vt /= K.  The marginal error every `check_every` iterations
// is || vt o (K0^T ut) - b ||, i.e. the product the next iteration needs anyway, and the
// result is sum_ij M_ij K0_ij ut_i vt_j.  Rounding differs from the reference form at the
// 1e-16 level with identical iteration/absorption schedules (SURVEY.md Appendix B.5).
//
// Mapping.  The two matvecs of 8 problems ("slots") at a time are the dense FP64 GEMMs
// K0^T [ut_1 .. ut_8] and K0 [vt_1 .. vt_8]; each warp runs them on the FP64 tensor path
// (mma.sync m8n8k4, DMMA): KP/8 accumulator tiles per warp, A fragments from the shared
// K0 / K0^T (XOR-swizzled: 2 wavefronts per fragment load, the minimum for 256 B), B fragments
// from the warp's private 8-column U / V panel (64-byte rows: conflict free as they are).  In
// the C-fragment layout lane (g = lane/4, t = lane%4) owns rows {8m+g} of the adjacent slots
// {2t, 2t+1}, so the element-wise update (one 128-bit store per row), the max/err reductions
// (3 xor-shuffles over the 8 lanes sharing t) and all per-slot state stay inside the warp: the
// 16 warps of a CTA are independent persistent workers, no CTA barrier in the loop, a finished
// slot is refilled at once from a global counter.  DMMA has the same peak as DFMA on B200
// (measured 37 TFLOP/s both) but needs 1/8 of the issue slots; with 4 warps per scheduler the
// epilogue (FP64 pipe, LSU) of three warps overlaps the DMMA stream of the fourth.
// Problems the scaled form cannot represent (NaN/Inf, |log ut| near the FP64 range) are queued
// for the reference-form kernel (sinkhorn_ref.cu).
#include "sinkhorn.cuh"

namespace pilot {

constexpr int SKB_WARPS = 16;
constexpr int SKB_SPW = 8;  // slots (problems in flight) per warp = panel columns

// K0, K0^T, M o K0 (all KP x KP, zero padded) and c0 = K0^T (1/K) into the workspace
__global__ void skb_setup_kernel(const double *__restrict__ M, int K, int KP, double reg,
                                 double *__restrict__ K0, double *__restrict__ K0T,
                                 double *__restrict__ MK, double *__restrict__ c0, int *__restrict__ asym)
{
    const int n = KP * KP;
    // asym != 0 when M differs from its transpose (asym was zeroed by the caller)
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < K * K; e += gridDim.x * blockDim.x) {
        const int i = e / K, j = e - i * K;
        if (i < j && M[i * K + j] != M[j * K + i]) *asym = 1;
    }
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
        const int i = e / KP, j = e - i * KP;
        double k0 = 0.0, mk = 0.0;
        if (i < K && j < K) {
            const double m = M[i * K + j];
            k0 = exp(-m / reg);
            mk = m * k0;
        }
        K0[i * KP + j] = k0;
        K0T[j * KP + i] = k0;
        MK[i * KP + j] = mk;
    }
    // c0_j = sum_i K0_ij / K: one warp per column, the exps in parallel (a serial loop of K double-precision
    // exps per thread made this the longest part of the kernel)
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int j = warp; j < KP; j += nwarps) {
        double s = 0.0;
        const double u0 = 1.0 / K;
        if (j < K)
            for (int i = lane; i < K; i += 32) s += exp(-M[i * K + j] / reg) * u0;
        s = warp_sum_d(s);
        if (lane == 0) c0[j] = s;
    }
}

__device__ __forceinline__ void dmma884(double &c0, double &c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// swizzled matrix addressing: column ^ 4 * (row % 4).  An A-fragment load reads rows 4*ks + t
// (t = 0..3) at columns 8*m + g; 64-bit shared loads are served per half-warp (g = 0..3 / 4..7), and
// with this swizzle the four rows of a half-warp fall into four different 8-bank groups: 2
// wavefronts per load, the minimum (an 8-column swizzle on odd rows gave 4).
__device__ __forceinline__ int swz(int row, int col) { return col ^ ((row & 3) << 2); }

// KP: storage extent (row stride of K0, panel rows; 16, 32, 48 or 64).  KC <= KP: compute extent, the
// multiple of 8 that covers K -- the DMMA tiles beyond it would only multiply zeros (K = 40: 25 instead
// of 36 tile products per k-step pair).
template <int KP, int KC, bool FULL, bool SYM>
__global__ void __launch_bounds__(SKB_WARPS * 32, 1)
sinkhorn_batched_kernel(const double *__restrict__ props, int K, SkParams prm, PairMap pm, int slot_cap, int warp_cap,
                        SkSetup s, double *__restrict__ scratch,  // [gridDim * WARPS * 8][2][KP] rea / reb
                        SkTail tail, unsigned long long *__restrict__ counter, double *__restrict__ out,
                        int *__restrict__ iters_out, int *__restrict__ abs_out, int *__restrict__ status_out,
                        long long *__restrict__ redo_list, unsigned long long *__restrict__ n_redo)
{
    const SkOut res{out, iters_out, abs_out, status_out, redo_list, n_redo};
    // the symmetric and the general variant are both enqueued; the setup kernel's asymmetry flag decides on
    // the device which one runs (no host read-back in a Sinkhorn call)
    if ((*s.asym != 0) == SYM) return;
    constexpr int MT = KC / 8;   // accumulator row tiles
    constexpr int KS = KC / 4;   // k-steps of 4
    constexpr int PS = SKB_SPW;  // panel row stride (doubles): 64-byte rows, conflict-free as they are
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // symmetric cost (always so in PILOT: squareform(pdist)): K0^T == K0, and the second matrix slot
    // holds M o K0 for the final cost instead; otherwise it holds K0^T and M o K0 is read from L2
    constexpr bool sym = SYM;
    double *sK0 = reinterpret_cast<double *>(smem_raw);  // [i][swz(i, j)]
    double *sSecond = sK0 + KP * KP;
    double *sK0T = sym ? sK0 : sSecond;                  // [j][swz(j, i)]
    double *sc0 = sSecond + KP * KP;
    double *sUV = sc0 + KP;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double *U = sUV + (size_t)warp * 2 * KP * PS;  // U[row][slot], then V
    double *V = U + KP * PS;
    // small K (latency-bound batches): the marginals a, b of the warp's 8 slots live in shared memory
    constexpr bool STAGE_AB = KP <= 32;
    double *sA = sUV + (size_t)SKB_WARPS * 2 * KP * PS + (size_t)warp * 2 * SKB_SPW * KP;  // [slot][KP], then b
    double *sB = sA + SKB_SPW * KP;
    for (int e = threadIdx.x; e < KP * KP; e += blockDim.x) {
        const int r = e / KP, c = e - r * KP;
        sK0[r * KP + swz(r, c)] = s.K0[e];
        if (sym) sSecond[e] = s.MK[e];                   // plain [i][j]
        else sSecond[r * KP + swz(r, c)] = s.K0T[e];
    }
    for (int e = threadIdx.x; e < KP; e += blockDim.x) sc0[e] = s.c0[e];
    __syncthreads();
    if (warp >= warp_cap) return;  // small batches: fewer warps per scheduler = shorter iteration latency

    // C-fragment ownership: lane (g, t) holds rows {8m + g} of the slots {2t, 2t + 1}
    const int g = lane >> 2, t = lane & 3;
    const unsigned gmask = 0x11111111u << t;  // the 8 lanes that share my 2 slots
    const int tsw = (t & 2) << 2, gsw = g ^ ((t & 1) << 2);             // K0 fragment rows 4*ks + t: swizzle 4 * t
    double *wscr = scratch + ((size_t)(blockIdx.x * SKB_WARPS + warp) * SKB_SPW) * 2 * KP;
    double *rea0 = wscr + (size_t)(2 * t) * 2 * KP;  // slot 2t: rea, then reb; slot 2t+1 follows
    const double invK = 1.0 / K;
    double *Uc = U + g * PS + 2 * t;  // my first element of U; rows advance by 8 * PS
    double *Vc = V + g * PS + 2 * t;

    // per-slot state (h = 0, 1), replicated in the 8 lanes of the group
    long long sl[2];
    const double *pa[2], *pb[2];
    int s_ii[2], s_abs[2];
    bool s_act[2], s_hasabs[2], s_pend[2], s_force[2], s_fresh[2], s_bad[2];

#define ROW_OK(r) (FULL || (r) < K)
#define SKB_ASSIGN(h, w)                                                                    \
    do {                                                                                    \
        sl[h] = (long long)(w);                                                             \
        s_act[h] = (w) != ~0ULL && (long long)(w) < pm.n_local;                             \
        int si_ = 0, sj_ = 0;                                                               \
        if (s_act[h]) global_to_ij(pm, local_to_global(pm, sl[h]), si_, sj_);               \
        pa[h] = props + (long long)si_ * K + g;                                             \
        pb[h] = props + (long long)sj_ * K + g;                                             \
        s_ii[h] = 0; s_abs[h] = 0; s_hasabs[h] = false; s_pend[h] = false; s_force[h] = false; \
        s_fresh[h] = true; s_bad[h] = false;                                                \
        _Pragma("unroll") for (int m = 0; m < MT; ++m) {                                    \
            const bool rok = s_act[h] && ROW_OK(8 * m + g);                                 \
            const double v0 = rok ? invK : 0.0;                                             \
            Uc[8 * m * PS + h] = v0;                                                        \
            Vc[8 * m * PS + h] = v0;                                                        \
            if (STAGE_AB) {                                                                 \
                sA[(2 * t + h) * KP + 8 * m + g] = rok ? __ldg(pa[h] + 8 * m) : 0.0;        \
                sB[(2 * t + h) * KP + 8 * m + g] = rok ? __ldg(pb[h] + 8 * m) : 0.0;        \
            }                                                                               \
        }                                                                                   \
    } while (0)

    // initial fill
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        unsigned long long w = ~0ULL;
        if (g == 0 && h < slot_cap) w = atomicAdd(counter, 1ULL);
        w = __shfl_sync(gmask, w, t);
        SKB_ASSIGN(h, w);
    }
    __syncwarp();

    for (;;) {
        if (!__any_sync(0xffffffffu, s_act[0] || s_act[1])) break;

        double acc[MT][2];
        double num[MT][2];
        // ======================= phase A: T = K0^T Ut =======================
#pragma unroll
        for (int m = 0; m < MT; ++m) { acc[m][0] = 0.0; acc[m][1] = 0.0; }
#pragma unroll 2
        for (int ks = 0; ks < KS; ++ks) {
            const int kr = 4 * ks + t;
            const double b0 = U[kr * PS + g];
            const double *arow = sK0 + kr * KP + gsw;
#pragma unroll
            for (int m = 0; m < MT; ++m) dmma884(acc[m][0], acc[m][1], arow[(8 * m) ^ tsw], b0);
        }
        // numerators of the v-update: b of my two slots
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int m = 0; m < MT; ++m)
                num[m][h] = STAGE_AB ? sB[(2 * t + h) * KP + 8 * m + g]
                                     : ((s_act[h] && ROW_OK(8 * m + g)) ? __ldg(pb[h] + 8 * m) : 0.0);

        // ---- resolve the pending convergence check / iteration cap of the previous iteration ----
        bool stop[2];
        int stop_status[2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            stop[h] = false; stop_status[h] = PILOT_ST_MAXITER;
            if (s_act[h] && !s_fresh[h]) {
                if (s_bad[h]) {
                    stop[h] = true; stop_status[h] = -1;  // handed to the reference-form kernel
                } else {
                    bool conv = false;
                    if (s_pend[h]) {
                        double e2 = 0.0;
#pragma unroll
                        for (int m = 0; m < MT; ++m)
                            if (ROW_OK(8 * m + g)) {
                                const double d = fma(Vc[8 * m * PS + h], acc[m][h], -num[m][h]);
                                e2 = fma(d, d, e2);
                            }
                        e2 += __shfl_xor_sync(gmask, e2, 4);
                        e2 += __shfl_xor_sync(gmask, e2, 8);
                        e2 += __shfl_xor_sync(gmask, e2, 16);
                        conv = sqrt(e2) <= prm.stop_thr;
                    }
                    if (conv) { stop[h] = true; stop_status[h] = PILOT_ST_CONVERGED; }
                    else if (s_force[h]) { stop[h] = true; stop_status[h] = PILOT_ST_MAXITER; }
                }
            }
        }
        // ---- warp-cooperative finalisation + refill of the stopped slots ----
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            unsigned mball = __ballot_sync(0xffffffffu, stop[h]) & 0xfu;  // one bit per group (lanes 0..3)
            while (mball) {
                const int tt = __ffs(mball) - 1;  // group id == its t
                mball &= mball - 1;
                const int col = 2 * tt + h;
                const int stt = __shfl_sync(0xffffffffu, stop_status[h], tt);
                double cost = 0.0;
                if (stt >= 0) {
                    // cost = sum_j Vt_j * sum_i (M o K0)_ij Ut_i ; lane = column j
                    const double *mk = sym ? sSecond : s.MK;
                    for (int j = lane; j < KC; j += 32) {  // panel rows >= KC are never written
                        double w0 = 0.0, w1 = 0.0;
                        for (int i = 0; i + 1 < K; i += 2) {
                            w0 = fma(mk[i * KP + j], U[i * PS + col], w0);
                            w1 = fma(mk[(i + 1) * KP + j], U[(i + 1) * PS + col], w1);
                        }
                        if (K & 1) w0 = fma(mk[(K - 1) * KP + j], U[(K - 1) * PS + col], w0);
                        cost = fma(V[j * PS + col], w0 + w1, cost);
                    }
                    cost = warp_sum_d(cost);
                }
                unsigned long long w = 0;
                if (lane == 0) w = atomicAdd(counter, 1ULL);
                w = __shfl_sync(0xffffffffu, w, 0);
                const bool mine = t == tt;
                __syncwarp();  // every lane has read the slot's U, V columns before its owners refill them
                if (mine && g == 0) sk_store(res, sl[h], stt, cost, s_ii[h], s_abs[h]);
                if (mine) {
                    SKB_ASSIGN(h, w);
#pragma unroll
                    for (int m = 0; m < MT; ++m)
                        num[m][h] = (s_act[h] && ROW_OK(8 * m + g)) ? __ldg(pb[h] + 8 * m) : 0.0;
                }
            }
        }
        __syncwarp();

        // ---- tail hand-over: the pool is empty (some slot could not be refilled) and this warp is
        // down to a few problems -- a DMMA panel at 1/8 .. 2/8 occupancy costs the stragglers ~6 us per
        // iteration; the warp-form tail kernel continues them at ~0.5 us (state is clean here: the
        // pending check / cap of every surviving slot has just been resolved) ----
        if (tail.rec) {
            const unsigned a0 = __ballot_sync(0xffffffffu, s_act[0]) & 0xfu;  // lanes 0..3: g == 0, t = 0..3
            const unsigned a1 = __ballot_sync(0xffffffffu, s_act[1]) & 0xfu;
            const int nact = __popc(a0) + __popc(a1);
            if (nact > 0 && nact < SKB_SPW && nact <= tail.evict_max) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    unsigned mb = h ? a1 : a0;
                    while (mb) {
                        const int tt = __ffs(mb) - 1;
                        mb &= mb - 1;
                        const int col = 2 * tt + h;
                        unsigned long long slot = 0;
                        if (lane == 0) slot = atomicAdd(tail.n_tail, 1ULL);
                        slot = __shfl_sync(0xffffffffu, slot, 0);
                        double *dst = tail.uv + slot * 2 * KP;
                        for (int r = lane; r < KC; r += 32) {
                            dst[r] = U[r * PS + col];
                            dst[KP + r] = V[r * PS + col];
                        }
                        if (t == tt && g == 0) {
                            SkTailRec rec;
                            rec.prob = sl[h]; rec.ii = s_ii[h]; rec.nabs = s_abs[h]; rec.hasabs = s_hasabs[h] ? 1 : 0;
                            rec.sslot = (blockIdx.x * SKB_WARPS + warp) * SKB_SPW + col;
                            tail.rec[slot] = rec;
                        }
                    }
                }
                break;
            }
        }

        // ---- v-update: Vt = b / T (my two slots are adjacent: one 128-bit store per row) ----
        long long mxv[2] = {0, 0};
        if (s_act[0] || s_act[1]) {
#pragma unroll
            for (int m = 0; m < MT; ++m) {
                const int row = 8 * m + g;
                double vv[2] = {0.0, 0.0};
                if (ROW_OK(row)) {
#pragma unroll
                    for (int h = 0; h < 2; ++h)
                        if (s_act[h]) {
                            const double tv = s_fresh[h] ? sc0[row] : acc[m][h];
                            vv[h] = sk_div(num[m][h], tv);
                            const double uu = s_hasabs[h] ? vv[h] * rea0[(2 * h + 1) * KP + row] : vv[h];
                            mxv[h] = max(mxv[h], sk_abs_bits(uu));
                        }
                }
                *reinterpret_cast<double2 *>(Vc + 8 * m * PS) = make_double2(vv[0], vv[1]);
            }
        }
        __syncwarp();

        // ======================= phase B: S = K0 Vt =======================
#pragma unroll
        for (int m = 0; m < MT; ++m) { acc[m][0] = 0.0; acc[m][1] = 0.0; }
#pragma unroll 2
        for (int ks = 0; ks < KS; ++ks) {
            const int kr = 4 * ks + t;
            const double b0 = V[kr * PS + g];
            const double *arow = sK0T + kr * KP + gsw;
#pragma unroll
            for (int m = 0; m < MT; ++m) dmma884(acc[m][0], acc[m][1], arow[(8 * m) ^ tsw], b0);
        }
        // ---- u-update: Ut = a / S, then the per-slot service (absorption, counters) ----
        if (s_act[0] || s_act[1]) {
#pragma unroll
            for (int h = 0; h < 2; ++h)
#pragma unroll
                for (int m = 0; m < MT; ++m)
                    num[m][h] = STAGE_AB ? sA[(2 * t + h) * KP + 8 * m + g]
                                         : ((s_act[h] && ROW_OK(8 * m + g)) ? __ldg(pa[h] + 8 * m) : 0.0);
            double un[MT][2];
            long long mxu[2] = {0, 0};
#pragma unroll
            for (int h = 0; h < 2; ++h)
#pragma unroll
                for (int m = 0; m < MT; ++m) {
                    const int row = 8 * m + g;
                    un[m][h] = 0.0;
                    if (s_act[h] && ROW_OK(row)) {
                        un[m][h] = sk_div(num[m][h], acc[m][h]);
                        const double uu = s_hasabs[h] ? un[m][h] * rea0[(2 * h) * KP + row] : un[m][h];
                        mxu[h] = max(mxu[h], sk_abs_bits(uu));
                    }
                }
            bool absorb[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                long long mx = max(mxu[h], mxv[h]);
#pragma unroll
                for (int o = 4; o < 32; o <<= 1) mx = max(mx, __shfl_xor_sync(gmask, mx, o));
                const bool bad = mx >= SK_NONFINITE_BITS;  // NaN or Inf anywhere in u, v
                absorb[h] = s_act[h] && !bad && mx > __double_as_longlong(prm.tau);
                if (s_act[h]) {
                    s_bad[h] = bad;
                    s_pend[h] = (s_ii[h] % prm.check_every) == 0;
                    ++s_ii[h];
                    s_force[h] = s_ii[h] >= prm.num_iter_max;
                    s_fresh[h] = false;
                }
            }
            if (absorb[0] || absorb[1]) {
                // u = v = 1/K in POT == divide the scaled iterates by K; remember 1/ut, 1/vt
                int rb[2] = {0, 0};
#pragma unroll
                for (int m = 0; m < MT; ++m) {
                    const int row = 8 * m + g;
                    double2 vo = *reinterpret_cast<double2 *>(Vc + 8 * m * PS);
                    if (ROW_OK(row)) {
#pragma unroll
                        for (int h = 0; h < 2; ++h)
                            if (absorb[h]) {
                                double &vref = h ? vo.y : vo.x;
                                rea0[(2 * h) * KP + row] = 1.0 / un[m][h];
                                rea0[(2 * h + 1) * KP + row] = 1.0 / vref;
                                // keep e^{+-alpha/reg} comfortably inside the FP64 range (spelled out here: through
                                // sk_out_of_range the KP = 48, 64 panels take a register or spill more)
                                rb[h] |= !(un[m][h] > 1e-250 && un[m][h] < 1e250 && vref > 1e-250 && vref < 1e250);
                                un[m][h] *= invK;
                                vref *= invK;
                            }
                    }
                    *reinterpret_cast<double2 *>(Vc + 8 * m * PS) = vo;
                }
#pragma unroll
                for (int h = 0; h < 2; ++h)
                    if (absorb[h]) {
                        int r = rb[h];
                        r |= __shfl_xor_sync(gmask, r, 4);
                        r |= __shfl_xor_sync(gmask, r, 8);
                        r |= __shfl_xor_sync(gmask, r, 16);
                        s_hasabs[h] = true;
                        ++s_abs[h];
                        s_bad[h] = s_bad[h] || r;
                    }
            }
#pragma unroll
            for (int m = 0; m < MT; ++m)
                *reinterpret_cast<double2 *>(Uc + 8 * m * PS) = make_double2(un[m][0], un[m][1]);
        }
        __syncwarp();
    }
#undef SKB_ASSIGN
#undef ROW_OK
}

size_t skb_setup_bytes(int KP) { return sizeof(double) * ((size_t)3 * KP * KP + KP + 32); }
// the flag is an int in the room behind c0
SkSetup sk_setup_view(const double *setup, int KP)
{
    const size_t n = (size_t)KP * KP;
    return {setup, setup + n, setup + 2 * n, setup + 3 * n, reinterpret_cast<const int *>(setup + 3 * n + KP)};
}
size_t skb_smem_bytes(int KP)
{
    const size_t stage = KP <= 32 ? (size_t)SKB_WARPS * 2 * SKB_SPW * KP : 0;  // a, b of every slot
    return sizeof(double) * ((size_t)2 * KP * KP + KP + (size_t)SKB_WARPS * 2 * KP * SKB_SPW + stage);
}
size_t skb_scratch_bytes(int KP, int ctas)
{
    return sizeof(double) * (size_t)ctas * SKB_WARPS * SKB_SPW * 2 * KP;
}
// padded problem size: the DMMA tiles need a multiple of 8, the work grows with KP^2
int skb_pad(int K) { return K <= 16 ? 16 : (K <= 32 ? 32 : (K <= 48 ? 48 : 64)); }
int sk_setup_extent(int K) { return K <= 64 ? skb_pad(K) : (K + 7) / 8 * 8; }
int skb_slots_per_cta() { return SKB_WARPS * SKB_SPW; }
int skb_slots_per_warp() { return SKB_SPW; }
int skb_warps() { return SKB_WARPS; }

template <int KP, int KC, bool FULL, bool SYM>
static int skb_launch_t(const double *props, int K, const SkParams &prm, const PairMap &pm, int slot_cap, int warp_cap,
                        const SkSetup &s, double *scratch, const SkTail &tail, int ctas, const SkOut &res,
                        unsigned long long *counter, cudaStream_t st)
{
    const size_t smem = skb_smem_bytes(KP);
    PILOT_CUDA(cudaFuncSetAttribute(sinkhorn_batched_kernel<KP, KC, FULL, SYM>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)smem));
    sinkhorn_batched_kernel<KP, KC, FULL, SYM><<<ctas, SKB_WARPS * 32, smem, st>>>(
        props, K, prm, pm, slot_cap, warp_cap, s, scratch, tail, counter, res.out, res.iters, res.absn, res.status,
        res.redo, res.n_redo);
    PILOT_LAUNCH_CHECK();
    return 0;
}

// fills the buffer sk_setup_view describes
int skb_setup(const double *cost, int K, const SkParams &prm, double *setup, cudaStream_t st)
{
    const int KP = sk_setup_extent(K);
    const SkSetup s = sk_setup_view(setup, KP);
    int *asym = const_cast<int *>(s.asym);
    PILOT_CUDA(cudaMemsetAsync(asym, 0, sizeof(int), st));
    skb_setup_kernel<<<8, 256, 0, st>>>(cost, K, KP, prm.reg, setup, const_cast<double *>(s.K0T),
                                        const_cast<double *>(s.MK), const_cast<double *>(s.c0), asym);
    PILOT_LAUNCH_CHECK();
    return 0;
}

// `setup` must already hold the output of skb_setup
int skb_launch(const double *props, int K, const SkParams &prm, const PairMap &pm, const double *setup,
               double *scratch, int ctas, int slot_cap, int warp_cap, bool symmetric, const SkTail &tail,
               const SkOut &res, unsigned long long *counter, cudaStream_t st)
{
    const int KP = skb_pad(K);
    const SkSetup s = sk_setup_view(setup, KP);
    // FULL: K fills the compute extent KC, no row masks
#define SKB_GO(KPV, KCV)                                                                                          \
    return (symmetric ? (K == KCV ? skb_launch_t<KPV, KCV, true, true> : skb_launch_t<KPV, KCV, false, true>)     \
                      : (K == KCV ? skb_launch_t<KPV, KCV, true, false> : skb_launch_t<KPV, KCV, false, false>))( \
        props, K, prm, pm, slot_cap, warp_cap, s, scratch, tail, ctas, res, counter, st)
    if (KP == 16) SKB_GO(16, 16);
    if (KP == 32) { if (K <= 24) SKB_GO(32, 24); SKB_GO(32, 32); }
    if (KP == 48) { if (K <= 40) SKB_GO(48, 40); SKB_GO(48, 48); }
    if (K <= 56) SKB_GO(64, 56);
    SKB_GO(64, 64);
#undef SKB_GO
}

}  // namespace pilot
