// Kernel (4): all-pairs exact EMD.  Replaces the loop over ot.emd2(a_i, a_j, cost)
// (reference pilotpy/tools/Trajectory.py:507-511; POT emd_c / LEMON network simplex).
//
// One warp per problem, persistent warps pulling problems from a global counter, ONE CTA of 32 warps
// per SM.  The kernel is instruction-issue bound (integer + shared-memory work, hardly any FP64), so
// every design choice below is about warp instructions per problem (round 1: 67 K, now ~20 K at K=64):
//   * basis tree = parent|size (packed u16) + flow[] + pi[] + a SUBTREE BITMASK per node
//     (<=128 nodes -> 4 x 32-bit words, stored word-major so that the owner lanes read conflict free;
//     node x = slot*32 + lane is owned by `lane`)
//   * start basis:  diagonal arcs (i,i) with min(a_i,b_i), then the LEAST-COST METHOD on the residual
//                   (surplus rows x deficit columns): the K(K-1) off-diagonal arcs are sorted ONCE per
//                   launch (the cost matrix is shared by all problems); a problem scans that list 32
//                   arcs at a time against two open-row/open-column bitmasks.  The node that an arc
//                   exhausts becomes the child of the other end, so parents close after their
//                   children and the subtree masks accumulate in the same sweep.  No artificial arcs,
//                   ~45 pivots to the optimum at K=64 (greedy north-west corner of round 1: 84; POT's
//                   artificial-root start: 331)
//   * pricing:      candidate list.  A major pass scans `scan_rows` rows x all columns (lane = column)
//                   and keeps the best row per column in registers; minor passes re-price only those
//                   <=64 arcs (2 per lane) after each pivot until none is eligible
//   * join / cycle: node y is on the i-side of the cycle iff sub[y] has i but not j (one AND per node,
//                   no walk); the ~7 cycle nodes are ballot-compacted so ONE lane handles ONE cycle node
//   * ratio test:   REDUX min over the decreasing arcs, Cunningham tie-break by cycle order
//   * re-hanging:   stem nodes find their stem child through a scatter, then sub[] of stem /
//                   ancestors are fixed with AND/OR of the cut mask
//   * potentials:   the cut subtree IS a bitmask -> one predicated add per node; the column
//                   potentials live in registers
//   * cycles longer than 32 nodes take a loop-based __noinline__ path (rare)
// Any exact solver returns the same optimum (SURVEY.md Appendix B.3); parity with the oracle is <1e-12
// relative in FP64.  precision = PILOT_F32 runs the same algorithm on float costs/flows/potentials
// (north_star's 1e-4 tier).
#include <stdlib.h>
#include "common.cuh"

namespace pilot {

constexpr int EMD_WARPS = 32;
constexpr unsigned FULLMASK = 0xffffffffu;

template <typename T> struct EmdReal;
template <> struct EmdReal<double> {
    __device__ static double eps() { return 8.8817841970012523e-15; }  // 40 ulp
    __device__ static double ninf() { return __longlong_as_double((long long)0xfff0000000000000ULL); }
};
template <> struct EmdReal<float> {
    __device__ static float eps() { return 4.76837158e-6f; }  // 40 ulp
    __device__ static float ninf() { return __uint_as_float(0xff800000u); }
};

// arg-max of a value >= 0 over the warp (0 means "no candidate"): winning lane or -1
__device__ __forceinline__ int warp_argmax_pos(double v, double &vmax)
{
    const unsigned long long kb = (unsigned long long)__double_as_longlong(v);
    const unsigned khi = (unsigned)(kb >> 32), klo = (unsigned)kb;
    const unsigned mhi = __reduce_max_sync(FULLMASK, khi);
    const unsigned mlo = __reduce_max_sync(FULLMASK, khi == mhi ? klo : 0u);
    if ((mhi | mlo) == 0u) return -1;
    vmax = __longlong_as_double((long long)(((unsigned long long)mhi << 32) | mlo));
    return __ffs(__ballot_sync(FULLMASK, khi == mhi && klo == mlo)) - 1;
}
__device__ __forceinline__ int warp_argmax_pos(float v, float &vmax)
{
    const unsigned kb = __float_as_uint(v);
    const unsigned m = __reduce_max_sync(FULLMASK, kb);
    if (m == 0u) return -1;
    vmax = __uint_as_float(m);
    return __ffs(__ballot_sync(FULLMASK, kb == m)) - 1;
}
// min of a value >= 0 over the lanes with `on`; `tie` = this lane holds the minimum
__device__ __forceinline__ double warp_min_pos(double v, bool on, bool &tie)
{
    const unsigned long long kb = on ? (unsigned long long)__double_as_longlong(v) : ~0ULL;
    const unsigned khi = (unsigned)(kb >> 32), klo = (unsigned)kb;
    const unsigned m1 = __reduce_min_sync(FULLMASK, khi);
    const unsigned m2 = __reduce_min_sync(FULLMASK, khi == m1 ? klo : 0xffffffffu);
    tie = on && khi == m1 && klo == m2;
    return __longlong_as_double((long long)(((unsigned long long)m1 << 32) | m2));
}
__device__ __forceinline__ float warp_min_pos(float v, bool on, bool &tie)
{
    const unsigned kb = on ? __float_as_uint(v) : 0xffffffffu;
    const unsigned m = __reduce_min_sync(FULLMASK, kb);
    tie = on && kb == m;
    return __uint_as_float(m);
}

template <int NW, typename T> struct EmdWarp {
    static constexpr int KP = 32 * NW;  // padded types per side
    static constexpr int N = 2 * KP;    // nodes: rows 0..KP-1, columns KP..2KP-1
    static constexpr int NS = 2 * NW;   // slots per lane == mask words
    static constexpr int SUBLD = N + 1; // odd word stride: the NS words of one node fall into different banks
    unsigned sub[NS][SUBLD];            // subtree masks, word-major
    T flow[N];                          // flow on the arc (node, parent)
    T pi[N];                            // potentials; residual supplies/demands while the start basis is built
    unsigned short info[N];             // parent (low byte, 255 = none) | subtree size << 8
    unsigned char tmpc[N];              // closing order (start basis) / stem-child scatter (pivots)
    unsigned char clist[N];             // compacted cycle nodes (bit 7: j-side)
};

// open-row / open-column sets of the start basis: one 64-bit mask each (warp-uniform)
__device__ __forceinline__ unsigned bit64(unsigned long long m, unsigned x) { return (unsigned)(m >> x) & 1u; }
__device__ __forceinline__ int lowest64(unsigned long long m) { return __ffsll((long long)m) - 1; }

// ---- K(K-1) off-diagonal arcs in ascending cost order (ties and 2^-40-relative near-ties by index) ----
__global__ void __launch_bounds__(1024) emd_sort_arcs_kernel(const double *__restrict__ cost, int K, int n_pad,
                                                            unsigned short *__restrict__ arcs)
{
    __shared__ unsigned long long key[4096];
    const int n = K * K;
    int np2 = 32;
    while (np2 < n) np2 <<= 1;
    for (int t = threadIdx.x; t < np2; t += blockDim.x) {
        unsigned long long k = ~0ULL;
        if (t < n) {
            const int i = t / K, j = t - i * K;
            if (i != j) {
                const unsigned long long u = (unsigned long long)__double_as_longlong(cost[t]);
                const unsigned long long o = (u >> 63) ? ~u : (u | 0x8000000000000000ULL);  // order preserving
                k = (o & ~0xfffULL) | (unsigned long long)t;
                if (k == ~0ULL) k -= 0x1000ULL;
            }
        }
        key[t] = k;
    }
    __syncthreads();
    for (int size = 2; size <= np2; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = threadIdx.x; t < np2; t += blockDim.x) {
                const int p = t ^ stride;
                if (p > t) {
                    const unsigned long long a = key[t], b = key[p];
                    const bool up = (t & size) == 0;
                    if ((a > b) == up) { key[t] = b; key[p] = a; }
                }
            }
            __syncthreads();
        }
    const int n_arcs = K * (K - 1);
    for (int t = threadIdx.x; t < n_pad; t += blockDim.x) {
        unsigned short e = 0x3f3fu;  // (63, 63): row 63 and column 63 are never open together (a diagonal arc)
        if (t < n_arcs) {
            const int idx = (int)(key[t] & 0xfffULL);
            const int i = idx / K, j = idx - i * K;
            e = (unsigned short)((i << 8) | j);
        }
        arcs[t] = e;
    }
}

// ---- pivot for cycles longer than the one-lane-per-node path handles: loops over 32-node rounds, the
// stem is re-hung by a serial walk (every lane executes it redundantly).  Rare; kept out of line so that
// its registers do not burden the main loop.  Column potentials are read/written in shared memory here.
template <int NW, typename T>
__device__ __noinline__ int emd_pivot_general(EmdWarp<NW, T> *sw, int ncyc, int ei, int jn, T erc, int lane)
{
    using W = EmdWarp<NW, T>;
    constexpr int KP = W::KP, NS = W::NS;
    // ratio test: min flow over the decreasing arcs, ties -> last in cycle order (Cunningham)
    T bf = (T)0;
    unsigned bod = 0;
    int by = 0, bsz = 0;
    bool bhas = false;
    for (int t = lane; t < ncyc; t += 32) {
        const unsigned ye = sw->clist[t];
        const int y = ye & 0x7f;
        const bool onJ = (ye >> 7) != 0;
        if (onJ == (y >= KP)) {
            const T f = sw->flow[y];
            const int sz = sw->info[y] >> 8;
            const unsigned od = onJ ? (unsigned)(256 + sz) : (unsigned)(256 - sz);
            if (!bhas || f < bf || (f == bf && od > bod)) { bf = f; bod = od; by = y; bsz = sz; bhas = true; }
        }
    }
    bool tie;
    const T delta = warp_min_pos(bf, bhas, tie);
    const unsigned m3 = __reduce_max_sync(FULLMASK, tie ? bod : 0u);
    if (m3 == 0u) return PILOT_ST_UNBOUNDED;
    const int wl = __ffs(__ballot_sync(FULLMASK, tie && bod == m3)) - 1;
    const int u_out = __shfl_sync(FULLMASK, by, wl);
    const int pc_out = __shfl_sync(FULLMASK, bsz, wl);
    const bool sideJ = m3 > 256u;
    const int u_in = sideJ ? jn : ei, v_in = sideJ ? ei : jn;
    const T sigma = sideJ ? erc : -erc;
    unsigned T2[NS];
#pragma unroll
    for (int w = 0; w < NS; ++w) T2[w] = sw->sub[w][u_out];
    // flows round the cycle; nodes off the stem gain / lose the cut subtree
    for (int t = lane; t < ncyc; t += 32) {
        const unsigned ye = sw->clist[t];
        const int y = ye & 0x7f;
        const bool onJ = (ye >> 7) != 0;
        const bool dec = onJ == (y >= KP);
        const T f = sw->flow[y];
        sw->flow[y] = dec ? f - delta : f + delta;
        const unsigned inf_ = sw->info[y];
        const int sz = inf_ >> 8;
        const bool same = onJ == sideJ;
        if (same && sz <= pc_out) continue;  // stem: below
        sw->info[y] = (unsigned short)((inf_ & 0xffu) | ((unsigned)(same ? sz - pc_out : sz + pc_out) << 8));
#pragma unroll
        for (int w = 0; w < NS; ++w) {
            const unsigned o = sw->sub[w][y];
            sw->sub[w][y] = same ? (o & ~T2[w]) : (o | T2[w]);
        }
    }
    __syncwarp();
    // stem u_in .. u_out: reverse the parent pointers
    {
        int y = u_in, npar = v_in, nsz = pc_out;
        T nflow = delta;
        unsigned nsub[NS];
#pragma unroll
        for (int w = 0; w < NS; ++w) nsub[w] = T2[w];
        for (int guard = 0; guard < W::N; ++guard) {
            const unsigned oinf = sw->info[y];
            const T oflow = sw->flow[y];
            unsigned osub[NS];
#pragma unroll
            for (int w = 0; w < NS; ++w) osub[w] = sw->sub[w][y];
            __syncwarp();
            sw->info[y] = (unsigned short)((unsigned)npar | ((unsigned)nsz << 8));
            sw->flow[y] = nflow;
#pragma unroll
            for (int w = 0; w < NS; ++w) sw->sub[w][y] = nsub[w];
            if (y == u_out) break;
            npar = y;
            nflow = oflow;
            nsz = pc_out - (int)(oinf >> 8);
#pragma unroll
            for (int w = 0; w < NS; ++w) nsub[w] = T2[w] & ~osub[w];
            y = oinf & 0xff;
        }
    }
    // potentials of the re-hung subtree
#pragma unroll
    for (int sl = 0; sl < NS; ++sl)
        if ((T2[sl] >> lane) & 1u) sw->pi[sl * 32 + lane] += sigma;
    __syncwarp();
    return PILOT_ST_CONVERGED;
}

// PLAN (double only): problems from the pair list of `plan`, and each problem's plan written from its basis
template <int NW, typename T, bool PLAN = false>
__global__ void __launch_bounds__(EMD_WARPS * 32, 1)
emd_pairs_kernel(const double *__restrict__ props, int K, const double *__restrict__ cost,
                 const unsigned short *__restrict__ arcs, int n_arcs_pad, PairMap pm, long long max_pivots,
                 double *__restrict__ out, int *__restrict__ status, int *__restrict__ pivots_out,
                 unsigned long long *__restrict__ counter, int fast_limit, int scan_rows, PlanArgs<PLAN> plan)
{
    static_assert(!PLAN || sizeof(T) == sizeof(double), "plans are FP64 only");
    using W = EmdWarp<NW, T>;
    constexpr int KP = W::KP, NS = W::NS;
    constexpr int LDM = KP + 1;  // odd row stride
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T *sM = reinterpret_cast<T *>(smem_raw);  // KP x LDM, row-major, zero padded
    unsigned short *sArcs = reinterpret_cast<unsigned short *>(smem_raw + sizeof(T) * KP * LDM);
    W *sw = reinterpret_cast<W *>(smem_raw + sizeof(T) * KP * LDM + sizeof(unsigned short) * n_arcs_pad) +
            (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    const unsigned lt_mask = (1u << lane) - 1u;
    const int wlane = lane & (NS - 1);

    for (int t = threadIdx.x; t < KP * KP; t += blockDim.x) {
        const int i = t / KP, j = t - i * KP;
        sM[i * LDM + j] = (i < K && j < K) ? (T)cost[i * K + j] : (T)0;
    }
    for (int t = threadIdx.x; t < n_arcs_pad; t += blockDim.x) sArcs[t] = arcs[t];
    __syncthreads();

    const T EPS = EmdReal<T>::eps();

    for (;;) {
        unsigned long long l = 0;
        if (lane == 0) l = atomicAdd(counter, 1ULL);
        l = __shfl_sync(FULLMASK, l, 0);
        if ((long long)l >= pm.n_local) break;
        int si_, sj_;
        if constexpr (PLAN) {
            if (!plan_pair(plan, (long long)l, si_, sj_)) {
                double *g = plan.plans + (long long)l * K * K;
                for (int e = lane; e < K * K; e += 32) g[e] = __longlong_as_double(PILOT_NAN_BITS);
                if (lane == 0) {
                    out[l] = __longlong_as_double(PILOT_NAN_BITS);
                    if (status) status[l] = PILOT_ST_NUMERIC;
                }
                continue;
            }
        } else {
            global_to_ij(pm, local_to_global(pm, (long long)l), si_, sj_);
        }
        const double *pa = props + (long long)si_ * K, *pb = props + (long long)sj_ * K;

        // ---------------- load a, b ; emd2's rescale of b ----------------
        T av[NW], bv[NW];
        bool valid[NW];
        {
            double ad[NW], bd[NW], sa = 0.0, sb = 0.0;
#pragma unroll
            for (int c = 0; c < NW; ++c) {
                const int idx = lane + 32 * c;
                valid[c] = idx < K;
                ad[c] = valid[c] ? pa[idx] : 0.0;
                bd[c] = valid[c] ? pb[idx] : 0.0;
                sa += ad[c];
                sb += bd[c];
            }
            sa = warp_sum_d(sa);
            sb = warp_sum_d(sb);
#pragma unroll
            for (int c = 0; c < NW; ++c) {
                av[c] = (T)ad[c];
                bv[c] = (T)__ddiv_rn(__dmul_rn(bd[c], sa), sb);
            }
        }

        // ---------------- start basis, parallel part: the diagonal arcs ----------------
        unsigned long long ro = 0ULL, co = 0ULL;  // open surplus rows / open deficit columns (warp-uniform)
#pragma unroll
        for (int c = 0; c < NW; ++c) {
            const int idx = lane + 32 * c;
            const int r = idx, cn = KP + idx;
            const bool sur = valid[c] && av[c] >= bv[c];
            ro |= (unsigned long long)__ballot_sync(FULLMASK, sur) << (32 * c);
            co |= (unsigned long long)__ballot_sync(FULLMASK, valid[c] && !sur) << (32 * c);
#pragma unroll
            for (int w = 0; w < NS; ++w) { sw->sub[w][r] = 0u; sw->sub[w][cn] = 0u; }
            unsigned short ir = 0x00ffu, ic = 0x00ffu;
            T fr = (T)0, fc = (T)0;
            if (valid[c]) {
                const unsigned bit = 1u << lane;
                if (sur) {  // column idx hangs under row idx (flow b); the row stays open with a - b
                    ic = (unsigned short)(r | 0x100);  fc = bv[c];
                    sw->sub[NW + c][cn] = bit;
                    sw->sub[c][r] = bit; sw->sub[NW + c][r] = bit;
                    ir = 0x02ffu;
                    sw->pi[r] = av[c] - bv[c];
                } else {    // row idx hangs under column idx (flow a); the column stays open with b - a
                    ir = (unsigned short)(cn | 0x100); fr = av[c];
                    sw->sub[c][r] = bit;
                    sw->sub[NW + c][cn] = bit; sw->sub[c][cn] = bit;
                    ic = 0x02ffu;
                    sw->pi[cn] = bv[c] - av[c];
                }
            }
            sw->info[r] = ir; sw->info[cn] = ic;
            sw->flow[r] = fr; sw->flow[cn] = fc;
        }
        __syncwarp();

        // ---------------- start basis, least-cost method on the residual (every lane runs it redundantly:
        // all stores are warp-uniform, so no lane ever reads another lane's value and no barrier is needed) ----
        int nr = __popcll(ro), nc = __popcll(co), n_ord = 0, root = 0;
        int st = PILOT_ST_CONVERGED;
        const bool greedy = nr > 0 && nc > 0;
        if (greedy) {
            for (int base = 0; nr + nc > 1 && base < n_arcs_pad; base += 32) {
                const unsigned e = sArcs[base + lane];
                const unsigned er = e >> 8, ec = e & 0xffu;
                unsigned hits = __ballot_sync(FULLMASK, (bit64(ro, er) & bit64(co, ec)) != 0u);
                while (hits) {
                    const int src = __ffs(hits) - 1;
                    const unsigned ee = __shfl_sync(FULLMASK, e, src);
                    const int i = (int)(ee >> 8), j = (int)(ee & 0xffu);
                    const int xr = i, xc = KP + j;
                    const T ra = sw->pi[xr], rb = sw->pi[xc];
                    const bool close_row = nr == 1 ? false : (nc == 1 ? true : ra <= rb);
                    const T f = ra < rb ? ra : rb;
                    const int x = close_row ? xr : xc, p = close_row ? xc : xr;
                    const T rest = (close_row ? rb : ra) - f;
                    sw->pi[p] = rest > (T)0 ? rest : (T)0;
                    const unsigned ix = sw->info[x], ip = sw->info[p];
                    sw->info[x] = (unsigned short)((ix & 0xff00u) | (unsigned)p);
                    sw->info[p] = (unsigned short)(ip + (ix & 0xff00u));
                    sw->flow[x] = f;
                    sw->sub[wlane][p] |= sw->sub[wlane][x];
                    sw->tmpc[n_ord++] = (unsigned char)x;
                    // the arcs of this chunk that touch the node just closed are stale now
                    if (close_row) { ro &= ~(1ULL << i); --nr; hits &= ~__ballot_sync(FULLMASK, er == (unsigned)i); }
                    else           { co &= ~(1ULL << j); --nc; hits &= ~__ballot_sync(FULLMASK, ec == (unsigned)j); }
                    if (nr + nc <= 1) break;
                }
            }
            if (nr + nc > 1) st = PILOT_ST_NUMERIC;  // cannot happen: every open (row, column) arc is in the list
            root = nr ? lowest64(ro) : KP + lowest64(co);
            // potentials, root first (reverse closing order)
            sw->pi[root] = (T)0;
            for (int t = n_ord - 1; t >= 0; --t) {
                const int x = sw->tmpc[t];
                const int p = sw->info[x] & 0xff;
                if (x < KP) sw->pi[x] = sw->pi[p] - sM[x * LDM + (p - KP)];
                else        sw->pi[x] = sw->pi[p] + sM[p * LDM + (x - KP)];
            }
        } else {
            // a >= b everywhere (or a < b everywhere, only through rounding): every residual is ~0.  Chain the
            // (row, leaf column) pairs with zero-flow arcs row_t -> column_{t-1} (resp. the mirror image)
            const bool rows_open = nr > 0;
            unsigned long long om = rows_open ? ro : co;
            int prev = lowest64(om);
            om &= om - 1;
            if (rows_open) {
                root = prev;
                sw->pi[prev] = (T)0;
                sw->pi[KP + prev] = sM[prev * LDM + prev];
            } else {
                root = KP + prev;
                sw->pi[KP + prev] = (T)0;
                sw->pi[prev] = -sM[prev * LDM + prev];
            }
            for (;;) {
                const int cur = lowest64(om);
                if (cur < 0) break;
                om &= om - 1;
                if (rows_open) {
                    sw->info[cur] = (unsigned short)((sw->info[cur] & 0xff00u) | (unsigned)(KP + prev));
                    sw->flow[cur] = (T)0;
                    sw->pi[cur] = sw->pi[KP + prev] - sM[cur * LDM + prev];
                    sw->pi[KP + cur] = sw->pi[cur] + sM[cur * LDM + cur];
                    sw->tmpc[n_ord++] = (unsigned char)cur;
                } else {
                    sw->info[KP + cur] = (unsigned short)((sw->info[KP + cur] & 0xff00u) | (unsigned)prev);
                    sw->flow[KP + cur] = (T)0;
                    sw->pi[KP + cur] = sw->pi[prev] + sM[prev * LDM + cur];
                    sw->pi[cur] = sw->pi[KP + cur] - sM[cur * LDM + cur];
                    sw->tmpc[n_ord++] = (unsigned char)(KP + cur);
                }
                prev = cur;
            }
            // subtree masks and sizes, leaves first: chain node x = tmpc[t] hangs under the leaf partner of
            // tmpc[t-1] (or of the root), which hangs under tmpc[t-1]
            for (int t = n_ord - 1; t >= 0; --t) {
                const int x = sw->tmpc[t];
                const int p = sw->info[x] & 0xff;      // leaf partner of the previous chain node
                const int pp = sw->info[p] & 0xff;     // the previous chain node itself
                const unsigned add = sw->info[x] & 0xff00u;
                sw->info[p] = (unsigned short)(sw->info[p] + add);
                sw->info[pp] = (unsigned short)(sw->info[pp] + add);
                const unsigned m = sw->sub[wlane][x];
                sw->sub[wlane][p] |= m;
                sw->sub[wlane][pp] |= m;
            }
        }
        __syncwarp();
        if (greedy) {
            // leaf potentials of the diagonal arcs (their parents are final now)
#pragma unroll
            for (int c = 0; c < NW; ++c) {
                const int idx = lane + 32 * c;
                if (valid[c]) {
                    const T m = sM[idx * LDM + idx];
                    if (av[c] >= bv[c]) sw->pi[KP + idx] = sw->pi[idx] + m;
                    else                sw->pi[idx] = sw->pi[KP + idx] - m;
                }
            }
            __syncwarp();
        }

        // ---------------- simplex iterations ----------------
        T pj[NW];
        int cand[NW];
#pragma unroll
        for (int c = 0; c < NW; ++c) {
            pj[c] = valid[c] ? sw->pi[KP + lane + 32 * c] : EmdReal<T>::ninf();
            cand[c] = -1;
        }
        int r0 = 0, since = 0, npiv = 0;
        bool have_cand = false;
        while (st == PILOT_ST_CONVERGED) {
            int ei = -1, ej = 0;
            T erc = (T)0;
            if (have_cand) {
                // ---- minor pass: re-price the stored candidates (one per column) ----
                T best = (T)0;
                int bi = 0, bc = 0;
#pragma unroll
                for (int c = 0; c < NW; ++c) {
                    const int i = cand[c] < 0 ? 0 : cand[c];
                    const T pr = sw->pi[i];
                    const T m = sM[i * LDM + lane + 32 * c];
                    const T rc = (m + pr) - pj[c];
                    const T tol = EPS * ((fabs(pr) + fabs(pj[c])) + fabs(m));
                    if (cand[c] >= 0 && rc < -tol && rc < best) { best = rc; bi = i; bc = c; }
                }
                T vmax;
                const int wl = warp_argmax_pos(fabs(best), vmax);  // best <= 0
                if (wl >= 0) {
                    ei = __shfl_sync(FULLMASK, bi, wl);
                    ej = __shfl_sync(FULLMASK, bc, wl) * 32 + wl;
                    erc = -vmax;
                } else {
                    have_cand = false;
                }
            }
            if (ei < 0) {
                if (since >= K) break;  // every row priced since the last pivot, nothing eligible: optimal
                // ---- major pass: best row per column over the next rows ----
                const int rows = min(scan_rows, K - since);
                T best[NW];
#pragma unroll
                for (int c = 0; c < NW; ++c) { best[c] = (T)0; cand[c] = -1; }
                // rows r0 .. r0+rows-1 (mod K) as at most two runs without a wrap test inside
                int i = r0, left = rows;
                while (left > 0) {
                    const int run = min(left, K - i);
                    const T *mrow = sM + i * LDM + lane;
                    const T *prow = sw->pi + i;
#pragma unroll 4
                    for (int rr = 0; rr < run; ++rr) {
                        const T pr = prow[rr];
#pragma unroll
                        for (int c = 0; c < NW; ++c) {
                            const T rc = (mrow[rr * LDM + 32 * c] + pr) - pj[c];
                            if (rc < best[c]) { best[c] = rc; cand[c] = i + rr; }
                        }
                    }
                    left -= run;
                    i += run;
                    if (i == K) i = 0;
                }
                r0 = i;
                since += rows;
                have_cand = true;
                continue;
            }
            if (++npiv > max_pivots) { st = PILOT_ST_MAXITER; break; }
            since = 0;

            // ---- compact the cycle of (ei -> KP+ej): i-side = has i but not j, j-side = has j but not i ----
            const int jn = KP + ej;
            int ncyc = 0;
            {
                const unsigned *subI = sw->sub[ei >> 5], *subJ = sw->sub[jn >> 5];
                const int shI = ei & 31, shJ = jn & 31;
#pragma unroll
                for (int sl = 0; sl < NS; ++sl) {
                    const int y = sl * 32 + lane;
                    const unsigned hi = (subI[y] >> shI) & 1u, hj = (subJ[y] >> shJ) & 1u;
                    const bool on = hi != hj;
                    const unsigned bal = __ballot_sync(FULLMASK, on);
                    if (on) sw->clist[ncyc + __popc(bal & lt_mask)] = (unsigned char)(y | (hj << 7));
                    ncyc += __popc(bal);
                }
            }
            __syncwarp();
            if (ncyc > fast_limit) {
                // ---------- long cycle: out-of-line path working on shared memory only ----------
#pragma unroll
                for (int c = 0; c < NW; ++c)
                    if (valid[c]) sw->pi[KP + lane + 32 * c] = pj[c];
                __syncwarp();
                const int rc_ = emd_pivot_general<NW, T>(sw, ncyc, ei, jn, erc, lane);
                if (rc_ != PILOT_ST_CONVERGED) { st = rc_; break; }
#pragma unroll
                for (int c = 0; c < NW; ++c)
                    if (valid[c]) pj[c] = sw->pi[KP + lane + 32 * c];
                continue;
            }
            // ---------- one lane per cycle node ----------
            const bool has = lane < ncyc;
            const unsigned ye = has ? sw->clist[lane] : 0u;
            const int y = ye & 0x7f;
            const bool onJ = (ye >> 7) != 0;
            const T f = has ? sw->flow[y] : (T)0;
            const unsigned inf_ = has ? sw->info[y] : 0u;
            const int sz = inf_ >> 8, par = inf_ & 0xff;
            const bool dec = has && (onJ == (y >= KP));  // i-side rows / j-side columns lose flow
            // ratio test: min flow, ties -> last in cycle order (Cunningham)
            bool tie;
            const T delta = warp_min_pos(f, dec, tie);
            const unsigned od = onJ ? (unsigned)(256 + sz) : (unsigned)(256 - sz);
            const unsigned m3 = __reduce_max_sync(FULLMASK, tie ? od : 0u);
            if (m3 == 0u) { st = PILOT_ST_UNBOUNDED; break; }
            const int wl = __ffs(__ballot_sync(FULLMASK, tie && od == m3)) - 1;
            const int u_out = __shfl_sync(FULLMASK, y, wl);
            const int pc_out = __shfl_sync(FULLMASK, sz, wl);
            const bool sideJ = m3 > 256u;
            const int u_in = sideJ ? jn : ei, v_in = sideJ ? ei : jn;
            const T sigma = sideJ ? erc : -erc;
            unsigned T2[NS];
#pragma unroll
            for (int w = 0; w < NS; ++w) T2[w] = sw->sub[w][u_out];
            // phase A: push delta round the cycle; stem children announce themselves
            const bool same = has && (onJ == sideJ);
            const bool stem = same && sz <= pc_out;
            if (has) sw->flow[y] = dec ? f - delta : f + delta;
            if (stem && y != u_out) sw->tmpc[par] = (unsigned char)y;
            __syncwarp();
            // phase B: own subtree; stem nodes fetch their stem child's (updated) flow, old subtree and size
            unsigned nsub[NS];
            unsigned ninfo = 0;
            T nflow = (T)0;
            if (stem) {
                if (y == u_in) {
                    ninfo = (unsigned)v_in | ((unsigned)pc_out << 8);
                    nflow = delta;
#pragma unroll
                    for (int w = 0; w < NS; ++w) nsub[w] = T2[w];
                } else {
                    const int ch = sw->tmpc[y];
                    nflow = sw->flow[ch];
                    ninfo = (unsigned)ch | ((unsigned)(pc_out - (int)(sw->info[ch] >> 8)) << 8);
#pragma unroll
                    for (int w = 0; w < NS; ++w) nsub[w] = T2[w] & ~sw->sub[w][ch];
                }
            } else if (has) {
                // above u_out on its side: loses the cut subtree; the other side (v_in and its ancestors
                // below the join) gains it
                ninfo = (unsigned)par | ((unsigned)(same ? sz - pc_out : sz + pc_out) << 8);
#pragma unroll
                for (int w = 0; w < NS; ++w) {
                    const unsigned o = sw->sub[w][y];
                    nsub[w] = same ? (o & ~T2[w]) : (o | T2[w]);
                }
            }
            __syncwarp();
            // phase C: rewrite parent / size / flow / sub of the cycle nodes
            if (has) {
                sw->info[y] = (unsigned short)ninfo;
                if (stem) sw->flow[y] = nflow;
#pragma unroll
                for (int w = 0; w < NS; ++w) sw->sub[w][y] = nsub[w];
            }
            // potentials of the re-hung subtree (rows in shared memory, columns in registers)
#pragma unroll
            for (int c = 0; c < NW; ++c) {
                if ((T2[c] >> lane) & 1u) sw->pi[c * 32 + lane] += sigma;
                if ((T2[NW + c] >> lane) & 1u) pj[c] += sigma;
            }
            __syncwarp();
        }

        // ---------------- objective: sum of flow * cost over the basic arcs ----------------
        double acc = 0.0;
#pragma unroll
        for (int s = 0; s < NS; ++s) {
            const int y = s * 32 + lane;
            const int p = sw->info[y] & 0xff;
            if (p != 255) {
                const T m = (s < NW) ? sM[y * LDM + (p - KP)] : sM[p * LDM + (y - KP)];
                acc += (double)sw->flow[y] * (double)m;
            }
        }
        acc = warp_sum_d(acc);
        if constexpr (PLAN) {
            // zero-fill, then the basis flows with the mapping of the objective loop: Gamma[row, column]
            double *g = plan.plans + (long long)l * K * K;
            for (int e = lane; e < K * K; e += 32) g[e] = 0.0;
            __syncwarp();
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                const int y = s * 32 + lane;
                const int p = sw->info[y] & 0xff;
                if (p != 255) g[(s < NW) ? y * K + (p - KP) : p * K + (y - KP)] = (double)sw->flow[y];
            }
        }
        if (lane == 0) {
            out[l] = st == PILOT_ST_NUMERIC ? __longlong_as_double(0x7ff8000000000000LL) : acc;
            if (status) status[l] = st;
            if (pivots_out) pivots_out[l] = npiv;
        }
        __syncwarp();
    }
}

template <int NW, typename T, bool PLAN = false>
static int emd_launch(const double *props, int K, const double *cost, const PairMap &pm, long long max_pivots,
                      double *out, int *status, int *pivots, void *workspace, cudaStream_t st,
                      const PlanArgs<PLAN> &plan = {})
{
    using W = EmdWarp<NW, T>;
    unsigned long long *counter = (unsigned long long *)workspace;
    unsigned short *arcs = (unsigned short *)((char *)workspace + 256);
    const int n_arcs_pad = ((K * (K - 1) + 31) / 32) * 32 + 32;  // >= one all-0xffff chunk at the end
    emd_sort_arcs_kernel<<<1, 1024, 0, st>>>(cost, K, n_arcs_pad, arcs);
    PILOT_LAUNCH_CHECK();
    const size_t smem = sizeof(T) * W::KP * (W::KP + 1) + sizeof(unsigned short) * n_arcs_pad + sizeof(W) * EMD_WARPS;
    PILOT_CUDA(cudaFuncSetAttribute(emd_pairs_kernel<NW, T, PLAN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)smem));
    long long ctas = sm_count();
    const long long need = (pm.n_local + EMD_WARPS - 1) / EMD_WARPS;
    if (ctas > need) ctas = need;
    if (ctas < 1) ctas = 1;
    // PILOT_EMD_FAST_LIMIT (0..32, tests only): longest cycle handled by the one-lane-per-node path
    int fast_limit = 32;
    if (const char *e = getenv("PILOT_EMD_FAST_LIMIT")) {
        fast_limit = atoi(e);
        if (fast_limit < 0) fast_limit = 0;
        if (fast_limit > 32) fast_limit = 32;
    }
    // rows per major pricing pass (PILOT_EMD_SCAN_ROWS overrides, measurements only)
    int scan_rows = K <= 16 ? K : (K <= 32 ? 16 : 32);  // measured at K = 64: 4/8/16/32/64 rows -> 25.6/29.1/31.7/33.3/32.3 M pairs/s
    if (const char *e = getenv("PILOT_EMD_SCAN_ROWS")) {
        scan_rows = atoi(e);
        if (scan_rows < 1) scan_rows = 1;
        if (scan_rows > K) scan_rows = K;
    }
    emd_pairs_kernel<NW, T, PLAN><<<(unsigned)ctas, EMD_WARPS * 32, smem, st>>>(
        props, K, cost, arcs, n_arcs_pad, pm, max_pivots, out, status, pivots, counter, fast_limit, scan_rows, plan);
    PILOT_LAUNCH_CHECK();
    return 0;
}

int emd_general_launch(const double *props, int K, const double *cost, const PairMap &pm, long long max_pivots,
                       double *out, int *status, int *pivots, void *workspace, cudaStream_t st);
int emd_general_plans_launch(const double *props, int K, const double *cost, const PairMap &pm, long long max_pivots,
                             double *out, int *status, void *workspace, const PlanArgs<true> &plan, cudaStream_t st);

size_t emd_ws_bytes(int K)
{
    (void)K;
    return 256 + sizeof(unsigned short) * (64 * 63 + 64);
}

}  // namespace pilot

extern "C" int pilot_emd_pairs(const double *props, int S, int K, const double *cost, int64_t max_pivots,
                               const pilot_pair_range *range, int precision, double *out, int32_t *status,
                               int32_t *pivots, void *workspace, size_t workspace_bytes, void *stream)
{
    using namespace pilot;
    PILOT_CHECK_ARG(props && cost && out && workspace, "pilot_emd_pairs: NULL pointer");
    PILOT_CHECK_ARG(S >= 1, "pilot_emd_pairs: S=%d", S);
    PILOT_CHECK_ARG(K >= 1 && K <= 256, "pilot_emd_pairs: K=%d outside the supported range [1, 256]", K);
    PILOT_CHECK_ARG(precision == PILOT_F64 || precision == PILOT_F32, "pilot_emd_pairs: precision=%d", precision);
    PILOT_CHECK_ARG(workspace_bytes >= emd_ws_bytes(K), "pilot_emd_pairs: workspace too small");
    PairMap pm;
    int rc = make_pair_map(range, S, &pm);
    if (rc) return rc;
    if (pm.n_local == 0) return 0;
    if (max_pivots <= 0) max_pivots = 100000;  // POT numItermax default
    cudaStream_t st = (cudaStream_t)stream;
    PILOT_CUDA(cudaMemsetAsync(workspace, 0, 256, st));
    if (K > 64)  // beyond the bit-mask solver: general network simplex (emd_general.cu), FP64 whatever the precision
        return emd_general_launch(props, K, cost, pm, max_pivots, out, status, pivots, workspace, st);
    if (precision == PILOT_F64) {
        if (K <= 32) return emd_launch<1, double>(props, K, cost, pm, max_pivots, out, status, pivots, workspace, st);
        return emd_launch<2, double>(props, K, cost, pm, max_pivots, out, status, pivots, workspace, st);
    }
    if (K <= 32) return emd_launch<1, float>(props, K, cost, pm, max_pivots, out, status, pivots, workspace, st);
    return emd_launch<2, float>(props, K, cost, pm, max_pivots, out, status, pivots, workspace, st);
}

extern "C" int pilot_emd_plans(const double *props, int S, int K, const double *cost, int64_t max_pivots,
                               const int32_t *pair_a, const int32_t *pair_b, int64_t n, double *plans, double *out,
                               int32_t *status, void *workspace, size_t workspace_bytes, void *stream)
{
    using namespace pilot;
    PILOT_CHECK_ARG(props && cost && pair_a && pair_b && plans && out && workspace, "pilot_emd_plans: NULL pointer");
    PILOT_CHECK_ARG(S >= 1, "pilot_emd_plans: S=%d", S);
    PILOT_CHECK_ARG(K >= 1 && K <= 256, "pilot_emd_plans: K=%d outside the supported range [1, 256]", K);
    PILOT_CHECK_ARG(n >= 0, "pilot_emd_plans: n=%lld", (long long)n);
    PILOT_CHECK_ARG(workspace_bytes >= emd_ws_bytes(K), "pilot_emd_plans: workspace too small");
    if (n == 0) return 0;
    if (max_pivots <= 0) max_pivots = 100000;  // POT numItermax default
    const PairMap pm = plan_pair_map(n, S);
    const PlanArgs<true> plan{pair_a, pair_b, S, plans};
    cudaStream_t st = (cudaStream_t)stream;
    PILOT_CUDA(cudaMemsetAsync(workspace, 0, 256, st));
    if (K > 64) return emd_general_plans_launch(props, K, cost, pm, max_pivots, out, status, workspace, plan, st);
    if (K <= 32)
        return emd_launch<1, double, true>(props, K, cost, pm, max_pivots, out, status, nullptr, workspace, st, plan);
    return emd_launch<2, double, true>(props, K, cost, pm, max_pivots, out, status, nullptr, workspace, st, plan);
}
