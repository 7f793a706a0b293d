// Kernel (3), wide variant: the batched shared-Gibbs-kernel solver of sinkhorn_batched.cu for 65 <= K <= 256.
// Same formulation (scaled iterates on the shared K0 = exp(-M/reg), mma.sync m8n8k4 FP64 panels of 8 problems,
// POT's schedule: absorption test every iteration, marginal error every `check_every`, NaN / Inf -> reference
// form), but K0 no longer fits one CTA's shared memory, so it is split over a thread-block cluster.
//
// Row stripes.  With KC = roundup(K, 8) the KC/8 row tiles are dealt out evenly over the CL CTAs of a cluster
// (the first KC/8 % CL members take one tile more).  Member r keeps in its shared memory the columns of K0 that
// produce its output rows: stripe[k][j - j0] = K0[k][j] for phase A (T = K0^T Ut) and K0[j][k] for phase B
// (S = K0 Vt).  For a symmetric cost (always so in PILOT) the two are the same array and a stripe is at most
// SKW_SH_SYM = 64 rows: 64 x 256 x 8 B = 128 KB at K = 256, CL = ceil(KC / 64) = 2..4.  The general variant
// holds both, in stripes half as tall: CL = ceil(KC / 32) <= 8, the portable maximum.
//
// Warp teams.  Warp w of every member forms one team that runs one 8-problem panel.  Every member keeps the
// whole KC x 8 panels Ut and Vt, computes the rows of its stripe with the DMMA loop of the panel kernel
// (k = 0 .. KC-1 ascending: each output row is the same FMA chain as in a KC-wide panel, whatever CL is or
// which slot a problem sits in) and then sends those rows to every member over DSMEM, together with its
// per-slot partials (max |u|, |v| as sk_abs_bits; the error^2 when a check is pending; the final cost of a
// problem that stops).  It arrives on every member's per-warp mbarrier (cluster scope) and waits on its own.
// Every member then reduces the partials in member order 0 .. CL-1 and so takes the same stop / absorb / redo
// decision with no further communication.  Member 0 draws refills from the global counter and sends their
// indices with the Ut exchange.  Absorptions are applied by every member to its full copy of the panels
// (the scaling is exact and elementwise, so the copies stay identical); the range test reads the full copy.
//
// Vt is double-buffered (Vt[p] of the previous iteration, Vt[q] of this one): a slot's convergence is known
// only after the Vt exchange of the next iteration, and its final cost sum_ij (M o K0)_ij Ut_i Vt_j still
// needs the previous Vt in full.  Member r sums it over its own rows i, reading M o K0 from the setup buffer
// (L2), and the partials are summed in member order.
//
// No tail hand-over: a panel whose problems run out keeps its stragglers (DESIGN.md section 6).
#include <cooperative_groups.h>
#include "sinkhorn.cuh"

namespace cg = cooperative_groups;

namespace pilot {

constexpr int SKW_MAX_WARPS = 8;   // warps (teams) per CTA; the shared-memory budget sets the actual count
constexpr int SKW_SPW = 8;         // slots per team = panel columns
constexpr int SKW_SH_SYM = 64;     // stripe height, symmetric cost: 8 accumulator tiles x 2 per lane
constexpr int SKW_SH_GEN = 32;     // stripe height, general cost (K0 and K0^T stripes)
__host__ __device__ constexpr int skw_max_cl(bool sym) { return 256 / (sym ? SKW_SH_SYM : SKW_SH_GEN); }  // 4 or 8

// per-warp exchange record of one slot
struct SkwPart {
    long long mx;  // max sk_abs_bits of the member's rows
    double x;      // V half: error^2 of a pending check; U half: cost of a problem that stopped
};
template <int CLM>  // CLM: largest cluster of the variant
struct SkwXchg {
    SkwPart v[CLM][SKW_SPW];
    SkwPart u[CLM][SKW_SPW];
    long long ids[SKW_SPW];        // refills drawn by member 0
    unsigned long long bar_v, bar_u;
};

__device__ __forceinline__ unsigned skw_smem_addr(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void skw_arrive_remote(unsigned long long *bar, unsigned rank)
{
    unsigned ra;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(skw_smem_addr(bar)), "r"(rank));
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(ra) : "memory");
}

__device__ __forceinline__ void skw_wait(unsigned long long *bar, unsigned parity)
{
    const unsigned a = skw_smem_addr(bar);
    unsigned done;
    do {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n"
                     " selp.u32 %0, 1, 0, p;\n}"
                     : "=r"(done) : "r"(a), "r"(parity) : "memory");
    } while (!done);
}

__device__ __forceinline__ void skw_dmma(double &c0, double &c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

__device__ __forceinline__ int skw_swz(int row, int col) { return col ^ ((row & 3) << 2); }

// shared memory of one CTA: stripe(s) [KC][SH] (swizzled), then per warp Ut [KC][8], Vt [2][KC][8], SkwXchg
// (K = 256, symmetric: 128 KB + 2 x 49.1 KB, two teams per CTA)
static size_t skw_smem_bytes(int KC, bool sym, int warps)
{
    const size_t xchg = sym ? sizeof(SkwXchg<skw_max_cl(true)>) : sizeof(SkwXchg<skw_max_cl(false)>);
    return sizeof(double) * (size_t)(sym ? 1 : 2) * KC * (sym ? SKW_SH_SYM : SKW_SH_GEN) +
           (size_t)warps * (sizeof(double) * 3 * KC * SKW_SPW + xchg);
}

// Buffer reuse without overwrite (X, Y members of one team, iteration n writes Vt[q], n+1 writes Vt[p]):
//  - Y writes X's Ut rows in the Ut exchange of n only after its wait on the Vt barrier of n, which needs X's
//    arrival there; X arrives after its phase A of n, the last read of the previous Ut rows of Y (the final cost
//    reads only X's own Ut rows, which only X writes).
//  - Y writes X's Vt[p] again in the Vt exchange of n+1 only after its wait on the Ut barrier of n, which needs
//    X's Ut arrival of n: X has then finished phase B of n-1 (the last read of Vt[p] as input), the error of a
//    pending check and the final cost of n (the last reads of Vt[p] as the previous iterate).
//  - The partial records follow the same argument (v at the Vt barrier, u and ids at the Ut barrier), and the
//    absorption scaling of X's full panels happens before X's next arrival.
//  - A member cannot arrive twice on one barrier phase: its next arrival on X's Vt barrier needs the completed Ut
//    phase of its own barrier, which needs X's arrival, made after X has waited on its Vt barrier.
template <int SH, bool SYM>
__global__ void __launch_bounds__(SKW_MAX_WARPS * 32, 1)
sinkhorn_wide_kernel(const double *__restrict__ props, int K, SkParams prm, PairMap pm, SkSetup s,
                     double *__restrict__ scratch,  // [gridDim * warps * 8][2][SH] rea / reb of the member's rows
                     unsigned long long *__restrict__ counter, double *__restrict__ out, int *__restrict__ iters_out,
                     int *__restrict__ abs_out, int *__restrict__ status_out, long long *__restrict__ redo_list,
                     unsigned long long *__restrict__ n_redo)
{
    const SkOut res{out, iters_out, abs_out, status_out, redo_list, n_redo};
    if ((*s.asym != 0) == SYM) return;  // both variants are enqueued; the setup kernel's flag picks one
    constexpr int MT = SH / 8;
    constexpr int PS = SKW_SPW;
    cg::cluster_group cluster = cg::this_cluster();
    const int CL = (int)cluster.num_blocks();
    const int me = (int)cluster.block_rank();
    const int KC = (K + 7) & ~7, KP = KC;  // the setup buffer's extent is KC for K > 64
    const int KS = KC / 4;
    const int tiles = KC / 8, tq = tiles / CL, tr = tiles % CL;
    const int nt = tq + (me < tr ? 1 : 0);               // my row tiles
    const int r0 = 8 * (me * tq + (me < tr ? me : tr));  // my first row
    const int nrows = 8 * nt;
    const int warps = blockDim.x >> 5;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *sA = reinterpret_cast<double *>(smem_raw);  // phase A: [k][swz(k, j - r0)] = K0[k][j]
    double *sB = SYM ? sA : sA + (size_t)KC * SH;       // phase B: [k][swz(k, i - r0)] = K0[i][k]
    double *panels = sA + (size_t)(SYM ? 1 : 2) * KC * SH;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double *U = panels + (size_t)warp * 3 * KC * PS;  // U[row][slot], then Vt[0], Vt[1]
    double *Vb = U + (size_t)KC * PS;
    using Xchg = SkwXchg<skw_max_cl(SYM)>;
    Xchg *xg = reinterpret_cast<Xchg *>(panels + (size_t)warps * 3 * KC * PS) + warp;

    for (int e = threadIdx.x; e < KC * SH; e += blockDim.x) {
        const int k = e / SH, c = e - k * SH;
        const bool in = c < nrows;
        sA[k * SH + skw_swz(k, c)] = in ? s.K0[(size_t)k * KP + r0 + c] : 0.0;
        if (!SYM) sB[k * SH + skw_swz(k, c)] = in ? s.K0T[(size_t)k * KP + r0 + c] : 0.0;
    }
    for (int e = lane; e < 3 * KC * PS; e += 32) U[e] = 0.0;  // rows >= K stay 0: the DMMA reads them

    const int g = lane >> 2, t = lane & 3;
    const unsigned gmask = 0x11111111u << t;  // the 8 lanes that share my 2 slots
    const int tsw = (t & 2) << 2, gsw = g ^ ((t & 1) << 2);
    double *rea0 = scratch + ((size_t)(blockIdx.x * warps + warp) * SKW_SPW + 2 * t) * 2 * SH;  // slot 2t, then 2t+1
    const double invK = 1.0 / K;

    long long sl[2];
    const double *pa[2], *pb[2];
    int s_ii[2], s_abs[2];
    bool s_act[2], s_hasabs[2], s_pend[2], s_force[2], s_fresh[2], s_bad[2];

#define ROW_OK(r) ((r) < K)
#define SKW_ASSIGN(h, w)                                                              \
    do {                                                                              \
        sl[h] = (w);                                                                  \
        s_act[h] = sl[h] >= 0 && sl[h] < pm.n_local;                                  \
        int si_ = 0, sj_ = 0;                                                         \
        if (s_act[h]) global_to_ij(pm, local_to_global(pm, sl[h]), si_, sj_);         \
        pa[h] = props + (long long)si_ * K + r0 + g;                                  \
        pb[h] = props + (long long)sj_ * K + r0 + g;                                  \
        s_ii[h] = 0; s_abs[h] = 0; s_hasabs[h] = false; s_pend[h] = false;            \
        s_force[h] = false; s_fresh[h] = true; s_bad[h] = false;                      \
    } while (0)

    // initial fill: member 0 draws, every member reads after the cluster barrier (which also publishes the
    // initialised mbarriers)
    if (lane == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(skw_smem_addr(&xg->bar_v)), "r"(CL));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(skw_smem_addr(&xg->bar_u)), "r"(CL));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (me == 0 && lane < SKW_SPW) {
        const long long w = (long long)atomicAdd(counter, 1ULL);
        for (int rr = 0; rr < CL; ++rr) cluster.map_shared_rank(xg, rr)->ids[lane] = w;
    }
    cluster.sync();
#pragma unroll
    for (int h = 0; h < 2; ++h) SKW_ASSIGN(h, xg->ids[2 * t + h]);

    int p = 0;         // Vt[p]: previous iterate, Vt[p ^ 1]: this iteration's
    unsigned ph = 0;   // barrier phase parity (both barriers complete once per iteration)
    for (;;) {
        if (!__any_sync(0xffffffffu, s_act[0] || s_act[1])) break;
        const double *Vp = Vb + (size_t)p * KC * PS;
        double *Vq = Vb + (size_t)(p ^ 1) * KC * PS;
        double acc[MT][2];
        // ======================= phase A: my rows of T = K0^T Ut =======================
#pragma unroll
        for (int m = 0; m < MT; ++m) { acc[m][0] = 0.0; acc[m][1] = 0.0; }
#pragma unroll 2
        for (int ks = 0; ks < KS; ++ks) {
            const int kr = 4 * ks + t;
            const double b0 = U[kr * PS + g];
            const double *arow = sA + kr * SH + gsw;
#pragma unroll
            for (int m = 0; m < MT; ++m)
                if (m < nt) skw_dmma(acc[m][0], acc[m][1], arow[(8 * m) ^ tsw], b0);
        }
        // ---- error^2 of a pending check (previous Vt, my rows) and the v-update ----
        double e2[2] = {0.0, 0.0};
        long long mxv[2] = {0, 0};
#pragma unroll
        for (int m = 0; m < MT; ++m) {
            if (m >= nt) break;
            const int lrow = 8 * m + g, row = r0 + lrow;
            double vv[2] = {0.0, 0.0};
            if (ROW_OK(row)) {
#pragma unroll
                for (int h = 0; h < 2; ++h)
                    if (s_act[h]) {
                        const double bj = __ldg(pb[h] + 8 * m);
                        if (s_pend[h] && !s_fresh[h]) {
                            const double d = fma(Vp[row * PS + 2 * t + h], acc[m][h], -bj);
                            e2[h] = fma(d, d, e2[h]);
                        }
                        const double tv = s_fresh[h] ? __ldg(s.c0 + row) : acc[m][h];
                        vv[h] = sk_div(bj, tv);
                        const double uu = s_hasabs[h] ? vv[h] * rea0[(2 * h + 1) * SH + lrow] : vv[h];
                        mxv[h] = max(mxv[h], sk_abs_bits(uu));
                    }
            }
            const double2 v2 = make_double2(vv[0], vv[1]);
            for (int rr = 0; rr < CL; ++rr)
                *reinterpret_cast<double2 *>(cluster.map_shared_rank(Vq, rr) + row * PS + 2 * t) = v2;
        }
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int o = 4; o < 32; o <<= 1) {
                e2[h] += __shfl_xor_sync(gmask, e2[h], o);
                mxv[h] = max(mxv[h], __shfl_xor_sync(gmask, mxv[h], o));
            }
        if (g == 0)
            for (int rr = 0; rr < CL; ++rr) {
                Xchg *x = cluster.map_shared_rank(xg, rr);
#pragma unroll
                for (int h = 0; h < 2; ++h) x->v[me][2 * t + h] = SkwPart{mxv[h], e2[h]};
            }
        asm volatile("fence.acq_rel.cluster;" ::: "memory");
        __syncwarp();
        if (lane < CL) skw_arrive_remote(&xg->bar_v, lane);
        skw_wait(&xg->bar_v, ph);

        // ---- stop decisions, identical in every member ----
        bool stop[2];
        int stt[2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            long long mx = 0;
            double e2s = 0.0;
            for (int rr = 0; rr < CL; ++rr) {
                const SkwPart q = xg->v[rr][2 * t + h];
                mx = max(mx, q.mx);
                e2s += q.x;
            }
            mxv[h] = mx;
            stop[h] = false;
            stt[h] = PILOT_ST_MAXITER;
            if (s_act[h] && !s_fresh[h]) {
                if (s_bad[h]) { stop[h] = true; stt[h] = -1; }
                else if (s_pend[h] && sqrt(e2s) <= prm.stop_thr) { stop[h] = true; stt[h] = PILOT_ST_CONVERGED; }
                else if (s_force[h]) stop[h] = true;
            }
        }
        // ---- my part of the cost of the problems that stopped: sum_{i mine} Ut_i sum_j (M o K0)_ij Vt_j ----
        double cpart[2] = {0.0, 0.0};
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            unsigned mb = __ballot_sync(0xffffffffu, stop[h] && stt[h] >= 0) & 0xfu;
            while (mb) {
                const int tt = __ffs(mb) - 1;
                mb &= mb - 1;
                const int col = 2 * tt + h;
                double c = 0.0;
                for (int j = lane; j < KC; j += 32) {
                    double w0 = 0.0;
                    for (int i = r0; i < r0 + nrows && i < K; ++i)
                        w0 = fma(s.MK[(size_t)i * KP + j], U[i * PS + col], w0);
                    c = fma(Vp[j * PS + col], w0, c);
                }
                c = warp_sum_d(c);
                if (t == tt) cpart[h] = c;
            }
        }
        // ---- member 0 draws the refills ----
        long long fill[2] = {-1, -1};
        if (me == 0) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                long long w = -1;
                if (g == 0 && stop[h]) w = (long long)atomicAdd(counter, 1ULL);
                fill[h] = w;
            }
        }
#pragma unroll
        for (int h = 0; h < 2; ++h)
            if (stop[h]) s_act[h] = false;
        __syncwarp();

        // ======================= phase B: my rows of S = K0 Vt =======================
#pragma unroll
        for (int m = 0; m < MT; ++m) { acc[m][0] = 0.0; acc[m][1] = 0.0; }
#pragma unroll 2
        for (int ks = 0; ks < KS; ++ks) {
            const int kr = 4 * ks + t;
            const double b0 = Vq[kr * PS + g];
            const double *arow = sB + kr * SH + gsw;
#pragma unroll
            for (int m = 0; m < MT; ++m)
                if (m < nt) skw_dmma(acc[m][0], acc[m][1], arow[(8 * m) ^ tsw], b0);
        }
        // ---- u-update of my rows ----
        long long mxu[2] = {0, 0};
#pragma unroll
        for (int m = 0; m < MT; ++m) {
            if (m >= nt) break;
            const int lrow = 8 * m + g, row = r0 + lrow;
            double un[2] = {0.0, 0.0};
            if (ROW_OK(row)) {
#pragma unroll
                for (int h = 0; h < 2; ++h)
                    if (s_act[h]) {
                        un[h] = sk_div(__ldg(pa[h] + 8 * m), acc[m][h]);
                        const double uu = s_hasabs[h] ? un[h] * rea0[(2 * h) * SH + lrow] : un[h];
                        mxu[h] = max(mxu[h], sk_abs_bits(uu));
                    }
            }
            const double2 u2 = make_double2(un[0], un[1]);
            for (int rr = 0; rr < CL; ++rr)
                *reinterpret_cast<double2 *>(cluster.map_shared_rank(U, rr) + row * PS + 2 * t) = u2;
        }
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int o = 4; o < 32; o <<= 1) mxu[h] = max(mxu[h], __shfl_xor_sync(gmask, mxu[h], o));
        if (g == 0)
            for (int rr = 0; rr < CL; ++rr) {
                Xchg *x = cluster.map_shared_rank(xg, rr);
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    x->u[me][2 * t + h] = SkwPart{mxu[h], cpart[h]};
                    if (me == 0 && stop[h]) x->ids[2 * t + h] = fill[h];
                }
            }
        asm volatile("fence.acq_rel.cluster;" ::: "memory");
        __syncwarp();
        if (lane < CL) skw_arrive_remote(&xg->bar_u, lane);
        skw_wait(&xg->bar_u, ph);
        ph ^= 1u;

        // ---- results of the stopped problems, absorption test and counters ----
        bool absorb[2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            long long mx = mxv[h];
            double cost = 0.0;
            for (int rr = 0; rr < CL; ++rr) {
                const SkwPart q = xg->u[rr][2 * t + h];
                mx = max(mx, q.mx);
                cost += q.x;
            }
            if (stop[h] && me == 0 && g == 0) sk_store(res, sl[h], stt[h], cost, s_ii[h], s_abs[h]);
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
            // u = v = 1/K in POT == divide the scaled iterates by K, here in every member's full copy; remember
            // 1/ut, 1/vt of my rows; the range test sees every row, so every member finds the same
#pragma unroll
            for (int h = 0; h < 2; ++h)
                if (absorb[h]) {
                    const int col = 2 * t + h;
                    int rb = 0;
                    for (int row = g; row < KC; row += 8) {
                        const double uo = U[row * PS + col], vo = Vq[row * PS + col];
                        if (ROW_OK(row)) {
                            const int lrow = row - r0;
                            if (lrow >= 0 && lrow < nrows) {
                                rea0[(2 * h) * SH + lrow] = 1.0 / uo;
                                rea0[(2 * h + 1) * SH + lrow] = 1.0 / vo;
                            }
                            rb |= sk_out_of_range(uo, vo);
                            U[row * PS + col] = uo * invK;
                            Vq[row * PS + col] = vo * invK;
                        }
                    }
                    rb |= __shfl_xor_sync(gmask, rb, 4);
                    rb |= __shfl_xor_sync(gmask, rb, 8);
                    rb |= __shfl_xor_sync(gmask, rb, 16);
                    s_hasabs[h] = true;
                    ++s_abs[h];
                    s_bad[h] = s_bad[h] || rb;
                }
        }
        // ---- refill the stopped slots with what member 0 drew ----
#pragma unroll
        for (int h = 0; h < 2; ++h)
            if (stop[h]) SKW_ASSIGN(h, xg->ids[2 * t + h]);
        __syncwarp();
        p ^= 1;
    }
#undef SKW_ASSIGN
#undef ROW_OK
    cluster.sync();  // no CTA exits while a peer may still write to its shared memory
}

size_t skw_scratch_bytes(int ctas) { return sizeof(double) * (size_t)ctas * SKW_MAX_WARPS * SKW_SPW * 2 * SKW_SH_SYM; }

template <int SH, bool SYM>
static int skw_launch_t(const double *props, int K, const SkParams &prm, const PairMap &pm, const SkSetup &s,
                        double *scratch, const SkOut &res, unsigned long long *counter, cudaStream_t st)
{
    const int KC = (K + 7) & ~7;
    const int CL = (KC + SH - 1) / SH;
    int dev = 0, smem_max = 0;
    PILOT_CUDA(cudaGetDevice(&dev));
    PILOT_CUDA(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    // as many warp teams per CTA as the shared memory holds
    int warps = SKW_MAX_WARPS;
    while (warps > 1 && skw_smem_bytes(KC, SYM, warps) > (size_t)smem_max) --warps;
    const size_t smem = skw_smem_bytes(KC, SYM, warps);
    PILOT_CHECK_ARG(smem <= (size_t)smem_max, "sinkhorn wide kernel: K=%d does not fit", K);
    auto kern = sinkhorn_wide_kernel<SH, SYM>;
    PILOT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CL;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cfg.blockDim = dim3(warps * 32);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    // persistent clusters, one wave (at most one CTA per SM: the scratch holds sm_count() CTAs)
    long long clusters = sm_count() / CL;
    cfg.gridDim = dim3((unsigned)(clusters * CL));
    int active = 0;
    PILOT_CUDA(cudaOccupancyMaxActiveClusters(&active, kern, &cfg));
    if (active >= 1 && active < clusters) clusters = active;
    // small batches: fewer teams per CTA (shorter iterations), spread over as many clusters as they fill
    const long long teams = (pm.n_local + SKW_SPW - 1) / SKW_SPW;
    long long per = (teams + clusters - 1) / clusters;
    if (per < warps) {
        cfg.blockDim = dim3((unsigned)(per * 32));
        clusters = (teams + per - 1) / per;
    }
    cfg.gridDim = dim3((unsigned)(clusters * CL));
    PILOT_CUDA(cudaLaunchKernelEx(&cfg, kern, props, K, prm, pm, s, scratch, counter, res.out, res.iters, res.absn,
                                  res.status, res.redo, res.n_redo));
    PILOT_LAUNCH_CHECK();
    return 0;
}

// `setup` must hold the output of skb_setup; scratch: skw_scratch_bytes(sm_count()) bytes
int skw_launch(const double *props, int K, const SkParams &prm, const PairMap &pm, const double *setup,
               double *scratch, bool symmetric, const SkOut &res, unsigned long long *counter, cudaStream_t st)
{
    PILOT_CHECK_ARG(K > 64 && K <= 256, "sinkhorn wide kernel: K=%d", K);
    const SkSetup s = sk_setup_view(setup, sk_setup_extent(K));
    return symmetric ? skw_launch_t<SKW_SH_SYM, true>(props, K, prm, pm, s, scratch, res, counter, st)
                     : skw_launch_t<SKW_SH_GEN, false>(props, K, prm, pm, s, scratch, res, counter, st);
}

}  // namespace pilot
