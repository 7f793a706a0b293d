// Kernel (4), general variant: exact EMD for 65 <= K <= 256 cell types.
//
// ot.emd2 (reference pilotpy/tools/Trajectory.py:511) has no limit on the histogram length; the bit-mask solver of
// emd.cu holds a problem's basis tree in 64-bit masks and stops at K = 64.  A Leiden clustering with more clusters
// takes this kernel instead: the same primal network simplex POT runs (artificial root, big-M star as the start
// basis, strongly feasible leaving rule -- strict '<' on the first path, '<=' on the second --, relative-epsilon
// entering test), one problem per warp, the tree as plain arrays (parent, orientation and flow of the parent arc,
// potential) in shared memory:
//   pricing   all lanes, blocks of 4 rows x K columns from a rotating start row; the first block holding an eligible
//             arc gives the entering arc (its most negative reduced cost)
//   pivot     lane 0 walks the cycle (join node by stamping the first path), finds the leaving arc, pushes delta and
//             reverses the parent pointers along the stem
//   update    all lanes: a node belongs to the re-hung subtree iff its root path meets the entering end; those
//             potentials shift by the entering arc's reduced cost
// Any exact method returns the same optimum, so the result agrees with the bit-mask kernel (and the oracle) to
// rounding.  Throughput is not the point here (about a thousand times the CPU loop, far below emd.cu): it removes a
// limit the reference does not have.  FP64 only.
#include "common.cuh"

namespace pilot {

constexpr int EMG_ROWS = 4;  // rows per pricing block

// per-warp state, N = 2K + 1 nodes (sources 0..K-1, sinks K..2K-1, root 2K)
struct EmgView {
    double *pi, *flow;      // [N] potential; flow on the arc to the parent
    short *parent;          // [N]
    unsigned short *stamp;  // [N] join search
    unsigned char *up;      // [N] 1: the parent arc runs node -> parent
};

__host__ __device__ __forceinline__ size_t emg_state_bytes(int K)
{
    const size_t N = 2 * (size_t)K + 1;
    return ((N * (8 + 8 + 2 + 2 + 1)) + 15) & ~(size_t)15;
}

// PLAN: problems from the pair list of `plan`, and each problem's plan written from the real tree arcs
template <bool PLAN>
__global__ void __launch_bounds__(512)
emd_general_kernel(const double *__restrict__ props, int K, const double *__restrict__ cost, PairMap pm,
                   long long max_pivots, double *__restrict__ out, int *__restrict__ status,
                   int *__restrict__ pivots_out, unsigned long long *__restrict__ counter,
                   const double *__restrict__ art_p, PlanArgs<PLAN> plan)
{
    const double art = *art_p;  // big-M cost of the artificial arcs (emg_art_kernel)
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int N = 2 * K + 1, root = 2 * K;
    unsigned char *base = smem_raw + (size_t)warp * emg_state_bytes(K);
    EmgView s;
    s.pi = reinterpret_cast<double *>(base);
    s.flow = s.pi + N;
    s.parent = reinterpret_cast<short *>(s.flow + N);
    s.stamp = reinterpret_cast<unsigned short *>(s.parent + N);
    s.up = reinterpret_cast<unsigned char *>(s.stamp + N);
    const double EPS = 2.2204460492503131e-15;  // 10 * DBL_EPSILON, as POT

    for (;;) {
        unsigned long long l = 0;
        if (lane == 0) l = atomicAdd(counter, 1ULL);
        l = __shfl_sync(0xffffffffu, l, 0);
        if ((long long)l >= pm.n_local) break;
        int si, sj;
        if constexpr (PLAN) {
            if (!plan_pair(plan, (long long)l, si, sj)) {
                double *g = plan.plans + (long long)l * K * K;
                for (int e = lane; e < K * K; e += 32) g[e] = __longlong_as_double(PILOT_NAN_BITS);
                if (lane == 0) {
                    out[l] = __longlong_as_double(PILOT_NAN_BITS);
                    if (status) status[l] = PILOT_ST_NUMERIC;
                }
                continue;
            }
        } else {
            global_to_ij(pm, local_to_global(pm, (long long)l), si, sj);
        }
        const double *pa = props + (long long)si * K, *pb = props + (long long)sj * K;

        // ---- a, b (emd2 rescales b to the mass of a), the artificial star ----
        double sa = 0.0, sb = 0.0;
        for (int j = lane; j < K; j += 32) { sa += pa[j]; sb += pb[j]; }
        sa = warp_sum_d(sa);
        sb = warp_sum_d(sb);
        for (int u = lane; u < N; u += 32) {
            s.stamp[u] = 0;
            if (u == root) { s.parent[u] = -1; s.pi[u] = 0.0; s.flow[u] = 0.0; s.up[u] = 0; continue; }
            const double sup = u < K ? pa[u] : -__ddiv_rn(__dmul_rn(pb[u - K], sa), sb);
            s.parent[u] = (short)root;
            if (sup >= 0.0) { s.up[u] = 1; s.flow[u] = sup; s.pi[u] = 0.0; }
            else            { s.up[u] = 0; s.flow[u] = -sup; s.pi[u] = art; }
        }
        __syncwarp();

        int st = PILOT_ST_CONVERGED;
        long long npiv = 0;
        int next_row = 0;
        unsigned short stamp_id = 0;
        for (;;) {
            // ---- pricing: blocks of EMG_ROWS rows from a rotating start; first block with an eligible arc ----
            double best = 0.0;
            int bi = -1, bj = -1;
            for (int scanned = 0; scanned < K && bi < 0; scanned += EMG_ROWS) {
                double lb = 0.0;
                int li = -1, lj = -1;
                for (int rr = 0; rr < EMG_ROWS && scanned + rr < K; ++rr) {
                    int i = next_row + scanned + rr;
                    if (i >= K) i -= K;
                    const double pi_i = s.pi[i];
                    const int par_i = s.parent[i];
                    const double *mrow = cost + (long long)i * K;
                    for (int j = lane; j < K; j += 32) {
                        const double m = __ldg(mrow + j), pj = s.pi[K + j];
                        const double rc = (m + pi_i) - pj;
                        // tree arcs are never candidates (their reduced cost is zero up to rounding)
                        const bool tree = par_i == K + j || s.parent[K + j] == i;
                        const double tol = EPS * fmax(fmax(fabs(pi_i), fabs(pj)), fabs(m));
                        if (!tree && rc < -tol && rc < lb) { lb = rc; li = i; lj = j; }
                    }
                }
                // warp argmin (ties: smallest row-major arc index, so the choice is deterministic)
                unsigned long long key = li < 0 ? ~0ULL : (unsigned long long)(li * K + lj);
                double v = lb;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const double ov = __shfl_xor_sync(0xffffffffu, v, o);
                    const unsigned long long ok = __shfl_xor_sync(0xffffffffu, key, o);
                    if (ov < v || (ov == v && ok < key)) { v = ov; key = ok; }
                }
                if (key != ~0ULL) { best = v; bi = (int)(key / (unsigned)K); bj = (int)(key % (unsigned)K); }
                if (bi >= 0) {
                    next_row += scanned + EMG_ROWS;
                    while (next_row >= K) next_row -= K;
                }
            }
            if (bi < 0) break;  // optimal
            if (++npiv > max_pivots) { st = PILOT_ST_MAXITER; break; }

            // ---- pivot (lane 0) ----
            int u_in = -1;
            double sigma = 0.0;
            if (lane == 0) {
                const int first = bi, second = K + bj;
                if (++stamp_id == 0) {  // wrapped: clear
                    for (int u = 0; u < N; ++u) s.stamp[u] = 0;
                    stamp_id = 1;
                }
                for (int u = first; u >= 0; u = s.parent[u]) s.stamp[u] = stamp_id;
                int join = second;
                while (s.stamp[join] != stamp_id) join = s.parent[join];
                double delta = __longlong_as_double(0x7ff0000000000000LL);
                int u_out = -1, side = 0;
                for (int u = first; u != join; u = s.parent[u])
                    if (s.up[u] && s.flow[u] < delta) { delta = s.flow[u]; u_out = u; side = 1; }
                for (int u = second; u != join; u = s.parent[u])
                    if (!s.up[u] && s.flow[u] <= delta) { delta = s.flow[u]; u_out = u; side = 2; }
                if (u_out < 0) {
                    u_in = -2;  // unbounded (cannot happen for a balanced problem)
                } else {
                    if (delta > 0.0) {
                        for (int u = first; u != join; u = s.parent[u]) s.flow[u] += s.up[u] ? -delta : delta;
                        for (int u = second; u != join; u = s.parent[u]) s.flow[u] += s.up[u] ? delta : -delta;
                    }
                    u_in = side == 1 ? first : second;
                    const int v_in = side == 1 ? second : first;
                    // reverse the stem u_in .. u_out: every node hangs under its former child
                    int child = u_in, new_parent = v_in;
                    double carry_flow = delta;                    // flow of the entering arc
                    unsigned char carry_up = u_in == first;       // entering arc runs first -> second
                    for (;;) {
                        const int old_parent = s.parent[child];
                        const double old_flow = s.flow[child];
                        const unsigned char old_up = s.up[child];
                        s.parent[child] = (short)new_parent;
                        s.flow[child] = carry_flow;
                        s.up[child] = carry_up;
                        if (child == u_out) break;
                        carry_flow = old_flow;
                        carry_up = !old_up;
                        new_parent = child;
                        child = old_parent;
                    }
                    sigma = u_in == first ? -best : best;
                }
            }
            u_in = __shfl_sync(0xffffffffu, u_in, 0);
            sigma = __shfl_sync(0xffffffffu, sigma, 0);
            __syncwarp();
            if (u_in == -2) { st = PILOT_ST_UNBOUNDED; break; }
            // ---- potentials of the re-hung subtree: every node whose root path meets u_in ----
            for (int x = lane; x < N; x += 32) {
                int y = x;
                while (y >= 0 && y != u_in) y = s.parent[y];
                if (y == u_in) s.pi[x] += sigma;
            }
            __syncwarp();
        }

        // ---- cost = sum of flow * M over the real tree arcs (an artificial arc hangs under the root) ----
        double acc = 0.0;
        bool infeasible = false;
        for (int u = lane; u < root; u += 32) {
            const int p = s.parent[u];
            if (p == root) { if (s.flow[u] > 1e-8) infeasible = true; continue; }
            const int i = u < K ? u : p, j = u < K ? p - K : u - K;
            acc = fma(s.flow[u], __ldg(cost + (long long)i * K + j), acc);
        }
        acc = warp_sum_d(acc);
        infeasible = __any_sync(0xffffffffu, infeasible);
        if constexpr (PLAN) {
            // zero-fill, then the flows of the real tree arcs with the mapping of the cost loop
            double *g = plan.plans + (long long)l * K * K;
            for (int e = lane; e < K * K; e += 32) g[e] = 0.0;
            __syncwarp();
            for (int u = lane; u < root; u += 32) {
                const int p = s.parent[u];
                if (p == root) continue;
                g[u < K ? (long long)u * K + (p - K) : (long long)p * K + (u - K)] = s.flow[u];
            }
        }
        if (lane == 0) {
            const bool bad = !(sa == sa) || !(sb == sb) || (st == PILOT_ST_CONVERGED && infeasible);
            out[l] = bad ? __longlong_as_double(0x7ff8000000000000LL) : acc;
            if (status) status[l] = bad ? PILOT_ST_NUMERIC : st;
            if (pivots_out) pivots_out[l] = (int)npiv;
        }
        __syncwarp();
    }
}

// max |cost| + 1, times (2K + 2): the big-M cost of the artificial arcs (EMD_wrap's choice)
__global__ void emg_art_kernel(const double *__restrict__ cost, int K, double *__restrict__ art)
{
    __shared__ double red[32];
    double m = 0.0;
    for (int t = threadIdx.x; t < K * K; t += blockDim.x) m = fmax(m, fabs(cost[t]));
    m = warp_max_d(m);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x < 32) {
        m = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.0;
        m = warp_max_d(m);
        if (threadIdx.x == 0) *art = (m + 1.0) * (double)(2 * K + 2);
    }
}

template <bool PLAN>
static int emg_launch(const double *props, int K, const double *cost, const PairMap &pm, long long max_pivots,
                      double *out, int *status, int *pivots, void *workspace, const PlanArgs<PLAN> &plan,
                      cudaStream_t st)
{
    unsigned long long *counter = (unsigned long long *)workspace;
    double *art = (double *)((char *)workspace + 128);
    emg_art_kernel<<<1, 1024, 0, st>>>(cost, K, art);
    PILOT_LAUNCH_CHECK();
    const size_t per_warp = emg_state_bytes(K);
    int warps = (int)((200 * 1024) / per_warp);
    if (warps > 16) warps = 16;
    if (warps < 1) warps = 1;
    const size_t smem = per_warp * warps;
    PILOT_CUDA(cudaFuncSetAttribute(emd_general_kernel<PLAN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)smem));
    long long ctas = sm_count();
    const long long need = (pm.n_local + warps - 1) / warps;
    if (ctas > need) ctas = need;
    if (ctas < 1) ctas = 1;
    emd_general_kernel<PLAN><<<(unsigned)ctas, warps * 32, smem, st>>>(props, K, cost, pm, max_pivots, out, status,
                                                                      pivots, counter, art, plan);
    PILOT_LAUNCH_CHECK();
    return 0;
}

int emd_general_launch(const double *props, int K, const double *cost, const PairMap &pm, long long max_pivots,
                       double *out, int *status, int *pivots, void *workspace, cudaStream_t st)
{
    return emg_launch<false>(props, K, cost, pm, max_pivots, out, status, pivots, workspace, {}, st);
}

int emd_general_plans_launch(const double *props, int K, const double *cost, const PairMap &pm, long long max_pivots,
                             double *out, int *status, void *workspace, const PlanArgs<true> &plan, cudaStream_t st)
{
    return emg_launch<true>(props, K, cost, pm, max_pivots, out, status, nullptr, workspace, plan, st);
}

}  // namespace pilot
