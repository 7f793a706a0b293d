// Kernel (3), reference-form variant: stabilised Sinkhorn with a PER-PROBLEM Gibbs
// kernel kept in shared memory, following the reference schedule statement by
// statement (ot.sinkhorn2(..., method="sinkhorn_stabilized") reached from
// pilotpy/tools/Trajectory.py:515; schedule in SURVEY.md Appendix A.2):
//   v = b/(K^T u); u = a/(K v); absorb into alpha/beta when max|u|,|v| > tau and
//   rebuild K = exp(-(M - alpha - beta)/reg); every `check_every` iterations
//   err = || sum_i exp(-(M-alpha-beta)/reg + log u + log v) - b ||_2 ; stop on
//   err <= stop_thr; NaN -> roll back to the previous (u, v); cap num_iter_max;
//   result sum(M * Gamma).
// One CTA of roundup(K, 32) >= 64 threads per problem (thread t owns row t and column t),
// persistent CTAs pulling problems from a global counter.  Up to K ~ 155 the Gibbs matrix sits in shared memory;
// above, each CTA keeps it in its own slice of the workspace (GK), at most one CTA per SM so that the slices
// stay few (K = 256: 514 KB each, 78 MB on 148 SMs, which should mostly stay in the 126 MB L2; not measured).
// This is the always-valid path: the batched shared-kernel solvers (sinkhorn_batched.cu, sinkhorn_wide.cu) hand
// it the problems they cannot represent.
#include "sinkhorn.cuh"

namespace pilot {

constexpr int SKR_MAX_WARPS = 8;   // K <= 256 by construction
constexpr size_t SKR_SMEM_MAX = 200 * 1024;  // larger Gibbs matrices go to the workspace
constexpr int SKR_SCAN = 256;      // problems per work item of the marker scan (mode 2)

static int skr_threads(int K) { return K <= 64 ? 64 : ((K + 31) / 32) * 32; }

// block reductions over the blockDim.x / 32 warps (2 for K <= 64), summed / maxed in warp order
__device__ __forceinline__ double block_max64(double v, double *red)
{
    v = warp_max_d(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double r = red[0];
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) r = fmax(r, red[w]);
    return r;
}
__device__ __forceinline__ double block_sum64(double v, double *red)
{
    v = warp_sum_d(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double r = red[0];
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) r += red[w];
    return r;
}

// mode 0: every local problem; mode 1: the problems of the redo list (at most max_list of them); mode 2: only if
// more than max_list problems were queued (the list overflowed): scan out[] for the redo marker the fast
// kernels left behind and solve those (the listed ones were overwritten by mode 1 already).
// GK: the Gibbs matrix lives in the CTA's slice of `gibbs` (K x (K | 1) doubles) instead of shared memory.
// PLAN (mode 0 only): problems from the pair list of `plan`; thread t writes column t of Gamma in the loop that
// accumulates the cost, so the plan sums, in that order, to out[l].
template <bool GK, bool PLAN = false>
__global__ void __launch_bounds__(SKR_MAX_WARPS * 32)
sinkhorn_ref_kernel(const double *__restrict__ props, int K, const double *__restrict__ M, SkParams prm,
                    PairMap pm, int mode, const long long *__restrict__ list,
                    const unsigned long long *__restrict__ n_list_dev, long long max_list,
                    double *__restrict__ out, int *__restrict__ iters_out, int *__restrict__ abs_out,
                    int *__restrict__ status_out, unsigned long long *__restrict__ counter, double *gibbs,
                    PlanArgs<PLAN> plan)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int KS = K | 1;  // odd row stride: row- and column-walks are both conflict-free
    double *Km = GK ? gibbs + (size_t)blockIdx.x * K * KS : reinterpret_cast<double *>(smem_raw);
    double *u = GK ? reinterpret_cast<double *>(smem_raw) : Km + (size_t)K * KS, *v = u + K, *up = v + K, *vp = up + K;
    double *al = vp + K, *be = al + K, *lu = be + K, *lv = lu + K, *red = lv + K;
    __shared__ long long s_l;
    __shared__ int s_nfound;
    __shared__ int s_found[SKR_SCAN];
    const int t = threadIdx.x;
    const int NT = blockDim.x;
    const bool act = t < K;
    long long n_work = pm.n_local;
    if (mode == 1) {
        n_work = (long long)*n_list_dev;
        if (n_work > max_list) n_work = max_list;
    } else if (mode == 2) {
        if ((long long)*n_list_dev <= max_list) return;
        n_work = (pm.n_local + SKR_SCAN - 1) / SKR_SCAN;
    }
    const double reg = prm.reg;
    int scan_pos = 0, scan_n = 0;
    long long scan_base = 0;

    for (;;) {
        long long l;
        if (mode == 2) {
            // next marked problem of the current chunk, else fetch and scan the next chunk
            while (scan_pos >= scan_n) {
                __syncthreads();
                if (t == 0) { s_l = (long long)atomicAdd(counter, 1ULL); s_nfound = 0; }
                __syncthreads();
                if (s_l >= n_work) return;
                scan_base = s_l * SKR_SCAN;
                for (int e = t; e < SKR_SCAN; e += NT) {
                    const long long q = scan_base + e;
                    if (q < pm.n_local && __double_as_longlong(out[q]) == SK_REDO_MARK)
                        s_found[atomicAdd(&s_nfound, 1)] = e;
                }
                __syncthreads();
                scan_n = s_nfound;
                scan_pos = 0;
            }
            l = scan_base + s_found[scan_pos++];
        } else {
            __syncthreads();
            if (t == 0) s_l = (long long)atomicAdd(counter, 1ULL);
            __syncthreads();
            const long long w = s_l;
            if (w >= n_work) break;
            l = mode == 1 ? list[w] : w;
        }
        int si, sj;
        if constexpr (PLAN) {
            if (!plan_pair(plan, l, si, sj)) {
                double *g = plan.plans + l * K * K;
                for (int e = t; e < K * K; e += NT) g[e] = __longlong_as_double(PILOT_NAN_BITS);
                if (t == 0) {
                    out[l] = __longlong_as_double(PILOT_NAN_BITS);
                    if (iters_out) iters_out[l] = 0;
                    if (abs_out) abs_out[l] = 0;
                    if (status_out) status_out[l] = PILOT_ST_NUMERIC;
                }
                continue;
            }
        } else {
            global_to_ij(pm, local_to_global(pm, l), si, sj);
        }
        const double a = act ? props[(long long)si * K + t] : 0.0;
        const double b = act ? props[(long long)sj * K + t] : 0.0;
        if (act) { al[t] = 0.0; be[t] = 0.0; u[t] = 1.0 / K; v[t] = 1.0 / K; }
        for (int e = t; e < K * K; e += NT) {
            const int i = e / K, j = e - i * K;
            Km[i * KS + j] = exp(-(__ldg(M + e)) / reg);
        }
        __syncthreads();
        double err = 1.0;
        int n_abs = 0, status = PILOT_ST_MAXITER, ii = 0;
        for (; ii < prm.num_iter_max; ++ii) {
            if (act) { up[t] = u[t]; vp[t] = v[t]; }
            // v = b / (K^T u)
            if (act) {
                double s = 0.0;
                for (int i = 0; i < K; ++i) s += Km[i * KS + t] * u[i];
                v[t] = b / s;
            }
            __syncthreads();
            // u = a / (K v)
            if (act) {
                double s = 0.0;
                for (int j = 0; j < K; ++j) s += Km[t * KS + j] * v[j];
                u[t] = a / s;
            }
            __syncthreads();
            // np.max(np.abs(x)) propagates NaN and `NaN > tau` is False: a vector holding a NaN
            // cannot trigger the absorption by itself, but the other vector still can.
            const double mu = block_max64(act ? fabs(u[t]) : 0.0, red);
            const double mv = block_max64(act ? fabs(v[t]) : 0.0, red);
            const bool nan_u = block_max64(act && u[t] != u[t] ? 1.0 : 0.0, red) > 0.0;
            const bool nan_v = block_max64(act && v[t] != v[t] ? 1.0 : 0.0, red) > 0.0;
            bool anynan = nan_u || nan_v;
            if ((!nan_u && mu > prm.tau) || (!nan_v && mv > prm.tau)) {
                if (act) {
                    al[t] += reg * log(u[t]);
                    be[t] += reg * log(v[t]);
                    u[t] = 1.0 / K;
                    v[t] = 1.0 / K;
                }
                anynan = false;  // u, v were just reset; the reference's NaN test sees the reset vectors
                __syncthreads();
                for (int e = t; e < K * K; e += NT) {
                    const int i = e / K, j = e - i * K;
                    Km[i * KS + j] = exp(-(__ldg(M + e) - al[i] - be[j]) / reg);
                }
                ++n_abs;
                __syncthreads();
            }
            if (ii % prm.check_every == 0) {
                if (act) { lu[t] = log(u[t]); lv[t] = log(v[t]); }
                __syncthreads();
                double d = 0.0;
                if (act) {
                    double cs = 0.0;
                    const double bj = be[t], lvj = lv[t];
                    for (int i = 0; i < K; ++i)
                        cs += exp(-(__ldg(M + i * K + t) - al[i] - bj) / reg + lu[i] + lvj);
                    d = cs - b;
                }
                err = sqrt(block_sum64(d * d, red));
            }
            if (err <= prm.stop_thr) { status = PILOT_ST_CONVERGED; ++ii; break; }
            if (anynan) {
                if (act) { u[t] = up[t]; v[t] = vp[t]; }
                status = PILOT_ST_NUMERIC;
                ++ii;
                break;
            }
        }
        __syncthreads();
        if (act) { lu[t] = log(u[t]); lv[t] = log(v[t]); }
        __syncthreads();
        double c = 0.0;
        if (act) {
            const double bj = be[t], lvj = lv[t];
            for (int i = 0; i < K; ++i) {
                const double m = __ldg(M + i * K + t);
                const double g = exp(-(m - al[i] - bj) / reg + lu[i] + lvj);
                if constexpr (PLAN) plan.plans[l * K * K + i * K + t] = g;
                c += m * g;
            }
        }
        c = block_sum64(c, red);
        if (t == 0) {
            out[l] = c;
            if (iters_out) iters_out[l] = ii;
            if (abs_out) abs_out[l] = n_abs;
            if (status_out) status_out[l] = status;
        }
    }
}

size_t sinkhorn_ref_smem(int K)
{
    const int KS = K | 1;
    return sizeof(double) * ((size_t)K * KS + 8 * (size_t)K + SKR_MAX_WARPS);
}
static bool skr_global_gibbs(int K) { return sinkhorn_ref_smem(K) > SKR_SMEM_MAX; }
size_t sinkhorn_ref_gibbs_bytes(int K)
{
    return skr_global_gibbs(K) ? sizeof(double) * (size_t)sm_count() * K * (K | 1) : 0;
}

template <bool PLAN>
static int skr_launch(const double *props, int K, const double *cost, const SkParams &prm, const PairMap &pm,
                      const SkOut &res, long long redo_cap, unsigned long long *counter, double *gibbs,
                      const PlanArgs<PLAN> &plan, cudaStream_t st)
{
    const bool queued = redo_cap != SK_SOLVE_ALL;
    // with a device-side list the amount of work is unknown here: launch one wave and let the CTAs loop
    const long long n_work = queued ? (long long)sm_count() * 4 : pm.n_local;
    if (n_work <= 0) return 0;
    const bool gk = skr_global_gibbs(K);
    PILOT_CHECK_ARG(!gk || gibbs, "sinkhorn reference-form kernel: K=%d needs a Gibbs workspace", K);
    const size_t smem = gk ? sizeof(double) * (8 * (size_t)K + SKR_MAX_WARPS) : sinkhorn_ref_smem(K);
    const int threads = skr_threads(K);
    PILOT_CHECK_ARG(threads <= SKR_MAX_WARPS * 32, "sinkhorn reference-form kernel: K=%d too large", K);
    const auto kern = gk ? sinkhorn_ref_kernel<true, PLAN> : sinkhorn_ref_kernel<false, PLAN>;
    PILOT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    PILOT_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem));
    if (per_sm < 1 || gk) per_sm = 1;  // gibbs holds one slice per SM
    long long ctas = (long long)sm_count() * per_sm;
    if (ctas > n_work) ctas = n_work;
    // modes 1 and 2 run back to back on the stream and share the counter: reset it before each
    for (int mode = queued ? 1 : 0; mode <= (queued ? 2 : 0); ++mode) {
        PILOT_CUDA(cudaMemsetAsync(counter, 0, sizeof(unsigned long long), st));
        kern<<<(unsigned)ctas, threads, smem, st>>>(props, K, cost, prm, pm, mode, res.redo, res.n_redo, redo_cap,
                                                    res.out, res.iters, res.absn, res.status, counter, gibbs,
                                                    plan);
        PILOT_LAUNCH_CHECK();
    }
    return 0;
}

int sinkhorn_ref_launch(const double *props, int K, const double *cost, const SkParams &prm, const PairMap &pm,
                        const SkOut &res, long long redo_cap, unsigned long long *counter, double *gibbs,
                        cudaStream_t st)
{
    return skr_launch<false>(props, K, cost, prm, pm, res, redo_cap, counter, gibbs, {}, st);
}

int sinkhorn_ref_plans_launch(const double *props, int K, const double *cost, const SkParams &prm,
                              const PairMap &pm, const SkOut &res, const PlanArgs<true> &plan,
                              unsigned long long *counter, double *gibbs, cudaStream_t st)
{
    return skr_launch<true>(props, K, cost, prm, pm, res, SK_SOLVE_ALL, counter, gibbs, plan, st);
}

}  // namespace pilot
