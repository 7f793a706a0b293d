// Kernel (3), FP32 mode (north_star's 1e-4 tier): all-pairs stabilised Sinkhorn in single precision.
// Replaces the loop over ot.sinkhorn2(a_i, a_j, cost, reg, method="sinkhorn_stabilized")
// (reference pilotpy/tools/Trajectory.py:513-515; schedule: SURVEY.md Appendix A.2).
//
// Why not the FP64 kernels' shared-Gibbs-kernel form: K0 = exp(-M/reg) itself underflows in float at
// reg = 0.01 (e^-100), and so do the scaled iterates e^{alpha/reg} u.  This kernel therefore keeps POT's own
// form -- a PER-PROBLEM kernel K = exp(-(M - alpha - beta)/reg), rebuilt at every absorption, whose entries
// are bounded because alpha, beta absorb the growth -- and makes it fast by holding K in REGISTERS:
//   * one warp per problem; the lanes form a 4 x 8 grid, lane (r, c) owns the K tile of KP/4 rows x KP/8
//     columns (KP = 64: 16 x 8 = 128 registers)
//   * t = K^T u: each lane multiplies its tile by its 16 entries of u, then a reduce-scatter over the 4 lanes
//     of a column group (2 butterfly steps) leaves every lane with the 2 column sums it owns
//   * s = K v: same with its 8 entries of v and a reduce-scatter over the 8 lanes of a row group (3 steps);
//     lane l ends up owning rows 2l, 2l+1
//   * the owned entries of u / v travel to the lanes that need them through a 256-byte shared buffer
//   * exponentials are exp2 of pre-scaled quantities (A = alpha log2e/reg, Ms = M log2e/reg): K = 2^(A_i+B_j-Ms_ij)
//   * same schedule as POT: v then u, absorption test after the update, marginal error every `check_every`
//     iterations (taken from the next iteration's K^T u, which is the same number), cap num_iter_max.
//     The stop threshold is raised to what float resolves (5e-7 against the 1e-9 default).
//   * a problem that produces NaN/Inf is handed to the FP64 reference-form kernel (sinkhorn_ref.cu)
// Per iteration and problem: 2 KP^2 FFMA-class + ~100 other warp instructions -- issue bound on the FP32 pipe.
#include "sinkhorn.cuh"

namespace pilot {

constexpr int SKF_WARPS = 8;
constexpr unsigned SKF_FULL = 0xffffffffu;
constexpr float SKF_MIN_THR = 5e-7f;

template <int KP> struct SkfShape {
    static constexpr int TR = KP / 4;    // tile rows per lane
    static constexpr int TC = KP / 8;    // tile columns per lane
    static constexpr int NV = KP / 32;   // owned vector entries per lane (rows NV*lane + e; columns TC*c + NV*r + e)
};

// reduce-scatter of x[0..N) over the lanes {lane ^ o : o in the given offsets}: after the call x[0..N/steps)
// holds the sums of the elements this lane owns.  Offsets from HI down to LO (powers of two).
template <int N, int HI, int LO> __device__ __forceinline__ void reduce_scatter(float (&x)[N], int lane)
{
    int n = N;
#pragma unroll
    for (int o = HI; o >= LO; o >>= 1) {
        const bool hi = (lane & o) != 0;
        n >>= 1;
#pragma unroll
        for (int k = 0; k < N / 2; ++k) {
            if (k < n) {
                const float keep = hi ? x[k + n] : x[k];
                const float send = hi ? x[k] : x[k + n];
                x[k] = keep + __shfl_xor_sync(SKF_FULL, send, o);
            }
        }
    }
}

__device__ __forceinline__ float fdiv_fast(float x, float y)
{
    // x / y for finite positive y: reciprocal seed + one Newton step on the quotient (error ~1 ulp)
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(y));
    const float q = x * r;
    return fmaf(fmaf(-y, q, x), r, q);
}

template <int KP>
__global__ void __launch_bounds__(SKF_WARPS * 32, 1)
sinkhorn_f32_kernel(const double *__restrict__ props, int K, const double *__restrict__ M, SkParams prm, PairMap pm,
                    unsigned long long *__restrict__ counter, double *__restrict__ out, int *__restrict__ iters_out,
                    int *__restrict__ abs_out, int *__restrict__ status_out, long long *__restrict__ redo_list,
                    unsigned long long *__restrict__ n_redo)
{
    const SkOut res{out, iters_out, abs_out, status_out, redo_list, n_redo};
    using S = SkfShape<KP>;
    constexpr int TR = S::TR, TC = S::TC, NV = S::NV;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *sMs = reinterpret_cast<float *>(smem_raw);  // M * log2e / reg, KP x KP row-major, +inf padded
    float *sK0 = sMs + KP * KP;                        // 2^-Ms (0 in the padding)
    float *sw = sK0 + KP * KP + (threadIdx.x >> 5) * 4 * KP;
    float *su = sw, *sv = sw + KP, *sA = sw + 2 * KP, *sB = sw + 3 * KP;
    const int lane = threadIdx.x & 31;
    const int r = lane >> 3, c = lane & 7;
    const float unscale = (float)(prm.reg / 1.4426950408889634);

    for (int e = threadIdx.x; e < KP * KP; e += blockDim.x) {
        const int i = e / KP, j = e - i * KP;
        const bool in = i < K && j < K;
        const float ms = in ? (float)(M[i * K + j] * (1.4426950408889634 / prm.reg)) : __int_as_float(0x7f800000);
        sMs[e] = ms;
        sK0[e] = in ? exp2f(-ms) : 0.0f;
    }
    __syncthreads();

    const float invK = 1.0f / (float)K;
    const float thr = fmaxf((float)prm.stop_thr, SKF_MIN_THR);
    const float tau = (float)prm.tau;
    const int row0 = NV * lane;               // owned rows row0 .. row0+NV-1
    const int col0 = TC * c + NV * r;         // owned columns col0 .. col0+NV-1
    const int trow = TR * r, tcol = TC * c;   // tile origin

    for (;;) {
        unsigned long long w = 0;
        if (lane == 0) w = atomicAdd(counter, 1ULL);
        w = __shfl_sync(SKF_FULL, w, 0);
        if ((long long)w >= pm.n_local) break;
        int si, sj;
        global_to_ij(pm, local_to_global(pm, (long long)w), si, sj);

        float a[NV], b[NV], u[NV], v[NV], A[NV], B[NV];
#pragma unroll
        for (int e = 0; e < NV; ++e) {
            a[e] = row0 + e < K ? (float)props[(long long)si * K + row0 + e] : 0.0f;
            b[e] = col0 + e < K ? (float)props[(long long)sj * K + col0 + e] : 0.0f;
            u[e] = row0 + e < K ? invK : 0.0f;
            v[e] = col0 + e < K ? invK : 0.0f;
            A[e] = 0.0f;
            B[e] = 0.0f;
        }
        // K tile = K0 tile
        float Kt[TR][TC];
#pragma unroll
        for (int i = 0; i < TR; ++i)
#pragma unroll
            for (int j = 0; j < TC; j += 4) {
                const float4 q = *reinterpret_cast<const float4 *>(sK0 + (trow + i) * KP + tcol + j);
                Kt[i][j] = q.x; Kt[i][j + 1] = q.y; Kt[i][j + 2] = q.z; Kt[i][j + 3] = q.w;
            }

        int ii = 0, nabs = 0, status = PILOT_ST_MAXITER;
        int until_check = 0;  // countdown to the next marginal check (ii % check_every == 0 without the modulo)
        bool pend = false, bad = false;
        for (;;) {
            // ---- t = K^T u ----
            __syncwarp();
#pragma unroll
            for (int e = 0; e < NV; ++e) su[row0 + e] = u[e];
            __syncwarp();
            float t[TC];
#pragma unroll
            for (int j = 0; j < TC; ++j) t[j] = 0.0f;
#pragma unroll
            for (int i = 0; i < TR; i += 4) {
                const float4 q = *reinterpret_cast<const float4 *>(su + trow + i);
                const float uu[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                for (int k = 0; k < 4; ++k)
#pragma unroll
                    for (int j = 0; j < TC; ++j) t[j] = fmaf(Kt[i + k][j], uu[k], t[j]);
            }
            reduce_scatter<TC, 16, 8>(t, lane);  // t[0..NV) = column sums of the owned columns
            // ---- resolve the pending marginal check / the iteration cap of the previous iteration ----
            if (pend || ii >= prm.num_iter_max || bad) {
                bool conv = false;
                if (pend && !bad) {
                    float e2 = 0.0f;
#pragma unroll
                    for (int e = 0; e < NV; ++e) {
                        const float d = fmaf(v[e], t[e], -b[e]);
                        e2 = fmaf(d, d, e2);
                    }
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) e2 += __shfl_xor_sync(SKF_FULL, e2, o);
                    conv = sqrtf(e2) <= thr;
                }
                if (bad) { status = -1; break; }
                if (conv) { status = PILOT_ST_CONVERGED; break; }
                if (ii >= prm.num_iter_max) { status = PILOT_ST_MAXITER; break; }
            }
            // ---- v = b / t ----
            unsigned mx = 0u;
#pragma unroll
            for (int e = 0; e < NV; ++e) {
                v[e] = col0 + e < K ? fdiv_fast(b[e], t[e]) : 0.0f;
                mx = max(mx, __float_as_uint(v[e]) & 0x7fffffffu);  // |v|: NaN / Inf sort above every finite value
            }
            __syncwarp();
#pragma unroll
            for (int e = 0; e < NV; ++e) sv[col0 + e] = v[e];
            __syncwarp();
            // ---- s = K v ----
            float s[TR];
            {
                float vv[TC];
#pragma unroll
                for (int j = 0; j < TC; j += 4) {
                    const float4 q = *reinterpret_cast<const float4 *>(sv + tcol + j);
                    vv[j] = q.x; vv[j + 1] = q.y; vv[j + 2] = q.z; vv[j + 3] = q.w;
                }
#pragma unroll
                for (int i = 0; i < TR; ++i) {
                    float acc = Kt[i][0] * vv[0];
#pragma unroll
                    for (int j = 1; j < TC; ++j) acc = fmaf(Kt[i][j], vv[j], acc);
                    s[i] = acc;
                }
            }
            reduce_scatter<TR, 4, 1>(s, lane);  // s[0..NV) = row sums of the owned rows
            // ---- u = a / s ; absorption test (max|u|, max|v| > tau), NaN / Inf test ----
#pragma unroll
            for (int e = 0; e < NV; ++e) {
                u[e] = row0 + e < K ? fdiv_fast(a[e], s[e]) : 0.0f;
                mx = max(mx, __float_as_uint(u[e]) & 0x7fffffffu);
            }
            mx = __reduce_max_sync(SKF_FULL, mx);
            bad = mx >= 0x7f800000u;
            pend = until_check == 0;
            until_check = pend ? prm.check_every - 1 : until_check - 1;
            ++ii;
            if (!bad && mx > __float_as_uint(tau)) {
                // alpha += reg log u, beta += reg log v (kept as A = alpha log2e / reg), u = v = 1/K, rebuild K
                bool under = false;
#pragma unroll
                for (int e = 0; e < NV; ++e) {
                    if (row0 + e < K) { under |= !(u[e] > 0.0f); A[e] += log2f(u[e]); u[e] = invK; }
                    if (col0 + e < K) { under |= !(v[e] > 0.0f); B[e] += log2f(v[e]); v[e] = invK; }
                }
                bad = __any_sync(SKF_FULL, under);  // a zero (zero mass, underflow): log = -inf -> POT's NaN path
                ++nabs;
                __syncwarp();
#pragma unroll
                for (int e = 0; e < NV; ++e) { sA[row0 + e] = A[e]; sB[col0 + e] = B[e]; }
                __syncwarp();
                float Bt[TC];
#pragma unroll
                for (int j = 0; j < TC; ++j) Bt[j] = sB[tcol + j];
#pragma unroll
                for (int i = 0; i < TR; ++i) {
                    const float Ai = sA[trow + i];
#pragma unroll
                    for (int j = 0; j < TC; ++j) Kt[i][j] = exp2f((Ai + Bt[j]) - sMs[(trow + i) * KP + tcol + j]);
                }
            }
        }

        float acc = 0.0f;
        if (status >= 0) {
            // cost = sum_ij M_ij u_i K_ij v_j with the state at the stop (su holds u, v is current)
            __syncwarp();
#pragma unroll
            for (int e = 0; e < NV; ++e) sv[col0 + e] = v[e];
            __syncwarp();
#pragma unroll
            for (int i = 0; i < TR; ++i) {
                const int gi = trow + i;
                if (gi < K) {
                    float rowacc = 0.0f;
#pragma unroll
                    for (int j = 0; j < TC; ++j)
                        if (tcol + j < K) rowacc = fmaf(Kt[i][j] * sMs[gi * KP + tcol + j], sv[tcol + j], rowacc);
                    acc = fmaf(rowacc, su[gi], acc);
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(SKF_FULL, acc, o);
        }
        if (lane == 0) sk_store(res, (long long)w, status, (double)(acc * unscale), ii, nabs);
        __syncwarp();
    }
}

template <int KP>
static int skf_launch_t(const double *props, int K, const double *cost, const SkParams &prm, const PairMap &pm,
                        const SkOut &res, unsigned long long *counter, cudaStream_t st)
{
    const size_t smem = sizeof(float) * ((size_t)2 * KP * KP + (size_t)SKF_WARPS * 4 * KP);
    PILOT_CUDA(cudaFuncSetAttribute(sinkhorn_f32_kernel<KP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    long long ctas = (pm.n_local + SKF_WARPS - 1) / SKF_WARPS;
    if (ctas > sm_count()) ctas = sm_count();
    if (ctas < 1) ctas = 1;
    sinkhorn_f32_kernel<KP><<<(unsigned)ctas, SKF_WARPS * 32, smem, st>>>(props, K, cost, prm, pm, counter, res.out,
                                                                         res.iters, res.absn, res.status, res.redo,
                                                                         res.n_redo);
    PILOT_LAUNCH_CHECK();
    return 0;
}

int skf_launch(const double *props, int K, const double *cost, const SkParams &prm, const PairMap &pm,
               const SkOut &res, unsigned long long *counter, cudaStream_t st)
{
    if (K <= 32) return skf_launch_t<32>(props, K, cost, prm, pm, res, counter, st);
    return skf_launch_t<64>(props, K, cost, prm, pm, res, counter, st);
}

}  // namespace pilot
