// Shared helpers for the pilot_b200 CUDA translation units (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/pilot_b200.h"

namespace pilot {

void set_error(const char *fmt, ...);

#define PILOT_CHECK_ARG(cond, ...)                     \
    do {                                               \
        if (!(cond)) {                                 \
            ::pilot::set_error(__VA_ARGS__);           \
            return -1;                                 \
        }                                              \
    } while (0)

#define PILOT_CUDA(call)                                                            \
    do {                                                                            \
        cudaError_t e_ = (call);                                                    \
        if (e_ != cudaSuccess) {                                                    \
            ::pilot::set_error("%s:%d %s: %s", __FILE__, __LINE__, #call,           \
                               cudaGetErrorString(e_));                             \
            return (int)e_;                                                         \
        }                                                                           \
    } while (0)

// every kernel launch of the library is followed by this: it also feeds pilot_launch_count()
#define PILOT_LAUNCH_CHECK()                \
    do {                                    \
        ::pilot::count_launch();            \
        PILOT_CUDA(cudaGetLastError());     \
    } while (0)

int sm_count();
void count_launch();

// ---- pair-space mapping (SURVEY.md 8e) -----------------------------------
struct PairMap {
    long long total, block, first;
    int nranks, rank, mode, S;
    long long n_local;
    // FULL and RECT rows: g = i*row_len + (j - col0).  FULL: (S, 0), RECT: (S - S_a, S_a); UPPER: (S, 0), the
    // dense matrix's row length
    int row_len, col0;
};

__host__ __device__ inline long long range_count(long long total, long long block, int nranks, int rank)
{
    if (total <= 0) return 0;
    long long nblocks = (total + block - 1) / block;
    long long full = nblocks / nranks;           // every rank has at least `full` blocks
    long long mine = full + ((nblocks % nranks) > rank ? 1 : 0);
    if (mine == 0) return 0;
    long long last_block = (mine - 1) * (long long)nranks + rank;  // my last block id
    long long cnt = mine * block;
    if (last_block == nblocks - 1) cnt -= (nblocks * block - total);
    return cnt;
}

__device__ __forceinline__ long long local_to_global(const PairMap &pm, long long l)
{
    long long lb = l / pm.block, off = l - lb * pm.block;
    return (lb * pm.nranks + pm.rank) * pm.block + off;
}

// strictly-upper-triangular row-major index -> (i, j), i < j
__device__ __forceinline__ void upper_to_ij(long long g, int S, int &i, int &j)
{
    // rows before i hold i*(2S-i-1)/2 entries
    double Sd = (double)S;
    double disc = (2.0 * Sd - 1.0) * (2.0 * Sd - 1.0) - 8.0 * (double)g;
    long long ii = (long long)(((2.0 * Sd - 1.0) - sqrt(disc)) * 0.5);
    if (ii < 0) ii = 0;
    if (ii > S - 2) ii = S - 2;
    while (ii * (2LL * S - ii - 1) / 2 > g) --ii;
    while ((ii + 1) * (2LL * S - ii - 2) / 2 <= g) ++ii;
    long long base = ii * (2LL * S - ii - 1) / 2;
    i = (int)ii;
    j = (int)(g - base + ii + 1);
}

// g counts from the start of the window [first, first + total)
__device__ __forceinline__ void global_to_ij(const PairMap &pm, long long g, int &i, int &j)
{
    g += pm.first;
    if (pm.mode != PILOT_PAIRS_UPPER) {  // FULL, RECT
        i = (int)(g / pm.row_len);
        j = pm.col0 + (int)(g - (long long)i * pm.row_len);
    } else {
        upper_to_ij(g, pm.S, i, j);
    }
}

int make_pair_map(const pilot_pair_range *r, int S, PairMap *pm);

// ---- transport plans (pilot_emd_plans, pilot_sinkhorn_plans) ------------------
// The extra arguments of a solver's plan variant: problem l is (a = props[pair_a[l]], b = props[pair_b[l]]) and its
// K x K plan goes to plans + l*K*K, row-major (rows: a's types).  The instances without a plan take the empty
// specialisation, so that their parameters and their code stay exactly as they were.
template <bool PLAN> struct PlanArgs {};
template <> struct PlanArgs<true> {
    const int *pair_a, *pair_b;
    int S;
    double *plans;
};

// (si, sj) of problem l; false when an index lies outside [0, S): that problem reads nothing and gets a NaN plan,
// a NaN cost and PILOT_ST_NUMERIC
__device__ __forceinline__ bool plan_pair(const PlanArgs<true> &pa, long long l, int &si, int &sj)
{
    si = pa.pair_a[l];
    sj = pa.pair_b[l];
    return si >= 0 && si < pa.S && sj >= 0 && sj < pa.S;
}
constexpr long long PILOT_NAN_BITS = 0x7ff8000000000000LL;

// the pair map of a plan call: n problems, l = 0..n-1 (no pair space behind it)
inline PairMap plan_pair_map(long long n, int S)
{
    PairMap pm{};
    pm.total = n;
    pm.block = n > 0 ? n : 1;
    pm.nranks = 1;
    pm.S = S;
    pm.n_local = n;
    return pm;
}

// ---- warp helpers -----------------------------------------------------------
__device__ __forceinline__ double shfl_d(double v, int src)
{
    return __shfl_sync(0xffffffffu, v, src);
}
__device__ __forceinline__ double warp_sum_d(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_max_d(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

}  // namespace pilot
