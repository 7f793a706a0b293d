// Kernel (5): packed per-rank results -> dense S x S matrix (EMD[i, j], i = row sample),
// mirroring the upper triangle for the symmetric exact-EMD case, or the dense S_a x S_b block of
// the RECT pair space (never mirrored: its rows and columns are different samples).  Replaces the NumPy
// element assignments EMD[i, j] = ... of the reference loop (pilotpy/tools/Trajectory.py:511,515).
// HBM-bound: 8 B read + 8 (or 16) B written per problem.
#include "common.cuh"

namespace pilot {

__global__ void unpack_kernel(const double *__restrict__ packed, long long chunk_stride, PairMap pm,
                              double diag_value, double *__restrict__ dense)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    const int S = pm.S;
    for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < pm.total; g += stride) {
        const long long b = g / pm.block, off = g - b * pm.block;
        const int owner = (int)(b % pm.nranks);
        const long long local = (b / pm.nranks) * pm.block + off;
        const double v = packed[(long long)owner * chunk_stride + local];
        int i, j;
        global_to_ij(pm, g, i, j);
        dense[(long long)i * pm.row_len + (j - pm.col0)] = v;
        if (pm.mode == PILOT_PAIRS_UPPER) dense[(long long)j * S + i] = v;
    }
    if (pm.mode == PILOT_PAIRS_UPPER)
        for (long long d = (long long)blockIdx.x * blockDim.x + threadIdx.x; d < S; d += stride)
            dense[d * S + d] = diag_value;
}

}  // namespace pilot

extern "C" int pilot_unpack_pairs(const double *packed, int64_t chunk_stride, int S, const pilot_pair_range *range,
                                  double diag_value, double *dense, void *stream)
{
    using namespace pilot;
    PILOT_CHECK_ARG(packed && dense && S >= 1, "pilot_unpack_pairs: bad argument");
    PairMap pm;
    int rc = make_pair_map(range, S, &pm);
    if (rc) return rc;
    long long work = pm.total > S ? pm.total : S;
    long long blocks = (work + 255) / 256;
    const long long cap = (long long)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    unpack_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(packed, chunk_stride, pm, diag_value, dense);
    PILOT_LAUNCH_CHECK();
    return 0;
}
