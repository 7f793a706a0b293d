// Kernel (2a): per-(cell type, dimension) MEDIAN of the embedding rows, in the
// input dtype.  Replaces data[annot.cell_type == k].median(axis=0)
// (reference pilotpy/tools/Trajectory.py:465-466; pandas nanmedian semantics:
// NaNs ignored, even counts -> (lo + hi) / 2 rounded in the input dtype).
//
// Two exact paths, chosen by median_path (end of this file):
//  * sampled-pivot streaming path (n >= 64K rows; second half of this file):
//    a hashed sample of ~2048-4096 rows per type gives, per (type, dim), two pivots lo <= hi that bracket the
//    median with ~4e-8 failure odds; ONE pass over X then counts x < lo and collects the ~10 % of elements
//    inside the bracket in per-pair lists (mn_stream_run_kernel: a CTA counting-sorts the row ids of a chunk
//    of <= 4096 rows by type in shared memory, so that a lane walks rows of ONE type with its pivots in
//    registers); a one-CTA-per-pair kernel finishes the selection inside the list.  If a pair's rank falls
//    outside its bracket (or its list overflows) the same CTA falls back to an exact radix select over
//    the type's rows -- no host round trip, results are always exact.
//    HBM traffic: one read of X + ~6 % for the sample + the lists (written once, read once).
//  * most-significant-digit radix select (every other input: fewer rows, a large K*D, more types than the stream
//    pass's shared memory holds, rows 1 MiB or more apart): every pass streams X once
//    and histograms the current 8-bit digit of the elements whose higher digits match the
//    running prefix of their (type, dim) query; 4 passes for f32, 8 for f64.
// Two queries per (type, dim) (ranks (n-1)/2 and n/2) so even counts need no second selection.
//
// Algorithmic bytes (SURVEY.md 8d): one read of X + codes.
#include <type_traits>
#include "common.cuh"

namespace pilot {

template <typename T> struct KeyOf;
template <> struct KeyOf<float> {
    using type = unsigned int;
    static constexpr int PASSES = 4;
    __device__ static unsigned int key(float x)
    {
        unsigned int u = __float_as_uint(x);
        return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
    }
    __device__ static float value(unsigned int k)
    {
        unsigned int u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
        return __uint_as_float(u);
    }
};
template <> struct KeyOf<double> {
    using type = unsigned long long;
    static constexpr int PASSES = 8;
    __device__ static unsigned long long key(double x)
    {
        unsigned long long u = (unsigned long long)__double_as_longlong(x);
        return (u >> 63) ? ~u : (u | 0x8000000000000000ULL);
    }
    __device__ static double value(unsigned long long k)
    {
        unsigned long long u = (k >> 63) ? (k & 0x7fffffffffffffffULL) : ~k;
        return __longlong_as_double((long long)u);
    }
};

struct MedianWs {
    unsigned int *hist;                          // KD * 2 * 256
    unsigned long long *prefix, *rank, *nvalid;  // KD * 2 keys (stored as u64), KD * 2, KD
};

// the radix path's workspace (all 8-byte aligned)
struct MedianLayout {
    MedianWs ws;
    size_t hist_bytes;  // zeroed before every pass
    size_t bytes;       // end of the last region
};

// carves the radix path's workspace at `base` (nullptr: only its size)
static MedianLayout median_workspace(void *base, int K, int D)
{
    const size_t kd = (size_t)K * D;
    uintptr_t p = (uintptr_t)base;
    const auto take = [&p](size_t bytes) { const uintptr_t r = p; p += bytes; return r; };
    MedianLayout l;
    l.hist_bytes = kd * 2 * 256 * sizeof(unsigned int);
    l.ws.hist = (unsigned int *)take(l.hist_bytes);
    l.ws.prefix = (unsigned long long *)take(kd * 2 * 8);
    l.ws.rank = (unsigned long long *)take(kd * 2 * 8);
    l.ws.nvalid = (unsigned long long *)take(kd * 8);
    l.bytes = p - (uintptr_t)base;
    return l;
}

template <typename T, int PASS>
__global__ void __launch_bounds__(256)
median_hist_kernel(const T *__restrict__ X, long long n, int D, long long ldx, const int *__restrict__ code,
                   int K, MedianWs ws)
{
    using KO = KeyOf<T>;
    using Key = typename KO::type;
    constexpr int BITS = sizeof(Key) * 8;
    constexpr int SHIFT = BITS - 8 * (PASS + 1);
    const long long total = n * D;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
        const long long r = e / D;
        const int d = (int)(e - r * D);
        const int k = __ldg(code + r);
        if ((unsigned)k >= (unsigned)K) continue;
        const T x = X[r * ldx + d];
        if (x != x) continue;  // nanmedian ignores NaN
        const Key key = KO::key(x);
        const int kd = k * D + d;
        const unsigned digit = (unsigned)(key >> SHIFT) & 0xffu;
        if constexpr (PASS == 0) {
            atomicAdd(&ws.hist[((size_t)kd * 2) * 256 + digit], 1u);
        } else {
            const Key hi = (Key)(key >> (SHIFT + 8));
            const Key p0 = (Key)ws.prefix[kd * 2] >> (SHIFT + 8);
            const Key p1 = (Key)ws.prefix[kd * 2 + 1] >> (SHIFT + 8);
            if (hi == p0) atomicAdd(&ws.hist[((size_t)kd * 2) * 256 + digit], 1u);
            if (hi == p1) atomicAdd(&ws.hist[((size_t)kd * 2 + 1) * 256 + digit], 1u);
        }
    }
}

// one warp per (kd, q)
template <typename T, int PASS>
__global__ void median_scan_kernel(int KD, MedianWs ws)
{
    using Key = typename KeyOf<T>::type;
    constexpr int BITS = sizeof(Key) * 8;
    constexpr int SHIFT = BITS - 8 * (PASS + 1);
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= KD * 2) return;
    const int kd = w >> 1, q = w & 1;
    unsigned int *h = ws.hist + ((size_t)kd * 2 + (PASS == 0 ? 0 : q)) * 256;
    unsigned int c[8];
    unsigned int mine = 0;
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        c[t] = h[lane * 8 + t];
        mine += c[t];
    }
    // inclusive warp scan of per-lane totals
    unsigned int incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        unsigned int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    const unsigned int total = __shfl_sync(0xffffffffu, incl, 31);
    unsigned long long rank;
    if (PASS == 0) {
        if (lane == 0 && q == 0) ws.nvalid[kd] = total;
        rank = total == 0 ? 0ULL : (q == 0 ? (unsigned long long)(total - 1) / 2 : (unsigned long long)total / 2);
    } else {
        rank = ws.rank[kd * 2 + q];
    }
    const unsigned int excl = incl - mine;
    const bool here = total > 0 && rank >= excl && rank < incl;
    if (here) {
        unsigned long long run = excl, below = 0;
        int digit = -1;
#pragma unroll
        for (int t = 0; t < 8; ++t) {
            if (digit < 0 && rank < run + c[t]) {
                digit = lane * 8 + t;
                below = run;
            }
            run += c[t];
        }
        Key p = PASS == 0 ? (Key)0 : (Key)ws.prefix[kd * 2 + q];
        p |= (Key)digit << SHIFT;
        ws.prefix[kd * 2 + q] = (unsigned long long)p;
        ws.rank[kd * 2 + q] = rank - below;
    }
    if (total == 0 && lane == 0) {
        ws.prefix[kd * 2 + q] = 0ULL;
        ws.rank[kd * 2 + q] = 0ULL;
    }
}

template <typename T>
__global__ void median_final_kernel(int KD, MedianWs ws, T *__restrict__ cent, double *__restrict__ cent64)
{
    using KO = KeyOf<T>;
    using Key = typename KO::type;
    const int kd = blockIdx.x * blockDim.x + threadIdx.x;
    if (kd >= KD) return;
    T med;
    if (ws.nvalid[kd] == 0) {
        med = (T)NAN;
    } else {
        const T lo = KO::value((Key)ws.prefix[kd * 2]);
        const T hi = KO::value((Key)ws.prefix[kd * 2 + 1]);
        if (lo == hi) med = lo;
        else if (sizeof(T) == 4) med = (T)__fdiv_rn(__fadd_rn((float)lo, (float)hi), 2.0f);
        else med = (T)__ddiv_rn(__dadd_rn((double)lo, (double)hi), 2.0);
    }
    cent[kd] = med;
    cent64[kd] = (double)med;
}

template <typename T, int PASS>
static int median_pass(const T *X, long long n, int D, long long ldx, const int *code, int K, MedianWs ws,
                       size_t hist_bytes, cudaStream_t st)
{
    PILOT_CUDA(cudaMemsetAsync(ws.hist, 0, hist_bytes, st));
    const long long total = n * D;
    long long blocks = (total + 255) / 256;
    const long long cap = (long long)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    median_hist_kernel<T, PASS><<<(unsigned)blocks, 256, 0, st>>>(X, n, D, ldx, code, K, ws);
    PILOT_LAUNCH_CHECK();
    const int KD = K * D;
    const int warps = KD * 2;
    median_scan_kernel<T, PASS><<<(warps * 32 + 255) / 256, 256, 0, st>>>(KD, ws);
    PILOT_LAUNCH_CHECK();
    return 0;
}

template <typename T>
static int median_run(const T *X, long long n, int D, long long ldx, const int *code, int K, T *cent,
                      double *cent64, void *workspace, cudaStream_t st)
{
    const size_t kd = (size_t)K * D;
    const MedianLayout l = median_workspace(workspace, K, D);
    int rc;
#define PILOT_MEDIAN_PASS(P) \
    if (KeyOf<T>::PASSES > P) { rc = median_pass<T, (P < KeyOf<T>::PASSES ? P : 0)>(X, n, D, ldx, code, K, l.ws, l.hist_bytes, st); if (rc) return rc; }
    PILOT_MEDIAN_PASS(0) PILOT_MEDIAN_PASS(1) PILOT_MEDIAN_PASS(2) PILOT_MEDIAN_PASS(3)
    PILOT_MEDIAN_PASS(4) PILOT_MEDIAN_PASS(5) PILOT_MEDIAN_PASS(6) PILOT_MEDIAN_PASS(7)
#undef PILOT_MEDIAN_PASS
    median_final_kernel<T><<<(unsigned)((kd + 127) / 128), 128, 0, st>>>((int)kd, l.ws, cent, cent64);
    PILOT_LAUNCH_CHECK();
    return 0;
}


// =====================================================================================
// sampled-pivot streaming path in NATURAL row order
// =====================================================================================
// Five small kernels around ONE pass over X:
//   count   : cells per type (shared-memory histogram of the codes)
//   plan    : per type the sampling stride, the candidate-list capacity and its offset in the pool (one warp)
//   sample  : ~2048-4096 hashed rows per type copied into a type-major sample buffer
//   pivot   : per (type, dim) two pivots lo <= hi at the sample ranks n_s/2 -+ 2.75 sqrt(n_s): the true median
//             lies outside with probability ~4e-8; the bracket holds ~9-12 % of the type's values
//   stream  : X is read exactly once (mn_stream_run_kernel, below): x < lo bumps a per-lane counter, an element
//             inside the closed bracket (or NaN) goes to a lane-private buffer and from there, once per item,
//             to its (type, dim) list with one global atomic on the list cursor
//   finish  : one CTA per (type, dim): rank bookkeeping (below / tie plateau / list / above), NaN count and radix
//             select inside the list staged in shared memory; if the rank fell outside the bracket or the list
//             overflowed, the same CTA runs an exact radix select over the type's rows -- no host round trip
// History of the stream pass (C3: 5 M x 50 f32, 40 types): round 1 gathered rows in GLOBAL type order (counting
// sort of all row ids, 1.46x the algorithmic DRAM bytes); round 2a read X in memory order with 128-bit loads and
// looked the pivots of every element up in shared memory (639 us, issue-bound at 78 instructions per element); a
// column-thread variant fed by 1-D bulk copies (cp.async.bulk + mbarriers) cut that to 42 instructions and 500 us;
// the chunk-sorted run form below needs ~15 and takes 376 us (2.7 TB/s), now bound by load latency.
constexpr int MN_SAMPLE_MIN = 2048;     // target sample rows per type: n_k / 16 clamped to [MIN, MAX]
constexpr int MN_SAMPLE_MAX = 4096;     //   (bracket width ~ 5.5 / sqrt(sample): 12 % ... 9 % of the type's values; measured best of 2048/4096/8192)
constexpr int MN_MCAP = MN_SAMPLE_MAX + MN_SAMPLE_MAX / 4;  // most sample rows a type can hold (pivot kernel's buffer)
constexpr double MED_SIGMAS = 5.5;      // half-width of the bracket in binomial sigmas
constexpr int MN_FIN_THREADS = 256;
constexpr int MN_REP = 32;              // replicas of every (type, dim) list: same-address global atomics serialise at ~20 ns
constexpr int MN_STAGE_MIN = 16384, MN_STAGE_MAX = 98304;  // bytes of candidates the finish kernel stages in shared memory

// shared-memory reduction without the compiler's warp-aggregation collective
__device__ __forceinline__ void red_shared_inc(unsigned int *p)
{
    const unsigned addr = (unsigned)__cvta_generic_to_shared(p);
    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(addr), "r"(1u) : "memory");
}

template <typename T> struct Inf;
template <> struct Inf<float> { __device__ static float pos() { return __int_as_float(0x7f800000); } };
template <> struct Inf<double> { __device__ static double pos() { return __longlong_as_double(0x7ff0000000000000LL); } };


struct MnHeader {
    unsigned int fail;  // pairs that took the exact full-column fallback (diagnostic, first word of the workspace)
    unsigned int pad[63];
};

template <typename T> struct MnWs {
    MnHeader *hdr;
    unsigned long long *type_cnt;          // K
    unsigned int *samp_cur;                // K: rows in the type's sample buffer
    unsigned int *below, *above;           // KD each: values below the bracket; values ON a tie plateau lo == hi
    unsigned int *ncand;                   // MN_REP x KD list cursors
    unsigned long long *cand_off;          // K: element offset of the type's candidate block; list (rep, d) at + (rep * D + d) * cap
    unsigned int *cap;                     // K: capacity of ONE replica list of a (type, dim)
    unsigned int *sstride;                 // K: keep a row when hash(row) % sstride == 0
    unsigned int *scap;                    // K: rows of the type's sample buffer
    unsigned long long *samp_off;          // K: first row of the type's sample buffer
    T *piv;                                // KD x 2
    T *samp;                               // per type a block of scap[k] sample rows of D values, row-major
    T *cand;                               // pool
};

__global__ void msort_count_kernel(const int *__restrict__ code, long long n, int K,
                                   unsigned long long *__restrict__ type_cnt)
{
    extern __shared__ unsigned int s_cnt[];
    for (int i = threadIdx.x; i < K; i += blockDim.x) s_cnt[i] = 0u;
    __syncthreads();
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int k = __ldg(code + i);
        if ((unsigned)k < (unsigned)K) atomicAdd(&s_cnt[k], 1u);  // ATOMS.POPC.INC: hardware warp aggregation
    }
    __syncthreads();
    for (int i = threadIdx.x; i < K; i += blockDim.x)
        if (s_cnt[i]) atomicAdd(&type_cnt[i], (unsigned long long)s_cnt[i]);
}


template <typename T> __global__ void mn_plan_kernel(int K, int D, int samp_max, MnWs<T> ws)
{
    // one warp: lane = type, 32 types per round, the two offsets by shuffle scans
    if (blockIdx.x != 0 || threadIdx.x >= 32) return;
    const int lane = threadIdx.x;
    unsigned long long off = 0, soff = 0;
    for (int b0 = 0; b0 < K; b0 += 32) {
        const int k = b0 + lane;
        const unsigned long long nk = k < K ? ws.type_cnt[k] : 0ULL;
        const unsigned cap = (unsigned)(0.35 * (double)nk / MN_REP) + 64u;
        unsigned long long target = nk / 16;
        target = target < MN_SAMPLE_MIN ? MN_SAMPLE_MIN : (target > (unsigned long long)samp_max ? (unsigned long long)samp_max : target);
        const unsigned long long sst = (nk + target - 1) / target;
        const unsigned long long expect = nk / (sst > 1 ? sst : 1);
        unsigned long long sc = expect + expect / 4 + 64;  // > 10 sigma of the binomial above the expectation
        if (sc > MN_MCAP) sc = MN_MCAP;
        const unsigned long long mine_s = k < K ? sc : 0ULL;
        const unsigned long long mine_c = k < K ? (unsigned long long)cap * (unsigned)D * MN_REP : 0ULL;
        unsigned long long is = mine_s, ic = mine_c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long vs = __shfl_up_sync(0xffffffffu, is, o), vc = __shfl_up_sync(0xffffffffu, ic, o);
            if (lane >= o) { is += vs; ic += vc; }
        }
        if (k < K) {
            ws.sstride[k] = (unsigned)(sst > 1 ? sst : 1);
            ws.scap[k] = (unsigned)sc;
            ws.samp_off[k] = soff + is - mine_s;
            ws.cap[k] = cap;
            ws.cand_off[k] = off + ic - mine_c;
        }
        soff += __shfl_sync(0xffffffffu, is, 31);
        off += __shfl_sync(0xffffffffu, ic, 31);
    }
}

__device__ __forceinline__ unsigned mn_hash(unsigned i)
{
    unsigned h = i * 0x9E3779B1u;
    h ^= h >> 15;
    h *= 0x85EBCA77u;
    h ^= h >> 13;
    return h;
}

// hashed row sample, type-major.  A CTA walks its contiguous block of rows, collects the selected ones in shared
// memory (position inside the CTA's share of the type through a shared-memory atomic), reserves its share of every
// type's sample buffer with ONE global atomic per type, then copies the rows (coalesced D-element rows).
constexpr int MN_SAMP_STAGE = 3072;  // selected rows a CTA can stage
template <typename T>
__global__ void __launch_bounds__(256)
mn_sample_kernel(const T *__restrict__ X, long long n, int D, long long ldx, const int *__restrict__ code, int K,
                 MnWs<T> ws)
{
    extern __shared__ __align__(16) unsigned int s_u[];  // cnt[K], base[K], sstride[K], scap[K], samp_off[K] (u64)
    unsigned int *s_cnt = s_u, *s_base = s_u + K, *s_sst = s_u + 2 * K, *s_scap = s_u + 3 * K;
    unsigned long long *s_soff = reinterpret_cast<unsigned long long *>(s_u + 4 * K);
    for (int i = threadIdx.x; i < K; i += blockDim.x) { s_sst[i] = ws.sstride[i]; s_scap[i] = ws.scap[i]; s_soff[i] = ws.samp_off[i]; }
    __shared__ unsigned int s_row[MN_SAMP_STAGE];
    __shared__ unsigned int s_kp[MN_SAMP_STAGE];  // type << 16 | position inside the CTA's share
    __shared__ unsigned int s_n;
    const long long per = (n + gridDim.x - 1) / gridDim.x;
    const long long c0 = (long long)blockIdx.x * per, c1 = c0 + per < n ? c0 + per : n;
    for (long long t0 = c0; t0 < c1; t0 += 32768) {  // in rounds, so that the stage cannot overflow
        const long long t1 = t0 + 32768 < c1 ? t0 + 32768 : c1;
        for (int i = threadIdx.x; i < K; i += blockDim.x) s_cnt[i] = 0u;
        if (threadIdx.x == 0) s_n = 0u;
        __syncthreads();
        for (long long i = t0 + threadIdx.x; i < t1; i += blockDim.x) {
            const int k = __ldg(code + i);
            if ((unsigned)k < (unsigned)K) {
                const unsigned sst = s_sst[k];
                if (sst <= 1u || (mn_hash((unsigned)i) % sst) == 0u) {
                    const unsigned lp = atomicAdd(&s_cnt[k], 1u);
                    const unsigned e = atomicAdd(&s_n, 1u);
                    if (e < (unsigned)MN_SAMP_STAGE && lp < 65536u) {
                        s_row[e] = (unsigned)i;
                        s_kp[e] = ((unsigned)k << 16) | lp;
                    }
                }
            }
        }
        __syncthreads();
        for (int i = threadIdx.x; i < K; i += blockDim.x)
            s_base[i] = s_cnt[i] ? atomicAdd(&ws.samp_cur[i], s_cnt[i]) : 0u;
        __syncthreads();
        const unsigned ne = s_n < (unsigned)MN_SAMP_STAGE ? s_n : (unsigned)MN_SAMP_STAGE;
        // copy: thread t moves the elements t, t + 256, ... of the staged rows (row-major): consecutive threads read
        // consecutive elements of a row; eight independent loads in flight per thread (the gather is latency-bound)
        {
            const unsigned total = ne * (unsigned)D;
            constexpr int CB = 8;
            for (unsigned idx0 = threadIdx.x; idx0 < total; idx0 += CB * blockDim.x) {
                T v[CB];
                size_t dst[CB];
                bool ok[CB];
#pragma unroll
                for (int c = 0; c < CB; ++c) {
                    const unsigned idx = idx0 + c * blockDim.x;
                    ok[c] = idx < total;
                    const unsigned e = ok[c] ? idx / (unsigned)D : 0u, d = ok[c] ? idx - e * (unsigned)D : 0u;
                    const unsigned kp = s_kp[e];
                    const unsigned k = kp >> 16, pos = s_base[k] + (kp & 0xffffu);
                    const unsigned scp = s_scap[k];
                    ok[c] = ok[c] && pos < scp;
                    // row-major inside the type's block: whole-row (coalesced) writes.  A dim-major block cost a 32-byte
                    // L2 sector per 4-byte element (15.6 M sector writes at C3, 165 us); the pivot kernel's strided column
                    // reads hit L2
                    dst[c] = (s_soff[k] + pos) * D + d;
                    v[c] = ok[c] ? X[(long long)s_row[e] * ldx + d] : (T)0;
                }
#pragma unroll
                for (int c = 0; c < CB; ++c)
                    if (ok[c]) ws.samp[dst[c]] = v[c];
            }
        }
        __syncthreads();
    }
}

// CTA-level radix select of two ranks over an arbitrary key source.  `known_prefix`/`first_shift`:
// digits above first_shift are already known to equal known_prefix for every key of interest.
template <typename T, typename Src>
__device__ void cta_select2_raw(Src src, long long r0, long long r1, unsigned int *hist /*[512]*/,
                                long long *sh /*[4]*/, typename KeyOf<T>::type known_prefix, int first_shift,
                                T &out0, T &out1)
{
    using KO = KeyOf<T>;
    using Key = typename KO::type;
    constexpr int BITS = sizeof(Key) * 8;
    Key p0 = known_prefix, p1 = known_prefix;
    long long q0 = r0, q1 = r1;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int shift = first_shift; shift >= 0; shift -= 8) {
        for (int b = threadIdx.x; b < 512; b += blockDim.x) hist[b] = 0u;
        __syncthreads();
        const bool top = shift + 8 >= BITS;
        const Key h0 = top ? (Key)0 : (Key)(p0 >> (shift + 8)), h1 = top ? (Key)0 : (Key)(p1 >> (shift + 8));
        src([&](T x) {
            const Key k = KO::key(x);
            const Key hi = top ? (Key)0 : (Key)(k >> (shift + 8));
            const unsigned dg = (unsigned)(k >> shift) & 0xffu;
            if (hi == h0) red_shared_inc(&hist[dg]);
            if (hi == h1) red_shared_inc(&hist[256 + dg]);
        });
        __syncthreads();
        if (warp < 2) {
            const unsigned int *h = hist + warp * 256;
            unsigned c[8];
            unsigned long long mine = 0;
#pragma unroll
            for (int t = 0; t < 8; ++t) { c[t] = h[lane * 8 + t]; mine += c[t]; }
            unsigned long long incl = mine;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long v = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += v;
            }
            const unsigned long long excl = incl - mine;
            const unsigned long long rank = (unsigned long long)(warp ? q1 : q0);
            if (rank >= excl && rank < incl) {
                unsigned long long run = excl, below = excl;
                int digit = lane * 8 + 7;
                bool found = false;
#pragma unroll
                for (int t = 0; t < 8; ++t) {
                    if (!found && rank < run + c[t]) { digit = lane * 8 + t; below = run; found = true; }
                    run += c[t];
                }
                sh[warp * 2] = digit;
                sh[warp * 2 + 1] = (long long)below;
            }
            const unsigned long long total = __shfl_sync(0xffffffffu, incl, 31);
            if (lane == 0 && rank >= total) { sh[warp * 2] = 255; sh[warp * 2 + 1] = (long long)total; }  // n == 0
        }
        __syncthreads();
        p0 |= (Key)sh[0] << shift; q0 -= sh[1];
        p1 |= (Key)sh[2] << shift; q1 -= sh[3];
        __syncthreads();
    }
    out0 = KO::value(p0);
    out1 = KO::value(p1);
}


constexpr int MN_LIN_BINS = 2048;  // linear bins of the one-pass selection
constexpr int MN_LIN_CAP = 512;    // most values its two target bins may hold
// CTA-level (256 threads) selection of the ranks r0 <= r1 among the values of `src` (no NaN), all of which lie in
// the finite interval [vlo, vhi], vlo < vhi.  ONE histogram pass over linear bins -- the values of a narrow bracket,
// or of a smooth sample, spread evenly over them: no hot bins, whereas the leading digits of a radix pass put
// thousands of values on a handful of shared-memory counters --, a scan, one pass that collects the (at most two)
// target bins, exact ranks inside them by counting.  Returns false (for every thread) when the target bins hold more
// than MN_LIN_CAP values -- a plateau of ties: the caller falls back to the radix select.
template <typename T, typename Src>
__device__ bool cta_select2_linear(Src src, long long r0, long long r1, T vlo, T vhi, unsigned int *hist /*[BINS]*/,
                                   T *coll /*[CAP + 2]*/, unsigned int *sh /*[16]*/, T &out0, T &out1)
{
    const T scale = (T)MN_LIN_BINS / (vhi - vlo);
    auto bin = [&](T x) -> int {
        const int b = (int)((x - vlo) * scale);  // monotone in x: equal values share a bin, bins order like the values
        return b < 0 ? 0 : (b >= MN_LIN_BINS ? MN_LIN_BINS - 1 : b);
    };
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int b = tid; b < MN_LIN_BINS; b += 256) hist[b] = 0u;
    if (tid == 0) sh[4] = 0u;
    __syncthreads();
    src([&](T x) { red_shared_inc(&hist[bin(x)]); });
    __syncthreads();
    {   // thread t owns the bins [8t, 8t + 8): CTA-wide exclusive scan, then the two ranks' bins
        unsigned c[8], mine = 0;
#pragma unroll
        for (int q = 0; q < 8; ++q) { c[q] = hist[8 * tid + q]; mine += c[q]; }
        unsigned incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) sh[8 + warp] = incl;
        __syncthreads();
        unsigned base = 0;
        for (int w = 0; w < warp; ++w) base += sh[8 + w];
        const unsigned excl = base + incl - mine;
#pragma unroll
        for (int which = 0; which < 2; ++which) {
            const unsigned r = (unsigned)(which ? r1 : r0);
            if (r >= excl && r < excl + mine) {
                unsigned run = excl;
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    if (r >= run && r < run + c[q]) { sh[2 * which] = 8 * tid + q; sh[2 * which + 1] = run; }
                    run += c[q];
                }
            }
        }
    }
    __syncthreads();
    const int b0 = (int)sh[0], b1 = (int)sh[2];
    const unsigned below0 = sh[1], below1 = sh[3];
    const unsigned n0 = hist[b0], cnt = n0 + (b1 != b0 ? hist[b1] : 0u);
    if (cnt > (unsigned)MN_LIN_CAP) return false;
    src([&](T x) {
        const int b = bin(x);
        if (b == b0 || b == b1) coll[atomicAdd(&sh[4], 1u)] = x;
    });
    __syncthreads();
    const unsigned q0 = (unsigned)r0 - below0, q1 = b1 == b0 ? (unsigned)r1 - below0 : n0 + ((unsigned)r1 - below1);
    for (unsigned i = tid; i < cnt; i += 256) {
        const T xi = coll[i];
        unsigned rank = 0;
        for (unsigned j = 0; j < cnt; ++j) {
            const T xj = coll[j];
            rank += (xj < xi || (xj == xi && j < i)) ? 1u : 0u;
        }
        if (rank == q0) coll[MN_LIN_CAP] = xi;
        if (rank == q1) coll[MN_LIN_CAP + 1] = xi;
    }
    __syncthreads();
    out0 = coll[MN_LIN_CAP];
    out1 = coll[MN_LIN_CAP + 1];
    __syncthreads();
    return true;
}

// CTA-level selection of the ranks r0 <= r1 among the values of `src` (no NaN), all of which lie in [vlo, vhi]: the
// linear bins when the interval is finite and not a point; otherwise, or on a plateau of ties, the radix select from
// the first digit in which key(vlo) and key(vhi) differ (every value shares the digits above it).
template <typename T, typename Src>
__device__ void cta_select2(Src src, long long r0, long long r1, T vlo, T vhi, unsigned int *hist /*[MN_LIN_BINS]*/,
                            T *coll /*[MN_LIN_CAP + 2]*/, unsigned int *lsh /*[16]*/, long long *sh /*[4]*/, T &out0,
                            T &out1)
{
    using KO = KeyOf<T>;
    using Key = typename KO::type;
    constexpr int BITS = sizeof(Key) * 8;
    if (vlo < vhi && vhi - vlo < Inf<T>::pos() &&
        cta_select2_linear<T>(src, r0, r1, vlo, vhi, hist, coll, lsh, out0, out1))
        return;
    const Key kl = KO::key(vlo), kh = KO::key(vhi);
    int first = BITS - 8;
    while (first > 0 && (kl >> first) == (kh >> first)) first -= 8;
    const Key prefix = first < BITS - 8 ? (Key)((kl >> (first + 8)) << (first + 8)) : (Key)0;
    cta_select2_raw<T>(src, r0, r1, hist, sh, prefix, first, out0, out1);
}

// one CTA per (type, dim): pivots lo <= hi bracketing the median, from the type's sample rows
template <typename T>
__global__ void __launch_bounds__(256, 6)
mn_pivot_kernel(int D, MnWs<T> ws)
{
    using Key = typename KeyOf<T>::type;
    constexpr int BITS = sizeof(Key) * 8;
    __shared__ long long sh[4];
    __shared__ unsigned int lhist[MN_LIN_BINS], lsh[16];
    unsigned int *hist = lhist;  // the radix fallback's 512 counters: never live together with the linear bins
    __shared__ T lcoll[MN_LIN_CAP + 2], red_mn[8], red_mx[8];
    extern __shared__ __align__(16) unsigned char pv_raw[];
    T *vals = reinterpret_cast<T *>(pv_raw);  // MN_MCAP
    const int kd = blockIdx.x;
    const int k = kd / D, d = kd - k * D;
    const unsigned cur = ws.samp_cur[k], scp = ws.scap[k];
    const int ns = (int)(cur < scp ? cur : scp);
    T lo = -Inf<T>::pos(), hi = Inf<T>::pos();
    if (ns >= 64) {
        const int delta = (int)ceil(0.5 * MED_SIGMAS * sqrt((double)ns)) + 1;
        const int jlo = (ns - 1) / 2 - delta, jhi = ns / 2 + delta;
        if (jlo > 0 && jhi < ns - 1) {
            const T *col = ws.samp + ws.samp_off[k] * D + d;  // column d of the type's row-major sample block
            for (int i = threadIdx.x; i < ns; i += 256) vals[i] = col[(size_t)i * D];
            __syncthreads();
            // valid count and range of the sample column (NaN samples sort last, as in np.sort)
            T mn = Inf<T>::pos(), mx = -Inf<T>::pos();
            unsigned mv = 0;
            for (int i = threadIdx.x; i < ns; i += 256) {
                const T x = vals[i];
                if (x == x) { mn = x < mn ? x : mn; mx = x > mx ? x : mx; ++mv; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const T a = __shfl_xor_sync(0xffffffffu, mn, o), b = __shfl_xor_sync(0xffffffffu, mx, o);
                mn = a < mn ? a : mn;
                mx = b > mx ? b : mx;
                mv += __shfl_xor_sync(0xffffffffu, mv, o);
            }
            if ((threadIdx.x & 31) == 0) { red_mn[threadIdx.x >> 5] = mn; red_mx[threadIdx.x >> 5] = mx; lsh[8 + (threadIdx.x >> 5)] = mv; }
            __syncthreads();
            int m = 0;
            for (int w = 0; w < 8; ++w) {
                mn = red_mn[w] < mn ? red_mn[w] : mn;
                mx = red_mx[w] > mx ? red_mx[w] : mx;
                m += (int)lsh[8 + w];
            }
            __syncthreads();
            auto smp = [&](auto f) {
                for (int i = threadIdx.x; i < ns; i += 256) {
                    const T x = vals[i];
                    if (x == x) f(x);
                }
            };
            if (jhi < m) {  // both ranks fall on valid samples; otherwise the bracket stays open (hi = +inf)
                if (mn == mx) lo = hi = mn;
                else cta_select2<T>(smp, jlo, jhi, mn, mx, lhist, lcoll, lsh, sh, lo, hi);
            } else if (jlo < m) {
                T dummy;
                cta_select2_raw<T>(smp, jlo, jlo, hist, sh, (Key)0, BITS - 8, lo, dummy);
            }
        }
    }
    if (threadIdx.x == 0) {
        ws.piv[2 * kd] = lo;
        ws.piv[2 * kd + 1] = hi;
    }
}

// The streaming pass, run form (any alignment; rows less than 1 MiB apart): a CTA takes a chunk of <= 4096
// consecutive rows, counting-sorts the chunk's row ids by type in shared memory (codes only: 4 bytes per row), and
// its warps then pull (type, 32-column group, 128-row segment) items: inside an item every row has the SAME type, so
// a lane keeps the (lo, hi) pivots of its (type, dim) in registers and an element costs a shared-memory broadcast of
// the row id, one address multiply-add, the load (a warp reads 32 consecutive elements of one row), two compares and
// a predicated store -- about 10 instructions against 40-75 in the earlier forms (history above), which looked up
// the pivots per element.  Bracket candidates collect in a lane-private shared-memory buffer and are appended to the
// (type, dim) list once per item: ONE global atomic per lane and item instead of one per candidate.  The rows of a
// chunk are read within microseconds of each other by one CTA, so the sectors two neighbouring rows share are
// fetched from DRAM once (round 1 gathered rows in GLOBAL type order and paid 1.46x).
constexpr int MN_RUN_THREADS = 512;
constexpr int MN_RUN_CMAX = 4096;      // rows per chunk: ids fit u16, <= 8 rows per thread in the sort
constexpr int MN_RUN_SEG = 128;        // rows per item
constexpr int MN_RUN_BUF = 128;        // bytes of a lane-private candidate buffer
constexpr size_t MN_RUN_SMEM_MAX = 100 * 1024;  // two CTAs per SM
template <typename T> struct MnRun {
    static constexpr int B = MN_RUN_BUF / (int)sizeof(T);  // its entries (32 f32 / 16 f64)
    static constexpr int U = 32 / (int)sizeof(T);   // loads in flight per lane (8 / 4)
};

template <typename T>
__global__ void __launch_bounds__(MN_RUN_THREADS, 2)
mn_stream_run_kernel(const T *__restrict__ X, long long n, int D, long long ldx, const int *__restrict__ code, int K,
                     int C, MnWs<T> ws)
{
    constexpr int B = MnRun<T>::B, U = MnRun<T>::U, NT = MN_RUN_THREADS;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T *buf = reinterpret_cast<T *>(smem_raw);                                   // [B][NT] lane-private candidate buffers
    unsigned int *s_off = reinterpret_cast<unsigned int *>(buf + (size_t)B * NT);  // [K + 1] first sorted slot of a type
    unsigned int *s_pos = s_off + K + 1;                                        // [K] counts, then scatter cursors
    unsigned int *s_eoff = s_pos + K;                                           // [K + 1] first item-table entry of a type
    unsigned int *s_tab = s_eoff + K + 1;                                       // [K + C / SEG + 1] type | segment << 16
    unsigned short *s_rid = reinterpret_cast<unsigned short *>(s_tab + K + C / MN_RUN_SEG + 1);  // [C]
    __shared__ unsigned int s_item, s_nitems;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int KD = K * D;
    const int CG = (D + 31) >> 5;
    const long long chunks = (n + C - 1) / C;
    for (long long chunk = blockIdx.x; chunk < chunks; chunk += gridDim.x) {
        const long long row0 = chunk * C;
        const int rows = (int)(n - row0 < C ? n - row0 : C);
        // ---- counting sort of the chunk's row ids by type ----
        for (int i = tid; i < K; i += NT) s_pos[i] = 0u;
        if (tid == 0) s_item = 0u;
        __syncthreads();
        int kreg[MN_RUN_CMAX / NT];
#pragma unroll
        for (int j = 0; j < MN_RUN_CMAX / NT; ++j) {
            const int i = tid + j * NT;
            int k = i < rows ? __ldg(code + row0 + i) : -1;
            if ((unsigned)k >= (unsigned)K) k = -1;
            kreg[j] = k;
            if (k >= 0) atomicAdd(&s_pos[k], 1u);
        }
        __syncthreads();
        if (warp == 0) {  // exclusive scans of the counts and of the segment counts
            unsigned run = 0, erun = 0;
            for (int b0 = 0; b0 < K; b0 += 32) {
                const int k = b0 + lane;
                const unsigned c = k < K ? s_pos[k] : 0u;
                const unsigned e = (c + MN_RUN_SEG - 1) / MN_RUN_SEG;
                unsigned ic = c, ie = e;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const unsigned vc = __shfl_up_sync(0xffffffffu, ic, o), ve = __shfl_up_sync(0xffffffffu, ie, o);
                    if (lane >= o) { ic += vc; ie += ve; }
                }
                if (k < K) {
                    s_off[k] = run + ic - c;
                    s_pos[k] = run + ic - c;
                    s_eoff[k] = erun + ie - e;
                    for (unsigned sgm = 0; sgm < e; ++sgm) s_tab[erun + ie - e + sgm] = (unsigned)k | (sgm << 16);
                }
                run += __shfl_sync(0xffffffffu, ic, 31);
                erun += __shfl_sync(0xffffffffu, ie, 31);
            }
            if (lane == 0) { s_off[K] = run; s_eoff[K] = erun; s_nitems = erun * (unsigned)CG; }
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < MN_RUN_CMAX / NT; ++j) {
            const int k = kreg[j];
            if (k >= 0) s_rid[atomicAdd(&s_pos[k], 1u)] = (unsigned short)(tid + j * NT);
        }
        __syncthreads();
        // ---- items ----
        const unsigned nitems = s_nitems;
        const T *xrow0 = X + row0 * ldx;
        const unsigned ldxb = (unsigned)ldx * (unsigned)sizeof(T);  // chunk-relative byte offsets stay below 2^32
        for (;;) {
            unsigned item = 0;
            if (lane == 0) item = atomicAdd(&s_item, 1u);
            item = __shfl_sync(0xffffffffu, item, 0);
            if (item >= nitems) break;
            const unsigned ent = s_tab[item / (unsigned)CG], cg = item % (unsigned)CG;
            const int k = (int)(ent & 0xffffu), sgm = (int)(ent >> 16);
            // list replica: by chunk and segment, so that a type whose rows sit in a few chunks (type-sorted input)
            // still spreads over all replicas
            const unsigned rep = (unsigned)(chunk + (chunk >> 5) + sgm) & (MN_REP - 1);
            const unsigned first = s_off[k] + (unsigned)sgm * MN_RUN_SEG;
            const unsigned tcnt = s_off[k + 1] - first;
            const int cnt = (int)(tcnt < (unsigned)MN_RUN_SEG ? tcnt : (unsigned)MN_RUN_SEG);
            const unsigned short *rid = s_rid + first;
            // lane -> (row slot, column): a column group narrower than 17 takes several rows per step
            const int Wc = D - (int)cg * 32 < 32 ? D - (int)cg * 32 : 32;
            const int RPS = 32 / Wc;
            const int sub = lane / Wc, d = (int)cg * 32 + (lane - sub * Wc);
            const bool active = sub < RPS;
            const int kd = k * D + (active ? d : 0);
            // a lane without a column compares against an empty bracket: it never lists anything that matters
            const T lo = active ? ws.piv[2 * kd] : Inf<T>::pos(), hi = active ? ws.piv[2 * kd + 1] : -Inf<T>::pos();
            const bool tie = active && lo == hi;
            const unsigned char *xpb = reinterpret_cast<const unsigned char *>(xrow0 + (active ? d : 0));
            const int subz = active ? sub : 0;
            const bool any_tie = __any_sync(0xffffffffu, tie);
            unsigned below = 0, ties = 0, nb = 0;
            T *mybuf = buf + tid;

            // append the lane's buffer to its list: one atomic reserves the space.  (A warp-cooperative variant -- one
            // list per store instruction, lane j = entry j, 1-2 sectors instead of 32 per instruction -- measured slower:
            // 414 vs 392 us at C3; the 32 shuffles and ballots cost more than the sector traffic they save.)
            auto flush_all = [&]() {
                if (active && nb) {
                    const unsigned pos = atomicAdd(&ws.ncand[(size_t)rep * KD + kd], nb);
                    const unsigned cap = ws.cap[k];
                    T *dst = ws.cand + ws.cand_off[k] + (size_t)(rep * (unsigned)D + (unsigned)d) * cap;
                    for (unsigned j = 0; j < nb; ++j)
                        if (pos + j < cap) dst[pos + j] = mybuf[(size_t)j * NT];
                }
                nb = 0;
            };
            // the closed bracket [lo, hi] and every NaN are listed; TIES: the ties of a plateau lo == hi are counted
            auto element = [&](T x, auto ties_tag) {
                const bool lt = x < lo;
                below += lt ? 1u : 0u;
                bool cand = !lt && !(x > hi);
                if (decltype(ties_tag)::value) {
                    if (tie && cand && x == lo) {
                        ++ties;
                        cand = false;
                    }
                }
                if (cand) {
                    mybuf[(size_t)nb * NT] = x;
                    ++nb;
                }
            };
            auto load_batch = [&](int j0, T (&x)[U]) {
#pragma unroll
                for (int u = 0; u < U; ++u)
                    x[u] = *reinterpret_cast<const T *>(xpb + (unsigned)rid[j0 + u * RPS + subz] * ldxb);
            };
            auto run_batch = [&](T (&x)[U]) {
                if (any_tie) {
#pragma unroll
                    for (int u = 0; u < U; ++u) element(x[u], std::true_type());
                } else {
#pragma unroll
                    for (int u = 0; u < U; ++u) element(x[u], std::false_type());
                }
                if (__any_sync(0xffffffffu, nb > (unsigned)(B - U))) flush_all();
            };
            const int stepr = RPS * U;
            const int nfull = cnt / stepr;
            // whole batches, software-pipelined: the loads of the next batch are in flight while this one is compared
            if (nfull > 0) {
                T xa[U], xb[U];
                load_batch(0, xa);
                int bi = 0;
                for (; bi + 2 <= nfull; bi += 2) {
                    load_batch((bi + 1) * stepr, xb);
                    run_batch(xa);
                    if (bi + 2 < nfull) load_batch((bi + 2) * stepr, xa);
                    run_batch(xb);
                }
                if (bi < nfull) run_batch(xa);
            }
            const int j0 = nfull * stepr;
            if (j0 < cnt) {  // the short last batch
                T x[U];
                bool ok[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int j = j0 + u * RPS + sub;
                    ok[u] = active && j < cnt;
                    x[u] = ok[u] ? *reinterpret_cast<const T *>(xpb + (unsigned)rid[j] * ldxb) : (T)0;
                }
#pragma unroll
                for (int u = 0; u < U; ++u)
                    if (ok[u]) element(x[u], std::true_type());
            }
            flush_all();
            if (active) {
                if (below) atomicAdd(&ws.below[kd], below);
                if (ties) atomicAdd(&ws.above[kd], ties);
            }
        }
        __syncthreads();
    }
}

// one CTA per (type, dim): rank bookkeeping (below / tie plateau / list / above), NaN count and selection inside
// the list, exact fallback over the type's own rows when the bracket missed or the list overflowed
template <typename T>
__global__ void __launch_bounds__(MN_FIN_THREADS, 5)
mn_finish_kernel(const T *__restrict__ X, long long n, int D, long long ldx, const int *__restrict__ code,
                 MnWs<T> ws, int STAGE, T *__restrict__ cent, double *__restrict__ cent64)
{
    using Key = typename KeyOf<T>::type;
    constexpr int BITS = sizeof(Key) * 8;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T *s_stage = reinterpret_cast<T *>(smem_raw);
    __shared__ long long sh[4];
    __shared__ unsigned int lhist[MN_LIN_BINS], lsh[16];
    unsigned int *hist = lhist;  // the radix paths' 512 counters: never live together with the linear bins
    __shared__ T lcoll[MN_LIN_CAP + 2];
    __shared__ unsigned long long s_nan, s_valid;
    const int kd = blockIdx.x;
    const int k = kd / D, d = kd - k * D;
    const long long Nk = (long long)ws.type_cnt[k];
    const long long below = ws.below[kd], tie_cnt = ws.above[kd];
    const unsigned cap = ws.cap[k];
    const int KD = gridDim.x;
    // the MN_REP replica lists of this (type, dim): counts and their exclusive prefix (one warp)
    __shared__ unsigned int s_roff[MN_REP + 1];
    __shared__ int s_over;
    if (threadIdx.x < 32) {
        static_assert(MN_REP == 32, "one lane per replica");
        const unsigned raw = ws.ncand[(size_t)threadIdx.x * KD + kd];
        const unsigned c = raw < cap ? raw : cap;
        const bool ov = __any_sync(0xffffffffu, raw > cap);
        unsigned incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned v = __shfl_up_sync(0xffffffffu, incl, o);
            if ((int)threadIdx.x >= o) incl += v;
        }
        s_roff[threadIdx.x + 1] = incl;
        if (threadIdx.x == 0) { s_roff[0] = 0u; s_over = ov ? 1 : 0; s_nan = 0ULL; s_valid = 0ULL; }
    }
    __syncthreads();
    const bool overflow = s_over != 0;
    const long long nlist = s_roff[MN_REP];
    const T *cl = ws.cand + ws.cand_off[k] + (size_t)d * cap;  // replica r at + r * D * cap
    const size_t rstride = (size_t)D * cap;
    const T lo = ws.piv[2 * kd], hi = ws.piv[2 * kd + 1];
    const long long ties = lo == hi ? tie_cnt : 0;
    const bool staged = !overflow && nlist <= STAGE;
    // every list element, NaN included: warp w walks the replicas w, w + 8, w + 16, w + 24 TOGETHER, sixteen
    // independent loads in flight per lane (one replica after the other made this the longest part of the kernel:
    // a dozen dependent round trips to L2 per CTA)
    auto lst_raw = [&](auto f) {
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
        constexpr int NQ = MN_REP / (MN_FIN_THREADS / 32);
        unsigned o[NQ], c[NQ], cm = 0;
        const T *src[NQ];
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
            const int r = warp + q * (MN_FIN_THREADS / 32);
            o[q] = s_roff[r];
            c[q] = s_roff[r + 1] - o[q];
            src[q] = cl + (size_t)r * rstride;
            cm = c[q] > cm ? c[q] : cm;
        }
        for (unsigned i0 = lane; i0 < cm; i0 += 128) {
            T v[NQ][4];
#pragma unroll
            for (int q = 0; q < NQ; ++q)
#pragma unroll
                for (int u = 0; u < 4; ++u) v[q][u] = i0 + 32 * u < c[q] ? src[q][i0 + 32 * u] : (T)0;
#pragma unroll
            for (int q = 0; q < NQ; ++q)
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (i0 + 32 * u < c[q]) f(o[q] + i0 + 32 * u, v[q][u]);
        }
    };
    unsigned my_nan = 0;
    if (staged) lst_raw([&](unsigned at, T x) { s_stage[at] = x; my_nan += x != x ? 1u : 0u; });  // NaNs counted on the way
    __syncthreads();
    auto lst_all = [&](auto f) {
        if (staged) {
            for (long long i = threadIdx.x; i < nlist; i += blockDim.x) f(s_stage[i]);
        } else {
            lst_raw([&](unsigned, T x) { f(x); });
        }
    };
    long long n_nan = 0;
    if (!overflow) {
        unsigned my = my_nan;
        if (!staged) lst_all([&](T x) { my += x != x ? 1u : 0u; });
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) my += __shfl_xor_sync(0xffffffffu, my, o);
        if ((threadIdx.x & 31) == 0 && my) atomicAdd(&s_nan, (unsigned long long)my);
        __syncthreads();
        n_nan = (long long)s_nan;
    }
    const long long nmid = nlist - n_nan;  // listed, orderable
    const long long nvalid = Nk - n_nan;
    T med;
    if (nvalid <= 0 && !overflow) {
        med = (T)NAN;
    } else {
        const long long q0 = (nvalid - 1) / 2, q1 = nvalid / 2;
        // where does each rank land?  0: < lo (fail) 1: the tie plateau lo == hi 2: the list 4: beyond (fail)
        auto region = [&](long long r, long long &rin) -> int {
            if (r < below) return 0;
            r -= below;
            if (r < ties) return 1;
            r -= ties;
            if (r < nmid) { rin = r; return 2; }
            return 4;
        };
        long long j0 = 0, j1 = 0;
        const int g0 = overflow ? 0 : region(q0, j0), g1 = overflow ? 0 : region(q1, j1);
        T v0, v1;
        if (overflow || g0 == 0 || g0 == 4 || g1 == 0 || g1 == 4) {
            // exact fallback: radix select over this type's own rows (found by scanning the codes)
            if (threadIdx.x == 0) atomicAdd(&ws.hdr->fail, 1u);
            {
                unsigned long long my = 0;
                for (long long i = threadIdx.x; i < n; i += blockDim.x)
                    if (__ldg(code + i) == k) {
                        const T x = X[i * ldx + d];
                        my += x == x ? 1ULL : 0ULL;
                    }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) my += __shfl_xor_sync(0xffffffffu, my, o);
                if ((threadIdx.x & 31) == 0 && my) atomicAdd(&s_valid, my);
            }
            __syncthreads();
            const long long nv = (long long)s_valid;
            if (nv <= 0) {
                v0 = v1 = (T)NAN;
            } else {
                auto col = [&](auto f) {
                    for (long long i = threadIdx.x; i < n; i += blockDim.x)
                        if (__ldg(code + i) == k) {
                            const T x = X[i * ldx + d];
                            if (x == x) f(x);
                        }
                };
                cta_select2_raw<T>(col, (nv - 1) / 2, nv / 2, hist, sh, (Key)0, BITS - 8, v0, v1);
            }
        } else {
            T m0 = lo, m1 = lo;
            if (g0 == 2 || g1 == 2) {
                auto lst = [&](auto f) { lst_all([&](T x) { if (x == x) f(x); }); };
                const long long s0 = g0 == 2 ? j0 : (g1 == 2 ? j1 : 0), s1 = g1 == 2 ? j1 : s0;  // s0 <= s1
                // every orderable list element lies in the bracket [lo, hi]
                cta_select2<T>(lst, s0, s1, lo, hi, lhist, lcoll, lsh, sh, m0, m1);
            }
            v0 = g0 == 1 ? lo : m0;
            v1 = g1 == 1 ? lo : m1;
        }
        if (v0 == v1) med = v0;
        else if (sizeof(T) == 4) med = (T)__fdiv_rn(__fadd_rn((float)v0, (float)v1), 2.0f);
        else med = (T)__ddiv_rn(__dadd_rn((double)v0, (double)v1), 2.0);
    }
    if (threadIdx.x == 0) {
        cent[kd] = med;
        cent64[kd] = (double)med;
    }
}

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// the stream path's workspace (256-byte aligned regions)
template <typename T> struct MnLayout {
    MnWs<T> ws;
    size_t zero;   // the prefix zeroed at the start of every call: header and counters
    size_t bytes;  // end of the last region
};

// carves the stream path's workspace at `base` (nullptr: only its size)
template <typename T> static MnLayout<T> mn_workspace(void *base, long long n, int K, int D)
{
    const size_t kd = (size_t)K * D;
    uintptr_t p = (uintptr_t)base;
    const auto take = [&p](size_t bytes) { const uintptr_t r = p; p += align256(bytes); return r; };
    MnLayout<T> l;
    MnWs<T> &ws = l.ws;
    ws.hdr = (MnHeader *)take(sizeof(MnHeader));
    ws.type_cnt = (unsigned long long *)take((size_t)K * 8);
    ws.samp_cur = (unsigned int *)take((size_t)K * 4);
    ws.below = (unsigned int *)take(kd * 4);
    ws.above = (unsigned int *)take(kd * 4);
    ws.ncand = (unsigned int *)take(kd * 4 * MN_REP);
    l.zero = p - (uintptr_t)base;
    ws.cand_off = (unsigned long long *)take((size_t)K * 8);
    ws.cap = (unsigned int *)take((size_t)K * 4);
    ws.sstride = (unsigned int *)take((size_t)K * 4);
    ws.scap = (unsigned int *)take((size_t)K * 4);
    ws.samp_off = (unsigned long long *)take((size_t)K * 8);
    ws.piv = (T *)take(kd * 2 * sizeof(T));
    ws.samp = (T *)take(((size_t)(n / 16) * 5 / 4 + (size_t)K * (MN_SAMPLE_MIN * 5 / 4 + 64 + 64)) * D * sizeof(T));
    ws.cand = (T *)take((size_t)(0.35 * (double)n * D) * sizeof(T) + (size_t)65 * MN_REP * kd * sizeof(T) + 4096);
    l.bytes = p - (uintptr_t)base;
    return l;
}

// which path computes the medians, and the run form's launch when it is the stream path
struct MedianPath {
    bool stream;        // the sampled-pivot stream path; otherwise the MSD radix select
    long long ctas, C;  // the run form's CTAs and rows per chunk
    size_t smem;        // its dynamic shared memory
};

// The stream path's limits on the shape alone, which is all the workspace query sees.  Its sample and list
// workspace grows with K*D (f64: ~38 KB per (type, dim) plus 0.35 n D list elements, against 2 KB of histograms on
// the radix path), so a large K*D takes the radix path.  The bound, 24 B per (type, dim) + 12 B per type within
// 160 KiB, is the shared memory of an earlier form of the pass; it stays so that every input keeps its path.
static bool mn_stream_shape_ok(long long n, int K, int D)
{
    return n >= 65536 && n < (1LL << 32) && K <= 4096 && 24 * (size_t)K * D + 12 * (size_t)K <= 160 * 1024;
}

// The stream path takes an input when its shape allows, its rows are less than 1 MiB apart (the run form's
// chunk-relative byte offsets stay below 2^32) and the run form's shared memory holds its types.
static MedianPath median_path(long long n, int K, int D, long long ldx, size_t elt)
{
    MedianPath p{};
    if (!mn_stream_shape_ok(n, K, D) || ldx * (long long)elt >= (1LL << 20)) return p;
    long long ctas = (n + 1023) / 1024;  // chunks of at least ~1024 rows
    const long long cta_cap = (long long)sm_count() * 2;
    if (ctas > cta_cap) ctas = cta_cap;
    const long long m = (n + ctas * MN_RUN_CMAX - 1) / (ctas * MN_RUN_CMAX);  // chunks per CTA
    long long C = (n + ctas * m - 1) / (ctas * m);
    C = (C + 7) & ~7LL;
    if (C > MN_RUN_CMAX) C = MN_RUN_CMAX;
    const long long chunks = (n + C - 1) / C;
    p.ctas = ctas < chunks ? ctas : chunks;
    p.C = C;
    // the kernel's dynamic shared memory: lane buffers, the sort's per-type tables, the item table, the row ids
    p.smem = (size_t)MN_RUN_BUF * MN_RUN_THREADS + ((size_t)4 * K + 3 + C / MN_RUN_SEG + 1) * 4 + (size_t)C * 2 + 16;
    p.stream = p.smem <= MN_RUN_SMEM_MAX;
    return p;
}

template <typename T>
static int median_run_stream(const T *X, long long n, int D, long long ldx, const int *code, int K,
                             const MedianPath &path, T *cent, double *cent64, void *workspace, cudaStream_t st)
{
    const size_t kd = (size_t)K * D;
    const MnLayout<T> l = mn_workspace<T>(workspace, n, K, D);
    const MnWs<T> ws = l.ws;
    PILOT_CUDA(cudaMemsetAsync(workspace, 0, l.zero, st));
    long long blocks = (n + 2047) / 2048;
    const long long cap = (long long)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    msort_count_kernel<<<(unsigned)blocks, 256, K * sizeof(unsigned int), st>>>(code, n, K, ws.type_cnt);
    PILOT_LAUNCH_CHECK();
    mn_plan_kernel<T><<<1, 32, 0, st>>>(K, D, MN_SAMPLE_MAX, ws);
    PILOT_LAUNCH_CHECK();
    {
        long long sblocks = (n + 1023) / 1024;  // one global atomic per (CTA, type): ~20 ns each, serialised per type
        if (sblocks > 4LL * sm_count()) sblocks = 4LL * sm_count();
        mn_sample_kernel<T><<<(unsigned)sblocks, 256, (6 * (size_t)K + 2) * sizeof(unsigned int), st>>>(X, n, D, ldx, code, K, ws);
    }
    PILOT_LAUNCH_CHECK();
    PILOT_CUDA(cudaFuncSetAttribute(mn_pivot_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)(MN_MCAP * sizeof(T))));
    mn_pivot_kernel<T><<<(unsigned)kd, 256, MN_MCAP * sizeof(T), st>>>(D, ws);
    PILOT_LAUNCH_CHECK();
    PILOT_CUDA(cudaFuncSetAttribute(mn_stream_run_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)path.smem));
    mn_stream_run_kernel<T><<<(unsigned)path.ctas, MN_RUN_THREADS, path.smem, st>>>(X, n, D, ldx, code, K, (int)path.C, ws);
    PILOT_LAUNCH_CHECK();
    {
        // stage size from the expected list length: bracket fraction 5.5 / sqrt(sample) of an average type, + 25 %;
        // a longer list is selected from global memory instead (L2 resident), a shorter stage lets more CTAs share an SM
        const double nk = (double)n / K;
        double ns = nk / 16;
        ns = ns < MN_SAMPLE_MIN ? MN_SAMPLE_MIN : (ns > MN_SAMPLE_MAX ? MN_SAMPLE_MAX : ns);
        if (ns > nk) ns = nk > 1 ? nk : 1;
        size_t bytes = (size_t)(1.25 * MED_SIGMAS / sqrt(ns) * nk) * sizeof(T);
        bytes = bytes < MN_STAGE_MIN ? MN_STAGE_MIN : (bytes > MN_STAGE_MAX ? MN_STAGE_MAX : bytes);
        bytes = (bytes + 1023) & ~(size_t)1023;
        PILOT_CUDA(cudaFuncSetAttribute(mn_finish_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, MN_STAGE_MAX));
        mn_finish_kernel<T><<<(unsigned)kd, MN_FIN_THREADS, bytes, st>>>(X, n, D, ldx, code, ws, (int)(bytes / sizeof(T)),
                                                                         cent, cent64);
    }
    PILOT_LAUNCH_CHECK();
    return 0;
}

size_t median_ws_bytes(long long n, int K, int D)
{
    // ldx and the dtype are unknown here: room for the f64 stream path whenever the shape allows it
    size_t a = median_workspace(nullptr, K, D).bytes;
    if (mn_stream_shape_ok(n, K, D)) {
        const size_t b = mn_workspace<double>(nullptr, n, K, D).bytes;
        if (b > a) a = b;
    }
    return a;
}
}  // namespace pilot

extern "C" int pilot_centroid_median(const void *X, int dtype, int64_t n_cells, int D, int64_t ldx,
                                     const int32_t *ct_code, int K, void *centroids, double *centroids_f64,
                                     void *workspace, size_t workspace_bytes, void *stream)
{
    using namespace pilot;
    PILOT_CHECK_ARG(dtype == PILOT_F32 || dtype == PILOT_F64, "pilot_centroid_median: dtype %d", dtype);
    PILOT_CHECK_ARG(K >= 1 && D >= 1 && n_cells >= 1 && ldx >= D, "pilot_centroid_median: bad shape");
    PILOT_CHECK_ARG(X && ct_code && centroids && centroids_f64 && workspace, "pilot_centroid_median: NULL pointer");
    PILOT_CHECK_ARG((long long)K * D < (1LL << 30), "pilot_centroid_median: K*D too large");
    PILOT_CHECK_ARG(n_cells < (1LL << 32), "pilot_centroid_median: n_cells must be < 2^32");
    PILOT_CHECK_ARG(workspace_bytes >= median_ws_bytes(n_cells, K, D),
                    "pilot_centroid_median: workspace %zu < %zu bytes", workspace_bytes,
                    median_ws_bytes(n_cells, K, D));
    cudaStream_t st = (cudaStream_t)stream;
    const MedianPath path = median_path(n_cells, K, D, ldx, dtype == PILOT_F32 ? sizeof(float) : sizeof(double));
    if (path.stream) {
        if (dtype == PILOT_F32)
            return median_run_stream<float>((const float *)X, n_cells, D, ldx, ct_code, K, path, (float *)centroids,
                                            centroids_f64, workspace, st);
        return median_run_stream<double>((const double *)X, n_cells, D, ldx, ct_code, K, path, (double *)centroids,
                                         centroids_f64, workspace, st);
    }
    if (dtype == PILOT_F32)
        return median_run<float>((const float *)X, n_cells, D, ldx, ct_code, K, (float *)centroids,
                                 centroids_f64, workspace, st);
    return median_run<double>((const double *)X, n_cells, D, ldx, ct_code, K, (double *)centroids,
                              centroids_f64, workspace, st);
}
