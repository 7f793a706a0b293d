// C-ABI plumbing: error string, pair-range helpers, workspace sizing.
#include <stdarg.h>
#include <string.h>
#include <atomic>
#include "common.cuh"

namespace pilot {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

static std::atomic<unsigned long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

int sm_count()
{
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

int make_pair_map(const pilot_pair_range *r, int S, PairMap *pm)
{
    PILOT_CHECK_ARG(r != nullptr, "pair range is NULL");
    PILOT_CHECK_ARG(r->block >= 1, "pair range: block must be >= 1 (got %lld)", (long long)r->block);
    PILOT_CHECK_ARG(r->nranks >= 1 && r->rank >= 0 && r->rank < r->nranks,
                    "pair range: bad rank %d of %d", r->rank, r->nranks);
    PILOT_CHECK_ARG(r->mode == PILOT_PAIRS_FULL || r->mode == PILOT_PAIRS_UPPER || r->mode == PILOT_PAIRS_RECT,
                    "pair range: bad mode %d", r->mode);
    const bool rect = r->mode == PILOT_PAIRS_RECT;
    PILOT_CHECK_ARG(!rect || (r->rows >= 1 && r->rows < S),
                    "pair range: RECT row count %d outside [1, %d)", r->rows, S);
    long long cap = rect ? (long long)r->rows * (S - r->rows)
                         : r->mode == PILOT_PAIRS_FULL ? (long long)S * S : (long long)S * (S - 1) / 2;
    PILOT_CHECK_ARG(r->first >= 0 && r->total >= 0 && r->first + r->total <= cap,
                    "pair range: window [%lld, +%lld) outside [0, %lld]", (long long)r->first, (long long)r->total, cap);
    pm->total = r->total;
    pm->block = r->block;
    pm->first = r->first;
    pm->nranks = r->nranks;
    pm->rank = r->rank;
    pm->mode = r->mode;
    pm->S = S;
    pm->row_len = rect ? S - r->rows : S;
    pm->col0 = rect ? r->rows : 0;
    pm->n_local = range_count(r->total, r->block, r->nranks, r->rank);
    return 0;
}

size_t median_ws_bytes(long long n, int K, int D);
size_t sinkhorn_ws_bytes(int K);
size_t emd_ws_bytes(int K);

}  // namespace pilot

extern "C" {

size_t pilot_workspace_bytes(int kind, int64_t n, int K, int S, int D)
{
    (void)S;
    switch (kind) {
    case PILOT_WS_MEDIAN:   return pilot::median_ws_bytes(n, K, D);
    case PILOT_WS_SINKHORN: return pilot::sinkhorn_ws_bytes(K);
    case PILOT_WS_EMD:      return pilot::emd_ws_bytes(K);
    default:                return 0;
    }
}

int pilot_abi_version(void) { return PILOT_B200_ABI_VERSION; }

uint64_t pilot_launch_count(void) { return (uint64_t)pilot::g_launches.load(std::memory_order_relaxed); }

const char *pilot_last_error(void) { return pilot::g_err; }

int64_t pilot_range_count(const pilot_pair_range *r)
{
    if (!r || r->block < 1 || r->nranks < 1 || r->rank < 0 || r->rank >= r->nranks) return -1;
    return pilot::range_count(r->total, r->block, r->nranks, r->rank);
}

}  // extern "C"
