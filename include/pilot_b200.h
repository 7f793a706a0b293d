/*
 * pilot_b200.h -- C ABI of the B200-native PILOT patient-distance hot path.
 *
 * The reference (CostaLab/PILOT, pilotpy 2.0.6) has no FFI/plugin interface: the
 * boundary is the Python function surface of pilotpy/tools/Trajectory.py plus
 * the adata.uns contract (SURVEY.md 8b).  Each entry point below replaces the
 * *native arithmetic* that one reference statement reaches, and is what a
 * ctypes binding inside pilotpy would call (see INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller unless its name
 *     starts with h_ ; the library allocates nothing persistent
 *   - scratch comes from a caller-provided workspace (pilot_workspace_bytes)
 *   - `stream` is a cudaStream_t (CUstream) passed as void*; all work is
 *     asynchronous on it
 *   - return value: 0 = OK, <0 = bad argument, >0 = CUDA error code;
 *     pilot_last_error() returns a thread-local message
 *   - no torch types, no C++ types
 */
#ifndef PILOT_B200_H
#define PILOT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PILOT_B200_ABI_VERSION 4

/* element types of the embedding handed to pilot_centroid_median; also the `precision`
 * of the two pair solvers (FP64 = the 1e-9 parity tier, FP32 = the 1e-4 tier) */
#define PILOT_F32 0
#define PILOT_F64 1

/* pdist metrics accepted by pilot_cdist (scipy.spatial.distance.pdist names) */
#define PILOT_METRIC_COSINE      0
#define PILOT_METRIC_EUCLIDEAN   1
#define PILOT_METRIC_SQEUCLIDEAN 2
#define PILOT_METRIC_CITYBLOCK   3
#define PILOT_METRIC_CHEBYSHEV   4
#define PILOT_METRIC_CORRELATION 5
#define PILOT_METRIC_BRAYCURTIS  6
#define PILOT_METRIC_CANBERRA    7
#define PILOT_METRIC_MINKOWSKI   8   /* SciPy's default p = 2 */
#define PILOT_METRIC_SEUCLIDEAN  9   /* V = var(centroids, axis=0, ddof=1), SciPy's default */
#define PILOT_METRIC_HAMMING     10

/* how a linear problem index g maps to a sample pair (i, j); S = rows of props */
#define PILOT_PAIRS_FULL  0   /* g = i*S + j, all S*S ordered pairs incl. diagonal     */
#define PILOT_PAIRS_UPPER 1   /* strictly upper triangle, row-major, S*(S-1)/2 pairs    */
/* two sample sets concatenated in props: rows i = 0..S_a-1 against columns
 * j = S_a + j', j' = 0..S_b-1 (S_b = S - S_a); g = i*S_b + j', S_a*S_b pairs, the
 * problem (a = props[i], b = props[S_a + j']).  S_a travels in pilot_pair_range.rows.
 * A problem is solved by the same arithmetic as the same pair of the FULL / UPPER
 * square over props, so a block is bit-identical to those entries of the square. */
#define PILOT_PAIRS_RECT  2

/* per-problem status written by the *_pairs kernels */
#define PILOT_ST_CONVERGED 0  /* Sinkhorn: err <= stopThr ; EMD: optimal               */
#define PILOT_ST_MAXITER   1  /* Sinkhorn: numItermax reached ; EMD: pivot cap reached */
#define PILOT_ST_NUMERIC   2  /* Sinkhorn: NaN roll-back (POT "Numerical errors")      */
#define PILOT_ST_UNBOUNDED 3  /* EMD only                                              */

/* workspace kinds for pilot_workspace_bytes */
#define PILOT_WS_MEDIAN   0
#define PILOT_WS_SINKHORN 1
#define PILOT_WS_EMD      2

/*
 * Partition of the window [first, first + total) of the linear pair space over
 * `nranks` processes: blocks of `block` consecutive problems are dealt
 * round-robin; rank r owns blocks r, r+nranks, ...  Its packed output holds its
 * blocks back to back.  nranks=1, rank=0, first=0 means "everything".  A window
 * (first > 0) lets the host solve, gather and copy out the matrix band by band.
 * (SURVEY.md 8e)
 */
typedef struct {
    int64_t total;   /* problems in the window: first + total <= S*S (FULL), S*(S-1)/2 (UPPER)
                        or S_a*(S - S_a) (RECT) */
    int64_t block;   /* problems per block (>=1) */
    int32_t nranks;
    int32_t rank;
    int32_t mode;    /* PILOT_PAIRS_* */
    int32_t rows;    /* row count S_a in PILOT_PAIRS_RECT (1 <= S_a < S), 0 otherwise */
    int64_t first;   /* linear index of the window's first problem */
} pilot_pair_range;

int         pilot_abi_version(void);
const char *pilot_last_error(void);
/* number of problems `range` assigns to range->rank */
int64_t     pilot_range_count(const pilot_pair_range *range);
size_t      pilot_workspace_bytes(int kind, int64_t n, int K, int S, int D);
/* kernels this library has launched in this process so far (bench.py's gpu_launches) */
uint64_t    pilot_launch_count(void);

/*
 * (1) Proportion counting -- replaces the pandas unique/value_counts/boolean-mask
 * scans of Cluster_Representations, Trajectory.py:402-425.
 * ct_code[i] in [0,K), smp_code[i] in [0,S) are arbitrary (not necessarily
 * first-appearance) integer codes of cell i.  Outputs: counts[s*K+k];
 * first_ct[k] / first_smp[s] = smallest cell index carrying that code
 * (n_cells if absent) so the host can restore `.unique()` order.
 */
int pilot_hist(const int32_t *ct_code, const int32_t *smp_code, int64_t n_cells,
               int K, int S, int64_t *counts, int64_t *first_ct,
               int64_t *first_smp, void *stream);

/*
 * Dirichlet-smoothed proportions, Trajectory.py:405-409 and :428-430, FP64,
 * bit-exact with the reference (sequential sums, no FMA contraction).
 * counts_raw is pilot_hist's table (S_raw x K_raw, raw-code order); perm_s[S] /
 * perm_k[K] (device int32, NULL = identity) list the raw codes in order of first
 * appearance, so props[s*K+k] and counts_out[s*K+k] (optional) come out in the
 * reference's `.unique()` order.  prior_out[K+1] receives the Dirichlet prior
 * n_k/(N-1)*regulizer and, last, its sequential sum.  normalization==0 copies
 * the raw counts (Trajectory.py:425).
 */
int pilot_props_finalize(const int64_t *counts_raw, int K_raw, int S_raw,
                         const int32_t *perm_k, const int32_t *perm_s, int K,
                         int S, int64_t n_cells, double regulizer,
                         int normalization, double *props, int64_t *counts_out,
                         double *prior_out, void *stream);

/*
 * (2a) Per-type, per-dimension MEDIAN of the embedding rows in the input dtype
 * (NaNs ignored, even counts -> (lo+hi)/2 rounded in the input dtype) --
 * replaces data[mask].median(axis=0), Trajectory.py:465-466.
 * X is row-major n_cells x D with leading dimension ldx (elements).
 * centroids (K*D, dtype of X) and centroids_f64 (K*D) are both written.
 */
int pilot_centroid_median(const void *X, int dtype, int64_t n_cells, int D,
                          int64_t ldx, const int32_t *ct_code, int K,
                          void *centroids, double *centroids_f64,
                          void *workspace, size_t workspace_bytes, void *stream);

/*
 * (2b) K x K distance matrix between centroids -- replaces
 * squareform(pdist(centroids, metric)), Trajectory.py:468-469.  Also writes
 * cost_norm = cost / max(cost) (Trajectory.py:101) and *cost_max; cost_norm
 * (required) doubles as scratch while the pairs are computed.
 */
int pilot_cdist(const double *centroids_f64, int K, int D, int metric,
                double *cost, double *cost_norm, double *cost_max, void *stream);

/*
 * (3) All-pairs stabilised Sinkhorn -- replaces the loop over
 * ot.sinkhorn2(a_i, a_j, cost, reg, method="sinkhorn_stabilized"),
 * Trajectory.py:513-515 (POT defaults: num_iter_max=1000, stop_thr=1e-9,
 * tau=1e3, check_every=20).  out[l] = sum(M * Gamma) of local problem l.
 * iters / absorptions / status may be NULL.
 * algo: 0 = shared-Gibbs-kernel solvers (fast path: one warp per problem with K0
 *           in registers for K <= 32 and a symmetric cost, else 8-problem DMMA
 *           panels whose stragglers are finished by a warp-form tail kernel;
 *           65 <= K <= 256: DMMA panels with K0 split in row stripes over a
 *           thread-block cluster; problems the scaled form cannot represent are
 *           re-solved by the reference-form kernel, however many they are),
 *       1 = reference-form kernel only (per-problem Gibbs kernel, literal schedule;
 *           the Gibbs matrix lives in the workspace when it does not fit shared
 *           memory, K > ~155),
 *       3 = DMMA-panel solver (+ tail) for every K <= 64, the cluster panels above.
 * Solver selection for algo = 0: the warp form runs for a symmetric cost when
 * 17 <= K <= 32, or K <= 16 and S*S < 200000, with S the rows of props (in
 * PILOT_PAIRS_RECT the concatenated sets, so a block is solved as the square over
 * them solves it); every other choice depends on K only.  It never depends on the
 * window, the rank or the partition, so results are bit-identical under them.
 * 1 <= K <= 256 (ot.sinkhorn2 itself has no limit).  The call is fully
 * asynchronous on `stream` (whether the cost is symmetric is decided on the
 * device: both variants of a solver are enqueued, one returns at once).
 * precision: PILOT_F64 = the schedule above in double (within 1e-9 of POT);
 * PILOT_F32 = log-domain Sinkhorn in float (within 1e-4; stop_thr is raised to
 * what float can resolve) for K <= 64; K > 64 runs the FP64 solvers whatever
 * the precision.
 */
int pilot_sinkhorn_pairs(const double *props, int S, int K, const double *cost,
                         double reg, int num_iter_max, double stop_thr,
                         double tau, int check_every,
                         const pilot_pair_range *range, int algo, int precision,
                         double *out, int32_t *iters, int32_t *absorptions,
                         int32_t *status,
                         void *workspace, size_t workspace_bytes, void *stream);

/*
 * (4) All-pairs exact EMD -- replaces the loop over ot.emd2(a_i, a_j, cost),
 * Trajectory.py:507-511 (b is rescaled to a's mass as emd2 does).
 * out[l] = optimal transport cost of local problem l; status/pivots may be NULL.
 * precision: PILOT_F64 (costs, flows and potentials in double: within 1e-9 of
 * POT) or PILOT_F32 (the same solver on float: within 1e-4).  1 <= K <= 256:
 * up to 64 types the bit-mask solver (emd.cu), 65..256 a general network simplex
 * (emd_general.cu, FP64 whatever the precision) -- ot.emd2 itself has no limit.
 */
int pilot_emd_pairs(const double *props, int S, int K, const double *cost,
                    int64_t max_pivots, const pilot_pair_range *range,
                    int precision, double *out, int32_t *status,
                    int32_t *pivots, void *workspace, size_t workspace_bytes,
                    void *stream);

/*
 * (3p, 4p) Transport plans of the n problems a caller lists -- what ot.sinkhorn
 * (method="sinkhorn_stabilized") and ot.emd return beside the costs of (3) and (4).
 * Problem l is (a = props[pair_a[l]], b = props[pair_b[l]]), solved as given (no
 * mirroring), on one device, in FP64:
 *   plans[l*K*K + r*K + c] = Gamma[r, c]  (n x K x K; row r: a cell type of a,
 *                                          column c: a cell type of b)
 *   out[l]                 = the cost, computed by the code that writes it in the
 *                            pair solvers above
 * pilot_emd_plans runs the exact solver of pilot_emd_pairs (bit-mask up to 64 types,
 * general network simplex above); Gamma holds the basis flows (at most 2K - 1
 * non-zeros), its rows sum to a and its columns to emd2's rescaled b.
 * pilot_sinkhorn_plans runs the reference-form kernel of pilot_sinkhorn_pairs
 * (algo = 1), whose cost it reproduces bit for bit; Gamma is
 * exp(-(M - alpha_i - beta_j)/reg + log u_i + log v_j), POT's statement.
 * 1 <= K <= 256, n >= 0.  status, iters and absorptions may be NULL.  A pair index
 * outside [0, S) is never read: that problem gets a NaN cost, a NaN plan and
 * PILOT_ST_NUMERIC.  Workspace: pilot_workspace_bytes(PILOT_WS_EMD, n, K, S, 0),
 * resp. PILOT_WS_SINKHORN.  Asynchronous on `stream`.
 */
int pilot_emd_plans(const double *props, int S, int K, const double *cost,
                    int64_t max_pivots, const int32_t *pair_a,
                    const int32_t *pair_b, int64_t n, double *plans,
                    double *out, int32_t *status, void *workspace,
                    size_t workspace_bytes, void *stream);
int pilot_sinkhorn_plans(const double *props, int S, int K, const double *cost,
                         double reg, int num_iter_max, double stop_thr,
                         double tau, int check_every, const int32_t *pair_a,
                         const int32_t *pair_b, int64_t n, double *plans,
                         double *out, int32_t *iters, int32_t *absorptions,
                         int32_t *status, void *workspace,
                         size_t workspace_bytes, void *stream);

/*
 * (5) Packed per-rank results (as laid out by an all-gather: rank r's chunk at
 * packed + r*chunk_stride) -> dense row-major matrix, EMD[i,j] with
 * i = row sample (a), j = column sample (b) as Trajectory.py:511/515.  Shape of
 * `dense` per mode (a window writes only its own entries):
 *   FULL : S x S;
 *   UPPER: S x S, mirrored into the lower triangle, `diag_value` on the diagonal;
 *   RECT : S_a x (S - S_a), dense[i*(S - S_a) + j'] = problem (i, S_a + j'); no
 *          mirror, no diagonal.
 */
int pilot_unpack_pairs(const double *packed, int64_t chunk_stride, int S,
                       const pilot_pair_range *range, double diag_value,
                       double *dense, void *stream);

/*
 * (f-1) Row k-nearest neighbours on the dense S x S distance matrix, the first step of the consumer
 * pilotpy.pl.trajectory (ploting.py:95-110: pydiffmap DiffusionMap.from_sklearn(k=64) ->
 * sklearn NearestNeighbors(n_neighbors=k).kneighbors_graph(X, mode='distance'), the rows of X = EMD/EMD.max()
 * as S-dimensional points, Euclidean metric, the query point itself included).
 * gram = X X^T (S x S row-major; a plain library GEMM on the caller's side).  Outputs, per row, the k
 * nearest rows sorted by (distance, index): idx[S*k] (int32) and dist[S*k] (Euclidean, double).
 * workspace: at least S doubles.  1 <= k <= min(S, 1024).
 */
int pilot_knn_rows(const double *gram, int S, int k, int32_t *idx, double *dist,
                   void *workspace, size_t workspace_bytes, void *stream);

/*
 * (f-2) Silhouette coefficient of every sample on the dense S x S matrix: the arithmetic of
 * Sil_computing(EMD, labels, metric) = sklearn.metrics.silhouette_score(EMD, labels, metric=metric)
 * (Trajectory.py:593-612; called at :107-113 and per resolution in ploting.py:310-324, :420-439), the ROWS of the
 * matrix as S-dimensional points.
 * metric = PILOT_METRIC_COSINE or PILOT_METRIC_EUCLIDEAN: `matrix` is the Gram matrix X X^T of the points (a plain
 * library GEMM on the caller's side); metric = PILOT_SIL_PRECOMPUTED: `matrix` is the distance matrix itself.
 * The samples come grouped by cluster: perm[S] lists the sample indices sorted by label, seg[n_labels + 1] are the
 * segment bounds inside perm, label[S] the compact label (0 .. n_labels - 1) of every sample.
 * Output sil[S]: (b - a) / max(a, b), 0 for singleton clusters; the score is their mean.
 * workspace: at least S doubles.  2 <= n_labels <= min(S - 1, 4096).
 */
#define PILOT_SIL_PRECOMPUTED 100
int pilot_silhouette_rows(const double *matrix, int S, int metric, const int32_t *perm, const int32_t *seg,
                          const int32_t *label, int n_labels, double *sil, void *workspace,
                          size_t workspace_bytes, void *stream);

/*
 * Pipe-peak microbenchmarks used as roofline denominators (SURVEY.md 8d):
 * kind 0 = FP64 FMA, 1 = FP32 FMA, 2 = FP64 mma.sync (DMMA m8n8k4).
 * Runs on `stream`, returns achieved TFLOP/s in *h_tflops (host pointer).
 */
int pilot_pipe_peak(int kind, double *h_tflops, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* PILOT_B200_H */
