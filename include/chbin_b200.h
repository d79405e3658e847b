/*
 * chbin_b200.h -- C-ABI of libchbin_b200.so: the B200-native replacement for CH-Bin's clustering hot path.
 *
 * Every entry point below names the reference interface it replaces (paths relative to the reference tree,
 * kdsuneraavinash/CH-Bin).  Plain C: pointers + sizes, no torch / numpy types.  Pointers are HOST memory
 * unless the parameter name ends in `_dev`.  The context owns all device memory; the caller owns every
 * buffer it passes; no pointer is retained after the call returns (except the stream handle).
 * All functions return CHB_OK (0) or a CHB_E* code; chb_last_error() gives the message.
 * One context = one CUDA device = one host thread at a time (the reference is single-threaded,
 * ch_bin/core/clustering/algorithm.py:43-60).  Multi-GPU = one context per GPU, either one process per GPU with the label
 * exchange above this ABI (torch.distributed / NCCL on the *_dev buffers), or one process driving a device group of
 * contexts that exchanges the labels itself (chb_group_*, below).
 *
 * There is no CPU fallback: chb_create fails with CHB_ENODEV when no sm_100 device is usable.
 */
#ifndef CHBIN_B200_H
#define CHBIN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CHB_ABI_VERSION 1

enum {
    CHB_OK = 0,
    CHB_EINVAL = 1,    /* bad argument / call order          -> Python ValueError            */
    CHB_ENODEV = 2,    /* no usable CUDA device              -> Python RuntimeError          */
    CHB_ECUDA = 3,     /* CUDA runtime fault                 -> Python RuntimeError          */
    CHB_ENOMEM = 4,    /* device allocation failed           -> Python MemoryError           */
    CHB_ENOTIMPL = 5,  /* unsupported metric / solver        -> Python NotImplementedError   */
                       /*   (hull_distance.py:108, solve_qp.py:132)                          */
    CHB_EUNASSIGNED = 6 /* un-clustered points left           -> ValueError (cli/clustering.py:79-80) */
};

/* AlgoDistanceMetric (config/default.ini:18 -> hull_distance.py:90-108) */
/* "affine" (hull_distance.py:69-87) is the SVD/orthogonal-projection form of the same geometric quantity as "affine-qp"
 * (hull_distance.py:38-66): the distance to the affine hull of the neighbours.  Both run the equality-constrained
 * solve of qp.cu; affinely dependent neighbours are dropped (the reference's scipy.linalg.orth drops the matching
 * null directions), so the two agree to rounding whenever the hull is the same. */
enum { CHB_METRIC_CONVEX = 0, CHB_METRIC_AFFINE_QP = 1, CHB_METRIC_AFFINE = 2 };

/* per-QP status written by chb_hull_distance_batch (SURVEY.md 8(b) "Errors") */
enum {
    CHB_QP_OK = 0,
    CHB_QP_DEGENERATE = 1, /* an affinely dependent neighbour set was met and handled          */
    CHB_QP_ITER_CAP = 2,   /* active-set iteration cap hit; alpha feasible, near-optimal       */
    CHB_QP_EMPTY_BIN = 3   /* m == 0: distance = +inf, never selected (algorithm.py:57 never fires) */
};

typedef struct chb_ctx chb_ctx;

typedef struct chb_timers {
    /* accumulated device time in milliseconds (CUDA events on the context's stream) and launch counts
     * since chb_create / chb_reset_timers */
    double ms_distance;  /* exact FP64 distance-row kernel (scipy cdist, distance_matrix.py:26,41)     */
    double ms_knn;       /* label-segmented top-k scan (find_nearest_from_cluster, distance_matrix.py:47-62) */
    double ms_qp;        /* batched hull-distance QP kernel (hull_distance.py:7-35 + solve_qp.py:18-51)  */
    double ms_commit;    /* argmin over bins + ordered-commit check (algorithm.py:47-60)               */
    int64_t launches_distance, launches_knn, launches_qp, launches_commit, launches_other;
    int64_t qps_solved;     /* QPs actually solved on the device (includes speculative re-solves)  */
    int64_t qps_reference;  /* QPs the reference would have solved: sum over iterations of U*C     */
    int64_t rounds;         /* speculate/repair rounds executed                                    */
    int64_t rows_scanned;   /* distance rows streamed by the kNN kernel                            */
    /* distance mode 2: the fused tensor-core Gram + per-bin selection kernel (fused.cu) is timed on its own; ms_knn
     * then holds the re-rank (and the rare exact-path scans) only */
    double ms_gram;
    int64_t launches_gram;
    int64_t gram_tiles;     /* 128 x 128 (query, column) tiles contracted, counted by the MMA-issuing warps themselves:
                             * 2*128*128*3*dp8 flop each, dp8 = d rounded up to 8 */
    int64_t gram_tiles_planned; /* the same count as the work-list planner predicted it (must agree) */
    int64_t qp_iter_cap;    /* QPs of the assignment rounds whose active-set method stopped on its iteration cap (CHB_QP_ITER_CAP):
                             * their distance comes from a feasible, possibly not optimal alpha (the reference would have fallen
                             * back to cvxopt, solve_qp.py:126-129); 0 on every workload tested */
} chb_timers;

/* ---- lifetime ---------------------------------------------------------------------------------------- */
int chb_abi_version(void);
/* device_id: CUDA ordinal.  Replaces nothing in the reference (it has no device); called by the
 * AlgoQpSolver=b200 branch added at cli/clustering.py:56. */
int chb_create(chb_ctx **out, int device_id);
int chb_destroy(chb_ctx *ctx);
const char *chb_last_error(const chb_ctx *ctx); /* ctx may be NULL: error of the last failed chb_create or chb_group_* call */
/* Run every kernel on this cudaStream_t (e.g. a torch stream; NULL = the legacy default stream) instead of the
 * context's own non-blocking stream; pass CHB_OWN_STREAM to go back.  Needed whenever another library (NCCL via
 * torch.distributed) touches the *_dev buffers: both must be ordered on the same stream. */
#define CHB_OWN_STREAM ((void *)(intptr_t)-1)
int chb_set_stream(chb_ctx *ctx, void *cuda_stream);
int chb_synchronize(chb_ctx *ctx);
int chb_get_timers(chb_ctx *ctx, chb_timers *out);
int chb_reset_timers(chb_ctx *ctx);
/* enable=1: bracket every kernel with CUDA events (adds two event records per launch). Default 1. */
int chb_enable_timers(chb_ctx *ctx, int enable);

/* ---- problem set-up ---------------------------------------------------------------------------------- */
/* `samples` of fit_cluster (algorithm.py:13): n x d float64, ROW-major (the Python wrapper converts the
 * F-ordered DataFrame.values of cli/clustering.py:53).  Copied to the device in a 16-byte-pitched layout. */
int chb_set_features(chb_ctx *ctx, const double *x_rowmajor, int64_t n, int32_t d);
int chb_set_features_dev(chb_ctx *ctx, const double *x_rowmajor_dev, int64_t n, int32_t d);
/* The same, returning as soon as the repack is ENQUEUED on the context's stream: x_rowmajor_dev may be released once work
 * enqueued on that stream after this call would be ordered behind it (e.g. a stream-ordered allocator on the same stream, or
 * after chb_build_distance_matrix / chb_synchronize).  For a buffer that an NCCL broadcast on the same stream just filled. */
int chb_set_features_dev_async(chb_ctx *ctx, const double *x_rowmajor_dev, int64_t n, int32_t d);
/* Same as chb_set_features, but returns as soon as the upload is ENQUEUED: when x_rowmajor is page-locked memory the
 * copy overlaps the caller's next host work (reading labels, drawing the first permutation).  The one exception to "no
 * pointer is retained": x_rowmajor must stay valid and unchanged until chb_build_distance_matrix (or chb_synchronize)
 * returns.  Pageable memory is staged before the call returns, as with chb_set_features. */
int chb_set_features_async(chb_ctx *ctx, const double *x_rowmajor, int64_t n, int32_t d);
/* Replication across GPUs (SURVEY 8e: "the small feature matrix replicated via NCCL broadcast over NVLink").  The context's
 * device feature matrix is n x ldx doubles (ldx = d rounded up to 2, pad columns zero).  chb_features_buffer makes sure it is
 * allocated for (n, d) and returns its device address and length.  The rank that holds the host array fills it with any
 * chb_set_features* call; every rank then takes part in ONE broadcast of *count doubles at *x_dev (ordered on the context's
 * stream, see chb_set_stream); the receiving ranks finish with chb_features_commit, which derives the FP32 copy / norms the
 * set_features calls derive (asynchronous as for chb_set_features_async). */
int chb_features_buffer(chb_ctx *ctx, int64_t n, int32_t d, double **x_dev, int64_t *count);
int chb_features_commit(chb_ctx *ctx, int asynchronous);
/* `samples` exactly as the reference holds it: cli/clustering.py:53 takes DataFrame.values of a single float64 block, an
 * F-ordered (n, d) array -- element (r, t) at x_colmajor[t * n + r].  The block is uploaded as it lies in host memory and
 * transposed into the device layout on the device (no host-side np.ascontiguousarray pass).  asynchronous != 0: returns
 * once the upload is enqueued, with chb_set_features_async's lifetime rule for x_colmajor. */
int chb_set_features_colmajor(chb_ctx *ctx, const double *x_colmajor, int64_t n, int32_t d, int asynchronous);
/* Builds `samples` on the device from its two sources instead of from features.csv (SURVEY 8f row 4):
 *   kmer      (n, dk)  normalised k-mer profiles of the sub-contigs (seq2vec output, cli/features.py:84-93), row-major;
 *   cov_raw   (P, S)   RAW per-sample coverages of the P parent contigs as read from the abundance file
 *                      (coverage.py:30), row-major;
 *   parent    (n,)     row of cov_raw each sub-contig inherits (the PARENT_NAME join of cli/features.py:107).
 * The coverages are normalised as coverage.py:35-41 does -- every column by its sum, then (S > 1) every row by its sum,
 * with pandas' summation orders so that the doubles are the ones parse_coverages returns -- and the device matrix becomes
 * [kmer | coverage] (n, dk + S), the column order left after cli/clustering.py:53 drops the name / label columns.
 * cov_norm_out (P, S), optional: the normalised coverages.  dk may be 0.  NaN (missing) coverages are not supported. */
int chb_set_features_merged(chb_ctx *ctx, const double *kmer, int64_t n, int32_t dk, const double *cov_raw, int64_t P,
                            int32_t S, const int64_t *parent, double *cov_norm_out);
/* The device feature matrix back on the host, (n, d) row-major. */
int chb_get_features(chb_ctx *ctx, double *out);
/* `initial_bins` + `num_clusters` of fit_cluster (algorithm.py:14-15): int64, -1 = to be assigned.
 * Defines points_to_assign = where(initial_bins == -1) (algorithm.py:38), ascending: "query slot" u is the
 * u-th such point.  [slot_begin, slot_end) is the slice of query slots THIS context owns (multi-GPU query
 * sharding); pass 0, -1 for all. */
int chb_set_labels(chb_ctx *ctx, const int64_t *initial_bins, int64_t n, int32_t num_clusters, int64_t slot_begin,
                   int64_t slot_end);
/* num_neighbors / metric of fit_cluster (algorithm.py:17,19). */
int chb_set_params(chb_ctx *ctx, int32_t num_neighbors, int32_t metric);
/* How the distances behind find_nearest_from_cluster are produced.
 *   mode 2 (default): nothing is stored; every round the tensor cores regenerate error-bounded FP32 candidate values
 *           and the per-bin selection happens in the same kernel's epilogue (fused.cu); exact scipy-cdist values are
 *           evaluated only where the FP32 bound cannot decide.  Bins that provably cannot be a query's nearest hull are
 *           pruned first.  num_neighbors >= 25: pruning, then exact selection for the surviving pairs (no Gram kernel).
 *           The library picks the kernel from the input: d <= 160 keeps a 128-row block's query operand resident in
 *           shared memory; 161 <= d <= 1024 streams it through the TMA ring with the column operand, and runs only when
 *           the stage has at least WIDE_FUSED_MIN_PAIRS = 250 000 (query, point) pairs, U x n over ALL query slots (the
 *           same on every rank; latched by chb_set_labels, env CHB_WIDE_FUSED_MIN_PAIRS read there).  That value is a
 *           compatibility floor that keeps tiny wide stages on mode 1, not a crossover: the fused path was faster at
 *           every size measured.  Below it, and for d > 1024 or num_neighbors > 32, mode 1 serves
 *           (chb_get_distance_path tells which).
 *   mode 1: the FP32 candidate matrix of the owned query rows is kept in HBM (InMemDistMatrix=yes) or recomputed per
 *           round (no) and scanned by knn.cu; exact values for candidates only.
 *   mode 0: every exact FP64 distance is formed (3 non-fusable FP64 ops per feature) and ranked directly.
 * In all modes the neighbour sets are bit-identical to ranking scipy's exact rows.  Call before
 * chb_build_distance_matrix. */
int chb_set_distance_mode(chb_ctx *ctx, int mode);
/* The distance mode the assignment rounds will run with the current features, labels, parameters and mode setting:
 * 2 = the fused path, 1 = the FP32 candidate filter, 0 = exact rows.  Call after chb_set_labels / chb_set_params /
 * chb_set_distance_mode.  After chb_set_features_async the features' magnitude check may still be in flight; it is then
 * assumed to pass (it fails only for features near FP32 overflow or underflow). */
int chb_get_distance_path(chb_ctx *ctx, int32_t *mode_out);
/* Engine of the FP32 candidate values in distance mode 1: 1 (default) = tcgen05 tensor cores, TF32 with a 3-term
 * hi/lo split, TMA-fed, TMEM accumulators (gram_tc.cu); 0 = FFMA on the CUDA cores (approx.cu). */
int chb_set_gram_engine(chb_ctx *ctx, int engine);
/* Test aid: the FP32 candidate values A (nrows x n) of owned slots, the relative bound eps_rel with
 * |A - d^2| <= eps_rel * (nrm[query] + max nrm), and nrm (n floats, may be NULL).  Mode 1, materialised only. */
int chb_get_candidate_rows(chb_ctx *ctx, int64_t slot0, int64_t nrows, float *out, double *eps_rel, float *nrm_out);
/* Test aid: the per-(query, bin) state the assignment rounds keep for owned slots [slot0, slot0+nslots): neighbour
 * lists (nslots*C*k int32, -1 padded, order unspecified), their lengths (nslots*C) and hull distances (nslots*C). */
int chb_get_pair_cache(chb_ctx *ctx, int64_t slot0, int64_t nslots, int32_t *idx_out, int32_t *cnt_out, double *dist_out);
/* Test aid (distance mode 2): what the fused Gram + selection kernel kept in the last round for owned slots
 * [slot0, slot0+nslots): 2*KR FP32 keys and point indices per (slot, bin) pair (key = +inf: empty entry), KR in
 * *kr_out (8 or 16), and the proven error bound of those keys, slack_out[c * nslots + s] >= |key - |x_q - x_i|^2|.
 * key_out / idx_out: nslots * C * 32 entries must be available (only nslots * C * 2 * KR are written). */
int chb_get_fused_candidates(chb_ctx *ctx, int64_t slot0, int64_t nslots, float *key_out, int32_t *idx_out, float *slack_out,
                             int32_t *kr_out);
/* Test aid (fused path): the bin-pruning bounds of owned slots [slot0, slot0+nslots) for the current label set: the
 * guessed bin (num_clusters = none), ub_out >= the distance to that bin's nearest seed contig, ubk2_out >= the squared
 * distance to its k-th nearest seed (+inf when it has fewer than k or more than 128 seeds). */
int chb_get_row_bounds(chb_ctx *ctx, int64_t slot0, int64_t nslots, int32_t *guess_out, float *ub_out, float *ubk2_out);
/* create_in_mem_distance_matrix / create_distance_matrix (distance_matrix.py:12-44) for the owned query
 * rows.  materialise=1: rows are computed once (exact cdist recipe) and kept in HBM (InMemDistMatrix=yes,
 * cli/clustering.py:57-59); fails with CHB_ENOMEM if they do not fit.  materialise=0: nothing is stored,
 * distances are recomputed bit-identically inside the kNN scan whenever consulted (stands in for the
 * on-disk memmap of cli/clustering.py:61-63). */
int chb_build_distance_matrix(chb_ctx *ctx, int materialise);
/* Copy distance rows of query slots [slot0, slot0+nrows) (must be owned) to the host: nrows x n float64. */
int chb_get_distance_rows(chb_ctx *ctx, int64_t slot0, int64_t nrows, double *out);

/* ---- building blocks (parity-testable stages) -------------------------------------------------------- */
/* find_nearest_from_cluster (distance_matrix.py:47-62) for every bin at once, against an explicit label
 * vector `labels` (int64, n; the query itself is always excluded, algorithm.py:50).  queries: point indices
 * that are owned query slots' points.  idx_out: nq*C*k int64, padded with -1, each list in canonical
 * (distance, index) order; m_out: nq*C int32 = min(k, |bin|). */
int chb_knn_per_bin(chb_ctx *ctx, const int64_t *labels, const int64_t *queries, int64_t nq, int64_t *idx_out,
                    int32_t *m_out);
/* calculate_distance / convex_hull_distance (hull_distance.py:7-35,90-108) for nq*C (query, bin) pairs with
 * given neighbour lists (layout as chb_knn_per_bin's output).  dist_out: nq*C float64 (+inf where m == 0);
 * status_out: nq*C int32 (may be NULL); alpha_out: nq*C*k float64 (may be NULL). */
int chb_hull_distance_batch(chb_ctx *ctx, const int64_t *queries, int64_t nq, const int64_t *idx, const int32_t *m,
                            double *dist_out, int32_t *status_out, double *alpha_out);

/* ---- the assignment loop (algorithm.py:43-72) --------------------------------------------------------- */
/* One iteration of fit_cluster's outer loop for the permutation `perm` (U int64 point indices = this
 * iteration's np.random.permutation(points_to_assign), algorithm.py:45).  Single-context form: runs the
 * speculate/repair rounds to the exact sequential fixed point, commits, and reports n_changed =
 * sum(initial_bins != curr_bins) (algorithm.py:63,68).  labels_out (n int64) may be NULL. */
int chb_fit_iteration(chb_ctx *ctx, const int64_t *perm, int64_t U, int64_t *labels_out, int64_t *n_changed);
/* Whole fit_cluster (algorithm.py:12-76): perms = max_iterations x U.  iterations_run / converged mirror the
 * loop's break (algorithm.py:64-66) and for-else (algorithm.py:74-75); changed_per_iter: max_iterations. */
int chb_fit(chb_ctx *ctx, const int64_t *perms, int64_t U, int32_t max_iterations, int64_t *labels_out,
            int32_t *iterations_run, int32_t *converged, int64_t *changed_per_iter);
int chb_get_labels(chb_ctx *ctx, int64_t *labels_out);

/* Multi-context (one per GPU) form of one iteration; the caller merges `tent_dev` across ranks between
 * chb_round_run and chb_round_commit (all-reduce MAX over int32; un-owned entries hold INT32_MIN).
 *   chb_iteration_begin(perm)                 once per iteration
 *   repeat: chb_round_run(lo, hi, tent_dev)   tentative labels of the owned positions in [lo, hi)
 *           <all-reduce MAX tent_dev[0 .. hi-lo)>
 *           chb_round_commit(lo, hi, tent_dev, &first_changed)   -> next lo = first_changed+1, or hi if -1
 *   chb_iteration_end(&n_changed)
 * window: suggested hi-lo (chb_get_window).  A single context that owns every slot may pass tent_dev = NULL to both calls
 * (the library keeps the tentative labels itself); chb_round_run only ENQUEUES work, chb_round_commit is the sync point,
 * so the host can overlap its own work (drawing the next permutation) with a round. */
/* In distance mode 2 the permutation is validated on the device: an entry that is out of range, not an un-assigned point
 * or repeated is reported (CHB_EINVAL, same messages) by the first chb_round_commit / chb_iteration_end that follows; the
 * iteration is then abandoned and the labels stay as they were before chb_iteration_begin. */
/* chb_round_commit / chb_round_commit_end may answer *first_changed = CHB_ROUND_AGAIN (a context that owns every slot
 * only): more (query, bin) pairs than expected needed the exact redo (many identical contigs), nothing was committed, the
 * library has enlarged its list -- run the same window [lo, hi) again. */
#define CHB_ROUND_AGAIN ((int64_t)-2)
int chb_iteration_begin(chb_ctx *ctx, const int64_t *perm, int64_t U);
/* The same with the permutation already in DEVICE memory (e.g. rank 0's draw after an NCCL broadcast): distance mode 2 only. */
int chb_iteration_begin_dev(chb_ctx *ctx, const int64_t *perm_dev, int64_t U);
/* Optional: the NEXT iteration's permutation (algorithm.py:45 draws one per iteration), uploaded on a side stream while the
 * current iteration's rounds run on the device.  The next chb_iteration_begin uses that copy iff it is called with the same
 * `perm` pointer (the host array must stay unchanged in between); any other pointer simply uploads as usual.  Call it after
 * chb_round_run has enqueued a round, before the commit that synchronises.  No-op outside distance mode 2. */
int chb_iteration_prefetch(chb_ctx *ctx, const int64_t *perm, int64_t U);
int chb_round_run(chb_ctx *ctx, int64_t lo, int64_t hi, int32_t *tent_dev);
int chb_round_commit(chb_ctx *ctx, int64_t lo, int64_t hi, const int32_t *tent_dev, int64_t *first_changed);
int chb_iteration_end(chb_ctx *ctx, int64_t *n_changed);
/* chb_round_commit and -- when the round changed nothing and hi is the last position -- chb_iteration_end in ONE call and
 * ONE host synchronisation (the "is the iteration over" decision is taken on the device): *iteration_done = 1 and
 * *n_changed = sum(initial_bins != curr_bins) (algorithm.py:63,68) in that case, else *iteration_done = 0 and the caller
 * continues with the next round as after chb_round_commit. */
int chb_round_commit_end(chb_ctx *ctx, int64_t lo, int64_t hi, const int32_t *tent_dev, int64_t *first_changed,
                         int64_t *n_changed, int32_t *iteration_done);
int chb_set_window(chb_ctx *ctx, int64_t window); /* 0 = whole iteration */
int64_t chb_get_window(chb_ctx *ctx);

/* Sharded contexts (distance mode 2), optional, between chb_build_distance_matrix and the FIRST chb_iteration_begin after
 * chb_set_labels: the speculation of the first iteration starts from every query's nearest seed centroid (any start leads to
 * the same result, algorithm.py:46-60; a good one saves a round).  chb_guess_export computes that start for the OWNED slots
 * only and writes it to guess_dev (U int32, slot order; un-owned entries INT32_MIN); the caller merges the ranks' vectors
 * (all-reduce MAX) and hands the result back with chb_guess_import.  *active = 0: nothing to exchange (other distance mode,
 * no queries) -- skip the collective and the import.  Without this pair every context computes all U guesses itself. */
int chb_guess_export(chb_ctx *ctx, int32_t *guess_dev, int32_t *active);
int chb_guess_import(chb_ctx *ctx, const int32_t *guess_dev);

/* ---- device groups: one host thread, N contexts ------------------------------------------------------------- */
/* A group is made of N existing, distinct contexts (one per GPU; the same device may appear more than once, each with a
 * context of its own).  Every member keeps its own stream and owned slot range (chb_set_labels); the group only moves
 * labels and features between members, with cudaMemcpyPeerAsync ordered by events on the members' streams.  All calls are
 * enqueued from one host thread; errors are reported by chb_last_error(NULL).  Destroy the group before its members.
 * The round protocol of a sharded stage over a group:
 *   chb_group_replicate_features(g, 0)          after a chb_set_features* call on member 0, before chb_set_labels
 *   repeat: chb_round_run(member m, lo, hi, buffer of m)   for every m
 *           chb_group_all_max(g, hi - lo)
 *           chb_round_commit(member m, lo, hi, buffer of m, ...)   for every m (they agree) */
typedef struct chb_group chb_group;
int chb_group_create(chb_group **out, chb_ctx *const *members, int32_t n);
int chb_group_destroy(chb_group *g);
/* A group-owned int32 device buffer of >= count entries on member m (tentative labels, guesses), on m's device.  Valid
 * until the group is destroyed or a later call for m asks for more entries (that call waits for every member's stream). */
int chb_group_buffer(chb_group *g, int32_t m, int64_t count, int32_t **buf_dev);
/* Element-wise MAX over the members' group buffers [0, count), result in every member's buffer; enqueued on the members'
 * streams, ordered after the work already enqueued there and before anything enqueued after.  Every member must hold a
 * buffer of >= count entries. */
int chb_group_all_max(chb_group *g, int64_t count);
/* The feature matrix of member `root` (after any chb_set_features* call) into every other member, then what
 * chb_features_commit derives there (asynchronously, as chb_features_commit(ctx, 1)). */
int chb_group_replicate_features(chb_group *g, int32_t root);

/* ---- measurement aid (bench.py only) ------------------------------------------------------------------ */
/* DFMA-saturating microbenchmark: measured FP64 pipe peak of this device in TFLOP/s (FMA = 2 flop). */
int chb_measure_fp64_tflops(chb_ctx *ctx, double *tflops);
/* L2 -> SM gather bandwidth in GB/s: 1104-byte rows (one d = 137 feature row) read at random from a 22 MB buffer with
 * 16-byte L2-only loads -- the ceiling of the QP kernels' neighbour-row gather while the feature matrix is L2-resident. */
int chb_measure_l2_gbs(chb_ctx *ctx, double *gbs);

#ifdef __cplusplus
}
#endif
#endif /* CHBIN_B200_H */
