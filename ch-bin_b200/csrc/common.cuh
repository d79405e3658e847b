// common.cuh -- context, error handling and launch helpers shared by the sm_100a kernels of libchbin_b200.
#pragma once

#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "chbin_b200.h"

#define CHB_WARP 32
#define CHB_FULL 0xffffffffu
#define CHB_KMAX 32          // largest AlgoNumNeighbors supported (one warp lane per neighbour slot)
#define CHB_UNOWNED INT32_MIN // tentative-label sentinel for positions another rank owns

struct chb_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    cudaStream_t own_stream = nullptr;
    // side stream (non-blocking): work that does not sit on the critical chain of a stage -- the upper-bound pass of the label
    // set-up (row_ub_kernel: only the first round's threshold_kernel reads its result) and the upload of the NEXT iteration's
    // permutation -- forked from / joined into `stream` with events
    cudaStream_t side_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_perm = nullptr;
    bool side_join_pending = false; // `stream` has not yet waited for ev_join
    bool round_counters_reset = false; // round_reset_kernel has put counters[1..3] into their pre-commit state for this round
    bool round_snapshot_pending = false; // the fused round's counters have not been read back yet (one copy at the commit)
    bool qp_fb_zeroed = false;         // ... and the QP fallback counter (counters[3]): chb_launch_qp skips its memset once
    std::string err;

    // ---- features: n x ldx float64, row pitch padded to 16 bytes, pad columns are zero
    int64_t n = 0;
    int32_t d = 0, ldx = 0;
    double *X = nullptr;
    float *Xf = nullptr;  // n x ldf FP32 copy of the features (candidate filter)
    float *nrm = nullptr; // n : |x - mu|^2 rounded up to FP32
    double *colsum = nullptr; // d : column sums of X (mu = colsum / n)
    double *colpart = nullptr; // per-256-row partial column sums (deterministic reduction)
    int64_t cap_colpart = 0;
    int32_t *seed_off = nullptr, *seed_idx = nullptr; // C + 1 offsets / seed points (initial label >= 0) sorted by (bin, index)
    int64_t cap_seed_off = 0, cap_seed_idx = 0;
    bool guess_pending = false; // first iteration after chb_set_labels: speculation starts from the nearest seed centroid
    bool guess_shared = false;  // sharded contexts exchange the speculation start (chb_guess_export / chb_guess_import): each
                                // computes the centroid terms of its OWN slots only
    bool guess_imported = false; // f_guess_all holds every slot's guess (after chb_guess_import)
    int32_t ldf = 0;
    int dist_mode = 2;    // 2: fused tensor-core Gram + selection (default); 1: FP32 candidate matrix + scan; 0: exact FP64 rows
    int gram_engine = 1;  // filter mode: 1 = tcgen05 TF32x3 tensor-core Gram (gram_tc.cu), 0 = FFMA Gram (approx.cu)
    float *Asplit = nullptr, *Bsplit = nullptr; // TF32 hi/lo split operands: rows x Kp (queries), n x Kp (points)
    int64_t cap_Asplit = 0, cap_Bsplit = 0;
    int32_t Kp = 0;
    bool bsplit_ready = false;
    bool filter_ok = true; // feature magnitudes inside the FP32 filter's validated range
    bool nmax_pending = false; // the read-back deciding filter_ok is still in flight (chb_set_features_async)
    bool wide_fused_size_ok = false; // 161 <= d <= 1024: the stage is large enough for the fused path (chb_set_labels)

    // ---- labels / slots
    int32_t C = 0;
    int64_t U = 0, u0 = 0, u1 = 0; // all query slots, owned slice [u0,u1)
    int32_t *old_label = nullptr;  // n : label at the start of the running iteration (seeds: fixed)
    int32_t *tent_pt = nullptr;    // n : tentative label of this iteration, by point
    int32_t *pos = nullptr;        // n : position in this iteration's permutation; -1 for seeds
    int32_t *qslot = nullptr;      // n : query slot of the point or -1
    int32_t *qpoint = nullptr;     // U : point of a slot
    int32_t *perm_pt = nullptr;    // U : this iteration's permutation (point indices)
    int32_t *own_pos = nullptr;    // n_own: ascending positions whose query this context owns
    int64_t n_own_pos = 0;
    int64_t *own_pos_host = nullptr;
    int64_t *perm64 = nullptr;     // U : this iteration's permutation as the caller passed it (device path of chb_iteration_begin)
    int64_t cap_perm64 = 0;
    int64_t *perm64_next = nullptr; // U : the next iteration's permutation, uploaded ahead on the side stream (chb_iteration_prefetch)
    int64_t cap_perm64_next = 0;
    const int64_t *perm_prefetch_src = nullptr; // host array the prefetched copy came from (nullptr: nothing prefetched)
    bool perm_check_pending = false; // the device-side validation of this iteration's permutation has not been read back yet
    bool own_pos_by_slot = false;  // own_pos is indexed by owned slot (device path) instead of ascending by position (host path)
    bool labels_set = false, in_iteration = false;
    std::vector<int32_t> h_lab, h_perm32, h_own32; // per-call scratch
    int32_t *pin_i32 = nullptr; // page-locked staging block of chb_set_labels
    int64_t pin_cap = 0;
    int32_t *h_qslot = nullptr; // host mirror of qslot (inside pin_i32), built on demand
    bool h_qslot_valid = false;
    int64_t *lab64 = nullptr; // n : labels widened to int64 for chb_get_labels
    int64_t cap_lab64 = 0;
    int64_t *pin_lab64 = nullptr; // page-locked staging block of chb_get_labels
    int64_t pin_lab_cap = 0;
    bool labels_staged = false; // pin_lab64 holds the current labels (they travelled with the commit that ended the iteration)
    int32_t *slot_tiles = nullptr; // per-1024-point tile counts / offsets of the slot scan
    int64_t cap_slot_tiles = 0;
    std::vector<uint8_t> h_seen;

    // ---- parameters
    int32_t k = 5, metric = CHB_METRIC_CONVEX;
    bool params_dirty = true;

    // ---- distances
    bool dist_ready = false, materialise = false;
    double *Dq = nullptr;       // (u1-u0) x n when materialised (dist_mode 0)
    double *Dscratch = nullptr; // scratch_rows x n otherwise
    int2 *packed = nullptr;     // n : packed labels for the kNN scan, rebuilt before every round
    int64_t lda = 0;            // row pitch (floats) of Aq / Ascratch: n rounded up to 4
    float *Aq = nullptr;        // (u1-u0) x lda FP32 approximate squared distances when materialised (dist_mode 1)
    float *Ascratch = nullptr;
    int64_t cap_Aq = 0, cap_Ascratch = 0;
    double *knn_dist = nullptr; // nown x C x k exact distances of the cached lists
    int64_t cap_knn_dist = 0;
    int64_t scratch_rows = 0;

    // ---- per (owned slot, bin) caches
    int32_t *knn_idx = nullptr;  // nown x C x k   canonical (distance, index) order
    int32_t *knn_cnt = nullptr;  // nown x C       -1 = never computed
    double *pair_dist = nullptr; // nown x C
    int32_t *pair_status = nullptr;
    int64_t cache_nown = 0;
    int32_t cache_C = 0, cache_k = 0;

    // ---- work list of dirty (slot_local, bin) pairs
    int2 *work = nullptr;
    int64_t work_cap = 0;
    int32_t *counters = nullptr;      // 16 ints: [0] work count, [1] first changed position, [2] n_changed, [3] QP fallback count,
                                      // [5] max |x - mu|^2 bits, [6] exact-redo pairs, [7] planned tiles, [8] tiles issued by the MMA warps
    int32_t *counters_host = nullptr; // pinned mirror (16 ints) + the commit's snapshot of all 16 device counters

    // capacities (elements) of the re-usable allocations above, so that repeated set-ups do not re-malloc
    int64_t cap_X = 0, cap_Xf = 0, cap_nrm = 0, cap_colsum = 0;
    double *stage_X = nullptr; // persistent staging area of chb_set_features
    int64_t cap_stage_X = 0;
    int64_t cap_n = 0, cap_U = 0, cap_own = 0, cap_Dq = 0, cap_scratch = 0, cap_pairs = 0, cap_knn = 0;

    // ---- distance mode 2 (fused.cu): column entries, permuted operand, candidate lists
    int32_t *f_bin_cnt = nullptr, *f_seg_off = nullptr, *f_cursor = nullptr, *f_tile_bin = nullptr, *f_ntiles = nullptr;
    int32_t *f_col_pt = nullptr, *f_col_a = nullptr, *f_col_b = nullptr;
    float *f_col_nrm = nullptr, *f_bperm = nullptr, *f_cand_key = nullptr;
    int32_t *f_cand_idx = nullptr;
    int2 *f_fb_pairs = nullptr; // (row, bin) pairs to redo exactly this round
    int2 *f_xs_slots = nullptr; // the same pairs regrouped per bin (16 <= k <= 24: exact_group_kernel redoes them)
    int64_t f_xs_cap = 0;
    int32_t f_fb_cap = 0;
    bool f_fb_worst = false; // the exact-redo list was grown to every (row, bin) pair after an overflow
    int64_t f_fb_alloc = 0; // entries allocated behind f_fb_pairs (f_fb_cap pairs + per-bin padding of the large-k path)
    int64_t f_cap_bins = 0, f_cap_cols = 0, f_cap_cand = 0, f_cap_thr = 0, f_cap_ldt = 0;
    float *f_thr = nullptr; // nown x C : largest FP32 key of the cached neighbour set (+inf: fewer than k members)
    float *f_t0 = nullptr;  // C x f_ldt : this round's admission threshold per (bin, owned slot)
    int64_t f_ldt = 0;
    float *f_a2 = nullptr;  // nown x Kp2 : TF32 [hi | lo] operand rows of the owned queries
    int64_t f_cap_a2 = 0, f_cap_bperm = 0;
    double *f_mc = nullptr, *f_mc2 = nullptr; // C x d : bin reference point minus the global mean; C : its squared norm
    int32_t *f_mcnt = nullptr;
    double *f_mcT = nullptr;        // d x Cp : the same table transposed (bins contiguous)
    int32_t *f_guess_all = nullptr; // U : bin of the nearest seed centroid of every query slot (C: none)
    int64_t f_cap_guess = 0, f_cap_mcT = 0, f_cap_seedT = 0;
    float *f_tqs = nullptr;         // U x Cp : |a_u - m_c|^2 of every query slot (slot order)
    int64_t f_cap_tqs = 0;
    float *f_seedT = nullptr;       // d x (#seeds) : centred FP32 seed contigs transposed, (bin, index) order
    int32_t *f_slot_row = nullptr;  // owned slot -> row
    float *f_sq_row = nullptr;      // per row: >= |a_q|
    int32_t *f_row_nb = nullptr, *f_row_bins = nullptr; // per row: number / list of the bins that survived pruning this round
    int32_t *f_row_pid = nullptr;   // per (row, j-th surviving bin): compact pair id of this round (compacted rounds)
    bool f_cand_dense = true;       // the candidate lists have a slot per (row, bin); false: per compact pair id only
    int64_t f_cap_mc = 0;
    float *f_tq = nullptr, *f_slack = nullptr; // C x f_ldt : |a_q - m_c|^2 and the key error bound per (bin, owned slot)
    int4 *f_items = nullptr;                   // surviving (row block, bin) work items of the fused kernel, row-block order
    int32_t *f_cta_begin = nullptr;            // sm_count + 1 : item range per CTA (balanced by tile count)
    int32_t *f_pair_row = nullptr, *f_pair_meta = nullptr, *f_mode = nullptr; // compact (row, bin) pairs: row per pair id; per-bin counters; mode flag
    float *f_ap = nullptr;                     // cap_pairs x Kp2 : query operand rows gathered in compact pair order
    int64_t f_cap_ap = 0, f_cap_pairs = 0;
    uint8_t *f_skip = nullptr;                 // (#row blocks) x C : tiles of this (row block, bin) are skipped this round
    int32_t *f_row_slot = nullptr, *f_row_pt = nullptr; // row -> owned slot / point
    float *f_ub = nullptr, *f_ubk2 = nullptr; // per row: upper bound of min_c hull distance; squared distance to the k-th nearest seed
    int32_t *f_row_guess = nullptr, *f_rhist = nullptr; // guessed bin per row; histogram / cursors of the row grouping
    float *f_ym2 = nullptr;                    // 2 (C + 1) : per-bin maxima of |y|^2 and |column term| of this round
    bool f_asplit_ready = false;

    int2 *fallback = nullptr; // pairs the small-k QP kernel hands to the general one
    int64_t fallback_cap = 0;
    double *qp_scratch = nullptr; // qp_lane.cu: the Gram matrices of one chunk of pairs, [batch of 32][entry][pair in batch]
    int64_t qp_scratch_cap = 0;   // doubles

    int64_t window = 0;
    int32_t *tent_win = nullptr; // window-sized tentative buffer for the single-context driver
    int64_t tent_win_cap = 0;

    // ---- timers: event pairs are recorded around launches and resolved lazily after a stream sync
    bool timers_on = true;
    chb_timers tm{};
    struct pending_ev { cudaEvent_t e0, e1; int stage; };
    std::vector<pending_ev> ev_pending;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev_free;
};

void chb_resolve_timers(chb_ctx *ctx); // call only when the stream is known to be idle

extern thread_local std::string g_chb_create_error;

int chb_fail(chb_ctx *ctx, int code, const char *fmt, ...);

#define CHB_CUDA(ctx, expr)                                                                             \
    do {                                                                                                \
        cudaError_t _e = (expr);                                                                        \
        if (_e != cudaSuccess)                                                                          \
            return chb_fail(ctx, _e == cudaErrorMemoryAllocation ? CHB_ENOMEM : CHB_ECUDA, "%s: %s (%s:%d)", #expr, \
                            cudaGetErrorString(_e), __FILE__, __LINE__);                               \
    } while (0)

#define CHB_CHECK(ctx, cond, code, ...)                     \
    do {                                                    \
        if (!(cond)) return chb_fail(ctx, code, __VA_ARGS__); \
    } while (0)

// ---- programmatic dependent launch (sm_90+) ---------------------------------------------------------------
// A clustering stage at 20k contigs is a chain of ~50 kernels of 3-70 us: between two of them the stream otherwise pays
// drain + launch (~2 us).  Kernels of that chain start with chb_pdl_enter() -- wait for the preceding grid (complete and
// flushed), then let the NEXT grid be scheduled -- and are launched through chb_launch_pdl, so that the next grid's CTAs
// are already resident (blocked in griddepcontrol.wait) when this one drains.  Rules: chb_pdl_enter() is the FIRST
// statement of the kernel, before any early return and before any global-memory access (a grid that exits without
// waiting would let its own dependents overtake the grid before it).  Both instructions are no-ops in a kernel launched
// the ordinary way.  CHB_NO_PDL=1 launches everything the ordinary way (A/B measurements).
#ifdef __CUDACC__
__device__ __forceinline__ void chb_pdl_enter()
{
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
// For kernels whose CTAs are all resident at once and run long (the persistent tensor-core kernel, the QP kernels, the
// exact redo): no early trigger -- the next grid's CTAs would sit beside them for the whole run (measured at 1M contigs:
// the stage 3.5 ms slower with the early trigger everywhere); the implicit trigger at CTA exit still lets the next grid
// move in while the last CTAs drain.
__device__ __forceinline__ void chb_pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

bool chb_pdl_enabled();

template <typename... KArgs, typename... Args>
inline cudaError_t chb_launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args &&...args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = chb_pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
#define CHB_PDL_LAUNCH(ctx, kern, grid, block, smem, ...) \
    CHB_CUDA(ctx, chb_launch_pdl(kern, dim3(grid), dim3(block), (size_t)(smem), (ctx)->stream, __VA_ARGS__))
#endif

enum chb_stage { CHB_ST_DISTANCE = 0, CHB_ST_KNN = 1, CHB_ST_QP = 2, CHB_ST_COMMIT = 3, CHB_ST_OTHER = 4, CHB_ST_GRAM = 5 };

// Brackets one kernel launch with events when timers are on; resolved by chb_resolve_timers.
struct chb_stage_timer {
    chb_ctx *c;
    chb_stage st;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    chb_stage_timer(chb_ctx *ctx, chb_stage s) : c(ctx), st(s)
    {
        if (!c->timers_on || st == CHB_ST_OTHER) return;
        if (c->ev_free.empty()) {
            cudaEventCreate(&e0);
            cudaEventCreate(&e1);
        } else {
            e0 = c->ev_free.back().first;
            e1 = c->ev_free.back().second;
            c->ev_free.pop_back();
        }
        cudaEventRecord(e0, c->stream);
    }
    ~chb_stage_timer()
    {
        int64_t *cnt = st == CHB_ST_DISTANCE ? &c->tm.launches_distance
                     : st == CHB_ST_KNN      ? &c->tm.launches_knn
                     : st == CHB_ST_QP       ? &c->tm.launches_qp
                     : st == CHB_ST_COMMIT   ? &c->tm.launches_commit
                     : st == CHB_ST_GRAM     ? &c->tm.launches_gram
                                             : &c->tm.launches_other;
        ++*cnt;
        if (e0) {
            cudaEventRecord(e1, c->stream);
            c->ev_pending.push_back({e0, e1, (int)st});
        }
    }
};

// ---- kernel launchers (each defined in its own .cu) ------------------------------------------------------
// distance.cu : out[r*n + i] = cdist(X[rows[r]], X[i]) with the exact scipy recipe
int chb_launch_distance_rows(chb_ctx *ctx, const int32_t *rows_dev, int64_t nrows, double *out_dev);

// approx.cu : FP32 feature copy + norms; FP32 approximate squared distance rows
int chb_launch_prep_f32(chb_ctx *ctx);
int chb_launch_approx_rows(chb_ctx *ctx, const int32_t *rows_dev, int64_t nrows, float *out_dev, int64_t ldo);

// gram_tc.cu : tcgen05 / TMA / TMEM version of the candidate-distance Gram contraction
int chb_gram_tc_prepare(chb_ctx *ctx, const int32_t *rows_dev, int64_t nrows, float *a_split, float *b_split, int32_t Kp,
                        bool do_b);
int chb_launch_gram_tc(chb_ctx *ctx, const float *a_split, const float *b_split, int32_t Kp, const int32_t *rows_dev,
                       int64_t nrows, float *out_dev, int64_t ldo);

// fused.cu : distance mode 2, Gram + per-bin selection in one tcgen05 kernel, then exact re-rank
constexpr int CHB_FUSED_RESIDENT_DMAX = 160; // widest d whose query operand stays resident in the fused kernel
bool chb_fused_supported(const chb_ctx *c); // the kernels can serve this d and k
bool chb_use_fused(const chb_ctx *c);       // api.cu: the rounds of this context run the fused path
int chb_round_fused(chb_ctx *c);
int chb_fused_setup(chb_ctx *c);  // allocations + once-per-label-set operands (idempotent)
int chb_fused_grow_redo_list(chb_ctx *c); // exact-redo list to its worst-case size (every (row, bin) pair)
int chb_fused_guess(chb_ctx *c);
int chb_fused_argmin(chb_ctx *c, const int32_t *own_pos_dev, int64_t cnt, int64_t lo, int64_t hi, int32_t *tent_dev); // argmin over surviving bins, positions in [lo, hi)
int chb_fused_mask_pair_cache(chb_ctx *c, int64_t slot0, int64_t nslots, int32_t *cnt_out, double *dist_out); // test aid  // tent_pt of every query point := bin of the nearest seed centroid
void chb_fused_free(chb_ctx *c);

// knn.cu
struct chb_knn_args {
    int filter;                // 0: `rows` = exact FP64 distances; 1: `arows` = FP32 approximate squared distances
    const float *arows;
    const float *nrm;          // |x|^2 rounded up to FP32 (filter)
    const unsigned int *nrm_max_bits;
    double eps_rel;            // |arows - d^2| <= eps_rel * (nrm[query] + nrm_max)
    const double *X;           // features, for the exact re-rank (filter)
    int32_t ldx, d;
    double *knn_dist;          // exact distances of the cached lists (filter, mode 0)
    const double *rows;        // distance rows
    int64_t row_stride;        // n
    int row_is_item;           // 0: row index = owned slot of the query; 1: row index = item (scratch rows)
    const int32_t *items;      // per CTA: position p (mode 0) or query point (mode 1)
    int64_t n_items;
    int mode;                  // 0 = round (effective labels from pos/tent/old), 1 = snapshot labels (old_label only)
    const int32_t *perm_pt, *qslot, *pos, *tent_pt, *old_label;
    const int2 *packed;        // optional: {pos, (tent << 16) | (old & 0xffff)} per point (C < 32768), 16-byte aligned
    int64_t n;
    int32_t C, k;
    int64_t u0;
    int32_t *knn_idx, *knn_cnt; // caches (mode 0) or plain outputs indexed by item (mode 1)
    int2 *work;
    int32_t *work_count;
};
int chb_launch_knn_scan(chb_ctx *ctx, const chb_knn_args &a);

// qp.cu
struct chb_qp_args {
    const double *X;
    int32_t ldx, d;
    const int2 *work;           // (row, c) pairs; row indexes knn/dist arrays
    const int32_t *work_count;  // device count (may be nullptr -> n_work)
    int64_t n_work;             // upper bound / exact count
    const int32_t *row_point;   // point index of row (query)
    const int32_t *knn_idx, *knn_cnt;
    int32_t C, k, metric;
    double *dist;
    int32_t *status;
    double *alpha; // optional rows x C x k
    int32_t *cap_count; // optional device counter: pairs whose active-set method ended on its iteration cap (CHB_QP_ITER_CAP)
};
int chb_launch_qp(chb_ctx *ctx, const chb_qp_args &a);
// qp_small.cu : k <= 5 fast path; ill-conditioned pairs are appended to `fallback`
int chb_launch_qp_small(chb_ctx *ctx, const chb_qp_args &a, int2 *fallback, int32_t *fallback_count);
// qp_mid.cu : 6 <= k <= 10
int chb_launch_qp_mid(chb_ctx *ctx, const chb_qp_args &a, int2 *fallback, int32_t *fallback_count);
// qp_lane.cu : 11 <= k <= 24 (FP64 tensor-core Gram, one lane per pair)
int chb_launch_qp_lane(chb_ctx *ctx, const chb_qp_args &a, int2 *fallback, int32_t *fallback_count);
