// api.cu -- host side of libchbin_b200's C-ABI (include/chbin_b200.h) plus the small ordering kernels.
//
// The assignment loop of the reference (/root/reference/ch_bin/core/clustering/algorithm.py:43-72) is a
// Gauss-Seidel sweep: the point at permutation position p sees the new labels of positions < p and last
// iteration's labels of positions > p.  It is reproduced EXACTLY by iterating a speculative map to its unique
// fixed point ("speculate + repair"):
//     T[p] = assign(p | new labels T[q] for q < p, old labels for q > p)          for every p in a window
// Round r recomputes T from the previous round's T.  All positions up to and including the first position whose
// T changed are final after the round (their inputs did not change), so the frontier strictly advances and the
// fixed point -- the sequential result, by induction over p -- is reached in at most `window` rounds; on
// binnable data it takes 2-4.  Per round only (query, bin) pairs whose neighbour list changed are re-solved.
#include <algorithm>
#include <cstdarg>
#include <cstring>
#include <vector>

#include "common.cuh"

thread_local std::string g_chb_create_error;

int chb_fail(chb_ctx *ctx, int code, const char *fmt, ...)
{
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf;
    else g_chb_create_error = buf;
    return code;
}

void chb_resolve_timers(chb_ctx *c)
{
    for (auto &p : c->ev_pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, p.e0, p.e1) == cudaSuccess) {
            switch (p.stage) {
            case CHB_ST_DISTANCE: c->tm.ms_distance += ms; break;
            case CHB_ST_KNN: c->tm.ms_knn += ms; break;
            case CHB_ST_QP: c->tm.ms_qp += ms; break;
            case CHB_ST_COMMIT: c->tm.ms_commit += ms; break;
            case CHB_ST_GRAM: c->tm.ms_gram += ms; break;
            default: break;
            }
        } else {
            (void)cudaGetLastError();
        }
        c->ev_free.emplace_back(p.e0, p.e1);
    }
    c->ev_pending.clear();
}

namespace {

template <typename T>
int dev_alloc(chb_ctx *ctx, T **p, int64_t count)
{
    if (*p) { cudaFree(*p); *p = nullptr; }
    if (count <= 0) return CHB_OK;
    cudaError_t e = cudaMalloc(reinterpret_cast<void **>(p), sizeof(T) * (size_t)count);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        *p = nullptr;
        return chb_fail(ctx, CHB_ENOMEM, "cudaMalloc of %lld bytes failed: %s", (long long)(sizeof(T) * (size_t)count),
                        cudaGetErrorString(e));
    }
    return CHB_OK;
}
// grow-only allocation: keeps the buffer when it is already large enough
template <typename T>
int dev_reserve(chb_ctx *ctx, T **p, int64_t *cap, int64_t count)
{
    if (*p && *cap >= count) return CHB_OK;
    *cap = 0;
    int rc = dev_alloc(ctx, p, count);
    if (rc == CHB_OK) *cap = count;
    return rc;
}
template <typename T>
void dev_free(T **p)
{
    if (*p) cudaFree(*p);
    *p = nullptr;
}

#define CHB_TRY(expr)                  \
    do {                               \
        int _rc = (expr);              \
        if (_rc != CHB_OK) return _rc; \
    } while (0)

inline unsigned nblk(int64_t n, int t) { return (unsigned)((n + t - 1) / t); }

// ---------------------------------------------------------------------------------------------------------
// small kernels
// ---------------------------------------------------------------------------------------------------------
__global__ void fill_i32_kernel(int32_t *p, int64_t n, int32_t v)
{
    chb_pdl_enter();
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

__global__ void set_pos_kernel(const int32_t *__restrict__ perm_pt, int64_t U, int32_t *__restrict__ pos)
{
    int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < U) pos[perm_pt[p]] = (int32_t)p;
}

__global__ void pack_labels_kernel(const int32_t *__restrict__ pos, const int32_t *__restrict__ tent, const int32_t *__restrict__ old,
                                   int64_t n, int2 *__restrict__ out)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = make_int2(pos[i], (int)(((unsigned)tent[i] << 16) | ((unsigned)old[i] & 0xffffu)));
}

// row-major n x d (contiguous) -> n x ldx (16-byte pitch, zero pad)
__global__ void repack_features_kernel(const double *__restrict__ src, int64_t n, int32_t d, int32_t ldx, double *__restrict__ dst)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * ldx) return;
    const int64_t r = i / ldx;
    const int32_t t = (int32_t)(i - r * ldx);
    dst[i] = t < d ? src[r * d + t] : 0.0;
}

// column-major n x d (the F-ordered DataFrame.values of cli/clustering.py:53: element (r, t) at src[t * n + r]) -> n x ldx
// row-major, through 32 x 32 shared-memory tiles so that both the reads and the writes are coalesced
__global__ void __launch_bounds__(256) repack_features_colmajor_kernel(const double *__restrict__ src, int64_t n, int32_t d,
                                                                       int32_t ldx, double *__restrict__ dst)
{
    __shared__ double tile[32][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int64_t r0 = (int64_t)blockIdx.x * 32;
    const int t0 = blockIdx.y * 32;
    for (int i = ty; i < 32; i += 8) {
        const int t = t0 + i;
        const int64_t r = r0 + tx;
        tile[i][tx] = (t < d && r < n) ? src[(int64_t)t * n + r] : 0.0;
    }
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        const int64_t r = r0 + i;
        const int t = t0 + tx;
        if (r < n && t < ldx) dst[r * ldx + t] = tile[tx][i];
    }
}

__global__ void gather_rows_kernel(const int32_t *__restrict__ own_pos, const int32_t *__restrict__ perm_pt, int64_t cnt,
                                   int32_t *__restrict__ rows)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < cnt) rows[i] = perm_pt[own_pos[i]];
}

// algorithm.py:47-48,57-58,60: strict '<' so the lowest bin wins ties and NaN never wins; when no bin wins the
// point keeps the label it had (min_cluster initialised to curr_bins[i_sample]).
__global__ void argmin_kernel(const int32_t *__restrict__ own_pos, int64_t cnt, const int32_t *__restrict__ perm_pt,
                              const int32_t *__restrict__ qslot, int64_t u0, const double *__restrict__ pair_dist, int32_t C,
                              const int32_t *__restrict__ old_label, int64_t lo, int32_t *__restrict__ tent)
{
    const int lane = threadIdx.x & 31;
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (w >= cnt) return;
    const int p = own_pos[w];
    const int j = perm_pt[p];
    const double *dr = pair_dist + ((int64_t)qslot[j] - u0) * C;
    double best = INFINITY;
    int bc = INT32_MAX;
    for (int c = lane; c < C; c += 32) {
        const double v = dr[c];
        if (v < best) { best = v; bc = c; } // ascending c per lane: first minimum kept
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(CHB_FULL, best, o);
        const int oc = __shfl_xor_sync(CHB_FULL, bc, o);
        if (ov < best || (ov == best && oc < bc)) { best = ov; bc = oc; }
    }
    if (lane == 0) tent[p - lo] = (best < INFINITY) ? bc : old_label[j];
}

__global__ void commit_kernel(const int32_t *__restrict__ tent, int64_t lo, int64_t hi, const int32_t *__restrict__ perm_pt,
                              int32_t *__restrict__ tent_pt, int32_t *__restrict__ counters, int32_t fb_cap)
{
    chb_pdl_enter();
    const int64_t p = lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= hi) return;
    // more pairs needed the exact redo than its list holds: this round's tentative labels are incomplete and must not be
    // committed -- the host grows the list and the caller runs the same window again (chb_round_commit)
    if (fb_cap > 0 && counters[6] > fb_cap) {
        if (p == lo) counters[1] = (int32_t)lo; // not the "nothing changed" pattern: end_if_done_kernel must not end the iteration
        return;
    }
    const int32_t v = tent[p - lo];
    const int j = perm_pt[p];
    if (v != tent_pt[j]) {
        tent_pt[j] = v;
        atomicMin(&counters[1], (int32_t)p);
    }
}

// Query slots on the device (chb_set_labels): slot of point i = number of un-assigned points before it (algorithm.py:38:
// points_to_assign is ascending) -- an exclusive scan over n flags in three small kernels (tile counts, scan of the tile
// counts, per-tile scan + scatter) instead of a host pass that writes three arrays of n entries.
constexpr int SLOT_TILE = 1024; // 256 threads x 4 points
__device__ __forceinline__ int block_exclusive_scan_256(int v, int *s_warp, int &total)
{
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(CHB_FULL, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) s_warp[w] = incl;
    __syncthreads();
    int woff = 0, tot = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int t = s_warp[i];
        if (i < w) woff += t;
        tot += t;
    }
    __syncthreads();
    total = tot;
    return woff + incl - v;
}
__global__ void __launch_bounds__(256) slots_count_kernel(const int32_t *__restrict__ lab, int64_t n, int32_t *__restrict__ tile_cnt)
{
    chb_pdl_enter();
    __shared__ int s_warp[8];
    const int64_t base = (int64_t)blockIdx.x * SLOT_TILE + threadIdx.x * 4;
    int v = 0;
#pragma unroll
    for (int u = 0; u < 4; ++u) v += (base + u < n && lab[base + u] == -1) ? 1 : 0;
    int total;
    block_exclusive_scan_256(v, s_warp, total);
    if (threadIdx.x == 0) tile_cnt[blockIdx.x] = total;
}
__global__ void __launch_bounds__(256) slots_tile_scan_kernel(int32_t *__restrict__ tile_cnt, int32_t ntiles)
{
    chb_pdl_enter();
    __shared__ int s_warp[8];
    int carry = 0;
    for (int32_t t0 = 0; t0 < ntiles; t0 += 256) {
        const int32_t t = t0 + threadIdx.x;
        const int v = t < ntiles ? tile_cnt[t] : 0;
        int total;
        const int ex = block_exclusive_scan_256(v, s_warp, total);
        if (t < ntiles) tile_cnt[t] = carry + ex;
        carry += total;
    }
}
__global__ void __launch_bounds__(256) slots_fill_kernel(const int32_t *__restrict__ lab, int64_t n, const int32_t *__restrict__ tile_off,
                                                         int32_t *__restrict__ qslot, int32_t *__restrict__ qpoint, int32_t *__restrict__ pos)
{
    chb_pdl_enter();
    __shared__ int s_warp[8];
    const int64_t base = (int64_t)blockIdx.x * SLOT_TILE + threadIdx.x * 4;
    bool f[4];
    int v = 0;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        f[u] = base + u < n && lab[base + u] == -1;
        v += f[u] ? 1 : 0;
    }
    int total;
    int slot = tile_off[blockIdx.x] + block_exclusive_scan_256(v, s_warp, total);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const int64_t i = base + u;
        if (i >= n) break;
        pos[i] = -1; // no permutation position yet (seeds keep -1 for good)
        if (f[u]) {
            qslot[i] = slot;
            qpoint[slot] = (int32_t)i;
            ++slot;
        } else {
            qslot[i] = -1;
        }
    }
}

// Device path of chb_iteration_begin: the caller's int64 permutation becomes perm_pt / pos / own_pos in one pass, and is
// validated on the way (out of range: counters[9], not a query point: counters[10]; repeats are found by
// check_perm_kernel once the scatter is complete: counters[11]) -- the first offending position of each kind, reported
// by the next commit.  An offending entry is replaced by a valid query point so that the round stays memory-safe.
__global__ void begin_perm_kernel(const int64_t *__restrict__ perm64, int64_t U, int64_t n, const int32_t *__restrict__ qslot,
                                  const int32_t *__restrict__ qpoint, int64_t u0, int64_t u1, int32_t *__restrict__ perm_pt,
                                  int32_t *__restrict__ pos, int32_t *__restrict__ own_pos, int32_t *__restrict__ counters,
                                  const int32_t *__restrict__ old_label, int32_t *__restrict__ tent_pt)
{
    chb_pdl_enter();
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n) tent_pt[p] = old_label[p]; // the iteration starts from the labels the last one ended on (grid covers max(U, n))
    if (p >= U) return;
    int64_t pt = perm64[p];
    if (pt < 0 || pt >= n) {
        atomicMin(&counters[9], (int32_t)p);
        pt = qpoint[p];
    } else if (qslot[pt] < 0) {
        atomicMin(&counters[10], (int32_t)p);
        pt = qpoint[p];
    }
    perm_pt[p] = (int32_t)pt;
    pos[pt] = (int32_t)p;
    const int64_t slot = qslot[pt];
    if (slot >= u0 && slot < u1) own_pos[slot - u0] = (int32_t)p;
}

__global__ void check_perm_kernel(const int32_t *__restrict__ perm_pt, int64_t U, const int32_t *__restrict__ pos,
                                  int32_t *__restrict__ counters)
{
    chb_pdl_enter();
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < U && pos[perm_pt[p]] != (int32_t)p) atomicMin(&counters[11], (int32_t)p);
}

// algorithm.py:63-72 on the device, taken only when the round just committed changed nothing (counters[1] still holds the
// "none" pattern): the iteration is over -- count sum(initial_bins != curr_bins) and make the new labels the old ones.
__global__ void end_if_done_kernel(int32_t *__restrict__ old_label, const int32_t *__restrict__ tent_pt, int64_t n,
                                   int32_t *__restrict__ counters, int64_t *__restrict__ lab64)
{
    chb_pdl_enter();
    if (counters[1] != 0x7f7f7f7f) return;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool ch = false;
    if (i < n) {
        const int32_t t = tent_pt[i];
        ch = old_label[i] != t;
        if (ch) old_label[i] = t;
        if (lab64) lab64[i] = t; // the caller's int64 labels, staged with this commit's read-back (stage_labels)
    }
    const unsigned m = __ballot_sync(CHB_FULL, ch);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(&counters[2], __popc(m));
}

__global__ void widen_labels_kernel(const int32_t *__restrict__ lab, int64_t n, int64_t *__restrict__ out)
{
    chb_pdl_enter();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = lab[i];
}

__global__ void count_changed_kernel(const int32_t *__restrict__ a, const int32_t *__restrict__ b, int64_t n,
                                     int32_t *__restrict__ counters)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool ch = (i < n) && (a[i] != b[i]);
    const unsigned m = __ballot_sync(CHB_FULL, ch);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(&counters[2], __popc(m));
}


int ensure_caches(chb_ctx *c)
{
    const int64_t nown = c->u1 - c->u0;
    if (c->cache_nown == nown && c->cache_C == c->C && c->cache_k == c->k && c->knn_idx) return CHB_OK;
    CHB_TRY(dev_reserve(c, &c->knn_idx, &c->cap_knn, nown * c->C * c->k));
    // exact distances of the cached lists: only the matrix-backed modes (knn.cu) keep them
    if (!chb_use_fused(c))
        CHB_TRY(dev_reserve(c, &c->knn_dist, &c->cap_knn_dist, nown * c->C * c->k));
    if (c->cap_pairs < nown * c->C) {
        CHB_TRY(dev_alloc(c, &c->knn_cnt, nown * c->C));
        CHB_TRY(dev_alloc(c, &c->pair_dist, nown * c->C));
        CHB_TRY(dev_alloc(c, &c->pair_status, nown * c->C));
        c->cap_pairs = nown * c->C;
    }
    c->cache_nown = nown;
    c->cache_C = c->C;
    c->cache_k = c->k;
    if (nown * c->C > 0) {
        // -1 in every count = "no cached neighbour set": all bytes 0xFF (the driver's memset runs at the HBM write rate; a
        // 4-byte-per-thread fill kernel reached a third of it on the 1.9 GB of the 1M x 500 configuration)
        CHB_CUDA(c, cudaMemsetAsync(c->knn_cnt, 0xFF, sizeof(int32_t) * (size_t)(nown * c->C), c->stream));
    }
    return CHB_OK;
}

int ensure_work(chb_ctx *c, int64_t items)
{
    const int64_t need = std::max<int64_t>(items * c->C, 1);
    if (need > c->work_cap) {
        CHB_TRY(dev_alloc(c, &c->work, need));
        c->work_cap = need;
    }
    return CHB_OK;
}

} // namespace

bool chb_pdl_enabled()
{
    static const bool on = getenv("CHB_NO_PDL") == nullptr;
    return on;
}

namespace {

int sync_stream(chb_ctx *c)
{
    CHB_CUDA(c, cudaStreamSynchronize(c->stream));
    chb_resolve_timers(c);
    if (c->nmax_pending) { // chb_set_features_async: the largest |x - mu|^2 has arrived now
        float nmax;
        memcpy(&nmax, &c->counters_host[5], sizeof(float));
        // the FP32 filter's error bound needs |x|^2 far from FP32 overflow / underflow; otherwise use exact rows
        c->filter_ok = (nmax > 1e-30f) && (nmax < 1e30f);
        c->nmax_pending = false;
    }
    return CHB_OK;
}

} // namespace

// Which path serves distance mode 2 -- decided here and nowhere else.  d <= 160: the fused kernel with the resident query
// operand.  161 <= d <= 1024: the fused kernel with the streamed query operand once the STAGE has at least
// WIDE_FUSED_MIN_PAIRS (query, point) pairs, U x n, else mode 1.  The pair count is the stage's, not the owned slice's, and
// it is latched by chb_set_labels, so that every rank of a sharded stage -- and every call within one stage -- takes the
// same path.  WIDE_FUSED_MIN_PAIRS is a compatibility floor, not a measured crossover: on a B200 at d = 200 the fused path
// was faster at every size measured, down to 72 k pairs (DESIGN.md section 8, tools/wide_features.py); the floor keeps the
// tiniest wide stages (< 250 k pairs, e.g. 500 contigs) on the mode-1 path they took before the streamed kernel existed.
// CHB_WIDE_FUSED_MIN_PAIRS overrides it (read at chb_set_labels).  Otherwise (d > 1024, k > 32, features outside the FP32
// filter's range) mode 1 or 0 serves.
constexpr int64_t WIDE_FUSED_MIN_PAIRS = 250000;
static int64_t wide_fused_min_pairs()
{
    const char *e = getenv("CHB_WIDE_FUSED_MIN_PAIRS");
    return e ? (int64_t)atoll(e) : WIDE_FUSED_MIN_PAIRS;
}
bool chb_use_fused(const chb_ctx *c)
{
    if (!(c->dist_mode == 2 && c->filter_ok && chb_fused_supported(c))) return false;
    return c->d <= CHB_FUSED_RESIDENT_DMAX || c->wide_fused_size_ok;
}

// =========================================================================================================
extern "C" {

int chb_abi_version(void) { return CHB_ABI_VERSION; }

const char *chb_last_error(const chb_ctx *ctx) { return ctx ? ctx->err.c_str() : g_chb_create_error.c_str(); }

int chb_create(chb_ctx **out, int device_id)
{
    if (!out) return chb_fail(nullptr, CHB_EINVAL, "chb_create: out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        (void)cudaGetLastError();
        return chb_fail(nullptr, CHB_ENODEV, "no CUDA device available (%s); libchbin_b200 has no CPU fallback",
                        e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    }
    if (device_id < 0 || device_id >= ndev)
        return chb_fail(nullptr, CHB_EINVAL, "device_id %d out of range [0,%d)", device_id, ndev);
    cudaDeviceProp prop{};
    if (cudaGetDeviceProperties(&prop, device_id) != cudaSuccess)
        return chb_fail(nullptr, CHB_ECUDA, "cudaGetDeviceProperties failed");
    if (prop.major != 10)
        return chb_fail(nullptr, CHB_ENODEV, "device %d is sm_%d%d; libchbin_b200 is built for sm_100a only", device_id,
                        prop.major, prop.minor);
    if (cudaSetDevice(device_id) != cudaSuccess) return chb_fail(nullptr, CHB_ECUDA, "cudaSetDevice failed");
    chb_ctx *c = new chb_ctx();
    c->device = device_id;
    c->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete c;
        return chb_fail(nullptr, CHB_ECUDA, "cudaStreamCreate failed");
    }
    c->stream = c->own_stream;
    if (cudaStreamCreateWithFlags(&c->side_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&c->ev_perm, cudaEventDisableTiming) != cudaSuccess) {
        delete c;
        return chb_fail(nullptr, CHB_ECUDA, "side stream / event creation failed");
    }
    if (cudaMalloc(&c->counters, sizeof(int32_t) * 16) != cudaSuccess ||
        cudaMallocHost(&c->counters_host, sizeof(int32_t) * 32) != cudaSuccess) {
        delete c;
        return chb_fail(nullptr, CHB_ENOMEM, "counter allocation failed");
    }
    cudaMemsetAsync(c->counters, 0, sizeof(int32_t) * 16, c->stream);
    memset(c->counters_host, 0, sizeof(int32_t) * 32);
    *out = c;
    return CHB_OK;
}

int chb_destroy(chb_ctx *c)
{
    if (!c) return CHB_OK;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    if (c->side_stream) cudaStreamSynchronize(c->side_stream);
    chb_resolve_timers(c);
    for (auto &p : c->ev_free) { cudaEventDestroy(p.first); cudaEventDestroy(p.second); }
    dev_free(&c->X); dev_free(&c->old_label); dev_free(&c->tent_pt); dev_free(&c->pos); dev_free(&c->qslot);
    dev_free(&c->perm64); dev_free(&c->perm64_next); dev_free(&c->lab64); dev_free(&c->slot_tiles); dev_free(&c->qpoint); dev_free(&c->perm_pt); dev_free(&c->own_pos); dev_free(&c->Dq); dev_free(&c->Dscratch);
    dev_free(&c->knn_idx); dev_free(&c->knn_cnt); dev_free(&c->pair_dist); dev_free(&c->pair_status);
    dev_free(&c->work); dev_free(&c->counters); dev_free(&c->tent_win); dev_free(&c->fallback); dev_free(&c->qp_scratch);
    dev_free(&c->Xf); dev_free(&c->nrm); dev_free(&c->packed); dev_free(&c->Asplit); dev_free(&c->Bsplit); dev_free(&c->colsum); dev_free(&c->stage_X); dev_free(&c->colpart); dev_free(&c->seed_off); dev_free(&c->seed_idx);
    chb_fused_free(c); dev_free(&c->Aq); dev_free(&c->Ascratch); dev_free(&c->knn_dist);
    if (c->counters_host) cudaFreeHost(c->counters_host);
    if (c->pin_i32) cudaFreeHost(c->pin_i32);
    if (c->pin_lab64) cudaFreeHost(c->pin_lab64);
    delete[] c->own_pos_host;
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_join) cudaEventDestroy(c->ev_join);
    if (c->ev_perm) cudaEventDestroy(c->ev_perm);
    if (c->side_stream) cudaStreamDestroy(c->side_stream);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
    return CHB_OK;
}

int chb_set_stream(chb_ctx *c, void *cuda_stream)
{
    CHB_CHECK(c, c, CHB_EINVAL, "ctx is NULL");
    CHB_CUDA(c, cudaSetDevice(c->device));
    CHB_TRY(sync_stream(c));
    CHB_CUDA(c, cudaStreamSynchronize(c->side_stream));
    // (void*)-1 = back to the context's own stream; anything else (including NULL, the legacy default stream) is adopted
    c->stream = (cuda_stream == reinterpret_cast<void *>(static_cast<intptr_t>(-1))) ? c->own_stream
                                                                                     : reinterpret_cast<cudaStream_t>(cuda_stream);
    return CHB_OK;
}

int chb_synchronize(chb_ctx *c)
{
    CHB_CHECK(c, c, CHB_EINVAL, "ctx is NULL");
    return sync_stream(c);
}

int chb_get_timers(chb_ctx *c, chb_timers *out)
{
    CHB_CHECK(c, c && out, CHB_EINVAL, "NULL argument");
    CHB_TRY(sync_stream(c));
    *out = c->tm;
    return CHB_OK;
}

int chb_reset_timers(chb_ctx *c)
{
    CHB_CHECK(c, c, CHB_EINVAL, "ctx is NULL");
    CHB_TRY(sync_stream(c));
    c->tm = chb_timers{};
    return CHB_OK;
}

int chb_enable_timers(chb_ctx *c, int enable)
{
    CHB_CHECK(c, c, CHB_EINVAL, "ctx is NULL");
    c->timers_on = enable != 0;
    return CHB_OK;
}

static inline bool use_filter(const chb_ctx *c) { return c->dist_mode >= 1 && c->filter_ok; }
static inline bool use_fused(const chb_ctx *c) { return chb_use_fused(c); }

// FP32 candidate rows for `nrows` query points (device list rows_dev), through the selected Gram engine
static int candidate_rows(chb_ctx *c, const int32_t *rows_dev, int64_t nrows, float *out, int64_t ldo)
{
    if (c->gram_engine == 0) return chb_launch_approx_rows(c, rows_dev, nrows, out, ldo);
    c->Kp = (3 * c->d + 31) & ~31;
    if (!c->bsplit_ready) {
        CHB_TRY(dev_reserve(c, &c->Bsplit, &c->cap_Bsplit, c->n * c->Kp));
    }
    CHB_TRY(dev_reserve(c, &c->Asplit, &c->cap_Asplit, nrows * c->Kp));
    CHB_TRY(chb_gram_tc_prepare(c, rows_dev, nrows, c->Asplit, c->Bsplit, c->Kp, !c->bsplit_ready));
    c->bsplit_ready = true;
    return chb_launch_gram_tc(c, c->Asplit, c->Bsplit, c->Kp, rows_dev, nrows, out, ldo);
}

static void fill_filter_args(chb_ctx *c, chb_knn_args &a, bool filt)
{
    a.filter = filt ? 1 : 0;
    a.nrm = c->nrm;
    a.nrm_max_bits = reinterpret_cast<const unsigned int *>(&c->counters[5]);
    a.eps_rel = c->gram_engine == 0 ? (double)(c->d + 16) * 1.1920928955078125e-07   // (d + 16) * 2^-23, approx.cu
                                    : (double)(3 * c->d + 64) * 1.1920928955078125e-07; // (3d + 64) * 2^-23, gram_tc.cu
    a.X = c->X;
    a.ldx = c->ldx;
    a.d = c->d;
}

// ---------------------------------------------------------------------------------------------------------
// Shapes and device arrays of a new feature matrix (shared by every chb_set_features* entry point)
static int features_begin(chb_ctx *c, int64_t n, int32_t d)
{
    CHB_CHECK(c, n < INT32_MAX, CHB_EINVAL, "n = %lld exceeds the 32-bit point index range", (long long)n);
    CHB_CUDA(c, cudaSetDevice(c->device));
    c->n = n;
    c->d = d;
    c->ldx = (d + 1) & ~1; // 16-byte row pitch
    c->ldf = (d + 3) & ~3;
    if (c->cap_X < n * c->ldx) { CHB_TRY(dev_alloc(c, &c->X, n * c->ldx)); c->cap_X = n * c->ldx; }
    if (c->cap_Xf < n * c->ldf) { CHB_TRY(dev_alloc(c, &c->Xf, n * c->ldf)); c->cap_Xf = n * c->ldf; }
    if (c->cap_nrm < n) { CHB_TRY(dev_alloc(c, &c->nrm, n)); c->cap_nrm = n; }
    if (c->cap_colsum < d) { CHB_TRY(dev_alloc(c, &c->colsum, d)); c->cap_colsum = d; }
    return CHB_OK;
}

// Derived arrays (FP32 copy, centred norms) once c->X holds the rows; invalidates everything built on the old matrix
static int features_finish(chb_ctx *c, bool defer_sync)
{
    CHB_TRY(chb_launch_prep_f32(c));
    CHB_CUDA(c, cudaMemcpyAsync(&c->counters_host[5], &c->counters[5], sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    c->nmax_pending = true; // resolved by the next stream synchronisation (sync_stream)
    if (!defer_sync) CHB_TRY(sync_stream(c));
    c->dist_ready = false;
    c->labels_set = false;
    c->bsplit_ready = false;
    c->f_asplit_ready = false;
    return CHB_OK;
}

static int set_features_common(chb_ctx *c, const double *src, int64_t n, int32_t d, cudaMemcpyKind kind, bool defer_sync = false,
                               bool colmajor = false)
{
    CHB_CHECK(c, c, CHB_EINVAL, "ctx is NULL");
    CHB_CHECK(c, src && n > 0 && d > 0, CHB_EINVAL, "samples must be a non-empty (n, d) float64 array");
    CHB_TRY(features_begin(c, n, d));
    {
        // one contiguous copy into a persistent staging buffer (a strided 2-D copy from pageable host memory is several
        // times slower, and allocating / freeing the staging area per call costs more than the copy), then repack
        const double *dsrc = src;
        if (kind == cudaMemcpyHostToDevice) {
            CHB_TRY(dev_reserve(c, &c->stage_X, &c->cap_stage_X, n * (int64_t)d));
            CHB_CUDA(c, cudaMemcpyAsync(c->stage_X, src, sizeof(double) * (size_t)n * d, cudaMemcpyHostToDevice, c->stream));
            dsrc = c->stage_X;
        }
        if (colmajor) {
            dim3 grid(nblk(n, 32), nblk(c->ldx, 32));
            repack_features_colmajor_kernel<<<grid, 256, 0, c->stream>>>(dsrc, n, d, c->ldx, c->X);
        } else {
            repack_features_kernel<<<nblk(n * c->ldx, 256), 256, 0, c->stream>>>(dsrc, n, d, c->ldx, c->X);
        }
        ++c->tm.launches_other;
        CHB_CUDA(c, cudaGetLastError());
    }
    return features_finish(c, defer_sync);
}

// ---------------------------------------------------------------------------------------------------------
// Coverage normalisation + feature merge on the device (coverage.py:35-41, cli/features.py:106-109).
//
// The reference divides every coverage column by its sum (DataFrame.sum(axis=0): numpy add.reduce over a contiguous
// float64 axis = pairwise summation: halves split at multiples of 8 down to leaves of <= 128 elements, each leaf summed
// with eight running sums), then -- with more than one sample -- every row by its sum (DataFrame.sum(axis=1): a
// left-to-right sequential sum over the columns).  Both orders are reproduced so that the merged rows are the same doubles
// pandas would have written (pinned by tests/golden, generated from coverage.py itself).
//
// The shape of the pairwise tree depends on P only: the host lists the leaves and a post-order program
// (>= 0: push that leaf's sum, -1: add the two topmost); leaves are summed in parallel, the program is run per column.
static void pairwise_plan(int64_t off, int64_t n, std::vector<int32_t> &leaf, std::vector<int32_t> &prog)
{
    if (n <= 128) {
        prog.push_back((int32_t)(leaf.size() / 2));
        leaf.push_back((int32_t)off);
        leaf.push_back((int32_t)n);
        return;
    }
    int64_t n2 = n / 2;
    n2 -= n2 % 8;
    pairwise_plan(off, n2, leaf, prog);
    pairwise_plan(off + n2, n - n2, leaf, prog);
    prog.push_back(-1);
}

__global__ void cov_leaf_sum_kernel(const double *__restrict__ raw, int32_t S, const int32_t *__restrict__ leaf, int32_t nleaf,
                                    double *__restrict__ leafsum)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)nleaf * S) return;
    const int32_t l = (int32_t)(i / S), j = (int32_t)(i - (int64_t)l * S);
    const int32_t n = leaf[2 * l + 1];
    const double *a = raw + (int64_t)leaf[2 * l] * S + j;
    double res;
    if (n < 8) {
        res = -0.0;
        for (int32_t t = 0; t < n; ++t) res = __dadd_rn(res, a[(int64_t)t * S]);
    } else {
        double r[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) r[u] = a[(int64_t)u * S];
        int32_t t = 8;
        for (; t < n - (n % 8); t += 8) {
#pragma unroll
            for (int u = 0; u < 8; ++u) r[u] = __dadd_rn(r[u], a[(int64_t)(t + u) * S]);
        }
        res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])), __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
        for (; t < n; ++t) res = __dadd_rn(res, a[(int64_t)t * S]);
    }
    leafsum[i] = res;
}

__global__ void cov_col_total_kernel(const double *__restrict__ leafsum, int32_t S, const int32_t *__restrict__ prog, int32_t nprog,
                                     double *__restrict__ colsum)
{
    const int32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= S) return;
    double st[48]; // tree depth <= log2(2^31 / 64) + 1
    int sp = 0;
    for (int32_t t = 0; t < nprog; ++t) {
        const int32_t op = prog[t];
        if (op >= 0) {
            st[sp++] = leafsum[(int64_t)op * S + j];
        } else {
            --sp;
            st[sp - 1] = __dadd_rn(st[sp - 1], st[sp]);
        }
    }
    colsum[j] = st[0];
}

__global__ void cov_normalise_kernel(const double *__restrict__ raw, int64_t P, int32_t S, const double *__restrict__ colsum,
                                     double *__restrict__ out)
{
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const double *a = raw + p * S;
    double *o = out + p * S;
    if (S == 1) { // a single sample is normalised over the column only (coverage.py:38)
        o[0] = __ddiv_rn(a[0], colsum[0]);
        return;
    }
    double rs = __ddiv_rn(a[0], colsum[0]);
    for (int32_t j = 1; j < S; ++j) rs = __dadd_rn(rs, __ddiv_rn(a[j], colsum[j]));
    for (int32_t j = 0; j < S; ++j) o[j] = __ddiv_rn(__ddiv_rn(a[j], colsum[j]), rs);
}

// X[i] = [ kmer[i] | cov[parent[i]] | 0-pad ]   (column order of the merged frame once the name / label columns are dropped,
// cli/features.py:106-109 and cli/clustering.py:53)
__global__ void merge_features_kernel(const double *__restrict__ kmer, int32_t dk, const double *__restrict__ cov, int32_t S,
                                      const int64_t *__restrict__ parent, int64_t n, int32_t ldx, double *__restrict__ dst)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * ldx) return;
    const int64_t r = i / ldx;
    const int32_t t = (int32_t)(i - r * ldx);
    double v = 0.0;
    if (t < dk) v = kmer[r * dk + t];
    else if (t < dk + S) v = cov[parent[r] * S + (t - dk)];
    dst[i] = v;
}

int chb_set_features_merged(chb_ctx *c, const double *kmer, int64_t n, int32_t dk, const double *cov_raw, int64_t P, int32_t S,
                            const int64_t *parent, double *cov_norm_out)
{
    CHB_CHECK(c, c, CHB_EINVAL, "ctx is NULL");
    CHB_CHECK(c, n > 0 && dk >= 0 && (dk == 0 || kmer), CHB_EINVAL, "k-mer profiles must be an (n, dk) float64 array");
    CHB_CHECK(c, cov_raw && P > 0 && S > 0 && P < INT32_MAX, CHB_EINVAL, "coverages must be a non-empty (P, S) float64 array");
    CHB_CHECK(c, parent, CHB_EINVAL, "parent index (n,) is NULL");
    for (int64_t i = 0; i < n; ++i)
        CHB_CHECK(c, parent[i] >= 0 && parent[i] < P, CHB_EINVAL, "parent[%lld] = %lld is not a coverage row (P = %lld)", (long long)i,
                  (long long)parent[i], (long long)P);
    const int32_t d = dk + S;
    CHB_TRY(features_begin(c, n, d));

    std::vector<int32_t> leaf, prog;
    pairwise_plan(0, P, leaf, prog);
    const int32_t nleaf = (int32_t)(leaf.size() / 2), nprog = (int32_t)prog.size();
    // staging block (doubles): kmer | raw | normalised | column sums | leaf sums | parent (int64) | leaf table + program (int32)
    const int64_t o_raw = n * (int64_t)dk, o_cov = o_raw + P * S, o_cs = o_cov + P * S, o_ls = o_cs + S, o_par = o_ls + (int64_t)nleaf * S,
                  o_tab = o_par + n, total = o_tab + (2 * (int64_t)nleaf + nprog + 1) / 2 + 1;
    CHB_TRY(dev_reserve(c, &c->stage_X, &c->cap_stage_X, total));
    double *s = c->stage_X;
    int32_t *tab = reinterpret_cast<int32_t *>(s + o_tab);
    if (dk > 0) CHB_CUDA(c, cudaMemcpyAsync(s, kmer, sizeof(double) * (size_t)n * dk, cudaMemcpyHostToDevice, c->stream));
    CHB_CUDA(c, cudaMemcpyAsync(s + o_raw, cov_raw, sizeof(double) * (size_t)P * S, cudaMemcpyHostToDevice, c->stream));
    CHB_CUDA(c, cudaMemcpyAsync(s + o_par, parent, sizeof(int64_t) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CHB_CUDA(c, cudaMemcpyAsync(tab, leaf.data(), sizeof(int32_t) * leaf.size(), cudaMemcpyHostToDevice, c->stream));
    CHB_CUDA(c, cudaMemcpyAsync(tab + 2 * nleaf, prog.data(), sizeof(int32_t) * prog.size(), cudaMemcpyHostToDevice, c->stream));
    cov_leaf_sum_kernel<<<nblk((int64_t)nleaf * S, 128), 128, 0, c->stream>>>(s + o_raw, S, tab, nleaf, s + o_ls);
    cov_col_total_kernel<<<nblk(S, 32), 32, 0, c->stream>>>(s + o_ls, S, tab + 2 * nleaf, nprog, s + o_cs);
    cov_normalise_kernel<<<nblk(P, 128), 128, 0, c->stream>>>(s + o_raw, P, S, s + o_cs, s + o_cov);
    merge_features_kernel<<<nblk(n * c->ldx, 256), 256, 0, c->stream>>>(s, dk, s + o_cov, S, reinterpret_cast<const int64_t *>(s + o_par), n,
                                                                        c->ldx, c->X);
    c->tm.launches_other += 4;
    CHB_CUDA(c, cudaGetLastError());
    if (cov_norm_out)
        CHB_CUDA(c, cudaMemcpyAsync(cov_norm_out, s + o_cov, sizeof(double) * (size_t)P * S, cudaMemcpyDeviceToHost, c->stream));
    return features_finish(c, false);
}

int chb_get_features(chb_ctx *c, double *out)
{
    CHB_CHECK(c, c && out, CHB_EINVAL, "NULL argument");
    CHB_CHECK(c, c->X && c->n > 0, CHB_EINVAL, "get_features: no feature matrix yet");
    CHB_CUDA(c, cudaSetDevice(c->device));
    CHB_CUDA(c, cudaMemcpy2DAsync(out, sizeof(double) * c->d, c->X, sizeof(double) * c->ldx, sizeof(double) * c->d, (size_t)c->n,
                                  cudaMemcpyDeviceToHost, c->stream));
    return sync_stream(c);
}

int chb_set_gram_engine(chb_ctx *c, int engine)
{
    CHB_CHECK(c, c, CHB_EINVAL, "ctx is NULL");
    CHB_CHECK(c, engine == 0 || engine == 1, CHB_EINVAL, "gram engine must be 0 (FFMA) or 1 (tcgen05 TF32x3)");
    if (engine != c->gram_engine) { c->dist_ready = false; c->cache_nown = -1; }
    c->gram_engine = engine;
    return CHB_OK;
}

int chb_get_candidate_rows(chb_ctx *c, int64_t slot0, int64_t nrows, float *out, double *eps_rel, float *nrm_out)
{
    CHB_CHECK(c, c && out, CHB_EINVAL, "NULL argument");
    CHB_CHECK(c, c->dist_ready && use_filter(c) && !use_fused(c) && c->materialise, CHB_EINVAL,
              "candidate rows exist only in distance mode 1 with a materialised matrix");
    CHB_CHECK(c, slot0 >= c->u0 && nrows >= 0 && slot0 + nrows <= c->u1, CHB_EINVAL, "slots not owned");
    CHB_CUDA(c, cudaSetDevice(c->device));
    CHB_CUDA(c, cudaMemcpy2DAsync(out, sizeof(float) * c->n, c->Aq + (slot0 - c->u0) * c->lda, sizeof(float) * c->lda,
                                  sizeof(float) * c->n, (size_t)nrows, cudaMemcpyDeviceToHost, c->stream));
    if (nrm_out) CHB_CUDA(c, cudaMemcpyAsync(nrm_out, c->nrm, sizeof(float) * (size_t)c->n, cudaMemcpyDeviceToHost, c->stream));
    if (eps_rel) {
        chb_knn_args a{};
        fill_filter_args(c, a, true);
        *eps_rel = a.eps_rel;
    }
    return sync_stream(c);
}

int chb_get_pair_cache(chb_ctx *c, int64_t slot0, int64_t nslots, int32_t *idx_out, int32_t *cnt_out, double *dist_out)
{
    CHB_CHECK(c, c && idx_out && cnt_out && dist_out, CHB_EINVAL, "NULL argument");
    CHB_CHECK(c, c->knn_idx && slot0 >= c->u0 && nslots >= 0 && slot0 + nslots <= c->u1, CHB_EINVAL, "slots not owned / no cache yet");
    CHB_CUDA(c, cudaSetDevice(c->device));
    const int64_t r0 = slot0 - c->u0, np = nslots * c->C;
    CHB_CUDA(c, cudaMemcpyAsync(idx_out, c->knn_idx + r0 * c->C * c->k, sizeof(int32_t) * (size_t)np * c->k, cudaMemcpyDeviceToHost, c->stream));
    CHB_CUDA(c, cudaMemcpyAsync(cnt_out, c->knn_cnt + r0 * c->C, sizeof(int32_t) * (size_t)np, cudaMemcpyDeviceToHost, c->stream));
    CHB_CUDA(c, cudaMemcpyAsync(dist_out, c->pair_dist + r0 * c->C, sizeof(double) * (size_t)np, cudaMemcpyDeviceToHost, c->stream));
    CHB_TRY(sync_stream(c));
    // distance mode 2 keeps no state for the bins its bounds ruled out: report them as "no neighbours, distance +inf"
    if (use_fused(c) && c->f_row_nb) CHB_TRY(chb_fused_mask_pair_cache(c, slot0, nslots, cnt_out, dist_out));
    return CHB_OK;
}

int chb_set_distance_mode(chb_ctx *c, int mode)
{
    CHB_CHECK(c, c, CHB_EINVAL, "ctx is NULL");
    CHB_CHECK(c, mode >= 0 && mode <= 2, CHB_EINVAL,
              "distance mode must be 0 (exact rows), 1 (FP32 filter + exact re-rank) or 2 (fused tensor-core Gram + selection)");
    if (mode != c->dist_mode) { c->dist_ready = false; c->cache_nown = -1; }
    c->dist_mode = mode;
    return CHB_OK;
}

int chb_get_distance_path(chb_ctx *c, int32_t *mode_out)
{
    CHB_CHECK(c, c && mode_out, CHB_EINVAL, "NULL argument");
    *mode_out = use_fused(c) ? 2 : (use_filter(c) ? 1 : 0);
    return CHB_OK;
}

int chb_set_features(chb_ctx *c, const double *x, int64_t n, int32_t d)
{
    return set_features_common(c, x, n, d, cudaMemcpyHostToDevice);
}
int chb_set_features_async(chb_ctx *c, const double *x, int64_t n, int32_t d)
{
    return set_features_common(c, x, n, d, cudaMemcpyHostToDevice, true);
}
int chb_set_features_colmajor(chb_ctx *c, const double *x, int64_t n, int32_t d, int asynchronous)
{
    return set_features_common(c, x, n, d, cudaMemcpyHostToDevice, asynchronous != 0, true);
}
int chb_set_features_dev(chb_ctx *c, const double *x_dev, int64_t n, int32_t d)
{
    return set_features_common(c, x_dev, n, d, cudaMemcpyDeviceToDevice);
}
int chb_set_features_dev_async(chb_ctx *c, const double *x_dev, int64_t n, int32_t d)
{
    return set_features_common(c, x_dev, n, d, cudaMemcpyDeviceToDevice, true);
}
// The device feature matrix itself (n x ldx, 16-byte row pitch): allocated for (n, d) if need be.  One rank fills it with any
// chb_set_features* call, broadcasts `count` doubles from *x_dev over NCCL, and the receivers call chb_features_commit.
int chb_features_buffer(chb_ctx *c, int64_t n, int32_t d, double **x_dev, int64_t *count)
{
    CHB_CHECK(c, c && x_dev && count, CHB_EINVAL, "NULL argument");
    CHB_CHECK(c, n > 0 && d > 0, CHB_EINVAL, "samples must be a non-empty (n, d) float64 array");
    CHB_TRY(features_begin(c, n, d));
    *x_dev = c->X;
    *count = n * (int64_t)c->ldx;
    return CHB_OK;
}
int chb_features_commit(chb_ctx *c, int asynchronous)
{
    CHB_CHECK(c, c, CHB_EINVAL, "ctx is NULL");
    CHB_CHECK(c, c->X && c->n > 0, CHB_EINVAL, "features_commit: call chb_features_buffer first");
    CHB_CUDA(c, cudaSetDevice(c->device));
    return features_finish(c, asynchronous != 0);
}

int chb_set_labels(chb_ctx *c, const int64_t *bins, int64_t n, int32_t C, int64_t slot_begin, int64_t slot_end)
{
    CHB_CHECK(c, c, CHB_EINVAL, "ctx is NULL");
    CHB_CHECK(c, c->X && n == c->n, CHB_EINVAL, "set_labels: call chb_set_features first with the same n");
    CHB_CHECK(c, bins && C >= 1, CHB_EINVAL, "initial_bins is NULL or num_clusters < 1");
    CHB_CUDA(c, cudaSetDevice(c->device));
    c->labels_set = false; // the staging block (and with it the host mirror of the slots) is rewritten below
    c->labels_staged = false;
    c->perm_prefetch_src = nullptr; // a permutation prefetched for the previous label set is void
    // Host staging in ONE page-locked block: lab[n] | qslot[n] | qpoint[n] | seed_idx[n] | seed_off[C + 1].  Copies from
    // page-locked memory neither stage nor wait for earlier work on the stream, so they (and the host loops here) overlap a
    // feature upload still in flight (chb_set_features_async).  The block is rewritten by the next chb_set_labels only.
    {
        const int64_t need = 4 * n + C + 1;
        if (c->pin_cap < need) {
            if (c->pin_i32) cudaFreeHost(c->pin_i32);
            c->pin_i32 = nullptr;
            c->pin_cap = 0;
            CHB_CUDA(c, cudaMallocHost(reinterpret_cast<void **>(&c->pin_i32), sizeof(int32_t) * (size_t)need));
            c->pin_cap = need;
        }
    }
    int32_t *lab = c->pin_i32, *qs = lab + n, *qp = qs + n, *seed_idx = qp + n, *seed_off = seed_idx + n;
    c->h_qslot = qs;          // host mirror of the slots: only the host path of chb_iteration_begin reads it ...
    c->h_qslot_valid = false; // ... and builds it on first use (ensure_host_slots)
    for (int32_t b = 0; b <= C; ++b) seed_off[b] = 0;
    int64_t ns = 0;
    int32_t *seed_tmp = qp; // seeds in index order first (compact), grouped by bin into seed_idx below
    {
        // one pass over n: labels to int32 and the compact seed list (a rarely taken branch); range check folded into a
        // min / max.  The query slots themselves are derived on the device (slots_*_kernel).
        // two passes: a branch-free one the compiler vectorises (narrowing + min / max), then the compaction over the int32
        // copy, eight labels at a time -- most blocks hold no seed (-1 & ... & -1 == -1) and are skipped.  At 1M contigs
        // this loop is on every rank's critical path (2 ms of a 12 ms stage on eight GPUs before the split).
        int64_t mn = 0, mx = -1;
        for (int64_t i = 0; i < n; ++i) {
            const int64_t b = bins[i];
            mn = b < mn ? b : mn;
            mx = b > mx ? b : mx;
            lab[i] = (int32_t)b;
        }
        int64_t i = 0;
        for (; i + 8 <= n; i += 8) {
            const int32_t *l = lab + i;
            if ((l[0] & l[1] & l[2] & l[3] & l[4] & l[5] & l[6] & l[7]) == -1) continue;
            for (int u = 0; u < 8; ++u)
                if (l[u] != -1) seed_tmp[ns++] = (int32_t)(i + u);
        }
        for (; i < n; ++i)
            if (lab[i] != -1) seed_tmp[ns++] = (int32_t)i;
        if (mn < -1 || mx >= C) {
            for (int64_t i = 0; i < n; ++i)
                CHB_CHECK(c, bins[i] >= -1 && bins[i] < C, CHB_EINVAL, "initial_bins[%lld] = %lld outside [-1, %d)", (long long)i,
                          (long long)bins[i], C);
        }
    }
    const int64_t U = n - ns;
    // seed contigs sorted by (bin, index): the bin reference points are summed in this fixed order on every rank.  Stable
    // counting sort over the ns seeds only.
    for (int64_t s = 0; s < ns; ++s) ++seed_off[lab[seed_tmp[s]] + 1];
    for (int32_t b = 0; b < C; ++b) seed_off[b + 1] += seed_off[b];
    {
        std::vector<int32_t> &cur = c->h_lab; // scratch: write cursor per bin
        cur.assign(seed_off, seed_off + C);
        for (int64_t s = 0; s < ns; ++s) seed_idx[cur[(size_t)lab[seed_tmp[s]]]++] = seed_tmp[s];
    }
    if (slot_end < 0) slot_end = U;
    CHB_CHECK(c, 0 <= slot_begin && slot_begin <= slot_end && slot_end <= U, CHB_EINVAL, "owned slot range [%lld,%lld) invalid for U=%lld",
              (long long)slot_begin, (long long)slot_end, (long long)U);
    c->C = C;
    c->U = U;
    c->u0 = slot_begin;
    c->u1 = slot_end;
    c->wide_fused_size_ok = U * n >= wide_fused_min_pairs(); // the stage's pair count: the same on every rank
    if (c->cap_n < n) {
        CHB_TRY(dev_alloc(c, &c->old_label, n));
        CHB_TRY(dev_alloc(c, &c->tent_pt, n));
        CHB_TRY(dev_alloc(c, &c->pos, n));
        CHB_TRY(dev_alloc(c, &c->qslot, n));
        CHB_TRY(dev_alloc(c, &c->packed, n + 4));
        c->cap_n = n;
    }
    if (c->cap_U < std::max<int64_t>(U, 1)) {
        CHB_TRY(dev_alloc(c, &c->qpoint, std::max<int64_t>(U, 1)));
        CHB_TRY(dev_alloc(c, &c->perm_pt, std::max<int64_t>(U, 1)));
        c->cap_U = std::max<int64_t>(U, 1);
    }
    if (c->cap_own < std::max<int64_t>(slot_end - slot_begin, 1)) {
        CHB_TRY(dev_alloc(c, &c->own_pos, std::max<int64_t>(slot_end - slot_begin, 1)));
        delete[] c->own_pos_host;
        c->own_pos_host = new int64_t[(size_t)std::max<int64_t>(slot_end - slot_begin, 1)];
        c->cap_own = std::max<int64_t>(slot_end - slot_begin, 1);
    }
    CHB_TRY(dev_reserve(c, &c->seed_off, &c->cap_seed_off, (int64_t)C + 1));
    CHB_TRY(dev_reserve(c, &c->seed_idx, &c->cap_seed_idx, std::max<int64_t>(n - U, 1)));
    CHB_CUDA(c, cudaMemcpyAsync(c->seed_off, seed_off, sizeof(int32_t) * ((size_t)C + 1), cudaMemcpyHostToDevice, c->stream));
    if (n - U > 0)
        CHB_CUDA(c, cudaMemcpyAsync(c->seed_idx, seed_idx, sizeof(int32_t) * (size_t)(n - U), cudaMemcpyHostToDevice, c->stream));
    CHB_CUDA(c, cudaMemcpyAsync(c->old_label, lab, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CHB_CUDA(c, cudaMemcpyAsync(c->tent_pt, c->old_label, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToDevice, c->stream));
    {
        const int32_t ntiles = (int32_t)((n + SLOT_TILE - 1) / SLOT_TILE);
        CHB_TRY(dev_reserve(c, &c->slot_tiles, &c->cap_slot_tiles, (int64_t)ntiles));
        CHB_PDL_LAUNCH(c, slots_count_kernel, (unsigned)ntiles, 256, 0, c->old_label, n, c->slot_tiles);
        CHB_PDL_LAUNCH(c, slots_tile_scan_kernel, 1, 256, 0, c->slot_tiles, ntiles);
        CHB_PDL_LAUNCH(c, slots_fill_kernel, (unsigned)ntiles, 256, 0, c->old_label, n, c->slot_tiles, c->qslot, c->qpoint, c->pos);
        CHB_CUDA(c, cudaGetLastError());
        c->tm.launches_other += 3;
    }
    c->labels_set = true;
    c->guess_pending = true;
    c->guess_shared = false; // the caller opts in again with chb_guess_export after every chb_set_labels
    c->guess_imported = false;
    c->in_iteration = false;
    c->dist_ready = false;
    c->f_asplit_ready = false;
    c->cache_nown = -1; // force cache re-initialisation
    return CHB_OK;
}

int chb_set_params(chb_ctx *c, int32_t k, int32_t metric)
{
    CHB_CHECK(c, c, CHB_EINVAL, "ctx is NULL");
    CHB_CHECK(c, k >= 1 && k <= CHB_KMAX, CHB_EINVAL, "num_neighbors must be in [1, %d], got %d", CHB_KMAX, k);
    CHB_CHECK(c, metric == CHB_METRIC_CONVEX || metric == CHB_METRIC_AFFINE_QP || metric == CHB_METRIC_AFFINE, CHB_ENOTIMPL,
              "Metric %d not implemented", metric);
    if (k != c->k || metric != c->metric) c->cache_nown = -1;
    c->k = k;
    c->metric = metric;
    return CHB_OK;
}

int chb_build_distance_matrix(chb_ctx *c, int materialise)
{
    CHB_CHECK(c, c, CHB_EINVAL, "ctx is NULL");
    CHB_CHECK(c, c->labels_set, CHB_EINVAL, "build_distance_matrix: call chb_set_features and chb_set_labels first");
    CHB_CUDA(c, cudaSetDevice(c->device));
    if (c->nmax_pending) CHB_TRY(sync_stream(c)); // chb_set_features_async: the upload ends here at the latest
    const int64_t nown = c->u1 - c->u0;
    c->materialise = materialise != 0;
    const bool filt = use_filter(c);
    c->lda = (c->n + 3) & ~int64_t(3);
    const int64_t step = 65535LL * 64;
    // scratch for recomputed rows: ~1 GiB, at least 64 rows
    int64_t srows = (1LL << 30) / ((filt ? 4 : 8) * c->n);
    srows = std::max<int64_t>(64, std::min<int64_t>(srows, std::max<int64_t>(nown, 64)));
    if (use_fused(c)) {
        // nothing is materialised: distances are regenerated on the tensor cores every round (fused.cu); a small
        // scratch serves the rare exact-path fallback
        dev_free(&c->Dq); c->cap_Dq = 0;
        dev_free(&c->Dscratch); c->cap_scratch = 0;
        dev_free(&c->Aq); c->cap_Aq = 0;
        srows = std::min<int64_t>(srows, 256);
        CHB_TRY(dev_reserve(c, &c->Ascratch, &c->cap_Ascratch, srows * c->lda));
        c->scratch_rows = srows;
        c->materialise = false;
        c->dist_ready = true; // nothing was enqueued: no synchronisation either (the label set-up keeps running underneath)
        return CHB_OK;
    } else if (filt) {
        dev_free(&c->Dq); c->cap_Dq = 0;
        dev_free(&c->Dscratch); c->cap_scratch = 0;
        if (c->materialise) {
            dev_free(&c->Ascratch); c->cap_Ascratch = 0;
            CHB_TRY(dev_reserve(c, &c->Aq, &c->cap_Aq, nown * c->lda));
            for (int64_t r0 = 0; r0 < nown; r0 += step)
                CHB_TRY(candidate_rows(c, c->qpoint + c->u0 + r0, std::min(step, nown - r0), c->Aq + r0 * c->lda, c->lda));
        } else {
            dev_free(&c->Aq); c->cap_Aq = 0;
            CHB_TRY(dev_reserve(c, &c->Ascratch, &c->cap_Ascratch, srows * c->lda));
            c->scratch_rows = srows;
        }
    } else {
        dev_free(&c->Aq); c->cap_Aq = 0;
        dev_free(&c->Ascratch); c->cap_Ascratch = 0;
        if (c->materialise) {
            dev_free(&c->Dscratch); c->cap_scratch = 0;
            CHB_TRY(dev_reserve(c, &c->Dq, &c->cap_Dq, nown * c->n));
            for (int64_t r0 = 0; r0 < nown; r0 += step)
                CHB_TRY(chb_launch_distance_rows(c, c->qpoint + c->u0 + r0, std::min(step, nown - r0), c->Dq + r0 * c->n));
        } else {
            dev_free(&c->Dq); c->cap_Dq = 0;
            CHB_TRY(dev_reserve(c, &c->Dscratch, &c->cap_scratch, srows * c->n));
            c->scratch_rows = srows;
        }
    }
    CHB_TRY(sync_stream(c));
    c->dist_ready = true;
    return CHB_OK;
}

int chb_get_distance_rows(chb_ctx *c, int64_t slot0, int64_t nrows, double *out)
{
    CHB_CHECK(c, c && out, CHB_EINVAL, "NULL argument");
    CHB_CHECK(c, c->dist_ready, CHB_EINVAL, "distance matrix not built");
    CHB_CHECK(c, slot0 >= c->u0 && nrows >= 0 && slot0 + nrows <= c->u1, CHB_EINVAL, "slots [%lld,%lld) not owned",
              (long long)slot0, (long long)(slot0 + nrows));
    CHB_CUDA(c, cudaSetDevice(c->device));
    if (c->materialise && !use_filter(c)) {
        CHB_CUDA(c, cudaMemcpyAsync(out, c->Dq + (slot0 - c->u0) * c->n, sizeof(double) * (size_t)nrows * c->n,
                                    cudaMemcpyDeviceToHost, c->stream));
        return sync_stream(c);
    }
    // exact rows are not stored in this mode: recompute them (same kernel, same recipe) through a temporary
    const int64_t chunk = std::max<int64_t>(1, std::min<int64_t>(std::max<int64_t>(nrows, 1), (1LL << 28) / (8 * c->n) + 1));
    double *tmp = nullptr;
    CHB_TRY(dev_alloc(c, &tmp, chunk * c->n));
    int rc = CHB_OK;
    for (int64_t r0 = 0; r0 < nrows && rc == CHB_OK; r0 += chunk) {
        const int64_t cnt = std::min(chunk, nrows - r0);
        if ((rc = chb_launch_distance_rows(c, c->qpoint + slot0 + r0, cnt, tmp))) break;
        cudaMemcpyAsync(out + r0 * c->n, tmp, sizeof(double) * (size_t)cnt * c->n, cudaMemcpyDeviceToHost, c->stream);
        rc = sync_stream(c);
    }
    dev_free(&tmp);
    return rc;
}

// ---------------------------------------------------------------------------------------------------------
int chb_knn_per_bin(chb_ctx *c, const int64_t *labels, const int64_t *queries, int64_t nq, int64_t *idx_out, int32_t *m_out)
{
    CHB_CHECK(c, c && labels && queries && idx_out && m_out, CHB_EINVAL, "NULL argument");
    CHB_CHECK(c, c->X && c->C > 0, CHB_EINVAL, "knn_per_bin: set features and labels first");
    CHB_CUDA(c, cudaSetDevice(c->device));
    if (c->nmax_pending) CHB_TRY(sync_stream(c));
    const int64_t n = c->n;
    const int32_t C = c->C, k = c->k;
    std::vector<int32_t> lab((size_t)n);
    for (int64_t i = 0; i < n; ++i) lab[(size_t)i] = (int32_t)labels[i];
    const int64_t chunk = std::max<int64_t>(1, std::min<int64_t>(nq, std::max<int64_t>(1, (1LL << 29) / (8 * n))));
    int32_t *d_lab = nullptr, *d_q = nullptr, *d_idx = nullptr, *d_cnt = nullptr;
    double *d_rows = nullptr;
    float *d_arows = nullptr;
    const bool filt = use_filter(c);
    int rc = CHB_OK;
    std::vector<int32_t> q32((size_t)chunk), idx32((size_t)chunk * C * k);
    do {
        if ((rc = dev_alloc(c, &d_lab, n)) || (rc = dev_alloc(c, &d_q, chunk)) || (rc = dev_alloc(c, &d_idx, chunk * C * k)) ||
            (rc = dev_alloc(c, &d_cnt, chunk * C)))
            break;
        const int64_t lda = (n + 3) & ~int64_t(3);
        if (filt ? (rc = dev_alloc(c, &d_arows, chunk * lda)) : (rc = dev_alloc(c, &d_rows, chunk * n))) break;
        cudaMemcpyAsync(d_lab, lab.data(), sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, c->stream);
        for (int64_t q0 = 0; q0 < nq && rc == CHB_OK; q0 += chunk) {
            const int64_t cnt = std::min(chunk, nq - q0);
            for (int64_t i = 0; i < cnt; ++i) {
                const int64_t q = queries[q0 + i];
                if (q < 0 || q >= n) { rc = chb_fail(c, CHB_EINVAL, "query index %lld out of range", (long long)q); break; }
                q32[(size_t)i] = (int32_t)q;
            }
            if (rc) break;
            cudaMemcpyAsync(d_q, q32.data(), sizeof(int32_t) * (size_t)cnt, cudaMemcpyHostToDevice, c->stream);
            if ((rc = filt ? candidate_rows(c, d_q, cnt, d_arows, lda) : chb_launch_distance_rows(c, d_q, cnt, d_rows))) break;
            chb_knn_args a{};
            fill_filter_args(c, a, filt);
            a.arows = d_arows;
            a.rows = d_rows; a.row_stride = filt ? lda : n; a.row_is_item = 1; a.items = d_q; a.n_items = cnt; a.mode = 1;
            a.old_label = d_lab; a.n = n; a.C = C; a.k = k; a.u0 = 0; a.knn_idx = d_idx; a.knn_cnt = d_cnt;
            if ((rc = chb_launch_knn_scan(c, a))) break;
            cudaMemcpyAsync(idx32.data(), d_idx, sizeof(int32_t) * (size_t)cnt * C * k, cudaMemcpyDeviceToHost, c->stream);
            cudaMemcpyAsync(m_out + q0 * C, d_cnt, sizeof(int32_t) * (size_t)cnt * C, cudaMemcpyDeviceToHost, c->stream);
            if ((rc = sync_stream(c))) break;
            for (int64_t i = 0; i < cnt * C * k; ++i) idx_out[q0 * C * k + i] = idx32[(size_t)i];
        }
    } while (0);
    dev_free(&d_lab); dev_free(&d_q); dev_free(&d_idx); dev_free(&d_cnt); dev_free(&d_rows); dev_free(&d_arows);
    return rc;
}

int chb_hull_distance_batch(chb_ctx *c, const int64_t *queries, int64_t nq, const int64_t *idx, const int32_t *m,
                            double *dist_out, int32_t *status_out, double *alpha_out)
{
    CHB_CHECK(c, c && queries && idx && m && dist_out, CHB_EINVAL, "NULL argument");
    CHB_CHECK(c, c->X && c->C > 0, CHB_EINVAL, "hull_distance_batch: set features and labels first");
    CHB_CUDA(c, cudaSetDevice(c->device));
    if (c->nmax_pending) CHB_TRY(sync_stream(c));
    const int32_t C = c->C, k = c->k;
    const int64_t np = nq * C;
    if (np == 0) return CHB_OK;
    std::vector<int32_t> q32((size_t)nq), idx32((size_t)np * k);
    std::vector<int2> work((size_t)np);
    for (int64_t i = 0; i < nq; ++i) {
        CHB_CHECK(c, queries[i] >= 0 && queries[i] < c->n, CHB_EINVAL, "query index out of range");
        q32[(size_t)i] = (int32_t)queries[i];
    }
    for (int64_t i = 0; i < np; ++i) {
        CHB_CHECK(c, m[i] >= 0 && m[i] <= k, CHB_EINVAL, "m[%lld] = %d outside [0, k=%d]", (long long)i, m[i], k);
        for (int32_t s = 0; s < k; ++s) {
            const int64_t v = idx[i * k + s];
            CHB_CHECK(c, s >= m[i] || (v >= 0 && v < c->n), CHB_EINVAL, "neighbour index out of range");
            idx32[(size_t)(i * k + s)] = (int32_t)v;
        }
        work[(size_t)i] = make_int2((int)(i / C), (int)(i % C));
    }
    int32_t *d_q = nullptr, *d_idx = nullptr, *d_m = nullptr, *d_st = nullptr;
    int2 *d_work = nullptr;
    double *d_dist = nullptr, *d_alpha = nullptr;
    int rc = CHB_OK;
    do {
        if ((rc = dev_alloc(c, &d_q, nq)) || (rc = dev_alloc(c, &d_idx, np * k)) || (rc = dev_alloc(c, &d_m, np)) ||
            (rc = dev_alloc(c, &d_st, np)) || (rc = dev_alloc(c, &d_work, np)) || (rc = dev_alloc(c, &d_dist, np)))
            break;
        if (alpha_out && (rc = dev_alloc(c, &d_alpha, np * k))) break;
        cudaMemcpyAsync(d_q, q32.data(), sizeof(int32_t) * (size_t)nq, cudaMemcpyHostToDevice, c->stream);
        cudaMemcpyAsync(d_idx, idx32.data(), sizeof(int32_t) * (size_t)np * k, cudaMemcpyHostToDevice, c->stream);
        cudaMemcpyAsync(d_m, m, sizeof(int32_t) * (size_t)np, cudaMemcpyHostToDevice, c->stream);
        cudaMemcpyAsync(d_work, work.data(), sizeof(int2) * (size_t)np, cudaMemcpyHostToDevice, c->stream);
        chb_qp_args a{};
        a.X = c->X; a.ldx = c->ldx; a.d = c->d; a.work = d_work; a.work_count = nullptr; a.n_work = np; a.row_point = d_q;
        a.knn_idx = d_idx; a.knn_cnt = d_m; a.C = C; a.k = k; a.metric = c->metric; a.dist = d_dist; a.status = d_st;
        a.alpha = d_alpha;
        if ((rc = chb_launch_qp(c, a))) break;
        c->tm.qps_solved += np;
        cudaMemcpyAsync(dist_out, d_dist, sizeof(double) * (size_t)np, cudaMemcpyDeviceToHost, c->stream);
        if (status_out) cudaMemcpyAsync(status_out, d_st, sizeof(int32_t) * (size_t)np, cudaMemcpyDeviceToHost, c->stream);
        if (alpha_out) cudaMemcpyAsync(alpha_out, d_alpha, sizeof(double) * (size_t)np * k, cudaMemcpyDeviceToHost, c->stream);
        rc = sync_stream(c);
    } while (0);
    dev_free(&d_q); dev_free(&d_idx); dev_free(&d_m); dev_free(&d_st); dev_free(&d_work); dev_free(&d_dist); dev_free(&d_alpha);
    return rc;
}

// ---------------------------------------------------------------------------------------------------------
int chb_set_window(chb_ctx *c, int64_t window)
{
    CHB_CHECK(c, c && window >= 0, CHB_EINVAL, "bad window");
    c->window = window;
    return CHB_OK;
}
int64_t chb_get_window(chb_ctx *c) { return c ? (c->window > 0 ? c->window : c->U) : 0; }

static int iteration_begin_common(chb_ctx *c, const int64_t *perm, int64_t U, bool perm_on_device);

int chb_iteration_begin(chb_ctx *c, const int64_t *perm, int64_t U) { return iteration_begin_common(c, perm, U, false); }

// The NEXT iteration's permutation, uploaded on the side stream while the current iteration's rounds run: a stage at 20k
// contigs spends ~20 us per iteration staging 140 KB of pageable host memory with the device idle (the upload sits right
// after the commit's synchronisation).  Used by the next chb_iteration_begin iff it is called with the same `perm`.
int chb_iteration_prefetch(chb_ctx *c, const int64_t *perm, int64_t U)
{
    CHB_CHECK(c, c && (perm || U == 0), CHB_EINVAL, "NULL argument");
    CHB_CHECK(c, c->labels_set && U == c->U, CHB_EINVAL, "permutation length %lld != number of points to assign %lld", (long long)U,
              (long long)c->U);
    c->perm_prefetch_src = nullptr;
    if (U == 0 || !use_fused(c)) return CHB_OK; // the host path of chb_iteration_begin reads the permutation on the host
    CHB_CUDA(c, cudaSetDevice(c->device));
    CHB_TRY(dev_reserve(c, &c->perm64_next, &c->cap_perm64_next, U));
    CHB_CUDA(c, cudaMemcpyAsync(c->perm64_next, perm, sizeof(int64_t) * (size_t)U, cudaMemcpyHostToDevice, c->side_stream));
    CHB_CUDA(c, cudaEventRecord(c->ev_perm, c->side_stream));
    c->perm_prefetch_src = perm;
    return CHB_OK;
}

int chb_iteration_begin_dev(chb_ctx *c, const int64_t *perm_dev, int64_t U)
{
    CHB_CHECK(c, c, CHB_EINVAL, "ctx is NULL");
    CHB_CHECK(c, use_fused(c) || U == 0, CHB_EINVAL, "chb_iteration_begin_dev needs the fused path of distance mode 2 (chb_get_distance_path); pass a host permutation otherwise");
    return iteration_begin_common(c, perm_dev, U, true);
}

static int iteration_begin_common(chb_ctx *c, const int64_t *perm, int64_t U, bool perm_on_device)
{
    CHB_CHECK(c, c && (perm || U == 0), CHB_EINVAL, "NULL argument");
    CHB_CHECK(c, c->labels_set && c->dist_ready, CHB_EINVAL, "iteration_begin: labels / distance matrix not set up");
    CHB_CHECK(c, U == c->U, CHB_EINVAL, "permutation length %lld != number of points to assign %lld", (long long)U,
              (long long)c->U);
    CHB_CUDA(c, cudaSetDevice(c->device));
    CHB_TRY(ensure_caches(c));
    c->own_pos_by_slot = false;
    c->labels_staged = false;
    if (use_fused(c) && U > 0) {
        // Device path (distance mode 2): the permutation is uploaded as it is and turned into perm_pt / pos / own_pos by
        // one kernel; its validation travels with the next commit's read-back (no host pass over U, no host mirror).
        const int64_t *src64 = nullptr;
        if (!perm_on_device && c->perm_prefetch_src && c->perm_prefetch_src == perm && c->cap_perm64_next >= U) {
            // uploaded ahead on the side stream while the previous iteration ran (chb_iteration_prefetch): the buffers swap roles
            std::swap(c->perm64, c->perm64_next);
            std::swap(c->cap_perm64, c->cap_perm64_next);
            CHB_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_perm, 0));
            src64 = c->perm64;
        } else {
            CHB_TRY(dev_reserve(c, &c->perm64, &c->cap_perm64, U));
            CHB_CUDA(c, cudaMemcpyAsync(c->perm64, perm, sizeof(int64_t) * (size_t)U,
                                        perm_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, c->stream));
            src64 = c->perm64;
        }
        c->perm_prefetch_src = nullptr;
        CHB_CUDA(c, cudaMemsetAsync(&c->counters[9], 0x7f, 3 * sizeof(int32_t), c->stream));
        CHB_PDL_LAUNCH(c, begin_perm_kernel, nblk(std::max<int64_t>(U, c->n), 256), 256, 0, src64, U, c->n, c->qslot, c->qpoint, c->u0, c->u1,
                       c->perm_pt, c->pos, c->own_pos, c->counters, c->old_label, c->tent_pt);
        CHB_PDL_LAUNCH(c, check_perm_kernel, nblk(U, 256), 256, 0, c->perm_pt, U, c->pos, c->counters);
        CHB_CUDA(c, cudaGetLastError());
        c->tm.launches_other += 2;
        c->n_own_pos = c->u1 - c->u0;
        c->own_pos_by_slot = true;
        c->perm_check_pending = true;
    } else {
    if (!c->h_qslot_valid) { // host mirror of the query slots (the device derives its own copy in chb_set_labels)
        int32_t *lab = c->pin_i32, *qs = lab + c->n;
        int32_t u = 0;
        for (int64_t i = 0; i < c->n; ++i) qs[i] = (lab[i] == -1) ? u++ : -1;
        c->h_qslot_valid = true;
    }
    // positions this context owns, ascending (a context owns the queries of slots [u0, u1)); host mirrors of
    // qslot / the permutation scratch are kept in the context so that nothing is allocated or read back per iteration
    std::vector<int32_t> &p32 = c->h_perm32;
    std::vector<int32_t> &own32 = c->h_own32;
    p32.resize((size_t)std::max<int64_t>(U, 1));
    own32.clear();
    {
        std::vector<uint8_t> &seen = c->h_seen;
        seen.assign((size_t)std::max<int64_t>(U, 1), 0);
        int64_t cnt = 0;
        for (int64_t p = 0; p < U; ++p) {
            const int64_t pt = perm[p];
            CHB_CHECK(c, pt >= 0 && pt < c->n, CHB_EINVAL, "permutation entry %lld out of range", (long long)pt);
            const int64_t slot = c->h_qslot[pt];
            CHB_CHECK(c, slot >= 0, CHB_EINVAL, "permutation entry %lld is not an un-assigned point", (long long)pt);
            CHB_CHECK(c, !seen[(size_t)slot], CHB_EINVAL, "permutation repeats point %lld", (long long)pt);
            seen[(size_t)slot] = 1;
            p32[(size_t)p] = (int32_t)pt;
            if (slot >= c->u0 && slot < c->u1) {
                own32.push_back((int32_t)p);
                c->own_pos_host[cnt++] = p;
            }
        }
        c->n_own_pos = cnt;
    }
    if (U) {
        CHB_CUDA(c, cudaMemcpyAsync(c->perm_pt, p32.data(), sizeof(int32_t) * (size_t)U, cudaMemcpyHostToDevice, c->stream));
        if (!own32.empty())
            CHB_CUDA(c, cudaMemcpyAsync(c->own_pos, own32.data(), sizeof(int32_t) * own32.size(), cudaMemcpyHostToDevice, c->stream));
        set_pos_kernel<<<nblk(U, 256), 256, 0, c->stream>>>(c->perm_pt, U, c->pos);
        CHB_CUDA(c, cudaGetLastError());
        ++c->tm.launches_other;
    }
    }
    if (!c->own_pos_by_slot) // (the device path's begin_perm_kernel has done this copy)
        CHB_CUDA(c, cudaMemcpyAsync(c->tent_pt, c->old_label, sizeof(int32_t) * (size_t)c->n, cudaMemcpyDeviceToDevice, c->stream));
    if (c->guess_pending && use_fused(c) && U > 0) {
        // First iteration: every query still carries -1.  Any starting vector T0 leads the speculate/repair rounds to
        // the same fixed point (position p is final once positions < p are, whatever it started from), so start from
        // the bin of the nearest seed centroid instead of "unassigned": when that guess is right the first round already
        // reproduces itself and the seed-only round (a full batch of QPs that the second round re-solves) is saved.
        CHB_CHECK(c, !c->guess_shared || c->guess_imported, CHB_EINVAL,
                  "iteration_begin: chb_guess_export was called without chb_guess_import (the other ranks' guesses are missing)");
        CHB_TRY(chb_fused_setup(c));
        CHB_TRY(chb_fused_guess(c));
    }
    c->guess_pending = false;
    // no sync: the host arrays are context-owned and pageable (the runtime stages them before returning)
    c->in_iteration = true;
    c->tm.qps_reference += (c->u1 - c->u0) * c->C;
    return CHB_OK;
}

// tent_dev == NULL: the context's own tentative buffer (single-context use: nothing to exchange between the two calls)
static int own_tent(chb_ctx *c, int64_t len, int32_t **out)
{
    if (c->tent_win_cap < len) {
        CHB_TRY(dev_alloc(c, &c->tent_win, len));
        c->tent_win_cap = len;
    }
    *out = c->tent_win;
    return CHB_OK;
}

int chb_round_run(chb_ctx *c, int64_t lo, int64_t hi, int32_t *tent_dev)
{
    CHB_CHECK(c, c, CHB_EINVAL, "ctx is NULL");
    CHB_CHECK(c, c->in_iteration, CHB_EINVAL, "round_run outside chb_iteration_begin/end");
    CHB_CHECK(c, 0 <= lo && lo < hi && hi <= c->U, CHB_EINVAL, "round window [%lld,%lld) invalid", (long long)lo, (long long)hi);
    CHB_CUDA(c, cudaSetDevice(c->device));
    if (!tent_dev) CHB_TRY(own_tent(c, hi - lo, &tent_dev));
    int64_t b = 0, cnt = c->n_own_pos; // device path: every owned position, the kernels skip those outside [lo, hi)
    if (!c->own_pos_by_slot) {
        const int64_t *ob = c->own_pos_host, *oe = c->own_pos_host + c->n_own_pos;
        b = std::lower_bound(ob, oe, lo) - ob;
        cnt = (std::lower_bound(ob, oe, hi) - ob) - b;
    }
    if (c->n_own_pos < c->U) { // positions of other ranks' queries stay CHB_UNOWNED; a context that owns them all skips the fill
        CHB_PDL_LAUNCH(c, fill_i32_kernel, nblk(hi - lo, 256), 256, 0, tent_dev, hi - lo, CHB_UNOWNED);
        CHB_CUDA(c, cudaGetLastError());
        ++c->tm.launches_other;
    }
    ++c->tm.rounds;
    if (cnt == 0) return CHB_OK;
    if (use_filter(c) && !use_fused(c) && c->C < 32768) {
        pack_labels_kernel<<<nblk(c->n, 256), 256, 0, c->stream>>>(c->pos, c->tent_pt, c->old_label, c->n, c->packed);
        CHB_CUDA(c, cudaGetLastError());
        ++c->tm.launches_other;
    }
    const bool filt = use_filter(c);
    if (use_fused(c)) {
        const int64_t nown = c->u1 - c->u0;
        CHB_TRY(ensure_work(c, nown)); // a pair is listed at most once per round (re-rank or exact redo)
        CHB_TRY(chb_round_fused(c)); // resets the work counter itself (round_reset_kernel)
        // pairs whose kept lists were incomplete were redone exactly inside chb_round_fused (no host round trip); the work /
        // tile / redo / cap counters all travel with the commit's ONE 64-byte read-back (commit_common) -- copy nodes between
        // the kernels would also break the programmatic launch chain
        chb_qp_args q{};
        q.X = c->X; q.ldx = c->ldx; q.d = c->d; q.work = c->work; q.work_count = c->counters; q.n_work = nown * c->C;
        q.row_point = c->qpoint + c->u0; q.knn_idx = c->knn_idx; q.knn_cnt = c->knn_cnt; q.C = c->C; q.k = c->k;
        q.metric = c->metric; q.dist = c->pair_dist; q.status = c->pair_status; q.alpha = nullptr;
        q.cap_count = &c->counters[14];
        CHB_TRY(chb_launch_qp(c, q));
        CHB_TRY(chb_fused_argmin(c, c->own_pos + b, cnt, lo, hi, tent_dev));
        c->round_snapshot_pending = true;
        return CHB_OK;
    }
    CHB_TRY(ensure_work(c, c->materialise ? cnt : std::min(cnt, c->scratch_rows)));
    const int64_t step = c->materialise ? cnt : c->scratch_rows;
    int32_t *rows_tmp = nullptr;
    if (!c->materialise) CHB_TRY(dev_alloc(c, &rows_tmp, step));
    int rc = CHB_OK;
    for (int64_t s0 = 0; s0 < cnt && rc == CHB_OK; s0 += step) {
        const int64_t sc = std::min(step, cnt - s0);
        cudaMemsetAsync(c->counters, 0, sizeof(int32_t), c->stream);
        chb_knn_args a{};
        a.row_stride = filt ? c->lda : c->n; a.items = c->own_pos + b + s0; a.n_items = sc; a.mode = 0; a.perm_pt = c->perm_pt;
        a.qslot = c->qslot; a.pos = c->pos; a.tent_pt = c->tent_pt; a.old_label = c->old_label; a.n = c->n; a.C = c->C;
        a.k = c->k; a.u0 = c->u0; a.knn_idx = c->knn_idx; a.knn_cnt = c->knn_cnt; a.work = c->work;
        a.work_count = c->counters;
        fill_filter_args(c, a, filt);
        a.knn_dist = c->knn_dist;
        a.packed = (filt && c->C < 32768) ? c->packed : nullptr;
        if (c->materialise) {
            a.rows = c->Dq;
            a.arows = c->Aq;
            a.row_is_item = 0;
        } else {
            gather_rows_kernel<<<nblk(sc, 256), 256, 0, c->stream>>>(c->own_pos + b + s0, c->perm_pt, sc, rows_tmp);
            ++c->tm.launches_other;
            if ((rc = filt ? candidate_rows(c, rows_tmp, sc, c->Ascratch, c->lda) : chb_launch_distance_rows(c, rows_tmp, sc, c->Dscratch)))
                break;
            a.rows = c->Dscratch;
            a.arows = c->Ascratch;
            a.row_is_item = 1;
        }
        if ((rc = chb_launch_knn_scan(c, a))) break;
        chb_qp_args q{};
        q.X = c->X; q.ldx = c->ldx; q.d = c->d; q.work = c->work; q.work_count = c->counters; q.n_work = sc * c->C;
        q.row_point = c->qpoint + c->u0; q.knn_idx = c->knn_idx; q.knn_cnt = c->knn_cnt; q.C = c->C; q.k = c->k;
        q.metric = c->metric; q.dist = c->pair_dist; q.status = c->pair_status; q.alpha = nullptr;
        if ((rc = chb_launch_qp(c, q))) break;
        // bookkeeping of solved QPs (read back lazily together with the commit counters)
        cudaMemcpyAsync(&c->counters_host[4], c->counters, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream);
        if (!c->materialise || s0 + step < cnt) {
            if ((rc = sync_stream(c))) break;
            c->tm.qps_solved += c->counters_host[4];
            c->counters_host[4] = 0;
        }
    }
    if (rows_tmp) { cudaStreamSynchronize(c->stream); cudaFree(rows_tmp); }
    if (rc) return rc;
    {
        chb_stage_timer t(c, CHB_ST_COMMIT);
        argmin_kernel<<<nblk(cnt * 32, 256), 256, 0, c->stream>>>(c->own_pos + b, cnt, c->perm_pt, c->qslot, c->u0, c->pair_dist,
                                                                  c->C, c->old_label, lo, tent_dev);
    }
    CHB_CUDA(c, cudaGetLastError());
    return CHB_OK;
}

// chb_iteration_begin's device-side validation of the permutation (the rounds ran on a sanitised copy): the caller has
// copied counters[9..11] to the host and synchronised
static int resolve_perm_check(chb_ctx *c)
{
    if (!c->perm_check_pending) return CHB_OK;
    c->perm_check_pending = false;
    const int32_t none = 0x7f7f7f7f;
    const int32_t bad = std::min(std::min(c->counters_host[9], c->counters_host[10]), c->counters_host[11]);
    if (bad == none) return CHB_OK;
    int64_t pt = -1;
    cudaMemcpy(&pt, c->perm64 + bad, sizeof(int64_t), cudaMemcpyDeviceToHost);
    c->in_iteration = false; // the iteration is abandoned; the next chb_iteration_begin starts from the old labels again
    if (c->counters_host[9] == bad) return chb_fail(c, CHB_EINVAL, "permutation entry %lld out of range", (long long)pt);
    if (c->counters_host[10] == bad) return chb_fail(c, CHB_EINVAL, "permutation entry %lld is not an un-assigned point", (long long)pt);
    return chb_fail(c, CHB_EINVAL, "permutation repeats point %lld", (long long)pt);
}

// Labels widened to the caller's int64 on the device and copied into the page-locked staging block (enqueued only)
constexpr int64_t LABEL_STAGE_MAX = 1 << 18;
static int ensure_label_stage(chb_ctx *c)
{
    CHB_TRY(dev_reserve(c, &c->lab64, &c->cap_lab64, c->n));
    if (c->pin_lab_cap < c->n) {
        CHB_CUDA(c, cudaStreamSynchronize(c->stream));
        if (c->pin_lab64) cudaFreeHost(c->pin_lab64);
        c->pin_lab64 = nullptr;
        c->pin_lab_cap = 0;
        CHB_CUDA(c, cudaMallocHost(reinterpret_cast<void **>(&c->pin_lab64), sizeof(int64_t) * (size_t)c->n));
        c->pin_lab_cap = c->n;
    }
    return CHB_OK;
}
static int stage_labels(chb_ctx *c, const int32_t *lab_dev, bool widened = false) // widened: lab64 is already filled
{
    CHB_TRY(ensure_label_stage(c));
    if (!widened) {
        CHB_PDL_LAUNCH(c, widen_labels_kernel, nblk(c->n, 256), 256, 0, lab_dev, c->n, c->lab64);
        ++c->tm.launches_other;
    }
    CHB_CUDA(c, cudaMemcpyAsync(c->pin_lab64, c->lab64, sizeof(int64_t) * (size_t)c->n, cudaMemcpyDeviceToHost, c->stream));
    return CHB_OK;
}

// Commit of one round; with n_changed != NULL also the end of the iteration when the round changed nothing and its window
// reached the last position -- decided on the device, so that the common "one round settles the iteration" case costs ONE
// host synchronisation instead of two.
static int commit_common(chb_ctx *c, int64_t lo, int64_t hi, const int32_t *tent_dev, int64_t *first_changed, int64_t *n_changed,
                         int32_t *iteration_done)
{
    CHB_CHECK(c, c && first_changed, CHB_EINVAL, "NULL argument");
    CHB_CHECK(c, c->in_iteration, CHB_EINVAL, "round_commit outside chb_iteration_begin/end");
    CHB_CHECK(c, 0 <= lo && lo < hi && hi <= c->U, CHB_EINVAL, "round window [%lld,%lld) invalid", (long long)lo, (long long)hi);
    CHB_CUDA(c, cudaSetDevice(c->device));
    if (!tent_dev) {
        CHB_CHECK(c, c->tent_win && c->tent_win_cap >= hi - lo, CHB_EINVAL, "round_commit(NULL) without a preceding round_run(NULL)");
        tent_dev = c->tent_win;
    }
    const bool may_end = n_changed != nullptr && hi == c->U;
    if (c->round_counters_reset) {
        c->round_counters_reset = false; // this round's round_reset_kernel left counters[1] = "none" and counters[2] = 0
    } else {
        CHB_CUDA(c, cudaMemsetAsync(&c->counters[1], 0x7f, sizeof(int32_t), c->stream)); // 0x7f7f7f7f: above any position
        if (may_end) CHB_CUDA(c, cudaMemsetAsync(&c->counters[2], 0, sizeof(int32_t), c->stream));
    }
    // if this commit ends the iteration the caller may well ask for the labels next: they are widened by end_if_done_kernel
    // itself and travel with the counters (if the iteration goes on the copy is simply not used)
    const bool stage = may_end && c->n <= LABEL_STAGE_MAX;
    if (stage) CHB_TRY(ensure_label_stage(c));
    {
        chb_stage_timer t(c, CHB_ST_COMMIT);
        CHB_PDL_LAUNCH(c, commit_kernel, nblk(hi - lo, 256), 256, 0, tent_dev, lo, hi, c->perm_pt, c->tent_pt, c->counters,
                                                                  (use_fused(c) && c->u1 - c->u0 == c->U) ? c->f_fb_cap : 0);
    }
    bool staged = false;
    if (may_end) {
        CHB_PDL_LAUNCH(c, end_if_done_kernel, nblk(c->n, 256), 256, 0, c->old_label, c->tent_pt, c->n, c->counters,
                       stage ? c->lab64 : nullptr);
        ++c->tm.launches_other;
        if (stage) {
            CHB_TRY(stage_labels(c, c->old_label, true));
            staged = true;
        }
    }
    if (c->round_snapshot_pending) {
        // fused path: every counter of the round in one 64-byte read-back (round_run enqueued none)
        c->round_snapshot_pending = false;
        int32_t *snap = c->counters_host + 16;
        CHB_CUDA(c, cudaMemcpyAsync(snap, c->counters, 16 * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
        CHB_TRY(sync_stream(c));
        int32_t *h = c->counters_host;
        h[1] = snap[1]; h[2] = snap[2];
        h[4] = snap[0];   // QPs solved this round (work-list length)
        for (int i = 6; i <= 12; ++i) h[i] = snap[i]; // exact-redo pairs, planned / issued tiles, permutation checks, refusal flag
        h[14] = snap[14]; // QPs that stopped on the iteration cap
    } else {
        CHB_CUDA(c, cudaMemcpyAsync(&c->counters_host[1], &c->counters[1], 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
        if (c->perm_check_pending)
            CHB_CUDA(c, cudaMemcpyAsync(&c->counters_host[9], &c->counters[9], 3 * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
        CHB_TRY(sync_stream(c));
    }
    c->tm.qps_solved += c->counters_host[4];
    c->counters_host[4] = 0;
    c->tm.qp_iter_cap += c->counters_host[14];
    c->counters_host[14] = 0;
    c->tm.gram_tiles_planned += c->counters_host[7]; // tiles left after bin pruning (pairs_plan_kernel), this round
    c->tm.gram_tiles += c->counters_host[8];         // tiles the MMA warps of gram_select_kernel actually issued
    c->counters_host[7] = c->counters_host[8] = 0;
    CHB_TRY(resolve_perm_check(c));
    if (c->counters_host[12]) {
        c->counters_host[12] = 0;
        c->in_iteration = false;
        return chb_fail(c, CHB_ENOMEM, "the pruning bounds left more (query, bin) pairs than the compact buffers hold and the per-pair candidate "
                                       "table (%lld x %d pairs) is beyond CHB_DENSE_LIST_GB: raise it or use distance mode 1",
                        (long long)(c->u1 - c->u0), c->C);
    }
    if (use_fused(c) && c->f_fb_cap > 0 && c->counters_host[6] > c->f_fb_cap) {
        const int32_t wanted = c->counters_host[6];
        c->counters_host[6] = 0;
        // a sharded context cannot take the round back on its own (its tentative labels are already merged with the other
        // ranks'): the fit fails there; a context that owns every slot committed nothing (commit_kernel saw the same
        // counter), grows the list to its worst case -- every (row, bin) pair -- and asks for the window again
        if (c->u1 - c->u0 != c->U)
            return chb_fail(c, CHB_ECUDA, "exact-redo list overflow: %d pairs, capacity %d", wanted, c->f_fb_cap);
        CHB_TRY(chb_fused_grow_redo_list(c));
        *first_changed = CHB_ROUND_AGAIN;
        if (iteration_done) *iteration_done = 0;
        return CHB_OK;
    }
    c->counters_host[6] = 0;
    *first_changed = (c->counters_host[1] == 0x7f7f7f7f) ? -1 : (int64_t)c->counters_host[1];
    if (iteration_done) *iteration_done = 0;
    if (may_end && *first_changed < 0) {
        *n_changed = c->counters_host[2];
        if (iteration_done) *iteration_done = 1;
        c->in_iteration = false;
        c->labels_staged = staged;
    }
    return CHB_OK;
}

int chb_round_commit(chb_ctx *c, int64_t lo, int64_t hi, const int32_t *tent_dev, int64_t *first_changed)
{
    return commit_common(c, lo, hi, tent_dev, first_changed, nullptr, nullptr);
}

int chb_round_commit_end(chb_ctx *c, int64_t lo, int64_t hi, const int32_t *tent_dev, int64_t *first_changed, int64_t *n_changed,
                         int32_t *iteration_done)
{
    CHB_CHECK(c, c && n_changed && iteration_done, CHB_EINVAL, "NULL argument");
    return commit_common(c, lo, hi, tent_dev, first_changed, n_changed, iteration_done);
}

int chb_iteration_end(chb_ctx *c, int64_t *n_changed)
{
    CHB_CHECK(c, c, CHB_EINVAL, "ctx is NULL");
    CHB_CHECK(c, c->in_iteration, CHB_EINVAL, "iteration_end without iteration_begin");
    CHB_CUDA(c, cudaSetDevice(c->device));
    CHB_CUDA(c, cudaMemsetAsync(&c->counters[2], 0, sizeof(int32_t), c->stream));
    count_changed_kernel<<<nblk(c->n, 256), 256, 0, c->stream>>>(c->old_label, c->tent_pt, c->n, c->counters);
    CHB_CUDA(c, cudaGetLastError());
    ++c->tm.launches_other;
    CHB_CUDA(c, cudaMemcpyAsync(&c->counters_host[2], &c->counters[2], sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    if (c->perm_check_pending) {
        CHB_CUDA(c, cudaMemcpyAsync(&c->counters_host[9], &c->counters[9], 3 * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
        CHB_TRY(sync_stream(c));
        CHB_TRY(resolve_perm_check(c)); // an invalid permutation: the labels stay as they were
    }
    CHB_CUDA(c, cudaMemcpyAsync(c->old_label, c->tent_pt, sizeof(int32_t) * (size_t)c->n, cudaMemcpyDeviceToDevice, c->stream));
    CHB_TRY(sync_stream(c));
    if (n_changed) *n_changed = c->counters_host[2];
    c->in_iteration = false;
    return CHB_OK;
}

int chb_get_labels(chb_ctx *c, int64_t *labels_out)
{
    CHB_CHECK(c, c && labels_out, CHB_EINVAL, "NULL argument");
    CHB_CHECK(c, c->labels_set, CHB_EINVAL, "labels not set");
    CHB_CUDA(c, cudaSetDevice(c->device));
    if (!(c->labels_staged && !c->in_iteration)) { // else: they came back with the commit that ended the last iteration
        CHB_TRY(stage_labels(c, c->in_iteration ? c->tent_pt : c->old_label));
        CHB_TRY(sync_stream(c));
    }
    memcpy(labels_out, c->pin_lab64, sizeof(int64_t) * (size_t)c->n);
    return CHB_OK;
}

static int fit_iteration_impl(chb_ctx *c, const int64_t *perm, const int64_t *next_perm, int64_t U, int64_t *labels_out, int64_t *n_changed);

int chb_fit_iteration(chb_ctx *c, const int64_t *perm, int64_t U, int64_t *labels_out, int64_t *n_changed)
{
    return fit_iteration_impl(c, perm, nullptr, U, labels_out, n_changed);
}

// next_perm != NULL: the permutation of the iteration after this one, uploaded ahead while this iteration's first round runs
static int fit_iteration_impl(chb_ctx *c, const int64_t *perm, const int64_t *next_perm, int64_t U, int64_t *labels_out, int64_t *n_changed)
{
    CHB_CHECK(c, c, CHB_EINVAL, "ctx is NULL");
    CHB_CHECK(c, c->u0 == 0 && c->u1 == c->U, CHB_EINVAL,
              "chb_fit_iteration needs a context that owns every query slot; use the chb_round_* calls when sharded");
    CHB_TRY(chb_iteration_begin(c, perm, U));
    const int64_t W = chb_get_window(c);
    if (U > 0) {
        if (c->tent_win_cap < W) {
            CHB_TRY(dev_alloc(c, &c->tent_win, W));
            c->tent_win_cap = W;
        }
        int64_t lo = 0, nch = 0;
        int32_t done = 0;
        while (lo < U) {
            const int64_t hi = std::min(U, lo + W);
            CHB_TRY(chb_round_run(c, lo, hi, c->tent_win));
            if (next_perm) { // after the round is enqueued: the staging copy on the host overlaps the round on the device
                CHB_TRY(chb_iteration_prefetch(c, next_perm, U));
                next_perm = nullptr;
            }
            int64_t first = -1;
            CHB_TRY(chb_round_commit_end(c, lo, hi, c->tent_win, &first, &nch, &done));
            if (first == CHB_ROUND_AGAIN) continue; // the exact-redo list was too small and has grown: same window again
            lo = (first < 0) ? hi : first + 1;
        }
        if (done) {
            if (n_changed) *n_changed = nch;
        } else {
            CHB_TRY(chb_iteration_end(c, n_changed));
        }
    } else {
        CHB_TRY(chb_iteration_end(c, n_changed));
    }
    if (labels_out) CHB_TRY(chb_get_labels(c, labels_out));
    return CHB_OK;
}

int chb_fit(chb_ctx *c, const int64_t *perms, int64_t U, int32_t max_iterations, int64_t *labels_out, int32_t *iterations_run,
            int32_t *converged, int64_t *changed_per_iter)
{
    CHB_CHECK(c, c && (perms || U == 0 || max_iterations == 0), CHB_EINVAL, "NULL argument");
    int32_t it = 0, conv = 0;
    for (; it < max_iterations; ++it) {
        int64_t nch = 0;
        CHB_TRY(fit_iteration_impl(c, perms + (int64_t)it * U, it + 1 < max_iterations ? perms + (int64_t)(it + 1) * U : nullptr, U, nullptr,
                                   &nch));
        if (changed_per_iter) changed_per_iter[it] = nch;
        if (nch == 0) { conv = 1; ++it; break; } // algorithm.py:63-66
    }
    if (iterations_run) *iterations_run = it;
    if (converged) *converged = conv;
    if (labels_out) CHB_TRY(chb_get_labels(c, labels_out));
    return CHB_OK;
}

} // extern "C"
