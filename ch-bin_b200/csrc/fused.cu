// fused.cu -- distance mode 2: tensor-core Gram contraction FUSED with the per-bin neighbour selection (sm_100a).
//
// Replaces, for one speculate/repair round, create_in_mem_distance_matrix + find_nearest_from_cluster
// (/root/reference/ch_bin/core/clustering/distance_matrix.py:33-62) for every (query, bin) pair, without ever
// writing a distance matrix.  Per label set (chb_fused_setup): bin reference points from the seed contigs, the
// U x C centroid terms (FP64 GEMM), the speculation start, per-query upper bounds, the row order (owned slots sorted
// by guessed bin) and the resident TF32 query operand.  Per round (chb_round_fused):
//
//  1. "column entries": every point becomes a column of the bin(s) in which some query can see it this round.
//     The label the query at permutation position p sees for point i is  pos[i] < p ? tent[i] : old[i]
//     (algorithm.py:46-60), so point i is a column of bin tent[i] visible when p > pos[i], and -- if different --
//     of bin old[i] visible when p < pos[i]; when both labels agree it is one column visible when p != pos[i]
//     (which also removes the query itself, algorithm.py:50).  Columns are counting-sorted by bin, each bin padded
//     to a multiple of 128; column_gather_kernel writes the per-bin-centred TF32 [hi | lo] operand rows in that order.
//  2. threshold_kernel: per (row, bin) the pruning test (bin cannot be the argmin: admission threshold -inf, nothing
//     else happens for the pair), else the key error bound E and the admission threshold T0 from the cached set;
//     the same kernel flags the (row block, bin) pairs none of whose rows survived; pairs_plan_kernel (and its tail, items_body) turn
//     the survivors into a balanced work list.
//  3. gram_select_kernel: one persistent CTA per SM walking its work items.  TMA: the row block's query operand is
//     loaded once and stays resident, the column operand streams through a 3-4-stage ring -> tcgen05.mma kind::tf32
//     (3-term hi/lo split, see gram_tc.cu) -> FP32 accumulators double-buffered in TMEM.  Eight decoupled epilogue
//     warps read a tile with one tcgen05.ld per thread (thread = query row x 64-column half), form
//     key = tq + column term - 2 acc, screen by visibility and T0, and keep the KR smallest (key, point) pairs of the
//     item's bin in REGISTERS (candidate stack in shared memory, one drain site, rank-by-counting insertion).
//  4. rerank_kernel, over each row's surviving bins: with |key - d^2| <= E the k smallest keys ARE the reference's
//     neighbours whenever key_(k+1) > key_(k) + 2E; otherwise only the candidates inside the 2E window get scipy's exact
//     recipe (sequential sum, no FMA) and are ranked by exact (distance, index).  A pair goes to the QP work list only
//     if its neighbour SET changed.  Pairs whose kept lists could be incomplete (more than KR keys inside the window:
//     duplicate contigs) are redone exactly on the device by exact_pairs_kernel.
//  5. k > 24 (one of the two 16-entry half-lists would overflow for most pairs): steps 3-4 are replaced by an exact selection over every pair
//     that survived step 2, regrouped per bin so that eight queries share each member row (exact_group_kernel).
//
// Roofline of gram_select_kernel: tensor pipe, co-limited by the CUDA-core selection epilogue (DESIGN.md section 4).
#include <cuda.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>

#include "common.cuh"

namespace {

constexpr int BM = 128, BN = 128, BK = 32;
constexpr int UMMA_K = 8;
constexpr uint32_t TILE_BYTES = BM * BK * 4; // one 128-row x 32-float operand box (128-byte swizzle atom rows)
constexpr int FUSED_THREADS = 320; // warp 0 TMA, warp 1 MMA, warps 2..9 epilogue (two per TMEM lane quadrant)
constexpr int EPI_THREADS = 256;
constexpr uint32_t TMEM_COLS = 256; // two 128-column accumulator buffers
constexpr int MAX_BOX = 10;         // resident query operand: at most 10 boxes = 160 KB  (d <= 160)
constexpr int SMEM_LIMIT = 232448;  // 227 KB opt-in shared memory per CTA
constexpr int DMAX_F = CHB_FUSED_RESIDENT_DMAX; // resident query operand (d <= 160)
constexpr int DMAX_W = 1024;        // streamed query operand (161 <= d <= 1024)
constexpr int NKT_STREAMED = -1;    // gram_select_kernel's NKT for the streamed query operand
constexpr int WIDE_STAGE_BOXES = 4; // streamed ring stage: {query hi, query lo, column hi, column lo} of one 32-feature block

// Operand layout (queries and columns alike), d <= 160: row = [hi(dp8) | lo(dp8) | 0...] floats, dp8 = d rounded up to 8,
// padded to nbox boxes of 32 floats.  hi/lo are the TF32 halves of the centred FP32 feature (gram_tc.cu).  The contraction
// hi.hi + hi.lo + lo.hi is issued as UMMA K=8 steps that pair step i of the RESIDENT query operand with step j of the
// streamed column operand, so the query operand is read from L2 once per row block instead of once per tile.
// d > 160: the query operand of a 128-row block no longer fits shared memory beside a ring.  Each half is padded to whole
// boxes instead, row = [hi(dp32) | lo(dp32)], so that box b holds the hi parts of features 32b .. 32b + 31 and box H + b
// (H = dp32 / 32) their lo parts; a ring stage carries the query AND column boxes of one 32-feature block and feeds
// 4 K-steps x 3 products.  The operand builders take the half width as their `dp8` argument and zero-fill past d.
constexpr int NC = 16; // per-thread candidate stack depth
struct SmemTail {
    // candidates that passed the screen wait here (thread-private stacks, [slot][thread]; their columns are remembered in
    // a per-thread 64-bit mask) until the warp drains them into the register lists: draining costs max-over-lanes
    // insertions, so it pays to drain rarely
    alignas(16) float cand_val[NC][EPI_THREADS];
    alignas(8) uint64_t full_bar[8];
    alignas(8) uint64_t empty_bar[8];
    alignas(8) uint64_t tmem_full_bar[2];
    alignas(8) uint64_t tmem_empty_bar[2];
    alignas(8) uint64_t a_full_bar;
    alignas(8) uint64_t a_empty_bar;
    alignas(8) uint2 prog[MAX_BOX * 8]; // per-tile MMA program: {query-operand descriptor (low word), column step offset}
    int prog_start[MAX_BOX + 1];        // first program entry of each column box
    uint32_t tmem_base;
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void st_shared_f32(uint32_t addr, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory"); }
__device__ __forceinline__ float ld_shared_f32(uint32_t addr)
{
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(void *smem_dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ bool elect_one_sync()
{
    uint32_t pred;
    asm volatile(
        "{\n"
        ".reg .pred P;\n"
        "elect.sync _|P, 0xffffffff;\n"
        "selp.b32 %0, 1, 0, P;\n"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void umma_commit(uint64_t *bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// everything a round starts from zero, in one launch: per-bin column counts, per-bin maxima, per-row survivor counts,
// per-bin pair counters, the work / redo counters, and the compact pair -> row table (-1 = padding)
__global__ void round_reset_kernel(int32_t *__restrict__ bin_cnt, int32_t nbin_cnt, float *__restrict__ ym2, int32_t nym2,
                                   int32_t *__restrict__ row_nb, int64_t nown, int32_t *__restrict__ pair_meta, int32_t nmeta,
                                   int32_t *__restrict__ pair_row, int64_t cap_pairs, int32_t *__restrict__ counters,
                                   int64_t ncol, int32_t *__restrict__ col_pt, int32_t *__restrict__ col_a, int32_t *__restrict__ col_b)
{
    chb_pdl_enter();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < ncol) { // padding columns: no point, never visible
        col_pt[i] = -1;
        col_a[i] = INT32_MAX;
        col_b[i] = INT32_MIN;
    }
    if (i < nbin_cnt) bin_cnt[i] = 0;
    if (i < nym2) ym2[i] = 0.f;
    if (i < nown) row_nb[i] = 0;
    if (i < nmeta) pair_meta[i] = 0;
    if (i < cap_pairs) pair_row[i] = -1;
    if (i == 0) {
        counters[0] = 0; counters[6] = 0; counters[7] = 0; counters[8] = 0; counters[12] = 0; counters[14] = 0;
        // the commit that follows this round (api.cu, commit_common) and the QP launch find their counters ready: first changed
        // position = "none", changed count, QP fallback count -- three memset nodes less on the round's chain
        counters[1] = 0x7f7f7f7f; counters[2] = 0; counters[3] = 0;
    }
}

// ---------------------------------------------------------------------------------------------------------
// column entries
// ---------------------------------------------------------------------------------------------------------
__global__ void entries_count_kernel(const int32_t *__restrict__ tent, const int32_t *__restrict__ old, int64_t n, int32_t C,
                                     int32_t *__restrict__ bin_cnt)
{
    chb_pdl_enter();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int t = tent[i], o = old[i];
    if (t >= 0 && t < C) atomicAdd(&bin_cnt[t], 1);
    if (o >= 0 && o < C && o != t) atomicAdd(&bin_cnt[o], 1);
}

// one block: segment offsets (each bin padded to a multiple of BN), tile -> bin map, cursors reset
__global__ void entries_scan_kernel(const int32_t *__restrict__ bin_cnt, int32_t C, int32_t *__restrict__ seg_off,
                                    int32_t *__restrict__ cursor, int32_t *__restrict__ tile_bin, int32_t *__restrict__ ntiles_out)
{
    chb_pdl_enter();
    if (threadIdx.x == 0) {
        int off = 0;
        for (int c = 0; c < C; ++c) {
            seg_off[c] = off;
            off += (bin_cnt[c] + BN - 1) / BN * BN;
        }
        seg_off[C] = off;
        *ntiles_out = off / BN;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        cursor[c] = 0;
        for (int t = seg_off[c] / BN; t < seg_off[c + 1] / BN; ++t) tile_bin[t] = c;
    }
}

__global__ void entries_scatter_kernel(const int32_t *__restrict__ tent, const int32_t *__restrict__ old,
                                       const int32_t *__restrict__ pos, int64_t n, int32_t C, const int32_t *__restrict__ seg_off,
                                       int32_t *__restrict__ cursor, int32_t *__restrict__ col_pt, int32_t *__restrict__ col_a,
                                       int32_t *__restrict__ col_b)
{
    chb_pdl_enter();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int t = tent[i], o = old[i], ps = pos[i];
    const bool tv = t >= 0 && t < C, ov = o >= 0 && o < C;
    if (tv) {
        const int e = seg_off[t] + atomicAdd(&cursor[t], 1);
        col_pt[e] = (int)i;
        col_a[e] = ps;                      // visible when p > pos[i] ...
        col_b[e] = (ov && o == t) ? ps : INT32_MIN; // ... and also when p < pos[i] if the old label agrees
    }
    if (ov && o != t) {
        const int e = seg_off[o] + atomicAdd(&cursor[o], 1);
        col_pt[e] = (int)i;
        col_a[e] = INT32_MAX;
        col_b[e] = ps;                      // visible only when p < pos[i]
    }
}

// Gathers rows of the centred FP32 features (Xf, prep_f32_kernel) through `idx` and writes them as TF32 operands in the
// [hi(dp8) | lo(dp8) | 0] layout, Kp2 floats per row; idx < 0 (padding columns) gives a zero row.  `count_tiles`
// (device, may be NULL) bounds the rows to *count_tiles * BN; otherwise nrows_max rows are written.
__global__ void split2_gather_kernel(const int32_t *__restrict__ idx, const int32_t *__restrict__ count_tiles, int64_t nrows_max,
                                     const float *__restrict__ Xf, int32_t ldf, int32_t d, int32_t dp8, int32_t Kp2,
                                     const float *__restrict__ nrm, float *__restrict__ out, float *__restrict__ out_nrm)
{
    chb_pdl_enter();
    const int64_t nr = count_tiles ? (int64_t)(*count_tiles) * BN : nrows_max;
    const int64_t kq = Kp2 / 4; // float4 per row
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nr * kq) return;
    const int64_t e = i / kq;
    const int q = (int)(i - e * kq);
    const int ptx = idx[e];
    float o[4] = {0.f, 0.f, 0.f, 0.f};
    if (ptx >= 0) {
        const float *xr = Xf + (int64_t)ptx * ldf;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int t = 4 * q + u;
            const int part = t >= dp8 ? 1 : 0;
            const int f = t - part * dp8;
            if (t < 2 * dp8 && f < d) {
                const float xf = __ldg(xr + f);
                const float hi = __uint_as_float(__float_as_uint(xf) & 0xffffe000u);
                o[u] = part ? __uint_as_float(__float_as_uint(xf - hi) & 0xffffe000u) : hi;
            }
        }
    }
    reinterpret_cast<float4 *>(out + e * Kp2)[q] = make_float4(o[0], o[1], o[2], o[3]);
    if (out_nrm && q == 0) out_nrm[e] = ptx >= 0 ? nrm[ptx] : 0.f;
}

// ---------------------------------------------------------------------------------------------------------
// per-bin centring.  The error of a tensor-core dot product scales with |a| |b|, and with one global centre the
// coverage dimensions keep both operands long (|x - mu| ~ 0.5 against in-bin distances ~ 0.03), so the filter slack
// 2E swallowed tens of bin members at 100k contigs.  Distances are translation invariant per COLUMN: with a fixed
// reference point mu_c per bin (mean of the bin's seed contigs; the global mean if it has none), m_c = mu_c - mu,
// the query operand a_q = fl32(x_q - mu) (unchanged) and the column operand y_i = fl32(x_i - mu_c),
//     |x_q - x_i|^2  ~  |a_q - m_c|^2  +  ( |y_i|^2 + 2 m_c.y_i )  -  2 a_q.y_i
//                        per (q, bin)        per column                  tensor core
// and the contraction error is bounded by eps |a_q| max_i |y_i| -- the column vectors are now in-bin offsets.
// The brackets are evaluated in FP64 from the FP32 operand values actually contracted and rounded once.
// ---------------------------------------------------------------------------------------------------------
// one block per bin: sum of its seed contigs (initial labels) in a FIXED order -- eight interleaved partial sums over the
// (bin, index)-ordered seed list, combined pairwise -- so that every rank gets the same bits; eight independent loads are
// in flight per thread instead of one dependent chain of gathers
__global__ void __launch_bounds__(256) centre_sum_kernel(const double *__restrict__ X, int32_t ldx, int32_t d,
                                                         const int32_t *__restrict__ seed_off, const int32_t *__restrict__ seed_idx,
                                                         double *__restrict__ sum, int32_t *__restrict__ cnt)
{
    chb_pdl_enter();
    const int c = blockIdx.x;
    const int b = seed_off[c], e = seed_off[c + 1];
    for (int t = threadIdx.x; t < d; t += blockDim.x) {
        double s[8] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        int i = b;
        for (; i + 8 <= e; i += 8) {
            double v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = X[(int64_t)seed_idx[i + u] * ldx + t];
#pragma unroll
            for (int u = 0; u < 8; ++u) s[u] += v[u];
        }
        for (int u = 0; i < e; ++i, ++u) s[u] += X[(int64_t)seed_idx[i] * ldx + t];
        sum[(int64_t)c * d + t] = ((s[0] + s[1]) + (s[2] + s[3])) + ((s[4] + s[5]) + (s[6] + s[7]));
    }
    if (threadIdx.x == 0) cnt[c] = e - b;
}

// m_c = mu_c - mu (zero for bins without seeds), mc2[c] = |m_c|^2
__global__ void centre_finish_kernel(double *__restrict__ mc, const int32_t *__restrict__ cnt, const double *__restrict__ colsum,
                                     double inv_n, int32_t d, double *__restrict__ mc2, double *__restrict__ mcT, int32_t Cp)
{
    chb_pdl_enter();
    const int c = blockIdx.x;
    __shared__ double red[128];
    const double inv = cnt[c] > 0 ? 1.0 / (double)cnt[c] : 0.0;
    double s = 0.0;
    for (int t = threadIdx.x; t < d; t += blockDim.x) {
        const double v = cnt[c] > 0 ? mc[(int64_t)c * d + t] * inv - colsum[t] * inv_n : 0.0;
        mc[(int64_t)c * d + t] = v;
        mcT[(int64_t)t * Cp + c] = v; // [feature][bin]: lanes of a warp read consecutive bins
        s += v * v;
    }
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = blockDim.x / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) mc2[c] = red[0];
}

// |a_u - m_c|^2 for every query slot u and every bin c, once per label set: an FP64 GEMM (U x C x d) on the FP64 tensor cores
// (mma.sync m8n8k4.f64 -> DMMA.8x8x4): 128 x 64 tiles per CTA, 8 warps of 32 x 32 (4 x 4 MMA tiles, 16 DMMA per 8 shared-memory
// reads), 16 features per shared-memory stage, the next stage's global loads in flight behind the arithmetic.
// tqs[u][c] = fl32( |a_u|^2 - 2 a_u.m_c + |m_c|^2 ), a_u = the FP32 centred feature row the tensor core contracts.  Both the
// speculation start (argmin over bins -- every rank must derive the same vector, and the summation order here is fixed) and
// the query terms of the owned rows come from it.
constexpr int CT_M = 128, CT_N = 64, CT_K = 16;
constexpr int CT_LDA = CT_M + 4, CT_LDB = CT_N + 4; // pitch = 4 mod 16 doubles: the (k-slot t, row g) fragment reads hit 16 bank pairs
constexpr size_t CT_SMEM = sizeof(double) * (2 * CT_K * (CT_LDA + CT_LDB) + 4 * CT_M);
__device__ __forceinline__ void ct_dmma(double (&c)[2], double a, double b)
{
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
}
__global__ void __launch_bounds__(256, 2) centroid_terms_kernel(const int32_t *__restrict__ qpoint, int64_t U, const float *__restrict__ Xf,
                                                                int32_t ldf, int32_t d, const double *__restrict__ mcT, int32_t Cp,
                                                                const double *__restrict__ mc2, int32_t C, float *__restrict__ tqs)
{
    chb_pdl_wait();
    // two stages: the stores of stage s + 1 overlap the MMAs of stage s (54 KB: dynamic shared memory, CT_SMEM)
    extern __shared__ __align__(16) unsigned char ct_smem[];
    double (*As)[CT_K][CT_LDA] = reinterpret_cast<double (*)[CT_K][CT_LDA]>(ct_smem);
    double (*Bs)[CT_K][CT_LDB] = reinterpret_cast<double (*)[CT_K][CT_LDB]>(ct_smem + sizeof(double) * 2 * CT_K * CT_LDA);
    double (*aa_s)[CT_M] = reinterpret_cast<double (*)[CT_M]>(ct_smem + sizeof(double) * 2 * CT_K * (CT_LDA + CT_LDB));
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int gq = lane >> 2, tq = lane & 3;
    const int wr = (warp >> 1) * 32, wc = (warp & 1) * 32; // the warp's 32 x 32 corner of the CTA tile
    const int64_t u0 = (int64_t)blockIdx.x * CT_M;
    // A CTA owns 128 query slots and walks over ALL bin tiles (64 bins each): the stages of consecutive tiles form one software
    // pipeline (the first loads of the next tile are in flight behind the last MMAs and the epilogue of the current one); the
    // query rows come from L1 / L2 after the first tile.
    // loader roles: A: query lq (two per thread: lq, lq + 64), features 4 lk .. 4 lk + 3 of the stage -- a warp covers 32
    // consecutive rows with one lk, so its shared-memory stores are conflict-free; B: feature bk, bins 4 bc .. 4 bc + 3
    const int lq = tid & 63, lk = tid >> 6;
    const int bk = tid >> 4, bc = tid & 15;
    const float *xrow[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int64_t uq = u0 + lq + 64 * h;
        xrow[h] = uq < U ? Xf + (int64_t)qpoint[uq] * ldf : nullptr;
    }
    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    double aa[2] = {0.0, 0.0}; // |a|^2 of the loader's two rows over its features (4 of every 16), first tile only; the 4 loaders are summed below
    float4 va[2];
    double2 vb[2];
    const int KS = (d + CT_K - 1) / CT_K, NT = (C + CT_N - 1) / CT_N, total = KS * NT;
    auto fetch = [&](int st) {
        const int nt = st / KS, k0 = (st - nt * KS) * CT_K;
        const int t = k0 + 4 * lk;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            va[h] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (xrow[h] && t < ldf) va[h] = *reinterpret_cast<const float4 *>(xrow[h] + t); // pads beyond d are zero (prep_f32_kernel)
            if (t + 0 >= d) va[h].x = 0.f;
            if (t + 1 >= d) va[h].y = 0.f;
            if (t + 2 >= d) va[h].z = 0.f;
            if (t + 3 >= d) va[h].w = 0.f;
        }
        const int tb = k0 + bk;
        const int c = nt * CT_N + 4 * bc; // Cp is a multiple of 32: a group of 4 bins is inside the padded row or outside
        vb[0] = vb[1] = make_double2(0.0, 0.0);
        if (tb < d && c + 3 < Cp) {
            vb[0] = *reinterpret_cast<const double2 *>(mcT + (int64_t)tb * Cp + c);
            vb[1] = *reinterpret_cast<const double2 *>(mcT + (int64_t)tb * Cp + c + 2);
        }
    };
    auto stash = [&](int buf, bool first_tile) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const double x0 = (double)va[h].x, x1 = (double)va[h].y, x2 = (double)va[h].z, x3 = (double)va[h].w;
            As[buf][4 * lk + 0][lq + 64 * h] = x0;
            As[buf][4 * lk + 1][lq + 64 * h] = x1;
            As[buf][4 * lk + 2][lq + 64 * h] = x2;
            As[buf][4 * lk + 3][lq + 64 * h] = x3;
            if (first_tile) {
                aa[h] = fma(x0, x0, aa[h]);
                aa[h] = fma(x1, x1, aa[h]);
                aa[h] = fma(x2, x2, aa[h]);
                aa[h] = fma(x3, x3, aa[h]);
            }
        }
        *reinterpret_cast<double2 *>(&Bs[buf][bk][4 * bc]) = vb[0];
        *reinterpret_cast<double2 *>(&Bs[buf][bk][4 * bc + 2]) = vb[1];
    };
    fetch(0);
    stash(0, true);
    __syncthreads();
    int buf = 0, ks = 0, nt = 0;
    for (int st = 0; st < total; ++st, buf ^= 1) {
        const bool more = st + 1 < total;
        if (more) fetch(st + 1);
#pragma unroll
        for (int k = 0; k < CT_K; k += 4) {
            // A fragment: (row g, k-slot t); B fragment: (k-slot t, column g)
            double af[4], bf[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) af[i] = As[buf][k + tq][wr + 8 * i + gq];
#pragma unroll
            for (int j = 0; j < 4; ++j) bf[j] = Bs[buf][k + tq][wc + 8 * j + gq];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) ct_dmma(acc[i][j], af[i], bf[j]);
        }
        const bool last_k = ks == KS - 1;
        if (last_k && nt == 0) { // |a_u|^2 is complete (every loader has stashed all its stages of the first tile)
#pragma unroll
            for (int h = 0; h < 2; ++h) aa_s[lk][lq + 64 * h] = aa[h];
        }
        if (more) stash(buf ^ 1, st + 1 < KS); // that buffer was last read in the previous iteration, which every warp has left
        __syncthreads();
        if (last_k) {
            // C fragment: lane (g, t) holds rows 8 i + g, columns 8 j + 2t, + 1 of the warp's corner
            const int cb = nt * CT_N + wc + 2 * tq;
            double m2[4][2];
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int e = 0; e < 2; ++e) m2[j][e] = cb + 8 * j + e < C ? mc2[cb + 8 * j + e] : 0.0;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int r = wr + 8 * i + gq;
                const int64_t u = u0 + r;
                const double au = (aa_s[0][r] + aa_s[1][r]) + (aa_s[2][r] + aa_s[3][r]);
                float *out = tqs + u * Cp + cb;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float v0 = (float)fmax(fma(-2.0, acc[i][j][0], au) + m2[j][0], 0.0);
                    const float v1 = (float)fmax(fma(-2.0, acc[i][j][1], au) + m2[j][1], 0.0);
                    if (u < U) {
                        if (cb + 8 * j + 1 < C) *reinterpret_cast<float2 *>(out + 8 * j) = make_float2(v0, v1);
                        else if (cb + 8 * j < C) out[8 * j] = v0;
                    }
                    acc[i][j][0] = acc[i][j][1] = 0.0;
                }
            }
            ks = 0;
            ++nt;
        } else {
            ++ks;
        }
    }
}

// one warp per query slot: bin with the smallest |a_u - m_c|^2 among the bins that have seeds (lowest bin on ties); C if none
__global__ void __launch_bounds__(256) guess_from_terms_kernel(const float *__restrict__ tqs, int64_t U, int32_t Cp, int32_t C,
                                                               const int32_t *__restrict__ mcnt, int32_t *__restrict__ guess_all)
{
    chb_pdl_enter();
    const int lane = threadIdx.x & 31;
    const int64_t u = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (u >= U) return;
    float best = INFINITY;
    int bc = C;
    for (int c = lane; c < C; c += 32) {
        if (mcnt[c] <= 0) continue;
        const float v = tqs[u * Cp + c];
        if (v < best) { best = v; bc = c; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(CHB_FULL, best, o);
        const int oc = __shfl_xor_sync(CHB_FULL, bc, o);
        if (ov < best || (ov == best && oc < bc)) { best = ov; bc = oc; }
    }
    if (lane == 0) guess_all[u] = bc;
}

// tq[c][r] = tqs[slot of row r][c] for the owned rows: tiles of 128 rows x 32 bins through shared memory, coalesced both ways,
// 16 independent 128-byte row reads per warp in flight (a 32 x 32 tile with 4 moved 2.4 TB/s on the 1.9 GB of 1M x 500)
constexpr int QT_ROWS = 128;
__global__ void __launch_bounds__(256) query_terms_gather_kernel(const float *__restrict__ tqs, int32_t Cp, int64_t u_first,
                                                                 const int32_t *__restrict__ row_slot, int64_t nown, int32_t C,
                                                                 int64_t ldt, float *__restrict__ tq)
{
    chb_pdl_enter();
    __shared__ float tile[QT_ROWS][33];
    const int x = threadIdx.x & 31, y = threadIdx.x >> 5;
    const int64_t r0 = (int64_t)blockIdx.x * QT_ROWS;
    const int c0 = blockIdx.y * 32;
    const int c = c0 + x;
#pragma unroll
    for (int i = 0; i < QT_ROWS / 8; ++i) {
        const int64_t r = r0 + y + 8 * i;
        tile[y + 8 * i][x] = (r < nown && c < C) ? tqs[(u_first + row_slot[r]) * Cp + c] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
        const int j = y + 8 * jj;
        if (c0 + j >= C) continue;
#pragma unroll
        for (int q = 0; q < QT_ROWS / 32; ++q) {
            const int64_t r = r0 + x + 32 * q;
            if (r < nown) tq[(int64_t)(c0 + j) * ldt + r] = tile[x + 32 * q][j];
        }
    }
}

__global__ void guess_scatter_kernel(const int32_t *__restrict__ qpoint, const int32_t *__restrict__ guess_all, int64_t U, int32_t C,
                                     int32_t *__restrict__ tent)
{
    chb_pdl_enter();
    const int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u < U && guess_all[u] < C) tent[qpoint[u]] = guess_all[u];
}

// ---------------------------------------------------------------------------------------------------------
// bin pruning.  The label of a query is the bin with the smallest hull distance (algorithm.py:47-58).  Two bounds
// decide most (query, bin) pairs without a neighbour search or a QP:
//   upper  UB(q)   = distance from q to the nearest SEED contig of its guessed bin g: seeds never change label and are
//                    visible to every query, the nearest visible member of a bin is one of its k neighbours, and the
//                    hull distance is at most the distance to a neighbour -- so min_c D(q, c) <= D(q, g) <= UB(q);
//   lower  LB(q,c) = |x_q - mu_c| - max_i |x_i - mu_c| over the bin's current members: the hull of any k of them lies in
//                    that ball -- so D(q, c) >= LB(q, c).
// A bin with LB(q, c) > UB(q) (strictly, with a rounding margin) cannot be the argmin, not even on a tie, and is
// pruned: admission threshold -inf, no candidates, no QP, hull distance +inf.  Rows are ordered by guessed bin so that
// whole 128-query row blocks prune the same bins and their tiles are skipped by the fused kernel.
// ---------------------------------------------------------------------------------------------------------
// seed contigs transposed, [feature][seed] in (bin, index) order, as the centred FP32 values fl32(x - mu) (prep_f32_kernel)
__global__ void seed_transpose_kernel(const float *__restrict__ Xf, int32_t ldf, int32_t d, const int32_t *__restrict__ seed_idx,
                                      int64_t ns, float *__restrict__ seedT)
{
    chb_pdl_enter();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ns * d) return;
    const int64_t sidx = i / d;
    const int t = (int)(i - sidx * d);
    seedT[(int64_t)t * ns + sidx] = Xf[(int64_t)seed_idx[sidx] * ldf + t];
}

// UB = an upper bound of the distance to the nearest seed of the guessed bin, and of the squared distance to its k-th nearest
// seed (an admission threshold for the first round, when there is no cached neighbour set yet: all seeds are visible members
// of the bin, so the bin's k-th smallest squared distance cannot exceed it).
//
// Both are BOUNDS, not distances, so they are evaluated in FP32 on the centred features a = fl32(x - mu) the tensor core
// contracts as well, and inflated rigorously: with D = x_q - x_s and D~ = a_q - a_s (exact difference of the stored floats),
//   | D~ - D |_2 <= 2^-24 (|x_q - mu| + |x_s - mu|)            (one rounding per stored coordinate)
//   S~ = fl32 sum of fl32(a_q,t - a_s,t)^2  >=  |D~|^2 (1 - (d + 3) 2^-24)   (all terms non-negative)
// and 1 / sqrt(1 - x) <= 1 + x for 0 <= x <= 1/2, hence
//   |D| <= sqrt(S~) f + 6e-8 (|a_q| + max_i |a_i|),   f = max(1 + 1e-5, 1 + (d + 3) 2^-24)   (ub_inflation)
// every operation rounded upwards; f = 1 + 1e-5 up to d = 164, 1 + 6.1e-5 at d = 1024.  The pruning test (threshold_kernel)
// keeps margins a hundred times wider than what this adds.
//
// Rows come grouped by guessed bin (row_end[c] = end of bin c's group), so a CTA takes 64 rows of ONE bin against that bin's
// seeds: a register-tiled squared-distance "GEMM" -- 4 rows x 4 seeds per thread, operands staged through shared memory in
// 32-feature slices -- then per row the minimum and k rounds of minimum extraction over the row's values (kept in shared
// memory, up to RU_MAXSEED seeds per bin; beyond that only the minimum, ubk2 = +inf).
constexpr int RU_ROWS = 64, RU_SEEDS = 32, RU_TK = 32, RU_THREADS = 128, RU_MAXSEED = 128;
constexpr int RU_QP = RU_ROWS + 4, RU_DP = RU_MAXSEED + 1;
inline float ub_inflation(int d)
{
    const double f = 1.0 + (double)(d + 3) * 5.9604644775390625e-08;
    const float fr = (float)f; // round to nearest: step up once if that went below
    return std::max(1.00001f, (double)fr >= f ? fr : std::nextafter(fr, 2.f));
}
__device__ __forceinline__ float ru_bound(float s2, float scale, float inflate)
{
    return __fadd_ru(__fmul_ru(__fsqrt_ru(s2), inflate), __fmul_ru(6e-8f, scale));
}
__global__ void __launch_bounds__(RU_THREADS) row_ub_kernel(const int32_t *__restrict__ row_pt, int64_t nown, const float *__restrict__ Xf,
                                                            int32_t ldf, int32_t d, int32_t C, int32_t k, const int32_t *__restrict__ seed_off,
                                                            const float *__restrict__ seedT, int64_t ns, const int32_t *__restrict__ row_end,
                                                            const float *__restrict__ sq_row, const unsigned int *__restrict__ nrm_max_bits,
                                                            float inflate, float *__restrict__ ub_out, float *__restrict__ ubk2_out)
{
    chb_pdl_wait();
    __shared__ float dist[RU_ROWS * RU_DP];                 // 33 KB
    __shared__ __align__(16) float qs[RU_TK * RU_QP];       // feature-major slice of the 64 query rows
    __shared__ __align__(16) float ss[RU_TK * RU_SEEDS];
    __shared__ int s_bin, s_r0, s_nr;
    __shared__ unsigned int s_min[RU_ROWS];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // which (bin, 64-row chunk) is this CTA?  bins 0..C (C = "no seeded bin": rows without any bound).  Warp 0 scans the chunk
    // counts 32 bins at a time.
    if (warp == 0) {
        int acc = 0, found = -1, r0 = 0, nr = 0;
        for (int cb = 0; cb <= C && found < 0; cb += 32) {
            const int c = cb + lane;
            const int beg = (c <= C && c > 0) ? row_end[c - 1] : 0, end = c <= C ? row_end[c] : beg;
            const int nch = c <= C ? (end - beg + RU_ROWS - 1) / RU_ROWS : 0;
            int incl = nch;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(CHB_FULL, incl, o);
                if (lane >= o) incl += v;
            }
            const int excl = acc + incl - nch;
            const bool mine = (int)blockIdx.x >= excl && (int)blockIdx.x < excl + nch;
            const unsigned who = __ballot_sync(CHB_FULL, mine);
            if (who) {
                const int src = __ffs(who) - 1;
                found = __shfl_sync(CHB_FULL, c, src);
                const int b0 = __shfl_sync(CHB_FULL, beg, src), e0 = __shfl_sync(CHB_FULL, end, src), x0 = __shfl_sync(CHB_FULL, excl, src);
                r0 = b0 + ((int)blockIdx.x - x0) * RU_ROWS;
                nr = min(RU_ROWS, e0 - r0);
            }
            acc += __shfl_sync(CHB_FULL, incl, 31);
        }
        if (lane == 0) { s_bin = found; s_r0 = r0; s_nr = nr; }
    }
    if (tid < RU_ROWS) s_min[tid] = 0x7f800000u; // +inf
    __syncthreads();
    const int c = s_bin, r0 = s_r0, nr = s_nr;
    if (c < 0) return;
    const int sbeg = c < C ? seed_off[c] : 0, nseed = c < C ? seed_off[c + 1] - seed_off[c] : 0;
    const int ty = tid >> 3, tx = tid & 7; // rows 4 ty .. 4 ty + 3, seeds 4 tx .. 4 tx + 3 of the tile
    // loader roles: query slice element e = tid + 128 i -> (row e >> 5, feature e & 31): 16 per thread; seed slice: 8 per thread
    const float *qrow[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const int rr = (tid + RU_THREADS * i) >> 5;
        qrow[i] = rr < nr ? Xf + (int64_t)row_pt[r0 + rr] * ldf : nullptr;
    }
    for (int sb = 0; sb < nseed; sb += RU_SEEDS) {
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
        for (int t0 = 0; t0 < d; t0 += RU_TK) {
            float qv_[16], sv_[8];
            const int tq = t0 + lane; // this thread's feature of the query slice (tid & 31 == lane)
#pragma unroll
            for (int i = 0; i < 16; ++i) qv_[i] = (qrow[i] && tq < d) ? __ldg(qrow[i] + tq) : 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int e = tid + RU_THREADS * i, t = e >> 5, sidx = e & 31;
                sv_[i] = (sb + sidx < nseed && t0 + t < d) ? __ldg(seedT + (int64_t)(t0 + t) * ns + sbeg + sb + sidx) : 0.f;
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) qs[lane * RU_QP + ((tid + RU_THREADS * i) >> 5)] = qv_[i];
#pragma unroll
            for (int i = 0; i < 8; ++i) ss[tid + RU_THREADS * i] = sv_[i];
            __syncthreads();
#pragma unroll 8
            for (int t = 0; t < RU_TK; ++t) {
                const float4 q4 = *reinterpret_cast<const float4 *>(&qs[t * RU_QP + 4 * ty]);
                const float4 s4 = *reinterpret_cast<const float4 *>(&ss[t * RU_SEEDS + 4 * tx]);
                const float qv[4] = {q4.x, q4.y, q4.z, q4.w}, sv[4] = {s4.x, s4.y, s4.z, s4.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float df = qv[i] - sv[j]; // pad features are 0 - 0
                        acc[i][j] = fmaf(df, df, acc[i][j]);
                    }
            }
            __syncthreads();
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int rr = 4 * ty + i;
            float mn = INFINITY;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int sidx = sb + 4 * tx + j;
                if (sidx < nseed) {
                    mn = fminf(mn, acc[i][j]);
                    if (sidx < RU_MAXSEED) dist[rr * RU_DP + sidx] = acc[i][j];
                }
            }
            if (mn < INFINITY) atomicMin(&s_min[rr], __float_as_uint(mn)); // non-negative floats order like their bits
        }
    }
    __syncthreads();
    // per row: warp w takes rows w, w + 4, ...; k-th smallest by k rounds of "extract the minimum" (as many lanes as seeds)
    const float amax = __fsqrt_ru(__uint_as_float(*nrm_max_bits));
    for (int rr = warp; rr < nr; rr += RU_THREADS / 32) {
        const float mn2 = __uint_as_float(s_min[rr]);
        float kth = INFINITY;
        if (nseed >= k && nseed <= RU_MAXSEED) {
            float v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) v[u] = (lane + 32 * u < nseed) ? dist[rr * RU_DP + lane + 32 * u] : INFINITY;
            for (int round = 0; round < k; ++round) {
                const float mine = fminf(fminf(v[0], v[1]), fminf(v[2], v[3]));
                float m = mine;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) m = fminf(m, __shfl_xor_sync(CHB_FULL, m, o));
                kth = m;
                const unsigned owners = __ballot_sync(CHB_FULL, mine == m);
                if (lane == __ffs(owners) - 1) { // remove one copy of the minimum
                    if (v[0] == m) v[0] = INFINITY; else if (v[1] == m) v[1] = INFINITY; else if (v[2] == m) v[2] = INFINITY; else v[3] = INFINITY;
                }
            }
        }
        if (lane == 0) {
            const float scale = __fadd_ru(sq_row[r0 + rr], amax);
            ub_out[r0 + rr] = mn2 < INFINITY ? ru_bound(mn2, scale, inflate) : INFINITY;
            const float bk = kth < INFINITY ? ru_bound(kth, scale, inflate) : INFINITY;
            ubk2_out[r0 + rr] = bk < INFINITY ? __fmul_ru(bk, bk) : INFINITY;
        }
    }
}

// rows = owned slots grouped by guessed bin (any order inside a group): histogram, scan, scatter -- no host round trip
__global__ void row_hist_kernel(const int32_t *__restrict__ guess_own, int64_t nown, int32_t *__restrict__ hist)
{
    chb_pdl_enter();
    const int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u < nown) atomicAdd(&hist[guess_own[u]], 1);
}
__global__ void row_scan_kernel(const int32_t *__restrict__ hist, int32_t nb, int32_t *__restrict__ cursor)
{
    chb_pdl_enter();
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        int acc = 0;
        for (int b = 0; b < nb; ++b) { cursor[b] = acc; acc += hist[b]; }
    }
}
__global__ void row_scatter_kernel(const int32_t *__restrict__ guess_own, int64_t nown, int32_t *__restrict__ cursor,
                                   int32_t *__restrict__ row_slot)
{
    chb_pdl_enter();
    const int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u < nown) row_slot[atomicAdd(&cursor[guess_own[u]], 1)] = (int32_t)u;
}

__global__ void row_gather_kernel(const int32_t *__restrict__ row_slot, const int32_t *__restrict__ qpoint_own,
                                  const int32_t *__restrict__ guess_own, const float *__restrict__ nrm, int64_t nown,
                                  int32_t *__restrict__ row_pt, int32_t *__restrict__ row_guess, int32_t *__restrict__ slot_row,
                                  float *__restrict__ sq_row)
{
    chb_pdl_enter();
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nown) return;
    const int sl = row_slot[r];
    const int pt = qpoint_own[sl];
    row_pt[r] = pt;
    row_guess[r] = guess_own[sl];
    slot_row[sl] = (int32_t)r;
    sq_row[r] = __fmul_ru(__fsqrt_ru(nrm[pt]), 1.000001f); // >= |a_q|
}

// one warp per column entry: y = fl32(x_i - mu_c) split into the [hi | lo] operand row, the column term
// |y|^2 + 2 m_c.y, and the per-bin maxima of |y|^2 and of |column term| (for the error bound); padding columns are zero
__global__ void __launch_bounds__(256) column_gather_kernel(const int32_t *__restrict__ col_pt, const int32_t *__restrict__ ntiles,
                                                            const int32_t *__restrict__ tile_bin, const double *__restrict__ X,
                                                            int32_t ldx, int32_t d, const double *__restrict__ colsum, double inv_n,
                                                            const double *__restrict__ mc, int32_t dp8, int32_t Kp2,
                                                            float *__restrict__ out, float *__restrict__ col_term,
                                                            unsigned int *__restrict__ ym2_bits, unsigned int *__restrict__ tcmax_bits)
{
    chb_pdl_enter();
    const int lane = threadIdx.x & 31;
    const int64_t e = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (e >= (int64_t)(*ntiles) * BN) return;
    const int ptx = col_pt[e];
    float *orow = out + e * Kp2;
    if (ptx < 0) {
        for (int t = lane; t < Kp2; t += 32) orow[t] = 0.f;
        if (lane == 0) col_term[e] = 0.f;
        return;
    }
    const int c = tile_bin[e / BN];
    const double *xr = X + (int64_t)ptx * ldx;
    const double *m = mc + (int64_t)c * d;
    double yy = 0.0, my = 0.0;
    for (int t = lane; t < dp8; t += 32) {
        float hi = 0.f, lo = 0.f;
        if (t < d) {
            const float yf = (float)(xr[t] - colsum[t] * inv_n - m[t]);
            hi = __uint_as_float(__float_as_uint(yf) & 0xffffe000u);
            lo = __uint_as_float(__float_as_uint(yf - hi) & 0xffffe000u);
            yy = fma((double)yf, (double)yf, yy);
            my = fma(m[t], (double)yf, my);
        }
        orow[t] = hi;
        orow[dp8 + t] = lo;
    }
    for (int t = 2 * dp8 + lane; t < Kp2; t += 32) orow[t] = 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        yy += __shfl_xor_sync(CHB_FULL, yy, o);
        my += __shfl_xor_sync(CHB_FULL, my, o);
    }
    if (lane == 0) {
        const double term = yy + 2.0 * my;
        col_term[e] = (float)term;
        atomicMax(&ym2_bits[c], __float_as_uint(__double2float_ru(yy)));          // non-negative floats order like their bits
        atomicMax(&tcmax_bits[c], __float_as_uint(__double2float_ru(fabs(term))));
    }
}

// ---- wide variant
__global__ void __launch_bounds__(256) column_gather_wide_kernel(const int32_t *__restrict__ col_pt, const int32_t *__restrict__ ntiles,
                                                            const int32_t *__restrict__ tile_bin, const double *__restrict__ X,
                                                            int32_t ldx, int32_t d, const double *__restrict__ colsum, double inv_n,
                                                            const double *__restrict__ mc, int32_t dp8, int32_t Kp2,
                                                            float *__restrict__ out, float *__restrict__ col_term,
                                                            unsigned int *__restrict__ ym2_bits, unsigned int *__restrict__ tcmax_bits)
{
    chb_pdl_enter();
    // The same for large inputs: a CTA takes CG_COLS consecutive column entries -- inside one 128-column tile, hence of one
    // bin -- CG_COLS / 8 per warp, and folds their maxima in shared memory: one atomic pair per CTA, a quarter of the CTAs.
    // 1M contigs: 1.30 -> 0.83 ms per launch (2.5 GB moved); at 20k contigs the one-column-per-warp kernel above is faster
    // (24 against 28 us: too few CTAs to fill the machine), so the host picks by the number of columns.
    constexpr int CG_COLS = 32;
    __shared__ unsigned int s_y[8], s_t[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t e0 = (int64_t)blockIdx.x * CG_COLS;
    if (e0 >= (int64_t)(*ntiles) * BN) return; // whole CTA (uniform)
    const int c = tile_bin[e0 / BN];
    const double *m = mc + (int64_t)c * d;
    unsigned int ymax = 0, tmax = 0; // non-negative floats order like their bits
    for (int w = 0; w < CG_COLS / 8; ++w) {
        const int64_t e = e0 + warp * (CG_COLS / 8) + w;
        const int ptx = col_pt[e];
        float *orow = out + e * Kp2;
        if (ptx < 0) { // padding column: zero row, never visible
            for (int t = lane; t < Kp2; t += 32) orow[t] = 0.f;
            if (lane == 0) col_term[e] = 0.f;
            continue;
        }
        const double *xr = X + (int64_t)ptx * ldx;
        double yy = 0.0, my = 0.0;
        for (int t = lane; t < dp8; t += 32) {
            float hi = 0.f, lo = 0.f;
            if (t < d) {
                const float yf = (float)(xr[t] - colsum[t] * inv_n - m[t]);
                hi = __uint_as_float(__float_as_uint(yf) & 0xffffe000u);
                lo = __uint_as_float(__float_as_uint(yf - hi) & 0xffffe000u);
                yy = fma((double)yf, (double)yf, yy);
                my = fma(m[t], (double)yf, my);
            }
            orow[t] = hi;
            orow[dp8 + t] = lo;
        }
        for (int t = 2 * dp8 + lane; t < Kp2; t += 32) orow[t] = 0.f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            yy += __shfl_xor_sync(CHB_FULL, yy, o);
            my += __shfl_xor_sync(CHB_FULL, my, o);
        }
        const double term = yy + 2.0 * my;
        if (lane == 0) col_term[e] = (float)term;
        ymax = max(ymax, __float_as_uint(__double2float_ru(yy)));
        tmax = max(tmax, __float_as_uint(__double2float_ru(fabs(term))));
    }
    if (lane == 0) { s_y[warp] = ymax; s_t[warp] = tmax; }
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
        for (int w = 1; w < 8; ++w) { ymax = max(ymax, s_y[w]); tmax = max(tmax, s_t[w]); }
        if (ymax) atomicMax(&ym2_bits[c], ymax);
        if (tmax) atomicMax(&tcmax_bits[c], tmax);
    }
}

// slack of (query r, bin c): bound on |key - |x_q - x_i|^2| for every column i of the bin (see the block comment above).
//   contraction: 2 * eps_rel * |a_q| * max|y|      (eps_rel = (3d + 64) 2^-23 bounds the dot-product error, gram_tc.cu)
//   FP32 roundings of the three terms and of the operands: 2^-21 * (tq + max|column term| + 2 |a_q| max|y| + D (|a_q| + max|y|) + D^2),  D = |a_q - m_c| + max|y|
__device__ __forceinline__ float pair_slack(double eps_rel, float nrm_q, float ym2, float tcmax, float tq)
{
    const double sq = sqrt((double)nrm_q), ym = sqrt((double)ym2), dq = sqrt((double)tq);
    const double e = 2.0 * eps_rel * sq * ym + 4.76837158203125e-07 * ((double)tq + (double)tcmax + 2.0 * sq * ym + (dq + ym) * (sq + ym) + (dq + ym) * (dq + ym));
    return __double2float_ru(e * (1.0 + 1e-6) + 1e-30);
}

// Work list of the fused kernel: one item per surviving (row block, bin) = {row block, bin, first tile, #tiles}, in row-block
// order, and for each of the G CTAs the contiguous range of items whose cumulative tile count falls into its 1/G share.
// Whole items only (a (query, bin) list is built by one CTA), so CTAs differ by at most one bin's tiles.  One block: the tail of
// pairs_plan_kernel when the compact buffer would overflow (mode 0); s_items / s_tiles: 1024 ints of shared memory each.
__device__ void items_body(const uint8_t *__restrict__ skip, int64_t nrb, int32_t C, const int32_t *__restrict__ seg_off, int32_t G,
                           int4 *__restrict__ items, int32_t *__restrict__ cta_begin, int32_t *__restrict__ totals, int *s_items,
                           int *s_tiles)
{
    __shared__ int tot_items, tot_tiles;
    const int tid = threadIdx.x;
    const int64_t ne = nrb * C;
    const int64_t per = (ne + 1023) / 1024;
    const int64_t e0 = tid * per < ne ? tid * per : ne, e1 = e0 + per < ne ? e0 + per : ne;
    int ni = 0, nt = 0;
    for (int64_t e = e0; e < e1; ++e) {
        const int c = (int)(e % C);
        const int w = (seg_off[c + 1] - seg_off[c]) / BN;
        if (!skip[e] && w > 0) { ++ni; nt += w; }
    }
    s_items[tid] = ni;
    s_tiles[tid] = nt;
    __syncthreads();
    // inclusive scan (Hillis-Steele) over the 1024 partial counts
    for (int o = 1; o < 1024; o <<= 1) {
        const int a = tid >= o ? s_items[tid - o] : 0, b = tid >= o ? s_tiles[tid - o] : 0;
        __syncthreads();
        s_items[tid] += a;
        s_tiles[tid] += b;
        __syncthreads();
    }
    if (tid == 1023) { tot_items = s_items[1023]; tot_tiles = s_tiles[1023]; }
    for (int b = tid; b <= G; b += 1024) cta_begin[b] = INT32_MAX;
    __syncthreads();
    const int TI = tot_items, TT = tot_tiles;
    int oi = s_items[tid] - ni, ot = s_tiles[tid] - nt; // exclusive prefixes of this thread's chunk
    for (int64_t e = e0; e < e1; ++e) {
        const int c = (int)(e % C);
        const int w = (seg_off[c + 1] - seg_off[c]) / BN;
        if (!skip[e] && w > 0) {
            items[oi] = make_int4((int)(e / C), c, seg_off[c] / BN, w);
            const int cta = (int)(((int64_t)ot * G) / (TT > 0 ? TT : 1));
            atomicMin(&cta_begin[cta], oi);
            ++oi;
            ot += w;
        }
    }
    __syncthreads();
    if (tid == 0) {
        cta_begin[G] = TI;
        for (int b = G - 1; b >= 0; --b)
            if (cta_begin[b] > cta_begin[b + 1]) cta_begin[b] = cta_begin[b + 1]; // CTAs without an item of their own
        totals[0] = TT;
    }
}

// ---------------------------------------------------------------------------------------------------------
// compaction.  After pruning, the rows that still need a bin are few and scattered over the row blocks (in a "side" bin
// of a row block typically 5-10 of the 128 rows survive), so contracting (row block x bin) tiles wastes most of every
// tile.  The surviving (row, bin) pairs are therefore regrouped PER BIN: bin c's survivors become ceil(n_c / 128) dense
// 128-row blocks whose query operand rows are gathered into a compact buffer.  mode = 1: work items are (pair block,
// bin); mode = 0 (the compact buffer would overflow: little pruning): items stay (row block, bin) as before.
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) pairs_plan_kernel(const int32_t *__restrict__ bin_surv, const int32_t *__restrict__ seg_off,
                                                          int32_t C, int64_t cap_pairs, int32_t G, int32_t *__restrict__ pair_off,
                                                          int32_t *__restrict__ scratch /* 2 (C + 1) */, int4 *__restrict__ items,
                                                          int32_t *__restrict__ cta_begin, int32_t *__restrict__ totals,
                                                          int32_t *__restrict__ mode, int32_t dense_ok,
                                                          const uint8_t *__restrict__ skip, int64_t nrb)
{
    chb_pdl_enter();
    __shared__ int s_mode, s_ti, s_tt;
    constexpr int PLAN_SMEM_BINS = 2048;
    __shared__ int s_nb[PLAN_SMEM_BINS], s_w[PLAN_SMEM_BINS];
    __shared__ int s_begin[1024 + 1]; // cta_begin while it is built (G <= 1024: the serial suffix-min then stays out of L2)
    int32_t *item_off = scratch, *tile_cum = scratch + C + 1;
    const int tid = threadIdx.x;
    const bool in_smem = C <= PLAN_SMEM_BINS; // the serial prefix below then walks shared memory instead of L2
    // per-bin block and tile counts first (all threads, coalesced), then one thread runs the three prefix sums over them
    for (int c = tid; c < C; c += 1024) {
        const int nb = (bin_surv[c] + BM - 1) / BM, w = (seg_off[c + 1] - seg_off[c]) / BN;
        if (in_smem) { s_nb[c] = nb; s_w[c] = w; }
        else { item_off[c] = nb; tile_cum[c] = w; }
    }
    __syncthreads();
    if (tid == 0) {
        int64_t po = 0;
        int io = 0, tc = 0;
        for (int c = 0; c < C; ++c) {
            const int nb = in_smem ? s_nb[c] : item_off[c], w = in_smem ? s_w[c] : tile_cum[c];
            pair_off[c] = (int32_t)po;
            item_off[c] = io;
            tile_cum[c] = tc;
            po += (int64_t)nb * BM;
            if (w > 0) { io += nb; tc += nb * w; }
        }
        pair_off[C] = (int32_t)(po < INT32_MAX ? po : INT32_MAX);
        item_off[C] = io;
        tile_cum[C] = tc;
        s_mode = po <= cap_pairs ? 1 : 0;
        if (!s_mode && !dense_ok) {
            // the survivors do not fit the compact buffers and there is no per-(row, bin) list table to fall back on (it
            // was beyond the memory budget, chb_fused_setup): the round is refused -- no items, nothing filled, nothing
            // re-ranked -- and the commit reports CHB_ENOMEM
            s_mode = 2;
            totals[5] = 1; // counters[12]
            io = 0;
            tc = 0;
        }
        s_ti = io;
        s_tt = tc;
        *mode = s_mode;
    }
    __syncthreads();
    if (s_mode == 2) {
        for (int b = tid; b <= G; b += 1024) cta_begin[b] = 0;
        if (tid == 0) totals[0] = 0;
        return;
    }
    if (!s_mode) { // little pruning: the (row block, bin) list instead (shared memory of the per-bin counts is free again)
        items_body(skip, nrb, C, seg_off, G, items, cta_begin, totals, s_nb, s_w);
        return;
    }
    const bool beg_smem = G <= 1024;
    int *beg = beg_smem ? s_begin : cta_begin;
    for (int b = tid; b <= G; b += 1024) beg[b] = INT32_MAX;
    __syncthreads();
    const int TI = s_ti, TT = s_tt;
    for (int c = tid; c < C; c += 1024) {
        const int w = (seg_off[c + 1] - seg_off[c]) / BN;
        if (w <= 0) continue;
        const int nb = item_off[c + 1] - item_off[c];
        for (int b = 0; b < nb; ++b) {
            const int it = item_off[c] + b;
            items[it] = make_int4(pair_off[c] / BM + b, c, seg_off[c] / BN, w);
            atomicMin(&beg[(int)(((int64_t)(tile_cum[c] + b * w) * G) / (TT > 0 ? TT : 1))], it);
        }
    }
    __syncthreads();
    if (tid == 0) {
        beg[G] = TI;
        int nxt = TI;
        for (int b = G - 1; b >= 0; --b) { // CTAs without an item of their own
            const int v = beg[b];
            nxt = v > nxt ? nxt : v;
            beg[b] = nxt;
        }
        totals[0] = TT;
    }
    if (beg_smem) {
        __syncthreads();
        for (int b = tid; b <= G; b += 1024) cta_begin[b] = s_begin[b];
    }
}

// compact pair id -> row, per bin (any order inside a bin), and the pair's query operand row copied into the compact
// buffer; one warp per row.  threshold_kernel left every pair's index inside its bin in row_pid: id = pair_off[bin] + index
// (lane j resolves the row's j-th surviving bin), the operand row is read once and written once per pair.  Padding ids
// keep pair_row = -1 (round_reset_kernel); their operand rows are never initialised -- accumulator rows are independent
// and the epilogue ignores rows without a query.  WIDE = false: rows of up to 96 float4 (d <= 160) stay in registers,
// three per lane; WIDE = true (streamed layout, up to 512 float4): the row is read again (L1) for every copy.
template <bool WIDE>
__global__ void __launch_bounds__(256) pairs_fill_kernel(const int32_t *__restrict__ mode, const int32_t *__restrict__ row_nb,
                                                         const int32_t *__restrict__ row_bins, int64_t nown, int32_t C,
                                                         const int32_t *__restrict__ pair_off, int32_t *__restrict__ pair_row,
                                                         int32_t *__restrict__ row_pid, const float *__restrict__ a2, int32_t Kp2,
                                                         float *__restrict__ ap)
{
    chb_pdl_enter();
    if (*mode != 1) return;
    const int lane = threadIdx.x & 31;
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= nown) return;
    const int nb = row_nb[r];
    if (nb == 0) return;
    const float4 *src = reinterpret_cast<const float4 *>(a2 + r * Kp2);
    const int nq = Kp2 / 4;
    float4 v[3];
    if constexpr (!WIDE) {
#pragma unroll
        for (int u = 0; u < 3; ++u) v[u] = (lane + 32 * u < nq) ? __ldg(src + lane + 32 * u) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    for (int jb = 0; jb < nb; jb += 32) {
        const int j = jb + lane;
        int id = -1;
        if (j < nb) {
            const int c = row_bins[r * C + j];
            id = pair_off[c] + row_pid[r * C + j];
            pair_row[id] = (int32_t)r;
            row_pid[r * C + j] = id; // the re-rank finds this pair's candidate lists under its compact id
        }
        const int cnt = nb - jb < 32 ? nb - jb : 32;
        for (int w = 0; w < cnt; ++w) {
            const int idw = __shfl_sync(CHB_FULL, id, w);
            float4 *dst = reinterpret_cast<float4 *>(ap + (int64_t)idw * Kp2);
            if constexpr (WIDE) {
                for (int u = lane; u < nq; u += 32) dst[u] = __ldg(src + u);
            } else {
#pragma unroll
                for (int u = 0; u < 3; ++u)
                    if (lane + 32 * u < nq) dst[lane + 32 * u] = v[u];
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// fused Gram + selection
// ---------------------------------------------------------------------------------------------------------
template <int KR>
struct TopList {
    float key[KR];
    int idx[KR];
    __device__ __forceinline__ void reset()
    {
#pragma unroll
        for (int s = 0; s < KR; ++s) { key[s] = INFINITY; idx[s] = INT32_MAX; }
    }
    // keeps the KR smallest keys (with their points) in ascending key order; branch-free.  The slot is found by counting
    // (independent compares) and every slot then updates on its own, so the dependency chain is short -- with two
    // epilogue warps per scheduler, latency rather than issue slots is what the epilogue runs out of.  Equal keys are not
    // ordered by index: the re-rank ranks by (key, index) itself, and its overflow test only needs "every dropped entry
    // has a key >= the largest kept key".
    __device__ __forceinline__ void insert(float ka, int ki)
    {
        int cnt = 0;
#pragma unroll
        for (int s = 0; s < KR; ++s) cnt += (key[s] <= ka) ? 1 : 0;
#pragma unroll
        for (int s = KR - 1; s >= 1; --s) {
            const bool shift = s > cnt, here = s == cnt;
            key[s] = shift ? key[s - 1] : (here ? ka : key[s]);
            idx[s] = shift ? idx[s - 1] : (here ? ki : idx[s]);
        }
        key[0] = cnt == 0 ? ka : key[0];
        idx[0] = cnt == 0 ? ki : idx[0];
    }
};

// NKT > 0: the number of K=8 steps per operand half is known at compile time and a tile's MMA sequence is straight-line
// code with immediate descriptor offsets (d = 137..160, the reference's 4-mer + coverage profiles); NKT = 0: any d, the
// sequence is tabulated in shared memory once per CTA; NKT = NKT_STREAMED: d = 161..1024, the query operand streams through
// the ring with the column operand (one stage per 32-feature block, see the layout note at the top).  Only the producer and
// MMA warps differ between the variants; the selection epilogue is the same code.
template <int KR, int NKT>
__global__ void __launch_bounds__(FUSED_THREADS, 1)
gram_select_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_ap,
                   const __grid_constant__ CUtensorMap map_b, const int32_t *__restrict__ mode_p,
                   const int32_t *__restrict__ pair_row, int nbox, int nk, int nstage,
                   const int32_t *__restrict__ col_pt,
                   const int32_t *__restrict__ col_a, const int32_t *__restrict__ col_b, const float *__restrict__ col_nrm,
                   const float *__restrict__ tq_tab, const int32_t *__restrict__ row_point, const int32_t *__restrict__ pos,
                   int64_t nrows, int32_t C, const float *__restrict__ t0_tab, int64_t ldt, const int4 *__restrict__ items,
                   const int32_t *__restrict__ cta_begin, float *__restrict__ cand_key, int32_t *__restrict__ cand_idx,
                   int32_t *__restrict__ tiles_issued)
{
    chb_pdl_wait();
    // This CTA's work: items [cta_begin[b], cta_begin[b + 1]) of the list built by pairs_plan_kernel, each one surviving
    // (row block, bin) = {row block, bin, first tile, #tiles}.  Pruned (row block, bin) pairs are not in the list: their
    // tiles are neither loaded, contracted nor screened.  All three warp roles walk the same items.
    const int item_begin = cta_begin[blockIdx.x], item_end = cta_begin[blockIdx.x + 1];
    // mode 1: item.x is a block of 128 compact (row, bin) pairs of bin item.y, operand rows in the compact buffer (map_ap),
    // pair_row[] names the query row of each; mode 0: item.x is a row block of the resident operand (map_a)
    const int mode = *mode_p;
    // dynamic shared memory: [resident query operand: nbox boxes][column ring: nstage boxes][SmemTail]; streamed:
    // [ring: nstage x 4 boxes][SmemTail]
    constexpr bool STREAM = NKT == NKT_STREAMED;
    constexpr uint32_t STAGE_BYTES = STREAM ? WIDE_STAGE_BOXES * TILE_BYTES : TILE_BYTES;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *base = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t *a_res = base;
    uint8_t *ring = STREAM ? base : base + (size_t)nbox * TILE_BYTES;
    SmemTail &S = *reinterpret_cast<SmemTail *>(ring + (size_t)nstage * STAGE_BYTES);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int s = 0; s < nstage; ++s) {
            mbar_init(&S.full_bar[s], 1);
            mbar_init(&S.empty_bar[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&S.tmem_full_bar[b], 1);
            mbar_init(&S.tmem_empty_bar[b], 8); // one arrival per epilogue warp
        }
        mbar_init(&S.a_full_bar, 1);
        mbar_init(&S.a_empty_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_ap) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&S.tmem_base)), "n"(TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = S.tmem_base;

    if (warp == 0) {
        // ---------------- TMA producer
        if (lane == 0) {
            int s = 0;
            uint32_t ph = 0;
            int cur_rb = -1, na = 0; // row block whose operand is resident, number of operand loads so far
            for (int it = item_begin; it < item_end; ++it) {
                const int4 item = items[it];
                if constexpr (STREAM) {
                    // per tile and 32-feature block b: query boxes b (hi), H + b (lo) and column boxes b, H + b in one stage
                    const int H = nbox >> 1;
                    const CUtensorMap *mq = mode ? &map_ap : &map_a;
                    for (int t = item.z; t < item.z + item.w; ++t) {
                        for (int b = 0; b < H; ++b) {
                            uint8_t *st = ring + (size_t)s * STAGE_BYTES;
                            mbar_wait(&S.empty_bar[s], ph ^ 1);
                            mbar_expect_tx(&S.full_bar[s], STAGE_BYTES);
                            tma_load_2d(st, mq, &S.full_bar[s], b * BK, item.x * BM);
                            tma_load_2d(st + TILE_BYTES, mq, &S.full_bar[s], (H + b) * BK, item.x * BM);
                            tma_load_2d(st + 2 * TILE_BYTES, &map_b, &S.full_bar[s], b * BK, t * BN);
                            tma_load_2d(st + 3 * TILE_BYTES, &map_b, &S.full_bar[s], (H + b) * BK, t * BN);
                            if (++s == nstage) { s = 0; ph ^= 1; }
                        }
                    }
                    continue;
                }
                if (item.x != cur_rb) {
                    // the resident operand may be overwritten once every MMA of the previous row block has completed
                    mbar_wait(&S.a_empty_bar, (uint32_t)((na & 1) ^ 1));
                    mbar_expect_tx(&S.a_full_bar, (uint32_t)nbox * TILE_BYTES);
                    for (int jb = 0; jb < nbox; ++jb)
                        tma_load_2d(a_res + (size_t)jb * TILE_BYTES, mode ? &map_ap : &map_a, &S.a_full_bar, jb * BK, item.x * BM);
                    cur_rb = item.x;
                    ++na;
                }
                for (int t = item.z; t < item.z + item.w; ++t) {
                    for (int jb = 0; jb < nbox; ++jb) {
                        mbar_wait(&S.empty_bar[s], ph ^ 1);
                        mbar_expect_tx(&S.full_bar[s], TILE_BYTES);
                        tma_load_2d(ring + (size_t)s * TILE_BYTES, &map_b, &S.full_bar[s], jb * BK, t * BN);
                        if (++s == nstage) { s = 0; ph ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ---------------- MMA issuer.  One thread feeds the tensor core, so its instruction stream is kept minimal:
        // the (query step, column step) pairing of a tile is the same for every tile and is tabulated once.  The whole
        // warp runs the loop (uniform control flow keeps descriptors in uniform registers); an elected lane issues.
        {
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
            const uint32_t a_addr = smem_u32(a_res);
            constexpr uint32_t DESC_HI = (1024u >> 4) | (1u << 14) | (2u << 29); // SBO = 1024 B, version 1, 128-byte swizzle
            if (NKT == 0 && lane == 0) {
                int m = 0;
                for (int jb = 0; jb < nbox; ++jb) {
                    S.prog_start[jb] = m;
                    for (int u = 0; u < BK / UMMA_K; ++u) {
                        const int j = jb * (BK / UMMA_K) + u; // K=8 step of the column operand
                        if (j >= 2 * nk) break;
                        // column hi step j pairs with query hi step j and query lo step nk + j;
                        // column lo step j - nk pairs with query hi step j - nk
                        const int i0 = j < nk ? j : j - nk;
                        const uint32_t boff = (uint32_t)((u * UMMA_K * 4) >> 4);
                        S.prog[m++] = make_uint2((((a_addr + (uint32_t)(i0 >> 2) * TILE_BYTES) & 0x3FFFFu) >> 4 | (1u << 16)) +
                                                     (uint32_t)(((i0 & 3) * UMMA_K * 4) >> 4), boff);
                        if (j < nk) {
                            const int i1 = nk + j;
                            S.prog[m++] = make_uint2((((a_addr + (uint32_t)(i1 >> 2) * TILE_BYTES) & 0x3FFFFu) >> 4 | (1u << 16)) +
                                                         (uint32_t)(((i1 & 3) * UMMA_K * 4) >> 4), boff);
                        }
                    }
                }
                S.prog_start[nbox] = m;
            }
            __syncwarp();
            const uint32_t ring_lo = ((smem_u32(ring) & 0x3FFFFu) >> 4) | (1u << 16);
            int s = 0;
            uint32_t ph = 0;
            int64_t tt = 0;
            int cur_rb = -1, na = 0;
            for (int it = item_begin; it < item_end; ++it) {
                const int4 item = items[it];
                if (!STREAM && item.x != cur_rb) {
                    // every MMA on the previous row block's operand has been issued: release it, then wait for the new one
                    if (cur_rb >= 0 && elect_one_sync()) umma_commit(&S.a_empty_bar);
                    mbar_wait(&S.a_full_bar, (uint32_t)(na & 1));
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    cur_rb = item.x;
                    ++na;
                }
                for (int t = item.z; t < item.z + item.w; ++t) {
                    const int buf = (int)(tt & 1);
                    const uint32_t tph = (uint32_t)((tt >> 1) & 1);
                    ++tt;
                    mbar_wait(&S.tmem_empty_bar[buf], tph ^ 1); // epilogue has drained this accumulator buffer
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t tmem_d = tmem_base + (uint32_t)(buf * BN);
                    if constexpr (STREAM) {
                        // stage = [query hi | query lo | column hi | column lo] of one 32-feature block: 4 K-steps x
                        // (hi.hi, lo.hi, hi.lo); zero pads past d contribute exact zeros
                        const int H = nbox >> 1;
                        for (int b = 0; b < H; ++b) {
                            const uint32_t st_lo = ring_lo + (uint32_t)s * (STAGE_BYTES >> 4);
                            mbar_wait(&S.full_bar[s], ph);
                            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                            if (elect_one_sync()) {
#pragma unroll
                                for (int u = 0; u < BK / UMMA_K; ++u) {
                                    const uint32_t ko = (uint32_t)((u * UMMA_K * 4) >> 4);
                                    const uint64_t qhi = ((uint64_t)DESC_HI << 32) | (st_lo + ko);
                                    const uint64_t qlo = ((uint64_t)DESC_HI << 32) | (st_lo + (TILE_BYTES >> 4) + ko);
                                    const uint64_t chi = ((uint64_t)DESC_HI << 32) | (st_lo + 2 * (TILE_BYTES >> 4) + ko);
                                    const uint64_t clo = ((uint64_t)DESC_HI << 32) | (st_lo + 3 * (TILE_BYTES >> 4) + ko);
                                    umma_tf32(tmem_d, qhi, chi, idesc, (b | u) != 0);
                                    umma_tf32(tmem_d, qlo, chi, idesc, 1u);
                                    umma_tf32(tmem_d, qhi, clo, idesc, 1u);
                                }
                                umma_commit(&S.empty_bar[s]);
                            }
                            if (++s == nstage) { s = 0; ph ^= 1; }
                        }
                    } else if constexpr (NKT > 0) {
                        constexpr int NBOX = (2 * NKT + 3) / 4;
                        const uint32_t a_lo = ((a_addr & 0x3FFFFu) >> 4) | (1u << 16);
#pragma unroll
                        for (int jb = 0; jb < NBOX; ++jb) {
                            const uint32_t b_lo = ring_lo + (uint32_t)s * (TILE_BYTES >> 4);
                            mbar_wait(&S.full_bar[s], ph);
                            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                            if (elect_one_sync()) {
#pragma unroll
                            for (int u = 0; u < BK / UMMA_K; ++u) {
                                const int j = jb * (BK / UMMA_K) + u;
                                if (j < 2 * NKT) {
                                    const int i0 = j < NKT ? j : j - NKT;
                                    const uint64_t bdesc = ((uint64_t)DESC_HI << 32) | (b_lo + (uint32_t)((u * UMMA_K * 4) >> 4));
                                    umma_tf32(tmem_d,
                                              ((uint64_t)DESC_HI << 32) |
                                                  (a_lo + (uint32_t)((i0 >> 2) * (TILE_BYTES >> 4) + (((i0 & 3) * UMMA_K * 4) >> 4))),
                                              bdesc, idesc, (jb | u) != 0);
                                    if (j < NKT) {
                                        const int i1 = NKT + j;
                                        umma_tf32(tmem_d,
                                                  ((uint64_t)DESC_HI << 32) |
                                                      (a_lo + (uint32_t)((i1 >> 2) * (TILE_BYTES >> 4) + (((i1 & 3) * UMMA_K * 4) >> 4))),
                                                  bdesc, idesc, 1u);
                                    }
                                }
                            }
                            umma_commit(&S.empty_bar[s]);
                            }
                            if (++s == nstage) { s = 0; ph ^= 1; }
                        }
                    } else {
                        uint32_t acc = 0;
                        int m = 0;
                        for (int jb = 0; jb < nbox; ++jb) {
                            const int m_end = S.prog_start[jb + 1];
                            const uint32_t b_lo = ring_lo + (uint32_t)s * (TILE_BYTES >> 4);
                            mbar_wait(&S.full_bar[s], ph);
                            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                            if (elect_one_sync()) {
                                for (int mm = m; mm < m_end; ++mm) {
                                    const uint2 e = S.prog[mm];
                                    const uint64_t adesc = ((uint64_t)DESC_HI << 32) | e.x;
                                    const uint64_t bdesc = ((uint64_t)DESC_HI << 32) | (b_lo + e.y);
                                    umma_tf32(tmem_d, adesc, bdesc, idesc, (mm | (int)acc) != 0);
                                }
                                umma_commit(&S.empty_bar[s]);
                            }
                            m = m_end;
                            acc = 1;
                            if (++s == nstage) { s = 0; ph ^= 1; }
                        }
                    }
                    if (elect_one_sync()) umma_commit(&S.tmem_full_bar[buf]);
                }
            }
            if (lane == 0 && tt > 0) atomicAdd(tiles_issued, (int32_t)tt); // measurement: tiles this CTA contracted
        }
    } else {
        // ---------------- epilogue warps 2..9: thread <-> (query row, column half).  The warps run decoupled: they
        // synchronise with the MMA warp only (TMEM full / empty barriers), so a warp that meets many candidates in one
        // tile does not hold up the other seven.  Column metadata is the same for all rows: it is read with warp-uniform
        // loads straight from global memory (L1 hits after a prefetch one tile ahead).
        const int q = warp & 3;                 // TMEM lane quadrant this warp may read
        const int half = (warp - 2) >> 2;       // 0: columns [0,64) of a tile, 1: columns [64,128)
        const int row = q * 32 + lane;          // TMEM lane == row within the block
        const int et = threadIdx.x - 64;        // 0..255 index among the epilogue threads
        TopList<KR> L;
        int64_t tt = 0;
        // the thread's candidate stack through explicit shared-space accesses (S is reached through a generic pointer: the
        // compiler emitted 64-bit generic ST.E / LD.E with an IMAD.WIDE each)
        const uint32_t cand_base = smem_u32(&S.cand_val[0][et]);
        for (int it = item_begin; it < item_end; ++it) {
            const int4 item = items[it];
            const int cur_bin = item.y;
            const int64_t gid = (int64_t)item.x * BM + row;
            const int64_t gr = mode ? (int64_t)pair_row[gid] : gid; // the query row this thread works for
            const bool rvalid = gr >= 0 && gr < nrows;
            const int p = rvalid ? pos[row_point[gr]] : INT32_MIN + 1;
            // admission threshold and query term |a_q - m_c|^2 of (this query, this bin): see threshold_kernel
            const float t0 = rvalid ? t0_tab[(int64_t)cur_bin * ldt + gr] : -INFINITY;
            const float nr = rvalid ? tq_tab[(int64_t)cur_bin * ldt + gr] : 0.f;
            L.reset();
            // rows are ordered by guessed bin, so in the "side" bins of a row block only a few rows survive the pruning:
            // a warp none of whose 32 rows admits anything (t0 = -inf) only hands the accumulator buffers back
            const bool wskip = __all_sync(CHB_FULL, !(t0 > -INFINITY));
            for (int t = item.z; t < item.z + item.w; ++t) {
                const int buf = (int)(tt & 1);
                const uint32_t tph = (uint32_t)((tt >> 1) & 1);
                ++tt;
                if (wskip) {
                    mbar_wait(&S.tmem_full_bar[buf], tph);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&S.tmem_empty_bar[buf]);
                    continue;
                }
                if (lane < 6 && (t + 1 < item.z + item.w || it + 1 < item_end)) {
                    // next tile's metadata -> L1: three arrays, two 128-byte lines each
                    const int tn = t + 1 < item.z + item.w ? t + 1 : items[it + 1].z;
                    const int64_t e = (int64_t)tn * BN + half * 64 + (lane & 1) * 32;
                    const void *pf = lane < 2 ? (const void *)(col_nrm + e) : (lane < 4 ? (const void *)(col_a + e) : (const void *)(col_b + e));
                    asm volatile("prefetch.global.L1 [%0];" ::"l"(pf));
                }
                const int64_t e0 = (int64_t)t * BN + half * 64;
                const float4 *mn = reinterpret_cast<const float4 *>(col_nrm + e0);
                const int4 *ma = reinterpret_cast<const int4 *>(col_a + e0);
                const int4 *mb = reinterpret_cast<const int4 *>(col_b + e0);
                const int32_t *tile_pt = col_pt + e0;
                mbar_wait(&S.tmem_full_bar[buf], tph);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                // the thread's 64 accumulator columns in one TMEM read; the buffer goes back to the MMA warp right away
                uint32_t v[64];
                {
                    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BN + half * 64);
                    asm volatile("tcgen05.ld.sync.aligned.32x32b.x64.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, %48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];"
                                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31]), "=r"(v[32]), "=r"(v[33]), "=r"(v[34]), "=r"(v[35]), "=r"(v[36]), "=r"(v[37]), "=r"(v[38]), "=r"(v[39]), "=r"(v[40]), "=r"(v[41]), "=r"(v[42]), "=r"(v[43]), "=r"(v[44]), "=r"(v[45]), "=r"(v[46]), "=r"(v[47]), "=r"(v[48]), "=r"(v[49]), "=r"(v[50]), "=r"(v[51]), "=r"(v[52]), "=r"(v[53]), "=r"(v[54]), "=r"(v[55]), "=r"(v[56]), "=r"(v[57]), "=r"(v[58]), "=r"(v[59]), "=r"(v[60]), "=r"(v[61]), "=r"(v[62]), "=r"(v[63])
                                 : "r"(taddr));
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&S.tmem_empty_bar[buf]);
                }
                // Screen the 64 columns four at a time; survivors go onto the thread's candidate stack (value in shared
                // memory, column in a bit mask).  The stacks are drained -- at ONE place in the code, the insertion is long
                // and the instruction cache small -- when one of them could overflow in the next group, and after the tile.
                int ncand = 0;
                unsigned cm_lo = 0, cm_hi = 0;
                int g = 0;
#define SCREEN_STEP(G)                                                                                              \
    case G: {                                                                                                       \
        const float thr = fminf(L.key[KR - 1], t0);                                                                 \
        const float4 n4 = __ldg(mn + G);                                                                            \
        const int4 a4 = __ldg(ma + G);                                                                              \
        const int4 b4 = __ldg(mb + G);                                                                              \
        const float nn[4] = {n4.x, n4.y, n4.z, n4.w};                                                               \
        const int aa[4] = {a4.x, a4.y, a4.z, a4.w};                                                                 \
        const int bb[4] = {b4.x, b4.y, b4.z, b4.w};                                                                 \
        _Pragma("unroll") for (int u = 0; u < 4; ++u) {                                                             \
            const float av = fmaf(-2.f, __uint_as_float(v[4 * G + u]), nr + nn[u]);                                 \
            if (((p > aa[u]) || (p < bb[u])) && (av <= thr)) {                                                      \
                st_shared_f32(cand_base + (uint32_t)ncand * (EPI_THREADS * 4), av);                                 \
                if (G < 8) cm_lo |= 1u << ((4 * G + u) & 31);                                                       \
                else cm_hi |= 1u << ((4 * G + u) & 31);                                                             \
                ++ncand;                                                                                            \
            }                                                                                                       \
        }                                                                                                           \
        if (G < 15 && __any_sync(CHB_FULL, ncand > NC - 4)) {                                                       \
            g = G + 1;                                                                                              \
            break;                                                                                                  \
        }                                                                                                           \
    }
                while (true) {
                    switch (g) {
                    SCREEN_STEP(0)
                    SCREEN_STEP(1)
                    SCREEN_STEP(2)
                    SCREEN_STEP(3)
                    SCREEN_STEP(4)
                    SCREEN_STEP(5)
                    SCREEN_STEP(6)
                    SCREEN_STEP(7)
                    SCREEN_STEP(8)
                    SCREEN_STEP(9)
                    SCREEN_STEP(10)
                    SCREEN_STEP(11)
                    SCREEN_STEP(12)
                    SCREEN_STEP(13)
                    SCREEN_STEP(14)
                    SCREEN_STEP(15)
                        g = 16;
                    }
                    while (__any_sync(CHB_FULL, ncand > 0)) {
                        if (ncand > 0) {
                            --ncand;
                            int col;
                            if (cm_hi) { col = 63 - __clz(cm_hi); cm_hi &= ~(1u << (col - 32)); }
                            else { col = 31 - __clz(cm_lo); cm_lo &= ~(1u << col); }
                            const float av = ld_shared_f32(cand_base + (uint32_t)ncand * (EPI_THREADS * 4));
                            if (av < L.key[KR - 1]) L.insert(av, __ldg(tile_pt + col));
                        }
                    }
                    if (g >= 16) break;
                }
#undef SCREEN_STEP
            }
            if (rvalid && !wskip) { // the item's (half-)list is complete (pruned rows' lists are never read)
                // compacted rounds: one list slot per compact pair id (what this thread's accumulator row is); otherwise per (row, bin)
                const int64_t lslot = mode ? gid : gr * C + cur_bin;
                float4 *ok = reinterpret_cast<float4 *>(cand_key + (lslot * 2 + half) * KR);
                int4 *oi = reinterpret_cast<int4 *>(cand_idx + (lslot * 2 + half) * KR);
#pragma unroll
                for (int s = 0; s < KR; s += 4) {
                    ok[s >> 2] = make_float4(L.key[s], L.key[s + 1], L.key[s + 2], L.key[s + 3]);
                    oi[s >> 2] = make_int4(L.idx[s], L.idx[s + 1], L.idx[s + 2], L.idx[s + 3]);
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 2) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS));
    }
}

// ---------------------------------------------------------------------------------------------------------
// admission thresholds.  The k cached neighbours of (query, bin) from the previous round bound this round's k-th
// smallest key as long as all of them are still visible members of the bin: the re-rank stores ub = (largest key of
// the chosen set) + (that round's slack) >= every member's true squared distance; with this round's slack E every
// re-evaluated member key is <= ub + E, so the k-th smallest key a_k of this round is too, and everything the re-rank
// may need (keys <= a_k + 2E) lies below T0 = ub + 3E.
// Columns above T0 are skipped by the fused kernel without touching the per-thread lists.  T0 = +inf when there is no
// usable cache (first round, fewer than k members, a member left the bin, exact-path fallback row).
// ---------------------------------------------------------------------------------------------------------
// THR_ROWS rows per thread: 4 (16-byte loads of the per-row tables, 16-byte stores of the pruned thresholds) when the pair
// table is large and nearly everything is pruned -- the kernel is then a stream over 8 bytes per pair; 1 when it is small and
// the surviving pairs' work (serial per thread) sets the time
constexpr int THR_BINS = 4;
template <int THR_ROWS>
__global__ void __launch_bounds__(256) threshold_kernel(const int32_t *__restrict__ knn_idx, const int32_t *__restrict__ knn_cnt, const float *__restrict__ thr,
                                 const int32_t *__restrict__ row_point, const int32_t *__restrict__ row_slot,
                                 const int32_t *__restrict__ pos, const int32_t *__restrict__ tent, const int32_t *__restrict__ old,
                                 const float *__restrict__ nrm, const unsigned int *__restrict__ nrm_max_bits,
                                 const float *__restrict__ ym2, const float *__restrict__ tcmax, const float *__restrict__ tq_tab,
                                 const float *__restrict__ ub_row, const float *__restrict__ sq_row,
                                 const float *__restrict__ ubk2_row, const int32_t *__restrict__ row_guess, double eps_rel, int64_t nown,
                                 int32_t C, int32_t k, int32_t prune, int64_t ldt, float *__restrict__ t0_tab, float *__restrict__ slack_tab,
                                 int32_t *__restrict__ row_nb, int32_t *__restrict__ row_bins, int32_t *__restrict__ bin_surv,
                                 uint8_t *__restrict__ skip, int32_t *__restrict__ row_pid)
{
    chb_pdl_enter();
    // grid: x = chunks of 1024 rows (eight 128-row blocks of the fused kernel; a thread takes 4 consecutive rows, a warp one
    // 128-row block), y = bin.  Besides the per-pair tables the block leaves skip[row block][bin] = "every row of the block
    // pruned the bin": the (row block, bin) work items of the uncompacted path, without a second pass over the thresholds.
    // THR_ROWS == 4 (large pair tables): a thread also walks THR_BINS consecutive bins -- the per-row bounds are read once for
    // them and the bins' query terms are all in flight before the first is used (the kernel is a stream over 8 B per pair)
    constexpr int NBIN = THR_ROWS == 4 ? THR_BINS : 1;
    const int lane = threadIdx.x & 31;
    const int64_t r0 = ((int64_t)blockIdx.x * 256 + threadIdx.x) * THR_ROWS; // first row (rows = owned slots ordered by guessed bin)
    float4 tq4s[NBIN], ub4 = make_float4(0.f, 0.f, 0.f, 0.f), sq4 = ub4;
    if (THR_ROWS == 4 && r0 < nown) {
        ub4 = *reinterpret_cast<const float4 *>(ub_row + r0);
        sq4 = *reinterpret_cast<const float4 *>(sq_row + r0);
#pragma unroll
        for (int cb = 0; cb < NBIN; ++cb) {
            const int cc = blockIdx.y * NBIN + cb;
            tq4s[cb] = cc < C ? *reinterpret_cast<const float4 *>(tq_tab + (int64_t)cc * ldt + r0) : ub4;
        }
    }
#pragma unroll
    for (int cb = 0; cb < NBIN; ++cb) {
    const int c = blockIdx.y * NBIN + cb;
    if (c >= C) break; // (uniform over the block)
    bool any_alive = false;
    if (r0 < nown) { // ldt is a multiple of 128 and the tables are allocated up to it: whole float4s may be touched
        float tqv[4], ubv[4], sqv[4];
        if (THR_ROWS == 4) {
            const float4 tq4 = tq4s[cb];
            tqv[0] = tq4.x; tqv[1] = tq4.y; tqv[2] = tq4.z; tqv[3] = tq4.w;
            ubv[0] = ub4.x; ubv[1] = ub4.y; ubv[2] = ub4.z; ubv[3] = ub4.w;
            sqv[0] = sq4.x; sqv[1] = sq4.y; sqv[2] = sq4.z; sqv[3] = sq4.w;
        } else {
            tqv[0] = tq_tab[(int64_t)c * ldt + r0];
            ubv[0] = ub_row[r0];
            sqv[0] = sq_row[r0];
        }
        const float ym = __fmul_ru(__fsqrt_ru(ym2[c]), 1.000001f), amax = __fsqrt_ru(__uint_as_float(*nrm_max_bits));
        float t0v[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
        bool alive[4] = {false, false, false, false};
#pragma unroll
        for (int u = 0; u < THR_ROWS; ++u) {
            alive[u] = r0 + u < nown;
            t0v[u] = -INFINITY;
            // pruning (97-99 % of the pairs end here, so this test is all FP32 and touches nothing per pair but tq and t0):
            // LB = |a_q - m_c| - max|y| > UB, with a margin far above the FP32 roundings of the operands and of this test.
            // Only the CONVEX hull of k members lies inside the ball around m_c: an affine hull is unbounded and may pass close
            // to a query far from every member, so the affine metrics (hull_distance.py:38-87) keep every bin (prune == 0).
            if (alive[u] && prune) {
                const float dq = __fsqrt_rd(tqv[u]), ub = ubv[u];
                const float scale = sqv[u] + amax;
                if (dq * 0.999999f - ym > ub + 1e-5f * (dq + ym + ub) + 4e-6f * scale) alive[u] = false;
            }
            any_alive = any_alive || alive[u];
        }
        if (any_alive) {
#pragma unroll
            for (int u = 0; u < THR_ROWS; ++u) {
                if (!alive[u]) continue;
                const int64_t r = r0 + u;
                const float tq = tqv[u];
                const int js = atomicAdd(&row_nb[r], 1); // surviving bins of this row, in any order
                row_bins[r * C + js] = c;
                // the pair's index among its bin's survivors: pairs_fill_kernel turns it into the compact pair id without a
                // second round of atomics on the C per-bin counters
                row_pid[r * C + js] = atomicAdd(&bin_surv[c], 1);
                const int64_t pair = (int64_t)row_slot[r] * C + c; // caches are indexed by slot
                const int jq = row_point[r];
                const float E = pair_slack(eps_rel, nrm[jq], ym2[c], tcmax[c], tq);
                slack_tab[(int64_t)c * ldt + r] = E;
                float out = INFINITY;
                if (knn_cnt[pair] == k) {
                    const float ub = thr[pair]; // upper bound on the true squared distance of every cached neighbour (re-rank)
                    if (ub < INFINITY) {
                        const int p = pos[jq];
                        bool ok = true;
                        // four neighbours at a time, loads of a kind issued together: index -> position -> label is a chain of
                        // three dependent L2 round trips per neighbour, and this thread is the tail of its CTA
                        for (int s0 = 0; s0 < k; s0 += 4) {
                            int jn[4], ps[4], lt[4], lo_[4];
#pragma unroll
                            for (int u = 0; u < 4; ++u) jn[u] = s0 + u < k ? knn_idx[pair * k + s0 + u] : -1;
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                ps[u] = jn[u] >= 0 ? pos[jn[u]] : 0;
                                lt[u] = jn[u] >= 0 ? tent[jn[u]] : c;
                                lo_[u] = jn[u] >= 0 ? old[jn[u]] : c;
                            }
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                const int lab = ps[u] < p ? lt[u] : (ps[u] > p ? lo_[u] : -1); // algorithm.py:46-60; the query itself never counts
                                ok = ok && (jn[u] < 0 || lab == c);
                            }
                        }
                        // this round's keys of the cached neighbours are <= ub + E, so is the k-th smallest key a_k, and the
                        // re-rank looks no further than a_k + 2E
                        if (ok) out = __fadd_ru(ub, __fmul_ru(3.f, E));
                    }
                }
                // no usable cache: in the query's guessed bin the k-th nearest SEED bounds the k-th smallest squared distance
                if (out == INFINITY && c == row_guess[r] && ubk2_row[r] < INFINITY) out = __fadd_ru(ubk2_row[r], __fmul_ru(3.f, E));
                t0v[u] = out;
            }
        }
        // rows beyond nown inside the last float4 hold -inf as well (never read)
        if (THR_ROWS == 4) *reinterpret_cast<float4 *>(t0_tab + (int64_t)c * ldt + r0) = make_float4(t0v[0], t0v[1], t0v[2], t0v[3]);
        else t0_tab[(int64_t)c * ldt + r0] = t0v[0];
    }
    if (THR_ROWS == 4) {
        // a warp covers exactly one 128-row block
        const bool warp_alive = __any_sync(CHB_FULL, any_alive);
        if (lane == 0) {
            const int64_t rb = ((int64_t)blockIdx.x * 256 + threadIdx.x) * THR_ROWS / BM;
            if (rb * BM < nown) skip[rb * C + c] = warp_alive ? 0 : 1;
        }
    } else {
        // 256 threads = two 128-row blocks
        __shared__ int s_alive[2];
        if (threadIdx.x < 2) s_alive[threadIdx.x] = 0;
        __syncthreads();
        if (any_alive) s_alive[threadIdx.x >> 7] = 1;
        __syncthreads();
        if ((threadIdx.x & 127) == 0) {
            const int64_t rb = (int64_t)blockIdx.x * 2 + (threadIdx.x >> 7);
            if (rb * BM < nown) skip[rb * C + c] = s_alive[threadIdx.x >> 7] ? 0 : 1;
        }
    }
    } // bins of this thread
}

// algorithm.py:47-48,57-58,60 over the surviving bins of each query: strict '<' so the lowest bin wins ties; a query
// always keeps its guessed bin, so there is a finite distance whenever that bin has a visible member
__global__ void argmin_rows_kernel(const int32_t *__restrict__ own_pos, int64_t cnt, const int32_t *__restrict__ perm_pt,
                                   const int32_t *__restrict__ qslot, int64_t u0, const int32_t *__restrict__ slot_row,
                                   const int32_t *__restrict__ row_nb, const int32_t *__restrict__ row_bins,
                                   const double *__restrict__ pair_dist, int32_t C, const int32_t *__restrict__ old_label,
                                   int64_t lo, int64_t hi, int32_t *__restrict__ tent)
{
    chb_pdl_enter();
    const int lane = threadIdx.x & 31;
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (w >= cnt) return;
    const int p = own_pos[w];
    if (p < lo || p >= hi) return; // outside this round's window (own_pos may list every owned position)
    const int j = perm_pt[p];
    const int64_t sl = (int64_t)qslot[j] - u0;
    const int64_t r = slot_row[sl];
    const int nb = row_nb[r];
    double best = INFINITY;
    int bc = INT32_MAX;
    for (int i = lane; i < nb; i += 32) {
        const int c = row_bins[r * C + i];
        const double v = pair_dist[sl * C + c];
        if (v < best || (v == best && c < bc)) { best = v; bc = c; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(CHB_FULL, best, o);
        const int oc = __shfl_xor_sync(CHB_FULL, bc, o);
        if (ov < best || (ov == best && oc < bc)) { best = ov; bc = oc; }
    }
    if (lane == 0) tent[p - lo] = (best < INFINITY) ? bc : old_label[j];
}

// ---------------------------------------------------------------------------------------------------------
// re-rank: candidates -> exact neighbour sets, dirty detection, QP work list
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double exact_distance_g(const double *__restrict__ xq_s, const double *__restrict__ xi, int d)
{
    double acc = 0.0;
    const int d8 = d & ~7;
    double v[8];
    if (d8 > 0) {
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = xi[u];
    }
    for (int t = 0; t < d8; t += 8) {
        double sq[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const double df = __dsub_rn(xq_s[t + u], v[u]);
            sq[u] = __dmul_rn(df, df);
        }
        if (t + 8 < d8) {
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = xi[t + 8 + u];
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) acc = __dadd_rn(acc, sq[u]);
    }
    for (int t = d8; t < d; ++t) {
        const double df = __dsub_rn(xq_s[t], xi[t]);
        acc = __dadd_rn(acc, __dmul_rn(df, df));
    }
    return __dsqrt_rn(acc);
}

// One warp per owned query.  A group of G lanes (G = 16 when the two half-lists of KR = 8 fit, else 32) handles
// one (query, bin) pair: lane s < 2*KR of the group holds one kept candidate.  Everything is predicated rather than
// branched so that the groups of a warp stay convergent for the shuffles; loops run over the set bits of the
// candidate masks (with admission thresholds most lists hold few more than k entries).
// Bins that never received a flush (no columns at all) are recognised through bin_cnt.
template <int G>
__global__ void __launch_bounds__(256) rerank_kernel(int64_t nrows, const float *__restrict__ cand_key, const int32_t *__restrict__ cand_idx, int KR,
                                                     const int32_t *__restrict__ bin_cnt, const double *__restrict__ X, int32_t ldx,
                                                     int32_t d, const int32_t *__restrict__ row_point,
                                                     const int32_t *__restrict__ row_slot,
                                                     const float *__restrict__ slack_tab, int32_t C,
                                                     int32_t k, int32_t *__restrict__ knn_idx, int32_t *__restrict__ knn_cnt,
                                                     int2 *__restrict__ work, int32_t *__restrict__ work_count,
                                                     int2 *__restrict__ fb_pairs, int32_t fb_cap, int32_t *__restrict__ fb_count,
                                                     const float *__restrict__ t0_tab, int64_t ldt, float *__restrict__ thr_out,
                                                     const int32_t *__restrict__ row_nb, const int32_t *__restrict__ row_bins,
                                                     const int32_t *__restrict__ row_pid, const int32_t *__restrict__ mode_p)
{
    chb_pdl_enter();
    const int mode = *mode_p; // 1: the fused kernel worked on compact (row, bin) pairs and filed the lists under their ids
    if (mode == 2) return;    // refused round (pairs_plan_kernel): there are no lists
    constexpr int NG = 32 / G;
    constexpr unsigned GM = G == 32 ? 0xffffffffu : ((1u << (G & 31)) - 1u);
    const int lane = threadIdx.x & 31;
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; // one warp per row: candidate lists, thresholds and
    if (r >= nrows) return;                                                   // slacks are per row ...
    const int64_t sl = row_slot[r];            // ... neighbour caches, hull distances and the work list per owned slot
    const int gl = lane & (G - 1), gsh = lane & ~(G - 1);
    const int jq = row_point[r];
    const double *xq_s = X + (int64_t)jq * ldx; // query row, read only for the (rare) exact evaluations
    const int K2 = 2 * KR;

    // only the bins that survived the pruning bounds (threshold_kernel lists them per row; pruned pairs were settled there)
    const int nb = row_nb[r];
    for (int jb = 0; jb < nb; jb += NG) {
        const int j = jb + lane / G;
        const bool act = j < nb;
        const int c = act ? row_bins[r * C + j] : 0;
        const int64_t pair = sl * C + c;
        const int64_t rpair = (act && mode) ? (int64_t)row_pid[r * C + j] : r * C + c;
        const float t0v = act ? t0_tab[(int64_t)c * ldt + r] : INFINITY;
        const int mo = act ? knn_cnt[pair] : 0;
        float ka = INFINITY;
        int ki = INT32_MAX;
        if (act && bin_cnt[c] > 0 && gl < K2) {
            ka = cand_key[rpair * K2 + gl];
            ki = cand_idx[rpair * K2 + gl];
        }
        const float E = act ? slack_tab[(int64_t)c * ldt + r] : 0.f; // |key - d^2| <= E for every column of this bin
        const float slack2 = __fmul_ru(2.f, E);
        const bool valid = ka < INFINITY; // +inf = empty slot
        const unsigned vm = (__ballot_sync(CHB_FULL, valid) >> gsh) & GM;
        const int nc = __popc(vm);
        const int m = nc < k ? nc : k; // |bin| <= k: all members (distance_matrix.py:58-59)
        const bool big = nc > k;
        // rank of every candidate by (key, index) among the valid ones, and the set of group lanes holding a smaller index
        // (for the canonical order of the chosen set below).  Full lists (no admission thresholds yet: first round): all G
        // lanes are visited, straight-line -- an empty slot holds (+inf, INT32_MAX) and never counts against a valid one, and
        // 2 x G independent shuffles pipeline where a walk over the set bits of `vm` is a serial chain of dependent shuffles
        int rnk = 0;
        unsigned lt_idx = 0; // bit t: group lane t holds a point index below this lane's
        const int niter = __reduce_max_sync(CHB_FULL, nc); // longest list among the warp's groups
        if (2 * niter > G) {
#pragma unroll
            for (int t = 0; t < G; ++t) {
                const float ok = __shfl_sync(CHB_FULL, ka, t, G);
                const int oi = __shfl_sync(CHB_FULL, ki, t, G);
                rnk += (ok < ka || (ok == ka && oi < ki)) ? 1 : 0;
                lt_idx |= (oi < ki ? 1u : 0u) << t;
            }
        } else {
            // short lists (admission thresholds at work: k + 2 candidates or so): visit the occupied slots only -- at 1M
            // contigs the kernel is bound by the shuffle unit, and 2 x G shuffles per pair cost 60 % more than this walk
            unsigned mm = vm;
            for (int it = 0; it < niter; ++it) {
                const bool had = mm != 0;
                const int t = had ? __ffs(mm) - 1 : 0;
                mm &= mm - 1;
                const float ok = __shfl_sync(CHB_FULL, ka, t, G);
                const int oi = __shfl_sync(CHB_FULL, ki, t, G);
                if (had) {
                    rnk += (ok < ka || (ok == ka && oi < ki)) ? 1 : 0;
                    lt_idx |= (oi < ki ? 1u : 0u) << t;
                }
            }
        }
        const unsigned bk = (__ballot_sync(CHB_FULL, valid && rnk == k - 1) >> gsh) & GM;
        const unsigned bk1 = (__ballot_sync(CHB_FULL, valid && rnk == k) >> gsh) & GM;
        const float a_k = __shfl_sync(CHB_FULL, ka, bk ? __ffs(bk) - 1 : 0, G);    // k-th smallest key   (big only)
        const float a_k1 = __shfl_sync(CHB_FULL, ka, bk1 ? __ffs(bk1) - 1 : 0, G); // (k+1)-th            (big only)
        const float hi = __fadd_ru(a_k, slack2);
        const bool could = valid && ka <= hi;                      // may belong to the exact top-k
        const bool sure = valid && (__fadd_ru(ka, slack2) < a_k1); // certainly belongs to it
        const unsigned cm = (__ballot_sync(CHB_FULL, could) >> gsh) & GM;
        const unsigned sm = (__ballot_sync(CHB_FULL, sure) >> gsh) & GM;
        const int nsure = __popc(sm);
        bool ovf = false; // the kept lists may be incomplete for this pair: it is redone exactly (exact_pairs_kernel)
        if (big) {
            // every key <= hi must have been admitted by the fused kernel's threshold (holds by construction of T0), and
            // a half-list that is full and entirely inside the slack may have dropped a closer point
            const unsigned lo_half = (1u << KR) - 1u;
            if (hi > t0v || __popc(cm & lo_half) == KR || __popc(cm >> KR) == KR) ovf = true;
        } else if (k >= KR) {
            // "at most k candidates" only means "the bin has at most k visible members" if no half-list is full: with k >= KR
            // a full half-list may have dropped members (k < KR: nc <= k < KR, no half-list can be full)
            const unsigned lo_half = (1u << KR) - 1u;
            if (__popc(vm & lo_half) == KR || __popc(vm >> KR) == KR) ovf = true;
        }
        // ambiguous candidates: exact scipy-recipe distance, rank by (distance, index)
        const bool amb = big && __popc(cm) != k && could && !sure;
        double de = 0.0;
        if (amb) de = exact_distance_g(xq_s, X + (int64_t)ki * ldx, d);
        const unsigned am = (__ballot_sync(CHB_FULL, amb) >> gsh) & GM;
        int rk = 0;
        {
            unsigned mm = am;
            while (__any_sync(CHB_FULL, mm != 0)) {
                const bool had = mm != 0;
                const int t = had ? __ffs(mm) - 1 : 0;
                mm &= mm - 1;
                const double od = __shfl_sync(CHB_FULL, de, t, G);
                const int oi = __shfl_sync(CHB_FULL, ki, t, G);
                if (had && (od < de || (od == de && oi < ki))) ++rk;
            }
        }
        const bool sel = !big ? valid : (__popc(cm) == k ? could : (sure || (amb && rk < k - nsure)));
        // largest FP32 key of the chosen set: next round's admission threshold derives from it (threshold_kernel)
        float mx = sel ? ka : -INFINITY;
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(CHB_FULL, mx, o));
        // neighbour set, stored in ascending index order (canonical for set comparison)
        const unsigned selm = (__ballot_sync(CHB_FULL, sel) >> gsh) & GM;
        const int srt = __popc(selm & lt_idx); // chosen points with a smaller index
        const bool diff = sel && (mo != m || knn_idx[pair * k + srt] != ki);
        const unsigned dm = (__ballot_sync(CHB_FULL, diff) >> gsh) & GM;
        const bool same = (mo == m) && dm == 0;
        if (act && ovf) {
            if (gl == 0) {
                thr_out[pair] = INFINITY;
                const int w = atomicAdd(fb_count, 1);
                if (w < fb_cap) fb_pairs[w] = make_int2((int)r, c);
            }
        } else if (act) {
            if (gl == 0) thr_out[pair] = (m == k) ? __fadd_ru(mx, E) : INFINITY;
            if (!same) {
                // slots [0, m) come from the selected lanes, slots [m, k) are cleared by the lanes sitting at those positions
                if (sel) knn_idx[pair * k + srt] = ki;
                if (gl >= m && gl < k) knn_idx[pair * k + gl] = -1;
                if (gl == 0) {
                    knn_cnt[pair] = m;
                    const int w = atomicAdd(work_count, 1);
                    work[w] = make_int2((int)sl, c);
                }
            }
        }
    }
}

// Exact redo of the (row, bin) pairs whose kept candidate lists may be incomplete (duplicate contigs: more than KR keys
// inside the slack window).  One CTA per pair walks the bin's column segment of this round, evaluates scipy's exact
// recipe for every visible member and selects the k smallest (distance, index) -- find_nearest_from_cluster
// (distance_matrix.py:47-62) verbatim.  Rare, so simple: per-thread sorted lists, then k block-wide argmin rounds.
template <int KX>
__global__ void __launch_bounds__(128) exact_pairs_kernel(const int2 *__restrict__ fb_pairs, const int32_t *__restrict__ fb_count,
                                                          int32_t fb_cap, const int32_t *__restrict__ seg_off,
                                                          const int32_t *__restrict__ bin_cnt, const int32_t *__restrict__ col_pt,
                                                          const int32_t *__restrict__ col_a, const int32_t *__restrict__ col_b,
                                                          const double *__restrict__ X, int32_t ldx, int32_t d,
                                                          const int32_t *__restrict__ row_point, const int32_t *__restrict__ row_slot,
                                                          const int32_t *__restrict__ pos, int32_t C, int32_t k,
                                                          int32_t *__restrict__ knn_idx, int32_t *__restrict__ knn_cnt,
                                                          int2 *__restrict__ work, int32_t *__restrict__ work_count)
{
    chb_pdl_wait();
    extern __shared__ __align__(16) double xq_s[];
    __shared__ double s_best[4];
    __shared__ int s_bidx[4], s_bthr[4];
    __shared__ int s_sel[KX];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nfb = min(*fb_count, fb_cap);
    for (int f = blockIdx.x; f < nfb; f += gridDim.x) {
        const int r = fb_pairs[f].x, c = fb_pairs[f].y;
        const int jq = row_point[r];
        const int p = pos[jq];
        __syncthreads();
        for (int t = tid; t < d; t += 128) xq_s[t] = X[(int64_t)jq * ldx + t];
        __syncthreads();
        double ld[KX];
        int li[KX];
#pragma unroll
        for (int s = 0; s < KX; ++s) { ld[s] = INFINITY; li[s] = INT32_MAX; }
        const int e0 = seg_off[c], e1 = e0 + bin_cnt[c];
        for (int e = e0 + tid; e < e1; e += 128) {
            const int pt = col_pt[e];
            if (pt < 0 || !((p > col_a[e]) || (p < col_b[e]))) continue;
            double dv = exact_distance_g(xq_s, X + (int64_t)pt * ldx, d);
            int iv = pt;
#pragma unroll
            for (int s = 0; s < KX; ++s) { // sorted insertion by (distance, index)
                const bool lt = dv < ld[s] || (dv == ld[s] && iv < li[s]);
                const double td = lt ? ld[s] : dv;
                const int ti = lt ? li[s] : iv;
                ld[s] = lt ? dv : ld[s];
                li[s] = lt ? iv : li[s];
                dv = td;
                iv = ti;
            }
        }
        int m = 0;
        for (int round = 0; round < k; ++round) {
            // block-wide argmin over the heads of the per-thread lists
            double bd = ld[0];
            int bi = li[0], bt = tid;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double od = __shfl_xor_sync(CHB_FULL, bd, o);
                const int oi = __shfl_xor_sync(CHB_FULL, bi, o);
                const int ot = __shfl_xor_sync(CHB_FULL, bt, o);
                if (od < bd || (od == bd && oi < bi)) { bd = od; bi = oi; bt = ot; }
            }
            if (lane == 0) { s_best[warp] = bd; s_bidx[warp] = bi; s_bthr[warp] = bt; }
            __syncthreads();
            int win = 0;
            for (int w = 1; w < 4; ++w)
                if (s_best[w] < s_best[win] || (s_best[w] == s_best[win] && s_bidx[w] < s_bidx[win])) win = w;
            const bool any = s_best[win] < INFINITY;
            const int wthr = s_bthr[win], widx = s_bidx[win];
            __syncthreads();
            if (!any) break;
            if (tid == 0) s_sel[m] = widx;
            ++m;
            if (tid == wthr) { // pop the head
#pragma unroll
                for (int s = 0; s + 1 < KX; ++s) { ld[s] = ld[s + 1]; li[s] = li[s + 1]; }
                ld[KX - 1] = INFINITY;
                li[KX - 1] = INT32_MAX;
            }
        }
        __syncthreads();
        if (tid == 0) {
            // ascending index order (canonical), compare with the cache, list for the QP kernel if the set changed
            for (int a = 1; a < m; ++a) {
                const int v = s_sel[a];
                int b = a - 1;
                while (b >= 0 && s_sel[b] > v) { s_sel[b + 1] = s_sel[b]; --b; }
                s_sel[b + 1] = v;
            }
            const int64_t pair = (int64_t)row_slot[r] * C + c;
            bool same = knn_cnt[pair] == m;
            for (int a = 0; same && a < m; ++a) same = knn_idx[pair * k + a] == s_sel[a];
            if (!same) {
                for (int a = 0; a < k; ++a) knn_idx[pair * k + a] = a < m ? s_sel[a] : -1;
                knn_cnt[pair] = m;
                work[atomicAdd(work_count, 1)] = make_int2(row_slot[r], c);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// Large neighbour counts (k > FUSED_KMAX: the 16-entry register half-lists of the fused kernel overflow for most pairs): exact selection for
// EVERY surviving (row, bin) pair.  With one pair per CTA every member row of the bin travels L2 -> SM once per pair and the
// L2 fabric is the bound; here the surviving pairs are regrouped per bin and XS_G queries of one bin share every member row
// they read (XS_G x fewer bytes, XS_G independent FP64 chains per thread), which leaves the FP64 pipe as the bound
// (|bin| x d x 3 operations per pair: scipy's recipe admits no FMA).
//   distances : a thread evaluates scipy's recipe for one member against the XS_G queries; (distance bits, index) composites of
//               the members visible to a query are appended to that query's shared-memory array -- non-negative doubles order
//               like their bit patterns and the index makes every composite unique;
//   selection : warp w owns query w.  tau = k-th smallest of 64 strided minima: at least k members are <= tau and, for
//               k << |bin|, few more; those are compacted and ranked by counting; ranks < k are find_nearest_from_cluster's
//               answer (distance_matrix.py:47-62, ties resolved by index as everywhere in this library).
// Bins larger than one pass are walked in chunks: the k kept so far stay at the front of the query's array.
constexpr int XS_G = 8, XS_THREADS = 32 * XS_G, XS_CHUNK = 4 * XS_THREADS, XS_KEEP = 32, XS_CAP = XS_CHUNK + XS_KEEP, XS_CAND = 128;
// largest k that goes through the fused tensor-core kernel's two 16-entry half-lists: the k + 1 smallest keys must all be kept,
// which holds unless one 64-column half holds 16 or more of them (the re-rank detects that and has the pair redone exactly).
// The members of a bin fall into the halves at random, so up to k = 24 that is the exception (a few per cent of the pairs at
// k = 20, about one in six at k = 24); beyond it is the rule and the exact selection below takes every pair.
constexpr int FUSED_KMAX = 24;
// XS_KEEP = the largest k the fused mode accepts (chb_fused_supported)

__device__ __forceinline__ bool comp_lt(unsigned long long ka, int ia, unsigned long long kb, int ib)
{
    return ka < kb || (ka == kb && ia < ib);
}

inline size_t exact_group_smem(int d)
{
    return (size_t)XS_G * (sizeof(double) * (size_t)((d + 1) & ~1) + (size_t)(XS_CAP + 64 + XS_CAND + XS_KEEP) * 12);
}

// offsets of the per-bin slot ranges, each rounded up to a multiple of XS_G (so that a group never mixes bins)
__global__ void xs_plan_kernel(const int32_t *__restrict__ bin_surv, int32_t C, int32_t *__restrict__ xs_off, int32_t *__restrict__ npairs)
{
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    int off = 0, np = 0;
    for (int c = 0; c < C; ++c) {
        xs_off[c] = off;
        const int s = bin_surv[c];
        np += s;
        off += (s + XS_G - 1) / XS_G * XS_G;
    }
    xs_off[C] = off;
    *npairs = np; // chb_round_commit reports an error if this exceeds the pair capacity
}

// the pairs the re-rank could not settle (16 < k <= FUSED_KMAX: overflowing half-lists are common), regrouped per bin so
// that exact_group_kernel can share each member row among eight of them
__global__ void fb_hist_kernel(const int2 *__restrict__ fb_pairs, const int32_t *__restrict__ fb_count, int32_t fb_cap,
                               int32_t *__restrict__ bin_cnt)
{
    const int n = min(*fb_count, fb_cap);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) atomicAdd(&bin_cnt[fb_pairs[i].y], 1);
}
__global__ void fb_scatter_kernel(const int2 *__restrict__ fb_pairs, const int32_t *__restrict__ fb_count, int32_t fb_cap,
                                  const int32_t *__restrict__ xs_off, int32_t *__restrict__ xs_cur, int2 *__restrict__ slots,
                                  int32_t cap_slots)
{
    const int n = min(*fb_count, fb_cap);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int2 pr = fb_pairs[i];
        const int sidx = xs_off[pr.y] + atomicAdd(&xs_cur[pr.y], 1);
        if (sidx < cap_slots) slots[sidx] = pr;
    }
}

__global__ void xs_fill_kernel(const int32_t *__restrict__ row_nb, const int32_t *__restrict__ row_bins, int64_t nown, int32_t C,
                               const int32_t *__restrict__ xs_off, int32_t *__restrict__ xs_cur, int2 *__restrict__ slots, int32_t cap_slots)
{
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nown) return;
    const int nb = row_nb[r];
    for (int j = 0; j < nb; ++j) {
        const int c = row_bins[r * C + j];
        const int s = xs_off[c] + atomicAdd(&xs_cur[c], 1);
        if (s < cap_slots) slots[s] = make_int2((int)r, c);
    }
}

// scipy's recipe (sequential sum of rounded squares, no FMA, then sqrt) for TWO member rows against XS_G query rows: every
// query value read from shared memory (a broadcast load still costs its 16 bytes x 32 lanes of return bandwidth) feeds two
// chains -- with one member per thread the kernel sat on the shared-memory pipe at 40 % FP64 utilisation (ncu)
__device__ __forceinline__ void group_distances2(const double *__restrict__ xq_s, int dpad, const double *__restrict__ xa,
                                                 const double *__restrict__ xb, int d, double (&accA)[XS_G], double (&accB)[XS_G])
{
#pragma unroll
    for (int g = 0; g < XS_G; ++g) accA[g] = accB[g] = 0.0;
    const int d4 = d & ~3;
    double va[4], vb[4];
    if (d4 > 0) {
#pragma unroll
        for (int u = 0; u < 4; ++u) { va[u] = xa[u]; vb[u] = xb[u]; }
    }
    for (int t = 0; t < d4; t += 4) {
        double wa[4], wb[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) { wa[u] = va[u]; wb[u] = vb[u]; }
        if (t + 4 < d4) {
#pragma unroll
            for (int u = 0; u < 4; ++u) { va[u] = xa[t + 4 + u]; vb[u] = xb[t + 4 + u]; }
        }
        // the query values of group g + 1 are fetched from shared memory while group g is being consumed
        double qn[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) qn[u] = xq_s[t + u];
#pragma unroll
        for (int g = 0; g < XS_G; ++g) {
            double qc[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) qc[u] = qn[u];
            if (g + 1 < XS_G) {
#pragma unroll
                for (int u = 0; u < 4; ++u) qn[u] = xq_s[(g + 1) * dpad + t + u];
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const double da = __dsub_rn(qc[u], wa[u]);
                const double db = __dsub_rn(qc[u], wb[u]);
                accA[g] = __dadd_rn(accA[g], __dmul_rn(da, da));
                accB[g] = __dadd_rn(accB[g], __dmul_rn(db, db));
            }
        }
    }
    for (int t = d4; t < d; ++t) {
        const double a = xa[t], b = xb[t];
#pragma unroll
        for (int g = 0; g < XS_G; ++g) {
            const double qv = xq_s[g * dpad + t];
            const double da = __dsub_rn(qv, a);
            const double db = __dsub_rn(qv, b);
            accA[g] = __dadd_rn(accA[g], __dmul_rn(da, da));
            accB[g] = __dadd_rn(accB[g], __dmul_rn(db, db));
        }
    }
#pragma unroll
    for (int g = 0; g < XS_G; ++g) { accA[g] = __dsqrt_rn(accA[g]); accB[g] = __dsqrt_rn(accB[g]); }
}

__global__ void __launch_bounds__(XS_THREADS, 1)
    exact_group_kernel(const int2 *__restrict__ slots, const int32_t *__restrict__ xs_off, int32_t cap_slots, const int32_t *__restrict__ seg_off,
                       const int32_t *__restrict__ bin_cnt, const int32_t *__restrict__ col_pt, const int32_t *__restrict__ col_a,
                       const int32_t *__restrict__ col_b, const double *__restrict__ X, int32_t ldx, int32_t d,
                       const int32_t *__restrict__ row_point, const int32_t *__restrict__ row_slot, const int32_t *__restrict__ pos, int32_t C,
                       int32_t k, int32_t *__restrict__ knn_idx, int32_t *__restrict__ knn_cnt, int2 *__restrict__ work,
                       int32_t *__restrict__ work_count)
{
    extern __shared__ __align__(16) unsigned char xs_raw[];
    typedef unsigned long long u64;
    const int dpad = (d + 1) & ~1;
    double *xq_s = reinterpret_cast<double *>(xs_raw); // [XS_G][dpad]
    u64 *key = reinterpret_cast<u64 *>(xq_s + XS_G * dpad); // 8-byte arrays first, then the 4-byte ones; all [XS_G][...]
    u64 *tmk = key + XS_G * XS_CAP;
    u64 *ck = tmk + XS_G * 64;
    u64 *selk = ck + XS_G * XS_CAND;
    int *idx = reinterpret_cast<int *>(selk + XS_G * XS_KEEP);
    int *tmi = idx + XS_G * XS_CAP;
    int *ci = tmi + XS_G * 64;
    int *seli = ci + XS_G * XS_CAND;
    __shared__ int s_n[XS_G], s_row[XS_G], s_p[XS_G], s_ti[XS_G];
    __shared__ u64 s_tk[XS_G];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const u64 KMAX = ~0ull;
    const int total = min(xs_off[C], cap_slots);
    for (int g0 = blockIdx.x * XS_G; g0 < total; g0 += gridDim.x * XS_G) {
        __syncthreads(); // the previous group's warps are done with the shared arrays
        if (tid < XS_G) {
            const int r = slots[g0 + tid].x; // -1: padding at the end of a bin's range
            s_row[tid] = r;
            s_n[tid] = 0;
            s_p[tid] = r >= 0 ? pos[row_point[r]] : 0;
        }
        const int c = slots[g0].y; // the first slot of a group is always a real pair
        __syncthreads();
        for (int i = tid; i < XS_G * dpad; i += XS_THREADS) {
            const int g = i / dpad, t = i - g * dpad;
            const int r = s_row[g];
            xq_s[i] = (r >= 0 && t < d) ? X[(int64_t)row_point[r] * ldx + t] : 0.0;
        }
        const int e0 = seg_off[c], e1 = e0 + bin_cnt[c];
        for (int cs = e0; cs < e1; cs += XS_CHUNK) {
            const int ce = min(cs + XS_CHUNK, e1);
            __syncthreads(); // query rows staged / previous chunk's selection finished
            // ---- distances of this chunk's members against the group's queries
            for (int e = cs + tid; e < ce; e += 2 * XS_THREADS) { // two members per thread and step
                const int e2 = e + XS_THREADS;
                const int pt = col_pt[e], pt2 = e2 < ce ? col_pt[e2] : -1; // -1: padding column
                if (pt < 0 && pt2 < 0) continue;
                const int ca = col_a[e], cb = col_b[e];
                const int ca2 = pt2 >= 0 ? col_a[e2] : 0, cb2 = pt2 >= 0 ? col_b[e2] : 0;
                double acc[XS_G], acc2[XS_G];
                group_distances2(xq_s, dpad, X + (int64_t)(pt >= 0 ? pt : pt2) * ldx, X + (int64_t)(pt2 >= 0 ? pt2 : pt) * ldx, d, acc, acc2);
#pragma unroll
                for (int g = 0; g < XS_G; ++g) {
                    if (s_row[g] < 0) continue;
                    if (pt >= 0 && ((s_p[g] > ca) || (s_p[g] < cb))) { // member visible to this query
                        const int slot = atomicAdd(&s_n[g], 1);
                        key[g * XS_CAP + slot] = (u64)__double_as_longlong(acc[g]);
                        idx[g * XS_CAP + slot] = pt;
                    }
                    if (pt2 >= 0 && ((s_p[g] > ca2) || (s_p[g] < cb2))) {
                        const int slot = atomicAdd(&s_n[g], 1);
                        key[g * XS_CAP + slot] = (u64)__double_as_longlong(acc2[g]);
                        idx[g * XS_CAP + slot] = pt2;
                    }
                }
            }
            __syncthreads();
            // ---- selection: warp w owns query w
            const int N = s_n[w];
            if (s_row[w] >= 0 && N > k) { // N <= k: all members so far (distance_matrix.py:58-59)
                u64 *K = key + w * XS_CAP;
                int *I = idx + w * XS_CAP;
                u64 m0k = KMAX, m1k = KMAX;
                int m0i = INT32_MAX, m1i = INT32_MAX;
                for (int j = lane; j < N; j += 64) {
                    if (comp_lt(K[j], I[j], m0k, m0i)) { m0k = K[j]; m0i = I[j]; }
                    const int j2 = j + 32;
                    if (j2 < N && comp_lt(K[j2], I[j2], m1k, m1i)) { m1k = K[j2]; m1i = I[j2]; }
                }
                tmk[w * 64 + lane] = m0k;
                tmi[w * 64 + lane] = m0i;
                tmk[w * 64 + 32 + lane] = m1k;
                tmi[w * 64 + 32 + lane] = m1i;
                __syncwarp();
                // tau = k-th smallest of the 64 minima (empty strides hold the sentinel; the position breaks their ties)
                int r0 = 0, r1 = 0;
                for (int t = 0; t < 64; ++t) {
                    const u64 ok = tmk[w * 64 + t];
                    const int oi = tmi[w * 64 + t];
                    r0 += (comp_lt(ok, oi, m0k, m0i) || (ok == m0k && oi == m0i && t < lane)) ? 1 : 0;
                    r1 += (comp_lt(ok, oi, m1k, m1i) || (ok == m1k && oi == m1i && t < lane + 32)) ? 1 : 0;
                }
                if (r0 == k - 1) { s_tk[w] = m0k; s_ti[w] = m0i; }
                if (r1 == k - 1) { s_tk[w] = m1k; s_ti[w] = m1i; }
                __syncwarp();
                const u64 tk = s_tk[w];
                const int ti = s_ti[w];
                // members <= tau (at least k of them), compacted in array order
                int M = 0;
                for (int base = 0; base < N; base += 32) {
                    const int j = base + lane;
                    const bool in = j < N && !comp_lt(tk, ti, K[j], I[j]);
                    const unsigned b = __ballot_sync(CHB_FULL, in);
                    if (in) {
                        const int slot = M + __popc(b & ((1u << lane) - 1u));
                        if (slot < XS_CAND) { ck[w * XS_CAND + slot] = K[j]; ci[w * XS_CAND + slot] = I[j]; }
                    }
                    M += __popc(b);
                }
                __syncwarp();
                const bool compact = M <= XS_CAND; // otherwise (a sentinel tau: fewer than k strides saw a member) rank in place
                const u64 *lk = compact ? ck + w * XS_CAND : K;
                const int *li = compact ? ci + w * XS_CAND : I;
                const int L = compact ? M : N;
                for (int j = lane; j < L; j += 32) {
                    const u64 a = lk[j];
                    const int ai = li[j];
                    if (!compact && comp_lt(tk, ti, a, ai)) continue;
                    int rk = 0;
                    for (int t = 0; t < L; ++t) rk += comp_lt(lk[t], li[t], a, ai) ? 1 : 0;
                    if (rk < k) { selk[w * XS_KEEP + rk] = a; seli[w * XS_KEEP + rk] = ai; }
                }
                __syncwarp();
                if (lane < k) { K[lane] = selk[w * XS_KEEP + lane]; I[lane] = seli[w * XS_KEEP + lane]; }
                if (lane == 0) s_n[w] = k;
            }
        }
        __syncthreads();
        // ---- ascending index order (canonical), compare with the cache, list for the QP kernel if the set changed
        if (s_row[w] >= 0) {
            const int r = s_row[w];
            const int m = s_n[w];
            const int *I = idx + w * XS_CAP;
            int *srt = seli + w * XS_KEEP;
            const int my = lane < m ? I[lane] : INT32_MAX;
            int rk = 0;
            for (int t = 0; t < m; ++t) rk += I[t] < my ? 1 : 0;
            __syncwarp();
            if (lane < m) srt[rk] = my;
            __syncwarp();
            const int64_t pair = (int64_t)row_slot[r] * C + c;
            const bool diff = lane < k && knn_idx[pair * k + lane] != (lane < m ? srt[lane] : -1);
            const bool same = knn_cnt[pair] == m && !__any_sync(CHB_FULL, diff);
            if (!same) {
                if (lane < k) knn_idx[pair * k + lane] = lane < m ? srt[lane] : -1;
                if (lane == 0) {
                    knn_cnt[pair] = m;
                    work[atomicAdd(work_count, 1)] = make_int2(row_slot[r], c);
                }
            }
        }
    }
}

typedef CUresult (*encode_fn_t)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
encode_fn_t get_encode_fn()
{
    static encode_fn_t fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<encode_fn_t>(p);
    }
    return fn;
}
int make_map(chb_ctx *ctx, CUtensorMap *map, float *base, int64_t nrows, int32_t Kp)
{
    encode_fn_t enc = get_encode_fn();
    CHB_CHECK(ctx, enc != nullptr, CHB_ECUDA, "cuTensorMapEncodeTiled entry point not available");
    const cuuint64_t gdim[2] = {(cuuint64_t)Kp, (cuuint64_t)nrows};
    const cuuint64_t gstr[1] = {(cuuint64_t)Kp * sizeof(float)};
    const cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)BM};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CHB_CHECK(ctx, r == CUDA_SUCCESS, CHB_ECUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
    return CHB_OK;
}

// dp8 = width of one operand half (d rounded up to 8, or to 32 when streamed), nk = its K=8 steps, nbox = 32-float boxes per
// operand row, Kp2 = floats per operand row, nstage = ring stages (boxes, or 4-box stages when streamed)
struct FusedGeom {
    int dp8, nk, nbox, Kp2, nstage;
    bool stream;
    size_t smem;
};
FusedGeom fused_geom(int d)
{
    FusedGeom g{};
    const int fixed = 1024 + (int)sizeof(SmemTail);
    g.stream = d > DMAX_F;
    if (g.stream) {
        g.dp8 = (d + BK - 1) & ~(BK - 1);
        g.nk = g.dp8 / UMMA_K;
        g.nbox = 2 * g.dp8 / BK;
        g.Kp2 = g.nbox * BK;
        const int stage = WIDE_STAGE_BOXES * (int)TILE_BYTES;
        g.nstage = std::min(8, (SMEM_LIMIT - fixed) / stage);
        g.smem = (size_t)fixed + (size_t)g.nstage * stage;
        return g;
    }
    g.dp8 = (d + 7) & ~7;
    g.nk = g.dp8 / UMMA_K;
    g.nbox = (2 * g.dp8 + BK - 1) / BK;
    g.Kp2 = g.nbox * BK;
    g.nstage = std::min(8, (SMEM_LIMIT - fixed - g.nbox * (int)TILE_BYTES) / (int)TILE_BYTES);
    g.smem = (size_t)fixed + (size_t)(g.nbox + std::max(g.nstage, 0)) * TILE_BYTES;
    return g;
}

template <int KR, int NKT>
int launch_fused(chb_ctx *c, const CUtensorMap &ma, const CUtensorMap &map, const CUtensorMap &mb, int64_t nrows, const FusedGeom &g)
{
    CHB_CUDA(c, cudaFuncSetAttribute(gram_select_kernel<KR, NKT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem));
    const int grid = c->sm_count; // persistent: one CTA per SM, work split by pairs_plan_kernel
    {
        chb_stage_timer t(c, CHB_ST_GRAM);
        CHB_PDL_LAUNCH(c, (gram_select_kernel<KR, NKT>), grid, FUSED_THREADS, g.smem,
            ma, map, mb, c->f_mode, c->f_pair_row, g.nbox, g.nk, g.nstage, c->f_col_pt, c->f_col_a, c->f_col_b, c->f_col_nrm, c->f_tq, c->f_row_pt, c->pos, nrows, c->C,
            c->f_t0, c->f_ldt, c->f_items, c->f_cta_begin, c->f_cand_key, c->f_cand_idx, &c->counters[8]);
    }
    CHB_CUDA(c, cudaGetLastError());
    return CHB_OK;
}

template <int KR>
int dispatch_nk(chb_ctx *c, const CUtensorMap &ma, const CUtensorMap &map, const CUtensorMap &mb, int64_t nrows, const FusedGeom &g)
{
    if (g.stream) return launch_fused<KR, NKT_STREAMED>(c, ma, map, mb, nrows, g);
    const bool generic = getenv("CHB_FUSED_GENERIC") != nullptr; // test aid: force the tabulated MMA sequence
    if (!generic && g.nk == 18) return launch_fused<KR, 18>(c, ma, map, mb, nrows, g);
    if (!generic && g.nk == 19) return launch_fused<KR, 19>(c, ma, map, mb, nrows, g);
    if (!generic && g.nk == 20) return launch_fused<KR, 20>(c, ma, map, mb, nrows, g);
    return launch_fused<KR, 0>(c, ma, map, mb, nrows, g);
}
int dispatch_fused(chb_ctx *c, const CUtensorMap &ma, const CUtensorMap &map, const CUtensorMap &mb, int64_t nrows, const FusedGeom &g,
                   int KR)
{
    return KR == 8 ? dispatch_nk<8>(c, ma, map, mb, nrows, g) : dispatch_nk<16>(c, ma, map, mb, nrows, g);
}

template <typename T>
int reserve(chb_ctx *ctx, T **p, int64_t *cap, int64_t count)
{
    if (*p && *cap >= count) return CHB_OK;
    if (*p) cudaFree(*p);
    *p = nullptr;
    *cap = 0;
    cudaError_t e = cudaMalloc(reinterpret_cast<void **>(p), sizeof(T) * (size_t)std::max<int64_t>(count, 1));
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return chb_fail(ctx, CHB_ENOMEM, "cudaMalloc of %lld bytes failed: %s", (long long)(sizeof(T) * (size_t)count),
                        cudaGetErrorString(e));
    }
    *cap = count;
    return CHB_OK;
}

inline unsigned nblk(int64_t n, int t) { return (unsigned)((n + t - 1) / t); }

} // namespace

// d <= 160: the resident query operand (2 * dp8 floats per row) fits MAX_BOX boxes with at least 3 ring stages left;
// 161 <= d <= 1024: the streamed kernel, 3 stages of 64 KB.  Up to k = 15 the k + 1 candidates the re-rank needs fit a
// 16-entry register half-list of the fused kernel, larger k uses pruning + exact selection only (chb_round_fused).  Whether
// a stage runs on this path is decided by chb_use_fused (api.cu) from the input size as well.
bool chb_fused_supported(const chb_ctx *c)
{
    const FusedGeom g = fused_geom(c->d);
    if (c->k > XS_KEEP || c->d > DMAX_W) return false;
    return g.nstage >= 3 && (g.stream || g.nbox <= MAX_BOX);
}

void chb_fused_free(chb_ctx *c)
{
    if (c->side_stream) cudaStreamSynchronize(c->side_stream);
    c->side_join_pending = false;
    cudaFree(c->f_bin_cnt); cudaFree(c->f_seg_off); cudaFree(c->f_cursor); cudaFree(c->f_tile_bin); cudaFree(c->f_ntiles);
    cudaFree(c->f_col_pt); cudaFree(c->f_col_a); cudaFree(c->f_col_b); cudaFree(c->f_col_nrm); cudaFree(c->f_bperm);
    cudaFree(c->f_cand_key); cudaFree(c->f_cand_idx); cudaFree(c->f_fb_pairs); cudaFree(c->f_xs_slots); cudaFree(c->f_thr); cudaFree(c->f_t0); cudaFree(c->f_a2); cudaFree(c->f_tq); cudaFree(c->f_slack); cudaFree(c->f_ym2);
    cudaFree(c->f_mc); cudaFree(c->f_mc2); cudaFree(c->f_mcnt); cudaFree(c->f_skip); cudaFree(c->f_pair_row); cudaFree(c->f_pair_meta); cudaFree(c->f_ap); cudaFree(c->f_mode); cudaFree(c->f_items); cudaFree(c->f_cta_begin); cudaFree(c->f_row_slot); cudaFree(c->f_row_pt);
    cudaFree(c->f_ub); cudaFree(c->f_ubk2); cudaFree(c->f_row_guess); cudaFree(c->f_rhist); cudaFree(c->f_mcT); cudaFree(c->f_guess_all); cudaFree(c->f_tqs);
    c->f_tqs = nullptr;
    c->f_cap_tqs = 0; cudaFree(c->f_seedT); cudaFree(c->f_row_nb); cudaFree(c->f_row_bins); cudaFree(c->f_row_pid); cudaFree(c->f_slot_row); cudaFree(c->f_sq_row);
    c->f_slot_row = nullptr;
    c->f_sq_row = nullptr;
    c->f_seedT = nullptr;
    c->f_row_nb = c->f_row_bins = c->f_row_pid = nullptr;
    c->f_cap_seedT = 0;
    c->f_mcT = nullptr;
    c->f_guess_all = nullptr;
    c->f_cap_guess = c->f_cap_mcT = 0;
    c->f_skip = nullptr;
    c->f_pair_row = c->f_pair_meta = c->f_mode = nullptr;
    c->f_ap = nullptr;
    c->f_cap_ap = c->f_cap_pairs = 0;
    c->f_items = nullptr;
    c->f_cta_begin = nullptr;
    c->f_row_slot = c->f_row_pt = nullptr;
    c->f_ub = c->f_ubk2 = nullptr;
    c->f_row_guess = c->f_rhist = nullptr;
    c->f_thr = c->f_t0 = c->f_a2 = c->f_tq = c->f_slack = c->f_ym2 = nullptr;
    c->f_mc = c->f_mc2 = nullptr;
    c->f_mcnt = nullptr;
    c->f_cap_mc = 0;
    c->f_cap_a2 = c->f_cap_bperm = 0;
    c->f_cap_bins = c->f_cap_cols = c->f_cap_cand = c->f_cap_thr = c->f_cap_ldt = 0;
    c->f_bin_cnt = c->f_seg_off = c->f_cursor = c->f_tile_bin = c->f_ntiles = c->f_col_pt = c->f_col_a = c->f_col_b = nullptr;
    c->f_col_nrm = c->f_bperm = c->f_cand_key = nullptr;
    c->f_cand_idx = nullptr;
    c->f_fb_pairs = nullptr;
    c->f_xs_slots = nullptr;
    c->f_xs_cap = 0;
    c->f_fb_alloc = 0;
}

// Runs steps 1-3 of the header comment for ALL owned query slots against the current (pos, tent, old) labels.
// Appends changed (slot_local, bin) pairs to ctx->work (count in counters[0]); queries needing the exact fallback are
// redone exactly on the device (exact_pairs_kernel; their count stays in counters[6]).
int chb_fused_argmin(chb_ctx *c, const int32_t *own_pos_dev, int64_t cnt, int64_t lo, int64_t hi, int32_t *tent_dev)
{
    if (cnt <= 0) return CHB_OK;
    {
        chb_stage_timer t(c, CHB_ST_COMMIT);
        CHB_PDL_LAUNCH(c, argmin_rows_kernel, nblk(cnt * 32, 256), 256, 0, own_pos_dev, cnt, c->perm_pt, c->qslot, c->u0, c->f_slot_row, c->f_row_nb,
                                                                       c->f_row_bins, c->pair_dist, c->C, c->old_label, lo, hi, tent_dev);
    }
    CHB_CUDA(c, cudaGetLastError());
    return CHB_OK;
}

int chb_fused_guess(chb_ctx *c)
{
    if (c->U <= 0) return CHB_OK;
    CHB_PDL_LAUNCH(c, guess_scatter_kernel, nblk(c->U, 256), 256, 0, c->qpoint, c->f_guess_all, c->U, c->C, c->tent_pt);
    CHB_CUDA(c, cudaGetLastError());
    ++c->tm.launches_other;
    return CHB_OK;
}

namespace {
__global__ void guess_export_kernel(const int32_t *__restrict__ guess_all, int64_t U, int64_t u0, int64_t u1, int32_t *__restrict__ out)
{
    const int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u < U) out[u] = (u >= u0 && u < u1) ? guess_all[u] : CHB_UNOWNED;
}
} // namespace

// Sharded contexts: every rank derives the speculation start of its OWN query slots (centroid terms = an U_own x C x d FP64
// contraction instead of U x C x d on every rank) and the ranks merge them with one all-reduce(MAX) over U int32 values.
extern "C" int chb_guess_export(chb_ctx *c, int32_t *guess_dev, int32_t *active)
{
    CHB_CHECK(c, c && guess_dev && active, CHB_EINVAL, "NULL argument");
    CHB_CHECK(c, c->labels_set && c->dist_ready, CHB_EINVAL, "guess_export: labels / distance structure not set up");
    *active = 0;
    if (!chb_use_fused(c) || c->U <= 0 || !c->guess_pending) return CHB_OK;
    CHB_CUDA(c, cudaSetDevice(c->device));
    if (!c->guess_shared) { c->guess_shared = true; c->f_asplit_ready = false; }
    c->guess_imported = false;
    {
        const int rc = chb_fused_setup(c);
        if (rc != CHB_OK) return rc;
    }
    guess_export_kernel<<<nblk(c->U, 256), 256, 0, c->stream>>>(c->f_guess_all, c->U, c->u0, c->u1, guess_dev);
    CHB_CUDA(c, cudaGetLastError());
    ++c->tm.launches_other;
    *active = 1;
    return CHB_OK;
}

extern "C" int chb_guess_import(chb_ctx *c, const int32_t *guess_dev)
{
    CHB_CHECK(c, c && guess_dev, CHB_EINVAL, "NULL argument");
    CHB_CHECK(c, c->guess_shared && c->f_guess_all, CHB_EINVAL, "guess_import without a preceding guess_export");
    CHB_CUDA(c, cudaSetDevice(c->device));
    CHB_CUDA(c, cudaMemcpyAsync(c->f_guess_all, guess_dev, sizeof(int32_t) * (size_t)c->U, cudaMemcpyDeviceToDevice, c->stream));
    c->guess_imported = true;
    return CHB_OK;
}

int chb_fused_grow_redo_list(chb_ctx *c)
{
    c->f_fb_worst = true; // chb_fused_setup sizes the list (and its regrouped copy) from this flag
    return chb_fused_setup(c);
}

int chb_fused_setup(chb_ctx *c)
{
    const int64_t nown = c->u1 - c->u0;
    const int64_t n = c->n;
    const int32_t C = c->C, k = c->k;
    const int KR = (k + 3 <= 8) ? 8 : 16;
    const FusedGeom g = fused_geom(c->d);
    const int64_t ncol_max = ((2 * n + (int64_t)BN * C + BN - 1) / BN) * BN;

    CHB_CHECK(c, chb_fused_supported(c), CHB_EINVAL, "fused mode supports num_neighbors <= 32 and d <= 1024");
    if (c->f_cap_bins < C + 1) {
        int64_t z = 0;
        z = 0; if (reserve(c, &c->f_bin_cnt, &z, C + 1)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_seg_off, &z, C + 2)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_cursor, &z, C + 1)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_ntiles, &z, 4)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_mode, &z, 4)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_pair_meta, &z, 5 * ((int64_t)C + 2))) return CHB_ENOMEM; // surv, off, cur, item_off, tile_cum
        z = 0; if (reserve(c, &c->f_ym2, &z, 2 * (C + 1))) return CHB_ENOMEM; // [0,C): max |y|^2, [C+1, 2C+1): max |column term|
        z = 0; if (reserve(c, &c->f_mcnt, &z, C + 1)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_mc2, &z, C + 1)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_rhist, &z, 2 * (C + 2))) return CHB_ENOMEM;
        c->f_cap_bins = C + 1;
    }
    if (reserve(c, &c->f_mcT, &c->f_cap_mcT, (int64_t)((C + 31) & ~31) * c->d)) return CHB_ENOMEM;
    if (reserve(c, &c->f_mc, &c->f_cap_mc, (int64_t)C * c->d)) return CHB_ENOMEM;
    if (reserve(c, &c->f_guess_all, &c->f_cap_guess, std::max<int64_t>(c->U, 1))) return CHB_ENOMEM;
    if (c->f_cap_cols < ncol_max) {
        int64_t z = 0;
        z = 0; if (reserve(c, &c->f_col_pt, &z, ncol_max)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_col_a, &z, ncol_max)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_col_b, &z, ncol_max)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_col_nrm, &z, ncol_max)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_tile_bin, &z, ncol_max / BN + 1)) return CHB_ENOMEM;
        c->f_cap_cols = ncol_max;
    }
    if (reserve(c, &c->f_bperm, &c->f_cap_bperm, ncol_max * g.Kp2)) return CHB_ENOMEM;
    {
        // Candidate lists (2 x KR keys + points per pair).  A slot per (row, bin) serves both kinds of round; at 1M contigs x
        // 500 bins that table alone is 61 GB for the 0.4 % of the pairs that survive the pruning, so beyond a budget
        // (CHB_DENSE_LIST_GB, default 8) only the compact pair ids get a slot -- rounds whose survivors do not fit the
        // compact buffers (hardly any pruning at that size) are then refused (pairs_plan_kernel -> CHB_ENOMEM at the commit).
        const int64_t per = (int64_t)KR * 2;
        const char *env = getenv("CHB_DENSE_LIST_GB");
        const double budget = (env ? atof(env) : 8.0) * (double)(1 << 30);
        const int64_t cap_pairs_now = ((4 * std::max<int64_t>(nown, 1) + (int64_t)BM * C + BM - 1) / BM) * BM;
        const bool dense = c->k > FUSED_KMAX ? false : (double)(nown * C * per) * 8.0 <= budget;
        // compacted rounds file the lists under compact pair ids (< cap_pairs, which exceeds nown * C when C < 4 + padding)
        const int64_t need = c->k > FUSED_KMAX ? 0 : (dense ? std::max<int64_t>(nown * C, cap_pairs_now) : cap_pairs_now) * per;
        if (c->f_cap_cand < need) {
            int64_t z = 0;
            z = 0; if (reserve(c, &c->f_cand_key, &z, need)) return CHB_ENOMEM;
            z = 0; if (reserve(c, &c->f_cand_idx, &z, need)) return CHB_ENOMEM;
            c->f_cap_cand = need;
        }
        c->f_cand_dense = dense;
    }
    {
        // pairs redone on exact distances: a few per row when they are the exception (k <= 15), every pair that survives
        // the pruning otherwise -- possibly all of them; + XS_G * C: that path pads every bin's range of the list to a
        // multiple of XS_G (exact_group_kernel)
        const int64_t per_row = (c->k > FUSED_KMAX || c->f_fb_worst) ? C : std::min<int64_t>(C, c->k > 15 ? 16 : 8);
        int64_t fbc = std::min<int64_t>(std::max<int64_t>(nown * per_row, 1024), INT32_MAX - 16 * (int64_t)C - 16);
        if (const char *t = getenv("CHB_TEST_FB_CAP")) // test aid: a tiny list, so that the overflow -> grow -> same window again path runs
            if (!c->f_fb_worst && c->k <= FUSED_KMAX) fbc = std::max<int64_t>(1, atoll(t));
        if (c->f_fb_alloc < fbc + 8 * (int64_t)C + 8) {
            int64_t z = 0;
            if (reserve(c, &c->f_fb_pairs, &z, fbc + 8 * (int64_t)C + 8)) return CHB_ENOMEM;
            c->f_fb_alloc = z;
        }
        c->f_fb_cap = (int32_t)fbc;
        if (c->k > 15 && c->k <= FUSED_KMAX && reserve(c, &c->f_xs_slots, &c->f_xs_cap, fbc + 8 * (int64_t)C + 8)) return CHB_ENOMEM;
    }
    c->f_ldt = (nown + 127) & ~int64_t(127);
    if (c->f_cap_thr < c->f_ldt * C || c->f_cap_ldt < c->f_ldt) {
        int64_t z = 0;
        c->f_cap_ldt = c->f_ldt;
        z = 0; if (reserve(c, &c->f_thr, &z, c->f_ldt * C)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_t0, &z, c->f_ldt * C)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_tq, &z, c->f_ldt * C)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_slack, &z, c->f_ldt * C)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_skip, &z, (c->f_ldt / BM) * C)) return CHB_ENOMEM;
        c->f_cap_pairs = ((4 * std::max<int64_t>(nown, 1) + (int64_t)BM * C + BM - 1) / BM) * BM;
        z = 0; if (reserve(c, &c->f_items, &z, std::max<int64_t>((c->f_ldt / BM) * C, c->f_cap_pairs / BM + C))) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_pair_row, &z, c->f_cap_pairs)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_cta_begin, &z, c->sm_count + 2)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_row_slot, &z, c->f_ldt)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_row_pt, &z, c->f_ldt)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_ub, &z, c->f_ldt)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_row_nb, &z, c->f_ldt)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_slot_row, &z, c->f_ldt)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_sq_row, &z, c->f_ldt)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_row_bins, &z, c->f_ldt * C)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_row_pid, &z, c->f_ldt * C)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_ubk2, &z, c->f_ldt)) return CHB_ENOMEM;
        z = 0; if (reserve(c, &c->f_row_guess, &z, c->f_ldt)) return CHB_ENOMEM;
        c->f_cap_thr = c->f_ldt * C;
        c->f_asplit_ready = false;
    }
    if (reserve(c, &c->f_ap, &c->f_cap_ap, c->f_cap_pairs * g.Kp2)) return CHB_ENOMEM;
    // once per (feature set, label set): bin reference points, row order, query operand and query terms
    if (!c->f_asplit_ready || c->f_cap_a2 < nown * g.Kp2) {
        if (reserve(c, &c->f_a2, &c->f_cap_a2, std::max<int64_t>(nown, 1) * g.Kp2)) return CHB_ENOMEM;
        // the side stream takes what only the first round's threshold_kernel needs (seed transpose, row_ub_kernel: 56 us at
        // 20k contigs, 2.5 ms at 1M) beside the chain that leads to the first round's column operand
        if (c->side_join_pending) { // a set-up that no round consumed
            CHB_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_join, 0));
            c->side_join_pending = false;
        }
        const int64_t ns_seed = std::max<int64_t>(n - c->U, 1);
        static const bool no_side = getenv("CHB_NO_SIDE") != nullptr; // A/B aid: everything on the one stream
        cudaStream_t side = no_side ? c->stream : c->side_stream;
        if (nown > 0) {
            if (reserve(c, &c->f_seedT, &c->f_cap_seedT, ns_seed * c->d)) return CHB_ENOMEM;
            if (!no_side) {
                CHB_CUDA(c, cudaEventRecord(c->ev_fork, c->stream));
                CHB_CUDA(c, cudaStreamWaitEvent(side, c->ev_fork, 0));
            }
            seed_transpose_kernel<<<nblk(ns_seed * c->d, 256), 256, 0, side>>>(c->Xf, c->ldf, c->d, c->seed_idx, n - c->U, c->f_seedT);
            ++c->tm.launches_other;
        }
        // bin reference points from the seed contigs (initial bins, fixed summation order)
        CHB_PDL_LAUNCH(c, centre_sum_kernel, (unsigned)C, 256, 0, c->X, c->ldx, c->d, c->seed_off, c->seed_idx, c->f_mc, c->f_mcnt);
        const int32_t Cp = (C + 31) & ~31;
        CHB_PDL_LAUNCH(c, centre_finish_kernel, (unsigned)C, 128, 0, c->f_mc, c->f_mcnt, c->colsum, 1.0 / (double)n, c->d, c->f_mc2,
                                                                 c->f_mcT, Cp);
        c->tm.launches_other += 2;
        // centroid terms |a_u - m_c|^2 and the nearest-centroid guess: for every slot, or -- when the ranks exchange their guesses
        // (chb_guess_export / chb_guess_import) -- for the owned slots only; f_tqs then starts at slot u0
        const int64_t t_first = c->guess_shared ? c->u0 : 0, t_cnt = c->guess_shared ? nown : c->U;
        if (t_cnt > 0) {
            if (reserve(c, &c->f_tqs, &c->f_cap_tqs, t_cnt * (int64_t)Cp)) return CHB_ENOMEM;
            dim3 gt((unsigned)((t_cnt + CT_M - 1) / CT_M), 1u);
            CHB_CUDA(c, cudaFuncSetAttribute(centroid_terms_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CT_SMEM));
            CHB_PDL_LAUNCH(c, centroid_terms_kernel, gt, 256, CT_SMEM, c->qpoint + t_first, t_cnt, c->Xf, c->ldf, c->d, c->f_mcT, Cp, c->f_mc2, C, c->f_tqs);
            CHB_PDL_LAUNCH(c, guess_from_terms_kernel, nblk(t_cnt * 32, 256), 256, 0, c->f_tqs, t_cnt, Cp, C, c->f_mcnt, c->f_guess_all + t_first);
            c->tm.launches_other += 2;
        }
        if (nown > 0) {
            // rows = owned slots grouped by guessed bin, so that a 128-row block prunes the same bins
            // (one single-CTA kernel for these four was tried for small inputs: slower -- one SM walking 20k entries with
            // dependent loads loses to four short launches over all SMs; likewise for the column entries below)
            c->tm.launches_other += 4;
            CHB_CUDA(c, cudaMemsetAsync(c->f_rhist, 0, sizeof(int32_t) * (size_t)(C + 2), c->stream));
            CHB_PDL_LAUNCH(c, row_hist_kernel, nblk(nown, 256), 256, 0, c->f_guess_all + c->u0, nown, c->f_rhist);
            CHB_PDL_LAUNCH(c, row_scan_kernel, 1, 32, 0, c->f_rhist, C + 1, c->f_rhist + C + 2);
            CHB_PDL_LAUNCH(c, row_scatter_kernel, nblk(nown, 256), 256, 0, c->f_guess_all + c->u0, nown, c->f_rhist + C + 2, c->f_row_slot);
            CHB_PDL_LAUNCH(c, row_gather_kernel, nblk(nown, 256), 256, 0, c->f_row_slot, c->qpoint + c->u0, c->f_guess_all + c->u0, c->nrm, nown,
                                                                      c->f_row_pt, c->f_row_guess, c->f_slot_row, c->f_sq_row);
            // fork: the row order is known; join: before the first round's threshold_kernel (chb_round_fused)
            if (!no_side) {
                CHB_CUDA(c, cudaEventRecord(c->ev_fork, c->stream));
                CHB_CUDA(c, cudaStreamWaitEvent(side, c->ev_fork, 0));
            }
            row_ub_kernel<<<(unsigned)(nown / RU_ROWS + C + 2), RU_THREADS, 0, side>>>(
                c->f_row_pt, nown, c->Xf, c->ldf, c->d, C, k, c->seed_off, c->f_seedT, n - c->U, c->f_rhist + C + 2, c->f_sq_row,
                reinterpret_cast<const unsigned int *>(&c->counters[5]), ub_inflation(c->d), c->f_ub, c->f_ubk2);
            if (!no_side) {
                CHB_CUDA(c, cudaEventRecord(c->ev_join, side));
                c->side_join_pending = true;
            }
            c->tm.launches_other += 1;
            CHB_PDL_LAUNCH(c, split2_gather_kernel, nblk(nown * (g.Kp2 / 4), 256), 256, 0, c->f_row_pt, nullptr, nown, c->Xf, c->ldf, c->d,
                                                                                      g.dp8, g.Kp2, c->nrm, c->f_a2, nullptr);
            dim3 gq((unsigned)((nown + QT_ROWS - 1) / QT_ROWS), (unsigned)((C + 31) / 32));
            CHB_PDL_LAUNCH(c, query_terms_gather_kernel, gq, 256, 0, c->f_tqs, Cp, c->u0 - t_first, c->f_row_slot, nown, C, c->f_ldt, c->f_tq);
            c->tm.launches_other += 2;
        }
        CHB_CUDA(c, cudaGetLastError());
        c->f_asplit_ready = true;
    }
    return CHB_OK;
}

int chb_round_fused(chb_ctx *c)
{
    const int64_t nown = c->u1 - c->u0;
    if (nown <= 0) return CHB_OK;
    const int64_t n = c->n;
    const int32_t C = c->C, k = c->k;
    const int KR = (k + 3 <= 8) ? 8 : 16;
    const FusedGeom g = fused_geom(c->d);
    const int64_t ncol_max = ((2 * n + (int64_t)BN * C + BN - 1) / BN) * BN;
    {
        const int rc0 = chb_fused_setup(c);
        if (rc0 != CHB_OK) return rc0;
    }

    // ---- 1. column entries
    CHB_PDL_LAUNCH(c, round_reset_kernel, nblk(std::max<int64_t>(std::max<int64_t>(std::max<int64_t>(nown, c->f_cap_pairs), ncol_max), 5 * (C + 2)), 256), 256, 0, c->f_bin_cnt, C + 1, c->f_ym2, 2 * (C + 1), c->f_row_nb, nown, c->f_pair_meta, 3 * (C + 2),
                                      c->f_pair_row, c->f_cap_pairs, c->counters, ncol_max, c->f_col_pt, c->f_col_a, c->f_col_b);
    CHB_PDL_LAUNCH(c, entries_count_kernel, nblk(n, 256), 256, 0, c->tent_pt, c->old_label, n, C, c->f_bin_cnt);
    CHB_PDL_LAUNCH(c, entries_scan_kernel, 1, 256, 0, c->f_bin_cnt, C, c->f_seg_off, c->f_cursor, c->f_tile_bin, c->f_ntiles);
    CHB_PDL_LAUNCH(c, entries_scatter_kernel, nblk(n, 256), 256, 0, c->tent_pt, c->old_label, c->pos, n, C, c->f_seg_off, c->f_cursor,
                                                                 c->f_col_pt, c->f_col_a, c->f_col_b);
    if (ncol_max >= (int64_t)1 << 18)
        CHB_PDL_LAUNCH(c, column_gather_wide_kernel, nblk(ncol_max, 32), 256, 0,
            c->f_col_pt, c->f_ntiles, c->f_tile_bin, c->X, c->ldx, c->d, c->colsum, 1.0 / (double)n, c->f_mc, g.dp8, g.Kp2, c->f_bperm,
            c->f_col_nrm, reinterpret_cast<unsigned int *>(c->f_ym2), reinterpret_cast<unsigned int *>(c->f_ym2 + C + 1));
    else
        CHB_PDL_LAUNCH(c, column_gather_kernel, nblk(ncol_max * 32, 256), 256, 0,
            c->f_col_pt, c->f_ntiles, c->f_tile_bin, c->X, c->ldx, c->d, c->colsum, 1.0 / (double)n, c->f_mc, g.dp8, g.Kp2, c->f_bperm,
            c->f_col_nrm, reinterpret_cast<unsigned int *>(c->f_ym2), reinterpret_cast<unsigned int *>(c->f_ym2 + C + 1));
    CHB_CUDA(c, cudaGetLastError());
    c->tm.launches_other += 5;

    c->round_counters_reset = c->qp_fb_zeroed = true; // round_reset_kernel (consumed by chb_launch_qp / commit_common)
    if (c->side_join_pending) { // row_ub_kernel of the label set-up (side stream)
        CHB_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_join, 0));
        c->side_join_pending = false;
    }

    // ---- 2. error slack and admission thresholds per (query, bin), then the fused Gram + selection.  eps_rel bounds the FP32
    // accumulation of the 3d products whatever the order the MMAs issue them in (the bound of a sum of n terms holds for any
    // summation tree); the streamed kernel's block-interleaved order and its zero pads past d (exact zeros) keep it.
    const double eps_rel = (double)(3 * c->d + 64) * 1.1920928955078125e-07;
    {
        const bool wide = nown * (int64_t)C >= (int64_t)1 << 24; // 16 M pairs and more: a stream over the pair table
        dim3 tg(nblk(nown, wide ? 1024 : 256), (unsigned)(wide ? (C + THR_BINS - 1) / THR_BINS : C));
        auto tk = wide ? threshold_kernel<4> : threshold_kernel<1>;
        CHB_PDL_LAUNCH(c, tk, tg, 256, 0, 
            c->knn_idx, c->knn_cnt, c->f_thr, c->f_row_pt, c->f_row_slot, c->pos, c->tent_pt, c->old_label, c->nrm,
            reinterpret_cast<const unsigned int *>(&c->counters[5]), c->f_ym2, c->f_ym2 + C + 1, c->f_tq, c->f_ub, c->f_sq_row, c->f_ubk2,
            c->f_row_guess, eps_rel, nown, C, k, c->metric == CHB_METRIC_CONVEX ? 1 : 0, c->f_ldt, c->f_t0, c->f_slack, c->f_row_nb,
            c->f_row_bins, c->f_pair_meta, c->f_skip, c->f_row_pid);
    }
    // KR = 16 serves k <= FUSED_KMAX: the re-rank needs the k + 1 smallest keys of the pair; they are all among the kept 2 x 16
    // unless one 64-column half holds 16 or more of them, which the re-rank's completeness tests detect (exact redo).  k + 3 <= KR
    // merely keeps those tests from firing often for small k.
    if (k > FUSED_KMAX) {
        // ---- 3'. large k: exact selection for every surviving pair (find_nearest_from_cluster on exact distances)
        chb_stage_timer t(c, CHB_ST_KNN);
        // surviving pairs regrouped per bin (threshold_kernel counted them per bin), XS_G queries of a bin per CTA pass
        int32_t *bin_surv = c->f_pair_meta, *xs_off = c->f_pair_meta + (C + 2), *xs_cur = c->f_pair_meta + 2 * (C + 2);
        const int32_t cap_slots = (int32_t)std::min<int64_t>(((int64_t)c->f_fb_cap + (int64_t)XS_G * C) & ~(int64_t)(XS_G - 1), INT32_MAX & ~(XS_G - 1));
        // per device, not per process: set on every call (a context may live on any device of this process)
        CHB_CUDA(c, cudaFuncSetAttribute(exact_group_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)exact_group_smem(c->d)));
        CHB_CUDA(c, cudaMemsetAsync(c->f_fb_pairs, 0xFF, sizeof(int2) * (size_t)cap_slots, c->stream));
        xs_plan_kernel<<<1, 32, 0, c->stream>>>(bin_surv, C, xs_off, &c->counters[6]);
        xs_fill_kernel<<<nblk(nown, 256), 256, 0, c->stream>>>(c->f_row_nb, c->f_row_bins, nown, C, xs_off, xs_cur, c->f_fb_pairs, cap_slots);
        exact_group_kernel<<<c->sm_count, XS_THREADS, exact_group_smem(c->d), c->stream>>>(
            c->f_fb_pairs, xs_off, cap_slots, c->f_seg_off, c->f_bin_cnt, c->f_col_pt, c->f_col_a, c->f_col_b, c->X, c->ldx, c->d, c->f_row_pt,
            c->f_row_slot, c->pos, C, k, c->knn_idx, c->knn_cnt, c->work, c->counters);
        CHB_CUDA(c, cudaGetLastError());
        c->tm.rows_scanned += nown;
        return CHB_OK;
    }
    const int64_t nrb = (nown + BM - 1) / BM;
    int32_t *bin_surv = c->f_pair_meta, *pair_off = c->f_pair_meta + (C + 2), *pair_cur = c->f_pair_meta + 2 * (C + 2);
    // test aid: CHB_FUSED_NO_COMPACT forces the (row block, bin) items that are otherwise only used when the compact buffer
    // would overflow
    const int64_t plan_cap = getenv("CHB_FUSED_NO_COMPACT") ? -1 : c->f_cap_pairs;
    CHB_PDL_LAUNCH(c, pairs_plan_kernel, 1, 1024, 0, bin_surv, c->f_seg_off, C, plan_cap, c->sm_count, pair_off,
                                                 c->f_pair_meta + 3 * (C + 2), c->f_items, c->f_cta_begin, &c->counters[7], c->f_mode,
                                                 c->f_cand_dense ? 1 : 0, c->f_skip, nrb);
    CHB_PDL_LAUNCH(c, g.stream ? pairs_fill_kernel<true> : pairs_fill_kernel<false>, nblk(nown * 32, 256), 256, 0, c->f_mode, c->f_row_nb, c->f_row_bins, nown, C, pair_off,
                   c->f_pair_row, c->f_row_pid, c->f_a2, g.Kp2, c->f_ap);
    CHB_CUDA(c, cudaGetLastError());
    c->tm.launches_other += 3;
    CUtensorMap ma, mb, map;
    int rc = make_map(c, &ma, c->f_a2, nown, g.Kp2);
    if (rc != CHB_OK) return rc;
    rc = make_map(c, &map, c->f_ap, c->f_cap_pairs, g.Kp2);
    if (rc != CHB_OK) return rc;
    rc = make_map(c, &mb, c->f_bperm, ncol_max, g.Kp2);
    if (rc != CHB_OK) return rc;
    rc = dispatch_fused(c, ma, map, mb, nown, g, KR);
    if (rc != CHB_OK) return rc;
    c->tm.rows_scanned += nown;

    // ---- 3. re-rank
    {
        chb_stage_timer t(c, CHB_ST_KNN);
        auto kern = (KR == 8) ? rerank_kernel<16> : rerank_kernel<32>;
        CHB_PDL_LAUNCH(c, kern, nblk(nown * 32, 256), 256, 0, 
            nown, c->f_cand_key, c->f_cand_idx, KR, c->f_bin_cnt, c->X, c->ldx, c->d, c->f_row_pt, c->f_row_slot, c->f_slack, C, k, c->knn_idx, c->knn_cnt, c->work, c->counters,
            c->f_fb_pairs, c->f_fb_cap, &c->counters[6], c->f_t0, c->f_ldt, c->f_thr, c->f_row_nb, c->f_row_bins, c->f_row_pid, c->f_mode);
        // pairs the re-rank could not settle from the kept lists (rare): exact redo, no host round trip -- the grid is
        // fixed and walks the device-side list
        const size_t xs = sizeof(double) * (size_t)((c->d + 1) & ~1);
        // one CTA per listed pair at a time (grid-stride over the device-side list): a handful at 20k contigs, tens of thousands
        // at 1M -- the grid follows the number of rows, up to eight resident CTAs per SM
        const unsigned xgrid = (unsigned)std::min<int64_t>((int64_t)c->sm_count * 8, std::max<int64_t>(64, nown / 256));
        if (KR == 8)
            CHB_PDL_LAUNCH(c, exact_pairs_kernel<5>, xgrid, 128, xs, c->f_fb_pairs, &c->counters[6], c->f_fb_cap, c->f_seg_off, c->f_bin_cnt, c->f_col_pt,
                                                              c->f_col_a, c->f_col_b, c->X, c->ldx, c->d, c->f_row_pt, c->f_row_slot, c->pos, C,
                                                              k, c->knn_idx, c->knn_cnt, c->work, c->counters);
        else if (k <= 15)
            CHB_PDL_LAUNCH(c, exact_pairs_kernel<15>, xgrid, 128, xs, c->f_fb_pairs, &c->counters[6], c->f_fb_cap, c->f_seg_off, c->f_bin_cnt,
                                                               c->f_col_pt, c->f_col_a, c->f_col_b, c->X, c->ldx, c->d, c->f_row_pt, c->f_row_slot,
                                                               c->pos, C, k, c->knn_idx, c->knn_cnt, c->work, c->counters);
        else {
            // 16 <= k <= FUSED_KMAX: a few per cent (k = 20) to one in six (k = 24) of the pairs overflow a half-list -- too many
            // for one CTA per pair; they are regrouped per bin and go through exact_group_kernel, eight pairs of a bin per pass
            int32_t *gb_cnt = c->f_pair_meta, *gb_off = c->f_pair_meta + (C + 2), *gb_cur = c->f_pair_meta + 2 * (C + 2); // free after the fused kernel
            const int32_t cap_slots = (int32_t)std::min<int64_t>(((int64_t)c->f_fb_cap + (int64_t)XS_G * C) & ~(int64_t)(XS_G - 1), INT32_MAX & ~(XS_G - 1));
            CHB_CUDA(c, cudaFuncSetAttribute(exact_group_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)exact_group_smem(c->d)));
            CHB_CUDA(c, cudaMemsetAsync(c->f_pair_meta, 0, sizeof(int32_t) * 3 * (size_t)(C + 2), c->stream));
            CHB_CUDA(c, cudaMemsetAsync(c->f_xs_slots, 0xFF, sizeof(int2) * (size_t)cap_slots, c->stream));
            fb_hist_kernel<<<c->sm_count, 256, 0, c->stream>>>(c->f_fb_pairs, &c->counters[6], c->f_fb_cap, gb_cnt);
            xs_plan_kernel<<<1, 32, 0, c->stream>>>(gb_cnt, C, gb_off, &c->counters[13]);
            fb_scatter_kernel<<<c->sm_count, 256, 0, c->stream>>>(c->f_fb_pairs, &c->counters[6], c->f_fb_cap, gb_off, gb_cur, c->f_xs_slots, cap_slots);
            exact_group_kernel<<<c->sm_count, XS_THREADS, exact_group_smem(c->d), c->stream>>>(
                c->f_xs_slots, gb_off, cap_slots, c->f_seg_off, c->f_bin_cnt, c->f_col_pt, c->f_col_a, c->f_col_b, c->X, c->ldx, c->d, c->f_row_pt,
                c->f_row_slot, c->pos, C, k, c->knn_idx, c->knn_cnt, c->work, c->counters);
        }
    }
    CHB_CUDA(c, cudaGetLastError());
    return CHB_OK;
}

extern "C" int chb_get_fused_candidates(chb_ctx *c, int64_t slot0, int64_t nslots, float *key_out, int32_t *idx_out, float *slack_out,
                                        int32_t *kr_out)
{
    CHB_CHECK(c, c && key_out && idx_out && slack_out && kr_out, CHB_EINVAL, "NULL argument");
    CHB_CHECK(c, c->f_cand_key && c->f_slack && slot0 >= c->u0 && nslots >= 0 && slot0 + nslots <= c->u1, CHB_EINVAL,
              "slots not owned / no fused round has run yet");
    CHB_CHECK(c, c->k <= FUSED_KMAX, CHB_EINVAL, "no candidate lists exist for num_neighbors > 24 (exact selection, chb_round_fused)");
    CHB_CUDA(c, cudaSetDevice(c->device));
    const int KR = (c->k + 3 <= 8) ? 8 : 16;
    const int64_t nown = c->u1 - c->u0, s0 = slot0 - c->u0, per = (int64_t)c->C * 2 * KR;
    *kr_out = KR;
    // the kernels keep these tables per ROW (owned slots ordered by guessed bin) and, in compacted rounds, the lists per
    // compact pair id: translate back to (slot, bin); bins the bounds ruled out have no list (keys +inf)
    const int32_t C = c->C;
    std::vector<int32_t> row_slot((size_t)std::max<int64_t>(nown, 1)), nb((size_t)std::max<int64_t>(nown, 1)), bins((size_t)C), pid((size_t)C);
    int32_t mode = 0;
    CHB_CUDA(c, cudaMemcpyAsync(row_slot.data(), c->f_row_slot, sizeof(int32_t) * (size_t)nown, cudaMemcpyDeviceToHost, c->stream));
    CHB_CUDA(c, cudaMemcpyAsync(nb.data(), c->f_row_nb, sizeof(int32_t) * (size_t)nown, cudaMemcpyDeviceToHost, c->stream));
    CHB_CUDA(c, cudaMemcpyAsync(&mode, c->f_mode, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    CHB_CUDA(c, cudaStreamSynchronize(c->stream));
    std::vector<float> srow((size_t)C);
    for (int64_t r = 0; r < nown; ++r) {
        const int64_t sl = row_slot[(size_t)r] - s0;
        if (sl < 0 || sl >= nslots) continue;
        for (int64_t e = 0; e < per; ++e) { key_out[sl * per + e] = INFINITY; idx_out[sl * per + e] = -1; }
        const int32_t n_b = nb[(size_t)r];
        CHB_CUDA(c, cudaMemcpyAsync(bins.data(), c->f_row_bins + r * C, sizeof(int32_t) * (size_t)n_b, cudaMemcpyDeviceToHost, c->stream));
        if (mode == 1)
            CHB_CUDA(c, cudaMemcpyAsync(pid.data(), c->f_row_pid + r * C, sizeof(int32_t) * (size_t)n_b, cudaMemcpyDeviceToHost, c->stream));
        CHB_CUDA(c, cudaMemcpy2DAsync(srow.data(), sizeof(float), c->f_slack + r, sizeof(float) * (size_t)c->f_ldt, sizeof(float),
                                      (size_t)C, cudaMemcpyDeviceToHost, c->stream));
        CHB_CUDA(c, cudaStreamSynchronize(c->stream));
        for (int32_t jb = 0; jb < n_b; ++jb) {
            const int32_t b = bins[(size_t)jb];
            const int64_t lslot = mode == 1 ? (int64_t)pid[(size_t)jb] : r * C + b;
            CHB_CUDA(c, cudaMemcpyAsync(key_out + sl * per + (int64_t)b * 2 * KR, c->f_cand_key + lslot * 2 * KR, sizeof(float) * 2 * KR,
                                        cudaMemcpyDeviceToHost, c->stream));
            CHB_CUDA(c, cudaMemcpyAsync(idx_out + sl * per + (int64_t)b * 2 * KR, c->f_cand_idx + lslot * 2 * KR, sizeof(int32_t) * 2 * KR,
                                        cudaMemcpyDeviceToHost, c->stream));
        }
        CHB_CUDA(c, cudaStreamSynchronize(c->stream));
        for (int32_t b = 0; b < C; ++b) slack_out[(int64_t)b * nslots + sl] = srow[(size_t)b];
    }
    CHB_CUDA(c, cudaStreamSynchronize(c->stream));
    return CHB_OK;
}

extern "C" int chb_get_row_bounds(chb_ctx *c, int64_t slot0, int64_t nslots, int32_t *guess_out, float *ub_out, float *ubk2_out)
{
    CHB_CHECK(c, c && guess_out && ub_out && ubk2_out, CHB_EINVAL, "NULL argument");
    CHB_CHECK(c, c->f_ub && c->f_asplit_ready && slot0 >= c->u0 && nslots >= 0 && slot0 + nslots <= c->u1, CHB_EINVAL,
              "slots not owned / the fused path has not set up this label set");
    CHB_CUDA(c, cudaSetDevice(c->device));
    if (c->side_join_pending) { // row_ub_kernel runs on the side stream
        CHB_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_join, 0));
        c->side_join_pending = false;
    }
    const int64_t nown = c->u1 - c->u0, s0 = slot0 - c->u0;
    std::vector<int32_t> slot_row((size_t)std::max<int64_t>(nown, 1)), guess((size_t)std::max<int64_t>(nown, 1));
    std::vector<float> ub((size_t)std::max<int64_t>(nown, 1)), ubk2((size_t)std::max<int64_t>(nown, 1));
    CHB_CUDA(c, cudaMemcpyAsync(slot_row.data(), c->f_slot_row, sizeof(int32_t) * (size_t)nown, cudaMemcpyDeviceToHost, c->stream));
    CHB_CUDA(c, cudaMemcpyAsync(guess.data(), c->f_row_guess, sizeof(int32_t) * (size_t)nown, cudaMemcpyDeviceToHost, c->stream));
    CHB_CUDA(c, cudaMemcpyAsync(ub.data(), c->f_ub, sizeof(float) * (size_t)nown, cudaMemcpyDeviceToHost, c->stream));
    CHB_CUDA(c, cudaMemcpyAsync(ubk2.data(), c->f_ubk2, sizeof(float) * (size_t)nown, cudaMemcpyDeviceToHost, c->stream));
    CHB_CUDA(c, cudaStreamSynchronize(c->stream));
    for (int64_t s = 0; s < nslots; ++s) {
        const int64_t r = slot_row[(size_t)(s0 + s)];
        guess_out[s] = guess[(size_t)r];
        ub_out[s] = ub[(size_t)r];
        ubk2_out[s] = ubk2[(size_t)r];
    }
    return CHB_OK;
}

int chb_fused_mask_pair_cache(chb_ctx *c, int64_t slot0, int64_t nslots, int32_t *cnt_out, double *dist_out)
{
    const int64_t nown = c->u1 - c->u0, s0 = slot0 - c->u0;
    const int32_t C = c->C;
    std::vector<int32_t> slot_row((size_t)std::max<int64_t>(nown, 1)), nb((size_t)std::max<int64_t>(nown, 1)), bins((size_t)C);
    CHB_CUDA(c, cudaMemcpyAsync(slot_row.data(), c->f_slot_row, sizeof(int32_t) * (size_t)nown, cudaMemcpyDeviceToHost, c->stream));
    CHB_CUDA(c, cudaMemcpyAsync(nb.data(), c->f_row_nb, sizeof(int32_t) * (size_t)nown, cudaMemcpyDeviceToHost, c->stream));
    CHB_CUDA(c, cudaStreamSynchronize(c->stream));
    std::vector<char> alive((size_t)C);
    for (int64_t s = 0; s < nslots; ++s) {
        const int64_t r = slot_row[(size_t)(s0 + s)];
        CHB_CUDA(c, cudaMemcpyAsync(bins.data(), c->f_row_bins + r * C, sizeof(int32_t) * (size_t)nb[(size_t)r], cudaMemcpyDeviceToHost, c->stream));
        CHB_CUDA(c, cudaStreamSynchronize(c->stream));
        std::fill(alive.begin(), alive.end(), 0);
        for (int32_t i = 0; i < nb[(size_t)r]; ++i) alive[(size_t)bins[(size_t)i]] = 1;
        for (int32_t b = 0; b < C; ++b)
            if (!alive[(size_t)b]) { cnt_out[s * C + b] = 0; dist_out[s * C + b] = INFINITY; }
    }
    return CHB_OK;
}
