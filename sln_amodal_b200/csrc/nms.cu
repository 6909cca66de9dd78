// nms.cu -- greedy NMS on the device, bit-compatible with the reference CPU extension.
//
// Reference semantics: nms/src/nms.c:4-69 (cpu_nms) behind nms/pth_nms.py:5-24.
// GPU baseline being replaced: nms/src/cuda/nms_kernel.cu:26-70 (full n x n mask incl.
// the useless lower triangle, ">" instead of ">=", FMA-contracted) followed by a
// synchronous D2H copy of the mask and a serial CPU scan (nms/src/nms_cuda.c:33-58).
//
// Pipeline (all on the caller's stream, no host round trip):
//   1. rank_kernel      stable rank of every box by (score desc, index asc)   O(n^2) compares, whole grid
//   2. gather_kernel    boxes/areas/classes permuted into visiting order
//   3. mask_kernel      upper-triangle 64x64 tiles of the "IoU >= thresh" bit matrix.  The
//                       IoU test reproduces nms.c's un-fused fp32 sequence; the divide is
//                       replaced by an exact sign test with a guarded fall-back to the
//                       IEEE divide (see iou_ge below)
//   4. scan_kernel      one CTA walks the 64-box chunks in order: a warp resolves each
//                       chunk against its diagonal tile with shuffles, the other warps
//                       OR the kept rows into the `removed` words in shared memory
#include "nms_core.cuh"

#include <cooperative_groups.h>

namespace sln {

// ---------------------------------------------------------------------------
// 1. rank sort
// ---------------------------------------------------------------------------
constexpr int RANK_ROWS = 256;     // elements ranked per CTA (one per thread)
constexpr int RANK_COLS = 1024;    // elements compared against per CTA (staged in smem)

// MODE 0: every column index is below every row index of this CTA  -> count key_j >= key_i
// MODE 1: every column index is above every row index              -> count key_j >  key_i
// MODE 2: index ranges overlap, or explicit tie ids                 -> full (key, tie) compare
// Carry-flag counting: `sub.cc` leaves the carry of a - b in CC.CF and `addc` adds it to the counter -- two
// instructions per compare, no predicate (ptxas even folds two carries into one IADD3.X).  Whether CF means
// "borrow" (a < b, the PTX manual's wording) or "no borrow" (a >= b, what the sm_100a SASS does) is NOT assumed:
// carry_counts_ge() probes it once per thread and the callers fold the answer in.
__device__ __forceinline__ void count_cf(int &cnt, unsigned a, unsigned b)
{
    asm("{\n\t.reg .u32 t;\n\tsub.cc.u32 t, %1, %2;\n\taddc.u32 %0, %0, 0;\n\t}" : "+r"(cnt) : "r"(a), "r"(b));
}
// same for (ahi, alo) - (bhi, blo) as 64-bit unsigned, three instructions
__device__ __forceinline__ void count_cf64(int &cnt, unsigned ahi, unsigned alo, unsigned bhi, unsigned blo)
{
    asm("{\n\t.reg .u32 t;\n\tsub.cc.u32 t, %1, %2;\n\tsubc.cc.u32 t, %3, %4;\n\taddc.u32 %0, %0, 0;\n\t}"
        : "+r"(cnt) : "r"(alo), "r"(blo), "r"(ahi), "r"(bhi));
}
__device__ __forceinline__ bool carry_counts_ge(unsigned one)    // `one` must be a run-time 1
{
    int probe = 0;
    count_cf(probe, one, 0u);                       // 1 - 0: no borrow
    return probe != 0;                              // true: count_cf counts a >= b; false: it counts a < b
}

// s_tie holds ~tie: "j precedes i" <=> (key_j, ~tie_j) > (key_i, ~tie_i) as one 64-bit unsigned compare.
// Returns, over the 4*n4 staged columns (padding: key 0, ~tie 0x80000000 -- never precedes anything and is never
// below anything):  MODE 0: #(key_j >= key_i)   MODE 1: #(key_j > key_i)   MODE 2: #(j precedes i)
template <int MODE>
__device__ __forceinline__ int rank_count(const uint4 *__restrict__ k4, const uint4 *__restrict__ t4, int n4,
                                          unsigned ki, unsigned nti, bool cf_is_ge)
{
    int c0 = 0, c1 = 0, c2 = 0, c3 = 0;            // four independent carry chains
#pragma unroll 4
    for (int q = 0; q < n4; ++q) {
        const uint4 k = k4[q];      // broadcast 16-byte shared load: four keys per instruction
        if (MODE == 0) {            // carry of key_j - key_i
            count_cf(c0, k.x, ki); count_cf(c1, k.y, ki); count_cf(c2, k.z, ki); count_cf(c3, k.w, ki);
        } else if (MODE == 1) {     // carry of key_i - key_j
            count_cf(c0, ki, k.x); count_cf(c1, ki, k.y); count_cf(c2, ki, k.z); count_cf(c3, ki, k.w);
        } else {                    // carry of K_i - K_j
            const uint4 t = t4[q];
            count_cf64(c0, ki, nti, k.x, t.x); count_cf64(c1, ki, nti, k.y, t.y);
            count_cf64(c2, ki, nti, k.z, t.z); count_cf64(c3, ki, nti, k.w, t.w);
        }
    }
    const int c = (c0 + c1) + (c2 + c3), all = 4 * n4;
    // MODE 0 wants #(key_j >= key_i); MODES 1/2 want #(K_i < K_j)
    if (MODE == 0) return cf_is_ge ? c : all - c;
    return cf_is_ge ? all - c : c;
}

// Optional epilogue of the rank kernel (sln_nms path): once the last column tile of a 256-row tile has added its
// counts -- detected with a ticket per row tile -- that CTA permutes its rows' boxes into visiting order.  This
// replaces a separate gather launch.  rank[] and the tickets are zeroed by one memset.
struct RankGather {
    const float *dets;         // [n][5]; nullptr: no gather
    const int *class_ids;      // may be nullptr
    float4 *boxes;
    float *areas;
    int *cls;
    int *order;
    int *tickets;              // [ceil(n / RANK_ROWS)]
};

__device__ __forceinline__ void rank_body(const float *scores, int stride, const int *tie_ids, int n,
                                          int *rank, RankGather ga)
{
    __shared__ __align__(16) unsigned s_key[RANK_COLS];
    __shared__ __align__(16) unsigned s_tie[RANK_COLS];     // ~tie id
    pdl_prologue();
    const int i0 = blockIdx.x * RANK_ROWS, i = i0 + threadIdx.x;
    const int j0 = blockIdx.y * RANK_COLS;
    const int jn = min(RANK_COLS, n - j0);
    // pad the tile to a multiple of 4 with entries that never count (key 0 with the largest tie id
    // loses every compare except against key 0 rows in MODE 0, handled by clamping below)
    // all loads of the thread (4 column keys, its own row key) are issued before the first use
    float sc[RANK_COLS / RANK_ROWS];
    int tie[RANK_COLS / RANK_ROWS];
#pragma unroll
    for (int q = 0; q < RANK_COLS / RANK_ROWS; ++q) {
        const int t = threadIdx.x + q * RANK_ROWS;
        sc[q] = 0.f;
        tie[q] = 0x7fffffff;
        if (t < jn) {
            sc[q] = __ldg(scores + (size_t)(j0 + t) * stride);
            tie[q] = tie_ids ? __ldg(tie_ids + j0 + t) : (j0 + t);
        }
    }
    float si = 0.f;
    int ti = i;
    if (i < n) {
        si = __ldg(scores + (size_t)i * stride);
        if (tie_ids) ti = __ldg(tie_ids + i);
    }
#pragma unroll
    for (int q = 0; q < RANK_COLS / RANK_ROWS; ++q) {
        const int t = threadIdx.x + q * RANK_ROWS;
        s_key[t] = t < jn ? score_key(sc[q]) : 0u;
        s_tie[t] = ~(unsigned)tie[q];
    }
    __syncthreads();
    int cnt = 0;
    if (i < n) {
    const unsigned ki = score_key(si);
    const int n4 = (jn + 3) >> 2, pad = n4 * 4 - jn;
    const uint4 *k4 = reinterpret_cast<const uint4 *>(s_key);
    const uint4 *t4 = reinterpret_cast<const uint4 *>(s_tie);
    const unsigned nti = ~(unsigned)ti;
    const bool cf_ge = carry_counts_ge((unsigned)(stride > 0));
    if (tie_ids == nullptr && j0 + jn <= i0) {
        cnt = rank_count<0>(k4, t4, n4, ki, nti, cf_ge);
        if (ki == 0u) cnt -= pad;                      // padded keys (0) satisfy 0 >= 0
    } else if (tie_ids == nullptr && j0 >= i0 + RANK_ROWS) {
        cnt = rank_count<1>(k4, t4, n4, ki, nti, cf_ge);
    } else {
        cnt = rank_count<2>(k4, t4, n4, ki, nti, cf_ge);
    }
    if (cnt) atomicAdd(rank + i, cnt);
    }
    if (ga.dets == nullptr) return;
    // ---- fused gather: the CTA that takes the last ticket of this row tile sees every column tile's counts
    __shared__ int s_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(ga.tickets + blockIdx.x, 1) == (int)gridDim.y - 1;
    __syncthreads();
    if (!s_last || i >= n) return;
    __threadfence();
    const int r = __ldcg(rank + i);
    const float c0 = ga.dets[5 * (size_t)i + 0], c1 = ga.dets[5 * (size_t)i + 1];
    const float c2 = ga.dets[5 * (size_t)i + 2], c3 = ga.dets[5 * (size_t)i + 3];
    ga.boxes[r] = make_float4(c0, c1, c2, c3);
    // pth_nms.py:16  areas = (x2 - x1 + 1) * (y2 - y1 + 1), one rounding per op
    ga.areas[r] = __fmul_rn(__fadd_rn(__fsub_rn(c3, c1), 1.f), __fadd_rn(__fsub_rn(c2, c0), 1.f));
    ga.order[r] = i;
    if (ga.class_ids) ga.cls[r] = ga.class_ids[i];
}

__global__ void __launch_bounds__(RANK_ROWS)
rank_kernel(const float *__restrict__ scores, int stride, const int *__restrict__ tie_ids, int n,
            int *__restrict__ rank, RankGather ga)
{
    rank_body(scores, stride, tie_ids, n, rank, ga);
}

// segment z = blockIdx.z.  Inputs move by in_stride bytes per segment (scores, tie ids, the gather's dets) and by
// cls_stride (the gather's class ids); rank and the gather's outputs and tickets by ws_stride.  Null pointers stay null.
__device__ __forceinline__ RankGather rank_gather_at(RankGather ga, size_t in_stride, size_t cls_stride, size_t ws_stride,
                                                     int z)
{
    if (ga.dets == nullptr) return ga;
    ga.dets = seg_at(ga.dets, in_stride, z);
    if (ga.class_ids) ga.class_ids = seg_at(ga.class_ids, cls_stride, z);
    ga.boxes = seg_at(ga.boxes, ws_stride, z);
    ga.areas = seg_at(ga.areas, ws_stride, z);
    ga.cls = seg_at(ga.cls, ws_stride, z);
    ga.order = seg_at(ga.order, ws_stride, z);
    ga.tickets = seg_at(ga.tickets, ws_stride, z);
    return ga;
}

__global__ void __launch_bounds__(RANK_ROWS)
rank_seg_kernel(const float *__restrict__ scores, int stride, const int *__restrict__ tie_ids, int n,
                int *__restrict__ rank, RankGather ga, size_t in_stride, size_t cls_stride, size_t ws_stride)
{
    const int z = blockIdx.z;
    rank_body(seg_at(scores, in_stride, z), stride, tie_ids ? seg_at(tie_ids, in_stride, z) : nullptr, n,
              seg_at(rank, ws_stride, z), rank_gather_at(ga, in_stride, cls_stride, ws_stride, z));
}

static int rank_launch(const float *scores, int stride, const int *tie_ids, int n, int *rank, const RankGather &ga,
                       cudaStream_t st)
{
    if (n <= 0) return SLN_OK;
    dim3 grid(cdiv(n, RANK_ROWS), cdiv(n, RANK_COLS));
    SLN_REQUIRE(grid.y <= 65535, SLN_ERR_ARG, "rank sort: n=%d too large", n);
    rank_kernel<<<grid, RANK_ROWS, 0, st>>>(scores, stride, tie_ids, n, rank, ga);
    SLN_LAUNCH_OK("rank_kernel");
    return SLN_OK;
}

int rank_sort_launch(const float *scores, int stride, const int *tie_ids, int n, int *rank, cudaStream_t st)
{
    return rank_launch(scores, stride, tie_ids, n, rank, RankGather{}, st);
}

static int rank_seg_launch(const float *scores, int stride, const int *tie_ids, int n, int B, int *rank,
                           const RankGather &ga, size_t in_stride, size_t cls_stride, size_t ws_stride, cudaStream_t st)
{
    if (n <= 0 || B <= 0) return SLN_OK;
    dim3 grid(cdiv(n, RANK_ROWS), cdiv(n, RANK_COLS), B);
    SLN_REQUIRE(grid.y <= 65535 && grid.z <= 65535, SLN_ERR_ARG, "rank sort: n=%d x %d segments too large", n, B);
    rank_seg_kernel<<<grid, RANK_ROWS, 0, st>>>(scores, stride, tie_ids, n, rank, ga, in_stride, cls_stride, ws_stride);
    SLN_LAUNCH_OK("rank_seg_kernel");
    return SLN_OK;
}

int rank_sort_batched_launch(const float *scores, const int *tie_ids, int n, int B, size_t stride_bytes, int *rank,
                             cudaStream_t st)
{
    return rank_seg_launch(scores, 1, tie_ids, n, B, rank, RankGather{}, stride_bytes, 0, stride_bytes, st);
}

// ---------------------------------------------------------------------------
// 3. IoU >= thresh bit matrix
// ---------------------------------------------------------------------------
// nms.c:51-61 restated:  w = max(0, min(x2)-max(x1)+1), h likewise, inter = w*h,
// ovr = inter / (area_i + area_j - inter), suppressed iff ovr >= thresh -- every
// operation rounded to fp32 separately (the CPU build has no FMA).
// The divide is avoided without changing the decision: d = fma(-thresh, den, inter)
// is inter - thresh*den rounded once; when den > 0 and |d| > 2^-20 * inter the true
// ratio is more than 2^-20 (relative) away from thresh, far outside the 2^-24 band in
// which the rounded quotient could land on the other side, so sign(d) decides.
// Anything else (near ties, den <= 0, inf/NaN) takes the IEEE divide.
__device__ __forceinline__ bool iou_ge(const float4 a, const float aa, const float4 b, const float ab,
                                       const float thresh)
{
    const float xx1 = fmaxf(a.x, b.x), yy1 = fmaxf(a.y, b.y);
    const float xx2 = fminf(a.z, b.z), yy2 = fminf(a.w, b.w);
    const float w = fmaxf(0.f, __fadd_rn(__fsub_rn(xx2, xx1), 1.f));
    const float h = fmaxf(0.f, __fadd_rn(__fsub_rn(yy2, yy1), 1.f));
    const float inter = __fmul_rn(w, h);
    const float den = __fsub_rn(__fadd_rn(aa, ab), inter);
    const float d = __fmaf_rn(-thresh, den, inter);
    if (den > 0.f && fabsf(d) > __fmul_rn(inter, 9.5367431640625e-07f)) return d > 0.f;
    return __fdiv_rn(inter, den) >= thresh;
}

// One 64-thread group per tile (row block rb, column block cb >= rb); 4 groups per CTA.
// Thread t owns row rb*64+t and produces one 64-bit word.  Diagonal tiles carry the
// full symmetric relation (bit t itself cleared).
constexpr int MASK_GROUPS = 4;

template <bool CLS>
__global__ void __launch_bounds__(64 * MASK_GROUPS)
nms_mask_kernel(const float4 *__restrict__ boxes, const float *__restrict__ areas, const int *__restrict__ cls,
                int n_host, const int *__restrict__ n_dev, int W_stride, float thresh,
                unsigned long long *__restrict__ mask, const int *__restrict__ skip,
                unsigned long long *__restrict__ fix_zero, int fix_words)
{
    if (skip && *skip == 1) return;                // the sparse path already produced the result
    // scratch of the resolve kernels that follow (removed sets, K, state): zeroed here instead of by a memset launch
    if (blockIdx.x == 0)
        for (int k = threadIdx.x; k < fix_words; k += blockDim.x) fix_zero[k] = 0ull;
    // n may live in device memory (second stage of the two-stage pipeline): the grid is sized for the
    // worst case and surplus CTAs leave at once
    const int n = n_dev ? *n_dev : n_host;
    const int W = (n + 63) >> 6;
    const long long n_tiles = (long long)W * (W + 1) / 2;
    __shared__ float4 s_box[MASK_GROUPS][64];
    __shared__ float s_area[MASK_GROUPS][64];
    __shared__ int s_cls[MASK_GROUPS][64];
    const int grp = threadIdx.x >> 6, t = threadIdx.x & 63;
    // grid-strided over blocks of MASK_GROUPS tiles (the grid is capped so that the "skip" exit above is cheap)
    for (long long tb = blockIdx.x; tb * MASK_GROUPS < n_tiles; tb += gridDim.x) {
        const long long tile = tb * MASK_GROUPS + grp;
        const bool active = tile < n_tiles;
        int rb = 0, cb = 0;
        __syncthreads();                           // the previous iteration's reads of s_box are done
        if (active) {
            // tiles are numbered row block by row block: row rb holds W-rb tiles (cb = rb..W-1)
            // start(rb) = rb*W - rb*(rb-1)/2
            const double Wd = (double)W + 0.5;
            rb = (int)(Wd - sqrt(Wd * Wd - 2.0 * (double)tile));
            if (rb < 0) rb = 0;
            if (rb > W - 1) rb = W - 1;
            while (rb > 0 && (long long)rb * W - (long long)rb * (rb - 1) / 2 > tile) --rb;
            while ((long long)(rb + 1) * W - (long long)(rb + 1) * rb / 2 <= tile) ++rb;
            cb = rb + (int)(tile - ((long long)rb * W - (long long)rb * (rb - 1) / 2));
            const int j = cb * 64 + t;
            if (j < n) {
                s_box[grp][t] = boxes[j];
                s_area[grp][t] = areas[j];
                if (CLS) s_cls[grp][t] = cls[j];
            }
        }
        __syncthreads();
        const int i = rb * 64 + t;
        if (!active || i >= n) continue;
        const float4 bi = boxes[i];
        const float ai = areas[i];
        const int ci = CLS ? cls[i] : 0;
        const int jn = min(64, n - cb * 64);
        unsigned long long bits = 0ull;
#pragma unroll 4
        for (int k = 0; k < jn; ++k) {
            bool hit = iou_ge(bi, ai, s_box[grp][k], s_area[grp][k], thresh);
            if (CLS) hit = hit && (s_cls[grp][k] == ci);
            bits |= (unsigned long long)hit << k;
        }
        if (rb == cb) bits &= ~(1ull << t);
        mask[(size_t)i * W_stride + cb] = bits;
    }
}

// ---------------------------------------------------------------------------
// 4. greedy scan (single CTA, software-pipelined over super-steps of 8 chunks = 512 boxes)
// ---------------------------------------------------------------------------
// The scan is inherently sequential in 64-box chunks: chunk c can only be resolved once the
// kept boxes of chunks < c have been ORed into its `removed` word.  To keep global-memory
// latency off that chain, the mask is consumed in two ways:
//   band(k)  rows of super-step k x the 16 words [8k, 8k+16): fetched UNCONDITIONALLY into
//            shared memory with cp.async one super-step ahead (double buffered).  Warp 0
//            resolves the 8 chunks of a super-step from shared memory alone: the diagonal word
//            gives the in-chunk relation (resolved by a ballot fixpoint, typically 2-3 rounds),
//            the other band words carry the kept rows into the next <= 15 words.
//   far(k)   kept rows of super-step k x words >= 8k+16: read from global memory by the other
//            31 warps while warp 0 already resolves super-step k+1 (they have a whole
//            super-step of slack); results land in the shared `removed` words via atomicOr.
// One block barrier per super-step; nothing else synchronises.
constexpr int SCAN_THREADS = 1024;
constexpr int SS_CHUNKS = 8;                       // chunks per super-step
constexpr int SS_ROWS = 64 * SS_CHUNKS;            // boxes per super-step
constexpr int BAND_WORDS = 2 * SS_CHUNKS;          // words of a band row
constexpr int BAND_STRIDE = BAND_WORDS + 1;        // padded row stride (u64) against bank conflicts

__device__ __forceinline__ void cp_async_8(void *smem_dst, const void *gmem_src)
{
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sa), "l"(gmem_src) : "memory");
}

__device__ __forceinline__ unsigned long long shfl_xor_u64(unsigned long long v, int m)
{
    const unsigned lo = __shfl_xor_sync(0xffffffffu, (unsigned)v, m);
    const unsigned hi = __shfl_xor_sync(0xffffffffu, (unsigned)(v >> 32), m);
    return ((unsigned long long)hi << 32) | lo;
}

__device__ __forceinline__ unsigned long long ballot64(bool a, bool b)
{
    const unsigned lo = __ballot_sync(0xffffffffu, a), hi = __ballot_sync(0xffffffffu, b);
    return ((unsigned long long)hi << 32) | lo;
}

// n may live in device memory (n_dev != nullptr): the two-stage pipeline compacts on the device
__global__ void __launch_bounds__(SCAN_THREADS)
nms_scan_kernel(const unsigned long long *__restrict__ mask, const int *__restrict__ order, int n_host,
                const int *__restrict__ n_dev, int W_stride, int max_keep_host, const int *__restrict__ keep_base_dev,
                int64_t *__restrict__ keep64, int *__restrict__ keep32, int *__restrict__ num_keep,
                const int *__restrict__ done_flag, const int *__restrict__ skip)
{
    extern __shared__ __align__(16) unsigned long long s_mem[];
    if (done_flag && *done_flag == 1) return;      // the parallel resolve already produced the result
    if (skip && *skip == 1) return;                // so did the sparse path
    const int n = n_dev ? *n_dev : n_host;
    const int W = (n + 63) >> 6;
    // keep_base: survivors already emitted by an earlier stage (they count against max_keep)
    const int keep_base = keep_base_dev ? *keep_base_dev : 0;
    const int max_keep = max_keep_host;
    unsigned long long *s_removed = s_mem;                                      // [W_stride]
    unsigned long long *s_band = s_mem + W_stride;                              // [2][SS_ROWS][BAND_STRIDE]
    int *s_klist = reinterpret_cast<int *>(s_band + 2 * SS_ROWS * BAND_STRIDE); // [2][SS_ROWS]
    __shared__ unsigned long long s_K[2][SS_CHUNKS];   // kept bits of the chunks of a super-step
    __shared__ int s_base[2];                          // survivors emitted before the super-step
    __shared__ int s_nk[2];
    __shared__ int s_total, s_stop;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int w = tid; w < W; w += SCAN_THREADS) s_removed[w] = 0ull;
    if (tid == 0) { s_total = keep_base; s_stop = (keep_base >= max_keep || n == 0) ? 1 : 0; s_nk[0] = s_nk[1] = 0; }

    auto prefetch_band = [&](int k, int first_thread, int nthreads) {
        unsigned long long *dst = s_band + (size_t)(k & 1) * SS_ROWS * BAND_STRIDE;
        const int row0 = k * SS_ROWS, w0 = k * SS_CHUNKS;
        for (int i = tid - first_thread; i < SS_ROWS * BAND_WORDS; i += nthreads) {
            const int rl = i / BAND_WORDS, wl = i - rl * BAND_WORDS;
            const int row = row0 + rl, w = w0 + wl;
            if (row < n && w < W) cp_async_8(dst + rl * BAND_STRIDE + wl, mask + (size_t)row * W_stride + w);
            else dst[rl * BAND_STRIDE + wl] = 0ull;
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    // emit the survivors of chunk j of super-step kk (kept bits in s_K, count before the super-step in
    // s_base): one warp per chunk, so the eight chunks' dependent order[] loads overlap
    auto emit = [&](int kk, int j) {
        const int c = kk * SS_CHUNKS + j;
        int before = 0, all = 0;
#pragma unroll
        for (int jj = 0; jj < SS_CHUNKS; ++jj) {
            const int cnt = __popcll(s_K[kk & 1][jj]);
            if (jj < j) before += cnt;
            all += cnt;
        }
        if (j == 0 && lane == 0) s_nk[kk & 1] = all;
        if (c >= W) return;
        const unsigned long long K = s_K[kk & 1][j];
        const int total = s_base[kk & 1] + before;
        int *klist = s_klist + (kk & 1) * SS_ROWS;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int b = lane + 32 * half;
            if ((K >> b) & 1ull) {
                const int off = __popcll(K & ((1ull << b) - 1ull));
                const int pos = c * 64 + b;
                const int idx = order ? order[pos] : pos;
                if (keep64) keep64[total + off] = idx;
                if (keep32) keep32[total + off] = idx;
                klist[before + off] = pos;
            }
        }
    };

    const int n_super = (W + SS_CHUNKS - 1) / SS_CHUNKS;
    prefetch_band(0, 0, SCAN_THREADS);
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();

    int k = 0;
    for (; k < n_super; ++k) {
        if (s_stop) break;
        const unsigned long long *band = s_band + (size_t)(k & 1) * SS_ROWS * BAND_STRIDE;
        if (warp == 0) {
            // ------------------------------------------------ resolve the 8 chunks of super-step k (the serial chain)
            int total = s_total;
            if (lane == 0) s_base[k & 1] = total;
            if (lane < SS_CHUNKS) s_K[k & 1][lane] = 0ull;
            __syncwarp();
            for (int j = 0; j < SS_CHUNKS; ++j) {
                const int c = k * SS_CHUNKS + j;
                if (c >= W) break;
                const int nb = min(64, n - c * 64);
                const unsigned long long valid = nb == 64 ? ~0ull : ((1ull << nb) - 1ull);
                // predecessor sets of my two boxes inside the chunk (diagonal tiles are symmetric)
                const unsigned long long p0 = band[(64 * j + lane) * BAND_STRIDE + j] & ((1ull << lane) - 1ull);
                const unsigned long long p1 = band[(64 * j + lane + 32) * BAND_STRIDE + j] & ((1ull << (lane + 32)) - 1ull);
                const unsigned long long U = ~s_removed[c] & valid;
                const bool u0 = (U >> lane) & 1ull, u1 = (U >> (lane + 32)) & 1ull;
                // K is the unique fixed point of  K = { b in U : no a in K, a < b, overlaps b }  (the
                // relation is acyclic); iterate from K = U until stable: 2 ANDs + 2 ballots per round
                unsigned long long K = U;
                for (;;) {
                    const unsigned long long Kn = ballot64(u0 && !(p0 & K), u1 && !(p1 & K));
                    if (Kn == K) break;
                    K = Kn;
                }
                int cnt = __popcll(K);
                if (total + cnt > max_keep) {          // keep only the first (max_keep-total) survivors
                    int need = max_keep - total;
                    unsigned long long k2 = 0ull, rest = K;
                    while (need-- > 0) {
                        const int b = __ffsll((long long)rest) - 1;
                        k2 |= 1ull << b;
                        rest &= ~(1ull << b);
                    }
                    K = k2;
                    cnt = __popcll(K);
                }
                if (lane == 0) s_K[k & 1][j] = K;
                total += cnt;
                if (total >= max_keep) { if (lane == 0) s_stop = 1; break; }
                // carry the kept rows into the band words after the diagonal: lane = (word wl, half of K);
                // only set bits of K are visited
                if (K) {
                    const int wl = lane & 15, half = lane >> 4;
                    unsigned long long acc = 0ull;
                    unsigned kb = (unsigned)(K >> (32 * half));
                    const unsigned long long *rows = band + (size_t)(64 * j + 32 * half) * BAND_STRIDE + wl;
                    while (kb) {
                        const int i = __ffs(kb) - 1;
                        kb &= kb - 1u;
                        acc |= rows[i * BAND_STRIDE];
                    }
                    acc |= shfl_xor_u64(acc, 16);
                    const int w = k * SS_CHUNKS + wl;
                    // atomic: the background warps OR into words >= 8k+8 at the same time
                    if (half == 0 && wl > j && w < W && acc) atomicOr(s_removed + w, acc);
                }
                __syncwarp();
            }
            if (lane == 0) s_total = total;
        } else {
            // ------------------------------------------------ background warps
            // (0) next band: asynchronous copies, waited for at the end of the iteration
            if (k + 1 < n_super) prefetch_band(k + 1, 32, SCAN_THREADS - 32);
            // (1) warps 1..8 write out the survivors of super-step k-1 and build its row list
            if (k >= 1 && warp <= SS_CHUNKS) emit(k - 1, warp - 1);
            asm volatile("bar.sync 1, %0;" ::"r"(SCAN_THREADS - 32) : "memory");
            // (2) far update: kept rows of super-step k-1 x words >= 8(k+1), straight from global memory
            if (k >= 1) {
                const int kp = k - 1;
                const int nk = s_nk[kp & 1];
                const int *klist = s_klist + (kp & 1) * SS_ROWS;
                const int wbeg = (kp + 2) * SS_CHUNKS;
                const int nw = W - wbeg;
                if (nw > 0 && nk > 0) {
                    // thread = (word, row group): a fixed word per thread, rows strided by the group
                    // count, eight independent loads in flight, one atomicOr per thread at the end
                    const int T = SCAN_THREADS - 32, t = tid - 32;
                    const int cols = min(nw, T);
                    const int groups = max(1, T / cols);
                    const int g = t / cols, wi = t - g * cols;
                    if (g < groups) {
                        for (int w = wbeg + wi; w < W; w += cols) {
                            const unsigned long long *col = mask + w;
                            unsigned long long acc = 0ull;
                            for (int r0 = g; r0 < nk; r0 += 8 * groups) {
                                unsigned long long v[8];
#pragma unroll
                                for (int u = 0; u < 8; ++u) {
                                    const int r = r0 + u * groups;
                                    v[u] = r < nk ? __ldg(col + (size_t)klist[r] * W_stride) : 0ull;
                                }
#pragma unroll
                                for (int u = 0; u < 8; ++u) acc |= v[u];
                            }
                            if (acc) atomicOr(s_removed + w, acc);
                        }
                    }
                }
            }
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();
    }
    // survivors of the last resolved super-step
    if (warp >= 1 && warp <= SS_CHUNKS && k >= 1) emit(k - 1, warp - 1);
    if (tid == 0) *num_keep = min(s_total, max_keep);
}

// ---------------------------------------------------------------------------
// 4b. parallel resolve: the greedy survivor set as a fixed point, computed by the whole GPU
// ---------------------------------------------------------------------------
// The greedy result is the unique K with  K = { b : no a in K, a < b, overlaps b }  (the relation
// is acyclic).  Iterating K <- F(K) from K = "all boxes" converges to it; on detector-like inputs in
// a handful of rounds (6 on the 12k RPN-like set, 3 on the low-overlap set), each round being one
// fully parallel pass: OR the mask rows of the current K into `removed`, then K' = ~removed.
// Persistent cooperative kernel: CTA = one 64-box chunk at a time (grid-strided), software grid
// barrier between the phases.  If MAX_ROUNDS is not enough, `status` is left at 0 and the serial
// scan kernel (launched right after, it exits at once when status == 1) produces the result.
constexpr int FIX_THREADS = 256;
constexpr int FIX_MAX_ROUNDS = 24;
constexpr int FIX_MIN_WORDS = 160;         // measured on RPN-like boxes: serial chain wins below ~10k boxes (8k: 183 vs 208 us), loses above (12k: 290 vs 251 us)

struct FixState {
    unsigned barrier;      // arrivals at the software grid barrier (monotone)
    int status;            // 1: converged, result written
    int changed[FIX_MAX_ROUNDS + 2];
};

__device__ __forceinline__ void grid_barrier(unsigned *counter, unsigned &generation, unsigned n_ctas)
{
    __syncthreads();
    ++generation;
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(counter, 1u);
        const unsigned target = generation * n_ctas;
        while (*reinterpret_cast<volatile unsigned *>(counter) < target) { }
        __threadfence();
    }
    __syncthreads();
}

__global__ void __launch_bounds__(FIX_THREADS)
nms_fixpoint_kernel(const unsigned long long *__restrict__ mask, const int *__restrict__ order, int n_host,
                    const int *__restrict__ n_dev, int W_stride, int max_keep, const int *__restrict__ keep_base_dev,
                    unsigned long long *__restrict__ removed /* [2][W_stride] */, unsigned long long *__restrict__ Kbuf /* [W_stride] */,
                    FixState *__restrict__ state, int64_t *__restrict__ keep64, int *__restrict__ keep32,
                    int *__restrict__ num_keep, const int *__restrict__ skip)
{
    if (skip && *skip == 1) return;                // uniform over the grid: nobody reaches a barrier
    const int n = n_dev ? *n_dev : n_host;
    const int W = (n + 63) >> 6;
    const int keep_base = keep_base_dev ? *keep_base_dev : 0;
    const int tid = threadIdx.x;
    const unsigned G = gridDim.x;
    unsigned gen = 0;
    __shared__ unsigned long long s_K;

    // Round r reads removed[r % 3] (round 0: nothing removed), ORs into removed[(r+1) % 3] and clears
    // removed[(r+2) % 3] for the round after -- so one grid barrier per round is enough (all three
    // buffers are zeroed by the host-side memset before the launch).
    int round = 0;
    bool converged = false;
    for (; round < FIX_MAX_ROUNDS; ++round) {
        const unsigned long long *rin = removed + (size_t)(round % 3) * W_stride;
        unsigned long long *rout = removed + (size_t)((round + 1) % 3) * W_stride;
        unsigned long long *rclr = removed + (size_t)((round + 2) % 3) * W_stride;
        for (int c = blockIdx.x; c < W; c += G) {
            if (tid == 0) {
                const int nb = min(64, n - c * 64);
                const unsigned long long valid = nb == 64 ? ~0ull : ((1ull << nb) - 1ull);
                const unsigned long long K = round == 0 ? valid : (valid & ~__ldcg(rin + c));   // L2: written by other SMs
                if (round == 0 || K != __ldcg(Kbuf + c)) atomicOr(&state->changed[round], 1);
                Kbuf[c] = K;
                rclr[c] = 0ull;
                s_K = K;
            }
            __syncthreads();
            const unsigned long long K = s_K;
            if (K) {
                // OR the rows of this chunk's kept boxes into the output words
                for (int w = c + tid; w < W; w += FIX_THREADS) {
                    const unsigned long long *col = mask + (size_t)c * 64 * W_stride + w;
                    unsigned long long acc = 0ull, k = K;
                    while (k) {                    // eight independent loads in flight
                        unsigned long long v[8];
#pragma unroll
                        for (int u = 0; u < 8; ++u) {
                            v[u] = 0ull;
                            if (k) {
                                const int b = __ffsll((long long)k) - 1;
                                k &= k - 1ull;
                                unsigned long long row = __ldg(col + (size_t)b * W_stride);
                                if (w == c) row &= ~((2ull << b) - 1ull);      // diagonal tile: successors only
                                v[u] = row;
                            }
                        }
#pragma unroll
                        for (int u = 0; u < 8; ++u) acc |= v[u];
                    }
                    if (acc) atomicOr(rout + w, acc);
                }
            }
            __syncthreads();
        }
        grid_barrier(&state->barrier, gen, G);
        // K of this round equals K of the previous one everywhere: it is the fixed point (uniform decision)
        if (*reinterpret_cast<volatile int *>(&state->changed[round]) == 0) { converged = true; break; }
    }
    if (!converged) return;            // status stays 0: the serial scan kernel takes over

    // emission: survivors in visiting order; each chunk's offset is the popcount of the chunks before it
    for (int c = blockIdx.x; c < W; c += G) {
        int before = 0;
        for (int cc = tid; cc < c; cc += FIX_THREADS) before += __popcll(__ldcg(Kbuf + cc));
        __shared__ int s_red[FIX_THREADS / 32];
        for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
        if ((tid & 31) == 0) s_red[tid >> 5] = before;
        __syncthreads();
        int total = keep_base;
        for (int k = 0; k < FIX_THREADS / 32; ++k) total += s_red[k];
        const unsigned long long K = __ldcg(Kbuf + c);
        if (tid < 64 && ((K >> tid) & 1ull)) {
            const int slot = total + __popcll(K & ((1ull << tid) - 1ull));
            if (slot < max_keep) {
                const int pos = c * 64 + tid;
                const int idx = order ? order[pos] : pos;
                if (keep64) keep64[slot] = idx;
                if (keep32) keep32[slot] = idx;
            }
        }
        if (c == W - 1 && tid == 0) {
            *num_keep = min(total + __popcll(K), max_keep);
            state->status = 1;
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------
// two-stage pipeline helpers
// ---------------------------------------------------------------------------
// Greedy NMS has a prefix property: the survivors of the first T boxes (in visiting order) are
// final, and every later box they overlap is certainly suppressed.  For clustered detections the
// top T boxes kill most of the rest, so the big IoU matrix is only built over what remains.
//
// suppress: dead[j] = 1 iff a stage-A survivor overlaps box j (j >= T).  Thread per box, survivors
// staged in shared memory 256 at a time.
template <bool CLS>
__global__ void __launch_bounds__(256)
nms_suppress_kernel(const float4 *__restrict__ boxes, const float *__restrict__ areas, const int *__restrict__ cls,
                    int T, int n, const int *__restrict__ keepA, const int *__restrict__ numA, float thresh,
                    unsigned char *__restrict__ dead, const int *__restrict__ skip)
{
    if (skip && *skip == 1) return;
    __shared__ float4 s_box[256];
    __shared__ float s_area[256];
    __shared__ int s_cls[256];
    const int j = T + blockIdx.x * 256 + threadIdx.x;
    const int nk = *numA;
    float4 bj = make_float4(0.f, 0.f, 0.f, 0.f);
    float aj = 0.f;
    int cj = 0;
    if (j < n) { bj = boxes[j]; aj = areas[j]; if (CLS) cj = cls[j]; }
    bool hit = false;
    for (int k0 = 0; k0 < nk; k0 += 256) {
        const int kk = k0 + threadIdx.x;
        if (kk < nk) {
            const int pos = keepA[kk];
            s_box[threadIdx.x] = boxes[pos];
            s_area[threadIdx.x] = areas[pos];
            if (CLS) s_cls[threadIdx.x] = cls[pos];
        }
        __syncthreads();
        const int m = min(256, nk - k0);
        if (j < n && !hit) {
            for (int k = 0; k < m; ++k) {
                bool h = iou_ge(s_box[k], s_area[k], bj, aj, thresh);
                if (CLS) h = h && (s_cls[k] == cj);
                if (h) { hit = true; break; }
            }
        }
        __syncthreads();
    }
    if (j < n) dead[j - T] = hit ? 1 : 0;
}

// compact: ordered (stable) compaction of the boxes j >= T that survived stage A into a second,
// smaller problem.  Single CTA; the visiting order is preserved, so stage B is again a greedy NMS.
__global__ void __launch_bounds__(1024)
nms_compact_kernel(const float4 *__restrict__ boxes, const float *__restrict__ areas, const int *__restrict__ cls,
                   const int *__restrict__ order, const unsigned char *__restrict__ dead, int T, int n,
                   float4 *__restrict__ boxes2, float *__restrict__ areas2, int *__restrict__ cls2,
                   int *__restrict__ order2, int *__restrict__ n2_out, const int *__restrict__ skip)
{
    if (skip && *skip == 1) return;
    __shared__ int s_warp[32];
    __shared__ int s_base;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int start = T; start < n; start += 1024) {
        const int j = start + tid;
        const bool take = j < n && !dead[j - T];
        const unsigned m = __ballot_sync(0xffffffffu, take);
        if (lane == 0) s_warp[warp] = __popc(m);
        __syncthreads();
        int off = s_base, total = 0;
        for (int k = 0; k < 32; ++k) {
            const int c = s_warp[k];
            if (k < warp) off += c;
            total += c;
        }
        if (take) {
            const int d = off + __popc(m & ((1u << lane) - 1u));
            boxes2[d] = boxes[j];
            areas2[d] = areas[j];
            if (cls) cls2[d] = cls[j];
            order2[d] = order ? order[j] : j;
        }
        __syncthreads();
        if (tid == 0) s_base += total;
        __syncthreads();
    }
    if (tid == 0) *n2_out = s_base;
}

// ---------------------------------------------------------------------------
// 5. sparse path: spatial binning -> exact pair tests on neighbours only -> in-CTA fixed point
// ---------------------------------------------------------------------------
// The dense pipeline above tests all n(n-1)/2 pairs (72 M at 12k boxes) although only a few edges per
// box exist.  A pair can only satisfy IoU >= t if the boxes' centres are close:
//   with W = x2-x1+1 (the reference's +1 widths), w = overlap length along x, IoU >= t implies
//   w >= t*max(W_a, W_b), W_b in [t*W_a, W_a/t] and w <= (W_a+W_b)/2 - |cx_a - cx_b|, hence
//   |cx_a - cx_b| <= W_a * (1-t) * max(1, 1/(2t))            (same along y).
// Boxes are bucketed by centre on a G x G grid (x CB class buckets for the class-aware call); a warp per
// box walks the cell rows its window meets and runs the SAME exact iou_ge test as the mask kernel on those
// candidates only.  Every hit (a before b in visiting order) becomes one packed edge (b << 16 | a).
// A single CTA then iterates  K <- { b : no a in K with edge a->b }  from K = all boxes to the fixed point
// -- the greedy survivor set, see section 4b -- with K in shared memory, and emits in visiting order.
// The window carries 1 % + 0.5 px of slack against fp32 rounding (coordinates are bounded by 32768, so one
// rounding is <= 0.004 px); the result does not depend on the order of cells, candidates or edges.
// Contract: 64 < n <= 65535, t >= 0.05, finite boxes with x2 >= x1, y2 >= y1, |coordinate| <= 32768, at
// most SP_EDGES_PER_BOX*n edges, fixed point within SP_MAX_ROUNDS rounds.  Anything else leaves status at 0
// and the dense kernels (launched right after; they exit at once when status == 1) produce the result.
constexpr int SP_MAX_N = 65535;
constexpr int SP_MIN_N = 65;
constexpr int SP_MAX_CELLS = 4096;
constexpr int SP_EDGES_PER_BOX = 16;
constexpr int SP_BIN_THREADS = 1024;
#ifndef SLN_SP_PAIR_WARPS
#define SLN_SP_PAIR_WARPS 8
#endif
#ifndef SLN_SP_PAIR_CTAS_PER_SM
#define SLN_SP_PAIR_CTAS_PER_SM 8
#endif
constexpr int SP_PAIR_WARPS = SLN_SP_PAIR_WARPS;
#ifndef SLN_SP_PAIR_UNROLL
#define SLN_SP_PAIR_UNROLL 4
#endif
constexpr int SP_PAIR_UNROLL = SLN_SP_PAIR_UNROLL;   // candidates per lane in flight
constexpr int SP_INLINE = 32;              // predecessors stored inline per box (one 64-byte row)
constexpr int SP_INL_V = SP_INLINE / 8;    // uint4 per row
constexpr int SP_WARP_BUF = 128;           // edges buffered per warp before one atomic allocation
constexpr int SP_MAX_ROUNDS = 96;
constexpr int SP_RESOLVE_THREADS = 1024;
constexpr float SP_MAX_COORD = 32768.f;
constexpr int SP_CLUSTER = 8;             // CTAs of the bin and resolve clusters

struct SparseHdr {
    int status;            // 1: the sparse path produced the result
    int bail;              // 1: outside the contract -> dense path
    unsigned edge_count;
    int G, CB;
    float minx, miny, invx, invy;
};

struct SparseBufs {
    SparseHdr *hdr;
    int *cell_start;       // [CB*G*G + 1]
    float4 *cbox;          // boxes / areas / positions / classes sorted by cell
    float *carea;
    int *cpos;
    int *ccls;
    uint4 *inl;            // [n][SP_INL_V] the first SP_INLINE predecessors of every box as u16 (0xffff: none)
    int2 *seg;             // [n] (first entry, count) of the rest of the list in `edges`
    unsigned *edges;       // [SP_EDGES_PER_BOX * n] overflow predecessor positions, grouped by box
};

static size_t nms_sparse_bytes(int n)
{
    if (n > SP_MAX_N) return 256;
    size_t b = 256;
    b += align_up(sizeof(int) * (SP_MAX_CELLS + 1), 256);
    b += align_up(sizeof(float4) * (size_t)n, 256);
    b += 3 * align_up(sizeof(int) * (size_t)n, 256);
    b += align_up(sizeof(int2) * (size_t)n, 256);
    b += align_up(sizeof(uint4) * SP_INL_V * (size_t)n, 256);
    b += align_up(sizeof(unsigned) * (size_t)SP_EDGES_PER_BOX * n, 256);
    return b;
}

static void sparse_carve(void *ws, int n, SparseBufs &b)
{
    unsigned char *p = static_cast<unsigned char *>(ws);
    b.hdr = reinterpret_cast<SparseHdr *>(p);     p += 256;
    b.cell_start = reinterpret_cast<int *>(p);    p += align_up(sizeof(int) * (SP_MAX_CELLS + 1), 256);
    b.cbox = reinterpret_cast<float4 *>(p);       p += align_up(sizeof(float4) * (size_t)n, 256);
    b.carea = reinterpret_cast<float *>(p);       p += align_up(sizeof(int) * (size_t)n, 256);
    b.cpos = reinterpret_cast<int *>(p);          p += align_up(sizeof(int) * (size_t)n, 256);
    b.ccls = reinterpret_cast<int *>(p);          p += align_up(sizeof(int) * (size_t)n, 256);
    b.seg = reinterpret_cast<int2 *>(p);          p += align_up(sizeof(int2) * (size_t)n, 256);
    b.inl = reinterpret_cast<uint4 *>(p);         p += align_up(sizeof(uint4) * SP_INL_V * (size_t)n, 256);
    b.edges = reinterpret_cast<unsigned *>(p);
}

// monotone in v (every fp32 operation is), so lo <= v <= hi implies cell(lo) <= cell(v) <= cell(hi)
__device__ __forceinline__ int sp_cell(float v, float minv, float inv, int G)
{
    const float f = floorf(__fmul_rn(__fsub_rn(v, minv), inv));
    return (int)fminf(fmaxf(f, 0.f), (float)(G - 1));
}

__device__ __forceinline__ bool sp_sane(const float4 b)
{
    return fabsf(b.x) <= SP_MAX_COORD && fabsf(b.y) <= SP_MAX_COORD && fabsf(b.z) <= SP_MAX_COORD &&
           fabsf(b.w) <= SP_MAX_COORD && b.z >= b.x && b.w >= b.y;       // false for NaN / inf
}

// One cluster of SP_CLUSTER CTAs: bounds of the centres, cell histogram, exclusive scan, scatter into cell order
// (a counting sort by cell).  CTA c owns the boxes i = c*1024 + tid + k*8192; partial bounds and histograms are
// exchanged through distributed shared memory, every CTA scans the summed histogram itself, and its scatter
// cursor of a cell starts after the boxes of lower-ranked CTAs.  A single CTA was bound by the scattered 36k
// 4..16-byte stores of one SM (31 us at 12k boxes); the cluster spreads them over 8 SMs.
constexpr int SP_BIN_ITEMS = (SP_MAX_N + SP_CLUSTER * SP_BIN_THREADS - 1) / (SP_CLUSTER * SP_BIN_THREADS);   // 8

template <bool CLS>
__device__ __forceinline__ void nms_bin_body(const float4 *boxes, const float *areas,
                                             const int *cls, int n, int G, int CB, SparseBufs sb,
                                             int *num_keep_preset)
{
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    __shared__ int s_hist[SP_MAX_CELLS];           // this CTA's counts (read by the whole cluster)
    __shared__ int s_cur[SP_MAX_CELLS];            // this CTA's scatter cursors
    __shared__ float s_red[4][SP_BIN_THREADS / 32];
    __shared__ float s_part[5];                    // this CTA's bounds + bad flag (read by the whole cluster)
    __shared__ int s_warp[SP_BIN_THREADS / 32];
    __shared__ int s_slice_tot;
    pdl_prologue();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int crank = (int)cluster.block_rank();
    const int NC = CB * G * G;
    constexpr int STEP = SP_CLUSTER * SP_BIN_THREADS;
    // sparse-only mode (SLN_NMS_SPARSE_ONLY): no dense kernels follow, a bail-out is reported as num_keep = -1
    if (num_keep_preset && crank == 0 && tid == 0) *num_keep_preset = -1;
    for (int k = tid; k < NC; k += SP_BIN_THREADS) s_hist[k] = 0;
    // ---- my boxes: loaded once (all loads in flight), kept in registers
    float4 v[SP_BIN_ITEMS];
    const int first = crank * SP_BIN_THREADS + tid;
#pragma unroll
    for (int u = 0; u < SP_BIN_ITEMS; ++u) {
        const int i = first + u * STEP;
        if (i < n) v[u] = boxes[i];
    }
    float mnx = 3.0e38f, mny = 3.0e38f, mxx = -3.0e38f, mxy = -3.0e38f;
    bool bad = false;
#pragma unroll
    for (int u = 0; u < SP_BIN_ITEMS; ++u) {
        if (first + u * STEP < n) {
            const float4 b = v[u];
            bad = bad || !sp_sane(b);
            const float cx = __fmul_rn(0.5f, __fadd_rn(b.x, b.z)), cy = __fmul_rn(0.5f, __fadd_rn(b.y, b.w));
            mnx = fminf(mnx, cx); mxx = fmaxf(mxx, cx);
            mny = fminf(mny, cy); mxy = fmaxf(mxy, cy);
        }
    }
    auto warp_bounds = [&]() {
        for (int o = 16; o > 0; o >>= 1) {
            mnx = fminf(mnx, __shfl_xor_sync(0xffffffffu, mnx, o));
            mny = fminf(mny, __shfl_xor_sync(0xffffffffu, mny, o));
            mxx = fmaxf(mxx, __shfl_xor_sync(0xffffffffu, mxx, o));
            mxy = fmaxf(mxy, __shfl_xor_sync(0xffffffffu, mxy, o));
        }
    };
    warp_bounds();
    if (lane == 0) { s_red[0][warp] = mnx; s_red[1][warp] = mny; s_red[2][warp] = mxx; s_red[3][warp] = mxy; }
    const int any_bad = __syncthreads_or(bad);
    if (warp == 0) {
        mnx = s_red[0][lane]; mny = s_red[1][lane]; mxx = s_red[2][lane]; mxy = s_red[3][lane];
        warp_bounds();
        if (lane == 0) { s_part[0] = mnx; s_part[1] = mny; s_part[2] = mxx; s_part[3] = mxy; s_part[4] = any_bad ? 1.f : 0.f; }
    }
    cluster.sync();
    float badf = 0.f;
    mnx = 3.0e38f; mny = 3.0e38f; mxx = -3.0e38f; mxy = -3.0e38f;
#pragma unroll
    for (int c = 0; c < SP_CLUSTER; ++c) {
        const float *q = cluster.map_shared_rank(s_part, c);
        mnx = fminf(mnx, q[0]); mny = fminf(mny, q[1]); mxx = fmaxf(mxx, q[2]); mxy = fmaxf(mxy, q[3]);
        badf = fmaxf(badf, q[4]);
    }
    if (badf != 0.f) {                             // uniform over the cluster
        if (crank == 0 && tid == 0) { sb.hdr->status = 0; sb.hdr->bail = 1; sb.hdr->edge_count = 0u; }
        cluster.sync();                            // nobody leaves while its s_part may still be read
        return;
    }
    const float invx = __fdiv_rn((float)G, fmaxf(__fsub_rn(mxx, mnx), 1e-3f));
    const float invy = __fdiv_rn((float)G, fmaxf(__fsub_rn(mxy, mny), 1e-3f));
    if (crank == 0 && tid == 0) {
        sb.hdr->status = 0; sb.hdr->bail = 0; sb.hdr->edge_count = 0u;
        sb.hdr->G = G; sb.hdr->CB = CB;
        sb.hdr->minx = mnx; sb.hdr->miny = mny; sb.hdr->invx = invx; sb.hdr->invy = invy;
    }
    // ---- keys and this CTA's histogram
    int key[SP_BIN_ITEMS];
#pragma unroll
    for (int u = 0; u < SP_BIN_ITEMS; ++u) {
        const int i = first + u * STEP;
        key[u] = 0;
        if (i < n) {
            const float4 b = v[u];
            const float cx = __fmul_rn(0.5f, __fadd_rn(b.x, b.z)), cy = __fmul_rn(0.5f, __fadd_rn(b.y, b.w));
            const int cb = CLS ? (int)((unsigned)cls[i] % (unsigned)CB) : 0;
            key[u] = (cb * G + sp_cell(cy, mny, invy, G)) * G + sp_cell(cx, mnx, invx, G);
            atomicAdd(&s_hist[key[u]], 1);
        }
    }
    cluster.sync();
    // ---- CTA c sums the 8 histograms over ITS slice of the cells (one cell per thread, consecutive lanes =
    // consecutive cells: each remote access is one coalesced row), scans the slice, and hands every CTA its
    // scatter cursors -- 16 DSMEM accesses per thread instead of every CTA reading every histogram
    {
        const int slice = (NC + SP_CLUSTER - 1) / SP_CLUSTER;   // <= 512
        const int k = crank * slice + tid;
        const bool mine = tid < slice && k < NC;
        int hc[SP_CLUSTER], tot = 0;
#pragma unroll
        for (int c = 0; c < SP_CLUSTER; ++c) {
            hc[c] = mine ? *cluster.map_shared_rank(s_hist + k, c) : 0;
            tot += hc[c];
        }
        int incl = tot;
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            int w = s_warp[lane], wi = w;
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, wi, o);
                if (lane >= o) wi += t;
            }
            s_warp[lane] = wi - w;
            if (lane == 31) s_slice_tot = wi;      // boxes in my slice of the cells
        }
        __syncthreads();
        const int local_excl = s_warp[warp] + incl - tot;
        cluster.sync();                            // slice totals visible
        int slice_off = 0;
#pragma unroll
        for (int c = 0; c < SP_CLUSTER; ++c) {
            const int t = *cluster.map_shared_rank(&s_slice_tot, c);
            if (c < crank) slice_off += t;
        }
        if (mine) {
            int run = slice_off + local_excl;
            sb.cell_start[k] = run;
#pragma unroll
            for (int c = 0; c < SP_CLUSTER; ++c) {
                *cluster.map_shared_rank(s_cur + k, c) = run;
                run += hc[c];
            }
        }
        if (crank == 0 && tid == 0) sb.cell_start[NC] = n;
    }
    cluster.sync();                                // cursors ready; nobody reads s_hist remotely after this point
    // ---- scatter my boxes (re-read: L1/L2 hits; keeping them in registers across the exchange spills)
#pragma unroll
    for (int u = 0; u < SP_BIN_ITEMS; ++u) {
        const int i = first + u * STEP;
        if (i < n) {
            const int p = atomicAdd(&s_cur[key[u]], 1);        // order inside a cell is irrelevant to the result
            sb.cbox[p] = boxes[i];
            sb.carea[p] = areas[i];
            sb.cpos[p] = i;
            if (CLS) sb.ccls[p] = cls[i];
        }
    }
}

template <bool CLS>
__global__ void __cluster_dims__(SP_CLUSTER, 1, 1) __launch_bounds__(SP_BIN_THREADS)
nms_bin_kernel(const float4 *__restrict__ boxes, const float *__restrict__ areas, const int *__restrict__ cls, int n,
               int G, int CB, SparseBufs sb, int *__restrict__ num_keep_preset)
{
    nms_bin_body<CLS>(boxes, areas, cls, n, G, CB, sb, num_keep_preset);
}

// problem b of a batched call (nms_sorted_batched_launch): every buffer moved by b * stride bytes
__device__ __forceinline__ SparseBufs sparse_at(SparseBufs sb, size_t stride, int b)
{
    sb.hdr = seg_at(sb.hdr, stride, b);
    sb.cell_start = seg_at(sb.cell_start, stride, b);
    sb.cbox = seg_at(sb.cbox, stride, b);
    sb.carea = seg_at(sb.carea, stride, b);
    sb.cpos = seg_at(sb.cpos, stride, b);
    sb.ccls = seg_at(sb.ccls, stride, b);
    sb.inl = seg_at(sb.inl, stride, b);
    sb.seg = seg_at(sb.seg, stride, b);
    sb.edges = seg_at(sb.edges, stride, b);
    return sb;
}

// grid (SP_CLUSTER, B): the cluster of blockIdx.y bins problem blockIdx.y
template <bool CLS>
__global__ void __cluster_dims__(SP_CLUSTER, 1, 1) __launch_bounds__(SP_BIN_THREADS)
nms_bin_seg_kernel(const float4 *__restrict__ boxes, const float *__restrict__ areas, const int *__restrict__ cls, int n,
                   int G, int CB, SparseBufs sb, size_t stride)
{
    const int b = blockIdx.y;
    nms_bin_body<CLS>(seg_at(boxes, stride, b), seg_at(areas, stride, b), CLS ? seg_at(cls, stride, b) : nullptr, n, G, CB,
                      sparse_at(sb, stride, b), nullptr);
}

// warp per box (grid-strided): exact tests against the boxes binned in the window's cells.  The window's cell
// rows are contiguous ranges of the cell-sorted arrays; their (start, running count) table is built once per box
// in shared memory (one row per lane, all loads in flight together) and the lanes then walk the concatenation of
// the ranges, so every pass tests 32 candidates whatever the row lengths are.
template <bool CLS>
__device__ __forceinline__ void nms_pairs_body(const float4 *boxes, const float *areas,
                                               const int *cls, int n, float thresh, float ct, unsigned edge_cap,
                                               SparseBufs sb)
{
    __shared__ unsigned s_buf[SP_PAIR_WARPS][SP_WARP_BUF];
    __shared__ int s_rs[SP_PAIR_WARPS][64];        // first item of each window row
    __shared__ int s_ri[SP_PAIR_WARPS][64];        // inclusive running count of candidates
    pdl_prologue();
    const SparseHdr h = *sb.hdr;
    if (h.bail) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned *buf = s_buf[warp];
    int *rs = s_rs[warp], *ri = s_ri[warp];
    int cnt = 0;                                   // warp-uniform: predecessors of the current box found so far
    const int G = h.G;                             // <= 64
    for (int b = blockIdx.x * SP_PAIR_WARPS + warp; b < n; b += gridDim.x * SP_PAIR_WARPS) {
        if (b == 0) {                              // nothing precedes the first box
            if (lane == 0) sb.seg[0] = make_int2(0, 0);
            if (lane < SP_INLINE) reinterpret_cast<unsigned short *>(sb.inl)[lane] = 0xffffu;
            continue;
        }
        const float4 bb = boxes[b];
        const float ab = areas[b];
        const int cbk = CLS ? cls[b] : 0;
        const float rx = __fadd_rn(__fmul_rn(__fadd_rn(__fsub_rn(bb.z, bb.x), 1.f), ct), 0.5f);
        const float ry = __fadd_rn(__fmul_rn(__fadd_rn(__fsub_rn(bb.w, bb.y), 1.f), ct), 0.5f);
        const float cx = __fmul_rn(0.5f, __fadd_rn(bb.x, bb.z)), cy = __fmul_rn(0.5f, __fadd_rn(bb.y, bb.w));
        const int ix0 = sp_cell(__fsub_rn(cx, rx), h.minx, h.invx, G), ix1 = sp_cell(__fadd_rn(cx, rx), h.minx, h.invx, G);
        const int iy0 = sp_cell(__fsub_rn(cy, ry), h.miny, h.invy, G), iy1 = sp_cell(__fadd_rn(cy, ry), h.miny, h.invy, G);
        const int plane = CLS ? (int)((unsigned)cbk % (unsigned)h.CB) * G : 0;
        const int nrows = iy1 - iy0 + 1;
        int total = 0;
        __syncwarp();                              // the previous box's table reads are done
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int r = lane + 32 * half;
            int s = 0, c = 0;
            if (r < nrows) {
                const int row = (plane + iy0 + r) * G;
                s = __ldg(sb.cell_start + row + ix0);
                c = __ldg(sb.cell_start + row + ix1 + 1) - s;
            }
            int incl = c;
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            rs[r] = s;
            ri[r] = total + incl;
            total += __shfl_sync(0xffffffffu, incl, 31);
            if (nrows <= 32) break;                // warp-uniform
        }
        __syncwarp();
        int r = 0;                                 // this lane's current row (monotone in t)
        for (int t0 = 0; t0 < total; t0 += 32 * SP_PAIR_UNROLL) {
            // SP_PAIR_UNROLL candidates per lane, every load issued before the first test
            int a[SP_PAIR_UNROLL], cc[SP_PAIR_UNROLL];
            float4 cb[SP_PAIR_UNROLL];
            float ca[SP_PAIR_UNROLL];
#pragma unroll
            for (int u = 0; u < SP_PAIR_UNROLL; ++u) {
                const int t = t0 + 32 * u + lane;
                a[u] = 0x7fffffff;                 // "not a predecessor"
                if (t < total) {
                    while (t >= ri[r]) ++r;
                    const int k = rs[r] + (t - (r ? ri[r - 1] : 0));
                    a[u] = sb.cpos[k];
                    cb[u] = sb.cbox[k];
                    ca[u] = sb.carea[k];
                    if (CLS) cc[u] = sb.ccls[k];
                }
            }
#pragma unroll
            for (int u = 0; u < SP_PAIR_UNROLL; ++u) {
                if (t0 + 32 * u >= total) break;   // warp-uniform
                bool hit = false;
                if (a[u] < b && (!CLS || cc[u] == cbk)) hit = iou_ge(cb[u], ca[u], bb, ab, thresh);
                const unsigned m = __ballot_sync(0xffffffffu, hit);
                if (m) {
                    const int slot = cnt + __popc(m & ((1u << lane) - 1u));
                    if (hit && slot < SP_WARP_BUF) buf[slot] = (unsigned)a[u];
                    cnt += __popc(m);
                }
            }
        }
        // the box's predecessor list: the first SP_INLINE entries inline (u16, one 32-byte row per box), the rest
        // in one contiguous segment of `edges`
        if (cnt > SP_WARP_BUF) {                   // more predecessors than the sparse path budgets for one box
            if (lane == 0) sb.hdr->bail = 1;
            cnt = 0;
        }
        __syncwarp();
        if (lane < SP_INLINE)
            reinterpret_cast<unsigned short *>(sb.inl)[(size_t)b * SP_INLINE + lane] = lane < cnt ? (unsigned short)buf[lane] : (unsigned short)0xffffu;
        const int over = cnt > SP_INLINE ? cnt - SP_INLINE : 0;
        unsigned base = 0u;
        if (lane == 0 && over) base = atomicAdd(&sb.hdr->edge_count, (unsigned)over);
        base = __shfl_sync(0xffffffffu, base, 0);
        for (int k = lane; k < over; k += 32)
            if (base + k < edge_cap) sb.edges[base + k] = buf[SP_INLINE + k];
        if (lane == 0) sb.seg[b] = make_int2((int)base, over);
        cnt = 0;
        __syncwarp();
    }
}

template <bool CLS>
__global__ void __launch_bounds__(32 * SP_PAIR_WARPS)
nms_pairs_kernel(const float4 *__restrict__ boxes, const float *__restrict__ areas, const int *__restrict__ cls, int n,
                 float thresh, float ct, unsigned edge_cap, SparseBufs sb)
{
    nms_pairs_body<CLS>(boxes, areas, cls, n, thresh, ct, edge_cap, sb);
}

template <bool CLS>
__global__ void __launch_bounds__(32 * SP_PAIR_WARPS)
nms_pairs_seg_kernel(const float4 *__restrict__ boxes, const float *__restrict__ areas, const int *__restrict__ cls, int n,
                     float thresh, float ct, unsigned edge_cap, SparseBufs sb, size_t stride)
{
    const int b = blockIdx.y;
    nms_pairs_body<CLS>(seg_at(boxes, stride, b), seg_at(areas, stride, b), CLS ? seg_at(cls, stride, b) : nullptr, n, thresh,
                        ct, edge_cap, sparse_at(sb, stride, b));
}

// One cluster of SP_CLUSTER CTAs: the greedy survivor set from the predecessor lists, then ordered emission.
// Two monotone sets, full copies in every CTA's shared memory:  KF = boxes known kept, DF = boxes known dead.
//   box b is dead   as soon as one predecessor is in KF,
//   box b is kept   as soon as all predecessors are in DF          (no predecessors: kept at once).
// Both rules only ever state final facts, so the sets can be read while other CTAs extend them and the fixed point
// (every box decided) is the greedy result whatever the interleaving.
//
// Why the reads that compute-sanitizer's racecheck flags (a warp publishing KF / DF words through DSMEM while another
// warp reads the same words in sp_scan8, no barrier in between) cannot change the result -- the argument, in full:
//   (1) Single writer: word w of KF and of DF is written only by the one warp that owns w (CTA w % SP_CLUSTER, a fixed
//       warp of it), in all SP_CLUSTER copies.  A 32-bit shared-memory store is atomic, so a reader sees either the old
//       or the new word, never a mixture.
//   (2) Monotone: the owner only ever ORs bits in; a bit, once set, stays set in every copy.  A stale read therefore
//       shows a SUBSET of the true sets at that instant.
//   (3) Soundness by induction over the visiting order (the greedy NMS order, nms.c:25-67): assume every bit that is
//       set for a box a < b is correct (a in KF => greedy keeps a; a in DF => greedy suppresses a).  Rule "dead" sets
//       b in DF only after reading some predecessor a (IoU(a, b) >= t, a < b) in KF: greedy keeps a, so it suppresses b.
//       Rule "kept" sets b in KF only after reading ALL predecessors in DF: greedy suppressed every box that could have
//       suppressed b, so it keeps b.  Both conclusions need only that the bits READ were correct, which (2) and the
//       induction hypothesis give for any subset.  KF and DF stay disjoint because a box is decided once by its owner.
//   (4) Progress: the lowest undecided box has all its predecessors decided; after the next cluster barrier
//       (barrier.cluster.arrive.release / wait.acquire: every copy sees every earlier store) its owner decides it.
//       So every round decides at least one box, and the loop ends with KF = the greedy survivors exactly.  Early
//       visibility between barriers can only decide boxes SOONER (fewer rounds), never differently.
//   (5) The sentinel word 2047 (bit 31 clear in KF, set in DF) is written once before the first barrier and never again.
// tests/test_gpu_parity.py::test_nms_sparse_resolve_is_interleaving_independent repeats the same inputs a few hundred
// times (the hardware interleaving differs from launch to launch) and demands identical survivors every time.  Ownership: 32-box word w belongs to CTA
// w % SP_CLUSTER, one warp per word, lane = box; the warp builds the word's new bits with ballots and stores the
// updated words into all SP_CLUSTER copies through DSMEM.  One hardware cluster barrier per round; a box costs work only while it is undecided, and its inline
// predecessor row sits in the owner's shared memory (one coalesced 32-byte load per box).
constexpr int SP_WORDS = 2048;             // 32-bit words of KF / DF (n <= 65535)
constexpr int SP_RES_ITEMS = SP_WORDS / SP_CLUSTER / (SP_RESOLVE_THREADS / 32);       // words per warp: 8
constexpr int SP_CACHE_ITEMS = 2;          // items whose inline rows are cached in shared memory (64 KB each)
constexpr int SP_OV_CACHE = 8192;          // u16 overflow entries cached per resolve CTA (16 KB)

// Branch-free scan of 8 inline entries: the sentinel 0xffff addresses bit 31 of word 2047 (box 65535 does not
// exist), which is kept clear in KF and set in DF, so an empty slot reads as "dead predecessor".
__device__ __forceinline__ void sp_scan8(const unsigned *KF, const unsigned *DF, uint4 v, unsigned &anyK, unsigned &anyN)
{
    const unsigned w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const unsigned a = (w[q] >> (16 * h)) & 0xffffu;
            anyK |= KF[a >> 5] >> (a & 31u);
            anyN |= ~DF[a >> 5] >> (a & 31u);
        }
    }
}

__device__ __forceinline__ void nms_sparse_resolve_body(const int *order, int n, int max_keep, unsigned edge_cap,
                                                        SparseBufs sb, int64_t *keep64, int *keep32,
                                                        int *num_keep)
{
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    extern __shared__ __align__(16) unsigned char s_raw[];
    __shared__ int s_wsum[SP_RESOLVE_THREADS / 32];
    __shared__ unsigned s_used;
    pdl_prologue();
    if (sb.hdr->bail) return;                      // uniform over the cluster: nobody is left at a barrier
    if (sb.hdr->edge_count > edge_cap) return;     // status stays 0: dense path
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int crank = (int)cluster.block_rank();
    unsigned *KF = reinterpret_cast<unsigned *>(s_raw);         // [SP_WORDS]
    unsigned *DF = KF + SP_WORDS;                               // [SP_WORDS]
    int *flags = reinterpret_cast<int *>(DF + SP_WORDS);        // [2][SP_CLUSTER] (+ padding)
    unsigned short *ov = reinterpret_cast<unsigned short *>(flags + 32);          // [SP_OV_CACHE] overflow entries
    uint4 *rows = reinterpret_cast<uint4 *>(ov + SP_OV_CACHE);  // [cache items][SP_RESOLVE_THREADS][2]
    const int W32 = (n + 31) >> 5;
    const int n_items = (W32 + SP_CLUSTER * 32 - 1) / (SP_CLUSTER * 32);          // words per warp actually used
    for (int w = tid; w < SP_WORDS; w += SP_RESOLVE_THREADS) { KF[w] = 0u; DF[w] = w == SP_WORDS - 1 ? 0x80000000u : 0u; }
    if (tid < 32) flags[tid] = 0;
    if (tid == 0) s_used = 0u;
    __syncthreads();
    // ---- my boxes: word w = (warp + 32*u) * SP_CLUSTER + crank, box = 32*w + lane
    unsigned undecided = 0u;                       // bit u: my box of item u is not decided yet
    // rest of the predecessor list beyond the inline row: count << 24 | offset (bit 23 set: offset into the
    // shared-memory cache `ov`, else into sb.edges); 0 = none.  Lists are copied by the whole warp, coalesced.
    unsigned p_over[SP_RES_ITEMS];
#pragma unroll
    for (int u = 0; u < SP_RES_ITEMS; ++u) {
        const int w = (warp + 32 * u) * SP_CLUSTER + crank;
        const int b = 32 * w + lane;
        int2 sg = make_int2(0, 0);
        if (u < n_items && w < W32 && b < n) {
            undecided |= 1u << u;
            if (u < SP_CACHE_ITEMS) {
#pragma unroll
                for (int v = 0; v < SP_INL_V; ++v)
                    rows[(u * SP_RESOLVE_THREADS + tid) * SP_INL_V + v] = __ldg(sb.inl + SP_INL_V * (size_t)b + v);
            }
            sg = __ldg(sb.seg + b);
        }
        p_over[u] = sg.y > 0 ? ((unsigned)sg.y << 24) | (unsigned)sg.x : 0u;        // sg.x < 16 n <= 2^20
        // every long list's lines are requested at once (lane-parallel prefetch): the copies below, one list after
        // the other, then find them on their way instead of paying one cold miss each
        for (int k = 0; k < sg.y; k += 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(sb.edges + sg.x + k));
        unsigned m = __ballot_sync(0xffffffffu, sg.y > 0);
        while (m) {
            const int L = __ffs(m) - 1;
            m &= m - 1u;
            const int st = __shfl_sync(0xffffffffu, sg.x, L), cn = __shfl_sync(0xffffffffu, sg.y, L);
            unsigned off = 0u;
            if (lane == 0) off = atomicAdd(&s_used, (unsigned)cn);
            off = __shfl_sync(0xffffffffu, off, 0);
            if (off + (unsigned)cn <= (unsigned)SP_OV_CACHE) {
                for (int k = lane; k < cn; k += 32) ov[off + k] = (unsigned short)__ldg(sb.edges + st + k);
                if (lane == L) p_over[u] = ((unsigned)cn << 24) | 0x800000u | off;
            }
        }
    }
    cluster.sync();                                // every CTA's shared memory is initialised before remote access
    bool done = false;
    for (int round = 0; round < SP_MAX_ROUNDS; ++round) {
#pragma unroll
        for (int u = 0; u < SP_RES_ITEMS; ++u) {
            if (u >= n_items) break;
            const int w = (warp + 32 * u) * SP_CLUSTER + crank;
            if (w >= W32) break;                   // warp-uniform
            if (__ballot_sync(0xffffffffu, (undecided >> u) & 1u) == 0u) continue;
            bool dead = false, kept = false, need_rest = false, all_dead_reg = true;
            if ((undecided >> u) & 1u) {
                const int b = 32 * w + lane;
                unsigned anyK = 0u, anyN = 0u;
                bool row_empty = false;
                // 8 entries at a time; rows are filled front to back, so the scan stops at the first chunk that
                // starts with the sentinel.  Round 0 knows (almost) nothing yet: only the first chunk is looked at,
                // a box without predecessors is kept at once, and no other box may be declared kept from a partial
                // scan (bits published by faster CTAs can already be visible).
#pragma unroll
                for (int v = 0; v < SP_INL_V; ++v) {
                    if (round == 0 && v > 0) break;
                    const uint4 rv = u < SP_CACHE_ITEMS ? rows[(u * SP_RESOLVE_THREADS + tid) * SP_INL_V + v]
                                                        : __ldg(sb.inl + SP_INL_V * (size_t)b + v);
                    if ((rv.x & 0xffffu) == 0xffffu) { row_empty = v == 0; break; }
                    sp_scan8(KF, DF, rv, anyK, anyN);
                }
                dead = anyK & 1u;
                const bool all_dead = round == 0 ? row_empty : !(anyN & 1u);
                all_dead_reg = all_dead;
                need_rest = !dead && p_over[u] != 0u && round > 0;
                kept = !dead && all_dead && !need_rest;
                if (dead || kept) undecided &= ~(1u << u);
            }
            // the rest of a long list: scanned by the whole warp, 32 entries per step
            unsigned m = __ballot_sync(0xffffffffu, need_rest);
            while (m) {
                const int L = __ffs(m) - 1;
                m &= m - 1u;
                const unsigned po = __shfl_sync(0xffffffffu, p_over[u], L);
                const int cn = (int)(po >> 24);
                const unsigned off = po & 0x7fffffu;
                bool hitK = false, notD = false;
                for (int k = lane; k < cn; k += 32) {
                    const unsigned a = (po & 0x800000u) ? (unsigned)ov[off + k] : __ldg(sb.edges + off + k);
                    const unsigned bit = 1u << (a & 31u);
                    if (KF[a >> 5] & bit) hitK = true;
                    else if (!(DF[a >> 5] & bit)) notD = true;
                }
                const bool anyK = __any_sync(0xffffffffu, hitK), anyN = __any_sync(0xffffffffu, notD);
                if (lane == L) {
                    dead = anyK;
                    kept = !anyK && all_dead_reg && !anyN;
                    if (dead || kept) undecided &= ~(1u << u);
                }
            }
            const unsigned kb = __ballot_sync(0xffffffffu, kept), db = __ballot_sync(0xffffffffu, dead);
            // (compute-sanitizer racecheck flags these stores against the reads in sp_scan8: that is the documented,
            // deliberate overlap -- 32-bit words, a single writer per word, bits only ever set, and either value a
            // reader can see is a valid state of the monotone sets)
            if (kb | db) {                         // the warp owns this word: plain stores of the updated words
                const unsigned nk = KF[w] | kb, nd = DF[w] | db;
                if (lane < SP_CLUSTER) {
                    *cluster.map_shared_rank(KF + w, lane) = nk;
                    *cluster.map_shared_rank(DF + w, lane) = nd;
                }
            }
        }
        // termination: every CTA tells every CTA whether it still has open boxes.  The flag words are double-buffered
        // by round parity, so the single barrier of the round is enough: a buffer is rewritten two rounds later, after
        // a barrier every CTA only reaches once it has read the old value.
        const int open = __syncthreads_or(undecided != 0u);
        if (tid < SP_CLUSTER) *cluster.map_shared_rank(flags + (round & 1) * SP_CLUSTER + crank, tid) = open;
        cluster.sync();
        int glob = 0;
#pragma unroll
        for (int c = 0; c < SP_CLUSTER; ++c) glob |= flags[(round & 1) * SP_CLUSTER + c];
        if (!glob) { done = true; break; }         // uniform over the cluster
    }
    if (!done) return;
    // ---- emission in visiting order: every CTA scans the per-word popcounts itself (2 words per thread) and
    // writes the survivors of the positions it owns
    const int c0 = __popc(KF[2 * tid]), c1 = __popc(KF[2 * tid + 1]);
    const int mine2 = c0 + c1;
    int incl = mine2;
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) s_wsum[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = s_wsum[lane], wi = w;
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += t;
        }
        s_wsum[lane] = wi - w;
    }
    __syncthreads();
    int *pre = reinterpret_cast<int *>(DF);        // DF is free now
    const int excl = s_wsum[warp] + incl - mine2;
    pre[2 * tid] = excl;
    pre[2 * tid + 1] = excl + c0;
    __syncthreads();
    for (int pos = crank * SP_RESOLVE_THREADS + tid; pos < n; pos += SP_CLUSTER * SP_RESOLVE_THREADS) {
        const unsigned kw = KF[pos >> 5];
        if ((kw >> (pos & 31)) & 1u) {
            const int slot = pre[pos >> 5] + __popc(kw & ((1u << (pos & 31)) - 1u));
            if (slot < max_keep) {
                const int idx = order ? order[pos] : pos;
                if (keep64) keep64[slot] = idx;
                if (keep32) keep32[slot] = idx;
            }
        }
    }
    if (crank == 0 && tid == SP_RESOLVE_THREADS - 1) {
        *num_keep = min(excl + mine2, max_keep);
        sb.hdr->status = 1;
    }
}

__global__ void __cluster_dims__(SP_CLUSTER, 1, 1) __launch_bounds__(SP_RESOLVE_THREADS, 1)
nms_sparse_resolve_kernel(const int *__restrict__ order, int n, int max_keep, unsigned edge_cap, SparseBufs sb,
                          int64_t *__restrict__ keep64, int *__restrict__ keep32, int *__restrict__ num_keep)
{
    nms_sparse_resolve_body(order, n, max_keep, edge_cap, sb, keep64, keep32, num_keep);
}

// grid (SP_CLUSTER, B): one cluster per problem; clusters beyond the GPU's cluster capacity queue.  order and the
// workspace move by `stride`; the outputs (keep64 or keep32, and num_keep) by their own strides, in bytes, so that
// they can live in the workspace or in a caller's [B, max_keep] / [B] arrays.  Null pointers stay null.
__global__ void __cluster_dims__(SP_CLUSTER, 1, 1) __launch_bounds__(SP_RESOLVE_THREADS, 1)
nms_sparse_resolve_seg_kernel(const int *__restrict__ order, int n, int max_keep, unsigned edge_cap, SparseBufs sb,
                              int64_t *__restrict__ keep64, int *__restrict__ keep32, size_t keep_stride,
                              int *__restrict__ num_keep, size_t num_stride, size_t stride)
{
    const int b = blockIdx.y;
    nms_sparse_resolve_body(order ? seg_at(order, stride, b) : nullptr, n, max_keep, edge_cap, sparse_at(sb, stride, b),
                            keep64 ? seg_at(keep64, keep_stride, b) : nullptr, keep32 ? seg_at(keep32, keep_stride, b) : nullptr,
                            seg_at(num_keep, num_stride, b));
}

// grid: ~3 boxes per cell; the class-aware call spends the cells on class buckets first.  ct: the window's half-width
// per unit of box width (see the contract above nms_bin_kernel)
static void sparse_params(int n, bool has_cls, float thresh, int &CB, int &G, float &ct)
{
    CB = 1; G = 64;
    if (has_cls) { CB = 64; G = 8; }
    while (G > 8 && (long long)CB * G * G > (long long)n / 2) G >>= 1;
    const float t = thresh > 1.f ? 1.f : thresh;
    ct = (1.f - t) * (t < 0.5f ? 0.5f / t : 1.f) * 1.01f;
}

static size_t sparse_resolve_smem(int n)
{
    int items = cdiv(cdiv(n, 32), SP_CLUSTER * 32);
    if (items > SP_CACHE_ITEMS) items = SP_CACHE_ITEMS;
    return sizeof(unsigned) * (2 * SP_WORDS + 32) + 2 * SP_OV_CACHE + (size_t)items * SP_RESOLVE_THREADS * sizeof(uint4) * SP_INL_V;
}

// returns the device address of the status word the dense kernels test (nullptr: sparse path not taken)
static int launch_sparse(const float4 *boxes, const float *areas, const int *cls, const int *order, int n, float thresh,
                         int max_keep, int64_t *keep64, int *keep32, int *num_keep, void *sparse, cudaStream_t st,
                         const int **skip_out, bool sparse_only)
{
    *skip_out = nullptr;
    if (sparse == nullptr || n < SP_MIN_N || n > SP_MAX_N || !(thresh >= 0.05f)) return SLN_OK;
    SparseBufs sb;
    sparse_carve(sparse, n, sb);
    int CB, G;
    float ct;
    sparse_params(n, cls != nullptr, thresh, CB, G, ct);
    const unsigned edge_cap = (unsigned)SP_EDGES_PER_BOX * (unsigned)n;
    // rank -> bin -> pairs -> resolve is a chain of short kernels: programmatic dependent launches (common.cuh)
    int *preset = sparse_only ? num_keep : nullptr;
    SLN_CUDA_OK(launch_chain(cls ? nms_bin_kernel<true> : nms_bin_kernel<false>, dim3(SP_CLUSTER), dim3(SP_BIN_THREADS), 0, st,
                             true, boxes, areas, cls, n, G, CB, sb, preset));
    int ctas = cdiv(n, SP_PAIR_WARPS);
    if (ctas > SLN_SP_PAIR_CTAS_PER_SM * sm_count()) ctas = SLN_SP_PAIR_CTAS_PER_SM * sm_count();
    SLN_CUDA_OK(launch_chain(cls ? nms_pairs_kernel<true> : nms_pairs_kernel<false>, dim3(ctas), dim3(32 * SP_PAIR_WARPS), 0, st,
                             true, boxes, areas, cls, n, thresh, ct, edge_cap, sb));
    const size_t smem = sparse_resolve_smem(n);
    SLN_CUDA_OK(cudaFuncSetAttribute(nms_sparse_resolve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    SLN_CUDA_OK(launch_chain(nms_sparse_resolve_kernel, dim3(SP_CLUSTER), dim3(SP_RESOLVE_THREADS), smem, st, true, order, n,
                             max_keep, edge_cap, sb, keep64, keep32, num_keep));
    *skip_out = &sb.hdr->status;
    return SLN_OK;
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
static size_t scan_smem_bytes(int W)
{
    return sizeof(unsigned long long) * ((size_t)W + 2 * (size_t)SS_ROWS * BAND_STRIDE) + sizeof(int) * 2 * SS_ROWS;
}

__global__ void nms_emit_stageA_kernel(const int *__restrict__ keepA, const int *__restrict__ numA,
                                       const int *__restrict__ order, int64_t *__restrict__ keep64,
                                       int *__restrict__ keep32, const int *__restrict__ skip)
{
    if (skip && *skip == 1) return;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= *numA) return;
    const int pos = keepA[i];
    const int idx = order ? order[pos] : pos;
    if (keep64) keep64[i] = idx;
    if (keep32) keep32[i] = idx;
}

static size_t nms_fix_bytes(int n_max);

constexpr int NMS_STAGE_A = 1024;          // boxes resolved by the first stage
constexpr int NMS_TWO_STAGE_MIN = 16384;   // below this one stage is cheaper (measured: no gain at 12k, loss at 6k)

static bool nms_two_stage(int n) { return n >= NMS_TWO_STAGE_MIN; }

size_t nms_buffers_bytes(int n)
{
    // one stage: mask over n.  two stages: mask over T (stage A) and over the n-T that may remain (stage B)
    const size_t nm = nms_two_stage(n) ? (size_t)(n - NMS_STAGE_A) : (size_t)n;
    const size_t W = (size_t)cdiv((int)nm, 64);
    size_t b = 0;
    b += align_up(sizeof(float4) * (size_t)n, 256);
    b += align_up(sizeof(float) * (size_t)n, 256);
    b += 3 * align_up(sizeof(int) * (size_t)n, 256);
    b += align_up(sizeof(int) * (size_t)cdiv(n, RANK_ROWS), 256);          // tickets (right after rank: one memset)
    b += align_up(sizeof(unsigned long long) * nm * W, 256);
    b += 2 * nms_fix_bytes(n);
    b += nms_sparse_bytes(n);
    if (nms_two_stage(n)) {
        b += align_up(sizeof(unsigned long long) * (size_t)NMS_STAGE_A * (NMS_STAGE_A / 64), 256);   // stage-A mask
        b += align_up(sizeof(float4) * nm, 256) + align_up(sizeof(float) * nm, 256);                   // boxes2, areas2
        b += 2 * align_up(sizeof(int) * nm, 256);                                                     // cls2, order2
        b += align_up(sizeof(int) * (size_t)NMS_STAGE_A, 256);                                         // keepA
        b += align_up(nm, 256);                                                                       // dead
        b += 256;                                                                                     // numA, n2
    }
    return b;
}

void nms_carve(void *ws, int n, NmsBuffers &b)
{
    unsigned char *p = static_cast<unsigned char *>(ws);
    const size_t nm = nms_two_stage(n) ? (size_t)(n - NMS_STAGE_A) : (size_t)n;
    const size_t W = (size_t)cdiv((int)nm, 64);
    b.boxes = reinterpret_cast<float4 *>(p); p += align_up(sizeof(float4) * (size_t)n, 256);
    b.areas = reinterpret_cast<float *>(p);  p += align_up(sizeof(float) * (size_t)n, 256);
    b.cls = reinterpret_cast<int *>(p);      p += align_up(sizeof(int) * (size_t)n, 256);
    b.order = reinterpret_cast<int *>(p);    p += align_up(sizeof(int) * (size_t)n, 256);
    b.rank = reinterpret_cast<int *>(p);     p += align_up(sizeof(int) * (size_t)n, 256);
    b.tickets = reinterpret_cast<int *>(p);  p += align_up(sizeof(int) * (size_t)cdiv(n, RANK_ROWS), 256);
    b.mask = reinterpret_cast<unsigned long long *>(p); p += align_up(sizeof(unsigned long long) * nm * W, 256);
    b.fix = p;                               p += 2 * nms_fix_bytes(n);
    b.sparse = p;                            p += nms_sparse_bytes(n);
    b.stage = p;
}

static int launch_mask(const float4 *boxes, const float *areas, const int *cls, int n_max, const int *n_dev,
                       int W_stride, float thresh, unsigned long long *mask, const int *skip, void *fix, cudaStream_t st)
{
    // words of the resolve scratch the kernel zeroes (see launch_scan): 4 W_stride + FixState
    unsigned long long *fz = static_cast<unsigned long long *>(fix);
    const int fw = (int)((align_up(sizeof(unsigned long long) * 4 * (size_t)W_stride, 256) + align_up(sizeof(FixState), 8)) / 8);
    const int W = cdiv(n_max, 64);
    const long long n_tiles = (long long)W * (W + 1) / 2;
    long long n_blocks = (n_tiles + MASK_GROUPS - 1) / MASK_GROUPS;
    if (n_blocks > 16LL * sm_count()) n_blocks = 16LL * sm_count();
    if (cls)
        nms_mask_kernel<true><<<(unsigned)n_blocks, 64 * MASK_GROUPS, 0, st>>>(boxes, areas, cls, n_max, n_dev, W_stride, thresh, mask, skip, fz, fw);
    else
        nms_mask_kernel<false><<<(unsigned)n_blocks, 64 * MASK_GROUPS, 0, st>>>(boxes, areas, cls, n_max, n_dev, W_stride, thresh, mask, skip, fz, fw);
    SLN_LAUNCH_OK("nms_mask_kernel");
    return SLN_OK;
}

// scratch of the parallel resolve, carved from `fix` (see nms_fix_bytes)
static size_t nms_fix_bytes(int n_max)
{
    const size_t W = (size_t)cdiv(n_max, 64);
    return align_up(sizeof(unsigned long long) * 4 * W, 256) + align_up(sizeof(FixState), 256);
}

static int launch_scan(const unsigned long long *mask, const int *order, int n_max, const int *n_dev, int W_stride,
                       int max_keep, const int *keep_base_dev, int64_t *keep64, int *keep32, int *num_keep,
                       void *fix, const int *skip, cudaStream_t st)
{
    // (1) parallel fixed-point resolve on the whole GPU
    const bool parallel = W_stride >= FIX_MIN_WORDS;     // short problems: the serial chain is cheaper than grid barriers
    unsigned long long *removed = static_cast<unsigned long long *>(fix);
    unsigned long long *Kbuf = removed + 3 * (size_t)W_stride;
    FixState *state = reinterpret_cast<FixState *>(static_cast<unsigned char *>(fix) + align_up(sizeof(unsigned long long) * 4 * (size_t)W_stride, 256));
    // (the three `removed` buffers, K and the state were zeroed by the mask kernel that precedes this call)
    static int max_ctas = 0;
    if (max_ctas == 0) {
        int per_sm = 0;
        SLN_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, nms_fixpoint_kernel, FIX_THREADS, 0));
        max_ctas = per_sm * sm_count();
        if (max_ctas < 1) max_ctas = 1;
    }
    int G = W_stride < max_ctas ? W_stride : max_ctas;
    if (G < 1) G = 1;
    int n_host = n_max;
    if (parallel) {
    void *args[] = {(void *)&mask, (void *)&order, (void *)&n_host, (void *)&n_dev, (void *)&W_stride, (void *)&max_keep,
                    (void *)&keep_base_dev, (void *)&removed, (void *)&Kbuf, (void *)&state, (void *)&keep64,
                    (void *)&keep32, (void *)&num_keep, (void *)&skip};
    SLN_CUDA_OK(cudaLaunchCooperativeKernel((const void *)nms_fixpoint_kernel, dim3(G), dim3(FIX_THREADS), args, 0, st));
    }
    // (2) serial scan: only does work when the fixed point was not reached in FIX_MAX_ROUNDS
    const size_t smem = scan_smem_bytes(W_stride);
    SLN_REQUIRE(smem <= 220 * 1024, SLN_ERR_ARG, "nms: n=%d too large for the scan kernel", n_max);
    SLN_CUDA_OK(cudaFuncSetAttribute(nms_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    nms_scan_kernel<<<1, SCAN_THREADS, smem, st>>>(mask, order, n_max, n_dev, W_stride, max_keep, keep_base_dev, keep64,
                                                  keep32, num_keep, &state->status, skip);
    SLN_LAUNCH_OK("nms_scan_kernel");
    return SLN_OK;
}

static int nms_dense_launch(const float4 *boxes, const float *areas, const int *cls, const int *order, int n, float thresh,
                            int max_keep, unsigned long long *mask, int64_t *keep64, int *keep32, int *num_keep,
                            cudaStream_t st, void *stage, void *fix, const int *skip);

// `stage`: scratch for the two-stage path (nullptr: single stage).  `order == nullptr`: kept entries
// are visiting positions.
int nms_sorted_launch(const float4 *boxes, const float *areas, const int *cls, const int *order, int n,
                      float thresh, int max_keep, unsigned long long *mask, int64_t *keep64, int *keep32,
                      int *num_keep, cudaStream_t st, void *stage, void *fix, void *sparse, bool sparse_only)
{
    if (max_keep <= 0 || max_keep > n) max_keep = n;
    if (n == 0) {
        SLN_CUDA_OK(cudaMemsetAsync(num_keep, 0, sizeof(int), st));
        return SLN_OK;
    }
    // sparse path first; the dense kernels below are launched regardless and leave at once when it succeeded
    const int *skip = nullptr;
    int rc = launch_sparse(boxes, areas, cls, order, n, thresh, max_keep, keep64, keep32, num_keep, sparse, st, &skip,
                           sparse_only);
    if (rc != SLN_OK) return rc;
    if (sparse_only && skip != nullptr) return SLN_OK;      // the caller retries with SLN_NMS_DENSE_ONLY on num_keep < 0
    return nms_dense_launch(boxes, areas, cls, order, n, thresh, max_keep, mask, keep64, keep32, num_keep, st, stage, fix, skip);
}

// The dense pipeline (one stage, or two for n >= NMS_TWO_STAGE_MIN with `stage`); every kernel leaves at once when
// *skip == 1 (the sparse path produced the result).  max_keep is already normalised to [1, n].
static int nms_dense_launch(const float4 *boxes, const float *areas, const int *cls, const int *order, int n, float thresh,
                            int max_keep, unsigned long long *mask, int64_t *keep64, int *keep32, int *num_keep,
                            cudaStream_t st, void *stage, void *fix, const int *skip)
{
    int rc;
    if (!nms_two_stage(n) || stage == nullptr) {
        const int W = cdiv(n, 64);
        rc = launch_mask(boxes, areas, cls, n, nullptr, W, thresh, mask, skip, fix, st);
        if (rc != SLN_OK) return rc;
        return launch_scan(mask, order, n, nullptr, W, max_keep, nullptr, keep64, keep32, num_keep, fix, skip, st);
    }
    // ---- two stages
    const int T = NMS_STAGE_A, nm = n - T, W2 = cdiv(nm, 64);
    unsigned char *p = static_cast<unsigned char *>(stage);
    unsigned long long *maskA = reinterpret_cast<unsigned long long *>(p); p += align_up(sizeof(unsigned long long) * (size_t)T * (T / 64), 256);
    float4 *boxes2 = reinterpret_cast<float4 *>(p);   p += align_up(sizeof(float4) * (size_t)nm, 256);
    float *areas2 = reinterpret_cast<float *>(p);     p += align_up(sizeof(float) * (size_t)nm, 256);
    int *cls2 = reinterpret_cast<int *>(p);           p += align_up(sizeof(int) * (size_t)nm, 256);
    int *order2 = reinterpret_cast<int *>(p);         p += align_up(sizeof(int) * (size_t)nm, 256);
    int *keepA = reinterpret_cast<int *>(p);          p += align_up(sizeof(int) * (size_t)T, 256);
    unsigned char *dead = p;                          p += align_up((size_t)nm, 256);
    int *numA = reinterpret_cast<int *>(p);
    int *n2 = numA + 1;
    // stage A: exact NMS of the first T boxes; survivors go straight to the output
    rc = launch_mask(boxes, areas, cls, T, nullptr, T / 64, thresh, maskA, skip, fix, st);
    if (rc != SLN_OK) return rc;
    rc = launch_scan(maskA, nullptr, T, nullptr, T / 64, max_keep, nullptr, nullptr, keepA, numA, fix, skip, st);
    if (rc != SLN_OK) return rc;
    // everything a stage-A survivor overlaps is gone; compact the rest (order preserved)
    if (cls) nms_suppress_kernel<true><<<cdiv(nm, 256), 256, 0, st>>>(boxes, areas, cls, T, n, keepA, numA, thresh, dead, skip);
    else nms_suppress_kernel<false><<<cdiv(nm, 256), 256, 0, st>>>(boxes, areas, cls, T, n, keepA, numA, thresh, dead, skip);
    SLN_LAUNCH_OK("nms_suppress_kernel");
    nms_compact_kernel<<<1, 1024, 0, st>>>(boxes, areas, cls, order, dead, T, n, boxes2, areas2, cls2, order2, n2, skip);
    SLN_LAUNCH_OK("nms_compact_kernel");
    // stage-A survivors -> output (positions -> original indices)
    nms_emit_stageA_kernel<<<cdiv(T, 256), 256, 0, st>>>(keepA, numA, order, keep64, keep32, skip);
    SLN_LAUNCH_OK("nms_emit_stageA_kernel");
    // stage B on the compacted remainder, appended after the stage-A survivors
    rc = launch_mask(boxes2, areas2, cls ? cls2 : nullptr, nm, n2, W2, thresh, mask, skip,
                     static_cast<unsigned char *>(fix) + nms_fix_bytes(n), st);
    if (rc != SLN_OK) return rc;
    return launch_scan(mask, order2, nm, n2, W2, max_keep, numA, keep64, keep32, num_keep,
                       static_cast<unsigned char *>(fix) + nms_fix_bytes(n), skip, st);
}

int nms_sorted_batched_launch(int B, size_t stride, const float4 *boxes, const float *areas, const int *cls,
                              const int *order, int n, float thresh, int max_keep, unsigned long long *mask,
                              int64_t *keep64, int *keep32, size_t keep_stride, int *num_keep, size_t num_stride,
                              cudaStream_t st, void *stage, void *fix, void *sparse)
{
    if (B <= 0) return SLN_OK;
    if (max_keep <= 0 || max_keep > n) max_keep = n;
    if (n == 0) {
        for (int b = 0; b < B; ++b) SLN_CUDA_OK(cudaMemsetAsync(seg_at(num_keep, num_stride, b), 0, sizeof(int), st));
        return SLN_OK;
    }
    // the same eligibility test as launch_sparse: n and thresh are common to all problems
    const bool sparse_ok = sparse != nullptr && n >= SP_MIN_N && n <= SP_MAX_N && thresh >= 0.05f;
    if (sparse_ok) {
        SLN_REQUIRE(B <= 65535, SLN_ERR_ARG, "nms: %d problems in one call", B);
        SparseBufs sb;
        sparse_carve(sparse, n, sb);
        int CB, G;
        float ct;
        sparse_params(n, cls != nullptr, thresh, CB, G, ct);
        const unsigned edge_cap = (unsigned)SP_EDGES_PER_BOX * (unsigned)n;
        SLN_CUDA_OK(launch_chain(cls ? nms_bin_seg_kernel<true> : nms_bin_seg_kernel<false>, dim3(SP_CLUSTER, B),
                                 dim3(SP_BIN_THREADS), 0, st, true, boxes, areas, cls, n, G, CB, sb, stride));
        // about the pair grid of one single-image call in all, at least one CTA per problem
        int ctas = cdiv(n, SP_PAIR_WARPS);
        const int cap = cdiv(SLN_SP_PAIR_CTAS_PER_SM * sm_count(), B);
        if (ctas > cap) ctas = cap;
        SLN_CUDA_OK(launch_chain(cls ? nms_pairs_seg_kernel<true> : nms_pairs_seg_kernel<false>, dim3(ctas, B),
                                 dim3(32 * SP_PAIR_WARPS), 0, st, true, boxes, areas, cls, n, thresh, ct, edge_cap, sb, stride));
        const size_t smem = sparse_resolve_smem(n);
        SLN_CUDA_OK(cudaFuncSetAttribute(nms_sparse_resolve_seg_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        SLN_CUDA_OK(launch_chain(nms_sparse_resolve_seg_kernel, dim3(SP_CLUSTER, B), dim3(SP_RESOLVE_THREADS), smem, st, true,
                                 order, n, max_keep, edge_cap, sb, keep64, keep32, keep_stride, num_keep, num_stride, stride));
    }
    // dense fallback, per problem and guarded by that problem's status word: without a host read nobody knows which
    // problems need it, so every problem gets the launches and those whose sparse pass succeeded leave at once
    for (int b = 0; b < B; ++b) {
        const int *skip = sparse_ok ? &seg_at(static_cast<SparseHdr *>(sparse), stride, b)->status : nullptr;
        const int rc = nms_dense_launch(seg_at(boxes, stride, b), seg_at(areas, stride, b), cls ? seg_at(cls, stride, b) : nullptr,
                                        order ? seg_at(order, stride, b) : nullptr, n, thresh, max_keep, seg_at(mask, stride, b),
                                        keep64 ? seg_at(keep64, keep_stride, b) : nullptr,
                                        keep32 ? seg_at(keep32, keep_stride, b) : nullptr, seg_at(num_keep, num_stride, b),
                                        st, stage ? seg_at(stage, stride, b) : nullptr, seg_at(fix, stride, b), skip);
        if (rc != SLN_OK) return rc;
    }
    return SLN_OK;
}

}  // namespace sln

using namespace sln;

extern "C" size_t sln_nms_workspace_bytes(int n)
{
    if (n < 0) return 0;
    return nms_buffers_bytes(n);
}

extern "C" int sln_nms_ex(const float *dets, const int *class_ids, int n, float thresh, int max_keep, int flags,
                          int64_t *keep, int *num_keep, int *path_out, void *workspace, size_t workspace_bytes,
                          void *stream)
{
    SLN_REQUIRE(n >= 0, SLN_ERR_ARG, "negative n");
    SLN_REQUIRE(num_keep != nullptr, SLN_ERR_ARG, "null num_keep");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (path_out) SLN_CUDA_OK(cudaMemsetAsync(path_out, 0, sizeof(int), st));
    if (n == 0) {
        SLN_CUDA_OK(cudaMemsetAsync(num_keep, 0, sizeof(int), st));
        return SLN_OK;
    }
    SLN_REQUIRE(dets && keep, SLN_ERR_ARG, "null pointer");
    SLN_REQUIRE(workspace && workspace_bytes >= nms_buffers_bytes(n), SLN_ERR_WORKSPACE,
                "nms workspace: need %zu bytes, got %zu", nms_buffers_bytes(n), workspace_bytes);
    NmsBuffers b;
    nms_carve(workspace, n, b);
    const bool try_sparse = !(flags & SLN_NMS_DENSE_ONLY) && n >= SP_MIN_N && n <= SP_MAX_N && thresh >= 0.05f;
    // rank[] and the row-tile tickets are adjacent: one memset
    SLN_CUDA_OK(cudaMemsetAsync(b.rank, 0, (size_t)(reinterpret_cast<unsigned char *>(b.tickets) - reinterpret_cast<unsigned char *>(b.rank)) +
                                               sizeof(int) * (size_t)cdiv(n, RANK_ROWS), st));
    RankGather ga{dets, class_ids, b.boxes, b.areas, b.cls, b.order, b.tickets};
    int rc = rank_launch(dets + 4, 5, nullptr, n, b.rank, ga, st);
    if (rc != SLN_OK) return rc;
    rc = nms_sorted_launch(b.boxes, b.areas, class_ids ? b.cls : nullptr, b.order, n, thresh, max_keep, b.mask,
                           keep, nullptr, num_keep, st, b.stage, b.fix, try_sparse ? b.sparse : nullptr,
                           (flags & SLN_NMS_SPARSE_ONLY) != 0);
    if (rc != SLN_OK) return rc;
    if (path_out && try_sparse)      // SparseHdr.status: 1 when the sparse path produced the result
        SLN_CUDA_OK(cudaMemcpyAsync(path_out, b.sparse, sizeof(int), cudaMemcpyDeviceToDevice, st));
    return SLN_OK;
}

extern "C" int sln_nms(const float *dets, const int *class_ids, int n, float thresh, int max_keep,
                       int64_t *keep, int *num_keep, void *workspace, size_t workspace_bytes, void *stream)
{
    return sln_nms_ex(dets, class_ids, n, thresh, max_keep, 0, keep, num_keep, nullptr, workspace, workspace_bytes, stream);
}

// B independent problems of n boxes.  The workspace is B copies of sln_nms_ex's, nms_buffers_bytes(n) apart (a multiple
// of 256); problem b runs sln_nms_ex's stages with sln_nms_ex's parameters in its copy, so its survivors are the same.
extern "C" size_t sln_nms_batched_workspace_bytes(int B, int n)
{
    if (B < 0 || n < 0) return 0;
    return (size_t)B * nms_buffers_bytes(n);
}

extern "C" int sln_nms_batched(const float *dets, const int *class_ids, int B, int n, float thresh, int max_keep, int flags,
                               int64_t *keep, int *num_keep, int *path_out, void *workspace, size_t workspace_bytes,
                               void *stream)
{
    SLN_REQUIRE(B >= 0 && n >= 0, SLN_ERR_ARG, "negative size (B=%d, n=%d)", B, n);
    SLN_REQUIRE(B <= 65535, SLN_ERR_ARG, "B=%d problems in one call (at most 65535)", B);
    SLN_REQUIRE(!(flags & SLN_NMS_SPARSE_ONLY), SLN_ERR_ARG, "SLN_NMS_SPARSE_ONLY needs a host retry: not for the batched call");
    if (B == 0) return SLN_OK;
    SLN_REQUIRE(num_keep != nullptr, SLN_ERR_ARG, "null num_keep");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (path_out) SLN_CUDA_OK(cudaMemsetAsync(path_out, 0, sizeof(int) * (size_t)B, st));
    if (n == 0) {
        SLN_CUDA_OK(cudaMemsetAsync(num_keep, 0, sizeof(int) * (size_t)B, st));
        return SLN_OK;
    }
    SLN_REQUIRE(dets && keep, SLN_ERR_ARG, "null pointer");
    const size_t S = nms_buffers_bytes(n);
    SLN_REQUIRE(workspace && workspace_bytes >= S * B, SLN_ERR_WORKSPACE, "batched nms workspace: need %zu bytes, got %zu",
                S * B, workspace_bytes);
    const int mk = (max_keep <= 0 || max_keep > n) ? n : max_keep;      // row length of keep
    NmsBuffers b;
    nms_carve(workspace, n, b);
    const bool try_sparse = !(flags & SLN_NMS_DENSE_ONLY) && n >= SP_MIN_N && n <= SP_MAX_N && thresh >= 0.05f;
    // every problem's rank[] and row-tile tickets (adjacent): one strided memset
    const size_t clear = (size_t)(reinterpret_cast<unsigned char *>(b.tickets) - reinterpret_cast<unsigned char *>(b.rank)) +
                         sizeof(int) * (size_t)cdiv(n, RANK_ROWS);
    SLN_CUDA_OK(cudaMemset2DAsync(b.rank, S, 0, clear, B, st));
    RankGather ga{dets, class_ids, b.boxes, b.areas, b.cls, b.order, b.tickets};
    int rc = rank_seg_launch(dets + 4, 5, nullptr, n, B, b.rank, ga, sizeof(float) * 5 * (size_t)n, sizeof(int) * (size_t)n,
                             S, st);
    if (rc != SLN_OK) return rc;
    rc = nms_sorted_batched_launch(B, S, b.boxes, b.areas, class_ids ? b.cls : nullptr, b.order, n, thresh, max_keep, b.mask,
                                   keep, nullptr, sizeof(int64_t) * (size_t)mk, num_keep, sizeof(int), st, b.stage, b.fix,
                                   try_sparse ? b.sparse : nullptr);
    if (rc != SLN_OK) return rc;
    if (path_out && try_sparse)      // SparseHdr.status of every problem: 1 when the sparse path produced its result
        SLN_CUDA_OK(cudaMemcpy2DAsync(path_out, sizeof(int), b.sparse, S, sizeof(int), B, cudaMemcpyDeviceToDevice, st));
    return SLN_OK;
}
