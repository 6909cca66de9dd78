// proposal.cu -- proposal_layer on the device (one image per call, no host sync).
//
// Reference semantics: modal/Functions.py:114-178 (proposal_layer) with
// apply_box_deltas :77-98 and clip_boxes :101-111; NMS through nms/pth_nms.py.
// The reference does a full descending sort of all A (=261 888) scores and keeps the
// first 6000 (:144-149), ~15 elementwise torch kernels for the decode, and the NMS
// host round trip.  Here:
//   1. radix select (3 histogram passes over the 32-bit order-preserving keys) finds
//      the exact k-th key; candidates above it are compacted in any order, candidates
//      equal to it are taken lowest-index-first (two-level ordered scan) -> exactly the
//      first k elements of the stable descending sort, as a set;
//   2. rank sort of the k candidates by (score desc, anchor index asc) -> visiting order;
//   3. decode + clip written directly in visiting order (one rounding per reference op,
//      exp via double so it is within 1 ulp of torch's);
//   4. the NMS mask + scan stages from nms.cu with max_keep = proposal_count;
//   5. gather + divide by [h,w,h,w], zero-fill the tail.
#include "nms_core.cuh"

namespace sln {

struct SelectState {
    unsigned prefix;     // high bits of the k-th key found so far
    int k_rem;           // how many elements are still wanted among keys matching prefix
    int count_gt;        // (final) number of keys strictly above the k-th key
    int counter;         // slot allocator for keys above the k-th key
};

constexpr int SEL_BINS = 2048;
constexpr int SEL_THREADS = 256;

__device__ __forceinline__ unsigned fg_key(const float *probs, int i) { return score_key(__ldg(probs + 2 * (size_t)i + 1)); }

// Walk a 2048-bin histogram from the top bin down to the bin holding the k_rem-th element (whole CTA of
// SEL_THREADS threads, 8 bins per thread); fold that bin into the prefix and reduce k_rem.  Every CTA of the kernel
// that consumes the result does this itself (the histogram is 8 KB in L2), which removes the three single-CTA
// "pick" launches of the first version; each pass has its own histogram, so nothing has to be cleared in between.
struct Pick {
    unsigned prefix;
    int k_rem;
};

template <int PASS>
__device__ Pick cta_pick(const unsigned *__restrict__ hist, unsigned prev_prefix, int k_rem)
{
    __shared__ unsigned s_wsum[SEL_THREADS / 32];
    __shared__ unsigned s_found[2];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    constexpr int PER = SEL_BINS / SEL_THREADS;     // 8
    unsigned h[PER], sum = 0u;
#pragma unroll
    for (int q = 0; q < PER; ++q) { h[q] = hist[PER * t + q]; sum += h[q]; }
    unsigned incl = sum;                            // inclusive suffix sum over the threads above (higher bins)
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned v = __shfl_down_sync(0xffffffffu, incl, o);
        if (lane + o < 32) incl += v;
    }
    __syncthreads();                                // the statics may still be read from a previous call
    if (lane == 0) s_wsum[warp] = incl;
    __syncthreads();
    unsigned above = incl - sum;                    // elements in bins above this thread's, same warp
    for (int w = warp + 1; w < SEL_THREADS / 32; ++w) above += s_wsum[w];
#pragma unroll
    for (int q = PER - 1; q >= 0; --q) {            // highest bin first
        if (above < (unsigned)k_rem && (unsigned)k_rem <= above + h[q]) { s_found[0] = (unsigned)(PER * t + q); s_found[1] = above; }
        above += h[q];
    }
    __syncthreads();
    Pick p;
    p.prefix = (prev_prefix << (PASS == 0 ? 0 : (PASS == 1 ? 11 : 10))) | s_found[0];
    p.k_rem = k_rem - (int)s_found[1];
    return p;
}

// pass 0: bits 31..21, pass 1: bits 20..10 (keys matching the 11-bit prefix), pass 2: bits 9..0.
// hist = three histograms [3][SEL_BINS], zeroed once per call.  Pass P > 0 first picks the bin of pass P-1 (from the
// state the previous launch left + that pass's histogram); CTA 0 publishes the new state for the next launch.
template <int PASS>
__device__ __forceinline__ void select_hist_body(const float *probs, int A, int K, SelectState *state,
                                                 unsigned *hist)
{
    __shared__ unsigned s_hist[SEL_BINS];
    pdl_prologue();
    for (int t = threadIdx.x; t < SEL_BINS; t += SEL_THREADS) s_hist[t] = 0u;
    unsigned prefix = 0u;
    if (PASS > 0) {
        const unsigned prev = PASS == 1 ? 0u : state[(PASS - 1) & 1].prefix;
        const int k_rem = PASS == 1 ? K : state[(PASS - 1) & 1].k_rem;
        const Pick p = PASS == 1 ? cta_pick<0>(hist, prev, k_rem) : cta_pick<1>(hist + SEL_BINS, prev, k_rem);
        prefix = p.prefix;
        // (the state words this launch reads are not the ones it writes: double-buffered by pass parity)
        if (blockIdx.x == 0 && threadIdx.x == 0) { state[PASS & 1].prefix = p.prefix; state[PASS & 1].k_rem = p.k_rem; }
    }
    __syncthreads();
    unsigned *out = hist + PASS * SEL_BINS;
    for (int i = blockIdx.x * SEL_THREADS + threadIdx.x; i < A; i += gridDim.x * SEL_THREADS) {
        const unsigned k = fg_key(probs, i);
        if (PASS == 0) atomicAdd(&s_hist[k >> 21], 1u);
        else if (PASS == 1) { if ((k >> 21) == prefix) atomicAdd(&s_hist[(k >> 10) & 0x7ffu], 1u); }
        else { if ((k >> 10) == prefix) atomicAdd(&s_hist[k & 0x3ffu], 1u); }
    }
    __syncthreads();
    for (int t = threadIdx.x; t < SEL_BINS; t += SEL_THREADS) {
        const unsigned v = s_hist[t];
        if (v) atomicAdd(out + t, v);
    }
}

template <int PASS>
__global__ void __launch_bounds__(SEL_THREADS)
select_hist_kernel(const float *__restrict__ probs, int A, int K, SelectState *__restrict__ state,
                   unsigned *__restrict__ hist)
{
    select_hist_body<PASS>(probs, A, K, state, hist);
}

// Batched forms (sln_proposal_layer_batched): image b = blockIdx.y reads probs + b*2A and works in the b-th copy of the
// single-image workspace, ws_stride bytes further on (seg_at).  The bodies are the single-image kernels' own.

template <int PASS>
__global__ void __launch_bounds__(SEL_THREADS)
select_hist_seg_kernel(const float *__restrict__ probs, int A, int K, SelectState *__restrict__ state,
                       unsigned *__restrict__ hist, size_t ws_stride)
{
    const int b = blockIdx.y;
    select_hist_body<PASS>(probs + 2 * (size_t)A * b, A, K, seg_at(state, ws_stride, b), seg_at(hist, ws_stride, b));
}

// Each CTA owns a contiguous slice of the anchors so that "ordered" means index order.
__device__ __forceinline__ void slice_of(int A, int &lo, int &hi)
{
    const int per = (A + gridDim.x - 1) / gridDim.x;
    lo = min(A, (int)blockIdx.x * per);
    hi = min(A, lo + per);
}

__device__ __forceinline__ void select_count_eq_body(const float *probs, int A, int K,
                                                     SelectState *state, const unsigned *hist,
                                                     int *blk_eq)
{
    __shared__ int s_cnt;
    pdl_prologue();
    if (threadIdx.x == 0) s_cnt = 0;
    // pick of pass 2: the exact k-th key T and how many keys equal to T are still wanted
    const Pick p = cta_pick<2>(hist + 2 * SEL_BINS, state[0].prefix, state[0].k_rem);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        state[1].prefix = p.prefix;
        state[1].k_rem = p.k_rem;
        state[1].count_gt = K - p.k_rem;
        state[1].counter = 0;
    }
    __syncthreads();
    const unsigned T = p.prefix;
    int lo, hi;
    slice_of(A, lo, hi);
    int c = 0;
    for (int i = lo + threadIdx.x; i < hi; i += SEL_THREADS) c += (fg_key(probs, i) == T);
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s_cnt, c);
    __syncthreads();
    if (threadIdx.x == 0) blk_eq[blockIdx.x] = s_cnt;
}

__global__ void __launch_bounds__(SEL_THREADS)
select_count_eq_kernel(const float *__restrict__ probs, int A, int K, SelectState *__restrict__ state,
                       const unsigned *__restrict__ hist, int *__restrict__ blk_eq)
{
    select_count_eq_body(probs, A, K, state, hist, blk_eq);
}

__global__ void __launch_bounds__(SEL_THREADS)
select_count_eq_seg_kernel(const float *__restrict__ probs, int A, int K, SelectState *__restrict__ state,
                           const unsigned *__restrict__ hist, int *__restrict__ blk_eq, size_t ws_stride)
{
    const int b = blockIdx.y;
    select_count_eq_body(probs + 2 * (size_t)A * b, A, K, seg_at(state, ws_stride, b), seg_at(hist, ws_stride, b),
                         seg_at(blk_eq, ws_stride, b));
}

__device__ __forceinline__ void select_compact_body(const float *probs, int A, SelectState *state,
                                                    const int *blk_eq, float *cand_score,
                                                    int *cand_idx)
{
    __shared__ int s_warp[SEL_THREADS / 32];
    __shared__ int s_base;
    pdl_prologue();
    state += 1;                                     // final state, published by select_count_eq_kernel
    const unsigned T = state->prefix;
    const int count_gt = state->count_gt, need_eq = state->k_rem;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int lo, hi;
    slice_of(A, lo, hi);
    // keys equal to T in the slices before mine (replaces the single-CTA scan launch)
    {
        int part = 0;
        for (int k = threadIdx.x; k < (int)blockIdx.x; k += SEL_THREADS) part += blk_eq[k];
        for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
        if (lane == 0) s_warp[warp] = part;
        __syncthreads();
        if (threadIdx.x == 0) {
            int tot = 0;
            for (int w = 0; w < SEL_THREADS / 32; ++w) tot += s_warp[w];
            s_base = tot;
        }
        __syncthreads();
    }
    int eq_base = s_base;
    __syncthreads();
    for (int start = lo; start < hi; start += SEL_THREADS) {
        const int i = start + threadIdx.x;
        unsigned k = 0;
        bool gt = false, eq = false;
        if (i < hi) {
            k = fg_key(probs, i);
            gt = k > T;
            eq = k == T;
        }
        if (gt) {
            const int slot = atomicAdd(&state->counter, 1);      // any order: a rank sort follows
            cand_score[slot] = __ldg(probs + 2 * (size_t)i + 1);
            cand_idx[slot] = i;
        }
        const unsigned m = __ballot_sync(0xffffffffu, eq);
        if (lane == 0) s_warp[warp] = __popc(m);
        __syncthreads();
        int off = 0, total = 0;
#pragma unroll
        for (int w = 0; w < SEL_THREADS / 32; ++w) {
            const int c = s_warp[w];
            if (w < warp) off += c;
            total += c;
        }
        if (eq) {
            const int tie_rank = eq_base + off + __popc(m & ((1u << lane) - 1u));
            if (tie_rank < need_eq) {                             // lowest indices first (stable)
                cand_score[count_gt + tie_rank] = __ldg(probs + 2 * (size_t)i + 1);
                cand_idx[count_gt + tie_rank] = i;
            }
        }
        eq_base += total;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(SEL_THREADS)
select_compact_kernel(const float *__restrict__ probs, int A, SelectState *__restrict__ state,
                      const int *__restrict__ blk_eq, float *__restrict__ cand_score,
                      int *__restrict__ cand_idx)
{
    select_compact_body(probs, A, state, blk_eq, cand_score, cand_idx);
}

__global__ void __launch_bounds__(SEL_THREADS)
select_compact_seg_kernel(const float *__restrict__ probs, int A, SelectState *__restrict__ state,
                          const int *__restrict__ blk_eq, float *__restrict__ cand_score, int *__restrict__ cand_idx,
                          size_t ws_stride)
{
    const int b = blockIdx.y;
    select_compact_body(probs + 2 * (size_t)A * b, A, seg_at(state, ws_stride, b), seg_at(blk_eq, ws_stride, b),
                        seg_at(cand_score, ws_stride, b), seg_at(cand_idx, ws_stride, b));
}

__device__ __forceinline__ void select_all_body(const float *probs, int A, float *cand_score,
                                                int *cand_idx)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= A) return;
    cand_score[i] = probs[2 * (size_t)i + 1];
    cand_idx[i] = i;
}

__global__ void select_all_kernel(const float *__restrict__ probs, int A, float *__restrict__ cand_score,
                                  int *__restrict__ cand_idx)
{
    select_all_body(probs, A, cand_score, cand_idx);
}

__global__ void select_all_seg_kernel(const float *__restrict__ probs, int A, float *__restrict__ cand_score,
                                      int *__restrict__ cand_idx, size_t ws_stride)
{
    const int b = blockIdx.y;
    select_all_body(probs + 2 * (size_t)A * b, A, seg_at(cand_score, ws_stride, b), seg_at(cand_idx, ws_stride, b));
}

__device__ __forceinline__ float clampf_nan(float v, float lo, float hi)
{
    return v < lo ? lo : (v > hi ? hi : v);      // NaN passes through like torch.clamp
}

struct Float4Std { float s0, s1, s2, s3; };

// Decode candidate j (anchor cand_idx[j]) and write it at its visiting position rank[j].
__device__ __forceinline__ void proposal_decode_body(const float *anchors, const float *deltas,
                                                     const int *cand_idx, const int *rank, int K,
                                                     Float4Std sd, float img_h, float img_w, float4 *boxes,
                                                     float *areas)
{
    pdl_prologue();
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= K) return;
    const int a = cand_idx[j];
    const float4 an = *reinterpret_cast<const float4 *>(anchors + 4 * (size_t)a);
    const float4 dl = *reinterpret_cast<const float4 *>(deltas + 4 * (size_t)a);
    const float dy = __fmul_rn(dl.x, sd.s0), dx = __fmul_rn(dl.y, sd.s1);      // Functions.py:137-140
    const float dh = __fmul_rn(dl.z, sd.s2), dw = __fmul_rn(dl.w, sd.s3);
    // apply_box_deltas, Functions.py:83-97 (one rounding per torch op)
    float height = __fsub_rn(an.z, an.x), width = __fsub_rn(an.w, an.y);
    float cy = __fadd_rn(an.x, __fmul_rn(0.5f, height));
    float cx = __fadd_rn(an.y, __fmul_rn(0.5f, width));
    cy = __fadd_rn(cy, __fmul_rn(dy, height));
    cx = __fadd_rn(cx, __fmul_rn(dx, width));
    height = __fmul_rn(height, (float)exp((double)dh));
    width = __fmul_rn(width, (float)exp((double)dw));
    float y1 = __fsub_rn(cy, __fmul_rn(0.5f, height));
    float x1 = __fsub_rn(cx, __fmul_rn(0.5f, width));
    float y2 = __fadd_rn(y1, height);
    float x2 = __fadd_rn(x1, width);
    // clip_boxes, Functions.py:101-111, window (0,0,h,w)
    y1 = clampf_nan(y1, 0.f, img_h); x1 = clampf_nan(x1, 0.f, img_w);
    y2 = clampf_nan(y2, 0.f, img_h); x2 = clampf_nan(x2, 0.f, img_w);
    const int p = rank[j];
    boxes[p] = make_float4(y1, x1, y2, x2);
    areas[p] = __fmul_rn(__fadd_rn(__fsub_rn(x2, x1), 1.f), __fadd_rn(__fsub_rn(y2, y1), 1.f));   // pth_nms.py:16
}

__global__ void proposal_decode_kernel(const float *__restrict__ anchors, const float *__restrict__ deltas,
                                       const int *__restrict__ cand_idx, const int *__restrict__ rank, int K,
                                       Float4Std sd, float img_h, float img_w, float4 *__restrict__ boxes,
                                       float *__restrict__ areas)
{
    proposal_decode_body(anchors, deltas, cand_idx, rank, K, sd, img_h, img_w, boxes, areas);
}

// anchors are shared by all images; deltas of image b start at b*4A
__global__ void proposal_decode_seg_kernel(const float *__restrict__ anchors, const float *__restrict__ deltas, int A,
                                           const int *__restrict__ cand_idx, const int *__restrict__ rank, int K,
                                           Float4Std sd, float img_h, float img_w, float4 *__restrict__ boxes,
                                           float *__restrict__ areas, size_t ws_stride)
{
    const int b = blockIdx.y;
    proposal_decode_body(anchors, deltas + 4 * (size_t)A * b, seg_at(cand_idx, ws_stride, b), seg_at(rank, ws_stride, b), K,
                         sd, img_h, img_w, seg_at(boxes, ws_stride, b), seg_at(areas, ws_stride, b));
}

__device__ __forceinline__ void proposal_finalize_body(const float4 *boxes, const int *keep,
                                                       const int *num_keep, int proposal_count, float img_h,
                                                       float img_w, float4 *out, int *num_out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int nk = min(*num_keep, proposal_count);
    if (i == 0) *num_out = nk;
    if (i >= proposal_count) return;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < nk) {
        const float4 b = boxes[keep[i]];
        v = make_float4(__fdiv_rn(b.x, img_h), __fdiv_rn(b.y, img_w), __fdiv_rn(b.z, img_h), __fdiv_rn(b.w, img_w));
    }
    out[i] = v;
}

__global__ void proposal_finalize_kernel(const float4 *__restrict__ boxes, const int *__restrict__ keep,
                                         const int *__restrict__ num_keep, int proposal_count, float img_h,
                                         float img_w, float4 *__restrict__ out, int *__restrict__ num_out)
{
    proposal_finalize_body(boxes, keep, num_keep, proposal_count, img_h, img_w, out, num_out);
}

__global__ void proposal_finalize_seg_kernel(const float4 *__restrict__ boxes, const int *__restrict__ keep,
                                             const int *__restrict__ num_keep, int proposal_count, float img_h,
                                             float img_w, float4 *__restrict__ out, int *__restrict__ num_out,
                                             size_t ws_stride)
{
    const int b = blockIdx.y;
    proposal_finalize_body(seg_at(boxes, ws_stride, b), seg_at(keep, ws_stride, b), seg_at(num_keep, ws_stride, b),
                           proposal_count, img_h, img_w, out + (size_t)proposal_count * b, num_out + b);
}

struct ProposalBuffers {
    SelectState *state;
    unsigned *hist;
    int *blk_eq;
    float *cand_score;
    int *cand_idx;
    int *keep;
    int *num_keep;
    void *nms;
};

constexpr int SEL_MAX_BLOCKS = 1024;

static size_t proposal_ws_bytes(int K)
{
    size_t b = 0;
    b += 256;                                                    // state
    b += align_up(sizeof(unsigned) * 3 * SEL_BINS, 256);         // hist (one per pass)
    b += align_up(sizeof(int) * SEL_MAX_BLOCKS, 256);            // blk_eq
    b += align_up(sizeof(float) * (size_t)K, 256);               // cand_score
    b += 2 * align_up(sizeof(int) * (size_t)K, 256);             // cand_idx, keep
    b += 256;                                                    // num_keep
    b += nms_buffers_bytes(K);
    return b;
}

static void proposal_carve(void *ws, int K, ProposalBuffers &b)
{
    unsigned char *p = static_cast<unsigned char *>(ws);
    b.state = reinterpret_cast<SelectState *>(p);  p += 256;
    b.hist = reinterpret_cast<unsigned *>(p);      p += align_up(sizeof(unsigned) * 3 * SEL_BINS, 256);
    b.blk_eq = reinterpret_cast<int *>(p);         p += align_up(sizeof(int) * SEL_MAX_BLOCKS, 256);
    b.cand_score = reinterpret_cast<float *>(p);   p += align_up(sizeof(float) * (size_t)K, 256);
    b.cand_idx = reinterpret_cast<int *>(p);       p += align_up(sizeof(int) * (size_t)K, 256);
    b.keep = reinterpret_cast<int *>(p);           p += align_up(sizeof(int) * (size_t)K, 256);
    b.num_keep = reinterpret_cast<int *>(p);       p += 256;
    b.nms = p;
}

}  // namespace sln

using namespace sln;

extern "C" size_t sln_proposal_workspace_bytes(int A, int pre_nms_limit)
{
    if (A < 0 || pre_nms_limit < 0) return 0;
    return proposal_ws_bytes(A < pre_nms_limit ? A : pre_nms_limit);
}

extern "C" int sln_proposal_layer(const float *probs, const float *deltas, const float *anchors, int A,
                                  int pre_nms_limit, int proposal_count, float nms_thresh,
                                  const float *std_dev_host, float img_h, float img_w, float *out_boxes,
                                  int *num_out, void *workspace, size_t workspace_bytes, void *stream)
{
    SLN_REQUIRE(A >= 0 && pre_nms_limit >= 0 && proposal_count >= 0, SLN_ERR_ARG, "negative size");
    SLN_REQUIRE(num_out && std_dev_host, SLN_ERR_ARG, "null pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int K = A < pre_nms_limit ? A : pre_nms_limit;
    if (proposal_count > 0) SLN_REQUIRE(out_boxes, SLN_ERR_ARG, "null out_boxes");
    if (K == 0 || proposal_count == 0) {
        SLN_CUDA_OK(cudaMemsetAsync(num_out, 0, sizeof(int), st));
        if (proposal_count > 0)
            SLN_CUDA_OK(cudaMemsetAsync(out_boxes, 0, sizeof(float) * 4 * (size_t)proposal_count, st));
        return SLN_OK;
    }
    SLN_REQUIRE(probs && deltas && anchors, SLN_ERR_ARG, "null pointer");
    SLN_REQUIRE((reinterpret_cast<uintptr_t>(deltas) & 15u) == 0 && (reinterpret_cast<uintptr_t>(anchors) & 15u) == 0 &&
                    (reinterpret_cast<uintptr_t>(out_boxes) & 15u) == 0,
                SLN_ERR_LAYOUT, "deltas / anchors / out_boxes must be 16-byte aligned");
    SLN_REQUIRE(workspace && workspace_bytes >= proposal_ws_bytes(K), SLN_ERR_WORKSPACE,
                "proposal workspace: need %zu bytes, got %zu", proposal_ws_bytes(K), workspace_bytes);
    ProposalBuffers b;
    proposal_carve(workspace, K, b);
    NmsBuffers nb;
    nms_carve(b.nms, K, nb);

    if (K == A) {
        select_all_kernel<<<cdiv(A, 256), 256, 0, st>>>(probs, A, b.cand_score, b.cand_idx);
        SLN_LAUNCH_OK("select_all_kernel");
    } else {
        int nblk = 4 * sm_count();
        if (nblk > SEL_MAX_BLOCKS) nblk = SEL_MAX_BLOCKS;
        if (nblk > cdiv(A, SEL_THREADS)) nblk = cdiv(A, SEL_THREADS);
        SLN_CUDA_OK(cudaMemsetAsync(b.hist, 0, sizeof(unsigned) * 3 * SEL_BINS, st));
        select_hist_kernel<0><<<nblk, SEL_THREADS, 0, st>>>(probs, A, K, b.state, b.hist);
        SLN_LAUNCH_OK("select_hist_kernel");
        // the rest of the select chain as programmatic dependent launches (common.cuh): every kernel starts with pdl_prologue()
        SLN_CUDA_OK(launch_chain(select_hist_kernel<1>, dim3(nblk), dim3(SEL_THREADS), 0, st, true, probs, A, K, b.state, b.hist));   // picks pass 0 -> state[1]
        SLN_CUDA_OK(launch_chain(select_hist_kernel<2>, dim3(nblk), dim3(SEL_THREADS), 0, st, true, probs, A, K, b.state, b.hist));   // picks pass 1 -> state[0]
        SLN_CUDA_OK(launch_chain(select_count_eq_kernel, dim3(nblk), dim3(SEL_THREADS), 0, st, true, probs, A, K, b.state,
                                 (const unsigned *)b.hist, b.blk_eq));                                                           // picks pass 2 -> state[1]
        SLN_CUDA_OK(launch_chain(select_compact_kernel, dim3(nblk), dim3(SEL_THREADS), 0, st, true, probs, A, b.state,
                                 (const int *)b.blk_eq, b.cand_score, b.cand_idx));
    }
    SLN_CUDA_OK(cudaMemsetAsync(nb.rank, 0, sizeof(int) * (size_t)K, st));
    int rc = rank_sort_launch(b.cand_score, 1, b.cand_idx, K, nb.rank, st);
    if (rc != SLN_OK) return rc;
    Float4Std sd{std_dev_host[0], std_dev_host[1], std_dev_host[2], std_dev_host[3]};
    SLN_CUDA_OK(launch_chain(proposal_decode_kernel, dim3(cdiv(K, 128)), dim3(128), 0, st, true, anchors, deltas,
                             (const int *)b.cand_idx, (const int *)nb.rank, K, sd, img_h, img_w, nb.boxes, nb.areas));
    rc = nms_sorted_launch(nb.boxes, nb.areas, nullptr, nullptr, K, nms_thresh, proposal_count, nb.mask, nullptr,
                           b.keep, b.num_keep, st, nb.stage, nb.fix, nb.sparse);
    if (rc != SLN_OK) return rc;
    proposal_finalize_kernel<<<cdiv(proposal_count, 128), 128, 0, st>>>(
        nb.boxes, b.keep, b.num_keep, proposal_count, img_h, img_w, reinterpret_cast<float4 *>(out_boxes), num_out);
    SLN_LAUNCH_OK("proposal_finalize_kernel");
    return SLN_OK;
}

// ---------------------------------------------------------------------------
// B images per call.  The workspace is B copies of the single-image one, ws_stride = proposal_ws_bytes(K) apart (a
// multiple of 256, so every array keeps its alignment); every stage is one launch over all images, the image on a grid
// dimension, except the dense NMS fallback, which runs per image behind that image's sparse status word
// (nms_sorted_batched_launch).  Each image goes through the single-image kernels' bodies with the single-image
// parameters (K, thresholds, grid shapes per image aside), so its result is sln_proposal_layer's bit for bit.
// ---------------------------------------------------------------------------
extern "C" size_t sln_proposal_batched_workspace_bytes(int B, int A, int pre_nms_limit)
{
    if (B < 0 || A < 0 || pre_nms_limit < 0) return 0;
    return (size_t)B * proposal_ws_bytes(A < pre_nms_limit ? A : pre_nms_limit);
}

extern "C" int sln_proposal_layer_batched(const float *probs, const float *deltas, const float *anchors, int B, int A,
                                          int pre_nms_limit, int proposal_count, float nms_thresh,
                                          const float *std_dev_host, float img_h, float img_w, float *out_boxes,
                                          int *num_out, void *workspace, size_t workspace_bytes, void *stream)
{
    SLN_REQUIRE(B >= 0 && A >= 0 && pre_nms_limit >= 0 && proposal_count >= 0, SLN_ERR_ARG, "negative size");
    SLN_REQUIRE(B <= 65535, SLN_ERR_ARG, "B=%d images in one call (at most 65535)", B);
    if (B == 0) return SLN_OK;
    SLN_REQUIRE(num_out && std_dev_host, SLN_ERR_ARG, "null pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int K = A < pre_nms_limit ? A : pre_nms_limit;
    if (proposal_count > 0) SLN_REQUIRE(out_boxes, SLN_ERR_ARG, "null out_boxes");
    if (K == 0 || proposal_count == 0) {
        SLN_CUDA_OK(cudaMemsetAsync(num_out, 0, sizeof(int) * (size_t)B, st));
        if (proposal_count > 0)
            SLN_CUDA_OK(cudaMemsetAsync(out_boxes, 0, sizeof(float) * 4 * (size_t)proposal_count * B, st));
        return SLN_OK;
    }
    SLN_REQUIRE(probs && deltas && anchors, SLN_ERR_ARG, "null pointer");
    SLN_REQUIRE((reinterpret_cast<uintptr_t>(deltas) & 15u) == 0 && (reinterpret_cast<uintptr_t>(anchors) & 15u) == 0 &&
                    (reinterpret_cast<uintptr_t>(out_boxes) & 15u) == 0,
                SLN_ERR_LAYOUT, "deltas / anchors / out_boxes must be 16-byte aligned");
    const size_t S = proposal_ws_bytes(K);
    SLN_REQUIRE(workspace && workspace_bytes >= S * B, SLN_ERR_WORKSPACE,
                "batched proposal workspace: need %zu bytes, got %zu", S * B, workspace_bytes);
    ProposalBuffers b;
    proposal_carve(workspace, K, b);
    NmsBuffers nb;
    nms_carve(b.nms, K, nb);

    if (K == A) {
        select_all_seg_kernel<<<dim3(cdiv(A, 256), B), 256, 0, st>>>(probs, A, b.cand_score, b.cand_idx, S);
        SLN_LAUNCH_OK("select_all_seg_kernel");
    } else {
        // about the grid of one single-image call in all: fewer CTAs per image as B grows
        int nblk = cdiv(4 * sm_count(), B);
        if (nblk > SEL_MAX_BLOCKS) nblk = SEL_MAX_BLOCKS;
        if (nblk > cdiv(A, SEL_THREADS)) nblk = cdiv(A, SEL_THREADS);
        // every image's three histograms: one strided memset
        SLN_CUDA_OK(cudaMemset2DAsync(b.hist, S, 0, sizeof(unsigned) * 3 * SEL_BINS, B, st));
        const dim3 grid(nblk, B);
        select_hist_seg_kernel<0><<<grid, SEL_THREADS, 0, st>>>(probs, A, K, b.state, b.hist, S);
        SLN_LAUNCH_OK("select_hist_seg_kernel");
        SLN_CUDA_OK(launch_chain(select_hist_seg_kernel<1>, grid, dim3(SEL_THREADS), 0, st, true, probs, A, K, b.state, b.hist, S));
        SLN_CUDA_OK(launch_chain(select_hist_seg_kernel<2>, grid, dim3(SEL_THREADS), 0, st, true, probs, A, K, b.state, b.hist, S));
        SLN_CUDA_OK(launch_chain(select_count_eq_seg_kernel, grid, dim3(SEL_THREADS), 0, st, true, probs, A, K, b.state,
                                 (const unsigned *)b.hist, b.blk_eq, S));
        SLN_CUDA_OK(launch_chain(select_compact_seg_kernel, grid, dim3(SEL_THREADS), 0, st, true, probs, A, b.state,
                                 (const int *)b.blk_eq, b.cand_score, b.cand_idx, S));
    }
    SLN_CUDA_OK(cudaMemset2DAsync(nb.rank, S, 0, sizeof(int) * (size_t)K, B, st));
    int rc = rank_sort_batched_launch(b.cand_score, b.cand_idx, K, B, S, nb.rank, st);
    if (rc != SLN_OK) return rc;
    Float4Std sd{std_dev_host[0], std_dev_host[1], std_dev_host[2], std_dev_host[3]};
    SLN_CUDA_OK(launch_chain(proposal_decode_seg_kernel, dim3(cdiv(K, 128), B), dim3(128), 0, st, true, anchors, deltas, A,
                             (const int *)b.cand_idx, (const int *)nb.rank, K, sd, img_h, img_w, nb.boxes, nb.areas, S));
    rc = nms_sorted_batched_launch(B, S, nb.boxes, nb.areas, nullptr, nullptr, K, nms_thresh, proposal_count, nb.mask, nullptr,
                                   b.keep, S, b.num_keep, S, st, nb.stage, nb.fix, nb.sparse);
    if (rc != SLN_OK) return rc;
    proposal_finalize_seg_kernel<<<dim3(cdiv(proposal_count, 128), B), 128, 0, st>>>(
        nb.boxes, b.keep, b.num_keep, proposal_count, img_h, img_w, reinterpret_cast<float4 *>(out_boxes), num_out, S);
    SLN_LAUNCH_OK("proposal_finalize_seg_kernel");
    return SLN_OK;
}
