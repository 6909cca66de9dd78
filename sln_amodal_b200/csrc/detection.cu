// detection.cu -- the elementwise front of refine_detections (reference modal/Functions.py:453-557) in one launch.
//
// Per ROI: class = argmax of the class probabilities (:468, first maximum), class-specific deltas scaled by
// RPN_BBOX_STD_DEV (:436-450), apply_box_deltas in normalised coordinates (:77-98), scale to pixels, clip to the
// window (:423-433), round half-to-even (:485), and the keep filter `class_id > 0 [and score >= min_confidence]`
// (:488-493).  The reference spends ~25 small torch kernels on this; every operation below is rounded separately in the
// same order, `exp` goes through double (within 1 ulp of torch's CPU exp, like proposal.cu).
//
// Output is laid out for sln_nms: dets [N][5] = (y1, x1, y2, x2, score) and a class id per box.  Boxes that fail the
// filter get score -inf and a unique negative class, so the class-aware NMS keeps them (nothing shares their class) at
// the very end of its score-ordered output; *n_excluded says how many to drop from the tail.
#include "common.cuh"

#include <math.h>

namespace sln {

__global__ void __launch_bounds__(128)
refine_decode_kernel(const float *__restrict__ rois, const float *__restrict__ probs, const float *__restrict__ deltas,
                     int N, int K, float s0, float s1, float s2, float s3, float img_h, float img_w, float wy1,
                     float wx1, float wy2, float wx2, float min_conf, int use_min_conf, float *__restrict__ dets,
                     int *__restrict__ cls_nms, int *__restrict__ class_ids, int *__restrict__ n_excluded)
{
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);      // warp per ROI: the K probabilities are one row
    if (i >= N) return;
    // argmax, first maximum (torch.max on the CPU reference); NaN never wins
    float best = -INFINITY;
    int arg = 0x7fffffff;
    for (int k = lane; k < K; k += 32) {
        const float p = __ldg(probs + (size_t)i * K + k);
        if (p > best) { best = p; arg = k; }
    }
    for (int o = 16; o > 0; o >>= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
        if (ob > best || (ob == best && oa < arg)) { best = ob; arg = oa; }
    }
    if (arg == 0x7fffffff) arg = 0;                                        // all NaN / -inf: class 0 (filtered out)
    if (lane != 0) return;
    const float score = __ldg(probs + (size_t)i * K + arg);
    const float4 r = *reinterpret_cast<const float4 *>(rois + 4 * (size_t)i);
    const float4 dl = *reinterpret_cast<const float4 *>(deltas + ((size_t)i * K + arg) * 4);
    const float dy = __fmul_rn(dl.x, s0), dx = __fmul_rn(dl.y, s1), dh = __fmul_rn(dl.z, s2), dw = __fmul_rn(dl.w, s3);
    float height = __fsub_rn(r.z, r.x), width = __fsub_rn(r.w, r.y);
    float cy = __fadd_rn(r.x, __fmul_rn(0.5f, height)), cx = __fadd_rn(r.y, __fmul_rn(0.5f, width));
    cy = __fadd_rn(cy, __fmul_rn(dy, height));
    cx = __fadd_rn(cx, __fmul_rn(dx, width));
    height = __fmul_rn(height, (float)exp((double)dh));
    width = __fmul_rn(width, (float)exp((double)dw));
    float y1 = __fsub_rn(cy, __fmul_rn(0.5f, height)), x1 = __fsub_rn(cx, __fmul_rn(0.5f, width));
    float y2 = __fadd_rn(y1, height), x2 = __fadd_rn(x1, width);
    y1 = __fmul_rn(y1, img_h); x1 = __fmul_rn(x1, img_w); y2 = __fmul_rn(y2, img_h); x2 = __fmul_rn(x2, img_w);
    // torch.clamp(min, max): NaN passes through
    auto clampf = [](float v, float lo, float hi) { return v < lo ? lo : (v > hi ? hi : v); };
    y1 = rintf(clampf(y1, wy1, wy2)); x1 = rintf(clampf(x1, wx1, wx2));
    y2 = rintf(clampf(y2, wy1, wy2)); x2 = rintf(clampf(x2, wx1, wx2));
    const bool keep = arg > 0 && (!use_min_conf || score >= min_conf);
    float *o = dets + 5 * (size_t)i;
    o[0] = y1; o[1] = x1; o[2] = y2; o[3] = x2;
    o[4] = keep ? score : -INFINITY;
    cls_nms[i] = keep ? arg : -(i + 1);
    class_ids[i] = arg;
    if (!keep) atomicAdd(n_excluded, 1);                                    // integer count: order-independent
}

}  // namespace sln

extern "C" int sln_refine_decode(const float *rois, const float *probs, const float *deltas, int N, int K,
                                 const float *std_dev_host, float img_h, float img_w, const float *window_host,
                                 float min_confidence, float *dets, int *cls_nms, int *class_ids, int *n_excluded,
                                 void *stream)
{
    SLN_REQUIRE(N >= 0 && K >= 1, SLN_ERR_ARG, "need N >= 0 and K >= 1 (got %d, %d)", N, K);
    SLN_REQUIRE(n_excluded && std_dev_host && window_host, SLN_ERR_ARG, "null pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    SLN_CUDA_OK(cudaMemsetAsync(n_excluded, 0, sizeof(int), st));
    if (N == 0) return SLN_OK;
    SLN_REQUIRE(rois && probs && deltas && dets && cls_nms && class_ids, SLN_ERR_ARG, "null pointer");
    SLN_REQUIRE((reinterpret_cast<uintptr_t>(rois) & 15u) == 0 && (reinterpret_cast<uintptr_t>(deltas) & 15u) == 0,
                SLN_ERR_LAYOUT, "rois / deltas must be 16-byte aligned");
    const int use_min = min_confidence != 0.f;                              // `if config.DETECTION_MIN_CONFIDENCE:` (:490)
    sln::refine_decode_kernel<<<sln::cdiv(N, 4), 128, 0, st>>>(rois, probs, deltas, N, K, std_dev_host[0], std_dev_host[1],
                                                               std_dev_host[2], std_dev_host[3], img_h, img_w,
                                                               window_host[0], window_host[1], window_host[2],
                                                               window_host[3], min_confidence, use_min, dets, cls_nms,
                                                               class_ids, n_excluded);
    SLN_LAUNCH_OK("refine_decode_kernel");
    return SLN_OK;
}

// ---------------------------------------------------------------------------
// refine_detections without NMS (the reference's shipped default, config.py:78 USE_NMS = False): of the ROIs whose
// argmax class is not background keep the `max_keep` best by score (Functions.py:528-532) and emit them in descending
// score order (:538-546).  Ties are broken by the lower ROI index (torch's sort leaves them unspecified; same rule as
// the NMS front).  Every thread ranks one ROI against all others (scores staged through shared memory, 4 keys per
// 16-byte load); ROIs ranked below max_keep write their output row directly, so select + sort + the three gathers +
// cat of the torch expression are this one launch.  dets / class_ids are sln_refine_decode's outputs (score = -inf for
// filtered ROIs, which therefore never take part).
namespace sln {

constexpr int TOPK_THREADS = 256;

// num_det (nullptr in the single-image kernel): one count per written row, i.e. min(#valid rows, max_keep) in all
__device__ __forceinline__ void refine_topk_body(const float *dets, const int *class_ids, int N,
                                                 int max_keep, float *result, long long *keep,
                                                 int *num_det)
{
    __shared__ __align__(16) float s_score[TOPK_THREADS];
    const int i = blockIdx.x * TOPK_THREADS + threadIdx.x;
    float si = -INFINITY;
    bool valid = false;
    if (i < N) {
        si = __ldg(dets + 5 * (size_t)i + 4);
        valid = __ldg(class_ids + i) > 0 && si > -INFINITY;
    }
    int rank = 0;
    for (int j0 = 0; j0 < N; j0 += TOPK_THREADS) {
        const int j = j0 + threadIdx.x;
        float sj = -INFINITY;                                  // filtered and out-of-range ROIs never precede anyone
        if (j < N && __ldg(class_ids + j) > 0) sj = __ldg(dets + 5 * (size_t)j + 4);
        __syncthreads();
        s_score[threadIdx.x] = sj;
        __syncthreads();
        const int lim = min(TOPK_THREADS, N - j0);
        // entries before i in index order win ties, entries after it do not
        const int split = min(max(i - j0, 0), lim);            // j0 + k < i  <=>  k < split
        int k = 0;
        for (; k + 4 <= split; k += 4) {
            const float4 v = *reinterpret_cast<const float4 *>(s_score + k);
            rank += (v.x >= si) + (v.y >= si) + (v.z >= si) + (v.w >= si);
        }
        for (; k < split; ++k) rank += s_score[k] >= si;
        k = split + ((i >= j0 && i < j0 + lim) ? 1 : 0);       // skip i itself
        for (; k < lim && (k & 3); ++k) rank += s_score[k] > si;
        for (; k + 4 <= lim; k += 4) {
            const float4 v = *reinterpret_cast<const float4 *>(s_score + k);
            rank += (v.x > si) + (v.y > si) + (v.z > si) + (v.w > si);
        }
        for (; k < lim; ++k) rank += s_score[k] > si;
    }
    if (!valid || rank >= max_keep) return;
    const float *d = dets + 5 * (size_t)i;
    float *o = result + 6 * (size_t)rank;
    o[0] = d[0]; o[1] = d[1]; o[2] = d[2]; o[3] = d[3];
    o[4] = (float)__ldg(class_ids + i);
    o[5] = si;
    keep[rank] = i;
    if (num_det) atomicAdd(num_det, 1);
}

__global__ void __launch_bounds__(TOPK_THREADS)
refine_topk_kernel(const float *__restrict__ dets, const int *__restrict__ class_ids, int N, int max_keep,
                   float *__restrict__ result, long long *__restrict__ keep)
{
    refine_topk_body(dets, class_ids, N, max_keep, result, keep, nullptr);
}

// image b = blockIdx.y: rows [b*N, (b+1)*N), ranked among themselves; keep holds row indices within the image
__global__ void __launch_bounds__(TOPK_THREADS)
refine_topk_seg_kernel(const float *__restrict__ dets, const int *__restrict__ class_ids, int N, int max_keep,
                       float *__restrict__ result, long long *__restrict__ keep, int *__restrict__ num_det)
{
    const size_t b = blockIdx.y;
    refine_topk_body(dets + 5 * (size_t)N * b, class_ids + (size_t)N * b, N, max_keep, result + 6 * (size_t)max_keep * b,
                     keep + (size_t)max_keep * b, num_det + b);
}

}  // namespace sln

extern "C" int sln_refine_topk(const float *dets, const int *class_ids, int N, int max_keep, float *result,
                               int64_t *keep, void *stream)
{
    SLN_REQUIRE(N >= 0 && max_keep >= 0, SLN_ERR_ARG, "negative size");
    if (N == 0 || max_keep == 0) return SLN_OK;
    SLN_REQUIRE(dets && class_ids && result && keep, SLN_ERR_ARG, "null pointer");
    sln::refine_topk_kernel<<<sln::cdiv(N, sln::TOPK_THREADS), sln::TOPK_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
        dets, class_ids, N, max_keep, result, reinterpret_cast<long long *>(keep));
    SLN_LAUNCH_OK("refine_topk_kernel");
    return SLN_OK;
}

extern "C" int sln_refine_topk_batched(const float *dets, const int *class_ids, int B, int N, int max_keep, float *result,
                                       int64_t *keep, int *num_det, void *stream)
{
    SLN_REQUIRE(B >= 0 && N >= 0 && max_keep >= 0, SLN_ERR_ARG, "negative size");
    SLN_REQUIRE(B <= 65535, SLN_ERR_ARG, "B=%d images in one call (at most 65535)", B);
    if (B == 0) return SLN_OK;
    SLN_REQUIRE(num_det, SLN_ERR_ARG, "null num_det");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    SLN_CUDA_OK(cudaMemsetAsync(num_det, 0, sizeof(int) * (size_t)B, st));
    if (N == 0 || max_keep == 0) return SLN_OK;
    SLN_REQUIRE(dets && class_ids && result && keep, SLN_ERR_ARG, "null pointer");
    sln::refine_topk_seg_kernel<<<dim3(sln::cdiv(N, sln::TOPK_THREADS), B), sln::TOPK_THREADS, 0, st>>>(
        dets, class_ids, N, max_keep, result, reinterpret_cast<long long *>(keep), num_det);
    SLN_LAUNCH_OK("refine_topk_seg_kernel");
    return SLN_OK;
}

// ---------------------------------------------------------------------------
// refine_detections with per-class NMS (USE_NMS = True), B images: the step after sln_nms_batched, which ran on
// sln_refine_decode's dets / cls_nms with max_keep = D.  Filtered rows carry score -inf and a class of their own, so the
// NMS never suppresses them and visits them last: the rows with a finite score are a prefix of every image's keep list,
// and its length is min(D, survivors).  Stopping the greedy NMS after D survivors does not change the first D, so this
// equals the first D rows of the single-image path (_refine_detections_fused), which runs the NMS to the end.
// One CTA per image (blockIdx.y), rows strided over its threads; rows at and beyond the count are zero.
namespace sln {

constexpr int EMIT_THREADS = 256;

__global__ void __launch_bounds__(EMIT_THREADS)
refine_nms_emit_seg_kernel(const float *__restrict__ dets, const int *__restrict__ class_ids, int N,
                           const long long *__restrict__ nms_keep, const int *__restrict__ nms_num, int nms_stride, int D,
                           float *__restrict__ result, long long *__restrict__ keep, int *__restrict__ num_det)
{
    const size_t b = blockIdx.y;
    const int nk = min(__ldg(nms_num + b), nms_stride);
    int count = 0;
    for (int r0 = 0; r0 < D; r0 += EMIT_THREADS) {
        const int r = r0 + threadIdx.x;
        long long idx = 0;
        float s = -INFINITY;
        if (r < D && r < nk) {
            idx = __ldg(nms_keep + b * (size_t)nms_stride + r);
            s = __ldg(dets + 5 * ((size_t)N * b + (size_t)idx) + 4);
        }
        const bool valid = s > -INFINITY;
        if (r < D) {
            float *o = result + 6 * ((size_t)D * b + r);
            if (valid) {
                const float *d = dets + 5 * ((size_t)N * b + (size_t)idx);
                o[0] = d[0]; o[1] = d[1]; o[2] = d[2]; o[3] = d[3];
                o[4] = (float)__ldg(class_ids + (size_t)N * b + (size_t)idx);
                o[5] = s;
            } else {
                o[0] = o[1] = o[2] = o[3] = o[4] = o[5] = 0.f;
            }
            keep[(size_t)D * b + r] = valid ? idx : 0;
        }
        count += __syncthreads_count(valid);
    }
    if (threadIdx.x == 0) num_det[b] = count;
}

}  // namespace sln

extern "C" int sln_refine_nms_emit_batched(const float *dets, const int *class_ids, int B, int N, const int64_t *nms_keep,
                                           const int *nms_num_keep, int nms_max_keep, int D, float *result, int64_t *keep,
                                           int *num_det, void *stream)
{
    SLN_REQUIRE(B >= 0 && N >= 0 && nms_max_keep >= 0 && D >= 0, SLN_ERR_ARG, "negative size");
    SLN_REQUIRE(B <= 65535, SLN_ERR_ARG, "B=%d images in one call (at most 65535)", B);
    if (B == 0) return SLN_OK;
    SLN_REQUIRE(num_det && nms_num_keep, SLN_ERR_ARG, "null pointer");
    SLN_REQUIRE(D == 0 || (result && keep), SLN_ERR_ARG, "null pointer");
    SLN_REQUIRE(N == 0 || nms_max_keep == 0 || (dets && class_ids && nms_keep), SLN_ERR_ARG, "null pointer");
    sln::refine_nms_emit_seg_kernel<<<dim3(1, B), sln::EMIT_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
        dets, class_ids, N, reinterpret_cast<const long long *>(nms_keep), nms_num_keep, nms_max_keep, D, result,
        reinterpret_cast<long long *>(keep), num_det);
    SLN_LAUNCH_OK("refine_nms_emit_seg_kernel");
    return SLN_OK;
}

// ---------------------------------------------------------------------------
// SURVEY 8(f)-1: detection targets -- IoU matching and box refinement
// ---------------------------------------------------------------------------
// bbox_overlaps (modal/Functions.py:184-218): IoU of every box of set 1 against every box of set 2, no "+1"
// convention, each operation rounded separately, 0/0 -> NaN like the torch expression.  The reference materialises
// two [N*G,4] repeat tensors and ~20 elementwise kernels; here one thread walks the G boxes of a row and optionally
// also produces what detection_target_layer wants from the matrix: the row maximum and its first index
// (torch.max semantics: a NaN in the row is the maximum).
namespace sln {

// IoU of box a (area1 = its area) against box g, bbox_overlaps' operation sequence.  Shared by bbox_overlaps_kernel and
// the batched match kernel, so that both round the same way.
__device__ __forceinline__ float iou_f32(const float4 a, float area1, const float4 g)
{
    const float y1 = fmaxf(a.x, g.x), x1 = fmaxf(a.y, g.y), y2 = fminf(a.z, g.z), x2 = fminf(a.w, g.w);
    // torch.max(x2 - x1, zeros): NaN-propagating in torch, fmaxf is not -- handled through `inter != inter` below
    const float dx = __fsub_rn(x2, x1), dy = __fsub_rn(y2, y1);
    float inter = __fmul_rn(dx > 0.f ? dx : (dx != dx ? dx : 0.f), dy > 0.f ? dy : (dy != dy ? dy : 0.f));
    const float area2 = __fmul_rn(__fsub_rn(g.z, g.x), __fsub_rn(g.w, g.y));
    const float uni = __fsub_rn(__fadd_rn(area1, area2), inter);
    return __fdiv_rn(inter, uni);
}

__device__ __forceinline__ float box_area_f32(const float4 a) { return __fmul_rn(__fsub_rn(a.z, a.x), __fsub_rn(a.w, a.y)); }

// torch.max(dim) over a row visited in index order: the first NaN is the maximum and stays, else the first strict maximum
__device__ __forceinline__ void row_max_update(float v, int j, float &best, int &arg, bool &best_nan)
{
    const bool vnan = v != v;
    if (!best_nan && (vnan || v > best)) { best = v; arg = j; best_nan = vnan; }
}

__global__ void __launch_bounds__(128)
bbox_overlaps_kernel(const float *__restrict__ b1, int N, const float *__restrict__ b2, int G,
                     float *__restrict__ overlaps, float *__restrict__ iou_max, int *__restrict__ argmax)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const float4 a = *reinterpret_cast<const float4 *>(b1 + 4 * (size_t)i);          // (y1, x1, y2, x2)
    const float area1 = box_area_f32(a);
    float best = -INFINITY;
    int arg = 0;
    bool best_nan = false;
    for (int j = 0; j < G; ++j) {
        const float4 g = __ldg(reinterpret_cast<const float4 *>(b2) + j);
        const float v = iou_f32(a, area1, g);
        if (overlaps) overlaps[(size_t)i * G + j] = v;
        const bool vnan = v != v;
        if (!best_nan && (vnan || v > best)) { best = v; arg = j; best_nan = vnan; }
    }
    if (iou_max) iou_max[i] = best;
    if (argmax) argmax[i] = arg;
}

// utils.box_refinement (utils.py:96-117) of box b onto gt box g, optionally divided by BBOX_STD_DEV (Functions.py:309-313)
__device__ __forceinline__ float4 box_refinement_f32(const float4 b, const float4 g, int use_std, float s0, float s1,
                                                     float s2, float s3)
{
    const float h = __fsub_rn(b.z, b.x), w = __fsub_rn(b.w, b.y);
    const float cy = __fadd_rn(b.x, __fmul_rn(0.5f, h)), cx = __fadd_rn(b.y, __fmul_rn(0.5f, w));
    const float gh = __fsub_rn(g.z, g.x), gw = __fsub_rn(g.w, g.y);
    const float gcy = __fadd_rn(g.x, __fmul_rn(0.5f, gh)), gcx = __fadd_rn(g.y, __fmul_rn(0.5f, gw));
    float dy = __fdiv_rn(__fsub_rn(gcy, cy), h), dx = __fdiv_rn(__fsub_rn(gcx, cx), w);
    float dh = (float)log((double)__fdiv_rn(gh, h)), dw = (float)log((double)__fdiv_rn(gw, w));   // within 1 ulp of torch's CPU log
    if (use_std) { dy = __fdiv_rn(dy, s0); dx = __fdiv_rn(dx, s1); dh = __fdiv_rn(dh, s2); dw = __fdiv_rn(dw, s3); }
    return make_float4(dy, dx, dh, dw);
}

__global__ void __launch_bounds__(128)
box_refinement_kernel(const float *__restrict__ box, const float *__restrict__ gt, int M, int use_std, float s0,
                      float s1, float s2, float s3, float *__restrict__ out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    const float4 b = *reinterpret_cast<const float4 *>(box + 4 * (size_t)i);
    const float4 g = *reinterpret_cast<const float4 *>(gt + 4 * (size_t)i);
    *reinterpret_cast<float4 *>(out + 4 * (size_t)i) = box_refinement_f32(b, g, use_std, s0, s1, s2, s3);
}

}  // namespace sln

extern "C" int sln_bbox_overlaps(const float *boxes1, int N, const float *boxes2, int G, float *overlaps,
                                 float *iou_max, int *argmax, void *stream)
{
    SLN_REQUIRE(N >= 0 && G >= 0, SLN_ERR_ARG, "negative size");
    if (N == 0) return SLN_OK;
    SLN_REQUIRE(boxes1 && (boxes2 || G == 0), SLN_ERR_ARG, "null pointer");
    SLN_REQUIRE((reinterpret_cast<uintptr_t>(boxes1) & 15u) == 0 && (reinterpret_cast<uintptr_t>(boxes2) & 15u) == 0,
                SLN_ERR_LAYOUT, "boxes must be 16-byte aligned");
    sln::bbox_overlaps_kernel<<<sln::cdiv(N, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(boxes1, N, boxes2, G,
                                                                                              overlaps, iou_max, argmax);
    SLN_LAUNCH_OK("bbox_overlaps_kernel");
    return SLN_OK;
}

extern "C" int sln_box_refinement(const float *box, const float *gt_box, int M, const float *std_dev_host, float *out,
                                  void *stream)
{
    SLN_REQUIRE(M >= 0, SLN_ERR_ARG, "negative size");
    if (M == 0) return SLN_OK;
    SLN_REQUIRE(box && gt_box && out, SLN_ERR_ARG, "null pointer");
    SLN_REQUIRE(((reinterpret_cast<uintptr_t>(box) | reinterpret_cast<uintptr_t>(gt_box) | reinterpret_cast<uintptr_t>(out)) & 15u) == 0,
                SLN_ERR_LAYOUT, "box / gt_box / out must be 16-byte aligned");
    const float *s = std_dev_host;
    sln::box_refinement_kernel<<<sln::cdiv(M, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
        box, gt_box, M, s != nullptr, s ? s[0] : 1.f, s ? s[1] : 1.f, s ? s[2] : 1.f, s ? s[3] : 1.f, out);
    SLN_LAUNCH_OK("box_refinement_kernel");
    return SLN_OK;
}

// ---------------------------------------------------------------------------
// mask targets (SURVEY 8a row A12 inside detection_target_layer, Functions.py:327-346)
// ---------------------------------------------------------------------------
// The reference gathers the assigned GT masks ([L,P,H,W] u8), converts every 1-MiB plane to float (280 MB per layer at
// P = 70), crops each with crop_and_resize and rounds.  Only mh*mw samples of a plane are ever read: one launch gathers
// by `assignment`, samples the u8 plane directly with the crop's exact tap arithmetic (common.cuh: axis_tap / lerp2;
// u8 -> f32 is exact) and rounds half-to-even.  out f32 [P, L, mh, mw].
namespace sln {

// Sample (y, x) of the mh x mw crop over box (y1,x1,y2,x2) of plane (l, g) of the u8 masks [L,G,H,W], before the
// rounding; 0 outside the plane (extrapolation value, :339).  Shared by mask_targets_kernel and the batched emit kernel.
__device__ __forceinline__ float mask_target_sample(const unsigned char *masks, int l, int G, int g, int H, int W,
                                                    float y1, float x1, float y2, float x2, int mh, int mw, int y, int x)
{
    float v = 0.f;
    const Tap ty = axis_tap(y1, y2, axis_scale(y1, y2, H, mh), H, mh, y);
    const Tap tx = axis_tap(x1, x2, axis_scale(x1, x2, W, mw), W, mw, x);
    if (ty.lo != INVALID_TAP && tx.lo != INVALID_TAP) {
        const unsigned char *pl = masks + ((size_t)l * G + g) * H * W;
        const int yh = ty.lo + (ty.lerp != 0.f), xh = tx.lo + (tx.lerp != 0.f);
        const float tl = (float)pl[(size_t)ty.lo * W + tx.lo], tr = (float)pl[(size_t)ty.lo * W + xh];
        const float bl = (float)pl[(size_t)yh * W + tx.lo], br = (float)pl[(size_t)yh * W + xh];
        v = lerp2(tl, tr, bl, br, tx.lerp, ty.lerp);
    }
    return v;
}

__global__ void __launch_bounds__(256)
mask_targets_kernel(const unsigned char *__restrict__ masks, int L, int G, int H, int W, const int *__restrict__ assignment,
                    const float *__restrict__ boxes, int P, int mh, int mw, float *__restrict__ out)
{
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)P * L * mh * mw;
    if (idx >= total) return;
    const int x = (int)(idx % mw);
    const int y = (int)((idx / mw) % mh);
    const int l = (int)((idx / ((long long)mw * mh)) % L);
    const int p = (int)(idx / ((long long)mw * mh * L));
    const int gidx = assignment[p];
    float v = 0.f;                                                        // extrapolation value 0 (:339)
    if (gidx >= 0 && gidx < G)
        v = mask_target_sample(masks, l, G, gidx, H, W, boxes[4 * p + 0], boxes[4 * p + 1], boxes[4 * p + 2],
                               boxes[4 * p + 3], mh, mw, y, x);
    out[idx] = rintf(v);                                                  // torch.round (:346)
}

}  // namespace sln

extern "C" int sln_mask_targets(const uint8_t *gt_masks, int L, int G, int H, int W, const int *assignment,
                                const float *boxes, int P, int mh, int mw, float *out, void *stream)
{
    SLN_REQUIRE(L >= 0 && G >= 0 && H >= 0 && W >= 0 && P >= 0 && mh >= 1 && mw >= 1, SLN_ERR_ARG, "bad size");
    const long long total = (long long)P * L * mh * mw;
    if (total == 0) return SLN_OK;
    SLN_REQUIRE(gt_masks && assignment && boxes && out, SLN_ERR_ARG, "null pointer");
    SLN_REQUIRE(H > 0 && W > 0 && H <= 32767 && W <= 32767, SLN_ERR_ARG, "mask side outside [1, 32767]");
    SLN_REQUIRE((total + 255) / 256 < (1ll << 31), SLN_ERR_ARG, "too many target samples");
    sln::mask_targets_kernel<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        gt_masks, L, G, H, W, assignment, boxes, P, mh, mw, out);
    SLN_LAUNCH_OK("mask_targets_kernel");
    return SLN_OK;
}

// ---------------------------------------------------------------------------
// detection_target_layer for B images: a match launch, one host round trip (sampling), an emit launch
// ---------------------------------------------------------------------------
// Match: one thread per proposal row of image b = blockIdx.y.  The candidates are the image's first num_gt[b] GT rows,
// or, when one of them has a class < 0 (a COCO crowd), its rows with class > 0 (Functions.py:253-267); the argmax is the
// candidate's index in gt_boxes[b] (the single-image path compacts the candidates in order, so its first maximum is the
// same box).  codes[b, i] bit 0 = positive (iou_max >= 0.5, :279), bit 1 = negative-eligible (iou_max < 0.5, and in a
// crowd image crowd_iou_max < 0.001, :351-352).  A row whose iou_max is NaN is neither, as in the reference (NaN
// compares false); rows at and beyond num_proposals[b] get 0.  The GT counts travel by value: no copy before the launch.
namespace sln {

template <int NB> struct TargetGtCounts { int v[NB]; };

constexpr int TARGET_BATCH_MAX = 512;

template <int NB>
__global__ void __launch_bounds__(128)
target_match_kernel(const float *__restrict__ proposals, int R, const int *__restrict__ num_proposals,
                    const float *__restrict__ gt_boxes, const int *__restrict__ gt_class_ids, int G, const __grid_constant__ TargetGtCounts<NB> ng,
                    unsigned char *__restrict__ codes, int *__restrict__ argmax)
{
    const int b = blockIdx.y;
    const int n_gt = ng.v[b];
    const int *cls = gt_class_ids + (size_t)b * G;
    const float4 *gt = reinterpret_cast<const float4 *>(gt_boxes) + (size_t)b * G;
    int crowd = 0;
    for (int j = threadIdx.x; j < n_gt; j += blockDim.x) crowd |= __ldg(cls + j) < 0;
    crowd = __syncthreads_or(crowd);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R) return;
    const size_t o = (size_t)b * R + i;
    const int n_prop = num_proposals ? min(max(__ldg(num_proposals + b), 0), R) : R;
    if (i >= n_prop) { codes[o] = 0; argmax[o] = 0; return; }
    const float4 a = *reinterpret_cast<const float4 *>(proposals + 4 * o);
    const float area1 = box_area_f32(a);
    float best = -INFINITY, cbest = -INFINITY;
    int arg = 0, carg = 0;
    bool best_nan = false, cbest_nan = false;
    for (int j = 0; j < n_gt; ++j) {
        const int c = crowd ? __ldg(cls + j) : 1;
        if (c == 0) continue;                                   // only reached in a crowd image
        const float v = iou_f32(a, area1, __ldg(gt + j));
        if (c > 0) row_max_update(v, j, best, arg, best_nan);
        else row_max_update(v, j, cbest, carg, cbest_nan);
    }
    codes[o] = (unsigned char)((best >= 0.5f ? 1 : 0) | (best < 0.5f && (!crowd || cbest < 0.001f) ? 2 : 0));
    argmax[o] = arg;
}

template <int NB>
static int launch_target_match(const float *proposals, int B, int R, const int *num_proposals, const float *gt_boxes,
                               const int *gt_class_ids, int G, const int *num_gt_host, uint8_t *codes, int *argmax,
                               cudaStream_t st)
{
    TargetGtCounts<NB> ng;
    for (int b = 0; b < NB; ++b) ng.v[b] = b < B ? num_gt_host[b] : 0;
    target_match_kernel<NB><<<dim3(cdiv(R, 128), B), 128, 0, st>>>(proposals, R, num_proposals, gt_boxes, gt_class_ids, G,
                                                                     ng, codes, argmax);
    SLN_LAUNCH_OK("target_match_kernel");
    return SLN_OK;
}

// Emit: one CTA per output row (b, t) of the padded [B,T] result, after the host has sampled the rows.  sel[b, t] is a
// proposal row of image b for t < num_rois[b]; the first num_positive[b] rows are the positives: their GT box and class
// come through the match kernel's argmax, the deltas through box_refinement_kernel's arithmetic, the L mask targets
// through mask_targets_kernel's sampling of image b's u8 planes (mask_planes[b] = [L, mask_g[b], H, W]) over the
// proposal, or over it in the GT box's frame under USE_MINI_MASK (:316-325).  Negative rows: the proposal, class 0, zero
// deltas and masks (:370-384).  Rows at and beyond num_rois[b]: zeros.  Every output element is written.
constexpr int TARGET_EMIT_THREADS = 256;

__global__ void __launch_bounds__(TARGET_EMIT_THREADS)
detection_targets_emit_kernel(const float *__restrict__ proposals, int R, const int *__restrict__ argmax,
                              const float *__restrict__ gt_boxes, const int *__restrict__ gt_class_ids, int G,
                              const int *__restrict__ sel, const int *__restrict__ num_positive,
                              const int *__restrict__ num_rois, const uint8_t *const *__restrict__ mask_planes,
                              const int *__restrict__ mask_g, int T, int L, int H, int W, int mh, int mw, int use_std,
                              float s0, float s1, float s2, float s3, int mini_mask, float *__restrict__ rois,
                              int *__restrict__ class_ids, float *__restrict__ deltas, float *__restrict__ masks)
{
    const int row = blockIdx.x;
    const int b = row / T, t = row - b * T;
    const bool live = t < __ldg(num_rois + b);
    const bool pos = live && t < __ldg(num_positive + b);
    const int n = L * mh * mw;
    float *mo = masks + (size_t)row * n;
    float4 roi = make_float4(0.f, 0.f, 0.f, 0.f);
    if (live) roi = *reinterpret_cast<const float4 *>(proposals + 4 * ((size_t)b * R + __ldg(sel + row)));
    if (!pos) {
        if (threadIdx.x == 0) {
            *reinterpret_cast<float4 *>(rois + 4 * (size_t)row) = roi;
            class_ids[row] = 0;
            *reinterpret_cast<float4 *>(deltas + 4 * (size_t)row) = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        for (int k = threadIdx.x; k < n; k += TARGET_EMIT_THREADS) mo[k] = 0.f;
        return;
    }
    const int g = __ldg(argmax + (size_t)b * R + __ldg(sel + row));
    const float4 gt = *reinterpret_cast<const float4 *>(gt_boxes + 4 * ((size_t)b * G + g));
    if (threadIdx.x == 0) {
        *reinterpret_cast<float4 *>(rois + 4 * (size_t)row) = roi;
        class_ids[row] = __ldg(gt_class_ids + (size_t)b * G + g);
        *reinterpret_cast<float4 *>(deltas + 4 * (size_t)row) = box_refinement_f32(roi, gt, use_std, s0, s1, s2, s3);
    }
    float4 box = roi;
    if (mini_mask) {
        const float gh = __fsub_rn(gt.z, gt.x), gw = __fsub_rn(gt.w, gt.y);
        box = make_float4(__fdiv_rn(__fsub_rn(roi.x, gt.x), gh), __fdiv_rn(__fsub_rn(roi.y, gt.y), gw),
                          __fdiv_rn(__fsub_rn(roi.z, gt.x), gh), __fdiv_rn(__fsub_rn(roi.w, gt.y), gw));
    }
    const uint8_t *planes = mask_planes[b];
    const int gs = __ldg(mask_g + b);
    for (int k = threadIdx.x; k < n; k += TARGET_EMIT_THREADS) {
        const int x = k % mw, y = (k / mw) % mh, l = k / (mw * mh);
        mo[k] = rintf(mask_target_sample(planes, l, gs, g, H, W, box.x, box.y, box.z, box.w, mh, mw, y, x));
    }
}

}  // namespace sln

extern "C" int sln_target_match_batched(const float *proposals, int B, int R, const int *num_proposals,
                                        const float *gt_boxes, const int *gt_class_ids, int G, const int *num_gt_host,
                                        uint8_t *codes, int *argmax, void *stream)
{
    SLN_REQUIRE(B >= 0 && R >= 0 && G >= 0, SLN_ERR_ARG, "target_match_batched: negative size");
    SLN_REQUIRE(B <= sln::TARGET_BATCH_MAX, SLN_ERR_ARG, "target_match_batched: B=%d images in one call (at most %d)", B,
                sln::TARGET_BATCH_MAX);
    if (B == 0 || R == 0) return SLN_OK;
    SLN_REQUIRE(proposals && codes && argmax && num_gt_host, SLN_ERR_ARG, "target_match_batched: null pointer");
    for (int b = 0; b < B; ++b)
        SLN_REQUIRE(num_gt_host[b] >= 0 && num_gt_host[b] <= G, SLN_ERR_ARG,
                    "target_match_batched: num_gt[%d] = %d outside [0, G=%d]", b, num_gt_host[b], G);
    SLN_REQUIRE(G == 0 || (gt_boxes && gt_class_ids), SLN_ERR_ARG, "target_match_batched: null pointer");
    SLN_REQUIRE(((reinterpret_cast<uintptr_t>(proposals) | reinterpret_cast<uintptr_t>(gt_boxes)) & 15u) == 0,
                SLN_ERR_LAYOUT, "target_match_batched: proposals / gt_boxes must be 16-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (B <= 16)
        return sln::launch_target_match<16>(proposals, B, R, num_proposals, gt_boxes, gt_class_ids, G, num_gt_host, codes, argmax, st);
    if (B <= 128)
        return sln::launch_target_match<128>(proposals, B, R, num_proposals, gt_boxes, gt_class_ids, G, num_gt_host, codes, argmax, st);
    return sln::launch_target_match<sln::TARGET_BATCH_MAX>(proposals, B, R, num_proposals, gt_boxes, gt_class_ids, G,
                                                           num_gt_host, codes, argmax, st);
}

extern "C" int sln_detection_targets_emit_batched(const float *proposals, int B, int R, const int *argmax,
                                                  const float *gt_boxes, const int *gt_class_ids, int G, const int *sel,
                                                  const int *num_positive, const int *num_rois,
                                                  const uint8_t *const *mask_planes, const int *mask_g, int T, int L,
                                                  int H, int W, int mh, int mw, const float *std_dev_host,
                                                  int use_mini_mask, float *rois, int *class_ids, float *deltas,
                                                  float *masks, void *stream)
{
    SLN_REQUIRE(B >= 0 && R >= 0 && G >= 0 && T >= 0 && L >= 0 && H >= 0 && W >= 0 && mh >= 1 && mw >= 1, SLN_ERR_ARG,
                "detection_targets_emit_batched: bad size");
    SLN_REQUIRE(B <= sln::TARGET_BATCH_MAX, SLN_ERR_ARG, "detection_targets_emit_batched: B=%d images in one call (at most %d)",
                B, sln::TARGET_BATCH_MAX);
    if ((long long)B * T == 0) return SLN_OK;
    SLN_REQUIRE(sel && num_positive && num_rois && rois && class_ids && deltas && masks, SLN_ERR_ARG,
                "detection_targets_emit_batched: null pointer");
    SLN_REQUIRE(R == 0 || (proposals && argmax), SLN_ERR_ARG, "detection_targets_emit_batched: null pointer");
    SLN_REQUIRE(G == 0 || (gt_boxes && gt_class_ids), SLN_ERR_ARG, "detection_targets_emit_batched: null pointer");
    SLN_REQUIRE(L == 0 || (mask_planes && mask_g), SLN_ERR_ARG, "detection_targets_emit_batched: null pointer");
    SLN_REQUIRE(H <= 32767 && W <= 32767, SLN_ERR_ARG, "detection_targets_emit_batched: mask side above 32767");
    SLN_REQUIRE((long long)L * mh * mw < (1ll << 31) && (long long)B * T < (1ll << 31), SLN_ERR_ARG,
                "detection_targets_emit_batched: too many targets");
    SLN_REQUIRE(((reinterpret_cast<uintptr_t>(proposals) | reinterpret_cast<uintptr_t>(gt_boxes) |
                  reinterpret_cast<uintptr_t>(rois) | reinterpret_cast<uintptr_t>(deltas)) & 15u) == 0, SLN_ERR_LAYOUT,
                "detection_targets_emit_batched: proposals / gt_boxes / rois / deltas must be 16-byte aligned");
    const float *s = std_dev_host;
    sln::detection_targets_emit_kernel<<<(unsigned)((long long)B * T), sln::TARGET_EMIT_THREADS, 0,
                                         static_cast<cudaStream_t>(stream)>>>(
        proposals, R, argmax, gt_boxes, gt_class_ids, G, sel, num_positive, num_rois, mask_planes, mask_g, T, L, H, W, mh,
        mw, s != nullptr, s ? s[0] : 1.f, s ? s[1] : 1.f, s ? s[2] : 1.f, s ? s[3] : 1.f, use_mini_mask != 0, rois, class_ids,
        deltas, masks);
    SLN_LAUNCH_OK("detection_targets_emit_kernel");
    return SLN_OK;
}

// ---------------------------------------------------------------------------
// SURVEY 8(f)-2: the overlap reductions of build_rpn_targets (modal/Functions.py:773-792)
// ---------------------------------------------------------------------------
// The reference builds the [A, G] IoU matrix in float64 numpy (utils.compute_overlaps, 261 888 x G, one pass per GT
// box) only to take three reductions of it: per anchor the maximum and its first index (:787-788), per GT box the first
// index of its column maximum (:792) -- plus the per-anchor maximum against the crowd boxes (:769-770).  Here the
// matrix is never materialised: kernel 1 walks the G boxes of an anchor, kernel 2 (one CTA per GT box) reduces a column
// with (value, lowest index) pairs.  float64 throughout, the same operation order as compute_iou (utils.py:65-76);
// numpy's argmax / amax treat NaN as the maximum, and so do these.
namespace sln {

__device__ __forceinline__ double iou_f64(const double4 a, double area_a, const double4 g, double area_g)
{
    const double y1 = fmax(g.x, a.x), y2 = fmin(g.z, a.z), x1 = fmax(g.y, a.y), x2 = fmin(g.w, a.w);
    const double dx = __dsub_rn(x2, x1), dy = __dsub_rn(y2, y1);
    // np.maximum(v, 0) propagates NaN; fmax does not
    const double inter = __dmul_rn(dx > 0.0 ? dx : (dx != dx ? dx : 0.0), dy > 0.0 ? dy : (dy != dy ? dy : 0.0));
    const double uni = __dsub_rn(__dadd_rn(area_g, area_a), inter);
    return __ddiv_rn(inter, uni);
}

__device__ __forceinline__ double box_area_f64(const double4 b) { return __dmul_rn(__dsub_rn(b.z, b.x), __dsub_rn(b.w, b.y)); }

// "v beats best" under numpy's argmax rule: NaN is the maximum, the first one wins
__device__ __forceinline__ bool beats(double v, int iv, double best, int ib)
{
    const bool vn = v != v, bn = best != best;
    if (vn != bn) return vn;
    if (!vn && v != best) return v > best;
    return iv < ib;                                  // equal values (or both NaN): lowest index
}

__global__ void __launch_bounds__(256)
rpn_anchor_reduce_kernel(const double *__restrict__ anchors, int A, const double *__restrict__ gt, int G,
                         double *__restrict__ iou_max, int *__restrict__ argmax)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= A) return;
    const double4 a = *reinterpret_cast<const double4 *>(anchors + 4 * (size_t)i);
    const double area_a = box_area_f64(a);
    double best = 0.0;
    int arg = 0;
    for (int j = 0; j < G; ++j) {
        const double4 g = *reinterpret_cast<const double4 *>(gt + 4 * (size_t)j);
        const double v = iou_f64(a, area_a, g, box_area_f64(g));
        if (j == 0 || beats(v, j, best, arg)) { best = v; arg = j; }
    }
    if (iou_max) iou_max[i] = best;
    if (argmax) argmax[i] = arg;
}

// Column argmax in two stages: RPN_GT_SLICES CTAs per GT box each reduce a slice of the anchors to one (value, lowest
// index) pair; a second, tiny launch reduces the slices.  (One CTA per GT box walked all 261 888 anchors in fp64: 237 us.)
constexpr int RPN_GT_SLICES = 128;

__device__ __forceinline__ void reduce_pair(double &best, int &arg)
{
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, arg, o);
        if (oi != 0x7fffffff && (arg == 0x7fffffff || beats(ov, oi, best, arg))) { best = ov; arg = oi; }
    }
}

__global__ void __launch_bounds__(256)
rpn_gt_argmax_kernel(const double *__restrict__ anchors, int A, const double *__restrict__ gt, int G,
                     double *__restrict__ part_v, int *__restrict__ part_i)
{
    __shared__ double s_v[8];
    __shared__ int s_i[8];
    const int j = blockIdx.x, slice = blockIdx.y;
    const double4 g = *reinterpret_cast<const double4 *>(gt + 4 * (size_t)j);
    const double area_g = box_area_f64(g);
    const int per = (A + RPN_GT_SLICES - 1) / RPN_GT_SLICES;
    const int i0 = slice * per, i1 = min(A, i0 + per);
    double best = 0.0;
    int arg = 0x7fffffff;
    for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
        const double4 a = *reinterpret_cast<const double4 *>(anchors + 4 * (size_t)i);
        const double v = iou_f64(a, box_area_f64(a), g, area_g);
        if (arg == 0x7fffffff || beats(v, i, best, arg)) { best = v; arg = i; }
    }
    reduce_pair(best, arg);
    if ((threadIdx.x & 31) == 0) { s_v[threadIdx.x >> 5] = best; s_i[threadIdx.x >> 5] = arg; }
    __syncthreads();
    if (threadIdx.x < 32) {
        best = threadIdx.x < 8 ? s_v[threadIdx.x] : 0.0;
        arg = threadIdx.x < 8 ? s_i[threadIdx.x] : 0x7fffffff;
        reduce_pair(best, arg);
        if (threadIdx.x == 0) { part_v[(size_t)j * RPN_GT_SLICES + slice] = best; part_i[(size_t)j * RPN_GT_SLICES + slice] = arg; }
    }
}

__global__ void __launch_bounds__(RPN_GT_SLICES)
rpn_gt_argmax_final_kernel(const double *__restrict__ part_v, const int *__restrict__ part_i, int *__restrict__ gt_argmax)
{
    __shared__ double s_v[RPN_GT_SLICES / 32];
    __shared__ int s_i[RPN_GT_SLICES / 32];
    const int j = blockIdx.x;
    double best = part_v[(size_t)j * RPN_GT_SLICES + threadIdx.x];
    int arg = part_i[(size_t)j * RPN_GT_SLICES + threadIdx.x];
    reduce_pair(best, arg);
    if ((threadIdx.x & 31) == 0) { s_v[threadIdx.x >> 5] = best; s_i[threadIdx.x >> 5] = arg; }
    __syncthreads();
    if (threadIdx.x < 32) {
        best = threadIdx.x < RPN_GT_SLICES / 32 ? s_v[threadIdx.x] : 0.0;
        arg = threadIdx.x < RPN_GT_SLICES / 32 ? s_i[threadIdx.x] : 0x7fffffff;
        reduce_pair(best, arg);
        if (threadIdx.x == 0) gt_argmax[j] = arg == 0x7fffffff ? 0 : arg;
    }
}

}  // namespace sln

extern "C" size_t sln_rpn_overlap_workspace_bytes(int G)
{
    if (G <= 0) return 0;
    return sln::align_up((sizeof(double) + sizeof(int)) * (size_t)G * sln::RPN_GT_SLICES, 256) + 256;
}

extern "C" int sln_rpn_overlap_reductions(const double *anchors, int A, const double *gt_boxes, int G,
                                          double *anchor_iou_max, int *anchor_argmax, int *gt_argmax, void *workspace,
                                          size_t workspace_bytes, void *stream)
{
    SLN_REQUIRE(A >= 0 && G >= 0, SLN_ERR_ARG, "negative size");
    if (A == 0 || G == 0) return SLN_OK;
    SLN_REQUIRE(anchors && gt_boxes, SLN_ERR_ARG, "null pointer");
    SLN_REQUIRE(((reinterpret_cast<uintptr_t>(anchors) | reinterpret_cast<uintptr_t>(gt_boxes)) & 31u) == 0, SLN_ERR_LAYOUT,
                "anchors / gt_boxes must be 32-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (anchor_iou_max || anchor_argmax) {
        sln::rpn_anchor_reduce_kernel<<<sln::cdiv(A, 256), 256, 0, st>>>(anchors, A, gt_boxes, G, anchor_iou_max, anchor_argmax);
        SLN_LAUNCH_OK("rpn_anchor_reduce_kernel");
    }
    if (gt_argmax) {
        SLN_REQUIRE(workspace && workspace_bytes >= sln_rpn_overlap_workspace_bytes(G), SLN_ERR_WORKSPACE,
                    "rpn overlap workspace: need %zu bytes, got %zu", sln_rpn_overlap_workspace_bytes(G), workspace_bytes);
        double *pv = static_cast<double *>(workspace);
        int *pi = reinterpret_cast<int *>(pv + (size_t)G * sln::RPN_GT_SLICES);
        sln::rpn_gt_argmax_kernel<<<dim3(G, sln::RPN_GT_SLICES), 256, 0, st>>>(anchors, A, gt_boxes, G, pv, pi);
        sln::rpn_gt_argmax_final_kernel<<<G, sln::RPN_GT_SLICES, 0, st>>>(pv, pi, gt_argmax);
        SLN_LAUNCH_OK("rpn_gt_argmax_kernel");
    }
    return SLN_OK;
}

// ---------------------------------------------------------------------------
// tight bounding boxes of binary planes (utils.extract_bboxes, utils.py:28-47, before its random jitter)
// ---------------------------------------------------------------------------
// One CTA per plane, 16-byte loads; per plane (y1, x1, y2, x2) with x2 / y2 exclusive like the reference (:44-45), or
// zeros when the plane is empty (:49).  Meant for the planes sln_layer_decode leaves on the device, so that
// load_image_gt's boxes (Functions.py:721) need no trip of the masks through the host.
namespace sln {

__global__ void __launch_bounds__(1024)
plane_bbox_kernel(const unsigned char *__restrict__ planes, int H, int W, int *__restrict__ out)
{
    __shared__ int s_red[4][32];
    const unsigned char *p = planes + (size_t)blockIdx.x * H * W;
    int y1 = 0x7fffffff, x1 = 0x7fffffff, y2 = -1, x2 = -1;
    const bool vec = (W % 16) == 0 && ((reinterpret_cast<uintptr_t>(planes) & 15u) == 0);
    if (vec) {
        const int wv = W / 16;
        const long long n = (long long)H * wv;
        for (long long k = threadIdx.x; k < n; k += blockDim.x) {
            const uint4 v = __ldg(reinterpret_cast<const uint4 *>(p) + k);
            if ((v.x | v.y | v.z | v.w) == 0u) continue;
            const int y = (int)(k / wv), xb = (int)(k - (long long)y * wv) * 16;
            const unsigned w4[4] = {v.x, v.y, v.z, v.w};
            int first = -1, last = -1;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (w4[q]) {
                    // lowest / highest non-zero byte of the word
                    const unsigned nz = __vcmpne4(w4[q], 0u);              // 0xff per non-zero byte
                    const int lo = (__ffs(nz) - 1) >> 3, hi = (31 - __clz(nz)) >> 3;
                    if (first < 0) first = 4 * q + lo;
                    last = 4 * q + hi;
                }
            }
            y1 = min(y1, y); y2 = max(y2, y);
            x1 = min(x1, xb + first); x2 = max(x2, xb + last);
        }
    } else {
        const long long n = (long long)H * W;
        for (long long k = threadIdx.x; k < n; k += blockDim.x) {
            if (p[k]) {
                const int y = (int)(k / W), x = (int)(k - (long long)y * W);
                y1 = min(y1, y); y2 = max(y2, y); x1 = min(x1, x); x2 = max(x2, x);
            }
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        y1 = min(y1, __shfl_xor_sync(0xffffffffu, y1, o)); x1 = min(x1, __shfl_xor_sync(0xffffffffu, x1, o));
        y2 = max(y2, __shfl_xor_sync(0xffffffffu, y2, o)); x2 = max(x2, __shfl_xor_sync(0xffffffffu, x2, o));
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { s_red[0][warp] = y1; s_red[1][warp] = x1; s_red[2][warp] = y2; s_red[3][warp] = x2; }
    __syncthreads();
    if (warp == 0) {
        const int nw = blockDim.x >> 5;
        y1 = lane < nw ? s_red[0][lane] : 0x7fffffff; x1 = lane < nw ? s_red[1][lane] : 0x7fffffff;
        y2 = lane < nw ? s_red[2][lane] : -1; x2 = lane < nw ? s_red[3][lane] : -1;
        for (int o = 16; o > 0; o >>= 1) {
            y1 = min(y1, __shfl_xor_sync(0xffffffffu, y1, o)); x1 = min(x1, __shfl_xor_sync(0xffffffffu, x1, o));
            y2 = max(y2, __shfl_xor_sync(0xffffffffu, y2, o)); x2 = max(x2, __shfl_xor_sync(0xffffffffu, x2, o));
        }
        if (lane == 0) {
            int4 r = make_int4(0, 0, 0, 0);
            if (y2 >= 0) r = make_int4(y1, x1, y2 + 1, x2 + 1);
            *reinterpret_cast<int4 *>(out + 4 * (size_t)blockIdx.x) = r;
        }
    }
}

}  // namespace sln

extern "C" int sln_plane_bboxes(const uint8_t *planes, int M, int H, int W, int *boxes, void *stream)
{
    SLN_REQUIRE(M >= 0 && H >= 0 && W >= 0, SLN_ERR_ARG, "negative size");
    if (M == 0) return SLN_OK;
    SLN_REQUIRE(boxes != nullptr && (reinterpret_cast<uintptr_t>(boxes) & 15u) == 0, SLN_ERR_ARG, "boxes must be a 16-byte aligned pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if ((size_t)H * W == 0) {
        SLN_CUDA_OK(cudaMemsetAsync(boxes, 0, sizeof(int) * 4 * (size_t)M, st));
        return SLN_OK;
    }
    SLN_REQUIRE(planes != nullptr, SLN_ERR_ARG, "null planes");
    sln::plane_bbox_kernel<<<M, 1024, 0, st>>>(planes, H, W, boxes);
    SLN_LAUNCH_OK("plane_bbox_kernel");
    return SLN_OK;
}

// ---------------------------------------------------------------------------
// nearest-neighbour zoom / flip of label planes (utils.resize_layer, utils.py:358-362: scipy.ndimage.zoom(order=0);
// np.fliplr in load_image_gt, Functions.py:712-715) as one gather
// ---------------------------------------------------------------------------
// dst[p][y][x] = src[p][iy[y]][ix[x]], or 0 where iy[y] < 0 or ix[x] < 0.  The index maps are computed by the caller
// (sln_amodal_b200/targets.py: scipy's own float64 rule, including its habit of zero-filling a last line whose sample
// position overshoots the input by one rounding error; a flip is the reversed column map), so the kernel is a pure,
// exact gather.  16 output bytes per thread.
namespace sln {

__global__ void __launch_bounds__(256)
gather_planes_kernel(const unsigned char *__restrict__ src, int H, int W, const int *__restrict__ iy,
                     const int *__restrict__ ix, int H2, int W2, unsigned char *__restrict__ dst)
{
    const int xs = (blockIdx.x * blockDim.x + threadIdx.x) * 16;
    const int y = blockIdx.y;
    if (xs >= W2) return;
    const unsigned char *sp = src + (size_t)blockIdx.z * H * W;
    unsigned char *dp = dst + ((size_t)blockIdx.z * H2 + y) * W2 + xs;
    const int sy = iy[y];
    unsigned char v[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        v[k] = 0;
        if (xs + k < W2) {
            const int sx = ix[xs + k];
            if (sy >= 0 && sx >= 0) v[k] = sp[(size_t)sy * W + sx];
        }
    }
    if (xs + 16 <= W2 && ((reinterpret_cast<uintptr_t>(dp) & 15u) == 0)) {
        uint4 o;
        o.x = v[0] | (v[1] << 8) | (v[2] << 16) | ((unsigned)v[3] << 24);
        o.y = v[4] | (v[5] << 8) | (v[6] << 16) | ((unsigned)v[7] << 24);
        o.z = v[8] | (v[9] << 8) | (v[10] << 16) | ((unsigned)v[11] << 24);
        o.w = v[12] | (v[13] << 8) | (v[14] << 16) | ((unsigned)v[15] << 24);
        *reinterpret_cast<uint4 *>(dp) = o;
    } else {
        for (int k = 0; k < 16 && xs + k < W2; ++k) dp[k] = v[k];
    }
}

}  // namespace sln

extern "C" int sln_gather_planes(const uint8_t *src, int n, int H, int W, const int *iy, const int *ix, int H2, int W2,
                                 uint8_t *dst, void *stream)
{
    SLN_REQUIRE(n >= 0 && H >= 0 && W >= 0 && H2 >= 0 && W2 >= 0, SLN_ERR_ARG, "negative size");
    if ((size_t)n * H2 * W2 == 0) return SLN_OK;
    SLN_REQUIRE(src && iy && ix && dst, SLN_ERR_ARG, "null pointer");
    SLN_REQUIRE(H2 <= 65535 && n <= 65535, SLN_ERR_ARG, "output height / plane count above 65535");
    dim3 grid(sln::cdiv(sln::cdiv(W2, 16), 256), H2, n);
    sln::gather_planes_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(src, H, W, iy, ix, H2, W2, dst);
    SLN_LAUNCH_OK("gather_planes_kernel");
    return SLN_OK;
}
