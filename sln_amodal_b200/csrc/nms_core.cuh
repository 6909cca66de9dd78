// nms_core.cuh -- internal interface shared by nms.cu (the sln_nms entry point) and
// proposal.cu (which feeds already-sorted boxes straight into the mask + scan stages).
#pragma once

#include "common.cuh"

namespace sln {

// Workspace carved up for one NMS problem of n boxes.
struct NmsBuffers {
    float4 *boxes;                 // [n] (c0,c1,c2,c3) in visiting (score) order
    float *areas;                  // [n] (c3-c1+1)*(c2-c0+1), pth_nms.py:16
    int *cls;                      // [n] class id in visiting order (only if class-aware)
    int *order;                    // [n] original index of the box at each visiting position
    int *rank;                     // [n] visiting position of each original box
    int *tickets;                  // [ceil(n/256)] row-tile tickets of the rank kernel's fused gather
    unsigned long long *mask;      // [n][W] IoU>=thresh bitmask, W = ceil(n/64)
    void *stage;                   // scratch of the two-stage pipeline (see nms.cu)
    void *fix;                     // scratch of the parallel fixed-point resolve
    void *sparse;                  // scratch of the sparse (binned) path
};

size_t nms_buffers_bytes(int n);
void nms_carve(void *ws, int n, NmsBuffers &b);

// Mask + greedy scan over boxes that are ALREADY in visiting order.
//   order == nullptr : kept entries are visiting positions themselves
//   keep64 / keep32  : either may be nullptr
int nms_sorted_launch(const float4 *boxes, const float *areas, const int *cls, const int *order, int n,
                      float thresh, int max_keep, unsigned long long *mask, int64_t *keep64, int *keep32,
                      int *num_keep, cudaStream_t st, void *stage, void *fix, void *sparse, bool sparse_only = false);

// Batched calls (sln_proposal_layer_batched) lay out B copies of the single-image workspace, stride_bytes apart: the
// array of image `seg` is the image-0 pointer moved by seg * stride_bytes.
template <typename T>
__host__ __device__ __forceinline__ T *seg_at(T *p, size_t stride_bytes, int seg)
{
    return (T *)((const unsigned char *)p + stride_bytes * (size_t)seg);
}

// B independent problems of n boxes each: boxes, areas, cls, order, mask, stage, fix and sparse are those of problem 0,
// problem b's are seg_at(.., stride_bytes, b); the outputs move by their own strides (keep64 / keep32 by keep_stride,
// num_keep by num_stride, in bytes).  cls, order, keep64 and keep32 may be nullptr.  One launch per sparse stage for all
// B (a cluster per problem); the dense kernels run per problem and leave at once where that problem's sparse pass
// succeeded.  Each problem's keep list is exactly nms_sorted_launch's.
int nms_sorted_batched_launch(int B, size_t stride_bytes, const float4 *boxes, const float *areas, const int *cls,
                              const int *order, int n, float thresh, int max_keep, unsigned long long *mask,
                              int64_t *keep64, int *keep32, size_t keep_stride, int *num_keep, size_t num_stride,
                              cudaStream_t st, void *stage, void *fix, void *sparse);

// Total order used everywhere a "descending score, stable" sort is needed:
// larger key first; NaN sorts as the largest value (torch.sort's convention);
// -0.0 == +0.0.  Ties are broken by ascending index.
__device__ __forceinline__ unsigned score_key(float s)
{
    unsigned u = __float_as_uint(s);
    if (s != s) return 0xffffffffu;
    if (u == 0x80000000u) u = 0u;
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// rank[i] = number of elements that precede element i in (score desc, tie id asc) order,
// score of element i = scores[i*stride], tie id = tie_ids[i] (or i when tie_ids is null;
// tie ids must be distinct).  rank must be zero-filled before the launch.
// O(n^2) compares spread over the whole grid: a stable, deterministic sort for the
// n <= ~16k this path sees, with no multi-pass radix machinery.
int rank_sort_launch(const float *scores, int stride, const int *tie_ids, int n, int *rank, cudaStream_t st);
// B segments of n elements each, segment z = blockIdx.z: scores / tie_ids / rank of segment z are seg_at(.., stride_bytes, z)
int rank_sort_batched_launch(const float *scores, const int *tie_ids, int n, int B, size_t stride_bytes, int *rank,
                             cudaStream_t st);

}  // namespace sln
