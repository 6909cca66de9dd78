// eval_tail.cuh -- what unmold.cu and rle.cu share for the batched evaluation tail (sln_unmold_rle_batched): the
// per-detection record the box prep writes, the launchers of rle.cu's kernels, and a block-wide prefix sum.
#pragma once

namespace sln {

// Exclusive prefix sum of v over the THREADS threads of the block (every thread must call it).  `warp_tot` is
// THREADS / 32 elements of shared memory; *total receives the block's sum.  Ends with a __syncthreads, so the
// shared array can be reused by the next call.
template <int THREADS, typename T>
__device__ __forceinline__ T block_excl_sum(T v, T *warp_tot, T *total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    T incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T u = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += u;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    T before = 0, sum = 0;
#pragma unroll
    for (int w = 0; w < THREADS / 32; ++w) {
        if (w < warp) before += warp_tot[w];
        sum += warp_tot[w];
    }
    *total = sum;
    __syncthreads();
    return before + incl - v;
}

// One kept detection, written by the box prep for the box-local paste and the run-length kernel.  bh / bw are the box's
// height and width, 0 / 0 for a kept box whose mask is empty (see unmold.cu); off is the byte offset of its
// column-major bh x bw mask in the mask buffer.
struct BoxRow {
    long long off;
    int y1, x1, bh, bw, H, W, src, ch;
};

// rle.cu: launch the run-length kernel over rows[B*D] (row b*D + k is live when k < nk[b]) and the string coder's scan
// and write kernels.  Return SLN_OK or an SLN_ERR_* code.
int launch_rle_boxes(const BoxRow *rows, const int *nk, int B, int D, const uint8_t *maskbuf, uint32_t *counts, int cap,
                     int *m_out, int *str_len, cudaStream_t st);
int launch_rle_strings(const uint32_t *counts, int n, int cap, const int *m, const int *str_len, int *str_off,
                       int *str_total, char *strings, cudaStream_t st);

}  // namespace sln
