// unmold.cu -- utils.unmold_mask (utils.py:447-465) for all detections of an image in one launch
// (SURVEY.md section 8(f), row 3: the step after the path, feeding the COCO run-length encoder of rle.cu).
//
// The reference resizes each small float mask to its detection box with scipy.misc.imresize(interp='bilinear')
// and thresholds at 0.5.  imresize is scipy's bytescale (min/max stretch to u8 in float32) followed by Pillow's
// 8-bit resampler (libImaging/Resample.c): triangle filter of support max(1, in/out), coefficients normalised in
// double and rounded to 22-bit fixed point, a horizontal pass whose result is clipped to 8 bits, then a vertical
// pass.  Every step is reproduced operation by operation (un-contracted double arithmetic for the coefficients,
// integer accumulation) so that the pasted mask is bit-identical; oracle/oracle.py restates the same steps and is
// pinned against Pillow itself.
//
// grid = (row slabs of 64 image rows, detections).  A CTA whose slab misses the box streams zeros; otherwise it
// rebuilds the u8 mask, computes the vertical coefficients of its own rows and the horizontal coefficients of the
// box columns, runs the horizontal pass only for the mask rows its vertical taps reach, and writes its slab once:
// 16 pixels per thread from one 16-byte shared-memory read per tap (the intermediate is stored at column offset
// x1 & 15, so image-aligned 16-pixel units are aligned in shared memory too).
//
// The batched evaluation tail (sln_unmold_rle_batched) runs the same resample into box-sized masks instead: a box prep
// kernel for all B images (padding cut, class collapse, float64 box arithmetic, keep rule, compaction, mask offsets) and
// a box-local paste that writes only each box's bh x bw binary mask, column-major, for rle.cu's run-length kernel.
#include <math.h>

#include "common.cuh"
#include "eval_tail.cuh"

namespace sln {

constexpr int UNMOLD_SLAB = 64;
constexpr int UNMOLD_THREADS = 256;
constexpr int PIL_BITS = 32 - 8 - 2;

struct UnmoldSmem {
    size_t f_off, src_off, hx_off, hk_off, tmp_off, vy_off, vk_off, total;
    int TS;
};

__host__ __device__ inline int imax_(int a, int b) { return a > b ? a : b; }

__host__ __device__ inline UnmoldSmem unmold_smem(int mh, int mw, int W)
{
    UnmoldSmem s;
    size_t o = 0;
    s.f_off = o;   o += (size_t)(((size_t)mh * mw * 4 + 15) / 16 * 16);
    s.src_off = o; o += (size_t)(((size_t)mh * mw + 15) / 16 * 16);
    s.hx_off = o;  o += (size_t)W * 4;
    s.hk_off = o;  o += (size_t)imax_(3 * W, mw * mw) * 4;
    o = (o + 15) / 16 * 16;
    s.TS = (W + 15) / 16 * 16 + 32;
    s.tmp_off = o; o += (size_t)mh * s.TS;
    s.vy_off = o;  o += (size_t)UNMOLD_SLAB * 4;
    s.vk_off = o;  o += (size_t)imax_(3 * UNMOLD_SLAB, mh * mh) * 4;
    s.total = o;
    return s;
}

// Resample.c precompute_coeffs + normalize_coeffs_8bpc for output sample xx of an axis resized in_size -> out_size
// with the triangle filter.  Writes <= tcap coefficients, returns xmin | count << 16.
__device__ __forceinline__ int pil_axis(int in_size, int out_size, int xx, int *k_out)
{
    const double scale = __ddiv_rn((double)in_size, (double)out_size);
    const double fs = scale < 1.0 ? 1.0 : scale;          // filterscale; support = 1.0 * filterscale
    const double ss = __ddiv_rn(1.0, fs);
    const double center = __dmul_rn((double)xx + 0.5, scale);
    int xmin = __double2int_rz(__dadd_rn(__dsub_rn(center, fs), 0.5));
    if (xmin < 0) xmin = 0;
    int xmax = __double2int_rz(__dadd_rn(__dadd_rn(center, fs), 0.5));
    if (xmax > in_size) xmax = in_size;
    const int cnt = xmax - xmin;
    double ww = 0.0;
    for (int x = 0; x < cnt; ++x) {
        double v = fabs(__dmul_rn(__dadd_rn(__dsub_rn((double)(x + xmin), center), 0.5), ss));
        ww = __dadd_rn(ww, v < 1.0 ? __dsub_rn(1.0, v) : 0.0);
    }
    for (int x = 0; x < cnt; ++x) {
        double v = fabs(__dmul_rn(__dadd_rn(__dsub_rn((double)(x + xmin), center), 0.5), ss));
        double w = v < 1.0 ? __dsub_rn(1.0, v) : 0.0;
        if (ww != 0.0) w = __ddiv_rn(w, ww);
        k_out[x] = __double2int_rz(__dadd_rn(0.5, __dmul_rn(w, (double)(1 << PIL_BITS))));
    }
    return xmin | (cnt << 16);
}

// ksize of Resample.c capped by the axis length: the stride of one output sample's coefficient row
__device__ __forceinline__ int pil_taps(int in_size, int out_size)
{
    const double scale = __ddiv_rn((double)in_size, (double)out_size);
    const double fs = scale < 1.0 ? 1.0 : scale;
    const int ksize = __double2int_rz(ceil(fs)) * 2 + 1;
    return ksize < in_size ? ksize : in_size;
}

// unmold_kernel's bytescale and horizontal pass as device functions, for the box-local paste below (unmold_kernel keeps
// its own inline copy: calling these from it reschedules its address arithmetic, and its benchmark figure moved by ~4 %).
// scipy.misc.bytescale of one [mh, mw] mask into src: min / max stretch in float32 (numpy-1.x scalar promotion), then
// round half up into u8.  load(i) returns element i in row-major order.  `between` runs after the per-warp min / max
// and before the barrier that publishes them (the callers compute their coefficient tables there).  Ends with a
// barrier: src is complete on return.
template <typename Load, typename Between>
__device__ __forceinline__ void bytescale_u8(Load load, int msz, float *fsrc, uint8_t *src, float *red_min, float *red_max,
                                             int tid, Between between)
{
    float lo = INFINITY, hi = -INFINITY;
    for (int i = tid; i < msz; i += UNMOLD_THREADS) {
        const float v = load(i);
        fsrc[i] = v;
        lo = fminf(lo, v);
        hi = fmaxf(hi, v);
    }
    for (int o = 16; o; o >>= 1) {
        lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if ((tid & 31) == 0) { red_min[tid >> 5] = lo; red_max[tid >> 5] = hi; }
    between();
    __syncthreads();
    for (int w = 0; w < UNMOLD_THREADS / 32; ++w) { lo = fminf(lo, red_min[w]); hi = fmaxf(hi, red_max[w]); }
    float cscale = __fsub_rn(hi, lo);
    if (cscale == 0.f) cscale = 1.f;
    const float scale = (float)(255.0 / (double)cscale);
    for (int i = tid; i < msz; i += UNMOLD_THREADS) {
        float b = __fmul_rn(__fsub_rn(fsrc[i], lo), scale);
        b = fminf(fmaxf(b, 0.f), 255.f);
        src[i] = (uint8_t)__float2int_rz(__fadd_rn(b, 0.5f));
    }
    __syncthreads();
}

// Pillow's horizontal pass for mask rows [r_lo, r_hi) and output columns [0, bw): tmp[r * TS + xoff + xx] =
// clip8((2^21 + sum_t src[r][xmin + t] * k[t]) >> 22)
__device__ __forceinline__ void pil_hpass(const uint8_t *src, int mw, const int *hx, const int *hk, int tH, int r_lo,
                                          int r_hi, int bw, uint8_t *tmp, int TS, int xoff, int tid)
{
    for (int idx = tid; idx < (r_hi - r_lo) * bw; idx += UNMOLD_THREADS) {
        const int r = r_lo + idx / bw, xx = idx - (idx / bw) * bw;
        const int pk = hx[xx], xmin = pk & 0xffff, cnt = pk >> 16;
        const int *k = hk + xx * tH;
        const uint8_t *s = src + r * mw + xmin;
        int acc = 1 << (PIL_BITS - 1);
        for (int t = 0; t < cnt; ++t) acc += (int)s[t] * k[t];
        acc >>= PIL_BITS;
        tmp[r * TS + xoff + xx] = (uint8_t)min(max(acc, 0), 255);
    }
}

template <bool VEC>
__device__ __forceinline__ void zero_rows(uint8_t *dst, long long count, int tid)
{
    if (VEC) {
        uint4 *d = reinterpret_cast<uint4 *>(dst);
        const uint4 z = make_uint4(0, 0, 0, 0);
        for (long long i = tid; i < count / 16; i += UNMOLD_THREADS) d[i] = z;
    } else {
        for (long long i = tid; i < count; i += UNMOLD_THREADS) dst[i] = 0;
    }
}

template <bool VEC>
__global__ void __launch_bounds__(UNMOLD_THREADS)
unmold_kernel(const float *__restrict__ masks, int mh, int mw, const int *__restrict__ boxes, int H, int W,
              uint8_t *__restrict__ out)
{
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ float red_min[UNMOLD_THREADS / 32], red_max[UNMOLD_THREADS / 32];
    const int n = blockIdx.y, tid = threadIdx.x;
    const int y0 = blockIdx.x * UNMOLD_SLAB, y_end = min(H, y0 + UNMOLD_SLAB);
    const int by1 = boxes[4 * n + 0], bx1 = boxes[4 * n + 1], by2 = boxes[4 * n + 2], bx2 = boxes[4 * n + 3];
    const int bh = by2 - by1, bw = bx2 - bx1;
    uint8_t *dst = out + ((size_t)n * H + y0) * (size_t)W;
    const int ra = max(y0, by1), rb = min(y_end, by2);         // image rows of this slab inside the box
    const bool inside = bh > 0 && bw > 0 && by1 >= 0 && bx1 >= 0 && by2 <= H && bx2 <= W;
    if (!inside || ra >= rb) {
        zero_rows<VEC>(dst, (long long)(y_end - y0) * W, tid);
        return;
    }
    const UnmoldSmem L = unmold_smem(mh, mw, W);
    float *fsrc = reinterpret_cast<float *>(smem + L.f_off);
    uint8_t *src = smem + L.src_off;
    int *hx = reinterpret_cast<int *>(smem + L.hx_off);
    int *hk = reinterpret_cast<int *>(smem + L.hk_off);
    uint8_t *tmp = smem + L.tmp_off;
    int *vy = reinterpret_cast<int *>(smem + L.vy_off);
    int *vk = reinterpret_cast<int *>(smem + L.vk_off);
    const int TS = L.TS;

    // ---- bytescale: min / max stretch in float32 (scipy.misc.bytescale under numpy-1.x scalar promotion)
    const int msz = mh * mw;
    const float *m = masks + (size_t)n * msz;
    float lo = INFINITY, hi = -INFINITY;
    for (int i = tid; i < msz; i += UNMOLD_THREADS) {
        const float v = __ldg(m + i);
        fsrc[i] = v;
        lo = fminf(lo, v);
        hi = fmaxf(hi, v);
    }
    for (int o = 16; o; o >>= 1) {
        lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if ((tid & 31) == 0) { red_min[tid >> 5] = lo; red_max[tid >> 5] = hi; }

    // ---- coefficients: horizontal for every box column, vertical for this slab's rows
    const int tH = pil_taps(mw, bw), tV = pil_taps(mh, bh);
    for (int xx = tid; xx < bw; xx += UNMOLD_THREADS) hx[xx] = pil_axis(mw, bw, xx, hk + xx * tH);
    for (int i = tid; i < rb - ra; i += UNMOLD_THREADS) vy[i] = pil_axis(mh, bh, ra - by1 + i, vk + i * tV);
    __syncthreads();
    for (int w = 0; w < UNMOLD_THREADS / 32; ++w) { lo = fminf(lo, red_min[w]); hi = fmaxf(hi, red_max[w]); }
    float cscale = __fsub_rn(hi, lo);
    if (cscale == 0.f) cscale = 1.f;
    const float scale = (float)(255.0 / (double)cscale);
    for (int i = tid; i < msz; i += UNMOLD_THREADS) {
        float b = __fmul_rn(__fsub_rn(fsrc[i], lo), scale);
        b = fminf(fmaxf(b, 0.f), 255.f);
        src[i] = (uint8_t)__float2int_rz(__fadd_rn(b, 0.5f));
    }
    __syncthreads();

    // ---- horizontal pass, only the mask rows the vertical taps of this slab reach (xmin and xmin + count are
    // monotone along an axis); the 8-bit result sits at column offset x1 & 15
    const int r_lo = vy[0] & 0xffff;
    const int v_last = vy[rb - ra - 1];
    const int r_hi = (v_last & 0xffff) + (v_last >> 16);
    const int xoff = bx1 & 15;
    for (int idx = tid; idx < (r_hi - r_lo) * bw; idx += UNMOLD_THREADS) {
        const int r = r_lo + idx / bw, xx = idx - (idx / bw) * bw;
        const int pk = hx[xx], xmin = pk & 0xffff, cnt = pk >> 16;
        const int *k = hk + xx * tH;
        const uint8_t *s = src + r * mw + xmin;
        int acc = 1 << (PIL_BITS - 1);
        for (int t = 0; t < cnt; ++t) acc += (int)s[t] * k[t];
        acc >>= PIL_BITS;
        tmp[r * TS + xoff + xx] = (uint8_t)min(max(acc, 0), 255);
    }
    __syncthreads();

    // ---- vertical pass + threshold (v / 255 >= 0.5  <=>  v >= 128) + paste, the slab written exactly once
    const int rows = y_end - y0;
    if (VEC) {
        const int UW = W >> 4, ubase = bx1 >> 4;
        uint4 *d4 = reinterpret_cast<uint4 *>(dst);
        for (int idx = tid; idx < rows * UW; idx += UNMOLD_THREADS) {
            const int yr = idx / UW, u = idx - yr * UW, y = y0 + yr;
            uint4 o = make_uint4(0, 0, 0, 0);
            if (y >= ra && y < rb && 16 * u + 16 > bx1 && 16 * u < bx2) {
                const int i = y - ra, pk = vy[i], ymin = pk & 0xffff, cnt = pk >> 16;
                const int *k = vk + i * tV;
                int acc[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) acc[j] = 1 << (PIL_BITS - 1);
                const uint8_t *t0 = tmp + ymin * TS + 16 * (u - ubase);
                for (int t = 0; t < cnt; ++t) {
                    const uint4 w = *reinterpret_cast<const uint4 *>(t0 + t * TS);
                    const int kt = k[t];
                    const unsigned ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                    for (int j = 0; j < 16; ++j) acc[j] += (int)((ww[j >> 2] >> (8 * (j & 3))) & 0xffu) * kt;
                }
                unsigned r[4] = {0, 0, 0, 0};
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const int x = 16 * u + j;
                    if (x >= bx1 && x < bx2 && (acc[j] >> PIL_BITS) >= 128) r[j >> 2] |= 1u << (8 * (j & 3));
                }
                o = make_uint4(r[0], r[1], r[2], r[3]);
            }
            d4[idx] = o;
        }
    } else {
        for (int idx = tid; idx < rows * W; idx += UNMOLD_THREADS) {
            const int yr = idx / W, x = idx - yr * W, y = y0 + yr;
            uint8_t o = 0;
            if (y >= ra && y < rb && x >= bx1 && x < bx2) {
                const int i = y - ra, pk = vy[i], ymin = pk & 0xffff, cnt = pk >> 16;
                const int *k = vk + i * tV;
                int acc = 1 << (PIL_BITS - 1);
                const uint8_t *t0 = tmp + ymin * TS + xoff + (x - bx1);
                for (int t = 0; t < cnt; ++t) acc += (int)t0[t * TS] * k[t];
                o = (acc >> PIL_BITS) >= 128 ? 1 : 0;
            }
            dst[idx] = o;
        }
    }
}

// ---------------------------------------------------------------------------
// utils.resize_image (utils.py:301-356): scipy.misc.imresize(image, (max_dim, max_dim)) of the uint8 RGB image =
// Pillow's 8-bit bilinear resample per band (no bytescale for uint8 input).  Same coefficient code as above:
// a table launch, a horizontal pass into an 8-bit intermediate [h, W2, C], a vertical pass.
// ---------------------------------------------------------------------------
struct ResizeTabs {
    int *hx, *hk, *vy, *vk;      // xmin | count << 16 and coefficient rows of the two axes
    int tH, tV;
};

__global__ void __launch_bounds__(256)
resize_coeffs_kernel(int h, int w, int H2, int W2, ResizeTabs t)
{
    pdl_prologue();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < W2) t.hx[i] = pil_axis(w, W2, i, t.hk + (size_t)i * t.tH);
    else if (i < W2 + H2) t.vy[i - W2] = pil_axis(h, H2, i - W2, t.vk + (size_t)(i - W2) * t.tV);
}

// tmp[r][xx][c] = clip8((2^21 + sum_t src[r][xmin+t][c] * k[t]) >> 22)
__global__ void __launch_bounds__(256)
resize_h_kernel(const uint8_t *__restrict__ src, int h, int w, int C, int W2, ResizeTabs t, uint8_t *__restrict__ tmp)
{
    pdl_prologue();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)h * W2) return;
    const int r = (int)(i / W2), xx = (int)(i - (long long)r * W2);
    const int pk = t.hx[xx], xmin = pk & 0xffff, cnt = pk >> 16;
    const int *k = t.hk + (size_t)xx * t.tH;
    const uint8_t *s = src + ((size_t)r * w + xmin) * C;
    uint8_t *d = tmp + ((size_t)r * W2 + xx) * C;
    if (C <= 4) {                                   // grey / RGB / RGBA: one pass over the taps for all bands
        int acc[4] = {1 << (PIL_BITS - 1), 1 << (PIL_BITS - 1), 1 << (PIL_BITS - 1), 1 << (PIL_BITS - 1)};
        for (int q = 0; q < cnt; ++q) {
            const int kq = __ldg(k + q);
#pragma unroll
            for (int c = 0; c < 4; ++c)
                if (c < C) acc[c] += (int)s[(size_t)q * C + c] * kq;
        }
#pragma unroll
        for (int c = 0; c < 4; ++c)
            if (c < C) d[c] = (uint8_t)min(max(acc[c] >> PIL_BITS, 0), 255);
        return;
    }
    for (int c = 0; c < C; ++c) {
        int acc = 1 << (PIL_BITS - 1);
        for (int q = 0; q < cnt; ++q) acc += (int)s[(size_t)q * C + c] * __ldg(k + q);
        acc >>= PIL_BITS;
        d[c] = (uint8_t)min(max(acc, 0), 255);
    }
}

// VEC4: four output bytes per thread (the row length in bytes is a multiple of 4: one 32-bit load per tap)
template <bool VEC4>
__global__ void __launch_bounds__(256)
resize_v_kernel(const uint8_t *__restrict__ tmp, int C, int H2, int W2, ResizeTabs t, uint8_t *__restrict__ out)
{
    pdl_prologue();
    constexpr int V = VEC4 ? 4 : 1;
    const long long rowb = (long long)W2 * C, rowu = rowb / V;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;     // one thread per V output bytes (x, c fastest)
    if (i >= (long long)H2 * rowu) return;
    const int yy = (int)(i / rowu);
    const long long xc = (i - (long long)yy * rowu) * V;
    const int pk = t.vy[yy], ymin = pk & 0xffff, cnt = pk >> 16;
    const int *k = t.vk + (size_t)yy * t.tV;
    if (VEC4) {
        int acc[4] = {1 << (PIL_BITS - 1), 1 << (PIL_BITS - 1), 1 << (PIL_BITS - 1), 1 << (PIL_BITS - 1)};
        for (int q = 0; q < cnt; ++q) {
            const unsigned w = *reinterpret_cast<const unsigned *>(tmp + (size_t)(ymin + q) * rowb + xc);
            const int kq = __ldg(k + q);
#pragma unroll
            for (int b = 0; b < 4; ++b) acc[b] += (int)((w >> (8 * b)) & 0xffu) * kq;
        }
        unsigned r = 0u;
#pragma unroll
        for (int b = 0; b < 4; ++b) r |= (unsigned)min(max(acc[b] >> PIL_BITS, 0), 255) << (8 * b);
        *reinterpret_cast<unsigned *>(out + (size_t)yy * rowb + xc) = r;
    } else {
        int acc = 1 << (PIL_BITS - 1);
        for (int q = 0; q < cnt; ++q) acc += (int)tmp[(size_t)(ymin + q) * rowb + xc] * __ldg(k + q);
        acc >>= PIL_BITS;
        out[(size_t)yy * rowb + xc] = (uint8_t)min(max(acc, 0), 255);
    }
}

static int resize_taps_host(int in_size, int out_size)
{
    const double scale = (double)in_size / (double)out_size;
    const double fs = scale < 1.0 ? 1.0 : scale;
    const int ksize = (int)ceil(fs) * 2 + 1;
    return ksize < in_size ? ksize : in_size;
}

static size_t resize_ws_layout(int h, int w, int C, int H2, int W2, size_t off[5])
{
    const int tH = resize_taps_host(w, W2), tV = resize_taps_host(h, H2);
    size_t o = 0;
    off[0] = o; o += align_up(sizeof(int) * (size_t)W2, 256);
    off[1] = o; o += align_up(sizeof(int) * (size_t)W2 * tH, 256);
    off[2] = o; o += align_up(sizeof(int) * (size_t)H2, 256);
    off[3] = o; o += align_up(sizeof(int) * (size_t)H2 * tV, 256);
    off[4] = o; o += align_up((size_t)h * W2 * C, 256);
    return o;
}

// ---------------------------------------------------------------------------
// Batched evaluation tail (sln_unmold_rle_batched): MaskRCNN.unmold_detections (model.py:747-806) for B images, ending
// in box-sized masks instead of H x W planes.  Two kernels here, then rle.cu's run-length kernel and string coder.
// ---------------------------------------------------------------------------
struct UnmoldImg {
    double sy, sx, shy, shx;     // h_scale, w_scale, window[0], window[1] as the reference computes them (float64)
    int H, W;
};
template <int NB> struct UnmoldImgs { UnmoldImg v[NB]; };   // by value: no host-to-device copy, graph capturable

constexpr int PREP_THREADS = 256;

// numpy's astype(int32) of a float64 (or a float32, exactly widened) as it behaves on x86-64: truncation toward zero,
// and INT_MIN (the "integer indefinite" of cvttsd2si) for NaN and values outside the int32 range.  __double2int_rz
// alone would saturate.  Such a coordinate drops the box under the keep rule below except as x2, where int32
// wrap-around can keep it; then both paths agree on boxes / class ids / scores, and the mask is empty here (the
// single-image paste is undefined for that box).
__device__ __forceinline__ int np_cast_i32(double v)
{
    return (v > -2147483649.0 && v < 2147483648.0) ? __double2int_rz(v) : (int)0x80000000;
}

// One CTA per image: (1) the padding cut, n = first row whose class is 0; (2) class collapse to 1 and the mask channel
// (numpy's negative indices wrap; a channel outside the mask makes the reference raise, reported as num_kept = -1);
// (3) astype(int32) of (box - shift) * scale, each operation rounded in float64; (4) the keep rule of
// unmold.unmold_detections, evaluated in int32 arithmetic with numpy's wrap-around, and compaction in order, with each
// kept mask's offset in the buffer (prefix sum of box areas from the image's base).  Rows at and beyond the count are
// zero in the outputs.
template <int NB>
__global__ void __launch_bounds__(PREP_THREADS)
unmold_box_prep_kernel(const float *__restrict__ det, int D, int K, UnmoldImgs<NB> P, int *__restrict__ boxes,
                       int *__restrict__ cls_out, float *__restrict__ scores, int *__restrict__ src_out,
                       int *__restrict__ num_kept, BoxRow *__restrict__ rows, int *__restrict__ nk)
{
    __shared__ int s_n, s_bad;
    __shared__ int s_wi[PREP_THREADS / 32];
    __shared__ long long s_wl[PREP_THREADS / 32];
    const int b = blockIdx.x, tid = threadIdx.x;
    const UnmoldImg I = P.v[b];
    const float *d0 = det + (size_t)b * D * 6;
    if (tid == 0) { s_n = D; s_bad = 0; }
    __syncthreads();
    for (int d = tid; d < D; d += PREP_THREADS)
        if (d0[6 * d + 4] == 0.f) atomicMin(&s_n, d);
    __syncthreads();
    const int n = s_n;
    for (int d = tid; d < n; d += PREP_THREADS) {
        int c = np_cast_i32((double)d0[6 * d + 4]);
        if (c > 0) c = 1;
        const long long ch = c < 0 ? (long long)c + K : c;
        if (ch < 0 || ch >= K) s_bad = 1;
    }
    long long base = 0;                                        // the image's slice of the mask buffer
    for (int q = 0; q < b; ++q) base += (long long)D * P.v[q].H * P.v[q].W;
    __syncthreads();
    const bool bad = s_bad != 0;
    int kept = 0;
    long long used = 0;
    for (int c0 = 0; c0 < (bad ? 0 : n); c0 += PREP_THREADS) {
        const int d = c0 + tid;
        int y1 = 0, x1 = 0, y2 = 0, x2 = 0, c = 0;
        bool keep = false;
        long long area = 0;
        if (d < n) {
            const float *r = d0 + 6 * d;
            y1 = np_cast_i32(__dmul_rn(__dsub_rn((double)r[0], I.shy), I.sy));
            x1 = np_cast_i32(__dmul_rn(__dsub_rn((double)r[1], I.shx), I.sx));
            y2 = np_cast_i32(__dmul_rn(__dsub_rn((double)r[2], I.shy), I.sy));
            x2 = np_cast_i32(__dmul_rn(__dsub_rn((double)r[3], I.shx), I.sx));
            const int a32 = (int)(((unsigned)y2 - (unsigned)y1) * ((unsigned)x2 - (unsigned)x1));   // numpy int32 wraps
            keep = a32 > 0 && y2 > y1 && y1 >= 0 && x1 >= 0 && y2 <= I.H && x2 <= I.W;
            if (keep && (long long)x2 - x1 > 0) area = (long long)(y2 - y1) * (x2 - x1);
            c = np_cast_i32((double)r[4]);
            if (c > 0) c = 1;
        }
        int cnt;
        long long area_sum;
        const int k = kept + block_excl_sum<PREP_THREADS>(keep ? 1 : 0, s_wi, &cnt);
        const long long off = used + block_excl_sum<PREP_THREADS>(area, s_wl, &area_sum);
        if (keep) {
            const size_t o = (size_t)b * D + k;
            boxes[4 * o + 0] = y1; boxes[4 * o + 1] = x1; boxes[4 * o + 2] = y2; boxes[4 * o + 3] = x2;
            cls_out[o] = c;
            scores[o] = d0[6 * d + 5];
            src_out[o] = d;
            BoxRow R;
            R.off = base + off;
            R.y1 = y1; R.x1 = x1;
            R.bh = area ? y2 - y1 : 0;
            R.bw = area ? x2 - x1 : 0;
            R.H = I.H; R.W = I.W;
            R.src = d;
            R.ch = c < 0 ? c + K : c;
            rows[o] = R;
        }
        kept += cnt;
        used += area_sum;
    }
    for (int k = kept + tid; k < D; k += PREP_THREADS) {
        const size_t o = (size_t)b * D + k;
        boxes[4 * o + 0] = 0; boxes[4 * o + 1] = 0; boxes[4 * o + 2] = 0; boxes[4 * o + 3] = 0;
        cls_out[o] = 0;
        scores[o] = 0.f;
        src_out[o] = 0;
    }
    if (tid == 0) {
        nk[b] = kept;
        num_kept[b] = bad ? -1 : kept;
    }
}

// Box-local paste: unmold_kernel's bytescale, coefficients, horizontal and vertical passes in the same operation order
// (bit-identical pixels), written as the bh x bw binary mask in column-major order (pycocotools' run order) and
// nothing else.  grid = (B*D rows, slabs of 64 box rows); a slab past the box's height and a row past the image's
// count return at once.  The mask element (y, x) of detection row src, channel ch of image b is read through strides.
__global__ void __launch_bounds__(UNMOLD_THREADS)
unmold_box_kernel(const float *__restrict__ mrcnn_mask, long long s0, long long s1, long long s2, long long s3,
                  long long s4, int mh, int mw, int Wmax, int D, const BoxRow *__restrict__ rows,
                  const int *__restrict__ nk, uint8_t *__restrict__ maskbuf)
{
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ float red_min[UNMOLD_THREADS / 32], red_max[UNMOLD_THREADS / 32];
    const int row = blockIdx.x, tid = threadIdx.x;
    const int b = row / D;
    if (row - b * D >= nk[b]) return;
    const BoxRow R = rows[row];
    const int bh = R.bh, bw = R.bw;
    const int ra = blockIdx.y * UNMOLD_SLAB;                   // box rows [ra, rb) of this slab
    if (ra >= bh) return;
    const int rb = min(bh, ra + UNMOLD_SLAB);
    const UnmoldSmem L = unmold_smem(mh, mw, Wmax);
    float *fsrc = reinterpret_cast<float *>(smem + L.f_off);
    uint8_t *src = smem + L.src_off;
    int *hx = reinterpret_cast<int *>(smem + L.hx_off);
    int *hk = reinterpret_cast<int *>(smem + L.hk_off);
    uint8_t *tmp = smem + L.tmp_off;
    int *vy = reinterpret_cast<int *>(smem + L.vy_off);
    int *vk = reinterpret_cast<int *>(smem + L.vk_off);
    const int TS = L.TS;

    const float *m = mrcnn_mask + b * s0 + R.src * s1 + R.ch * s4;
    const int tH = pil_taps(mw, bw), tV = pil_taps(mh, bh);
    bytescale_u8([&](int i) { const int y = i / mw; return __ldg(m + y * s2 + (i - y * mw) * s3); }, mh * mw, fsrc, src,
                 red_min, red_max, tid, [&] {
        for (int xx = tid; xx < bw; xx += UNMOLD_THREADS) hx[xx] = pil_axis(mw, bw, xx, hk + xx * tH);
        for (int i = tid; i < rb - ra; i += UNMOLD_THREADS) vy[i] = pil_axis(mh, bh, ra + i, vk + i * tV);
    });
    const int r_lo = vy[0] & 0xffff;
    const int v_last = vy[rb - ra - 1];
    pil_hpass(src, mw, hx, hk, tH, r_lo, (v_last & 0xffff) + (v_last >> 16), bw, tmp, TS, 0, tid);
    __syncthreads();

    // vertical pass + threshold (v >= 128), box row fastest: consecutive threads write consecutive bytes of a column
    const int nr = rb - ra;
    uint8_t *dst = maskbuf + R.off;
    for (int idx = tid; idx < nr * bw; idx += UNMOLD_THREADS) {
        const int xx = idx / nr, i = idx - xx * nr;
        const int pk = vy[i], ymin = pk & 0xffff, cnt = pk >> 16;
        const int *k = vk + i * tV;
        int acc = 1 << (PIL_BITS - 1);
        const uint8_t *t0 = tmp + ymin * TS + xx;
        for (int t = 0; t < cnt; ++t) acc += (int)t0[t * TS] * k[t];
        dst[(size_t)xx * bh + ra + i] = (acc >> PIL_BITS) >= 128 ? 1 : 0;
    }
}

template <int NB>
static int launch_box_prep(const float *det, int B, int D, int K, const int *H_host, const int *W_host,
                           const double *scale_shift_host, int *boxes, int *cls, float *scores, int *src_row,
                           int *num_kept, BoxRow *rows, int *nk, cudaStream_t st)
{
    UnmoldImgs<NB> P;
    for (int b = 0; b < NB; ++b) {
        UnmoldImg &I = P.v[b];
        const bool live = b < B;
        I.sy = live ? scale_shift_host[4 * b + 0] : 0.0;
        I.sx = live ? scale_shift_host[4 * b + 1] : 0.0;
        I.shy = live ? scale_shift_host[4 * b + 2] : 0.0;
        I.shx = live ? scale_shift_host[4 * b + 3] : 0.0;
        I.H = live ? H_host[b] : 0;
        I.W = live ? W_host[b] : 0;
    }
    unmold_box_prep_kernel<NB><<<B, PREP_THREADS, 0, st>>>(det, D, K, P, boxes, cls, scores, src_row, num_kept, rows, nk);
    SLN_LAUNCH_OK("unmold_box_prep_kernel");
    return SLN_OK;
}

constexpr int UNMOLD_BATCH_MAX = 512;

struct TailLayout {
    size_t rows, nk, counts, masks, total;
};

static TailLayout tail_layout(int B, int D, const int *H_host, const int *W_host, int cap)
{
    TailLayout t;
    size_t o = 0;
    long long area = 0;
    for (int b = 0; b < B; ++b) area += (long long)D * H_host[b] * W_host[b];
    t.rows = o;   o += align_up(sizeof(BoxRow) * (size_t)B * D, 256);
    t.nk = o;     o += align_up(sizeof(int) * (size_t)B, 256);
    t.counts = o; o += align_up(sizeof(uint32_t) * (size_t)B * D * cap, 256);
    t.masks = o;  o += align_up((size_t)area, 256);
    t.total = o;
    return t;
}

}  // namespace sln

using namespace sln;

extern "C" size_t sln_resize_image_workspace_bytes(int h, int w, int C, int H2, int W2)
{
    if (h <= 0 || w <= 0 || C <= 0 || H2 <= 0 || W2 <= 0) return 0;
    size_t off[5];
    return resize_ws_layout(h, w, C, H2, W2, off);
}

extern "C" int sln_resize_image_u8(const uint8_t *src, int h, int w, int C, int H2, int W2, uint8_t *out, void *workspace,
                                   size_t workspace_bytes, void *stream)
{
    SLN_REQUIRE(h > 0 && w > 0 && C > 0 && H2 > 0 && W2 > 0, SLN_ERR_ARG, "bad resize shape");
    SLN_REQUIRE(h < 65536 && w < 65536 && H2 < 65536 && W2 < 65536 && C <= 16, SLN_ERR_ARG, "resize: sides < 65536, C <= 16");
    SLN_REQUIRE(src && out, SLN_ERR_ARG, "null pointer");
    size_t off[5];
    const size_t need = resize_ws_layout(h, w, C, H2, W2, off);
    SLN_REQUIRE(workspace && workspace_bytes >= need, SLN_ERR_WORKSPACE, "resize workspace: need %zu bytes, got %zu", need, workspace_bytes);
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    ResizeTabs t;
    t.hx = reinterpret_cast<int *>(ws + off[0]);
    t.hk = reinterpret_cast<int *>(ws + off[1]);
    t.vy = reinterpret_cast<int *>(ws + off[2]);
    t.vk = reinterpret_cast<int *>(ws + off[3]);
    t.tH = resize_taps_host(w, W2);
    t.tV = resize_taps_host(h, H2);
    uint8_t *tmp = ws + off[4];
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    resize_coeffs_kernel<<<cdiv(W2 + H2, 256), 256, 0, st>>>(h, w, H2, W2, t);
    SLN_LAUNCH_OK("resize_coeffs_kernel");
    const bool vec4 = ((long long)W2 * C) % 4 == 0 && (reinterpret_cast<uintptr_t>(out) & 3u) == 0 && (reinterpret_cast<uintptr_t>(tmp) & 3u) == 0;
    const long long nh = (long long)h * W2, nv = (long long)H2 * W2 * C / (vec4 ? 4 : 1);
    SLN_REQUIRE((nh + 255) / 256 < (1ll << 31) && (nv + 255) / 256 < (1ll << 31), SLN_ERR_ARG, "resize: image too large");
    SLN_CUDA_OK(launch_chain(resize_h_kernel, dim3((unsigned)((nh + 255) / 256)), dim3(256), 0, st, true, src, h, w, C, W2, t, tmp));
    SLN_CUDA_OK(launch_chain(vec4 ? resize_v_kernel<true> : resize_v_kernel<false>, dim3((unsigned)((nv + 255) / 256)), dim3(256), 0, st, true,
                             (const uint8_t *)tmp, C, H2, W2, t, out));
    return SLN_OK;
}

extern "C" int sln_unmold_masks(const float *masks, int N, int mh, int mw, const int *boxes, int H, int W,
                                uint8_t *out, void *stream)
{
    SLN_REQUIRE(N >= 0 && mh > 0 && mw > 0 && H > 0 && W > 0, SLN_ERR_ARG, "bad unmold shape");
    SLN_REQUIRE(mh <= 256 && mw <= 256 && H < 65536 && W < 65536, SLN_ERR_ARG, "unmold: mask <= 256^2, image < 65536^2");
    if (N == 0) return SLN_OK;
    SLN_REQUIRE(masks && boxes && out, SLN_ERR_ARG, "null pointer");
    SLN_REQUIRE(N <= 65535, SLN_ERR_ARG, "unmold: at most 65535 masks per call");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const UnmoldSmem L = unmold_smem(mh, mw, W);
    SLN_REQUIRE(L.total <= 200 * 1024, SLN_ERR_ARG, "unmold: mask / image too large for shared memory (%zu bytes)", L.total);
    const bool vec = (W % 16 == 0) && (reinterpret_cast<uintptr_t>(out) % 16 == 0);
    dim3 grid(cdiv(H, UNMOLD_SLAB), N);
    if (vec) {
        SLN_CUDA_OK(cudaFuncSetAttribute(unmold_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
        unmold_kernel<true><<<grid, UNMOLD_THREADS, L.total, st>>>(masks, mh, mw, boxes, H, W, out);
    } else {
        SLN_CUDA_OK(cudaFuncSetAttribute(unmold_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
        unmold_kernel<false><<<grid, UNMOLD_THREADS, L.total, st>>>(masks, mh, mw, boxes, H, W, out);
    }
    SLN_LAUNCH_OK("unmold_kernel");
    return SLN_OK;
}

extern "C" size_t sln_unmold_rle_batched_workspace_bytes(int B, int D, const int *H_host, const int *W_host, int cap)
{
    if (B <= 0 || D <= 0 || cap < 1 || !H_host || !W_host) return 0;
    for (int b = 0; b < B; ++b)
        if (H_host[b] <= 0 || W_host[b] <= 0) return 0;
    return tail_layout(B, D, H_host, W_host, cap).total;
}

extern "C" int sln_unmold_rle_batched(const float *detections, int B, int D, const float *mrcnn_mask, int mh, int mw,
                                      int K, const long long *mask_strides_host, const int *H_host, const int *W_host,
                                      const double *scale_shift_host, int cap, int *boxes, int *class_ids, float *scores,
                                      int *src_row, int *num_kept, int *m_out, int *str_off, int *str_len,
                                      int *str_total, char *strings, long long strings_cap, void *workspace,
                                      size_t workspace_bytes, void *stream)
{
    SLN_REQUIRE(B >= 0 && D >= 0 && cap >= 1, SLN_ERR_ARG, "unmold_rle_batched: bad B / D / cap");
    SLN_REQUIRE(B <= UNMOLD_BATCH_MAX, SLN_ERR_ARG, "unmold_rle_batched: at most %d images per call", UNMOLD_BATCH_MAX);
    SLN_REQUIRE(mh > 0 && mw > 0 && mh <= 256 && mw <= 256 && K >= 1, SLN_ERR_ARG, "unmold_rle_batched: mask <= 256^2, K >= 1");
    if (B == 0) return SLN_OK;
    SLN_REQUIRE(H_host && W_host && scale_shift_host && mask_strides_host, SLN_ERR_ARG, "unmold_rle_batched: null host array");
    int Wmax = 1;
    for (int b = 0; b < B; ++b) {
        SLN_REQUIRE(H_host[b] > 0 && W_host[b] > 0 && H_host[b] < 65536 && W_host[b] < 65536, SLN_ERR_ARG,
                    "unmold_rle_batched: image %d is %dx%d (sides in [1, 65535])", b, H_host[b], W_host[b]);
        Wmax = W_host[b] > Wmax ? W_host[b] : Wmax;
    }
    SLN_REQUIRE((long long)B * D < (1ll << 31) / 8 && (long long)cap * B * D < (1ll << 40), SLN_ERR_ARG,
                "unmold_rle_batched: too many detections");
    SLN_REQUIRE(strings_cap >= 7ll * cap * B * D && strings_cap < (1ll << 31), SLN_ERR_ARG,
                "unmold_rle_batched: strings_cap must be >= 7 * cap * B * D and < 2^31 (got %lld)", strings_cap);
    if (D == 0) {
        SLN_REQUIRE(num_kept && str_total, SLN_ERR_ARG, "unmold_rle_batched: null pointer");
        SLN_CUDA_OK(cudaMemsetAsync(num_kept, 0, sizeof(int) * B, static_cast<cudaStream_t>(stream)));
        SLN_CUDA_OK(cudaMemsetAsync(str_total, 0, sizeof(int), static_cast<cudaStream_t>(stream)));
        return SLN_OK;
    }
    SLN_REQUIRE(detections && mrcnn_mask && boxes && class_ids && scores && src_row && num_kept && m_out && str_off &&
                str_len && str_total && strings, SLN_ERR_ARG, "unmold_rle_batched: null pointer");
    const TailLayout T = tail_layout(B, D, H_host, W_host, cap);
    SLN_REQUIRE(workspace && workspace_bytes >= T.total, SLN_ERR_WORKSPACE,
                "unmold_rle_batched workspace: need %zu bytes, got %zu", T.total, workspace_bytes);
    const UnmoldSmem L = unmold_smem(mh, mw, Wmax);
    SLN_REQUIRE(L.total <= 200 * 1024, SLN_ERR_ARG, "unmold_rle_batched: mask / image too large for shared memory (%zu bytes)", L.total);
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    BoxRow *rows = reinterpret_cast<BoxRow *>(ws + T.rows);
    int *nk = reinterpret_cast<int *>(ws + T.nk);
    uint32_t *counts = reinterpret_cast<uint32_t *>(ws + T.counts);
    uint8_t *maskbuf = ws + T.masks;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int rc;
    if (B <= 16)
        rc = launch_box_prep<16>(detections, B, D, K, H_host, W_host, scale_shift_host, boxes, class_ids, scores, src_row, num_kept, rows, nk, st);
    else if (B <= 128)
        rc = launch_box_prep<128>(detections, B, D, K, H_host, W_host, scale_shift_host, boxes, class_ids, scores, src_row, num_kept, rows, nk, st);
    else
        rc = launch_box_prep<UNMOLD_BATCH_MAX>(detections, B, D, K, H_host, W_host, scale_shift_host, boxes, class_ids, scores, src_row, num_kept, rows, nk, st);
    if (rc != SLN_OK) return rc;
    int Hmax = 1;
    for (int b = 0; b < B; ++b) Hmax = H_host[b] > Hmax ? H_host[b] : Hmax;
    const long long *s = mask_strides_host;
    SLN_CUDA_OK(cudaFuncSetAttribute(unmold_box_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
    unmold_box_kernel<<<dim3((unsigned)(B * D), (unsigned)cdiv(Hmax, UNMOLD_SLAB)), UNMOLD_THREADS, L.total, st>>>(
        mrcnn_mask, s[0], s[1], s[2], s[3], s[4], mh, mw, Wmax, D, rows, nk, maskbuf);
    SLN_LAUNCH_OK("unmold_box_kernel");
    rc = launch_rle_boxes(rows, nk, B, D, maskbuf, counts, cap, m_out, str_len, st);
    if (rc != SLN_OK) return rc;
    return launch_rle_strings(counts, B * D, cap, m_out, str_len, str_off, str_total, strings, st);
}
