// crop.cu -- RoIAlign (TF-style crop_and_resize) forward / backward for sm_100a.
//
// Reference semantics: roialign/roi_align/src/crop_and_resize.c:6-112 (forward),
// :157-252 (backward); GPU baseline being replaced:
// roialign/roi_align/src/cuda/crop_and_resize_kernel.cu:10-82 / :84-165.
//
// Design (DESIGN.md section "RoIAlign"):
//   forward, NHWC   one CTA per ROI; threadIdx.x walks the channel vectors of one
//                   sample point (float4, 512 B per warp-load, 4 loads in flight per
//                   sample, two samples per iteration), threadIdx.y walks sample
//                   points; per-ROI tap tables live in shared memory so the box is
//                   decoded once per CTA, not once per output element.
//   forward, NCHW   one CTA per (ROI, channel chunk); a warp owns one channel plane
//                   at a time and its lanes walk the ph*pw samples, so the writes are
//                   contiguous and the 4 taps come through L1.
//   backward, NHWC  gather form, no atomics, no memset: one CTA per 8x8 pixel tile of
//                   one image; it bins that image's ROIs against the tile (ordered
//                   ballot compaction, so the list keeps the original box order), and
//                   one warp per destination pixel then sums every contribution in
//                   the reference's serial order (box, y, x, tap) in registers and
//                   writes the pixel exactly once.  Result is bit-identical to the
//                   reference's CPU backward and independent of scheduling.
#include <stdlib.h>

#include "common.cuh"

namespace sln {

// ===========================================================================
// forward, NHWC
// ===========================================================================
struct PyramidMaps {
    const void *map[8];       // elements of the kernel's type T
    int H[8];
    int W[8];
};

// Per-sample record built once per CTA: offsets of the four taps inside the ROI's image (units of
// VEC floats, channel vector 0) and the two lerp weights; o00 < 0 marks an extrapolated sample.
struct SampleRec {
    int o00, o01, o10, o11;
    float xl, yl;
};

// img/out addressed in units of VEC elements of T (float, or a 2-byte type: see CropIO).  LEVELS: take the source map
// from `pm` by level[r]; otherwise use pm.map[0].
template <typename T, int VEC, bool LEVELS>
__global__ void __launch_bounds__(256)
crop_fwd_nhwc_kernel(PyramidMaps pm, int B, int C, const float *__restrict__ boxes,
                     const int *__restrict__ box_ind, const int *__restrict__ level, int n_levels,
                     int ph, int pw, int band, float ext, T *__restrict__ out)
{
    using IO = CropIO<T, VEC>;
    using V = typename IO::V;
    extern __shared__ __align__(16) unsigned char s_fwd_raw[];
    SampleRec *rec = reinterpret_cast<SampleRec *>(s_fwd_raw);      // [band]: samples [s_lo, s_hi) of the crop

    const int r = blockIdx.x;
    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    const int nthr = blockDim.x * blockDim.y;
    const int b = box_ind[r];
    int lv = 0;
    if (LEVELS) lv = level[r];
    const bool ok = (b >= 0 && b < B) && (!LEVELS || (lv >= 0 && lv < n_levels));
    // select the level with static indices (dynamic indexing would spill the
    // by-value parameter struct to local memory)
    int H = pm.H[0], W = pm.W[0];
    const void *mp = pm.map[0];
    if (LEVELS && ok) {
#pragma unroll
        for (int l = 1; l < 8; ++l)
            if (l == lv) { H = pm.H[l]; W = pm.W[l]; mp = pm.map[l]; }
    }
    V *__restrict__ o = reinterpret_cast<V *>(out);
    const int CV = C / VEC;
    const int s_lo = blockIdx.y * band, S = min(ph * pw - s_lo, band);     // this CTA's slice of the crop
    const size_t out_base = ((size_t)r * ph * pw + s_lo) * CV;

    if (!ok) {   // reference GPU kernel skips such boxes (kernel.cu:34-38): rows stay zero
        const V z = IO::splat(0.f);
        for (int i = tid; i < S * CV; i += nthr) o[out_base + i] = z;
        return;
    }

    const float y1 = boxes[4 * r + 0], x1 = boxes[4 * r + 1];
    const float y2 = boxes[4 * r + 2], x2 = boxes[4 * r + 3];
    const float sc_y = axis_scale(y1, y2, H, ph), sc_x = axis_scale(x1, x2, W, pw);
    for (int s = tid; s < S; s += nthr) {
        const int y = (s_lo + s) / pw, x = (s_lo + s) - y * pw;
        const Tap ty = axis_tap(y1, y2, sc_y, H, ph, y), tx = axis_tap(x1, x2, sc_x, W, pw, x);
        SampleRec q;
        q.o00 = -1; q.o01 = q.o10 = q.o11 = 0;
        q.xl = tx.lerp; q.yl = ty.lerp;
        if (ty.lo != INVALID_TAP && tx.lo != INVALID_TAP) {
            const int yh = ty.lo + (ty.lerp != 0.f), xh = tx.lo + (tx.lerp != 0.f);
            q.o00 = (ty.lo * W + tx.lo) * CV; q.o01 = (ty.lo * W + xh) * CV;
            q.o10 = (yh * W + tx.lo) * CV;    q.o11 = (yh * W + xh) * CV;
        }
        rec[s] = q;
    }
    __syncthreads();

    const V vext = IO::splat(ext);
    const V *__restrict__ img = static_cast<const V *>(mp) + (size_t)b * H * W * CV;
    const int sstep = blockDim.y;

    for (int cv = threadIdx.x; cv < CV; cv += blockDim.x) {
        const V *__restrict__ imc = img + cv;
        V *__restrict__ oc = o + out_base + cv;
        int s = threadIdx.y;
        // two sample points per iteration: 8 independent 16-byte loads in flight
        for (; s + sstep < S; s += 2 * sstep) {
            const SampleRec qa = rec[s], qb = rec[s + sstep];
            V a0, a1, a2, a3, b0, b1, b2, b3;
            if (qa.o00 >= 0) {
                a0 = IO::ld(imc + qa.o00); a1 = IO::ld(imc + qa.o01);
                a2 = IO::ld(imc + qa.o10); a3 = IO::ld(imc + qa.o11);
            }
            if (qb.o00 >= 0) {
                b0 = IO::ld(imc + qb.o00); b1 = IO::ld(imc + qb.o01);
                b2 = IO::ld(imc + qb.o10); b3 = IO::ld(imc + qb.o11);
            }
            const V ra = qa.o00 >= 0 ? IO::lerp(a0, a1, a2, a3, qa.xl, qa.yl) : vext;
            const V rb = qb.o00 >= 0 ? IO::lerp(b0, b1, b2, b3, qb.xl, qb.yl) : vext;
            __stcs(oc + (size_t)s * CV, ra);
            __stcs(oc + (size_t)(s + sstep) * CV, rb);
        }
        if (s < S) {
            const SampleRec q = rec[s];
            V res = vext;
            if (q.o00 >= 0)
                res = IO::lerp(IO::ld(imc + q.o00), IO::ld(imc + q.o01), IO::ld(imc + q.o10), IO::ld(imc + q.o11), q.xl, q.yl);
            __stcs(oc + (size_t)s * CV, res);
        }
    }
}

// ===========================================================================
// forward, NCHW (the reference's native layout; API default for NCHW tensors)
// ===========================================================================
__global__ void __launch_bounds__(256)
crop_fwd_nchw_kernel(const float *__restrict__ img, int B, int C, int H, int W,
                     const float *__restrict__ boxes, const int *__restrict__ box_ind,
                     int ph, int pw, float ext, int c_chunk, float *__restrict__ out)
{
    extern __shared__ Tap s_tab[];
    Tap *ytab = s_tab;
    Tap *xtab = s_tab + ph;
    const int r = blockIdx.x;
    const int c0 = blockIdx.y * c_chunk;
    const int c1 = min(C, c0 + c_chunk);
    const int tid = threadIdx.x;
    const int S = ph * pw;
    const int b = box_ind[r];
    float *__restrict__ o = out + ((size_t)r * C) * S;
    if (b < 0 || b >= B) {
        for (int i = c0 * S + tid; i < c1 * S; i += blockDim.x) o[i] = 0.f;
        return;
    }
    const float y1 = boxes[4 * r + 0], x1 = boxes[4 * r + 1];
    const float y2 = boxes[4 * r + 2], x2 = boxes[4 * r + 3];
    for (int k = tid; k < ph + pw; k += blockDim.x) {
        if (k < ph) ytab[k] = axis_tap(y1, y2, axis_scale(y1, y2, H, ph), H, ph, k);
        else xtab[k - ph] = axis_tap(x1, x2, axis_scale(x1, x2, W, pw), W, pw, k - ph);
    }
    __syncthreads();
    const int lane = tid & 31, warp = tid >> 5, nwarp = blockDim.x >> 5;
    const size_t plane = (size_t)H * W;
    for (int s = lane; s < S; s += 32) {
        const int y = s / pw, x = s - y * pw;
        const Tap ty = ytab[y], tx = xtab[x];
        const bool valid = ty.lo != INVALID_TAP && tx.lo != INVALID_TAP;
        const int yh = ty.lo + (ty.lerp != 0.f), xh = tx.lo + (tx.lerp != 0.f);
        const int o00 = ty.lo * W + tx.lo, o01 = ty.lo * W + xh;
        const int o10 = yh * W + tx.lo, o11 = yh * W + xh;
        for (int c = c0 + warp; c < c1; c += nwarp) {
            float v = ext;
            if (valid) {
                const float *p = img + ((size_t)b * C + c) * plane;
                v = lerp2(__ldg(p + o00), __ldg(p + o01), __ldg(p + o10), __ldg(p + o11), tx.lerp, ty.lerp);
            }
            __stcs(o + (size_t)c * S + s, v);
        }
    }
}

// ===========================================================================
// backward, NHWC
// ===========================================================================
// Pixel window [y0,y1]x[x0,x1] (inclusive, clamped) that a ROI's valid samples can
// touch, or an empty window.  Sample positions are monotone in k, so the first and
// last sample bound the window; a conservative superset is fine (exact per-sample
// tests happen in the accumulate phase).
struct RoiWin {
    short y0, y1, x0, x1;
};

__device__ __forceinline__ void axis_window(float a1, float a2, int extent, int crop, int &w0, int &w1)
{
    const float em1 = (float)(extent - 1);
    const float scale = axis_scale(a1, a2, extent, crop);
    float p0, p1;
    if (crop > 1) {
        p0 = __fmul_rn(a1, em1);
        p1 = __fadd_rn(p0, __fmul_rn((float)(crop - 1), scale));
    } else {
        p0 = p1 = (float)(0.5 * (double)__fadd_rn(a1, a2) * (double)(extent - 1));
    }
    if (!(p0 == p0) || !(p1 == p1)) { w0 = 1; w1 = 0; return; }   // NaN: nothing
    const float lo = fminf(p0, p1), hi = fmaxf(p0, p1);
    if (hi < 0.f || lo > em1) { w0 = 1; w1 = 0; return; }
    w0 = (int)floorf(fmaxf(lo, 0.f));
    w1 = (int)ceilf(fminf(hi, em1));
}

// Supertiles: every destination map is cut into at most 8x8 supertiles per image (side a
// multiple of 32 pixels); the prep kernels build, per supertile, the ordered list of ROIs
// whose window meets it, so a warp scans tens of entries instead of the whole ROI list.
struct SuperGrid {
    int side;      // pixels per supertile side
    int nx, ny;    // supertiles per image
};

static SuperGrid super_grid(int H, int W)
{
    SuperGrid g;
    int side = 32;
    while (cdiv(H, side) > 8 || cdiv(W, side) > 8) side *= 2;
    g.side = side;
    g.nx = cdiv(W, side);
    g.ny = cdiv(H, side);
    return g;
}

constexpr int BWD_MAX_LEVELS = 8;

struct BwdLevel {
    float *out;        // grad map of this level, NHWC [B,H,W,C]
    int H, W;
    int tiles_x, tiles_y;
    float rcp_tiles_x, rcp_tiles_y;
    SuperGrid sg;
    int sg_shift;      // log2(sg.side)
    int st_base;       // first supertile id of this level
    int tile_base;     // first tile (CTA) id of this level
};

struct BwdParams {
    BwdLevel lv[BWD_MAX_LEVELS];
    int n_levels;
    int sched_base[BWD_MAX_LEVELS];   // CTA numbering: smallest maps first (their strips see the longest
    int sched_lvl[BWD_MAX_LEVELS];    // ROI lists, so they must not form the tail of the launch)
};

struct BwdTileBases {  // passed by value to the main kernel: static-index compares only
    int base[BWD_MAX_LEVELS];   // first CTA of the j-th scheduled level (ascending)
    int lvl[BWD_MAX_LEVELS];    // which level that is
    int n_levels;
};

// Per-ROI sampling grid, evaluated once: pos(k) = base + k*scale on each axis, the same
// expression (and rounding) as axis_tap / crop_and_resize.c:44-56.
struct RoiAxes {
    float by, sy, bx, sx;
};

// supertile list entry: the ROI's sampling grid rides along, so that the gather kernels need no second, dependent load
// per ROI
struct __align__(16) ListEntryA {
    RoiWin win;
    int roi;
    int pad;
    RoiAxes ax;
};

__device__ __forceinline__ void axis_base_scale(float a1, float a2, int extent, int crop, float &base, float &scale)
{
    if (crop > 1) {
        base = __fmul_rn(a1, (float)(extent - 1));
        scale = axis_scale(a1, a2, extent, crop);
    } else {
        base = (float)(0.5 * (double)__fadd_rn(a1, a2) * (double)(extent - 1));
        scale = 0.f;
    }
}

// tap k of an axis from its sampling grid (axis_base_scale): the same fp32 operations as axis_tap for crop > 1; for
// crop == 1 the base plus 0 * k at k = 0, which is the base itself
__device__ __forceinline__ Tap tap_at(float base, float scale, float em1, int k)
{
    const float pos = __fadd_rn(base, __fmul_rn((float)k, scale));
    Tap t;
    if (!(pos >= 0.f && pos <= em1)) {
        t.lo = INVALID_TAP;
        t.lerp = 0.f;
    } else {
        const float fl = floorf(pos);
        t.lo = (int)fl;
        t.lerp = __fsub_rn(pos, fl);
    }
    return t;
}

// static-index copy of P.lv[l] (dynamic indexing would spill the parameter struct)
__device__ __forceinline__ BwdLevel pick_level(const BwdParams &P, int l)
{
    BwdLevel r = P.lv[0];
#pragma unroll
    for (int k = 1; k < BWD_MAX_LEVELS; ++k)
        if (k == l) r = P.lv[k];
    return r;
}

// prep 1: per-ROI axes and pixel window on its level + per-supertile counts (integer atomics:
// order-independent result); thread 0 also publishes the level table for the main kernel.
__global__ void crop_bwd_windows_kernel(const float *__restrict__ boxes, const int *__restrict__ box_ind,
                                        const int *__restrict__ level, int N, int B, int ph, int pw,
                                        BwdParams P, RoiWin *__restrict__ win, RoiAxes *__restrict__ axes,
                                        int *__restrict__ st_count,
                                        BwdLevel *__restrict__ lv_table, int *__restrict__ queue, int queue_init,
                                        int *__restrict__ gid)
{
    pdl_prologue();          // the prep launches and the main kernel are a chain of programmatic dependents (common.cuh)
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < BWD_MAX_LEVELS) lv_table[r] = pick_level(P, r);
    if (r == 0) *queue = queue_init;                 // ticket counter of the bulk-async kernel
    if (r >= N) return;
    RoiWin w;
    w.y0 = 1; w.y1 = 0; w.x0 = 1; w.x1 = 0;
    int my_gid = -1;                                 // (image, level) group of the ROI; -1: contributes nothing
    const int b = box_ind[r];
    const int l = level ? level[r] : 0;
    if (b >= 0 && b < B && l >= 0 && l < P.n_levels) {
        const BwdLevel L = pick_level(P, l);
        const float y1 = boxes[4 * r + 0], x1 = boxes[4 * r + 1], y2 = boxes[4 * r + 2], x2 = boxes[4 * r + 3];
        RoiAxes a;
        axis_base_scale(y1, y2, L.H, ph, a.by, a.sy);
        axis_base_scale(x1, x2, L.W, pw, a.bx, a.sx);
        axes[r] = a;
        int a0, a1, c0, c1;
        axis_window(y1, y2, L.H, ph, a0, a1);
        axis_window(x1, x2, L.W, pw, c0, c1);
        if (a0 <= a1 && c0 <= c1) {
            my_gid = b * P.n_levels + l;
            w.y0 = (short)a0; w.y1 = (short)a1; w.x0 = (short)c0; w.x1 = (short)c1;
            for (int sy = a0 >> L.sg_shift; sy <= (a1 >> L.sg_shift); ++sy)
                for (int sx = c0 >> L.sg_shift; sx <= (c1 >> L.sg_shift); ++sx)
                    atomicAdd(st_count + L.st_base + (b * L.sg.ny + sy) * L.sg.nx + sx, 1);
        }
    }
    win[r] = w;
    gid[r] = my_gid;
}

// prep 2: ordered ROI list of every (image, level) group.  One CTA per group walks the group ids of all ROIs (4 bytes each)
// and compacts the ids of its own ROIs in index order; the supertile fill below then looks at its group's ROIs only
// (~N / groups of them) instead of all N.  glist [n_groups][N], gcount [n_groups].
constexpr int GROUP_THREADS = 1024;
constexpr int GROUP_PER_THREAD = 8;

// SLN_BWD_PLANNED: the lists in the workspace were built by an earlier SLN_BWD_PLAN_ONLY call on the same ROIs; only the
// level table (it carries the gradient maps' addresses, unknown at plan time) and the ticket counter are refreshed.
__global__ void crop_bwd_republish_kernel(BwdParams P, BwdLevel *__restrict__ lv_table, int *__restrict__ queue, int queue_init)
{
    pdl_prologue();
    const int r = threadIdx.x;
    if (r < BWD_MAX_LEVELS) lv_table[r] = pick_level(P, r);
    if (r == 0) *queue = queue_init;
}

__global__ void __launch_bounds__(GROUP_THREADS)
crop_bwd_group_kernel(const int *__restrict__ gid, int N, int *__restrict__ glist, int *__restrict__ gcount)
{
    __shared__ int s_cnt[GROUP_PER_THREAD][GROUP_THREADS / 32];
    __shared__ int s_total;
    pdl_prologue();
    const int g = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int *__restrict__ out = glist + (size_t)g * N;
    int base = 0;
    for (int start = 0; start < N; start += GROUP_THREADS * GROUP_PER_THREAD) {
        unsigned masks[GROUP_PER_THREAD];
        __syncthreads();                                          // s_cnt reuse
#pragma unroll
        for (int it = 0; it < GROUP_PER_THREAD; ++it) {
            const int r = start + it * GROUP_THREADS + tid;
            const bool take = r < N && gid[r] == g;
            masks[it] = __ballot_sync(0xffffffffu, take);
            if (lane == 0) s_cnt[it][warp] = __popc(masks[it]);
        }
        __syncthreads();
        if (warp == 0) {                                          // exclusive scan over the (it, warp) grid in ROI order
            int run = 0;
#pragma unroll
            for (int it = 0; it < GROUP_PER_THREAD; ++it) {
                const int c = s_cnt[it][lane];
                int incl = c;
                for (int o = 1; o < 32; o <<= 1) {
                    const int v = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += v;
                }
                s_cnt[it][lane] = run + incl - c;
                run += __shfl_sync(0xffffffffu, incl, 31);
            }
            if (lane == 0) s_total = run;
        }
        __syncthreads();
#pragma unroll
        for (int it = 0; it < GROUP_PER_THREAD; ++it)
            if ((masks[it] >> lane) & 1u)
                out[base + s_cnt[it][warp] + __popc(masks[it] & ((1u << lane) - 1u))] = start + it * GROUP_THREADS + tid;
        base += s_total;
    }
    if (tid == 0) gcount[g] = base;
}

// prep 3: ordered fill.  One CTA per supertile: its list offset is the sum of the counts of
// the supertiles before it; it then takes the ROIs in index order, FILL_PER_THREAD x 1024 at
// a time (all loads issued up front), and compacts the hits with one block-wide scan so the
// list keeps the original box order.  st_off[st] is published for the main kernel.
constexpr int FILL_THREADS = 1024;
constexpr int FILL_PER_THREAD = 2;

__global__ void __launch_bounds__(FILL_THREADS)
crop_bwd_fill_kernel(const int *__restrict__ glist, const int *__restrict__ gcount,
                     const RoiWin *__restrict__ win, const RoiAxes *__restrict__ axes, int N, BwdParams P,
                     const int *__restrict__ st_count, int *__restrict__ st_off, ListEntryA *__restrict__ entries)
{
    __shared__ int s_cnt[FILL_PER_THREAD][FILL_THREADS / 32];
    __shared__ int s_base;
    pdl_prologue();
    const int st = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // offset = sum of counts before st
    int part = 0;
    for (int i = tid; i < st; i += FILL_THREADS) part += st_count[i];
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if (lane == 0) s_cnt[0][warp] = part;
    __syncthreads();
    if (tid == 0) {
        int t = 0;
        for (int k = 0; k < FILL_THREADS / 32; ++k) t += s_cnt[0][k];
        s_base = t;
        st_off[st] = t;
    }
    __syncthreads();
    int base = s_base;
    if (st_count[st] == 0) return;
    int l = 0;
#pragma unroll
    for (int k = 1; k < BWD_MAX_LEVELS; ++k)
        if (k < P.n_levels && st >= P.lv[k].st_base) l = k;
    const BwdLevel L = pick_level(P, l);
    const int local = st - L.st_base;
    const int sx = local % L.sg.nx, sy = (local / L.sg.nx) % L.sg.ny, b = local / (L.sg.nx * L.sg.ny);
    const int y0 = sy << L.sg_shift, y1 = y0 + L.sg.side - 1, x0 = sx << L.sg_shift, x1 = x0 + L.sg.side - 1;
    // the ROIs of this supertile's (image, level) group, in index order
    const int g = b * P.n_levels + l;
    const int n_g = gcount[g];
    const int *__restrict__ gl = glist + (size_t)g * N;
    for (int start = 0; start < n_g; start += FILL_THREADS * FILL_PER_THREAD) {
        RoiWin w[FILL_PER_THREAD];
        int roi[FILL_PER_THREAD];
#pragma unroll
        for (int it = 0; it < FILL_PER_THREAD; ++it) {          // all loads first
            const int i = start + it * FILL_THREADS + tid;
            roi[it] = i < n_g ? gl[i] : -1;
        }
#pragma unroll
        for (int it = 0; it < FILL_PER_THREAD; ++it)
            if (roi[it] >= 0) w[it] = win[roi[it]];
        unsigned masks[FILL_PER_THREAD];
        __syncthreads();                                          // s_cnt reuse
#pragma unroll
        for (int it = 0; it < FILL_PER_THREAD; ++it) {
            const bool take = roi[it] >= 0 && !(w[it].y1 < y0 || w[it].y0 > y1 || w[it].x1 < x0 || w[it].x0 > x1);
            masks[it] = __ballot_sync(0xffffffffu, take);
            if (lane == 0) s_cnt[it][warp] = __popc(masks[it]);
        }
        __syncthreads();
        // exclusive scan over the (it, warp) grid in ROI order: warp 0 does it serially per lane group
        if (warp == 0) {
            int run = 0;
#pragma unroll
            for (int it = 0; it < FILL_PER_THREAD; ++it) {
                const int c = s_cnt[it][lane];
                int incl = c;
                for (int o = 1; o < 32; o <<= 1) {
                    const int v = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += v;
                }
                s_cnt[it][lane] = run + incl - c;
                run += __shfl_sync(0xffffffffu, incl, 31);
            }
            if (lane == 0) s_base = run;
        }
        __syncthreads();
#pragma unroll
        for (int it = 0; it < FILL_PER_THREAD; ++it) {
            if ((masks[it] >> lane) & 1u) {
                const int slot = base + s_cnt[it][warp] + __popc(masks[it] & ((1u << lane) - 1u));
                ListEntryA e;
                e.win = w[it];
                e.roi = roi[it];
                e.pad = 0;
                e.ax = axes[roi[it]];
                entries[slot] = e;
            }
        }
        base += s_base;
    }
}

template <bool EXACT>
__device__ __forceinline__ float accum1(float s, float g, float wy, float wx, float w)
{
    if (EXACT) return __fadd_rn(s, __fmul_rn(wx, __fmul_rn(wy, g)));   // crop_and_resize.c:241-247
    return __fmaf_rn(w, g, s);
}
template <bool EXACT>
__device__ __forceinline__ float accum(float s, float g, float wy, float wx, float w) { return accum1<EXACT>(s, g, wy, wx, w); }
template <bool EXACT>
__device__ __forceinline__ float4 accum(float4 s, float4 g, float wy, float wx, float w)
{
    return make_float4(accum1<EXACT>(s.x, g.x, wy, wx, w), accum1<EXACT>(s.y, g.y, wy, wx, w),
                       accum1<EXACT>(s.z, g.z, wy, wx, w), accum1<EXACT>(s.w, g.w, wy, wx, w));
}

constexpr int BWD_ROWS = 8;            // warps per CTA; warp w owns row w of the tile
constexpr int BWD_THREADS = 32 * BWD_ROWS;
constexpr int BWD_TW = 4;              // destination pixels per warp (one strip)

// t / d for 0 <= t < 2^24 with a precomputed float reciprocal (exact after one correction)
__device__ __forceinline__ int fast_div(int t, int d, float rcp)
{
    int q = __float2int_rz(__fmul_rn(__int2float_rn(t), rcp));
    const int r = t - q * d;
    q += (r >= d) - (r < 0);
    return q;
}

// Backward kernel: gather form, no atomics, no shared memory, no block barriers; every
// destination pixel is written exactly once (zeros included, so no memset).
//   warp  = one strip of 4 horizontally adjacent destination pixels of one image and level
//   lanes = channel vectors (NV per lane), accumulators in registers
// The warp walks its supertile's ROI list in original box order.  For every ROI whose window
// meets the strip, lane k evaluates tap k of the y axis and of the x axis from the entry's
// sampling grid (tap_at: same arithmetic as the forward; the grid is read from the list at
// each use, since holding it in registers spills); ballots give the samples that touch the
// strip's row and columns; the warp then visits those samples in (y, x) order and adds each
// tap's term to the pixel it lands on.  Per destination pixel the summation order is (ROI, y, x, tap TL/TR/BL/BR) --
// the reference's serial order (crop_and_resize.c:190-250).
// EXACT: each term is wx*(wy*g) with every operation rounded like crop_and_resize.c:241-247
// (bit-identical to the reference CPU backward); otherwise fma(wy*wx, g, acc).
// 4 resident CTAs per SM (<= 64 registers): measured best on B200 (A/B runs, profiles/README.md)
template <int VEC, int NV, bool EXACT>
__global__ void __launch_bounds__(BWD_THREADS, 4)
crop_bwd_nhwc_kernel(const float *__restrict__ grads, const ListEntryA *__restrict__ entries, const int *__restrict__ st_off,
                     const int *__restrict__ st_count, const BwdLevel *__restrict__ lv_table,
                     BwdTileBases TB, int C, int ph, int pw)
{
    using V = typename VecT<VEC>::type;
    constexpr int TW = BWD_TW;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int l = TB.lvl[0];
#pragma unroll
    for (int k = 1; k < BWD_MAX_LEVELS; ++k)
        if (k < TB.n_levels && (int)blockIdx.x >= TB.base[k]) l = TB.lvl[k];
    const BwdLevel L = lv_table[l];
    int t = blockIdx.x - L.tile_base;
    const int q1 = fast_div(t, L.tiles_x, L.rcp_tiles_x);
    const int tx_i = t - q1 * L.tiles_x;
    const int b = fast_div(q1, L.tiles_y, L.rcp_tiles_y);
    const int ty_i = q1 - b * L.tiles_y;
    const int H = L.H, W = L.W;
    const int py = ty_i * BWD_ROWS + warp;
    if (py >= H) return;
    const int tx0 = tx_i * TW, tx1 = min(tx0 + TW, W) - 1;
    const float em1y = (float)(H - 1), em1x = (float)(W - 1);
    const int CV = C / VEC;
    const int cvbase = blockIdx.y * (32 * NV) + lane;

    // accumulators of the strip's 4 pixels x NV channel vectors: named scalars, so they
    // stay in registers (an indexed array ends up in local memory here)
    static_assert(NV == 1 || NV == 2, "1-2 vectors per lane");
    const V zero = make_splat(0.f, (V *)nullptr);
    V p0a = zero, p1a = zero, p2a = zero, p3a = zero;
    V p0b = zero, p1b = zero, p2b = zero, p3b = zero;
    const bool va_ok = cvbase < CV, vb_ok = NV == 2 && cvbase + 32 < CV;

    const int st = L.st_base + (b * L.sg.ny + (py >> L.sg_shift)) * L.sg.nx + (tx0 >> L.sg_shift);
    const int n_list = st_count[st];
    const ListEntryA *__restrict__ list = entries + (n_list ? st_off[st] : 0);
    const V *__restrict__ g = reinterpret_cast<const V *>(grads) + cvbase;
    const int S = ph * pw;

#define SLN_BWD_ADD(PA, PB, WX, WW)                                   \
    {                                                                 \
        PA = accum<EXACT>(PA, ga, wy, WX, WW);                        \
        if (NV == 2) PB = accum<EXACT>(PB, gb, wy, WX, WW);           \
    }

    for (int base = 0; base < n_list; base += 32) {
        const int li = base + lane;
        int my_roi = -1;
        bool take = false;
        if (li < n_list) {
            const RoiWin w = list[li].win;
            my_roi = list[li].roi;
            take = !(w.y1 < py || w.y0 > py || w.x1 < tx0 || w.x0 > tx1);
        }
        unsigned todo = __ballot_sync(0xffffffffu, take);
        while (todo) {
            const int bit = __ffs(todo) - 1;
            todo &= todo - 1;
            const int r = __shfl_sync(0xffffffffu, my_roi, bit);
            const RoiAxes *__restrict__ ax = &list[base + bit].ax;
            const V *gr = g + (size_t)r * S * CV;
            for (int ky0 = 0; ky0 < ph; ky0 += 32) {
                Tap ty;
                ty.lo = INVALID_TAP; ty.lerp = 0.f;
                if (ky0 + lane < ph) ty = tap_at(ax->by, ax->sy, em1y, ky0 + lane);
                unsigned ym = __ballot_sync(0xffffffffu, ty.lo == py || (ty.lo + 1 == py && ty.lerp != 0.f));
                while (ym) {
                    const int yb = __ffs(ym) - 1;
                    ym &= ym - 1;
                    const int ylo = __shfl_sync(0xffffffffu, ty.lo, yb);
                    const float yl = __shfl_sync(0xffffffffu, ty.lerp, yb);
                    // row weight that lands on py; when the sample row is integral (floor == ceil)
                    // both the top and the bottom tap hit this row, weights 1 and 0, in that order
                    const bool y_int = (yl == 0.f);
                    const float wy0 = (ylo == py) ? __fsub_rn(1.f, yl) : yl;
                    const int yoff = (ky0 + yb) * pw;
                    for (int kx0 = 0; kx0 < pw; kx0 += 32) {
                        Tap tx;
                        tx.lo = INVALID_TAP; tx.lerp = 0.f;
                        if (kx0 + lane < pw) tx = tap_at(ax->bx, ax->sx, em1x, kx0 + lane);
                        unsigned xm = __ballot_sync(0xffffffffu, tx.lo != INVALID_TAP && tx.lo <= tx1 &&
                                                                     tx.lo + (tx.lerp != 0.f) >= tx0);
                        while (xm) {
                            const int xb = __ffs(xm) - 1;
                            xm &= xm - 1;
                            const int xlo = __shfl_sync(0xffffffffu, tx.lo, xb);
                            const float xl = __shfl_sync(0xffffffffu, tx.lerp, xb);
                            const float wl = __fsub_rn(1.f, xl), wr = xl;
                            const int pl = xlo - tx0;               // strip pixel of the left tap (-1 .. 3)
                            V ga = zero, gb = zero;
                            if (va_ok) ga = ldg_vec(gr + (size_t)(yoff + kx0 + xb) * CV);
                            if (vb_ok) gb = ldg_vec(gr + (size_t)(yoff + kx0 + xb) * CV + 32);
                            if (!y_int && xl != 0.f) {
                                // generic sample: one row weight; left tap on pl, right tap on pl+1
                                const float wy = wy0;
                                const float w_l = __fmul_rn(wy, wl), w_r = __fmul_rn(wy, wr);
                                switch (pl) {
                                case -1: SLN_BWD_ADD(p0a, p0b, wr, w_r) break;
                                case 0: SLN_BWD_ADD(p0a, p0b, wl, w_l) SLN_BWD_ADD(p1a, p1b, wr, w_r) break;
                                case 1: SLN_BWD_ADD(p1a, p1b, wl, w_l) SLN_BWD_ADD(p2a, p2b, wr, w_r) break;
                                case 2: SLN_BWD_ADD(p2a, p2b, wl, w_l) SLN_BWD_ADD(p3a, p3b, wr, w_r) break;
                                default: SLN_BWD_ADD(p3a, p3b, wl, w_l) break;
                                }
                            } else {
                                // integral sample position on an axis: taps coincide; keep the reference's
                                // TL, TR, BL, BR order per pixel
                                const int pr = (xl == 0.f) ? pl : pl + 1;
                                for (int pass = 0; pass < (y_int ? 2 : 1); ++pass) {
                                    const float wy = pass == 0 ? wy0 : yl;
                                    const float w_l = __fmul_rn(wy, wl), w_r = __fmul_rn(wy, wr);
                                    if (pl == 0) SLN_BWD_ADD(p0a, p0b, wl, w_l)
                                    else if (pl == 1) SLN_BWD_ADD(p1a, p1b, wl, w_l)
                                    else if (pl == 2) SLN_BWD_ADD(p2a, p2b, wl, w_l)
                                    else if (pl == 3) SLN_BWD_ADD(p3a, p3b, wl, w_l)
                                    if (pr == 0) SLN_BWD_ADD(p0a, p0b, wr, w_r)
                                    else if (pr == 1) SLN_BWD_ADD(p1a, p1b, wr, w_r)
                                    else if (pr == 2) SLN_BWD_ADD(p2a, p2b, wr, w_r)
                                    else if (pr == 3) SLN_BWD_ADD(p3a, p3b, wr, w_r)
                                }
                            }
                        }
                    }
                }
            }
        }
    }
#undef SLN_BWD_ADD

    // ---- write every pixel of the strip exactly once (zeros included)
    V *__restrict__ o = reinterpret_cast<V *>(L.out) + (((size_t)b * H + py) * W + tx0) * CV + cvbase;
    if (va_ok) {
        __stcs(o, p0a);
        if (tx0 + 1 <= tx1) __stcs(o + (size_t)CV, p1a);
        if (tx0 + 2 <= tx1) __stcs(o + 2 * (size_t)CV, p2a);
        if (tx0 + 3 <= tx1) __stcs(o + 3 * (size_t)CV, p3a);
    }
    if (vb_ok) {
        __stcs(o + 32, p0b);
        if (tx0 + 1 <= tx1) __stcs(o + (size_t)CV + 32, p1b);
        if (tx0 + 2 <= tx1) __stcs(o + 2 * (size_t)CV + 32, p2b);
        if (tx0 + 3 <= tx1) __stcs(o + 3 * (size_t)CV + 32, p3b);
    }
}

#include "crop_bwd_tma.cuh"

// ===========================================================================
// layout converters: per image, [C][HW] <-> [HW][C]
// ===========================================================================
// T: float, or unsigned short for every 2-byte type (the transposes move bits)
template <typename T>
__global__ void __launch_bounds__(256)
transpose_kernel(const T *__restrict__ src, T *__restrict__ dst, int rows, int cols)
{
    // src [batch][rows][cols] -> dst [batch][cols][rows]
    __shared__ T tile[32][33];
    const size_t boff = (size_t)blockIdx.z * rows * cols;
    const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int j = ty; j < 32; j += 8) {
        const int r = r0 + j, c = c0 + tx;
        if (r < rows && c < cols) tile[j][tx] = __ldg(src + boff + (size_t)r * cols + c);
    }
    __syncthreads();
    for (int j = ty; j < 32; j += 8) {
        const int c = c0 + j, r = r0 + tx;
        if (r < rows && c < cols) dst[boff + (size_t)c * rows + r] = tile[tx][j];
    }
}

// Vector form for rows % 4 == 0, cols % 4 == 0 and 16-byte aligned pointers (every FPN map and crop tensor): a 64 x 64
// tile per CTA, 16-byte loads along the source rows, 16-byte stores along the destination rows.  The tile is stored
// transposed with a 65-word pitch, so the four scalar writes of a loaded vector hit four different rows (banks 4 apart
// plus the lane's own offset: conflict-free per quarter warp) and the 16-byte reads along a row are contiguous.
// 2-byte elements move as 8-byte vectors of four (ushort4), with the same tile and thread mapping.
template <typename T> struct Vec4T;
template <> struct Vec4T<float> { using type = float4; };
template <> struct Vec4T<unsigned short> { using type = ushort4; };

template <typename T>
__global__ void __launch_bounds__(256)
transpose_v4_kernel(const T *__restrict__ src, T *__restrict__ dst, int rows, int cols)
{
    using V4 = typename Vec4T<T>::type;
    __shared__ T tile[64][65];                                  // tile[c][r] = src[r0 + r][c0 + c]
    const size_t boff = (size_t)blockIdx.z * rows * cols;
    const int c0 = blockIdx.x * 64, r0 = blockIdx.y * 64;
    const int q = threadIdx.x & 15, j0 = threadIdx.x >> 4;      // 16 vectors per 64-float row, 16 rows per pass
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int r = r0 + j0 + 16 * k, c = c0 + 4 * q;
        if (r < rows && c < cols) {
            const V4 v = __ldcs(reinterpret_cast<const V4 *>(src + boff + (size_t)r * cols + c));
            tile[4 * q + 0][j0 + 16 * k] = v.x;
            tile[4 * q + 1][j0 + 16 * k] = v.y;
            tile[4 * q + 2][j0 + 16 * k] = v.z;
            tile[4 * q + 3][j0 + 16 * k] = v.w;
        }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int c = c0 + j0 + 16 * k, r = r0 + 4 * q;          // destination row c, columns r .. r + 3
        if (c < cols && r < rows) {
            const T *t = &tile[j0 + 16 * k][4 * q];
            V4 o;
            o.x = t[0]; o.y = t[1]; o.z = t[2]; o.w = t[3];
            __stcs(reinterpret_cast<V4 *>(dst + boff + (size_t)c * rows + r), o);
        }
    }
}

template <typename T>
static int launch_transpose(const T *src, T *dst, int batch, int rows, int cols, cudaStream_t st)
{
    constexpr uintptr_t a = 4 * sizeof(T) - 1;
    const bool al = ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & a) == 0;
    if (batch == 0 || rows == 0 || cols == 0) return SLN_OK;
    if (rows % 4 == 0 && cols % 4 == 0 && al && batch <= 65535 && cdiv(rows, 64) <= 65535) {
        dim3 grid(cdiv(cols, 64), cdiv(rows, 64), batch);
        transpose_v4_kernel<T><<<grid, 256, 0, st>>>(src, dst, rows, cols);
        SLN_LAUNCH_OK("transpose_v4_kernel");
        return SLN_OK;
    }
    SLN_REQUIRE(cdiv(rows, 32) <= 65535 && batch <= 65535, SLN_ERR_ARG,
                "transpose: rows/batch too large (%d, %d)", rows, batch);
    dim3 grid(cdiv(cols, 32), cdiv(rows, 32), batch);
    transpose_kernel<T><<<grid, 256, 0, st>>>(src, dst, rows, cols);
    SLN_LAUNCH_OK("transpose_kernel");
    return SLN_OK;
}

// ===========================================================================
// host-side launch logic
// ===========================================================================
static bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// max_crop: 255 for the backward (sample ranges are packed in bytes), 4096 for the forward
static int check_crop_args(const void *image, const void *boxes, const void *box_ind, const void *out,
                           int B, int C, int H, int W, int N, int ph, int pw, int max_crop = 255)
{
    SLN_REQUIRE(B >= 0 && C >= 0 && H >= 0 && W >= 0 && N >= 0, SLN_ERR_ARG, "negative size");
    SLN_REQUIRE(ph >= 1 && pw >= 1 && ph <= max_crop && pw <= max_crop, SLN_ERR_ARG,
                "crop size %dx%d outside [1,%d]", ph, pw, max_crop);
    SLN_REQUIRE(H <= 32767 && W <= 32767, SLN_ERR_ARG, "map side > 32767");
    if (N > 0 && C > 0) {
        SLN_REQUIRE(boxes && box_ind && out, SLN_ERR_ARG, "null pointer");
        SLN_REQUIRE(B == 0 || H == 0 || W == 0 || image, SLN_ERR_ARG, "null image");
    }
    return SLN_OK;
}

static void fwd_block_shape(int CV, dim3 &block)
{
    int bx = CV < 256 ? CV : 256;
    if (bx >= 32) bx = (bx / 32) * 32;          // whole warps along the channel axis
    int by = 256 / bx;
    if (by < 1) by = 1;
    block = dim3(bx, by, 1);
}

// widest vector of VEC elements that C and every pointer allow: 16 bytes (float4 / 8 x 2-byte) down to one element
template <typename T, int VEC>
static bool fwd_vec_ok(const PyramidMaps &pm, int n_levels, int C, const void *out)
{
    constexpr uintptr_t a = sizeof(T) * VEC - 1;
    bool ok = C % VEC == 0 && (reinterpret_cast<uintptr_t>(out) & a) == 0;
    for (int l = 0; l < n_levels; ++l) ok = ok && (reinterpret_cast<uintptr_t>(pm.map[l]) & a) == 0;
    return ok;
}

template <typename T, int VEC>
static void launch_fwd_nhwc(dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool levels, const PyramidMaps &pm, int n_levels,
                            int B, int C, const float *boxes, const int *box_ind, const int *level, int ph, int pw, int band,
                            float ext, T *out)
{
    if (levels) crop_fwd_nhwc_kernel<T, VEC, true><<<grid, block, smem, st>>>(pm, B, C, boxes, box_ind, level, n_levels, ph, pw, band, ext, out);
    else crop_fwd_nhwc_kernel<T, VEC, false><<<grid, block, smem, st>>>(pm, B, C, boxes, box_ind, level, n_levels, ph, pw, band, ext, out);
}

template <typename T>
static int crop_fwd_nhwc(const PyramidMaps &pm, int n_levels, bool levels, int B, int C,
                         const float *boxes, const int *box_ind, const int *level, int N, int ph, int pw,
                         float ext, T *out, cudaStream_t st)
{
    constexpr bool F32 = sizeof(T) == 4;
    constexpr int VMAX = 16 / sizeof(T);                     // elements per 16-byte vector
    int vec = 1;
    if (fwd_vec_ok<T, VMAX>(pm, n_levels, C, out)) vec = VMAX;
    else if (!F32 && fwd_vec_ok<T, 4>(pm, n_levels, C, out)) vec = 4;
    else if (!F32 && fwd_vec_ok<T, 2>(pm, n_levels, C, out)) vec = 2;
    const int CV = C / vec;
    dim3 block;
    fwd_block_shape(CV, block);
    const int band = ph * pw < 2048 ? ph * pw : 2048;        // samples per CTA (48 KB of records at most)
    const size_t smem = sizeof(SampleRec) * (size_t)band;
    size_t plane_max = 0;
    for (int l = 0; l < n_levels; ++l) plane_max = plane_max > (size_t)pm.H[l] * pm.W[l] ? plane_max : (size_t)pm.H[l] * pm.W[l];
    SLN_REQUIRE(plane_max * (size_t)CV < (1ull << 31), SLN_ERR_ARG, "feature map too large for 32-bit tap offsets");
    dim3 grid(N, cdiv(ph * pw, band));
    SLN_REQUIRE(grid.y <= 65535, SLN_ERR_ARG, "crop too large");
    if constexpr (F32) {
        if (vec == 4) launch_fwd_nhwc<T, 4>(grid, block, smem, st, levels, pm, n_levels, B, C, boxes, box_ind, level, ph, pw, band, ext, out);
        else launch_fwd_nhwc<T, 1>(grid, block, smem, st, levels, pm, n_levels, B, C, boxes, box_ind, level, ph, pw, band, ext, out);
    } else {
        if (vec == 8) launch_fwd_nhwc<T, 8>(grid, block, smem, st, levels, pm, n_levels, B, C, boxes, box_ind, level, ph, pw, band, ext, out);
        else if (vec == 4) launch_fwd_nhwc<T, 4>(grid, block, smem, st, levels, pm, n_levels, B, C, boxes, box_ind, level, ph, pw, band, ext, out);
        else if (vec == 2) launch_fwd_nhwc<T, 2>(grid, block, smem, st, levels, pm, n_levels, B, C, boxes, box_ind, level, ph, pw, band, ext, out);
        else launch_fwd_nhwc<T, 1>(grid, block, smem, st, levels, pm, n_levels, B, C, boxes, box_ind, level, ph, pw, band, ext, out);
    }
    SLN_LAUNCH_OK("crop_fwd_nhwc_kernel");
    return SLN_OK;
}

// the forward of a call whose element type is named by an SLN_DTYPE_* code
static int crop_fwd_nhwc_dt(int dtype, const PyramidMaps &pm, int n_levels, bool levels, int B, int C, const float *boxes,
                            const int *box_ind, const int *level, int N, int ph, int pw, float ext, void *out, cudaStream_t st)
{
    switch (dtype) {
    case SLN_DTYPE_F32:
        return crop_fwd_nhwc(pm, n_levels, levels, B, C, boxes, box_ind, level, N, ph, pw, ext, static_cast<float *>(out), st);
    case SLN_DTYPE_BF16:
        return crop_fwd_nhwc(pm, n_levels, levels, B, C, boxes, box_ind, level, N, ph, pw, ext, static_cast<__nv_bfloat16 *>(out), st);
    case SLN_DTYPE_F16:
        return crop_fwd_nhwc(pm, n_levels, levels, B, C, boxes, box_ind, level, N, ph, pw, ext, static_cast<__half *>(out), st);
    }
    SLN_REQUIRE(false, SLN_ERR_ARG, "unknown dtype %d", dtype);
    return SLN_ERR_ARG;
}

struct BwdWs {
    RoiWin *win;
    RoiAxes *axes;
    int *st_count;
    int *st_off;
    BwdLevel *lv_table;
    int *queue;
    int *gid;       // [N] (image, level) group of every ROI
    int *gcount;    // [B * n_levels]
    int *glist;     // [B * n_levels][N] ROI ids per group, in index order
    ListEntryA *entries;
};

constexpr int BWD_MAX_ST = 64;        // supertiles per image and level (8 x 8)

static size_t bwd_ws_bytes(int N, int B, int n_levels)
{
    // every ROI lives on one level and meets at most 64 supertiles of its image
    const size_t n_st = (size_t)B * BWD_MAX_ST * (size_t)n_levels + 1;
    return align_up(sizeof(RoiWin) * (size_t)N, 256) + align_up(sizeof(RoiAxes) * (size_t)N, 256) +
           2 * align_up(sizeof(int) * n_st, 256) + align_up(sizeof(BwdLevel) * BWD_MAX_LEVELS, 256) + 256 +
           align_up(sizeof(int) * (size_t)N, 256) + align_up(sizeof(int) * (size_t)B * n_levels, 256) +
           align_up(sizeof(int) * (size_t)B * n_levels * (size_t)N, 256) +
           align_up(sizeof(ListEntryA) * (size_t)N * BWD_MAX_ST, 256);
}

// Which gather kernel serves an fp32 call: the bulk-async kernel (crop_bwd_tma.cuh) when C % 4 == 0, grads and grad maps
// are 16-byte aligned and the crop is at most 32 samples per side; the strip form (crop_bwd_nhwc_kernel) for every other
// shape.  DESIGN.md section 4.3 has the timings of both.
static bool bwd_use_tma(int ph, int pw, bool vec4)
{
    return vec4 && ph <= bwdtma::MAX_POOL && pw <= bwdtma::MAX_POOL;
}

// persistent grid of the bulk-async kernel: two CTAs per SM; CTA i starts with work item i and then draws tickets
// (heaviest levels first)
static unsigned bwd_tma_grid(long long n_work)
{
    const long long resident = 2LL * sm_count();
    return (unsigned)(n_work < resident ? n_work : resident);
}

// One configuration of the bulk-async kernel (stage size, ring depth; see crop_bwd_tma.cuh).  2-byte element types keep
// the fp32 stage geometry (samples per stage, ring depth); their stages take half the bytes.
template <typename T, bool EXACT, int STG_S, int NST>
static int launch_bwd_tma_cfg(const T *grads, const BwdWs &ws, const BwdTileBases &TB, long long n_work, int chunks, int C,
                              int ph, int pw, cudaStream_t st)
{
    const size_t smem = bwdtma::smem_bytes<STG_S, NST, sizeof(T)>();
    void (*kern)(const T *, const ListEntryA *, const int *, const int *, const BwdLevel *, BwdTileBases, int, int, int, int,
                 int, int *);
    if constexpr (sizeof(T) == 4) {
        kern = C % 256 == 0  ? bwdtma::crop_bwd_tma_kernel<2, EXACT, true, STG_S, NST>
               : C == 128    ? bwdtma::crop_bwd_tma_kernel<1, EXACT, true, STG_S, NST>
               : C > 128     ? bwdtma::crop_bwd_tma_kernel<2, EXACT, false, STG_S, NST>
                             : bwdtma::crop_bwd_tma_kernel<1, EXACT, false, STG_S, NST>;
    } else {
        kern = C % 256 == 0 ? bwdtma::crop_bwd_tma_b16_kernel<T, EXACT, true, STG_S, NST>
                            : bwdtma::crop_bwd_tma_b16_kernel<T, EXACT, false, STG_S, NST>;
    }
    SLN_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // work-item tickets: tickets below `grid` are the CTAs' first items (the counter starts there, set by the windows kernel)
    const unsigned grid = bwd_tma_grid(n_work);
    // programmatic dependent of the prep chain: its CTAs are placed and set their barriers up while the fill kernel's last
    // wave drains, and block (griddepcontrol.wait in the kernel) before they read anything the prep wrote
    SLN_CUDA_OK(launch_chain(kern, dim3(grid), dim3(bwdtma::THREADS), smem, st, true, grads,
                             (const ListEntryA *)ws.entries, (const int *)ws.st_off, (const int *)ws.st_count,
                             (const BwdLevel *)ws.lv_table, TB, C, ph, pw, (int)n_work, chunks, ws.queue));
    SLN_LAUNCH_OK("crop_bwd_tma_kernel");
    return SLN_OK;
}

template <typename T, bool EXACT>
static int launch_bwd_tma(const T *grads, const BwdWs &ws, const BwdParams &P, long long tiles, int C, int ph, int pw,
                          cudaStream_t st)
{
    const int chunks = cdiv(C, bwdtma::CH_MAX);
    const long long n_work = tiles * chunks;                 // work item = (tile, channel chunk)
    SLN_REQUIRE(n_work < (1ll << 24), SLN_ERR_ARG, "too many tiles x channel chunks (%lld)", n_work);
    if (n_work == 0) return SLN_OK;
    BwdTileBases TB{};
    TB.n_levels = P.n_levels;
    for (int j = 0; j < P.n_levels; ++j) { TB.base[j] = P.sched_base[j]; TB.lvl[j] = P.sched_lvl[j]; }
    // small crops stage ~8 samples per (ROI, tile) hit: more, smaller stages; large crops: fewer, larger ones.
    // SLN_BWD_CFG=0/1 in the environment forces one for A/B runs.
    const char *e = getenv("SLN_BWD_CFG");
    const bool small = (e && (e[0] == '0' || e[0] == '1')) ? e[0] == '1' : ph * pw <= 64;
    if (small) return launch_bwd_tma_cfg<T, EXACT, 16, 6>(grads, ws, TB, n_work, chunks, C, ph, pw, st);
    return launch_bwd_tma_cfg<T, EXACT, 32, 3>(grads, ws, TB, n_work, chunks, C, ph, pw, st);
}

// the bulk-async kernel for the element type named by an SLN_DTYPE_* code
static int launch_bwd_tma_dt(int dtype, const void *grads, bool exact, const BwdWs &ws, const BwdParams &P, long long tiles,
                             int C, int ph, int pw, cudaStream_t st)
{
    switch (dtype) {
    case SLN_DTYPE_BF16: {
        const __nv_bfloat16 *g = static_cast<const __nv_bfloat16 *>(grads);
        return exact ? launch_bwd_tma<__nv_bfloat16, true>(g, ws, P, tiles, C, ph, pw, st)
                     : launch_bwd_tma<__nv_bfloat16, false>(g, ws, P, tiles, C, ph, pw, st);
    }
    case SLN_DTYPE_F16: {
        const __half *g = static_cast<const __half *>(grads);
        return exact ? launch_bwd_tma<__half, true>(g, ws, P, tiles, C, ph, pw, st)
                     : launch_bwd_tma<__half, false>(g, ws, P, tiles, C, ph, pw, st);
    }
    default: {
        const float *g = static_cast<const float *>(grads);
        return exact ? launch_bwd_tma<float, true>(g, ws, P, tiles, C, ph, pw, st)
                     : launch_bwd_tma<float, false>(g, ws, P, tiles, C, ph, pw, st);
    }
    }
}

template <int VEC, int NV, bool EXACT>
static int launch_bwd(const float *grads, const BwdWs &ws, const BwdParams &P, long long tiles, int C, int ph, int pw,
                      cudaStream_t st)
{
    const int chunks = cdiv(C / VEC, 32 * NV);
    SLN_REQUIRE(chunks <= 65535, SLN_ERR_ARG, "too many channel chunks");
    if (tiles == 0) return SLN_OK;
    BwdTileBases TB{};
    TB.n_levels = P.n_levels;
    for (int j = 0; j < P.n_levels; ++j) { TB.base[j] = P.sched_base[j]; TB.lvl[j] = P.sched_lvl[j]; }
    dim3 grid((unsigned)tiles, chunks);
    crop_bwd_nhwc_kernel<VEC, NV, EXACT><<<grid, BWD_THREADS, 0, st>>>(grads, ws.entries, ws.st_off, ws.st_count, ws.lv_table,
                                                                      TB, C, ph, pw);
    SLN_LAUNCH_OK("crop_bwd_nhwc_kernel");
    return SLN_OK;
}

template <int VEC, bool EXACT>
static int dispatch_bwd(const float *grads, const BwdWs &ws, const BwdParams &P, long long tiles, int C, int ph, int pw,
                        cudaStream_t st)
{
    const int CV = C / VEC;
    // two channel vectors per lane halve the control work per byte, but also the CTA count:
    // only use them when the maps provide enough strips to fill the machine
    if (CV > 32 && tiles >= 6LL * sm_count()) return launch_bwd<VEC, 2, EXACT>(grads, ws, P, tiles, C, ph, pw, st);
    return launch_bwd<VEC, 1, EXACT>(grads, ws, P, tiles, C, ph, pw, st);
}

// grads [N,ph,pw,C]; one grad map per level (NHWC); level[i] selects the map of ROI i (null: level 0)
// mode 0: plan + run; 1 (SLN_BWD_PLAN_ONLY): build the lists only (grads / maps are not touched; maps[l] only need to be
// plausible addresses); 2 (SLN_BWD_PLANNED): the workspace holds the lists of a mode-1 call with the same boxes, box_ind,
// level, N, C, ph, pw, B and map sizes -- skip the three prep launches and only republish the level table (grad map
// addresses and the tile geometry of the gather kernel that runs) and the ticket counter.  The lists do not depend on
// which gather kernel runs, so every shape plans ahead the same way.
// dtype: element type of grads and maps (SLN_DTYPE_*).  2-byte types run the bulk-async kernel only (C % 8 == 0, crops
// of at most 32 per side, 16-byte aligned pointers); other shapes are refused.  A plan does not depend on the dtype: the
// prep kernels see boxes and sizes only, and the tile grid (8 x 8) and channel chunks (256) are the same for every type.
static int crop_bwd_nhwc(int dtype, const void *grads, const float *boxes, const int *box_ind, const int *level, int N, int C,
                         int ph, int pw, float *const *maps, const int *Hs, const int *Ws, int n_levels, int B,
                         bool exact, void *wsp, size_t ws_bytes, cudaStream_t st, int mode = 0)
{
    SLN_REQUIRE(dtype == SLN_DTYPE_F32 || dtype == SLN_DTYPE_BF16 || dtype == SLN_DTYPE_F16, SLN_ERR_ARG, "unknown dtype %d", dtype);
    if (B == 0 || C == 0) return SLN_OK;
    SLN_REQUIRE(ws_bytes >= bwd_ws_bytes(N, B, n_levels), SLN_ERR_WORKSPACE,
                "crop bwd workspace: need %zu bytes, got %zu", bwd_ws_bytes(N, B, n_levels), ws_bytes);
    SLN_REQUIRE(wsp != nullptr, SLN_ERR_WORKSPACE, "null workspace");
    BwdParams P{};
    P.n_levels = n_levels;
    int n_st = 0;
    long long tiles = 0;
    bool vec4 = C % 4 == 0 && aligned16(grads);
    for (int l = 0; l < n_levels; ++l) vec4 = vec4 && aligned16(maps[l]);
    const bool use_tma = bwd_use_tma(ph, pw, vec4);
    // 2-byte shapes that pass this check are bulk-async shapes (C % 8 == 0 implies C % 4 == 0)
    SLN_REQUIRE(dtype == SLN_DTYPE_F32 || mode == 1 || (C % 8 == 0 && use_tma), SLN_ERR_LAYOUT,
                "2-byte crop backward needs C %% 8 == 0 (C = %d), crops of at most 32 per side (%dx%d) and 16-byte aligned "
                "grads and grad maps", C, ph, pw);
    for (int l = 0; l < n_levels; ++l) {
        BwdLevel &L = P.lv[l];
        L.out = maps[l];
        L.H = Hs[l];
        L.W = Ws[l];
        L.sg = super_grid(L.H, L.W);
        L.sg_shift = 0;
        while ((1 << L.sg_shift) < L.sg.side) ++L.sg_shift;
        L.st_base = n_st;
        n_st += B * L.sg.nx * L.sg.ny;
        L.tiles_x = cdiv(L.W, use_tma ? bwdtma::TW : BWD_TW);
        L.tiles_y = cdiv(L.H, use_tma ? bwdtma::TH : BWD_ROWS);
        L.rcp_tiles_x = L.tiles_x ? 1.0f / (float)L.tiles_x : 0.f;
        L.rcp_tiles_y = L.tiles_y ? 1.0f / (float)L.tiles_y : 0.f;
        SLN_REQUIRE((size_t)L.H * L.W == 0 || maps[l] != nullptr, SLN_ERR_ARG, "null grad map");
    }
    {   // schedule levels by ascending map area
        int ord[BWD_MAX_LEVELS];
        for (int l = 0; l < n_levels; ++l) ord[l] = l;
        for (int a = 0; a < n_levels; ++a)
            for (int b2 = a + 1; b2 < n_levels; ++b2)
                if ((long long)P.lv[ord[b2]].H * P.lv[ord[b2]].W < (long long)P.lv[ord[a]].H * P.lv[ord[a]].W) {
                    const int t = ord[a]; ord[a] = ord[b2]; ord[b2] = t;
                }
        for (int j = 0; j < n_levels; ++j) {
            BwdLevel &L = P.lv[ord[j]];
            L.tile_base = (int)tiles;
            P.sched_base[j] = (int)tiles;
            P.sched_lvl[j] = ord[j];
            tiles += (long long)L.tiles_x * L.tiles_y * B;
        }
    }
    SLN_REQUIRE(tiles < (1ll << 24), SLN_ERR_ARG, "too many tiles (%lld)", tiles);
    unsigned char *p = static_cast<unsigned char *>(wsp);
    const size_t n_st_cap = (size_t)B * BWD_MAX_ST * (size_t)n_levels + 1;
    BwdWs ws;
    ws.win = reinterpret_cast<RoiWin *>(p);        p += align_up(sizeof(RoiWin) * (size_t)N, 256);
    ws.axes = reinterpret_cast<RoiAxes *>(p);      p += align_up(sizeof(RoiAxes) * (size_t)N, 256);
    ws.st_count = reinterpret_cast<int *>(p);      p += align_up(sizeof(int) * n_st_cap, 256);
    ws.st_off = reinterpret_cast<int *>(p);        p += align_up(sizeof(int) * n_st_cap, 256);
    ws.lv_table = reinterpret_cast<BwdLevel *>(p); p += align_up(sizeof(BwdLevel) * BWD_MAX_LEVELS, 256);
    ws.queue = reinterpret_cast<int *>(p);         p += 256;
    ws.gid = reinterpret_cast<int *>(p);           p += align_up(sizeof(int) * (size_t)N, 256);
    ws.gcount = reinterpret_cast<int *>(p);        p += align_up(sizeof(int) * (size_t)B * n_levels, 256);
    ws.glist = reinterpret_cast<int *>(p);         p += align_up(sizeof(int) * (size_t)B * n_levels * (size_t)N, 256);
    ws.entries = reinterpret_cast<ListEntryA *>(p);

    const int queue_init = (int)bwd_tma_grid(tiles * cdiv(C, bwdtma::CH_MAX));   // ticket counter of the bulk-async kernel
    if (mode == 2) {
        SLN_CUDA_OK(launch_chain(crop_bwd_republish_kernel, dim3(1), dim3(32), 0, st, true, P, ws.lv_table, ws.queue, queue_init));
        SLN_LAUNCH_OK("crop_bwd_republish_kernel");
    } else {
        SLN_CUDA_OK(cudaMemsetAsync(ws.st_count, 0, sizeof(int) * (size_t)(n_st + 1), st));
        // the windows kernel also publishes the level table, so it always runs (>= 1 CTA)
        SLN_CUDA_OK(launch_chain(crop_bwd_windows_kernel, dim3(cdiv(N > BWD_MAX_LEVELS ? N : BWD_MAX_LEVELS, 256)), dim3(256), 0, st,
                                 true, boxes, box_ind, level, N, B, ph, pw, P, ws.win, ws.axes, ws.st_count, ws.lv_table,
                                 ws.queue, queue_init, ws.gid));
        SLN_LAUNCH_OK("crop_bwd_windows_kernel");
        if (N > 0 && n_st > 0) {
            SLN_CUDA_OK(launch_chain(crop_bwd_group_kernel, dim3(B * n_levels), dim3(GROUP_THREADS), 0, st, true, (const int *)ws.gid,
                                     N, ws.glist, ws.gcount));
            SLN_LAUNCH_OK("crop_bwd_group_kernel");
            SLN_CUDA_OK(launch_chain(crop_bwd_fill_kernel, dim3(n_st), dim3(FILL_THREADS), 0, st, true, (const int *)ws.glist,
                                     (const int *)ws.gcount, (const RoiWin *)ws.win, (const RoiAxes *)ws.axes, N, P,
                                     (const int *)ws.st_count, ws.st_off, ws.entries));
            SLN_LAUNCH_OK("crop_bwd_fill_kernel");
        }
        if (mode == 1) return SLN_OK;
    }
    if (use_tma) return launch_bwd_tma_dt(dtype, grads, exact, ws, P, tiles, C, ph, pw, st);
    const float *g32 = static_cast<const float *>(grads);
    if (vec4) {
        if (exact) return dispatch_bwd<4, true>(g32, ws, P, tiles, C, ph, pw, st);
        return dispatch_bwd<4, false>(g32, ws, P, tiles, C, ph, pw, st);
    }
    if (exact) return dispatch_bwd<1, true>(g32, ws, P, tiles, C, ph, pw, st);
    return dispatch_bwd<1, false>(g32, ws, P, tiles, C, ph, pw, st);
}

}  // namespace sln

// ===========================================================================
// C ABI
// ===========================================================================
using namespace sln;

extern "C" int sln_crop_and_resize_fwd_ex(int dtype, const void *image, int B, int C, int H, int W, int layout,
                                          const float *boxes, const int *box_ind, int N, int ph, int pw,
                                          float ext, void *crops, void *stream)
{
    SLN_REQUIRE(dtype == SLN_DTYPE_F32 || dtype == SLN_DTYPE_BF16 || dtype == SLN_DTYPE_F16, SLN_ERR_ARG, "unknown dtype %d", dtype);
    int rc = check_crop_args(image, boxes, box_ind, crops, B, C, H, W, N, ph, pw, 4096);
    if (rc != SLN_OK) return rc;
    if (N == 0 || C == 0) return SLN_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (layout == SLN_LAYOUT_NHWC) {
        PyramidMaps pm{};
        pm.map[0] = image; pm.H[0] = H; pm.W[0] = W;
        return crop_fwd_nhwc_dt(dtype, pm, 1, false, B, C, boxes, box_ind, nullptr, N, ph, pw, ext, crops, st);
    }
    SLN_REQUIRE(layout == SLN_LAYOUT_NCHW, SLN_ERR_LAYOUT, "unknown layout %d", layout);
    SLN_REQUIRE(dtype == SLN_DTYPE_F32, SLN_ERR_LAYOUT, "2-byte crop forward is NHWC-only; convert with sln_nchw_to_nhwc_b16");
    // channel chunks so that small-N calls still fill the machine
    int c_chunk = C;
    const int want_ctas = 4 * sm_count();
    if (N < want_ctas) {
        const int split = cdiv(want_ctas, N);
        c_chunk = cdiv(C, split);
        if (c_chunk < 8) c_chunk = C < 8 ? C : 8;
    }
    dim3 grid(N, cdiv(C, c_chunk));
    SLN_REQUIRE(grid.y <= 65535, SLN_ERR_ARG, "too many channel chunks");
    // tap tables: 64 KB at 4096 x 4096, so crops with ph + pw > 6144 need more than the 48 KB granted without opting in
    const size_t smem = sizeof(Tap) * (size_t)(ph + pw);
    if (smem > 48 * 1024)
        SLN_CUDA_OK(cudaFuncSetAttribute(crop_fwd_nchw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    crop_fwd_nchw_kernel<<<grid, 256, smem, st>>>(static_cast<const float *>(image), B, C, H, W, boxes, box_ind, ph, pw, ext,
                                                  c_chunk, static_cast<float *>(crops));
    SLN_LAUNCH_OK("crop_fwd_nchw_kernel");
    return SLN_OK;
}

extern "C" int sln_crop_and_resize_fwd(const float *image, int B, int C, int H, int W, int layout,
                                       const float *boxes, const int *box_ind, int N, int ph, int pw,
                                       float ext, float *crops, void *stream)
{
    return sln_crop_and_resize_fwd_ex(SLN_DTYPE_F32, image, B, C, H, W, layout, boxes, box_ind, N, ph, pw, ext, crops, stream);
}

extern "C" size_t sln_crop_and_resize_bwd_workspace_bytes(int N, int B, int ph, int pw)
{
    if (N < 0 || B < 0 || ph < 1 || pw < 1) return 0;
    return bwd_ws_bytes(N, B, 1);
}

extern "C" int sln_crop_and_resize_bwd_ex(int dtype, const void *grads, const float *boxes, const int *box_ind, int N,
                                          int C, int ph, int pw, void *grad_image, int B, int H, int W,
                                          int layout, int flags, void *workspace, size_t workspace_bytes, void *stream)
{
    SLN_REQUIRE(layout == SLN_LAYOUT_NHWC, SLN_ERR_LAYOUT,
                "crop backward is NHWC-only; convert with sln_nchw_to_nhwc / sln_nhwc_to_nchw");
    int rc = check_crop_args(grad_image, boxes, box_ind, grad_image, B, C, H, W, N, ph, pw);
    if (rc != SLN_OK) return rc;
    SLN_REQUIRE(N == 0 || C == 0 || grads, SLN_ERR_ARG, "null grads");
    if (H == 0 || W == 0) return SLN_OK;
    float *maps[1] = {static_cast<float *>(grad_image)};
    return crop_bwd_nhwc(dtype, grads, boxes, box_ind, nullptr, N, C, ph, pw, maps, &H, &W, 1, B,
                         (flags & SLN_BWD_EXACT) != 0, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

extern "C" int sln_crop_and_resize_bwd(const float *grads, const float *boxes, const int *box_ind, int N,
                                       int C, int ph, int pw, float *grad_image, int B, int H, int W,
                                       int layout, int flags, void *workspace, size_t workspace_bytes, void *stream)
{
    return sln_crop_and_resize_bwd_ex(SLN_DTYPE_F32, grads, boxes, box_ind, N, C, ph, pw, grad_image, B, H, W, layout, flags,
                                      workspace, workspace_bytes, stream);
}

extern "C" int sln_pyramid_crop_fwd_ex(int dtype, const void *const *maps_host, const int *H_host, const int *W_host,
                                       int n_levels, int B, int C, const float *boxes, const int *box_ind,
                                       const int *level, int N, int ph, int pw, float ext, void *crops,
                                       void *stream)
{
    SLN_REQUIRE(n_levels >= 1 && n_levels <= 8, SLN_ERR_ARG, "n_levels %d outside [1,8]", n_levels);
    SLN_REQUIRE(maps_host && H_host && W_host && level, SLN_ERR_ARG, "null pointer");
    PyramidMaps pm{};
    for (int l = 0; l < n_levels; ++l) {
        int rc = check_crop_args(maps_host[l], boxes, box_ind, crops, B, C, H_host[l], W_host[l], N, ph, pw, 4096);
        if (rc != SLN_OK) return rc;
        pm.map[l] = maps_host[l]; pm.H[l] = H_host[l]; pm.W[l] = W_host[l];
    }
    if (N == 0 || C == 0) return SLN_OK;
    return crop_fwd_nhwc_dt(dtype, pm, n_levels, true, B, C, boxes, box_ind, level, N, ph, pw, ext, crops,
                            static_cast<cudaStream_t>(stream));
}

extern "C" int sln_pyramid_crop_fwd(const float *const *maps_host, const int *H_host, const int *W_host,
                                    int n_levels, int B, int C, const float *boxes, const int *box_ind,
                                    const int *level, int N, int ph, int pw, float ext, float *crops,
                                    void *stream)
{
    return sln_pyramid_crop_fwd_ex(SLN_DTYPE_F32, reinterpret_cast<const void *const *>(maps_host), H_host, W_host, n_levels, B, C,
                                   boxes, box_ind, level, N, ph, pw, ext, crops, stream);
}

extern "C" size_t sln_pyramid_crop_bwd_workspace_bytes(int N, int B, int n_levels, int ph, int pw)
{
    if (N < 0 || B < 0 || n_levels < 1 || n_levels > BWD_MAX_LEVELS || ph < 1 || pw < 1) return 0;
    return bwd_ws_bytes(N, B, n_levels);
}

extern "C" int sln_pyramid_crop_bwd_ex(int dtype, const void *grads, const float *boxes, const int *box_ind, const int *level,
                                       int N, int C, int ph, int pw, void *const *grad_maps_host, const int *H_host,
                                       const int *W_host, int n_levels, int B, int flags, void *workspace,
                                       size_t workspace_bytes, void *stream)
{
    SLN_REQUIRE(n_levels >= 1 && n_levels <= BWD_MAX_LEVELS, SLN_ERR_ARG, "n_levels %d outside [1,8]", n_levels);
    SLN_REQUIRE(grad_maps_host && H_host && W_host, SLN_ERR_ARG, "null pointer");
    SLN_REQUIRE(n_levels == 1 || level || N == 0, SLN_ERR_ARG, "level array required for n_levels > 1");
    for (int l = 0; l < n_levels; ++l) {
        int rc = check_crop_args(grad_maps_host[l], boxes, box_ind, grad_maps_host[l], B, C, H_host[l], W_host[l], N, ph, pw);
        if (rc != SLN_OK) return rc;
    }
    const int mode = (flags & SLN_BWD_PLAN_ONLY) ? 1 : ((flags & SLN_BWD_PLANNED) ? 2 : 0);
    SLN_REQUIRE(N == 0 || C == 0 || grads || mode == 1, SLN_ERR_ARG, "null grads");
    return crop_bwd_nhwc(dtype, grads, boxes, box_ind, level, N, C, ph, pw, reinterpret_cast<float *const *>(grad_maps_host),
                         H_host, W_host, n_levels, B, (flags & SLN_BWD_EXACT) != 0, workspace, workspace_bytes,
                         static_cast<cudaStream_t>(stream), mode);
}

extern "C" int sln_pyramid_crop_bwd(const float *grads, const float *boxes, const int *box_ind, const int *level,
                                    int N, int C, int ph, int pw, float *const *grad_maps_host, const int *H_host,
                                    const int *W_host, int n_levels, int B, int flags, void *workspace,
                                    size_t workspace_bytes, void *stream)
{
    return sln_pyramid_crop_bwd_ex(SLN_DTYPE_F32, grads, boxes, box_ind, level, N, C, ph, pw,
                                   reinterpret_cast<void *const *>(grad_maps_host), H_host, W_host, n_levels, B, flags,
                                   workspace, workspace_bytes, stream);
}

// FPN level of every ROI, modal/modals.py:53-64, with the exact fp32 operation sequence the reference's torch
// expression evaluates on a CUDA tensor (`224.0 / t` is reciprocal-then-multiply in torch; sqrt, divide and log are the
// IEEE / libdevice ones; round is half-to-even; the float -> int conversion maps NaN to 0 before the clamp):
//   lvl = clamp(int(round(4 + log(sqrt(h*w) / (224 / sqrt(H*W))) / log(2))), 2, 5)          -> level_out = lvl - 2
// One launch instead of the ten elementwise launches of the torch expression.
namespace sln {
__global__ void roi_level_kernel(const float *__restrict__ boxes, int N, float image_area, int *__restrict__ level_out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const float4 b = *reinterpret_cast<const float4 *>(boxes + 4 * (size_t)i);
    const float h = __fsub_rn(b.z, b.x), w = __fsub_rn(b.w, b.y);
    const float d = __fmul_rn(__fdiv_rn(1.f, __fsqrt_rn(image_area)), 224.f);
    const float q = __fdiv_rn(__fsqrt_rn(__fmul_rn(h, w)), d);
    const float v = __fadd_rn(__fdiv_rn(logf(q), logf(2.f)), 4.f);
    const float r = rintf(v);
    int lv = (r != r) ? 0 : (r >= 2147483648.f ? 2147483647 : (r <= -2147483648.f ? (-2147483647 - 1) : (int)r));
    lv = lv < 2 ? 2 : (lv > 5 ? 5 : lv);
    level_out[i] = lv - 2;
}
}  // namespace sln

extern "C" int sln_roi_levels(const float *boxes, int N, int image_h, int image_w, int *level_out, void *stream)
{
    SLN_REQUIRE(N >= 0, SLN_ERR_ARG, "negative N");
    if (N == 0) return SLN_OK;
    SLN_REQUIRE(boxes && level_out, SLN_ERR_ARG, "null pointer");
    SLN_REQUIRE((reinterpret_cast<uintptr_t>(boxes) & 15u) == 0, SLN_ERR_LAYOUT, "boxes must be 16-byte aligned");
    // torch.tensor([float(H * W)], dtype=float32): the product in exact integer arithmetic, rounded once
    const float area = (float)((double)image_h * (double)image_w);
    sln::roi_level_kernel<<<cdiv(N, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(boxes, N, area, level_out);
    SLN_LAUNCH_OK("roi_level_kernel");
    return SLN_OK;
}

template <typename T>
static int nchw_to_nhwc(const T *src, T *dst, int B, int C, int H, int W, void *stream)
{
    SLN_REQUIRE(B >= 0 && C >= 0 && H >= 0 && W >= 0, SLN_ERR_ARG, "negative size");
    SLN_REQUIRE((size_t)H * W < (1ull << 31), SLN_ERR_ARG, "plane too large");
    if ((size_t)B * C * H * W == 0) return SLN_OK;
    SLN_REQUIRE(src && dst && src != dst, SLN_ERR_ARG, "null or aliased pointers");
    return launch_transpose(src, dst, B, C, H * W, static_cast<cudaStream_t>(stream));
}

template <typename T>
static int nhwc_to_nchw(const T *src, T *dst, int B, int C, int H, int W, void *stream)
{
    SLN_REQUIRE(B >= 0 && C >= 0 && H >= 0 && W >= 0, SLN_ERR_ARG, "negative size");
    SLN_REQUIRE((size_t)H * W < (1ull << 31), SLN_ERR_ARG, "plane too large");
    if ((size_t)B * C * H * W == 0) return SLN_OK;
    SLN_REQUIRE(src && dst && src != dst, SLN_ERR_ARG, "null or aliased pointers");
    return launch_transpose(src, dst, B, H * W, C, static_cast<cudaStream_t>(stream));
}

extern "C" int sln_nchw_to_nhwc(const float *src, float *dst, int B, int C, int H, int W, void *stream)
{
    return nchw_to_nhwc(src, dst, B, C, H, W, stream);
}

extern "C" int sln_nhwc_to_nchw(const float *src, float *dst, int B, int C, int H, int W, void *stream)
{
    return nhwc_to_nchw(src, dst, B, C, H, W, stream);
}

extern "C" int sln_nchw_to_nhwc_b16(const uint16_t *src, uint16_t *dst, int B, int C, int H, int W, void *stream)
{
    return nchw_to_nhwc(src, dst, B, C, H, W, stream);
}

extern "C" int sln_nhwc_to_nchw_b16(const uint16_t *src, uint16_t *dst, int B, int C, int H, int W, void *stream)
{
    return nhwc_to_nchw(src, dst, B, C, H, W, stream);
}
