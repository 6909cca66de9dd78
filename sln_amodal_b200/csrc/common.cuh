// common.cuh -- shared helpers for libsln_b200 (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/sln_b200.h"

namespace sln {

// thread-local error text behind sln_last_error_string()
void set_error(const char *fmt, ...);

#define SLN_REQUIRE(cond, code, ...)                 \
    do {                                             \
        if (!(cond)) {                               \
            ::sln::set_error(__VA_ARGS__);           \
            return (code);                           \
        }                                            \
    } while (0)

#define SLN_CUDA_OK(expr)                                                                  \
    do {                                                                                   \
        cudaError_t _e = (expr);                                                           \
        if (_e != cudaSuccess) {                                                           \
            ::sln::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),       \
                             __FILE__, __LINE__);                                          \
            return SLN_ERR_CUDA;                                                           \
        }                                                                                  \
    } while (0)

#define SLN_LAUNCH_OK(name)                                                                \
    do {                                                                                   \
        cudaError_t _e = cudaGetLastError();                                               \
        if (_e != cudaSuccess) {                                                           \
            ::sln::set_error("launch of %s failed: %s", name, cudaGetErrorString(_e));     \
            return SLN_ERR_CUDA;                                                           \
        }                                                                                  \
    } while (0)

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
static inline int cdiv(int a, int b) { return (a + b - 1) / b; }

int sm_count();   // of the current device (not cached)

// ---------------------------------------------------------------------------
// Programmatic dependent launch (sm_90+): a kernel launched with launch_chain(pdl = true) may be scheduled while its
// predecessor in the stream is still running; pdl_prologue() at the very top of BOTH kernels makes the predecessor
// allow that as soon as all of its CTAs are resident and makes the successor block until the predecessor has
// completed and flushed -- only the launch latency and CTA placement overlap, never the bodies.  Without the launch
// attribute both instructions are no-ops.  SLN_PDL=0 in the environment turns the attribute off (A/B).
// ---------------------------------------------------------------------------
__device__ __forceinline__ void pdl_prologue()
{
    asm volatile("griddepcontrol.launch_dependents;");
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

bool pdl_enabled();   // lib.cu: getenv("SLN_PDL") != "0", cached

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_chain(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                       bool pdl, Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = (pdl && pdl_enabled()) ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---------------------------------------------------------------------------
// One axis of the crop sampling grid, bit-compatible with crop_and_resize.c:44-56
// (scale and sample position, un-fused fp32; the single-sample case is evaluated in
// double like the reference's `0.5 * (y1 + y2) * (image_height - 1)`), :58/:80 (range
// test) and :71-73/:89-91 (floorf / ceilf taps, lerp = pos - floor).
// lo == INVALID_TAP marks a sample outside [0, extent-1] (or a NaN position, which is
// undefined behaviour in the reference and is treated as "outside" here).
// hi is not stored: ceilf(pos) == lo + (lerp != 0) exactly, because pos - floorf(pos)
// is exact in fp32.
// ---------------------------------------------------------------------------
constexpr int INVALID_TAP = -(1 << 30);

struct Tap {
    int lo;
    float lerp;
};

__device__ __forceinline__ float axis_scale(float a1, float a2, int extent, int crop)
{
    return crop > 1 ? __fdiv_rn(__fmul_rn(__fsub_rn(a2, a1), (float)(extent - 1)), (float)(crop - 1))
                    : 0.f;
}

__device__ __forceinline__ Tap axis_tap(float a1, float a2, float scale, int extent, int crop, int k)
{
    const float em1 = (float)(extent - 1);
    float pos;
    if (crop > 1) {
        pos = __fadd_rn(__fmul_rn(a1, em1), __fmul_rn((float)k, scale));
    } else {
        pos = (float)(0.5 * (double)__fadd_rn(a1, a2) * (double)(extent - 1));
    }
    Tap t;
    if (!(pos >= 0.f && pos <= em1)) {   // also catches NaN
        t.lo = INVALID_TAP;
        t.lerp = 0.f;
    } else {
        const float fl = floorf(pos);
        t.lo = (int)fl;
        t.lerp = __fsub_rn(pos, fl);
    }
    return t;
}

// bilinear blend with the reference's rounding sequence (crop_and_resize.c:102-106)
__device__ __forceinline__ float lerp2(float tl, float tr, float bl, float br, float xl, float yl)
{
    const float top = __fadd_rn(tl, __fmul_rn(__fsub_rn(tr, tl), xl));
    const float bot = __fadd_rn(bl, __fmul_rn(__fsub_rn(br, bl), xl));
    return __fadd_rn(top, __fmul_rn(__fsub_rn(bot, top), yl));
}

template <int VEC> struct VecT;
template <> struct VecT<1> { using type = float; };
template <> struct VecT<4> { using type = float4; };

__device__ __forceinline__ float ldg_vec(const float *p) { return __ldg(p); }
__device__ __forceinline__ float4 ldg_vec(const float4 *p) { return __ldg(p); }

__device__ __forceinline__ float4 make_splat(float v, float4 *) { return make_float4(v, v, v, v); }
__device__ __forceinline__ float make_splat(float v, float *) { return v; }

__device__ __forceinline__ float lerp2v(float tl, float tr, float bl, float br, float xl, float yl)
{
    return lerp2(tl, tr, bl, br, xl, yl);
}
// ---------------------------------------------------------------------------
// Packed fp32 pairs (sm_100: FADD2 / FMUL2 / FFMA2, PTX .f32x2): two IEEE-rounded fp32 operations per instruction, each
// half rounded exactly like the scalar instruction.  The bit-parity kernels need the reference's UN-fused sequence
// (every multiply and add rounded on its own, crop_and_resize.c:102-106), and ptxas (12.9) contracts mul.rn.f32x2 +
// add.rn.f32x2 into one FFMA2 -- unlike the scalar mul.rn / add.rn pair, which it never fuses; it even sees through
// fma.rn.f32x2(a, b, -0.0) as a product and contracts that (checked in SASS).  So in the un-fused kernels only the
// subtraction and the addition are packed and the product stays two scalar mul.rn.f32: 4 instructions per pair of
// lerps instead of 6.  Where fusing is the defined behaviour (the backward's default mode) FFMA2 is used as it is.
// ---------------------------------------------------------------------------
typedef unsigned long long f32x2_t;
__device__ __forceinline__ f32x2_t pk2(float lo, float hi)
{
    f32x2_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpk2(f32x2_t v, float &lo, float &hi)
{
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2_t add2_rn(f32x2_t a, f32x2_t b)
{
    f32x2_t r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2_t sub2_rn(f32x2_t a, f32x2_t b)
{
    f32x2_t r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2_t fma2_rn(f32x2_t a, f32x2_t b, f32x2_t c)
{
    f32x2_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
// a + (b - a) * w on a pair, each operation rounded on its own (the reference's sequence): FADD2, 2 x FMUL, FADD2
__device__ __forceinline__ f32x2_t lerp_pair(f32x2_t a, f32x2_t b, float w)
{
    float d0, d1;
    unpk2(sub2_rn(b, a), d0, d1);
    return add2_rn(a, pk2(__fmul_rn(d0, w), __fmul_rn(d1, w)));
}

__device__ __forceinline__ float4 lerp2v(float4 tl, float4 tr, float4 bl, float4 br, float xl, float yl)
{
    // 24 instructions instead of 36 per float4, same bits as lerp2() on every component
    const f32x2_t top0 = lerp_pair(pk2(tl.x, tl.y), pk2(tr.x, tr.y), xl), top1 = lerp_pair(pk2(tl.z, tl.w), pk2(tr.z, tr.w), xl);
    const f32x2_t bot0 = lerp_pair(pk2(bl.x, bl.y), pk2(br.x, br.y), xl), bot1 = lerp_pair(pk2(bl.z, bl.w), pk2(br.z, br.w), xl);
    const f32x2_t r0 = lerp_pair(top0, bot0, yl), r1 = lerp_pair(top1, bot1, yl);
    float4 r;
    unpk2(r0, r.x, r.y);
    unpk2(r1, r.z, r.w);
    return r;
}

// ---------------------------------------------------------------------------
// 2-byte elements (bf16 / fp16 maps under autocast).  Widening to fp32 is exact, so a kernel that widens its inputs,
// runs the fp32 operation sequence and rounds its result once (to nearest even) gives the bits of the fp32 kernel run
// on the widened tensor, rounded.  Elements travel as raw 16-bit words.
// ---------------------------------------------------------------------------
template <typename T> struct Elem16;
template <> struct Elem16<__nv_bfloat16> {
    static __device__ __forceinline__ float widen(unsigned short h) { return __uint_as_float((unsigned)h << 16); }
    static __device__ __forceinline__ void widen2(unsigned w, float &lo, float &hi)
    {
        lo = __uint_as_float(w << 16);
        hi = __uint_as_float(w & 0xffff0000u);
    }
    static __device__ __forceinline__ unsigned short narrow(float f) { return __bfloat16_as_ushort(__float2bfloat16_rn(f)); }
    static __device__ __forceinline__ unsigned narrow2(float lo, float hi)
    {
        const __nv_bfloat162 r = __floats2bfloat162_rn(lo, hi);
        return *reinterpret_cast<const unsigned *>(&r);
    }
};
template <> struct Elem16<__half> {
    static __device__ __forceinline__ float widen(unsigned short h) { return __half2float(__ushort_as_half(h)); }
    static __device__ __forceinline__ void widen2(unsigned w, float &lo, float &hi)
    {
        const float2 f = __half22float2(*reinterpret_cast<const __half2 *>(&w));
        lo = f.x;
        hi = f.y;
    }
    static __device__ __forceinline__ unsigned short narrow(float f) { return __half_as_ushort(__float2half_rn(f)); }
    static __device__ __forceinline__ unsigned narrow2(float lo, float hi)
    {
        const __half2 r = __floats2half2_rn(lo, hi);
        return *reinterpret_cast<const unsigned *>(&r);
    }
};

// 16 bytes of a 2-byte type (8 elements) <-> two float4 (elements 0..3, 4..7)
template <typename T>
__device__ __forceinline__ void widen8(uint4 v, float4 &a, float4 &b)
{
    Elem16<T>::widen2(v.x, a.x, a.y);
    Elem16<T>::widen2(v.y, a.z, a.w);
    Elem16<T>::widen2(v.z, b.x, b.y);
    Elem16<T>::widen2(v.w, b.z, b.w);
}
template <typename T>
__device__ __forceinline__ uint4 narrow8(float4 a, float4 b)
{
    return make_uint4(Elem16<T>::narrow2(a.x, a.y), Elem16<T>::narrow2(a.z, a.w), Elem16<T>::narrow2(b.x, b.y),
                      Elem16<T>::narrow2(b.z, b.w));
}

// Vector I/O of the forward gather: VEC elements per load / store.  fp32: float / float4 as before.  2-byte types:
// 8 / 4 / 2 / 1 elements (16 / 8 / 4 / 2 bytes), widened on load, the lerp run on packed fp32 pairs (same bits as
// lerp2() per element), rounded once on store.
template <typename T, int VEC> struct CropIO {
    using V = typename VecT<VEC>::type;
    static __device__ __forceinline__ V ld(const V *p) { return ldg_vec(p); }
    static __device__ __forceinline__ V splat(float v) { return make_splat(v, (V *)nullptr); }
    static __device__ __forceinline__ V lerp(V tl, V tr, V bl, V br, float xl, float yl) { return lerp2v(tl, tr, bl, br, xl, yl); }
};

template <int VEC> struct Vec16;
template <> struct Vec16<8> { using type = uint4; };
template <> struct Vec16<4> { using type = uint2; };
template <> struct Vec16<2> { using type = unsigned; };
template <> struct Vec16<1> { using type = unsigned short; };

template <typename T, int VEC> struct CropIO16 {
    using V = typename Vec16<VEC>::type;
    static constexpr int NW = VEC >= 2 ? VEC / 2 : 1;     // 32-bit words per vector
    static __device__ __forceinline__ V ld(const V *p) { return __ldg(p); }
    static __device__ __forceinline__ V splat(float v)
    {
        if constexpr (VEC == 1) {
            return Elem16<T>::narrow(v);
        } else {
            unsigned w[NW];
            const unsigned h = Elem16<T>::narrow2(v, v);
#pragma unroll
            for (int i = 0; i < NW; ++i) w[i] = h;
            V r;
            __builtin_memcpy(&r, w, sizeof(V));
            return r;
        }
    }
    static __device__ __forceinline__ V lerp(V tl, V tr, V bl, V br, float xl, float yl)
    {
        using E = Elem16<T>;
        if constexpr (VEC == 1) {
            return E::narrow(lerp2(E::widen(tl), E::widen(tr), E::widen(bl), E::widen(br), xl, yl));
        } else {
            unsigned a[NW], b[NW], c[NW], d[NW], r[NW];
            __builtin_memcpy(a, &tl, sizeof(V));
            __builtin_memcpy(b, &tr, sizeof(V));
            __builtin_memcpy(c, &bl, sizeof(V));
            __builtin_memcpy(d, &br, sizeof(V));
#pragma unroll
            for (int i = 0; i < NW; ++i) {
                float a0, a1, b0, b1, c0, c1, d0, d1;
                E::widen2(a[i], a0, a1);
                E::widen2(b[i], b0, b1);
                E::widen2(c[i], c0, c1);
                E::widen2(d[i], d0, d1);
                const f32x2_t top = lerp_pair(pk2(a0, a1), pk2(b0, b1), xl), bot = lerp_pair(pk2(c0, c1), pk2(d0, d1), xl);
                float r0, r1;
                unpk2(lerp_pair(top, bot, yl), r0, r1);
                r[i] = E::narrow2(r0, r1);
            }
            V out;
            __builtin_memcpy(&out, r, sizeof(V));
            return out;
        }
    }
};
template <int VEC> struct CropIO<__nv_bfloat16, VEC> : CropIO16<__nv_bfloat16, VEC> {};
template <int VEC> struct CropIO<__half, VEC> : CropIO16<__half, VEC> {};

}  // namespace sln
