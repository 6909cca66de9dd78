// rle.cu -- COCO run-length encoding of binary masks on the device (SURVEY.md section 8(f), row 3).
//
// Reference: cocoapi/common/maskApi.c:32-41 (rleEncode: one serial pass per mask, counts of alternating runs starting
// with the run of zeros) and :204-216 (rleToString: LEB128-like, 6 bits per char, delta against counts[i-2]).
// The evaluation path of the reference (amodal_train.py:371-400) pastes every detection mask into a full-resolution
// plane and encodes it on the host.  Here one cluster of 8 CTAs per mask finds the run boundaries with word-wide compares:
//   pass 1  every thread counts the value changes in its contiguous chunk (a change at j <=> T[j] != T[j-1], T[-1] = 0)
//   scan    block-wide exclusive scan of the counts, and a running maximum of "last change position so far"
//   pass 2  every thread walks its chunk again and writes, for its k-th change at j, counts[k] = j - previous change
// The masks are read in the memory order given (pycocotools encodes column-major planes: pass them transposed).
// Bytes per mask: a (read twice, the second pass from L2) + 4 m written.
// For sln_unmold_rle_batched the runs come from box-sized masks instead (rle_box_kernel: the plane is never built), and
// the strings are made on the device too (rle_str_*_kernel: maskApi.c's rleToString, packed for all masks).
#include <stdlib.h>

#include "common.cuh"
#include "eval_tail.cuh"

#include <cooperative_groups.h>

namespace sln {

constexpr int RLE_THREADS = 1024;
constexpr int RLE_CLUSTER = 8;             // CTAs per mask

// value changes inside one 32-bit word: bit 8q set <=> byte q differs from the byte before it
__device__ __forceinline__ unsigned change_bits(unsigned w, unsigned prev_byte)
{
    const unsigned shifted = (w << 8) | prev_byte;
    return __vcmpne4(w, shifted) & 0x01010101u;
}

// One cluster of RLE_CLUSTER CTAs per mask (8192 threads, 16-byte loads): a 1024^2 mask is 128 bytes per thread.  The
// per-CTA totals (number of changes, last change position) are exchanged through distributed shared memory.
__global__ void __cluster_dims__(RLE_CLUSTER, 1, 1) __launch_bounds__(RLE_THREADS)
rle_encode_kernel(const unsigned char *__restrict__ masks, long long a, unsigned *__restrict__ counts, int cap,
                  int *__restrict__ m_out)
{
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    __shared__ int s_cnt[RLE_THREADS / 32];
    __shared__ long long s_last[RLE_THREADS / 32];
    __shared__ int s_cta_cnt;                      // read by the whole cluster
    __shared__ long long s_cta_last;
    const int mask_id = blockIdx.x / RLE_CLUSTER, crank = (int)cluster.block_rank();
    const unsigned char *T = masks + (size_t)mask_id * a;
    unsigned *out = counts + (size_t)mask_id * cap;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // chunk of this thread: a multiple of 16 bytes so that vector loads stay aligned when the mask base is
    long long len = (a + RLE_CLUSTER * RLE_THREADS - 1) / (RLE_CLUSTER * RLE_THREADS);
    len = (len + 15) & ~15ll;
    const long long gt = (long long)crank * RLE_THREADS + tid;
    const long long j0 = min(a, gt * len), j1 = min(a, j0 + len);
    const bool vec = ((reinterpret_cast<uintptr_t>(T) & 15u) == 0);

    auto walk = [&](auto &&on_change) {
        unsigned prev = j0 > 0 ? T[j0 - 1] : 0u;
        long long j = j0;
        if (vec) {
            auto vec16 = [&](const uint4 v, long long jj) {
                const unsigned w[4] = {v.x, v.y, v.z, v.w};
                // byte-wise "differs from the byte before": four XORs; almost every 16-byte piece of a mask is constant,
                // so the per-byte extraction only runs where something changes
                const unsigned d[4] = {w[0] ^ ((w[0] << 8) | prev), w[1] ^ ((w[1] << 8) | (w[0] >> 24)),
                                       w[2] ^ ((w[2] << 8) | (w[1] >> 24)), w[3] ^ ((w[3] << 8) | (w[2] >> 24))};
                prev = w[3] >> 24;
                if ((d[0] | d[1] | d[2] | d[3]) == 0u) return;
#pragma unroll
                for (int q4 = 0; q4 < 4; ++q4) {
                    unsigned ch = __vcmpne4(d[q4], 0u) & 0x01010101u;
                    while (ch) {
                        const int q = (__ffs(ch) - 1) >> 3;
                        ch &= ch - 1;
                        on_change(jj + 4 * q4 + q);
                    }
                }
            };
            for (; j + 16 <= j1; j += 16) vec16(__ldg(reinterpret_cast<const uint4 *>(T + j)), j);
        }
        for (; j < j1; ++j) {
            const unsigned v = T[j];
            if (v != prev) on_change(j);
            prev = v;
        }
    };

    // ---- pass 1: count, remember the last change
    int cnt = 0;
    long long last = -1;
    walk([&](long long j) { ++cnt; last = j; });
    // ---- exclusive scan of cnt, inclusive running max of last (positions grow with the thread index)
    int incl = cnt;
    long long lmax = last;
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        const long long l = __shfl_up_sync(0xffffffffu, lmax, o);
        if (lane >= o) { incl += v; lmax = max(lmax, l); }
    }
    if (lane == 31) { s_cnt[warp] = incl; s_last[warp] = lmax; }
    __syncthreads();
    int base = 0, cta_total = 0;
    long long before = -1, cta_last = -1;          // last change in the warps before mine / in this CTA
    for (int k = 0; k < RLE_THREADS / 32; ++k) {
        if (k < warp) { base += s_cnt[k]; before = max(before, s_last[k]); }
        cta_total += s_cnt[k];
        cta_last = max(cta_last, s_last[k]);
    }
    if (tid == 0) { s_cta_cnt = cta_total; s_cta_last = cta_last; }
    cluster.sync();
    int total = 0;
    long long last_all = -1;
#pragma unroll
    for (int c = 0; c < RLE_CLUSTER; ++c) {
        const int tc = *cluster.map_shared_rank(&s_cta_cnt, c);
        const long long lc = *cluster.map_shared_rank(&s_cta_last, c);
        if (c < crank) { base += tc; before = max(before, lc); }
        total += tc;
        last_all = max(last_all, lc);
    }
    cluster.sync();                                // nobody leaves while its totals may still be read
    const int off = base + incl - cnt;
    long long prev_change = __shfl_up_sync(0xffffffffu, lmax, 1);        // last change in the lanes before mine
    if (lane == 0) prev_change = -1;
    prev_change = max(prev_change, before);
    // ---- pass 2: counts.  counts[k] = position of change k - position of change k-1 (0 for k = 0); the final
    // run closes the mask: counts[total] = a - last change
    const int m = total + 1;
    if (m <= cap) {
        int k = off;
        long long pc = prev_change < 0 ? 0 : prev_change;
        walk([&](long long j) { out[k++] = (unsigned)(j - pc); pc = j; });
        if (crank == 0 && tid == 0) out[total] = (unsigned)(a - (last_all < 0 ? 0 : last_all));
    }
    if (crank == 0 && tid == 0) m_out[mask_id] = m <= cap ? m : -m;
}


// ---------------------------------------------------------------------------
// Coalesced form (16-byte aligned masks, a % 16 == 0 -- the 1024^2 planes): a warp owns a contiguous span of the mask
// and reads it 512 bytes per instruction (lane = 16 consecutive bytes), so every 128-byte line is fetched once per pass
// instead of 16 bytes at a time by 8 different instructions (the chunk-per-thread form above moves 2-3x the mask through
// L2).  The scan unit is the warp: changes are counted per 16-byte piece as a 16-bit mask, the running output index and
// the position of the previous change are warp-uniform, and a warp-wide prefix (sum of counts, maximum of last change
// positions) is only taken for the 512-byte steps that contain a change at all.
// ---------------------------------------------------------------------------
__device__ __forceinline__ unsigned piece_changes(const uint4 v, unsigned prev_byte)
{
    const unsigned w[4] = {v.x, v.y, v.z, v.w};
    const unsigned d[4] = {w[0] ^ ((w[0] << 8) | prev_byte), w[1] ^ ((w[1] << 8) | (w[0] >> 24)),
                           w[2] ^ ((w[2] << 8) | (w[1] >> 24)), w[3] ^ ((w[3] << 8) | (w[2] >> 24))};
    if ((d[0] | d[1] | d[2] | d[3]) == 0u) return 0u;
    unsigned cm = 0u;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const unsigned ch = __vcmpne4(d[q], 0u) & 0x01010101u;          // bit 8b <=> byte b differs from the one before
        cm |= (((ch * 0x01020408u) >> 24) & 0xfu) << (4 * q);           // -> 4 adjacent bits
    }
    return cm;                                                          // bit b <=> change at byte b of the piece
}

// 512 threads and <= 32 registers: four CTAs per SM.  (The 1024-thread form above needs 38-40 registers, i.e. ONE CTA per
// SM, and a cluster of 8 needs 8 SMs of one GPC: 16 clusters at a time on 128 of the 148 SMs, 6 waves for 100 masks --
// that, not the access pattern, is what held both forms at ~110 us.)
constexpr int RLEC_THREADS = 512;
#ifndef SLN_RLEC_CTAS
#define SLN_RLEC_CTAS 4
#endif
constexpr int RLEC_CTAS_PER_SM = SLN_RLEC_CTAS;

__global__ void __cluster_dims__(RLE_CLUSTER, 1, 1) __launch_bounds__(RLEC_THREADS, RLEC_CTAS_PER_SM)
rle_encode_coalesced_kernel(const unsigned char *__restrict__ masks, long long a, unsigned *__restrict__ counts, int cap,
                            int *__restrict__ m_out)
{
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    constexpr unsigned FULL = 0xffffffffu;
    __shared__ int s_cnt[RLEC_THREADS / 32];
    __shared__ unsigned s_last[RLEC_THREADS / 32];  // last change position + 1 (0: none)
    __shared__ int s_cta_cnt;                      // read by the whole cluster
    __shared__ unsigned s_cta_last;
    const int mask_id = blockIdx.x / RLE_CLUSTER, crank = (int)cluster.block_rank();
    const unsigned char *T = masks + (size_t)mask_id * a;
    unsigned *out = counts + (size_t)mask_id * cap;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int WARPS = RLE_CLUSTER * (RLEC_THREADS / 32);
    long long span = (a + WARPS - 1) / WARPS;
    span = (span + 511) & ~511ll;                  // whole 512-byte steps
    const long long w0 = min(a, ((long long)crank * (RLEC_THREADS / 32) + warp) * span), w1 = min(a, w0 + span);
    const unsigned carry0 = (w0 > 0 && w0 < a) ? T[w0 - 1] : 0u;

    // ---- pass 1: changes of this warp's span, last change position
    int cnt = 0;
    unsigned lastp1 = 0u;
    {
        unsigned carry = carry0;
        for (long long p0 = w0; p0 < w1; p0 += 512) {
            const long long p = p0 + 16 * lane;
            const bool ok = p < w1;
            const uint4 v = ok ? __ldg(reinterpret_cast<const uint4 *>(T + p)) : make_uint4(0, 0, 0, 0);
            const unsigned lastb = v.w >> 24;
            unsigned pb = __shfl_up_sync(FULL, lastb, 1);
            if (lane == 0) pb = carry;
            carry = __shfl_sync(FULL, lastb, 31);
            const unsigned cm = ok ? piece_changes(v, pb) : 0u;
            if (cm) {
                cnt += __popc(cm);
                lastp1 = (unsigned)p + (31 - __clz(cm)) + 1u;
            }
        }
    }
    for (int o = 16; o; o >>= 1) {
        cnt += __shfl_xor_sync(FULL, cnt, o);
        lastp1 = max(lastp1, __shfl_xor_sync(FULL, lastp1, o));
    }
    if (lane == 0) { s_cnt[warp] = cnt; s_last[warp] = lastp1; }
    __syncthreads();
    int base = 0, cta_total = 0;
    unsigned before = 0u, cta_last = 0u;           // last change (+1) in the warps before mine / in this CTA
    for (int k = 0; k < RLEC_THREADS / 32; ++k) {
        if (k < warp) { base += s_cnt[k]; before = max(before, s_last[k]); }
        cta_total += s_cnt[k];
        cta_last = max(cta_last, s_last[k]);
    }
    if (tid == 0) { s_cta_cnt = cta_total; s_cta_last = cta_last; }
    cluster.sync();
    int total = 0;
    unsigned last_all = 0u;
#pragma unroll
    for (int c = 0; c < RLE_CLUSTER; ++c) {
        const int tc = *cluster.map_shared_rank(&s_cta_cnt, c);
        const unsigned lc = *cluster.map_shared_rank(&s_cta_last, c);
        if (c < crank) { base += tc; before = max(before, lc); }
        total += tc;
        last_all = max(last_all, lc);
    }
    cluster.sync();                                // nobody leaves while its totals may still be read
    // ---- pass 2: counts[k] = position of change k - position of change k-1 (0 for k = 0); counts[total] closes the mask
    const int m = total + 1;
    if (m <= cap && cnt > 0) {
        int k = base;                              // warp-uniform: index of the next change
        unsigned pc1 = before;                     // warp-uniform: previous change position + 1 (0: none)
        unsigned carry = carry0;
        for (long long p0 = w0; p0 < w1; p0 += 512) {
            const long long p = p0 + 16 * lane;
            const bool ok = p < w1;
            const uint4 v = ok ? __ldg(reinterpret_cast<const uint4 *>(T + p)) : make_uint4(0, 0, 0, 0);
            const unsigned lastb = v.w >> 24;
            unsigned pb = __shfl_up_sync(FULL, lastb, 1);
            if (lane == 0) pb = carry;
            carry = __shfl_sync(FULL, lastb, 31);
            unsigned cm = ok ? piece_changes(v, pb) : 0u;
            if (!__any_sync(FULL, cm != 0u)) continue;
            const int c = __popc(cm);
            int incl = c;
            unsigned lmax = cm ? (unsigned)p + (31 - __clz(cm)) + 1u : 0u;
            for (int o = 1; o < 32; o <<= 1) {
                const int vi = __shfl_up_sync(FULL, incl, o);
                const unsigned vl = __shfl_up_sync(FULL, lmax, o);
                if (lane >= o) { incl += vi; lmax = max(lmax, vl); }
            }
            unsigned prev1 = __shfl_up_sync(FULL, lmax, 1);             // last change (+1) in the lanes before mine
            if (lane == 0) prev1 = 0u;
            prev1 = max(prev1, pc1);
            int kk = k + incl - c;
            unsigned pos_prev = prev1 ? prev1 - 1u : 0u;
            while (cm) {
                const unsigned j = (unsigned)p + (__ffs(cm) - 1);
                cm &= cm - 1;
                out[kk++] = j - pos_prev;
                pos_prev = j;
            }
            k += __shfl_sync(FULL, incl, 31);
            pc1 = max(pc1, __shfl_sync(FULL, lmax, 31));
        }
    }
    if (crank == 0 && tid == 0) {
        if (m <= cap) out[total] = (unsigned)(a - (last_all ? (long long)last_all - 1 : 0));
        m_out[mask_id] = m <= cap ? m : -m;
    }
}

// ---------------------------------------------------------------------------
// Runs from a box-sized mask (sln_unmold_rle_batched).  The column-major H x W plane that pycocotools encodes is zero
// outside the box, so its value changes lie in the box's column segments [x*H + y1, x*H + y2) or right after them.  A
// segment's first pixel is compared with 0, except in a full-height box (y1 == 0, y2 == H) past its first column:
// there the plane runs straight on from the previous column's last box pixel (the box is one contiguous stretch of the
// plane).  After a segment the plane is 0 again, so a set last pixel makes a change one past it, unless the next
// column's segment follows at once (full height) or the plane ends there.  The final run closes at a = H*W.
// One CTA per detection; each thread takes a contiguous chunk of the bh*bw box bytes, in two passes like
// rle_encode_kernel (count, block scan, write).  The string length of maskApi.c's rleToString is added up at the end.
// ---------------------------------------------------------------------------
constexpr int RLEB_THREADS = 256;

// characters rleToString spends on one delta x (maskApi.c:204-216): 5 bits per char until the rest is the sign
__device__ __forceinline__ int rle_chars(long long x)
{
    int n = 0;
    bool more = true;
    while (more) {
        const int c = (int)(x & 0x1f);
        x >>= 5;
        more = (c & 0x10) ? x != -1 : x != 0;
        ++n;
    }
    return n;
}

__device__ __forceinline__ void rle_put(long long x, char *o)
{
    bool more = true;
    while (more) {
        char c = (char)(x & 0x1f);
        x >>= 5;
        more = (c & 0x10) ? x != -1 : x != 0;
        if (more) c |= 0x20;
        *o++ = (char)(c + 48);
    }
}

// maskApi.c's delta: counts[k] against counts[k-2], from k = 3 on (sic: `if (i > 2)`)
__device__ __forceinline__ long long rle_delta(const uint32_t *c, int k)
{
    long long x = (long long)c[k];
    if (k > 2) x -= (long long)c[k - 2];
    return x;
}

template <int THREADS>
__device__ __forceinline__ int block_string_length(const uint32_t *c, int m, int *warp_tot)
{
    int n = 0;
    for (int k = threadIdx.x; k < m; k += THREADS) n += rle_chars(rle_delta(c, k));
    int total;
    block_excl_sum<THREADS>(n, warp_tot, &total);
    return total;
}

__global__ void __launch_bounds__(RLEB_THREADS)
rle_box_kernel(const BoxRow *__restrict__ rows, const int *__restrict__ nk, int D, const uint8_t *__restrict__ maskbuf,
               uint32_t *__restrict__ counts, int cap, int *__restrict__ m_out, int *__restrict__ str_len)
{
    __shared__ int s_cnt[RLEB_THREADS / 32];
    __shared__ long long s_last[RLEB_THREADS / 32];
    const int row = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = row / D;
    if (row - b * D >= nk[b]) {
        if (tid == 0) { m_out[row] = 0; str_len[row] = 0; }
        return;
    }
    const BoxRow R = rows[row];
    const long long H = R.H, a = H * R.W, area = (long long)R.bh * R.bw;
    const uint8_t *T = maskbuf + R.off;
    uint32_t *out = counts + (size_t)row * cap;
    const bool merge = R.y1 == 0 && R.bh == R.H;
    const long long len = (area + RLEB_THREADS - 1) / RLEB_THREADS;
    const long long i0 = min(area, tid * len), i1 = min(area, i0 + len);

    auto walk = [&](auto &&on_change) {
        if (i0 >= i1) return;
        int c = (int)(i0 / R.bh), r = (int)(i0 - (long long)c * R.bh);
        long long col = (long long)(R.x1 + c) * H + R.y1;      // plane position of box row 0 of column c
        unsigned prev = (r > 0 || (merge && i0 > 0)) ? T[i0 - 1] : 0u;
        for (long long i = i0; i < i1; ++i) {
            const unsigned v = T[i];
            if (v != prev) on_change(col + r);
            if (r == R.bh - 1) {
                if (v && (!merge || c == R.bw - 1) && col + r + 1 < a) on_change(col + r + 1);
                ++c;
                r = 0;
                col += H;
                prev = merge ? v : 0u;
            } else {
                ++r;
                prev = v;
            }
        }
    };

    // ---- pass 1: count, remember the last change; then the exclusive count and the last change before each thread
    int cnt = 0;
    long long last = -1;
    walk([&](long long j) { ++cnt; last = j; });
    long long lmax = last;
    for (int o = 1; o < 32; o <<= 1) {
        const long long l = __shfl_up_sync(0xffffffffu, lmax, o);
        if (lane >= o) lmax = max(lmax, l);
    }
    if (lane == 31) s_last[warp] = lmax;
    int total;
    const int off = block_excl_sum<RLEB_THREADS>(cnt, s_cnt, &total);   // its barriers publish s_last too
    long long before = -1, last_all = -1;
    for (int w = 0; w < RLEB_THREADS / 32; ++w) {
        if (w < warp) before = max(before, s_last[w]);
        last_all = max(last_all, s_last[w]);
    }
    long long prev_change = __shfl_up_sync(0xffffffffu, lmax, 1);
    if (lane == 0) prev_change = -1;
    prev_change = max(prev_change, before);
    // ---- pass 2: counts[k] = change k - change k-1 (the first from 0); counts[total] closes the plane
    const int m = total + 1;
    if (m <= cap) {
        int k = off;
        long long pc = prev_change < 0 ? 0 : prev_change;
        walk([&](long long j) { out[k++] = (uint32_t)(j - pc); pc = j; });
        if (tid == 0) out[total] = (uint32_t)(a - (last_all < 0 ? 0 : last_all));
    }
    __syncthreads();                                   // the counts are read back below by other threads
    const int slen = m <= cap ? block_string_length<RLEB_THREADS>(out, m, s_cnt) : 0;
    if (tid == 0) {
        m_out[row] = m <= cap ? m : -m;
        str_len[row] = slen;
    }
}

// ---------------------------------------------------------------------------
// Device string coder: rleToString (maskApi.c:204-216) for n count lists, packed into one buffer.  The characters of
// counts[k] depend only on counts[k] and counts[k-2], so a mask's string is per-count lengths, a scan and the writes;
// the masks' strings follow one another in mask order (a scan over the n lengths).  Byte for byte what the host
// helper sln_rle_to_string writes, without its terminating 0.
// ---------------------------------------------------------------------------
constexpr int STR_THREADS = 256;
constexpr int STR_SCAN_THREADS = 1024;

__global__ void __launch_bounds__(STR_THREADS)
rle_str_len_kernel(const uint32_t *__restrict__ counts, int cap, const int *__restrict__ m, int *__restrict__ str_len)
{
    __shared__ int s_w[STR_THREADS / 32];
    const int i = blockIdx.x, mi = m[i];
    const int len = (mi > 0 && mi <= cap) ? block_string_length<STR_THREADS>(counts + (size_t)i * cap, mi, s_w) : 0;
    if (threadIdx.x == 0) str_len[i] = len;
}

__global__ void __launch_bounds__(STR_SCAN_THREADS)
rle_str_scan_kernel(const int *__restrict__ str_len, int n, int *__restrict__ str_off, int *__restrict__ str_total)
{
    __shared__ int s_w[STR_SCAN_THREADS / 32];
    int run = 0;
    for (int c0 = 0; c0 < n; c0 += STR_SCAN_THREADS) {
        const int i = c0 + threadIdx.x;
        const int v = i < n ? str_len[i] : 0;
        int t;
        const int e = block_excl_sum<STR_SCAN_THREADS>(v, s_w, &t);
        if (i < n) str_off[i] = run + e;
        run += t;
    }
    if (threadIdx.x == 0) *str_total = run;
}

__global__ void __launch_bounds__(STR_THREADS)
rle_str_write_kernel(const uint32_t *__restrict__ counts, int cap, const int *__restrict__ m,
                     const int *__restrict__ str_off, const int *__restrict__ str_len, char *__restrict__ strings)
{
    __shared__ int s_w[STR_THREADS / 32];
    const int i = blockIdx.x;
    if (str_len[i] == 0) return;
    const int mi = m[i];
    const uint32_t *c = counts + (size_t)i * cap;
    char *o = strings + str_off[i];
    int run = 0;
    for (int k0 = 0; k0 < mi; k0 += STR_THREADS) {
        const int k = k0 + threadIdx.x;
        const long long x = k < mi ? rle_delta(c, k) : 0;
        int t;
        const int e = block_excl_sum<STR_THREADS>(k < mi ? rle_chars(x) : 0, s_w, &t);
        if (k < mi) rle_put(x, o + run + e);
        run += t;
    }
}

int launch_rle_boxes(const BoxRow *rows, const int *nk, int B, int D, const uint8_t *maskbuf, uint32_t *counts, int cap,
                     int *m_out, int *str_len, cudaStream_t st)
{
    rle_box_kernel<<<B * D, RLEB_THREADS, 0, st>>>(rows, nk, D, maskbuf, counts, cap, m_out, str_len);
    SLN_LAUNCH_OK("rle_box_kernel");
    return SLN_OK;
}

int launch_rle_strings(const uint32_t *counts, int n, int cap, const int *m, const int *str_len, int *str_off,
                       int *str_total, char *strings, cudaStream_t st)
{
    rle_str_scan_kernel<<<1, STR_SCAN_THREADS, 0, st>>>(str_len, n, str_off, str_total);
    SLN_LAUNCH_OK("rle_str_scan_kernel");
    rle_str_write_kernel<<<n, STR_THREADS, 0, st>>>(counts, cap, m, str_off, str_len, strings);
    SLN_LAUNCH_OK("rle_str_write_kernel");
    return SLN_OK;
}

}  // namespace sln

extern "C" int sln_rle_encode(const uint8_t *masks, int n, long long a, uint32_t *counts, int cap, int *m_out, void *stream)
{
    SLN_REQUIRE(n >= 0 && a >= 0 && cap >= 1, SLN_ERR_ARG, "bad size");
    SLN_REQUIRE(a < (1ll << 32), SLN_ERR_ARG, "mask too large for 32-bit run lengths");
    SLN_REQUIRE((long long)n * sln::RLE_CLUSTER < (1ll << 31), SLN_ERR_ARG, "too many masks");
    if (n == 0) return SLN_OK;
    SLN_REQUIRE(masks != nullptr || a == 0, SLN_ERR_ARG, "null masks");
    SLN_REQUIRE(counts && m_out, SLN_ERR_ARG, "null pointer");
    const char *e = getenv("SLN_RLE_CHUNKED");                         // A/B: the chunk-per-thread form for every shape
    const bool coalesced = (a % 16 == 0) && ((reinterpret_cast<uintptr_t>(masks) & 15u) == 0) && !(e && e[0] == '1');
    if (coalesced)
        sln::rle_encode_coalesced_kernel<<<n * sln::RLE_CLUSTER, sln::RLEC_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(masks, a, counts, cap, m_out);
    else
        sln::rle_encode_kernel<<<n * sln::RLE_CLUSTER, sln::RLE_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(masks, a, counts, cap, m_out);
    SLN_LAUNCH_OK("rle_encode_kernel");
    return SLN_OK;
}

// Host helper (no CUDA): maskApi.c:204-216.  Returns the string length (without the terminating 0), or the required
// capacity negated when `cap` is too small.
extern "C" long long sln_rle_to_string(const uint32_t *counts, long long m, char *out, long long cap)
{
    long long p = 0;
    for (long long i = 0; i < m; ++i) {
        long long x = (long long)counts[i];
        if (i > 2) x -= (long long)counts[i - 2];
        int more = 1;
        while (more) {
            char c = (char)(x & 0x1f);
            x >>= 5;
            more = (c & 0x10) ? x != -1 : x != 0;
            if (more) c |= 0x20;
            c += 48;
            if (p < cap) out[p] = c;
            ++p;
        }
    }
    if (p < cap) out[p] = 0;
    return p < cap ? p : -(p + 1);
}

extern "C" int sln_rle_strings(const uint32_t *counts, int n, int cap, const int *m, int *str_off, int *str_len,
                               int *str_total, char *strings, long long strings_cap, void *stream)
{
    SLN_REQUIRE(n >= 0 && cap >= 1, SLN_ERR_ARG, "rle_strings: bad n / cap");
    SLN_REQUIRE(strings_cap >= 7ll * cap * n && strings_cap < (1ll << 31), SLN_ERR_ARG,
                "rle_strings: strings_cap must be >= 7 * cap * n and < 2^31 (got %lld)", strings_cap);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    SLN_REQUIRE(str_total, SLN_ERR_ARG, "rle_strings: null pointer");
    if (n == 0) {
        SLN_CUDA_OK(cudaMemsetAsync(str_total, 0, sizeof(int), st));
        return SLN_OK;
    }
    SLN_REQUIRE(counts && m && str_off && str_len && strings, SLN_ERR_ARG, "rle_strings: null pointer");
    sln::rle_str_len_kernel<<<n, sln::STR_THREADS, 0, st>>>(counts, cap, m, str_len);
    SLN_LAUNCH_OK("rle_str_len_kernel");
    return sln::launch_rle_strings(counts, n, cap, m, str_len, str_off, str_total, strings, st);
}
