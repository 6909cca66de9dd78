// crop_bwd_tma.cuh -- RoIAlign backward, persistent bulk-async ("TMA") form.  Included by crop.cu inside namespace sln.
//
// Reference semantics: roialign/roi_align/src/crop_and_resize.c:157-252 (serial scatter, order (box, y, x, tap));
// GPU baseline being replaced: cuda/crop_and_resize_kernel.cu:84-165 (atomicAdd scatter).
//
// Why another form: the strip kernel (crop.cu) spends ~7 warp instructions on search and addressing
// per useful FMA and stall on every gradient load (ncu, round 1: 389 M warp instructions for 50 M warp-FMAs at 14x14,
// 48 % of the stall samples on the first FMA after the loads).  Here the search, the data movement and the arithmetic
// are three decoupled agents of a persistent CTA (two CTAs per SM, each walking tiles blockIdx.x, + gridDim.x, ...):
//   * one PRODUCER warp does all the search.  Per 8x8 pixel tile it walks the supertile's ordered ROI list, intersects
//     each ROI's tap tables (one tap per lane) with the tile, and cuts the hit -- the sub-rectangle of the crop whose
//     samples reach the tile -- into STAGES of up to STG_S samples (whole sample rows).  A stage is a descriptor
//     (per tile row the range of stage rows that reach it; per stage row its top tile row and lerp; per sample column
//     the tile column of its left tap and its lerp) plus the gradient vectors themselves, fetched by cp.async.bulk
//     (one per sample row: n * C * sizeof(T) contiguous bytes; SASS UBLKCP) into a ring of shared-memory stages.  An mbarrier
//     per stage counts the bytes in (complete_tx); a second one counts the eight consumers out.  The producer runs
//     ahead of the consumers by the depth of the ring, across tile boundaries: the list heads of the next two tiles and
//     the tap tables of the next ROI are in flight while the current ROI is planned.
//   * eight CONSUMER warps own one pixel row of the tile each, with the row's accumulators (8 pixels x C channels) in
//     registers.  For every stage a consumer waits once, looks up its row range, reads each staged vector of those rows
//     from shared memory once and applies both x taps with a warp-uniform switch on the tap's tile column.  No ballots,
//     no shuffles, no global loads, no search.  An end-of-tile stage makes it write its row -- every output pixel exactly
//     once, zeros included (no memset, no atomics) -- and clear the accumulators.
// Every consumer takes part in every stage, so a parity wait can never be more than one phase behind (no ABA).
// Per destination pixel the terms are added in the reference's order (ROI, y, x, tap TL/TR/BL/BR): stages are issued in
// (ROI, sy) order, samples inside a stage row ascend in sx, and a pixel row belongs to one warp.  EXACT = the reference's
// rounding sequence wx*(wy*g) per term, incl. the zero-weight taps of integral sample positions (bit-identical to
// crop_and_resize.c); otherwise one fma per term with the fused weight wy*wx.
#pragma once

namespace bwdtma {

constexpr int TH = 8;                  // tile rows = consumer warps
constexpr int TW = 8;                  // tile columns = accumulator pixels per consumer lane
constexpr int NCONS = TH;
constexpr int THREADS = 32 * (NCONS + 1);
constexpr int MAX_POOL = 32;           // one sample row / column per lane
constexpr int CH_MAX = 256;            // channels per CTA (two float4 per consumer lane)
// Per launch configuration (template parameters of the kernel): STG_S samples per stage (and at most as many rows /
// sample columns), 8 .. 32; NST stages in the ring.  Shared memory allows STG_S * NST = 96 KB per CTA at two CTAs per SM.
// Measured on B200 (8 x 1000 ROIs, C = 256, ms per call incl. prep; A/B in profiles/README.md): 7x7 prefers 16 x 6
// (0.309 against 0.318 for 32 x 3), 14x14 and 16x16 prefer 32 x 3 (0.497 / 0.578 against 0.510 / 0.599).

struct XEnt {
    int pl;          // tile column of the left tap (-1 .. 7)
    float xl;        // lerp
};
enum { ST_DATA = 0, ST_TILE_END = 1, ST_EXIT = 2 };
template <int STG_S>
struct StageDesc {
    int flags;       // ST_*
    int n_s;         // ST_DATA: samples per stage row.  ST_TILE_END: channels of the work item
    int n_rows;
    int chb;         // bytes per staged sample (channels of the work item * 4)
    int2 rows[TH];   // ST_TILE_END: the write-out record (TileOut)
    int2 rowd[STG_S];   // per stage row: (tile row of its top tap, -1 .. 7; lerp bits)
    XEnt x[STG_S];      // per sample column of the stage
};
struct TileOut {     // overlays StageDesc::rows for ST_TILE_END
    unsigned long long out;   // address of pixel (b, y0, x0), channel c0
    int row_stride;           // 16-byte vectors per map row
    int pix_stride;           // 16-byte vectors per pixel
    int ny, nx;               // valid rows / columns of the tile
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// try_wait suspends the thread in hardware for a bounded time, so the loop does not spin on the issue port
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "SLN_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra SLN_DONE;\n"
        "bra SLN_WAIT;\n"
        "SLN_DONE:\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}
// global -> shared bulk copy (SASS UBLKCP); completion is counted in bytes on `bar`
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}

template <bool EXACT>
__device__ __forceinline__ float4 term(float4 a, float4 g, float w, float wy, float wx)
{
    if (EXACT) {   // crop_and_resize.c:241-247: image += wx * (wy * g), every operation rounded
        return make_float4(__fadd_rn(a.x, __fmul_rn(wx, __fmul_rn(wy, g.x))), __fadd_rn(a.y, __fmul_rn(wx, __fmul_rn(wy, g.y))),
                           __fadd_rn(a.z, __fmul_rn(wx, __fmul_rn(wy, g.z))), __fadd_rn(a.w, __fmul_rn(wx, __fmul_rn(wy, g.w))));
    }
    // one fma per component, two components per instruction (FFMA2: each half rounded like the scalar fma)
    const f32x2_t ww = pk2(w, w);
    float4 r;
    unpk2(fma2_rn(ww, pk2(g.x, g.y), pk2(a.x, a.y)), r.x, r.y);
    unpk2(fma2_rn(ww, pk2(g.z, g.w), pk2(a.z, a.w)), r.z, r.w);
    return r;
}

// acc[K] += weight * g for a warp-uniform, run-time K: a switch over statically indexed registers
#define SLN_TMA_ADD(K, W, WY, WX)                                                  \
    {                                                                              \
        acc[K][0] = term<EXACT>(acc[K][0], g0, W, WY, WX);                         \
        if (NACC == 2) acc[K][1] = term<EXACT>(acc[K][1], g1, W, WY, WX);          \
    }

// The run [k0, k0 + n) of sample indices k in [0, crop) whose position pos(k) = base + k * scale (rounded exactly like
// tap_at / crop_and_resize.c:44-56) is inside the map, [0, extent - 1], and has floor(pos) <= t1 and ceil(pos) >= t0, i.e.
// whose taps reach pixel rows (columns) t0 .. t1.  pos is monotone in k, so the set is a run; its ends come from a
// division and are then corrected against the exact predicate, so rounding in the estimate cannot change the result.
__device__ __forceinline__ void sample_run(float base, float scale, float em1, int crop, int t0, int t1, int extent,
                                           int &k0, int &n)
{
    // above(k): pos is past the lower bound; below(k): pos is before the upper bound
    const float lo_b = (float)(t0 - 1), hi_b = (float)(t1 + 1);
    const bool lo_closed = t0 == 0, hi_closed = t1 == extent - 1;       // bounds 0 / extent - 1 are inclusive
    auto pos = [&](int k) { return __fadd_rn(base, __fmul_rn((float)k, scale)); };
    auto above = [&](int k) { const float p = pos(k); return lo_closed ? p >= 0.f : p > lo_b; };
    auto below = [&](int k) { const float p = pos(k); return hi_closed ? p <= em1 : p < hi_b; };
    k0 = 0;
    n = 0;
    if (scale == 0.f || crop == 1) {
        if (above(0) && below(0)) n = crop;
        return;
    }
    // first k where a predicate that is monotone false -> true turns true (crop if never)
    auto first_true = [&](float bound, bool want_above) {
        int k = __float2int_rd(__fdiv_rn(__fsub_rn(bound, base), scale));
        k = max(0, min(crop, k));
        if (want_above) {
            while (k > 0 && above(k - 1)) --k;
            while (k < crop && !above(k)) ++k;
        } else {
            while (k > 0 && !below(k - 1)) --k;
            while (k < crop && below(k)) ++k;
        }
        return k;
    };
    int a, b;
    if (scale > 0.f) {          // pos increasing: [first above, first not-below)
        a = first_true(lo_closed ? 0.f : lo_b, true);
        b = first_true(hi_closed ? em1 : hi_b, false);
    } else {                    // pos decreasing: [first below, first not-above)
        // mirrored predicates: below is false -> true, above is true -> false
        int k = __float2int_rd(__fdiv_rn(__fsub_rn(hi_closed ? em1 : hi_b, base), scale));
        k = max(0, min(crop, k));
        while (k > 0 && below(k - 1)) --k;
        while (k < crop && !below(k)) ++k;
        a = k;
        k = __float2int_rd(__fdiv_rn(__fsub_rn(lo_closed ? 0.f : lo_b, base), scale));
        k = max(0, min(crop, k));
        while (k > 0 && !above(k - 1)) --k;
        while (k < crop && above(k)) ++k;
        b = k;
    }
    if (b > a) { k0 = a; n = b - a; }
}

// whole sample rows of nsx samples that fit a stage of STG_S samples (1 for longer rows: they take several stages).
// STG_S / nsx without the integer divide (~25 dependent instructions): floor((STG_S + 0.5) / nsx) is exact for
// 1 <= nsx <= STG_S <= 32 under the approximate divide's 2 ulp.
template <int STG_S>
__device__ __forceinline__ int rows_per_stage(int nsx)
{
    return nsx <= STG_S ? __float2int_rz(__fdividef((float)STG_S + 0.5f, (float)nsx)) : 1;
}

struct TileGeom {
    int l, b, y0, x0, y1, x1, c0, st;
};

// work item w -> (tile, channel chunk) -> level / image / tile origin / supertile.  lv: level table in shared memory.
__device__ __forceinline__ TileGeom tile_geom(int w, int chunks, const BwdTileBases &TB, const BwdLevel *lv)
{
    TileGeom g;
    const int tile = w / chunks;
    g.c0 = (w - tile * chunks) * CH_MAX;
    int l = TB.lvl[0];
#pragma unroll
    for (int k = 1; k < BWD_MAX_LEVELS; ++k)
        if (k < TB.n_levels && tile >= TB.base[k]) l = TB.lvl[k];
    g.l = l;
    const BwdLevel &L = lv[l];
    const int t = tile - L.tile_base;
    const int q1 = fast_div(t, L.tiles_x, L.rcp_tiles_x);
    const int tx_i = t - q1 * L.tiles_x;
    g.b = fast_div(q1, L.tiles_y, L.rcp_tiles_y);
    const int ty_i = q1 - g.b * L.tiles_y;
    g.y0 = ty_i * TH;
    g.x0 = tx_i * TW;
    g.y1 = min(g.y0 + TH, L.H) - 1;
    g.x1 = min(g.x0 + TW, L.W) - 1;
    g.st = L.st_base + (g.b * L.sg.ny + (g.y0 >> L.sg_shift)) * L.sg.nx + (g.x0 >> L.sg_shift);
    return g;
}

// T: element type of grads and grad maps -- float, or a 2-byte type (__nv_bfloat16 / __half) that the consumers widen on
// the shared-memory read and round once on the write; the accumulators and their arithmetic are fp32 either way.
// NV: 16-byte vectors per consumer lane (fp32: 1 or 2, i.e. 4 or 8 channels; 2-byte types: 1, i.e. 8 channels).
// FULL: the CTA's channel chunk fills every lane's vectors (CH == 32 * NV * 16 / sizeof(T)), so no lane predicates.
// The kernels are the two __global__ wrappers below: crop_bwd_tma_kernel (f32) and crop_bwd_tma_b16_kernel (2-byte types).
template <typename T, int NV, bool EXACT, bool FULL, int STG_S, int NST>
__device__ __forceinline__ void
crop_bwd_tma_body(const T *__restrict__ grads, const ListEntryA *__restrict__ entries, const int *__restrict__ st_off,
                  const int *__restrict__ st_count, const BwdLevel *__restrict__ lv_table,
                  BwdTileBases TB, int C, int ph, int pw, int n_work, int chunks, int *__restrict__ queue)
{
    extern __shared__ __align__(128) unsigned char s_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    static_assert(STG_S >= 8 && STG_S <= 32, "a consumer finds its sample columns with one 32-lane ballot");
    constexpr int ESZ = sizeof(T);
    constexpr int VPV = 16 / ESZ;                         // elements per 16-byte vector
    constexpr int NACC = ESZ == 4 ? NV : 2;               // float4 accumulators per pixel and lane
    static_assert(ESZ == 4 || NV == 1, "2-byte elements: one 16-byte vector (8 channels) per lane");
    constexpr int STAGE_BYTES = STG_S * CH_MAX * ESZ;
    using Desc = StageDesc<STG_S>;
    // ---- shared memory carve-up
    unsigned char *stages = s_raw;                                                    // [NST][STAGE_BYTES]
    Desc *sdesc = reinterpret_cast<Desc *>(s_raw + (size_t)NST * STAGE_BYTES);
    BwdLevel *lv = reinterpret_cast<BwdLevel *>(sdesc + NST);
    uint64_t *bars = reinterpret_cast<uint64_t *>(lv + BWD_MAX_LEVELS);
    const uint32_t full0 = smem_u32(bars), empty0 = full0 + 8 * NST;
    asm volatile("griddepcontrol.launch_dependents;");
    if (threadIdx.x == 0) {
        for (int i = 0; i < NST; ++i) {
            mbar_init(full0 + 8 * i, 1);                   // the producer's arrive(.expect_tx) (+ the bytes)
            mbar_init(empty0 + 8 * i, NCONS);              // every consumer releases every stage
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    // everything below reads what the prep launches wrote (level table, lists, ticket counter): wait for them here
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (threadIdx.x < BWD_MAX_LEVELS) lv[threadIdx.x] = lv_table[threadIdx.x];
    __syncthreads();

    if (warp == NCONS) {
        // =========================================================== producer
        const int S = ph * pw;
        unsigned slot = 0, epar = 1;                       // ring slot of the next stage; parity that marks it released
        auto acquire = [&]() -> unsigned {                 // next ring stage, released by all consumers
            mbar_wait(empty0 + 8 * slot, epar);
            return slot;
        };
        auto advance = [&]() {                             // (no % and / by NST on the per-stage chain)
            if (++slot == NST) {
                slot = 0;
                epar ^= 1u;
            }
        };
        auto no_entry = []() {
            ListEntryA e;
            e.roi = -1;
            e.pad = 0;
            e.win.y0 = e.win.x0 = 1;
            e.win.y1 = e.win.x1 = 0;
            e.ax.by = e.ax.sy = e.ax.bx = e.ax.sx = 0.f;
            return e;
        };
        // tile pipeline: work items come from a global ticket counter (heaviest levels first, so the light P2 tiles fill
        // the tail); while item C is planned, the first list chunk of item B, the list count / offset of item A and the
        // ticket of the item after that are in flight.  Tickets 0 .. gridDim.x - 1 are the CTAs' first items.
        auto ticket = [&]() -> int {
            int t = 0;
            if (lane == 0) t = atomicAdd(queue, 1);
            return t;                                      // lane 0 only; broadcast when it is needed
        };
        int wC = blockIdx.x;
        int wB = __shfl_sync(0xffffffffu, ticket(), 0), wA = __shfl_sync(0xffffffffu, ticket(), 0);
        int cntC = 0, offC = 0, cntB = 0, offB = 0;
        TileGeom gC{}, gB{};
        ListEntryA eC = no_entry();
        if (wC < n_work) {
            gC = tile_geom(wC, chunks, TB, lv);
            cntC = st_count[gC.st];
            offC = st_off[gC.st];
            if (lane < cntC) eC = entries[offC + lane];
        }
        if (wB < n_work) {
            gB = tile_geom(wB, chunks, TB, lv);
            cntB = st_count[gB.st];
            offB = st_off[gB.st];
        }
        while (wC < n_work) {
            const int tF = ticket();
            ListEntryA eB = no_entry();
            if (wB < n_work && lane < cntB) eB = entries[offB + lane];
            int cntA = 0, offA = 0;
            TileGeom gA{};
            if (wA < n_work) {
                gA = tile_geom(wA, chunks, TB, lv);
                cntA = st_count[gA.st];
                offA = st_off[gA.st];                      // written for every supertile, also the empty ones
            }

            const BwdLevel &L = lv[gC.l];
            const int y0 = gC.y0, x0 = gC.x0, y1 = gC.y1, x1 = gC.x1, c0 = gC.c0;
            const int CH = min(C - c0, CH_MAX);
            const int chb = CH * ESZ;
            const float em1y = (float)(L.H - 1), em1x = (float)(L.W - 1);
            const int n_list = cntC;
            const ListEntryA *__restrict__ list = entries + offC;

            for (int base = 0; base < n_list; base += 32) {
                ListEntryA e = eC;
                if (base > 0) {
                    e = no_entry();
                    if (base + lane < n_list) e = list[base + lane];
                }
                // ---- plan 32 ROIs at once, one per lane: the runs of sample rows / columns that reach the tile
                int ky0 = 0, nky = 0, kx0 = 0, nkx = 0;
                if (e.roi >= 0 && !(e.win.y1 < y0 || e.win.y0 > y1 || e.win.x1 < x0 || e.win.x0 > x1)) {
                    sample_run(e.ax.by, e.ax.sy, em1y, ph, y0, y1, L.H, ky0, nky);
                    if (nky > 0) sample_run(e.ax.bx, e.ax.sx, em1x, pw, x0, x1, L.W, kx0, nkx);
                }
                unsigned todo = __ballot_sync(0xffffffffu, nky > 0 && nkx > 0);
                const int packed = ky0 | (nky << 8) | (kx0 << 16) | (nkx << 24);
                // per hit, still one ROI per lane: where its first staged sample lives and how its rows pack into stages --
                // computed 32 at a time here instead of once per hit on the serial chain below
                const long long goff = ((long long)e.roi * S + (long long)ky0 * pw + kx0) * C + c0;
                const int pack2 = rows_per_stage<STG_S>(nkx > 0 ? nkx : 1) | (min(nkx, STG_S) << 8);
                while (todo) {
                    const int bit = __ffs(todo) - 1;
                    todo &= todo - 1;
                    const long long go = __shfl_sync(0xffffffffu, goff, bit);
                    const int pk = __shfl_sync(0xffffffffu, packed, bit), pk2 = __shfl_sync(0xffffffffu, pack2, bit);
                    const float by = __shfl_sync(0xffffffffu, e.ax.by, bit), sy = __shfl_sync(0xffffffffu, e.ax.sy, bit);
                    const float bx = __shfl_sync(0xffffffffu, e.ax.bx, bit), sx = __shfl_sync(0xffffffffu, e.ax.sx, bit);
                    const int sy0 = pk & 0xff, nsy = (pk >> 8) & 0xff, sx0 = (pk >> 16) & 0xff, nsx = (pk >> 24) & 0xff;
                    // lane i: tap of sample row sy0 + i and of sample column sx0 + i (same arithmetic as the forward)
                    const Tap ty = tap_at(by, sy, em1y, sy0 + lane), tx = tap_at(bx, sx, em1x, sx0 + lane);
                    const int2 my_row = make_int2(ty.lo - y0, __float_as_int(ty.lerp));
                    XEnt my_col;
                    my_col.pl = tx.lo - x0;
                    my_col.xl = tx.lerp;
                    const T *gr = grads + go;
                    // stages: whole sample rows, as many as fit; a row longer than a stage takes several stages
                    const int n_s_full = pk2 >> 8;
                    const int rows_per = pk2 & 0xff;
                    for (int ra = 0; ra < nsy; ra += rows_per) {
                        const int n_rows = min(rows_per, nsy - ra);
                        for (int sb = 0; sb < nsx; sb += STG_S) {
                            const int n_s = min(n_s_full, nsx - sb);
                            const unsigned s = acquire();
                            Desc *d = sdesc + s;
                            if (lane == 0) *reinterpret_cast<int4 *>(d) = make_int4(ST_DATA, n_s, n_rows, chb);
                            const int rrow = lane - ra, rcol = lane - sb;
                            const bool row_mine = rrow >= 0 && rrow < n_rows;
                            if (row_mine) d->rowd[rrow] = my_row;
                            if (rcol >= 0 && rcol < n_s) d->x[rcol] = my_col;
                            const uint32_t bar = full0 + 8 * s;
                            // the copies go out first; the stage's phase cannot complete before lane 0's arrival below (one
                            // pending arrival), so bytes landing ahead of the expect_tx only drive the count negative for a while
                            if (row_mine) {                  // lane ra + i fetches stage row i
                                const uint32_t dst = smem_u32(stages + (size_t)s * STAGE_BYTES) + rrow * n_s * chb;
                                const T *src = gr + ((size_t)lane * pw + sb) * C;
                                if (CH == C) {
                                    bulk_g2s(dst, src, (uint32_t)(n_s * chb), bar);
                                } else {                     // channel chunk of a wider map: one copy per sample
                                    for (int k = 0; k < n_s; ++k) bulk_g2s(dst + k * chb, src + (size_t)k * C, (uint32_t)chb, bar);
                                }
                            }
                            __syncwarp();                    // the descriptor stores of all lanes before the arrival
                            if (lane == 0) mbar_arrive_expect_tx(bar, (uint32_t)(n_rows * n_s * chb));
                            advance();
                        }
                    }
                }
            }
            // end of tile: the write-out record
            {
                const unsigned s = acquire();
                Desc *d = sdesc + s;
                if (lane == 0) {
                    d->flags = ST_TILE_END;
                    d->n_s = CH;
                    TileOut o;
                    o.out = (unsigned long long)(reinterpret_cast<T *>(L.out) + (((size_t)gC.b * L.H + y0) * L.W + x0) * C + c0);
                    o.row_stride = L.W * (C / VPV);
                    o.pix_stride = C / VPV;
                    o.ny = y1 - y0 + 1;
                    o.nx = x1 - x0 + 1;
                    *reinterpret_cast<TileOut *>(d->rows) = o;
                    mbar_arrive(full0 + 8 * s);
                }
                advance();
            }
            wC = wB; cntC = cntB; offC = offB; eC = eB; gC = gB;
            wB = wA; cntB = cntA; offB = offA; gB = gA;
            wA = __shfl_sync(0xffffffffu, tF, 0);
        }
        const unsigned s = acquire();
        if (lane == 0) {
            sdesc[s].flags = ST_EXIT;
            mbar_arrive(full0 + 8 * s);
        }
        return;
    }

    // =============================================================== consumers
    // Warp c owns pixel COLUMN c of the tile (8 rows x C channels in registers).  A staged sample row reaches two pixel
    // rows but, with its ~8-16 samples, every column of the tile: column ownership keeps all eight warps busy on every
    // stage row (row ownership, the first version of this kernel, had two of eight at work and was latency-bound).
    const int c = warp;                                     // tile column
    float4 acc[TH][NACC];
#pragma unroll
    for (int k = 0; k < TH; ++k)
#pragma unroll
        for (int v = 0; v < NACC; ++v) acc[k][v] = make_float4(0.f, 0.f, 0.f, 0.f);

    for (unsigned s = 0, fpar = 0;; fpar ^= (++s == NST), s = s == NST ? 0u : s) {
        mbar_wait(full0 + 8 * s, fpar);
        const Desc *d = sdesc + s;
        const int4 hdr = *reinterpret_cast<const int4 *>(d);        // flags, n_s, n_rows, chb
        if (hdr.x != ST_DATA) {
            if (hdr.x == ST_EXIT) break;
            // ---- end of tile: write the column exactly once (zeros included), clear the accumulators
            const TileOut o = *reinterpret_cast<const TileOut *>(d->rows);
            const int CH = hdr.y;
            const bool ok0 = FULL || lane * VPV < CH, ok1 = NV == 2 && (FULL || lane * 4 + 128 < CH);
            if (c < o.nx) {
                if constexpr (ESZ == 4) {
                    float4 *__restrict__ op = reinterpret_cast<float4 *>(o.out) + (size_t)c * o.pix_stride + lane;
#pragma unroll
                    for (int k = 0; k < TH; ++k) {
                        if (k < o.ny) {
                            if (ok0) __stcs(op + (size_t)k * o.row_stride, acc[k][0]);
                            if (ok1) __stcs(op + (size_t)k * o.row_stride + 32, acc[k][1]);
                        }
                    }
                } else {        // 8 channels per lane, rounded once: 16 bytes per pixel
                    uint4 *__restrict__ op = reinterpret_cast<uint4 *>(o.out) + (size_t)c * o.pix_stride + lane;
#pragma unroll
                    for (int k = 0; k < TH; ++k)
                        if (k < o.ny && ok0) __stcs(op + (size_t)k * o.row_stride, narrow8<T>(acc[k][0], acc[k][1]));
                }
            }
#pragma unroll
            for (int k = 0; k < TH; ++k)
#pragma unroll
                for (int v = 0; v < NACC; ++v) acc[k][v] = make_float4(0.f, 0.f, 0.f, 0.f);
            __syncwarp();
            if (lane == 0) mbar_arrive(empty0 + 8 * s);
            continue;
        }
        // the samples of a stage row whose left or right tap lands on my column: a run (tap columns are monotone in sx)
        const int n_s = hdr.y;
        int s0, ns;
        {
            bool hit = false;
            if (lane < n_s) {
                const XEnt e = d->x[lane];
                hit = e.pl == c || (e.pl == c - 1 && e.xl != 0.f);
            }
            const unsigned m = __ballot_sync(0xffffffffu, hit);
            s0 = m ? __ffs(m) - 1 : 0;
            ns = __popc(m);
        }
#ifdef SLN_BWD_PROBE_NO_COMPUTE
        ns = 0;                             // diagnostic build: the consumers only shake hands (pace of producer + copies)
#endif
        if (ns > 0) {
            const int chb = FULL ? NV * 512 : hdr.w;
            const bool ok0 = FULL || lane * 16 < chb, ok1 = NV == 2 && (FULL || lane * 16 + 512 < chb);
            const unsigned char *stage = stages + (size_t)s * STAGE_BYTES + (size_t)s0 * chb + lane * 16;
            for (int r = 0; r < hdr.z; ++r) {
                const int2 rd = d->rowd[r];
                const int rel = rd.x;                           // tile row of the top tap, -1 .. 7 (other values: no tap here)
                const float yl = __int_as_float(rd.y);
                const float wt = __fsub_rn(1.f, yl);
                const unsigned char *rowp = stage + (size_t)r * n_s * chb;
                const XEnt *xe = d->x + s0;
                for (int k = ns; k > 0; --k, rowp += chb, ++xe) {
                    const XEnt e = *xe;
                    float4 g0, g1;
                    if constexpr (ESZ != 4) {       // widen the lane's 8 staged channels
                        uint4 raw = make_uint4(0u, 0u, 0u, 0u);
                        if (FULL || ok0) raw = *reinterpret_cast<const uint4 *>(rowp);
                        widen8<T>(raw, g0, g1);
                    } else if (FULL) {
                        g0 = *reinterpret_cast<const float4 *>(rowp);
                        if (NV == 2) g1 = *reinterpret_cast<const float4 *>(rowp + 512);
                    } else {
                        g0 = make_float4(0.f, 0.f, 0.f, 0.f);
                        g1 = g0;
                        if (ok0) g0 = *reinterpret_cast<const float4 *>(rowp);
                        if (ok1) g1 = *reinterpret_cast<const float4 *>(rowp + 512);
                    }
                    const float wl = __fsub_rn(1.f, e.xl);
                    if (!EXACT) {
                        // one x tap of the sample is mine (an integral column has its whole weight on the left tap)
                        const float wx = e.pl == c ? wl : e.xl;
                        const float a = __fmul_rn(wt, wx), bb = __fmul_rn(yl, wx);
                        switch (rel) {
                        case -1: SLN_TMA_ADD(0, bb, 0.f, 0.f) break;
                        case 0: SLN_TMA_ADD(0, a, 0.f, 0.f) SLN_TMA_ADD(1, bb, 0.f, 0.f) break;
                        case 1: SLN_TMA_ADD(1, a, 0.f, 0.f) SLN_TMA_ADD(2, bb, 0.f, 0.f) break;
                        case 2: SLN_TMA_ADD(2, a, 0.f, 0.f) SLN_TMA_ADD(3, bb, 0.f, 0.f) break;
                        case 3: SLN_TMA_ADD(3, a, 0.f, 0.f) SLN_TMA_ADD(4, bb, 0.f, 0.f) break;
                        case 4: SLN_TMA_ADD(4, a, 0.f, 0.f) SLN_TMA_ADD(5, bb, 0.f, 0.f) break;
                        case 5: SLN_TMA_ADD(5, a, 0.f, 0.f) SLN_TMA_ADD(6, bb, 0.f, 0.f) break;
                        case 6: SLN_TMA_ADD(6, a, 0.f, 0.f) SLN_TMA_ADD(7, bb, 0.f, 0.f) break;
                        case 7: SLN_TMA_ADD(7, a, 0.f, 0.f) break;
                        default: break;                      // not a row of this tile
                        }
                    } else {
                        // reference order per sample and pixel: TL, TR on the top row, then BL, BR on the bottom row, which
                        // is the same row (weight 0) when the sample row is integral; the right tap coincides with the left
                        // one when the sample column is integral
                        const int pr = e.pl + (e.xl != 0.f);
                        const int rb = rel + (yl != 0.f);
#pragma unroll
                        for (int pass = 0; pass < 2; ++pass) {
                            const int row = pass == 0 ? rel : rb;
                            const float w_y = pass == 0 ? wt : yl;
#pragma unroll
                            for (int side = 0; side < 2; ++side) {
                                if ((side == 0 ? e.pl : pr) != c) continue;
                                const float w_x = side == 0 ? wl : e.xl;
                                switch (row) {
                                case 0: SLN_TMA_ADD(0, 0.f, w_y, w_x) break;
                                case 1: SLN_TMA_ADD(1, 0.f, w_y, w_x) break;
                                case 2: SLN_TMA_ADD(2, 0.f, w_y, w_x) break;
                                case 3: SLN_TMA_ADD(3, 0.f, w_y, w_x) break;
                                case 4: SLN_TMA_ADD(4, 0.f, w_y, w_x) break;
                                case 5: SLN_TMA_ADD(5, 0.f, w_y, w_x) break;
                                case 6: SLN_TMA_ADD(6, 0.f, w_y, w_x) break;
                                case 7: SLN_TMA_ADD(7, 0.f, w_y, w_x) break;
                                default: break;              // -1 / 8: the neighbouring tile's pixel
                                }
                            }
                        }
                    }
                }
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty0 + 8 * s);
    }
}
#undef SLN_TMA_ADD

template <int NV, bool EXACT, bool FULL, int STG_S, int NST>
__global__ void __launch_bounds__(THREADS, 2)
crop_bwd_tma_kernel(const float *__restrict__ grads, const ListEntryA *__restrict__ entries, const int *__restrict__ st_off,
                    const int *__restrict__ st_count, const BwdLevel *__restrict__ lv_table,
                    BwdTileBases TB, int C, int ph, int pw, int n_work, int chunks, int *__restrict__ queue)
{
    crop_bwd_tma_body<float, NV, EXACT, FULL, STG_S, NST>(grads, entries, st_off, st_count, lv_table, TB, C, ph, pw, n_work, chunks,
                                                          queue);
}

// T = __nv_bfloat16 / __half: 8 channels (one 16-byte vector) per consumer lane
template <typename T, bool EXACT, bool FULL, int STG_S, int NST>
__global__ void __launch_bounds__(THREADS, 2)
crop_bwd_tma_b16_kernel(const T *__restrict__ grads, const ListEntryA *__restrict__ entries, const int *__restrict__ st_off,
                        const int *__restrict__ st_count, const BwdLevel *__restrict__ lv_table,
                        BwdTileBases TB, int C, int ph, int pw, int n_work, int chunks, int *__restrict__ queue)
{
    crop_bwd_tma_body<T, 1, EXACT, FULL, STG_S, NST>(grads, entries, st_off, st_count, lv_table, TB, C, ph, pw, n_work, chunks, queue);
}

template <int STG_S, int NST, int ESZ = 4>
static size_t smem_bytes()
{
    return (size_t)NST * STG_S * CH_MAX * ESZ + sizeof(StageDesc<STG_S>) * NST + sizeof(BwdLevel) * BWD_MAX_LEVELS +
           sizeof(uint64_t) * 2 * NST + 128;
}

}  // namespace bwdtma
