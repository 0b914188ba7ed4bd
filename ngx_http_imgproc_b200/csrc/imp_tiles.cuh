// imp_tiles.cuh — shared-memory tile kernels (sm_100a): the source rectangle a CTA needs is staged into
// shared memory by the TMA engine (one cp.async.bulk per source row, completion counted on an mbarrier),
// the gather + op list run out of shared memory / registers, and the result is stored coalesced.
//
// The direct-from-global kernels in imp_kernels.cu remain the general path (any pitch/alignment, any
// footprint); these are selected per job when the source rows are 16-byte addressable
// (pick_launch, imp_gpu.cu) and the footprint fits the shared-memory budget.
#pragma once
#include "imp_gather.cuh"

// ---- debug build (-DIMP_DEBUG_BOUNDS; ngx_http_imgproc_b200/build.py --debug -> libimp_gpu_dbg.so) -----------------------
// compute-sanitizer is not available on the GPU pool, so the tile kernels carry their own bounds assertions on every
// staged-tile, lookup-table, out-stage and destination address they form; a violated one sets a bit that
// imp_gpu_debug_flags() reads back (tests/test_gpu_host_path.py runs the request fuzz over the debug build). Bits:
// 0-1 blur (border fill, out stage), 2-3 cubic, 4-6 gather tile, 8-11 strip kernels (tile reads, taps, destination).
#if defined(IMP_DEBUG_BOUNDS)
static __device__ unsigned g_imp_dbg_flags;
#define IMP_DBG(cond, bit) do { if (!(cond)) atomicOr(&g_imp_dbg_flags, 1u << (bit)); } while (0)
static inline unsigned imp_debug_flags_tu() { unsigned v = 0; cudaMemcpyFromSymbol(&v, g_imp_dbg_flags, sizeof v); return v; }
#else
#define IMP_DBG(cond, bit) do { } while (0)
static inline unsigned imp_debug_flags_tu() { return 0; }
#endif

namespace imp_tiles {

// ---- PTX: mbarrier + 1-D bulk async copy (TMA, SASS UBLKCP) ---------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// The same on a 32-bit shared-window address: the ring loops convert their barrier arrays ONCE (the generic->shared cvta per
// poll was 5-9 % of the strip kernels' instructions in the round-2 captures).
__device__ __forceinline__ void mbar_wait_a(uint32_t bar_addr, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(bar_addr), "r"(parity) : "memory");
}
__device__ __forceinline__ void mbar_arrive_a(uint32_t bar_addr) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_addr) : "memory");
}
// global -> shared, 16-byte aligned on both sides, size a multiple of 16.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// 2-D tiled TMA load (SASS UTMALDG): box of the job's tensor map at element coordinates (c0, c1).
__device__ __forceinline__ void tma_load_2d(void* dst_smem, const void* tmap, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(smem_u32(dst_smem)), "l"(tmap), "r"(c0), "r"(c1), "r"(smem_u32(bar)) : "memory");
}

// u8 -> f32 product without the XU pipe: m = 2^23 + S (PRMT), fma(m, a, -(2^23*a)) == RN(S*a) exactly,
// because m*a - 2^23*a == S*a in exact arithmetic and FMA rounds once.
__device__ __forceinline__ float byte_times(uint32_t word, int sel, float a, float neg_a23) {
    const float m = __uint_as_float(__byte_perm(word, 0x4B000000u, 0x7650 | sel));
    return __fmaf_rn(m, a, neg_a23);
}
__device__ __forceinline__ float u8_times(uint32_t byte, float a, float neg_a23) {
    return __fmaf_rn(__uint_as_float(byte | 0x4B000000u), a, neg_a23);
}

// Loads NB consecutive bytes that start at an arbitrarily aligned shared-memory address into NB/4 (rounded up)
// registers: aligned 32-bit loads + funnel shifts, so packed 3-channel pixels cost ~1/4 LDS + 1/4 SHF per byte
// instead of one LDS.U8 each, and every byte then sits at a compile-time position.
template <int NB>
__device__ __forceinline__ void load_bytes(const uint8_t* p, uint32_t (&w)[(NB + 3) / 4]) {
    constexpr int NW = (NB + 3) / 4;
    // plain pointer arithmetic (no integer round trip), so the compiler still knows these are shared-memory loads (LDS,
    // 32-bit addresses) — through uintptr_t they became generic LD.E with 64-bit address maths
    // the low address bits are the same in the generic and the shared window: no cvta (10 % of the cfg1 kernel's instructions)
    const unsigned mis = (unsigned)reinterpret_cast<uintptr_t>(p) & 3u;
    const uint32_t* base = reinterpret_cast<const uint32_t*>(p - mis);
    const unsigned sh = mis * 8;
    uint32_t raw[NW + 1];
#pragma unroll
    for (int i = 0; i <= NW; i++) raw[i] = base[i];
#pragma unroll
    for (int i = 0; i < NW; i++) w[i] = __funnelshift_r(raw[i], raw[i + 1], sh);
}

constexpr int TW = 32, TH = 8;          // output tile
constexpr int MAX_SMEM = 96 * 1024;     // source-tile budget per CTA

// ---- INTER_AREA, fractional scale (SURVEY App. A.3), from a shared-memory tile ----------------------------
// One thread per output pixel; a warp is one output row of the tile, so the y taps are warp-uniform.
// area_rows() accumulates one output pixel from the staged rows.
// The x taps of a column are NT contiguous source pixels whose weights sit in registers. Columns with
// fewer taps than NT are zero-padded on the right: the padded products are exactly +0, and adding +0
// leaves a running float sum bit-identical, so the result equals OpenCV's ordered accumulation.
// (A padded tap may read a byte past the staged pixels; any byte converts to a finite float.)
template <int SC, int NT>
__device__ __forceinline__ void area_rows(const uint8_t* __restrict__ row /* first source row, my first tap */, int rs, const ImpAreaTap* yt /* shared memory */, int ycount,
                                          const float (&a)[NT], const float (&na)[NT], float (&sum)[SC]) {
    // the y taps of an output row are consecutive source rows and were staged next to the pixels by the producer, so
    // this loop touches no global memory at all
    // OpenCV assigns the first row's product and adds the rest; 0 + p == p exactly (p >= +0), so the sum starts at 0
#pragma unroll
    for (int c = 0; c < SC; c++) sum[c] = 0.0f;
    for (int j = 0; j < ycount; j++, row += rs) {
        const float beta = yt[j].a;
        float h[SC];
        uint32_t seg[SC == 4 ? 1 : (NT * SC + 3) / 4];
        if (SC != 4) load_bytes<(SC == 4 ? 4 : NT * SC)>(row, seg);
#pragma unroll
        for (int k = 0; k < NT; k++) {
            if (SC == 4) {
                const uint32_t w = *reinterpret_cast<const uint32_t*>(row + k * 4);
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    const float pr = byte_times(w, c, a[k], na[k]);
                    h[c] = (k == 0) ? pr : __fadd_rn(h[c], pr);
                }
            } else {
#pragma unroll
                for (int c = 0; c < SC; c++) {
                    const int pos = k * SC + c;
                    const float pr = byte_times(seg[pos / 4], pos % 4, a[k], na[k]);
                    h[c] = (k == 0) ? pr : __fadd_rn(h[c], pr);
                }
            }
        }
#pragma unroll
        for (int c = 0; c < SC; c++) {
            sum[c] = __fadd_rn(sum[c], __fmul_rn(beta, h[c]));
        }
    }
}

// Integer-scale INTER_AREA (SURVEY App. A.2): plain byte sums over the NT x ycount block. For 4 channels two
// PRMTs split a pixel into two packed u16 pairs, so a pixel costs LDS + 2 PRMT + 2 IADD (block <= 256 px).
template <int SC, int NT>
__device__ __forceinline__ void area_int_rows(const uint8_t* __restrict__ row, int rs, int ycount, int (&isum)[SC]) {
    unsigned lo = 0, hi = 0;                       // SC == 4: {B,R} and {G,A} as u16 pairs
#pragma unroll
    for (int c = 0; c < SC; c++) isum[c] = 0;
    for (int j = 0; j < ycount; j++, row += rs) {
#pragma unroll
        for (int k = 0; k < NT; k++) {
            if (SC == 4) {
                const uint32_t w = *reinterpret_cast<const uint32_t*>(row + k * 4);
                lo += __byte_perm(w, 0, 0x4240);   // bytes 0 and 2 -> low halves
                hi += __byte_perm(w, 0, 0x4341);   // bytes 1 and 3
            }
        }
        if (SC != 4) {
            uint32_t seg[SC == 4 ? 1 : (NT * SC + 3) / 4];
            load_bytes<(SC == 4 ? 4 : NT * SC)>(row, seg);
            // per channel: dp4a of each word with the 0/1 mask of that channel's byte positions (compile-time)
#pragma unroll
            for (int c = 0; c < SC; c++) {
#pragma unroll
                for (int wi = 0; wi < (NT * SC + 3) / 4; wi++) {
                    unsigned mask = 0;
#pragma unroll
                    for (int bpos = 0; bpos < 4; bpos++) {
                        const int pos = wi * 4 + bpos;
                        if (pos < NT * SC && pos % SC == c) mask |= 1u << (8 * bpos);
                    }
                    if (mask) isum[c] = __dp4a(seg[wi], mask, (unsigned)isum[c]);
                }
            }
        }
    }
    if (SC == 4) { isum[0] = lo & 0xFFFF; isum[2 % SC] = lo >> 16; isum[1 % SC] = hi & 0xFFFF; isum[3 % SC] = hi >> 16; }
}

// Round-half-even of 0 <= x < 2^22 without F2I (FADD + IADD).
__device__ __forceinline__ int rint_pos(float x) { return __float_as_int(__fadd_rn(x, 12582912.0f)) - 0x4B400000; }

// Persistent strip kernel. A CTA owns a strip of 32 output columns of one job and walks down its 8-row
// tiles. Warp 8 is the TMA producer: it stages the source rows of tile t+1 into the other half of a
// multi-stage shared-memory ring (2..8 stages, as many as fit ~64 KB) while warps 0-7 (one output row each) consume tile t. full[]/empty[]
// mbarriers carry the hand-off; the per-thread x weights are loaded once per strip.
//   blob tables (host, imp_planner.cpp): xtile[tx] = {first source px, last source px} of tile column tx,
//   ytile[ty] = {first source row, number of source rows} of tile row ty.
constexpr int STRIP_CONSUMERS = TW * TH;          // 256 threads, 8 warps
constexpr int STRIP_PRODUCER_WARPS = 1;         // UBLKCP issue is serialised per warp: spread the rows over 4 warps
constexpr int STRIP_THREADS = STRIP_CONSUMERS + 32 * STRIP_PRODUCER_WARPS;

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Orders this thread's earlier generic-proxy accesses to shared memory (plain LDS) before later async-proxy ones (the TMA
// refill a released stage receives). The AREA consumers do not need it: their arithmetic has consumed every loaded byte
// before the stage is released. The plain gathers only LOAD before releasing — the values are first used by the
// epilogue — and without the fence the refill overtook loads still queued behind the scattered byte stores of a
// rotated 3-channel store (round 2: rotate=90/270 on 3-channel frames read the tile of 8 rows later).
__device__ __forceinline__ void fence_generic_to_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// The destination address of base pixel (bx, by) is affine in by for a fixed bx under all eight output orientations
// (dst + Y*pitch + X*dc with (X,Y) = imp_map_xy): a thread of a strip owns one bx, so it keeps {address of (bx,0), step
// per by} instead of re-evaluating the frame map from the pass header for every pixel.
struct StripStore { uint8_t* base; int step; int rows; };
__device__ __forceinline__ StripStore strip_store_line(const ImpFrameMap& om, uint8_t* dst, int pitch, int dc, int bx) {
    int X0, Y0, X1, Y1;
    imp_map_xy(om, bx, 0, X0, Y0);
    imp_map_xy(om, bx, 1, X1, Y1);
    StripStore s;
    s.base = dst + (ptrdiff_t)Y0 * pitch + (ptrdiff_t)X0 * dc;
    s.step = (Y1 - Y0) * pitch + (X1 - X0) * dc;
    s.rows = om.h;
    return s;
}

// Rows of column bx on which the op list can change a pixel. A list made only of watermarks (the common request:
// resize + watermark) touches nothing outside the watermark rectangles, so a thread asks once per strip for the
// by-interval its column shares with them and skips the op loop elsewhere. Any other op -> every row.
struct StripOpsRows { int y0, y1; };
__device__ __forceinline__ StripOpsRows strip_ops_rows(const uint8_t* s_ops, int nops, int bx) {
    StripOpsRows r; r.y0 = 0x7fffffff; r.y1 = -1;
    const ImpOp* ops = reinterpret_cast<const ImpOp*>(s_ops);
    for (int k = 0; k < nops; k++) {
        const ImpOp& op = ops[k];
        if (op.kind != IMP_OP_WATERMARK) { r.y0 = 0; r.y1 = 0x7fffffff; return r; }
        // watermark rectangle [i0, i0+i2) x [i1, i1+i3) of the op's frame, pulled back through imp_map_xy
        const ImpFrameMap m = op.map;
        const int ulo = m.flipx ? m.w - op.i[0] - op.i[2] : op.i[0], uhi = ulo + op.i[2] - 1;
        const int vlo = m.flipy ? m.h - op.i[1] - op.i[3] : op.i[1], vhi = vlo + op.i[3] - 1;
        const int xlo = m.swap ? vlo : ulo, xhi = m.swap ? vhi : uhi, ylo = m.swap ? ulo : vlo, yhi = m.swap ? uhi : vhi;
        if (bx >= xlo && bx <= xhi) { r.y0 = min(r.y0, ylo); r.y1 = max(r.y1, yhi); }
    }
    return r;
}

// Shared epilogue of the strip kernels: op list + store of one pixel. Inlined: an out-of-line call (v[] through
// local memory + call/return) measured 12-20 % slower on cfg1/cfg2 than the larger code.
template <int SC, int FL>
__device__ __forceinline__ void strip_epilogue(const ImpJob& job, int oc, int dc, const StripStore& st, const StripOpsRows& orows, const uint8_t* s_ops, int nops, int bx, int by, const int* v) {
    ImpPx p;
    if (SC == 1) { p.b = p.g = p.r = v[0]; p.a = 255; }
    else { p.b = v[0]; p.g = v[SC > 1 ? 1 : 0]; p.r = v[SC > 2 ? 2 : 0]; p.a = (SC == 4) ? v[SC - 1] : 255; }
    if (by >= orows.y0 && by <= orows.y1) {
        ImpPx px[1] = {p};
        const int xs[1] = {bx}, ys[1] = {by};
        imp_run_ops_n<1, FL == 1, false, FL == 2>(px, oc, xs, ys, reinterpret_cast<const ImpOp*>(s_ops), nops, s_ops + nops * sizeof(ImpOp), job.wm, job.wm_pitch, job.wm_c);
        p = px[0];
    }
    uint8_t* d = st.base + (ptrdiff_t)by * st.step;
    IMP_DBG(d >= job.dst && d + dc <= job.dst + (size_t)st.rows * job.dst_pitch, 11);
    if (dc == 4) *reinterpret_cast<uchar4*>(d) = make_uchar4((unsigned char)p.b, (unsigned char)p.g, (unsigned char)p.r, (unsigned char)p.a);
    else { d[0] = (unsigned char)p.b; d[1] = (unsigned char)p.g; d[2] = (unsigned char)p.r; }
}

template <int SC, int NT, int MODE, int FL>
__device__ __forceinline__ void area_strip_consume(const ImpJob& job, const ImpPass* __restrict__ P, const uint8_t* __restrict__ blob,
                                                   const uint8_t* tile0, int stage_bytes, uint64_t* full, uint64_t* empty,
                                                   const uint8_t* s_ops, int nops, int bx0, int col_off, int tiles_y, int NSTAGE) {
    const ImpRange* __restrict__ xr = reinterpret_cast<const ImpRange*>(blob + P->xofs_off);
    const ImpAreaTap* __restrict__ xt = reinterpret_cast<const ImpAreaTap*>(blob + P->xcoef_off);
    const int bw = P->bw, bh = P->bh, rs = P->tile_rs;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool in_x = bx0 + lane < bw;
    const int bx = min(bx0 + lane, bw - 1);
    const int2 rxv = __ldg(reinterpret_cast<const int2*>(xr + bx));
    float a[MODE == 0 ? NT : 1], na[MODE == 0 ? NT : 1];
    if (MODE == 0) {
#pragma unroll
        for (int k = 0; k < (MODE == 0 ? NT : 1); k++) {
            a[k] = (k < rxv.y) ? __int_as_float(__ldg(reinterpret_cast<const int2*>(xt + rxv.x + k)).y) : 0.0f;
            na[k] = -8388608.0f * a[k];
        }
    }
    const int box_2x2 = (P->nx == 2 && P->ny == 2);
    const float box_scale = P->area_scale;
    const int my_off = col_off + __ldg(reinterpret_cast<const int*>(xt + rxv.x)) * SC;    // byte offset of my first tap in a tile row

    const int box_bytes = rs * P->tile_rows;
    const int ytap_bytes = (P->tile_ytaps * 8 + 15) & ~15;
    const int oc = P->oc, dc = P->dc;
    const StripStore st = strip_store_line(P->out, job.dst, job.dst_pitch, dc, bx);
    const StripOpsRows orows = strip_ops_rows(s_ops, nops, bx);
    int stage = 0, phase = 0;
    const uint32_t full_a = smem_u32(full), empty_a = smem_u32(empty);
    for (int t = 0; t < tiles_y; t++) {
        const int by = min(t * TH + warp, bh - 1);
        const bool in_y = t * TH + warp < bh;
        mbar_wait_a(full_a + stage * 8, phase);
        const uint8_t* sbase = tile0 + stage * stage_bytes;
        const ImpAreaTap* s_yt = reinterpret_cast<const ImpAreaTap*>(sbase + box_bytes);              // the tile's y taps
        // {byte offset of my first source row in the tile, taps, first tap}: one 16-byte load starts the row
        const int4 yrow = reinterpret_cast<const int4*>(sbase + box_bytes + ytap_bytes)[by - t * TH];
        int v[SC];
        if (MODE == 0) {
            float sum[SC];
            // rows [yrow.x/rs, +yrow.y) of the box, NT taps (the zero-weight padded ones included, +4 for the aligned word loads)
            IMP_DBG(my_off >= 0 && yrow.x >= 0 && yrow.x + (yrow.y - 1) * rs + my_off + NT * SC + (SC == 4 ? 0 : 4) <= box_bytes + (SC == 4 ? 0 : 4) && my_off + NT * SC <= rs + 4, 8);
            IMP_DBG(yrow.z >= 0 && (yrow.z + yrow.y) * 8 <= ytap_bytes, 9);
            area_rows<SC, (MODE == 0 ? NT : 1)>(sbase + my_off + yrow.x, rs, s_yt + yrow.z, yrow.y, a, na, sum);
#pragma unroll
            for (int c = 0; c < SC; c++) v[c] = min(rint_pos(sum[c]), 255);          // sums are >= 0
        } else {
            // integer-scale mode lives in area_int_strip_consume()
#pragma unroll
            for (int c = 0; c < SC; c++) v[c] = box_2x2 ? (v[c] + 2) >> 2 : min(rint_pos(__fmul_rn(imp_u2f(v[c]), box_scale)), 255);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive_a(empty_a + stage * 8);             // this warp is done with the stage
        if (in_x && in_y) strip_epilogue<SC, FL>(job, oc, dc, st, orows, s_ops, nops, bx, by, v);
        if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
    }
}

// Integer-scale consumer (INTER_AREA NxM): no tap tables at all — output row y reads source rows y*ny .. y*ny+ny-1 and
// output column x reads source pixels x*nx .. — and the store map is hoisted (registers are plentiful here).
// Kept separate from the fractional consumer: sharing one body cost that one 4 % (register allocation).
template <int SC, int NT, int FL>
__device__ __forceinline__ void area_int_strip_consume(const ImpJob& job, const ImpPass* __restrict__ P, const uint8_t* tile0, int stage_bytes,
                                                       uint64_t* full, uint64_t* empty, const uint8_t* s_ops, int nops, int bx0, int col_off,
                                                       int tiles_y, int NSTAGE) {
    const int bw = P->bw, bh = P->bh, rs = P->tile_rs, oc = P->oc, dc = P->dc, ny = P->ny;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool in_x = bx0 + lane < bw;
    const int bx = min(bx0 + lane, bw - 1);
    const int box_2x2 = (P->nx == 2 && ny == 2);
    const float box_scale = P->area_scale;
    const int my_off = col_off + bx * NT * SC;                        // byte offset of my first source pixel in a tile row
    const StripStore st = strip_store_line(P->out, job.dst, job.dst_pitch, dc, bx);
    const StripOpsRows orows = strip_ops_rows(s_ops, nops, bx);
    int stage = 0, phase = 0;
    const uint32_t full_a = smem_u32(full), empty_a = smem_u32(empty);
    for (int t = 0; t < tiles_y; t++) {
        const int by = min(t * TH + warp, bh - 1);
        const bool in_y = t * TH + warp < bh;
        mbar_wait_a(full_a + stage * 8, phase);
        int v[SC];
        IMP_DBG(my_off >= 0 && my_off + NT * SC <= rs + 4 && (by * ny - t * TH * ny) >= 0 && (by * ny - t * TH * ny + ny) <= P->tile_rows, 8);
        area_int_rows<SC, NT>(tile0 + (stage * stage_bytes + my_off + (by * ny - t * TH * ny) * rs), rs, ny, v);
#pragma unroll
        for (int c = 0; c < SC; c++) v[c] = box_2x2 ? (v[c] + 2) >> 2 : min(rint_pos(__fmul_rn(imp_u2f(v[c]), box_scale)), 255);
        __syncwarp();
        if (lane == 0) mbar_arrive_a(empty_a + stage * 8);             // this warp is done with the stage
        if (in_x && in_y) strip_epilogue<SC, FL>(job, oc, dc, st, orows, s_ops, nops, bx, by, v);
        if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
    }
}

// INTER_LINEAR consumer of the strip kernel (mode 3; shrinking only, the gather tile kernel enlarges): the same TMA ring,
// one output row per warp, each pixel from 2x2 staged source pixels. The per-column part of the gather (source offsets,
// x coefficients) is loaded once per strip.
template <int SC, int FL>
__device__ __forceinline__ void linear_strip_consume(const ImpJob& job, const ImpPass* __restrict__ P, const uint8_t* __restrict__ blob,
                                                     const uint8_t* tile0, int stage_bytes, uint64_t* full, uint64_t* empty,
                                                     const uint8_t* s_ops, int nops, int bx0, int col_off, int tiles_y, int NSTAGE) {
    const int bw = P->bw, bh = P->bh, sw = P->sw, sh = P->sh, rs = P->tile_rs, oc = P->oc, dc = P->dc;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool in_x = bx0 + lane < bw;
    const int bx = min(bx0 + lane, bw - 1);
    const int* __restrict__ yofs = reinterpret_cast<const int*>(blob + P->yofs_off);
    const int4* __restrict__ ytile = reinterpret_cast<const int4*>(blob + P->ytile_off);
    const int xs = __ldg(reinterpret_cast<const int*>(blob + P->xofs_off) + bx);
    const int xo0 = col_off + min(max(xs, 0), sw - 1) * SC, xo1 = col_off + min(max(xs + 1, 0), sw - 1) * SC;
    const short* xa = reinterpret_cast<const short*>(blob + P->xcoef_off);
    const int a0 = __ldg(xa + bx * 2), a1 = __ldg(xa + bx * 2 + 1);
    const StripStore st = strip_store_line(P->out, job.dst, job.dst_pitch, dc, bx);
    const StripOpsRows orows = strip_ops_rows(s_ops, nops, bx);
    int stage = 0, phase = 0;
    const uint32_t full_a = smem_u32(full), empty_a = smem_u32(empty);
    for (int t = 0; t < tiles_y; t++) {
        const int by = min(t * TH + warp, bh - 1);
        const bool in_y = t * TH + warp < bh;
        const int row0 = __ldg(ytile + t).x;                            // first source row staged for this tile
        const int ys = __ldg(yofs + by);
        const int r0 = min(max(ys, 0), sh - 1) - row0, r1 = min(max(ys + 1, 0), sh - 1) - row0;
        const short* yb = reinterpret_cast<const short*>(blob + P->ycoef_off);
        const int b0 = __ldg(yb + by * 2), b1 = __ldg(yb + by * 2 + 1);
        mbar_wait_a(full_a + stage * 8, phase);
        const uint8_t* sbase = tile0 + stage * stage_bytes;
        int v[SC];
        IMP_DBG(r0 >= 0 && r0 < P->tile_rows && xo0 >= 0 && xo0 + SC <= rs && (r1 >= 0 && r1 < P->tile_rows && xo1 >= 0 && xo1 + SC <= rs), 10);
        const uint8_t* q0 = sbase + r0 * rs; const uint8_t* q1 = sbase + r1 * rs;
        int p00[SC], p01[SC], p10[SC], p11[SC];
        if (SC == 4) {
            const uint32_t w00 = *reinterpret_cast<const uint32_t*>(q0 + xo0), w01 = *reinterpret_cast<const uint32_t*>(q0 + xo1);
            const uint32_t w10 = *reinterpret_cast<const uint32_t*>(q1 + xo0), w11 = *reinterpret_cast<const uint32_t*>(q1 + xo1);
#pragma unroll
            for (int c = 0; c < SC; c++) { p00[c] = (w00 >> (8 * c)) & 255; p01[c] = (w01 >> (8 * c)) & 255; p10[c] = (w10 >> (8 * c)) & 255; p11[c] = (w11 >> (8 * c)) & 255; }
        } else {
#pragma unroll
            for (int c = 0; c < SC; c++) { p00[c] = q0[xo0 + c]; p01[c] = q0[xo1 + c]; p10[c] = q1[xo0 + c]; p11[c] = q1[xo1 + c]; }
        }
#pragma unroll
        for (int c = 0; c < SC; c++) {                                  // SURVEY App. A.4 / imp_gather_linear
            const int h0 = p00[c] * a0 + p01[c] * a1, h1 = p10[c] * a0 + p11[c] * a1;
            v[c] = ((((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2) & 255;
        }
        // every lane's loads must have been performed before lane 0 hands the stage back to the TMA producer
        fence_generic_to_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive_a(empty_a + stage * 8);             // this warp is done with the stage
        if (in_x && in_y) strip_epilogue<SC, FL>(job, oc, dc, st, orows, s_ops, nops, bx, by, v);
        if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
    }
}

// LIGHT: the pass has no ops or only fused tables (ImpPass::light — every plain resize): the instantiation without the general
// op interpreter fits 56 registers, so four CTAs share an SM instead of three.
// FL 2: compositing ops and fused tables only ("resize + watermark", cfg2 / cfg5): the interpreter without the HSV code.
template <int SC, int MODE, int FL>
__global__ void __launch_bounds__(STRIP_THREADS, (FL == 1 && MODE != 0) ? 4 : 3)      // the fractional mode keeps 12 x weights in registers: 72
imp_strip_kernel(const ImpJob* __restrict__ jobs, int first, int count, const __grid_constant__ ImpJob one, const int NSTAGE) {
    extern __shared__ __align__(128) uint8_t smem[];
    const int jn = blockIdx.y + blockIdx.z * 65535;
    if (jn >= count) return;
    const ImpJob* __restrict__ jp = jobs ? jobs + first + jn : &one;
    ImpJob job;                                                        // everything but the tensor map
    job.src = jp->src; job.dst = jp->dst; job.pass = jp->pass; job.wm = jp->wm;
    job.src_pitch = jp->src_pitch; job.dst_pitch = jp->dst_pitch; job.wm_pitch = jp->wm_pitch; job.wm_c = jp->wm_c; job.tm_x0 = jp->tm_x0;
    const uint8_t* __restrict__ blob = job.pass;
    const ImpPass* __restrict__ P = reinterpret_cast<const ImpPass*>(blob);
    const int bw = P->bw, bh = P->bh;
    const int tiles_x = (bw + TW - 1) / TW, tiles_y = (bh + TH - 1) / TH;
    if ((int)blockIdx.x >= tiles_x) return;

    uint64_t* full = reinterpret_cast<uint64_t*>(smem);               // [NSTAGE]
    uint64_t* empty = full + NSTAGE;                                  // [NSTAGE]
    const int nops = P->nops;
    const int ops_bytes = (nops * (int)sizeof(ImpOp) + P->lut_bytes + 15) & ~15;
    uint8_t* s_ops = smem + 128;                                      // up to 8 stages: 16 mbarriers
    uint8_t* tile0 = s_ops + ((ops_bytes + 127) & ~127);              // 128-byte aligned
    const int rs = P->tile_rs;
    // stage = [pixel box][y taps of the tile][y ranges of its 8 output rows] (the last two only in fractional mode)
    const int ytap_bytes = (MODE == 0) ? ((P->tile_ytaps * 8 + 15) & ~15) : 0;
    const int stage_bytes = (rs * P->tile_rows + ytap_bytes + (MODE == 0 ? 128 : 0) + 127) & ~127;
    const int tid = threadIdx.x;
    if (tid == 0) {
        for (int i = 0; i < NSTAGE; i++) { mbar_init(full + i, 1); mbar_init(empty + i, TH); }
    }
    {
        const uint4* gsrc = reinterpret_cast<const uint4*>(blob + P->ops_off);
        uint4* sdst = reinterpret_cast<uint4*>(s_ops);
        for (int i = tid; i < ops_bytes / 16; i += STRIP_THREADS) sdst[i] = __ldg(gsrc + i);
    }
    // x placement of this strip inside the tensor map (8-byte elements)
    const int px0 = __ldg(reinterpret_cast<const int2*>(blob + P->xtile_off) + blockIdx.x).x;     // first source pixel of the strip
    const int xbyte = job.tm_x0 + px0 * SC;                           // its byte offset in the map's row
    const int c0 = (xbyte >> 4) << 1;                                 // element coordinate of the box; TMA wants the box origin 16-byte aligned
    __syncthreads();

    if (tid >= STRIP_CONSUMERS) {
        // ---- TMA producer: one elected thread, one instruction per tile ----
        if (tid == STRIP_CONSUMERS) {
            const int4* __restrict__ ytile = reinterpret_cast<const int4*>(blob + P->ytile_off);
            const uint8_t* __restrict__ g_yt = blob + P->ycoef_off;
            const uint8_t* __restrict__ g_yr = blob + P->yrow4_off;
            const uint32_t box_bytes = (uint32_t)(rs * P->tile_rows);
            int stage = 0, phase = 0;
            for (int t = 0; t < tiles_y; t++) {
                const int4 yt4 = __ldg(ytile + t);                       // {first source row, rows, first y tap, y taps}
                mbar_wait(empty + stage, phase ^ 1);
                uint8_t* sdst = tile0 + stage * stage_bytes;
                if (MODE == 0) {
                    // the tile's y taps and row ranges ride along as two small bulk copies, so the consumers' inner
                    // loops never leave shared memory
                    const int tapbase = yt4.z & ~1;
                    const uint32_t tapbytes = (uint32_t)(((yt4.w + (yt4.z & 1)) * 8 + 15) & ~15);
                    mbar_expect_tx(full + stage, box_bytes + tapbytes + 128u);
                    tma_load_2d(sdst, jp->tmap, c0, yt4.x, full + stage);
                    bulk_g2s(sdst + box_bytes, g_yt + (size_t)tapbase * 8, tapbytes, full + stage);
                    bulk_g2s(sdst + box_bytes + ytap_bytes, g_yr + (size_t)t * TH * 16, 128u, full + stage);
                } else {
                    mbar_expect_tx(full + stage, box_bytes);
                    tma_load_2d(sdst, jp->tmap, c0, yt4.x, full + stage);
                }
                if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
            }
        }
        return;
    }
    // ---- consumers ----
    const int col_off = job.tm_x0 - c0 * 8;                           // tile byte offset of source pixel 0
    const int bx0 = blockIdx.x * TW;
    if constexpr (MODE == 3) {
        linear_strip_consume<SC, FL>(job, P, blob, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE);
    } else if constexpr (MODE == 0) {
        switch (P->max_xtaps) {                                       // uniform over the pass
        case 1: area_strip_consume<SC, 1, 0, FL>(job, P, blob, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        case 2: area_strip_consume<SC, 2, 0, FL>(job, P, blob, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        case 3: area_strip_consume<SC, 3, 0, FL>(job, P, blob, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        case 4: area_strip_consume<SC, 4, 0, FL>(job, P, blob, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        case 5: area_strip_consume<SC, 5, 0, FL>(job, P, blob, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        case 6: area_strip_consume<SC, 6, 0, FL>(job, P, blob, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        case 7: area_strip_consume<SC, 7, 0, FL>(job, P, blob, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        case 8: area_strip_consume<SC, 8, 0, FL>(job, P, blob, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        case 9: area_strip_consume<SC, 9, 0, FL>(job, P, blob, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        case 10: area_strip_consume<SC, 10, 0, FL>(job, P, blob, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        case 11: area_strip_consume<SC, 11, 0, FL>(job, P, blob, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        default: area_strip_consume<SC, 12, 0, FL>(job, P, blob, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        }
    } else {
        switch (P->nx) {
        case 1: area_int_strip_consume<SC, 1, FL>(job, P, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        case 2: area_int_strip_consume<SC, 2, FL>(job, P, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        case 3: area_int_strip_consume<SC, 3, FL>(job, P, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        case 4: area_int_strip_consume<SC, 4, FL>(job, P, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        case 5: area_int_strip_consume<SC, 5, FL>(job, P, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        case 6: area_int_strip_consume<SC, 6, FL>(job, P, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        case 7: area_int_strip_consume<SC, 7, FL>(job, P, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        case 8: area_int_strip_consume<SC, 8, FL>(job, P, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        case 9: area_int_strip_consume<SC, 9, FL>(job, P, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        case 10: area_int_strip_consume<SC, 10, FL>(job, P, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        case 11: area_int_strip_consume<SC, 11, FL>(job, P, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        default: area_int_strip_consume<SC, 12, FL>(job, P, tile0, stage_bytes, full, empty, s_ops, nops, bx0, col_off, tiles_y, NSTAGE); break;
        }
    }
}

// Copies `rows` rows of `row_bytes` bytes from a shared-memory stage (row stride `ss`, a multiple of 16, stage 16-byte
// aligned) to global rows: 16 bytes per thread when the destination rows are 16-byte addressable (the library's own
// buffers always are), 4 bytes or single bytes otherwise. Consecutive threads write consecutive chunks of a row.
__device__ __forceinline__ void tile_copy_out(const uint8_t* s, int ss, uint8_t* d, int dp, int row_bytes, int rows, int tid, int nt) {
    const unsigned mis = (unsigned)(reinterpret_cast<uintptr_t>(d) | (unsigned)dp);
    if ((mis & 15) == 0 && row_bytes <= 256) {
        // rows of up to 16 chunks: chunk slots padded to a power of two, so (row, chunk) come from a shift and a mask
        const int nch = row_bytes >> 4, tail = row_bytes & 15;
        const int sl = nch <= 2 ? 1 : nch <= 4 ? 2 : nch <= 8 ? 3 : 4;
        for (int i = tid; i < (rows << sl); i += nt) {
            const int ry = i >> sl, ch = i & ((1 << sl) - 1);
            if (ch >= nch) continue;
            *reinterpret_cast<uint4*>(d + (size_t)ry * dp + 16 * ch) = *reinterpret_cast<const uint4*>(s + ry * ss + 16 * ch);
        }
        if (tail) for (int i = tid; i < rows * tail; i += nt) {
            const int ry = i / tail, b = (nch << 4) + i - ry * tail;
            d[(size_t)ry * dp + b] = s[ry * ss + b];
        }
    } else if ((mis & 3) == 0) {
        const int nch = row_bytes >> 2, tail = row_bytes & 3;
        for (int i = tid; i < rows * nch; i += nt) {
            const int ry = i / nch, ch = i - ry * nch;
            *reinterpret_cast<uint32_t*>(d + (size_t)ry * dp + 4 * ch) = *reinterpret_cast<const uint32_t*>(s + ry * ss + 4 * ch);
        }
        for (int i = tid; i < rows * tail; i += nt) {
            const int ry = i / tail, b = (nch << 2) + i - ry * tail;
            d[(size_t)ry * dp + b] = s[ry * ss + b];
        }
    } else {
        for (int i = tid; i < rows * row_bytes; i += nt) {
            const int ry = i / row_bytes, b = i - ry * row_bytes;
            d[(size_t)ry * dp + b] = s[ry * ss + b];
        }
    }
}

// Same for a stage whose rows are only 4-byte aligned (row stride `ss` a multiple of 4, odd in words: see imp_blur.cuh):
// a 16-byte global chunk is assembled from four 32-bit shared loads.
__device__ __forceinline__ void tile_copy_out_w(const uint8_t* s, int ss, uint8_t* d, int dp, int row_bytes, int rows, int tid, int nt) {
    const unsigned mis = (unsigned)(reinterpret_cast<uintptr_t>(d) | (unsigned)dp);
    if ((mis & 15) == 0 && row_bytes <= 256) {
        // rows of up to 16 chunks: chunk slots padded to a power of two, so (row, chunk) come from a shift and a mask
        const int nch = row_bytes >> 4, tail = row_bytes & 15;
        const int sl = nch <= 2 ? 1 : nch <= 4 ? 2 : nch <= 8 ? 3 : 4;
        for (int i = tid; i < (rows << sl); i += nt) {
            const int ry = i >> sl, ch = i & ((1 << sl) - 1);
            if (ch >= nch) continue;
            const uint32_t* q = reinterpret_cast<const uint32_t*>(s + ry * ss + 16 * ch);
            *reinterpret_cast<uint4*>(d + (size_t)ry * dp + 16 * ch) = make_uint4(q[0], q[1], q[2], q[3]);
        }
        if (tail) for (int i = tid; i < rows * tail; i += nt) {
            const int ry = i / tail, b = (nch << 4) + i - ry * tail;
            d[(size_t)ry * dp + b] = s[ry * ss + b];
        }
    } else if ((mis & 3) == 0) {
        const int nch = row_bytes >> 2, tail = row_bytes & 3;
        for (int i = tid; i < rows * nch; i += nt) {
            const int ry = i / nch, ch = i - ry * nch;
            *reinterpret_cast<uint32_t*>(d + (size_t)ry * dp + 4 * ch) = *reinterpret_cast<const uint32_t*>(s + ry * ss + 4 * ch);
        }
        for (int i = tid; i < rows * tail; i += nt) {
            const int ry = i / tail, b = (nch << 2) + i - ry * tail;
            d[(size_t)ry * dp + b] = s[ry * ss + b];
        }
    } else {
        for (int i = tid; i < rows * row_bytes; i += nt) {
            const int ry = i / row_bytes, b = i - ry * row_bytes;
            d[(size_t)ry * dp + b] = s[ry * ss + b];
        }
    }
}

}  // namespace imp_tiles
