// imp_plan.h — structures shared by the host planner and the device kernels.
//
// A request (crop / resize / filter list / watermark / flatten; RunJob steps 3-7, bridge.c:574-656) is
// lowered on the host into 1..n PASSES. Pass 0 gathers from the decoded frame (crop folded into the
// source addressing, resize as the gather); every Gaussian blur (filters.c:192-207) starts a new pass
// whose gather is the stencil. All other filters, the watermark and the paper-flatten are pointwise
// OPS executed in registers between a pass's gather and its store, so a blur-free request is a single
// kernel and each frame makes one HBM round trip.
//
// Geometry filters (flip, rotate; filters.c:72-133) never move pixels by themselves: all passes work
// in the orientation of the BASE frame (the frame right after crop+resize). Each coordinate-dependent
// op carries the map base(x,y) -> its own frame, and the last pass applies the accumulated map when
// storing. This is exact because the Gaussian kernel is symmetric and sigma_x == sigma_y, so blur
// commutes with the eight flips/transposes.
#pragma once
#include <stdint.h>

enum ImpGather : int {
    IMP_G_COPY = 0,       // index map only (crop / no resize)
    IMP_G_NN,             // cvResize CV_INTER_NN        (SURVEY App. A.1)
    IMP_G_AREA_INT,       // cvResize CV_INTER_AREA, integer scales (A.2)
    IMP_G_AREA_FRAC,      // cvResize CV_INTER_AREA, generic        (A.3)
    IMP_G_CUBIC,          // cvResize CV_INTER_CUBIC     (A.4)
    IMP_G_LINEAR,         // cv::INTER_LINEAR extension  (A.4)
    IMP_G_BLUR,           // cvSmooth CV_GAUSSIAN        (A.5)
    IMP_G_COUNT
};

enum ImpOpKind : int {
    IMP_OP_MODULATE = 1,  // ModulateHSV filters.c:524-547
    IMP_OP_ADDCOLOR,      // AlphaBlendAddColor filters.c:608-616
    IMP_OP_LUT_ALL,       // ApplyGamma filters.c:549-559 (every channel, alpha too)
    IMP_OP_CONTRAST,      // BrightnessContrast filters.c:595-605
    IMP_OP_GRADMAP,       // Gradmap filters.c:260-277
    IMP_OP_VIGNETTE,      // Vignette filters.c:295-323 + RadialGradient :693-703
    IMP_OP_LOMO,          // Lomo filters.c:335-346
    IMP_OP_RAINBOW,       // Rainbow filters.c:356-403
    IMP_OP_SCANLINE,      // Scanline filters.c:405-455
    IMP_OP_WATERMARK,     // Watermark bridge.c:239-281 + AlphaBlendOver filters.c:619-662
    IMP_OP_PAPER,         // BlendWithPaper filters.c:666-687
    // planner-made (imp_planner.cpp "fusion of channel-separable ops"): a run of AlphaBlendAddColor / ApplyGamma /
    // BrightnessContrast / Lomo composed into one table per channel; i[0] = LUT offset of u8[3 or 4][256] (B,G,R[,A]),
    // i[1] = 1 when the alpha table is present and to be applied
    IMP_OP_LUT3,          // c = tab[c][c]
    IMP_OP_MAXLUT3,       // c = tab[c][max(B,G,R)] (a saturation-0 ModulateHSV opened the run); alpha: tab[3][A]
};

// base-frame (x,y) -> coordinates in another frame of size w x h:
//   (u,v) = swap ? (y,x) : (x,y);  X = flipx ? w-1-u : u;  Y = flipy ? h-1-v : v
struct ImpFrameMap {
    int swap, flipx, flipy, w, h;
};

struct ImpOp {                // 64 bytes
    int   kind;
    int   i[6];
    float f[4];
    ImpFrameMap map;          // frame the op sees (vignette, scanline, watermark)
};

#define IMP_MAX_OPS 48

// One pass, as the kernels see it. Lives at offset 0 of the pass blob in device memory; every *_off
// is a byte offset into that blob (0 = absent).
struct ImpPass {
    int kind;                 // ImpGather
    int sc;                   // channels of the pass input (1, 3 or 4)
    int oc;                   // channels the ops and the store see (3 or 4; 1 only when sc==1 and gray is kept)
    int sx0, sy0;             // origin of the source window inside the input image (crop), pixels
    int sw, sh;               // size of the source window == clamp bounds of the gather
    int bw, bh;               // base-frame size == the gather's output size
    int nx, ny;               // AREA_INT block size
    int ksize;                // CUBIC 4 / LINEAR 2 ; BLUR: tap count n
    int simd_end;             // CUBIC: bytes of a row handled by OpenCV's float path (A.4)
    float area_scale;         // AREA_INT: f32(1/(nx*ny))
    int xofs_off, xcoef_off;  // NN: xofs[bw]; CUBIC/LINEAR: xofs[bw], short xcoef[bw*ksize];
    int yofs_off, ycoef_off;  // AREA_FRAC: int2 range[b] (first tap, count) + coef = {int si; float a}[taps]
    int taps_off;             // BLUR: int taps[n]; CUBIC: float ycoef[bh*4] = short coefficient * 2^-22 (exact)
    int blur_r;               // BLUR tile kernel: padded tap radius (3, 6, 9 or 12); 0 = generic two-launch path only
    int tapsr_off;            // BLUR tile kernel: int taps[2*blur_r+1] (zero taps trimmed, then zero-padded symmetrically)
    int taph_off, tapv_off;   // BLUR tile kernel: the same taps as u8 dot-product words: u32 taph[4][NWH] (dp4a, four byte
                              // alignments), u32 tapv[2][NWV] (dp2a, two parities); ImpBlurDims<R> below
    int max_xtaps, max_ytaps; // AREA_FRAC: largest tap count per output column / row
    int tile_rs, tile_rows;   // tile kernels: shared-memory row stride (bytes) and max source rows per 32x8 tile
    int tile_smem;            // tile kernels: source-tile bytes (tile_rs*tile_rows); 0 = no tile kernel for this pass
    int xtile_off, ytile_off; // tile kernels: int2 per tile column {first px, last px}; int4 per tile row {first src row, rows, first y tap, y taps}
    int light;                // bit 0: every op of the pass is a fused table (IMP_OP_LUT3 / IMP_OP_MAXLUT3) or there is none: the strip,
                              // gather and cubic kernels then run an instantiation whose op interpreter knows only those two (fewer
                              // registers, more CTAs per SM); bit 1: no compositing op (watermark, paper): the blur kernel's flavour; bit 2: nothing but
                              // compositing ops and fused tables ("resize + watermark"): the strip kernels' flavour without the HSV code
    int gt;                   // gather tile kernel (imp_gathertile.cuh; COPY / NN / LINEAR): destination tile edge, 64 or 32; 0 = none
    int tile_ytaps;           // strip kernel: y-tap entries staged per tile (max over tiles, incl. alignment slack)
    int yrow4_off;            // strip kernel: int4 per output row {byte offset of its first source row inside the tile, y taps, index of its first tap in the tile's staged taps, 0}
    int nops;
    int ops_off;              // ImpOp[nops]
    int lut_off, lut_bytes;   // LUT area (gamma 256 B each, gradmap 768 B each)
    ImpFrameMap out;          // base (x,y) -> destination pixel
    int dc;                   // destination channels (== oc)
    int blob_bytes;
};

// Geometry of the fused blur tile kernel (imp_blur.cuh), shared with the planner (tap tables, TMA box) and the runtime
// (shared-memory size). A CTA blurs a BTW x BTH tile of the base frame with taps padded to radius R.
// imp_cubic.cuh: floats per row of the horizontal-pass buffer of a T-wide tile (+4 / +1: bank spread), and the launch's
// dynamic shared memory: [bar 128][ops][TMA box][hbuf rows x HRS floats][T x {int4, float4} row lookups][T x T*3 out stage]
// Columns are stored group-transposed — column lx at position (lx & 3) * (T/4 + 1) + (lx >> 2) — so that the vertical pass,
// where a thread owns columns 4t .. 4t+3, reads consecutive positions across a warp (conflict-free), hence T + 4 positions
// per row; the row stride is 4 mod 32 words (float4 rows of 8 lanes spread over all banks) or odd.
#define IMP_CUBIC_HRS(sc, T) ((sc) == 4 ? ((T) + 4) * 4 + 20 : ((T) + 4) * (sc) + 1)
#define IMP_CUBIC_POS(lx, T) (((lx) & 3) * ((T) / 4 + 1) + ((lx) >> 2))
inline int imp_cubic_dyn_smem(int sc, int ops_bytes16, int tile_rs, int tile_rows, int T, int dc) {
    return 128 + ((ops_bytes16 + 127) & ~127) + ((tile_rs * tile_rows + 127) & ~127) + ((tile_rows * IMP_CUBIC_HRS(sc, T) * 4 + 15) & ~15) + T * 32 +
           (dc == 4 ? 0 : T * T * 3) + 64;
}
// imp_gathertile.cuh: [bar 128][ops][TMA box][6*T lookup words][T rows of T*3 bytes: out stage of 3-channel results]
#define IMP_GATHER_TPC 4      // consecutive tiles one CTA walks (two TMA boxes: the next tile's is in flight)
inline int imp_gather_dyn_smem(int gt, int ops_bytes16, int tile_rs, int tile_rows, int dc) {
    return 128 + ((ops_bytes16 + 127) & ~127) + 2 * ((tile_rs * tile_rows + 127) & ~127) + 6 * gt * 4 + (dc == 4 ? 0 : gt * gt * 3) + 64;
}
// vignette mask table: entries beyond the frame's largest |dx|, |dy| (>= the tile kernels' overhang: 64)
#define IMP_VIGNETTE_MARGIN 64
#define IMP_BLUR_TW 32
#define IMP_BLUR_TH 64
template <int R> struct ImpBlurDims {
    static constexpr int SPANX = IMP_BLUR_TW + 2 * R, SPANY = IMP_BLUR_TH + 2 * R;   // source neighbourhood
    static constexpr int NWH = (2 * R + 4 + 3) / 4;           // tap words per byte alignment (2R+1 taps shifted by up to 3)
    static constexpr int NWIN = NWH + 1;                      // planar words a thread loads for 8 adjacent outputs
    static constexpr int PWW = (6 + NWIN) | 1;                // planar row stride in words: covers SPANX bytes, odd (banks)
    static constexpr int NDV = R + 1;                         // dp2a per output: ceil((2R+1 taps + 1 parity shift) / 2)
    static constexpr int NWV = (NDV + 1) / 2;                 // tap words per parity (one word feeds a dp2a.lo and a dp2a.hi)
    static constexpr int NV128 = (8 + 2 * R + 7) / 8;         // 16-byte loads covering the 8+2R u16 window of 8 outputs
    static constexpr int HNEED = SPANY > IMP_BLUR_TH - 8 + 8 * NV128 ? SPANY : IMP_BLUR_TH - 8 + 8 * NV128;
    static constexpr int HS = ((HNEED - 8 + 15) & ~15) + 8;   // u16 row stride of the transposed sums: % 16 == 8 (banks)
    static constexpr int planar_bytes(int sc) { return (sc * SPANY * PWW * 4 + 127) & ~127; }
    static constexpr int hbuf_bytes(int sc) { return sc * IMP_BLUR_TW * HS * 2; }
};
inline int imp_blur_dyn_smem(int sc, int r, int ops_bytes16, int tile_rs) {
    const int spany = IMP_BLUR_TH + 2 * r;
    int planar = 0, hbuf = 0;
    switch (r) {
        case 3:  planar = ImpBlurDims<3>::planar_bytes(sc);  hbuf = ImpBlurDims<3>::hbuf_bytes(sc);  break;
        case 6:  planar = ImpBlurDims<6>::planar_bytes(sc);  hbuf = ImpBlurDims<6>::hbuf_bytes(sc);  break;
        case 9:  planar = ImpBlurDims<9>::planar_bytes(sc);  hbuf = ImpBlurDims<9>::hbuf_bytes(sc);  break;
        default: planar = ImpBlurDims<12>::planar_bytes(sc); hbuf = ImpBlurDims<12>::hbuf_bytes(sc); break;
    }
    return 128 + ((ops_bytes16 + 127) & ~127) + ((tile_rs * spany + 127) & ~127) + planar + hbuf + 64;
}

// One job of a batch: which pass blob, where the pixels are.
struct ImpJob {
    const uint8_t* src;       // input image of this pass (top-left of the whole image, not of the window)
    uint8_t*       dst;
    const uint8_t* pass;      // device pointer to the ImpPass blob
    const uint8_t* wm;        // watermark pixels on this device (or null)
    int src_pitch, dst_pitch, wm_pitch, wm_c;
    int tm_x0;                // strip kernels: byte offset of the source window's first pixel inside the tensor map's row
    int pad_[15];
    // strip kernels: CUtensorMap (2-D, 8-byte elements) over the 16-byte aligned source window of this job, so the
    // TMA engine fetches a whole tile (box = tile_rs bytes x tile_rows rows) with ONE instruction.
    alignas(64) unsigned char tmap[128];
};

// One GIF frame as the producer of the hot path sees it (advancedio.c:126-186): palette indices in FreeImage scanline
// order (bottom-up), placement on the canvas, disposal and transparency key, palette as RGBQUAD (B,G,R,x).
struct ImpGifFrame {
    const uint8_t* indices;   // device pointer
    const uint8_t* palette;   // device pointer, 256 * 4 bytes
    int pitch, w, h, left, top, dispose, key, pad_;
};
