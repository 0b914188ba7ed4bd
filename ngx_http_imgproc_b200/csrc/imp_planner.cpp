// imp_planner.cpp — host side of the drop-in: the reference's argument grammar and validation
// (Crop bridge.c:18-128, Resize bridge.c:143-190, Filter + callbacks filters.c:43-455, Watermark
// placement bridge.c:254-274) restated so that every request yields the SAME return code at the SAME
// RunJob step as the reference, and the lowering of a valid request into kernel passes (imp_plan.h).
//
// Nothing here touches pixels. Tables the kernels need (resize taps, Gaussian taps, gamma / gradient
// LUTs, alpha constants) are computed here in C with the same libm and double/float sequence the
// reference and OpenCV use, so no pow/exp/division-by-table ever runs on the device.
//
// Deliberate deviations (all turn a reference crash/UB into IMP_ERROR_INVALID_ARGS; SURVEY App. C):
//   C-4  gradmap with <2 or >8 colours            (uninitialised LUT / heap overflow in the reference)
//   C-8  watermark ROI empty after clipping       (OpenCV assert in the reference)
//   C-9  blur sigma == 0                          (OpenCV assert)
//   C-10 scanline with no argument token          (NULL dereference)
//   crop/gravity offsets that are negative or a gravity string with fewer than two tokens (OpenCV
//   assert / strcmp(NULL)); resize to a zero-sized target (cvCreateImage error).
// Two more differences from "same code at the same step", both on purpose (DESIGN.md §6):
//   * Crop tokenises `gravity` in place (bridge.c:73): frames 2.. of a multi-frame GIF then see a string of <= 2 characters
//     and fail with INVALID_ARGS at the crop step. Here every frame of a job sees the same string and succeeds.
//   * no cap on the op count of a pass surfaces as an error: a chain longer than IMP_MAX_OPS (or with more tables than a
//     pass's shared memory takes) continues in an index-map pass (Lower::reserve_op), as the reference would accept it.
#include "imp_internal.h"
#include "imp_pixel.cuh"            // host instantiation of the per-pixel ops: composed LUTs are tabulated with the very code the kernels run
#include <math.h>
#include <float.h>
#include <limits.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <mutex>

// ---- overlay registry: one shared image per distinct watermark content -----------------------------------------
void (*imp_wm_dev_release)(ImpWmImage*) = nullptr;
ImpWmImage::~ImpWmImage() { if (imp_wm_dev_release) imp_wm_dev_release(this); }

namespace {
std::mutex g_wm_mu;
std::vector<std::shared_ptr<ImpWmImage>> g_wm_registry;     // most recently used last
constexpr size_t kWmRegistryCap = 32;

unsigned long long hash_bytes(unsigned long long h, const uint8_t* p, size_t n) {
    // 8 bytes per step (multiply-xorshift); collisions are harmless: a hit is confirmed with memcmp
    size_t i = 0;
    for (; i + 8 <= n; i += 8) { unsigned long long v; memcpy(&v, p + i, 8); h = (h ^ v) * 0x9E3779B97F4A7C15ull; h ^= h >> 29; }
    for (; i < n; i++) { h = (h ^ p[i]) * 0x100000001B3ull; }
    return h;
}
}  // namespace

std::shared_ptr<ImpWmImage> imp_wm_intern(const imp_gpu_watermark* wm) {
    const size_t row = (size_t)wm->width * wm->channels;
    unsigned long long h = 0xcbf29ce484222325ull ^ ((unsigned long long)wm->width << 40) ^ ((unsigned long long)wm->height << 16) ^ (unsigned)wm->channels;
    for (int y = 0; y < wm->height; y++) h = hash_bytes(h, wm->pixels + (size_t)y * wm->step, row);
    std::lock_guard<std::mutex> lk(g_wm_mu);
    for (size_t i = g_wm_registry.size(); i-- > 0;) {
        const std::shared_ptr<ImpWmImage>& e = g_wm_registry[i];
        if (e->hash != h || e->w != wm->width || e->h != wm->height || e->c != wm->channels) continue;
        bool same = true;
        for (int y = 0; y < wm->height && same; y++) same = memcmp(e->pixels.data() + (size_t)y * row, wm->pixels + (size_t)y * wm->step, row) == 0;
        if (!same) continue;
        std::shared_ptr<ImpWmImage> hit = e;
        if (i + 1 != g_wm_registry.size()) { g_wm_registry.erase(g_wm_registry.begin() + i); g_wm_registry.push_back(hit); }
        return hit;
    }
    auto img = std::make_shared<ImpWmImage>();
    img->w = wm->width; img->h = wm->height; img->c = wm->channels; img->hash = h;
    img->pixels.resize(row * wm->height);
    for (int y = 0; y < wm->height; y++) memcpy(img->pixels.data() + (size_t)y * row, wm->pixels + (size_t)y * wm->step, row);
    if (g_wm_registry.size() >= kWmRegistryCap) g_wm_registry.erase(g_wm_registry.begin());   // plans keep theirs alive
    g_wm_registry.push_back(img);
    return img;
}

void imp_wm_registry_clear() {
    std::vector<std::shared_ptr<ImpWmImage>> drop;
    { std::lock_guard<std::mutex> lk(g_wm_mu); drop.swap(g_wm_registry); }
}

// ---- launch choice (the runtime picks `tiled` or `fallback` per job: imp_gpu.cu, pick_launch) ---------------------------
ImpLaunch imp_pass_launch(const ImpPass& h, ImpKernel k) {
    const int ops16 = (h.nops * (int)sizeof(ImpOp) + h.lut_bytes + 15) & ~15;
    ImpLaunch l{k, 0, 0, std::max(16, h.nops * (int)sizeof(ImpOp) + h.lut_bytes), 0, 0};     // the direct kernels stage only the ops
    switch (k) {
        case ImpKernel::BlurGeneric: break;
        case ImpKernel::Direct: l.ctas_per_job = ((h.bw + 31) / 32) * ((h.bh + 31) / 32); break;
        case ImpKernel::CubicRun: l.ctas_per_job = ((h.bw + 31) / 32) * ((h.bh + 8 * IMP_CUBIC_RUN - 1) / (8 * IMP_CUBIC_RUN)); break;
        case ImpKernel::Strip: {
            // one ring stage: the source box (+ the staged y taps and the 8 rows' int4 descriptors of fractional AREA)
            const int extra = h.kind == IMP_G_AREA_FRAC ? (((h.tile_ytaps * 8 + 15) & ~15) + 128) : 0;
            const int stage = (h.tile_smem + extra + 127) & ~127;
            // The table-ops-only instantiation runs four CTAs per SM (56 registers), the others three. Ring depth: as many
            // stages as fit 72 KB (three CTAs of 72 KB + ops still share an SM's 227 KB; 54 KB for four), between 2 and 8.
            // Small tiles (cfg1: 7 KB) need the depth to keep enough bytes in flight; cfg2's 23.7 KB stage gets 3 (1.5 % over 2).
            const bool four = (h.light & 1) && h.kind != IMP_G_AREA_FRAC;
            l.param = std::max(2, std::min(8, ((four ? 54 : 72) * 1024) / stage));
            l.flavour = (h.light & 1) ? 1 : (h.light & 4) ? 2 : 0;
            l.smem_bytes = 128 + ((ops16 + 127) & ~127) + l.param * stage + 64;      // +64: padded taps past the last row
            l.ctas_per_job = (h.bw + 31) / 32;                                          // strips (tile columns)
            // A launch takes the largest footprint of its group, so strip jobs are grouped by this class as well: a few big
            // tiles must not drag thousands of small ones down to two CTAs per SM.
            l.ctas_per_sm = std::max(1, std::min(four ? 4 : 3, (227 * 1024) / (l.smem_bytes + 1024)));
        } break;
        case ImpKernel::BlurTile:
            l.param = h.blur_r;
            l.flavour = (h.light >> 1) & 1;
            l.smem_bytes = imp_blur_dyn_smem(h.sc, h.blur_r, ops16, h.tile_rs);
            l.ctas_per_job = ((h.bw + IMP_BLUR_TW - 1) / IMP_BLUR_TW) * ((h.bh + IMP_BLUR_TH - 1) / IMP_BLUR_TH);    // same count in destination space
            break;
        case ImpKernel::CubicTile:
            l.param = h.gt;
            l.flavour = h.light & 1;
            l.smem_bytes = imp_cubic_dyn_smem(h.sc, ops16, h.tile_rs, h.tile_rows, h.gt, h.dc);
            l.ctas_per_job = ((h.bw + h.gt - 1) / h.gt) * ((h.bh + h.gt - 1) / h.gt);                          // same count in destination space
            break;
        case ImpKernel::GatherTile:
            l.param = h.gt;
            l.flavour = h.light & 1;
            l.smem_bytes = imp_gather_dyn_smem(h.gt, ops16, h.tile_rs, h.tile_rows, h.dc);
            l.ctas_per_job = (((h.bw + h.gt - 1) / h.gt) * ((h.bh + h.gt - 1) / h.gt) + IMP_GATHER_TPC - 1) / IMP_GATHER_TPC;   // IMP_GATHER_TPC tiles each
            break;
    }
    return l;
}

void imp_pass_launches(const ImpPass& h, ImpLaunch* tiled, ImpLaunch* fallback) {
    const ImpKernel fb = h.kind == IMP_G_CUBIC ? ImpKernel::CubicRun : h.kind == IMP_G_BLUR ? ImpKernel::BlurGeneric : ImpKernel::Direct;
    ImpKernel k = fb;
    if (h.tile_smem > 0) {
        if (h.kind == IMP_G_CUBIC) k = ImpKernel::CubicTile;
        else if (h.gt > 0) k = ImpKernel::GatherTile;
        else if (h.kind == IMP_G_BLUR) k = h.blur_r > 0 ? ImpKernel::BlurTile : fb;
        else if (h.kind != IMP_G_COPY && h.kind != IMP_G_NN) k = ImpKernel::Strip;
    }
    *fallback = imp_pass_launch(h, fb);
    *tiled = imp_pass_launch(h, k);
    if (tiled->smem_bytes > IMP_SMEM_OPTIN) *tiled = *fallback;
}

namespace {

// ---- C-library-faithful helpers ---------------------------------------------------------------------
// strtok_r semantics: separators collapse, no empty tokens.
std::vector<std::string> tokens(const char* s, char sep) {
    std::vector<std::string> out;
    if (!s) return out;
    const char* p = s;
    while (*p) {
        while (*p == sep) p++;
        if (!*p) break;
        const char* q = p;
        while (*q && *q != sep) q++;
        out.emplace_back(p, q - p);
        p = q;
    }
    return out;
}

struct Num { long v; std::string rest; };
Num parse_long(const std::string& s, int base = 10) {
    char* end = nullptr;
    long v = strtol(s.c_str(), &end, base);
    return Num{v, std::string(end)};
}
float parse_float(const std::string& s) { return strtof(s.c_str(), nullptr); }

// (int)x for double x as x86-64 cvttsd2si does it.
int d2i_x86(double v) { return (v > -2147483649.0 && v < 2147483648.0) ? (int)v : INT_MIN; }
int f2i_x86(float v) { return (v > -2147483904.0f && v < 2147483648.0f) ? (int)v : INT_MIN; }

// ---- frame-map algebra (imp_plan.h) -----------------------------------------------------------------
struct Frame {
    int w, h, c;
    int swap = 0, fx = 0, fy = 0;            // base -> this frame
    ImpFrameMap map() const { return ImpFrameMap{swap, fx, fy, w, h}; }
    void flip_h() { fx ^= 1; }               // cvFlip(…, 1)  filters.c:97
    void flip_v() { fy ^= 1; }               // cvFlip(…, 0)  filters.c:99
    void rot90()  { int nfx = !fy, nfy = fx; swap ^= 1; fx = nfx; fy = nfy; std::swap(w, h); }   // filters.c:116-119, 270-90 = flip y-axis
    void rot270() { int nfx = fy, nfy = !fx; swap ^= 1; fx = nfx; fy = nfy; std::swap(w, h); }   // filters.c:116-119, 270-270 = flip x-axis
};

// ---- blob assembly ------------------------------------------------------------------------------------
struct BlobBuilder {
    std::vector<uint8_t> b;
    BlobBuilder() { b.resize((sizeof(ImpPass) + 15) & ~size_t(15), 0); }
    int add(const void* p, size_t n) {
        size_t off = (b.size() + 15) & ~size_t(15);
        b.resize(off + n, 0);
        if (n) memcpy(b.data() + off, p, n);
        return (int)off;
    }
};

struct AreaTap { int si; float a; };
struct Range { int first, count; };

// SURVEY App. A.3 (OpenCV computeResizeAreaTab), grouped per output index.
void area_table(int ssize, int dsize, double scale, std::vector<Range>& ranges, std::vector<AreaTap>& taps, int& max_taps) {
    ranges.resize(dsize); taps.clear(); max_taps = 0;
    for (int d = 0; d < dsize; d++) {
        double f1 = d * scale, f2 = f1 + scale;
        double cell = std::min(scale, ssize - f1);
        int s1 = (int)ceil(f1), s2 = (int)floor(f2);
        s2 = std::min(s2, ssize - 1);
        s1 = std::min(s1, s2);
        int first = (int)taps.size();
        if (s1 - f1 > 1e-3) taps.push_back(AreaTap{s1 - 1, (float)((s1 - f1) / cell)});
        for (int s = s1; s < s2; s++) taps.push_back(AreaTap{s, (float)(1.0 / cell)});
        if (f2 - s2 > 1e-3) taps.push_back(AreaTap{s2, (float)(std::min(std::min(f2 - s2, 1.), cell) / cell)});
        ranges[d] = Range{first, (int)taps.size() - first};
        max_taps = std::max(max_taps, ranges[d].count);
    }
}

short sat_i16(float v) { long r = lrintf(v); return (short)std::max(-32768L, std::min(32767L, r)); }

// SURVEY App. A.4: offsets + 11-bit coefficients for INTER_LINEAR / INTER_CUBIC.
void interp_table(int ssize, int dsize, double scale, bool cubic, bool is_x, std::vector<int>& ofs, std::vector<short>& coef) {
    const int ks = cubic ? 4 : 2;
    ofs.resize(dsize); coef.resize((size_t)dsize * ks);
    for (int d = 0; d < dsize; d++) {
        float f = (float)((d + 0.5) * scale - 0.5);
        int s = (int)floor((double)f);
        f -= (float)s;
        if (!cubic && is_x) {
            if (s < 0) { f = 0; s = 0; }
            if (s >= ssize - 1) { f = 0; s = ssize - 1; }
        }
        ofs[d] = s;
        float cb[4];
        if (cubic) {
            const float A = -0.75f;
            float x = f;
            cb[0] = ((A * (x + 1) - 5 * A) * (x + 1) + 8 * A) * (x + 1) - 4 * A;
            cb[1] = ((A + 2) * x - (A + 3)) * x * x + 1;
            cb[2] = ((A + 2) * (1 - x) - (A + 3)) * (1 - x) * (1 - x) + 1;
            cb[3] = 1.f - cb[0] - cb[1] - cb[2];
        } else { cb[0] = 1.f - f; cb[1] = f; }
        for (int k = 0; k < ks; k++) coef[(size_t)d * ks + k] = sat_i16(cb[k] * 2048);
    }
}

// SURVEY App. A.1.
void nn_table(int ssize, int dsize, std::vector<int>& ofs) {
    double inv = 1.0 / ((double)dsize / ssize);
    ofs.resize(dsize);
    for (int d = 0; d < dsize; d++) ofs[d] = std::min((int)floor(d * inv), ssize - 1);
}

// SURVEY App. A.5: 8-bit Gaussian taps with error diffusion, sum == 256.
std::vector<int> gaussian_taps(double sigma) {
    int n = (int)lrint(sigma * 6 + 1) | 1;
    std::vector<double> t(n);
    double s2 = -0.5 / (sigma * sigma), sum = 0;
    for (int i = 0; i < n; i++) { double x = i - (n - 1) * 0.5; t[i] = exp(s2 * x * x); sum += t[i]; }
    double inv = 1. / sum, err = 0;
    std::vector<int> k(n);
    int isum = 0;
    for (int i = 0; i < n / 2; i++) {
        double adj = t[i] * inv * 256 + err;
        int v = (int)lrint(adj);
        err = adj - v;
        k[i] = k[n - 1 - i] = v;
        isum += v;
    }
    k[n / 2] = 256 - 2 * isum;
    return k;
}

// Strip-kernel tables for shrinking INTER_LINEAR (imp_tiles.cuh, mode 3): per strip of 32 output columns the
// first and last source pixel it touches, per tile of 8 output rows the first source row and the row count; the TMA box is
// the largest such rectangle. x_lo/x_hi(bx), y_lo/y_hi(by): clamped source coordinates an output column / row reads.
template <class FXL, class FXH, class FYL, class FYH>
void gather_strip_tables(BlobBuilder& bb, ImpPass& P, int c, FXL x_lo, FXH x_hi, FYL y_lo, FYH y_hi) {
    const int rw = P.bw, rh = P.bh;
    int span = 0, rows = 0;
    std::vector<int> xtile, ytile;
    for (int x0 = 0; x0 < rw; x0 += 32) {
        int p0 = x_lo(x0), p1 = x_hi(std::min(x0 + 32, rw) - 1);
        for (int x = x0; x < std::min(x0 + 32, rw); x++) { p0 = std::min(p0, x_lo(x)); p1 = std::max(p1, x_hi(x)); }
        xtile.push_back(p0); xtile.push_back(p1);
        span = std::max(span, p1 - p0 + 1);
    }
    for (int y0 = 0; y0 < rh; y0 += 8) {
        int p0 = y_lo(y0), p1 = y_hi(std::min(y0 + 8, rh) - 1);
        for (int y = y0; y < std::min(y0 + 8, rh); y++) { p0 = std::min(p0, y_lo(y)); p1 = std::max(p1, y_hi(y)); }
        ytile.push_back(p0); ytile.push_back(p1 - p0 + 1); ytile.push_back(0); ytile.push_back(0);
        rows = std::max(rows, p1 - p0 + 1);
    }
    P.xtile_off = bb.add(xtile.data(), xtile.size() * 4);
    P.ytile_off = bb.add(ytile.data(), ytile.size() * 4);
    P.tile_rs = (span * c + 15 + 15) & ~15;                     // +15 for the 16-byte alignment of the box origin
    if ((P.tile_rs / 4) % 32 == 0) P.tile_rs += 16;
    P.tile_rows = rows;
    P.tile_smem = (P.tile_rs <= 2048 && rows <= 256 && (long long)P.tile_rs * rows <= 64 * 1024) ? P.tile_rs * rows : 0;
}

// Gather tile kernel (imp_gathertile.cuh; index map, NN, LINEAR): T x T tiles of the destination at ANY base origin (it
// tiles in destination space, so flips move the origin). The TMA box is the largest source rectangle such a tile reads;
// T = 64 when that box stays small (upscales, copies), 32 otherwise, none when even that is too large.
// x_lo/x_hi(bx), y_lo/y_hi(by): clamped source coordinates a base column / row reads; non-decreasing in bx / by.
template <class FXL, class FXH, class FYL, class FYH>
void gather_tile_tables(ImpPass& P, int c, FXL x_lo, FXH x_hi, FYL y_lo, FYH y_hi) {
    const int rw = P.bw, rh = P.bh;
    for (int T : {64, 32}) {
        int span = 0, rows = 0;
        for (int x0 = 0; x0 < rw; x0++) span = std::max(span, x_hi(std::min(x0 + T, rw) - 1) - x_lo(x0) + 1);
        for (int y0 = 0; y0 < rh; y0++) rows = std::max(rows, y_hi(std::min(y0 + T, rh) - 1) - y_lo(y0) + 1);
        const int rs = (span * c + 15 + 15) & ~15;                  // +15 for the 16-byte alignment of the box origin
        const long long bytes = (long long)rs * rows;
        if (rs <= 2048 && rows <= 256 && bytes <= (T == 64 ? 24 : 40) * 1024) {
            P.gt = T; P.tile_rs = rs; P.tile_rows = rows; P.tile_smem = (int)bytes;
            return;
        }
    }
}

// ---- lowering state -----------------------------------------------------------------------------------
struct Lower {
    imp_gpu_plan* plan;
    Frame fr;                       // current logical frame
    // pass under construction
    ImpPass hdr;
    BlobBuilder bb;
    std::vector<ImpOp> ops;
    std::vector<uint8_t> luts;
    int in_w, in_h, in_c;
    bool uses_wm = false;
    bool dry = false;               // validate only: no tables, LUTs or blobs
    double sigma = 0;

    // ---- fusion of channel-separable ops ----------------------------------------------------------------------------
    // AlphaBlendAddColor, ApplyGamma, BrightnessContrast and Lomo map every channel byte on its own (filters.c:549-616,
    // 335-346), so a run of them — gotham is three in a row, kelvin and "sepia" end in one — composes into ONE 256-entry
    // table per channel, tabulated here with the host instantiation of the kernels' own per-pixel functions: the same
    // bytes, one shared-memory load per channel instead of the float sequence of every op. A modulate with saturation
    // factor 0 (sepia) turns the pixel into (V,V,V) with V = scaled max(B,G,R): it OPENS such a run as a table over the
    // maximum (IMP_OP_MAXLUT3). Geometry filters do not close a run (pointwise ops commute with index maps).
    int fuse_mode = 0;              // 0 none, 1 per-channel tables of the channel's own value, 2 tables of max(B,G,R)
    bool fuse_alpha = false;        // the alpha table is not the identity (gamma runs over alpha too, filters.c:554)
    uint8_t fuse_tab[4][256];
    void fuse_open(int mode) {
        fuse_mode = mode; fuse_alpha = false;
        if (!dry) for (int c = 0; c < 4; c++) for (int v = 0; v < 256; v++) fuse_tab[c][v] = (uint8_t)v;
    }
    // f(ImpPx&) is one separable op on a whole pixel; it is tabulated channel by channel through the running tables
    template <class F> void fuse(F f, bool touches_alpha) {
        if (!fuse_mode) fuse_open(1);
        if (touches_alpha && hdr.oc == 4) fuse_alpha = true;
        if (dry) return;
        for (int v = 0; v < 256; v++) {
            ImpPx p{fuse_tab[0][v], fuse_tab[1][v], fuse_tab[2][v], fuse_tab[3][v]};
            f(p);
            fuse_tab[0][v] = (uint8_t)p.b; fuse_tab[1][v] = (uint8_t)p.g; fuse_tab[2][v] = (uint8_t)p.r;
            if (touches_alpha && hdr.oc == 4) fuse_tab[3][v] = (uint8_t)p.a;
        }
    }
    void fuse_flush() {
        if (!fuse_mode) return;
        ImpOp o{}; o.kind = fuse_mode == 2 ? IMP_OP_MAXLUT3 : IMP_OP_LUT3;
        o.i[1] = fuse_alpha ? 1 : 0;
        fuse_mode = 0;
        reserve_op();
        if (!dry) o.i[0] = add_lut(&fuse_tab[0][0], fuse_alpha ? 1024 : 768);
        ops.push_back(o);
    }
    // every op that is not channel-separable closes the running table first
    void push(const ImpOp& o) { fuse_flush(); reserve_op(); ops.push_back(o); }
    // The reference takes as many filters as imgproc_max_filters_count allows (bridge.c:360-363). A pass holds IMP_MAX_OPS ops
    // and ~30 KB of tables (shared memory of the kernels): when the next op would not fit, the running pass is stored in base
    // orientation and an index-map pass continues the chain — same pixels, one more round trip through the L2-resident scratch.
    void reserve_op() {
        if ((int)ops.size() < IMP_MAX_OPS && luts.size() <= 30 * 1024) return;
        ImpFrameMap ident{0, 0, 0, hdr.bw, hdr.bh};
        const int bw = hdr.bw, bh = hdr.bh, oc = hdr.oc;
        if (hdr.kind == IMP_G_COPY && !dry) copy_tables();
        end_pass(ident, bw, bh);
        begin_pass(IMP_G_COPY, bw, bh, oc);
        hdr.oc = oc; hdr.sx0 = hdr.sy0 = 0; hdr.sw = hdr.bw = bw; hdr.sh = hdr.bh = bh;
    }

    void begin_pass(int kind, int in_w_, int in_h_, int in_c_) {
        memset(&hdr, 0, sizeof hdr);
        bb = BlobBuilder(); ops.clear(); luts.clear(); uses_wm = false; sigma = 0;
        hdr.kind = kind; in_w = in_w_; in_h = in_h_; in_c = in_c_;
        hdr.sc = in_c_;
    }
    void copy_tables() {
        gather_tile_tables(hdr, hdr.sc, [](int x) { return x; }, [](int x) { return x; }, [](int y) { return y; }, [](int y) { return y; });
    }
    int add_lut(const uint8_t* p, int n) { int off = (int)luts.size(); luts.insert(luts.end(), p, p + n); return off; }
    int final_dc = 0;              // destination channels of the LAST pass when the encoder-side packing changes them
    void end_pass(const ImpFrameMap& out, int out_w, int out_h) {
        fuse_flush();
        if (dry) return;
        hdr.nops = (int)ops.size();
        while (luts.size() % 16) luts.push_back(0);
        std::vector<uint8_t> tail(ops.size() * sizeof(ImpOp) + luts.size());
        if (!ops.empty()) memcpy(tail.data(), ops.data(), ops.size() * sizeof(ImpOp));
        if (!luts.empty()) memcpy(tail.data() + ops.size() * sizeof(ImpOp), luts.data(), luts.size());
        static const uint8_t pad[16] = {0};
        hdr.ops_off = tail.empty() ? bb.add(pad, 16) : bb.add(tail.data(), tail.size());
        hdr.lut_off = hdr.ops_off + (int)(ops.size() * sizeof(ImpOp));
        hdr.lut_bytes = (int)luts.size();
        hdr.out = out;
        hdr.dc = final_dc ? final_dc : hdr.oc;
        hdr.light = 7;                         // bit 0: only fused tables (or no op at all); bit 1: no compositing op; bit 2: only compositing + tables
        for (const ImpOp& o : ops) {
            const bool table = o.kind == IMP_OP_LUT3 || o.kind == IMP_OP_MAXLUT3, comp = o.kind == IMP_OP_WATERMARK || o.kind == IMP_OP_PAPER;
            if (!table) hdr.light &= ~1;
            if (comp) hdr.light &= ~2;
            if (!table && !comp) hdr.light &= ~4;
        }
        bb.b.resize(((bb.b.size() + 15) & ~size_t(15)) + 64, 0);     // tail slack: the strip kernels' 16/64-byte table copies may over-read
        hdr.blob_bytes = (int)bb.b.size();
        memcpy(bb.b.data(), &hdr, sizeof hdr);
        ImpHostPass hp;
        hp.hdr = hdr; hp.blob = bb.b;
        hp.in_w = in_w; hp.in_h = in_h; hp.in_c = in_c;
        hp.out_w = out_w; hp.out_h = out_h; hp.out_c = hdr.dc;
        hp.uses_watermark = uses_wm; hp.sigma = sigma;
        imp_pass_launches(hdr, &hp.tiled, &hp.fallback);
        plan->passes.push_back(std::move(hp));
    }
    // A Gaussian blur: close the running pass (stored in base orientation) and open a stencil pass.
    void split_for_blur(double sg) {
        fuse_flush();
        if (dry) {                                  // only what later validation depends on: a new pass starts an empty op list
            if (!(hdr.kind == IMP_G_COPY && ops.empty() && hdr.sc >= 3)) { ops.clear(); hdr.sc = hdr.oc; }
            hdr.kind = IMP_G_BLUR;
            return;
        }
        std::vector<int> k = gaussian_taps(sg);
        const bool trivial = hdr.kind == IMP_G_COPY && ops.empty() && hdr.sc >= 3;
        if (trivial) {
            hdr.kind = IMP_G_BLUR;                  // blur reads the (cropped) source directly
        } else {
            ImpFrameMap ident{0, 0, 0, hdr.bw, hdr.bh};
            int bw = hdr.bw, bh = hdr.bh, oc = hdr.oc;
            if (hdr.kind == IMP_G_COPY) copy_tables();
            end_pass(ident, bw, bh);
            begin_pass(IMP_G_BLUR, bw, bh, oc);
            hdr.oc = oc; hdr.sx0 = hdr.sy0 = 0; hdr.sw = hdr.bw = bw; hdr.sh = hdr.bh = bh;
        }
        hdr.ksize = (int)k.size();
        hdr.taps_off = bb.add(k.data(), k.size() * sizeof(int));
        sigma = sg;
        // tile kernel (imp_blur.cuh): effective radius after trimming zero outer taps, padded up to 3/6/9/12
        int lo = 0, hi = (int)k.size() - 1;
        while (lo < hi && k[lo] == 0 && k[hi] == 0) { lo++; hi--; }
        const int r_eff = (hi - lo) / 2;
        hdr.blur_r = r_eff <= 3 ? 3 : r_eff <= 6 ? 6 : r_eff <= 9 ? 9 : r_eff <= 12 ? 12 : 0;
        if (k.size() == 1) hdr.blur_r = 0;                          // n == 1 holds the single tap 256, a plain copy
        for (int v : k) if (v < 0 || v > 255) hdr.blur_r = 0;       // the dot-product taps are u8 (a lone centre tap of 256 is not)
        if (hdr.blur_r) {
            const int R = hdr.blur_r;
            std::vector<int> kr(2 * R + 1, 0);
            for (int i = lo; i <= hi; i++) kr[R - r_eff + (i - lo)] = k[i];
            hdr.tapsr_off = bb.add(kr.data(), kr.size() * sizeof(int));
            // taph[m][w]: byte e of word w = tap (4w + e - m), i.e. the taps shifted right by m bytes (horizontal, dp4a);
            // tapv[m][w]: the same with m in {0,1} (vertical, dp2a: bytes 0,1 feed .lo, bytes 2,3 feed .hi)
            const int nwh = (2 * R + 4 + 3) / 4, nwv = ((R + 1) + 1) / 2;
            std::vector<uint32_t> th((size_t)4 * nwh, 0), tv((size_t)2 * nwv, 0);
            for (int m = 0; m < 4; m++)
                for (int b = 0; b < 4 * nwh; b++) {
                    const int t = b - m;
                    if (t >= 0 && t <= 2 * R) th[(size_t)m * nwh + b / 4] |= (uint32_t)kr[t] << (8 * (b % 4));
                }
            for (int m = 0; m < 2; m++)
                for (int b = 0; b < 4 * nwv; b++) {
                    const int t = b - m;
                    if (t >= 0 && t <= 2 * R) tv[(size_t)m * nwv + b / 4] |= (uint32_t)kr[t] << (8 * (b % 4));
                }
            hdr.taph_off = bb.add(th.data(), th.size() * 4);
            hdr.tapv_off = bb.add(tv.data(), tv.size() * 4);
            hdr.tile_rows = IMP_BLUR_TH + 2 * R;
            hdr.tile_rs = ((IMP_BLUR_TW + 2 * R) * hdr.sc + 15 + 15) & ~15;
            hdr.tile_smem = hdr.tile_rs * hdr.tile_rows;
        }
    }
};


const char* const kFilterNames[] = {"flip", "rotate", "modulate", "colorize", "blur", "gamma", "contrast", "gradmap",
                                    "vignette", "gotham", "lomo", "kelvin", "rainbow", "scanline"};   // filters.c:10-24
const bool kExperimental[] = {false, false, false, false, false, false, false, false, true, true, true, true, true, true};

void gamma_lut(float gamma, uint8_t* lut) {          // filters.c:561-570, stored through char (filters.c:556)
    float inverse = 1 / gamma;
    for (int i = 0; i < 256; i++) lut[i] = (uint8_t)(unsigned)d2i_x86(pow(i / 255.0, inverse) * 255.0);
}

void push_modulate(Lower& L, int h, int s, int v) {
    if (s == 0) {
        // S becomes 0 whatever it was and HSV2RGB's S == 0 branch (helpers.c:117) returns (V,V,V): the pixel only depends on
        // max(B,G,R) from here on, so the op opens a table over that maximum and the separable ops after it fold in
        L.fuse_flush();
        L.fuse_open(2);
        if (!L.dry) for (int m = 0; m < 256; m++) { ImpPx p{m, m, m, 255}; imp_op_modulate(p, h, 0, v); L.fuse_tab[0][m] = (uint8_t)p.b; L.fuse_tab[1][m] = (uint8_t)p.g; L.fuse_tab[2][m] = (uint8_t)p.r; }
        return;
    }
    ImpOp o{}; o.kind = IMP_OP_MODULATE; o.i[0] = h; o.i[1] = s; o.i[2] = v; L.push(o);
}
void push_addcolor(Lower& L, const int* rgb, float alpha) {     // filters.c:608-616
    ImpOp o{}; o.kind = IMP_OP_ADDCOLOR;
    float beta = 1 - alpha;
    o.f[0] = beta; o.f[1] = (float)rgb[2] * alpha; o.f[2] = (float)rgb[1] * alpha; o.f[3] = (float)rgb[0] * alpha;
    o.i[0] = (beta >= 0 && o.f[1] >= 0 && o.f[2] >= 0 && o.f[3] >= 0) ? 1 : 0;     // enables the XU-free truncation path
    const float f0 = o.f[0], f1 = o.f[1], f2 = o.f[2], f3 = o.f[3]; const bool nonneg = o.i[0] != 0;
    L.fuse([=](ImpPx& p) { imp_op_addcolor(p, f0, f1, f2, f3, nonneg); }, false);
}
void push_gamma(Lower& L, float g) {
    uint8_t lut[256];
    if (!L.dry) gamma_lut(g, lut);
    L.fuse([&](ImpPx& p) { p.b = lut[p.b]; p.g = lut[p.g]; p.r = lut[p.r]; p.a = lut[p.a]; }, true);     // every channel, alpha too (filters.c:554)
}
void push_contrast(Lower& L, float br, float ct) {
    const float f0 = ct, f1 = br * 255;
    L.fuse([=](ImpPx& p) { p.b = imp_contrast1(p.b, f0, f1); p.g = imp_contrast1(p.g, f0, f1); p.r = imp_contrast1(p.r, f0, f1); }, false);
}

int hex2(const std::string& s, int i) { return (int)strtol(s.substr(i * 2, 2).c_str(), nullptr, 16); }

// One "name=args" request (filters.c:43-70 + callbacks). Returns IMP_* code.
int lower_filter(Lower& L, const char* request, int allow) {
    std::vector<std::string> parts = tokens(request, '=');
    if (parts.empty()) return IMP_ERROR_NO_SUCH_FILTER;
    if (parts.size() < 2) return IMP_ERROR_INVALID_ARGS;
    const std::string& name = parts[0];
    const std::string& args = parts[1];
    int id = -1;
    for (int i = 0; i < 14; i++)
        if (name == kFilterNames[i] && (allow || !kExperimental[i])) { id = i; break; }
    if (id < 0) return IMP_ERROR_NO_SUCH_FILTER;
    std::vector<std::string> t = tokens(args.c_str(), ',');
    Frame& fr = L.fr;
    switch (id) {
        case 0: {   // flip filters.c:72-109
            if (args.size() != 2) return IMP_ERROR_INVALID_ARGS;
            int hz = 0, vt = 0;
            if (args[0] == '1') hz = 1; else if (args[0] != '0') return IMP_ERROR_INVALID_ARGS;
            if (args[1] == '1') vt = 1; else if (args[1] != '0') return IMP_ERROR_INVALID_ARGS;
            if (hz) fr.flip_h();
            if (vt) fr.flip_v();
            return IMP_OK;
        }
        case 1: {   // rotate filters.c:111-133
            int amount = (int)strtol(args.c_str(), nullptr, 10);
            if (amount == 90) fr.rot90();
            else if (amount == 270) fr.rot270();
            else if (amount == 180) { fr.flip_h(); fr.flip_v(); }
            else return IMP_ERROR_INVALID_ARGS;
            return IMP_OK;
        }
        case 2: {   // modulate filters.c:135-158
            if (t.size() < 3) return IMP_ERROR_INVALID_ARGS;
            int p[3];
            for (int i = 0; i < 3; i++) p[i] = (int)strtol(t[i].c_str(), nullptr, 10);
            if (p[0] < 0 || p[0] > 180) return IMP_ERROR_INVALID_ARGS;
            if (p[2] <= 0) return IMP_ERROR_INVALID_ARGS;
            push_modulate(L, p[0], p[1], p[2]);
            return IMP_OK;
        }
        case 3: {   // colorize filters.c:160-190
            if (t.empty() || t[0].size() != 6) return IMP_ERROR_INVALID_ARGS;
            int rgb[3] = {hex2(t[0], 0), hex2(t[0], 1), hex2(t[0], 2)};
            float opacity = t.size() > 1 ? parse_float(t[1]) : 0.5f;
            if (opacity < 0 || opacity > 1) return IMP_ERROR_INVALID_ARGS;
            push_addcolor(L, rgb, opacity);
            return IMP_OK;
        }
        case 4: {   // blur filters.c:192-207
            if (t.empty()) return IMP_ERROR_INVALID_ARGS;
            float sigma = parse_float(t[0]);
            if (sigma < 0) return IMP_ERROR_INVALID_ARGS;
            if (!(sigma > 0)) return IMP_ERROR_INVALID_ARGS;           // App. C-9
            double sg = (double)sigma;
            if (sg * 6 + 1 > 2047) return IMP_ERROR_INVALID_ARGS;      // documented cap on the stencil size
            L.split_for_blur(sg);
            return IMP_OK;
        }
        case 5:     // gamma filters.c:209-212
            push_gamma(L, parse_float(args));
            return IMP_OK;
        case 6: {   // contrast filters.c:214-221
            float v = parse_float(args);
            if (v <= 0) return IMP_ERROR_INVALID_ARGS;
            push_contrast(L, 0, v);
            return IMP_OK;
        }
        case 7: {   // gradmap filters.c:223-286 + CalculateGradientLUT :572-593
            for (const std::string& tok : t) if (tok.size() != 6) return IMP_ERROR_INVALID_ARGS;
            if (t.size() < 2 || t.size() > 8) return IMP_ERROR_INVALID_ARGS;   // App. C-4
            uint8_t lut[768];
            memset(lut, 0, sizeof lut);                                        // tail defined as 0 (App. C-4)
            int segments = (int)t.size() - 1, ptr = 0;
            float inner = 256 / (float)segments;
            for (int c = 0; c < segments; c++) {
                uint8_t from[3], to[3];
                for (int j = 0; j < 3; j++) { from[j] = (uint8_t)hex2(t[c], j); to[j] = (uint8_t)hex2(t[c + 1], j); }
                for (int i = 0; i < (int)inner; i++) {
                    float step = i / inner;
                    for (int j = 0; j < 3; j++) {
                        float v = (float)from[j] + step * (float)(to[j] - from[j]);
                        lut[ptr++] = (uint8_t)(unsigned)d2i_x86(round((double)v));
                    }
                }
            }
            ImpOp o{}; o.kind = IMP_OP_GRADMAP; L.fuse_flush(); L.reserve_op(); o.i[0] = L.add_lut(lut, 768); L.ops.push_back(o);
            return IMP_OK;
        }
        case 8: {   // vignette filters.c:295-323; centre/maxr from helpers.c:46-66
            float intensity = t.size() > 0 ? parse_float(t[0]) : 0.5f;
            float radius = t.size() > 1 ? parse_float(t[1]) : 1.0f;
            int w = fr.w, h = fr.h, cx = w / 2, cy = h / 2;
            int xs[4] = {0, w, 0, w}, ys[4] = {0, 0, h, h};
            float maxd = 0;
            for (int i = 0; i < 4; i++) {
                float d = (float)sqrt(pow((double)(float)(xs[i] - cx), 2) + pow((double)(float)(ys[i] - cy), 2));
                if (maxd < d) maxd = d;
            }
            ImpOp o{}; o.kind = IMP_OP_VIGNETTE; o.i[0] = cx; o.i[1] = cy; o.f[0] = radius * maxd; o.f[1] = intensity; o.map = fr.map();
            // The mask depends on the pixel only through (|dx|, |dy|): the runtime tabulates it once per plan and device as
            // mask[|dy|][|dx|] (same double-precision code as the per-pixel path) when the table stays below 64 MB. Indexed
            // by d2 = dx*dx + dy*dy it was half the entries, but the 32 lanes of a warp then hit 32 different sectors of
            // it; row-major in |dx| they read one or two.
            {
                long long mx = std::max(cx, w - 1 - cx) + IMP_VIGNETTE_MARGIN, my = std::max(cy, h - 1 - cy) + IMP_VIGNETTE_MARGIN;
                long long entries = (mx + 1) * (my + 1);
                if (entries <= (16ll << 20)) { o.i[2] = (int)(mx + 1); o.i[3] = (int)(my + 1); }
            }
            L.push(o);
            return IMP_OK;
        }
        case 9: {   // gotham filters.c:325-333
            push_modulate(L, 120, 5, 100);
            int rgb[3] = {17, 27, 93};
            push_addcolor(L, rgb, (float)0.15);
            push_gamma(L, (float)0.3);
            push_contrast(L, (float)-0.07, (float)1.5);
            return IMP_OK;
        }
        case 10:    // lomo filters.c:335-346
            L.fuse([](ImpPx& p) { p.g = imp_lomo1(p.g); p.r = imp_lomo1(p.r); }, false);
            return IMP_OK;
        case 11: {  // kelvin filters.c:348-354
            push_modulate(L, 120, 50, 100);
            int rgb[3] = {255, 153, 0};
            push_addcolor(L, rgb, (float)0.5);
            return IMP_OK;
        }
        case 12: {  // rainbow filters.c:356-403
            int sat;
            if (args == "full") sat = 255; else if (args == "mid") sat = 190; else if (args == "pale") sat = 120;
            else return IMP_ERROR_INVALID_ARGS;
            ImpOp o{}; o.kind = IMP_OP_RAINBOW; o.i[0] = sat; L.push(o);
            return IMP_OK;
        }
        case 13: {  // scanline filters.c:405-455
            if (t.empty()) return IMP_ERROR_INVALID_ARGS;                      // App. C-10
            float intensity = parse_float(t[0]);
            if (intensity < 0 || intensity > 1) return IMP_ERROR_INVALID_ARGS;
            float opacity = t.size() > 1 ? parse_float(t[1]) : 0;
            if (opacity < 0 || opacity > 1) return IMP_ERROR_INVALID_ARGS;
            int freq = t.size() > 2 ? (int)strtol(t[2].c_str(), nullptr, 10) : 1;
            if (freq < 1) return IMP_ERROR_INVALID_ARGS;
            int width = t.size() > 3 ? (int)strtol(t[3].c_str(), nullptr, 10) : 1;
            if (width < 1) return IMP_ERROR_INVALID_ARGS;
            if ((long long)freq + width + 1 > INT_MAX) return IMP_ERROR_INVALID_ARGS;
            ImpOp o{}; o.kind = IMP_OP_SCANLINE;
            o.i[0] = freq + width + 1; o.i[1] = freq; o.i[2] = width;
            o.i[3] = f2i_x86(255 * opacity) & 255; o.i[4] = f2i_x86(255 * intensity) & 255;
            o.map = fr.map();
            L.push(o);
            return IMP_OK;
        }
    }
    return IMP_ERROR_NO_SUCH_FILTER;
}

// bridge.c:18-128. col,row: current image size. Returns code; window in x,y,w,h.
int parse_crop(const char* args_s, const char* gravity, size_t col, size_t row, int& X, int& Y, int& W, int& H) {
    std::vector<std::string> t = tokens(args_s, ',');
    Num nw = parse_long(t.size() > 0 ? t[0] : std::string());
    Num nh = parse_long(t.size() > 1 ? t[1] : std::string());
    unsigned ww = (unsigned)nw.v, wh = (unsigned)nh.v;
    bool respect = false;
    if (gravity) {
        if (strlen(gravity) > 2) respect = true; else return IMP_ERROR_INVALID_ARGS;
    }
    if (nw.rest.empty() && nh.rest.empty()) {                 // ratio mode, float32 (bridge.c:47-57)
        float px = (float)col;
        float py = px / (float)ww * (float)wh;
        if (py > (float)row) { py = (float)row; px = py / (float)wh * (float)ww; }
        ww = (unsigned)d2i_x86(round((double)px));
        wh = (unsigned)d2i_x86(round((double)py));
    } else if (nw.rest == "px" && nh.rest == "px") {
    } else return IMP_ERROR_INVALID_ARGS;
    if (ww == 0 || ww > col || wh == 0 || wh > row) return IMP_ERROR_INVALID_ARGS;

    std::vector<std::string> g;
    if (respect) g = tokens(gravity, ',');
    else if (t.size() > 2) g.assign(t.begin() + 2, t.end());
    if (respect && g.size() < 2) return IMP_ERROR_INVALID_ARGS;   // reference: strcmp(NULL)
    auto axis = [](const std::string* tok, const char* lo, const char* hi, const char* dflt, long size, long win, int& out) -> bool {
        std::string s = tok ? *tok : std::string(dflt);
        if (s == lo) { out = 0; return true; }
        if (s == hi) { out = (int)(size - win); return true; }
        if (s == "c") { out = d2i_x86(round((double)(size - win) / 2.0)); return true; }
        Num n = parse_long(s);
        if (n.rest == "px") { out = (int)(unsigned)n.v; return true; }
        return false;
    };
    int wx, wy;
    if (!axis(g.size() > 0 ? &g[0] : nullptr, "l", "r", "c", (long)col, (long)ww, wx)) return IMP_ERROR_INVALID_ARGS;
    if (!axis(g.size() > 1 ? &g[1] : nullptr, "t", "b", "t", (long)row, (long)wh, wy)) return IMP_ERROR_INVALID_ARGS;
    if (wx < 0 || wy < 0) return IMP_ERROR_INVALID_ARGS;          // reference: OpenCV size-mismatch assert
    // 64-bit: a pixel offset near INT_MAX must not wrap past the bound (the reference stops it at cvSetImageROI)
    if ((long long)wx + (long long)ww > (long long)col || (long long)wy + (long long)wh > (long long)row) return IMP_ERROR_INVALID_ARGS;
    X = wx; Y = wy; W = (int)ww; H = (int)wh;
    return IMP_OK;
}

// bridge.c:143-190.
int parse_resize(const char* args_s, size_t col, size_t row, const imp_gpu_config* cfg, int simple, int& W, int& H, int& mode) {
    std::vector<std::string> t = tokens(args_s, ',');
    unsigned width = (unsigned)parse_long(t.size() > 0 ? t[0] : std::string()).v;
    unsigned height = (unsigned)parse_long(t.size() > 1 ? t[1] : std::string()).v;
    if (width == 0 && height == 0) return IMP_ERROR_INVALID_ARGS;
    if (width == 0) width = (unsigned)d2i_x86(round((double)((float)height / (float)row * (float)col)));
    if (height == 0) height = (unsigned)d2i_x86(round((double)((float)width / (float)col * (float)row)));
    bool up = t.size() > 2 && t[2] == "up";
    if (!up) {
        width = (unsigned)fmin((double)width, (double)col);
        height = (unsigned)fmin((double)height, (double)row);
    }
    unsigned mw = cfg ? cfg->max_target_w : 0, mh = cfg ? cfg->max_target_h : 0;
    if ((mw > 0 && width > mw) || (mh > 0 && width > mh)) return IMP_ERROR_TOO_BIG_TARGET;    // sic: bridge.c:184
    if (width == 0 || height == 0) return IMP_ERROR_INVALID_ARGS;                               // cvCreateImage would fail
    if (width > 65535u || height > 65535u) return IMP_ERROR_TOO_BIG_TARGET;                     // documented hard cap
    W = (int)width; H = (int)height;
    mode = simple ? 0 : ((width > col || height > row) ? 2 : 3);                                // CV_INTER_NN / CUBIC / AREA
    return IMP_OK;
}

}  // namespace

int imp_build_plan(const imp_gpu_request* req, const imp_gpu_config* cfg, int w, int h, int c, imp_gpu_plan* plan, int* step, bool dry) {
    int dummy; if (!step) step = &dummy;
    *step = 0;                                   // IMP_STEP_START: the filter-count guard fires while RunJob
    if (!req || w <= 0 || h <= 0 || (c != 1 && c != 3 && c != 4)) return IMP_ERROR_INVALID_ARGS;
    if (req->filter_count < 0 || (req->filter_count > 0 && !req->filters)) return IMP_ERROR_INVALID_ARGS;
    // is still parsing the query (bridge.c:360-363), i.e. before any operator validates its arguments
    if (cfg && req->filter_count > cfg->max_filters) return IMP_ERROR_TOO_MUCH_FILTERS;
    *step = IMP_STEP_CROP;
    plan->src_w = w; plan->src_h = h; plan->src_c = c;
    Lower L; L.plan = plan; L.dry = dry;

    // step 3: crop (bridge.c:576-586)
    int cx = 0, cy = 0, cw = w, ch = h;
    if (req->crop) {
        int code = parse_crop(req->crop, req->gravity, (size_t)w, (size_t)h, cx, cy, cw, ch);
        if (code) return code;
    }
    // every kernel and the host paths address src + win_y*step + win_x*c: the window must lie inside the frame
    if (cx < 0 || cy < 0 || cw <= 0 || ch <= 0 || (long long)cx + cw > w || (long long)cy + ch > h) return IMP_ERROR_INVALID_ARGS;
    plan->win_x = cx; plan->win_y = cy; plan->win_w = cw; plan->win_h = ch;

    // step 4: resize (bridge.c:589-604)
    *step = IMP_STEP_RESIZE;
    int rw = cw, rh = ch, mode = -1;
    if (req->resize) {
        int code = parse_resize(req->resize, (size_t)cw, (size_t)ch, cfg, req->simple_resize, rw, rh, mode);
        if (code) return code;
        if (req->interp == IMP_INTERP_LINEAR && mode != 0) mode = 1;
    }
    L.begin_pass(IMP_G_COPY, w, h, c);
    ImpPass& P = L.hdr;
    P.sx0 = cx; P.sy0 = cy; P.sw = cw; P.sh = ch; P.bw = rw; P.bh = rh;
    if (dry && mode >= 0 && !(rw == cw && rh == ch)) P.kind = IMP_G_NN;      // "not an index map" is all the validation needs
    if (!dry && mode >= 0 && !(rw == cw && rh == ch)) {
        double scale_x = 1.0 / ((double)rw / cw), scale_y = 1.0 / ((double)rh / ch);
        int isx = (int)lrint(scale_x), isy = (int)lrint(scale_y);
        bool fast = fabs(scale_x - isx) < DBL_EPSILON && fabs(scale_y - isy) < DBL_EPSILON;
        if (mode == 1 && fast && isx == 2 && isy == 2) mode = 3;
        if (mode == 0) {
            std::vector<int> xo, yo;
            nn_table(cw, rw, xo); nn_table(ch, rh, yo);
            P.kind = IMP_G_NN;
            P.xofs_off = L.bb.add(xo.data(), xo.size() * 4);
            P.yofs_off = L.bb.add(yo.data(), yo.size() * 4);
            // staging pays while most staged rows are used: a nearest-neighbour shrink reads one row in scale_y, which the
            // direct kernel fetches sector by sector instead
            if (scale_y <= 1.5 && scale_x <= 2.0)
                gather_tile_tables(P, c, [&](int x) { return xo[x]; }, [&](int x) { return xo[x]; },
                                   [&](int y) { return yo[y]; }, [&](int y) { return yo[y]; });
        } else if (mode == 3 && scale_x >= 1 && scale_y >= 1) {
            {
                // The strip kernel (imp_tiles.cuh) walks the same tap tables for both flavours; with integer scales
                // every column/row has exactly nx/ny taps and the weights are unused.
                std::vector<Range> xr, yr; std::vector<AreaTap> xt, yt;
                area_table(cw, rw, scale_x, xr, xt, P.max_xtaps);
                area_table(ch, rh, scale_y, yr, yt, P.max_ytaps);
                if (fast) { P.kind = IMP_G_AREA_INT; P.nx = isx; P.ny = isy; P.area_scale = 1.f / (isx * isy); }
                else P.kind = IMP_G_AREA_FRAC;
                // footprint of the 32x8 output tiles of the shared-memory kernel (imp_tiles.cuh)
                int span = 0, rows = 0;
                std::vector<int> xtile, ytile;
                for (int x0 = 0; x0 < rw; x0 += 32) {
                    int x1 = std::min(x0 + 32, rw) - 1;
                    int p0 = xt[xr[x0].first].si, p1 = xt[xr[x1].first + xr[x1].count - 1].si;
                    xtile.push_back(p0); xtile.push_back(p1);
                    span = std::max(span, p1 - p0 + 1);
                }
                int ytaps = 0;
                for (int y0 = 0; y0 < rh; y0 += 8) {
                    int y1 = std::min(y0 + 8, rh) - 1;
                    int p0 = yt[yr[y0].first].si, p1 = yt[yr[y1].first + yr[y1].count - 1].si;
                    int t0 = yr[y0].first, tn = yr[y1].first + yr[y1].count - t0;
                    ytile.push_back(p0); ytile.push_back(p1 - p0 + 1); ytile.push_back(t0); ytile.push_back(tn);   // int4 per tile row
                    rows = std::max(rows, p1 - p0 + 1);
                    ytaps = std::max(ytaps, tn + 2);           // +1 for the even alignment of the first tap, +1 for the 16-byte rounding
                }
                P.tile_ytaps = ytaps;
                P.xtile_off = L.bb.add(xtile.data(), xtile.size() * 4);
                P.ytile_off = L.bb.add(ytile.data(), ytile.size() * 4);
                // TMA box: tile_rs bytes x rows; +2 px for the zero-weight padded taps of narrower columns, +15 for the
                // 16-byte alignment of the box origin, +4 for the aligned word loads of packed 3-channel pixels
                P.tile_rs = ((span + 2) * c + 15 + 4 + 15) & ~15;
                if ((P.tile_rs / 4) % 32 == 0) P.tile_rs += 16;
                P.tile_rows = rows;
                P.tile_smem = (P.max_xtaps <= 12 && P.tile_rs <= 2048 && rows <= 256 && (long long)P.tile_rs * rows <= 100 * 1024 &&
                               (!fast || isx * isy <= 256)) ? P.tile_rs * rows : 0;
                {
                    // what a consumer warp needs to start an output row, relative to the tile it is staged with
                    std::vector<int> yrow4;
                    const int padded = (rh + 7) & ~7;              // the producer always copies 8 entries
                    for (int y = 0; y < padded; y++) {
                        const int yy = std::min(y, rh - 1), t = yy / 8;
                        const int p0 = ytile[t * 4], tapbase = ytile[t * 4 + 2] & ~1;
                        yrow4.push_back((yt[yr[yy].first].si - p0) * P.tile_rs); yrow4.push_back(yr[yy].count);
                        yrow4.push_back(yr[yy].first - tapbase); yrow4.push_back(0);
                    }
                    P.yrow4_off = L.bb.add(yrow4.data(), yrow4.size() * 4);
                }
                P.xofs_off = L.bb.add(xr.data(), xr.size() * sizeof(Range));
                P.xcoef_off = L.bb.add(xt.data(), xt.size() * sizeof(AreaTap));
                P.yofs_off = L.bb.add(yr.data(), yr.size() * sizeof(Range));
                P.ycoef_off = L.bb.add(yt.data(), yt.size() * sizeof(AreaTap));
            }
        } else {
            bool cubic = (mode == 2);
            // (AREA with an upscaled axis cannot come out of bridge.c:190; LINEAR/CUBIC otherwise)
            if (mode == 3) cubic = false;
            std::vector<int> xo, yo; std::vector<short> xa, yb;
            interp_table(cw, rw, scale_x, cubic, true, xo, xa);
            interp_table(ch, rh, scale_y, cubic, false, yo, yb);
            P.kind = cubic ? IMP_G_CUBIC : IMP_G_LINEAR;
            P.ksize = cubic ? 4 : 2;
            P.simd_end = (rw * c) - ((rw * c) % 8);
            P.xofs_off = L.bb.add(xo.data(), xo.size() * 4);
            P.xcoef_off = L.bb.add(xa.data(), xa.size() * 2);
            P.yofs_off = L.bb.add(yo.data(), yo.size() * 4);
            P.ycoef_off = L.bb.add(yb.data(), yb.size() * 2);
            auto clampi = [](int v, int lo, int hi) { return std::min(std::max(v, lo), hi); };
            if (cubic) {
                // the float form OpenCV's SIMD vertical pass multiplies with: b * 2^-22, exact (imp_cubic.cuh)
                std::vector<float> ybf(yb.size());
                for (size_t i = 0; i < yb.size(); i++) ybf[i] = (float)yb[i] * (1.0f / 4194304.0f);
                P.taps_off = L.bb.add(ybf.data(), ybf.size() * 4);
                // tile kernel (imp_cubic.cuh): T x T output tiles at ANY origin (it tiles in destination space); the TMA box is
                // the largest source rectangle such a tile's clamped 4x4 footprints span. T = 64 while the box and the
                // horizontal-pass buffer stay within ~52 KB (four CTAs per SM), else 32, else the column-run kernel.
                for (int T : {64, 32}) {
                    int span = 0, rows = 0;
                    for (int x0 = 0; x0 < rw; x0++) {
                        const int x1 = std::min(x0 + T, rw) - 1;
                        span = std::max(span, clampi(xo[x1] + 2, 0, cw - 1) - clampi(xo[x0] - 1, 0, cw - 1) + 1);
                    }
                    for (int y0 = 0; y0 < rh; y0++) {
                        const int y1 = std::min(y0 + T, rh) - 1;
                        rows = std::max(rows, clampi(yo[y1] + 2, 0, ch - 1) - clampi(yo[y0] - 1, 0, ch - 1) + 1);
                    }
                    const int rs = (span * c + 15 + 15) & ~15;
                    const long long bytes = (long long)rs * rows + (long long)rows * IMP_CUBIC_HRS(c, T) * 4;
                    if (rs <= 2048 && rows <= 160 && bytes <= 52 * 1024) {
                        P.gt = T; P.tile_rs = rs; P.tile_rows = rows; P.tile_smem = rs * rows;
                        break;
                    }
                }
            } else {
                // shrinking reads a large source rectangle per output tile: the persistent strip kernel streams it through its
                // TMA ring (cfg1l: 0.36 ms against 0.56 ms for one box per tile); enlarging reads a small one and is bound by
                // the stores, which the tile kernel issues 16 bytes at a time
                if (scale_x > 1.25 || scale_y > 1.25)
                    gather_strip_tables(L.bb, P, c, [&](int x) { return clampi(xo[x], 0, cw - 1); }, [&](int x) { return clampi(xo[x] + 1, 0, cw - 1); },
                                        [&](int y) { return clampi(yo[y], 0, ch - 1); }, [&](int y) { return clampi(yo[y] + 1, 0, ch - 1); });
                else
                    gather_tile_tables(P, c, [&](int x) { return clampi(xo[x], 0, cw - 1); }, [&](int x) { return clampi(xo[x] + 1, 0, cw - 1); },
                                       [&](int y) { return clampi(yo[y], 0, ch - 1); }, [&](int y) { return clampi(yo[y] + 1, 0, ch - 1); });
            }
        }
    }

    // step 5: gray -> BGR, then filters in query order (bridge.c:606-627)
    *step = IMP_STEP_FILTERING;
    P.oc = (c == 1) ? 3 : c;
    L.fr = Frame{rw, rh, P.oc};
    for (int i = 0; i < req->filter_count; i++) {
        int code = lower_filter(L, req->filters[i] ? req->filters[i] : "", cfg ? cfg->allow_experiments : 0);
        if (code) return code;
    }

    // a pass 0 that stayed a plain index map (crop / no resize) takes the gather tile kernel as well
    if (!dry && L.hdr.kind == IMP_G_COPY) L.copy_tables();

    // step 6: watermark (bridge.c:629-640, 239-281)
    *step = IMP_STEP_WATERMARK;
    unsigned long long wm_bytes = 0;
    if (cfg && cfg->watermark) {
        const imp_gpu_watermark* wm = cfg->watermark;
        if (!wm->pixels || wm->width <= 0 || wm->height <= 0 || (wm->channels != 3 && wm->channels != 4))
            return IMP_ERROR_NO_SUCH_WATERMARK;
        int basew = L.fr.w, baseh = L.fr.h, left, top;
        if (wm->gravity_x == 'c') left = (basew - wm->width) / 2 + wm->offset_x;
        else if (wm->gravity_x == 'r') left = basew - wm->width - wm->offset_x;
        else left = wm->offset_x;
        if (wm->gravity_y == 'c') top = (baseh - wm->height) / 2 + wm->offset_y;
        else if (wm->gravity_y == 'b') top = baseh - wm->height - wm->offset_y;
        else top = wm->offset_y;
        // cvSetImageROI clips the work area to the image (App. C-8)
        int x0 = std::max(left, 0), y0 = std::max(top, 0);
        int x1 = std::min(left + wm->width, basew), y1 = std::min(top + wm->height, baseh);
        if (x1 <= x0 || y1 <= y0) return IMP_ERROR_INVALID_ARGS;
        int ew = std::min(wm->width, basew - x0), eh = std::min(wm->height, baseh - y0);     // filters.c:624-625
        ImpOp o{}; o.kind = IMP_OP_WATERMARK;
        o.i[0] = x0; o.i[1] = y0; o.i[2] = ew; o.i[3] = eh;
        float opacity = (float)(wm->opacity / 100.0);
        o.f[0] = 1 - opacity;
        o.map = L.fr.map();
        L.push(o);
        L.uses_wm = true;
        if (!dry) plan->wm = imp_wm_intern(wm);         // shared by content: PrepareWatermark decodes once (bridge.c:199-237)
        wm_bytes = (unsigned long long)ew * eh * wm->channels;
    }

    // flatten (bridge.c:642-656)
    if (req->flatten && L.fr.c == 4) { ImpOp o{}; o.kind = IMP_OP_PAPER; L.push(o); }
    L.fuse_flush();

    *step = IMP_STEP_ENCODE;
    // encoder-side pixel prep (advancedio.c:65-101 IplToFI32 / IplToFI24): FreeImage bitmaps are bottom-up, 32-bit ones
    // get alpha 255 when the frame has none, 24-bit ones drop the alpha. A final vertical flip of the store map plus a
    // destination channel count; no extra pass.
    if (req->pack != IMP_PACK_NONE && req->pack != IMP_PACK_FI24 && req->pack != IMP_PACK_FI32) return IMP_ERROR_INVALID_ARGS;
    if (req->pack != IMP_PACK_NONE) {
        L.fr.flip_v();
        L.final_dc = req->pack == IMP_PACK_FI32 ? 4 : 3;
    }
    L.end_pass(L.fr.map(), L.fr.w, L.fr.h);
    plan->out_w = L.fr.w; plan->out_h = L.fr.h; plan->out_c = L.final_dc ? L.final_dc : L.fr.c;
    plan->algo_bytes = (unsigned long long)cw * ch * c + (unsigned long long)plan->out_w * plan->out_h * plan->out_c + wm_bytes;
    return IMP_OK;
}
