// imp_pixel.cuh — per-pixel arithmetic of the filter chain, written once for device and host.
//
// Device code is the product. The host instantiation exists only so that the test suite can walk this
// exact source on a machine without a GPU (a test-only harness under tests/, built with g++); the
// shipped library never runs pixel math on the CPU.
//
// Every float operation below rounds exactly once, in the order the reference's C evaluates it
// (SURVEY §8a "Spec check"): device code uses the __f*_rn intrinsics (never contracted into FMA), host
// code is compiled with -ffp-contract=off. Stores through the reference's `char* imageData`
// (helpers.h:2) are "truncate toward zero, keep the low byte", with x86's out-of-range result
// (INT_MIN) reproduced by f2i_x86().
#pragma once
#include <stdint.h>
#include <math.h>
#include <string.h>
#include "imp_plan.h"

#if defined(__CUDACC__)
#define IMP_HD __host__ __device__ __forceinline__
#else
#define IMP_HD inline
#endif

#if defined(__CUDACC__)
// x/255.0f and (2x)/60.0f for every byte x, divided on the host with IEEE float division (imp_gpu_init). The library is
// built without relocatable device code, so every kernel translation unit carries its own copy (2 KB) and exports an
// uploader built from imp_upload_tables_tu(); imp_upload_tables() (imp_kernels.cu) calls them all.
static __device__ float g_imp_div255[256];
static __device__ float g_imp_div30[256];
// ceil(2^31 / d) for d = 1..255 (0 for d = 0): floor(n / d) == umulhi(2n + 1, g_imp_recip31[d]) for 0 <= n < 2^16.
// (2n+1) * (2^31/d + e) / 2^32 = (n + 1/2)/d + (2n+1)e/2^32 with 0 <= e < 1: the first term lies at least 1/(2d) >= 2^-9
// below the next integer and never below floor(n/d); the second is < 2^-15.
static __device__ unsigned g_imp_recip31[256];
// HSV2RGB per hue byte H (helpers.c:109-176): h = 2H/60, sector i = floor(h), f = h - i. Of q = v(1 - s f) and
// t = v(1 - s(1 - f)) a sector uses exactly one: .x = the float bits of the factor it needs (f in odd sectors and in
// `default`, 1 - f in even ones, computed on the host in the reference's float order), .y = the PRMT selector that places
// {V, that value, p} into (b, g, r) for the sector.
static __device__ int2 g_imp_hsv[256];
#endif

#if defined(__CUDA_ARCH__)
#define IMP_FMUL(a, b) __fmul_rn((a), (b))
#define IMP_FADD(a, b) __fadd_rn((a), (b))
#define IMP_FSUB(a, b) __fsub_rn((a), (b))
#define IMP_FDIV(a, b) __fdiv_rn((a), (b))
#define IMP_RINT(a)    __float2int_rn(a)
#else
#define IMP_FMUL(a, b) ((float)(a) * (float)(b))
#define IMP_FADD(a, b) ((float)(a) + (float)(b))
#define IMP_FSUB(a, b) ((float)(a) - (float)(b))
#define IMP_FDIV(a, b) ((float)(a) / (float)(b))
#define IMP_RINT(a)    ((int)lrintf(a))
#endif

struct ImpPx { int b, g, r, a; };

// ---- device-only fast paths that keep int<->float conversions and divisions off the XU pipe -----------------
// (16 lanes/clk/SM on sm_100 vs 64+ for the ALU/FMA pipes; the first ncu capture of the pass kernel showed
// I2F alone at >100 % of the XU pipe). All of them are exact for the ranges stated.
#if defined(__CUDA_ARCH__)
// 0 <= x < 2^23 -> float, exact (LOP3 + FADD)
__device__ __forceinline__ float imp_u2f(int x) { return __fadd_rn(__uint_as_float(0x4B000000u | (unsigned)x), -8388608.0f); }
// 0 <= x < 2^23 -> trunc(x) (FADD.RZ + LOP3); NaN -> 0x400000 (low byte 0, like x86's INT_MIN)
__device__ __forceinline__ int imp_f2u(float x) { return __float_as_int(__fadd_rz(x, 8388608.0f)) & 0x7FFFFF; }
// floor(n / d) for 0 <= n <= 65535, 0 <= d <= 255 (0 when d == 0), exact: one table load + LEA + IMAD.HI (see g_imp_recip31)
__device__ __forceinline__ int imp_udiv16(int n, int d) {
    return (int)__umulhi(2u * (unsigned)n + 1u, __ldg(&g_imp_recip31[d]));
}
// |x| < 2^22 -> float, exact (IADD + FADD); float |x| < 2^22 -> round-half-even int (FADD + IADD)
__device__ __forceinline__ float imp_i2f22(int x) { return __fadd_rn(__int_as_float(0x4B400000 + x), -12582912.0f); }
__device__ __forceinline__ int imp_rint22(float x) { return __float_as_int(__fadd_rn(x, 12582912.0f)) - 0x4B400000; }
#else
inline float imp_i2f22(int x) { return (float)x; }
inline int imp_rint22(float x) { return (int)lrintf(x); }
inline float imp_u2f(int x) { return (float)x; }
inline int imp_f2u(float x) { return (x == x) ? (int)x : 0x400000; }
inline int imp_udiv16(int n, int d) { return d ? n / d : 0; }
#endif

// x86 cvttss2si: truncate; NaN / out of range -> 0x80000000.
IMP_HD int imp_f2i_x86(float v) {
    return (v > -2147483904.0f && v < 2147483648.0f) ? (int)v : (int)0x80000000;
}
IMP_HD int imp_f2b(float v) { return imp_f2i_x86(v) & 255; }
IMP_HD int imp_sat8(int v) { return v < 0 ? 0 : (v > 255 ? 255 : v); }
IMP_HD int imp_min(int a, int b) { return a < b ? a : b; }
IMP_HD int imp_max(int a, int b) { return a > b ? a : b; }

#if defined(__CUDACC__)
static inline cudaError_t imp_upload_tables_tu() {
    float a[256], b[256];
    for (int i = 0; i < 256; i++) { a[i] = (float)i / 255.0f; b[i] = (float)(i * 2) / 60.0f; }     // IEEE float division on the host
    unsigned r[256];
    r[0] = 0;
    for (unsigned d = 1; d < 256; d++) r[d] = (unsigned)(((1ull << 31) + d - 1) / d);
    int2 hs[256];
    for (int H = 0; H < 256; H++) {
        const float h = b[H];
        const int i = (int)h;
        const float f = h - (float)i;
        const bool use_q = (i & 1) != 0 || i >= 5;
        const float ff = use_q ? f : 1.0f - f;
        // source bytes of the packed word: 0 = V, 1 = q|t, 2 = p; result bytes: 0 = b, 1 = g, 2 = r, 3 = 0
        static const int sel[6] = {0x4012, 0x4102, 0x4201, 0x4210, 0x4120, 0x4021};     // sectors 0..4, default
        memcpy(&hs[H].x, &ff, 4);
        hs[H].y = sel[i < 5 ? i : 5];
    }
    cudaError_t e = cudaMemcpyToSymbol(g_imp_div255, a, sizeof a);
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(g_imp_div30, b, sizeof b);
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(g_imp_recip31, r, sizeof r);
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(g_imp_hsv, hs, sizeof hs);
    return e;
}
#endif

IMP_HD void imp_map_xy(const ImpFrameMap& m, int bx, int by, int& x, int& y) {
    int u = m.swap ? by : bx, v = m.swap ? bx : by;
    x = m.flipx ? m.w - 1 - u : u;
    y = m.flipy ? m.h - 1 - v : v;
}

// helpers.c:70-107 RGB2HSV (integer; C division truncates toward zero).
// Branch-free: the reference's `if (v != 0)` / `if (s != 0)` guards only skip work whose result is 0 anyway — v == 0
// means delta == 0, and s == 0 <=> delta == 0 (255*delta >= v as soon as delta >= 1), where the first maximum is r and
// num = g - b = 0 — and imp_udiv16 returns 0 for a zero divisor.
IMP_HD void imp_rgb2hsv(int b, int g, int r, int& h, int& s, int& v) {
    const int mn = imp_min(b, imp_min(g, r)), mx = imp_max(b, imp_max(g, r));
    const int delta = mx - mn;
    v = mx;
    s = imp_udiv16(255 * delta, v);
    const bool ir = mx == r, ig = mx == g;                                  // the reference tests r, then g, else b
    const int num = ir ? g - b : (ig ? b - r : r - g);
    const int base = ir ? 0 : (ig ? 60 : 120);
    const int q = imp_udiv16(30 * (num < 0 ? -num : num), delta);          // C division truncates toward zero
    h = base + (num < 0 ? -q : q);
    if (h < 0) h += 180;
}

// helpers.c:109-176 HSV2RGB (float32; `default:` also takes sector 6, i.e. H == 180).
// Inputs are the BYTES the reference would have stored (0..255).
// Branch-free: with S == 0 every product below is v * 1.0f, i.e. (V,V,V) like the reference's early return; of q and t only
// the one the sector uses is evaluated (q in odd sectors and in `default`, t in even ones), by the expression the
// reference evaluates; the sector switch is three selects.
IMP_HD void imp_hsv2rgb(int H, int S, int V, int& b, int& g, int& r) {
    const float v = imp_u2f(V);
#if defined(__CUDA_ARCH__)
    // device: the effective fraction and the sector's byte placement come from one 8-byte table entry (see g_imp_hsv)
    const float s = __ldg(&g_imp_div255[S]);
    const int2 e = __ldg(&g_imp_hsv[H]);
    const int p = imp_f2u(IMP_FMUL(v, IMP_FSUB(1.0f, s)));
    const int x = imp_f2u(IMP_FMUL(v, IMP_FSUB(1.0f, IMP_FMUL(s, __int_as_float(e.x)))));
    const unsigned o = __byte_perm((unsigned)V | ((unsigned)x << 8) | ((unsigned)p << 16), 0u, (unsigned)e.y);
    b = o & 255; g = (o >> 8) & 255; r = o >> 16;
#else
    const float s = IMP_FDIV((float)S, 255.0f);
    const float h = IMP_FDIV((float)(H * 2), 60.0f);
    const int i = imp_f2u(h);                                               // h >= 0: floor == trunc
    const float f = IMP_FSUB(h, imp_u2f(i));
    // v in [0,255], factors in [0,1]: plain truncation is in range
    const int p = imp_f2u(IMP_FMUL(v, IMP_FSUB(1.0f, s)));
    const bool use_q = (i & 1) != 0 || i >= 5;
    const float ff = use_q ? f : IMP_FSUB(1.0f, f);
    const int x = imp_f2u(IMP_FMUL(v, IMP_FSUB(1.0f, IMP_FMUL(s, ff))));    // q = v(1 - s f) or t = v(1 - s(1 - f))
    // sector:  0 (V,t,p)  1 (q,V,p)  2 (p,V,t)  3 (p,q,V)  4 (t,p,V)  default (V,p,q)      as (r,g,b)
    r = (i == 0 || i >= 5) ? V : ((i == 1 || i == 4) ? x : p);
    g = (i == 1 || i == 2) ? V : ((i == 0 || i == 3) ? x : p);
    b = (i == 3 || i == 4) ? V : ((i == 2 || i >= 5) ? x : p);
    // v in [0,255] and the factors in [0,1]: p, x are already bytes
#endif
}

// filters.c:524-547: (int)fmin(c*k/100.0, 255) stored through char == C-truncating (c*k)/100 capped at
// 255, low byte (SURVEY §8a "Simplifications"); the int product wraps like the reference's.
IMP_HD int imp_modulate_scale(int c, int k) {
    int t = (int)((unsigned)c * (unsigned)k);
    int q = t / 100;
    return (q > 255 ? 255 : q) & 255;
}

IMP_HD void imp_op_modulate(ImpPx& p, int dh, int ks, int kv) {
    if (ks == 0) {
        // saturation factor 0 ("sepia" = modulate=..,0,.. + colorize): S becomes 0 whatever it was, and HSV2RGB's S == 0
        // branch (helpers.c:117) returns (V,V,V) whatever the hue, with V = max(B,G,R) scaled. Same bytes, no divisions.
        p.b = p.g = p.r = imp_modulate_scale(imp_max(p.b, imp_max(p.g, p.r)), kv);
        return;
    }
    int h, s, v;
    imp_rgb2hsv(p.b, p.g, p.r, h, s, v);
    if (dh != 0) { h += dh; if (h > 180) h -= 180; h &= 255; }
    s = imp_modulate_scale(s, ks);
    v = imp_modulate_scale(v, kv);
    imp_hsv2rgb(h, s, v, p.b, p.g, p.r);
}

// filters.c:608-616: px[c] = (char)(beta*px[c] + rgb[2-c]*alpha); ca[] = rgb[2-c]*alpha from the host.
IMP_HD void imp_op_addcolor(ImpPx& p, float beta, float cb, float cg, float cr, bool nonneg) {
    if (nonneg) {           // beta, cb, cg, cr >= 0 (host-checked): sums are in [0, 2^23)
        p.b = imp_f2u(IMP_FADD(IMP_FMUL(beta, imp_u2f(p.b)), cb)) & 255;
        p.g = imp_f2u(IMP_FADD(IMP_FMUL(beta, imp_u2f(p.g)), cg)) & 255;
        p.r = imp_f2u(IMP_FADD(IMP_FMUL(beta, imp_u2f(p.r)), cr)) & 255;
    } else {
        p.b = imp_f2b(IMP_FADD(IMP_FMUL(beta, (float)p.b), cb));
        p.g = imp_f2b(IMP_FADD(IMP_FMUL(beta, (float)p.g), cg));
        p.r = imp_f2b(IMP_FADD(IMP_FMUL(beta, (float)p.r), cr));
    }
}

// filters.c:595-605: val = (int)(ct*val + br*255); clamp to [0,255]. br255 = br*255 from the host.
IMP_HD int imp_contrast1(int v, float ct, float br255) {
    const float x = IMP_FADD(IMP_FMUL(ct, imp_u2f(v)), br255);
    // (int)x on x86 then clamp: x < 0 -> 0; x < 256 -> trunc; x < 2^31 -> 255; x >= 2^31, inf, NaN -> INT_MIN -> 0
    if (!(x < 2147483648.0f)) return 0;
    const float c = x < 0.0f ? 0.0f : (x > 255.0f ? 255.0f : x);
    return imp_f2u(c);
}

// filters.c:335-346: fmax(fmin(v*1.5-50,255),0) truncated == (3v-100)>>1 clamped.
IMP_HD int imp_lomo1(int v) {
    int t = 3 * v - 100;
    return t < 0 ? 0 : imp_min(t >> 1, 255);
}

// filters.c:356-403 Rainbow on HSV bytes; returns via hsv2rgb. Hue bytes are (char)(hue/2.0).
IMP_HD void imp_op_rainbow(ImpPx& p, int sat) {
    int h, s, v;
    imp_rgb2hsv(p.b, p.g, p.r, h, s, v);
    int hue = h * 2, light = v, saturation = sat, hb;
    if (light < 20) { light = 0; saturation = 0; hb = h; }
    else if (light > 254) { saturation = 0; hb = h; }
    else if (hue <= 10 || hue > 340) hb = 0;
    else if (hue < 35) hb = 15;
    else if (hue < 68) hb = 30;
    else if (hue < 150) hb = 60;
    else if (hue < 200) hb = 97;     // 195/2.0 = 97.5 -> 97
    else if (hue < 250) hb = 112;    // 225/2.0 = 112.5 -> 112
    else hb = 142;                   // 285/2.0 = 142.5 -> 142 (run-time truncation, App. C-1)
    imp_hsv2rgb(hb, saturation & 255, light, p.b, p.g, p.r);
}

// filters.c:405-455 Scanline: every row takes the HSV round trip; rows with freq <= (y mod period) <
// freq+width get S,V overwritten (closed form of the row state machine, SURVEY a19).
IMP_HD void imp_op_scanline(ImpPx& p, int y, int period, int freq, int sbyte, int vbyte) {
    int h, s, v;
    imp_rgb2hsv(p.b, p.g, p.r, h, s, v);
    int ph = y % period;
    if (ph >= freq && ph < period - 1) { s = sbyte; v = vbyte; }
    imp_hsv2rgb(h, s, v, p.b, p.g, p.r);
}

// filters.c:693-703 RadialGradient + helpers.c:46-48 Dist for one pixel.
// dx*dx+dy*dy is exact in double, sqrt is correctly rounded, narrowing matches the reference; cos and the 4th power are
// double, then narrowed: within 9.5 double ulp of cos^4 for glibc's cos+pow and CUDA's cos+2 squarings, so the float agrees
// unless a float rounding boundary is that close (no such entry in any frame the tests use: tests/vignette_ref.py).
#if defined(__CUDACC__)
static __host__ __device__ __noinline__     // double cos + its slow path: large and rare, keep one copy per kernel
#else
inline
#endif
float imp_vignette_mask(int x, int y, int cx, int cy, float maxr, float intensity) {
    double dx = (double)(cx - x), dy = (double)(cy - y);
    float distance = (float)sqrt(dx * dx + dy * dy);
    float raw = IMP_FMUL(IMP_FDIV(distance, maxr), intensity);
    double c = cos((double)raw);
    double c2 = c * c;
    return (float)(c2 * c2);
}

IMP_HD void imp_op_vignette_masked(ImpPx& p, float mask) {
    int h, s, v;
    imp_rgb2hsv(p.b, p.g, p.r, h, s, v);
    v = imp_f2u(IMP_FMUL(imp_u2f(v), mask)) & 255;          // mask = cos^4 >= 0 (NaN -> low byte 0, as on x86)
    imp_hsv2rgb(h, s, v, p.b, p.g, p.r);
}

IMP_HD void imp_op_vignette(ImpPx& p, int x, int y, int cx, int cy, float maxr, float intensity) {
    float mask = imp_vignette_mask(x, y, cx, cy, maxr, intensity);
    int h, s, v;
    imp_rgb2hsv(p.b, p.g, p.r, h, s, v);
    v = imp_f2u(IMP_FMUL(imp_u2f(v), mask)) & 255;          // mask = cos^4 >= 0 (NaN -> low byte 0, as on x86)
    imp_hsv2rgb(h, s, v, p.b, p.g, p.r);
}

// x/255.0 narrowed to float == x/255.0f correctly rounded for every byte x (checked exhaustively in
// the CPU test suite, test_alpha_unit_identity), so one IEEE float division replaces the double divide + narrowing.
IMP_HD float imp_alpha_unit(int a) {
#if defined(__CUDA_ARCH__)
    return __ldg(&g_imp_div255[a]);
#else
    return IMP_FDIV((float)a, 255.0f);
#endif
}

// filters.c:619-662 AlphaBlendOver for one pixel. alpha = 1 - opacity (host float).
// dst_has_a / src_has_a: nChannels == 4.
IMP_HD void imp_op_over(ImpPx& d, bool dst_has_a, int sb, int sg, int sr, int sa, bool src_has_a, float alpha) {
    float dA = dst_has_a ? imp_alpha_unit(d.a) : 1.0f;
    float sA = src_has_a ? imp_alpha_unit(sa) : 1.0f;
    sA = IMP_FSUB(sA, alpha);
    sA = sA > 0.0f ? sA : 0.0f;                      // fmax(sA - alpha, 0)
    float one_m = IMP_FSUB(1.0f, sA);
    float tA = IMP_FADD(sA, IMP_FMUL(dA, one_m));
    if (tA == 0.0f) { d.b = d.g = d.r = 0; }
    else {
        // all terms are >= 0 and the quotients stay far below 2^23
        d.b = imp_f2u(IMP_FDIV(IMP_FADD(IMP_FMUL(imp_u2f(sb), sA), IMP_FMUL(IMP_FMUL(imp_u2f(d.b), dA), one_m)), tA)) & 255;
        d.g = imp_f2u(IMP_FDIV(IMP_FADD(IMP_FMUL(imp_u2f(sg), sA), IMP_FMUL(IMP_FMUL(imp_u2f(d.g), dA), one_m)), tA)) & 255;
        d.r = imp_f2u(IMP_FDIV(IMP_FADD(IMP_FMUL(imp_u2f(sr), sA), IMP_FMUL(IMP_FMUL(imp_u2f(d.r), dA), one_m)), tA)) & 255;
    }
    if (dst_has_a) d.a = imp_f2u(IMP_FMUL(tA, 255.0f)) & 255;
}

// filters.c:666-687 BlendWithPaper for one pixel.
IMP_HD void imp_op_paper(ImpPx& p) {
    float diff = imp_u2f(255 - p.a);
    float pa = imp_alpha_unit(p.a);
    p.b = imp_f2u(IMP_FADD(diff, IMP_FMUL(imp_u2f(p.b), pa))) & 255;
    p.g = imp_f2u(IMP_FADD(diff, IMP_FMUL(imp_u2f(p.g), pa))) & 255;
    p.r = imp_f2u(IMP_FADD(diff, IMP_FMUL(imp_u2f(p.r), pa))) & 255;
    p.a = 255;
}

// Runs the op list of a pass on N pixels at base coordinates (bx[n],by[n]): the op loop is the outer one, so an op's
// parameters and its dispatch are paid once per N pixels and the N bodies are independent instruction streams.
// lut: the pass's LUT area; wm*: this job's watermark.
// LIGHT: the pass holds nothing but fused tables (ImpPass::light): the interpreter then knows only IMP_OP_LUT3 / IMP_OP_MAXLUT3,
// which keeps the HSV / watermark / vignette code and its registers out of the kernel instantiation.
// NOCOMP: the pass holds no compositing op (IMP_OP_WATERMARK / IMP_OP_PAPER; ImpPass::light == 2): the instantiation leaves
// AlphaBlendOver's float divisions and their registers out.
// COMPONLY: nothing but compositing ops and fused tables (ImpPass::light & 4 — the standard "resize + watermark" request):
// the HSV / vignette / gradmap code stays out.
template <int N, bool LIGHT = false, bool NOCOMP = false, bool COMPONLY = false>
IMP_HD void imp_run_ops_n(ImpPx (&px)[N], int oc, const int (&bx)[N], const int (&by)[N], const ImpOp* ops, int nops, const uint8_t* lut,
                          const uint8_t* wm, int wm_pitch, int wm_c) {
    if (LIGHT) {
        for (int k = 0; k < nops; k++) {
            const ImpOp& op = ops[k];
            const uint8_t* t = lut + op.i[0];
            const bool al = op.i[1] != 0 && oc == 4, mx = op.kind == IMP_OP_MAXLUT3;
#pragma unroll
            for (int n = 0; n < N; n++) {
                ImpPx& p = px[n];
                const int m = imp_max(p.b, imp_max(p.g, p.r));
                p.b = t[mx ? m : p.b]; p.g = t[256 + (mx ? m : p.g)]; p.r = t[512 + (mx ? m : p.r)];
                if (al) p.a = t[768 + p.a];
            }
        }
        return;
    }
    for (int k = 0; k < nops; k++) {
        const ImpOp& op = ops[k];
        switch (op.kind) {
            case IMP_OP_MODULATE: {
                if (COMPONLY) break;
                const int a = op.i[0], b = op.i[1], c = op.i[2];
#pragma unroll
                for (int n = 0; n < N; n++) imp_op_modulate(px[n], a, b, c);
            } break;
            case IMP_OP_ADDCOLOR: {
                if (COMPONLY) break;
                const float f0 = op.f[0], f1 = op.f[1], f2 = op.f[2], f3 = op.f[3];
                const bool nonneg = op.i[0] != 0;
#pragma unroll
                for (int n = 0; n < N; n++) imp_op_addcolor(px[n], f0, f1, f2, f3, nonneg);
            } break;
            case IMP_OP_LUT_ALL: {
                if (COMPONLY) break;
                const uint8_t* t = lut + op.i[0];
#pragma unroll
                for (int n = 0; n < N; n++) {
                    ImpPx& p = px[n];
                    p.b = t[p.b]; p.g = t[p.g]; p.r = t[p.r];
                    if (oc == 4) p.a = t[p.a];
                }
            } break;
            case IMP_OP_CONTRAST: {
                if (COMPONLY) break;
                const float f0 = op.f[0], f1 = op.f[1];
#pragma unroll
                for (int n = 0; n < N; n++) {
                    ImpPx& p = px[n];
                    p.b = imp_contrast1(p.b, f0, f1);
                    p.g = imp_contrast1(p.g, f0, f1);
                    p.r = imp_contrast1(p.r, f0, f1);
                }
            } break;
            case IMP_OP_GRADMAP: {
                if (COMPONLY) break;
                const uint8_t* t0 = lut + op.i[0];
#pragma unroll
                for (int n = 0; n < N; n++) {
                    ImpPx& p = px[n];
                    const uint8_t* t = t0 + ((p.r + p.g + p.b) / 3) * 3;
                    p.r = t[0]; p.g = t[1]; p.b = t[2];
                }
            } break;
            case IMP_OP_VIGNETTE: {
                if (COMPONLY) break;
#if defined(__CUDA_ARCH__)
                const float* tab = reinterpret_cast<const float*>(((unsigned long long)(unsigned)op.i[5] << 32) | (unsigned)op.i[4]);
                if (tab) {           // mask[|dy|][|dx|], tabulated per plan by imp_vignette_table_kernel with the code of imp_vignette_mask
                    const int stride = op.i[2];
                    // dx = cx - x with x = flipx ? w-1-u : u and u = swap ? by : bx is affine in the base coordinates:
                    // dx = ox + xa*bx + xb*by, dy = oy + ya*bx + yb*by. The runtime stores that form into the device copy
                    // of the op when it attaches the table (plan_to_device: i[0..1] = ox, oy; the map's fields = xa, xb, ya,
                    // yb), so nothing is derived here, and a caller whose pixels share a column (or a row) leaves one add
                    // per pixel. The table carries IMP_VIGNETTE_MARGIN entries beyond the frame in both directions: tile
                    // kernels may evaluate (never store) pixels of a partial tile that lie up to that far outside.
                    const int ox = op.i[0], oy = op.i[1];
                    const int xa = op.map.swap, xb = op.map.flipx, ya = op.map.flipy, yb = op.map.w;
                    float mask[N];
#pragma unroll
                    for (int n = 0; n < N; n++) {
                        const int dx = ox + xa * bx[n] + xb * by[n], dy = oy + ya * bx[n] + yb * by[n];
                        mask[n] = __ldg(tab + (dy < 0 ? -dy : dy) * stride + (dx < 0 ? -dx : dx));
                    }
#pragma unroll
                    for (int n = 0; n < N; n++) imp_op_vignette_masked(px[n], mask[n]);
                    break;
                }
#endif
                for (int n = 0; n < N; n++) {
                    int x, y; imp_map_xy(op.map, bx[n], by[n], x, y);
                    imp_op_vignette(px[n], x, y, op.i[0], op.i[1], op.f[0], op.f[1]);
                }
            } break;
            case IMP_OP_LOMO:
                if (COMPONLY) break;
#pragma unroll
                for (int n = 0; n < N; n++) { px[n].g = imp_lomo1(px[n].g); px[n].r = imp_lomo1(px[n].r); }
                break;
            case IMP_OP_RAINBOW: {
                if (COMPONLY) break;
                const int a = op.i[0];
#pragma unroll
                for (int n = 0; n < N; n++) imp_op_rainbow(px[n], a);
            } break;
            case IMP_OP_SCANLINE:
                if (COMPONLY) break;
#pragma unroll
                for (int n = 0; n < N; n++) {
                    int x, y; imp_map_xy(op.map, bx[n], by[n], x, y);
                    imp_op_scanline(px[n], y, op.i[0], op.i[1], op.i[3], op.i[4]);
                }
                break;
            case IMP_OP_WATERMARK:
                if (NOCOMP) break;
#pragma unroll
                for (int n = 0; n < N; n++) {
                    int x, y; imp_map_xy(op.map, bx[n], by[n], x, y);
                    int wx = x - op.i[0], wy = y - op.i[1];
                    if (wx >= 0 && wy >= 0 && wx < op.i[2] && wy < op.i[3]) {
                        const uint8_t* s = wm + (size_t)wy * wm_pitch + (size_t)wx * wm_c;
                        imp_op_over(px[n], oc == 4, s[0], s[1], s[2], wm_c == 4 ? s[3] : 255, wm_c == 4, op.f[0]);
                    }
                }
                break;
            case IMP_OP_LUT3: {
                const uint8_t* t = lut + op.i[0];
                const bool al = op.i[1] != 0 && oc == 4;
#pragma unroll
                for (int n = 0; n < N; n++) {
                    ImpPx& p = px[n];
                    p.b = t[p.b]; p.g = t[256 + p.g]; p.r = t[512 + p.r];
                    if (al) p.a = t[768 + p.a];
                }
            } break;
            case IMP_OP_MAXLUT3: {
                const uint8_t* t = lut + op.i[0];
                const bool al = op.i[1] != 0 && oc == 4;
#pragma unroll
                for (int n = 0; n < N; n++) {
                    ImpPx& p = px[n];
                    const int m = imp_max(p.b, imp_max(p.g, p.r));
                    p.b = t[m]; p.g = t[256 + m]; p.r = t[512 + m];
                    if (al) p.a = t[768 + p.a];
                }
            } break;
            case IMP_OP_PAPER:
                if (NOCOMP) break;
                if (oc == 4) {
#pragma unroll
                    for (int n = 0; n < N; n++) imp_op_paper(px[n]);
                }
                break;
            default: break;
        }
    }
}

// One pixel.
IMP_HD void imp_run_ops(ImpPx& p, int oc, int bx, int by, const ImpOp* ops, int nops, const uint8_t* lut,
                        const uint8_t* wm, int wm_pitch, int wm_c) {
    ImpPx px[1] = {p};
    const int xs[1] = {bx}, ys[1] = {by};
    imp_run_ops_n<1>(px, oc, xs, ys, ops, nops, lut, wm, wm_pitch, wm_c);
    p = px[0];
}
