/*
 * imp_oracle.c — CPU restatement of IMP's decoded-pixel hot path.
 *
 * TEST INFRASTRUCTURE ONLY. This file is the checker the CUDA path is compared against; it is
 * never linked into, imported by, or called from the product (ngx_http_imgproc_b200/). Only
 * tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may use it.
 *
 * Two families of functions:
 *   1. hand-written reference arithmetic, restated from /root/reference/{filters,helpers,bridge}.c
 *      (each function cites the file:line it follows). Pinned against the reference's own code
 *      compiled unmodified (oracle/_ref/libimp_ref.so, see oracle/Makefile) in tests/test_oracle_*.py.
 *   2. the OpenCV calls the reference makes (cvCopy+ROI, cvResize, cvFlip, cvTranspose, cvSmooth,
 *      cvCvtColor). OpenCV 2.4.9 (docs/01 - Installation.md:25, config:5) is NOT vendored under
 *      /root/reference, so these restate OpenCV's published algorithms (SURVEY.md Appendix A) and are
 *      pinned against cv2 4.13.0 with IPP off, the only OpenCV in this image. Known version gap
 *      (2.4.9 vs 4.13: Gaussian tap rounding, SIMD cubic path) is stated in DESIGN.md.
 *
 * Conventions: 8-bit unsigned interleaved images, channel order B,G,R[,A] (required.h:65-69),
 * pixel (x,y,c) at data[step*y + x*channels + c] (helpers.h:1). Build: gcc -O2 -ffp-contract=off
 * (no FMA contraction; every float op rounds once, like the reference built with nginx's -O).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <limits.h>
#include <float.h>

typedef struct {
    unsigned char* data;
    int width, height, channels, step;
} orc_img;

#define PX(im, x, y, c) ((im)->data[(size_t)(im)->step * (y) + (size_t)(x) * (im)->channels + (c)])

/* float/double -> int exactly as x86-64 cvttss2si/cvttsd2si do (what gcc emits for the reference's
 * implicit conversions): truncate toward zero; out of range or NaN -> INT_MIN ("integer indefinite").
 * A following store through char* keeps the low byte (helpers.h:2, SURVEY finding 5). */
static inline int f2i(float v)  { return (v > -2147483904.0f && v < 2147483648.0f) ? (int)v : INT_MIN; }
static inline int d2i(double v) { return (v > -2147483649.0 && v < 2147483648.0) ? (int)v : INT_MIN; }
static inline unsigned char f2b(float v)  { return (unsigned char)(unsigned)f2i(v); }
static inline unsigned char d2b(double v) { return (unsigned char)(unsigned)d2i(v); }
static inline unsigned char i2b(int v)    { return (unsigned char)(unsigned)v; }
static inline int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }
static inline unsigned char sat_u8(int v) { return (unsigned char)(v < 0 ? 0 : (v > 255 ? 255 : v)); }

/* ------------------------------------------------------------------------------------------ */
/* 1. Hand-written reference arithmetic                                                        */
/* ------------------------------------------------------------------------------------------ */

/* helpers.c:70-107 RGB2HSV — integer, C division truncates toward zero, hue in [0,180). */
void orc_rgb2hsv_px(unsigned char* p) {
    int b = p[0], g = p[1], r = p[2];
    int mn = (g <= b) ? (r <= g ? r : g) : (r <= b ? r : b);      /* helpers.h:20 MIN3(r,g,b) */
    int mx = (g >= b) ? (r >= g ? r : g) : (r >= b ? r : b);      /* helpers.h:21 MAX3(r,g,b) */
    int delta = mx - mn, h = 0, s = 0, v = mx;
    if (v != 0) s = 255 * delta / v;
    if (s != 0) {
        if (mx == r)      h = 30 * (g - b) / delta;
        else if (mx == g) h = 60 + 30 * (b - r) / delta;
        else              h = 120 + 30 * (r - g) / delta;
    }
    if (h < 0) h += 180;
    p[0] = (unsigned char)h; p[1] = (unsigned char)s; p[2] = (unsigned char)v;
}

/* helpers.c:109-176 HSV2RGB — float32, one rounding per op, truncating stores;
 * `default:` also takes sector 6 (H==180), SURVEY App. C-3. */
void orc_hsv2rgb_px(unsigned char* p) {
    float h = (float)(p[0] * 2), s = (float)p[1], v = (float)p[2];
    int r, g, b;
    if (s == 0) {
        r = g = b = f2i(v);
    } else {
        s = s / 255.0f;
        h = h / 60.0f;
        int i = (int)floor((double)h);
        float f = h - (float)i;
        int pp = f2i(v * (1.0f - s));
        int q  = f2i(v * (1.0f - s * f));
        int t  = f2i(v * (1.0f - s * (1.0f - f)));
        int vi = f2i(v);
        switch (i) {
            case 0:  r = vi; g = t;  b = pp; break;
            case 1:  r = q;  g = vi; b = pp; break;
            case 2:  r = pp; g = vi; b = t;  break;
            case 3:  r = pp; g = q;  b = vi; break;
            case 4:  r = t;  g = pp; b = vi; break;
            default: r = vi; g = pp; b = q;  break;
        }
    }
    p[0] = i2b(b); p[1] = i2b(g); p[2] = i2b(r);
}

void orc_rgb2hsv(orc_img* im) {
    for (int y = 0; y < im->height; y++) for (int x = 0; x < im->width; x++) orc_rgb2hsv_px(&PX(im, x, y, 0));
}
void orc_hsv2rgb(orc_img* im) {
    for (int y = 0; y < im->height; y++) for (int x = 0; x < im->width; x++) orc_hsv2rgb_px(&PX(im, x, y, 0));
}

/* filters.c:524-547 ModulateHSV. hsv[] are the already-validated ints of Modulate (filters.c:135-158). */
void orc_modulate_hsv(orc_img* im, const int* hsv) {
    for (int y = 0; y < im->height; y++) for (int x = 0; x < im->width; x++) {
        unsigned char* p = &PX(im, x, y, 0);
        orc_rgb2hsv_px(p);
        if (hsv[0] != 0) {
            int hue = p[0] + hsv[0];
            if (hue > 180) hue -= 180;                    /* required.h:64 CV_HUE_WHEEL_RESOLUTION */
            p[0] = i2b(hue);
        }
        for (int c = 1; c < 3; c++) {
            int cval = p[c];
            /* int*int wraps in the reference's build; /100.0 and fmin are double; then (int) */
            cval = d2i(fmin((double)(int)((unsigned)cval * (unsigned)hsv[c]) / 100.0, 255));
            p[c] = i2b(cval);
        }
        orc_hsv2rgb_px(p);
    }
}

/* filters.c:608-616 AlphaBlendAddColor (Colorize core): float32, truncating char store. */
void orc_add_color(orc_img* im, const int* rgb, float alpha) {
    float beta = 1 - alpha;
    for (int y = 0; y < im->height; y++) for (int x = 0; x < im->width; x++)
        for (int c = 0; c < 3; c++) {
            float v = (beta * (float)PX(im, x, y, c)) + ((float)rgb[2 - c] * alpha);
            PX(im, x, y, c) = f2b(v);
        }
}

/* filters.c:561-570 CalculateGammaLUT: inverse is float32, pow/divide/multiply are double. */
void orc_gamma_lut(float gamma, int* lut) {
    float inverse = 1 / gamma;
    for (int i = 0; i < 256; i++) lut[i] = d2i(pow(i / 255.0, inverse) * 255.0);
}

/* filters.c:549-559 ApplyGamma: ALL channels, alpha included (App. C-5). */
void orc_gamma(orc_img* im, float gamma) {
    int lut[256];
    orc_gamma_lut(gamma, lut);
    for (int y = 0; y < im->height; y++) for (int x = 0; x < im->width; x++)
        for (int c = 0; c < im->channels; c++) PX(im, x, y, c) = i2b(lut[PX(im, x, y, c)]);
}

/* filters.c:595-605 BrightnessContrast: first min(C,3) channels, float32 then clamp. */
void orc_brightness_contrast(orc_img* im, float br, float ct) {
    int nc = im->channels < 3 ? im->channels : 3;
    for (int y = 0; y < im->height; y++) for (int x = 0; x < im->width; x++)
        for (int c = 0; c < nc; c++) {
            int val = PX(im, x, y, c);
            val = f2i((ct * (float)val) + (br * 255));
            val = val > 255 ? 255 : val;
            val = val < 0 ? 0 : val;
            PX(im, x, y, c) = (unsigned char)val;
        }
}

/* filters.c:572-593 CalculateGradientLUT. The reference leaves lut[(int)inner*(n-1)*3 ..] uninitialised
 * (App. C-4); the restatement defines that tail as 0 and callers exclude it from parity. */
void orc_gradient_lut(const unsigned char* colors /* n*3, as parsed: [0]=RR [1]=GG [2]=BB */, int n, unsigned char* lut /* 768 */) {
    int segments = n - 1;
    float inner = 256 / (float)segments;
    int pointer = 0;
    memset(lut, 0, 768);
    for (int c = 0; c < segments; c++) {
        const unsigned char* from = colors + 3 * c;
        const unsigned char* to = colors + 3 * (c + 1);
        for (int i = 0; i < (int)inner; i++) {
            float step = i / inner;
            for (int j = 0; j < 3; j++) {
                float v = (float)from[j] + step * (float)(to[j] - from[j]);
                lut[pointer++] = (unsigned char)d2i(round((double)v));
            }
        }
    }
}

/* filters.c:260-277 Gradmap per-pixel remap. */
void orc_gradmap(orc_img* im, const unsigned char* lut) {
    for (int y = 0; y < im->height; y++) for (int x = 0; x < im->width; x++) {
        unsigned char* p = &PX(im, x, y, 0);
        int offset = ((p[2] + p[1] + p[0]) / 3) * 3;
        p[2] = lut[offset + 0]; p[1] = lut[offset + 1]; p[0] = lut[offset + 2];
    }
}

/* helpers.c:46-48 Dist: float args promoted to double, pow(.,2), sqrt, narrowed to float. */
static float orc_dist(int ax, int ay, int bx, int by) {
    return (float)sqrt(pow((double)(float)(ax - bx), 2) + pow((double)(float)(ay - by), 2));
}
/* helpers.c:50-66 GetMaxDisFromCorners. */
static float orc_max_corner_dist(int w, int h, int cx, int cy) {
    int xs[4] = {0, w, 0, w}, ys[4] = {0, 0, h, h};
    float m = 0;
    for (int i = 0; i < 4; i++) { float d = orc_dist(xs[i], ys[i], cx, cy); if (m < d) m = d; }
    return m;
}
/* filters.c:693-703 RadialGradient for one pixel. */
float orc_vignette_mask(int x, int y, int w, int h, float power, float radius) {
    int cx = w / 2, cy = h / 2;
    float maxr = radius * orc_max_corner_dist(w, h, cx, cy);
    float distance = orc_dist(cx, cy, x, y);
    float raw = distance / maxr * power;
    return (float)pow(cos((double)raw), 4);
}
/* orc_vignette_mask at |dx| = i < nx, |dy| = j < ny from the centre of a w x h frame, into out[j * nx + i]. */
void orc_vignette_mask_table(float* out, int nx, int ny, int w, int h, float power, float radius) {
    for (int j = 0; j < ny; j++) for (int i = 0; i < nx; i++) out[(long)j * nx + i] = orc_vignette_mask(w / 2 - i, h / 2 - j, w, h, power, radius);
}
/* filters.c:295-323 Vignette. */
void orc_vignette(orc_img* im, float intensity, float radius) {
    int w = im->width, h = im->height, cx = w / 2, cy = h / 2;
    float maxr = radius * orc_max_corner_dist(w, h, cx, cy);
    for (int y = 0; y < h; y++) for (int x = 0; x < w; x++) {
        unsigned char* p = &PX(im, x, y, 0);
        float distance = orc_dist(cx, cy, x, y);
        float raw = distance / maxr * intensity;
        float mask = (float)pow(cos((double)raw), 4);
        orc_rgb2hsv_px(p);
        p[2] = f2b((float)p[2] * mask);
        orc_hsv2rgb_px(p);
    }
}

/* filters.c:335-346 Lomo: channels 1,2 (G,R), double math, float store. */
void orc_lomo(orc_img* im) {
    for (int y = 0; y < im->height; y++) for (int x = 0; x < im->width; x++)
        for (int c = 1; c < 3; c++) {
            float val = PX(im, x, y, c);
            val = (float)fmax(fmin(val * 1.5 - 50, 255), 0);
            PX(im, x, y, c) = f2b(val);
        }
}

/* filters.c:325-333 Gotham, :348-354 Kelvin — compositions. */
void orc_gotham(orc_img* im) {
    int hsv[3] = {120, 5, 100}, rgb[3] = {17, 27, 93};
    orc_modulate_hsv(im, hsv);
    orc_add_color(im, rgb, (float)0.15);
    orc_gamma(im, (float)0.3);
    orc_brightness_contrast(im, (float)-0.07, (float)1.5);
}
void orc_kelvin(orc_img* im) {
    int hsv[3] = {120, 50, 100}, rgb[3] = {255, 153, 0};
    orc_modulate_hsv(im, hsv);
    orc_add_color(im, rgb, (float)0.5);
}

/* filters.c:356-403 Rainbow. hue/2.0 is stored through char: truncation at run time (-O1), App. C-1. */
void orc_rainbow(orc_img* im, int sat) {
    for (int y = 0; y < im->height; y++) for (int x = 0; x < im->width; x++) {
        unsigned char* p = &PX(im, x, y, 0);
        orc_rgb2hsv_px(p);
        int hue = p[0] * 2, light = p[2], saturation = sat;
        if (light < 20) { light = 0; saturation = 0; }
        else if (light > 254) { saturation = 0; }
        else if (hue <= 10 || hue > 340) hue = 0;
        else if (hue >= 10 && hue < 35) hue = 30;
        else if (hue >= 35 && hue < 68) hue = 60;
        else if (hue >= 68 && hue < 150) hue = 120;
        else if (hue >= 150 && hue < 200) hue = 195;
        else if (hue >= 200 && hue < 250) hue = 225;
        else hue = 285;
        p[0] = d2b(hue / 2.0); p[1] = i2b(saturation); p[2] = i2b(light);
        orc_hsv2rgb_px(p);
    }
}

/* filters.c:432-452 Scanline row state machine, kept as the reference wrote it. */
void orc_scanline(orc_img* im, float intensity, float opacity, int freq, int width) {
    for (int y = 0; y < im->height; y++) for (int x = 0; x < im->width; x++) orc_rgb2hsv_px(&PX(im, x, y, 0));
    int skipped = 0, drawed = 0;
    for (int y = 0; y < im->height; y++) {
        if (skipped == freq) {
            if (drawed == width) { skipped = drawed = 0; }
            else {
                for (int x = 0; x < im->width; x++) {
                    PX(im, x, y, 1) = f2b(255 * opacity);
                    PX(im, x, y, 2) = f2b(255 * intensity);
                }
                drawed++;
            }
        } else skipped++;
    }
    for (int y = 0; y < im->height; y++) for (int x = 0; x < im->width; x++) orc_hsv2rgb_px(&PX(im, x, y, 0));
}

/* filters.c:619-662 AlphaBlendOver with the ROI origin (x0,y0) that Watermark sets (bridge.c:273-276).
 * x0,y0 are the ROI offsets AFTER cvSetImageROI's clipping (App. C-8). */
void orc_alpha_over(orc_img* dst, int x0, int y0, const orc_img* src, float opacity) {
    float alpha = 1 - opacity;
    int maxrow = src->height < dst->height - y0 ? src->height : dst->height - y0;
    int maxcol = src->width < dst->width - x0 ? src->width : dst->width - x0;
    for (int row = 0; row < maxrow; row++) for (int col = 0; col < maxcol; col++) {
        unsigned char* d = &PX(dst, col + x0, row + y0, 0);
        const unsigned char* s = &PX(src, col, row, 0);
        int dB = d[0], dG = d[1], dR = d[2];
        float dA = dst->channels == 4 ? (float)(d[3] / 255.0) : 1;
        int sB = s[0], sG = s[1], sR = s[2];
        float sA = src->channels == 4 ? (float)(s[3] / 255.0) : 1;
        sA = (float)fmax(sA - alpha, 0);
        float tA = sA + dA * (1 - sA);
        int tB, tG, tR;
        if (tA == 0) { tB = tG = tR = 0; }
        else {
            tB = f2i(((float)sB * sA + (float)dB * dA * (1 - sA)) / tA);
            tG = f2i(((float)sG * sA + (float)dG * dA * (1 - sA)) / tA);
            tR = f2i(((float)sR * sA + (float)dR * dA * (1 - sA)) / tA);
        }
        d[0] = i2b(tB); d[1] = i2b(tG); d[2] = i2b(tR);
        if (dst->channels == 4) d[3] = f2b(tA * 255);
    }
}

/* bridge.c:254-276 Watermark placement + cvSetImageROI clipping -> ROI origin. Returns 0 if the
 * clipped ROI is empty (the reference would assert inside OpenCV, App. C-8), else 1. */
int orc_watermark_origin(int basew, int baseh, int overw, int overh, char gx, char gy, int ox, int oy, int* x0, int* y0) {
    int left, top;
    if (gx == 'c') left = (basew - overw) / 2 + ox; else if (gx == 'r') left = basew - overw - ox; else left = ox;
    if (gy == 'c') top = (baseh - overh) / 2 + oy; else if (gy == 'b') top = baseh - overh - oy; else top = oy;
    /* cvSetImageROI: rect &= (0,0,w,h) */
    int rx0 = left < 0 ? 0 : left, ry0 = top < 0 ? 0 : top;
    int rx1 = left + overw > basew ? basew : left + overw, ry1 = top + overh > baseh ? baseh : top + overh;
    if (rx1 <= rx0 || ry1 <= ry0) return 0;
    *x0 = rx0; *y0 = ry0;
    return 1;
}

/* filters.c:666-687 BlendWithPaper (4-channel only). */
void orc_blend_with_paper(orc_img* im) {
    for (int y = 0; y < im->height; y++) for (int x = 0; x < im->width; x++) {
        unsigned char* p = &PX(im, x, y, 0);
        int oB = p[0], oG = p[1], oR = p[2], oA = p[3];
        int diffalpha = 255 - oA;
        float prodalpha = (float)(oA / 255.0);
        p[0] = i2b(f2i((float)diffalpha + ((float)oB * prodalpha)));
        p[1] = i2b(f2i((float)diffalpha + ((float)oG * prodalpha)));
        p[2] = i2b(f2i((float)diffalpha + ((float)oR * prodalpha)));
        p[3] = 255;
    }
}

/* filters.c:707-729 CalcPerceivedBrightness: x-outer/y-inner float32 running sum. */
float orc_perceived_brightness(const orc_img* im) {
    float sum = 0;
    if (im->channels == 1) {
        for (int x = 0; x < im->width; x++) for (int y = 0; y < im->height; y++) sum += PX(im, x, y, 0);
    } else {
        for (int x = 0; x < im->width; x++) for (int y = 0; y < im->height; y++) {
            int r = PX(im, x, y, 2), g = PX(im, x, y, 1), b = PX(im, x, y, 0);
            sum += sqrt(r * r * 0.241 + g * g * 0.691 + b * b * 0.068);
        }
    }
    return sum / (im->width * im->height) / 255.0;
}

/* filters.c:486-522 ASCII: density = floor(V / factor), V = max(B,G,R) (RGB2HSV's value), factor = 256.0/len as float. */
long orc_ascii(const orc_img* im, int wide, unsigned char* out) {
    static const char w70[] = "$@B%8&WM#*oahkbdpqwmZO0QLCJUYXzcvunxrjft/\\|()1{}[]?-_+~<>i!lI;:,\"^`'. ";
    static const char n10[] = "@%8#*+=-:. ";
    const char* table = wide ? w70 : n10;
    int tablelen = (int)strlen(table);
    float factor = 256.0 / tablelen;
    int width = im->width, height = im->height;
    for (int y = 0; y < height; y++) {
        long rowoffset = (long)y * (width + 1);
        for (int x = 0; x < width; x++) {
            const unsigned char* p = &PX(im, x, y, 0);
            int v = im->channels == 1 ? p[0] : (p[0] > p[1] ? (p[0] > p[2] ? p[0] : p[2]) : (p[1] > p[2] ? p[1] : p[2]));
            int density = (int)floor(v / factor);
            out[rowoffset + x] = (unsigned char)table[density];
        }
        if (rowoffset > 0) out[rowoffset - 1] = '\n';
    }
    return (long)(width + 1) * height - 1;
}

/* advancedio.c:195-248 LoadGIF's per-pixel loop. Pinned against the reference's own LoadGIF (advancedio.c compiled
 * unmodified over oracle/fake_freeimage.c, tests/test_oracle.py). Three accidents of that loop, as restated here:
 *  - `x > left + w` (advancedio.c:203) lets x == left+w read row[w]: the scanline's pad byte or the first index of
 *    the next scanline. Restated while the byte lies inside the page's pitch*height block; past it -> the key.
 *  - a page without a transparent colour has key == -1 and uncovered pixels index palette[-1], which aliases the
 *    BITMAPINFOHEADER's biClrImportant (256 for 8-bit pages): bytes {0,1,0,0}.
 *  - `master` is uninitialised pool memory in the reference; it is only read before being written when frame 0 has
 *    DISPOSAL_BACKGROUND and transparent pixels. Zero here. */
typedef struct { const unsigned char* indices; int pitch, width, height, left, top, dispose, key; const unsigned char* palette; } orc_gif_frame;
void orc_gif_expand(const orc_gif_frame* frames, int n, int cw, int ch, int destructive, unsigned char* const* canvases, int cstep) {
    int* master = (int*)calloc((size_t)cw * ch, sizeof(int));
    for (int f = 0; f < n; f++) {
        const orc_gif_frame* fr = &frames[f];
        for (int y = 0; y < ch; y++) {
            int rowidx = fr->height + fr->top - y - 1;
            const unsigned char* row = (rowidx >= 0 && rowidx < fr->height) ? fr->indices + (size_t)rowidx * fr->pitch : NULL;
            for (int x = 0; x < cw; x++) {
                int coloridx;
                if (!row || x < fr->left || y < fr->top || x > fr->left + fr->width || y > fr->top + fr->height) coloridx = fr->key;
                else if (rowidx * fr->pitch + (x - fr->left) >= fr->height * fr->pitch) coloridx = fr->key;   /* past the block */
                else coloridx = row[x - fr->left];
                if (destructive) {
                    int offset = y * cw + x;
                    if (fr->dispose == 2) { if (coloridx == fr->key) coloridx = 0; else master[offset] = coloridx; }
                    else { if (coloridx == fr->key && f > 0) coloridx = master[offset]; else master[offset] = coloridx; }
                }
                unsigned char* d = canvases[f] + (size_t)y * cstep + (size_t)x * 4;
                static const unsigned char clr_important[4] = {0, 1, 0, 0};
                const unsigned char* q = (coloridx >= 0 && coloridx < 256) ? fr->palette + coloridx * 4 : clr_important;
                d[0] = q[0]; d[1] = q[1]; d[2] = q[2]; d[3] = coloridx == fr->key ? 0 : 255;
            }
        }
    }
    free(master);
}

/* ------------------------------------------------------------------------------------------ */
/* 2. OpenCV ops the reference calls (SURVEY Appendix A; pinned against cv2 4.13 IPP-off)        */
/* ------------------------------------------------------------------------------------------ */

/* bridge.c:130-135 cvSetImageROI + cvCopy. */
void orc_copy_roi(const orc_img* src, int x, int y, orc_img* dst) {
    for (int r = 0; r < dst->height; r++)
        memcpy(dst->data + (size_t)dst->step * r, src->data + (size_t)src->step * (y + r) + (size_t)x * src->channels,
               (size_t)dst->width * dst->channels);
}

/* filters.c:95-99,119,126 cvFlip: mode 0 = around x axis (rows reversed), >0 = around y axis, <0 = both. */
void orc_flip(const orc_img* src, orc_img* dst, int mode) {
    int w = src->width, h = src->height, c = src->channels;
    for (int y = 0; y < h; y++) for (int x = 0; x < w; x++) {
        int sx = (mode != 0) ? w - 1 - x : x;
        int sy = (mode <= 0) ? h - 1 - y : y;
        memcpy(&PX(dst, x, y, 0), &PX(src, sx, sy, 0), (size_t)c);
    }
}

/* filters.c:118 cvTranspose. dst is (h x w). */
void orc_transpose(const orc_img* src, orc_img* dst) {
    for (int y = 0; y < dst->height; y++) for (int x = 0; x < dst->width; x++)
        memcpy(&PX(dst, x, y, 0), &PX(src, y, x, 0), (size_t)src->channels);
}

/* bridge.c:613-618 cvCvtColor(CV_GRAY2BGR). */
void orc_gray2bgr(const orc_img* src, orc_img* dst) {
    for (int y = 0; y < src->height; y++) for (int x = 0; x < src->width; x++) {
        unsigned char v = PX(src, x, y, 0);
        PX(dst, x, y, 0) = v; PX(dst, x, y, 1) = v; PX(dst, x, y, 2) = v;
    }
}

/* App. A.1 INTER_NEAREST. */
static void resize_nn(const orc_img* s, orc_img* d) {
    double ifx = 1.0 / ((double)d->width / s->width), ify = 1.0 / ((double)d->height / s->height);
    for (int y = 0; y < d->height; y++) {
        int sy = (int)floor(y * ify); if (sy > s->height - 1) sy = s->height - 1;
        for (int x = 0; x < d->width; x++) {
            int sx = (int)floor(x * ifx); if (sx > s->width - 1) sx = s->width - 1;
            memcpy(&PX(d, x, y, 0), &PX(s, sx, sy, 0), (size_t)s->channels);
        }
    }
}

/* App. A.2 INTER_AREA with both scales integer. */
static void resize_area_int(const orc_img* s, orc_img* d, int nx, int ny) {
    int c = s->channels;
    float scale = 1.f / (nx * ny);
    for (int y = 0; y < d->height; y++) for (int x = 0; x < d->width; x++) for (int k = 0; k < c; k++) {
        int sum = 0;
        for (int j = 0; j < ny; j++) for (int i = 0; i < nx; i++) sum += PX(s, x * nx + i, y * ny + j, k);
        if (nx == 2 && ny == 2) PX(d, x, y, k) = (unsigned char)((sum + 2) >> 2);
        else PX(d, x, y, k) = sat_u8((int)lrintf((float)sum * scale));
    }
}

typedef struct { int si, di; float alpha; } area_tap;

/* App. A.3 tap table for one axis (OpenCV computeResizeAreaTab). Returns tap count. */
int orc_area_tab(int ssize, int dsize, double scale, area_tap* tab) {
    int k = 0;
    for (int dx = 0; dx < dsize; dx++) {
        double fsx1 = dx * scale, fsx2 = fsx1 + scale;
        double cell = fmin(scale, ssize - fsx1);
        int sx1 = (int)ceil(fsx1), sx2 = (int)floor(fsx2);
        if (sx2 > ssize - 1) sx2 = ssize - 1;
        if (sx1 > sx2) sx1 = sx2;
        if (sx1 - fsx1 > 1e-3) { tab[k].di = dx; tab[k].si = sx1 - 1; tab[k++].alpha = (float)((sx1 - fsx1) / cell); }
        for (int sx = sx1; sx < sx2; sx++) { tab[k].di = dx; tab[k].si = sx; tab[k++].alpha = (float)(1.0 / cell); }
        if (fsx2 - sx2 > 1e-3) { tab[k].di = dx; tab[k].si = sx2; tab[k++].alpha = (float)(fmin(fmin(fsx2 - sx2, 1.), cell) / cell); }
    }
    return k;
}

/* App. A.3 INTER_AREA, generic: ordered float32 accumulation, no FMA. */
static void resize_area_frac(const orc_img* s, orc_img* d, double scale_x, double scale_y) {
    int c = s->channels, dw = d->width, dh = d->height;
    area_tap* xt = (area_tap*)malloc(sizeof(area_tap) * ((size_t)s->width * 2 + 2 * dw + 4));
    area_tap* yt = (area_tap*)malloc(sizeof(area_tap) * ((size_t)s->height * 2 + 2 * dh + 4));
    int nx = orc_area_tab(s->width, dw, scale_x, xt), ny = orc_area_tab(s->height, dh, scale_y, yt);
    float* buf = (float*)malloc(sizeof(float) * dw * c);
    float* sum = (float*)malloc(sizeof(float) * dw * c);
    int prev_dy = -1;
    for (int j = 0; j < ny; j++) {
        float beta = yt[j].alpha; int dy = yt[j].di, sy = yt[j].si;
        for (int i = 0; i < dw * c; i++) buf[i] = 0;
        for (int k = 0; k < nx; k++) {
            float a = xt[k].alpha; int dxn = xt[k].di * c, sxn = xt[k].si * c;
            for (int ch = 0; ch < c; ch++) buf[dxn + ch] += (float)s->data[(size_t)s->step * sy + sxn + ch] * a;
        }
        if (dy != prev_dy) {
            if (prev_dy >= 0) for (int i = 0; i < dw * c; i++) d->data[(size_t)d->step * prev_dy + i] = sat_u8((int)lrintf(sum[i]));
            for (int i = 0; i < dw * c; i++) sum[i] = beta * buf[i];
            prev_dy = dy;
        } else {
            for (int i = 0; i < dw * c; i++) sum[i] += beta * buf[i];
        }
    }
    if (prev_dy >= 0) for (int i = 0; i < dw * c; i++) d->data[(size_t)d->step * prev_dy + i] = sat_u8((int)lrintf(sum[i]));
    free(xt); free(yt); free(buf); free(sum);
}

static short sat_i16_rint(float v) { long r = lrintf(v); return (short)(r < -32768 ? -32768 : (r > 32767 ? 32767 : r)); }

/* App. A.4 cubic coefficients (OpenCV interpolateCubic, A = -0.75), float32. */
static void cubic_coeffs(float x, float* co) {
    const float A = -0.75f;
    co[0] = ((A * (x + 1) - 5 * A) * (x + 1) + 8 * A) * (x + 1) - 4 * A;
    co[1] = ((A + 2) * x - (A + 3)) * x * x + 1;
    co[2] = ((A + 2) * (1 - x) - (A + 3)) * (1 - x) * (1 - x) + 1;
    co[3] = 1.f - co[0] - co[1] - co[2];
}

/* App. A.4: per-axis offsets and 11-bit integer coefficients. ksize 2 (linear) or 4 (cubic). */
void orc_interp_tab(int ssize, int dsize, double scale, int cubic, int is_x, int* ofs, short* coef) {
    int ksize = cubic ? 4 : 2;
    for (int d = 0; d < dsize; d++) {
        float f = (float)((d + 0.5) * scale - 0.5);
        int sidx = (int)floor((double)f);
        f -= (float)sidx;
        if (!cubic && is_x) {
            if (sidx < 0) { f = 0; sidx = 0; }
            if (sidx >= ssize - 1) { f = 0; sidx = ssize - 1; }
        }
        ofs[d] = sidx;
        float cb[4];
        if (cubic) cubic_coeffs(f, cb); else { cb[0] = 1.f - f; cb[1] = f; }
        for (int k = 0; k < ksize; k++) coef[d * ksize + k] = sat_i16_rint(cb[k] * 2048);
    }
}

/* App. A.4 INTER_LINEAR / INTER_CUBIC, 8-bit fixed point. */
static void resize_interp(const orc_img* s, orc_img* d, double scale_x, double scale_y, int cubic) {
    int c = s->channels, dw = d->width, dh = d->height, ks = cubic ? 4 : 2, k0 = cubic ? 1 : 0;
    int* xofs = (int*)malloc(sizeof(int) * dw); short* xa = (short*)malloc(sizeof(short) * dw * ks);
    int* yofs = (int*)malloc(sizeof(int) * dh); short* yb = (short*)malloc(sizeof(short) * dh * ks);
    orc_interp_tab(s->width, dw, scale_x, cubic, 1, xofs, xa);
    orc_interp_tab(s->height, dh, scale_y, cubic, 0, yofs, yb);
    int rowlen = dw * c;
    int simd_end = rowlen - (rowlen % 8);           /* 128-bit universal intrinsics: 8 x int16 per step */
    int* H = (int*)malloc(sizeof(int) * rowlen * ks);
    for (int dy = 0; dy < dh; dy++) {
        for (int k = 0; k < ks; k++) {
            int sy = clampi(yofs[dy] - k0 + k, 0, s->height - 1);
            const unsigned char* S = s->data + (size_t)s->step * sy;
            for (int dx = 0; dx < dw; dx++) for (int ch = 0; ch < c; ch++) {
                int v = 0;
                for (int t = 0; t < ks; t++) {
                    int sx = clampi(xofs[dx] - k0 + t, 0, s->width - 1);
                    v += S[sx * c + ch] * xa[dx * ks + t];
                }
                H[k * rowlen + dx * c + ch] = v;
            }
        }
        const short* b = yb + dy * ks;
        unsigned char* D = d->data + (size_t)d->step * dy;
        if (!cubic) {
            for (int i = 0; i < rowlen; i++)
                D[i] = (unsigned char)((((b[0] * (H[i] >> 4)) >> 16) + ((b[1] * (H[rowlen + i] >> 4)) >> 16) + 2) >> 2);
        } else {
            const float sc = 1.f / (2048.f * 2048.f);
            float b0 = b[0] * sc, b1 = b[1] * sc, b2 = b[2] * sc, b3 = b[3] * sc;
            for (int i = 0; i < rowlen; i++) {
                int h0 = H[i], h1 = H[rowlen + i], h2 = H[2 * rowlen + i], h3 = H[3 * rowlen + i];
                if (i < simd_end) {
                    float t3 = (float)h3 * b3;
                    float t2 = (float)h2 * b2 + t3;
                    float t1 = (float)h1 * b1 + t2;
                    float t0 = (float)h0 * b0 + t1;
                    D[i] = sat_u8((int)lrintf(t0));
                } else {
                    D[i] = sat_u8((h0 * b[0] + h1 * b[1] + h2 * b[2] + h3 * b[3] + (1 << 21)) >> 22);
                }
            }
        }
    }
    free(xofs); free(xa); free(yofs); free(yb); free(H);
}

/* bridge.c:191 cvResize. mode: 0 NN, 1 LINEAR, 2 CUBIC, 3 AREA (same values as CV_INTER_*). */
void orc_resize(const orc_img* s, orc_img* d, int mode) {
    if (d->width == s->width && d->height == s->height) { orc_copy_roi(s, 0, 0, d); return; }
    double scale_x = 1.0 / ((double)d->width / s->width), scale_y = 1.0 / ((double)d->height / s->height);
    if (mode == 0) { resize_nn(s, d); return; }
    int isx = (int)lrint(scale_x), isy = (int)lrint(scale_y);
    int fast = fabs(scale_x - isx) < DBL_EPSILON && fabs(scale_y - isy) < DBL_EPSILON;
    if (mode == 1 && fast && isx == 2 && isy == 2) mode = 3;
    if (mode == 3 && scale_x >= 1 && scale_y >= 1) {
        if (fast) resize_area_int(s, d, isx, isy); else resize_area_frac(s, d, scale_x, scale_y);
        return;
    }
    /* AREA with upscaling does not occur through bridge.c:190; LINEAR/CUBIC otherwise. */
    resize_interp(s, d, scale_x, scale_y, mode == 2);
}

/* App. A.5 Gaussian taps: n = rint(6*sigma+1)|1, 8-bit fixed point with error diffusion, sum == 256. */
int orc_gaussian_taps(double sigma, int* taps /* >= n */, int maxn) {
    int n = (int)lrint(sigma * 6 + 1) | 1;
    if (n > maxn) return -n;
    double* t = (double*)malloc(sizeof(double) * n);
    double scale2x = -0.5 / (sigma * sigma), sum = 0;
    for (int i = 0; i < n; i++) { double x = i - (n - 1) * 0.5; t[i] = exp(scale2x * x * x); sum += t[i]; }
    double inv = 1. / sum;
    double err = 0; int isum = 0;
    for (int i = 0; i < n / 2; i++) {
        double adj = t[i] * inv * 256 + err;
        int v = (int)lrint(adj);
        err = adj - v;
        taps[i] = taps[n - 1 - i] = v;
        isum += v;
    }
    taps[n / 2] = 256 - 2 * isum;
    free(t);
    return n;
}

/* filters.c:204 cvSmooth(CV_GAUSSIAN,0,0,sigma) == GaussianBlur(ksize 0, sigma, BORDER_REPLICATE), all channels. */
int orc_gaussian(const orc_img* s, orc_img* d, double sigma) {
    int w = s->width, h = s->height, c = s->channels;
    int n = (int)lrint(sigma * 6 + 1) | 1;
    int* k = (int*)malloc(sizeof(int) * n);
    orc_gaussian_taps(sigma, k, n);
    int r = n / 2;
    unsigned short* tmp = (unsigned short*)malloc(sizeof(unsigned short) * (size_t)w * h * c);
    for (int y = 0; y < h; y++) for (int x = 0; x < w; x++) for (int ch = 0; ch < c; ch++) {
        unsigned acc = 0;
        for (int i = 0; i < n; i++) acc += (unsigned)PX(s, clampi(x + i - r, 0, w - 1), y, ch) * k[i];
        tmp[((size_t)y * w + x) * c + ch] = (unsigned short)acc;
    }
    for (int y = 0; y < h; y++) for (int x = 0; x < w; x++) for (int ch = 0; ch < c; ch++) {
        unsigned acc = 0;
        for (int j = 0; j < n; j++) acc += (unsigned)tmp[((size_t)clampi(y + j - r, 0, h - 1) * w + x) * c + ch] * k[j];
        PX(d, x, y, ch) = (unsigned char)((acc + 32768u) >> 16);
    }
    free(tmp); free(k);
    return n;
}
