// area_exact_shim.cpp — a C face over the planner's exact integer INTER_AREA taps (imp_planner.cpp, area_exact) for
// tests/test_area_exact_int.py. Built together with hostsim.cpp (plan creation) and imp_planner.cpp; no device involved.
#include "../../ngx_http_imgproc_b200/csrc/imp_internal.h"
#include "../../ngx_http_imgproc_b200/csrc/imp_gather.cuh"
#include <string.h>

extern "C" {

// Pass k's header: kind, sc, sw, sh, bw, bh, max_xtaps, max_ytaps, area_d, area_bias, area_magic, x taps, y taps
void shim_area_info(const imp_gpu_plan* p, int k, long long* out) {
    const ImpHostPass& hp = p->passes[k];
    const ImpPass& h = hp.hdr;
    long long nxt = 0, nyt = 0;
    if (h.kind == IMP_G_AREA_FRAC || h.kind == IMP_G_AREA_INT) {
        const ImpRange* xr = (const ImpRange*)(hp.blob.data() + h.xofs_off);
        const ImpRange* yr = (const ImpRange*)(hp.blob.data() + h.yofs_off);
        nxt = xr[h.bw - 1].first + xr[h.bw - 1].count;
        nyt = yr[h.bh - 1].first + yr[h.bh - 1].count;
    }
    const long long v[13] = {h.kind, h.sc, h.sw, h.sh, h.bw, h.bh, h.max_xtaps, h.max_ytaps, h.area_d, h.area_bias, (long long)h.area_magic, nxt, nyt};
    memcpy(out, v, sizeof v);
}

// The tap ranges and the integer weights of an exact pass: xr[2 bw], yr[2 bh] as {first tap, count}; xk[2 nx], yk[2 ny] as
// {source index, k}. Returns 0, or 1 when the pass has no integer tables.
int shim_area_tables(const imp_gpu_plan* p, int k, int* xr, int* yr, int* xk, int* yk, int nxk, int nyk) {
    const ImpHostPass& hp = p->passes[k];
    const ImpPass& h = hp.hdr;
    if (!h.area_d || !h.ixcoef_off || !h.iycoef_off) return 1;
    const uint8_t* b = hp.blob.data();
    memcpy(xr, b + h.xofs_off, (size_t)h.bw * sizeof(ImpRange));
    memcpy(yr, b + h.yofs_off, (size_t)h.bh * sizeof(ImpRange));
    memcpy(xk, b + h.ixcoef_off, (size_t)nxk * sizeof(ImpAreaKTap));
    memcpy(yk, b + h.iycoef_off, (size_t)nyk * sizeof(ImpAreaKTap));
    return 0;
}

// The float gather of pass k (imp_gather_area_frac, the code the direct kernel compiles) for every base pixel, before any
// op: out[(by * bw + bx) * sc + c]. src: the pass's input image, rows of sp bytes.
int shim_area_float(const imp_gpu_plan* p, int k, const uint8_t* src, int sp, uint8_t* out) {
    const ImpHostPass& hp = p->passes[k];
    const ImpPass* P = &hp.hdr;
    const uint8_t* blob = hp.blob.data();
    if (P->kind != IMP_G_AREA_FRAC) return 1;
    const ImpRange* xr = (const ImpRange*)(blob + P->xofs_off);
    const ImpRange* yr = (const ImpRange*)(blob + P->yofs_off);
    const ImpAreaTap* xt = (const ImpAreaTap*)(blob + P->xcoef_off);
    const ImpAreaTap* yt = (const ImpAreaTap*)(blob + P->ycoef_off);
    for (int by = 0; by < P->bh; by++)
        for (int bx = 0; bx < P->bw; bx++) {
            int v[4] = {0, 0, 0, 0};
            uint8_t* d = out + ((size_t)by * P->bw + bx) * P->sc;
            switch (P->sc) {
                case 1: { ImpSrcGlobal<1> S; S.base = src + (size_t)P->sy0 * sp + (size_t)P->sx0; S.pitch = sp; imp_gather_area_frac<1>(S, xr, xt, yr, yt, bx, by, v); } break;
                case 3: { ImpSrcGlobal<3> S; S.base = src + (size_t)P->sy0 * sp + (size_t)P->sx0 * 3; S.pitch = sp; imp_gather_area_frac<3>(S, xr, xt, yr, yt, bx, by, v); } break;
                case 4: { ImpSrcGlobal<4> S; S.base = src + (size_t)P->sy0 * sp + (size_t)P->sx0 * 4; S.pitch = sp; imp_gather_area_frac<4>(S, xr, xt, yr, yt, bx, by, v); } break;
                default: return 1;
            }
            for (int c = 0; c < P->sc; c++) d[c] = (uint8_t)v[c];
        }
    return 0;
}

}  // extern "C"
