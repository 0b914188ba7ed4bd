// hostsim.cpp — TEST-ONLY. Walks a plan's passes on the CPU with the SAME headers the CUDA kernels
// compile (imp_pixel.cuh, imp_gather.cuh) and the SAME planner (imp_planner.cpp), so that the planner,
// the frame-map algebra and the per-pixel arithmetic can be checked against the oracle on a machine
// without a GPU (`pytest -m "not gpu"`). It is built into tests/hostsim/libimp_hostsim.so by
// tests/conftest.py, is never linked into libimp_gpu.so and is not a fallback: the product has none.
#include "../../ngx_http_imgproc_b200/csrc/imp_internal.h"
#include "../../ngx_http_imgproc_b200/csrc/imp_gather.cuh"
#include <vector>
#include <string.h>

template <int SC>
static void run_pass(const ImpHostPass& hp, const uint8_t* src, int sp, uint8_t* dst, int dp, const uint8_t* wm, int wm_pitch, int wm_c) {
    const uint8_t* blob = hp.blob.data();
    const ImpPass* P = (const ImpPass*)blob;
    ImpSrcGlobal<SC> S; S.base = src + (size_t)P->sy0 * sp + (size_t)P->sx0 * SC; S.pitch = sp;
    const ImpOp* ops = (const ImpOp*)(blob + P->ops_off);
    const uint8_t* lut = blob + P->lut_off;
    std::vector<uint16_t> tmp;
    const int* taps = (const int*)(blob + P->taps_off);
    if (P->kind == IMP_G_BLUR) {
        const int w = P->sw, h = P->sh, n = P->ksize, r = n / 2;
        tmp.resize((size_t)w * h * SC);
        for (int y = 0; y < h; y++) for (int x = 0; x < w; x++) for (int c = 0; c < SC; c++) {
            unsigned acc = 0;
            for (int i = 0; i < n; i++) acc += (unsigned)S.at(imp_min(imp_max(x + i - r, 0), w - 1), y, c) * (unsigned)taps[i];
            tmp[((size_t)y * w + x) * SC + c] = (uint16_t)acc;
        }
    }
    for (int by = 0; by < P->bh; by++) for (int bx = 0; bx < P->bw; bx++) {
        int v[4] = {0, 0, 0, 255};
        switch (P->kind) {
            case IMP_G_COPY: imp_gather_copy<SC>(S, bx, by, v); break;
            case IMP_G_NN: imp_gather_nn<SC>(S, (const int*)(blob + P->xofs_off), (const int*)(blob + P->yofs_off), bx, by, v); break;
            case IMP_G_AREA_INT: imp_gather_area_int<SC>(S, P->nx, P->ny, P->area_scale, bx, by, v); break;
            case IMP_G_AREA_FRAC: imp_gather_area_frac<SC>(S, (const ImpRange*)(blob + P->xofs_off), (const ImpAreaTap*)(blob + P->xcoef_off),
                                                           (const ImpRange*)(blob + P->yofs_off), (const ImpAreaTap*)(blob + P->ycoef_off), bx, by, v); break;
            case IMP_G_CUBIC: imp_gather_cubic<SC>(S, P->sw, P->sh, (const int*)(blob + P->xofs_off), (const short*)(blob + P->xcoef_off),
                                                   (const int*)(blob + P->yofs_off), (const short*)(blob + P->ycoef_off), P->simd_end, bx, by, v); break;
            case IMP_G_LINEAR: imp_gather_linear<SC>(S, P->sw, P->sh, (const int*)(blob + P->xofs_off), (const short*)(blob + P->xcoef_off),
                                                     (const int*)(blob + P->yofs_off), (const short*)(blob + P->ycoef_off), bx, by, v); break;
            case IMP_G_BLUR: {
                const int w = P->sw, h = P->sh, n = P->ksize, r = n / 2;
                for (int c = 0; c < SC; c++) {
                    unsigned acc = 0;
                    for (int j = 0; j < n; j++) acc += (unsigned)tmp[((size_t)imp_min(imp_max(by + j - r, 0), h - 1) * w + bx) * SC + c] * (unsigned)taps[j];
                    v[c] = (int)((acc + 32768u) >> 16);
                }
            } break;
        }
        ImpPx p;
        if (SC == 1) { p.b = p.g = p.r = v[0]; p.a = 255; } else { p.b = v[0]; p.g = v[1]; p.r = v[2]; p.a = SC == 4 ? v[3] : 255; }
        imp_run_ops(p, P->oc, bx, by, ops, P->nops, lut, wm, wm_pitch, wm_c);
        int X, Y; imp_map_xy(P->out, bx, by, X, Y);
        uint8_t* d = dst + (size_t)Y * dp + (size_t)X * P->dc;
        d[0] = (uint8_t)p.b; d[1] = (uint8_t)p.g; d[2] = (uint8_t)p.r; if (P->dc == 4) d[3] = (uint8_t)p.a;
    }
}

extern "C" {
int hostsim_plan_create(const imp_gpu_request* req, const imp_gpu_config* cfg, int w, int h, int c, imp_gpu_plan** out, int* step) {
    imp_gpu_plan* p = new imp_gpu_plan();
    int rc = imp_build_plan(req, cfg, w, h, c, p, step);
    if (rc) { delete p; *out = nullptr; return rc; }
    *out = p; return 0;
}
// validate-only mode of the planner (what the operator layer runs per recorded op): code, step and output geometry only
int hostsim_plan_validate(const imp_gpu_request* req, const imp_gpu_config* cfg, int w, int h, int c, int* step, int* out3) {
    imp_gpu_plan p;
    int rc = imp_build_plan(req, cfg, w, h, c, &p, step, true);
    if (!rc) { out3[0] = p.out_w; out3[1] = p.out_h; out3[2] = p.out_c; }
    return rc;
}
void hostsim_plan_destroy(imp_gpu_plan* p) { delete p; }
void hostsim_plan_output(const imp_gpu_plan* p, int* w, int* h, int* c) { *w = p->out_w; *h = p->out_h; *c = p->out_c; }
int hostsim_plan_passes(const imp_gpu_plan* p) { return (int)p->passes.size(); }
int hostsim_plan_pass_kind(const imp_gpu_plan* p, int k) { return p->passes[k].hdr.kind; }
unsigned long long hostsim_plan_bytes(const imp_gpu_plan* p) { return p->algo_bytes; }
int hostsim_run(const imp_gpu_plan* p, const uint8_t* src, int sp, uint8_t* dst, int dp) {
    std::vector<uint8_t> prev, cur;
    const uint8_t* in = src; int in_pitch = sp;
    const uint8_t* wm = p->wm ? p->wm->pixels.data() : nullptr;
    const int wm_w = p->wm ? p->wm->w : 0, wm_c = p->wm ? p->wm->c : 0;
    for (size_t k = 0; k < p->passes.size(); k++) {
        const ImpHostPass& hp = p->passes[k];
        uint8_t* out; int out_pitch;
        if (k + 1 == p->passes.size()) { out = dst; out_pitch = dp; }
        else { out_pitch = (hp.out_w * hp.out_c + 15) & ~15; cur.assign((size_t)out_pitch * hp.out_h, 0); out = cur.data(); }
        switch (hp.hdr.sc) {
            case 1: run_pass<1>(hp, in, in_pitch, out, out_pitch, wm, wm_w * wm_c, wm_c); break;
            case 3: run_pass<3>(hp, in, in_pitch, out, out_pitch, wm, wm_w * wm_c, wm_c); break;
            case 4: run_pass<4>(hp, in, in_pitch, out, out_pitch, wm, wm_w * wm_c, wm_c); break;
            default: return 1;
        }
        prev.swap(cur); in = prev.data(); in_pitch = out_pitch;
    }
    return 0;
}
}
extern "C" void hostsim_plan_tile_info(const imp_gpu_plan* p, int k, int* out) {
    const ImpPass& h = p->passes[k].hdr;
    out[0] = h.tile_rs; out[1] = h.tile_rows; out[2] = h.tile_smem; out[3] = h.max_xtaps; out[4] = h.max_ytaps; out[5] = h.kind;
}
// the launch a job of pass k takes (ImpHostPass::tiled when its source rows are 16-byte addressable, else ::fallback):
// kernel (ImpKernel), param, flavour, ctas_per_job, smem_bytes, ctas_per_sm
extern "C" void hostsim_plan_launch(const imp_gpu_plan* p, int k, int tiled, int* out) {
    const ImpLaunch& l = tiled ? p->passes[k].tiled : p->passes[k].fallback;
    out[0] = (int)l.kernel; out[1] = l.param; out[2] = l.flavour; out[3] = l.ctas_per_job; out[4] = l.smem_bytes; out[5] = l.ctas_per_sm;
}
// What decides the device code a job of pass k runs (the `tiled` launch when its source rows are 16-byte addressable, else
// `fallback`): kind, sc, dc, kernel (ImpKernel), flavour, param, max_xtaps, nx, ny, gt, blur_r, the blur's effective tap
// radius (zero outer taps trimmed, as the planner does before it pads to blur_r), tile_rs, tile_rows, tile_smem, smem_bytes.
extern "C" void hostsim_plan_branch(const imp_gpu_plan* p, int k, int tiled, int* out) {
    const ImpHostPass& hp = p->passes[k];
    const ImpPass& h = hp.hdr;
    const ImpLaunch& l = tiled ? hp.tiled : hp.fallback;
    int r_eff = 0;
    if (h.kind == IMP_G_BLUR) {
        const int* t = (const int*)(hp.blob.data() + h.taps_off);
        int lo = 0, hi = h.ksize - 1;
        while (lo < hi && t[lo] == 0 && t[hi] == 0) { lo++; hi--; }
        r_eff = (hi - lo) / 2;
    }
    const int v[16] = {h.kind, h.sc, h.dc, (int)l.kernel, l.flavour, l.param, h.max_xtaps, h.nx, h.ny, h.gt, h.blur_r, r_eff,
                       h.tile_rs, h.tile_rows, h.tile_smem, l.smem_bytes};
    memcpy(out, v, sizeof v);
}
// Per vignette op of the plan, in pass and op order, 8 ints: cx, cy, the op's frame w, h, the table's nx, ny as the
// planner sized it (0, 0: no table, each pixel evaluates imp_vignette_mask), the frame map's swap and flip flags packed
// as swap | flipx << 1 | flipy << 2, and 0; and 2 floats: maxr, intensity. Returns the number of ops (at most cap are written).
extern "C" int hostsim_vignette_ops(const imp_gpu_plan* p, int* iout, float* fout, int cap) {
    int n = 0;
    for (const ImpHostPass& hp : p->passes) {
        const ImpOp* ops = (const ImpOp*)(hp.blob.data() + hp.hdr.ops_off);
        for (int k = 0; k < hp.hdr.nops; k++) {
            const ImpOp& o = ops[k];
            if (o.kind != IMP_OP_VIGNETTE) continue;
            if (n < cap) {
                const int v[8] = {o.i[0], o.i[1], o.map.w, o.map.h, o.i[2], o.i[3], o.map.swap | o.map.flipx << 1 | o.map.flipy << 2, 0};
                memcpy(iout + 8 * n, v, sizeof v);
                fout[2 * n] = o.f[0]; fout[2 * n + 1] = o.f[1];
            }
            n++;
        }
    }
    return n;
}
// out[j * nx + i] = the CPU build of imp_vignette_mask at |dx| = i, |dy| = j (the code the device table kernel and the
// per-pixel path compile).
extern "C" void hostsim_vignette_mask_table(float* out, int nx, int ny, float maxr, float intensity) {
    for (int j = 0; j < ny; j++)
        for (int i = 0; i < nx; i++) out[(size_t)j * nx + i] = imp_vignette_mask(0, 0, i, j, maxr, intensity);
}
