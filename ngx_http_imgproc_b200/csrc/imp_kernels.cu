// imp_kernels.cu — sm_100a kernels of the decoded-pixel path and their launchers.
//
// Round-1 layout: one thread per base-frame pixel, 32x8 pixel tiles, one CTA per (tile, job).
// Each CTA stages its pass's op list + LUTs in shared memory once; the gather reads the source through
// the read-only path, the op list runs in registers, and the store applies the accumulated
// flip/rotate map. A whole batch (GIF frames, concurrent requests) is one launch per kernel variant:
// grid = (tiles, jobs). See DESIGN.md §Kernels for the roofline of each variant.
#include "imp_internal.h"
#include <algorithm>
#include "imp_gather.cuh"

#include <atomic>
static std::atomic<unsigned long long> g_imp_launches{0};
unsigned long long imp_launches() { return g_imp_launches.load(); }
void imp_count_launches(int n) { g_imp_launches += (unsigned long long)n; }

// every kernel translation unit has its own copy of the per-byte division tables (imp_pixel.cuh)
cudaError_t imp_upload_tables() {
    cudaError_t e = imp_upload_tables_tu();
    if (e == cudaSuccess) e = imp_upload_tables_strip();
    if (e == cudaSuccess) e = imp_upload_tables_blur();
    if (e == cudaSuccess) e = imp_upload_tables_cubic();
    if (e == cudaSuccess) e = imp_upload_tables_gather();
    return e;
}

// mask[j][i] for |dx| = i < nx, |dy| = j < ny: the per-pixel code of imp_vignette_mask, which sees the pixel only through
// sqrt(dx*dx + dy*dy).
__global__ void imp_vignette_table_kernel(float* __restrict__ tab, int nx, int ny, float maxr, float intensity) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
    if (i >= nx || j >= ny) return;
    const float distance = (float)sqrt((double)i * (double)i + (double)j * (double)j);
    const float raw = __fmul_rn(__fdiv_rn(distance, maxr), intensity);
    const double c = cos((double)raw);
    const double c2 = c * c;
    tab[(size_t)j * nx + i] = (float)(c2 * c2);
}

cudaError_t imp_build_vignette_table(float* d_tab, int nx, int ny, float maxr, float intensity, cudaStream_t st) {
    imp_vignette_table_kernel<<<dim3((nx + 255) / 256, ny), 256, 0, st>>>(d_tab, nx, ny, maxr, intensity);
    g_imp_launches++;
    return cudaGetLastError();
}

// CalcPerceivedBrightness (filters.c:707-729): sum over pixels of sqrt(r*r*0.241 + g*g*0.691 + b*b*0.068) (or of the gray
// value), as a device reduction so that `format=json` (Info, bridge.c:283-300) needs 8 bytes back instead of the frame.
// The reference's running float32 sum in column-major order is not reproducible in parallel; this sums in double and the
// caller divides by w*h*255. Parity is stated on the JSON integer round(brightness*100) (tests/test_gpu_parity.py).
__global__ void __launch_bounds__(256) imp_brightness_kernel(const uint8_t* __restrict__ img, int pitch, int w, int h, int c, double* __restrict__ acc) {
    double s = 0.0;
    for (int y = blockIdx.y; y < h; y += gridDim.y) {
        const uint8_t* row = img + (size_t)y * pitch;
        for (int x = blockIdx.x * blockDim.x + threadIdx.x; x < w; x += gridDim.x * blockDim.x) {
            if (c == 1) s += (double)row[x];
            else {
                const uint8_t* p = row + (size_t)x * c;
                const int b = p[0], g = p[1], r = p[2];
                s += sqrt(r * r * 0.241 + g * g * 0.691 + b * b * 0.068);
            }
        }
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    __shared__ double ws[8];
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < 8; i++) t += ws[i];
        atomicAdd(acc, t);
    }
}

cudaError_t imp_launch_brightness(const uint8_t* d_img, int pitch, int w, int h, int c, double* d_acc, cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(d_acc, 0, sizeof(double), st);
    if (e != cudaSuccess) return e;
    dim3 grid((w + 255) / 256 > 8 ? 8 : (w + 255) / 256, h < 1184 ? h : 1184);
    imp_brightness_kernel<<<grid, 256, 0, st>>>(d_img, pitch, w, h, c, d_acc);
    g_imp_launches++;
    return cudaGetLastError();
}

// ASCII (filters.c:486-522, `format=text`): one character per pixel from the HSV value V = max(B,G,R) through a 256-entry
// table the host derives with the reference's float maths; rows are separated by '\n' (no trailing newline).
__global__ void __launch_bounds__(256) imp_ascii_kernel(const uint8_t* __restrict__ img, int pitch, int w, int h, int c,
                                                        const uint8_t* __restrict__ lut, uint8_t* __restrict__ out) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x > w || y >= h) return;
    uint8_t* o = out + (size_t)y * (w + 1) + x;
    if (x == w) { if (y + 1 < h) *o = '\n'; return; }
    const uint8_t* p = img + (size_t)y * pitch + (size_t)x * c;
    const int v = c == 1 ? p[0] : max(p[0], max(p[1], p[2]));
    *o = __ldg(lut + v);
}

cudaError_t imp_launch_ascii(const uint8_t* d_img, int pitch, int w, int h, int c, const uint8_t* d_lut, uint8_t* d_out, cudaStream_t st) {
    dim3 grid((w + 1 + 255) / 256, h);
    imp_ascii_kernel<<<grid, 256, 0, st>>>(d_img, pitch, w, h, c, d_lut, d_out);
    g_imp_launches++;
    return cudaGetLastError();
}

// Window extraction / re-pitching on the device for the end-to-end path: the host frame's rows travel as ONE linear copy
// (a 2-D host-to-device copy costs ~0.15 us per row, i.e. only 23 GB/s for 3.5 KB rows) and this kernel then lays the crop
// window out with the 16-byte-aligned pitch the TMA kernels need. One thread per 4 destination bytes.
__global__ void __launch_bounds__(256) imp_repitch_kernel(const uint8_t* __restrict__ src, int sp, uint8_t* __restrict__ dst, int dp,
                                                          int row_bytes, int rows) {
    const int words = (row_bytes + 3) >> 2;
    const long long total = (long long)words * rows;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(i / words), xw = (int)(i - (long long)y * words);
        const uint8_t* s = src + (size_t)y * sp + (size_t)xw * 4;
        const int n = min(4, row_bytes - xw * 4);
        uint32_t w = 0;
        if ((reinterpret_cast<uintptr_t>(s) & 3) == 0 && n == 4) w = __ldg(reinterpret_cast<const uint32_t*>(s));
        else for (int b = 0; b < n; b++) w |= (uint32_t)__ldg(s + b) << (8 * b);
        *reinterpret_cast<uint32_t*>(dst + (size_t)y * dp + (size_t)xw * 4) = w;       // the pad bytes of the last word are inside the pitch
    }
}

cudaError_t imp_launch_repitch(const uint8_t* d_src, int sp, uint8_t* d_dst, int dp, int row_bytes, int rows, cudaStream_t st) {
    const long long total = (long long)((row_bytes + 3) >> 2) * rows;
    const int blocks = (int)std::min<long long>((total + 255) / 256, 148 * 16);
    imp_repitch_kernel<<<std::max(blocks, 1), 256, 0, st>>>(d_src, sp, d_dst, dp, row_bytes, rows);
    return cudaGetLastError();                 // a copy, not a pixel stage: not counted by imp_gpu_launch_count()
}

// GIF canvas expansion (SURVEY 8f-2; advancedio.c:195-248): every canvas pixel walks the frames in order, carrying the
// reference's `master` index for the disposal replay in a register, and writes one BGRA pixel per frame. Frames travel
// over PCIe as 8-bit indices (4x fewer bytes than the BGRA canvases the CPU path builds).
__global__ void __launch_bounds__(256) imp_gif_expand_kernel(const ImpGifFrame* __restrict__ frames, int n, int cw, int ch, int destructive,
                                                             uint8_t* __restrict__ canvases, int cpitch) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= cw || y >= ch) return;
    int master = 0;
    for (int f = 0; f < n; f++) {
        const ImpGifFrame fr = frames[f];
        const int rowidx = fr.h + fr.top - y - 1;
        int idx;
        // advancedio.c:203 tests `x > left + w`, so the column right of the frame reads row[w]: a pad byte of the
        // scanline or the first index of the next one. Reproduced while that byte is inside the page's pixel block.
        const int col = x - fr.left;
        if (rowidx < 0 || rowidx >= fr.h || col < 0 || col > fr.w || rowidx * fr.pitch + col >= fr.h * fr.pitch) idx = fr.key;
        else idx = __ldg(fr.indices + (size_t)rowidx * fr.pitch + col);
        if (destructive) {
            if (fr.dispose == 2) {                       // GIF_DISPOSAL_BACKGROUND
                if (idx == fr.key) idx = 0; else master = idx;
            } else {                                     // LEAVE / PREVIOUS / UNSPECIFIED
                if (idx == fr.key && f > 0) idx = master; else master = idx;
            }
        }
        // idx is 0..255 or -1 (a page without a transparent colour). palette[-1] aliases FreeImage's biClrImportant == 256,
        // i.e. the bytes {0,1,0,0} (advancedio.c:232 with FreeImage_GetTransparentIndex == -1).
        uchar4 q = make_uchar4(0, 1, 0, 0);
        if (idx >= 0 && idx < 256) q = __ldg(reinterpret_cast<const uchar4*>(fr.palette) + idx);
        const uchar4 px = make_uchar4(q.x, q.y, q.z, idx == fr.key ? 0 : 255);
        *reinterpret_cast<uchar4*>(canvases + ((size_t)f * ch + y) * cpitch + (size_t)x * 4) = px;
    }
}

cudaError_t imp_launch_gif_expand(const ImpGifFrame* d_frames, int n, int cw, int ch, int destructive, uint8_t* d_canvases, int cpitch, cudaStream_t st) {
    dim3 grid((cw + 255) / 256, ch);
    imp_gif_expand_kernel<<<grid, 256, 0, st>>>(d_frames, n, cw, ch, destructive, d_canvases, cpitch);
    g_imp_launches++;
    return cudaGetLastError();
}

namespace {

constexpr int TILE_W = 32, TILE_H = 8;

struct OpsSmem {
    const ImpOp* ops; const uint8_t* lut;
};

// Copies ops[] + LUT area (contiguous in the blob, 16-byte aligned) into shared memory.
__device__ __forceinline__ OpsSmem stage_ops(const ImpPass* P, const uint8_t* blob, uint8_t* smem) {
    const int bytes = P->nops * (int)sizeof(ImpOp) + P->lut_bytes;
    const uint4* g = reinterpret_cast<const uint4*>(blob + P->ops_off);
    uint4* s = reinterpret_cast<uint4*>(smem);
    const int tid = threadIdx.y * blockDim.x + threadIdx.x, nt = blockDim.x * blockDim.y;
    for (int i = tid; i < (bytes + 15) / 16; i += nt) s[i] = __ldg(g + i);
    __syncthreads();
    OpsSmem o;
    o.ops = reinterpret_cast<const ImpOp*>(smem);
    o.lut = smem + P->nops * sizeof(ImpOp);
    return o;
}

template <int DC>
__device__ __forceinline__ void store_px(const ImpJob& job, const ImpPass* P, int bx, int by, const ImpPx& p) {
    int X, Y;
    imp_map_xy(P->out, bx, by, X, Y);
    uint8_t* d = job.dst + (size_t)Y * job.dst_pitch + (size_t)X * DC;
    if (DC == 4) {
        *reinterpret_cast<uchar4*>(d) = make_uchar4((unsigned char)p.b, (unsigned char)p.g, (unsigned char)p.r, (unsigned char)p.a);
    } else {
        d[0] = (unsigned char)p.b; d[1] = (unsigned char)p.g; d[2] = (unsigned char)p.r;
    }
}

template <int SC>
__device__ __forceinline__ void promote(const int* v, ImpPx& p) {
    if (SC == 1) { p.b = p.g = p.r = v[0]; p.a = 255; }
    else { p.b = v[0]; p.g = v[1]; p.r = v[2]; p.a = (SC == 4) ? v[3] : 255; }
}

// The general pass kernel: one thread owns PASS_PPT output pixels of a column (rows TILE_H apart inside a
// 32 x 32 tile). The job and pass headers are staged in shared memory together with the ops, so the per-thread
// set-up (about 130 instructions when it was paid per pixel) and every op's parameter fetch + dispatch are
// shared by PASS_PPT pixels, and the PASS_PPT gathers are independent loads in flight together.
constexpr int PASS_PPT = 4;

struct PassHdrSmem {
    ImpPass P;
    const uint8_t* src; uint8_t* dst; const uint8_t* wm;
    int src_pitch, dst_pitch, wm_pitch, wm_c;
};

template <int KIND, int SC>
__global__ void __launch_bounds__(TILE_W * TILE_H, 6)
imp_pass_kernel(const ImpJob* __restrict__ jobs, int first, int count, const ImpJob one) {
    extern __shared__ __align__(16) uint8_t smem[];
    __shared__ __align__(16) PassHdrSmem H;
    const int j = blockIdx.y + blockIdx.z * 65535;
    if (j >= count) return;
    const int tid = threadIdx.y * TILE_W + threadIdx.x;
    const ImpJob* jp = jobs ? jobs + first + j : nullptr;
    const uint8_t* blob = jp ? jp->pass : one.pass;
    {
        static_assert(sizeof(ImpPass) % 4 == 0, "ImpPass is copied by words");
        const int* g = reinterpret_cast<const int*>(blob);
        int* sP = reinterpret_cast<int*>(&H.P);
        if (tid < (int)(sizeof(ImpPass) / 4)) sP[tid] = __ldg(g + tid);
        if (tid == 64) {
            H.src = jp ? jp->src : one.src; H.dst = jp ? jp->dst : one.dst; H.wm = jp ? jp->wm : one.wm;
            H.src_pitch = jp ? jp->src_pitch : one.src_pitch; H.dst_pitch = jp ? jp->dst_pitch : one.dst_pitch;
            H.wm_pitch = jp ? jp->wm_pitch : one.wm_pitch; H.wm_c = jp ? jp->wm_c : one.wm_c;
        }
        const ImpPass* gP = reinterpret_cast<const ImpPass*>(blob);
        const int bytes = __ldg(&gP->nops) * (int)sizeof(ImpOp) + __ldg(&gP->lut_bytes);
        const uint4* go = reinterpret_cast<const uint4*>(blob + __ldg(&gP->ops_off));
        uint4* so = reinterpret_cast<uint4*>(smem);
        for (int i = tid; i < (bytes + 15) / 16; i += TILE_W * TILE_H) so[i] = __ldg(go + i);
    }
    __syncthreads();
    const ImpPass& P = H.P;
    const int bw = P.bw, bh = P.bh;
    const int tiles_x = (bw + TILE_W - 1) / TILE_W, tiles_y = (bh + TILE_H * PASS_PPT - 1) / (TILE_H * PASS_PPT);
    if ((int)blockIdx.x >= tiles_x * tiles_y) return;
    const int x = (blockIdx.x % tiles_x) * TILE_W + threadIdx.x;
    const int y0 = (blockIdx.x / tiles_x) * (TILE_H * PASS_PPT) + threadIdx.y;
    if (x >= bw || y0 >= bh) return;
    const int nops = P.nops;
    const ImpOp* ops = reinterpret_cast<const ImpOp*>(smem);
    const uint8_t* lut = smem + nops * sizeof(ImpOp);

    ImpSrcGlobal<SC> S;
    S.pitch = H.src_pitch;
    S.base = H.src + (size_t)P.sy0 * S.pitch + (size_t)P.sx0 * SC;
    // rows past the bottom edge repeat the last row (computed, never stored)
    int bx[PASS_PPT], by[PASS_PPT];
#pragma unroll
    for (int n = 0; n < PASS_PPT; n++) { bx[n] = x; by[n] = min(y0 + n * TILE_H, bh - 1); }
    ImpPx px[PASS_PPT];
#pragma unroll
    for (int n = 0; n < PASS_PPT; n++) {
        int v[4] = {0, 0, 0, 255};
        if (KIND == IMP_G_COPY) {
            imp_gather_copy<SC>(S, x, by[n], v);
        } else if (KIND == IMP_G_NN) {
            imp_gather_nn<SC>(S, reinterpret_cast<const int*>(blob + P.xofs_off), reinterpret_cast<const int*>(blob + P.yofs_off), x, by[n], v);
        } else if (KIND == IMP_G_AREA_INT) {
            imp_gather_area_int<SC>(S, P.nx, P.ny, P.area_scale, x, by[n], v);
        } else if (KIND == IMP_G_AREA_FRAC) {
            imp_gather_area_frac<SC>(S, reinterpret_cast<const ImpRange*>(blob + P.xofs_off), reinterpret_cast<const ImpAreaTap*>(blob + P.xcoef_off),
                                     reinterpret_cast<const ImpRange*>(blob + P.yofs_off), reinterpret_cast<const ImpAreaTap*>(blob + P.ycoef_off), x, by[n], v);
        } else if (KIND == IMP_G_CUBIC) {
            imp_gather_cubic<SC>(S, P.sw, P.sh, reinterpret_cast<const int*>(blob + P.xofs_off), reinterpret_cast<const short*>(blob + P.xcoef_off),
                                 reinterpret_cast<const int*>(blob + P.yofs_off), reinterpret_cast<const short*>(blob + P.ycoef_off), P.simd_end, x, by[n], v);
        } else if (KIND == IMP_G_LINEAR) {
            imp_gather_linear<SC>(S, P.sw, P.sh, reinterpret_cast<const int*>(blob + P.xofs_off), reinterpret_cast<const short*>(blob + P.xcoef_off),
                                  reinterpret_cast<const int*>(blob + P.yofs_off), reinterpret_cast<const short*>(blob + P.ycoef_off), x, by[n], v);
        }
        promote<SC>(v, px[n]);
    }
    if (nops) imp_run_ops_n<PASS_PPT>(px, P.oc, bx, by, ops, nops, lut, H.wm, H.wm_pitch, H.wm_c);
    const ImpFrameMap out = P.out;
    const int dc = P.dc, dpitch = H.dst_pitch;
    uint8_t* dst = H.dst;
#pragma unroll
    for (int n = 0; n < PASS_PPT; n++) {
        if (y0 + n * TILE_H >= bh) break;
        int X, Y;
        imp_map_xy(out, x, by[n], X, Y);
        uint8_t* d = dst + (size_t)Y * dpitch + (size_t)X * dc;
        const ImpPx& p = px[n];
        if (dc == 4) {
            *reinterpret_cast<uchar4*>(d) = make_uchar4((unsigned char)p.b, (unsigned char)p.g, (unsigned char)p.r, (unsigned char)p.a);
        } else {
            d[0] = (unsigned char)p.b; d[1] = (unsigned char)p.g; d[2] = (unsigned char)p.r;
        }
    }
}

// ---- INTER_CUBIC with the horizontal pass shared down a column run ------------------------------------------------
// A thread produces CUBIC_RUN vertically adjacent output pixels of one column. OpenCV's H[row][dx] (int32, SURVEY
// App. A.4) depends only on the source row and the output column, so a sliding window of four H rows is carried
// down the run: at 2x upscale that is ~1.4 horizontal rows per output instead of 4. The window is held as floats
// (the conversion is exact, |H| < 2^22) because the vertical pass of every byte below simd_end is OpenCV's float
// form; the last <8 bytes of a row take the integer form through the generic per-pixel gather.
constexpr int CUBIC_RUN = IMP_CUBIC_RUN;      // imp_internal.h (the host sizes the grid with it)

template <int SC>
__device__ __forceinline__ void cubic_hrow(const ImpSrcGlobal<SC>& S, const int (&sx)[4], int sy, int a0, int a1, int a2, int a3, float (&hf)[SC]) {
    int p0[SC], p1[SC], p2[SC], p3[SC];
    S.px(sx[0], sy, p0); S.px(sx[1], sy, p1); S.px(sx[2], sy, p2); S.px(sx[3], sy, p3);
#pragma unroll
    for (int c = 0; c < SC; c++) hf[c] = imp_i2f22(p0[c] * a0 + p1[c] * a1 + p2[c] * a2 + p3[c] * a3);
}

template <int SC>
__global__ void __launch_bounds__(TILE_W * TILE_H, 4)
imp_cubic_run_kernel(const ImpJob* __restrict__ jobs, int first, int count, const ImpJob one) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int jn = blockIdx.y + blockIdx.z * 65535;
    if (jn >= count) return;
    const ImpJob job = jobs ? jobs[first + jn] : one;
    const uint8_t* blob = job.pass;
    const ImpPass* __restrict__ P = reinterpret_cast<const ImpPass*>(blob);
    const int bw = P->bw, bh = P->bh;
    const int tiles_x = (bw + TILE_W - 1) / TILE_W, tiles_y = (bh + TILE_H * CUBIC_RUN - 1) / (TILE_H * CUBIC_RUN);
    if ((int)blockIdx.x >= tiles_x * tiles_y) return;
    OpsSmem os = stage_ops(P, blob, smem);
    const int bx = (blockIdx.x % tiles_x) * TILE_W + threadIdx.x;
    const int by0 = ((blockIdx.x / tiles_x) * TILE_H + threadIdx.y) * CUBIC_RUN;
    if (bx >= bw || by0 >= bh) return;
    ImpSrcGlobal<SC> S;
    S.base = job.src + (size_t)P->sy0 * job.src_pitch + (size_t)P->sx0 * SC;
    S.pitch = job.src_pitch;
    const int sw = P->sw, sh = P->sh, oc = P->oc, dc = P->dc, nops = P->nops, simd_end = P->simd_end;
    const int* __restrict__ xofs = reinterpret_cast<const int*>(blob + P->xofs_off);
    const short* __restrict__ xa = reinterpret_cast<const short*>(blob + P->xcoef_off);
    const int* __restrict__ yofs = reinterpret_cast<const int*>(blob + P->yofs_off);
    const short* __restrict__ yb = reinterpret_cast<const short*>(blob + P->ycoef_off);
    const float* __restrict__ ybf = reinterpret_cast<const float*>(blob + P->taps_off);
    const bool fast = bx * SC + SC <= simd_end;                        // every byte of this pixel is on the float path
    int sx[4];
    const int x0 = __ldg(xofs + bx) - 1;
#pragma unroll
    for (int t = 0; t < 4; t++) sx[t] = min(max(x0 + t, 0), sw - 1);
    const int2 av = __ldg(reinterpret_cast<const int2*>(xa + bx * 4));   // 4 shorts, 8-byte aligned
    const int a0 = (short)(av.x & 0xffff), a1 = av.x >> 16, a2 = (short)(av.y & 0xffff), a3 = av.y >> 16;
    // Code size matters here (ncu: the first fully unrolled version was 14.6 K instructions and its top stall reason was
    // instruction fetch): the four-row window is loaded once before the run, the run only slides it, the rare non-SIMD
    // tail pixels take a rolled loop of their own, and the op list is instantiated once for both groups of four.
    unsigned q[CUBIC_RUN];                      // gathered pixels, packed B|G<<8|R<<16|A<<24 while the H window is live
    if (fast) {
        float h0[SC], h1[SC], h2[SC], h3[SC];
        int top = __ldg(yofs + by0) - 1;
        cubic_hrow<SC>(S, sx, min(max(top, 0), sh - 1), a0, a1, a2, a3, h0);
        cubic_hrow<SC>(S, sx, min(max(top + 1, 0), sh - 1), a0, a1, a2, a3, h1);
        cubic_hrow<SC>(S, sx, min(max(top + 2, 0), sh - 1), a0, a1, a2, a3, h2);
        cubic_hrow<SC>(S, sx, min(max(top + 3, 0), sh - 1), a0, a1, a2, a3, h3);
#pragma unroll
        for (int o = 0; o < CUBIC_RUN; o++) {
            const int by = min(by0 + o, bh - 1);                       // past the bottom edge: the last row again, never stored
            const int want = __ldg(yofs + by) - 1;                     // non-decreasing in by
            while (top < want) {
#pragma unroll
                for (int c = 0; c < SC; c++) { h0[c] = h1[c]; h1[c] = h2[c]; h2[c] = h3[c]; }
                top++;
                cubic_hrow<SC>(S, sx, min(max(top + 3, 0), sh - 1), a0, a1, a2, a3, h3);
            }
            const float4 fv = __ldg(reinterpret_cast<const float4*>(ybf) + by);          // coefficient * 2^-22, tabulated by the planner
            int v[4] = {0, 0, 0, 255};
#pragma unroll
            for (int c = 0; c < SC; c++) {
                const float t3 = __fmul_rn(h3[c], fv.w);
                const float t2 = __fadd_rn(__fmul_rn(h2[c], fv.z), t3);
                const float t1 = __fadd_rn(__fmul_rn(h1[c], fv.y), t2);
                const float t0 = __fadd_rn(__fmul_rn(h0[c], fv.x), t1);
                v[c] = imp_sat8(imp_rint22(t0));
            }
            ImpPx p;
            promote<SC>(v, p);
            q[o] = (unsigned)p.b | ((unsigned)p.g << 8) | ((unsigned)p.r << 16) | ((unsigned)p.a << 24);
        }
    } else {
#pragma unroll 1
        for (int o = 0; o < CUBIC_RUN; o++) {
            int v[4] = {0, 0, 0, 255};
            imp_gather_cubic<SC>(S, sw, sh, xofs, xa, yofs, yb, simd_end, bx, min(by0 + o, bh - 1), v);
            ImpPx p;
            promote<SC>(v, p);
            const unsigned w = (unsigned)p.b | ((unsigned)p.g << 8) | ((unsigned)p.r << 16) | ((unsigned)p.a << 24);
#pragma unroll
            for (int k = 0; k < CUBIC_RUN; k++) if (k == o) q[k] = w;          // register select, no local-memory array
        }
    }
    // op list + store, four pixels at a time (the op loop is the outer loop inside imp_run_ops_n)
    static_assert(CUBIC_RUN == 8, "two groups of four below");
#pragma unroll 1
    for (int g = 0; g < CUBIC_RUN; g += 4) {
        if (by0 + g >= bh) break;
        ImpPx px[4];
        int bxs[4], bys[4];
#pragma unroll
        for (int o = 0; o < 4; o++) {
            const unsigned w = g ? q[4 + o] : q[o];
            bxs[o] = bx; bys[o] = min(by0 + g + o, bh - 1);
            px[o].b = w & 255; px[o].g = (w >> 8) & 255; px[o].r = (w >> 16) & 255; px[o].a = w >> 24;
        }
        if (nops) imp_run_ops_n<4>(px, oc, bxs, bys, os.ops, nops, os.lut, job.wm, job.wm_pitch, job.wm_c);
#pragma unroll
        for (int o = 0; o < 4; o++) {
            if (by0 + g + o >= bh) break;
            if (dc == 4) store_px<4>(job, P, bx, by0 + g + o, px[o]); else store_px<3>(job, P, bx, by0 + g + o, px[o]);
        }
    }
}

// ---- generic Gaussian (any sigma): horizontal pass to a u16 scratch, vertical pass + ops + store ----
template <int SC>
__global__ void __launch_bounds__(256) imp_blur_h_kernel(const ImpJob job, uint16_t* __restrict__ tmp) {
    const uint8_t* blob = job.pass;
    const ImpPass* __restrict__ P = reinterpret_cast<const ImpPass*>(blob);
    const int w = P->sw, h = P->sh, n = P->ksize, r = n / 2;
    const int x = blockIdx.x * TILE_W + threadIdx.x, y = blockIdx.y * TILE_H + threadIdx.y;
    if (x >= w || y >= h) return;
    const int* taps = reinterpret_cast<const int*>(blob + P->taps_off);
    const uint8_t* row = job.src + (size_t)(P->sy0 + y) * job.src_pitch + (size_t)P->sx0 * SC;
    unsigned acc[SC];
#pragma unroll
    for (int c = 0; c < SC; c++) acc[c] = 0;
    for (int i = 0; i < n; i++) {
        const int sx = min(max(x + i - r, 0), w - 1);
        const unsigned k = (unsigned)__ldg(taps + i);
#pragma unroll
        for (int c = 0; c < SC; c++) acc[c] += (unsigned)__ldg(row + sx * SC + c) * k;
    }
#pragma unroll
    for (int c = 0; c < SC; c++) tmp[((size_t)y * w + x) * SC + c] = (uint16_t)acc[c];
}

template <int SC>
__global__ void __launch_bounds__(256) imp_blur_v_kernel(const ImpJob job, const uint16_t* __restrict__ tmp) {
    extern __shared__ __align__(16) uint8_t smem[];
    const uint8_t* blob = job.pass;
    const ImpPass* __restrict__ P = reinterpret_cast<const ImpPass*>(blob);
    OpsSmem os = stage_ops(P, blob, smem);
    const int w = P->sw, h = P->sh, n = P->ksize, r = n / 2;
    const int x = blockIdx.x * TILE_W + threadIdx.x, y = blockIdx.y * TILE_H + threadIdx.y;
    if (x >= w || y >= h) return;
    const int* taps = reinterpret_cast<const int*>(blob + P->taps_off);
    unsigned acc[SC];
#pragma unroll
    for (int c = 0; c < SC; c++) acc[c] = 0;
    for (int jj = 0; jj < n; jj++) {
        const int sy = min(max(y + jj - r, 0), h - 1);
        const unsigned k = (unsigned)__ldg(taps + jj);
#pragma unroll
        for (int c = 0; c < SC; c++) acc[c] += (unsigned)__ldg(tmp + ((size_t)sy * w + x) * SC + c) * k;
    }
    int v[4] = {0, 0, 0, 255};
#pragma unroll
    for (int c = 0; c < SC; c++) v[c] = (int)((acc[c] + 32768u) >> 16);
    ImpPx p;
    promote<SC>(v, p);
    const int oc = P->oc;
    imp_run_ops(p, oc, x, y, os.ops, P->nops, os.lut, job.wm, job.wm_pitch, job.wm_c);
    if (P->dc == 4) store_px<4>(job, P, x, y, p); else store_px<3>(job, P, x, y, p);
}

template <int KIND>
cudaError_t launch_direct_sc(const ImpLaunchGroup& g, const ImpJob* d_jobs, const ImpJob* one, cudaStream_t st) {
    const dim3 block(TILE_W, TILE_H);                  // grid.x: 32 x (8 * PASS_PPT) tiles
    switch (g.sc) {
        case 1: return imp_launch_jobs<imp_pass_kernel<KIND, 1>, false>(g, block, d_jobs, one, st);
        case 3: return imp_launch_jobs<imp_pass_kernel<KIND, 3>, false>(g, block, d_jobs, one, st);
        case 4: return imp_launch_jobs<imp_pass_kernel<KIND, 4>, false>(g, block, d_jobs, one, st);
    }
    return cudaErrorInvalidValue;
}

cudaError_t launch_direct(const ImpLaunchGroup& g, const ImpJob* d_jobs, const ImpJob* one, cudaStream_t st) {
    switch (g.kind) {
        case IMP_G_COPY:      return launch_direct_sc<IMP_G_COPY>(g, d_jobs, one, st);
        case IMP_G_NN:        return launch_direct_sc<IMP_G_NN>(g, d_jobs, one, st);
        case IMP_G_AREA_INT:  return launch_direct_sc<IMP_G_AREA_INT>(g, d_jobs, one, st);
        case IMP_G_AREA_FRAC: return launch_direct_sc<IMP_G_AREA_FRAC>(g, d_jobs, one, st);
        case IMP_G_CUBIC:     return launch_direct_sc<IMP_G_CUBIC>(g, d_jobs, one, st);
        case IMP_G_LINEAR:    return launch_direct_sc<IMP_G_LINEAR>(g, d_jobs, one, st);
    }
    return cudaErrorInvalidValue;
}

cudaError_t launch_cubic_run(const ImpLaunchGroup& g, const ImpJob* d_jobs, const ImpJob* one, cudaStream_t st) {
    const dim3 block(TILE_W, TILE_H);                  // grid.x: 32 x (8 * CUBIC_RUN) tiles
    switch (g.sc) {
        case 1: return imp_launch_jobs<imp_cubic_run_kernel<1>, false>(g, block, d_jobs, one, st);
        case 3: return imp_launch_jobs<imp_cubic_run_kernel<3>, false>(g, block, d_jobs, one, st);
        case 4: return imp_launch_jobs<imp_cubic_run_kernel<4>, false>(g, block, d_jobs, one, st);
    }
    return cudaErrorInvalidValue;
}

}  // namespace

cudaError_t imp_launch_group(const ImpLaunchGroup& g, const ImpJob* d_jobs, const ImpJob* one, cudaStream_t st) {
    switch (g.kernel) {
        case ImpKernel::Direct:     return launch_direct(g, d_jobs, one, st);
        case ImpKernel::Strip:      return imp_launch_strip(g, d_jobs, one, st);          // imp_k_strip.cu
        case ImpKernel::BlurTile:   return imp_launch_blur_tile(g, d_jobs, one, st);      // imp_k_blur.cu
        case ImpKernel::CubicRun:   return launch_cubic_run(g, d_jobs, one, st);
        case ImpKernel::CubicTile:  return imp_launch_cubic_tile(g, d_jobs, one, st);     // imp_k_cubic.cu
        case ImpKernel::GatherTile: return imp_launch_gather_tile(g, d_jobs, one, st);    // imp_k_gather.cu
        case ImpKernel::BlurGeneric: break;                                               // imp_launch_blur_generic
    }
    return cudaErrorInvalidValue;
}

cudaError_t imp_launch_blur_generic(const ImpJob& job, const ImpPass& hdr, uint16_t* d_scratch, int smem_bytes, cudaStream_t st) {
    dim3 block(TILE_W, TILE_H);
    dim3 grid((hdr.sw + TILE_W - 1) / TILE_W, (hdr.sh + TILE_H - 1) / TILE_H);
    switch (hdr.sc) {
        case 3:
            imp_blur_h_kernel<3><<<grid, block, 0, st>>>(job, d_scratch);
            imp_blur_v_kernel<3><<<grid, block, smem_bytes, st>>>(job, d_scratch);
            break;
        case 4:
            imp_blur_h_kernel<4><<<grid, block, 0, st>>>(job, d_scratch);
            imp_blur_v_kernel<4><<<grid, block, smem_bytes, st>>>(job, d_scratch);
            break;
        default: return cudaErrorInvalidValue;
    }
    g_imp_launches += 2;
    return cudaGetLastError();
}
