// imp_internal.h — host-side internals of libimp_gpu.so (not part of the ABI).
#pragma once
#include <stdint.h>
#include <atomic>
#include <memory>
#include <string>
#include <vector>
#include <cuda_runtime.h>
#include "imp_plan.h"
#include "../../include/imp_gpu.h"

// ---- launch choice --------------------------------------------------------------------------------
// The kernel that runs a pass. The values order a pass's launch groups (batch_compile sorts by them); BlurGeneric sorts
// before BlurTile, where the two-launch Gaussian has always stood.
enum class ImpKernel : int {
    BlurGeneric = -1,    // imp_blur_h_kernel + imp_blur_v_kernel through a u16 plane, one job per launch pair (any sigma)
    Direct = 0,          // imp_pass_kernel<KIND, C> (imp_kernels.cu): any pitch, alignment and footprint
    Strip = 1,           // imp_strip_kernel<C, MODE, FL> (imp_tiles.cuh): INTER_AREA, shrinking INTER_LINEAR
    BlurTile = 2,        // imp_blur_tile_kernel<C, R, NOCOMP> (imp_blur.cuh): tap radius <= 12
    CubicRun = 3,        // imp_cubic_run_kernel<C> (imp_kernels.cu): INTER_CUBIC, any pitch and alignment
    CubicTile = 4,       // imp_cubic_tile_kernel<C, LIGHT> (imp_cubic.cuh)
    GatherTile = 5,      // imp_gather_tile_kernel<C, KIND, LIGHT> (imp_gathertile.cuh): index map, NN, enlarging INTER_LINEAR
};
// Dynamic shared memory the tile kernels are configured for (cudaFuncAttributeMaxDynamicSharedMemorySize); a tile launch
// whose footprint exceeds it (many LUT filters can push a pass over) takes the pass's fallback kernel instead.
constexpr int IMP_SMEM_OPTIN = 200 * 1024;
// How one job of a pass is launched.
struct ImpLaunch {
    ImpKernel kernel;
    int param;           // Strip: ring stages; BlurTile: tap radius; CubicTile, GatherTile: tile edge; otherwise 0
    int flavour;         // op interpreter: 0 general, 1 fused tables only, 2 (Strip) compositing + tables; BlurTile: 1 = NOCOMP
    int smem_bytes;      // dynamic shared memory
    int ctas_per_job;    // grid.x (BlurGeneric: 0, its launches size their own 2-D grid)
    int ctas_per_sm;     // Strip: CTAs of this footprint an SM holds, the occupancy class strip jobs are grouped by; otherwise 0
};
// imp_planner.cpp: the launch of pass `h` on kernel `k` (one that serves the pass's kind), and the pass's two choices
// (ImpHostPass::tiled, ::fallback below).
ImpLaunch imp_pass_launch(const ImpPass& h, ImpKernel k);
void imp_pass_launches(const ImpPass& h, ImpLaunch* tiled, ImpLaunch* fallback);

// ---- planner output (host) ------------------------------------------------------------------------
struct ImpHostPass {
    ImpPass hdr;                       // offsets filled by finalize()
    std::vector<uint8_t> blob;         // ImpPass + tables + ops + LUTs, ready to upload
    int in_w, in_h, in_c;              // input image of the pass (whole image, before the window)
    int out_w, out_h, out_c;           // stored image
    int uses_watermark;
    double sigma;                      // BLUR only
    // Jobs whose source rows are 16-byte addressable take `tiled` (a shared-memory tile kernel when the pass has one and
    // its footprint fits IMP_SMEM_OPTIN, else the same as `fallback`); every other job takes `fallback`: Direct, CubicRun
    // or BlurGeneric by kind.
    ImpLaunch tiled, fallback;
};

// A decoded overlay (what PrepareWatermark leaves in the conf pool, bridge.c:199-237). The reference decodes it ONCE at
// configuration time and every request blends the same pixels (bridge.c:239-281); here it is interned by content, shared
// by every plan that uses it and uploaded once per device (imp_gpu_upload_watermark, or lazily on first use).
struct ImpWmImage {
    std::vector<uint8_t> pixels;       // tightly packed, w*c bytes per row
    int w = 0, h = 0, c = 0;
    unsigned long long hash = 0;
    struct Dev { uint8_t* d = nullptr; int pitch = 0; };
    Dev dev[16];
    ~ImpWmImage();                     // releases the device copies through imp_wm_dev_release (set by imp_gpu.cu)
};
extern void (*imp_wm_dev_release)(ImpWmImage*);
// imp_planner.cpp: the shared image holding exactly these pixels (registered on first sight; bounded registry).
std::shared_ptr<ImpWmImage> imp_wm_intern(const imp_gpu_watermark* wm);
void imp_wm_registry_clear();

struct imp_gpu_plan {
    std::vector<ImpHostPass> passes;
    int src_w, src_h, src_c;
    int win_x, win_y, win_w, win_h;    // crop window in the source
    int out_w, out_h, out_c;
    unsigned long long algo_bytes;     // SURVEY §8d
    std::shared_ptr<ImpWmImage> wm;    // overlay the plan blends (shared, uploaded once per device), or null
    int pack = IMP_PACK_NONE;          // the request's IMP_PACK_*: the layout of the stored result
    std::atomic<int> refs{1};          // the plan cache and every imp_gpu_plan_create caller hold one reference each
    // per-device state: ONE stream-ordered allocation holds every pass blob (+ vignette tables), filled by an
    // asynchronous copy from pinned staging; `ready_ev` orders the first kernels behind it
    struct Dev {
        std::vector<uint8_t*> pass_blobs;          // pointers into `arena`
        uint8_t* arena = nullptr;
        cudaEvent_t ready_ev = nullptr;
        std::atomic<bool> settled{false};          // the upload is known to have completed
        bool ready = false;
    };
    Dev dev[16];
};

// imp_planner.cpp. `dry`: validate only — same codes, steps and output geometry, but no tables, LUTs, blobs or
// watermark pixels are materialised (what each recorded operator of the imp_ops layer needs).
int imp_build_plan(const imp_gpu_request* req, const imp_gpu_config* cfg, int w, int h, int c,
                   imp_gpu_plan* plan, int* step, bool dry = false);

inline int align16(int v) { return (v + 15) & ~15; }
inline size_t align256(size_t v) { return (v + 255) & ~size_t(255); }

// ---- host jobs and how they cross the link (imp_transfer.cpp: pure host logic, no CUDA call) ----------------------
// One job of the chunked host path. A frame result goes to (dst, dst_step); an answer is a one-row result: brightness
// writes 4 bytes (a float) at dst, ASCII imp_gpu_ascii_length bytes with the 70-level ramp where `wide`.
struct ImpHostJob { imp_gpu_plan* plan; const uint8_t* src; int src_step; uint8_t* dst; int dst_step; bool wide; };
enum class ImpResult { Frame, Brightness, Ascii };
constexpr int IMP_CHUNK_JOBS = 256;                  // the most jobs a chunk holds
constexpr size_t IMP_CHUNK_BYTES = 128u << 20;       // the most crop-window + result bytes a chunk holds (one job may exceed it)
// The chunk boundaries [0, e1, ..., n] of n jobs over n_streams lanes (clamped to 1..8).
std::vector<int> imp_chunk_bounds(const ImpHostJob* jobs, int n, int n_streams);

// How a job's source reaches the device and its result the host.
enum class ImpRoute : uint8_t {
    Resident,        // source: already on this device (GIF canvases), nothing to upload
    Staged,          // pageable host memory, through the lane's pinned staging (h_in / h_out)
    Linear,          // pinned: one linear copy (source: into d_in at the device pitch; frame result: out of d_out)
    LinearRepitch,   // pinned source of short rows: one linear copy of the rows the window touches into d_stage, then a
                     // re-pitch kernel into d_in
    Rows2D,          // pinned: one 2-D copy
    Direct,          // pinned answer: straight from the device into the destination
};
struct ImpJobLayout {
    ImpRoute src, dst;
    int in_pitch, out_pitch;     // device pitches of the crop window (d_in) and of the result (d_out)
    size_t in_off, out_off;      // d_in, d_out
    size_t lin_bytes;            // Linear, LinearRepitch sources: bytes of the one copy
    size_t stage_off;            // LinearRepitch: d_stage
    size_t hin_off;              // Staged source: h_in, rows at in_pitch
    size_t hout_off;             // Staged result: h_out, frame rows packed at out_w*out_c
    size_t res_bytes;            // bytes handed to the host: the frame's rows, 4 (brightness) or the text's length
    int slices;                  // Staged source: uploaded in this many row slices (each as soon as it is staged)
};
struct ImpChunkLayout {
    std::vector<ImpJobLayout> jobs;
    size_t in_total = 0, out_total = 0, stage_total = 0, hin_total = 0, hout_total = 0;   // buffer sizes the chunk needs
};
// The routes and offsets of a chunk of m jobs. `resident`: every source is already on the device; src_pinned[k] /
// dst_pinned[k]: whether job k's source / destination is page-locked (brightness: dst_pinned[0] decides for the chunk,
// whose floats come back in one copy).
ImpChunkLayout imp_chunk_layout(const ImpHostJob* jobs, int m, ImpResult kind, bool resident, const bool* src_pinned, const bool* dst_pinned);

// imp_kernels.cu
#define IMP_CUBIC_RUN 8           // imp_cubic_run_kernel: output rows per thread; a CTA covers 32 x (8 * IMP_CUBIC_RUN) pixels
unsigned long long imp_launches();
void imp_count_launches(int n);
// One launch over jobs that share kind, source channels and the launch choice (kernel, param, flavour).
struct ImpLaunchGroup {
    int kind, sc;                // ImpGather and source channels of every job
    ImpKernel kernel;            // never BlurGeneric (imp_launch_blur_generic)
    int param, flavour;          // as in ImpLaunch
    int first, count;            // jobs [first, first+count) of the device job table
    int ctas;                    // grid.x: the largest ctas_per_job of the group
    int smem_bytes;              // the largest smem_bytes of the group
};
// d_jobs == nullptr: a single job passed by value (`one`), no device job table needed.
cudaError_t imp_launch_group(const ImpLaunchGroup& g, const ImpJob* d_jobs, const ImpJob* one, cudaStream_t st);
#if defined(__CUDACC__)
// Launches Kernel(jobs, first, count, one, extra...) over a group: grid.x = g.ctas, the jobs over grid.y (and z beyond
// 65535). OptIn: the kernel is configured for IMP_SMEM_OPTIN bytes of dynamic shared memory, once per device.
template <auto Kernel, bool OptIn = true, class... Extra>
cudaError_t imp_launch_jobs(const ImpLaunchGroup& g, dim3 block, const ImpJob* d_jobs, const ImpJob* one, cudaStream_t st, Extra... extra) {
    if (OptIn) {
        static std::atomic<bool> attr_set[16];             // per device; setting the attribute twice is harmless
        int dev = 0; cudaGetDevice(&dev);
        if (!attr_set[dev & 15]) {
            cudaError_t e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, IMP_SMEM_OPTIN);
            if (e != cudaSuccess) return e;
            attr_set[dev & 15] = true;
        }
    }
    const ImpJob dummy{};
    dim3 grid(g.ctas, g.count < 65535 ? g.count : 65535, (g.count + 65534) / 65535);
    Kernel<<<grid, block, g.smem_bytes, st>>>(d_jobs, g.first, g.count, one ? *one : dummy, extra...);
    imp_count_launches(1);
    return cudaGetLastError();
}
#endif
// Two-kernel Gaussian through a u16 scratch (any sigma). One job, passed by value.
cudaError_t imp_launch_blur_generic(const ImpJob& job, const ImpPass& hdr, uint16_t* d_scratch, int smem_bytes, cudaStream_t st);
cudaError_t imp_upload_tables();
// one translation unit per kernel family (each with its own copy of the per-byte division tables, imp_pixel.cuh)
cudaError_t imp_upload_tables_strip();
cudaError_t imp_upload_tables_blur();
cudaError_t imp_upload_tables_cubic();
cudaError_t imp_upload_tables_gather();
unsigned imp_debug_flags_strip(); unsigned imp_debug_flags_blur(); unsigned imp_debug_flags_cubic(); unsigned imp_debug_flags_gather();
cudaError_t imp_launch_strip(const ImpLaunchGroup& g, const ImpJob* d_jobs, const ImpJob* one, cudaStream_t st);        // imp_k_strip.cu
cudaError_t imp_launch_blur_tile(const ImpLaunchGroup& g, const ImpJob* d_jobs, const ImpJob* one, cudaStream_t st);    // imp_k_blur.cu
cudaError_t imp_launch_cubic_tile(const ImpLaunchGroup& g, const ImpJob* d_jobs, const ImpJob* one, cudaStream_t st);   // imp_k_cubic.cu
cudaError_t imp_launch_gather_tile(const ImpLaunchGroup& g, const ImpJob* d_jobs, const ImpJob* one, cudaStream_t st);  // imp_k_gather.cu
// rows of `row_bytes` bytes from (src, sp) to (dst, dp); dst and dp are multiples of 4 (the library's own pitched buffers)
cudaError_t imp_launch_repitch(const uint8_t* d_src, int sp, uint8_t* d_dst, int dp, int row_bytes, int rows, cudaStream_t st);
cudaError_t imp_launch_gif_expand(const ImpGifFrame* d_frames, int n, int cw, int ch, int destructive, uint8_t* d_canvases, int cpitch, cudaStream_t st);
// One frame of a brightness or ASCII launch: a result on the device and where its answer goes.
struct ImpInfoJob {
    const uint8_t* img;          // rows of w*c bytes (c in {1,3,4}), `pitch` apart
    long long text_off;          // ASCII: the job's first byte in the text arena
    int pitch, w, h, c;
    int vec;                     // 1: img and pitch are multiples of 16 (rows are read 16 bytes at a time)
    int ctas;                    // CTAs over this job: imp_brightness_ctas / imp_ascii_ctas of (w, h)
    int part_off;                // brightness: the first of the job's `ctas` partial sums
    int wide;                    // ASCII: 1 = the 70-level ramp, 0 = the 10-level one
};
struct ImpAsciiRamps { uint8_t lut[2][256]; };   // HSV value -> character, [0] 10-level ramp, [1] 70-level ramp
int imp_brightness_ctas(int w, int h);
int imp_ascii_ctas(int w, int h);
// n jobs from the device table d_jobs, or (d_jobs == nullptr, n == 1) the job `one` passed by value; grid.x = max_ctas, the
// largest ctas of the jobs. Brightness: out[j] = brightness of job j; tickets[0..n) must be 0 and are left 0.
cudaError_t imp_launch_brightness(const ImpInfoJob* d_jobs, const ImpInfoJob& one, int n, int max_ctas, double* partials, unsigned* tickets, float* out, cudaStream_t st);
cudaError_t imp_launch_ascii(const ImpInfoJob* d_jobs, const ImpInfoJob& one, int n, int max_ctas, const ImpAsciiRamps& ramps, uint8_t* text, cudaStream_t st);
cudaError_t imp_build_vignette_table(float* d_tab, int nx, int ny, float maxr, float intensity, cudaStream_t st);          // per-device constant tables of imp_pixel.cuh
