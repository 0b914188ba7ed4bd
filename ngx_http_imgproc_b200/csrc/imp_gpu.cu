// imp_gpu.cu — the C ABI of libimp_gpu.so (include/imp_gpu.h): device contexts, plan upload,
// batches, the end-to-end host paths (pinned staging + streams) and the multi-GPU farm.
// No CPU fallback exists anywhere in this file: if CUDA is unusable every compute call fails with
// IMP_ERROR_GPU and a message in imp_gpu_last_error().
#include "imp_internal.h"
#include <cuda.h>
#include <stdio.h>
#include <math.h>
#include <string.h>
#include <stdlib.h>
#include <unistd.h>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <deque>
#include <functional>
#include <list>
#include <mutex>
#include <new>
#include <thread>
#include <tuple>
#include <unordered_map>

namespace {

constexpr int MAX_DEV = 16;
thread_local char t_err[512] = "";
thread_local int t_dev = -1;

int fail(cudaError_t e, const char* what, int line) {
    snprintf(t_err, sizeof t_err, "%s failed at imp_gpu.cu:%d: %s", what, line, cudaGetErrorString(e));
    return IMP_ERROR_GPU;
}
int fail_msg(const char* msg) { snprintf(t_err, sizeof t_err, "%s", msg); return IMP_ERROR_GPU; }

#define CK(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return fail(e__, #call, __LINE__); } while (0)

// A growable buffer (device or pinned host) that is only ever re-allocated when a request outgrows it.
struct Buf {
    uint8_t* p = nullptr; size_t cap = 0;
    int grow(size_t need, bool host) {
        if (need <= cap) return IMP_OK;
        if (p) { if (host) CK(cudaFreeHost(p)); else CK(cudaFree(p)); p = nullptr; cap = 0; }
        need = (need * 5 / 4 + 4095) & ~size_t(4095);
        if (host) CK(cudaHostAlloc((void**)&p, need, cudaHostAllocDefault)); else CK(cudaMalloc((void**)&p, need));
        cap = need;
        return IMP_OK;
    }
    void release(bool host) { if (p) { if (host) cudaFreeHost(p); else cudaFree(p); } p = nullptr; cap = 0; }
};

}  // namespace

// ---- batch ---------------------------------------------------------------------------------------------
struct ImpTmKey {
    uintptr_t a0; unsigned long long g0, g1; int pitch; unsigned b0, b1;
    bool operator==(const ImpTmKey& o) const { return a0 == o.a0 && g0 == o.g0 && g1 == o.g1 && pitch == o.pitch && b0 == o.b0 && b1 == o.b1; }
};
struct ImpTmKeyHash {
    size_t operator()(const ImpTmKey& k) const {
        unsigned long long h = k.a0 * 0x9E3779B97F4A7C15ull;
        h ^= (k.g0 + 0x632BE59BD9B4E019ull + (h << 6) + (h >> 2));
        h ^= (k.g1 * 0xC2B2AE3D27D4EB4Full + (h << 6) + (h >> 2));
        h ^= ((unsigned long long)(unsigned)k.pitch << 32 | k.b0) + (h << 6) + (h >> 2);
        h ^= k.b1 + (h << 6) + (h >> 2);
        return (size_t)h;
    }
};
struct ImpTmap { unsigned char bytes[128]; };

struct imp_gpu_batch {
    struct Item { imp_gpu_plan* plan; const uint8_t* src; int sp; uint8_t* dst; int dp; };
    std::vector<Item> items;
    int dev = -1;
    bool dirty = true;
    // compiled form
    std::vector<ImpJob> h_jobs;
    ImpJob* d_jobs = nullptr; size_t jobs_cap = 0;
    Buf h_pin;                                   // pinned staging of the job table (the upload is asynchronous)
    cudaEvent_t up_ev = nullptr; bool up_pending = false;
    bool table_needed = false;                   // false when every launch group holds one job (passed by value)
    Buf scratch;
    struct Step { ImpLaunchGroup g; ImpPass hdr; uint16_t* plane; };     // hdr, plane: BlurGeneric only (its u16 plane)
    std::vector<Step> steps;
    unsigned long long algo_bytes = 0;
    int launches = 0;
    // tensor maps are encoded once per (buffer, geometry): the staging lanes present the same addresses again and again
    using TmCache = std::unordered_map<ImpTmKey, ImpTmap, ImpTmKeyHash>;
    TmCache tmaps;
};

namespace {

struct Lane {            // one in-flight chunk of host jobs of the end-to-end path
    cudaStream_t st = nullptr;
    cudaEvent_t up_done = nullptr;               // this chunk's uploads have been issued up to here: the next chunk's wait for it
    Buf d_in, d_out, d_stage;                    // device: re-pitched crop windows, results, linear landing zone of short rows
    Buf h_in, h_out;                             // pinned staging for host buffers that are not page-locked
    imp_gpu_batch batch;                         // the chunk's job table, scratch and tensor maps
    Buf d_info, h_info;                          // brightness / ASCII: job table, partial sums, answers, texts; the table's pinned staging
    Buf d_tickets;                               // brightness: one ticket per job of a chunk, zeroed once (the kernel leaves them 0)
    bool busy = false;                           // a chunk was issued and is not finished
    struct Out { uint8_t* dst; size_t dst_step, row_bytes; int rows; size_t hout_off; };   // staged results: copied from h_out after the sync
    std::vector<Out> pend;
};
struct DevCtx {
    bool ready = false;
    cudaStream_t stream = nullptr;               // uploads (plans, overlays) and the library's default stream
    Buf h_up; cudaEvent_t up_ev = nullptr; bool up_pending = false;   // pinned staging of plan uploads
    std::vector<Lane*> lanes;                    // persistent staging, reused across calls
    std::mutex run_mu;                           // serialises users of `lanes`
    Buf h_gif, d_gif, d_canvas; cudaEvent_t gif_ev = nullptr;   // GIF albums: packed pages (pinned / device), expanded BGRA canvases
};
DevCtx g_dev[MAX_DEV];
std::mutex g_mu;

int cur_dev() {
    if (t_dev >= 0) return t_dev;
    std::lock_guard<std::mutex> lk(g_mu);
    for (int d = 0; d < MAX_DEV; d++) if (g_dev[d].ready) { t_dev = d; return d; }
    return -1;
}

int bind() {          // make the thread's device current
    int d = cur_dev();
    if (d < 0) return fail_msg("imp_gpu_init() has not been called (no CUDA device initialised; there is no CPU fallback)");
    CK(cudaSetDevice(d));
    return IMP_OK;
}

cudaStream_t pick_stream(void* s) { return s ? (cudaStream_t)s : g_dev[t_dev].stream; }

// The overlay on device `d` (uploaded once per device for the life of the image; caller holds g_mu).
int wm_to_device(ImpWmImage* wm, int d) {
    ImpWmImage::Dev& wd = wm->dev[d];
    if (wd.d) return IMP_OK;
    wd.pitch = align16(wm->w * wm->c);
    CK(cudaMalloc((void**)&wd.d, (size_t)wd.pitch * wm->h));
    // `pixels` lives as long as the image does, so the copy may stay in flight on the upload stream
    CK(cudaMemcpy2DAsync(wd.d, wd.pitch, wm->pixels.data(), (size_t)wm->w * wm->c, (size_t)wm->w * wm->c, wm->h, cudaMemcpyHostToDevice, g_dev[d].stream));
    return IMP_OK;
}

void wm_release_device(ImpWmImage* wm) {
    for (int d = 0; d < MAX_DEV; d++) {
        if (!wm->dev[d].d) continue;
        if (g_dev[d].ready && cudaSetDevice(d) == cudaSuccess) cudaFree(wm->dev[d].d);
        wm->dev[d].d = nullptr;
    }
    if (t_dev >= 0) cudaSetDevice(t_dev);
}
struct WmHook { WmHook() { imp_wm_dev_release = wm_release_device; } } g_wm_hook;

// Uploads the plan's pass blobs (+ vignette tables, overlay) to the current device, once. Nothing here blocks on the GPU:
// one stream-ordered allocation, one copy from pinned staging on the device's upload stream, an event for the consumers.
int plan_to_device(imp_gpu_plan* plan) {
    const int d = t_dev;
    imp_gpu_plan::Dev& pd = plan->dev[d];
    std::lock_guard<std::mutex> lk(g_mu);
    if (pd.ready) return IMP_OK;
    DevCtx& ctx = g_dev[d];
    std::vector<size_t> off(plan->passes.size());
    size_t blob_total = 0;
    for (size_t i = 0; i < plan->passes.size(); i++) { off[i] = blob_total; blob_total += align256(plan->passes[i].blob.size()); }
    size_t total = blob_total;
    struct Tab { size_t pass, op, off; };
    std::vector<Tab> tabs;
    for (size_t i = 0; i < plan->passes.size(); i++) {
        const ImpPass& h = plan->passes[i].hdr;
        const ImpOp* ops = reinterpret_cast<const ImpOp*>(plan->passes[i].blob.data() + h.ops_off);
        for (int k = 0; k < h.nops; k++)
            if (ops[k].kind == IMP_OP_VIGNETTE && ops[k].i[2] > 0) { tabs.push_back(Tab{i, (size_t)k, total}); total += align256((size_t)ops[k].i[2] * ops[k].i[3] * sizeof(float)); }
    }
    if (ctx.up_pending) { CK(cudaEventSynchronize(ctx.up_ev)); ctx.up_pending = false; }      // the staging buffer is free again
    int rc = ctx.h_up.grow(blob_total, true); if (rc) return rc;
    CK(cudaMallocAsync((void**)&pd.arena, std::max<size_t>(total, 256), ctx.stream));
    pd.pass_blobs.assign(plan->passes.size(), nullptr);
    for (size_t i = 0; i < plan->passes.size(); i++) {
        memcpy(ctx.h_up.p + off[i], plan->passes[i].blob.data(), plan->passes[i].blob.size());
        pd.pass_blobs[i] = pd.arena + off[i];
    }
    for (const Tab& t : tabs) {                  // per-device copy of the op: the table pointer is patched in
        const ImpPass& h = plan->passes[t.pass].hdr;
        ImpOp* op = reinterpret_cast<ImpOp*>(ctx.h_up.p + off[t.pass] + h.ops_off) + t.op;
        float* tab = reinterpret_cast<float*>(pd.arena + t.off);
        CK(imp_build_vignette_table(tab, op->i[2], op->i[3], op->f[0], op->f[1], ctx.stream));
        const unsigned long long v = (unsigned long long)(uintptr_t)tab;
        op->i[4] = (int)(unsigned)(v & 0xffffffffu); op->i[5] = (int)(unsigned)(v >> 32);
        // With a table the device never takes the per-pixel path, so this device's copy of the op carries the lookup's affine
        // form instead of the centre and the frame map (imp_pixel.cuh, IMP_OP_VIGNETTE): dx = ox + xa*bx + xb*by,
        // dy = oy + ya*bx + yb*by, where dx = cx - x, x = flipx ? w-1-u : u, u = swap ? by : bx (and likewise dy)
        {
            const ImpFrameMap m = op->map;
            const int sx = m.flipx ? 1 : -1, ox = op->i[0] - (m.flipx ? m.w - 1 : 0);
            const int sy = m.flipy ? 1 : -1, oy = op->i[1] - (m.flipy ? m.h - 1 : 0);
            op->i[0] = ox; op->i[1] = oy;
            op->map.swap = m.swap ? 0 : sx;      // xa
            op->map.flipx = m.swap ? sx : 0;     // xb
            op->map.flipy = m.swap ? sy : 0;     // ya
            op->map.w = m.swap ? 0 : sy;         // yb
            op->map.h = 0;
        }
    }
    if (blob_total) CK(cudaMemcpyAsync(pd.arena, ctx.h_up.p, blob_total, cudaMemcpyHostToDevice, ctx.stream));
    if (plan->wm) { rc = wm_to_device(plan->wm.get(), d); if (rc) return rc; }
    if (!pd.ready_ev) CK(cudaEventCreateWithFlags(&pd.ready_ev, cudaEventDisableTiming));
    CK(cudaEventRecord(pd.ready_ev, ctx.stream));
    CK(cudaEventRecord(ctx.up_ev, ctx.stream));
    ctx.up_pending = true;
    pd.settled = false;
    pd.ready = true;
    return IMP_OK;
}

// Orders work on `st` behind the plan's upload (a no-op once the upload is known to be complete).
int plan_wait_ready(imp_gpu_plan* plan, cudaStream_t st) {
    imp_gpu_plan::Dev& pd = plan->dev[t_dev];
    if (pd.settled.load(std::memory_order_acquire)) return IMP_OK;
    cudaError_t e = cudaEventQuery(pd.ready_ev);
    if (e == cudaSuccess) { pd.settled.store(true, std::memory_order_release); return IMP_OK; }
    if (e != cudaErrorNotReady) return fail(e, "cudaEventQuery", __LINE__);
    if (st != g_dev[t_dev].stream) CK(cudaStreamWaitEvent(st, pd.ready_ev, 0));
    return IMP_OK;
}

// Device memory of plans that were destroyed (cache evictions, mostly): kernels on any stream may still be reading the
// blobs, so the arenas are parked and released in batches behind ONE device synchronisation (caller holds g_mu).
struct Parked { int dev; uint8_t* arena; };
std::vector<Parked> g_parked;
void parked_release(bool all) {
    if (g_parked.empty() || (!all && g_parked.size() < 32)) return;
    bool synced[MAX_DEV] = {false};
    for (const Parked& p : g_parked) {
        if (!g_dev[p.dev].ready || cudaSetDevice(p.dev) != cudaSuccess) continue;
        if (!synced[p.dev]) { cudaDeviceSynchronize(); synced[p.dev] = true; }
        cudaFreeAsync(p.arena, g_dev[p.dev].stream);     // back into the pool, no further synchronisation
    }
    g_parked.clear();
    if (t_dev >= 0) cudaSetDevice(t_dev);
}

void plan_free_device(imp_gpu_plan* plan) {
    for (int d = 0; d < MAX_DEV; d++) {
        imp_gpu_plan::Dev& pd = plan->dev[d];
        if (!pd.ready) continue;
        if (g_dev[d].ready && cudaSetDevice(d) == cudaSuccess) {
            if (pd.arena) g_parked.push_back(Parked{d, pd.arena});
            if (pd.ready_ev) cudaEventDestroy(pd.ready_ev);
        }
        pd.arena = nullptr; pd.ready_ev = nullptr; pd.pass_blobs.clear();
        pd.ready = false;
    }
    parked_release(false);
}

void plan_release(imp_gpu_plan* plan) {          // drops one reference
    if (!plan) return;
    if (plan->refs.fetch_sub(1) > 1) return;
    { std::lock_guard<std::mutex> lk(g_mu); plan_free_device(plan); }
    if (t_dev >= 0) cudaSetDevice(t_dev);
    delete plan;
}

// ---- plan cache: the same request on the same frame geometry under the same configuration is lowered once ---------------
// (the reference re-parses every request, bridge.c:346-372; its per-config work, PrepareWatermark, happens once per cycle)
struct PlanCache {
    std::mutex mu;
    std::list<std::pair<std::string, imp_gpu_plan*>> lru;             // most recent first; the cache holds one reference each
    std::unordered_map<std::string, std::list<std::pair<std::string, imp_gpu_plan*>>::iterator> map;
    size_t cap = 128;
    unsigned long long hits = 0, misses = 0;
    PlanCache() { const char* e = getenv("IMP_GPU_PLAN_CACHE"); if (e) cap = (size_t)std::max(0, atoi(e)); }
};
PlanCache g_cache;

void key_str(std::string& k, const char* s) { if (s) { k += '1'; k += s; } else k += '0'; k += '\x1f'; }
void key_int(std::string& k, long long v) { char b[32]; snprintf(b, sizeof b, "%lld\x1f", v); k += b; }

std::string plan_key(const imp_gpu_request* req, const imp_gpu_config* cfg, int w, int h, int c, const ImpWmImage* wm) {
    std::string k; k.reserve(192);
    key_int(k, w); key_int(k, h); key_int(k, c);
    key_str(k, req->crop); key_str(k, req->gravity); key_str(k, req->resize);
    key_int(k, req->filter_count);
    for (int i = 0; i < req->filter_count; i++) key_str(k, req->filters[i]);
    key_int(k, req->simple_resize); key_int(k, req->flatten); key_int(k, req->interp); key_int(k, req->pack);
    if (cfg) {
        key_int(k, cfg->max_target_w); key_int(k, cfg->max_target_h); key_int(k, cfg->max_filters); key_int(k, cfg->allow_experiments);
        if (cfg->watermark) {
            const imp_gpu_watermark* m = cfg->watermark;
            key_int(k, (long long)(uintptr_t)wm); key_int(k, m->gravity_x); key_int(k, m->gravity_y);
            key_int(k, m->offset_x); key_int(k, m->offset_y); key_int(k, m->opacity);
        } else k += "nowm";
    } else k += "nocfg";
    return k;
}

void cache_clear() {
    std::vector<imp_gpu_plan*> drop;
    {
        std::lock_guard<std::mutex> lk(g_cache.mu);
        for (auto& e : g_cache.lru) drop.push_back(e.second);
        g_cache.lru.clear(); g_cache.map.clear();
    }
    for (imp_gpu_plan* p : drop) plan_release(p);
    std::lock_guard<std::mutex> lk(g_mu);
    parked_release(true);
}

int pass_pitch(const ImpHostPass& hp) { return align16(hp.out_w * hp.out_c); }

// cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda link dependency).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) p = nullptr;
        return (EncodeTiledFn)p;
    }();
    return fn;
}

// Tensor map over the job's source window for the strip kernels: 8-byte elements, rows = window rows, origin =
// the window's first byte aligned down to 16; box = tile_rs bytes x tile_rows rows. Out-of-range box parts are
// zero-filled by the TMA unit, so edge tiles never touch memory outside the window's rows.
int encode_job_tmap(const ImpPass& h, ImpJob& j, imp_gpu_batch::TmCache* cache) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return fail_msg("cuTensorMapEncodeTiled is unavailable in this driver");
    const uintptr_t win = (uintptr_t)j.src + (size_t)h.sy0 * j.src_pitch + (size_t)h.sx0 * h.sc;
    const uintptr_t a0 = win & ~uintptr_t(15);
    j.tm_x0 = (int)(win - a0);
    const cuuint64_t gdim[2] = {(cuuint64_t)((j.tm_x0 + (size_t)h.sw * h.sc + 7) / 8), (cuuint64_t)h.sh};
    const cuuint64_t gstride[1] = {(cuuint64_t)j.src_pitch};
    const cuuint32_t box[2] = {(cuuint32_t)(h.tile_rs / 8), (cuuint32_t)h.tile_rows};
    const cuuint32_t estr[2] = {1, 1};
    static_assert(sizeof(CUtensorMap) == 128, "CUtensorMap size");
    const ImpTmKey key{a0, gdim[0], gdim[1], j.src_pitch, box[0], box[1]};
    if (cache) {
        auto it = cache->find(key);
        if (it != cache->end()) { memcpy(j.tmap, it->second.bytes, 128); return IMP_OK; }
    }
    CUtensorMap tm;
    CUresult r = enc(&tm, CU_TENSOR_MAP_DATA_TYPE_UINT64, 2, (void*)a0, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { snprintf(t_err, sizeof t_err, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r); return IMP_ERROR_GPU; }
    memcpy(j.tmap, &tm, 128);
    if (cache) {
        if (cache->size() > 8192) cache->clear();
        ImpTmap v; memcpy(v.bytes, &tm, 128);
        cache->emplace(key, v);
    }
    return IMP_OK;
}

// Which of its pass's launches a job takes: `tiled` when the job's source rows are 16-byte addressable — pitch % 16 == 0
// and either the image rows or the window rows start 16-byte aligned (imp_tiles.cuh) — and tensor maps can be encoded,
// `fallback` otherwise. IMP_GPU_FORCE_DIRECT=1 routes every job through imp_pass_kernel (INTER_CUBIC included) or the
// two-launch Gaussian (used by the tests to keep the general paths — unaligned pitches, oversized footprints, large
// sigma — covered on the GPU).
ImpLaunch pick_launch(const ImpHostPass& hp, const uint8_t* src, int sp) {
    static const bool force_direct = [] { const char* e = getenv("IMP_GPU_FORCE_DIRECT"); return e && *e == '1'; }();
    const ImpPass& h = hp.hdr;
    if (force_direct) return imp_pass_launch(h, h.kind == IMP_G_BLUR ? ImpKernel::BlurGeneric : ImpKernel::Direct);
    const uintptr_t img = (uintptr_t)src, win = img + (size_t)h.sy0 * sp + (size_t)h.sx0 * h.sc;
    return encode_tiled() && sp % 16 == 0 && (img % 16 == 0 || win % 16 == 0) ? hp.tiled : hp.fallback;
}
bool uses_tmap(ImpKernel k) { return k == ImpKernel::Strip || k == ImpKernel::BlurTile || k == ImpKernel::CubicTile || k == ImpKernel::GatherTile; }

// Scratch a plan needs on the device: intermediates between passes + the u16 plane of each generic blur.
// off[k] = offset of pass k's output (non-final passes); blur_off[k] = offset of pass k's u16 plane.
// `src`/`sp`: the job's source (null = one of the library's own aligned buffers). The u16 plane is only reserved for a
// blur that takes the generic kernels (radius > 12, or a pass-0 source whose rows are not 16-byte addressable).
size_t plan_scratch_layout(const imp_gpu_plan* p, size_t base, std::vector<size_t>& off, std::vector<size_t>& blur_off,
                           const uint8_t* src = nullptr, int sp = 0) {
    size_t cur = base;
    auto take = [&](size_t bytes) { size_t o = cur; cur += (bytes + 255) & ~size_t(255); return o; };
    off.assign(p->passes.size(), 0); blur_off.assign(p->passes.size(), 0);
    for (size_t k = 0; k < p->passes.size(); k++) {
        const ImpHostPass& hp = p->passes[k];
        if (k + 1 < p->passes.size()) off[k] = take((size_t)pass_pitch(hp) * hp.out_h);
        if (hp.hdr.kind == IMP_G_BLUR && pick_launch(hp, k == 0 ? src : nullptr, k == 0 ? sp : 0).kernel == ImpKernel::BlurGeneric)
            blur_off[k] = take((size_t)hp.hdr.sw * hp.hdr.sh * hp.hdr.sc * 2);
    }
    return cur;
}

ImpJob make_job(const imp_gpu_plan* p, int d, size_t k, const uint8_t* src, int sp, uint8_t* dst, int dp,
                uint8_t* scratch, const std::vector<size_t>& off) {
    const imp_gpu_plan::Dev& pd = p->dev[d];
    ImpJob j{};
    j.pass = pd.pass_blobs[k];
    if (p->wm) { j.wm = p->wm->dev[d].d; j.wm_pitch = p->wm->dev[d].pitch; j.wm_c = p->wm->c; }
    if (k == 0) { j.src = src; j.src_pitch = sp; }
    else { j.src = scratch + off[k - 1]; j.src_pitch = pass_pitch(p->passes[k - 1]); }
    if (k + 1 == p->passes.size()) { j.dst = dst; j.dst_pitch = dp; }
    else { j.dst = scratch + off[k]; j.dst_pitch = pass_pitch(p->passes[k]); }
    return j;
}

// Turns `items` into launch steps and the jobs they cover (in device-table order), pass by pass. Within a pass the jobs are
// grouped by (kind, exact integer AREA taps, sc, kernel, param, flavour, ctas_per_sm), one launch per group in that order; a generic blur is a step
// of its own. alloc(bytes, &p): where the items' scratch lives (plan_scratch_layout, item after item).
template <class Alloc>
int build_steps(const std::vector<imp_gpu_batch::Item>& items, Alloc alloc, imp_gpu_batch::TmCache* tmaps,
                std::vector<imp_gpu_batch::Step>& steps, std::vector<ImpJob>& jobs) {
    steps.clear(); jobs.clear();
    std::vector<std::vector<size_t>> off(items.size()), boff(items.size());
    size_t bytes = 0;
    size_t max_passes = 0;
    for (size_t i = 0; i < items.size(); i++) {
        bytes = plan_scratch_layout(items[i].plan, bytes, off[i], boff[i], items[i].src, items[i].sp);
        max_passes = std::max(max_passes, items[i].plan->passes.size());
    }
    uint8_t* scratch = nullptr;
    if (int rc = alloc(bytes, &scratch)) return rc;
    struct Pending {
        const ImpPass* hdr; ImpLaunch l; ImpJob job; uint16_t* plane;
        auto key() const { return std::make_tuple(hdr->kind, hdr->area_d != 0, hdr->sc, l.kernel, l.param, l.flavour, l.ctas_per_sm); }
    };
    std::vector<Pending> pend;
    for (size_t k = 0; k < max_passes; k++) {
        pend.clear();
        for (size_t i = 0; i < items.size(); i++) {
            const auto& it = items[i];
            if (it.plan->passes.size() <= k) continue;
            const ImpHostPass& hp = it.plan->passes[k];
            ImpJob jb = make_job(it.plan, t_dev, k, it.src, it.sp, it.dst, it.dp, scratch, off[i]);
            const ImpLaunch l = pick_launch(hp, jb.src, jb.src_pitch);
            if (uses_tmap(l.kernel)) { int rc = encode_job_tmap(hp.hdr, jb, tmaps); if (rc) return rc; }
            pend.push_back(Pending{&hp.hdr, l, jb, reinterpret_cast<uint16_t*>(scratch + boff[i][k])});
        }
        std::stable_sort(pend.begin(), pend.end(), [](const Pending& a, const Pending& c) { return a.key() < c.key(); });
        for (size_t s = 0, e; s < pend.size(); s = e) {
            const bool generic = pend[s].l.kernel == ImpKernel::BlurGeneric;
            for (e = s + 1; e < pend.size() && !generic && pend[e].key() == pend[s].key(); e++) {}
            imp_gpu_batch::Step st{};
            st.g = ImpLaunchGroup{pend[s].hdr->kind, pend[s].hdr->sc, pend[s].l.kernel, pend[s].l.param, pend[s].l.flavour, (int)jobs.size(), (int)(e - s), 0, 0,
                                  pend[s].hdr->area_d != 0};
            if (generic) { st.hdr = *pend[s].hdr; st.plane = pend[s].plane; }
            for (size_t j = s; j < e; j++) {
                st.g.ctas = std::max(st.g.ctas, pend[j].l.ctas_per_job);
                st.g.smem_bytes = std::max(st.g.smem_bytes, pend[j].l.smem_bytes);
                jobs.push_back(pend[j].job);
            }
            steps.push_back(st);
        }
    }
    return IMP_OK;
}

// d_jobs: the device copy of `jobs`; a group of one job takes it by value instead (kernel parameter).
int launch_steps(const std::vector<imp_gpu_batch::Step>& steps, const std::vector<ImpJob>& jobs, const ImpJob* d_jobs, cudaStream_t st) {
    for (const auto& s : steps) {
        if (s.g.kernel == ImpKernel::BlurGeneric) CK(imp_launch_blur_generic(jobs[s.g.first], s.hdr, s.plane, s.g.smem_bytes, st));
        else if (s.g.count == 1) { ImpLaunchGroup g = s.g; g.first = 0; CK(imp_launch_group(g, nullptr, &jobs[s.g.first], st)); }
        else CK(imp_launch_group(s.g, d_jobs, nullptr, st));
    }
    return IMP_OK;
}

// `up`: the stream the job table is uploaded on (the stream the launches follow on). Nothing here blocks unless a buffer
// has to grow or the previous table of this batch is still being copied out of the pinned staging.
int batch_compile(imp_gpu_batch* b, cudaStream_t up) {
    b->dev = t_dev;
    b->algo_bytes = 0; b->launches = 0;
    for (const auto& it : b->items) {
        int rc = plan_to_device(it.plan);
        if (rc) return rc;
        if ((rc = plan_wait_ready(it.plan, up))) return rc;
        b->algo_bytes += it.plan->algo_bytes;
    }
    auto grow = [b](size_t bytes, uint8_t** p) { int rc = b->scratch.grow(bytes, false); *p = b->scratch.p; return rc; };
    if (int rc = build_steps(b->items, grow, &b->tmaps, b->steps, b->h_jobs)) return rc;
    b->table_needed = false;
    for (const auto& st : b->steps) {
        b->launches += st.g.kernel == ImpKernel::BlurGeneric ? 2 : 1;
        if (st.g.count > 1) b->table_needed = true;
    }
    if (b->table_needed) {
        if (b->h_jobs.size() > b->jobs_cap) {
            if (b->d_jobs) CK(cudaFree(b->d_jobs));
            b->d_jobs = nullptr; b->jobs_cap = 0;
            const size_t cap = b->h_jobs.size() * 5 / 4 + 16;
            CK(cudaMalloc((void**)&b->d_jobs, cap * sizeof(ImpJob)));
            b->jobs_cap = cap;
        }
        const size_t bytes = b->h_jobs.size() * sizeof(ImpJob);
        if (b->up_pending) { CK(cudaEventSynchronize(b->up_ev)); b->up_pending = false; }
        int rc = b->h_pin.grow(bytes, true); if (rc) return rc;
        memcpy(b->h_pin.p, b->h_jobs.data(), bytes);
        CK(cudaMemcpyAsync(b->d_jobs, b->h_pin.p, bytes, cudaMemcpyHostToDevice, up));
        if (!b->up_ev) CK(cudaEventCreateWithFlags(&b->up_ev, cudaEventDisableTiming));
        CK(cudaEventRecord(b->up_ev, up));
        b->up_pending = true;
    }
    b->dirty = false;
    return IMP_OK;
}

void batch_release(imp_gpu_batch* b) {          // device/pinned memory of a batch (its device must be current)
    if (b->d_jobs) cudaFree(b->d_jobs);
    b->d_jobs = nullptr; b->jobs_cap = 0;
    b->scratch.release(false); b->h_pin.release(true);
    if (b->up_ev) cudaEventDestroy(b->up_ev);
    b->up_ev = nullptr; b->up_pending = false;
}


// ---- the chunked end-to-end path over host buffers ---------------------------------------------------------------------
// Requests are cut into CHUNKS of consecutive jobs (imp_chunk_bounds); a chunk owns one lane (stream + staging) while it is
// in flight: H2D of every window, ONE launch per (pass, kernel choice) over the whole chunk through a device job table (the
// path the device-resident batches take), D2H of every result. Lanes rotate, so the copies of chunk k+1 overlap the kernels
// of chunk k and the D2H of chunk k-1 (PCIe is full duplex). How each job's bytes travel is imp_chunk_layout's choice.
// What comes back: the frames, or one more launch per chunk reduces the results on the device and only the answers come
// back (ImpResult::Brightness, ::Ascii).

bool is_pinned(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

// Host-side copies between pageable frames and the pinned staging run on several cores at once: one core moves 4-10 GB/s
// (page-granular source, TLB-bound), a fraction of the link. stage_threads(): the most threads one copy is split over
// (IMP_GPU_STAGE_THREADS, default 8 or half the cores if fewer); a copy gets one thread per 2 MB up to that.
int stage_threads() {
    static const int v = [] {
        const char* e = getenv("IMP_GPU_STAGE_THREADS");
        int n = e ? atoi(e) : 0;
        if (n <= 0) { const unsigned hc = std::thread::hardware_concurrency(); n = (int)std::min<unsigned>(8u, std::max<unsigned>(1u, hc / 2)); }
        return std::max(1, std::min(n, 32));
    }();
    return v;
}
int stage_parts(size_t bytes, int items) {
    return (int)std::max<size_t>(1, std::min<size_t>({(size_t)stage_threads(), bytes >> 20, (size_t)std::max(items, 1)}));
}
// The big host-side copies (pageable frame -> pinned staging, pinned staging -> pageable result) use streaming stores: the
// destination is written once and not read by this core again, so it need not be read into the cache first as a plain
// memcpy's write-allocate does — on the B200 box one request's 29 MB window went from 2.4 to 1.2 ms, a 64-request batch
// from 29 to 42 GB/s.
void copy_stream(uint8_t* dst, const uint8_t* src, size_t n) {
#if defined(__SSE2__)
    if (n >= 4096) {
        const size_t head = (16 - (reinterpret_cast<uintptr_t>(dst) & 15)) & 15;
        if (head) { memcpy(dst, src, head); dst += head; src += head; n -= head; }
        const size_t v = n >> 6;
        for (size_t i = 0; i < v; i++) {
            const __m128i a = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src + 64 * i)), b = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src + 64 * i + 16));
            const __m128i c = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src + 64 * i + 32)), d = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src + 64 * i + 48));
            _mm_stream_si128(reinterpret_cast<__m128i*>(dst + 64 * i), a); _mm_stream_si128(reinterpret_cast<__m128i*>(dst + 64 * i + 16), b);
            _mm_stream_si128(reinterpret_cast<__m128i*>(dst + 64 * i + 32), c); _mm_stream_si128(reinterpret_cast<__m128i*>(dst + 64 * i + 48), d);
        }
        _mm_sfence();
        if (n & 63) memcpy(dst + (v << 6), src + (v << 6), n & 63);
        return;
    }
#endif
    memcpy(dst, src, n);
}
// `rows` rows of `row_bytes`: one copy when both sides are dense, else row by row
void copy_rows(uint8_t* dst, size_t dst_step, const uint8_t* src, size_t src_step, size_t row_bytes, int rows) {
    if (dst_step == row_bytes && src_step == row_bytes) copy_stream(dst, src, row_bytes * rows);
    else for (int y = 0; y < rows; y++) copy_stream(dst + (size_t)y * dst_step, src + (size_t)y * src_step, row_bytes);
}
// The copy workers: a small persistent pool (spawning threads per copy costs ~50 us each, more than a 2 MB slice takes).
// Created on first use — after nginx has forked its workers — and again in a child should a process fork later.
class CopyPool {
    std::mutex mu; std::condition_variable cv;
    std::deque<std::function<void()>> q;
    std::vector<std::thread> th;
    bool stop = false; pid_t owner = 0;
    // after a fork() the handles name threads that do not exist in this process: they are set aside, never joined or detached
    void abandon() { if (!th.empty()) new std::vector<std::thread>(std::move(th)); th.clear(); }
    void work() {
        for (;;) {
            std::function<void()> f;
            {
                std::unique_lock<std::mutex> lk(mu);
                cv.wait(lk, [&] { return stop || !q.empty(); });
                if (q.empty()) return;
                f = std::move(q.front()); q.pop_front();
            }
            f();
        }
    }
public:
    int ensure(int n) {                      // number of workers available (0: run inline)
        std::lock_guard<std::mutex> lk(mu);
        if (owner != getpid()) { abandon(); q.clear(); owner = getpid(); }   // threads do not cross fork()
        while ((int)th.size() < n) {
            try { th.emplace_back([this] { work(); }); } catch (...) { break; }
        }
        return (int)th.size();
    }
    void submit(std::function<void()> f) {
        { std::lock_guard<std::mutex> lk(mu); q.push_back(std::move(f)); }
        cv.notify_one();
    }
    void shutdown() {
        std::vector<std::thread> old;
        { std::lock_guard<std::mutex> lk(mu); if (owner != getpid()) abandon(); stop = true; old.swap(th); }
        cv.notify_all();
        for (std::thread& t : old) if (t.joinable()) t.join();
        std::lock_guard<std::mutex> lk(mu); stop = false;
    }
};
// never destroyed: its threads may outlive main() when the host does not call imp_gpu_shutdown (joinable std::thread destructors abort)
CopyPool& g_copy_pool = *new CopyPool;

// fn(i0, i1) over [0, n) cut into `parts` contiguous ranges: the first on the calling thread, the others on the pool
template <class F> void run_parts(int n, int parts, F fn) {
    if (parts > 1) parts = std::min(parts, g_copy_pool.ensure(stage_threads() - 1) + 1);
    if (parts <= 1 || n < parts) { fn(0, n); return; }
    struct Latch { std::mutex m; std::condition_variable c; int left; } latch;
    latch.left = parts - 1;
    for (int t = 1; t < parts; t++) {
        const int i0 = (int)((long long)n * t / parts), i1 = (int)((long long)n * (t + 1) / parts);
        try {
            g_copy_pool.submit([&latch, &fn, i0, i1] {
                fn(i0, i1);
                std::lock_guard<std::mutex> lk(latch.m);
                if (--latch.left == 0) latch.c.notify_one();
            });
        } catch (...) {                        // no memory for the task: this range runs here; the latch must not be left waiting
            fn(i0, i1);
            std::lock_guard<std::mutex> lk(latch.m);
            --latch.left;
        }
    }
    fn(0, (int)((long long)n / parts));
    std::unique_lock<std::mutex> lk(latch.m);
    latch.c.wait(lk, [&] { return latch.left == 0; });
}

int lane_finish(Lane& L) {
    if (!L.busy) return IMP_OK;
    cudaError_t e = cudaStreamSynchronize(L.st);
    if (e == cudaSuccess) {
        // results for pageable destinations (the frames cvCreateImage hands out) leave the pinned staging here; a 200-frame GIF
        // is 400 MB of it. Big frames one after the other, each frame's rows over the threads; the other results of the
        // chunk (answers whatever their size) shared out whole.
        const uint8_t* h_out = L.h_out.p;
        std::vector<const Lane::Out*> small; size_t small_bytes = 0;
        for (const Lane::Out& o : L.pend) {
            const size_t bytes = o.row_bytes * o.rows;
            if (o.rows == 1 || bytes < (4u << 20)) { small.push_back(&o); small_bytes += bytes; continue; }
            run_parts(o.rows, stage_parts(bytes, o.rows), [&o, h_out](int y0, int y1) {
                copy_rows(o.dst + (size_t)y0 * o.dst_step, o.dst_step, h_out + o.hout_off + y0 * o.row_bytes, o.row_bytes, o.row_bytes, y1 - y0);
            });
        }
        const Lane::Out* const* sm = small.data();
        run_parts((int)small.size(), stage_parts(small_bytes, (int)small.size()), [sm, h_out](int k0, int k1) {
            for (int k = k0; k < k1; k++) copy_rows(sm[k]->dst, sm[k]->dst_step, h_out + sm[k]->hout_off, sm[k]->row_bytes, sm[k]->row_bytes, sm[k]->rows);
        });
    }
    L.pend.clear(); L.busy = false;
    if (e != cudaSuccess) return fail(e, "cudaStreamSynchronize", __LINE__);
    return IMP_OK;
}

// The 256-entry ramps of ASCII (filters.c:486-522), derived with the reference's float maths (filters.c:496,509).
const ImpAsciiRamps& ascii_ramps() {
    static const ImpAsciiRamps r = [] {
        static const char kWide[] = "$@B%8&WM#*oahkbdpqwmZO0QLCJUYXzcvunxrjft/\\|()1{}[]?-_+~<>i!lI;:,\"^`'. ";   // filters.c:486-487
        static const char kNarrow[] = "@%8#*+=-:. ";
        ImpAsciiRamps t;
        for (int wide = 0; wide < 2; wide++) {
            const char* table = wide ? kWide : kNarrow;
            const float factor = 256.0 / (int)strlen(table);
            for (int v = 0; v < 256; v++) t.lut[wide][v] = (uint8_t)table[(int)floor((double)((float)v / factor))];
        }
        return t;
    }();
    return r;
}

// Brightness / ASCII of the chunk's m results (in L.d_out): ONE launch over all of them, then only the answers cross the
// link — straight into pinned destinations, through h_out otherwise (lane_finish copies on).
int lane_answers(Lane& L, const ImpHostJob* jobs, int m, ImpResult kind, const ImpChunkLayout& lay) {
    const bool ascii = kind == ImpResult::Ascii;
    std::vector<ImpInfoJob> tab(m);
    int parts = 0, max_ctas = 1;
    size_t text_total = 0;
    for (int k = 0; k < m; k++) {
        const imp_gpu_plan* p = jobs[k].plan;
        const ImpJobLayout& l = lay.jobs[k];
        ImpInfoJob& q = tab[k];
        q = ImpInfoJob{};
        q.img = L.d_out.p + l.out_off; q.pitch = l.out_pitch;                // 256-byte aligned slot, 16-byte pitch
        q.w = p->out_w; q.h = p->out_h; q.c = p->out_c; q.vec = 1;
        if (ascii) {
            q.ctas = imp_ascii_ctas(q.w, q.h); q.wide = jobs[k].wide ? 1 : 0;
            q.text_off = (long long)text_total; text_total += align256(l.res_bytes);
        } else {
            q.ctas = imp_brightness_ctas(q.w, q.h); q.part_off = parts; parts += q.ctas;
        }
        max_ctas = std::max(max_ctas, q.ctas);
    }
    const size_t tab_bytes = align256(sizeof(ImpInfoJob) * m), part_bytes = align256(sizeof(double) * parts), ans_bytes = align256(sizeof(float) * m);
    int r;
    if ((r = L.d_info.grow(tab_bytes + part_bytes + ans_bytes + text_total, false)) || (r = L.h_info.grow(tab_bytes, true))) return r;
    if (!ascii && !L.d_tickets.p) {
        if ((r = L.d_tickets.grow(sizeof(unsigned) * IMP_CHUNK_JOBS, false))) return r;
        CK(cudaMemsetAsync(L.d_tickets.p, 0, L.d_tickets.cap, L.st));
    }
    memcpy(L.h_info.p, tab.data(), sizeof(ImpInfoJob) * m);
    CK(cudaMemcpyAsync(L.d_info.p, L.h_info.p, sizeof(ImpInfoJob) * m, cudaMemcpyHostToDevice, L.st));
    const ImpInfoJob* d_tab = reinterpret_cast<const ImpInfoJob*>(L.d_info.p);
    uint8_t* d_ans = L.d_info.p + tab_bytes + part_bytes;
    uint8_t* d_text = d_ans + ans_bytes;
    auto dst = [&](int k) { return lay.jobs[k].dst == ImpRoute::Staged ? L.h_out.p + lay.jobs[k].hout_off : jobs[k].dst; };
    if (ascii) CK(imp_launch_ascii(d_tab, tab[0], m, max_ctas, ascii_ramps(), d_text, L.st));
    else CK(imp_launch_brightness(d_tab, tab[0], m, max_ctas, reinterpret_cast<double*>(L.d_info.p + tab_bytes),
                                  reinterpret_cast<unsigned*>(L.d_tickets.p), reinterpret_cast<float*>(d_ans), L.st));
    if (!ascii) CK(cudaMemcpyAsync(dst(0), d_ans, sizeof(float) * m, cudaMemcpyDeviceToHost, L.st));
    for (int k = 0; k < m; k++) {
        const ImpJobLayout& l = lay.jobs[k];
        if (ascii) CK(cudaMemcpyAsync(dst(k), d_text + tab[k].text_off, l.res_bytes, cudaMemcpyDeviceToHost, L.st));
        if (l.dst == ImpRoute::Staged) L.pend.push_back(Lane::Out{jobs[k].dst, l.res_bytes, l.res_bytes, 1, l.hout_off});
    }
    return IMP_OK;
}

// Issues one chunk of m jobs on lane L. The order on the lane's stream: every upload in job order, the up_done record, the
// window extractions (a kernel never sits between two copies of the stream and idles the copy engine), the grouped
// launches, then the answer launch or the downloads.
int lane_issue(Lane& L, const ImpHostJob* jobs, int m, ImpResult kind, bool resident) {
    std::unique_ptr<bool[]> pinned(new bool[2 * (size_t)m]);
    bool* src_pinned = pinned.get(); bool* dst_pinned = src_pinned + m;
    for (int k = 0; k < m; k++) {
        src_pinned[k] = resident || is_pinned(jobs[k].src);
        dst_pinned[k] = is_pinned(jobs[k].dst);
    }
    const ImpChunkLayout lay = imp_chunk_layout(jobs, m, kind, resident, src_pinned, dst_pinned);
    int r;
    if ((r = L.d_in.grow(lay.in_total, false)) || (r = L.d_out.grow(lay.out_total, false)) || (r = L.d_stage.grow(lay.stage_total, false)) ||
        (r = L.h_in.grow(lay.hin_total, true)) || (r = L.h_out.grow(lay.hout_total, true))) return r;
    L.busy = true;
    imp_gpu_batch& B = L.batch;
    B.items.clear(); B.dirty = true;
    struct Repitch { const uint8_t* src; int sp; uint8_t* dst; int dp, row_bytes, rows; };
    std::vector<Repitch> repitch;
    for (int k = 0; k < m; k++) {
        const ImpHostJob& j = jobs[k];
        const ImpJobLayout& l = lay.jobs[k];
        imp_gpu_plan* p = j.plan;
        const int sc = p->src_c;
        const size_t in_row = (size_t)p->win_w * sc;
        uint8_t* d_in = L.d_in.p + l.in_off;
        uint8_t* d_out = L.d_out.p + l.out_off;
        const uint8_t* rows = j.src + (size_t)p->win_y * j.src_step;          // the rows the crop window touches
        switch (l.src) {
        case ImpRoute::Resident:
            B.items.push_back(imp_gpu_batch::Item{p, j.src, j.src_step, d_out, l.out_pitch});
            continue;
        case ImpRoute::Staged: {
            // a pageable frame (what cvDecodeImage hands RunJob) goes through the lane's pinned staging, laid out with the
            // device pitch, by several cores at once (stage_threads above), in row slices each uploaded once staged
            uint8_t* h = L.h_in.p + l.hin_off;
            const uint8_t* win = rows + (size_t)p->win_x * sc;
            for (int s = 0; s < l.slices; s++) {
                const int r0 = (int)((long long)p->win_h * s / l.slices), r1 = (int)((long long)p->win_h * (s + 1) / l.slices);
                run_parts(r1 - r0, stage_parts(in_row * (size_t)(r1 - r0), r1 - r0), [=, &j](int y0, int y1) {
                    copy_rows(h + (size_t)(r0 + y0) * l.in_pitch, l.in_pitch, win + (size_t)(r0 + y0) * j.src_step, j.src_step, in_row, y1 - y0);
                });
                CK(cudaMemcpyAsync(d_in + (size_t)r0 * l.in_pitch, h + (size_t)r0 * l.in_pitch, (size_t)l.in_pitch * (r1 - r0), cudaMemcpyHostToDevice, L.st));
            }
            break;
        }
        case ImpRoute::Linear:
            CK(cudaMemcpyAsync(d_in, rows, l.lin_bytes, cudaMemcpyHostToDevice, L.st));
            break;
        case ImpRoute::LinearRepitch: {
            uint8_t* stage = L.d_stage.p + l.stage_off;
            CK(cudaMemcpyAsync(stage, rows, l.lin_bytes, cudaMemcpyHostToDevice, L.st));
            repitch.push_back(Repitch{stage + (size_t)p->win_x * sc, j.src_step, d_in, l.in_pitch, (int)in_row, p->win_h});
            break;
        }
        default:                                                               // Rows2D
            CK(cudaMemcpy2DAsync(d_in, l.in_pitch, rows + (size_t)p->win_x * sc, j.src_step, in_row, p->win_h, cudaMemcpyHostToDevice, L.st));
        }
        // The device copy holds only the crop window; bias the base pointer so the pass's (sx0,sy0) lands on it.
        const uint8_t* biased = d_in - ((size_t)p->win_y * l.in_pitch + (size_t)p->win_x * sc);
        B.items.push_back(imp_gpu_batch::Item{p, biased, l.in_pitch, d_out, l.out_pitch});
    }
    if (L.up_done) CK(cudaEventRecord(L.up_done, L.st));
    for (const Repitch& q : repitch) CK(imp_launch_repitch(q.src, q.sp, q.dst, q.dp, q.row_bytes, q.rows, L.st));
    if ((r = batch_compile(&B, L.st))) return r;
    if ((r = launch_steps(B.steps, B.h_jobs, B.d_jobs, L.st))) return r;
    if (kind != ImpResult::Frame) return lane_answers(L, jobs, m, kind, lay);
    for (int k = 0; k < m; k++) {
        const ImpHostJob& j = jobs[k];
        const ImpJobLayout& l = lay.jobs[k];
        const imp_gpu_plan* p = j.plan;
        const size_t out_row = (size_t)p->out_w * p->out_c;
        const uint8_t* d_out = L.d_out.p + l.out_off;
        if (l.dst == ImpRoute::Linear) CK(cudaMemcpyAsync(j.dst, d_out, (size_t)l.out_pitch * (p->out_h - 1) + out_row, cudaMemcpyDeviceToHost, L.st));
        else if (l.dst == ImpRoute::Rows2D) CK(cudaMemcpy2DAsync(j.dst, j.dst_step, d_out, l.out_pitch, out_row, p->out_h, cudaMemcpyDeviceToHost, L.st));
        else {
            CK(cudaMemcpy2DAsync(L.h_out.p + l.hout_off, out_row, d_out, l.out_pitch, out_row, p->out_h, cudaMemcpyDeviceToHost, L.st));
            L.pend.push_back(Lane::Out{j.dst, (size_t)j.dst_step, out_row, p->out_h, l.hout_off});
        }
    }
    return IMP_OK;
}

// Runs jobs [0, n) over n_streams lanes of the current device. `resident`: the sources are already on the device;
// `after`: an event every lane waits for before its first chunk (their producer). Caller holds run_mu.
int run_host_chunked_locked(const ImpHostJob* jobs, int n, ImpResult kind, int n_streams, bool resident, cudaEvent_t after) {
    DevCtx& ctx = g_dev[t_dev];
    n_streams = std::max(1, std::min(n_streams, 8));
    while ((int)ctx.lanes.size() < n_streams) {
        Lane* L = new (std::nothrow) Lane();
        if (!L) return IMP_ERROR_MALLOC_FAILED;
        cudaError_t e = cudaStreamCreateWithFlags(&L->st, cudaStreamNonBlocking);
        if (e != cudaSuccess) { delete L; return fail(e, "cudaStreamCreateWithFlags", __LINE__); }
        e = cudaEventCreateWithFlags(&L->up_done, cudaEventDisableTiming);
        if (e != cudaSuccess) { cudaStreamDestroy(L->st); delete L; return fail(e, "cudaEventCreateWithFlags", __LINE__); }
        ctx.lanes.push_back(L);
    }
    if (after) for (int k = 0; k < n_streams; k++) CK(cudaStreamWaitEvent(ctx.lanes[k]->st, after, 0));
    int result = IMP_OK;
    try {
        const std::vector<int> bounds = imp_chunk_bounds(jobs, n, n_streams);
        Lane* prev = nullptr;
        for (size_t c = 0; c + 1 < bounds.size() && result == IMP_OK; c++) {
            Lane& L = *ctx.lanes[c % n_streams];
            if ((result = lane_finish(L))) break;
            // each chunk's uploads wait for the previous chunk's: they run back to back in chunk order (imp_chunk_bounds)
            if (prev && prev != &L && !resident) CK(cudaStreamWaitEvent(L.st, prev->up_done, 0));
            prev = &L;
            result = lane_issue(L, jobs + bounds[c], bounds[c + 1] - bounds[c], kind, resident);
        }
    } catch (const std::bad_alloc&) { result = IMP_ERROR_MALLOC_FAILED; }
    for (Lane* L : ctx.lanes) { int r = lane_finish(*L); if (result == IMP_OK) result = r; }
    return result;
}
int run_host_chunked(const std::vector<ImpHostJob>& jobs, ImpResult kind, int n_streams) {
    if (jobs.empty()) return IMP_OK;
    std::lock_guard<std::mutex> run_lk(g_dev[t_dev].run_mu);
    return run_host_chunked_locked(jobs.data(), (int)jobs.size(), kind, n_streams, false, nullptr);
}

// Every job of a host call is checked before any work starts, so a bad one leaves every output as it was. A packed
// (bottom-up) result would reverse an answer's text, and the JSON and text exits never reach the FreeImage packer.
// text_caps: ASCII only, the capacity of each text.
int check_host_jobs(ImpResult kind, const std::vector<ImpHostJob>& jobs, const long* text_caps = nullptr) {
    for (size_t i = 0; i < jobs.size(); i++) {
        const ImpHostJob& j = jobs[i];
        const imp_gpu_plan* p = j.plan;
        if (!p || !j.src || !j.dst || (long long)j.src_step < (long long)p->src_w * p->src_c) return IMP_ERROR_INVALID_ARGS;
        if (kind == ImpResult::Frame ? (long long)j.dst_step < (long long)p->out_w * p->out_c : p->pack != IMP_PACK_NONE) return IMP_ERROR_INVALID_ARGS;
        if (kind == ImpResult::Ascii && text_caps[i] < imp_gpu_ascii_length(p->out_w, p->out_h)) return IMP_ERROR_INVALID_ARGS;
    }
    return IMP_OK;
}

// The job list of a host call (answers fill in dst themselves).
std::vector<ImpHostJob> host_jobs(int n, imp_gpu_plan* const* plans, const unsigned char* const* srcs, const int* src_steps,
                                  unsigned char* const* dsts = nullptr, const int* dst_steps = nullptr) {
    std::vector<ImpHostJob> v(n);
    for (int i = 0; i < n; i++) v[i] = ImpHostJob{plans[i], srcs[i], src_steps[i], dsts ? dsts[i] : nullptr, dst_steps ? dst_steps[i] : 0, false};
    return v;
}

// The "build and check" halves of the frame, brightness and ASCII calls: the job list the run takes (empty when n <= 0), or
// the code the call refuses with. The synchronous call and its submit both take their jobs from here.
int frame_jobs(int n, imp_gpu_plan* const* plans, const unsigned char* const* srcs, const int* src_steps,
               unsigned char* const* dsts, const int* dst_steps, std::vector<ImpHostJob>& jobs) {
    if (n <= 0) return IMP_OK;
    if (!plans || !srcs || !src_steps || !dsts || !dst_steps) return IMP_ERROR_INVALID_ARGS;
    jobs = host_jobs(n, plans, srcs, src_steps, dsts, dst_steps);
    return check_host_jobs(ImpResult::Frame, jobs);
}
int brightness_jobs(int n, imp_gpu_plan* const* plans, const unsigned char* const* srcs, const int* src_steps, float* brightness,
                    std::vector<ImpHostJob>& jobs) {
    if (n <= 0) return IMP_OK;
    if (!plans || !srcs || !src_steps || !brightness) return IMP_ERROR_INVALID_ARGS;
    jobs = host_jobs(n, plans, srcs, src_steps);
    for (int i = 0; i < n; i++) jobs[i].dst = reinterpret_cast<uint8_t*>(brightness + i);
    return check_host_jobs(ImpResult::Brightness, jobs);
}
int ascii_jobs(int n, imp_gpu_plan* const* plans, const unsigned char* const* srcs, const int* src_steps, const char* const* args,
               unsigned char* const* texts, const long* text_caps, std::vector<ImpHostJob>& jobs) {
    if (n <= 0) return IMP_OK;
    if (!plans || !srcs || !src_steps || !args || !texts || !text_caps) return IMP_ERROR_INVALID_ARGS;
    jobs = host_jobs(n, plans, srcs, src_steps);
    for (int i = 0; i < n; i++) {
        jobs[i].dst = texts[i];
        jobs[i].wide = args[i] && strcmp(args[i], "wide") == 0;                  // filters.c:490-494
    }
    return check_host_jobs(ImpResult::Ascii, jobs, text_caps);
}

// The checks imp_gpu_run_device and imp_gpu_batch_add make on a device job.
int check_device_job(const imp_gpu_plan* plan, const void* d_src, int sp, const void* d_dst, int dp) {
    if (!plan || !d_src || !d_dst) return IMP_ERROR_INVALID_ARGS;
    if (sp < plan->src_w * plan->src_c || dp < plan->out_w * plan->out_c) return IMP_ERROR_INVALID_ARGS;
    if (plan->out_c == 4 && (dp % 4 || ((uintptr_t)d_dst) % 4)) return IMP_ERROR_INVALID_ARGS;
    if (plan->src_c == 4 && (sp % 4 || ((uintptr_t)d_src) % 4)) return IMP_ERROR_INVALID_ARGS;
    return IMP_OK;
}

// How many devices the box has; IMP_ERROR_GPU with the reason when it has none.
int count_devices(int* n) {
    *n = 0;
    cudaError_t e = cudaGetDeviceCount(n);
    if (e != cudaSuccess || *n == 0) {
        *n = 0;
        snprintf(t_err, sizeof t_err, "no CUDA device available (%s); libimp_gpu has no CPU fallback", e == cudaSuccess ? "count == 0" : cudaGetErrorString(e));
        return IMP_ERROR_GPU;
    }
    return IMP_OK;
}

int bad_device_list(const char* spec, int entry, const char* tok, int tok_len, const char* why) {
    snprintf(t_err, sizeof t_err, "device list \"%s\": entry %d (\"%.*s\") %s", spec, entry, std::min(tok_len, 64), tok, why);
    return IMP_ERROR_INVALID_ARGS;
}

// Which devices this process may use, in order: the one parser of IMP_GPU_DEVICES (the worker mapping and the farm both
// read the list through here). `spec` NULL or empty: 0 .. n_devices-1, at most MAX_DEV of them. Otherwise comma-separated
// decimal ordinals, each below n_devices and MAX_DEV, none twice, at most MAX_DEV entries; anything else is
// IMP_ERROR_INVALID_ARGS with the offending entry in t_err.
int device_list(const char* spec, int n_devices, int* list, int* len) {
    *len = 0;
    if (n_devices <= 0) return fail_msg("no CUDA device to choose from (0 devices); libimp_gpu has no CPU fallback");
    if (!spec || !*spec) {
        for (int d = 0; d < std::min(n_devices, MAX_DEV); d++) list[(*len)++] = d;
        return IMP_OK;
    }
    for (const char* p = spec;; p++) {
        const char* tok = p;
        const int entry = *len + 1;
        long v = 0;
        for (; *p >= '0' && *p <= '9'; p++) v = std::min(v * 10 + (*p - '0'), 1000000L);
        if (*p && *p != ',') {
            while (*p && *p != ',') p++;
            return bad_device_list(spec, entry, tok, (int)(p - tok), "is not a decimal device ordinal");
        }
        const int tok_len = (int)(p - tok);
        if (tok_len == 0) return bad_device_list(spec, entry, tok, 0, "is empty");
        if (*len == MAX_DEV) return bad_device_list(spec, entry, tok, tok_len, "is past the 16 entries a list may hold");
        if (v >= n_devices) {
            char why[48];
            snprintf(why, sizeof why, "names no device: %d present", n_devices);
            return bad_device_list(spec, entry, tok, tok_len, why);
        }
        if (v >= MAX_DEV) return bad_device_list(spec, entry, tok, tok_len, "is beyond device 15, the last libimp_gpu drives");
        for (int k = 0; k < *len; k++)
            if (list[k] == v) return bad_device_list(spec, entry, tok, tok_len, "names a device already listed");
        list[(*len)++] = (int)v;
        if (!*p) return IMP_OK;
    }
}

}  // namespace

// A host call in flight: what its "build and check" half captured, and its "run" half, which a helper thread applies to
// that on the device the caller had current at the submit.
struct imp_gpu_ticket {
    std::thread th;
    int rc = IMP_OK; std::string err;
    std::atomic<bool> done{false};
    std::vector<ImpHostJob> jobs;                        // each plan holds one more reference until the wait
    std::function<int(std::vector<ImpHostJob>&)> run;
};

namespace {

// Every submit ends here once its call's checks have passed: the ticket takes the job list and the run, and the helper
// thread starts. Nothing throws out of it; an allocation that fails leaves no ticket and no extra plan reference.
int start_ticket(std::vector<ImpHostJob> jobs, std::function<int(std::vector<ImpHostJob>&)> run, imp_gpu_ticket** ticket) {
    imp_gpu_ticket* t = nullptr;
    bool held = false;
    try {
        t = new imp_gpu_ticket();
        t->jobs = std::move(jobs); t->run = std::move(run);
        for (const ImpHostJob& j : t->jobs) j.plan->refs.fetch_add(1);       // the call keeps its plans alive
        held = true;
        const int dev = t_dev;
        t->th = std::thread([t, dev]() {
            int r = imp_gpu_set_device(dev);
            if (r == IMP_OK) {
                try { r = t->run(t->jobs); } catch (const std::bad_alloc&) { r = IMP_ERROR_MALLOC_FAILED; }
            }
            t->rc = r;
            if (r) t->err = t_err;
            t->done.store(true, std::memory_order_release);
        });
    } catch (...) {
        if (t) { if (held) for (const ImpHostJob& j : t->jobs) plan_release(j.plan); delete t; }
        return IMP_ERROR_MALLOC_FAILED;
    }
    *ticket = t;
    return IMP_OK;
}

// The "run" half of the frame, brightness and ASCII calls.
std::function<int(std::vector<ImpHostJob>&)> chunked_run(ImpResult kind, int n_streams) {
    return [kind, n_streams](std::vector<ImpHostJob>& jobs) { return run_host_chunked(jobs, kind, n_streams); };
}

}  // namespace

extern "C" {

int imp_gpu_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int imp_gpu_init(int device) {
    if (device < 0 || device >= MAX_DEV) return fail_msg("imp_gpu_init: device index out of range");
    int n = 0;
    if (int rc = count_devices(&n)) return rc;
    if (device >= n) return fail_msg("imp_gpu_init: no such device");
    CK(cudaSetDevice(device));
    {
        std::lock_guard<std::mutex> lk(g_mu);
        DevCtx& c = g_dev[device];
        if (!c.ready) {
            cudaDeviceProp prop;
            CK(cudaGetDeviceProperties(&prop, device));
            if (prop.major != 10) {
                snprintf(t_err, sizeof t_err, "device %d is sm_%d%d; libimp_gpu is built for sm_100a only", device, prop.major, prop.minor);
                return IMP_ERROR_GPU;
            }
            CK(cudaFree(0));
            CK(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
            CK(cudaEventCreateWithFlags(&c.up_ev, cudaEventDisableTiming));
            // stream-ordered allocations (plan arenas, per-call scratch) keep their memory in the pool instead of going
            // back to the driver at every synchronisation
            cudaMemPool_t pool;
            if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
                unsigned long long keep = ~0ull;
                cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
                // prime the pool: the first plans of a worker then sub-allocate instead of mapping fresh memory
                void* prime = nullptr;
                if (cudaMallocAsync(&prime, 32u << 20, c.stream) == cudaSuccess) cudaFreeAsync(prime, c.stream);
                else cudaGetLastError();
            }
            CK(imp_upload_tables());
            c.ready = true;
        }
    }
    t_dev = device;
    return IMP_OK;
}

// Pure host logic, like imp_gpu_farm_assign: testable without a device.
int imp_gpu_worker_device(int worker, int n_devices, const char* devices, int* device) {
    if (!device) return IMP_ERROR_INVALID_ARGS;
    *device = -1;
    if (worker < 0) { snprintf(t_err, sizeof t_err, "worker index %d is negative", worker); return IMP_ERROR_INVALID_ARGS; }
    int list[MAX_DEV], len = 0;
    if (int rc = device_list(devices, n_devices, list, &len)) return rc;
    *device = list[worker % len];
    return IMP_OK;
}

int imp_gpu_init_worker(int worker, int* device) {
    if (device) *device = -1;
    int n = 0, d = -1, rc = count_devices(&n);
    if (rc == IMP_OK) rc = imp_gpu_worker_device(worker, n, getenv("IMP_GPU_DEVICES"), &d);
    if (rc == IMP_OK) rc = imp_gpu_init(d);
    if (rc == IMP_OK && device) *device = d;
    return rc;
}

int imp_gpu_set_device(int device) {
    if (device < 0 || device >= MAX_DEV) return fail_msg("imp_gpu_set_device: device index out of range");
    if (!g_dev[device].ready) { int rc = imp_gpu_init(device); if (rc) return rc; }
    t_dev = device;
    CK(cudaSetDevice(device));
    return IMP_OK;
}

void imp_gpu_shutdown(void) {
    g_copy_pool.shutdown();
    cache_clear();                     // cached plans and registered overlays go first: their device memory is still reachable
    imp_wm_registry_clear();
    std::lock_guard<std::mutex> lk(g_mu);
    for (int d = 0; d < MAX_DEV; d++) {
        DevCtx& c = g_dev[d];
        if (!c.ready) continue;
        if (cudaSetDevice(d) == cudaSuccess) {
            cudaDeviceSynchronize();
            for (Lane* L : c.lanes) {
                L->d_in.release(false); L->d_out.release(false); L->d_stage.release(false);
                L->h_in.release(true); L->h_out.release(true);
                L->d_info.release(false); L->h_info.release(true); L->d_tickets.release(false);
                batch_release(&L->batch);
                if (L->up_done) cudaEventDestroy(L->up_done);
                if (L->st) cudaStreamDestroy(L->st);
                delete L;
            }
            c.lanes.clear();
            c.h_up.release(true);
            c.h_gif.release(true); c.d_gif.release(false); c.d_canvas.release(false);
            if (c.gif_ev) { cudaEventDestroy(c.gif_ev); c.gif_ev = nullptr; }
            if (c.up_ev) cudaEventDestroy(c.up_ev);
            if (c.stream) cudaStreamDestroy(c.stream);
        }
        c.stream = nullptr; c.up_ev = nullptr; c.up_pending = false; c.ready = false;
    }
    t_dev = -1;
}

const char* imp_gpu_last_error(void) { return t_err; }
unsigned imp_gpu_debug_flags(void) {
    if (bind() != IMP_OK) return 0;
    cudaDeviceSynchronize();
    return imp_debug_flags_kernels() | imp_debug_flags_strip() | imp_debug_flags_blur() | imp_debug_flags_cubic() | imp_debug_flags_gather();
}
unsigned long long imp_gpu_launch_count(void) { return imp_launches(); }

// ---- overlays -------------------------------------------------------------------------------------------
int imp_gpu_upload_watermark(const imp_gpu_watermark* wm) {
    int rc = bind(); if (rc) return rc;
    if (!wm || !wm->pixels || wm->width <= 0 || wm->height <= 0 || (wm->channels != 3 && wm->channels != 4) || wm->step < wm->width * wm->channels)
        return IMP_ERROR_NO_SUCH_WATERMARK;
    try {
        std::shared_ptr<ImpWmImage> img = imp_wm_intern(wm);
        std::lock_guard<std::mutex> lk(g_mu);
        return wm_to_device(img.get(), t_dev);
    } catch (const std::bad_alloc&) { return IMP_ERROR_MALLOC_FAILED; }
}

// ---- plans ---------------------------------------------------------------------------------------------
int imp_gpu_plan_create(const imp_gpu_request* req, const imp_gpu_config* cfg, int w, int h, int c, imp_gpu_plan** out, int* step) {
    if (out) *out = nullptr;
    if (!out) return IMP_ERROR_INVALID_ARGS;
    imp_gpu_plan* p = nullptr;
    try {
        std::string key;
        const bool cacheable = g_cache.cap > 0 && req && w > 0 && h > 0 && req->filter_count >= 0 && (req->filter_count == 0 || req->filters);
        if (cacheable) {
            std::shared_ptr<ImpWmImage> wm;
            const imp_gpu_watermark* m = cfg ? cfg->watermark : nullptr;
            if (m && m->pixels && m->width > 0 && m->height > 0 && (m->channels == 3 || m->channels == 4)) wm = imp_wm_intern(m);
            key = plan_key(req, cfg, w, h, c, wm.get());
            std::lock_guard<std::mutex> lk(g_cache.mu);
            auto it = g_cache.map.find(key);
            if (it != g_cache.map.end()) {
                g_cache.lru.splice(g_cache.lru.begin(), g_cache.lru, it->second);
                imp_gpu_plan* hit = it->second->second;
                hit->refs.fetch_add(1);
                g_cache.hits++;
                if (step) *step = IMP_STEP_ENCODE;
                *out = hit;
                return IMP_OK;
            }
            g_cache.misses++;
        }
        p = new imp_gpu_plan();
        int rc = imp_build_plan(req, cfg, w, h, c, p, step);
        if (rc) { delete p; return rc; }
        if (cacheable) {
            imp_gpu_plan* evicted = nullptr;
            {
                std::lock_guard<std::mutex> lk(g_cache.mu);
                if (g_cache.map.find(key) == g_cache.map.end()) {
                    p->refs.fetch_add(1);                              // the cache's reference
                    g_cache.lru.emplace_front(key, p);
                    g_cache.map[key] = g_cache.lru.begin();
                    if (g_cache.lru.size() > g_cache.cap) {
                        evicted = g_cache.lru.back().second;
                        g_cache.map.erase(g_cache.lru.back().first);
                        g_cache.lru.pop_back();
                    }
                }
            }
            if (evicted) plan_release(evicted);
        }
    } catch (const std::bad_alloc&) {
        delete p; return IMP_ERROR_MALLOC_FAILED;
    } catch (...) {
        delete p; return IMP_ERROR_INVALID_ARGS;
    }
    *out = p;
    return IMP_OK;
}

void imp_gpu_plan_destroy(imp_gpu_plan* plan) { plan_release(plan); }

void imp_gpu_plan_cache_stats(unsigned long long* hits, unsigned long long* misses, int* entries) {
    std::lock_guard<std::mutex> lk(g_cache.mu);
    if (hits) *hits = g_cache.hits; if (misses) *misses = g_cache.misses; if (entries) *entries = (int)g_cache.lru.size();
}
void imp_gpu_plan_cache_clear(void) { cache_clear(); }

void imp_gpu_plan_output(const imp_gpu_plan* p, int* w, int* h, int* c) {
    if (w) *w = p->out_w; if (h) *h = p->out_h; if (c) *c = p->out_c;
}
void imp_gpu_plan_source_window(const imp_gpu_plan* p, int* x, int* y, int* w, int* h) {
    if (x) *x = p->win_x; if (y) *y = p->win_y; if (w) *w = p->win_w; if (h) *h = p->win_h;
}
int imp_gpu_plan_passes(const imp_gpu_plan* p) { return (int)p->passes.size(); }
unsigned long long imp_gpu_plan_algorithmic_bytes(const imp_gpu_plan* p) { return p->algo_bytes; }

// ---- batches -------------------------------------------------------------------------------------------
int imp_gpu_batch_create(imp_gpu_batch** out) {
    if (!out) return IMP_ERROR_INVALID_ARGS;
    *out = new (std::nothrow) imp_gpu_batch();
    return *out ? IMP_OK : IMP_ERROR_MALLOC_FAILED;
}
void imp_gpu_batch_destroy(imp_gpu_batch* b) {
    if (!b) return;
    if (b->dev >= 0 && cudaSetDevice(b->dev) == cudaSuccess) {
        batch_release(b);
        if (t_dev >= 0) cudaSetDevice(t_dev);
    }
    delete b;
}
int imp_gpu_batch_clear(imp_gpu_batch* b) { b->items.clear(); b->dirty = true; return IMP_OK; }
int imp_gpu_batch_size(const imp_gpu_batch* b) { return (int)b->items.size(); }
unsigned long long imp_gpu_batch_algorithmic_bytes(const imp_gpu_batch* b) { return b->algo_bytes; }
int imp_gpu_batch_launches_per_run(const imp_gpu_batch* b) { return b->launches; }

int imp_gpu_batch_add(imp_gpu_batch* b, imp_gpu_plan* plan, const void* d_src, int sp, void* d_dst, int dp) {
    if (!b) return IMP_ERROR_INVALID_ARGS;
    if (int rc = check_device_job(plan, d_src, sp, d_dst, dp)) return rc;
    try { b->items.push_back(imp_gpu_batch::Item{plan, (const uint8_t*)d_src, sp, (uint8_t*)d_dst, dp}); }
    catch (...) { return IMP_ERROR_MALLOC_FAILED; }
    b->dirty = true;
    return IMP_OK;
}

int imp_gpu_batch_launch(imp_gpu_batch* b, void* stream) {
    int rc = bind(); if (rc) return rc;
    if (!b) return IMP_ERROR_INVALID_ARGS;
    if (b->items.empty()) return IMP_OK;
    cudaStream_t st = pick_stream(stream);
    if (b->dirty || b->dev != t_dev) {
        try { rc = batch_compile(b, st); } catch (const std::bad_alloc&) { return IMP_ERROR_MALLOC_FAILED; }
        if (rc) return rc;
    }
    return launch_steps(b->steps, b->h_jobs, b->d_jobs, st);
}

// ---- one frame -----------------------------------------------------------------------------------------
int imp_gpu_run_device(imp_gpu_plan* plan, const void* d_src, int sp, void* d_dst, int dp, void* stream) {
    int rc = bind(); if (rc) return rc;
    if ((rc = check_device_job(plan, d_src, sp, d_dst, dp))) return rc;
    if ((rc = plan_to_device(plan))) return rc;
    cudaStream_t st = pick_stream(stream);
    if ((rc = plan_wait_ready(plan, st))) return rc;
    // the batch's steps over this one frame: every group holds one job, passed by value (no device job table)
    uint8_t* scratch = nullptr;
    auto alloc = [&](size_t bytes, uint8_t** p) {
        if (bytes) CK(cudaMallocAsync((void**)&scratch, bytes, st));      // stream-ordered: stays asynchronous
        *p = scratch;
        return IMP_OK;
    };
    std::vector<imp_gpu_batch::Step> steps;
    std::vector<ImpJob> jobs;
    try { rc = build_steps({imp_gpu_batch::Item{plan, (const uint8_t*)d_src, sp, (uint8_t*)d_dst, dp}}, alloc, nullptr, steps, jobs); }
    catch (const std::bad_alloc&) { rc = IMP_ERROR_MALLOC_FAILED; }
    if (!rc) rc = launch_steps(steps, jobs, nullptr, st);
    if (scratch) CK(cudaFreeAsync(scratch, st));
    return rc;
}

int imp_gpu_run_host(imp_gpu_plan* plan, const unsigned char* src, int src_step, unsigned char* dst, int dst_step) {
    if (!plan || !src || !dst) return IMP_ERROR_INVALID_ARGS;
    imp_gpu_plan* plans[1] = {plan};
    const unsigned char* srcs[1] = {src}; unsigned char* dsts[1] = {dst};
    int ss[1] = {src_step}, ds[1] = {dst_step};
    return imp_gpu_batch_run_host(1, plans, srcs, ss, dsts, ds, 1);
}

// End to end over host buffers (see run_host_chunked above). Only the crop window of a frame travels; a host pointer
// that is not page-locked goes through the lane's pinned staging.
int imp_gpu_batch_run_host(int n, imp_gpu_plan* const* plans, const unsigned char* const* srcs, const int* src_steps,
                           unsigned char* const* dsts, const int* dst_steps, int n_streams) {
    int rc = bind(); if (rc) return rc;
    try {
        std::vector<ImpHostJob> jobs;
        if ((rc = frame_jobs(n, plans, srcs, src_steps, dsts, dst_steps, jobs))) return rc;
        return run_host_chunked(jobs, ImpResult::Frame, n_streams);
    } catch (const std::bad_alloc&) { return IMP_ERROR_MALLOC_FAILED; }
}

// Asynchronous form: the jobs are checked, then the call returns, a helper thread of the library drives the batch on the
// caller's current device, imp_gpu_batch_wait() joins it. The argument arrays are copied; the pixel buffers must stay valid
// until the wait.
int imp_gpu_batch_submit_host(int n, imp_gpu_plan* const* plans, const unsigned char* const* srcs, const int* src_steps,
                              unsigned char* const* dsts, const int* dst_steps, int n_streams, imp_gpu_ticket** ticket) {
    if (!ticket) return IMP_ERROR_INVALID_ARGS;
    *ticket = nullptr;
    int rc = bind(); if (rc) return rc;
    if (n < 0) return IMP_ERROR_INVALID_ARGS;
    try {
        std::vector<ImpHostJob> jobs;
        if ((rc = frame_jobs(n, plans, srcs, src_steps, dsts, dst_steps, jobs))) return rc;
        return start_ticket(std::move(jobs), chunked_run(ImpResult::Frame, n_streams), ticket);
    } catch (const std::bad_alloc&) { return IMP_ERROR_MALLOC_FAILED; }
}

int imp_gpu_batch_poll(const imp_gpu_ticket* ticket) { return ticket && ticket->done.load(std::memory_order_acquire) ? 1 : 0; }

int imp_gpu_batch_wait(imp_gpu_ticket* ticket) {
    if (!ticket) return IMP_ERROR_INVALID_ARGS;
    if (ticket->th.joinable()) ticket->th.join();
    const int rc = ticket->rc;
    if (rc) snprintf(t_err, sizeof t_err, "%s", ticket->err.c_str());
    for (const ImpHostJob& j : ticket->jobs) plan_release(j.plan);
    delete ticket;
    return rc;
}

// Which GPU runs which job (pure host logic: no device is touched). Round-robin: job i -> GPU i mod n_gpus. Size-aware:
// largest job first onto the GPU with the least algorithmic bytes so far (ties: lowest GPU index; equal sizes keep
// request order), the assignment SURVEY 8e asks for on mixed-size farms.
int imp_gpu_farm_assign(int n, imp_gpu_plan* const* plans, int n_gpus, int policy, int* owner) {
    if (n < 0 || n_gpus <= 0 || !owner || (n > 0 && !plans)) return IMP_ERROR_INVALID_ARGS;
    if (policy != IMP_FARM_ROUND_ROBIN && policy != IMP_FARM_SIZE_AWARE) return IMP_ERROR_INVALID_ARGS;
    try {
        if (policy == IMP_FARM_ROUND_ROBIN) { for (int i = 0; i < n; i++) owner[i] = i % n_gpus; return IMP_OK; }
        std::vector<int> order(n);
        for (int i = 0; i < n; i++) { if (!plans[i]) return IMP_ERROR_INVALID_ARGS; order[i] = i; }
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return plans[a]->algo_bytes > plans[b]->algo_bytes; });
        std::vector<unsigned long long> load(n_gpus, 0);
        for (int i : order) {
            int g = 0;
            for (int k = 1; k < n_gpus; k++) if (load[k] < load[g]) g = k;
            load[g] += plans[i]->algo_bytes; owner[i] = g;
        }
    } catch (const std::bad_alloc&) { return IMP_ERROR_MALLOC_FAILED; }
    return IMP_OK;
}

// Independent frames over the GPUs of one box, one host thread per GPU, no inter-GPU traffic.
// IMP_FARM_ROUND_ROBIN: job i -> GPU i mod n_gpus. IMP_FARM_SIZE_AWARE: largest job first onto the GPU with the least
// algorithmic bytes so far (mixed-size farms: evens out the bytes per GPU).
int imp_gpu_farm_run_host_policy(int n, imp_gpu_plan* const* plans, const unsigned char* const* srcs, const int* src_steps,
                                 unsigned char* const* dsts, const int* dst_steps, int n_gpus, int n_streams, int policy) {
    if (n < 0 || n_gpus <= 0 || (policy != IMP_FARM_ROUND_ROBIN && policy != IMP_FARM_SIZE_AWARE)) return IMP_ERROR_INVALID_ARGS;
    if (n > 0 && (!plans || !srcs || !src_steps || !dsts || !dst_steps)) return IMP_ERROR_INVALID_ARGS;
    const int avail = imp_gpu_device_count();
    if (avail <= 0) return fail_msg("no CUDA device available; libimp_gpu has no CPU fallback");
    int devs[MAX_DEV], n_devs = 0;                      // GPU g of the assignment runs on device devs[g]
    if (int rc = device_list(getenv("IMP_GPU_DEVICES"), avail, devs, &n_devs)) return rc;
    if (n_gpus > n_devs) return fail_msg("imp_gpu_farm_run_host: more GPUs requested than present");
    std::vector<std::vector<ImpHostJob>> share(n_gpus);
    try {
        const std::vector<ImpHostJob> jobs = host_jobs(n, plans, srcs, src_steps, dsts, dst_steps);
        int rc = check_host_jobs(ImpResult::Frame, jobs);
        if (rc) return rc;
        std::vector<int> owner(std::max(n, 1));
        if ((rc = imp_gpu_farm_assign(n, plans, n_gpus, policy, owner.data()))) return rc;
        for (int i = 0; i < n; i++) share[owner[i]].push_back(jobs[i]);    // each GPU walks its jobs in request order
    } catch (const std::bad_alloc&) { return IMP_ERROR_MALLOC_FAILED; }
    std::vector<int> rcs(n_gpus, IMP_OK);
    std::vector<std::string> errs(n_gpus);
    std::vector<std::thread> th;
    const int caller_dev = t_dev;
    for (int g = 0; g < n_gpus; g++) {
        th.emplace_back([&, g]() {
            int rc = imp_gpu_set_device(devs[g]);
            if (rc == IMP_OK && !share[g].empty()) {
                try { rc = run_host_chunked(share[g], ImpResult::Frame, n_streams); } catch (const std::bad_alloc&) { rc = IMP_ERROR_MALLOC_FAILED; }
            }
            rcs[g] = rc;
            if (rc) errs[g] = t_err;
        });
    }
    for (auto& t : th) t.join();
    if (caller_dev >= 0) { t_dev = caller_dev; cudaSetDevice(caller_dev); }
    for (int g = 0; g < n_gpus; g++) if (rcs[g]) { snprintf(t_err, sizeof t_err, "gpu %d: %s", devs[g], errs[g].c_str()); return rcs[g]; }
    return IMP_OK;
}

int imp_gpu_farm_run_host(int n, imp_gpu_plan* const* plans, const unsigned char* const* srcs, const int* src_steps,
                          unsigned char* const* dsts, const int* dst_steps, int n_gpus, int n_streams) {
    return imp_gpu_farm_run_host_policy(n, plans, srcs, src_steps, dsts, dst_steps, n_gpus, n_streams, IMP_FARM_ROUND_ROBIN);
}

// ---- format=json / format=text without the frames: brightness and ASCII of the results, reduced on the device ---------
int imp_gpu_batch_brightness_host(int n, imp_gpu_plan* const* plans, const unsigned char* const* srcs, const int* src_steps,
                                  float* brightness, int n_streams) {
    int rc = bind(); if (rc) return rc;
    try {
        std::vector<ImpHostJob> jobs;
        if ((rc = brightness_jobs(n, plans, srcs, src_steps, brightness, jobs))) return rc;
        return run_host_chunked(jobs, ImpResult::Brightness, n_streams);
    } catch (const std::bad_alloc&) { return IMP_ERROR_MALLOC_FAILED; }
}

int imp_gpu_batch_ascii_host(int n, imp_gpu_plan* const* plans, const unsigned char* const* srcs, const int* src_steps,
                             const char* const* args, unsigned char* const* texts, const long* text_caps, int n_streams) {
    int rc = bind(); if (rc) return rc;
    try {
        std::vector<ImpHostJob> jobs;
        if ((rc = ascii_jobs(n, plans, srcs, src_steps, args, texts, text_caps, jobs))) return rc;
        return run_host_chunked(jobs, ImpResult::Ascii, n_streams);
    } catch (const std::bad_alloc&) { return IMP_ERROR_MALLOC_FAILED; }
}

// Asynchronous forms of the two above (imp_gpu_batch_submit_host's contract): each ASCII job's ramp is taken at the submit.
int imp_gpu_batch_brightness_submit_host(int n, imp_gpu_plan* const* plans, const unsigned char* const* srcs, const int* src_steps,
                                         float* brightness, int n_streams, imp_gpu_ticket** ticket) {
    if (!ticket) return IMP_ERROR_INVALID_ARGS;
    *ticket = nullptr;
    int rc = bind(); if (rc) return rc;
    try {
        std::vector<ImpHostJob> jobs;
        if ((rc = brightness_jobs(n, plans, srcs, src_steps, brightness, jobs))) return rc;
        return start_ticket(std::move(jobs), chunked_run(ImpResult::Brightness, n_streams), ticket);
    } catch (const std::bad_alloc&) { return IMP_ERROR_MALLOC_FAILED; }
}

int imp_gpu_batch_ascii_submit_host(int n, imp_gpu_plan* const* plans, const unsigned char* const* srcs, const int* src_steps,
                                    const char* const* args, unsigned char* const* texts, const long* text_caps, int n_streams,
                                    imp_gpu_ticket** ticket) {
    if (!ticket) return IMP_ERROR_INVALID_ARGS;
    *ticket = nullptr;
    int rc = bind(); if (rc) return rc;
    try {
        std::vector<ImpHostJob> jobs;
        if ((rc = ascii_jobs(n, plans, srcs, src_steps, args, texts, text_caps, jobs))) return rc;
        return start_ticket(std::move(jobs), chunked_run(ImpResult::Ascii, n_streams), ticket);
    } catch (const std::bad_alloc&) { return IMP_ERROR_MALLOC_FAILED; }
}

// One frame: the batch kernels over a single job passed by value. Rows take the 16-byte path when base and pitch allow it.
int imp_gpu_brightness_device(const void* d_img, int pitch, int w, int h, int c, float* brightness, void* stream) {
    int rc = bind(); if (rc) return rc;
    if (!d_img || !brightness || w <= 0 || h <= 0 || (c != 1 && c != 3 && c != 4)) return IMP_ERROR_INVALID_ARGS;
    cudaStream_t st = pick_stream(stream);
    ImpInfoJob q{};
    q.img = (const uint8_t*)d_img; q.pitch = pitch; q.w = w; q.h = h; q.c = c;
    q.vec = (reinterpret_cast<uintptr_t>(d_img) % 16 == 0 && pitch % 16 == 0) ? 1 : 0;
    q.ctas = imp_brightness_ctas(w, h);
    const size_t part = align256(sizeof(double) * q.ctas);
    uint8_t* d = nullptr;                                              // partials | ticket | answer
    CK(cudaMallocAsync((void**)&d, part + 256, st));
    unsigned* ticket = reinterpret_cast<unsigned*>(d + part);
    float* d_ans = reinterpret_cast<float*>(d + part + 16);
    float v = 0;
    cudaError_t e = cudaMemsetAsync(ticket, 0, sizeof(unsigned), st);
    if (e == cudaSuccess) e = imp_launch_brightness(nullptr, q, 1, q.ctas, reinterpret_cast<double*>(d), ticket, d_ans, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&v, d_ans, sizeof(float), cudaMemcpyDeviceToHost, st);
    cudaFreeAsync(d, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return fail(e, "brightness", __LINE__);
    *brightness = v;
    return IMP_OK;
}

int imp_gpu_brightness_host(const unsigned char* img, int step, int w, int h, int c, float* brightness) {
    int rc = bind(); if (rc) return rc;
    if (!img || !brightness || w <= 0 || h <= 0 || (c != 1 && c != 3 && c != 4)) return IMP_ERROR_INVALID_ARGS;
    cudaStream_t st = g_dev[t_dev].stream;
    const int pitch = align16(w * c);                                  // staged aligned: the 16-byte path, as on the batch path
    uint8_t* d = nullptr;
    CK(cudaMallocAsync((void**)&d, (size_t)pitch * h, st));
    CK(cudaMemcpy2DAsync(d, pitch, img, step, (size_t)w * c, h, cudaMemcpyHostToDevice, st));
    rc = imp_gpu_brightness_device(d, pitch, w, h, c, brightness, st);
    cudaFreeAsync(d, st);
    return rc;
}

int imp_gpu_ascii_host(const unsigned char* img, int step, int w, int h, int c, const char* args, unsigned char* out, long out_cap) {
    int rc = bind(); if (rc) return rc;
    if (!img || !out || w <= 0 || h <= 0 || (c != 1 && c != 3 && c != 4)) return IMP_ERROR_INVALID_ARGS;
    const long len = imp_gpu_ascii_length(w, h);
    if (out_cap < len) return IMP_ERROR_INVALID_ARGS;
    cudaStream_t st = g_dev[t_dev].stream;
    ImpInfoJob q{};
    q.pitch = align16(w * c); q.w = w; q.h = h; q.c = c; q.vec = 1;
    q.ctas = imp_ascii_ctas(w, h);
    q.wide = (args && strcmp(args, "wide") == 0) ? 1 : 0;                                  // filters.c:490-494
    uint8_t *d_img = nullptr, *d_out = nullptr;
    CK(cudaMallocAsync((void**)&d_img, (size_t)q.pitch * h, st));
    CK(cudaMallocAsync((void**)&d_out, (size_t)len + 1, st));
    q.img = d_img;
    CK(cudaMemcpy2DAsync(d_img, q.pitch, img, step, (size_t)w * c, h, cudaMemcpyHostToDevice, st));
    CK(imp_launch_ascii(nullptr, q, 1, q.ctas, ascii_ramps(), d_out, st));
    CK(cudaMemcpyAsync(out, d_out, (size_t)len, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    cudaFreeAsync(d_img, st); cudaFreeAsync(d_out, st);
    return IMP_OK;
}

// ---- "next" row §8f-2: GIF canvas expansion ------------------------------------------------------------------
// The checks every GIF entry point makes on a GIF's pages.
static int gif_check_pages(const imp_gpu_gif_frame* frames, int n) {
    if (!frames || n <= 0) return IMP_ERROR_INVALID_ARGS;
    for (int f = 0; f < n; f++)
        if (!frames[f].indices || !frames[f].palette || frames[f].width <= 0 || frames[f].height <= 0 || frames[f].pitch < frames[f].width) return IMP_ERROR_INVALID_ARGS;
    return IMP_OK;
}
// Packs a round into h_buf, uploads it to d_buf as one copy and launches its one expansion into d_arena. The pages are
// pageable host memory: a long animation (tens of MB) is packed by several cores (run_parts).
static cudaError_t gif_round_expand(const ImpGifRound& r, uint8_t* h_buf, uint8_t* d_buf, uint8_t* d_arena, cudaStream_t st) {
    const int np = (int)r.pages.size();
    run_parts(np, stage_parts(r.pack_bytes, np), [&r, h_buf, d_buf](int k0, int k1) {
        for (int k = k0; k < k1; k++) imp_gif_pack_page(r, k, h_buf, d_buf, copy_stream);
    });
    cudaError_t e = cudaMemcpyAsync(d_buf, h_buf, r.pack_bytes, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = imp_launch_gif_expand(reinterpret_cast<const ImpGifAlbum*>(d_buf), (int)r.albums.size(),
                                                    reinterpret_cast<const ImpGifFrame*>(d_buf + r.page_off), r.blocks, d_arena, r.arena_bytes, st);
    return e;
}

int imp_gpu_gif_expand_device(const imp_gpu_gif_frame* frames, int n, int canvas_w, int canvas_h, int destructive,
                              void* d_canvases, int canvas_pitch, void* stream) {
    int rc = bind(); if (rc) return rc;
    if (!frames || n <= 0 || canvas_w <= 0 || canvas_h <= 0 || !d_canvases || canvas_pitch < canvas_w * 4 || canvas_pitch % 4) return IMP_ERROR_INVALID_ARGS;
    cudaStream_t st = pick_stream(stream);
    if ((rc = gif_check_pages(frames, n))) return rc;
    const imp_gpu_gif_album album{frames, n, canvas_w, canvas_h, destructive, nullptr, nullptr, nullptr};
    ImpGifRound r;
    try { r = imp_gif_round_layout(&album, 1, canvas_pitch); } catch (const std::bad_alloc&) { return IMP_ERROR_MALLOC_FAILED; }
    uint8_t* h_buf = nullptr; uint8_t* d_buf = nullptr;
    CK(cudaHostAlloc((void**)&h_buf, r.pack_bytes, cudaHostAllocDefault));
    cudaError_t e = cudaMallocAsync((void**)&d_buf, r.pack_bytes, st);
    if (e != cudaSuccess) { cudaFreeHost(h_buf); return fail(e, "cudaMallocAsync", __LINE__); }
    try { e = gif_round_expand(r, h_buf, d_buf, (uint8_t*)d_canvases, st); }
    catch (const std::bad_alloc&) { cudaFreeAsync(d_buf, st); cudaFreeHost(h_buf); return IMP_ERROR_MALLOC_FAILED; }
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);          // h_buf / d_buf are released below
    cudaFreeAsync(d_buf, st);
    cudaFreeHost(h_buf);
    if (e != cudaSuccess) return fail(e, "gif expand", __LINE__);
    return IMP_OK;
}

// A whole GIF request: the pages travel as palette indices (1 byte per pixel instead of the 4 of a decoded canvas), are
// expanded into BGRA canvases on the device (LoadGIF's loop, advancedio.c:195-248) and feed the frame loop of RunJob
// (bridge.c:576-656) without leaving it: grouped launches over all frames, results D2H as in imp_gpu_batch_run_host.
int imp_gpu_gif_album_run_host(const imp_gpu_gif_frame* frames, int n, int canvas_w, int canvas_h, int destructive,
                               imp_gpu_plan* const* plans, unsigned char* const* dsts, const int* dst_steps, int n_streams) {
    const imp_gpu_gif_album album{frames, n, canvas_w, canvas_h, destructive, plans, dsts, dst_steps};
    return imp_gpu_gif_albums_run_host(&album, 1, n_streams);
}

// What the run of an albums call needs besides its job list, all of it the library's own: a submit keeps it until the wait.
struct GifRounds {
    std::vector<imp_gpu_gif_frame> pages;    // every album's page descriptors, copied; `lay` points into them
    std::vector<int> page;                   // job k runs on page page[k] of its album
    std::vector<int> job0;                   // album a's jobs: [job0[a], job0[a + 1])
    std::vector<int> rounds;                 // imp_gif_round_bounds
    std::vector<ImpGifRound> lay;
    size_t pack_max = 0, arena_max = 0;
};

// The "build and check" half of imp_gpu_gif_albums_run_host. A frame's source is its page's canvas; the page stands in for
// it until the canvases are placed, so that a bad job of any album is refused before any buffer grows or any work starts.
static int gif_albums_build(const imp_gpu_gif_album* albums, int n_albums, std::vector<ImpHostJob>& jobs, GifRounds& g) {
    if (n_albums < 0 || (n_albums > 0 && !albums)) return IMP_ERROR_INVALID_ARGS;
    std::vector<imp_gpu_gif_album> own(albums, albums + n_albums);   // their `pages` are pointed at g.pages below
    g.job0.assign((size_t)n_albums + 1, 0);
    for (int a = 0; a < n_albums; a++) {
        const imp_gpu_gif_album& al = albums[a];
        if (al.canvas_w <= 0 || al.canvas_h <= 0 || !al.plans || !al.dsts || !al.dst_steps) return IMP_ERROR_INVALID_ARGS;
        if (int rc = gif_check_pages(al.pages, al.n_pages)) return rc;
        g.job0[a] = (int)jobs.size();
        for (int f = 0; f < al.n_pages; f++) {
            imp_gpu_plan* p = al.plans[f];                            // null: replayed for the pages after it, no result wanted
            if (!p) continue;
            if (p->src_w != al.canvas_w || p->src_h != al.canvas_h || p->src_c != 4) return IMP_ERROR_INVALID_ARGS;
            jobs.push_back(ImpHostJob{p, al.pages[f].indices, align16(al.canvas_w * 4), al.dsts[f], al.dst_steps[f], false});
            g.page.push_back(f);
        }
        g.pages.insert(g.pages.end(), al.pages, al.pages + al.n_pages);
    }
    g.job0[n_albums] = (int)jobs.size();
    if (int rc = check_host_jobs(ImpResult::Frame, jobs)) return rc;
    for (int a = 0, f0 = 0; a < n_albums; f0 += own[a].n_pages, a++) own[a].pages = g.pages.data() + f0;
    g.rounds = imp_gif_round_bounds(own.data(), n_albums);
    for (size_t r = 0; r + 1 < g.rounds.size(); r++) {
        g.lay.push_back(imp_gif_round_layout(own.data() + g.rounds[r], g.rounds[r + 1] - g.rounds[r]));
        g.pack_max = std::max(g.pack_max, g.lay.back().pack_bytes);
        g.arena_max = std::max(g.arena_max, g.lay.back().arena_bytes);
    }
    return IMP_OK;
}

// The "run" half: per round one pack of all its albums' pages, one upload, one expansion launch and one chunked frame loop
// over all its albums' frames, so that chunks and grouped launches span requests.
static int gif_albums_run(const GifRounds& g, std::vector<ImpHostJob>& jobs, int n_streams) {
    if (g.lay.empty()) return IMP_OK;
    DevCtx& ctx = g_dev[t_dev];
    std::lock_guard<std::mutex> run_lk(ctx.run_mu);
    int rc;
    if ((rc = ctx.h_gif.grow(g.pack_max, true)) || (rc = ctx.d_gif.grow(g.pack_max, false)) || (rc = ctx.d_canvas.grow(g.arena_max, false))) return rc;
    if (!ctx.gif_ev) CK(cudaEventCreateWithFlags(&ctx.gif_ev, cudaEventDisableTiming));
    try {                                                             // the C caller cannot unwind: bad_alloc ends as a code
    for (size_t r = 0; r < g.lay.size() && rc == IMP_OK; r++) {       // one after another: the pack and the arena are reused
        const ImpGifRound& R = g.lay[r];
        const int a0 = g.rounds[r], a1 = g.rounds[r + 1];
        for (int a = a0; a < a1; a++) {
            const ImpGifAlbum& A = R.albums[a - a0];
            for (int k = g.job0[a]; k < g.job0[a + 1]; k++) jobs[k].src = ctx.d_canvas.p + A.canvas_off + (size_t)g.page[k] * A.pitch * A.ch;
        }
        CK(gif_round_expand(R, ctx.h_gif.p, ctx.d_gif.p, ctx.d_canvas.p, ctx.stream));
        CK(cudaEventRecord(ctx.gif_ev, ctx.stream));
        const int j0 = g.job0[a0], j1 = g.job0[a1];
        if (j0 == j1) CK(cudaStreamSynchronize(ctx.stream));
        else rc = run_host_chunked_locked(jobs.data() + j0, j1 - j0, ImpResult::Frame, n_streams, true, ctx.gif_ev);
    }
    } catch (const std::bad_alloc&) { rc = IMP_ERROR_MALLOC_FAILED; }
    if (rc != IMP_OK) cudaStreamSynchronize(ctx.stream);           // the staging buffers are reused by the next call
    return rc;
}

int imp_gpu_gif_albums_run_host(const imp_gpu_gif_album* albums, int n_albums, int n_streams) {
    int rc = bind(); if (rc) return rc;
    std::vector<ImpHostJob> jobs;
    GifRounds g;
    try { if ((rc = gif_albums_build(albums, n_albums, jobs, g))) return rc; }
    catch (const std::bad_alloc&) { return IMP_ERROR_MALLOC_FAILED; }
    return gif_albums_run(g, jobs, n_streams);
}

int imp_gpu_gif_albums_submit_host(const imp_gpu_gif_album* albums, int n_albums, int n_streams, imp_gpu_ticket** ticket) {
    if (!ticket) return IMP_ERROR_INVALID_ARGS;
    *ticket = nullptr;
    int rc = bind(); if (rc) return rc;
    try {
        std::vector<ImpHostJob> jobs;
        auto g = std::make_shared<GifRounds>();
        if ((rc = gif_albums_build(albums, n_albums, jobs, *g))) return rc;
        return start_ticket(std::move(jobs), [g, n_streams](std::vector<ImpHostJob>& j) { return gif_albums_run(*g, j, n_streams); }, ticket);
    } catch (const std::bad_alloc&) { return IMP_ERROR_MALLOC_FAILED; }
}

int imp_gpu_gif_expand_host(const imp_gpu_gif_frame* frames, int n, int canvas_w, int canvas_h, int destructive,
                            unsigned char* const* canvases, int canvas_step) {
    int rc = bind(); if (rc) return rc;
    if (!canvases || canvas_step < canvas_w * 4) return IMP_ERROR_INVALID_ARGS;
    cudaStream_t st = g_dev[t_dev].stream;
    const int pitch = align16(canvas_w * 4);
    uint8_t* d = nullptr;
    CK(cudaMalloc((void**)&d, (size_t)pitch * canvas_h * n));
    rc = imp_gpu_gif_expand_device(frames, n, canvas_w, canvas_h, destructive, d, pitch, st);
    for (int f = 0; f < n && rc == IMP_OK; f++) {
        cudaError_t e = cudaMemcpy2D(canvases[f], canvas_step, d + (size_t)f * pitch * canvas_h, pitch, (size_t)canvas_w * 4, canvas_h, cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) rc = fail(e, "cudaMemcpy2D", __LINE__);
    }
    cudaFree(d);
    return rc;
}

// ---- memory helpers ------------------------------------------------------------------------------------
int imp_gpu_malloc(void** p, size_t bytes) { int rc = bind(); if (rc) return rc; CK(cudaMalloc(p, bytes)); return IMP_OK; }
int imp_gpu_free(void* p) { int rc = bind(); if (rc) return rc; CK(cudaFree(p)); return IMP_OK; }
int imp_gpu_malloc_pitch(void** p, int* pitch, int width_bytes, int height) {
    int rc = bind(); if (rc) return rc;
    const int pt = align16(width_bytes);
    CK(cudaMalloc(p, (size_t)pt * (size_t)std::max(height, 1)));
    if (pitch) *pitch = pt;
    return IMP_OK;
}
int imp_gpu_host_alloc(void** p, size_t bytes) { int rc = bind(); if (rc) return rc; CK(cudaHostAlloc(p, bytes, cudaHostAllocDefault)); return IMP_OK; }
int imp_gpu_host_free(void* p) { int rc = bind(); if (rc) return rc; CK(cudaFreeHost(p)); return IMP_OK; }
int imp_gpu_upload_2d(void* d, int dp, const void* h, int hs, int wb, int rows, void* stream) {
    int rc = bind(); if (rc) return rc;
    CK(cudaMemcpy2DAsync(d, dp, h, hs, wb, rows, cudaMemcpyHostToDevice, pick_stream(stream)));
    return IMP_OK;
}
int imp_gpu_download_2d(void* h, int hs, const void* d, int dp, int wb, int rows, void* stream) {
    int rc = bind(); if (rc) return rc;
    CK(cudaMemcpy2DAsync(h, hs, d, dp, wb, rows, cudaMemcpyDeviceToHost, pick_stream(stream)));
    return IMP_OK;
}
int imp_gpu_sync(void* stream) {
    int rc = bind(); if (rc) return rc;
    if (stream) CK(cudaStreamSynchronize((cudaStream_t)stream));
    else CK(cudaDeviceSynchronize());
    return IMP_OK;
}

}  // extern "C"
