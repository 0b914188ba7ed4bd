// imp_ops.cpp — reference-signature operators (include/imp_ops.h): record + validate now, run fused later.
#include "../../include/imp_ops.h"
#include "imp_internal.h"
#include <string.h>
#include <stdlib.h>
#include <map>
#include <mutex>
#include <string>
#include <vector>

namespace {

struct Pending {
    // the decoded frame as it was before the first recorded op
    char* data; int w, h, c, step;
    // what the header was last set to (to recognise a recycled IplImage address)
    int cur_w, cur_h, cur_c;
    bool has_crop = false, has_gravity = false, has_resize = false;
    std::string crop, gravity, resize;
    std::vector<std::string> filters;
    int simple = 0, flatten = 0, allow = 0, n_ops = 0;
    bool has_wm = false; imp_gpu_watermark wm{};
    unsigned max_w = 0, max_h = 0;
};

std::map<const IplImage*, Pending> g_pending;
std::mutex g_ops_mu;
imp_ops_create_image_fn g_create = nullptr;
imp_ops_release_image_fn g_release = nullptr;

IplImage* default_create(int w, int h, int depth, int c) {
    IplImage* im = (IplImage*)calloc(1, sizeof(IplImage));
    if (!im) return nullptr;
    im->nSize = (int)sizeof(IplImage); im->nChannels = c; im->depth = depth; im->width = w; im->height = h; im->align = 4;
    im->widthStep = (w * c + 3) & ~3;                 // cvCreateImage's 4-byte row alignment
    im->imageSize = im->widthStep * h;
    im->imageData = im->imageDataOrigin = (char*)malloc(im->imageSize > 0 ? (size_t)im->imageSize : 1);
    if (!im->imageData) { free(im); return nullptr; }
    return im;
}
void default_release(IplImage** p) {
    if (p && *p) { free((*p)->imageDataOrigin); free((*p)->roi); free(*p); *p = nullptr; }
}

Pending from_header(const IplImage* im) {
    Pending p;
    p.data = im->imageData; p.w = p.cur_w = im->width; p.h = p.cur_h = im->height; p.c = p.cur_c = im->nChannels; p.step = im->widthStep;
    return p;
}

Pending& entry(IplImage* im) {
    auto it = g_pending.find(im);
    if (it != g_pending.end()) {
        Pending& p = it->second;
        if (p.data == im->imageData && p.cur_w == im->width && p.cur_h == im->height && p.cur_c == im->nChannels) return p;
        g_pending.erase(it);                              // a different image now lives at this address
    }
    return g_pending.emplace(im, from_header(im)).first->second;
}

struct Built { imp_gpu_request req; imp_gpu_config cfg; std::vector<const char*> fp; };
void to_request(const Pending& p, Built& b) {
    b.fp.clear();
    for (const std::string& f : p.filters) b.fp.push_back(f.c_str());
    b.req.crop = p.has_crop ? p.crop.c_str() : nullptr;
    b.req.gravity = p.has_gravity ? p.gravity.c_str() : nullptr;
    b.req.resize = p.has_resize ? p.resize.c_str() : nullptr;
    b.req.filters = b.fp.empty() ? nullptr : b.fp.data();
    b.req.filter_count = (int)b.fp.size();
    b.req.simple_resize = p.simple; b.req.flatten = p.flatten; b.req.interp = IMP_INTERP_REFERENCE; b.req.pack = IMP_PACK_NONE;
    b.cfg.max_target_w = p.max_w; b.cfg.max_target_h = p.max_h;
    b.cfg.max_filters = 1 << 20;                         // RunJob enforces the count while parsing (bridge.c:361)
    b.cfg.allow_experiments = p.allow;
    b.cfg.watermark = p.has_wm ? &p.wm : nullptr;
}

// Validates the recorded chain (the newest op included); on success fixes the header up. The planner runs in its
// validate-only mode: same codes and geometry, no tables, LUTs or overlay pixels (the lowering happens once, at the flush,
// and is served from the plan cache for every further frame and request of the same shape).
int validate(IplImage* im, Pending& p) {
    Built b; to_request(p, b);
    imp_gpu_plan plan;
    int step = 0;
    int rc = imp_build_plan(&b.req, &b.cfg, p.w, p.h, p.c, &plan, &step, true);
    if (rc) return rc;
    im->width = p.cur_w = plan.out_w; im->height = p.cur_h = plan.out_h; im->nChannels = p.cur_c = plan.out_c;
    // imageData still holds the undisturbed source; widthStep/imageSize keep describing THAT buffer until imp_Flush
    p.n_ops++;
    return IMP_OK;
}

// What a flush runs for `im` (caller holds g_ops_mu): the recorded chain, or — nothing recorded, `*idle` — the frame as it
// is, held in `scratch`. An idle frame only has to run when it has 1 channel: the empty plan promotes gray to BGR
// (bridge.c:613-618).
const Pending& flush_entry(IplImage* im, Pending& scratch, bool* idle) {
    auto it = g_pending.find(im);
    *idle = it == g_pending.end() || it->second.n_ops == 0;
    if (!*idle) return it->second;
    scratch = from_header(im);
    return scratch;
}

int make_plan(const Pending& p, imp_gpu_plan** plan_out) {
    Built b; to_request(p, b);
    int step = 0;
    return imp_gpu_plan_create(&b.req, &b.cfg, p.w, p.h, p.c, plan_out, &step);
}

int run_one(IplImage** pointer, const Pending& p, imp_gpu_plan** plan_out, IplImage** out_img) {
    int rc = make_plan(p, plan_out);
    if (rc) return rc;
    imp_ops_create_image_fn create = g_create ? g_create : default_create;
    IplImage* out = create((*plan_out)->out_w, (*plan_out)->out_h, (*pointer)->depth ? (*pointer)->depth : 8, (*plan_out)->out_c);
    if (!out) { imp_gpu_plan_destroy(*plan_out); *plan_out = nullptr; return IMP_ERROR_MALLOC_FAILED; }
    *out_img = out;
    return IMP_OK;
}

}  // namespace

// The C frames of bridge.c cannot unwind: a C++ exception (bad_alloc, length_error) ends as a return code.
#define IMP_OPS_TRY try {
#define IMP_OPS_CATCH } catch (const std::bad_alloc&) { return IMP_ERROR_MALLOC_FAILED; } catch (...) { return IMP_ERROR_INVALID_ARGS; }

extern "C" {

void imp_ops_set_image_allocator(imp_ops_create_image_fn create, imp_ops_release_image_fn release) {
    std::lock_guard<std::mutex> lk(g_ops_mu);
    g_create = create; g_release = release;
}

int imp_Crop(IplImage** pointer, char* args, char* gravity) {
    IMP_OPS_TRY
    if (!pointer || !*pointer || !args) return IMP_ERROR_INVALID_ARGS;
    std::lock_guard<std::mutex> lk(g_ops_mu);
    Pending& p = entry(*pointer);
    if (p.has_crop || p.has_resize || !p.filters.empty() || p.has_wm || p.flatten) return IMP_ERROR_UNSUPPORTED;   // RunJob's order is fixed: flush first
    Pending saved = p;
    p.has_crop = true; p.crop = args;
    p.has_gravity = gravity != nullptr; if (gravity) p.gravity = gravity;
    int rc = validate(*pointer, p);
    if (rc) p = saved;
    return rc;
    IMP_OPS_CATCH
}

int imp_Resize(IplImage** pointer, char* args, const imp_gpu_config* config, int simple) {
    IMP_OPS_TRY
    if (!pointer || !*pointer || !args) return IMP_ERROR_INVALID_ARGS;
    std::lock_guard<std::mutex> lk(g_ops_mu);
    Pending& p = entry(*pointer);
    if (p.has_resize || !p.filters.empty() || p.has_wm || p.flatten) return IMP_ERROR_UNSUPPORTED;
    Pending saved = p;
    p.has_resize = true; p.resize = args; p.simple = simple ? 1 : 0;
    p.max_w = config ? config->max_target_w : 0; p.max_h = config ? config->max_target_h : 0;
    int rc = validate(*pointer, p);
    if (rc) p = saved;
    return rc;
    IMP_OPS_CATCH
}

int imp_Filter(IplImage** pointer, char* request, int allowExperiments) {
    IMP_OPS_TRY
    if (!pointer || !*pointer || !request) return IMP_ERROR_INVALID_ARGS;
    std::lock_guard<std::mutex> lk(g_ops_mu);
    Pending& p = entry(*pointer);
    if (p.has_wm || p.flatten) return IMP_ERROR_UNSUPPORTED;
    Pending saved = p;
    p.filters.push_back(request); p.allow = allowExperiments ? 1 : 0;
    int rc = validate(*pointer, p);
    if (rc) p = saved;
    return rc;
    IMP_OPS_CATCH
}

int imp_Watermark(IplImage* image, const imp_gpu_config* config) {
    IMP_OPS_TRY
    if (!image) return IMP_ERROR_INVALID_ARGS;
    if (!config || !config->watermark) return IMP_OK;
    std::lock_guard<std::mutex> lk(g_ops_mu);
    Pending& p = entry(image);
    if (p.has_wm || p.flatten) return IMP_ERROR_UNSUPPORTED;
    Pending saved = p;
    p.has_wm = true; p.wm = *config->watermark;
    int rc = validate(image, p);
    if (rc) p = saved;
    return rc;
    IMP_OPS_CATCH
}

int imp_BlendWithPaper(IplImage* image) {
    IMP_OPS_TRY
    if (!image) return IMP_ERROR_INVALID_ARGS;
    std::lock_guard<std::mutex> lk(g_ops_mu);
    Pending& p = entry(image);
    Pending saved = p;
    p.flatten = 1;
    int rc = validate(image, p);
    if (rc) p = saved;
    return rc;
    IMP_OPS_CATCH
}

int imp_ops_pending(const IplImage* image) {
    std::lock_guard<std::mutex> lk(g_ops_mu);
    auto it = g_pending.find(image);
    return it == g_pending.end() ? 0 : it->second.n_ops;
}

void imp_Discard(IplImage* image) {
    std::lock_guard<std::mutex> lk(g_ops_mu);
    auto it = g_pending.find(image);
    if (it == g_pending.end()) return;
    // restore the header to the buffer it really describes
    image->width = it->second.w; image->height = it->second.h; image->nChannels = it->second.c;
    g_pending.erase(it);
}

// pages != nullptr: the album of a GIF whose canvases live on the device only (imp_FlushAllGif) — every frame takes part,
// the sources are the pages, and frames[i]'s own pixels are never read.
static int flush_all(IplImage** frames, int count, const imp_gpu_gif_frame* pages, int n_pages, int destructive) {
    IMP_OPS_TRY
    if (!frames || count < 0) return IMP_ERROR_INVALID_ARGS;
    std::vector<imp_gpu_plan*> plans; std::vector<IplImage*> outs; std::vector<int> idx;
    std::vector<const unsigned char*> srcs; std::vector<unsigned char*> dsts; std::vector<int> ss, ds;
    int rc = IMP_OK, cw = 0, ch = 0;                                  // GIF: the canvas every page is composed onto
    {
        std::lock_guard<std::mutex> lk(g_ops_mu);
        for (int i = 0; i < count && rc == IMP_OK; i++) {
            if (!frames[i]) { if (pages) rc = IMP_ERROR_INVALID_ARGS; continue; }
            Pending scratch; bool idle;
            const Pending& p = flush_entry(frames[i], scratch, &idle);
            if (idle && frames[i]->nChannels != 1 && !pages) { g_pending.erase(frames[i]); continue; }
            if (pages) {
                if (i == 0) { cw = p.w; ch = p.h; }
                if (p.c != 4 || p.w != cw || p.h != ch) { rc = IMP_ERROR_INVALID_ARGS; break; }
            }
            imp_gpu_plan* plan = nullptr; IplImage* out = nullptr;
            rc = run_one(&frames[i], p, &plan, &out);
            if (rc) break;
            plans.push_back(plan); outs.push_back(out); idx.push_back(i);
            srcs.push_back((const unsigned char*)p.data); ss.push_back(p.step);
            dsts.push_back((unsigned char*)out->imageData); ds.push_back(out->widthStep);
        }
    }
    if (rc == IMP_OK && !plans.empty()) {
        if (pages) {
            // frame k is page k, or (a `page` request) the one frame is the last page and the earlier pages are only replayed
            const int skip = n_pages - (int)plans.size();
            std::vector<imp_gpu_plan*> pp((size_t)n_pages, nullptr); std::vector<unsigned char*> pd((size_t)n_pages, nullptr); std::vector<int> ps((size_t)n_pages, 0);
            for (size_t k = 0; k < plans.size(); k++) { pp[skip + k] = plans[k]; pd[skip + k] = dsts[k]; ps[skip + k] = ds[k]; }
            rc = imp_gpu_gif_album_run_host(pages, n_pages, cw, ch, destructive, pp.data(), pd.data(), ps.data(), 4);
        } else {
            rc = imp_gpu_batch_run_host((int)plans.size(), plans.data(), srcs.data(), ss.data(), dsts.data(), ds.data(), 4);
        }
    }
    imp_ops_release_image_fn release = g_release ? g_release : default_release;
    {
        std::lock_guard<std::mutex> lk(g_ops_mu);
        for (size_t k = 0; k < plans.size(); k++) {
            IplImage* old = frames[idx[k]];
            if (rc == IMP_OK) {
                g_pending.erase(old);
                frames[idx[k]] = outs[k];
                release(&old);
            } else {
                release(&outs[k]);
            }
            imp_gpu_plan_destroy(plans[k]);
        }
    }
    return rc;
    IMP_OPS_CATCH
}

int imp_FlushAll(IplImage** frames, int count) { return flush_all(frames, count, nullptr, 0, 0); }

int imp_FlushAllGif(IplImage** frames, int count, const imp_gpu_gif_frame* pages, int n_pages, int destructive) {
    if (!pages || count <= 0 || !(n_pages == count || (count == 1 && n_pages >= 1))) return IMP_ERROR_INVALID_ARGS;
    return flush_all(frames, count, pages, n_pages, destructive);
}

int imp_Flush(IplImage** pointer) {
    if (!pointer || !*pointer) return IMP_ERROR_INVALID_ARGS;
    return imp_FlushAll(pointer, 1);
}

// The job imp_Flush would run for `image` (an idle multi-channel frame: the empty plan, a copy), its answer computed on the
// device. Nothing recorded is consumed.
static int answer_job(IplImage* image, imp_gpu_plan** plan, const unsigned char** src, int* step) {
    std::lock_guard<std::mutex> lk(g_ops_mu);
    Pending scratch; bool idle;
    const Pending& p = flush_entry(image, scratch, &idle);
    *src = (const unsigned char*)p.data; *step = p.step;
    return make_plan(p, plan);
}

int imp_Brightness(IplImage* image, float* brightness) {
    IMP_OPS_TRY
    if (!image || !brightness) return IMP_ERROR_INVALID_ARGS;
    imp_gpu_plan* plan = nullptr; const unsigned char* src = nullptr; int step = 0;
    int rc = answer_job(image, &plan, &src, &step);
    if (rc) return rc;
    rc = imp_gpu_batch_brightness_host(1, &plan, &src, &step, brightness, 1);
    imp_gpu_plan_destroy(plan);
    return rc;
    IMP_OPS_CATCH
}

int imp_Ascii(IplImage* image, const char* args, unsigned char* out, long out_cap) {
    IMP_OPS_TRY
    if (!image || !out) return IMP_ERROR_INVALID_ARGS;
    imp_gpu_plan* plan = nullptr; const unsigned char* src = nullptr; int step = 0;
    int rc = answer_job(image, &plan, &src, &step);
    if (rc) return rc;
    unsigned char* texts[1] = {out};
    rc = imp_gpu_batch_ascii_host(1, &plan, &src, &step, &args, texts, &out_cap, 1);
    imp_gpu_plan_destroy(plan);
    return rc;
    IMP_OPS_CATCH
}

}  // extern "C"
