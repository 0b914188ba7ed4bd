/*
 * imp_dropin.c — the reference's OWN operator symbols (bridge.h:2-7, filters.h:1-16,30) implemented on libimp_gpu.so.
 *
 * This file is compiled INSIDE the nginx module, next to bridge.c (add it to NGX_ADDON_SRCS in the module's `config`), so
 * it sees the module's real required.h — Config, Album, IplImage come from there, nothing is re-declared. With it linked
 * in, the definitions it replaces are deleted from the reference and every call site stays as it is:
 *
 *   bridge.c   OnEnvStart, OnEnvDestroy (:10-16), Crop (:18-141), Resize (:143-197), Watermark (:239-281)
 *   filters.c  the 14 filter callbacks Flip .. Scanline (:72-455) and BlendWithPaper (:666-687)
 *
 * filters.c's Filter / CallbackMap / CheckDestructive (:5-70) stay untouched and now dispatch to the callbacks below;
 * ASCII, CalcPerceivedBrightness and helpers.c stay on the host. RunJob itself gains ONE statement before its
 * "alternative exit points" (bridge.c:658):   answer->Code = imp_FlushAlbum(&album); if (answer->Code) goto finalize;
 * and its gray->BGR block (bridge.c:613-618) goes away (INTEGRATION.md §2). Every function here validates its arguments
 * exactly like the one it replaces (same IMP_* code, image untouched on error), records the operation and fixes the
 * IplImage header up; imp_FlushAlbum runs what was recorded for all frames as fused GPU passes.
 */
#include <ngx_config.h>
#include <ngx_core.h>
#include "required.h"
#include "bridge.h"
#include "filters.h"
#include "imp_ops.h"
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

/* frames stay owned by OpenCV's allocator: RunJob releases them with cvReleaseImage (bridge.c:714-722) */
static IplImage* imp_create(int w, int h, int depth, int ch) { return cvCreateImage(cvSize(w, h), depth, ch); }
static void      imp_release(IplImage** im)                  { cvReleaseImage(im); }

/* Config (required.h:110-120) -> the plain struct of imp_gpu.h; the watermark pixels stay in the conf pool
 * (PrepareWatermark, bridge.c:199-237) and are interned + uploaded once per worker by the library */
static void imp_config_from(const Config* c, imp_gpu_config* g, imp_gpu_watermark* w) {
    g->max_target_w = c->MaxTargetDimensions ? c->MaxTargetDimensions->W : 0;
    g->max_target_h = c->MaxTargetDimensions ? c->MaxTargetDimensions->H : 0;
    g->max_filters = (int)c->MaxFiltersCount;
    g->allow_experiments = (int)c->AllowExperiments;
    g->watermark = NULL;
    if (c->WatermarkInfo) {
        w->pixels = c->WatermarkInfo->Pointer;
        w->width = c->WatermarkInfo->Size.width;  w->height = c->WatermarkInfo->Size.height;
        w->channels = c->WatermarkInfo->Channels; w->step = c->WatermarkInfo->Step;
        w->gravity_x = c->WatermarkPosition->GravityX; w->gravity_y = c->WatermarkPosition->GravityY;
        w->offset_x = c->WatermarkPosition->OffsetX;   w->offset_y = c->WatermarkPosition->OffsetY;
        w->opacity = (int)c->WatermarkOpacity;
        g->watermark = w;
    }
}

/* The worker's index (nginx's ngx_process_cycle.c sets it before the worker's init_process handlers run). Weak: inside
 * nginx its own definition is the one linked, and a host built without nginx (the reference's RunJob linked against
 * stand-in headers for testing) still links, as worker 0 unless it sets the symbol. */
ngx_uint_t ngx_worker __attribute__((weak));

/* module.c:100-107 calls these per worker process, i.e. after fork: the CUDA context is created here, on the device the
 * worker's index selects (IMP_GPU_DEVICES, imp_gpu.h), so that worker_processes spreads the workers over every GPU of the
 * box. Without a device every request answers IMP_ERROR_GPU; the startup log says why. */
void OnEnvStart() {
    int dev = -1;
    if (imp_gpu_init_worker((int)ngx_worker, &dev) == IMP_OK)
        ngx_log_error(NGX_LOG_NOTICE, ngx_cycle->log, 0, "imgproc: worker %d on GPU %d", (int)ngx_worker, dev);
    else
        ngx_log_error(NGX_LOG_EMERG, ngx_cycle->log, 0, "imgproc: worker %d has no GPU: %s", (int)ngx_worker, imp_gpu_last_error());
    imp_ops_set_image_allocator(imp_create, imp_release);
}
void OnEnvDestroy() { imp_gpu_shutdown(); }

int Crop(IplImage** pointer, char* args, char* gravity) { return imp_Crop(pointer, args, gravity); }

int Resize(IplImage** pointer, char* args, Config* config, int simple) {
    imp_gpu_config g; imp_gpu_watermark w;
    imp_config_from(config, &g, &w);
    return imp_Resize(pointer, args, &g, simple);
}

int Watermark(IplImage* image, Config* config) {
    imp_gpu_config g; imp_gpu_watermark w;
    imp_config_from(config, &g, &w);
    return imp_Watermark(image, &g);
}

void BlendWithPaper(IplImage* source) { imp_BlendWithPaper(source); }

/* The callbacks filters.c's CallbackMap points at. Filter (filters.c:43-70, unchanged) has already split "name=args",
 * matched the name and checked the experimental flag, so the operation is recorded as allowed. */
static int imp_record(IplImage** pointer, const char* name, char* args) {
    size_t n = strlen(name) + 1 + strlen(args) + 1;
    char* request = (char*)malloc(n);
    int rc;
    if (!request) return IMP_ERROR_MALLOC_FAILED;
    snprintf(request, n, "%s=%s", name, args);
    rc = imp_Filter(pointer, request, 1);
    free(request);
    return rc;
}
int Flip    (IplImage** pointer, char* args) { return imp_record(pointer, "flip", args); }
int Rotate  (IplImage** pointer, char* args) { return imp_record(pointer, "rotate", args); }
int Modulate(IplImage** pointer, char* args) { return imp_record(pointer, "modulate", args); }
int Colorize(IplImage** pointer, char* args) { return imp_record(pointer, "colorize", args); }
int Blur    (IplImage** pointer, char* args) { return imp_record(pointer, "blur", args); }
int Gamma   (IplImage** pointer, char* args) { return imp_record(pointer, "gamma", args); }
int Contrast(IplImage** pointer, char* args) { return imp_record(pointer, "contrast", args); }
int Gradmap (IplImage** pointer, char* args) { return imp_record(pointer, "gradmap", args); }
int Vignette(IplImage** pointer, char* args) { return imp_record(pointer, "vignette", args); }
int Gotham  (IplImage** pointer, char* args) { return imp_record(pointer, "gotham", args); }
int Lomo    (IplImage** pointer, char* args) { return imp_record(pointer, "lomo", args); }
int Kelvin  (IplImage** pointer, char* args) { return imp_record(pointer, "kelvin", args); }
int Rainbow (IplImage** pointer, char* args) { return imp_record(pointer, "rainbow", args); }
int Scanline(IplImage** pointer, char* args) { return imp_record(pointer, "scanline", args); }

/* ---- GIF albums: LoadGIF's per-pixel loop (advancedio.c:195-248) on the device -------------------------------------
 * With INTEGRATION.md §4's edit LoadGIF no longer composes the canvases: for every page it walks it calls
 * imp_AlbumGifPage, which keeps a copy of the page's index bits (1 byte per pixel) and palette; the canvas-sized frames it
 * still creates are placeholders. imp_FlushAlbum recognises the album by its last frame and expands the pages on the
 * device, straight into the frame loop. One album is in flight per worker (RunJob is synchronous): a single slot. */
static struct {
    IplImage* last;                 /* Image of the newest registered page: Frames[Count-1] of the album, also after a `page` request */
    unsigned char stamp[16];        /* written into that placeholder's (never read) pixels: a recycled address cannot pass for it */
    imp_gpu_gif_frame* pages;
    unsigned char** blocks;         /* one malloc per page: palette (1024 bytes) then the index bits */
    int count, cap, destructive;
} imp_gif;

static void imp_gif_reset(void) {
    int k;
    for (k = 0; k < imp_gif.count; k++) free(imp_gif.blocks[k]);
    imp_gif.count = 0; imp_gif.last = NULL;
}

int imp_AlbumGifPage(Album* album, int frameid, int isdestructive, const unsigned char* bits, int pitch, int width, int height,
                     int left, int top, const void* palette) {
    unsigned char* block;
    imp_gpu_gif_frame* pg;
    if (!album || frameid < 0 || !bits || !palette || pitch < width || width <= 0 || height <= 0) return IMP_ERROR_INVALID_ARGS;
    if (frameid == 0) imp_gif_reset();
    if (frameid != imp_gif.count) return IMP_ERROR_INVALID_ARGS;            /* LoadGIF walks the pages in order */
    if (imp_gif.count == imp_gif.cap) {
        int cap = imp_gif.cap ? imp_gif.cap * 2 : 64;
        imp_gpu_gif_frame* np = (imp_gpu_gif_frame*)realloc(imp_gif.pages, sizeof(imp_gpu_gif_frame) * (size_t)cap);
        unsigned char** nb;
        if (!np) return IMP_ERROR_MALLOC_FAILED;
        imp_gif.pages = np;
        nb = (unsigned char**)realloc(imp_gif.blocks, sizeof(unsigned char*) * (size_t)cap);
        if (!nb) return IMP_ERROR_MALLOC_FAILED;
        imp_gif.blocks = nb; imp_gif.cap = cap;
    }
    block = (unsigned char*)malloc(1024 + (size_t)pitch * (size_t)height);
    if (!block) return IMP_ERROR_MALLOC_FAILED;
    memcpy(block, palette, 1024);
    memcpy(block + 1024, bits, (size_t)pitch * (size_t)height);
    pg = &imp_gif.pages[imp_gif.count];
    pg->indices = block + 1024; pg->pitch = pitch; pg->width = width; pg->height = height;
    pg->left = left; pg->top = top;
    pg->dispose = album->Frames[frameid].Dispose;
    pg->transparency_key = album->Frames[frameid].TransparencyKey;
    pg->palette = block;
    imp_gif.blocks[imp_gif.count++] = block;
    imp_gif.destructive = isdestructive;
    imp_gif.last = album->Frames[frameid].Image;
    {   /* RunJob may fail between LoadGIF and the flush and release the frames; a later album's frame can then live at the
         * same address. The placeholder's pixels carry a stamp that an image decoded there would have overwritten. */
        static unsigned long long serial = 0;
        int nb = imp_gif.last->imageSize < 16 ? imp_gif.last->imageSize : 16;
        serial++;
        memcpy(imp_gif.stamp, "IMPGIFPG", 8);
        memcpy(imp_gif.stamp + 8, &serial, 8);
        if (nb > 0 && imp_gif.last->imageData) memcpy(imp_gif.last->imageData, imp_gif.stamp, (size_t)nb);
    }
    return IMP_OK;
}

static int imp_gif_is_album(IplImage* last, int count) {
    int nb;
    if (!imp_gif.count || imp_gif.last != last || !(imp_gif.count == count || count == 1)) return 0;
    nb = last->imageSize < 16 ? last->imageSize : 16;
    return nb <= 0 || !last->imageData || memcmp(last->imageData, imp_gif.stamp, (size_t)nb) == 0;
}

/* Runs everything recorded for the album's frames (bridge.c:576-656 loops) as fused GPU passes: one batched call.
 * The album of a GIF whose pages were handed to imp_AlbumGifPage takes its pixels from them (expanded on the device). */
int imp_FlushAlbum(Album* album) {
    IplImage* stack[64];
    IplImage** fr = stack;
    int k, rc;
    if (album->Count <= 0) return IMP_OK;
    if (album->Count > 64) { fr = (IplImage**)malloc(sizeof(IplImage*) * (size_t)album->Count); if (!fr) return IMP_ERROR_MALLOC_FAILED; }
    for (k = 0; k < album->Count; k++) fr[k] = album->Frames[k].Image;
    if (imp_gif_is_album(fr[album->Count - 1], album->Count)) {
        rc = imp_FlushAllGif(fr, album->Count, imp_gif.pages, imp_gif.count, imp_gif.destructive);
        imp_gif_reset();
    } else {
        rc = imp_FlushAll(fr, album->Count);
    }
    for (k = 0; k < album->Count; k++) album->Frames[k].Image = fr[k];
    if (fr != stack) free(fr);
    return rc;
}
