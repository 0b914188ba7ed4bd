/*
 * imp_gpu.h — C ABI of libimp_gpu.so: the B200 (sm_100a) implementation of IMP's decoded-pixel
 * hot path (RunJob steps 3-7, /root/reference/bridge.c:574-656): crop, resize, filter chain,
 * watermark alpha-composite, alpha flatten.
 *
 * This is the drop-in boundary below bridge.c. Host code stays C; every entry point takes plain
 * pointers and sizes (no CUDA, torch or C++ types), returns the reference's own IMP_* codes
 * (required.h:27-41) and never throws or exits. There is NO CPU fallback: without a usable CUDA
 * device every compute entry point returns IMP_ERROR_GPU.
 *
 * What each group replaces in the reference:
 *   imp_gpu_init_worker / imp_gpu_shutdown OnEnvStart / OnEnvDestroy      bridge.c:10-16 (no-ops there;
 *                                          called per worker from module.c:100-107, i.e. after fork): worker k
 *                                          takes device list[k % length] of IMP_GPU_DEVICES (below)
 *   imp_gpu_request + imp_gpu_config       the strings RunJob extracts from the query (bridge.c:346-372)
 *                                          and the Config fields the ops read (required.h:110-120)
 *   imp_gpu_plan_create                    argument validation of Crop (bridge.c:18-128), Resize
 *                                          (bridge.c:143-190), Filter + 14 callbacks (filters.c:43-455),
 *                                          Watermark placement (bridge.c:254-274): same grammar, same
 *                                          codes, same failing step, before any pixel is touched
 *   imp_gpu_run_host / _run_device         the per-frame loops bridge.c:576-656 for ONE frame
 *   imp_gpu_batch_*                        the same loops over album.Frames[] (GIF frames) and over
 *                                          concurrent requests: one fused launch per kernel variant
 *   imp_gpu_farm_run_host                  independent frames sharded round-robin over the GPUs of
 *                                          one box (no collective: nothing crosses GPUs)
 *   imp_gpu_batch_brightness_host /        Info (bridge.c:283-300) and ASCII (filters.c:486-522) after the frame loops:
 *   imp_gpu_batch_ascii_host               the brightness or the text comes back, not the frame
 * The reference-signature operator layer (Crop/Resize/Filter/Watermark/BlendWithPaper on IplImage)
 * is declared in imp_ops.h and is implemented on top of this ABI.
 *
 * IMP_GPU_DEVICES (environment): the devices this process may use, in order, as comma-separated decimal
 * ordinals ("4,0,5,1"); unset or empty means 0..n-1 for the n devices present. imp_gpu_init_worker maps
 * nginx worker k onto entry k % length, and the farm runs GPU g of its assignment on entry g. Read at each
 * of those calls; imp_gpu_init(device) ignores it.
 */
#ifndef IMP_GPU_H
#define IMP_GPU_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- return codes: required.h:27-41, plus one new code for CUDA failures (maps to HTTP 500) ---- */
#define IMP_OK                      0
#define IMP_ERROR_UNSUPPORTED       1
#define IMP_ERROR_MALLOC_FAILED     2
#define IMP_ERROR_INVALID_ARGS      50
#define IMP_ERROR_UPSCALE           51
#define IMP_ERROR_NO_SUCH_FILTER    52
#define IMP_ERROR_NO_SUCH_WATERMARK 53
#define IMP_ERROR_TOO_BIG_TARGET    54
#define IMP_ERROR_TOO_MUCH_FILTERS  55
#define IMP_ERROR_FEATURE_DISABLED  56
#define IMP_ERROR_GPU               100

/* ---- job steps: required.h:46-54 ---------------------------------------------------------------- */
#define IMP_STEP_CROP      3
#define IMP_STEP_RESIZE    4
#define IMP_STEP_FILTERING 5
#define IMP_STEP_WATERMARK 6
#define IMP_STEP_ENCODE    8

/* ---- resize interpolation override (extension; 0 keeps the reference rule bridge.c:190) --------- */
#define IMP_INTERP_REFERENCE 0   /* simple ? NN : (upscale ? CUBIC : AREA) */
#define IMP_INTERP_LINEAR    1   /* cv::INTER_LINEAR instead of CUBIC/AREA (north_star "bilinear") */

/* The decoded watermark as PrepareWatermark leaves it in the conf pool (RecoverInfo, required.h:101-108,
 * bridge.c:221-234) plus its placement (Position, required.h:86-91) and opacity (module.c directive). */
/* ---- encoder-side pixel prep folded into the final store (advancedio.c:65-101; SURVEY 8f-3) ------ */
#define IMP_PACK_NONE 0          /* rows top-down, channel count of the chain (what cvEncodeImage wants) */
#define IMP_PACK_FI24 24         /* IplToFI24: rows bottom-up, 3 bytes per pixel (alpha dropped) */
#define IMP_PACK_FI32 32         /* IplToFI32: rows bottom-up, 4 bytes per pixel (alpha 255 when the frame has none) */

typedef struct imp_gpu_watermark {
    const unsigned char* pixels;   /* RecoverInfo.Pointer: 8-bit B,G,R[,A] interleaved, host memory */
    int  width, height;            /* RecoverInfo.Size */
    int  channels;                 /* RecoverInfo.Channels: 3 or 4 */
    int  step;                     /* RecoverInfo.Step (bytes per row) */
    char gravity_x, gravity_y;     /* Position.GravityX/Y: 'l'|'c'|'r', 't'|'c'|'b' */
    int  offset_x, offset_y;       /* Position.OffsetX/Y */
    int  opacity;                  /* Config.WatermarkOpacity, 1..100 */
} imp_gpu_watermark;

/* The Config fields the hot path reads (required.h:110-120). */
typedef struct imp_gpu_config {
    unsigned int max_target_w, max_target_h;   /* MaxTargetDimensions (0 = unlimited) */
    int max_filters;                           /* MaxFiltersCount */
    int allow_experiments;                     /* AllowExperiments */
    const imp_gpu_watermark* watermark;        /* WatermarkInfo or NULL */
} imp_gpu_config;

/* What RunJob hands to steps 3-7 (bridge.c:318-372, 594, 642-656). Strings are the raw GET values,
 * NUL-terminated, caller-owned and never modified (the reference's in-place tokenising of `gravity`,
 * bridge.c:73, is not reproduced: every frame of a job sees the same string). */
typedef struct imp_gpu_request {
    const char*        crop;          /* "W,H[,gx,gy]" or NULL */
    const char*        gravity;       /* "gx,gy" or NULL */
    const char*        resize;        /* "W[,H[,up]]" or NULL */
    const char* const* filters;       /* filter_count strings "name=args" (text after "filter-") */
    int                filter_count;
    int                simple_resize; /* 1 when the encoder is GIF -> INTER_NN (bridge.c:594) */
    int                flatten;       /* 1 when the encoder has no alpha -> BlendWithPaper (bridge.c:642-656) */
    int                interp;        /* IMP_INTERP_* */
    int                pack;          /* IMP_PACK_*: encoder-side layout of the result (SURVEY 8f-3) */
} imp_gpu_request;

typedef struct imp_gpu_plan   imp_gpu_plan;    /* validated, lowered, device-resident job recipe */
typedef struct imp_gpu_batch  imp_gpu_batch;   /* a set of (plan, source, destination) jobs launched together */
typedef struct imp_gpu_ticket imp_gpu_ticket;  /* an asynchronous host batch in flight */

/* ---- lifetime ----------------------------------------------------------------------------------- */
/* Creates the CUDA context on `device` for this process (call after fork). Idempotent per device. */
int  imp_gpu_init(int device);
void imp_gpu_shutdown(void);
int  imp_gpu_device_count(void);
/* Selects which initialised device subsequent calls from THIS thread use. */
int  imp_gpu_set_device(int device);
/* The device worker `worker` takes (pure host logic, needs no device): *device = list[worker % length], where the list
 * is `devices` in IMP_GPU_DEVICES's syntax, or 0..n_devices-1 when `devices` is NULL or empty. IMP_ERROR_INVALID_ARGS
 * for a negative worker or a bad list (an empty or non-decimal entry, a trailing comma, an ordinal >= n_devices or
 * >= 16, a repeated ordinal, more than 16 entries; imp_gpu_last_error() names the entry); IMP_ERROR_GPU for
 * n_devices <= 0. *device = -1 on failure. */
int  imp_gpu_worker_device(int worker, int n_devices, const char* devices, int* device);
/* OnEnvStart of nginx worker `worker` (ngx_worker): counts the devices, maps the worker through imp_gpu_worker_device
 * with IMP_GPU_DEVICES from the environment, then imp_gpu_init on the result, which also makes it the calling thread's
 * device. *device (may be NULL) = the device, or -1 on failure; then nothing is initialised and compute calls fail
 * with IMP_ERROR_GPU as they do before any imp_gpu_init. */
int  imp_gpu_init_worker(int worker, int* device);
const char* imp_gpu_last_error(void);          /* thread-local text of the last IMP_ERROR_GPU or rejected device list */
/* Diagnostics: bounds assertions violated by the tile kernels on the current device since start-up, as a bit set. Always 0
 * for the release build; the debug build (python -m ngx_http_imgproc_b200.build --debug -> libimp_gpu_dbg.so, compiled
 * with -DIMP_DEBUG_BOUNDS) checks every staged-tile, lookup, out-stage and destination address the tile kernels form —
 * the stand-in for compute-sanitizer, which the GPU pool does not offer. Synchronises the device. */
unsigned imp_gpu_debug_flags(void);
/* Pixel-stage kernels launched by this library since process start (all devices). The host paths' window
 * re-pitch copy (short rows travel as one linear H2D copy and are laid out on the device) is not counted. */
unsigned long long imp_gpu_launch_count(void);

/* ---- overlays: PrepareWatermark (bridge.c:199-237) decodes the watermark ONCE per configuration --------- */
/* Registers the decoded overlay and uploads it to the current device (call from OnEnvStart, after imp_gpu_init; or
 * never: the first plan that uses an overlay registers it). Overlays are interned by CONTENT: every plan whose
 * config carries the same pixels shares one host copy and one device copy per GPU, so a request never re-uploads it.
 * Returns IMP_ERROR_NO_SUCH_WATERMARK for an unusable descriptor (what Watermark returns, bridge.c:240-242). */
int  imp_gpu_upload_watermark(const imp_gpu_watermark* wm);

/* ---- plans -------------------------------------------------------------------------------------- */
/* Validates `req` against a source frame of src_w x src_h x src_c (8-bit, c in {1,3,4}) exactly as the
 * reference's operators would, in the reference's order; on success returns IMP_OK and a plan, else the
 * reference's error code with *step = the IMP_STEP_* at which RunJob would have stopped. */
int  imp_gpu_plan_create(const imp_gpu_request* req, const imp_gpu_config* cfg,
                         int src_w, int src_h, int src_c, imp_gpu_plan** plan, int* step);
void imp_gpu_plan_destroy(imp_gpu_plan* plan);
/* Plans are immutable and reference counted: imp_gpu_plan_create serves a repeated (request, frame geometry, config)
 * from an LRU cache (128 entries; IMP_GPU_PLAN_CACHE=n in the environment, 0 disables) without re-running the
 * planner or touching the device; imp_gpu_plan_destroy drops the caller's reference. */
void imp_gpu_plan_cache_stats(unsigned long long* hits, unsigned long long* misses, int* entries);
void imp_gpu_plan_cache_clear(void);
void imp_gpu_plan_output(const imp_gpu_plan* plan, int* w, int* h, int* c);
/* Source window the plan actually reads (the crop window), for callers that upload only those rows. */
void imp_gpu_plan_source_window(const imp_gpu_plan* plan, int* x, int* y, int* w, int* h);
/* Number of kernel passes (1 unless a blur splits the chain) and algorithmic bytes (SURVEY §8d). */
int  imp_gpu_plan_passes(const imp_gpu_plan* plan);
unsigned long long imp_gpu_plan_algorithmic_bytes(const imp_gpu_plan* plan);

/* ---- one frame ---------------------------------------------------------------------------------- */
/* Host buffers: H2D of the crop window, kernels, D2H; synchronous. dst must hold out_h rows of dst_step. */
int  imp_gpu_run_host(imp_gpu_plan* plan, const unsigned char* src, int src_step,
                      unsigned char* dst, int dst_step);
/* Device buffers; asynchronous on `stream` (a cudaStream_t passed as void*, NULL = the library's stream for this
 * device). Any pitch at least one row long (src_w*src_c, out_w*out_c bytes) and any base are accepted, except that
 * 4-channel rows (a 4-channel source, a 4-channel or FI32 result) must have a pitch and a base that are multiples of 4;
 * anything else returns IMP_ERROR_INVALID_ARGS. Only the out_w*out_c bytes of each result row are written, never the
 * pitch padding. A source whose pitch is a multiple of 16 and whose image or crop window starts 16-byte aligned takes
 * the shared-memory tile kernels; any other source the general kernels, with the same results. imp_gpu_batch_add takes
 * the same buffers. */
int  imp_gpu_run_device(imp_gpu_plan* plan, const void* d_src, int src_pitch,
                        void* d_dst, int dst_pitch, void* stream);

/* ---- batches: GIF frames / concurrent requests ---------------------------------------------------- */
int  imp_gpu_batch_create(imp_gpu_batch** batch);
void imp_gpu_batch_destroy(imp_gpu_batch* batch);
int  imp_gpu_batch_clear(imp_gpu_batch* batch);
int  imp_gpu_batch_add(imp_gpu_batch* batch, imp_gpu_plan* plan, const void* d_src, int src_pitch,
                       void* d_dst, int dst_pitch);
/* Uploads the job table once (until the next add/clear) and launches one kernel per pass and kernel
 * variant over all jobs; asynchronous on `stream`. */
int  imp_gpu_batch_launch(imp_gpu_batch* batch, void* stream);
int  imp_gpu_batch_size(const imp_gpu_batch* batch);
unsigned long long imp_gpu_batch_algorithmic_bytes(const imp_gpu_batch* batch);
int  imp_gpu_batch_launches_per_run(const imp_gpu_batch* batch);

/* End to end over host buffers, on the current device; synchronous. The n jobs are cut into chunks of consecutive
 * jobs; each chunk's crop windows are copied H2D, the whole chunk runs as ONE grouped launch per kernel variant
 * (device job table, as imp_gpu_batch_launch), its results are copied D2H; `n_streams` (1..8) chunks are in flight on
 * their own streams and pinned staging lanes, so copies and kernels overlap. The frame loops of RunJob
 * (bridge.c:576-656) over album.Frames[] map onto one call. Every job is checked before any work starts: a NULL plan,
 * source or destination, or a step shorter than its row returns IMP_ERROR_INVALID_ARGS with nothing written. */
int  imp_gpu_batch_run_host(int n, imp_gpu_plan* const* plans, const unsigned char* const* srcs,
                            const int* src_steps, unsigned char* const* dsts, const int* dst_steps,
                            int n_streams);
/* Asynchronous form (SURVEY 8b-4 submit/wait): checks every job (a bad one: IMP_ERROR_INVALID_ARGS, no ticket), then
 * returns at once with a ticket; a helper thread drives the batch on the caller's current device. The argument arrays
 * are copied, the pixel buffers must stay valid until imp_gpu_batch_wait, which blocks, returns the batch's code and
 * frees the ticket. imp_gpu_batch_poll: 1 when finished, 0 while running. Every plan holds a reference until the wait,
 * so imp_gpu_plan_destroy right after the submit is safe. On any failure *ticket = NULL and nothing is written; n == 0
 * gives a ticket whose wait returns IMP_OK. imp_gpu_batch_brightness_submit_host, imp_gpu_batch_ascii_submit_host and
 * imp_gpu_gif_albums_submit_host (below) are the same for their calls, and poll and wait serve every kind of ticket. */
int  imp_gpu_batch_submit_host(int n, imp_gpu_plan* const* plans, const unsigned char* const* srcs,
                               const int* src_steps, unsigned char* const* dsts, const int* dst_steps,
                               int n_streams, imp_gpu_ticket** ticket);
int  imp_gpu_batch_poll(const imp_gpu_ticket* ticket);
int  imp_gpu_batch_wait(imp_gpu_ticket* ticket);
/* Same work sharded over devices 0..n_gpus-1 with one host thread per GPU; no inter-GPU traffic (nothing crosses
 * GPUs: docs/02 - Configuration.md:18 worker_processes is the reference's scale-out model). All devices are
 * initialised on demand. imp_gpu_farm_run_host is round-robin (job i -> GPU i mod n_gpus). With IMP_GPU_DEVICES set,
 * GPU g runs on its entry g, n_gpus larger than the list returns IMP_ERROR_GPU like n_gpus larger than the box, and a
 * bad list returns IMP_ERROR_INVALID_ARGS before any work. */
#define IMP_FARM_ROUND_ROBIN 0
#define IMP_FARM_SIZE_AWARE  1   /* largest job first onto the GPU with the fewest algorithmic bytes so far (mixed sizes) */
/* The assignment itself (pure host logic, needs no device): owner[i] = the GPU job i runs on under `policy`. */
int  imp_gpu_farm_assign(int n, imp_gpu_plan* const* plans, int n_gpus, int policy, int* owner);
int  imp_gpu_farm_run_host(int n, imp_gpu_plan* const* plans, const unsigned char* const* srcs,
                           const int* src_steps, unsigned char* const* dsts, const int* dst_steps,
                           int n_gpus, int n_streams);
int  imp_gpu_farm_run_host_policy(int n, imp_gpu_plan* const* plans, const unsigned char* const* srcs,
                                  const int* src_steps, unsigned char* const* dsts, const int* dst_steps,
                                  int n_gpus, int n_streams, int policy);

/* ---- format=json / format=text: an answer instead of the frame (SURVEY 8f-1, 8f-4) ------------------------------- */
/* format=json / format=text (bridge.c:659-677) for n jobs without their frames leaving the device: job i runs plans[i]
 * on srcs[i] exactly as imp_gpu_batch_run_host would, then brightness[i] = CalcPerceivedBrightness of the result
 * (filters.c:707-729; double sum, deterministic: the same frame gives the same bits whatever the batch, chunking or
 * n_streams), or texts[i] receives ASCII of the result (filters.c:486-522; args[i] as the reference takes it, NULL = the
 * 10-level ramp), imp_gpu_ascii_length(out_w, out_h) bytes. Synchronous, on the current device.
 * Each chunk of jobs costs one launch more than imp_gpu_batch_run_host, and only the floats or the texts cross the bus.
 * Every job is checked first; IMP_ERROR_INVALID_ARGS, with nothing written, for a NULL array or plan, a plan whose request
 * packs the result for FreeImage (pack != IMP_PACK_NONE: bottom-up rows would reverse the text) or text_caps[i] smaller
 * than the text. n == 0: IMP_OK. */
int  imp_gpu_batch_brightness_host(int n, imp_gpu_plan* const* plans, const unsigned char* const* srcs, const int* src_steps,
                                   float* brightness, int n_streams);
int  imp_gpu_batch_ascii_host(int n, imp_gpu_plan* const* plans, const unsigned char* const* srcs, const int* src_steps,
                              const char* const* args, unsigned char* const* texts, const long* text_caps, int n_streams);
/* Asynchronous forms of the two calls above, as imp_gpu_batch_submit_host is of imp_gpu_batch_run_host: every check of the
 * synchronous call runs at the submit (a packed answer or a text_caps[i] smaller than the text: IMP_ERROR_INVALID_ARGS,
 * no ticket, nothing written). The argument arrays are copied, each ASCII job's ramp is taken from args[i] at the submit;
 * the sources and the brightness / texts buffers must stay valid until imp_gpu_batch_wait. */
int  imp_gpu_batch_brightness_submit_host(int n, imp_gpu_plan* const* plans, const unsigned char* const* srcs,
                                          const int* src_steps, float* brightness, int n_streams, imp_gpu_ticket** ticket);
int  imp_gpu_batch_ascii_submit_host(int n, imp_gpu_plan* const* plans, const unsigned char* const* srcs, const int* src_steps,
                                     const char* const* args, unsigned char* const* texts, const long* text_caps,
                                     int n_streams, imp_gpu_ticket** ticket);

/* One frame already decoded: what Info() (bridge.c:283-300) prints as round(brightness*100). The reference accumulates
 * float32 in column-major order; the device sums in double (the same reduction as the batch call, so a frame gives the same
 * bits here as there when its rows are 16-byte aligned: the host form stages them so), and the values agree to ~1e-5
 * relative. Any base and pitch are accepted on the device. */
int  imp_gpu_brightness_device(const void* d_img, int pitch, int width, int height, int channels, float* brightness, void* stream);
int  imp_gpu_brightness_host(const unsigned char* img, int step, int width, int height, int channels, float* brightness);

/* ASCII of one frame. `args` as the reference takes it ("wide" selects the 70-level ramp, anything else the 10-level one).
 * Writes (width+1)*height-1 bytes: one character per pixel, rows separated by '\n'. The frame itself is not modified (the
 * reference converts it to HSV in place, filters.c:504, which nothing reads afterwards). */
long imp_gpu_ascii_length(int width, int height);
int  imp_gpu_ascii_host(const unsigned char* img, int step, int width, int height, int channels, const char* args,
                        unsigned char* out, long out_cap);

/* ---- SURVEY 8f-2: GIF canvas expansion (advancedio.c:195-248, LoadGIF's per-pixel loop) on the device ------------- */
/* A frame exactly as LoadGIF holds it after FreeImage_LockPage (+ConvertTo8Bits): 8-bit palette indices in FreeImage
 * scanline order (bottom-up), FrameLeft/FrameTop, DisposalMethod, FreeImage_GetTransparentIndex, the RGBQUAD palette. */
typedef struct imp_gpu_gif_frame {
    const unsigned char* indices;      /* host memory, height rows of `pitch` bytes, row 0 = bottom scanline */
    int pitch, width, height;
    int left, top;
    int dispose;                       /* advancedio.h:3-6: 0 unspecified, 1 leave, 2 background, 3 previous */
    int transparency_key;              /* -1 when the frame has none */
    const unsigned char* palette;      /* 256 x {B,G,R,reserved} */
} imp_gpu_gif_frame;
/* Expands n frames into n BGRA canvases of canvas_w x canvas_h laid out back to back on the device
 * (frame f at d_canvases + f*canvas_pitch*canvas_h), ready to be fed to imp_gpu_batch_add. `destructive` as
 * LoadGIF's isdestructive (replay disposal through the master index canvas). Uploads 1 byte per pixel.
 * The loop's accidents are kept: the off-by-one at x == left+width (advancedio.c:203) reads row[width] — the pad
 * byte or the next scanline's first index — as long as it lies inside the page's pitch*height block (so pass the
 * page bits as FreeImage holds them), and uncovered pixels of a page without a transparent colour read palette[-1],
 * FreeImage's biClrImportant == 256, i.e. {B,G,R} = {0,1,0} with alpha 0. `master` starts at 0 (uninitialised pool
 * memory in the reference, only observable when frame 0 has DISPOSAL_BACKGROUND and transparent pixels). */
int  imp_gpu_gif_expand_device(const imp_gpu_gif_frame* frames, int n, int canvas_w, int canvas_h, int destructive,
                               void* d_canvases, int canvas_pitch, void* stream);
int  imp_gpu_gif_expand_host(const imp_gpu_gif_frame* frames, int n, int canvas_w, int canvas_h, int destructive,
                             unsigned char* const* canvases, int canvas_step);
/* A whole GIF request end to end: LoadGIF's loop and RunJob's frame loop (bridge.c:576-656) without the canvases ever
 * visiting the host. The pages are uploaded as indices (1 byte per pixel), expanded on the device, and frame f runs
 * plans[f] (created for a canvas_w x canvas_h 4-channel source; usually one cached plan repeated) into dsts[f]; chunks
 * of frames are in flight on `n_streams` lanes exactly as in imp_gpu_batch_run_host. plans[f] == NULL: page f only takes
 * part in the disposal replay (LoadGIF's `page` request, advancedio.c:253-272, keeps the last page alone). Synchronous. */
int  imp_gpu_gif_album_run_host(const imp_gpu_gif_frame* frames, int n, int canvas_w, int canvas_h, int destructive,
                                imp_gpu_plan* const* plans, unsigned char* const* dsts, const int* dst_steps,
                                int n_streams);
/* Many GIF requests in one call: each album is what imp_gpu_gif_album_run_host takes. */
typedef struct imp_gpu_gif_album {
    const imp_gpu_gif_frame* pages; int n_pages;          /* as imp_gpu_gif_album_run_host takes them */
    int canvas_w, canvas_h, destructive;
    imp_gpu_plan* const* plans;                           /* n_pages entries; NULL = page only replayed (a `page` request) */
    unsigned char* const* dsts; const int* dst_steps;     /* n_pages entries, used where plans[f] != NULL */
} imp_gpu_gif_album;
/* Runs every album: each album's results are byte-identical to what imp_gpu_gif_album_run_host gives for that album
 * alone, whatever the neighbouring albums, their order or n_streams. Consecutive albums whose canvases fit 256 MB together
 * form a round (an album above that is a round alone): one upload of all their pages, one expansion launch, and one
 * chunked frame loop whose grouped launches span albums; rounds run one after another. Every album is checked before any
 * work (page and palette pointers, page geometry, each plan's source a canvas_w x canvas_h 4-channel canvas, destination
 * steps): one bad album returns IMP_ERROR_INVALID_ARGS and no destination of any album is written. n_albums == 0 returns
 * IMP_OK. Synchronous, on the current device. */
int  imp_gpu_gif_albums_run_host(const imp_gpu_gif_album* albums, int n_albums, int n_streams);
/* Asynchronous form, as imp_gpu_batch_submit_host is of imp_gpu_batch_run_host: every album is checked at the submit (one
 * bad album: IMP_ERROR_INVALID_ARGS, no ticket, nothing written). The album descriptors and their pages, plans, dsts and
 * dst_steps arrays are copied; the index planes, palettes and destinations must stay valid until imp_gpu_batch_wait. */
int  imp_gpu_gif_albums_submit_host(const imp_gpu_gif_album* albums, int n_albums, int n_streams, imp_gpu_ticket** ticket);

/* ---- memory helpers so a C host needs no CUDA headers --------------------------------------------- */
int  imp_gpu_malloc(void** d_ptr, size_t bytes);
int  imp_gpu_free(void* d_ptr);
int  imp_gpu_malloc_pitch(void** d_ptr, int* pitch, int width_bytes, int height);
int  imp_gpu_host_alloc(void** h_ptr, size_t bytes);      /* pinned */
int  imp_gpu_host_free(void* h_ptr);
int  imp_gpu_upload_2d(void* d_dst, int d_pitch, const void* h_src, int h_step, int width_bytes, int height, void* stream);
int  imp_gpu_download_2d(void* h_dst, int h_step, const void* d_src, int d_pitch, int width_bytes, int height, void* stream);
int  imp_gpu_sync(void* stream);                          /* NULL = whole device */

#ifdef __cplusplus
}
#endif
#endif /* IMP_GPU_H */
