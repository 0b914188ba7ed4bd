/*
 * imp_ops.h — the reference's operator signatures (bridge.h:4-7, filters.h:1,30) on top of libimp_gpu.so.
 *
 * RunJob (bridge.c:574-656) calls Crop, Resize, Filter, Watermark, BlendWithPaper one after another, each
 * walking the whole frame on the CPU. The functions below keep those names' arguments, return codes and
 * "image unchanged on error" behaviour, but only RECORD the operation (after validating it exactly like the
 * reference does) and fix up the IplImage header (width/height/nChannels/widthStep/imageSize) so the next
 * operator sees the geometry it expects. imp_Flush() then runs everything recorded for that frame as ONE
 * fused GPU plan (one H2D of the crop window, one kernel unless a blur splits the chain, one D2H) and
 * replaces the frame. ngx_http_imgproc_b200/dropin/imp_dropin.c wraps these under the reference's exact names and
 * prototypes (Crop, Resize(…, Config*, …), the 14 filter callbacks, Watermark, BlendWithPaper) for a module that is
 * compiled against its own required.h; INTEGRATION.md shows what changes in bridge.c / filters.c (call sites: nothing).
 *
 *   reference (file:line)                                replacement
 *   int Crop(IplImage**, char*, char*)       bridge.c:18   imp_Crop
 *   int Resize(IplImage**, char*, Config*, int) bridge.c:143 imp_Resize  (Config -> imp_gpu_config, see INTEGRATION.md)
 *   int Filter(IplImage**, char*, int)       filters.c:43  imp_Filter
 *   int Watermark(IplImage*, Config*)        bridge.c:239  imp_Watermark
 *   void BlendWithPaper(IplImage*)           filters.c:666 imp_BlendWithPaper
 *   gray->BGR block                          bridge.c:613-618  implicit (a 1-channel frame leaves imp_Flush as BGR, also when nothing was recorded)
 *   (none)                                   before bridge.c:659   imp_Flush / imp_FlushAll
 *   CalcPerceivedBrightness / ASCII          bridge.c:296, 668     imp_Brightness / imp_Ascii (the frame stays on the device)
 *   LoadGIF's canvas loop                    advancedio.c:195-248  imp_FlushAllGif (pages expanded on the device; imp_AlbumGifPage in the drop-in)
 *   cvReleaseImage on an error path          bridge.c:714-722  imp_Discard first
 *
 * Not reproduced on purpose: Crop tokenising `gravity` in place (bridge.c:73), which makes the 2nd frame of a
 * GIF fail with 400; the double free of a frame when a filter fails after flip/rotate/gray->BGR
 * (bridge.c:609-627).
 */
#ifndef IMP_OPS_H
#define IMP_OPS_H

#include "imp_gpu.h"

#ifdef __cplusplus
extern "C" {
#endif

/* IplImage: use OpenCV's own definition when <opencv/cv.h> (types_c.h) was included first; otherwise a
 * layout-identical declaration (OpenCV 2.4 types_c.h; sizeof == 144 on x86-64). */
#if !defined(__OPENCV_CORE_TYPES_H__) && !defined(OPENCV_CORE_TYPES_H) && !defined(IMP_ORACLE_SHIM_CV_H) && !defined(IMP_HAVE_IPLIMAGE)
#define IMP_HAVE_IPLIMAGE
typedef struct _IplROI { int coi, xOffset, yOffset, width, height; } IplROI;
typedef struct _IplImage {
    int nSize, ID, nChannels, alphaChannel, depth;
    char colorModel[4], channelSeq[4];
    int dataOrder, origin, align, width, height;
    struct _IplROI* roi;
    struct _IplImage* maskROI;
    void* imageId;
    void* tileInfo;
    int imageSize;
    char* imageData;
    int widthStep;
    int BorderMode[4], BorderConst[4];
    char* imageDataOrigin;
} IplImage;
#endif

/* How imp_Flush obtains / frees frames: pass thin wrappers of cvCreateImage / cvReleaseImage so that frames
 * stay owned by OpenCV's allocator (RunJob releases them at bridge.c:714-722). */
typedef IplImage* (*imp_ops_create_image_fn)(int width, int height, int depth, int channels);
typedef void (*imp_ops_release_image_fn)(IplImage** image);
void imp_ops_set_image_allocator(imp_ops_create_image_fn create, imp_ops_release_image_fn release);

int  imp_Crop(IplImage** pointer, char* args, char* gravity);
int  imp_Resize(IplImage** pointer, char* args, const imp_gpu_config* config, int simple);
int  imp_Filter(IplImage** pointer, char* request, int allowExperiments);
int  imp_Watermark(IplImage* image, const imp_gpu_config* config);
int  imp_BlendWithPaper(IplImage* image);          /* the reference returns void; 0 here unless the frame is unknown */

/* Executes what was recorded for *pointer. On success *pointer holds the result (a new frame from the
 * allocator when size or channel count changed, the old one released). Returns IMP_OK or IMP_ERROR_GPU. */
int  imp_Flush(IplImage** pointer);
/* Same for all frames of an album in one overlapped batch (GIF frames; bridge.c:576-656 loops). */
int  imp_FlushAll(IplImage** frames, int count);
/* The album of a GIF whose canvases were NOT expanded on the host: frames[] are the canvas-sized 4-channel IplImages
 * LoadGIF created (advancedio.c:188-193; their pixels are never read), pages[] the FreeImage pages its per-pixel loop
 * (:195-248) would have walked. Expands on the device and runs what was recorded for each frame (a frame with nothing
 * recorded just receives its canvas). n_pages == count: frame i is page i. count == 1 < n_pages: LoadGIF's `page`
 * request (:264-272) — the frame is the LAST page, the earlier ones are only replayed for their disposal. */
int  imp_FlushAllGif(IplImage** frames, int count, const imp_gpu_gif_frame* pages, int n_pages, int destructive);
/* Brightness / ASCII of what imp_Flush would leave in `image`, computed on the device; the frame is not brought back.
 * What was recorded for `image` STAYS recorded: a later imp_Flush still produces the pixels, imp_Discard still works.
 * A 1-channel frame is answered as BGR, recorded operators or not (imp_Flush promotes it, bridge.c:613-618). `args` and
 * out_cap as imp_gpu_ascii_host takes them. Returns IMP_OK, IMP_ERROR_INVALID_ARGS or IMP_ERROR_GPU. */
int  imp_Brightness(IplImage* image, float* brightness);
int  imp_Ascii(IplImage* image, const char* args, unsigned char* out, long out_cap);
/* Forget anything recorded for `image` (call before releasing a frame that was never flushed). */
void imp_Discard(IplImage* image);
/* Number of operations currently recorded for `image` (0 = pixels are up to date). */
int  imp_ops_pending(const IplImage* image);

#ifdef __cplusplus
}
#endif
#endif /* IMP_OPS_H */
