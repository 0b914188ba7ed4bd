// imp_gif.cuh — GIF canvas expansion (SURVEY 8f-2; LoadGIF's loop, advancedio.c:195-248), written once for device and
// host: imp_gif_expand_kernel (imp_kernels.cu) runs imp_gif_expand_thread for every thread of its grid, and a CPU test
// harness (tests/test_gif_albums.py) runs the same function over the same packed table.
#pragma once
#include "imp_pixel.cuh"

#if defined(__CUDA_ARCH__)
#define IMP_GIF_LDG(p) __ldg(p)
#else
#define IMP_GIF_LDG(p) (*(p))
#endif

// Canvas pixel (x, y) of an album over its n pages, carrying the reference's `master` index for the disposal replay in a
// register; page f's pixel goes to canvases + f * canvas_bytes + y * cpitch + 4x.
IMP_HD void imp_gif_replay_pixel(const ImpGifFrame* pages, int n, int destructive, int x, int y,
                                 uint8_t* canvases, size_t canvas_bytes, int cpitch) {
    int master = 0;
    uint8_t* const end = canvases + (size_t)n * canvas_bytes;
    uint8_t* px = canvases + (size_t)y * cpitch + (size_t)x * 4;
    for (int f = 0; f < n; f++, px += canvas_bytes) {
        const ImpGifFrame fr = pages[f];
        const int rowidx = fr.h + fr.top - y - 1;
        int idx;
        // advancedio.c:203 tests `x > left + w`, so the column right of the frame reads row[w]: a pad byte of the
        // scanline or the first index of the next one. Reproduced while that byte is inside the page's pixel block.
        const int col = x - fr.left;
        if (rowidx < 0 || rowidx >= fr.h || col < 0 || col > fr.w || rowidx * fr.pitch + col >= fr.h * fr.pitch) idx = fr.key;
        else {
            const size_t off = (size_t)rowidx * fr.pitch + col;
            IMP_DBG(off < (size_t)fr.h * fr.pitch, 12);
            idx = IMP_GIF_LDG(fr.indices + off);
        }
        if (destructive) {
            if (fr.dispose == 2) {                       // GIF_DISPOSAL_BACKGROUND
                if (idx == fr.key) idx = 0; else master = idx;
            } else {                                     // LEAVE / PREVIOUS / UNSPECIFIED
                if (idx == fr.key && f > 0) idx = master; else master = idx;
            }
        }
        // idx is 0..255 or -1 (a page without a transparent colour). palette[-1] aliases FreeImage's biClrImportant == 256,
        // i.e. the bytes {0,1,0,0} (advancedio.c:232 with FreeImage_GetTransparentIndex == -1).
        uint32_t q = 0x100u;
        if (idx >= 0 && idx < 256) q = IMP_GIF_LDG(reinterpret_cast<const uint32_t*>(fr.palette) + idx);
        IMP_DBG(px + 4 <= end && x * 4 + 4 <= cpitch, 13);
        *reinterpret_cast<uint32_t*>(px) = (q & 0xFFFFFFu) | (idx == fr.key ? 0u : 0xFF000000u);
    }
}

// Thread `lane` of expansion block `block`: the block's album is the last one whose blk0 <= block, and the album's pixels
// are enumerated row by row from its first block, so a narrow canvas fills whole blocks with its following rows.
IMP_HD void imp_gif_expand_thread(const ImpGifAlbum* albums, int n_albums, const ImpGifFrame* pages, uint8_t* arena,
                                  size_t arena_bytes, long long block, int lane) {
    int lo = 0, hi = n_albums - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (albums[mid].blk0 <= block) lo = mid; else hi = mid - 1;
    }
    const ImpGifAlbum a = albums[lo];
    const long long p = (block - a.blk0) * IMP_GIF_THREADS + lane;
    if (p >= (long long)a.cw * a.ch) return;
    const int y = (int)(p / a.cw), x = (int)(p - (long long)y * a.cw);
    const size_t canvas_bytes = (size_t)a.pitch * a.ch;
    IMP_DBG(a.canvas_off + (size_t)a.n * canvas_bytes <= arena_bytes, 13);
    imp_gif_replay_pixel(pages + a.first, a.n, a.destructive, x, y, arena + a.canvas_off, canvas_bytes, a.pitch);
}
