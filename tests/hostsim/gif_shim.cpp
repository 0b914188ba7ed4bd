// gif_shim.cpp — a C face over the GIF album part of imp_transfer.cpp (the round cutter and the round pack) and over the
// expansion's per-thread code (imp_gif.cuh) for tests/test_gif_albums.py. Built together with imp_transfer.cpp (and
// transfer_shim.cpp, whose chunk cutter the launch-count test restates); neither the planner nor a device is involved.
#include "../../ngx_http_imgproc_b200/csrc/imp_internal.h"
#include "../../ngx_http_imgproc_b200/csrc/imp_gif.cuh"
#include <string.h>

extern "C" {

// imp_gif_round_bounds into out[0 .. n+1) (only each album's canvas_w, canvas_h and n_pages are read); returns how many
// boundaries there are
int shim_gif_round_bounds(int n, const imp_gpu_gif_album* albums, int* out) {
    const std::vector<int> b = imp_gif_round_bounds(albums, n);
    for (size_t i = 0; i < b.size(); i++) out[i] = b[i];
    return (int)b.size();
}

// Albums [0, n) expanded as ONE round on the CPU: imp_gif_round_layout, imp_gif_pack_page into one host block (the "device"
// pointers are host pointers), then imp_gif_expand_thread for every thread of the launch's grid, the code
// imp_gif_expand_kernel compiles. canvases[a] receives album a's pages, canvas_h rows of 4 * canvas_w bytes each, back to
// back. Returns the grid's block count.
long long shim_gif_expand(int n, const imp_gpu_gif_album* albums, unsigned char* const* canvases) {
    const ImpGifRound r = imp_gif_round_layout(albums, n);
    std::vector<uint8_t> pack(r.pack_bytes + 16), arena(r.arena_bytes + 16, 0xCD);
    uint8_t* h = pack.data() + ((16 - ((uintptr_t)pack.data() & 15)) & 15);
    uint8_t* ar = arena.data() + ((16 - ((uintptr_t)arena.data() & 15)) & 15);
    for (int k = 0; k < (int)r.pages.size(); k++)
        imp_gif_pack_page(r, k, h, h, [](uint8_t* d, const uint8_t* s, size_t b) { memcpy(d, s, b); });
    const ImpGifAlbum* tab = reinterpret_cast<const ImpGifAlbum*>(h);
    const ImpGifFrame* pages = reinterpret_cast<const ImpGifFrame*>(h + r.page_off);
    for (long long b = 0; b < r.blocks; b++)
        for (int t = 0; t < IMP_GIF_THREADS; t++) imp_gif_expand_thread(tab, n, pages, ar, r.arena_bytes, b, t);
    for (int a = 0; a < n; a++) {
        const ImpGifAlbum& A = r.albums[a];
        const size_t row = (size_t)A.cw * 4;
        for (int f = 0; f < A.n; f++)
            for (int y = 0; y < A.ch; y++)
                memcpy(canvases[a] + ((size_t)f * A.ch + y) * row, ar + A.canvas_off + ((size_t)f * A.ch + y) * A.pitch, row);
    }
    return r.blocks;
}

}  // extern "C"
