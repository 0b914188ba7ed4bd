// imp_transfer.cpp — how the chunked host path moves a batch over the link: where the batch is cut into chunks, and
// how each job's source reaches the device and its result comes back. Pure host logic (no CUDA call): the caller says
// which buffers are page-locked, so tests/test_transfer_plan.py pins every decision on the CPU.
#include "imp_internal.h"
#include <algorithm>

// The size of an ASCII answer (include/imp_gpu.h). Defined here because it is a rule of the layout below (an ASCII job's
// result bytes), so the layout and its CPU test need nothing from the CUDA side.
extern "C" long imp_gpu_ascii_length(int width, int height) { return (long)(width + 1) * height - 1; }

namespace {
// What a job moves: its crop window at the device pitch and its result.
size_t job_bytes(const imp_gpu_plan* p) {
    return (size_t)align16(p->win_w * p->src_c) * p->win_h + (size_t)p->out_w * p->out_c * p->out_h;
}
}  // namespace

// Uploads of different lanes issued together are time-sliced by the copy engines: every chunk's upload then ends at the
// END of all uploads and nothing overlaps the way back. The runtime therefore chains each chunk's uploads behind the
// previous chunk's, and a call is cut into at least 2 chunks per lane when its bytes allow (>= 4 MB per chunk), so that
// the pipeline has stages to overlap. Small batches are spread over the lanes instead of filling one chunk.
std::vector<int> imp_chunk_bounds(const ImpHostJob* jobs, int n, int n_streams) {
    n_streams = std::max(1, std::min(n_streams, 8));
    size_t total = 0;
    for (int i = 0; i < n; i++) total += job_bytes(jobs[i].plan);
    const size_t chunk_bytes = std::min(IMP_CHUNK_BYTES, std::max<size_t>(4u << 20, total / (2 * (size_t)n_streams)));
    const int max_jobs = std::max(1, std::min(IMP_CHUNK_JOBS, (n + n_streams - 1) / n_streams));
    std::vector<int> bounds{0};
    for (int i = 0; i < n;) {
        int e = i; size_t bytes = 0;
        while (e < n && e - i < max_jobs) {
            const size_t need = job_bytes(jobs[e].plan);
            if (e > i && bytes + need > chunk_bytes) break;
            bytes += need; e++;
        }
        bounds.push_back(e);
        i = e;
    }
    return bounds;
}

ImpChunkLayout imp_chunk_layout(const ImpHostJob* jobs, int m, ImpResult kind, bool resident, const bool* src_pinned, const bool* dst_pinned) {
    ImpChunkLayout c;
    c.jobs.resize(m);
    for (int k = 0; k < m; k++) {
        const ImpHostJob& j = jobs[k];
        const imp_gpu_plan* p = j.plan;
        ImpJobLayout& l = c.jobs[k];
        l = ImpJobLayout{};
        const size_t in_row = (size_t)p->win_w * p->src_c, out_row = (size_t)p->out_w * p->out_c;
        l.in_pitch = align16((int)in_row); l.out_pitch = align16((int)out_row);
        l.in_off = c.in_total;
        if (!resident) c.in_total += align256((size_t)l.in_pitch * p->win_h);             // landing zone of the crop window
        l.out_off = c.out_total; c.out_total += align256((size_t)l.out_pitch * p->out_h);
        l.res_bytes = kind == ImpResult::Frame ? out_row * p->out_h
                    : kind == ImpResult::Ascii ? (size_t)imp_gpu_ascii_length(p->out_w, p->out_h) : sizeof(float);

        // A 2-D host-to-device copy pays ~0.15 us per row whatever its width (measured: 3.5 KB rows move at 23 GB/s, 14 KB
        // rows at the link's 54 GB/s). Short rows therefore travel as ONE linear copy of the rows the window touches (full
        // width) and a small kernel extracts / re-pitches the window on the device; a window that IS the frame's contiguous
        // rows is one linear copy whatever its row length.
        const bool short_rows = j.src_step <= 8192;
        if (resident) {
            l.src = ImpRoute::Resident;
        } else if (!src_pinned[k]) {
            l.src = ImpRoute::Staged;
            l.hin_off = c.hin_total; c.hin_total += align256((size_t)l.in_pitch * p->win_h);
            // a lone large window is staged and uploaded in row slices, so that the copy engine works on slice k while the
            // cores stage slice k+1 (cfg2's 29 MB window: 1.16 -> 1.04 ms); smaller ones do not repay the extra dispatches
            l.slices = std::min(p->win_h, (m > 1 || in_row * p->win_h < (16u << 20)) ? 1 : 4);
        } else if (j.src_step == l.in_pitch && p->win_x == 0 && (short_rows || in_row == (size_t)l.in_pitch)) {
            l.src = ImpRoute::Linear;
        } else if (short_rows) {
            l.src = ImpRoute::LinearRepitch;
        } else {
            l.src = ImpRoute::Rows2D;
        }
        if (l.src == ImpRoute::Linear || l.src == ImpRoute::LinearRepitch)
            l.lin_bytes = (size_t)(p->win_h - 1) * j.src_step + (size_t)p->win_x * p->src_c + in_row;
        if (l.src == ImpRoute::LinearRepitch) { l.stage_off = c.stage_total; c.stage_total += align256(l.lin_bytes); }

        if (!dst_pinned[kind == ImpResult::Brightness ? 0 : k]) {
            l.dst = ImpRoute::Staged;
            l.hout_off = c.hout_total;
            // brightness answers are staged back to back: the chunk's floats come back in one copy
            c.hout_total += kind == ImpResult::Brightness ? sizeof(float) : align256(l.res_bytes);
        } else if (kind != ImpResult::Frame) {
            l.dst = ImpRoute::Direct;
        } else {
            l.dst = j.dst_step == l.out_pitch ? ImpRoute::Linear : ImpRoute::Rows2D;
        }
    }
    return c;
}
