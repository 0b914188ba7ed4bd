// transfer_shim.cpp — a C face over imp_transfer.cpp (the chunk cutter and the transfer layout of the host path) for
// tests/test_transfer_plan.py. Plans are bare: only the geometry fields those functions read are filled, so neither the
// planner nor a device is involved.
#include "../../ngx_http_imgproc_b200/csrc/imp_internal.h"

namespace {
std::vector<ImpHostJob> jobs_of(int n, imp_gpu_plan* const* plans, const int* src_steps, const int* dst_steps) {
    std::vector<ImpHostJob> v(n);
    for (int i = 0; i < n; i++) v[i] = ImpHostJob{plans[i], nullptr, src_steps ? src_steps[i] : 0, nullptr, dst_steps ? dst_steps[i] : 0, false};
    return v;
}
}  // namespace

extern "C" {

imp_gpu_plan* shim_plan(int src_w, int src_h, int src_c, int win_x, int win_y, int win_w, int win_h, int out_w, int out_h, int out_c) {
    imp_gpu_plan* p = new imp_gpu_plan();
    p->src_w = src_w; p->src_h = src_h; p->src_c = src_c;
    p->win_x = win_x; p->win_y = win_y; p->win_w = win_w; p->win_h = win_h;
    p->out_w = out_w; p->out_h = out_h; p->out_c = out_c;
    p->algo_bytes = 0;
    return p;
}
void shim_plan_free(imp_gpu_plan* p) { delete p; }

// imp_chunk_bounds into out[0 .. n+1); returns how many boundaries there are
int shim_bounds(int n, imp_gpu_plan* const* plans, int n_streams, int* out) {
    const std::vector<ImpHostJob> jobs = jobs_of(n, plans, nullptr, nullptr);
    const std::vector<int> b = imp_chunk_bounds(jobs.data(), n, n_streams);
    for (size_t i = 0; i < b.size(); i++) out[i] = b[i];
    return (int)b.size();
}

// imp_chunk_layout: per job 12 values (src route, dst route, in_pitch, out_pitch, in_off, out_off, lin_bytes, stage_off,
// hin_off, hout_off, res_bytes, slices), then the 5 totals (in, out, stage, h_in, h_out)
void shim_layout(int m, imp_gpu_plan* const* plans, const int* src_steps, const int* dst_steps, int kind, int resident,
                 const unsigned char* src_pinned, const unsigned char* dst_pinned, long long* per_job, long long* totals) {
    const std::vector<ImpHostJob> jobs = jobs_of(m, plans, src_steps, dst_steps);
    std::unique_ptr<bool[]> sp(new bool[m + 1]), dp(new bool[m + 1]);
    for (int k = 0; k < m; k++) { sp[k] = src_pinned[k] != 0; dp[k] = dst_pinned[k] != 0; }
    const ImpChunkLayout c = imp_chunk_layout(jobs.data(), m, (ImpResult)kind, resident != 0, sp.get(), dp.get());
    for (int k = 0; k < m; k++) {
        const ImpJobLayout& l = c.jobs[k];
        const long long v[12] = {(long long)l.src, (long long)l.dst, l.in_pitch, l.out_pitch, (long long)l.in_off, (long long)l.out_off,
                                 (long long)l.lin_bytes, (long long)l.stage_off, (long long)l.hin_off, (long long)l.hout_off,
                                 (long long)l.res_bytes, l.slices};
        for (int f = 0; f < 12; f++) per_job[12 * k + f] = v[f];
    }
    const long long t[5] = {(long long)c.in_total, (long long)c.out_total, (long long)c.stage_total, (long long)c.hin_total, (long long)c.hout_total};
    for (int f = 0; f < 5; f++) totals[f] = t[f];
}

}  // extern "C"
