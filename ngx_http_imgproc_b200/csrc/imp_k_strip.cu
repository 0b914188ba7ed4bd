// imp_k_strip.cu — translation unit of the persistent TMA strip kernels (imp_tiles.cuh): INTER_AREA fractional / integer.
#include "imp_internal.h"
#include "imp_tiles.cuh"

cudaError_t imp_upload_tables_strip() { return imp_upload_tables_tu(); }
unsigned imp_debug_flags_strip() { return imp_debug_flags_tu(); }

template <int SC, int MODE>
static cudaError_t launch_strip(const ImpLaunchGroup& g, const ImpJob* d_jobs, const ImpJob* one, cudaStream_t st) {
    using imp_tiles::imp_strip_kernel;
    const dim3 block(imp_tiles::STRIP_THREADS);
    switch (g.flavour) {
        case 1:  return imp_launch_jobs<imp_strip_kernel<SC, MODE, 1>>(g, block, d_jobs, one, st, g.param);
        case 2:  return imp_launch_jobs<imp_strip_kernel<SC, MODE, 2>>(g, block, d_jobs, one, st, g.param);
        default: return imp_launch_jobs<imp_strip_kernel<SC, MODE, 0>>(g, block, d_jobs, one, st, g.param);
    }
}

template <int MODE>
static cudaError_t launch_strip_sc(const ImpLaunchGroup& g, const ImpJob* d_jobs, const ImpJob* one, cudaStream_t st) {
    switch (g.sc) {
        case 1: return launch_strip<1, MODE>(g, d_jobs, one, st);
        case 3: return launch_strip<3, MODE>(g, d_jobs, one, st);
        case 4: return launch_strip<4, MODE>(g, d_jobs, one, st);
    }
    return cudaErrorInvalidValue;
}

// strip kernel modes (imp_tiles.cuh): 0 fractional INTER_AREA, 1 integer INTER_AREA, 3 INTER_LINEAR
cudaError_t imp_launch_strip(const ImpLaunchGroup& g, const ImpJob* d_jobs, const ImpJob* one, cudaStream_t st) {
    switch (g.kind) {
        case IMP_G_AREA_FRAC: return launch_strip_sc<0>(g, d_jobs, one, st);
        case IMP_G_AREA_INT:  return launch_strip_sc<1>(g, d_jobs, one, st);
        case IMP_G_LINEAR:    return launch_strip_sc<3>(g, d_jobs, one, st);
    }
    return cudaErrorInvalidValue;
}
