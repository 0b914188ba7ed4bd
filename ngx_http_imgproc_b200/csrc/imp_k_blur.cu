// imp_k_blur.cu — translation unit of the fused Gaussian blur tile kernel (imp_blur.cuh).
#include "imp_internal.h"
#include "imp_blur.cuh"

cudaError_t imp_upload_tables_blur() { return imp_upload_tables_tu(); }
unsigned imp_debug_flags_blur() { return imp_debug_flags_tu(); }

template <int SC, int R>
static cudaError_t launch_blur_tile(const ImpLaunchGroup& g, const ImpJob* d_jobs, const ImpJob* one, cudaStream_t st) {
    using imp_tiles::imp_blur_tile_kernel;
    const dim3 block(imp_tiles::BLUR_THREADS);
    return g.flavour ? imp_launch_jobs<imp_blur_tile_kernel<SC, R, true>>(g, block, d_jobs, one, st)
                     : imp_launch_jobs<imp_blur_tile_kernel<SC, R, false>>(g, block, d_jobs, one, st);
}

template <int SC>
static cudaError_t launch_blur_tile_r(const ImpLaunchGroup& g, const ImpJob* d_jobs, const ImpJob* one, cudaStream_t st) {
    switch (g.param) {                                     // tap radius
        case 3:  return launch_blur_tile<SC, 3>(g, d_jobs, one, st);
        case 6:  return launch_blur_tile<SC, 6>(g, d_jobs, one, st);
        case 9:  return launch_blur_tile<SC, 9>(g, d_jobs, one, st);
        case 12: return launch_blur_tile<SC, 12>(g, d_jobs, one, st);
    }
    return cudaErrorInvalidValue;
}

cudaError_t imp_launch_blur_tile(const ImpLaunchGroup& g, const ImpJob* d_jobs, const ImpJob* one, cudaStream_t st) {
    if (g.sc == 3) return launch_blur_tile_r<3>(g, d_jobs, one, st);
    if (g.sc == 4) return launch_blur_tile_r<4>(g, d_jobs, one, st);
    return cudaErrorInvalidValue;
}
