// imp_k_gather.cu — translation unit of the destination-tiled plain gathers (imp_gathertile.cuh): index map, NN, LINEAR.
#include "imp_internal.h"
#include "imp_gathertile.cuh"

cudaError_t imp_upload_tables_gather() { return imp_upload_tables_tu(); }
unsigned imp_debug_flags_gather() { return imp_debug_flags_tu(); }

template <int KIND>
static cudaError_t launch_gather_sc(const ImpLaunchGroup& g, const ImpJob* d_jobs, const ImpJob* one, cudaStream_t st) {
    using imp_tiles::imp_gather_tile_kernel;
    const dim3 block(imp_tiles::GATHER_THREADS);
    switch (g.sc) {
        case 1: return g.flavour ? imp_launch_jobs<imp_gather_tile_kernel<1, KIND, true>>(g, block, d_jobs, one, st) : imp_launch_jobs<imp_gather_tile_kernel<1, KIND, false>>(g, block, d_jobs, one, st);
        case 3: return g.flavour ? imp_launch_jobs<imp_gather_tile_kernel<3, KIND, true>>(g, block, d_jobs, one, st) : imp_launch_jobs<imp_gather_tile_kernel<3, KIND, false>>(g, block, d_jobs, one, st);
        case 4: return g.flavour ? imp_launch_jobs<imp_gather_tile_kernel<4, KIND, true>>(g, block, d_jobs, one, st) : imp_launch_jobs<imp_gather_tile_kernel<4, KIND, false>>(g, block, d_jobs, one, st);
    }
    return cudaErrorInvalidValue;
}

cudaError_t imp_launch_gather_tile(const ImpLaunchGroup& g, const ImpJob* d_jobs, const ImpJob* one, cudaStream_t st) {
    switch (g.kind) {
        case IMP_G_COPY:   return launch_gather_sc<IMP_G_COPY>(g, d_jobs, one, st);
        case IMP_G_NN:     return launch_gather_sc<IMP_G_NN>(g, d_jobs, one, st);
        case IMP_G_LINEAR: return launch_gather_sc<IMP_G_LINEAR>(g, d_jobs, one, st);
    }
    return cudaErrorInvalidValue;
}
