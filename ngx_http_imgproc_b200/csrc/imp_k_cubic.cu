// imp_k_cubic.cu — translation unit of the INTER_CUBIC tile kernel (imp_cubic.cuh).
#include "imp_internal.h"
#include "imp_cubic.cuh"

cudaError_t imp_upload_tables_cubic() { return imp_upload_tables_tu(); }
unsigned imp_debug_flags_cubic() { return imp_debug_flags_tu(); }

cudaError_t imp_launch_cubic_tile(const ImpLaunchGroup& g, const ImpJob* d_jobs, const ImpJob* one, cudaStream_t st) {
    using imp_tiles::imp_cubic_tile_kernel;
    const dim3 block(imp_tiles::CUBIC_THREADS);
    switch (g.sc) {
        case 1: return g.flavour ? imp_launch_jobs<imp_cubic_tile_kernel<1, true>>(g, block, d_jobs, one, st) : imp_launch_jobs<imp_cubic_tile_kernel<1, false>>(g, block, d_jobs, one, st);
        case 3: return g.flavour ? imp_launch_jobs<imp_cubic_tile_kernel<3, true>>(g, block, d_jobs, one, st) : imp_launch_jobs<imp_cubic_tile_kernel<3, false>>(g, block, d_jobs, one, st);
        case 4: return g.flavour ? imp_launch_jobs<imp_cubic_tile_kernel<4, true>>(g, block, d_jobs, one, st) : imp_launch_jobs<imp_cubic_tile_kernel<4, false>>(g, block, d_jobs, one, st);
    }
    return cudaErrorInvalidValue;
}
