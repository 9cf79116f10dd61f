// bsx_map_pe_wide.cu -- the paired-end WGBS kernel for indexes built with -v >= 8 (16-byte context entries).
struct MapKernel {
    static constexpr bool pe = true, rrbs = false, wide = true;
    static constexpr bool owner_sched = false;
    static constexpr bool run_advance = true;      // long lists, see bsx_map_se_rrbs.cu
};
#include "bsx_map_impl.cuh"

namespace {
__global__ void __launch_bounds__(BSX_WARPS_PER_CTA * 32, 4) bsx_map_pe_wide_kernel(const __grid_constant__ MapArgs A) { map_pe(A); }
}
extern const void *const bsx_map_pe_wide = (const void *)bsx_map_pe_wide_kernel;
