// bsx_map_se_wide.cu -- the single-end WGBS kernel for indexes built with -v >= 8: 16-byte context entries (32 + 32 bases
// around the seed) staged and tested in one go, where 32 bases would let a fifth of config 5's candidates through.
struct MapKernel {
    static constexpr bool pe = false, rrbs = false, wide = true;
    static constexpr bool owner_sched = false;
    static constexpr bool run_advance = true;      // long lists (-v 15 repeats), see bsx_map_se_rrbs.cu
};
#include "bsx_map_impl.cuh"

namespace {
__global__ void __launch_bounds__(BSX_WARPS_PER_CTA * 32, 5) bsx_map_se_wide_kernel(const __grid_constant__ MapArgs A) { map_se(A); }
}
extern const void *const bsx_map_se_wide = (const void *)bsx_map_se_wide_kernel;
