// bsx_map_se_rrbs.cu -- the single-end RRBS (-D) mapping kernel: same source, RRBS fixed at compile time.
struct MapKernel {
    static constexpr bool pe = false, rrbs = true, wide = false;
    static constexpr bool owner_sched = false;
    // rounds that stay inside one long list advance the previous schedule instead of rebuilding it: pays where lists run
    // to thousands of entries (config 4 +2 %, config 5 +9 %), costs 1-3 % on configs 2 / 3
    static constexpr bool run_advance = true;
};
#include "bsx_map_impl.cuh"

namespace {
__global__ void __launch_bounds__(BSX_WARPS_PER_CTA * 32, 5) bsx_map_se_rrbs_kernel(const __grid_constant__ MapArgs A) { map_se(A); }
}
extern const void *const bsx_map_se_rrbs = (const void *)bsx_map_se_rrbs_kernel;
