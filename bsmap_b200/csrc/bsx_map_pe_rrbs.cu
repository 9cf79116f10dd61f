// bsx_map_pe_rrbs.cu -- the paired-end RRBS (-D) mapping kernel: same source, RRBS fixed at compile time.
struct MapKernel {
    static constexpr bool pe = true, rrbs = true, wide = false;
    static constexpr bool owner_sched = false;
    static constexpr bool run_advance = true;      // long lists, see bsx_map_se_rrbs.cu
};
#include "bsx_map_impl.cuh"

namespace {
__global__ void __launch_bounds__(BSX_WARPS_PER_CTA * 32, 4) bsx_map_pe_rrbs_kernel(const __grid_constant__ MapArgs A) { map_pe(A); }
}
extern const void *const bsx_map_pe_rrbs = (const void *)bsx_map_pe_rrbs_kernel;
