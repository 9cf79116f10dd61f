// bsx_map_se.cu -- the single-end WGBS mapping kernel (SingleAlign::Do_Batch): RRBS and wide-context code compiled out
// (the kernel is instruction-cache and register sensitive: 90 KB of SASS with RRBS, -7 % with the wide-context registers
// live in the list loop).
struct MapKernel {
    static constexpr bool pe = false, rrbs = false, wide = false;
    // short lists (a few half-steps each): the owning lane writes its list's schedule entries (+1 % on config 2; the
    // RRBS / wide kernels, whose lists run to thousands of entries, keep the per-half-step lookup: -9 % / -2 % there)
    static constexpr bool owner_sched = true;
    static constexpr bool run_advance = false;
};
#include "bsx_map_impl.cuh"

namespace {
__global__ void __launch_bounds__(BSX_WARPS_PER_CTA * 32, 5) bsx_map_se_wgbs_kernel(const __grid_constant__ MapArgs A) { map_se(A); }
}
extern const void *const bsx_map_se_wgbs = (const void *)bsx_map_se_wgbs_kernel;
