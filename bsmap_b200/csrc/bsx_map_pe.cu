// bsx_map_pe.cu -- the paired-end WGBS mapping kernel (PairAlign::Do_Batch): inlined whole; every big device function has
// one call site (bsx_map_impl.cuh loops over the mates), so the list walk exists once in the binary.  RRBS is compiled out
// (bsx_map_pe_rrbs.cu): the kernel is instruction-fetch sensitive.  Four resident CTAs per SM at 64 registers: five at
// 48 registers measured slower (config 3 64.9 -> 59.2 M pairs/s).
struct MapKernel {
    static constexpr bool pe = true, rrbs = false;
    static constexpr bool wide = false;            // 8-byte context entries; indexes built for -v >= 8 take bsx_map_pe_wide.cu
    static constexpr bool owner_sched = false, run_advance = false;
};
#include "bsx_map_impl.cuh"

namespace {
__global__ void __launch_bounds__(BSX_WARPS_PER_CTA * 32, 4) bsx_map_pe_wgbs_kernel(const __grid_constant__ MapArgs A) { map_pe(A); }
}
extern const void *const bsx_map_pe_wgbs = (const void *)bsx_map_pe_wgbs_kernel;
