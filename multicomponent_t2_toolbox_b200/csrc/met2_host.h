// met2_host.h — host-side plumbing shared by the translation units of libmet2.so (error state, launch accounting).
#pragma once
#ifdef MET2_HOST_EMU
#include "simt_emu.h"
#else
#include <cuda_runtime.h>
#endif
#include <stdint.h>

#include "../../include/met2.h"

// Kernel launch: `MET2_LAUNCH(grid, block, dynamic_smem_bytes, stream, kernel<...>)(args...)` is the CUDA launch
// `kernel<...><<<grid, block, smem, stream>>>(args...)`; under MET2_HOST_EMU (tests/emu, CPU) the same host code drives
// the SIMT emulator instead.  The kernel name comes last so that template argument lists may contain commas.
#ifdef MET2_HOST_EMU
#define MET2_LAUNCH(grid, block, smem, stream, ...) simt::make_launch(dim3(grid), dim3(block), (size_t)(smem), __VA_ARGS__)
#else
#define MET2_LAUNCH(grid, block, smem, stream, ...) __VA_ARGS__<<<(grid), (block), (smem), (stream)>>>
#endif

namespace met2 {

int set_error(int code, const char* fmt, ...);
int check_launch(const char* what);
void count_launch(int n = 1);
int sm_count();
inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// Test hooks: environment variables that force paths the default geometry takes only at sizes too large for the tests.
// read_overrides() is the one place they are read.  met2_fa_fit, met2_t2_fit(_echo) and their *_workspace_bytes call it
// once per call and never cache the result, because tests change the variables between calls in one process; a fit
// sees the values its workspace_bytes call saw as long as nobody changes them in between (MET2_T2_TILE sizes the tile
// list inside the workspace).
//   MET2_T2_WARPS=<w>        caps the warps per CTA of every T2 fit kernel, Gram-domain and echo-space (never raises the
//                            limit): the emulated T2 fits run with 2 or 3 warps (tests/emu/emu.py, t2_fit)
//   MET2_T2_TILE=<n>         uniform tiles of n voxels instead of guided self-scheduling, so that one flip angle spans
//                            several tiles (test_emu_kernels.py, test_odd_sizes_and_tile_scheduling)
//   MET2_LCURVE_SWITCH=<x>   lambda below which the echo-space L-curve tries a grid point in the Gram domain first
//                            (default T2_LCURVE_SWITCH): 100 forces the fall-back from a full Gram-domain factor to echo
//                            space, 0 the whole grid in echo space (test_emu_kernels.py,
//                            test_echo_space_lcurve_and_bayesreg_against_oracle)
//   MET2_FA_SEARCH=warp      switches the thread-per-voxel FA search off: the warp-per-voxel kernel searches every voxel
//                            (test_emu_kernels.py, test_fa_stage_kernels_against_reference; test_gpu_parity_r2.py,
//                            test_fa_search_thread_kernel_equals_warp_kernel)
//   MET2_FA_THREAD_PCAP=<c>  runs the thread-per-voxel FA search at any voxel count and, for 1 <= c < FT_PM, caps its
//                            positive sets at c columns, so that voxels are handed back to the warp kernel (same tests)
struct Overrides {
    int t2_warps;            // 0: unset
    int t2_tile;             // 0: unset
    bool lcurve_switch_set;
    double lcurve_switch;
    bool fa_search_warp;
    bool fa_thread_pcap_set;
    int fa_thread_pcap;
};
Overrides read_overrides();

}  // namespace met2
