// Launcher of the fused DSTD-GC kernel, instantiated for the fused shapes of kernel_shapes.h with one translation unit
// per (T, V, threads) so that nvcc can compile them in parallel (dstd_inst_*.cu).  Returns 0 or a CUDA error code.
//
// Two CTA shapes: 512 threads x 1 CTA per SM (wide blocks: the fp32 working set of E >= 32 fills the SM's
// shared memory) and 256 threads x 2 CTAs per SM (narrow blocks: two samples in flight per SM hide each
// other's barrier and latency stalls).  cistgcn_api.cu picks by what the shared-memory plan allows.
#pragma once
#include "dstd_block.cuh"
#include "host_util.h"
#include "kernel_shapes.h"

namespace cg {

constexpr int DSTD_NT_WIDE = 512;      // 1 CTA / SM, up to 227 KB of shared memory
constexpr int DSTD_NT_NARROW = 256;    // 2 CTAs / SM, up to 113 KB each
constexpr int DSTD_SMEM_NARROW_BYTES = (233472 - 2 * 1024) / 2;

template <int T, int V, int NT, bool TC = false>
int launch_dstd_impl(const DstdArgs& a, void* stream) {
#ifndef CISTGCN_EMU
  auto kfn = dstd_block_kernel<T, V, NT, TC>;
#else
  auto kfn = dstd_block_kernel<T, V, NT, false>;    // the emulator has no tensor cores: the TC slot runs the FFMA kernel
#endif
  const size_t smem = (size_t)a.smem_floats * sizeof(float);
  int err = 0;
  const int per_sm = prepared_blocks_per_sm(kfn, NT, smem, &err);
  if (err) return err;
  const int grid = grid_for(a.batch, per_sm);
  CG_LAUNCH(kfn, grid, NT, smem, stream, a);
  return last_launch_error();
}

#define CG_EXTERN_FUSED(T, V, TC)                                          \
  extern template int launch_dstd_impl<T, V, 256>(const DstdArgs&, void*); \
  extern template int launch_dstd_impl<T, V, 512>(const DstdArgs&, void*); \
  CG_IF_##TC(extern template int launch_dstd_impl<T, V, 512, true>(const DstdArgs&, void*);)
CG_FUSED_SHAPES(CG_EXTERN_FUSED)
#undef CG_EXTERN_FUSED

}  // namespace cg
