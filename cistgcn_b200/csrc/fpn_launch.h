// Launcher of the FPN-chain kernel, one translation unit per joint count of kernel_shapes.h (fpn_inst_*.cu).
#pragma once
#include "fpn_chain.cuh"
#include "host_util.h"
#include "kernel_shapes.h"

namespace cg {

template <int V>
int launch_fpn_impl(const FpnArgs& a, void* stream) {
  auto kfn = fpn_chain_kernel<V>;
  const size_t smem = (size_t)a.smem_floats * sizeof(float);
  int err = 0;
  const int per_sm = prepared_blocks_per_sm(kfn, FPN_NT, smem, &err);
  if (err) return err;
  const int grid = grid_for(a.batch, per_sm);
  CG_LAUNCH(kfn, grid, FPN_NT, smem, stream, a);
  return last_launch_error();
}

#define CG_EXTERN_FPN(V) extern template int launch_fpn_impl<V>(const FpnArgs&, void*);
CG_FPN_JOINTS(CG_EXTERN_FPN)
#undef CG_EXTERN_FPN

}  // namespace cg
