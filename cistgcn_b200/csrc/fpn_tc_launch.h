// Launcher of the tensor-core FPN kernel (fpn_tc.cuh), one translation unit per joint count of kernel_shapes.h and
// operand form (fpn_tc_inst_*.cu).  BF16: single-term bf16 operands, bf16 input (cistgcn_forward_bf16).
#pragma once
#ifndef CISTGCN_EMU
#include "fpn_tc.cuh"
#include "host_util.h"
#include "kernel_shapes.h"

namespace cg {

template <int V, bool BF16 = false>
int launch_fpn_tc_impl(const FpnTcArgs& a, void* stream) {
  auto kfn = fpn_tc_kernel<V, BF16>;
  const size_t smem = (size_t)FtcGeom<V>::SMEM_BYTES;
  int err = 0;
  prepared_blocks_per_sm(kfn, FTC_NT, smem, &err);       // raises the opt-in shared-memory limit once
  if (err) return err;
  const int grid = grid_for(a.batch, 1);                  // one CTA per SM: it owns all 512 TMEM columns
  CG_LAUNCH(kfn, grid, FTC_NT, smem, stream, a);
  return last_launch_error();
}

#define CG_EXTERN_FPN_TC(V)                                                    \
  extern template int launch_fpn_tc_impl<V, false>(const FpnTcArgs&, void*); \
  extern template int launch_fpn_tc_impl<V, true>(const FpnTcArgs&, void*);
CG_FPN_JOINTS(CG_EXTERN_FPN_TC)
#undef CG_EXTERN_FPN_TC

}  // namespace cg
#endif
