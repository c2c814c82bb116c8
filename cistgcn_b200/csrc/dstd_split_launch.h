// Launchers of the three-stage DSTD-GC path (dstd_reduce.cuh, dstd_adj.cuh, dstd_mix*.cuh).  Each table shape of
// kernel_shapes.h is instantiated in its own translation units (dstd_split_inst_*.cu, dstd_mix_inst_*.cu,
// dstd_mix_mma_inst_*.cu) so that nvcc compiles them in parallel; the declarations below keep every other unit from
// instantiating them again.  Launchers return 0 or a CUDA error code.
#pragma once
#include "dstd_adj.cuh"
#include "dstd_mix.cuh"
#include "dstd_mix_mma.cuh"
#include "dstd_mix_narrow.cuh"
#include "dstd_reduce.cuh"
#include "host_util.h"
#include "kernel_shapes.h"

namespace cg {

#define CG_EXTERN_SPLIT(T, V, MMA, NARROW)                                                      \
  extern template int launch_reduce_impl<T, V, 1>(const ReduceArgs&, void*);                     \
  extern template int launch_reduce_impl<T, V, 2>(const ReduceArgs&, void*);                     \
  extern template int launch_adj_impl<T, V>(const AdjArgs&, void*);                               \
  extern template int launch_mix_impl<T, V, 256, 4>(const MixArgs&, void*);                       \
  extern template int launch_mix_impl<T, V, 256, 8>(const MixArgs&, void*);                       \
  extern template int launch_mix_impl<T, V, 512, 8>(const MixArgs&, void*);                       \
  CG_IF_##MMA(extern template int launch_mix_mma_impl<T, V>(const MixArgs&, void*);)              \
  CG_IF_##NARROW(extern template int launch_mix_narrow_impl<T, V, 3>(const MixArgs&, void*);)
CG_SPLIT_SHAPES(CG_EXTERN_SPLIT)
#undef CG_EXTERN_SPLIT

}  // namespace cg
