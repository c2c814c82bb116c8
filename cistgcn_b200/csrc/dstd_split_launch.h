// Launchers of the three-stage DSTD-GC path (dstd_reduce.cuh, dstd_adj.cuh, dstd_mix.cuh), one translation unit per
// instantiation group so that nvcc compiles them in parallel (dstd_split_inst_*.cu, dstd_mix_inst_*.cu).
// Return 0 or a CUDA error code.
#pragma once
#include "dstd_adj.cuh"
#include "dstd_mix.cuh"
#include "dstd_mix_mma.cuh"
#include "dstd_mix_narrow.cuh"
#include "dstd_reduce.cuh"
#include "host_util.h"

namespace cg {

#define CG_DECL_SPLIT(T, V) \
  int launch_reduce_##T##_##V##_1(const ReduceArgs& a, void* stream); \
  int launch_reduce_##T##_##V##_2(const ReduceArgs& a, void* stream); \
  int launch_adj_##T##_##V(const AdjArgs& a, void* stream); \
  int launch_mix_##T##_##V##_256_4(const MixArgs& a, void* stream); \
  int launch_mix_##T##_##V##_256_8(const MixArgs& a, void* stream); \
  int launch_mix_##T##_##V##_512_8(const MixArgs& a, void* stream);
CG_DECL_SPLIT(10, 22)
CG_DECL_SPLIT(10, 18)
CG_DECL_SPLIT(22, 25)
CG_DECL_SPLIT(18, 25)
CG_DECL_SPLIT(22, 10)
CG_DECL_SPLIT(18, 10)
#undef CG_DECL_SPLIT
int launch_mix_mma_10_22(const MixArgs& a, void* stream);
int launch_mix_mma_10_18(const MixArgs& a, void* stream);
int launch_mix_narrow_22_25(const MixArgs& a, void* stream);
int launch_mix_narrow_18_25(const MixArgs& a, void* stream);
int launch_mix_narrow_22_10(const MixArgs& a, void* stream);
int launch_mix_narrow_18_10(const MixArgs& a, void* stream);

}  // namespace cg
