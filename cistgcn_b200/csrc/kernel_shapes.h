// The block shapes the DSTD-GC and FPN kernels are compiled for: the one list of them.  The launch headers declare an
// `extern template` for every entry and cistgcn_api.cu dispatches over them; both are generated from the lists below.
//
// Adding a shape: add its line here, then add the translation units that explicitly instantiate its launchers (copy
// the units of a shape with the same variants and change the numbers; one unit per group so nvcc builds them in
// parallel).  A line without its units fails at link time.
#pragma once

// Three-stage path (dstd_reduce.cuh -> dstd_adj.cuh -> stage 3): X(T, V, MMA, NARROW), one line per (T, V).
// Every shape has the reduce stage (NE = 1, 2: dstd_split_inst_T_V.cu), the adjacency stage (same unit) and the FFMA
// tile mix (dstd_mix.cuh) at 256 threads / TM 4, 256 / 8 and 512 / 8 (dstd_mix_inst_T_V_NT_TM.cu).
//   MMA = 1: stage 3 also has the 3xTF32 mma.sync channel mix (dstd_mix_mma.cuh, dstd_mix_mma_inst_T_V.cu).
//   NARROW = 1: stage 3 also has the warp-per-sample mix of 3 -> 3 blocks (dstd_mix_narrow.cuh, C = 3; it is
//   instantiated next to the reduce stage, in dstd_split_inst_T_V.cu).
#define CG_SPLIT_SHAPES(X) \
  X(10, 22, 1, 0)          \
  X(10, 18, 1, 0)          \
  X(22, 25, 0, 1)          \
  X(18, 25, 0, 1)          \
  X(22, 10, 0, 1)          \
  X(18, 10, 0, 1)

// Round-1 fused kernel (dstd_block.cuh): X(T, V, TC), at 256 and 512 threads (dstd_inst_T_V_NT.cu).
//   TC = 1: also the 512-thread instantiation with the tcgen05 channel mixes (dstd_inst_T_V_512_tc.cu).
#define CG_FUSED_SHAPES(X) \
  X(10, 22, 1)             \
  X(10, 18, 1)             \
  X(22, 25, 0)             \
  X(18, 25, 0)

// FPN chain: X(V) joint counts, each with the FP32-FMA kernel (fpn_chain.cuh, fpn_inst_V.cu) and the tcgen05 kernel
// (fpn_tc.cuh) in its split-fp32 and bf16 forms (fpn_tc_inst_V.cu, fpn_tc_inst_V_bf16.cu).
#define CG_FPN_JOINTS(X) \
  X(22)                  \
  X(18)

// CG_IF_1(code) is code, CG_IF_0(code) is nothing: expands a table line's variant bit
#define CG_IF_0(...)
#define CG_IF_1(...) __VA_ARGS__

namespace cg {

struct SplitShape { int T, V; bool mix_mma, mix_narrow; };
struct FusedShape { int T, V; bool tc; };

#define CG_SPLIT_ROW(T, V, MMA, NARROW) {T, V, MMA, NARROW},
#define CG_FUSED_ROW(T, V, TC) {T, V, TC},
#define CG_FPN_ROW(V) V,
constexpr SplitShape kSplitShapes[] = {CG_SPLIT_SHAPES(CG_SPLIT_ROW)};
constexpr FusedShape kFusedShapes[] = {CG_FUSED_SHAPES(CG_FUSED_ROW)};
constexpr int kFpnJoints[] = {CG_FPN_JOINTS(CG_FPN_ROW)};
#undef CG_SPLIT_ROW
#undef CG_FUSED_ROW
#undef CG_FPN_ROW

// The table line of (T, V), or nullptr when the path has no kernel for it
constexpr const SplitShape* split_shape(int T, int V) {
  for (const SplitShape& s : kSplitShapes)
    if (s.T == T && s.V == V) return &s;
  return nullptr;
}
constexpr const FusedShape* fused_shape(int T, int V) {
  for (const FusedShape& s : kFusedShapes)
    if (s.T == T && s.V == V) return &s;
  return nullptr;
}
constexpr bool fpn_joints_built(int V) {
  for (int j : kFpnJoints)
    if (j == V) return true;
  return false;
}

}  // namespace cg
