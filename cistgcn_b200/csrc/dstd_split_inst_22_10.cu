// Explicit instantiations: reduce + adjacency stages (+ the narrow 3-channel mix stage) of the three-stage DSTD-GC path for (T, V) = (22, 10).
#include "dstd_adj.cuh"
#include "dstd_mix_narrow.cuh"
#include "dstd_reduce.cuh"
namespace cg {
int launch_reduce_22_10_1(const ReduceArgs& a, void* stream) { return launch_reduce_impl<22, 10, 1>(a, stream); }
int launch_reduce_22_10_2(const ReduceArgs& a, void* stream) { return launch_reduce_impl<22, 10, 2>(a, stream); }
int launch_adj_22_10(const AdjArgs& a, void* stream) { return launch_adj_impl<22, 10>(a, stream); }
int launch_mix_narrow_22_10(const MixArgs& a, void* stream) { return launch_mix_narrow_impl<22, 10, 3>(a, stream); }
}  // namespace cg
