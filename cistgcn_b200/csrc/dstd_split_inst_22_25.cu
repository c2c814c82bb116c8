// Explicit instantiations: reduce + adjacency stages (+ the narrow 3-channel mix stage) of the three-stage DSTD-GC path for (T, V) = (22, 25).
#include "dstd_adj.cuh"
#include "dstd_mix_narrow.cuh"
#include "dstd_reduce.cuh"
template int cg::launch_reduce_impl<22, 25, 1>(const cg::ReduceArgs&, void*);
template int cg::launch_reduce_impl<22, 25, 2>(const cg::ReduceArgs&, void*);
template int cg::launch_adj_impl<22, 25>(const cg::AdjArgs&, void*);
template int cg::launch_mix_narrow_impl<22, 25, 3>(const cg::MixArgs&, void*);
