// Explicit instantiations: reduce + adjacency stages of the three-stage DSTD-GC path for (T, V) = (10, 22).
#include "dstd_adj.cuh"
#include "dstd_reduce.cuh"
template int cg::launch_reduce_impl<10, 22, 1>(const cg::ReduceArgs&, void*);
template int cg::launch_reduce_impl<10, 22, 2>(const cg::ReduceArgs&, void*);
template int cg::launch_adj_impl<10, 22>(const cg::AdjArgs&, void*);
