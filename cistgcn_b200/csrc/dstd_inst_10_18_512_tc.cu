// Explicit instantiation of the fused DSTD-GC kernel for T = 10, V = 18, 512 threads, tensor-core channel mixes.
#include "dstd_launch.h"
template int cg::launch_dstd_impl<10, 18, 512, true>(const cg::DstdArgs&, void*);
