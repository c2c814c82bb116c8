// Explicit instantiation of the fused DSTD-GC kernel for (T, V) = (18, 25), 512 threads per CTA.
#include "dstd_launch.h"
template int cg::launch_dstd_impl<18, 25, 512>(const cg::DstdArgs&, void*);
