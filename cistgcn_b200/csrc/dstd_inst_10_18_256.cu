// Explicit instantiation of the fused DSTD-GC kernel for (T, V) = (10, 18), 256 threads per CTA.
#include "dstd_launch.h"
template int cg::launch_dstd_impl<10, 18, 256>(const cg::DstdArgs&, void*);
