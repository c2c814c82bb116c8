// Explicit instantiation: mix stage of the three-stage DSTD-GC path, (T, V) = (22, 25), 256 threads, TM = 8.
#include "dstd_mix.cuh"
template int cg::launch_mix_impl<22, 25, 256, 8>(const cg::MixArgs&, void*);
