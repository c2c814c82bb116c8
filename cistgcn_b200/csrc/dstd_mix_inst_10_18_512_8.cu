// Explicit instantiation: mix stage of the three-stage DSTD-GC path, (T, V) = (10, 18), 512 threads, TM = 8.
#include "dstd_mix.cuh"
template int cg::launch_mix_impl<10, 18, 512, 8>(const cg::MixArgs&, void*);
