// Explicit instantiation: mix stage of the three-stage DSTD-GC path, (T, V) = (18, 25), 256 threads, TM = 4.
#include "dstd_mix.cuh"
template int cg::launch_mix_impl<18, 25, 256, 4>(const cg::MixArgs&, void*);
