// Explicit instantiation: tensor-core (3xTF32 mma.sync) mix stage of the three-stage DSTD-GC path, (T, V) = (10, 18).
#include "dstd_mix_mma.cuh"
template int cg::launch_mix_mma_impl<10, 18>(const cg::MixArgs&, void*);
