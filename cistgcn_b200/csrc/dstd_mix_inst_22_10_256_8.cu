// Explicit instantiation: mix stage of the three-stage DSTD-GC path, (T, V) = (22, 10), 256 threads, TM = 8.
#include "dstd_mix.cuh"
namespace cg {
int launch_mix_22_10_256_8(const MixArgs& a, void* stream) { return launch_mix_impl<22, 10, 256, 8>(a, stream); }
}  // namespace cg
