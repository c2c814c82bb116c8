// Explicit instantiation: mix stage of the three-stage DSTD-GC path, (T, V) = (18, 10), 256 threads, TM = 4.
#include "dstd_mix.cuh"
namespace cg {
int launch_mix_18_10_256_4(const MixArgs& a, void* stream) { return launch_mix_impl<18, 10, 256, 4>(a, stream); }
}  // namespace cg
