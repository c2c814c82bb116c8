// Explicit instantiation: mix stage of the three-stage DSTD-GC path, (T, V) = (18, 10), 512 threads, TM = 8.
#include "dstd_mix.cuh"
namespace cg {
int launch_mix_18_10_512_8(const MixArgs& a, void* stream) { return launch_mix_impl<18, 10, 512, 8>(a, stream); }
}  // namespace cg
