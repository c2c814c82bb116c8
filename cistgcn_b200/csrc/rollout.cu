// Autoregressive rollout past output_n (cistgcn_rollout_f32 / _bf16 in cistgcn_api.cu): what runs between two forwards of
// one chunk.  The step's prediction p_k (n, To, V, 3) is read once; its frames that fall inside the horizon go to the
// caller's output at frame offset k * To (optionally with per-frame MPJPE sums against the caller's target, the
// summation scheme of mpjpe_kernel), and its last Tin frames become the next step's input window.
#include <math.h>

#include "host_util.h"
#include "simt.h"

namespace cg {

constexpr int ROLLOUT_NT = 256;

struct RolloutStepArgs {
  const float* pred;      // (n, To, V, 3) this step's prediction
  float* out;             // (n, H, V, 3) at the chunk's first sample
  float* window;          // (n, Tin, V, 3) next step's input = pred[:, To - Tin:]; NULL after the last step
  const float* target;    // (n, H, V, 3) at the chunk's first sample, or NULL
  double* frame_sums;     // [H], accumulated into (with target)
  long long n;            // samples of the chunk
  int t0, nf;             // this step fills frames [t0, t0 + nf) of out, nf <= To
  int H, Tin, To, V;
};

// One thread per predicted joint position (3 floats), grid-stride.
__global__ void __launch_bounds__(ROLLOUT_NT) rollout_step_kernel(const RolloutStepArgs a) {
  __shared__ double fs[64];
  const int tid = threadIdx.x;
  for (int i = tid; i < 64; i += ROLLOUT_NT) fs[i] = 0.0;
  __syncthreads();
  const int TV = a.To * a.V, skip = a.To - a.Tin;       // Tin <= To: the FPN launcher rejects anything else first
  const long long total = a.n * TV;
  const long long stride = (long long)gridDim.x * ROLLOUT_NT;
  for (long long i = (long long)blockIdx.x * ROLLOUT_NT + tid; i < total; i += stride) {
    const long long b = i / TV;
    const int r = (int)(i - b * TV), f = r / a.V, v = r - f * a.V;
    const float* p = a.pred + i * 3;
    const float p0 = __ldg(p), p1 = __ldg(p + 1), p2 = __ldg(p + 2);
    if (a.window && f >= skip) {
      float* w = a.window + ((b * a.Tin + (f - skip)) * a.V + v) * 3;
      w[0] = p0; w[1] = p1; w[2] = p2;
    }
    if (f < a.nf) {
      const long long o = ((b * a.H + a.t0 + f) * a.V + v) * 3;
      float* q = a.out + o;
      q[0] = p0; q[1] = p1; q[2] = p2;
      if (a.target) {
        const float* tg = a.target + o;
        const float d0 = p0 - __ldg(tg), d1 = p1 - __ldg(tg + 1), d2 = p2 - __ldg(tg + 2);
        const float e = sqrtf(fmaf(d0, d0, fmaf(d1, d1, d2 * d2)));
        if (a.To <= 64) atomicAdd(&fs[f], (double)e);
        else atomicAdd(&a.frame_sums[a.t0 + f], (double)e);
      }
    }
  }
  __syncthreads();
  if (a.target && a.To <= 64)
    for (int f = tid; f < a.nf; f += ROLLOUT_NT) atomicAdd(&a.frame_sums[a.t0 + f], fs[f]);
}

// Host: one launch over a chunk; returns 0 or a CUDA error code.
int launch_rollout_step(const float* pred, float* out, float* window, const float* target, double* frame_sums,
                        long long n, int t0, int nf, int H, int Tin, int To, int V, void* stream) {
  RolloutStepArgs a;
  a.pred = pred; a.out = out; a.window = window; a.target = target; a.frame_sums = frame_sums;
  a.n = n; a.t0 = t0; a.nf = nf; a.H = H; a.Tin = Tin; a.To = To; a.V = V;
  const long long blocks = (n * To * V + ROLLOUT_NT - 1) / ROLLOUT_NT;
  const long long cap = (long long)cached_sm_count() * 8;
  CG_LAUNCH(rollout_step_kernel, (int)(blocks < cap ? blocks : cap), ROLLOUT_NT, 0, stream, a);
  return last_launch_error();
}

}  // namespace cg
