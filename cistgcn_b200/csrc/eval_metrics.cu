// Fused evaluation metrics (reference: environment/test.py:65-94 Metrics.compute and :125-129 the scatter of the used
// joints back into the full skeleton; losses/losses.py:50-61 mpjpe, :64-77 weighted_mpjpe, :79-144 pa_mpjpe, :147-161
// n_mpjpe, :164-179 mean_velocity_error, :200-239 bone_length_error).  The reference runs each metric as its own chain of
// ATen kernels with a `.cpu()` sync after every one; here ONE kernel reads (pred, target) once and accumulates every
// metric's per-frame sum.  One warp per (sample, frame); lanes = joints; poses staged in shared memory.
#include "eval_metrics.cuh"
#include "host_util.h"

namespace cgt { int fail_train(int code, const char* fmt, ...); }

namespace cgm {

__global__ void __launch_bounds__(NT) eval_metrics_kernel(const Args a) {
  __shared__ float sp[NW][2][MAXJ * 3];       // assembled pose at t and t + 1
  __shared__ float st[NW][2][MAXJ * 3];       // target pose at t and t + 1
  __shared__ double acc[CISTGCN_METRIC_COUNT][32];     // per-CTA per-frame sums (To <= 32 per pass)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int To = a.To;
  for (int i = threadIdx.x; i < CISTGCN_METRIC_COUNT * 32; i += NT) (&acc[0][0])[i] = 0.0;
  __syncthreads();
  const long long items = a.B * To;
  for (long long it = (long long)blockIdx.x * NW + warp; it < items; it += (long long)gridDim.x * NW) {
    const long long b = it / To;
    const int t = (int)(it - b * To);
    float m[CISTGCN_METRIC_COUNT];
    metrics_item(a, sp[warp], st[warp], b, t, lane, m);
    if (lane == 0) {
      atomicAdd(&acc[CISTGCN_METRIC_MPJPE][t], (double)m[CISTGCN_METRIC_MPJPE]);
      atomicAdd(&acc[CISTGCN_METRIC_PA_MPJPE][t], (double)m[CISTGCN_METRIC_PA_MPJPE]);
      atomicAdd(&acc[CISTGCN_METRIC_N_MPJPE][t], (double)m[CISTGCN_METRIC_N_MPJPE]);
      if (t + 1 < To) atomicAdd(&acc[CISTGCN_METRIC_VELOCITY][t], (double)m[CISTGCN_METRIC_VELOCITY]);
      atomicAdd(&acc[CISTGCN_METRIC_BONE_LENGTH][t], (double)m[CISTGCN_METRIC_BONE_LENGTH]);
      atomicAdd(&acc[CISTGCN_METRIC_WEIGHTED0][t], (double)m[CISTGCN_METRIC_WEIGHTED0]);
      atomicAdd(&acc[CISTGCN_METRIC_WEIGHTED1][t], (double)m[CISTGCN_METRIC_WEIGHTED1]);
    }
    __syncwarp();
  }
  __syncthreads();
  for (int i = threadIdx.x; i < CISTGCN_METRIC_COUNT * To; i += NT) {
    const int m = i / To, t = i - m * To;
    if (acc[m][t] != 0.0) atomicAdd(a.sums + m * To + t, acc[m][t]);
  }
}

}  // namespace cgm

extern "C" int cistgcn_eval_metrics_f32(const float* pred, const float* target, const int32_t* src_map, const int32_t* bones,
                                        int32_t n_bones, const float* weights0, const float* weights1, float* assembled,
                                        double* sums, int64_t batch, int32_t To, int32_t Vu, int32_t Vf, void* stream) {
  if (!pred || !target || !src_map || !sums) return cgt::fail_train(-1, "eval_metrics: NULL buffer");
  if (batch < 0 || To < 1 || To > 32 || Vu < 1 || Vf < 1 || Vf > cgm::MAXJ || n_bones < 0 || (n_bones > 0 && !bones))
    return cgt::fail_train(-1, "eval_metrics: bad geometry (output_n <= 32, joints <= %d)", cgm::MAXJ);
  if (batch == 0) return 0;
  cgm::Args a;
  a.pred = pred; a.target = target; a.src_map = src_map; a.bones = bones; a.wt[0] = weights0; a.wt[1] = weights1;
  a.assembled = assembled; a.sums = sums; a.B = batch; a.To = To; a.Vu = Vu; a.Vf = Vf; a.NB = n_bones;
  const long long items = (long long)batch * To;
  long long grid = (items + cgm::NW - 1) / cgm::NW;
  const long long cap = (long long)cg::cached_sm_count() * 4;
  if (grid > cap) grid = cap;
  CG_LAUNCH(cgm::eval_metrics_kernel, (int)grid, cgm::NT, 0, stream, a);
  if (int e = cg::last_launch_error()) return cgt::fail_train(-4, "eval_metrics_kernel launch: %s", cg::launch_error_string(e));
  return 0;
}
