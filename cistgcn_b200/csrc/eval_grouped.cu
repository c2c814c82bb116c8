// Grouped evaluation: per-group (action, sub-dataset) per-frame sums in one pass over a whole test set.
//
// grouped_mpjpe_kernel (behind cistgcn_mpjpe_grouped_f32 in cistgcn_api.cu) is mpjpe_kernel's summation scheme -- fp32
// per-joint L2 error, fp64 shared then global atomics -- with the frame sums split by a per-sample group id:
// sums[G][T] and counts[G] (samples).  eval_metrics_grouped_kernel (cistgcn_eval_metrics_grouped_f32 below) is
// eval_metrics_kernel's warp work (eval_metrics.cuh) accumulated into sums[G][CISTGCN_METRIC_COUNT][To] + counts[G], with
// no frame limit.  Both keep a per-CTA accumulator in dynamic shared memory when it fits kAccSmemBytes and add straight
// into the global sums otherwise.  A sample whose id is outside [0, G) is skipped and not counted.
#include "eval_metrics.cuh"
#include "host_util.h"

namespace cgt { int fail_train(int code, const char* fmt, ...); }

namespace cg {

constexpr size_t kAccSmemBytes = 48 * 1024;   // largest per-CTA accumulator (sums + counts) kept in shared memory
constexpr int GMPJPE_NT = 256;

CG_DEV void add_count(long long* p, long long v) {
#ifdef CISTGCN_EMU
  __atomic_fetch_add(p, v, __ATOMIC_RELAXED);
#else
  atomicAdd(reinterpret_cast<unsigned long long*>(p), (unsigned long long)v);
#endif
}

struct GroupedMpjpeArgs {
  const float* pred;      // (B, T, V, 3)
  const float* target;    // (B, T, V, 3)
  const int* groups;      // [B] group ids, or NULL = every sample in group 0
  double* sums;           // [G][T], accumulated
  long long* counts;      // [G], accumulated
  long long n;            // B*T*V
  int T, V, G;
  int smem;               // 1: per-CTA accumulator in dynamic shared memory ([G][T] doubles, then [G] counts)
};

// One thread per joint position (3 floats), grid-stride, as mpjpe_kernel.
__global__ void __launch_bounds__(GMPJPE_NT) grouped_mpjpe_kernel(const GroupedMpjpeArgs a) {
  CG_DYN_SMEM(dyn);
  const int tid = threadIdx.x, GT = a.G * a.T, TV = a.T * a.V;
  double* fs = reinterpret_cast<double*>(dyn);
  long long* cs = reinterpret_cast<long long*>(fs + GT);
  if (a.smem) {
    for (int i = tid; i < GT; i += GMPJPE_NT) fs[i] = 0.0;
    for (int i = tid; i < a.G; i += GMPJPE_NT) cs[i] = 0;
  }
  __syncthreads();
  double* sums = a.smem ? fs : a.sums;
  long long* counts = a.smem ? cs : a.counts;
  const long long stride = (long long)gridDim.x * GMPJPE_NT;
  for (long long i = (long long)blockIdx.x * GMPJPE_NT + tid; i < a.n; i += stride) {
    const long long b = i / TV;
    const int r = (int)(i - b * TV);
    const int g = a.groups ? __ldg(a.groups + b) : 0;
    if ((unsigned)g >= (unsigned)a.G) continue;
    const float* p = a.pred + i * 3;
    const float* q = a.target + i * 3;
    const float d0 = p[0] - q[0], d1 = p[1] - q[1], d2 = p[2] - q[2];
    const float e = sqrtf(fmaf(d0, d0, fmaf(d1, d1, d2 * d2)));
    atomicAdd(&sums[(long long)g * a.T + r / a.V], (double)e);
    if (r == 0) add_count(&counts[g], 1);
  }
  __syncthreads();
  if (a.smem) {
    for (int i = tid; i < GT; i += GMPJPE_NT)
      if (fs[i] != 0.0) atomicAdd(&a.sums[i], fs[i]);
    for (int i = tid; i < a.G; i += GMPJPE_NT)
      if (cs[i] != 0) add_count(&a.counts[i], cs[i]);
  }
}

// Host: one launch; returns 0 or a CUDA error code.  The arguments are checked by the caller.
int launch_mpjpe_grouped(const float* pred, const float* target, const int* groups, int G, long long batch, int T, int V,
                         double* sums, long long* counts, void* stream) {
  GroupedMpjpeArgs a;
  a.pred = pred; a.target = target; a.groups = groups; a.sums = sums; a.counts = counts;
  a.n = batch * T * V; a.T = T; a.V = V; a.G = G;
  const size_t smem = ((size_t)G * T + G) * 8;
  a.smem = smem <= kAccSmemBytes;
  const long long blocks = (a.n + GMPJPE_NT - 1) / GMPJPE_NT;
  const long long cap = (long long)cached_sm_count() * 8;
  CG_LAUNCH(grouped_mpjpe_kernel, (int)(blocks < cap ? blocks : cap), GMPJPE_NT, a.smem ? smem : 0, stream, a);
  return last_launch_error();
}

}  // namespace cg

namespace cgm {

struct GroupedArgs {
  Args m;                 // m.sums: [G][CISTGCN_METRIC_COUNT][To], accumulated
  const int* groups;      // [B] group ids, or NULL = every sample in group 0
  long long* counts;      // [G], accumulated
  int G;
  int smem;               // 1: per-CTA accumulator in dynamic shared memory (sums as m.sums, then [G] counts)
};

__global__ void __launch_bounds__(NT) eval_metrics_grouped_kernel(const GroupedArgs a) {
  __shared__ float sp[NW][2][MAXJ * 3];       // assembled pose at t and t + 1
  __shared__ float st[NW][2][MAXJ * 3];       // target pose at t and t + 1
  CG_DYN_SMEM(dyn);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int To = a.m.To, S = a.G * CISTGCN_METRIC_COUNT * To;
  double* acc = reinterpret_cast<double*>(dyn);
  long long* cnt = reinterpret_cast<long long*>(acc + S);
  if (a.smem) {
    for (int i = threadIdx.x; i < S; i += NT) acc[i] = 0.0;
    for (int i = threadIdx.x; i < a.G; i += NT) cnt[i] = 0;
  }
  __syncthreads();
  double* sums = a.smem ? acc : a.m.sums;
  long long* counts = a.smem ? cnt : a.counts;
  const long long items = a.m.B * To;
  for (long long it = (long long)blockIdx.x * NW + warp; it < items; it += (long long)gridDim.x * NW) {
    const long long b = it / To;
    const int t = (int)(it - b * To);
    float m[CISTGCN_METRIC_COUNT];
    metrics_item(a.m, sp[warp], st[warp], b, t, lane, m);    // also for skipped ids: `assembled` is written for every sample
    const int g = a.groups ? __ldg(a.groups + b) : 0;
    if (lane == 0 && (unsigned)g < (unsigned)a.G) {
      double* s = sums + (long long)g * CISTGCN_METRIC_COUNT * To + t;
      for (int k = 0; k < CISTGCN_METRIC_COUNT; ++k)
        if (k != CISTGCN_METRIC_VELOCITY || t + 1 < To) atomicAdd(s + k * To, (double)m[k]);
      if (t == 0) cg::add_count(&counts[g], 1);
    }
    __syncwarp();
  }
  __syncthreads();
  if (a.smem) {
    for (int i = threadIdx.x; i < S; i += NT)
      if (acc[i] != 0.0) atomicAdd(a.m.sums + i, acc[i]);
    for (int i = threadIdx.x; i < a.G; i += NT)
      if (cnt[i] != 0) cg::add_count(a.counts + i, cnt[i]);
  }
}

}  // namespace cgm

extern "C" int cistgcn_eval_metrics_grouped_f32(const float* pred, const float* target, const int32_t* groups,
                                                int32_t n_groups, const int32_t* src_map, const int32_t* bones,
                                                int32_t n_bones, const float* weights0, const float* weights1,
                                                float* assembled, double* sums, int64_t* counts, int64_t batch,
                                                int32_t To, int32_t Vu, int32_t Vf, void* stream) {
  if (!pred || !target || !src_map || !sums || !counts) return cgt::fail_train(-1, "eval_metrics_grouped: NULL buffer");
  if (n_groups < 1 || (long long)n_groups * CISTGCN_METRIC_COUNT * To > 0x7fffffffLL)
    return cgt::fail_train(-1, "eval_metrics_grouped: n_groups = %d (>= 1, n_groups * %d * To < 2^31)", n_groups,
                           CISTGCN_METRIC_COUNT);
  if (batch < 0 || To < 1 || Vu < 1 || Vf < 1 || Vf > cgm::MAXJ || n_bones < 0 || (n_bones > 0 && !bones))
    return cgt::fail_train(-1, "eval_metrics_grouped: bad geometry (batch >= 0, To >= 1, joints <= %d)", cgm::MAXJ);
  if (batch == 0) return 0;
  cgm::GroupedArgs a;
  a.m.pred = pred; a.m.target = target; a.m.src_map = src_map; a.m.bones = bones; a.m.wt[0] = weights0; a.m.wt[1] = weights1;
  a.m.assembled = assembled; a.m.sums = sums; a.m.B = batch; a.m.To = To; a.m.Vu = Vu; a.m.Vf = Vf; a.m.NB = n_bones;
  a.groups = groups; a.counts = reinterpret_cast<long long*>(counts); a.G = n_groups;
  const size_t smem_need = ((size_t)n_groups * CISTGCN_METRIC_COUNT * To + n_groups) * 8;
  a.smem = smem_need <= cg::kAccSmemBytes;
  const size_t smem = a.smem ? smem_need : 0;
  int err = 0;
  const int per_sm = cg::prepared_blocks_per_sm(cgm::eval_metrics_grouped_kernel, cgm::NT, smem, &err);
  if (err) return cgt::fail_train(-4, "eval_metrics_grouped_kernel shared-memory opt-in: %s", cg::launch_error_string(err));
  const long long items = (long long)batch * To;
  long long grid = (items + cgm::NW - 1) / cgm::NW;
  const long long cap = (long long)cg::cached_sm_count() * per_sm;
  if (grid > cap) grid = cap;
  CG_LAUNCH(cgm::eval_metrics_grouped_kernel, (int)grid, cgm::NT, smem, stream, a);
  if (int e = cg::last_launch_error())
    return cgt::fail_train(-4, "eval_metrics_grouped_kernel launch: %s", cg::launch_error_string(e));
  return 0;
}
