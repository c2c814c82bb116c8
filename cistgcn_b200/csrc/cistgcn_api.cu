// C-ABI of the B200-native CIST-GCN forward path (declared in include/cistgcn_b200.h).
// Host-side orchestration only: descriptor validation, shared-memory planning, launches.
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <mutex>
#include <string>
#include <vector>

#include "../../include/cistgcn_b200.h"
#include "dstd_launch.h"
#include "dstd_split_launch.h"
#include "fpn_launch.h"
#include "fpn_tc_launch.h"
#include "host_util.h"
#include "simt.h"
#include "tail.cuh"

#ifndef CISTGCN_MAX_CHUNK
#define CISTGCN_MAX_CHUNK 32768
#endif

namespace cg {
// csrc/rollout.cu: moves one rollout step's prediction into the output and the next input window; 0 or a CUDA error
int launch_rollout_step(const float* pred, float* out, float* window, const float* target, double* frame_sums,
                        long long n, int t0, int nf, int H, int Tin, int To, int V, void* stream);
// csrc/eval_grouped.cu: per-group per-frame MPJPE sums and sample counts; 0 or a CUDA error
int launch_mpjpe_grouped(const float* pred, const float* target, const int* groups, int G, long long batch, int T, int V,
                         double* sums, long long* counts, void* stream);
}  // namespace cg

namespace {

thread_local std::string g_err;

constexpr int kMaxSmemBytes = 227 * 1024;

}  // namespace

namespace cgt {
// Records the message for cistgcn_last_error() and returns code: the error sink of every entry point, also those of
// train_ops.cu, augment.cu, eval_metrics.cu and eval_grouped.cu
int fail_train(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}
}  // namespace cgt

namespace {

constexpr auto& fail = cgt::fail_train;
using cg::sm_count;
using cg::grid_for;

// e: what a launcher returned (a CUDA error code or 0)
int check_launch(int e, const char* what) {
  if (e) return fail(-4, "%s launch: %s", what, cg::launch_error_string(e));
  return 0;
}

// ---- optional per-kernel CUDA-event timing (bench.py's live roofline numbers) ------------------
enum { KIND_DSTD = 0, KIND_FPN = 1, KIND_TAIL = 2, KIND_MPJPE = 3, KIND_REDUCE = 4, KIND_ADJ = 5, KIND_MIX = 6, KIND_OTHER = 7,
       KIND_COUNT = CISTGCN_PROFILE_KINDS };
const char* const kKindNames[KIND_COUNT] = {"dstd_block_kernel", "fpn_kernel", "tail_kernel", "mpjpe_kernel",
                                            "dstd_reduce_kernel", "dstd_adj_kernel", "dstd_mix_kernel", "other"};
#ifndef CISTGCN_EMU
struct ProfSlot { cudaEvent_t beg, end; int kind; };
struct Profiler {
  std::mutex mu;                   // process-wide instrumentation: every access holds the lock
  bool on = false;
  std::vector<ProfSlot> slots;     // events are recycled after every read
  size_t used = 0;
  long long launches[KIND_COUNT] = {};
  ProfSlot* next(int kind) {
    if (used == slots.size()) {
      if (slots.size() >= 16384) return nullptr;
      ProfSlot s;
      if (cudaEventCreate(&s.beg) != cudaSuccess || cudaEventCreate(&s.end) != cudaSuccess) return nullptr;
      slots.push_back(s);
    }
    slots[used].kind = kind;
    return &slots[used++];
  }
};
Profiler g_prof;
struct ProfScope {
  ProfSlot* s = nullptr;
  cudaStream_t st;
  ProfScope(int kind, void* stream) : st((cudaStream_t)stream) {
    std::lock_guard<std::mutex> lock(g_prof.mu);
    if (!g_prof.on) return;
    g_prof.launches[kind]++;
    s = g_prof.next(kind);
    if (s) cudaEventRecord(s->beg, st);
  }
  ~ProfScope() { if (s) cudaEventRecord(s->end, st); }
};
#else
struct ProfScope { ProfScope(int, void*) {} };
#endif

// ---------------------------------------------------------------------------------------------
#ifdef CISTGCN_PROFILE
long long* g_phase_clocks = nullptr;   // debug hooks of -DCISTGCN_PROFILE builds, see cistgcn_debug_phase_clocks
int g_stamp_iter = 0;
#else
constexpr long long* g_phase_clocks = nullptr;
constexpr int g_stamp_iter = 0;
#endif

int check_block_desc(const int32_t* d) {
  const int Ci = d[CB_CI], Co = d[CB_CO];
  if (Ci < 2 || Co < 1) return fail(-2, "DSTD-GC block needs Ci >= 2 (got %d -> %d)", Ci, Co);
  if (Co > 64 || Ci > 64) return fail(-2, "DSTD-GC block: %d -> %d channels exceed the 64 supported", Ci, Co);
  if (d[CB_IN_MODE] == 1 && Ci != 10) return fail(-2, "feature-building input mode needs Ci == 10");
  return 0;
}

// one " (T,V)" per table line, for the "built:" list of an error message
#define CG_SHAPE_NAME(T, V, ...) " (" #T "," #V ")"
#define CG_JOINTS_NAME(V) " " #V

// ---- round-1 fused kernel (one CTA per sample, csrc/dstd_block.cuh): E = 64 blocks and CISTGCN_FLAG_DSTD_FUSED
template <int T, int V>
int launch_fused_shape(const cg::DstdArgs& a, int nt, void* stream) {
  if constexpr (cg::fused_shape(T, V)->tc)
    if (nt == 512 && a.tc) return cg::launch_dstd_impl<T, V, 512, true>(a, stream);
  return nt == 256 ? cg::launch_dstd_impl<T, V, 256>(a, stream) : cg::launch_dstd_impl<T, V, 512>(a, stream);
}

int launch_dstd_fused(const int32_t* desc, const float* weights, const float* in, float* out, long long batch,
                      const cistgcn_block_taps* taps, uint32_t flags, int in_bf16, int out_bf16, void* stream) {
  cg::DstdArgs a;
  memcpy(a.d, desc, sizeof(a.d));
  a.w = weights; a.in = in; a.out = out; a.batch = (int)batch;
  a.in_bf16 = in_bf16; a.out_bf16 = out_bf16;
  if (in_bf16 || out_bf16) flags &= ~(uint32_t)CISTGCN_FLAG_DSTD_TC;      // the tcgen05 epilogues store fp32 only
  a.tap_adj_s = taps ? taps->adj_s : nullptr;
  a.tap_adj_t = taps ? taps->adj_t : nullptr;
  a.tap_w1 = taps ? taps->w1 : nullptr;
  a.tap_w2 = taps ? taps->w2 : nullptr;
  const int T = a.d[CB_T], V = a.d[CB_V], Ci = a.d[CB_CI], Co = a.d[CB_CO];
  // the 10-frame output blocks (output_n = 10) among others: they run on the three-stage path only
  const cg::FusedShape* shape = cg::fused_shape(T, V);
  if (!shape)
    return fail(-2, "DSTD-GC block: (T, V) = (%d, %d) has no fused kernel (built:" CG_FUSED_SHAPES(CG_SHAPE_NAME) ")", T, V);
  if (!a.d[CB_INTERP]) { a.tap_adj_s = nullptr; a.tap_adj_t = nullptr; }
  a.phase_clocks = g_phase_clocks;
  a.stamp_iter = g_stamp_iter;
  // narrow blocks: 256 threads, two CTAs per SM (if the whole plan fits half an SM's shared memory);
  // wide blocks: 512 threads, one CTA per SM
  // (the tensor-core flag asks for the wide plan outright: only that instantiation carries the tcgen05 channel mixes)
  const bool tc_ok = (flags & CISTGCN_FLAG_DSTD_TC) && shape->tc;
  int nt = cg::DSTD_NT_NARROW;
  if (tc_ok || !cg::dstd_plan(a, nt, cg::DSTD_SMEM_NARROW_BYTES / 4)) {
    nt = cg::DSTD_NT_WIDE;
    if (!cg::dstd_plan(a, nt, kMaxSmemBytes / 4, tc_ok) || (size_t)a.smem_floats * 4 > (size_t)kMaxSmemBytes)
      return fail(-2, "DSTD-GC block (%d->%d, T=%d, V=%d) needs %zu B of shared memory (> %d)", Ci, Co, T, V,
                  (size_t)a.smem_floats * 4, kMaxSmemBytes);
  }
  ProfScope prof(KIND_DSTD, stream);
  int e = 0;
#define CG_FUSED_CASE(TT, VV, TC) \
  if (T == TT && V == VV) e = launch_fused_shape<TT, VV>(a, nt, stream);
  CG_FUSED_SHAPES(CG_FUSED_CASE)
#undef CG_FUSED_CASE
  return check_launch(e, "dstd_block_kernel");
}

// ---- three-stage path (csrc/dstd_reduce.cuh -> dstd_adj.cuh -> dstd_mix.cuh)
struct SplitPlan {
  cg::ReduceArgs r;
  cg::AdjArgs j;
  cg::MixArgs m;
  int mix_nt, mix_tm, ne;
  bool mix_mma;                                               // stage 3 on 3xTF32 mma.sync (dstd_mix_mma.cuh)
  bool mix_narrow;                                            // stage 3 warp-per-sample, streamed adjacencies (dstd_mix_narrow.cuh)
  size_t red_floats, wg_floats, adjs_floats, adjt_floats;     // scratch per sample
};

// Fills the three argument blocks' plans; false if the shape / widths are outside what the split kernels tile.
bool split_plan(const int32_t* desc, SplitPlan& sp, uint32_t flags = 0) {
  const int T = desc[CB_T], V = desc[CB_V], Co = desc[CB_CO], Ch = desc[CB_CH], Cg = desc[CB_CG];
  const bool interp = desc[CB_INTERP] != 0;
  const cg::SplitShape* shape = cg::split_shape(T, V);
  if (!shape) return false;
  memcpy(sp.r.d, desc, sizeof(sp.r.d));
  memcpy(sp.j.d, desc, sizeof(sp.j.d));
  memcpy(sp.m.d, desc, sizeof(sp.m.d));
  const int cap = kMaxSmemBytes / 4;
  if (!cg::reduce_plan(sp.r, cap, !(flags & CISTGCN_FLAG_DSTD_REDUCE_FFMA))) return false;
  if (!((!(flags & CISTGCN_FLAG_DSTD_ADJ_FFMA) && cg::adj_plan(sp.j, cap, true)) || cg::adj_plan(sp.j, cap, false))) return false;
  sp.ne = interp ? (4 * Ch + 31) / 32 : 1;
  if (sp.ne < 1) sp.ne = 1;
  // mix stage: two 256-thread CTAs per SM when the plan fits half an SM, else one 512-thread CTA
  const int TV = T * V;
  const int tn = (TV % 4 == 0) ? 4 : 2;
  const int ng = ((TV / tn) + 31) / 32;
  auto fits = [&](int nt, int tm) { return ((Co + tm - 1) / tm) * ng <= (tm == 8 ? 1 : 2) * (nt / 32); };
  sp.mix_nt = 0;
  sp.mix_mma = false;
  sp.mix_narrow = false;
  // 3 -> 3 blocks (the output block): one warp per sample, adjacencies streamed from global memory
  if (!(flags & CISTGCN_FLAG_DSTD_MIX_FFMA) && shape->mix_narrow && cg::mix_narrow_plan<3>(sp.m, cap)) {
    sp.mix_narrow = true; sp.mix_nt = 32 * sp.m.nwarps; sp.mix_tm = 0;
  } else
  // tensor-core channel mixes: the input blocks (T = 10) from 16 channels up -- below that a 16-row MMA tile is mostly
  // padding and the FFMA loops are already short
  if (!(flags & CISTGCN_FLAG_DSTD_MIX_FFMA) && shape->mix_mma && (desc[CB_CI] >= 16 || Co >= 16) &&
      cg::mix_mma_plan(sp.m, cg::DSTD_SMEM_NARROW_BYTES / 4)) {
    sp.mix_mma = true; sp.mix_nt = 256; sp.mix_tm = 0;
  } else if (cg::mix_plan(sp.m, 256, cg::DSTD_SMEM_NARROW_BYTES / 4)) {
    if (Co > 16 && fits(256, 8)) { sp.mix_nt = 256; sp.mix_tm = 8; }
    else if (fits(256, 4)) { sp.mix_nt = 256; sp.mix_tm = 4; }
  }
  if (!sp.mix_nt) {
    if (!cg::mix_plan(sp.m, 512, cap) || !fits(512, 8)) return false;
    sp.mix_nt = 512; sp.mix_tm = 8;
  }
  const cg::RedLayout RL(T, V, Cg, Ch, interp);
  sp.red_floats = (size_t)RL.total;
  sp.wg_floats = (size_t)((2 * Co + 3) & ~3);
  sp.adjs_floats = interp ? (size_t)((V * T * T + 3) & ~3) : 0;
  sp.adjt_floats = interp ? (size_t)((T * V * V + 3) & ~3) : 0;
  return true;
}

size_t split_scratch_floats(const SplitPlan& sp, long long batch, bool with_adj) {
  size_t n = (size_t)batch * sp.red_floats + (((size_t)batch * 2 * sp.r.d[CB_CO] + 3) & ~(size_t)3);
  if (with_adj) n += (((size_t)batch * sp.r.d[CB_V] * sp.r.d[CB_T] * sp.r.d[CB_T] + 3) & ~(size_t)3) +
                     (((size_t)batch * sp.r.d[CB_T] * sp.r.d[CB_V] * sp.r.d[CB_V] + 3) & ~(size_t)3);
  return n;
}

bool use_split(const int32_t* desc, uint32_t flags, SplitPlan& sp) {
  if (flags & (CISTGCN_FLAG_DSTD_FUSED | CISTGCN_FLAG_DSTD_TC)) return false;
  return split_plan(desc, sp, flags);
}

int no_split_kernel(int T, int V) {
  return fail(-2, "DSTD-GC block: (T, V) = (%d, %d) has no compiled kernel (built:" CG_SPLIT_SHAPES(CG_SHAPE_NAME) ")", T, V);
}

// The three stages of one table shape; stage 3 as split_plan chose it, among the variants the table line has
template <int T, int V>
int launch_split_shape(const SplitPlan& sp, void* stream) {
  constexpr cg::SplitShape shape = *cg::split_shape(T, V);
  int e;
  { ProfScope prof(KIND_REDUCE, stream);
    e = sp.ne == 1 ? cg::launch_reduce_impl<T, V, 1>(sp.r, stream) : cg::launch_reduce_impl<T, V, 2>(sp.r, stream); }
  if (e) return check_launch(e, "dstd_reduce_kernel");
  { ProfScope prof(KIND_ADJ, stream); e = cg::launch_adj_impl<T, V>(sp.j, stream); }
  if (e) return check_launch(e, "dstd_adj_kernel");
  ProfScope prof(KIND_MIX, stream);
  if constexpr (shape.mix_narrow)
    if (sp.mix_narrow) return check_launch(cg::launch_mix_narrow_impl<T, V, 3>(sp.m, stream), "dstd_mix_kernel");
  if constexpr (shape.mix_mma)
    if (sp.mix_mma) return check_launch(cg::launch_mix_mma_impl<T, V>(sp.m, stream), "dstd_mix_kernel");
  e = sp.mix_nt == 512 ? cg::launch_mix_impl<T, V, 512, 8>(sp.m, stream)
      : sp.mix_tm == 8 ? cg::launch_mix_impl<T, V, 256, 8>(sp.m, stream) : cg::launch_mix_impl<T, V, 256, 4>(sp.m, stream);
  return check_launch(e, "dstd_mix_kernel");
}

int launch_dstd_split(SplitPlan& sp, const float* weights, const float* in, float* out, long long batch,
                      const cistgcn_block_taps* taps, float* scratch, int in_bf16, int out_bf16, void* stream) {
  const int* d = sp.r.d;
  const int T = d[CB_T], V = d[CB_V], Co = d[CB_CO];
  const bool interp = d[CB_INTERP] != 0;
  // scratch: [B x red record][B x 2 x Co gates][B x (V,T,T)][B x (T,V,V)], every region 16-byte aligned
  float* red = scratch;
  float* wg = red + (size_t)batch * sp.red_floats;
  float* adj_s = wg + (((size_t)batch * 2 * Co + 3) & ~(size_t)3);
  float* adj_t = adj_s + (((size_t)batch * V * T * T + 3) & ~(size_t)3);
  // the adjacency taps have exactly the layout stage 3 reads: write them once, in place
  if (interp && taps && taps->adj_s && taps->adj_t) { adj_s = taps->adj_s; adj_t = taps->adj_t; }
  sp.r.w = weights; sp.r.in = in; sp.r.red = red; sp.r.batch = (int)batch; sp.r.red_stride = (int)sp.red_floats;
  sp.r.in_bf16 = in_bf16; sp.m.in_bf16 = in_bf16; sp.m.out_bf16 = out_bf16;
  sp.j.w = weights; sp.j.red = red; sp.j.red_stride = (int)sp.red_floats; sp.j.wg = wg;
  sp.j.adj_s = adj_s; sp.j.adj_t = adj_t; sp.j.batch = (int)batch;
  sp.j.tap_w1 = taps ? taps->w1 : nullptr; sp.j.tap_w2 = taps ? taps->w2 : nullptr;
  sp.m.w = weights; sp.m.in = in; sp.m.out = out; sp.m.wg = wg; sp.m.adj_s = adj_s; sp.m.adj_t = adj_t; sp.m.batch = (int)batch;
#define CG_SPLIT_CASE(TT, VV, MMA, NARROW) \
  if (T == TT && V == VV) return launch_split_shape<TT, VV>(sp, stream);
  CG_SPLIT_SHAPES(CG_SPLIT_CASE)
#undef CG_SPLIT_CASE
  return no_split_kernel(T, V);
}

// Scratch floats of one block for `batch` samples (0 when the block runs on the fused kernel).
size_t dstd_scratch_floats(const int32_t* desc, uint32_t flags, long long batch) {
  SplitPlan sp;
  if (!use_split(desc, flags, sp)) return 0;
  return split_scratch_floats(sp, batch, true);
}

int launch_dstd(const int32_t* desc, const float* weights, const float* in, float* out, long long batch,
                const cistgcn_block_taps* taps, float* scratch, size_t scratch_floats, uint32_t flags, void* stream,
                int in_bf16 = 0, int out_bf16 = 0) {
  if (int rc = check_block_desc(desc)) return rc;
  if (in_bf16 && (desc[CB_IN_MODE] == 1 || desc[CB_IN_SV] != 1 || (desc[CB_V] & 1)))
    return fail(-2, "DSTD-GC block: bf16 input needs an activation tensor with contiguous, even-length joint rows");
  SplitPlan sp;
  if (use_split(desc, flags, sp)) {
    const bool taps_hold = desc[CB_INTERP] && taps && taps->adj_s && taps->adj_t;
    const size_t need = split_scratch_floats(sp, batch, !taps_hold);
    if (!scratch || scratch_floats < need)
      return fail(-1, "DSTD-GC block: scratch too small (%zu floats given, %zu needed)", scratch_floats, need);
    return launch_dstd_split(sp, weights, in, out, batch, taps, scratch, in_bf16, out_bf16, stream);
  }
  // a shape neither path is built for: name the shapes of the default (three-stage) path
  if (!(flags & (CISTGCN_FLAG_DSTD_FUSED | CISTGCN_FLAG_DSTD_TC)) && !cg::split_shape(desc[CB_T], desc[CB_V]))
    return no_split_kernel(desc[CB_T], desc[CB_V]);
  return launch_dstd_fused(desc, weights, in, out, batch, taps, flags, in_bf16, out_bf16, stream);
}

#ifndef CISTGCN_EMU
// tcgen05 kernel (fpn_tc.cuh): 32-wide channel tiles, two 128-position tiles, weights packed with CF_TC_*.
// A layer's K is its input channels padded to 16 (one k-step): 2 k-chunks for input_n <= 16 and output_n <= 16,
// 4 for 16 < output_n <= 25.  The map's channels past output_n stay zero, so a 2-chunk layer reads only channels 0..15.
bool fpn_tc_supported(const int32_t* fpn_descs, int n_fpn, const int32_t* tail_desc) {
  const int To = tail_desc[CT_TOUT], V = tail_desc[CT_V], Tin = tail_desc[CT_TIN];
  if (To > 25 || Tin > 16 || tail_desc[CT_F] != cg::FTC_F || !cg::fpn_joints_built(V) || n_fpn > 4) return false;
  for (int l = 0; l < n_fpn; ++l) {
    const int32_t* f = fpn_descs + l * CF_COUNT;
    if (f[CF_TC_KC] != (f[CF_CIN] + 15) / 16 * 2 || f[CF_TC_W] <= 0 || f[CF_TC_PRM] <= 0) return false;
    if ((f[CF_RESID] != 0) != (l > 0)) return false;       // layer 0 reads the separate input buffer, no residual there
  }
  return true;
}

int launch_fpn_tc(const int32_t* fpn_descs, int n_fpn, const int32_t* tail_desc, const float* weights,
                  const float* in, float* x7, long long batch, void* stream, bool bf16 = false) {
  cg::FpnTcArgs a;
  memcpy(a.f, fpn_descs, sizeof(int32_t) * CF_COUNT * n_fpn);
  memcpy(a.t, tail_desc, sizeof(a.t));
  a.n_layers = n_fpn; a.w = weights; a.in = in; a.x7 = x7; a.batch = (int)batch;
  a.dbg = g_phase_clocks;     // nullptr outside -DCISTGCN_PROFILE builds
  ProfScope prof(KIND_FPN, stream);
  int e = 0;
#define CG_FPN_TC_CASE(VV) \
  if (a.t[CT_V] == VV) e = bf16 ? cg::launch_fpn_tc_impl<VV, true>(a, stream) : cg::launch_fpn_tc_impl<VV, false>(a, stream);
  CG_FPN_JOINTS(CG_FPN_TC_CASE)
#undef CG_FPN_TC_CASE
  return check_launch(e, "fpn_tc_kernel");
}
#endif

int launch_fpn(const int32_t* fpn_descs, int n_fpn, const int32_t* tail_desc, const float* weights,
               const float* in, float* x7, long long batch, uint32_t flags, void* stream, bool bf16 = false) {
  if (n_fpn < 1 || n_fpn > cg::FPN_MAX_LAYERS) return fail(-2, "FPN chain: %d layers unsupported", n_fpn);
  // descriptor consistency first: both kernels rely on it
  {
    const int To = tail_desc[CT_TOUT], Tin = tail_desc[CT_TIN], V = tail_desc[CT_V];
    if (To < 1 || Tin < 1 || V < 1) return fail(-2, "FPN chain: bad geometry (Tin=%d, Tout=%d, V=%d)", Tin, To, V);
    if (To % 5 != 0) return fail(-2, "FPN chain: output_n = %d must be a multiple of 5", To);
    if (Tin > To) return fail(-2, "FPN chain: input_n > output_n unsupported");
    if (tail_desc[CT_F] != 10) return fail(-2, "FPN chain: feature width %d unsupported (in_ch is fixed at 10)", tail_desc[CT_F]);
    for (int l = 0; l < n_fpn; ++l) {
      const int32_t* f = fpn_descs + l * CF_COUNT;
      if (f[CF_COUT] != To || f[CF_CIN] != (l == 0 ? Tin : To)) return fail(-2, "FPN chain: layer %d channel mismatch", l);
    }
  }
#ifndef CISTGCN_EMU
  if (bf16) {
    bool ok = fpn_tc_supported(fpn_descs, n_fpn, tail_desc);
    for (int l = 0; ok && l < n_fpn; ++l) ok = fpn_descs[l * CF_COUNT + CF_TC_W16] > 0;
    if (!ok) return fail(-2, "bf16 forward: the FPN stack has no tcgen05 operand image for this shape / these weights");
    return launch_fpn_tc(fpn_descs, n_fpn, tail_desc, weights, in, x7, batch, stream, true);
  }
  if (!(flags & CISTGCN_FLAG_FPN_FP32) && fpn_tc_supported(fpn_descs, n_fpn, tail_desc))
    return launch_fpn_tc(fpn_descs, n_fpn, tail_desc, weights, in, x7, batch, stream);
#else
  (void)flags;
  if (bf16) return fail(-2, "bf16 forward needs the tensor-core FPN kernel (not available in the emulator build)");
#endif
  cg::FpnArgs a;
  memcpy(a.f, fpn_descs, sizeof(int32_t) * CF_COUNT * n_fpn);
  memcpy(a.t, tail_desc, sizeof(a.t));
  a.n_layers = n_fpn; a.w = weights; a.in = in; a.x7 = x7; a.batch = (int)batch;
  const int V = a.t[CT_V];
  cg::fpn_plan(a);
  const size_t smem = (size_t)a.smem_floats * sizeof(float);
  if (smem > (size_t)kMaxSmemBytes) return fail(-2, "FPN chain needs %zu B of shared memory", smem);
  if (!cg::fpn_joints_built(V))
    return fail(-2, "FPN chain: joints = %d has no compiled kernel (built:" CG_FPN_JOINTS(CG_JOINTS_NAME) ")", V);
  ProfScope prof(KIND_FPN, stream);
  int e = 0;
#define CG_FPN_CASE(VV) \
  if (V == VV) e = cg::launch_fpn_impl<VV>(a, stream);
  CG_FPN_JOINTS(CG_FPN_CASE)
#undef CG_FPN_CASE
  return check_launch(e, "fpn_chain_kernel");
}

int launch_tail(const int32_t* tail_desc, const float* weights, const float* x, const float* x7, const float* x8,
                float* pred, const float* target, double* frame_sums, long long batch, const cistgcn_taps* taps,
                long long tap_offset, void* stream) {
  cg::TailArgs a;
  memcpy(a.t, tail_desc, sizeof(a.t));
  a.w = weights; a.x = x; a.x7 = x7; a.x8 = x8; a.pred = pred; a.target = target; a.frame_sums = frame_sums;
  a.batch = (int)batch;
  const int To = a.t[CT_TOUT], V = a.t[CT_V], H = a.t[CT_HID];
  if (H < 64 || cg::TAIL_NT % H != 0) return fail(-2, "ContextLayer hidden_dim = %d unsupported (64, 128, 256)", H);
  if (a.t[CT_SEH1] > 8 || a.t[CT_SEH2] > 8) return fail(-2, "SE hidden width > 8 unsupported");
  if (To < 1 || To > cg::TAIL_NT || V < 1) return fail(-2, "ContextLayer: output_n = %d / joints = %d unsupported (1 <= output_n <= %d)", To, V, cg::TAIL_NT);
  a.tap_joints = taps && taps->ctx_joints ? taps->ctx_joints + tap_offset * V : nullptr;
  a.tap_disp = taps && taps->ctx_displacements ? taps->ctx_displacements + tap_offset * To : nullptr;
  a.tap_sjn = taps && taps->ctx_seq_joints_n ? taps->ctx_seq_joints_n + tap_offset * To * V : nullptr;
  a.tap_sjd = taps && taps->ctx_seq_joints_dims ? taps->ctx_seq_joints_dims + tap_offset * 3 * To * V : nullptr;
  cg::tail_plan(a);
  const size_t smem = (size_t)a.smem_floats * sizeof(float);
  if (smem > (size_t)kMaxSmemBytes) return fail(-2, "ContextLayer needs %zu B of shared memory (> %d)", smem, kMaxSmemBytes);
  auto kfn = cg::tail_kernel;
  int perr = 0;
  const int per_sm = cg::prepared_blocks_per_sm(kfn, cg::TAIL_NT, smem, &perr);
  if (perr) return fail(-3, "cudaFuncSetAttribute(%zu B): %s", smem, cg::launch_error_string(perr));
  const int grid = grid_for(batch, per_sm);
  ProfScope prof(KIND_TAIL, stream);
  CG_LAUNCH(kfn, grid, cg::TAIL_NT, smem, stream, a);
  return check_launch(cg::last_launch_error(), "tail_kernel");
}

struct PlanView {
  const int32_t* hdr;
  const int32_t* in_blocks;
  const int32_t* fpn;
  const int32_t* tail;
  const int32_t* out_blocks;
  int n_in, n_fpn, n_out, len;
};

int parse_plan(const int32_t* plan, int plan_len, PlanView& pv) {
  if (!plan) return fail(-1, "plan is NULL");
  if (plan_len >= 0 && plan_len < CP_HEADER_COUNT) return fail(-1, "plan too short");
  if (plan[CP_ABI] != CISTGCN_ABI_VERSION) return fail(-1, "plan ABI %d != library ABI %d", plan[CP_ABI], CISTGCN_ABI_VERSION);
  pv.hdr = plan;
  pv.n_in = plan[CP_N_IN_BLOCKS]; pv.n_fpn = plan[CP_N_FPN]; pv.n_out = plan[CP_N_OUT_BLOCKS];
  if (pv.n_in < 1 || pv.n_in > CISTGCN_MAX_BLOCKS || pv.n_out < 1 || pv.n_out > CISTGCN_MAX_BLOCKS || pv.n_fpn < 1 ||
      pv.n_fpn > CISTGCN_MAX_FPN)
    return fail(-1, "plan block counts out of range");
  pv.len = CP_HEADER_COUNT + (pv.n_in + pv.n_out) * CB_COUNT + pv.n_fpn * CF_COUNT + CT_COUNT;
  if (plan_len >= 0 && plan_len != pv.len) return fail(-1, "plan length %d, expected %d", plan_len, pv.len);
  pv.in_blocks = plan + CP_HEADER_COUNT;
  pv.fpn = pv.in_blocks + pv.n_in * CB_COUNT;
  pv.tail = pv.fpn + pv.n_fpn * CF_COUNT;
  pv.out_blocks = pv.tail + CT_COUNT;
  return 0;
}

size_t act_floats_per_sample(const int32_t* hdr) {
  const int T = hdr[CP_TIN], To = hdr[CP_TOUT], V = hdr[CP_V];
  return (size_t)hdr[CP_CMAX] * V * (T > To ? T : To);
}

}  // namespace

extern "C" {

const char* cistgcn_last_error(void) { return g_err.c_str(); }
int cistgcn_abi_version(void) { return CISTGCN_ABI_VERSION; }

int cistgcn_debug_phase_clocks(void* device_buffer) {
#ifdef CISTGCN_PROFILE
  g_phase_clocks = reinterpret_cast<long long*>(device_buffer);
  return 0;
#else
  (void)device_buffer;
  return fail(-5, "cistgcn_debug_phase_clocks: library built without -DCISTGCN_PROFILE (the kernels carry no clock reads)");
#endif
}

int cistgcn_debug_stamp_iteration(int iteration) {
#ifdef CISTGCN_PROFILE
  g_stamp_iter = iteration < 0 ? 0 : iteration;
  return 0;
#else
  (void)iteration;
  return fail(-5, "cistgcn_debug_stamp_iteration: library built without -DCISTGCN_PROFILE");
#endif
}

const char* cistgcn_profile_kind_name(int kind) {
  return (kind >= 0 && kind < KIND_COUNT) ? kKindNames[kind] : "";
}

int cistgcn_profile_enable(int on) {
#ifndef CISTGCN_EMU
  std::lock_guard<std::mutex> lock(g_prof.mu);
  g_prof.on = on != 0;
  g_prof.used = 0;
  for (int k = 0; k < KIND_COUNT; ++k) g_prof.launches[k] = 0;
#else
  (void)on;
#endif
  return 0;
}

int cistgcn_profile_read(double* ms_by_kind, int64_t* launches_by_kind) {
  for (int k = 0; k < KIND_COUNT; ++k) { if (ms_by_kind) ms_by_kind[k] = 0.0; if (launches_by_kind) launches_by_kind[k] = 0; }
#ifndef CISTGCN_EMU
  if (cudaDeviceSynchronize() != cudaSuccess) return fail(-4, "profile_read: device synchronize failed");
  std::lock_guard<std::mutex> lock(g_prof.mu);
  for (size_t i = 0; i < g_prof.used; ++i) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, g_prof.slots[i].beg, g_prof.slots[i].end) == cudaSuccess && ms_by_kind)
      ms_by_kind[g_prof.slots[i].kind] += ms;
  }
  for (int k = 0; k < KIND_COUNT; ++k) { if (launches_by_kind) launches_by_kind[k] = g_prof.launches[k]; g_prof.launches[k] = 0; }
  g_prof.used = 0;
#endif
  return 0;
}

// workspace layout per chunk: [act0][act1][x7][x8][DSTD scratch (max over blocks)], every region 256-byte aligned
static size_t align64f(size_t floats) { return (floats + 63) & ~(size_t)63; }

static size_t plan_scratch_floats(const PlanView& pv, uint32_t flags, long long chunk) {
  size_t mx = 0;
  for (int i = 0; i < pv.n_in; ++i) { const size_t n = dstd_scratch_floats(pv.in_blocks + i * CB_COUNT, flags, chunk); if (n > mx) mx = n; }
  for (int i = 0; i < pv.n_out; ++i) { const size_t n = dstd_scratch_floats(pv.out_blocks + i * CB_COUNT, flags, chunk); if (n > mx) mx = n; }
  return mx;
}

size_t cistgcn_workspace_bytes(const int32_t* plan, int64_t batch) {
  PlanView pv;
  if (parse_plan(plan, -1, pv)) return 0;
  const long long chunk = batch < CISTGCN_MAX_CHUNK ? (batch > 0 ? batch : 1) : CISTGCN_MAX_CHUNK;
  const size_t act = align64f((size_t)chunk * act_floats_per_sample(plan));
  const size_t xo = align64f((size_t)chunk * plan[CP_TOUT] * plan[CP_V] * 3);
  const size_t scratch = align64f(plan_scratch_floats(pv, (uint32_t)plan[CP_FLAGS], chunk));
  return (2 * act + 2 * xo + scratch) * sizeof(float) + 256;
}

// The forward's per-chunk regions inside a caller's workspace (layout above); `end` is the first float past them
struct ChunkWorkspace {
  float *act0, *act1, *x7, *x8, *scratch, *end;
  size_t scratch_floats;
};

static ChunkWorkspace chunk_workspace(const PlanView& pv, const int32_t* plan, long long chunk_max, void* workspace) {
  const size_t act = align64f((size_t)chunk_max * act_floats_per_sample(plan));
  const size_t xo = align64f((size_t)chunk_max * plan[CP_TOUT] * plan[CP_V] * 3);
  ChunkWorkspace w;
  w.act0 = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
  w.act1 = w.act0 + act;
  w.x7 = w.act1 + act;
  w.x8 = w.x7 + xo;
  w.scratch = w.x8 + xo;
  w.scratch_floats = align64f(plan_scratch_floats(pv, (uint32_t)plan[CP_FLAGS], chunk_max));
  w.end = w.scratch + w.scratch_floats;
  return w;
}

// The whole model on one chunk of n samples: x (n, Tin, V, 3) -> pred (n, Tout, V, 3) (+ MPJPE sums against target);
// s = the chunk's first sample in the taps
static int forward_chunk(const PlanView& pv, const float* weights, const float* x, float* pred, const float* target,
                         double* frame_sums, long long n, const cistgcn_taps* taps, long long s, const ChunkWorkspace& w,
                         uint32_t flags, void* stream, bool act_bf16) {
  auto block_taps = [&](const cistgcn_block_taps& src, const int32_t* bd) {
    cistgcn_block_taps bt = {nullptr, nullptr, nullptr, nullptr};
    const size_t tv = (size_t)bd[CB_T] * bd[CB_V];
    bt.adj_s = src.adj_s ? src.adj_s + (size_t)s * tv * bd[CB_T] : nullptr;
    bt.adj_t = src.adj_t ? src.adj_t + (size_t)s * tv * bd[CB_V] : nullptr;
    bt.w1 = src.w1 ? src.w1 + (size_t)s * bd[CB_CO] : nullptr;
    bt.w2 = src.w2 ? src.w2 + (size_t)s * bd[CB_CO] : nullptr;
    return bt;
  };
  const float* cur = x;
  float* bufs[2] = {w.act0, w.act1};
  int flip = 0;
  for (int i = 0; i < pv.n_in; ++i) {
    const int32_t* bd = pv.in_blocks + i * CB_COUNT;
    cistgcn_block_taps bt = {nullptr, nullptr, nullptr, nullptr};
    if (taps) bt = block_taps(taps->in_blocks[i], bd);
    float* dst = bufs[flip];
    // bf16 forward: every inter-block activation of the input stack (and the FPN's input) is stored as bf16
    if (int rc = launch_dstd(bd, weights, cur, dst, n, taps ? &bt : nullptr, w.scratch, w.scratch_floats, flags, stream,
                             act_bf16 && i > 0, act_bf16))
      return rc;
    cur = dst;
    flip ^= 1;
  }
  if (int rc = launch_fpn(pv.fpn, pv.n_fpn, pv.tail, weights, cur, w.x7, n, flags, stream, act_bf16)) return rc;
  cur = w.x7;
  for (int i = 0; i < pv.n_out; ++i) {
    const int32_t* bd = pv.out_blocks + i * CB_COUNT;
    cistgcn_block_taps bt = {nullptr, nullptr, nullptr, nullptr};
    if (taps) bt = block_taps(taps->out_blocks[i], bd);
    float* dst = (i == pv.n_out - 1) ? w.x8 : bufs[flip];
    if (int rc = launch_dstd(bd, weights, cur, dst, n, taps ? &bt : nullptr, w.scratch, w.scratch_floats, flags, stream)) return rc;
    cur = dst;
    flip ^= 1;
  }
  return launch_tail(pv.tail, weights, x, w.x7, w.x8, pred, target, frame_sums, n, taps, s, stream);
}

static int forward_impl(const int32_t* plan, int32_t plan_len, const float* weights, const float* x, float* pred,
                        const float* target, double* frame_sums, void* workspace, size_t workspace_bytes,
                        int64_t batch, const cistgcn_taps* taps, void* stream, bool act_bf16) {
  PlanView pv;
  if (int rc = parse_plan(plan, plan_len, pv)) return rc;
  if (batch < 0) return fail(-1, "negative batch");
  if (batch == 0) return 0;
  if (!weights || !x || !pred || !workspace) return fail(-1, "NULL buffer");
  if ((target == nullptr) != (frame_sums == nullptr)) return fail(-1, "target and frame_sums must be given together");
  if (workspace_bytes < cistgcn_workspace_bytes(plan, batch)) return fail(-1, "workspace too small");
  const uint32_t flags = (uint32_t)plan[CP_FLAGS];
  const int T = plan[CP_TIN], To = plan[CP_TOUT], V = plan[CP_V];
  const long long chunk_max = batch < CISTGCN_MAX_CHUNK ? batch : CISTGCN_MAX_CHUNK;
  const ChunkWorkspace w = chunk_workspace(pv, plan, chunk_max, workspace);
  for (long long s = 0; s < batch; s += chunk_max) {
    const long long n = (batch - s) < chunk_max ? (batch - s) : chunk_max;
    if (int rc = forward_chunk(pv, weights, x + (size_t)s * T * V * 3, pred + (size_t)s * To * V * 3,
                               target ? target + (size_t)s * To * V * 3 : nullptr, frame_sums, n, taps, s, w, flags,
                               stream, act_bf16))
      return rc;
  }
  return 0;
}

int cistgcn_forward_f32(const int32_t* plan, int32_t plan_len, const float* weights, const float* x, float* pred,
                        const float* target, double* frame_sums, void* workspace, size_t workspace_bytes,
                        int64_t batch, const cistgcn_taps* taps, void* stream) {
  return forward_impl(plan, plan_len, weights, x, pred, target, frame_sums, workspace, workspace_bytes, batch, taps, stream, false);
}

int cistgcn_forward_bf16(const int32_t* plan, int32_t plan_len, const float* weights, const float* x, float* pred,
                         const float* target, double* frame_sums, void* workspace, size_t workspace_bytes,
                         int64_t batch, const cistgcn_taps* taps, void* stream) {
  return forward_impl(plan, plan_len, weights, x, pred, target, frame_sums, workspace, workspace_bytes, batch, taps, stream, true);
}

// rollout workspace per chunk: the forward's, then [window (Tin frames)][step prediction (Tout frames)], 256-byte aligned
size_t cistgcn_rollout_workspace_bytes(const int32_t* plan, int64_t batch) {
  const size_t fwd = cistgcn_workspace_bytes(plan, batch);
  if (!fwd) return 0;
  const long long chunk = batch < CISTGCN_MAX_CHUNK ? (batch > 0 ? batch : 1) : CISTGCN_MAX_CHUNK;
  const size_t pose = (size_t)chunk * plan[CP_V] * 3;
  return fwd + (align64f(pose * plan[CP_TIN]) + align64f(pose * plan[CP_TOUT])) * sizeof(float);
}

// K = ceil(horizon / Tout) forwards per chunk, back to back on the caller's stream; step k reads the window written by
// step k - 1 (the chunk's x for k = 0) and rollout_step_kernel scatters its prediction
static int rollout_impl(const int32_t* plan, int32_t plan_len, const float* weights, const float* x, int32_t horizon,
                        float* out, const float* target, double* frame_sums, void* workspace, size_t workspace_bytes,
                        int64_t batch, void* stream, bool act_bf16) {
  PlanView pv;
  if (int rc = parse_plan(plan, plan_len, pv)) return rc;
  if (batch < 0) return fail(-1, "negative batch");
  if (horizon < 1) return fail(-1, "rollout: horizon = %d, must be >= 1", horizon);
  if (batch == 0) return 0;
  if (!weights || !x || !out || !workspace) return fail(-1, "NULL buffer");
  if ((target == nullptr) != (frame_sums == nullptr)) return fail(-1, "target and frame_sums must be given together");
  const size_t need = cistgcn_rollout_workspace_bytes(plan, batch);
  if (workspace_bytes < need) return fail(-1, "rollout: workspace too small (%zu bytes given, %zu needed)", workspace_bytes, need);
  const uint32_t flags = (uint32_t)plan[CP_FLAGS];
  const int T = plan[CP_TIN], To = plan[CP_TOUT], V = plan[CP_V];
  const long long chunk_max = batch < CISTGCN_MAX_CHUNK ? batch : CISTGCN_MAX_CHUNK;
  const ChunkWorkspace w = chunk_workspace(pv, plan, chunk_max, workspace);
  float* window = w.end;
  float* step = window + align64f((size_t)chunk_max * T * V * 3);
  const int K = (horizon + To - 1) / To;
  for (long long s = 0; s < batch; s += chunk_max) {
    const long long n = (batch - s) < chunk_max ? (batch - s) : chunk_max;
    const float* in = x + (size_t)s * T * V * 3;
    for (int k = 0; k < K; ++k) {
      if (int rc = forward_chunk(pv, weights, in, step, nullptr, nullptr, n, nullptr, 0, w, flags, stream, act_bf16)) return rc;
      const int t0 = k * To, nf = horizon - t0 < To ? horizon - t0 : To;
      int e;
      { ProfScope prof(KIND_OTHER, stream);
        e = cg::launch_rollout_step(step, out + (size_t)s * horizon * V * 3, k + 1 < K ? window : nullptr,
                                    target ? target + (size_t)s * horizon * V * 3 : nullptr, frame_sums, n, t0, nf,
                                    horizon, T, To, V, stream); }
      if (e) return check_launch(e, "rollout_step_kernel");
      in = window;
    }
  }
  return 0;
}

int cistgcn_rollout_f32(const int32_t* plan, int32_t plan_len, const float* weights, const float* x, int32_t horizon,
                        float* out, const float* target, double* frame_sums, void* workspace, size_t workspace_bytes,
                        int64_t batch, void* stream) {
  return rollout_impl(plan, plan_len, weights, x, horizon, out, target, frame_sums, workspace, workspace_bytes, batch,
                      stream, false);
}

int cistgcn_rollout_bf16(const int32_t* plan, int32_t plan_len, const float* weights, const float* x, int32_t horizon,
                         float* out, const float* target, double* frame_sums, void* workspace, size_t workspace_bytes,
                         int64_t batch, void* stream) {
  return rollout_impl(plan, plan_len, weights, x, horizon, out, target, frame_sums, workspace, workspace_bytes, batch,
                      stream, true);
}

size_t cistgcn_dstd_block_workspace_bytes(const int32_t* block_desc, int64_t batch) {
  if (!block_desc || batch <= 0) return 0;
  return dstd_scratch_floats(block_desc, 0, batch) * sizeof(float) + 256;
}

int cistgcn_dstd_block_f32(const int32_t* block_desc, const float* weights, const float* in, float* out,
                           int64_t batch, const cistgcn_block_taps* taps, void* workspace, size_t workspace_bytes,
                           uint32_t flags, void* stream) {
  if (!block_desc || !weights || !in || !out) return fail(-1, "NULL buffer");
  if (batch <= 0) return batch == 0 ? 0 : fail(-1, "negative batch");
  float* ws = nullptr;
  size_t ws_floats = 0;
  if (workspace) {
    const uintptr_t base = (reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255);
    const size_t skipped = base - reinterpret_cast<uintptr_t>(workspace);
    if (workspace_bytes > skipped) { ws = reinterpret_cast<float*>(base); ws_floats = (workspace_bytes - skipped) / sizeof(float); }
  }
  return launch_dstd(block_desc, weights, in, out, batch, taps, ws, ws_floats, flags, stream);
}

int cistgcn_fpn_chain_f32(const int32_t* fpn_descs, int32_t n_fpn, const int32_t* tail_desc, const float* weights,
                          const float* in, float* x7, int64_t batch, uint32_t flags, void* stream) {
  if (!fpn_descs || !tail_desc || !weights || !in || !x7) return fail(-1, "NULL buffer");
  if (batch <= 0) return batch == 0 ? 0 : fail(-1, "negative batch");
  return launch_fpn(fpn_descs, n_fpn, tail_desc, weights, in, x7, batch, flags, stream);
}

int cistgcn_tail_f32(const int32_t* tail_desc, const float* weights, const float* x, const float* x7,
                     const float* x8, float* pred, const float* target, double* frame_sums, int64_t batch,
                     const cistgcn_taps* taps, void* stream) {
  if (!tail_desc || !weights || !x || !x7 || !x8 || !pred) return fail(-1, "NULL buffer");
  if ((target == nullptr) != (frame_sums == nullptr)) return fail(-1, "target and frame_sums must be given together");
  if (batch <= 0) return batch == 0 ? 0 : fail(-1, "negative batch");
  return launch_tail(tail_desc, weights, x, x7, x8, pred, target, frame_sums, batch, taps, 0, stream);
}

int cistgcn_mpjpe_f32(const float* pred, const float* target, int64_t batch, int32_t T, int32_t V, float* err,
                      double* frame_sums, void* stream) {
  if (!pred || !target) return fail(-1, "NULL buffer");
  if (T <= 0 || V <= 0) return fail(-1, "mpjpe: T = %d, V = %d must be positive", T, V);
  if (batch <= 0) return batch == 0 ? 0 : fail(-1, "negative batch");
  cg::MpjpeArgs a;
  a.pred = pred; a.target = target; a.err = err; a.frame_sums = frame_sums;
  a.n = (long long)batch * T * V; a.T = T; a.V = V;
  long long blocks = (a.n + 255) / 256;
  const long long cap = (long long)sm_count() * 8;
  auto kfn = cg::mpjpe_kernel;
  ProfScope prof(KIND_MPJPE, stream);
  CG_LAUNCH(kfn, (int)(blocks < cap ? blocks : cap), 256, 0, stream, a);
  return check_launch(cg::last_launch_error(), "mpjpe_kernel");
}

int cistgcn_mpjpe_grouped_f32(const float* pred, const float* target, const int32_t* groups, int32_t n_groups, int64_t batch,
                              int32_t T, int32_t V, double* sums, int64_t* counts, void* stream) {
  if (!pred || !target || !sums || !counts) return fail(-1, "mpjpe_grouped: NULL buffer");
  if (n_groups < 1 || T < 1 || V < 1 || (long long)n_groups * T > 0x7fffffffLL)
    return fail(-1, "mpjpe_grouped: n_groups = %d, T = %d, V = %d must be positive (n_groups * T < 2^31)", n_groups, T, V);
  if (batch <= 0) return batch == 0 ? 0 : fail(-1, "negative batch");
  ProfScope prof(KIND_MPJPE, stream);
  return check_launch(cg::launch_mpjpe_grouped(pred, target, groups, n_groups, batch, T, V, sums,
                                               reinterpret_cast<long long*>(counts), stream), "grouped_mpjpe_kernel");
}

}  // extern "C"
