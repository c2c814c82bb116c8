// DSTD-GC block, stage 1 of 3: everything that REDUCES the normalised tile to small per-sample vectors
// (reference: models/CISTGCN/CISTGCN.py:360-371 _get_stats_, :323-326 conv_{s,t}.0-3, :138-142 / :146-150 the first
// two convolutions of Map2Adj's time_compress / joint_compress, for both domains).
//
// Round 1 ran these phases inside the fused per-sample CTA: ~8 barrier-separated phases on 16 warps at 7 % FMA
// efficiency.  Here ONE WARP owns one sample and there is no block-level barrier at all: the warp streams the sample
// frame by frame ("slab" = one t, Ci x V values), so its live state is a 3 KB slab instead of the 28 KB tile, and
// 12-16 independent samples are in flight per SM.  Per slab:
//   load     lanes = joints: coalesced row loads (or the 10-feature build of CISTGCN.py:568-577), global_norm folded
//   stats    lanes = channels: row mean / variance over the joints; merged over frames with Chan's update
//   mix      lanes = OUTPUT channels of the stacked 1x1 convolutions (4*Ch Map2Adj entry maps + 2*Cg gate-conv maps),
//            register tile over the V joints: per input channel one conflict-free weight LDS per output + V/4 broadcast
//            LDS.128 of the slab row feed 3*V FFMAs.  The gate conv (T,1) is the same GEMM with per-frame weights,
//            accumulated over the slabs in registers.
//            MMA variant (T = 10, Ci >= 16): the same GEMMs as 3xTF32 mma.sync.m16n8k8 -- rows = output channels,
//            columns = joints, k = input channels; the slab rows are split into hi + lo once per k step and shared by
//            the entry maps and the gate conv; the weights are ONE fp32 fragment image per matrix, split in the loop
//            (a second, lo image would cost resident warps); the accumulator fragments go to the map buffer with
//            conflict-free 64-bit stores (row stride = 8 mod 16).
//   collapse lanes = the 2*Ch outputs (both domains) of time_compress.3 (accumulated over slabs) and
//            joint_compress.3 (complete per slab; MMA variant: its weights as [c'][v / 4][lane][4], one LDS.128 per
//            four FFMAs on four independent chains).
// Output per sample (the `red` record, float offsets from RedLayout): tc [2*Ch][V] and jc [2*Ch][T] (after BN), then
// stats [2+2T] and h1 [2*Cg][V] (after BN + PReLU) -- the gate inputs come last because stage 2 (dstd_adj.cuh), which
// turns the record into the gates and the adjacencies, reuses their room for dim_seq / dim_space.
#pragma once
#include "../../include/cistgcn_b200.h"
#include "host_util.h"
#include "simt.h"

namespace cg {

__host__ __device__ inline int rpad4(int n) { return (n + 3) & ~3; }
__host__ __device__ inline int rpad32(int n) { return (n + 31) & ~31; }
__host__ __device__ inline int rmin(int a, int b) { return a < b ? a : b; }
__host__ __device__ inline int rmax(int a, int b) { return a > b ? a : b; }
constexpr int RED_MAX_WARPS = 12;      // 384 threads: up to 168 registers per thread
// Row stride of the per-warp map buffer.  FFMA variant: 4 x odd, so that lanes = rows conflict only 4-way on the transposing
// store; tensor-core variant: = 8 (mod 16), so that the accumulator-fragment stores (8 rows x 4 column pairs per
// half-warp) are conflict free.
__host__ __device__ constexpr int red_as(int V, bool mma) {
  const int xs = (V + 3) & ~3;
  return mma ? ((xs + 7) / 16) * 16 + 8 : ((xs % 8 == 4) ? xs : xs + 4);
}

// Float offsets inside one sample's `red` record.  The Map2Adj maps come first and the gate inputs (statistics, hidden
// maps) last: stage 2 is done with the latter before it needs room for dim_seq / dim_space, which alias them.
struct RedLayout {
  int stats, h1, h1g, tc, jc, total;
  __host__ __device__ RedLayout(int T, int V, int Cg, int Ch, bool interp) {
    tc = 0;
    jc = tc + (interp ? rpad4(2 * Ch * V) : 0);
    stats = jc + (interp ? rpad4(2 * Ch * T) : 0);
    h1 = stats + rpad4(2 + 2 * T);
    h1g = rpad4(Cg * V);                 // each gate's hidden map starts 16-byte aligned (stage 2 reads it with LDS.128)
    total = h1 + 2 * h1g;
  }
};

struct ReduceArgs {
  int d[CB_COUNT];
  const float* w;
  const float* in;
  float* red;
  int batch, red_stride;
  int in_bf16;                      // the input activation tensor is stored as bf16 (cistgcn_forward_bf16; needs sv == 1, V even)
  int nwarps;                       // warps per CTA (= samples in flight per CTA)
  int o_a0, o_g0, o_tc3, o_jc3;     // resident matrices (shared-memory float offsets)
  int o_gn_s, o_gn_b, o_a0_b, o_a0_a, o_g0_b, o_g0_a, o_tc3_b, o_jc3_b;   // resident vectors
  int mp_e, mp_g, mp_c;             // row lengths: pad32(4Ch), pad32(2Cg), pad32(2Ch)
  int o_warp, warp_floats, smem_floats;
  int mma;                          // stacked 1x1 convolutions (Map2Adj entry maps + gate conv) on 3xTF32 mma.sync
  int ks, mte, mtg;                 // MMA variant: k steps of 8 input channels, 16-row tiles of the entry maps / the gate conv
};

// Host: shared-memory plan.  Returns false when the shape is outside this kernel's register tiling
// (4*Ch <= 32*NE_MAX, 2*Cg <= 32, Ci <= 32) or the resident weights leave no room for >= 4 warps.
constexpr int RED_NE_MAX = 2;
inline bool reduce_plan(ReduceArgs& a, int max_smem_floats, bool mma = true) {
  const int* d = a.d;
  const int Ci = d[CB_CI], T = d[CB_T], V = d[CB_V], Ch = d[CB_CH], Cg = d[CB_CG];
  const bool interp = d[CB_INTERP] != 0;
  if (Ci > 32 || 2 * Cg > 32 || (interp && 4 * Ch > 32 * RED_NE_MAX)) return false;
  a.mp_e = rpad32(4 * Ch); a.mp_g = rpad32(2 * Cg); a.mp_c = rpad32(2 * Ch);
  int cur = 0;
  auto take = [&](int n) { const int o = cur; cur += rpad4(n); return o; };
  // tensor-core variant: the input blocks (T = 10) from 16 input channels up (K = 10 padded to 16 loses to the FFMA loops); the matrices of the stacked 1x1 convolutions
  // are then held as fragment-ordered images [row tile][k step][lane][4]
  a.mma = mma && T == 10 && Ci >= 16;
  a.ks = (Ci + 7) / 8; a.mte = interp ? (4 * Ch + 15) / 16 : 0; a.mtg = (2 * Cg + 15) / 16;
  a.o_g0 = take(a.mma ? T * a.mtg * a.ks * 128 : Ci * T * a.mp_g);
  a.o_a0 = interp ? take(a.mma ? a.mte * a.ks * 128 : Ci * a.mp_e) : 0;
  a.o_tc3 = interp ? take(a.mma ? T * 2 * ((Ch + 7) / 8) * 128 : Ch * T * a.mp_c) : 0;   // tensor-core variant: [t][domain][k step][lane][4]
  a.o_jc3 = interp ? take(Ch * (a.mma ? rpad4(V) : V) * a.mp_c) : 0;     // tensor-core variant: [c'][v / 4][lane][4], v padded
  a.o_gn_s = take(Ci); a.o_gn_b = take(Ci);
  a.o_g0_b = take(a.mp_g); a.o_g0_a = take(2);
  a.o_a0_b = take(a.mp_e); a.o_a0_a = take(4);
  a.o_tc3_b = take(a.mp_c); a.o_jc3_b = take(a.mp_c);
  const int XS = rpad4(V), XT = V | 1, AS = red_as(V, a.mma != 0);
  const int rows_ag = interp ? 4 * Ch : 0;
  int region = Ci * XT;                                           // transposed slab copy (stats) aliases the map buffer
  if (rows_ag * AS > region) region = rows_ag * AS;
  if (2 * Cg * AS > region) region = 2 * Cg * AS;                 // output staging of h1 / tc
  if (2 * Ch * AS > region) region = 2 * Ch * AS;
  a.warp_floats = rpad4(Ci * XS) + rpad4(region);
  a.o_warp = cur;
  int nw = (max_smem_floats - cur) / a.warp_floats;
  if (nw > RED_MAX_WARPS) nw = RED_MAX_WARPS;
  if (nw < 4) return false;
  a.nwarps = nw;
  a.smem_floats = cur + nw * a.warp_floats;
  return true;
}

// c[mt][nt] += W (fragment image of an fp32 matrix, split into hi + lo here) * slab (B fragments, already split), k step ks.
// Row tiles go in pairs and the three products of one accumulator are issued 2 * NTL MMAs apart, smallest terms first.
template <int MT, int NTL>
CG_DEV void reduce_mma_rows(float (&acc)[MT][NTL][4], const float* frag, int mt_used, int KS, int ks,
                            const float (&bh)[NTL][2], const float (&bl)[NTL][2]) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int mp = 0; mp < MT; mp += 2) {
    if (mp < mt_used) {
      const bool two = mp + 1 < MT && mp + 1 < mt_used;
      float ah[2][4], al[2][4];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int mt = (u == 0 || two) ? mp + u : mp;
        const float4 w4 = *reinterpret_cast<const float4*>(frag + ((mt * KS + ks) * 32 + lane) * 4);
        tf32_split(w4.x, ah[u][0], al[u][0]); tf32_split(w4.y, ah[u][1], al[u][1]);
        tf32_split(w4.z, ah[u][2], al[u][2]); tf32_split(w4.w, ah[u][3], al[u][3]);
      }
#pragma unroll
      for (int term = 0; term < 3; ++term)
#pragma unroll
        for (int u = 0; u < 2; ++u)
          if (mp + u < MT && (u == 0 || two)) {
#pragma unroll
            for (int nt = 0; nt < NTL; ++nt) {
              if (term == 0) mma_tf32(acc[mp + u][nt], al[u], bh[nt]);
              else if (term == 1) mma_tf32(acc[mp + u][nt], ah[u], bl[nt]);
              else mma_tf32(acc[mp + u][nt], ah[u], bh[nt]);
            }
          }
    }
  }
}

// Fragment-ordered image of an M x K matrix given as src(m, k): dst[((mt * KS + ks) * 32 + lane) * 4 + j] with
// m = 16 mt + lane / 4 + 8 (j & 1), k = 8 ks + lane % 4 + 4 (j >> 1); zero outside the matrix.
template <class SRC>
CG_DEV void build_reduce_frags(float* dst, int MT, int KS, int M, int K, int nthreads, SRC src) {
  for (int i = threadIdx.x; i < MT * KS * 128; i += nthreads) {
    const int j = i & 3, ln = (i >> 2) & 31, tile = i >> 7, ks = tile % KS, mt = tile / KS;
    const int m = 16 * mt + (ln >> 2) + ((j & 1) ? 8 : 0), k = 8 * ks + (ln & 3) + ((j & 2) ? 4 : 0);
    dst[i] = (m < M && k < K) ? src(m, k) : 0.f;
  }
}

template <int T, int V, int NE, bool MMA = false>
__global__ void __launch_bounds__(32 * RED_MAX_WARPS, 1) dstd_reduce_kernel(const ReduceArgs a) {
  CG_DYN_SMEM(smem);
  constexpr int XS = (V + 3) & ~3;                 // slab row stride (LDS.128 broadcast reads)
  constexpr int XT = V | 1;                        // transposed-use copy: odd stride, lanes = channels read columns
  constexpr int AS = red_as(V, MMA);               // map row stride
  constexpr int V4 = XS / 4;
  constexpr int TV = T * V;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nthreads = blockDim.x;
  const int* d = a.d;
  const int Ci = d[CB_CI], Ch = d[CB_CH], Cg = d[CB_CG];
  const bool interp = d[CB_INTERP] != 0;
  const RedLayout RL(T, V, Cg, Ch, interp);
  const float* __restrict__ W = a.w;

  // ---------------- once per launch: resident weights -> shared memory
  {
    auto cp = [&](int dst, int field, int n) {
      for (int i = threadIdx.x; i < n; i += nthreads) smem[dst + i] = __ldg(W + d[field] + i);
    };
    if constexpr (MMA) {
      const int mpg_ = a.mp_g, mpe_ = a.mp_e;
      for (int t = 0; t < T; ++t)                    // gate conv (T,1): one image per frame, rows (c*T + t) of the k-major matrix
        build_reduce_frags(smem + a.o_g0 + t * a.mtg * a.ks * 128, a.mtg, a.ks, 2 * Cg, Ci, nthreads,
                           [&](int m, int k) { return __ldg(W + d[CB_R_G0_WT] + (size_t)(k * T + t) * mpg_ + m); });
      if (interp)
        build_reduce_frags(smem + a.o_a0, a.mte, a.ks, 4 * Ch, Ci, nthreads,
                           [&](int m, int k) { return __ldg(W + d[CB_R_A0_WT] + (size_t)k * mpe_ + m); });
    } else {
      cp(a.o_g0, CB_R_G0_WT, Ci * T * a.mp_g);
      if (interp) cp(a.o_a0, CB_R_A0_WT, Ci * a.mp_e);
    }
    cp(a.o_gn_s, CB_GN_S, Ci); cp(a.o_gn_b, CB_GN_B, Ci);
    cp(a.o_g0_b, CB_R_G0_B, a.mp_g); cp(a.o_g0_a, CB_G0_A, 2);
    if (interp) {
      if constexpr (MMA) {
        // time_compress.3 (T,1): per frame and domain one 16 x Ch fragment image (rows = outputs o, k = input channel c')
        const int mpc_ = a.mp_c, ksc = (Ch + 7) / 8;
        for (int tl = 0; tl < T * 2; ++tl) {
          const int t = tl >> 1, L = tl & 1;
          build_reduce_frags(smem + a.o_tc3 + tl * ksc * 128, 1, ksc, Ch, Ch, nthreads,
                             [&](int m, int k) { return __ldg(W + d[CB_R_TC3_WT] + (size_t)(k * T + t) * mpc_ + L * Ch + m); });
        }
      } else {
        cp(a.o_tc3, CB_R_TC3_WT, Ch * T * a.mp_c);
      }
      if constexpr (MMA) {
        // joint_compress.3 weights as [c'][v / 4][lane = output][4 joints]: one conflict-free LDS.128 per four FFMAs
        const int mpc_ = a.mp_c;
        for (int i = threadIdx.x; i < Ch * XS * mpc_; i += nthreads) {
          const int e = i & 3, ln = (i >> 2) % mpc_, rest = (i >> 2) / mpc_, v = 4 * (rest % V4) + e, cp_ = rest / V4;
          smem[a.o_jc3 + i] = v < V ? __ldg(W + d[CB_R_JC3_WT] + (size_t)(cp_ * V + v) * mpc_ + ln) : 0.f;
        }
      } else {
        cp(a.o_jc3, CB_R_JC3_WT, Ch * V * a.mp_c);
      }
      cp(a.o_a0_b, CB_R_A0_B, a.mp_e); cp(a.o_a0_a, CB_A0_A, 4);
      cp(a.o_tc3_b, CB_R_TC3_B, a.mp_c); cp(a.o_jc3_b, CB_R_JC3_B, a.mp_c);
    }
  }
  if constexpr (MMA) {
    // the padding joints of the map rows meet zero weights in the collapse stage: they must hold finite values
    for (int i = threadIdx.x; i < a.nwarps * a.warp_floats; i += nthreads) smem[a.o_warp + i] = 0.f;
  }
  __syncthreads();
  const float* gs = smem + a.o_gn_s;
  const float* gb = smem + a.o_gn_b;
  const float* wa0 = smem + a.o_a0;
  const float* wg0 = smem + a.o_g0;
  const float* wtc = smem + a.o_tc3;
  const float* wjc = smem + a.o_jc3;
  const int mpe = a.mp_e, mpg = a.mp_g, mpc = a.mp_c;
  float* xs = smem + a.o_warp + warp * a.warp_floats;      // [Ci][XS]
  float* ag = xs + rpad4(Ci * XS);                         // [4Ch][AS] maps | [Ci][XT] transposed slab | output staging
  const bool wactive = warp < a.nwarps;

  // per-lane constants of the collapse stage: lane = output (L, o) of both domains
  const int L3 = (lane < 2 * Ch && Ch > 0) ? lane / Ch : 0;
  const float* arow_tc = ag + (2 * L3 * Ch) * AS;          // time_compress map rows of domain L3
  const float* arow_jc = ag + ((2 * L3 + 1) * Ch) * AS;    // joint_compress map rows
  float e_b[NE], e_a[NE];
#pragma unroll
  for (int j = 0; j < NE; ++j) {
    const int m = lane + 32 * j;
    e_b[j] = interp ? smem[a.o_a0_b + m] : 0.f;
    e_a[j] = interp ? smem[a.o_a0_a + rmin(m / rmax(Ch, 1), 3)] : 0.f;
  }

  // tensor-core variant: fragment geometry (lane = 4 g + q) and the epilogue constants of the rows this lane holds
  constexpr int NTL = (V + 7) / 8, MTE = 2 * NE;
  const int g = lane >> 2, q = lane & 3;
  float me_b[MTE][2], me_a[MTE][2];
  if constexpr (MMA) {
#pragma unroll
    for (int mt = 0; mt < MTE; ++mt)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int m = rmin(16 * mt + g + 8 * h, rmax(4 * Ch - 1, 0));
        me_b[mt][h] = interp ? smem[a.o_a0_b + m] : 0.f;
        me_a[mt][h] = interp ? smem[a.o_a0_a + rmin(m / rmax(Ch, 1), 3)] : 0.f;
      }
  }

  bool first_sample = true;
  for (int b = blockIdx.x * a.nwarps + warp; wactive && b < a.batch; b += gridDim.x * a.nwarps) {
    float* red = a.red + (size_t)b * a.red_stride;
    const float* src = a.in + (size_t)b * d[CB_IN_SB];
    const int sc = d[CB_IN_SC], st = d[CB_IN_ST], sv = d[CB_IN_SV];
    const bool ibf = a.in_bf16 != 0;
    auto gather_slab = [&](size_t sample_off, int tt) {    // lanes = joints: Ci coalesced row copies, no register staging
      if (!ibf) {
        if (lane < V) {
          const float* p = a.in + sample_off + tt * st + lane * sv;
#pragma unroll 8
          for (int c = 0; c < Ci; ++c) cp_async4(xs + c * XS + lane, p + c * sc);
        }
      } else if (lane < V / 2) {                           // bf16 rows: joint pairs as 4-byte copies into the row's first words
        const unsigned short* p = reinterpret_cast<const unsigned short*>(a.in) + sample_off + tt * st + 2 * lane;
#pragma unroll 8
        for (int c = 0; c < Ci; ++c) cp_async4(xs + c * XS + lane, reinterpret_cast<const float*>(p + c * sc));
      }
      cp_async_commit();
    };
    const size_t sample_off = (size_t)b * d[CB_IN_SB];
    const bool gathered = d[CB_IN_MODE] != 1;
    if (gathered && first_sample) { gather_slab(sample_off, 0); first_sample = false; }
    float ch_mean = 0.f, ch_m2 = 0.f;                      // Chan accumulators over (t, v), lane = channel
    float acc_g[V], acc_tc[V];
#pragma unroll
    for (int v = 0; v < V; ++v) { acc_g[v] = 0.f; acc_tc[v] = 0.f; }
    float mtc[2][NTL][4];                                  // tensor-core variant: time_compress.3 accumulators, per domain
#pragma unroll
    for (int L = 0; L < 2; ++L)
#pragma unroll
      for (int nt = 0; nt < NTL; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) mtc[L][nt][e] = 0.f;
    float mg[2][NTL][4];                                   // tensor-core variant: gate-conv accumulator fragments
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < NTL; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) mg[mt][nt][e] = 0.f;

#pragma unroll 1
    for (int t = 0; t < T; ++t) {
      // ---- load slab t (lanes = joints), global_norm folded (:375); block 0 builds the 10 features (:568-577)
      if (d[CB_IN_MODE] == 1) {
        if (lane < V) {
          float f[10];
          float sp = 0.f;
          const float* p = src + (t * V + lane) * 3;
#pragma unroll
          for (int k = 0; k < 3; ++k) {
            const float p0 = __ldg(p + k);
            float vel, acc;
            if (t < T - 1) {
              const float p1 = __ldg(p + V * 3 + k);
              vel = p1 - p0;
              const float veln = (t < T - 2) ? __ldg(p + 2 * V * 3 + k) - p1 : p1;   // vel[T-1] = x[T-1]
              acc = veln - vel;
            } else {
              vel = p0;        // vel[:, -1] = x[:, -1]
              acc = p0;        // acc[:, -1] = vel[:, -1]
            }
            f[k] = p0; f[3 + k] = acc; f[6 + k] = vel;
            sp = fmaf(vel, vel, sp);
          }
          f[9] = sqrtf(sp);
#pragma unroll
          for (int c = 0; c < 10; ++c) {
            const float val = fmaf(gs[c], f[c], gb[c]);
            xs[c * XS + lane] = val;
            ag[c * XT + lane] = val;
          }
        }
      } else {
        // the raw slab was gathered into xs by cp.async one stage ahead (below): every row load of the slab is in
        // flight at once and its latency hides behind the previous slab's collapse stage.  Normalise in place.
        cp_async_wait_all();
        __syncwarp();
        if (!ibf) {
          if (lane < V) {
            int c = 0;
#pragma unroll 2
            for (; c + 4 <= Ci; c += 4) {                        // scale / shift of four channels per 128-bit load
              const float4 s4 = *reinterpret_cast<const float4*>(gs + c);
              const float4 b4 = *reinterpret_cast<const float4*>(gb + c);
              const float sc4[4] = {s4.x, s4.y, s4.z, s4.w}, sh4[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const float val = fmaf(sc4[i], xs[(c + i) * XS + lane], sh4[i]);
                xs[(c + i) * XS + lane] = val;
                ag[(c + i) * XT + lane] = val;
              }
            }
            for (; c < Ci; ++c) {
              const float val = fmaf(gs[c], xs[c * XS + lane], gb[c]);
              xs[c * XS + lane] = val;
              ag[c * XT + lane] = val;
            }
          }
        } else {
          // expand the packed bf16 pairs in place, eight rows at a time: every lane reads before any lane writes
          const unsigned* xw = reinterpret_cast<const unsigned*>(xs);
          for (int c0 = 0; c0 < Ci; c0 += 8) {
            float val[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              const int c = rmin(c0 + k, Ci - 1);
              const unsigned w = lane < V ? xw[c * XS + (lane >> 1)] : 0u;
              val[k] = fmaf(gs[c], bits_f32((lane & 1) ? (w & 0xFFFF0000u) : (w << 16)), gb[c]);
            }
            __syncwarp();
            if (lane < V) {
#pragma unroll
              for (int k = 0; k < 8; ++k)
                if (c0 + k < Ci) { xs[(c0 + k) * XS + lane] = val[k]; ag[(c0 + k) * XT + lane] = val[k]; }
            }
          }
        }
      }
      // (the XS - V padding columns of a row are loaded by the LDS.128 reads below but never enter an FMA)
      __syncwarp();
      // ---- statistics of the slab (:360-371), lanes = channels; Bessel-corrected like torch.std
      {
        float mu = 0.f, q = 0.f;
        if (lane < Ci) {
          const float* xr = ag + lane * XT;
          float xv[V];
          float s = 0.f;
#pragma unroll
          for (int v = 0; v < V; ++v) { xv[v] = xr[v]; s += xv[v]; }
          mu = s / V;
#pragma unroll
          for (int v = 0; v < V; ++v) { const float dd = xv[v] - mu; q = fmaf(dd, dd, q); }
          // merge (n_b = V, mean mu, M2 q) into the running (n_a = t*V, ch_mean, ch_m2)
          const float na = (float)(t * V), nb = (float)V;
          const float delta = mu - ch_mean;
          ch_mean += delta * (nb / (na + nb));
          ch_m2 += q + delta * delta * (na * nb / (na + nb));
        }
        const float sd = lane < Ci ? sqrtf(q / (V - 1)) : 0.f;
        const float s1 = warp_sum(lane < Ci ? mu : 0.f);
        const float m2 = warp_sum(sd) / Ci;
        const float dd = lane < Ci ? sd - m2 : 0.f;
        const float q2 = warp_sum(dd * dd);
        if (lane == 0) { red[RL.stats + 1 + t] = s1 / Ci; red[RL.stats + 2 + T + t] = sqrtf(q2 / (Ci - 1)); }
      }
      __syncwarp();            // the transposed copy is dead: its region becomes the map buffer
      // ---- stacked 1x1 convolutions over the slab
      float acc_e[NE][V];
      float me[MTE][NTL][4];
      if constexpr (MMA) {
        // tensor cores: rows = output channels (16 per tile), columns = joints (8 per tile), k = input channels; the slab
        // rows are split into hi + lo once per k step and shared by the entry maps and the gate conv
#pragma unroll
        for (int mt = 0; mt < MTE; ++mt)
#pragma unroll
          for (int nt = 0; nt < NTL; ++nt)
#pragma unroll
            for (int e = 0; e < 4; ++e) me[mt][nt][e] = 0.f;
        const float* fg = wg0 + t * a.mtg * a.ks * 128;
#pragma unroll 1
        for (int ks = 0; ks < a.ks; ++ks) {
          const int k0 = 8 * ks + q, k1 = k0 + 4;
          const float* x0 = xs + (k0 < Ci ? k0 : 0) * XS + g;       // rows beyond Ci meet zero weights: any finite row
          const float* x1 = xs + (k1 < Ci ? k1 : 0) * XS + g;
          float bh[NTL][2], bl[NTL][2];
#pragma unroll
          for (int nt = 0; nt < NTL; ++nt) {                         // (columns beyond V: garbage in accumulator columns never stored)
            tf32_split(x0[8 * nt], bh[nt][0], bl[nt][0]);
            tf32_split(x1[8 * nt], bh[nt][1], bl[nt][1]);
          }
          if (interp) reduce_mma_rows<MTE, NTL>(me, wa0, a.mte, a.ks, ks, bh, bl);
          reduce_mma_rows<2, NTL>(mg, fg, a.mtg, a.ks, ks, bh, bl);
        }
      } else {
      // FP32 FMA: lanes = output channels, registers = joints
#pragma unroll
      for (int j = 0; j < NE; ++j)
#pragma unroll
        for (int v = 0; v < V; ++v) acc_e[j][v] = 0.f;
      {
        const float* we = wa0 + lane;
        const float* wgp = wg0 + t * mpg + lane;                    // row (c*T + t)
        const float* xr = xs;
#pragma unroll 2
        for (int c = 0; c < Ci; ++c) {
          float x[XS];
#pragma unroll
          for (int i = 0; i < V4; ++i) {
            const float4 q4 = *reinterpret_cast<const float4*>(xr + 4 * i);
            x[4 * i] = q4.x; x[4 * i + 1] = q4.y; x[4 * i + 2] = q4.z; x[4 * i + 3] = q4.w;
          }
          const float wgv = wgp[0];
          if (interp) {
#pragma unroll
            for (int j = 0; j < NE; ++j) {
              const float wv = we[32 * j];
#pragma unroll
              for (int v = 0; v < V; ++v) acc_e[j][v] = fmaf(wv, x[v], acc_e[j][v]);
            }
          }
#pragma unroll
          for (int v = 0; v < V; ++v) acc_g[v] = fmaf(wgv, x[v], acc_g[v]);
          we += mpe;
          wgp += T * mpg;
          xr += XS;
        }
      }
      }
      if (gathered) {
        __syncwarp();            // every lane is done reading the slab: gather the next one (or the next sample's first)
        const int bn = b + gridDim.x * a.nwarps;
        if (t + 1 < T) gather_slab(sample_off, t + 1);
        else if (bn < a.batch) gather_slab((size_t)bn * d[CB_IN_SB], 0);
      }
      if (interp) {
        // ---- BN + PReLU of the entry maps -> ag[m][v]  (:139-140, :147-148)
        if constexpr (MMA) {
#pragma unroll
          for (int mt = 0; mt < MTE; ++mt)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const int m = 16 * mt + g + 8 * h;
              if (m < 4 * Ch) {
                float* ar = ag + m * AS + 2 * q;
#pragma unroll
                for (int nt = 0; nt < NTL; ++nt) {
                  const float v0 = prelu(me[mt][nt][2 * h] + me_b[mt][h], me_a[mt][h]);
                  const float v1 = prelu(me[mt][nt][2 * h + 1] + me_b[mt][h], me_a[mt][h]);
                  if constexpr (V % 2 == 0) {
                    if (8 * nt + 2 * q < V) *reinterpret_cast<float2*>(ar + 8 * nt) = make_float2(v0, v1);
                  } else {
                    if (8 * nt + 2 * q < V) ar[8 * nt] = v0;
                    if (8 * nt + 2 * q + 1 < V) ar[8 * nt + 1] = v1;
                  }
                }
              }
            }
        } else {
#pragma unroll
          for (int j = 0; j < NE; ++j) {
            const int m = lane + 32 * j;
            if (m < 4 * Ch) {
              float* ar = ag + m * AS;
#pragma unroll
              for (int v = 0; v < V; ++v) ar[v] = prelu(acc_e[j][v] + e_b[j], e_a[j]);
            }
          }
        }
        __syncwarp();
        // ---- collapsing convolutions (:141-142, :149-150)
        if constexpr (MMA) {
          // time_compress.3 on the tensor cores: per domain rows = outputs (Ch <= 16: one tile), k = the Ch map rows,
          // columns = joints; both domains share the MMA stream so that one accumulator is revisited 2 * NTL MMAs later
          const int ksc = (Ch + 7) / 8;
          const float* ft = wtc + t * 2 * ksc * 128;
#pragma unroll 1
          for (int ks = 0; ks < ksc; ++ks) {
            const int k0 = 8 * ks + q, k1 = k0 + 4;
            float ah[2][4], al[2][4], bh[2][NTL][2], bl[2][NTL][2];
#pragma unroll
            for (int L = 0; L < 2; ++L) {
              const float4 w4 = *reinterpret_cast<const float4*>(ft + ((L * ksc + ks) * 32 + lane) * 4);
              tf32_split(w4.x, ah[L][0], al[L][0]); tf32_split(w4.y, ah[L][1], al[L][1]);
              tf32_split(w4.z, ah[L][2], al[L][2]); tf32_split(w4.w, ah[L][3], al[L][3]);
              const float* r0 = ag + (2 * L * Ch + (k0 < Ch ? k0 : 0)) * AS + g;    // rows beyond Ch meet zero weights
              const float* r1 = ag + (2 * L * Ch + (k1 < Ch ? k1 : 0)) * AS + g;
#pragma unroll
              for (int nt = 0; nt < NTL; ++nt) {
                tf32_split(r0[8 * nt], bh[L][nt][0], bl[L][nt][0]);
                tf32_split(r1[8 * nt], bh[L][nt][1], bl[L][nt][1]);
              }
            }
#pragma unroll
            for (int term = 0; term < 3; ++term)
#pragma unroll
              for (int L = 0; L < 2; ++L)
#pragma unroll
                for (int nt = 0; nt < NTL; ++nt) {
                  if (term == 0) mma_tf32(mtc[L][nt], al[L], bh[L][nt]);
                  else if (term == 1) mma_tf32(mtc[L][nt], ah[L], bl[L][nt]);
                  else mma_tf32(mtc[L][nt], ah[L], bh[L][nt]);
                }
          }
        }
        {                                                           // lanes = outputs (domain L3, channel o)
          const float* wt = wtc + t * mpc + lane;                   // row (c'*T + t)
          const float* wj = wjc + lane;                             // row (c'*V + v)
          float jsum = 0.f;
#pragma unroll 2
          for (int cp_ = 0; cp_ < Ch; ++cp_) {
            float xa[XS], xg[XS];
#pragma unroll
            for (int i = 0; i < V4; ++i) {
              if constexpr (!MMA) {
                const float4 q4 = *reinterpret_cast<const float4*>(arow_tc + cp_ * AS + 4 * i);
                xa[4 * i] = q4.x; xa[4 * i + 1] = q4.y; xa[4 * i + 2] = q4.z; xa[4 * i + 3] = q4.w;
              }
              const float4 g4 = *reinterpret_cast<const float4*>(arow_jc + cp_ * AS + 4 * i);
              xg[4 * i] = g4.x; xg[4 * i + 1] = g4.y; xg[4 * i + 2] = g4.z; xg[4 * i + 3] = g4.w;
            }
            if constexpr (!MMA) {
              const float wtv = wt[cp_ * T * mpc];
#pragma unroll
              for (int v = 0; v < V; ++v) acc_tc[v] = fmaf(wtv, xa[v], acc_tc[v]);
            }
            if constexpr (MMA) {
              const float* wjr = wjc + ((size_t)cp_ * V4 * mpc + lane) * 4;
              float j0 = 0.f, j1 = 0.f, j2 = 0.f, j3 = 0.f;
#pragma unroll
              for (int i = 0; i < V4; ++i) {
                const float4 w4 = *reinterpret_cast<const float4*>(wjr + (size_t)i * mpc * 4);
                j0 = fmaf(w4.x, xg[4 * i], j0); j1 = fmaf(w4.y, xg[4 * i + 1], j1);
                j2 = fmaf(w4.z, xg[4 * i + 2], j2); j3 = fmaf(w4.w, xg[4 * i + 3], j3);
              }
              jsum += (j0 + j1) + (j2 + j3);
            } else {
            const float* wjr = wj + cp_ * V * mpc;
            float j0 = 0.f, j1 = 0.f;
#pragma unroll
            for (int v = 0; v + 1 < V; v += 2) {
              j0 = fmaf(wjr[v * mpc], xg[v], j0);
              j1 = fmaf(wjr[(v + 1) * mpc], xg[v + 1], j1);
            }
            if (V & 1) j0 = fmaf(wjr[(V - 1) * mpc], xg[V - 1], j0);
            jsum += j0 + j1;
            }
          }
          if (lane < 2 * Ch) red[RL.jc + lane * T + t] = jsum + smem[a.o_jc3_b + lane];
        }
      }
      __syncwarp();              // slab and map rows are read: the next slab may overwrite them
    }

    // ---------------- per-sample results
    {
      // channel-level statistics: mean over channels of the channel means, std over channels of the channel stds
      const float cm = lane < Ci ? ch_mean : 0.f;
      const float sd = lane < Ci ? sqrtf(ch_m2 / (TV - 1)) : 0.f;
      const float s1 = warp_sum(cm);
      const float m2 = warp_sum(sd) / Ci;
      const float dd = lane < Ci ? sd - m2 : 0.f;
      const float q2 = warp_sum(dd * dd);
      if (lane == 0) { red[RL.stats] = s1 / Ci; red[RL.stats + 1 + T] = sqrtf(q2 / (Ci - 1)); }
    }
    // gate conv (T,1) + BN + PReLU -> h1 (:323-326); staged through shared memory for coalesced stores
    if constexpr (MMA) {
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int m = 16 * mt + g + 8 * h;
          if (m < 2 * Cg) {
            const float bb = smem[a.o_g0_b + m], sl = smem[a.o_g0_a + m / Cg];
            float* ar = ag + m * AS + 2 * q;
#pragma unroll
            for (int nt = 0; nt < NTL; ++nt) {
              if (8 * nt + 2 * q < V) ar[8 * nt] = prelu(mg[mt][nt][2 * h] + bb, sl);
              if (8 * nt + 2 * q + 1 < V) ar[8 * nt + 1] = prelu(mg[mt][nt][2 * h + 1] + bb, sl);
            }
          }
        }
    } else if (lane < 2 * Cg) {
      const float bb = smem[a.o_g0_b + lane], sl = smem[a.o_g0_a + lane / Cg];
      float* ar = ag + lane * AS;
#pragma unroll
      for (int v = 0; v < V; ++v) ar[v] = prelu(acc_g[v] + bb, sl);
    }
    __syncwarp();
    for (int i = lane; i < 2 * RL.h1g; i += 32) {
      const int g = i / RL.h1g, r = i - g * RL.h1g;
      red[RL.h1 + i] = r < Cg * V ? ag[(g * Cg + r / V) * AS + (r % V)] : 0.f;
    }
    __syncwarp();
    if (interp) {
      if constexpr (MMA) {
#pragma unroll
        for (int L = 0; L < 2; ++L)
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int o = g + 8 * h;
            if (o < Ch) {
              const float bb = smem[a.o_tc3_b + L * Ch + o];
              float* ar = ag + (L * Ch + o) * AS + 2 * q;
#pragma unroll
              for (int nt = 0; nt < NTL; ++nt) {
                if (8 * nt + 2 * q < V) ar[8 * nt] = mtc[L][nt][2 * h] + bb;
                if (8 * nt + 2 * q + 1 < V) ar[8 * nt + 1] = mtc[L][nt][2 * h + 1] + bb;
              }
            }
          }
      } else if (lane < 2 * Ch) {
        const float bb = smem[a.o_tc3_b + lane];
        float* ar = ag + lane * AS;
#pragma unroll
        for (int v = 0; v < V; ++v) ar[v] = acc_tc[v] + bb;
      }
      __syncwarp();
      for (int i = lane; i < 2 * Ch * V; i += 32) red[RL.tc + i] = ag[(i / V) * AS + (i % V)];
      __syncwarp();
    }
  }
}

template <int T, int V, int NE>
int launch_reduce_impl(const ReduceArgs& a, void* stream) {
  if constexpr (T == 10) {
    if (a.mma) return launch_warp_per_sample(dstd_reduce_kernel<T, V, NE, true>, a, stream);
  }
  return launch_warp_per_sample(dstd_reduce_kernel<T, V, NE, false>, a, stream);
}

}  // namespace cg
