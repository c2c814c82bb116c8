// DSTD-GC block, stage 3 of 3: the TILE path -- adjacency products, channel mixes, gating, compressor, squeeze-excitation
// and the block residual (reference: models/CISTGCN/CISTGCN.py:110, 117, 123 ConvTemporalGraphical; :229-247, 259-269
// Domain_GCNN_layer; :305-318, 386-390 DSTD_GC; models/layers/SE.py:24-41), with the gates and the sample-specific
// adjacencies read from stage 2 (dstd_adj.cuh).
//
// One CTA per sample at a time, but -- unlike round 1's fused kernel -- the working set is TWO tiles, not three plus the
// adjacency scratch of both domains, so an E = 32 block fits two 256-thread CTAs per SM (the barrier and latency stalls
// of one sample hide behind the other):
//   * the two domains run one after the other through the SAME work tile;
//   * the compressor's 1x1 over cat(u1, u2) (:305) is accumulated in registers, domain by domain (K = Co each), so the
//     concatenated 2*Co-channel map never exists;
//   * only one adjacency is resident at a time; the second is copied in (cp.async) behind the first domain's channel mix.
// Every weight matrix of the stage is resident in shared memory for the whole launch.
#pragma once
#include "../../include/cistgcn_b200.h"
#include "dstd_block.cuh"
#include "host_util.h"
#include "simt.h"

namespace cg {

struct MixArgs {
  int d[CB_COUNT];
  int res[CB_COUNT];       // shared-memory float offset of the resident copy of weight field f (all fields used here)
  int wsz[CB_COUNT];
  const float* w;
  const float* in;
  float* out;
  const float* wg;         // (B, 2, Co) gates from stage 2
  const float* adj_s;      // (B, V, T, T) from stage 2 (ignored when the block carries static adjacencies)
  const float* adj_t;      // (B, T, V, V)
  int in_bf16, out_bf16;   // activation tensors stored as bf16 (cistgcn_forward_bf16); strides stay in elements
  int batch;
  int o_xn, o_a, o_adj, o_sm, smem_floats;
  int nwarps, o_warp, warp_floats;      // warp-per-sample variant (dstd_mix_narrow.cuh)
};

// Host: shared-memory plan for `nt` threads.  All matrices must be resident.
inline bool mix_plan(MixArgs& a, int nt, int max_smem_floats) {
  const int* d = a.d;
  const int Ci = d[CB_CI], Co = d[CB_CO], T = d[CB_T], V = d[CB_V], Hs = d[CB_HS];
  const bool has_res = d[CB_HAS_RES] != 0;
  const int TV = T * V, cmax = imax(Ci, Co), Cop = pad8i(Co);
  for (int f = 0; f < CB_COUNT; ++f) { a.wsz[f] = 0; a.res[f] = -1; }
  int* z = a.wsz;
  z[CB_GN_S] = z[CB_GN_B] = Ci;
  for (int L = 0; L < 2; ++L) {
    z[CB_TCN_WT_S + L] = Ci * (has_res ? 2 : 1) * Cop; z[CB_TCN_B_S + L] = Co; z[CB_TCN_A_S + L] = 1;
    z[CB_P_S_S + L] = Co; z[CB_P_B_S + L] = Co; z[CB_P_A_S + L] = 1;
  }
  z[CB_CP_WT] = 2 * Co * Cop; z[CB_CP_B] = Co; z[CB_CP_A] = 1;
  z[CB_SE1_WT] = Co * pad8i(Hs); z[CB_SE2_WT] = Hs * Cop;
  if (has_res) { z[CB_RS_WT] = Ci * Cop; z[CB_RS_B] = Co; }
  for (int f = 0; f < CB_COUNT; ++f) z[f] = pad4i(z[f]);
  a.o_xn = 0;
  a.o_a = pad4i(Ci * TV);
  a.o_adj = a.o_a + pad4i(cmax * TV);
  const int adj = imax(pad4i(T * T * (V | 1)), T * pad4i(V * V));
  a.o_sm = a.o_adj + adj;
  int cur = a.o_sm + pad4i(2 * Co) + 2 * pad4i(Co) + pad4i(Hs) + 2 * (nt / 32) * 8;
  for (int f = 0; f < CB_COUNT; ++f)
    if (z[f]) { a.res[f] = cur; cur += z[f]; }
  a.smem_floats = cur;
  return cur <= max_smem_floats;
}

// Work-unit mapping of the register-accumulated compressor: unit (pass, warp) -> TM output rows x 32 lanes x TN columns.
template <int TM, int TN, int N, int NT>
struct AccMap {
  static constexpr int NW = NT / 32, NCOLS = N / TN, NG = (NCOLS + 31) / 32;
  CG_DEV static bool locate(int pass, int M, int& m0, int& n0) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int mtiles = (M + TM - 1) / TM;
    const int item = pass * NW + warp;
    const int slot = (item / mtiles) * 32 + lane;
    const bool active = item < mtiles * NG && slot < NCOLS;
    m0 = active ? (item % mtiles) * TM : 0;
    n0 = active ? slot * TN : 0;
    return active;
  }
  static bool fits(int M, int npass) { return ((M + TM - 1) / TM) * NG <= npass * NW; }
};

template <int TM, int TN, int LD, int N, int NT, int NPASS>
CG_DEV void gemm_accumulate(float (&acc)[NPASS][TM][TN], const float* ws, int Mp, int M, int K, const float* X) {
#pragma unroll
  for (int pass = 0; pass < NPASS; ++pass) {
    int m0, n0;
    if (!AccMap<TM, TN, N, NT>::locate(pass, M, m0, n0)) continue;
    const float* wp = ws + m0;
    const float* xp = X + n0;
#pragma unroll 4
    for (int k = 0; k < K; ++k) {
      float w[TM], x[TN];
      lds_vec<TM>(wp, w);
      lds_vec<TN>(xp, x);
      wp += Mp;
      xp += LD;
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[pass][i][j] = fmaf(w[i], x[j], acc[pass][i][j]);
    }
  }
}

// TM = output rows per thread of the compressor accumulation: 8 (one pass) for wide blocks, 4 (up to two passes) else.
template <int T, int V, int NT, int TM>
__global__ void __launch_bounds__(NT, NT <= 256 ? 2 : 1) dstd_mix_kernel(const MixArgs a) {
  CG_DYN_SMEM(smem);
  constexpr int TV = T * V, TT = T * T, VV = V * V, VP = V | 1;
  constexpr int NW = NT / 32;
  constexpr int TNW = (TV % 4 == 0) ? 4 : 2;
  constexpr int VVP = (VV + 3) & ~3;
  constexpr int NPASS = TM == 8 ? 1 : 2;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int* d = a.d;
  const float* __restrict__ W = a.w;
  const int Ci = d[CB_CI], Co = d[CB_CO], Hs = d[CB_HS];
  const bool has_res = d[CB_HAS_RES] != 0, interp = d[CB_INTERP] != 0;
  const int Cop = pad8i(Co);

  float* XN = smem + a.o_xn;
  float* A = smem + a.o_a;
  float* ADJ = smem + a.o_adj;
  float* p = smem + a.o_sm;
  float* wg = p;      p += pad4i(2 * Co);
  float* semean = p;  p += pad4i(Co);
  float* gate = p;    p += pad4i(Co);
  float* hid = p;     p += pad4i(Hs);
  float* separt = p;                                   // [NPASS * NW][TM] squeeze partial sums
  auto P = [&](int f) -> const float* { return smem + a.res[f]; };

  for (int f = 0; f < CB_COUNT; ++f)
    if (a.res[f] >= 0) copy_async<NT>(smem + a.res[f], W + d[f], a.wsz[f]);
  cp_async_commit();
  cp_async_wait_all();
  __syncthreads();

  const float* gs = P(CB_GN_S);
  const float* gb = P(CB_GN_B);
  const float* tb0 = P(CB_TCN_B_S); const float* tb1 = P(CB_TCN_B_T);
  const float* ps0 = P(CB_P_S_S);   const float* ps1 = P(CB_P_S_T);
  const float* pb0 = P(CB_P_B_S);   const float* pb1 = P(CB_P_B_T);
  const float ta0 = P(CB_TCN_A_S)[0], ta1 = P(CB_TCN_A_T)[0], pa0 = P(CB_P_A_S)[0], pa1 = P(CB_P_A_T)[0];
  const float* cb = P(CB_CP_B);
  const float ca = P(CB_CP_A)[0];
  const int K2 = has_res ? Ci : 0;

  for (int b = blockIdx.x; b < a.batch; b += gridDim.x) {
    // ---------------- load + global_norm (:375); block 0 builds the 10 features (:568-577); gates; Adj_s
    if (tid < 2 * Co) wg[tid] = __ldg(a.wg + (size_t)b * 2 * Co + tid);
    {
      const float* as = interp ? a.adj_s + (size_t)b * V * TT : W + d[CB_ADJ_S];     // (V,T,T) -> [t][q][v], odd row stride
      for (int i = tid; i < V * TT; i += NT) { const int v = i / TT, r = i - v * TT; ADJ[r * VP + v] = __ldg(as + i); }
    }
    if (d[CB_IN_MODE] == 1) {
      const float* src = a.in + (size_t)b * d[CB_IN_SB];
      float* raw = A;
      for (int i = tid; i < TV * 3; i += NT) raw[i] = __ldg(src + i);
      __syncthreads();
      for (int n = tid; n < TV; n += NT) {
        const int t = n / V;
        float f[10];
        float sp = 0.f;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const float p0 = raw[n * 3 + k];
          float vel, acc;
          if (t < T - 1) {
            const float p1 = raw[(n + V) * 3 + k];
            vel = p1 - p0;
            const float veln = (t < T - 2) ? raw[(n + 2 * V) * 3 + k] - p1 : p1;   // vel[T-1] = x[T-1]
            acc = veln - vel;
          } else {
            vel = p0;      // vel[:, -1] = x[:, -1]
            acc = p0;      // acc[:, -1] = vel[:, -1]
          }
          f[k] = p0; f[3 + k] = acc; f[6 + k] = vel;
          sp = fmaf(vel, vel, sp);
        }
        f[9] = sqrtf(sp);
#pragma unroll
        for (int c = 0; c < 10; ++c) XN[c * TV + n] = fmaf(gs[c], f[c], gb[c]);
      }
    } else {
      const bool ibf = a.in_bf16 != 0;
      const size_t sbase_ = (size_t)b * d[CB_IN_SB];
      const int sc = d[CB_IN_SC], st = d[CB_IN_ST], sv = d[CB_IN_SV];
      if (sv == 1 && st == V && sc == TV && (TV % 4) == 0 && (d[CB_IN_SB] % 4) == 0) {       // contiguous tile: 128-bit (64-bit bf16) loads
        for (int i = tid; i < Ci * TV / 4; i += NT) {
          const int c = (i * 4) / TV;
          float4 v4 = ld_act4(a.in, sbase_ + (size_t)i * 4, ibf);
          const float g0 = gs[c], b0 = gb[c];
          v4.x = fmaf(g0, v4.x, b0); v4.y = fmaf(g0, v4.y, b0); v4.z = fmaf(g0, v4.z, b0); v4.w = fmaf(g0, v4.w, b0);
          reinterpret_cast<float4*>(XN)[i] = v4;
        }
      } else {
        for (int i = tid; i < Ci * TV; i += NT) {
          const int c = i / TV, n = i - c * TV, t = n / V, v = n - t * V;
          XN[i] = fmaf(gs[c], ld_act(a.in, sbase_ + (size_t)c * sc + t * st + v * sv, ibf), gb[c]);
        }
      }
    }
    __syncthreads();

    float cacc[NPASS][TM][TNW];
#pragma unroll
    for (int q = 0; q < NPASS; ++q)
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TNW; ++j) cacc[q][i][j] = 0.f;

#pragma unroll 1
    for (int L = 0; L < 2; ++L) {
      // ---------------- g = XN x Adj  (:110, :117, :123) -> A
      if (L == 0) {
        if (Ci >= 4 && ((Ci + 3) / 4) * V >= NT) gcn_space<T, V, 4, NT>(XN, ADJ, A, Ci);
        else if (Ci >= 2) gcn_space<T, V, 2, NT>(XN, ADJ, A, Ci);
        else gcn_space<T, V, 1, NT>(XN, ADJ, A, Ci);
      } else {
        if (Ci >= 4 && ((Ci + 3) / 4) * T * 2 >= NT) gcn_time<T, V, 4, NT>(XN, ADJ, A, Ci);
        else if (Ci >= 2) gcn_time<T, V, 2, NT>(XN, ADJ, A, Ci);
        else gcn_time<T, V, 1, NT>(XN, ADJ, A, Ci);
      }
      __syncthreads();
      if (L == 0) {
        // Adj_s is dead: bring Adj_t in behind the channel mix ((T,V,V) rows padded to a float4)
        const float* at = interp ? a.adj_t + (size_t)b * T * VV : W + d[CB_ADJ_T];
        if constexpr (VV % 4 == 0) {
          for (int i = tid * 4; i < T * VV; i += NT * 4) cp_async16(ADJ + i, at + i);
          cp_async_commit();
        } else {
          for (int i = tid; i < T * VV; i += NT) ADJ[(i / VV) * VVP + i % VV] = __ldg(at + i);
          constexpr int PADC = VVP - VV;
          for (int i = tid; i < T * PADC; i += NT) ADJ[(i / PADC) * VVP + VV + i % PADC] = 0.f;
        }
      }
      // ---------------- x_L = PReLU(BN(W g + b) + res); u_L = PReLU(BN(w_L * x_L)), in place  (:266-268, :388)
      {
        const float* tb = L ? tb1 : tb0;
        const float* ps = L ? ps1 : ps0;
        const float* pb = L ? pb1 : pb0;
        const float ta = L ? ta1 : ta0, pa = L ? pa1 : pa0;
        const float* wgl = wg + L * Co;
        const WideOp ops[1] = {{nullptr, P(CB_TCN_WT_S + L), A, XN}};
        gemm_wide_auto<TNW, TV, TV, NT, true, 1>(ops, Cop, Co, Ci, K2, nullptr, 0,
          [&](int, int m, int n0, float (&v)[TNW]) {
            const float tbm = tb[m], sc = ps[m] * wgl[m], pbm = pb[m];
            float r[TNW];
            if (!has_res) lds_vec<TNW>(XN + m * TV + n0, r);
#pragma unroll
            for (int j = 0; j < TNW; ++j) {
              float x = v[j] + tbm;
              if (!has_res) x += r[j];
              x = prelu(x, ta);
              v[j] = prelu(fmaf(sc, x, pbm), pa);
            }
            store_vec<TNW>(A + m * TV + n0, v);
          });
      }
      // ---------------- compressor, this domain's half of the K range, into registers  (:305)
      gemm_accumulate<TM, TNW, TV, TV, NT, NPASS>(cacc, P(CB_CP_WT) + L * Co * Cop, Cop, Co, Co, A);
      if (L == 0) cp_async_wait_all();
      __syncthreads();            // everyone is done reading u_L (and Adj_t has landed)
    }
    // ---------------- c = PReLU(BN(.)) -> A, with the squeeze sums on the way  (:306-307, SE.py:39)
    // (per-(pass, warp, row) partial sums, added up in a fixed order below: bit-reproducible, no atomics)
#pragma unroll
    for (int q = 0; q < NPASS; ++q) {
      int m0, n0;
      const bool act = AccMap<TM, TNW, TV, NT>::locate(q, Co, m0, n0);
#pragma unroll
      for (int i = 0; i < TM; ++i) {
        float rs = 0.f;
        if (act && m0 + i < Co) {
          const float bias = cb[m0 + i];
          float v[TNW];
#pragma unroll
          for (int j = 0; j < TNW; ++j) { v[j] = prelu(cacc[q][i][j] + bias, ca); rs += v[j]; }
          store_vec<TNW>(A + (m0 + i) * TV + n0, v);
        }
        rs = warp_sum(rs);
        if (lane == 0) separt[((q * NW + warp) * TM) + i] = rs;
      }
    }
    __syncthreads();
    if (tid < Co) {
      const int mtiles = (Co + TM - 1) / TM, mt = tid / TM, i = tid - mt * TM;
      float s = 0.f;
      for (int item = mt; item < NPASS * NW; item += mtiles) s += separt[item * TM + i];   // units of this row tile
      semean[tid] = s * (1.f / TV);
    }
    __syncthreads();
    // ---------------- squeeze-excitation (SE.py:37-41)
    for (int h = warp; h < Hs; h += NW) {
      const float* wt = P(CB_SE1_WT) + h;
      float acc = 0.f;
      for (int c = lane; c < Co; c += 32) acc = fmaf(wt[c * pad8i(Hs)], semean[c], acc);
      acc = warp_sum(acc);
      if (lane == 0) hid[h] = fmaxf(acc, 0.f);
    }
    __syncthreads();
    for (int o = tid; o < Co; o += NT) {
      const float* wt = P(CB_SE2_WT) + o;
      float acc = 0.f;
      for (int h = 0; h < Hs; ++h) acc = fmaf(wt[h * Cop], hid[h], acc);
      gate[o] = sigmoidf(acc);
    }
    __syncthreads();
    // ---------------- out = c * gate + residual(xn)   (:390)
    {
      const bool obf = a.out_bf16 != 0;
      const size_t obase = (size_t)b * d[CB_OUT_SB];
      const int sc = d[CB_OUT_SC], st = d[CB_OUT_ST], sv = d[CB_OUT_SV];
      const bool contiguous = sv == 1 && st == V && sc == TV && (TV % 4) == 0 && (d[CB_OUT_SB] % 4) == 0;
      if (has_res) {
        const float* rbias = P(CB_RS_B);
        const WideOp ops[1] = {{nullptr, P(CB_RS_WT), XN, nullptr}};
        gemm_wide_auto<TNW, TV, TV, NT, false, 1>(ops, Cop, Co, Ci, 0, nullptr, 0,
          [&](int, int m, int n0, float (&v)[TNW]) {
            const float gm = gate[m], bias = rbias[m];
            float c[TNW];
            lds_vec<TNW>(A + m * TV + n0, c);
#pragma unroll
            for (int j = 0; j < TNW; ++j) v[j] = fmaf(c[j], gm, v[j] + bias);
            if (contiguous) {
              if constexpr (TNW == 4) st_act4(a.out, obase + (size_t)m * TV + n0, make_float4(v[0], v[1], v[2], v[3]), obf);
              else { st_act(a.out, obase + (size_t)m * TV + n0, v[0], obf); st_act(a.out, obase + (size_t)m * TV + n0 + 1, v[1], obf); }
            } else {
              int t = n0 / V, vv = n0 - t * V;
#pragma unroll
              for (int j = 0; j < TNW; ++j) {
                st_act(a.out, obase + (size_t)m * sc + t * st + vv * sv, v[j], obf);
                if (++vv == V) { vv = 0; ++t; }
              }
            }
          });
      } else if (contiguous) {
        for (int i = tid; i < Co * TV / 4; i += NT) {
          const float gm = gate[(i * 4) / TV];
          const float4 c4 = reinterpret_cast<const float4*>(A)[i];
          const float4 x4 = reinterpret_cast<const float4*>(XN)[i];
          st_act4(a.out, obase + (size_t)i * 4,
                  make_float4(fmaf(c4.x, gm, x4.x), fmaf(c4.y, gm, x4.y), fmaf(c4.z, gm, x4.z), fmaf(c4.w, gm, x4.w)), obf);
        }
      } else {
        for (int i = tid; i < Co * TV; i += NT) {
          const int m = i / TV, n = i - m * TV, t = n / V, v = n - t * V;
          st_act(a.out, obase + (size_t)m * sc + t * st + v * sv, fmaf(A[i], gate[m], XN[i]), obf);
        }
      }
    }
    __syncthreads();
  }
}

template <int T, int V, int NT, int TM>
int launch_mix_impl(const MixArgs& a, void* stream) {
  auto kfn = dstd_mix_kernel<T, V, NT, TM>;
  const size_t smem = (size_t)a.smem_floats * sizeof(float);
  int err = 0;
  const int per_sm = prepared_blocks_per_sm(kfn, NT, smem, &err);
  if (err) return err;
  const int grid = grid_for(a.batch, per_sm);
  CG_LAUNCH(kfn, grid, NT, smem, stream, a);
  return last_launch_error();
}

}  // namespace cg
