// DSTD-GC block, stage 3 of 3, NARROW variant: blocks with Ci = Co = C <= 4 channels and an identity block residual --
// the output block st_gcnns_o (3 -> 3 on the (xyz, joints, frames) view; models/CISTGCN/CISTGCN.py:110-123, 229-269,
// 305-318, 386-390, models/layers/SE.py:24-41).
//
// At 3 channels the stage is not arithmetic at all: a sample carries 2 x 3 x T x V x (T + V) = 0.16 M MACs against
// V*T*T + T*V*V = 25 850 adjacency values (103 KB) that are each used exactly C times.  The tile kernel (dstd_mix.cuh)
// staged both adjacencies through shared memory behind block barriers with two samples in flight per SM and ran at
// 1.0 TB/s; here ONE WARP owns one sample, the adjacencies stream from global memory straight into registers (each
// (T x T) / (V x V) slice is one contiguous run, a row per load instruction, the next slice's rows in flight while the
// current slice is consumed) and 12-16 samples are in flight per SM with no block barrier:
//   space domain  lane = q:  g[c] = sum_t xn[c][t][v] * A_s[v][t][q]   for one joint-axis index v at a time
//   time domain   lane = w:  g[c] = sum_v xn[c][t][v] * A_t[t][v][w]   for one frame-axis index t at a time
// and the lane that holds position (q, v) / (t, w) runs the whole per-position epilogue on its C values in registers:
// tcn 1x1 + BN + identity residual + PReLU, gate * (.) + BN + PReLU, this domain's half of the compressor.  The
// compressor sums of the space domain wait in shared memory for the time domain; squeeze-excitation and the block
// residual finish the sample.  Per warp: the normalised tile and the compressor tile, 2 x C x T x V floats.
#pragma once
#include "../../include/cistgcn_b200.h"
#include "dstd_mix.cuh"
#include "host_util.h"
#include "simt.h"

namespace cg {

#ifdef CISTGCN_EMU
constexpr int MIXN_MAX_WARPS = 4;           // emulator: one OS thread per CUDA thread -- keep the CTAs small
#else
constexpr int MIXN_MAX_WARPS = 16;          // 512 threads: up to 128 registers per thread
#endif

// Host: plan of the narrow variant (extends MixArgs: nwarps / o_warp / warp_floats).  False when the block is not narrow.
template <int C>
inline bool mix_narrow_plan(MixArgs& a, int max_smem_floats) {
  const int* d = a.d;
  const int Ci = d[CB_CI], Co = d[CB_CO], T = d[CB_T], V = d[CB_V], Hs = d[CB_HS];
  if (Ci != C || Co != C || d[CB_HAS_RES] != 0 || d[CB_IN_MODE] == 1 || T > 32 || V > 32 || Hs > 32) return false;
  const int TV = T * V, Cop = pad8i(Co);
  for (int f = 0; f < CB_COUNT; ++f) { a.wsz[f] = 0; a.res[f] = -1; }
  int* z = a.wsz;
  z[CB_GN_S] = z[CB_GN_B] = Ci;
  for (int L = 0; L < 2; ++L) {
    z[CB_TCN_WT_S + L] = Ci * Cop; z[CB_TCN_B_S + L] = Co; z[CB_TCN_A_S + L] = 1;
    z[CB_P_S_S + L] = Co; z[CB_P_B_S + L] = Co; z[CB_P_A_S + L] = 1;
  }
  z[CB_CP_WT] = 2 * Co * Cop; z[CB_CP_B] = Co; z[CB_CP_A] = 1;
  z[CB_SE1_WT] = Co * pad8i(Hs); z[CB_SE2_WT] = Hs * Cop;
  int cur = 0;
  for (int f = 0; f < CB_COUNT; ++f)
    if (z[f]) { z[f] = pad4i(z[f]); a.res[f] = cur; cur += z[f]; }
  a.o_warp = cur;
  a.warp_floats = 2 * pad4i(C * TV) + 8;
  int nw = (max_smem_floats - cur) / a.warp_floats;
  if (nw > MIXN_MAX_WARPS) nw = MIXN_MAX_WARPS;
  if (nw < 4) return false;
  a.nwarps = nw;
  a.smem_floats = cur + nw * a.warp_floats;
  return true;
}

template <int T, int V, int C>
__global__ void __launch_bounds__(32 * MIXN_MAX_WARPS, 1) dstd_mix_narrow_kernel(const MixArgs a) {
  CG_DYN_SMEM(smem);
  constexpr int TV = T * V, TT = T * T, VV = V * V, Cop = 8;
  constexpr int PF_AHEAD = 4;              // slices between the L2 prefetch and the register loads (one slice ahead of use)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nthreads = blockDim.x;
  const int* d = a.d;
  const float* __restrict__ W = a.w;
  const int Hs = d[CB_HS];
  const bool interp = d[CB_INTERP] != 0;

  for (int f = 0; f < CB_COUNT; ++f)
    if (a.res[f] >= 0)
      for (int i = threadIdx.x; i < a.wsz[f]; i += nthreads) smem[a.res[f] + i] = __ldg(W + d[f] + i);
  __syncthreads();
  auto P = [&](int f) -> const float* { return smem + a.res[f]; };
  const float* gs = P(CB_GN_S);
  const float* gb = P(CB_GN_B);
  const float* cpw = P(CB_CP_WT);
  const float* cb = P(CB_CP_B);
  const float ca = P(CB_CP_A)[0];

  float* XN = smem + a.o_warp + warp * a.warp_floats;      // [C][T*V] normalised input
  float* CA = XN + pad4i(C * TV);                          // [C][T*V] compressor sums, then c
  float* sv = CA + pad4i(C * TV);                          // [8] squeeze means / gates

  const bool ibf = a.in_bf16 != 0, obf = a.out_bf16 != 0;
  const int isc = d[CB_IN_SC], ist = d[CB_IN_ST], isv = d[CB_IN_SV];
  const int osc = d[CB_OUT_SC], ost = d[CB_OUT_ST], osv = d[CB_OUT_SV];
  // channel-fastest views ((B, frames, joints, xyz) tensors seen as (xyz, joints, frames)): walk memory in its own order
  const bool in_cfast = isc == 1 && ist == C && isv == C * T;
  const bool out_cfast = osc == 1 && ost == C && osv == C * T;

  // Per-position epilogue of domain L on the lane's C adjacency-product values g at position n (:266-268, :388), then
  // this domain's half of the compressor (:305): returns the C partial sums.
  auto domain_epilogue = [&](int L, const float (&g)[C], int n, const float* wgl, float (&cacc)[C]) {
    const float* wt = P(CB_TCN_WT_S + L);
    const float* tb = P(CB_TCN_B_S + L);
    const float* ps = P(CB_P_S_S + L);
    const float* pb = P(CB_P_B_S + L);
    const float ta = P(CB_TCN_A_S + L)[0], pa = P(CB_P_A_S + L)[0];
    float u[C];
#pragma unroll
    for (int m = 0; m < C; ++m) {
      float x = tb[m];
#pragma unroll
      for (int k = 0; k < C; ++k) x = fmaf(wt[k * Cop + m], g[k], x);
      x = prelu(x + XN[m * TV + n], ta);
      u[m] = prelu(fmaf(ps[m] * wgl[m], x, pb[m]), pa);
    }
#pragma unroll
    for (int mo = 0; mo < C; ++mo) {
      float s = 0.f;
#pragma unroll
      for (int m = 0; m < C; ++m) s = fmaf(cpw[(L * C + m) * Cop + mo], u[m], s);
      cacc[mo] = s;
    }
  };

  for (int b = blockIdx.x * a.nwarps + warp; warp < a.nwarps && b < a.batch; b += gridDim.x * a.nwarps) {
    // ---------------- load + global_norm (:375)
    {
      const size_t sbase_ = (size_t)b * d[CB_IN_SB];
      if (in_cfast) {
        for (int j = lane; j < C * TV; j += 32) {
          const int c = j % C, r = j / C, t = r % T, v = r / T;
          XN[c * TV + t * V + v] = fmaf(gs[c], ld_act(a.in, sbase_ + j, ibf), gb[c]);
        }
      } else {
        for (int i = lane; i < C * TV; i += 32) {
          const int c = i / TV, n = i - c * TV, t = n / V, v = n - t * V;
          XN[i] = fmaf(gs[c], ld_act(a.in, sbase_ + (size_t)c * isc + t * ist + v * isv, ibf), gb[c]);
        }
      }
    }
    float wgl[2][C];
#pragma unroll
    for (int L = 0; L < 2; ++L)
#pragma unroll
      for (int m = 0; m < C; ++m) wgl[L][m] = __ldg(a.wg + (size_t)b * 2 * C + L * C + m);
    __syncwarp();

    // ---------------- space domain: g[c][q][v] = sum_t xn[c][t][v] * A_s[v][t][q]  (:110, 'nctv,nvtq->ncqv'); lane = q
    {
      const float* as = (interp ? a.adj_s + (size_t)b * V * TT : W + d[CB_ADJ_S]) + (lane < T ? lane : T - 1);
      float cur[T], nxt[T];
#pragma unroll
      for (int t = 0; t < T; ++t) cur[t] = __ldg(as + t * T);
#pragma unroll 1
      for (int v = 0; v < V; ++v) {
        if (v + PF_AHEAD < V) prefetch_l2_warp(as - (lane < T ? lane : T - 1) + (v + PF_AHEAD) * TT, TT * 4);
        if (v + 1 < V) {
          const float* an = as + (v + 1) * TT;
#pragma unroll
          for (int t = 0; t < T; ++t) nxt[t] = __ldg(an + t * T);
        }
        float g[C];
#pragma unroll
        for (int c = 0; c < C; ++c) g[c] = 0.f;
#pragma unroll
        for (int t = 0; t < T; ++t)
#pragma unroll
          for (int c = 0; c < C; ++c) g[c] = fmaf(XN[c * TV + t * V + v], cur[t], g[c]);
        if (lane < T) {
          const int n = lane * V + v;
          float cacc[C];
          domain_epilogue(0, g, n, wgl[0], cacc);
#pragma unroll
          for (int m = 0; m < C; ++m) CA[m * TV + n] = cacc[m];
        }
#pragma unroll
        for (int t = 0; t < T; ++t) cur[t] = nxt[t];
      }
    }
    __syncwarp();
    // ---------------- time domain: g[c][t][w] = sum_v xn[c][t][v] * A_t[t][v][w]  (:117, 'nctv,ntvw->nctw'); lane = w
    float ssum[C];
#pragma unroll
    for (int m = 0; m < C; ++m) ssum[m] = 0.f;
    {
      const float* at = (interp ? a.adj_t + (size_t)b * T * VV : W + d[CB_ADJ_T]) + (lane < V ? lane : V - 1);
      float cur[V], nxt[V];
#pragma unroll
      for (int v = 0; v < V; ++v) cur[v] = __ldg(at + v * V);
#pragma unroll 1
      for (int t = 0; t < T; ++t) {
        if (t + PF_AHEAD < T) prefetch_l2_warp(at - (lane < V ? lane : V - 1) + (t + PF_AHEAD) * VV, VV * 4);
        if (t + 1 < T) {
          const float* an = at + (t + 1) * VV;
#pragma unroll
          for (int v = 0; v < V; ++v) nxt[v] = __ldg(an + v * V);
        }
        float g[C];
#pragma unroll
        for (int c = 0; c < C; ++c) g[c] = 0.f;
#pragma unroll
        for (int v = 0; v < V; ++v)
#pragma unroll
          for (int c = 0; c < C; ++c) g[c] = fmaf(XN[c * TV + t * V + v], cur[v], g[c]);
        if (lane < V) {
          const int n = t * V + lane;
          float cacc[C];
          domain_epilogue(1, g, n, wgl[1], cacc);
          // ---- c = PReLU(BN(compressor)) with the squeeze sums on the way (:306-307, SE.py:39)
#pragma unroll
          for (int m = 0; m < C; ++m) {
            const float cv = prelu(CA[m * TV + n] + cacc[m] + cb[m], ca);
            CA[m * TV + n] = cv;
            ssum[m] += cv;
          }
        }
#pragma unroll
        for (int v = 0; v < V; ++v) cur[v] = nxt[v];
      }
    }
    // ---------------- squeeze-excitation (SE.py:37-41): every lane computes the tiny MLP redundantly
    float gate[C];
    {
      float mean[C];
#pragma unroll
      for (int m = 0; m < C; ++m) mean[m] = warp_sum(ssum[m]) * (1.f / TV);
      const float* se1 = P(CB_SE1_WT);
      const float* se2 = P(CB_SE2_WT);
      const int hp = pad8i(Hs);
      float acc[C];
#pragma unroll
      for (int m = 0; m < C; ++m) acc[m] = 0.f;
      for (int h = 0; h < Hs; ++h) {
        float hv = 0.f;
#pragma unroll
        for (int c = 0; c < C; ++c) hv = fmaf(se1[c * hp + h], mean[c], hv);
        hv = fmaxf(hv, 0.f);
#pragma unroll
        for (int m = 0; m < C; ++m) acc[m] = fmaf(se2[h * Cop + m], hv, acc[m]);
      }
#pragma unroll
      for (int m = 0; m < C; ++m) gate[m] = sigmoidf(acc[m]);
    }
    if (lane == 0) {
#pragma unroll
      for (int m = 0; m < C; ++m) sv[m] = gate[m];
    }
    __syncwarp();
    // ---------------- out = c * gate + xn   (:390, identity block residual)
    {
      const size_t obase = (size_t)b * d[CB_OUT_SB];
      if (out_cfast) {
        for (int j = lane; j < C * TV; j += 32) {
          const int c = j % C, r = j / C, t = r % T, v = r / T, i = c * TV + t * V + v;
          st_act(a.out, obase + j, fmaf(CA[i], sv[c], XN[i]), obf);
        }
      } else {
        for (int i = lane; i < C * TV; i += 32) {
          const int c = i / TV, n = i - c * TV, t = n / V, v = n - t * V;
          st_act(a.out, obase + (size_t)c * osc + t * ost + v * osv, fmaf(CA[i], sv[c], XN[i]), obf);
        }
      }
    }
    __syncwarp();
  }
}

template <int T, int V, int C>
int launch_mix_narrow_impl(const MixArgs& a, void* stream) {
  return launch_warp_per_sample(dstd_mix_narrow_kernel<T, V, C>, a, stream);
}

}  // namespace cg
