// DSTD-GC block, stage 3 of 3, TENSOR-CORE variant: the same tile path as dstd_mix.cuh (adjacency products, channel
// mixes, gating, compressor, squeeze-excitation, block residual; models/CISTGCN/CISTGCN.py:110-123, 229-269, 305-318,
// 386-390, models/layers/SE.py:24-41), with every 1x1 channel mix -- tcn of both domains (+ the domain layers' residual
// conv), the compressor over cat(u1, u2) and the block residual conv -- on the tensor cores.
//
// Why warp-level mma.sync and not tcgen05 here: a channel mix of one sample is M = Co <= 32 rows x N = T*V = 220
// positions x K = Ci <= 32 -- per sample 0.23 MFLOP.  Round 1 put these GEMMs on tcgen05 (dstd_block.cuh, tc_gemm) and
// lost to the FP32-FMA loops: the fp32 [c][t*v] tiles had to be converted into a K-major split-16-bit staging operand
// before every MMA and read back from TMEM one position per lane after it (1.8 K + 4 K cycles per call around 0.5 K
// cycles of MMAs).  Register-operand MMAs need neither: a B fragment is two LDS.32 straight from the fp32 tile, the
// accumulator fragment is already in the registers of the lanes that run the epilogue, and every warp owns whole
// columns (positions) of the tile, so the in-place epilogue and the compressor that consumes it need no block barrier.
//
// fp32 accuracy on the TF32 pipe (3xTF32): x = hi + lo with hi = rna_tf32(x), lo = x - hi (exact in fp32, truncated to
// TF32 by the MMA); w likewise; x*w ~= lo*hi + hi*lo + hi*hi, accumulated in fp32, smallest terms first.  hi*hi is exact (11 x 11
// significant bits), the dropped lo*lo term is < 2^-22 |x w|: 3e-7 relative per product against 6e-8 for an FFMA.
// mma.sync.m16n8k8.tf32 issues at 0.47 / clk / SM on B200 (profiles/mma_sync_r1.log) = 159 effective MAC / clk / SM
// after the 3x, against the ~50 the FFMA tile loops of dstd_mix.cuh sustain (FMA pipe 39 % active, issue 60 %).
//
// Weights are re-laid at launch start into FRAGMENT order in shared memory: for (row tile mt of 16, k step ks of 8) one
// float4 per lane = {W[m][k], W[m+8][k], W[m][k+4], W[m+8][k+4]}, m = 16 mt + lane/4, k = 8 ks + lane%4 (zero outside the
// matrix), stored twice -- the hi image and the lo image of the 3xTF32 split, computed once per launch -- so an A
// fragment pair is two conflict-free LDS.128 shared by the warp's 3-4 column tiles and only the activations are split
// in the loop (2 LDS.32 + 6 ALU instructions per 6 MMAs).
#pragma once
#include "../../include/cistgcn_b200.h"
#include "dstd_block.cuh"
#include "dstd_mix.cuh"
#include "host_util.h"
#include "simt.h"

namespace cg {

constexpr int MMA_NT = 256;                 // threads per CTA (two CTAs per SM)

// Row stride of the two activation tiles: = 8 (mod 32), so that the B-fragment loads (lane = 4 g + q reads row q, column
// g: bank 8 q + g) and the float2 accesses of the epilogues (rows g, columns 2 q) are bank-conflict free; with the
// natural stride T*V = 220 = 28 (mod 32) both were 2-way conflicted (ncu: half of their wavefronts excessive).
__host__ __device__ constexpr int mma_ld(int TV) { return ((TV + 31) / 32) * 32 + 8; }
__host__ __device__ inline int mma_mt(int M) { return (M + 15) / 16; }
__host__ __device__ inline int mma_ks(int K) { return (K + 7) / 8; }

// Host: shared-memory plan of the tensor-core variant.  Same regions as mix_plan; the four GEMM weight fields hold the
// fragment-ordered images.
inline bool mix_mma_plan(MixArgs& a, int max_smem_floats) {
  const int* d = a.d;
  const int Ci = d[CB_CI], Co = d[CB_CO], T = d[CB_T], V = d[CB_V], Hs = d[CB_HS];
  const bool has_res = d[CB_HAS_RES] != 0;
  if (Ci > 32 || Co > 32) return false;                      // accumulator budget: two row tiles per warp
  const int TV = T * V, cmax = imax(Ci, Co), Cop = pad8i(Co);
  const int MT = mma_mt(Co), KSi = mma_ks(Ci), KSo = mma_ks(Co);
  if (((TV + 7) / 8 + 7) / 8 > 4) return false;              // at most four column tiles per warp
  for (int f = 0; f < CB_COUNT; ++f) { a.wsz[f] = 0; a.res[f] = -1; }
  int* z = a.wsz;
  z[CB_GN_S] = z[CB_GN_B] = Ci;
  for (int L = 0; L < 2; ++L) {
    z[CB_TCN_WT_S + L] = 2 * MT * KSi * (has_res ? 2 : 1) * 128; z[CB_TCN_B_S + L] = Co; z[CB_TCN_A_S + L] = 1;
    z[CB_P_S_S + L] = Co; z[CB_P_B_S + L] = Co; z[CB_P_A_S + L] = 1;
  }
  z[CB_CP_WT] = 2 * MT * 2 * KSo * 128; z[CB_CP_B] = Co; z[CB_CP_A] = 1;
  z[CB_SE1_WT] = Co * pad8i(Hs); z[CB_SE2_WT] = Hs * Cop;
  if (has_res) { z[CB_RS_WT] = 2 * MT * KSi * 128; z[CB_RS_B] = Co; }
  for (int f = 0; f < CB_COUNT; ++f) z[f] = pad4i(z[f]);
  const int LD = mma_ld(TV);
  a.o_xn = 0;
  a.o_a = pad4i(Ci * LD);
  // (the B fragments of the last, partial column tile read the row padding behind column T*V: column-local garbage in
  // accumulator columns that are never stored)
  a.o_adj = a.o_a + pad4i(cmax * LD);
  // adjacency region; the squeeze partial sums [NW][32] alias it behind Adj_s (Adj_t is dead by then)
  // (the next sample's Adj_s is copied in behind the second domain's channel mix, so the partials sit behind it)
  const int adj = imax(imax(pad4i(T * T * (V | 1)) + (MMA_NT / 32) * 32, T * pad4i(V * V)), (MMA_NT / 32) * 32);
  a.o_sm = a.o_adj + adj;
  int cur = a.o_sm + pad4i(2 * Co) + 2 * pad4i(Co) + pad4i(Hs);
  for (int f = 0; f < CB_COUNT; ++f)
    if (z[f]) { a.res[f] = cur; cur += z[f]; }
  a.smem_floats = cur;
  return cur <= max_smem_floats;
}

// (TF32 helpers tf32_rna / tf32_split / mma_tf32: simt.h)

// Fragment-ordered hi | lo images of a k-major weight matrix W[k][Mp] (rows k0 .. k0+K-1 of it), M x K, zero padded:
// dst[0 .. n) = hi, dst[n .. 2n) = lo, n = MT * KS * 128.
template <int NT>
CG_DEV void build_frag_image(float* dst, const float* __restrict__ W, int Mp, int M, int K, int k0) {
  const int MT = mma_mt(M), KS = mma_ks(K), n = MT * KS * 128;
  for (int i = threadIdx.x; i < n; i += NT) {
    const int j = i & 3, ln = (i >> 2) & 31, tile = i >> 7, ks = tile % KS, mt = tile / KS;
    const int m = mt * 16 + (ln >> 2) + ((j & 1) ? 8 : 0), k = ks * 8 + (ln & 3) + ((j & 2) ? 4 : 0);
    const float w = (m < M && k < K) ? __ldg(W + (size_t)(k0 + k) * Mp + m) : 0.f;
    float hi, lo;
    tf32_split(w, hi, lo);
    dst[i] = hi; dst[n + i] = lo;
  }
}

// acc[nt][mt] += Wfrag (MT x KS fragment tiles, hi image then lo image) * X[k][n] for `ntiles` (<= NTP) of the warp's
// column tiles, tile i at columns nbase + i * NSTRIDE; X is an fp32 tile in shared memory with row stride LD.
template <int NTP, int MT, int LD, int NSTRIDE>
CG_DEV void mma_gemm(float (&acc)[NTP][MT][4], const float* wfrag, int KS, int K, const float* X, int nbase, int ntiles) {
  const int lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3;
  const float* wlo = wfrag + MT * KS * 128;
#pragma unroll 1
  for (int ks = 0; ks < KS; ++ks) {
    float ah[MT][4], al[MT][4];
#pragma unroll
    for (int mt = 0; mt < MT; ++mt) {
      const float4 h4 = *reinterpret_cast<const float4*>(wfrag + ((mt * KS + ks) * 32 + lane) * 4);
      const float4 l4 = *reinterpret_cast<const float4*>(wlo + ((mt * KS + ks) * 32 + lane) * 4);
      ah[mt][0] = h4.x; ah[mt][1] = h4.y; ah[mt][2] = h4.z; ah[mt][3] = h4.w;
      al[mt][0] = l4.x; al[mt][1] = l4.y; al[mt][2] = l4.z; al[mt][3] = l4.w;
    }
    const int k0 = ks * 8 + q, k1 = k0 + 4;
    const float* x0 = X + (k0 < K ? k0 : 0) * LD + g;      // rows beyond K meet zero weights; keep the address inside the tile
    const float* x1 = X + (k1 < K ? k1 : 0) * LD + g;
    // splits of all (<= NTP) tiles first, then the MMAs term by term: the three products of one accumulator are issued
    // NTP * MT MMAs apart, so that a warp does not sit out the MMA latency between them
    float bh[NTP][2], bl[NTP][2];
#pragma unroll
    for (int nt = 0; nt < NTP; ++nt) {
      const int col = nt < ntiles ? nbase + nt * NSTRIDE : nbase;      // inactive tile: a valid address, no MMA
      tf32_split(x0[col], bh[nt][0], bl[nt][0]);
      tf32_split(x1[col], bh[nt][1], bl[nt][1]);
    }
#pragma unroll
    for (int nt = 0; nt < NTP; ++nt)
      if (nt == 0 || nt < ntiles) {
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) mma_tf32(acc[nt][mt], al[mt], bh[nt]);
      }
#pragma unroll
    for (int nt = 0; nt < NTP; ++nt)
      if (nt == 0 || nt < ntiles) {
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) mma_tf32(acc[nt][mt], ah[mt], bl[nt]);
      }
#pragma unroll
    for (int nt = 0; nt < NTP; ++nt)
      if (nt == 0 || nt < ntiles) {
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) mma_tf32(acc[nt][mt], ah[mt], bh[nt]);
      }
  }
}

template <class ACC>
CG_DEV void zero_acc(ACC& acc) {
  float* p = &acc[0][0][0];
#pragma unroll
  for (int i = 0; i < (int)(sizeof(ACC) / sizeof(float)); ++i) p[i] = 0.f;
}

// MT = row tiles of 16 output channels (1: Co <= 16, 2: Co <= 32)
template <int T, int V, int MT>
__global__ void __launch_bounds__(MMA_NT, 2) dstd_mix_mma_kernel(const MixArgs a) {
  CG_DYN_SMEM(smem);
  constexpr int NT = MMA_NT, NW = NT / 32;
  constexpr int TV = T * V, TT = T * T, VV = V * V, VP = V | 1;
  constexpr int VVP = (VV + 3) & ~3;
  constexpr int NTP = 2;
  constexpr int NTILES = (TV + 7) / 8, NTW = (((NTILES + NW - 1) / NW + NTP - 1) / NTP) * NTP;    // per warp, padded to whole passes                               // column tiles per pass of the in-place phases (register budget)
  constexpr int LD = mma_ld(TV);                       // row stride of the XN / A tiles
  static_assert(TV % 2 == 0, "column pairs");
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, q = lane & 3;
  const int* d = a.d;
  const float* __restrict__ W = a.w;
  const int Ci = d[CB_CI], Co = d[CB_CO], Hs = d[CB_HS];
  const bool has_res = d[CB_HAS_RES] != 0, interp = d[CB_INTERP] != 0;
  const int Cop = pad8i(Co);
  const int KSi = mma_ks(Ci), KSo = mma_ks(Co);

  float* XN = smem + a.o_xn;
  float* A = smem + a.o_a;
  float* ADJ = smem + a.o_adj;
  float* p = smem + a.o_sm;
  float* wg = p;      p += pad4i(2 * Co);
  float* semean = p;  p += pad4i(Co);
  float* gate = p;    p += pad4i(Co);
  float* hid = p;     p += pad4i(Hs);
  float* separt = ADJ + pad4i(TT * VP);                // [NW][32] squeeze partial sums (row m of the warp's columns); Adj_t is dead by then
  auto P = [&](int f) -> const float* { return smem + a.res[f]; };
  auto Pw = [&](int f) -> float* { return smem + a.res[f]; };

  // ---------------- once per launch: resident vectors (plain copies) and fragment images of the four GEMM operands
  for (int f = 0; f < CB_COUNT; ++f) {
    if (a.res[f] < 0) continue;
    const bool frag = f == CB_TCN_WT_S || f == CB_TCN_WT_T || f == CB_CP_WT || f == CB_RS_WT;
    if (!frag) copy_async<NT>(smem + a.res[f], W + d[f], a.wsz[f]);
  }
  cp_async_commit();
  for (int L = 0; L < 2; ++L) {
    build_frag_image<NT>(Pw(CB_TCN_WT_S + L), W + d[CB_TCN_WT_S + L], Cop, Co, Ci, 0);
    if (has_res) build_frag_image<NT>(Pw(CB_TCN_WT_S + L) + 2 * MT * KSi * 128, W + d[CB_TCN_WT_S + L], Cop, Co, Ci, Ci);
    build_frag_image<NT>(Pw(CB_CP_WT) + L * 2 * MT * KSo * 128, W + d[CB_CP_WT], Cop, Co, Co, L * Co);
  }
  if (has_res) build_frag_image<NT>(Pw(CB_RS_WT), W + d[CB_RS_WT], Cop, Co, Ci, 0);
  cp_async_wait_all();
  __syncthreads();

  const float* gs = P(CB_GN_S);
  const float* gb = P(CB_GN_B);
  const float* cb = P(CB_CP_B);
  const float ca = P(CB_CP_A)[0];

  // the warp's column tiles (8 positions each): tiles warp, warp + NW, ... -> columns 8 warp + i * NS
  constexpr int NS = NW * 8;
  const int ntiles_w = (NTILES - warp + NW - 1) / NW;

  // ---- operands fetched a sample ahead
  // Adj_s (V,T,T) -> [t][q][v] with an odd row stride, as 4-byte cp.async gathers (no register staging)
  auto adj_s_fetch = [&](int bb) {
    const float* as = interp ? a.adj_s + (size_t)bb * V * TT : W + d[CB_ADJ_S];
    for (int i = tid; i < V * TT; i += NT) { const int v = i / TT, r = i - v * TT; cp_async4(ADJ + r * VP + v, as + i); }
    cp_async_commit();
  };
  bool adj_ahead = false;                              // CTA-uniform
  // channels per thread of the adjacency products: every thread runs ceil(items / NT) items of tc channels one after the
  // other, so the phase lasts rounds * tc; ties go to the wider tile (fewer operand loads per FMA).  32 channels: tc = 3
  // (242 / 220 items, one round) instead of two rounds of 2.
  auto pick_tc = [&](int per_ctile) {
    if (Ci < 16) return Ci >= 2 ? 2 : 1;               // measured: at 10 channels one round of 2 beats one round of 1 (operand loads)
    int best = 1, cost = 1 << 30;
    for (int tc = 1; tc <= 4; ++tc) {
      const int items = ((Ci + tc - 1) / tc) * per_ctile, c = ((items + NT - 1) / NT) * tc;
      if (c <= cost) { cost = c; best = tc; }
    }
    return best;
  };
  constexpr int GT_TW = (V % 11 == 0) ? 11 : ((V % 9 == 0) ? 9 : ((V % 5 == 0) ? 5 : 1));   // gcn_time's column tile
  const int tc_space = pick_tc(V), tc_time = pick_tc(T * (V / GT_TW));

  for (int b = blockIdx.x; b < a.batch; b += gridDim.x) {
    // the next sample's operands (input tile, both adjacencies) start their way from HBM into L2 now: the tile load at the
    // top of the next iteration is exposed (two samples in flight per SM), an L2 hit halves what it waits for.  (Loading the
    // next tile into registers behind the squeeze-excitation was tried: at the 128-register cap it spilled and cost 9 %.)
    if (b + (int)gridDim.x < a.batch) {
      const size_t bn = (size_t)b + gridDim.x;
      if (d[CB_IN_MODE] == 1) prefetch_l2_range<NT>(a.in + bn * d[CB_IN_SB], (size_t)TV * 3 * 4);
      else if (d[CB_IN_SV] == 1 && d[CB_IN_ST] == V && d[CB_IN_SC] == TV)
        prefetch_l2_range<NT>(reinterpret_cast<const char*>(a.in) + bn * d[CB_IN_SB] * (a.in_bf16 ? 2 : 4), (size_t)Ci * TV * (a.in_bf16 ? 2 : 4));
      if (interp) {
        prefetch_l2_range<NT>(a.adj_s + bn * V * TT, (size_t)V * TT * 4);
        prefetch_l2_range<NT>(a.adj_t + bn * T * VV, (size_t)T * VV * 4);
      }
    }
    // ---------------- load + global_norm (:375); block 0 builds the 10 features (:568-577); gates; Adj_s
    if (tid < 2 * Co) wg[tid] = __ldg(a.wg + (size_t)b * 2 * Co + tid);
    if (!adj_ahead) adj_s_fetch(b);                    // first sample of the CTA; later ones were fetched a sample ahead
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
        for (int c = 0; c < 10; ++c) XN[c * LD + n] = fmaf(gs[c], f[c], gb[c]);
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
          *reinterpret_cast<float4*>(XN + c * LD + (i * 4 - c * TV)) = v4;
        }
      } else {
        for (int i = tid; i < Ci * TV; i += NT) {
          const int c = i / TV, n = i - c * TV, t = n / V, v = n - t * V;
          XN[c * LD + n] = fmaf(gs[c], ld_act(a.in, sbase_ + (size_t)c * sc + t * st + v * sv, ibf), gb[c]);
        }
      }
    }
    cp_async_wait_all();                               // Adj_s
    __syncthreads();

    float cacc[NTW][MT][4];                            // compressor accumulators over both domains (:305)
    zero_acc(cacc);

#pragma unroll 1
    for (int L = 0; L < 2; ++L) {
      // ---------------- g = XN x Adj  (:110, :117, :123) -> A   (FP32 FMA: per-sample operands on both sides)
      if (L == 0) {
        switch (tc_space) {
          case 4: gcn_space<T, V, 4, NT, LD>(XN, ADJ, A, Ci); break;
          case 3: gcn_space<T, V, 3, NT, LD>(XN, ADJ, A, Ci); break;
          case 2: gcn_space<T, V, 2, NT, LD>(XN, ADJ, A, Ci); break;
          default: gcn_space<T, V, 1, NT, LD>(XN, ADJ, A, Ci);
        }
      } else {
        switch (tc_time) {
          case 4: gcn_time<T, V, 4, NT, LD>(XN, ADJ, A, Ci); break;
          case 3: gcn_time<T, V, 3, NT, LD>(XN, ADJ, A, Ci); break;
          case 2: gcn_time<T, V, 2, NT, LD>(XN, ADJ, A, Ci); break;
          default: gcn_time<T, V, 1, NT, LD>(XN, ADJ, A, Ci);
        }
      }
      __syncthreads();
      if (L == 1) {
        // Adj_t is dead: the NEXT sample's Adj_s comes in behind this domain's channel mix, the compressor and the SE
        adj_ahead = b + (int)gridDim.x < a.batch;
        if (adj_ahead) adj_s_fetch(b + (int)gridDim.x);
      }
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
      // ---------------- x_L = PReLU(BN(W g + b) + res); u_L = PReLU(BN(w_L * x_L))  (:266-268, :388), in place on the
      // warp's own columns, NTP column tiles at a time
      {
        const float* wt = P(CB_TCN_WT_S + L);
        const float* tb = P(CB_TCN_B_S + L);
        const float* ps = P(CB_P_S_S + L);
        const float* pb = P(CB_P_B_S + L);
        const float ta = P(CB_TCN_A_S + L)[0], pa = P(CB_P_A_S + L)[0];
        const float* wgl = wg + L * Co;
#pragma unroll 1
        for (int i0 = 0; i0 < ntiles_w; i0 += NTP) {
          const int nti = ntiles_w - i0 < NTP ? ntiles_w - i0 : NTP;
          float acc[NTP][MT][4];
          zero_acc(acc);
          const int nb0 = warp * 8 + i0 * NS;
          mma_gemm<NTP, MT, LD, NS>(acc, wt, KSi, Ci, A, nb0, nti);
          if (has_res) mma_gemm<NTP, MT, LD, NS>(acc, wt + 2 * MT * KSi * 128, KSi, Ci, XN, nb0, nti);   // domain layer's residual conv
          __syncwarp();                                // every lane of the warp is done reading the columns it overwrites
#pragma unroll
          for (int mt = 0; mt < MT; ++mt) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const int m = mt * 16 + g + 8 * h;
              if (m < Co) {
                const float tbm = tb[m], sc = ps[m] * wgl[m], pbm = pb[m];
#pragma unroll
                for (int i = 0; i < NTP; ++i) {
                  const int n = nb0 + i * NS + 2 * q;
                  if (i < nti && n < TV) {
                    float x0 = acc[i][mt][2 * h] + tbm, x1 = acc[i][mt][2 * h + 1] + tbm;
                    if (!has_res) { const float2 r = *reinterpret_cast<const float2*>(XN + m * LD + n); x0 += r.x; x1 += r.y; }
                    x0 = prelu(x0, ta); x1 = prelu(x1, ta);
                    *reinterpret_cast<float2*>(A + m * LD + n) = make_float2(prelu(fmaf(sc, x0, pbm), pa), prelu(fmaf(sc, x1, pbm), pa));
                  }
                }
              }
            }
          }
        }
        __syncwarp();
      }
      // ---------------- compressor, this domain's half of the K range  (:305)
#pragma unroll
      for (int i0 = 0; i0 < NTW; i0 += NTP) {
        if (i0 < ntiles_w)
          mma_gemm<NTP, MT, LD, NS>(*reinterpret_cast<float (*)[NTP][MT][4]>(&cacc[i0][0][0]), P(CB_CP_WT) + L * 2 * MT * KSo * 128, KSo, Co,
                                    A, warp * 8 + i0 * NS, ntiles_w - i0);
      }
      if (L == 0) cp_async_wait_all();
      __syncthreads();            // everyone is done reading u_L (and Adj_t has landed)
    }
    // ---------------- c = PReLU(BN(.)) -> A, with the squeeze sums on the way  (:306-307, SE.py:39)
#pragma unroll
    for (int mt = 0; mt < MT; ++mt) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int m = mt * 16 + g + 8 * h;
        float rs = 0.f;
        if (m < Co) {
          const float bias = cb[m];
#pragma unroll
          for (int i = 0; i < NTW; ++i) {
            const int n = warp * 8 + i * NS + 2 * q;
            if (i < ntiles_w && n < TV) {
              const float v0 = prelu(cacc[i][mt][2 * h] + bias, ca), v1 = prelu(cacc[i][mt][2 * h + 1] + bias, ca);
              rs += v0 + v1;
              *reinterpret_cast<float2*>(A + m * LD + n) = make_float2(v0, v1);
            }
          }
        }
        rs += __shfl_xor_sync(0xffffffffu, rs, 1);     // the four lanes that share row m
        rs += __shfl_xor_sync(0xffffffffu, rs, 2);
        if (q == 0) separt[warp * 32 + m] = rs;
      }
    }
    __syncthreads();
    if (tid < Co) {
      float s = 0.f;
      for (int w = 0; w < NW; ++w) s += separt[w * 32 + tid];      // fixed order: bit-reproducible
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
#pragma unroll 1
        for (int i0 = 0; i0 < ntiles_w; i0 += NTP) {
          const int nti = ntiles_w - i0 < NTP ? ntiles_w - i0 : NTP;
          float acc[NTP][MT][4];
          zero_acc(acc);
          const int nb0 = warp * 8 + i0 * NS;
          mma_gemm<NTP, MT, LD, NS>(acc, P(CB_RS_WT), KSi, Ci, XN, nb0, nti);
#pragma unroll
          for (int mt = 0; mt < MT; ++mt) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const int m = mt * 16 + g + 8 * h;
              if (m < Co) {
                const float gm = gate[m], bias = rbias[m];
#pragma unroll
                for (int i = 0; i < NTP; ++i) {
                  const int n = nb0 + i * NS + 2 * q;
                  if (i < nti && n < TV) {
                    const float2 c2 = *reinterpret_cast<const float2*>(A + m * LD + n);
                    const float v0 = fmaf(c2.x, gm, acc[i][mt][2 * h] + bias), v1 = fmaf(c2.y, gm, acc[i][mt][2 * h + 1] + bias);
                    if (contiguous) {
                      st_act(a.out, obase + (size_t)m * TV + n, v0, obf);
                      st_act(a.out, obase + (size_t)m * TV + n + 1, v1, obf);
                    } else {
                      const int t0 = n / V, v0i = n - t0 * V;
                      st_act(a.out, obase + (size_t)m * sc + t0 * st + v0i * sv, v0, obf);
                      const int n1 = n + 1, t1 = n1 / V, v1i = n1 - t1 * V;
                      st_act(a.out, obase + (size_t)m * sc + t1 * st + v1i * sv, v1, obf);
                    }
                  }
                }
              }
            }
          }
        }
      } else if (contiguous) {
        for (int i = tid; i < Co * TV / 4; i += NT) {
          const int m = (i * 4) / TV, n = i * 4 - m * TV;
          const float gm = gate[m];
          const float4 c4 = *reinterpret_cast<const float4*>(A + m * LD + n);
          const float4 x4 = *reinterpret_cast<const float4*>(XN + m * LD + n);
          st_act4(a.out, obase + (size_t)i * 4,
                  make_float4(fmaf(c4.x, gm, x4.x), fmaf(c4.y, gm, x4.y), fmaf(c4.z, gm, x4.z), fmaf(c4.w, gm, x4.w)), obf);
        }
      } else {
        for (int i = tid; i < Co * TV; i += NT) {
          const int m = i / TV, n = i - m * TV, t = n / V, v = n - t * V;
          st_act(a.out, obase + (size_t)m * sc + t * st + v * sv, fmaf(A[m * LD + n], gate[m], XN[m * LD + n]), obf);
        }
      }
    }
    __syncthreads();
  }
}

template <int T, int V, int MT>
inline int launch_mix_mma_mt(const MixArgs& a, void* stream) {
  auto kfn = dstd_mix_mma_kernel<T, V, MT>;
  const size_t smem = (size_t)a.smem_floats * sizeof(float);
  int err = 0;
  const int per_sm = prepared_blocks_per_sm(kfn, MMA_NT, smem, &err);
  if (err) return err;
  const int grid = grid_for(a.batch, per_sm);
  CG_LAUNCH(kfn, grid, MMA_NT, smem, stream, a);
  return last_launch_error();
}
template <int T, int V>
int launch_mix_mma_impl(const MixArgs& a, void* stream) {
  return mma_mt(a.d[CB_CO]) == 1 ? launch_mix_mma_mt<T, V, 1>(a, stream) : launch_mix_mma_mt<T, V, 2>(a, stream);
}

}  // namespace cg
