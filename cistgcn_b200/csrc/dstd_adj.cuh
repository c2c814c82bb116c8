// DSTD-GC block, stage 2 of 3: the per-sample VECTOR path -- from the `red` record of stage 1 (dstd_reduce.cuh) to the
// two context gates and the two sample-specific adjacencies (reference: models/CISTGCN/CISTGCN.py:327-352, 378-384 the
// gate nets conv_{s,t}.4-7 + map_{s,t}; :144, :152 the last 1x1 of Map2Adj's compress branches; :155-170, :183-189 the
// outer products and the expansor).
//
// In round 1 these were ~10 serial phases of one 16-warp CTA per sample (gate matvecs alone: 14 K cycles for 25 K MACs).
// Here one WARP owns one sample, end to end, with warp-level synchronisation only; every weight matrix is resident in
// shared memory and shared by all warps of the CTA; 8-16 samples are in flight per SM.
//   gate conv (1,V) and the gate MLP: lanes = output channels, the input vector is broadcast from shared memory;
//   dim_seq / dim_space: lanes = joints, register tile over the frames;
//   expansor: lanes = columns of the outer-product map o (never materialised); the hidden column lives in registers,
//             weight rows are warp-uniform 128-bit loads; the result is written with coalesced stores in the
//             reference's own (V,T,T) / (T,V,V) layout, i.e. the interpretability taps of environment/test.py:146-157
//             and the operand of stage 3 are the same buffer.
//   expansor on the tensor cores (default): the two layers are CHAINED register-operand 3xTF32 mma.sync.m16n8k8 GEMMs
//             with the map COLUMNS as the M dimension (16 per tile, two tiles per round): the A fragment of layer 1 is
//             the outer product itself, computed in the lanes that feed it; the accumulator fragment of layer 1
//             (bias + PReLU applied in place) IS the A fragment of layer 2 once the k slots of layer 2's weight image
//             are permuted to the accumulator's column order (slot q <-> hidden 2q, slot q + 4 <-> hidden 2q + 1), so
//             the hidden map never leaves the registers and needs no shuffle.  Weights: fragment-ordered hi | lo
//             images built once per launch (one conflict-free LDS.128 per 8 x 8 tile).  2.3-2.7x fewer warp
//             instructions than the FFMA column loops at N = 22 / 25, about the same at N = 10 (16 x 16 padding).
#pragma once
#include "../../include/cistgcn_b200.h"
#include "dstd_reduce.cuh"
#include "simt.h"

namespace cg {

constexpr int ADJ_CPL = 2;            // expansor columns per lane and weight-row read
constexpr int ADJ_MAX_WARPS = 8;      // 256 threads: up to 255 registers per thread (the 25-wide expansor columns need ~200)
#ifdef CISTGCN_EMU
constexpr int ADJ_MMA_MAX_WARPS = 4;  // emulator: one OS thread per CUDA thread -- keep the CTAs small
#else
constexpr int ADJ_MMA_MAX_WARPS = 16; // tensor-core expansor: 512 threads, up to 128 registers per thread
#endif

struct AdjArgs {
  int d[CB_COUNT];
  int res[CB_COUNT];       // shared-memory float offset of the resident copy of weight field f, or -1 (read through L1/L2)
  int wsz[CB_COUNT];       // floats of weight field f (multiple of 4), 0 if unused here
  const float* w;
  const float* red;
  int red_stride;
  float* wg;               // (B, 2, Co) gates w1 | w2
  float* adj_s;            // (B, V, T, T)
  float* adj_t;            // (B, T, V, V)
  float* tap_w1;           // optional (B, Co) copies for the interpretability taps
  float* tap_w2;
  int batch, nwarps;
  int o_warp, warp_floats, smem_floats;
  int mma;                 // expansor as chained 3xTF32 mma.sync GEMMs (default) instead of the FFMA column loops
  int o_f1[2], o_f2[2];    // shared-memory float offsets of the fragment images of expansor.0 / expansor.4, per domain
};

__host__ __device__ inline int apad8(int n) { return (n + 7) & ~7; }
__host__ __device__ inline int imax_(int a, int b) { return a > b ? a : b; }

// Host: residency plan.  Vectors first, then matrices by reuse; what does not fit is read through L1 / L2.
__host__ __device__ inline int adj_frag_floats(int n) { const int ks = (n + 7) / 8; return ks * ks * 128; }

inline bool adj_plan(AdjArgs& a, int max_smem_floats, bool mma = true) {
  const int* d = a.d;
  const int Co = d[CB_CO], T = d[CB_T], V = d[CB_V], Ch = d[CB_CH], Cg = d[CB_CG];
  const bool interp = d[CB_INTERP] != 0;
  const int Cop = apad8(Co), TV = T * V;
  if (Co > 32 || T > 32 || V > 32) return false;
  for (int f = 0; f < CB_COUNT; ++f) { a.wsz[f] = 0; a.res[f] = -1; }
  int* z = a.wsz;
  z[CB_G4_WT] = 2 * Cg * V * Cop; z[CB_G4_B] = 2 * Co; z[CB_G4_A] = 2;
  z[CB_M0_WT] = 2 * (Co + 2 + 2 * T) * Cop; z[CB_M0_B] = 2 * Co; z[CB_M0_A] = 2;
  z[CB_M4_WT] = 2 * Co * Cop;
  if (interp) {
    for (int L = 0; L < 2; ++L) {
      const int n = L == 0 ? V : T;
      z[CB_TC6_WT_S + L] = Ch * apad8(T); z[CB_JC6_WT_S + L] = Ch * apad8(V);
      z[CB_E0_B_S + L] = n; z[CB_E0_A_S + L] = 1;
      if (!mma) { z[CB_E0_WT_S + L] = n * apad8(n); z[CB_E4N_WT_S + L] = n * apad8(n); }
    }
  }
  a.mma = mma && interp;
  for (int f = 0; f < CB_COUNT; ++f) z[f] = rpad4(z[f]);
  const RedLayout RL(T, V, Cg, Ch, interp);
  // per warp: the red record; dim_seq / dim_space (4 x T*V) start where the gate inputs (statistics, hidden maps) begin --
  // the gates are finished before Map2Adj starts -- and run past the record's end if they need to; then the gate vectors
  a.warp_floats = imax_(rpad4(RL.total), interp ? RL.stats + 4 * rpad4(TV) : 0) + 4 * rpad4(Co);
  const int order[] = {CB_G4_B, CB_G4_A, CB_M0_B, CB_M0_A, CB_E0_B_S, CB_E0_B_T, CB_E0_A_S, CB_E0_A_T,
                       CB_E0_WT_S, CB_E0_WT_T, CB_E4N_WT_S, CB_E4N_WT_T, CB_TC6_WT_S, CB_TC6_WT_T, CB_JC6_WT_S, CB_JC6_WT_T,
                       CB_M0_WT, CB_M4_WT, CB_G4_WT};
  const int min_warps = 8;
  int cur = 0;
  if (a.mma)
    for (int L = 0; L < 2; ++L) {                     // fragment images: always resident
      const int n = L == 0 ? V : T;
      a.o_f1[L] = cur; cur += adj_frag_floats(n);
      a.o_f2[L] = cur; cur += adj_frag_floats(n);
    }
  for (int f : order) {
    if (z[f] == 0) continue;
    if (cur + z[f] + min_warps * a.warp_floats <= max_smem_floats) { a.res[f] = cur; cur += z[f]; }
  }
  if (a.mma)                                          // the tensor-core kernel addresses its weights as shared memory only
    for (int f = 0; f < CB_COUNT; ++f)
      if (z[f] && a.res[f] < 0) return false;
  a.o_warp = cur;
  int nw = (max_smem_floats - cur) / a.warp_floats;
  if (nw > (a.mma ? ADJ_MMA_MAX_WARPS : ADJ_MAX_WARPS)) nw = a.mma ? ADJ_MMA_MAX_WARPS : ADJ_MAX_WARPS;
  if (nw < 2) return false;
  a.nwarps = nw;
  a.smem_floats = cur + nw * a.warp_floats;
  return true;
}

// Map2Adj.expansor (CISTGCN.py:165-170) as an independent two-layer N -> N -> N MLP for every column of the outer-product
// map: out[:, col] = W4 PReLU(W0 o[:, col] + b0).  w0 k-major [k][pad8(N)], w4 row-major [m][pad8(N)].
// Every lane owns CPL columns at a time (col, col + 32, ...): a warp-uniform weight row is read ONCE (128-bit broadcast
// loads, the scarce resource: 2 wavefronts per 4 floats) and feeds CPL * N FFMAs per lane; the hidden columns live in
// registers and the result goes straight to memory, one output row at a time (coalesced over the lanes).
template <int N, int NCOLS, int CPL, class OFN, class STORE>
CG_DEV void expansor_warp(const float* w0, const float* b0, float a0, const float* w4, OFN o_at, STORE store) {
  constexpr int NPW = (N + 7) & ~7;
  const int lane = threadIdx.x & 31;
#pragma unroll 1
  for (int c0 = 0; c0 < NCOLS; c0 += 32 * CPL) {
    bool active[CPL];
    int col[CPL];
#pragma unroll
    for (int u = 0; u < CPL; ++u) {
      active[u] = c0 + 32 * u + lane < NCOLS;
      col[u] = active[u] ? c0 + 32 * u + lane : NCOLS - 1;
    }
    w0 = opaque_ptr(w0);                            // the weight rows are re-read every round, not hoisted out of it
    w4 = opaque_ptr(w4);
    b0 = opaque_ptr(b0);
    float h[CPL][N];
#pragma unroll
    for (int u = 0; u < CPL; ++u)
#pragma unroll
      for (int j = 0; j < N; ++j) h[u][j] = 0.f;
#pragma unroll 2
    for (int k = 0; k < N; ++k) {
      float ok[CPL];
#pragma unroll
      for (int u = 0; u < CPL; ++u) ok[u] = o_at(k, col[u]);
      float wrow[NPW];
#pragma unroll
      for (int i = 0; i < NPW / 4; ++i) {
        const float4 q = *reinterpret_cast<const float4*>(w0 + k * NPW + 4 * i);
        wrow[4 * i] = q.x; wrow[4 * i + 1] = q.y; wrow[4 * i + 2] = q.z; wrow[4 * i + 3] = q.w;
      }
#pragma unroll
      for (int u = 0; u < CPL; ++u)
#pragma unroll
        for (int j = 0; j < N; ++j) h[u][j] = fmaf(wrow[j], ok[u], h[u][j]);
    }
#pragma unroll
    for (int j = 0; j < N; ++j) {
      const float bj = b0[j];
#pragma unroll
      for (int u = 0; u < CPL; ++u) h[u][j] = prelu(h[u][j] + bj, a0);
    }
#pragma unroll 1
    for (int m = 0; m < N; ++m) {
      float wrow[NPW];
#pragma unroll
      for (int i = 0; i < NPW / 4; ++i) {
        const float4 q = *reinterpret_cast<const float4*>(w4 + m * NPW + 4 * i);
        wrow[4 * i] = q.x; wrow[4 * i + 1] = q.y; wrow[4 * i + 2] = q.z; wrow[4 * i + 3] = q.w;
      }
#pragma unroll
      for (int u = 0; u < CPL; ++u) {
        float o0 = 0.f, o1 = 0.f;
#pragma unroll
        for (int k = 0; k + 1 < N; k += 2) { o0 = fmaf(wrow[k], h[u][k], o0); o1 = fmaf(wrow[k + 1], h[u][k + 1], o1); }
        if (N & 1) o0 = fmaf(wrow[N - 1], h[u][N - 1], o0);
        if (active[u]) store(m, col[u], o0 + o1);
      }
    }
  }
}

// ---- expansor on the tensor cores ------------------------------------------------------------------------------------
// Fragment images of the two expansor matrices for mma.sync.m16n8k8 (B operand, 8 x 8 tiles, tile index kt * NKS + nt),
// one float4 per lane = {b0 hi, b1 hi, b0 lo, b1 lo} of the 3xTF32 split; lane = 4 g + q:
//   layer 1 (w0 k-major [k][pad8(N)]):  b0 = W0[j = 8 nt + g][k = 8 kt + q], b1 = same j, k + 4
//   layer 2 (w4 row-major [m][pad8(N)]): the k slots follow the ACCUMULATOR column order of layer 1, slot q <-> hidden
//            8 kt + 2 q, slot q + 4 <-> hidden 8 kt + 2 q + 1:  b0 = W4[m = 8 nt + g][8 kt + 2 q], b1 = W4[m][8 kt + 2 q + 1]
template <int N>
CG_DEV void build_expansor_frags(float* f1, float* f2, const float* __restrict__ w0, const float* __restrict__ w4, int nthreads) {
  constexpr int NKS = (N + 7) / 8, NPW = (N + 7) & ~7;
  for (int i = threadIdx.x; i < NKS * NKS * 32; i += nthreads) {
    const int ln = i & 31, tile = i >> 5, nt = tile % NKS, kt = tile / NKS, g = ln >> 2, q = ln & 3;
    const int n = 8 * nt + g;
    float v[4];
    v[0] = (n < N && 8 * kt + q < N) ? __ldg(w0 + (8 * kt + q) * NPW + n) : 0.f;
    v[1] = (n < N && 8 * kt + q + 4 < N) ? __ldg(w0 + (8 * kt + q + 4) * NPW + n) : 0.f;
    v[2] = (n < N && 8 * kt + 2 * q < N) ? __ldg(w4 + n * NPW + 8 * kt + 2 * q) : 0.f;
    v[3] = (n < N && 8 * kt + 2 * q + 1 < N) ? __ldg(w4 + n * NPW + 8 * kt + 2 * q + 1) : 0.f;
    float hi[4], lo[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) tf32_split(v[e], hi[e], lo[e]);
    f1[4 * i] = hi[0]; f1[4 * i + 1] = hi[1]; f1[4 * i + 2] = lo[0]; f1[4 * i + 3] = lo[1];
    f2[4 * i] = hi[2]; f2[4 * i + 1] = hi[3]; f2[4 * i + 2] = lo[2]; f2[4 * i + 3] = lo[3];
  }
}

// acc[tile][nt] += A[tile] (16 x 8 fragments, hi / lo) * B[kt][nt] for all NKS column tiles of the weight image; the three
// products of one accumulator are issued 2 * NKS MMAs apart (smallest terms first) so a warp does not wait out the MMA latency.
template <int NKS>
CG_DEV void expansor_mma_step(float (&acc)[2][NKS][4], const float (&ah)[2][4], const float (&al)[2][4], const float* frag, int kt) {
  const int lane = threadIdx.x & 31;
  float bh[NKS][2], bl[NKS][2];
#pragma unroll
  for (int nt = 0; nt < NKS; ++nt) {
    const float4 b4 = *reinterpret_cast<const float4*>(frag + ((kt * NKS + nt) * 32 + lane) * 4);
    bh[nt][0] = b4.x; bh[nt][1] = b4.y; bl[nt][0] = b4.z; bl[nt][1] = b4.w;
  }
#pragma unroll
  for (int nt = 0; nt < NKS; ++nt)
#pragma unroll
    for (int tl = 0; tl < 2; ++tl) mma_tf32(acc[tl][nt], al[tl], bh[nt]);
#pragma unroll
  for (int nt = 0; nt < NKS; ++nt)
#pragma unroll
    for (int tl = 0; tl < 2; ++tl) mma_tf32(acc[tl][nt], ah[tl], bl[nt]);
#pragma unroll
  for (int nt = 0; nt < NKS; ++nt)
#pragma unroll
    for (int tl = 0; tl < 2; ++tl) mma_tf32(acc[tl][nt], ah[tl], bh[nt]);
}

// Same contract as expansor_warp.  Rows of the MMA tiles = map columns: a round covers 32 columns (two 16-row tiles);
// lane = 4 g + q owns rows g and g + 8 of each tile.
template <int N, int NCOLS, class OFN, class STORE>
CG_DEV void expansor_mma_warp(const float* f1_, const float* f2_, const float* b0, float a0, OFN o_at, STORE store) {
  constexpr int NKS = (N + 7) / 8;
  const int lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3;
#pragma unroll 1
  for (int c0 = 0; c0 < NCOLS; c0 += 32) {
    bool active[4];
    int col[4];                                           // tile tl: rows g -> col[2 tl], g + 8 -> col[2 tl + 1]
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      active[u] = c0 + 8 * u + g < NCOLS;
      col[u] = active[u] ? c0 + 8 * u + g : NCOLS - 1;
    }
    const int oz = opaque_zero();                       // the fragment images are re-read every round, not hoisted out of it
    const float* f1 = f1_ + oz;
    const float* f2 = f2_ + oz;
    float acc[2][NKS][4];
#pragma unroll
    for (int tl = 0; tl < 2; ++tl)
#pragma unroll
      for (int nt = 0; nt < NKS; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[tl][nt][e] = 0.f;
    // ---- layer 1: hidden[col][j] = sum_k o[k][col] W0[j][k]; the A fragment is the outer-product map itself
#pragma unroll
    for (int kt = 0; kt < NKS; ++kt) {
      const int k0 = 8 * kt + q, k1 = k0 + 4;
      float ah[2][4], al[2][4];
#pragma unroll
      for (int tl = 0; tl < 2; ++tl) {
        const float o0 = k0 < N ? o_at(k0, col[2 * tl]) : 0.f, o1 = k0 < N ? o_at(k0, col[2 * tl + 1]) : 0.f;
        const float o2 = k1 < N ? o_at(k1, col[2 * tl]) : 0.f, o3 = k1 < N ? o_at(k1, col[2 * tl + 1]) : 0.f;
        tf32_split(o0, ah[tl][0], al[tl][0]); tf32_split(o1, ah[tl][1], al[tl][1]);
        tf32_split(o2, ah[tl][2], al[tl][2]); tf32_split(o3, ah[tl][3], al[tl][3]);
      }
      expansor_mma_step<NKS>(acc, ah, al, f1, kt);
    }
    // ---- layer 2: out[col][m] = sum_j PReLU(hidden[col][j] + b0[j]) W4[m][j]; accumulator tile jt -> A fragment of k step jt
    float out[2][NKS][4];
#pragma unroll
    for (int tl = 0; tl < 2; ++tl)
#pragma unroll
      for (int nt = 0; nt < NKS; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) out[tl][nt][e] = 0.f;
#pragma unroll
    for (int jt = 0; jt < NKS; ++jt) {
      const int j0 = 8 * jt + 2 * q;
      const float bj0 = b0[j0 < N ? j0 : N - 1], bj1 = b0[j0 + 1 < N ? j0 + 1 : N - 1];   // padded hidden units meet zero weights
      float ah[2][4], al[2][4];
#pragma unroll
      for (int tl = 0; tl < 2; ++tl) {
        // accumulator: [0] = (row g, hidden j0), [1] = (g, j0 + 1), [2] = (g + 8, j0), [3] = (g + 8, j0 + 1)
        // A fragment:  [0] = (row g, slot q), [1] = (g + 8, slot q), [2] = (g, slot q + 4), [3] = (g + 8, slot q + 4)
        tf32_split(prelu(acc[tl][jt][0] + bj0, a0), ah[tl][0], al[tl][0]);
        tf32_split(prelu(acc[tl][jt][2] + bj0, a0), ah[tl][1], al[tl][1]);
        tf32_split(prelu(acc[tl][jt][1] + bj1, a0), ah[tl][2], al[tl][2]);
        tf32_split(prelu(acc[tl][jt][3] + bj1, a0), ah[tl][3], al[tl][3]);
      }
      expansor_mma_step<NKS>(out, ah, al, f2, jt);
    }
    // ---- store: out[tl][mt]: [0] = (col[2 tl], m0), [1] = (col[2 tl], m0 + 1), [2] = (col[2 tl + 1], m0), [3] = (col[2 tl + 1], m0 + 1)
#pragma unroll
    for (int mt = 0; mt < NKS; ++mt) {
      const int m0 = 8 * mt + 2 * q;
#pragma unroll
      for (int tl = 0; tl < 2; ++tl) {
        if (m0 < N) {
          if (active[2 * tl]) store(m0, col[2 * tl], out[tl][mt][0]);
          if (active[2 * tl + 1]) store(m0, col[2 * tl + 1], out[tl][mt][2]);
        }
        if (m0 + 1 < N) {
          if (active[2 * tl]) store(m0 + 1, col[2 * tl], out[tl][mt][1]);
          if (active[2 * tl + 1]) store(m0 + 1, col[2 * tl + 1], out[tl][mt][3]);
        }
      }
    }
  }
}

// y[m] = sum_k W[k][m] * x[k] for the lane's output column m (clamped by the caller); x broadcast from shared memory.
CG_DEV float warp_col_dot(const float* __restrict__ wcol, int Mp, int K, const float* x) {
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  int k = 0;
#pragma unroll 2
  for (; k + 4 <= K; k += 4) {
    const float4 xv = *reinterpret_cast<const float4*>(x + k);
    a0 = fmaf(wcol[(k + 0) * Mp], xv.x, a0);
    a1 = fmaf(wcol[(k + 1) * Mp], xv.y, a1);
    a2 = fmaf(wcol[(k + 2) * Mp], xv.z, a2);
    a3 = fmaf(wcol[(k + 3) * Mp], xv.w, a3);
  }
  for (; k < K; ++k) a0 = fmaf(wcol[k * Mp], x[k], a0);
  return (a0 + a1) + (a2 + a3);
}

template <int T, int V, bool MMA>
__global__ void __launch_bounds__(32 * (MMA ? ADJ_MMA_MAX_WARPS : ADJ_MAX_WARPS), 1) dstd_adj_kernel(const AdjArgs a) {
  CG_DYN_SMEM(smem);
  constexpr int TV = T * V, TT = T * T, VV = V * V;
  constexpr int TP = (T + 3) & ~3, VQ = (V + 3) & ~3;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nthreads = blockDim.x;
  const int* d = a.d;
  const int Co = d[CB_CO], Ch = d[CB_CH], Cg = d[CB_CG];
  const bool interp = d[CB_INTERP] != 0;
  const int Cop = apad8(Co);
  const RedLayout RL(T, V, Cg, Ch, interp);
  const float* __restrict__ W = a.w;

  for (int f = 0; f < CB_COUNT; ++f)
    if (a.res[f] >= 0)
      for (int i = threadIdx.x; i < a.wsz[f]; i += nthreads) smem[a.res[f] + i] = __ldg(W + d[f] + i);
  if constexpr (MMA) {
    build_expansor_frags<V>(smem + a.o_f1[0], smem + a.o_f2[0], W + d[CB_E0_WT_S], W + d[CB_E4N_WT_S], nthreads);
    build_expansor_frags<T>(smem + a.o_f1[1], smem + a.o_f2[1], W + d[CB_E0_WT_T], W + d[CB_E4N_WT_T], nthreads);
  }
  __syncthreads();
  // MMA variant: the plan guarantees every field resident, so the pointers are provably shared-memory pointers (LDS with
  // 32-bit address arithmetic; the either-or form compiles to generic loads, ~8 instead of ~3 instructions per weight)
  auto P = [&](int f) -> const float* {
    if constexpr (MMA) return smem + a.res[f];
    else return a.res[f] >= 0 ? smem + a.res[f] : W + d[f];
  };

  float* rr = smem + a.o_warp + warp * a.warp_floats;      // the sample's red record
  float* dseq = rr + RL.stats;                             // [2][T][V]   dim_seq of both domains (aliases the gate inputs)
  float* dsp = dseq + 2 * rpad4(TV);                       // [2][V][T]   dim_space
  const int Co4 = rpad4(Co);                               // per-gate stride of the small vectors (16-byte aligned rows)
  float* h2 = rr + imax_(rpad4(RL.total), interp ? RL.stats + 4 * rpad4(TV) : 0);       // [2][Co4]
  float* zz = h2 + 2 * Co4;                                // [2][Co4]
  const int oc = lane < Co ? lane : Co - 1;

  for (int b = blockIdx.x * a.nwarps + warp; warp < a.nwarps && b < a.batch; b += gridDim.x * a.nwarps) {
    {
      const float4* src = reinterpret_cast<const float4*>(a.red + (size_t)b * a.red_stride);
      for (int i = lane; i < RL.total / 4; i += 32) reinterpret_cast<float4*>(rr)[i] = __ldg(src + i);
    }
    __syncwarp();
    // ---------------- gate conv (1,V) + BN + PReLU -> h2 (:327-330), lanes = output channels
    {
      const float* w4 = P(CB_G4_WT);
      const float* b4 = P(CB_G4_B);
      const float* a4 = P(CB_G4_A);
      const int K = Cg * V;
#pragma unroll 1
      for (int g = 0; g < 2; ++g) {
        const float acc = warp_col_dot(w4 + (size_t)g * K * Cop + oc, Cop, K, rr + RL.h1 + g * RL.h1g);
        if (lane < Co) h2[g * Co4 + lane] = prelu(acc + b4[g * Co + lane], a4[g]);
      }
    }
    __syncwarp();
    // ---------------- gate MLP: Linear(Co + 2 + 2T -> Co) + BN + PReLU, Linear(Co -> Co)  (:341-352, 378-384)
    {
      const float* m0 = P(CB_M0_WT);
      const float* m0b = P(CB_M0_B);
      const float* m0a = P(CB_M0_A);
      const float* m4 = P(CB_M4_WT);
      const int NS = 2 + 2 * T;
#pragma unroll 1
      for (int g = 0; g < 2; ++g) {
        const float* w0 = m0 + (size_t)g * (Co + NS) * Cop + oc;
        float acc = warp_col_dot(w0, Cop, Co, h2 + g * Co4);
        acc += warp_col_dot(w0 + (size_t)Co * Cop, Cop, NS, rr + RL.stats);
        if (lane < Co) zz[g * Co4 + lane] = prelu(acc + m0b[g * Co + lane], m0a[g]);
      }
      __syncwarp();
#pragma unroll 1
      for (int g = 0; g < 2; ++g) {
        const float acc = warp_col_dot(m4 + (size_t)g * Co * Cop + oc, Cop, Co, zz + g * Co4);
        if (lane < Co) {
          a.wg[((size_t)b * 2 + g) * Co + lane] = acc;
          float* tp = g == 0 ? a.tap_w1 : a.tap_w2;
          if (tp) tp[(size_t)b * Co + lane] = acc;
        }
      }
    }
    if (interp) {
      // ---------------- dim_seq / dim_space: last 1x1 of each compress branch (:144, :152); lanes = joints
#pragma unroll 1
      for (int L = 0; L < 2; ++L) {
        const float* w6 = P(CB_TC6_WT_S + L);              // [Ch][pad8(T)]
        const float* wj = P(CB_JC6_WT_S + L);              // [Ch][pad8(V)]
        const float* tcv = rr + RL.tc + L * Ch * V;        // [Ch][V]
        const float* jcv = rr + RL.jc + L * Ch * T;        // [Ch][T]
        const int vl = lane < V ? lane : V - 1;
        float s[T], p[T];
#pragma unroll
        for (int t = 0; t < T; ++t) { s[t] = 0.f; p[t] = 0.f; }
#pragma unroll 2
        for (int o = 0; o < Ch; ++o) {
          const float xv = tcv[o * V + vl];                // dim_seq[t'][v] = sum_o W6[o][t'] * tc[o][v]
          const float wv = wj[o * apad8(V) + vl];          // dim_space[v'][t] = sum_o Wj6[o][v'] * jc[o][t]
#pragma unroll
          for (int t = 0; t < T; ++t) {
            s[t] = fmaf(w6[o * apad8(T) + t], xv, s[t]);
            p[t] = fmaf(wv, jcv[o * T + t], p[t]);
          }
        }
        if (lane < V) {
#pragma unroll
          for (int t = 0; t < T; ++t) { dseq[L * rpad4(TV) + t * V + lane] = s[t]; dsp[L * rpad4(TV) + lane * T + t] = p[t]; }
        }
      }
      __syncwarp();
      // ---------------- space domain: o[v'][t][q] = dsp[v'][t] * dseq[q][v'] (:155-158, 187), expansor over the joint axis
      {
        float* out = a.adj_s + (size_t)b * V * TT;
        const float* ds = dseq;
        const float* dp = dsp;
        auto o_at = [&](int k, int col) { const int t = col / T, q = col - t * T; return dp[k * T + t] * ds[q * V + k]; };
        auto store = [&](int m, int col, float val) { out[m * TT + col] = val; };
        if constexpr (MMA) expansor_mma_warp<V, TT>(smem + a.o_f1[0], smem + a.o_f2[0], P(CB_E0_B_S), P(CB_E0_A_S)[0], o_at, store);
        else expansor_warp<V, TT, ADJ_CPL>(P(CB_E0_WT_S), P(CB_E0_B_S), P(CB_E0_A_S)[0], P(CB_E4N_WT_S), o_at, store);
      }
      // ---------------- time domain: o[t'][v][w] = dsp[v][t'] * dseq[t'][w] (:159-162, 187), expansor over the frame axis
      {
        float* out = a.adj_t + (size_t)b * T * VV;
        const float* ds = dseq + rpad4(TV);
        const float* dp = dsp + rpad4(TV);
        auto o_at = [&](int k, int col) { const int v = col / V, w = col - v * V; return dp[v * T + k] * ds[k * V + w]; };
        auto store = [&](int m, int col, float val) { out[m * VV + col] = val; };
        if constexpr (MMA) expansor_mma_warp<T, VV>(smem + a.o_f1[1], smem + a.o_f2[1], P(CB_E0_B_T), P(CB_E0_A_T)[0], o_at, store);
        else expansor_warp<T, VV, ADJ_CPL>(P(CB_E0_WT_T), P(CB_E0_B_T), P(CB_E0_A_T)[0], P(CB_E4N_WT_T), o_at, store);
      }
    }
    __syncwarp();
  }
  (void)TP; (void)VQ;
}

template <int T, int V>
int launch_adj_impl(const AdjArgs& a, void* stream) {
  if (a.mma) return launch_warp_per_sample(dstd_adj_kernel<T, V, true>, a, stream);
  return launch_warp_per_sample(dstd_adj_kernel<T, V, false>, a, stream);
}

}  // namespace cg
