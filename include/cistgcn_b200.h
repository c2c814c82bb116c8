/*
 * cistgcn_b200 -- C-ABI of the B200-native CIST-GCN forward path.
 *
 * Plain C: pointers, sizes and int32 descriptor arrays only (no torch / C++ types).  Every
 * buffer (packed weights, activations, workspace) is allocated and owned by the caller on the
 * device the call runs on; `stream` is a cudaStream_t passed as void*.  All entry points
 * return 0 on success and a negative code on error; cistgcn_last_error() returns the message of
 * the last failing call on the calling thread (thread-local).  Kernel choices travel with the call
 * (CP_FLAGS in the plan, `flags` arguments): calls from different host threads on distinct streams,
 * workspaces and outputs are independent.  The only process-wide state is instrumentation: the
 * optional launch timer (cistgcn_profile_*, mutex-protected) and, in -DCISTGCN_PROFILE builds only,
 * the phase-clock debug hooks.
 *
 * What each entry point replaces in the reference (QualityMinds/cistgcn, paths relative to
 * human_motion_prediction/):
 *   cistgcn_forward_f32 /    models/CISTGCN/CISTGCN.py:567-597  CISTGCN.forward, called from
 *   cistgcn_forward_bf16
 *                            environment/train.py:59 and environment/test.py:101,103
 *                            (+ losses/losses.py:50-61 mpjpe when `target` is given)
 *   cistgcn_rollout_f32 /    no counterpart: the autoregressive loop a caller writes around CISTGCN.forward to reach
 *   cistgcn_rollout_bf16     horizons past output_n (+ losses.mpjpe over the whole horizon when `target` is given)
 *   cistgcn_dstd_block_f32   models/CISTGCN/CISTGCN.py:373-390  DSTD_GC.forward (one block)
 *   cistgcn_fpn_chain_f32    models/CISTGCN/CISTGCN.py:582-589  FPN stack + dim_conversor + cumsum
 *   cistgcn_tail_f32         models/CISTGCN/CISTGCN.py:591-597  ContextLayer + output assembly
 *   cistgcn_mpjpe_f32        losses/losses.py:50-61             mpjpe (all three reduce_axis modes)
 *   cistgcn_mpjpe_grouped_f32  the same per-frame sums split by a per-sample group id (one row per action / sub-dataset)
 *
 * Descriptors are flat int32 arrays indexed by the enums below.  Weight fields are offsets (in
 * floats) into the packed weight blob produced by cistgcn_b200/pack.py (BatchNorm folded,
 * matrices stored k-major with the output dimension padded to a multiple of CISTGCN_MPAD).
 */
#ifndef CISTGCN_B200_H
#define CISTGCN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CISTGCN_ABI_VERSION 6
#define CISTGCN_MPAD 8          /* output-dimension padding of every k-major matrix */
#define CISTGCN_MAX_BLOCKS 8    /* input + output DSTD-GC blocks in one plan */
#define CISTGCN_MAX_FPN 8
#define CISTGCN_PROFILE_KINDS 8  /* 0 fused DSTD-GC block, 1 FPN chain, 2 context+assembly, 3 mpjpe,
                                    4 DSTD reduce stage, 5 DSTD adjacency stage, 6 DSTD mix stage, 7 other */

/* kernel-choice flags (CP_FLAGS of a plan; `flags` of the per-stage entry points); 0 = defaults */
#define CISTGCN_FLAG_FPN_FP32   1  /* FPN stack on the FP32-FMA kernel (csrc/fpn_chain.cuh) instead of tcgen05 (csrc/fpn_tc.cuh) */
#define CISTGCN_FLAG_DSTD_FUSED 2  /* DSTD-GC blocks on the round-1 fused one-CTA-per-sample kernel (csrc/dstd_block.cuh) instead
                                      of the three-stage reduce / adjacency / mix kernels */
#define CISTGCN_FLAG_DSTD_TC    4  /* with DSTD_FUSED: channel mixes as tcgen05 MMAs where the shared-memory plan fits */
#define CISTGCN_FLAG_DSTD_MIX_FFMA 8  /* three-stage path: channel mixes of stage 3 on the FP32-FMA tile loops (csrc/dstd_mix.cuh)
                                        instead of 3xTF32 mma.sync (csrc/dstd_mix_mma.cuh, the default where Ci, Co <= 32) and of the
                                        warp-per-sample streaming kernel of the 3 -> 3 output block (csrc/dstd_mix_narrow.cuh) */
#define CISTGCN_FLAG_DSTD_ADJ_FFMA 16 /* three-stage path: Map2Adj expansor of stage 2 on the FP32-FMA column loops instead of
                                        the chained 3xTF32 mma.sync GEMMs (csrc/dstd_adj.cuh, the default) */
#define CISTGCN_FLAG_DSTD_REDUCE_FFMA 32 /* three-stage path: stacked 1x1 convolutions of stage 1 (Map2Adj entry maps, gate conv) on
                                        the FP32-FMA lane-per-channel loops instead of 3xTF32 mma.sync (csrc/dstd_reduce.cuh) */

/* ---- one DSTD-GC block (CISTGCN.py:273-390).  *_S/_T pairs: index +0 = dsgn ("space" domain,
 *      TxT adjacency per joint), +1 = tsgn ("time" domain, VxV adjacency per frame). ---------- */
enum cistgcn_block_field {
  CB_CI = 0,      /* input channels */
  CB_CO,          /* output channels */
  CB_T,           /* length of the block's "time" axis  (10; V for the output block) */
  CB_V,           /* length of the block's "joint" axis (V; output_n, 25 or 10, for the output block) */
  CB_CH,          /* Map2Adj inter channels = Ci/2            (CISTGCN.py:137) */
  CB_CG,          /* gate inter channels = max(Co/2,1)        (CISTGCN.py:321) */
  CB_HS,          /* SE hidden width = max(Co/reduction,1)    (SE.py:28-29)    */
  CB_HAS_RES,     /* 1 when Ci != Co: residual paths are conv1x1+BN (CISTGCN.py:239-247,310-318) */
  CB_INTERP,      /* 1: adjacency generated per sample by Map2Adj; 0: static A parameters */
  CB_IN_MODE,     /* 0: activation tensor with the strides below; 1: raw poses (T,V,3) -> 10 features */
  CB_IN_SB, CB_IN_SC, CB_IN_ST, CB_IN_SV,      /* input strides in floats: sample, c, t, v */
  CB_OUT_SB, CB_OUT_SC, CB_OUT_ST, CB_OUT_SV,  /* output strides */
  CB_GN_S, CB_GN_B,                 /* global_norm folded scale / shift               [Ci]        */
  CB_G0_WT, CB_G0_B, CB_G0_A,       /* conv_{s,t}.0 stacked: [Ci*T][pad(2Cg)], [2Cg], slopes [2]  */
  CB_G4_WT, CB_G4_B, CB_G4_A,       /* conv_{s,t}.4: 2 x [Cg*V][pad(Co)], [2][Co], slopes [2]     */
  CB_M0_WT, CB_M0_B, CB_M0_A,       /* map_{s,t}.0:  2 x [Co+2+2T][pad(Co)], [2][Co], slopes [2]  */
  CB_M4_WT,                         /* map_{s,t}.4:  2 x [Co][pad(Co)]                            */
  CB_A0_WT, CB_A0_B, CB_A0_A,       /* Map2Adj first 1x1 convs stacked (dsgn.tc, dsgn.jc, tsgn.tc, tsgn.jc):
                                       [Ci][pad(4Ch)], [4Ch], slopes [4] */
  CB_TC3_WT_S, CB_TC3_WT_T,         /* time_compress.3 (+BN .4):  [Ch*T][pad(Ch)] */
  CB_TC3_B_S, CB_TC3_B_T,           /* [Ch] */
  CB_TC6_WT_S, CB_TC6_WT_T,         /* time_compress.6:           [Ch][pad(T)]   */
  CB_JC3_WT_S, CB_JC3_WT_T,         /* joint_compress.3 (+BN .4): [Ch*V][pad(Ch)] */
  CB_JC3_B_S, CB_JC3_B_T,
  CB_JC6_WT_S, CB_JC6_WT_T,         /* joint_compress.6:          [Ch][pad(V)]   */
  CB_E0_WT_S, CB_E0_WT_T,           /* expansor.0 (+BN .1): [n][pad(n)], n = V (dsgn) / T (tsgn) */
  CB_E0_B_S, CB_E0_B_T,
  CB_E0_A_S, CB_E0_A_T,             /* expansor.3 PReLU slope */
  CB_E4_WT_S, CB_E4_WT_T,           /* expansor.4: [n][pad(n)] */
  CB_ADJ_S, CB_ADJ_T,               /* static adjacency gcn.A: (V,T,T) / (T,V,V); used when !INTERP */
  CB_TCN_WT_S, CB_TCN_WT_T,         /* tcn.0 (+BN .1) [Ci (+Ci residual rows when HAS_RES)][pad(Co)] */
  CB_TCN_B_S, CB_TCN_B_T,           /* combined bias [Co] */
  CB_TCN_A_S, CB_TCN_A_T,           /* Domain_GCNN_layer.prelu slope */
  CB_P_S_S, CB_P_S_T,               /* prelu{1,2}.0 BN scale [Co] */
  CB_P_B_S, CB_P_B_T,               /* prelu{1,2}.0 BN shift [Co] */
  CB_P_A_S, CB_P_A_T,               /* prelu{1,2}.1 slope */
  CB_CP_WT, CB_CP_B, CB_CP_A,       /* compressor.0 (+BN .1): [2Co][pad(Co)], [Co], slope */
  CB_SE1_WT, CB_SE2_WT,             /* compressor.3.excitation.{0,2}: [Co][pad(Hs)], [Hs][pad(Co)] */
  CB_RS_WT, CB_RS_B,                /* block residual conv (+BN): [Ci][pad(Co)], [Co]  (HAS_RES only) */
  /* tcgen05 operand images of the channel-mixing 1x1 convolutions (csrc/dstd_block.cuh, tc_gemm), 0 = absent:
   * [K/8 k-chunks][4*Np rows][8 x 16 bit], rows j*Np + m = bf16 term j of output channel m (j = 0,1,2), rows 3*Np + m =
   * its fp16 rounding; Np = pad16(outputs); K = the same row blocks as the fp32 matrix, each padded to 16 */
  CB_TC_A0,                         /* Map2Adj first 1x1 convs stacked (4*Ch outputs, K = Ci) */
  CB_TC_TCN_S, CB_TC_TCN_T,         /* tcn.0 (+BN) [+ residual conv rows]  (Co outputs, K = Ci [+ Ci]) */
  CB_TC_CP,                         /* compressor.0 (+BN)  (Co outputs, K = Co + Co) */
  CB_TC_RS,                         /* block residual conv (+BN)  (Co outputs, K = Ci; HAS_RES only) */
  /* operands of the reduce stage (csrc/dstd_reduce.cuh): rows padded to 32 outputs so that lane = output channel */
  CB_R_A0_WT, CB_R_A0_B,            /* Map2Adj first 1x1 convs stacked: [Ci][pad32(4Ch)], bias [pad32(4Ch)] */
  CB_R_G0_WT, CB_R_G0_B,            /* conv_{s,t}.0 stacked: [Ci*T][pad32(2Cg)] (row c*T + t), bias [pad32(2Cg)] */
  CB_R_TC3_WT, CB_R_TC3_B,          /* time_compress.3 of dsgn | tsgn side by side: [Ch*T][pad32(2Ch)] (row c*T + t), bias */
  CB_R_JC3_WT, CB_R_JC3_B,          /* joint_compress.3 of dsgn | tsgn side by side: [Ch*V][pad32(2Ch)] (row c*V + v), bias */
  /* operand of the adjacency stage (csrc/dstd_adj.cuh): expansor.4 row-major (output row, inputs padded to 8) */
  CB_E4N_WT_S, CB_E4N_WT_T,         /* [n][pad(n)], n = V (dsgn) / T (tsgn) */
  CB_COUNT
};

/* ---- one FPN layer (CISTGCN.py:38-79) + the caller's PReLU / residual (:584-586) ------------ */
enum cistgcn_fpn_field {
  CF_CIN = 0,     /* input channels (= frames): input_n for layer 0, output_n afterwards */
  CF_COUT,        /* output_n (25 or 10) */
  CF_RESID,       /* 1: x6 = PReLU(FPN(x6)) + x6 (layers >= 1) */
  CF_W_D1, CF_W_D2, CF_W_D3,   /* block{1,2,3}.0 (+BN .1): [Cin][3][5 otiles][16] (kw-major, 5 outs, 1 pad) */
  CF_B_D1, CF_B_D2, CF_B_D3,   /* folded bias [Cout] */
  CF_A_D1, CF_A_D2, CF_A_D3,   /* block{1,2,3}.3 slope */
  CF_CP_WT,       /* compress weights for the 3*Cout branch channels: [3*Cout][pad(Cout)] */
  CF_CP_AVG_WT,   /* compress weights for the Cin global-average channels: [Cin][pad(Cout)] */
  CF_CP_B,        /* compress bias [Cout] */
  CF_OUT_A,       /* prelus.{i} slope */
  /* tensor-core (tcgen05) image of the same layer, see csrc/fpn_tc.cuh.  Weights are split into three bf16
   * terms (w = w1 + w2 + w3 to 24 bits) so that fp32 accuracy survives the bf16 tensor pipe. */
  CF_TC_KC,       /* 16-byte k-chunks (8 input channels each) per kernel tap: pad16(Cin) / 8 */
  CF_TC_W,        /* 3 branches x { 9 tap slices [KC][96][8 bf16], 1 compress slice [4][96][8 bf16] }; row = 32*term + cout */
  CF_TC_PRM,      /* fp32: bias[3][32], slope[3], out slope, compress bias[32], avg-branch weights [32 cin][32 cout] */
  CF_TC_W16,      /* bf16-only image for cistgcn_forward_bf16: same slices, [KC][32][8 bf16] (row = cout), 4 chunks for compress */
  CF_COUNT
};

/* ---- FPN chain + dim_conversor + cumsum, ContextLayer, output assembly ---------------------- */
enum cistgcn_tail_field {
  CT_TIN = 0,     /* input_n  */
  CT_TOUT,        /* output_n */
  CT_V,           /* joints   */
  CT_F,           /* feature channels leaving the input block stack (in_ch = 10, CISTGCN.py:512) */
  CT_HID,         /* ContextLayer hidden_dim (64) */
  CT_SEH1,        /* SELayer1d hidden = Tout / reduction      (SE.py:10)    */
  CT_SEH2,        /* SELayer2d hidden = max(Tout/reduction,1) (SE.py:28-29) */
  CT_DC0_WT, CT_DC0_B, CT_DC0_A,    /* dim_conversor.0 (+BN .1): [F][pad(3)], [3], slope */
  CT_DC3_WT, CT_DC3_A,              /* dim_conversor.3: [3][pad(3)]; dim_conversor.4 slopes [3] */
  CT_C1_S, CT_C1_B, CT_C1_A,        /* context_conv1 folded per-channel scale/shift [HID], slope */
  CT_C2_WT, CT_C2_B, CT_C2_A,       /* context_conv2 (+BN): [Tout][pad(HID)], [HID], slope */
  CT_C3_S, CT_C3_B, CT_C3_A,        /* context_conv3 */
  CT_MAP_WT, CT_MAP_A,              /* map{1,2,3}.0: 3 x [HID][pad(Tout)]; slopes [3] */
  CT_FS_WT, CT_FS_B,                /* fmap_s (+BN): [3*Tout][pad(V)], [V] */
  CT_FT_WT, CT_FT_B,                /* fmap_t (+BN): [3*Tout][pad(Tout)], [Tout] */
  CT_N0_WT, CT_N0_B, CT_N0_A,       /* norm_map.0 (+BN .1): [Tout][pad(Tout)], [Tout], slope (.3) */
  CT_NSE1_WT, CT_NSE2_WT,           /* norm_map.4.excitation.{0,2}: [Tout][pad(SEH1)], [SEH1][pad(Tout)] */
  CT_N5_WT, CT_N5_B, CT_N5_A,       /* norm_map.5 (+BN .6), slope (.8) */
  CT_FC0_S, CT_FC0_B, CT_FC0_A,     /* fconv.0 (+BN .1): per-dim scale/shift [3], slope */
  CT_FC3_WT, CT_FC3_B, CT_FC3_A,    /* fconv.3 (+BN .4): [3][pad(3)], [3], slope */
  CT_SE1_WT, CT_SE2_WT,             /* SE.excitation.{0,2}: [Tout][pad(SEH2)], [SEH2][pad(Tout)] */
  CT_COUNT
};

/* ---- whole-model plan: header, then the block / FPN / tail descriptors back to back --------- */
enum cistgcn_plan_field {
  CP_ABI = 0,     /* must equal CISTGCN_ABI_VERSION */
  CP_TIN, CP_TOUT, CP_V,
  CP_N_IN_BLOCKS, /* DSTD-GC blocks before the FPN stack (5) */
  CP_N_FPN,       /* FPN layers (4) */
  CP_N_OUT_BLOCKS,/* DSTD-GC blocks after the ContextLayer (1) */
  CP_CMAX,        /* widest channel count of any inter-block activation */
  CP_WEIGHT_FLOATS, /* size of the packed weight blob, for bounds checking */
  CP_FLAGS,       /* CISTGCN_FLAG_* kernel choices for this plan (0 = defaults) */
  CP_HEADER_COUNT
};
/* plan layout: [CP_HEADER_COUNT] [n_in x CB_COUNT] [n_fpn x CF_COUNT] [CT_COUNT] [n_out x CB_COUNT] */

/* Optional interpretability outputs (environment/test.py:146-157 reads them off the module).
 * Any pointer may be NULL.  Shapes per sample: adj_s (V,T,T), adj_t (T,V,V), w1/w2 (Co). */
typedef struct cistgcn_block_taps {
  float* adj_s;
  float* adj_t;
  float* w1;
  float* w2;
} cistgcn_block_taps;

typedef struct cistgcn_taps {
  cistgcn_block_taps in_blocks[CISTGCN_MAX_BLOCKS];
  cistgcn_block_taps out_blocks[CISTGCN_MAX_BLOCKS];
  float* ctx_joints;          /* (B, V)          context_layer.joints          */
  float* ctx_displacements;   /* (B, Tout)       context_layer.displacements   */
  float* ctx_seq_joints_n;    /* (B, Tout, V)    context_layer.seq_joints_n    */
  float* ctx_seq_joints_dims; /* (B, 3, Tout, V) context_layer.seq_joints_dims */
} cistgcn_taps;

const char* cistgcn_last_error(void);
int cistgcn_abi_version(void);

/* Bytes of scratch the forward needs for `batch` samples (it chunks internally above
 * CISTGCN_MAX_CHUNK samples, so this saturates). */
size_t cistgcn_workspace_bytes(const int32_t* plan, int64_t batch);

/* Full forward.  x: (B, Tin, V, 3) fp32 contiguous; pred: (B, Tout, V, 3).
 * target (optional, same shape as pred) + frame_sums (optional, double[Tout], ACCUMULATED into:
 * the caller zeroes it): sum over samples and joints of ||pred - target||_2 per output frame, from
 * which mpjpe's `[]` and `(0,2)` reductions follow by dividing by B*V*Tout resp. B*V. */
int cistgcn_forward_f32(const int32_t* plan, int32_t plan_len, const float* weights,
                        const float* x, float* pred, const float* target, double* frame_sums,
                        void* workspace, size_t workspace_bytes, int64_t batch,
                        const cistgcn_taps* taps, void* stream);

/* Same call with bf16 STORAGE and bf16 tensor-core operands where the path is a dense GEMM (BASELINE.json configs[3]):
 * every activation tensor between the kernels of the input block stack and the FPN stack's input are stored as bf16
 * (half the HBM traffic of the widest tensors); the FPN stack's convolutions run as single-term bf16 tcgen05 MMAs with
 * fp32 accumulation (one MMA per k-step instead of the two split-operand ones of the fp32 path); the per-sample vector
 * math (statistics, gates, adjacency generation, squeeze-excitation) and x / pred / x7 / x8 stay fp32.
 * Stated bound against the fp32 reference on unit-scale inputs: max-abs <= 3e-2 on the predicted coordinates, MPJPE
 * agreement <= 5e-3 (tests/test_bf16_forward.py).  Needs the tcgen05 FPN kernel (joints 22 / 18). */
int cistgcn_forward_bf16(const int32_t* plan, int32_t plan_len, const float* weights,
                         const float* x, float* pred, const float* target, double* frame_sums,
                         void* workspace, size_t workspace_bytes, int64_t batch,
                         const cistgcn_taps* taps, void* stream);

/* Autoregressive rollout to `horizon` >= 1 frames: K = ceil(horizon / Tout) forwards per chunk of CISTGCN_MAX_CHUNK
 * samples, back to back on `stream` (no host synchronisation).  Step 0 reads x (B, Tin, V, 3); step k + 1 reads the last
 * Tin frames of step k's prediction p_k (Tin <= Tout, so exactly p_k[:, Tout - Tin:]).  out (B, horizon, V, 3):
 * p_0, ..., p_{K-1} concatenated along the frames and cut to `horizon`, bit-identical to the same loop over
 * cistgcn_forward_f32 (_bf16) at the same batch size.  target (optional, same shape as out) + frame_sums (optional, double[horizon], ACCUMULATED into):
 * per-frame sums of ||out - target||_2 as in cistgcn_forward_f32.  No taps.  Unsupported shapes fail as in the
 * forward, before anything is written.  The workspace is the forward's plus one window and one step prediction per
 * chunk: cistgcn_rollout_workspace_bytes(plan, batch) bytes. */
size_t cistgcn_rollout_workspace_bytes(const int32_t* plan, int64_t batch);
int cistgcn_rollout_f32(const int32_t* plan, int32_t plan_len, const float* weights, const float* x,
                        int32_t horizon, float* out, const float* target, double* frame_sums,
                        void* workspace, size_t workspace_bytes, int64_t batch, void* stream);
/* Same with the bf16 activation storage of cistgcn_forward_bf16. */
int cistgcn_rollout_bf16(const int32_t* plan, int32_t plan_len, const float* weights, const float* x,
                         int32_t horizon, float* out, const float* target, double* frame_sums,
                         void* workspace, size_t workspace_bytes, int64_t batch, void* stream);

/* One DSTD-GC block on `batch` samples with the strides in the descriptor.  The three-stage path needs
 * cistgcn_dstd_block_workspace_bytes(desc, batch) bytes of scratch (stage records + gates + adjacencies). */
size_t cistgcn_dstd_block_workspace_bytes(const int32_t* block_desc, int64_t batch);
int cistgcn_dstd_block_f32(const int32_t* block_desc, const float* weights, const float* in,
                           float* out, int64_t batch, const cistgcn_block_taps* taps,
                           void* workspace, size_t workspace_bytes, uint32_t flags, void* stream);

/* FPN stack + dim_conversor + cumsum.  in: (B, Tin, F, V) (frames as channels); out x7: (B, Tout, V, 3). */
int cistgcn_fpn_chain_f32(const int32_t* fpn_descs, int32_t n_fpn, const int32_t* tail_desc,
                          const float* weights, const float* in, float* x7, int64_t batch,
                          uint32_t flags, void* stream);

/* ContextLayer(x7) + output assembly: pred = x[:, -1:] + x8 + act (+ optional MPJPE partial sums). */
int cistgcn_tail_f32(const int32_t* tail_desc, const float* weights, const float* x, const float* x7,
                     const float* x8, float* pred, const float* target, double* frame_sums,
                     int64_t batch, const cistgcn_taps* taps, void* stream);

/* mpjpe: err (optional): (B, T, V) per-joint L2 error; frame_sums (optional): double[T] accumulated. */
int cistgcn_mpjpe_f32(const float* pred, const float* target, int64_t batch, int32_t T, int32_t V,
                      float* err, double* frame_sums, void* stream);

/* Grouped mpjpe for per-group (per action, per sub-dataset) tables in one pass.  pred, target (B, T, V, 3); groups[B]
 * int32 group id of every sample, or NULL = every sample in group 0.  ACCUMULATES into sums[n_groups][T] (double: sum over
 * the group's samples and the joints of ||pred - target||_2 per frame, the scheme of cistgcn_mpjpe_f32) and counts[n_groups]
 * (int64: samples).  Group g's per-frame MPJPE is sums[g] / (counts[g] * V).  A sample whose id is outside [0, n_groups)
 * is skipped and not counted; nothing outside sums / counts is written.  -1: NULL pred / target / sums / counts,
 * n_groups < 1, T < 1, V < 1, negative batch; batch 0 is a no-op.  Timed under the profile kind "mpjpe_kernel". */
int cistgcn_mpjpe_grouped_f32(const float* pred, const float* target, const int32_t* groups, int32_t n_groups,
                              int64_t batch, int32_t T, int32_t V, double* sums, int64_t* counts, void* stream);

/* Fused evaluation metrics (environment/test.py:65-94 Metrics.compute, :125-129 the scatter of the model's joints into the
 * full skeleton).  pred (B, To, Vu, 3) = model output on the used joints; target (B, To, Vf, 3) = full skeleton;
 * src_map[Vf]: index into pred's joints or -1 (keep the target's joint: dim_used / dim_repeat_32 <- dim_repeat_22 of
 * loaders/h36m_motion_3d.py:55-59 folded into one table).  One kernel accumulates, for every output frame, the sum over
 * samples and joints of each metric below into sums[metric][To] (double, ACCUMULATED into; divide by B*Vf -- bones: B*n_bones
 * -- for the reference's reduce_axis=(0, 2) values); `assembled` (optional) receives the scattered prediction. */
enum cistgcn_metric {
  CISTGCN_METRIC_MPJPE = 0,     /* losses.mpjpe                 losses/losses.py:50-61   */
  CISTGCN_METRIC_PA_MPJPE,      /* losses.pa_mpjpe (Procrustes) losses/losses.py:79-144  */
  CISTGCN_METRIC_N_MPJPE,       /* losses.n_mpjpe               losses/losses.py:147-161 */
  CISTGCN_METRIC_VELOCITY,      /* losses.mean_velocity_error   losses/losses.py:164-179 (frames 0 .. To-2) */
  CISTGCN_METRIC_BONE_LENGTH,   /* losses.bone_length_error     losses/losses.py:200-215 */
  CISTGCN_METRIC_WEIGHTED0,     /* losses.weighted_mpjpe with weights0 (B, To, Vf), losses/losses.py:64-77 */
  CISTGCN_METRIC_WEIGHTED1,     /* ... with weights1 */
  CISTGCN_METRIC_COUNT
};
int cistgcn_eval_metrics_f32(const float* pred, const float* target, const int32_t* src_map, const int32_t* bones,
                             int32_t n_bones, const float* weights0, const float* weights1, float* assembled,
                             double* sums, int64_t batch, int32_t To, int32_t Vu, int32_t Vf, void* stream);
/* Grouped form of cistgcn_eval_metrics_f32, with no limit on To (cistgcn_eval_metrics_f32 takes To <= 32).  groups[B]
 * int32 group id of every sample, or NULL = every sample in group 0.  ACCUMULATES into sums[n_groups][CISTGCN_METRIC_COUNT][To]
 * (each group's block means what cistgcn_eval_metrics_f32's sums mean for that group's samples) and counts[n_groups]
 * (int64: samples).  A sample whose id is outside [0, n_groups) is skipped and not counted (its `assembled` rows are still
 * written); nothing outside sums / counts / assembled is written.  -1: NULL pred / target / src_map / sums / counts,
 * n_groups < 1, To < 1, joints out of range, negative batch; batch 0 is a no-op.  Not timed by cistgcn_profile_*, like
 * cistgcn_eval_metrics_f32. */
int cistgcn_eval_metrics_grouped_f32(const float* pred, const float* target, const int32_t* groups, int32_t n_groups,
                                     const int32_t* src_map, const int32_t* bones, int32_t n_bones, const float* weights0,
                                     const float* weights1, float* assembled, double* sums, int64_t* counts,
                                     int64_t batch, int32_t To, int32_t Vu, int32_t Vf, void* stream);

/* GPU-side training-batch pipeline (loaders/h36m_motion_3d.py:94-108 window split + velocity / speed targets;
 * environment/custom_transforms.py:10-419 RandomFlip, RandomRotation, RandomScale, RandomNoise, RandomTranslation in the
 * order loaders/loader.py:42-130 composes them).  windows (N, S, V, 3): the resident dataset; index[B]: the window of every
 * batch element; params (B, CISTGCN_AUG_PARAMS): the host-drawn random parameters (0 = transform does not fire);
 * noise (optional) (B, V, 3): RandomNoise's uniform(-1, 1) draws.  Outputs: sample (B, Tin, V, 3), target (B, S-Tin, V, 3)
 * and (optional) sample_vel, target_vel (cumulated velocities), target_gvel (B, S-Tin, V) (cumulated speeds). */
enum cistgcn_aug_param {
  CISTGCN_AUG_FLIP = 0,      /* [3] 1 = mirror that coordinate about the window's centroid        */
  CISTGCN_AUG_ROT_ON = 3,    /* 1 = rotate about the centroid with ...                            */
  CISTGCN_AUG_ROT = 4,       /* [9] row-major rotation matrix R: x <- (x - c) R + c               */
  CISTGCN_AUG_SCALE_ON = 13,
  CISTGCN_AUG_SCALE = 14,    /* [3] per-coordinate scale                                          */
  CISTGCN_AUG_NOISE = 17,    /* amplitude (0 = off): x <- x + amp * u[joint, k] * (max - min)_k   */
  CISTGCN_AUG_TRANS_ON = 18,
  CISTGCN_AUG_TRANS = 19,    /* [3] translation as a fraction of the window's extent per coordinate */
  CISTGCN_AUG_PARAMS = 24
};
int cistgcn_augment_windows_f32(const float* windows, const int64_t* index, const float* params, const float* noise,
                                float* sample, float* target, float* sample_vel, float* target_vel, float* target_gvel,
                                int64_t batch, int32_t seq_len, int32_t joints, int32_t input_n, void* stream);

/* Optional per-kernel timing for benchmarks (no reference counterpart).  While enabled every launch
 * (of every host thread) is bracketed by CUDA events on its stream; cistgcn_profile_read synchronises
 * the device, sums the elapsed milliseconds and launch counts per kernel kind (arrays of
 * CISTGCN_PROFILE_KINDS) and resets the counters.  Process-wide instrumentation behind a mutex; leave
 * disabled in production. */
int cistgcn_profile_enable(int on);
int cistgcn_profile_read(double* ms_by_kind, int64_t* launches_by_kind);
const char* cistgcn_profile_kind_name(int kind);
/* Debug, -DCISTGCN_PROFILE builds only (otherwise they return -5 and the kernels carry no clock reads):
 * while non-NULL, thread 0 of the first CTA of every fused DSTD-GC / tcgen05 FPN launch stamps clock64() at
 * its phase boundaries into device_buffer (>= 32 x int64).  Process-wide, not thread-safe. */
int cistgcn_debug_phase_clocks(void* device_buffer);
/* Debug: stamp the CTA's `iteration`-th sample instead of its first (0 = cold caches, >= 1 = steady state). */
int cistgcn_debug_stamp_iteration(int iteration);

#ifdef __cplusplus
}
#endif
#endif /* CISTGCN_B200_H */
