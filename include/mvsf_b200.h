/*
 * libmvsf_b200 - C ABI of the B200-native MVSFormer++ depth-inference hot path.
 *
 * The reference (maybeLx/MVSFormerPlusPlus) has no FFI layer: its seams are Python callables
 * (SURVEY.md §8b).  Each entry point below states the reference callable (file:line, relative to the
 * reference repo root) whose arithmetic it replaces.  Conventions:
 *   - every pointer is a DEVICE pointer to fp32 data unless marked "host"; buffers are owned by the
 *     caller and borrowed for the duration of the call (the reference's torch tensors play this role);
 *   - one sample per call (the reference's eval path is batch-1: DINOv2_mvsformer_model.py:88);
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*); calls never synchronise;
 *   - return 0 on success, a negative mvsf_status otherwise; mvsf_last_error() gives the message
 *     (the Python host raises RuntimeError, mirroring the reference's Python exceptions);
 *   - there is no CPU fallback and no dispatch: a missing/failed CUDA path is an error.
 *
 * Layouts (HBM):  feature maps are channels-last  [V][H][W][C];  hypothesis / probability volumes are
 * depth-major [D][H][W] (the reference's [B,D,H,W] with B=1);  cost volumes are [D][H][W][G] (NDHWC);
 * tokens are [L][C].  Packed-weight layouts are documented per function and produced by
 * mvsformerplusplus_b200/packing.py from a reference state_dict (BatchNorm folded, eval mode).
 */
#ifndef MVSF_B200_H
#define MVSF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* mvsf_stream_t; /* cudaStream_t */

enum mvsf_status {
  MVSF_OK = 0,
  MVSF_ERR_INVALID = -1,     /* bad argument / unsupported shape (reference: AssertionError / NotImplementedError) */
  MVSF_ERR_CUDA = -2,        /* CUDA launch or runtime error */
  MVSF_ERR_WORKSPACE = -3    /* workspace too small */
};

const char* mvsf_last_error(void);
int mvsf_abi_version(void);
/* number of kernel launches issued by this library on the calling thread since the last reset (bench.py's gpu_launches) */
long long mvsf_launch_count(int reset);
/* opt-in device timers around single kernels launched from inside a multi-kernel entry point ("attention_tc"):
 * CUDA events on the launching stream; read = device ms + launches since the last read (synchronises, resets). */
int mvsf_ktimer_enable(int on);
int mvsf_ktimer_read(const char* name, double* ms, long long* launches);

/* ---- layout helpers at the boundary (reference tensors are NCHW: DINOv2_mvsformer_model.py:95-98) */
int mvsf_nchw_to_nhwc(const float* src, float* dst, int N, int C, int HW, mvsf_stream_t stream);
int mvsf_nhwc_to_nchw(const float* src, float* dst, int N, int C, int HW, mvsf_stream_t stream);

/* ---- W1: projection prep.  models/cost_volume.py:68-71 + models/warping.py:80-82 (src@inv(ref), rot/trans)
 *      and torch.inverse(K) of models/position_encoding.py:146.
 * proj [V][2][4][4] (slot 0 extrinsic, slot 1[:3,:3] intrinsic; view 0 = reference view).
 * homs [(V-1)][12]: rot row-major (9) then trans (3) of  P_src * P_ref^-1.   kinv_ref [9] row-major. */
int mvsf_compose_geometry(const float* proj, int V, float* homs, float* kinv_ref, mvsf_stream_t stream);

/* ---- W2 prep for the warp seam: models/warping.py:80-82  proj = src_proj @ inverse(ref_proj) on composed 4x4
 * projections [B][4][4] (fp64 on device) -> homs [B][12] = rot row-major (9) then trans (3). */
int mvsf_homography_from_proj(const float* src_proj, const float* ref_proj, int B, float* homs, mvsf_stream_t stream);

/* ---- F5: models/module.py:692-704 init_inverse_range.  depth_values [Dn] -> out [D][H][W] */
int mvsf_init_inverse_range(const float* depth_values, int Dn, float* out, int D, int H, int W, mvsf_stream_t stream);
/* ---- F6: models/module.py:707-724 schedule_inverse_range (shift=False).
 * prev_depth [H/2][W/2], prev_hypo [Dp][H/2][W/2] (only planes 1 and 2 are read) -> out [D][H][W] */
int mvsf_schedule_inverse_range(const float* prev_depth, const float* prev_hypo, int Dp, float split_itv, float* out,
                                int D, int H, int W, mvsf_stream_t stream);
/* ---- F7: models/position_encoding.py:138-161 get_position_3d(normalize=True).
 * stats [6] = {width_min,width_max,height_min,height_max,depth_min,depth_max}.  pos [3][D][H][W].
 * compute_minmax: 1 = extents from this call's positions + depth range of depth_values, then normalise (B == 1);
 *                 0 = reuse the extents, refresh the depth range, normalise.
 * Batched callers (the reference reduces extents and depth_values.min()/max() over the whole batch,
 * position_encoding.py:152-157, DINOv2_mvsformer_model.py:156):  2 = reset + accumulate this sample's extents,
 * 3 = accumulate, 4 = finalise (decode extents, depth range over depth_values[0..Dn), Dn = B * numdepth),
 * 5 = normalise only.  Unused pointers may be NULL in modes 2-5. */
int mvsf_position3d(const float* kinv_ref, const float* depth, const float* depth_values, int Dn, float* stats,
                    int compute_minmax, float* pos, int D, int H, int W, mvsf_stream_t stream);

/* ---- W2 (finest seam): models/warping.py:69-109 homo_warping_3D_with_mask.
 * src [H][W][C], hom [12], depth [D][H][W] -> warped [C][D][H][W] (reference layout), mask [D][H][W] u8 or NULL */
int mvsf_homo_warp(const float* src_nhwc, const float* hom, const float* depth, float* warped, uint8_t* mask, int C,
                   int D, int H, int W, mvsf_stream_t stream);

/* ---- test hooks: the cost-volume passes have two organisations computing the same function - L1 gathers
 * from global memory (warp_corr.cu, any C in 8/16/32/64) and TMA-staged shared-memory windows (warp_tile.cu, C = 8/16, even H).
 * mode 0: force the L1 organisation everywhere; 1 (default): adaptive - the window kernels of the two-gather plan where they
 * apply, and for mvsf_warp_corr_entropy_store at C = 8, D = 4 a per-call choice made ON THE DEVICE from the call's own
 * geometry (share of sampled taps that miss the pipeline kernel's predicted windows <= 60 per mille -> pipeline kernel,
 * else L1 kernel; both are launched, the one not chosen returns at once); 2: force the pipeline kernel at C = 8, D = 4 and
 * the window kernels elsewhere.  mvsf_warp_corr_last_selection reads the most recent decision back (synchronises). */
int mvsf_warp_corr_set_tile_path(int mode);
int mvsf_warp_corr_last_selection(int* used_pipeline, int* miss_permille);

/* ---- which of the two cost-volume plans to run for a stage shape: 1 = two gathers (mvsf_warp_corr_entropy, mvsf_vis_cnn,
 * mvsf_warp_corr_aggregate; no intermediate buffer), 0 = spill plan (mvsf_warp_corr_entropy_store, mvsf_vis_cnn,
 * mvsf_corr_aggregate; needs a [(V-1)][D][H][W][8] fp32 buffer; the faster one on B200).  Both give the same volume. */
int mvsf_warp_corr_plan(int C, int G, int D, int H, int W, int V, size_t spill_budget_bytes);

/* ---- W2+W3+W4 pass A: warp + group correlation summed over groups + softmax-entropy over D.
 * models/cost_volume.py:72-92.  feat [V][H][W][C] (view 0 = reference), homs [(V-1)][12], depth [D][H][W]
 * -> entropy [(V-1)][H][W].   The (V-1,C,D,H,W) warped volume is never written. */
int mvsf_warp_corr_entropy(const float* feat, const float* homs, const float* depth, float* entropy, int V, int C,
                           int G, int D, int H, int W, mvsf_stream_t stream);
/* ---- W4 visibility CNN: models/cost_volume.py:37,93.  entropy [N][H][W] -> vis [N][H][W].
 * wts: packed, BN folded: w1[9][16] b1[16] w2[16 ic][9][16 oc] b2[16] w3[16 ic][9][8 oc] b3[8] w4[8] b4[1] (=3649 floats) */
int mvsf_vis_cnn(const float* entropy, const float* wts, float* vis, int N, int H, int W, mvsf_stream_t stream);
/* ---- W2+W3+W4 pass B: recompute warp + group correlation, weight by vis, reduce over views.
 * models/cost_volume.py:72-101 -> volume [D][H][W][G] = sum_v w_v*inprod_v / (sum_v w_v + 1e-6) */
int mvsf_warp_corr_aggregate(const float* feat, const float* homs, const float* depth, const float* vis,
                             float* volume, int V, int C, int G, int D, int H, int W, mvsf_stream_t stream);
/* Faster variant of the two calls above (the one hotpath.py uses): pass A additionally stores the per-view group
 * correlations corr [V-1][D][H*W][G] (G must be 8; 4*G*D*H*W*(V-1) bytes), the view aggregation then streams them
 * instead of gathering the source features a second time (the gather is L1-request bound, HBM has headroom). */
int mvsf_warp_corr_entropy_store(const float* feat, const float* homs, const float* depth, float* entropy, float* corr,
                                 int V, int C, int G, int D, int H, int W, mvsf_stream_t stream);
int mvsf_corr_aggregate(const float* corr, const float* vis, float* volume, int V, int G, int D, int H, int W,
                        mvsf_stream_t stream);

/* ---- R2-R4: models/module.py:367-408 (kind 0: CostRegNet, stride 2, 3^3 prob no bias) and
 *      :453-504 (kind 1: CostRegNet3D, stride (1,2,2), 1^3 prob + bias).  volume [D][H][W][C] -> logits [D][H][W].
 * wts: packed by packing.pack_costreg_unet (per layer [27][Cin][Cout] with BN scale folded, then bias[Cout]). */
int mvsf_costreg_unet_workspace_bytes(int kind, int C, int D, int H, int W, size_t* bytes);
/* install time: wts -> wts_tc, the fp16 hi/lo weight slabs of the tcgen05 implicit-GEMM convolutions (csrc/conv3d_tc.cu) */
int mvsf_costreg_unet_tc_bytes(size_t* bytes);
int mvsf_costreg_unet_pack_tc(int kind, const float* wts, void* wts_tc, size_t wts_tc_bytes, mvsf_stream_t stream);
int mvsf_costreg_unet_forward(int kind, const float* volume, const float* wts, const void* wts_tc, float* logits,
                              void* workspace, size_t workspace_bytes, int C, int D, int H, int W, mvsf_stream_t stream);
/* test seam: ONE 3x3x3 layer of the U-Nets on the tcgen05 implicit-GEMM path, fp32 in / out (module.py:367-504:
 * Conv3d / strided Conv3d / ConvTranspose3d(output_padding = stride - 1) + folded BN + ReLU, optional skip added after the
 * ReLU).  mode 0: stride 1, 1: stride (sd,2,2), 2: transposed (sd,2,2).  in [ID][IH][IW][cin]; w32 = [27][cin][cout] then
 * bias[cout]; skip (or NULL) and out [OD][OH][OW][cout]; workspace >= 4*(nin + 2*nout) + 216*cin*max(cout,16) + 512 bytes. */
int mvsf_conv3d_tc_layer(int mode, int sd, const float* in, const float* w32, const float* skip, float* out,
                         void* workspace, size_t workspace_bytes, int cin, int cout, int ID, int IH, int IW,
                         mvsf_stream_t stream);

/* ---- R1: models/module.py:602-646 PureTransformerCostReg (+ position_encoding.py:164-189 PositionEncoding3D).
 * volume [D][H][W][C] is modified in place by the PE add; pos [3][D][H][W] or NULL.
 * Fixed by the shipped config: down_rate (2,4,4), mid 64, heads 4, mlp 256.  softmax_scale = hd^-0.5*log_tal(N).
 * wts16 = mvsf_split_weights_f16(wts) (fp16 hi|lo parts for the tcgen05 GEMMs), n_wts = number of floats in wts. */
int mvsf_costreg_tr_workspace_bytes(int C, int D, int H, int W, size_t* bytes);
int mvsf_costreg_tr_forward(float* volume, const float* pos, const float* wts, const void* wts16, size_t n_wts,
                            float* logits, void* workspace, size_t workspace_bytes, int C, int D, int H, int W,
                            int layers, float softmax_scale, mvsf_stream_t stream);
/* install-time helper: fp32 weight blob (n floats, n % 8 == 0) -> out16 = [n fp16 hi parts | n fp16 lo parts] (4n bytes) */
int mvsf_split_weights_f16(const float* wts, void* out16, size_t n, mvsf_stream_t stream);

/* softmax attention of R1 alone: models/dino/layers/attention.py:141-170 (FlashAttention2.forward after the qkv linear).
 * qkv [N][3][4][16] fp32 -> out [N][64]; workspace >= (N+128)*896 bytes.  tcgen05 tensor cores, 3-term split-fp16 operands,
 * fp32 accumulation in TMEM; |q*scale|, |k|, |v| must be < 65504. */
int mvsf_attention_forward(const float* qkv, float* out, void* workspace, size_t workspace_bytes, int N,
                           float softmax_scale, mvsf_stream_t stream);

/* token-wise linear layer alone (nn.Linear, e.g. models/module.py:520-522 FFN.linear1): C[M,N] = act(A[M,K] W[N,K]^T + bias)
 * on the tcgen05 tensor cores with fp16 hi/lo split operands (fp32-class accuracy).  N % 16 == 0, N <= 256, K % 64 == 0.
 * workspace >= (M+N)*2K*2 + 256 bytes.  gelu != 0 applies the exact-erf GELU. */
int mvsf_linear_tc_forward(const float* A, const float* W, const float* bias, float* C, void* workspace,
                           size_t workspace_bytes, int M, int N, int K, int gelu, mvsf_stream_t stream);

/* ---- S1: models/cost_volume.py:105-117 + models/module.py:649-655 (eval, depth_type 'ce').
 * logits [D][H][W], depth hypotheses [D][H][W] -> prob [D][H][W], depth [H][W], conf [H][W] */
int mvsf_softargmax(const float* logits, const float* depth_hypo, float tmp, float* prob, float* depth, float* conf,
                    int D, int H, int W, mvsf_stream_t stream);
/* ---- S2: DINOv2_mvsformer_model.py:167-177: acc (+)= scale * nearest_upsample(conf) ; init!=0 overwrites */
int mvsf_conf_accumulate(const float* conf, int h, int w, float* acc, int H, int W, float scale, int init,
                         mvsf_stream_t stream);

/* ---- F1-F4: models/FMT.py:164-206 FMT_with_pathway.forward.
 * Inputs are the reference's NCHW pyramids: f1 [V][64][H1][W1], f2 [V][32][2H1][2W1], f3 [V][16][4H1][4W1],
 * f4 [V][8][8H1][8W1]; pe [H1*W1][64] is the PositionEncodingSineNorm table (position_encoding.py:61-74).
 * Outputs are channels-last: o1 [V][H1][W1][64] ... o4 [V][8H1][8W1][8].  wts: packing.pack_fmt. */
int mvsf_fmt_workspace_bytes(int V, int H1, int W1, size_t* bytes);
int mvsf_fmt_forward(const float* f1, const float* f2, const float* f3, const float* f4, const float* pe,
                     const float* wts, const void* wts16, size_t n_wts, float* o1, float* o2, float* o3, float* o4,
                     void* workspace, size_t workspace_bytes, int V, int H1, int W1, mvsf_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* MVSF_B200_H */
