// R1: stage-1 transformer cost regulariser, models/module.py:602-646 (PureTransformerCostReg) with
// FlashAttnBlock post-norm blocks (:569-582), LayerNorm3D (:586-599), PositionEncoding3D
// (models/position_encoding.py:164-189) and the entropy-invariance softmax scale (attention.py:158-161).
//
// volume [D][H][W][8] --(+pe_proj(PE3D))--> patchify (2,4,4) GEMM K=256 + LN3D --> tokens [N][64]
//   6 x { qkv GEMM -> softmax attention (4 heads x 16) -> proj GEMM + gamma1/residual/LN -> FFN GEMMs + gamma2/residual/LN }
//   --> un-patchify GEMM (64 -> 2*4*4*8) --> per-voxel LN3D(8) + 1x1x1 prob --> logits [D][H][W]
// Softmax attention is order-free over tokens, so tokens are kept in (d', h', w') raster order instead of the
// reference's "(h w d)" (module.py:573) - the result is identical.
#include <cuda_fp16.h>
#include <float.h>

#include "linear_tc.cuh"
#include "umma.cuh"

namespace mvsf {

// packed weights (floats), produced by packing.pack_costreg_tr:
//   pe_w[8][24] | down_w[64][256] (k = ((kd*4+kh)*4+kw)*8+ci) | down_b[64] | down_ln_w[64] | down_ln_b[64]
//   per layer: qkv_w[192][64] | proj_w[64][64] | proj_b[64] | gamma1[64] | n1_w[64] | n1_b[64]
//              | f1_w[256][64] | f1_b[256] | f2_w[64][256] | f2_b[64] | gamma2[64] | n2_w[64] | n2_b[64]
//   up_w[256][64] (n = ((kd*4+kh)*4+kw)*8+co) | up_b[256] | up_ln_w[8] | up_ln_b[8] | prob_w[8] | prob_b[1] (+3 pad)
constexpr int TR_PE = 0, TR_DOWN_W = 192, TR_DOWN_B = TR_DOWN_W + 64 * 256, TR_DOWN_LNW = TR_DOWN_B + 64,
              TR_DOWN_LNB = TR_DOWN_LNW + 64, TR_LAYER0 = TR_DOWN_LNB + 64;
constexpr int L_QKV = 0, L_PROJ_W = 192 * 64, L_PROJ_B = L_PROJ_W + 64 * 64, L_G1 = L_PROJ_B + 64, L_N1W = L_G1 + 64,
              L_N1B = L_N1W + 64, L_F1W = L_N1B + 64, L_F1B = L_F1W + 256 * 64, L_F2W = L_F1B + 256,
              L_F2B = L_F2W + 64 * 256, L_G2 = L_F2B + 64, L_N2W = L_G2 + 64, L_N2B = L_N2W + 64, TR_LAYER = L_N2B + 64;
constexpr int U_W = 0, U_B = 256 * 64, U_LNW = U_B + 256, U_LNB = U_LNW + 8, U_PW = U_LNB + 8, U_PB = U_PW + 8;

// volume[d,y,x,:] += pe_w (8x24) * PE3D(pos[:,d,y,x])
__global__ void pe3d_add_kernel(float* __restrict__ vol, const float* __restrict__ pos, const float* __restrict__ pe_w,
                                size_t nvox) {
  __shared__ float w[8 * 24];
  for (int i = threadIdx.x; i < 192; i += blockDim.x) w[i] = __ldg(pe_w + i);
  __syncthreads();
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nvox) return;
  // div_term = exp(arange(0,8,2) * (-ln(1e4)/8))  (position_encoding.py:169)
  const float div[4] = {1.0f, 0.1f, 0.01f, 0.001f};
  float pe[24];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    float p = __ldg(pos + a * nvox + i);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float arg = __fmul_rn(__fmul_rn(p, 4.0f), div[k]);
      pe[a * 8 + 2 * k] = sinf(arg);
      pe[a * 8 + 2 * k + 1] = cosf(arg);
    }
  }
  float4* v = reinterpret_cast<float4*>(vol + i * 8);
  float4 v0 = v[0], v1 = v[1];
  float o[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 24; ++k) s = fmaf(w[c * 24 + k], pe[k], s);
    o[c] += s;
  }
  v[0] = make_float4(o[0], o[1], o[2], o[3]);
  v[1] = make_float4(o[4], o[5], o[6], o[7]);
}

// im2col for the (2,4,4)/(2,4,4) patchify conv, emitted as the fp16 hi|lo split the tensor-core GEMM consumes:
// patches2[t] = [hi(256) | lo(256)], k = ((kd*4+kh)*4+kw)*8 + ci
__global__ void patch_gather_kernel(const float* __restrict__ vol, __half* __restrict__ patches2, int D, int H, int W) {
  const int Hp = H / 4, Wp = W / 4;
  size_t total = (size_t)(D / 2) * Hp * Wp * 32;  // one thread per (token, voxel): 8 channels
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int vox = (int)(i & 31);
  size_t t = i >> 5;
  int wp = (int)(t % Wp), hp = (int)((t / Wp) % Hp), dp = (int)(t / ((size_t)Wp * Hp));
  int kw = vox & 3, kh = (vox >> 2) & 3, kd = vox >> 4;
  const float* src = vol + (((size_t)(dp * 2 + kd) * H + hp * 4 + kh) * W + wp * 4 + kw) * 8;
  float4 a = ldg4(src), b = ldg4(src + 4);
  float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  __half* row = patches2 + t * 512 + vox * 8;
  split_store8(row, row + 256, v);
}

__device__ __forceinline__ void split_f16(float x, __half& hi, __half& lo) {
  hi = __float2half_rn(x);
  lo = __float2half_rn(x - __half2float(hi));
}
__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

#include "attention_fa.cuh"   // second-generation attention kernel (inside namespace mvsf)

// un-patchify epilogue: u [N][256] (n = vox*8+co) -> LayerNorm3D over the 8 channels of each voxel (eps 1e-6)
// -> prob 1x1x1 (8 -> 1) + bias -> logits [D][H][W]
__global__ void unpatch_ln_prob_kernel(const float* __restrict__ u, const float* __restrict__ tail,
                                       float* __restrict__ logits, int D, int H, int W) {
  const int Hp = H / 4, Wp = W / 4;
  size_t total = (size_t)D * H * W;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  // thread order follows u's memory order (token-major, voxel-minor) so the 32-byte reads are coalesced
  int vox = (int)(i & 31);
  size_t t = i >> 5;
  int wp = (int)(t % Wp), hp = (int)((t / Wp) % Hp), dp = (int)(t / ((size_t)Wp * Hp));
  int kw = vox & 3, kh = (vox >> 2) & 3, kd = vox >> 4;
  float4 a = ldg4(u + i * 8), b = ldg4(u + i * 8 + 4);
  float x[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  float mean = 0.f;
#pragma unroll
  for (int c = 0; c < 8; ++c) mean += x[c];
  mean *= 0.125f;
  float var = 0.f;
#pragma unroll
  for (int c = 0; c < 8; ++c) { float dd = x[c] - mean; var = fmaf(dd, dd, var); }
  var *= 0.125f;
  const float sd = sqrtf(var + 1e-6f);
  float s = __ldg(tail + (U_PB - U_LNW));
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    float y = __ldg(tail + c) * __fdiv_rn(x[c] - mean, sd) + __ldg(tail + 8 + c);
    s = fmaf(y, __ldg(tail + 16 + c), s);
  }
  logits[((size_t)(dp * 2 + kd) * H + hp * 4 + kh) * W + wp * 4 + kw] = s;
}


static int run_attention(const float* qkv, float* o, __half* o2, __half* tiled, int N, float scale_log2e, cudaStream_t s) {
  const int ntiles = cdiv(N, 128);
  qkv_tile_kernel<<<cdiv((long long)ntiles * 128 * 24, 256), 256, 0, s>>>(qkv, tiled, N, ntiles, scale_log2e);
  MVSF_LAUNCH_CHECK("qkv_tile");
  static DeviceOnce once;
  const int dev = current_device();
  if (once.need(dev)) {
    MVSF_CUDA_OK(cudaFuncSetAttribute(attention_fa_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fa6::SMEM));
    once.done(dev);
  }
  cudaEvent_t kt = ktimer_enabled() ? ktimer_begin("attention_tc", s) : nullptr;
  const dim3 grid(cdiv(ntiles, 2), 4);
  attention_fa_kernel<<<grid, fa6::THREADS, fa6::SMEM, s>>>(tiled, o, o2, N, ntiles);
  if (kt) ktimer_end(kt, s);
  MVSF_LAUNCH_CHECK("attention_tc");
  return MVSF_OK;
}

}  // namespace mvsf

using namespace mvsf;

extern "C" {

int mvsf_costreg_tr_workspace_bytes(int C, int D, int H, int W, size_t* bytes) {
  MVSF_REQUIRE(bytes && C == 8, "costreg_tr: base channel must be 8");
  MVSF_REQUIRE(D % 2 == 0 && H % 4 == 0 && W % 4 == 0 && D > 0 && H > 0 && W > 0,
               "costreg_tr: D %% 2, H %% 4, W %% 4 must be 0 (down_rate (2,4,4))");
  size_t N = (size_t)(D / 2) * (H / 4) * (W / 4);
  // per token (in floats): big 256 (patches2 / ffn hidden split / un-patchify out), x 64, y 64, x2 64, y2 64, o2 64,
  // qkv 192, attention operand split 192
  *bytes = (N * (256 + 64 + 64 + 64 + 64 + 64 + 192) + (N + 128) * 224) * sizeof(float);
  return MVSF_OK;
}

int mvsf_costreg_tr_forward(float* volume, const float* pos, const float* wts, const void* wts16, size_t n_wts,
                            float* logits, void* workspace, size_t workspace_bytes, int C, int D, int H, int W,
                            int layers, float softmax_scale, mvsf_stream_t stream) {
  MVSF_REQUIRE(volume && wts && wts16 && logits && workspace && layers >= 0, "costreg_tr: bad arguments");
  size_t need = 0;
  int rc = mvsf_costreg_tr_workspace_bytes(C, D, H, W, &need);
  if (rc) return rc;
  if (workspace_bytes < need) return fail(MVSF_ERR_WORKSPACE, "costreg_tr: workspace %zu < %zu bytes", workspace_bytes, need);
  MVSF_REQUIRE(((uintptr_t)workspace & 15) == 0 && ((uintptr_t)wts & 15) == 0 && ((uintptr_t)volume & 15) == 0 &&
                   ((uintptr_t)wts16 & 15) == 0 && (n_wts % 8) == 0,
               "costreg_tr: pointers must be 16-byte aligned");
  MVSF_REQUIRE(n_wts >= (size_t)TR_LAYER0 + (size_t)layers * TR_LAYER + U_PB + 1, "costreg_tr: weight blob too small");
  cudaStream_t s = (cudaStream_t)stream;
  const size_t nvox = (size_t)D * H * W;
  const int N = (int)((size_t)(D / 2) * (H / 4) * (W / 4));
  const __half* wh = reinterpret_cast<const __half*>(wts16);  // fp16 hi parts, same indexing as wts
  const __half* wl = wh + n_wts;                              // fp16 lo parts
  float* big = (float*)workspace;                             // [N][256] floats
  __half* big2 = reinterpret_cast<__half*>(big);             // [N][512] halves: row = [hi(256) | lo(256)]
  float* x = big + (size_t)N * 256;                           // [N][64]
  float* y = x + (size_t)N * 64;                              // [N][64]
  __half* x2 = reinterpret_cast<__half*>(y + (size_t)N * 64);    // [N][128] = [hi(64) | lo(64)]
  __half* y2 = x2 + (size_t)N * 128;
  __half* o2 = y2 + (size_t)N * 128;
  float* qkv = reinterpret_cast<float*>(o2 + (size_t)N * 128);   // [N][192]
  __half* split = reinterpret_cast<__half*>(qkv + (size_t)N * 192);  // [6][4][N][16] fp16

  if (pos) {
    pe3d_add_kernel<<<cdiv((long long)nvox, 256), 256, 0, s>>>(volume, pos, wts + TR_PE, nvox);
    MVSF_LAUNCH_CHECK("pe3d_add");
  }
  patch_gather_kernel<<<cdiv((long long)N * 32, 256), 256, 0, s>>>(volume, big2, D, H, W);
  MVSF_LAUNCH_CHECK("patch_gather");

  TcLinArgs a{};
  a.Ah = big2; a.Al = big2 + 256; a.lda = 512; a.Bh = wh + TR_DOWN_W; a.Bl = wl + TR_DOWN_W; a.ldb = 256;
  a.M = N; a.N = 64; a.K = 256; a.bias = wts + TR_DOWN_B; a.ln_w = wts + TR_DOWN_LNW; a.ln_b = wts + TR_DOWN_LNB; a.ln_eps = 1e-6f;
  a.C = x; a.ldc = 64; a.C2 = x2; a.ldc2 = 128;
  if ((rc = launch_linear_tc(a, LIN_LN, s))) return rc;

  const float scale_log2e = softmax_scale * 1.4426950408889634f;
  for (int l = 0; l < layers; ++l) {
    const size_t lo = (size_t)TR_LAYER0 + (size_t)l * TR_LAYER;
    const float* lw = wts + lo;
    TcLinArgs q{};
    q.Ah = x2; q.Al = x2 + 64; q.lda = 128; q.Bh = wh + lo + L_QKV; q.Bl = wl + lo + L_QKV; q.ldb = 64;
    q.M = N; q.N = 192; q.K = 64; q.C = qkv; q.ldc = 192;
    if ((rc = launch_linear_tc(q, LIN_BIAS, s))) return rc;
    if ((rc = run_attention(qkv, nullptr, o2, split, N, scale_log2e, s))) return rc;
    TcLinArgs p{};
    p.Ah = o2; p.Al = o2 + 64; p.lda = 128; p.Bh = wh + lo + L_PROJ_W; p.Bl = wl + lo + L_PROJ_W; p.ldb = 64;
    p.M = N; p.N = 64; p.K = 64; p.bias = lw + L_PROJ_B; p.res = x; p.ldres = 64; p.gamma = lw + L_G1;
    p.ln_w = lw + L_N1W; p.ln_b = lw + L_N1B; p.ln_eps = 1e-5f; p.C = y; p.ldc = 64; p.C2 = y2; p.ldc2 = 128;
    if ((rc = launch_linear_tc(p, LIN_RES_LN, s))) return rc;
    TcLinArgs f1{};
    f1.Ah = y2; f1.Al = y2 + 64; f1.lda = 128; f1.Bh = wh + lo + L_F1W; f1.Bl = wl + lo + L_F1W; f1.ldb = 64;
    f1.M = N; f1.N = 256; f1.K = 64; f1.bias = lw + L_F1B; f1.C2 = big2; f1.ldc2 = 512;
    if ((rc = launch_linear_tc(f1, LIN_GELU, s))) return rc;
    TcLinArgs f2{};
    f2.Ah = big2; f2.Al = big2 + 256; f2.lda = 512; f2.Bh = wh + lo + L_F2W; f2.Bl = wl + lo + L_F2W; f2.ldb = 256;
    f2.M = N; f2.N = 64; f2.K = 256; f2.bias = lw + L_F2B; f2.res = y; f2.ldres = 64; f2.gamma = lw + L_G2;
    f2.ln_w = lw + L_N2W; f2.ln_b = lw + L_N2B; f2.ln_eps = 1e-5f; f2.C = x; f2.ldc = 64; f2.C2 = x2; f2.ldc2 = 128;
    if ((rc = launch_linear_tc(f2, LIN_RES_LN, s))) return rc;
  }
  const size_t uo = (size_t)TR_LAYER0 + (size_t)layers * TR_LAYER;
  TcLinArgs u{};
  u.Ah = x2; u.Al = x2 + 64; u.lda = 128; u.Bh = wh + uo + U_W; u.Bl = wl + uo + U_W; u.ldb = 64;
  u.M = N; u.N = 256; u.K = 64; u.bias = wts + uo + U_B; u.C = big; u.ldc = 256;
  if ((rc = launch_linear_tc(u, LIN_BIAS, s))) return rc;
  unpatch_ln_prob_kernel<<<cdiv((long long)nvox, 256), 256, 0, s>>>(big, wts + uo + U_LNW, logits, D, H, W);
  MVSF_LAUNCH_CHECK("unpatch_ln_prob");
  return MVSF_OK;
}

/* Softmax attention alone (attention.py:141-170): qkv [N][3][4][16] fp32 -> out [N][64].  workspace >= N*768 bytes. */
int mvsf_attention_forward(const float* qkv, float* out, void* workspace, size_t workspace_bytes, int N,
                           float softmax_scale, mvsf_stream_t stream) {
  MVSF_REQUIRE(qkv && out && workspace && N > 0, "attention_forward: bad arguments");
  if (workspace_bytes < (size_t)(N + 128) * 896) return fail(MVSF_ERR_WORKSPACE, "attention_forward: workspace %zu < %zu bytes", workspace_bytes, (size_t)(N + 128) * 896);
  return run_attention(qkv, out, nullptr, reinterpret_cast<__half*>(workspace), N, softmax_scale * 1.4426950408889634f, (cudaStream_t)stream);
}
}
