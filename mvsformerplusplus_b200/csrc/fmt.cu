// F1-F4: FMT_with_pathway.forward (models/FMT.py:164-206): cross-view feature transformer on the 1/8-resolution
// features (FMT.forward :81-137, CrossBlock block.py:336-346 pre-norm with pre_norm_query=False, linear attention
// attention.py:261-291, LayerScale, Mlp) followed by the top-down pathway
//   stage_{k+1} = smooth_k( bilinear_up(dim_reduction_k(stage_k)) + lateral_{k+1} )      (FMT.py:154-162,195-197).
// Tokens "(h w) c" of the reference are exactly channels-last pixels, so the stage-1 output is produced directly in
// the [V][H][W][64] layout the warp kernels consume.  All source views are processed as one batch; the K/V
// summaries of the two cross layers depend only on the reference view and are computed once.
#include "linear_tc.cuh"
#include "umma.cuh"

namespace mvsf {

// packed weights per CrossBlock (floats): n1_w[64] n1_b[64] qkv_w[192][64] proj_w[64][64] proj_b[64] g1[64]
//                                          n2_w[64] n2_b[64] f1_w[256][64] f1_b[256] f2_w[64][256] f2_b[64] g2[64]
constexpr int B_N1W = 0, B_N1B = 64, B_QKV = 128, B_PW = B_QKV + 192 * 64, B_PB = B_PW + 64 * 64, B_G1 = B_PB + 64,
              B_N2W = B_G1 + 64, B_N2B = B_N2W + 64, B_F1W = B_N2B + 64, B_F1B = B_F1W + 256 * 64,
              B_F2W = B_F1B + 256, B_F2B = B_F2W + 64 * 256, B_G2 = B_F2B + 64, B_SIZE = B_G2 + 64;
// after 4 blocks: dr1[32][64] dr2[16][32] dr3[8][16] sm1[9][32][32] sm2[9][16][16] sm3[9][8][8]   ([tap][ci][co])
constexpr int P_DR1 = 4 * B_SIZE, P_DR2 = P_DR1 + 32 * 64, P_DR3 = P_DR2 + 16 * 32, P_SM1 = P_DR3 + 8 * 16,
              P_SM2 = P_SM1 + 9 * 32 * 32, P_SM3 = P_SM2 + 9 * 16 * 16, FMT_WTS = P_SM3 + 9 * 8 * 8;
constexpr int KVSZ = 4 * 16 * 16 + 64;  // KV[h][m][d] + ksum[h][d]

// f [V][64][L] (NCHW) + pe [L][64] -> tok [V][L][64]
__global__ void tokens_add_pe_kernel(const float* __restrict__ f, const float* __restrict__ pe, float* __restrict__ tok,
                                     int L) {
  __shared__ float tile[32][33];
  const int v = blockIdx.z;
  const float* s = f + (size_t)v * 64 * L;
  float* d = tok + (size_t)v * 64 * L;
  int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int c = c0 + i, p = p0 + threadIdx.x;
    if (p < L) tile[i][threadIdx.x] = s[(size_t)c * L + p];
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int p = p0 + i, c = c0 + threadIdx.x;
    if (p < L) d[(size_t)p * 64 + c] = tile[threadIdx.x][i] + __ldg(pe + (size_t)p * 64 + c);
  }
}

// partial[view][blk][KVSZ]: KV[h][m][d] = sum_s k[s,h,d] v[s,h,m] ; ksum[h][d] = sum_s k[s,h,d]  over a 256-token chunk
constexpr int KV_CHUNK = 256, KV_TILE = 64;
__global__ void __launch_bounds__(256)
kv_partial_kernel(const float* __restrict__ kv, int ld, int koff, int voff, int L, float* __restrict__ partial) {
  __shared__ __align__(16) float ks[KV_TILE][64];
  __shared__ __align__(16) float vs[KV_TILE][64];
  const int view = blockIdx.y, blk = blockIdx.x, tid = threadIdx.x;
  const float* base = kv + (size_t)view * L * ld;
  const int h = tid >> 6, m = (tid >> 2) & 15, d0 = (tid & 3) * 4;
  float acc[4] = {0.f, 0.f, 0.f, 0.f}, ksum[4] = {0.f, 0.f, 0.f, 0.f};
  const int s_begin = blk * KV_CHUNK, s_end = min(L, s_begin + KV_CHUNK);
  for (int s0 = s_begin; s0 < s_end; s0 += KV_TILE) {
    __syncthreads();
    for (int i = tid; i < KV_TILE * 16; i += 256) {
      int r = i >> 4, c = (i & 15) * 4;
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
      if (s0 + r < s_end) {
        a = ldg4(base + (size_t)(s0 + r) * ld + koff + c);
        b = ldg4(base + (size_t)(s0 + r) * ld + voff + c);
      }
      *reinterpret_cast<float4*>(&ks[r][c]) = a;
      *reinterpret_cast<float4*>(&vs[r][c]) = b;
    }
    __syncthreads();
#pragma unroll 8
    for (int r = 0; r < KV_TILE; ++r) {
      float4 k4 = *reinterpret_cast<const float4*>(&ks[r][h * 16 + d0]);
      float vv = vs[r][h * 16 + m];
      acc[0] = fmaf(k4.x, vv, acc[0]); acc[1] = fmaf(k4.y, vv, acc[1]);
      acc[2] = fmaf(k4.z, vv, acc[2]); acc[3] = fmaf(k4.w, vv, acc[3]);
      ksum[0] += k4.x; ksum[1] += k4.y; ksum[2] += k4.z; ksum[3] += k4.w;
    }
  }
  float* o = partial + ((size_t)view * gridDim.x + blk) * KVSZ;
  *reinterpret_cast<float4*>(o + (h * 16 + m) * 16 + d0) = make_float4(acc[0], acc[1], acc[2], acc[3]);
  if (m == 0) *reinterpret_cast<float4*>(o + 1024 + h * 16 + d0) = make_float4(ksum[0], ksum[1], ksum[2], ksum[3]);
}
__global__ void kv_final_kernel(const float* __restrict__ partial, int nblk, float* __restrict__ fin) {
  const int view = blockIdx.y;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= KVSZ) return;
  float s = 0.f;
  for (int b = 0; b < nblk; ++b) s += partial[((size_t)view * nblk + b) * KVSZ + i];
  fin[(size_t)view * KVSZ + i] = s;
}

// Row LayerNorm over 64 channels emitting the fp16 hi|lo split [hi(64) | lo(64)] the tensor-core GEMMs consume
__global__ void __launch_bounds__(256)
layernorm64_split_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ b,
                         __half* __restrict__ y2, int M, float eps) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= M) return;
  float2 v = ldg2(x + (size_t)row * 64 + lane * 2);
  float s = v.x + v.y;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s * (1.0f / 64.0f);
  float d0 = v.x - mean, d1 = v.y - mean;
  float q = d0 * d0 + d1 * d1;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  const float sd = sqrtf(q * (1.0f / 64.0f) + eps);
  float2 ww = ldg2(w + lane * 2), bb = ldg2(b + lane * 2);
  const float o0 = __fdiv_rn(d0, sd) * ww.x + bb.x, o1 = __fdiv_rn(d1, sd) * ww.y + bb.y;
  const __half2 hh = __floats2half2_rn(o0, o1);
  const float2 hf = __half22float2(hh);
  *reinterpret_cast<__half2*>(y2 + (size_t)row * 128 + lane * 2) = hh;
  *reinterpret_cast<__half2*>(y2 + (size_t)row * 128 + 64 + lane * 2) = __floats2half2_rn(o0 - hf.x, o1 - hf.y);
}

// out[s][h*16+m] = (sum_d q[s,h,d] KV[h][m][d]) / (q[s,h,:] . ksum[h,:] + 1e-6)     (attention.py:281-284)
__global__ void __launch_bounds__(128)
linattn_apply_kernel(const float* __restrict__ q, int ldq, const float* __restrict__ kvfin, size_t kv_view_stride,
                     __half* __restrict__ out2, int L, int M) {
  __shared__ __align__(16) float kvs[256 + 16];
  const int h = blockIdx.y;
  const int s = blockIdx.x * 128 + threadIdx.x;
  const int view = (blockIdx.x * 128) / L;  // host guarantees L % 128 == 0 or a single view per launch
  const float* kvp = kvfin + (size_t)view * kv_view_stride;
  for (int i = threadIdx.x; i < 256; i += 128) kvs[i] = __ldg(kvp + h * 256 + i);
  if (threadIdx.x < 16) kvs[256 + threadIdx.x] = __ldg(kvp + 1024 + h * 16 + threadIdx.x);
  __syncthreads();
  if (s >= M) return;
  float qv[16];
  const float* qp = q + (size_t)s * ldq + h * 16;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    float4 t = ldg4(qp + c * 4);
    qv[c * 4] = t.x; qv[c * 4 + 1] = t.y; qv[c * 4 + 2] = t.z; qv[c * 4 + 3] = t.w;
  }
  float den = 0.f;
#pragma unroll
  for (int d = 0; d < 16; ++d) den = fmaf(qv[d], kvs[256 + d], den);
  const float z = __fdiv_rn(1.0f, den + 1e-6f);
  __half* op = out2 + (size_t)s * 128 + h * 16;  // fp16 hi|lo split rows [hi(64) | lo(64)]
#pragma unroll
  for (int mq = 0; mq < 4; ++mq) {
    float r[4];
#pragma unroll
    for (int mm = 0; mm < 4; ++mm) {
      const float4* kp = reinterpret_cast<const float4*>(&kvs[(mq * 4 + mm) * 16]);
      float4 a = kp[0], b = kp[1], c = kp[2], e = kp[3];
      float t = qv[0] * a.x;
      t = fmaf(qv[1], a.y, t); t = fmaf(qv[2], a.z, t); t = fmaf(qv[3], a.w, t);
      t = fmaf(qv[4], b.x, t); t = fmaf(qv[5], b.y, t); t = fmaf(qv[6], b.z, t); t = fmaf(qv[7], b.w, t);
      t = fmaf(qv[8], c.x, t); t = fmaf(qv[9], c.y, t); t = fmaf(qv[10], c.z, t); t = fmaf(qv[11], c.w, t);
      t = fmaf(qv[12], e.x, t); t = fmaf(qv[13], e.y, t); t = fmaf(qv[14], e.z, t); t = fmaf(qv[15], e.w, t);
      r[mm] = t * z;
    }
    const __half2 h01 = __floats2half2_rn(r[0], r[1]), h23 = __floats2half2_rn(r[2], r[3]);
    const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
    *reinterpret_cast<__half2*>(op + mq * 4) = h01;
    *reinterpret_cast<__half2*>(op + mq * 4 + 2) = h23;
    *reinterpret_cast<__half2*>(op + 64 + mq * 4) = __floats2half2_rn(r[0] - f01.x, r[1] - f01.y);
    *reinterpret_cast<__half2*>(op + 64 + mq * 4 + 2) = __floats2half2_rn(r[2] - f23.x, r[3] - f23.y);
  }
}

#include "fmt_smooth_tc.cuh"   // fused upsample + lateral add + 3x3 smooth conv on tcgen05

struct FmtWs {
  __half *xn2, *att2, *hid2;   // fp16 hi|lo split activations: [M][128], [M][128], [M][512]
  float *qkv, *ref0, *kvpart, *kvfin, *kvc;
  const __half *wh, *wl;       // fp16 hi / lo parts of the packed weight blob (same indexing as the fp32 blob)
};

// one CrossBlock over `M` tokens (nviews views of L tokens each) stored at x (in place).
// self attention: kv_src == nullptr ; cross attention: kvc = precomputed K/V summary of the reference view.
// LayerNorms are fused into the epilogue of the GEMM that produces their input: proj emits x (residual stream) and
// split(norm2(x)), FFN2 emits x and split(norm1 of the NEXT block) when `next_bw` is given; `ln1_ready` says the previous
// block already left split(norm1(x)) in ws.xn2.
static int run_block(float* x, int nviews, int L, const float* bw, size_t boff, const float* kvc, const FmtWs& ws,
                     cudaStream_t s, bool ln1_ready = false, const float* next_bw = nullptr) {
  const int M = nviews * L;
  int rc;
  if (!ln1_ready) {
    layernorm64_split_kernel<<<cdiv(M, 8), 256, 0, s>>>(x, bw + B_N1W, bw + B_N1B, ws.xn2, M, 1e-5f);
    MVSF_LAUNCH_CHECK("fmt_ln1");
  }
  const float* kvsum;
  size_t kv_stride;
  int ldq;
  TcLinArgs a{};
  a.Ah = ws.xn2; a.Al = ws.xn2 + 64; a.lda = 128; a.Bh = ws.wh + boff + B_QKV; a.Bl = ws.wl + boff + B_QKV; a.ldb = 64;
  a.M = M; a.K = 64; a.C = ws.qkv;
  if (!kvc) {
    a.N = 192; a.ldc = 192; a.elu_cols = 128;
    if ((rc = launch_linear_tc(a, LIN_ELU1, s))) return rc;
    const int nblk = cdiv(L, KV_CHUNK);
    kv_partial_kernel<<<dim3(nblk, nviews), 256, 0, s>>>(ws.qkv, 192, 64, 128, L, ws.kvpart);
    MVSF_LAUNCH_CHECK("fmt_kv_partial");
    kv_final_kernel<<<dim3(cdiv(KVSZ, 256), nviews), 256, 0, s>>>(ws.kvpart, nblk, ws.kvfin);
    MVSF_LAUNCH_CHECK("fmt_kv_final");
    kvsum = ws.kvfin; kv_stride = KVSZ; ldq = 192;
  } else {
    a.N = 64; a.ldc = 64; a.elu_cols = 64;
    if ((rc = launch_linear_tc(a, LIN_ELU1, s))) return rc;
    kvsum = kvc; kv_stride = 0; ldq = 64;
  }
  if (L % 128 == 0 || nviews == 1) {
    linattn_apply_kernel<<<dim3(cdiv(M, 128), 4), 128, 0, s>>>(ws.qkv, ldq, kvsum, kv_stride, ws.att2, L, M);
    MVSF_LAUNCH_CHECK("fmt_linattn_apply");
  } else {
    for (int v = 0; v < nviews; ++v) {  // views do not align with 128-token blocks: one launch per view
      linattn_apply_kernel<<<dim3(cdiv(L, 128), 4), 128, 0, s>>>(ws.qkv + (size_t)v * L * ldq, ldq,
                                                                 kvsum + (size_t)v * kv_stride, 0,
                                                                 ws.att2 + (size_t)v * L * 128, L, L);
      MVSF_LAUNCH_CHECK("fmt_linattn_apply");
    }
  }
  TcLinArgs p{};
  p.Ah = ws.att2; p.Al = ws.att2 + 64; p.lda = 128; p.Bh = ws.wh + boff + B_PW; p.Bl = ws.wl + boff + B_PW; p.ldb = 64;
  p.M = M; p.N = 64; p.K = 64; p.bias = bw + B_PB; p.res = x; p.ldres = 64; p.gamma = bw + B_G1;
  p.Cpre = x; p.ldcpre = 64; p.ln_w = bw + B_N2W; p.ln_b = bw + B_N2B; p.ln_eps = 1e-5f; p.C2 = ws.xn2; p.ldc2 = 128;
  if ((rc = launch_linear_tc(p, LIN_RES_LN, s))) return rc;   // x += gamma1 * proj(...), xn2 = split(norm2(x))
  TcLinArgs f1{};
  f1.Ah = ws.xn2; f1.Al = ws.xn2 + 64; f1.lda = 128; f1.Bh = ws.wh + boff + B_F1W; f1.Bl = ws.wl + boff + B_F1W; f1.ldb = 64;
  f1.M = M; f1.N = 256; f1.K = 64; f1.bias = bw + B_F1B; f1.C2 = ws.hid2; f1.ldc2 = 512;
  if ((rc = launch_linear_tc(f1, LIN_GELU, s))) return rc;
  TcLinArgs f2{};
  f2.Ah = ws.hid2; f2.Al = ws.hid2 + 256; f2.lda = 512; f2.Bh = ws.wh + boff + B_F2W; f2.Bl = ws.wl + boff + B_F2W; f2.ldb = 256;
  f2.M = M; f2.N = 64; f2.K = 256; f2.bias = bw + B_F2B; f2.res = x; f2.ldres = 64; f2.gamma = bw + B_G2;
  if (next_bw) {   // x += gamma2 * ffn(...), xn2 = split(norm1_next(x))
    f2.Cpre = x; f2.ldcpre = 64; f2.ln_w = next_bw + B_N1W; f2.ln_b = next_bw + B_N1B; f2.ln_eps = 1e-5f; f2.C2 = ws.xn2; f2.ldc2 = 128;
    if ((rc = launch_linear_tc(f2, LIN_RES_LN, s))) return rc;
  } else {
    f2.C = x; f2.ldc = 64;
    if ((rc = launch_linear_tc(f2, LIN_RES, s))) return rc;
  }
  return MVSF_OK;
}

// K/V summary of a cross layer: key = value = norm1_layer(ref_feature)   (block.py:341-343, FMT.py:121-125)
static int run_cross_kv(const float* ref_tok, int L, const float* bw, size_t boff, float* kvc_out, const FmtWs& ws,
                        cudaStream_t s) {
  int rc;
  layernorm64_split_kernel<<<cdiv(L, 8), 256, 0, s>>>(ref_tok, bw + B_N1W, bw + B_N1B, ws.xn2, L, 1e-5f);
  MVSF_LAUNCH_CHECK("fmt_ln_key");
  TcLinArgs a{};
  a.Ah = ws.xn2; a.Al = ws.xn2 + 64; a.lda = 128;
  a.Bh = ws.wh + boff + B_QKV + 64 * 64; a.Bl = ws.wl + boff + B_QKV + 64 * 64; a.ldb = 64;
  a.M = L; a.N = 128; a.K = 64; a.C = ws.qkv; a.ldc = 128; a.elu_cols = 64;
  if ((rc = launch_linear_tc(a, LIN_ELU1, s))) return rc;
  const int nblk = cdiv(L, KV_CHUNK);
  kv_partial_kernel<<<dim3(nblk, 1), 256, 0, s>>>(ws.qkv, 128, 0, 64, L, ws.kvpart);
  MVSF_LAUNCH_CHECK("fmt_kv_partial");
  kv_final_kernel<<<dim3(cdiv(KVSZ, 256), 1), 256, 0, s>>>(ws.kvpart, nblk, kvc_out);
  MVSF_LAUNCH_CHECK("fmt_kv_final");
  return MVSF_OK;
}

// 1x1 dim_reduction_k of the pathway (FMT.py:186-189, a bias-free conv = per-pixel CIN -> COUT linear map), channels-last.
// One pixel per thread: the CIN inputs sit in registers, the [COUT][CIN] weights in shared memory (every lane reads the
// same weight: broadcast), HBM traffic = CIN + COUT floats per pixel.  (The generic SIMT GEMM tile this replaces ran at
// 39 / 76 / 185 us for the three levels, ~7x its memory time.)
template <int CIN, int COUT>
__global__ void __launch_bounds__(128)
reduce1x1_kernel(const float* __restrict__ x, const float* __restrict__ w, float* __restrict__ y, int M) {
  __shared__ __align__(16) float ws[COUT * CIN];
  for (int i = threadIdx.x; i < COUT * CIN / 4; i += 128) reinterpret_cast<float4*>(ws)[i] = ldg4(w + 4 * i);
  __syncthreads();
  const int m = blockIdx.x * 128 + threadIdx.x;
  if (m >= M) return;
  float4 xv[CIN / 4];
#pragma unroll
  for (int k = 0; k < CIN / 4; ++k) xv[k] = ldg4(x + (size_t)m * CIN + 4 * k);
  float* yo = y + (size_t)m * COUT;
#pragma unroll
  for (int n4 = 0; n4 < COUT / 4; ++n4) {
    float o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4* wr = reinterpret_cast<const float4*>(ws + (n4 * 4 + j) * CIN);
      float acc = 0.f;
#pragma unroll
      for (int k = 0; k < CIN / 4; ++k) {
        const float4 wv = wr[k];
        acc = fmaf(xv[k].x, wv.x, acc); acc = fmaf(xv[k].y, wv.y, acc);
        acc = fmaf(xv[k].z, wv.z, acc); acc = fmaf(xv[k].w, wv.w, acc);
      }
      o[j] = acc;
    }
    *reinterpret_cast<float4*>(yo + n4 * 4) = make_float4(o[0], o[1], o[2], o[3]);
  }
}

template <int CIN, int COUT>
static int run_pathway_level(const float* prev, const float* lat, const float* dr_w, const float* sm_w, float* red,
                             float* pre, float* out, int V, int h, int w, cudaStream_t s) {
  const int M = V * h * w;
  reduce1x1_kernel<CIN, COUT><<<cdiv(M, 128), 128, 0, s>>>(prev, dr_w, red, M);
  MVSF_LAUNCH_CHECK("fmt_reduce1x1");
  (void)pre;
  return launch_fmt_smooth_tc<COUT>(red, lat, sm_w, out, V, h, w, s);
}

}  // namespace mvsf

using namespace mvsf;

extern "C" {

int mvsf_fmt_workspace_bytes(int V, int H1, int W1, size_t* bytes) {
  MVSF_REQUIRE(bytes && V >= 2 && H1 > 0 && W1 > 0, "fmt: bad arguments");
  size_t L = (size_t)H1 * W1, VL = (size_t)V * L;
  size_t nblk = (L + KV_CHUNK - 1) / KV_CHUNK;
  size_t n = 640 * VL + 64 * L + (size_t)V * nblk * KVSZ + (size_t)(V + 2) * KVSZ + 64;
  *bytes = n * sizeof(float);
  return MVSF_OK;
}

int mvsf_fmt_forward(const float* f1, const float* f2, const float* f3, const float* f4, const float* pe,
                     const float* wts, const void* wts16, size_t n_wts, float* o1, float* o2, float* o3, float* o4,
                     void* workspace, size_t workspace_bytes, int V, int H1, int W1, mvsf_stream_t stream) {
  MVSF_REQUIRE(f1 && f2 && f3 && f4 && pe && wts && wts16 && o1 && o2 && o3 && o4 && workspace, "fmt: null pointer");
  MVSF_REQUIRE(n_wts >= (size_t)FMT_WTS && (n_wts % 8) == 0 && ((uintptr_t)wts16 & 15) == 0, "fmt: bad fp16 weight blob");
  size_t need = 0;
  int rc = mvsf_fmt_workspace_bytes(V, H1, W1, &need);
  if (rc) return rc;
  if (workspace_bytes < need) return fail(MVSF_ERR_WORKSPACE, "fmt: workspace %zu < %zu bytes", workspace_bytes, need);
  MVSF_REQUIRE(((uintptr_t)workspace & 15) == 0 && ((uintptr_t)wts & 15) == 0, "fmt: pointers must be 16-byte aligned");
  cudaStream_t s = (cudaStream_t)stream;
  const int L = H1 * W1;
  const size_t VL = (size_t)V * L;
  float* base = (float*)workspace;
  FmtWs ws;
  ws.xn2 = reinterpret_cast<__half*>(base);                  // [V*L][128] halves (= 64 floats / token)
  ws.qkv = base + 64 * VL;                                   // [V*L][192]
  ws.att2 = reinterpret_cast<__half*>(ws.qkv + 192 * VL);    // [V*L][128] halves
  ws.hid2 = ws.att2 + 128 * VL;                              // [V*L][512] halves  (576 VL floats in total; the pathway reuses 640 VL)
  ws.wh = reinterpret_cast<const __half*>(wts16);
  ws.wl = ws.wh + n_wts;
  ws.ref0 = base + 640 * VL;          // [L][64]
  const size_t nblk = (L + KV_CHUNK - 1) / KV_CHUNK;
  ws.kvpart = ws.ref0 + 64 * (size_t)L;
  ws.kvfin = ws.kvpart + (size_t)V * nblk * KVSZ;
  ws.kvc = ws.kvfin + (size_t)V * KVSZ;   // [2][KVSZ]

  MVSF_REQUIRE(V <= 65535, "fmt: too many views");
  tokens_add_pe_kernel<<<dim3(cdiv(L, 32), 2, V), dim3(32, 8), 0, s>>>(f1, pe, o1, L);
  MVSF_LAUNCH_CHECK("fmt_tokens_add_pe");

  const float* b0 = wts; const float* b1 = wts + B_SIZE; const float* b2 = wts + 2 * B_SIZE; const float* b3 = wts + 3 * B_SIZE;
  // reference view: the two self layers (FMT.py:96-107); keep the output of the first one for cross layer 1
  if ((rc = run_block(o1, 1, L, b0, 0, nullptr, ws, s, false, b2))) return rc;
  MVSF_CUDA_OK(cudaMemcpyAsync(ws.ref0, o1, (size_t)L * 64 * sizeof(float), cudaMemcpyDeviceToDevice, s));
  if ((rc = run_block(o1, 1, L, b2, 2 * (size_t)B_SIZE, nullptr, ws, s, true, nullptr))) return rc;
  if ((rc = run_cross_kv(ws.ref0, L, b1, (size_t)B_SIZE, ws.kvc, ws, s))) return rc;
  if ((rc = run_cross_kv(o1, L, b3, 3 * (size_t)B_SIZE, ws.kvc + KVSZ, ws, s))) return rc;
  // source views as one batch: self, cross(ref_list[0]), self, cross(ref_list[1])   (FMT.py:119-135)
  float* xs = o1 + (size_t)L * 64;
  if ((rc = run_block(xs, V - 1, L, b0, 0, nullptr, ws, s, false, b1))) return rc;
  if ((rc = run_block(xs, V - 1, L, b1, (size_t)B_SIZE, ws.kvc, ws, s, true, b2))) return rc;
  if ((rc = run_block(xs, V - 1, L, b2, 2 * (size_t)B_SIZE, nullptr, ws, s, true, b3))) return rc;
  if ((rc = run_block(xs, V - 1, L, b3, 3 * (size_t)B_SIZE, ws.kvc + KVSZ, ws, s, true, nullptr))) return rc;

  // top-down pathway (FMT.py:195-197), all views batched
  float* red = base;                  // <= 128 VL floats
  float* pre = base + 128 * VL;       // <= 512 VL floats
  if ((rc = run_pathway_level<64, 32>(o1, f2, wts + P_DR1, wts + P_SM1, red, pre, o2, V, H1, W1, s))) return rc;
  if ((rc = run_pathway_level<32, 16>(o2, f3, wts + P_DR2, wts + P_SM2, red, pre, o3, V, 2 * H1, 2 * W1, s))) return rc;
  if ((rc = run_pathway_level<16, 8>(o3, f4, wts + P_DR3, wts + P_SM3, red, pre, o4, V, 4 * H1, 4 * W1, s))) return rc;
  return MVSF_OK;
}
}
