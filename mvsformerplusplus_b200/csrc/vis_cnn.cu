// W4 visibility CNN: models/cost_volume.py:37,93
//   ConvBnReLU(1,16) -> ConvBnReLU(16,16) -> ConvBnReLU(16,8) -> Conv1x1(8,1) -> Sigmoid      (BN folded, fp32-class)
// One fused, persistent kernel; a CTA works on 14 x 30 output tiles and never writes the 16-channel intermediates to HBM
// (HBM traffic = 4 B in + 4 B out per pixel).
//   layer 1 (1 -> 16, 144 FMA / pixel)  SIMT over the 18 x 34 halo region; the result is stored as fp16 hi|lo VOXEL-OCTET
//                                       PLANES in shared memory (plane[row][col] = 8 channels = 16 B), the layout in
//                                       which a 3x3 tap is just another UMMA descriptor start address (see conv3d_tc.cu)
//   layer 2 (16 -> 16) and 3 (16 -> 8)  implicit GEMMs on tcgen05: M-tile = 16 rows x 8 columns of pixels, N = 16, K = 16
//                                       channels; per tap two MMAs: x_hi x [w_hi | w_lo] (N = 32, both products side by
//                                       side) and x_lo x w_hi (N = 16, accumulated onto the first), fp32 accumulators in
//                                       TMEM (a small-N tcgen05.mma costs ~50 clk whatever N is: fewer, wider MMAs); the layer-2 epilogue (bias, ReLU, zero outside the
//                                       image = layer 3's padding) writes the planes of layer 3's input
//   layer 4 + sigmoid                   in the layer-3 epilogue (one TMEM lane = one pixel per thread)
// The 16 x 32 region of layer 2 and the 14 x 30 tile of layer 3 are both covered by four 16 x 8 M-tiles; rows / columns of
// an M-tile that fall outside the useful region read the zero border of the plane buffers and are discarded.
// Two CTAs per SM (101 KB of shared memory each) overlap one CTA's SIMT phases with the other's MMAs.
// The fp32 SIMT version this replaces ran at 48 % of the FMA peak (1.9 ms per DTU depth map).
#include "common.cuh"
#include "linear_tc.cuh"
#include "umma.cuh"

namespace mvsf {

using namespace umma;

namespace vc {
constexpr int TH = 14, TW = 30;                 // output tile
constexpr int PR = 18, PC = 34;                 // plane rows / columns (a1: all valid; a2: 16 x 32 valid, rest zero)
constexpr uint32_t PLANE = PR * PC * 16;        // 9792 B: one octet of channels, hi or lo
constexpr uint32_t PITCH = PC * 16;
constexpr int IN_R = 20, IN_C = 36;             // input region (3-pixel halo)
// packed weights (floats): w1[9][16] b1[16] w2[16][9][16] b2[16] w3[16][9][8] b3[8] w4[8] b4[1]
constexpr int OFF_W2 = 160, OFF_B2 = 160 + 2304, OFF_W3 = OFF_B2 + 16,
              OFF_B3 = OFF_W3 + 1152, OFF_W4 = OFF_B3 + 8, OFF_B4 = OFF_W4 + 8;
// shared memory (bytes): planes a1 [hi o0 | hi o1 | lo o0 | lo o1], planes a2, weight tiles, input, small params, barrier
constexpr uint32_t OFF_A1 = 0, OFF_A2 = 4 * PLANE, OFF_B2T = 8 * PLANE, BT_LAYER = 9 * 1024,      // [tap][2 kc][32 rows: w_hi | w_lo][8]
                   OFF_B3T = OFF_B2T + BT_LAYER, OFF_IN = OFF_B3T + BT_LAYER, OFF_PAR = OFF_IN + IN_R * IN_C * 4,
                   OFF_BAR = OFF_PAR + 1024, SMEM = OFF_BAR + 32;
// small parameter block (floats): w1[144] b1[16] b2[16] b3[8] w4[8] b4[1]
constexpr int P_W1 = 0, P_B1 = 144, P_B2 = 160, P_B3 = 176, P_W4 = 184, P_B4 = 192;
}  // namespace vc

// Layer-2/3 activations stay fp16 hi + lo.  Rounding them to fp16 once (x_hi x [w_hi | w_lo] only: half the MMAs, 0.26 ms
// less per DTU depth map) was measured and removed: 1.4e-4..4.6e-4 on the visibility weight, 1.3e-4 on the stage-4
// probability at the full DTU size, outside the 1e-4 bar.
__global__ void __launch_bounds__(256, 2)
vis_cnn_kernel(const float* __restrict__ entropy, const float* __restrict__ wts, float* __restrict__ vis, int H, int W,
               int tiles_x, int tiles_y, int ntiles) {
  using namespace vc;
  extern __shared__ __align__(128) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sb = smem_u32(smem);
  float* in_s = reinterpret_cast<float*>(smem + OFF_IN);
  float* par = reinterpret_cast<float*>(smem + OFF_PAR);
  const uint32_t bar = sb + OFF_BAR;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + OFF_BAR + 16);

  // ---- once per CTA: parameters, fp16 hi|lo weight tiles in the canonical K-major B layout, zero border of a2
  for (int i = tid; i < 160; i += 256) par[i] = __ldg(wts + i);                      // w1, b1
  if (tid < 16) par[P_B2 + tid] = __ldg(wts + OFF_B2 + tid);
  if (tid < 8) { par[P_B3 + tid] = __ldg(wts + OFF_B3 + tid); par[P_W4 + tid] = __ldg(wts + OFF_W4 + tid); }
  if (tid == 0) par[P_B4] = __ldg(wts + OFF_B4);
  for (int i = tid; i < 2 * 9 * 2 * 16 * 8; i += 256) {   // (layer, tap, k-chunk, row n, e) -> hi and lo tiles
    const int e = i & 7, n = (i >> 3) & 15, kc = (i >> 7) & 1, tap = (i >> 8) % 9, layer = i / (9 * 256);
    const int ci = kc * 8 + e;
    float w = 0.f;
    if (layer == 0) w = __ldg(wts + OFF_W2 + (ci * 9 + tap) * 16 + n);
    else if (n < 8) w = __ldg(wts + OFF_W3 + (ci * 9 + tap) * 8 + n);
    const __half hi = __float2half_rn(w), lo = __float2half_rn(w - __half2float(hi));
    __half* t = reinterpret_cast<__half*>(smem + (layer ? OFF_B3T : OFF_B2T) + tap * 1024);
    t[kc * 256 + n * 8 + e] = hi;
    t[kc * 256 + (16 + n) * 8 + e] = lo;
  }
  for (int i = tid; i < (int)(4 * PLANE / 16); i += 256) reinterpret_cast<uint4*>(smem + OFF_A2)[i] = make_uint4(0, 0, 0, 0);
  if (tid == 0) { mbar_init(bar, 1); fence_barrier_init(); }
  if (warp == 0) tmem_alloc(sb + OFF_BAR + 16, 256);
  fence_proxy_async();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t el = elect_one();
  constexpr uint32_t a_hi = desc_hi(PITCH), b_hi = desc_hi(128);
  const uint32_t idesc16 = make_idesc_f16(128, 16), idesc32 = make_idesc_f16(128, 32);
  uint32_t phase = 0;

  // MMAs of one 3x3 layer over the four M-tiles: planes at `pl`, weight tiles at `bt`, accumulators at TMEM column `col`
  auto issue_layer = [&](uint32_t pl, uint32_t bt, uint32_t col) {
#pragma unroll
    for (int kh = 0; kh < 3; ++kh) {
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        const uint32_t aoff = (uint32_t)(kh * PC + kw) * 16u;
        const uint32_t ah = desc_lo(pl + aoff, PLANE), al = desc_lo(pl + 2 * PLANE + aoff, PLANE);   // K = two octets
        const uint32_t wb = desc_lo(bt + (kh * 3 + kw) * 1024, 512);
        const uint32_t acc = (kh | kw) ? 1u : 0u;
        // accumulator columns of M-tile ct: [32 ct, +16) = x_hi w_hi + x_lo w_hi, [32 ct + 16, +16) = x_hi w_lo
#pragma unroll
        for (int ct = 0; ct < 4; ++ct) mma_f16_ss_lh(el, tmem_base + col + ct * 32, ah + ct * 8, a_hi, wb, b_hi, idesc32, acc);
#pragma unroll
        for (int ct = 0; ct < 4; ++ct) mma_f16_ss_lh(el, tmem_base + col + ct * 32, al + ct * 8, a_hi, wb, b_hi, idesc16, 1u);
      }
    }
    commit_el(el, bar);
  };

  // epilogue geometry: warp w reads TMEM lanes 32 (w % 4) ..., warps 0-3 take M-tiles 0 and 1, warps 4-7 M-tiles 2 and 3
  const int quarter = warp & 3, m = quarter * 32 + lane;
  const int er = m >> 3, ec0 = (warp >> 2) * 16 + (m & 7);     // row and first column (second M-tile: + 8)
  const uint32_t trow = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)((warp >> 2) * 64);

  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int tx = tile % tiles_x, ty = (tile / tiles_x) % tiles_y, n = tile / (tiles_x * tiles_y);
    const int x0 = tx * TW, y0 = ty * TH;
    const float* __restrict__ E = entropy + (size_t)n * H * W;
    // ---- input region (zero outside the image: layer 1's padding)
    for (int i = tid; i < IN_R * IN_C; i += 256) {
      const int r = i / IN_C, c = i - r * IN_C;
      const int gy = y0 - 3 + r, gx = x0 - 3 + c;
      in_s[i] = (gy >= 0 && gy < H && gx >= 0 && gx < W) ? __ldg(E + (size_t)gy * W + gx) : 0.0f;
    }
    __syncthreads();
    // ---- layer 1 on the 18 x 34 region -> planes a1 (zero outside the image: layer 2's padding)
    for (int i = tid; i < PR * PC; i += 256) {
      const int r = i / PC, c = i - r * PC;
      const int gy = y0 - 2 + r, gx = x0 - 2 + c;
      const bool inside = gy >= 0 && gy < H && gx >= 0 && gx < W;
      float acc[16];
#pragma unroll
      for (int oc = 0; oc < 16; ++oc) acc[oc] = par[P_B1 + oc];
#pragma unroll
      for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const float v = in_s[(r + ky) * IN_C + c + kx];
          const float* wp = par + P_W1 + (ky * 3 + kx) * 16;
#pragma unroll
          for (int oc = 0; oc < 16; ++oc) acc[oc] = fmaf(v, wp[oc], acc[oc]);
        }
#pragma unroll
      for (int oc = 0; oc < 16; ++oc) acc[oc] = inside ? fmaxf(acc[oc], 0.0f) : 0.0f;
      __half* p = reinterpret_cast<__half*>(smem + OFF_A1 + (uint32_t)i * 16u);
      const float (&lo8)[8] = reinterpret_cast<const float (&)[8]>(acc[0]);
      const float (&hi8)[8] = reinterpret_cast<const float (&)[8]>(acc[8]);
      // p is a __half*: + PLANE / 2 elements = + PLANE bytes.  Planes: [hi o0 | hi o1 | lo o0 | lo o1]
      split_store8(p, p + PLANE, lo8);                           // channels 0-7 : hi -> plane 0, lo -> plane 2
      split_store8(p + PLANE / 2, p + PLANE / 2 + PLANE, hi8);   // channels 8-15: hi -> plane 1, lo -> plane 3
    }
    fence_proxy_async();
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) { tc_fence_after_sync(); issue_layer(sb + OFF_A1, sb + OFF_B2T, 0u); }
    // ---- layer-2 epilogue: bias, ReLU, zero outside the image -> planes a2 (16 x 32 region anchored at row 0, column 0)
    mbar_wait(bar, phase);
    phase ^= 1u;
    tc_fence_after_sync();
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      float v[16], v2[16];
      tmem_ld16(trow + k * 32, v);
      tmem_ld16(trow + k * 32 + 16, v2);
#pragma unroll
      for (int oc = 0; oc < 16; ++oc) v[oc] += v2[oc];
      const int c = ec0 + k * 8;
      const int gy = y0 - 1 + er, gx = x0 - 1 + c;
      const bool inside = gy >= 0 && gy < H && gx >= 0 && gx < W;
#pragma unroll
      for (int oc = 0; oc < 16; ++oc) v[oc] = inside ? fmaxf(v[oc] + par[P_B2 + oc], 0.0f) : 0.0f;
      __half* p = reinterpret_cast<__half*>(smem + OFF_A2 + (uint32_t)(er * PC + c) * 16u);
      const float (&lo8)[8] = reinterpret_cast<const float (&)[8]>(v[0]);
      const float (&hi8)[8] = reinterpret_cast<const float (&)[8]>(v[8]);
      split_store8(p, p + PLANE, lo8);
      split_store8(p + PLANE / 2, p + PLANE / 2 + PLANE, hi8);
    }
    fence_proxy_async();
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) { tc_fence_after_sync(); issue_layer(sb + OFF_A2, sb + OFF_B3T, 128u); }
    // ---- layer-3 epilogue: bias, ReLU, 1x1 conv, sigmoid
    mbar_wait(bar, phase);
    phase ^= 1u;
    tc_fence_after_sync();
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      float v[16], v2[16];
      tmem_ld16(trow + 128 + k * 32, v);
      tmem_ld16(trow + 128 + k * 32 + 16, v2);
#pragma unroll
      for (int oc = 0; oc < 8; ++oc) v[oc] += v2[oc];
      const int ox = ec0 + k * 8;
      const int gy = y0 + er, gx = x0 + ox;
      if (er < TH && ox < TW && gy < H && gx < W) {
        float s = par[P_B4];
#pragma unroll
        for (int oc = 0; oc < 8; ++oc) s = fmaf(fmaxf(v[oc] + par[P_B3 + oc], 0.f), par[P_W4 + oc], s);
        vis[((size_t)n * H + gy) * W + gx] = __fdiv_rn(1.0f, 1.0f + expf(-s));
      }
    }
    tc_fence_before_sync();
    __syncthreads();   // a1, the input tile and the TMEM columns are free again
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 256);
}

}  // namespace mvsf

using namespace mvsf;

extern "C" int mvsf_vis_cnn(const float* entropy, const float* wts, float* vis, int N, int H, int W,
                            mvsf_stream_t stream) {
  MVSF_REQUIRE(entropy && wts && vis && N > 0 && N <= 65535 && H > 0 && W > 0, "vis_cnn: bad arguments");
  static DeviceOnce once;
  const int dev = current_device();
  const int num_sms = device_sm_count(dev);
  if (once.need(dev)) {
    MVSF_CUDA_OK(cudaFuncSetAttribute(vis_cnn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)vc::SMEM));
    once.done(dev);
  }
  const int tiles_x = cdiv(W, vc::TW), tiles_y = cdiv(H, vc::TH);
  const long long ntiles = (long long)tiles_x * tiles_y * N;
  MVSF_REQUIRE(ntiles < (1ll << 30), "vis_cnn: image too large");
  const int grid = (int)(ntiles < 2 * num_sms ? ntiles : 2 * num_sms);
  vis_cnn_kernel<<<grid, 256, vc::SMEM, (cudaStream_t)stream>>>(entropy, wts, vis, H, W, tiles_x, tiles_y, (int)ntiles);
  MVSF_LAUNCH_CHECK("vis_cnn");
  return MVSF_OK;
}
