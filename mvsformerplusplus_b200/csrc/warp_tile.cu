// W2+W3+W4 for the fine stages (C = 8 / 16 feature channels): homography warp fused with group-wise correlation
// (models/warping.py:69-109, models/cost_volume.py:72-101) around TMA-staged source windows in shared memory.
//
// Why a second organisation next to warp_corr.cu: with 8 or 16 channels one bilinear corner is only 32 / 64 bytes, so a
// warp-wide global gather touches 16 / 8 different 128-byte lines per instruction and runs at 25-50 % of the L1
// wavefront rate, and the taps of neighbouring pixels are NOT coherent at stages 2-4 (the hypothesis planes follow the
// previous stage's per-pixel depth).  Here
//   * a CTA owns a tile of reference pixels; per (source view, chunk of <= 8 hypotheses) it computes its tap
//     coordinates, reduces their bounding box, and one thread issues ONE cp.async.bulk.tensor (TMA) box load of the
//     source footprint: a 5-D view (c, y-parity, x, y/2, view) of the channels-last feature tensor, so the window lands
//     in shared memory as [y/2][x][y&1][C] and everything outside the image is zero-filled by the TMA unit
//     (= grid_sample's padding_mode='zeros', no per-corner masking);
//   * every lane then owns whole taps: the 4 corners x 8 channels of a tap are 8 pieces of 16 bytes that, in this
//     layout, fall on 8 DIFFERENT 16-byte bank groups whatever the tap position is; lane l reads them in the order
//     (round i) bank group = i XOR (l mod 8), so the 8 lanes of every LDS.128 phase hit 8 different bank groups:
//     conflict-free shared-memory gathers at 128 B/clk/SM for arbitrary (incoherent) tap positions.  Which corner a
//     round delivers depends on the tap's x/y parity; that is folded into per-tap swaps of the two x / y weights and
//     base addresses (lane-constant predicates), so the 8 rounds themselves are straight-line code;
//   * taps outside the staged window (depth outliers) fall back to global loads for that lane only.
// Measured on B200 (DTU stage 4, 28.3 M taps per pass; DESIGN.md "warp + correlation" has the full table): pass A 0.37 ms,
// pass B 0.42 ms - faster than the L1-gather kernels doing the same two gathers (0.43 / 0.50 ms), 28 % faster on the
// plane-sweep microbenchmark, but slower than warp_corr.cu's spill plan (gather once, stream the stored correlations:
// 0.51 + 0.19 ms), which therefore stays the default of the cascade; these kernels serve the two-gather plan (plane sweeps,
// spill buffers over budget).  A variant that staged the window rows with cp.async.bulk (2-4 KB requests, odd row pitch)
// instead of the tensor box measured slower (0.58 / 0.69 ms); with D = 4..8 taps per lane and window the per-window
// skeleton (coordinates, bounding box, CTA barrier, staging latency) costs more than the conflict-free gather itself.
#include <cuda.h>
#include <float.h>
#include <limits.h>

#include "umma.cuh"

namespace mvsf {
namespace wt {
using namespace umma;

constexpr int TW = 32, THREADS = 256;   // reference-pixel tile: 32 columns, one warp per tile row
constexpr int kMaxD = 512;
// resident CTAs per SM of the C = 8 pipeline kernel and its ring of windows of 32 KB each; measured at DTU stage 4:
// 2 CTAs x 3 windows 0.367 ms, 3 CTAs x 2 windows 0.444 ms
constexpr int kPsBlocks8 = 2, kPsNbuf8 = 3;
constexpr int kPassBBlocks8 = 3;   // resident CTAs per SM of the C = 8, D <= 4 aggregation kernel (3 costs ~20 spilled registers)
// the pipeline kernel serves a pass-A call when at most this many of every 1000 sampled in-bound taps miss its windows
// (DTU stage 4: 28, pipeline faster; Tanks&Temples: 287, L1-gather kernel faster; see warp_stream_select_kernel)
constexpr int kMaxWindowMissPermille = 60;

template <int C>
struct Cfg {
  static constexpr int LPX = C / 8;                  // lanes per pixel: every lane owns 8 channels of a tap
  static constexpr int PIX = THREADS / LPX;          // pixels per CTA
  static constexpr int TROWS = PIX / TW;             // tile rows
  static constexpr int WX = 64, WY = 16;             // staged window (source texels); WY even
  static constexpr int POS = 2 * C * 4;              // bytes of one window position [y&1][C]
  static constexpr int P = WX * POS;                 // pitch of one row pair
  static constexpr uint32_t BYTES = (WY / 2) * P;    // 32 KB (C = 8), 64 KB (C = 16)
};

__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
// acc (4 channels) += w * t, as two packed fp32x2 FMAs (FFMA2: one issue slot per two FMAs)
__device__ __forceinline__ void fma4(float4& acc, float w, const float4& t) {
  const float2 ww = make_float2(w, w);
  float2 lo = __ffma2_rn(make_float2(t.x, t.y), ww, make_float2(acc.x, acc.y));
  float2 hi = __ffma2_rn(make_float2(t.z, t.w), ww, make_float2(acc.z, acc.w));
  acc = make_float4(lo.x, lo.y, hi.x, hi.y);
}
__device__ __forceinline__ float dot4(const float4& a, const float4& b) { return fmaf(a.w, b.w, fmaf(a.z, b.z, fmaf(a.y, b.y, a.x * b.x))); }

// per-lane constants of the rotated read order
struct Lane {
  bool b0, b1, b2;      // bits of (lane & 7) that are XORed into the bank-group index of a round
  uint32_t base[2];     // window base + 16-byte piece offset for rounds with i0 = 0 / 1
};
// Read order of a consumer lane that owns 8-channel slice `sub` of its pixel, with base[] relative to the window (the caller
// adds the window address), and the first channel of the lane's quad A / quad B.
template <int C>
__device__ __forceinline__ Lane make_lane(int lane, int sub, int& chA, int& chB) {
  Lane L;
  if (C == 8) {
    L.b0 = lane & 1; L.b1 = (lane >> 1) & 1; L.b2 = (lane >> 2) & 1;
    L.base[0] = L.b0 ? 16 : 0;
    L.base[1] = L.b0 ? 0 : 16;
    chA = L.b0 ? 4 : 0; chB = L.b0 ? 0 : 4;
  } else {
    // lanes 2j, 2j+1 = the two channel halves of one pixel; bits 1-2 of the lane = tap slot inside an LDS.128 phase
    L.b0 = false; L.b1 = (lane >> 1) & 1; L.b2 = (lane >> 2) & 1;
    const int q0 = 2 * sub + (L.b1 ? 1 : 0), q1 = 2 * sub + (L.b1 ? 0 : 1);
    L.base[0] = q0 * 16;
    L.base[1] = q1 * 16;
    chA = q0 * 4; chB = q1 * 4;
  }
  return L;
}

// One tap (4 corners x 8 channels of this lane) from the staged window: sA / sB receive the bilinear sample of the lane's
// two channel quads (quad A = the one read in rounds with i0 = 0).  (lx, ly) = integer tap position relative to the window
// origin (both rows / columns inside the window), (fx, fy) = fractional parts.
// C = 8 : position = [y&1][8 ch] = 64 B; 16-byte bank group of a piece = (x&1)<<2 | (y&1)<<1 | quad.
// C = 16: position = [y&1][16 ch] = 128 B (one line); bank group = (y&1)<<2 | channel quarter; a lane owns quarters
//         {2k, 2k+1} (k = lane & 1 is the "b0" group bit here, the x corner is a compile-time round bit).
template <int C>
__device__ __forceinline__ void gather_window(const Lane& L, int lx, int ly, float fx, float fy, float4& sA, float4& sB) {
  using K = Cfg<C>;
  const float gx = 1.0f - fx, gy = 1.0f - fy;
  const bool yodd = ly & 1;
  // byte offsets (window-relative) of the even-parity and odd-parity source row of this tap
  const uint32_t rE = (uint32_t)((ly + 1) >> 1) * K::P;
  const uint32_t rO = (uint32_t)(ly >> 1) * K::P + C * 4;
  const float wE = yodd ? fy : gy, wO = yodd ? gy : fy;   // weight of the even / odd row
  if (C == 8) {
    const bool xodd = lx & 1;
    const uint32_t cE = (uint32_t)((lx + 1) & ~1) * K::POS, cO = (uint32_t)(lx | 1) * K::POS;
    const float vE = xodd ? fx : gx, vO = xodd ? gx : fx;  // weight of the even / odd column
    // rounds: i2 selects the x parity (XOR b2), i1 the y parity (XOR b1), i0 the channel quad (XOR b0, folded in base[])
    const uint32_t X0 = L.b2 ? cO : cE, X1 = L.b2 ? cE : cO;
    const float wx0 = L.b2 ? vO : vE, wx1 = L.b2 ? vE : vO;
    const uint32_t R0 = L.b1 ? rO : rE, R1 = L.b1 ? rE : rO;
    const float wy0 = L.b1 ? wO : wE, wy1 = L.b1 ? wE : wO;
    const float w00 = wx0 * wy0, w01 = wx0 * wy1, w10 = wx1 * wy0, w11 = wx1 * wy1;
    const float4 a0 = lds128(X0 + R0 + L.base[0]), b0 = lds128(X0 + R0 + L.base[1]);
    const float4 a1 = lds128(X0 + R1 + L.base[0]), b1 = lds128(X0 + R1 + L.base[1]);
    const float4 a2 = lds128(X1 + R0 + L.base[0]), b2 = lds128(X1 + R0 + L.base[1]);
    const float4 a3 = lds128(X1 + R1 + L.base[0]), b3 = lds128(X1 + R1 + L.base[1]);
    fma4(sA, w00, a0); fma4(sB, w00, b0);
    fma4(sA, w01, a1); fma4(sB, w01, b1);
    fma4(sA, w10, a2); fma4(sB, w10, b2);
    fma4(sA, w11, a3); fma4(sB, w11, b3);
  } else {
    // C == 16: x corner = compile-time (both columns are whole lines), y parity XOR b2, low quarter bit XOR b1
    const uint32_t c0 = (uint32_t)lx * K::POS;
    const uint32_t R0 = (L.b2 ? rO : rE) + c0, R1 = (L.b2 ? rE : rO) + c0;
    const float wy0 = L.b2 ? wO : wE, wy1 = L.b2 ? wE : wO;
    const float w00 = gx * wy0, w01 = gx * wy1, w10 = fx * wy0, w11 = fx * wy1;
    const float4 a0 = lds128(R0 + L.base[0]), b0 = lds128(R0 + L.base[1]);
    const float4 a1 = lds128(R1 + L.base[0]), b1 = lds128(R1 + L.base[1]);
    const float4 a2 = lds128(R0 + L.base[0] + K::POS), b2 = lds128(R0 + L.base[1] + K::POS);
    const float4 a3 = lds128(R1 + L.base[0] + K::POS), b3 = lds128(R1 + L.base[1] + K::POS);
    fma4(sA, w00, a0); fma4(sB, w00, b0);
    fma4(sA, w01, a1); fma4(sB, w01, b1);
    fma4(sA, w10, a2); fma4(sB, w10, b2);
    fma4(sA, w11, a3); fma4(sB, w11, b3);
  }
}

// same tap through global memory (zero padding by masked weights, as warp_corr.cu): the rare out-of-window taps
template <int C>
__device__ __forceinline__ void gather_global(const float* __restrict__ srcA, const float* __restrict__ srcB, float ix, float iy,
                                              int W, int H, float4& sA, float4& sB) {
  int4 off;
  float4 wt;
  make_tap_fast(ix, iy, W, H, C, off, wt);
  fma4(sA, wt.x, ldg4(srcA + off.x)); fma4(sB, wt.x, ldg4(srcB + off.x));
  fma4(sA, wt.y, ldg4(srcA + off.y)); fma4(sB, wt.y, ldg4(srcB + off.y));
  fma4(sA, wt.z, ldg4(srcA + off.z)); fma4(sB, wt.z, ldg4(srcB + off.z));
  fma4(sA, wt.w, ldg4(srcA + off.w)); fma4(sB, wt.w, ldg4(srcB + off.w));
}

struct TapCoord {
  float fx, fy;
  int x0, y0;
  bool inb;   // sample position inside (-1, W) x (-1, H): otherwise every corner is outside the image -> contributes 0
};
__device__ __forceinline__ TapCoord split_coord(float ix, float iy, int W, int H) {
  TapCoord t;
  t.inb = (ix > -1.0f) && (ix < (float)W) && (iy > -1.0f) && (iy < (float)H);   // false for NaN / Inf
  const float sx = t.inb ? ix : 0.0f, sy = t.inb ? iy : 0.0f;
  const float MAGIC = 12582912.0f;   // 1.5 * 2^23: round-down add = floor (|s| < 2^22)
  const float tx = __fadd_rd(sx, MAGIC), ty = __fadd_rd(sy, MAGIC);
  t.x0 = __float_as_int(tx) - 0x4B400000;
  t.y0 = __float_as_int(ty) - 0x4B400000;
  t.fx = sx - (tx - MAGIC);
  t.fy = sy - (ty - MAGIC);
  return t;
}

// Origin (ox, oy even) of the WX x WY window centred on the bounding box [mnx, mxx] x [mny, mxy] of tap positions; (0, 0)
// for an empty box.
template <int C>
__device__ __forceinline__ void window_origin(int mnx, int mxx, int mny, int mxy, int& ox, int& oy) {
  using K = Cfg<C>;
  ox = 0;
  oy = 0;
  if (mnx <= mxx) {
    const int slack_x = K::WX - (mxx + 2 - mnx), slack_y = K::WY - (mxy + 2 - mny);
    ox = mnx - (slack_x > 0 ? slack_x / 2 : 0);
    oy = (mny - (slack_y > 0 ? slack_y / 2 : 0)) & ~1;
  }
}
// The pipeline kernel's window for one (tile, view), predicted by a whole warp: each lane contributes the taps of its sample
// pixel at the first and the last hypothesis.  The producer warp and warp_stream_select_kernel both call this, so the
// selection replays the producer's windows exactly.
template <int C>
__device__ __forceinline__ void predict_window(const TapCoord& first, const TapCoord& last, int& ox, int& oy) {
  int mnx = INT_MAX, mxx = INT_MIN, mny = INT_MAX, mxy = INT_MIN;
  if (first.inb) { mnx = min(mnx, first.x0); mxx = max(mxx, first.x0); mny = min(mny, first.y0); mxy = max(mxy, first.y0); }
  if (last.inb) { mnx = min(mnx, last.x0); mxx = max(mxx, last.x0); mny = min(mny, last.y0); mxy = max(mxy, last.y0); }
  mnx = __reduce_min_sync(0xffffffffu, mnx);
  mxx = __reduce_max_sync(0xffffffffu, mxx);
  mny = __reduce_min_sync(0xffffffffu, mny);
  mxy = __reduce_max_sync(0xffffffffu, mxy);
  window_origin<C>(mnx, mxx, mny, mxy, ox, oy);
}

struct Shared {
  unsigned long long bar;
  int bbox[2][4];   // double-buffered {min x0, max x0, min y0, max y0} of the current window's taps
};

// Stages one window: reduces the bounding box of the CTA's taps, centres the WX x WY box on it, issues the TMA load and
// waits for it.  Returns the window origin (ox, oy even) to every thread.  `slot` alternates per call.
template <int C>
__device__ __forceinline__ void stage_window(const CUtensorMap* map, Shared& sh, uint32_t win, int slot, uint32_t& phase, int view,
                                             int mnx, int mxx, int mny, int mxy, int& ox, int& oy) {
  using K = Cfg<C>;
  mnx = __reduce_min_sync(0xffffffffu, mnx);
  mxx = __reduce_max_sync(0xffffffffu, mxx);
  mny = __reduce_min_sync(0xffffffffu, mny);
  mxy = __reduce_max_sync(0xffffffffu, mxy);
  if ((threadIdx.x & 31) == 0) {
    atomicMin(&sh.bbox[slot][0], mnx);
    atomicMax(&sh.bbox[slot][1], mxx);
    atomicMin(&sh.bbox[slot][2], mny);
    atomicMax(&sh.bbox[slot][3], mxy);
  }
  __syncthreads();   // bbox complete; every lane has also finished reading the previous window
  window_origin<C>(sh.bbox[slot][0], sh.bbox[slot][1], sh.bbox[slot][2], sh.bbox[slot][3], ox, oy);
  if (threadIdx.x == 0) {
    sh.bbox[slot ^ 1][0] = INT_MAX; sh.bbox[slot ^ 1][1] = INT_MIN;   // reset the other slot for the next window
    sh.bbox[slot ^ 1][2] = INT_MAX; sh.bbox[slot ^ 1][3] = INT_MIN;
    const uint32_t bar = smem_u32(&sh.bar);
    expect_tx(bar, K::BYTES);
    tma_load_5d(win, map, 0, 0, ox, oy >> 1, view, bar);
  }
  mbar_wait_warp(smem_u32(&sh.bar), phase);
  phase ^= 1;
}

// Everything a lane needs to sample source view `view` for its pixel.
template <int C>
struct ViewCtx {
  Hom m;
  float rx, ry, rz;
  const float* srcA;
  const float* srcB;
};

// One (view, hypothesis chunk [d0, d0 + n)) of this lane's pixel: tap coordinates, window staging, gather.
// consume(k, sA, sB) receives the bilinear sample of hypothesis d0 + k (quad A / quad B channels of the lane).
// The bounding box is taken from the first and last hypothesis of the chunk: taps of one pixel lie on its epipolar line
// and move monotonically with the (monotone) hypotheses, so those two bound the rest; a tap that still falls outside the
// window (non-monotone caller-supplied hypotheses, depth outliers of neighbours) goes through global memory.
template <int C, int DCHT, typename F>
__device__ __forceinline__ void process_chunk(const CUtensorMap* map, Shared& sh, uint32_t win, int& slot, uint32_t& phase,
                                              const Lane& L, const ViewCtx<C>& vc, int view, const float* __restrict__ depth_p,
                                              int HW, int d0, int n, bool active, const CoordConst& cc, int W, int H, F&& consume) {
  using K = Cfg<C>;
  float ix, iy;
  warp_coord_lean(vc.rx, vc.ry, vc.rz, vc.m, __ldg(depth_p + (size_t)d0 * HW), cc, ix, iy);
  TapCoord tF = split_coord(ix, iy, W, H);
  tF.inb = tF.inb && active;
  TapCoord tL = tF;
  if (n > 1) {
    warp_coord_lean(vc.rx, vc.ry, vc.rz, vc.m, __ldg(depth_p + (size_t)(d0 + n - 1) * HW), cc, ix, iy);
    tL = split_coord(ix, iy, W, H);
    tL.inb = tL.inb && active;
  }
  int mnx = INT_MAX, mxx = INT_MIN, mny = INT_MAX, mxy = INT_MIN;
  if (tF.inb) { mnx = mxx = tF.x0; mny = mxy = tF.y0; }
  if (tL.inb) { mnx = min(mnx, tL.x0); mxx = max(mxx, tL.x0); mny = min(mny, tL.y0); mxy = max(mxy, tL.y0); }
  int ox, oy;
  stage_window<C>(map, sh, win, slot, phase, view, mnx, mxx, mny, mxy, ox, oy);
  slot ^= 1;
#pragma unroll
  for (int k = 0; k < DCHT; ++k) {
    if (k < n) {
      TapCoord t;
      if (k == 0) t = tF;
      else if (k == n - 1) t = tL;
      else {
        warp_coord_lean(vc.rx, vc.ry, vc.rz, vc.m, __ldg(depth_p + (size_t)(d0 + k) * HW), cc, ix, iy);
        t = split_coord(ix, iy, W, H);
        t.inb = t.inb && active;
      }
      float4 sA = make_float4(0.f, 0.f, 0.f, 0.f), sB = sA;
      const int lx = t.x0 - ox, ly = t.y0 - oy;
      const bool inwin = t.inb && (unsigned)lx <= (unsigned)(K::WX - 2) && (unsigned)ly <= (unsigned)(K::WY - 2);
      gather_window<C>(L, inwin ? lx : 0, inwin ? ly : 0, t.fx, t.fy, sA, sB);
      if (!inwin) {
        sA = make_float4(0.f, 0.f, 0.f, 0.f); sB = sA;
        if (t.inb) {   // rare: sample through global memory (coordinates recomputed: they are not kept in registers)
          warp_coord_lean(vc.rx, vc.ry, vc.rz, vc.m, __ldg(depth_p + (size_t)(d0 + k) * HW), cc, ix, iy);
          gather_global<C>(vc.srcA, vc.srcB, ix, iy, W, H, sA, sB);
        }
      }
      consume(k, sA, sB);
    }
  }
}

// ----------------------------------------------------------------------------------------------------------------------
// MODE 0: pass A  -> entropy[v][pixel]      (cost_volume.py:89-92)
// MODE 1: pass B  -> volume[d][pixel][g]    (cost_volume.py:95-101), G = 8 groups
// DCHT: hypotheses per window (4 or 8).  GENERIC (pass A only): D > DCHT, similarities parked in a per-thread array.
// ----------------------------------------------------------------------------------------------------------------------
template <int C, int MODE, int DCHT, bool GENERIC>
__global__ void __launch_bounds__(THREADS, C == 8 && MODE == 0 ? 3 : (C == 8 && DCHT == 4 ? kPassBBlocks8 : 2))
warp_tile_kernel(const __grid_constant__ CUtensorMap map, const float* __restrict__ feat, const float* __restrict__ homs,
                 const float* __restrict__ depth, const float* __restrict__ vis, float* __restrict__ out, int V, int D, int H,
                 int W, int dch) {
  using K = Cfg<C>;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ Shared sh;
  const uint32_t win = (smem_u32(smem_raw) + 127u) & ~127u;
  const int tid = threadIdx.x, lane = tid & 31;
  const int HW = H * W;
  // pixel of this lane: LPX adjacent lanes share a pixel
  const int pix_in_cta = tid / K::LPX;
  const int px = blockIdx.x * TW + (pix_in_cta % TW), py = blockIdx.y * K::TROWS + (pix_in_cta / TW);
  const bool active = (px < W) && (py < H);
  const int p = min(py, H - 1) * W + min(px, W - 1);
  const int sub = tid % K::LPX;           // which 8-channel slice of the pixel
  int chA, chB;
  Lane L = make_lane<C>(lane, sub, chA, chB);
  L.base[0] += win;
  L.base[1] += win;
  if (tid == 0) {
    mbar_init(smem_u32(&sh.bar), 1);
    fence_barrier_init();
    sh.bbox[0][0] = INT_MAX; sh.bbox[0][1] = INT_MIN; sh.bbox[0][2] = INT_MAX; sh.bbox[0][3] = INT_MIN;
    sh.bbox[1][0] = INT_MAX; sh.bbox[1][1] = INT_MIN; sh.bbox[1][2] = INT_MAX; sh.bbox[1][3] = INT_MIN;
  }
  __syncthreads();
  uint32_t phase = 0;
  int slot = 0;
  const CoordConst cc = make_coord_const(W, H);
  const float fxp = (float)min(px, W - 1), fyp = (float)min(py, H - 1);
  const float4 rA = ldg4(feat + (size_t)p * C + chA), rB = ldg4(feat + (size_t)p * C + chB);
  constexpr float inv_cpg = 8.0f / (float)C;   // G / C with G = 8 groups: mean over the channels of a group
  const float* __restrict__ depth_p = depth + p;

  auto make_view = [&](int v) {
    ViewCtx<C> vc;
    vc.m = load_hom(homs + (size_t)v * 12);
    pixel_ray(vc.m, fxp, fyp, vc.rx, vc.ry, vc.rz);
    vc.srcA = feat + (size_t)(v + 1) * HW * C + chA;
    vc.srcB = feat + (size_t)(v + 1) * HW * C + chB;
    return vc;
  };

  if (MODE == 0) {
    // ------------------------------------------------------------------ pass A: views outer, hypothesis chunks inner
    float sims[GENERIC ? kMaxD : DCHT];
    for (int v = 0; v < V - 1; ++v) {
      const ViewCtx<C> vc = make_view(v);
      float mx = -FLT_MAX;
      for (int d0 = 0; d0 < D; d0 += dch) {
        const int n = min(dch, D - d0);
        process_chunk<C, DCHT>(&map, sh, win, slot, phase, L, vc, v + 1, depth_p, HW, d0, n, active, cc, W, H,
                               [&](int k, const float4& sA, const float4& sB) {
                                 float s = dot4(rA, sA) + dot4(rB, sB);
                                 if (K::LPX == 2) s += __shfl_xor_sync(0xffffffffu, s, 1);
                                 s *= inv_cpg;
                                 sims[GENERIC ? d0 + k : k] = s;
                                 mx = fmaxf(mx, s);
                               });
        if (!GENERIC) break;
      }
      // softmax over D -> entropy (cost_volume.py:90-92): p = exp(s - max) / Z ; H = -sum p * log(p + 1e-7)
      float Z = 0.f, ent = 0.f;
      if (GENERIC) {
        for (int d = 0; d < D; ++d) { sims[d] = expf(sims[d] - mx); Z += sims[d]; }
        for (int d = 0; d < D; ++d) { const float pr = __fdiv_rn(sims[d], Z); ent -= pr * logf(pr + 1e-7f); }
      } else {
#pragma unroll
        for (int k = 0; k < DCHT; ++k)
          if (k < D) { sims[k] = expf(sims[k] - mx); Z += sims[k]; }
#pragma unroll
        for (int k = 0; k < DCHT; ++k)
          if (k < D) { const float pr = __fdiv_rn(sims[k], Z); ent -= pr * logf(pr + 1e-7f); }
      }
      if (active && sub == 0) out[(size_t)v * HW + p] = ent;
    }
  } else {
    // ------------------------------------------------------------------ pass B: hypothesis chunks outer, views inner
    float wsum = 0.f;
    for (int v = 0; v < V - 1; ++v) wsum = __fadd_rn(wsum, __ldg(vis + (size_t)v * HW + p));
    const float den = __fadd_rn(wsum, 1e-6f);
    // ref * (1 / channels per group): what every warped channel is multiplied with before the visibility weight
    const float4 qA = make_float4(rA.x * inv_cpg, rA.y * inv_cpg, rA.z * inv_cpg, rA.w * inv_cpg);
    const float4 qB = make_float4(rB.x * inv_cpg, rB.y * inv_cpg, rB.z * inv_cpg, rB.w * inv_cpg);
    for (int d0 = 0; d0 < D; d0 += dch) {
      const int n = min(dch, D - d0);
      float4 accA[DCHT], accB[DCHT];
#pragma unroll
      for (int k = 0; k < DCHT; ++k) accA[k] = accB[k] = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int v = 0; v < V - 1; ++v) {
        const ViewCtx<C> vc = make_view(v);
        const float w = __ldg(vis + (size_t)v * HW + p);
        process_chunk<C, DCHT>(&map, sh, win, slot, phase, L, vc, v + 1, depth_p, HW, d0, n, active, cc, W, H,
                               [&](int k, const float4& sA, const float4& sB) {
                                 // group correlation of this view (cost_volume.py:78-85) times its weight (:97)
                                 accA[k].x = fmaf(qA.x * sA.x, w, accA[k].x); accA[k].y = fmaf(qA.y * sA.y, w, accA[k].y);
                                 accA[k].z = fmaf(qA.z * sA.z, w, accA[k].z); accA[k].w = fmaf(qA.w * sA.w, w, accA[k].w);
                                 accB[k].x = fmaf(qB.x * sB.x, w, accB[k].x); accB[k].y = fmaf(qB.y * sB.y, w, accB[k].y);
                                 accB[k].z = fmaf(qB.z * sB.z, w, accB[k].z); accB[k].w = fmaf(qB.w * sB.w, w, accB[k].w);
                               });
      }
      if (active) {
#pragma unroll
        for (int k = 0; k < DCHT; ++k) {
          if (k < n) {
            float* o = out + ((size_t)(d0 + k) * HW + p) * 8;
            if (C == 8) {   // channels == groups
              *reinterpret_cast<float4*>(o + chA) = make_float4(__fdiv_rn(accA[k].x, den), __fdiv_rn(accA[k].y, den),
                                                                __fdiv_rn(accA[k].z, den), __fdiv_rn(accA[k].w, den));
              *reinterpret_cast<float4*>(o + chB) = make_float4(__fdiv_rn(accB[k].x, den), __fdiv_rn(accB[k].y, den),
                                                                __fdiv_rn(accB[k].z, den), __fdiv_rn(accB[k].w, den));
            } else {        // 2 channels per group: a quad is 2 groups
              *reinterpret_cast<float2*>(o + chA / 2) = make_float2(__fdiv_rn(accA[k].x + accA[k].y, den), __fdiv_rn(accA[k].z + accA[k].w, den));
              *reinterpret_cast<float2*>(o + chB / 2) = make_float2(__fdiv_rn(accB[k].x + accB[k].y, den), __fdiv_rn(accB[k].z + accB[k].w, den));
            }
          }
        }
      }
    }
  }
}

// ======================================================================================================================
// Pass A of the SPILL plan for the finest stage (C = 8, D = 4), as a persistent producer / consumer pipeline (the
// cascade's default path):
//   out: entropy[v][pixel]  and  corr[v][d][pixel][8]   (then vis CNN, then corr_aggregate streams corr).
// One producer warp runs ahead of eight consumer warps through a ring of NBUF window buffers:
//   producer, per (tile, view): wait empty[buf] -> predict the window origin from 32 sample pixels of the tile (first and last
//             hypothesis: the taps of a pixel lie between them on its epipolar line) -> origin to shared memory ->
//             expect_tx + ONE cp.async.bulk.tensor box -> full[buf]
//   consumers, per (tile, view): wait full[buf] -> D taps per lane from the window (conflict-free rotated LDS.128; taps
//             outside the window through global memory) -> similarity, per-view entropy, correlation store -> arrive empty[buf]
// No CTA-wide barrier, no bounding-box reduction and no staging latency on the consumers' path (the first window kernels
// above pay all three per (view, chunk) and measured 0.37 ms at DTU stage 4; the L1-gather pass A 0.51 ms).
// ======================================================================================================================
struct PsCfg {
  static constexpr int NCONS = 256;           // consumer threads: an 8 x 32 pixel tile, one lane per pixel
  static constexpr int THREADS = NCONS + 32;  // + the producer warp
  static constexpr int TROWS = 8;
};

template <int NBUF>
struct PsShared {
  unsigned long long full[NBUF], empty[NBUF];
  int origin[NBUF][2];
};

template <int C, int D, int NBUF>
__global__ void __launch_bounds__(PsCfg::THREADS, kPsBlocks8)
warp_stream_entropy_store_kernel(const __grid_constant__ CUtensorMap map, const float* __restrict__ feat,
                                 const float* __restrict__ homs, const float* __restrict__ depth, float* __restrict__ entropy,
                                 float* __restrict__ corr, int V, int H, int W, int tiles_x, int ntiles, const int* __restrict__ select) {
  static_assert(C == 8, "one consumer lane per pixel owns all 8 channels");
  using K = Cfg<C>;
  using P = PsCfg;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ PsShared<NBUF> sh;
  if (select && *select == 0) return;   // warp_stream_select_kernel chose the L1-gather kernel for this call (launched next)
  const uint32_t win0 = (smem_u32(smem_raw) + 127u) & ~127u;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int HW = H * W;
  if (tid == 0) {
    for (int b = 0; b < NBUF; ++b) { mbar_init(smem_u32(&sh.full[b]), 1); mbar_init(smem_u32(&sh.empty[b]), P::NCONS / 32); }
    fence_barrier_init();
  }
  __syncthreads();
  const CoordConst cc = make_coord_const(W, H);
  const int my_tiles = (ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (warp == P::NCONS / 32) {
    // ------------------------------------------------------------------------------------------------ producer warp
    // sample pixel of this lane inside a tile: 4 rows x 8 columns spread over the 8 x 32 tile
    const int sr = (lane >> 3) * 2 + 1, sc = (lane & 7) * 4 + 1;
    int j = 0;
    for (int t = 0; t < my_tiles; ++t) {
      const int tile = (int)blockIdx.x + t * (int)gridDim.x;
      const int px = min((tile % tiles_x) * TW + sc, W - 1), py = min((tile / tiles_x) * P::TROWS + sr, H - 1);
      const int p = py * W + px;
      const float d_first = __ldg(depth + p), d_last = __ldg(depth + (size_t)(D - 1) * HW + p);
      const float fxp = (float)px, fyp = (float)py;
      for (int v = 0; v < V - 1; ++v, ++j) {
        const int buf = j % NBUF;
        const Hom m = load_hom(homs + (size_t)v * 12);
        float rx, ry, rz;
        pixel_ray(m, fxp, fyp, rx, ry, rz);
        TapCoord tc[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          float ix, iy;
          warp_coord_lean(rx, ry, rz, m, e ? d_last : d_first, cc, ix, iy);
          tc[e] = split_coord(ix, iy, W, H);
        }
        int ox, oy;
        predict_window<C>(tc[0], tc[1], ox, oy);
        mbar_wait_warp(smem_u32(&sh.empty[buf]), (uint32_t)(((j / NBUF) & 1) ^ 1));   // consumers released this buffer
        if (lane == 0) {
          sh.origin[buf][0] = ox;
          sh.origin[buf][1] = oy;
          const uint32_t bar = smem_u32(&sh.full[buf]);
          expect_tx(bar, K::BYTES);
          tma_load_5d(win0 + (uint32_t)buf * K::BYTES, &map, 0, 0, ox, oy >> 1, v + 1, bar);
        }
        __syncwarp();
      }
    }
    return;
  }

  // -------------------------------------------------------------------------------------------------- consumer warps
  int chA, chB;
  Lane L = make_lane<C>(lane, 0, chA, chB);
  const uint32_t base0 = L.base[0], base1 = L.base[1];   // + the address of the current window
  int j = 0;
  for (int t = 0; t < my_tiles; ++t) {
    const int tile = (int)blockIdx.x + t * (int)gridDim.x;
    const int px = (tile % tiles_x) * TW + (tid % TW), py = (tile / tiles_x) * P::TROWS + (tid / TW);
    const bool active = (px < W) && (py < H);
    const int p = min(py, H - 1) * W + min(px, W - 1);
    const float fxp = (float)min(px, W - 1), fyp = (float)min(py, H - 1);
    const float4 rA = ldg4(feat + (size_t)p * C + chA), rB = ldg4(feat + (size_t)p * C + chB);
    float dv[D];
#pragma unroll
    for (int k = 0; k < D; ++k) dv[k] = __ldg(depth + (size_t)k * HW + p);
    for (int v = 0; v < V - 1; ++v, ++j) {
      const int buf = j % NBUF;
      const Hom m = load_hom(homs + (size_t)v * 12);
      float rx, ry, rz;
      pixel_ray(m, fxp, fyp, rx, ry, rz);
      mbar_wait_warp(smem_u32(&sh.full[buf]), (uint32_t)((j / NBUF) & 1));
      const int ox = sh.origin[buf][0], oy = sh.origin[buf][1];
      L.base[0] = win0 + (uint32_t)buf * K::BYTES + base0;
      L.base[1] = win0 + (uint32_t)buf * K::BYTES + base1;
      float sims[D];
      float mx = -FLT_MAX;
#pragma unroll
      for (int k = 0; k < D; ++k) {
        float ix, iy;
        warp_coord_lean(rx, ry, rz, m, dv[k], cc, ix, iy);
        TapCoord tc = split_coord(ix, iy, W, H);
        tc.inb = tc.inb && active;
        float4 sA = make_float4(0.f, 0.f, 0.f, 0.f), sB = sA;
        const int lx = tc.x0 - ox, ly = tc.y0 - oy;
        const bool inwin = tc.inb && (unsigned)lx <= (unsigned)(K::WX - 2) && (unsigned)ly <= (unsigned)(K::WY - 2);
        gather_window<C>(L, inwin ? lx : 0, inwin ? ly : 0, tc.fx, tc.fy, sA, sB);
        if (!inwin) {
          sA = make_float4(0.f, 0.f, 0.f, 0.f); sB = sA;
          if (tc.inb) {   // rare: the source pointers are formed here so that they hold no registers in the loop
            const float* __restrict__ src = feat + (size_t)(v + 1) * HW * C;
            gather_global<C>(src + chA, src + chB, ix, iy, W, H, sA, sB);
          }
        }
        // per-view group correlations exactly as the aggregation pass consumes them (cost_volume.py:78-85); channels == groups
        if (active) {
          float* cp = corr + (((size_t)v * D + k) * HW + p) * 8;
          *reinterpret_cast<float4*>(cp + chA) = make_float4(rA.x * sA.x, rA.y * sA.y, rA.z * sA.z, rA.w * sA.w);
          *reinterpret_cast<float4*>(cp + chB) = make_float4(rB.x * sB.x, rB.y * sB.y, rB.z * sB.z, rB.w * sB.w);
        }
        const float s = dot4(rA, sA) + dot4(rB, sB);   // sum over the 8 one-channel groups
        sims[k] = s;
        mx = fmaxf(mx, s);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&sh.empty[buf]));   // this warp is done with the window
      // softmax over D -> entropy (cost_volume.py:90-92).  Intrinsic exp / log (ex2 / lg2 based, ~1e-6 relative here: the
      // arguments are <= 0 resp. in (1e-7, 1]); the entropy feeds a CNN whose output is compared at 5e-4.
      float Z = 0.f, ent = 0.f;
#pragma unroll
      for (int k = 0; k < D; ++k) { sims[k] = __expf(sims[k] - mx); Z += sims[k]; }
      const float rZ = __fdiv_rn(1.0f, Z);
#pragma unroll
      for (int k = 0; k < D; ++k) { const float pr = sims[k] * rZ; ent -= pr * __logf(pr + 1e-7f); }
      if (active) entropy[(size_t)v * HW + p] = ent;
    }
  }
}


// Which pass-A kernel should serve this call?  The pipeline kernel wins as long as nearly every tap lies in the 64 x 16 texel
// window its producer predicts (DTU stage 4: 28 misses per 1000 taps, 0.36 vs 0.51 ms); a tap outside goes through a divergent
// global gather, and with wide baselines + noisy hypotheses (Tanks&Temples, 9 source views: 287 per 1000, 1.57 vs 1.43 ms)
// the L1-gather kernel is faster.  CTA b replays the producer's prediction for sample tile b (one warp per source view) and
// counts, for the tile's 32 sample pixels, the hypotheses whose tap misses the window; the last CTA to finish turns the
// totals into the decision (at most kMaxWindowMissPermille -> pipeline) and clears the scratch counters for the slot's next use.
//   select[0] = 1: pipeline kernel, 0: L1 kernel;  select[1] = misses per 1000 in-bound taps (diagnostics);
//   select[2..4] = scratch: taps, misses, finished CTAs (zero between calls).
// Both kernels are launched behind it; the one not chosen returns at once.
template <int C, int D>
__global__ void __launch_bounds__(1024)
warp_stream_select_kernel(const float* __restrict__ homs, const float* __restrict__ depth, int V, int H, int W, int tiles_x,
                          int ntiles, int* __restrict__ select) {
  using K = Cfg<C>;
  using P = PsCfg;
  const int lane = threadIdx.x & 31, HW = H * W;
  const CoordConst cc = make_coord_const(W, H);
  const int sr = (lane >> 3) * 2 + 1, sc = (lane & 7) * 4 + 1;   // the producer's sample pixels
  const int tile = (int)(((long long)blockIdx.x * ntiles) / gridDim.x);
  const int px = min((tile % tiles_x) * TW + sc, W - 1), py = min((tile / tiles_x) * P::TROWS + sr, H - 1);
  const int p = py * W + px;
  const float fxp = (float)px, fyp = (float)py;
  float dv[D];
#pragma unroll
  for (int k = 0; k < D; ++k) dv[k] = __ldg(depth + (size_t)k * HW + p);
  unsigned int tot = 0u, miss = 0u;
  for (int v = threadIdx.x >> 5; v < V - 1; v += blockDim.x >> 5) {
    const Hom m = load_hom(homs + (size_t)v * 12);
    float rx, ry, rz;
    pixel_ray(m, fxp, fyp, rx, ry, rz);
    TapCoord tc[D];
#pragma unroll
    for (int k = 0; k < D; ++k) {
      float ix, iy;
      warp_coord_lean(rx, ry, rz, m, dv[k], cc, ix, iy);
      tc[k] = split_coord(ix, iy, W, H);
    }
    int ox, oy;
    predict_window<C>(tc[0], tc[D - 1], ox, oy);
#pragma unroll
    for (int k = 0; k < D; ++k) {
      if (!tc[k].inb) continue;
      ++tot;
      const int lx = tc[k].x0 - ox, ly = tc[k].y0 - oy;
      if (!((unsigned)lx <= (unsigned)(K::WX - 2) && (unsigned)ly <= (unsigned)(K::WY - 2))) ++miss;
    }
  }
  tot = __reduce_add_sync(0xffffffffu, tot);
  miss = __reduce_add_sync(0xffffffffu, miss);
  if (lane == 0) { atomicAdd(select + 2, (int)tot); atomicAdd(select + 3, (int)miss); }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(select + 4, 1) == (int)gridDim.x - 1) {   // last CTA: every other CTA's counts are visible
      __threadfence();
      const unsigned int t = (unsigned int)atomicExch(select + 2, 0), ms = (unsigned int)atomicExch(select + 3, 0);
      const unsigned int permille = t ? (unsigned int)(((unsigned long long)ms * 1000ull) / t) : 0u;
      select[1] = (int)permille;
      select[0] = permille <= (unsigned int)kMaxWindowMissPermille ? 1 : 0;
      atomicExch(select + 4, 0);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// 5-D view (c, y&1, x, y/2, view) of the channels-last feature tensor [V][H][W][C] (H even)
template <int C>
static int make_window_map(CUtensorMap* m, const float* feat, int V, int H, int W) {
  using K = Cfg<C>;
  EncodeTiledFn enc = encode_tiled_fn();
  MVSF_REQUIRE(enc, "warp_tile: cuTensorMapEncodeTiled is not available from this driver");
  const cuuint64_t row = (cuuint64_t)W * C * 4;
  const cuuint64_t dims[5] = {(cuuint64_t)C, 2, (cuuint64_t)W, (cuuint64_t)(H / 2), (cuuint64_t)V};
  const cuuint64_t strides[4] = {row, (cuuint64_t)C * 4, 2 * row, (cuuint64_t)H * row};
  const cuuint32_t box[5] = {(cuuint32_t)C, 2, (cuuint32_t)K::WX, (cuuint32_t)(K::WY / 2), 1};
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, const_cast<float*>(feat), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(MVSF_ERR_CUDA, "warp_tile: cuTensorMapEncodeTiled failed (%d) for V=%d H=%d W=%d C=%d", (int)r, V, H, W, C);
  return MVSF_OK;
}

template <int C, int MODE, int DCHT, bool GENERIC>
static int launch(const float* feat, const float* homs, const float* depth, const float* vis, float* out, int V, int D, int H,
                  int W, int dch, cudaStream_t s) {
  using K = Cfg<C>;
  auto kern = warp_tile_kernel<C, MODE, DCHT, GENERIC>;
  static DeviceOnce once;
  const int dev = current_device();
  const size_t smem = K::BYTES + 128;
  if (once.need(dev)) {
    MVSF_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    once.done(dev);
  }
  CUtensorMap map;
  int rc = make_window_map<C>(&map, feat, V, H, W);
  if (rc) return rc;
  dim3 grid(cdiv(W, TW), cdiv(H, K::TROWS));
  kern<<<grid, THREADS, smem, s>>>(map, feat, homs, depth, vis, out, V, D, H, W, dch);
  return MVSF_OK;
}

template <int C>
static int dispatch(int mode, const float* feat, const float* homs, const float* depth, const float* vis, float* out, int V,
                    int D, int H, int W, cudaStream_t s) {
  if (mode == 0) {
    if (D <= 4) return launch<C, 0, 4, false>(feat, homs, depth, vis, out, V, D, H, W, D, s);
    if (D <= 8) return launch<C, 0, 8, false>(feat, homs, depth, vis, out, V, D, H, W, D, s);
    int c = D / 24;   // plane sweeps: the epipolar span of a chunk has to stay inside the window
    c = c < 2 ? 2 : (c > 8 ? 8 : c);
    return launch<C, 0, 8, true>(feat, homs, depth, vis, out, V, D, H, W, c, s);
  }
  if (D <= 4) return launch<C, 1, 4, false>(feat, homs, depth, vis, out, V, D, H, W, D, s);
  int c = D <= 8 ? D : D / 24;
  c = c < 2 ? 2 : (c > 8 ? 8 : c);
  return launch<C, 1, 8, false>(feat, homs, depth, vis, out, V, D, H, W, c, s);
}

template <int C, int D, int NBUF>
static int launch_stream_store(const float* feat, const float* homs, const float* depth, float* entropy, float* corr, int V,
                               int H, int W, int* select, cudaStream_t s) {
  using K = Cfg<C>;
  auto kern = warp_stream_entropy_store_kernel<C, D, NBUF>;
  static DeviceOnce once;
  const int dev = current_device();
  const size_t smem = (size_t)NBUF * K::BYTES + 128;
  if (once.need(dev)) {
    MVSF_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    once.done(dev);
  }
  CUtensorMap map;
  int rc = make_window_map<C>(&map, feat, V, H, W);
  if (rc) return rc;
  const int tiles_x = cdiv(W, TW), tiles_y = cdiv(H, PsCfg::TROWS), ntiles = tiles_x * tiles_y;
  const int cap = device_sm_count(dev) * kPsBlocks8;
  if (select) {
    const int nsample = ntiles < 96 ? ntiles : 96, warps = V - 1 < 32 ? V - 1 : 32;
    warp_stream_select_kernel<C, D><<<nsample, 32 * warps, 0, s>>>(homs, depth, V, H, W, tiles_x, ntiles, select);
  }
  kern<<<ntiles < cap ? ntiles : cap, PsCfg::THREADS, smem, s>>>(map, feat, homs, depth, entropy, corr, V, H, W, tiles_x, ntiles, select);
  return MVSF_OK;
}

}  // namespace wt

// Used by warp_corr.cu's entry points.  Returns false when this organisation does not apply (other channel counts, odd H:
// the y-parity view of the tensor map needs an even number of rows, misaligned pointers).
bool warp_tile_supported(const float* feat, int C, int G, int D, int H, int W) {
  return (C == 8 || C == 16) && G == 8 && (H % 2 == 0) && H >= 2 && W >= 2 && D >= 1 && D <= wt::kMaxD &&
         ((uintptr_t)feat & 15) == 0 && ((long long)W * C * 4) % 16 == 0;
}
// pass A: entropy [V-1][H][W]
int warp_tile_entropy(const float* feat, const float* homs, const float* depth, float* entropy, int V, int C, int D, int H,
                      int W, cudaStream_t s) {
  return C == 8 ? wt::dispatch<8>(0, feat, homs, depth, nullptr, entropy, V, D, H, W, s)
                : wt::dispatch<16>(0, feat, homs, depth, nullptr, entropy, V, D, H, W, s);
}
// pass B: volume [D][H][W][8]
int warp_tile_aggregate(const float* feat, const float* homs, const float* depth, const float* vis, float* volume, int V, int C,
                        int D, int H, int W, cudaStream_t s) {
  return C == 8 ? wt::dispatch<8>(1, feat, homs, depth, vis, volume, V, D, H, W, s)
                : wt::dispatch<16>(1, feat, homs, depth, vis, volume, V, D, H, W, s);
}

// pass A of the spill plan (entropy + per-view group correlations) for the shape the pipeline kernel is built for
bool warp_stream_store_supported(const float* feat, const float* corr, int C, int G, int D, int H, int W) {
  return warp_tile_supported(feat, C, G, D, H, W) && C == 8 && D == 4 && ((uintptr_t)corr & 15) == 0;
}
// select != nullptr: five device ints (decision, miss share, three zeroed scratch counters); a small kernel decides from the geometry of THIS call whether the pipeline kernel runs
// (select[0] = 1) or leaves the call to the L1-gather kernel the caller launches next (select[0] = 0)
int warp_stream_entropy_store(const float* feat, const float* homs, const float* depth, float* entropy, float* corr, int V,
                              int H, int W, int* select, cudaStream_t s) {
  return wt::launch_stream_store<8, 4, wt::kPsNbuf8>(feat, homs, depth, entropy, corr, V, H, W, select, s);
}

}  // namespace mvsf
