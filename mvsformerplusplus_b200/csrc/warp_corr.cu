// W2+W3+W4: homography warp fused with group-wise correlation (models/warping.py:69-109,
// models/cost_volume.py:72-101).  The (V-1,C,D,H,W) warped volume is never written to HBM.
//
// Data layout: feature maps channels-last [V][H][W][C] so one bilinear corner is C contiguous floats.
// Thread mapping: LPP = C/4 lanes cooperate on one reference pixel, each lane owning 4 consecutive channels
// and loading them with one 128-bit LDG per corner; a warp therefore covers 32/LPP consecutive pixels and each
// warp-wide load touches 512 contiguous bytes of the source map when neighbouring pixels map to neighbouring
// source texels (the common case).  Tap coordinates are computed once per warp and shared through shared memory;
// partial dot products are combined across the LPP lanes with a butterfly reduce-scatter.
//
//   pass A (warp_corr_entropy):   sim[d] = sum_g mean_{c in g} ref[c]*warp[c,d]  ->  softmax_D -> entropy
//   pass B (warp_corr_aggregate): vol[g,d] = sum_v w_v * mean_{c in g} ref*warp_v / (sum_v w_v + 1e-6)
//
// Two passes because the visibility weight w_v is a 7x7-receptive-field CNN of the entropy map
// (cost_volume.py:89-93).  Two plans bridge them: the spill plan (the cascade's default) has pass A also store the
// (V-1) x G x D x H x W per-view group correlations and streams them in corr_aggregate_kernel; the recompute plan gathers
// a second time in pass B and needs no buffer (plane sweeps, spill buffers over budget).  See mvsf_warp_corr_plan.
#include <float.h>

#include <atomic>
#include <mutex>

#include "common.cuh"

namespace mvsf {

// warp_tile.cu: TMA-staged shared-memory windows, for C = 8 / 16 (the fine stages)
bool warp_tile_supported(const float* feat, int C, int G, int D, int H, int W);
int warp_tile_entropy(const float* feat, const float* homs, const float* depth, float* entropy, int V, int C, int D, int H,
                      int W, cudaStream_t s);
int warp_tile_aggregate(const float* feat, const float* homs, const float* depth, const float* vis, float* volume, int V, int C,
                        int D, int H, int W, cudaStream_t s);
bool warp_stream_store_supported(const float* feat, const float* corr, int C, int G, int D, int H, int W);
int warp_stream_entropy_store(const float* feat, const float* homs, const float* depth, float* entropy, float* corr, int V,
                              int H, int W, int* select, cudaStream_t s);

constexpr int kMaxGenericD = 512;

// v2 organisation (r1 ncu: v1 was instruction-issue bound because all C/4 lanes of a pixel recomputed the exact-rounding
// coordinate math: ~220 warp instructions per tap):
//   A warp owns P = 32/LPP consecutive pixels (LPP = C/4 lanes per pixel) and works on chunks of DCH = 2*LPP
//   hypotheses, i.e. always 64 (pixel, hypothesis) taps per chunk.
//   phase 1: every lane computes exactly two of the 64 taps (coordinates -> 4 corner offsets + 4 weights) and parks them
//            in a per-warp shared-memory table (2 KB);  phase 2: the LPP lanes of a pixel read each tap back with two
//            broadcast LDS.128 and do the 4-corner gather + correlation for their 4 channels.
// For the shipped stages DCH equals the stage's hypothesis count (C=64/32/16/8 <-> D=32/16/8/4): one chunk per view.
template <int C>
struct WC {
  static constexpr int LPP = C / 4, P = 32 / LPP, DCH = 2 * LPP;
};
struct __align__(16) TapTable {
  int4 off[64];
  float4 wt[64];
};

// phase 1 for one (view, chunk): taps t = lane and lane+32, t = di*P + pi
template <int C>
__device__ __forceinline__ void build_taps(TapTable& tb, const float* __restrict__ depth, const Hom& m, float rx, float ry,
                                           float rz, const CoordConst& cc, int p1, int d0, int D, int HW, int H, int W,
                                           int lane) {
  constexpr int P = WC<C>::P;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int t = lane + 32 * k;
    const int d = d0 + t / P;
    const float dv = (d < D) ? __ldg(depth + (size_t)d * HW + p1) : 1.0f;
    float ix, iy;
    warp_coord_fast(rx, ry, rz, m, dv, cc, ix, iy);
    int4 off;
    float4 wt;
    make_tap_fast(ix, iy, W, H, C, off, wt);
    tb.off[t] = off;
    tb.wt[t] = wt;
  }
}
__device__ __forceinline__ float4 gather4(const float* __restrict__ base, const int4& o, const float4& w) {
  float4 a = ldg4(base + o.x), b = ldg4(base + o.y), c = ldg4(base + o.z), d = ldg4(base + o.w);
  float4 s;
  s.x = fmaf(d.x, w.w, fmaf(c.x, w.z, fmaf(b.x, w.y, a.x * w.x)));
  s.y = fmaf(d.y, w.w, fmaf(c.y, w.z, fmaf(b.y, w.y, a.y * w.x)));
  s.z = fmaf(d.z, w.w, fmaf(c.z, w.z, fmaf(b.z, w.y, a.z * w.x)));
  s.w = fmaf(d.w, w.w, fmaf(c.w, w.z, fmaf(b.w, w.y, a.w * w.x)));
  return s;
}

// Butterfly reduce-scatter over the LPP lanes of a pixel: in: v[0..N) partial sums per lane; out: lane `lip` holds the
// complete sums of elements [lip*N/LPP, (lip+1)*N/LPP) in v[0..N/LPP).
template <int N, int LANES>
struct ReduceScatter {
  static __device__ __forceinline__ void run(float (&v)[N > 0 ? N : 1], int lip) {
    if constexpr (LANES > 1) {
      constexpr int H = N / 2, O = LANES / 2;
      const bool upper = (lip & O) != 0;
#pragma unroll
      for (int i = 0; i < H; ++i) {
        float send = upper ? v[i] : v[i + H];
        float keep = upper ? v[i + H] : v[i];
        v[i] = keep + __shfl_xor_sync(0xffffffffu, send, O);
      }
      float (&lo)[H > 0 ? H : 1] = reinterpret_cast<float (&)[H > 0 ? H : 1]>(v);
      ReduceScatter<H, O>::run(lo, lip);
    }
  }
};

// ---------------------------------------------------------------------------------------------- pass A
// CPGS > 0: also store the per-view GROUP correlations corr[v][d][pixel][g] (G = C / CPGS = 8 groups) so that the view
// aggregation becomes a streaming pass (corr_aggregate_kernel) instead of a second gather: the gather is bound by L1
// requests, the extra 4 * G * D * HW * (V-1) bytes of HBM traffic each way are cheaper.
template <int C, bool GENERIC, int CPGS, bool STRIDED = false>
__global__ void __launch_bounds__(256)
warp_corr_entropy_kernel(const float* __restrict__ feat, const float* __restrict__ homs,
                         const float* __restrict__ depth, float* __restrict__ entropy, float* __restrict__ corr, int G,
                         int D, int H, int W, const int* __restrict__ skip_if) {
  constexpr int LPP = WC<C>::LPP, P = WC<C>::P, DCH = WC<C>::DCH;
  if (skip_if && *skip_if != 0) return;   // the pipeline kernel (warp_tile.cu) served this call
  constexpr int SPL = DCH / LPP;  // complete sims per lane per chunk (= 2)
  constexpr int MAXCH = GENERIC ? (kMaxGenericD + DCH - 1) / DCH : 1;
  __shared__ TapTable tables[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  TapTable& tb = tables[warp];
  const int HW = H * W;
  const int v = blockIdx.y;
  // STRIDED (the adaptive launch behind the selection kernel, C = 8): a capped grid strides over the 8-warp pixel blocks, so
  // that the launch that finds skip_if set costs microseconds instead of 55 000 exiting CTAs (and the kernel itself is
  // faster at C = 8, T&T 1.43 -> 1.24 ms; at C = 16..64 the loop costs registers - 143 at C = 64 - and is not used)
  int bx = blockIdx.x;
  do {
  const int pix0 = (bx * 8 + warp) * P;
  if (pix0 >= HW) return;  // whole warp exits together (later blocks lie further out still)
  // phase-1 pixel (lane % P) and phase-2 pixel (lane / LPP)
  const int p1 = min(pix0 + lane % P, HW - 1);
  const int p2raw = pix0 + lane / LPP;
  const bool active = p2raw < HW;
  const int p2 = active ? p2raw : HW - 1;
  const int lip = lane % LPP;
  const Hom m = load_hom(homs + (size_t)v * 12);
  const CoordConst cc = make_coord_const(W, H);
  const int y1 = p1 / W, x1 = p1 - y1 * W;
  const float fx = (float)x1, fy = (float)y1;
  float rx, ry, rz;
  pixel_ray(m, fx, fy, rx, ry, rz);
  const float4 r = ldg4(feat + (size_t)p2 * C + lip * 4);
  const float* __restrict__ src = feat + (size_t)(v + 1) * HW * C + lip * 4;
  const float gscale = (float)G / (float)C;

  float sims[MAXCH * SPL];
  const int nch = GENERIC ? (D + DCH - 1) / DCH : 1;
  for (int ch = 0; ch < nch; ++ch) {
    const int d0 = ch * DCH;
    build_taps<C>(tb, depth, m, rx, ry, rz, cc, p1, d0, D, HW, H, W, lane);
    __syncwarp();
    float part[DCH];
    const int pi = lane / LPP;
#pragma unroll
    for (int di = 0; di < DCH; ++di) {
      const int4 o = tb.off[di * P + pi];
      const float4 w = tb.wt[di * P + pi];
      const float4 s = gather4(src, o, w);
      part[di] = fmaf(r.w, s.w, fmaf(r.z, s.z, fmaf(r.y, s.y, r.x * s.x)));
      if (CPGS > 0 && d0 + di < D) {   // group correlations exactly as the aggregation pass forms them
        constexpr float inv_cpg = 1.0f / (float)(CPGS > 0 ? CPGS : 1);
        float* cp = corr + (((size_t)v * D + d0 + di) * HW + p2) * 8;
        if (CPGS == 1) {
          if (active) *reinterpret_cast<float4*>(cp + lip * 4) = make_float4(r.x * s.x, r.y * s.y, r.z * s.z, r.w * s.w);
        } else if (CPGS == 2) {
          if (active) *reinterpret_cast<float2*>(cp + lip * 2) = make_float2(fmaf(r.y, s.y, r.x * s.x) * inv_cpg, fmaf(r.w, s.w, r.z * s.z) * inv_cpg);
        } else if (CPGS == 4) {
          if (active) cp[lip] = part[di] * inv_cpg;
        } else {  // 8 channels per group: two lanes share a group
          const float both = part[di] + __shfl_xor_sync(0xffffffffu, part[di], 1);
          if (active && (lip & 1) == 0) cp[lip >> 1] = both * inv_cpg;
        }
      }
    }
    __syncwarp();
    ReduceScatter<DCH, LPP>::run(part, lip);
#pragma unroll
    for (int i = 0; i < SPL; ++i) {
      const int d = d0 + lip * SPL + i;
      sims[ch * SPL + i] = (d < D) ? part[i] * gscale : -FLT_MAX;
    }
  }
  // softmax over D -> entropy; a pixel's sims are spread over its LPP lanes (nch*SPL each)
  float mx = -FLT_MAX;
  for (int i = 0; i < nch * SPL; ++i) mx = fmaxf(mx, sims[i]);
#pragma unroll
  for (int o = LPP / 2; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float Z = 0.f;
  for (int i = 0; i < nch * SPL; ++i) {
    sims[i] = (sims[i] == -FLT_MAX) ? 0.f : expf(sims[i] - mx);
    Z += sims[i];
  }
#pragma unroll
  for (int o = LPP / 2; o > 0; o >>= 1) Z += __shfl_xor_sync(0xffffffffu, Z, o);
  float ent = 0.f;
  for (int i = 0; i < nch * SPL; ++i) {
    float pr = __fdiv_rn(sims[i], Z);
    ent -= pr * logf(pr + 1e-7f);
  }
#pragma unroll
  for (int o = LPP / 2; o > 0; o >>= 1) ent += __shfl_xor_sync(0xffffffffu, ent, o);
  if (active && lip == 0) entropy[(size_t)v * HW + p2] = ent;
  if (STRIDED) __syncwarp();   // the warp's tap table is rewritten by the next trip
  } while (STRIDED && (bx += (int)gridDim.x) * 8 * P < HW);
}

// ---------------------------------------------------------------------------------------------- pass B
// CPG = C/G channels per group.  A lane owns NGL = max(1, 4/CPG) groups; for CPG = 8 two lanes share a group and their
// partial sums are combined once at the end (the view reduction is linear).
template <int C, int CPG>
__global__ void __launch_bounds__(256)
warp_corr_aggregate_kernel(const float* __restrict__ feat, const float* __restrict__ homs,
                           const float* __restrict__ depth, const float* __restrict__ vis,
                           float* __restrict__ volume, int V, int D, int H, int W) {
  constexpr int LPP = WC<C>::LPP, P = WC<C>::P, DCH = WC<C>::DCH;
  constexpr int G = C / CPG;
  constexpr int NGL = (CPG >= 4) ? 1 : 4 / CPG;
  constexpr int LPG = (CPG >= 4) ? CPG / 4 : 1;  // lanes per group (1 or 2)
  static_assert(LPG == 1 || LPG == 2, "C/G must be 1, 2, 4 or 8");
  __shared__ TapTable tables[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  TapTable& tb = tables[warp];
  const int HW = H * W;
  const int pix0 = (blockIdx.x * 8 + warp) * P;
  if (pix0 >= HW) return;
  const int p1 = min(pix0 + lane % P, HW - 1);
  const int p2raw = pix0 + lane / LPP;
  const bool active = p2raw < HW;
  const int p2 = active ? p2raw : HW - 1;
  const int lip = lane % LPP, pi = lane / LPP;
  const CoordConst cc = make_coord_const(W, H);
  const int y1 = p1 / W, x1 = p1 - y1 * W;
  const float fx = (float)x1, fy = (float)y1;
  const float4 r = ldg4(feat + (size_t)p2 * C + lip * 4);
  constexpr float inv_cpg = 1.0f / (float)CPG;

  for (int d0 = 0; d0 < D; d0 += DCH) {
    float acc[NGL][DCH];
#pragma unroll
    for (int g = 0; g < NGL; ++g)
#pragma unroll
      for (int i = 0; i < DCH; ++i) acc[g][i] = 0.f;
    float wsum = 0.f;
    for (int v = 0; v < V - 1; ++v) {
      const Hom m = load_hom(homs + (size_t)v * 12);
      float rx, ry, rz;
      pixel_ray(m, fx, fy, rx, ry, rz);
      build_taps<C>(tb, depth, m, rx, ry, rz, cc, p1, d0, D, HW, H, W, lane);
      __syncwarp();
      const float* __restrict__ src = feat + (size_t)(v + 1) * HW * C + lip * 4;
      const float w = __ldg(vis + (size_t)v * HW + p2);
      wsum = __fadd_rn(wsum, w);
#pragma unroll
      for (int di = 0; di < DCH; ++di) {
        const int4 o = tb.off[di * P + pi];
        const float4 wt = tb.wt[di * P + pi];
        const float4 s = gather4(src, o, wt);
        if (CPG >= 4) {
          float part = fmaf(r.w, s.w, fmaf(r.z, s.z, fmaf(r.y, s.y, r.x * s.x))) * inv_cpg;
          acc[0][di] = fmaf(part, w, acc[0][di]);
        } else if (CPG == 2) {
          acc[0][di] = fmaf(fmaf(r.y, s.y, r.x * s.x) * inv_cpg, w, acc[0][di]);
          acc[NGL > 1 ? 1 : 0][di] = fmaf(fmaf(r.w, s.w, r.z * s.z) * inv_cpg, w, acc[NGL > 1 ? 1 : 0][di]);
        } else {  // CPG == 1: plain product (cost_volume.py:84-85)
          acc[0][di] = fmaf(r.x * s.x, w, acc[0][di]);
          acc[NGL > 1 ? 1 : 0][di] = fmaf(r.y * s.y, w, acc[NGL > 1 ? 1 : 0][di]);
          acc[NGL > 2 ? 2 : 0][di] = fmaf(r.z * s.z, w, acc[NGL > 2 ? 2 : 0][di]);
          acc[NGL > 3 ? 3 : 0][di] = fmaf(r.w * s.w, w, acc[NGL > 3 ? 3 : 0][di]);
        }
      }
      __syncwarp();
    }
    const float den = __fadd_rn(wsum, 1e-6f);
    if (LPG == 2) {
      // the two lanes of a group exchange halves: even lane ends with hypotheses [0, DCH/2), odd lane with [DCH/2, DCH)
      ReduceScatter<DCH, 2>::run(acc[0], lip & 1);
      if (active) {
        const int dbase = d0 + (lip & 1) * (DCH / 2);
#pragma unroll
        for (int i = 0; i < DCH / 2; ++i)
          if (dbase + i < D) volume[((size_t)(dbase + i) * HW + p2) * G + (lip >> 1)] = __fdiv_rn(acc[0][i], den);
      }
    } else if (active) {
#pragma unroll
      for (int di = 0; di < DCH; ++di) {
        if (d0 + di < D) {
          float* o = volume + ((size_t)(d0 + di) * HW + p2) * G;
          if (NGL == 1) {
            o[lip] = __fdiv_rn(acc[0][di], den);
          } else if (NGL == 2) {
            *reinterpret_cast<float2*>(o + lip * 2) = make_float2(__fdiv_rn(acc[0][di], den), __fdiv_rn(acc[NGL > 1 ? 1 : 0][di], den));
          } else {
            *reinterpret_cast<float4*>(o + lip * 4) =
                make_float4(__fdiv_rn(acc[0][di], den), __fdiv_rn(acc[NGL > 1 ? 1 : 0][di], den),
                            __fdiv_rn(acc[NGL > 2 ? 2 : 0][di], den), __fdiv_rn(acc[NGL > 3 ? 3 : 0][di], den));
          }
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------- finest seam
// models/warping.py:69-109 as a standalone op (materialises [C][D][H][W]; used for seam parity, not by the hot path)
__global__ void homo_warp_kernel(const float* __restrict__ src, const float* __restrict__ hom,
                                 const float* __restrict__ depth, float* __restrict__ warped,
                                 uint8_t* __restrict__ mask, int C, int D, int H, int W) {
  const int HW = H * W;
  int p = blockIdx.x * blockDim.x + threadIdx.x;
  int d = blockIdx.y;
  if (p >= HW) return;
  int y = p / W, x = p - y * W;
  const Hom m = load_hom(hom);
  const float fx = (float)x, fy = (float)y;
  float rx, ry, rz;
  pixel_ray(m, fx, fy, rx, ry, rz);
  const float half_w = (float)(W - 1) * 0.5f, half_h = (float)(H - 1) * 0.5f;
  float ix, iy, z;
  warp_coord(rx, ry, rz, m, __ldg(depth + (size_t)d * HW + p), half_w, half_h, (float)(W - 1), (float)(H - 1), ix, iy, z);
  Tap t = make_tap(ix, iy, W, H, C);
  for (int c = 0; c < C; ++c) {
    float a = __ldg(src + t.o00 + c), b = __ldg(src + t.o01 + c), cc = __ldg(src + t.o10 + c), dd = __ldg(src + t.o11 + c);
    warped[((size_t)c * D + d) * HW + p] = fmaf(dd, t.w11, fmaf(cc, t.w10, fmaf(b, t.w01, a * t.w00)));
  }
  if (mask) {
    // warping.py:98-103: |normalised coordinate| > 1 or z <= 0.  ix = (g+1)/2*(W-1)  =>  g>1 <=> ix > W-1 etc.
    bool out = (ix > (float)(W - 1)) || (ix < 0.0f) || (iy > (float)(H - 1)) || (iy < 0.0f) || (z <= 0.0f);
    mask[(size_t)d * HW + p] = out ? 1 : 0;
  }
}

template <int C>
static void launch_entropy(const float* feat, const float* homs, const float* depth, float* entropy, float* corr, int V, int G,
                           int D, int H, int W, cudaStream_t s) {
  constexpr int P = WC<C>::P;
  dim3 grid(cdiv((long long)H * W, 8 * P), V - 1);
  if (corr) {   // G == 8 (checked by the caller)
    if (D == WC<C>::DCH)
      warp_corr_entropy_kernel<C, false, C / 8><<<grid, 256, 0, s>>>(feat, homs, depth, entropy, corr, G, D, H, W, nullptr);
    else
      warp_corr_entropy_kernel<C, true, C / 8><<<grid, 256, 0, s>>>(feat, homs, depth, entropy, corr, G, D, H, W, nullptr);
  } else if (D == WC<C>::DCH) {
    warp_corr_entropy_kernel<C, false, 0><<<grid, 256, 0, s>>>(feat, homs, depth, entropy, nullptr, G, D, H, W, nullptr);
  } else {
    warp_corr_entropy_kernel<C, true, 0><<<grid, 256, 0, s>>>(feat, homs, depth, entropy, nullptr, G, D, H, W, nullptr);
  }
}
// The spill plan at C = 8, D = 4 behind the selection kernel, which may have left it nothing to do (skip_if set): a capped,
// grid-strided grid.
static void launch_entropy_adaptive(const float* feat, const float* homs, const float* depth, float* entropy, float* corr,
                                    int V, int G, int D, int H, int W, cudaStream_t s, const int* skip_if) {
  constexpr int P = WC<8>::P;
  const int blocks = cdiv((long long)H * W, 8 * P), cap = device_sm_count(current_device()) * 16;
  dim3 grid(blocks < cap ? blocks : cap, V - 1);
  warp_corr_entropy_kernel<8, false, 1, true><<<grid, 256, 0, s>>>(feat, homs, depth, entropy, corr, G, D, H, W, skip_if);
}

// volume[d][p][g] = sum_v vis[v][p] * corr[v][d][p][g] / (sum_v vis[v][p] + 1e-6)   (cost_volume.py:95-101), G = 8
__global__ void __launch_bounds__(256)
corr_aggregate_kernel(const float* __restrict__ corr, const float* __restrict__ vis, float* __restrict__ volume, int V, int D,
                      int HW) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;   // (d, pixel, half of the 8 groups)
  const size_t total = (size_t)D * HW * 2;
  if (i >= total) return;
  const size_t dp = i >> 1;
  const int p = (int)(dp % HW);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  float wsum = 0.f;
  for (int v = 0; v < V - 1; ++v) {
    const float w = __ldg(vis + (size_t)v * HW + p);
    const float4 c = ldg4(corr + ((size_t)v * D * HW + dp) * 8 + (i & 1) * 4);
    wsum = __fadd_rn(wsum, w);
    acc.x = fmaf(c.x, w, acc.x); acc.y = fmaf(c.y, w, acc.y); acc.z = fmaf(c.z, w, acc.z); acc.w = fmaf(c.w, w, acc.w);
  }
  const float den = __fadd_rn(wsum, 1e-6f);
  *reinterpret_cast<float4*>(volume + dp * 8 + (i & 1) * 4) =
      make_float4(__fdiv_rn(acc.x, den), __fdiv_rn(acc.y, den), __fdiv_rn(acc.z, den), __fdiv_rn(acc.w, den));
}

template <int C, int CPG>
static int launch_aggregate(const float* feat, const float* homs, const float* depth, const float* vis, float* volume,
                            int V, int D, int H, int W, cudaStream_t s) {
  constexpr int P = WC<C>::P;
  dim3 grid(cdiv((long long)H * W, 8 * P));
  warp_corr_aggregate_kernel<C, CPG><<<grid, 256, 0, s>>>(feat, homs, depth, vis, volume, V, D, H, W);
  return 0;
}

}  // namespace mvsf

using namespace mvsf;

// test hook: 0 forces the L1-gather organisation (warp_corr.cu) for every shape, 1 (default) lets C = 8 / 16 stages use
// the TMA-staged window kernels (warp_tile.cu).  Both compute the same function; tests compare them.
static int g_use_tile = 1;   // 0: L1-gather kernels everywhere, 1: adaptive (default), 2: window / pipeline kernels wherever they exist

// Selection slots of the adaptive pass-A choice: 8 ints per call (decision, miss share, 3 scratch counters), a ring per device so that calls in
// flight on different streams do not share a slot.  Allocated on the first call (like the kernels' attribute set-up).
constexpr int kSelectSlots = 256;
static int* g_select[16] = {};
static std::atomic<unsigned> g_select_next{0};
static std::atomic<int*> g_select_last{nullptr};
static std::mutex g_select_mu;
static int* select_slot() {
  const int dev = current_device();
  if (dev < 0 || dev >= 16) return nullptr;
  if (!g_select[dev]) {
    std::lock_guard<std::mutex> lock(g_select_mu);
    if (!g_select[dev]) {
      int* p = nullptr;
      if (cudaMalloc(&p, sizeof(int) * 8 * kSelectSlots) != cudaSuccess) return nullptr;
      cudaMemset(p, 0, sizeof(int) * 8 * kSelectSlots);
      g_select[dev] = p;
    }
  }
  int* slot = g_select[dev] + 8 * (g_select_next.fetch_add(1) % kSelectSlots);
  g_select_last.store(slot);
  return slot;
}

extern "C" {

int mvsf_warp_corr_set_tile_path(int enable) {
  g_use_tile = enable < 0 ? 0 : (enable > 2 ? 2 : enable);
  return MVSF_OK;
}
int mvsf_warp_corr_last_selection(int* used_pipeline, int* miss_permille) {
  int* slot = g_select_last.load();
  MVSF_REQUIRE(slot && used_pipeline && miss_permille, "warp_corr_last_selection: no adaptive call has been made yet");
  int h[2] = {0, 0};
  MVSF_CUDA_OK(cudaMemcpy(h, slot, sizeof(h), cudaMemcpyDeviceToHost));   // synchronises: diagnostics / tests only
  *used_pipeline = h[0];
  *miss_permille = h[1];
  return MVSF_OK;
}

static int warp_corr_entropy_impl(const float* feat, const float* homs, const float* depth, float* entropy, float* corr, int V,
                                  int C, int G, int D, int H, int W, mvsf_stream_t stream);

/* 1: run the cost volume as two gathers (mvsf_warp_corr_entropy + mvsf_warp_corr_aggregate, no intermediate buffer);
 * 0: spill plan (mvsf_warp_corr_entropy_store + mvsf_corr_aggregate, needs 4*(V-1)*G*D*H*W bytes).  Measured on B200 the
 * spill plan is the faster one at every stage of the shipped cascade (the gather is bound by the SM's load path, the
 * streaming pass by HBM), so the recommendation only depends on the buffer size the caller is willing to spend. */
int mvsf_warp_corr_plan(int C, int G, int D, int H, int W, int V, size_t spill_budget_bytes) {
  if (G != 8 || !(C == 8 || C == 16 || C == 32 || C == 64)) return 1;   // the spill kernels exist for G == 8 only
  const size_t spill = (size_t)4 * (size_t)(V > 1 ? V - 1 : 1) * G * D * H * W;
  return spill > spill_budget_bytes ? 1 : 0;
}
int mvsf_warp_corr_entropy(const float* feat, const float* homs, const float* depth, float* entropy, int V, int C,
                           int G, int D, int H, int W, mvsf_stream_t stream) {
  return warp_corr_entropy_impl(feat, homs, depth, entropy, nullptr, V, C, G, D, H, W, stream);
}

int mvsf_warp_corr_entropy_store(const float* feat, const float* homs, const float* depth, float* entropy, float* corr,
                                 int V, int C, int G, int D, int H, int W, mvsf_stream_t stream) {
  MVSF_REQUIRE(corr && ((uintptr_t)corr & 15) == 0 && G == 8, "warp_corr_entropy_store: corr must be 16-byte aligned and G == 8");
  return warp_corr_entropy_impl(feat, homs, depth, entropy, corr, V, C, G, D, H, W, stream);
}

int mvsf_corr_aggregate(const float* corr, const float* vis, float* volume, int V, int G, int D, int H, int W,
                        mvsf_stream_t stream) {
  MVSF_REQUIRE(corr && vis && volume && V >= 2 && G == 8 && D >= 1 && H > 0 && W > 0, "corr_aggregate: bad arguments (G must be 8)");
  const size_t total = (size_t)D * H * W * 2;
  corr_aggregate_kernel<<<cdiv((long long)total, 256), 256, 0, (cudaStream_t)stream>>>(corr, vis, volume, V, D, H * W);
  MVSF_LAUNCH_CHECK("corr_aggregate");
  return MVSF_OK;
}

static int warp_corr_entropy_impl(const float* feat, const float* homs, const float* depth, float* entropy, float* corr, int V,
                                  int C, int G, int D, int H, int W, mvsf_stream_t stream) {
  MVSF_REQUIRE(feat && homs && depth && entropy, "warp_corr_entropy: null pointer");
  MVSF_REQUIRE(V >= 2 && H > 0 && W > 0 && D >= 1, "warp_corr_entropy: bad shape");
  MVSF_REQUIRE(G <= C, "G must <= C!");  // models/cost_volume.py:87
  MVSF_REQUIRE(C % G == 0 && (C == 8 || C == 16 || C == 32 || C == 64), "warp_corr_entropy: C must be 8/16/32/64, C %% G == 0");
  MVSF_REQUIRE(D <= kMaxGenericD, "warp_corr_entropy: D <= %d", kMaxGenericD);
  cudaStream_t s = (cudaStream_t)stream;
  if (corr && g_use_tile && warp_stream_store_supported(feat, corr, C, G, D, H, W)) {
    // finest stage of the cascade (C = 8, D = 4): persistent TMA producer / consumer pipeline kernel, as long as the taps of
    // this call fit its windows (decided on the device, per call: see warp_stream_select_kernel)
    const bool forced = g_use_tile == 2;
    int* select = forced ? nullptr : select_slot();
    if (forced || select) {
      int rc = warp_stream_entropy_store(feat, homs, depth, entropy, corr, V, H, W, select, s);
      if (rc) return rc;
      MVSF_LAUNCH_CHECK("warp_stream_entropy_store");
      if (forced) return MVSF_OK;
      count_launch();   // the selection kernel
      launch_entropy_adaptive(feat, homs, depth, entropy, corr, V, G, D, H, W, s, select);   // returns at once unless select[0] == 0
      MVSF_LAUNCH_CHECK("warp_corr_entropy");
      return MVSF_OK;
    }
  }
  if (!corr && g_use_tile && warp_tile_supported(feat, C, G, D, H, W)) {
    int rc = warp_tile_entropy(feat, homs, depth, entropy, V, C, D, H, W, s);
    if (rc) return rc;
    MVSF_LAUNCH_CHECK("warp_tile_entropy");
    return MVSF_OK;
  }
  switch (C) {
    case 8: launch_entropy<8>(feat, homs, depth, entropy, corr, V, G, D, H, W, s); break;
    case 16: launch_entropy<16>(feat, homs, depth, entropy, corr, V, G, D, H, W, s); break;
    case 32: launch_entropy<32>(feat, homs, depth, entropy, corr, V, G, D, H, W, s); break;
    default: launch_entropy<64>(feat, homs, depth, entropy, corr, V, G, D, H, W, s); break;
  }
  MVSF_LAUNCH_CHECK("warp_corr_entropy");
  return MVSF_OK;
}

int mvsf_warp_corr_aggregate(const float* feat, const float* homs, const float* depth, const float* vis,
                             float* volume, int V, int C, int G, int D, int H, int W, mvsf_stream_t stream) {
  MVSF_REQUIRE(feat && homs && depth && vis && volume, "warp_corr_aggregate: null pointer");
  MVSF_REQUIRE(V >= 2 && H > 0 && W > 0 && D >= 1, "warp_corr_aggregate: bad shape");
  MVSF_REQUIRE(G <= C, "G must <= C!");
  MVSF_REQUIRE(G == 8 && (C == 8 || C == 16 || C == 32 || C == 64), "warp_corr_aggregate: G must be 8 and C in 8/16/32/64");
  cudaStream_t s = (cudaStream_t)stream;
  if (g_use_tile && warp_tile_supported(feat, C, G, D, H, W)) {
    int rc = warp_tile_aggregate(feat, homs, depth, vis, volume, V, C, D, H, W, s);
    if (rc) return rc;
    MVSF_LAUNCH_CHECK("warp_tile_aggregate");
    return MVSF_OK;
  }
  switch (C) {
    case 8: launch_aggregate<8, 1>(feat, homs, depth, vis, volume, V, D, H, W, s); break;
    case 16: launch_aggregate<16, 2>(feat, homs, depth, vis, volume, V, D, H, W, s); break;
    case 32: launch_aggregate<32, 4>(feat, homs, depth, vis, volume, V, D, H, W, s); break;
    default: launch_aggregate<64, 8>(feat, homs, depth, vis, volume, V, D, H, W, s); break;
  }
  MVSF_LAUNCH_CHECK("warp_corr_aggregate");
  return MVSF_OK;
}

int mvsf_homo_warp(const float* src_nhwc, const float* hom, const float* depth, float* warped, uint8_t* mask, int C,
                   int D, int H, int W, mvsf_stream_t stream) {
  MVSF_REQUIRE(src_nhwc && hom && depth && warped && C > 0 && D > 0 && H > 0 && W > 0 && D <= 65535, "homo_warp: bad arguments");
  dim3 grid(cdiv(H * W, 128), D);
  homo_warp_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(src_nhwc, hom, depth, warped, mask, C, D, H, W);
  MVSF_LAUNCH_CHECK("homo_warp");
  return MVSF_OK;
}
}
