// 3x3x3 convolutions of the U-Net cost regularisers (models/module.py:367-408 CostRegNet, :453-504 CostRegNet3D) as
// implicit GEMMs on the 5th-generation tensor cores, fp32-class accuracy.
//
//   * activations live in HBM as two fp16 tensors (hi, lo; x ~= hi + lo carries 22 mantissa bits), NDHWC.  A tile is
//     16 (h) x 8*NT (w) cells of one depth slice.  Per (input depth slice, group of KG channel octets) "unit" ONE thread
//     issues TMA box loads (cp.async.bulk.tensor.5d over (c, w, h, d, hi|lo); the conv padding is TMA's out-of-bounds
//     zero fill) that land the halo of the tile in shared memory as PLANES of voxel octets: plane[row][col] = 8 channels
//     = 16 bytes.  Eight w-neighbours are then 128 contiguous bytes = one UMMA "core matrix" of the canonical no-swizzle
//     K-major layout, the h rows are the 8-row groups (SBO = row pitch) and hi / lo planes (or the two octets) are the
//     two K-chunks of a K = 16 MMA (LBO = plane distance).  A filter tap (kh, kw) is nothing but a different descriptor
//     start address: no im2col, no per-element address arithmetic anywhere;
//   * KG = 1: per tap two tcgen05.mma.kind::f16 (M = 128 cells, N = Cout, K = 16)
//         [x_hi | x_lo] x [w_hi ; w_hi]   and   [x_hi | x_lo] x [w_lo ; 0]       (x_lo*w_lo ~ 2^-22 is dropped)
//     KG = 2 (16 channels per unit): K = 16 spans the two octets and three MMAs x_lo*w_hi, x_hi*w_lo, x_hi*w_hi are
//     issued; fp32 accumulation in TMEM; the weight slabs come pre-arranged from conv3d_tc_pack and travel with the
//     unit (one cp.async.bulk) through the same mbarrier ring (expect_tx / complete_tx);
//   * stride-(SD,2,2) convolutions keep four parity planes (even/odd h x even/odd w, one strided tensor map each) so
//     that every tap is again a dense plane access; transposed convolutions run in gather form over INPUT cells with
//     four accumulators, one per output parity class (every (kh, kw) tap feeds exactly one class).  Taps that read the
//     same input shift (dih, diw) are fused along N: the class accumulators sit in TMEM in the order [0, 1, 3, 2] so
//     that the 4 / 2 / 2 / 1 classes fed by the shifts (0,0) / (0,1) / (1,0) / (1,1) are contiguous column ranges;
//   * persistent, warp-specialised CTAs (one per SM, tiles strided by gridDim.x): warp 0 = TMA producer, warp 1 = MMA
//     issuer, warps 2-9 = two epilogue warpgroups (one TMEM lane = one cell per thread: bias (folded BatchNorm), ReLU,
//     skip add, fp16 hi|lo split or the fused 1x1x1 `prob` conv).  Rings: full[s]/empty[s] for the operand stages,
//     accf[b]/acce[b] for the two TMEM accumulator buffers, so loads, MMAs and the epilogue of consecutive tiles overlap.
#include "conv3d_tc.cuh"

#include <cuda.h>

#include "linear_tc.cuh"
#include "umma.cuh"

namespace mvsf {

using namespace umma;

namespace c3 {
constexpr int NEPI = 256, THREADS = 64 + NEPI, MAX_STAGES = 8;   // warp 0: TMA, warp 1: MMA, warps 2-9: epilogue
template <int MODE, int NT>
struct Geo {
  static constexpr int TW = 8 * NT, TH = 16;
  static constexpr int PR = MODE == CONV_S1 ? TH + 2 : TH + 1;   // plane rows
  static constexpr int PC = MODE == CONV_S1 ? TW + 2 : TW + 1;   // plane columns (voxel octets)
  static constexpr int NSUB = MODE == CONV_S2 ? 4 : 1;           // parity sub-planes
  static constexpr uint32_t SUB_BYTES = PR * PC * 16;            // one plane; a TMA box = hi plane + lo plane
  static constexpr uint32_t PAIR = (2 * SUB_BYTES + 127) / 128 * 128;
  static constexpr uint32_t OCT_BYTES = NSUB * PAIR;             // everything of one channel octet
  static constexpr uint32_t PITCH = PC * 16;
};
__host__ __device__ inline int npad(int cout) { return cout < 16 ? 16 : cout; }
__host__ __device__ inline uint32_t slab_bytes(int cout) { return (uint32_t)npad(cout) * 576u; }  // 9 blocks x 2 variants x (2 x NPAD x 16 B)

struct alignas(64) Maps { CUtensorMap m[4]; };   // CONV_S2: one map per (h, w) parity; otherwise m[0]
}  // namespace c3

// depth taps (kd, id) of output slice od
struct DepthTaps { int n, kd[3], id[3]; };
template <int MODE>
__device__ __forceinline__ DepthTaps depth_taps(int od, int SD, int ID) {
  DepthTaps t;
  t.n = 0;
#pragma unroll
  for (int kd = 0; kd < 3; ++kd) {
    int id;
    bool ok = true;
    if (MODE == CONV_S1) id = od + kd - 1;
    else if (MODE == CONV_S2) id = od * SD + kd - 1;
    else {
      const int num = od + 1 - kd;
      if (SD == 1) id = num;
      else { ok = (num & 1) == 0; id = num >> 1; }
    }
    if (ok && id >= 0 && id < ID) { t.kd[t.n] = kd; t.id[t.n] = id; ++t.n; }
  }
  return t;
}

template <int MODE, int OUT>
__device__ __forceinline__ void conv_epilogue_item(const ConvTcArgs& a, uint32_t tcol, int NPAD, bool valid, size_t vox) {
  const int COUT = a.COUT;
  float prob = 0.f;
  for (int c16 = 0; c16 < NPAD / 16; ++c16) {
    float v[16];
    tmem_ld16(tcol + c16 * 16, v);
#pragma unroll
    for (int g = 0; g < 2; ++g) {
      const int c0 = c16 * 16 + g * 8;
      if (c0 >= COUT) continue;
      float x[8];
      const float4 b0 = ldg4(a.bias + c0), b1 = ldg4(a.bias + c0 + 4);
      x[0] = fmaxf(v[g * 8 + 0] + b0.x, 0.f); x[1] = fmaxf(v[g * 8 + 1] + b0.y, 0.f);
      x[2] = fmaxf(v[g * 8 + 2] + b0.z, 0.f); x[3] = fmaxf(v[g * 8 + 3] + b0.w, 0.f);
      x[4] = fmaxf(v[g * 8 + 4] + b1.x, 0.f); x[5] = fmaxf(v[g * 8 + 5] + b1.y, 0.f);
      x[6] = fmaxf(v[g * 8 + 6] + b1.z, 0.f); x[7] = fmaxf(v[g * 8 + 7] + b1.w, 0.f);
      if (!valid) continue;
      if (OUT == OUT_SPLIT) {
        if (a.skip_hi) {
          const uint4 sh = *reinterpret_cast<const uint4*>(a.skip_hi + vox * COUT + c0);
          const uint4 sl = *reinterpret_cast<const uint4*>(a.skip_lo + vox * COUT + c0);
          const __half2* h2 = reinterpret_cast<const __half2*>(&sh);
          const __half2* l2 = reinterpret_cast<const __half2*>(&sl);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 fh = __half22float2(h2[e]), fl = __half22float2(l2[e]);
            x[2 * e] += fh.x + fl.x;
            x[2 * e + 1] += fh.y + fl.y;
          }
        }
        split_store8(a.out_hi + vox * COUT + c0, a.out_lo + vox * COUT + c0, x);
      } else {
        const float4 s0 = ldg4(a.skip32 + vox * COUT + c0), s1 = ldg4(a.skip32 + vox * COUT + c0 + 4);
        x[0] += s0.x; x[1] += s0.y; x[2] += s0.z; x[3] += s0.w;
        x[4] += s1.x; x[5] += s1.y; x[6] += s1.z; x[7] += s1.w;
        if (OUT == OUT_F32) {
          float* op = a.out32 + vox * COUT + c0;
          *reinterpret_cast<float4*>(op) = make_float4(x[0], x[1], x[2], x[3]);
          *reinterpret_cast<float4*>(op + 4) = make_float4(x[4], x[5], x[6], x[7]);
        } else {
          if (c0 == 0) prob = __ldg(a.probw + COUT);
#pragma unroll
          for (int e = 0; e < 8; ++e) prob = fmaf(x[e], __ldg(a.probw + c0 + e), prob);
        }
      }
    }
  }
  if (OUT == OUT_PROB && valid) a.out32[vox] = prob;
}

// Persistent kernel: CTA i works on tiles i, i + gridDim.x, ...; tile = (output depth slice, 16 x 8*NT cells).
template <int MODE, int NT, int OUT>
__global__ void __launch_bounds__(c3::THREADS, 1)
conv3d_tc_kernel(const __grid_constant__ c3::Maps maps, ConvTcArgs a, int NS, int OD, int OH, int OW, int tiles_w,
                 int tiles_h, int ntiles) {
  using G = c3::Geo<MODE, NT>;
  constexpr int PC = G::PC, NSUB = G::NSUB;
  constexpr int NCLS = MODE == DECONV_S2 ? 4 : 1;
  extern __shared__ __align__(1024) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int CIN = a.CIN, COUT = a.COUT, SD = a.SD, ID = a.ID, IH = a.IH, IW = a.IW;
  const int NPAD = c3::npad(COUT);
  const int KG = a.KG;                                            // channel octets per unit
  const uint32_t b_bytes = c3::slab_bytes(COUT);
  const uint32_t a_bytes = (uint32_t)KG * G::OCT_BYTES;
  const uint32_t stage_bytes = (a_bytes + b_bytes + 127u) / 128u * 128u;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bars = sbase + NS * stage_bytes;                 // full[8] | empty[8] | accf[2] | acce[2] | tmem slot
  const uint32_t bar_full = bars, bar_empty = bars + 64, bar_accf = bars + 128, bar_acce = bars + 144;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + NS * stage_bytes + 160);
  const int ngroups = (CIN >> 3) / KG;
  const uint32_t acc_cols = (uint32_t)(NT * NCLS * NPAD);         // one accumulator buffer

  uint32_t ncols = 32;
  while (ncols < 2 * acc_cols) ncols <<= 1;
  if (tid == 0) {
    for (int i = 0; i < c3::MAX_STAGES; ++i) { mbar_init(bar_full + 8 * i, 1); mbar_init(bar_empty + 8 * i, 1); }
    mbar_init(bar_accf, 1); mbar_init(bar_accf + 8, 1);
    mbar_init(bar_acce, c3::NEPI); mbar_init(bar_acce + 8, c3::NEPI);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_slot)), ncols);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // --------------------------------------------------------------------------------------- TMA producer
    if (lane == 0) {
      uint32_t g = 0;
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int tw = tile % tiles_w, th = (tile / tiles_w) % tiles_h, od = tile / (tiles_w * tiles_h);
        const int c0h = th * 16, c0w = tw * G::TW;
        const DepthTaps dt = depth_taps<MODE>(od, SD, ID);
        for (int ds = 0; ds < dt.n; ++ds) {
          for (int grp = 0; grp < ngroups; ++grp, ++g) {
            const int s = g % NS;
            mbar_wait(bar_empty + 8 * s, (uint32_t)(((g / NS) & 1) ^ 1));
            const uint32_t st = sbase + s * stage_bytes, full = bar_full + 8 * s;
            expect_tx(full, (uint32_t)(KG * NSUB) * 2u * G::SUB_BYTES + b_bytes);
            for (int og = 0; og < KG; ++og) {
              const int c = (grp * KG + og) * 8;
#pragma unroll
              for (int sub = 0; sub < NSUB; ++sub) {
                int w0, h0;
                if (MODE == CONV_S1) { w0 = c0w - 1; h0 = c0h - 1; }
                else if (MODE == CONV_S2) { w0 = c0w - (sub & 1); h0 = c0h - (sub >> 1); }   // odd plane: index j <-> 2j + 1
                else { w0 = c0w; h0 = c0h; }
                tma_load_5d(st + (uint32_t)(og * NSUB + sub) * G::PAIR, &maps.m[sub], c, w0, h0, dt.id[ds], 0, full);
              }
            }
            bulk_load(st + a_bytes, a.wtc + (size_t)(dt.kd[ds] * ngroups + grp) * (b_bytes / 2), b_bytes, full);
          }
        }
      }
    }
  } else if (warp == 1) {
    // --------------------------------------------------------------------------------------- MMA issue
    {   // converged warp, one elected lane per tcgen05 instruction (see conv3d_col_kernel)
      const uint32_t blk = (uint32_t)NPAD * 32u;   // one weight block: NPAD rows x 2 k-chunks
      uint32_t g = 0;
      int it = 0;
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
        const int od = tile / (tiles_w * tiles_h);
        const DepthTaps dt = depth_taps<MODE>(od, SD, ID);
        const int U = dt.n * ngroups;
        const int buf = it & 1;
        mbar_wait(bar_acce + 8 * buf, (uint32_t)(((it >> 1) & 1) ^ 1));   // the epilogue has drained this accumulator buffer
        tc_fence_after_sync();
        const uint32_t tacc0 = tmem_base + (uint32_t)buf * acc_cols;
        for (int u = 0; u < U; ++u, ++g) {
          const int s = g % NS;
          mbar_wait(bar_full + 8 * s, (uint32_t)((g / NS) & 1));
          tc_fence_after_sync();
          const uint32_t sA = sbase + s * stage_bytes, sB = sA + a_bytes;
          // one fused tap group: A start offset, first weight block, number of blocks (N = nb * NPAD), accumulator column
          auto issue = [&](uint32_t aoff, int bstart, int nb, int dcol, bool overwrite) {
            const uint32_t n = (uint32_t)(nb * NPAD);
            const uint32_t idesc = make_idesc_f16(128, (int)n);
            const uint32_t t0 = sB + (uint32_t)bstart * 2u * blk, t1 = t0 + (uint32_t)nb * blk;
            const uint64_t b0 = make_desc(t0, n * 16u, 128), b1 = make_desc(t1, n * 16u, 128);
            // consecutive MMAs go to different accumulators (M-tiles): back-to-back MMAs on one accumulator serialise
            if (KG == 1) {
#pragma unroll
              for (int t = 0; t < NT; ++t)                                                       // K = [hi | lo] of one octet
                mma_f16_ss_elect(tacc0 + (uint32_t)(t * NCLS * NPAD + dcol), make_desc(sA + aoff + t * 128, G::SUB_BYTES, G::PITCH), b0,
                           idesc, overwrite ? 0u : 1u);                                        // x [w_hi ; w_hi]
#pragma unroll
              for (int t = 0; t < NT; ++t)
                mma_f16_ss_elect(tacc0 + (uint32_t)(t * NCLS * NPAD + dcol), make_desc(sA + aoff + t * 128, G::SUB_BYTES, G::PITCH), b1,
                           idesc, 1u);                                                         // x [w_lo ; 0]
            } else {
#pragma unroll
              for (int t = 0; t < NT; ++t)                                                       // K = two octets; lo planes
                mma_f16_ss_elect(tacc0 + (uint32_t)(t * NCLS * NPAD + dcol),
                           make_desc(sA + G::SUB_BYTES + aoff + t * 128, G::OCT_BYTES, G::PITCH), b0, idesc, overwrite ? 0u : 1u);  // x_lo * w_hi
#pragma unroll
              for (int t = 0; t < NT; ++t)
                mma_f16_ss_elect(tacc0 + (uint32_t)(t * NCLS * NPAD + dcol), make_desc(sA + aoff + t * 128, G::OCT_BYTES, G::PITCH), b1,
                           idesc, 1u);                                                         // x_hi * w_lo
#pragma unroll
              for (int t = 0; t < NT; ++t)
                mma_f16_ss_elect(tacc0 + (uint32_t)(t * NCLS * NPAD + dcol), make_desc(sA + aoff + t * 128, G::OCT_BYTES, G::PITCH), b0,
                           idesc, 1u);                                                         // x_hi * w_hi
            }
          };
          if (MODE == DECONV_S2) {
            // input shift (dih, diw) -> fused classes; weight blocks in conv3d_tc_pack's order
            issue(0u, 0, 4, 0, u == 0);                                   // (0,0): taps (1,1) (1,2) (2,2) (2,1) -> classes 0 1 3 2
            issue(16u, 4, 2, NPAD, false);                                // (0,1): taps (1,0) (2,0)             -> classes 1 3
            issue((uint32_t)PC * 16u, 6, 2, 2 * NPAD, false);             // (1,0): taps (0,2) (0,1)             -> classes 3 2
            issue((uint32_t)(PC + 1) * 16u, 8, 1, 2 * NPAD, false);       // (1,1): tap  (0,0)                   -> class 3
          } else {
#pragma unroll
            for (int kh = 0; kh < 3; ++kh) {
#pragma unroll
              for (int kw = 0; kw < 3; ++kw) {
                int sub = 0, rs = kh, cs = kw;
                if (MODE == CONV_S2) {
                  sub = (kh == 1 ? 0 : 2) + (kw == 1 ? 0 : 1);
                  rs = kh == 2 ? 1 : 0; cs = kw == 2 ? 1 : 0;
                }
                issue((uint32_t)sub * G::PAIR + (uint32_t)(rs * PC + cs) * 16u, kh * 3 + kw, 1, 0, u == 0 && kh == 0 && kw == 0);
              }
            }
          }
          commit_elect(bar_empty + 8 * s);
        }
        commit_elect(bar_accf + 8 * buf);
      }
    }
  } else {
    // --------------------------------------------------------------------------------------- epilogue (2 warpgroups)
    const int wg = (warp - 2) >> 2, quarter = warp & 3;   // a warp may only touch TMEM lanes 32 * (warp % 4) ...
    const int m = quarter * 32 + lane;                    // TMEM lane = GEMM row = cell (h = m / 8, w = m % 8) of an M-tile
    int it = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
      const int tw = tile % tiles_w, th = (tile / tiles_w) % tiles_h, od = tile / (tiles_w * tiles_h);
      const int buf = it & 1;
      mbar_wait(bar_accf + 8 * buf, (uint32_t)((it >> 1) & 1));
      tc_fence_after_sync();
      const uint32_t trow = tmem_base + (uint32_t)buf * acc_cols + ((uint32_t)(quarter * 32) << 16);
      const int ch = th * 16 + (m >> 3);
#pragma unroll 1
      for (int item = wg; item < NT * NCLS; item += 2) {
        const int t = item / NCLS, cls = item % NCLS;
        const int cw = tw * G::TW + t * 8 + (m & 7);
        int oh, ow;
        bool valid;
        if (MODE == DECONV_S2) { oh = 2 * ch + (cls >> 1); ow = 2 * cw + (cls & 1); valid = ch < IH && cw < IW; }
        else { oh = ch; ow = cw; valid = ch < OH && cw < OW; }
        const size_t vox = valid ? ((size_t)od * OH + oh) * OW + ow : 0;
        const uint32_t tcol = trow + (uint32_t)((t * NCLS + (cls ^ (cls >> 1))) * NPAD);   // class order [0, 1, 3, 2]
        conv_epilogue_item<MODE, OUT>(a, tcol, NPAD, valid, vox);
      }
      tc_fence_before_sync();
      mbar_arrive(bar_acce + 8 * buf);
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, ncols);
}


// ---------------------------------------------------------------------------------------------------------------------
// Depth-streaming variant for layers whose DEPTH stride is 1 (every 3x3x3 conv of CostRegNet3D, the stride-1 convs of
// CostRegNet).  The MMAs above are bound by the shared-memory read of the A operand (4 KB per instruction whatever N is),
// so instead of visiting an input slice three times - once per output slice it feeds - a work item is a COLUMN: a tile
// x a run of output depth slices [d0, d1).  Input slice `id` is loaded ONCE and one MMA per tap multiplies it with
// [W(kd=2) ; W(kd=1) ; W(kd=0)] (N = 3 * Cout), feeding the accumulators of the output slices id-1, id, id+1 at once.
// The accumulators live in a ring of 4 TMEM slots per M-tile (slot = od % 4, consecutive slots are contiguous columns,
// a window that wraps is issued as two MMAs); slice id-1 is complete once the MMAs of input slice id have retired and is
// drained by the epilogue warps while the next input slice is multiplied.  3x fewer A-operand reads and TMA bytes.
template <int MODE, int NT>
__global__ void __launch_bounds__(c3::THREADS, 1)
conv3d_col_kernel(const __grid_constant__ c3::Maps maps, ConvTcArgs a, int NS, int wres, int OH, int OW, int tiles_w,
                  int tiles_h, int DC, int nitems) {
  using G = c3::Geo<MODE, NT>;
  constexpr int PC = G::PC, NSUB = G::NSUB;
  extern __shared__ __align__(1024) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int CIN = a.CIN, COUT = a.COUT, D = a.ID;
  const int NPAD = c3::npad(COUT);
  const int KG = a.KG;
  const int ngroups = (CIN >> 3) / KG;
  const uint32_t slab = (uint32_t)NPAD * 1728u;                   // 9 taps x 2 variants x (2 k-chunks x 3*NPAD rows x 16 B)
  const uint32_t a_bytes = (uint32_t)KG * G::OCT_BYTES;
  const uint32_t stage_bytes = (a_bytes + (wres ? 0u : slab) + 127u) / 128u * 128u;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t wbase = sbase;                                   // resident weight slabs (wres)
  const uint32_t ring = sbase + (wres ? ((uint32_t)ngroups * slab + 127u) / 128u * 128u : 0u);
  const uint32_t bars = ring + NS * stage_bytes;                  // full[8] | empty[8] | accf[4] | acce[4] | wbar | tmem slot
  const uint32_t bar_full = bars, bar_empty = bars + 64, bar_accf = bars + 128, bar_acce = bars + 160, bar_w = bars + 192;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + (bars - sbase) + 200);

  uint32_t ncols = 32;
  while (ncols < (uint32_t)(4 * NT * NPAD)) ncols <<= 1;
  if (tid == 0) {
    for (int i = 0; i < c3::MAX_STAGES; ++i) { mbar_init(bar_full + 8 * i, 1); mbar_init(bar_empty + 8 * i, 1); }
    for (int i = 0; i < 4; ++i) { mbar_init(bar_accf + 8 * i, 1); mbar_init(bar_acce + 8 * i, c3::NEPI); }
    mbar_init(bar_w, 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_slot)), ncols);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  const int tiles_hw = tiles_w * tiles_h;

  if (warp == 0) {
    // --------------------------------------------------------------------------------------- TMA producer
    if (lane == 0) {
      if (wres) {
        expect_tx(bar_w, (uint32_t)ngroups * slab);
        for (int grp = 0; grp < ngroups; ++grp) bulk_load(wbase + grp * slab, a.wtc + (size_t)grp * (slab / 2), slab, bar_w);
      }
      uint32_t g = 0;
      for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
        const int tw = item % tiles_w, th = (item / tiles_w) % tiles_h, ck = item / tiles_hw;
        const int c0h = th * 16, c0w = tw * G::TW;
        const int d0 = ck * DC, d1 = min(D, d0 + DC);
        const int first_id = max(d0 - 1, 0), last_id = min(d1, D - 1);
        for (int id = first_id; id <= last_id; ++id) {
          for (int grp = 0; grp < ngroups; ++grp, ++g) {
            const int s = g % NS;
            mbar_wait(bar_empty + 8 * s, (uint32_t)(((g / NS) & 1) ^ 1));
            const uint32_t st = ring + s * stage_bytes, full = bar_full + 8 * s;
            expect_tx(full, (uint32_t)(KG * NSUB) * 2u * G::SUB_BYTES + (wres ? 0u : slab));
            for (int og = 0; og < KG; ++og) {
              const int c = (grp * KG + og) * 8;
#pragma unroll
              for (int sub = 0; sub < NSUB; ++sub) {
                int w0, h0;
                if (MODE == CONV_S1) { w0 = c0w - 1; h0 = c0h - 1; }
                else { w0 = c0w - (sub & 1); h0 = c0h - (sub >> 1); }
                tma_load_5d(st + (uint32_t)(og * NSUB + sub) * G::PAIR, &maps.m[sub], c, w0, h0, id, 0, full);
              }
            }
            if (!wres) bulk_load(st + a_bytes, a.wtc + (size_t)grp * (slab / 2), slab, full);
          }
        }
      }
    }
  } else if (warp == 1) {
    // --------------------------------------------------------------------------------------- MMA issue
    // The whole warp runs this code converged (every value is warp-uniform and lives in uniform registers); one elected
    // lane issues each tcgen05 instruction.  An `if (lane == 0)` version costs ~20 instructions per MMA (per-instruction
    // divergence handling + register -> uniform register moves) and the issuing thread is the bottleneck of the kernel.
    {
      if (wres) mbar_wait(bar_w, 0u);
      const uint32_t btile = (uint32_t)NPAD * 96u;    // one (tap, variant) weight tile: 2 k-chunks x 3*NPAD rows x 16 B
      const uint32_t blbo = (uint32_t)NPAD * 48u;     // k-chunk stride inside a weight tile
      uint32_t g = 0, pm = 0;                         // pm bit s: parity of the number of completed uses of slot s
      for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
        const int ck = item / tiles_hw;
        const int d0 = ck * DC, d1 = min(D, d0 + DC);
        const int first_id = max(d0 - 1, 0), last_id = min(d1, D - 1);
        for (int id = first_id; id <= last_id; ++id) {
          const int oa = max(id - 1, d0), ob = min(id + 1, d1 - 1);       // output slices fed by this input slice
          const int fa = id == first_id ? oa : id + 1;                    // [fa, ob]: slices that receive their FIRST contribution
          for (int od = fa; od <= ob; ++od) mbar_wait(bar_acce + 8 * (od & 3), ((pm >> (od & 3)) & 1u) ^ 1u);  // slot drained
          tc_fence_after_sync();
          for (int grp = 0; grp < ngroups; ++grp, ++g) {
            const int s = g % NS;
            mbar_wait(bar_full + 8 * s, (uint32_t)((g / NS) & 1));
            tc_fence_after_sync();
            const uint32_t sA = ring + s * stage_bytes;
            const uint32_t sB = wres ? wbase + grp * slab : sA + a_bytes;
            // MMAs of one (tap, variant) over the output slices [x, y]; a window that wraps around the 4-slot ring is split
            auto mma_range = [&](int x, int y, bool overwrite, uint32_t astart, uint32_t albo, uint32_t tile) {
              while (x <= y) {
                const int sx = x & 3;
                const int len = min(y - x + 1, 4 - sx);
                const uint32_t n = (uint32_t)(len * NPAD);
                const uint32_t idesc = make_idesc_f16(128, (int)n);
                const uint64_t bd = make_desc(tile + (uint32_t)((x - id + 1) * NPAD) * 16u, blbo, 128);
#pragma unroll
                for (int t = 0; t < NT; ++t)
                  mma_f16_ss_elect(tmem_base + (uint32_t)((t * 4 + sx) * NPAD), make_desc(astart + t * 128, albo, G::PITCH), bd, idesc,
                                   overwrite ? 0u : 1u);
                x += len;
              }
            };
#pragma unroll
            for (int kh = 0; kh < 3; ++kh) {
#pragma unroll
              for (int kw = 0; kw < 3; ++kw) {
                int sub = 0, rs = kh, cs = kw;
                if (MODE == CONV_S2) {
                  sub = (kh == 1 ? 0 : 2) + (kw == 1 ? 0 : 1);
                  rs = kh == 2 ? 1 : 0; cs = kw == 2 ? 1 : 0;
                }
                const uint32_t aoff = sA + (uint32_t)sub * G::PAIR + (uint32_t)(rs * PC + cs) * 16u;
                const uint32_t t0 = sB + (uint32_t)(kh * 3 + kw) * 2u * btile, t1 = t0 + btile;   // w_hi tile, w_lo tile
                const bool first = grp == 0 && kh == 0 && kw == 0;
                // variant list: (A start, A k-chunk stride, weight tile)
                const uint32_t va[3] = {KG == 1 ? aoff : aoff + G::SUB_BYTES, KG == 1 ? aoff : aoff, aoff};
                const uint32_t vl = KG == 1 ? G::SUB_BYTES : G::OCT_BYTES;
                const uint32_t vt[3] = {t0, t1, t0};
                const int nv = KG == 1 ? 2 : 3;     // KG 1: x [w_hi;w_hi], x [w_lo;0]   KG 2: x_lo*w_hi, x_hi*w_lo, x_hi*w_hi
#pragma unroll
                for (int v = 0; v < 3; ++v) {
                  if (v >= nv) break;
                  if (first && v == 0) {
                    if (fa > oa) mma_range(oa, fa - 1, false, va[v], vl, vt[v]);
                    if (fa <= ob) mma_range(fa, ob, true, va[v], vl, vt[v]);
                  } else {
                    mma_range(oa, ob, false, va[v], vl, vt[v]);
                  }
                }
              }
            }
            commit_elect(bar_empty + 8 * s);
          }
          if (id - 1 >= d0) { commit_elect(bar_accf + 8 * ((id - 1) & 3)); pm ^= 1u << ((id - 1) & 3); }
          if (id == last_id && id <= d1 - 1) { commit_elect(bar_accf + 8 * (id & 3)); pm ^= 1u << (id & 3); }
        }
      }
    }
  } else {
    // --------------------------------------------------------------------------------------- epilogue (2 warpgroups)
    const int wg = (warp - 2) >> 2, quarter = warp & 3;
    const int m = quarter * 32 + lane;
    uint32_t pm = 0;
    for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
      const int tw = item % tiles_w, th = (item / tiles_w) % tiles_h, ck = item / tiles_hw;
      const int d0 = ck * DC, d1 = min(D, d0 + DC);
      const int ch = th * 16 + (m >> 3);
      for (int od = d0; od < d1; ++od) {
        const int slot = od & 3;
        mbar_wait(bar_accf + 8 * slot, (pm >> slot) & 1u);
        pm ^= 1u << slot;
        tc_fence_after_sync();
        const uint32_t trow = tmem_base + ((uint32_t)(quarter * 32) << 16);
#pragma unroll 1
        for (int t = wg; t < NT; t += 2) {
          const int cw = tw * G::TW + t * 8 + (m & 7);
          const bool valid = ch < OH && cw < OW;
          const size_t vox = valid ? ((size_t)od * OH + ch) * OW + cw : 0;
          conv_epilogue_item<MODE, OUT_SPLIT>(a, trow + (uint32_t)((t * 4 + slot) * NPAD), NPAD, valid, vox);
        }
        tc_fence_before_sync();
        mbar_arrive(bar_acce + 8 * slot);
      }
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, ncols);
}

// ------------------------------------------------------------------------------------------------------- host
int conv3d_tc_kg(int mode, int cin) { return (mode != CONV_S2 && cin >= 16) ? 2 : 1; }
// depth-streaming kernel: convolutions with depth stride 1 whose 3*Cout-wide weight tiles still fit shared memory
int conv3d_tc_col(int mode, int sd, int cout) { return (mode == CONV_S1 || (mode == CONV_S2 && sd == 1)) && c3::npad(cout) <= 32; }

size_t conv3d_tc_packed_halves(int mode, int cin, int cout) {   // the same for both layouts
  return (size_t)3 * (cin / 8 / conv3d_tc_kg(mode, cin)) * (c3::slab_bytes(cout) / 2);
}

// slab (kd, channel group g) = 9 weight blocks of [2 MMA variants][2 k-chunks][NPAD rows][8 halves]; blocks that are fused
// into one MMA are interleaved as [variant][k-chunk][nb * NPAD rows][8] (conv: nb = 1; deconv: 4, 2, 2, 1)
// col layout (depth-streaming kernel): slab (channel group g) = [9 taps][2 variants][2 k-chunks][kd = 2, 1, 0][NPAD rows][8]
__global__ void conv3d_tc_pack_kernel(const float* __restrict__ w32, __half* __restrict__ out, int cin, int cout, int NPAD,
                                      int KG, int deconv, int col, size_t total) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int e = (int)(i & 7);
  const size_t q = i >> 3;                           // 16-byte chunk
  const int per_slab = col ? NPAD * 108 : NPAD * 36;
  const int slab = (int)(q / per_slab), c = (int)(q % per_slab);
  const int ngroups = cin / 8 / KG;
  int kd = slab / ngroups, g = slab % ngroups;
  int mm, kc, n, kh, kw;
  if (col) {
    g = slab;
    n = c % NPAD;
    int r = c / NPAD;
    kd = 2 - r % 3; r /= 3;
    kc = r & 1; r >>= 1;
    mm = r & 1; r >>= 1;
    kh = r / 3; kw = r % 3;
  } else if (!deconv) {
    n = c % NPAD;
    int r = c / NPAD;
    kc = r & 1; r >>= 1;
    mm = r & 1; r >>= 1;
    kh = r / 3; kw = r % 3;
  } else {
    const int bs[4] = {0, 4, 6, 8}, nbs[4] = {4, 2, 2, 1};
    const int tkh[4][4] = {{1, 1, 2, 2}, {1, 2, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}};
    const int tkw[4][4] = {{1, 2, 2, 1}, {0, 0, 0, 0}, {2, 1, 0, 0}, {0, 0, 0, 0}};
    int t = 3;
    for (int k = 0; k < 3; ++k)
      if (c < bs[k + 1] * 4 * NPAD) { t = k; break; }
    const int cc = c - bs[t] * 4 * NPAD, nb = nbs[t];
    mm = cc / (2 * nb * NPAD);
    kc = (cc / (nb * NPAD)) & 1;
    const int nn = cc % (nb * NPAD);
    const int b = nn / NPAD;
    n = nn % NPAD;
    kh = tkh[t][b]; kw = tkw[t][b];
  }
  const int ci = (KG == 1 ? g : g * 2 + kc) * 8 + e;
  float w = 0.f;
  if (n < cout) w = w32[((size_t)((kd * 3 + kh) * 3 + kw) * cin + ci) * cout + n];
  const __half hi = __float2half_rn(w);
  const __half lo = __float2half_rn(w - __half2float(hi));
  __half v;
  if (KG == 1) v = mm == 0 ? hi : (kc == 0 ? lo : __float2half_rn(0.f));
  else v = mm == 0 ? hi : lo;
  out[i] = v;
}

int conv3d_tc_pack(const float* w32, __half* out, int mode, int sd, int cin, int cout, cudaStream_t s) {
  MVSF_REQUIRE(w32 && out && cin % 8 == 0 && cout % 8 == 0, "conv3d_tc_pack: bad arguments");
  const size_t total = conv3d_tc_packed_halves(mode, cin, cout);
  conv3d_tc_pack_kernel<<<cdiv((long long)total, 256), 256, 0, s>>>(w32, out, cin, cout, c3::npad(cout),
                                                                     conv3d_tc_kg(mode, cin), mode == DECONV_S2 ? 1 : 0,
                                                                     conv3d_tc_col(mode, sd, cout), total);
  MVSF_LAUNCH_CHECK("conv3d_tc_pack");
  return MVSF_OK;
}

__global__ void split_vec8_kernel(const float* __restrict__ x, __half* __restrict__ hi, __half* __restrict__ lo, size_t n8) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n8) return;
  const float4 a = ldg4(x + i * 8), b = ldg4(x + i * 8 + 4);
  const float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  split_store8(hi + i * 8, lo + i * 8, v);
}
__global__ void merge_vec8_kernel(const __half* __restrict__ hi, const __half* __restrict__ lo, float* __restrict__ x, size_t n8) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n8) return;
  const uint4 h = *reinterpret_cast<const uint4*>(hi + i * 8), l = *reinterpret_cast<const uint4*>(lo + i * 8);
  const __half2* h2 = reinterpret_cast<const __half2*>(&h);
  const __half2* l2 = reinterpret_cast<const __half2*>(&l);
  float r[8];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float2 fh = __half22float2(h2[e]), fl = __half22float2(l2[e]);
    r[2 * e] = fh.x + fl.x;
    r[2 * e + 1] = fh.y + fl.y;
  }
  *reinterpret_cast<float4*>(x + i * 8) = make_float4(r[0], r[1], r[2], r[3]);
  *reinterpret_cast<float4*>(x + i * 8 + 4) = make_float4(r[4], r[5], r[6], r[7]);
}
int launch_split_vec8(const float* x, __half* hi, __half* lo, size_t n, cudaStream_t s) {
  MVSF_REQUIRE(x && hi && lo && n > 0 && n % 8 == 0, "split_vec8: bad arguments");
  split_vec8_kernel<<<cdiv((long long)(n / 8), 256), 256, 0, s>>>(x, hi, lo, n / 8);
  MVSF_LAUNCH_CHECK("split_vec8");
  return MVSF_OK;
}
int launch_merge_vec8(const __half* hi, const __half* lo, float* x, size_t n, cudaStream_t s) {
  MVSF_REQUIRE(x && hi && lo && n > 0 && n % 8 == 0, "merge_vec8: bad arguments");
  merge_vec8_kernel<<<cdiv((long long)(n / 8), 256), 256, 0, s>>>(hi, lo, x, n / 8);
  MVSF_LAUNCH_CHECK("merge_vec8");
  return MVSF_OK;
}

// 5-D map (c, w, h, d, hi|lo) over the fp16 activation pair; sh/sw = 2 and (ph, pw) select one parity plane of (h, w)
static int make_map(CUtensorMap* m, const __half* hi, const __half* lo, int C, int D, int H, int W, int sh, int sw, int ph,
                    int pw, int box_w, int box_h) {
  EncodeTiledFn enc = encode_tiled_fn();
  MVSF_REQUIRE(enc, "conv3d_tc: cuTensorMapEncodeTiled is not available from this driver");
  const long long lo_off = (lo - hi) * (long long)sizeof(__half);
  MVSF_REQUIRE(lo_off > 0 && lo_off % 16 == 0, "conv3d_tc: the lo tensor must follow the hi tensor at a 16-byte multiple");
  const cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)((W - pw + sw - 1) / sw), (cuuint64_t)((H - ph + sh - 1) / sh), (cuuint64_t)D, 2};
  const cuuint64_t strides[4] = {(cuuint64_t)sw * C * 2, (cuuint64_t)sh * W * C * 2, (cuuint64_t)H * W * C * 2, (cuuint64_t)lo_off};
  const cuuint32_t box[5] = {8, (cuuint32_t)box_w, (cuuint32_t)box_h, 1, 2};
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  void* base = const_cast<__half*>(hi + ((size_t)ph * W + pw) * C);
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(MVSF_ERR_CUDA, "conv3d_tc: cuTensorMapEncodeTiled failed (%d) for C=%d D=%d H=%d W=%d", (int)r, C, D, H, W);
  return MVSF_OK;
}

template <int MODE, int NT, int OUT>
static int launch_one(const ConvTcArgs& a, int NS, size_t smem, int OD, int OH, int OW, int cells_h, int cells_w,
                      int num_sms, cudaStream_t s) {
  using G = c3::Geo<MODE, NT>;
  auto kern = conv3d_tc_kernel<MODE, NT, OUT>;
  static DeviceOnce once;
  const int dev = current_device();
  if (once.need(dev)) {
    MVSF_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    once.done(dev);
  }
  c3::Maps maps;
  int rc;
  if (MODE == CONV_S2) {
    for (int sub = 0; sub < 4; ++sub)
      if ((rc = make_map(&maps.m[sub], a.in_hi, a.in_lo, a.CIN, a.ID, a.IH, a.IW, 2, 2, sub >> 1, sub & 1, G::PC, G::PR))) return rc;
  } else {
    if ((rc = make_map(&maps.m[0], a.in_hi, a.in_lo, a.CIN, a.ID, a.IH, a.IW, 1, 1, 0, 0, G::PC, G::PR))) return rc;
    maps.m[1] = maps.m[2] = maps.m[3] = maps.m[0];
  }
  const int tiles_w = cdiv(cells_w, 8 * NT), tiles_h = cdiv(cells_h, 16);
  const long long ntiles = (long long)tiles_w * tiles_h * OD;
  MVSF_REQUIRE(ntiles < (1ll << 30), "conv3d_tc: volume too large");
  const int grid = (int)(ntiles < num_sms ? ntiles : num_sms);
  kern<<<grid, c3::THREADS, smem, s>>>(maps, a, NS, OD, OH, OW, tiles_w, tiles_h, (int)ntiles);
  MVSF_LAUNCH_CHECK("conv3d_tc");
  return MVSF_OK;
}

template <int MODE, int OUT>
static int launch_mode(const ConvTcArgs& a, cudaStream_t s) {
  int OD, OH, OW, cells_h, cells_w;
  if (MODE == CONV_S1) { OD = a.ID; OH = a.IH; OW = a.IW; cells_h = OH; cells_w = OW; }
  else if (MODE == CONV_S2) { OD = (a.ID - 1) / a.SD + 1; OH = (a.IH - 1) / 2 + 1; OW = (a.IW - 1) / 2 + 1; cells_h = OH; cells_w = OW; }
  else { OD = a.ID * a.SD; OH = a.IH * 2; OW = a.IW * 2; cells_h = a.IH; cells_w = a.IW; }
  const int num_sms = device_sm_count(current_device());
  const int NPAD = c3::npad(a.COUT);
  const uint32_t b_bytes = c3::slab_bytes(a.COUT);
  const int ncls = MODE == DECONV_S2 ? 4 : 1;
  // tile width: the widest tile (least halo) whose two accumulator buffers fit TMEM and that keeps the persistent CTAs busy
  int best_nt = 0;
  double best_eff = -1.0;
  const int nts[3] = {4, 2, 1};
  size_t stage_of[5] = {0, 0, 0, 0, 0};
  for (int k = 0; k < 3; ++k) {
    const int nt = nts[k];
    const uint32_t oct = nt == 4 ? c3::Geo<MODE, 4>::OCT_BYTES : (nt == 2 ? c3::Geo<MODE, 2>::OCT_BYTES : c3::Geo<MODE, 1>::OCT_BYTES);
    const size_t stage = align_up((size_t)a.KG * oct + b_bytes, 128);
    stage_of[nt] = stage;
    if (2 * nt * ncls * NPAD > 512 || 2 * stage + 256 > 227 * 1024) continue;
    const long long ntiles = (long long)cdiv(cells_w, 8 * nt) * cdiv(cells_h, 16) * OD;
    const double eff = (double)ntiles / (double)(cdiv(ntiles, num_sms) * (long long)num_sms);
    if (eff >= 0.85) { best_nt = nt; break; }
    if (eff > best_eff) { best_eff = eff; best_nt = nt; }
  }
  MVSF_REQUIRE(best_nt > 0, "conv3d_tc: no tile shape fits (COUT %d)", a.COUT);
  const size_t stage = stage_of[best_nt];
  int NS = (int)((227 * 1024 - 256) / stage);
  if (NS > c3::MAX_STAGES) NS = c3::MAX_STAGES;
  const size_t smem = NS * stage + 256;
  switch (best_nt) {
    case 4: return launch_one<MODE, 4, OUT>(a, NS, smem, OD, OH, OW, cells_h, cells_w, num_sms, s);
    case 2: return launch_one<MODE, 2, OUT>(a, NS, smem, OD, OH, OW, cells_h, cells_w, num_sms, s);
    default: return launch_one<MODE, 1, OUT>(a, NS, smem, OD, OH, OW, cells_h, cells_w, num_sms, s);
  }
}


template <int MODE, int NT>
static int launch_col_one(const ConvTcArgs& a, int NS, int wres, size_t smem, int OH, int OW, int DC, int num_sms, cudaStream_t s) {
  using G = c3::Geo<MODE, NT>;
  auto kern = conv3d_col_kernel<MODE, NT>;
  static DeviceOnce once;
  const int dev = current_device();
  if (once.need(dev)) {
    MVSF_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    once.done(dev);
  }
  c3::Maps maps;
  int rc;
  if (MODE == CONV_S2) {
    for (int sub = 0; sub < 4; ++sub)
      if ((rc = make_map(&maps.m[sub], a.in_hi, a.in_lo, a.CIN, a.ID, a.IH, a.IW, 2, 2, sub >> 1, sub & 1, G::PC, G::PR))) return rc;
  } else {
    if ((rc = make_map(&maps.m[0], a.in_hi, a.in_lo, a.CIN, a.ID, a.IH, a.IW, 1, 1, 0, 0, G::PC, G::PR))) return rc;
    maps.m[1] = maps.m[2] = maps.m[3] = maps.m[0];
  }
  const int tiles_w = cdiv(OW, 8 * NT), tiles_h = cdiv(OH, 16);
  const long long nitems = (long long)tiles_w * tiles_h * cdiv(a.ID, DC);
  MVSF_REQUIRE(nitems < (1ll << 30), "conv3d_tc: volume too large");
  const int grid = (int)(nitems < num_sms ? nitems : num_sms);
  kern<<<grid, c3::THREADS, smem, s>>>(maps, a, NS, wres, OH, OW, tiles_w, tiles_h, DC, (int)nitems);
  MVSF_LAUNCH_CHECK("conv3d_col");
  return MVSF_OK;
}

template <int MODE>
static int launch_col(const ConvTcArgs& a, cudaStream_t s) {
  const int D = a.ID;
  const int OH = MODE == CONV_S1 ? a.IH : (a.IH - 1) / 2 + 1, OW = MODE == CONV_S1 ? a.IW : (a.IW - 1) / 2 + 1;
  const int num_sms = device_sm_count(current_device());
  const int NPAD = c3::npad(a.COUT);
  const int ngroups = a.CIN / 8 / a.KG;
  const size_t slab = (size_t)NPAD * 1728;
  const size_t wres_bytes = align_up(ngroups * slab, 128);
  const int wres = wres_bytes <= 112 * 1024 ? 1 : 0;            // all weight slabs stay resident in shared memory
  // (tile width, depth run) with the least redundant halo traffic per useful output at full occupancy of the persistent CTAs
  int best_nt = 0, best_dc = 0, best_ns = 0;
  size_t best_smem = 0;
  double best_cost = 1e30;
  const int nts[3] = {4, 2, 1};
  for (int k = 0; k < 3; ++k) {
    const int nt = nts[k];
    if (4 * nt * NPAD > 512) continue;
    const uint32_t oct = nt == 4 ? c3::Geo<MODE, 4>::OCT_BYTES : (nt == 2 ? c3::Geo<MODE, 2>::OCT_BYTES : c3::Geo<MODE, 1>::OCT_BYTES);
    const size_t stage = align_up((size_t)a.KG * oct + (wres ? 0 : slab), 128);
    const size_t fixed = (wres ? wres_bytes : 0) + 256;
    int ns = (int)((227 * 1024 - fixed) / stage);
    if (ns > c3::MAX_STAGES) ns = c3::MAX_STAGES;
    if (ns < 2) continue;
    for (int div = 1; div <= 8; div *= 2) {
      const int dc = cdiv(D, div);
      if (div > 1 && dc == cdiv(D, div / 2)) continue;
      const long long items = (long long)cdiv(OW, 8 * nt) * cdiv(OH, 16) * cdiv(D, dc);
      const double eff = (double)items / (double)(cdiv(items, num_sms) * (long long)num_sms);
      const double halo_w = MODE == CONV_S1 ? (8.0 * nt + 2) / (8.0 * nt) : (16.0 * nt + 1) / (16.0 * nt);
      const double halo_d = dc >= D ? 1.0 : (dc + 2.0) / dc;
      const double cost = halo_w * halo_d / eff;
      if (cost < best_cost) { best_cost = cost; best_nt = nt; best_dc = dc; best_ns = ns; best_smem = fixed + ns * stage; }
    }
  }
  MVSF_REQUIRE(best_nt > 0, "conv3d_col: no tile shape fits (CIN %d COUT %d)", a.CIN, a.COUT);
  switch (best_nt) {
    case 4: return launch_col_one<MODE, 4>(a, best_ns, wres, best_smem, OH, OW, best_dc, num_sms, s);
    case 2: return launch_col_one<MODE, 2>(a, best_ns, wres, best_smem, OH, OW, best_dc, num_sms, s);
    default: return launch_col_one<MODE, 1>(a, best_ns, wres, best_smem, OH, OW, best_dc, num_sms, s);
  }
}

int launch_conv3d_tc(const ConvTcArgs& a, int mode, int out_mode, cudaStream_t s) {
  MVSF_REQUIRE(a.in_hi && a.in_lo && a.wtc && a.bias, "conv3d_tc: null pointer");
  MVSF_REQUIRE(a.CIN % 8 == 0 && a.CIN >= 8 && a.CIN <= 64 && a.COUT % 8 == 0 && a.COUT >= 8 && a.COUT <= 64 &&
                   (a.COUT == 8 || a.COUT % 16 == 0), "conv3d_tc: channels must be 8, 16, 32, 48 or 64");
  MVSF_REQUIRE(a.SD == 1 || a.SD == 2, "conv3d_tc: depth stride must be 1 or 2");
  MVSF_REQUIRE(a.KG == conv3d_tc_kg(mode, a.CIN), "conv3d_tc: KG must be conv3d_tc_kg(mode, CIN) (it fixes the weight slab layout)");
  MVSF_REQUIRE(((uintptr_t)a.in_hi & 15) == 0 && ((uintptr_t)a.in_lo & 15) == 0 && ((uintptr_t)a.wtc & 15) == 0,
               "conv3d_tc: operands must be 16-byte aligned");
  MVSF_REQUIRE(a.col == conv3d_tc_col(mode, a.SD, a.COUT), "conv3d_tc: col must be conv3d_tc_col(mode, SD, COUT) (weight slab layout)");
  if (out_mode == OUT_SPLIT) {
    MVSF_REQUIRE(a.out_hi && a.out_lo, "conv3d_tc: split output missing");
    if (a.col) return mode == CONV_S1 ? launch_col<CONV_S1>(a, s) : launch_col<CONV_S2>(a, s);
    if (mode == CONV_S1) return launch_mode<CONV_S1, OUT_SPLIT>(a, s);
    if (mode == CONV_S2) return launch_mode<CONV_S2, OUT_SPLIT>(a, s);
    if (mode == DECONV_S2) return launch_mode<DECONV_S2, OUT_SPLIT>(a, s);
  } else if (mode == DECONV_S2 && (out_mode == OUT_F32 || out_mode == OUT_PROB)) {
    MVSF_REQUIRE(a.out32 && a.skip32 && a.COUT == 8 && (out_mode == OUT_F32 || a.probw), "conv3d_tc: fp32 output needs out32, skip32, COUT == 8");
    if (out_mode == OUT_F32) return launch_mode<DECONV_S2, OUT_F32>(a, s);
    return launch_mode<DECONV_S2, OUT_PROB>(a, s);
  }
  return fail(MVSF_ERR_INVALID, "conv3d_tc: unsupported mode %d / output %d", mode, out_mode);
}

}  // namespace mvsf

using namespace mvsf;

/* Test entry: one 3x3x3 layer through the tensor-core path with fp32 in/out (split, pack and merge done here).
 * in [ID][IH][IW][cin]; w32 = [27][cin][cout] then bias[cout]; skip (optional) and out [OD][OH][OW][cout]. */
extern "C" int mvsf_conv3d_tc_layer(int mode, int sd, const float* in, const float* w32, const float* skip, float* out,
                                    void* workspace, size_t workspace_bytes, int cin, int cout, int ID, int IH, int IW,
                                    mvsf_stream_t stream) {
  MVSF_REQUIRE(in && w32 && out && workspace && (mode >= 0 && mode <= 2) && (sd == 1 || sd == 2), "conv3d_tc_layer: bad arguments");
  MVSF_REQUIRE(cin % 8 == 0 && cout % 8 == 0, "conv3d_tc_layer: channels must be multiples of 8");
  int OD, OH, OW;
  if (mode == CONV_S1) { OD = ID; OH = IH; OW = IW; }
  else if (mode == CONV_S2) { OD = (ID - 1) / sd + 1; OH = (IH - 1) / 2 + 1; OW = (IW - 1) / 2 + 1; }
  else { OD = ID * sd; OH = IH * 2; OW = IW * 2; }
  const size_t nin = (size_t)ID * IH * IW * cin, nout = (size_t)OD * OH * OW * cout;
  const size_t nw = align_up(conv3d_tc_packed_halves(mode, cin, cout), 64);
  const size_t need = (2 * nin + 4 * nout + nw) * sizeof(__half) + 256;
  if (workspace_bytes < need) return fail(MVSF_ERR_WORKSPACE, "conv3d_tc_layer: workspace %zu < %zu bytes", workspace_bytes, need);
  cudaStream_t s = (cudaStream_t)stream;
  __half* xin = reinterpret_cast<__half*>(workspace);
  __half* xout = xin + 2 * nin;
  __half* xskip = xout + 2 * nout;
  __half* wtc = xskip + 2 * nout;
  int rc;
  if ((rc = launch_split_vec8(in, xin, xin + nin, nin, s))) return rc;
  if (skip && (rc = launch_split_vec8(skip, xskip, xskip + nout, nout, s))) return rc;
  if ((rc = conv3d_tc_pack(w32, wtc, mode, sd, cin, cout, s))) return rc;
  ConvTcArgs a{};
  a.in_hi = xin; a.in_lo = xin + nin; a.wtc = wtc; a.bias = w32 + (size_t)27 * cin * cout;
  if (skip) { a.skip_hi = xskip; a.skip_lo = xskip + nout; }
  a.out_hi = xout; a.out_lo = xout + nout;
  a.CIN = cin; a.COUT = cout; a.SD = sd; a.ID = ID; a.IH = IH; a.IW = IW; a.KG = conv3d_tc_kg(mode, cin);
  a.col = conv3d_tc_col(mode, sd, cout);
  if ((rc = launch_conv3d_tc(a, mode, OUT_SPLIT, s))) return rc;
  return launch_merge_vec8(xout, xout + nout, out, nout, s);
}
