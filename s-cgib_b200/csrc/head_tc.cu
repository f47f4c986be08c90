// head_tc.cu - head MLP forward on the tensor cores (hidden 64, fp32 data):
//     Z = Wm2 relu(Wm1 [noisy || alpha C] + bm1) + bm2                  (reference models.py:676, 749)
// Same warp-specialised persistent pipeline as the GIN forward kernels (producer warps -> GEMM1 -> epilogue 1 -> GEMM2 ->
// epilogue 2, two stages of operand tiles and TMEM accumulators, mbarrier hand-offs), with the operand scheme of
// contrastive_tc.cu: every fp32 operand is a TWO-TERM FP16 SPLIT v = hi + 2^-11 lo' (hi = fp16(v), lo' = fp16((v - hi) 2^11):
// 22 significand bits at every magnitude) and a product is two kind::f16 MMAs per K = 16 step: A_hi x [B_hi | B_lo'] (N = 128:
// the hi hi and hi lo' parts in separate accumulator columns) and A_lo' x B_hi accumulated into the lo' columns; the epilogue
// forms hh + 2^-11 (hl' + l'h) - the same 2^-22-class product as the 3xTF32 scheme of the GIN kernels, with half the MMAs
// (16 + 8 per 128-row tile) and half the operand bytes.  The weights are scaled by 2^4 (undone exactly in the epilogues).  The
// inputs are used as they are when their magnitudes stay below 2^5 (GIN: relu(BN(.)) features, O(1)); otherwise (GraphSAGE /
// GCN features end without an activation, and the op entry accepts any magnitude) the caller passes max |noisy|, max |C| and
// max |alpha| in device slots (xmax) and the producers multiply [noisy || alpha C] by the power of two S that brings that bound
// into [2^4, 2^5).  The head is positively homogeneous up to its biases, so r' = relu(W1 S x + S b1) = S r and the epilogues undo
// S exactly with the 2^-4 of the weights: no rounding changes, no host synchronisation.  fp16's range then holds r' up to
// ||W1||_inf ~ 2^11; the operands are still clamped to +-65504 as a last resort.  r = relu(u + b1) goes to GEMM2 through TENSOR
// MEMORY (16-bit A operand: two K values per column).
// Producers build [noisy || alpha C] (never materialised in HBM unless the caller asks for interaction_map) with 32-byte
// loads of 8 channels; alpha C and r are saved for the head backward.  Replaces the FP32-FFMA head_fwd_kernel (75 -> ~25 us
// at N = 61 k rows), which remains the hidden-128 / cross-check path (SCGIB_HEAD_FFMA=1).  bf16 mode: optional bf16 copies of
// r and alpha C for its head backward.
#include "kernels.cuh"
#include "umma.cuh"

namespace scgib {
using namespace umma;

namespace htc {
constexpr int TM = 128;
constexpr int kEpiWarps = 8, kMmaWarp = kEpiWarps, kProdWarps = 8, PT = kProdWarps * 32;
constexpr int kThreadsH = (kEpiWarps + 1 + kProdWarps) * 32;
constexpr int kABlk = TM * 128;                 // one [128 rows][64 fp16] format-B block
constexpr int kStage = 4 * kABlk;               // hi: noisy block, alpha-C block | lo: the same two
constexpr int kW1Blk = HID * 128;               // one [64 out rows][64 fp16 K columns] block
constexpr float kWScale = 16.f;
constexpr uint32_t kId = (1u << 4) | ((uint32_t)(HID >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);   // kind::f16, fp16 x fp16, M 128, N 64, K-major A and B
constexpr uint32_t kId2 = (1u << 4) | ((uint32_t)(2 * HID >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);   // N 128
// TMEM columns of stage s (base 192 s): D (128: hh | hl' + l'h; D1, later overwritten by D2) | r hi (32) | r lo' (32)
constexpr int kColD1 = 0, kColD2 = 0, kColR = 128, kStageCols = 192;
constexpr float kLoScale = 1.f / 2048.f;

struct Smem {
  static constexpr int off_a = 0;                                 // 2 stages
  static constexpr int off_w1 = 2 * kStage;                       // per K block: hi | lo'  (rows 0..63 | 64..127 of one N = 128 operand)
  static constexpr int off_w2 = off_w1 + 4 * kW1Blk;              // hi | lo'
  static constexpr int off_f = off_w2 + 2 * kW1Blk;               // b1[64] b2[64]
  static constexpr int off_bar = off_f + 2 * HID * 4;             // 12 mbarriers + tmem slot
  static constexpr int total = off_bar + 128;
  static_assert(total <= 227 * 1024, "shared memory budget");
};
enum { B_FULL = 0, B_EMPTY = 2, B_D1 = 4, B_R = 6, B_D2 = 8, B_E2 = 10, B_COUNT = 12 };

__device__ __forceinline__ void mma_h(uint32_t d, uint64_t a, uint64_t b, uint32_t id, bool acc) { if (elect_one()) mma_bf16(d, a, b, id, acc); }
__device__ __forceinline__ void mma_h_ta(uint32_t d, uint32_t a_tmem, uint64_t b, uint32_t id, bool acc) { if (elect_one()) mma_bf16_ta(d, a_tmem, b, id, acc); }
__device__ __forceinline__ void tmem_st16u(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
      :: "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
         "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]) : "memory");
}
__device__ __forceinline__ float clamp16(float v) { return fminf(fmaxf(v, -65504.f), 65504.f); }

// natural fp32 weights [OUT = 64 rows][IN cols] (scaled by kWScale) -> fp16 K-major B operand: per block of 64 K columns the
// hi tile [64][64] followed by the lo' tile (rows 64..127 of the block's N = 128 operand)
template <int IN>
__device__ __forceinline__ void stage_weight16(unsigned char* dst, const float* __restrict__ W, int tid, int nthreads) {
  for (int i = tid; i < HID * (IN / 8); i += nthreads) {
    const int o = i / (IN / 8), c8 = i % (IN / 8);
    const float4 v0 = ldg4(W + (size_t)o * IN + c8 * 8), v1 = ldg4(W + (size_t)o * IN + c8 * 8 + 4);
    const float v[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) split_f16x2_s11(v[2 * q] * kWScale, v[2 * q + 1] * kWScale, hi[q], lo[q]);
    const int off = (c8 >> 3) * 2 * kW1Blk + tile_b_off(o, c8 & 7);
    *reinterpret_cast<uint4*>(dst + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(dst + off + kW1Blk) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}

// GATE = true: the compressor's first layer on the same pipeline (one GEMM): H = relu(BN(y)) is formed by the producers (and
// stored), q = H Wc1^T + bc1 by epilogue 1; arguments: noisy = y, bn = {mean, rstd, gamma, beta}, W1n = Wc1 [64][64], b1 = bc1,
// r = H (out), Z = q (out).
template <bool GATE>
__global__ void __launch_bounds__(kThreadsH, 1)
head_fwd_tc_kernel(HeadFwdArgs p) {
  using L = Smem;
  extern __shared__ __align__(1024) unsigned char smem[];
  float* s_b1 = reinterpret_cast<float*>(smem + L::off_f);
  float* s_b2 = s_b1 + HID;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::off_bar);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + L::off_bar + B_COUNT * 8);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = (p.N + TM - 1) / TM;
  const int bid = (int)blockIdx.x, nblk = (int)gridDim.x;
  const int my_tiles = (n_tiles - bid + nblk - 1) / nblk;       // tiles bid + i * nblk
  auto tile_base = [&](int i) { return (bid + i * nblk) * TM; };

  if (threadIdx.x == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(&bars[B_FULL + s], kProdWarps);
      mbar_init(&bars[B_EMPTY + s], 1);
      mbar_init(&bars[B_D1 + s], 1);
      mbar_init(&bars[B_R + s], kEpiWarps);
      mbar_init(&bars[B_D2 + s], 1);
      mbar_init(&bars[B_E2 + s], kEpiWarps);
    }
  }
  if (warp == kMmaWarp) tmem_alloc(s_tmem, 512);
  // parameters only (they precede the programmatic-dependency wait: the weights are never written inside a step's forward)
  if (GATE) stage_weight16<HID>(smem + L::off_w1, p.W1n, threadIdx.x, kThreadsH);
  else {
    stage_weight16<2 * HID>(smem + L::off_w1, p.W1n, threadIdx.x, kThreadsH);
    stage_weight16<HID>(smem + L::off_w2, p.W2n, threadIdx.x, kThreadsH);
  }
  if (threadIdx.x < HID) { s_b1[threadIdx.x] = p.b1[threadIdx.x]; s_b2[threadIdx.x] = GATE ? 0.f : p.b2[threadIdx.x]; }
  pdl_sync();
  fence_smem_to_async();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *s_tmem;
  float S = 1.f;                                              // input pre-scale (header): 1 unless the inputs exceed 2^5
  if (!GATE && p.xmax) {
    const float bound = fmaxf(__uint_as_float(__ldcg(p.xmax)), __uint_as_float(__ldcg(p.xmax + 1)) * __uint_as_float(__ldcg(p.xmax + 2)));
    if (bound >= 32.f && bound <= 3.0e38f) {
      int e;
      (void)frexpf(bound, &e);                                // bound = m 2^e, m in [0.5, 1): S bound in [2^4, 2^5)
      S = exp2f((float)(5 - e));
    }
  }
  const float kInvS = (1.f / kWScale) / S;                    // exact: powers of two

  if (warp > kMmaWarp) {
    // =========================================================================== producers: [noisy || alpha C] -> fp16 hi / lo tiles
    const int pt = (warp - (kMmaWarp + 1)) * 32 + lane;
    if (GATE) {
      const int c8 = pt & 7, r0 = pt >> 3;                      // 8-channel chunk of the 64, first row (rows r0 + 32 j)
      const int c = c8 * 8;
      float mu[8], sc[8], be[8];                                // relu(BN(y)) = max((y - mean) * (rstd * gamma) + beta, 0)
#pragma unroll
      for (int q = 0; q < 8; ++q) { mu[q] = p.bn[c + q]; sc[q] = p.bn[HID + c + q] * p.bn[2 * HID + c + q]; be[q] = p.bn[3 * HID + c + q]; }
      for (int i = 0; i < my_tiles; ++i) {
        const int s = i & 1, use = i >> 1;
        const int base = tile_base(i);
        if (use > 0) mbar_wait(&bars[B_EMPTY + s], (uint32_t)((use - 1) & 1));
        unsigned char* ahi = smem + L::off_a + s * kStage;
        unsigned char* alo = ahi + 2 * kABlk;
        float v[4][8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int gv = base + r0 + 32 * j;
          if (gv < p.N) {
            if (p.in_bf16) {                                    // bf16 mode: y is bf16 storage
              const uint4 w = *reinterpret_cast<const uint4*>(reinterpret_cast<const bf16_t*>(p.noisy) + (size_t)gv * HID + c);
              v[j][0] = bf16_lo(w.x); v[j][1] = bf16_hi(w.x); v[j][2] = bf16_lo(w.y); v[j][3] = bf16_hi(w.y);
              v[j][4] = bf16_lo(w.z); v[j][5] = bf16_hi(w.z); v[j][6] = bf16_lo(w.w); v[j][7] = bf16_hi(w.w);
            } else {
              ld8(p.noisy + (size_t)gv * HID + c, v[j]);
            }
          } else {
#pragma unroll
            for (int q = 0; q < 8; ++q) v[j][q] = 0.f;
          }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int r = r0 + 32 * j, gv = base + r;
          if (gv < p.N) {
#pragma unroll
            for (int q = 0; q < 8; ++q) v[j][q] = fmaxf(fmaf(v[j][q] - mu[q], sc[q], be[q]), 0.f);
            st8(p.r + (size_t)gv * HID + c, v[j]);
          }
          uint32_t hi[4], lo[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) split_f16x2_s11(fminf(v[j][2 * q], 65504.f), fminf(v[j][2 * q + 1], 65504.f), hi[q], lo[q]);
          const int off = tile_b_off(r, c8);
          *reinterpret_cast<uint4*>(ahi + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
          *reinterpret_cast<uint4*>(alo + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        }
        fence_smem_to_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars[B_FULL + s]);
      }
    } else {
    const int ch = pt & 15, r0 = pt >> 4;                       // this thread's 8-channel chunk of the 128 and its first row
    const bool second = ch >= 8;                                // alpha C half
    const int c8 = ch & 7;
    for (int i = 0; i < my_tiles; ++i) {
      const int s = i & 1, use = i >> 1;
      const int base = tile_base(i);
      if (use > 0) mbar_wait(&bars[B_EMPTY + s], (uint32_t)((use - 1) & 1));   // GEMM1 of the stage's previous tile has read it
      unsigned char* ahi = smem + L::off_a + s * kStage + (second ? kABlk : 0);
      unsigned char* alo = ahi + 2 * kABlk;
#pragma unroll
      for (int bt = 0; bt < 2; ++bt) {
        float v[4][8];
        float al[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int r = r0 + 16 * (4 * bt + j), gv = base + r;
          al[j] = 1.f;
          if (gv < p.N) {
            ld8((second ? p.C : p.noisy) + (size_t)gv * HID + c8 * 8, v[j]);
            if (second) al[j] = __ldg(p.alpha + gv);
          } else {
#pragma unroll
            for (int q = 0; q < 8; ++q) v[j][q] = 0.f;
          }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int r = r0 + 16 * (4 * bt + j), gv = base + r;
#pragma unroll
          for (int q = 0; q < 8; ++q) v[j][q] *= al[j];
          if (gv < p.N) {
            if (second && p.aC) st8(p.aC + (size_t)gv * HID + c8 * 8, v[j]);
            if (second && p.aC_bf)       // bf16 mode: the head backward's operand copy
              *reinterpret_cast<uint4*>(p.aC_bf + (size_t)gv * HID + c8 * 8) =
                  make_uint4(pack_bf16x2(v[j][0], v[j][1]), pack_bf16x2(v[j][2], v[j][3]), pack_bf16x2(v[j][4], v[j][5]), pack_bf16x2(v[j][6], v[j][7]));
            if (p.imap) st8(p.imap + (size_t)gv * 2 * HID + ch * 8, v[j]);
          }
          uint32_t hi[4], lo[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) split_f16x2_s11(clamp16(v[j][2 * q] * S), clamp16(v[j][2 * q + 1] * S), hi[q], lo[q]);
          const int off = tile_b_off(r, c8);
          *reinterpret_cast<uint4*>(ahi + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
          *reinterpret_cast<uint4*>(alo + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        }
      }
      fence_smem_to_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars[B_FULL + s]);
    }
    }
  } else if (warp == kMmaWarp) {
    // =========================================================================== MMA issuer (converged warp, elected lane)
    const uint32_t w1 = smem_u32(smem + L::off_w1), w2 = smem_u32(smem + L::off_w2);
    auto gemm1 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      mbar_wait(&bars[B_FULL + s], (uint32_t)(use & 1));
      if (use > 0) mbar_wait(&bars[B_E2 + s], (uint32_t)((use - 1) & 1));     // the epilogue has read the stage's previous D2
      fence_after_sync();
      const uint32_t ah = smem_u32(smem + L::off_a + s * kStage), al = ah + 2 * kABlk;
      const uint32_t d = tmem + s * kStageCols + kColD1;
#pragma unroll
      for (int k = 0; k < (GATE ? HID : 2 * HID) / 16; ++k) {
        const uint32_t kb = (uint32_t)(k >> 2);
        const uint64_t db = desc_b_kmajor(w1 + kb * 2 * kW1Blk, k & 3);        // hi tile; the N = 128 view continues into the lo' tile
        mma_h(d, desc_b_kmajor(ah + kb * kABlk, k & 3), db, kId2, k > 0);
        mma_h(d + HID, desc_b_kmajor(al + kb * kABlk, k & 3), db, kId, true);
      }
      mma_commit_w(&bars[B_D1 + s]);
      mma_commit_w(&bars[B_EMPTY + s]);
    };
    auto gemm2 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      mbar_wait(&bars[B_R + s], (uint32_t)(use & 1));
      fence_after_sync();
      const uint32_t d = tmem + s * kStageCols + kColD2;
      const uint32_t rh = tmem + s * kStageCols + kColR, rl = rh + 32;
#pragma unroll
      for (int k = 0; k < HID / 16; ++k) {
        const uint64_t db = desc_b_kmajor(w2, k);
        mma_h_ta(d, rh + 8 * k, db, kId2, k > 0);
        mma_h_ta(d + HID, rl + 8 * k, db, kId, true);
      }
      mma_commit_w(&bars[B_D2 + s]);
    };
    if (my_tiles > 0) gemm1(0);
    for (int i = 0; i < my_tiles; ++i) {
      if (i + 1 < my_tiles) gemm1(i + 1);
      if (!GATE) gemm2(i);
    }
  } else {
    // =========================================================================== epilogue
    // warp w: TMEM lane quarter w & 3 (rows 32 (w & 3) ..), column half w >> 2 (columns 32 (w >> 2) ..)
    const int q = warp & 3, half = warp >> 2;
    const int row = q * 32 + lane;
    const int c0 = half * 32;
    const uint32_t tl = (uint32_t)(q * 32) << 16;
    auto epi1 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      const int gv = tile_base(i) + row;
      mbar_wait(&bars[B_D1 + s], (uint32_t)(use & 1));
      fence_after_sync();
      const uint32_t t0 = tmem + s * kStageCols + tl;
      float v[32], v2[32];
      tmem_ld16_nowait(t0 + kColD1 + c0, *reinterpret_cast<float (*)[16]>(v));
      tmem_ld16_nowait(t0 + kColD1 + c0 + 16, *reinterpret_cast<float (*)[16]>(v + 16));
      tmem_ld16_nowait(t0 + kColD1 + HID + c0, *reinterpret_cast<float (*)[16]>(v2));
      tmem_ld16_nowait(t0 + kColD1 + HID + c0 + 16, *reinterpret_cast<float (*)[16]>(v2 + 16));
      tmem_ld_wait();
      if (GATE) {                                               // q = H Wc1^T + bc1: no activation, nothing goes back to the tensor pipe
        fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars[B_E2 + s]);           // the stage's TMEM columns may be overwritten by its next tile
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = fmaf(fmaf(v2[j], kLoScale, v[j]), kInvS, s_b1[c0 + j]);
        if (gv < p.N) {
#pragma unroll
          for (int j = 0; j < 4; ++j) st8(p.Z + (size_t)gv * HID + c0 + 8 * j, v + 8 * j);
        }
        return;
      }
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = fmaxf(fmaf(fmaf(v2[j], kLoScale, v[j]), kInvS, s_b1[c0 + j]), 0.f);
      uint32_t hi[16], lo[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) split_f16x2_s11(fminf(v[2 * j] * S, 65504.f), fminf(v[2 * j + 1] * S, 65504.f), hi[j], lo[j]);
      tmem_st16u(t0 + kColR + c0 / 2, hi);
      tmem_st16u(t0 + kColR + 32 + c0 / 2, lo);
      if (p.r && gv < p.N) {
#pragma unroll
        for (int j = 0; j < 4; ++j) st8(p.r + (size_t)gv * HID + c0 + 8 * j, v + 8 * j);
      }
      if (p.r_bf && gv < p.N) {      // bf16 mode: the head backward's operand copy
#pragma unroll
        for (int j = 0; j < 4; ++j)
          *reinterpret_cast<uint4*>(p.r_bf + (size_t)gv * HID + c0 + 8 * j) =
              make_uint4(pack_bf16x2(v[8 * j], v[8 * j + 1]), pack_bf16x2(v[8 * j + 2], v[8 * j + 3]), pack_bf16x2(v[8 * j + 4], v[8 * j + 5]),
                         pack_bf16x2(v[8 * j + 6], v[8 * j + 7]));
      }
      tmem_st_wait();
      fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars[B_R + s]);
    };
    auto epi2 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      const int gv = tile_base(i) + row;
      mbar_wait(&bars[B_D2 + s], (uint32_t)(use & 1));
      fence_after_sync();
      const uint32_t t0 = tmem + s * kStageCols + tl;
      float y[32], y2[32];
      tmem_ld16_nowait(t0 + kColD2 + c0, *reinterpret_cast<float (*)[16]>(y));
      tmem_ld16_nowait(t0 + kColD2 + c0 + 16, *reinterpret_cast<float (*)[16]>(y + 16));
      tmem_ld16_nowait(t0 + kColD2 + HID + c0, *reinterpret_cast<float (*)[16]>(y2));
      tmem_ld16_nowait(t0 + kColD2 + HID + c0 + 16, *reinterpret_cast<float (*)[16]>(y2 + 16));
      tmem_ld_wait();
      fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars[B_E2 + s]);           // the stage's TMEM columns may be overwritten by its next tile
#pragma unroll
      for (int j = 0; j < 32; ++j) y[j] = fmaf(fmaf(y2[j], kLoScale, y[j]), kInvS, s_b2[c0 + j]);
      if (gv < p.N) {
#pragma unroll
        for (int j = 0; j < 4; ++j) st8(p.Z + (size_t)gv * HID + c0 + 8 * j, y + 8 * j);
      }
    };
    if (my_tiles > 0) epi1(0);
    for (int i = 0; i < my_tiles; ++i) {
      if (i + 1 < my_tiles) epi1(i + 1);
      if (!GATE) epi2(i);
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc(tmem, 512);
}
}  // namespace htc

void launch_head_fwd_tc(const HeadFwdArgs& a, cudaStream_t s) {
  static bool once = (cudaFuncSetAttribute(htc::head_fwd_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, htc::Smem::total), true);
  (void)once;
  const int grid = max(1, min((a.N + htc::TM - 1) / htc::TM, num_sms()));
  launch_k((htc::head_fwd_tc_kernel<false>), dim3(grid), dim3(htc::kThreadsH), htc::Smem::total, s, a);
}

// H = relu(BN(y)); q = H Wc1^T + bc1 on the same pipeline (hidden 64, fp32 y)
void launch_gate_lin_fwd_tc(const GateLinFwdArgs& g, const float* Wc1, cudaStream_t s) {
  static bool once = (cudaFuncSetAttribute(htc::head_fwd_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, htc::Smem::total), true);
  (void)once;
  HeadFwdArgs a{};
  a.noisy = g.y; a.bn = g.bn; a.N = g.N; a.W1n = Wc1; a.b1 = g.bc1; a.r = g.H; a.Z = g.q; a.in_bf16 = g.y_bf16;
  const int grid = max(1, min((a.N + htc::TM - 1) / htc::TM, num_sms()));
  launch_k((htc::head_fwd_tc_kernel<true>), dim3(grid), dim3(htc::kThreadsH), htc::Smem::total, s, a);
}

}  // namespace scgib
