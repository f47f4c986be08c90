// gin_bwd_h.cu - GIN layer backward (part 2) on tcgen05 with TWO-TERM FP16 operand splits: 128-row tiles, K = 16 MMAs.
//
// Reference: autograd of models.py:66-72.  Runs every fp32 GIN layer at hidden 64 (the 32-wide layer 0 runs zero-padded to
// 64 input channels), the head MLP and, in half mode, the compressor's first linear layer:
//   g_y = rstd * (gamma*g_o - c1 - yhat*c2);  G1: g_r = g_y W2;  G3: dW2 += g_y^T r;  g_u = g_r * [r > 0];
//   G2: g_a = g_u W1;  G4: dW1 += g_u^T a;  db2 += sum g_y;  db1 += sum g_u.
// Every operand is a two-term fp16 split (22 significand bits, the precision of 3xTF32 products at twice the K per MMA):
//   * forward activations r, a and the weights (x 2^4): v = hi + lo, lo = fp16(v - hi) UNSCALED (|v| = O(1): absolute error
//     <= 2^-25), so their hi and lo products accumulate into the SAME columns.  Where a and r are not O(1) (the head MLP
//     operator: GraphSAGE / GCN features are unbounded) the caller leaves max |a| and max |r| in device slots, and a, r are
//     first normalised by powers of two Sa, Sr as the gradients below; dW1 / dW2 undo them where they leave tensor memory;
//   * gradients g_y, g_u: first normalised by a power of two S (max |g| of the launch -> ~2^8: the producing kernel leaves
//     max |g_o| in a device slot by an order-independent atomicMax, the BN-backward factors are known here), then
//     v = hi + 2^-11 lo' with the residual SCALED into fp16's normal range: small gradient entries keep their relative
//     precision; the lo' products land in separate accumulator columns / TMEM lanes and are folded in with 2^-11 by the epilogues.
// A 128-row tile needs 12 + 16 + 12 + 16 = 56 kind::f16 MMAs (K = 16), two 128-row stages of fp16 tiles fit in shared
// memory, and UMMA M = 128 uses all 128 TMEM lanes (8 epilogue warps: lane quarter x 32-column half).  All scalings are exact
// powers of two, undone exactly.  Roles: 8 epilogue warps, 1 MMA warp, 16 loader warps (the role timeline showed the loaders'
// dependent 32-byte row loads as the serial bottleneck of a tile: 6 us with 8 warps); hand-offs are mbarriers with one arrival
// per warp.
#include <stdlib.h>
#include "kernels.cuh"
#include "umma.cuh"

namespace scgib {
using namespace umma;

// per-tile role timestamps (SCGIB_DBG bit 2048; experiments only, tests/gpu_tc2_trace.py bwdh); tiles >= 16 are not recorded
__device__ long long g_bwdh_trace[160 * 16 * 12];
#define BWDH_TRACE(ev, tile) do { if (trace_on && (tile) < 16 && blockIdx.x < 160) g_bwdh_trace[((size_t)blockIdx.x * 16 + (tile)) * 12 + (ev)] = clock64(); } while (0)

namespace bwdh {
constexpr int TM = 128;
constexpr int kEpiWarps = 8, kLoadWarps = 16;
constexpr int kMmaWarp = kEpiWarps;
constexpr int kThreadsB = (kEpiWarps + 1 + kLoadWarps) * 32;
constexpr int LT = kLoadWarps * 32;                 // loader threads
constexpr int kTile = TM * 128;                     // one [128 rows][64 fp16] format-B tile (16 KB)
constexpr int kStage = 4 * kTile;                   // X hi | X lo' | Y hi | Y lo
constexpr int kWTile = HID * 128;                   // one [64][64 fp16] weight tile
constexpr float kWScale = 16.f, kLo = 1.f / 2048.f;
// TMEM columns: D1[2] (g_r: [hh + hl | l'h], 128 each) | D2 (g_a, 128) | D3 (dW2, 64: TMEM lanes 0..63 hi rows, 64..127 lo' rows) | D4 (dW1, 64)
constexpr int kColD1 = 0, kColD2 = 256, kColD3 = 384, kColD4 = 448;
enum { B_FULL1 = 0, B_FULL2 = 2, B_GU = 4, B_D1 = 6, B_D2 = 8, B_E2 = 10, B_COUNT = 11 };

__host__ __device__ constexpr uint32_t idh(int M, int N, bool a_mn, bool b_mn) {     // kind::f16, fp16 A / B, fp32 accumulate
  return (1u << 4) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
constexpr uint32_t kIdRow = idh(TM, HID, false, false);      // G1 / G2: A = X K-major, B = transposed weight tile K-major
constexpr uint32_t kIdCol = idh(128, HID, true, true);       // G3 / G4: A = [g_hi | g_lo']^T (M-stacked, MN-major), B = Y MN-major

struct Smem {
  static constexpr int off_stage = 0;
  static constexpr int off_w2 = 2 * kStage;                         // W2t hi | lo   ([in][out])
  static constexpr int off_w1 = off_w2 + 2 * kWTile;                // W1t hi | lo   ([kin][out])
  static constexpr int off_mask = off_w1 + 2 * kWTile;              // uint2 [2][TM]: r > 0 bits
  static constexpr int off_k = off_mask + 2 * TM * 8;               // float ka kd ke mean [HID]
  static constexpr int off_db1 = off_k + 4 * HID * 4;               // float [TM][HID + 1]: per-row (TMEM lane) sums of S * g_u
  static constexpr int off_db2 = off_db1 + TM * (HID + 1) * 4;      // float [LT / 8][HID]: per-loader-row-group sums of g_y
  static constexpr int off_bar = off_db2 + (LT / 8) * HID * 4;
  static constexpr int total = off_bar + 128;
  static_assert(total <= 227 * 1024, "shared memory budget");
};

__device__ __forceinline__ void mma_h(uint32_t d, uint64_t a, uint64_t b, uint32_t id, bool acc) { if (elect_one()) mma_bf16(d, a, b, id, acc); }
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" :: "l"(p)); }
__device__ __forceinline__ void ld8cs(const float* p, float* v) {
  asm volatile("ld.global.cs.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]),
               "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]) : "l"(p));
}
__device__ __forceinline__ float clamp16(float v) { return fminf(fmaxf(v, -65504.f), 65504.f); }
// the power of two 2^(8 - e) for bound = m * 2^e (m in [0.5, 1)): it takes the bound into [2^7, 2^8); 1 for a bound of 0 or inf
__device__ __forceinline__ float pow2_norm(float bound) {
  if (!(bound > 0.f && bound < 3.0e38f)) return 1.f;
  int e;
  (void)frexpf(bound, &e);
  return exp2f((float)max(-100, min(100, 8 - e)));
}
__device__ __forceinline__ float slot_norm(const unsigned int* slot) { return slot ? pow2_norm(__uint_as_float(__ldcg(slot))) : 1.f; }

// transposed weight tile for the input-gradient GEMMs: B[n = input channel][k = output channel] = 16 W[out][in], fp16 hi / lo
// (`in` < 64 input channels: the missing rows of the tile are zero)
__device__ __forceinline__ void stage_wt(unsigned char* hi_t, unsigned char* lo_t, const float* __restrict__ W, int in, int tid, int nthreads) {
  for (int i = tid; i < HID * 8; i += nthreads) {
    const int n = i & (HID - 1), c8 = i >> 6;                    // consecutive threads: consecutive input channels (coalesced)
    float v[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) v[q] = n < in ? __ldg(W + (size_t)(c8 * 8 + q) * in + n) * kWScale : 0.f;
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) split_f16x2_plain(v[2 * q], v[2 * q + 1], hi[q], lo[q]);
    const int off = tile_b_off(n, c8);
    *reinterpret_cast<uint4*>(hi_t + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(lo_t + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}

template <bool HALF>
__global__ void __launch_bounds__(kThreadsB, 1)
gin_bwd_h_kernel(GinBwdMainPair pp) {
  using L = Smem;
  constexpr int KIN = HID;                                    // tile width of a / g_a / W1t: narrower layers (kin = 32) are zero-padded
  const int kin = pp.kin;
  // half mode (one linear layer, the compressor's first: gH += g_q Wc1, dWc1 = g_q^T H, dbc1 = sum g_q): only G1 / G3 run,
  // epilogue 1 adds g_r to the rows of g_a (in / out) instead of masking and re-splitting it; identity BN constants; r = H
  constexpr bool half_mode = HALF;
  const bool second = (int)blockIdx.x >= pp.split;
  const GinBwdMainArgs& p = pp.a[second ? 1 : 0];
  const int bid = second ? (int)blockIdx.x - pp.split : (int)blockIdx.x;          // CTA index / count inside its problem
  const int nblk = second ? (int)gridDim.x - pp.split : pp.split;
  extern __shared__ __align__(1024) unsigned char smem[];
  uint2* s_mask = reinterpret_cast<uint2*>(smem + L::off_mask);
  float* s_k = reinterpret_cast<float*>(smem + L::off_k);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::off_bar);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + L::off_bar + B_COUNT * 8);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = (p.V + TM - 1) / TM;
  const int my_tiles = max(0, (n_tiles - bid + nblk - 1) / nblk);
  // descending row order: gin_bwd_pre (the previous launch) walks ascending, so the rows it touched last (g_o just written,
  // y just read) are still in L2 when this kernel starts, and the g_a rows written last here (the lowest) are the ones the
  // next layer's gin_bwd_pre gathers first
  const bool rev = pp.reverse != 0;
  const bool trace_on = pp.trace != 0;
  auto tile_base = [&](int i) { return (bid + (rev ? my_tiles - 1 - i : i) * nblk) * TM; };
  auto Xs = [&](int s) { return smem + L::off_stage + s * kStage; };
  auto Ys = [&](int s) { return smem + L::off_stage + s * kStage + 2 * kTile; };

  if (threadIdx.x == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(&bars[B_FULL1 + s], kLoadWarps);
      mbar_init(&bars[B_FULL2 + s], kLoadWarps);
      mbar_init(&bars[B_GU + s], kEpiWarps);
      mbar_init(&bars[B_D1 + s], 1);
      mbar_init(&bars[B_D2 + s], 1);
    }
    mbar_init(&bars[B_E2], kEpiWarps);
  }
  if (warp == kMmaWarp) tmem_alloc(s_tmem, 512);
  if (pp.wait_first) pdl_sync();
  stage_wt(smem + L::off_w2, smem + L::off_w2 + kWTile, p.W2, HID, threadIdx.x, kThreadsB);
  if (!half_mode) stage_wt(smem + L::off_w1, smem + L::off_w1 + kWTile, p.W1, kin, threadIdx.x, kThreadsB);
  if (!pp.wait_first) pdl_sync();   // the weights above are parameters; bn / cvec / g_o / y / r / a / gmax below come from the previous kernels
  // BN-backward constants: g_y = ka*g_o - kd*y + (kd*mean - ke)      (ka = rstd*gamma, kd = rstd^2*c2, ke = rstd*c1)
  if (threadIdx.x < HID) {
    const int c = threadIdx.x;
    const float mean = p.bn[c], rstd = p.bn[HID + c], gamma = p.bn[2 * HID + c];
    const float kd = rstd * rstd * p.cvec[HID + c];
    s_k[c] = rstd * gamma; s_k[HID + c] = kd; s_k[2 * HID + c] = fmaf(kd, mean, -rstd * p.cvec[c]); s_k[3 * HID + c] = mean;   // ka, kd, kd*mean - ke
  }
  fence_smem_to_async();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *s_tmem;
  // gradient normalisation: S = 2^e with S * max|g_o| * max|ka| in [2^7, 2^8): the other BN-backward terms are of the same order
  // and g_u = g_r * mask sums 64 weighted terms, so fp16's 2^16 keeps 2^8 of headroom (values are clamped to the fp16 range
  // before conversion), while entries down to 2^-22 of the largest one keep the full 22-bit two-term precision.  Sa, Sr: the
  // same rule for a and r (1 without a slot); g_a, db1, db2 and the r > 0 mask do not depend on them.
  float kamax = 0.f;
  for (int c = 0; c < HID; ++c) kamax = fmaxf(kamax, fabsf(s_k[c]));
  const float S = pow2_norm((p.gmax ? __uint_as_float(__ldcg(p.gmax)) : 0.f) * kamax);
  const float Sa = slot_norm(p.amax), Sr = slot_norm(p.rmax);
  const float invS = 1.f / S;

  float* s_db1 = reinterpret_cast<float*>(smem + L::off_db1);
  float* s_db2 = reinterpret_cast<float*>(smem + L::off_db2);

  if (warp > kMmaWarp) {
    // =========================================================================== loaders
    const int pt = (warp - (kMmaWarp + 1)) * 32 + lane;
    constexpr int RPP = LT / 8, UPT = TM / RPP;                 // rows per pass, (row, chunk) units per thread
    const int c8 = pt & 7, r0 = pt >> 3;                        // this thread's 8-channel chunk and first row (rows r0 + RPP u)
    const int c = c8 * 8;
    float db2[8];                    // column sums of g_y for channels 8*c8 .. 8*c8+7 over this thread's rows
#pragma unroll
    for (int q = 0; q < 8; ++q) db2[q] = 0.f;
    // phase 1 of tile i: g_o, y, r rows -> S * g_y (hi / lo'), r (hi / lo), r > 0 bits -> X, Y, mask of stage i & 1
    auto phase1 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      const int base = tile_base(i);
      unsigned char* X = Xs(s);
      unsigned char* Y = Ys(s);
      if (pt == 0) BWDH_TRACE(0, i);
      if (i + 1 < my_tiles) {                                   // next tile -> L2: 256 lines of 128 B per [128][64] fp32 tensor
        const size_t off = (size_t)tile_base(i + 1) * HID + (size_t)(pt & 255) * 32;
        if (pt < 256 && off < (size_t)p.V * HID) {
          prefetch_l2(p.g_o + off); prefetch_l2(p.y + off); prefetch_l2(p.r + off);
          const size_t aoff = (size_t)tile_base(i + 1) * kin + (size_t)(pt & 255) * 32;
          if ((pt & 255) * 32 < TM * kin && aoff < (size_t)p.V * kin) prefetch_l2(p.a + aoff);
        }
      }
      bool waited = use == 0;
#pragma unroll
      for (int u = 0; u < UPT; ++u) {                           // one (row, 8-channel chunk) unit at a time: three 32-byte loads in flight
        // (measured: issuing both units' loads before the wait costs registers / spills and is slower, 110 vs 99 us per launch)
        const int row = r0 + RPP * u;
        const bool ok = base + row < p.V;
        float go[1][8], yy[1][8], rr[1][8];
        if (ok) {
          const size_t o = (size_t)(base + row) * HID + c;
          ld8(p.g_o + o, go[0]); ld8cs(p.y + o, yy[0]); ld8cs(p.r + o, rr[0]);
        } else {
#pragma unroll
          for (int q = 0; q < 8; ++q) { go[0][q] = 0.f; yy[0][q] = 0.f; rr[0][q] = 0.f; }
        }
        if (!waited) {                                          // the stage's previous tile: G2 / G4 (half mode: G1 / G3) are done
          mbar_wait(&bars[(half_mode ? B_D1 : B_D2) + s], (uint32_t)((use - 1) & 1)); waited = true; if (pt == 0) BWDH_TRACE(1, i);
        }
        uint32_t hi[4], lo[4], rh[4], rl[4];
        unsigned bits = 0;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const float4 ka = ld4(s_k + c + 4 * h), kd = ld4(s_k + HID + c + 4 * h), ke = ld4(s_k + 2 * HID + c + 4 * h);
          const float kav[4] = {ka.x, ka.y, ka.z, ka.w}, kdv[4] = {kd.x, kd.y, kd.z, kd.w}, kev[4] = {ke.x, ke.y, ke.z, ke.w};
          float gy[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float g = ok ? fmaf(kav[q], go[0][4 * h + q], fmaf(-kdv[q], yy[0][4 * h + q], kev[q])) : 0.f;   // ke' = kd * mean - ke
            db2[4 * h + q] += g;
            gy[q] = clamp16(g * S);
            bits |= (rr[0][4 * h + q] > 0.f ? 1u : 0u) << (4 * h + q);
          }
          split_f16x2_s11(gy[0], gy[1], hi[2 * h], lo[2 * h]);
          split_f16x2_s11(gy[2], gy[3], hi[2 * h + 1], lo[2 * h + 1]);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) split_f16x2_plain(fminf(rr[0][2 * q] * Sr, 65504.f), fminf(rr[0][2 * q + 1] * Sr, 65504.f), rh[q], rl[q]);
        const int off = tile_b_off(row, c8);
        *reinterpret_cast<uint4*>(X + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4*>(X + kTile + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        *reinterpret_cast<uint4*>(Y + off) = make_uint4(rh[0], rh[1], rh[2], rh[3]);
        *reinterpret_cast<uint4*>(Y + kTile + off) = make_uint4(rl[0], rl[1], rl[2], rl[3]);
        // r > 0 bits of the row: the 8 lanes of a row hold 8 channels each -> one 64-bit word (bit = channel)
        unsigned mlo = c8 < 4 ? bits << (8 * c8) : 0u, mhi = c8 >= 4 ? bits << (8 * (c8 - 4)) : 0u;
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) { mlo |= __shfl_xor_sync(0xffffffffu, mlo, o); mhi |= __shfl_xor_sync(0xffffffffu, mhi, o); }
        if (c8 == 0) s_mask[s * TM + row] = make_uint2(mlo, mhi);
      }
      fence_smem_to_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars[B_FULL1 + s]);
      if (pt == 0) BWDH_TRACE(2, i);
    };
    if (my_tiles > 0) phase1(0);
    for (int i = 0; i < my_tiles; ++i) {
      const int s = i & 1, use = i >> 1;
      const int base = tile_base(i);
      unsigned char* Y = Ys(s);
      // the next tile's g_y / r go into the other stage while the tensor pipe works on this one
      if (i + 1 < my_tiles) phase1(i + 1);
      if (half_mode) continue;
      // ---- phase 2 of tile i: a rows -> (after G1 / G3 have read Y) -> Y
      float aa[UPT][8];                                         // the thread's a rows are in flight during the wait
#pragma unroll
      for (int j = 0; j < UPT; ++j) {
        const int v = base + r0 + RPP * j;
        if (v < p.V && c < kin) ld8cs(p.a + (size_t)v * kin + c, aa[j]);
        else {
#pragma unroll
          for (int q = 0; q < 8; ++q) aa[j][q] = 0.f;
        }
      }
      mbar_wait(&bars[B_D1 + s], (uint32_t)(use & 1));
      if (pt == 0) BWDH_TRACE(3, i);
#pragma unroll
      for (int j = 0; j < UPT; ++j) {
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) split_f16x2_plain(clamp16(aa[j][2 * q] * Sa), clamp16(aa[j][2 * q + 1] * Sa), hi[q], lo[q]);
        const int off = tile_b_off(r0 + RPP * j, c8);
        *reinterpret_cast<uint4*>(Y + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4*>(Y + kTile + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
      }
      fence_smem_to_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars[B_FULL2 + s]);
      if (pt == 0) BWDH_TRACE(4, i);
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) s_db2[r0 * HID + c + q] = db2[q];
  } else if (warp == kMmaWarp) {
    // =========================================================================== MMA issuer (converged warp, elected lane)
    const uint32_t w2h = smem_u32(smem + L::off_w2), w2l = w2h + kWTile, w1h = smem_u32(smem + L::off_w1), w1l = w1h + kWTile;
    auto g13 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      const uint32_t xh = smem_u32(Xs(s)), xl = xh + kTile, yh = smem_u32(Ys(s)), yl = yh + kTile;
      mbar_wait(&bars[B_FULL1 + s], (uint32_t)(use & 1));
      if (half_mode && use > 0) mbar_wait(&bars[B_GU + s], (uint32_t)((use - 1) & 1));   // the epilogue has read this D1 buffer's previous tile
      fence_after_sync();
      if (lane == 0) BWDH_TRACE(5, i);
      const uint32_t d1 = tmem + kColD1 + s * 128;
      // G1: S * 16 * g_r = (g_hi + 2^-11 g_lo') (W2t_hi + W2t_lo):  columns [0, 64) hh + hl, columns [64, 128) l'h
#pragma unroll
      for (int k = 0; k < HID / 16; ++k) {
        const uint64_t ah = desc_b_kmajor(xh, k), al = desc_b_kmajor(xl, k), bh = desc_b_kmajor(w2h, k), bl = desc_b_kmajor(w2l, k);
        mma_h(d1, ah, bh, kIdRow, k > 0);
        mma_h(d1, ah, bl, kIdRow, true);
        mma_h(d1 + HID, al, bh, kIdRow, k > 0);
      }
      // G3: S * dW2 += [g_hi | g_lo']^T (r_hi + r_lo)   (X, Y MN-major; hi and lo' tiles of X adjacent = M 128), over all tiles
#pragma unroll
      for (int k = 0; k < TM / 16; ++k) {
        const uint64_t a = desc_b_mnmajor(xh, kTile, k);
        mma_h(tmem + kColD3, a, desc_b_mnmajor(yh, kTile, k), kIdCol, i > 0 || k > 0);
        mma_h(tmem + kColD3, a, desc_b_mnmajor(yl, kTile, k), kIdCol, true);
      }
      mma_commit_w(&bars[B_D1 + s]);
    };
    auto g24 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      const uint32_t xh = smem_u32(Xs(s)), xl = xh + kTile, yh = smem_u32(Ys(s)), yl = yh + kTile;
      mbar_wait(&bars[B_GU + s], (uint32_t)(use & 1));
      mbar_wait(&bars[B_FULL2 + s], (uint32_t)(use & 1));
      if (i > 0) mbar_wait(&bars[B_E2], (uint32_t)((i - 1) & 1));      // epilogue 2 of the previous tile has read D2
      fence_after_sync();
      if (lane == 0) BWDH_TRACE(6, i);
      // G2: S * 16 * g_a = (gu_hi + 2^-11 gu_lo') (W1t_hi + W1t_lo)
#pragma unroll
      for (int k = 0; k < HID / 16; ++k) {
        const uint64_t ah = desc_b_kmajor(xh, k), al = desc_b_kmajor(xl, k), bh = desc_b_kmajor(w1h, k), bl = desc_b_kmajor(w1l, k);
        mma_h(tmem + kColD2, ah, bh, kIdRow, k > 0);
        mma_h(tmem + kColD2, ah, bl, kIdRow, true);
        mma_h(tmem + kColD2 + KIN, al, bh, kIdRow, k > 0);
      }
      // G4: S * dW1 += [gu_hi | gu_lo']^T (a_hi + a_lo)
#pragma unroll
      for (int k = 0; k < TM / 16; ++k) {
        const uint64_t a = desc_b_mnmajor(xh, kTile, k);
        mma_h(tmem + kColD4, a, desc_b_mnmajor(yh, kTile, k), kIdCol, i > 0 || k > 0);
        mma_h(tmem + kColD4, a, desc_b_mnmajor(yl, kTile, k), kIdCol, true);
      }
      mma_commit_w(&bars[B_D2 + s]);
    };
    // G1/G3 of tile i+1 are queued BEFORE G2/G4 of tile i: they run while the epilogue produces g_u of tile i
    if (my_tiles > 0) g13(0);
    for (int i = 0; i < my_tiles; ++i) {
      if (i + 1 < my_tiles) g13(i + 1);
      if (!half_mode) g24(i);
    }
  } else {
    // =========================================================================== epilogue
    // warp w: TMEM lane quarter q = w & 3 (rows 32 q + lane), column half w >> 2 (channels 32 (w >> 2) ..)
    const int q = warp & 3, half = warp >> 2;
    const int row = q * 32 + lane;
    const int c0 = half * 32;
    const uint32_t tl = (uint32_t)(q * 32) << 16;
    float db1[32];                   // S * g_u sums of this thread's row (TMEM lane) for its 32 columns over all tiles
#pragma unroll
    for (int j = 0; j < 32; ++j) db1[j] = 0.f;
    // epilogue 1 of tile i: S * g_u = S * g_r * [r > 0] -> X (hi / lo'), column sums for db1
    auto epi1 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      unsigned char* X = Xs(s);
      mbar_wait(&bars[B_D1 + s], (uint32_t)(use & 1));
      fence_after_sync();
      if (threadIdx.x == 0) BWDH_TRACE(7, i);
      const uint32_t d1 = tmem + tl + kColD1 + s * 128;
      if (half_mode) {                                          // g_a rows (in / out) += g_r; nothing goes back to the tensor pipe
        const int gv = tile_base(i) + row;
        const float k = invS * (1.f / kWScale);
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
          float g[16], t2[16], old[16];
          tmem_ld16_nowait(d1 + c0 + 16 * cc, g);
          tmem_ld16_nowait(d1 + HID + c0 + 16 * cc, t2);
          if (gv < p.V) { ld8(p.g_a + (size_t)gv * HID + c0 + 16 * cc, old); ld8(p.g_a + (size_t)gv * HID + c0 + 16 * cc + 8, old + 8); }
          tmem_ld_wait();
          if (gv < p.V) {
#pragma unroll
            for (int j = 0; j < 16; ++j) old[j] += fmaf(t2[j], kLo, g[j]) * k;
            st8(p.g_a + (size_t)gv * HID + c0 + 16 * cc, old);
            st8(p.g_a + (size_t)gv * HID + c0 + 16 * cc + 8, old + 8);
          }
        }
        fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars[B_GU + s]);
        return;
      }
      const uint2 m = s_mask[s * TM + row];
      const unsigned mbits = half == 0 ? m.x : m.y;
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        float g[16], t2[16];
        tmem_ld16_nowait(d1 + c0 + 16 * cc, g);
        tmem_ld16_nowait(d1 + HID + c0 + 16 * cc, t2);
        tmem_ld_wait();
        uint32_t hi[8], lo[8];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float v = fmaf(t2[j], kLo, g[j]) * (1.f / kWScale);
          g[j] = ((mbits >> (16 * cc + j)) & 1u) ? v : 0.f;
          db1[16 * cc + j] += g[j];
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) split_f16x2_s11(clamp16(g[2 * j]), clamp16(g[2 * j + 1]), hi[j], lo[j]);
        const int o0 = tile_b_off(row, (c0 >> 3) + 2 * cc), o1 = tile_b_off(row, (c0 >> 3) + 2 * cc + 1);
        *reinterpret_cast<uint4*>(X + o0) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4*>(X + o1) = make_uint4(hi[4], hi[5], hi[6], hi[7]);
        *reinterpret_cast<uint4*>(X + kTile + o0) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        *reinterpret_cast<uint4*>(X + kTile + o1) = make_uint4(lo[4], lo[5], lo[6], lo[7]);
      }
      fence_smem_to_async();
      fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars[B_GU + s]);
      if (threadIdx.x == 0) BWDH_TRACE(8, i);
    };
    // epilogue 2 of tile i: g_a -> global
    auto epi2 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      const int gv = tile_base(i) + row;
      mbar_wait(&bars[B_D2 + s], (uint32_t)(use & 1));
      fence_after_sync();
      if (threadIdx.x == 0) BWDH_TRACE(9, i);
      float g[32], t2[32];
      tmem_ld16_nowait(tmem + tl + kColD2 + c0, *reinterpret_cast<float (*)[16]>(g));
      tmem_ld16_nowait(tmem + tl + kColD2 + c0 + 16, *reinterpret_cast<float (*)[16]>(g + 16));
      tmem_ld16_nowait(tmem + tl + kColD2 + KIN + c0, *reinterpret_cast<float (*)[16]>(t2));
      tmem_ld16_nowait(tmem + tl + kColD2 + KIN + c0 + 16, *reinterpret_cast<float (*)[16]>(t2 + 16));
      tmem_ld_wait();
      fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars[B_E2]);                  // D2 may be overwritten by G2 of the next tile
      const float k = invS * (1.f / kWScale);
#pragma unroll
      for (int j = 0; j < 32; ++j) g[j] = fmaf(t2[j], kLo, g[j]) * k;
      if (gv < p.V && c0 < kin) {
#pragma unroll
        for (int j = 0; j < 4; ++j) st8(p.g_a + (size_t)gv * kin + c0 + 8 * j, g + 8 * j);
      }
      if (threadIdx.x == 0) BWDH_TRACE(10, i);
    };
    // g_r of tile i+1 is ready before g_a of tile i (MMA issue order): mask / re-split it first
    if (my_tiles > 0) epi1(0);
    for (int i = 0; i < my_tiles; ++i) {
      if (i + 1 < my_tiles) epi1(i + 1);
      if (!half_mode) epi2(i);
    }
#pragma unroll
    for (int j = 0; j < 32; ++j) s_db1[row * (HID + 1) + c0 + j] = db1[j];
  }
  // ---- every CTA writes its partial gradients (zeros when it had no tile)
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  float* part = p.part + (size_t)blockIdx.x * p.pstride;
  // dW2 / dW1 from tensor memory: accumulator row L (TMEM lane L): L < 64 = hi part of out-channel L, L >= 64 = lo' part of
  // out-channel L - 64 (both summed over B_hi + B_lo).  dW2[o][i] = (row o + 2^-11 row 64 + o) / (S Sr), dW1: / (S Sa).
  float* s_x = reinterpret_cast<float*>(smem);          // [64][HID + 1] exchange buffer (the stages are dead)
  for (int pass = 0; pass < (half_mode ? 1 : 2); ++pass) {   // pass 0: dW2, pass 1: dW1
    const uint32_t col = pass == 0 ? kColD3 : kColD4;
    const int64_t offW = pass == 0 ? p.off_W2 : p.off_W1;
    const float kW = invS * (1.f / (pass == 0 ? Sr : Sa));
    float t[64];
    if (warp < 4) {
      const uint32_t tl = (uint32_t)(warp * 32) << 16;
      const int Lr = warp * 32 + lane;
#pragma unroll
      for (int c16 = 0; c16 < 4; ++c16) {
        float a0[16];
        if (my_tiles > 0) tmem_ld16(tmem + tl + col + c16 * 16, a0);
#pragma unroll
        for (int j = 0; j < 16; ++j) t[c16 * 16 + j] = my_tiles > 0 ? a0[j] : 0.f;
      }
      if (Lr >= 64) {
#pragma unroll
        for (int j = 0; j < 64; ++j) s_x[(Lr - 64) * (HID + 1) + j] = t[j];
      }
    }
    __syncthreads();
    const int C = pass == 0 ? HID : kin;                // columns of the parameter (dW1 of a kin = 32 layer: [64][32])
    if (warp < 2) {
      const int o = warp * 32 + lane;
      for (int j = 0; j < C; j += 4) {
        float4 v;
        v.x = fmaf(s_x[o * (HID + 1) + j], kLo, t[j]) * kW;         v.y = fmaf(s_x[o * (HID + 1) + j + 1], kLo, t[j + 1]) * kW;
        v.z = fmaf(s_x[o * (HID + 1) + j + 2], kLo, t[j + 2]) * kW; v.w = fmaf(s_x[o * (HID + 1) + j + 3], kLo, t[j + 3]) * kW;
        st4(part + offW + (size_t)o * C + j, v);
      }
    }
    __syncthreads();
  }
  // db1: the epilogue threads' per-row sums, column sums in row order (fixed); db2: the loaders' 32 row groups per channel
  if (threadIdx.x < HID) {
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    for (int r = 0; r < TM; r += 4) {
      s0 += s_db1[r * (HID + 1) + threadIdx.x]; s1 += s_db1[(r + 1) * (HID + 1) + threadIdx.x];
      s2 += s_db1[(r + 2) * (HID + 1) + threadIdx.x]; s3 += s_db1[(r + 3) * (HID + 1) + threadIdx.x];
    }
    if (!half_mode) part[p.off_b1 + threadIdx.x] = ((s0 + s1) + (s2 + s3)) * invS;
    float sum = 0.f;
#pragma unroll
    for (int g = 0; g < LT / 8; ++g) sum += s_db2[g * HID + threadIdx.x];
    part[p.off_b2 + threadIdx.x] = sum;
  }
  fence_before_sync();
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc(tmem, 512);
}

}  // namespace bwdh

// the same layer of both encoders (or the two K halves of the head MLP) in one launch: CTAs [0, split) write the partial
// gradients of a0, [split, grid) of a1 (split = pair_split on the 128-row tile counts: the callers' partial-sum reduction
// ranges use the same rule)
void launch_gin_bwd_main_h_pair(const GinBwdMainArgs& a0, const GinBwdMainArgs& a1, int kin, int grid, cudaStream_t s, bool weights_from_prev_kernel) {
  static bool once = (cudaFuncSetAttribute(bwdh::gin_bwd_h_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bwdh::Smem::total), true);
  (void)once;
  GinBwdMainPair pp;
  pp.a[0] = a0; pp.a[1] = a1;
  pp.wait_first = weights_from_prev_kernel ? 1 : 0;
  pp.kin = kin;
  pp.half = 0;
  pp.split = pair_split(grid, (a0.V + 127) / 128, (a1.V + 127) / 128);
  static int tr = -1;
  if (tr < 0) { const char* e = getenv("SCGIB_DBG"); tr = (e && (atoi(e) & 2048)) ? 1 : 0; }
  pp.trace = tr;
  pp.reverse = 1;
  launch_k((bwdh::gin_bwd_h_kernel<false>), dim3(grid), dim3(bwdh::kThreadsB), bwdh::Smem::total, s, pp);
}

void launch_gin_bwd_main_h(const GinBwdMainArgs& a, int kin, int grid, cudaStream_t s) {
  static bool once = (cudaFuncSetAttribute(bwdh::gin_bwd_h_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bwdh::Smem::total), true);
  (void)once;
  GinBwdMainPair pp;
  pp.a[0] = a; pp.a[1] = a;
  pp.split = grid; pp.kin = kin; pp.half = 0; pp.wait_first = 0; pp.trace = 0; pp.reverse = 0;
  launch_k((bwdh::gin_bwd_h_kernel<false>), dim3(grid), dim3(bwdh::kThreadsB), bwdh::Smem::total, s, pp);
}

// one linear layer on the same kernel (half mode): g_in (in / out) += g W;  dW = g^T x;  db = sum g      (gate_lin_bwd on tcgen05)
void launch_linear_bwd_h(const float* g, const float* x, const float* W, int V, float* g_in, const float* bn_identity, const float* cvec_zero,
                         const unsigned int* gmax, float* part, int64_t pstride, int64_t off_W, int64_t off_b, int grid, cudaStream_t s) {
  static bool once = (cudaFuncSetAttribute(bwdh::gin_bwd_h_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bwdh::Smem::total), true);
  (void)once;
  GinBwdMainPair pp;
  GinBwdMainArgs a;
  a.g_o = g; a.y = x; a.r = x; a.a = x; a.bn = bn_identity; a.cvec = cvec_zero; a.W1 = W; a.W2 = W; a.V = V; a.g_a = g_in;
  a.part = part; a.pstride = pstride; a.off_W1 = off_W; a.off_b1 = off_b; a.off_W2 = off_W; a.off_b2 = off_b; a.gmax = gmax;
  pp.a[0] = a; pp.a[1] = a;
  pp.split = grid; pp.kin = HID; pp.half = 1; pp.wait_first = 0; pp.trace = 0; pp.reverse = 0;
  launch_k((bwdh::gin_bwd_h_kernel<true>), dim3(grid), dim3(bwdh::kThreadsB), bwdh::Smem::total, s, pp);
}

}  // namespace scgib
extern "C" __attribute__((visibility("default"))) int scgib_debug_bwdh_trace(long long* host_out, int n) {
  return (int)cudaMemcpyFromSymbol(host_out, scgib::g_bwdh_trace, (size_t)n * sizeof(long long));
}
