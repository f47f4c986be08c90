// gin_bwd_tc2.cu - GIN layer backward (part 2) on tcgen05, second generation: 64-row tiles, DOUBLE-BUFFERED operand tiles.
//
// Same contract and math as gin_bwd_tc.cu / gin_bwd_main_kernel (reference: autograd of models.py:66-72):
//   g_y = rstd * (gamma*g_o - c1 - yhat*c2);  G1: g_r = g_y W2;  G3: dW2 += g_y^T r;  g_u = g_r * [r > 0];
//   G2: g_a = g_u W1;  G4: dW1 += g_u^T a;  db2 += sum g_y;  db1 += sum g_u.
// The role timeline of gin_bwd_tc (tests/gpu_tc2_trace.py bwd) showed a fully serialised 128-row tile: loader store
// 2.0 us -> G1+G3 1.5 us -> epilogue 2.1 us -> G2+G4 1.2 us, because its two 64 KB buffers leave no room for a second
// tile.  Here a tile is 64 rows (X = g_y then g_u, Y = r then a: 2 x 32 KB), so TWO tiles fit: the loaders fill tile
// i+1 while the tensor pipe and the epilogue work on tile i.  Further changes:
//   * the weight-gradient GEMMs take an M-STACKED A operand: the hi and lo copies of g (adjacent tiles) are read as
//     one MN-major A with M = 128 ([g_hi | g_lo]^T); two MMAs per K step (B = r_hi, then r_lo, same 64 accumulator
//     columns) give rows 0..63 = g_hi^T r and rows 64..127 = g_lo^T r: 16 MMAs per tile instead of 32;
//   * the g_r accumulator is double-buffered in tensor memory, so G1/G3 of tile i+1 run while the epilogue masks and
//     re-splits g_u of tile i (tensor pipe and epilogue each need ~1.8 us per tile and now overlap);
//   * 8 epilogue warps (TMEM lane quarter x column half), 8 loader warps, 1 MMA warp: 17 warps, 96 registers, no spills.
// UMMA M = 64 keeps accumulator row i in TMEM lane (i/16)*32 + i%16: an epilogue warp owns 16 rows (lanes 0..15).
#include <stdlib.h>
#include "kernels.cuh"
#include "umma.cuh"

namespace scgib {
using namespace umma;

// per-tile role timestamps (SCGIB_DBG bit 2048; experiments only, tests/gpu_tc2_trace.py bwd); tiles >= 16 are not recorded
__device__ long long g_bwd2_trace[160 * 16 * 12];
#define BWD2_TRACE(ev, tile) do { if (trace_on && (tile) < 16 && blockIdx.x < 160) g_bwd2_trace[((size_t)blockIdx.x * 16 + (tile)) * 12 + (ev)] = clock64(); } while (0)

namespace bwd2 {
constexpr int TM = 64;
constexpr int kEpiWarps = 8, kLoadWarps = 8;
constexpr int kMmaWarp = kEpiWarps;
constexpr int kThreadsB = (kEpiWarps + 1 + kLoadWarps) * 32;
constexpr int LT = kLoadWarps * 32;                 // loader threads
constexpr int kTile = TM * HID * 4;                 // one [64][64] fp32 tile in format S (16 KB)
constexpr int kStage = 4 * kTile;                   // X hi | X lo | Y hi | Y lo
// TMEM columns: D1[2] (g_r, 128 each: hi*hi | hi*lo halves) | D2 (g_a, 2*KIN) | D3 (dW2, 64, M = 128 stacked) | D4 (dW1, KIN)
constexpr int kColD1 = 0, kColD2 = 256, kColD3 = 384, kColD4 = 448;
enum { B_FULL1 = 0, B_FULL2 = 2, B_GU = 4, B_D1 = 6, B_D2 = 8, B_E2 = 10, B_COUNT = 11 };

template <int KIN>
struct Smem {
  static constexpr int W2B = HID * HID * 4, W1B = KIN * HID * 4;     // one hi (or lo) transposed weight tile
  static constexpr int off_stage = 0;
  static constexpr int off_w2 = 2 * kStage;                          // W2t hi | lo   ([in][out], dense cores)
  static constexpr int off_w1 = off_w2 + 2 * W2B;                    // W1t hi | lo   ([kin][out])
  static constexpr int off_mask = off_w1 + 2 * W1B;                  // uint2 [2][TM]: r > 0 bits
  static constexpr int off_red = off_mask + 2 * TM * 8;              // float [16][HID] column-sum scratch
  static constexpr int off_bar = off_red + 16 * HID * 4;
  static constexpr int total = off_bar + 128;
};

__device__ __forceinline__ float warp_colsum32(float (&v)[32], int lane) {
#pragma unroll
  for (int h = 16, off = 16; h >= 1; h >>= 1, off >>= 1) {
    const bool up = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < h; ++i) {
      const float send = up ? v[i] : v[i + h];
      const float keep = up ? v[i + h] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  return v[0];
}

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" :: "l"(p)); }

template <int KIN>
__global__ void __launch_bounds__(kThreadsB, 1)
gin_bwd_tc2_kernel(GinBwdMainPair pp) {
  using L = Smem<KIN>;
  const bool second = (int)blockIdx.x >= pp.split;
  const GinBwdMainArgs& p = pp.a[second ? 1 : 0];
  const int bid = second ? (int)blockIdx.x - pp.split : (int)blockIdx.x;          // CTA index / count inside its problem
  const int nblk = second ? (int)gridDim.x - pp.split : pp.split;
  const bool trace_on = pp.trace != 0;
  extern __shared__ __align__(1024) unsigned char smem[];
  uint2* s_mask = reinterpret_cast<uint2*>(smem + L::off_mask);
  float* s_red = reinterpret_cast<float*>(smem + L::off_red);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::off_bar);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + L::off_bar + B_COUNT * 8);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = (p.V + TM - 1) / TM;
  const int my_tiles = max(0, (n_tiles - bid + nblk - 1) / nblk);
  // Tiles are walked in DESCENDING row order: gin_bwd_pre (the previous launch) walks ascending, so the rows it touched
  // last (g_o just written, y just read) are still in the 126 MB L2 when this kernel starts, and the g_a rows this kernel
  // writes last (the lowest) are the ones the next layer's gin_bwd_pre gathers first.
  const bool rev = pp.reverse != 0;
  auto tile_base = [&](int i) { return (bid + (rev ? my_tiles - 1 - i : i) * nblk) * TM; };
  auto Xs = [&](int s) { return smem + L::off_stage + s * kStage; };
  auto Ys = [&](int s) { return smem + L::off_stage + s * kStage + 2 * kTile; };

  if (threadIdx.x == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(&bars[B_FULL1 + s], kLoadWarps);
      mbar_init(&bars[B_FULL2 + s], kLoadWarps);
      mbar_init(&bars[B_GU + s], kEpiWarps * 32);
      mbar_init(&bars[B_D1 + s], 1);
      mbar_init(&bars[B_D2 + s], 1);
    }
    mbar_init(&bars[B_E2], kEpiWarps * 32);
  }
  if (warp == kMmaWarp) tmem_alloc(s_tmem, 512);
  if (pp.wait_first) pdl_sync();
  // transposed weights, hi/lo split: W2t[in][out] = W2[out][in], W1t[kin][out] = W1[out][kin]  (K-major B operands)
  for (int i = threadIdx.x; i < HID * HID; i += kThreadsB) {
    const int o = i / HID, c = i % HID;                       // coalesced read of W2[o][c]
    const float v = __ldg(p.W2 + i), hi = tf32_rna(v), lo = tf32_rna(v - hi);
    const int off = tile_off4(HID, c, o >> 2, 128) + (o & 3) * 4;
    *reinterpret_cast<float*>(smem + L::off_w2 + off) = hi;
    *reinterpret_cast<float*>(smem + L::off_w2 + L::W2B + off) = lo;
  }
  for (int i = threadIdx.x; i < HID * KIN; i += kThreadsB) {
    const int o = i / KIN, c = i % KIN;
    const float v = __ldg(p.W1 + i), hi = tf32_rna(v), lo = tf32_rna(v - hi);
    const int off = tile_off4(HID, c, o >> 2, 128) + (o & 3) * 4;
    *reinterpret_cast<float*>(smem + L::off_w1 + off) = hi;
    *reinterpret_cast<float*>(smem + L::off_w1 + L::W1B + off) = lo;
  }
  if (!pp.wait_first) pdl_sync();   // the weights above are parameters; bn / cvec / g_o / y / r / a below come from the previous kernels
  fence_smem_to_async();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *s_tmem;

  float4 db2 = make4(0.f);          // loaders: column sums of g_y for channels 4*gl..4*gl+3 over this thread's rows
  float db1 = 0.f;                  // epilogue: column sums of g_u for column 32*half + lane over this warp's rows

  if (warp > kMmaWarp) {
    // =========================================================================== loaders
    const int pt = (warp - (kMmaWarp + 1)) * 32 + lane;
    constexpr int RPP = LT / 16, NR = TM / RPP;               // 16 rows per pass, 4 passes
    const int gl = pt & 15, gr = pt >> 4;
    const int c = gl * 4;
    const float4 mean = ldg4(p.bn + c), rstd = ldg4(p.bn + HID + c), gamma = ldg4(p.bn + 2 * HID + c);
    const float4 c1 = ldg4(p.cvec + c), c2 = ldg4(p.cvec + HID + c);
    // g_y = ka*g_o - kd*(y - mean) - ke      (ka = rstd*gamma, kd = rstd^2*c2, ke = rstd*c1)
    const float4 ka = make_float4(rstd.x * gamma.x, rstd.y * gamma.y, rstd.z * gamma.z, rstd.w * gamma.w);
    const float4 kd = make_float4(rstd.x * rstd.x * c2.x, rstd.y * rstd.y * c2.y, rstd.z * rstd.z * c2.z, rstd.w * rstd.w * c2.w);
    const float4 ke = make_float4(rstd.x * c1.x, rstd.y * c1.y, rstd.z * c1.z, rstd.w * c1.w);
    constexpr int ALPR = KIN / 4, ARPP = LT / ALPR, ANR = TM / ARPP;   // `a` rows: lanes per row, rows per pass, passes
    const int al = pt % ALPR, ar = pt / ALPR;
    // phase 1 of tile i: g_o, y, r rows -> g_y, r (hi/lo) -> X, Y of stage i & 1
    auto phase1 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      const int base = tile_base(i);
      unsigned char* X = Xs(s);
      unsigned char* Y = Ys(s);
      if (pt == 0) BWD2_TRACE(0, i);
      float4 go[NR], yy[NR], rr[NR];
#pragma unroll
      for (int j = 0; j < NR; ++j) {
        const int v = base + gr + j * RPP;
        const bool ok = v < p.V;
        const size_t o = (size_t)(ok ? v : 0) * HID + c;
        go[j] = ok ? ld4(p.g_o + o) : make4(0.f);
        yy[j] = ok ? ld4_cs(p.y + o) : make4(0.f);
        rr[j] = ok ? ld4_cs(p.r + o) : make4(0.f);
      }
      if (i + 2 < my_tiles) {                                 // two tiles ahead -> L2: 128 lines of 128 B per [64][64] tile
        const int nb = tile_base(i + 2), line = pt & 127;
        const size_t off = (size_t)nb * HID + (size_t)line * 32;
        if (off < (size_t)p.V * HID) {
          if (pt < 128) { prefetch_l2(p.y + off); prefetch_l2(p.g_o + off); }
          else {
            prefetch_l2(p.r + off);
            const size_t aoff = (size_t)nb * KIN + (size_t)line * 32;
            if (line * 32 < TM * KIN && aoff < (size_t)p.V * KIN) prefetch_l2(p.a + aoff);
          }
        }
      }
      if (use > 0) mbar_wait(&bars[B_D2 + s], (uint32_t)((use - 1) & 1));   // G2 / G4 of the stage's previous tile are done
      if (pt == 0) BWD2_TRACE(1, i);
#pragma unroll
      for (int j = 0; j < NR; ++j) {
        const int row = gr + j * RPP;
        const bool ok = base + row < p.V;
        float4 gy;
        gy.x = ka.x * go[j].x - kd.x * (yy[j].x - mean.x) - ke.x;
        gy.y = ka.y * go[j].y - kd.y * (yy[j].y - mean.y) - ke.y;
        gy.z = ka.z * go[j].z - kd.z * (yy[j].z - mean.z) - ke.z;
        gy.w = ka.w * go[j].w - kd.w * (yy[j].w - mean.w) - ke.w;
        if (!ok) gy = make4(0.f);
        db2 = add4(db2, gy);
        store_split4_s(X, X + kTile, TM, row, gl, gy);
        store_split4_s(Y, Y + kTile, TM, row, gl, rr[j]);
        // r > 0 bits of the row: field q of the two words holds channel 4*l + q at bit l
        const unsigned b0 = __ballot_sync(0xffffffffu, rr[j].x > 0.f), b1 = __ballot_sync(0xffffffffu, rr[j].y > 0.f);
        const unsigned b2 = __ballot_sync(0xffffffffu, rr[j].z > 0.f), b3 = __ballot_sync(0xffffffffu, rr[j].w > 0.f);
        if (gl == 0) {
          const int sh = lane & 16;
          s_mask[s * TM + row] = make_uint2(((b0 >> sh) & 0xffffu) | (((b1 >> sh) & 0xffffu) << 16),
                                            ((b2 >> sh) & 0xffffu) | (((b3 >> sh) & 0xffffu) << 16));
        }
      }
      fence_smem_to_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars[B_FULL1 + s]);
      if (pt == 0) BWD2_TRACE(2, i);
    };
    if (my_tiles > 0) phase1(0);
    for (int i = 0; i < my_tiles; ++i) {
      const int s = i & 1, use = i >> 1;
      const int base = tile_base(i);
      unsigned char* Y = Ys(s);
      // the next tile's g_y / r go into the other stage while the tensor pipe works on this one
      if (i + 1 < my_tiles) phase1(i + 1);
      // ---- phase 2 of tile i: a rows -> (after G1 / G3 have read Y) -> Y
      float4 aa[ANR];
#pragma unroll
      for (int j = 0; j < ANR; ++j) {
        const int v = base + ar + j * ARPP;
        aa[j] = v < p.V ? ld4_cs(p.a + (size_t)v * KIN + al * 4) : make4(0.f);
      }
      mbar_wait(&bars[B_D1 + s], (uint32_t)(use & 1));
      if (pt == 0) BWD2_TRACE(3, i);
#pragma unroll
      for (int j = 0; j < ANR; ++j) store_split4_s(Y, Y + TM * KIN * 4, TM, ar + j * ARPP, al, aa[j]);
      fence_smem_to_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars[B_FULL2 + s]);
      if (pt == 0) BWD2_TRACE(4, i);
    }
  } else if (warp == kMmaWarp) {
    // =========================================================================== MMA issuer (converged warp, elected lane)
    const uint32_t w2 = smem_u32(smem + L::off_w2), w1 = smem_u32(smem + L::off_w1);
    constexpr uint32_t idG1a = idesc_tf32(TM, 2 * HID, false, false), idG1b = idesc_tf32(TM, HID, false, false);
    constexpr uint32_t idG2a = idesc_tf32(TM, 2 * KIN, false, false), idG2b = idesc_tf32(TM, KIN, false, false);
    constexpr uint32_t idG3 = idesc_tf32(128, HID, true, true);          // [g_hi | g_lo]^T x r_hi (then r_lo)
    constexpr uint32_t idG4 = idesc_tf32(128, KIN, true, true);          // [g_hi | g_lo]^T x a_hi (then a_lo)
    auto g13 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      const uint32_t xh = smem_u32(Xs(s)), xl = xh + kTile, yh = smem_u32(Ys(s)), yl = yh + kTile;
      mbar_wait(&bars[B_FULL1 + s], (uint32_t)(use & 1));
      fence_after_sync();
      if (lane == 0) BWD2_TRACE(5, i);
      const uint32_t d1 = tmem + kColD1 + s * 128;
      // G1: g_r = g_y W2          (A = X K-major, B = [W2t_hi | W2t_lo])
#pragma unroll
      for (int k = 0; k < HID / 8; ++k) {
        const uint64_t b = desc_g_dense(w2, HID, k);
        mma_tf32_w(d1, desc_s_kmajor(xh, TM, k), b, idG1a, k > 0);
        mma_tf32_w(d1, desc_s_kmajor(xl, TM, k), b, idG1b, true);
      }
      // G3: dW2 += [g_hi | g_lo]^T (r_hi + r_lo)   (X, Y MN-major; hi and lo tiles of X adjacent), accumulated over all tiles
#pragma unroll
      for (int k = 0; k < TM / 8; ++k) {
        const uint64_t a = desc_s_mnmajor(xh, TM, k);
        mma_tf32_w(tmem + kColD3, a, desc_s_mnmajor(yh, TM, k), idG3, i > 0 || k > 0);
        mma_tf32_w(tmem + kColD3, a, desc_s_mnmajor(yl, TM, k), idG3, true);
      }
      mma_commit_w(&bars[B_D1 + s]);
    };
    auto g24 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      const uint32_t xh = smem_u32(Xs(s)), xl = xh + kTile, yh = smem_u32(Ys(s)), yl = yh + TM * KIN * 4;
      mbar_wait(&bars[B_GU + s], (uint32_t)(use & 1));
      mbar_wait(&bars[B_FULL2 + s], (uint32_t)(use & 1));
      if (i > 0) mbar_wait(&bars[B_E2], (uint32_t)((i - 1) & 1));      // epilogue 2 of the previous tile has read D2
      fence_after_sync();
      if (lane == 0) BWD2_TRACE(6, i);
      // G2: g_a = g_u W1          (A = X K-major, B = [W1t_hi | W1t_lo])
#pragma unroll
      for (int k = 0; k < HID / 8; ++k) {
        const uint64_t b = desc_g_dense(w1, HID, k);
        mma_tf32_w(tmem + kColD2, desc_s_kmajor(xh, TM, k), b, idG2a, k > 0);
        mma_tf32_w(tmem + kColD2, desc_s_kmajor(xl, TM, k), b, idG2b, true);
      }
      // G4: dW1 += [g_hi | g_lo]^T (a_hi + a_lo)
#pragma unroll
      for (int k = 0; k < TM / 8; ++k) {
        const uint64_t a = desc_s_mnmajor(xh, TM, k);
        mma_tf32_w(tmem + kColD4, a, desc_s_mnmajor(yh, TM, k), idG4, i > 0 || k > 0);
        mma_tf32_w(tmem + kColD4, a, desc_s_mnmajor(yl, TM, k), idG4, true);
      }
      mma_commit_w(&bars[B_D2 + s]);
    };
    // G1/G3 of tile i+1 are queued BEFORE G2/G4 of tile i: they run while the epilogue produces g_u of tile i
    if (my_tiles > 0) g13(0);
    for (int i = 0; i < my_tiles; ++i) {
      if (i + 1 < my_tiles) g13(i + 1);
      g24(i);
    }
  } else {
    // =========================================================================== epilogue
    // warp w: TMEM lane quarter q = w & 3 (rows 16q + lane, lanes 0..15), column half h = w >> 2 (channels 32h ..)
    const int q = warp & 3, half = warp >> 2;
    const int row = q * 16 + (lane & 15);
    const bool act = lane < 16;
    const int c0 = half * 32;
    const uint32_t tl = (uint32_t)(q * 32) << 16;
    // epilogue 1 of tile i: g_u = g_r * [r > 0] -> X (hi/lo), column sums for db1
    auto epi1 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      unsigned char* X = Xs(s);
      mbar_wait(&bars[B_D1 + s], (uint32_t)(use & 1));
      fence_after_sync();
      if (threadIdx.x == 0) BWD2_TRACE(7, i);
      const uint32_t d1 = tmem + tl + kColD1 + s * 128;
      const uint2 m = s_mask[s * TM + row];
      float g[32], t2[32];
      tmem_ld16_nowait(d1 + c0, *reinterpret_cast<float (*)[16]>(g));
      tmem_ld16_nowait(d1 + c0 + 16, *reinterpret_cast<float (*)[16]>(g + 16));
      tmem_ld16_nowait(d1 + HID + c0, *reinterpret_cast<float (*)[16]>(t2));
      tmem_ld16_nowait(d1 + HID + c0 + 16, *reinterpret_cast<float (*)[16]>(t2 + 16));
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const int cc = c0 + j;                                // channel 4*l + f  ->  bit l of 16-bit field f
        const unsigned word = (cc & 2) ? m.y : m.x;
        const bool on = act && ((word >> (((cc & 1) << 4) + (cc >> 2))) & 1u);
        g[j] = on ? g[j] + t2[j] : 0.f;
      }
      if (act) {
#pragma unroll
        for (int f = 0; f < 8; ++f)
          store_split4_s(X, X + kTile, TM, row, 8 * half + f, make_float4(g[4 * f], g[4 * f + 1], g[4 * f + 2], g[4 * f + 3]));
      }
      db1 += warp_colsum32(g, lane);                          // inactive lanes and rows beyond V hold zeros
      fence_smem_to_async();
      fence_before_sync();
      mbar_arrive(&bars[B_GU + s]);
      if (threadIdx.x == 0) BWD2_TRACE(8, i);
    };
    // epilogue 2 of tile i: g_a -> global
    auto epi2 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      const int gv = tile_base(i) + row;
      mbar_wait(&bars[B_D2 + s], (uint32_t)(use & 1));
      fence_after_sync();
      if (threadIdx.x == 0) BWD2_TRACE(9, i);
      if (KIN == HID || half == 0) {
        const int cb = KIN == HID ? c0 : 0;                   // 32 columns per warp (two halves for KIN = 64, one for KIN = 32)
        float g[32], t2[32];
        tmem_ld16_nowait(tmem + tl + kColD2 + cb, *reinterpret_cast<float (*)[16]>(g));
        tmem_ld16_nowait(tmem + tl + kColD2 + cb + 16, *reinterpret_cast<float (*)[16]>(g + 16));
        tmem_ld16_nowait(tmem + tl + kColD2 + KIN + cb, *reinterpret_cast<float (*)[16]>(t2));
        tmem_ld16_nowait(tmem + tl + kColD2 + KIN + cb + 16, *reinterpret_cast<float (*)[16]>(t2 + 16));
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) g[j] += t2[j];
        if (act && gv < p.V) {
#pragma unroll
          for (int j = 0; j < 4; ++j) st8(p.g_a + (size_t)gv * KIN + cb + 8 * j, g + 8 * j);
        }
      }
      fence_before_sync();
      mbar_arrive(&bars[B_E2]);                               // D2 may be overwritten by G2 of the next tile
      if (threadIdx.x == 0) BWD2_TRACE(10, i);
    };
    // g_r of tile i+1 is ready before g_a of tile i (MMA issue order): mask / re-split it first
    if (my_tiles > 0) epi1(0);
    for (int i = 0; i < my_tiles; ++i) {
      if (i + 1 < my_tiles) epi1(i + 1);
      epi2(i);
    }
  }
  // ---- every CTA writes its partial gradients (zeros when it had no tile)
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  float* part = p.part + (size_t)blockIdx.x * p.pstride;
  // dW2 / dW1 from tensor memory: accumulator row L (TMEM lane L): L < 64 = hi part of out-channel L, L >= 64 = lo part of
  // out-channel L - 64 (both already summed over B_hi + B_lo).  dW[o][i] = row o + row 64 + o.
  float* s_x = reinterpret_cast<float*>(smem);          // [64][HID + 1] exchange buffer (the stages are dead)
  for (int pass = 0; pass < 2; ++pass) {                // pass 0: dW2 (C = HID), pass 1: dW1 (C = KIN)
    const int C = pass == 0 ? HID : KIN;
    const uint32_t col = pass == 0 ? kColD3 : kColD4;
    const int64_t offW = pass == 0 ? p.off_W2 : p.off_W1;
    float t[64];
    if (warp < 4) {
      const uint32_t tl = (uint32_t)(warp * 32) << 16;
      const int Lr = warp * 32 + lane;
#pragma unroll
      for (int c16 = 0; c16 < 4; ++c16) {
        float a0[16];
        if (my_tiles > 0 && c16 * 16 < C) tmem_ld16(tmem + tl + col + c16 * 16, a0);
#pragma unroll
        for (int j = 0; j < 16; ++j) t[c16 * 16 + j] = (my_tiles > 0 && c16 * 16 < C) ? a0[j] : 0.f;
      }
      if (Lr >= 64) {
#pragma unroll
        for (int j = 0; j < 64; ++j) s_x[(Lr - 64) * (HID + 1) + j] = t[j];
      }
    }
    __syncthreads();
    if (warp < 2) {
      const int o = warp * 32 + lane;
      for (int j = 0; j < C; j += 4) {
        float4 v;
        v.x = t[j] + s_x[o * (HID + 1) + j];         v.y = t[j + 1] + s_x[o * (HID + 1) + j + 1];
        v.z = t[j + 2] + s_x[o * (HID + 1) + j + 2]; v.w = t[j + 3] + s_x[o * (HID + 1) + j + 3];
        st4(part + offW + (size_t)o * C + j, v);
      }
    }
    __syncthreads();
  }
  // db1: the four lane-quarter warps of each column half, fixed order
  if (warp < kEpiWarps) s_red[(warp & 3) * HID + (warp >> 2) * 32 + lane] = db1;
  __syncthreads();
  if (threadIdx.x < HID)
    part[p.off_b1 + threadIdx.x] = (s_red[threadIdx.x] + s_red[HID + threadIdx.x]) + (s_red[2 * HID + threadIdx.x] + s_red[3 * HID + threadIdx.x]);
  __syncthreads();
  // db2: loaders' per-thread sums, 16 row groups per channel quad, fixed order
  if (warp > kMmaWarp) {
    const int pt = (warp - (kMmaWarp + 1)) * 32 + lane;
    st4(s_red + (pt >> 4) * HID + (pt & 15) * 4, db2);
  }
  __syncthreads();
  if (threadIdx.x < HID) {
    float sum = 0.f;
#pragma unroll
    for (int g = 0; g < 16; ++g) sum += s_red[g * HID + threadIdx.x];
    part[p.off_b2 + threadIdx.x] = sum;
  }
  fence_before_sync();
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc(tmem, 512);
}

}  // namespace bwd2

template <int KIN>
static void launch_bwd2(const GinBwdMainPair& pp, int grid, cudaStream_t s) {
  using L = bwd2::Smem<KIN>;
  static bool once = (cudaFuncSetAttribute(bwd2::gin_bwd_tc2_kernel<KIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::total), true);
  (void)once;
  launch_k((bwd2::gin_bwd_tc2_kernel<KIN>), dim3(grid), dim3(bwd2::kThreadsB), L::total, s, pp);
}

}  // namespace scgib
extern "C" __attribute__((visibility("default"))) int scgib_debug_bwd_trace(long long* host_out, int n) {
  return (int)cudaMemcpyFromSymbol(host_out, scgib::g_bwd2_trace, (size_t)n * sizeof(long long));
}
namespace scgib {
static int bwd2_trace_flag() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("SCGIB_DBG"); v = (e && (atoi(e) & 2048)) ? 1 : 0; }
  return v;
}

void launch_gin_bwd_main_tc2(const GinBwdMainArgs& a, int kin, int grid, cudaStream_t s) {
  GinBwdMainPair pp;
  pp.a[0] = a; pp.a[1] = a;
  pp.split = grid;
  pp.trace = 0;
  pp.reverse = 0;
  if (kin == 32) launch_bwd2<32>(pp, grid, s); else launch_bwd2<HID>(pp, grid, s);
}

// the same layer of both encoders in one launch: CTAs [0, split) write the partial gradients of a0, [split, grid) of a1
// (split as computed by pair_split on 128-row tile counts: api.cu uses the same rule for the partial-sum ranges)
void launch_gin_bwd_main_tc2_pair(const GinBwdMainArgs& a0, const GinBwdMainArgs& a1, int kin, int grid, cudaStream_t s,
                                  bool weights_from_prev_kernel) {
  GinBwdMainPair pp;
  pp.a[0] = a0; pp.a[1] = a1;
  pp.wait_first = weights_from_prev_kernel ? 1 : 0;
  pp.split = pair_split(grid, (a0.V + 127) / 128, (a1.V + 127) / 128);
  pp.trace = bwd2_trace_flag();
  static int rev = -1;
  if (rev < 0) { const char* e = getenv("SCGIB_BWD_REV"); rev = (e && e[0] == '0') ? 0 : 1; }
  pp.reverse = rev;
  if (kin == 32) launch_bwd2<32>(pp, grid, s); else launch_bwd2<HID>(pp, grid, s);
}

}  // namespace scgib
