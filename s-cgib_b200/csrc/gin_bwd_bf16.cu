// gin_bwd_bf16.cu - GIN layer BACKWARD in bf16 mode (ScgibDims.act_dtype = SCGIB_ACT_BF16), hidden width H = 64 or 128.
//
// Same math as gin_bwd_pre_kernel + gin_bwd_h (reference: autograd of models.py:66-72), on bf16 activations / layer
// gradients with fp32 accumulation everywhere:
//   pre : G_v = Ga_v + sum_{u in N(v)} Ga_u (bf16x8 gathers through the symmetric CSR; top layer: fp32 rows through a map),
//         g_o = G * [relu(BN(y)) > 0] -> bf16, d gamma / d beta (of the ROUNDED g_o, so that the BatchNorm backward
//         below is exactly consistent), fixed-order in-kernel finalise, c1 = gamma*dbeta/V, c2 = gamma*dgamma/V.
//   main: g_y = rstd*(gamma*g_o - c1 - yhat*c2);  G1 g_r = g_y W2;  G3 dW2 += g_y^T r;  g_u = g_r * [r > 0];
//         G2 g_a = g_u W1;  G4 dW1 += g_u^T a;  db2 += sum g_y;  db1 += sum g_u
//         as SINGLE-PASS tcgen05 kind::f16 MMAs on 128-row tiles: the row tiles X (g_y, then g_u in place) and Y (r, then
//         a in place) are stored ONCE in format B (umma.cuh) and read K-major by G1 / G2 and MN-major by G3 / G4; the
//         weights stay in their natural [out][in] layout and are read MN-major (no transposed copies); dW2 / dW1
//         accumulate in tensor memory over all tiles of the CTA.  24 MMAs per 128 rows at H = 64 (the 3xTF32 kernel: 128).
#include <stdlib.h>
#include "kernels.cuh"
#include "umma.cuh"

namespace scgib {
using namespace umma;

namespace bfb {

__device__ __forceinline__ uint4 ldg16(const void* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }
__device__ __forceinline__ uint4 ldg16_cs(const void* p) { return __ldcs(reinterpret_cast<const uint4*>(p)); }
__device__ __forceinline__ void unpack8(uint4 h, float (&v)[8]) {
  v[0] = bf16_lo(h.x); v[1] = bf16_hi(h.x); v[2] = bf16_lo(h.y); v[3] = bf16_hi(h.y);
  v[4] = bf16_lo(h.z); v[5] = bf16_hi(h.z); v[6] = bf16_lo(h.w); v[7] = bf16_hi(h.w);
}
__device__ __forceinline__ uint4 pack8(const float (&v)[8]) {
  return make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
}

// ------------------------------------------------------------------------------------------------
// part 1: upstream gradient of h' = relu(BN(y)), ReLU mask, d gamma / d beta
// ------------------------------------------------------------------------------------------------
template <int H, int MINB>
__global__ void __launch_bounds__(kThreads, MINB)
gin_bwd_pre_bf16_kernel(GinBwdPrePair pp) {
  pdl_sync();
  const bool second = (int)blockIdx.x >= pp.split;
  const GinBwdPreArgs& p = pp.a[second ? 1 : 0];
  const int bid = second ? (int)blockIdx.x - pp.split : (int)blockIdx.x;
  const int nblk = second ? (int)gridDim.x - pp.split : pp.split;
  constexpr int LPR = H / 8, RPC = kThreads / LPR;            // lanes per row (8 channels each), rows per CTA pass
  __shared__ __align__(16) float s_red[RPC * 2 * H];
  __shared__ double s_d[kThreads];
  const int l = threadIdx.x % LPR, hw = threadIdx.x / LPR;
  const bf16_t* y = reinterpret_cast<const bf16_t*>(p.y);
  bf16_t* g_o = reinterpret_cast<bf16_t*>(p.g_o);
  float mean[8], rstd[8], sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int c = l * 8 + j;
    mean[j] = __ldg(p.bn + c); rstd[j] = __ldg(p.bn + H + c);
    sc[j] = rstd[j] * __ldg(p.bn + 2 * H + c); sh[j] = __ldg(p.bn + 3 * H + c) - mean[j] * sc[j];
  }
  float db[8], dg[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { db[j] = 0.f; dg[j] = 0.f; }
  constexpr int NR = 4;
  for (int v0 = bid * RPC + hw; v0 < p.V; v0 += nblk * RPC * NR) {
    int vv[NR];
    uint4 yy[NR];
    float g[NR][8];
#pragma unroll
    for (int j = 0; j < NR; ++j) {
      vv[j] = v0 + j * nblk * RPC;
      yy[j] = vv[j] < p.V ? ldg16_cs(y + (size_t)vv[j] * H + l * 8) : make_uint4(0, 0, 0, 0);
    }
    if (p.indptr) {     // G_v = Ga_v + sum_{u in N(v)} Ga_u, neighbours in CSR order, two slots of NR rows in flight
      const bf16_t* src = reinterpret_cast<const bf16_t*>(p.src);
      int e0[NR], deg[NR], maxd = 0;
#pragma unroll
      for (int j = 0; j < NR; ++j) {
        const bool ok = vv[j] < p.V;
        e0[j] = ok ? __ldg(p.indptr + vv[j]) : 0;
        deg[j] = ok ? __ldg(p.indptr + vv[j] + 1) - e0[j] : 0;
        maxd = max(maxd, deg[j]);
      }
      int u0[NR], u1[NR];
#pragma unroll
      for (int j = 0; j < NR; ++j) {
        u0[j] = deg[j] > 0 ? __ldg(p.indices + e0[j]) : -1;
        u1[j] = deg[j] > 1 ? __ldg(p.indices + e0[j] + 1) : -1;
      }
      uint4 hs[NR], h0[NR], h1[NR];
#pragma unroll
      for (int j = 0; j < NR; ++j) {
        hs[j] = vv[j] < p.V ? ldg16(src + (size_t)vv[j] * H + l * 8) : make_uint4(0, 0, 0, 0);
        h0[j] = u0[j] >= 0 ? ldg16(src + (size_t)u0[j] * H + l * 8) : make_uint4(0, 0, 0, 0);
        h1[j] = u1[j] >= 0 ? ldg16(src + (size_t)u1[j] * H + l * 8) : make_uint4(0, 0, 0, 0);
      }
#pragma unroll
      for (int j = 0; j < NR; ++j) {
        float a[8], b[8], c[8];
        unpack8(hs[j], a); unpack8(h0[j], b); unpack8(h1[j], c);
#pragma unroll
        for (int q = 0; q < 8; ++q) g[j][q] = (a[q] + b[q]) + c[q];
      }
      for (int d = 2; d < maxd; d += 2) {
#pragma unroll
        for (int j = 0; j < NR; ++j) {
          u0[j] = deg[j] > d ? __ldg(p.indices + e0[j] + d) : -1;
          u1[j] = deg[j] > d + 1 ? __ldg(p.indices + e0[j] + d + 1) : -1;
        }
#pragma unroll
        for (int j = 0; j < NR; ++j) {
          h0[j] = u0[j] >= 0 ? ldg16(src + (size_t)u0[j] * H + l * 8) : make_uint4(0, 0, 0, 0);
          h1[j] = u1[j] >= 0 ? ldg16(src + (size_t)u1[j] * H + l * 8) : make_uint4(0, 0, 0, 0);
        }
#pragma unroll
        for (int j = 0; j < NR; ++j) {
          float b[8], c[8];
          unpack8(h0[j], b); unpack8(h1[j], c);
#pragma unroll
          for (int q = 0; q < 8; ++q) g[j][q] = (g[j][q] + b[q]) + c[q];
        }
      }
    } else {            // top layer: fp32 rows of gH / gC, optionally through a row map
#pragma unroll
      for (int j = 0; j < NR; ++j) {
        float4 a = make4(0.f), b = make4(0.f);
        if (vv[j] < p.V) {
          const float* s = p.src + (size_t)(p.map ? __ldg(p.map + vv[j]) : vv[j]) * H + l * 8;
          a = ld4(s); b = ld4(s + 4);
        }
        g[j][0] = a.x; g[j][1] = a.y; g[j][2] = a.z; g[j][3] = a.w; g[j][4] = b.x; g[j][5] = b.y; g[j][6] = b.z; g[j][7] = b.w;
      }
    }
#pragma unroll
    for (int j = 0; j < NR; ++j) {
      if (vv[j] >= p.V) continue;
      float yv[8];
      unpack8(yy[j], yv);
#pragma unroll
      for (int q = 0; q < 8; ++q) g[j][q] = fmaf(yv[q], sc[q], sh[q]) > 0.f ? g[j][q] : 0.f;
      const uint4 pk = pack8(g[j]);
      *reinterpret_cast<uint4*>(g_o + (size_t)vv[j] * H + l * 8) = pk;
      float gr[8];
      unpack8(pk, gr);
#pragma unroll
      for (int q = 0; q < 8; ++q) { db[q] += gr[q]; dg[q] = fmaf(gr[q], (yv[q] - mean[q]) * rstd[q], dg[q]); }
    }
  }
#pragma unroll
  for (int q = 0; q < 8; ++q) { s_red[hw * 2 * H + l * 8 + q] = db[q]; s_red[hw * 2 * H + H + l * 8 + q] = dg[q]; }
  __syncthreads();
  for (int j = threadIdx.x; j < 2 * H; j += kThreads) {
    float s = 0.f;
#pragma unroll
    for (int h = 0; h < RPC; ++h) s += s_red[h * 2 * H + j];
    p.part[(size_t)bid * 2 * H + j] = s;
  }
  if (!last_cta_arrives(p.counter, (unsigned)nblk)) return;
  {
    constexpr int NSEG = kThreads / (2 * H);                 // 2 (H = 64) or 1 (H = 128) interleaved segments per column
    const int j = threadIdx.x % (2 * H), seg = threadIdx.x / (2 * H);
    s_d[seg * 2 * H + j] = sum_partials(p.part + j, 2 * H, nblk, seg, NSEG);
    __syncthreads();
    if (threadIdx.x < H) {
      const int c = threadIdx.x;
      double dbeta = 0.0, dgamma = 0.0;
#pragma unroll
      for (int s = 0; s < NSEG; ++s) { dbeta += s_d[s * 2 * H + c]; dgamma += s_d[s * 2 * H + H + c]; }
      p.d_beta[c] = (float)dbeta;
      p.d_gamma[c] = (float)dgamma;
      const double gamma = (double)p.bn[2 * H + c];
      p.cvec[c] = (float)(gamma * dbeta / (double)p.V);
      p.cvec[H + c] = (float)(gamma * dgamma / (double)p.V);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// part 2: BatchNorm backward + the four MLP gradient GEMMs (persistent, one CTA per SM)
// ------------------------------------------------------------------------------------------------
constexpr int TM = 128;
constexpr int kEpiWarps = 8, kLoadWarps = 8;
constexpr int kMmaWarp = kEpiWarps;
constexpr int kThreadsB = (kEpiWarps + 1 + kLoadWarps) * 32;
constexpr int LT = kLoadWarps * 32;
enum { B_FULL1 = 0, B_FULL2 = 2, B_GU = 4, B_D1 = 6, B_D2 = 8, B_E2 = 10, B_COUNT = 11 };

template <int KIN, int H>
struct BwdSmem {
  static constexpr int KP = KIN < 64 ? 64 : KIN;                      // the `a` tile / g_a accumulator are padded to 64 columns
  static constexpr int HB = H / 64, KB = KP / 64;
  static constexpr int kX = HB * TM * 128;                             // g_y, then g_u
  static constexpr int kY = (HB > KB ? HB : KB) * TM * 128;            // r, then a
  static constexpr int kStage = kX + kY;
  static constexpr int W2B = HB * H * 128, W1B = KB * H * 128;         // natural [out rows][in columns] (MN-major B operands)
  static constexpr int off_stage = 0;
  static constexpr int off_w2 = 2 * kStage, off_w1 = off_w2 + W2B;
  static constexpr int off_mask = off_w1 + W1B;                        // uint8 [2][TM][H / 8]: r > 0 bits
  static constexpr int off_bar = off_mask + 2 * TM * (H / 8);
  static constexpr int total = off_bar + 128;
  static_assert(total <= 227 * 1024, "shared memory budget");
  static constexpr int D1BUF = H == 64 ? 2 : 1;
  static constexpr int colD1 = 0, colD2 = D1BUF * H, colD3 = colD2 + KP, colD4 = colD3 + H;
  static_assert(colD4 + KP <= 512, "tensor memory budget");
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

template <int OUT, int IN, int INP>
__device__ __forceinline__ void stage_weight(unsigned char* dst, const float* __restrict__ W, int tid, int nthreads) {
  for (int i = tid; i < OUT * (INP / 8); i += nthreads) {
    const int o = i / (INP / 8), c8 = i % (INP / 8);
    uint4 pk = make_uint4(0, 0, 0, 0);
    if (c8 * 8 < IN) {
      const float4 v0 = ldg4(W + (size_t)o * IN + c8 * 8), v1 = ldg4(W + (size_t)o * IN + c8 * 8 + 4);
      pk = make_uint4(pack_bf16x2(v0.x, v0.y), pack_bf16x2(v0.z, v0.w), pack_bf16x2(v1.x, v1.y), pack_bf16x2(v1.z, v1.w));
    }
    *reinterpret_cast<uint4*>(dst + (c8 >> 3) * (OUT * 128) + tile_b_off(o, c8 & 7)) = pk;
  }
}

// GA_F32: g_a is written as fp32 (layer 0: its consumer input_proj_bwd reads fp32)
template <int KIN, int H, bool GA_F32>
__global__ void __launch_bounds__(kThreadsB, 1)
gin_bwd_bf16_kernel(GinBwdMainPair pp) {
  using L = BwdSmem<KIN, H>;
  constexpr int KP = L::KP, CH = H / 64;
  const bool second = (int)blockIdx.x >= pp.split;
  const GinBwdMainArgs& p = pp.a[second ? 1 : 0];
  const int bid = second ? (int)blockIdx.x - pp.split : (int)blockIdx.x;
  const int nblk = second ? (int)gridDim.x - pp.split : pp.split;
  const bf16_t* p_go = reinterpret_cast<const bf16_t*>(p.g_o);
  const bf16_t* p_y = reinterpret_cast<const bf16_t*>(p.y);
  const bf16_t* p_r = reinterpret_cast<const bf16_t*>(p.r);
  const bf16_t* p_a = reinterpret_cast<const bf16_t*>(p.a);
  extern __shared__ __align__(1024) unsigned char smem[];
  unsigned char* s_mask = smem + L::off_mask;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::off_bar);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + L::off_bar + B_COUNT * 8);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = (p.V + TM - 1) / TM;
  const int my_tiles = max(0, (n_tiles - bid + nblk - 1) / nblk);
  const bool rev = pp.reverse != 0;
  auto tile_base = [&](int i) { return (bid + (rev ? my_tiles - 1 - i : i) * nblk) * TM; };
  auto Xs = [&](int s) { return smem + L::off_stage + s * L::kStage; };
  auto Ys = [&](int s) { return smem + L::off_stage + s * L::kStage + L::kX; };

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
  stage_weight<H, H, H>(smem + L::off_w2, p.W2, threadIdx.x, kThreadsB);
  stage_weight<H, KIN, KP>(smem + L::off_w1, p.W1, threadIdx.x, kThreadsB);
  pdl_sync();      // the weights above are parameters; bn / cvec / g_o / y / r / a below come from the previous kernels
  fence_smem_to_async();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *s_tmem;

  float db2[8];                      // loaders: column sums of g_y for channels 8*gl.. over this thread's rows
#pragma unroll
  for (int j = 0; j < 8; ++j) db2[j] = 0.f;
  float db1[CH];                     // epilogue: column sums of g_u for column half*(H/2) + 32 c + lane over this warp's rows
#pragma unroll
  for (int c = 0; c < CH; ++c) db1[c] = 0.f;

  if (warp > kMmaWarp) {
    // =========================================================================== loaders
    const int pt = (warp - (kMmaWarp + 1)) * 32 + lane;
    constexpr int LPR = H / 8, RPP = LT / LPR, NRT = TM / RPP;          // lanes per row, rows per pass, passes per tile
    constexpr int NB = 4;                                               // passes in flight
    const int gl = pt % LPR, gr = pt / LPR;
    float ka[8], kd[8], ke[8], mean[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = gl * 8 + j;
      const float rstd = __ldg(p.bn + H + c), gamma = __ldg(p.bn + 2 * H + c);
      mean[j] = __ldg(p.bn + c);
      ka[j] = rstd * gamma; kd[j] = rstd * rstd * __ldg(p.cvec + H + c); ke[j] = rstd * __ldg(p.cvec + c);
    }
    constexpr int ALPR = KIN / 8, ARPP = LT / ALPR, ANR = TM / ARPP;
    const int al = pt % ALPR, ar = pt / ALPR;
    auto phase1 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      const int base = tile_base(i);
      unsigned char* X = Xs(s);
      unsigned char* Y = Ys(s);
#pragma unroll 1
      for (int b0 = 0; b0 < NRT; b0 += NB) {
        uint4 go[NB], yy[NB], rr[NB];
#pragma unroll
        for (int j = 0; j < NB; ++j) {
          const int v = base + gr + (b0 + j) * RPP;
          const bool ok = v < p.V;
          const size_t o = (size_t)(ok ? v : 0) * H + gl * 8;
          go[j] = ok ? ldg16(p_go + o) : make_uint4(0, 0, 0, 0);
          yy[j] = ok ? ldg16_cs(p_y + o) : make_uint4(0, 0, 0, 0);
          rr[j] = ok ? ldg16_cs(p_r + o) : make_uint4(0, 0, 0, 0);
        }
        if (b0 == 0 && use > 0) mbar_wait(&bars[B_D2 + s], (uint32_t)((use - 1) & 1));   // G2 / G4 of the stage's previous tile are done
#pragma unroll
        for (int j = 0; j < NB; ++j) {
          const int row = gr + (b0 + j) * RPP;
          const bool ok = base + row < p.V;
          float g[8], yv[8], rv[8];
          unpack8(go[j], g); unpack8(yy[j], yv); unpack8(rr[j], rv);
          unsigned m = 0;
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            g[q] = ok ? ka[q] * g[q] - kd[q] * (yv[q] - mean[q]) - ke[q] : 0.f;
            m |= (rv[q] > 0.f ? 1u : 0u) << q;
          }
          const uint4 pk = pack8(g);
          float gq[8];
          unpack8(pk, gq);
#pragma unroll
          for (int q = 0; q < 8; ++q) db2[q] += gq[q];
          *reinterpret_cast<uint4*>(X + (gl >> 3) * (TM * 128) + tile_b_off(row, gl & 7)) = pk;
          *reinterpret_cast<uint4*>(Y + (gl >> 3) * (TM * 128) + tile_b_off(row, gl & 7)) = rr[j];
          s_mask[(s * TM + row) * (H / 8) + gl] = (unsigned char)m;
        }
      }
      fence_smem_to_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars[B_FULL1 + s]);
    };
    if (my_tiles > 0) phase1(0);
    for (int i = 0; i < my_tiles; ++i) {
      const int s = i & 1, use = i >> 1;
      const int base = tile_base(i);
      unsigned char* Y = Ys(s);
      if (i + 1 < my_tiles) phase1(i + 1);
      // phase 2 of tile i: a rows -> (after G1 / G3 have read Y) -> Y
      uint4 aa[ANR];
#pragma unroll
      for (int j = 0; j < ANR; ++j) {
        const int v = base + ar + j * ARPP;
        aa[j] = v < p.V ? ldg16_cs(p_a + (size_t)v * KIN + al * 8) : make_uint4(0, 0, 0, 0);
      }
      mbar_wait(&bars[B_D1 + s], (uint32_t)(use & 1));
#pragma unroll
      for (int j = 0; j < ANR; ++j) {
        const int row = ar + j * ARPP;
        *reinterpret_cast<uint4*>(Y + (al >> 3) * (TM * 128) + tile_b_off(row, al & 7)) = aa[j];
        if (KIN < 64) *reinterpret_cast<uint4*>(Y + tile_b_off(row, 4 + al)) = make_uint4(0, 0, 0, 0);   // padding columns: finite
      }
      fence_smem_to_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars[B_FULL2 + s]);
    }
  } else if (warp == kMmaWarp) {
    // =========================================================================== MMA issuer (converged warp, elected lane)
    const uint32_t w2 = smem_u32(smem + L::off_w2), w1 = smem_u32(smem + L::off_w1);
    constexpr uint32_t idG1 = idesc_bf16(TM, H, false, true);            // A = X K-major, B = W2 natural (MN-major)
    constexpr uint32_t idG2 = idesc_bf16(TM, KP, false, true);           // A = X K-major, B = W1 natural (MN-major)
    constexpr uint32_t idG3 = idesc_bf16(H, H, true, true);              // A = X^T, B = Y (r), K = tile rows
    constexpr uint32_t idG4 = idesc_bf16(H, KP, true, true);             // A = X^T, B = Y (a)
    auto g13 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      const uint32_t x = smem_u32(Xs(s)), y = smem_u32(Ys(s));
      mbar_wait(&bars[B_FULL1 + s], (uint32_t)(use & 1));
      if (L::D1BUF == 1 && i > 0) mbar_wait(&bars[B_GU + (s ^ 1)], (uint32_t)(((i - 1) >> 1) & 1));   // epilogue 1 of tile i-1 has read D1
      fence_after_sync();
      const uint32_t d1 = tmem + L::colD1 + (L::D1BUF == 2 ? s * H : 0);
#pragma unroll
      for (int k = 0; k < H / 16; ++k)       // G1: K = out channels; W2 rows 16k.. (MN-major: 2048 B per step), N blocks H*128 apart
        mma_bf16_w(d1, desc_b_kmajor(x + (k >> 2) * (TM * 128), k & 3), desc_b_mnmajor(w2, H * 128, k), idG1, k > 0);
#pragma unroll
      for (int k = 0; k < TM / 16; ++k)      // G3: K = tile rows
        mma_bf16_w(tmem + L::colD3, desc_b_mnmajor(x, TM * 128, k), desc_b_mnmajor(y, TM * 128, k), idG3, i > 0 || k > 0);
      mma_commit_w(&bars[B_D1 + s]);
    };
    auto g24 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      const uint32_t x = smem_u32(Xs(s)), y = smem_u32(Ys(s));
      mbar_wait(&bars[B_GU + s], (uint32_t)(use & 1));
      mbar_wait(&bars[B_FULL2 + s], (uint32_t)(use & 1));
      if (i > 0) mbar_wait(&bars[B_E2], (uint32_t)((i - 1) & 1));        // epilogue 2 of the previous tile has read D2
      fence_after_sync();
#pragma unroll
      for (int k = 0; k < H / 16; ++k)       // G2
        mma_bf16_w(tmem + L::colD2, desc_b_kmajor(x + (k >> 2) * (TM * 128), k & 3), desc_b_mnmajor(w1, H * 128, k), idG2, k > 0);
#pragma unroll
      for (int k = 0; k < TM / 16; ++k)      // G4
        mma_bf16_w(tmem + L::colD4, desc_b_mnmajor(x, TM * 128, k), desc_b_mnmajor(y, TM * 128, k), idG4, i > 0 || k > 0);
      mma_commit_w(&bars[B_D2 + s]);
    };
    if (my_tiles > 0) g13(0);
    for (int i = 0; i < my_tiles; ++i) {
      if (i + 1 < my_tiles) g13(i + 1);
      g24(i);
    }
  } else {
    // =========================================================================== epilogue
    const int q = warp & 3, half = warp >> 2;
    const int row = q * 32 + lane;
    const uint32_t tl = (uint32_t)(q * 32) << 16;
    auto epi1 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      unsigned char* X = Xs(s);
      mbar_wait(&bars[B_D1 + s], (uint32_t)(use & 1));
      fence_after_sync();
      const uint32_t d1 = tmem + tl + L::colD1 + (L::D1BUF == 2 ? s * H : 0);
#pragma unroll
      for (int c = 0; c < CH; ++c) {
        const int c0 = half * (H / 2) + 32 * c;
        const uint32_t m = *reinterpret_cast<const uint32_t*>(s_mask + (s * TM + row) * (H / 8) + c0 / 8);
        float g[32];
        tmem_ld16_nowait(d1 + c0, *reinterpret_cast<float (*)[16]>(g));
        tmem_ld16_nowait(d1 + c0 + 16, *reinterpret_cast<float (*)[16]>(g + 16));
        tmem_ld_wait();
#pragma unroll
        for (int f = 0; f < 4; ++f) {
          float v8[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) v8[j] = ((m >> (8 * f + j)) & 1u) ? g[8 * f + j] : 0.f;
          const uint4 pk = pack8(v8);
          const int c8 = c0 / 8 + f;
          *reinterpret_cast<uint4*>(X + (c8 >> 3) * (TM * 128) + tile_b_off(row, c8 & 7)) = pk;
          unpack8(pk, v8);
#pragma unroll
          for (int j = 0; j < 8; ++j) g[8 * f + j] = v8[j];
        }
        db1[c] += warp_colsum32(g, lane);                      // rows beyond V hold zeros
      }
      fence_smem_to_async();
      fence_before_sync();
      mbar_arrive(&bars[B_GU + s]);
    };
    auto epi2 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      const int gv = tile_base(i) + row;
      mbar_wait(&bars[B_D2 + s], (uint32_t)(use & 1));
      fence_after_sync();
      constexpr int CK = KIN >= 64 ? KIN / 64 : 1;             // 32-column chunks per warp (KIN = 32: the half-0 warps only)
      if (KIN >= 64 || half == 0) {
#pragma unroll
        for (int c = 0; c < CK; ++c) {
          const int c0 = KIN >= 64 ? half * (KIN / 2) + 32 * c : 0;
          float g[32];
          tmem_ld16_nowait(tmem + tl + L::colD2 + c0, *reinterpret_cast<float (*)[16]>(g));
          tmem_ld16_nowait(tmem + tl + L::colD2 + c0 + 16, *reinterpret_cast<float (*)[16]>(g + 16));
          tmem_ld_wait();
          if (gv < p.V) {
            if (GA_F32) {
#pragma unroll
              for (int j = 0; j < 4; ++j) st8(p.g_a + (size_t)gv * KIN + c0 + 8 * j, g + 8 * j);
            } else {
              bf16_t* dst = reinterpret_cast<bf16_t*>(p.g_a) + (size_t)gv * KIN + c0;
#pragma unroll
              for (int j = 0; j < 4; ++j)
                *reinterpret_cast<uint4*>(dst + 8 * j) = make_uint4(pack_bf16x2(g[8 * j], g[8 * j + 1]), pack_bf16x2(g[8 * j + 2], g[8 * j + 3]),
                                                                    pack_bf16x2(g[8 * j + 4], g[8 * j + 5]), pack_bf16x2(g[8 * j + 6], g[8 * j + 7]));
            }
          }
        }
      }
      fence_before_sync();
      mbar_arrive(&bars[B_E2]);
    };
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
  // dW2 [o][j] = D3, dW1 [o][i] = D4 (first KIN columns): accumulator row o is TMEM lane o (H = 128) or (o/16)*32 + o%16 (H = 64)
  if (warp < 4) {
    const uint32_t tl = (uint32_t)(warp * 32) << 16;
    const bool act = H == 128 || lane < 16;
    const int o = H == 128 ? warp * 32 + lane : warp * 16 + (lane & 15);
    for (int pass = 0; pass < 2; ++pass) {
      const int C = pass == 0 ? H : KIN;
      const uint32_t col = pass == 0 ? L::colD3 : L::colD4;
      float* dst = part + (pass == 0 ? p.off_W2 : p.off_W1) + (size_t)o * C;
      for (int c16 = 0; c16 < C; c16 += 16) {
        float t[16];
        if (my_tiles > 0) tmem_ld16(tmem + tl + col + c16, t);
        if (act) {
#pragma unroll
          for (int j = 0; j < 16; j += 4)
            st4(dst + c16 + j, my_tiles > 0 ? make_float4(t[j], t[j + 1], t[j + 2], t[j + 3]) : make4(0.f));
        }
      }
    }
  }
  float* s_red = reinterpret_cast<float*>(smem);                // [RPP or 4][H] scratch (the stages are dead)
  __syncthreads();
  if (warp < kEpiWarps) {
#pragma unroll
    for (int c = 0; c < CH; ++c) s_red[(warp & 3) * H + (warp >> 2) * (H / 2) + 32 * c + lane] = db1[c];
  }
  __syncthreads();
  if (threadIdx.x < H)
    part[p.off_b1 + threadIdx.x] = (s_red[threadIdx.x] + s_red[H + threadIdx.x]) + (s_red[2 * H + threadIdx.x] + s_red[3 * H + threadIdx.x]);
  __syncthreads();
  constexpr int RPPL = LT / (H / 8);
  if (warp > kMmaWarp) {
    const int pt = (warp - (kMmaWarp + 1)) * 32 + lane;
    const int gl = pt % (H / 8), gr = pt / (H / 8);
#pragma unroll
    for (int j = 0; j < 8; ++j) s_red[gr * H + gl * 8 + j] = db2[j];
  }
  __syncthreads();
  if (threadIdx.x < H) {
    float sum = 0.f;
#pragma unroll 8
    for (int g = 0; g < RPPL; ++g) sum += s_red[g * H + threadIdx.x];
    part[p.off_b2 + threadIdx.x] = sum;
  }
  fence_before_sync();
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc(tmem, 512);
}

}  // namespace bfb

int gin_bwd_pre_bf16_grid(int V, int hidden) { return gin_bwd_pre_grid(V); }
template <int H>
static void launch_pre_bf16_t(const GinBwdPrePair& pp, int grid, cudaStream_t s) {
  const int occ = gin_bwd_pre_occ();
  if (occ == 2) launch_k((bfb::gin_bwd_pre_bf16_kernel<H, 2>), dim3(grid), dim3(kThreads), 0, s, pp);
  else if (occ == 3) launch_k((bfb::gin_bwd_pre_bf16_kernel<H, 3>), dim3(grid), dim3(kThreads), 0, s, pp);
  else launch_k((bfb::gin_bwd_pre_bf16_kernel<H, 4>), dim3(grid), dim3(kThreads), 0, s, pp);
}

void launch_gin_bwd_pre_bf16(const GinBwdPreArgs& a0, const GinBwdPreArgs* a1, int hidden, cudaStream_t s) {
  GinBwdPrePair pp;
  pp.a[0] = a0; pp.a[1] = a1 ? *a1 : a0;
  const int grid = max(a1 ? 2 : 1, gin_bwd_pre_bf16_grid(a0.V + (a1 ? a1->V : 0), hidden));
  pp.split = a1 ? pair_split(grid, a0.V, a1->V) : grid;
  if (hidden == 64) launch_pre_bf16_t<64>(pp, grid, s); else launch_pre_bf16_t<128>(pp, grid, s);
}

template <int KIN, int H, bool GA_F32>
static void launch_bwd_bf16_t(const GinBwdMainPair& pp, int grid, cudaStream_t s) {
  using L = bfb::BwdSmem<KIN, H>;
  static bool once = (cudaFuncSetAttribute(bfb::gin_bwd_bf16_kernel<KIN, H, GA_F32>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::total), true);
  (void)once;
  launch_k((bfb::gin_bwd_bf16_kernel<KIN, H, GA_F32>), dim3(grid), dim3(bfb::kThreadsB), L::total, s, pp);
}

// CTAs [0, split) write the partial gradients of a0, [split, grid) of a1 (a1 == nullptr: one problem).  g_o / y / r / a are
// bf16; g_a is bf16, except with ga_f32 (layer 0 and the head backward), where it is fp32.  kin < hidden happens at layer 0
// only, which always takes fp32 g_a.
void launch_gin_bwd_main_bf16(const GinBwdMainArgs& a0, const GinBwdMainArgs* a1, int kin, int hidden, int grid, cudaStream_t s,
                              bool ga_f32) {
  GinBwdMainPair pp;
  pp.a[0] = a0; pp.a[1] = a1 ? *a1 : a0;
  pp.split = a1 ? pair_split(grid, (a0.V + 127) / 128, (a1->V + 127) / 128) : grid;
  pp.trace = 0;
  pp.reverse = 1;
  if (hidden == 64) {
    if (kin == 32) launch_bwd_bf16_t<32, 64, true>(pp, grid, s);
    else if (ga_f32) launch_bwd_bf16_t<64, 64, true>(pp, grid, s);
    else launch_bwd_bf16_t<64, 64, false>(pp, grid, s);
  } else {
    if (kin == 32) launch_bwd_bf16_t<32, 128, true>(pp, grid, s);
    else if (kin == 64) launch_bwd_bf16_t<64, 128, true>(pp, grid, s);
    else if (ga_f32) launch_bwd_bf16_t<128, 128, true>(pp, grid, s);
    else launch_bwd_bf16_t<128, 128, false>(pp, grid, s);
  }
}

}  // namespace scgib
