// gin_bf16.cu - GIN layer FORWARD in bf16 mode (ScgibDims.act_dtype = SCGIB_ACT_BF16), hidden width H = 64 or 128.
//
// Same contract as gin_fwd_tc3 (reference models.py:66-72: DGL GINConv 'sum' + MLP + BatchNorm1d statistics) and the
// same warp-specialised persistent pipeline (TMA window one tile ahead -> CSR gather out of shared memory -> GEMM1 ->
// epilogue 1 -> GEMM2 -> epilogue 2 + statistics), but every activation tensor is bf16 in HBM (`in`, a, r, y: half the
// bytes of the fp32 path) and the two 64 / 128-wide GEMMs are SINGLE-PASS tcgen05 kind::f16 MMAs with fp32 accumulation:
//   * gathers are 16-byte loads of 8 bf16 channels (bf16x8), accumulated in fp32; BN + ReLU of the producing layer is one
//     FMA + max per element (scale = rstd*gamma, shift = beta - mean*scale);
//   * operand tiles are format B of umma.cuh (dense 128-byte rows, SWIZZLE_128B): 1 MMA per K = 16 step instead of the
//     3xTF32 path's 2 x (K = 8) hi/lo pairs - 8 instead of 32 MMAs per 128-row tile at H = 64;
//   * r = relu(u + b1) is packed to bf16x2 in registers and handed to GEMM2 through TENSOR MEMORY (A operand in TMEM:
//     16 r columns = 8 TMEM columns per K step), never through shared memory;
//   * y is rounded to bf16 once; the batch statistics are those of the ROUNDED values (what the consumers normalise),
//     per-warp Chan/Welford triples in fp64, fixed-order combine.
// Operand formats pinned on B200 by tests/csrc/umma_probe_bf16.cu (profiles/r02_umma_probe_bf16.txt).
#include <stdlib.h>
#include "kernels.cuh"
#include "umma.cuh"

namespace scgib {
using namespace umma;

// per-tile role timestamps (SCGIB_DBG bit 1024; experiments only, tests/gpu_tc2_trace.py)
__device__ long long g_bf16_trace[160 * 16 * 12];
#define BF_TRACE(ev, tile) do { if ((p.dbg & 1024) && (tile) < 16 && blockIdx.x < 160) g_bf16_trace[((size_t)blockIdx.x * 16 + (tile)) * 12 + (ev)] = clock64(); } while (0)

namespace bf {
constexpr int TM = 128;                       // rows per tile = UMMA M
constexpr int kEpiWarps = 8;
constexpr int kMmaWarp = kEpiWarps;
constexpr int kIdxBufs = 3;
constexpr int HALO = 64, WIN = TM + 2 * HALO;

template <int KIN, int H>
struct FwdSmem {
  static constexpr int KB = (KIN + 63) / 64, HB = H / 64;             // 64-column blocks of the A tile / of r
  static constexpr int ROWB = KIN * 2;                                 // bytes of a raw window row
  static constexpr int kWin = WIN * ROWB, kA = KB * TM * 128;
  static constexpr int kStage = ((kWin > kA ? kWin : kA) + 1023) / 1024 * 1024;
  static constexpr int W1B = KB * H * 128, W2B = HB * H * 128;         // K-major B operands [H out rows][64-col blocks]
  static constexpr int kIdxCap = 1024;
  static constexpr int off_stage = 0;
  static constexpr int off_w1 = 2 * kStage, off_w2 = off_w1 + W1B;
  static constexpr int off_f = off_w2 + W2B;                           // b1[H] b2[H] scale[H] shift[H]
  static constexpr int off_bar = off_f + 4 * H * 4;
  static constexpr int off_ip = off_bar + 128;                         // int [3][TM + 4]
  static constexpr int off_self = off_ip + kIdxBufs * (TM + 4) * 4;    // int [3][WIN]
  static constexpr int off_ix = off_self + kIdxBufs * WIN * 4;         // int [3][kIdxCap]
  static constexpr int total = off_ix + kIdxBufs * kIdxCap * 4;
  static_assert(total <= 227 * 1024, "shared memory budget");
  static_assert(2 * kStage >= (8 * 3 * (H / 2) + 4 * 3 * H) * 8, "statistics scratch aliases the stages");
};

enum { B_FULL_A = 0, B_EMPTY_A = 2, B_D1 = 4, B_R = 6, B_D2 = 8, B_RAW = 10, B_COUNT = 12 };

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

__device__ __forceinline__ void tmem_st16u(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
      :: "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
         "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]) : "memory");
}
__device__ __forceinline__ void stg16(void* p, uint4 v) { *reinterpret_cast<uint4*>(p) = v; }
__device__ __forceinline__ void stg16_cs(void* p, uint4 v) {
  asm volatile("st.global.cs.v4.b32 [%0], {%1,%2,%3,%4};" :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void mma_bf16_ta_w(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, bool accumulate) {
  if (elect_one()) mma_bf16_ta(d_tmem, a_tmem, b_desc, idesc, accumulate);
}
// acc[0..7] += f(h) for the 8 bf16 channels packed in h; f = relu(h*scale + shift) (BN) or identity
template <bool BN>
__device__ __forceinline__ void acc8(float (&acc)[8], uint4 h, const float (&sc)[8], const float (&sh)[8]) {
  const uint32_t w[4] = {h.x, h.y, h.z, h.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float lo = bf16_lo(w[i]), hi = bf16_hi(w[i]);
    if (BN) {
      acc[2 * i] += fmaxf(fmaf(lo, sc[2 * i], sh[2 * i]), 0.f);
      acc[2 * i + 1] += fmaxf(fmaf(hi, sc[2 * i + 1], sh[2 * i + 1]), 0.f);
    } else {
      acc[2 * i] += lo;
      acc[2 * i + 1] += hi;
    }
  }
}

// weights: natural fp32 [OUT rows][IN cols] -> bf16 K-major B operand (format B blocks of 64 columns, OUT rows each)
template <int OUT, int IN>
__device__ __forceinline__ void stage_weight(unsigned char* dst, const float* __restrict__ W, int tid, int nthreads) {
  for (int i = tid; i < OUT * (IN / 8); i += nthreads) {
    const int o = i / (IN / 8), c8 = i % (IN / 8);
    const float4 v0 = ldg4(W + (size_t)o * IN + c8 * 8), v1 = ldg4(W + (size_t)o * IN + c8 * 8 + 4);
    const uint4 pk = make_uint4(pack_bf16x2(v0.x, v0.y), pack_bf16x2(v0.z, v0.w), pack_bf16x2(v1.x, v1.y), pack_bf16x2(v1.z, v1.w));
    *reinterpret_cast<uint4*>(dst + (c8 >> 3) * (OUT * 128) + tile_b_off(o, c8 & 7)) = pk;
  }
}

template <int KIN, int H, int PW>
__global__ void __launch_bounds__((kEpiWarps + 1 + PW) * 32, 1)
gin_fwd_bf16_kernel(GinFwdPair pp) {
  using L = FwdSmem<KIN, H>;
  constexpr int kThreadsF = (kEpiWarps + 1 + PW) * 32;
  constexpr int PT = PW * 32;
  constexpr int CH = H / 64;                                  // 32-column chunks per epilogue warp
  constexpr uint32_t kIdesc = idesc_bf16(TM, H, false, false);
  const bool second = (int)blockIdx.x >= pp.split;
  const GinFwdArgs& p = pp.a[second ? 1 : 0];
  const int bid = second ? (int)blockIdx.x - pp.split : (int)blockIdx.x;
  const int nblk = second ? (int)gridDim.x - pp.split : pp.split;
  const bf16_t* p_in = reinterpret_cast<const bf16_t*>(p.in);
  bf16_t* p_a = reinterpret_cast<bf16_t*>(p.a_out);
  bf16_t* p_r = reinterpret_cast<bf16_t*>(p.r_out);
  bf16_t* p_y = reinterpret_cast<bf16_t*>(p.y_out);
  extern __shared__ __align__(1024) unsigned char smem[];
  float* s_b1 = reinterpret_cast<float*>(smem + L::off_f);
  float* s_b2 = s_b1 + H;
  float* s_sc = s_b2 + H;
  float* s_sh = s_sc + H;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::off_bar);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + L::off_bar + B_COUNT * 8);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = (p.V + TM - 1) / TM;
  const int my_tiles = max(0, (n_tiles - bid + nblk - 1) / nblk);
  const bool rev = p.reverse != 0;
  auto tile_base = [&](int i) { return (bid + (rev ? my_tiles - 1 - i : i) * nblk) * TM; };

  if (threadIdx.x == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(&bars[B_FULL_A + s], PW);
      mbar_init(&bars[B_EMPTY_A + s], 1);
      mbar_init(&bars[B_D1 + s], 1);
      mbar_init(&bars[B_R + s], kEpiWarps * 32);
      mbar_init(&bars[B_D2 + s], 1);
      mbar_init(&bars[B_RAW + s], 1);
    }
  }
  if (warp == kMmaWarp) tmem_alloc(s_tmem, 4 * H);
  stage_weight<H, KIN>(smem + L::off_w1, p.W1, threadIdx.x, kThreadsF);
  stage_weight<H, H>(smem + L::off_w2, p.W2, threadIdx.x, kThreadsF);
  pdl_sync();      // everything above reads parameters only; from here on: the previous kernel's outputs (bn_in, activations)
  if (threadIdx.x < H) {
    const int c = threadIdx.x;
    s_b1[c] = p.b1[c]; s_b2[c] = p.b2[c];
    if (p.bn_in) {
      const float sc = p.bn_in[H + c] * p.bn_in[2 * H + c];
      s_sc[c] = sc; s_sh[c] = p.bn_in[3 * H + c] - p.bn_in[c] * sc;
    }
  }
  fence_smem_to_async();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *s_tmem;
  // TMEM columns of stage s (base 2H s): D1 [0, H) - overwritten in place by packed r: r columns [0, H/2) in TMEM columns
  // [0, H/4), r columns [H/2, H) in TMEM columns [H/2, 3H/4) (each epilogue warp packs inside the columns it has read);
  // D2 [H, 2H)

  double run_n = 0.0, run_mean[CH], run_m2[CH];
#pragma unroll
  for (int c = 0; c < CH; ++c) { run_mean[c] = 0.0; run_m2[c] = 0.0; }

  if (warp > kMmaWarp) {
    // =========================================================================== producers
    constexpr int LPR = KIN / 8, RPP = PT / LPR, NR = (TM + RPP - 1) / RPP;   // lanes per row (8 channels each), rows per pass
    const int pt = (warp - (kMmaWarp + 1)) * 32 + lane;
    const int gl = pt % LPR, gr = pt / LPR;
    int* s_ip = reinterpret_cast<int*>(smem + L::off_ip);
    int* s_self = reinterpret_cast<int*>(smem + L::off_self);
    int* s_ix = reinterpret_cast<int*>(smem + L::off_ix);
    const bool has_bn = (p.bn_in != nullptr);
    float sc[8], sh[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { sc[j] = has_bn ? s_sc[gl * 8 + j] : 1.f; sh[j] = has_bn ? s_sh[gl * 8 + j] : 0.f; }
    auto prod_sync = [&]() { asm volatile("bar.sync 1, %0;" :: "n"(PT) : "memory"); };
    auto raw_of = [&](int s) { return smem + L::off_stage + s * L::kStage; };
    auto win_start = [&](int i) { return max(0, tile_base(i) - HALO); };
    auto stage_indices = [&](int i, int e_begin, int e_end) {
      const int buf = i % kIdxBufs, base = tile_base(i), ws = win_start(i);
      for (int r = pt; r <= TM; r += PT) cp_async4(&s_ip[buf * (TM + 4) + r], p.indptr + min(base + r, p.V));
      if (p.row_map)
        for (int r = pt; r < WIN; r += PT) cp_async4(&s_self[buf * WIN + r], p.row_map + min(ws + r, p.V - 1));
      const int n = min(e_end - e_begin, L::kIdxCap);
      for (int e = pt; e < n; e += PT) cp_async4(&s_ix[buf * L::kIdxCap + e], p.indices + e_begin + e);
    };
    auto copy_window = [&](int i) {
      const int s = i & 1, buf = i % kIdxBufs, ws = win_start(i);
      const int wn = min(WIN, p.V - ws);
      unsigned char* raw = raw_of(s);
      if (pt == 0) mbar_arrive_expect_tx(&bars[B_RAW + s], (uint32_t)(wn * L::ROWB));
      if (p.row_map) {
        for (int r = pt; r < wn; r += PT)
          bulk_copy_g2s(raw + r * L::ROWB, p_in + (size_t)s_self[buf * WIN + r] * KIN, L::ROWB, &bars[B_RAW + s]);
      } else if (pt < 4) {
        const int r0 = pt * (WIN / 4), nr = min(WIN / 4, wn - r0);
        if (nr > 0) bulk_copy_g2s(raw + r0 * L::ROWB, p_in + (size_t)(ws + r0) * KIN, (uint32_t)(nr * L::ROWB), &bars[B_RAW + s]);
      }
    };
    auto bounds = [&](int i, int& e_begin, int& e_end) {
      const int base = tile_base(i);
      e_begin = __ldg(p.indptr + base); e_end = __ldg(p.indptr + min(base + TM, p.V));
    };
    int nb_begin = 0, nb_end = 0;
    if (my_tiles > 0) { bounds(0, nb_begin, nb_end); stage_indices(0, nb_begin, nb_end); }
    cp_async_commit();
    cp_async_wait_all();
    prod_sync();
    if (my_tiles > 0) copy_window(0);
    if (my_tiles > 1) { bounds(1, nb_begin, nb_end); stage_indices(1, nb_begin, nb_end); }
    cp_async_commit();
    if (my_tiles > 2) bounds(2, nb_begin, nb_end);
    for (int i = 0; i < my_tiles; ++i) {
      const int s = i & 1, use = i >> 1, buf = i % kIdxBufs;
      const int base = tile_base(i), ws = win_start(i);
      if (pt == 0) BF_TRACE(0, i);
      // [1] indices of tile i+1 and the window of tile i have landed
      cp_async_wait_all();
      mbar_wait(&bars[B_RAW + s], (uint32_t)(use & 1));
      prod_sync();
      if (pt == 0) BF_TRACE(1, i);
      // [2] one tile ahead: window of tile i+1 (its stage is free once GEMM1 of tile i-1 has read it), indices of tile i+2
      if (i + 1 < my_tiles) {
        if (i >= 1) mbar_wait(&bars[B_EMPTY_A + (s ^ 1)], (uint32_t)(((i - 1) >> 1) & 1));
        copy_window(i + 1);
      }
      if (i + 2 < my_tiles) stage_indices(i + 2, nb_begin, nb_end);
      cp_async_commit();
      if (i + 3 < my_tiles) bounds(i + 3, nb_begin, nb_end);
      if (pt == 0) BF_TRACE(2, i);
      // [3] a_v = f(h_v) + sum_u f(h_u), neighbours in CSR order, out of the raw window (fp32 accumulation)
      const int* ip = s_ip + buf * (TM + 4);
      const int* ix = s_ix + buf * L::kIdxCap;
      const unsigned char* raw = raw_of(s);
      const int e_begin = ip[0];
      float agg[NR][8];
      int e0[NR], deg[NR], maxd = 0;
#pragma unroll
      for (int j = 0; j < NR; ++j) {
        const int r = min(gr + j * RPP, TM - 1);
        const bool ok = gr + j * RPP < TM && base + r < p.V;
        e0[j] = ip[r] - e_begin;
        deg[j] = ok ? ip[r + 1] - ip[r] : 0;
        maxd = max(maxd, deg[j]);
#pragma unroll
        for (int q = 0; q < 8; ++q) agg[j][q] = 0.f;
        if (ok) {
          const uint4 h = *reinterpret_cast<const uint4*>(raw + (base - ws + r) * L::ROWB + gl * 16);
          if (has_bn) acc8<true>(agg[j], h, sc, sh); else acc8<false>(agg[j], h, sc, sh);
        }
      }
      for (int d = 0; d < maxd; ++d) {
#pragma unroll
        for (int j = 0; j < NR; ++j) {
          if (d < deg[j]) {
            const int e = e0[j] + d;
            const int u = (e < L::kIdxCap) ? ix[e] : __ldg(p.indices + e_begin + e);
            const int ul = u - ws;
            uint4 h;
            if ((unsigned)ul < (unsigned)WIN) h = *reinterpret_cast<const uint4*>(raw + ul * L::ROWB + gl * 16);
            else h = __ldg(reinterpret_cast<const uint4*>(p_in + (size_t)(p.row_map ? __ldg(p.row_map + u) : u) * KIN + gl * 8));
            if (has_bn) acc8<true>(agg[j], h, sc, sh); else acc8<false>(agg[j], h, sc, sh);
          }
        }
      }
      // [4] every producer has finished reading the raw window: overwrite the stage with the bf16 operand tile
      prod_sync();
      if (pt == 0) BF_TRACE(3, i);
      unsigned char* At = smem + L::off_stage + s * L::kStage;
#pragma unroll
      for (int j = 0; j < NR; ++j) {
        const int r = gr + j * RPP;
        if (r < TM) {
          const uint4 pk = make_uint4(pack_bf16x2(agg[j][0], agg[j][1]), pack_bf16x2(agg[j][2], agg[j][3]),
                                      pack_bf16x2(agg[j][4], agg[j][5]), pack_bf16x2(agg[j][6], agg[j][7]));
          if (p_a && base + r < p.V) stg16_cs(p_a + (size_t)(base + r) * KIN + gl * 8, pk);
          *reinterpret_cast<uint4*>(At + (gl >> 3) * (TM * 128) + tile_b_off(r, gl & 7)) = pk;
        }
      }
      fence_smem_to_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars[B_FULL_A + s]);
      if (pt == 0) BF_TRACE(4, i);
    }
    cp_async_wait_all();
  } else if (warp == kMmaWarp) {
    // =========================================================================== MMA issuer (converged warp, elected lane)
    const uint32_t w1 = smem_u32(smem + L::off_w1), w2 = smem_u32(smem + L::off_w2);
    auto gemm1 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      mbar_wait(&bars[B_FULL_A + s], (uint32_t)(use & 1));
      fence_after_sync();
      if (lane == 0) BF_TRACE(5, i);
      const uint32_t at = smem_u32(smem + L::off_stage + s * L::kStage);
      const uint32_t d = tmem + s * 2 * H;
#pragma unroll
      for (int k = 0; k < KIN / 16; ++k)
        mma_bf16_w(d, desc_b_kmajor(at + (k >> 2) * (TM * 128), k & 3), desc_b_kmajor(w1 + (k >> 2) * (H * 128), k & 3), kIdesc, k > 0);
      mma_commit_w(&bars[B_D1 + s]);
      mma_commit_w(&bars[B_EMPTY_A + s]);
    };
    auto gemm2 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      mbar_wait(&bars[B_R + s], (uint32_t)(use & 1));
      fence_after_sync();
      if (lane == 0) BF_TRACE(6, i);
      const uint32_t d = tmem + s * 2 * H + H;
      const uint32_t rb = tmem + s * 2 * H;
#pragma unroll
      for (int k = 0; k < H / 16; ++k) {
        const uint32_t ra = rb + (k < H / 32 ? 8 * k : H / 2 + 8 * (k - H / 32));
        mma_bf16_ta_w(d, ra, desc_b_kmajor(w2 + (k >> 2) * (H * 128), k & 3), kIdesc, k > 0);
      }
      mma_commit_w(&bars[B_D2 + s]);
    };
    if (my_tiles > 0) gemm1(0);
    for (int i = 0; i < my_tiles; ++i) {
      if (i + 1 < my_tiles) gemm1(i + 1);
      gemm2(i);
    }
  } else {
    // =========================================================================== epilogue
    // warp w: TMEM lane quarter w & 3 (rows 32 (w&3) ..), column half w >> 2 (columns (H/2)(w>>2) .., CH chunks of 32)
    const int q = warp & 3, half = warp >> 2;
    const int row = q * 32 + lane;
    const uint32_t tl = (uint32_t)(q * 32) << 16;
    auto epi1 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      const int gv = tile_base(i) + row;
      mbar_wait(&bars[B_D1 + s], (uint32_t)(use & 1));
      fence_after_sync();
      if (threadIdx.x == 0) BF_TRACE(7, i);
      const uint32_t t0 = tmem + s * 2 * H + tl;
      uint32_t pk[CH][16];
#pragma unroll
      for (int c = 0; c < CH; ++c) {
        const int c0 = half * (H / 2) + 32 * c;
        float v[32];
        tmem_ld16_nowait(t0 + c0, *reinterpret_cast<float (*)[16]>(v));
        tmem_ld16_nowait(t0 + c0 + 16, *reinterpret_cast<float (*)[16]>(v + 16));
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j)
          pk[c][j] = pack_bf16x2(fmaxf(v[2 * j] + s_b1[c0 + 2 * j], 0.f), fmaxf(v[2 * j + 1] + s_b1[c0 + 2 * j + 1], 0.f));
      }
      // all D1 columns of this warp have been read: pack r in place (TMEM columns half*(H/2) + 16 c ..)
#pragma unroll
      for (int c = 0; c < CH; ++c) {
        tmem_st16u(t0 + half * (H / 2) + 16 * c, pk[c]);
        if (p_r && gv < p.V) {
          bf16_t* dst = p_r + (size_t)gv * H + half * (H / 2) + 32 * c;
#pragma unroll
          for (int j = 0; j < 4; ++j) stg16_cs(dst + 8 * j, make_uint4(pk[c][4 * j], pk[c][4 * j + 1], pk[c][4 * j + 2], pk[c][4 * j + 3]));
        }
      }
      tmem_st_wait();
      fence_before_sync();
      mbar_arrive(&bars[B_R + s]);
      if (threadIdx.x == 0) BF_TRACE(8, i);
    };
    auto epi2 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      const int base = tile_base(i);
      const int gv = base + row;
      const bool valid = gv < p.V;
      const int cnt = max(0, min(32, p.V - (base + q * 32)));
      mbar_wait(&bars[B_D2 + s], (uint32_t)(use & 1));
      fence_after_sync();
      if (threadIdx.x == 0) BF_TRACE(9, i);
      double nt = run_n;
#pragma unroll
      for (int c = 0; c < CH; ++c) {
        const int c0 = half * (H / 2) + 32 * c;
        const uint32_t t0 = tmem + s * 2 * H + H + tl + c0;
        float y[32], t[32];
        tmem_ld16_nowait(t0, *reinterpret_cast<float (*)[16]>(y));
        tmem_ld16_nowait(t0 + 16, *reinterpret_cast<float (*)[16]>(y + 16));
        tmem_ld_wait();
        uint32_t pk[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          pk[j] = pack_bf16x2(y[2 * j] + s_b2[c0 + 2 * j], y[2 * j + 1] + s_b2[c0 + 2 * j + 1]);
          y[2 * j] = bf16_lo(pk[j]); y[2 * j + 1] = bf16_hi(pk[j]);       // statistics of what is stored
        }
        if (valid) {
          bf16_t* dst = p_y + (size_t)gv * H + c0;
#pragma unroll
          for (int j = 0; j < 4; ++j) stg16(dst + 8 * j, make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]));
        }
        if (cnt > 0) {
#pragma unroll
          for (int j = 0; j < 32; ++j) t[j] = valid ? y[j] : 0.f;
          const float mu = warp_colsum32(t, lane) / (float)cnt;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float d = y[j] - __shfl_sync(0xffffffffu, mu, j);
            t[j] = valid ? d * d : 0.f;
          }
          const float m2 = warp_colsum32(t, lane);
          const double nb = (double)cnt, dl = (double)mu - run_mean[c];
          nt = run_n + nb;
          run_m2[c] += (double)m2 + dl * dl * run_n * nb / nt;
          run_mean[c] += dl * nb / nt;
        }
      }
      run_n = nt;
      fence_before_sync();
      if (threadIdx.x == 0) BF_TRACE(10, i);
    };
    if (my_tiles > 0) epi1(0);
    for (int i = 0; i < my_tiles; ++i) {
      if (i + 1 < my_tiles) epi1(i + 1);
      epi2(i);
    }
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  if (warp == kMmaWarp) tmem_dealloc(tmem, 4 * H);
  // ---- CTA partial (n, mean, M2) per column (the stages are dead: scratch aliases them)
  constexpr int CW = H / 2;                                  // columns per epilogue warp
  double* s_stat = reinterpret_cast<double*>(smem);           // [8 warps][3][CW]
  double* s_comb = s_stat + kEpiWarps * 3 * CW;               // [4][3][H]
  if (warp < kEpiWarps) {
#pragma unroll
    for (int c = 0; c < CH; ++c) {
      s_stat[(warp * 3 + 0) * CW + 32 * c + lane] = run_n;
      s_stat[(warp * 3 + 1) * CW + 32 * c + lane] = run_mean[c];
      s_stat[(warp * 3 + 2) * CW + 32 * c + lane] = run_m2[c];
    }
  }
  __syncthreads();
  if (threadIdx.x < H) {
    const int c = threadIdx.x, half = c / CW, l = c % CW;
    double n = 0.0, mean = 0.0, m2 = 0.0;
    for (int q = 0; q < 4; ++q) {
      const int w = half * 4 + q;
      const double nb = s_stat[(w * 3 + 0) * CW + l];
      if (nb > 0.0) {
        const double mb = s_stat[(w * 3 + 1) * CW + l], qb = s_stat[(w * 3 + 2) * CW + l];
        const double nt = n + nb, dl = mb - mean;
        m2 += qb + dl * dl * n * nb / nt;
        mean += dl * nb / nt;
        n = nt;
      }
    }
    double* part = reinterpret_cast<double*>(p.part) + (size_t)bid * 3 * H;
    part[c] = n; part[H + c] = mean; part[2 * H + c] = m2;
  }
  if (!last_cta_arrives(p.counter, (unsigned)nblk)) return;
  {
    constexpr int SEGS = 4, BATCH = 8;
    const int c = threadIdx.x % H, seg = threadIdx.x / H;
    const double* part = reinterpret_cast<const double*>(p.part);
    if (seg < SEGS) {
      double n = 0.0, mean = 0.0, m2 = 0.0;
      for (int b0 = seg; b0 < nblk; b0 += SEGS * BATCH) {
        double pn[BATCH], pm[BATCH], pq[BATCH];
#pragma unroll
        for (int k = 0; k < BATCH; ++k) {
          const int b = b0 + k * SEGS;
          const bool ok = b < nblk;
          pn[k] = ok ? __ldcg(part + (size_t)b * 3 * H + c) : 0.0;
          pm[k] = ok ? __ldcg(part + (size_t)b * 3 * H + H + c) : 0.0;
          pq[k] = ok ? __ldcg(part + (size_t)b * 3 * H + 2 * H + c) : 0.0;
        }
#pragma unroll
        for (int k = 0; k < BATCH; ++k) {
          const double nt = n + pn[k], dl = pm[k] - mean, w = pn[k] / fmax(nt, 1.0);
          m2 += pq[k] + dl * dl * n * w;
          mean += dl * w;
          n = nt;
        }
      }
      s_comb[(seg * 3 + 0) * H + c] = n; s_comb[(seg * 3 + 1) * H + c] = mean; s_comb[(seg * 3 + 2) * H + c] = m2;
    }
    __syncthreads();
    if (threadIdx.x < H) {
      double n = 0.0, mean = 0.0, m2 = 0.0;
#pragma unroll
      for (int w4 = 0; w4 < SEGS; ++w4) {
        const double nb = s_comb[(w4 * 3 + 0) * H + c], mb = s_comb[(w4 * 3 + 1) * H + c], qb = s_comb[(w4 * 3 + 2) * H + c];
        const double nt = n + nb, dl = mb - mean, w = nb / fmax(nt, 1.0);
        m2 += qb + dl * dl * n * w;
        mean += dl * w;
        n = nt;
      }
      const double var = m2 / (double)p.V;
      p.bn_out[c] = (float)mean;
      p.bn_out[H + c] = (float)(1.0 / sqrt(var + (double)kBnEps));
      if (p.gamma) { p.bn_out[2 * H + c] = p.gamma[c]; p.bn_out[3 * H + c] = p.beta[c]; }
      if (p.running) {
        const double unb = p.V > 1 ? var * (double)p.V / (double)(p.V - 1) : var;
        p.running[c] = 0.9f * p.running[c] + 0.1f * (float)mean;
        p.running[H + c] = 0.9f * p.running[H + c] + 0.1f * (float)unb;
      }
    }
  }
}

}  // namespace bf

template <int KIN, int H>
static void launch_fwd_bf16(const GinFwdPair& pp, int grid, cudaStream_t s) {
  using L = bf::FwdSmem<KIN, H>;
  constexpr int PW = 16;
  static bool once = (cudaFuncSetAttribute(bf::gin_fwd_bf16_kernel<KIN, H, PW>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::total), true);
  (void)once;
  launch_k((bf::gin_fwd_bf16_kernel<KIN, H, PW>), dim3(grid), dim3((bf::kEpiWarps + 1 + PW) * 32), L::total, s, pp);
}

}  // namespace scgib
extern "C" __attribute__((visibility("default"))) int scgib_debug_bf16_trace(long long* host_out, int n) {
  return (int)cudaMemcpyFromSymbol(host_out, scgib::g_bf16_trace, (size_t)n * sizeof(long long));
}
namespace scgib {

size_t gin_fwd_bf16_part_floats(int hidden) { return (size_t)num_sms() * 3 * hidden * 2; }   // per-CTA (n, mean, M2) in fp64

// the same layer of both encoders in one launch (a1 == nullptr: one problem); in / a_out / r_out / y_out point to bf16 data
void launch_gin_fwd_bf16(const GinFwdArgs& a0, const GinFwdArgs* a1, int kin, int hidden, cudaStream_t s) {
  GinFwdPair pp;
  pp.a[0] = a0; pp.a[1] = a1 ? *a1 : a0;
  const int t0 = (a0.V + bf::TM - 1) / bf::TM, t1 = a1 ? (a1->V + bf::TM - 1) / bf::TM : 0;
  const int grid = min(t0 + t1, num_sms());
  pp.split = a1 ? pair_split(grid, t0, t1) : grid;
  static int dbg = -1;
  if (dbg < 0) { const char* e = getenv("SCGIB_DBG"); dbg = e ? atoi(e) : 0; }
  pp.a[0].dbg = pp.a[1].dbg = dbg;
  if (hidden == 64) {
    if (kin == 32) launch_fwd_bf16<32, 64>(pp, grid, s); else launch_fwd_bf16<64, 64>(pp, grid, s);
  } else {
    if (kin == 32) launch_fwd_bf16<32, 128>(pp, grid, s);
    else if (kin == 64) launch_fwd_bf16<64, 128>(pp, grid, s);      // layer 0 at d_transfer 64
    else launch_fwd_bf16<128, 128>(pp, grid, s);
  }
}

}  // namespace scgib
