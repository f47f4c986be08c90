// gin_tc3.cu - GIN layer forward, third-generation tcgen05 kernel: the gather runs out of SHARED MEMORY.
//
// Same contract as gin_fwd_kernel (gin_kernels.cu; reference models.py:66-72: DGL GINConv 'sum' + MLP + BatchNorm1d
// statistics) and the same tensor-core pipeline as gin_tc2.cu (3xTF32, N-stacked B operands, r handed to GEMM2 through
// tensor memory), but the producer no longer issues dependent global gathers.  Measured on B200 (role timeline of
// gin_tc2, tests/gpu_tc2_trace.py): a 128-row tile spent 6-9 us between the first index read and the last neighbour
// row arriving, against ~2 us of tensor-pipe and ~4 us of epilogue work - the gather latency bounded the kernel.
// Molecular batches are LOCAL: every neighbour of a row lives in the same graph (or ego-net), i.e. within a few rows
// of it, so almost every gathered row belongs to the tile itself.  Therefore:
//   * a WINDOW of 256 input rows - the tile's 128 rows plus a 64-row halo on either side - is copied by TMA
//     (cp.async.bulk: one bulk copy for a contiguous window, one per row through the ego row map for layer 0) into the
//     stage's 64 KB shared-memory buffer ONE TILE AHEAD, completion on an mbarrier: HBM latency hides behind a tile period;
//   * the CSR gather reads neighbour rows from that window (LDS, ~30 cycles); only neighbours further than the halo
//     (graphs larger than 64 nodes) fall back to a global load;
//   * after a producer barrier the aggregated rows overwrite the same buffer as tf32 hi/lo operand tiles.
// Roles: 8 epilogue warps (TMEM lane quarter x column half), 1 MMA warp, 8 producer warps; one CTA per SM,
// two stages; Encoder1 and Encoder2 rows share the launch (GinFwdPair).
#include <stdlib.h>
#include "kernels.cuh"
#include "umma.cuh"

namespace scgib {
using namespace umma;

// per-tile role timestamps (GinFwdArgs::dbg bit 1024; experiments only, tests/gpu_tc2_trace.py)
__device__ long long g_tc3_trace[160 * 16 * 12];
#define TC3_TRACE(ev, tile) do { if ((p.dbg & 1024) && (tile) < 16 && blockIdx.x < 160) g_tc3_trace[((size_t)blockIdx.x * 16 + (tile)) * 12 + (ev)] = clock64(); } while (0)

namespace tc3 {
constexpr int TM = 128;                       // rows per tile = UMMA M
constexpr int kEpiWarps = 8;
constexpr int kMmaWarp = kEpiWarps;
constexpr int kIdxCap = 1024;                 // staged neighbour indices per tile (more edges: read from global)
constexpr int kStageBytes = 2 * TM * HID * 4; // hi + lo tile of one stage (format S); first holds the raw row window
constexpr int HALO = 64, WIN = TM + 2 * HALO;  // window rows (WIN * 64 floats = the whole stage)
constexpr uint32_t kIdesc = idesc_tf32(TM, HID, false, false);
constexpr uint32_t kIdesc2 = idesc_tf32(TM, 2 * HID, false, false);
// TMEM columns of stage s (base + 256 s): D1 (128: hi*hi | hi*lo halves; overwritten in place by r_hi | r_lo) | D2 (128)
constexpr int kColD1 = 0, kColRhi = 0, kColRlo = 64, kColD2 = 128;
constexpr int kIdxBufs = 3;                   // index buffers: tile being gathered, tile being copied, tile being staged

template <int KIN>
struct Smem {
  static constexpr int W1B = HID * KIN * 4, W2B = HID * HID * 4;
  static constexpr int off_stage = 0;
  static constexpr int off_w1_hi = 2 * kStageBytes, off_w1_lo = off_w1_hi + W1B;
  static constexpr int off_w2_hi = off_w1_lo + W1B, off_w2_lo = off_w2_hi + W2B;
  static constexpr int off_f = off_w2_lo + W2B;                       // b1[64] b2[64] bn_in[4][64]
  static constexpr int off_stat = off_f + 6 * HID * 4;                // double [8 warps][3][32]
  static constexpr int off_bar = off_stat + kEpiWarps * 3 * 32 * 8;   // 10 mbarriers + tmem slot
  static constexpr int off_ip = off_bar + 128;                        // int [3][TM + 4]   indptr slice of the tile
  static constexpr int off_self = off_ip + kIdxBufs * (TM + 4) * 4;   // int [3][WIN]      mapped rows of the window (layer 0 of Encoder2)
  static constexpr int off_ix = off_self + kIdxBufs * WIN * 4;        // int [3][kIdxCap]  neighbour rows (unmapped)
  static constexpr int total = off_ix + kIdxBufs * kIdxCap * 4;
  static_assert(total <= 227 * 1024, "shared memory budget");
};

enum { B_FULL_A = 0, B_EMPTY_A = 2, B_D1 = 4, B_R = 6, B_D2 = 8, B_RAW = 10, B_COUNT = 12 };

// column sums of a [32 rows (lanes)][32 columns (registers)] block by a transpose-reduce: lane l returns column l
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
// non-blocking test of an mbarrier phase (true: the phase with this parity has completed)
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
               : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}

template <int KIN, int PW>
__global__ void __launch_bounds__((kEpiWarps + 1 + PW) * 32, 1)
gin_fwd_tc3_kernel(GinFwdPair pp) {
  using L = Smem<KIN>;
  constexpr int kThreads3 = (kEpiWarps + 1 + PW) * 32;
  constexpr int PT = PW * 32;                                 // producer threads
  const bool second = (int)blockIdx.x >= pp.split;
  const GinFwdArgs& p = pp.a[second ? 1 : 0];
  const int bid = second ? (int)blockIdx.x - pp.split : (int)blockIdx.x;          // CTA index / count inside its problem
  const int nblk = second ? (int)gridDim.x - pp.split : pp.split;
  extern __shared__ __align__(1024) unsigned char smem[];
  float* s_b1 = reinterpret_cast<float*>(smem + L::off_f);
  float* s_b2 = s_b1 + HID;
  float* s_bn = s_b2 + HID;                                   // {mean, rstd, gamma, beta}[HID] of the producing layer
  double* s_stat = reinterpret_cast<double*>(smem + L::off_stat);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::off_bar);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + L::off_bar + B_COUNT * 8);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = (p.V + TM - 1) / TM;
  const int my_tiles = (n_tiles - bid + nblk - 1) / nblk;     // tiles bid + i*nblk
  const bool rev = p.reverse != 0;
  auto tile_base = [&](int i) { return (bid + (rev ? my_tiles - 1 - i : i) * nblk) * TM; };

  // ---- one-time setup: barriers, TMEM, weights (natural [out][in] = K-major B operand, dense cores), biases
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
  if (warp == kMmaWarp) tmem_alloc(s_tmem, 512);
  for (int i = threadIdx.x; i < HID * (KIN / 4); i += kThreads3) {
    const int o = i / (KIN / 4), c4 = i % (KIN / 4);
    store_split4(smem + L::off_w1_hi, smem + L::off_w1_lo, KIN, o, c4, ldg4(p.W1 + (size_t)o * KIN + c4 * 4), 128);
  }
  for (int i = threadIdx.x; i < HID * (HID / 4); i += kThreads3) {
    const int o = i / (HID / 4), c4 = i % (HID / 4);
    store_split4(smem + L::off_w2_hi, smem + L::off_w2_lo, HID, o, c4, ldg4(p.W2 + (size_t)o * HID + c4 * 4), 128);
  }
  if (threadIdx.x < HID) { s_b1[threadIdx.x] = p.b1[threadIdx.x]; s_b2[threadIdx.x] = p.b2[threadIdx.x]; }
  pdl_sync();      // everything above reads parameters only; from here on: the previous kernel's outputs (bn_in, activations)
  if (p.bn_in && threadIdx.x < 4 * HID) s_bn[threadIdx.x] = p.bn_in[threadIdx.x];
  fence_smem_to_async();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *s_tmem;

  if (warp > kMmaWarp) {
    // =========================================================================== producers
    // A lane owns EIGHT channels of a row (two float4: channel quads gl and gl + LPR, so that the 8 lanes of a row read 128
    // contiguous bytes per load - no bank conflicts): the per-row index work of the gather (edge range, neighbour index, window
    // offset, halo test) - most of the loop's instructions in the ncu source profile - is replicated in 8 instead of 16 lanes
    constexpr int LPR = KIN / 8, RPP = PT / LPR, NR = (TM + RPP - 1) / RPP;   // lanes per row, rows per pass, passes (last one guarded)
    const int pt = (warp - (kMmaWarp + 1)) * 32 + lane;
    const int gl = pt % LPR, gr = pt / LPR;
    int* s_ip = reinterpret_cast<int*>(smem + L::off_ip);
    int* s_self = reinterpret_cast<int*>(smem + L::off_self);
    int* s_ix = reinterpret_cast<int*>(smem + L::off_ix);
    const bool has_bn = (p.bn_in != nullptr);
    // relu(BN(y)) = max((y - mean) * (rstd * gamma) + beta, 0) for this lane's two channel quads
    float4 mu[2], sc[2], be[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      mu[h] = make4(0.f); sc[h] = make4(1.f); be[h] = make4(0.f);
      if (has_bn) {
        const int c = (gl + LPR * h) * 4;
        const float4 rs = ld4(s_bn + HID + c), ga = ld4(s_bn + 2 * HID + c);
        mu[h] = ld4(s_bn + c); be[h] = ld4(s_bn + 3 * HID + c);
        sc[h] = make_float4(rs.x * ga.x, rs.y * ga.y, rs.z * ga.z, rs.w * ga.w);
      }
    }
    auto act = [&](float4 y, int h) {
      if (!has_bn) return y;
      return make_float4(fmaxf(fmaf(y.x - mu[h].x, sc[h].x, be[h].x), 0.f), fmaxf(fmaf(y.y - mu[h].y, sc[h].y, be[h].y), 0.f),
                         fmaxf(fmaf(y.z - mu[h].z, sc[h].z, be[h].z), 0.f), fmaxf(fmaf(y.w - mu[h].w, sc[h].w, be[h].w), 0.f));
    };
    auto prod_sync = [&]() { asm volatile("bar.sync 1, %0;" :: "n"(PT) : "memory"); };
    // raw window of stage s: plain row-major [WIN][KIN] at the start of the stage
    auto raw_of = [&](int s) { return reinterpret_cast<float*>(smem + L::off_stage + s * kStageBytes); };
    auto win_start = [&](int i) { return max(0, tile_base(i) - HALO); };
    // indptr slice, mapped window rows and (unmapped) neighbour rows of tile i -> index buffer i % 3 (cp.async)
    auto stage_indices = [&](int i, int e_begin, int e_end) {
      const int buf = i % kIdxBufs, base = tile_base(i), ws = win_start(i);
      for (int r = pt; r <= TM; r += PT) cp_async4(&s_ip[buf * (TM + 4) + r], p.indptr + min(base + r, p.V));
      if (p.row_map)
        for (int r = pt; r < WIN; r += PT) cp_async4(&s_self[buf * WIN + r], p.row_map + min(ws + r, p.V - 1));
      const int n = min(e_end - e_begin, kIdxCap);
      for (int e = pt; e < n; e += PT) cp_async4(&s_ix[buf * kIdxCap + e], p.indices + e_begin + e);
    };
    // the window of tile i -> its stage, by TMA bulk copies completing on B_RAW (rows >= V are never referenced)
    auto copy_window = [&](int i) {
      const int s = i & 1, buf = i % kIdxBufs, ws = win_start(i);
      const int wn = min(WIN, p.V - ws);
      float* raw = raw_of(s);
      if (pt == 0) mbar_arrive_expect_tx(&bars[B_RAW + s], (uint32_t)(wn * KIN * 4));
      if (p.row_map) {
        for (int r = pt; r < wn; r += PT)
          bulk_copy_g2s(raw + r * KIN, p.in + (size_t)s_self[buf * WIN + r] * KIN, KIN * 4, &bars[B_RAW + s]);
      } else if (pt < 4) {                                      // contiguous window: 4 bulk copies of up to 64 rows
        const int r0 = pt * (WIN / 4), nr = min(WIN / 4, wn - r0);
        if (nr > 0) bulk_copy_g2s(raw + r0 * KIN, p.in + (size_t)(ws + r0) * KIN, (uint32_t)(nr * KIN * 4), &bars[B_RAW + s]);
      }
    };
    auto bounds = [&](int i, int& e_begin, int& e_end) {
      const int base = tile_base(i);
      e_begin = __ldg(p.indptr + base); e_end = __ldg(p.indptr + min(base + TM, p.V));
    };
    // ---- prologue: indices of tiles 0 and 1, window of tile 0, index range of tile 2
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
      if (pt == 0) TC3_TRACE(0, i);
      // ---- [1] indices of tile i+1 (cp.async group of the previous iteration) and the window of tile i have landed
      cp_async_wait_all();
      mbar_wait(&bars[B_RAW + s], (uint32_t)(use & 1));
      prod_sync();
      if (pt == 0) TC3_TRACE(1, i);
      // ---- [2] one tile ahead: window of tile i+1 into the other stage (free once GEMM1 of tile i-1 has read it; its
      //          mapped row ids arrived with the group above), indices of tile i+2, index range of tile i+3.
      //          GEMM1 of tile i-1 was issued only when the previous iteration ended, so the stage is normally NOT free yet:
      //          waiting here cost ~1 us of every ~5.5 us tile period (role timeline).  If it is not free, the copy is issued
      //          after the gather of this tile instead, and the window is pulled into L2 meanwhile so that the late copy is short.
      bool window_issued = i + 1 >= my_tiles;
      if (!window_issued) {
        if (i < 1 || mbar_test(&bars[B_EMPTY_A + (s ^ 1)], (uint32_t)(((i - 1) >> 1) & 1))) { copy_window(i + 1); window_issued = true; }
        else if (!p.row_map) {
          const int ws1 = win_start(i + 1), wn1 = min(WIN, p.V - ws1);
          for (int l = pt; l < wn1 * (KIN / 32); l += PT) prefetch_l2(p.in + (size_t)ws1 * KIN + (size_t)l * 32);
        }
      }
      if (i + 2 < my_tiles) stage_indices(i + 2, nb_begin, nb_end);
      cp_async_commit();
      if (i + 3 < my_tiles) bounds(i + 3, nb_begin, nb_end);
      if (pt == 0) TC3_TRACE(2, i);
      // ---- [3] a_v = f(h_v) + sum_u f(h_u), neighbours in CSR order, out of the raw window
      const int* ip = s_ip + buf * (TM + 4);
      const int* ix = s_ix + buf * kIdxCap;
      const float* raw = raw_of(s);
      const int e_begin = ip[0];
      float4 agg[NR][2];
      int e0[NR], deg[NR], maxd = 0;
#pragma unroll
      for (int j = 0; j < NR; ++j) {
        const int r = min(gr + j * RPP, TM - 1);
        const bool ok = gr + j * RPP < TM && base + r < p.V;
        e0[j] = ip[r] - e_begin;
        deg[j] = ok ? ip[r + 1] - ip[r] : 0;
        maxd = max(maxd, deg[j]);
        const float* src = raw + (base - ws + r) * KIN + gl * 4;
        agg[j][0] = ok ? act(ld4(src), 0) : make4(0.f);
        agg[j][1] = ok ? act(ld4(src + LPR * 4), 1) : make4(0.f);
      }
      for (int d = 0; d < maxd; ++d) {
#pragma unroll
        for (int j = 0; j < NR; ++j) {
          if (d < deg[j]) {
            const int e = e0[j] + d;
            const int u = (e < kIdxCap) ? ix[e] : __ldg(p.indices + e_begin + e);
            const int ul = u - ws;
            const float* src = (unsigned)ul < (unsigned)WIN ? raw + ul * KIN + gl * 4
                                                            : p.in + (size_t)(p.row_map ? __ldg(p.row_map + u) : u) * KIN + gl * 4;   // beyond the halo: global
            agg[j][0] = add4(agg[j][0], act(ld4(src), 0));
            agg[j][1] = add4(agg[j][1], act(ld4(src + LPR * 4), 1));
          }
        }
      }
      if (!window_issued) {                                     // (block-uniform) the deferred window copy: GEMM1 of tile i-1 is long done
        mbar_wait(&bars[B_EMPTY_A + (s ^ 1)], (uint32_t)(((i - 1) >> 1) & 1));
        copy_window(i + 1);
      }
      // ---- [4] every producer has finished reading the raw window: overwrite the stage with the hi/lo operand tiles
      prod_sync();
      if (pt == 0) TC3_TRACE(3, i);
      unsigned char* hi = smem + L::off_stage + s * kStageBytes;
      unsigned char* lo = hi + TM * KIN * 4;
#pragma unroll
      for (int j = 0; j < NR; ++j) {
        const int r = gr + j * RPP;
        if (r < TM) {
          if (p.a_out && base + r < p.V) {
            st4_cs(p.a_out + (size_t)(base + r) * KIN + gl * 4, agg[j][0]);
            st4_cs(p.a_out + (size_t)(base + r) * KIN + (gl + LPR) * 4, agg[j][1]);
          }
          store_split4_s(hi, lo, TM, r, gl, agg[j][0]);
          store_split4_s(hi, lo, TM, r, gl + LPR, agg[j][1]);
        }
      }
      fence_smem_to_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars[B_FULL_A + s]);
      if (pt == 0) TC3_TRACE(4, i);
      (void)use;
    }
    cp_async_wait_all();
  } else if (warp == kMmaWarp) {
    // =========================================================================== MMA issuer
    {   // the whole warp runs the loop (uniform descriptors); one elected lane issues each instruction
      const uint32_t w1h = smem_u32(smem + L::off_w1_hi), w2h = smem_u32(smem + L::off_w2_hi);
      static_assert(L::off_w1_lo == L::off_w1_hi + L::W1B && L::off_w2_lo == L::off_w2_hi + L::W2B, "hi/lo weight tiles must be adjacent");
      auto gemm1 = [&](int i) {
        const int s = i & 1, use = i >> 1;
        mbar_wait(&bars[B_FULL_A + s], (uint32_t)(use & 1));
        fence_after_sync();
        if (lane == 0) TC3_TRACE(5, i);
        const uint32_t ah = smem_u32(smem + L::off_stage + s * kStageBytes), al = ah + TM * KIN * 4;
        const uint32_t d = tmem + s * 256 + kColD1;
#pragma unroll
        for (int k = 0; k < KIN / 8; ++k) {
          const uint64_t dah = desc_s_kmajor(ah, TM, k), dal = desc_s_kmajor(al, TM, k);
          const uint64_t dbh = desc_g_dense(w1h, KIN, k);   // hi tile; the N = 128 view continues into the lo tile
          mma_tf32_w(d, dah, dbh, kIdesc2, k > 0);
          mma_tf32_w(d, dal, dbh, kIdesc, true);
        }
        mma_commit_w(&bars[B_D1 + s]);
        mma_commit_w(&bars[B_EMPTY_A + s]);
      };
      auto gemm2 = [&](int i) {
        const int s = i & 1, use = i >> 1;
        mbar_wait(&bars[B_R + s], (uint32_t)(use & 1));
        fence_after_sync();
        if (lane == 0) TC3_TRACE(6, i);
        const uint32_t d = tmem + s * 256 + kColD2;
        const uint32_t rh = tmem + s * 256 + kColRhi, rl = tmem + s * 256 + kColRlo;
#pragma unroll
        for (int k = 0; k < HID / 8; ++k) {
          const uint64_t dbh = desc_g_dense(w2h, HID, k);
          mma_tf32_ta_w(d, rh + 8 * k, dbh, kIdesc2, k > 0);
          mma_tf32_ta_w(d, rl + 8 * k, dbh, kIdesc, true);
        }
        mma_commit_w(&bars[B_D2 + s]);
      };
      // GEMM2(i) is issued as soon as its r is ready; GEMM1 runs up to two tiles ahead
      if (my_tiles > 0) gemm1(0);
      for (int i = 0; i < my_tiles; ++i) {
        if (i + 1 < my_tiles) gemm1(i + 1);
        gemm2(i);
      }
    }
  } else {
    // =========================================================================== epilogue
    // warp w: TMEM lane quarter w & 3 (rows 32 (w&3) ..), column half w >> 2 (columns 32 (w>>2) ..)
    const int q = warp & 3, half = warp >> 2;
    const int row = q * 32 + lane;
    const int c0 = half * 32;
    const uint32_t tl = (uint32_t)(q * 32) << 16;
    double run_n = 0.0, run_mean = 0.0, run_m2 = 0.0;         // column c0 + lane over this warp's rows
    auto epi1 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      const int gv = tile_base(i) + row;
      mbar_wait(&bars[B_D1 + s], (uint32_t)(use & 1));
      fence_after_sync();
      if (threadIdx.x == 0) TC3_TRACE(7, i);
      const uint32_t t0 = tmem + s * 256 + tl;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        float v[16], v2[16], hi[16], lo[16];
        tmem_ld16_nowait(t0 + kColD1 + c0 + 16 * c, v);
        tmem_ld16_nowait(t0 + kColD1 + HID + c0 + 16 * c, v2);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          v[j] = fmaxf((v[j] + v2[j]) + s_b1[c0 + 16 * c + j], 0.f);
          hi[j] = tf32_rna(v[j]);
          lo[j] = tf32_rna(v[j] - hi[j]);
        }
        tmem_st16(t0 + kColRhi + c0 + 16 * c, hi);          // in place: these columns have just been read by this thread
        tmem_st16(t0 + kColRlo + c0 + 16 * c, lo);
        if (p.r_out && gv < p.V) {
          st8_cs(p.r_out + (size_t)gv * HID + c0 + 16 * c, v);
          st8_cs(p.r_out + (size_t)gv * HID + c0 + 16 * c + 8, v + 8);
        }
      }
      tmem_st_wait();
      fence_before_sync();
      mbar_arrive(&bars[B_R + s]);
      if (threadIdx.x == 0) TC3_TRACE(8, i);
    };
    auto epi2 = [&](int i) {
      const int s = i & 1, use = i >> 1;
      const int base = tile_base(i);
      const int gv = base + row;
      const bool valid = gv < p.V;
      const int cnt = max(0, min(32, p.V - (base + q * 32)));   // valid rows of this warp (warp-uniform)
      mbar_wait(&bars[B_D2 + s], (uint32_t)(use & 1));
      fence_after_sync();
      if (threadIdx.x == 0) TC3_TRACE(9, i);
      const uint32_t t0 = tmem + s * 256 + tl + kColD2 + c0;
      float y[32], t[32];
      tmem_ld16_nowait(t0, *reinterpret_cast<float (*)[16]>(y));
      tmem_ld16_nowait(t0 + 16, *reinterpret_cast<float (*)[16]>(y + 16));
      tmem_ld16_nowait(t0 + HID, *reinterpret_cast<float (*)[16]>(t));
      tmem_ld16_nowait(t0 + HID + 16, *reinterpret_cast<float (*)[16]>(t + 16));
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; ++j) y[j] = (y[j] + t[j]) + s_b2[c0 + j];
      if (valid) {
#pragma unroll
        for (int j = 0; j < 4; ++j) st8(p.y_out + (size_t)gv * HID + c0 + 8 * j, y + 8 * j);
      }
      // statistics of this warp's rows: column mean, then centred M2 (two transpose-reduces; lane l <-> column c0 + l)
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
        const double nb = (double)cnt, nt = run_n + nb, dl = (double)mu - run_mean;   // Chan update of the running triple
        run_m2 += (double)m2 + dl * dl * run_n * nb / nt;
        run_mean += dl * nb / nt;
        run_n = nt;
      }
      fence_before_sync();   // TMEM reads of this stage are complete before GEMM2 of its next user (ordered through B_R)
      if (threadIdx.x == 0) TC3_TRACE(10, i);
    };
    if (my_tiles > 0) epi1(0);
    for (int i = 0; i < my_tiles; ++i) {
      if (i + 1 < my_tiles) epi1(i + 1);
      epi2(i);
    }
    s_stat[(warp * 3 + 0) * 32 + lane] = run_n;
    s_stat[(warp * 3 + 1) * 32 + lane] = run_mean;
    s_stat[(warp * 3 + 2) * 32 + lane] = run_m2;
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  if (warp == kMmaWarp) tmem_dealloc(tmem, 512);
  // ---- CTA partial (n, mean, M2) per column: Chan combine of the 4 row-quarter warps of the column's half in fp64
  if (threadIdx.x < HID) {
    const int c = threadIdx.x, half = c >> 5, l = c & 31;
    double n = 0.0, mean = 0.0, m2 = 0.0;
    for (int q = 0; q < 4; ++q) {
      const int w = half * 4 + q;
      const double nb = s_stat[(w * 3 + 0) * 32 + l];
      if (nb > 0.0) {
        const double mb = s_stat[(w * 3 + 1) * 32 + l], qb = s_stat[(w * 3 + 2) * 32 + l];
        const double nt = n + nb, dl = mb - mean;
        m2 += qb + dl * dl * n * nb / nt;
        mean += dl * nb / nt;
        n = nt;
      }
    }
    double* part = reinterpret_cast<double*>(p.part) + (size_t)bid * 3 * HID;
    part[c] = n; part[HID + c] = mean; part[2 * HID + c] = m2;
  }
  if (!last_cta_arrives(p.counter, (unsigned)nblk)) return;
  // ---- batch statistics: the last CTA of the problem combines the per-CTA partials in fp64.  Thread (c, seg) first LOADS
  //      a batch of partials (independent loads), then Chan-combines them in a fixed order; 4 segments, then a serial 4-way.
  {
    constexpr int SEGS = 4, BATCH = 8;
    const int c = threadIdx.x & (HID - 1), seg = threadIdx.x >> 6;
    const double* part = reinterpret_cast<const double*>(p.part);
    double* s_comb = reinterpret_cast<double*>(smem);        // [SEGS][3][HID] (the stages are dead by now)
    if (seg < SEGS) {
      double n = 0.0, mean = 0.0, m2 = 0.0;
      for (int b0 = seg; b0 < nblk; b0 += SEGS * BATCH) {
        double pn[BATCH], pm[BATCH], pq[BATCH];
#pragma unroll
        for (int k = 0; k < BATCH; ++k) {
          const int b = b0 + k * SEGS;
          const bool ok = b < nblk;
          pn[k] = ok ? __ldcg(part + (size_t)b * 3 * HID + c) : 0.0;
          pm[k] = ok ? __ldcg(part + (size_t)b * 3 * HID + HID + c) : 0.0;
          pq[k] = ok ? __ldcg(part + (size_t)b * 3 * HID + 2 * HID + c) : 0.0;
        }
#pragma unroll
        for (int k = 0; k < BATCH; ++k) {
          const double nt = n + pn[k], dl = pm[k] - mean, w = pn[k] / fmax(nt, 1.0);
          m2 += pq[k] + dl * dl * n * w;
          mean += dl * w;
          n = nt;
        }
      }
      s_comb[(seg * 3 + 0) * HID + c] = n; s_comb[(seg * 3 + 1) * HID + c] = mean; s_comb[(seg * 3 + 2) * HID + c] = m2;
    }
    __syncthreads();
    if (threadIdx.x < HID) {
      double n = 0.0, mean = 0.0, m2 = 0.0;
#pragma unroll
      for (int w4 = 0; w4 < SEGS; ++w4) {
        const double nb = s_comb[(w4 * 3 + 0) * HID + c], mb = s_comb[(w4 * 3 + 1) * HID + c], qb = s_comb[(w4 * 3 + 2) * HID + c];
        const double nt = n + nb, dl = mb - mean, w = nb / fmax(nt, 1.0);
        m2 += qb + dl * dl * n * w;
        mean += dl * w;
        n = nt;
      }
      const double var = m2 / (double)p.V;
      p.bn_out[c] = (float)mean;
      p.bn_out[HID + c] = (float)(1.0 / sqrt(var + (double)kBnEps));
      if (p.gamma) { p.bn_out[2 * HID + c] = p.gamma[c]; p.bn_out[3 * HID + c] = p.beta[c]; }
      if (p.running) {
        const double unb = p.V > 1 ? var * (double)p.V / (double)(p.V - 1) : var;
        p.running[c] = 0.9f * p.running[c] + 0.1f * (float)mean;
        p.running[HID + c] = 0.9f * p.running[HID + c] + 0.1f * (float)unb;
      }
    }
  }
}

}  // namespace tc3

template <int KIN, int PW>
static void launch_tc3_pw(const GinFwdPair& pp, int grid, cudaStream_t s) {
  using L = tc3::Smem<KIN>;
  static bool once = (cudaFuncSetAttribute(tc3::gin_fwd_tc3_kernel<KIN, PW>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::total), true);
  (void)once;
  launch_k((tc3::gin_fwd_tc3_kernel<KIN, PW>), dim3(grid), dim3((tc3::kEpiWarps + 1 + PW) * 32), L::total, s, pp);
}
template <int KIN>
static void launch_tc3(const GinFwdPair& pp, int grid, cudaStream_t s) {
  static int pw = -1;                     // producer warps: SCGIB_TC3_PW = 8 | 12 | 16 (default) | 20
  if (pw < 0) { const char* e = getenv("SCGIB_TC3_PW"); pw = e ? atoi(e) : 16; }
  if (pw == 20) launch_tc3_pw<KIN, 20>(pp, grid, s);
  else if (pw == 16) launch_tc3_pw<KIN, 16>(pp, grid, s);
  else if (pw == 12) launch_tc3_pw<KIN, 12>(pp, grid, s);
  else launch_tc3_pw<KIN, 8>(pp, grid, s);
}

}  // namespace scgib
extern "C" __attribute__((visibility("default"))) int scgib_debug_tc2_trace(long long* host_out, int n) {
  return (int)cudaMemcpyFromSymbol(host_out, scgib::g_tc3_trace, (size_t)n * sizeof(long long));
}
namespace scgib {

static int dbg_mask3() {
  static int dbg = -1;
  if (dbg < 0) { const char* e = getenv("SCGIB_DBG"); dbg = e ? atoi(e) : 0; }
  return dbg;
}

void launch_gin_fwd_tc3(const GinFwdArgs& a, int kin, cudaStream_t s) {
  GinFwdPair pp;
  pp.a[0] = a; pp.a[1] = a;
  const int grid = min((a.V + tc3::TM - 1) / tc3::TM, num_sms());
  pp.split = grid;                                   // single problem: every CTA works on a[0]
  if (kin == 32) launch_tc3<32>(pp, grid, s); else launch_tc3<HID>(pp, grid, s);
}

// the same layer of both encoders in one launch (separate part / counter / bn_out buffers per problem)
void launch_gin_fwd_tc3_pair(const GinFwdArgs& a0, const GinFwdArgs& a1, int kin, cudaStream_t s) {
  GinFwdPair pp;
  pp.a[0] = a0; pp.a[1] = a1;
  const int t0 = (a0.V + tc3::TM - 1) / tc3::TM, t1 = (a1.V + tc3::TM - 1) / tc3::TM;
  const int grid = min(t0 + t1, num_sms());
  pp.split = pair_split(grid, t0, t1);
  pp.a[0].dbg = pp.a[1].dbg = dbg_mask3();
  if (kin == 32) launch_tc3<32>(pp, grid, s); else launch_tc3<HID>(pp, grid, s);
}

}  // namespace scgib
