// contrastive_tc.cu - the B x B similarity blocks of the contrastive loss on the 5th-generation tensor cores.
//
// reference: sim / batched_semi_loss, models.py:606-629:  refl = exp(z1 z1^T), between = exp(z1 z2^T), row sums.
//
// Operands are TWO-TERM FP16 SPLITS (kind::f16, fp32 accumulation): the normalised rows satisfy |z| <= 1, so
// z = hi + lo with hi = fp16(z), lo = fp16(z - hi) carries 22 significand bits (absolute error <= 2^-25 per element - the
// same 2^-22-class products as the 3xTF32 scheme used before) at HALF the bytes and with K = 16 per instruction:
//     S = A_hi B_hi^T + A_hi B_lo^T + A_lo B_hi^T        (three accumulating MMAs per K step, the lo x lo term is < 2^-24)
// A column block of z1 and z2 is stored as [z1 hi | z2 hi | z1 lo | z2 lo] (four [64][64] format-B tiles of umma.cuh, copied by
// cp.async straight from the pre-split rows graph_gate_fwd / normalize_kernel write), so ONE N = 128 MMA covers the refl and
// the between block at once: 12 MMAs per column block instead of 48.  The backward's weighted probabilities P (scaled by
// 2^k ~ B into fp16's normal range, un-scaled exactly at the end) are split the same way in registers and handed to the
// P Z GEMMs through TENSOR MEMORY (16-bit A operand: two K values per column), double-buffered.
// Roles: 8 worker warps (copies, exp / P epilogues, results) + ONE MMA-issuing warp; every hand-off is an mbarrier.
// Side jobs of other kernels ride along the forward as extra CTAs (ConFwdSides, kernels.cuh).
#include "kernels.cuh"
#include "umma.cuh"
#include "side_jobs.cuh"

namespace scgib {
using namespace umma;

constexpr int CI = 128;          // rows of z1 per CTA (UMMA M)
constexpr int CJ = 64;           // columns (rows of z1 / z2) per block
constexpr int ZI16 = CI * 128;   // one [128][64 fp16] format-B tile (16 KB)
constexpr int ZJ16 = CJ * 128;   // one [64][64 fp16] tile (8 KB)
constexpr int kStage16 = 4 * ZJ16;   // z1 hi | z2 hi | z1 lo | z2 lo
constexpr int kWorkers = 512;                // 16 worker warps: TMEM lane quarter (warp & 3) x 16-column chunk (warp >> 2)
constexpr int kConThreads = kWorkers + 32;   // + the MMA warp
constexpr int kMmaW = kWorkers / 32;
constexpr int kSideWarps = kThreads / 32;    // side-job bodies are written for kThreads threads

__host__ __device__ constexpr uint32_t idesc_f16c(int M, int N, bool a_mn, bool b_mn) {   // kind::f16, fp16 A / B, fp32 accumulate
  return (1u << 4) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
constexpr uint32_t kIdSim128 = idesc_f16c(CI, 2 * CJ, false, false), kIdSim64 = idesc_f16c(CI, CJ, false, false);
constexpr uint32_t kIdPV128 = idesc_f16c(CI, 2 * HID, false, true), kIdPV64 = idesc_f16c(CI, HID, false, true);

__device__ __forceinline__ void mma_f16c_w(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, bool acc) {
  if (elect_one()) mma_bf16(d, a, b, idesc, acc);                       // kind::f16; the operand formats are in idesc
}
__device__ __forceinline__ void mma_f16c_ta_w(uint32_t d, uint32_t a_tmem, uint64_t b, uint32_t idesc, bool acc) {
  if (elect_one()) mma_bf16_ta(d, a_tmem, b, idesc, acc);
}
__device__ __forceinline__ void tmem_st8u(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               :: "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}
__device__ __forceinline__ void tmem_st16u(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
      :: "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
         "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]) : "memory");
}

// rows [base, base+R) of a [B][64] fp16 matrix -> a format-B tile (16-byte chunks XOR-swizzled with row % 8); rows >= B zero-filled
template <int R>
__device__ __forceinline__ void cp_async_tile16(unsigned char* dst, const uint16_t* __restrict__ src, int base, int B) {
  for (int i = threadIdx.x; i < R * 8; i += kWorkers) {
    const int r = i >> 3, c8 = i & 7;
    const bool ok = base + r < B;
    cp_async16(dst + tile_b_off(r, c8), src + (size_t)(ok ? base + r : 0) * HID + c8 * 8, ok);
  }
}
__device__ __forceinline__ void worker_sync() { asm volatile("bar.sync 1, %0;" :: "n"(kWorkers) : "memory"); }

// ------------------------------------------------------------------------------------------------
// forward: row sums of exp(z1 z1^T) (diagonal excluded) + exp(z1 z2^T) over this CTA's column blocks
// ------------------------------------------------------------------------------------------------
struct ConTcLayout {
  static constexpr int off_zi = 0;                          // hi, lo
  static constexpr int off_zj = 2 * ZI16;                   // [2 stages][z1 hi | z2 hi | z1 lo | z2 lo]
  static constexpr int off_rs = off_zj + 2 * kStage16;      // float [4][128]
  static constexpr int off_bar = off_rs + 4 * CI * 4;       // tile[2], sim[2], free[2] + tmem slot
  static constexpr int total = off_bar + 64;
};
enum { CF_TILE = 0, CF_SIM = 2, CF_FREE = 4 };

// Grid: CTAs [0, iblocks * jsplit) are the similarity CTAs (row block b % iblocks, column split b / iblocks); the CTAs
// after them run the side jobs of ConFwdSides (recon_reduce, then compressor_ema); the CTA that finishes last runs
// loss_finalize when sd.finalize is set.
__device__ __forceinline__ void con_fwd_finish(const ConFwdSides& sd) {
  if (!sd.finalize) return;
  if (!last_cta_arrives(sd.counter)) return;
  loss_finalize_body<kThreads>(sd.fin);
}

__global__ void __launch_bounds__(kConThreads, 1)
contrastive_fwd_tc_kernel(ContrastiveFwdArgs p, ConFwdSides sd, int iblocks) {
  pdl_sync();
  using L = ConTcLayout;
  extern __shared__ __align__(1024) unsigned char smem[];
  const int nmain = iblocks * p.jsplit;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if ((int)blockIdx.x >= nmain) {
    const int side = (int)blockIdx.x - nmain;
    if (warp >= kSideWarps) return;        // the side bodies are written for kThreads threads (exited warps leave the CTA barriers)
    if (side < sd.n_reduce) recon_reduce_body(sd.rpart, sd.rgrid, sd.G, sd.edge, HID, side, sd.n_reduce);
    else compressor_ema_body<HID, kThreads>(sd.cstat, p.B, sd.running);
    con_fwd_finish(sd);
    return;
  }
  const int bx = (int)blockIdx.x % iblocks, by = (int)blockIdx.x / iblocks, gy = p.jsplit;
  unsigned char* zi = smem + L::off_zi;
  unsigned char* zj = smem + L::off_zj;
  float* s_rs = reinterpret_cast<float*>(smem + L::off_rs);
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(smem + L::off_bar);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + L::off_bar + 56);
  const size_t n = (size_t)p.B * HID;
  const uint16_t* zs = reinterpret_cast<const uint16_t*>(p.zsplit);
  const uint16_t *z1h = zs, *z1l = zs + n, *z2h = zs + 2 * n, *z2l = zs + 3 * n;
  const int ibase = bx * CI;
  const int jblocks = (p.B + CJ - 1) / CJ;
  const int nblk = (jblocks - by + gy - 1) / gy;   // blocks of this CTA
  auto jb_of = [&](int t) { return by + t * gy; };
  const bool is_mma = warp == kMmaW;

  if (is_mma) tmem_alloc(s_tmem, 256);
  if (threadIdx.x == 0) {
    for (int s = 0; s < 2; ++s) { mbar_init(&s_bar[CF_TILE + s], kMmaW); mbar_init(&s_bar[CF_SIM + s], 1); mbar_init(&s_bar[CF_FREE + s], kMmaW); }
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *s_tmem;

  if (is_mma) {
    const uint32_t zih = smem_u32(zi), zil = zih + ZI16;
    for (int t = 0; t < nblk; ++t) {
      const int s = t & 1, use = t >> 1;
      mbar_wait(&s_bar[CF_TILE + s], (uint32_t)(use & 1));
      if (use > 0) mbar_wait(&s_bar[CF_FREE + s], (uint32_t)((use - 1) & 1));      // the workers have read S set s of block t-2
      fence_after_sync();
      const uint32_t buf = smem_u32(zj + s * kStage16);
      const uint32_t d = tmem + s * 128;                  // columns [z1 z1_j^T | z1 z2_j^T]
#pragma unroll
      for (int k = 0; k < HID / 16; ++k) {
        const uint64_t ah = desc_b_kmajor(zih, k), al = desc_b_kmajor(zil, k);
        const uint64_t bh = desc_b_kmajor(buf, k), bl = desc_b_kmajor(buf + 2 * ZJ16, k);
        mma_f16c_w(d, ah, bh, kIdSim128, k > 0);
        mma_f16c_w(d, ah, bl, kIdSim128, true);
        mma_f16c_w(d, al, bh, kIdSim128, true);
      }
      mma_commit_w(&s_bar[CF_SIM + s]);
    }
  } else {
    auto load_j = [&](int t) {
      unsigned char* buf = zj + (t & 1) * kStage16;
      const int jbase = jb_of(t) * CJ;
      cp_async_tile16<CJ>(buf, z1h, jbase, p.B);
      cp_async_tile16<CJ>(buf + ZJ16, z2h, jbase, p.B);
      cp_async_tile16<CJ>(buf + 2 * ZJ16, z1l, jbase, p.B);
      cp_async_tile16<CJ>(buf + 3 * ZJ16, z2l, jbase, p.B);
    };
    auto tile_landed = [&](int t) {                      // this thread's copies of block t are complete and visible to the tensor core
      cp_async_commit();
      cp_async_wait_all();
      fence_smem_to_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s_bar[CF_TILE + (t & 1)]);         // one arrival per worker warp
    };
    cp_async_tile16<CI>(zi, z1h, ibase, p.B);
    cp_async_tile16<CI>(zi + ZI16, z1l, ibase, p.B);
    if (nblk > 0) { load_j(0); tile_landed(0); }
    if (nblk > 1) load_j(1);
    const int row = 32 * (warp & 3) + lane;              // UMMA M = 128: accumulator row = TMEM lane
    const int ccol = (warp >> 2) * 16;                   // this thread's 16 of the 64 columns
    const int gi = ibase + row;
    const uint32_t tl = (uint32_t)(32 * (warp & 3)) << 16;
    const bool rows_full = ibase + CI <= p.B;
    float rs = 0.f;
    for (int t = 0; t < nblk; ++t) {
      const int s = t & 1, use = t >> 1;
      if (t + 1 < nblk) tile_landed(t + 1);              // block t+1 (copied one iteration ago) -> the MMA warp
      mbar_wait(&s_bar[CF_SIM + s], (uint32_t)(use & 1));
      fence_after_sync();
      if (t + 2 < nblk) load_j(t + 2);                   // the similarity GEMMs of block t are done: its stage is free
      const int jbase = jb_of(t) * CJ;
      const uint32_t d = tmem + s * 128 + tl + ccol;
      float v[16], v2[16];
      tmem_ld16_nowait(d, v);                            // refl (z1 z1^T, diagonal excluded)
      tmem_ld16_nowait(d + 64, v2);                      // between
      tmem_ld_wait();
      fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s_bar[CF_FREE + s]);   // S set s may be overwritten by block t+2
      // |s| <= 1: ex2.approx is good to ~2e-7 relative.  Interior blocks (no row / column beyond B, no diagonal) skip the masks.
      const bool interior = rows_full && jbase + CJ <= p.B && (jbase + CJ <= ibase || jbase >= ibase + CI);
      if (interior) {
#pragma unroll
        for (int j = 0; j < 16; ++j) rs += __expf(v[j]) + __expf(v2[j]);
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int gj = jbase + ccol + j;
          rs += (gj < p.B && gj != gi) ? __expf(v[j]) : 0.f;
          rs += (gj < p.B) ? __expf(v2[j]) : 0.f;
        }
      }
    }
    cp_async_commit();
    cp_async_wait_all();
    s_rs[(warp >> 2) * CI + row] = rs;
    worker_sync();
    if (threadIdx.x < CI && ibase + threadIdx.x < p.B)
      p.rowsum[(size_t)by * p.B + ibase + threadIdx.x] = (s_rs[threadIdx.x] + s_rs[CI + threadIdx.x]) + (s_rs[2 * CI + threadIdx.x] + s_rs[3 * CI + threadIdx.x]);
  }
  fence_before_sync();
  __syncthreads();
  if (is_mma) tmem_dealloc(tmem, 256);
  con_fwd_finish(sd);
}

// ------------------------------------------------------------------------------------------------
// backward (same math as contrastive_bwd_kernel, loss_kernels.cu):
//   mode 0 (rows i of z1):  g1_i = sum_{j != i} e^{z1_i.z1_j} (1/D_i + 1/D_j) z1_j + sum_j e^{z1_i.z2_j}/D_i z2_j
//   mode 1 (rows j of z2):  g2_j = sum_i e^{z1_i.z2_j}/D_i z1_i
// Per 128-row block and 64-row column block: S = Zrow Zcol^T -> TMEM; the workers turn S into the weighted probabilities
// P' = pscale * P (exp, 1/D weights, masks), split P' into fp16 hi/lo and write it BACK to tensor memory, where it is the A
// operand of acc += P' Zcol (B = the same shared-memory column tiles read MN-major: [Z hi | Z lo] = one N = 128 MMA, plus
// P'_lo Z_hi).  P never touches shared memory and the B x B matrices never exist in HBM.
// TMEM: S set s at 128 s (S1 | S2), P buffer b at 256 + 64 b (hi 32 columns | lo 32 columns), acc 384 (hi part | lo part).
// ------------------------------------------------------------------------------------------------
constexpr int kColP = 256, kColAcc = 384;

struct ConBwdTcLayout {
  static constexpr int off_zi = 0;                            // hi, lo
  static constexpr int off_zj = 2 * ZI16;                     // [2 stages][z1 hi | z2 hi | z1 lo | z2 lo]
  static constexpr int off_di = off_zj + 2 * kStage16;        // float [128]
  static constexpr int off_dj = off_di + CI * 4;              // float [2][64]
  static constexpr int off_bar = off_dj + 2 * CJ * 4;         // tile[2], sim[2], p[2], pv[2] + tmem slot
  static constexpr int total = off_bar + 128;
};
enum { CB_TILE = 0, CB_SIM = 2, CB_P = 4, CB_PV = 6 };

__global__ void __launch_bounds__(kConThreads, 1)
contrastive_bwd_tc_kernel(ContrastiveBwdArgs p, const float* __restrict__ zsplit, int iblocks, float pscale) {
  pdl_sync();
  using L = ConBwdTcLayout;
  extern __shared__ __align__(1024) unsigned char smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int bx = (int)blockIdx.x % iblocks, by = (int)blockIdx.x / iblocks, gy = p.jsplit;
  unsigned char* zi = smem + L::off_zi;
  unsigned char* zj = smem + L::off_zj;
  float* s_di = reinterpret_cast<float*>(smem + L::off_di);
  float* s_dj = reinterpret_cast<float*>(smem + L::off_dj);
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(smem + L::off_bar);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + L::off_bar + 96);
  const size_t n = (size_t)p.B * HID;
  const uint16_t* zs = reinterpret_cast<const uint16_t*>(zsplit);
  const uint16_t *z1h = zs, *z1l = zs + n, *z2h = zs + 2 * n, *z2l = zs + 3 * n;
  const int ibase = bx * CI;
  const int jblocks = (p.B + CJ - 1) / CJ;
  const int nblk = (jblocks - by + gy - 1) / gy;
  auto jb_of = [&](int t) { return (by + t * gy) * CJ; };
  const bool is_mma = warp == kMmaW;

  if (is_mma) tmem_alloc(s_tmem, 512);
  if (threadIdx.x == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(&s_bar[CB_TILE + s], kMmaW); mbar_init(&s_bar[CB_SIM + s], 1);      // worker barriers: one arrival per warp
      mbar_init(&s_bar[CB_P + s], kMmaW); mbar_init(&s_bar[CB_PV + s], 1);
    }
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *s_tmem;

  if (is_mma) {
    // =========================================================================== MMA issuer (converged warp, elected lane)
    const uint32_t zih = smem_u32(zi), zil = zih + ZI16;
    int n_tile[2] = {0, 0}, n_p[2] = {0, 0}, round = 0;   // completed waits per barrier (phase bookkeeping); P rounds issued
    for (int mode = 0; mode < 2; ++mode) {
      const int nsrc = mode == 1 ? 1 : 2;
      auto issue_sim = [&](int t) {                      // similarity GEMMs of block t into S set t & 1
        const int s = t & 1;
        mbar_wait(&s_bar[CB_TILE + s], (uint32_t)(n_tile[s] & 1));
        ++n_tile[s];
        fence_after_sync();
        const uint32_t buf = smem_u32(zj + s * kStage16);
        const uint32_t d = tmem + s * 128;
#pragma unroll
        for (int k = 0; k < HID / 16; ++k) {
          const uint64_t ah = desc_b_kmajor(zih, k), al = desc_b_kmajor(zil, k);
          const uint64_t bh = desc_b_kmajor(buf, k), bl = desc_b_kmajor(buf + 2 * ZJ16, k);
          if (mode == 0) {                               // [z1 | z2] column tiles: refl and between in one N = 128 MMA
            mma_f16c_w(d, ah, bh, kIdSim128, k > 0);
            mma_f16c_w(d, ah, bl, kIdSim128, true);
            mma_f16c_w(d, al, bh, kIdSim128, true);
          } else {                                       // rows of z2 against the z1 column tile only
            mma_f16c_w(d, ah, bh, kIdSim64, k > 0);
            mma_f16c_w(d, ah, bl, kIdSim64, true);
            mma_f16c_w(d, al, bh, kIdSim64, true);
          }
        }
        mma_commit_w(&s_bar[CB_SIM + s]);
      };
      if (nblk > 0) issue_sim(0);
      int pv_in_mode = 0;
      for (int t = 0; t < nblk; ++t) {
        for (int q = 0; q < nsrc; ++q) {
          const int pb = round & 1;
          mbar_wait(&s_bar[CB_P + pb], (uint32_t)(n_p[pb] & 1));
          ++n_p[pb];
          fence_after_sync();
          // acc += P' Zcol for source q (0: z1 tiles, 1: z2 tiles) of block t; P' (hi | lo) is in tensor memory
          const uint32_t bh = smem_u32(zj + (t & 1) * kStage16) + q * ZJ16;     // hi tile; its lo tile is 2 * ZJ16 further
          const uint32_t ph = tmem + kColP + pb * 64, pl = ph + 32;
#pragma unroll
          for (int k = 0; k < CJ / 16; ++k) {
            const uint64_t b = desc_b_mnmajor(bh, 2 * ZJ16, k);
            mma_f16c_ta_w(tmem + kColAcc, ph + 8 * k, b, kIdPV128, !(pv_in_mode == 0 && k == 0));
            mma_f16c_ta_w(tmem + kColAcc, pl + 8 * k, b, kIdPV64, true);
          }
          mma_commit_w(&s_bar[CB_PV + pb]);
          ++pv_in_mode;
          ++round;
          // the similarity GEMMs of block t+1 queue BEHIND the first PV GEMM of block t (the tensor pipe is in order)
          if (q == 0 && t + 1 < nblk) issue_sim(t + 1);
        }
      }
    }
  } else {
    // =========================================================================== workers
    const int row = 32 * (warp & 3) + lane;              // TMEM lane = row of the 128-row block
    const int ccol = (warp >> 2) * 16;                   // this thread's 16 of the 64 columns
    const bool rows_full = ibase + CI <= p.B;
    const int gi = ibase + row;
    const uint32_t tl = (uint32_t)(32 * (warp & 3)) << 16;
    int n_sim[2] = {0, 0}, n_pv[2] = {0, 0}, round = 0;  // completed waits per barrier; P rounds handed over
    int last_pv_round = -1;                              // every PV GEMM up to this round has been observed complete
    auto wait_pv_upto = [&](int r) {                     // PV GEMMs of rounds <= r have completed (in-order tensor pipe)
      while (last_pv_round < r) {
        ++last_pv_round;
        const int pb = last_pv_round & 1;
        mbar_wait(&s_bar[CB_PV + pb], (uint32_t)(n_pv[pb] & 1));
        ++n_pv[pb];
      }
      fence_after_sync();
    };
    auto tile_landed = [&](int t) {                      // this thread's copies of tile t are complete and visible to the tensor core
      cp_async_commit();
      cp_async_wait_all();
      fence_smem_to_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s_bar[CB_TILE + (t & 1)]);
    };
    for (int mode = 0; mode < 2; ++mode) {
      const bool mode1 = (mode == 1);
      auto load_j = [&](int t) {
        unsigned char* buf = zj + (t & 1) * kStage16;
        const int jbase = jb_of(t);
        cp_async_tile16<CJ>(buf, z1h, jbase, p.B);
        cp_async_tile16<CJ>(buf + 2 * ZJ16, z1l, jbase, p.B);
        if (!mode1) {
          cp_async_tile16<CJ>(buf + ZJ16, z2h, jbase, p.B);
          cp_async_tile16<CJ>(buf + 3 * ZJ16, z2l, jbase, p.B);
        }
        if (threadIdx.x < CJ) s_dj[(t & 1) * CJ + threadIdx.x] = (jbase + threadIdx.x < p.B) ? pscale / __ldg(p.D + jbase + threadIdx.x) : 0.f;
      };
      // ---- prologue of the mode: row tile + two column blocks (every MMA of the previous mode has completed, see the end of the loop)
      cp_async_tile16<CI>(zi, mode1 ? z2h : z1h, ibase, p.B);
      cp_async_tile16<CI>(zi + ZI16, mode1 ? z2l : z1l, ibase, p.B);
      if (mode == 0 && threadIdx.x < CI) s_di[threadIdx.x] = (ibase + threadIdx.x < p.B) ? pscale / __ldg(p.D + ibase + threadIdx.x) : 0.f;
      if (nblk > 0) { load_j(0); tile_landed(0); }
      if (nblk > 1) load_j(1);
      worker_sync();                                     // s_di / s_dj (pscale / D) of the first blocks visible to all workers
      const float di = s_di[row];
      const int nsrc = mode1 ? 1 : 2;
      for (int t = 0; t < nblk; ++t) {
        // block t+1 has landed (copied one iteration ago): hand it to the MMA warp; make its 1/D_j visible to the workers
        if (t + 1 < nblk) tile_landed(t + 1);
        worker_sync();
        mbar_wait(&s_bar[CB_SIM + (t & 1)], (uint32_t)(n_sim[t & 1] & 1));      // similarities of block t are in tensor memory
        ++n_sim[t & 1];
        fence_after_sync();
        const int jbase = jb_of(t);
        const float* dj = s_dj + (t & 1) * CJ;
        const uint32_t sset = tmem + tl + (t & 1) * 128 + ccol;
        // interior blocks (no row / column beyond B, no diagonal entry) skip the masks
        const bool interior = rows_full && jbase + CJ <= p.B && (mode1 || jbase + CJ <= ibase || jbase >= ibase + CI);
        float djv[16];
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4) {
          const float4 t4 = ld4(dj + ccol + 4 * j4);
          djv[4 * j4] = t4.x; djv[4 * j4 + 1] = t4.y; djv[4 * j4 + 2] = t4.z; djv[4 * j4 + 3] = t4.w;
        }
        for (int q = 0; q < nsrc; ++q) {
          // one weighted-probability block: S (16 columns of this thread) -> P' hi/lo (fp16 pairs) in tensor memory
          const int kind = mode1 ? 2 : q;                // 0: refl (z1 z1), 1: between, 2: mode 1
          float v[16];
          tmem_ld16(sset + q * 64, v);
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float w = kind == 0 ? di + djv[j] : (kind == 1 ? di : djv[j]);
            v[j] = __expf(v[j]) * w;                      // |s| <= 1: ex2.approx is good to ~2e-7 relative
          }
          if (!interior) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const int gj = jbase + ccol + j;
              if (gj >= p.B || gi >= p.B || (kind == 0 && gj == gi)) v[j] = 0.f;
            }
          }
          uint32_t hi[8], lo[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) split_f16x2_plain(v[2 * j], v[2 * j + 1], hi[j], lo[j]);
          const int pb = round & 1;
          wait_pv_upto(round - 2);                         // the PV GEMM that last read P buffer pb has completed
          tmem_st8u(tmem + tl + kColP + pb * 64 + ccol / 2, hi);
          tmem_st8u(tmem + tl + kColP + pb * 64 + 32 + ccol / 2, lo);
          tmem_st_wait();
          fence_before_sync();
          __syncwarp();
          if (lane == 0) mbar_arrive(&s_bar[CB_P + pb]);
          ++round;
        }
        // stage t & 1 is free once the PV GEMMs of block t have completed: prefetch block t+2 into it
        if (t + 2 < nblk) { wait_pv_upto(round - 1); load_j(t + 2); }
      }
      // ---- result rows of this mode: acc = (columns 0..63 + columns 64..127) / pscale
      float* out = (mode1 ? p.g2p : p.g1p) + (size_t)by * p.B * HID;
      if (nblk > 0) {
        wait_pv_upto(round - 1);
        float a0[16], a1[16];
        tmem_ld16_nowait(tmem + tl + kColAcc + ccol, a0);
        tmem_ld16_nowait(tmem + tl + kColAcc + 64 + ccol, a1);
        tmem_ld_wait();
        const float inv = 1.f / pscale;
#pragma unroll
        for (int j = 0; j < 16; ++j) a0[j] = (a0[j] + a1[j]) * inv;
        if (gi < p.B) {
          st8(out + (size_t)gi * HID + ccol, a0);
          st8(out + (size_t)gi * HID + ccol + 8, a0 + 8);
        }
      } else if (gi < p.B) {
        const float z[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        st8(out + (size_t)gi * HID + ccol, z);
        st8(out + (size_t)gi * HID + ccol + 8, z);
      }
      // every MMA of this mode has completed (the last PV GEMM follows every similarity GEMM in the in-order tensor pipe) and
      // every worker has read its accumulator rows before the next mode's copies overwrite the tiles and its GEMMs the tensor memory
      fence_before_sync();
      worker_sync();
      fence_after_sync();
    }
    cp_async_commit();
    cp_async_wait_all();
  }
  fence_before_sync();
  __syncthreads();
  if (is_mma) tmem_dealloc(tmem, 512);
}

static float con_pscale(int B) {          // power of two >= B: P' = pscale * P is O(1), inside fp16's normal range
  float s = 1.f;
  while (s < (float)B && s < 16777216.f) s *= 2.f;
  return s;
}

void launch_contrastive_fwd_tc_sides(const ContrastiveFwdArgs& a, const ConFwdSides& sides, cudaStream_t s) {
  static bool once = (cudaFuncSetAttribute(contrastive_fwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           ConTcLayout::total), true);
  (void)once;
  const int iblocks = (a.B + CI - 1) / CI;
  const int grid = iblocks * a.jsplit + sides.n_reduce + sides.n_ema;
  launch_k((contrastive_fwd_tc_kernel), dim3(grid), dim3(kConThreads), ConTcLayout::total, s, a, sides, iblocks);
}
void launch_contrastive_fwd_tc(const ContrastiveFwdArgs& a, cudaStream_t s) { launch_contrastive_fwd_tc_sides(a, ConFwdSides{}, s); }

void launch_contrastive_bwd_tc(const ContrastiveBwdArgs& a, const float* zsplit, cudaStream_t s) {
  static bool once = (cudaFuncSetAttribute(contrastive_bwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           ConBwdTcLayout::total), true);
  (void)once;
  const int iblocks = (a.B + CI - 1) / CI;
  launch_k((contrastive_bwd_tc_kernel), dim3(iblocks * a.jsplit), dim3(kConThreads), ConBwdTcLayout::total, s, a, zsplit, iblocks,
           con_pscale(a.B));
}

}  // namespace scgib
