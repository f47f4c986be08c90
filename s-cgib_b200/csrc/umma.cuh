// umma.cuh - 5th-generation tensor-core (tcgen05) primitives for the 64-wide tile GEMMs of the S-CGIB path.
//
// All GEMM operands live in shared memory in ONE tile format ("format G", the no-swizzle / interleaved canonical
// layout of the UMMA shared-memory descriptors): a [R rows][C cols] fp32 tile is a grid of 8-row x 4-column core
// matrices of 128 contiguous bytes (row r of a core at byte 16*(r%8)); cores of one 8-row group are kCoreStride = 144
// bytes apart (the 16 bytes of padding spread the 16 chunks of a row over all banks), 8-row groups C/4 * 144 bytes.
// Format G is the K-major operand format (MN index = row, K index = col): D[row][n] += sum_col A[row][col] * B[n][col].
// Reductions over the tile ROWS (weight gradients) and natural-layout weights as B of the input-gradient GEMMs use
// MN-major operands, which for 32-bit types need format S below.
//
// fp32 parity: every product runs as 3xTF32 - hi = rna_tf32(v), lo = rna_tf32(v - hi);  D = hi*hi' + lo*hi' + hi*lo'
// with fp32 accumulation in tensor memory (error ~2^-21 per product).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace scgib {
namespace umma {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

constexpr int kCoreStride = 144;   // bytes between the 4-column cores of one 8-row group

// bytes of an [R][C] tile and of one 8-row group
__host__ __device__ constexpr int group_bytes(int C, int core = kCoreStride) { return (C / 4) * core; }
__host__ __device__ constexpr int tile_bytes(int R, int C, int core = kCoreStride) { return (R / 8) * group_bytes(C, core); }
// byte offset of the 16-byte chunk holding cols [4*c4, 4*c4+4) of `row` in a tile with C columns
__device__ __forceinline__ int tile_off4(int C, int row, int c4, int core = kCoreStride) {
  return (row >> 3) * group_bytes(C, core) + c4 * core + ((row & 7) << 4);
}

__device__ __forceinline__ float tf32_rna(float v) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return __uint_as_float(r);
}
__device__ __forceinline__ void split4(float4 v, float4& hi, float4& lo) {
  hi = make_float4(tf32_rna(v.x), tf32_rna(v.y), tf32_rna(v.z), tf32_rna(v.w));
  lo = make_float4(tf32_rna(v.x - hi.x), tf32_rna(v.y - hi.y), tf32_rna(v.z - hi.z), tf32_rna(v.w - hi.w));
}
// store 4 consecutive columns of a row into the hi and lo copies of a format-G tile with C columns
__device__ __forceinline__ void store_split4(unsigned char* hi_tile, unsigned char* lo_tile, int C, int row, int c4, float4 v,
                                             int core = kCoreStride) {
  float4 hi, lo;
  split4(v, hi, lo);
  const int off = tile_off4(C, row, c4, core);
  *reinterpret_cast<float4*>(hi_tile + off) = hi;
  *reinterpret_cast<float4*>(lo_tile + off) = lo;
}

// ---- shared-memory matrix descriptors (no swizzle, version 1 = Blackwell)
__device__ __forceinline__ uint64_t desc_base(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;   // descriptor version
  return d;
}

// instruction descriptor: kind::tf32, fp32 accumulate
__host__ __device__ constexpr uint32_t idesc_tf32(int M, int N, bool a_mn, bool b_mn) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void mma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, bool accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
      :: "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"((uint32_t)accumulate) : "memory");
}

// D[M][N] (+)= A * B over a K extent of `ksteps` * 8, as 3xTF32.
//   K-major view : LBO = core stride (the two 4-column cores of one K=8 step), SBO = 8-row group stride;
//                  a step advances two cores (288 B).
//   MN-major view: LBO = 8-row (= 8 K) group stride, SBO = core stride (4-column MN groups); a step advances one group.
// MN-major operands of 32-bit types need their own tile format ("format S": SWIZZLE_128B_BASE32B - measured: the
// no-swizzle and 16-byte-swizzled MN-major views yield zeros for kind::tf32).  An [R rows = K][64 cols = MN] tile is
// two column halves of [R][32 floats]; each row of a half is a 128-byte line whose 32-byte chunks are XOR-swizzled
// with (row % 4).  Descriptor: LBO = half stride (R*128), SBO = 512 (4-row groups); one K=8 step advances 1024 B.
__host__ __device__ constexpr int tile_s_bytes(int R) { return 2 * R * 128; }
__device__ __forceinline__ int tile_s_off4(int R, int row, int c4) {
  const int half = c4 >> 3, c = c4 & 7;
  return half * (R * 128) + row * 128 + ((((c >> 1) ^ (row & 3))) << 5) + ((c & 1) << 4);
}
__device__ __forceinline__ void store_split4_s(unsigned char* hi_tile, unsigned char* lo_tile, int R, int row, int c4, float4 v) {
  float4 hi, lo;
  split4(v, hi, lo);
  const int off = tile_s_off4(R, row, c4);
  *reinterpret_cast<float4*>(hi_tile + off) = hi;
  *reinterpret_cast<float4*>(lo_tile + off) = lo;
}

// D[M][N] (+)= A * B over a K extent of `ksteps` * 8, as 3xTF32.
//   K-major operand (format G): LBO = core stride (the two 4-column cores of one K=8 step), SBO = 8-row group stride;
//                               a step advances two cores (288 B).  `stride` = group_bytes(C).
//   MN-major operand (format S): `stride` = R*128 (half stride).
struct Operand {
  uint32_t hi, lo;       // shared-memory addresses of the hi / lo tiles
  bool mn;               // MN-major view (format S)?
  uint32_t stride;       // format G: 8-row group stride; format S: half stride
  uint32_t core;         // format G: core stride (kCoreStride for activation tiles, 128 for dense weight tiles)
  __device__ __forceinline__ uint64_t desc(uint32_t base, int step) const {
    if (mn) return desc_base(base + step * 1024, stride, 512) | ((uint64_t)1 << 61);   // SWIZZLE_128B_BASE32B
    return desc_base(base + step * 2 * core, core, stride);
  }
};
__device__ __forceinline__ void gemm_3xtf32(uint32_t d_tmem, const Operand& a, const Operand& b, int ksteps, uint32_t idesc,
                                            bool accumulate_first) {
  for (int s = 0; s < ksteps; ++s) {
    const uint64_t ah = a.desc(a.hi, s), al = a.desc(a.lo, s), bh = b.desc(b.hi, s), bl = b.desc(b.lo, s);
    mma_tf32(d_tmem, al, bh, idesc, accumulate_first || s > 0);   // small terms first
    mma_tf32(d_tmem, ah, bl, idesc, true);
    mma_tf32(d_tmem, ah, bh, idesc, true);
  }
}

// ---- tensor memory
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {   // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(smem_result)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {          // the same warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// generic-proxy smem writes -> visible to the tensor core (async proxy)
__device__ __forceinline__ void fence_smem_to_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// all previously issued MMAs of this thread arrive on `bar` when complete
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}\n"
      :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}

// 32 lanes x 16 consecutive columns: thread t of the warp gets lane (lane_base + t), columns col..col+15
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ uint32_t tmem_addr(uint32_t base, int lane, int col) { return base + ((uint32_t)lane << 16) + (uint32_t)col; }

// the same without the wait (issue several, then tmem_ld_wait once)
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// registers -> tensor memory: thread t of the warp writes lane (lane_base + t), columns col..col+15
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
      :: "r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
         "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])),
         "r"(__float_as_uint(v[7])), "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])),
         "r"(__float_as_uint(v[11])), "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])),
         "r"(__float_as_uint(v[15])) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// A operand in tensor memory (M = 128: accumulator-style layout, row = lane, K index = column; 8 columns per K step)
__device__ __forceinline__ void mma_tf32_ta(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, bool accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}\n"
      :: "r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"((uint32_t)accumulate) : "memory");
}

// Format-S tile ([halves of 32 columns][R rows][128 B], 32-byte chunks XOR-swizzled with row % 4) read as a K-MAJOR
// operand (MN index = tile row, K index = column): layout type SWIZZLE_128B_BASE32B, SBO = 512, LBO = half stride;
// K step s (8 columns = 32 B) starts at half s/4, byte 32*(s%4) of the row (measured on B200: tests/gpu_umma_probe2.py).
__device__ __forceinline__ uint64_t desc_s_kmajor(uint32_t tile, int R, int s) {
  return desc_base(tile + (uint32_t)(s >> 2) * (uint32_t)(R * 128) + (uint32_t)(s & 3) * 32u, (uint32_t)R * 128u, 512u) | ((uint64_t)1 << 61);
}
// dense format-G weight tile [n rows][C cols] (128-byte cores) as the K-major B operand, K step s
__device__ __forceinline__ uint64_t desc_g_dense(uint32_t tile, int C, int s) {
  return desc_base(tile + (uint32_t)s * 256u, 128u, (uint32_t)(C / 4) * 128u);
}

// one elected lane of a fully converged warp (the compiler then knows the MMA issue region is single-threaded)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\t"
      "elect.sync rx|px, 0xffffffff;\n\t"
      "@px mov.s32 %0, 1;\n\t}\n"
      : "+r"(pred));
  return pred != 0;
}

// MMA issue from a fully converged warp: every lane computes the (warp-uniform) descriptors, so they stay in uniform
// registers, and one elected lane issues.  Issuing from inside an `if (lane == 0)` region instead makes the compiler
// rebuild every descriptor in vector registers and move it to the uniform file per instruction (R2UR), which costs
// more than the ~54-cycle tcgen05.mma itself for the small N = 64, K = 8 MMAs of this path.
__device__ __forceinline__ void mma_tf32_w(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, bool accumulate) {
  if (elect_one()) mma_tf32(d_tmem, a_desc, b_desc, idesc, accumulate);
}
__device__ __forceinline__ void mma_tf32_ta_w(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, bool accumulate) {
  if (elect_one()) mma_tf32_ta(d_tmem, a_tmem, b_desc, idesc, accumulate);
}
__device__ __forceinline__ void mma_commit_w(uint64_t* bar) {
  if (elect_one()) mma_commit(bar);
}

// TMA bulk copy global -> shared (1-D, size a multiple of 16 bytes, 16-byte aligned addresses), completion on an mbarrier
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_copy_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               :: "r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}

// ------------------------------------------------------------------------------------------------
// bf16 operands (kind::f16, fp32 accumulation; K = 16 per instruction).  Tile format "B": a [R rows][64 bf16] block is
// R dense 128-byte rows whose 16-byte chunks are XOR-swizzled with (row % 8) (SWIZZLE_128B; block base 1024-byte
// aligned); wider tiles are column blocks of 64.  The same physical block is read
//   K-major  (MN index = row, K = column): SBO = 1024 (8-row groups), K step s starts 32*s bytes into the row;
//   MN-major (MN index = column, K = row): SBO = 1024 (8-row K groups), LBO = block stride (next 64 MN columns),
//                                          K step s (16 rows) starts at byte 2048*s.
// Pinned on B200 by tests/csrc/umma_probe_bf16.cu (tests/gpu_umma_probe_bf16.py).
// ------------------------------------------------------------------------------------------------
__host__ __device__ constexpr uint32_t idesc_bf16(int M, int N, bool a_mn, bool b_mn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void mma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, bool accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
      :: "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"((uint32_t)accumulate) : "memory");
}
__device__ __forceinline__ void mma_bf16_ta(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, bool accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
      :: "r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"((uint32_t)accumulate) : "memory");
}
__device__ __forceinline__ void mma_bf16_w(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, bool accumulate) {
  if (elect_one()) mma_bf16(d_tmem, a_desc, b_desc, idesc, accumulate);
}
constexpr uint64_t kSw128 = (uint64_t)2 << 61;
// byte offset of the 16-byte chunk c8 (8 bf16) of `row` inside a format-B block
__device__ __forceinline__ int tile_b_off(int row, int c8) { return row * 128 + ((c8 ^ (row & 7)) << 4); }
__device__ __forceinline__ uint64_t desc_b_kmajor(uint32_t block, int s) {          // K step s of one 64-column block
  return desc_base(block + (uint32_t)s * 32u, 16u, 1024u) | kSw128;
}
__device__ __forceinline__ uint64_t desc_b_mnmajor(uint32_t block, uint32_t block_stride, int s) {   // K step s = rows 16s..16s+15
  return desc_base(block + (uint32_t)s * 2048u, block_stride, 1024u) | kSw128;
}
// two fp32 -> packed bf16x2 (round to nearest even): lo half = a, hi half = b
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
__device__ __forceinline__ float bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t v) { return __uint_as_float(v & 0xffff0000u); }

}  // namespace umma
}  // namespace scgib
