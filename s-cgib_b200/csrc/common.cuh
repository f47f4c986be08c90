// common.cuh - shared device helpers for the S-CGIB sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace scgib {

constexpr int HID = 64;        // hidden width (exp_pretraining.py:390)
// d_transfer (exp_pretraining.py:378, the layer-0 input width of the encoders): 32, 64 or 128 and at most hidden.  Tensor-core
// tiles are built from 32-column lines and the gin_fwd_tc3 stage holds windows of at most 64 columns.
constexpr int kMaxTransfer = 128;
__host__ __device__ constexpr bool transfer_width_ok(int d, int hidden) { return (d == 32 || d == 64 || d == 128) && d <= hidden; }
constexpr int kThreads = 256;  // CTA size of every tile kernel
constexpr int kMaxInDim = 128; // widest raw node-feature input (transfer_d, s2s_rev on the H = 128 Set2Set instance)
constexpr int kMaxClasses = 1024;   // widest fine-tuning head output (C; 2 * kMaxInDim for r_transfer_d)
constexpr float kBnEps = 1e-5f;
typedef uint16_t bf16_t;       // raw bfloat16 storage (bf16 mode: activations of the GIN encoders)

// Programmatic dependent launch (PDL): a kernel launched with launch_k() below may be scheduled while its predecessor in
// the stream is still running; it must not touch anything the predecessor writes before pdl_wait() returns (the
// predecessor grid has then completed and its memory is visible).  pdl_trigger() lets the NEXT kernel in the stream be
// scheduled; it is always issued after this kernel's own pdl_wait(), so a kernel's pre-wait section only ever overlaps its
// immediate predecessor.  Without a programmatic dependency both are no-ops.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_sync() { pdl_wait(); pdl_trigger(); }

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
// 256-bit global accesses (sm_100+): one full 32-byte sector per thread - used where a thread owns a whole row
__device__ __forceinline__ void st8(float* p, const float* v) {
  asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" :: "l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]),
               "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]) : "memory");
}
__device__ __forceinline__ void ld8(const float* p, float* v) {
  asm volatile("ld.global.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]),
               "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]) : "l"(p));
}
// streaming variants (L2 evict-first): tensors saved for the backward pass / read exactly once must not push the next
// layer's gather source out of L2
__device__ __forceinline__ void st8_cs(float* p, const float* v) {
  asm volatile("st.global.cs.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" :: "l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]),
               "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]) : "memory");
}
__device__ __forceinline__ void st4_cs(float* p, float4 v) { __stcs(reinterpret_cast<float4*>(p), v); }
__device__ __forceinline__ float4 ld4_cs(const float* p) { return __ldcs(reinterpret_cast<const float4*>(p)); }
// 4 consecutive channels of an activation row stored as fp32 or (bf16 mode) bf16: `p` is the tensor base, idx the element index
template <bool BF>
__device__ __forceinline__ float4 ld4a(const float* p, size_t idx) {
  if (BF) {
    const uint2 w = *reinterpret_cast<const uint2*>(reinterpret_cast<const bf16_t*>(p) + idx);
    return make_float4(__uint_as_float(w.x << 16), __uint_as_float(w.x & 0xffff0000u), __uint_as_float(w.y << 16),
                       __uint_as_float(w.y & 0xffff0000u));
  }
  return *reinterpret_cast<const float4*>(p + idx);
}
template <bool BF>
__device__ __forceinline__ void st4a(float* p, size_t idx, float4 v) {
  if (BF) {
    uint2 w;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(w.x) : "f"(v.y), "f"(v.x));
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(w.y) : "f"(v.w), "f"(v.z));
    *reinterpret_cast<uint2*>(reinterpret_cast<bf16_t*>(p) + idx) = w;
  } else {
    *reinterpret_cast<float4*>(p + idx) = v;
  }
}
__device__ __forceinline__ float4 make4(float a) { return make_float4(a, a, a, a); }
__device__ __forceinline__ float4 add4(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ float4 relu4(float4 a) {
  return make_float4(fmaxf(a.x, 0.f), fmaxf(a.y, 0.f), fmaxf(a.z, 0.f), fmaxf(a.w, 0.f));
}

// (a, b) -> packed fp16 pairs of the two-term split v = hi + lo: hi = fp16(v), lo = fp16(v - hi) (UNSCALED residual: for
// |v| <= 1 its absolute error is <= 2^-25, the fp16 subnormal spacing / 2); element a in the low 16 bits
__device__ __forceinline__ void split_f16x2_plain(float a, float b, uint32_t& hi, uint32_t& lo) {
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(b), "f"(a));
  float ha, hb;
  asm("{\n\t.reg .b16 l, h;\n\tmov.b32 {l, h}, %2;\n\tcvt.f32.f16 %0, l;\n\tcvt.f32.f16 %1, h;\n\t}" : "=f"(ha), "=f"(hb) : "r"(hi));
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(b - hb), "f"(a - ha));
}

// the same with the residual SCALED by 2^11: lo' = fp16((v - hi) * 2048) stays in fp16's normal range whenever hi does, so
// hi + 2^-11 lo' carries 22 significand bits for every magnitude (products with lo' land in separate accumulator columns
// and are scaled back by 2^-11 in the epilogue)
__device__ __forceinline__ void split_f16x2_s11(float a, float b, uint32_t& hi, uint32_t& lo) {
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(b), "f"(a));
  float ha, hb;
  asm("{\n\t.reg .b16 l, h;\n\tmov.b32 {l, h}, %2;\n\tcvt.f32.f16 %0, l;\n\tcvt.f32.f16 %1, h;\n\t}" : "=f"(ha), "=f"(hb) : "r"(hi));
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"((b - hb) * 2048.f), "f"((a - ha) * 2048.f));
}

// relu(BN(y)) for 4 consecutive channels: ((y - mean) * rstd) * gamma + beta
struct Bn4 {
  float4 mean, rstd, gamma, beta;
  __device__ __forceinline__ void load(const float* bn, int c, int H = HID) {  // bn = {mean[H], rstd[H], gamma[H], beta[H]}
    mean = ldg4(bn + c); rstd = ldg4(bn + H + c); gamma = ldg4(bn + 2 * H + c); beta = ldg4(bn + 3 * H + c);
  }
  __device__ __forceinline__ float4 xhat(float4 y) const {
    return make_float4((y.x - mean.x) * rstd.x, (y.y - mean.y) * rstd.y, (y.z - mean.z) * rstd.z, (y.w - mean.w) * rstd.w);
  }
  __device__ __forceinline__ float4 pre(float4 y) const {  // BN output before the ReLU
    float4 h = xhat(y);
    return make_float4(fmaf(h.x, gamma.x, beta.x), fmaf(h.y, gamma.y, beta.y), fmaf(h.z, gamma.z, beta.z), fmaf(h.w, gamma.w, beta.w));
  }
  __device__ __forceinline__ float4 act(float4 y) const { return relu4(pre(y)); }
};

// GIN aggregation a_v = f(in[map(v)]) + sum_{u in N(v)} f(in[map(u)]) for NR rows at once per thread (lane `gl` owns
// 4 channels).  The gather is latency-bound, not bandwidth-bound (degree ~2, 256-byte rows), so it is organised for
// memory-level parallelism: every dependent stage (indptr -> indices -> [row_map] -> feature rows) is issued for all
// NR rows and for TWO neighbour slots at once before anything is consumed.  Neighbours are added in CSR order.
// SELF = false: the neighbour sum alone (A Z of the reconstruction loss)
template <int KIN, int NR, bool SELF = true>
__device__ __forceinline__ void gather_aggregate(const float* __restrict__ in, const int32_t* __restrict__ row_map,
                                                 const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                                 int V, const int (&v)[NR], int gl, const Bn4* bn, float4 (&acc)[NR]) {
  int e0[NR], deg[NR], sv[NR];
#pragma unroll
  for (int j = 0; j < NR; ++j) {
    const bool ok = v[j] < V;
    e0[j] = ok ? __ldg(indptr + v[j]) : 0;
    deg[j] = ok ? __ldg(indptr + v[j] + 1) : 0;
    sv[j] = (ok && row_map) ? __ldg(row_map + v[j]) : v[j];
  }
  int maxd = 0;
#pragma unroll
  for (int j = 0; j < NR; ++j) { deg[j] -= e0[j]; maxd = max(maxd, deg[j]); }
  int u0[NR], u1[NR];
#pragma unroll
  for (int j = 0; j < NR; ++j) {
    u0[j] = deg[j] > 0 ? __ldg(indices + e0[j]) : -1;
    u1[j] = deg[j] > 1 ? __ldg(indices + e0[j] + 1) : -1;
  }
  float4 hs[NR];
#pragma unroll
  for (int j = 0; j < NR; ++j) hs[j] = (SELF && v[j] < V) ? ld4(in + (size_t)sv[j] * KIN + gl * 4) : make4(0.f);
  if (row_map) {
#pragma unroll
    for (int j = 0; j < NR; ++j) {
      if (u0[j] >= 0) u0[j] = __ldg(row_map + u0[j]);
      if (u1[j] >= 0) u1[j] = __ldg(row_map + u1[j]);
    }
  }
  float4 h0[NR], h1[NR];
#pragma unroll
  for (int j = 0; j < NR; ++j) {
    h0[j] = u0[j] >= 0 ? ld4(in + (size_t)u0[j] * KIN + gl * 4) : make4(0.f);
    h1[j] = u1[j] >= 0 ? ld4(in + (size_t)u1[j] * KIN + gl * 4) : make4(0.f);
  }
#pragma unroll
  for (int j = 0; j < NR; ++j) {
    acc[j] = make4(0.f);
    if (SELF && v[j] < V) acc[j] = bn ? bn->act(hs[j]) : hs[j];
    if (u0[j] >= 0) acc[j] = add4(acc[j], bn ? bn->act(h0[j]) : h0[j]);
    if (u1[j] >= 0) acc[j] = add4(acc[j], bn ? bn->act(h1[j]) : h1[j]);
  }
  for (int d = 2; d < maxd; d += 2) {                    // rows with more than two neighbours
#pragma unroll
    for (int j = 0; j < NR; ++j) {
      u0[j] = deg[j] > d ? __ldg(indices + e0[j] + d) : -1;
      u1[j] = deg[j] > d + 1 ? __ldg(indices + e0[j] + d + 1) : -1;
    }
    if (row_map) {
#pragma unroll
      for (int j = 0; j < NR; ++j) {
        if (u0[j] >= 0) u0[j] = __ldg(row_map + u0[j]);
        if (u1[j] >= 0) u1[j] = __ldg(row_map + u1[j]);
      }
    }
#pragma unroll
    for (int j = 0; j < NR; ++j) {
      h0[j] = u0[j] >= 0 ? ld4(in + (size_t)u0[j] * KIN + gl * 4) : make4(0.f);
      h1[j] = u1[j] >= 0 ? ld4(in + (size_t)u1[j] * KIN + gl * 4) : make4(0.f);
    }
#pragma unroll
    for (int j = 0; j < NR; ++j) {
      if (u0[j] >= 0) acc[j] = add4(acc[j], bn ? bn->act(h0[j]) : h0[j]);
      if (u1[j] >= 0) acc[j] = add4(acc[j], bn ? bn->act(h1[j]) : h1[j]);
    }
  }
}

// Deterministic sum of `n` per-CTA partials part[b * stride] (b = start, start + step, ...) in fp64, fixed order.  The
// loads are independent of the adds, so the unrolled loop keeps several in flight (a hand-batched variant with an
// explicit array of loads measured slower on B200).
__device__ __forceinline__ double sum_partials(const float* part, size_t stride, int n, int start, int step) {
  // four interleaved chains: 32 independent L2 loads in flight instead of 8 (the chain of round trips is the whole cost
  // of a last-CTA finalise); combined as (s0 + s1) + (s2 + s3)
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  int b = start;
#pragma unroll 8
  for (; b + 3 * step < n; b += 4 * step) {
    s0 += (double)__ldcg(part + (size_t)b * stride);
    s1 += (double)__ldcg(part + (size_t)(b + step) * stride);
    s2 += (double)__ldcg(part + (size_t)(b + 2 * step) * stride);
    s3 += (double)__ldcg(part + (size_t)(b + 3 * step) * stride);
  }
  for (; b < n; b += step) s0 += (double)__ldcg(part + (size_t)b * stride);
  return (s0 + s1) + (s2 + s3);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ------------------------------------------------------------------------------------------------
// "last CTA finalises" pattern: every CTA publishes its partials, the last one to arrive reduces
// them in a fixed order (deterministic, no float atomics) and resets the counter for the next launch.
// ------------------------------------------------------------------------------------------------
// (`ncta` = number of CTAs working on this problem: a launch may carry two independent problems, see GinFwdPair)
__device__ __forceinline__ bool last_cta_arrives(unsigned int* counter, unsigned int ncta) {
  __shared__ bool is_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int prev = atomicAdd(counter, 1u);
    is_last = (prev == ncta - 1);
    if (is_last) *counter = 0u;
  }
  __syncthreads();
  if (is_last) __threadfence();
  return is_last;
}
__device__ __forceinline__ bool last_cta_arrives(unsigned int* counter) { return last_cta_arrives(counter, gridDim.x); }

// ------------------------------------------------------------------------------------------------
// Register-tiled FP32 tile GEMMs out of shared memory (256 threads).
//   gemm_nn : C[TILE_M][N] += A[TILE_M][K] (row-major, lda) * B[K][N] (k-major, ldb)
//             thread (tr, tc): rows tr*TM..+TM, cols tc*4..+4 ; TM = TILE_M*N/1024
//   gemm_tn : C[NX][NY]   += X[rows][NX]^T * Y[rows][NY]    (reduction over the tile rows)
//             thread (ti, tj) of a 16x16 arrangement: ti*TO..+TO of NX, tj*TJ..+TJ of NY
// ------------------------------------------------------------------------------------------------
template <int TILE_M, int N>
struct NNMap {
  static constexpr int CG = N / 4;
  static constexpr int RG = kThreads / CG;
  static constexpr int TM = TILE_M / RG;
  static_assert(TM >= 1 && TM * RG == TILE_M, "bad tile");
  __device__ static __forceinline__ int tc() { return threadIdx.x % CG; }
  __device__ static __forceinline__ int tr() { return threadIdx.x / CG; }
  __device__ static __forceinline__ int row0() { return tr() * TM; }
  __device__ static __forceinline__ int col0() { return tc() * 4; }
};

template <int TILE_M, int K, int N>
__device__ __forceinline__ void gemm_nn(const float* __restrict__ As, int lda, const float* __restrict__ Bs, int ldb,
                                        float (&acc)[NNMap<TILE_M, N>::TM][4]) {
  using M = NNMap<TILE_M, N>;
  const float* a0 = As + M::row0() * lda;
  const float* b0 = Bs + M::col0();
#pragma unroll 2
  for (int k = 0; k < K; k += 4) {
    float4 b[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) b[i] = ld4(b0 + (k + i) * ldb);
#pragma unroll
    for (int m = 0; m < M::TM; ++m) {
      const float4 a = ld4(a0 + m * lda + k);
      acc[m][0] = fmaf(a.x, b[0].x, acc[m][0]); acc[m][1] = fmaf(a.x, b[0].y, acc[m][1]);
      acc[m][2] = fmaf(a.x, b[0].z, acc[m][2]); acc[m][3] = fmaf(a.x, b[0].w, acc[m][3]);
      acc[m][0] = fmaf(a.y, b[1].x, acc[m][0]); acc[m][1] = fmaf(a.y, b[1].y, acc[m][1]);
      acc[m][2] = fmaf(a.y, b[1].z, acc[m][2]); acc[m][3] = fmaf(a.y, b[1].w, acc[m][3]);
      acc[m][0] = fmaf(a.z, b[2].x, acc[m][0]); acc[m][1] = fmaf(a.z, b[2].y, acc[m][1]);
      acc[m][2] = fmaf(a.z, b[2].z, acc[m][2]); acc[m][3] = fmaf(a.z, b[2].w, acc[m][3]);
      acc[m][0] = fmaf(a.w, b[3].x, acc[m][0]); acc[m][1] = fmaf(a.w, b[3].y, acc[m][1]);
      acc[m][2] = fmaf(a.w, b[3].z, acc[m][2]); acc[m][3] = fmaf(a.w, b[3].w, acc[m][3]);
    }
  }
}

template <int NX, int NY>
struct TNMap {
  static constexpr int TO = NX / 16;
  static constexpr int TJ = NY / 16;
  static_assert(TO >= 1 && TJ >= 1 && TO % 2 == 0 && TJ % 2 == 0, "bad tn tile");
  __device__ static __forceinline__ int ti() { return threadIdx.x / 16; }
  __device__ static __forceinline__ int tj() { return threadIdx.x % 16; }
  __device__ static __forceinline__ int o0() { return ti() * TO; }
  __device__ static __forceinline__ int j0() { return tj() * TJ; }
};

template <int NX, int NY>
__device__ __forceinline__ void gemm_tn(const float* __restrict__ Xs, int ldx, const float* __restrict__ Ys, int ldy,
                                        int rows, float (&acc)[TNMap<NX, NY>::TO][TNMap<NX, NY>::TJ]) {
  using M = TNMap<NX, NY>;
  const float* x0 = Xs + M::o0();
  const float* y0 = Ys + M::j0();
#pragma unroll 4
  for (int r = 0; r < rows; ++r) {
    float xv[M::TO], yv[M::TJ];
#pragma unroll
    for (int i = 0; i < M::TO; i += 2) {
      const float2 t = *reinterpret_cast<const float2*>(x0 + r * ldx + i);
      xv[i] = t.x; xv[i + 1] = t.y;
    }
#pragma unroll
    for (int j = 0; j < M::TJ; j += 2) {
      const float2 t = *reinterpret_cast<const float2*>(y0 + r * ldy + j);
      yv[j] = t.x; yv[j + 1] = t.y;
    }
#pragma unroll
    for (int i = 0; i < M::TO; ++i)
#pragma unroll
      for (int j = 0; j < M::TJ; ++j) acc[i][j] = fmaf(xv[i], yv[j], acc[i][j]);
  }
}

// ---- asynchronous global -> shared copies (LDGSTS): no register staging, every copy of a tile in flight at once
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, bool valid) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  const int sz = valid ? 16 : 0;   // src-size 0: the 16 destination bytes are zero-filled
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" :: "r"(s), "l"(gsrc), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gsrc) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(s), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// [TILE_M][COLS] row tile of a global [V][COLS] matrix -> smem (leading dim ld), rows >= V zero-filled
template <int TILE_M, int COLS>
__device__ __forceinline__ void cp_async_row_tile(float* __restrict__ dst, int ld, const float* __restrict__ src,
                                                  int row_base, int V) {
  constexpr int C4 = COLS / 4;
  for (int i = threadIdx.x; i < TILE_M * C4; i += kThreads) {
    const int r = i / C4, c = (i % C4) * 4;
    const int v = row_base + r;
    const bool ok = v < V;
    cp_async16(dst + r * ld + c, src + (size_t)(ok ? v : 0) * COLS + c, ok);
  }
}

// cooperative copy of a dense [rows][cols] fp32 matrix (global, contiguous) into smem with leading dim ld
template <int COLS>
__device__ __forceinline__ void load_matrix(float* __restrict__ dst, int ld, const float* __restrict__ src, int rows) {
  constexpr int C4 = COLS / 4;
  for (int i = threadIdx.x; i < rows * C4; i += kThreads) {
    const int r = i / C4, c = (i % C4) * 4;
    st4(dst + r * ld + c, ldg4(src + (size_t)r * COLS + c));
  }
}

// load a [TILE_M][COLS] row tile of a global [V][COLS] matrix into smem (zero-fill rows >= V)
template <int TILE_M, int COLS>
__device__ __forceinline__ void load_row_tile(float* __restrict__ dst, int ld, const float* __restrict__ src,
                                              int row_base, int V) {
  constexpr int C4 = COLS / 4;
  for (int i = threadIdx.x; i < TILE_M * C4; i += kThreads) {
    const int r = i / C4, c = (i % C4) * 4;
    const int v = row_base + r;
    float4 val = make4(0.f);
    if (v < V) val = ld4(src + (size_t)v * COLS + c);
    st4(dst + r * ld + c, val);
  }
}

// Host side: launch with the programmatic-stream-serialization attribute (SCGIB_PDL=0 disables: plain stream order)
bool pdl_enabled();
template <typename... KArgs, typename... Args>
inline void launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = pdl_enabled() ? 1 : 0;
  cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

}  // namespace scgib
