// encoder_bf16.cu - the operators of the --encoder GraphSAGE / GCN variants in bf16 mode (--dtype bf16): the same contracts
// as encoder_ops.cu on bf16 activations, with fp32 accumulation everywhere.
//
//   scgib_graph_aggregate_bf16 : bf16x8 (16-byte) row gathers, fp32 accumulation in CSR order, bf16 or fp32 output.
//   scgib_linear_fwd_bf16      : single-pass tcgen05 kind::f16 MMAs (bf16 operands, fp32 accumulator in tensor memory) on
//                                128-row tiles; the weights are rounded to bf16 once per CTA and stay in shared memory.
//   scgib_linear_bwd_w_bf16    : the contraction over rows on tcgen05 from the same bf16 row tiles read MN-major, accumulated
//                                in tensor memory over the CTA's row chunk; per-CTA partials, then the fixed-order reduction
//                                of the fp32 path (encoder_ops.cu).
//
// Rounding points (DESIGN §3.5; the bf16 emulation of the tests follows them exactly):
//   aggregation  out = rnd(fd * sum_u fs * in[u] + add)                (one rounding; fp32 output: none)
//   linear       Y   = rnd(act(sum_p (Xp (.) (Mp > 0)) rnd(Wp) + bias)) (X, M are bf16 already; fp32 output: no final rnd)
//   weight grad  dW  = (G (.) (M > 0))^T X,  db = column sums of G (.) (M > 0)   (bf16 inputs, fp32 sums, fp32 outputs)
// Every reduction runs in a fixed order: reruns are bit-identical.
#include "kernels.cuh"
#include "umma.cuh"
#include "../../include/scgib.h"

namespace scgib {
using namespace umma;

namespace encb {

constexpr int TM = 128;                       // rows per tile = the MMA M
constexpr int kSmemMax = 227 * 1024;          // opt-in dynamic shared memory per CTA
constexpr int kSmemSM = 228 * 1024;           // shared memory per SM

__device__ __forceinline__ void unpack8(uint4 h, float (&v)[8]) {
  v[0] = bf16_lo(h.x); v[1] = bf16_hi(h.x); v[2] = bf16_lo(h.y); v[3] = bf16_hi(h.y);
  v[4] = bf16_lo(h.z); v[5] = bf16_hi(h.z); v[6] = bf16_lo(h.w); v[7] = bf16_hi(h.w);
}
__device__ __forceinline__ uint4 pack8(const float (&v)[8]) {
  return make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
}
// x (.) (m > 0), 8 bf16 lanes (a NaN mask zeroes, as in the fp32 kernels)
__device__ __forceinline__ uint4 mask8(uint4 x, uint4 m) {
  auto h = [](uint32_t xv, uint32_t mv) {
    return (bf16_lo(mv) > 0.f ? (xv & 0xffffu) : 0u) | (bf16_hi(mv) > 0.f ? (xv & 0xffff0000u) : 0u);
  };
  return make_uint4(h(x.x, m.x), h(x.y, m.y), h(x.z, m.z), h(x.w, m.w));
}
__device__ __forceinline__ float deg_norm(int mode, int deg) {
  const float d = (float)max(deg, 1);
  return mode == 0 ? 1.f : (mode == 1 ? 1.f / d : 1.f / sqrtf(d));
}

// ------------------------------------------------------------------------------------------------
// aggregation: W / 8 lanes (capped at 32) own one row, 8 channels each
// ------------------------------------------------------------------------------------------------
template <int W, bool OUT_F32>
__global__ void __launch_bounds__(kThreads)
graph_aggregate_bf16_kernel(const bf16_t* __restrict__ in, const int32_t* __restrict__ row_map, const int32_t* __restrict__ indptr,
                            const int32_t* __restrict__ indices, int V, int src_norm, int dst_norm, const bf16_t* __restrict__ add,
                            void* __restrict__ out) {
  pdl_sync();
  constexpr int LPR = W / 8, RPC = kThreads / LPR;
  const int l = threadIdx.x % LPR;
  for (int v = blockIdx.x * RPC + threadIdx.x / LPR; v < V; v += gridDim.x * RPC) {
    const int e0 = __ldg(indptr + v), e1 = __ldg(indptr + v + 1);
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    for (int e = e0; e < e1; ++e) {
      const int u = __ldg(indices + e);
      const float fs = src_norm ? deg_norm(src_norm, __ldg(indptr + u + 1) - __ldg(indptr + u)) : 1.f;
      float x[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(in + (size_t)(row_map ? __ldg(row_map + u) : u) * W + l * 8)), x);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = fmaf(fs, x[j], acc[j]);
    }
    const float fd = deg_norm(dst_norm, e1 - e0);
    float r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = acc[j] * fd;
    if (add) {
      float a[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(add + (size_t)v * W + l * 8)), a);
#pragma unroll
      for (int j = 0; j < 8; ++j) r[j] += a[j];
    }
    if (OUT_F32) st8(reinterpret_cast<float*>(out) + (size_t)v * W + l * 8, r);
    else *reinterpret_cast<uint4*>(reinterpret_cast<bf16_t*>(out) + (size_t)v * W + l * 8) = pack8(r);
  }
}

// ------------------------------------------------------------------------------------------------
// linear forward.  Shared memory (format B of umma.cuh, 64-column blocks, 1024-byte aligned), per operand pair p:
//   W_p: ceil(Kp / 64) blocks of [O rows][64 bf16] (row o = output channel, K-major B operand; [K][O] weights are
//        transposed while staged), X_p: ceil(Kp / 64) blocks of [128 rows][64 bf16] (K-major A operand).
// Persistent CTAs; per 128-row tile: 8 warps load X (map / mask on load) -> one elected lane issues Kp / 16 MMAs per pair
// into one fp32 accumulator [128 lanes][O columns] -> every warp reads a quarter of the lanes x half of the columns, adds
// the bias, applies the ReLU and writes bf16 or fp32 rows.
// ------------------------------------------------------------------------------------------------
struct LinBf16Args {
  const bf16_t* X[2]; const bf16_t* M[2]; const float* W[2]; int K[2]; int kxo[2];
  const int32_t* map0;
  int nop, V, O, relu, y_f32;
  const float* bias;
  void* Y;
};
__host__ __device__ inline int kblocks(int K) { return (K + 63) / 64; }
__host__ __device__ inline int lin_w_off(const LinBf16Args& a, int p) { return p == 0 ? 0 : kblocks(a.K[0]) * a.O * 128; }
__host__ __device__ inline int lin_x_off(const LinBf16Args& a, int p) {
  int o = (kblocks(a.K[0]) + (a.nop > 1 ? kblocks(a.K[1]) : 0)) * a.O * 128;
  return p == 0 ? o : o + kblocks(a.K[0]) * TM * 128;
}
__host__ __device__ inline int lin_bar_off(const LinBf16Args& a) {
  return lin_x_off(a, 0) + (kblocks(a.K[0]) + (a.nop > 1 ? kblocks(a.K[1]) : 0)) * TM * 128;
}
__host__ inline int lin_smem_bytes(const LinBf16Args& a) { return lin_bar_off(a) + 64 + 1024; }   // + base alignment slack
__host__ __device__ inline uint32_t tmem_cols(int n) { uint32_t c = 32; while ((int)c < n) c <<= 1; return c; }

__global__ void __launch_bounds__(kThreads, 1) linear_fwd_bf16_kernel(LinBf16Args p) {
  pdl_sync();
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + lin_bar_off(p));
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bar + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, O = p.O;
  const uint32_t ncols = tmem_cols(O);
  if (threadIdx.x == 0) mbar_init(bar, 1);
  if (warp == 0) tmem_alloc(s_tmem, ncols);
  // weights -> bf16, [O rows][K] format B
  for (int q = 0; q < p.nop; ++q) {
    unsigned char* w = smem + lin_w_off(p, q);
    const int K = p.K[q], K8 = K / 8;
    for (int i = threadIdx.x; i < O * K8; i += kThreads) {
      int o, c8;
      float v[8];
      if (p.kxo[q]) {          // [K][O]: consecutive threads take consecutive o (coalesced per k)
        o = i % O; c8 = i / O;
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = __ldg(p.W[q] + (size_t)(c8 * 8 + j) * O + o);
      } else {
        o = i / K8; c8 = i % K8;
        const float4 a = ldg4(p.W[q] + (size_t)o * K + c8 * 8), b = ldg4(p.W[q] + (size_t)o * K + c8 * 8 + 4);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
      }
      *reinterpret_cast<uint4*>(w + (c8 >> 3) * (O * 128) + tile_b_off(o, c8 & 7)) = pack8(v);
    }
  }
  fence_smem_to_async();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *s_tmem;
  const uint32_t idesc = idesc_bf16(TM, O, false, false);
  const int q4 = warp & 3, half = warp >> 2, row = q4 * 32 + lane;
  const int n_tiles = (p.V + TM - 1) / TM;
  uint32_t phase = 0;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, phase ^= 1) {
    const int base = tile * TM;
    for (int q = 0; q < p.nop; ++q) {
      unsigned char* x = smem + lin_x_off(p, q);
      const int K = p.K[q], K8 = K / 8;
      const bf16_t* X = p.X[q];
      const bf16_t* M = p.M[q];
      const int32_t* map = q == 0 ? p.map0 : nullptr;
      for (int i = threadIdx.x; i < TM * K8; i += kThreads) {
        const int r = i / K8, c8 = i % K8, v = base + r;
        uint4 val = make_uint4(0, 0, 0, 0);
        if (v < p.V) {
          const size_t src = (size_t)(map ? __ldg(map + v) : v) * K + c8 * 8;
          val = __ldg(reinterpret_cast<const uint4*>(X + src));
          if (M) val = mask8(val, __ldg(reinterpret_cast<const uint4*>(M + src)));
        }
        *reinterpret_cast<uint4*>(x + (c8 >> 3) * (TM * 128) + tile_b_off(r, c8 & 7)) = val;
      }
    }
    fence_smem_to_async();
    __syncthreads();
    if (warp == 0) {
      fence_after_sync();
      for (int q = 0; q < p.nop; ++q) {
        const uint32_t x = smem_u32(smem + lin_x_off(p, q)), w = smem_u32(smem + lin_w_off(p, q));
        for (int k = 0; k < p.K[q] / 16; ++k)
          mma_bf16_w(tmem, desc_b_kmajor(x + (k >> 2) * (TM * 128), k & 3), desc_b_kmajor(w + (k >> 2) * (O * 128), k & 3), idesc,
                     q > 0 || k > 0);
      }
      mma_commit_w(bar);
    }
    mbar_wait(bar, phase);
    fence_after_sync();
    const int v = base + row;
    for (int c0 = half * (O / 2); c0 < (half + 1) * (O / 2); c0 += 16) {
      float y[16];
      tmem_ld16(tmem + ((uint32_t)(q4 * 32) << 16) + c0, y);
      if (p.bias) {
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
          const float4 b = ldg4(p.bias + c0 + j);
          y[j] += b.x; y[j + 1] += b.y; y[j + 2] += b.z; y[j + 3] += b.w;
        }
      }
      if (p.relu) {
#pragma unroll
        for (int j = 0; j < 16; ++j) y[j] = fmaxf(y[j], 0.f);
      }
      if (v < p.V) {
        if (p.y_f32) {
          float* dst = reinterpret_cast<float*>(p.Y) + (size_t)v * O + c0;
          st8(dst, y); st8(dst + 8, y + 8);
        } else {
          uint4* dst = reinterpret_cast<uint4*>(reinterpret_cast<bf16_t*>(p.Y) + (size_t)v * O + c0);
          dst[0] = pack8(*reinterpret_cast<float (*)[8]>(y));
          dst[1] = pack8(*reinterpret_cast<float (*)[8]>(y + 8));
        }
      }
    }
    fence_before_sync();
    __syncthreads();          // the accumulator and the X tiles are free for the next tile
  }
  if (warp == 0) tmem_dealloc(tmem, ncols);
}

// ------------------------------------------------------------------------------------------------
// weight gradient: CTA c reduces the rows [c * rows_per_chunk, ...) in 128-row tiles.  Gm = G (.) (M > 0) is stored as
// [128 rows][O] and X[map] as [128 rows][KP] (KP = max(K, 64)), both format B; read MN-major (K = tile rows) they give
// D[o][k] += sum_r Gm[r][o] X[r][k] as M = 128 (O = 64: M = 64) x N = KP MMAs, accumulated in tensor memory over the chunk.
// db: each loader thread owns 8 fixed channels and sums the bf16 values it stored, then a fixed-order sum over threads.
// ------------------------------------------------------------------------------------------------
struct BwdWBf16Args {
  const bf16_t* G; const bf16_t* M; const bf16_t* X; const int32_t* map;
  int V, O, K, rows_per_chunk;
  float* part;       // [chunks][O*K + O]
};
__host__ __device__ inline int bw_kp(int K) { return K < 64 ? 64 : K; }
__host__ __device__ inline int bw_x_off(int O) { return O / 64 * TM * 128; }
__host__ __device__ inline int bw_red_off(int O, int K) { return bw_x_off(O) + bw_kp(K) / 64 * TM * 128; }
__host__ __device__ inline int bw_bar_off(int O, int K) { return bw_red_off(O, K) + kThreads * 8 * 4; }
__host__ inline int bw_smem_bytes(int O, int K) { return bw_bar_off(O, K) + 64 + 1024; }

__global__ void __launch_bounds__(kThreads, 1) linear_bwd_w_bf16_kernel(BwdWBf16Args p) {
  pdl_sync();
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const int O = p.O, K = p.K, KP = bw_kp(K);
  unsigned char* g_tile = smem;
  unsigned char* x_tile = smem + bw_x_off(O);
  float* s_red = reinterpret_cast<float*>(smem + bw_red_off(O, K));
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + bw_bar_off(O, K));
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bar + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int MM = O == 64 ? 64 : 128, nM = O / MM;
  const uint32_t ncols = tmem_cols(nM * KP);
  if (threadIdx.x == 0) mbar_init(bar, 1);
  if (warp == 0) tmem_alloc(s_tmem, ncols);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *s_tmem;
  const uint32_t idesc = idesc_bf16(MM, KP, true, true);
  const int O8 = O / 8, K8 = KP / 8;
  const int gc = threadIdx.x % O8, gr = threadIdx.x / O8, GRP = kThreads / O8;   // this thread's G channels 8*gc.., rows gr + j*GRP
  float db[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) db[j] = 0.f;
  const int r_begin = blockIdx.x * p.rows_per_chunk, r_end = min(r_begin + p.rows_per_chunk, p.V);
  uint32_t phase = 0;
  int t = 0;
  for (int rb = r_begin; rb < r_end; rb += TM, ++t, phase ^= 1) {
    for (int r = gr; r < TM; r += GRP) {
      const int v = rb + r;
      uint4 g = make_uint4(0, 0, 0, 0);
      if (v < r_end) {
        const size_t gi = (size_t)v * O + gc * 8;
        g = __ldg(reinterpret_cast<const uint4*>(p.G + gi));
        if (p.M) g = mask8(g, __ldg(reinterpret_cast<const uint4*>(p.M + gi)));
      }
      float gv[8];
      unpack8(g, gv);
#pragma unroll
      for (int j = 0; j < 8; ++j) db[j] += gv[j];
      *reinterpret_cast<uint4*>(g_tile + (gc >> 3) * (TM * 128) + tile_b_off(r, gc & 7)) = g;
    }
    for (int i = threadIdx.x; i < TM * K8; i += kThreads) {
      const int r = i / K8, c8 = i % K8, v = rb + r;
      uint4 x = make_uint4(0, 0, 0, 0);
      if (v < r_end && c8 * 8 < K)
        x = __ldg(reinterpret_cast<const uint4*>(p.X + (size_t)(p.map ? __ldg(p.map + v) : v) * K + c8 * 8));
      *reinterpret_cast<uint4*>(x_tile + (c8 >> 3) * (TM * 128) + tile_b_off(r, c8 & 7)) = x;
    }
    fence_smem_to_async();
    __syncthreads();
    if (warp == 0) {
      fence_after_sync();
      const uint32_t ga = smem_u32(g_tile), xa = smem_u32(x_tile);
      for (int m = 0; m < nM; ++m)
#pragma unroll
        for (int s = 0; s < TM / 16; ++s)
          mma_bf16_w(tmem + (uint32_t)(m * KP), desc_b_mnmajor(ga + (uint32_t)(m * 2 * TM * 128), TM * 128, s),
                     desc_b_mnmajor(xa, TM * 128, s), idesc, t > 0 || s > 0);
      mma_commit_w(bar);
    }
    mbar_wait(bar, phase);     // the tiles are free again
    fence_after_sync();
    __syncthreads();
  }
  // partials of this chunk: dW [o][k] from the accumulator (row o: lane o of block m, or lane (o/16)*32 + o%16 at M = 64)
  float* part = p.part + (size_t)blockIdx.x * ((size_t)O * K + O);
  const int q4 = warp & 3, half = warp >> 2;
  for (int m = 0; m < nM; ++m) {
    const bool act = MM == 128 || lane < 16;
    const int o = MM == 128 ? m * 128 + q4 * 32 + lane : q4 * 16 + (lane & 15);
    for (int c0 = half * (K / 2); c0 < (half + 1) * (K / 2); c0 += 16) {
      float d[16];
      tmem_ld16(tmem + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(m * KP + c0), d);
      if (act) {
        float* dst = part + (size_t)o * K + c0;
#pragma unroll
        for (int j = 0; j < 16; j += 4) st4(dst + j, make_float4(d[j], d[j + 1], d[j + 2], d[j + 3]));
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) s_red[(gr * O8 + gc) * 8 + j] = db[j];
  __syncthreads();
  for (int o = threadIdx.x; o < O; o += kThreads) {
    float s = 0.f;
    for (int g = 0; g < GRP; ++g) s += s_red[(g * O8 + o / 8) * 8 + o % 8];
    part[(size_t)O * K + o] = s;
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, ncols);
}

}  // namespace encb

// persistent grid: as many CTAs per SM as shared and tensor memory allow, and no more (the dynamic shared memory request
// is raised so that a further CTA cannot fit: an SM never holds a CTA that would wait for tensor-memory columns)
static int persistent_ctas(int smem, uint32_t tcols, int work, int& smem_req) {
  int occ = encb::kSmemSM / (smem + 1024);
  occ = min(occ, (int)(512 / tcols));
  occ = max(occ, 1);
  smem_req = max(smem, encb::kSmemSM / (occ + 1) - 1024 + 16);
  smem_req = min(smem_req, encb::kSmemMax);
  return max(1, min(work, occ * num_sms()));
}

// row chunks of the weight-gradient reduction: at least 4 tiles per chunk, at most one chunk per SM
static int bwd_w_bf16_chunks(int V) {
  const int tiles = (V + encb::TM - 1) / encb::TM;
  return max(1, min(num_sms(), (tiles + 3) / 4));
}

}  // namespace scgib

using namespace scgib;

static bool width_ok_b(int W) { return W == 32 || W == 64 || W == 128 || W == 256; }
static bool al16(const void* p) { return ((uintptr_t)p & 15u) == 0; }

// DT: 32, 64 or 128 (the *_d entry); scgib_input_proj_fwd_bf16 keeps its contract DT = 32
static int input_proj_fwd_bf16(const float* x, const float* Wt, int32_t N, int32_t F, int32_t DT, int32_t max_dt, void* t,
                               void* stream) {
  if (!x || !Wt || !t) return SCGIB_E_NULL;
  if (!transfer_width_ok(DT, max_dt) || F < 1 || F > kMaxInDim) return SCGIB_E_SHAPE;
  if (N < 1) return SCGIB_E_RANGE;
  if (!al16(t)) return SCGIB_E_ALIGN;
  launch_input_proj_fwd(x, Wt, N, F, DT, 1, reinterpret_cast<float*>(t), (cudaStream_t)stream, true);
  return (int)cudaGetLastError();
}
extern "C" SCGIB_API int scgib_input_proj_fwd_bf16(const float* x, const float* Wt, int32_t N, int32_t F, int32_t DT, void* t,
                                                   void* stream) {
  return input_proj_fwd_bf16(x, Wt, N, F, DT, 32, t, stream);
}
extern "C" SCGIB_API int scgib_input_proj_fwd_d_bf16(const float* x, const float* Wt, int32_t N, int32_t F, int32_t DT, void* t,
                                                     void* stream) {
  return input_proj_fwd_bf16(x, Wt, N, F, DT, kMaxTransfer, t, stream);
}

extern "C" SCGIB_API int scgib_f32_to_bf16(const float* in, int64_t n, void* out, void* stream) {
  if (!in || !out) return SCGIB_E_NULL;
  if (n < 1) return SCGIB_E_RANGE;
  if (n % 8) return SCGIB_E_SHAPE;
  if (!al16(in) || !al16(out)) return SCGIB_E_ALIGN;
  launch_f32_to_bf16(in, out, (size_t)n, (cudaStream_t)stream);
  return (int)cudaGetLastError();
}

extern "C" SCGIB_API int scgib_graph_aggregate_bf16(const void* in, int32_t W, const int32_t* row_map, const int32_t* indptr,
                                                    const int32_t* indices, int32_t V, int32_t src_norm, int32_t dst_norm,
                                                    const void* add, void* out, int32_t out_f32, void* stream) {
  if (!in || !indptr || !out) return SCGIB_E_NULL;
  if (!width_ok_b(W) || src_norm < 0 || src_norm > 2 || dst_norm < 0 || dst_norm > 2) return SCGIB_E_SHAPE;
  if (V < 1) return SCGIB_E_RANGE;
  if (!al16(in) || !al16(out) || !al16(add)) return SCGIB_E_ALIGN;
  cudaStream_t s = (cudaStream_t)stream;
  const bf16_t* i = reinterpret_cast<const bf16_t*>(in);
  const bf16_t* a = reinterpret_cast<const bf16_t*>(add);
  const int rpc = kThreads / (W / 8);
  const int grid = min((V + rpc - 1) / rpc, 16 * num_sms());
#define AGG_B(WW)                                                                                                              \
  if (out_f32) launch_k((encb::graph_aggregate_bf16_kernel<WW, true>), dim3(grid), dim3(kThreads), 0, s, i, row_map, indptr, indices, V, src_norm, dst_norm, a, out); \
  else launch_k((encb::graph_aggregate_bf16_kernel<WW, false>), dim3(grid), dim3(kThreads), 0, s, i, row_map, indptr, indices, V, src_norm, dst_norm, a, out);
  switch (W) {
    case 32: AGG_B(32) break;
    case 64: AGG_B(64) break;
    case 128: AGG_B(128) break;
    default: AGG_B(256) break;
  }
#undef AGG_B
  return (int)cudaGetLastError();
}

extern "C" SCGIB_API int scgib_linear_fwd_bf16(const void* X0, const void* M0, const int32_t* map0, const float* W0, int32_t K0,
                                               int32_t w0_kxo, const void* X1, const void* M1, const float* W1, int32_t K1,
                                               int32_t w1_kxo, const float* bias, int32_t relu, int32_t V, int32_t O, void* Y,
                                               int32_t y_f32, void* stream) {
  if (!X0 || !W0 || !Y || (X1 && !W1)) return SCGIB_E_NULL;
  if (!width_ok_b(K0) || !width_ok_b(O) || (X1 && !width_ok_b(K1))) return SCGIB_E_SHAPE;
  if (V < 1) return SCGIB_E_RANGE;
  if (!al16(X0) || !al16(M0) || !al16(W0) || !al16(X1) || !al16(M1) || !al16(W1) || !al16(bias) || !al16(Y)) return SCGIB_E_ALIGN;
  encb::LinBf16Args a;
  a.X[0] = reinterpret_cast<const bf16_t*>(X0); a.M[0] = reinterpret_cast<const bf16_t*>(M0); a.W[0] = W0; a.K[0] = K0; a.kxo[0] = w0_kxo;
  a.X[1] = reinterpret_cast<const bf16_t*>(X1); a.M[1] = reinterpret_cast<const bf16_t*>(M1); a.W[1] = W1; a.K[1] = X1 ? K1 : 0;
  a.kxo[1] = w1_kxo;
  a.map0 = map0; a.nop = X1 ? 2 : 1; a.V = V; a.O = O; a.relu = relu; a.y_f32 = y_f32; a.bias = bias; a.Y = Y;
  const int smem = encb::lin_smem_bytes(a);
  if (smem > encb::kSmemMax) return SCGIB_E_SHAPE;      // two wide pairs: weights + row tiles exceed shared memory
  int req;
  const int grid = persistent_ctas(smem, encb::tmem_cols(O), (V + encb::TM - 1) / encb::TM, req);
  static bool once = (cudaFuncSetAttribute(encb::linear_fwd_bf16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, encb::kSmemMax), true);
  (void)once;
  launch_k((encb::linear_fwd_bf16_kernel), dim3(grid), dim3(kThreads), req, (cudaStream_t)stream, a);
  return (int)cudaGetLastError();
}

extern "C" SCGIB_API size_t scgib_linear_bwd_w_bf16_workspace_bytes(int32_t V, int32_t O, int32_t K) {
  if (V < 1) return 256;
  return (size_t)bwd_w_bf16_chunks(V) * ((size_t)O * K + O) * sizeof(float) + 256;
}

// dW (+)= (G (.) (M > 0))^T X[map]  ([O][K], or [K][O] with kxo), db (+)= column sums (optional); G, M, X bf16, dW / db fp32
extern "C" SCGIB_API int scgib_linear_bwd_w_bf16(const void* G, const void* M, const void* X, const int32_t* map, int32_t V,
                                                 int32_t O, int32_t K, int32_t kxo, int32_t accumulate, float* dW, float* db,
                                                 void* workspace, size_t workspace_bytes, void* stream) {
  if (!G || !X || !dW || !workspace) return SCGIB_E_NULL;
  if (!(O == 64 || O == 128 || O == 256) || !width_ok_b(K)) return SCGIB_E_SHAPE;
  if (V < 1) return SCGIB_E_RANGE;
  if (!al16(G) || !al16(M) || !al16(X) || !al16(workspace)) return SCGIB_E_ALIGN;
  if (workspace_bytes < scgib_linear_bwd_w_bf16_workspace_bytes(V, O, K)) return SCGIB_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  const int chunks = bwd_w_bf16_chunks(V);
  const int rpc = ((V + chunks - 1) / chunks + encb::TM - 1) / encb::TM * encb::TM;
  encb::BwdWBf16Args a{reinterpret_cast<const bf16_t*>(G), reinterpret_cast<const bf16_t*>(M), reinterpret_cast<const bf16_t*>(X),
                       map, V, O, K, rpc, (float*)workspace};
  const int nchunks = (V + rpc - 1) / rpc;
  int req;
  const int KP = encb::bw_kp(K);
  persistent_ctas(encb::bw_smem_bytes(O, K), encb::tmem_cols((O == 256 ? 2 : 1) * KP), nchunks, req);
  static bool once = (cudaFuncSetAttribute(encb::linear_bwd_w_bf16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, encb::kSmemMax), true);
  (void)once;
  launch_k((encb::linear_bwd_w_bf16_kernel), dim3(nchunks), dim3(kThreads), req, s, a);
  launch_linear_bwd_w_reduce((const float*)workspace, nchunks, O, K, kxo, accumulate, dW, db, s);
  return (int)cudaGetLastError();
}
