// encoder_ops.cu - the building blocks of the --encoder GraphSAGE / GCN variants (SURVEY 8 f4, second half) as individual
// operators behind the C ABI: normalised neighbourhood aggregation, a tiled FP32 linear layer with up to two operand pairs,
// its weight-gradient reduction, and a width-generic segment sum.
//
// Reference call sites replaced (paths relative to the reference tree):
//   GraphSAGE.forward  models.py:91-104  (DGL SAGEConv 'mean': fc_self(h) + fc_neigh(mean_{u in N(v)} h_u))
//   GCN.forward        models.py:75-88   (DGL GraphConv norm='both': D^-1/2 A D^-1/2 h W + b, degrees clamped to 1)
// The molecular graphs and their induced ego-nets are stored symmetric (both directions of every bond), so the backward
// of an aggregation is the same gather with the two degree normalisations exchanged - no transposed CSR, no atomics; every
// reduction runs in a fixed order (bit-identical reruns).
//
// These layers are plain FP32 FFMA tiles (the host composes them per layer; s-cgib_b200/encoders.py): the tensor-core
// pipeline of this library is built around the GIN layer (gin_tc3.cu / gin_bwd_h.cu), which the CLI default selects.
// --dtype bf16 runs the same operators on bf16 activations with tcgen05 products: encoder_bf16.cu.
#include "kernels.cuh"
#include "../../include/scgib.h"

namespace scgib {

// degree normalisation codes of scgib_graph_aggregate_f32
__device__ __forceinline__ float deg_norm(int mode, int deg) {
  const float d = (float)max(deg, 1);
  return mode == 0 ? 1.f : (mode == 1 ? 1.f / d : 1.f / sqrtf(d));
}

// out[v] = (add ? add[v] : 0) + fd(deg v) * sum_{u in N(v)} fs(deg u) * in[map(u)]      (W channels, W / 4 <= 64 float4 lanes)
// LPR lanes own one row (4 * NQ channels each)
template <int W>
__global__ void __launch_bounds__(kThreads)
graph_aggregate_kernel(const float* __restrict__ in, const int32_t* __restrict__ row_map, const int32_t* __restrict__ indptr,
                       const int32_t* __restrict__ indices, int V, int src_norm, int dst_norm, const float* __restrict__ add,
                       float* __restrict__ out) {
  pdl_sync();
  constexpr int Q = W / 4, LPR = Q < 32 ? Q : 32, NQ = Q / LPR, RPC = kThreads / LPR;
  const int l = threadIdx.x % LPR;
  for (int v = blockIdx.x * RPC + threadIdx.x / LPR; v < V; v += gridDim.x * RPC) {
    const int e0 = __ldg(indptr + v), e1 = __ldg(indptr + v + 1);
    float4 acc[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) acc[q] = make4(0.f);
    for (int e = e0; e < e1; ++e) {
      const int u = __ldg(indices + e);
      const float fs = src_norm ? deg_norm(src_norm, __ldg(indptr + u + 1) - __ldg(indptr + u)) : 1.f;
      const float* row = in + (size_t)(row_map ? __ldg(row_map + u) : u) * W;
#pragma unroll
      for (int q = 0; q < NQ; ++q) {
        const float4 x = ld4(row + (l + q * LPR) * 4);
        acc[q].x = fmaf(fs, x.x, acc[q].x); acc[q].y = fmaf(fs, x.y, acc[q].y);
        acc[q].z = fmaf(fs, x.z, acc[q].z); acc[q].w = fmaf(fs, x.w, acc[q].w);
      }
    }
    const float fd = deg_norm(dst_norm, e1 - e0);
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
      float4 r = make_float4(acc[q].x * fd, acc[q].y * fd, acc[q].z * fd, acc[q].w * fd);
      if (add) r = add4(r, ld4(add + (size_t)v * W + (l + q * LPR) * 4));
      st4(out + (size_t)v * W + (l + q * LPR) * 4, r);
    }
  }
}

// out[s] = sum of the rows of segment s (dgl.sum_nodes), any width W
template <int W>
__global__ void __launch_bounds__(kThreads)
segment_sum_w_kernel(const float* __restrict__ in, const int32_t* __restrict__ seg_ptr, int S, float* __restrict__ out) {
  pdl_sync();
  constexpr int Q = W / 4, LPR = Q < 32 ? Q : 32, NQ = Q / LPR, RPC = kThreads / LPR;
  const int l = threadIdx.x % LPR;
  for (int s = blockIdx.x * RPC + threadIdx.x / LPR; s < S; s += gridDim.x * RPC) {
    const int r0 = __ldg(seg_ptr + s), r1 = __ldg(seg_ptr + s + 1);
    float4 acc[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) acc[q] = make4(0.f);
    for (int r = r0; r < r1; ++r)
#pragma unroll
      for (int q = 0; q < NQ; ++q) acc[q] = add4(acc[q], ld4(in + (size_t)r * W + (l + q * LPR) * 4));
#pragma unroll
    for (int q = 0; q < NQ; ++q) st4(out + (size_t)s * W + (l + q * LPR) * 4, acc[q]);
  }
}

// ------------------------------------------------------------------------------------------------
// Y[V][O] = act( sum_p Xp[mapp(r)][Kp] (.) (Mp > 0) * Wp + bias )       p = 0, 1 (second pair optional)
//   Wp is [O][Kp] (nn.Linear layout, w_kxo = 0) or [Kp][O] (GraphConv layout / a transposed product, w_kxo = 1).
//   Mp (optional, same shape as Xp): ReLU mask of a backward product, g (.) (h > 0).
// CTA tile: 128 rows x 32 output columns, K chunks of 32; thread = 4 rows x 4 columns.
// ------------------------------------------------------------------------------------------------
struct LinOperand {
  const float* X; const float* M; const int32_t* map; const float* Wt; int K; int w_kxo;
};
struct LinearArgs {
  LinOperand op[2];
  int nop, V, O, relu;
  const float* bias;
  float* Y;
};
constexpr int LTM = 128, LTN = 32, LTK = 32;

__global__ void __launch_bounds__(kThreads) linear_fwd_kernel(LinearArgs p) {
  pdl_sync();
  __shared__ float s_x[LTM][LTK + 1];
  __shared__ __align__(16) float s_w[LTK][LTN];
  const int row0 = blockIdx.x * LTM, col0 = blockIdx.y * LTN;
  const int tc = threadIdx.x & 7, tr = threadIdx.x >> 3;         // columns tc*4..+3, rows tr*4..+3
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int o = 0; o < p.nop; ++o) {
    const LinOperand& q = p.op[o];
    for (int k0 = 0; k0 < q.K; k0 += LTK) {
      __syncthreads();
      // X chunk: 128 rows x 32 columns, 8 lanes x float4 per row
      for (int i = threadIdx.x; i < LTM * (LTK / 4); i += kThreads) {
        const int r = i >> 3, c = (i & 7) * 4;
        const int v = row0 + r;
        float4 x = make4(0.f);
        if (v < p.V) {
          const size_t src = (size_t)(q.map ? __ldg(q.map + v) : v) * q.K + k0 + c;
          x = ld4(q.X + src);
          if (q.M) {
            const float4 m = ld4(q.M + src);
            x = make_float4(m.x > 0.f ? x.x : 0.f, m.y > 0.f ? x.y : 0.f, m.z > 0.f ? x.z : 0.f, m.w > 0.f ? x.w : 0.f);
          }
        }
        s_x[r][c] = x.x; s_x[r][c + 1] = x.y; s_x[r][c + 2] = x.z; s_x[r][c + 3] = x.w;
      }
      // W chunk -> s_w[k][n]
      for (int i = threadIdx.x; i < LTK * LTN; i += kThreads) {
        if (q.w_kxo) { const int k = i / LTN, n = i % LTN; s_w[k][n] = __ldg(q.Wt + (size_t)(k0 + k) * p.O + col0 + n); }
        else { const int n = i / LTK, k = i % LTK; s_w[k][n] = __ldg(q.Wt + (size_t)(col0 + n) * q.K + k0 + k); }
      }
      __syncthreads();
#pragma unroll 8
      for (int k = 0; k < LTK; ++k) {
        const float4 w = ld4(&s_w[k][tc * 4]);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float x = s_x[tr * 4 + i][k];
          acc[i][0] = fmaf(x, w.x, acc[i][0]); acc[i][1] = fmaf(x, w.y, acc[i][1]);
          acc[i][2] = fmaf(x, w.z, acc[i][2]); acc[i][3] = fmaf(x, w.w, acc[i][3]);
        }
      }
    }
  }
  const float4 b = p.bias ? ldg4(p.bias + col0 + tc * 4) : make4(0.f);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int v = row0 + tr * 4 + i;
    if (v >= p.V) continue;
    float4 y = make_float4(acc[i][0] + b.x, acc[i][1] + b.y, acc[i][2] + b.z, acc[i][3] + b.w);
    if (p.relu) y = relu4(y);
    st4(p.Y + (size_t)v * p.O + col0 + tc * 4, y);
  }
}

// ------------------------------------------------------------------------------------------------
// dW[o][k] = sum_r Gm[r][o] X[map(r)][k],  db[o] = sum_r Gm[r][o],  Gm = G (.) (M > 0)
// grid (row chunks, O tiles of 64, K tiles of 64): per-chunk partial tiles, then a fixed-order reduction over the chunks
// (kxo: dW stored [K][O], the GraphConv weight layout; accumulate: add to the destination - a layer applied twice).
// ------------------------------------------------------------------------------------------------
struct LinearBwdWArgs {
  const float* G; const float* M; const float* X; const int32_t* map;
  int V, O, K, rows_per_chunk;
  float* part;       // [chunks][O*K + O]
};
constexpr int WT = 64, WR = 32;

__global__ void __launch_bounds__(kThreads) linear_bwd_w_kernel(LinearBwdWArgs p) {
  pdl_sync();
  __shared__ __align__(16) float s_g[WR][WT];
  __shared__ __align__(16) float s_x[WR][WT];
  const int chunk = blockIdx.x, o0 = blockIdx.y * WT, k0 = blockIdx.z * WT;
  const int to = threadIdx.x >> 4, tk = threadIdx.x & 15;        // outputs o0 + to*4..+3, k0 + tk*4..+3
  float acc[4][4], accb[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const int r_begin = chunk * p.rows_per_chunk, r_end = min(r_begin + p.rows_per_chunk, p.V);
  const int kw = min(WT, p.K - k0);                                // valid K columns of this tile (32 or 64)
  for (int rb = r_begin; rb < r_end; rb += WR) {
    __syncthreads();
    for (int i = threadIdx.x; i < WR * (WT / 4); i += kThreads) {
      const int r = i >> 4, c = (i & 15) * 4;
      const int v = rb + r;
      float4 g = make4(0.f), x = make4(0.f);
      if (v < r_end) {
        const size_t gi = (size_t)v * p.O + o0 + c;
        g = ld4(p.G + gi);
        if (p.M) {
          const float4 m = ld4(p.M + gi);
          g = make_float4(m.x > 0.f ? g.x : 0.f, m.y > 0.f ? g.y : 0.f, m.z > 0.f ? g.z : 0.f, m.w > 0.f ? g.w : 0.f);
        }
        if (c < kw) x = ld4(p.X + (size_t)(p.map ? __ldg(p.map + v) : v) * p.K + k0 + c);
      }
      st4(&s_g[r][c], g);
      st4(&s_x[r][c], x);
    }
    __syncthreads();
#pragma unroll 4
    for (int r = 0; r < WR; ++r) {
      const float4 g = ld4(&s_g[r][to * 4]), x = ld4(&s_x[r][tk * 4]);
      const float gv[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        acc[i][0] = fmaf(gv[i], x.x, acc[i][0]); acc[i][1] = fmaf(gv[i], x.y, acc[i][1]);
        acc[i][2] = fmaf(gv[i], x.z, acc[i][2]); acc[i][3] = fmaf(gv[i], x.w, acc[i][3]);
        if (tk == 0) accb[i] += gv[i];
      }
    }
  }
  float* part = p.part + (size_t)chunk * ((size_t)p.O * p.K + p.O);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int o = o0 + to * 4 + i;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + tk * 4 + j;
      if (k < p.K) part[(size_t)o * p.K + k] = acc[i][j];
    }
    if (tk == 0 && blockIdx.z == 0) part[(size_t)p.O * p.K + o] = accb[i];
  }
}

__global__ void __launch_bounds__(kThreads)
linear_bwd_w_reduce_kernel(const float* __restrict__ part, int chunks, int O, int K, int kxo, int accumulate,
                           float* __restrict__ dW, float* __restrict__ db) {
  pdl_sync();
  const int n = O * K + O;
  for (int i = blockIdx.x * kThreads + threadIdx.x; i < n; i += gridDim.x * kThreads) {
    double s0 = 0.0, s1 = 0.0;
    int c = 0;
    for (; c + 1 < chunks; c += 2) {
      s0 += (double)__ldcg(part + (size_t)c * n + i);
      s1 += (double)__ldcg(part + (size_t)(c + 1) * n + i);
    }
    if (c < chunks) s0 += (double)__ldcg(part + (size_t)c * n + i);
    const float v = (float)(s0 + s1);
    if (i < O * K) {
      const int o = i / K, k = i % K;
      float* d = dW + (kxo ? (size_t)k * O + o : (size_t)i);
      *d = accumulate ? *d + v : v;
    } else if (db) {
      float* d = db + (i - O * K);
      *d = accumulate ? *d + v : v;
    }
  }
}

void launch_linear_plain(const float* X, const float* W, const float* bias, int V, int K, int O, float* Y, cudaStream_t s) {
  LinearArgs a;
  a.op[0] = LinOperand{X, nullptr, nullptr, W, K, 0};
  a.op[1] = LinOperand{nullptr, nullptr, nullptr, nullptr, 0, 0};
  a.nop = 1; a.V = V; a.O = O; a.relu = 0; a.bias = bias; a.Y = Y;
  launch_k((linear_fwd_kernel), dim3((V + LTM - 1) / LTM, O / LTN), dim3(kThreads), 0, s, a);
}

void launch_linear_bwd_w_reduce(const float* part, int chunks, int O, int K, int kxo, int accumulate, float* dW, float* db,
                                cudaStream_t s) {
  const int n = O * K + O;
  launch_k((linear_bwd_w_reduce_kernel), dim3(min((n + kThreads - 1) / kThreads, 4 * num_sms())), dim3(kThreads), 0, s,
           part, chunks, O, K, kxo, accumulate, dW, db);
}

// row chunks of the weight-gradient reduction: enough (chunks x output tiles) CTAs for two per SM, at least 256 rows per chunk
static int bwd_w_chunks(int V, int O, int K) {
  int tiles = (O / WT) * ((K + WT - 1) / WT);
  if (tiles < 1) tiles = 1;
  int c = (2 * num_sms() + tiles - 1) / tiles;
  const int cmax = (V + 255) / 256;
  if (c > cmax) c = cmax;
  return c < 1 ? 1 : c;
}

}  // namespace scgib

using namespace scgib;

static bool width_ok(int W) { return W == 32 || W == 64 || W == 128 || W == 256; }

// in [rows][W]; out[v] = (add ? add[v] : 0) + fd(v) * sum_{u in N(v)} fs(u) in[map(u)];  norms: 0 none, 1 1/deg, 2 deg^-1/2
extern "C" SCGIB_API int scgib_graph_aggregate_f32(const float* in, int32_t W, const int32_t* row_map, const int32_t* indptr,
                                                   const int32_t* indices, int32_t V, int32_t src_norm, int32_t dst_norm,
                                                   const float* add, float* out, void* stream) {
  if (!in || !indptr || !out) return SCGIB_E_NULL;
  if (!width_ok(W) || src_norm < 0 || src_norm > 2 || dst_norm < 0 || dst_norm > 2) return SCGIB_E_SHAPE;
  if (V < 1) return SCGIB_E_RANGE;
  cudaStream_t s = (cudaStream_t)stream;
  const int lpr = W / 4 < 32 ? W / 4 : 32, rpc = kThreads / lpr;
  const int grid = min((V + rpc - 1) / rpc, 16 * num_sms());
  switch (W) {
    case 32: launch_k((graph_aggregate_kernel<32>), dim3(grid), dim3(kThreads), 0, s, in, row_map, indptr, indices, V, src_norm, dst_norm, add, out); break;
    case 64: launch_k((graph_aggregate_kernel<64>), dim3(grid), dim3(kThreads), 0, s, in, row_map, indptr, indices, V, src_norm, dst_norm, add, out); break;
    case 128: launch_k((graph_aggregate_kernel<128>), dim3(grid), dim3(kThreads), 0, s, in, row_map, indptr, indices, V, src_norm, dst_norm, add, out); break;
    default: launch_k((graph_aggregate_kernel<256>), dim3(grid), dim3(kThreads), 0, s, in, row_map, indptr, indices, V, src_norm, dst_norm, add, out); break;
  }
  return (int)cudaGetLastError();
}

extern "C" SCGIB_API int scgib_segment_sum_w_f32(const float* in, const int32_t* seg_ptr, int32_t S, int32_t W, float* out, void* stream) {
  if (!in || !seg_ptr || !out) return SCGIB_E_NULL;
  if (!width_ok(W)) return SCGIB_E_SHAPE;
  if (S < 1) return SCGIB_E_RANGE;
  cudaStream_t s = (cudaStream_t)stream;
  const int lpr = W / 4 < 32 ? W / 4 : 32, rpc = kThreads / lpr;
  const int grid = min((S + rpc - 1) / rpc, 16 * num_sms());
  switch (W) {
    case 32: launch_k((segment_sum_w_kernel<32>), dim3(grid), dim3(kThreads), 0, s, in, seg_ptr, S, out); break;
    case 64: launch_k((segment_sum_w_kernel<64>), dim3(grid), dim3(kThreads), 0, s, in, seg_ptr, S, out); break;
    case 128: launch_k((segment_sum_w_kernel<128>), dim3(grid), dim3(kThreads), 0, s, in, seg_ptr, S, out); break;
    default: launch_k((segment_sum_w_kernel<256>), dim3(grid), dim3(kThreads), 0, s, in, seg_ptr, S, out); break;
  }
  return (int)cudaGetLastError();
}

// Y = act(X0[map0] (.) (M0 > 0) * W0 + X1 (.) (M1 > 0) * W1 + bias); X1 == NULL: one operand pair.  K0, K1, O multiples of 32.
extern "C" SCGIB_API int scgib_linear_fwd_f32(const float* X0, const float* M0, const int32_t* map0, const float* W0, int32_t K0,
                                              int32_t w0_kxo, const float* X1, const float* M1, const float* W1, int32_t K1,
                                              int32_t w1_kxo, const float* bias, int32_t relu, int32_t V, int32_t O, float* Y,
                                              void* stream) {
  if (!X0 || !W0 || !Y || (X1 && !W1)) return SCGIB_E_NULL;
  if (K0 < 32 || K0 % 32 || O < 32 || O % 32 || (X1 && (K1 < 32 || K1 % 32))) return SCGIB_E_SHAPE;
  if (V < 1) return SCGIB_E_RANGE;
  LinearArgs a;
  a.op[0] = LinOperand{X0, M0, map0, W0, K0, w0_kxo};
  a.op[1] = LinOperand{X1, M1, nullptr, W1, K1, w1_kxo};
  a.nop = X1 ? 2 : 1; a.V = V; a.O = O; a.relu = relu; a.bias = bias; a.Y = Y;
  launch_k((linear_fwd_kernel), dim3((V + LTM - 1) / LTM, O / LTN), dim3(kThreads), 0, (cudaStream_t)stream, a);
  return (int)cudaGetLastError();
}

extern "C" SCGIB_API size_t scgib_linear_bwd_w_workspace_bytes(int32_t V, int32_t O, int32_t K) {
  return (size_t)bwd_w_chunks(V, O, K) * ((size_t)O * K + O) * sizeof(float) + 256;
}

// dW (+)= (G (.) (M > 0))^T X[map]  ([O][K], or [K][O] with kxo), db (+)= column sums (optional)
extern "C" SCGIB_API int scgib_linear_bwd_w_f32(const float* G, const float* M, const float* X, const int32_t* map, int32_t V,
                                                int32_t O, int32_t K, int32_t kxo, int32_t accumulate, float* dW, float* db,
                                                void* workspace, size_t workspace_bytes, void* stream) {
  if (!G || !X || !dW || !workspace) return SCGIB_E_NULL;
  if (O < 64 || O % 64 || K < 32 || K % 32) return SCGIB_E_SHAPE;
  if (V < 1) return SCGIB_E_RANGE;
  if (workspace_bytes < scgib_linear_bwd_w_workspace_bytes(V, O, K)) return SCGIB_E_WORKSPACE;
  if (((uintptr_t)workspace & 15u) != 0) return SCGIB_E_ALIGN;
  cudaStream_t s = (cudaStream_t)stream;
  const int chunks = bwd_w_chunks(V, O, K);
  LinearBwdWArgs a{G, M, X, map, V, O, K, ((V + chunks - 1) / chunks + WR - 1) / WR * WR, (float*)workspace};
  launch_k((linear_bwd_w_kernel), dim3(chunks, O / WT, (K + WT - 1) / WT), dim3(kThreads), 0, s, a);
  launch_linear_bwd_w_reduce((const float*)workspace, chunks, O, K, kxo, accumulate, dW, db, s);
  return (int)cudaGetLastError();
}
