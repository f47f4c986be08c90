// logm_kernels.cu - the `--recons_type logM` reconstruction loss (reference models.py:770-782 `loss_recon`, with the
// k-step log transition matrices of util.py:60-91 `GetProbTranMat` / `getM_logM`) without any dense n x n matrix and
// without the offline `pts/*_M_khop_k.pt` files:
//
//   loss = (1/k) sum_g sum_{i=1..k} || Z_g Z_g^T - L_{g,i} ||_F^2 / n_g^2,
//   L_{g,i}[r][c] = max( log( (A_g^i)[r][c] / colsum_c(A_g^i) ) - log(1/n_g), 0 )       (nan / -inf -> 0)
//
// || Z Z^T - L ||^2 = || Z^T Z ||_F^2 - 2 sum_{rc} (z_r . z_c) L_rc + sum_{rc} L_rc^2, and L_{g,i} is SPARSE: (A^i)[r][c] is the
// number of i-step walks r -> c, non-zero only inside the i-hop ball of r.  So the loss is a per-graph H x H Gram term (H = 64 or 128)
// plus a sum over the (seed, ball node) pairs of the k-hop ego-nets - the same warp-per-seed machinery as the ego-net
// extraction, with a walk-count dynamic programme on the ball.  A is symmetric, so colsum_c(A^i) = rowsum_c(A^i) = the
// number of i-step walks starting at c (`walks`), and L_i[c][r] follows from the same count as L_i[r][c].
//
// Gradient:  gZ_g = (4 / n^2) Z_g (Z_g^T Z_g) - (2 / (k n^2)) sum_i (L_i + L_i^T) Z_g.
// Every reduction is in a fixed order (per-seed / per-graph terms, then one fp64 reduce): no float atomics.
#include "kernels.cuh"
#include "../../include/scgib.h"

namespace scgib {

namespace {
constexpr int LCAP = SCGIB_EGO_CAP;    // ball capacity (nodes within k hops of a seed)
constexpr int LK = 8;                  // max walk length
constexpr int kWarps = 8;

// walks[i][v] = number of (i+1)-step walks starting at v; one CTA per graph (the steps need a graph-wide barrier)
__global__ void __launch_bounds__(128)
logm_walks_kernel(const int32_t* __restrict__ graph_ptr, const int32_t* __restrict__ indptr,
                  const int32_t* __restrict__ indices, int N, int k, float* __restrict__ walks) {
  const int g = blockIdx.x;
  const int v0 = graph_ptr[g], v1 = graph_ptr[g + 1];
  for (int v = v0 + threadIdx.x; v < v1; v += blockDim.x) walks[v] = (float)(indptr[v + 1] - indptr[v]);
  for (int i = 1; i < k; ++i) {
    __syncthreads();
    const float* prev = walks + (size_t)(i - 1) * N;
    float* cur = walks + (size_t)i * N;
    for (int v = v0 + threadIdx.x; v < v1; v += blockDim.x) {
      float s = 0.f;
      for (int e = indptr[v]; e < indptr[v + 1]; ++e) s += prev[indices[e]];
      cur[v] = s;
    }
  }
}

// per graph: G = Z_g^T Z_g in shared memory (thread (ty, tx) owns an H/16 x H/16 block)
template <int H>
__device__ __forceinline__ void graph_gram(const float* __restrict__ Z, int v0, int v1, float* sG) {
  constexpr int TM = H / 16;
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
  float acc[TM][TM];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TM; ++j) acc[i][j] = 0.f;
  for (int r = v0; r < v1; ++r) {
    float av[TM], bv[TM];
#pragma unroll
    for (int q = 0; q < TM; q += 4) {
      const float4 a = ldg4(Z + (size_t)r * H + ty * TM + q), b = ldg4(Z + (size_t)r * H + tx * TM + q);
      av[q] = a.x; av[q + 1] = a.y; av[q + 2] = a.z; av[q + 3] = a.w;
      bv[q] = b.x; bv[q + 1] = b.y; bv[q + 2] = b.z; bv[q + 3] = b.w;
    }
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
      for (int j = 0; j < TM; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
  }
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TM; ++j) sG[(ty * TM + i) * H + tx * TM + j] = acc[i][j];
}

// the H x H Gram matrix lives in dynamic shared memory: 16 KB at H = 64, 64 KB (opt-in) at H = 128
template <int H>
constexpr int gram_smem_bytes() { return H * H * (int)sizeof(float); }

template <int H>
__global__ void __launch_bounds__(kThreads)
logm_gram_fwd_kernel(const float* __restrict__ Z, const int32_t* __restrict__ graph_ptr, float* __restrict__ gram) {
  extern __shared__ float sG[];
  __shared__ float s_red[kThreads / 32];
  const int g = blockIdx.x;
  const int v0 = graph_ptr[g], v1 = graph_ptr[g + 1];
  graph_gram<H>(Z, v0, v1, sG);
  __syncthreads();
  float s = 0.f;
  for (int i = threadIdx.x; i < H * H; i += kThreads) s = fmaf(sG[i], sG[i], s);
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < kThreads / 32; ++w) t += s_red[w];
    const float n = (float)(v1 - v0);
    gram[g] = t / (n * n);
  }
}

// gZ_g = scale * (4 / n^2) Z_g G_g   (overwrites gZ; logm_pair_bwd adds the sparse part afterwards)
template <int H>
__global__ void __launch_bounds__(kThreads)
logm_gram_bwd_kernel(const float* __restrict__ Z, const int32_t* __restrict__ graph_ptr, float scale, float* __restrict__ gZ) {
  extern __shared__ float sG[];
  const int g = blockIdx.x;
  const int v0 = graph_ptr[g], v1 = graph_ptr[g + 1];
  graph_gram<H>(Z, v0, v1, sG);
  __syncthreads();
  const float n = (float)(v1 - v0);
  const float f = scale * 4.f / (n * n);
  const int c = threadIdx.x & (H - 1);
  for (int r = v0 + threadIdx.x / H; r < v1; r += kThreads / H) {
    const float* z = Z + (size_t)r * H;
    float s = 0.f;
#pragma unroll 8
    for (int q = 0; q < H; ++q) s = fmaf(__ldg(z + q), sG[q * H + c], s);
    gZ[(size_t)r * H + c] = f * s;
  }
}

// k-hop ball of seed v (BFS order, then rank-sorted ascending) in `sorted`; returns its size (0 on overflow)
__device__ __forceinline__ int sorted_ball(const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices, int v, int k,
                                           int* ball, int* sorted, int lane, int32_t* status) {
  int m = 1;
  if (lane == 0) ball[0] = v;
  __syncwarp();
  int fb = 0, fe = 1;
  bool overflow = false;
  for (int hop = 0; hop < k && fb < fe && !overflow; ++hop) {
    for (int f = fb; f < fe && !overflow; ++f) {
      const int u = ball[f];
      const int e0 = __ldg(indptr + u), e1 = __ldg(indptr + u + 1);
      for (int eb = e0; eb < e1; eb += 32) {
        const int e = eb + lane;
        const int w = (e < e1) ? __ldg(indices + e) : -1;
        bool isnew = (w >= 0);
        if (isnew)
          for (int i = 0; i < m; ++i)
            if (ball[i] == w) { isnew = false; break; }
        const unsigned mask = __ballot_sync(0xffffffffu, isnew);
        const int pos = m + __popc(mask & ((1u << lane) - 1u));
        if (isnew && pos < LCAP) ball[pos] = w;
        m += __popc(mask);
        if (m > LCAP) { overflow = true; }
        __syncwarp();
        if (overflow) break;
      }
    }
    fb = fe;
    fe = min(m, LCAP);
  }
  if (overflow) { if (lane == 0) atomicExch(status, 1); return 0; }
  for (int i = lane; i < m; i += 32) {
    const int val = ball[i];
    int rank = 0;
    for (int j = 0; j < m; ++j) rank += (ball[j] < val);
    sorted[rank] = val;
  }
  __syncwarp();
  return m;
}

__device__ __forceinline__ int find_pos(const int* sorted, int m, int w) {
  int lo = 0, hi = m;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (sorted[mid] < w) lo = mid + 1; else hi = mid;
  }
  return (lo < m && sorted[lo] == w) ? lo : -1;
}

__device__ __forceinline__ int graph_of(const int32_t* __restrict__ graph_ptr, int B, int v) {   // graph_ptr[g] <= v < graph_ptr[g+1]
  int lo = 0, hi = B;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(graph_ptr + mid) <= v) lo = mid; else hi = mid;
  }
  return lo;
}

struct LogmPairArgs {
  const float* Z; const int32_t *graph_ptr, *indptr, *indices; int B, N, k;
  const float* walks;        // [k][N]
  float* pair;               // fwd: [N] per-seed term
  float* gZ; float scale;    // bwd: gZ_r += ...
  int32_t* status;
};

// A lane's H / 32 channels of a Z row: float2 at H = 64, float4 at H = 128.
template <int H> struct LaneZ;
template <> struct LaneZ<64> {
  float2 v;
  __device__ __forceinline__ static LaneZ load(const float* p) { return {*reinterpret_cast<const float2*>(p)}; }
  __device__ __forceinline__ void store(float* p) const { *reinterpret_cast<float2*>(p) = v; }
  __device__ __forceinline__ float dot(const LaneZ& o) const { return v.x * o.v.x + v.y * o.v.y; }
  __device__ __forceinline__ void fma(float f, const LaneZ& z) { v.x = fmaf(f, z.v.x, v.x); v.y = fmaf(f, z.v.y, v.y); }
};
template <> struct LaneZ<128> {
  float4 v;
  __device__ __forceinline__ static LaneZ load(const float* p) { return {*reinterpret_cast<const float4*>(p)}; }
  __device__ __forceinline__ void store(float* p) const { *reinterpret_cast<float4*>(p) = v; }
  __device__ __forceinline__ float dot(const LaneZ& o) const { return (v.x * o.v.x + v.y * o.v.y) + (v.z * o.v.z + v.w * o.v.w); }
  __device__ __forceinline__ void fma(float f, const LaneZ& z) {
    v.x = fmaf(f, z.v.x, v.x); v.y = fmaf(f, z.v.y, v.y); v.z = fmaf(f, z.v.z, v.z); v.w = fmaf(f, z.v.w, v.w);
  }
};

// One warp per seed r.  x[i][a] = (A^i)[r][sorted[a]] by dynamic programming on the ball (a neighbour outside the ball is
// further than k hops from r, so its count is 0 for every step that matters).
template <bool BWD, int H>
__global__ void __launch_bounds__(kWarps * 32, H == 64 ? 0 : 4)
logm_pair_kernel(LogmPairArgs p) {
  using LZ = LaneZ<H>;
  __shared__ int s_ball[kWarps][LCAP];
  __shared__ int s_sorted[kWarps][LCAP];
  __shared__ float s_x[kWarps][2][LCAP];
  __shared__ float s_coef[kWarps][LCAP];     // fwd: sum_i L_i[r][c] ; bwd: sum_i (L_i[r][c] + L_i[c][r])
  __shared__ float s_l2[kWarps][LCAP];       // fwd: sum_i L_i[r][c]^2
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c2 = (H / 32) * lane;
  for (int r = blockIdx.x * kWarps + warp; r < p.N; r += gridDim.x * kWarps) {
    const int m = sorted_ball(p.indptr, p.indices, r, p.k, s_ball[warp], s_sorted[warp], lane, p.status);
    const int g = graph_of(p.graph_ptr, p.B, r);
    const float n = (float)(__ldg(p.graph_ptr + g + 1) - __ldg(p.graph_ptr + g));
    const int* sorted = s_sorted[warp];
    float* coef = s_coef[warp];
    float* l2 = s_l2[warp];
    for (int a = lane; a < m; a += 32) { s_x[warp][0][a] = (sorted[a] == r) ? 1.f : 0.f; coef[a] = 0.f; l2[a] = 0.f; }
    __syncwarp();
    for (int i = 0; i < p.k; ++i) {
      const float* xp = s_x[warp][i & 1];
      float* xc = s_x[warp][(i + 1) & 1];
      const float wr = __ldg(p.walks + (size_t)i * p.N + r);
      for (int a = lane; a < m; a += 32) {
        const int c = sorted[a];
        float s = 0.f;
        for (int e = __ldg(p.indptr + c); e < __ldg(p.indptr + c + 1); ++e) {
          const int pos = find_pos(sorted, m, __ldg(p.indices + e));
          if (pos >= 0) s += xp[pos];
        }
        xc[a] = s;
        if (s > 0.f) {
          const float wc = __ldg(p.walks + (size_t)i * p.N + c);
          const float lrc = fmaxf(logf(n * s / wc), 0.f);                 // L_i[r][c]: column c is normalised by walks_i(c)
          if (BWD) {
            const float lcr = fmaxf(logf(n * s / wr), 0.f);               // L_i[c][r] = log(n (A^i)[c][r] / walks_i(r)), A^i symmetric
            coef[a] += lrc + lcr;
          } else {
            coef[a] += lrc;
            l2[a] = fmaf(lrc, lrc, l2[a]);
          }
        }
      }
      __syncwarp();
    }
    const LZ zr = LZ::load(p.Z + (size_t)r * H + c2);
    if (BWD) {
      LZ acc{};
      for (int a = 0; a < m; ++a) {
        const float cf = coef[a];
        if (cf == 0.f) continue;
        acc.fma(cf, LZ::load(p.Z + (size_t)sorted[a] * H + c2));
      }
      const float f = -2.f * p.scale / ((float)p.k * n * n);
      float* dst = p.gZ + (size_t)r * H + c2;
      LZ cur = LZ::load(dst);
      cur.fma(f, acc);
      cur.store(dst);
    } else {
      float t = 0.f;                                                      // sum_c ( -2 (z_r . z_c) sum_i L + sum_i L^2 )
      for (int a = 0; a < m; ++a) {
        const float cf = coef[a];
        if (cf == 0.f) continue;
        const float h = warp_sum(zr.dot(LZ::load(p.Z + (size_t)sorted[a] * H + c2)));
        t += fmaf(-2.f * h, cf, l2[a]);
      }
      if (lane == 0) p.pair[r] = t / (n * n);
    }
    __syncwarp();
  }
}

// loss = sum_g gram[g] + (1/k) sum_r pair[r]     (one CTA, fp64, fixed order)
__global__ void __launch_bounds__(kThreads)
logm_reduce_kernel(const float* __restrict__ gram, int B, const float* __restrict__ pair, int N, int k, float* __restrict__ out) {
  __shared__ double s_a[kThreads];
  double a = 0.0, b = 0.0;
  for (int i = threadIdx.x; i < B; i += kThreads) a += (double)gram[i];
  for (int i = threadIdx.x; i < N; i += kThreads) b += (double)pair[i];
  s_a[threadIdx.x] = a + b / (double)k;
  __syncthreads();
  for (int o = kThreads / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) s_a[threadIdx.x] += s_a[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = (float)s_a[0];
}

}  // namespace

int logm_max_steps() { return LK; }

template <int H>
static void launch_logm_fwd_t(const float* Z, const int32_t* graph_ptr, const int32_t* indptr, const int32_t* indices, int B, int N,
                              int k, float* walks, float* gram, float* pair, float* loss_out, int32_t* status, cudaStream_t s) {
  static bool once = (cudaFuncSetAttribute(logm_gram_fwd_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, gram_smem_bytes<H>()), true);
  (void)once;
  logm_walks_kernel<<<B, 128, 0, s>>>(graph_ptr, indptr, indices, N, k, walks);
  logm_gram_fwd_kernel<H><<<B, kThreads, gram_smem_bytes<H>(), s>>>(Z, graph_ptr, gram);
  LogmPairArgs a{Z, graph_ptr, indptr, indices, B, N, k, walks, pair, nullptr, 0.f, status};
  const int grid = min((N + kWarps - 1) / kWarps, 16 * num_sms());
  logm_pair_kernel<false, H><<<grid, kWarps * 32, 0, s>>>(a);
  logm_reduce_kernel<<<1, kThreads, 0, s>>>(gram, B, pair, N, k, loss_out);
}

template <int H>
static void launch_logm_bwd_t(const float* Z, const int32_t* graph_ptr, const int32_t* indptr, const int32_t* indices, int B, int N,
                              int k, const float* walks, float scale, float* gZ, int32_t* status, cudaStream_t s) {
  static bool once = (cudaFuncSetAttribute(logm_gram_bwd_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, gram_smem_bytes<H>()), true);
  (void)once;
  logm_gram_bwd_kernel<H><<<B, kThreads, gram_smem_bytes<H>(), s>>>(Z, graph_ptr, scale, gZ);
  LogmPairArgs a{Z, graph_ptr, indptr, indices, B, N, k, walks, nullptr, gZ, scale, status};
  const int grid = min((N + kWarps - 1) / kWarps, 16 * num_sms());
  logm_pair_kernel<true, H><<<grid, kWarps * 32, 0, s>>>(a);
}

void launch_logm_fwd(const float* Z, const int32_t* graph_ptr, const int32_t* indptr, const int32_t* indices, int B, int N,
                     int k, float* walks, float* gram, float* pair, float* loss_out, int32_t* status, int hidden, cudaStream_t s) {
  if (hidden == 64) launch_logm_fwd_t<64>(Z, graph_ptr, indptr, indices, B, N, k, walks, gram, pair, loss_out, status, s);
  else launch_logm_fwd_t<128>(Z, graph_ptr, indptr, indices, B, N, k, walks, gram, pair, loss_out, status, s);
}

void launch_logm_bwd(const float* Z, const int32_t* graph_ptr, const int32_t* indptr, const int32_t* indices, int B, int N,
                     int k, const float* walks, float scale, float* gZ, int32_t* status, int hidden, cudaStream_t s) {
  if (hidden == 64) launch_logm_bwd_t<64>(Z, graph_ptr, indptr, indices, B, N, k, walks, scale, gZ, status, s);
  else launch_logm_bwd_t<128>(Z, graph_ptr, indptr, indices, B, N, k, walks, scale, gZ, status, s);
}

}  // namespace scgib
