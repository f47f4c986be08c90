// gin_kernels.cu - input projection and the GIN encoder (forward + backward) as fused row-tile kernels.
//
// Reference call sites replaced (paths relative to the reference tree):
//   F.normalize + transfer_d        exp_pretraining.py:312-314, models.py:668-669
//   GIN.forward                     models.py:66-72   (DGL GINConv 'sum', eps = 0 buffer; MLP models.py:38-49;
//                                                      BatchNorm1d train mode over all rows; ReLU)
// One forward launch per GINConv layer:
//   gather-aggregate (CSR segmented reduce, float4 lanes, BN+ReLU of the previous layer applied on load)
//   -> 2-GEMM MLP out of shared memory -> y (pre-BN) + per-tile (mean, M2) -> last CTA finalises the batch
//   statistics (Chan combine in fp64, fixed order) and the running-stat EMA.
// Backward per layer: `gin_bwd_pre` (gather of the upstream gradient, ReLU/BN mask, d gamma / d beta with an
// in-kernel deterministic finalise) then `gin_bwd_main` (BN backward, 4 tile GEMMs: g_r, g_a, dW2, dW1).
#include <stdlib.h>
#include "kernels.cuh"

namespace scgib {

// ------------------------------------------------------------------------------------------------
// x_hat = x / max(||x||_2, 1e-12);  t = x_hat Wt^T          (Wt [DT][F], F <= FMAX, DT = 32, 64 or 128)
// The row norm and each output are sequential sums over f = 0..F-1, whatever FMAX: FMAX only sizes the weight copy.
// The outputs are computed in passes over 32-column groups (kProjGroup): the weight copy holds one group, so it stays
// within the static shared-memory limit at F = 128, DT = 128, and DT = 32 is the single pass it always was.
// ------------------------------------------------------------------------------------------------
constexpr int kProjGroup = 32;

// the rows [v0, N) step vstep of one 32-column output group g0 of a projection CTA (s_w: this group's weights, [f][o])
template <bool OUT_BF16>
__device__ __forceinline__ void input_proj_rows(const float* __restrict__ x, const float* s_w, int v0, int vstep, int N, int F,
                                                int DT, int g0, int normalize, float* __restrict__ t) {
  const int q = threadIdx.x & 7;  // output quad
  for (int v = v0 + (threadIdx.x >> 3); v < N; v += vstep) {
    const float* xr = x + (size_t)v * F;
    float ss = 0.f;
    for (int f = 0; f < F; ++f) { const float a = __ldg(xr + f); ss = fmaf(a, a, ss); }
    const float inv = normalize ? 1.f / fmaxf(sqrtf(ss), 1e-12f) : 1.f;
    float4 acc = make4(0.f);
    for (int f = 0; f < F; ++f) {
      const float a = __ldg(xr + f) * inv;
      const float4 w = ld4(s_w + f * kProjGroup + q * 4);
      acc.x = fmaf(a, w.x, acc.x); acc.y = fmaf(a, w.y, acc.y); acc.z = fmaf(a, w.z, acc.z); acc.w = fmaf(a, w.w, acc.w);
    }
    st4a<OUT_BF16>(t, (size_t)v * DT + g0 + q * 4, acc);
  }
}
__device__ __forceinline__ void stage_proj_group(float* s_w, const float* __restrict__ Wt, int F, int g0) {
  for (int i = threadIdx.x; i < F * kProjGroup; i += kThreads) {
    const int o = i / F, f = i % F;
    s_w[f * kProjGroup + o] = Wt[(size_t)g0 * F + i];
  }
}

template <bool OUT_BF16, int FMAX>
__global__ void __launch_bounds__(kThreads)
input_proj_fwd_kernel(const float* __restrict__ x, const float* __restrict__ Wt, int N, int F, int DT, int normalize,
                      float* __restrict__ t) {
  pdl_sync();
  __shared__ __align__(16) float s_w[FMAX * kProjGroup];  // [f][o]
  for (int g0 = 0; g0 < DT; g0 += kProjGroup) {
    if (g0 > 0) __syncthreads();     // every reader of the previous group's weights is done
    stage_proj_group(s_w, Wt, F, g0);
    __syncthreads();
    input_proj_rows<OUT_BF16>(x, s_w, blockIdx.x * (kThreads / 8), gridDim.x * (kThreads / 8), N, F, DT, g0, normalize, t);
  }
}

// out_bf16: t is bf16 storage (bf16 mode: the layer-0 input of the GIN encoders)
void launch_input_proj_fwd(const float* x, const float* Wt, int N, int F, int DT, int normalize, float* t, cudaStream_t s, bool out_bf16) {
  const int grid = min((N + 31) / 32, 148 * 8);
  if (F <= 32) {
    if (out_bf16) launch_k((input_proj_fwd_kernel<true, 32>), dim3(grid), dim3(kThreads), 0, s, x, Wt, N, F, DT, normalize, t);
    else launch_k((input_proj_fwd_kernel<false, 32>), dim3(grid), dim3(kThreads), 0, s, x, Wt, N, F, DT, normalize, t);
  } else {
    if (out_bf16) launch_k((input_proj_fwd_kernel<true, kMaxInDim>), dim3(grid), dim3(kThreads), 0, s, x, Wt, N, F, DT, normalize, t);
    else launch_k((input_proj_fwd_kernel<false, kMaxInDim>), dim3(grid), dim3(kThreads), 0, s, x, Wt, N, F, DT, normalize, t);
  }
}

// ------------------------------------------------------------------------------------------------
// The parameter-only prologue of a step in ONE launch (three independent jobs, CTA ranges): input projection
// (CTAs [0, nproj)), the k-major weight copies of the FFMA kernels (one CTA per job) and the head backward's operand
// preparation (8 CTAs: W1a = W1[:, :H], W1b = W1[:, H:], identity BatchNorm-backward constants).
// ------------------------------------------------------------------------------------------------
// one thread per row of {parent rows, ego rows}: xagg_v = x_hat[p(v)] + sum_{u in N(v)} x_hat[p(u)], FC >= F columns in registers
template <int FC>
__device__ __forceinline__ void xagg_rows(const FwdPrepArgs& p, int cta) {
  const int V0 = p.xa_V[0], V1 = p.xa_V[1], F = p.F;
  for (int i = cta * kThreads + threadIdx.x; i < V0 + V1; i += p.nxagg * kThreads) {
    const int set = i < V0 ? 0 : 1, v = set == 0 ? i : i - V0;
    const int32_t* indices = p.xa_indices[set];
    const int32_t* map = set == 0 ? nullptr : p.xa_map;
    const int32_t* ip = p.xa_indptr[set];          // null: the row itself only (x_hat[p(v)])
    const int e0 = ip ? __ldg(ip + v) : 0, e1 = ip ? __ldg(ip + v + 1) : 0;
    float acc[FC];
#pragma unroll
    for (int f = 0; f < FC; ++f) acc[f] = 0.f;
    for (int e = e0 - 1; e < e1; ++e) {          // e0 - 1: the row itself
      const int u = e < e0 ? v : __ldg(indices + e);
      const float* xr = p.xa_x + (size_t)(map ? __ldg(map + u) : u) * F;
      float xv[FC];
      float ss = 0.f;
#pragma unroll
      for (int f = 0; f < FC; ++f) { xv[f] = f < F ? __ldg(xr + f) : 0.f; ss = fmaf(xv[f], xv[f], ss); }
      const float inv = p.normalize ? 1.f / fmaxf(sqrtf(ss), 1e-12f) : 1.f;
#pragma unroll
      for (int f = 0; f < FC; ++f) acc[f] = fmaf(xv[f], inv, acc[f]);
    }
    float* d = p.xagg[set] + (size_t)v * p.xa_stride;
#pragma unroll
    for (int f = 0; f < FC; f += 4)
      if (f < p.xa_stride) st4(d + f, make_float4(acc[f], acc[f + 1], acc[f + 2], acc[f + 3]));
  }
}

// F > 32: one warp per row, lane l holds the columns l, l + 32, l + 64, l + 96 (coalesced loads, four accumulators).
// The norm of a neighbour row is the lane partials summed by a butterfly: the same fixed order on every lane and run.
__device__ __forceinline__ void xagg_rows_wide(const FwdPrepArgs& p, int cta) {
  constexpr int NC = kMaxInDim / 32;
  const int V0 = p.xa_V[0], V1 = p.xa_V[1], F = p.F;
  const int lane = threadIdx.x & 31, wpc = kThreads / 32;
  for (int i = cta * wpc + (threadIdx.x >> 5); i < V0 + V1; i += p.nxagg * wpc) {
    const int set = i < V0 ? 0 : 1, v = set == 0 ? i : i - V0;
    const int32_t* indices = p.xa_indices[set];
    const int32_t* map = set == 0 ? nullptr : p.xa_map;
    const int32_t* ip = p.xa_indptr[set];
    const int e0 = ip ? __ldg(ip + v) : 0, e1 = ip ? __ldg(ip + v + 1) : 0;
    float acc[NC];
#pragma unroll
    for (int c = 0; c < NC; ++c) acc[c] = 0.f;
    for (int e = e0 - 1; e < e1; ++e) {          // e0 - 1: the row itself
      const int u = e < e0 ? v : __ldg(indices + e);
      const float* xr = p.xa_x + (size_t)(map ? __ldg(map + u) : u) * F;
      float xv[NC];
      float ss = 0.f;
#pragma unroll
      for (int c = 0; c < NC; ++c) { const int f = lane + 32 * c; xv[c] = f < F ? __ldg(xr + f) : 0.f; ss = fmaf(xv[c], xv[c], ss); }
      ss = warp_sum(ss);
      const float inv = p.normalize ? 1.f / fmaxf(sqrtf(ss), 1e-12f) : 1.f;
#pragma unroll
      for (int c = 0; c < NC; ++c) acc[c] = fmaf(xv[c], inv, acc[c]);
    }
    float* d = p.xagg[set] + (size_t)v * p.xa_stride;
#pragma unroll
    for (int c = 0; c < NC; ++c)
      if (lane + 32 * c < p.xa_stride) d[lane + 32 * c] = acc[c];
  }
}

// FMAX: 32 for F <= 32, kMaxInDim above (the weight copy of the projection CTAs and the xagg row scheme)
template <bool OUT_BF16, int FMAX>
__global__ void __launch_bounds__(kThreads) fwd_prep_kernel(FwdPrepArgs p) {
  pdl_sync();
  __shared__ __align__(16) float s_w[FMAX * kProjGroup];  // [f][o] of one 32-column output group
  int b = (int)blockIdx.x;
  if (b < p.nxagg) {
    if constexpr (FMAX > 32) xagg_rows_wide(p, b);
    else if (p.F <= 12) xagg_rows<12>(p, b);
    else xagg_rows<32>(p, b);
    return;
  }
  b -= p.nxagg;
  if (b < p.nproj) {
    for (int g0 = 0; g0 < p.DT; g0 += kProjGroup) {
      if (g0 > 0) __syncthreads();
      stage_proj_group(s_w, p.Wt, p.F, g0);
      __syncthreads();
      input_proj_rows<OUT_BF16>(p.x, s_w, b * (kThreads / 8), p.nproj * (kThreads / 8), p.N, p.F, p.DT, g0, p.normalize, p.t);
    }
    return;
  }
  if (b < p.nproj + p.jobs.n) {
    const TransposeJob j = p.jobs.job[b - p.nproj];
    for (int i = threadIdx.x; i < j.rows * j.cols; i += kThreads) {
      const int c = i / j.rows, r = i % j.rows;   // consecutive threads write consecutive dst elements
      j.dst[(size_t)c * j.rows + r] = __ldg(j.src + (size_t)r * j.cols + c);
    }
    return;
  }
  const int hb = b - p.nproj - p.jobs.n, H = p.hid;      // head backward prep, 8 CTAs
  for (int i = hb * kThreads + threadIdx.x; i < H * 2 * H; i += 8 * kThreads) {
    const int o = i / (2 * H), k = i % (2 * H);
    const float w = __ldg(p.headW1 + i);
    if (k < H) p.W1a[o * H + k] = w; else p.W1b[o * H + k - H] = w;
  }
  if (hb == 0) {
    for (int i = threadIdx.x; i < 4 * H; i += kThreads) p.bn[i] = (i >= H && i < 3 * H) ? 1.f : 0.f;   // mean 0, rstd 1, gamma 1, beta 0
    for (int i = threadIdx.x; i < 2 * H; i += kThreads) p.cvec[i] = 0.f;
  }
}
void launch_fwd_prep(FwdPrepArgs a, cudaStream_t s, bool out_bf16) {
  a.nproj = a.x ? min((a.N + 31) / 32, 148 * 8) : 0;
  const bool wide = a.F > 32;
  const int rows_per_cta = wide ? kThreads / 32 : kThreads;     // xagg: a warp per row (wide) or a thread per row
  a.nxagg = (a.xa_x && a.xagg[0]) ? min((a.xa_V[0] + a.xa_V[1] + rows_per_cta - 1) / rows_per_cta, 148 * 8) : 0;
  const int grid = a.nxagg + a.nproj + a.jobs.n + (a.headW1 ? 8 : 0);
  if (grid == 0) return;
  if (wide) {
    if (out_bf16) launch_k((fwd_prep_kernel<true, kMaxInDim>), dim3(grid), dim3(kThreads), 0, s, a);
    else launch_k((fwd_prep_kernel<false, kMaxInDim>), dim3(grid), dim3(kThreads), 0, s, a);
  } else {
    if (out_bf16) launch_k((fwd_prep_kernel<true, 32>), dim3(grid), dim3(kThreads), 0, s, a);
    else launch_k((fwd_prep_kernel<false, 32>), dim3(grid), dim3(kThreads), 0, s, a);
  }
}

template <bool VEC>      // VEC: float4 loads (x 16-byte aligned, n a multiple of 4)
__global__ void __launch_bounds__(kThreads) absmax_kernel(const float* __restrict__ x, size_t n, unsigned int* __restrict__ slot) {
  pdl_sync();
  float m = 0.f;
  for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < (VEC ? n / 4 : n); i += (size_t)gridDim.x * kThreads) {
    if (VEC) {
      const float4 v = ld4(x + 4 * i);
      m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
    } else {
      m = fmaxf(m, fabsf(x[i]));
    }
  }
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(slot, __float_as_uint(m));
}
void launch_absmax(const float* x, size_t n, unsigned int* slot, cudaStream_t s) {
  const bool vec = (n & 3) == 0 && ((uintptr_t)x & 15u) == 0;
  const size_t units = vec ? n / 4 : n;
  const int grid = (int)min((size_t)(4 * num_sms()), (units + kThreads - 1) / kThreads);
  if (units == 0) return;
  if (vec) launch_k((absmax_kernel<true>), dim3(grid), dim3(kThreads), 0, s, x, n, slot);
  else launch_k((absmax_kernel<false>), dim3(grid), dim3(kThreads), 0, s, x, n, slot);
}

__global__ void __launch_bounds__(kThreads) f32_to_bf16_kernel(const float* __restrict__ in, bf16_t* __restrict__ out, size_t n4) {
  pdl_sync();
  for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < n4; i += (size_t)gridDim.x * kThreads)
    st4a<true>(reinterpret_cast<float*>(out), 4 * i, ld4(in + 4 * i));
}
void launch_f32_to_bf16(const float* in, void* out, size_t n, cudaStream_t s) {   // n multiple of 4
  const size_t n4 = n / 4;
  const int grid = (int)min((size_t)(4 * num_sms()), (n4 + kThreads - 1) / kThreads);
  if (n4 > 0) launch_k((f32_to_bf16_kernel), dim3(grid), dim3(kThreads), 0, s, in, reinterpret_cast<bf16_t*>(out), n4);
}

__global__ void bn_from_running_kernel(const float* __restrict__ running, const float* __restrict__ gamma,
                                       const float* __restrict__ beta, float* __restrict__ bn, int HID) {
  pdl_sync();
  const int c = threadIdx.x;
  if (c >= HID) return;
  bn[c] = running[c];
  bn[HID + c] = 1.f / sqrtf(running[HID + c] + kBnEps);
  bn[2 * HID + c] = gamma[c];
  bn[3 * HID + c] = beta[c];
}
void launch_bn_from_running(const float* running, const float* gamma, const float* beta, float* bn, int hidden, cudaStream_t s) {
  launch_k((bn_from_running_kernel), dim3(1), dim3(hidden), 0, s, running, gamma, beta, bn, hidden);
}

// ------------------------------------------------------------------------------------------------
// batched transposes of small weight matrices (forward kernels want k-major copies)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) transpose_many_kernel(TransposeJobs jobs) {
  pdl_sync();
  const TransposeJob j = jobs.job[blockIdx.x];
  for (int i = threadIdx.x; i < j.rows * j.cols; i += kThreads) {
    const int c = i / j.rows, r = i % j.rows;   // consecutive threads write consecutive dst elements
    j.dst[(size_t)c * j.rows + r] = __ldg(j.src + (size_t)r * j.cols + c);
  }
}
void launch_transposes(const TransposeJobs& jobs, cudaStream_t s) {
  if (jobs.n > 0) launch_k((transpose_many_kernel), dim3(jobs.n), dim3(kThreads), 0, s, jobs);
}

// ------------------------------------------------------------------------------------------------
// GIN layer forward
// ------------------------------------------------------------------------------------------------
constexpr int GT = 128;        // rows per tile

template <int KIN, int HID>
struct GinFwdSmem {
  static constexpr int GLD = HID + 4;   // smem leading dim (row-major tiles)
  float tile[GT * GLD];        // A tile [GT][KIN+4] then R tile [GT][HID+4]
  float w1t[KIN * HID];
  float w2t[HID * HID];
  float red[16 * HID];
  float b1[HID], b2[HID], mean[HID];
  double dred[4 * HID];
};

template <int KIN, int HID>
__global__ void __launch_bounds__(kThreads, HID == 64 ? 2 : 1)
gin_fwd_kernel(GinFwdArgs p) {
  pdl_sync();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  GinFwdSmem<KIN, HID>& sm = *reinterpret_cast<GinFwdSmem<KIN, HID>*>(smem_raw);
  constexpr int GLD = HID + 4;
  constexpr int LDA = KIN + 4;
  constexpr int LPR = KIN / 4;             // lanes per row in the gather
  constexpr int RPP = kThreads / LPR;      // rows per pass
  using M = NNMap<GT, HID>;

  load_matrix<HID>(sm.w1t, HID, p.W1t, KIN);
  load_matrix<HID>(sm.w2t, HID, p.W2t, HID);
  if (threadIdx.x < HID) { sm.b1[threadIdx.x] = p.b1[threadIdx.x]; sm.b2[threadIdx.x] = p.b2[threadIdx.x]; }

  const int n_tiles = (p.V + GT - 1) / GT;
  const int gl = threadIdx.x % LPR, gr = threadIdx.x / LPR;
  Bn4 bn;
  const bool has_bn = (p.bn_in != nullptr);
  if (has_bn) bn.load(p.bn_in, gl * 4, HID);   // KIN == HID whenever a BN precedes the layer

  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int base = tile * GT;
    __syncthreads();  // previous tile's readers of sm.tile are done (also covers the weight loads)
    // ---- gather-aggregate: a_v = f(in[map(v)]) + sum_u f(in[map(u)])   (all row passes of the thread interleaved)
    {
      constexpr int NRT = GT / RPP, NR = NRT < 8 ? NRT : 8;    // row passes of the thread, at most 8 in flight together
#pragma unroll 1
      for (int j0 = 0; j0 < NRT; j0 += NR) {
        int vv[NR];
        float4 agg[NR];
#pragma unroll
        for (int j = 0; j < NR; ++j) vv[j] = base + gr + (j0 + j) * RPP;
        gather_aggregate<KIN, NR>(p.in, p.row_map, p.indptr, p.indices, p.V, vv, gl, has_bn ? &bn : nullptr, agg);
#pragma unroll
        for (int j = 0; j < NR; ++j) {
          if (p.a_out && vv[j] < p.V) st4(p.a_out + (size_t)vv[j] * KIN + gl * 4, agg[j]);
          st4(sm.tile + (gr + (j0 + j) * RPP) * LDA + gl * 4, agg[j]);
        }
      }
    }
    __syncthreads();
    // ---- u = W1 a + b1 ; r = relu(u)
    float acc[M::TM][4];
    const int c0 = M::col0(), r0 = M::row0();
#pragma unroll
    for (int m = 0; m < M::TM; ++m) { acc[m][0] = sm.b1[c0]; acc[m][1] = sm.b1[c0 + 1]; acc[m][2] = sm.b1[c0 + 2]; acc[m][3] = sm.b1[c0 + 3]; }
    gemm_nn<GT, KIN, HID>(sm.tile, LDA, sm.w1t, HID, acc);
    __syncthreads();  // everyone finished reading the A tile
#pragma unroll
    for (int m = 0; m < M::TM; ++m) {
      const float4 rv = relu4(make_float4(acc[m][0], acc[m][1], acc[m][2], acc[m][3]));
      st4(sm.tile + (r0 + m) * GLD + c0, rv);
      const int v = base + r0 + m;
      if (p.r_out && v < p.V) st4(p.r_out + (size_t)v * HID + c0, rv);
    }
    __syncthreads();
    // ---- y = W2 r + b2
#pragma unroll
    for (int m = 0; m < M::TM; ++m) { acc[m][0] = sm.b2[c0]; acc[m][1] = sm.b2[c0 + 1]; acc[m][2] = sm.b2[c0 + 2]; acc[m][3] = sm.b2[c0 + 3]; }
    gemm_nn<GT, HID, HID>(sm.tile, GLD, sm.w2t, HID, acc);
    float ps[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int m = 0; m < M::TM; ++m) {
      const int v = base + r0 + m;
      if (v < p.V) {
        st4(p.y_out + (size_t)v * HID + c0, make_float4(acc[m][0], acc[m][1], acc[m][2], acc[m][3]));
        ps[0] += acc[m][0]; ps[1] += acc[m][1]; ps[2] += acc[m][2]; ps[3] += acc[m][3];
      }
    }
    // ---- per-tile column mean and centred second moment
    const int cnt = min(GT, p.V - base);
    st4(sm.red + M::tr() * HID + c0, make_float4(ps[0], ps[1], ps[2], ps[3]));
    __syncthreads();
    if (threadIdx.x < HID) {
      float s = 0.f;
#pragma unroll
      for (int g = 0; g < M::RG; ++g) s += sm.red[g * HID + threadIdx.x];
      sm.mean[threadIdx.x] = s / (float)cnt;
    }
    __syncthreads();
    {
      const float4 mu = ld4(sm.mean + c0);
      ps[0] = ps[1] = ps[2] = ps[3] = 0.f;
#pragma unroll
      for (int m = 0; m < M::TM; ++m) {
        if (base + r0 + m < p.V) {
          float d;
          d = acc[m][0] - mu.x; ps[0] = fmaf(d, d, ps[0]);
          d = acc[m][1] - mu.y; ps[1] = fmaf(d, d, ps[1]);
          d = acc[m][2] - mu.z; ps[2] = fmaf(d, d, ps[2]);
          d = acc[m][3] - mu.w; ps[3] = fmaf(d, d, ps[3]);
        }
      }
      st4(sm.red + M::tr() * HID + c0, make_float4(ps[0], ps[1], ps[2], ps[3]));
    }
    __syncthreads();
    if (threadIdx.x < HID) {
      float s = 0.f;
#pragma unroll
      for (int g = 0; g < M::RG; ++g) s += sm.red[g * HID + threadIdx.x];
      p.part[(size_t)tile * 2 * HID + threadIdx.x] = sm.mean[threadIdx.x];
      p.part[(size_t)tile * 2 * HID + HID + threadIdx.x] = s;
    }
  }
  // ---- batch statistics: last CTA combines the per-tile (n, mean, M2) in fp64, fixed order
  if (!last_cta_arrives(p.counter)) return;
  constexpr int NSEG = kThreads / HID;     // interleaved segments per column (4 at HID = 64, 2 at HID = 128)
  const int c = threadIdx.x % HID, seg = threadIdx.x / HID;
  double s = 0.0;
  for (int t = seg; t < n_tiles; t += NSEG) {
    const double n = (double)min(GT, p.V - t * GT);
    s += n * (double)__ldcg(p.part + (size_t)t * 2 * HID + c);
  }
  sm.dred[seg * HID + c] = s;
  __syncthreads();
  double msum = 0.0;
#pragma unroll
  for (int g = 0; g < NSEG; ++g) msum += sm.dred[g * HID + c];
  const double mean = msum / (double)p.V;
  __syncthreads();
  double q = 0.0;
  for (int t = seg; t < n_tiles; t += NSEG) {
    const double n = (double)min(GT, p.V - t * GT);
    const double d = (double)__ldcg(p.part + (size_t)t * 2 * HID + c) - mean;
    q += (double)__ldcg(p.part + (size_t)t * 2 * HID + HID + c) + n * d * d;
  }
  sm.dred[seg * HID + c] = q;
  __syncthreads();
  if (threadIdx.x < HID) {
    double qsum = 0.0;
#pragma unroll
    for (int g = 0; g < NSEG; ++g) qsum += sm.dred[g * HID + c];
    const double var = qsum / (double)p.V;
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

int gin_fwd_grid(int V) {
  const int n_tiles = (V + GT - 1) / GT;
  return min(n_tiles, 2 * num_sms());
}

template <int KIN, int H>
static void launch_gin_fwd_t(const GinFwdArgs& a, cudaStream_t s) {
  static bool once = (cudaFuncSetAttribute(gin_fwd_kernel<KIN, H>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)sizeof(GinFwdSmem<KIN, H>)), true);
  (void)once;
  const int n_tiles = (a.V + GT - 1) / GT;
  const int grid = min(n_tiles, (H == 64 ? 2 : 1) * num_sms());
  launch_k((gin_fwd_kernel<KIN, H>), dim3(grid), dim3(kThreads), sizeof(GinFwdSmem<KIN, H>), s, a);
}
void launch_gin_fwd(const GinFwdArgs& a, int kin, int hidden, cudaStream_t s) {
  if (hidden == 64) { if (kin == 32) launch_gin_fwd_t<32, 64>(a, s); else launch_gin_fwd_t<64, 64>(a, s); }
  else if (kin == 32) launch_gin_fwd_t<32, 128>(a, s);
  else if (kin == 64) launch_gin_fwd_t<64, 128>(a, s);        // layer 0 at d_transfer 64
  else launch_gin_fwd_t<128, 128>(a, s);
}

// ------------------------------------------------------------------------------------------------
// GIN layer backward, part 1: upstream gradient of h' = relu(BN(y)), ReLU mask, d gamma / d beta
//   mode CSR   : G_v = Ga_v + sum_{u in N(v)} Ga_u      (A symmetric => gather form, no atomics)
//   mode direct: G_v = src[map ? map[v] : v]
//   g_o = G * [gamma*yhat+beta > 0] ; dbeta = sum g_o ; dgamma = sum g_o*yhat
// Last CTA: dgamma/dbeta -> grads, and the BN-backward constants c1 = gamma*dbeta/V, c2 = gamma*dgamma/V.
// ------------------------------------------------------------------------------------------------
template <int HID, int MINB>
__global__ void __launch_bounds__(kThreads, MINB)
gin_bwd_pre_kernel(GinBwdPrePair pp) {
  pdl_sync();
  const bool second = (int)blockIdx.x >= pp.split;
  const GinBwdPreArgs& p = pp.a[second ? 1 : 0];
  const int bid = second ? (int)blockIdx.x - pp.split : (int)blockIdx.x;          // CTA index / count inside its problem
  const int nblk = second ? (int)gridDim.x - pp.split : pp.split;
  constexpr int LPR = HID / 4, RPC = kThreads / LPR;       // lanes per row (4 channels each), rows per CTA pass
  __shared__ __align__(16) float s_red[RPC * 2 * HID];
  __shared__ double s_d[kThreads];
  const int l = threadIdx.x % LPR, hw = threadIdx.x / LPR;
  Bn4 bn;
  bn.load(p.bn, l * 4, HID);
  float4 db = make4(0.f), dg = make4(0.f);
  float gm = 0.f;
  constexpr int NR = 4;
  for (int v0 = bid * RPC + hw; v0 < p.V; v0 += nblk * RPC * NR) {
    int vv[NR];
    float4 g[NR];
#pragma unroll
    for (int j = 0; j < NR; ++j) vv[j] = v0 + j * nblk * RPC;
    float4 y[NR];   // issued first: independent of the gather's dependent index chain
#pragma unroll
    for (int j = 0; j < NR; ++j) y[j] = vv[j] < p.V ? ld4_cs(p.y + (size_t)vv[j] * HID + l * 4) : make4(0.f);
    if (p.indptr) {
      gather_aggregate<HID, NR>(p.src, nullptr, p.indptr, p.indices, p.V, vv, l, nullptr, g);
    } else {
#pragma unroll
      for (int j = 0; j < NR; ++j) {
        g[j] = make4(0.f);
        if (vv[j] < p.V) g[j] = ld4(p.src + (size_t)(p.map ? __ldg(p.map + vv[j]) : vv[j]) * HID + l * 4);
      }
    }
#pragma unroll
    for (int j = 0; j < NR; ++j) {
      if (vv[j] >= p.V) continue;
      const float4 xh = bn.xhat(y[j]);
      const float4 o = bn.pre(y[j]);
      float4 gg = g[j];
      gg.x = o.x > 0.f ? gg.x : 0.f; gg.y = o.y > 0.f ? gg.y : 0.f; gg.z = o.z > 0.f ? gg.z : 0.f; gg.w = o.w > 0.f ? gg.w : 0.f;
      st4(p.g_o + (size_t)vv[j] * HID + l * 4, gg);
      gm = fmaxf(fmaxf(gm, fmaxf(fabsf(gg.x), fabsf(gg.y))), fmaxf(fabsf(gg.z), fabsf(gg.w)));
      db = add4(db, gg);
      dg.x = fmaf(gg.x, xh.x, dg.x); dg.y = fmaf(gg.y, xh.y, dg.y); dg.z = fmaf(gg.z, xh.z, dg.z); dg.w = fmaf(gg.w, xh.w, dg.w);
    }
  }
  st4(s_red + hw * 2 * HID + l * 4, db);
  st4(s_red + hw * 2 * HID + HID + l * 4, dg);
  if (p.gmax) {                  // max is order-independent: the atomic keeps the result deterministic
    gm = warp_max(gm);
    if ((threadIdx.x & 31) == 0 && gm > 0.f) atomicMax(p.gmax, __float_as_uint(gm));
  }
  __syncthreads();
  if (threadIdx.x < 2 * HID) {
    float s = 0.f;
#pragma unroll
    for (int h = 0; h < RPC; ++h) s += s_red[h * 2 * HID + threadIdx.x];
    p.part[(size_t)bid * 2 * HID + threadIdx.x] = s;
  }
  if (!last_cta_arrives(p.counter, (unsigned)nblk)) return;
  // 256 threads: column j (0..H-1 dbeta, H..2H-1 dgamma), NSEG interleaved segments, batched loads
  constexpr int NSEG = kThreads / (2 * HID);
  {
    const int j = threadIdx.x % (2 * HID), seg = threadIdx.x / (2 * HID);
    s_d[seg * 2 * HID + j] = sum_partials(p.part + j, 2 * HID, nblk, seg, NSEG);
  }
  __syncthreads();
  if (threadIdx.x < HID) {
    const int c = threadIdx.x;
    double dbeta = 0.0, dgamma = 0.0;
#pragma unroll
    for (int sg = 0; sg < NSEG; ++sg) { dbeta += s_d[sg * 2 * HID + c]; dgamma += s_d[sg * 2 * HID + HID + c]; }
    p.d_beta[c] = (float)dbeta;
    p.d_gamma[c] = (float)dgamma;
    const double gamma = (double)p.bn[2 * HID + c];
    p.cvec[c] = (float)(gamma * dbeta / (double)p.V);
    p.cvec[HID + c] = (float)(gamma * dgamma / (double)p.V);
  }
}

// resident CTAs per SM of the gather kernels: SCGIB_PRE_OCC = 2 (default) | 3 | 4.  Measured on B200 (B = 4096): 52 / 58 / 59 us
// per launch in fp32 and 42 / 63 / 68 us in bf16 - the register cap of the higher occupancies spills the rows in flight.
// Also measured and NOT kept: the CSR index chain software-pipelined one row group ahead (offsets and the first four
// neighbour ids of the next group requested while this group's rows are in flight): 63 instead of 52.6 us per launch at
// 128 registers - the kernel is bound by its L2 / DRAM traffic, not by the dependent index loads.
int gin_bwd_pre_occ() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("SCGIB_PRE_OCC"); v = (e && e[0] >= '2' && e[0] <= '4') ? e[0] - '0' : 2; }
  return v;
}
int gin_bwd_pre_grid(int V) { return min((V + 63) / 64, gin_bwd_pre_occ() * num_sms()); }
template <int H>
static void launch_pre_t(const GinBwdPrePair& pp, int grid, cudaStream_t s) {
  const int occ = gin_bwd_pre_occ();
  if (occ == 2) launch_k((gin_bwd_pre_kernel<H, 2>), dim3(grid), dim3(kThreads), 0, s, pp);
  else if (occ == 3) launch_k((gin_bwd_pre_kernel<H, 3>), dim3(grid), dim3(kThreads), 0, s, pp);
  else launch_k((gin_bwd_pre_kernel<H, 4>), dim3(grid), dim3(kThreads), 0, s, pp);
}

void launch_gin_bwd_pre(const GinBwdPreArgs& a, int hidden, cudaStream_t s) {
  GinBwdPrePair pp;
  pp.a[0] = a; pp.a[1] = a;
  const int grid = gin_bwd_pre_grid(a.V);
  pp.split = grid;
  if (hidden == 64) launch_pre_t<64>(pp, grid, s); else launch_pre_t<128>(pp, grid, s);
}

int pair_split(int grid, int work0, int work1) {
  if (grid < 2) return grid;
  int s0 = (int)(((long long)grid * work0 + (work0 + work1) / 2) / (work0 + work1));
  return max(1, min(grid - 1, s0));
}

void launch_gin_bwd_pre_pair(const GinBwdPreArgs& a0, const GinBwdPreArgs& a1, int hidden, cudaStream_t s) {
  GinBwdPrePair pp;
  pp.a[0] = a0; pp.a[1] = a1;
  const int grid = max(2, gin_bwd_pre_grid(a0.V + a1.V));
  pp.split = pair_split(grid, a0.V, a1.V);
  if (hidden == 64) launch_pre_t<64>(pp, grid, s); else launch_pre_t<128>(pp, grid, s);
}

// ------------------------------------------------------------------------------------------------
// GIN layer backward, part 2 (persistent, one CTA per SM, static tile striding => deterministic):
//   g_y = rstd * (gamma*g_o - c1 - yhat*c2)
//   g_u = (g_y W2) * [r > 0] ; g_a = g_u W1 -> Ga
//   dW2 += g_y^T r ; db2 += sum g_y ; dW1 += g_u^T a ; db1 += sum g_u     (per-CTA partials)
// ------------------------------------------------------------------------------------------------
template <int KIN, int HID, int GT>
struct GinBwdSmem {
  static constexpr int GLD = HID + 4;
  float gy[GT * GLD];
  float gu[GT * GLD];
  float r[GT * GLD];
  float a[GT * (KIN + 4)];
  float w2[HID * HID];     // natural [out][in]  = k-major for g_y W2
  float w1[HID * KIN];     // natural [out][in]  = k-major for g_u W1
};

// GT = rows per tile (128 at HID = 64; 32 at HID = 128: three [GT][HID] tiles + both weight matrices must fit 227 KB)
template <int KIN, int HID, int GT>
__global__ void __launch_bounds__(kThreads, 1)
gin_bwd_main_kernel(GinBwdMainArgs p) {
  pdl_sync();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  GinBwdSmem<KIN, HID, GT>& sm = *reinterpret_cast<GinBwdSmem<KIN, HID, GT>*>(smem_raw);
  constexpr int GLD = HID + 4;
  constexpr int LDA = KIN + 4;
  using M2 = NNMap<GT, HID>;   // g_r tile
  using M1 = NNMap<GT, KIN>;   // g_a tile
  using T2 = TNMap<HID, HID>;  // dW2
  using T1 = TNMap<HID, KIN>;  // dW1

  load_matrix<HID>(sm.w2, HID, p.W2, HID);
  load_matrix<KIN>(sm.w1, KIN, p.W1, HID);

  float dW2[T2::TO][T2::TJ], dW1[T1::TO][T1::TJ];
#pragma unroll
  for (int i = 0; i < T2::TO; ++i)
#pragma unroll
    for (int j = 0; j < T2::TJ; ++j) dW2[i][j] = 0.f;
#pragma unroll
  for (int i = 0; i < T1::TO; ++i)
#pragma unroll
    for (int j = 0; j < T1::TJ; ++j) dW1[i][j] = 0.f;
  float dbias = 0.f;  // threads 0..63: db2[c]; threads 64..127: db1[c-64]

  const int n_tiles = (p.V + GT - 1) / GT;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int base = tile * GT;
    __syncthreads();
    // ---- stage g_o, y, r, a with cp.async (the whole 128 KB tile in flight at once), then g_y in place:
    //      g_y = rstd * (gamma*g_o - c1 - yhat*c2)
    cp_async_row_tile<GT, HID>(sm.gy, GLD, p.g_o, base, p.V);
    cp_async_row_tile<GT, HID>(sm.gu, GLD, p.y, base, p.V);
    cp_async_row_tile<GT, HID>(sm.r, GLD, p.r, base, p.V);
    cp_async_row_tile<GT, KIN>(sm.a, LDA, p.a, base, p.V);
    cp_async_commit();
    cp_async_wait_all();
    __syncthreads();
    {
      const int c = (threadIdx.x % (HID / 4)) * 4;
      const float4 mean = ldg4(p.bn + c), rstd = ldg4(p.bn + HID + c), gamma = ldg4(p.bn + 2 * HID + c);
      const float4 c1 = ldg4(p.cvec + c), c2 = ldg4(p.cvec + HID + c);
      for (int r = threadIdx.x / (HID / 4); r < GT; r += kThreads / (HID / 4)) {
        float4 gy = make4(0.f);
        if (base + r < p.V) {
          const float4 go = ld4(sm.gy + r * GLD + c);
          const float4 y = ld4(sm.gu + r * GLD + c);
          gy.x = rstd.x * (gamma.x * go.x - c1.x - (y.x - mean.x) * rstd.x * c2.x);
          gy.y = rstd.y * (gamma.y * go.y - c1.y - (y.y - mean.y) * rstd.y * c2.y);
          gy.z = rstd.z * (gamma.z * go.z - c1.z - (y.z - mean.z) * rstd.z * c2.z);
          gy.w = rstd.w * (gamma.w * go.w - c1.w - (y.w - mean.w) * rstd.w * c2.w);
        }
        st4(sm.gy + r * GLD + c, gy);
      }
    }
    __syncthreads();
    // ---- g_u = (g_y W2) * [r > 0]
    {
      float acc[M2::TM][4];
#pragma unroll
      for (int m = 0; m < M2::TM; ++m) acc[m][0] = acc[m][1] = acc[m][2] = acc[m][3] = 0.f;
      gemm_nn<GT, HID, HID>(sm.gy, GLD, sm.w2, HID, acc);
      const int c0 = M2::col0(), r0 = M2::row0();
#pragma unroll
      for (int m = 0; m < M2::TM; ++m) {
        const float4 rr = ld4(sm.r + (r0 + m) * GLD + c0);
        st4(sm.gu + (r0 + m) * GLD + c0,
            make_float4(rr.x > 0.f ? acc[m][0] : 0.f, rr.y > 0.f ? acc[m][1] : 0.f,
                        rr.z > 0.f ? acc[m][2] : 0.f, rr.w > 0.f ? acc[m][3] : 0.f));
      }
    }
    __syncthreads();
    // ---- g_a = g_u W1 -> global
    {
      float acc[M1::TM][4];
#pragma unroll
      for (int m = 0; m < M1::TM; ++m) acc[m][0] = acc[m][1] = acc[m][2] = acc[m][3] = 0.f;
      gemm_nn<GT, HID, KIN>(sm.gu, GLD, sm.w1, KIN, acc);
      const int c0 = M1::col0(), r0 = M1::row0();
#pragma unroll
      for (int m = 0; m < M1::TM; ++m) {
        const int v = base + r0 + m;
        if (v < p.V) st4(p.g_a + (size_t)v * KIN + c0, make_float4(acc[m][0], acc[m][1], acc[m][2], acc[m][3]));
      }
    }
    // ---- weight gradients (rows beyond V are zero in gy/gu)
    gemm_tn<HID, HID>(sm.gy, GLD, sm.r, GLD, GT, dW2);
    gemm_tn<HID, KIN>(sm.gu, GLD, sm.a, LDA, GT, dW1);
    if (threadIdx.x < 2 * HID) {
      const float* src = (threadIdx.x < HID) ? sm.gy : sm.gu;
      const int c = threadIdx.x & (HID - 1);
      float s = 0.f;
#pragma unroll 8
      for (int r = 0; r < GT; ++r) s += src[r * GLD + c];
      dbias += s;
    }
  }
  // ---- per-CTA partials (every CTA writes, also when it had no tile)
  float* part = p.part + (size_t)blockIdx.x * p.pstride;
#pragma unroll
  for (int i = 0; i < T2::TO; ++i)
#pragma unroll
    for (int j = 0; j < T2::TJ; ++j) part[p.off_W2 + (T2::o0() + i) * HID + T2::j0() + j] = dW2[i][j];
#pragma unroll
  for (int i = 0; i < T1::TO; ++i)
#pragma unroll
    for (int j = 0; j < T1::TJ; ++j) part[p.off_W1 + (T1::o0() + i) * KIN + T1::j0() + j] = dW1[i][j];
  if (threadIdx.x < HID) part[p.off_b2 + threadIdx.x] = dbias;
  else if (threadIdx.x < 2 * HID) part[p.off_b1 + threadIdx.x - HID] = dbias;
}

template <int KIN, int H, int GTB>
static void launch_gin_bwd_main_t(const GinBwdMainArgs& a, int grid, cudaStream_t s) {
  using S = GinBwdSmem<KIN, H, GTB>;
  static bool once = (cudaFuncSetAttribute(gin_bwd_main_kernel<KIN, H, GTB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(S)), true);
  (void)once;
  launch_k((gin_bwd_main_kernel<KIN, H, GTB>), dim3(grid), dim3(kThreads), sizeof(S), s, a);
}
void launch_gin_bwd_main(const GinBwdMainArgs& a, int kin, int hidden, int grid, cudaStream_t s) {
  if (hidden == 64) { if (kin == 32) launch_gin_bwd_main_t<32, 64, 128>(a, grid, s); else launch_gin_bwd_main_t<64, 64, 128>(a, grid, s); }
  else if (kin == 32) launch_gin_bwd_main_t<32, 128, 32>(a, grid, s);
  else if (kin == 64) launch_gin_bwd_main_t<64, 128, 32>(a, grid, s);     // layer 0 at d_transfer 64
  else launch_gin_bwd_main_t<128, 128, 32>(a, grid, s);
}

// ------------------------------------------------------------------------------------------------
// transfer_d backward: dWt[o][f] = sum_rows gt_row[o] * x_hat[map(row)][f] with gt_row = Ga0_row + sum_{u in N(row)} Ga0_u
// (layer-0 aggregation backward; Ga0 is [V][DT]).  The adjacency is symmetric, so the gather moves to the features:
//   dWt[o][f] = sum_u Ga0_u[o] * xagg_u[f],   xagg_u = x_hat[p(u)] + sum_{v in N(u)} x_hat[p(v)]
// xagg is a constant of the batch, produced by side CTAs of the forward's prologue launch (fwd_prep); this kernel only
// streams Ga0 and xagg (it was a latency-bound CSR gather of 128-byte rows before: 59 us at B = 4096).
// Two row sets (parent batch, ego batch) in one launch; last CTA finalises into grads.
// ------------------------------------------------------------------------------------------------
// padded feature width of a partial row: 32 up to F = 32, else F rounded up to the FC = 16 columns of a pass
__host__ __device__ __forceinline__ int ipb_fp(int F) { return F <= 32 ? 32 : (F + 15) / 16 * 16; }
constexpr int IPB_THREADS = 1024;   // 32 warps per CTA, one CTA per SM: 148 partials for the final (last-CTA) reduction

// lane = output channel og + o of transfer_d (og: 32-channel group, one pass over the rows each); every warp streams 32-row
// blocks straight from global memory (coalesced 128-byte Ga0 row segments, xagg rows one per lane and broadcast by shuffles)
// into acc[f] = sum_r Ga0_r[og + o] xagg_r[f]
template <int FC, bool WIDE, int DT>     // WIDE: F > 32; DT: d_transfer (a compile-time stride, so DT = 32 keeps its code)
__global__ void __launch_bounds__(IPB_THREADS, 1)
input_proj_bwd_kernel(InputProjBwdArgs p) {
  pdl_sync();
  __shared__ __align__(16) float s_red[32 * 32 * 4];     // [warp][o][4 features]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int V0 = p.V[0], Vt = p.V[0] + p.V[1], XS = p.xa_stride;
  const int nwarps = (int)gridDim.x * 32;
  const int gw = (int)blockIdx.x * 32 + warp;
  const int FP = WIDE ? ipb_fp(p.F) : 32;
  for (int og = 0; og < DT; og += 32)
  for (int fb = 0; fb < XS; fb += FC) {      // FC feature columns per pass over the rows (one pass for F <= 16)
  float acc[FC];
#pragma unroll
  for (int f = 0; f < FC; ++f) acc[f] = 0.f;
  // blocks of 32 rows: lane j holds xagg of row j (coalesced), broadcast by shuffles against the row's Ga0 line
  for (int rb = gw * 32; rb < Vt; rb += nwarps * 32) {
    float4 xm[FC / 4];
    {
      const int r = rb + lane;
      const int set = r < V0 ? 0 : 1, v = r < V0 ? r : r - V0;
      const float* xr = p.xagg[set] + (size_t)v * XS + fb;
#pragma unroll
      for (int q = 0; q < FC / 4; ++q) xm[q] = (r < Vt && fb + q * 4 < XS) ? ld4_cs(xr + q * 4) : make4(0.f);
    }
#pragma unroll
    for (int j0 = 0; j0 < 32; j0 += 8) {
      float g[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int r = rb + j0 + j;
        const int set = r < V0 ? 0 : 1, v = r < V0 ? r : r - V0;
        g[j] = r < Vt ? __ldcs(p.ga[set] + (size_t)v * DT + og + lane) : 0.f;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j)
#pragma unroll
        for (int q = 0; q < FC / 4; ++q) {
          acc[q * 4 + 0] = fmaf(g[j], __shfl_sync(0xffffffffu, xm[q].x, j0 + j), acc[q * 4 + 0]);
          acc[q * 4 + 1] = fmaf(g[j], __shfl_sync(0xffffffffu, xm[q].y, j0 + j), acc[q * 4 + 1]);
          acc[q * 4 + 2] = fmaf(g[j], __shfl_sync(0xffffffffu, xm[q].z, j0 + j), acc[q * 4 + 2]);
          acc[q * 4 + 3] = fmaf(g[j], __shfl_sync(0xffffffffu, xm[q].w, j0 + j), acc[q * 4 + 3]);
        }
    }
  }
  // CTA partial [o][f] (stride FP): the 32 warps are summed in a fixed order, four feature columns at a time
  float* part = p.part + ((size_t)blockIdx.x * DT + og) * FP;
#pragma unroll
  for (int q = 0; q < FC / 4; ++q) {
    __syncthreads();
    st4(s_red + (warp * 32 + lane) * 4, make_float4(acc[q * 4], acc[q * 4 + 1], acc[q * 4 + 2], acc[q * 4 + 3]));
    __syncthreads();
    if (threadIdx.x < 128) {
      const int o = threadIdx.x >> 2, k = threadIdx.x & 3;
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < 32; ++w) t += s_red[(w * 32 + o) * 4 + k];
      part[o * FP + fb + q * 4 + k] = t;
    }
  }
  }
  if (!last_cta_arrives(p.counter)) return;
  // only the F real feature columns; interleaved partial sums keep the loads of a thread independent; fixed order
  for (int o2 = threadIdx.x; o2 < DT * p.F; o2 += IPB_THREADS) {
    const int oo = o2 / p.F, f = o2 % p.F;
    const float* src = p.part + oo * FP + f;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    const int nb = (int)gridDim.x;
    int b = 0;
#pragma unroll 8
    for (; b + 3 < nb; b += 4) {
      s0 += (double)__ldcg(src + (size_t)b * DT * FP);
      s1 += (double)__ldcg(src + (size_t)(b + 1) * DT * FP);
      s2 += (double)__ldcg(src + (size_t)(b + 2) * DT * FP);
      s3 += (double)__ldcg(src + (size_t)(b + 3) * DT * FP);
    }
    for (; b < nb; ++b) s0 += (double)__ldcg(src + (size_t)b * DT * FP);
    p.d_Wt[oo * p.F + f] = (float)((s0 + s1) + (s2 + s3));
  }
}

int input_proj_bwd_grid(int V0, int V1) {
  (void)V0; (void)V1;
  return num_sms();
}
size_t input_proj_bwd_part_floats(int V0, int V1, int F, int DT) { return (size_t)input_proj_bwd_grid(V0, V1) * DT * ipb_fp(F); }
template <int FC, bool WIDE>
static void launch_ipb(const InputProjBwdArgs& a, int grid, cudaStream_t s) {
  if (a.DT == 32) launch_k((input_proj_bwd_kernel<FC, WIDE, 32>), dim3(grid), dim3(IPB_THREADS), 0, s, a);
  else if (a.DT == 64) launch_k((input_proj_bwd_kernel<FC, WIDE, 64>), dim3(grid), dim3(IPB_THREADS), 0, s, a);
  else launch_k((input_proj_bwd_kernel<FC, WIDE, 128>), dim3(grid), dim3(IPB_THREADS), 0, s, a);
}
void launch_input_proj_bwd(const InputProjBwdArgs& a, cudaStream_t s) {
  const int grid = input_proj_bwd_grid(a.V[0], a.V[1]);
  if (a.F <= 12) launch_ipb<12, false>(a, grid, s);
  else if (a.F <= 32) launch_ipb<16, false>(a, grid, s);
  else launch_ipb<16, true>(a, grid, s);
}

}  // namespace scgib
