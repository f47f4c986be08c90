// side_jobs.cuh - device bodies of the step's small serial jobs, shared by their stand-alone kernels (loss_kernels.cu,
// head_kernels.cu: op-level C ABI, FFMA / hidden-128 paths) and, for the forward jobs, by the tcgen05 contrastive forward
// launch, where they run as EXTRA CTAs on the SMs that launch leaves idle (ConFwdSides, kernels.cuh).
//
// Reference call sites replaced: loss_recon_adj (models.py:762-768, Gram identity), the compressor BatchNorm's B sequential
// running-statistics updates (models.py:642 per graph), KL + recon + contrastive (exp_pretraining.py:321).
#pragma once
#include "kernels.cuh"

namespace scgib {

// G[j] = sum over the recon_fwd partials (fp64, fixed order: 8 interleaved chains); output j = HID*HID is the edge-dot sum.
// CTA idx of n (blockDim = kThreads) takes outputs idx*kThreads + t, stride n*kThreads.
__device__ __forceinline__ void recon_reduce_body(const float* __restrict__ part, int grid, float* __restrict__ G,
                                                  float* __restrict__ edge_sum, int HID, int idx, int n) {
  const int total = HID * HID + 1;
  const size_t ST = (size_t)HID * HID + 4;
  for (int j = idx * kThreads + (int)threadIdx.x; j < total; j += n * kThreads) {
    double s[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) s[k] = 0.0;
    int c = 0;
#pragma unroll 2
    for (; c + 7 < grid; c += 8) {
#pragma unroll
      for (int k = 0; k < 8; ++k) s[k] += (double)__ldcg(part + (size_t)(c + k) * ST + j);
    }
    for (; c < grid; ++c) s[0] += (double)__ldcg(part + (size_t)c * ST + j);
    const double t = ((s[0] + s[1]) + (s[2] + s[3])) + ((s[4] + s[5]) + (s[6] + s[7]));
    if (j < HID * HID) G[j] = (float)t; else edge_sum[0] = (float)t;
  }
}

// running stats of the compressor BN after B sequential per-graph updates (closed form, fixed order)
// r_B = 0.9^B r_0 + sum_g 0.1 * 0.9^(B-1-g) stat_g ; graphs older than kEmaWindow contribute < 0.9^768 ~ 1e-35.
constexpr int kEmaWindow = 768;
template <int HID, int NT>       // one CTA of NT threads (a multiple of 2*HID)
__device__ __forceinline__ void compressor_ema_body(const float* __restrict__ cstat, int B, float* __restrict__ running) {
  constexpr int kSeg = NT / (2 * HID);
  static_assert(kSeg >= 1 && kSeg * 2 * HID == NT, "EMA CTA size");
  __shared__ double s_part[kSeg][2 * HID];
  const int j = threadIdx.x % (2 * HID);  // 0..H-1 mean, H..2H-1 var
  const int seg = threadIdx.x / (2 * HID);
  const int g0 = B > kEmaWindow ? B - kEmaWindow : 0;
  // newest graph first: weight 0.1 * 0.9^k for age k = B-1-g, advanced by a constant factor (two pow() per thread
  // instead of one per term: the fp64 pow dominated this kernel)
  double acc = 0.0;
  double w = 0.1 * pow(0.9, (double)seg);
  const double step = pow(0.9, (double)kSeg);
#pragma unroll 8
  for (int g = B - 1 - seg; g >= g0; g -= kSeg) {
    acc += w * (double)__ldcg(cstat + (size_t)g * 2 * HID + j);
    w *= step;
  }
  s_part[seg][j] = acc;
  __syncthreads();
  if (seg == 0) {
    double r = pow(0.9, (double)B) * (double)running[j];
#pragma unroll
    for (int k = 0; k < kSeg; ++k) r += s_part[k][j];
    running[j] = (float)r;
  }
}

// losses = {KL, contrastive, recon, total}; also the contrastive denominators D_i (saved for backward).  One CTA of NT threads.
template <int NT>
__device__ __forceinline__ void loss_finalize_body(const LossFinalizeArgs& p) {
  __shared__ double s_a[NT], s_b[NT];
  double con = 0.0, fro = 0.0;
  const bool act = threadIdx.x < NT;       // a CTA may have more threads than NT: the extra ones only join the barriers
  if (act) {
  // four rows per thread and pass: 4 x jsplit independent loads in flight (the serial chain of L2 round trips is the whole
  // cost of this one-CTA job); every row's partial sums are still added in column-split order
  for (int i0 = threadIdx.x; i0 < p.B; i0 += 4 * NT) {
    float d[4] = {0.f, 0.f, 0.f, 0.f}, dg[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) dg[u] = i0 + u * NT < p.B ? __ldcg(p.diag + i0 + u * NT) : 0.f;
    for (int js = 0; js < p.jsplit; ++js) {
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (i0 + u * NT < p.B) d[u] += __ldcg(p.rowsum + (size_t)js * p.B + i0 + u * NT);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (i0 + u * NT < p.B) {
        p.D[i0 + u * NT] = d[u];
        con += (double)(logf(d[u]) - dg[u]);      // -log(exp(s_b(i,i)) / D_i)
      }
  }
  if (!p.recon_override) {
#pragma unroll 8
    for (int j = threadIdx.x; j < p.hidden * p.hidden; j += NT) { const double g = (double)__ldcg(p.G + j); fro += g * g; }
  }
  s_a[threadIdx.x] = con; s_b[threadIdx.x] = fro;
  }
  __syncthreads();
  for (int o = NT / 2; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) { s_a[threadIdx.x] += s_a[threadIdx.x + o]; s_b[threadIdx.x] += s_b[threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const float kl = __ldcg(p.kl);
    const float c = (float)(s_a[0] / (double)p.B);
    const float r = p.recon_override ? __ldcg(p.recon_override)
                                     : (float)((s_b[0] - 2.0 * (double)__ldcg(p.edge_sum) + (double)p.E) / (double)p.N);
    p.losses[0] = kl; p.losses[1] = c; p.losses[2] = r; p.losses[3] = kl + r + c;
  }
}

// recon backward: gZ = scale * (4/N) * (Z G - A Z); CTA idx of n walks row tiles idx, idx + n, ...
constexpr int kReconTile = 128;
template <int HID> struct ReconBwdSmem { float z[kReconTile * (HID + 4)]; float g[HID * HID]; };

template <int HID>
__device__ __forceinline__ void recon_bwd_body(const ReconBwdArgs& p, unsigned char* smem_raw, int idx, int n) {
  constexpr int GT = kReconTile;
  ReconBwdSmem<HID>& sm = *reinterpret_cast<ReconBwdSmem<HID>*>(smem_raw);
  constexpr int GLD = HID + 4;
  using M = NNMap<GT, HID>;
  load_matrix<HID>(sm.g, HID, p.G, HID);
  const float k = p.scale * 4.f / (float)p.N;
  const int n_tiles = (p.N + GT - 1) / GT;
  float gm = 0.f;
  for (int tile = idx; tile < n_tiles; tile += n) {
    const int base = tile * GT;
    __syncthreads();
    load_row_tile<GT, HID>(sm.z, GLD, p.Z, base, p.N);
    __syncthreads();
    float acc[M::TM][4];
#pragma unroll
    for (int m = 0; m < M::TM; ++m) acc[m][0] = acc[m][1] = acc[m][2] = acc[m][3] = 0.f;
    const int c0 = M::col0(), r0 = M::row0();
    // the neighbour sums (A Z) of this thread's rows are issued before the tile GEMM: their L2 latency hides behind it
    // (hidden 64; at 128 the 16 extra float4 per thread would spill, so the sums follow the GEMM there)
    constexpr bool EARLY = HID == 64;
    float4 nb[EARLY ? M::TM : 1];
    auto neigh = [&](int v) {
      float4 t = make4(0.f);
      const int e0 = __ldg(p.indptr + v), e1 = __ldg(p.indptr + v + 1);
      for (int e = e0; e < e1; ++e) t = add4(t, ld4(p.Z + (size_t)__ldg(p.indices + e) * HID + c0));
      return t;
    };
    if (EARLY) {
#pragma unroll
      for (int m = 0; m < M::TM; ++m) {
        const int v = base + r0 + m;
        nb[EARLY ? m : 0] = v < p.N ? neigh(v) : make4(0.f);
      }
    }
    gemm_nn<GT, HID, HID>(sm.z, GLD, sm.g, HID, acc);
#pragma unroll
    for (int m = 0; m < M::TM; ++m) {
      const int v = base + r0 + m;
      if (v < p.N) {
        const float4 t = EARLY ? nb[EARLY ? m : 0] : neigh(v);
        const float4 o = make_float4(k * (acc[m][0] - t.x), k * (acc[m][1] - t.y), k * (acc[m][2] - t.z), k * (acc[m][3] - t.w));
        st4(p.gZ + (size_t)v * HID + c0, o);
        gm = fmaxf(fmaxf(gm, fmaxf(fabsf(o.x), fabsf(o.y))), fmaxf(fabsf(o.z), fabsf(o.w)));
      }
    }
  }
  if (p.gmax) {                  // max is order-independent: the atomic keeps the result deterministic
    gm = warp_max(gm);
    if ((threadIdx.x & 31) == 0 && gm > 0.f) atomicMax(p.gmax, __float_as_uint(gm));
  }
}

}  // namespace scgib
