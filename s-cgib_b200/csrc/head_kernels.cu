// head_kernels.cu - everything between the two GIN encoders and the losses:
//   ego sum-pooling + attention logit, compressor linear, the per-graph information-bottleneck gate with
//   the core/graph readouts, KL and the core-candidate softmax fused in one segment kernel, and the head MLP.
//
// Reference call sites replaced (paths relative to the reference tree):
//   dgl.sum_nodes                         models.py:716, 725, 733, 684
//   compress / compression (Python loop)  models.py:595-604, 631-660
//   attention (Python loop)               models.py:738-749
//   self.MLP(interaction_map)             models.py:569-572, 676
#include <stdlib.h>
#include "kernels.cuh"
#include "side_jobs.cuh"

namespace scgib {

constexpr int GT = 128;

// ------------------------------------------------------------------------------------------------
// segment sums (half-warp per segment, float4 lanes)
// ------------------------------------------------------------------------------------------------
template <int HID>
__global__ void __launch_bounds__(kThreads)
segment_sum_kernel(const float* __restrict__ in, const int32_t* __restrict__ seg_ptr, int S, const float* __restrict__ bn,
                   float* __restrict__ out) {
  pdl_sync();
  constexpr int LPR = HID / 4, SPC = kThreads / LPR;      // lanes per segment (4 channels each), segments per CTA pass
  const int l = threadIdx.x % LPR;
  Bn4 b;
  if (bn) b.load(bn, l * 4, HID);
  for (int s = blockIdx.x * SPC + (threadIdx.x / LPR); s < S; s += gridDim.x * SPC) {
    const int r0 = __ldg(seg_ptr + s), r1 = __ldg(seg_ptr + s + 1);
    float4 acc = make4(0.f);
    for (int r = r0; r < r1; ++r) {
      const float4 y = ld4(in + (size_t)r * HID + l * 4);
      acc = add4(acc, bn ? b.act(y) : y);
    }
    st4(out + (size_t)s * HID + l * 4, acc);
  }
}
void launch_segment_sum(const float* in, const int32_t* seg_ptr, int S, const float* bn, float* out, int hidden, cudaStream_t s) {
  const int spc = kThreads / (hidden / 4);
  const int grid = min((S + spc - 1) / spc, 16 * num_sms());
  if (hidden == 64) launch_k((segment_sum_kernel<64>), dim3(grid), dim3(kThreads), 0, s, in, seg_ptr, S, bn, out);
  else launch_k((segment_sum_kernel<128>), dim3(grid), dim3(kThreads), 0, s, in, seg_ptr, S, bn, out);
}

// C_v = sum over the ego-net of v of relu(BN(y)) ; logit_v = w_cand . C_v
// TWO consecutive seeds per lane group: their rows are contiguous, so one unrolled pass over [r0, r2) keeps up to 8
// independent row loads in flight per lane (one seed's ~3 rows leave the memory pipeline idle behind the ego_ptr -> row chain)
template <bool BF, int HID>
__global__ void __launch_bounds__(kThreads)
ego_pool_fwd_kernel(EgoPoolFwdArgs p) {
  pdl_sync();
  constexpr int LPR = HID / 4, SPC = kThreads / LPR;
  const int l = threadIdx.x % LPR;
  Bn4 b;
  b.load(p.bn, l * 4, HID);
  const float4 w = ldg4(p.w_cand + l * 4);
  const unsigned hmask = LPR == 32 ? 0xffffffffu : ((threadIdx.x & 16) ? 0xffff0000u : 0x0000ffffu);   // half-warps may diverge at the tail
  // the segment offsets of the NEXT pair are requested before this pair's rows are consumed (persistent grid: the
  // ego_ptr -> rows dependency of one iteration overlaps the row loads of the previous one)
  const int stride = 2 * gridDim.x * SPC;
  int v = 2 * (blockIdx.x * SPC + (threadIdx.x / LPR));
  int n0 = 0, n1 = 0, n2 = 0;
  if (v < p.N) { n0 = __ldg(p.ego_ptr + v); n1 = __ldg(p.ego_ptr + v + 1); n2 = v + 1 < p.N ? __ldg(p.ego_ptr + v + 2) : n1; }
  for (; v < p.N; v += stride) {
    const bool two = v + 1 < p.N;
    const int r0 = n0, r1 = n1, r2 = n2;
    const int vn = v + stride;
    if (vn < p.N) { n0 = __ldg(p.ego_ptr + vn); n1 = __ldg(p.ego_ptr + vn + 1); n2 = vn + 1 < p.N ? __ldg(p.ego_ptr + vn + 2) : n1; }
    float4 accA = make4(0.f), accB = make4(0.f);
    for (int rb = r0; rb < r2; rb += 8) {
      float4 x[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i] = rb + i < r2 ? ld4a<BF>(p.y, (size_t)(rb + i) * HID + l * 4) : make4(0.f);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (rb + i >= r2) break;
        const float4 a = b.act(x[i]);
        if (rb + i < r1) accA = add4(accA, a); else accB = add4(accB, a);
      }
    }
    st4(p.C + (size_t)v * HID + l * 4, accA);
    if (two) st4(p.C + (size_t)(v + 1) * HID + l * 4, accB);
    float dA = accA.x * w.x + accA.y * w.y + accA.z * w.z + accA.w * w.w;
    float dB = accB.x * w.x + accB.y * w.y + accB.z * w.z + accB.w * w.w;
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) { dA += __shfl_xor_sync(hmask, dA, o); dB += __shfl_xor_sync(hmask, dB, o); }
    if (l == 0) { p.logit[v] = dA; if (two) p.logit[v + 1] = dB; }
  }
}

void launch_ego_pool_fwd(const EgoPoolFwdArgs& a, int hidden, cudaStream_t s) {
  const int spc = 2 * (kThreads / (hidden / 4));                 // seeds per CTA pass
  const int grid = min((a.N + spc - 1) / spc, 3 * num_sms());    // persistent: 3 CTAs per SM
  if (hidden == 64) {
    if (a.y_bf16) launch_k((ego_pool_fwd_kernel<true, 64>), dim3(grid), dim3(kThreads), 0, s, a);
    else launch_k((ego_pool_fwd_kernel<false, 64>), dim3(grid), dim3(kThreads), 0, s, a);
  } else {
    if (a.y_bf16) launch_k((ego_pool_fwd_kernel<true, 128>), dim3(grid), dim3(kThreads), 0, s, a);
    else launch_k((ego_pool_fwd_kernel<false, 128>), dim3(grid), dim3(kThreads), 0, s, a);
  }
}

// ------------------------------------------------------------------------------------------------
// H = relu(BN(y_last)) ; q = H Wc1^T + bc1
// ------------------------------------------------------------------------------------------------
template <int HID> struct GateLinFwdSmem { float tile[GT * (HID + 4)]; float w[HID * HID]; };

template <bool BF, int HID>
__global__ void __launch_bounds__(kThreads, HID == 64 ? 2 : 1)
gate_lin_fwd_kernel(GateLinFwdArgs p) {
  pdl_sync();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  GateLinFwdSmem<HID>& sm = *reinterpret_cast<GateLinFwdSmem<HID>*>(smem_raw);
  constexpr int GLD = HID + 4;
  using M = NNMap<GT, HID>;
  load_matrix<HID>(sm.w, HID, p.Wc1t, HID);
  const int n_tiles = (p.N + GT - 1) / GT;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int base = tile * GT;
    __syncthreads();
    for (int i = threadIdx.x; i < GT * (HID / 4); i += kThreads) {
      const int r = i / (HID / 4), c = (i % (HID / 4)) * 4;
      const int v = base + r;
      float4 h = make4(0.f);
      if (v < p.N) {
        Bn4 b;
        b.load(p.bn, c, HID);
        h = b.act(ld4a<BF>(p.y, (size_t)v * HID + c));
        st4(p.H + (size_t)v * HID + c, h);
      }
      st4(sm.tile + r * GLD + c, h);
    }
    __syncthreads();
    float acc[M::TM][4];
    const int c0 = M::col0(), r0 = M::row0();
    const float4 bias = ldg4(p.bc1 + c0);
#pragma unroll
    for (int m = 0; m < M::TM; ++m) { acc[m][0] = bias.x; acc[m][1] = bias.y; acc[m][2] = bias.z; acc[m][3] = bias.w; }
    gemm_nn<GT, HID, HID>(sm.tile, GLD, sm.w, HID, acc);
#pragma unroll
    for (int m = 0; m < M::TM; ++m) {
      const int v = base + r0 + m;
      if (v < p.N) st4(p.q + (size_t)v * HID + c0, make_float4(acc[m][0], acc[m][1], acc[m][2], acc[m][3]));
    }
  }
}
template <bool BF, int H>
static void launch_gate_lin_fwd_t(const GateLinFwdArgs& a, cudaStream_t s) {
  static bool once = (cudaFuncSetAttribute(gate_lin_fwd_kernel<BF, H>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(GateLinFwdSmem<H>)), true);
  (void)once;
  const int grid = min((a.N + GT - 1) / GT, (H == 64 ? 2 : 1) * num_sms());
  launch_k((gate_lin_fwd_kernel<BF, H>), dim3(grid), dim3(kThreads), sizeof(GateLinFwdSmem<H>), s, a);
}
void launch_gate_lin_fwd(const GateLinFwdArgs& a, int hidden, cudaStream_t s) {
  static int gate_ffma = -1;                 // SCGIB_HEAD_FFMA=1: FFMA tiles also at hidden 64 (cross-check)
  if (gate_ffma < 0) { const char* e = getenv("SCGIB_HEAD_FFMA"); gate_ffma = (e && e[0] == '1') ? 1 : 0; }
  if (hidden == 64 && a.Wc1n && tensor_core_mode() != 0 && !gate_ffma &&
      ((((uintptr_t)a.y | (uintptr_t)a.H | (uintptr_t)a.q) & 31u) == 0)) {
    launch_gate_lin_fwd_tc(a, a.Wc1n, s);
    return;
  }
  if (hidden == 64) { if (a.y_bf16) launch_gate_lin_fwd_t<true, 64>(a, s); else launch_gate_lin_fwd_t<false, 64>(a, s); }
  else { if (a.y_bf16) launch_gate_lin_fwd_t<true, 128>(a, s); else launch_gate_lin_fwd_t<false, 128>(a, s); }
}

// gH += g_q Wc1 ; dWc1 += g_q^T H ; dbc1 += sum g_q
template <int HID, int GT> struct GateLinBwdSmem { float gq[2][GT * (HID + 4)]; float h[2][GT * (HID + 4)]; float w[HID * HID]; };   // two tile buffers: cp.async prefetch

template <int HID, int GT>       // GT rows per tile: 128 at HID = 64, 32 at HID = 128 (four tiles + the weights in 227 KB)
__global__ void __launch_bounds__(kThreads, 1)
gate_lin_bwd_kernel(GateLinBwdArgs p) {
  pdl_sync();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  GateLinBwdSmem<HID, GT>& sm = *reinterpret_cast<GateLinBwdSmem<HID, GT>*>(smem_raw);
  constexpr int GLD = HID + 4;
  using M = NNMap<GT, HID>;
  using T = TNMap<HID, HID>;
  load_matrix<HID>(sm.w, HID, p.Wc1, HID);
  float dW[T::TO][T::TJ];
#pragma unroll
  for (int i = 0; i < T::TO; ++i)
#pragma unroll
    for (int j = 0; j < T::TJ; ++j) dW[i][j] = 0.f;
  float dbias = 0.f;
  const int n_tiles = (p.N + GT - 1) / GT;
  // the next tile's g_q / H rows are copied (cp.async, no register staging) while this tile's GEMMs run
  if ((int)blockIdx.x < n_tiles) {
    cp_async_row_tile<GT, HID>(sm.gq[0], GLD, p.g_q, blockIdx.x * GT, p.N);
    cp_async_row_tile<GT, HID>(sm.h[0], GLD, p.H, blockIdx.x * GT, p.N);
  }
  cp_async_commit();
  int it = 0;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
    const int base = tile * GT;
    const float* gq = sm.gq[it & 1];
    const float* hh = sm.h[it & 1];
    cp_async_wait_all();
    __syncthreads();                      // tile `it` has landed; every thread is done with the other buffer (tile it-1)
    if (tile + (int)gridDim.x < n_tiles) {
      cp_async_row_tile<GT, HID>(sm.gq[(it + 1) & 1], GLD, p.g_q, (tile + gridDim.x) * GT, p.N);
      cp_async_row_tile<GT, HID>(sm.h[(it + 1) & 1], GLD, p.H, (tile + gridDim.x) * GT, p.N);
    }
    cp_async_commit();
    float acc[M::TM][4];
#pragma unroll
    for (int m = 0; m < M::TM; ++m) acc[m][0] = acc[m][1] = acc[m][2] = acc[m][3] = 0.f;
    gemm_nn<GT, HID, HID>(gq, GLD, sm.w, HID, acc);
    const int c0 = M::col0(), r0 = M::row0();
#pragma unroll
    for (int m = 0; m < M::TM; ++m) {
      const int v = base + r0 + m;
      if (v < p.N) {
        float* dst = p.gH + (size_t)v * HID + c0;
        const float4 old = ld4(dst);
        st4(dst, make_float4(old.x + acc[m][0], old.y + acc[m][1], old.z + acc[m][2], old.w + acc[m][3]));
      }
    }
    gemm_tn<HID, HID>(gq, GLD, hh, GLD, GT, dW);
    if (threadIdx.x < HID) {
      float s = 0.f;
#pragma unroll 8
      for (int r = 0; r < GT; ++r) s += gq[r * GLD + threadIdx.x];
      dbias += s;
    }
  }
  cp_async_wait_all();
  float* part = p.part + (size_t)blockIdx.x * p.pstride;
#pragma unroll
  for (int i = 0; i < T::TO; ++i)
#pragma unroll
    for (int j = 0; j < T::TJ; ++j) part[p.off_W + (T::o0() + i) * HID + T::j0() + j] = dW[i][j];
  if (threadIdx.x < HID) part[p.off_b + threadIdx.x] = dbias;
}
template <int H, int GTB>
static void launch_gate_lin_bwd_t(const GateLinBwdArgs& a, int grid, cudaStream_t s) {
  using S = GateLinBwdSmem<H, GTB>;
  static bool once = (cudaFuncSetAttribute(gate_lin_bwd_kernel<H, GTB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(S)), true);
  (void)once;
  launch_k((gate_lin_bwd_kernel<H, GTB>), dim3(grid), dim3(kThreads), sizeof(S), s, a);
}
void launch_gate_lin_bwd(const GateLinBwdArgs& a, int hidden, int grid, cudaStream_t s) {
  if (hidden == 64) launch_gate_lin_bwd_t<64, 128>(a, grid, s); else launch_gate_lin_bwd_t<128, 32>(a, grid, s);
}

// ------------------------------------------------------------------------------------------------
// per-graph gate (warp per graph, lane owns channels 2l, 2l+1)
// ------------------------------------------------------------------------------------------------
// A lane owns CPL = HID / 32 consecutive channels (2 at HID = 64, 4 at HID = 128): vector loads / stores of CPL floats
template <int CPL> struct LaneVec { float v[CPL]; };
template <int CPL>
__device__ __forceinline__ LaneVec<CPL> ldv(const float* p) {
  LaneVec<CPL> r;
  if (CPL == 2) { const float2 t = *reinterpret_cast<const float2*>(p); r.v[0] = t.x; r.v[1] = t.y; }
  else { const float4 t = *reinterpret_cast<const float4*>(p); r.v[0] = t.x; r.v[1] = t.y; r.v[CPL - 2] = t.z; r.v[CPL - 1] = t.w; }
  return r;
}
template <int CPL>
__device__ __forceinline__ void stv(float* p, const LaneVec<CPL>& a) {
  if (CPL == 2) *reinterpret_cast<float2*>(p) = make_float2(a.v[0], a.v[1]);
  else *reinterpret_cast<float4*>(p) = make_float4(a.v[0], a.v[1], a.v[CPL - 2], a.v[CPL - 1]);
}
template <int CPL>
__device__ __forceinline__ void stv_bf16(bf16_t* p, const LaneVec<CPL>& a) {      // round-to-nearest-even bf16 copy
  uint32_t w0, w1;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(w0) : "f"(a.v[1]), "f"(a.v[0]));
  if (CPL == 2) { *reinterpret_cast<uint32_t*>(p) = w0; return; }
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(w1) : "f"(a.v[CPL - 1]), "f"(a.v[CPL - 2]));
  *reinterpret_cast<uint2*>(p) = make_uint2(w0, w1);
}
template <int CPL>
__device__ __forceinline__ LaneVec<CPL> zerov() {
  LaneVec<CPL> r;
#pragma unroll
  for (int k = 0; k < CPL; ++k) r.v[k] = 0.f;
  return r;
}

constexpr float kKlEps = 0.0000001f;   // models.py:632
__device__ __forceinline__ float tf32_rna_f(float v) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return __uint_as_float(r);
}

// Measured and NOT kept: graphs of <= 24 nodes with their H / q rows cached in registers (one round of loads instead of three
// passes of 4-row batches): 170 registers -> one resident CTA per SM, 62 instead of 43 us - the warps-per-SM count, not the
// per-graph chain, sets this kernel's time.
template <int HID, int RB>      // RB rows in flight per warp in the gate pass (4 for molecule-sized graphs, 8 for ~150-node graphs)
__global__ void __launch_bounds__(kThreads)
graph_gate_fwd_kernel(GraphGateFwdArgs p) {
  pdl_sync();
  constexpr int CPL = HID / 32;
  using V = LaneVec<CPL>;
  const int lane = threadIdx.x & 31;
  const int c = CPL * lane;
  const V gam = ldv<CPL>(p.gamma_c + c), bet = ldv<CPL>(p.beta_c + c), w2 = ldv<CPL>(p.wc2 + c);
  const float bc2 = __ldg(p.bc2);
  const int warps = gridDim.x * (kThreads / 32);
  for (int g = blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); g < p.B; g += warps) {
    const int v0 = __ldg(p.graph_ptr + g), v1 = __ldg(p.graph_ptr + g + 1);
    const float n = (float)(v1 - v0);
    // pass 1: means
    V sH = zerov<CPL>(), sQ = zerov<CPL>();
#pragma unroll 4
    for (int v = v0; v < v1; ++v) {
      const V h = ldv<CPL>(p.H + (size_t)v * HID + c), q = ldv<CPL>(p.q + (size_t)v * HID + c);
#pragma unroll
      for (int k = 0; k < CPL; ++k) { sH.v[k] += h.v[k]; sQ.v[k] += q.v[k]; }
    }
    V muH, muQ;
#pragma unroll
    for (int k = 0; k < CPL; ++k) { muH.v[k] = sH.v[k] / n; muQ.v[k] = sQ.v[k] / n; }
    // pass 2: centred second moments
    V vH = zerov<CPL>(), vQ = zerov<CPL>();
#pragma unroll 4
    for (int v = v0; v < v1; ++v) {
      const V h = ldv<CPL>(p.H + (size_t)v * HID + c), q = ldv<CPL>(p.q + (size_t)v * HID + c);
#pragma unroll
      for (int k = 0; k < CPL; ++k) {
        float d = h.v[k] - muH.v[k]; vH.v[k] = fmaf(d, d, vH.v[k]);
        d = q.v[k] - muQ.v[k]; vQ.v[k] = fmaf(d, d, vQ.v[k]);
      }
    }
    V sd, rstd, muQe = muQ, uvar;
#pragma unroll
    for (int k = 0; k < CPL; ++k) {
      sd.v[k] = sqrtf(vH.v[k] / (n - 1.f));                       // torch.std_mean: unbiased
      rstd.v[k] = 1.f / sqrtf(vQ.v[k] / n + kBnEps);              // BN: biased
      uvar.v[k] = vQ.v[k] / (n - 1.f);
    }
    if (p.eval_running) {       // model.eval(): nn.BatchNorm1d normalises with its running statistics
      const V rm = ldv<CPL>(p.eval_running + c), rv = ldv<CPL>(p.eval_running + HID + c);
      muQe = rm;
#pragma unroll
      for (int k = 0; k < CPL; ++k) rstd.v[k] = 1.f / sqrtf(rv.v[k] + kBnEps);
    }
    stv<CPL>(p.readout + (size_t)g * HID + c, sH);
    float* gs = p.gstat + (size_t)g * 4 * HID;
    stv<CPL>(gs + c, muH); stv<CPL>(gs + HID + c, sd); stv<CPL>(gs + 2 * HID + c, muQe); stv<CPL>(gs + 3 * HID + c, rstd);
    if (p.cstat) {
      stv<CPL>(p.cstat + (size_t)g * 2 * HID + c, muQ);
      stv<CPL>(p.cstat + (size_t)g * 2 * HID + HID + c, uvar);
    }
    // pass 3: gate, noisy features, core readout, KL of the last graph
    const bool last = (g == p.B - 1);
    V core = zerov<CPL>(), kl1 = zerov<CPL>(), kl2 = zerov<CPL>(), isd;
#pragma unroll
    for (int k = 0; k < CPL; ++k) isd.v[k] = 1.f / (sd.v[k] + kKlEps);
    // latency-bound loop: the loads and shuffle chains of RB rows overlap
    for (int vb = v0; vb < v1; vb += RB) {
      V h[RB], q[RB], fu[RB];
      float u[RB], pv[RB];
#pragma unroll
      for (int i = 0; i < RB; ++i) {
        const int v = min(vb + i, v1 - 1);
        h[i] = ldv<CPL>(p.H + (size_t)v * HID + c); q[i] = ldv<CPL>(p.q + (size_t)v * HID + c);
        fu[i] = ldv<CPL>(p.feat_u + (size_t)v * HID + c); u[i] = __ldg(p.gate_u + v);
      }
#pragma unroll
      for (int i = 0; i < RB; ++i) {
        float acc = 0.f;
#pragma unroll
        for (int k = 0; k < CPL; ++k) {
          const float o = fmaf((q[i].v[k] - muQe.v[k]) * rstd.v[k], gam.v[k], bet.v[k]);
          acc = k == 0 ? fmaxf(o, 0.f) * w2.v[k] : acc + fmaxf(o, 0.f) * w2.v[k];
        }
        pv[i] = acc;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int i = 0; i < RB; ++i) pv[i] += __shfl_xor_sync(0xffffffffu, pv[i], o);
      }
#pragma unroll
      for (int i = 0; i < RB; ++i) {
        const int v = vb + i;
        if (v >= v1) break;
        const float eps = __fadd_rn(__fmul_rn(-0.9998f, u[i]), 0.9999f);       // (bias-(1-bias))*u + (1-bias), bias=1e-4
        const float gi = logf(eps) - logf(1.f - eps);
        const float lam = 1.f / (1.f + expf(-(gi + (pv[i] + bc2))));
        const float ln = 1.f - lam;
        V z;
#pragma unroll
        for (int k = 0; k < CPL; ++k) {
          const float m = lam * h[i].v[k] + ln * muH.v[k];
          const float sg = ln * sd.v[k];
          z.v[k] = m + fu[i].v[k] * sg;
          core.v[k] += z.v[k];
          if (last) {
            float t = sg * isd.v[k]; kl1.v[k] = fmaf(0.5f * t, t, kl1.v[k]);
            t = (m - muH.v[k]) * isd.v[k]; kl2.v[k] = fmaf(t, t, kl2.v[k]);
          }
        }
        stv<CPL>(p.noisy + (size_t)v * HID + c, z);
        if (p.noisy_bf) stv_bf16<CPL>(p.noisy_bf + (size_t)v * HID + c, z);
        if (lane == 0) p.lam[v] = lam;
      }
    }
    stv<CPL>(p.core + (size_t)g * HID + c, core);
    if (p.z1) {
      // the contrastive loss' row normalisation (models.py:606-610, F.normalize) of this graph's two readouts, fused here:
      // z1 = core / max(||core||, 1e-12), z2 = readout / max(||readout||, 1e-12), diag = z1 . z2, tf32 hi / lo copies
      float qa = 0.f, qb = 0.f;
#pragma unroll
      for (int k = 0; k < CPL; ++k) { qa = fmaf(core.v[k], core.v[k], qa); qb = fmaf(sH.v[k], sH.v[k], qb); }
      const float na = fmaxf(sqrtf(warp_sum(qa)), 1e-12f), nb = fmaxf(sqrtf(warp_sum(qb)), 1e-12f);
      V za, zb;
      float dd = 0.f;
#pragma unroll
      for (int k = 0; k < CPL; ++k) { za.v[k] = core.v[k] / na; zb.v[k] = sH.v[k] / nb; dd = fmaf(za.v[k], zb.v[k], dd); }
      const size_t o = (size_t)g * HID + c;
      stv<CPL>(p.z1 + o, za); stv<CPL>(p.z2 + o, zb);
      if (p.zsplit) {      // fp16 hi / lo parts [4][B][HID] halves (z1 hi, z1 lo, z2 hi, z2 lo) for the tensor-core kernels (hidden 64)
        uint32_t* zs = reinterpret_cast<uint32_t*>(p.zsplit);
        const size_t nn = (size_t)p.B * HID / 2, o2 = o / 2;
        uint32_t ah, al, bh, bl;
        split_f16x2_plain(za.v[0], za.v[1], ah, al);
        split_f16x2_plain(zb.v[0], zb.v[1], bh, bl);
        if (CPL == 2) { zs[o2] = ah; zs[nn + o2] = al; zs[2 * nn + o2] = bh; zs[3 * nn + o2] = bl; }
      }
      dd = warp_sum(dd);
      if (lane == 0) { p.n1[g] = na; p.n2[g] = nb; p.diag[g] = dd; }
    }
    if (last) {
      float a1 = 0.f, a2 = 0.f;
#pragma unroll
      for (int k = 0; k < CPL; ++k) { a1 = k == 0 ? kl1.v[k] : a1 + kl1.v[k]; a2 = k == 0 ? kl2.v[k] : a2 + kl2.v[k]; }
      const float tot = warp_sum(a1 + n * a2);
      if (lane == 0) p.kl[0] = tot / ((float)HID * n);
    }
    // attention softmax over the graph's nodes (core half and bias cancel: SURVEY F14)
    float mx = -INFINITY;
    for (int v = v0 + lane; v < v1; v += 32) mx = fmaxf(mx, __ldg(p.logit + v));
    mx = warp_max(mx);
    float se = 0.f;
    for (int v = v0 + lane; v < v1; v += 32) se += expf(__ldg(p.logit + v) - mx);
    se = warp_sum(se);
    for (int v = v0 + lane; v < v1; v += 32) p.alpha[v] = expf(__ldg(p.logit + v) - mx) / se;
  }
}
void launch_graph_gate_fwd(const GraphGateFwdArgs& a, int hidden, cudaStream_t s) {
  const int grid = min((a.B + 7) / 8, 8 * num_sms());
  const bool big = a.N / max(a.B, 1) >= 48;
  if (hidden == 64) {
    if (big) launch_k((graph_gate_fwd_kernel<64, 8>), dim3(grid), dim3(kThreads), 0, s, a);
    else launch_k((graph_gate_fwd_kernel<64, 4>), dim3(grid), dim3(kThreads), 0, s, a);
  } else {
    if (big) launch_k((graph_gate_fwd_kernel<128, 8>), dim3(grid), dim3(kThreads), 0, s, a);
    else launch_k((graph_gate_fwd_kernel<128, 4>), dim3(grid), dim3(kThreads), 0, s, a);
  }
}

// running stats of the compressor BN after B sequential per-graph updates: compressor_ema_body (side_jobs.cuh)
template <int HID>
__global__ void __launch_bounds__(1024)
compressor_ema_kernel(const float* __restrict__ cstat, int B, float* __restrict__ running) {
  pdl_sync();
  compressor_ema_body<HID, 1024>(cstat, B, running);
}
void launch_compressor_ema(const float* cstat, int B, float* running, int hidden, cudaStream_t s) {
  if (hidden == 64) launch_k((compressor_ema_kernel<64>), dim3(1), dim3(1024), 0, s, cstat, B, running);
  else launch_k((compressor_ema_kernel<128>), dim3(1), dim3(1024), 0, s, cstat, B, running);
}

// NT threads per CTA (measured at B = 4096, hidden 64: 256 threads / 512 CTAs and 512 threads / 256 CTAs - at 128 registers or
// capped to 64 with spills for two resident CTAs per SM - all take 88 us: the kernel is bound by the per-graph dependent chains)
template <int HID, int NT>
__global__ void __launch_bounds__(NT)
graph_gate_bwd_kernel(GraphGateBwdArgs p) {
  pdl_sync();
  constexpr int CPL = HID / 32;
  using V = LaneVec<CPL>;
  __shared__ __align__(16) float s_red[(NT / 32) * 5 * HID];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = CPL * lane;
  const V gam = ldv<CPL>(p.gamma_c + c), bet = ldv<CPL>(p.beta_c + c), w2 = ldv<CPL>(p.wc2 + c), wc = ldv<CPL>(p.w_cand + c);
  V a_dg = zerov<CPL>(), a_db = zerov<CPL>(), a_dw2 = zerov<CPL>(), a_dwc = zerov<CPL>();
  float a_dbc2 = 0.f, gqmax = 0.f;
  const int warps = gridDim.x * (NT / 32);
  auto dot = [](const V& a, const V& b) {
    float r = a.v[0] * b.v[0];
#pragma unroll
    for (int k = 1; k < CPL; ++k) r += a.v[k] * b.v[k];
    return r;
  };
  for (int g = blockIdx.x * (NT / 32) + warp; g < p.B; g += warps) {
    const int v0 = __ldg(p.graph_ptr + g), v1 = __ldg(p.graph_ptr + g + 1);
    const float n = (float)(v1 - v0);
    const float* gs = p.gstat + (size_t)g * 4 * HID;
    const V muH = ldv<CPL>(gs + c), sd = ldv<CPL>(gs + HID + c), muQ = ldv<CPL>(gs + 2 * HID + c), rstd = ldv<CPL>(gs + 3 * HID + c);
    V gcore, gread;
    if (p.con_g1p) {
      // (g - z_hat (z_hat . g)) / max(||z||, 1e-12) with g = scale / B * (sum of the column-split partials - the other view's z_hat)
      const size_t o = (size_t)g * HID + c;
      V g1 = zerov<CPL>(), g2 = zerov<CPL>();
      for (int js = 0; js < p.con_jsplit; ++js) {
        const V a = ldv<CPL>(p.con_g1p + (size_t)js * p.B * HID + o), bb = ldv<CPL>(p.con_g2p + (size_t)js * p.B * HID + o);
#pragma unroll
        for (int k = 0; k < CPL; ++k) { g1.v[k] += a.v[k]; g2.v[k] += bb.v[k]; }
      }
      const V z1 = ldv<CPL>(p.con_z1 + o), z2 = ldv<CPL>(p.con_z2 + o);
      const float kk = p.con_scale / (float)p.B;
      float t1 = 0.f, t2 = 0.f;
#pragma unroll
      for (int k = 0; k < CPL; ++k) {
        g1.v[k] = kk * (g1.v[k] - z2.v[k]); g2.v[k] = kk * (g2.v[k] - z1.v[k]);
        t1 = fmaf(z1.v[k], g1.v[k], t1); t2 = fmaf(z2.v[k], g2.v[k], t2);
      }
      const float d1 = warp_sum(t1), d2 = warp_sum(t2);
      const float n1 = __ldg(p.con_n1 + g), n2 = __ldg(p.con_n2 + g);
#pragma unroll
      for (int k = 0; k < CPL; ++k) { gcore.v[k] = (g1.v[k] - z1.v[k] * d1) / n1; gread.v[k] = (g2.v[k] - z2.v[k] * d2) / n2; }
    } else {
      gcore = ldv<CPL>(p.g_core + (size_t)g * HID + c); gread = ldv<CPL>(p.g_readout + (size_t)g * HID + c);
    }
    const bool last = (g == p.B - 1) && (p.kl_scale != 0.f);
    V isd;
#pragma unroll
    for (int k = 0; k < CPL; ++k) isd.v[k] = 1.f / (sd.v[k] + kKlEps);
    // ---- attention pass A: S = sum_v alpha_v (gT_v . C_v)
    float S = 0.f;
#pragma unroll 8
    for (int v = v0; v < v1; ++v) {
      const V gT = ldv<CPL>(p.gI2 + (size_t)v * p.gI_stride + c), C = ldv<CPL>(p.C + (size_t)v * HID + c);
      S += __ldg(p.alpha + v) * warp_sum(dot(gT, C));
    }
    // ---- pass B: attention backward, gate backward (scalar part), per-graph BN sums.  The loop is latency-bound (one
    //      warp per graph, two dependent shuffle reductions per row): the loads of RB rows are issued together and the
    //      rows' shuffle chains interleave; sums are still accumulated in row order.
    V m1 = zerov<CPL>(), m2 = zerov<CPL>();
    constexpr int RB = 4;
    for (int vb = v0; vb < v1; vb += RB) {
      V gT[RB], C[RB], gz0[RB], h[RB], fu[RB], q[RB];
      float al[RB], lam[RB];
#pragma unroll
      for (int i = 0; i < RB; ++i) {
        const int v = min(vb + i, v1 - 1);
        gT[i] = ldv<CPL>(p.gI2 + (size_t)v * p.gI_stride + c); C[i] = ldv<CPL>(p.C + (size_t)v * HID + c);
        gz0[i] = ldv<CPL>(p.gI + (size_t)v * p.gI_stride + c); h[i] = ldv<CPL>(p.H + (size_t)v * HID + c);
        fu[i] = ldv<CPL>(p.feat_u + (size_t)v * HID + c); q[i] = ldv<CPL>(p.q + (size_t)v * HID + c);
        al[i] = __ldg(p.alpha + v); lam[i] = __ldg(p.lam + v);
      }
      float dt[RB], part[RB];
      V gh[RB];
#pragma unroll
      for (int i = 0; i < RB; ++i) {
        dt[i] = dot(gT[i], C[i]);
        float pa = 0.f, kr1 = 0.f, kr2 = 0.f;
#pragma unroll
        for (int k = 0; k < CPL; ++k) {
          const float gz = gz0[i].v[k] + gcore.v[k];
          const float t = gz * (h[i].v[k] - muH.v[k] - fu[i].v[k] * sd.v[k]);
          pa = k == 0 ? t : pa + t;
          gh[i].v[k] = fmaf(lam[i], gz, gread.v[k]);
          if (last) {
            const float r1 = sd.v[k] * isd.v[k];                              // sigma/(sigma+e)
            const float r2 = (h[i].v[k] - muH.v[k]) * isd.v[k];               // (H-mu)/(sigma+e)
            kr1 = k == 0 ? r1 * r1 : kr1 + r1 * r1;
            kr2 = k == 0 ? r2 * r2 : kr2 + r2 * r2;
            gh[i].v[k] += (p.kl_scale / ((float)HID * n)) * 2.f * n * lam[i] * lam[i] * r2 * isd.v[k];
          }
        }
        if (last) pa += (p.kl_scale / ((float)HID * n)) * (-(1.f - lam[i]) * kr1 + 2.f * n * lam[i] * kr2);
        part[i] = pa;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int i = 0; i < RB; ++i) {
          dt[i] += __shfl_xor_sync(0xffffffffu, dt[i], o);
          part[i] += __shfl_xor_sync(0xffffffffu, part[i], o);
        }
      }
#pragma unroll
      for (int i = 0; i < RB; ++i) {
        const int v = vb + i;
        if (v >= v1) break;
        const float dl = al[i] * (dt[i] - S);
        const float gpv = part[i] * lam[i] * (1.f - lam[i]);
        V gc;
#pragma unroll
        for (int k = 0; k < CPL; ++k) {
          gc.v[k] = fmaf(dl, wc.v[k], al[i] * gT[i].v[k]);
          a_dwc.v[k] = fmaf(dl, C[i].v[k], a_dwc.v[k]);
          const float qh = (q[i].v[k] - muQ.v[k]) * rstd.v[k];
          const float o = fmaf(qh, gam.v[k], bet.v[k]);
          a_dw2.v[k] = fmaf(gpv, fmaxf(o, 0.f), a_dw2.v[k]);
          const float go = o > 0.f ? gpv * w2.v[k] : 0.f;
          a_db.v[k] += go;
          a_dg.v[k] = fmaf(go, qh, a_dg.v[k]);
          m1.v[k] = fmaf(gam.v[k], go, m1.v[k]);
          m2.v[k] = fmaf(gam.v[k] * go, qh, m2.v[k]);
        }
        stv<CPL>(p.gC + (size_t)v * HID + c, gc);
        stv<CPL>(p.gH + (size_t)v * HID + c, gh[i]);
        if (lane == 0) p.gp[v] = gpv;
        a_dbc2 += gpv;
      }
    }
#pragma unroll
    for (int k = 0; k < CPL; ++k) { m1.v[k] /= n; m2.v[k] /= n; }
    __syncwarp();
    // ---- pass C: per-graph BN backward -> g_q (two loads per row: 8 rows in flight)
    constexpr int RBC = 8;
    for (int vb = v0; vb < v1; vb += RBC) {
      float gpv[RBC];
      V q[RBC];
#pragma unroll
      for (int i = 0; i < RBC; ++i) {
        const int v = min(vb + i, v1 - 1);
        gpv[i] = __ldcg(p.gp + v);
        q[i] = ldv<CPL>(p.q + (size_t)v * HID + c);
      }
#pragma unroll
      for (int i = 0; i < RBC; ++i) {
        const int v = vb + i;
        if (v >= v1) break;
        V gq;
#pragma unroll
        for (int k = 0; k < CPL; ++k) {
          const float qh = (q[i].v[k] - muQ.v[k]) * rstd.v[k];
          const float o = fmaf(qh, gam.v[k], bet.v[k]);
          const float go = o > 0.f ? gpv[i] * w2.v[k] : 0.f;
          gq.v[k] = rstd.v[k] * (gam.v[k] * go - m1.v[k] - qh * m2.v[k]);
        }
        stv<CPL>(p.g_q + (size_t)v * HID + c, gq);
#pragma unroll
        for (int k = 0; k < CPL; ++k) gqmax = fmaxf(gqmax, fabsf(gq.v[k]));
      }
    }
  }
  if (p.gmax_q) {                // max is order-independent: the atomic keeps the result deterministic
    gqmax = warp_max(gqmax);
    if (lane == 0 && gqmax > 0.f) atomicMax(p.gmax_q, __float_as_uint(gqmax));
  }
  // ---- parameter-gradient partials: warp -> CTA -> last CTA
  float* r = s_red + warp * 5 * HID;
  stv<CPL>(r + c, a_dg); stv<CPL>(r + HID + c, a_db); stv<CPL>(r + 2 * HID + c, a_dw2); stv<CPL>(r + 3 * HID + c, a_dwc);
  if (lane == 0) r[4 * HID] = a_dbc2;
  __syncthreads();
  for (int j = threadIdx.x; j < 4 * HID + 1; j += NT) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < NT / 32; ++w) s += s_red[w * 5 * HID + j];
    p.part[(size_t)blockIdx.x * 5 * HID + j] = s;
  }
  if (!last_cta_arrives(p.counter)) return;
  for (int j = threadIdx.x; j < 4 * HID + 1; j += NT) {
    // four interleaved partial sums: 32 independent loads in flight instead of a chain of ~300 L2 round trips
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    const int nb = (int)gridDim.x;
    const float* src = p.part + j;
    int b = 0;
#pragma unroll 8
    for (; b + 3 < nb; b += 4) {
      s0 += (double)__ldcg(src + (size_t)b * 5 * HID);
      s1 += (double)__ldcg(src + (size_t)(b + 1) * 5 * HID);
      s2 += (double)__ldcg(src + (size_t)(b + 2) * 5 * HID);
      s3 += (double)__ldcg(src + (size_t)(b + 3) * 5 * HID);
    }
    for (; b < nb; ++b) s0 += (double)__ldcg(src + (size_t)b * 5 * HID);
    const float f = (float)((s0 + s1) + (s2 + s3));
    if (j < HID) p.d_gamma_c[j] = f;
    else if (j < 2 * HID) p.d_beta_c[j - HID] = f;
    else if (j < 3 * HID) p.d_wc2[j - 2 * HID] = f;
    else if (j < 4 * HID) { p.d_attn_w[HID + j - 3 * HID] = f; p.d_attn_w[j - 3 * HID] = 0.f; }  // core half: exactly 0 (F14)
    else { p.d_bc2[0] = f; p.d_attn_b[0] = 0.f; }
  }
}
void launch_graph_gate_bwd(const GraphGateBwdArgs& a, int hidden, cudaStream_t s) {
  // latency-bound warp-per-graph loops: as many resident warps as fit
  if (hidden == 64) {
    const int grid = min((a.B + 7) / 8, 4 * num_sms());
    launch_k((graph_gate_bwd_kernel<64, kThreads>), dim3(grid), dim3(kThreads), 0, s, a);
  } else {
    const int grid = min((a.B + 7) / 8, 4 * num_sms());
    launch_k((graph_gate_bwd_kernel<128, kThreads>), dim3(grid), dim3(kThreads), 0, s, a);
  }
}

// ------------------------------------------------------------------------------------------------
// head MLP forward: Z = Wm2 relu(Wm1 [noisy || alpha*C] + bm1) + bm2
// ------------------------------------------------------------------------------------------------
// HT rows per tile: 64 at HID = 64; 32 at HID = 128 (tile [HT][2H] + W1t [2H][H] + W2t [H][H] = 225 KB)
template <int HID, int HT> struct HeadFwdSmem { float tile[HT * (2 * HID + 4)]; float w1t[2 * HID * HID]; float w2t[HID * HID]; };

template <int HID, int HT>
__device__ __forceinline__ void head_load_tile(float* tile, const float* __restrict__ noisy, const float* __restrict__ C,
                                               const float* __restrict__ alpha, int base, int N, float* imap, float* aC,
                                               bf16_t* aC_bf) {
  constexpr int HLD = 2 * HID + 4, LPR = 2 * HID / 4;      // lanes per row of the [noisy || alpha C] tile (4 channels each)
  for (int i = threadIdx.x; i < HT * LPR; i += kThreads) {
    const int r = i / LPR, l = i % LPR;
    const int v = base + r;
    float4 val = make4(0.f);
    if (v < N) {
      if (l < LPR / 2) {
        val = ld4(noisy + (size_t)v * HID + l * 4);
      } else {
        const float al = __ldg(alpha + v);
        const float4 cc = ld4(C + (size_t)v * HID + (l - LPR / 2) * 4);
        val = make_float4(al * cc.x, al * cc.y, al * cc.z, al * cc.w);
        if (aC) st4(aC + (size_t)v * HID + (l - LPR / 2) * 4, val);
        if (aC_bf) st4a<true>(reinterpret_cast<float*>(aC_bf), (size_t)v * HID + (l - LPR / 2) * 4, val);
      }
      if (imap) st4(imap + (size_t)v * 2 * HID + l * 4, val);
    }
    st4(tile + r * HLD + l * 4, val);
  }
}

template <int HID, int HT>
__global__ void __launch_bounds__(kThreads, HID == 64 ? 2 : 1)
head_fwd_kernel(HeadFwdArgs p) {
  pdl_sync();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  HeadFwdSmem<HID, HT>& sm = *reinterpret_cast<HeadFwdSmem<HID, HT>*>(smem_raw);
  constexpr int GLD = HID + 4, HLD = 2 * HID + 4;
  using M = NNMap<HT, HID>;
  load_matrix<HID>(sm.w1t, HID, p.W1t, 2 * HID);
  load_matrix<HID>(sm.w2t, HID, p.W2t, HID);
  const int n_tiles = (p.N + HT - 1) / HT;
  const int c0 = M::col0(), r0 = M::row0();
  const float4 b1 = ldg4(p.b1 + c0), b2 = ldg4(p.b2 + c0);
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int base = tile * HT;
    __syncthreads();
    head_load_tile<HID, HT>(sm.tile, p.noisy, p.C, p.alpha, base, p.N, p.imap, p.aC, p.aC_bf);
    __syncthreads();
    float acc[M::TM][4];
#pragma unroll
    for (int m = 0; m < M::TM; ++m) { acc[m][0] = b1.x; acc[m][1] = b1.y; acc[m][2] = b1.z; acc[m][3] = b1.w; }
    gemm_nn<HT, 2 * HID, HID>(sm.tile, HLD, sm.w1t, HID, acc);
    __syncthreads();
#pragma unroll
    for (int m = 0; m < M::TM; ++m) {
      const float4 rv = relu4(make_float4(acc[m][0], acc[m][1], acc[m][2], acc[m][3]));
      st4(sm.tile + (r0 + m) * GLD + c0, rv);
      const int v = base + r0 + m;
      if (v < p.N) {
        if (p.r) st4(p.r + (size_t)v * HID + c0, rv);
        if (p.r_bf) st4a<true>(reinterpret_cast<float*>(p.r_bf), (size_t)v * HID + c0, rv);
      }
    }
    __syncthreads();
#pragma unroll
    for (int m = 0; m < M::TM; ++m) { acc[m][0] = b2.x; acc[m][1] = b2.y; acc[m][2] = b2.z; acc[m][3] = b2.w; }
    gemm_nn<HT, HID, HID>(sm.tile, GLD, sm.w2t, HID, acc);
#pragma unroll
    for (int m = 0; m < M::TM; ++m) {
      const int v = base + r0 + m;
      if (v < p.N) st4(p.Z + (size_t)v * HID + c0, make_float4(acc[m][0], acc[m][1], acc[m][2], acc[m][3]));
    }
  }
}
template <int H, int HT>
static void launch_head_fwd_t(const HeadFwdArgs& a, cudaStream_t s) {
  using S = HeadFwdSmem<H, HT>;
  static bool once = (cudaFuncSetAttribute(head_fwd_kernel<H, HT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(S)), true);
  (void)once;
  const int grid = min((a.N + HT - 1) / HT, (H == 64 ? 2 : 1) * num_sms());
  launch_k((head_fwd_kernel<H, HT>), dim3(grid), dim3(kThreads), sizeof(S), s, a);
}
void launch_head_fwd(const HeadFwdArgs& a, int hidden, cudaStream_t s) {
  const uintptr_t al32 = (uintptr_t)a.noisy | (uintptr_t)a.C | (uintptr_t)a.Z | (uintptr_t)a.r | (uintptr_t)a.aC | (uintptr_t)a.imap |
                         (uintptr_t)a.r_bf | (uintptr_t)a.aC_bf;
  static int head_ffma = -1;                 // SCGIB_HEAD_FFMA=1: FFMA tiles also at hidden 64 (cross-check)
  if (head_ffma < 0) { const char* e = getenv("SCGIB_HEAD_FFMA"); head_ffma = (e && e[0] == '1') ? 1 : 0; }
  if (hidden == 64 && a.W1n && a.W2n && (al32 & 31u) == 0 && tensor_core_mode() != 0 && !head_ffma) {   // 32-byte row accesses
    launch_head_fwd_tc(a, s);
    return;
  }
  if (hidden == 64) launch_head_fwd_t<64, 64>(a, s); else launch_head_fwd_t<128, 32>(a, s);
}

// The head MLP backward is the GIN layer backward kernel run on the two K = H halves of the first head layer (api.cu).
// prep: dense copies W1a = W1[:, :H], W1b = W1[:, H:] and the identity BatchNorm-backward constants
// (bn = {0, 1, 1, 0}, cvec = 0: g_y = g_o).  interleave: grads slot [2][H][H] (dW1a | dW1b) -> [H][2H] in place.
__global__ void __launch_bounds__(kThreads)
head_bwd_prep_kernel(const float* __restrict__ W1, float* __restrict__ W1a, float* __restrict__ W1b, float* __restrict__ bn,
                     float* __restrict__ cvec, int HID) {
  pdl_sync();
  for (int i = blockIdx.x * kThreads + threadIdx.x; i < HID * 2 * HID; i += gridDim.x * kThreads) {
    const int o = i / (2 * HID), k = i % (2 * HID);
    const float w = W1[i];
    if (k < HID) W1a[o * HID + k] = w; else W1b[o * HID + k - HID] = w;
  }
  if (blockIdx.x == 0) {
    for (int i = threadIdx.x; i < 4 * HID; i += kThreads) bn[i] = (i >= HID && i < 3 * HID) ? 1.f : 0.f;   // mean 0, rstd 1, gamma 1, beta 0
    for (int i = threadIdx.x; i < 2 * HID; i += kThreads) cvec[i] = 0.f;
  }
}
__global__ void identity_bn_kernel(float* __restrict__ bn, int HID) {
  pdl_sync();
  for (int i = threadIdx.x; i < 4 * HID; i += blockDim.x) bn[i] = (i >= HID && i < 3 * HID) ? 1.f : 0.f;
}
void launch_identity_bn(float* bn, int hidden, cudaStream_t s) { identity_bn_kernel<<<1, 128, 0, s>>>(bn, hidden); }
void launch_head_bwd_prep(const float* W1, float* W1a, float* W1b, float* bn, float* cvec, int hidden, cudaStream_t s) {
  launch_k((head_bwd_prep_kernel), dim3(8), dim3(kThreads), 0, s, W1, W1a, W1b, bn, cvec, hidden);
}

__global__ void __launch_bounds__(kThreads) head_dw1_interleave_kernel(float* __restrict__ dW1, int HID) {
  pdl_sync();
  extern __shared__ __align__(16) float s_w[];            // [2 * HID * HID]
  for (int i = threadIdx.x; i < 2 * HID * HID; i += kThreads) s_w[i] = dW1[i];
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * HID * HID; i += kThreads) {
    const int o = i / (2 * HID), k = i % (2 * HID);
    dW1[i] = k < HID ? s_w[o * HID + k] : s_w[HID * HID + o * HID + k - HID];
  }
}
void launch_head_dw1_interleave(float* dW1, int hidden, cudaStream_t s) {
  const int bytes = 2 * hidden * hidden * (int)sizeof(float);
  static bool once = (cudaFuncSetAttribute(head_dw1_interleave_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 128 * 128 * 4), true);
  (void)once;
  launch_k((head_dw1_interleave_kernel), dim3(1), dim3(kThreads), bytes, s, dW1, hidden);
}

}  // namespace scgib

// ------------------------------------------------------------------------------------------------
// Stand-alone operators behind the op-level C ABI (scgib_core_cand_attn_*_f32, scgib_segment_sum_bwd_f32): the whole-step
// functions run the same math fused into ego_pool_fwd / graph_gate_fwd / graph_gate_bwd.
// ------------------------------------------------------------------------------------------------
namespace scgib {

// attention over the candidates of each graph (models.py:738-748; the core half of attn_layer and its bias cancel in the
// softmax, SURVEY F14): logit_v = w_cand . C_v, alpha = softmax over the graph's nodes, T_v = alpha_v C_v.  Warp per graph.
__global__ void __launch_bounds__(kThreads)
attn_fwd_kernel(const float* __restrict__ C, const int32_t* __restrict__ graph_ptr, int B, int H, const float* __restrict__ w_cand,
                float* __restrict__ alpha, float* __restrict__ T) {
  pdl_sync();
  const int lane = threadIdx.x & 31;
  for (int g = blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); g < B; g += gridDim.x * (kThreads / 32)) {
    const int v0 = __ldg(graph_ptr + g), v1 = __ldg(graph_ptr + g + 1);
    float mx = -INFINITY;
    for (int v = v0; v < v1; ++v) {
      float d = 0.f;
      for (int c = lane; c < H; c += 32) d = fmaf(__ldg(w_cand + c), C[(size_t)v * H + c], d);
      d = warp_sum(d);
      if (lane == 0) alpha[v] = d;                 // logits first
      mx = fmaxf(mx, d);
    }
    __syncwarp();
    float se = 0.f;
    for (int v = v0 + lane; v < v1; v += 32) se += expf(alpha[v] - mx);
    se = warp_sum(se);
    __syncwarp();
    for (int v = v0 + lane; v < v1; v += 32) alpha[v] = expf(alpha[v] - mx) / se;
    __syncwarp();
    if (T)
      for (int v = v0; v < v1; ++v) {
        const float a = alpha[v];
        for (int c = lane; c < H; c += 32) T[(size_t)v * H + c] = a * C[(size_t)v * H + c];
      }
  }
}
void launch_attn_fwd(const float* C, const int32_t* graph_ptr, int B, int H, const float* w_cand, float* alpha, float* T, cudaStream_t s) {
  launch_k((attn_fwd_kernel), dim3(min((B + 7) / 8, 8 * num_sms())), dim3(kThreads), 0, s, C, graph_ptr, B, H, w_cand, alpha, T);
}

// backward: d alpha_v = gT_v . C_v;  d logit_v = alpha_v (d alpha_v - sum_u alpha_u d alpha_u);  gC_v = alpha_v gT_v + d logit_v w_cand;
// d w_cand = sum_v d logit_v C_v  (per-graph partials dwp [B][H], summed by the caller's reduction in graph order)
__global__ void __launch_bounds__(kThreads)
attn_bwd_kernel(const float* __restrict__ C, const float* __restrict__ alpha, const float* __restrict__ gT,
                const int32_t* __restrict__ graph_ptr, int B, int H, const float* __restrict__ w_cand, float* __restrict__ gC,
                float* __restrict__ dwp, float* __restrict__ scratch) {
  pdl_sync();
  const int lane = threadIdx.x & 31;
  for (int g = blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); g < B; g += gridDim.x * (kThreads / 32)) {
    const int v0 = __ldg(graph_ptr + g), v1 = __ldg(graph_ptr + g + 1);
    float S = 0.f;
    for (int v = v0; v < v1; ++v) {
      float d = 0.f;
      for (int c = lane; c < H; c += 32) d = fmaf(gT[(size_t)v * H + c], C[(size_t)v * H + c], d);
      d = warp_sum(d);
      if (lane == 0) scratch[v] = d;
      S = fmaf(alpha[v], d, S);
    }
    __syncwarp();
    for (int c = lane; c < H; c += 32) {
      const float w = __ldg(w_cand + c);
      float dw = 0.f;
      for (int v = v0; v < v1; ++v) {
        const float a = alpha[v], dl = a * (scratch[v] - S);
        gC[(size_t)v * H + c] = fmaf(dl, w, a * gT[(size_t)v * H + c]);
        dw = fmaf(dl, C[(size_t)v * H + c], dw);
      }
      dwp[(size_t)g * H + c] = dw;
    }
  }
}
void launch_attn_bwd(const float* C, const float* alpha, const float* gT, const int32_t* graph_ptr, int B, int H, const float* w_cand,
                     float* gC, float* dwp, float* scratch, cudaStream_t s) {
  launch_k((attn_bwd_kernel), dim3(min((B + 7) / 8, 8 * num_sms())), dim3(kThreads), 0, s, C, alpha, gT, graph_ptr, B, H, w_cand, gC, dwp, scratch);
}

// backward of dgl.sum_nodes: g_in[row] = g_out[segment of row]
__global__ void __launch_bounds__(kThreads)
segment_sum_bwd_kernel(const float* __restrict__ g_out, const int32_t* __restrict__ seg_ptr, int S, int H, float* __restrict__ g_in) {
  pdl_sync();
  const int lane = threadIdx.x & 31;
  for (int sgm = blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); sgm < S; sgm += gridDim.x * (kThreads / 32)) {
    const int r0 = __ldg(seg_ptr + sgm), r1 = __ldg(seg_ptr + sgm + 1);
    for (int c = lane * 4; c < H; c += 128) {
      const float4 g = ld4(g_out + (size_t)sgm * H + c);
      for (int r = r0; r < r1; ++r) st4(g_in + (size_t)r * H + c, g);
    }
  }
}
void launch_segment_sum_bwd(const float* g_out, const int32_t* seg_ptr, int S, int H, float* g_in, cudaStream_t s) {
  launch_k((segment_sum_bwd_kernel), dim3(min((S + 7) / 8, 16 * num_sms())), dim3(kThreads), 0, s, g_out, seg_ptr, S, H, g_in);
}

// out[c] = sum_g part[g][c] in graph order (fp64 accumulate): fixed-order column sums of per-graph partials
__global__ void __launch_bounds__(kThreads)
colsum_rows_kernel(const float* __restrict__ part, int R, int H, float* __restrict__ out) {
  pdl_sync();
  for (int c = blockIdx.x * kThreads + threadIdx.x; c < H; c += gridDim.x * kThreads) {
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    int r = 0;
    for (; r + 3 < R; r += 4) {
      s0 += (double)part[(size_t)r * H + c]; s1 += (double)part[(size_t)(r + 1) * H + c];
      s2 += (double)part[(size_t)(r + 2) * H + c]; s3 += (double)part[(size_t)(r + 3) * H + c];
    }
    for (; r < R; ++r) s0 += (double)part[(size_t)r * H + c];
    out[c] = (float)((s0 + s1) + (s2 + s3));
  }
}
void launch_colsum_rows(const float* part, int R, int H, float* out, cudaStream_t s) {
  launch_k((colsum_rows_kernel), dim3(1), dim3(kThreads), 0, s, part, R, H, out);
}

}  // namespace scgib
