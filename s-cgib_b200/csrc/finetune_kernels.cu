// finetune_kernels.cu - the fine-tuning head of Mainmodel_finetuning.forward (reference models.py:501-520):
//   Set2Set(hidden, n_iters = 2, 1 LSTM layer) readout (DGL 1.1.0 dgl.nn.Set2Set, call site models.py:365, 515)
//   -> predict = Linear(2H, H) - ReLU - Linear(H, C)  (models.py:386-397) -> optional sigmoid (models.py:519-520).
//
// Every graph is independent in this head (the LSTM runs over the batch of graphs, not over time across graphs), so
// the whole forward is ONE kernel: a CTA owns G graphs, runs the LSTM cell for them out of shared memory (weights are
// streamed k-major from L2 and reused by the G graphs), then one warp per graph does the node attention
// (e_v = z_v . q, softmax over the graph, r = sum alpha_v z_v), and after the last iteration the predict MLP.
// The backward is one per-graph kernel of the same shape (activation gradients, g_Z) followed by small fixed-order
// A^T B reductions over the graphs for the weight gradients (no float atomics).
// Heads with more than kMaxC outputs keep everything up to u = relu(Wp1 q* + bp1) in the per-graph kernels; the output
// layer scores = act(u Wp2^T + bp2) and its backward g_u = relu'(u) * ((g_scores . act') Wp2) run as tiled kernels over
// [B x C] / [B x H] instead of one Wp2 row per thread.
#include "kernels.cuh"

namespace scgib {

namespace {
constexpr int FG = 8;   // graphs per CTA = warps per CTA
constexpr int kMaxC = 64;   // widest output layer run inside the per-graph kernels (s_gpre of the backward)

__device__ __forceinline__ float sigmoidf_acc(float x) { return 1.f / (1.f + expf(-x)); }

// out[g][j] = bias(j) + sum_k in[g][k] * WT[k][j]   for the CTA's FG graphs (in/out in shared memory)
template <class BiasF>
__device__ __forceinline__ void matvec_kmajor(const float* __restrict__ WT, int K, int NOUT, const float* s_in, int ld_in,
                                              float* s_out, int ld_out, BiasF bias) {
  for (int j = threadIdx.x; j < NOUT; j += kThreads) {
    float acc[FG];
    const float b = bias(j);
#pragma unroll
    for (int g = 0; g < FG; ++g) acc[g] = b;
#pragma unroll 4
    for (int k = 0; k < K; ++k) {
      const float w = __ldg(WT + (size_t)k * NOUT + j);
#pragma unroll
      for (int g = 0; g < FG; ++g) acc[g] = fmaf(w, s_in[g * ld_in + k], acc[g]);
    }
#pragma unroll
    for (int g = 0; g < FG; ++g) s_out[g * ld_out + j] = acc[g];
  }
}

// per-lane channel slice of a row: H/32 consecutive floats
template <int H> struct Lane;
template <> struct Lane<32> {   // small feature widths (Set2Set over raw features, zero-padded to 32 channels)
  float v[1];
  __device__ __forceinline__ void load(const float* row, int lane) { v[0] = row[lane]; }
  __device__ __forceinline__ void store(float* row, int lane) const { row[lane] = v[0]; }
  static constexpr int W = 1;
};
template <> struct Lane<64> {
  float v[2];
  __device__ __forceinline__ void load(const float* row, int lane) { const float2 t = *reinterpret_cast<const float2*>(row + lane * 2); v[0] = t.x; v[1] = t.y; }
  __device__ __forceinline__ void store(float* row, int lane) const { *reinterpret_cast<float2*>(row + lane * 2) = make_float2(v[0], v[1]); }
  static constexpr int W = 2;
};
template <> struct Lane<128> {
  float v[4];
  __device__ __forceinline__ void load(const float* row, int lane) { const float4 t = ld4(row + lane * 4); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; }
  __device__ __forceinline__ void store(float* row, int lane) const { st4(row + lane * 4, make_float4(v[0], v[1], v[2], v[3])); }
  static constexpr int W = 4;
};
template <int H>
__device__ __forceinline__ float lane_dot(const Lane<H>& a, const Lane<H>& b) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < Lane<H>::W; ++i) s = fmaf(a.v[i], b.v[i], s);
  return warp_sum(s);
}

template <int H>
struct FtSmem {
  float in[FG][3 * H];     // [q* (2H) | h (H)]  LSTM input of the next step
  float gates[FG][4 * H];
  float c[FG][H];
  float mid[FG][H];
};

template <int H>
__global__ void __launch_bounds__(kThreads) finetune_head_fwd_kernel(FinetuneHeadFwdArgs p) {
  __shared__ FtSmem<H> sm;
  const int g0 = blockIdx.x * FG;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int B = p.B, T = p.T;
  for (int i = threadIdx.x; i < FG * 3 * H; i += kThreads) (&sm.in[0][0])[i] = 0.f;
  for (int i = threadIdx.x; i < FG * H; i += kThreads) (&sm.c[0][0])[i] = 0.f;
  __syncthreads();
  for (int t = 0; t < T; ++t) {
    // ---- LSTM cell (torch gate order i, f, g, o): gates = W_ih q* + b_ih + W_hh h + b_hh
    {
      const float* bih = p.b_ih; const float* bhh = p.b_hh;
      // [WihT ; WhhT] are stored back to back: one k-major [3H][4H] matrix
      matvec_kmajor(p.WlstmT, 3 * H, 4 * H, &sm.in[0][0], 3 * H, &sm.gates[0][0], 4 * H,
                    [&](int j) { return __ldg(bih + j) + __ldg(bhh + j); });
    }
    __syncthreads();
    for (int i = threadIdx.x; i < FG * H; i += kThreads) {
      const int g = i / H, c = i % H;
      const float ig = sigmoidf_acc(sm.gates[g][c]), fg = sigmoidf_acc(sm.gates[g][H + c]);
      const float gg = tanhf(sm.gates[g][2 * H + c]), og = sigmoidf_acc(sm.gates[g][3 * H + c]);
      const float cn = fmaf(fg, sm.c[g][c], ig * gg);
      const float h = og * tanhf(cn);
      sm.c[g][c] = cn;
      sm.in[g][c] = h;             // q half of q*
      sm.in[g][2 * H + c] = h;     // hidden state
      if (g0 + g < B) {
        float* gs = p.gates + ((size_t)t * B + g0 + g) * 4 * H;
        gs[c] = ig; gs[H + c] = fg; gs[2 * H + c] = gg; gs[3 * H + c] = og;
        p.cst[((size_t)t * B + g0 + g) * H + c] = cn;
      }
    }
    __syncthreads();
    // ---- node attention of graph g0 + warp
    const int g = g0 + warp;
    if (g < B) {
      const int v0 = __ldg(p.graph_ptr + g), v1 = __ldg(p.graph_ptr + g + 1);
      Lane<H> q;
      q.load(&sm.in[warp][0], lane);
      float* al = p.alpha + (size_t)t * p.N;
      float mx = -INFINITY;
      constexpr int RB = 4;               // rows in flight: the loads and the shuffle reductions of RB rows overlap
      for (int vb = v0; vb < v1; vb += RB) {
        Lane<H> z[RB];
        float e[RB];
#pragma unroll
        for (int r = 0; r < RB; ++r) z[r].load(p.Z + (size_t)min(vb + r, v1 - 1) * H, lane);
#pragma unroll
        for (int r = 0; r < RB; ++r) {
          e[r] = 0.f;
#pragma unroll
          for (int i = 0; i < Lane<H>::W; ++i) e[r] = fmaf(z[r].v[i], q.v[i], e[r]);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
          for (int r = 0; r < RB; ++r) e[r] += __shfl_xor_sync(0xffffffffu, e[r], o);
        }
#pragma unroll
        for (int r = 0; r < RB; ++r) {
          if (vb + r < v1) {
            if (lane == 0) al[vb + r] = e[r];
            mx = fmaxf(mx, e[r]);
          }
        }
      }
      __syncwarp();
      Lane<H> acc;
#pragma unroll
      for (int i = 0; i < Lane<H>::W; ++i) acc.v[i] = 0.f;
      float den = 0.f;
      for (int vb = v0; vb < v1; vb += RB) {
        Lane<H> z[RB];
        float ex[RB];
#pragma unroll
        for (int r = 0; r < RB; ++r) {
          const int v = min(vb + r, v1 - 1);
          z[r].load(p.Z + (size_t)v * H, lane);
          ex[r] = al[v];
        }
#pragma unroll
        for (int r = 0; r < RB; ++r) {
          if (vb + r < v1) {
            const float x = expf(ex[r] - mx);
            den += x;
#pragma unroll
            for (int i = 0; i < Lane<H>::W; ++i) acc.v[i] = fmaf(x, z[r].v[i], acc.v[i]);
          }
        }
      }
      const float inv = den > 0.f ? 1.f / den : 0.f;
      __syncwarp();
      for (int v = v0 + lane; v < v1; v += 32) al[v] = expf(al[v] - mx) * inv;
#pragma unroll
      for (int i = 0; i < Lane<H>::W; ++i) acc.v[i] *= inv;
      acc.store(&sm.in[warp][H], lane);                                 // r half of q*
      float* qs = p.qstar + ((size_t)t * B + g) * 2 * H;
      q.store(qs, lane);
      acc.store(qs + H, lane);
    }
    __syncthreads();
  }
  if (p.C == 0) return;                 // readout only (Set2Set without a predict head)
  // ---- predict: u = relu(Wp1 q* + bp1), s = Wp2 u + bp2, optional sigmoid
  {
    const float* b1 = p.bp1;
    matvec_kmajor(p.Wp1T, 2 * H, H, &sm.in[0][0], 3 * H, &sm.mid[0][0], H, [&](int j) { return __ldg(b1 + j); });
  }
  __syncthreads();
  for (int i = threadIdx.x; i < FG * H; i += kThreads) {
    const int g = i / H, c = i % H;
    const float u = fmaxf(sm.mid[g][c], 0.f);
    sm.mid[g][c] = u;
    if (g0 + g < B) p.rp[(size_t)(g0 + g) * H + c] = u;
  }
  if (p.C > kMaxC) return;              // the output layer runs as a tiled kernel (ft_out_fwd_kernel)
  __syncthreads();
  for (int i = threadIdx.x; i < FG * p.C; i += kThreads) {
    const int g = i / p.C, c = i % p.C;
    if (g0 + g >= B) continue;
    float s = __ldg(p.bp2 + c);
    const float* w = p.Wp2 + (size_t)c * H;      // natural [C][H]
    for (int k = 0; k < H; ++k) s = fmaf(__ldg(w + k), sm.mid[g][k], s);
    if (p.sigmoid) s = sigmoidf_acc(s);
    p.scores[(size_t)(g0 + g) * p.C + c] = s;
  }
}

// out[g][k] = sum_j in[g][j] * W[j][k]   (W natural [J][K]: coalesced over k)
__device__ __forceinline__ void matvec_natural(const float* __restrict__ W, int J, int K, const float* s_in, int ld_in,
                                               float* s_out, int ld_out) {
  for (int k = threadIdx.x; k < K; k += kThreads) {
    float acc[FG];
#pragma unroll
    for (int g = 0; g < FG; ++g) acc[g] = 0.f;
#pragma unroll 4
    for (int j = 0; j < J; ++j) {
      const float w = __ldg(W + (size_t)j * K + k);
#pragma unroll
      for (int g = 0; g < FG; ++g) acc[g] = fmaf(w, s_in[g * ld_in + j], acc[g]);
    }
#pragma unroll
    for (int g = 0; g < FG; ++g) s_out[g * ld_out + k] = acc[g];
  }
}

template <int H>
struct FtBwdSmem {
  float gq[FG][2 * H];     // gradient wrt q*_t
  float gh[FG][H];         // gradient wrt h_t from step t+1 (W_hh path)
  float gc[FG][H];         // gradient wrt c_t from step t+1
  float dg[FG][4 * H];     // pre-activation gate gradients of step t
  float tmp[FG][H];
};

template <int H>
__global__ void __launch_bounds__(kThreads) finetune_head_bwd_kernel(FinetuneHeadBwdArgs p) {
  __shared__ FtBwdSmem<H> sm;
  __shared__ float s_gpre[FG][kMaxC];
  const int g0 = blockIdx.x * FG;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int B = p.B, T = p.T, C = p.C;
  for (int i = threadIdx.x; i < FG * H; i += kThreads) { (&sm.gh[0][0])[i] = 0.f; (&sm.gc[0][0])[i] = 0.f; }
  if (C > kMaxC) {
    // ---- predict backward from g_u (masked, written by ft_out_bwd_kernel)
    for (int i = threadIdx.x; i < FG * H; i += kThreads) {
      const int g = i / H, c = i % H;
      sm.tmp[g][c] = g0 + g < B ? p.g_u[(size_t)(g0 + g) * H + c] : 0.f;
    }
    __syncthreads();
    matvec_natural(p.Wp1, H, 2 * H, &sm.tmp[0][0], H, &sm.gq[0][0], 2 * H);    // g wrt q*_{T-1}
  } else if (C > 0) {
    // ---- predict backward
    for (int i = threadIdx.x; i < FG * C; i += kThreads) {
      const int g = i / C, c = i % C;
      float v = 0.f;
      if (g0 + g < B) {
        v = p.g_scores[(size_t)(g0 + g) * C + c];
        if (p.sigmoid) { const float s = p.scores[(size_t)(g0 + g) * C + c]; v *= s * (1.f - s); }
        p.g_pre[(size_t)(g0 + g) * C + c] = v;
      }
      s_gpre[g][c] = v;
    }
    __syncthreads();
    matvec_natural(p.Wp2, C, H, &s_gpre[0][0], kMaxC, &sm.tmp[0][0], H);       // g_u (before the ReLU mask)
    __syncthreads();
    for (int i = threadIdx.x; i < FG * H; i += kThreads) {
      const int g = i / H, c = i % H;
      float v = 0.f;
      if (g0 + g < B) {
        v = p.rp[(size_t)(g0 + g) * H + c] > 0.f ? sm.tmp[g][c] : 0.f;
        p.g_u[(size_t)(g0 + g) * H + c] = v;
      }
      sm.tmp[g][c] = v;
    }
    __syncthreads();
    matvec_natural(p.Wp1, H, 2 * H, &sm.tmp[0][0], H, &sm.gq[0][0], 2 * H);    // g wrt q*_{T-1}
  } else {
    for (int i = threadIdx.x; i < FG * 2 * H; i += kThreads) (&sm.gq[0][0])[i] = 0.f;
  }
  __syncthreads();
  if (p.g_readout) {                      // upstream gradient given directly at the Set2Set output q*_{T-1}
    for (int i = threadIdx.x; i < FG * 2 * H; i += kThreads) {
      const int g = i / (2 * H), c = i % (2 * H);
      if (g0 + g < B) sm.gq[g][c] += p.g_readout[(size_t)(g0 + g) * 2 * H + c];
    }
    __syncthreads();
  }
  for (int t = T - 1; t >= 0; --t) {
    // ---- attention backward of graph g0 + warp; adds the attention path to the q half of gq
    const int g = g0 + warp;
    if (g < B) {
      const int v0 = __ldg(p.graph_ptr + g), v1 = __ldg(p.graph_ptr + g + 1);
      const float* al = p.alpha + (size_t)t * p.N;
      const float* qs = p.qstar + ((size_t)t * B + g) * 2 * H;
      Lane<H> q, gr;
      q.load(qs, lane);
      gr.load(&sm.gq[warp][H], lane);
      float S = 0.f;
      constexpr int RB = 4;
      for (int vb = v0; vb < v1; vb += RB) {
        Lane<H> z[RB];
        float ga[RB], av[RB];
#pragma unroll
        for (int r = 0; r < RB; ++r) {
          const int v = min(vb + r, v1 - 1);
          z[r].load(p.Z + (size_t)v * H, lane);
          av[r] = __ldg(al + v);
        }
#pragma unroll
        for (int r = 0; r < RB; ++r) {
          ga[r] = 0.f;
#pragma unroll
          for (int i = 0; i < Lane<H>::W; ++i) ga[r] = fmaf(z[r].v[i], gr.v[i], ga[r]);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
          for (int r = 0; r < RB; ++r) ga[r] += __shfl_xor_sync(0xffffffffu, ga[r], o);
        }
#pragma unroll
        for (int r = 0; r < RB; ++r) {
          if (vb + r < v1) {
            if (lane == 0) p.gp[vb + r] = ga[r];
            S = fmaf(av[r], ga[r], S);
          }
        }
      }
      __syncwarp();
      Lane<H> accq;
#pragma unroll
      for (int i = 0; i < Lane<H>::W; ++i) accq.v[i] = 0.f;
      for (int vb = v0; vb < v1; vb += RB) {
        Lane<H> z[RB], gz[RB];
        float a[RB], gpv[RB];
#pragma unroll
        for (int r = 0; r < RB; ++r) {
          const int v = min(vb + r, v1 - 1);
          z[r].load(p.Z + (size_t)v * H, lane);
          a[r] = __ldg(al + v);
          gpv[r] = p.gp[v];
          if (t == T - 1) {
#pragma unroll
            for (int i = 0; i < Lane<H>::W; ++i) gz[r].v[i] = 0.f;
          } else {
            gz[r].load(p.gZ + (size_t)v * H, lane);
          }
        }
#pragma unroll
        for (int r = 0; r < RB; ++r) {
          if (vb + r < v1) {
            const float ge = a[r] * (gpv[r] - S);
#pragma unroll
            for (int i = 0; i < Lane<H>::W; ++i) {
              gz[r].v[i] += fmaf(a[r], gr.v[i], ge * q.v[i]);
              accq.v[i] = fmaf(ge, z[r].v[i], accq.v[i]);
            }
            gz[r].store(p.gZ + (size_t)(vb + r) * H, lane);
          }
        }
      }
      Lane<H> gqv;
      gqv.load(&sm.gq[warp][0], lane);
#pragma unroll
      for (int i = 0; i < Lane<H>::W; ++i) gqv.v[i] += accq.v[i];
      gqv.store(&sm.gq[warp][0], lane);
    }
    __syncthreads();
    // ---- LSTM cell backward
    for (int i = threadIdx.x; i < FG * H; i += kThreads) {
      const int gg_ = i / H, c = i % H;
      float di = 0.f, df = 0.f, dgg = 0.f, dout = 0.f, gcp = 0.f;
      if (g0 + gg_ < B) {
        const float* gs = p.gates + ((size_t)t * B + g0 + gg_) * 4 * H;
        const float ig = gs[c], fg = gs[H + c], gg = gs[2 * H + c], og = gs[3 * H + c];
        const float ct = p.cst[((size_t)t * B + g0 + gg_) * H + c];
        const float cprev = t > 0 ? p.cst[((size_t)(t - 1) * B + g0 + gg_) * H + c] : 0.f;
        const float tc = tanhf(ct);
        const float ghv = sm.gq[gg_][c] + sm.gh[gg_][c];
        const float gcv = sm.gc[gg_][c] + ghv * og * (1.f - tc * tc);
        di = gcv * gg * ig * (1.f - ig);
        df = gcv * cprev * fg * (1.f - fg);
        dgg = gcv * ig * (1.f - gg * gg);
        dout = ghv * tc * og * (1.f - og);
        gcp = gcv * fg;
        float* dgp = p.dgates + ((size_t)t * B + g0 + gg_) * 4 * H;
        dgp[c] = di; dgp[H + c] = df; dgp[2 * H + c] = dgg; dgp[3 * H + c] = dout;
      }
      sm.dg[gg_][c] = di; sm.dg[gg_][H + c] = df; sm.dg[gg_][2 * H + c] = dgg; sm.dg[gg_][3 * H + c] = dout;
      sm.gc[gg_][c] = gcp;
    }
    __syncthreads();
    if (t > 0) {
      matvec_natural(p.Wih, 4 * H, 2 * H, &sm.dg[0][0], 4 * H, &sm.gq[0][0], 2 * H);
      matvec_natural(p.Whh, 4 * H, H, &sm.dg[0][0], 4 * H, &sm.gh[0][0], H);
      __syncthreads();
    }
  }
}

// Output layer of heads with C > kMaxC.  A CTA owns a tile of RI * 16 graphs x 64 columns; thread (tx, ty) of the
// 16 x 16 grid owns graphs ty + 16 i and columns tx + 16 j (coalesced stores).  Operands go through shared memory in
// k-major chunks of 32.  Each output is a sequential fmaf chain over k (over c in the backward) from the bias (from 0),
// the order of the in-kernel path.
constexpr int OT = 64, OK = 32;

// scores[b][c] = act(bp2[c] + sum_k rp[b][k] Wp2[c][k])
__global__ void __launch_bounds__(kThreads) ft_out_fwd_kernel(const float* __restrict__ rp, const float* __restrict__ Wp2,
                                                              const float* __restrict__ bp2, int B, int C, int H, int sigmoid,
                                                              float* __restrict__ scores) {
  constexpr int RI = 4;
  __shared__ float sa[OK][RI * 16 + 1], sw[OK][OT + 1];     // [k][graph], [k][class]
  const int g0 = blockIdx.y * RI * 16, c0 = blockIdx.x * OT;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float acc[RI][4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int c = c0 + tx + 16 * j;
    const float b = c < C ? __ldg(bp2 + c) : 0.f;
#pragma unroll
    for (int i = 0; i < RI; ++i) acc[i][j] = b;
  }
  for (int k0 = 0; k0 < H; k0 += OK) {
    __syncthreads();
    for (int e = threadIdx.x; e < RI * 16 * OK; e += kThreads) {
      const int r = e / OK, k = e % OK;
      sa[k][r] = g0 + r < B ? __ldg(rp + (size_t)(g0 + r) * H + k0 + k) : 0.f;
    }
    for (int e = threadIdx.x; e < OT * OK; e += kThreads) {
      const int r = e / OK, k = e % OK;
      sw[k][r] = c0 + r < C ? __ldg(Wp2 + (size_t)(c0 + r) * H + k0 + k) : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int k = 0; k < OK; ++k) {
      float a[RI], w[4];
#pragma unroll
      for (int i = 0; i < RI; ++i) a[i] = sa[k][ty + 16 * i];
#pragma unroll
      for (int j = 0; j < 4; ++j) w[j] = sw[k][tx + 16 * j];
#pragma unroll
      for (int i = 0; i < RI; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(w[j], a[i], acc[i][j]);
    }
  }
#pragma unroll
  for (int i = 0; i < RI; ++i) {
    const int g = g0 + ty + 16 * i;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = c0 + tx + 16 * j;
      if (g < B && c < C) scores[(size_t)g * C + c] = sigmoid ? sigmoidf_acc(acc[i][j]) : acc[i][j];
    }
  }
}

// g_pre[b][c] = g_scores[b][c] * act'(scores[b][c])  (written by the CTAs of the first column tile);
// g_u[b][k] = rp[b][k] > 0 ? sum_c g_pre[b][c] Wp2[c][k] : 0
__global__ void __launch_bounds__(kThreads) ft_out_bwd_kernel(const float* __restrict__ rp, const float* __restrict__ Wp2,
                                                              const float* __restrict__ scores, const float* __restrict__ g_scores,
                                                              int B, int C, int H, int sigmoid, float* __restrict__ g_pre,
                                                              float* __restrict__ g_u) {
  constexpr int RI = 2;
  __shared__ float sg[OK][RI * 16 + 1], sw[OK][OT + 1];     // [c][graph], [c][k]
  const int g0 = blockIdx.y * RI * 16, k0 = blockIdx.x * OT;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const bool write_pre = blockIdx.x == 0;
  float acc[RI][4];
#pragma unroll
  for (int i = 0; i < RI; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int cb = 0; cb < C; cb += OK) {
    __syncthreads();
    for (int e = threadIdx.x; e < RI * 16 * OK; e += kThreads) {
      const int r = e / OK, c = e % OK;
      const int g = g0 + r, cc = cb + c;
      float v = 0.f;
      if (g < B && cc < C) {
        v = __ldg(g_scores + (size_t)g * C + cc);
        if (sigmoid) { const float sc = __ldg(scores + (size_t)g * C + cc); v *= sc * (1.f - sc); }
        if (write_pre) g_pre[(size_t)g * C + cc] = v;
      }
      sg[c][r] = v;
    }
    for (int e = threadIdx.x; e < OK * OT; e += kThreads) {
      const int c = e / OT, k = e % OT;
      sw[c][k] = (cb + c < C && k0 + k < H) ? __ldg(Wp2 + (size_t)(cb + c) * H + k0 + k) : 0.f;
    }
    __syncthreads();
    const int nc = min(OK, C - cb);
    for (int c = 0; c < nc; ++c) {
      float a[RI], w[4];
#pragma unroll
      for (int i = 0; i < RI; ++i) a[i] = sg[c][ty + 16 * i];
#pragma unroll
      for (int j = 0; j < 4; ++j) w[j] = sw[c][tx + 16 * j];
#pragma unroll
      for (int i = 0; i < RI; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(w[j], a[i], acc[i][j]);
    }
  }
#pragma unroll
  for (int i = 0; i < RI; ++i) {
    const int g = g0 + ty + 16 * i;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + tx + 16 * j;
      if (g < B && k < H) g_u[(size_t)g * H + k] = __ldg(rp + (size_t)g * H + k) > 0.f ? acc[i][j] : 0.f;
    }
  }
}

// part[z][m][n] = sum over the rows of split z of A[r][m] * Bm[r][n]   (32x32 output tile per CTA, blockIdx.z = row split;
// Bm == nullptr: Bm is a column of ones (column sums of A, Nn = 1)).  atb_reduce_kernel adds the splits in order:
// out[m][n] = sum_z part[z][m][n] - a fixed order, no float atomics.
__global__ void __launch_bounds__(kThreads) atb_partial_kernel(const float* __restrict__ A, int lda, const float* __restrict__ Bm,
                                                               int ldb, float* __restrict__ part, int R, int M, int Nn,
                                                               int rows_per_split) {
  __shared__ float sa[32][33], sb[32][33];
  const int m0 = blockIdx.x * 32, n0 = blockIdx.y * 32;
  const int rbeg = blockIdx.z * rows_per_split, rend = min(R, rbeg + rows_per_split);
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;     // ty in 0..7 -> 4 output rows each
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int r0 = rbeg; r0 < rend; r0 += 32) {
    for (int i = threadIdx.x; i < 32 * 32; i += kThreads) {
      const int rr = i >> 5, cc = i & 31;
      const int r = r0 + rr;
      sa[rr][cc] = (r < rend && m0 + cc < M) ? A[(size_t)r * lda + m0 + cc] : 0.f;
      sb[rr][cc] = (r < rend && n0 + cc < Nn) ? (Bm ? Bm[(size_t)r * ldb + n0 + cc] : 1.f) : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int rr = 0; rr < 32; ++rr) {
      const float bv = sb[rr][tx];
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[i] = fmaf(sa[rr][ty * 4 + i], bv, acc[i]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i, n = n0 + tx;
    if (m < M && n < Nn) part[((size_t)blockIdx.z * M + m) * Nn + n] = acc[i];
  }
}

__global__ void __launch_bounds__(kThreads) atb_reduce_kernel(const float* __restrict__ part, int S, int M, int Nn,
                                                              float* __restrict__ out, int ldo, float* __restrict__ out2) {
  const int i = blockIdx.x * kThreads + threadIdx.x;
  if (i >= M * Nn) return;
  float s = 0.f;
  for (int z = 0; z < S; ++z) s += part[(size_t)z * M * Nn + i];
  const int m = i / Nn, n = i % Nn;
  out[(size_t)m * ldo + n] = s;
  if (out2) out2[(size_t)m * ldo + n] = s;
}

}  // namespace

void launch_finetune_head_fwd(const FinetuneHeadFwdArgs& a, cudaStream_t s) {
  const int grid = (a.B + FG - 1) / FG;
  if (a.H == 32) finetune_head_fwd_kernel<32><<<grid, kThreads, 0, s>>>(a);
  else if (a.H == 64) finetune_head_fwd_kernel<64><<<grid, kThreads, 0, s>>>(a);
  else finetune_head_fwd_kernel<128><<<grid, kThreads, 0, s>>>(a);
  if (a.C > kMaxC)
    ft_out_fwd_kernel<<<dim3((a.C + OT - 1) / OT, (a.B + 63) / 64), kThreads, 0, s>>>(a.rp, a.Wp2, a.bp2, a.B, a.C, a.H, a.sigmoid, a.scores);
}

void launch_finetune_head_bwd(const FinetuneHeadBwdArgs& a, cudaStream_t s) {
  const int grid = (a.B + FG - 1) / FG;
  if (a.C > kMaxC)
    ft_out_bwd_kernel<<<dim3((a.H + OT - 1) / OT, (a.B + 31) / 32), kThreads, 0, s>>>(a.rp, a.Wp2, a.scores, a.g_scores, a.B, a.C, a.H,
                                                                                   a.sigmoid, a.g_pre, a.g_u);
  if (a.H == 32) finetune_head_bwd_kernel<32><<<grid, kThreads, 0, s>>>(a);
  else if (a.H == 64) finetune_head_bwd_kernel<64><<<grid, kThreads, 0, s>>>(a);
  else finetune_head_bwd_kernel<128><<<grid, kThreads, 0, s>>>(a);
}

int atb_splits(int R) { const int sp = (R + 127) / 128; return sp < 1 ? 1 : (sp > 64 ? 64 : sp); }

// out[m][n] = sum_r A[r][m] * Bm[r][n] (Bm == nullptr: column sums of A, Nn = 1); scratch >= atb_splits(R) * M * Nn floats
void launch_atb(const float* A, int lda, const float* Bm, int ldb, float* out, int ldo, float* out2, int R, int M, int Nn,
                float* scratch, cudaStream_t s) {
  const int S = atb_splits(R);
  const int rows_per_split = ((R + S - 1) / S + 31) / 32 * 32;
  dim3 grid((M + 31) / 32, (Nn + 31) / 32, S);
  atb_partial_kernel<<<grid, kThreads, 0, s>>>(A, lda, Bm, ldb, scratch, R, M, Nn, rows_per_split);
  atb_reduce_kernel<<<(M * Nn + kThreads - 1) / kThreads, kThreads, 0, s>>>(scratch, S, M, Nn, out, ldo, out2);
}

int finetune_max_classes() { return kMaxClasses; }

}  // namespace scgib
