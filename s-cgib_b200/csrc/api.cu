// api.cu - the extern "C" surface of libscgib.so (include/scgib.h): parameter layout, workspace carving and the
// launch sequences of the whole pre-training forward / backward.  No device memory is allocated here.
#include <stdio.h>
#include <string.h>
#include <stdlib.h>
#include "kernels.cuh"
#include "../../include/scgib.h"
#include "scgib_private.h"

namespace scgib {

int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = 148;
  }
  return n;
}

// SCGIB_TC / SCGIB_TC_BWD: 1 (default) = the tcgen05 kernels (gin_tc3.cu / gin_bwd_tc2.cu), 0 = the FP32 FFMA
// register-tile kernels of gin_kernels.cu (the cross-check implementation)
static int g_use_tc = -1;
int tensor_core_mode() {
  if (g_use_tc < 0) { const char* e = getenv("SCGIB_TC"); g_use_tc = (e && e[0] == '0') ? 0 : 1; }
  return g_use_tc;
}
static int g_bwd_tc = -1;
int bwd_tensor_core_mode() {
  if (g_bwd_tc < 0) { const char* e = getenv("SCGIB_TC_BWD"); g_bwd_tc = (e && e[0] == '0') ? 0 : 1; }
  return g_bwd_tc;
}
// SCGIB_RECON_SIDE=1: the adjacency-reconstruction backward as side CTAs of the contrastive backward launch (measured: the
// 20 SMs that launch leaves idle need longer for it than the separate 29 us launch on all SMs; default off)
static bool recon_side_mode() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("SCGIB_RECON_SIDE"); v = (e && e[0] == '1') ? 1 : 0; }
  return v == 1;
}
// CTAs of recon_fwd (= its per-CTA partial Gram matrices): two resident CTAs per SM at hidden 64 overlap the copy / Gram / gather phases
static int recon_fwd_grid() { return 2 * num_sms(); }
static int g_bwd_h = -1;
int bwd_h_mode() {
  if (g_bwd_h < 0) { const char* e = getenv("SCGIB_BWD_H"); g_bwd_h = (e && e[0] == '0') ? 0 : 1; }
  return g_bwd_h;
}
static int g_fwd4 = -1;
int fwd_tc4_mode() {
  if (g_fwd4 < 0) { const char* e = getenv("SCGIB_FWD4"); g_fwd4 = (e && e[0] == '1') ? 1 : 0; }
  return g_fwd4;
}
static void launch_gin_fwd_any(const GinFwdArgs& a, int kin, cudaStream_t s) {      // op-level entry: hidden 64
  if (tensor_core_mode() == 0) launch_gin_fwd(a, kin, HID, s);
  else if (kin == HID && !a.row_map && fwd_tc4_mode()) launch_gin_fwd_tc4(a, s);
  else launch_gin_fwd_tc3(a, kin, s);
}

// contrastive similarity blocks on tcgen05 (default on; SCGIB_CON_FFMA=1 selects the FFMA tiles)
static int g_con_tc = -1;
static bool use_tc_contrastive() {
  if (g_con_tc < 0) { const char* e = getenv("SCGIB_CON_FFMA"); g_con_tc = (e && e[0] == '1') ? 0 : 1; }
  return g_con_tc == 1;
}

// layers alternate the direction in which they walk the row tiles (SCGIB_FWD_ALT=0 disables): layer l+1 starts with the
// rows layer l wrote last, which are still in L2
static bool fwd_alternate() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("SCGIB_FWD_ALT"); v = (e && e[0] == '0') ? 0 : 1; }
  return v == 1;
}

bool pdl_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("SCGIB_PDL"); v = (e && e[0] == '0') ? 0 : 1; }
  return v == 1;
}

static inline size_t al(size_t x) { return (x + 255) / 256 * 256; }

// Optional per-launch timing with CUDA events on the launching stream (bench.py's roofline numbers).
struct Prof {
  bool on = false;
  int n = 0;
  static constexpr int kMax = 512;
  cudaEvent_t ev[2 * kMax];
  int made = 0;
  const char* name[kMax];
};
static Prof g_prof;
static inline void prof_begin(const char* name, cudaStream_t s) {
  if (!g_prof.on || g_prof.n >= Prof::kMax) return;
  while (g_prof.made < 2 * (g_prof.n + 1)) cudaEventCreate(&g_prof.ev[g_prof.made++]);
  g_prof.name[g_prof.n] = name;
  cudaEventRecord(g_prof.ev[2 * g_prof.n], s);
}
static inline void prof_end(cudaStream_t s) {
  if (!g_prof.on || g_prof.n >= Prof::kMax) return;
  cudaEventRecord(g_prof.ev[2 * g_prof.n + 1], s);
  ++g_prof.n;
}
// SCGIB_DEBUG_SYNC=1: synchronise after every launch and report the first failing kernel by name.
static inline bool debug_sync() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("SCGIB_DEBUG_SYNC"); v = (e && e[0] == '1') ? 1 : 0; }
  return v == 1;
}
static inline void debug_check(const char* name, cudaStream_t s) {
  if (!debug_sync()) return;
  cudaError_t e = cudaStreamSynchronize(s);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) { fprintf(stderr, "[scgib] kernel '%s' failed: %s\n", name, cudaGetErrorString(e)); fflush(stderr); }
}
#define PROF(name, stmt) do { prof_begin(name, s); stmt; prof_end(s); debug_check(name, s); } while (0)

static bool dims_ok(const ScgibDims* d) {
  return d && (d->hidden == 64 || d->hidden == 128) && d->d_transfer == DTR && d->gin_layers >= 1 && d->gin_layers <= 8 && d->in_dim >= 1 &&
         d->in_dim <= 32 && (d->act_dtype == SCGIB_ACT_F32 || d->act_dtype == SCGIB_ACT_BF16);
}

struct Layout {
  int64_t off[SCGIB_P_ENC + 2 * 8 * SCGIB_ENC_SLOTS];
  int64_t size[SCGIB_P_ENC + 2 * 8 * SCGIB_ENC_SLOTS];
  int n;
  int64_t total;
  int64_t enc(int e, int l, int L, int slot) const { return off[SCGIB_P_ENC + (e * L + l) * SCGIB_ENC_SLOTS + slot]; }
};

static Layout make_layout(const ScgibDims* d) {
  Layout lo;
  const int L = d->gin_layers, HID = d->hidden;
  int64_t sizes[SCGIB_P_ENC] = {
      (int64_t)HID * 2 * HID, HID, (int64_t)HID * HID, HID,      // head
      (int64_t)HID * HID, HID, HID, HID, HID, 1,                  // compressor
      2 * HID, 1,                                                 // attention
      (int64_t)DTR * d->in_dim};                                  // transfer_d
  int n = 0;
  int64_t o = 0;
  auto push = [&](int64_t s) { lo.off[n] = o; lo.size[n] = s; o += (s + 3) / 4 * 4; ++n; };
  for (int i = 0; i < SCGIB_P_ENC; ++i) push(sizes[i]);
  for (int e = 0; e < 2; ++e)
    for (int l = 0; l < L; ++l) {
      const int kin = (l == 0) ? DTR : HID;
      push((int64_t)HID * kin); push(HID); push((int64_t)HID * HID); push(HID); push(HID); push(HID);
    }
  lo.n = n;
  lo.total = o;
  return lo;
}

// ---------------------------------------------------------------- workspace
struct Ws {
  // transposed weights
  float *enc_w1t[2][8], *enc_w2t[2][8], *head_w1t, *head_w2t, *comp_w1t;
  float* t;
  float *a[2][8], *r[2][8], *y[2][8];
  float* bn[2][8];      // {mean, rstd, gamma, beta}
  float* cvec[2];
  float* small_part;    // BN partials (fwd) / dgamma,dbeta partials (bwd) / gate partials / input-proj partials
  float* small_part2;   // the same for Encoder2 when both encoders share a launch
  unsigned int* counters;
  float *H, *q, *C, *logit, *alpha, *lam, *noisy, *Z, *r_head, *readout, *core, *gstat, *cstat, *kl;
  float *rpart, *G, *edge;
  float *z1, *z2, *n1, *n2, *diag, *D, *rowsum, *g1p, *g2p, *g_core, *g_readout, *zsplit;
  float *gZ, *gI, *gp, *g_q, *gH, *gC, *g_o[2], *Ga[2], *ga0[2];
  float* xagg[2];       // aggregated normalised features of the parent / ego rows, [V][xagg_stride] (transfer_d backward)
  float *logm_walks, *logm_gram, *logm_pair, *logm_loss;     // --recons_type logM (logm_kernels.cu)
  float *aC, *head_w1a, *head_w1b, *head_bn, *head_cvec;     // tensor-core head backward (the GIN backward kernel on two K halves)
  bf16_t *noisy_bf, *aC_bf, *r_head_bf, *gZ_bf;              // bf16 mode: its operands in bf16 (the bf16 GIN backward kernel)
  float* ppart;
  size_t bytes;
};

static inline int xagg_stride(const ScgibDims* d) { return (d->in_dim + 3) / 4 * 4; }

static size_t small_part_floats(int N, int Ns, int HID) {
  const int Vmax = N > Ns ? N : Ns;
  size_t a = (size_t)((Vmax + 63) / 64) * 2 * HID;                   // gin fwd tile partials (64-row tiles)
  const size_t a2 = (size_t)num_sms() * 3 * HID * 2;                  // gin_tc2: per-CTA (n, mean, M2) in fp64
  a = a > a2 ? a : a2;
  size_t b = (size_t)(gin_bwd_pre_grid(N + Ns) + 2) * 2 * HID;       // dgamma/dbeta partials (per problem of a shared launch)
  size_t c = (size_t)4 * num_sms() * 5 * HID;                        // gate partials
  size_t d = (size_t)input_proj_bwd_grid(N, Ns) * DTR * 32;          // transfer_d partials
  size_t m = a > b ? a : b;
  m = m > c ? m : c;
  return m > d ? m : d;
}

static Ws carve(const ScgibDims* d, const Layout& lo, int B, int N, int E, int Ns, int Es, void* base) {
  Ws w;
  char* p = (char*)base;
  size_t o = 0;
  auto take = [&](size_t nfloats) { float* r = (float*)(p + o); o += al(nfloats * sizeof(float)); return r; };
  // activations of the GIN encoders (t, a, r, y, the layer gradients g_o / Ga): fp32, or bf16 in bf16 mode - carved by bytes
  const size_t es = d->act_dtype == SCGIB_ACT_BF16 ? 2 : 4;
  auto take_act = [&](size_t nelems) { float* r = (float*)(p + o); o += al(nelems * es); return r; };
  const int L = d->gin_layers, HID = d->hidden;
  const int V[2] = {N, Ns};
  const int Vmax = N > Ns ? N : Ns;
  for (int e = 0; e < 2; ++e)
    for (int l = 0; l < L; ++l) {
      const int kin = l == 0 ? DTR : HID;
      w.enc_w1t[e][l] = take((size_t)kin * HID);
      w.enc_w2t[e][l] = take((size_t)HID * HID);
      w.a[e][l] = take_act((size_t)V[e] * kin);
      w.r[e][l] = take_act((size_t)V[e] * HID);
      w.y[e][l] = take_act((size_t)V[e] * HID);
      w.bn[e][l] = take(4 * HID);
    }
  w.head_w1t = take(2 * HID * HID); w.head_w2t = take(HID * HID); w.comp_w1t = take(HID * HID);
  w.t = take_act((size_t)N * DTR);
  w.cvec[0] = take(2 * HID); w.cvec[1] = take(2 * HID);
  w.small_part = take(small_part_floats(N, Ns, HID)); w.small_part2 = take(small_part_floats(N, Ns, HID));
  w.counters = (unsigned int*)take(64);
  w.H = take((size_t)N * HID); w.q = take((size_t)N * HID); w.C = take((size_t)N * HID);
  w.logit = take(N); w.alpha = take(N); w.lam = take(N);
  w.noisy = take((size_t)N * HID); w.Z = take((size_t)N * HID); w.r_head = take((size_t)N * HID);
  w.readout = take((size_t)B * HID); w.core = take((size_t)B * HID);
  w.gstat = take((size_t)B * 4 * HID); w.cstat = take((size_t)B * 2 * HID); w.kl = take(4);
  w.rpart = take((size_t)recon_fwd_grid() * (HID * HID + 4)); w.G = take(HID * HID); w.edge = take(4);
  const int js = contrastive_jsplit(B);
  w.z1 = take((size_t)B * HID); w.z2 = take((size_t)B * HID); w.zsplit = take((size_t)4 * B * HID);
  w.n1 = take(B); w.n2 = take(B); w.diag = take(B); w.D = take(B);
  w.rowsum = take((size_t)js * B);
  w.g1p = take((size_t)js * B * HID); w.g2p = take((size_t)js * B * HID);
  w.g_core = take((size_t)B * HID); w.g_readout = take((size_t)B * HID);
  w.gZ = take((size_t)N * HID); w.gI = take((size_t)N * 2 * HID); w.gp = take(N);
  w.g_q = take((size_t)N * HID); w.gH = take((size_t)N * HID); w.gC = take((size_t)N * HID);
  w.g_o[0] = take_act((size_t)N * HID); w.g_o[1] = take_act((size_t)Ns * HID);
  w.Ga[0] = take_act((size_t)N * HID); w.Ga[1] = take_act((size_t)Ns * HID);
  (void)Vmax;
  w.ga0[0] = take((size_t)N * DTR); w.ga0[1] = take((size_t)Ns * DTR);
  w.xagg[0] = take((size_t)N * xagg_stride(d)); w.xagg[1] = take((size_t)Ns * xagg_stride(d));
  w.logm_walks = take((size_t)logm_max_steps() * N); w.logm_gram = take(B); w.logm_pair = take(N); w.logm_loss = take(4);
  w.aC = take((size_t)N * HID); w.head_w1a = take(HID * HID); w.head_w1b = take(HID * HID);
  w.head_bn = take(4 * HID); w.head_cvec = take(2 * HID);
  if (d->act_dtype == SCGIB_ACT_BF16) {
    w.noisy_bf = (bf16_t*)take_act((size_t)N * HID); w.aC_bf = (bf16_t*)take_act((size_t)N * HID);
    w.r_head_bf = (bf16_t*)take_act((size_t)N * HID); w.gZ_bf = (bf16_t*)take_act((size_t)N * HID);
  } else {
    w.noisy_bf = w.aC_bf = w.r_head_bf = w.gZ_bf = nullptr;
  }
  w.ppart = take((size_t)num_sms() * lo.total);
  w.bytes = o;
  (void)E; (void)Es;
  return w;
}

static int check_batch(const ScgibBatch* b) {
  if (!b) return SCGIB_E_NULL;
  if (b->struct_size != (int32_t)sizeof(ScgibBatch)) return SCGIB_E_ABI;
  if (b->B < 1 || b->N < 2 || b->Ns < b->N || b->E < 0 || b->Es < 0) return SCGIB_E_RANGE;
  if (!b->graph_ptr || !b->indptr || !b->ego_ptr || !b->ego_nodes || !b->ego_seed || !b->sub_indptr ||
      (!b->x && !b->t_override) || !b->gate_u || !b->feat_u)
    return SCGIB_E_NULL;
  if ((b->E > 0 && !b->indices) || (b->Es > 0 && !b->sub_indices)) return SCGIB_E_NULL;
  if (((uintptr_t)b->feat_u & 15u) != 0) return SCGIB_E_ALIGN;
  if (b->recon_logm_steps < 0 || b->recon_logm_steps > logm_max_steps()) return SCGIB_E_RANGE;
  return SCGIB_OK;
}

}  // namespace scgib

using namespace scgib;

extern "C" SCGIB_API int scgib_version(void) { return SCGIB_VERSION; }

extern "C" SCGIB_API const char* scgib_error_string(int code) {
  switch (code) {
    case SCGIB_OK: return "ok";
    case SCGIB_E_NULL: return "required pointer is NULL";
    case SCGIB_E_SHAPE: return "unsupported dimensions (hidden must be 64 or 128, d_transfer 32, 1 <= gin_layers <= 8, in_dim <= 32; --recons_type logM and the op-level entries: hidden 64)";
    case SCGIB_E_ALIGN: return "pointer not 16-byte aligned";
    case SCGIB_E_WORKSPACE: return "workspace too small";
    case SCGIB_E_RANGE: return "size out of range";
    case SCGIB_E_ABI: return "ScgibBatch.struct_size does not match this library (binding built against another scgib.h)";
    default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown scgib error";
  }
}

extern "C" SCGIB_API int scgib_num_sms(void) { return num_sms(); }
extern "C" SCGIB_API int32_t scgib_batch_abi_size(void) { return (int32_t)sizeof(ScgibBatch); }

extern "C" SCGIB_API int32_t scgib_param_slots(const ScgibDims* d) {
  if (!dims_ok(d)) return SCGIB_E_SHAPE;
  return SCGIB_P_ENC + 2 * d->gin_layers * SCGIB_ENC_SLOTS;
}

extern "C" SCGIB_API int64_t scgib_param_layout(const ScgibDims* d, int64_t* offsets, int64_t* sizes) {
  if (!dims_ok(d)) return SCGIB_E_SHAPE;
  const Layout lo = make_layout(d);
  for (int i = 0; i < lo.n; ++i) {
    if (offsets) offsets[i] = lo.off[i];
    if (sizes) sizes[i] = lo.size[i];
  }
  return lo.total;
}

extern "C" SCGIB_API size_t scgib_pretrain_workspace_bytes(const ScgibDims* d, int32_t B, int32_t N, int32_t E, int32_t Ns, int32_t Es) {
  if (!dims_ok(d)) return 0;
  const Layout lo = make_layout(d);
  return carve(d, lo, B, N, E, Ns, Es, nullptr).bytes;
}

// features_only: stop after the head MLP (Z); the pre-training losses are not evaluated (fine-tuning forward)
static int forward_impl(const ScgibDims* d, const float* params, float* bn_running, const ScgibBatch* b, float* losses,
                        float* interaction_map, float* Z, float* noisy, float* graph_readout, void* workspace,
                        size_t workspace_bytes, void* stream_, bool features_only) {
  if (!dims_ok(d)) return SCGIB_E_SHAPE;
  if (!params || (!losses && !features_only) || !workspace) return SCGIB_E_NULL;
  int rc = check_batch(b);
  if (rc) return rc;
  if (((uintptr_t)workspace & 255u) != 0 || ((uintptr_t)params & 15u) != 0) return SCGIB_E_ALIGN;
  const Layout lo = make_layout(d);
  const Ws w = carve(d, lo, b->B, b->N, b->E, b->Ns, b->Es, workspace);
  if (workspace_bytes < w.bytes) return SCGIB_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream_;
  const int L = d->gin_layers, HID = d->hidden;
  const bool eval = b->eval_mode != 0;       // model.eval(): BatchNorm layers use (and do not update) their running statistics
  if (eval && !bn_running) return SCGIB_E_NULL;
  const bool bf = d->act_dtype == SCGIB_ACT_BF16;   // bf16 mode: GIN activations in bf16, single-pass bf16 tensor-core MLPs
  const bool tc64 = HID == 64;                      // the 3xTF32 tcgen05 kernels (fp32 data) exist for hidden = 64; 128: FFMA tiles
  if (b->recon_logm_steps > 0 && HID != 64 && !features_only) return SCGIB_E_SHAPE;   // --recons_type logM: hidden 64 only

  cudaMemsetAsync(w.counters, 0, 64 * sizeof(float), s);
  // Parameter-only prologue, ONE launch: k-major weight copies for the FFMA forward GEMMs (the tensor-core GIN kernels read
  // the natural layout: their copies are skipped), the head backward's operands (W1 halves, identity BN constants: the
  // backward pass of the same step finds them in the workspace) and the input projection.
  {
    FwdPrepArgs pa;
    TransposeJobs& jobs = pa.jobs;
    jobs.n = 0;
    auto add = [&](const float* src, float* dst, int rows, int cols) { jobs.job[jobs.n++] = TransposeJob{src, dst, rows, cols}; };
    const bool enc_ffma = !bf && !(tc64 && tensor_core_mode() != 0);
    if (enc_ffma)
      for (int e = 0; e < 2; ++e)
        for (int l = 0; l < L; ++l) {
          add(params + lo.enc(e, l, L, SCGIB_ENC_W1), w.enc_w1t[e][l], HID, l == 0 ? DTR : HID);
          add(params + lo.enc(e, l, L, SCGIB_ENC_W2), w.enc_w2t[e][l], HID, HID);
          if (jobs.n >= 20) { launch_transposes(jobs, s); jobs.n = 0; }
        }
    add(params + lo.off[SCGIB_P_HEAD_W1], w.head_w1t, HID, 2 * HID);
    add(params + lo.off[SCGIB_P_HEAD_W2], w.head_w2t, HID, HID);
    add(params + lo.off[SCGIB_P_COMP_W1], w.comp_w1t, HID, HID);
    pa.headW1 = params + lo.off[SCGIB_P_HEAD_W1]; pa.W1a = w.head_w1a; pa.W1b = w.head_w1b; pa.bn = w.head_bn; pa.cvec = w.head_cvec;
    pa.hid = HID;
    if (b->t_override && bf)
      launch_f32_to_bf16(b->t_override, w.t, (size_t)b->N * DTR, s);
    else if (b->t_override)
      cudaMemcpyAsync(w.t, b->t_override, (size_t)b->N * DTR * sizeof(float), cudaMemcpyDeviceToDevice, s);
    else {
      pa.x = b->x; pa.Wt = params + lo.off[SCGIB_P_TRANSFER]; pa.N = b->N; pa.F = d->in_dim; pa.normalize = b->normalize_x; pa.t = w.t;
      if (!eval) {      // the backward pass of this step contracts the layer-0 input gradients with the aggregated features
        pa.xa_indptr[0] = b->indptr; pa.xa_indptr[1] = b->sub_indptr; pa.xa_indices[0] = b->indices; pa.xa_indices[1] = b->sub_indices;
        pa.xa_x = b->x; pa.xa_map = b->ego_nodes; pa.xa_V[0] = b->N; pa.xa_V[1] = b->Ns;
        pa.xagg[0] = w.xagg[0]; pa.xagg[1] = w.xagg[1]; pa.xa_stride = xagg_stride(d);
      }
    }
    PROF("fwd_prep", launch_fwd_prep(pa, s, bf));
  }
  // the two GIN encoders (models.py:704, 707): layer l of Encoder1 and of Encoder2 are independent, so they share a launch
  for (int l = 0; l < L; ++l) {
    GinFwdArgs ga[2];
    for (int e = 0; e < 2; ++e) {
      GinFwdArgs& a = ga[e];
      a.in = l == 0 ? w.t : w.y[e][l - 1];
      a.row_map = (e == 1 && l == 0) ? b->ego_nodes : nullptr;
      a.bn_in = l == 0 ? nullptr : w.bn[e][l - 1];
      a.indptr = e == 0 ? b->indptr : b->sub_indptr;
      a.indices = e == 0 ? b->indices : b->sub_indices;
      a.V = e == 0 ? b->N : b->Ns;
      a.W1t = w.enc_w1t[e][l]; a.b1 = params + lo.enc(e, l, L, SCGIB_ENC_B1);
      a.W2t = w.enc_w2t[e][l]; a.b2 = params + lo.enc(e, l, L, SCGIB_ENC_B2);
      a.W1 = params + lo.enc(e, l, L, SCGIB_ENC_W1); a.W2 = params + lo.enc(e, l, L, SCGIB_ENC_W2);
      a.gamma = params + lo.enc(e, l, L, SCGIB_ENC_GAMMA); a.beta = params + lo.enc(e, l, L, SCGIB_ENC_BETA);
      a.a_out = w.a[e][l]; a.r_out = w.r[e][l]; a.y_out = w.y[e][l];
      a.part = e == 0 ? w.small_part : w.small_part2; a.counter = w.counters + (e == 0 ? 0 : 8);
      a.bn_out = w.bn[e][l];
      a.running = (bn_running && !eval) ? bn_running + (size_t)(e * L + l) * 2 * HID : nullptr;
      a.reverse = (l & 1) && fwd_alternate();
    }
    const int kin = l == 0 ? DTR : HID;
    if (bf) {
      PROF("gin_fwd_bf16.enc1+2", launch_gin_fwd_bf16(ga[0], &ga[1], kin, HID, s));
    } else if (tc64 && tensor_core_mode() != 0) {
      if (kin == HID && fwd_tc4_mode()) PROF("gin_fwd_tc4.enc1+2", launch_gin_fwd_tc4_pair(ga[0], ga[1], s));
      else PROF("gin_fwd_tc.enc1+2", launch_gin_fwd_tc3_pair(ga[0], ga[1], kin, s));
    } else {
      for (int e = 0; e < 2; ++e) PROF(e == 0 ? "gin_fwd_ffma.enc1" : "gin_fwd_ffma.enc2", launch_gin_fwd(ga[e], kin, HID, s));
    }
    if (eval)
      for (int e = 0; e < 2; ++e)
        launch_bn_from_running(bn_running + (size_t)(e * L + l) * 2 * HID, params + lo.enc(e, l, L, SCGIB_ENC_GAMMA),
                               params + lo.enc(e, l, L, SCGIB_ENC_BETA), w.bn[e][l], HID, s);
  }
  // forward tail on the tcgen05 contrastive launch: recon_reduce + compressor_ema as side CTAs, loss_finalize by its last CTA
  const bool fuse_tail = !features_only && tc64 && use_tc_contrastive();
  {
    GateLinFwdArgs a{w.y[0][L - 1], w.bn[0][L - 1], b->N, w.comp_w1t, params + lo.off[SCGIB_P_COMP_B1], w.H, w.q, bf};
    a.Wc1n = params + lo.off[SCGIB_P_COMP_W1];
    PROF("gate_lin_fwd", launch_gate_lin_fwd(a, HID, s));
  }
  {
    EgoPoolFwdArgs a{w.y[1][L - 1], w.bn[1][L - 1], b->ego_ptr, b->N, params + lo.off[SCGIB_P_ATTN_W] + HID, w.C, w.logit, bf};
    PROF("ego_pool_fwd", launch_ego_pool_fwd(a, HID, s));
  }
  {
    GraphGateFwdArgs a;
    a.graph_ptr = b->graph_ptr; a.B = b->B; a.N = b->N; a.H = w.H; a.q = w.q;
    a.gamma_c = params + lo.off[SCGIB_P_COMP_GAMMA]; a.beta_c = params + lo.off[SCGIB_P_COMP_BETA];
    a.wc2 = params + lo.off[SCGIB_P_COMP_W2]; a.bc2 = params + lo.off[SCGIB_P_COMP_B2];
    a.gate_u = b->gate_u; a.feat_u = b->feat_u; a.logit = w.logit;
    a.noisy = w.noisy; a.lam = w.lam; a.alpha = w.alpha; a.readout = w.readout; a.core = w.core;
    a.gstat = w.gstat; a.cstat = (bn_running && !eval) ? w.cstat : nullptr; a.kl = w.kl;
    a.eval_running = eval ? bn_running + (size_t)2 * L * 2 * HID : nullptr;
    a.noisy_bf = w.noisy_bf;
    if (!features_only) {      // the contrastive loss' row normalisation rides in the per-graph warps
      a.z1 = w.z1; a.z2 = w.z2; a.n1 = w.n1; a.n2 = w.n2; a.diag = w.diag; a.zsplit = tc64 ? w.zsplit : nullptr;
    }
    PROF("graph_gate_fwd", launch_graph_gate_fwd(a, HID, s));
    if (bn_running && !eval && !fuse_tail)
      PROF("compressor_ema", launch_compressor_ema(w.cstat, b->B, bn_running + (size_t)2 * L * 2 * HID, HID, s));
  }
  {
    HeadFwdArgs a{w.noisy, w.C, w.alpha, b->N, w.head_w1t, params + lo.off[SCGIB_P_HEAD_B1], w.head_w2t,
                  params + lo.off[SCGIB_P_HEAD_B2], interaction_map, bf ? nullptr : w.aC, bf ? nullptr : w.r_head, w.Z,
                  w.r_head_bf, w.aC_bf};       // bf16 mode: the backward's operands are kept in bf16 only
    a.W1n = params + lo.off[SCGIB_P_HEAD_W1]; a.W2n = params + lo.off[SCGIB_P_HEAD_W2];
    PROF("head_fwd", launch_head_fwd(a, HID, s));
  }
  const int logm = b->recon_logm_steps;
  if (!features_only && logm > 0) {
    PROF("logm_fwd", launch_logm_fwd(w.Z, b->graph_ptr, b->indptr, b->indices, b->B, b->N, logm, w.logm_walks, w.logm_gram,
                                     w.logm_pair, w.logm_loss, (int32_t*)(w.counters + 32), HID, s));
  } else if (!features_only) {
    const int grid = recon_fwd_grid();
    ReconFwdArgs a{w.Z, b->indptr, b->indices, b->N, w.rpart};
    PROF("recon_fwd", launch_recon_fwd(a, HID, grid, s));
    if (!fuse_tail) PROF("recon_reduce", launch_recon_reduce(w.rpart, grid, w.G, w.edge, HID, s));
  }
  const int js = contrastive_jsplit(b->B);
  if (!features_only) {
    ContrastiveFwdArgs c{w.z1, w.z2, b->B, js, w.rowsum, w.zsplit};
    LossFinalizeArgs fin{w.rowsum, js, w.diag, b->B, w.G, w.edge, b->N, b->E, logm > 0 ? w.logm_loss : nullptr, w.kl, w.D, losses, HID};
    if (fuse_tail) {
      ConFwdSides sd;
      if (logm <= 0) { sd.rpart = w.rpart; sd.rgrid = recon_fwd_grid(); sd.G = w.G; sd.edge = w.edge; sd.n_reduce = 8; }
      if (bn_running && !eval) { sd.cstat = w.cstat; sd.running = bn_running + (size_t)2 * L * 2 * HID; sd.n_ema = 1; }
      sd.finalize = 1; sd.fin = fin; sd.counter = w.counters + 4;
      PROF("contrastive_fwd_tc", launch_contrastive_fwd_tc_sides(c, sd, s));
    } else {
      PROF("contrastive_fwd", launch_contrastive_fwd(c, HID, s));
      PROF("loss_finalize", launch_loss_finalize(fin, s));
    }
  }
  if (Z) cudaMemcpyAsync(Z, w.Z, (size_t)b->N * HID * sizeof(float), cudaMemcpyDeviceToDevice, s);
  if (noisy) cudaMemcpyAsync(noisy, w.noisy, (size_t)b->N * HID * sizeof(float), cudaMemcpyDeviceToDevice, s);
  if (graph_readout) cudaMemcpyAsync(graph_readout, w.readout, (size_t)b->B * HID * sizeof(float), cudaMemcpyDeviceToDevice, s);
  return (int)cudaGetLastError();
}

extern "C" SCGIB_API int scgib_pretrain_forward_f32(const ScgibDims* d, const float* params, float* bn_running,
                                          const ScgibBatch* b, float* losses, float* interaction_map, float* Z,
                                          float* noisy, float* graph_readout, void* workspace, size_t workspace_bytes,
                                          void* stream) {
  return forward_impl(d, params, bn_running, b, losses, interaction_map, Z, noisy, graph_readout, workspace,
                      workspace_bytes, stream, false);
}

extern "C" SCGIB_API int scgib_extract_forward_f32(const ScgibDims* d, const float* params, float* bn_running,
                                         const ScgibBatch* b, float* interaction_map, float* Z, float* noisy,
                                         float* graph_readout, void* workspace, size_t workspace_bytes, void* stream) {
  return forward_impl(d, params, bn_running, b, nullptr, interaction_map, Z, noisy, graph_readout, workspace,
                      workspace_bytes, stream, true);
}

// gZ_ext == nullptr: gradients of scale . {KL, contrastive, recon};  gZ_ext != nullptr: gradients of <gZ_ext, Z> (the
// upstream gradient of a head applied to Z = MLP(interaction_map): the fine-tuning models, models.py:501-520)
static int backward_impl(const ScgibDims* d, const float* params, const ScgibBatch* b, const float* loss_scale,
                         const float* gZ_ext, float* grads, void* workspace, size_t workspace_bytes, void* stream_) {
  if (!dims_ok(d)) return SCGIB_E_SHAPE;
  if (!params || !grads || !workspace || !loss_scale) return SCGIB_E_NULL;
  int rc = check_batch(b);
  if (rc) return rc;
  if (b->t_override) return SCGIB_E_NULL;   // forward-only mode: no gradient path to transfer_d
  if (b->eval_mode) return SCGIB_E_RANGE;   // the BatchNorm backward is the training-mode one (batch statistics)
  if (((uintptr_t)workspace & 255u) != 0 || ((uintptr_t)params & 15u) != 0 || ((uintptr_t)grads & 15u) != 0) return SCGIB_E_ALIGN;
  const Layout lo = make_layout(d);
  const Ws w = carve(d, lo, b->B, b->N, b->E, b->Ns, b->Es, workspace);
  if (workspace_bytes < w.bytes) return SCGIB_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream_;
  const int L = d->gin_layers, HID = d->hidden;
  const int GP = num_sms();
  const float s_kl = loss_scale[0], s_con = loss_scale[1], s_rec = loss_scale[2];
  const bool bf = d->act_dtype == SCGIB_ACT_BF16;
  const bool tc_bwd = HID == 64 && bwd_tensor_core_mode() != 0;    // 3xTF32 tcgen05 backward (fp32 data): hidden 64; else FFMA tiles
  if (b->recon_logm_steps > 0 && HID != 64 && !gZ_ext) return SCGIB_E_SHAPE;

  cudaMemsetAsync(w.counters, 0, 64 * sizeof(float), s);
  // gin_bwd_h.cu (two-term fp16 splits) normalises the gradients of a launch by a power of two derived from max |g_o|: the kernel
  // that produces g_o leaves it in one of these slots (zeroed above) with an order-independent atomicMax
  const bool use_h = tc_bwd && bwd_h_mode() != 0;
  unsigned int* gm_head = w.counters + 52;
  auto gm_layer = [&](int e, int l) { return w.counters + 40 + e * 6 + l; };
  const int js = contrastive_jsplit(b->B);
  if (gZ_ext) {
    if (((uintptr_t)gZ_ext & 15u) != 0) return SCGIB_E_ALIGN;
    cudaMemcpyAsync(w.gZ, gZ_ext, (size_t)b->N * HID * sizeof(float), cudaMemcpyDeviceToDevice, s);
    cudaMemsetAsync(w.g_core, 0, (size_t)b->B * HID * sizeof(float), s);
    cudaMemsetAsync(w.g_readout, 0, (size_t)b->B * HID * sizeof(float), s);
  } else {
    // contrastive backward; its normalisation backward (contrastive_bwd_finalize) is fused into graph_gate_bwd below.  On the
    // tcgen05 launch the adjacency-reconstruction backward rides along as side CTAs on the SMs the 128-row blocks leave idle.
    ContrastiveBwdArgs a{w.z1, w.z2, w.D, b->B, js, w.g1p, w.g2p};
    const bool con_tc = HID == 64 && use_tc_contrastive();
    const bool logm = b->recon_logm_steps > 0;
    ReconBwdArgs ra{w.Z, w.G, b->indptr, b->indices, b->N, s_rec, w.gZ};
    if (use_h && !logm) ra.gmax = gm_head;          // max |gZ| for the head backward's gradient normalisation (gin_bwd_h.cu)
    if (con_tc) {
      ConBwdSides sd;
      const bool recon_side = !logm && recon_side_mode();
      if (recon_side) { sd.recon = ra; sd.n_recon = max(1, num_sms() - ((b->B + 127) / 128) * js); }
      PROF("contrastive_bwd_tc", launch_contrastive_bwd_tc_sides(a, w.zsplit, sd, s));
      if (!logm && !recon_side) PROF("recon_bwd", launch_recon_bwd(ra, HID, s));
    } else {
      PROF("contrastive_bwd_ffma", launch_contrastive_bwd(a, HID, s));
    }
    if (logm) {
      PROF("logm_bwd", launch_logm_bwd(w.Z, b->graph_ptr, b->indptr, b->indices, b->B, b->N, b->recon_logm_steps, w.logm_walks,
                                       s_rec, w.gZ, (int32_t*)(w.counters + 32), HID, s));
    } else if (!con_tc) {
      PROF("recon_bwd", launch_recon_bwd(ra, HID, s));
    }
  }
  // head MLP backward: Z = W2 relu(W1a noisy + W1b (alpha C) + b1) + b2 is the GIN MLP with its first layer split over two
  // K = H inputs, so its backward is the GIN backward kernel run on both halves (problem 0: a = noisy, W1a -> gI[:, :H], dW1a,
  // dW2, db1, db2; problem 1: a = alpha C, W1b -> gI[:, H:], dW1b; its duplicate dW2 / bias partials are not reduced) with an
  // identity BatchNorm backward (g_y = gZ).  tcgen05 kernel: both problems in ONE launch (CTAs split); FFMA tiles: two launches.
  const bool head_pair = tc_bwd || bf;         // one shared launch (CTAs split between the two K halves)
  const int head_split = head_pair ? pair_split(GP, (b->N + 127) / 128, (b->N + 127) / 128) : GP;
  {
    // (W1a / W1b / head_bn / head_cvec were prepared by the forward pass of this step: fwd_prep)
    if (bf) PROF("head_gz_bf16", launch_f32_to_bf16(w.gZ, w.gZ_bf, (size_t)b->N * HID, s));
    if (use_h && (gZ_ext || b->recon_logm_steps > 0)) PROF("head_gz_absmax", launch_absmax(w.gZ, (size_t)b->N * HID, gm_head, s));
    GinBwdMainArgs m[2];
    for (int h = 0; h < 2; ++h) {
      m[h].g_o = w.gZ; m[h].y = w.Z; m[h].r = w.r_head; m[h].a = h == 0 ? w.noisy : w.aC;
      m[h].bn = w.head_bn; m[h].cvec = w.head_cvec;
      m[h].W1 = h == 0 ? w.head_w1a : w.head_w1b; m[h].W2 = params + lo.off[SCGIB_P_HEAD_W2];
      m[h].V = b->N; m[h].g_a = w.gI + (size_t)h * b->N * HID; m[h].part = w.ppart; m[h].pstride = lo.total;
      m[h].off_W1 = lo.off[SCGIB_P_HEAD_W1] + (int64_t)h * HID * HID; m[h].off_b1 = lo.off[SCGIB_P_HEAD_B1];
      m[h].off_W2 = lo.off[SCGIB_P_HEAD_W2]; m[h].off_b2 = lo.off[SCGIB_P_HEAD_B2];
      m[h].gmax = gm_head;
    }
    if (bf) {
      // bf16 mode: the bf16 GIN backward kernel (single-pass bf16 MMAs) on bf16 copies of gZ / r / noisy / alpha C; gI stays fp32.
      // Its weight staging precedes its PDL wait: W1a / W1b come from head_bwd_prep, TWO launches upstream (complete by then).
      for (int h = 0; h < 2; ++h) {
        m[h].g_o = (const float*)w.gZ_bf; m[h].y = (const float*)w.gZ_bf; m[h].r = (const float*)w.r_head_bf;
        m[h].a = (const float*)(h == 0 ? w.noisy_bf : w.aC_bf);
      }
      PROF("head_bwd_bf16", launch_gin_bwd_main_bf16(m[0], &m[1], HID, HID, GP, s, true));
    } else if (use_h) {
      PROF("head_bwd_h", launch_gin_bwd_main_h_pair(m[0], m[1], HID, GP, s));
    } else if (tc_bwd) {
      PROF("head_bwd_tc", launch_gin_bwd_main_tc2_pair(m[0], m[1], HID, GP, s));
    } else {
      PROF("head_bwd_ffma.a", launch_gin_bwd_main(m[0], HID, HID, GP, s));
      PROF("head_bwd_ffma.b", launch_gin_bwd_main(m[1], HID, HID, GP, s));   // rewrites the (identical) dW2 / bias partials of .a
    }
  }
  {
    GraphGateBwdArgs a;
    a.graph_ptr = b->graph_ptr; a.B = b->B; a.N = b->N; a.H = w.H; a.q = w.q; a.C = w.C;
    a.gamma_c = params + lo.off[SCGIB_P_COMP_GAMMA]; a.beta_c = params + lo.off[SCGIB_P_COMP_BETA];
    a.wc2 = params + lo.off[SCGIB_P_COMP_W2]; a.w_cand = params + lo.off[SCGIB_P_ATTN_W] + HID;
    a.feat_u = b->feat_u; a.lam = w.lam; a.alpha = w.alpha; a.gstat = w.gstat;
    a.gI = w.gI; a.gI2 = w.gI + (size_t)b->N * HID; a.gI_stride = HID;      // dense halves [N][H] | [N][H]
    a.g_core = w.g_core; a.g_readout = w.g_readout; a.kl_scale = s_kl;
    if (!gZ_ext) {
      a.con_g1p = w.g1p; a.con_g2p = w.g2p; a.con_z1 = w.z1; a.con_z2 = w.z2; a.con_n1 = w.n1; a.con_n2 = w.n2;
      a.con_jsplit = js; a.con_scale = s_con;
    }
    a.gp = w.gp; a.g_q = w.g_q; a.gH = w.gH; a.gC = w.gC;
    a.part = w.small_part; a.counter = w.counters + 1;
    a.d_gamma_c = grads + lo.off[SCGIB_P_COMP_GAMMA]; a.d_beta_c = grads + lo.off[SCGIB_P_COMP_BETA];
    a.d_wc2 = grads + lo.off[SCGIB_P_COMP_W2]; a.d_bc2 = grads + lo.off[SCGIB_P_COMP_B2];
    a.d_attn_w = grads + lo.off[SCGIB_P_ATTN_W]; a.d_attn_b = grads + lo.off[SCGIB_P_ATTN_B];
    a.gmax_q = use_h ? w.counters + 53 : nullptr;
    PROF("graph_gate_bwd", launch_graph_gate_bwd(a, HID, s));
  }
  if (use_h) {      // compressor.0 backward = one linear layer on the fp16-split tensor-core kernel (half mode of gin_bwd_h.cu)
    PROF("gate_lin_bwd_h", launch_linear_bwd_h(w.g_q, w.H, params + lo.off[SCGIB_P_COMP_W1], b->N, w.gH, w.head_bn, w.head_cvec,
                                               w.counters + 53, w.ppart, lo.total, lo.off[SCGIB_P_COMP_W1], lo.off[SCGIB_P_COMP_B1], GP, s));
  } else {
    GateLinBwdArgs a{w.g_q, w.H, b->N, params + lo.off[SCGIB_P_COMP_W1], w.gH, w.ppart, lo.total,
                     lo.off[SCGIB_P_COMP_W1], lo.off[SCGIB_P_COMP_B1]};
    PROF("gate_lin_bwd", launch_gate_lin_bwd(a, HID, GP, s));
  }
  const int enc_split = pair_split(GP, (b->N + 127) / 128, (b->Ns + 127) / 128);   // CTAs of Encoder1 in a shared launch
  const bool pair_main = bf || tc_bwd;
  for (int l = L - 1; l >= 0; --l) {
    const int kin = l == 0 ? DTR : HID;
    GinBwdPreArgs pa[2];
    GinBwdMainArgs ma[2];
    for (int e = 0; e < 2; ++e) {
      const int V = e == 0 ? b->N : b->Ns;
      GinBwdPreArgs& q = pa[e];
      if (l == L - 1) {
        q.src = e == 0 ? w.gH : w.gC; q.indptr = nullptr; q.indices = nullptr; q.map = e == 0 ? nullptr : b->ego_seed;
      } else {
        q.src = w.Ga[e]; q.indptr = e == 0 ? b->indptr : b->sub_indptr; q.indices = e == 0 ? b->indices : b->sub_indices; q.map = nullptr;
      }
      q.y = w.y[e][l]; q.bn = w.bn[e][l]; q.V = V; q.g_o = w.g_o[e];
      q.part = e == 0 ? w.small_part : w.small_part2; q.counter = w.counters + (e == 0 ? 2 : 10);
      q.d_gamma = grads + lo.enc(e, l, L, SCGIB_ENC_GAMMA); q.d_beta = grads + lo.enc(e, l, L, SCGIB_ENC_BETA);
      q.cvec = w.cvec[e];
      q.gmax = use_h ? gm_layer(e, l) : nullptr;
      GinBwdMainArgs& m = ma[e];
      m.gmax = gm_layer(e, l);
      m.g_o = w.g_o[e]; m.y = w.y[e][l]; m.r = w.r[e][l]; m.a = w.a[e][l]; m.bn = w.bn[e][l]; m.cvec = w.cvec[e];
      m.W1 = params + lo.enc(e, l, L, SCGIB_ENC_W1); m.W2 = params + lo.enc(e, l, L, SCGIB_ENC_W2);
      m.V = V; m.g_a = l == 0 ? w.ga0[e] : w.Ga[e]; m.part = w.ppart; m.pstride = lo.total;
      m.off_W1 = lo.enc(e, l, L, SCGIB_ENC_W1); m.off_b1 = lo.enc(e, l, L, SCGIB_ENC_B1);
      m.off_W2 = lo.enc(e, l, L, SCGIB_ENC_W2); m.off_b2 = lo.enc(e, l, L, SCGIB_ENC_B2);
    }
    if (bf) {
      PROF("gin_bwd_pre_bf16.enc1+2", launch_gin_bwd_pre_bf16(pa[0], &pa[1], HID, s));
      PROF("gin_bwd_main_bf16.enc1+2", launch_gin_bwd_main_bf16(ma[0], &ma[1], kin, HID, GP, s));
      continue;
    }
    PROF("gin_bwd_pre.enc1+2", launch_gin_bwd_pre_pair(pa[0], pa[1], HID, s));
    if (use_h) {
      PROF("gin_bwd_main_h.enc1+2", launch_gin_bwd_main_h_pair(ma[0], ma[1], kin, GP, s));
    } else if (pair_main) {
      PROF("gin_bwd_main_tc.enc1+2", launch_gin_bwd_main_tc2_pair(ma[0], ma[1], kin, GP, s));
    } else {
      PROF("gin_bwd_main_ffma.enc1", launch_gin_bwd_main(ma[0], kin, HID, GP, s));
      PROF("gin_bwd_main_ffma.enc2", launch_gin_bwd_main(ma[1], kin, HID, GP, s));
    }
  }
  {
    InputProjBwdArgs a;
    a.ga[0] = w.ga0[0]; a.ga[1] = w.ga0[1]; a.xagg[0] = w.xagg[0]; a.xagg[1] = w.xagg[1]; a.xa_stride = xagg_stride(d);
    a.V[0] = b->N; a.V[1] = b->Ns; a.F = d->in_dim; a.part = w.small_part; a.counter = w.counters + 3;
    a.d_Wt = grads + lo.off[SCGIB_P_TRANSFER];
    PROF("input_proj_bwd", launch_input_proj_bwd(a, s));
  }
  {
    ReduceRanges r;
    r.n = 0;
    auto add = [&](int64_t off, int64_t len, int c0, int c1) { r.off[r.n] = off; r.len[r.n] = len; r.c0[r.n] = c0; r.c1[r.n] = c1; ++r.n; };
    // shared tcgen05 launch: partial rows [0, head_split) = problem 0 (dW1a and everything else), [head_split, GP) = problem 1
    // (dW1b); FFMA: two launches, every partial row holds both.  The partial slot holds [dW1a | dW1b] ([2][H][H]); the
    // reduction writes them interleaved as the parameter's [H][2H] layout.
    add(lo.off[SCGIB_P_HEAD_W1], (int64_t)HID * HID, 0, head_split);
    r.dst[r.n - 1] = lo.off[SCGIB_P_HEAD_W1]; r.ilv[r.n - 1] = HID;
    add(lo.off[SCGIB_P_HEAD_W1] + (int64_t)HID * HID, (int64_t)HID * HID, head_pair ? head_split : 0, GP);
    r.dst[r.n - 1] = lo.off[SCGIB_P_HEAD_W1] + HID; r.ilv[r.n - 1] = HID;
    add(lo.off[SCGIB_P_HEAD_B1], lo.off[SCGIB_P_HEAD_B2] + HID - lo.off[SCGIB_P_HEAD_B1], 0, head_split);
    add(lo.off[SCGIB_P_COMP_W1], lo.off[SCGIB_P_COMP_B1] + HID - lo.off[SCGIB_P_COMP_W1], 0, GP);
    for (int e = 0; e < 2; ++e)        // shared launches: partial rows [0, split) belong to Encoder1, [split, GP) to Encoder2
      for (int l = 0; l < L; ++l)
        add(lo.enc(e, l, L, SCGIB_ENC_W1), lo.enc(e, l, L, SCGIB_ENC_B2) + HID - lo.enc(e, l, L, SCGIB_ENC_W1),
            pair_main ? (e == 0 ? 0 : enc_split) : 0, pair_main ? (e == 0 ? enc_split : GP) : GP);
    PROF("reduce_partials", launch_reduce_partials(w.ppart, lo.total, GP, r, grads, s));
  }
  return (int)cudaGetLastError();
}

extern "C" SCGIB_API int scgib_pretrain_backward_f32(const ScgibDims* d, const float* params, const ScgibBatch* b,
                                           const float* loss_scale, float* grads, void* workspace,
                                           size_t workspace_bytes, void* stream) {
  return backward_impl(d, params, b, loss_scale, nullptr, grads, workspace, workspace_bytes, stream);
}

extern "C" SCGIB_API int scgib_extract_backward_f32(const ScgibDims* d, const float* params, const ScgibBatch* b,
                                          const float* gZ, float* grads, void* workspace, size_t workspace_bytes,
                                          void* stream) {
  if (!gZ) return SCGIB_E_NULL;
  const float zero[3] = {0.f, 0.f, 0.f};
  return backward_impl(d, params, b, zero, gZ, grads, workspace, workspace_bytes, stream);
}

extern "C" SCGIB_API int scgib_adam_step_f32(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                                   int64_t step, float lr, float beta1, float beta2, float eps, float weight_decay,
                                   float grad_scale, void* stream) {
  if (!params || !grads || !exp_avg || !exp_avg_sq) return SCGIB_E_NULL;
  if (n < 1 || step < 1) return SCGIB_E_RANGE;
  cudaStream_t s = (cudaStream_t)stream;
  PROF("adam", launch_adam(params, grads, exp_avg, exp_avg_sq, n, step, lr, beta1, beta2, eps, weight_decay, grad_scale, s));
  return (int)cudaGetLastError();
}

// ---------------------------------------------------------------- fine-tuning head (Set2Set + predict)
namespace scgib {
struct FtLayout { int64_t off[SCGIB_FT_SLOTS], size[SCGIB_FT_SLOTS], total; };
static FtLayout ft_layout(int H, int C) {
  FtLayout lo;
  const int64_t sz[SCGIB_FT_SLOTS] = {(int64_t)4 * H * 2 * H, (int64_t)4 * H * H, 4 * H, 4 * H, (int64_t)H * 2 * H, H, (int64_t)C * H, C};
  int64_t o = 0;
  for (int i = 0; i < SCGIB_FT_SLOTS; ++i) { lo.off[i] = o; lo.size[i] = sz[i]; o += (sz[i] + 3) / 4 * 4; }
  lo.total = o;
  return lo;
}
struct FtWs { float *WlstmT, *Wp1T, *gates, *cst, *qstar, *alpha, *rp, *g_pre, *g_u, *dgates, *gp, *scratch; size_t bytes; };
static FtWs ft_carve(int H, int C, int T, int B, int N, void* base) {
  FtWs w;
  char* p = (char*)base;
  size_t o = 0;
  auto take = [&](size_t nfloats) { float* r = (float*)(p + o); o += al(nfloats * sizeof(float)); return r; };
  w.WlstmT = take((size_t)3 * H * 4 * H); w.Wp1T = take((size_t)2 * H * H);
  w.gates = take((size_t)T * B * 4 * H); w.cst = take((size_t)T * B * H); w.qstar = take((size_t)T * B * 2 * H);
  w.alpha = take((size_t)T * N); w.rp = take((size_t)B * H); w.g_pre = take((size_t)B * C); w.g_u = take((size_t)B * H);
  w.dgates = take((size_t)T * B * 4 * H); w.gp = take(N);
  w.scratch = take((size_t)atb_splits(T * B) * 4 * H * 2 * H);     // row-split partials of the weight-gradient reductions
  w.bytes = o;
  return w;
}
static bool ft_dims_ok(int H, int C, int T) { return (H == 32 || H == 64 || H == 128) && C >= 0 && C <= finetune_max_classes() && T >= 1 && T <= 8; }
}  // namespace scgib

extern "C" SCGIB_API int64_t scgib_finetune_head_layout(int32_t H, int32_t C, int64_t* offsets, int64_t* sizes) {
  if (!ft_dims_ok(H, C, 1)) return SCGIB_E_SHAPE;
  const FtLayout lo = ft_layout(H, C);
  for (int i = 0; i < SCGIB_FT_SLOTS; ++i) {
    if (offsets) offsets[i] = lo.off[i];
    if (sizes) sizes[i] = lo.size[i];
  }
  return lo.total;
}

extern "C" SCGIB_API size_t scgib_finetune_head_workspace_bytes(int32_t H, int32_t C, int32_t T, int32_t B, int32_t N) {
  if (!ft_dims_ok(H, C, T) || B < 1 || N < 1) return 0;
  return ft_carve(H, C, T, B, N, nullptr).bytes;
}

extern "C" SCGIB_API int scgib_finetune_head_fwd_f32(const float* head_params, int32_t H, int32_t C, int32_t T, int32_t sigmoid,
                                           const float* Z, const int32_t* graph_ptr, int32_t B, int32_t N, float* scores,
                                           float* readout, void* workspace, size_t workspace_bytes, void* stream_) {
  if (!ft_dims_ok(H, C, T)) return SCGIB_E_SHAPE;
  if (!head_params || !Z || !graph_ptr || (!scores && C > 0) || !workspace) return SCGIB_E_NULL;
  if (B < 1 || N < 1) return SCGIB_E_RANGE;
  if (((uintptr_t)workspace & 255u) != 0 || ((uintptr_t)head_params & 15u) != 0 || ((uintptr_t)Z & 15u) != 0) return SCGIB_E_ALIGN;
  const FtLayout lo = ft_layout(H, C);
  const FtWs w = ft_carve(H, C, T, B, N, workspace);
  if (workspace_bytes < w.bytes) return SCGIB_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream_;
  TransposeJobs jobs;
  jobs.n = 3;
  jobs.job[0] = TransposeJob{head_params + lo.off[SCGIB_FT_LSTM_WIH], w.WlstmT, 4 * H, 2 * H};
  jobs.job[1] = TransposeJob{head_params + lo.off[SCGIB_FT_LSTM_WHH], w.WlstmT + (size_t)2 * H * 4 * H, 4 * H, H};
  jobs.job[2] = TransposeJob{head_params + lo.off[SCGIB_FT_PRED_W1], w.Wp1T, H, 2 * H};
  PROF("ft_transpose_weights", launch_transposes(jobs, s));
  FinetuneHeadFwdArgs a;
  a.Z = Z; a.graph_ptr = graph_ptr; a.B = B; a.N = N; a.H = H; a.C = C; a.T = T; a.sigmoid = sigmoid;
  a.WlstmT = w.WlstmT; a.b_ih = head_params + lo.off[SCGIB_FT_LSTM_BIH]; a.b_hh = head_params + lo.off[SCGIB_FT_LSTM_BHH];
  a.Wp1T = w.Wp1T; a.bp1 = head_params + lo.off[SCGIB_FT_PRED_B1];
  a.Wp2 = head_params + lo.off[SCGIB_FT_PRED_W2]; a.bp2 = head_params + lo.off[SCGIB_FT_PRED_B2];
  a.gates = w.gates; a.cst = w.cst; a.qstar = w.qstar; a.alpha = w.alpha; a.rp = w.rp; a.scores = scores;
  PROF("finetune_head_fwd", launch_finetune_head_fwd(a, s));
  if (readout)
    cudaMemcpyAsync(readout, w.qstar + (size_t)(T - 1) * B * 2 * H, (size_t)B * 2 * H * sizeof(float), cudaMemcpyDeviceToDevice, s);
  return (int)cudaGetLastError();
}

extern "C" SCGIB_API int scgib_finetune_head_bwd_f32(const float* head_params, int32_t H, int32_t C, int32_t T, int32_t sigmoid,
                                           const float* Z, const int32_t* graph_ptr, int32_t B, int32_t N,
                                           const float* scores, const float* g_scores, const float* g_readout, float* gZ,
                                           float* head_grads, void* workspace, size_t workspace_bytes, void* stream_) {
  if (!ft_dims_ok(H, C, T)) return SCGIB_E_SHAPE;
  if (!head_params || !Z || !graph_ptr || !gZ || !head_grads || !workspace) return SCGIB_E_NULL;
  if ((C > 0 && (!scores || !g_scores)) || (C == 0 && !g_readout)) return SCGIB_E_NULL;
  if (B < 1 || N < 1) return SCGIB_E_RANGE;
  if (((uintptr_t)workspace & 255u) != 0 || ((uintptr_t)head_params & 15u) != 0 || ((uintptr_t)Z & 15u) != 0 ||
      ((uintptr_t)gZ & 15u) != 0)
    return SCGIB_E_ALIGN;
  const FtLayout lo = ft_layout(H, C);
  const FtWs w = ft_carve(H, C, T, B, N, workspace);
  if (workspace_bytes < w.bytes) return SCGIB_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream_;
  FinetuneHeadBwdArgs a;
  a.Z = Z; a.graph_ptr = graph_ptr; a.B = B; a.N = N; a.H = H; a.C = C; a.T = T; a.sigmoid = sigmoid;
  a.Wih = head_params + lo.off[SCGIB_FT_LSTM_WIH]; a.Whh = head_params + lo.off[SCGIB_FT_LSTM_WHH];
  a.Wp1 = head_params + lo.off[SCGIB_FT_PRED_W1]; a.Wp2 = head_params + lo.off[SCGIB_FT_PRED_W2];
  a.gates = w.gates; a.cst = w.cst; a.qstar = w.qstar; a.alpha = w.alpha; a.rp = w.rp; a.scores = scores;
  a.g_scores = g_scores; a.g_readout = g_readout; a.g_pre = w.g_pre; a.g_u = w.g_u; a.dgates = w.dgates; a.gp = w.gp; a.gZ = gZ;
  PROF("finetune_head_bwd", launch_finetune_head_bwd(a, s));
  // weight gradients: fixed-order reductions over the graphs
  float* g = head_grads;
  if (T > 1) {   // the LSTM input of step t is q*_{t-1} (zero at t = 0)
    PROF("ft_dWih", launch_atb(w.dgates + (size_t)B * 4 * H, 4 * H, w.qstar, 2 * H, g + lo.off[SCGIB_FT_LSTM_WIH], 2 * H, nullptr, (T - 1) * B, 4 * H, 2 * H, w.scratch, s));
    PROF("ft_dWhh", launch_atb(w.dgates + (size_t)B * 4 * H, 4 * H, w.qstar, 2 * H, g + lo.off[SCGIB_FT_LSTM_WHH], H, nullptr, (T - 1) * B, 4 * H, H, w.scratch, s));
  } else {
    cudaMemsetAsync(g + lo.off[SCGIB_FT_LSTM_WIH], 0, (size_t)(lo.off[SCGIB_FT_LSTM_BIH] - lo.off[SCGIB_FT_LSTM_WIH]) * sizeof(float), s);
  }
  PROF("ft_dbias", launch_atb(w.dgates, 4 * H, nullptr, 0, g + lo.off[SCGIB_FT_LSTM_BIH], 1, g + lo.off[SCGIB_FT_LSTM_BHH], T * B, 4 * H, 1, w.scratch, s));
  if (C == 0) {     // readout only: the predict slots get zero gradients
    cudaMemsetAsync(g + lo.off[SCGIB_FT_PRED_W1], 0, (size_t)(lo.total - lo.off[SCGIB_FT_PRED_W1]) * sizeof(float), s);
    return (int)cudaGetLastError();
  }
  PROF("ft_dWp1", launch_atb(w.g_u, H, w.qstar + (size_t)(T - 1) * B * 2 * H, 2 * H, g + lo.off[SCGIB_FT_PRED_W1], 2 * H, nullptr, B, H, 2 * H, w.scratch, s));
  PROF("ft_dbp1", launch_atb(w.g_u, H, nullptr, 0, g + lo.off[SCGIB_FT_PRED_B1], 1, nullptr, B, H, 1, w.scratch, s));
  PROF("ft_dWp2", launch_atb(w.g_pre, C, w.rp, H, g + lo.off[SCGIB_FT_PRED_W2], H, nullptr, B, C, H, w.scratch, s));
  PROF("ft_dbp2", launch_atb(w.g_pre, C, nullptr, 0, g + lo.off[SCGIB_FT_PRED_B2], 1, nullptr, B, C, 1, w.scratch, s));
  return (int)cudaGetLastError();
}

// ---------------------------------------------------------------- individual operators
extern "C" SCGIB_API int scgib_input_proj_fwd_f32(const float* x, const float* Wt, int32_t N, int32_t F, int32_t DT, float* t, void* stream) {
  if (!x || !Wt || !t) return SCGIB_E_NULL;
  if (DT != DTR || F < 1 || F > 32) return SCGIB_E_SHAPE;
  if (N < 1) return SCGIB_E_RANGE;
  launch_input_proj_fwd(x, Wt, N, F, 1, t, (cudaStream_t)stream);
  return (int)cudaGetLastError();
}

// transfer_d backward as an operator: dWt[o][f] = sum over both row sets of g_r[o] * xrow_r[f], xrow_r = x_hat[p(r)] (+ the
// x_hat rows of r's neighbours when a CSR is given: the layer-0 aggregation backward of the GIN path moved to the features)
extern "C" SCGIB_API size_t scgib_transfer_bwd_workspace_bytes(int32_t V0, int32_t V1, int32_t F) {
  const size_t xs = (size_t)(F + 3) / 4 * 4;
  return al((size_t)V0 * xs * 4) + al((size_t)V1 * xs * 4) + al((size_t)input_proj_bwd_grid(V0, V1) * DTR * 32 * 4) + 256;
}
extern "C" SCGIB_API int scgib_transfer_bwd_f32(const float* x, int32_t F, int32_t normalize, const float* g0, int32_t V0,
                                                const int32_t* indptr0, const int32_t* indices0, const float* g1, int32_t V1,
                                                const int32_t* indptr1, const int32_t* indices1, const int32_t* map1,
                                                float* dWt, void* workspace, size_t workspace_bytes, void* stream) {
  if (!x || !g0 || !dWt || !workspace || (V1 > 0 && (!g1 || !map1))) return SCGIB_E_NULL;
  if (F < 1 || F > 32) return SCGIB_E_SHAPE;
  if (V0 < 1 || V1 < 0) return SCGIB_E_RANGE;
  if (((uintptr_t)workspace & 255u) != 0) return SCGIB_E_ALIGN;
  if (workspace_bytes < scgib_transfer_bwd_workspace_bytes(V0, V1, F)) return SCGIB_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  const int xs = (F + 3) / 4 * 4;
  char* p = (char*)workspace;
  float* xa0 = (float*)p; p += al((size_t)V0 * xs * 4);
  float* xa1 = (float*)p; p += al((size_t)V1 * xs * 4);
  float* part = (float*)p; p += al((size_t)input_proj_bwd_grid(V0, V1) * DTR * 32 * 4);
  unsigned int* counter = (unsigned int*)p;
  cudaMemsetAsync(counter, 0, 64, s);
  FwdPrepArgs pa;
  pa.jobs.n = 0;
  pa.F = F; pa.normalize = normalize;
  pa.xa_indptr[0] = indptr0; pa.xa_indices[0] = indices0; pa.xa_indptr[1] = indptr1; pa.xa_indices[1] = indices1;
  pa.xa_map = map1; pa.xa_V[0] = V0; pa.xa_V[1] = V1; pa.xagg[0] = xa0; pa.xagg[1] = xa1; pa.xa_stride = xs;
  pa.xa_x = x;
  launch_fwd_prep(pa, s, false);
  InputProjBwdArgs a;
  a.ga[0] = g0; a.ga[1] = g1 ? g1 : g0; a.xagg[0] = xa0; a.xagg[1] = xa1; a.xa_stride = xs;
  a.V[0] = V0; a.V[1] = V1; a.F = F; a.part = part; a.counter = counter; a.d_Wt = dWt;
  launch_input_proj_bwd(a, s);
  return (int)cudaGetLastError();
}

extern "C" SCGIB_API size_t scgib_gin_workspace_bytes(int32_t V) {
  size_t part = (size_t)((V + 63) / 64) * 2 * HID * sizeof(float);
  const size_t part2 = (size_t)num_sms() * 3 * HID * sizeof(double);
  if (part2 > part) part = part2;
  return al(part) + al(HID * HID * sizeof(float)) * 2 + 256;
}

extern "C" SCGIB_API int scgib_gin_layer_fwd_f32(const float* in, int32_t kin, const int32_t* row_map, const float* bn_in,
                                       const int32_t* indptr, const int32_t* indices, int32_t V, const float* W1,
                                       const float* b1, const float* W2, const float* b2, float* a_out, float* r_out,
                                       float* y_out, float* bn_out, float* running, void* workspace,
                                       size_t workspace_bytes, void* stream_) {
  if (!in || !indptr || !W1 || !b1 || !W2 || !b2 || !y_out || !bn_out || !workspace) return SCGIB_E_NULL;
  if (kin != DTR && kin != HID) return SCGIB_E_SHAPE;
  if (bn_in && kin != HID) return SCGIB_E_SHAPE;
  if (V < 1) return SCGIB_E_RANGE;
  if (workspace_bytes < scgib_gin_workspace_bytes(V)) return SCGIB_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream_;
  char* p = (char*)workspace;
  float* w1t = (float*)p; p += al(HID * HID * sizeof(float));
  float* w2t = (float*)p; p += al(HID * HID * sizeof(float));
  unsigned int* counter = (unsigned int*)p; p += 256;
  float* part = (float*)p;
  cudaMemsetAsync(counter, 0, 256, s);
  TransposeJobs jobs;
  jobs.n = 2;
  jobs.job[0] = TransposeJob{W1, w1t, HID, kin};
  jobs.job[1] = TransposeJob{W2, w2t, HID, HID};
  launch_transposes(jobs, s);
  GinFwdArgs a;
  a.in = in; a.row_map = row_map; a.bn_in = bn_in; a.indptr = indptr; a.indices = indices; a.V = V;
  a.W1t = w1t; a.b1 = b1; a.W2t = w2t; a.b2 = b2; a.W1 = W1; a.W2 = W2;
  a.gamma = nullptr; a.beta = nullptr;
  a.a_out = a_out; a.r_out = r_out; a.y_out = y_out; a.part = part; a.counter = counter; a.bn_out = bn_out; a.running = running;
  launch_gin_fwd_any(a, kin, s);
  return (int)cudaGetLastError();
}

// One GINConv + BatchNorm + ReLU layer backward (the three kernels the whole-step backward uses per layer)
namespace scgib {
struct GinBwdOpWs { float *g_o, *cvec, *part2, *ppart; unsigned int* counter; int64_t off[4], pstride; size_t bytes; };
static GinBwdOpWs gin_bwd_op_carve(int V, int kin, void* base) {
  GinBwdOpWs w;
  char* p = (char*)base;
  size_t o = 0;
  auto take = [&](size_t nfloats) { float* r = (float*)(p + o); o += al(nfloats * sizeof(float)); return r; };
  w.g_o = take((size_t)V * HID); w.cvec = take(2 * HID);
  w.part2 = take((size_t)(gin_bwd_pre_grid(V) + 2) * 2 * HID);
  w.counter = (unsigned int*)take(64);
  w.off[0] = 0; w.off[1] = (int64_t)HID * kin; w.off[2] = w.off[1] + HID; w.off[3] = w.off[2] + (int64_t)HID * HID;   // W1 b1 W2 b2
  w.pstride = w.off[3] + HID;
  w.ppart = take((size_t)num_sms() * w.pstride);
  w.bytes = o;
  return w;
}
}  // namespace scgib

extern "C" SCGIB_API size_t scgib_gin_layer_bwd_workspace_bytes(int32_t V, int32_t kin) {
  if (V < 1 || (kin != DTR && kin != HID)) return 0;
  return gin_bwd_op_carve(V, kin, nullptr).bytes;
}

extern "C" SCGIB_API int scgib_gin_layer_bwd_f32(const float* g_next, const int32_t* indptr, const int32_t* indices, int32_t V,
                                       int32_t kin, const float* y, const float* r, const float* a, const float* bn,
                                       const float* W1, const float* W2, float* g_a, float* dW1, float* db1, float* dW2,
                                       float* db2, float* dgamma, float* dbeta, void* workspace, size_t workspace_bytes,
                                       void* stream_) {
  if (!g_next || !y || !r || !a || !bn || !W1 || !W2 || !g_a || !dW1 || !db1 || !dW2 || !db2 || !dgamma || !dbeta || !workspace)
    return SCGIB_E_NULL;
  if (indptr && !indices) return SCGIB_E_NULL;
  if (kin != DTR && kin != HID) return SCGIB_E_SHAPE;
  if (V < 1) return SCGIB_E_RANGE;
  if (((uintptr_t)workspace & 255u) != 0) return SCGIB_E_ALIGN;
  const GinBwdOpWs w = gin_bwd_op_carve(V, kin, workspace);
  if (workspace_bytes < w.bytes) return SCGIB_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream_;
  const int GP = num_sms();
  cudaMemsetAsync(w.counter, 0, 256, s);
  GinBwdPreArgs q;
  q.src = g_next; q.indptr = indptr; q.indices = indptr ? indices : nullptr; q.map = nullptr;
  q.y = y; q.bn = bn; q.V = V; q.g_o = w.g_o; q.part = w.part2; q.counter = w.counter;
  q.d_gamma = dgamma; q.d_beta = dbeta; q.cvec = w.cvec;
  const bool use_h = bwd_tensor_core_mode() != 0 && bwd_h_mode() != 0 && (((uintptr_t)y | (uintptr_t)r | (uintptr_t)a | (uintptr_t)g_a) & 31u) == 0;
  q.gmax = use_h ? w.counter + 32 : nullptr;         // max |g_o| for the fp16-split kernel's gradient normalisation (zeroed above)
  launch_gin_bwd_pre(q, HID, s);
  GinBwdMainArgs m;
  m.g_o = w.g_o; m.y = y; m.r = r; m.a = a; m.bn = bn; m.cvec = w.cvec; m.W1 = W1; m.W2 = W2; m.V = V; m.g_a = g_a;
  m.part = w.ppart; m.pstride = w.pstride; m.off_W1 = w.off[0]; m.off_b1 = w.off[1]; m.off_W2 = w.off[2]; m.off_b2 = w.off[3];
  m.gmax = w.counter + 32;
  if (use_h) launch_gin_bwd_main_h(m, kin, GP, s);
  else if (bwd_tensor_core_mode() != 0) launch_gin_bwd_main_tc2(m, kin, GP, s);
  else launch_gin_bwd_main(m, kin, HID, GP, s);
  // per-CTA partials -> the four gradient tensors (fixed order)
  float* outs[4] = {dW1, db1, dW2, db2};
  const int64_t lens[4] = {(int64_t)HID * kin, HID, (int64_t)HID * HID, HID};
  for (int i = 0; i < 4; ++i) {
    ReduceRanges rr;
    rr.n = 1; rr.off[0] = w.off[i]; rr.len[0] = lens[i]; rr.c0[0] = 0; rr.c1[0] = GP;
    launch_reduce_partials(w.ppart, w.pstride, GP, rr, outs[i] - w.off[i], s);
  }
  return (int)cudaGetLastError();
}

// ---- loss operators (forward + gradient in one call; the units of the whole-step functions)
namespace scgib {
struct LossOpWs { float *rpart, *G, *edge, *z1, *z2, *zsplit, *n1, *n2, *diag, *D, *rowsum, *g1p, *g2p, *kl, *losses; size_t bytes; };
static LossOpWs loss_op_carve(int B, void* base, int HID = scgib::HID) {
  LossOpWs w;
  char* p = (char*)base;
  size_t o = 0;
  auto take = [&](size_t nfloats) { float* r = (float*)(p + o); o += al(nfloats * sizeof(float)); return r; };
  const int js = contrastive_jsplit(B > 0 ? B : 1);
  w.rpart = take((size_t)recon_fwd_grid() * (HID * HID + 4)); w.G = take(HID * HID); w.edge = take(4);
  w.z1 = take((size_t)B * HID); w.z2 = take((size_t)B * HID); w.zsplit = take((size_t)4 * B * HID);
  w.n1 = take(B); w.n2 = take(B); w.diag = take(B); w.D = take(B); w.rowsum = take((size_t)js * B);
  w.g1p = take((size_t)js * B * HID); w.g2p = take((size_t)js * B * HID); w.kl = take(4); w.losses = take(4);
  w.bytes = o;
  return w;
}
}  // namespace scgib

extern "C" SCGIB_API size_t scgib_loss_workspace_bytes(int32_t B) { return B < 0 ? 0 : loss_op_carve(B, nullptr).bytes; }
extern "C" SCGIB_API size_t scgib_loss_workspace_bytes_h(int32_t B, int32_t hidden) {
  return (B < 0 || (hidden != 64 && hidden != 128)) ? 0 : loss_op_carve(B, nullptr, hidden).bytes;
}

static int recon_adj_impl(const float* Z, const int32_t* indptr, const int32_t* indices, int32_t N, int32_t E, const int HID,
                          float scale, float* loss, float* gZ, void* workspace, size_t workspace_bytes, void* stream_) {
  if (!Z || !indptr || !loss || !workspace || (E > 0 && !indices)) return SCGIB_E_NULL;
  if (HID != 64 && HID != 128) return SCGIB_E_SHAPE;
  if (N < 1 || E < 0) return SCGIB_E_RANGE;
  if (((uintptr_t)workspace & 255u) != 0 || ((uintptr_t)Z & 15u) != 0 || ((uintptr_t)gZ & 15u) != 0) return SCGIB_E_ALIGN;
  const LossOpWs w = loss_op_carve(1, workspace, HID);
  if (workspace_bytes < w.bytes) return SCGIB_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream_;
  const int grid = num_sms();
  ReconFwdArgs a{Z, indptr, indices, N, w.rpart};
  launch_recon_fwd(a, HID, grid, s);
  launch_recon_reduce(w.rpart, grid, w.G, w.edge, HID, s);
  cudaMemsetAsync(w.kl, 0, 4 * sizeof(float), s);
  cudaMemsetAsync(w.rowsum, 0, sizeof(float), s);
  cudaMemsetAsync(w.diag, 0, sizeof(float), s);
  LossFinalizeArgs f{w.rowsum, 1, w.diag, 0, w.G, w.edge, N, E, nullptr, w.kl, w.D, w.losses, HID};   // B = 0: only the recon term
  launch_loss_finalize(f, s);
  cudaMemcpyAsync(loss, w.losses + 2, sizeof(float), cudaMemcpyDeviceToDevice, s);
  if (gZ) {
    ReconBwdArgs ra{Z, w.G, indptr, indices, N, scale, gZ};
    launch_recon_bwd(ra, HID, s);
  }
  return (int)cudaGetLastError();
}

extern "C" SCGIB_API int scgib_recon_adj_f32(const float* Z, const int32_t* indptr, const int32_t* indices, int32_t N, int32_t E,
                                   float scale, float* loss, float* gZ, void* workspace, size_t workspace_bytes, void* stream_) {
  return recon_adj_impl(Z, indptr, indices, N, E, HID, scale, loss, gZ, workspace, workspace_bytes, stream_);
}
extern "C" SCGIB_API int scgib_recon_adj_h_f32(const float* Z, const int32_t* indptr, const int32_t* indices, int32_t N, int32_t E,
                                     int32_t hidden, float scale, float* loss, float* gZ, void* workspace, size_t workspace_bytes,
                                     void* stream_) {
  return recon_adj_impl(Z, indptr, indices, N, E, hidden, scale, loss, gZ, workspace, workspace_bytes, stream_);
}

static int contrastive_impl(const float* core, const float* readout, int32_t B, const int HID, float scale, float* loss,
                            float* g_core, float* g_readout, void* workspace, size_t workspace_bytes, void* stream_) {
  if (!core || !readout || !loss || !workspace) return SCGIB_E_NULL;
  if ((g_core == nullptr) != (g_readout == nullptr)) return SCGIB_E_NULL;
  if (HID != 64 && HID != 128) return SCGIB_E_SHAPE;
  if (B < 1) return SCGIB_E_RANGE;
  if (((uintptr_t)workspace & 255u) != 0 || ((uintptr_t)core & 15u) != 0 || ((uintptr_t)readout & 15u) != 0) return SCGIB_E_ALIGN;
  const LossOpWs w = loss_op_carve(B, workspace, HID);
  if (workspace_bytes < w.bytes) return SCGIB_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream_;
  const int js = contrastive_jsplit(B);
  const bool tc = HID == 64 && use_tc_contrastive();          // the tcgen05 contrastive kernels are built for hidden 64
  NormalizeArgs na{core, readout, B, w.z1, w.z2, w.n1, w.n2, w.diag, tc ? w.zsplit : nullptr};
  launch_normalize(na, HID, s);
  ContrastiveFwdArgs c{w.z1, w.z2, B, js, w.rowsum, w.zsplit};
  if (tc) launch_contrastive_fwd_tc(c, s); else launch_contrastive_fwd(c, HID, s);
  cudaMemsetAsync(w.kl, 0, 4 * sizeof(float), s);
  cudaMemsetAsync(w.G, 0, HID * HID * sizeof(float), s);
  cudaMemsetAsync(w.edge, 0, 4 * sizeof(float), s);
  LossFinalizeArgs f{w.rowsum, js, w.diag, B, w.G, w.edge, 1, 0, nullptr, w.kl, w.D, w.losses, HID};
  launch_loss_finalize(f, s);
  cudaMemcpyAsync(loss, w.losses + 1, sizeof(float), cudaMemcpyDeviceToDevice, s);
  if (g_core) {
    ContrastiveBwdArgs a{w.z1, w.z2, w.D, B, js, w.g1p, w.g2p};
    if (tc) launch_contrastive_bwd_tc(a, w.zsplit, s); else launch_contrastive_bwd(a, HID, s);
    ContrastiveBwdFinArgs fa{w.g1p, w.g2p, w.z1, w.z2, w.n1, w.n2, B, js, scale, g_core, g_readout};
    launch_contrastive_bwd_finalize(fa, HID, s);
  }
  return (int)cudaGetLastError();
}
extern "C" SCGIB_API int scgib_contrastive_f32(const float* core, const float* readout, int32_t B, float scale, float* loss,
                                     float* g_core, float* g_readout, void* workspace, size_t workspace_bytes, void* stream_) {
  return contrastive_impl(core, readout, B, HID, scale, loss, g_core, g_readout, workspace, workspace_bytes, stream_);
}
extern "C" SCGIB_API int scgib_contrastive_h_f32(const float* core, const float* readout, int32_t B, int32_t hidden, float scale,
                                       float* loss, float* g_core, float* g_readout, void* workspace, size_t workspace_bytes,
                                       void* stream_) {
  return contrastive_impl(core, readout, B, hidden, scale, loss, g_core, g_readout, workspace, workspace_bytes, stream_);
}

// ---- --recons_type logM as an operator (logm_kernels.cu): hidden 64 or 128
namespace scgib {
struct LogmOpWs { float *walks, *gram, *pair, *loss; size_t bytes; };
static LogmOpWs logm_op_carve(int B, int N, int k, void* base) {
  LogmOpWs w;
  char* p = (char*)base;
  size_t o = 0;
  auto take = [&](size_t nfloats) { float* r = (float*)(p + o); o += al(nfloats * sizeof(float)); return r; };
  w.walks = take((size_t)k * N); w.gram = take(B); w.pair = take(N); w.loss = take(4);
  w.bytes = o;
  return w;
}
}  // namespace scgib

extern "C" SCGIB_API size_t scgib_recon_logm_workspace_bytes(int32_t B, int32_t N, int32_t k) {
  if (B < 1 || N < 2 || k < 1 || k > logm_max_steps()) return 0;
  return logm_op_carve(B, N, k, nullptr).bytes;
}

extern "C" SCGIB_API int scgib_recon_logm_h_f32(const float* Z, const int32_t* graph_ptr, const int32_t* indptr, const int32_t* indices,
                                                int32_t B, int32_t N, int32_t hidden, int32_t k, float scale, float* loss, float* gZ,
                                                int32_t* status, void* workspace, size_t workspace_bytes, void* stream_) {
  if (!Z || !graph_ptr || !indptr || !indices || !loss || !status || !workspace) return SCGIB_E_NULL;
  if (hidden != 64 && hidden != 128) return SCGIB_E_SHAPE;
  if (k < 1 || k > logm_max_steps() || B < 1 || N < 2) return SCGIB_E_RANGE;
  if (((uintptr_t)workspace & 255u) || ((uintptr_t)Z & 15u) || ((uintptr_t)gZ & 15u)) return SCGIB_E_ALIGN;
  const LogmOpWs w = logm_op_carve(B, N, k, workspace);
  if (workspace_bytes < w.bytes) return SCGIB_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream_;
  cudaMemsetAsync(status, 0, sizeof(int32_t), s);
  launch_logm_fwd(Z, graph_ptr, indptr, indices, B, N, k, w.walks, w.gram, w.pair, w.loss, status, hidden, s);
  cudaMemcpyAsync(loss, w.loss, sizeof(float), cudaMemcpyDeviceToDevice, s);
  if (gZ) launch_logm_bwd(Z, graph_ptr, indptr, indices, B, N, k, w.walks, scale, gZ, status, hidden, s);
  return (int)cudaGetLastError();
}

extern "C" SCGIB_API int scgib_segment_sum_f32(const float* in, const int32_t* seg_ptr, int32_t S, const float* bn, float* out, void* stream) {
  if (!in || !seg_ptr || !out) return SCGIB_E_NULL;
  if (S < 1) return SCGIB_E_RANGE;
  launch_segment_sum(in, seg_ptr, S, bn, out, HID, (cudaStream_t)stream);
  return (int)cudaGetLastError();
}

// ---------------------------------------------------------------- op-level entries: core gate, attention, head MLP
namespace scgib {
struct GateOpWs {
  float *Hc, *q, *gstat, *lam, *alpha0, *logit0, *zeros, *gp, *g_q, *gC, *w1t, *bnid, *part, *ppart, *kl, *cstat;
  unsigned int* counters;
  int64_t pstride;
  size_t bytes;
};
static GateOpWs gate_op_carve(int H, int B, int N, void* base) {
  GateOpWs w;
  char* p = (char*)base;
  size_t o = 0;
  auto take = [&](size_t nfloats) { float* r = (float*)(p + o); o += al(nfloats * sizeof(float)); return r; };
  w.Hc = take((size_t)N * H); w.q = take((size_t)N * H); w.gstat = take((size_t)B * 4 * H); w.lam = take(N);
  w.alpha0 = take(N); w.logit0 = take(N); w.zeros = take((size_t)N * H); w.gp = take(N); w.g_q = take((size_t)N * H);
  w.gC = take((size_t)N * H); w.w1t = take((size_t)H * H); w.bnid = take(4 * H);
  w.part = take((size_t)4 * num_sms() * 5 * H);
  w.pstride = (int64_t)H * H + H;
  w.ppart = take((size_t)num_sms() * w.pstride);
  w.kl = take(4);
  w.counters = (unsigned int*)take(64);
  w.cstat = take((size_t)B * 2 * H);
  w.bytes = o;
  return w;
}
static bool hidden_ok(int H) { return H == 64 || H == 128; }
}  // namespace scgib

extern "C" SCGIB_API size_t scgib_core_gate_workspace_bytes(int32_t hidden, int32_t B, int32_t N) {
  if (!hidden_ok(hidden) || B < 1 || N < 2) return 0;
  return gate_op_carve(hidden, B, N, nullptr).bytes;
}

// running == nullptr: training-mode BatchNorm (per-graph batch statistics, kept in cstat for scgib_core_gate_ema_f32);
// otherwise model.eval(): q is normalised with running = {mean, var} and cstat is not written
static int core_gate_fwd_impl(const float* Hfeat, const int32_t* graph_ptr, int32_t B, int32_t N, int32_t hidden, const float* Wc1,
                              const float* bc1, const float* gamma_c, const float* beta_c, const float* wc2, const float* bc2,
                              const float* running, const float* gate_u, const float* feat_u, float* noisy, float* lam,
                              float* graph_readout, float* core_readout, float* kl, void* workspace, size_t workspace_bytes,
                              void* stream_) {
  if (!Hfeat || !graph_ptr || !Wc1 || !bc1 || !gamma_c || !beta_c || !wc2 || !bc2 || !gate_u || !feat_u || !noisy || !graph_readout ||
      !core_readout || !workspace)
    return SCGIB_E_NULL;
  if (!hidden_ok(hidden)) return SCGIB_E_SHAPE;
  if (B < 1 || N < 2) return SCGIB_E_RANGE;
  if (((uintptr_t)workspace & 255u) || ((uintptr_t)Hfeat & 15u) || ((uintptr_t)feat_u & 15u) || ((uintptr_t)noisy & 15u) ||
      ((uintptr_t)running & 15u))
    return SCGIB_E_ALIGN;
  const GateOpWs w = gate_op_carve(hidden, B, N, workspace);
  if (workspace_bytes < w.bytes) return SCGIB_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream_;
  const int H = hidden;
  // Hfeat is used as given (signed features: the GraphSAGE / GCN encoders end without an activation, models.py:88, 103;
  // the fused GIN path applies relu(BN(.)) on load instead): q = compressor.0(Hfeat) on the FP32 linear tiles
  cudaMemcpyAsync(w.Hc, Hfeat, (size_t)N * H * sizeof(float), cudaMemcpyDeviceToDevice, s);
  cudaMemsetAsync(w.logit0, 0, (size_t)N * sizeof(float), s);
  launch_linear_plain(Hfeat, Wc1, bc1, N, H, H, w.q, s);
  GraphGateFwdArgs a;
  a.graph_ptr = graph_ptr; a.B = B; a.N = N; a.H = w.Hc; a.q = w.q;
  a.gamma_c = gamma_c; a.beta_c = beta_c; a.wc2 = wc2; a.bc2 = bc2; a.gate_u = gate_u; a.feat_u = feat_u; a.logit = w.logit0;
  a.noisy = noisy; a.lam = w.lam; a.alpha = w.alpha0; a.readout = graph_readout; a.core = core_readout; a.gstat = w.gstat;
  a.eval_running = running;
  a.cstat = running ? nullptr : w.cstat;      // per-graph batch statistics of q: scgib_core_gate_ema_f32
  a.kl = w.kl;
  launch_graph_gate_fwd(a, H, s);
  if (lam) cudaMemcpyAsync(lam, w.lam, (size_t)N * sizeof(float), cudaMemcpyDeviceToDevice, s);
  if (kl) cudaMemcpyAsync(kl, w.kl, sizeof(float), cudaMemcpyDeviceToDevice, s);
  return (int)cudaGetLastError();
}

extern "C" SCGIB_API int scgib_core_gate_fwd_f32(const float* Hfeat, const int32_t* graph_ptr, int32_t B, int32_t N, int32_t hidden,
                                       const float* Wc1, const float* bc1, const float* gamma_c, const float* beta_c,
                                       const float* wc2, const float* bc2, const float* gate_u, const float* feat_u, float* noisy,
                                       float* lam, float* graph_readout, float* core_readout, float* kl, void* workspace,
                                       size_t workspace_bytes, void* stream_) {
  return core_gate_fwd_impl(Hfeat, graph_ptr, B, N, hidden, Wc1, bc1, gamma_c, beta_c, wc2, bc2, nullptr, gate_u, feat_u, noisy, lam,
                            graph_readout, core_readout, kl, workspace, workspace_bytes, stream_);
}

extern "C" SCGIB_API int scgib_core_gate_eval_fwd_f32(const float* Hfeat, const int32_t* graph_ptr, int32_t B, int32_t N,
                                                      int32_t hidden, const float* Wc1, const float* bc1, const float* gamma_c,
                                                      const float* beta_c, const float* wc2, const float* bc2, const float* running,
                                                      const float* gate_u, const float* feat_u, float* noisy, float* lam,
                                                      float* graph_readout, float* core_readout, float* kl, void* workspace,
                                                      size_t workspace_bytes, void* stream_) {
  if (!running) return SCGIB_E_NULL;
  return core_gate_fwd_impl(Hfeat, graph_ptr, B, N, hidden, Wc1, bc1, gamma_c, beta_c, wc2, bc2, running, gate_u, feat_u, noisy, lam,
                            graph_readout, core_readout, kl, workspace, workspace_bytes, stream_);
}

// compressor.1's running statistics after the B per-graph BatchNorm calls of the forward that filled `workspace`
// (models.py:642: one nn.BatchNorm1d call per graph, momentum 0.1, unbiased variance): running = {mean[H], var[H]}
extern "C" SCGIB_API int scgib_core_gate_ema_f32(int32_t B, int32_t N, int32_t hidden, float* running, void* workspace,
                                                 size_t workspace_bytes, void* stream_) {
  if (!running || !workspace) return SCGIB_E_NULL;
  if (!hidden_ok(hidden)) return SCGIB_E_SHAPE;
  if (B < 1 || N < 2) return SCGIB_E_RANGE;
  if ((uintptr_t)workspace & 255u) return SCGIB_E_ALIGN;
  const GateOpWs w = gate_op_carve(hidden, B, N, workspace);
  if (workspace_bytes < w.bytes) return SCGIB_E_WORKSPACE;
  launch_compressor_ema(w.cstat, B, running, hidden, (cudaStream_t)stream_);
  return (int)cudaGetLastError();
}

extern "C" SCGIB_API int scgib_core_gate_bwd_f32(const int32_t* graph_ptr, int32_t B, int32_t N, int32_t hidden, const float* Wc1,
                                       const float* gamma_c, const float* beta_c, const float* wc2, const float* feat_u,
                                       const float* g_noisy, const float* g_core, const float* g_readout, float kl_scale,
                                       float* gH, float* dWc1, float* dbc1, float* dgamma_c, float* dbeta_c, float* dwc2, float* dbc2,
                                       void* workspace, size_t workspace_bytes, void* stream_) {
  if (!graph_ptr || !Wc1 || !gamma_c || !beta_c || !wc2 || !feat_u || !g_noisy || !g_core || !g_readout || !gH || !dWc1 || !dbc1 ||
      !dgamma_c || !dbeta_c || !dwc2 || !dbc2 || !workspace)
    return SCGIB_E_NULL;
  if (!hidden_ok(hidden)) return SCGIB_E_SHAPE;
  if (B < 1 || N < 2) return SCGIB_E_RANGE;
  if (((uintptr_t)workspace & 255u) || ((uintptr_t)g_noisy & 15u) || ((uintptr_t)gH & 15u)) return SCGIB_E_ALIGN;
  const GateOpWs w = gate_op_carve(hidden, B, N, workspace);
  if (workspace_bytes < w.bytes) return SCGIB_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream_;
  const int H = hidden, GP = num_sms();
  cudaMemsetAsync(w.counters, 0, 64 * sizeof(float), s);
  cudaMemsetAsync(w.zeros, 0, (size_t)N * H * sizeof(float), s);
  cudaMemsetAsync(w.alpha0, 0, (size_t)N * sizeof(float), s);
  GraphGateBwdArgs a;
  a.graph_ptr = graph_ptr; a.B = B; a.N = N; a.H = w.Hc; a.q = w.q; a.C = w.zeros;
  a.gamma_c = gamma_c; a.beta_c = beta_c; a.wc2 = wc2; a.w_cand = w.zeros;     // no attention branch: zero candidates / weights
  a.feat_u = feat_u; a.lam = w.lam; a.alpha = w.alpha0; a.gstat = w.gstat;
  a.gI = g_noisy; a.gI2 = w.zeros; a.gI_stride = H; a.g_core = g_core; a.g_readout = g_readout; a.kl_scale = kl_scale;
  a.gp = w.gp; a.g_q = w.g_q; a.gH = gH; a.gC = w.gC; a.part = w.part; a.counter = w.counters + 1;
  a.d_gamma_c = dgamma_c; a.d_beta_c = dbeta_c; a.d_wc2 = dwc2; a.d_bc2 = dbc2;
  a.d_attn_w = w.bnid; a.d_attn_b = w.kl + 1;                                   // discarded (the attention weights are not part of this op)
  launch_graph_gate_bwd(a, H, s);
  GateLinBwdArgs g{w.g_q, w.Hc, N, Wc1, gH, w.ppart, w.pstride, 0, (int64_t)H * H};
  launch_gate_lin_bwd(g, H, GP, s);
  float* outs[2] = {dWc1, dbc1};
  const int64_t offs[2] = {0, (int64_t)H * H}, lens[2] = {(int64_t)H * H, H};
  for (int i = 0; i < 2; ++i) {
    ReduceRanges rr;
    rr.n = 1; rr.off[0] = offs[i]; rr.len[0] = lens[i]; rr.c0[0] = 0; rr.c1[0] = GP;
    launch_reduce_partials(w.ppart, w.pstride, GP, rr, outs[i] - offs[i], s);
  }
  return (int)cudaGetLastError();
}

// core-candidate attention (models.py:738-748): alpha = softmax_g(w_cand . C_v), T = alpha C.  The core half of attn_layer
// and its bias cancel in the per-graph softmax (their gradients are exactly zero), so only w_cand = attn_layer.weight[0, H:] enters.
extern "C" SCGIB_API int scgib_core_cand_attn_fwd_f32(const float* C, const int32_t* graph_ptr, int32_t B, int32_t N, int32_t hidden,
                                            const float* w_cand, float* alpha, float* T, void* stream) {
  if (!C || !graph_ptr || !w_cand || !alpha) return SCGIB_E_NULL;
  if (hidden < 1 || (hidden & 3)) return SCGIB_E_SHAPE;
  if (B < 1 || N < 1) return SCGIB_E_RANGE;
  launch_attn_fwd(C, graph_ptr, B, hidden, w_cand, alpha, T, (cudaStream_t)stream);
  return (int)cudaGetLastError();
}
// workspace: (N + B * hidden) floats, 256-byte aligned
extern "C" SCGIB_API int scgib_core_cand_attn_bwd_f32(const float* C, const float* alpha, const float* gT, const int32_t* graph_ptr, int32_t B,
                                            int32_t N, int32_t hidden, const float* w_cand, float* gC, float* dw_cand, void* workspace,
                                            size_t workspace_bytes, void* stream_) {
  if (!C || !alpha || !gT || !graph_ptr || !w_cand || !gC || !dw_cand || !workspace) return SCGIB_E_NULL;
  if (hidden < 1 || (hidden & 3)) return SCGIB_E_SHAPE;
  if (B < 1 || N < 1) return SCGIB_E_RANGE;
  if (workspace_bytes < ((size_t)N + (size_t)B * hidden) * sizeof(float) + 256) return SCGIB_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream_;
  float* scratch = (float*)workspace;
  float* dwp = (float*)((char*)workspace + al((size_t)N * sizeof(float)));
  launch_attn_bwd(C, alpha, gT, graph_ptr, B, hidden, w_cand, gC, dwp, scratch, s);
  launch_colsum_rows(dwp, B, hidden, dw_cand, s);
  return (int)cudaGetLastError();
}

extern "C" SCGIB_API int scgib_segment_sum_bwd_f32(const float* g_out, const int32_t* seg_ptr, int32_t S, int32_t hidden, float* g_in,
                                         void* stream) {
  if (!g_out || !seg_ptr || !g_in) return SCGIB_E_NULL;
  if (hidden < 4 || (hidden & 3)) return SCGIB_E_SHAPE;
  if (S < 1) return SCGIB_E_RANGE;
  launch_segment_sum_bwd(g_out, seg_ptr, S, hidden, g_in, (cudaStream_t)stream);
  return (int)cudaGetLastError();
}

// head MLP (models.py:569-572, 676): Z = W2 relu(W1 [noisy || alpha C] + b1) + b2
namespace scgib {
struct HeadOpWs { float *w1t, *w2t, *aC, *r, *Zc, *w1a, *w1b, *bnid, *cvec, *ppart; unsigned int* xmax; int64_t off[4], pstride; size_t bytes; };
static HeadOpWs head_op_carve(int H, int N, void* base) {
  HeadOpWs w;
  char* p = (char*)base;
  size_t o = 0;
  auto take = [&](size_t nfloats) { float* r = (float*)(p + o); o += al(nfloats * sizeof(float)); return r; };
  w.w1t = take((size_t)2 * H * H); w.w2t = take((size_t)H * H); w.aC = take((size_t)N * H); w.r = take((size_t)N * H);
  w.Zc = take((size_t)N * H); w.w1a = take((size_t)H * H); w.w1b = take((size_t)H * H); w.bnid = take(4 * H); w.cvec = take(2 * H);
  w.off[0] = 0; w.off[1] = (int64_t)2 * H * H; w.off[2] = w.off[1] + H; w.off[3] = w.off[2] + (int64_t)H * H;   // W1 b1 W2 b2
  w.pstride = w.off[3] + H;
  w.ppart = take((size_t)num_sms() * w.pstride);
  w.xmax = (unsigned int*)take(4);
  w.bytes = o;
  return w;
}
}  // namespace scgib

extern "C" SCGIB_API size_t scgib_head_mlp_workspace_bytes(int32_t hidden, int32_t N) {
  if (!hidden_ok(hidden) || N < 1) return 0;
  return head_op_carve(hidden, N, nullptr).bytes;
}

extern "C" SCGIB_API int scgib_head_mlp_fwd_f32(const float* noisy, const float* C, const float* alpha, int32_t N, int32_t hidden,
                                      const float* W1, const float* b1, const float* W2, const float* b2, float* interaction_map,
                                      float* Z, void* workspace, size_t workspace_bytes, void* stream_) {
  if (!noisy || !C || !alpha || !W1 || !b1 || !W2 || !b2 || !Z || !workspace) return SCGIB_E_NULL;
  if (!hidden_ok(hidden)) return SCGIB_E_SHAPE;
  if (N < 1) return SCGIB_E_RANGE;
  if (((uintptr_t)workspace & 255u) || ((uintptr_t)noisy & 15u) || ((uintptr_t)C & 15u) || ((uintptr_t)Z & 15u)) return SCGIB_E_ALIGN;
  const HeadOpWs w = head_op_carve(hidden, N, workspace);
  if (workspace_bytes < w.bytes) return SCGIB_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream_;
  const int H = hidden;
  TransposeJobs jobs;
  jobs.n = 2;
  jobs.job[0] = TransposeJob{W1, w.w1t, H, 2 * H};
  jobs.job[1] = TransposeJob{W2, w.w2t, H, H};
  launch_transposes(jobs, s);
  HeadFwdArgs a{noisy, C, alpha, N, w.w1t, b1, w.w2t, b2, interaction_map, w.aC, w.r, w.Zc};
  a.W1n = W1; a.W2n = W2;
  if (H == 64) {      // any input magnitude (GraphSAGE / GCN features are unbounded): the tensor-core head's power-of-two pre-scale
    cudaMemsetAsync(w.xmax, 0, 3 * sizeof(unsigned int), s);
    launch_absmax(noisy, (size_t)N * H, w.xmax, s);
    launch_absmax(C, (size_t)N * H, w.xmax + 1, s);
    launch_absmax(alpha, (size_t)N, w.xmax + 2, s);
    a.xmax = w.xmax;
  }
  launch_head_fwd(a, H, s);
  cudaMemcpyAsync(Z, w.Zc, (size_t)N * H * sizeof(float), cudaMemcpyDeviceToDevice, s);
  return (int)cudaGetLastError();
}

// gI [N, 2H] = d<gZ, Z>/d interaction_map (first half: noisy, second half: alpha C); call after the forward with the same workspace
extern "C" SCGIB_API int scgib_head_mlp_bwd_f32(const float* gZ, const float* noisy, int32_t N, int32_t hidden, const float* W1,
                                      const float* W2, float* gI, float* dW1, float* db1, float* dW2, float* db2, void* workspace,
                                      size_t workspace_bytes, void* stream_) {
  if (!gZ || !noisy || !W1 || !W2 || !gI || !dW1 || !db1 || !dW2 || !db2 || !workspace) return SCGIB_E_NULL;
  if (!hidden_ok(hidden)) return SCGIB_E_SHAPE;
  if (N < 1) return SCGIB_E_RANGE;
  if (((uintptr_t)workspace & 255u) || ((uintptr_t)gZ & 15u) || ((uintptr_t)gI & 15u)) return SCGIB_E_ALIGN;
  const HeadOpWs w = head_op_carve(hidden, N, workspace);
  if (workspace_bytes < w.bytes) return SCGIB_E_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream_;
  const int H = hidden, GP = num_sms();
  const bool tc = H == 64 && bwd_tensor_core_mode() != 0;
  launch_head_bwd_prep(W1, w.w1a, w.w1b, w.bnid, w.cvec, H, s);
  // the GIN backward kernel on the two K = H halves of the first layer (identity BatchNorm backward: g_y = gZ; its `y` operand
  // only enters multiplied by zero).  gI is returned as two dense halves [2][N][H]: gradient wrt noisy, then wrt alpha C.
  GinBwdMainArgs m[2];
  for (int h = 0; h < 2; ++h) {
    m[h].g_o = gZ; m[h].y = gZ; m[h].r = w.r; m[h].a = h == 0 ? noisy : w.aC;
    m[h].bn = w.bnid; m[h].cvec = w.cvec; m[h].W1 = h == 0 ? w.w1a : w.w1b; m[h].W2 = W2; m[h].V = N;
    m[h].g_a = gI + (size_t)h * N * H;
    m[h].part = w.ppart; m[h].pstride = w.pstride;
    m[h].off_W1 = w.off[0] + (int64_t)h * H * H; m[h].off_b1 = w.off[1]; m[h].off_W2 = w.off[2]; m[h].off_b2 = w.off[3];
  }
  int split = GP;
  if (tc) {
    launch_gin_bwd_main_tc2_pair(m[0], m[1], H, GP, s, true);
    split = pair_split(GP, (N + 127) / 128, (N + 127) / 128);
  } else {
    launch_gin_bwd_main(m[0], H, H, GP, s);
    launch_gin_bwd_main(m[1], H, H, GP, s);
  }
  ReduceRanges rr;
  rr.n = 0;
  auto add = [&](int64_t off, int64_t len, int c0, int c1) { rr.off[rr.n] = off; rr.len[rr.n] = len; rr.c0[rr.n] = c0; rr.c1[rr.n] = c1; ++rr.n; };
  add(w.off[0], (int64_t)H * H, 0, split);
  add(w.off[0] + (int64_t)H * H, (int64_t)H * H, tc ? split : 0, GP);
  launch_reduce_partials(w.ppart, w.pstride, GP, rr, dW1 - w.off[0], s);
  launch_head_dw1_interleave(dW1, H, s);
  float* outs[3] = {db1, dW2, db2};
  const int64_t lens[3] = {H, (int64_t)H * H, H};
  for (int i = 0; i < 3; ++i) {
    ReduceRanges r1;
    r1.n = 1; r1.off[0] = w.off[i + 1]; r1.len[0] = lens[i]; r1.c0[0] = 0; r1.c1[0] = split;
    launch_reduce_partials(w.ppart, w.pstride, GP, r1, outs[i] - w.off[i + 1], s);
  }
  return (int)cudaGetLastError();
}

// ---------------------------------------------------------------- debugging aid
// Byte offset of a named workspace buffer (tests compare intermediates with the oracle); -1 if unknown.
extern "C" SCGIB_API int64_t scgib_pretrain_workspace_offset(const ScgibDims* d, int32_t B, int32_t N, int32_t E,
                                                             int32_t Ns, int32_t Es, const char* name) {
  if (!dims_ok(d) || !name) return -1;
  const Layout lo = make_layout(d);
  const Ws w = carve(d, lo, B, N, E, Ns, Es, nullptr);
  struct { const char* n; const void* p; } tab[] = {
      {"t", w.t}, {"H", w.H}, {"q", w.q}, {"C", w.C}, {"logit", w.logit}, {"alpha", w.alpha}, {"lam", w.lam},
      {"noisy", w.noisy}, {"Z", w.Z}, {"r_head", w.r_head}, {"readout", w.readout}, {"core", w.core}, {"gstat", w.gstat},
      {"kl", w.kl}, {"G", w.G}, {"edge", w.edge}, {"z1", w.z1}, {"z2", w.z2}, {"D", w.D}, {"diag", w.diag},
      {"g_core", w.g_core}, {"g_readout", w.g_readout}, {"gZ", w.gZ}, {"gI", w.gI}, {"gp", w.gp}, {"g_q", w.g_q},
      {"gH", w.gH}, {"gC", w.gC}, {"ga0_1", w.ga0[0]}, {"ga0_2", w.ga0[1]}, {"cvec", w.cvec[0]}};
  for (auto& e : tab)
    if (!strcmp(e.n, name)) return (int64_t)((const char*)e.p - (const char*)nullptr);
  int e = 0, l = 0;
  char kind = 0;
  if (sscanf(name, "%c%d_%d", &kind, &e, &l) == 3 && (e == 1 || e == 2) && l >= 0 && l < d->gin_layers) {
    const void* p = kind == 'y' ? w.y[e - 1][l] : kind == 'a' ? w.a[e - 1][l] : kind == 'r' ? w.r[e - 1][l]
                    : kind == 'b' ? w.bn[e - 1][l] : nullptr;
    if (p) return (int64_t)((const char*)p - (const char*)nullptr);
  }
  return -1;
}

// ---------------------------------------------------------------- per-launch timing (bench.py)
extern "C" SCGIB_API void scgib_profile_enable(int on) { g_prof.on = on != 0; g_prof.n = 0; }
extern "C" SCGIB_API int scgib_profile_count(void) { return g_prof.n; }
// Name and elapsed milliseconds of recorded launch i (the caller has synchronised the stream).
extern "C" SCGIB_API int scgib_profile_get(int i, const char** name, float* ms) {
  if (i < 0 || i >= g_prof.n || !name || !ms) return SCGIB_E_RANGE;
  *name = g_prof.name[i];
  return (int)cudaEventElapsedTime(ms, g_prof.ev[2 * i], g_prof.ev[2 * i + 1]);
}

// scgib_private.h: select the GIN implementation (1 = tcgen05, 0 = FP32 FFMA cross-check; < 0: back to the default)
extern "C" SCGIB_API void scgib_set_tensor_cores_bwd(int mode) { g_bwd_tc = (mode == 0 || mode == 1) ? mode : -1; }
extern "C" SCGIB_API void scgib_set_tensor_cores(int mode) { g_use_tc = (mode == 0 || mode == 1) ? mode : -1; }
