// kernels.cuh - argument blocks and host launchers shared by the .cu files of libscgib.
#pragma once
#include "common.cuh"

namespace scgib {

int num_sms();

// ---------------------------------------------------------------- gin_kernels.cu
struct TransposeJob { const float* src; float* dst; int rows, cols; };  // dst[c][r] = src[r][c]
struct TransposeJobs { TransposeJob job[24]; int n; };
void launch_transposes(const TransposeJobs& jobs, cudaStream_t s);

// eval mode (model.eval()): bn = {running_mean, 1/sqrt(running_var + eps), gamma, beta} replaces the batch statistics a
// GIN forward kernel has just written, before the next layer / the pooling kernels read them
void launch_bn_from_running(const float* running, const float* gamma, const float* beta, float* bn, int hidden, cudaStream_t s);
void launch_input_proj_fwd(const float* x, const float* Wt, int N, int F, int normalize, float* t, cudaStream_t s, bool out_bf16 = false);
void launch_f32_to_bf16(const float* in, void* out, size_t n, cudaStream_t s);
// input projection + weight transposes + head-backward operand preparation in one launch (any part optional:
// x == nullptr, jobs.n == 0, headW1 == nullptr)
struct FwdPrepArgs {
  TransposeJobs jobs;
  const float* headW1 = nullptr; float *W1a = nullptr, *W1b = nullptr, *bn = nullptr, *cvec = nullptr; int hid = 64;
  const float* x = nullptr; const float* Wt = nullptr; int N = 0, F = 0, normalize = 0; float* t = nullptr;
  // aggregated normalised features xagg_v = x_hat[p(v)] + sum_{u in N(v)} x_hat[p(u)] of the parent rows and the ego rows
  // (a constant of the batch: the transfer_d backward contracts the layer-0 input gradient with it, input_proj_bwd)
  const int32_t* xa_indptr[2] = {nullptr, nullptr}; const int32_t* xa_indices[2] = {nullptr, nullptr};
  const float* xa_x = nullptr; const int32_t* xa_map = nullptr; int xa_V[2] = {0, 0}; float* xagg[2] = {nullptr, nullptr}; int xa_stride = 0;
  int nproj = 0, nxagg = 0;            // set by the launcher
};
void launch_fwd_prep(FwdPrepArgs a, cudaStream_t s, bool out_bf16);

struct GinFwdArgs {
  const float* in;          // [*, KIN]  t (layer 0) or the previous layer's pre-BN output y
  const int32_t* row_map;   // optional: input row of output row j (ego batch layer 0: ego_nodes)
  const float* bn_in;       // optional {mean, rstd, gamma, beta}[HID] of the producing layer
  const int32_t* indptr;
  const int32_t* indices;
  int V;
  const float *W1t, *b1, *W2t, *b2;   // W1t [KIN][HID], W2t [HID][HID]  (k-major copies, FFMA kernel)
  const float *W1, *W2;               // natural [out][in] (tensor-core kernel: K-major B operand)
  const float *gamma, *beta;          // this layer's BN affine (copied into bn_out for the consumers)
  float *a_out, *r_out, *y_out;       // a/r optional (saved for backward)
  float* part;                        // [n_tiles][2][HID]
  unsigned int* counter;
  float* bn_out;                      // {mean, rstd, gamma, beta}[HID]
  float* running;                     // optional {running_mean, running_var}[HID]
  int reverse = 0;                    // gin_tc3: walk the row tiles in descending order (alternate layers: the rows the
                                      //  previous layer wrote last are still in L2)
  int dbg = 0;                        // gin_tc2 experiments (SCGIB_DBG bit mask): 1 no r/y stores, 2 no stats, 4 no gather loads, 8 no a store
};
// Two independent problems of the same shape class (the same layer of Encoder1 and Encoder2) in ONE launch: CTAs
// [0, split) work on a[0], CTAs [split, grid) on a[1]; split is chosen proportional to the tile counts, so the 148
// persistent CTAs are balanced over both row sets and the per-launch fixed costs are paid once.
struct GinFwdPair { GinFwdArgs a[2]; int split; };
int gin_fwd_grid(int V);
void launch_gin_fwd(const GinFwdArgs& a, int kin, int hidden, cudaStream_t s);        // FP32 FFMA tiles (gin_kernels.cu), hidden 64 / 128
void launch_gin_fwd_tc3(const GinFwdArgs& a, int kin, cudaStream_t s);              // tcgen05 3xTF32, shared-memory window gather (gin_tc3.cu)
void launch_gin_fwd_tc3_pair(const GinFwdArgs& a0, const GinFwdArgs& a1, int kin, cudaStream_t s);
void launch_gin_fwd_tc4(const GinFwdArgs& a, cudaStream_t s);                       // tcgen05, aggregation on the tensor cores too (gin_tc4.cu); KIN = 64
void launch_gin_fwd_tc4_pair(const GinFwdArgs& a0, const GinFwdArgs& a1, cudaStream_t s);
int fwd_tc4_mode();                                                       // SCGIB_FWD4: 1 = gin_tc4.cu for the KIN = 64 layers
// bf16 mode (gin_bf16.cu, gin_bwd_bf16.cu): the float* activation fields of the argument blocks point to bf16 data
size_t gin_fwd_bf16_part_floats(int hidden);
void launch_gin_fwd_bf16(const GinFwdArgs& a0, const GinFwdArgs* a1, int kin, int hidden, cudaStream_t s);
int tensor_core_mode();                                                   // SCGIB_TC: 1 gin_tc3.cu (default), 0 FFMA cross-check
inline bool use_tensor_cores() { return tensor_core_mode() != 0; }

struct GinBwdPreArgs {
  const float* src;         // CSR mode: Ga [V][HID]; direct mode: rows gathered through map
  const int32_t* indptr;    // non-null => CSR mode
  const int32_t* indices;
  const int32_t* map;       // direct mode only, optional
  const float* y;           // [V][HID] this layer's pre-BN output
  const float* bn;          // {mean, rstd, gamma, beta}
  int V;
  float* g_o;               // [V][HID]
  float* part;              // [grid][2][HID]
  unsigned int* counter;
  float *d_gamma, *d_beta;  // [HID] final gradients
  float* cvec;              // {c1, c2}[HID]
  unsigned int* gmax = nullptr;   // optional: atomicMax of the bits of max |g_o| (zeroed by the caller): gradient scale of gin_bwd_h
};
struct GinBwdPrePair { GinBwdPreArgs a[2]; int split; };
int gin_bwd_pre_grid(int V);
int gin_bwd_pre_occ();          // resident CTAs per SM of the gather kernels (SCGIB_PRE_OCC)
void launch_gin_bwd_pre(const GinBwdPreArgs& a, int hidden, cudaStream_t s);
void launch_gin_bwd_pre_pair(const GinBwdPreArgs& a0, const GinBwdPreArgs& a1, int hidden, cudaStream_t s);   // grid = gin_bwd_pre_grid(V0 + V1)
int pair_split(int grid, int work0, int work1);     // CTAs given to problem 0

struct GinBwdMainArgs {
  const float *g_o, *y, *r, *a;
  const float *bn, *cvec;
  const float *W1, *W2;     // natural [out][in]
  int V;
  float* g_a;               // [V][KIN]
  float* part;              // per-CTA partial gradients: part[cta * pstride + off_*]
  int64_t pstride;
  int64_t off_W1, off_b1, off_W2, off_b2;
  const unsigned int* gmax = nullptr;   // gin_bwd_h: bits of max |g_o| (left by the kernel that produced g_o)
};
void launch_gin_bwd_main(const GinBwdMainArgs& a, int kin, int hidden, int grid, cudaStream_t s);      // FP32 FFMA tiles, hidden 64 / 128
struct GinBwdMainPair {
  GinBwdMainArgs a[2]; int split; int trace; int reverse = 0;
  int kin = HID;            // gin_bwd_h: input width of the layer (32 | 64)
  int half = 0;             // gin_bwd_h: one linear layer only (G1 / G3; g_a rows += g_r)
  int wait_first = 0;       // PDL: W1 / W2 are written by the kernel launched right before this one (the head backward's de-interleaved
                            //  W1 halves): wait for it before staging the weights instead of after
};
void launch_gin_bwd_main_tc2(const GinBwdMainArgs& a, int kin, int grid, cudaStream_t s);  // tcgen05 3xTF32, 64-row double-buffered tiles (gin_bwd_tc2.cu)
void launch_gin_bwd_main_tc2_pair(const GinBwdMainArgs& a0, const GinBwdMainArgs& a1, int kin, int grid, cudaStream_t s,
                                  bool weights_from_prev_kernel = false);
int gin_bwd_pre_bf16_grid(int V, int hidden);
void launch_gin_bwd_pre_bf16(const GinBwdPreArgs& a0, const GinBwdPreArgs* a1, int hidden, cudaStream_t s);
void launch_gin_bwd_main_bf16(const GinBwdMainArgs& a0, const GinBwdMainArgs* a1, int kin, int hidden, int grid, cudaStream_t s,
                              bool ga_f32 = false);      // ga_f32: g_a is written as fp32 also for kin == hidden (head backward)
void launch_gin_bwd_main_h_pair(const GinBwdMainArgs& a0, const GinBwdMainArgs& a1, int kin, int grid, cudaStream_t s,
                                bool weights_from_prev_kernel = false);     // tcgen05, two-term fp16 splits, 128-row tiles (gin_bwd_h.cu); kin 32 | 64
void launch_gin_bwd_main_h(const GinBwdMainArgs& a, int kin, int grid, cudaStream_t s);   // single problem
void launch_linear_bwd_h(const float* g, const float* x, const float* W, int V, float* g_in, const float* bn_identity, const float* cvec_zero,
                         const unsigned int* gmax, float* part, int64_t pstride, int64_t off_W, int64_t off_b, int grid, cudaStream_t s);
void launch_absmax(const float* x, size_t n, unsigned int* slot, cudaStream_t s);   // atomicMax(slot, bits of max |x|)
int bwd_h_mode();                                                          // SCGIB_BWD_H: 1 (default) gin_bwd_h.cu for the KIN = 64 layers and the head
int bwd_tensor_core_mode();                                                                // SCGIB_TC_BWD: 1 gin_bwd_tc2.cu (default), 0 FFMA cross-check

struct InputProjBwdArgs {
  const float* ga[2];       // layer-0 input gradients of the two encoders, [V][DTR]
  const float* xagg[2];     // aggregated normalised features of the rows, [V][xa_stride] (fwd_prep)
  int xa_stride;
  int V[2];
  int F;
  float* part;              // [grid][DTR*32]
  unsigned int* counter;
  float* d_Wt;              // [DTR][F]
};
int input_proj_bwd_grid(int V0, int V1);
void launch_input_proj_bwd(const InputProjBwdArgs& a, cudaStream_t s);

// ---------------------------------------------------------------- encoder_ops.cu
// Y[V][O] = X[V][K] W^T + bias, W [O][K] (nn.Linear layout); K, O multiples of 32
void launch_linear_plain(const float* X, const float* W, const float* bias, int V, int K, int O, float* Y, cudaStream_t s);

// ---------------------------------------------------------------- head_kernels.cu
// H = relu(BN(y_last)) materialised; q = H Wc1^T + bc1   (compressor.0, models.py:590)
struct GateLinFwdArgs {
  const float* y; const float* bn; int N;   // y: fp32, or bf16 storage when y_bf16
  const float* Wc1t; const float* bc1;   // Wc1t [HID][HID] k-major
  float* H; float* q;
  bool y_bf16 = false;
  const float* Wc1n = nullptr;           // natural [HID][HID]: when set (hidden 64, fp32 y) the tensor-core kernel runs
};
void launch_gate_lin_fwd(const GateLinFwdArgs& a, int hidden, cudaStream_t s);

// gH += g_q Wc1 ; dWc1 = g_q^T H ; dbc1 = sum g_q     (persistent, per-CTA partials)
struct GateLinBwdArgs {
  const float* g_q; const float* H; int N;
  const float* Wc1;                      // natural
  float* gH;                             // in/out [N][HID]
  float* part; int64_t pstride; int64_t off_W, off_b;
};
void launch_gate_lin_bwd(const GateLinBwdArgs& a, int hidden, int grid, cudaStream_t s);

// C_v = sum_{j in ego(v)} relu(BN(y2_last_j)) ; logit_v = w_cand . C_v
struct EgoPoolFwdArgs {
  const float* y; const float* bn; const int32_t* ego_ptr; int N;
  const float* w_cand;                   // attn_layer.weight[0, HID:2*HID]
  float* C; float* logit;
  bool y_bf16 = false;                   // y is bf16 storage (bf16 mode)
};
void launch_ego_pool_fwd(const EgoPoolFwdArgs& a, int hidden, cudaStream_t s);

void launch_segment_sum(const float* in, const int32_t* seg_ptr, int S, const float* bn, float* out, int hidden, cudaStream_t s);

// Per-graph gate + attention softmax (warp per graph): models.py:595-604, 631-660, 738-748
struct GraphGateFwdArgs {
  const int32_t* graph_ptr; int B; int N;
  const float *H, *q;                    // [N][HID]
  const float *gamma_c, *beta_c, *wc2, *bc2;
  const float *gate_u, *feat_u;          // [N], [N][HID]
  const float* logit;                    // [N]
  float* noisy;                          // [N][HID]  Z^c
  float* lam;                            // [N]
  float* alpha;                          // [N]
  float* readout;                        // [B][HID]  R_g   (graph_features_readout)
  float* core;                           // [B][HID]  sum_v Z^c_v
  float* gstat;                          // [B][4][HID] mu_g, sigma_g, mu^c_g, rstd^c_g (saved)
  const float* eval_running;             // optional {running_mean, running_var}[HID] of the compressor BatchNorm: eval mode
                                         //  (normalise with the running statistics instead of the per-graph ones)
  float* cstat;                          // optional [B][2][HID] compressor-BN batch mean / unbiased var per graph
  float* kl;                             // [1] KL loss (last graph)
  bf16_t* noisy_bf = nullptr;            // optional bf16 copy of noisy (bf16 mode: `a` operand of the head backward)
  // optional (z1 != nullptr): the contrastive loss' row normalisation fused into the per-graph warp (normalize_kernel's
  // outputs: z1 = core / max(||core||, 1e-12), z2 = readout / ..., norms, diag = z1 . z2, tf32 hi/lo copies)
  float *z1 = nullptr, *z2 = nullptr, *n1 = nullptr, *n2 = nullptr, *diag = nullptr, *zsplit = nullptr;
};
void launch_graph_gate_fwd(const GraphGateFwdArgs& a, int hidden, cudaStream_t s);

// compressor BatchNorm running stats: B sequential EMA updates in closed form (models.py:642 per graph)
void launch_compressor_ema(const float* cstat, int B, float* running, int hidden, cudaStream_t s);

struct GraphGateBwdArgs {
  const int32_t* graph_ptr; int B; int N;
  const float *H, *q, *C;                // saved
  const float *gamma_c, *beta_c, *wc2;
  const float* w_cand;
  const float *feat_u, *lam, *alpha, *gstat;
  const float* gI;                       // gradient wrt the noisy half of interaction_map, row stride gI_stride
  const float* gI2;                      // gradient wrt the alpha*C half, row stride gI_stride  (interleaved [N][2*HID]
  int gI_stride;                         //  from the FFMA head backward: gI2 = gI + HID, stride 2*HID; dense halves: HID)
  const float* g_core;                   // [B][HID]  contrastive gradient wrt core readout
  const float* g_readout;                // [B][HID]  contrastive gradient wrt graph readout
  float kl_scale;                        // d total / d KL
  float* gp;                             // [N] scratch
  float* g_q;                            // [N][HID]
  float* gH;                             // [N][HID]  direct part (lin backward adds g_q Wc1)
  float* gC;                             // [N][HID]
  float* part;                           // [grid][5*HID]: dgamma_c, dbeta_c, dwc2, dw_cand, (dbc2 at [4*HID])
  unsigned int* counter;
  float *d_gamma_c, *d_beta_c, *d_wc2, *d_bc2, *d_attn_w, *d_attn_b;   // final gradients
  unsigned int* gmax_q = nullptr;        // optional: atomicMax of the bits of max |g_q| (gradient scale of the tensor-core gate_lin backward)
  // optional (con_g1p != nullptr): contrastive_bwd_finalize fused into the per-graph warp - g_core / g_readout are formed
  // from the contrastive kernel's column-split partials [con_jsplit][B][HID] (g_core / g_readout above are then unused)
  const float *con_g1p = nullptr, *con_g2p = nullptr, *con_z1 = nullptr, *con_z2 = nullptr, *con_n1 = nullptr, *con_n2 = nullptr;
  int con_jsplit = 0; float con_scale = 0.f;
};
void launch_graph_gate_bwd(const GraphGateBwdArgs& a, int hidden, cudaStream_t s);

// Z = Wm2 relu(Wm1 [noisy || alpha*C] + bm1) + bm2       (models.py:676, 749)
struct HeadFwdArgs {
  const float *noisy, *C, *alpha; int N;
  const float *W1t, *b1, *W2t, *b2;      // W1t [2*HID][HID], W2t [HID][HID]
  float* imap;                           // optional [N][2*HID]
  float* aC;                             // optional [N][HID]: alpha*C, the second half of interaction_map (saved for the
                                         //  tensor-core head backward)
  float* r;                              // [N][HID] saved (optional)
  float* Z;                              // [N][HID]
  bf16_t* r_bf = nullptr;                // optional bf16 copies of r and alpha*C (bf16 mode: operands of the head backward)
  bf16_t* aC_bf = nullptr;
  bool in_bf16 = false;                         // head_tc.cu GATE mode only: `noisy` (= y) is bf16 storage
  const float* bn = nullptr;                    // head_tc.cu GATE mode only: {mean, rstd, gamma, beta}[HID] of the producing layer
  const float *W1n = nullptr, *W2n = nullptr;   // natural [HID][2*HID], [HID][HID]: when set (hidden 64, fp32 saves) the tensor-core
                                                //  kernel head_tc.cu runs instead of the FFMA tiles
  const unsigned int* xmax = nullptr;           // head_tc.cu: optional device slots {max |noisy|, max |C|, max |alpha|} (float bits,
                                                //  launch_absmax): inputs beyond 2^5 are pre-scaled by a power of two (see head_tc.cu)
};
void launch_head_fwd(const HeadFwdArgs& a, int hidden, cudaStream_t s);
void launch_head_fwd_tc(const HeadFwdArgs& a, cudaStream_t s);
void launch_gate_lin_fwd_tc(const GateLinFwdArgs& g, const float* Wc1, cudaStream_t s);   // compressor.0 forward on the same tensor-core pipeline

// Head backward = the GIN backward kernel run on the two K = H halves of the first head layer (api.cu).
// prep: dense copies W1a = W1[:, :HID], W1b = W1[:, HID:] and the identity BatchNorm-backward constants
// (bn = {0, 1, 1, 0}, cvec = 0: g_y = g_o).  fix: grads slot [2][HID][HID] (dW1a | dW1b) -> [HID][2*HID] in place.
void launch_head_bwd_prep(const float* W1, float* W1a, float* W1b, float* bn, float* cvec, int hidden, cudaStream_t s);
void launch_head_dw1_interleave(float* dW1, int hidden, cudaStream_t s);
void launch_identity_bn(float* bn, int hidden, cudaStream_t s);        // bn = {mean 0, rstd 1, gamma 1, beta 0}

// stand-alone attention / segment-broadcast operators (op-level C ABI)
void launch_attn_fwd(const float* C, const int32_t* graph_ptr, int B, int H, const float* w_cand, float* alpha, float* T, cudaStream_t s);
void launch_attn_bwd(const float* C, const float* alpha, const float* gT, const int32_t* graph_ptr, int B, int H, const float* w_cand,
                     float* gC, float* dwp, float* scratch, cudaStream_t s);
void launch_segment_sum_bwd(const float* g_out, const int32_t* seg_ptr, int S, int H, float* g_in, cudaStream_t s);
void launch_colsum_rows(const float* part, int R, int H, float* out, cudaStream_t s);

// ---------------------------------------------------------------- loss_kernels.cu
// recon: per-CTA partials of Z^T Z and of sum_{(i,j) in E} z_i . z_j     (models.py:762-768, Gram identity)
struct ReconFwdArgs {
  const float* Z; const int32_t* indptr; const int32_t* indices; int N;
  float* part;                           // [grid][HID*HID + 4]
};
void launch_recon_fwd(const ReconFwdArgs& a, int hidden, int grid, cudaStream_t s);
// G = sum of partials; edge = sum; one small kernel
void launch_recon_reduce(const float* part, int grid, float* G, float* edge_sum, int hidden, cudaStream_t s);
// gZ = scale * (4/N) * (Z G - A Z)
struct ReconBwdArgs {
  const float* Z; const float* G; const int32_t* indptr; const int32_t* indices; int N;
  float scale; float* gZ;
  unsigned int* gmax = nullptr;          // optional: atomicMax of the bits of max |gZ|
};
void launch_recon_bwd(const ReconBwdArgs& a, int hidden, cudaStream_t s);

// contrastive (models.py:606-629)
struct NormalizeArgs { const float *core, *readout; int B; float *z1, *z2, *n1, *n2, *diag; float* zsplit; };  // zsplit: optional [4][B][HID] tf32 hi/lo of z1, z2
void launch_normalize(const NormalizeArgs& a, int hidden, cudaStream_t s);
struct ContrastiveFwdArgs { const float *z1, *z2; int B; int jsplit; float* rowsum; const float* zsplit; };  // rowsum [jsplit][B]
void launch_contrastive_fwd(const ContrastiveFwdArgs& a, int hidden, cudaStream_t s);        // FP32 FFMA tiles (hidden 64 / 128)
void launch_contrastive_fwd_tc(const ContrastiveFwdArgs& a, cudaStream_t s);     // tcgen05 3xTF32 (contrastive_tc.cu)
struct ContrastiveBwdArgs {
  const float *z1, *z2, *D; int B; int jsplit;
  float* g1p; float* g2p;                // [jsplit][B][HID] partial gradients wrt z1_hat / z2_hat
};
void launch_contrastive_bwd(const ContrastiveBwdArgs& a, int hidden, cudaStream_t s);                          // FP32 FFMA tiles (hidden 64 / 128)
void launch_contrastive_bwd_tc(const ContrastiveBwdArgs& a, const float* zsplit, cudaStream_t s);   // tcgen05 (contrastive_tc.cu)
struct ContrastiveBwdFinArgs {
  const float *g1p, *g2p, *z1, *z2, *n1, *n2; int B; int jsplit; float scale;
  float *g_core, *g_readout;
};
void launch_contrastive_bwd_finalize(const ContrastiveBwdFinArgs& a, int hidden, cudaStream_t s);
int contrastive_jsplit(int B);

struct LossFinalizeArgs {
  const float* rowsum; int jsplit; const float* diag; int B;   // contrastive
  const float* G; const float* edge_sum; int N; int E;          // recon (adjacency)
  const float* recon_override;                                  // non-null: the recon loss was computed elsewhere (logM)
  const float* kl;
  float* D;                                                      // [B] contrastive denominators (saved)
  float* losses;                                                 // {KL, contrastive, recon, total}
  int hidden = HID;                                              // G is [hidden][hidden]
};
void launch_loss_finalize(const LossFinalizeArgs& a, cudaStream_t s);

// Horizontal fusion of the step's small serial jobs: the tcgen05 contrastive kernels run one CTA per SM on 128-row blocks
// and leave SMs idle (128 of 148 CTAs at B = 4096), so independent latency-bound jobs of the same phase ride along as
// EXTRA CTAs of those launches (side_jobs.cuh) instead of paying a launch + drain each:
//   forward : recon_reduce (n_reduce CTAs), compressor_ema (n_ema = 0 | 1 CTA), and loss_finalize run by whichever CTA
//             of the launch finishes last (`counter`, self-resetting);
//   backward: recon_bwd (n_recon CTAs walking all row tiles).
constexpr int kConSideCtas = 12;          // SMs contrastive_jsplit() leaves to the side jobs
struct ConFwdSides {
  const float* rpart = nullptr; int rgrid = 0; float* G = nullptr; float* edge = nullptr; int n_reduce = 0;
  const float* cstat = nullptr; float* running = nullptr; int n_ema = 0;
  int finalize = 0; LossFinalizeArgs fin; unsigned int* counter = nullptr;
};
struct ConBwdSides { int n_recon = 0; ReconBwdArgs recon; };
void launch_contrastive_fwd_tc_sides(const ContrastiveFwdArgs& a, const ConFwdSides& sides, cudaStream_t s);
void launch_contrastive_bwd_tc_sides(const ContrastiveBwdArgs& a, const float* zsplit, const ConBwdSides& sides, cudaStream_t s);

// grads[off..off+len) = sum_c part[c*pstride + off + i] for each listed range
// partial rows [c0, c1) hold the range; ilv > 0: element i of the range goes to dst + (i / ilv) * 2 * ilv + i % ilv instead of
// off + i (the head MLP's dW1 halves [2][H][H] -> [H][2H]: the former head_dw1_interleave kernel)
struct ReduceRanges { int64_t off[40]; int64_t len[40]; int c0[40]; int c1[40]; int64_t dst[40] = {}; int ilv[40] = {}; int n; };
void launch_reduce_partials(const float* part, int64_t pstride, int nparts, const ReduceRanges& r, float* grads,
                            cudaStream_t s);

void launch_adam(float* params, const float* grads, float* m, float* v, int64_t n, int64_t step, float lr, float b1,
                 float b2, float eps, float wd, float gscale, cudaStream_t s);

// ---------------------------------------------------------------- finetune_kernels.cu
// Fine-tuning head (Mainmodel_finetuning.forward, models.py:501-520): Set2Set(H, T iterations, 1 LSTM layer) -> predict MLP
// -> optional sigmoid, one kernel per direction; per-graph state saved in the caller's workspace.
struct FinetuneHeadFwdArgs {
  const float* Z; const int32_t* graph_ptr; int B, N, H, C, T, sigmoid;
  const float* WlstmT;                   // k-major [3H][4H] = [W_ih^T ; W_hh^T]
  const float *b_ih, *b_hh;              // [4H]
  const float* Wp1T; const float* bp1;   // k-major [2H][H], [H]
  const float* Wp2; const float* bp2;    // natural [C][H], [C]
  float *gates, *cst, *qstar, *alpha;    // saved: [T][B][4H] (activated i,f,g,o), [T][B][H], [T][B][2H], [T][N]
  float *rp, *scores;                    // [B][H] predict hidden (post-ReLU), [B][C]
};
void launch_finetune_head_fwd(const FinetuneHeadFwdArgs& a, cudaStream_t s);
struct FinetuneHeadBwdArgs {
  const float* Z; const int32_t* graph_ptr; int B, N, H, C, T, sigmoid;
  const float *Wih, *Whh, *Wp1, *Wp2;    // natural layouts
  const float *gates, *cst, *qstar, *alpha, *rp, *scores;
  const float* g_scores;                 // [B][C]  (unused when C == 0)
  const float* g_readout;                // optional [B][2H]: upstream gradient at the Set2Set output itself
  float *g_pre, *g_u, *dgates, *gp;      // [B][C], [B][H], [T][B][4H], [N] scratch
  float* gZ;                             // [N][H]
};
void launch_finetune_head_bwd(const FinetuneHeadBwdArgs& a, cudaStream_t s);
// out[m][n] = sum_r A[r][m] * Bm[r][n] (Bm == nullptr: column sums of A, Nn = 1); row splits are reduced in a fixed order
int atb_splits(int R);
void launch_atb(const float* A, int lda, const float* Bm, int ldb, float* out, int ldo, float* out2, int R, int M, int Nn,
                float* scratch, cudaStream_t s);
int finetune_max_classes();

// ---------------------------------------------------------------- logm_kernels.cu
// `--recons_type logM` (models.py:770-782 with util.py:60-91): per-graph Gram term + sparse k-hop pair term, no dense n x n.
// walks [k][N], gram [B], pair [N] are workspace; loss_out[0] = the loss; bwd OVERWRITES gZ with scale * d loss / d Z.
// Z is [N][hidden], hidden 64 or 128.
int logm_max_steps();
void launch_logm_fwd(const float* Z, const int32_t* graph_ptr, const int32_t* indptr, const int32_t* indices, int B, int N,
                     int k, float* walks, float* gram, float* pair, float* loss_out, int32_t* status, int hidden, cudaStream_t s);
void launch_logm_bwd(const float* Z, const int32_t* graph_ptr, const int32_t* indptr, const int32_t* indices, int B, int N,
                     int k, const float* walks, float scale, float* gZ, int32_t* status, int hidden, cudaStream_t s);

}  // namespace scgib
