/*
 * scgib.h - C ABI of libscgib.so: the B200 (sm_100a) implementation of the S-CGIB per-batch
 * pre-training hot path.
 *
 * The reference (O-JounLee/S-CGIB) has no FFI layer: its hot path is Python (models.py) calling
 * DGL 1.1.0 / PyTorch kernels.  Each entry point below replaces the reference call sites it
 * cites (file:line relative to the reference tree); INTEGRATION.md shows the ctypes binding a
 * maintainer adds on the reference side.
 *
 * Conventions
 *  - plain pointers and sizes only; every pointer is DEVICE memory unless marked (host).
 *  - the caller owns every buffer (inputs, outputs, workspace); the library never allocates or
 *    frees device memory and keeps no pointer after return.
 *  - fp32 tensors are row-major, contiguous, rows 16-byte aligned; index arrays are int32.
 *  - every function is asynchronous on `stream` (a cudaStream_t passed as void*), re-entrant
 *    and stateless.  No host synchronisation unless documented.
 *  - return value: 0 = ok; negative = SCGIB_E_* (argument/shape error, nothing launched);
 *    positive = cudaError_t of the failing launch.
 */
#ifndef SCGIB_H_
#define SCGIB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SCGIB_VERSION 100
#if defined(__GNUC__)
#define SCGIB_API __attribute__((visibility("default")))
#else
#define SCGIB_API
#endif

enum {
  SCGIB_OK = 0,
  SCGIB_E_NULL = -1,      /* required pointer is NULL */
  SCGIB_E_SHAPE = -2,     /* unsupported dimension (hidden must be 64 or 128, d_transfer 32 / 64 / 128 and <= hidden, 1 <= L <= 8, 1 <= F <= 128, fine-tuning head C <= 1024) */
  SCGIB_E_ALIGN = -3,     /* pointer not 16-byte aligned */
  SCGIB_E_WORKSPACE = -4, /* workspace too small */
  SCGIB_E_RANGE = -5,     /* size out of range (e.g. k < 1, graph with < 2 nodes) */
  SCGIB_E_ABI = -6,       /* ScgibBatch.struct_size != sizeof(ScgibBatch): caller built against another header */
};

SCGIB_API int scgib_version(void);
SCGIB_API const char* scgib_error_string(int code);
/* Number of SMs of the current device (host query, cached). */
SCGIB_API int scgib_num_sms(void);

/* ------------------------------------------------------------------------------------------
 * Model description.  Parameters live in ONE flat fp32 buffer (so the gradient all-reduce and
 * the optimiser touch a single tensor); scgib_param_layout gives the offset of every tensor.
 * State-dict names on the reference side are listed in INTEGRATION.md.
 * ------------------------------------------------------------------------------------------ */
typedef struct ScgibDims {
  int32_t in_dim;     /* F: raw feature width (9 PCQM4Mv2 / mol-PCBA, 11 QM9, 37 NCI1, 89 DD), 1 <= F <= 128  exp_pretraining.py:219 */
  int32_t d_transfer; /* DT: 32, 64 or 128, at most hidden (the layer-0 input width)  exp_pretraining.py:378 */
  int32_t hidden;     /* 64 or 128 (--dims)                                      exp_pretraining.py:390 */
  int32_t gin_layers; /* L: GINConv per encoder (4 in models.py:57-58)                               */
  int32_t act_dtype;  /* SCGIB_ACT_F32 (reference precision, 1e-5) or SCGIB_ACT_BF16: the GIN encoders keep their
                         activations (t, a, r, y and the layer gradients) in bf16 and run their MLPs as single-pass
                         bf16 tensor-core GEMMs with fp32 accumulation and fp32 / fp64 statistics (2e-2 tolerance);
                         parameters, gradients, optimiser state and everything the caller sees stay fp32 */
} ScgibDims;
enum { SCGIB_ACT_F32 = 0, SCGIB_ACT_BF16 = 1 };

/* Slots of the flat parameter buffer, in layout order.  Per-encoder/per-layer slots are
 * addressed as SCGIB_P_ENC + (enc * L + layer) * SCGIB_ENC_SLOTS + {W1,B1,W2,B2,GAMMA,BETA}. */
enum {
  SCGIB_ENC_W1 = 0, SCGIB_ENC_B1, SCGIB_ENC_W2, SCGIB_ENC_B2, SCGIB_ENC_GAMMA, SCGIB_ENC_BETA,
  SCGIB_ENC_SLOTS
};
enum {
  SCGIB_P_HEAD_W1 = 0, /* MLP.0.weight [H,2H]        models.py:569-572 */
  SCGIB_P_HEAD_B1,     /* MLP.0.bias   [H]                              */
  SCGIB_P_HEAD_W2,     /* MLP.2.weight [H,H]                            */
  SCGIB_P_HEAD_B2,     /* MLP.2.bias   [H]                              */
  SCGIB_P_COMP_W1,     /* compressor.0.weight [H,H]  models.py:589-593 */
  SCGIB_P_COMP_B1,     /* compressor.0.bias [H]                         */
  SCGIB_P_COMP_GAMMA,  /* compressor.1.weight [H]                       */
  SCGIB_P_COMP_BETA,   /* compressor.1.bias [H]                         */
  SCGIB_P_COMP_W2,     /* compressor.3.weight [1,H]                     */
  SCGIB_P_COMP_B2,     /* compressor.3.bias [1]                         */
  SCGIB_P_ATTN_W,      /* attn_layer.weight [1,2H]   models.py:562     */
  SCGIB_P_ATTN_B,      /* attn_layer.bias [1]                           */
  SCGIB_P_TRANSFER,    /* transfer_d.weight [DT,F]   models.py:559     */
  SCGIB_P_ENC,         /* first encoder slot; 2*L*SCGIB_ENC_SLOTS slots follow */
};
/* Number of slots for `d`; offsets[i], sizes[i] (in floats) for each slot; returns total floats
 * (each slot padded to a multiple of 4 floats).  (host) pointers; either may be NULL. */
SCGIB_API int64_t scgib_param_layout(const ScgibDims* d, int64_t* offsets, int64_t* sizes);
SCGIB_API int32_t scgib_param_slots(const ScgibDims* d);

/* One mini-batch: the batched parent graph (dgl.batch, molecules.py:359) and the flattened
 * batch of one k-hop ego-net per node (exp_pretraining.py:308-309), both as symmetric CSR. */
typedef struct ScgibBatch {
  int32_t struct_size;         /* = sizeof(ScgibBatch) (scgib_batch_abi_size()); checked on entry: SCGIB_E_ABI      */
  int32_t B, N, E;             /* graphs, nodes, directed edges of the parent batch            */
  int32_t Ns, Es;              /* rows / directed edges of the ego batch                        */
  const int32_t* graph_ptr;    /* [B+1] node offset of each graph   (batch_num_nodes)           */
  const int32_t* indptr;       /* [N+1]                                                         */
  const int32_t* indices;      /* [E]   global node ids, ascending per row                      */
  const int32_t* ego_ptr;      /* [N+1] ego-net v = rows ego_ptr[v]..ego_ptr[v+1]               */
  const int32_t* ego_nodes;    /* [Ns]  parent node of each ego row (ascending per ego-net)     */
  const int32_t* ego_seed;     /* [Ns]  seed node v of the ego-net each row belongs to          */
  const int32_t* sub_indptr;   /* [Ns+1]                                                        */
  const int32_t* sub_indices;  /* [Es]  ego-batch row ids                                       */
  const float* x;              /* [N,F] node features                                           */
  int32_t normalize_x;         /* 1: apply F.normalize(x) (exp_pretraining.py:312) inside; 0: x is used as given */
  const float* gate_u;         /* [N]   U[0,1) gate noise       (torch.rand,  models.py:599)    */
  const float* feat_u;         /* [N,H] U[0,1) feature noise    (rand_like,   models.py:650)    */
  const float* t_override;     /* optional [N,DT]: already-transferred features (the batch_x argument of
                                  extract_features, models.py:702); x / transfer_d are then not used (forward only) */
  int32_t eval_mode;           /* 1: model.eval() - every BatchNorm (GIN layers, compressor) normalises with the running
                                  statistics in `bn_running` (required, not updated); forward only (evaluate_network,
                                  train_pep_func.py:187-230).  0: training mode (batch statistics) */
  int32_t recon_logm_steps;    /* 0: recons_type 'adj' (models.py:762-768, the default).  k >= 1: recons_type 'logM'
                                  (models.py:770-782) with the k-step log transition matrices of util.py:60-91 computed
                                  on the fly from the CSR (k = --k_transition, <= 8); no pts/*_M_khop_k.pt files */
} ScgibBatch;

/* sizeof(ScgibBatch) of the library build: a binding fills ScgibBatch.struct_size with its own idea of the size. */
SCGIB_API int32_t scgib_batch_abi_size(void);

/* ------------------------------------------------------------------------------------------
 * k-hop ego-network extraction  (replaces dgl.khop_in_subgraph per node + dgl.batch:
 * exp_pretraining.py:271, 308-309; exp_pcqm4mv2.py:422,425).  Two phases around one
 * host-visible size read:
 *   1. scgib_ego_count : per-seed ball size and induced edge count, exclusive scans.
 *                        ego_ptr[N+1], ego_eptr[N+1] are written; ego_ptr[N] = Ns, ego_eptr[N] = Es.
 *   2. scgib_ego_fill  : node lists (bit-exact with the reference: ascending parent ids,
 *                        containing the seed), seed ids and the induced CSR.
 * status[0] is set non-zero if a ball exceeds SCGIB_EGO_CAP nodes (fill output is then invalid).
 * ------------------------------------------------------------------------------------------ */
#define SCGIB_EGO_CAP 128
SCGIB_API size_t scgib_ego_workspace_bytes(int32_t N);
SCGIB_API int scgib_ego_count(const int32_t* indptr, const int32_t* indices, int32_t N, int32_t k,
                    int32_t* ego_ptr, int32_t* ego_eptr, int32_t* status,
                    void* workspace, size_t workspace_bytes, void* stream);
SCGIB_API int scgib_ego_fill(const int32_t* indptr, const int32_t* indices, int32_t N, int32_t k,
                   const int32_t* ego_ptr, const int32_t* ego_eptr,
                   int32_t* ego_nodes, int32_t* ego_seed, int32_t* sub_indptr, int32_t* sub_indices,
                   void* stream);

/* ------------------------------------------------------------------------------------------
 * On-device batch assembly  (replaces DataLoader + MoleculeDataset.collate + dgl.batch: molecules.py:349-362,
 * exp_pretraining.py:283, 303-306, and the per-step H2D of the batch).  The packed dataset shard - every molecule of the
 * dataset as ONE symmetric CSR: mol_ptr[M+1] node offsets, ds_indptr[Nt+1], ds_indices[Et] (dataset-global node ids),
 * ds_x[Nt,F] - stays resident in HBM; a mini-batch is a device array of B molecule ids (any order, repeats allowed).
 * dgl.batch semantics: molecules in list order, node / edge ids offset.  Two phases around one host read of (N, E):
 *   1. count: graph_ptr[B+1], edge_ptr[B+1] (exclusive scans; graph_ptr[B] = N, edge_ptr[B] = E)
 *   2. fill : indptr[N+1], indices[E], x[N,F] of the batch.
 * ------------------------------------------------------------------------------------------ */
SCGIB_API size_t scgib_batch_workspace_bytes(int32_t B);
SCGIB_API int scgib_batch_assemble_count(const int32_t* mol_ptr, const int32_t* ds_indptr, const int32_t* ids, int32_t B,
                                         int32_t* graph_ptr, int32_t* edge_ptr, void* workspace, size_t workspace_bytes,
                                         void* stream);
SCGIB_API int scgib_batch_assemble_fill(const int32_t* mol_ptr, const int32_t* ds_indptr, const int32_t* ds_indices,
                                        const float* ds_x, int32_t F, const int32_t* ids, int32_t B,
                                        const int32_t* graph_ptr, const int32_t* edge_ptr, int32_t* indptr,
                                        int32_t* indices, float* x, void* stream);

/* Input validation on the device (failure detection; the reference's preprocessing swallows errors with bare `except:`,
 * exp_pretraining.py:276-278, and a 1-node graph surfaces as a BatchNorm ValueError / NaN std, models.py:642-647).
 * status[0] (device int32[2]) = 0 if the batch is well formed, else the smallest violated condition: 1 graph_ptr does not
 * cover [0,N); 2 indptr does not cover [0,E); 3 a graph with < 2 nodes; 4 indptr not monotone; 5 a neighbour outside the
 * node's own graph; 6 neighbours not strictly ascending (to_bidirected order, duplicate edges); 7 a self loop.
 * status[1] = an offending graph / node id. */
SCGIB_API int scgib_batch_validate(const int32_t* graph_ptr, const int32_t* indptr, const int32_t* indices, int32_t B,
                                   int32_t N, int32_t E, int32_t* status, void* stream);

/* ------------------------------------------------------------------------------------------
 * Whole pre-training step (Mainmodel.forward / Mainmodel_continue.forward, models.py:662-700,
 * 1158-1195, + loss.backward(), exp_pretraining.py:315-322).
 *
 * Workspace: one caller-owned device buffer of scgib_pretrain_workspace_bytes() bytes, 256-byte
 * aligned.  `forward` leaves the saved activations there; `backward` must be called with the
 * same workspace, batch and params before the next forward.
 *
 * outputs (device): losses[4] = {KL, contrastive, recon, KL+recon+contrastive};
 *   optional embeddings (NULL to skip): interaction_map [N,2H] (models.py:749), Z [N,H]
 *   (models.py:676), noisy [N,H], graph_readout [B,H] (models.py:716).
 * bn_running: [2*L+1][2][H] running_mean/running_var of Encoder1 BNs, Encoder2 BNs, compressor
 *   BN (in that order), updated in place like nn.BatchNorm1d(momentum 0.1) in train mode
 *   (NULL to skip).
 * ------------------------------------------------------------------------------------------ */
SCGIB_API size_t scgib_pretrain_workspace_bytes(const ScgibDims* d, int32_t B, int32_t N, int32_t E,
                                      int32_t Ns, int32_t Es);
SCGIB_API int scgib_pretrain_forward_f32(const ScgibDims* d, const float* params, float* bn_running,
                               const ScgibBatch* batch, float* losses,
                               float* interaction_map, float* Z, float* noisy, float* graph_readout,
                               void* workspace, size_t workspace_bytes, void* stream);
/* grads: flat buffer with the layout of `params`; every used slot is overwritten (not
 * accumulated); unused reference parameters are not part of the buffer.
 * loss_scale[3] (host): d(total)/d{KL, contrastive, recon}; the reference uses {1,1,1}. */
SCGIB_API int scgib_pretrain_backward_f32(const ScgibDims* d, const float* params, const ScgibBatch* batch,
                                const float* loss_scale, float* grads,
                                void* workspace, size_t workspace_bytes, void* stream);
/* Backward of the feature path only: gradients of <gZ, Z> with respect to every parameter, where Z = MLP(interaction_map)
 * is the output of scgib_pretrain_forward_f32 (its `Z` argument) and gZ [N, hidden] is the upstream gradient of whatever
 * head consumes Z - the fine-tuning models' Set2Set / predict head (Mainmodel_finetuning.forward, models.py:501-520;
 * autograd through model.extract_features + self.MLP).  Same workspace / grads contract as scgib_pretrain_backward_f32;
 * the pre-training losses contribute nothing. */
SCGIB_API int scgib_extract_backward_f32(const ScgibDims* d, const float* params, const ScgibBatch* batch,
                                         const float* gZ, float* grads, void* workspace, size_t workspace_bytes,
                                         void* stream);

/* Forward of the feature path only: everything scgib_pretrain_forward_f32 does up to Z = MLP(interaction_map), without
 * the pre-training losses - what Mainmodel_finetuning.forward runs before its readout (models.py:508-513:
 * transfer_d, model.extract_features, self.MLP).  Same workspace; pair with scgib_extract_backward_f32. */
SCGIB_API int scgib_extract_forward_f32(const ScgibDims* d, const float* params, float* bn_running,
                                        const ScgibBatch* batch, float* interaction_map, float* Z, float* noisy,
                                        float* graph_readout, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Fine-tuning head (Mainmodel_finetuning.forward, models.py:515-520): dgl.nn.Set2Set(H, n_iters = T, n_layers = 1)
 * readout of Z (models.py:365, 515; per iteration: q = LSTM(q*), e_v = z_v . q_g, alpha = softmax over the graph,
 * r_g = sum alpha_v z_v, q* = [q || r]) -> predict = Linear(2H,H)-ReLU-Linear(H,C) (models.py:386-397) -> sigmoid
 * (models.py:519-520; sigmoid = 0 for the regression datasets, models.py:516-517).  One kernel per direction.
 * head_params / head_grads: one flat fp32 buffer, slots below (scgib_finetune_head_layout gives offsets, each slot
 * padded to 4 floats).  H in {32, 64, 128}, 0 <= C <= 1024 (above 64 the output layer
 * runs as tiled kernels over [B x C]), T <= 8.  The forward leaves its saved state in `workspace`
 * (scgib_finetune_head_workspace_bytes, 256-byte aligned); the backward must get the same workspace and Z.
 *   fwd: scores [B,C]; optional readout [B,2H] (= q* after the last iteration, the Set2Set output).
 *   bwd: gZ [N,H] (overwritten) = d(<g_scores, scores> + <g_readout, readout>)/dZ; g_readout [B,2H] is optional;
 *        head_grads: every slot overwritten.
 * C = 0 is the bare Set2Set readout (no predict head; scores / g_scores unused, g_readout required): with H = 32 and
 * zero-padded weights and features it serves Set2Set over the raw node features (Mainmodel_domainadapt.s2s_rev,
 * models.py:114, 267 - padded hidden units have zero gates weights and stay exactly 0).
 * ------------------------------------------------------------------------------------------ */
enum {
  SCGIB_FT_LSTM_WIH = 0, /* s2s.lstm.weight_ih_l0 [4H,2H]  (gate order i,f,g,o) */
  SCGIB_FT_LSTM_WHH,     /* s2s.lstm.weight_hh_l0 [4H,H]  */
  SCGIB_FT_LSTM_BIH,     /* s2s.lstm.bias_ih_l0 [4H]      */
  SCGIB_FT_LSTM_BHH,     /* s2s.lstm.bias_hh_l0 [4H]      */
  SCGIB_FT_PRED_W1,      /* predict.0.weight [H,2H]       */
  SCGIB_FT_PRED_B1,      /* predict.0.bias [H]            */
  SCGIB_FT_PRED_W2,      /* predict.2.weight [C,H]        */
  SCGIB_FT_PRED_B2,      /* predict.2.bias [C]            */
  SCGIB_FT_SLOTS
};
SCGIB_API int64_t scgib_finetune_head_layout(int32_t H, int32_t C, int64_t* offsets, int64_t* sizes);
SCGIB_API size_t scgib_finetune_head_workspace_bytes(int32_t H, int32_t C, int32_t T, int32_t B, int32_t N);
SCGIB_API int scgib_finetune_head_fwd_f32(const float* head_params, int32_t H, int32_t C, int32_t T, int32_t sigmoid,
                                          const float* Z, const int32_t* graph_ptr, int32_t B, int32_t N, float* scores,
                                          float* readout, void* workspace, size_t workspace_bytes, void* stream);
SCGIB_API int scgib_finetune_head_bwd_f32(const float* head_params, int32_t H, int32_t C, int32_t T, int32_t sigmoid,
                                          const float* Z, const int32_t* graph_ptr, int32_t B, int32_t N,
                                          const float* scores, const float* g_scores, const float* g_readout, float* gZ,
                                          float* head_grads, void* workspace, size_t workspace_bytes, void* stream);

/* Adam with L2-in-gradient weight decay over one flat buffer (torch.optim.Adam(lr, weight_decay),
 * exp_pretraining.py:86,112,323).  step = 1-based step count; grad_scale multiplies the gradient
 * first (1/world_size after a sum all-reduce). */
SCGIB_API int scgib_adam_step_f32(float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                        int64_t n, int64_t step, float lr, float beta1, float beta2, float eps,
                        float weight_decay, float grad_scale, void* stream);

/* ------------------------------------------------------------------------------------------
 * Individual operators (what the autograd Functions of the drop-in modules call; also the
 * unit-test surface).  H = 64.
 * ------------------------------------------------------------------------------------------ */
/* F.normalize(x) then transfer_d (exp_pretraining.py:312-314, models.py:668): t[N,DT].  1 <= F <= 128, DT 32, 64 or 128. */
SCGIB_API int scgib_input_proj_fwd_f32(const float* x, const float* Wt, int32_t N, int32_t F, int32_t DT,
                             float* t, void* stream);

/* One GINConv + (deferred) BatchNorm layer (models.py:66-72; DGL GINConv sum, eps=0):
 *   a_v = f(in[map(v)]) + sum_{u in N(v)} f(in[map(u)]),  f = relu(BN_in(.)) or identity (bn_in NULL)
 *   y   = W2 relu(W1 a + b1) + b2          (pre-BN output, saved)
 * and the batch statistics of y over all V rows: bn_out = {mean[H], rstd[H]} (biased var, eps 1e-5).
 * bn_in = {mean[H], rstd[H], gamma[H], beta[H]} of the producing layer.  a_out/r_out (saved for
 * backward) may be NULL.  running = {running_mean[H], running_var[H]} or NULL.
 * workspace >= scgib_gin_workspace_bytes(V). */
SCGIB_API size_t scgib_gin_workspace_bytes(int32_t V);
SCGIB_API int scgib_gin_layer_fwd_f32(const float* in, int32_t kin, const int32_t* row_map, const float* bn_in,
                            const int32_t* indptr, const int32_t* indices, int32_t V,
                            const float* W1, const float* b1, const float* W2, const float* b2,
                            float* a_out, float* r_out, float* y_out, float* bn_out, float* running,
                            void* workspace, size_t workspace_bytes, void* stream);

/* Backward of one GINConv + BatchNorm(train) + ReLU layer (autograd through models.py:66-72), the per-layer unit of
 * scgib_pretrain_backward_f32:
 *   g_next : indptr == NULL: [V,H] gradient wrt the layer OUTPUT h' = relu(BN(y));
 *            indptr != NULL: [V,H] gradient wrt the NEXT layer's aggregated input, gathered here through the symmetric
 *            CSR (G_v = g_next[v] + sum_{u in N(v)} g_next[u]: the transpose of the GIN aggregation, no atomics);
 *   y, r, a: what scgib_gin_layer_fwd_f32 saved (pre-BN output, hidden relu(W1 a + b1), aggregated input);
 *   bn     : {mean, rstd, gamma, beta}[H] of this layer;
 *   outputs: g_a [V,kin] (gradient wrt the aggregated input a), dW1 [H,kin], db1 [H], dW2 [H,H], db2 [H], dgamma [H],
 *            dbeta [H] - all overwritten. */
SCGIB_API size_t scgib_gin_layer_bwd_workspace_bytes(int32_t V, int32_t kin);
SCGIB_API int scgib_gin_layer_bwd_f32(const float* g_next, const int32_t* indptr, const int32_t* indices, int32_t V,
                                      int32_t kin, const float* y, const float* r, const float* a, const float* bn,
                                      const float* W1, const float* W2, float* g_a, float* dW1, float* db1, float* dW2,
                                      float* db2, float* dgamma, float* dbeta, void* workspace, size_t workspace_bytes,
                                      void* stream);

/* The same layer in bf16 mode (the kernels of the fused step with SCGIB_ACT_BF16), hidden H = 64 (kin 32 or 64) or 128
 * (kin 32, 64 or 128); other shapes return SCGIB_E_SHAPE.  Activations are bf16 (16-byte aligned rows), weights, biases,
 * BatchNorm constants and weight gradients fp32.
 *  forward : in, a_out, r_out, y_out bf16; y is rounded once and bn_out holds the statistics of the rounded y.
 *            workspace >= scgib_gin_layer_fwd_bf16_workspace_bytes(V, H), 256-byte aligned.
 *  backward: g_next bf16 [V,H] with indptr (CSR mode), fp32 [V,H] without (gradient wrt the layer output); y, r, a bf16;
 *            g_a fp32 when ga_f32 != 0 or kin < H, else bf16.  workspace >= scgib_gin_layer_bwd_bf16_workspace_bytes. */
SCGIB_API size_t scgib_gin_layer_fwd_bf16_workspace_bytes(int32_t V, int32_t hidden);
SCGIB_API int scgib_gin_layer_fwd_bf16(const void* in, int32_t kin, int32_t hidden, const int32_t* row_map, const float* bn_in,
                                       const int32_t* indptr, const int32_t* indices, int32_t V,
                                       const float* W1, const float* b1, const float* W2, const float* b2,
                                       void* a_out, void* r_out, void* y_out, float* bn_out, float* running,
                                       void* workspace, size_t workspace_bytes, void* stream);
SCGIB_API size_t scgib_gin_layer_bwd_bf16_workspace_bytes(int32_t V, int32_t kin, int32_t hidden);
SCGIB_API int scgib_gin_layer_bwd_bf16(const void* g_next, const int32_t* indptr, const int32_t* indices, int32_t V,
                                       int32_t kin, int32_t hidden, int32_t ga_f32, const void* y, const void* r, const void* a,
                                       const float* bn, const float* W1, const float* W2, void* g_a, float* dW1, float* db1,
                                       float* dW2, float* db2, float* dgamma, float* dbeta, void* workspace,
                                       size_t workspace_bytes, void* stream);

/* Loss operators: value and gradient in one call (the units of the whole-step functions).  workspace >=
 * scgib_loss_workspace_bytes(B) (B = 1 for the reconstruction loss), 256-byte aligned; loss = device float[1].
 *  scgib_recon_adj_f32  : loss_recon_adj (models.py:762-768) = sum_{ij} (z_i . z_j - A_ij)^2 / N over the WHOLE batch
 *                         (cross-graph pairs included, as the reference does) through the Gram identity
 *                         ||Z^T Z||_F^2 - 2 sum_E z_i . z_j + E; gZ (optional) = scale * d loss / d Z = scale 4/N (Z G - A Z).
 *  scgib_contrastive_f32: batched_semi_loss (models.py:606-629, tau = 1, one chunk) of z1 = core readout, z2 = graph
 *                         readout ([B,H], un-normalised); g_core / g_readout (optional, both or none) = scale * gradients. */
SCGIB_API size_t scgib_loss_workspace_bytes(int32_t B);
SCGIB_API int scgib_recon_adj_f32(const float* Z, const int32_t* indptr, const int32_t* indices, int32_t N, int32_t E,
                                  float scale, float* loss, float* gZ, void* workspace, size_t workspace_bytes, void* stream);
SCGIB_API int scgib_contrastive_f32(const float* core, const float* readout, int32_t B, float scale, float* loss,
                                    float* g_core, float* g_readout, void* workspace, size_t workspace_bytes, void* stream);
/* the same operators at hidden = 64 or 128 (the entries above are the hidden-64 instances) */
SCGIB_API size_t scgib_loss_workspace_bytes_h(int32_t B, int32_t hidden);
SCGIB_API int scgib_recon_adj_h_f32(const float* Z, const int32_t* indptr, const int32_t* indices, int32_t N, int32_t E,
                                    int32_t hidden, float scale, float* loss, float* gZ, void* workspace, size_t workspace_bytes,
                                    void* stream);
SCGIB_API int scgib_contrastive_h_f32(const float* core, const float* readout, int32_t B, int32_t hidden, float scale, float* loss,
                                      float* g_core, float* g_readout, void* workspace, size_t workspace_bytes, void* stream);
/* loss_recon of --recons_type logM (models.py:770-782 with the k-step log transition matrices of util.py:60-91):
 *   loss = (1/k) sum_g sum_{i=1..k} || Z_g Z_g^T - logM_{g,i} ||_F^2 / n_g^2,   Z [N][hidden], hidden 64 or 128,
 * computed per graph (graph_ptr [B+1]) on the symmetric CSR without any dense n x n matrix.  gZ (optional) = scale * d loss / d Z.
 * status = device int32[1]: set to 0, then to 1 when a k-hop ball exceeds SCGIB_EGO_CAP nodes (its terms are then dropped).
 * workspace >= scgib_recon_logm_workspace_bytes(B, N, k), 256-byte aligned; Z / gZ 16-byte aligned.
 * Codes: hidden not 64 / 128 -> SCGIB_E_SHAPE; k outside [1, 8], B < 1 or N < 2 -> SCGIB_E_RANGE. */
SCGIB_API size_t scgib_recon_logm_workspace_bytes(int32_t B, int32_t N, int32_t k);
SCGIB_API int scgib_recon_logm_h_f32(const float* Z, const int32_t* graph_ptr, const int32_t* indptr, const int32_t* indices,
                                     int32_t B, int32_t N, int32_t hidden, int32_t k, float scale, float* loss, float* gZ,
                                     int32_t* status, void* workspace, size_t workspace_bytes, void* stream);

/* out[s] = sum_{rows in segment s} f(in[row])  (dgl.sum_nodes, models.py:716,725,733,684);
 * f = relu(BN(.)) when bn = {mean,rstd,gamma,beta} is given, identity otherwise. */
SCGIB_API int scgib_segment_sum_f32(const float* in, const int32_t* seg_ptr, int32_t S, const float* bn,
                          float* out, void* stream);

/* ------------------------------------------------------------------------------------------
 * Per-graph core gate, core-candidate attention, head MLP and the sum_nodes broadcast as individual operators (SURVEY 8b):
 * the units scgib_extract_forward/backward_f32 run fused.  hidden in {64, 128}.
 *
 *  scgib_core_gate_fwd/bwd_f32 : compress + compression (models.py:595-604, 631-660) on Hfeat = graph_features [N,H]
 *      (the Encoder1 output, any sign): q = compressor.0(H), per-graph BatchNorm (compressor.1, training mode), p = compressor.3(relu),
 *      lambda = sigmoid(logit(eps(gate_u)) + p), noisy = lambda H + (1 - lambda) mu_g + feat_u (1 - lambda) sigma_g,
 *      graph_readout = sum_nodes(H), core_readout = sum_nodes(noisy), kl = KL of the LAST graph (models.py:657-659).
 *      bwd: gradients of <g_noisy, noisy> + <g_core, core_readout> + <g_readout, graph_readout> + kl_scale * kl; call after
 *      the forward with the same workspace (scgib_core_gate_workspace_bytes, 256-byte aligned).
 *  scgib_core_cand_attn_fwd/bwd_f32 : the attention loop (models.py:738-748): alpha = per-graph softmax of
 *      attn_layer([core || C_v]); the core half and the bias cancel in the softmax, so only w_cand = attn_layer.weight[0, H:]
 *      enters (their gradients are exactly zero).  T = alpha C (optional).  bwd workspace: (N + B*hidden) floats + 256 bytes.
 *  scgib_head_mlp_fwd/bwd_f32 : self.MLP(interaction_map) (models.py:569-572, 676) with interaction_map = [noisy || alpha C];
 *      bwd returns gI as TWO dense halves [2][N][H] (gradient wrt noisy, then wrt alpha C) and the four parameter gradients.
 *  scgib_segment_sum_bwd_f32 : backward of dgl.sum_nodes: g_in[row] = g_out[segment(row)].
 * ------------------------------------------------------------------------------------------ */
SCGIB_API size_t scgib_core_gate_workspace_bytes(int32_t hidden, int32_t B, int32_t N);
SCGIB_API int scgib_core_gate_fwd_f32(const float* Hfeat, const int32_t* graph_ptr, int32_t B, int32_t N, int32_t hidden,
                                      const float* Wc1, const float* bc1, const float* gamma_c, const float* beta_c,
                                      const float* wc2, const float* bc2, const float* gate_u, const float* feat_u,
                                      float* noisy, float* lam, float* graph_readout, float* core_readout, float* kl,
                                      void* workspace, size_t workspace_bytes, void* stream);
/* model.eval() instance of scgib_core_gate_fwd_f32: compressor.1 normalises q with its running statistics
 * running = {mean[H], var[H]} (nn.BatchNorm1d in eval mode) instead of the per-graph batch statistics, and nothing is kept
 * for a backward or for scgib_core_gate_ema_f32 (forward only).  Same codes as scgib_core_gate_fwd_f32. */
SCGIB_API int scgib_core_gate_eval_fwd_f32(const float* Hfeat, const int32_t* graph_ptr, int32_t B, int32_t N, int32_t hidden,
                                           const float* Wc1, const float* bc1, const float* gamma_c, const float* beta_c,
                                           const float* wc2, const float* bc2, const float* running, const float* gate_u,
                                           const float* feat_u, float* noisy, float* lam, float* graph_readout,
                                           float* core_readout, float* kl, void* workspace, size_t workspace_bytes, void* stream);
/* running = {mean[H], var[H]} of compressor.1 after the B per-graph BatchNorm calls of the forward that filled `workspace`. */
SCGIB_API int scgib_core_gate_ema_f32(int32_t B, int32_t N, int32_t hidden, float* running, void* workspace,
                                      size_t workspace_bytes, void* stream);
SCGIB_API int scgib_core_gate_bwd_f32(const int32_t* graph_ptr, int32_t B, int32_t N, int32_t hidden, const float* Wc1,
                                      const float* gamma_c, const float* beta_c, const float* wc2, const float* feat_u,
                                      const float* g_noisy, const float* g_core, const float* g_readout, float kl_scale,
                                      float* gH, float* dWc1, float* dbc1, float* dgamma_c, float* dbeta_c, float* dwc2,
                                      float* dbc2, void* workspace, size_t workspace_bytes, void* stream);
SCGIB_API int scgib_core_cand_attn_fwd_f32(const float* C, const int32_t* graph_ptr, int32_t B, int32_t N, int32_t hidden,
                                           const float* w_cand, float* alpha, float* T, void* stream);
SCGIB_API int scgib_core_cand_attn_bwd_f32(const float* C, const float* alpha, const float* gT, const int32_t* graph_ptr,
                                           int32_t B, int32_t N, int32_t hidden, const float* w_cand, float* gC,
                                           float* dw_cand, void* workspace, size_t workspace_bytes, void* stream);
SCGIB_API size_t scgib_head_mlp_workspace_bytes(int32_t hidden, int32_t N);
SCGIB_API int scgib_head_mlp_fwd_f32(const float* noisy, const float* C, const float* alpha, int32_t N, int32_t hidden,
                                     const float* W1, const float* b1, const float* W2, const float* b2,
                                     float* interaction_map, float* Z, void* workspace, size_t workspace_bytes, void* stream);
SCGIB_API int scgib_head_mlp_bwd_f32(const float* gZ, const float* noisy, int32_t N, int32_t hidden, const float* W1,
                                     const float* W2, float* gI, float* dW1, float* db1, float* dW2, float* db2,
                                     void* workspace, size_t workspace_bytes, void* stream);
SCGIB_API int scgib_segment_sum_bwd_f32(const float* g_out, const int32_t* seg_ptr, int32_t S, int32_t hidden, float* g_in,
                                        void* stream);

/* ------------------------------------------------------------------------------------------
 * Building blocks of the --encoder GraphSAGE / GCN variants (models.py:75-104; csrc/encoder_ops.cu) and the transfer_d
 * backward as operators.  FP32 FFMA tiles; widths W, K, O in {32, 64, 128, 256} (multiples of 32).  The adjacency is
 * symmetric (molecular graphs and their induced ego-nets), so the backward of an aggregation is the same call with the two
 * degree normalisations exchanged.
 *
 *  scgib_graph_aggregate_f32 : out[v] = (add ? add[v] : 0) + fd(deg v) sum_{u in N(v)} fs(deg u) in[map(u)]
 *      norm codes: 0 = 1, 1 = 1 / max(deg, 1) (SAGEConv 'mean'), 2 = max(deg, 1)^-1/2 (GraphConv norm='both').
 *  scgib_segment_sum_w_f32   : dgl.sum_nodes at any supported width.
 *  scgib_linear_fwd_f32      : Y[V,O] = act(X0[map0] (.) (M0 > 0) W0 + X1 (.) (M1 > 0) W1 + bias); Wp is [O][Kp]
 *      (nn.Linear, wp_kxo = 0) or [Kp][O] (GraphConv weight / a transposed product, wp_kxo = 1); Mp optional ReLU masks
 *      (backward products g (.) (h > 0)); X1 NULL = one operand pair.
 *  scgib_linear_bwd_w_f32    : dW (+)= (G (.) (M > 0))^T X[map] as [O][K] (kxo = 0) or [K][O] (kxo = 1), db (+)= column sums;
 *      fixed-order two-stage reduction (bit-identical reruns).  O multiple of 64.  workspace 16-byte aligned.
 *  scgib_transfer_bwd_d_f32  : d transfer_d.weight [DT][F] = sum over two row sets of g_r (x) xrow_r, xrow_r = x_hat[p(r)]
 *      (+ the x_hat rows of r's neighbours when a CSR is given); g0 / g1 are [V][DT].  1 <= F <= 128, DT 32, 64 or 128.
 *      workspace 256-byte aligned, from scgib_transfer_bwd_workspace_bytes_d (0 for an unsupported DT).
 *  scgib_transfer_bwd_f32    : scgib_transfer_bwd_d_f32 at DT = 32 (and its workspace query).
 * ------------------------------------------------------------------------------------------ */
SCGIB_API int scgib_graph_aggregate_f32(const float* in, int32_t W, const int32_t* row_map, const int32_t* indptr,
                                        const int32_t* indices, int32_t V, int32_t src_norm, int32_t dst_norm,
                                        const float* add, float* out, void* stream);
SCGIB_API int scgib_segment_sum_w_f32(const float* in, const int32_t* seg_ptr, int32_t S, int32_t W, float* out, void* stream);
SCGIB_API int scgib_linear_fwd_f32(const float* X0, const float* M0, const int32_t* map0, const float* W0, int32_t K0,
                                   int32_t w0_kxo, const float* X1, const float* M1, const float* W1, int32_t K1,
                                   int32_t w1_kxo, const float* bias, int32_t relu, int32_t V, int32_t O, float* Y, void* stream);
SCGIB_API size_t scgib_linear_bwd_w_workspace_bytes(int32_t V, int32_t O, int32_t K);
SCGIB_API int scgib_linear_bwd_w_f32(const float* G, const float* M, const float* X, const int32_t* map, int32_t V, int32_t O,
                                     int32_t K, int32_t kxo, int32_t accumulate, float* dW, float* db, void* workspace,
                                     size_t workspace_bytes, void* stream);
SCGIB_API size_t scgib_transfer_bwd_workspace_bytes(int32_t V0, int32_t V1, int32_t F);
SCGIB_API int scgib_transfer_bwd_f32(const float* x, int32_t F, int32_t normalize, const float* g0, int32_t V0,
                                     const int32_t* indptr0, const int32_t* indices0, const float* g1, int32_t V1,
                                     const int32_t* indptr1, const int32_t* indices1, const int32_t* map1, float* dWt,
                                     void* workspace, size_t workspace_bytes, void* stream);
SCGIB_API size_t scgib_transfer_bwd_workspace_bytes_d(int32_t V0, int32_t V1, int32_t F, int32_t DT);
SCGIB_API int scgib_transfer_bwd_d_f32(const float* x, int32_t F, int32_t DT, int32_t normalize, const float* g0, int32_t V0,
                                       const int32_t* indptr0, const int32_t* indices0, const float* g1, int32_t V1,
                                       const int32_t* indptr1, const int32_t* indices1, const int32_t* map1, float* dWt,
                                       void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * The same building blocks in bf16 mode (--dtype bf16; csrc/encoder_bf16.cu): activations, masks and layer gradients are
 * bf16 storage (raw 16-bit words), weights / bias / dW / db fp32; every sum is fp32.  All data pointers 16-byte aligned
 * (SCGIB_E_ALIGN), widths in {32, 64, 128, 256} (SCGIB_E_SHAPE), V >= 1 (SCGIB_E_RANGE); checked before any launch.
 *
 *  scgib_input_proj_fwd_d_bf16 : scgib_input_proj_fwd_f32 with the [N][DT] output rounded to bf16, DT 32, 64 or 128.
 *  scgib_input_proj_fwd_bf16  : scgib_input_proj_fwd_d_bf16 at DT = 32 (any other DT: SCGIB_E_SHAPE).
 *  scgib_f32_to_bf16          : out = rnd(in), n a multiple of 8.
 *  scgib_graph_aggregate_bf16 : scgib_graph_aggregate_f32 on bf16 in / add; out bf16, or fp32 when out_f32.
 *  scgib_linear_fwd_bf16      : scgib_linear_fwd_f32 on bf16 Xp / Mp, single-pass tcgen05 MMAs with the weights rounded to
 *      bf16 and an fp32 accumulator; Y bf16, or fp32 when y_f32.  The weights and one 128-row tile per pair live in shared
 *      memory: a pair of wide operands beyond 227 KB (e.g. K0 = K1 = 256 at O = 256) is SCGIB_E_SHAPE.
 *  scgib_linear_bwd_w_bf16    : scgib_linear_bwd_w_f32 on bf16 G / M / X (O in {64, 128, 256}); the row contraction runs on
 *      tcgen05; workspace from scgib_linear_bwd_w_bf16_workspace_bytes.
 * ------------------------------------------------------------------------------------------ */
SCGIB_API int scgib_input_proj_fwd_bf16(const float* x, const float* Wt, int32_t N, int32_t F, int32_t DT, void* t, void* stream);
SCGIB_API int scgib_input_proj_fwd_d_bf16(const float* x, const float* Wt, int32_t N, int32_t F, int32_t DT, void* t, void* stream);
SCGIB_API int scgib_f32_to_bf16(const float* in, int64_t n, void* out, void* stream);
SCGIB_API int scgib_graph_aggregate_bf16(const void* in, int32_t W, const int32_t* row_map, const int32_t* indptr,
                                         const int32_t* indices, int32_t V, int32_t src_norm, int32_t dst_norm,
                                         const void* add, void* out, int32_t out_f32, void* stream);
SCGIB_API int scgib_linear_fwd_bf16(const void* X0, const void* M0, const int32_t* map0, const float* W0, int32_t K0,
                                    int32_t w0_kxo, const void* X1, const void* M1, const float* W1, int32_t K1,
                                    int32_t w1_kxo, const float* bias, int32_t relu, int32_t V, int32_t O, void* Y,
                                    int32_t y_f32, void* stream);
SCGIB_API size_t scgib_linear_bwd_w_bf16_workspace_bytes(int32_t V, int32_t O, int32_t K);
SCGIB_API int scgib_linear_bwd_w_bf16(const void* G, const void* M, const void* X, const int32_t* map, int32_t V, int32_t O,
                                      int32_t K, int32_t kxo, int32_t accumulate, float* dW, float* db, void* workspace,
                                      size_t workspace_bytes, void* stream);


/* Debugging aid: byte offset of a named intermediate inside the pre-training workspace ("t", "H", "q", "C",
 * "alpha", "lam", "y<enc>_<layer>", "gH", ...), -1 if unknown.  Tests compare intermediates with the oracle. */
SCGIB_API int64_t scgib_pretrain_workspace_offset(const ScgibDims* d, int32_t B, int32_t N, int32_t E, int32_t Ns,
                                                  int32_t Es, const char* name);

/* ------------------------------------------------------------------------------------------
 * Data parallelism: gradient all-reduce fused with Adam over NVLink peer memory (peer_kernels.cu).  Replaces
 * loss.backward()'s gradient exchange + optimizer.step() (exp_pretraining.py:321-323) for one process per GPU.
 *  scgib_peer_alloc  : cudaMalloc + zero a buffer and return its 64-byte CUDA IPC handle (the one place where the
 *                      library allocates: an IPC handle must name a whole allocation);
 *  scgib_peer_open   : map a peer process's buffer (handle exchanged by the host, e.g. torch.distributed);
 *  scgib_allreduce_adam_f32 : peer_grads[r] / peer_flags[r] (HOST arrays of device pointers, r < world <= 16) are rank
 *                      r's gradient buffer of this step's parity and its flag array (uint32[world], zero-initialised);
 *                      seq = 1, 2, ... is the step number, identical on every rank; gradients are double-buffered by
 *                      seq & 1 (see peer_kernels.cu).  Every rank applies the identical rank-ordered mean gradient.
 * ------------------------------------------------------------------------------------------ */
SCGIB_API int scgib_peer_alloc(size_t bytes, void** dev_ptr, unsigned char* handle64);
SCGIB_API int scgib_peer_open(const unsigned char* handle64, void** dev_ptr);
SCGIB_API int scgib_peer_close(void* dev_ptr);
SCGIB_API int scgib_peer_free(void* dev_ptr);
SCGIB_API int scgib_allreduce_adam_f32(float* params, float* exp_avg, float* exp_avg_sq, int64_t n,
                                       const void* const* peer_grads, const void* const* peer_flags, int32_t rank,
                                       int32_t world, uint32_t seq, int64_t step, float lr, float beta1, float beta2,
                                       float eps, float weight_decay, void* stream);

/* Per-launch timing with CUDA events recorded on the launching stream (used by bench.py for the roofline
 * numbers).  enable(1) clears the record; every later kernel launch of this library is bracketed by two events;
 * after synchronising the stream, profile_get(i) returns the static kernel-family name and the elapsed ms. */
SCGIB_API void scgib_profile_enable(int on);
SCGIB_API int scgib_profile_count(void);
SCGIB_API int scgib_profile_get(int i, const char** name, float* ms);

#ifdef __cplusplus
}
#endif
#endif /* SCGIB_H_ */
