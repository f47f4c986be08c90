"""Thin wrappers over the individual-operator entry points of the C ABI (unit-test surface and the
building blocks of the drop-in modules).  Every function requires CUDA tensors; nothing falls back to torch."""
from __future__ import annotations

import ctypes

import torch

from . import _lib

HID = 64


def _stream(t):
    return torch.cuda.current_stream(t.device).cuda_stream


def _cuda(*ts):
    for t in ts:
        if t is not None and t.device.type != "cuda":
            raise RuntimeError("scgib_b200 ops need CUDA tensors (no CPU fallback)")


def input_proj(x: torch.Tensor, Wt: torch.Tensor, out_dtype=torch.float32) -> torch.Tensor:
    """transfer_d(F.normalize(x))  (exp_pretraining.py:312, models.py:668): [N, d_transfer] with d_transfer = Wt.shape[0]
    (32, 64 or 128); ``out_dtype`` torch.bfloat16 rounds the output."""
    _cuda(x, Wt)
    x, Wt = x.contiguous().float(), Wt.contiguous().float()
    t = torch.empty(x.shape[0], Wt.shape[0], device=x.device, dtype=out_dtype)
    entry = _lib.load().scgib_input_proj_fwd_d_bf16 if out_dtype == torch.bfloat16 else _lib.load().scgib_input_proj_fwd_f32
    _lib.check(entry(_lib.ptr(x), _lib.ptr(Wt), x.shape[0], x.shape[1], Wt.shape[0], _lib.ptr(t), _stream(x)), "input_proj_fwd")
    return t


def to_bf16(t: torch.Tensor) -> torch.Tensor:
    """round an fp32 tensor (numel a multiple of 8) to bf16 on the device."""
    _cuda(t)
    t = _c32(t)
    out = torch.empty(t.shape, device=t.device, dtype=torch.bfloat16)
    _lib.check(_lib.load().scgib_f32_to_bf16(_lib.ptr(t), t.numel(), _lib.ptr(out), _stream(t)), "f32_to_bf16")
    return out


def gin_layer_fwd(h, indptr, indices, W1, b1, W2, b2, row_map=None, bn_in=None, running=None, save=False):
    """One GINConv + batch statistics (models.py:66-72).  Returns (y, bn{mean,rstd}[2,H], a, r), H = W1.shape[0].
    A torch.bfloat16 ``h`` runs the bf16-mode kernel (H 64 or 128): y, a, r bf16, bn the statistics of the rounded y."""
    _cuda(h, indptr, W1)
    lib = _lib.load()
    V = indptr.numel() - 1
    kin, H = h.shape[1], W1.shape[0]
    if h.dtype == torch.bfloat16:
        h = _b16(h)
        W1, b1, W2, b2 = _c32(W1), _c32(b1), _c32(W2), _c32(b2)
        y = torch.empty(V, H, device=h.device, dtype=torch.bfloat16)
        a = torch.empty(V, kin, device=h.device, dtype=torch.bfloat16) if save else None
        r = torch.empty(V, H, device=h.device, dtype=torch.bfloat16) if save else None
        bn_out = torch.zeros(4, H, device=h.device)
        ws = _ws(lib.scgib_gin_layer_fwd_bf16_workspace_bytes(V, H), h.device)
        off = (-ws.data_ptr()) % 256
        _lib.check(lib.scgib_gin_layer_fwd_bf16(_lib.ptr(h), kin, H, _lib.ptr(row_map), _lib.ptr(bn_in), _lib.ptr(indptr),
                                                _lib.ptr(indices), V, _lib.ptr(W1), _lib.ptr(b1), _lib.ptr(W2), _lib.ptr(b2),
                                                _lib.ptr(a), _lib.ptr(r), _lib.ptr(y), _lib.ptr(bn_out),
                                                _lib.ptr(running), ctypes.c_void_p(ws.data_ptr() + off), ws.numel() - off,
                                                _stream(h)), "gin_layer_fwd_bf16")
        return y, bn_out[:2], a, r
    if H != HID:
        raise ValueError("gin_layer_fwd: the fp32 layer entry is hidden %d (got %d)" % (HID, H))
    y = torch.empty(V, HID, device=h.device)
    a = torch.empty(V, kin, device=h.device) if save else None
    r = torch.empty(V, HID, device=h.device) if save else None
    bn_out = torch.zeros(4, HID, device=h.device)
    ws = torch.empty(lib.scgib_gin_workspace_bytes(V), dtype=torch.uint8, device=h.device)
    _lib.check(lib.scgib_gin_layer_fwd_f32(_lib.ptr(h.contiguous()), kin, _lib.ptr(row_map), _lib.ptr(bn_in),
                                           _lib.ptr(indptr), _lib.ptr(indices), V, _lib.ptr(W1.contiguous()),
                                           _lib.ptr(b1), _lib.ptr(W2.contiguous()), _lib.ptr(b2), _lib.ptr(a),
                                           _lib.ptr(r), _lib.ptr(y), _lib.ptr(bn_out), _lib.ptr(running), _lib.ptr(ws),
                                           ws.numel(), _stream(h)), "gin_layer_fwd")
    return y, bn_out[:2], a, r


def segment_sum(h, seg_ptr, bn=None):
    """dgl.sum_nodes (models.py:716, 725, 733, 684); optional fused relu(BN(.)) on load."""
    _cuda(h, seg_ptr)
    S = seg_ptr.numel() - 1
    out = torch.empty(S, HID, device=h.device)
    _lib.check(_lib.load().scgib_segment_sum_f32(_lib.ptr(h.contiguous()), _lib.ptr(seg_ptr), S, _lib.ptr(bn),
                                                 _lib.ptr(out), _stream(h)), "segment_sum")
    return out


def gin_layer_bwd(g_next, y, r, a, bn, W1, W2, indptr=None, indices=None, ga_f32=False):
    """Backward of one GINConv + BatchNorm(train) + ReLU layer.  ``g_next``: gradient wrt the layer output (``indptr`` None)
    or wrt the next layer's aggregated input (gathered through the CSR).  ``bn`` = [4,H] {mean, rstd, gamma, beta}, H = W1.shape[0].
    Returns (g_a, dW1, db1, dW2, db2, dgamma, dbeta).
    A torch.bfloat16 ``y`` runs the bf16-mode kernels: y, r, a bf16, g_next bf16 with ``indptr`` and fp32 without; g_a is fp32
    with ``ga_f32`` or a.shape[1] < H, else bf16."""
    _cuda(g_next, y, r, a, bn, W1, W2)
    lib = _lib.load()
    V, kin, dev = y.shape[0], a.shape[1], y.device
    H = W1.shape[0]
    if y.dtype == torch.bfloat16:
        y, r, a = _b16(y), _b16(r), _b16(a)
        g_next = _b16(g_next) if indptr is not None else _c32(g_next)
        bn, W1, W2 = _c32(bn), _c32(W1), _c32(W2)
        f32 = bool(ga_f32) or kin < H
        g_a = torch.empty(V, kin, device=dev, dtype=torch.float32 if f32 else torch.bfloat16)
        dW1, db1 = torch.empty(H, kin, device=dev), torch.empty(H, device=dev)
        dW2, db2 = torch.empty(H, H, device=dev), torch.empty(H, device=dev)
        dgamma, dbeta = torch.empty(H, device=dev), torch.empty(H, device=dev)
        ws = _ws(lib.scgib_gin_layer_bwd_bf16_workspace_bytes(V, kin, H), dev)
        off = (-ws.data_ptr()) % 256
        _lib.check(lib.scgib_gin_layer_bwd_bf16(_lib.ptr(g_next), _lib.ptr(indptr), _lib.ptr(indices), V, kin, H, int(f32),
                                                _lib.ptr(y), _lib.ptr(r), _lib.ptr(a), _lib.ptr(bn), _lib.ptr(W1), _lib.ptr(W2),
                                                _lib.ptr(g_a), _lib.ptr(dW1), _lib.ptr(db1), _lib.ptr(dW2),
                                                _lib.ptr(db2), _lib.ptr(dgamma), _lib.ptr(dbeta),
                                                ctypes.c_void_p(ws.data_ptr() + off), ws.numel() - off, _stream(y)),
                   "gin_layer_bwd_bf16")
        return g_a, dW1, db1, dW2, db2, dgamma, dbeta
    g_a = torch.empty(V, kin, device=dev)
    dW1, db1 = torch.empty(HID, kin, device=dev), torch.empty(HID, device=dev)
    dW2, db2 = torch.empty(HID, HID, device=dev), torch.empty(HID, device=dev)
    dgamma, dbeta = torch.empty(HID, device=dev), torch.empty(HID, device=dev)
    ws = torch.empty(lib.scgib_gin_layer_bwd_workspace_bytes(V, kin) + 256, dtype=torch.uint8, device=dev)
    _lib.check(lib.scgib_gin_layer_bwd_f32(_lib.ptr(g_next.contiguous()), _lib.ptr(indptr), _lib.ptr(indices), V, kin,
                                           _lib.ptr(y.contiguous()), _lib.ptr(r.contiguous()), _lib.ptr(a.contiguous()),
                                           _lib.ptr(bn.contiguous()), _lib.ptr(W1.contiguous()), _lib.ptr(W2.contiguous()),
                                           _lib.ptr(g_a), _lib.ptr(dW1), _lib.ptr(db1), _lib.ptr(dW2), _lib.ptr(db2),
                                           _lib.ptr(dgamma), _lib.ptr(dbeta), _lib.ptr(ws), ws.numel(), _stream(y)),
               "gin_layer_bwd")
    return g_a, dW1, db1, dW2, db2, dgamma, dbeta


def recon_adj(Z, indptr, indices, scale=1.0, want_grad=True):
    """loss_recon_adj (models.py:762-768) and scale * d loss / d Z; returns (loss[1], gZ or None)."""
    _cuda(Z, indptr)
    lib = _lib.load()
    Z = Z.contiguous().float()
    N, E = Z.shape[0], indices.numel()
    loss = torch.empty(1, device=Z.device)
    gZ = torch.empty_like(Z) if want_grad else None
    H = Z.shape[1]
    ws = torch.empty(lib.scgib_loss_workspace_bytes_h(1, H) + 256, dtype=torch.uint8, device=Z.device)
    _lib.check(lib.scgib_recon_adj_h_f32(_lib.ptr(Z), _lib.ptr(indptr), _lib.ptr(indices), N, E, H, float(scale), _lib.ptr(loss),
                                         _lib.ptr(gZ), _lib.ptr(ws), ws.numel(), _stream(Z)), "recon_adj")
    return loss, gZ


def recon_logm(Z, graph_ptr, indptr, indices, k, scale=1.0, want_grad=True):
    """loss_recon of --recons_type logM (models.py:770-782, k-step log transition matrices of util.py:60-91) and
    scale * d loss / d Z, hidden 64 or 128; returns (loss[1], gZ or None, status[1]).  status is 1 when a k-hop ball
    exceeded the ego-net capacity (its terms are dropped); it is left on the device (no host sync)."""
    _cuda(Z, graph_ptr, indptr, indices)
    lib = _lib.load()
    Z = _c32(Z)
    N, H, B = Z.shape[0], Z.shape[1], graph_ptr.numel() - 1
    loss = torch.empty(1, device=Z.device)
    status = torch.empty(1, dtype=torch.int32, device=Z.device)
    gZ = torch.empty_like(Z) if want_grad else None
    ws = _ws(lib.scgib_recon_logm_workspace_bytes(B, N, int(k)), Z.device)
    _lib.check(lib.scgib_recon_logm_h_f32(_lib.ptr(Z), _lib.ptr(graph_ptr), _lib.ptr(indptr), _lib.ptr(indices), B, N, H, int(k),
                                          float(scale), _lib.ptr(loss), _lib.ptr(gZ), _lib.ptr(status),
                                          _lib.ptr(ws), ws.numel(), _stream(Z)), "recon_logm")
    return loss, gZ, status


def contrastive(core, readout, scale=1.0, want_grad=True):
    """batched_semi_loss (models.py:606-629) of the core / graph readouts and its gradients; returns (loss[1], g_core, g_readout)."""
    _cuda(core, readout)
    lib = _lib.load()
    core, readout = core.contiguous().float(), readout.contiguous().float()
    B = core.shape[0]
    loss = torch.empty(1, device=core.device)
    g1 = torch.empty_like(core) if want_grad else None
    g2 = torch.empty_like(core) if want_grad else None
    H = core.shape[1]
    ws = torch.empty(lib.scgib_loss_workspace_bytes_h(B, H) + 256, dtype=torch.uint8, device=core.device)
    _lib.check(lib.scgib_contrastive_h_f32(_lib.ptr(core), _lib.ptr(readout), B, H, float(scale), _lib.ptr(loss), _lib.ptr(g1),
                                           _lib.ptr(g2), _lib.ptr(ws), ws.numel(), _stream(core)), "contrastive")
    return loss, g1, g2


def _c32(t):
    """contiguous fp32 view / copy (the kernels read raw pointers)."""
    return t.detach().contiguous().float()


def _ws(nbytes, dev):
    return torch.empty(int(nbytes) + 256, dtype=torch.uint8, device=dev)


class CoreGate:
    """compress + compression (models.py:595-604, 631-660) as one operator pair; ``forward`` keeps its saved state in a
    workspace that ``backward`` reuses (one forward, then its backward)."""

    def __init__(self, hidden, Wc1, bc1, gamma_c, beta_c, wc2, bc2):
        self.H = int(hidden)
        self.p = [t.contiguous().float() for t in (Wc1, bc1, gamma_c, beta_c, wc2, bc2)]

    def forward(self, Hfeat, graph_ptr, gate_u, feat_u, running=None):
        """``running`` = (running_mean, running_var) of compressor.1: model.eval() BatchNorm, forward only (no backward and
        no running-statistics update may follow)."""
        _cuda(Hfeat, graph_ptr, gate_u, feat_u)
        lib, H, dev = _lib.load(), self.H, Hfeat.device
        N, B = Hfeat.shape[0], graph_ptr.numel() - 1
        self.ws = _ws(lib.scgib_core_gate_workspace_bytes(H, B, N), dev)
        self.saved = (graph_ptr, B, N, feat_u.contiguous())
        self.eval_forward = running is not None
        noisy, lam = torch.empty(N, H, device=dev), torch.empty(N, device=dev)
        readout, core, kl = torch.empty(B, H, device=dev), torch.empty(B, H, device=dev), torch.empty(1, device=dev)
        W, b, g, be, w2, b2 = self.p
        common = (_lib.ptr(Hfeat.contiguous()), _lib.ptr(graph_ptr), B, N, H, _lib.ptr(W), _lib.ptr(b), _lib.ptr(g), _lib.ptr(be),
                  _lib.ptr(w2), _lib.ptr(b2))
        tail = (_lib.ptr(gate_u.contiguous()), _lib.ptr(self.saved[3]), _lib.ptr(noisy), _lib.ptr(lam), _lib.ptr(readout),
                _lib.ptr(core), _lib.ptr(kl), _lib.ptr(self.ws), self.ws.numel(), _stream(Hfeat))
        if running is None:
            _lib.check(lib.scgib_core_gate_fwd_f32(*common, *tail), "core_gate_fwd")
        else:
            run = torch.stack([_c32(running[0]), _c32(running[1])]).contiguous()
            _lib.check(lib.scgib_core_gate_eval_fwd_f32(*common, _lib.ptr(run), *tail), "core_gate_eval_fwd")
        return noisy, lam, readout, core, kl

    def _check_train_forward(self, what):
        if self.eval_forward:
            raise RuntimeError("CoreGate.%s() after an eval-mode forward (running statistics): the eval gate is forward only" % what)

    def update_running(self, running_mean, running_var):
        """compressor.1's running statistics after this forward's B per-graph BatchNorm calls (models.py:642), in place."""
        self._check_train_forward("update_running")
        graph_ptr, B, N, feat_u = self.saved
        run = torch.stack([running_mean, running_var]).contiguous().float()
        _lib.check(_lib.load().scgib_core_gate_ema_f32(B, N, self.H, _lib.ptr(run), _lib.ptr(self.ws), self.ws.numel(), _stream(run)),
                   "core_gate_ema")
        running_mean.copy_(run[0]); running_var.copy_(run[1])

    def backward(self, g_noisy, g_core, g_readout, kl_scale=1.0):
        self._check_train_forward("backward")
        lib, H = _lib.load(), self.H
        graph_ptr, B, N, feat_u = self.saved
        dev = feat_u.device
        W, b, g, be, w2, b2 = self.p
        gH = torch.empty(N, H, device=dev)
        out = [torch.empty(H, H, device=dev), torch.empty(H, device=dev), torch.empty(H, device=dev), torch.empty(H, device=dev),
               torch.empty(H, device=dev), torch.empty(1, device=dev)]
        _lib.check(lib.scgib_core_gate_bwd_f32(_lib.ptr(graph_ptr), B, N, H, _lib.ptr(W), _lib.ptr(g), _lib.ptr(be), _lib.ptr(w2),
                                               _lib.ptr(feat_u), _lib.ptr(g_noisy.contiguous()), _lib.ptr(g_core.contiguous()),
                                               _lib.ptr(g_readout.contiguous()), float(kl_scale), _lib.ptr(gH), *[_lib.ptr(t) for t in out],
                                               _lib.ptr(self.ws), self.ws.numel(), _stream(gH)), "core_gate_bwd")
        return (gH, *out)


def core_cand_attn_fwd(C, graph_ptr, w_cand):
    """attention loop of models.py:738-748 -> (alpha [N], T = alpha C [N,H])."""
    _cuda(C, graph_ptr, w_cand)
    N, H = C.shape
    alpha, T = torch.empty(N, device=C.device), torch.empty_like(C)
    _lib.check(_lib.load().scgib_core_cand_attn_fwd_f32(_lib.ptr(C.contiguous()), _lib.ptr(graph_ptr), graph_ptr.numel() - 1, N, H,
                                                        _lib.ptr(w_cand.contiguous()), _lib.ptr(alpha), _lib.ptr(T), _stream(C)), "attn_fwd")
    return alpha, T


def core_cand_attn_bwd(C, alpha, gT, graph_ptr, w_cand):
    _cuda(C, alpha, gT, graph_ptr, w_cand)
    N, H = C.shape
    B = graph_ptr.numel() - 1
    gC, dw = torch.empty_like(C), torch.empty(H, device=C.device)
    ws = _ws((N + B * H) * 4 + 512, C.device)
    _lib.check(_lib.load().scgib_core_cand_attn_bwd_f32(_lib.ptr(C.contiguous()), _lib.ptr(alpha), _lib.ptr(gT.contiguous()), _lib.ptr(graph_ptr),
                                                        B, N, H, _lib.ptr(w_cand.contiguous()), _lib.ptr(gC), _lib.ptr(dw), _lib.ptr(ws),
                                                        ws.numel(), _stream(C)), "attn_bwd")
    return gC, dw


class HeadMLP:
    """self.MLP(interaction_map), interaction_map = [noisy || alpha C] (models.py:569-572, 676, 749)."""

    def __init__(self, hidden, W1, b1, W2, b2):
        self.H = int(hidden)
        self.p = [t.contiguous().float() for t in (W1, b1, W2, b2)]

    def forward(self, noisy, C, alpha):
        _cuda(noisy, C, alpha)
        lib, H, dev = _lib.load(), self.H, noisy.device
        N = noisy.shape[0]
        self.ws = _ws(lib.scgib_head_mlp_workspace_bytes(H, N), dev)
        self.saved = (noisy.contiguous(), N)
        imap, Z = torch.empty(N, 2 * H, device=dev), torch.empty(N, H, device=dev)
        W1, b1, W2, b2 = self.p
        _lib.check(lib.scgib_head_mlp_fwd_f32(_lib.ptr(self.saved[0]), _lib.ptr(C.contiguous()), _lib.ptr(alpha.contiguous()), N, H, _lib.ptr(W1),
                                              _lib.ptr(b1), _lib.ptr(W2), _lib.ptr(b2), _lib.ptr(imap), _lib.ptr(Z), _lib.ptr(self.ws),
                                              self.ws.numel(), _stream(noisy)), "head_mlp_fwd")
        return Z, imap

    def backward(self, gZ):
        lib, H = _lib.load(), self.H
        noisy, N = self.saved
        dev = noisy.device
        W1, b1, W2, b2 = self.p
        gI = torch.empty(2, N, H, device=dev)
        dW1, db1, dW2, db2 = torch.empty(H, 2 * H, device=dev), torch.empty(H, device=dev), torch.empty(H, H, device=dev), torch.empty(H, device=dev)
        _lib.check(lib.scgib_head_mlp_bwd_f32(_lib.ptr(gZ.contiguous()), _lib.ptr(noisy), N, H, _lib.ptr(W1), _lib.ptr(W2), _lib.ptr(gI),
                                              _lib.ptr(dW1), _lib.ptr(db1), _lib.ptr(dW2), _lib.ptr(db2), _lib.ptr(self.ws), self.ws.numel(),
                                              _stream(noisy)), "head_mlp_bwd")
        return gI, dW1, db1, dW2, db2


def segment_sum_bwd(g_out, seg_ptr, rows):
    """backward of dgl.sum_nodes: g_in[row] = g_out[segment(row)]."""
    _cuda(g_out, seg_ptr)
    S, H = g_out.shape
    g_in = torch.empty(rows, H, device=g_out.device)
    _lib.check(_lib.load().scgib_segment_sum_bwd_f32(_lib.ptr(g_out.contiguous()), _lib.ptr(seg_ptr), S, H, _lib.ptr(g_in), _stream(g_out)),
               "segment_sum_bwd")
    return g_in


# ---------------------------------------------------------------- building blocks of --encoder GraphSAGE / GCN (csrc/encoder_ops.cu)
NORM_NONE, NORM_MEAN, NORM_SQRT = 0, 1, 2


def _b16(t):
    """contiguous bf16 operand of the bf16-mode entries (csrc/encoder_bf16.cu); refuses other dtypes."""
    if t is None:
        return None
    if t.dtype != torch.bfloat16:
        raise TypeError("bf16-mode operator: every activation operand must be torch.bfloat16, got %s" % t.dtype)
    return t.detach().contiguous()


def graph_aggregate(h, indptr, indices, src_norm, dst_norm, row_map=None, add=None, out_dtype=None):
    """out[v] = (add[v]) + fd(deg v) sum_{u in N(v)} fs(deg u) h[map(u)]; the SAGEConv mean (NONE, MEAN), its backward
    (MEAN, NONE) and the GraphConv normalised sum (SQRT, SQRT; self-adjoint) on the symmetric CSR.
    A torch.bfloat16 ``h`` (and ``add``) runs the bf16-mode kernel: output bf16, or fp32 with ``out_dtype=torch.float32``."""
    _cuda(h, indptr, indices)
    if h.dtype == torch.bfloat16:
        h, add = _b16(h), _b16(add)
        V, W = indptr.numel() - 1, h.shape[1]
        od = torch.bfloat16 if out_dtype is None else out_dtype
        out = torch.empty(V, W, device=h.device, dtype=od)
        _lib.check(_lib.load().scgib_graph_aggregate_bf16(_lib.ptr(h), W, _lib.ptr(row_map), _lib.ptr(indptr), _lib.ptr(indices), V,
                                                          src_norm, dst_norm, _lib.ptr(add), _lib.ptr(out),
                                                          int(od == torch.float32), _stream(h)), "graph_aggregate_bf16")
        return out
    h = _c32(h)
    add = None if add is None else _c32(add)
    V, W = indptr.numel() - 1, h.shape[1]
    out = torch.empty(V, W, device=h.device)
    _lib.check(_lib.load().scgib_graph_aggregate_f32(_lib.ptr(h), W, _lib.ptr(row_map), _lib.ptr(indptr), _lib.ptr(indices), V,
                                                     src_norm, dst_norm, _lib.ptr(add), _lib.ptr(out), _stream(h)), "graph_aggregate")
    return out


def segment_sum_w(h, seg_ptr):
    """dgl.sum_nodes at width 32 / 64 / 128 / 256."""
    _cuda(h, seg_ptr)
    h = _c32(h)
    S, W = seg_ptr.numel() - 1, h.shape[1]
    out = torch.empty(S, W, device=h.device)
    _lib.check(_lib.load().scgib_segment_sum_w_f32(_lib.ptr(h), _lib.ptr(seg_ptr), S, W, _lib.ptr(out), _stream(h)), "segment_sum_w")
    return out


def linear_fwd(X0, W0, O, w0_kxo=False, X1=None, W1=None, w1_kxo=False, bias=None, relu=False, map0=None, M0=None, M1=None, V=None,
               out_dtype=None):
    """Y[V,O] = act(X0[map0] (.) (M0 > 0) W0 + X1 (.) (M1 > 0) W1 + bias); W [O,K] (nn.Linear) or [K,O] (w_kxo).
    A torch.bfloat16 ``X0`` runs the bf16-mode tensor-core kernel (X1, M0, M1 bf16 too; weights and bias fp32): output bf16,
    or fp32 with ``out_dtype=torch.float32``."""
    _cuda(X0, W0)
    if X0.dtype == torch.bfloat16:
        X0, X1, M0, M1 = (_b16(t) for t in (X0, X1, M0, M1))
        W0, W1, bias = (None if t is None else _c32(t) for t in (W0, W1, bias))
        V = int(V if V is not None else (map0.numel() if map0 is not None else X0.shape[0]))
        od = torch.bfloat16 if out_dtype is None else out_dtype
        Y = torch.empty(V, O, device=X0.device, dtype=od)
        _lib.check(_lib.load().scgib_linear_fwd_bf16(_lib.ptr(X0), _lib.ptr(M0), _lib.ptr(map0), _lib.ptr(W0), X0.shape[1], int(w0_kxo),
                                                     _lib.ptr(X1), _lib.ptr(M1), _lib.ptr(W1), 0 if X1 is None else X1.shape[1],
                                                     int(w1_kxo), _lib.ptr(bias), int(relu), V, O, _lib.ptr(Y),
                                                     int(od == torch.float32), _stream(X0)), "linear_fwd_bf16")
        return Y
    X0, W0, X1, W1, bias, M0, M1 = (None if t is None else _c32(t) for t in (X0, W0, X1, W1, bias, M0, M1))
    V = int(V if V is not None else (map0.numel() if map0 is not None else X0.shape[0]))
    Y = torch.empty(V, O, device=X0.device)
    _lib.check(_lib.load().scgib_linear_fwd_f32(_lib.ptr(X0), _lib.ptr(M0), _lib.ptr(map0), _lib.ptr(W0), X0.shape[1], int(w0_kxo),
                                                _lib.ptr(X1), _lib.ptr(M1), _lib.ptr(W1), 0 if X1 is None else X1.shape[1],
                                                int(w1_kxo), _lib.ptr(bias), int(relu), V, O, _lib.ptr(Y), _stream(X0)), "linear_fwd")
    return Y


def linear_bwd_w(G, X, dW, db=None, M=None, map=None, kxo=False, accumulate=False):
    """dW (+)= (G (.) (M > 0))^T X[map] ([O,K], or [K,O] with kxo), db (+)= column sums; in place on dW / db.
    A torch.bfloat16 ``G`` runs the bf16-mode tensor-core kernel (M, X bf16 too; dW / db stay fp32)."""
    _cuda(G, X, dW)
    if not (dW.is_contiguous() and dW.dtype == torch.float32) or (db is not None and not db.is_contiguous()):
        raise ValueError("linear_bwd_w writes dW / db in place: contiguous fp32 tensors")
    if G.dtype == torch.bfloat16:
        G, X, M = _b16(G), _b16(X), _b16(M)
        lib = _lib.load()
        V, O, K = G.shape[0], G.shape[1], X.shape[1]
        ws = _ws(lib.scgib_linear_bwd_w_bf16_workspace_bytes(V, O, K), G.device)
        _lib.check(lib.scgib_linear_bwd_w_bf16(_lib.ptr(G), _lib.ptr(M), _lib.ptr(X), _lib.ptr(map), V, O, K, int(kxo), int(accumulate),
                                               _lib.ptr(dW), _lib.ptr(db), _lib.ptr(ws), ws.numel(), _stream(G)), "linear_bwd_w_bf16")
        return dW, db
    G, X, M = _c32(G), _c32(X), None if M is None else _c32(M)
    lib = _lib.load()
    V, O, K = G.shape[0], G.shape[1], X.shape[1]
    ws = _ws(lib.scgib_linear_bwd_w_workspace_bytes(V, O, K), G.device)
    _lib.check(lib.scgib_linear_bwd_w_f32(_lib.ptr(G), _lib.ptr(M), _lib.ptr(X), _lib.ptr(map), V, O, K, int(kxo), int(accumulate),
                                          _lib.ptr(dW), _lib.ptr(db), _lib.ptr(ws), ws.numel(), _stream(G)), "linear_bwd_w")
    return dW, db


def transfer_bwd(x, g0, g1, map1, normalize=True, csr0=None, csr1=None):
    """d transfer_d.weight [d_transfer, F] from the input gradients [V, d_transfer] of the two row sets (parent rows / ego rows
    through map1); d_transfer = g0.shape[1] (32, 64 or 128)."""
    _cuda(x, g0)
    x, g0, g1 = _c32(x), _c32(g0), None if g1 is None else _c32(g1)
    lib = _lib.load()
    F, DT, V0, V1 = x.shape[1], g0.shape[1], g0.shape[0], 0 if g1 is None else g1.shape[0]
    if g1 is not None and g1.shape[1] != DT:
        raise ValueError("transfer_bwd: g0 and g1 differ in width (%d, %d)" % (DT, g1.shape[1]))
    dWt = torch.empty(DT, F, device=x.device)
    nbytes = lib.scgib_transfer_bwd_workspace_bytes_d(V0, V1, F, DT)
    ws = torch.empty(int(nbytes) + 256, dtype=torch.uint8, device=x.device)
    off = (-ws.data_ptr()) % 256
    ip0, ix0 = csr0 if csr0 is not None else (None, None)
    ip1, ix1 = csr1 if csr1 is not None else (None, None)
    _lib.check(lib.scgib_transfer_bwd_d_f32(_lib.ptr(x), F, DT, int(normalize), _lib.ptr(g0), V0, _lib.ptr(ip0), _lib.ptr(ix0), _lib.ptr(g1),
                                            V1, _lib.ptr(ip1), _lib.ptr(ix1), _lib.ptr(map1), _lib.ptr(dWt),
                                            ctypes.c_void_p(ws.data_ptr() + off), int(nbytes), _stream(x)), "transfer_bwd")
    return dWt
