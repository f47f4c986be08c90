"""--encoder GraphSAGE / GCN on the B200 path (reference models.py:75-104, selected at models.py:573-587).

The CLI default (--encoder GIN) runs the fused tensor-core engine (engine.py / csrc/api.cu).  The two other message-passing
encoders of the reference are composed here, layer by layer, from the hand-written operator kernels behind the C ABI
(csrc/encoder_ops.cu: normalised aggregation, FP32 linear tiles, weight-gradient reduction; csrc/api.cu: core gate,
core-candidate attention, head MLP, the two batch losses, the transfer_d backward).  Host code only sequences the
launches and keeps the saved activations: no torch kernels compute anything on this path except the final scaling of the
parameter gradients by the upstream loss gradient, and nothing falls back to torch or the CPU.

The parameter containers reproduce DGL 1.1.x's state-dict keys and default initialisation (``convN.fc_self.weight`` /
``convN.fc_neigh.weight`` / ``convN.fc_self.bias`` for SAGEConv, ``convN.weight`` [in, out] / ``convN.bias`` for GraphConv), so a
reference checkpoint loads unchanged.  DGL itself is not available offline: its semantics are restated
(tests/golden/dgl_stub), "DGL internals unpinned" as everywhere else in this repository.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops
from .ops import NORM_MEAN, NORM_NONE, NORM_SQRT

DTR = 32


# ---------------------------------------------------------------------------------------------- parameter containers
class SAGEConv(nn.Module):
    """dgl.nn.SAGEConv(in_feats, out_feats, 'mean'): rst = fc_self(h) + fc_neigh(mean_{u in N(v)} h_u)."""

    def __init__(self, in_feats, out_feats, aggregator_type="mean"):
        super().__init__()
        if aggregator_type != "mean":
            raise NotImplementedError("SAGEConv aggregator '%s' (the reference uses 'mean', models.py:94-96)" % aggregator_type)
        self.fc_neigh = nn.Linear(in_feats, out_feats, bias=False)
        self.fc_self = nn.Linear(in_feats, out_feats, bias=True)
        gain = nn.init.calculate_gain("relu")
        nn.init.xavier_uniform_(self.fc_self.weight, gain=gain)
        nn.init.xavier_uniform_(self.fc_neigh.weight, gain=gain)


class GraphSAGE(nn.Module):
    """reference models.py:91-104: conv1, ReLU, conv2, ReLU, conv2 again (conv3 is constructed and never called), no final
    ReLU.  ``conv3`` is kept for state-dict compatibility."""
    kind = "GraphSAGE"

    def __init__(self, in_feats, h_feats):
        super().__init__()
        self.in_feats, self.hidden_dim = in_feats, h_feats
        self.conv1 = SAGEConv(in_feats, h_feats, "mean")
        self.conv2 = SAGEConv(h_feats, h_feats, "mean")
        self.conv3 = SAGEConv(h_feats, h_feats, "mean")

    def run_forward(self, t, indptr, indices, row_map=None):
        """t [rows, in_feats]; row r of this encoder reads t[row_map[r]] (the ego batch).  Returns (out [V, h], saved)."""
        H, c1, c2 = self.hidden_dim, self.conv1, self.conv2
        V = indptr.numel() - 1
        agg = lambda h, rm=None: ops.graph_aggregate(h, indptr, indices, NORM_NONE, NORM_MEAN, row_map=rm)
        m0 = agg(t, row_map)
        h1 = ops.linear_fwd(t, c1.fc_self.weight, H, X1=m0, W1=c1.fc_neigh.weight, bias=c1.fc_self.bias, relu=True, map0=row_map, V=V)
        m1 = agg(h1)
        h2 = ops.linear_fwd(h1, c2.fc_self.weight, H, X1=m1, W1=c2.fc_neigh.weight, bias=c2.fc_self.bias, relu=True)
        m2 = agg(h2)
        h3 = ops.linear_fwd(h2, c2.fc_self.weight, H, X1=m2, W1=c2.fc_neigh.weight, bias=c2.fc_self.bias, relu=False)
        return h3, (t, row_map, indptr, indices, m0, h1, m1, h2, m2)

    def run_backward(self, saved, g_out, weights=True):
        """-> (gradient wrt the gathered input rows [V, in_feats], {parameter name: gradient}); ``weights=False`` (every
        parameter of this encoder frozen) skips the weight-gradient launches and returns an empty dict."""
        t, row_map, indptr, indices, m0, h1, m1, h2, m2 = saved
        H, c1, c2 = self.hidden_dim, self.conv1, self.conv2
        dev = g_out.device
        new = lambda *s: torch.empty(*s, device=dev)
        dWs1, dWn1, db1 = new(H, self.in_feats), new(H, self.in_feats), new(H)
        dWs2, dWn2, db2 = new(H, H), new(H, H), new(H)
        bwd_w = ops.linear_bwd_w if weights else (lambda *a, **k: None)
        aggT = lambda u, add: ops.graph_aggregate(u, indptr, indices, NORM_MEAN, NORM_NONE, add=add)

        def through(g, mask, conv, width):      # gradient wrt the layer input: g Ws + A^T(g Wn), g masked by the layer's ReLU
            u = ops.linear_fwd(g, conv.fc_neigh.weight, width, w0_kxo=True, M0=mask)
            gs = ops.linear_fwd(g, conv.fc_self.weight, width, w0_kxo=True, M0=mask)
            return aggT(u, gs)

        # third layer: conv2 without ReLU
        bwd_w(g_out, h2, dWs2, db2)
        bwd_w(g_out, m2, dWn2)
        g_h2 = through(g_out, None, c2, H)
        # second layer: conv2 (its second use: the weight gradients accumulate), ReLU mask h2 > 0
        bwd_w(g_h2, h1, dWs2, db2, M=h2, accumulate=True)
        bwd_w(g_h2, m1, dWn2, M=h2, accumulate=True)
        g_h1 = through(g_h2, h2, c2, H)
        # first layer: conv1 on the gathered t rows
        bwd_w(g_h1, t, dWs1, db1, M=h1, map=row_map)
        bwd_w(g_h1, m0, dWn1, M=h1)
        g_t = through(g_h1, h1, c1, self.in_feats)
        if not weights:
            return g_t, {}
        return g_t, {"conv1.fc_self.weight": dWs1, "conv1.fc_neigh.weight": dWn1, "conv1.fc_self.bias": db1,
                     "conv2.fc_self.weight": dWs2, "conv2.fc_neigh.weight": dWn2, "conv2.fc_self.bias": db2}


class GraphConv(nn.Module):
    """dgl.nn.pytorch.conv.GraphConv(in, out, norm='both', allow_zero_in_degree=True): D^-1/2 A D^-1/2 h W + b."""

    def __init__(self, in_feats, out_feats, allow_zero_in_degree=True):
        super().__init__()
        self.weight = nn.Parameter(torch.empty(in_feats, out_feats))
        self.bias = nn.Parameter(torch.zeros(out_feats))
        nn.init.xavier_uniform_(self.weight)


class GCN(nn.Module):
    """reference models.py:75-88: widths in -> 2h -> 2h -> h, ReLU between the layers, none after conv3."""
    kind = "GCN"

    def __init__(self, num_features, hidden_dim=64):
        super().__init__()
        self.in_feats, self.hidden_dim = num_features, hidden_dim
        self.conv1 = GraphConv(num_features, hidden_dim * 2)
        self.conv2 = GraphConv(hidden_dim * 2, hidden_dim * 2)
        self.conv3 = GraphConv(hidden_dim * 2, hidden_dim)

    def run_forward(self, t, indptr, indices, row_map=None):
        H = self.hidden_dim
        agg = lambda h, rm=None: ops.graph_aggregate(h, indptr, indices, NORM_SQRT, NORM_SQRT, row_map=rm)
        a0 = agg(t, row_map)
        h1 = ops.linear_fwd(a0, self.conv1.weight, 2 * H, w0_kxo=True, bias=self.conv1.bias, relu=True)
        a1 = agg(h1)
        h2 = ops.linear_fwd(a1, self.conv2.weight, 2 * H, w0_kxo=True, bias=self.conv2.bias, relu=True)
        a2 = agg(h2)
        h3 = ops.linear_fwd(a2, self.conv3.weight, H, w0_kxo=True, bias=self.conv3.bias, relu=False)
        return h3, (indptr, indices, a0, h1, a1, h2, a2)

    def run_backward(self, saved, g_out, weights=True):
        indptr, indices, a0, h1, a1, h2, a2 = saved
        H, dev = self.hidden_dim, g_out.device
        new = lambda *s: torch.empty(*s, device=dev)
        agg = lambda h: ops.graph_aggregate(h, indptr, indices, NORM_SQRT, NORM_SQRT)       # self-adjoint on the symmetric CSR
        dW1, db1 = new(self.in_feats, 2 * H), new(2 * H)
        dW2, db2 = new(2 * H, 2 * H), new(2 * H)
        dW3, db3 = new(2 * H, H), new(H)
        bwd_w = ops.linear_bwd_w if weights else (lambda *a, **k: None)
        bwd_w(g_out, a2, dW3, db3, kxo=True)
        g_h2 = agg(ops.linear_fwd(g_out, self.conv3.weight, 2 * H))                      # g W3^T: W3 [2h, h] read as [O, K]
        bwd_w(g_h2, a1, dW2, db2, M=h2, kxo=True)
        g_h1 = agg(ops.linear_fwd(g_h2, self.conv2.weight, 2 * H, M0=h2))
        bwd_w(g_h1, a0, dW1, db1, M=h1, kxo=True)
        g_t = agg(ops.linear_fwd(g_h1, self.conv1.weight, self.in_feats, M0=h1))
        if not weights:
            return g_t, {}
        return g_t, {"conv1.weight": dW1, "conv1.bias": db1, "conv2.weight": dW2, "conv2.bias": db2,
                     "conv3.weight": dW3, "conv3.bias": db3}


def make_encoder(encoder, in_dim, hidden_dim):
    if encoder == "GraphSAGE":
        return GraphSAGE(in_dim, hidden_dim)
    if encoder == "GCN":
        return GCN(in_dim, hidden_dim)
    raise ValueError(encoder)


# ---------------------------------------------------------------------------------------------- the composed step
def _f(t):
    return t.detach().contiguous().float()


def inner_of(model):
    """Mainmodel_continue (models.py:1010-1276) trains its own transfer_d / MLP around the LOADED module's encoders,
    compressor and attention layer (``self.model``); Mainmodel owns everything."""
    return getattr(model, "model", None) or model


def resolve_param(model, name):
    root = model if (name.startswith("transfer_d") or name.startswith("MLP.")) else inner_of(model)
    obj = root
    for p in name.split("."):
        obj = obj[int(p)] if p.isdigit() else getattr(obj, p)
    return obj


def composed_features(outer, g, ego, t, gate_u, feat_u):
    """reference models.py:702-750 on operator kernels.  ``t`` [N, d_transfer] transferred features.  Returns the outputs
    and everything the backward needs."""
    model = inner_of(outer)
    Hd = int(outer.hidden_dim)
    Hf, sv1 = model.Encoder1.run_forward(t, g.indptr, g.indices)
    S, sv2 = model.Encoder2.run_forward(t, ego.sub_indptr, ego.sub_indices, row_map=ego.ego_nodes)
    c = model.compressor
    gate = ops.CoreGate(Hd, _f(c[0].weight), _f(c[0].bias), _f(c[1].weight), _f(c[1].bias), _f(c[3].weight), _f(c[3].bias))
    bn = c[1]
    # compressor.1 follows its own training flag, as nn.BatchNorm1d does: per-graph batch statistics and B sequential
    # running-statistics updates, one per graph (models.py:642), or - in eval - the running statistics (forward only).
    # The gate / feature noise is drawn in both modes (models.py:599, 650).
    if bn.training:
        noisy, lam, readout, core, kl = gate.forward(Hf, g.graph_ptr, gate_u, feat_u)
        gate.update_running(bn.running_mean, bn.running_var)
    else:
        noisy, lam, readout, core, kl = gate.forward(Hf, g.graph_ptr, gate_u, feat_u, running=(bn.running_mean, bn.running_var))
    C = ops.segment_sum_w(S, ego.ego_ptr)
    w_cand = _f(model.attn_layer.weight[0, Hd:])
    alpha, _ = ops.core_cand_attn_fwd(C, g.graph_ptr, w_cand)
    mlp = outer.MLP
    head = ops.HeadMLP(Hd, _f(mlp[0].weight), _f(mlp[0].bias), _f(mlp[2].weight), _f(mlp[2].bias))
    Z, imap = head.forward(noisy, C, alpha)
    st = dict(sv1=sv1, sv2=sv2, gate=gate, head=head, C=C, alpha=alpha, w_cand=w_cand, Ns=int(ego.sub_indptr.numel() - 1))
    return dict(interaction_map=imap, Z=Z, noisy=noisy, graph_readout=readout, core_readout=core, kl=kl), st


def composed_param_names(model):
    """The parameters the composed step differentiates, in the order the autograd Function receives them."""
    names = ["transfer_d.weight", "attn_layer.weight", "attn_layer.bias", "MLP.0.weight", "MLP.0.bias", "MLP.2.weight", "MLP.2.bias"]
    enc = ["conv1.fc_self.weight", "conv1.fc_neigh.weight", "conv1.fc_self.bias", "conv2.fc_self.weight", "conv2.fc_neigh.weight",
           "conv2.fc_self.bias"] if inner_of(model).Encoder1.kind == "GraphSAGE" else \
          ["conv1.weight", "conv1.bias", "conv2.weight", "conv2.bias", "conv3.weight", "conv3.bias"]
    names += ["Encoder1." + n for n in enc] + ["Encoder2." + n for n in enc]
    names += ["compressor.0.weight", "compressor.0.bias", "compressor.1.weight", "compressor.1.bias", "compressor.3.weight",
              "compressor.3.bias"]
    return names


def composed_backward(outer, st, gZ, g_core, g_readout, kl_scale, names):
    """The backward of ``composed_features`` + head MLP: gradients of <gZ, Z> + <g_core, core_readout> +
    <g_readout, graph_readout> + kl_scale * KL for the parameter ``names`` (composed_param_names order), as a dict.
    The input-gradient chain always runs down to transfer_d; an encoder none of whose parameters is named (all frozen:
    fine-tuning) skips its weight-gradient launches."""
    model = inner_of(outer)
    g, ego = st["g"], st["ego"]
    Hd = int(outer.hidden_dim)
    gI, dW1h, db1h, dW2h, db2h = st["head"].backward(gZ)
    gC, dw_cand = ops.core_cand_attn_bwd(st["C"], st["alpha"], gI[1], g.graph_ptr, st["w_cand"])
    gH, dWc1, dbc1, dgam, dbet, dwc2, dbc2 = st["gate"].backward(gI[0], g_core, g_readout, kl_scale=kl_scale)
    gS = ops.segment_sum_bwd(gC, ego.ego_ptr, st["Ns"])
    w1 = any(n.startswith("Encoder1.") for n in names)
    w2 = any(n.startswith("Encoder2.") for n in names)
    gt0, ge1 = model.Encoder1.run_backward(st["sv1"], gH, weights=w1)
    gt1, ge2 = model.Encoder2.run_backward(st["sv2"], gS, weights=w2)
    dWt = ops.transfer_bwd(st["x"], gt0, gt1, ego.ego_nodes, normalize=True)
    d_attn = torch.zeros(1, 2 * Hd, device=gH.device)
    d_attn[0, Hd:] = dw_cand            # the core half and the bias cancel inside the per-graph softmax: exactly zero
    grads = {"transfer_d.weight": dWt, "attn_layer.weight": d_attn, "attn_layer.bias": torch.zeros(1, device=gH.device),
             "MLP.0.weight": dW1h, "MLP.0.bias": db1h, "MLP.2.weight": dW2h, "MLP.2.bias": db2h,
             "compressor.0.weight": dWc1, "compressor.0.bias": dbc1, "compressor.1.weight": dgam, "compressor.1.bias": dbet,
             "compressor.3.weight": dwc2.reshape(1, Hd), "compressor.3.bias": dbc2.reshape(1)}
    grads.update({"Encoder1." + n: v for n, v in ge1.items()})
    grads.update({"Encoder2." + n: v for n, v in ge2.items()})
    return {n: grads[n] for n in names}


def trainable_param_names(outer):
    """composed_param_names restricted to the parameters that require a gradient (fine-tuning freezes the loaded model)."""
    return [n for n in composed_param_names(outer) if resolve_param(outer, n).requires_grad]


class ComposedPretrainFn(torch.autograd.Function):
    """Mainmodel.forward (models.py:662-700) for --encoder GraphSAGE / GCN: (KL, contrastive, reconstruction)."""

    @staticmethod
    def forward(ctx, model, g, ego, x, gate_u, feat_u, names, *params):
        t = ops.input_proj(x, _f(model.transfer_d.weight))                 # F.normalize + transfer_d (idempotent on normalised x)
        out, st = composed_features(model, g, ego, t, gate_u, feat_u)
        if getattr(model, "recons_type", "adj") == "logM":                 # models.py:693-694: k-step log transition matrices
            rec, gZ, _ = ops.recon_logm(out["Z"], g.graph_ptr, g.indptr, g.indices, int(model.k_transition), 1.0)
        else:
            rec, gZ = ops.recon_adj(out["Z"], g.indptr, g.indices, 1.0)    # value and gradient in one launch sequence
        con, g_core, g_readout = ops.contrastive(out["core_readout"], out["graph_readout"], 1.0)
        st.update(gZ=gZ, g_core=g_core, g_readout=g_readout, x=x, g=g, ego=ego)
        ctx.model, ctx.st, ctx.names = model, st, names
        model._composed_last = out
        return out["kl"].reshape(()).clone(), con.reshape(()), rec.reshape(())

    @staticmethod
    def backward(ctx, g_kl, g_con, g_rec):
        model, st, names = ctx.model, ctx.st, ctx.names
        same = g_kl.data_ptr() == g_con.data_ptr() == g_rec.data_ptr() and g_kl.numel() == 1
        if same:        # loss = KL + recon + contrastive (exp_pretraining.py:320): scale the parameter gradients once, no host read
            s_kl = s_con = s_rec = 1.0
        else:
            s_kl, s_con, s_rec = torch.stack([g_kl.reshape(()), g_con.reshape(()), g_rec.reshape(())]).tolist()
        gZ = st["gZ"] if s_rec == 1.0 else st["gZ"] * s_rec
        g_core = st["g_core"] if s_con == 1.0 else st["g_core"] * s_con
        g_readout = st["g_readout"] if s_con == 1.0 else st["g_readout"] * s_con
        grads = composed_backward(model, st, gZ, g_core, g_readout, s_kl, names)
        out = [grads[n] for n in names]
        if same:
            torch._foreach_mul_(out, g_kl.reshape(()).to(out[0].dtype))
        ctx.st = None
        return (None,) * 7 + tuple(out)


def _zero_readout_grads(st, outer):
    B, Hd = st["g"].batch_size, int(outer.hidden_dim)
    z = torch.zeros(B, Hd, device=st["x"].device)
    return z, z


class ComposedFinetuneFn(torch.autograd.Function):
    """Mainmodel_finetuning.forward (models.py:501-520) around GraphSAGE / GCN encoders: transfer_d -> the loaded model's
    extract_features -> MLP -> Set2Set -> predict (-> sigmoid).  Parameters: ``names`` (composed_param_names of the ones that
    require a gradient), then the head's FT_NAMES slots."""

    @staticmethod
    def forward(ctx, owner, g, ego, x, gate_u, feat_u, names, *params):
        head = owner._head
        t = ops.input_proj(x, _f(owner.transfer_d.weight))
        out, st = composed_features(owner, g, ego, t, gate_u, feat_u)
        scores = head.forward(out["Z"], g.graph_ptr)
        st.update(x=x, g=g, ego=ego)
        ctx.owner, ctx.st, ctx.names, ctx.params = owner, st, names, params
        ctx.serial = head.fwd_serial
        return scores

    @staticmethod
    def backward(ctx, g_scores):
        from .models import _check_serial, _detach_aliased_grads
        from .engine import FT_NAMES
        owner, st, names = ctx.owner, ctx.st, ctx.names
        head = owner._head
        _check_serial("Mainmodel_finetuning (head)", head, ctx.serial)
        _detach_aliased_grads(ctx.params, head.grads)
        gZ = head.backward(g_scores)
        g_core, g_readout = _zero_readout_grads(st, owner)
        grads = composed_backward(owner, st, gZ, g_core, g_readout, 0.0, names)
        hv = head.views(grads=True)
        ctx.st = None
        return (None,) * 7 + tuple(grads[n] for n in names) + tuple(hv.pop(n) for n in FT_NAMES)


class ComposedDomainAdaptFn(torch.autograd.Function):
    """Mainmodel_domainadapt.forward (models.py:254-269) around GraphSAGE / GCN encoders -> (r_transfer_d(s2s(MLP(
    extract_features))) [B, 2 in_dim], s2s_rev(x) [B, 2 in_dim]).  Parameters: ``names``, the head's slots (r_transfer_d in
    the predict slots), the four s2s_rev LSTM tensors."""

    @staticmethod
    def forward(ctx, owner, g, ego, x, gate_u, feat_u, x_norm, names, *params):
        head, rev = owner._head, owner._rev
        t = ops.input_proj(x, _f(owner.transfer_d.weight))
        out, st = composed_features(owner, g, ego, t, gate_u, feat_u)
        rec = head.forward(out["Z"], g.graph_ptr)
        org = rev.forward(x_norm, g.graph_ptr)
        st.update(x=x, g=g, ego=ego)
        ctx.owner, ctx.st, ctx.names, ctx.params = owner, st, names, params
        ctx.serial = (head.fwd_serial, rev.head.fwd_serial)
        return rec, org

    @staticmethod
    def backward(ctx, g_rec, g_org):
        from .models import _check_serial, _detach_aliased_grads
        from .engine import FT_NAMES
        owner, st, names = ctx.owner, ctx.st, ctx.names
        head, rev = owner._head, owner._rev
        _check_serial("Mainmodel_domainadapt (head)", head, ctx.serial[0])
        _check_serial("Mainmodel_domainadapt (s2s_rev)", rev.head, ctx.serial[1])
        _detach_aliased_grads(ctx.params, head.grads)
        gZ = head.backward(g_rec)
        g_core, g_readout = _zero_readout_grads(st, owner)
        grads = composed_backward(owner, st, gZ, g_core, g_readout, 0.0, names)
        hv = head.views(grads=True)
        ctx.st = None
        return ((None,) * 8 + tuple(grads[n] for n in names) + tuple(hv.pop(n) for n in FT_NAMES) +
                tuple(rev.backward(g_org)))
