"""Drop-in replacements for the reference's model classes on the pre-training hot path.

Same class names, constructor arguments, ``forward`` signatures, return values and state-dict keys as the reference
(models.py:38-72 MLP / GIN, :546-782 Mainmodel, :1010-1276 Mainmodel_continue); the computation runs in the sm_100a
kernels of libscgib.so through one autograd Function per step.  There is no PyTorch fallback: on a CPU device or
without the library the forward raises.

Parameters stay ordinary ``nn.Parameter`` objects (optimisers, ``state_dict`` and ``torch.save(model)`` work), but
their storage is re-pointed at one flat device buffer so the kernels, the gradient all-reduce and the fused Adam
see a single tensor.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from .engine import (FT_NAMES, HID, DeviceBatch, FinetuneHead, PaddedSet2Set, PretrainEngine, bn_buffer_names,
                     param_names)
from .graph import BatchedGraph, EgoBatch, khop_ego_batch

_CPU_GATE_NOISE = __import__("os").environ.get("SCGIB_CPU_GATE_NOISE", "0") == "1"
DEFAULT_GIN_LAYERS = 4   # reference models.py:57-58: ``num_layers = 5; range(num_layers - 1)``


class MLP(nn.Module):
    """reference models.py:38-49."""

    def __init__(self, num_features, num_classes, dims=16):
        super().__init__()
        self.mlp = nn.Sequential(nn.Linear(num_features, dims), nn.ReLU(), nn.Linear(dims, num_classes))

    def forward(self, x):
        return self.mlp(x)


class GINConv(nn.Module):
    """Parameter container with DGL GINConv's attribute names (``apply_func``, buffer ``eps`` = [0.])."""

    def __init__(self, apply_func=None, aggregator_type="sum", init_eps=0, learn_eps=False):
        super().__init__()
        if aggregator_type != "sum" or learn_eps:
            raise NotImplementedError("only GINConv('sum', learn_eps=False) is on the S-CGIB path (models.py:63)")
        self.apply_func = apply_func
        self.register_buffer("eps", torch.FloatTensor([init_eps]))


class GIN(nn.Module):
    """reference models.py:52-72.  ``forward(g, h)`` runs the fused CUDA layers (inference of the encoder alone:
    no autograd; training goes through Mainmodel.forward)."""

    def __init__(self, input_dim, hidden_dim=64, num_gin_layers=DEFAULT_GIN_LAYERS):
        super().__init__()
        if hidden_dim not in (64, 128):
            raise NotImplementedError("libscgib is built for hidden_dim 64 or 128 (--dims, exp_pretraining.py:390)")
        self.hidden_dim = hidden_dim
        self.ginlayers = nn.ModuleList()
        self.batch_norms = nn.ModuleList()
        for layer in range(num_gin_layers):
            mlp = MLP(input_dim if layer == 0 else hidden_dim, hidden_dim, hidden_dim)
            self.ginlayers.append(GINConv(mlp, learn_eps=False))
            self.batch_norms.append(nn.BatchNorm1d(hidden_dim))

    @torch.no_grad()
    def forward(self, g, h):
        from . import ops
        if self.hidden_dim != HID:
            raise NotImplementedError("the stand-alone GIN.forward (op-level entry) is built for hidden_dim=64; the models run 128 "
                                      "through Mainmodel.forward")
        indptr, indices = (g.sub_indptr, g.sub_indices) if isinstance(g, EgoBatch) else (g.indptr, g.indices)
        bn_in = None
        for i, layer in enumerate(self.ginlayers):
            lin1, lin2 = layer.apply_func.mlp[0], layer.apply_func.mlp[2]
            bn = self.batch_norms[i]
            running = torch.stack([bn.running_mean, bn.running_var]).contiguous() if self.training else None
            y, stats, _, _ = ops.gin_layer_fwd(h, indptr, indices, lin1.weight, lin1.bias, lin2.weight, lin2.bias,
                                               bn_in=bn_in, running=running)
            if self.training:
                bn.running_mean.copy_(running[0]); bn.running_var.copy_(running[1]); bn.num_batches_tracked += 1
                mean, rstd = stats[0], stats[1]
            else:
                mean, rstd = bn.running_mean, torch.rsqrt(bn.running_var + bn.eps)
            bn_in = torch.stack([mean, rstd, bn.weight, bn.bias]).contiguous()
            h = y
        return torch.relu((h - bn_in[0]) * bn_in[1] * bn_in[2] + bn_in[3])


class _Set2SetParams(nn.Module):
    """``dgl.nn.Set2Set(hidden, 2, 1)`` as a parameter container (``s2s.lstm.*`` keys); the pre-training default
    readout is 'sum' (exp_pretraining.py:380), so it never runs on this path."""

    def __init__(self, input_dim, n_iters, n_layers):
        super().__init__()
        self.input_dim, self.output_dim, self.n_iters, self.n_layers = input_dim, 2 * input_dim, n_iters, n_layers
        self.lstm = nn.LSTM(2 * input_dim, input_dim, n_layers)
        self.lstm.reset_parameters()          # DGL's Set2Set.__init__ re-initialises the LSTM (second RNG draw)


def _check_serial(what, obj, serial):
    """The engine keeps ONE workspace of saved activations: backward must belong to the most recent forward."""
    if obj.fwd_serial != serial:
        raise RuntimeError("scgib_b200: %s.backward() after another forward on the same model - the saved activations of "
                           "this forward were overwritten (one forward, then its backward; see INTEGRATION.md)" % what)


def _detach_aliased_grads(params, flat):
    """The backward kernels overwrite the flat gradient buffer.  A parameter whose .grad still aliases it (adopted from
    an earlier backward and not reset by zero_grad) gets a private copy first, so gradient accumulation is preserved."""
    lo, hi = flat.data_ptr(), flat.data_ptr() + flat.numel() * flat.element_size()
    for p in params:
        g = p.grad
        if g is not None and lo <= g.data_ptr() < hi:
            p.grad = g.clone()


class _PretrainFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, bridge, batch, gate_u, feat_u, *params):
        eng = bridge.engine
        losses = eng.forward(batch, gate_u, feat_u, update_running=bridge.training)
        ctx.bridge = bridge
        ctx.params = params
        ctx.serial = eng.fwd_serial
        out = losses.clone()
        return out[0], out[1], out[2]

    @staticmethod
    def backward(ctx, g_kl, g_con, g_rec):
        eng = ctx.bridge.engine
        _check_serial("Mainmodel", eng, ctx.serial)
        _detach_aliased_grads(ctx.params, eng.grads)
        if g_kl.data_ptr() == g_con.data_ptr() == g_rec.data_ptr() and g_kl.numel() == 1:
            # loss = KL + recon + contrastive (exp_pretraining.py:320): the three upstream gradients are one tensor.  Run the
            # backward at scale 1 and multiply the flat gradient buffer by it on the device - no host read, no sync.
            eng.backward((1.0, 1.0, 1.0))
            eng.grads.mul_(g_kl.reshape(()).to(eng.grads.dtype))
        else:
            scale = torch.stack([g_kl, g_con, g_rec]).tolist()    # individually weighted losses: one host read
            eng.backward(tuple(scale))
        gv = eng.grad_views()
        # views of the flat gradient buffer, no copies: autograd's AccumulateGrad adopts them as .grad when .grad is None
        # (zero_grad(set_to_none=True), the default); gradients that are still live from an earlier backward were moved
        # out of the buffer by _detach_aliased_grads, so accumulation across backward calls stays correct
        return (None, None, None, None) + tuple(gv.pop(name) for name in ctx.bridge.slot_names)   # pop: no second reference


class _Bridge:
    """Keeps the module's parameters / BN buffers aliased to the engine's flat buffers."""

    def __init__(self, owner, in_dim, gin_layers):
        self.owner, self.in_dim, self.gin_layers = owner, in_dim, gin_layers
        self.engine = None
        self.slot_names = param_names(gin_layers)
        self.training = True

    def _resolve(self, name):
        """Slot name -> (module holding it, attribute path).  transfer_d / MLP come from the outer module, the rest
        from the module whose extract_features runs (the loaded ``self.model`` for Mainmodel_continue)."""
        o = self.owner
        inner = getattr(o, "model", None) or o
        root = o if (name.startswith("transfer_d") or name.startswith("MLP.")) else inner
        obj = root
        parts = name.split(".")
        for p in parts[:-1]:
            obj = obj[int(p)] if p.isdigit() else getattr(obj, p)
        return obj, parts[-1]

    def sync(self, device):
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("S-CGIB B200 path: the model must be on a CUDA device (no CPU fallback)")
        cached = getattr(self, "_cached", None)
        if cached is not None and self.engine is not None and self.engine.device == device and \
                all(p.data_ptr() == ptr for p, ptr in cached[1]) and all(b.data_ptr() == ptr for b, ptr in cached[2]):
            return cached[0]          # every parameter / BN buffer still aliases the flat buffers: nothing to do
        params = self._sync_slow(device)
        inner = self._bn_modules
        bufs = []
        for i, base in enumerate(bn_buffer_names(self.gin_layers)):
            obj = inner
            for q in base.split("."):
                obj = obj[int(q)] if q.isdigit() else getattr(obj, q)
            bufs += [(obj.running_mean, obj.running_mean.data_ptr()), (obj.running_var, obj.running_var.data_ptr())]
        self._cached = (params, [(p, p.data_ptr()) for p in params], bufs)
        return params

    def _sync_slow(self, device):
        if self.engine is None or self.engine.device != device:
            self.engine = PretrainEngine(self.in_dim, gin_layers=self.gin_layers, hidden=int(getattr(self.owner, "hidden_dim", HID)),
                                         device=device, dtype=getattr(self.owner, "act_dtype", "fp32"))
        views = self.engine.views()
        params = []
        for name in self.slot_names:
            mod, attr = self._resolve(name)
            p = getattr(mod, attr)
            v = views[name]
            if p.data_ptr() != v.data_ptr():
                v.copy_(p.data.to(device).reshape(v.shape))
                p.data = v
            params.append(p)
        inner = getattr(self.owner, "model", None) or self.owner
        for i, base in enumerate(bn_buffer_names(self.gin_layers)):
            obj = inner
            for p in base.split("."):
                obj = obj[int(p)] if p.isdigit() else getattr(obj, p)
            for j, attr in enumerate(("running_mean", "running_var")):
                buf = getattr(obj, attr)
                v = self.engine.bn_running[i, j]
                if buf.data_ptr() != v.data_ptr():
                    v.copy_(buf.data.to(device))
                    buf.data = v
        self._bn_modules = inner
        return params


def _check_composed_width(encoder, hidden_dim):
    if encoder != "GIN" and int(hidden_dim) not in (64, 128):
        raise NotImplementedError("--encoder %s runs at --dims 64 or 128 on the B200 path" % encoder)


def _check_args(args, encoder, allowed=("GIN",)):
    if encoder not in allowed:
        # the reference's own unknown-encoder branch (models.py:585-587); Transformer is outside SURVEY section 8
        print("scgib_b200: --encoder %s is not implemented on the B200 path for this class (available: %s)" % (encoder, ", ".join(allowed)))
        raise SystemExit()
    if getattr(args, "readout_f", "sum") != "sum" or getattr(args, "recons_type", "adj") not in ("adj", "logM") or \
            not getattr(args, "useAtt", 1):
        raise NotImplementedError("B200 path covers --readout_f sum --recons_type adj|logM --useAtt 1")


def _own_encoders(encoder, in_dim, hidden_dim, gin_layers):
    """Encoder1 / Encoder2 of the fine-tuning / domain-adaptation wrappers: constructed (state-dict keys, RNG draws) and never
    called, with the switch Mainmodel_continue uses (models.py:576-581)."""
    if encoder == "GIN":
        return GIN(in_dim, hidden_dim, gin_layers), GIN(in_dim, hidden_dim, gin_layers)
    from .encoders import make_encoder
    return make_encoder(encoder, in_dim, hidden_dim), make_encoder(encoder, in_dim, hidden_dim)


def _bump_compressor_batches(loaded, B):
    """num_batches_tracked of the loaded compressor.1 after a composed forward: one BatchNorm call per graph (models.py:642)."""
    bn = loaded.compressor[1]
    if bn.training:
        bn.num_batches_tracked += B


def _loaded_encoder_kind(loaded):
    """The encoders a fine-tuning / domain-adaptation forward runs are the LOADED module's (``self.model.Encoder1``,
    models.py:508, 262), whatever the wrapper's own ``encoder`` argument: after domain adaptation that is the adapter's own
    encoders (SURVEY 3.1).  They select the path: the fused GIN engine or the operator-composed GraphSAGE / GCN step."""
    return getattr(loaded.Encoder1, "kind", "GIN")


class _HotPathMixin:
    """forward / extract_features shared by Mainmodel and Mainmodel_continue."""

    def _device_batch(self, batch_g, batch_x, flatten_batch_subgraphs, device, t_override=None):
        g = batch_g if batch_g.device == torch.device(device) else batch_g.to(device)
        ego = flatten_batch_subgraphs
        if not isinstance(ego, EgoBatch):
            raise TypeError("flatten_batch_subgraphs must be an scgib_b200.graph.EgoBatch (khop_ego_batch)")
        if ego.device != g.device:
            ego = ego.to(g.device)
        x = None if batch_x is None else batch_x.to(g.device).float()
        # exp_pretraining.py:312 already applied F.normalize to batch_x: use it as given
        b = DeviceBatch(g, ego, x, normalize_x=False, t_override=t_override)
        b.eval_mode = not self.training              # model.eval(): running statistics in every BatchNorm (forward only)
        if getattr(self, "recons_type", "adj") == "logM":      # models.py:693-694; the k-step matrices are computed on the GPU
            b.recon_logm_steps = int(self.k_transition)
        return b

    def _noise(self, N, device):
        # reference: gate noise from the CPU generator (models.py:599), feature noise on the device (models.py:650).
        # Both are drawn on the device here (the CPU draw + copy costs ~0.3 ms per step at B = 4096 and the reference's
        # per-graph CPU stream is not reproducible from a batched draw anyway); SCGIB_CPU_GATE_NOISE=1 restores the CPU draw.
        H = int(self.hidden_dim)
        if _CPU_GATE_NOISE:
            return torch.rand(N).to(device, non_blocking=True), torch.rand(N, H, device=device)
        return torch.rand(N, device=device), torch.rand(N, H, device=device)

    def _composed_inputs(self, batch_g, flatten_batch_subgraphs, device):
        g = batch_g if batch_g.device == torch.device(device) else batch_g.to(device)
        ego = flatten_batch_subgraphs
        if not isinstance(ego, EgoBatch):
            raise TypeError("flatten_batch_subgraphs must be an scgib_b200.graph.EgoBatch (khop_ego_batch)")
        if ego.device != g.device:
            ego = ego.to(g.device)
        if g.device.type != "cuda":
            raise RuntimeError("S-CGIB B200 path: the model must be on a CUDA device (no CPU fallback)")
        return g, ego

    def _forward_composed(self, batch_g, batch_x, flatten_batch_subgraphs, device):
        """--encoder GraphSAGE / GCN: the step composed from operator kernels (encoders.py)."""
        from . import encoders
        if not self.training:
            raise NotImplementedError("model.eval() forward with --encoder GraphSAGE / GCN: the pre-training losses are built for "
                                      "training mode (eval-mode features: extract_features, Mainmodel_finetuning)")
        g, ego = self._composed_inputs(batch_g, flatten_batch_subgraphs, device)
        x = batch_x.to(g.device).float().contiguous()
        gate_u, feat_u = self._noise(x.shape[0], g.device)
        names = encoders.composed_param_names(self)
        kl, con, rec = encoders.ComposedPretrainFn.apply(self, g, ego, x, gate_u.contiguous(), feat_u.contiguous(), names,
                                                         *[encoders.resolve_param(self, n) for n in names])
        _bump_compressor_batches(encoders.inner_of(self), g.batch_size)
        return None, kl, con, rec

    def forward(self, batch_g, batch_x, flatten_batch_subgraphs, batch_logMs, x_subs, current_epoch, edge_index,
                k_transition, device, batch_size=16):
        """reference models.py:662-700 / 1158-1195 -> (None, KL_Loss, contrastive_loss, reconstruction_loss)."""
        self.batch_size = batch_size
        self.device = device
        if batch_size < batch_g.batch_size:
            raise NotImplementedError("batched_semi_loss with batch_size < number of graphs (never the case in the CLI)")
        if getattr(self, "encoder_kind", "GIN") != "GIN":
            return self._forward_composed(batch_g, batch_x, flatten_batch_subgraphs, device)
        params = self._bridge.sync(device)
        self._bridge.training = self.training
        b = self._device_batch(batch_g, batch_x, flatten_batch_subgraphs, device)
        gate_u, feat_u = self._noise(b.N, b.g.device)
        kl, con, rec = _PretrainFn.apply(self._bridge, b, gate_u, feat_u, *params)
        if self.training:
            self._bump_batches_tracked(b.B)
        return None, kl, con, rec

    def _bump_batches_tracked(self, B):
        inner = self._bridge._bn_modules
        for enc in (inner.Encoder1, inner.Encoder2):
            for bn in enc.batch_norms:
                bn.num_batches_tracked += 1
        inner.compressor[1].num_batches_tracked += B     # one BatchNorm call per graph (models.py:642)

    @torch.no_grad()
    def extract_features(self, nodes_list, batch_g, batch_x, flatten_batch_subgraphs, x_subs, device):
        """reference models.py:702-750 (forward only here): ``batch_x`` is already transfer_d'ed [N, d_transfer].
        Returns (interaction_map [N,2d], KL_tensor, noisy_node_feature [N,d], graph_features_readout [B,d])."""
        if getattr(self, "encoder_kind", "GIN") != "GIN":
            from . import encoders
            g, ego = self._composed_inputs(batch_g, flatten_batch_subgraphs, device)
            gate_u, feat_u = self._noise(g.num_nodes(), g.device)
            out, _ = encoders.composed_features(self, g, ego, batch_x.to(g.device).float().contiguous(), gate_u.contiguous(),
                                                feat_u.contiguous())
            return out["interaction_map"], out["kl"].clone(), out["noisy"], out["graph_readout"]
        br = getattr(self, "_bridge", None) or _Bridge(self, self.in_dim_raw, self.gin_layers)
        self._bridge = br
        br.sync(device)
        b = self._device_batch(batch_g, None, flatten_batch_subgraphs, device, t_override=batch_x.to(device))
        gate_u, feat_u = self._noise(b.N, b.g.device)
        losses, emb = br.engine.forward(b, gate_u, feat_u, want=True, update_running=self.training)
        self.graph_features = None
        return emb["interaction_map"], losses[0:1].clone(), emb["noisy"], emb["graph_readout"]


class Mainmodel(_HotPathMixin, nn.Module):
    """reference models.py:546-782.  Construction order follows the reference so a seeded default init gives the same
    weights; the modules the default configuration never uses (fc1, embedding_h, reduce_d, s2s, reconstructX) are kept
    for state-dict compatibility."""

    def __init__(self, args, in_dim, hidden_dim, num_layers, num_heads, k_transition, encoder):
        super().__init__()
        _check_args(args, encoder, allowed=("GIN", "GraphSAGE", "GCN"))
        _check_composed_width(encoder, hidden_dim)
        self.encoder_kind = encoder
        self.tau = 1.0
        self.recons_type = args.recons_type
        self.useAtt = args.useAtt
        self.readout = args.readout_f
        self.hidden_dim = hidden_dim
        self.k_transition = k_transition
        self.gin_layers = int(getattr(args, "gin_layers", DEFAULT_GIN_LAYERS))
        self.act_dtype = getattr(args, "dtype", "fp32")      # "bf16": bf16 activations in the GIN encoders (--dtype bf16)
        self.in_dim_raw = in_dim
        self.fc1 = nn.Linear(hidden_dim, 1)
        self.in_dim = args.d_transfer
        self.transfer_d = nn.Linear(in_dim, self.in_dim, bias=False)
        self.embedding_h = nn.Linear(self.in_dim, hidden_dim, bias=False)
        self.attn_layer = nn.Linear(self.hidden_dim * 2, 1)
        self.reduce_d = nn.Linear(2 * self.hidden_dim, self.hidden_dim)
        self.device = args.device
        self.s2s = _Set2SetParams(hidden_dim, 2, 1)
        self.reconstructX = nn.Sequential(nn.Linear(self.hidden_dim, self.in_dim))
        self.MLP = nn.Sequential(nn.Linear(2 * self.hidden_dim, self.hidden_dim), nn.ReLU(),
                                 nn.Linear(self.hidden_dim, self.hidden_dim))
        if encoder == "GIN":
            self.Encoder1 = GIN(self.in_dim, hidden_dim, self.gin_layers)
            self.Encoder2 = GIN(self.in_dim, hidden_dim, self.gin_layers)
        else:                       # models.py:576-581: composed from operator kernels, see encoders.py
            from .encoders import make_encoder
            self.Encoder1 = make_encoder(encoder, self.in_dim, hidden_dim)
            self.Encoder2 = make_encoder(encoder, self.in_dim, hidden_dim)
        self.compressor = nn.Sequential(nn.Linear(self.hidden_dim, self.hidden_dim), nn.BatchNorm1d(self.hidden_dim),
                                        nn.ReLU(), nn.Linear(self.hidden_dim, 1))
        self._bridge = _Bridge(self, in_dim, self.gin_layers) if encoder == "GIN" else None

    def __getstate__(self):     # torch.save(model) (exp_pretraining.py:107): drop the engine, keep plain tensors
        st = self.__dict__.copy()
        st["_bridge"] = None
        st.pop("_composed_last", None)
        return st

    def __setstate__(self, st):
        self.__dict__.update(st)
        for p in self.parameters():
            p.data = p.data.clone()
        self._bridge = _Bridge(self, self.in_dim_raw, self.gin_layers) if getattr(self, "encoder_kind", "GIN") == "GIN" else None


class Mainmodel_continue(_HotPathMixin, nn.Module):
    """reference models.py:1010-1276: wraps a pickled model (``torch.load(cp_filename)``), owns a new transfer_d and
    MLP head and trains them together with the LOADED module's encoders/compressor/attention (models.py:1167)."""

    def __init__(self, args, in_dim, hidden_dim, num_layers, num_heads, k_transition, num_classes, cp_filename, encoder):
        super().__init__()
        _check_args(args, encoder, allowed=("GIN", "GraphSAGE", "GCN"))
        _check_composed_width(encoder, hidden_dim)
        self.encoder_kind = encoder
        self.tau = 1.0
        self.readout = args.readout_f
        self.gin_layers = int(getattr(args, "gin_layers", DEFAULT_GIN_LAYERS))
        self.act_dtype = getattr(args, "dtype", "fp32")      # "bf16": bf16 activations in the GIN encoders (--dtype bf16)
        self.in_dim_raw = in_dim
        self.s2s = _Set2SetParams(hidden_dim, 2, 1)
        self.s2s_rev = _Set2SetParams(in_dim, 2, 1)
        self.in_dim = args.d_transfer
        self.transfer_d = nn.Linear(in_dim, self.in_dim, bias=False)
        self.recons_type = args.recons_type
        self.batch_size = args.batch_size
        self.useAtt = args.useAtt
        self.embedding_h = nn.Linear(self.in_dim, hidden_dim, bias=False)
        self.hidden_dim = hidden_dim
        self.k_transition = k_transition
        self.reduce_d = nn.Linear(2 * self.hidden_dim, self.hidden_dim)
        self.attn_layer = nn.Linear(2 * self.hidden_dim, 1)
        self.num_nodes = -1
        self.device = args.device
        self.r_transfer_d = nn.Sequential(nn.Linear(2 * self.hidden_dim, self.hidden_dim), nn.ReLU(),
                                          nn.Linear(self.hidden_dim, in_dim * 2))
        out_dim = 1 if getattr(args, "task", "graph_classification") == "graph_regression" else num_classes
        self.predict = nn.Sequential(nn.Linear(2 * self.hidden_dim, self.hidden_dim), nn.ReLU(),
                                     nn.Linear(self.hidden_dim, out_dim))
        self.MLP = nn.Sequential(nn.Linear(2 * self.hidden_dim, self.hidden_dim), nn.ReLU(),
                                 nn.Linear(self.hidden_dim, self.hidden_dim))
        if encoder == "GIN":
            self.Encoder1 = GIN(self.in_dim, hidden_dim, self.gin_layers)
            self.Encoder2 = GIN(self.in_dim, hidden_dim, self.gin_layers)
        else:
            from .encoders import make_encoder
            self.Encoder1 = make_encoder(encoder, self.in_dim, hidden_dim)
            self.Encoder2 = make_encoder(encoder, self.in_dim, hidden_dim)
        self.model = torch.load(cp_filename, map_location=args.device, weights_only=False)
        for p in self.model.parameters():
            p.requires_grad = True
        self.compressor = nn.Sequential(nn.Linear(self.hidden_dim, self.hidden_dim), nn.BatchNorm1d(self.hidden_dim),
                                        nn.ReLU(), nn.Linear(self.hidden_dim, 1))
        self.reconstructX = nn.Sequential(nn.Linear(self.hidden_dim, self.hidden_dim), nn.ReLU(),
                                          nn.Linear(self.hidden_dim, in_dim))
        self._bridge = _Bridge(self, in_dim, self.gin_layers) if encoder == "GIN" else None

    __getstate__ = Mainmodel.__getstate__
    __setstate__ = Mainmodel.__setstate__


class _FinetuneFn(torch.autograd.Function):
    """transfer_d -> model.extract_features -> MLP -> Set2Set -> predict (-> sigmoid) as one autograd node."""

    @staticmethod
    def forward(ctx, owner, batch, gate_u, feat_u, *params):
        eng, head = owner._bridge.engine, owner._head
        Z = eng.forward_features(batch, gate_u, feat_u, update_running=owner.training)
        scores = head.forward(Z, batch.g.graph_ptr)
        ctx.owner = owner
        ctx.params = params
        ctx.serial = (eng.fwd_serial, head.fwd_serial)
        return scores

    @staticmethod
    def backward(ctx, g_scores):
        owner = ctx.owner
        eng, head = owner._bridge.engine, owner._head
        _check_serial("Mainmodel_finetuning", eng, ctx.serial[0])
        _check_serial("Mainmodel_finetuning (head)", head, ctx.serial[1])
        _detach_aliased_grads(ctx.params, eng.grads)
        _detach_aliased_grads(ctx.params, head.grads)
        gZ = head.backward(g_scores)
        eng.extract_backward(gZ)
        gv, hv = eng.grad_views(), head.views(grads=True)
        grads = [gv.pop(n) for n in owner._bridge.slot_names] + [hv.pop(n) for n in FT_NAMES]
        return (None, None, None, None) + tuple(grads)


class Mainmodel_finetuning(nn.Module):
    """reference models.py:358-543: fine-tuning wrapper around a pickled pre-trained model.  Owns transfer_d, MLP, the
    Set2Set readout and the predict head; the loaded ``self.model`` supplies the encoders, compressor and attention layer
    through ``extract_features`` with only the ``layers.2`` parameters left trainable (models.py:424-435).
    ``forward`` returns ``(scores, 0, 0, 0)`` like the reference; the loss helpers are the reference's."""

    def __init__(self, args, in_dim, hidden_dim, num_layers, num_heads, k_transition, num_classes, cp_filename, encoder):
        super().__init__()
        _check_args(args, encoder, allowed=("GIN", "GraphSAGE", "GCN"))
        _check_composed_width(encoder, hidden_dim)
        self.tau = 1.0
        self.dataset = args.dataset
        self.readout = args.readout_f
        self.gin_layers = int(getattr(args, "gin_layers", DEFAULT_GIN_LAYERS))
        self.act_dtype = getattr(args, "dtype", "fp32")      # "bf16": bf16 activations in the GIN encoders (--dtype bf16)
        self.in_dim_raw = in_dim
        self.s2s = _Set2SetParams(hidden_dim, 2, 1)
        self.in_dim = args.d_transfer
        self.transfer_d = nn.Linear(in_dim, self.in_dim, bias=False)
        self.batch_size = args.batch_size
        self.useAtt = args.useAtt
        self.embedding_h = nn.Linear(self.in_dim, hidden_dim, bias=False)
        self.hidden_dim = hidden_dim
        self.k_transition = k_transition
        self.reduce_d = nn.Linear(2 * self.hidden_dim, self.hidden_dim)
        self.attn_layer = nn.Linear(2 * self.hidden_dim, 1)
        self.num_nodes = -1
        self.device = args.device
        self.tasks = ['ZINC', 'Peptides-struct', 'FreeSolv', 'ESOL']
        if args.task == "graph_regression":
            out_dim = 1
        elif args.task == "graph_classification":
            out_dim = num_classes
        else:
            raise NotImplementedError("task must be graph_regression or graph_classification (models.py:385-399)")
        self.predict = nn.Sequential(nn.Linear(2 * self.hidden_dim, self.hidden_dim), nn.ReLU(),
                                     nn.Linear(self.hidden_dim, out_dim))
        self.MLP = nn.Sequential(nn.Linear(2 * self.hidden_dim, self.hidden_dim), nn.ReLU(),
                                 nn.Linear(self.hidden_dim, self.hidden_dim))
        self.Encoder1, self.Encoder2 = _own_encoders(encoder, self.in_dim, hidden_dim, self.gin_layers)
        print("Loading pre-trained model .pt  ... ")
        self.model = torch.load(cp_filename, map_location=args.device, weights_only=False)
        for name, para in self.model.named_parameters():     # models.py:424-435: the last list entry decides
            para.requires_grad = "layers.2" in name          # (no GraphSAGE / GCN name contains it: all frozen)
        self.compressor = nn.Sequential(nn.Linear(self.hidden_dim, self.hidden_dim), nn.BatchNorm1d(self.hidden_dim),
                                        nn.ReLU(), nn.Linear(self.hidden_dim, 1))
        self.encoder_kind = _loaded_encoder_kind(self.model)
        _check_composed_width(self.encoder_kind, hidden_dim)
        self._bridge = _Bridge(self, in_dim, self.gin_layers) if self.encoder_kind == "GIN" else None
        self._head = None

    def __getstate__(self):
        st = Mainmodel.__getstate__(self)
        st["_head"] = None                      # engine objects (ctypes handles, device buffers) are rebuilt on demand
        return st

    def __setstate__(self, st):
        Mainmodel.__setstate__(self, st)
        self._head = None

    _device_batch = _HotPathMixin._device_batch
    _noise = _HotPathMixin._noise
    _composed_inputs = _HotPathMixin._composed_inputs

    def _sync_head(self, device):
        device = torch.device(device)
        sigmoid = self.dataset not in self.tasks              # models.py:516-520
        if self._head is None or self._head.device != device:
            self._head = FinetuneHead(self.hidden_dim, self.predict[2].out_features, n_iters=self.s2s.n_iters,
                                      sigmoid=sigmoid, device=device)
        views = self._head.views()
        params = []
        for name in FT_NAMES:
            obj = self
            parts = name.split(".")
            for p in parts[:-1]:
                obj = obj[int(p)] if p.isdigit() else getattr(obj, p)
            prm = getattr(obj, parts[-1])
            v = views[name]
            if prm.data_ptr() != v.data_ptr():
                v.copy_(prm.data.to(device).reshape(v.shape))
                prm.data = v
            params.append(prm)
        return params

    def forward(self, batch_g, batch_x, flatten_batch_subgraphs, x_subs, current_epoch, edge_index, k_transition,
                device, batch_size=2):
        """reference models.py:501-520 -> (scores [B,C], 0, 0, 0)."""
        self.batch_size = batch_size
        self.device = device
        if getattr(self, "encoder_kind", "GIN") != "GIN":         # (wrappers pickled before encoder_kind existed are GIN)
            return self._forward_composed(batch_g, batch_x, flatten_batch_subgraphs, device), 0, 0, 0
        params = self._bridge.sync(device) + self._sync_head(device)
        self._bridge.training = self.training
        b = self._device_batch(batch_g, batch_x, flatten_batch_subgraphs, device)
        gate_u, feat_u = self._noise(b.N, b.g.device)
        scores = _FinetuneFn.apply(self, b, gate_u, feat_u, *params)
        if self.training:
            _HotPathMixin._bump_batches_tracked(self, b.B)
        return scores, 0, 0, 0

    def _forward_composed(self, batch_g, batch_x, flatten_batch_subgraphs, device):
        """GraphSAGE / GCN encoders in the loaded module: the feature path composed from operator kernels (encoders.py)."""
        from . import encoders
        g, ego = self._composed_inputs(batch_g, flatten_batch_subgraphs, device)
        head_params = self._sync_head(device)
        x = batch_x.to(g.device).float().contiguous()
        gate_u, feat_u = self._noise(x.shape[0], g.device)
        names = encoders.trainable_param_names(self)
        scores = encoders.ComposedFinetuneFn.apply(self, g, ego, x, gate_u.contiguous(), feat_u.contiguous(), names,
                                                   *[encoders.resolve_param(self, n) for n in names], *head_params)
        _bump_compressor_batches(self.model, g.batch_size)
        return scores

    # loss helpers: reference models.py:522-543 (operate on the [B,C] scores)
    def loss(self, scores, targets):
        return nn.BCELoss()(scores.float(), targets.float())

    def loss_CrossEntropy(self, scores, targets):
        return nn.CrossEntropyLoss()(scores.to(torch.float32), targets.squeeze(dim=-1))

    def loss_RMSE(self, scores, targets):
        return torch.sqrt(nn.MSELoss()(scores, targets))

    def BCEWithLogitsLoss(self, scores, targets):
        return nn.BCEWithLogitsLoss()(scores, targets)

    def lossMAE(self, scores, targets):
        return nn.L1Loss()(scores, targets)


DA_NAMES = ["s2s.lstm.weight_ih_l0", "s2s.lstm.weight_hh_l0", "s2s.lstm.bias_ih_l0", "s2s.lstm.bias_hh_l0",
            "r_transfer_d.0.weight", "r_transfer_d.0.bias", "r_transfer_d.2.weight", "r_transfer_d.2.bias"]
REV_NAMES = ["weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0"]


class _DomainAdaptFn(torch.autograd.Function):
    """-> (r_transfer_d(s2s(MLP(extract_features))) [B, 2 in_dim], s2s_rev(x) [B, 2 in_dim])."""

    @staticmethod
    def forward(ctx, owner, batch, gate_u, feat_u, x_norm, *params):
        eng, head, rev = owner._bridge.engine, owner._head, owner._rev
        Z = eng.forward_features(batch, gate_u, feat_u, update_running=owner.training)
        rec = head.forward(Z, batch.g.graph_ptr)
        org = rev.forward(x_norm, batch.g.graph_ptr)
        ctx.owner = owner
        ctx.params = params
        ctx.serial = (eng.fwd_serial, head.fwd_serial, rev.head.fwd_serial)
        return rec, org

    @staticmethod
    def backward(ctx, g_rec, g_org):
        owner = ctx.owner
        eng, head, rev = owner._bridge.engine, owner._head, owner._rev
        _check_serial("Mainmodel_domainadapt", eng, ctx.serial[0])
        _check_serial("Mainmodel_domainadapt (head)", head, ctx.serial[1])
        _check_serial("Mainmodel_domainadapt (s2s_rev)", rev.head, ctx.serial[2])
        _detach_aliased_grads(ctx.params, eng.grads)
        _detach_aliased_grads(ctx.params, head.grads)
        gZ = head.backward(g_rec)
        eng.extract_backward(gZ)
        gv, hv = eng.grad_views(), head.views(grads=True)
        grads = [gv.pop(n) for n in owner._bridge.slot_names] + [hv.pop(n) for n in FT_NAMES]
        grads += list(rev.backward(g_org))
        return (None, None, None, None, None) + tuple(grads)


class Mainmodel_domainadapt(nn.Module):
    """reference models.py:107-355: domain adaptation of a pre-trained model to a new dataset's feature space.
    ``forward(...) -> X_loss = sum((r_transfer_d(s2s(MLP(extract_features))) - s2s_rev(batch_x))**2)`` (models.py:254-275);
    every parameter of the loaded model is trainable (models.py:176-178).  Both Set2Set readouts and the r_transfer_d
    MLP run in the fine-tuning head kernels (csrc/finetune_kernels.cu); the squared-error sum over the [B, 2 in_dim]
    outputs is the reference's one-liner."""

    def __init__(self, args, in_dim, hidden_dim, num_layers, num_heads, k_transition, num_classes, cp_filename, encoder):
        super().__init__()
        _check_args(args, encoder, allowed=("GIN", "GraphSAGE", "GCN"))
        _check_composed_width(encoder, hidden_dim)
        self.tau = 1.0
        self.readout = args.readout_f
        self.gin_layers = int(getattr(args, "gin_layers", DEFAULT_GIN_LAYERS))
        self.act_dtype = getattr(args, "dtype", "fp32")      # "bf16": bf16 activations in the GIN encoders (--dtype bf16)
        self.in_dim_raw = in_dim
        self.s2s = _Set2SetParams(hidden_dim, 2, 1)
        self.s2s_rev = _Set2SetParams(in_dim, 2, 1)
        self.in_dim = args.d_transfer
        self.transfer_d = nn.Linear(in_dim, self.in_dim, bias=False)
        self.batch_size = args.batch_size
        self.useAtt = args.useAtt
        self.embedding_h = nn.Linear(self.in_dim, hidden_dim, bias=False)
        self.hidden_dim = hidden_dim
        self.k_transition = k_transition
        self.reduce_d = nn.Linear(2 * self.hidden_dim, self.hidden_dim)
        self.attn_layer = nn.Linear(2 * self.hidden_dim, 1)
        self.num_nodes = -1
        self.device = args.device
        self.r_transfer_d = nn.Sequential(nn.Linear(2 * self.hidden_dim, self.hidden_dim), nn.ReLU(),
                                          nn.Linear(self.hidden_dim, in_dim * 2))
        out_dim = 1 if getattr(args, "task", "graph_classification") == "graph_regression" else num_classes
        self.predict = nn.Sequential(nn.Linear(2 * self.hidden_dim, self.hidden_dim), nn.ReLU(),
                                     nn.Linear(self.hidden_dim, out_dim))
        self.MLP = nn.Sequential(nn.Linear(2 * self.hidden_dim, self.hidden_dim), nn.ReLU(),
                                 nn.Linear(self.hidden_dim, self.hidden_dim))
        self.Encoder1, self.Encoder2 = _own_encoders(encoder, self.in_dim, hidden_dim, self.gin_layers)
        print("Loading pre-trained model .pt  ... ")
        self.model = torch.load(cp_filename, map_location=args.device, weights_only=False)
        for p in self.model.parameters():
            p.requires_grad = True
        self.compressor = nn.Sequential(nn.Linear(self.hidden_dim, self.hidden_dim), nn.BatchNorm1d(self.hidden_dim),
                                        nn.ReLU(), nn.Linear(self.hidden_dim, 1))
        self.reconstructX = nn.Sequential(nn.Linear(self.hidden_dim, self.hidden_dim), nn.ReLU(),
                                          nn.Linear(self.hidden_dim, in_dim))
        self.encoder_kind = _loaded_encoder_kind(self.model)
        _check_composed_width(self.encoder_kind, hidden_dim)
        self._bridge = _Bridge(self, in_dim, self.gin_layers) if self.encoder_kind == "GIN" else None
        self._head = None
        self._rev = None

    def __getstate__(self):
        st = Mainmodel.__getstate__(self)
        st["_head"] = None
        st["_rev"] = None
        return st

    def __setstate__(self, st):
        Mainmodel.__setstate__(self, st)
        self._head = None
        self._rev = None

    _device_batch = _HotPathMixin._device_batch
    _noise = _HotPathMixin._noise
    _composed_inputs = _HotPathMixin._composed_inputs

    def _sync_heads(self, device):
        device = torch.device(device)
        if self._head is None or self._head.device != device:
            self._head = FinetuneHead(self.hidden_dim, 2 * self.in_dim_raw, n_iters=self.s2s.n_iters, sigmoid=False,
                                      device=device)
            self._rev = PaddedSet2Set(self.in_dim_raw, n_iters=self.s2s_rev.n_iters, device=device)
        views = self._head.views()
        params = []
        for name, slot in zip(DA_NAMES, FT_NAMES):          # r_transfer_d sits in the head's predict slots
            obj = self
            parts = name.split(".")
            for p in parts[:-1]:
                obj = obj[int(p)] if p.isdigit() else getattr(obj, p)
            prm = getattr(obj, parts[-1])
            v = views[slot]
            if prm.data_ptr() != v.data_ptr():
                v.copy_(prm.data.to(device).reshape(v.shape))
                prm.data = v
            params.append(prm)
        rev_params = [getattr(self.s2s_rev.lstm, n) for n in REV_NAMES]
        self._rev.set_params(*[p.data.to(device) for p in rev_params])
        return params + rev_params

    def forward(self, batch_g, batch_x, flatten_batch_subgraphs, batch_logMs, x_subs, current_epoch, edge_index,
                k_transition, device, batch_size=16):
        """reference models.py:254-269 -> X_loss (scalar)."""
        self.batch_size = batch_size
        self.device = device
        if getattr(self, "encoder_kind", "GIN") != "GIN":
            return self._forward_composed(batch_g, batch_x, flatten_batch_subgraphs, device)
        params = self._bridge.sync(device) + self._sync_heads(device)
        self._bridge.training = self.training
        b = self._device_batch(batch_g, batch_x, flatten_batch_subgraphs, device)
        gate_u, feat_u = self._noise(b.N, b.g.device)
        rec, org = _DomainAdaptFn.apply(self, b, gate_u, feat_u, b.x, *params)
        if self.training:
            _HotPathMixin._bump_batches_tracked(self, b.B)
        return self.loss_X(org, rec)

    def _forward_composed(self, batch_g, batch_x, flatten_batch_subgraphs, device):
        """GraphSAGE / GCN encoders in the loaded module: the feature path composed from operator kernels (encoders.py);
        every parameter of the loaded model is trainable."""
        from . import encoders
        g, ego = self._composed_inputs(batch_g, flatten_batch_subgraphs, device)
        head_params = self._sync_heads(device)
        x = batch_x.to(g.device).float().contiguous()
        gate_u, feat_u = self._noise(x.shape[0], g.device)
        names = encoders.trainable_param_names(self)
        rec, org = encoders.ComposedDomainAdaptFn.apply(self, g, ego, x, gate_u.contiguous(), feat_u.contiguous(), x, names,
                                                        *[encoders.resolve_param(self, n) for n in names], *head_params)
        _bump_compressor_batches(self.model, g.batch_size)
        return self.loss_X(org, rec)

    def loss_X(self, batch_x_org, interaction_map):
        return torch.sum((interaction_map - batch_x_org) ** 2)
