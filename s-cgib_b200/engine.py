"""PretrainEngine - host driver of the S-CGIB pre-training step on one GPU.

Owns the flat parameter / gradient / Adam-state buffers and the kernel workspace and calls the
C ABI (include/scgib.h).  One forward = one C call (~30 kernel launches), one backward = one C call;
there is no per-graph Python loop and no host synchronisation inside a step.

Reference path replaced: exp_pretraining.py:300-324 (train_epoch_pre_training body) and
models.py:662-700 / 1158-1195 (Mainmodel(.continue).forward).
"""
from __future__ import annotations

import ctypes
from collections import OrderedDict
from typing import Dict, Optional

import torch

from . import _lib
from .graph import BatchedGraph, EgoBatch, EgoWorkspace, khop_ego_batch

HID = 64
_VALIDATE = __import__("os").environ.get("SCGIB_VALIDATE", "0") == "1"     # per-batch input validation (one extra host read)


def param_names(gin_layers: int):
    """Reference state-dict name of every slot of the flat parameter buffer (INTEGRATION.md)."""
    names = ["MLP.0.weight", "MLP.0.bias", "MLP.2.weight", "MLP.2.bias",
             "compressor.0.weight", "compressor.0.bias", "compressor.1.weight", "compressor.1.bias",
             "compressor.3.weight", "compressor.3.bias", "attn_layer.weight", "attn_layer.bias", "transfer_d.weight"]
    for e in (1, 2):
        for l in range(gin_layers):
            p = "Encoder%d." % e
            names += [p + "ginlayers.%d.apply_func.mlp.0.weight" % l, p + "ginlayers.%d.apply_func.mlp.0.bias" % l,
                      p + "ginlayers.%d.apply_func.mlp.2.weight" % l, p + "ginlayers.%d.apply_func.mlp.2.bias" % l,
                      p + "batch_norms.%d.weight" % l, p + "batch_norms.%d.bias" % l]
    return names


def param_shapes(in_dim: int, gin_layers: int, hidden: int = HID, d_transfer: int = 32):
    H, D = hidden, d_transfer
    shapes = [(H, 2 * H), (H,), (H, H), (H,), (H, H), (H,), (H,), (H,), (1, H), (1,),
              (1, 2 * H), (1,), (D, in_dim)]
    for _e in range(2):
        for l in range(gin_layers):
            shapes += [(H, D if l == 0 else H), (H,), (H, H), (H,), (H,), (H,)]
    return shapes


def bn_buffer_names(gin_layers: int):
    names = []
    for e in (1, 2):
        for l in range(gin_layers):
            names.append("Encoder%d.batch_norms.%d" % (e, l))
    names.append("compressor.1")
    return names


class DeviceBatch:
    """Everything one step needs, resident on the device: parent CSR, ego CSR, features, noise."""

    def __init__(self, g: BatchedGraph, ego: EgoBatch, x: torch.Tensor, normalize_x: bool = True, t_override=None):
        self.g, self.ego, self.x, self.normalize_x = g, ego, (None if x is None else x.contiguous()), normalize_x
        self.t_override = None if t_override is None else t_override.contiguous().float()
        self.recon_logm_steps = 0        # k >= 1: --recons_type logM with k-step matrices (models.py:770-782)
        self.eval_mode = False           # model.eval(): BatchNorm layers use their running statistics (forward only)
        self.B, self.N, self.E = g.batch_size, g.num_nodes(), g.num_edges()
        self.Ns, self.Es = ego.num_nodes(), ego.num_edges()

    def c_struct(self, gate_u, feat_u):
        b = _lib.Batch()
        b.struct_size = ctypes.sizeof(_lib.Batch)
        b.B, b.N, b.E, b.Ns, b.Es = self.B, self.N, self.E, self.Ns, self.Es
        g, e = self.g, self.ego
        b.graph_ptr, b.indptr, b.indices = g.graph_ptr.data_ptr(), g.indptr.data_ptr(), g.indices.data_ptr()
        b.ego_ptr, b.ego_nodes, b.ego_seed = e.ego_ptr.data_ptr(), e.ego_nodes.data_ptr(), e.ego_seed.data_ptr()
        b.sub_indptr, b.sub_indices = e.sub_indptr.data_ptr(), e.sub_indices.data_ptr()
        b.x, b.normalize_x = (self.x.data_ptr() if self.x is not None else None), int(self.normalize_x)
        b.t_override = None if self.t_override is None else self.t_override.data_ptr()
        b.gate_u, b.feat_u = gate_u.data_ptr(), feat_u.data_ptr()
        b.recon_logm_steps = int(self.recon_logm_steps)
        b.eval_mode = int(bool(self.eval_mode))
        return b

    def algorithmic_bytes(self, gin_layers=4, F=9, s=4, hidden=HID, d_transfer=32):   # s = bytes per activation element (2 in bf16 mode)
        """SURVEY.md §8(d) 'algorithmic bytes per training step' evaluated on this batch's actual sizes."""
        N, E, Ns, Es, d, dt = self.N, self.E, self.Ns, self.Es, hidden, d_transfer

        def enc(V, D):
            tot = 0
            for l in range(gin_layers):
                din = dt if l == 0 else d
                tot += V * (din + d) * s + 4 * (V + 1 + D)
            return tot
        fwd = enc(N, E) + enc(Ns, Es) + N * F * 4 + Ns * 4 + N * dt * s + (Ns + N) * d * s + 2 * N * d * s + \
            (N + 1) * d * s + 2 * N * d * s + N * d * s + 4 * (N + 1 + E) + 4 * d * s
        ego = 4 * (N + 1 + E) + 4 * (2 * Ns + 1 + Es + N + 1)
        return 3 * fwd + ego


class PretrainEngine:
    def __init__(self, in_dim: int, gin_layers: int = 4, hidden: int = 64, d_transfer: int = 32,
                 device="cuda:0", seed: Optional[int] = None, dtype: str = "fp32"):
        """``dtype``: "fp32" (reference precision, 1e-5) or "bf16" (the GIN encoders keep their activations in bf16 and run
        single-pass bf16 tensor-core MLPs; parameters, gradients, optimiser state and all outputs stay fp32; 2e-2)."""
        self.lib = _lib.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("PretrainEngine needs a CUDA device: the hot path has no CPU fallback")
        if dtype not in ("fp32", "bf16"):
            raise ValueError("dtype must be 'fp32' or 'bf16'")
        self.dtype = dtype
        self.hidden = int(hidden)
        self.dims = _lib.Dims(int(in_dim), int(d_transfer), int(hidden), int(gin_layers),
                              _lib.ACT_BF16 if dtype == "bf16" else _lib.ACT_F32)
        n = self.lib.scgib_param_slots(ctypes.byref(self.dims))
        if n < 0:
            _lib.check(n, "param_slots")
        off = (ctypes.c_int64 * n)()
        sz = (ctypes.c_int64 * n)()
        self.total = int(self.lib.scgib_param_layout(ctypes.byref(self.dims), off, sz))
        self.offsets, self.sizes = list(off), list(sz)
        self.names = param_names(gin_layers)
        self.shapes = param_shapes(in_dim, gin_layers, self.hidden, int(d_transfer))
        assert len(self.names) == n == len(self.shapes)
        self.params = torch.zeros(self.total, dtype=torch.float32, device=self.device)
        self.grads = torch.zeros_like(self.params)
        self.exp_avg = torch.zeros_like(self.params)
        self.exp_avg_sq = torch.zeros_like(self.params)
        self.bn_running = torch.zeros(2 * gin_layers + 1, 2, hidden, dtype=torch.float32, device=self.device)
        self.bn_running[:, 1] = 1.0
        self.num_batches_tracked = 0
        self.step_count = 0
        self.losses = torch.zeros(4, dtype=torch.float32, device=self.device)
        self._ws = None
        self._loss_scale = (ctypes.c_float * 3)(1.0, 1.0, 1.0)
        self.ego_ws = EgoWorkspace()
        self.recon_logm_steps = 0        # k >= 1: batches made by this engine use --recons_type logM with k-step matrices
        self.fwd_serial = 0              # bumped by every forward: an autograd node of an older forward must not run backward
        self._noise_gen = torch.Generator(device=self.device)
        if seed is not None:
            self._noise_gen.manual_seed(seed)
            self.reset_parameters(seed)
        else:
            # unseeded: follow torch's global seed (torch.manual_seed) and decorrelate data-parallel ranks
            rank = int(__import__("os").environ.get("RANK", "0"))
            self._noise_gen.manual_seed((torch.initial_seed() + 7919 * rank) % (2 ** 63))

    # ---------------------------------------------------------------- parameters
    def views(self) -> "OrderedDict[str, torch.Tensor]":
        out = OrderedDict()
        for name, o, s, shp in zip(self.names, self.offsets, self.sizes, self.shapes):
            out[name] = self.params[o:o + s].view(shp)
        return out

    def grad_views(self):
        out = OrderedDict()
        for name, o, s, shp in zip(self.names, self.offsets, self.sizes, self.shapes):
            out[name] = self.grads[o:o + s].view(shp)
        return out

    def reset_parameters(self, seed=0):
        """nn.Linear / BatchNorm1d default initialisation (kaiming_uniform(a=sqrt(5)), bias U(-1/sqrt(fan_in), ..))."""
        gen = torch.Generator().manual_seed(seed)
        v = self.views()
        for name, t in v.items():
            if "batch_norms" in name or name.startswith("compressor.1"):
                t.fill_(1.0 if name.endswith("weight") else 0.0)
                continue
            wname = name[:-4] + "weight" if name.endswith("bias") else name
            fan_in = v[wname].shape[1]
            bound = 1.0 / fan_in ** 0.5
            t.copy_((torch.rand(t.shape, generator=gen) * 2 - 1) * bound)

    def load_state_dict(self, sd: Dict[str, torch.Tensor], strict=False):
        """Load reference-named tensors (e.g. a state_dict of models.Mainmodel)."""
        v = self.views()
        for name, t in v.items():
            if name in sd:
                t.copy_(sd[name].reshape(t.shape))
            elif strict:
                raise KeyError(name)
        for i, base in enumerate(bn_buffer_names(self.dims.gin_layers)):
            if base + ".running_mean" in sd:
                self.bn_running[i, 0].copy_(sd[base + ".running_mean"])
                self.bn_running[i, 1].copy_(sd[base + ".running_var"])

    def state_dict(self):
        sd = OrderedDict((k, t.detach().clone()) for k, t in self.views().items())
        for i, base in enumerate(bn_buffer_names(self.dims.gin_layers)):
            sd[base + ".running_mean"] = self.bn_running[i, 0].clone()
            sd[base + ".running_var"] = self.bn_running[i, 1].clone()
        return sd

    def checkpoint(self):
        """Everything needed to resume training bit-identically: parameters, BN running statistics, Adam moments and step,
        the noise generator state (the reference checkpoints by pickling the whole module, exp_pretraining.py:103-132,
        and loses the optimiser state; this keeps it)."""
        return dict(params=self.params.detach().clone(), bn_running=self.bn_running.detach().clone(),
                    exp_avg=self.exp_avg.detach().clone(), exp_avg_sq=self.exp_avg_sq.detach().clone(),
                    step_count=self.step_count, num_batches_tracked=self.num_batches_tracked,
                    noise_state=self._noise_gen.get_state(), gin_layers=int(self.dims.gin_layers),
                    in_dim=int(self.dims.in_dim), hidden=self.hidden)

    def restore(self, ck):
        if int(ck["gin_layers"]) != int(self.dims.gin_layers) or int(ck["in_dim"]) != int(self.dims.in_dim) or \
                int(ck.get("hidden", HID)) != self.hidden:
            raise ValueError("checkpoint was written for different model dimensions")
        self.params.copy_(ck["params"])
        self.bn_running.copy_(ck["bn_running"])
        self.exp_avg.copy_(ck["exp_avg"])
        self.exp_avg_sq.copy_(ck["exp_avg_sq"])
        self.step_count, self.num_batches_tracked = int(ck["step_count"]), int(ck["num_batches_tracked"])
        self._noise_gen.set_state(ck["noise_state"].cpu())

    # ---------------------------------------------------------------- data
    def make_batch(self, g: BatchedGraph, k: int = 1, normalize_x: bool = True) -> DeviceBatch:
        """H2D of a host batch (if needed) + on-GPU k-hop ego-net extraction."""
        if g.device != self.device:
            g = g.to(self.device, non_blocking=True)
        if _VALIDATE:
            g.validate()
        ego = khop_ego_batch(g, k, self.ego_ws)
        b = DeviceBatch(g, ego, g.ndata["x"].float(), normalize_x)
        b.recon_logm_steps = self.recon_logm_steps
        return b

    def prefetch_batch(self, g: BatchedGraph, k: int = 1, normalize_x: bool = True, slots: int = 3):
        """Data-loader style pipelining: H2D (if ``g`` is a pinned host batch) and k-hop ego-net extraction of the
        NEXT batch on a side stream while the current step's kernels run.  The one host read of (Ns, Es) waits for the
        side stream only, so the launch queue of the training stream never drains.  Buffers come from a small ring of
        preallocated slots (no allocator traffic in steady state); a slot is reused only after the training stream has
        finished the step that read it.  Pair with ``wait_batch``."""
        if not hasattr(self, "_side"):
            self._side = torch.cuda.Stream(self.device)
            self._slots = [dict(bufs={}, done=None, dev={}) for _ in range(slots)]
            self._slot_i = 0
        slot = self._slots[self._slot_i % len(self._slots)]
        self._slot_i += 1
        train_stream = torch.cuda.current_stream(self.device)
        with torch.cuda.stream(self._side):
            if slot["done"] is not None:
                self._side.wait_event(slot["done"])
            if g.device != self.device:                      # pinned host batch: H2D into the slot's device buffers
                def put(name, t):
                    d = slot["dev"].get(name)
                    if d is None or d.numel() < t.numel() or d.dtype != t.dtype:
                        d = torch.empty(int(t.numel() * 1.25) + 16, dtype=t.dtype, device=self.device)
                        slot["dev"][name] = d
                    v = d[:t.numel()].view(t.shape)
                    v.copy_(t, non_blocking=True)
                    return v
                gd = BatchedGraph.__new__(BatchedGraph)
                gd.graph_ptr, gd.indptr, gd.indices = put("graph_ptr", g.graph_ptr), put("indptr", g.indptr), put("indices", g.indices)
                gd.ndata = {"x": put("x", g.ndata["x"])}
                g = gd
            ego = khop_ego_batch(g, k, self.ego_ws, out=slot["bufs"])
            x = g.ndata["x"]
            if x.dtype != torch.float32:                     # the fp32 copy is allocated on the side stream but read by
                x = x.float()                                # the training stream: keep its block out of the side pool
                x.record_stream(train_stream)                # until that work has run
            b = DeviceBatch(g, ego, x, normalize_x)
            b.recon_logm_steps = self.recon_logm_steps
            b._slot = slot
            ev = torch.cuda.Event()
            ev.record(self._side)
        return b, ev

    def prefetch_ids(self, dataset, ids: torch.Tensor, k: int = 1, normalize_x: bool = True, slots: int = 3):
        """The same pipelining for a dataset resident in HBM (graph.DeviceDataset): H2D of the B molecule ids, GPU-side
        batch assembly and ego-net extraction of the NEXT batch on the side stream.  Pair with ``wait_batch``."""
        if not hasattr(self, "_side"):
            self._side = torch.cuda.Stream(self.device)
            self._slots = [dict(bufs={}, done=None, dev={}) for _ in range(slots)]
            self._slot_i = 0
        slot = self._slots[self._slot_i % len(self._slots)]
        self._slot_i += 1
        with torch.cuda.stream(self._side):
            if slot["done"] is not None:
                self._side.wait_event(slot["done"])
            g = dataset.assemble(ids, out=slot["dev"])
            ego = khop_ego_batch(g, k, self.ego_ws, out=slot["bufs"])
            b = DeviceBatch(g, ego, g.ndata["x"], normalize_x)
            b.recon_logm_steps = self.recon_logm_steps
            b._slot = slot
            ev = torch.cuda.Event()
            ev.record(self._side)
        return b, ev

    def wait_batch(self, handle) -> DeviceBatch:
        b, ev = handle
        torch.cuda.current_stream(self.device).wait_event(ev)
        return b

    def draw_noise(self, N):
        """U[0,1) gate / feature noise (reference: CPU torch.rand per graph, device rand_like: models.py:599, 650)."""
        return (torch.rand(N, device=self.device, generator=self._noise_gen),
                torch.rand(N, self.hidden, device=self.device, generator=self._noise_gen))

    def _workspace(self, b: DeviceBatch):
        need = self.lib.scgib_pretrain_workspace_bytes(ctypes.byref(self.dims), b.B, b.N, b.E, b.Ns, b.Es)
        if self._ws is None or self._ws.numel() < need:
            self._ws = None
            self._ws = torch.empty(int(need * 1.1) + 256, dtype=torch.uint8, device=self.device)
        return self._ws

    def debug_buffer(self, name: str, shape):
        """View of a named intermediate of the last forward/backward inside the workspace (tests only)."""
        b = self._last[0]
        off = self.lib.scgib_pretrain_workspace_offset(ctypes.byref(self.dims), b.B, b.N, b.E, b.Ns, b.Es, name.encode())
        if off < 0:
            raise KeyError(name)
        n = 1
        for v in shape:
            n *= v
        return self._ws[off:off + 4 * n].view(torch.float32).view(shape)

    # ---------------------------------------------------------------- step
    def forward(self, b: DeviceBatch, gate_u=None, feat_u=None, want=False, update_running=True,
                params: Optional[torch.Tensor] = None):
        """Returns the device tensor losses[4] = {KL, contrastive, recon, total}; with ``want`` also a dict of
        embeddings (interaction_map [N,128], Z, noisy, graph_readout)."""
        if gate_u is None:
            gate_u, feat_u = self.draw_noise(b.N)
        self._last = (b, gate_u.contiguous(), feat_u.contiguous())
        self.fwd_serial += 1
        cb = b.c_struct(self._last[1], self._last[2])
        ws = self._workspace(b)
        emb = None
        if want:
            H = self.hidden
            emb = dict(interaction_map=torch.empty(b.N, 2 * H, device=self.device),
                       Z=torch.empty(b.N, H, device=self.device), noisy=torch.empty(b.N, H, device=self.device),
                       graph_readout=torch.empty(b.B, H, device=self.device))
        p = self.params if params is None else params
        st = torch.cuda.current_stream(self.device).cuda_stream
        _lib.check(self.lib.scgib_pretrain_forward_f32(
            ctypes.byref(self.dims), _lib.ptr(p), _lib.ptr(self.bn_running) if (update_running or b.eval_mode) else None,
            ctypes.byref(cb), _lib.ptr(self.losses),
            _lib.ptr(emb["interaction_map"]) if want else None, _lib.ptr(emb["Z"]) if want else None,
            _lib.ptr(emb["noisy"]) if want else None, _lib.ptr(emb["graph_readout"]) if want else None,
            _lib.ptr(ws), ws.numel(), st), "pretrain_forward")
        if update_running and not b.eval_mode:
            self.num_batches_tracked += 1
        return (self.losses, emb) if want else self.losses

    def backward(self, loss_scale=(1.0, 1.0, 1.0), params: Optional[torch.Tensor] = None):
        """Gradients of scale . {KL, contrastive, recon} into the flat ``grads`` buffer (overwritten)."""
        b, gate_u, feat_u = self._last
        cb = b.c_struct(gate_u, feat_u)
        ws = self._workspace(b)
        self._loss_scale[0], self._loss_scale[1], self._loss_scale[2] = loss_scale
        p = self.params if params is None else params
        st = torch.cuda.current_stream(self.device).cuda_stream
        _lib.check(self.lib.scgib_pretrain_backward_f32(ctypes.byref(self.dims), _lib.ptr(p), ctypes.byref(cb),
                                                        self._loss_scale, _lib.ptr(self.grads), _lib.ptr(ws),
                                                        ws.numel(), st), "pretrain_backward")
        self._release_slot(b)
        return self.grads

    def forward_features(self, b: DeviceBatch, gate_u=None, feat_u=None, want_imap=False, update_running=True,
                         params: Optional[torch.Tensor] = None):
        """Feature path only (transfer_d -> extract_features -> head MLP; models.py:508-513), no pre-training losses.
        Returns Z [N,64] (and interaction_map [N,128] with ``want_imap``); ``extract_backward`` is its backward."""
        if gate_u is None:
            gate_u, feat_u = self.draw_noise(b.N)
        self._last = (b, gate_u.contiguous(), feat_u.contiguous())
        self.fwd_serial += 1
        cb = b.c_struct(self._last[1], self._last[2])
        ws = self._workspace(b)
        Z = torch.empty(b.N, self.hidden, device=self.device)
        imap = torch.empty(b.N, 2 * self.hidden, device=self.device) if want_imap else None
        p = self.params if params is None else params
        st = torch.cuda.current_stream(self.device).cuda_stream
        _lib.check(self.lib.scgib_extract_forward_f32(
            ctypes.byref(self.dims), _lib.ptr(p), _lib.ptr(self.bn_running) if (update_running or b.eval_mode) else None,
            ctypes.byref(cb), _lib.ptr(imap), _lib.ptr(Z), None, None, _lib.ptr(ws), ws.numel(), st), "extract_forward")
        if update_running and not b.eval_mode:
            self.num_batches_tracked += 1
        return (Z, imap) if want_imap else Z

    def extract_backward(self, gZ: torch.Tensor, params: Optional[torch.Tensor] = None):
        """Gradients of <gZ, Z> into the flat ``grads`` buffer (overwritten): the backward of ``extract_features`` + head
        MLP for a downstream head that consumes Z (fine-tuning, models.py:501-520).  Call after ``forward``."""
        b, gate_u, feat_u = self._last
        cb = b.c_struct(gate_u, feat_u)
        ws = self._workspace(b)
        gZ = gZ.contiguous().float()
        assert gZ.shape == (b.N, self.hidden) and gZ.device == self.device
        p = self.params if params is None else params
        st = torch.cuda.current_stream(self.device).cuda_stream
        _lib.check(self.lib.scgib_extract_backward_f32(ctypes.byref(self.dims), _lib.ptr(p), ctypes.byref(cb), _lib.ptr(gZ),
                                                       _lib.ptr(self.grads), _lib.ptr(ws), ws.numel(), st),
                   "extract_backward")
        self._release_slot(b)
        return self.grads

    def adam_step(self, lr=1e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=5e-5, grad_scale=1.0):
        """torch.optim.Adam(lr, weight_decay=5e-5) of exp_pretraining.py:86 over the flat buffer."""
        self.step_count += 1
        st = torch.cuda.current_stream(self.device).cuda_stream
        _lib.check(self.lib.scgib_adam_step_f32(_lib.ptr(self.params), _lib.ptr(self.grads), _lib.ptr(self.exp_avg),
                                                _lib.ptr(self.exp_avg_sq), self.total, self.step_count, lr, betas[0],
                                                betas[1], eps, weight_decay, grad_scale, st), "adam")

    def enable_peer_allreduce(self, group=None):
        """Data parallelism without NCCL on the hot path: gradients live in NVLink-mapped peer memory and ONE fused
        kernel per step does the rank-ordered all-reduce and Adam (dist.PeerAllreduce, csrc/peer_kernels.cu)."""
        from .dist import PeerAllreduce
        self._peer = PeerAllreduce(self.lib, self.total, self.device, group)
        self.grads = self._peer.grads(1)
        return self._peer

    def train_step(self, b: DeviceBatch, gate_u=None, feat_u=None, lr=1e-4, weight_decay=5e-5, world_size=1):
        """forward + backward (+ gradient all-reduce) + Adam; returns the device losses tensor (no host sync)."""
        peer = getattr(self, "_peer", None)
        losses = self.forward(b, gate_u, feat_u)
        if peer is not None and world_size > 1:
            peer.seq += 1
            self.grads = peer.grads(peer.seq)                 # this step's parity buffer (peers read it over NVLink)
            self.backward()
            self.step_count += 1
            peer.step(self.params, self.exp_avg, self.exp_avg_sq, peer.seq, self.step_count, lr, (0.9, 0.999), 1e-8,
                      weight_decay, torch.cuda.current_stream(self.device).cuda_stream)
        else:
            self.backward()
            if world_size > 1:
                import torch.distributed as dist
                dist.all_reduce(self.grads, op=dist.ReduceOp.SUM)
            self.adam_step(lr=lr, weight_decay=weight_decay, grad_scale=1.0 / world_size)
        self._release_slot(b)
        return losses

    def _release_slot(self, b):
        """A prefetch slot's buffers may be overwritten once the work queued so far on the training stream has run."""
        slot = getattr(b, "_slot", None)
        if slot is not None:
            slot["done"] = torch.cuda.Event()
            slot["done"].record(torch.cuda.current_stream(self.device))


FT_NAMES = ["s2s.lstm.weight_ih_l0", "s2s.lstm.weight_hh_l0", "s2s.lstm.bias_ih_l0", "s2s.lstm.bias_hh_l0",
            "predict.0.weight", "predict.0.bias", "predict.2.weight", "predict.2.bias"]


class FinetuneHead:
    """Set2Set(hidden, n_iters, 1) readout + predict MLP (+ sigmoid) of Mainmodel_finetuning.forward
    (models.py:515-520) on the CUDA path: one forward kernel, one backward kernel + fixed-order weight-gradient
    reductions (csrc/finetune_kernels.cu).  Parameters / gradients live in one flat buffer (slots = FT_NAMES)."""

    def __init__(self, hidden: int, num_out: int, n_iters: int = 2, sigmoid: bool = True, device="cuda:0"):
        self.lib = _lib.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("FinetuneHead needs a CUDA device: the hot path has no CPU fallback")
        self.H, self.C, self.T, self.sigmoid = int(hidden), int(num_out), int(n_iters), bool(sigmoid)
        off = (ctypes.c_int64 * _lib.FT_SLOTS)()
        sz = (ctypes.c_int64 * _lib.FT_SLOTS)()
        total = int(self.lib.scgib_finetune_head_layout(self.H, self.C, off, sz))
        if total < 0:
            _lib.check(total, "finetune_head_layout")
        self.total, self.offsets, self.sizes = total, list(off), list(sz)
        H, C = self.H, self.C
        self.shapes = [(4 * H, 2 * H), (4 * H, H), (4 * H,), (4 * H,), (H, 2 * H), (H,), (C, H), (C,)]
        if C == 0:
            self.shapes[6], self.shapes[7] = (0, H), (0,)
        self.names = list(FT_NAMES)
        self.params = torch.zeros(total, dtype=torch.float32, device=self.device)
        self.grads = torch.zeros_like(self.params)
        self._ws = None
        self._saved = None
        self.fwd_serial = 0

    def views(self, grads=False):
        buf = self.grads if grads else self.params
        return OrderedDict((n, buf[o:o + s].view(shp)) for n, o, s, shp in zip(self.names, self.offsets, self.sizes, self.shapes))

    def load_state_dict(self, sd):
        for n, t in self.views().items():
            if t.numel():
                t.copy_(sd[n].reshape(t.shape))

    def _workspace(self, B, N):
        need = self.lib.scgib_finetune_head_workspace_bytes(self.H, self.C, self.T, B, N)
        if self._ws is None or self._ws.numel() < need:
            self._ws = None
            self._ws = torch.empty(int(need * 1.1) + 256, dtype=torch.uint8, device=self.device)
        return self._ws

    def forward(self, Z: torch.Tensor, graph_ptr: torch.Tensor, want_readout=False):
        """scores [B,C] (after the sigmoid if enabled); with ``want_readout`` also the Set2Set output q* [B,2H]."""
        Z = Z.contiguous()
        B, N = graph_ptr.numel() - 1, Z.shape[0]
        assert Z.shape[1] == self.H and Z.dtype == torch.float32 and graph_ptr.dtype == torch.int32
        ws = self._workspace(B, N)
        scores = torch.empty(B, max(self.C, 1), device=self.device)
        readout = torch.empty(B, 2 * self.H, device=self.device) if (want_readout or self.C == 0) else None
        st = torch.cuda.current_stream(self.device).cuda_stream
        _lib.check(self.lib.scgib_finetune_head_fwd_f32(_lib.ptr(self.params), self.H, self.C, self.T, int(self.sigmoid),
                                                        _lib.ptr(Z), _lib.ptr(graph_ptr), B, N, _lib.ptr(scores),
                                                        _lib.ptr(readout), _lib.ptr(ws), ws.numel(), st), "finetune_head_fwd")
        self._saved = (Z, graph_ptr, scores)
        self.fwd_serial += 1
        if self.C == 0:
            return readout
        return (scores, readout) if want_readout else scores

    def backward(self, g_scores: Optional[torch.Tensor] = None, g_readout: Optional[torch.Tensor] = None):
        """Returns gZ [N,H]; the head's parameter gradients are written to ``self.grads`` (overwritten).  ``g_readout``
        [B,2H]: optional upstream gradient at the Set2Set output (required when the head has no predict MLP, C = 0)."""
        Z, graph_ptr, scores = self._saved
        B, N = graph_ptr.numel() - 1, Z.shape[0]
        g_scores = None if g_scores is None else g_scores.contiguous().float()
        g_readout = None if g_readout is None else g_readout.contiguous().float()
        gZ = torch.empty_like(Z)
        ws = self._workspace(B, N)
        st = torch.cuda.current_stream(self.device).cuda_stream
        _lib.check(self.lib.scgib_finetune_head_bwd_f32(_lib.ptr(self.params), self.H, self.C, self.T, int(self.sigmoid),
                                                        _lib.ptr(Z), _lib.ptr(graph_ptr), B, N, _lib.ptr(scores),
                                                        _lib.ptr(g_scores), _lib.ptr(g_readout), _lib.ptr(gZ), _lib.ptr(self.grads),
                                                        _lib.ptr(ws), ws.numel(), st), "finetune_head_bwd")
        return gZ


class PaddedSet2Set:
    """``dgl.nn.Set2Set(h, n_iters, 1)`` for a feature width h <= 128 (Mainmodel_domainadapt.s2s_rev over the raw
    node features, models.py:114, 267) on the smallest H in {32, 64, 128} >= h of the head kernels: weights and features
    are zero-padded to H channels.  A padded hidden unit has zero gate pre-activations (i = f = o = 1/2, g = 0), so its
    cell and hidden state stay exactly 0 and the real channels are untouched.  The scatter / gather between the module's
    real-shaped LSTM parameters and the padded flat buffer is index plumbing on four small tensors."""

    WIDTHS = (32, 64, 128)

    def __init__(self, h: int, n_iters: int = 2, device="cuda:0"):
        if not 1 <= h <= self.WIDTHS[-1]:
            raise NotImplementedError("PaddedSet2Set: feature width must be between 1 and %d, got %d" % (self.WIDTHS[-1], h))
        self.P = next(w for w in self.WIDTHS if w >= h)
        self.h, self.device = int(h), torch.device(device)
        self.head = FinetuneHead(self.P, 0, n_iters=n_iters, sigmoid=False, device=device)
        P, dev = self.P, self.device
        gate_rows = torch.cat([g * P + torch.arange(h) for g in range(4)]).to(dev)                 # [4h] rows of the padded gates
        in_cols = torch.cat([torch.arange(h), P + torch.arange(h)]).to(dev)                        # [2h] q half | readout half
        self.idx = dict(rows=gate_rows, in_cols=in_cols, hid_cols=torch.arange(h, device=dev),
                        out_cols=in_cols)

    def set_params(self, w_ih, w_hh, b_ih, b_hh):
        v = self.head.views()
        self.head.params.zero_()
        ix = self.idx
        v["s2s.lstm.weight_ih_l0"][ix["rows"][:, None], ix["in_cols"][None, :]] = w_ih.detach().float()
        v["s2s.lstm.weight_hh_l0"][ix["rows"][:, None], ix["hid_cols"][None, :]] = w_hh.detach().float()
        v["s2s.lstm.bias_ih_l0"][ix["rows"]] = b_ih.detach().float()
        v["s2s.lstm.bias_hh_l0"][ix["rows"]] = b_hh.detach().float()

    def forward(self, x: torch.Tensor, graph_ptr: torch.Tensor):
        """x [N, h] -> Set2Set output [B, 2h]."""
        xp = torch.zeros(x.shape[0], self.P, device=self.device)
        xp[:, :self.h] = x
        ro = self.head.forward(xp, graph_ptr)
        return ro[:, self.idx["out_cols"]]

    def backward(self, g_out: torch.Tensor):
        """g_out [B, 2h] -> gradients of the four LSTM tensors in their real shapes."""
        gp = torch.zeros(g_out.shape[0], 2 * self.P, device=self.device)
        gp[:, self.idx["out_cols"]] = g_out.float()
        self.head.backward(None, gp)
        gv, ix = self.head.views(grads=True), self.idx
        return (gv["s2s.lstm.weight_ih_l0"][ix["rows"][:, None], ix["in_cols"][None, :]].clone(),
                gv["s2s.lstm.weight_hh_l0"][ix["rows"][:, None], ix["hid_cols"][None, :]].clone(),
                gv["s2s.lstm.bias_ih_l0"][ix["rows"]].clone(), gv["s2s.lstm.bias_hh_l0"][ix["rows"]].clone())
