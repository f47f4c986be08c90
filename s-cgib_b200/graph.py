"""DGL-free batched graphs for the S-CGIB hot path.

``BatchedGraph`` re-provides the slice of the DGLGraph surface the reference uses
(``dgl.batch`` molecules.py:359; ``.to / .ndata / .edges / .batch_num_nodes / .adj().to_dense()``
exp_pretraining.py:303-310, models.py:665, 764) on top of int32 CSR tensors, and
``khop_ego_batch`` replaces the offline ``dgl.khop_in_subgraph`` loop + per-step ``dgl.batch`` of
the ego-nets (exp_pretraining.py:271, 308-309) with two CUDA kernels per batch.
"""
from __future__ import annotations

from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _lib


class _DenseAdj:
    def __init__(self, g):
        self._g = g

    def to_dense(self):
        src, dst = self._g.edges()
        n = self._g.num_nodes()
        a = torch.zeros(n, n, dtype=torch.float32, device=src.device)
        a[src.long(), dst.long()] = 1.0
        return a


class BatchedGraph:
    """A batch of undirected graphs stored as one symmetric CSR (neighbours ascending, global ids)."""

    def __init__(self, graph_ptr, indptr, indices, x=None):
        self.graph_ptr = torch.as_tensor(graph_ptr, dtype=torch.int32)
        self.indptr = torch.as_tensor(indptr, dtype=torch.int32)
        self.indices = torch.as_tensor(indices, dtype=torch.int32)
        self.ndata = {}
        if x is not None:
            self.ndata["x"] = torch.as_tensor(x)

    # ---- DGLGraph-compatible surface
    @property
    def device(self):
        return self.indptr.device

    @property
    def batch_size(self):
        return self.graph_ptr.numel() - 1

    def num_nodes(self):
        return self.indptr.numel() - 1

    def num_edges(self):
        return self.indices.numel()

    def nodes(self):
        return torch.arange(self.num_nodes(), device=self.device)

    def batch_num_nodes(self):
        return (self.graph_ptr[1:] - self.graph_ptr[:-1]).long()

    def edges(self):
        deg = (self.indptr[1:] - self.indptr[:-1]).long()
        dst = torch.repeat_interleave(torch.arange(self.num_nodes(), device=self.device), deg)
        return self.indices.long(), dst

    def adj(self):
        return _DenseAdj(self)

    def to(self, device, non_blocking=False):
        g = BatchedGraph.__new__(BatchedGraph)
        g.graph_ptr = self.graph_ptr.to(device, non_blocking=non_blocking)
        g.indptr = self.indptr.to(device, non_blocking=non_blocking)
        g.indices = self.indices.to(device, non_blocking=non_blocking)
        g.ndata = {k: v.to(device, non_blocking=non_blocking) for k, v in self.ndata.items()}
        return g

    def pin_memory(self):
        g = BatchedGraph.__new__(BatchedGraph)
        g.graph_ptr, g.indptr, g.indices = self.graph_ptr.pin_memory(), self.indptr.pin_memory(), self.indices.pin_memory()
        g.ndata = {k: v.pin_memory() for k, v in self.ndata.items()}
        return g

    VALIDATE_ERRORS = {1: "graph_ptr does not cover [0, N)", 2: "indptr does not cover [0, E)",
                       3: "a graph has fewer than 2 nodes (per-graph BatchNorm / unbiased std, models.py:642-647)",
                       4: "indptr is not monotone", 5: "an edge leaves its graph", 6: "neighbours are not strictly ascending "
                       "(duplicate edge or unsorted row; build graphs with graph() / to_bidirected)", 7: "self loop"}

    def validate(self):
        """Checks what the kernels rely on; on a CUDA device with one kernel (scgib_batch_validate) and one host read.
        Raises ValueError naming the violated condition.  The engine calls it per batch when SCGIB_VALIDATE=1."""
        if self.device.type == "cuda":
            lib = _lib.load()
            status = torch.zeros(2, dtype=torch.int32, device=self.device)
            st = torch.cuda.current_stream(self.device).cuda_stream
            _lib.check(lib.scgib_batch_validate(_lib.ptr(self.graph_ptr), _lib.ptr(self.indptr), _lib.ptr(self.indices),
                                                self.batch_size, self.num_nodes(), self.num_edges(), _lib.ptr(status), st),
                       "batch_validate")
            code, where = status.tolist()
            if code:
                raise ValueError("invalid batch: %s (at graph / node %d)" % (self.VALIDATE_ERRORS.get(code, code), where))
            return self
        n = self.batch_num_nodes()
        if int(n.min()) < 2:
            raise ValueError("every graph needs >= 2 nodes (per-graph BatchNorm / unbiased std, models.py:642-647)")
        return self


def graph(edges, num_nodes: Optional[int] = None, x=None) -> BatchedGraph:
    """``dgl.graph((src, dst))`` followed by ``dgl.to_bidirected`` (util.py:317-318): reverse edges
    added, duplicates dropped, num_nodes = max id + 1, neighbours ascending."""
    src = np.asarray(edges[0], dtype=np.int64)
    dst = np.asarray(edges[1], dtype=np.int64)
    if num_nodes is None:
        num_nodes = int(max(src.max(initial=-1), dst.max(initial=-1)) + 1)
    s = np.concatenate([src, dst])
    d = np.concatenate([dst, src])
    key = np.unique(d * num_nodes + s)          # sorted by (dst, src): CSR rows with ascending neighbours
    dd, ss = key // num_nodes, key % num_nodes
    indptr = np.zeros(num_nodes + 1, dtype=np.int64)
    np.add.at(indptr, dd + 1, 1)
    return BatchedGraph(np.asarray([0, num_nodes]), np.cumsum(indptr), ss, x)


to_bidirected = lambda g: g  # graphs built by ``graph`` are already bidirected


def batch(graphs: Sequence[BatchedGraph]) -> BatchedGraph:
    """``dgl.batch``: concatenate in list order with node-id offsets; ``ndata`` concatenated."""
    gp, ip, idx = [torch.zeros(1, dtype=torch.int32)], [torch.zeros(1, dtype=torch.int32)], []
    noff = eoff = 0
    for g in graphs:
        gp.append(g.graph_ptr[1:] + noff)
        ip.append(g.indptr[1:] + eoff)
        idx.append(g.indices + noff)
        noff += g.num_nodes()
        eoff += g.num_edges()
    out = BatchedGraph(torch.cat(gp), torch.cat(ip), torch.cat(idx) if idx else torch.zeros(0, dtype=torch.int32))
    keys = graphs[0].ndata.keys() if graphs else ()
    for k in keys:
        out.ndata[k] = torch.cat([g.ndata[k] for g in graphs], 0)
    return out


def sum_nodes(g: BatchedGraph, key: str):
    """``dgl.sum_nodes`` through the CUDA segment kernel."""
    from .ops import segment_sum
    return segment_sum(g.ndata[key], g.graph_ptr)


class EgoBatch:
    """Flattened batch of one k-hop ego-net per parent node (what ``dgl.batch(chain(batch_subgraphs))``
    yields in the reference).  Row j is parent node ``ego_nodes[j]`` inside the ego-net of ``ego_seed[j]``."""

    def __init__(self, parent: BatchedGraph, k, ego_ptr, ego_nodes, ego_seed, sub_indptr, sub_indices):
        self.parent, self.k = parent, k
        self.ego_ptr, self.ego_nodes, self.ego_seed = ego_ptr, ego_nodes, ego_seed
        self.sub_indptr, self.sub_indices = sub_indptr, sub_indices

    @property
    def device(self):
        return self.ego_ptr.device

    @property
    def batch_size(self):
        return self.ego_ptr.numel() - 1

    def num_nodes(self):
        return self.ego_nodes.numel()

    def num_edges(self):
        return self.sub_indices.numel()

    def batch_num_nodes(self):
        return (self.ego_ptr[1:] - self.ego_ptr[:-1]).long()

    def to(self, device, non_blocking=False):
        return self if torch.device(device) == self.device else EgoBatch(
            self.parent.to(device), self.k, *[t.to(device) for t in (self.ego_ptr, self.ego_nodes, self.ego_seed,
                                                                     self.sub_indptr, self.sub_indices)])

    @property
    def ndata(self):
        # x_subs rows are copies of parent rows (SURVEY F10): a lazy gather, only for API compatibility
        return {k: v[self.ego_nodes.long()] for k, v in self.parent.ndata.items()}


class EgoWorkspace:
    """Reusable device buffers for ``khop_ego_batch`` (grown on demand)."""

    def __init__(self):
        self.ws = None
        self.ptrs = None
        self.status = None
        self.host = None


_DEFAULT_EGO_WS = {}     # per device: the pinned 3-int read-back buffer and the scan workspace are reused across calls


def khop_ego_batch(g: BatchedGraph, k: int, ws: Optional[EgoWorkspace] = None, stream=None, out=None) -> EgoBatch:
    """k-hop ego-net of every node of ``g`` on the GPU (bit-exact with ``dgl.khop_in_subgraph`` node lists).
    One host synchronisation (to read Ns / Es between the count and the fill kernel).
    ``out``: optional dict of preallocated int32 device buffers {ego_ptr, ego_eptr, ego_nodes, ego_seed, sub_indptr,
    sub_indices, status}; buffers that are too small are replaced in the dict."""
    lib = _lib.load()
    if g.device.type != "cuda":
        raise RuntimeError("khop_ego_batch needs the graph on a CUDA device (no CPU fallback)")
    dev = g.device
    N = g.num_nodes()
    st = torch.cuda.current_stream(dev).cuda_stream if stream is None else stream
    if ws is None:          # callers of the reference's loop pass nothing: a pinned allocation per call would cost ~2 ms
        ws = _DEFAULT_EGO_WS.setdefault(str(dev), EgoWorkspace())
    need = lib.scgib_ego_workspace_bytes(N)
    if ws.ws is None or ws.ws.numel() < need or ws.ws.device != dev:
        ws.ws = torch.empty(int(need * 1.5), dtype=torch.uint8, device=dev)
    if ws.host is None:
        ws.host = torch.empty(3, dtype=torch.int32).pin_memory()
    out = {} if out is None else out

    def buf(name, n):
        t = out.get(name)
        if t is None or t.numel() < n or t.device != dev:
            t = torch.empty(int(n * 1.25) + 16, dtype=torch.int32, device=dev)
            out[name] = t
        return t

    ego_ptr, ego_eptr, status = buf("ego_ptr", N + 1), buf("ego_eptr", N + 1), buf("status", 1)
    _lib.check(lib.scgib_ego_count(_lib.ptr(g.indptr), _lib.ptr(g.indices), N, int(k), _lib.ptr(ego_ptr),
                                   _lib.ptr(ego_eptr), _lib.ptr(status), _lib.ptr(ws.ws), ws.ws.numel(), st),
               "ego_count")
    ws.host[0:1].copy_(ego_ptr[N:N + 1], non_blocking=True)
    ws.host[1:2].copy_(ego_eptr[N:N + 1], non_blocking=True)
    ws.host[2:3].copy_(status[0:1], non_blocking=True)
    torch.cuda.current_stream(dev).synchronize()
    Ns, Es, bad = (int(v) for v in ws.host)
    if bad:
        raise RuntimeError("an ego-net exceeds SCGIB_EGO_CAP=%d nodes" % _lib.EGO_CAP)
    ego_nodes, ego_seed = buf("ego_nodes", Ns), buf("ego_seed", Ns)
    sub_indptr, sub_indices = buf("sub_indptr", Ns + 1), buf("sub_indices", max(Es, 1))
    _lib.check(lib.scgib_ego_fill(_lib.ptr(g.indptr), _lib.ptr(g.indices), N, int(k), _lib.ptr(ego_ptr),
                                  _lib.ptr(ego_eptr), _lib.ptr(ego_nodes), _lib.ptr(ego_seed), _lib.ptr(sub_indptr),
                                  _lib.ptr(sub_indices), st), "ego_fill")
    return EgoBatch(g, k, ego_ptr[:N + 1], ego_nodes[:Ns], ego_seed[:Ns], sub_indptr[:Ns + 1], sub_indices[:Es])


class DeviceDataset:
    """A packed dataset shard resident in HBM (every molecule as one symmetric CSR; the format of ``pts/<name>_csr.pt``,
    keys graph_ptr / indptr / indices / x) + GPU-side batch assembly: ``assemble(ids)`` builds the ``dgl.batch`` of the
    listed molecules on the device (csrc/graph_kernels.cu).  Replaces DataLoader + ``MoleculeDataset.collate``
    (molecules.py:349-362) and the per-step H2D of the batch: only the B molecule ids cross PCIe."""

    def __init__(self, graph_ptr, indptr, indices, x, device="cuda:0"):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("DeviceDataset needs a CUDA device (no CPU fallback)")
        self.lib = _lib.load()
        self.mol_ptr = torch.as_tensor(graph_ptr, dtype=torch.int32).to(self.device)
        self.indptr = torch.as_tensor(indptr, dtype=torch.int32).to(self.device)
        self.indices = torch.as_tensor(indices, dtype=torch.int32).to(self.device)
        self.x = torch.as_tensor(x).float().contiguous().to(self.device)
        self.F = int(self.x.shape[1])
        self._ws = None
        self._host = torch.empty(2, dtype=torch.int32).pin_memory()

    @classmethod
    def from_batched(cls, g: BatchedGraph, device="cuda:0"):
        return cls(g.graph_ptr, g.indptr, g.indices, g.ndata["x"], device)

    def __len__(self):
        return self.mol_ptr.numel() - 1

    def nbytes(self):
        return sum(t.numel() * t.element_size() for t in (self.mol_ptr, self.indptr, self.indices, self.x))

    def assemble(self, ids: torch.Tensor, out=None) -> BatchedGraph:
        """``ids``: int32 molecule ids (device, or pinned host: copied asynchronously).  One host read of (N, E) between
        the count and the fill kernels, on the current stream.  ``out``: optional dict of reusable device buffers."""
        dev = self.device
        if ids.device != dev:
            ids = ids.to(dev, non_blocking=True)
        ids = ids.to(torch.int32).contiguous()
        B = ids.numel()
        st = torch.cuda.current_stream(dev).cuda_stream
        need = self.lib.scgib_batch_workspace_bytes(B)
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(int(need * 1.5), dtype=torch.uint8, device=dev)
        out = {} if out is None else out

        def buf(name, n, dtype=torch.int32):
            t = out.get(name)
            if t is None or t.numel() < n or t.device != dev or t.dtype != dtype:
                t = torch.empty(int(n * 1.25) + 16, dtype=dtype, device=dev)
                out[name] = t
            return t

        graph_ptr, edge_ptr = buf("b_graph_ptr", B + 1), buf("b_edge_ptr", B + 1)
        _lib.check(self.lib.scgib_batch_assemble_count(_lib.ptr(self.mol_ptr), _lib.ptr(self.indptr), _lib.ptr(ids), B,
                                                       _lib.ptr(graph_ptr), _lib.ptr(edge_ptr), _lib.ptr(self._ws),
                                                       self._ws.numel(), st), "batch_assemble_count")
        self._host[0:1].copy_(graph_ptr[B:B + 1], non_blocking=True)
        self._host[1:2].copy_(edge_ptr[B:B + 1], non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
        N, E = int(self._host[0]), int(self._host[1])
        indptr, indices = buf("b_indptr", N + 1), buf("b_indices", max(E, 1))
        x = buf("b_x", N * self.F, torch.float32)
        _lib.check(self.lib.scgib_batch_assemble_fill(_lib.ptr(self.mol_ptr), _lib.ptr(self.indptr), _lib.ptr(self.indices),
                                                      _lib.ptr(self.x), self.F, _lib.ptr(ids), B, _lib.ptr(graph_ptr),
                                                      _lib.ptr(edge_ptr), _lib.ptr(indptr), _lib.ptr(indices), _lib.ptr(x),
                                                      st), "batch_assemble_fill")
        g = BatchedGraph.__new__(BatchedGraph)
        g.graph_ptr, g.indptr, g.indices = graph_ptr[:B + 1], indptr[:N + 1], indices[:E]
        g.ndata = {"x": x[:N * self.F].view(N, self.F)}
        return g


# --------------------------------------------------------------------------------------------------
# On-disk format: one packed CSR shard per dataset (replaces pts/<name>.bin + pts/<name>_subgraphs_khop_<k>.pt +
# pts/<name>_M_khop_<k>.pt of the reference, exp_pretraining.py:171-206, 285: ego-nets and log-transition matrices are
# computed on the GPU per batch and never stored)
# --------------------------------------------------------------------------------------------------
def pack_shard(molecules, path: Optional[str] = None):
    """``molecules``: iterable of (edge_index [2,E] as in a PyG ``Data``, x [n,F], y) triples.  Each molecule goes through
    ``graph`` (= ``util.load_dgl_fromPyG``, util.py:277-325: dgl.graph + to_bidirected) and all of them are concatenated
    like ``dgl.batch``.  Returns (and optionally ``torch.save``s) the dict that ``pts/<name>_csr.pt`` holds."""
    gs, ys = [], []
    for edge_index, x, y in molecules:
        edge_index = np.asarray(edge_index)
        x = torch.as_tensor(np.asarray(x)).float()
        gs.append(graph((edge_index[0], edge_index[1]), num_nodes=x.shape[0], x=x))
        ys.append(torch.as_tensor(np.asarray(y)).float().reshape(-1))
    big = batch(gs)
    shard = dict(graph_ptr=big.graph_ptr, indptr=big.indptr, indices=big.indices, x=big.ndata["x"], y=torch.stack(ys))
    if path is not None:
        torch.save(shard, path)
    return shard


def load_shard(path: str) -> "tuple[BatchedGraph, torch.Tensor]":
    shard = torch.load(path)
    return BatchedGraph(shard["graph_ptr"], shard["indptr"], shard["indices"], shard["x"]), shard.get("y")


class DeviceLoader:
    """Drop-in for ``DataLoader(dataset, batch_size, shuffle=True, collate_fn=dataset.collate)`` (exp_pretraining.py:283) over
    a ``DeviceDataset``: iterating yields the reference's 4-tuples ``(batched_graph, labels, subgraphs, logMs)`` with the
    batch assembled on the GPU from B molecule ids (no Python object per molecule, no collate, no H2D of graph data).
    ``rank`` / ``world`` shard every epoch's permutation like a ``DistributedSampler(drop_last=True)``.  With
    ``shard_batches=True`` they shard whole batches instead: rank r takes batches r, r + world, r + 2 world, ... of the
    single-process batch list, so the ranks together see every molecule exactly once (evaluation splits)."""

    def __init__(self, dataset: DeviceDataset, batch_size: int, shuffle: bool = True, drop_last: bool = False,
                 labels: Optional[torch.Tensor] = None, rank: int = 0, world: int = 1, seed: int = 0,
                 shard_batches: bool = False):
        self.dataset, self.batch_size, self.shuffle, self.drop_last = dataset, int(batch_size), shuffle, drop_last
        self.labels = None if labels is None else labels.to(dataset.device)
        self.rank, self.world, self.seed, self.epoch = rank, world, seed, 0
        self.shard_batches = shard_batches
        self.sampler = self                      # ``loader.sampler.set_epoch(e)`` works as with a DistributedSampler
        self._bufs = [{}, {}]                    # two sets of reusable device buffers (consecutive batches never share one)

    def set_epoch(self, epoch: int):
        self.epoch = int(epoch)

    def _per_rank(self):
        n = len(self.dataset)
        return n // self.world if self.world > 1 and not self.shard_batches else n

    def _ranges(self):
        """[lo, hi) positions in the pass's id list of this rank's batches."""
        n, B = self._per_rank(), self.batch_size
        if self.drop_last:
            n -= n % B
        if self.shard_batches:
            from .dist import round_robin_batches
            return round_robin_batches(n, B, self.rank, self.world)
        return [(lo, min(lo + B, n)) for lo in range(0, n, B)]

    def __len__(self):
        return len(self._ranges())

    def id_batches(self):
        """The epoch's mini-batches as device tensors of molecule ids (what ``__iter__`` assembles one by one)."""
        ids_dev = self._epoch_ids()
        for lo, hi in self._ranges():
            yield ids_dev[lo:hi]

    def _epoch_ids(self):
        """Permutation of this pass, then advance the epoch: like ``DataLoader(shuffle=True)`` every pass reshuffles
        without anybody calling ``set_epoch`` (which stays as the data-parallel override: all ranks must agree)."""
        n = len(self.dataset)
        if self.shuffle:
            perm = torch.randperm(n, generator=torch.Generator().manual_seed(self.seed + self.epoch))
            self.epoch += 1
        else:
            perm = torch.arange(n)
        if self.world > 1 and not self.shard_batches:
            per = n // self.world
            perm = perm[self.rank * per:(self.rank + 1) * per]
        return perm.to(torch.int32).to(self.dataset.device)

    def __iter__(self):
        ids_dev = self._epoch_ids()
        for i, (lo, hi) in enumerate(self._ranges()):
            ids = ids_dev[lo:hi]
            g = self.dataset.assemble(ids, out=self._bufs[i & 1])
            labels = self.labels[ids.long()] if self.labels is not None else torch.zeros(ids.numel(), 1, device=self.dataset.device)
            yield g, labels, None, None
