"""Oracle graph utilities (numpy, CPU).  TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Restates, without DGL, the graph semantics the reference hot path relies on:

* ``to_bidirected_ref``   - ``dgl.graph((s,d))`` + ``dgl.to_bidirected``  (reference util.py:317-318)
* ``batch_ref``           - ``dgl.batch`` node/edge id offsets          (reference molecules.py:359)
* ``khop_ball_ref``       - ``dgl.khop_in_subgraph(g, v, k)[0]`` node set (reference exp_pretraining.py:271)
* ``ego_batch_ref``       - the flattened ``dgl.batch`` of all ego-nets  (reference exp_pretraining.py:308-309)
* ``synth_molecule`` / ``synth_batch`` - the synthetic PCQM4Mv2-/Peptides-shape generator of SURVEY.md §8(d)

All index arrays are int32 / int64 numpy; features float32.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Sequence, Tuple

import numpy as np


# --------------------------------------------------------------------------------------
# DGL graph construction semantics
# --------------------------------------------------------------------------------------
def to_bidirected_ref(src: Sequence[int], dst: Sequence[int], num_nodes: int | None = None):
    """dgl.graph((src,dst)) then dgl.to_bidirected: add reverse edges, drop duplicates,
    edges sorted lexicographically by (src, dst).  num_nodes = max id + 1 (dgl.graph default).

    Returns (num_nodes, src_sorted, dst_sorted) as int64 arrays.
    """
    src = np.asarray(src, dtype=np.int64)
    dst = np.asarray(dst, dtype=np.int64)
    if num_nodes is None:
        num_nodes = int(max(src.max(initial=-1), dst.max(initial=-1)) + 1)
    s = np.concatenate([src, dst])
    d = np.concatenate([dst, src])
    key = np.unique(s * num_nodes + d)  # sorted => (src,dst) lexicographic
    return num_nodes, key // num_nodes, key % num_nodes


def csr_from_edges(num_nodes: int, src: np.ndarray, dst: np.ndarray):
    """In-neighbour CSR (row = dst, entries = src ascending).  For symmetric graphs this equals
    the out-neighbour CSR.  Returns (indptr[int32, n+1], indices[int32, E])."""
    order = np.lexsort((src, dst))
    s = src[order]
    d = dst[order]
    indptr = np.zeros(num_nodes + 1, dtype=np.int64)
    np.add.at(indptr, d + 1, 1)
    indptr = np.cumsum(indptr)
    return indptr.astype(np.int32), s.astype(np.int32)


@dataclass
class RefGraph:
    """One graph (or a batch of graphs) in CSR form with DGL-equivalent bookkeeping."""
    graph_ptr: np.ndarray  # int32 [B+1] node offsets per graph
    indptr: np.ndarray     # int32 [N+1]
    indices: np.ndarray    # int32 [E]   global node ids, ascending inside each row
    x: np.ndarray          # float32 [N, F]

    @property
    def num_graphs(self) -> int:
        return len(self.graph_ptr) - 1

    @property
    def num_nodes(self) -> int:
        return len(self.indptr) - 1

    @property
    def num_edges(self) -> int:
        return len(self.indices)

    def batch_num_nodes(self) -> np.ndarray:
        return np.diff(self.graph_ptr)

    def edges(self) -> Tuple[np.ndarray, np.ndarray]:
        """(src, dst) of every directed edge, in CSR (dst-major) order."""
        dst = np.repeat(np.arange(self.num_nodes, dtype=np.int64), np.diff(self.indptr))
        return self.indices.astype(np.int64), dst

    def dense_adj(self) -> np.ndarray:
        """DGL ``g.adj().to_dense()``: A[src, dst] = 1."""
        a = np.zeros((self.num_nodes, self.num_nodes), dtype=np.float32)
        s, d = self.edges()
        a[s, d] = 1.0
        return a


def batch_ref(graphs: List[RefGraph]) -> RefGraph:
    """dgl.batch: concatenate in list order, offsetting node ids."""
    gp = [0]
    ip = [np.zeros(1, dtype=np.int64)]
    idx = []
    xs = []
    noff = 0
    eoff = 0
    for g in graphs:
        assert g.num_graphs == 1
        ip.append(g.indptr[1:].astype(np.int64) + eoff)
        idx.append(g.indices.astype(np.int64) + noff)
        xs.append(g.x)
        noff += g.num_nodes
        eoff += g.num_edges
        gp.append(noff)
    return RefGraph(
        graph_ptr=np.asarray(gp, dtype=np.int32),
        indptr=np.concatenate(ip).astype(np.int32),
        indices=(np.concatenate(idx) if idx else np.zeros(0)).astype(np.int32),
        x=np.concatenate(xs, axis=0).astype(np.float32),
    )


# --------------------------------------------------------------------------------------
# k-hop ego networks (dgl.khop_in_subgraph restated)
# --------------------------------------------------------------------------------------
def khop_ball_ref(indptr: np.ndarray, indices: np.ndarray, v: int, k: int) -> np.ndarray:
    """Node set of dgl.khop_in_subgraph(g, v, k): hop h = unique(in_edges(frontier).src);
    result = unique(cat(seed, all hops)) => ascending original ids, contains v."""
    frontier = np.asarray([v], dtype=np.int64)
    hops = [frontier]
    for _ in range(k):
        if len(frontier) == 0:
            break
        nb = [indices[indptr[u]:indptr[u + 1]] for u in frontier]
        frontier = np.unique(np.concatenate(nb)) if nb else np.zeros(0, dtype=np.int64)
        hops.append(frontier.astype(np.int64))
    return np.unique(np.concatenate(hops)).astype(np.int64)


@dataclass
class RefEgoBatch:
    """Flattened batch of one ego-net per parent node (SURVEY.md Appendix A.0)."""
    ego_ptr: np.ndarray      # int32 [N+1]  ego-net v occupies rows ego_ptr[v]:ego_ptr[v+1]
    ego_nodes: np.ndarray    # int32 [Ns]   parent (global) node id of each ego row
    sub_indptr: np.ndarray   # int32 [Ns+1] induced CSR over ego rows
    sub_indices: np.ndarray  # int32 [Es]   ego-batch-local row ids

    @property
    def num_rows(self) -> int:
        return len(self.ego_nodes)

    @property
    def num_edges(self) -> int:
        return len(self.sub_indices)


def ego_batch_ref(g: RefGraph, k: int) -> RefEgoBatch:
    """For every node v (in node order) the induced k-hop in-subgraph, batched like
    ``dgl.batch(chain.from_iterable(batch_subgraphs))``."""
    N = g.num_nodes
    ego_ptr = np.zeros(N + 1, dtype=np.int64)
    nodes = []
    sub_ip = [0]
    sub_idx = []
    row0 = 0
    for v in range(N):
        ball = khop_ball_ref(g.indptr, g.indices, v, k)
        m = len(ball)
        pos = {int(u): i for i, u in enumerate(ball)}
        for u in ball:
            nb = g.indices[g.indptr[u]:g.indptr[u + 1]]
            loc = [row0 + pos[int(w)] for w in nb if int(w) in pos]  # ascending since nb ascending
            sub_idx.extend(loc)
            sub_ip.append(len(sub_idx))
        nodes.append(ball)
        row0 += m
        ego_ptr[v + 1] = row0
    return RefEgoBatch(
        ego_ptr=ego_ptr.astype(np.int32),
        ego_nodes=(np.concatenate(nodes) if nodes else np.zeros(0)).astype(np.int32),
        sub_indptr=np.asarray(sub_ip, dtype=np.int32),
        sub_indices=np.asarray(sub_idx, dtype=np.int32),
    )


# --------------------------------------------------------------------------------------
# Synthetic molecules (SURVEY.md §8(d))
# --------------------------------------------------------------------------------------
def _synth_bonds(rng: np.random.Generator, n: int, window: int, p_chain: float, n_rings: int,
                 max_deg: int = 4):
    deg = np.zeros(n, dtype=np.int64)
    adj = [set() for _ in range(n)]
    bonds = []

    def add(a, b):
        bonds.append((a, b))
        adj[a].add(b)
        adj[b].add(a)
        deg[a] += 1
        deg[b] += 1

    for v in range(1, n):
        lo = max(0, v - window)
        cand = [u for u in range(lo, v) if deg[u] < max_deg]
        if not cand:  # widen until something is free (a tree always has a leaf)
            cand = [u for u in range(0, v) if deg[u] < max_deg]
        if p_chain > 0 and deg[v - 1] < max_deg and rng.random() < p_chain:
            u = v - 1
        else:
            u = cand[int(rng.integers(len(cand)))]
        add(u, v)
    for _ in range(n_rings):
        for _attempt in range(32):
            a = int(rng.integers(n))
            lo, hi = max(0, a - window), min(n - 1, a + window)
            b = int(rng.integers(lo, hi + 1))
            if a == b or b in adj[a] or deg[a] >= max_deg or deg[b] >= max_deg:
                continue
            if adj[a] & adj[b]:  # would close a triangle
                continue
            add(a, b)
            break
    return bonds, deg


def _macrocycle_bonds(rng: np.random.Generator, n: int):
    """Peptides-shape chain with a head-to-tail closure (atom 0 - atom n-1) and 3 closures 65 .. 200 atoms apart: the bonds
    of a macrocyclic peptide, whose neighbours lie further apart in atom order than the local ring closures of ``peptides``."""
    bonds, deg = _synth_bonds(rng, n, window=6, p_chain=0.5, n_rings=3)
    have = {(min(a, b), max(a, b)) for a, b in bonds}
    extra = [(0, n - 1)]
    while len(extra) < 4:
        a = int(rng.integers(n))
        b = a + int(rng.integers(65, 201)) * (1 if rng.random() < 0.5 else -1)
        if 0 <= b < n and (min(a, b), max(a, b)) not in have and (min(a, b), max(a, b)) not in extra:
            extra.append((min(a, b), max(a, b)))
    for a, b in extra:
        if (a, b) not in have:
            bonds.append((a, b))
            deg[a] += 1
            deg[b] += 1
    return bonds, deg


def synth_molecule(rng: np.random.Generator, shape: str = "pcqm") -> RefGraph:
    """One synthetic molecule.  ``pcqm``: n~U[8,22], tree + 2 ring closures (bonds ~ n+1).
    ``peptides``: n~U[120,180], chain-biased tree + 3 ring closures.  ``macrocycle``: a ``peptides`` chain with a head-to-tail
    closure and 3 closures 65 .. 200 atoms apart (_macrocycle_bonds)."""
    if shape == "pcqm":
        n = int(rng.integers(8, 23))
        bonds, deg = _synth_bonds(rng, n, window=6, p_chain=0.0, n_rings=2)
    elif shape == "peptides":
        n = int(rng.integers(120, 181))
        bonds, deg = _synth_bonds(rng, n, window=6, p_chain=0.5, n_rings=3)
    elif shape == "macrocycle":
        n = int(rng.integers(120, 181))
        bonds, deg = _macrocycle_bonds(rng, n)
    else:
        raise ValueError(shape)
    return _molecule(rng, n, bonds, deg)


def _molecule(rng: np.random.Generator, n: int, bonds, deg) -> RefGraph:
    b = np.asarray(bonds, dtype=np.int64)
    nn_, s, d = to_bidirected_ref(b[:, 0], b[:, 1], n)
    indptr, indices = csr_from_edges(n, s, d)
    x = np.stack([
        rng.integers(1, 36, n), rng.integers(0, 4, n), deg, rng.integers(0, 11, n),
        rng.integers(0, 5, n), rng.integers(0, 5, n), rng.integers(0, 6, n),
        rng.integers(0, 2, n), rng.integers(0, 2, n)], axis=1).astype(np.float32)
    return RefGraph(np.asarray([0, n], dtype=np.int32), indptr, indices, x)


def synth_batch(seed: int, num_graphs: int, shape: str = "pcqm") -> RefGraph:
    rng = np.random.default_rng(seed)
    return batch_ref([synth_molecule(rng, shape) for _ in range(num_graphs)])


def synth_batch_fast(seed: int, num_graphs: int, shape: str = "pcqm", pool: int = 512) -> RefGraph:
    """Large batches for timing: draw ``pool`` distinct molecules once, then sample the batch
    from the pool with replacement (features re-drawn per instance is not needed for timing)."""
    rng = np.random.default_rng(seed)
    mols = [synth_molecule(rng, shape) for _ in range(min(pool, num_graphs))]
    pick = rng.integers(len(mols), size=num_graphs)
    return batch_ref([mols[i] for i in pick])


def path_graph(n: int, F: int = 9, seed: int = 0) -> RefGraph:
    s = np.arange(n - 1)
    _, ss, dd = to_bidirected_ref(s, s + 1, n)
    indptr, indices = csr_from_edges(n, ss, dd)
    x = np.random.default_rng(seed).random((n, F), dtype=np.float32) + 0.1
    return RefGraph(np.asarray([0, n], dtype=np.int32), indptr, indices, x)


def graph_from_bonds(n: int, bonds, F: int = 9, seed: int = 0) -> RefGraph:
    b = np.asarray(bonds, dtype=np.int64).reshape(-1, 2)
    _, ss, dd = to_bidirected_ref(b[:, 0], b[:, 1], n)
    indptr, indices = csr_from_edges(n, ss, dd)
    x = np.random.default_rng(seed).random((n, F), dtype=np.float32) + 0.1
    return RefGraph(np.asarray([0, n], dtype=np.int32), indptr, indices, x)


# --------------------------------------------------------------------------------------
# Non-local and dense graphs: the gather paths of the GIN forward kernels (csrc/gin_tc3.cu, gin_bf16.cu) beyond the
# 256-row window (a 128-row tile + a 64-row halo on each side) and beyond the 1024 staged neighbour indices of a tile
# --------------------------------------------------------------------------------------
GIN_TILE, GIN_HALO, GIN_IDX_CAP = 128, 64, 1024


def macrocycle_batch(seed: int, num_graphs: int, big: int = 420) -> RefGraph:
    """``num_graphs`` macrocyclic peptides (synth_molecule "macrocycle") and, with ``big`` > 0, one macrocycle of ``big``
    atoms: neighbours up to 200 rows apart, beyond the gather window."""
    rng = np.random.default_rng(seed)
    mols = [synth_molecule(rng, "macrocycle") for _ in range(num_graphs)]
    if big:
        mols.append(_molecule(rng, big, *_macrocycle_bonds(rng, big)))
    return batch_ref(mols)


def shuffle_nodes(g: RefGraph, seed: int) -> RefGraph:
    """The same graphs with the node ids randomly permuted inside each graph (arbitrary atom order: neighbours anywhere in
    the graph's row range)."""
    rng = np.random.default_rng(seed)
    N = g.num_nodes
    perm = np.concatenate([lo + rng.permutation(hi - lo) for lo, hi in zip(g.graph_ptr[:-1], g.graph_ptr[1:])]).astype(np.int64)
    src, dst = g.edges()
    indptr, indices = csr_from_edges(N, perm[src], perm[dst])
    x = np.empty_like(g.x)
    x[perm] = g.x
    return RefGraph(g.graph_ptr.copy(), indptr, indices, x)


def halo_graph(V: int, F: int = 9) -> RefGraph:
    """One graph of V rows: a path, plus edges from rows 0 and 127 of every tile to the rows just inside and just outside
    its window [ws, ws + 256), ws = max(0, base - 64): u = ws (inside), ws - 1 (outside), ws + 255 (inside), ws + 256
    (outside), where those rows exist.  Tile 0 has its window clipped at row 0, the last tile at V."""
    bonds = [(i, i + 1) for i in range(V - 1)]
    for base in range(0, V, GIN_TILE):
        ws = max(0, base - GIN_HALO)
        for v in (base, base + GIN_TILE - 1):
            for u in (ws - 1, ws, ws + 2 * GIN_HALO + GIN_TILE - 1, ws + 2 * GIN_HALO + GIN_TILE):
                if v < V and 0 <= u < V and u != v:
                    bonds.append((v, u))
    return graph_from_bonds(V, bonds, F)


def circulant_bonds(V: int, half_degree: int = 4):
    """Bonds of the circulant graph with offsets 1 .. half_degree (wrapping): every row has 2 * half_degree neighbours."""
    return [(i, (i + k) % V) for i in range(V) for k in range(1, half_degree + 1)]


def dense_tiles_graph(F: int = 9) -> RefGraph:
    """Three tiles of a degree-8 circulant (1024 edges each) with one bond removed between tiles 0 and 1 and one added
    between tiles 1 and 2: tiles of exactly 1023, 1024 and 1025 edges."""
    V = 3 * GIN_TILE
    bonds = [b for b in circulant_bonds(V) if b != (127, 128)] + [(200, 300)]
    return graph_from_bonds(V, bonds, F)


def dense_walk_graph(ctas: int = 148, walk: int = 4, F: int = 9) -> RefGraph:
    """``walk`` tiles per CTA of a ``ctas``-CTA persistent grid (tile t is the (t // ctas)-th tile its CTA walks): a degree-8
    circulant (1024 edges per tile) where every odd step of the walk gets 64 more bonds inside the tile (1152 edges, over
    the staged-index capacity), so that overflowing and fitting tiles alternate through the three index buffers."""
    V = ctas * walk * GIN_TILE
    bonds = circulant_bonds(V)
    for t in range(V // GIN_TILE):
        if (t // ctas) % 2 == 1:
            base = t * GIN_TILE
            bonds += [(base + r, base + r + GIN_HALO) for r in range(GIN_HALO)]
    return graph_from_bonds(V, bonds, F)


def star_graph(leaves: int, F: int = 9) -> RefGraph:
    """A hub (row 0) bonded to ``leaves`` leaves: the hub row alone exceeds the staged indices of its tile, and most leaves,
    and the hub for every leaf past row 255, lie outside the window."""
    return graph_from_bonds(leaves + 1, [(0, i) for i in range(1, leaves + 1)], F)
