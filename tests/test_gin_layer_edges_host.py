"""CPU side of the GIN layer edge suite (tests/test_gpu_gin_layer_edges.py): the graph families it runs, and proof from the
CSR alone that each family reaches the gather path it is meant for.

The GIN forward kernels (csrc/gin_tc3.cu fp32, csrc/gin_bf16.cu bf16) gather a 128-row tile out of a 256-row window in shared
memory, [ws, ws + 256) with ws = max(0, base - 64), and stage at most 1024 neighbour indices per tile.  A neighbour outside
the window is read from global memory (through row_map in layer 0 of Encoder2), edge slots past 1024 are read from the
global index array, and the window is clipped at row 0 and at V.  The counts below are computed per tile exactly as the
kernels decide them.  The batches the other GPU tests build reach none of these paths (test_existing_batches_stay_local).
No device is touched."""
import numpy as np
import pytest
import torch

from oracle.graph_ref import (GIN_HALO, GIN_IDX_CAP, GIN_TILE, dense_tiles_graph, dense_walk_graph, ego_batch_ref, graph_from_bonds,
                              halo_graph, macrocycle_batch, path_graph, batch_ref, shuffle_nodes, star_graph, synth_batch)

WIN = GIN_TILE + 2 * GIN_HALO


def family(name):
    """dict(V, indptr, indices, row_map, n_in) of one family: a layer over V rows reading n_in input rows (through row_map)."""
    def plain(g):
        return dict(V=g.num_nodes, indptr=g.indptr, indices=g.indices, row_map=None, n_in=g.num_nodes)
    if name == "macrocycles":               # Peptides-func macrocycles (head-to-tail + 65 .. 200-atom closures) and a 420-atom one
        return plain(macrocycle_batch(1, 12))
    if name == "shuffled":                  # synth_batch molecules, atom order permuted inside each graph
        return plain(shuffle_nodes(synth_batch(2, 30, "peptides"), 3))
    if name.startswith("halo_"):            # edges exactly at the window limits; tile 0 and the last tile clipped
        return plain(halo_graph(int(name[5:])))
    if name == "dense_tiles":               # tiles of exactly 1023, 1024, 1025 edges
        return plain(dense_tiles_graph())
    if name == "dense_walk":                # 4 tiles per CTA, alternating 1024 / 1152 edges
        return plain(dense_walk_graph())
    if name == "star":                      # a 1500-leaf star: the hub row alone exceeds the staged indices
        return plain(star_graph(1500))
    if name == "ego_macrocycles":           # layer 0 of Encoder2: the k = 2 ego batch of the macrocycles, row_map = ego_nodes
        g = macrocycle_batch(1, 12)
        e = ego_batch_ref(g, 2)
        return dict(V=e.num_rows, indptr=e.sub_indptr, indices=e.sub_indices, row_map=e.ego_nodes, n_in=g.num_nodes)
    if name == "random_map":                # a random row map with repeated ids over a macrocycle CSR
        g = macrocycle_batch(4, 12)
        n_in = g.num_nodes // 3
        rm = np.random.default_rng(5).integers(0, n_in, g.num_nodes).astype(np.int32)
        return dict(V=g.num_nodes, indptr=g.indptr, indices=g.indices, row_map=rm, n_in=n_in)
    raise ValueError(name)


HALO_V = (127, 128, 129, 255, 257, 677)
FAMILIES = ["macrocycles", "shuffled"] + ["halo_%d" % v for v in HALO_V] + ["dense_tiles", "dense_walk", "star", "ego_macrocycles",
                                                                             "random_map"]


def tile_report(indptr, indices):
    """Per row tile, as the kernels decide it: neighbours outside the window, edges of the tile, window clipped at 0 / at V."""
    indptr = np.asarray(indptr, dtype=np.int64)
    V = len(indptr) - 1
    n_tiles = (V + GIN_TILE - 1) // GIN_TILE
    base = np.arange(n_tiles) * GIN_TILE
    ws = np.maximum(0, base - GIN_HALO)
    rows = np.repeat(np.arange(V), np.diff(indptr))
    tile = rows // GIN_TILE
    ul = np.asarray(indices, dtype=np.int64) - ws[tile]
    outside = np.bincount(tile[(ul < 0) | (ul >= WIN)], minlength=n_tiles)
    edges = indptr[np.minimum(base + GIN_TILE, V)] - indptr[base]
    return dict(outside=outside, edges=edges, clip_lo=base - GIN_HALO < 0, clip_hi=ws + WIN > V)


def summary(f):
    t = tile_report(f["indptr"], f["indices"])
    return dict(V=f["V"], tiles=len(t["edges"]), outside=int(t["outside"].sum()), max_tile_edges=int(t["edges"].max()),
                tiles_over_cap=int((t["edges"] > GIN_IDX_CAP).sum()), clipped_hi=bool(t["clip_hi"][-1]), row_map=f["row_map"] is not None)


@pytest.mark.parametrize("name", FAMILIES)
def test_family_reaches_its_path(name):
    f = family(name)
    V, ip, ix = f["V"], f["indptr"], f["indices"]
    assert len(ip) == V + 1 and ix.min() >= 0 and ix.max() < V
    src, dst = ix.astype(np.int64), np.repeat(np.arange(V), np.diff(ip.astype(np.int64)))
    assert np.array_equal(np.sort(src * V + dst), np.sort(dst * V + src))          # symmetric, as every GIN CSR is
    if f["row_map"] is not None:
        assert len(f["row_map"]) == V and f["row_map"].min() >= 0 and f["row_map"].max() < f["n_in"]
    t = tile_report(ip, ix)
    print(name, summary(f))
    if name in ("macrocycles", "shuffled", "star", "random_map", "halo_677", "halo_257", "halo_129"):
        assert t["outside"].sum() > 0                                               # beyond-window global reads
    if name == "macrocycles":
        assert np.abs(src - dst).max() > GIN_HALO + GIN_TILE                         # some closure is out of reach of any tile
    if name == "ego_macrocycles":
        # ego rows are local (every neighbour inside the window), but the window is copied row by row through the map, from
        # input rows further apart than a window
        assert t["outside"].sum() == 0
        rm = f["row_map"].astype(np.int64)
        span = [np.ptp(rm[max(0, b - GIN_HALO):b + GIN_TILE + GIN_HALO]) for b in range(0, V, GIN_TILE)]
        assert max(span) >= WIN
    if name == "random_map":
        assert len(np.unique(f["row_map"])) < V                                      # repeated ids
    if name.startswith("halo_"):
        assert t["clip_lo"][0] and t["clip_hi"][-1]
        # every rule of the window test is hit on both sides, wherever the rows exist
        base = np.arange(len(t["edges"])) * GIN_TILE
        ws = np.maximum(0, base - GIN_HALO)
        ul = src - ws[dst // GIN_TILE]
        for lim in (0, WIN - 1, WIN):
            assert (ul == lim).any() or V <= lim, lim
        if V > WIN:
            assert (ul == -1).any()
    if name == "dense_tiles":
        assert list(t["edges"]) == [GIN_IDX_CAP - 1, GIN_IDX_CAP, GIN_IDX_CAP + 1]
    if name == "dense_walk":
        over = t["edges"] > GIN_IDX_CAP
        assert V > 3 * 148 * GIN_TILE and over.any() and (~over).any()
        walk = over.reshape(-1, 148)                                                  # [step of the walk][CTA]
        assert (walk[1::2].all() and not walk[0::2].any())                           # overflowing and fitting tiles alternate
        assert set(t["edges"]) == {GIN_IDX_CAP, GIN_IDX_CAP + GIN_TILE}
    if name == "star":
        assert np.diff(ip.astype(np.int64))[0] > GIN_IDX_CAP and t["edges"][0] > GIN_IDX_CAP


def test_existing_batches_stay_local():
    """The batches of the other GPU tests (synth_batch molecules, their ego batches, the hand-built rings and stars) never leave
    the window and never overflow the staged indices: without the families above, those paths would run untested."""
    star13 = graph_from_bonds(13, [(0, i) for i in range(1, 13)], seed=3)
    ring40 = graph_from_bonds(40, [(i, (i + 1) % 40) for i in range(40)], seed=4)
    cases = {"pcqm_b300": synth_batch(1, 300), "pcqm_b4096": synth_batch(21, 4096), "peptides_b6": synth_batch(22, 6, "peptides"),
             "ragged": batch_ref([path_graph(2, seed=1), synth_batch(23, 1, "peptides"), star13, path_graph(3, seed=2), ring40])}
    rows = {}
    for name, g in cases.items():
        rows[name] = summary(dict(V=g.num_nodes, indptr=g.indptr, indices=g.indices, row_map=None))
    for name, (seed, B, k, shape) in {"ego_pcqm_b96_k2": (12, 96, 2, "pcqm"), "ego_peptides_b4_k3": (13, 4, 3, "peptides")}.items():
        e = ego_batch_ref(synth_batch(seed, B, shape), k)
        rows[name] = summary(dict(V=e.num_rows, indptr=e.sub_indptr, indices=e.sub_indices, row_map=e.ego_nodes))
    for name, r in rows.items():
        print(name, r)
        assert r["outside"] == 0 and r["tiles_over_cap"] == 0, (name, r)


def test_bf16_layer_reference_without_rounding_is_the_oracle():
    """tests/bf16_emulation.py's GIN layer reference with its rounding switched off computes GINConvRef + MLP (the oracle)
    operation for operation, and its backward matches autograd through GINConv -> BatchNorm(train) -> ReLU."""
    from oracle.scgib_oracle import GINConvRef, MLP, tgraph_from_ref
    from tests.bf16_emulation import gin_aggregate_ref, gin_bn_act_terms, gin_bwd_ref, gin_mlp_ref
    g = macrocycle_batch(7, 3)
    tg = tgraph_from_ref(g)
    V = g.num_nodes
    torch.manual_seed(3)
    conv = GINConvRef(MLP(32, 64, 64)).double()
    l1, l2 = conv.apply_func.mlp[0], conv.apply_func.mlp[2]
    h = torch.randn(V, 32, dtype=torch.float64)
    y_ref = conv(tg, h)
    terms, _ = gin_bn_act_terms(h, None, True)
    a = gin_aggregate_ref(terms, tg.src, tg.dst)
    r, y = gin_mlp_ref(a, l1.weight, l1.bias, l2.weight, l2.bias, emulate=False)
    assert torch.equal(y, y_ref)
    r2, y2 = gin_mlp_ref(a, l1.weight, l1.bias, l2.weight, l2.bias, emulate=True)
    assert 0 < float((y2.detach() - y.detach()).abs().max() / y.detach().abs().max()) <= 2e-2
    y, a = y.detach(), a.detach()
    # backward (direct and CSR mode) against autograd
    bnm = torch.nn.BatchNorm1d(64).double().train()
    with torch.no_grad():
        bnm.weight.uniform_(0.5, 1.5); bnm.bias.uniform_(-0.3, 0.3)
    for csr in (False, True):
        a_in = a.detach().clone().requires_grad_(True)
        for p in conv.parameters():
            p.grad = None
        bnm.zero_grad()
        y_ag = l2(torch.relu(l1(a_in)))
        out = torch.relu(bnm(y_ag))
        g_up = torch.randn(V, 64, dtype=torch.float64)
        G = g_up + torch.zeros_like(g_up).index_add(0, tg.dst, g_up[tg.src]) if csr else g_up
        (out * G).sum().backward()
        yd = y_ag.detach()
        bn = torch.stack([yd.mean(0), 1.0 / torch.sqrt(yd.var(0, unbiased=False) + 1e-5), bnm.weight.detach(), bnm.bias.detach()])
        res, _ = gin_bwd_ref(g_up, tg.src if csr else None, tg.dst if csr else None, yd, torch.relu(l1(a)).detach(), a, bn.float(),
                             l1.weight.detach(), l2.weight.detach(), True, emulate=False)
        want = (a_in.grad, l1.weight.grad, l1.bias.grad, l2.weight.grad, l2.bias.grad, bnm.weight.grad, bnm.bias.grad)
        for i, (got, w) in enumerate(zip(res, want)):
            if i == 4:                      # db2: a bias in front of a BatchNorm, mathematically zero
                assert float(got.abs().max()) <= 1e-5 * float(G.abs().max()), csr
                continue
            # bn is handed over in fp32 (as the kernels take it): the mask and BatchNorm constants move at 1e-7
            assert float((got - w).abs().max()) <= 1e-5 * float(w.abs().max()), (csr, i)


def test_bf16_layer_entries_validate_before_launching():
    """scgib_gin_layer_fwd_bf16 / scgib_gin_layer_bwd_bf16 return SCGIB_E_* for shapes without a kernel instance, a bn_in with
    kin != H, misaligned rows and short workspaces, before touching the device (every pointer below is a dummy)."""
    import ctypes
    from tests.test_abi import _lib as load
    lib = load().load()
    E_NULL, E_SHAPE, E_ALIGN, E_WORKSPACE, E_RANGE = -1, -2, -3, -4, -5
    P, Q, W = ctypes.c_void_p(0x10000), ctypes.c_void_p(0x10008), ctypes.c_void_p(0x20000)

    def fwd(kin=64, H=64, bn=None, V=10, a=None, ws=1 << 30, h=P):
        return lib.scgib_gin_layer_fwd_bf16(h, kin, H, None, bn, P, P, V, P, P, P, P, a, None, P, P, None, W, ws, None)

    def bwd(kin=64, H=64, V=10, y=P, ws=1 << 30, g_a=P):
        return lib.scgib_gin_layer_bwd_bf16(P, None, None, V, kin, H, 1, y, P, P, P, P, P, g_a, P, P, P, P, P, P, W, ws, None)
    for kin, H in ((128, 64), (16, 64), (32, 96), (48, 128), (64, 256)):
        assert fwd(kin, H) == E_SHAPE and bwd(kin, H) == E_SHAPE, (kin, H)
        assert lib.scgib_gin_layer_bwd_bf16_workspace_bytes(10, kin, H) == 0
    assert fwd(32, 64, bn=P) == E_SHAPE and fwd(64, 128, bn=P) == E_SHAPE
    assert fwd(h=None) == E_NULL and fwd(V=0) == E_RANGE and bwd(V=0) == E_RANGE
    assert fwd(a=Q) == E_ALIGN and fwd(h=Q) == E_ALIGN and bwd(y=Q) == E_ALIGN and bwd(g_a=Q) == E_ALIGN
    assert lib.scgib_gin_layer_fwd_bf16_workspace_bytes(10, 96) == 0
    for kin, H in ((32, 64), (64, 64), (32, 128), (64, 128), (128, 128)):
        need_f, need_b = lib.scgib_gin_layer_fwd_bf16_workspace_bytes(100000, H), lib.scgib_gin_layer_bwd_bf16_workspace_bytes(100000, kin, H)
        assert need_f > 0 and need_b > 100000 * H * 2
        assert fwd(kin, H, V=100000, ws=need_f - 1) == E_WORKSPACE and bwd(kin, H, V=100000, ws=need_b - 1) == E_WORKSPACE
