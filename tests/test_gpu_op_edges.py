"""Operator edge suite: the per-graph and tensor-core kernels behind the op-level C ABI against fp64 references at the
shapes where their code paths change (RB = 4 / 8 of the core gate, the warp-per-graph loops that wrap past the grid cap,
the head's tensor-core / FFMA branches, the logM / ego-net ball capacity, the Set2Set class and step limits, the
contrastive row blocks) and at input magnitudes away from 1.

The fp64 references are the oracle's functions where they are cheap; where the oracle loops per graph and a batch has ~10^4
graphs, the vectorised restatements below are used instead.  tests/test_op_edge_refs_host.py checks every restatement
against the oracle on small batches, without a GPU.

Bounds are those of the existing op tests: 1e-5 forward, 2e-5 / 5e-5 gradients (2e-4 for the core gate backward, as
tests/test_gpu_ops.py), max-norm relative error (tests/helpers.rel)."""
import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle.graph_ref import batch_ref, ego_batch_ref, graph_from_bonds, khop_ball_ref, path_graph, synth_batch
from oracle.scgib_oracle import OracleMainmodel, Set2SetRef, TGraph, get_logm, loss_recon_logm, tgraph_from_ref
from tests.helpers import product_graph, rel

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
EGO_CAP = 128
KL_EPS, BN_EPS, GATE_BIAS = 1e-7, 1e-5, 1e-4


# ------------------------------------------------------------------------------------------------ fp64 restatements
def seg_of(sizes):
    return torch.repeat_interleave(torch.arange(len(sizes)), torch.as_tensor(sizes, dtype=torch.int64))


def seg_sum(x, seg, B):
    return torch.zeros((B,) + x.shape[1:], dtype=x.dtype).index_add(0, seg, x)


def gate_ref(Hf, sizes, Wc1, bc1, gamma, beta, w2, b2, gate_u, feat_u, running=None):
    """OracleMainmodel.compression + sum_nodes (models.py:595-604, 631-660) for all graphs at once.  Returns noisy, graph
    readout, core readout, KL of the last graph, and each graph's batch mean / unbiased variance of q (the running-statistics
    update of compressor.1).  ``running`` = (mean, var): the eval-mode BatchNorm."""
    B, seg = len(sizes), seg_of(sizes)
    n = torch.as_tensor(sizes, dtype=Hf.dtype)
    Hd = Hf.detach()                                         # models.py:645: std / mean of a detached copy
    mu = seg_sum(Hd, seg, B) / n[:, None]
    sd = torch.sqrt(seg_sum((Hd - mu[seg]) ** 2, seg, B) / (n - 1)[:, None])
    q = Hf @ Wc1.t() + bc1
    qm = seg_sum(q, seg, B) / n[:, None]
    qc2 = seg_sum((q - qm[seg]) ** 2, seg, B)
    if running is None:
        qhat = (q - qm[seg]) / torch.sqrt(qc2 / n[:, None] + BN_EPS)[seg]
    else:
        qhat = (q - running[0]) / torch.sqrt(running[1] + BN_EPS)
    p = torch.relu(qhat * gamma + beta) @ w2.reshape(-1) + b2.reshape(())
    eps = (GATE_BIAS - (1 - GATE_BIAS)) * gate_u.reshape(-1) + (1 - GATE_BIAS)
    lam = torch.sigmoid(torch.log(eps) - torch.log(1 - eps) + p)[:, None]
    noisy_mean = lam * Hf + (1 - lam) * mu[seg]
    noisy_std = (1 - lam) * sd[seg]
    noisy = noisy_mean + feat_u * noisy_std
    last = slice(int(sum(sizes[:-1])), int(sum(sizes)))
    den = sd[-1] + KL_EPS
    KL = 0.5 * (noisy_std[last] ** 2 / den ** 2) + torch.sum(((noisy_mean[last] - mu[-1]) / den) ** 2, dim=0)
    return noisy, seg_sum(Hf, seg, B), seg_sum(noisy, seg, B), KL.mean(), qm.detach(), (qc2 / (n - 1)[:, None]).detach()


def bn_ema_ref(qm, qv, mean0, var0, momentum=0.1):
    """compressor.1's running statistics after one nn.BatchNorm1d train call per graph, in graph order."""
    m, v = mean0.clone(), var0.clone()
    for g in range(qm.shape[0]):
        m = (1 - momentum) * m + momentum * qm[g]
        v = (1 - momentum) * v + momentum * qv[g]
    return m, v


def attn_ref(C, sizes, w):
    """models.py:738-748 (core half and bias of attn_layer cancel): alpha = per-graph softmax of C w, T = alpha C."""
    B, seg = len(sizes), seg_of(sizes)
    logit = C @ w
    mx = torch.full((B,), -float("inf"), dtype=C.dtype).scatter_reduce(0, seg, logit.detach(), "amax")
    ex = torch.exp(logit - mx[seg])
    alpha = ex / seg_sum(ex, seg, B)[seg]
    return alpha, C * alpha[:, None]


def adjacency_blocks(g):
    """Dense adjacency of every graph of a RefGraph batch."""
    out = []
    for b in range(g.num_graphs):
        v0, v1 = int(g.graph_ptr[b]), int(g.graph_ptr[b + 1])
        A = np.zeros((v1 - v0, v1 - v0))
        for v in range(v0, v1):
            A[v - v0, g.indices[g.indptr[v]:g.indptr[v + 1]] - v0] = 1.0
        out.append((v0, v1, A))
    return out


def ball_sizes(g, k):
    return np.asarray([len(khop_ball_ref(g.indptr, g.indices, v, k)) for v in range(g.num_nodes)])


def logm_ref(Z, g, k, cap=EGO_CAP):
    """loss_recon of --recons_type logM (models.py:770-782) in the per-seed form of csrc/logm_kernels.cu, with the terms of every
    seed whose k-hop ball exceeds ``cap`` nodes dropped (the operator's documented status-1 result):
        loss = sum_g ||Z_g^T Z_g||^2 / n^2 + (1/k) sum_{kept seeds r} sum_c (-2 (z_r . z_c) Ls_rc + L2_rc) / n^2,
        gZ_r = 4/n^2 (Z_g Z_g^T Z_g)_r - [r kept] 2/(k n^2) sum_c (Ls + Ls^T)_rc z_c,
    Ls = sum_i logM_i, L2 = sum_i logM_i^2.  With no ball over ``cap`` this is loss_recon_logm and its gradient."""
    kept = torch.from_numpy(ball_sizes(g, k) <= cap).to(Z.dtype)
    loss = Z.new_zeros(())
    gZ = torch.zeros_like(Z)
    for v0, v1, A in adjacency_blocks(g):
        n = v1 - v0
        Ls = [torch.from_numpy(m) for m in get_logm(A, k)]
        L1, L2 = sum(Ls), sum(m ** 2 for m in Ls)
        Zg, kp = Z[v0:v1], kept[v0:v1]
        G = Zg.t() @ Zg
        loss = loss + (G ** 2).sum() / n ** 2 + (kp[:, None] * (-2 * (Zg @ Zg.t()) * L1 + L2)).sum() / (k * n ** 2)
        gZ[v0:v1] = 4 / n ** 2 * Zg @ G - 2 / (k * n ** 2) * kp[:, None] * ((L1 + L1.t()) @ Zg)
    return loss, gZ


# ------------------------------------------------------------------------------------------------ batch shapes
def gate_sizes(kind):
    """Graph sizes (>= 2 nodes: a graph's std is unbiased) around the RB = 4 / 8 switch (mean N / B >= 48) and the grid cap."""
    from scgib_b200 import _lib
    rng = np.random.default_rng(len(kind))
    if kind == "mean_lt48_with_400":
        s = rng.integers(2, 23, size=60); s[17] = 400
    elif kind == "mean_gt48_with_2":
        s = np.asarray([2, 150, 2, 2, 150, 150, 2, 150, 150, 2])
    elif kind == "b1":
        s = np.asarray([37])
    elif kind == "last_2":
        s = np.concatenate([rng.integers(2, 23, size=20), [2]])
    elif kind == "last_150":
        s = np.concatenate([rng.integers(2, 23, size=20), [150]])
    elif kind == "grid_wrap":                 # forward: 8 warps x 8 SMs-multiples CTAs; backward 4 x SMs CTAs: both loops wrap
        s = rng.integers(2, 7, size=8 * 8 * int(_lib.load().scgib_num_sms()) + 37)
    else:
        raise KeyError(kind)
    mean = s.sum() / len(s)
    assert s.min() >= 2 and (mean < 48 if kind == "mean_lt48_with_400" else True) and (mean >= 48 if kind == "mean_gt48_with_2" else True)
    return [int(v) for v in s]


GATE_KINDS = ["mean_lt48_with_400", "mean_gt48_with_2", "b1", "last_2", "last_150", "grid_wrap"]


def _ptr(sizes):
    return torch.from_numpy(np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)).to(DEV)


def _f(t):
    return t.detach().float().to(DEV)


def _f64(t):
    """fp64 copy of the fp32-rounded value: the reference sees exactly the operator's inputs."""
    return t.detach().float().double()


# ------------------------------------------------------------------------------------------------ core gate
@pytest.mark.parametrize("H", [64, 128])
@pytest.mark.parametrize("kind", GATE_KINDS)
def test_core_gate_edges(kind, H):
    from scgib_b200 import ops
    sizes = gate_sizes(kind)
    N = sum(sizes)
    torch.manual_seed(H + N)
    m = OracleMainmodel(9, H).double()
    c = m.compressor
    P = [_f64(t) for t in (c[0].weight, c[0].bias, c[1].weight, c[1].bias, c[3].weight, c[3].bias)]
    for t in P:
        t.requires_grad_(True)
    Hf = _f64(torch.randn(N, H, dtype=torch.float64)).requires_grad_(True)
    gate_u, feat_u = torch.rand(N, dtype=torch.float64).float(), torch.rand(N, H, dtype=torch.float64).float()
    noisy, readout, core, kl, qm, qv = gate_ref(Hf, sizes, *P, gate_u.double(), feat_u.double())
    gn, gc, gr = torch.randn_like(noisy), torch.randn_like(core), torch.randn_like(readout)
    ((noisy * gn).sum() + (core * gc).sum() + (readout * gr).sum() + 0.7 * kl).backward()

    op = ops.CoreGate(H, *[_f(t) for t in P])
    gp = _ptr(sizes)
    out = op.forward(_f(Hf), gp, gate_u.to(DEV), feat_u.to(DEV))
    for name, got, ref in (("noisy", out[0], noisy), ("readout", out[2], readout), ("core", out[3], core), ("kl", out[4], kl.reshape(1))):
        assert rel(got, ref) <= 1e-5, (name, rel(got, ref))
    grads = op.backward(_f(gn), _f(gc), _f(gr), 0.7)
    refs = (Hf.grad, *[t.grad for t in P])
    gmax = max(float(r.abs().max()) for r in refs)
    for i, (got, ref) in enumerate(zip(grads, refs)):
        if i == 2:                                             # compressor.0.bias in front of a BatchNorm: zero gradient
            assert float(ref.abs().max()) <= 1e-9 * gmax and float(got.abs().max()) <= 1e-4 * gmax
            continue
        assert rel(got.reshape(ref.shape), ref) <= 2e-4, (i, rel(got.reshape(ref.shape), ref))

    # compressor.1's running statistics: B sequential BatchNorm1d(momentum 0.1) calls, one per graph
    rm0, rv0 = torch.randn(H, dtype=torch.float64) * 0.1, 1 + torch.rand(H, dtype=torch.float64)
    run_m, run_v = _f(rm0), _f(rv0)
    op.forward(_f(Hf), gp, gate_u.to(DEV), feat_u.to(DEV))
    op.update_running(run_m, run_v)
    em, ev = bn_ema_ref(qm, qv, _f64(rm0), _f64(rv0))
    assert rel(run_m, em) <= 1e-5 and rel(run_v, ev) <= 1e-5, (rel(run_m, em), rel(run_v, ev))

    # model.eval(): the BatchNorm normalises with the running statistics
    rmv = (_f64(rm0), _f64(rv0))
    with torch.no_grad():
        noisy_e, readout_e, core_e, kl_e, _, _ = gate_ref(Hf, sizes, *P, gate_u.double(), feat_u.double(), running=rmv)
    out_e = op.forward(_f(Hf), gp, gate_u.to(DEV), feat_u.to(DEV), running=(_f(rm0), _f(rv0)))
    torch.cuda.synchronize()
    for name, got, ref in (("noisy", out_e[0], noisy_e), ("readout", out_e[2], readout_e), ("core", out_e[3], core_e),
                           ("kl", out_e[4], kl_e.reshape(1))):
        assert rel(got, ref) <= 1e-5, ("eval " + name, rel(got, ref))


# ------------------------------------------------------------------------------------------------ core-candidate attention
def _exact_logits(sizes, H, centre):
    """C [N,H] and w [H] with every logit C_v . w EXACT in fp32 (entries on a 1/64 grid, w = +-1/8): the operator's error is
    then its softmax's own.  Graph b's logits are centre[b] + U(-8, 8)."""
    N = sum(sizes)
    C = torch.round(torch.randn(N, H, dtype=torch.float64) * 64) / 64
    w = (torch.randint(0, 2, (H,)).double() * 2 - 1) / 8
    target = torch.round((centre[seg_of(sizes)] + (torch.rand(N, dtype=torch.float64) * 16 - 8)) * 512) / 512
    C[:, 0] = (target - C[:, 1:] @ w[1:]) / w[0]
    assert torch.equal(C @ w, target) and torch.equal(C.float().double(), C)
    return C, w


@pytest.mark.parametrize("H", [64, 128])
@pytest.mark.parametrize("kind,logits", [(k, "randn") for k in GATE_KINDS] +
                         [("mean_lt48_with_400", "pm80"), ("grid_wrap", "pm80"), ("mean_gt48_with_2", "equal")])
def test_core_cand_attention_edges(kind, logits, H):
    from scgib_b200 import ops
    sizes = gate_sizes(kind)
    N, B = sum(sizes), len(sizes)
    torch.manual_seed(7 * H + N)
    if logits == "pm80":                      # a softmax without the max shift overflows (exp(88.7) = inf in fp32)
        C, w = _exact_logits(sizes, H, torch.where(torch.arange(B) % 2 == 0, 80.0, -80.0).double())
    else:
        C, w = _f64(torch.randn(N, H, dtype=torch.float64)), _f64(torch.randn(H, dtype=torch.float64) * 0.3)
        if logits == "equal":                 # every row of graph 1 the same: equal logits, alpha = 1 / n
            C[sizes[0]:sizes[0] + sizes[1]] = C[sizes[0]]
    C.requires_grad_(True); w.requires_grad_(True)
    alpha, T = attn_ref(C, sizes, w)
    gT = _f64(torch.randn_like(T))
    (T * gT).sum().backward()
    gp = _ptr(sizes)
    a, Tg = ops.core_cand_attn_fwd(_f(C), gp, _f(w))
    assert rel(a, alpha) <= 1e-5 and rel(Tg, T) <= 1e-5, (rel(a, alpha), rel(Tg, T))
    if logits == "equal":
        n1 = sizes[1]
        assert rel(a[sizes[0]:sizes[0] + n1], torch.full((n1,), 1.0 / n1, dtype=torch.float64)) <= 1e-6
    gC, dw = ops.core_cand_attn_bwd(_f(C), a, _f(gT), gp, _f(w))
    torch.cuda.synchronize()
    assert rel(gC, C.grad) <= 2e-5 and rel(dw, w.grad) <= 2e-5, (rel(gC, C.grad), rel(dw, w.grad))


# ------------------------------------------------------------------------------------------------ head MLP
def _offset_copy(t):
    """The same values in a view whose data pointer is 16 (not 32) bytes past an allocation: the FFMA branch at hidden 64."""
    buf = torch.empty(t.numel() + 4, device=DEV)
    v = buf[4:].view(t.shape)
    v.copy_(t)
    assert v.data_ptr() % 32 == 16
    return v


def _away_from_kink(noisy, C, alpha, W1, b1, scale):
    """Redraw the rows with a hidden pre-activation within 1e-5 of the largest one from the ReLU kink: there two correct fp32
    products may take different sides, and the flipped unit moves that row's input gradient by O(1) (tests/helpers.py)."""
    while True:
        u = torch.cat((noisy, C * alpha[:, None]), -1) @ W1.t() + b1
        bad = (u.abs() < 1e-5 * float(u.abs().max())).any(1)
        if not bad.any():
            return noisy, C
        k = int(bad.sum())
        noisy[bad] = _f64(torch.randn(k, noisy.shape[1], dtype=torch.float64) * scale)
        C[bad] = _f64(torch.randn(k, C.shape[1], dtype=torch.float64) * scale)


@pytest.mark.parametrize("H", [64, 128])
@pytest.mark.parametrize("N", [1, 127, 128, 129, 61440])
@pytest.mark.parametrize("scale", [1e-3, 1.0, 1e3, 1e5])
def test_head_mlp_edges(scale, N, H):
    from scgib_b200 import ops
    torch.manual_seed(H + N)
    mlp = nn.Sequential(nn.Linear(2 * H, H), nn.ReLU(), nn.Linear(H, H)).double()
    with torch.no_grad():
        for p in mlp.parameters():
            p.copy_(_f64(p))
    alpha = _f64(torch.rand(N, dtype=torch.float64))
    noisy, C = _away_from_kink(_f64(torch.randn(N, H, dtype=torch.float64) * scale), _f64(torch.randn(N, H, dtype=torch.float64) * scale),
                               alpha, mlp[0].weight.detach(), mlp[0].bias.detach(), scale)
    noisy.requires_grad_()
    aC = (C * alpha[:, None]).requires_grad_()
    imap = torch.cat((noisy, aC), -1)
    Z = mlp(imap)
    gZ = _f64(torch.randn_like(Z))
    (Z * gZ).sum().backward()
    refs = ((mlp[0].weight.grad, "dW1"), (mlp[0].bias.grad, "db1"), (mlp[2].weight.grad, "dW2"), (mlp[2].bias.grad, "db2"))
    op = ops.HeadMLP(H, _f(mlp[0].weight), _f(mlp[0].bias), _f(mlp[2].weight), _f(mlp[2].bias))
    branches = [("aligned", lambda t: t)] + ([("offset16", _offset_copy)] if H == 64 else [])
    Zs = {}
    for br, place in branches:                   # hidden 64: aligned operands run head_tc.cu, 16-byte offsets the FFMA tiles
        Zg, ig = op.forward(place(_f(noisy)), place(_f(C)), _f(alpha))
        Zs[br] = Zg.clone()
        assert rel(Zg, Z) <= 1e-5 and rel(ig, imap) <= 1e-6, (br, rel(Zg, Z), rel(ig, imap))
        gI, *dW = op.backward(_f(gZ))
        torch.cuda.synchronize()
        assert rel(gI[0], noisy.grad) <= 2e-5 and rel(gI[1], aC.grad) <= 2e-5, (br, rel(gI[0], noisy.grad), rel(gI[1], aC.grad))
        for got, (ref, name) in zip(dW, refs):
            assert rel(got, ref) <= 2e-5, (br, name, rel(got, ref))
    if H == 64 and N == 61440 and scale == 1.0:   # two different kernels ran: different roundings of the same product
        assert not torch.equal(Zs["aligned"], Zs["offset16"])


# ------------------------------------------------------------------------------------------------ GIN layer backward
@pytest.mark.parametrize("kin,csr", [(64, False), (32, False), (64, True), (32, True)])
@pytest.mark.parametrize("act_scale", [1e-3, 1e2])
@pytest.mark.parametrize("g_scale", [1e-6, 1e4])
def test_gin_layer_backward_magnitudes(kin, csr, act_scale, g_scale):
    """scgib_gin_layer_bwd_f32 with the forward activations a, r and the upstream gradient far from 1 (the fp16-split kernel
    scales the gradients by a power of two and splits a, r as they are)."""
    from scgib_b200 import ops
    from oracle.scgib_oracle import GINConvRef, MLP
    g = synth_batch(5, 400)
    tg = tgraph_from_ref(g)
    V = g.num_nodes
    torch.manual_seed(kin + int(csr))
    conv = GINConvRef(MLP(kin, 64, 64)).double()
    bnm = torch.nn.BatchNorm1d(64).double().train()
    lin1, lin2 = conv.apply_func.mlp[0], conv.apply_func.mlp[2]
    with torch.no_grad():
        bnm.weight.uniform_(0.5, 1.5); bnm.bias.uniform_(-0.3, 0.3)
        lin1.bias.mul_(act_scale); lin2.bias.mul_(act_scale)       # a, r, y all scale with the input
        for p in (lin1.weight, lin1.bias, lin2.weight, lin2.bias):
            p.copy_(_f64(p))
    h = torch.randn(V, kin, dtype=torch.float64) * act_scale
    neigh = torch.zeros_like(h).index_add(0, tg.dst, h[tg.src])
    a_ref = _f64(h + neigh).requires_grad_(True)
    r_ref = torch.relu(lin1(a_ref))
    y_ref = lin2(r_ref)
    # the operator takes the saved fp32 y / r: the reference continues from exactly those values
    y_in = _f64(y_ref).requires_grad_(True)
    out = torch.relu(bnm(y_in))
    g_up = _f64(torch.randn(V, 64, dtype=torch.float64) * g_scale)
    G = g_up + torch.zeros_like(g_up).index_add(0, tg.dst, g_up[tg.src]) if csr else g_up
    (out * G).sum().backward()
    y_ref.backward(y_in.grad)
    mean, var = y_in.detach().mean(0), y_in.detach().var(0, unbiased=False)
    bn = torch.stack([mean, 1.0 / torch.sqrt(var + BN_EPS), bnm.weight.detach(), bnm.bias.detach()]).float().to(DEV)
    pg = product_graph(g, DEV)
    res = ops.gin_layer_bwd(_f(g_up), _f(y_in), _f(r_ref), _f(a_ref), bn, _f(lin1.weight), _f(lin2.weight),
                            indptr=pg.indptr if csr else None, indices=pg.indices if csr else None)
    torch.cuda.synchronize()
    want = (a_ref.grad, lin1.weight.grad, lin1.bias.grad, lin2.weight.grad, lin2.bias.grad, bnm.weight.grad, bnm.bias.grad)
    names = ("g_a", "dW1", "db1", "dW2", "db2", "dgamma", "dbeta")
    gmax = max(float(w.abs().max()) for w in want)
    for name, got, w in zip(names, res, want):
        if name == "db2":        # a bias in front of a BatchNorm: mathematically zero
            assert float(got.abs().max()) <= 1e-5 * gmax, name
            continue
        assert rel(got, w) <= 5e-5, (name, rel(got, w))


# ------------------------------------------------------------------------------------------------ logM operator
def star(leaves):
    return graph_from_bonds(leaves + 1, [(0, i) for i in range(1, leaves + 1)])


def ring(n):
    return graph_from_bonds(n, [(i, (i + 1) % n) for i in range(n)])


def _logm_case(g, k, H, seed):
    from scgib_b200 import ops
    torch.manual_seed(seed)
    Z = _f64(torch.randn(g.num_nodes, H, dtype=torch.float64) * 0.15)
    dropped = bool((ball_sizes(g, k) > EGO_CAP).any())
    if dropped:
        ref, gref = logm_ref(Z, g, k)
    else:
        Zr = Z.clone().requires_grad_(True)
        ref = loss_recon_logm(Zr, tgraph_from_ref(g), k)
        ref.backward()
        gref = Zr.grad
    pg = product_graph(g, DEV)
    loss, gZ, status = ops.recon_logm(_f(Z), pg.graph_ptr, pg.indptr, pg.indices, k, scale=0.5)
    torch.cuda.synchronize()
    assert int(status) == int(dropped)
    assert torch.isfinite(loss).all() and torch.isfinite(gZ).all()
    assert abs(float(loss) - float(ref)) <= 1e-5 * abs(float(ref)), (float(loss), float(ref))
    assert rel(gZ, 0.5 * gref) <= 2e-5, rel(gZ, 0.5 * gref)
    return dropped


@pytest.mark.parametrize("H", [64, 128])
@pytest.mark.parametrize("k", [4, 5, 6, 7, 8])
@pytest.mark.parametrize("shape,B", [("pcqm", 40), ("peptides", 4)])
def test_recon_logm_long_walks(shape, B, k, H):
    _logm_case(synth_batch(500 + k + H, B, shape), k, H, H + k)


@pytest.mark.parametrize("H", [64, 128])
@pytest.mark.parametrize("k", [1, 3, 8])
def test_recon_logm_ball_at_capacity(k, H):
    """A 127-leaf star (every k >= 1 ball is exactly 128 nodes), a 40-ring, a graph with isolated nodes, 2-node graphs."""
    g = batch_ref([star(127), ring(40), graph_from_bonds(6, [(0, 1), (1, 2)]), graph_from_bonds(2, [(0, 1)]),
                   graph_from_bonds(2, [(0, 1)])])
    assert ball_sizes(g, k).max() == EGO_CAP
    assert not _logm_case(g, k, H, 31 + k)


@pytest.mark.parametrize("H", [64, 128])
def test_recon_logm_ball_over_capacity(H):
    """A 200-leaf star at k = 1: the centre's ball has 201 nodes.  status = 1 and the centre's seed terms are dropped, exactly
    as the fp64 reference that drops the same seeds."""
    g = batch_ref([graph_from_bonds(2, [(0, 1)]), star(200), ring(40)])
    assert _logm_case(g, 1, H, 77)


# ------------------------------------------------------------------------------------------------ ego-net extraction
def test_ego_extraction_at_and_over_capacity():
    from scgib_b200.graph import khop_ego_batch
    g = batch_ref([ring(12), star(127), graph_from_bonds(2, [(0, 1)])])
    e = ego_batch_ref(g, 1)
    got = khop_ego_batch(product_graph(g, DEV), 1)
    for name in ("ego_ptr", "ego_nodes", "sub_indptr", "sub_indices"):
        assert np.array_equal(getattr(got, name).cpu().numpy(), getattr(e, name)), name
    assert int(np.diff(e.ego_ptr).max()) == EGO_CAP
    with pytest.raises(RuntimeError, match="SCGIB_EGO_CAP"):
        khop_ego_batch(product_graph(batch_ref([ring(12), star(128)]), DEV), 1)


def test_dropin_logm_refuses_ball_over_capacity():
    """Mainmodel --recons_type logM takes its ego-nets from khop_ego_batch, which refuses a ball over the capacity: a loss with
    silently dropped logM terms (the operator's status 1) is never returned."""
    import types
    import models
    from scgib_b200.graph import khop_ego_batch
    args = types.SimpleNamespace(recons_type="logM", useAtt=1, readout_f="sum", d_transfer=32, device=DEV, batch_size=128,
                                 task="graph_classification", dataset="Peptides-func", k_transition=1)
    m = models.Mainmodel(args, 9, hidden_dim=64, num_layers=4, num_heads=4, k_transition=1, encoder="GraphSAGE").to(DEV)
    m.train()
    g = batch_ref([ring(12), star(200)])
    pg = product_graph(g, DEV)
    with pytest.raises(RuntimeError, match="SCGIB_EGO_CAP"):
        m.forward(pg, F.normalize(pg.ndata["x"].float()), khop_ego_batch(pg, 1), None, None, 1, None, 2, DEV, g.num_graphs)


# ------------------------------------------------------------------------------------------------ Set2Set + predict head
def _seg_graph(sizes):
    ptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    z = torch.zeros(0, dtype=torch.int64)
    return TGraph(seg_ptr=torch.from_numpy(ptr), indptr=torch.zeros(int(ptr[-1]) + 1, dtype=torch.int64), indices=z, src=z, dst=z)


S2S_CASES = [  # H, C, T, sizes
    (64, 64, 8, [1, 150, 450, 3, 17, 1, 40]),
    (128, 64, 8, [450, 1, 150, 9, 2, 33, 1, 150, 5]),
    (64, 0, 2, [1, 150, 450, 3, 17, 1, 40]),
    (128, 0, 3, [450, 1, 150, 9, 2, 33, 1, 150, 5]),
    (64, 64, 8, [450]),
    (128, 10, 2, [1]),
    (64, 5, 2, "b8300"),
]


@pytest.mark.parametrize("H,C,T,sizes", S2S_CASES, ids=["H%d-C%d-T%d-%s" % (c[0], c[1], c[2], c[3] if isinstance(c[3], str) else "B%d" % len(c[3]))
                                                       for c in S2S_CASES])
def test_set2set_head_edges(H, C, T, sizes):
    """Set2Set(H, T, 1) + predict + sigmoid (C > 0), or the Set2Set readout alone with its upstream gradient g_readout (C = 0).
    B = 8300 at T = 2: the weight-gradient reductions over (T - 1) B and T B rows reach their 64-split limit."""
    from scgib_b200.engine import FinetuneHead
    if sizes == "b8300":
        sizes = np.random.default_rng(8300).integers(1, 40, size=8300)
    sizes = np.asarray(sizes)
    B, N = len(sizes), int(sizes.sum())
    tg = _seg_graph(sizes)
    torch.manual_seed(B + C + T)
    s2s = Set2SetRef(H, T, 1).double()
    predict = nn.Sequential(nn.Linear(2 * H, H), nn.ReLU(), nn.Linear(H, max(C, 1))).double()
    with torch.no_grad():
        for p in list(s2s.parameters()) + list(predict.parameters()):
            p.copy_(_f64(p))
    Z = _f64(torch.randn(N, H, dtype=torch.float64) * 0.7).requires_grad_(True)
    q = s2s(tg, Z)
    g_r = _f64(torch.randn(B, 2 * H, dtype=torch.float64))
    obj = (q * g_r).sum()
    if C > 0:
        s = torch.sigmoid(predict(q))
        g_s = _f64(torch.randn(B, C, dtype=torch.float64))
        obj = obj + (s * g_s).sum()
    obj.backward()

    head = FinetuneHead(H, C, n_iters=T, sigmoid=True, device=DEV)
    sd = {"s2s." + n: p for n, p in s2s.state_dict().items()}
    if C > 0:
        sd.update({"predict." + n: p for n, p in predict.state_dict().items()})
    else:
        sd.update({"predict.0." + n: p for n, p in predict[0].state_dict().items()})
    head.load_state_dict({n: t.float() for n, t in sd.items()})
    gp = torch.from_numpy(np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)).to(DEV)
    if C > 0:
        scores, readout = head.forward(_f(Z), gp, want_readout=True)
        assert rel(scores, s) <= 1e-5, rel(scores, s)
        gZ = head.backward(_f(g_s), g_readout=_f(g_r))
    else:
        readout = head.forward(_f(Z), gp)
        gZ = head.backward(None, g_readout=_f(g_r))
    torch.cuda.synchronize()
    assert rel(readout, q) <= 1e-5, rel(readout, q)
    assert rel(gZ, Z.grad) <= 2e-5, rel(gZ, Z.grad)
    ref = {"s2s." + n: p.grad for n, p in s2s.named_parameters()}
    if C > 0:
        ref.update({"predict." + n: p.grad for n, p in predict.named_parameters()})
    for n, got in head.views(grads=True).items():
        if C == 0 and n.startswith("predict."):                  # no predict MLP: nothing flows through it
            continue
        assert rel(got, ref[n]) <= 2e-5, (n, rel(got, ref[n]))


# ------------------------------------------------------------------------------------------------ contrastive, recon adj
@pytest.mark.parametrize("H", [64, 128])
@pytest.mark.parametrize("B", [127, 128, 129, 255, 257, 4097])
def test_contrastive_block_edges(B, H):
    from scgib_b200 import ops
    torch.manual_seed(B + H)
    m = OracleMainmodel(9, H).double()
    core = _f64(torch.randn(B, H, dtype=torch.float64) * 2).requires_grad_(True)
    ro = _f64(torch.randn(B, H, dtype=torch.float64) * 3).requires_grad_(True)
    con = m.batched_semi_loss(core, ro, B)
    con.backward()
    loss, g1, g2 = ops.contrastive(_f(core), _f(ro), scale=2.0)
    torch.cuda.synchronize()
    assert abs(float(loss) - float(con)) <= 1e-5 * abs(float(con)), (float(loss), float(con))
    assert rel(g1, 2.0 * core.grad) <= 5e-5 and rel(g2, 2.0 * ro.grad) <= 5e-5, (rel(g1, 2.0 * core.grad), rel(g2, 2.0 * ro.grad))


@pytest.mark.parametrize("H", [64, 128])
@pytest.mark.parametrize("N", [2, 37, 1031])
def test_recon_adj_tile_edges(N, H):
    from scgib_b200 import ops
    g = path_graph(N)
    torch.manual_seed(N + H)
    m = OracleMainmodel(9, H).double()
    Z = _f64(torch.randn(N, H, dtype=torch.float64) * 0.3).requires_grad_(True)
    rec = m.loss_recon_adj(Z, tgraph_from_ref(g))
    rec.backward()
    pg = product_graph(g, DEV)
    loss, gZ = ops.recon_adj(_f(Z), pg.indptr, pg.indices, scale=0.5)
    torch.cuda.synchronize()
    assert abs(float(loss) - float(rec)) <= 1e-5 * abs(float(rec)), (float(loss), float(rec))
    assert rel(gZ, 0.5 * Z.grad) <= 2e-5, rel(gZ, 0.5 * Z.grad)
