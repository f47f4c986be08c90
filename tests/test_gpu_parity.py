"""GPU parity tests (run on the B200 box: `pytest -m gpu`).  The CUDA path is called through the C ABI
(ctypes) and compared with (1) the golden vectors recorded from the unmodified reference models.py and
(2) the CPU oracle on seeded synthetic batches.

Tolerances (BASELINE.json north_star): embeddings and losses 1e-5 relative (fp32, max-norm) against the fp64
oracle; gradients: median over the 61 parameter tensors <= 5e-5, every tensor <= 5e-3 (a ReLU mask that flips
between two correct fp32 implementations moves downstream gradients by O(1/rows); tests/helpers.py).  Where fp32 arithmetic itself cannot reach that (sums over ~10^5 rows with cancellation,
1/sigma^2 terms of the KL), the bound is 5x the error of the fp32 torch reference-precision run against the same fp64 truth
(tests/helpers.py:check_against_truth).  Ego-net index lists are bit-exact.
"""
import glob
import os

import numpy as np
import pytest
import torch

from oracle.graph_ref import (RefEgoBatch, RefGraph, batch_ref, ego_batch_ref, graph_from_bonds, macrocycle_batch, path_graph,
                              shuffle_nodes, synth_batch)
from oracle.scgib_oracle import (OracleMainmodel, draw_noise_like_reference, normalize_rows, tgraph_from_ego,
                                 tgraph_from_ref)
from tests.helpers import (GRAD_TOL_MAX, GRAD_TOL_MEDIAN, check_against_truth, engine_from_oracle, fp64_truth,
                           is_zero_grad_param, oracle_grads, product_ego_from_ref, product_graph, rel)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLD = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "pretrain_*.pt")) +
              glob.glob(os.path.join(os.path.dirname(__file__), "golden", "logm_*.pt")))     # logm_*: --recons_type logM
FWD_TOL = 1e-5


def _ego_equal(ego, e: RefEgoBatch):
    assert np.array_equal(ego.ego_ptr.cpu().numpy(), e.ego_ptr)
    assert np.array_equal(ego.ego_nodes.cpu().numpy(), e.ego_nodes)
    assert np.array_equal(ego.sub_indptr.cpu().numpy(), e.sub_indptr)
    assert np.array_equal(ego.sub_indices.cpu().numpy(), e.sub_indices)
    seed = np.repeat(np.arange(len(e.ego_ptr) - 1), np.diff(e.ego_ptr))
    assert np.array_equal(ego.ego_seed.cpu().numpy(), seed)


@pytest.mark.parametrize("k", [1, 2, 3])
@pytest.mark.parametrize("seed,B", [(0, 64), (3, 257)])
def test_ego_extraction_bit_exact(seed, B, k):
    from scgib_b200.graph import khop_ego_batch
    g = synth_batch(seed, B)
    _ego_equal(khop_ego_batch(product_graph(g, DEV), k), ego_batch_ref(g, k))


@pytest.mark.parametrize("k", [1, 2, 4])
def test_ego_extraction_adversarial(k):
    from scgib_b200.graph import khop_ego_batch
    ring = graph_from_bonds(12, [(i, (i + 1) % 12) for i in range(12)])
    star = graph_from_bonds(40, [(0, i) for i in range(1, 40)])          # degree 39 > one warp of neighbours
    iso = graph_from_bonds(6, [(0, 5), (2, 3)])                          # isolated interior nodes 1, 4
    g = batch_ref([ring, star, iso, path_graph(2), path_graph(33)])
    _ego_equal(khop_ego_batch(product_graph(g, DEV), k), ego_batch_ref(g, k))


def test_ego_extraction_large_matches_properties():
    """Full-size batch (B=4096): sizes, sortedness, seed membership, symmetry of the induced CSR."""
    from scgib_b200.graph import khop_ego_batch
    from scgib_b200.synth import synth_batch as psynth
    g = psynth(5, 4096).to(DEV)
    ego = khop_ego_batch(g, 2)
    ptr, nodes, seed = ego.ego_ptr.long(), ego.ego_nodes.long(), ego.ego_seed.long()
    assert int(ptr[-1]) == nodes.numel() and int(ego.sub_indptr[-1]) == ego.sub_indices.numel()
    d = nodes[1:] - nodes[:-1]
    same = seed[1:] == seed[:-1]
    assert bool((d[same] > 0).all())                                        # ascending inside each ego-net
    assert int((nodes == seed).sum()) == g.num_nodes()                      # each ego-net contains its seed once
    deg = (ego.sub_indptr[1:] - ego.sub_indptr[:-1]).long()
    dst = torch.repeat_interleave(torch.arange(nodes.numel(), device=DEV), deg)
    src = ego.sub_indices.long()
    assert bool((seed[src] == seed[dst]).all())
    key = src * nodes.numel() + dst
    assert torch.equal(torch.sort(key)[0], torch.sort(dst * nodes.numel() + src)[0])   # symmetric


def test_input_proj_and_segment_sum():
    from scgib_b200 import ops
    torch.manual_seed(0)
    x = torch.rand(1000, 9) * 10
    W = torch.randn(32, 9)
    ref = torch.nn.functional.normalize(x) @ W.t()
    assert rel(ops.input_proj(x.to(DEV), W.to(DEV)), ref) <= 2e-6
    h = torch.randn(1000, 64)
    ptr = torch.tensor([0, 3, 3, 500, 1000], dtype=torch.int32)
    ref = torch.stack([h[0:3].sum(0), h[3:3].sum(0), h[3:500].sum(0), h[500:].sum(0)])
    assert rel(ops.segment_sum(h.to(DEV), ptr.to(DEV)), ref) <= 2e-6


@pytest.mark.parametrize("kin", [32, 64])
def test_gin_layer_forward(kin):
    from scgib_b200 import ops
    from oracle.scgib_oracle import GINConvRef, MLP
    g = synth_batch(1, 300)
    tg = tgraph_from_ref(g)
    torch.manual_seed(kin)
    conv = GINConvRef(MLP(kin, 64, 64))
    h = torch.randn(g.num_nodes, kin)
    y_ref = conv(tg, h)
    lin1, lin2 = conv.apply_func.mlp[0], conv.apply_func.mlp[2]
    pg = product_graph(g, DEV)
    y, bn, a, r = ops.gin_layer_fwd(h.to(DEV), pg.indptr, pg.indices, lin1.weight.detach().to(DEV),
                                    lin1.bias.detach().to(DEV), lin2.weight.detach().to(DEV),
                                    lin2.bias.detach().to(DEV), save=True)
    assert rel(y, y_ref) <= 2e-6
    assert rel(bn[0], y_ref.mean(0)) <= 1e-5
    assert rel(bn[1], 1.0 / torch.sqrt(y_ref.var(0, unbiased=False) + 1e-5)) <= 1e-5
    neigh = torch.zeros_like(h).index_add(0, tg.dst, h[tg.src])
    assert rel(a, h + neigh) <= 2e-6


def _run_engine(m, g, e, k, gate_u, feat_u, from_gpu_ego=True, recon_logm_steps=0):
    from scgib_b200.engine import DeviceBatch
    from scgib_b200.graph import khop_ego_batch
    eng = engine_from_oracle(m, DEV)
    pg = product_graph(g, DEV)
    ego = khop_ego_batch(pg, k) if from_gpu_ego else product_ego_from_ref(pg, e, k, DEV)
    b = DeviceBatch(pg, ego, pg.ndata["x"], normalize_x=True)
    b.recon_logm_steps = recon_logm_steps
    losses, emb = eng.forward(b, gate_u.to(DEV), feat_u.to(DEV), want=True)
    eng.backward()
    torch.cuda.synchronize()
    return eng, losses.cpu(), emb


@pytest.mark.parametrize("path", GOLD, ids=[os.path.basename(p) for p in GOLD])
def test_golden_reference_parity(path):
    """CUDA path vs the unmodified reference models.py (golden vectors): losses, embeddings, all 61 gradients,
    BN running statistics."""
    fx = torch.load(path, weights_only=False)
    g, e = RefGraph(**fx["graph"]), RefEgoBatch(**fx["ego"])
    k, H = fx["meta"]["k"], int(fx["meta"].get("hidden", 64))
    m = OracleMainmodel(9, H, 32, 4)
    m.load_state_dict(fx["state"], strict=False)
    gate_u, feat_u = draw_noise_like_reference(g.batch_num_nodes().tolist(), H, fx["meta"]["noise_seed"])
    logm = k if fx["meta"].get("recons_type", "adj") == "logM" else 0
    eng, losses, emb = _run_engine(m, g, e, k, gate_u, feat_u, recon_logm_steps=logm)
    truth_out, truth_grads = fp64_truth(m, g, e, gate_u, feat_u, recon_logm_steps=logm)
    check_against_truth(eng, losses, emb, fx["out"], fx["grads"], truth_out, truth_grads, tag="golden_" + os.path.basename(path)[:-3])
    # direct comparison with the recorded reference numbers as well (these batches are tiny: fp32 noise is small)
    for i, name in enumerate(("KL", "contrastive", "recon")):
        assert abs(float(losses[i]) - float(fx["out"][name])) <= FWD_TOL * abs(float(fx["out"][name])), name
    for name in ("interaction_map", "Z", "noisy", "graph_readout"):
        assert rel(emb[name], fx["out"][name]) <= FWD_TOL, (name, rel(emb[name], fx["out"][name]))
    sd = eng.state_dict()
    for n, t in fx["state_after"].items():
        if t.dtype.is_floating_point:
            assert rel(sd[n], t) <= 1e-5, n


@pytest.mark.parametrize("seed,B,k", [(11, 128, 1), (12, 96, 2), (13, 40, 3)])
def test_parity_vs_faithful_oracle(seed, B, k):
    """config 1 size (B=128): loop-for-loop oracle incl. the dense N x N reconstruction."""
    g = synth_batch(seed, B)
    e = ego_batch_ref(g, k)
    torch.manual_seed(seed)
    m = OracleMainmodel(9)
    x = normalize_rows(torch.from_numpy(g.x))
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    gate_u, feat_u = draw_noise_like_reference(g.batch_num_nodes().tolist(), 64, seed + 100)
    out = m.forward_faithful(tgraph_from_ref(g), x, tgraph_from_ego(e), x[en], gate_u, feat_u)
    ref_grads = oracle_grads(m, out)
    m.zero_grad()
    eng, losses, emb = _run_engine(m, g, e, k, gate_u, feat_u)
    truth_out, truth_grads = fp64_truth(m, g, e, gate_u, feat_u)
    check_against_truth(eng, losses, emb, out, ref_grads, truth_out, truth_grads, tag="h64_faithful_b%d_k%d" % (B, k))


@pytest.mark.parametrize("B,k", [(4096, 1)])
def test_parity_full_size_vs_vectorised_oracle_fp64(B, k):
    """config 2 size (B=4096, ~61k nodes, ~192k ego rows): fp64 vectorised oracle = truth, fp32 vectorised oracle =
    the reference-precision yardstick."""
    g = synth_batch(21, B)
    e = ego_batch_ref(g, k)
    torch.manual_seed(21)
    m = OracleMainmodel(9)
    gate_u, feat_u = draw_noise_like_reference(g.batch_num_nodes().tolist(), 64, 121)
    eng, losses, emb = _run_engine(m, g, e, k, gate_u, feat_u)
    x = normalize_rows(torch.from_numpy(g.x))
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    out = m.forward_vectorised(tgraph_from_ref(g), x, tgraph_from_ego(e), en, gate_u, feat_u)
    ref_grads = oracle_grads(m, out)
    m.zero_grad()
    truth_out, truth_grads = fp64_truth(m, g, e, gate_u, feat_u)
    rep = check_against_truth(eng, losses, emb, out, ref_grads, truth_out, truth_grads, tag="h64_vectorised_b%d_k%d" % (B, k))
    worst = max(rep, key=lambda r: r[1])
    print("worst cuda-vs-fp64 %.3e (%s); fp32 torch oracle on the same tensor %.3e" % (worst[1], worst[0], worst[2]))


def test_extract_backward_external_upstream_gradient():
    """Backward of the feature path for a downstream head (fine-tuning, models.py:501-520): gradients of <G, Z> for a
    random upstream gradient G against autograd of the fp64 oracle."""
    g = synth_batch(21, 96)
    e = ego_batch_ref(g, 1)
    torch.manual_seed(5)
    m = OracleMainmodel(9)
    gate_u, feat_u = draw_noise_like_reference(g.batch_num_nodes().tolist(), 64, 7)
    G = torch.randn(g.num_nodes, 64, generator=torch.Generator().manual_seed(3))
    m64 = OracleMainmodel(9).double()
    m64.load_state_dict({n: (v.double() if v.dtype.is_floating_point else v) for n, v in m.state_dict().items()})
    x = normalize_rows(torch.from_numpy(g.x).double())
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    out = m64.forward_vectorised(tgraph_from_ref(g), x, tgraph_from_ego(e), en, gate_u.double(), feat_u.double())
    (out["Z"] * G.double()).sum().backward()
    truth = {n: p.grad.detach().clone() for n, p in m64.named_parameters() if p.grad is not None}
    from scgib_b200.engine import DeviceBatch
    eng = engine_from_oracle(m, DEV)
    pg = product_graph(g, DEV)
    b = DeviceBatch(pg, product_ego_from_ref(pg, e, 1, DEV), pg.ndata["x"])
    _, emb = eng.forward(b, gate_u.to(DEV), feat_u.to(DEV), want=True, update_running=False)
    assert rel(emb["Z"], out["Z"]) <= 1e-5
    eng.extract_backward(G.to(DEV))
    torch.cuda.synchronize()
    errs = []
    for n, gv in eng.grad_views().items():
        if n not in truth or is_zero_grad_param(n):
            continue
        errs.append(rel(gv, truth[n]))
    errs.sort()
    assert errs[len(errs) // 2] <= GRAD_TOL_MEDIAN and errs[-1] <= GRAD_TOL_MAX, errs[-5:]


def test_forward_backward_deterministic():
    """No float atomics anywhere: two runs are bit-identical."""
    g = synth_batch(31, 512)
    e = ego_batch_ref(g, 1)
    torch.manual_seed(31)
    m = OracleMainmodel(9)
    gate_u, feat_u = draw_noise_like_reference(g.batch_num_nodes().tolist(), 64, 131)
    eng1, l1, emb1 = _run_engine(m, g, e, 1, gate_u, feat_u)
    g1 = eng1.grads.clone()
    eng2, l2, emb2 = _run_engine(m, g, e, 1, gate_u, feat_u)
    assert torch.equal(l1, l2) and torch.equal(emb1["Z"], emb2["Z"]) and torch.equal(g1, eng2.grads)


def test_adam_matches_torch():
    from scgib_b200.engine import PretrainEngine
    eng = PretrainEngine(9, device=DEV, seed=3)
    p0 = eng.params.clone()
    ref = torch.nn.Parameter(p0.clone())
    opt = torch.optim.Adam([ref], lr=1e-4, weight_decay=5e-5)
    gen = torch.Generator(device=DEV).manual_seed(0)
    for step in range(5):
        gr = torch.randn(eng.total, device=DEV, generator=gen)
        eng.grads.copy_(gr)
        eng.adam_step(lr=1e-4, weight_decay=5e-5)
        ref.grad = gr.clone()
        opt.step()
    assert rel(eng.params, ref.detach()) <= 1e-6
    assert rel(eng.params - p0, ref.detach() - p0) <= 2e-4      # p - p0 cancels ~4 digits of an fp32 parameter


def test_train_steps_follow_oracle_trajectory():
    """5 optimiser steps (forward + backward + Adam) track the oracle's loss trajectory."""
    from scgib_b200.engine import DeviceBatch
    from scgib_b200.graph import khop_ego_batch
    g = synth_batch(41, 64)
    e = ego_batch_ref(g, 1)
    torch.manual_seed(41)
    m = OracleMainmodel(9)
    opt = torch.optim.Adam(m.parameters(), lr=1e-4, weight_decay=5e-5)        # exp_pretraining.py:86, 386
    eng = engine_from_oracle(m, DEV)
    pg = product_graph(g, DEV)
    b = DeviceBatch(pg, khop_ego_batch(pg, 1), pg.ndata["x"])
    x = normalize_rows(torch.from_numpy(g.x))
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    tg, te = tgraph_from_ref(g), tgraph_from_ego(e)
    for step in range(5):
        gate_u, feat_u = draw_noise_like_reference(g.batch_num_nodes().tolist(), 64, 200 + step)
        opt.zero_grad()
        out = m.forward_faithful(tg, x, te, x[en], gate_u, feat_u)
        loss = out["KL"] + out["recon"] + out["contrastive"]
        loss.backward()
        opt.step()
        got = eng.train_step(b, gate_u.to(DEV), feat_u.to(DEV), lr=1e-4)
        # Adam normalises every gradient to a +-lr step, so fp32 rounding differences in tiny gradients are
        # amplified step over step: the trajectory is compared at 1e-3
        assert abs(float(got[3]) - float(loss)) <= 1e-3 * abs(float(loss)), (step, float(got[3]), float(loss))


def test_bad_arguments_raise():
    from scgib_b200 import _lib
    from scgib_b200.engine import PretrainEngine
    with pytest.raises(RuntimeError):
        PretrainEngine(9, hidden=48, device=DEV)          # unsupported width -> SCGIB_E_SHAPE
    with pytest.raises(RuntimeError):
        PretrainEngine(9, device="cpu")                   # no CPU fallback


def _edge_case_batch(kind):
    if kind == "pairs":            # the smallest graphs the reference accepts (per-graph BatchNorm / unbiased std need n >= 2)
        return batch_ref([path_graph(2, seed=i) for i in range(7)])
    if kind == "single":           # B = 1: the contrastive loss has no negatives, the KL graph is the only graph
        return synth_batch(21, 1)
    if kind == "peptides":         # ~150-node graphs (BASELINE configs[4] shape): long per-graph loops, tiles spanning few graphs
        return synth_batch(22, 6, "peptides")
    if kind == "ragged":           # 2-node graphs next to 150-node graphs, a star (degree 12) and a 40-ring
        star = graph_from_bonds(13, [(0, i) for i in range(1, 13)], seed=3)
        ring = graph_from_bonds(40, [(i, (i + 1) % 40) for i in range(40)], seed=4)
        mols = [path_graph(2, seed=1), synth_batch(23, 1, "peptides"), star, path_graph(3, seed=2), ring,
                synth_batch(24, 1, "peptides"), path_graph(2, seed=5)]
        return batch_ref(mols)
    if kind == "macrocycles":      # head-to-tail and 65 .. 200-atom ring closures, one 420-atom ring: neighbours beyond the gather window
        return macrocycle_batch(25, 5)
    if kind == "shuffled":         # Peptides-shape molecules with the atom order permuted inside each graph
        return shuffle_nodes(synth_batch(26, 5, "peptides"), 27)
    raise ValueError(kind)


@pytest.mark.parametrize("kind,k", [("pairs", 1), ("peptides", 1), ("peptides", 3), ("ragged", 2), ("macrocycles", 2), ("shuffled", 1)])
def test_parity_edge_shapes(kind, k):
    """Ragged / extreme batches against the faithful oracle (same policy as test_parity_vs_faithful_oracle)."""
    g = _edge_case_batch(kind)
    e = ego_batch_ref(g, k)
    torch.manual_seed(7)
    m = OracleMainmodel(9)
    x = normalize_rows(torch.from_numpy(g.x))
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    gate_u, feat_u = draw_noise_like_reference(g.batch_num_nodes().tolist(), 64, 300)
    out = m.forward_faithful(tgraph_from_ref(g), x, tgraph_from_ego(e), x[en], gate_u, feat_u)
    ref_grads = oracle_grads(m, out)
    m.zero_grad()
    eng, losses, emb = _run_engine(m, g, e, k, gate_u, feat_u)
    truth_out, truth_grads = fp64_truth(m, g, e, gate_u, feat_u)
    check_against_truth(eng, losses, emb, out, ref_grads, truth_out, truth_grads)


def test_single_graph_batch():
    """B = 1: the contrastive loss is -log(e^s / e^s) = 0 (no negatives) - compared absolutely; everything else as usual."""
    g = _edge_case_batch("single")
    e = ego_batch_ref(g, 2)
    torch.manual_seed(7)
    m = OracleMainmodel(9).double()
    x = normalize_rows(torch.from_numpy(g.x)).double()
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    gate_u, feat_u = draw_noise_like_reference(g.batch_num_nodes().tolist(), 64, 300)
    out = m.forward_faithful(tgraph_from_ref(g), x, tgraph_from_ego(e), x[en], gate_u.double(), feat_u.double())
    eng, losses, emb = _run_engine(m.float(), g, e, 2, gate_u, feat_u)
    assert torch.isfinite(losses).all() and torch.isfinite(eng.grads).all()
    assert abs(float(losses[1])) <= 1e-6 and abs(float(out["contrastive"])) <= 1e-12
    for i, name in ((0, "KL"), (2, "recon")):
        assert abs(float(losses[i]) - float(out[name])) <= 1e-5 * abs(float(out[name])), name
    for name in ("interaction_map", "Z", "noisy", "graph_readout"):
        assert rel(emb[name].cpu(), out[name].detach()) <= 1e-5, name


@pytest.mark.parametrize("seed,B,k,shape", [(41, 96, 1, "pcqm"), (42, 64, 2, "pcqm"), (43, 48, 3, "pcqm"), (44, 4, 2, "peptides")])
def test_logm_reconstruction_vs_faithful_oracle(seed, B, k, shape):
    """--recons_type logM (models.py:770-782 + util.py:60-91): the sparse Gram/pair formulation on the GPU against the
    dense per-graph loop of the oracle, forward and gradients."""
    g = synth_batch(seed, B, shape)
    e = ego_batch_ref(g, k)
    torch.manual_seed(seed)
    m = OracleMainmodel(9)
    x = normalize_rows(torch.from_numpy(g.x))
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    gate_u, feat_u = draw_noise_like_reference(g.batch_num_nodes().tolist(), 64, seed + 100)
    out = m.forward_faithful(tgraph_from_ref(g), x, tgraph_from_ego(e), x[en], gate_u, feat_u, recon_logm_steps=k)
    ref_grads = oracle_grads(m, out)
    m.zero_grad()
    eng, losses, emb = _run_engine(m, g, e, k, gate_u, feat_u, recon_logm_steps=k)
    truth_out, truth_grads = fp64_truth(m, g, e, gate_u, feat_u, recon_logm_steps=k)
    check_against_truth(eng, losses, emb, out, ref_grads, truth_out, truth_grads)


def test_eval_mode_uses_running_statistics():
    """model.eval(): GIN BatchNorms and the compressor BatchNorm normalise with their running statistics.  Two training
    forwards (to move the running statistics away from their initial values), then an eval forward, against the torch
    oracle driven the same way."""
    g = synth_batch(91, 80)
    e = ego_batch_ref(g, 1)
    torch.manual_seed(91)
    m = OracleMainmodel(9)
    x = normalize_rows(torch.from_numpy(g.x))
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    tg, te = tgraph_from_ref(g), tgraph_from_ego(e)
    from scgib_b200.engine import DeviceBatch
    from scgib_b200.graph import khop_ego_batch
    eng = engine_from_oracle(m, DEV)
    pg = product_graph(g, DEV)
    b = DeviceBatch(pg, khop_ego_batch(pg, 1), pg.ndata["x"], normalize_x=True)
    m.train()
    for step in range(2):
        gate_u, feat_u = draw_noise_like_reference(g.batch_num_nodes().tolist(), 64, 500 + step)
        m.forward_faithful(tg, x, te, x[en], gate_u, feat_u)
        eng.forward(b, gate_u.to(DEV), feat_u.to(DEV))
    gate_u, feat_u = draw_noise_like_reference(g.batch_num_nodes().tolist(), 64, 600)
    m.eval()
    with torch.no_grad():
        out = m.forward_faithful(tg, x, te, x[en], gate_u, feat_u)
    b.eval_mode = True
    before = eng.bn_running.clone()
    losses, emb = eng.forward(b, gate_u.to(DEV), feat_u.to(DEV), want=True, update_running=False)
    assert torch.equal(before, eng.bn_running)                      # eval never updates the running statistics
    for i, name in enumerate(("KL", "contrastive", "recon")):
        assert abs(float(losses[i]) - float(out[name])) <= 2e-5 * abs(float(out[name])), (name, float(losses[i]), float(out[name]))
    for name in ("interaction_map", "Z", "noisy", "graph_readout"):
        assert rel(emb[name].cpu(), out[name]) <= 2e-5, (name, rel(emb[name].cpu(), out[name]))
    with pytest.raises(RuntimeError):
        eng.backward()                                              # the backward is the training-mode one


def test_checkpoint_resume_is_bit_identical(tmp_path):
    """PretrainEngine.checkpoint / restore: 4 training steps == 2 steps + save + load into a fresh engine + 2 steps, bit for
    bit (parameters, Adam moments, BN running statistics, noise stream)."""
    from scgib_b200.engine import PretrainEngine
    from scgib_b200.synth import synth_batch as product_synth
    batches = [product_synth(100 + i, 64).to(DEV) for i in range(4)]

    def steps(eng, lo, hi):
        out = []
        for i in range(lo, hi):
            b = eng.make_batch(batches[i], 1)
            out.append(eng.train_step(b).clone())
        return out

    a = PretrainEngine(9, gin_layers=4, device=DEV, seed=11)
    la = steps(a, 0, 4)
    b1 = PretrainEngine(9, gin_layers=4, device=DEV, seed=11)
    lb = steps(b1, 0, 2)
    torch.save(b1.checkpoint(), tmp_path / "ck.pt")
    b2 = PretrainEngine(9, gin_layers=4, device=DEV, seed=999)          # different init: everything must come from the file
    b2.restore(torch.load(tmp_path / "ck.pt", weights_only=False))
    lb += steps(b2, 2, 4)
    for x, y in zip(la, lb):
        assert torch.equal(x, y)
    assert torch.equal(a.params, b2.params) and torch.equal(a.exp_avg_sq, b2.exp_avg_sq)
    assert torch.equal(a.bn_running, b2.bn_running) and a.step_count == b2.step_count == 4


@pytest.mark.parametrize("kin,csr", [(64, False), (32, False), (64, True)])
def test_gin_layer_backward_op(kin, csr):
    """scgib_gin_layer_bwd_f32 (the per-layer unit of the backward) against torch autograd through GINConv -> BatchNorm
    (train) -> ReLU, with the upstream gradient given at the layer output or gathered through the CSR."""
    from scgib_b200 import ops
    from oracle.scgib_oracle import GINConvRef, MLP
    g = synth_batch(5, 400)
    tg = tgraph_from_ref(g)
    V = g.num_nodes
    torch.manual_seed(kin + int(csr))
    conv = GINConvRef(MLP(kin, 64, 64)).double()
    bnm = torch.nn.BatchNorm1d(64).double().train()
    with torch.no_grad():
        bnm.weight.uniform_(0.5, 1.5); bnm.bias.uniform_(-0.3, 0.3)
    h = torch.randn(V, kin, dtype=torch.float64)
    neigh = torch.zeros_like(h).index_add(0, tg.dst, h[tg.src])
    a_ref = (h + neigh).requires_grad_(True)
    lin1, lin2 = conv.apply_func.mlp[0], conv.apply_func.mlp[2]
    r_ref = torch.relu(lin1(a_ref))
    y_ref = lin2(r_ref)
    out = torch.relu(bnm(y_ref))
    g_up = torch.randn(V, 64, dtype=torch.float64)
    G = g_up + torch.zeros_like(g_up).index_add(0, tg.dst, g_up[tg.src]) if csr else g_up   # transpose of the aggregation
    (out * G).sum().backward()
    mean, var = y_ref.mean(0), y_ref.var(0, unbiased=False)
    bn = torch.stack([mean, 1.0 / torch.sqrt(var + 1e-5), bnm.weight, bnm.bias]).detach().float().to(DEV)
    pg = product_graph(g, DEV)
    res = ops.gin_layer_bwd(g_up.float().to(DEV), y_ref.detach().float().to(DEV), r_ref.detach().float().to(DEV),
                            a_ref.detach().float().to(DEV), bn, lin1.weight.detach().float().to(DEV),
                            lin2.weight.detach().float().to(DEV), indptr=pg.indptr if csr else None,
                            indices=pg.indices if csr else None)
    want = (a_ref.grad, lin1.weight.grad, lin1.bias.grad, lin2.weight.grad, lin2.bias.grad, bnm.weight.grad, bnm.bias.grad)
    names = ("g_a", "dW1", "db1", "dW2", "db2", "dgamma", "dbeta")
    gmax = max(float(w.abs().max()) for w in want)
    for name, got, w in zip(names, res, want):
        if name == "db2":        # a bias in front of a BatchNorm: mathematically zero
            assert float(got.abs().max()) <= 1e-5 * gmax
            continue
        assert rel(got.cpu(), w) <= 5e-5, (name, rel(got.cpu(), w))


def test_loss_operators_recon_and_contrastive():
    """scgib_recon_adj_f32 / scgib_contrastive_f32 (value + gradient) against the oracle's dense formulas in fp64."""
    from scgib_b200 import ops
    g = synth_batch(8, 200)
    tg = tgraph_from_ref(g)
    torch.manual_seed(8)
    m = OracleMainmodel(9).double()
    Z = (torch.randn(g.num_nodes, 64, dtype=torch.float64) * 0.3).requires_grad_(True)
    rec = m.loss_recon_adj(Z, tg)
    rec.backward()
    pg = product_graph(g, DEV)
    loss, gZ = ops.recon_adj(Z.detach().float().to(DEV), pg.indptr, pg.indices, scale=0.5)
    assert abs(float(loss) - float(rec)) <= 1e-5 * abs(float(rec))
    assert rel(gZ.cpu(), 0.5 * Z.grad) <= 2e-5
    for B in (1, 7, 300, 1100):
        core = (torch.randn(B, 64, dtype=torch.float64) * 2).requires_grad_(True)
        ro = (torch.randn(B, 64, dtype=torch.float64) * 3).requires_grad_(True)
        con = m.batched_semi_loss(core, ro, B)
        con.backward()
        loss, g1, g2 = ops.contrastive(core.detach().float().to(DEV), ro.detach().float().to(DEV), scale=2.0)
        if B == 1:
            assert abs(float(loss)) <= 1e-6
            continue
        assert abs(float(loss) - float(con)) <= 1e-5 * abs(float(con)), B
        assert rel(g1.cpu(), 2.0 * core.grad) <= 5e-5 and rel(g2.cpu(), 2.0 * ro.grad) <= 5e-5, B
