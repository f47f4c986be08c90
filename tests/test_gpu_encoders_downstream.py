"""--encoder GraphSAGE / GCN after pre-training: the logM loss operator at hidden 64 / 128, logM pre-training, eval-mode
features, fine-tuning and domain adaptation around GraphSAGE / GCN checkpoints, and the exp_pep_func_5.py CLI, against the fp64
oracle.  Thresholds follow tests/helpers.py: values 1e-5 relative; gradients median <= 5e-5 and every tensor <= 5e-3."""
import os
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle.graph_ref import ego_batch_ref, synth_batch
from oracle.scgib_oracle import (OracleDomainAdapt, OracleFinetune, OracleMainmodel, loss_recon_logm, make_encoder,
                                 normalize_rows, tgraph_from_ego, tgraph_from_ref)
from tests.helpers import GRAD_TOL_MAX, GRAD_TOL_MEDIAN, product_graph, rel

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _args(**kw):
    a = types.SimpleNamespace(recons_type="adj", useAtt=1, readout_f="sum", d_transfer=32, device=DEV, batch_size=128,
                              task="graph_classification", dataset="Peptides-func", k_transition=1)
    a.__dict__.update(kw)
    return a


def _grad_errors(got, ref, skip_core_half=()):
    """Max-norm relative errors of every reference gradient; mathematically-zero ones (bias in front of a BatchNorm, the
    softmax-shift-invariant attention bias) must be zero up to rounding."""
    assert set(got) == set(ref), (sorted(set(got) ^ set(ref)))
    gmax = max(float(v.abs().max()) for v in ref.values())
    errs = []
    for n, gref in ref.items():
        g = got[n].detach().cpu()
        if n in skip_core_half:                       # attn_layer.weight: the core half is exactly zero, compare the candidates
            H = g.shape[1] // 2
            assert float(g[:, :H].abs().max()) == 0.0, n
            g, gref = g[:, H:], gref[:, H:]
        if float(gref.abs().max()) <= 1e-6 * gmax:
            assert float(g.abs().max()) <= 1e-4 * gmax, n
            continue
        errs.append((rel(g, gref), n))
    errs.sort()
    assert errs[len(errs) // 2][0] <= GRAD_TOL_MEDIAN and errs[-1][0] <= GRAD_TOL_MAX, errs[-3:]
    return errs


# ------------------------------------------------------------------------------------------------ 1. logM operator
@pytest.mark.parametrize("shape,B", [("pcqm", 40), ("peptides", 6)])
@pytest.mark.parametrize("H", [64, 128])
@pytest.mark.parametrize("k", [1, 2, 3])
def test_recon_logm_operator_matches_oracle(shape, B, H, k):
    from scgib_b200 import ops
    g = synth_batch(300 + k + H, B, shape)
    tg = tgraph_from_ref(g)
    torch.manual_seed(H + k)
    Z = (torch.randn(g.num_nodes, H, dtype=torch.float64) * 0.15).requires_grad_(True)
    ref = loss_recon_logm(Z, tg, k)
    ref.backward()
    pg = product_graph(g, DEV)
    Zd = Z.detach().float().to(DEV)
    loss, gZ, status = ops.recon_logm(Zd, pg.graph_ptr, pg.indptr, pg.indices, k, scale=0.5)
    assert int(status) == 0
    assert abs(float(loss) - float(ref)) <= 1e-5 * abs(float(ref)), (float(loss), float(ref))
    assert rel(gZ.cpu(), 0.5 * Z.grad) <= 2e-5, rel(gZ.cpu(), 0.5 * Z.grad)
    loss2, none, _ = ops.recon_logm(Zd, pg.graph_ptr, pg.indptr, pg.indices, k, want_grad=False)
    assert none is None and torch.equal(loss2, loss)             # fixed-order reductions: the same value without the gradient


# ------------------------------------------------------------------------------------------------ 2. logM pre-training
def _mainmodel(encoder, hidden, k, state, **kw):
    import models
    m = models.Mainmodel(_args(k_transition=k, **kw), 9, hidden_dim=hidden, num_layers=4, num_heads=4, k_transition=k,
                         encoder=encoder)
    missing, unexpected = m.load_state_dict(state, strict=False)
    assert not unexpected, unexpected
    return m.to(DEV)


@pytest.mark.parametrize("encoder,hidden,k", [("GraphSAGE", 64, 1), ("GCN", 64, 2), ("GraphSAGE", 128, 2), ("GCN", 128, 1)])
def test_logm_pretraining_matches_oracle(encoder, hidden, k, monkeypatch):
    from scgib_b200.graph import khop_ego_batch
    g = synth_batch(410 + hidden + k, 24)
    e = ego_batch_ref(g, k)
    torch.manual_seed(11)
    ref = OracleMainmodel(9, hidden, 32, 4, encoder=encoder).double()
    gate_u, feat_u = torch.rand(g.num_nodes), torch.rand(g.num_nodes, hidden)
    m = _mainmodel(encoder, hidden, k, {n: t.float() for n, t in ref.state_dict().items()}, recons_type="logM")
    pg = product_graph(g, DEV)
    monkeypatch.setattr(m, "_noise", lambda N, dev: (gate_u.to(dev), feat_u.to(dev)))
    m.train()
    _, kl, con, rec = m.forward(pg, F.normalize(pg.ndata["x"].float()), khop_ego_batch(pg, k), None, None, 1, None, 2, DEV,
                                g.num_graphs)
    (kl + rec + con).backward()
    xr = normalize_rows(torch.from_numpy(g.x)).double()
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    out = ref.forward_faithful(tgraph_from_ref(g), xr, tgraph_from_ego(e), xr[en], gate_u.double(), feat_u.double(),
                               recon_logm_steps=k)
    (out["KL"] + out["recon"] + out["contrastive"]).backward()
    for name, got in (("KL", kl), ("contrastive", con), ("recon", rec)):
        assert abs(float(got) - float(out[name])) <= 1e-5 * abs(float(out[name])), (name, float(got), float(out[name]))
    refg = {n: p.grad for n, p in ref.named_parameters() if p.grad is not None}
    got = {n: p.grad for n, p in m.named_parameters() if p.grad is not None}
    _grad_errors({n: got[n] for n in refg}, refg, skip_core_half=("attn_layer.weight",))


# ------------------------------------------------------------------------------------------------ 3. eval-mode features
@pytest.mark.parametrize("encoder,hidden", [("GraphSAGE", 64), ("GCN", 128)])
def test_eval_extract_features_matches_oracle(encoder, hidden, monkeypatch):
    from scgib_b200.graph import khop_ego_batch
    g = synth_batch(520 + hidden, 30)
    e = ego_batch_ref(g, 1)
    torch.manual_seed(13)
    ref = OracleMainmodel(9, hidden, 32, 4, encoder=encoder).double()
    bn = ref.compressor[1]
    with torch.no_grad():                               # non-trivial running statistics of compressor.1
        bn.running_mean.copy_(torch.randn(hidden, dtype=torch.float64) * 0.3)
        bn.running_var.copy_(torch.rand(hidden, dtype=torch.float64) * 2 + 0.2)
    gate_u, feat_u = torch.rand(g.num_nodes), torch.rand(g.num_nodes, hidden)
    m = _mainmodel(encoder, hidden, 1, {n: t.float() if t.dtype.is_floating_point else t for n, t in ref.state_dict().items()})
    m.eval()
    ref.eval()
    monkeypatch.setattr(m, "_noise", lambda N, dev: (gate_u.to(dev), feat_u.to(dev)))
    pg = product_graph(g, DEV)
    xr = normalize_rows(torch.from_numpy(g.x)).double()
    t = m.transfer_d(xr.float().to(DEV)).detach()
    before = {n: v.clone() for n, v in m.state_dict().items() if "compressor.1" in n}
    imap, kl_t, noisy, readout = m.extract_features(pg.batch_num_nodes(), pg, t, khop_ego_batch(pg, 1), None, DEV)
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    with torch.no_grad():
        bx = ref.transfer_d(xr)
        r_imap, _, r_noisy, r_readout = ref.extract_features(tgraph_from_ref(g), bx, tgraph_from_ego(e), bx[en], gate_u.double(),
                                                             feat_u.double())
    for name, got, want in (("interaction_map", imap, r_imap), ("noisy", noisy, r_noisy), ("graph_readout", readout, r_readout)):
        assert rel(got, want) <= 1e-5, (name, rel(got, want))
    for n, v in before.items():                          # eval: the running statistics stay
        assert torch.equal(m.state_dict()[n], v), n


# ------------------------------------------------------------------------------------------------ 4. fine-tuning
def _oracle_wrapper(cls, encoder, hidden, **kw):
    inner = OracleMainmodel(9, hidden, 32, 4, encoder=encoder)
    with torch.no_grad():
        bn = inner.compressor[1]
        bn.running_mean.copy_(torch.randn(hidden) * 0.2)
        bn.running_var.copy_(torch.rand(hidden) + 0.5)
    ref = cls(inner, 9, hidden_dim=hidden, **kw)
    # the outer, never-called encoders of the wrapper follow --encoder (state-dict keys of the product's wrapper)
    ref.Encoder1, ref.Encoder2 = make_encoder(encoder, 32, hidden), make_encoder(encoder, 32, hidden)
    return ref


def _checkpoint(tmp_path, encoder, hidden, k):
    import models
    pre = models.Mainmodel(_args(k_transition=k), 9, hidden_dim=hidden, num_layers=4, num_heads=4, k_transition=k, encoder=encoder)
    ckpt = str(tmp_path / ("pre_training_synth_%s_%d_4_%d.pt" % (encoder, hidden, k)))
    torch.save(pre, ckpt)
    return ckpt


@pytest.mark.parametrize("encoder,hidden,k,regression", [("GraphSAGE", 64, 1, False), ("GCN", 64, 2, True),
                                                         ("GraphSAGE", 128, 2, True), ("GCN", 128, 1, False)])
def test_finetuning_sage_gcn_matches_oracle(encoder, hidden, k, regression, tmp_path, monkeypatch):
    import models
    from scgib_b200.graph import khop_ego_batch
    B, C = 40, 1 if regression else 10
    g = synth_batch(600 + hidden + k, B)
    e = ego_batch_ref(g, k)
    torch.manual_seed(17 + k)
    task = "graph_regression" if regression else "graph_classification"
    ref = _oracle_wrapper(OracleFinetune, encoder, hidden, num_classes=C, task=task, regression_dataset=regression)
    args = _args(k_transition=k, task=task, dataset="ZINC" if regression else "Peptides-func")
    m = models.Mainmodel_finetuning(args, 9, hidden, 4, 4, k, C, _checkpoint(tmp_path, encoder, hidden, k), encoder)
    missing, unexpected = m.load_state_dict(ref.state_dict(), strict=False)
    assert not unexpected, unexpected
    m = m.to(DEV).train()
    ref = ref.double().train()
    assert sorted(n for n, p in m.named_parameters() if p.requires_grad) == sorted(n for n, p in ref.named_parameters() if p.requires_grad)
    pg = product_graph(g, DEV)
    ego = khop_ego_batch(pg, k)
    x = F.normalize(pg.ndata["x"].float())
    gate_u, feat_u = torch.rand(g.num_nodes), torch.rand(g.num_nodes, hidden)
    monkeypatch.setattr(m, "_noise", lambda N, dev: (gate_u.to(dev), feat_u.to(dev)))
    scores, z1, z2, z3 = m.forward(pg, x, ego, None, 1, None, 2, DEV, B)
    assert (z1, z2, z3) == (0, 0, 0)
    xr = normalize_rows(torch.from_numpy(g.x)).double()
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    tg, te = tgraph_from_ref(g), tgraph_from_ego(e)
    out = ref(tg, xr, te, xr[en], gate_u.double(), feat_u.double())
    assert rel(scores.detach().cpu(), out["scores"].detach()) <= 1e-5
    if regression:
        targets = torch.randn(B, 1)
        m.lossMAE(scores, targets.to(DEV)).backward()
        F.l1_loss(out["scores"], targets.double()).backward()
    else:
        targets = (torch.rand(B, C) < 0.3).float()
        (m.loss(scores, targets.to(DEV)) / 2).backward()
        (F.binary_cross_entropy(out["scores"], targets.double()) / 2).backward()
    refg = {n: p.grad for n, p in ref.named_parameters() if p.grad is not None}
    got = {n: p.grad for n, p in m.named_parameters() if p.grad is not None}
    _grad_errors(got, refg)
    # the loaded compressor.1 advanced as B per-graph BatchNorm calls do
    sd, rsd = m.state_dict(), ref.state_dict()
    for n in ("model.compressor.1.running_mean", "model.compressor.1.running_var"):
        assert rel(sd[n].cpu(), rsd[n]) <= 1e-5, n
    assert int(sd["model.compressor.1.num_batches_tracked"]) == int(rsd["model.compressor.1.num_batches_tracked"])
    # evaluate_network: model.eval(), running statistics, no autograd
    m.eval()
    ref.eval()
    gu2, fu2 = torch.rand(g.num_nodes), torch.rand(g.num_nodes, hidden)
    monkeypatch.setattr(m, "_noise", lambda N, dev: (gu2.to(dev), fu2.to(dev)))
    with torch.no_grad():
        s_eval, _, _, _ = m.forward(pg, x, ego, None, 1, None, 2, DEV)
        r_eval = ref(tg, xr, te, xr[en], gu2.double(), fu2.double())["scores"]
    assert rel(s_eval.cpu(), r_eval) <= 1e-5
    assert int(m.state_dict()["model.compressor.1.num_batches_tracked"]) == int(rsd["model.compressor.1.num_batches_tracked"])


# ------------------------------------------------------------------------------------------------ 5. domain adaptation
@pytest.mark.parametrize("encoder,hidden,k", [("GraphSAGE", 64, 2), ("GCN", 64, 1), ("GraphSAGE", 128, 1)])
def test_domainadapt_sage_gcn_matches_oracle(encoder, hidden, k, tmp_path, monkeypatch):
    import models
    from scgib_b200.graph import khop_ego_batch
    B = 32
    g = synth_batch(700 + hidden + k, B)
    e = ego_batch_ref(g, k)
    torch.manual_seed(19 + k)
    ref = _oracle_wrapper(OracleDomainAdapt, encoder, hidden, num_classes=10)
    m = models.Mainmodel_domainadapt(_args(k_transition=k), 9, hidden, 4, 4, k, 10, _checkpoint(tmp_path, encoder, hidden, k), encoder)
    missing, unexpected = m.load_state_dict(ref.state_dict(), strict=False)
    assert not unexpected, unexpected
    m = m.to(DEV).train()
    ref = ref.double().train()
    pg = product_graph(g, DEV)
    gate_u, feat_u = torch.rand(g.num_nodes), torch.rand(g.num_nodes, hidden)
    monkeypatch.setattr(m, "_noise", lambda N, dev: (gate_u.to(dev), feat_u.to(dev)))
    loss = m.forward(pg, F.normalize(pg.ndata["x"].float()), khop_ego_batch(pg, k), None, None, 1, None, 2, DEV, B)
    loss.backward()
    xr = normalize_rows(torch.from_numpy(g.x)).double()
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    out = ref(tgraph_from_ref(g), xr, tgraph_from_ego(e), xr[en], gate_u.double(), feat_u.double())
    out["X_loss"].backward()
    assert abs(float(loss) - float(out["X_loss"])) <= 1e-5 * abs(float(out["X_loss"]))
    refg = {n: p.grad for n, p in ref.named_parameters() if p.grad is not None}
    got = {n: p.grad for n, p in m.named_parameters() if p.grad is not None}
    assert any(n.startswith("model.Encoder1.") for n in got) and any(n.startswith("model.Encoder2.") for n in got)
    _grad_errors(got, refg, skip_core_half=("model.attn_layer.weight",))


# ------------------------------------------------------------------------------------------------ 6. CLI
@pytest.mark.parametrize("encoder", ["GraphSAGE", "GCN"])
def test_exp_pep_func_cli_pretrain_adapt_finetune_with_encoder(encoder, tmp_path, monkeypatch):
    """exp_pep_func_5.py --encoder GraphSAGE|GCN: pre-train, domain-adapt, fine-tune with evaluation (model.eval()) on synthetic
    Peptides-shape molecules; the reference's checkpoint names and a finite test metric."""
    import exp_pep_func_5 as ep
    monkeypatch.chdir(tmp_path)
    out = str(tmp_path) + "/outputs/"
    common = ["--device", DEV, "--batch_size", "16", "--synthetic", "48", "--output_path", out, "--num_layers", "4",
              "--encoder", encoder]
    ep.args = ep.build_parser().parse_args(common + ["--pretrained_mode", "1", "--pt_epoches", "2"])
    ep.device = torch.device(DEV)
    with pytest.raises(SystemExit):
        ep.main()
    first = "Peptides-func_%s_64_4_1.pt" % encoder
    assert os.listdir(tmp_path / "outputs") == [first]
    ep.args = ep.build_parser().parse_args(common + ["--pretrained_ds", "Peptides-func", "--domain_adapt", "1",
                                                     "--adapt_epoches", "2", "--ft_epoches", "3"])
    metric = ep.main()
    assert sorted(os.listdir(tmp_path / "outputs")) == [first, "Peptides-func_%s_64_4_1_Peptides-func.pt" % encoder]
    assert metric == metric and 0.0 < metric < 10.0


def test_eval_forward_then_backward_is_refused():
    """The eval-mode core gate is forward only: a backward after it raises instead of using stale saved state."""
    from scgib_b200 import ops
    H, gp = 64, torch.tensor([0, 5, 12], dtype=torch.int32, device=DEV)
    N = 12
    p = [torch.randn(H, H, device=DEV), torch.randn(H, device=DEV), torch.ones(H, device=DEV), torch.zeros(H, device=DEV),
         torch.randn(H, device=DEV), torch.zeros(1, device=DEV)]
    gate = ops.CoreGate(H, *p)
    Hf = torch.randn(N, H, device=DEV)
    gate.forward(Hf, gp, torch.rand(N, device=DEV), torch.rand(N, H, device=DEV),
                 running=(torch.zeros(H, device=DEV), torch.ones(H, device=DEV)))
    with pytest.raises(RuntimeError):
        gate.backward(torch.zeros(N, H, device=DEV), torch.zeros(2, H, device=DEV), torch.zeros(2, H, device=DEV))
