"""Raw node features wider than 32 channels (1 <= in_dim <= 128: NCI1 37, DD 89) and fine-tuning heads with more than 64
outputs (C <= 1024: ogbg-molpcba 128 tasks, ToxCast 617), against fp64.

Operators: the input projection (fp32 and bf16 output), the transfer_d weight gradient with and without the ego rows, and
the Set2Set + predict head on its tiled output layer.  Whole steps: GIN pre-training (adjacency and logM losses, fp32 and
bf16), GraphSAGE / GCN pre-training, Mainmodel_finetuning with NaN-masked BCE and Mainmodel_domainadapt, whose s2s_rev runs
on the zero-padded H = 64 / 128 Set2Set instances.  End to end: exp_pretraining.py from F = 89 shards.

Bounds are the repository's: 1e-5 forward and the gradient policy of tests/helpers.py (median <= 5e-5, every tensor
<= 5e-3) in fp32; in bf16 the two yardsticks of tests/test_gpu_bf16.py: against the fp64 oracle with the kernels' bf16
rounding points emulated (2e-2 values, median gradient 4e-2) and against plain fp64 (2e-2 losses, or the emulated
algorithm's own deviation where that is larger)."""
import dataclasses
import os
import types

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle.graph_ref import ego_batch_ref, synth_batch
from oracle.scgib_oracle import (OracleDomainAdapt, OracleFinetune, OracleMainmodel, Set2SetRef, draw_noise_like_reference,
                                 make_encoder, normalize_rows, tgraph_from_ego, tgraph_from_ref)
from tests.helpers import (GRAD_TOL_MAX, GRAD_TOL_MEDIAN, check_against_truth, engine_from_oracle, fp64_truth, is_zero_grad_param,
                           oracle_grads, product_graph, rel)
from tests.test_gpu_op_edges import _f, _f64, _seg_graph

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
WIDTHS = [1, 9, 32, 33, 37, 64, 89, 128]
TOL_BF16, GRAD_MEDIAN_BF16 = 2e-2, 4e-2


def _wide(g, F_, seed, signed=False):
    """The batch ``g`` with F_ random features per node in place of its 9 molecular ones: uniform in [0.05, 1.05), or
    standard normal (``signed``: row directions spread over the sphere, as for embeddings)."""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((g.num_nodes, F_), dtype=np.float32) if signed else rng.random((g.num_nodes, F_), dtype=np.float32) + 0.05
    return dataclasses.replace(g, x=x)


def _csr(g):
    ip = torch.from_numpy(g.indptr.astype(np.int64))
    ix = torch.from_numpy(g.indices.astype(np.int64))
    return ip, ix, torch.repeat_interleave(torch.arange(g.num_nodes), ip[1:] - ip[:-1])


# ------------------------------------------------------------------------------------------------ operators
@pytest.mark.parametrize("F_", WIDTHS)
@pytest.mark.parametrize("out_dtype", [torch.float32, torch.bfloat16])
def test_input_proj_wide(F_, out_dtype):
    from scgib_b200 import ops
    torch.manual_seed(F_)
    N = 5003
    x = torch.rand(N, F_) * 3 - 1
    x[7] = 0.0                                                  # a zero row: the 1e-12 floor of F.normalize
    Wt = torch.randn(32, F_) / F_ ** 0.5
    ref = F.normalize(x.double()) @ Wt.double().t()
    got = ops.input_proj(x.to(DEV), Wt.to(DEV), out_dtype=out_dtype)
    torch.cuda.synchronize()
    assert got.dtype == out_dtype and got.shape == (N, 32)
    assert float(got[7].abs().max()) == 0.0
    assert rel(got.float(), ref) <= (1e-5 if out_dtype == torch.float32 else TOL_BF16), rel(got.float(), ref)


@pytest.mark.parametrize("F_", WIDTHS)
@pytest.mark.parametrize("ego", [False, True])
def test_transfer_bwd_wide(F_, ego):
    from scgib_b200 import ops
    g = _wide(synth_batch(300 + F_, 61), F_, F_)
    e = ego_batch_ref(g, 1)
    x = torch.from_numpy(g.x).double()
    xn = F.normalize(x)
    N, Ns = g.num_nodes, e.num_rows
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    torch.manual_seed(F_)
    g0, g1 = torch.randn(N, 32, dtype=torch.float64), torch.randn(Ns, 32, dtype=torch.float64)
    ip, ix, dst = _csr(g)
    sip = torch.from_numpy(e.sub_indptr.astype(np.int64))
    six = torch.from_numpy(e.sub_indices.astype(np.int64))
    sdst = torch.repeat_interleave(torch.arange(Ns), sip[1:] - sip[:-1])
    xa0 = xn + torch.zeros_like(xn).index_add(0, dst, xn[ix])
    xe = xn[en]
    xa1 = xe + torch.zeros_like(xe).index_add(0, sdst, xe[six])
    d = lambda t: t.to(DEV)
    if ego:
        ref_plain = g0.t() @ xn + g1.t() @ xn[en]
        ref_csr = g0.t() @ xa0 + g1.t() @ xa1
        plain = ops.transfer_bwd(d(x.float()), d(g0.float()), d(g1.float()), d(en.int()), normalize=True)
        csr = ops.transfer_bwd(d(x.float()), d(g0.float()), d(g1.float()), d(en.int()), normalize=True,
                               csr0=(d(ip.int()), d(ix.int())), csr1=(d(sip.int()), d(six.int())))
    else:                                                       # V1 = 0: the parent rows only
        ref_plain, ref_csr = g0.t() @ xn, g0.t() @ xa0
        plain = ops.transfer_bwd(d(x.float()), d(g0.float()), None, None, normalize=True)
        csr = ops.transfer_bwd(d(x.float()), d(g0.float()), None, None, normalize=True, csr0=(d(ip.int()), d(ix.int())))
    torch.cuda.synchronize()
    assert plain.shape == (32, F_)
    assert rel(plain, ref_plain) <= 1e-5, rel(plain, ref_plain)
    assert rel(csr, ref_csr) <= 1e-5, rel(csr, ref_csr)


def _head_case(H, C, T, sigmoid, sizes, seed):
    from scgib_b200.engine import FinetuneHead
    sizes = np.asarray(sizes)
    B, N = len(sizes), int(sizes.sum())
    tg = _seg_graph(sizes)
    torch.manual_seed(seed)
    s2s = Set2SetRef(H, T, 1).double()
    predict = nn.Sequential(nn.Linear(2 * H, H), nn.ReLU(), nn.Linear(H, C)).double()
    with torch.no_grad():
        for p in list(s2s.parameters()) + list(predict.parameters()):
            p.copy_(_f64(p))
    Z = _f64(torch.randn(N, H, dtype=torch.float64) * 0.7).requires_grad_(True)
    q = s2s(tg, Z)
    s = predict(q)
    if sigmoid:
        s = torch.sigmoid(s)
    g_r = _f64(torch.randn(B, 2 * H, dtype=torch.float64))
    g_s = _f64(torch.randn(B, C, dtype=torch.float64))
    ((q * g_r).sum() + (s * g_s).sum()).backward()

    head = FinetuneHead(H, C, n_iters=T, sigmoid=sigmoid, device=DEV)
    sd = {"s2s." + n: p for n, p in s2s.state_dict().items()}
    sd.update({"predict." + n: p for n, p in predict.state_dict().items()})
    head.load_state_dict({n: t.float() for n, t in sd.items()})
    gp = torch.from_numpy(np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)).to(DEV)
    scores, readout = head.forward(_f(Z), gp, want_readout=True)
    gZ = head.backward(_f(g_s), g_readout=_f(g_r))
    torch.cuda.synchronize()
    assert rel(scores, s) <= 1e-5, rel(scores, s)
    assert rel(readout, q) <= 1e-5, rel(readout, q)
    assert rel(gZ, Z.grad) <= 2e-5, rel(gZ, Z.grad)
    ref = {"s2s." + n: p.grad for n, p in s2s.named_parameters()}
    ref.update({"predict." + n: p.grad for n, p in predict.named_parameters()})
    for n, got in head.views(grads=True).items():
        assert rel(got, ref[n]) <= 2e-5, (n, rel(got, ref[n]))
    # reruns are bit-identical (fixed-order reductions, no float atomics)
    g1 = head.grads.clone()
    s2 = head.forward(_f(Z), gp).clone()
    head.backward(_f(g_s), g_readout=_f(g_r))
    torch.cuda.synchronize()
    assert torch.equal(s2, scores) and torch.equal(head.grads, g1)


@pytest.mark.parametrize("C", [65, 128, 617, 1024])
@pytest.mark.parametrize("H", [64, 128])
@pytest.mark.parametrize("T", [1, 2, 3])
@pytest.mark.parametrize("sigmoid", [True, False])
def test_set2set_head_wide_outputs(C, H, T, sigmoid):
    """The output layer on the tiled kernels (C > 64), with the Set2Set readout gradient g_readout added; 70 graphs cover
    partial 64-graph / 32-graph tiles and graphs of 1 to 120 nodes."""
    sizes = np.random.default_rng(C + H + T).integers(1, 120, size=70)
    _head_case(H, C, T, sigmoid, sizes, seed=C * 7 + H + T + int(sigmoid))


def test_set2set_head_wide_outputs_b8300():
    """B = 8300: the dWp2 [617][64] reduction over B rows reaches the 64-split limit of the weight-gradient scratch."""
    sizes = np.random.default_rng(8300).integers(1, 40, size=8300)
    _head_case(64, 617, 2, True, sizes, seed=8300)


# ------------------------------------------------------------------------------------------------ GIN pre-training steps
def _oracle_out(m, g, e, gate_u, feat_u, steps, emulate_bf16):
    """fp64 oracle (optionally with the bf16 rounding points of the kernels emulated) and its parameter gradients."""
    m64 = OracleMainmodel(m.transfer_d.in_features, m.attn_layer.in_features // 2, 32, len(m.Encoder1.ginlayers)).double()
    m64.load_state_dict({n: (v.double() if v.dtype.is_floating_point else v) for n, v in m.state_dict().items()})
    m64.Encoder1.emulate_bf16 = m64.Encoder2.emulate_bf16 = emulate_bf16
    x = normalize_rows(torch.from_numpy(g.x).double())
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    if steps:
        out = m64.forward_faithful(tgraph_from_ref(g), x, tgraph_from_ego(e), x[en], gate_u.double(), feat_u.double(),
                                   recon_logm_steps=steps)
    else:
        out = m64.forward_vectorised(tgraph_from_ref(g), x, tgraph_from_ego(e), en, gate_u.double(), feat_u.double())
    return out, oracle_grads(m64, out)


def _bf16_step_check(eng, losses, emb, m, g, e, gate_u, feat_u, steps):
    """The yardsticks of tests/test_gpu_bf16.py: (A) against the emulated bf16 algorithm, (B) against fp64 relative to
    that algorithm's own deviation."""
    truth_out, truth_grads = _oracle_out(m, g, e, gate_u, feat_u, steps, False)
    emul_out, emul_grads = _oracle_out(m, g, e, gate_u, feat_u, steps, True)
    for i, name in enumerate(("KL", "contrastive", "recon")):
        den = max(abs(float(truth_out[name])), 1e-3)
        got, emul, truth = float(losses[i]), float(emul_out[name]), float(truth_out[name])
        assert abs(got - emul) / den <= TOL_BF16, ("vs bf16 emulation", name, got, emul)
        assert abs(got - truth) / den <= max(TOL_BF16, 2.0 * abs(emul - truth) / den), ("vs fp64", name, got, truth)
    for name in ("interaction_map", "Z", "noisy", "graph_readout"):
        assert rel(emb[name], emul_out[name]) <= TOL_BF16, (name, rel(emb[name], emul_out[name]))
    assert torch.isfinite(eng.grads).all()
    gerr, gerr_emul, ginh = [], [], []
    for n, got in eng.grad_views().items():
        if is_zero_grad_param(n):
            continue
        truth, emul = truth_grads[n].reshape(got.shape), emul_grads[n].reshape(got.shape)
        if n == "attn_layer.weight":
            H = got.shape[1] // 2
            got, truth, emul = got[:, H:], truth[:, H:], emul[:, H:]
        gerr.append(rel(got, truth))
        gerr_emul.append(rel(got, emul))
        ginh.append(rel(emul, truth))
    med = lambda v: sorted(v)[len(v) // 2]
    assert med(gerr_emul) <= GRAD_MEDIAN_BF16, ("median gradient error vs bf16 emulation", med(gerr_emul))
    assert med(gerr) <= 1.5 * med(ginh) + GRAD_MEDIAN_BF16, ("median gradient error vs fp64", med(gerr), med(ginh))


def _pretrain_case(F_, H, k, dtype, seed, logm=False):
    from scgib_b200.engine import DeviceBatch
    from scgib_b200.graph import khop_ego_batch
    g = _wide(synth_batch(seed, 48), F_, seed, signed=True)
    e = ego_batch_ref(g, k)
    torch.manual_seed(seed)
    m = OracleMainmodel(F_, H)
    x = normalize_rows(torch.from_numpy(g.x))
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    gate_u, feat_u = draw_noise_like_reference(g.batch_num_nodes().tolist(), H, seed + 100)
    steps = k if logm else 0
    out = m.forward_faithful(tgraph_from_ref(g), x, tgraph_from_ego(e), x[en], gate_u, feat_u, recon_logm_steps=steps)
    ref_grads = oracle_grads(m, out)
    m.zero_grad()
    eng = engine_from_oracle(m, DEV, in_dim=F_, dtype=dtype)
    pg = product_graph(g, DEV)
    b = DeviceBatch(pg, khop_ego_batch(pg, k), pg.ndata["x"], normalize_x=True)
    b.recon_logm_steps = steps
    losses, emb = eng.forward(b, gate_u.to(DEV), feat_u.to(DEV), want=True)
    eng.backward()
    torch.cuda.synchronize()
    if dtype == "fp32":
        truth_out, truth_grads = fp64_truth(m, g, e, gate_u, feat_u, recon_logm_steps=steps)
    assert eng.grad_views()["transfer_d.weight"].shape == (32, F_)
    if dtype == "bf16":
        _bf16_step_check(eng, losses.cpu(), emb, m, g, e, gate_u, feat_u, steps)
    else:
        check_against_truth(eng, losses.cpu(), emb, out, ref_grads, truth_out, truth_grads)
    l2 = eng.forward(b, gate_u.to(DEV), feat_u.to(DEV), update_running=False).clone()      # bit-identical rerun
    g1 = eng.grads.clone()
    eng.backward()
    torch.cuda.synchronize()
    assert torch.equal(l2, losses.to(DEV)) and torch.equal(eng.grads, g1)


def _with_flip_retries(case, seed, *a, **kw):
    """A hidden unit within rounding distance of a ReLU kink takes different sides in two correct implementations and
    moves the gradients below it in discrete jumps (tests/helpers.py, tests/test_gpu_hidden128.py).  A gradient bound may
    therefore miss on one batch: up to three seeds.  The forward bounds hold on every attempt."""
    last = None
    for attempt in range(3):
        try:
            return case(*a, seed=seed + 1000 * attempt, **kw)
        except AssertionError as err:
            if "gradient error" not in str(err) and "'grad " not in str(err):
                raise
            last = err
    raise last


@pytest.mark.parametrize("F_", [37, 89, 128])
@pytest.mark.parametrize("H", [64, 128])
@pytest.mark.parametrize("k", [1, 2])
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_gin_pretrain_step_wide_features(F_, H, k, dtype):
    _with_flip_retries(_pretrain_case, 40 + F_ + H + k, F_, H, k, dtype)


@pytest.mark.parametrize("F_", [37, 89, 128])
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_gin_pretrain_step_wide_features_logm(F_, dtype):
    _with_flip_retries(_pretrain_case, 70 + F_, F_, 64, 2, dtype, logm=True)


def _args(**kw):
    a = types.SimpleNamespace(recons_type="adj", useAtt=1, readout_f="sum", d_transfer=32, device=DEV, batch_size=128,
                              task="graph_classification", dataset="Peptides-func", k_transition=1)
    a.__dict__.update(kw)
    return a


def _grad_errors(got, ref, skip_core_half=()):
    assert set(got) == set(ref), (sorted(set(got) ^ set(ref)))
    gmax = max(float(v.abs().max()) for v in ref.values())
    errs = []
    for n, gref in ref.items():
        g = got[n].detach().cpu()
        if n in skip_core_half:
            H = g.shape[1] // 2
            assert float(g[:, :H].abs().max()) == 0.0, n
            g, gref = g[:, H:], gref[:, H:]
        if float(gref.abs().max()) <= 1e-6 * gmax:
            assert float(g.abs().max()) <= 1e-4 * gmax, n
            continue
        errs.append((rel(g, gref), n))
    errs.sort()
    return errs


@pytest.mark.parametrize("encoder", ["GraphSAGE", "GCN"])
def test_sage_gcn_pretrain_step_f89(encoder, monkeypatch):
    import models
    from scgib_b200.graph import khop_ego_batch
    F_, H, k = 89, 64, 1
    g = _wide(synth_batch(89, 120), F_, 89)
    e = ego_batch_ref(g, k)
    torch.manual_seed(8)
    ref = OracleMainmodel(F_, H, 32, 4, encoder=encoder).double()
    gate_u, feat_u = torch.rand(g.num_nodes), torch.rand(g.num_nodes, H)
    m = models.Mainmodel(_args(k_transition=k), F_, hidden_dim=H, num_layers=4, num_heads=4, k_transition=k, encoder=encoder)
    missing, unexpected = m.load_state_dict({n: t.float() for n, t in ref.state_dict().items()}, strict=False)
    assert not unexpected, unexpected
    m = m.to(DEV).train()
    pg = product_graph(g, DEV)
    monkeypatch.setattr(m, "_noise", lambda N, dev: (gate_u.to(dev), feat_u.to(dev)))
    _, kl, con, rec = m.forward(pg, F.normalize(pg.ndata["x"].float()), khop_ego_batch(pg, k), None, None, 1, None, 2, DEV, 120)
    (kl + rec + con).backward()
    torch.cuda.synchronize()
    xr = normalize_rows(torch.from_numpy(g.x)).double()
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    out = ref.forward_vectorised(tgraph_from_ref(g), xr, tgraph_from_ego(e), en, gate_u.double(), feat_u.double())
    (out["KL"] + out["recon"] + out["contrastive"]).backward()
    for name, got in (("KL", kl), ("contrastive", con), ("recon", rec)):
        assert abs(float(got) - float(out[name])) <= 1e-5 * abs(float(out[name])), (name, float(got), float(out[name]))
    refg = {n: p.grad for n, p in ref.named_parameters() if p.grad is not None}
    got = {n: p.grad for n, p in m.named_parameters() if p.grad is not None}
    assert got["transfer_d.weight"].shape == (32, F_)
    errs = _grad_errors(got, refg)
    assert errs[len(errs) // 2][0] <= GRAD_TOL_MEDIAN and errs[-1][0] <= GRAD_TOL_MAX, errs[-3:]


# ------------------------------------------------------------------------------------------------ fine-tuning, adaptation
def _oracle_wrapper(cls, encoder, F_, hidden, **kw):
    inner = OracleMainmodel(F_, hidden, 32, 4, encoder=encoder)
    with torch.no_grad():
        bn = inner.compressor[1]
        bn.running_mean.copy_(torch.randn(hidden) * 0.2)
        bn.running_var.copy_(torch.rand(hidden) + 0.5)
    ref = cls(inner, F_, hidden_dim=hidden, **kw)
    ref.Encoder1, ref.Encoder2 = make_encoder(encoder, 32, hidden), make_encoder(encoder, 32, hidden)
    return ref


def _checkpoint(tmp_path, encoder, F_, hidden, k, dtype="fp32"):
    import models
    pre = models.Mainmodel(_args(k_transition=k, dtype=dtype), F_, hidden_dim=hidden, num_layers=4, num_heads=4, k_transition=k,
                           encoder=encoder)
    ckpt = str(tmp_path / ("pre_training_synth_%s_%d_%d_%d.pt" % (encoder, F_, hidden, k)))
    torch.save(pre, ckpt)
    return ckpt


@pytest.mark.parametrize("encoder,dtype", [("GIN", "fp32"), ("GIN", "bf16"), ("GCN", "fp32")])
@pytest.mark.parametrize("C", [128, 617])
def test_finetuning_many_tasks_masked_bce(encoder, dtype, C, tmp_path, monkeypatch):
    """Mainmodel_finetuning with 128 (ogbg-molpcba) and 617 (ToxCast) tasks at F = 37, NaN targets dropped by
    train_pep_func.masked_loss as the reference's MetricWrapper does, then the eval() scores."""
    import models
    from scgib_b200.graph import khop_ego_batch
    from train_pep_func import masked_loss
    F_, H, k, B = 37, 64, 1, 40
    g = _wide(synth_batch(900 + C, B), F_, C)
    e = ego_batch_ref(g, k)
    torch.manual_seed(C)
    ref = _oracle_wrapper(OracleFinetune, encoder, F_, H, num_classes=C)
    ref.model.Encoder1.emulate_bf16 = ref.model.Encoder2.emulate_bf16 = dtype == "bf16"    # yardstick (A) of test_gpu_bf16.py
    args = _args(k_transition=k, dtype=dtype)
    m = models.Mainmodel_finetuning(args, F_, H, 4, 4, k, C, _checkpoint(tmp_path, encoder, F_, H, k, dtype), encoder)
    missing, unexpected = m.load_state_dict(ref.state_dict(), strict=False)
    assert not unexpected, unexpected
    m = m.to(DEV).train()
    ref = ref.double().train()
    pg = product_graph(g, DEV)
    ego = khop_ego_batch(pg, k)
    x = F.normalize(pg.ndata["x"].float())
    gate_u, feat_u = torch.rand(g.num_nodes), torch.rand(g.num_nodes, H)
    monkeypatch.setattr(m, "_noise", lambda N, dev: (gate_u.to(dev), feat_u.to(dev)))
    scores, _, _, _ = m.forward(pg, x, ego, None, 1, None, 2, DEV, B)
    assert scores.shape == (B, C)
    xr = normalize_rows(torch.from_numpy(g.x)).double()
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    tg, te = tgraph_from_ref(g), tgraph_from_ego(e)
    out = ref(tg, xr, te, xr[en], gate_u.double(), feat_u.double())
    fwd_tol = TOL_BF16 if dtype == "bf16" else 1e-5
    assert rel(scores.detach().cpu(), out["scores"].detach()) <= fwd_tol
    targets = (torch.rand(B, C) < 0.3).double()
    targets[torch.rand(B, C) < 0.4] = float("nan")
    masked_loss(F.binary_cross_entropy, scores, targets.float().to(DEV)).backward()
    masked_loss(F.binary_cross_entropy, out["scores"], targets).backward()
    refg = {n: p.grad for n, p in ref.named_parameters() if p.grad is not None}
    got = {n: p.grad for n, p in m.named_parameters() if p.grad is not None}
    assert got["predict.2.weight"].shape == (C, H)
    errs = _grad_errors(got, refg)
    if dtype == "bf16":
        assert errs[len(errs) // 2][0] <= GRAD_MEDIAN_BF16, errs[-3:]
    else:
        assert errs[len(errs) // 2][0] <= GRAD_TOL_MEDIAN and errs[-1][0] <= GRAD_TOL_MAX, errs[-3:]
    m.eval()
    ref.eval()
    # eval(): against plain fp64 (the bf16 emulation of the oracle models the batch-statistics forward only; measured here,
    # the bf16 eval scores sit within 1.3e-3 of fp64 and the emulation 2.5e-2 .. 4.6e-2 away from both)
    ref.model.Encoder1.emulate_bf16 = ref.model.Encoder2.emulate_bf16 = False
    gu2, fu2 = torch.rand(g.num_nodes), torch.rand(g.num_nodes, H)
    monkeypatch.setattr(m, "_noise", lambda N, dev: (gu2.to(dev), fu2.to(dev)))
    with torch.no_grad():
        s_eval, _, _, _ = m.forward(pg, x, ego, None, 1, None, 2, DEV)
        r_eval = ref(tg, xr, te, xr[en], gu2.double(), fu2.double())["scores"]
    assert rel(s_eval.cpu(), r_eval) <= fwd_tol


@pytest.mark.parametrize("F_", [37, 89])
def test_domainadapt_wide_features(F_, tmp_path, monkeypatch):
    """r_transfer_d ends in Linear(hidden, 2 F): C = 74 / 178 on the tiled output layer; s2s_rev pads F to 64 / 128."""
    import models
    from scgib_b200.graph import khop_ego_batch
    H, k, B = 64, 1, 32
    g = _wide(synth_batch(700 + F_, B), F_, F_)
    e = ego_batch_ref(g, k)
    torch.manual_seed(19 + F_)
    ref = _oracle_wrapper(OracleDomainAdapt, "GIN", F_, H, num_classes=10)
    m = models.Mainmodel_domainadapt(_args(k_transition=k), F_, H, 4, 4, k, 10, _checkpoint(tmp_path, "GIN", F_, H, k), "GIN")
    missing, unexpected = m.load_state_dict(ref.state_dict(), strict=False)
    assert not unexpected, unexpected
    m = m.to(DEV).train()
    ref = ref.double().train()
    pg = product_graph(g, DEV)
    gate_u, feat_u = torch.rand(g.num_nodes), torch.rand(g.num_nodes, H)
    monkeypatch.setattr(m, "_noise", lambda N, dev: (gate_u.to(dev), feat_u.to(dev)))
    loss = m.forward(pg, F.normalize(pg.ndata["x"].float()), khop_ego_batch(pg, k), None, None, 1, None, 2, DEV, B)
    loss.backward()
    assert m._rev.P == (64 if F_ <= 64 else 128)
    xr = normalize_rows(torch.from_numpy(g.x)).double()
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    out = ref(tgraph_from_ref(g), xr, tgraph_from_ego(e), xr[en], gate_u.double(), feat_u.double())
    out["X_loss"].backward()
    assert abs(float(loss) - float(out["X_loss"])) <= 1e-5 * abs(float(out["X_loss"]))
    refg = {n: p.grad for n, p in ref.named_parameters() if p.grad is not None}
    got = {n: p.grad for n, p in m.named_parameters() if p.grad is not None}
    assert got["s2s_rev.lstm.weight_ih_l0"].shape == (4 * F_, 2 * F_)
    errs = _grad_errors(got, refg, skip_core_half=("model.attn_layer.weight",))
    assert errs[len(errs) // 2][0] <= GRAD_TOL_MEDIAN and errs[-1][0] <= GRAD_TOL_MAX, errs[-3:]


# ------------------------------------------------------------------------------------------------ end to end
def test_exp_pretraining_from_f89_shards(tmp_path, monkeypatch):
    """pts/<name>_csr.pt shards with 89 node features: load_graphdataset takes F from the shard's x, and the three stages
    pre-train on it."""
    import exp_pretraining as ep
    from scgib_b200.graph import pack_shard
    monkeypatch.chdir(tmp_path)
    os.makedirs("pts")
    for i, name in enumerate(["PCQM4Mv2", "QM9", "mol-PCBA"]):
        g = _wide(synth_batch(500 + i, 64), 89, 500 + i)
        mols = []
        for j in range(g.num_graphs):
            n0, n1 = int(g.graph_ptr[j]), int(g.graph_ptr[j + 1])
            e0, e1 = int(g.indptr[n0]), int(g.indptr[n1])
            src = np.repeat(np.arange(n1 - n0), np.diff(g.indptr[n0:n1 + 1]))
            mols.append((np.stack([src, g.indices[e0:e1] - n0]), g.x[n0:n1], [0.0]))
        pack_shard(mols, "pts/%s_csr.pt" % name)
    ep.args = ep.build_parser().parse_args(["--device", DEV, "--pt_epoches", "1", "--batch_size", "32",
                                            "--output_path", str(tmp_path) + "/outputs/"])
    ep.device = torch.device(DEV)
    ep.main()
    names = sorted(os.listdir(tmp_path / "outputs"))
    assert names == ["pre_training_PCQM4Mv2_GIN_64_4_1.pt", "pre_training_PCQM4Mv2_QM9_GIN_64_4_1.pt",
                     "pre_training_PCQM4Mv2_QM9_mol-PCBA_GIN_64_4_1.pt"]
    last = torch.load(tmp_path / "outputs" / names[-1], weights_only=False)
    assert last.transfer_d.weight.shape == (32, 89)
    assert all(torch.isfinite(p).all() for p in last.parameters())
