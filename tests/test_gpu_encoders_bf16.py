"""bf16 mode of the --encoder GraphSAGE / GCN path (--dtype bf16, csrc/encoder_bf16.cu).

Operators: fp64 references computed from the SAME bf16-rounded operands; fp32 outputs within the fp32 op tests' bounds,
bf16 outputs within one bf16 ulp of the rounded fp64 value (plus the fp32-accumulation slack of a cancelling sum).
Models: Mainmodel in bf16 mode against (A) the fp64 oracle with the bf16 rounding points emulated (tests/bf16_emulation.py)
and (B) the plain fp64 oracle, with the bounds of tests/test_gpu_bf16.py; fine-tuning / domain adaptation against plain
fp64; bit-identical reruns."""
import copy
import os
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle.graph_ref import ego_batch_ref, synth_batch
from oracle.scgib_oracle import OracleMainmodel, normalize_rows, tgraph_from_ego, tgraph_from_ref
from tests.bf16_emulation import emulate
from tests.helpers import product_graph, rel

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _bf(t):
    """fp64 values of the bf16 rounding of t."""
    return t.to(torch.bfloat16).double()


def _within_ulp(got, ref, slack):
    """|got - rnd(ref)| <= one bf16 ulp of rnd(ref) + slack (absolute)."""
    got, r = got.double().cpu(), _bf(ref)
    ulp = torch.where(r == 0, torch.zeros_like(r), torch.exp2(torch.floor(torch.log2(r.abs().clamp(min=1e-38))) - 7))
    err = (got - r).abs() - ulp - slack
    return float(err.max()) <= 0, float(((got - r).abs() / ulp.clamp(min=1e-38)).max())


def _csr(g):
    ip = torch.from_numpy(g.indptr.astype(np.int64))
    ix = torch.from_numpy(g.indices.astype(np.int64))
    dst = torch.repeat_interleave(torch.arange(g.num_nodes), ip[1:] - ip[:-1])
    return ip, ix, dst


def _b(t):
    return t.to(torch.bfloat16).to(DEV).contiguous()


# ---------------------------------------------------------------------------------------------- operators
@pytest.mark.parametrize("W", [32, 64, 128, 256])
@pytest.mark.parametrize("norms", [(0, 0), (0, 1), (1, 0), (1, 1), (2, 2), (0, 2), (2, 0), (1, 2), (2, 1)])
@pytest.mark.parametrize("mapped", [False, True])
def test_graph_aggregate_bf16_op(W, norms, mapped):
    from scgib_b200 import ops
    g = synth_batch(81, 37)
    ip, ix, dst = _csr(g)
    V = g.num_nodes
    # a few isolated (zero-degree) rows at the end: degrees clamp to 1, the sum is empty
    ip = torch.cat([ip, ip[-1:].repeat(3)])
    V += 3
    dst = torch.repeat_interleave(torch.arange(V), ip[1:] - ip[:-1])
    torch.manual_seed(W + 7 * norms[0] + norms[1])
    rows = V + 11
    h = _bf(torch.randn(rows, W, dtype=torch.float64))
    row_map = torch.randint(0, rows, (V,)) if mapped else None
    add = _bf(torch.randn(V, W, dtype=torch.float64)) if mapped else None
    deg = (ip[1:] - ip[:-1]).double().clamp(min=1)
    f = lambda mode: torch.ones(V, dtype=torch.float64) if mode == 0 else (1.0 / deg if mode == 1 else deg.pow(-0.5))
    fs, fd = f(norms[0]), f(norms[1])
    src = h[row_map] if mapped else h[:V]
    ref = torch.zeros(V, W, dtype=torch.float64).index_add(0, dst, src[ix] * fs[ix][:, None]) * fd[:, None]
    mag = torch.zeros(V, W, dtype=torch.float64).index_add(0, dst, (src[ix] * fs[ix][:, None]).abs()) * fd[:, None]
    if mapped:
        ref, mag = ref + add, mag + add.abs()
    args = (_b(h) if mapped else _b(h[:V]), ip.int().to(DEV), ix.int().to(DEV), norms[0], norms[1])
    kw = dict(row_map=row_map.int().to(DEV), add=_b(add)) if mapped else {}
    got = ops.graph_aggregate(*args, **kw)
    assert got.dtype == torch.bfloat16
    ok, worst = _within_ulp(got, ref, 1e-6 * mag)
    assert ok, worst
    got32 = ops.graph_aggregate(*args, out_dtype=torch.float32, **kw)
    assert got32.dtype == torch.float32 and rel(got32, ref) <= 1e-5
    assert torch.equal(got32, ops.graph_aggregate(*args, out_dtype=torch.float32, **kw))
    assert torch.equal(got, got32.to(torch.bfloat16))          # one rounding of the same fp32 value


# (K0, K1, O) of the encoders: SAGE layers at hidden 64 / 128 (in 32), their backward products (O = 32), GCN at 2h = 256
_LIN = [(32, 32, 64), (64, 64, 64), (32, 32, 128), (128, 128, 128), (64, 0, 32), (128, 0, 32), (64, 0, 64), (128, 0, 128),
        (32, 0, 128), (128, 0, 128), (32, 0, 256), (256, 0, 256), (256, 0, 128), (128, 0, 256), (64, 0, 128)]


@pytest.mark.parametrize("K0,K1,O", _LIN)
@pytest.mark.parametrize("kxo", [False, True])
@pytest.mark.parametrize("V", [1, 127, 128, 129, 3001])
def test_linear_fwd_bf16_op(K0, K1, O, kxo, V):
    from scgib_b200 import ops
    torch.manual_seed(V + O + K0 + K1)
    rows = V + 5
    X0 = _bf(torch.randn(rows, K0, dtype=torch.float64))
    M0 = _bf(torch.randn(rows, K0, dtype=torch.float64))
    map0 = torch.randint(0, rows, (V,))
    W0 = torch.randn(O, K0, dtype=torch.float64) / K0 ** 0.5
    bias = torch.randn(O, dtype=torch.float64)
    ref = (X0 * (M0 > 0))[map0] @ _bf(W0).t() + bias
    mag = (X0 * (M0 > 0))[map0].abs() @ _bf(W0).abs().t() + bias.abs()
    f = lambda t: t.float().to(DEV).contiguous()
    kw = {}
    if K1:
        X1, M1 = _bf(torch.randn(V, K1, dtype=torch.float64)), _bf(torch.randn(V, K1, dtype=torch.float64))
        W1 = torch.randn(O, K1, dtype=torch.float64) / K1 ** 0.5
        ref = ref + (X1 * (M1 > 0)) @ _bf(W1).t()
        mag = mag + (X1 * (M1 > 0)).abs() @ _bf(W1).abs().t()
        kw = dict(X1=_b(X1), M1=_b(M1), W1=f(W1.t()) if kxo else f(W1), w1_kxo=kxo)
    args = (_b(X0), f(W0.t()) if kxo else f(W0), O)
    kw.update(w0_kxo=kxo, bias=f(bias), map0=map0.int().to(DEV), M0=_b(M0), V=V)
    y32 = ops.linear_fwd(*args, relu=False, out_dtype=torch.float32, **kw)
    assert y32.dtype == torch.float32 and float(((y32.double().cpu() - ref).abs() - 1e-5 * mag).max()) <= 0
    y = ops.linear_fwd(*args, relu=True, **kw)
    assert y.dtype == torch.bfloat16
    ok, worst = _within_ulp(y, torch.relu(ref), 2e-6 * mag)
    assert ok, worst
    assert torch.equal(y, torch.relu(y32).to(torch.bfloat16))
    assert torch.equal(y32, ops.linear_fwd(*args, relu=False, out_dtype=torch.float32, **kw))


def test_linear_fwd_bf16_pcqm_ego_batch():
    """one ego batch of PCQM size through the first SAGE layer: row_map gather, two operand pairs."""
    from scgib_b200 import ops
    torch.manual_seed(3)
    N, V, H = 60000, 600000, 64
    t = torch.randn(N, 32, device=DEV).to(torch.bfloat16)
    m0 = torch.randn(V, 32, device=DEV).to(torch.bfloat16)
    rm = torch.randint(0, N, (V,), device=DEV, dtype=torch.int32)
    Ws, Wn, b = torch.randn(H, 32, device=DEV) / 6, torch.randn(H, 32, device=DEV) / 6, torch.randn(H, device=DEV)
    y = ops.linear_fwd(t, Ws, H, X1=m0, W1=Wn, bias=b, relu=True, map0=rm, V=V, out_dtype=torch.float32)
    sel = torch.randint(0, V, (4096,), device=DEV)
    ref = torch.relu(t.double()[rm[sel].long()] @ Ws.to(torch.bfloat16).double().t() +
                     m0.double()[sel] @ Wn.to(torch.bfloat16).double().t() + b.double())
    assert rel(y[sel], ref) <= 1e-5


@pytest.mark.parametrize("V,O,K", [(1000, 64, 32), (5000, 64, 64), (40000, 128, 128), (300, 256, 32), (2000, 128, 256),
                                   (70000, 256, 256), (129, 128, 32), (1, 64, 64), (20000, 64, 128), (9000, 128, 64)])
@pytest.mark.parametrize("kxo", [False, True])
def test_linear_bwd_w_bf16_op(V, O, K, kxo):
    from scgib_b200 import ops
    torch.manual_seed(V + K)
    rows = V + 3
    G, M = _bf(torch.randn(V, O, dtype=torch.float64)), _bf(torch.randn(V, O, dtype=torch.float64))
    X = _bf(torch.randn(rows, K, dtype=torch.float64))
    mp = torch.randint(0, rows, (V,))
    Gm = G * (M > 0)
    dW_ref, db_ref = Gm.t() @ X[mp], Gm.sum(0)
    dW = torch.empty(K, O, device=DEV) if kxo else torch.empty(O, K, device=DEV)
    db = torch.empty(O, device=DEV)
    ops.linear_bwd_w(_b(G), _b(X), dW, db, M=_b(M), map=mp.int().to(DEV), kxo=kxo)
    first = dW.clone()
    assert rel(dW.t() if kxo else dW, dW_ref) <= 2e-5 and rel(db, db_ref) <= 2e-5
    ops.linear_bwd_w(_b(G), _b(X), dW, db, M=_b(M), map=mp.int().to(DEV), kxo=kxo, accumulate=True)
    assert rel(dW.t() if kxo else dW, 2 * dW_ref) <= 2e-5 and rel(db, 2 * db_ref) <= 2e-5
    again = torch.empty_like(first)
    ops.linear_bwd_w(_b(G), _b(X), again, None, M=_b(M), map=mp.int().to(DEV), kxo=kxo)
    assert torch.equal(first, again)
    # without the mask and the map
    ops.linear_bwd_w(_b(G), _b(X[:V]), again, None, kxo=kxo)
    assert rel(again.t() if kxo else again, G.t() @ X[:V]) <= 2e-5


def test_bf16_operators_refuse_mixed_dtypes():
    from scgib_b200 import ops
    X = torch.randn(10, 32, device=DEV).to(torch.bfloat16)
    with pytest.raises(TypeError):
        ops.linear_fwd(X, torch.randn(32, 32, device=DEV), 32, X1=torch.randn(10, 32, device=DEV), W1=torch.randn(32, 32, device=DEV))
    with pytest.raises(TypeError):
        ops.linear_bwd_w(torch.randn(10, 64, device=DEV).to(torch.bfloat16), torch.randn(10, 32, device=DEV),
                         torch.empty(64, 32, device=DEV))


# ---------------------------------------------------------------------------------------------- models
def _args(**kw):
    a = types.SimpleNamespace(recons_type="adj", useAtt=1, readout_f="sum", d_transfer=32, device=DEV, batch_size=128,
                              task="graph_classification", k_transition=1, dtype="bf16")
    a.__dict__.update(kw)
    return a


def _pretrain(encoder, hidden, k, recons, dtype, g, state, gate_u, feat_u, monkeypatch):
    import models
    from scgib_b200.graph import khop_ego_batch
    m = models.Mainmodel(_args(k_transition=k, recons_type=recons, dtype=dtype), 9, hidden_dim=hidden, num_layers=4, num_heads=4,
                         k_transition=k, encoder=encoder)
    m.load_state_dict(state, strict=False)
    m = m.to(DEV)
    pg = product_graph(g, DEV)
    ego = khop_ego_batch(pg, k)
    x = F.normalize(pg.ndata["x"].float())
    monkeypatch.setattr(m, "_noise", lambda N, dev: (gate_u.to(dev), feat_u.to(dev)))
    m.train()
    _, kl, con, rec = m.forward(pg, x, ego, None, None, 1, None, 2, DEV, max(16, g.num_graphs))
    (kl + rec + con).backward()
    torch.cuda.synchronize()
    return m, kl, con, rec


@pytest.mark.parametrize("encoder", ["GraphSAGE", "GCN"])
@pytest.mark.parametrize("hidden", [64, 128])
@pytest.mark.parametrize("k,recons", [(1, "adj"), (2, "adj"), (2, "logM")])
def test_mainmodel_bf16_against_fp64_oracle(encoder, hidden, k, recons, monkeypatch):
    g = synth_batch(91 + hidden + k, 200)
    e = ego_batch_ref(g, k)
    torch.manual_seed(7)
    ref = OracleMainmodel(9, hidden, 32, 4, encoder=encoder).double()
    gate_u, feat_u = torch.rand(g.num_nodes), torch.rand(g.num_nodes, hidden)
    state = {n: t.float() for n, t in ref.state_dict().items()}
    m, kl, con, rec = _pretrain(encoder, hidden, k, recons, "bf16", g, state, gate_u, feat_u, monkeypatch)
    m32, *_ = _pretrain(encoder, hidden, k, recons, "fp32", g, state, gate_u, feat_u, monkeypatch)
    xr = normalize_rows(torch.from_numpy(g.x)).double()
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    emu = copy.deepcopy(ref)
    emulate(emu.Encoder1)
    emulate(emu.Encoder2)

    def run(model):
        if recons == "logM":
            o = model.forward_faithful(tgraph_from_ref(g), xr, tgraph_from_ego(e), xr[en], gate_u.double(), feat_u.double(),
                                       recon_logm_steps=k)
        else:
            o = model.forward_vectorised(tgraph_from_ref(g), xr, tgraph_from_ego(e), en, gate_u.double(), feat_u.double())
        (o["KL"] + o["recon"] + o["contrastive"]).backward()
        return o, {n: p.grad for n, p in model.named_parameters() if p.grad is not None}
    out, refg = run(ref)
    oute, emug = run(emu)
    last = m._composed_last
    got = {n: p.grad for n, p in m.named_parameters() if p.grad is not None}
    got32 = {n: p.grad for n, p in m32.named_parameters() if p.grad is not None}
    gmax = max(float(v.abs().max()) for v in refg.values())
    keep = [n for n, v in refg.items() if float(v.abs().max()) > 1e-6 * gmax]
    med = lambda errs: sorted(errs)[len(errs) // 2]
    # (A) against the fp64 oracle with the bf16 rounding points emulated
    for name, got_l in (("KL", kl), ("contrastive", con), ("recon", rec)):
        assert abs(float(got_l) - float(oute[name])) <= 2e-2 * abs(float(oute[name])), (name, float(got_l), float(oute[name]))
    embs = [n for n in ("Z", "noisy", "graph_readout") if n in out]
    for name in embs:
        assert rel(last[name], oute[name]) <= 2e-2, (name, rel(last[name], oute[name]))
    assert med([rel(got[n].cpu(), emug[n]) for n in keep]) <= 4e-2
    # (B) against plain fp64: losses 2e-2; embeddings and gradients within 3x the emulated algorithm's own deviation
    for name, got_l in (("KL", kl), ("contrastive", con), ("recon", rec)):
        assert abs(float(got_l) - float(out[name])) <= 2e-2 * abs(float(out[name])), (name, float(got_l), float(out[name]))
    for name in embs:
        assert rel(last[name], out[name]) <= 3 * rel(oute[name].detach(), out[name]) + 1e-3, name
    assert med([rel(got[n].cpu(), refg[n]) for n in keep]) <= 3 * med([rel(emug[n], refg[n]) for n in keep]) + 1e-3
    assert med([rel(got32[n].cpu(), refg[n]) for n in keep]) <= 5e-5    # the same module in fp32 mode: unchanged path
    # the encoders ran in bf16: their saved activations are bf16, the output fp32
    assert last["Z"].dtype == torch.float32


@pytest.mark.parametrize("encoder", ["GraphSAGE", "GCN"])
def test_bf16_composed_step_is_bit_identical_on_rerun(encoder, monkeypatch):
    g = synth_batch(17, 150)
    torch.manual_seed(11)
    ref = OracleMainmodel(9, 64, 32, 4, encoder=encoder)
    state = {n: t.float() for n, t in ref.state_dict().items()}
    gate_u, feat_u = torch.rand(g.num_nodes), torch.rand(g.num_nodes, 64)
    runs = []
    for _ in range(2):
        m, kl, con, rec = _pretrain(encoder, 64, 1, "adj", "bf16", g, state, gate_u, feat_u, monkeypatch)
        runs.append(([float(kl), float(con), float(rec)], {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None},
                     {n: b.clone() for n, b in m.named_buffers()}))
    assert runs[0][0] == runs[1][0]
    assert runs[0][1].keys() == runs[1][1].keys() and all(torch.equal(runs[0][1][n], runs[1][1][n]) for n in runs[0][1])
    assert all(torch.equal(runs[0][2][n], runs[1][2][n]) for n in runs[0][2])


def test_encoder_activations_are_bf16_inside():
    """run_forward on a bf16 t keeps m0..h2 / a0..a2 in bf16 and returns an fp32 h3; the input gradient is fp32."""
    from scgib_b200 import encoders, ops
    g = synth_batch(5, 40)
    pg = product_graph(g, DEV)
    for enc in (encoders.GraphSAGE(32, 64), encoders.GCN(32, 64)):
        enc = enc.to(DEV)
        t = torch.randn(g.num_nodes, 32, device=DEV)
        h3, saved = enc.run_forward(ops.to_bf16(t), pg.indptr, pg.indices)
        assert h3.dtype == torch.float32
        acts = [s for s in saved if torch.is_tensor(s) and s.dim() == 2]
        assert acts and all(a.dtype == torch.bfloat16 for a in acts)
        g_t, grads = enc.run_backward(saved, torch.randn_like(h3))
        assert g_t.dtype == torch.float32 and g_t.shape == (g.num_nodes, 32)
        assert all(v.dtype == torch.float32 and torch.isfinite(v).all() for v in grads.values())
        h3_32, _ = enc.run_forward(t, pg.indptr, pg.indices)
        assert rel(h3, h3_32) <= 3e-2


def test_extract_features_eval_bf16():
    import models
    from scgib_b200.graph import khop_ego_batch
    g = synth_batch(52, 16)
    torch.manual_seed(52)
    feats = {}
    for dt in ("fp32", "bf16"):
        torch.manual_seed(52)
        m = models.Mainmodel(_args(dtype=dt), 9, 64, 4, 4, 1, "GCN").to(DEV).eval()
        pg = product_graph(g, DEV)
        ego = khop_ego_batch(pg, 1)
        t = m.transfer_d(F.normalize(pg.ndata["x"].float())).detach()
        m._noise = lambda N, dev: (torch.full((N,), 0.5, device=dev), torch.full((N, 64), 0.5, device=dev))
        imap, kl_t, noisy, readout = m.extract_features(pg.batch_num_nodes(), pg, t, ego, None, DEV)
        feats[dt] = (imap, readout)
    assert rel(feats["bf16"][0], feats["fp32"][0]) <= 2e-2 and rel(feats["bf16"][1], feats["fp32"][1]) <= 2e-2


def test_exp_pretraining_cli_gcn_bf16(tmp_path, monkeypatch):
    import exp_pretraining as ep
    monkeypatch.chdir(tmp_path)
    ep.args = ep.build_parser().parse_args(["--device", DEV, "--pt_epoches", "2", "--batch_size", "32", "--synthetic", "96",
                                            "--encoder", "GCN", "--dtype", "bf16", "--output_path", str(tmp_path) + "/outputs/"])
    ep.device = torch.device(DEV)
    ep.main()
    names = sorted(os.listdir(tmp_path / "outputs"))
    assert len(names) == 3
    last = torch.load(tmp_path / "outputs" / names[-1], weights_only=False)
    assert last.act_dtype == "bf16" and type(last.model.Encoder1).__name__ == "GCN"
    assert all(torch.isfinite(p).all() for p in last.parameters())


def _median_grad_err(got, refg):
    gmax = max(float(v.abs().max()) for v in refg.values())
    errs = sorted(rel(got[n].cpu(), g) for n, g in refg.items() if float(g.abs().max()) > 1e-6 * gmax)
    return errs[len(errs) // 2]


@pytest.mark.parametrize("encoder,hidden,k", [("GraphSAGE", 64, 1), ("GCN", 128, 2)])
def test_finetuning_bf16_against_fp64_oracle(encoder, hidden, k, tmp_path, monkeypatch):
    import models
    from oracle.scgib_oracle import OracleFinetune
    from scgib_b200.graph import khop_ego_batch
    from tests.test_gpu_encoders_downstream import _checkpoint, _oracle_wrapper
    B, C = 40, 10
    g = synth_batch(600 + hidden + k, B)
    e = ego_batch_ref(g, k)
    torch.manual_seed(17 + k)
    ref = _oracle_wrapper(OracleFinetune, encoder, hidden, num_classes=C, task="graph_classification", regression_dataset=False)
    args = _args(k_transition=k, task="graph_classification", dataset="Peptides-func")
    m = models.Mainmodel_finetuning(args, 9, hidden, 4, 4, k, C, _checkpoint(tmp_path, encoder, hidden, k), encoder)
    m.load_state_dict(ref.state_dict(), strict=False)
    m = m.to(DEV).train()
    ref = ref.double().train()
    pg = product_graph(g, DEV)
    gate_u, feat_u = torch.rand(g.num_nodes), torch.rand(g.num_nodes, hidden)
    monkeypatch.setattr(m, "_noise", lambda N, dev: (gate_u.to(dev), feat_u.to(dev)))
    scores, _, _, _ = m.forward(pg, F.normalize(pg.ndata["x"].float()), khop_ego_batch(pg, k), None, 1, None, 2, DEV, B)
    xr = normalize_rows(torch.from_numpy(g.x)).double()
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    out = ref(tgraph_from_ref(g), xr, tgraph_from_ego(e), xr[en], gate_u.double(), feat_u.double())
    assert rel(scores.detach().cpu(), out["scores"].detach()) <= 2e-2
    targets = (torch.rand(B, C) < 0.3).float()
    loss = m.loss(scores, targets.to(DEV))
    rloss = F.binary_cross_entropy(out["scores"], targets.double())
    assert abs(float(loss) - float(rloss)) <= 2e-2 * abs(float(rloss))
    loss.backward()
    rloss.backward()
    refg = {n: p.grad for n, p in ref.named_parameters() if p.grad is not None}
    got = {n: p.grad for n, p in m.named_parameters() if p.grad is not None}
    assert _median_grad_err(got, refg) <= 4e-2


@pytest.mark.parametrize("encoder,hidden,k", [("GCN", 64, 1), ("GraphSAGE", 128, 1)])
def test_domainadapt_bf16_against_fp64_oracle(encoder, hidden, k, tmp_path, monkeypatch):
    import models
    from oracle.scgib_oracle import OracleDomainAdapt
    from scgib_b200.graph import khop_ego_batch
    from tests.test_gpu_encoders_downstream import _checkpoint, _oracle_wrapper
    B = 32
    g = synth_batch(700 + hidden + k, B)
    e = ego_batch_ref(g, k)
    torch.manual_seed(19 + k)
    ref = _oracle_wrapper(OracleDomainAdapt, encoder, hidden, num_classes=10)
    m = models.Mainmodel_domainadapt(_args(k_transition=k), 9, hidden, 4, 4, k, 10, _checkpoint(tmp_path, encoder, hidden, k), encoder)
    m.load_state_dict(ref.state_dict(), strict=False)
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
    assert abs(float(loss) - float(out["X_loss"])) <= 2e-2 * abs(float(out["X_loss"]))
    refg = {n: p.grad for n, p in ref.named_parameters() if p.grad is not None}
    got = {n: p.grad for n, p in m.named_parameters() if p.grad is not None}
    assert _median_grad_err(got, refg) <= 4e-2
