"""Driver-visible GPU tests for claims that round 1 only covered with scripts (VERDICT r01 item 5):
the fused peer all-reduce + Adam kernel, the L = 5 (paper / shipped-checkpoint) variant incl. the reference's shipped
weights, odd / extreme batch sizes, a short training run, and the one-forward-one-backward guard of the drop-in modules."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle.graph_ref import ego_batch_ref, synth_batch
from oracle.scgib_oracle import (OracleMainmodel, draw_noise_like_reference, normalize_rows, tgraph_from_ego,
                                 tgraph_from_ref)
from tests.helpers import check_against_truth, engine_from_oracle, fp64_truth, oracle_grads, product_graph, rel

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---------------------------------------------------------------- fused all-reduce + Adam (csrc/peer_kernels.cu)
def test_allreduce_adam_world1_matches_adam_kernel():
    """world = 1: the fused kernel degenerates to Adam on the rank's own gradient buffer (replaces loss.backward()'s
    exchange + optimizer.step(), exp_pretraining.py:321-323): must equal scgib_adam_step_f32 bit for bit, and both must
    follow torch.optim.Adam(lr, weight_decay) to fp32 rounding."""
    import ctypes
    from scgib_b200 import _lib
    lib = _lib.load()
    n = 80680
    gen = torch.Generator(device=DEV).manual_seed(0)
    p0 = torch.randn(n, device=DEV, generator=gen)
    pa, ma, va = p0.clone(), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    pb, mb, vb = p0.clone(), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    pt = torch.nn.Parameter(p0.clone())
    opt = torch.optim.Adam([pt], lr=1e-3, weight_decay=5e-5)
    gbuf = [torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)]
    flags = torch.zeros(64, dtype=torch.int32, device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    for step in range(1, 6):
        g = torch.randn(n, device=DEV, generator=gen)
        gbuf[step & 1].copy_(g)
        grads = (ctypes.c_void_p * 1)(gbuf[step & 1].data_ptr())
        fl = (ctypes.c_void_p * 1)(flags.data_ptr())
        _lib.check(lib.scgib_allreduce_adam_f32(_lib.ptr(pa), _lib.ptr(ma), _lib.ptr(va), n, grads, fl, 0, 1, step, step,
                                                1e-3, 0.9, 0.999, 1e-8, 5e-5, st), "allreduce_adam")
        _lib.check(lib.scgib_adam_step_f32(_lib.ptr(pb), _lib.ptr(g), _lib.ptr(mb), _lib.ptr(vb), n, step, 1e-3, 0.9, 0.999,
                                           1e-8, 5e-5, 1.0, st), "adam")
        pt.grad = g.clone()
        opt.step()
    torch.cuda.synchronize()
    assert torch.equal(pa, pb) and torch.equal(ma, mb) and torch.equal(va, vb)
    assert rel(pa, pt.detach()) <= 2e-6


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs on one node")
def test_allreduce_adam_two_ranks():
    """2-process run over NVLink peer memory: fused kernel == NCCL all-reduce + Adam kernel, replicas bit-identical."""
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29541", os.path.join(ROOT, "tests", "gpu_peer_allreduce.py")],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "replicas bit-identical: True" in r.stdout


# ---------------------------------------------------------------- L = 5 (SURVEY F4) and the shipped checkpoint
def _run(m, g, e, k, gate_u, feat_u, L):
    from scgib_b200.engine import DeviceBatch
    from scgib_b200.graph import khop_ego_batch
    eng = engine_from_oracle(m, DEV, gin_layers=L)
    pg = product_graph(g, DEV)
    b = DeviceBatch(pg, khop_ego_batch(pg, k), pg.ndata["x"], normalize_x=True)
    losses, emb = eng.forward(b, gate_u.to(DEV), feat_u.to(DEV), want=True)
    eng.backward()
    torch.cuda.synchronize()
    return eng, b, losses.cpu(), emb


@pytest.mark.parametrize("L", [5, 2])
def test_parity_other_layer_counts(L):
    """gin_layers = 5 is the paper / shipped-checkpoint variant (`num_layers - 1` = 4 in the published code)."""
    g = synth_batch(31, 100)
    e = ego_batch_ref(g, 1)
    torch.manual_seed(31)
    m = OracleMainmodel(9, 64, 32, L)
    x = normalize_rows(torch.from_numpy(g.x))
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    gate_u, feat_u = draw_noise_like_reference(g.batch_num_nodes().tolist(), 64, 131)
    out = m.forward_faithful(tgraph_from_ref(g), x, tgraph_from_ego(e), x[en], gate_u, feat_u)
    ref_grads = oracle_grads(m, out)
    m.zero_grad()
    eng, _, losses, emb = _run(m, g, e, 1, gate_u, feat_u, L)
    m64 = OracleMainmodel(9, 64, 32, L).double()
    m64.load_state_dict({n: (v.double() if v.dtype.is_floating_point else v) for n, v in m.state_dict().items()})
    o64 = m64.forward_vectorised(tgraph_from_ref(g), x.double(), tgraph_from_ego(e), en, gate_u.double(), feat_u.double())
    check_against_truth(eng, losses, emb, out, ref_grads, o64, oracle_grads(m64, o64))


def test_shipped_checkpoint_weights_l5():
    """The reference's shipped weights (outputs/pre_training_v1_GIN_64_5_1.pt, 5 GINConv per encoder; fixture made by
    tests/golden/make_ckpt_fixture.py) through PretrainEngine(gin_layers=5): finite, oracle-matching forward and
    gradients in training mode, and the eval-mode forward (running statistics of the checkpoint)."""
    fx = torch.load(os.path.join(ROOT, "tests", "golden", "shipped_ckpt_v1_GIN_64_5_1.pt"))
    assert fx["meta"]["gin_layers"] == 5
    m = OracleMainmodel(9, 64, 32, 5)
    missing, unexpected = m.load_state_dict(fx["state"], strict=False)
    used = [n for n, _ in m.named_parameters() if n.startswith(("transfer_d", "MLP.", "Encoder", "compressor", "attn_layer"))]
    assert not [n for n in used if n in missing], missing
    g = synth_batch(41, 64)
    e = ego_batch_ref(g, 1)
    x = normalize_rows(torch.from_numpy(g.x))
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    gate_u, feat_u = draw_noise_like_reference(g.batch_num_nodes().tolist(), 64, 141)
    out = m.forward_faithful(tgraph_from_ref(g), x, tgraph_from_ego(e), x[en], gate_u, feat_u)
    ref_grads = oracle_grads(m, out)
    m.zero_grad()
    m.load_state_dict(fx["state"], strict=False)          # the training-mode forward moved the running statistics
    eng, b, losses, emb = _run(m, g, e, 1, gate_u, feat_u, 5)
    assert torch.isfinite(losses).all() and torch.isfinite(eng.grads).all()
    truth_out, truth_grads = fp64_truth(m, g, e, gate_u, feat_u)
    check_against_truth(eng, losses, emb, out, ref_grads, truth_out, truth_grads)
    # eval mode: every BatchNorm normalises with the checkpoint's running statistics
    m.load_state_dict(fx["state"], strict=False)
    m.eval()
    with torch.no_grad():
        oe = m.forward_faithful(tgraph_from_ref(g), x, tgraph_from_ego(e), x[en], gate_u, feat_u)
    eng2 = engine_from_oracle(m, DEV, gin_layers=5)
    b.eval_mode = True
    _, emb2 = eng2.forward(b, gate_u.to(DEV), feat_u.to(DEV), want=True)
    torch.cuda.synchronize()
    for name in ("interaction_map", "Z", "noisy", "graph_readout"):
        assert rel(emb2[name], oe[name]) <= 2e-5, (name, rel(emb2[name], oe[name]))


# ---------------------------------------------------------------- robustness (was tests/gpu_size_sweep.py)
@pytest.mark.parametrize("B,k,shape", [(1, 1, "pcqm"), (2, 1, "pcqm"), (3, 2, "pcqm"), (100, 1, "pcqm"), (1000, 3, "pcqm"),
                                       (4097, 1, "pcqm"), (16384, 1, "pcqm"), (7, 1, "peptides"), (300, 2, "peptides"),
                                       (129, 4, "pcqm")])
def test_size_sweep_finite_and_deterministic(B, k, shape):
    from scgib_b200.engine import PretrainEngine
    from scgib_b200.synth import synth_batch as psynth
    eng = PretrainEngine(9, gin_layers=4, device=DEV, seed=1)
    b = eng.make_batch(psynth(B, B, shape).to(DEV), k)
    gen = torch.Generator(device=DEV).manual_seed(3)
    gu, fu = torch.rand(b.N, device=DEV, generator=gen), torch.rand(b.N, 64, device=DEV, generator=gen)
    res = []
    for _ in range(2):
        losses = eng.forward(b, gu, fu).clone()
        res.append((losses, eng.backward().clone()))
    torch.cuda.synchronize()
    assert torch.isfinite(res[0][0]).all() and torch.isfinite(res[0][1]).all()
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])
    del eng
    torch.cuda.empty_cache()


def test_training_run_loss_goes_down():
    """300 steps at B = 2048 on a resident dataset of 16k synthetic molecules, lr 1e-3 (was tests/gpu_train_sanity.py)."""
    from scgib_b200.engine import PretrainEngine
    from scgib_b200.graph import DeviceDataset, batch
    from scgib_b200.synth import synth_batch as psynth
    eng = PretrainEngine(9, gin_layers=4, device=DEV, seed=0)
    ds = DeviceDataset.from_batched(batch([psynth(i, 4096) for i in range(4)]), DEV)
    gen = torch.Generator().manual_seed(0)
    ids = lambda: torch.randperm(len(ds), generator=gen)[:2048].to(torch.int32).pin_memory()
    hist = []
    handle = eng.prefetch_ids(ds, ids(), 1)
    for step in range(300):
        b = eng.wait_batch(handle)
        losses = eng.train_step(b, lr=1e-3)
        handle = eng.prefetch_ids(ds, ids(), 1)
        if step % 50 == 0 or step == 299:
            hist.append(losses.cpu().tolist())
            assert all(v == v and abs(v) < 1e12 for v in hist[-1]), hist[-1]
    assert hist[-1][3] < 0.7 * hist[0][3], hist
    assert torch.isfinite(eng.params).all()


# ---------------------------------------------------------------- API guards (ADVICE r01)
def test_backward_after_second_forward_raises():
    """The engine keeps ONE workspace of saved activations: a backward that belongs to an older forward must raise
    instead of silently using the newer batch's activations."""
    import types
    from scgib_b200 import models
    from scgib_b200.graph import khop_ego_batch
    from scgib_b200.synth import synth_batch as psynth
    args = types.SimpleNamespace(recons_type="adj", useAtt=1, readout_f="sum", d_transfer=32, device=DEV)
    torch.manual_seed(0)
    model = models.Mainmodel(args, 9, hidden_dim=64, num_layers=4, num_heads=4, k_transition=1, encoder="GIN").to(DEV)
    outs = []
    for seed in (1, 2):
        g = psynth(seed, 16).to(DEV)
        ego = khop_ego_batch(g, 1)
        x = torch.nn.functional.normalize(g.ndata["x"].float())
        _, kl, con, rec = model.forward(g, x, ego, None, None, 1, None, 1, DEV, batch_size=16)
        outs.append(kl + con + rec)
    with pytest.raises(RuntimeError, match="another forward"):
        outs[0].backward()
    outs[1].backward()          # the latest forward's backward is fine
    assert all(p.grad is None or torch.isfinite(p.grad).all() for p in model.parameters())


def test_device_loader_reshuffles_every_pass():
    from scgib_b200.graph import DeviceDataset, DeviceLoader, batch
    from scgib_b200.synth import synth_batch as psynth
    ds = DeviceDataset.from_batched(batch([psynth(0, 64)]), DEV)
    loader = DeviceLoader(ds, 16, shuffle=True)
    first = torch.cat([ids for ids in loader.id_batches()]).cpu()
    second = torch.cat([ids for ids in loader.id_batches()]).cpu()
    assert not torch.equal(first, second) and torch.equal(first.sort()[0], second.sort()[0])
    loader.set_epoch(0)
    assert torch.equal(torch.cat([ids for ids in loader.id_batches()]).cpu(), first)      # the DP override still pins the order


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"SCGIB_HEAD_FFMA": "1", "SCGIB_CON_FFMA": "1"}], ids=["ffma_head_contrastive"])
def test_implementation_switches_stay_parity_green(env):
    """The cross-check kernels behind the environment switches (INTEGRATION.md) pass the same parity tests as the
    defaults: the FFMA head / contrastive kernels with the un-fused forward tail.  The switches are read once per
    process, hence the subprocess."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_parity.py", "-q", "-x", "-k",
                        "gin_layer or golden_reference_parity or faithful_oracle or loss_operators"],
                       cwd=root, env={**os.environ, **env}, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
