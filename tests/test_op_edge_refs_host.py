"""The vectorised fp64 restatements of tests/test_gpu_op_edges.py against the oracle's own per-graph functions, on small
batches (no GPU needed): a wrong reference would otherwise pass or fail the CUDA kernels for the wrong reason."""
import numpy as np
import torch
import torch.nn.functional as F

from oracle.graph_ref import batch_ref, graph_from_bonds, synth_batch
from oracle.scgib_oracle import OracleMainmodel, loss_recon_logm, sum_nodes, tgraph_from_ref
from tests.helpers import rel
from tests.test_gpu_op_edges import _exact_logits, attn_ref, ball_sizes, bn_ema_ref, gate_ref, logm_ref, ring, seg_of, star


def _sizes_graph(sizes):
    return batch_ref([graph_from_bonds(n, [(i, i + 1) for i in range(n - 1)]) for n in sizes])


def test_gate_ref_matches_oracle_compression():
    sizes = [5, 2, 17, 150, 2, 9]
    N, H = sum(sizes), 64
    torch.manual_seed(0)
    m = OracleMainmodel(9, H).double()
    c = m.compressor
    rm0, rv0 = torch.randn(H, dtype=torch.float64) * 0.1, 1 + torch.rand(H, dtype=torch.float64)
    c[1].running_mean.copy_(rm0); c[1].running_var.copy_(rv0)
    Hf = torch.randn(N, H, dtype=torch.float64).requires_grad_()
    gate_u, feat_u = torch.rand(N, dtype=torch.float64), torch.rand(N, H, dtype=torch.float64)
    noisy, _, KL_tensor = m.compression(Hf, sizes, gate_u, feat_u)        # nn.BatchNorm1d train calls, one per graph
    tg = tgraph_from_ref(_sizes_graph(sizes))
    readout, core = sum_nodes(tg, Hf), sum_nodes(tg, noisy)
    gn, gc, gr = torch.randn_like(noisy), torch.randn_like(core), torch.randn_like(readout)
    ((noisy * gn).sum() + (core * gc).sum() + (readout * gr).sum() + 0.7 * KL_tensor.mean()).backward()
    want = [Hf.grad.clone()] + [p.grad.clone() for p in (c[0].weight, c[1].weight, c[1].bias, c[3].weight, c[3].bias)]

    P = [t.detach().clone().requires_grad_(True) for t in (c[0].weight, c[0].bias, c[1].weight, c[1].bias, c[3].weight, c[3].bias)]
    H2 = Hf.detach().clone().requires_grad_()
    n2, r2, c2, kl2, qm, qv = gate_ref(H2, sizes, *P, gate_u, feat_u)
    for got, ref in ((n2, noisy), (r2, readout), (c2, core), (kl2, KL_tensor.mean())):
        assert rel(got, ref) <= 1e-12
    ((n2 * gn).sum() + (c2 * gc).sum() + (r2 * gr).sum() + 0.7 * kl2).backward()
    for got, ref in zip([H2.grad] + [P[i].grad for i in (0, 2, 3, 4, 5)], want):
        assert rel(got, ref) <= 1e-10
    em, ev = bn_ema_ref(qm, qv, rm0, rv0)
    assert rel(em, c[1].running_mean) <= 1e-12 and rel(ev, c[1].running_var) <= 1e-12

    # model.eval(): compressor.1 normalises with its running statistics
    m.eval()
    with torch.no_grad():
        noisy_e, _, KL_e = m.compression(Hf, sizes, gate_u, feat_u)
        n3, _, _, kl3, _, _ = gate_ref(H2, sizes, *P, gate_u, feat_u, running=(c[1].running_mean, c[1].running_var))
    assert rel(n3, noisy_e) <= 1e-12 and rel(kl3, KL_e.mean()) <= 1e-12


def test_attn_ref_matches_per_graph_softmax():
    sizes = [3, 1, 40, 7]
    torch.manual_seed(1)
    for C, w in ((torch.randn(sum(sizes), 64, dtype=torch.float64), torch.randn(64, dtype=torch.float64)),
                 _exact_logits(sizes, 64, torch.tensor([80.0, -80.0, 80.0, -80.0], dtype=torch.float64))):
        seg = seg_of(sizes)
        logit = C @ w
        alpha = torch.cat([F.softmax(logit[seg == b], 0) for b in range(len(sizes))])
        a, T = attn_ref(C, sizes, w)
        assert rel(a, alpha) <= 1e-13 and rel(T, C * alpha[:, None]) <= 1e-13


def test_logm_ref_matches_oracle_and_drops_overflowing_seeds():
    for g, k in ((synth_batch(3, 6), 4), (synth_batch(4, 2, "peptides"), 3), (batch_ref([star(127), ring(40)]), 1)):
        torch.manual_seed(k)
        Z = (torch.randn(g.num_nodes, 64, dtype=torch.float64) * 0.15).requires_grad_(True)
        ref = loss_recon_logm(Z, tgraph_from_ref(g), k)
        ref.backward()
        loss, gZ = logm_ref(Z.detach(), g, k)
        assert abs(float(loss) - float(ref.detach())) <= 1e-6 * abs(float(ref.detach())) and rel(gZ, Z.grad) <= 1e-6   # the oracle's logM are fp32
    # dropping: a capacity below the star's centre ball removes exactly the centre's seed terms
    g = batch_ref([star(6), graph_from_bonds(2, [(0, 1)])])
    assert list(ball_sizes(g, 1)) == [7, 2, 2, 2, 2, 2, 2, 2, 2]
    torch.manual_seed(5)
    Z = torch.randn(g.num_nodes, 64, dtype=torch.float64)
    full, g_full = logm_ref(Z, g, 1, cap=128)
    part, g_part = logm_ref(Z, g, 1, cap=6)
    n = 7
    A = np.zeros((n, n)); A[0, 1:] = A[1:, 0] = 1
    L = np.log(np.maximum(A / A.sum(0) * n, 1e-300)).clip(min=0) * (A > 0)                      # logM_1 of the star
    Lc, z = torch.from_numpy(L), Z[:n]
    centre_terms = (-2 * (z[0] @ z.t()) * Lc[0] + Lc[0] ** 2).sum() / n ** 2
    assert abs(float(full - part - centre_terms)) <= 1e-12 * abs(float(full))
    expect = g_full.clone()
    expect[0] += 2 / n ** 2 * (Lc + Lc.t())[0] @ z
    assert rel(g_part, expect) <= 1e-12
