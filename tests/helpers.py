"""Shared helpers for the GPU parity tests: build product-side batches/engines from oracle-side objects."""
import numpy as np
import torch

from oracle.graph_ref import RefEgoBatch, RefGraph, ego_batch_ref
from oracle.scgib_oracle import OracleMainmodel, normalize_rows, tgraph_from_ego, tgraph_from_ref


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def is_zero_grad_param(n):
    """Gradients that are mathematically zero (bias in front of a BatchNorm; softmax shift, SURVEY F14)."""
    return n.endswith("apply_func.mlp.2.bias") or n in ("attn_layer.bias", "compressor.0.bias")


def product_graph(g: RefGraph, device):
    from scgib_b200.graph import BatchedGraph
    return BatchedGraph(torch.from_numpy(g.graph_ptr), torch.from_numpy(g.indptr), torch.from_numpy(g.indices),
                        torch.from_numpy(g.x)).to(device)


def product_ego_from_ref(pg, e: RefEgoBatch, k, device):
    from scgib_b200.graph import EgoBatch
    seed = np.repeat(np.arange(len(e.ego_ptr) - 1, dtype=np.int32), np.diff(e.ego_ptr))
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a.astype(np.int32))).to(device)
    return EgoBatch(pg, k, t(e.ego_ptr), t(e.ego_nodes), t(seed), t(e.sub_indptr), t(e.sub_indices))


def hidden_of(m) -> int:
    return m.attn_layer.in_features // 2


def engine_from_oracle(m: OracleMainmodel, device, gin_layers=4, in_dim=9, dtype="fp32"):
    from scgib_b200.engine import PretrainEngine
    eng = PretrainEngine(in_dim, gin_layers=gin_layers, hidden=hidden_of(m), device=device, dtype=dtype)
    eng.load_state_dict({k: v.detach().float().to(device) for k, v in m.state_dict().items()}, strict=False)
    return eng


def oracle_grads(m, out):
    (out["KL"] + out["recon"] + out["contrastive"]).backward()
    return {n: p.grad.detach().clone() for n, p in m.named_parameters() if p.grad is not None}


def fp64_truth(m, g, e, gate_u, feat_u, recon_logm_steps=0):
    """fp64 vectorised oracle (forward + all parameter gradients) with the weights of ``m``: the ground truth
    both the fp32 reference run and the fp32 CUDA path are measured against."""
    m64 = OracleMainmodel(m.transfer_d.in_features, hidden_of(m), 32, len(m.Encoder1.ginlayers)).double()
    m64.load_state_dict({n: (v.double() if v.dtype.is_floating_point else v) for n, v in m.state_dict().items()})
    x = normalize_rows(torch.from_numpy(g.x).double())
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    if recon_logm_steps:      # --recons_type logM: only the faithful flavour restates it
        out = m64.forward_faithful(tgraph_from_ref(g), x, tgraph_from_ego(e), x[en], gate_u.double(), feat_u.double(),
                                   recon_logm_steps=recon_logm_steps)
    else:
        out = m64.forward_vectorised(tgraph_from_ref(g), x, tgraph_from_ego(e), en, gate_u.double(), feat_u.double())
    return out, oracle_grads(m64, out)


GRAD_TOL_MEDIAN, GRAD_TOL_MAX = 5e-5, 5e-3


def dump_parity(tag, report):
    """Measured errors of a parity case -> gpurun_out/parity_fp32/<tag>.json (kept in profiles/parity_r02.json)."""
    import json
    import os
    if any(os.environ.get(k) for k in ("SCGIB_FWD4", "SCGIB_HEAD_FFMA", "SCGIB_CON_FFMA", "SCGIB_TC", "SCGIB_TC_BWD")):
        return      # a cross-check run (tests/test_gpu_round2.py): keep the default build's numbers
    out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out", "parity_fp32")
    os.makedirs(out, exist_ok=True)
    fwd = {r[0]: dict(cuda_vs_fp64=r[1], fp32_torch_vs_fp64=r[2], bound=r[3]) for r in report if not r[0].startswith("grad ")}
    g = sorted(r[1] for r in report if r[0].startswith("grad "))
    gr = sorted(r[2] for r in report if r[0].startswith("grad "))
    worst = max((r for r in report if r[0].startswith("grad ")), key=lambda r: r[1])
    with open(os.path.join(out, tag + ".json"), "w") as fh:
        json.dump(dict(case=tag, forward=fwd, grad_median_cuda_vs_fp64=g[len(g) // 2], grad_max_cuda_vs_fp64=g[-1],
                       grad_worst=worst[0], grad_median_fp32_torch_vs_fp64=gr[len(gr) // 2], grad_max_fp32_torch_vs_fp64=gr[-1]), fh, indent=1)


def check_against_truth(eng, losses, emb, ref_out, ref_grads, truth_out, truth_grads, fwd_tol=1e-5, slack=5.0, tag=None):
    """The CUDA fp32 result is measured against the fp64 oracle ("truth"), next to the reference-precision (fp32
    torch) run of the same math.

    Forward (losses, embeddings): 1e-5 relative (BASELINE.json), or ``slack`` x the fp32 reference run's own distance
    from the truth where fp32 cannot do better.

    Gradients: fp32 gradients of this network are not a smooth function of rounding.  A hidden unit whose
    pre-activation lies within rounding distance of the ReLU kink takes different sides in two correct fp32
    implementations; its mask flips in the backward pass and every gradient downstream moves by O(1/rows) ~ 1e-3
    (verified on the torch oracle itself: perturbing the inputs by 1e-7 relative moves single gradients by 2e-4 in
    discrete jumps).  So: the MEDIAN over the parameter tensors of the max-norm relative error must be <= 5e-5
    (rounding-level agreement wherever no mask flipped) and every tensor must be within 5e-3 (flip allowance) or
    ``slack`` x the fp32 reference run's error."""
    report = []

    def one(name, got, ref, truth, tol):
        e_got, e_ref = rel(got, truth), rel(ref, truth)
        bound = max(tol, slack * e_ref)
        report.append((name, e_got, e_ref, bound))
        assert e_got <= bound, (name, "cuda-vs-fp64 %.3e" % e_got, "fp32ref-vs-fp64 %.3e" % e_ref, "bound %.3e" % bound)

    for i, name in enumerate(("KL", "contrastive", "recon")):
        one(name, losses[i].reshape(1), ref_out[name].reshape(1), truth_out[name].reshape(1), fwd_tol)
    for name in ("interaction_map", "Z", "noisy", "graph_readout"):
        one(name, emb[name], ref_out[name], truth_out[name], fwd_tol)
    gv = eng.grad_views()
    gmax = max(float(v.abs().max()) for v in truth_grads.values())
    for n, got in gv.items():
        truth = truth_grads[n].reshape(got.shape)
        ref = ref_grads[n].reshape(got.shape)
        if is_zero_grad_param(n):
            assert float(got.abs().max()) <= 1e-5 * gmax, n
            continue
        if n == "attn_layer.weight":
            H = got.shape[1] // 2
            assert float(got[:, :H].abs().max()) == 0.0          # core half: exactly zero (SURVEY F14)
            got, ref, truth = got[:, H:], ref[:, H:], truth[:, H:]
        one("grad " + n, got, ref, truth, GRAD_TOL_MAX)
    gerr = sorted(r[1] for r in report if r[0].startswith("grad "))
    rerr = sorted(r[2] for r in report if r[0].startswith("grad "))
    med, med_ref = gerr[len(gerr) // 2], rerr[len(rerr) // 2]
    if tag is not None:
        dump_parity(tag, report)
    # at full size (~3e7 ReLU units) mask flips are everywhere: the yardstick is the fp32 reference run's own median, with
    # the same ``slack`` as every other bound here.  (Measured, round 2: the B = 96, k = 2 case sits at 2.0e-5 with the FFMA
    # head forward and at 6.2e-5 with the tensor-core one - identical for its two operand splittings of different precision,
    # i.e. one flipped unit, not rounding - while the fp32 torch run of the same math is at 1.6e-5; profiles/parity_r02.json.)
    assert med <= max(GRAD_TOL_MEDIAN, slack * med_ref), ("median gradient error", med, "fp32 reference run", med_ref)
    return report
