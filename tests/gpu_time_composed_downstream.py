"""Time the GraphSAGE / GCN fine-tuning and domain-adaptation steps and the logM loss operator (measurement, no target):

    python -m tests.gpu_time_composed_downstream

One JSON line per case.  A step is forward + loss + backward + torch Adam on a batch already resident in HBM (its k-hop
ego-nets built once, outside the timed region), timed with CUDA events after warm-up steps.  The GPU name and power limit
are read in the same run."""
import json
import os
import subprocess
import tempfile
import types

import torch
import torch.nn.functional as F

DEV = torch.device("cuda:0")


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    name, _, power = q.partition(",")
    return {"gpu": name.strip() or torch.cuda.get_device_name(DEV), "power_limit": power.strip() or None}


def timed(fn, warmup, iters):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters          # ms per call


def _args(**kw):
    a = types.SimpleNamespace(recons_type="adj", useAtt=1, readout_f="sum", d_transfer=32, device=str(DEV), batch_size=4096,
                              task="graph_classification", dataset="Peptides-func", k_transition=1)
    a.__dict__.update(kw)
    return a


def step_case(kind, encoder, shape, B, hidden, tmp, info):
    import models
    from scgib_b200.graph import khop_ego_batch
    from scgib_b200.synth import synth_batch
    torch.manual_seed(0)
    pre = models.Mainmodel(_args(), 9, hidden, 4, 4, 1, encoder)
    ckpt = os.path.join(tmp, "%s_%d.pt" % (encoder, hidden))
    torch.save(pre, ckpt)
    cls = models.Mainmodel_finetuning if kind == "finetune" else models.Mainmodel_domainadapt
    m = cls(_args(), 9, hidden, 4, 4, 1, 10, ckpt, encoder).to(DEV).train()
    opt = torch.optim.Adam([p for p in m.parameters() if p.requires_grad], lr=1e-4)
    g = synth_batch(1, B, shape).to(DEV)
    ego = khop_ego_batch(g, 1)
    x = F.normalize(g.ndata["x"].float())
    targets = (torch.rand(B, 10, device=DEV) < 0.1).float()

    def step():
        opt.zero_grad()
        if kind == "finetune":
            scores, _, _, _ = m.forward(g, x, ego, None, 1, None, 2, DEV, B)
            loss = m.loss(scores, targets)
        else:
            loss = m.forward(g, x, ego, None, None, 1, None, 2, DEV, B)
        loss.backward()
        opt.step()

    ms = timed(step, 3, 20)
    print(json.dumps(dict(case="%s_step" % kind, encoder=encoder, shape=shape, batch=B, hidden=hidden, ms_per_step=round(ms, 3),
                          graphs_per_s=round(B / ms * 1e3), **info)), flush=True)


def logm_cases(info):
    from scgib_b200 import ops
    from scgib_b200.synth import synth_batch
    B = 4096
    g = synth_batch(2, B, "pcqm").to(DEV)
    for H in (64, 128):
        Z = torch.randn(g.num_nodes(), H, device=DEV) * 0.1
        ms = timed(lambda: ops.recon_adj(Z, g.indptr, g.indices, 1.0), 5, 50)
        print(json.dumps(dict(case="recon_adj", batch=B, hidden=H, us_per_call=round(ms * 1e3, 1), **info)), flush=True)
        for k in (1, 2, 3):
            for want in (False, True):
                ms = timed(lambda: ops.recon_logm(Z, g.graph_ptr, g.indptr, g.indices, k, 1.0, want_grad=want), 5, 50)
                print(json.dumps(dict(case="recon_logm", batch=B, hidden=H, k=k, with_grad=want, us_per_call=round(ms * 1e3, 1),
                                      **info)), flush=True)


def main():
    info = gpu_info()
    logm_cases(info)
    with tempfile.TemporaryDirectory() as tmp:
        for encoder in ("GraphSAGE", "GCN"):
            step_case("finetune", encoder, "peptides", 1024, 64, tmp, info)
            step_case("finetune", encoder, "peptides", 1024, 128, tmp, info)
            step_case("finetune", encoder, "pcqm", 4096, 64, tmp, info)
            step_case("domainadapt", encoder, "pcqm", 4096, 64, tmp, info)


if __name__ == "__main__":
    main()
