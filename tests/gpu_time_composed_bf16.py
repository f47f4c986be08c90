"""Time --dtype bf16 against fp32 on the GraphSAGE / GCN composed path (measurement, no target):

    python -m tests.gpu_time_composed_bf16

Cases: pre-training at PCQM shape, B = 4096, and fine-tuning at Peptides shape, B = 1024, hidden 64 and 128, both encoders.
A step is forward + loss + backward + torch Adam on a batch resident in HBM (k-hop ego-nets built once, outside the timed
region), timed with CUDA events after warm-up.  fp32 and bf16 alternate (two rounds) in one process, so both see the same
machine state.  Per case and dtype, one more run under torch.profiler gives the device time per kernel (the operator
breakdown).  One JSON line per measurement; the GPU name and power limit are read in the same run."""
import json
import os
import tempfile

import torch
import torch.nn.functional as F

from tests.gpu_time_composed_downstream import DEV, _args, gpu_info, timed


def build_step(kind, encoder, B, hidden, dtype, tmp):
    import models
    from scgib_b200.graph import khop_ego_batch
    from scgib_b200.synth import synth_batch
    torch.manual_seed(0)
    shape = "pcqm" if kind == "pretrain" else "peptides"
    g = synth_batch(1, B, shape).to(DEV)
    ego = khop_ego_batch(g, 1)
    x = F.normalize(g.ndata["x"].float())
    if kind == "pretrain":
        m = models.Mainmodel(_args(batch_size=B, dtype=dtype), 9, hidden, 4, 4, 1, encoder).to(DEV).train()

        def loss_fn():
            _, kl, con, rec = m.forward(g, x, ego, None, None, 1, None, 2, DEV, B)
            return kl + con + rec
    else:
        pre = models.Mainmodel(_args(), 9, hidden, 4, 4, 1, encoder)
        ckpt = os.path.join(tmp, "%s_%d.pt" % (encoder, hidden))
        torch.save(pre, ckpt)
        m = models.Mainmodel_finetuning(_args(dtype=dtype), 9, hidden, 4, 4, 1, 10, ckpt, encoder).to(DEV).train()
        targets = (torch.rand(B, 10, device=DEV) < 0.1).float()

        def loss_fn():
            scores, _, _, _ = m.forward(g, x, ego, None, 1, None, 2, DEV, B)
            return m.loss(scores, targets)
    opt = torch.optim.Adam([p for p in m.parameters() if p.requires_grad], lr=1e-4)

    def step():
        opt.zero_grad()
        loss_fn().backward()
        opt.step()
    return step


def kernel_breakdown(step, steps=3):
    """device time per kernel name (ms per step), largest first"""
    from torch.profiler import ProfilerActivity, profile
    step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            step()
        torch.cuda.synchronize()
    tot = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            tot[e.key] = tot.get(e.key, 0.0) + t / 1e3 / steps
    return {k[:80]: round(v, 4) for k, v in sorted(tot.items(), key=lambda kv: -kv[1])[:14]}


def main():
    info = gpu_info()
    cases = [(kind, enc, B, h) for kind, B in (("pretrain", 4096), ("finetune", 1024)) for enc in ("GraphSAGE", "GCN")
             for h in (64, 128)]
    with tempfile.TemporaryDirectory() as tmp:
        for kind, enc, B, h in cases:
            steps = {dt: build_step(kind, enc, B, h, dt, tmp) for dt in ("fp32", "bf16")}
            res = {"fp32": [], "bf16": []}
            for _ in range(2):
                for dt in ("fp32", "bf16"):
                    res[dt].append(timed(steps[dt], 3, 20))
            for dt in ("fp32", "bf16"):
                ms = min(res[dt])
                print(json.dumps(dict(case="%s_step" % kind, encoder=enc, batch=B, hidden=h, dtype=dt, ms_per_step=round(ms, 3),
                                      runs_ms=[round(v, 3) for v in res[dt]], graphs_per_s=round(B / ms * 1e3), **info)), flush=True)
            for dt in ("fp32", "bf16"):
                print(json.dumps(dict(case="%s_kernels" % kind, encoder=enc, batch=B, hidden=h, dtype=dt,
                                      ms_per_step_by_kernel=kernel_breakdown(steps[dt]))), flush=True)


if __name__ == "__main__":
    main()
