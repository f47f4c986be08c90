"""Weak scaling of the data-parallel fine-tuning step (Mainmodel_finetuning, GIN engine, AllReduceAdam).

Driver (no torchrun environment): launches this script under torchrun at world 1, 2, 4 and 8 (as many as there are
GPUs), reads the card name and power limit with nvidia-smi in the same call, and prints one JSON line per configuration
and world with the weak-scaling efficiency against world 1.

    python tests/gpu_time_finetune_dp.py [--out profiles/r03_finetune_dp.jsonl]

Worker (under torchrun): per configuration, one batch per rank resident in HBM; the timed step is the loop body of
train_pep_func.train_epoch_graph_classification (ego-net extraction, forward, loss / 2, backward, optimizer.step()),
with the optimizer stepping every batch.  CUDA events around the step, and around every all-reduce inside
AllReduceAdam.step (torch.distributed.all_reduce wrapped for the measurement)."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CONFIGS = [  # (name, shape, graphs per GPU, hidden, dtype)
    ("peptides_B1024_h128_fp32", "peptides", 1024, 128, "fp32"),
    ("peptides_B1024_h128_bf16", "peptides", 1024, 128, "bf16"),
    ("pcqm_B4096_h64_fp32", "pcqm", 4096, 64, "fp32"),
]


def worker(steps, warmup):
    import torch
    import torch.distributed as dist
    import torch.nn.functional as F
    from scgib_b200 import dist as sdist
    rank, local, world = sdist.init_from_env("nccl")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    import models
    from scgib_b200.graph import khop_ego_batch
    from scgib_b200.optim import AllReduceAdam
    from scgib_b200.synth import synth_batch

    ar_events = []
    real_all_reduce = dist.all_reduce

    def timed_all_reduce(t, *a, **kw):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = real_all_reduce(t, *a, **kw)
        e1.record()
        ar_events.append((e0, e1, t.numel()))
        return out

    tmp = tempfile.mkdtemp(prefix="scgib_dp_") if rank == 0 else None
    holder = [tmp]
    if world > 1:
        dist.broadcast_object_list(holder, 0)
    tmp = holder[0]
    for name, shape, B, H, dtype in CONFIGS:
        args = types.SimpleNamespace(recons_type="adj", useAtt=1, readout_f="sum", d_transfer=32, device=str(dev), batch_size=B,
                                     task="graph_classification", dataset="Peptides-func", k_transition=1, gin_layers=4,
                                     dtype=dtype, encoder="GIN")
        ckpt = os.path.join(tmp, "%s.pt" % name)
        if rank == 0:
            torch.manual_seed(5)
            torch.save(models.Mainmodel(args, 9, hidden_dim=H, num_layers=4, num_heads=4, k_transition=1, encoder="GIN"), ckpt)
        if world > 1:
            dist.barrier()
        torch.manual_seed(7)
        model = models.Mainmodel_finetuning(args, 9, hidden_dim=H, num_layers=4, num_heads=4, k_transition=1, num_classes=10,
                                            cp_filename=ckpt, encoder="GIN").to(dev)
        torch.cuda.manual_seed(100 + rank)
        opt = AllReduceAdam(model.parameters(), lr=1e-3, weight_decay=1e-5)
        g = synth_batch(50 + rank, B, shape).to(dev)
        y = (torch.rand(B, 10, generator=torch.Generator().manual_seed(2 + rank)) < 0.1).float().to(dev)
        model.train()

        def step():
            opt.zero_grad()
            ego = khop_ego_batch(g, 1)
            x = F.normalize(g.ndata["x"].float())
            scores, _, _, _ = model.forward(g, x, ego, None, 1, None, 2, dev, B)
            loss = model.loss(scores, y) / 2
            loss.backward()
            opt.step()

        dist.all_reduce = timed_all_reduce
        for _ in range(warmup):
            step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ar_events.clear()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        dist.all_reduce = real_all_reduce
        ms = e0.elapsed_time(e1) / steps
        ar_ms = sum(a.elapsed_time(b) for a, b, _ in ar_events) / steps
        n_floats = ar_events[0][2] if ar_events else 0
        # the slowest rank sets the pace of a synchronous step: report the max over ranks
        t = torch.tensor([ms, ar_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ar_ms = t.tolist()
        if rank == 0:
            print(json.dumps({"config": name, "shape": shape, "graphs_per_gpu": B, "hidden": H, "dtype": dtype, "gin_layers": 4,
                              "world": world, "steps": steps, "warmup": warmup, "step_ms": ms, "graphs_per_s": world * B / ms * 1e3,
                              "allreduce_ms": ar_ms if world > 1 else 0.0, "allreduce_floats": n_floats,
                              "allreduce_share": (ar_ms / ms) if world > 1 else 0.0}), flush=True)
        del model, opt
        torch.cuda.empty_cache()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        shutil.rmtree(tmp, ignore_errors=True)


def driver(steps, warmup, out):
    import torch
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    gpu = [l.strip() for l in smi.stdout.strip().splitlines()]
    n = torch.cuda.device_count()
    lines, base = [], {}
    for world in (1, 2, 4, 8):
        if world > n:
            break
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
                            "--master-addr", "127.0.0.1", "--master-port", str(29610 + world), os.path.abspath(__file__),
                            "--worker", "--steps", str(steps), "--warmup", str(warmup)], capture_output=True, text=True,
                           cwd=ROOT, timeout=1800)
        if r.returncode != 0:
            sys.stderr.write(r.stdout[-4000:] + r.stderr[-4000:])
            raise SystemExit("world %d failed" % world)
        for l in r.stdout.splitlines():
            if not l.startswith("{"):
                continue
            d = json.loads(l)
            if world == 1:
                base[d["config"]] = d["step_ms"]
            d["weak_scaling_efficiency"] = base[d["config"]] / d["step_ms"] if d["config"] in base else None
            d["gpu"] = gpu[0] if gpu else None
            d["gpus_seen"] = gpu
            lines.append(d)
            print(json.dumps(d), flush=True)
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.worker:
        worker(a.steps, a.warmup)
    else:
        driver(a.steps, a.warmup, a.out)
