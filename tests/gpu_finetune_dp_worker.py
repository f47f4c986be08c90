"""Two-rank data-parallel fine-tuning / domain adaptation against a single-process emulation (run under torchrun by
tests/test_gpu_finetune_dp.py).

Every rank trains one epoch of the real loop (train_pep_func.py) with AllReduceAdam, averages its BatchNorm running
statistics and evaluates its whole-batch shard of the validation split.  Rank 0 then replays both ranks' batches on one
replica: before each forward it restores that rank's CUDA generator state and BatchNorm buffers, and before
``torch.optim.Adam.step()`` it sets the gradient to (g0 + g1) / 2.  The last stdout line is ``RESULT <json>``.

    python -m torch.distributed.run --nproc-per-node 2 tests/gpu_finetune_dp_worker.py --mode ft --encoder GIN --out DIR
    [--backend gloo]
"""
import argparse
import json
import os
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch                                      # noqa: E402
import torch.distributed as dist                  # noqa: E402
import torch.nn.functional as F                   # noqa: E402

NOISE_SEED = 100


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", choices=["ft", "da"], default="ft")
    ap.add_argument("--encoder", default="GIN", choices=["GIN", "GraphSAGE", "GCN"])
    ap.add_argument("--dtype", default="fp32", choices=["fp32", "bf16"])
    ap.add_argument("--batch", type=int, default=48)
    ap.add_argument("--batches", type=int, default=6, help="training batches per rank")
    ap.add_argument("--backend", default="nccl", choices=["nccl", "gloo"],
                    help="gloo: both ranks share cuda:0 (the same exchange semantics on a one-GPU machine)")
    ap.add_argument("--out", required=True)
    opt = ap.parse_args()

    from scgib_b200 import dist as sdist
    rank, local, world = sdist.init_from_env(opt.backend)
    dev = torch.device("cuda", local if opt.backend == "nccl" else 0)
    torch.cuda.set_device(dev)
    import models
    import train_pep_func as tpf
    from scgib_b200.graph import DeviceDataset, DeviceLoader, khop_ego_batch
    from scgib_b200.optim import AllReduceAdam
    from scgib_b200.synth import synth_batch

    B, C = opt.batch, 10
    args = types.SimpleNamespace(recons_type="adj", useAtt=1, readout_f="sum", d_transfer=32, device=str(dev), batch_size=B,
                                 task="graph_classification", dataset="Peptides-func", k_transition=1, gin_layers=4,
                                 dtype=opt.dtype, encoder=opt.encoder)
    ckpt = os.path.join(opt.out, "pretrained.pt")
    if rank == 0:
        torch.manual_seed(5)
        torch.save(models.Mainmodel(args, 9, hidden_dim=64, num_layers=4, num_heads=4, k_transition=1, encoder=opt.encoder), ckpt)
    dist.barrier()

    n_train, n_val = world * opt.batches * B, 4 * B + B // 2            # 5 validation batches, the last one short
    train_g, val_g = synth_batch(11, n_train, "peptides"), synth_batch(12, n_val, "peptides")
    gen = torch.Generator().manual_seed(13)
    train_y, val_y = (torch.rand(n_train, C, generator=gen) < 0.1).float(), (torch.rand(n_val, C, generator=gen) < 0.1).float()
    lr, wd = 1e-3, (1e-5 if opt.mode == "ft" else 5e-5)

    def replica():
        torch.manual_seed(7)
        cls = models.Mainmodel_finetuning if opt.mode == "ft" else models.Mainmodel_domainadapt
        return cls(args, 9, hidden_dim=64, num_layers=4, num_heads=4, k_transition=1, num_classes=C, cp_filename=ckpt,
                   encoder=opt.encoder).to(dev)

    def train_loader(r):
        return DeviceLoader(DeviceDataset.from_batched(train_g, dev), B, shuffle=True, labels=train_y, rank=r, world=world)

    def snapshot(m):
        return [t.detach().cpu().clone() for _, t in sorted(list(m.named_parameters()) + list(m.named_buffers()))]

    # ------------------------------------------------------------------ data parallel
    model = replica()
    torch.cuda.manual_seed(NOISE_SEED + rank)
    optimizer = AllReduceAdam(model.parameters(), lr=lr, weight_decay=wd)
    if opt.mode == "ft":
        epoch_vals = tpf.train_epoch_graph_classification(args, model, optimizer, dev, train_loader(rank), 1, B)[:2]
    else:
        epoch_vals = tpf.train_epoch_domainadaptation(model, args, optimizer, dev, train_loader(rank), 1, 1, B)
    epoch_vals = [float(v) for v in epoch_vals]
    sdist.average_bn_buffers_(model)
    ev = None
    if opt.mode == "ft":
        val = DeviceLoader(DeviceDataset.from_batched(val_g, dev), B, shuffle=False, labels=val_y, rank=rank, world=world,
                           shard_batches=True)
        ev = [float(v) for v in tpf.evaluate_network(args, model, None, dev, val, 1, B)]
    torch.save(snapshot(model), os.path.join(opt.out, "rank%d.pt" % rank))
    dist.barrier()
    if rank != 0:
        dist.barrier()
        dist.destroy_process_group()
        return
    mine, other = snapshot(model), torch.load(os.path.join(opt.out, "rank1.pt"))
    names = [n for n, _ in sorted(list(model.named_parameters()) + list(model.named_buffers()))]
    res = {"world": world, "epoch": epoch_vals, "eval": ev,
           "ranks_differ": [n for n, a, b in zip(names, mine, other) if not torch.equal(a, b)]}

    # ------------------------------------------------------------------ single-process emulation on this GPU
    emu = replica()
    ref_opt = torch.optim.Adam(emu.parameters(), lr=lr, weight_decay=wd)
    bns = [m for m in emu.modules() if isinstance(m, torch.nn.modules.batchnorm._BatchNorm)]

    def bn_state():
        return [t.clone() for m in bns for t in (m.running_mean, m.running_var, m.num_batches_tracked)]

    def set_bn(state):
        for t, s in zip([t for m in bns for t in (m.running_mean, m.running_var, m.num_batches_tracked)], state):
            t.copy_(s)

    states = []
    for r in range(world):
        torch.cuda.manual_seed(NOISE_SEED + r)
        states.append([torch.cuda.get_rng_state(), bn_state()])
    loaders = [train_loader(r) for r in range(world)]
    n_batches = len(loaders[0])
    seen = []
    emu.train()
    for it, batches in enumerate(zip(*loaders)):
        step = opt.mode == "da" or (it + 1) % 2 == 0 or it + 1 == n_batches
        grads = []
        for r, (g, t, _, _) in enumerate(batches):
            torch.cuda.set_rng_state(states[r][0])
            set_bn(states[r][1])
            ref_opt.zero_grad()
            ego = khop_ego_batch(g, 1)
            x = F.normalize(g.ndata["x"].float())
            if opt.mode == "ft":
                scores, _, _, _ = emu.forward(g, x, ego, None, 1, None, 2, dev, B)
                loss = tpf.masked_loss(emu.loss, scores, t) / 2
            else:
                loss = emu.forward(g, x, ego, None, None, 1, None, 2, dev, B)
            loss.backward()
            seen.append(loss.item())
            states[r] = [torch.cuda.get_rng_state(), bn_state()]
            if step:
                grads.append([None if p.grad is None else p.grad.clone() for p in emu.parameters()])
        if step:
            with torch.no_grad():
                for p, *gs in zip(emu.parameters(), *grads):
                    p.grad = None if gs[0] is None else (gs[0] + gs[1]) / 2
            ref_opt.step()
    res["emu_epoch_loss"] = sum(seen) / len(seen)
    with torch.no_grad():
        set_bn([(a + b) / 2 if a.is_floating_point() else a for a, b in zip(states[0][1], states[1][1])])
    emu_snap = snapshot(emu)
    res["emu_differs"] = [n for n, a, b in zip(names, mine, emu_snap) if not torch.equal(a, b)]
    res["emu_max_diff"] = max([float((a.double() - b.double()).abs().max()) for a, b in zip(mine, emu_snap) if a.numel()] + [0.0])
    if opt.mode == "ft":
        emu.eval()
        single = DeviceLoader(DeviceDataset.from_batched(val_g, dev), B, shuffle=False, labels=val_y)
        losses, aps = [], []
        with torch.no_grad():
            for i, (g, t, _, _) in enumerate(single):
                r = i % world
                torch.cuda.set_rng_state(states[r][0])
                scores, _, _, _ = emu.forward(g, F.normalize(g.ndata["x"].float()), khop_ego_batch(g, 1), None, 1, None, 2, dev)
                losses.append(tpf.masked_loss(emu.loss, scores, t).item())
                aps.append(float(emu.BCEWithLogitsLoss(scores, t)))
                states[r][0] = torch.cuda.get_rng_state()
        res["emu_eval"] = [sum(losses) / len(losses), sum(aps) / len(aps)]
    print("RESULT " + json.dumps(res), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
