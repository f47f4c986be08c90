"""Drop-in for the reference's ``exp_pep_func_5.py`` CLI (Peptides-func: pre-train / domain-adapt / fine-tune; same flags
and defaults, reference exp_pep_func_5.py:505-553; flow of ``run`` :96-160 and ``run_epoch_graph_classification``
:168-230) on the B200 path.

    python exp_pep_func_5.py --pretrained_mode 1                       # pre-train on the dataset, save the checkpoint
    python exp_pep_func_5.py --pretrained_ds Peptides-func --domain_adapt 1      # adapt + fine-tune a checkpoint

Under torchrun (one process per GPU) every stage trains data-parallel: each rank takes ``--batch_size`` graphs per
mini-batch of its shard, the gradients are averaged in ``optimizer.step()``, evaluation splits are sharded by whole
batches and every reported value is reduced over the ranks (DESIGN.md section 6).

    torchrun --nproc-per-node 8 exp_pep_func_5.py --pretrained_mode 1
    torchrun --nproc-per-node 8 exp_pep_func_5.py --pretrained_ds Peptides-func --domain_adapt 1

The LRGB dataset is not available offline: ``pts/<dataset>_csr.pt`` (keys graph_ptr / indptr / indices / x / y) is read
if present, otherwise ``--synthetic`` Peptides-shape molecules with Bernoulli(0.1) labels are generated.  The Excel
bookkeeping of the reference (update_evaluation_value) is not reproduced.
"""
import argparse
import os
import time

import numpy as np
import torch
from torch.utils.data import DataLoader
from torch.utils.data.distributed import DistributedSampler

import exp_pretraining as pre
from models import Mainmodel, Mainmodel_domainadapt, Mainmodel_finetuning
from molecules import MoleculeDataset
from scgib_b200 import dist as sdist
from scgib_b200.graph import BatchedGraph, DeviceDataset, DeviceLoader, batch as _batch
from scgib_b200.optim import AllReduceAdam
from scgib_b200.synth import synth_batch
from train_pep_func import evaluate_network, train_epoch_domainadaptation, train_epoch_graph_classification


def load_dataset():
    path = "pts/%s_csr.pt" % args.dataset
    if os.path.exists(path):
        shard = torch.load(path)
        big = BatchedGraph(shard["graph_ptr"], shard["indptr"], shard["indices"], shard["x"])
        labels = shard["y"].float()
    else:
        print("[I] %s not found: generating %d synthetic Peptides-shape molecules" % (path, args.synthetic))
        big = synth_batch(7, args.synthetic, "peptides")
        labels = (torch.rand(args.synthetic, args.num_classes, generator=torch.Generator().manual_seed(7)) < 0.1).float()
    gp, ip = big.graph_ptr.tolist(), big.indptr
    samples = []
    for i in range(len(gp) - 1):
        n0, n1 = gp[i], gp[i + 1]
        e0, e1 = int(ip[n0]), int(ip[n1])
        g = BatchedGraph([0, n1 - n0], ip[n0:n1 + 1] - e0, big.indices[e0:e1] - n0, big.ndata["x"][n0:n1])
        samples.append((g, labels[i], None, None))
    return MoleculeDataset(samples, args.dataset), big.ndata["x"].shape[1]


REPLICA_SEED = 2024


def build_replica(cls, *a, **kw):
    """``cls(*a, **kw).to(device)``.  Data-parallel: every rank builds the same initial weights (same seed, same checkpoint),
    then the default CUDA generator, which draws the gate / feature noise, is reseeded per rank so that the ranks draw
    independent noise for their different molecules."""
    rank, world = sdist.rank_world()
    if world > 1:
        torch.manual_seed(REPLICA_SEED)
    model = cls(*a, **kw).to(device)
    if world > 1:
        torch.cuda.manual_seed(REPLICA_SEED + rank)
    return model


def set_epoch(loader, epoch):
    """DistributedSampler reshuffles per epoch only when told (DeviceLoader reshuffles on its own)."""
    if isinstance(getattr(loader, "sampler", None), DistributedSampler):
        loader.sampler.set_epoch(epoch)


def exists_on_rank0(path):
    """The same "checkpoint exists" answer on every rank: rank 0's."""
    exists = os.path.exists(path)
    if sdist.rank_world()[1] > 1:
        import torch.distributed as dist
        flag = torch.tensor([int(exists)], device=device)
        dist.broadcast(flag, 0)
        exists = bool(flag.item())
    return exists


def print_checksum(model, what):
    """Data parallel: the replicas must stay identical; each rank prints the sum of its parameters and buffers."""
    rank, world = sdist.rank_world()
    if world > 1:
        chk = float(sum(t.detach().double().sum() for t in list(model.parameters()) + list(model.buffers())))
        print("rank %d parameter checksum %s %.10f" % (rank, what, chk))


def save_checkpoint(model, path):
    """Average the BatchNorm running statistics over the ranks, write the file from rank 0, and let no rank go on (and
    load it) before it is written."""
    rank, world = sdist.rank_world()
    sdist.average_bn_buffers_(model)
    if rank == 0:
        torch.save(model, path)
        print("[I] saved %s" % path)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    print_checksum(model, os.path.basename(path))


def run_domain_adaptation(file_name, pre_train_loader, batch_size, device):
    """reference exp_pep_func_5.py:77-95."""
    rank = sdist.rank_world()[0]
    model = build_replica(Mainmodel_domainadapt, args, args.num_features, hidden_dim=args.dims, num_layers=args.num_layers,
                          num_heads=args.num_heads, k_transition=args.k_transition, num_classes=args.num_classes,
                          cp_filename=file_name, encoder=args.encoder)
    optimizer = AllReduceAdam(model.parameters(), lr=args.lr, weight_decay=5e-5)
    best_model, best_loss, best_epoch = model, 100000000, 0
    for epoch in range(1, args.adapt_epoches):
        set_epoch(pre_train_loader, epoch)
        epoch_train_loss, reconstruction_loss = train_epoch_domainadaptation(model, args, optimizer, device, pre_train_loader,
                                                                             epoch, 1, batch_size)
        if best_loss >= epoch_train_loss:
            best_model, best_epoch, best_loss = model, epoch, epoch_train_loss
        if epoch - best_epoch > 20:
            break
        if rank == 0:
            print("Epoch:%d	|Best_epoch:%d	|Train_loss:%0.4f	 |reconstruction_loss:%0.4f	" % (epoch, best_epoch, epoch_train_loss, reconstruction_loss))
    return best_model, best_epoch


def run_epoch_graph_classification(train_loader, val_loader, test_loader, num_features, file_name, batch_size):
    """reference exp_pep_func_5.py:168-230."""
    rank = sdist.rank_world()[0]
    model = build_replica(Mainmodel_finetuning, args, num_features, hidden_dim=args.dims, num_layers=args.num_layers,
                          num_heads=args.num_heads, k_transition=args.k_transition, num_classes=args.num_classes,
                          cp_filename=file_name, encoder=args.encoder)
    best_model = model
    optimizer = AllReduceAdam(model.parameters(), lr=args.lr, weight_decay=1e-5)
    best_loss, best_epoch, epoch = 100000000, 0, 0
    t0 = time.time()
    tr, va, te = [], [], []
    for epoch in range(1, args.ft_epoches):
        set_epoch(train_loader, epoch)
        loss, tr_m, optimizer = train_epoch_graph_classification(args, model, optimizer, device, train_loader, epoch, batch_size)
        sdist.average_bn_buffers_(model)          # evaluation runs on the running statistics: the same on every rank
        val_loss, va_m = evaluate_network(args, model, optimizer, device, val_loader, epoch, batch_size)
        _, te_m = evaluate_network(args, model, optimizer, device, test_loader, epoch, batch_size)
        tr.append(float(tr_m)); va.append(float(va_m)); te.append(float(te_m))
        if best_loss >= loss:
            best_model, best_epoch, best_loss = model, epoch, loss
        if epoch - best_epoch > 50:
            break
        if rank == 0:
            print(f'Epoch: {epoch}	|Best_epoch: {best_epoch}	|Train_loss: {np.round(loss, 6)}	|Val_loss: {np.round(val_loss, 6)}	'
                  f'| Train_ap: {np.round(tr[-1], 6)}	| Val_ap: {np.round(va[-1], 6)}	| epoch_test_ap: {np.round(te[-1], 6)} ')
    sdist.average_bn_buffers_(best_model)
    _, test_ap = evaluate_network(args, best_model, optimizer, device, test_loader, epoch, batch_size)
    print_checksum(best_model, "fine-tuned")
    print("TOTAL TIME TAKEN: {:.4f}s".format(time.time() - t0))
    return test_ap.cpu(), best_epoch


def run(i, dataset_full, num_features, num_classes):
    """reference exp_pep_func_5.py:96-160."""
    batch_size = args.batch_size
    collate = dataset_full.collate
    rank, world = sdist.rank_world()
    # data parallel: the training splits are sharded by molecules (equal counts per rank, the remainder dropped), the
    # evaluation splits by whole batches, round robin, so that every molecule is evaluated exactly once
    if args.device_loader and device.type == "cuda":
        # every split resident in HBM, mini-batches assembled on the GPU from molecule ids (scgib_b200.graph.DeviceLoader)
        def dev_loader(samples, shuffle):
            ds = DeviceDataset.from_batched(_batch([smp[0] for smp in samples]), device)
            return DeviceLoader(ds, batch_size, shuffle=shuffle, labels=torch.stack([torch.as_tensor(smp[1]) for smp in samples]),
                                rank=rank, world=world, shard_batches=not shuffle)
        train_loader, val_loader, test_loader = dev_loader(dataset_full.train, True), dev_loader(dataset_full.val, False), dev_loader(dataset_full.test, False)
        pre_train_loader = dev_loader(dataset_full.data_all, True)
    elif world > 1:
        def train_dl(samples):
            return DataLoader(samples, batch_size=batch_size, collate_fn=collate,
                              sampler=DistributedSampler(samples, num_replicas=world, rank=rank, shuffle=True, drop_last=True))

        def eval_dl(samples):
            shard = [list(range(lo, hi)) for lo, hi in sdist.round_robin_batches(len(samples), batch_size, rank, world)]
            return DataLoader(samples, batch_sampler=shard, collate_fn=collate)
        train_loader, val_loader, test_loader = train_dl(dataset_full.train), eval_dl(dataset_full.val), eval_dl(dataset_full.test)
        pre_train_loader = train_dl(dataset_full.data_all)
    else:
        train_loader = DataLoader(dataset_full.train, batch_size=batch_size, shuffle=True, collate_fn=collate)
        val_loader = DataLoader(dataset_full.val, batch_size=batch_size, shuffle=False, collate_fn=collate)
        test_loader = DataLoader(dataset_full.test, batch_size=batch_size, shuffle=False, collate_fn=collate)
        pre_train_loader = DataLoader(dataset_full.data_all, batch_size=batch_size, shuffle=True, collate_fn=collate)
    tag = f'{args.encoder}_{args.dims}_{args.num_layers}_{args.k_transition}'
    file_name_cpt = args.output_path + f'{args.dataset}_{tag}.pt'
    os.makedirs(args.output_path, exist_ok=True)
    if args.pretrained_mode == 1:
        if not exists_on_rank0(file_name_cpt):
            model = build_replica(Mainmodel, args, num_features, hidden_dim=args.dims, num_layers=args.num_layers,
                                  num_heads=args.num_heads, k_transition=args.k_transition, encoder=args.encoder)
            optimizer = pre.make_optimizer(model, args.lr)
            pre.args = args
            best_model, _ = pre.run_pretraining(model, pre_train_loader, optimizer, batch_size, device)
            save_checkpoint(best_model, file_name_cpt)
            print("\nFinished pre-trained model ...")
        else:
            print("\nexists pretrained model, quiting ...")
        raise SystemExit()
    ds = args.pretrained_ds
    file_name_cpt = args.output_path + f'{ds}_{tag}.pt'
    if args.domain_adapt == 1:
        file_domain_adapt = args.output_path + f'{ds}_{tag}_{args.dataset}.pt'
        if not exists_on_rank0(file_domain_adapt):
            print("\nDomain adaptation starting ...")
            best_model, _ = run_domain_adaptation(file_name_cpt, pre_train_loader, batch_size, device)
            save_checkpoint(best_model, file_domain_adapt)
        file_name_cpt = file_domain_adapt
        print("\nDomain adaptation finished ...")
    print("\nFine tunning the pre-trained model ...")
    acc, best_epoch = run_epoch_graph_classification(train_loader, val_loader, test_loader, num_features, file_name_cpt, batch_size)
    print("Graph classification: Mean %0.4f, Std %0.4f" % (float(acc), 0.0))
    return float(acc)


def main():
    args.num_classes = 10
    dataset_full, num_features = load_dataset()
    args.num_features = num_features
    res = None
    for i in range(args.run_times):
        res = run(i, dataset_full, num_features, args.num_classes)
    return res


def build_parser():
    parser = argparse.ArgumentParser(description="Experiments")
    parser.add_argument("--dataset", default="Peptides-func", help="Dataset")
    parser.add_argument("--model", default="Mainmodel", help="GNN Model")
    parser.add_argument("--run_times", type=int, default=1)
    parser.add_argument("--drop", type=float, default=0.1, help="dropout")
    parser.add_argument("--custom_masks", default=True, action='store_true', help="custom train/val/test masks")
    parser.add_argument("--device", default="cuda:0", help="GPU ids")
    parser.add_argument("--batch_size", type=int, default=128)
    parser.add_argument("--testmode", type=int, default=0)
    parser.add_argument("--pretrained_mode", type=int, default=0)
    parser.add_argument("--domain_adapt", type=int, default=0)
    parser.add_argument("--pretrained_ds", default="pre_training_v1", help="Loading pretrained model ")
    parser.add_argument("--d_transfer", type=int, default=32,
                        help="width of transfer_d, the encoders' input: 32, 64 or 128, at most --dims (default 32)")
    parser.add_argument("--layer_relax", type=int, default=0)
    parser.add_argument("--readout_f", default="sum")
    parser.add_argument("--adapt_epoches", type=int, default=50)
    parser.add_argument("--lr", type=float, default=1e-3, help="learning rate")
    parser.add_argument("--pt_epoches", type=int, default=50)
    parser.add_argument("--ft_epoches", type=int, default=50)
    parser.add_argument("--useAtt", type=int, default=1)
    parser.add_argument("--dims", type=int, default=64, help="hidden dims")
    parser.add_argument("--task", default="graph_classification")
    parser.add_argument("--encoder", default="GIN")
    parser.add_argument("--recons_type", default="adj")
    parser.add_argument("--k_transition", type=int, default=1)
    parser.add_argument("--num_layers", type=int, default=5)
    parser.add_argument("--num_heads", type=int, default=4)
    parser.add_argument("--output_path", default="outputs/", help="outputs model")
    parser.add_argument("--pre_training", default="1", help="pre_training or not")
    parser.add_argument("--index_excel", type=int, default="-1", help="index_excel")
    parser.add_argument("--file_name", default="outputs_excels.xlsx", help="file_name dataset")
    # additions of the B200 port (not in the reference)
    parser.add_argument("--gin_layers", type=int, default=4, help="GINConv per encoder (4 in the published models.py)")
    parser.add_argument("--device_loader", type=int, default=1, help="1: splits resident in HBM + GPU-side batch assembly; 0: torch DataLoader + collate")
    parser.add_argument("--dtype", default="fp32", choices=["fp32", "bf16"], help="bf16 = bf16 activations inside the GIN / GraphSAGE / GCN encoders (see exp_pretraining.py)")
    parser.add_argument("--engine_loop", type=int, default=1, help="pre-training stage: epoch through the engine API (see exp_pretraining.py)")
    parser.add_argument("--synthetic", type=int, default=512, help="synthetic molecules when pts/<dataset>_csr.pt is absent")
    return parser


if __name__ == '__main__':
    args = build_parser().parse_args()
    distributed = int(os.environ.get("WORLD_SIZE", "1")) > 1
    if distributed:             # torchrun: one process per GPU, --device is replaced by the local rank's GPU
        _rank, _local, _world = sdist.init_from_env("nccl")
        args.device = "cuda:%d" % _local
    print(args)
    device = torch.device(args.device)
    try:
        main()
    except SystemExit as e:     # --pretrained_mode 1 quits after the pre-training stage, as the reference does
        if e.code not in (None, 0) or not distributed:
            raise
    if distributed:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
