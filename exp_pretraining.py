"""Drop-in for the reference's ``exp_pretraining.py`` CLI (same flags and defaults, reference
exp_pretraining.py:359-406) on the B200 path.

    python exp_pretraining.py --encoder GIN --dims 64 --num_layers 4 --k_transition 1 --device cuda:0

Differences forced by the environment: the OGB / QM9 / mol-PCBA datasets and the DGL ``pts/*.bin`` files are not
available offline, so ``load_graphdataset`` reads a packed CSR shard ``pts/<name>_csr.pt`` if present and otherwise
generates ``--synthetic`` molecules of the dataset's shape; k-hop ego-nets are extracted on the GPU per batch
instead of being loaded from ``pts/<name>_subgraphs_khop_<k>.pt``.
"""
import argparse
import logging
import os
import random
import time
import zlib
from pathlib import Path

import torch
import torch.nn.functional as F
from torch.utils.data import DataLoader

from molecules import MoleculeDataset
from models import Mainmodel, Mainmodel_continue
from scgib_b200.graph import BatchedGraph, DeviceDataset, DeviceLoader, batch as _batch, khop_ego_batch, load_shard
from scgib_b200.synth import synth_batch


def make_optimizer(model, lr):
    """reference exp_pretraining.py:86,112: Adam(lr, weight_decay=5e-5) over the model's parameters.  For the drop-in
    modules this is scgib_b200.optim.FlatAdam: the same update as ONE kernel over the flat parameter buffer (same
    zero_grad() / step() surface); SCGIB_TORCH_ADAM=1 keeps torch.optim.Adam on the parameter views."""
    if getattr(model, "_bridge", None) is not None and os.environ.get("SCGIB_TORCH_ADAM", "0") != "1":
        from scgib_b200.optim import FlatAdam
        return FlatAdam(model, lr=lr, weight_decay=5e-5)
    from scgib_b200.optim import AllReduceAdam          # torch.optim.Adam (+ the gradient all-reduce under torchrun)
    return AllReduceAdam(model.parameters(), lr=lr, weight_decay=5e-5)


def run_pretraining(model, pre_train_loader1, optimizer, batch_size, device):
    best_epoch, best_model, best_loss = 0, model, 100000000
    rank, world = _rank_world()
    for epoch in range(1, args.pt_epoches):
        if hasattr(pre_train_loader1.sampler, "set_epoch"):
            pre_train_loader1.sampler.set_epoch(epoch)
        t0 = time.time()
        fast = getattr(args, "engine_loop", 0) and isinstance(pre_train_loader1, DeviceLoader) and type(optimizer).__name__ == "FlatAdam"
        epoch_fn = train_epoch_pre_training_engine if fast else train_epoch_pre_training
        epoch_train_loss, KL_Loss, contrastive_loss, reconstruction_loss = epoch_fn(
            model, args, optimizer, device, pre_train_loader1, epoch, 1, batch_size)
        if world > 1:        # every rank must take the same early-stopping decision: use the mean loss over the ranks
            import torch.distributed as dist
            t = torch.tensor([epoch_train_loss], device=device, dtype=torch.float64)
            dist.all_reduce(t)
            epoch_train_loss = float(t) / world
        if rank == 0:
            n_graphs = len(pre_train_loader1) * batch_size * world
            print('{"epoch": %d, "graphs_per_s": %.0f, "world": %d}' % (epoch, n_graphs / max(time.time() - t0, 1e-9), world))
        if best_loss >= epoch_train_loss:
            best_model, best_epoch, best_loss = model, epoch, epoch_train_loss
        if epoch - best_epoch > 50:
            break
        if rank == 0:
            print("Epoch:%d	|Best_epoch:%d	|Train_loss:%0.4f" % (epoch, best_epoch, epoch_train_loss))
    return best_model, best_epoch


def train_epoch_pre_training_engine(model, args, optimizer, device, data_loader, epoch, k_transition, batch_size=16):
    """The same epoch as ``train_epoch_pre_training`` driven through the engine API (``--engine_loop 1``, the default when
    the data comes from a ``DeviceLoader`` and the optimiser is ``FlatAdam``): the next batch (ids -> GPU batch assembly ->
    ego-nets) is prepared on a side stream while the current step runs, forward / backward / Adam are three library calls
    on the shared flat buffers, and the per-step ``loss.item()`` of the reference loop (exp_pretraining.py:324) is replaced
    by ONE device-to-host read per epoch.  Same parameters, BatchNorm buffers, Adam state and return values."""
    model.train()
    bridge = model._bridge
    bridge.sync(device)
    eng = bridge.engine
    eng.recon_logm_steps = int(model.k_transition) if getattr(model, "recons_type", "adj") == "logM" else 0
    g = optimizer.param_groups[0]
    rank, world = _rank_world()
    acc = torch.zeros(4, device=device, dtype=torch.float64)
    steps = n_graphs = 0
    it = data_loader.id_batches()
    ids = next(it, None)
    handle = None if ids is None else eng.prefetch_ids(data_loader.dataset, ids, args.k_transition, normalize_x=True)
    while handle is not None:
        b = eng.wait_batch(handle)
        losses = eng.train_step(b, lr=g["lr"], weight_decay=g["weight_decay"], world_size=world)
        acc += losses.double()
        steps += 1
        n_graphs += b.B
        ids = next(it, None)
        handle = None if ids is None else eng.prefetch_ids(data_loader.dataset, ids, args.k_transition, normalize_x=True)
    inner = bridge._bn_modules                                   # nn.BatchNorm1d bookkeeping of the module view
    for enc in (inner.Encoder1, inner.Encoder2):
        for bn in enc.batch_norms:
            bn.num_batches_tracked += steps
    inner.compressor[1].num_batches_tracked += n_graphs          # one BatchNorm call per graph (models.py:642)
    kl, con, rec, tot = (acc / max(steps, 1)).tolist()            # the epoch's one host read
    return tot, torch.tensor(kl), torch.tensor(con), torch.tensor(rec)


def train_epoch_pre_training(model, args, optimizer, device, data_loader, epoch, k_transition, batch_size=16):
    """reference exp_pretraining.py:290-333, one difference: ego-nets come from the GPU extraction kernel."""
    model.train()
    epoch_loss = epoch_KL = epoch_con = epoch_rec = 0
    count = 0
    for it, (batch_graphs, _, batch_subgraphs, batch_logMs) in enumerate(data_loader):
        count = it
        batch_graphs = batch_graphs.to(device)
        batch_x = batch_graphs.ndata['x'].float().to(device)
        edge_index = None
        optimizer.zero_grad()
        flatten_batch_subgraphs = khop_ego_batch(batch_graphs, args.k_transition)
        x_subs = None                                   # rows of batch_x (ego_nodes); never materialised
        batch_x = F.normalize(batch_x)
        _, KL_Loss, contrastive_loss, reconstruction_loss = model.forward(
            batch_graphs, batch_x, flatten_batch_subgraphs, batch_logMs, x_subs, 1, edge_index, 2, device, batch_size)
        loss = KL_Loss + reconstruction_loss + contrastive_loss
        loss.backward()
        optimizer.step()
        epoch_loss += loss.detach().item()
        epoch_KL += KL_Loss.detach(); epoch_con += contrastive_loss.detach(); epoch_rec += reconstruction_loss.detach()
    n = count + 1
    return epoch_loss / n, epoch_KL / n, epoch_con / n, epoch_rec / n


def load_graphdataset(dataset_name):
    args.dataset = dataset_name
    args.num_features = dict(zip(args.dataset_list, args.feature_list))[dataset_name]
    path = "pts/%s_csr.pt" % dataset_name
    samples_all = []
    if os.path.exists(path):
        big, _ = load_shard(path)             # written by scgib_b200.graph.pack_shard from PyG-style (edge_index, x, y)
        args.num_features = int(big.ndata["x"].shape[1])      # the shard's own feature width (e.g. NCI1 37, DD 89)
    else:
        print("[I] %s not found: generating %d synthetic molecules of the %s shape" % (path, args.synthetic, dataset_name))
        big = synth_batch(zlib.crc32(dataset_name.encode()) % 1000, args.synthetic)     # the same molecules in every process
        if args.num_features != big.ndata["x"].shape[1]:
            big.ndata["x"] = torch.cat([big.ndata["x"], torch.rand(big.num_nodes(), args.num_features - 9)], 1)
    gp, ip = big.graph_ptr.tolist(), big.indptr
    for i in range(len(gp) - 1):
        n0, n1 = gp[i], gp[i + 1]
        e0, e1 = int(ip[n0]), int(ip[n1])
        g = BatchedGraph([0, n1 - n0], ip[n0:n1 + 1] - e0, big.indices[e0:e1] - n0, big.ndata["x"][n0:n1])
        samples_all.append((g, torch.zeros(1), None, None))
    random.Random(0).shuffle(samples_all) if int(os.environ.get("WORLD_SIZE", "1")) > 1 else random.shuffle(samples_all)
    return MoleculeDataset(samples_all, 'pre_training'), args.num_features


def _rank_world():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def _barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()


def run(i, dataset_full1, feature1, dataset_full2, feature2, dataset_full3, feature3):
    """Three-stage sequential pre-training, reference exp_pretraining.py:81-145."""
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        torch.manual_seed(2024)                            # identical initial weights on every rank
    model = Mainmodel(args, feature1, hidden_dim=args.dims, num_layers=args.num_layers, num_heads=args.num_heads,
                      k_transition=args.k_transition, encoder=args.encoder).to(device)
    batch_size = args.batch_size
    rank, world = _rank_world()
    if args.device_loader and device.type == "cuda":
        # the datasets stay resident in HBM and every mini-batch is assembled on the GPU from its molecule ids (no Python
        # object per molecule, no collate, no H2D of graph data): the host-side DataLoader tops out far below the kernels
        loaders = [DeviceLoader(DeviceDataset.from_batched(_batch([smp[0] for smp in d.data_all]), device), batch_size,
                                shuffle=True, drop_last=world > 1, rank=rank, world=world) for d in (dataset_full1, dataset_full2, dataset_full3)]
    elif world > 1:    # data parallelism (torchrun): every rank takes its shard of each epoch; FlatAdam all-reduces the gradients
        from torch.utils.data.distributed import DistributedSampler
        loaders = [DataLoader(d.data_all, batch_size=batch_size, collate_fn=d.collate,
                              sampler=DistributedSampler(d.data_all, num_replicas=world, rank=rank, shuffle=True, drop_last=True))
                   for d in (dataset_full1, dataset_full2, dataset_full3)]
    else:
        loaders = [DataLoader(d.data_all, batch_size=batch_size, shuffle=True, collate_fn=d.collate)
                   for d in (dataset_full1, dataset_full2, dataset_full3)]
    features = [feature1, feature2, feature3]
    Path(args.output_path).mkdir(parents=True, exist_ok=True)
    if args.pretrained_mode == 1:
        tag = f'{args.encoder}_{args.dims}_{args.num_layers}_{args.k_transition}.pt'
        file_name_cpt = args.output_path + f'pre_training_{args.dataset_list[0]}_{tag}'
        prev = file_name_cpt
        for stage in range(len(args.dataset_list)):
            name = "_".join(args.dataset_list[:stage + 1])
            file_check = args.output_path + f'pre_training_{name}_{tag}'
            todo = not os.path.exists(file_check)
            if world > 1:                                  # every rank takes the same branch (rank 0 writes the files)
                import torch.distributed as dist
                flag = torch.tensor([int(todo)], device=device)
                dist.broadcast(flag, 0)
                todo = bool(flag.item())
            if todo:
                if stage == 0:
                    if rank == 0:
                        torch.save(model, file_check)
                    _barrier(world)
                if world > 1:
                    torch.manual_seed(20240 + stage)       # identical initialisation of the new transfer_d / MLP on every rank
                wrapped = Mainmodel_continue(args, features[stage], hidden_dim=args.dims, num_layers=args.num_layers,
                                             num_heads=args.num_heads, k_transition=args.k_transition, num_classes=1,
                                             cp_filename=prev if stage else file_check, encoder=args.encoder).to(device)
                optimizer = make_optimizer(wrapped, args.lr)
                best_model, _ = run_pretraining(wrapped, loaders[stage], optimizer, batch_size, device)
                if world > 1:
                    chk = float(sum(p.detach().double().sum() for p in best_model.parameters()))
                    print("rank %d stage %d parameter checksum %.10f" % (rank, stage + 1, chk))
                if rank == 0:
                    torch.save(best_model, file_check)
                _barrier(world)
            prev = file_check
            print(f"Finished pre-trained model step {stage + 1}...")
    print(f"\nFinished pretraining models on {str(args.dataset_list)} ...")
    return 0


def main():
    timestr = time.strftime("%Y%m%d-%H%M%S")
    Path("./exp_logs").mkdir(parents=True, exist_ok=True)
    logging.basicConfig(filename="exp_logs/" + args.dataset + "-" + timestr + ".log", filemode="w", level=logging.INFO)
    logging.info("Starting on device: %s", device)
    logging.info("Config: %s ", args)
    args.dataset_list = ['PCQM4Mv2', 'QM9', 'mol-PCBA']
    args.feature_list = [9, 11, 9]
    sets = [load_graphdataset(n) for n in args.dataset_list]
    for i in range(args.run_times):
        run(i, sets[0][0], sets[0][1], sets[1][0], sets[1][1], sets[2][0], sets[2][1])


def build_parser():
    parser = argparse.ArgumentParser(description="Experiments")
    parser.add_argument("--dataset", default="pre-train", help="Dataset")
    parser.add_argument("--model", default="Mainmodel", help="GNN Model")
    parser.add_argument("--run_times", type=int, default=1)
    parser.add_argument("--drop", type=float, default=0.1, help="dropout")
    parser.add_argument("--custom_masks", default=True, action='store_true', help="custom train/val/test masks")
    parser.add_argument("--device", default="cuda:0", help="GPU ids")
    parser.add_argument("--pretrained_mode", type=int, default=1)
    parser.add_argument("--domain_adapt", type=int, default=0)
    parser.add_argument("--d_transfer", type=int, default=32,
                        help="width of transfer_d, the encoders' input: 32, 64 or 128, at most --dims (default 32)")
    parser.add_argument("--layer_relax", type=int, default=0)
    parser.add_argument("--readout_f", default="sum")
    parser.add_argument("--batch_size", type=int, default=128)
    parser.add_argument("--testmode", type=int, default=0)
    parser.add_argument("--lr", type=float, default=1e-4, help="learning rate")
    parser.add_argument("--pt_epoches", type=int, default=100)
    parser.add_argument("--ft_epoches", type=int, default=100)
    parser.add_argument("--useAtt", type=int, default=1)
    parser.add_argument("--dims", type=int, default=64, help="hidden dims")
    parser.add_argument("--task", default="graph_classification")
    parser.add_argument("--encoder", default="GIN")
    parser.add_argument("--recons_type", default="adj")
    parser.add_argument("--k_transition", type=int, default=1)
    parser.add_argument("--num_layers", type=int, default=4)
    parser.add_argument("--num_heads", type=int, default=4)
    parser.add_argument("--output_path", default="outputs/", help="outputs model")
    parser.add_argument("--pre_training", default="1", help="pre_training or not")
    parser.add_argument("--index_excel", type=int, default="-1", help="index_excel")
    parser.add_argument("--file_name", default="outputs_excels.xlsx", help="file_name dataset")
    # additions of the B200 port (not in the reference)
    parser.add_argument("--gin_layers", type=int, default=4, help="GINConv per encoder (4 in the published models.py; 5 = paper / shipped checkpoint)")
    parser.add_argument("--dtype", default="fp32", choices=["fp32", "bf16"], help="fp32 = reference precision; bf16 = bf16 activations inside the encoders, on single-pass bf16 tensor-core products (the GIN MLPs; the GraphSAGE / GCN linear layers and their weight gradients); parameters / optimiser stay fp32")
    parser.add_argument("--engine_loop", type=int, default=1, help="1: drive the epoch through the engine API (prefetch stream, one host read per epoch); 0: the reference's loop body")
    parser.add_argument("--device_loader", type=int, default=1, help="1: datasets resident in HBM + GPU-side batch assembly (DeviceLoader); 0: torch DataLoader + collate as in the reference")
    parser.add_argument("--synthetic", type=int, default=2048, help="synthetic molecules per dataset when pts/<name>_csr.pt is absent")
    return parser


if __name__ == '__main__':
    args = build_parser().parse_args()
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:         # torchrun: one process per GPU, --device is replaced by the local rank's GPU
        from scgib_b200.dist import init_from_env
        _rank, _local, _world = init_from_env("nccl")
        args.device = "cuda:%d" % _local
    print(args)
    device = torch.device(args.device)
    main()
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
