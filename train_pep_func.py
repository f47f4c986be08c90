"""Drop-in for the reference's ``train_pep_func.py`` training / evaluation loops (reference train_pep_func.py:91-230) on the
B200 path: same function names, arguments and return values.  Differences: the ego-nets come from the GPU extraction
kernel (``khop_ego_batch``) instead of pickled DGLGraph lists, and the NaN-masking of ``MetricWrapper`` (goli / ogb are not
installable here) is restated in ``masked_loss``.

Under torch.distributed (one process per GPU) every function returns the per-batch mean over the union of all ranks'
batches (``scgib_b200.dist.mean_over_ranks``), identical on every rank; single process, the values are the reference's."""
import torch
import torch.nn.functional as F

from scgib_b200.dist import mean_over_ranks, rank_world
from scgib_b200.graph import khop_ego_batch


def masked_loss(loss_fn, scores, targets):
    """MetricWrapper(metric, target_nan_mask="ignore-flatten") (train_pep_func.py:139): drop NaN targets, flatten."""
    mask = ~torch.isnan(targets)
    if bool(mask.all()):
        return loss_fn(scores, targets)
    return loss_fn(scores[mask], targets[mask])


def train_epoch_domainadaptation(model, args, optimizer, device, data_loader, epoch, k_transition, batch_size=16):
    """reference train_pep_func.py:91-124 -> (epoch_loss, epoch_reconstruction_loss)."""
    model.train()
    epoch_loss = 0
    epoch_reconstruction_loss = 0
    count = 0
    for it, (batch_graphs, _, batch_subgraphs, batch_logMs) in enumerate(data_loader):
        count = it
        batch_graphs = batch_graphs.to(device)
        batch_x = batch_graphs.ndata['x'].float().to(device)
        optimizer.zero_grad()
        flatten_batch_subgraphs = khop_ego_batch(batch_graphs, args.k_transition)
        batch_x = F.normalize(batch_x)
        reconstruction_loss = model.forward(batch_graphs, batch_x, flatten_batch_subgraphs, batch_logMs, None, 1, None, 2,
                                            device, batch_size)
        loss = reconstruction_loss
        loss.backward()
        optimizer.step()
        epoch_loss += loss.detach().item()
        epoch_reconstruction_loss += reconstruction_loss.detach()
    if rank_world()[1] > 1:
        epoch_loss, rec = mean_over_ranks([epoch_loss, epoch_reconstruction_loss], count + 1, device)
        return epoch_loss, torch.tensor(rec, dtype=torch.float32, device=device)
    epoch_loss /= (count + 1)
    epoch_reconstruction_loss /= (count + 1)
    return epoch_loss, epoch_reconstruction_loss


def train_epoch_graph_classification(args, model, optimizer, device, data_loader, epoch, batch_size):
    """reference train_pep_func.py:130-184 (gradient accumulation over 2 mini-batches) -> (loss, train metric, optimizer)."""
    model.train()
    epoch_loss = 0
    epoch_train_ap = 0
    it = -1
    n_batches = len(data_loader)
    for it, (batch_graphs, batch_targets, batch_subgraphs, _) in enumerate(data_loader):
        batch_targets = batch_targets.to(device)
        batch_graphs = batch_graphs.to(device)
        batch_x = batch_graphs.ndata['x'].float().to(device)
        optimizer.zero_grad()       # as the reference does (train_pep_func.py:152): every iteration, before the forward
        flatten_batch_subgraphs = khop_ego_batch(batch_graphs, args.k_transition)
        batch_x = F.normalize(batch_x)
        batch_scores, _, _, _ = model.forward(batch_graphs, batch_x, flatten_batch_subgraphs, None, 1, None, 2, device,
                                              batch_size)
        loss = masked_loss(model.loss, batch_scores, batch_targets)
        loss = loss / 2
        loss.backward()
        if ((it + 1) % 2 == 0) or (it + 1 == n_batches):
            optimizer.step()
            optimizer.zero_grad()
        epoch_loss += loss.detach().item()
        epoch_train_ap += model.BCEWithLogitsLoss(batch_scores.detach(), batch_targets)
    if rank_world()[1] > 1:
        epoch_loss, ap = mean_over_ranks([epoch_loss, epoch_train_ap], it + 1, device)
        return epoch_loss, torch.tensor(ap, dtype=torch.float32), optimizer
    epoch_train_ap /= (it + 1)
    epoch_loss /= (it + 1)
    return epoch_loss, epoch_train_ap.detach().cpu(), optimizer


def evaluate_network(args, model, optimizer, device, data_loader, epoch, batch_size):
    """reference train_pep_func.py:187-230: model.eval() (running statistics in every BatchNorm) -> (loss, metric)."""
    model.eval()
    epoch_test_loss = 0
    epoch_test_ap = 0
    it = -1
    with torch.no_grad():
        for it, (batch_graphs, batch_targets, batch_subgraphs, _) in enumerate(data_loader):
            batch_graphs = batch_graphs.to(device)
            batch_x = batch_graphs.ndata['x'].float().to(device)
            batch_targets = batch_targets.to(device)
            flatten_batch_subgraphs = khop_ego_batch(batch_graphs, args.k_transition)
            batch_x = F.normalize(batch_x)
            batch_scores, _, _, _ = model.forward(batch_graphs, batch_x, flatten_batch_subgraphs, None, 1, None, 2, device)
            loss = masked_loss(model.loss, batch_scores, batch_targets)
            epoch_test_loss += loss.detach().item()
            epoch_test_ap += model.BCEWithLogitsLoss(batch_scores, batch_targets)
    if rank_world()[1] > 1:         # whole-batch shards (round robin): a rank may hold fewer batches, or none
        loss, ap = mean_over_ranks([epoch_test_loss, epoch_test_ap], it + 1, device)
        return loss, torch.tensor(ap, dtype=torch.float32)
    epoch_test_ap /= (it + 1)
    epoch_test_loss /= (it + 1)
    return epoch_test_loss, epoch_test_ap.detach().cpu()
