"""Host logic of data-parallel fine-tuning / domain adaptation on CPU (world 2, gloo): the whole-batch evaluation shard,
the training shards, BatchNorm running-statistics averaging through aliased buffers, the reductions of
train_pep_func.py and the early-stopping decision built on them."""
import os
import socket
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


class _IdDataset:
    """What DeviceLoader needs of a DeviceDataset to produce id batches."""
    device = "cpu"

    def __init__(self, n):
        self.n = n

    def __len__(self):
        return self.n


@pytest.mark.parametrize("B", [1, 4, 7])
def test_round_robin_eval_shard_covers_every_batch_once(B):
    from scgib_b200.dist import round_robin_batches
    from scgib_b200.graph import DeviceLoader
    for W in range(1, 9):
        for n in (B * W * 3, B * W * 3 + 1, B * W * 3 - 1, B * W + B - 1, B - 1, 0, 1):
            single = [(lo, min(lo + B, n)) for lo in range(0, n, B)]
            shards = [round_robin_batches(n, B, r, W) for r in range(W)]
            assert sorted(sum(shards, [])) == single
            for r in range(W):                                   # rank r holds batches r, r + W, ... in order
                assert shards[r] == single[r::W]
            loaders = [DeviceLoader(_IdDataset(n), B, shuffle=False, rank=r, world=W, shard_batches=True) for r in range(W)]
            ids = [[b.tolist() for b in ld.id_batches()] for ld in loaders]
            assert [len(ld) for ld in loaders] == [len(s) for s in shards]
            got = sorted(sum(ids, []))
            assert got == [list(range(lo, hi)) for lo, hi in single]
            assert sorted(i for b in got for i in b) == list(range(n))


def test_shard_batches_world1_is_the_plain_loader():
    from scgib_b200.graph import DeviceLoader
    for n, B in ((10, 3), (12, 4), (0, 2)):
        a = DeviceLoader(_IdDataset(n), B, shuffle=False)
        b = DeviceLoader(_IdDataset(n), B, shuffle=False, shard_batches=True)
        assert [x.tolist() for x in a.id_batches()] == [x.tolist() for x in b.id_batches()] and len(a) == len(b)


def test_train_shards_have_equal_lengths():
    from torch.utils.data import DataLoader
    from torch.utils.data.distributed import DistributedSampler
    from scgib_b200.graph import DeviceLoader
    for W in range(1, 9):
        for n, B in ((307, 16), (64, 8), (1000, 128), (9, 4)):
            lens = [len(DeviceLoader(_IdDataset(n), B, shuffle=True, rank=r, world=W)) for r in range(W)]
            assert len(set(lens)) == 1
            ids = [torch.cat(list(DeviceLoader(_IdDataset(n), B, shuffle=True, rank=r, world=W).id_batches())).tolist()
                   for r in range(W)]
            assert len(set(map(len, ids))) == 1 and len(set(sum(ids, []))) == len(sum(ids, []))   # equal, disjoint
            data = list(range(n))
            dl = [len(DataLoader(data, batch_size=B, sampler=DistributedSampler(data, num_replicas=W, rank=r, shuffle=True,
                                                                                drop_last=True))) for r in range(W)]
            assert len(set(dl)) == 1


class _Graphs:
    def __init__(self, x):
        self.ndata = {"x": x}

    def to(self, device):
        return self


class _FakeModel(torch.nn.Module):
    """Stands in for the fine-tuning / domain-adaptation wrappers: sigmoid(x W) scores; records every per-batch value the
    loops accumulate."""

    def __init__(self):
        super().__init__()
        torch.manual_seed(0)
        self.w = torch.nn.Parameter(torch.randn(5, 3) * 0.3)
        self.bn = torch.nn.BatchNorm1d(3)
        self.seen = {"loss": [], "metric": [], "da": []}

    def forward(self, *a):
        x = a[1]
        if len(a) == 10:                                  # domain adaptation: (g, x, subgraphs, logMs, ..., batch_size)
            v = ((x @ self.w) ** 2).sum()
            self.seen["da"].append(float(v.detach()))
            return v
        return torch.sigmoid(self.bn(x @ self.w)), 0, 0, 0

    def loss(self, scores, targets):
        v = torch.nn.BCELoss()(scores, targets)
        self.seen["loss"].append(float(v.detach()))
        return v

    def BCEWithLogitsLoss(self, scores, targets):
        v = torch.nn.BCEWithLogitsLoss()(scores, targets)
        self.seen["metric"].append(float(v.detach()))
        return v


def _batches(seed, n):
    g = torch.Generator().manual_seed(seed)
    return [(_Graphs(torch.randn(4 + i, 5, generator=g)), (torch.rand(4 + i, 3, generator=g) < 0.3).float(), None, None)
            for i in range(n)]


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    torch.set_num_threads(1)
    from scgib_b200 import dist as sdist
    from scgib_b200.optim import AllReduceAdam
    import train_pep_func as tpf
    sdist.init_from_env("gloo")
    tpf.khop_ego_batch = lambda g, k: None
    out = {}

    # BatchNorm buffers as views into one flat tensor, as the GIN engine's bn_running holds them
    m = torch.nn.Sequential(torch.nn.BatchNorm1d(4), torch.nn.Linear(4, 4), torch.nn.BatchNorm1d(6))
    flat = torch.zeros(2, 2, 6)
    for i, bn in enumerate((m[0], m[2])):
        n = bn.num_features
        flat[i, 0, :n] = torch.arange(n) + 10.0 * rank
        flat[i, 1, :n] = 1.0 + rank * torch.arange(n)
        bn.running_mean.data = flat[i, 0, :n]
        bn.running_var.data = flat[i, 1, :n]
    ptrs = [(bn.running_mean.data_ptr(), bn.running_var.data_ptr()) for bn in (m[0], m[2])]
    before = [t.clone() for bn in (m[0], m[2]) for t in (bn.running_mean, bn.running_var)]
    sdist.average_bn_buffers_(m)
    out["bn_before"] = [t.numpy() for t in before]
    out["bn_after"] = [t.clone().numpy() for bn in (m[0], m[2]) for t in (bn.running_mean, bn.running_var)]
    out["bn_alias"] = ptrs == [(bn.running_mean.data_ptr(), bn.running_var.data_ptr()) for bn in (m[0], m[2])] and \
        m[0].running_mean.data_ptr() == flat[0, 0].data_ptr() and m[2].running_var.data_ptr() == flat[1, 1].data_ptr()
    out["bn_flat"] = flat.numpy()

    args = types.SimpleNamespace(k_transition=1)
    model = _FakeModel()
    # evaluation: 5 batches round robin -> rank 0 holds 3, rank 1 holds 2
    everything = _batches(1, 5)
    mine = [everything[lo] for lo, _ in sdist.round_robin_batches(5, 1, rank, world)]
    loss, ap = tpf.evaluate_network(args, model, None, "cpu", mine, 0, 1)
    out["eval"] = (loss, float(ap))
    out["eval_seen"] = dict(loss=list(model.seen["loss"]), metric=list(model.seen["metric"]))
    # an empty shard (fewer batches than ranks) still takes part in the reduction
    model.seen = {"loss": [], "metric": [], "da": []}
    mine = [everything[lo] for lo, _ in sdist.round_robin_batches(1, 1, rank, world)]
    loss, ap = tpf.evaluate_network(args, model, None, "cpu", mine, 0, 1)
    out["eval1"] = (loss, float(ap))
    out["eval1_seen"] = dict(loss=list(model.seen["loss"]), metric=list(model.seen["metric"]))
    # one training epoch (4 batches per rank, different data per rank) and one domain-adaptation epoch
    model.seen = {"loss": [], "metric": [], "da": []}
    opt = AllReduceAdam(model.parameters(), lr=1e-2)
    loss, ap, _ = tpf.train_epoch_graph_classification(args, model, opt, "cpu", _batches(10 + rank, 4), 1, 4)
    out["train"] = (loss, float(ap))
    out["train_seen"] = dict(loss=list(model.seen["loss"]), metric=list(model.seen["metric"]))
    out["w"] = model.w.detach().clone().numpy()
    model.seen = {"loss": [], "metric": [], "da": []}
    da_loss, da_rec = tpf.train_epoch_domainadaptation(model, args, opt, "cpu", _batches(20 + rank, 3), 1, 1, 4)
    out["da"] = (da_loss, float(da_rec))
    out["da_seen"] = list(model.seen["da"])

    # early stopping on per-rank losses that differ: each rank decides from the reduced loss
    local = {0: [5.0, 4.0, 4.5, 4.6, 4.7], 1: [5.0, 4.9, 3.0, 3.5, 3.6]}[rank]
    best_loss, best_epoch, decisions = 1e8, 0, []
    for epoch, l in enumerate(local, 1):
        l = sdist.mean_over_ranks([l], 1)[0]
        if best_loss >= l:
            best_epoch, best_loss = epoch, l
        decisions.append((best_epoch, epoch - best_epoch > 1))
    out["decisions"] = decisions
    q.put((rank, out))
    dist.barrier()
    dist.destroy_process_group()


@pytest.fixture(scope="module")
def two_ranks():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=240) for _ in range(world))
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    return res


@pytest.mark.timeout(300)
def test_bn_buffer_average_in_place(two_ranks):
    r0, r1 = two_ranks[0], two_ranks[1]
    for a, b, x0, x1 in zip(r0["bn_after"], r1["bn_after"], r0["bn_before"], r1["bn_before"]):
        assert np.array_equal(a, b)
        assert np.allclose(a, (x0 + x1) / 2, rtol=0, atol=1e-6)
        assert not np.array_equal(x0, x1)
    assert r0["bn_alias"] and r1["bn_alias"]
    assert np.array_equal(r0["bn_flat"][0, 0, :4], r0["bn_after"][0])       # the averaged values landed in the flat base
    assert np.array_equal(r0["bn_flat"][1, 1, :6], r0["bn_after"][3])


def _mean(xs):
    return sum(xs) / len(xs)


@pytest.mark.timeout(300)
def test_evaluation_reduction_over_the_union_of_batches(two_ranks):
    for key, seen in (("eval", "eval_seen"), ("eval1", "eval1_seen")):
        loss = two_ranks[0][seen]["loss"] + two_ranks[1][seen]["loss"]
        metric = two_ranks[0][seen]["metric"] + two_ranks[1][seen]["metric"]
        (l0, m0), (l1, m1) = two_ranks[0][key], two_ranks[1][key]
        assert l0 == l1 and float(m0) == float(m1)
        assert abs(l0 - _mean(loss)) <= 1e-6 * abs(_mean(loss))
        assert abs(float(m0) - _mean(metric)) <= 1e-6 * abs(_mean(metric))
    assert len(two_ranks[0]["eval_seen"]["loss"]) == 3 and len(two_ranks[1]["eval_seen"]["loss"]) == 2
    assert len(two_ranks[1]["eval1_seen"]["loss"]) == 0


@pytest.mark.timeout(300)
def test_epoch_reductions_over_the_union_of_batches(two_ranks):
    r0, r1 = two_ranks[0], two_ranks[1]
    assert r0["train"] == r1["train"] and r0["da"] == r1["da"]
    loss = [v / 2 for v in r0["train_seen"]["loss"] + r1["train_seen"]["loss"]]           # the reference's loss / 2
    metric = r0["train_seen"]["metric"] + r1["train_seen"]["metric"]
    assert abs(r0["train"][0] - _mean(loss)) <= 1e-6 * _mean(loss)
    assert abs(r0["train"][1] - _mean(metric)) <= 1e-6 * _mean(metric)
    da = r0["da_seen"] + r1["da_seen"]
    assert abs(r0["da"][0] - _mean(da)) <= 1e-6 * _mean(da) and abs(r0["da"][1] - _mean(da)) <= 1e-6 * _mean(da)
    assert r0["train_seen"]["loss"] != r1["train_seen"]["loss"]
    assert np.array_equal(r0["w"], r1["w"])                               # AllReduceAdam kept the replicas identical


@pytest.mark.timeout(300)
def test_early_stopping_decision_agrees_across_ranks(two_ranks):
    assert two_ranks[0]["decisions"] == two_ranks[1]["decisions"]
    # on their own local losses the ranks would have disagreed (rank 0 stops improving at epoch 2, rank 1 at epoch 3)
    assert two_ranks[0]["decisions"][-1] == (3, True)
