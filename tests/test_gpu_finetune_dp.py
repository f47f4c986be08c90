"""Data-parallel fine-tuning and domain adaptation on two GPUs: replicas stay bit-identical, equal bit for bit to a
single-process emulation of both ranks (tests/gpu_finetune_dp_worker.py), evaluation reduced over whole-batch shards, and
the exp_pep_func_5.py CLI under torchrun."""
import json
import os
import re
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _torchrun(port, script_args, cwd, timeout=900):
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", str(port)] + script_args, capture_output=True, text=True, timeout=timeout,
                       cwd=cwd)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return r.stdout


two_gpus = pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs on one node")


@pytest.mark.parametrize("backend", [pytest.param("nccl", marks=two_gpus), "gloo"])
@pytest.mark.parametrize("mode,encoder,dtype,port", [("ft", "GIN", "fp32", 29571), ("ft", "GIN", "bf16", 29572),
                                                     ("ft", "GraphSAGE", "fp32", 29573), ("da", "GIN", "fp32", 29574)])
def test_two_ranks_match_single_process_emulation(mode, encoder, dtype, port, backend, tmp_path):
    """nccl: one GPU per rank; gloo: both ranks on cuda:0, which runs the same check on a one-GPU machine."""
    batches = 6 if mode == "ft" else 2                      # three optimizer steps / two optimizer steps per rank
    out = _torchrun(port + (10 if backend == "gloo" else 0),
                    [os.path.join(ROOT, "tests", "gpu_finetune_dp_worker.py"), "--mode", mode, "--encoder", encoder,
                     "--dtype", dtype, "--batches", str(batches), "--backend", backend, "--out", str(tmp_path)], ROOT)
    res = json.loads(out.strip().splitlines()[-1].split("RESULT ", 1)[1])
    assert res["world"] == 2
    assert res["ranks_differ"] == []                        # parameters and BatchNorm buffers bit-identical on both ranks
    assert res["emu_differs"] == [], res["emu_max_diff"]    # ... and to the single-process emulation
    assert abs(res["epoch"][0] - res["emu_epoch_loss"]) <= 1e-6 * abs(res["emu_epoch_loss"])
    if mode == "ft":
        for got, ref in zip(res["eval"], res["emu_eval"]):
            assert abs(got - ref) <= 1e-6 * abs(ref), (res["eval"], res["emu_eval"])


@two_gpus
def test_cli_pretrain_adapt_finetune_two_ranks(tmp_path):
    """torchrun exp_pep_func_5.py --pretrained_mode 1, then --domain_adapt 1 with fine-tuning: each checkpoint is written
    once (rank 0), only rank 0 prints epoch lines, and the replicas end identical."""
    out_dir = str(tmp_path / "outputs") + "/"
    common = [os.path.join(ROOT, "exp_pep_func_5.py"), "--batch_size", "32", "--synthetic", "256", "--output_path", out_dir,
              "--num_layers", "4"]
    pre = _torchrun(29575, common + ["--pretrained_mode", "1", "--pt_epoches", "3"], str(tmp_path))
    ft = _torchrun(29576, common + ["--pretrained_ds", "Peptides-func", "--domain_adapt", "1", "--adapt_epoches", "3",
                                    "--ft_epoches", "3"], str(tmp_path))
    files = ["Peptides-func_GIN_64_4_1.pt", "Peptides-func_GIN_64_4_1_Peptides-func.pt"]
    assert sorted(os.listdir(tmp_path / "outputs")) == files
    for text, f in ((pre, files[0]), (ft, files[1])):
        assert text.count("[I] saved %s%s" % (out_dir, f)) == 1
    assert len(re.findall(r"^Epoch:\d", pre, re.M)) == 2                   # pre-training: epochs 1, 2 on rank 0 only
    assert len(re.findall(r"^Epoch:\d", ft, re.M)) == 2                    # domain adaptation
    assert len(re.findall(r"^Epoch: \d", ft, re.M)) == 2                   # fine-tuning
    sums = {}
    for rank, what, val in re.findall(r"rank (\d) parameter checksum (\S+) (\S+)", pre + ft):
        sums.setdefault(what, {})[rank] = val
    assert sorted(sums) == sorted(files + ["fine-tuned"])
    for what, per_rank in sums.items():
        assert sorted(per_rank) == ["0", "1"] and per_rank["0"] == per_rank["1"], (what, per_rank)
