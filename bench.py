#!/usr/bin/env python
"""bench.py - S-CGIB pre-training throughput (graphs/s) on N B200s + roofline + CPU baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--k 1] [--impl reference] [--dump-outputs DIR]

Metric (BASELINE.json): pre-training graphs/s, PCQM4Mv2-shape synthetic molecules, GIN-4x64 (models.py:57-58),
k_transition=1, fp32.  A "step" is one full pre-training step on one mini-batch per GPU:
on-GPU k-hop ego-net extraction + noise draw + forward + backward + gradient all-reduce (N>1) + Adam.

  value : steps timed with CUDA events, batches already resident in HBM.
  e2e   : the same step through the public API with HOST (pinned) batches: H2D of the batch arrays and
          D2H of the losses inside the timed region.
  --impl reference : the reference's CPU path (oracle restatement, loop-for-loop; DGL cannot be installed
          here) on the host cores, B=128 mini-batches (the reference's default --batch_size).
  --dump-outputs DIR : after the timed steps, what the timed path computed in its last step (losses or scores, parameters
          after the optimiser step, gradients, BatchNorm running statistics) as DIR/<name>.npy in float32.  Inputs, weights
          and noise are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "pretrain graphs/s (PCQM4Mv2-shape GIN-4x64 k=1)"
UNIT = "graphs/s"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def dump_outputs(out_dir, arrays):
    """--dump-outputs: one DIR/<name>.npy (float32) per device tensor."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


class NvmlClockSampler:
    """SM clock + throttle reasons read through NVML (nvidia_ml_py) every 5 ms from a thread while the timed region
    runs: a 100-step timed region is ~0.25 s, too short for nvidia-smi's own start-up."""

    def __init__(self, torch_index):
        import pynvml
        self.nv = pynvml
        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(torch_index).uuid)
        try:
            self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
        except Exception:
            self.h = pynvml.nvmlDeviceGetHandleByUUID("GPU-" + uuid)
        self.sm, self.reasons, self.stop_flag = [], set(), False
        self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))

    def _loop(self):
        nv = self.nv
        bits = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self.stop_flag:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for n, b in bits.items():
                    if r & b:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        self.t = threading.Thread(target=self._loop, daemon=True)
        self.t.start()

    def stop(self):
        self.stop_flag = True
        self.t.join(timeout=1)
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.mx, "reasons": sorted(self.reasons),
                "samples": len(sm), "source": "nvml"}


def make_clock_sampler(torch_index, smi_index):
    try:
        return NvmlClockSampler(torch_index)
    except Exception:
        return ClockSampler(smi_index)


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [v.strip() for v in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------
# CPU baseline: the reference's path restated loop-for-loop (oracle), forward + backward + Adam
# ----------------------------------------------------------------------------------------------------
def cpu_reference_run(steps, warmup, batch=128, k=1, hidden=64):
    import numpy as np
    from oracle.graph_ref import ego_batch_ref, synth_batch
    from oracle.scgib_oracle import OracleMainmodel, normalize_rows, oracle_train_step, tgraph_from_ego, tgraph_from_ref
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    model = OracleMainmodel(9, hidden)
    opt = torch.optim.Adam(model.parameters(), lr=1e-4, weight_decay=5e-5)
    data = []
    for s in range(2):
        g = synth_batch(100 + s, batch)
        e = ego_batch_ref(g, k)      # the reference loads pre-extracted ego-nets from disk: not timed
        x = normalize_rows(torch.from_numpy(g.x))
        en = torch.from_numpy(e.ego_nodes.astype(np.int64))
        data.append((tgraph_from_ref(g), x, tgraph_from_ego(e), x[en]))
    for i in range(warmup):
        oracle_train_step(model, opt, *data[i % 2])
    if steps is None:                      # bounded sample: about 12 s of CPU work
        t0 = time.perf_counter()
        for i in range(3):
            oracle_train_step(model, opt, *data[i % 2])
        steps = max(10, min(400, int(12.0 / ((time.perf_counter() - t0) / 3))))
    t0 = time.perf_counter()
    for i in range(steps):
        oracle_train_step(model, opt, *data[i % 2])
    dt = time.perf_counter() - t0
    return {"value": batch * steps / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "sample": "%d steps of B=%d (reference default --batch_size), fwd+bwd+Adam, faithful per-graph loops + dense NxN "
                      "recon, %.1f s wall" % (steps, batch, dt)}, dt / steps * 1e3


def torch_gpu_reference_run(dev, k=1, hidden=64):
    """The "reference torch path on the same GPU" (north_star): the oracle's restatement of the reference run with plain
    torch on the B200 - `faithful` = what the reference really executes (per-graph Python loops, dense N x N recon) at its
    default batch 128; `vectorised` = a strong torch baseline the reference does not have (segment ops + Gram identity)
    at B = 4096.  Forward + backward + torch.optim.Adam, CUDA events, ego-nets prepared outside the timed region (the
    reference loads them from disk)."""
    import numpy as np
    from oracle.graph_ref import ego_batch_ref, synth_batch_fast
    from oracle.scgib_oracle import OracleMainmodel, normalize_rows, tgraph_from_ego, tgraph_from_ref
    out = {}
    for name, B, steps in (("faithful_b128", 128, 10), ("vectorised_b4096", 4096, 20)):
        torch.manual_seed(0)
        model = OracleMainmodel(9, hidden).to(dev)
        opt = torch.optim.Adam(model.parameters(), lr=1e-4, weight_decay=5e-5)
        g = synth_batch_fast(100, B)
        e = ego_batch_ref(g, k)
        x = normalize_rows(torch.from_numpy(g.x)).to(dev)
        en = torch.from_numpy(e.ego_nodes.astype(np.int64)).to(dev)
        tg, te = tgraph_from_ref(g).to(dev), tgraph_from_ego(e).to(dev)
        xs = x[en]

        def step():
            opt.zero_grad()
            if name.startswith("faithful"):
                o = model.forward_faithful(tg, x, te, xs)
            else:
                o = model.forward_vectorised(tg, x, te, en, torch.rand(x.shape[0], device=dev), torch.rand(x.shape[0], hidden, device=dev))
            loss = o["KL"] + o["recon"] + o["contrastive"]
            loss.backward()
            opt.step()
            return loss.detach().item()          # the reference reads the loss every step (exp_pretraining.py:324)
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out[name] = {"value": B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "batch": B, "steps": steps}
        del model, opt
        torch.cuda.empty_cache()
    out["note"] = ("plain PyTorch (the oracle's restatement of the reference's math; DGL itself is not installable here) on the "
                   "same B200: the north_star's 'reference torch path on the same GPU'")
    return out


def run_reference(args, rank, emit):
    if rank != 0:
        return
    base, ms = cpu_reference_run(args.steps, args.warmup, batch=128, k=args.k, hidden=args.dims)
    line = {"metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": "S-CGIB pre-training step GIN-4x64 k=%d, PCQM4Mv2-shape synthetic molecules, CPU sample: "
                                   "mini-batches of 128 graphs" % args.k},
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ----------------------------------------------------------------------------------------------------
# Secondary workload (BASELINE configs[4], SURVEY 8 a20): fine-tuning step of Mainmodel_finetuning
# ----------------------------------------------------------------------------------------------------
def cpu_finetune_run(shape, batch, k=1, budget_s=10.0, hidden=64):
    import numpy as np
    from oracle.graph_ref import ego_batch_ref, synth_batch
    from oracle.scgib_oracle import OracleFinetune, OracleMainmodel, normalize_rows, tgraph_from_ego, tgraph_from_ref
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(0)
    model = OracleFinetune(OracleMainmodel(9, hidden), 9, hidden, num_classes=10)
    opt = torch.optim.Adam([p for p in model.parameters() if p.requires_grad], lr=1e-4)
    g = synth_batch(100, batch, shape)
    e = ego_batch_ref(g, k)
    x = normalize_rows(torch.from_numpy(g.x))
    en = torch.from_numpy(e.ego_nodes.astype(np.int64))
    tg, te, xs = tgraph_from_ref(g), tgraph_from_ego(e), x[en]
    y = (torch.rand(batch, 10) < 0.1).float()

    def step():
        opt.zero_grad()
        out = model(tg, x, te, xs)
        (torch.nn.functional.binary_cross_entropy(out["scores"], y) / 2).backward()
        opt.step()
    step()
    t0 = time.perf_counter()
    n = 0
    while time.perf_counter() - t0 < budget_s:
        step(); n += 1
    dt = time.perf_counter() - t0
    return {"value": batch * n / dt, "unit": "graphs/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": "%d steps of B=%d %s-shape graphs, Mainmodel_finetuning fwd+bwd+Adam (per-graph loops), %.1f s wall" % (n, batch, shape, dt)}


def run_finetune(args, emit):
    """graphs/s of one fine-tuning step (features forward, Set2Set + predict head, BCE gradient, head backward, feature
    backward, Adam on both flat buffers) on one GPU; hidden = 64 (the reference default --dims)."""
    from scgib_b200 import _lib
    from scgib_b200.engine import FinetuneHead, PretrainEngine
    from scgib_b200.synth import synth_batch
    dev = torch.device("cuda", 0)
    lib = _lib.load()
    H, es = args.dims, (2 if args.dtype == "bf16" else 4)
    eng = PretrainEngine(9, gin_layers=4, hidden=H, device=dev, seed=0, dtype=args.dtype)
    head = FinetuneHead(H, 10, n_iters=2, sigmoid=True, device=dev)
    head.params.copy_((torch.rand(head.total, generator=torch.Generator().manual_seed(1)) * 0.25 - 0.125).to(dev))
    hm, hv = torch.zeros_like(head.params), torch.zeros_like(head.params)
    B = args.batch
    nb = 3
    host = [synth_batch(50 + i, B, args.shape).pin_memory() for i in range(nb)]
    resident = [h.to(dev) for h in host]
    targets = (torch.rand(B, 10, generator=torch.Generator().manual_seed(2)) < 0.1).float().to(dev)
    state = {"n": 0}

    def run_steps(src, steps, read):
        handle = eng.prefetch_batch(src[0], args.k)
        for i in range(steps):
            b = eng.wait_batch(handle)
            Z = eng.forward_features(b)
            scores = head.forward(Z, b.g.graph_ptr)
            g_s = (scores - targets) / (scores * (1 - scores)).clamp_min(1e-12) / (2.0 * B * 10)   # d(BCE/2)/d scores
            gZ = head.backward(g_s)
            eng.extract_backward(gZ)
            eng.adam_step(lr=1e-4, weight_decay=0.0)
            state["n"] += 1
            st = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(lib.scgib_adam_step_f32(_lib.ptr(head.params), _lib.ptr(head.grads), _lib.ptr(hm), _lib.ptr(hv),
                                               head.total, state["n"], 1e-4, 0.9, 0.999, 1e-8, 0.0, 1.0, st), "adam")
            slot = getattr(b, "_slot", None)
            if slot is not None:
                slot["done"] = torch.cuda.Event(); slot["done"].record(torch.cuda.current_stream(dev))
            if i + 1 < steps:
                handle = eng.prefetch_batch(src[(i + 1) % nb], args.k)
            if read:
                state["scores"] = scores.cpu()
        state["b"], state["last_scores"] = b, scores

    def timed(src, steps, read):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); run_steps(src, steps, read); e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    run_steps(resident, max(args.warmup, 3), False)
    sampler = make_clock_sampler(0, 0)
    sampler.start()
    ms = timed(resident, args.steps, False)
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"scores": state["last_scores"], "params": eng.params, "grads": eng.grads,
                                         "head_params": head.params, "head_grads": head.grads})
    run_steps(host, 3, True)
    ms_e2e = timed(host, args.steps, True)
    prof = {}
    lib.scgib_profile_enable(1)
    run_steps(resident, 1, False)
    torch.cuda.synchronize()
    name, t = ctypes.c_char_p(), ctypes.c_float()
    for j in range(lib.scgib_profile_count()):
        lib.scgib_profile_get(j, ctypes.byref(name), ctypes.byref(t))
        cur = prof.setdefault(name.value.decode(), [0.0, 0]); cur[0] += t.value; cur[1] += 1
    nlaunch = lib.scgib_profile_count()
    lib.scgib_profile_enable(0)
    b = state["b"]
    hbm, peak_src = peaks()
    # roofline unit = ONE GIN layer of both encoders (layer average); a layer's backward = gin_bwd_pre + gin_bwd_main
    fam = {}
    for k_, v in prof.items():
        f = "gin_bwd (pre + main)" if k_.startswith(("gin_bwd_pre", "gin_bwd_main")) else k_
        cur = fam.setdefault(f, [0.0, []]); cur[0] += v[0]; cur[1].append(k_)
    dom = max(fam, key=lambda k_: fam[k_][0])
    V, D = b.N + b.Ns, b.E + b.Es
    fwd_layer = sum(V * (di + H) * es + 4 * (V + 1 + D) for di in (32, H, H, H)) / 4.0
    if dom.startswith("gin_bwd"):
        abytes, unit_ms = 2.0 * fwd_layer, fam[dom][0] / 4.0
    elif dom.startswith("gin_fwd"):
        abytes, unit_ms = fwd_layer, fam[dom][0] / 4.0
    else:
        abytes, unit_ms = 3 * b.N * H * 4, prof[dom][0] / prof[dom][1]
    achieved = abytes / (unit_ms * 1e-3) / 1e9
    step_bytes = b.algorithmic_bytes(gin_layers=4, s=es, hidden=H) - 3 * (b.N * H * es + 4 * (b.N + 1 + b.E))   # no recon / contrastive in fine-tuning
    h2d = sum(t_.numel() * t_.element_size() for t_ in (host[0].graph_ptr, host[0].indptr, host[0].indices, host[0].ndata["x"]))
    line = {"metric": "finetune graphs/s (%s-shape GIN-4x%d k=%d, Set2Set readout)" % (args.shape, H, args.k),
            "value": B * args.steps / (ms * 1e-3), "unit": "graphs/s", "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if args.dtype == "bf16" else "f32", "data": "synthetic",
            "config": {"workload": "Mainmodel_finetuning step (ego extraction + features fwd + Set2Set/predict head + BCE + bwd + Adam), "
                                   "GIN-4x%d (--dims %d; BASELINE configs[4] = GIN-5x128 in the paper's layer count), k=%d, batch %d %s-shape graphs"
                                   % (H, H, args.k, B, args.shape),
                       "nodes": b.N, "edges": b.E, "ego_rows": b.Ns, "ego_edges": b.Es,
                       "l2": "no flush: per-step working set exceeds the 126 MB L2"},
            "clocks": clocks,
            "e2e": {"value": B * args.steps / (ms_e2e * 1e-3), "unit": "graphs/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": B * 10 * 4, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": (nlaunch + 8) * args.steps,
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": hbm, "unit": "GB/s", "frac": achieved / hbm,
                         "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_unit": abytes, "unit_ms": unit_ms,
                         "members": fam[dom][1], "note": "unit = one GIN layer of both encoders (layer average); backward = pre + main"},
            "step_roofline": {"algorithmic_bytes_per_step": step_bytes, "achieved": step_bytes / (ms / args.steps * 1e-3) / 1e9,
                              "peak": hbm, "unit": "GB/s", "frac": step_bytes / (ms / args.steps * 1e-3) / 1e9 / hbm},
            "kernels": {k_: {"ms_per_step": v[0], "launches_per_step": v[1]} for k_, v in prof.items()}}
    if not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_finetune_run(args.shape, 32 if args.shape == "peptides" else 128, args.k, hidden=H)
    emit(line)


# ----------------------------------------------------------------------------------------------------
def run_encoder_variant(args, emit):
    """--encoder GraphSAGE / GCN (reference models.py:75-104): graphs/s of the pre-training step through the drop-in module
    (models.Mainmodel composed from the operator kernels, s-cgib_b200/encoders.py) with torch.optim.Adam over the module's
    parameters - the loop body of exp_pretraining.train_epoch_pre_training.  One GPU; `value` from batches resident in HBM,
    `e2e` from pinned host batches with the per-step loss read."""
    import types
    import torch.nn.functional as F
    import models as dropin_models
    from scgib_b200.graph import khop_ego_batch
    from scgib_b200.synth import synth_batch
    dev = torch.device("cuda", 0)
    H, B = args.dims, args.batch
    ns = types.SimpleNamespace(recons_type="adj", useAtt=1, readout_f="sum", d_transfer=32, device=str(dev), batch_size=B,
                               k_transition=args.k, dtype="fp32")
    torch.manual_seed(0)
    dm = dropin_models.Mainmodel(ns, 9, H, 4, 4, args.k, args.encoder).to(dev)
    dm.train()
    opt = torch.optim.Adam(dm.parameters(), lr=1e-4, weight_decay=5e-5)      # exp_pretraining.py:86
    nb = 4
    host = [synth_batch(1000 + i, B).pin_memory() for i in range(nb)]
    resident = [h.to(dev) for h in host]
    state = {}

    def run_steps(src, steps, read):
        for i in range(steps):
            bg = src[i % nb].to(dev, non_blocking=True)
            bx = F.normalize(bg.ndata["x"].float())
            opt.zero_grad()
            ego = khop_ego_batch(bg, args.k)
            _, kl, con, rec = dm.forward(bg, bx, ego, None, None, 1, None, 2, dev, B)
            loss = kl + rec + con
            loss.backward()
            opt.step()
            if read:
                state["loss"] = loss.detach().item()
        state["last_loss"] = loss
        state["shape"] = (bg.num_nodes(), bg.num_edges(), int(ego.sub_indptr.numel() - 1), int(ego.sub_indices.numel()))

    def timed(src, steps, read):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); run_steps(src, steps, read); e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    run_steps(resident, max(args.warmup, 3), False)
    sampler = make_clock_sampler(0, 0)
    sampler.start()
    ms = timed(resident, args.steps, False)
    clocks = sampler.stop()
    if args.dump_outputs:
        flat = lambda ts: torch.cat([t.detach().float().reshape(-1) for t in ts])
        dump_outputs(args.dump_outputs, {
            "loss": state["last_loss"].reshape(1),
            "params": flat(dm.parameters()),
            "grads": flat(p.grad if p.grad is not None else torch.zeros_like(p) for p in dm.parameters()),
            "bn_running": flat(v for n, v in dm.state_dict().items() if n.endswith(("running_mean", "running_var")))})
    run_steps(host, 3, True)
    ms_e2e = timed(host, args.steps, True)
    N, E, Ns, Es = state["shape"]
    h2d = sum(t_.numel() * t_.element_size() for t_ in (host[0].graph_ptr, host[0].indptr, host[0].indices, host[0].ndata["x"]))
    launches = {"GraphSAGE": 2 * (3 + 3 + 6 * 2 + 9), "GCN": 2 * (3 + 3 + 6 + 6)}[args.encoder] + 24
    line = {"metric": "pretrain graphs/s (PCQM4Mv2-shape %s x%d k=%d, operator-composed step)" % (args.encoder, H, args.k),
            "value": B * args.steps / (ms * 1e-3), "unit": "graphs/s", "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": "S-CGIB pre-training step with --encoder %s (models.py:75-104): ego extraction + forward + backward + "
                                   "torch Adam through models.Mainmodel, FP32 FFMA operator kernels, batch %d synthetic PCQM4Mv2-shape "
                                   "graphs, k_transition=%d" % (args.encoder, B, args.k),
                       "nodes": N, "edges": E, "ego_rows": Ns, "ego_edges": Es,
                       "l2": "no flush: per-step working set exceeds the 126 MB L2"},
            "clocks": clocks,
            "e2e": {"value": B * args.steps / (ms_e2e * 1e-3), "unit": "graphs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches * args.steps}
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--batch", type=int, default=4096, help="graphs per GPU per step")
    ap.add_argument("--k", type=int, default=1)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="pretrain", choices=["pretrain", "finetune"],
                    help="pretrain = the headline metric (default); finetune = Mainmodel_finetuning step (1 GPU)")
    ap.add_argument("--recons_type", default="adj", choices=["adj", "logM"],
                    help="adj = the reference default (the headline); logM = k-step log transition matrices (models.py:770-782)")
    ap.add_argument("--shape", default="pcqm", choices=["pcqm", "peptides"], help="synthetic molecule shape (finetune workload)")
    ap.add_argument("--dims", type=int, default=64, choices=[64, 128], help="hidden width (--dims of the reference CLI); 128 = BASELINE configs[4]")
    ap.add_argument("--dtype", default="fp32", choices=["fp32", "bf16"],
                    help="fp32 = the headline (reference precision); bf16 = bf16 activations + single-pass bf16 tensor-core MLPs in the GIN encoders")
    ap.add_argument("--encoder", default="GIN", choices=["GIN", "GraphSAGE", "GCN"],
                    help="GIN = the headline (fused tensor-core engine); GraphSAGE / GCN = the operator-composed variants (1 GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed path computed in its last step to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; --impl reference has none")
    # stdout carries exactly ONE JSON line: anything libraries print (e.g. the NCCL version banner) goes to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, emit)
        return
    if args.warmup < 3:
        args.warmup = 3
    if args.encoder != "GIN":
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (the hot path has no CPU fallback)")
        if rank == 0:
            run_encoder_variant(args, emit)
        return
    if args.workload == "finetune":
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (the hot path has no CPU fallback)")
        if rank == 0:
            run_finetune(args, emit)
        return

    import torch.distributed as dist
    from scgib_b200 import _lib
    from scgib_b200.engine import PretrainEngine
    from scgib_b200.synth import synth_batch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the hot path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    bf16 = args.dtype == "bf16"
    H = args.dims
    eng = PretrainEngine(9, gin_layers=4, hidden=H, device=dev, seed=0, dtype=args.dtype)     # same seed on every rank: replicas start equal
    eng._noise_gen.manual_seed(1234 + rank)
    if args.recons_type == "logM":
        eng.recon_logm_steps = args.k
    fused_dp = world > 1 and os.environ.get("SCGIB_DP", "peer") == "peer"
    if fused_dp:
        eng.enable_peer_allreduce()      # gradient all-reduce fused with Adam over NVLink peer memory (no NCCL per step)

    n_batches = 4
    host = [synth_batch(1000 * rank + i, args.batch).pin_memory() for i in range(n_batches)]
    resident = [h.to(dev) for h in host]
    torch.cuda.synchronize()

    # Pipelined input: the next batch's H2D + ego-net extraction run on a side stream during the current step
    # (engine.prefetch_batch); every step still extracts the ego-nets of its own batch on the GPU.
    state = {}

    # D2H of every step's {KL, contrastive, recon, total}: an async copy into pinned memory right behind the step, read on
    # the host one step later (after the next step has been launched), so the GPU never drains for the read
    loss_host = torch.empty(2, 4).pin_memory()
    loss_ev = [torch.cuda.Event(), torch.cuda.Event()]

    def read_loss_async(i, losses):
        loss_host[i & 1].copy_(losses, non_blocking=True)
        loss_ev[i & 1].record()
        if i > 0:
            loss_ev[(i - 1) & 1].synchronize()
            state["loss"] = loss_host[(i - 1) & 1].clone()

    def read_loss_last(steps):
        loss_ev[(steps - 1) & 1].synchronize()
        state["loss"] = loss_host[(steps - 1) & 1].clone()

    def run_steps(src, steps, read_loss):
        handle = eng.prefetch_batch(src[0], args.k)
        for i in range(steps):
            b = eng.wait_batch(handle)
            losses = eng.train_step(b, world_size=world)
            if read_loss:
                read_loss_async(i, losses)
            if i + 1 < steps:
                handle = eng.prefetch_batch(src[(i + 1) % n_batches], args.k)
        if read_loss:
            read_loss_last(steps)
        state["last"] = b

    def step_resident(steps):
        run_steps(resident, steps, False)

    def step_e2e(steps):
        run_steps(host, steps, True)     # H2D of graph_ptr/indptr/indices/x from pinned host memory every step

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn(steps)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    # third feed: the dataset resident in HBM, a step's input is its B molecule ids (GPU-side batch assembly)
    from scgib_b200.graph import DeviceDataset, batch as batch_graphs
    dataset = DeviceDataset.from_batched(batch_graphs(host), dev)
    gen = torch.Generator().manual_seed(77 + rank)
    id_lists = [torch.randperm(len(dataset), generator=gen)[:args.batch].to(torch.int32).pin_memory() for _ in range(8)]

    def step_ids(steps):
        handle = eng.prefetch_ids(dataset, id_lists[0], args.k)
        for i in range(steps):
            b = eng.wait_batch(handle)
            losses = eng.train_step(b, world_size=world)
            read_loss_async(i, losses)
            if i + 1 < steps:
                handle = eng.prefetch_ids(dataset, id_lists[(i + 1) % len(id_lists)], args.k)
        read_loss_last(steps)

    step_resident(args.warmup)
    sampler = make_clock_sampler(local_rank, torch.cuda.current_device() if "CUDA_VISIBLE_DEVICES" not in os.environ else local_rank)
    if rank == 0:
        sampler.start()
    ms = timed(step_resident, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:          # the e2e / dropin / profiling passes below keep training this engine
        dump_outputs(args.dump_outputs, {"losses": eng.losses, "params": eng.params, "grads": eng.grads,
                                         "bn_running": eng.bn_running})
    step_e2e(3)
    ms_e2e = timed(step_e2e, args.steps)
    step_ids(3)
    ms_ids = timed(step_ids, args.steps)

    # ---- the reference-facing drop-in surface: exp_pretraining.train_epoch_pre_training's loop body (reference
    #      exp_pretraining.py:300-324) on models.Mainmodel with torch.optim.Adam over the module parameters, host batches,
    #      one .item() per step - what a user of the reference gets by swapping the imports (rank 0 timing, N = 1 only)
    ms_dropin = None
    if world == 1:
        import types
        import torch.nn.functional as F
        import models as dropin_models
        from scgib_b200.graph import khop_ego_batch
        ns = types.SimpleNamespace(recons_type=args.recons_type, useAtt=1, readout_f="sum", d_transfer=32, device=str(dev),
                                   batch_size=args.batch, k_transition=args.k, dtype=args.dtype)
        torch.manual_seed(0)
        dm = dropin_models.Mainmodel(ns, 9, H, 4, 4, args.k, "GIN").to(dev)
        dm.train()
        from exp_pretraining import make_optimizer
        dopt = make_optimizer(dm, 1e-4)          # what the drop-in exp_pretraining.py builds: Adam(lr, wd 5e-5) as one flat kernel

        def step_dropin(steps):
            for i in range(steps):
                bg = host[i % n_batches].to(dev, non_blocking=True)
                bx = bg.ndata["x"].float()
                dopt.zero_grad()
                ego = khop_ego_batch(bg, args.k)
                bx = F.normalize(bx)
                _, kl, con, rec = dm.forward(bg, bx, ego, None, None, 1, None, 2, dev, args.batch)
                loss = kl + rec + con
                loss.backward()
                dopt.step()
                state["loss_item"] = loss.detach().item()

        step_dropin(3)
        ms_dropin = timed(step_dropin, args.steps)

    # ---- per-kernel timing pass (CUDA events on the launching stream around every launch of the library)
    prof = {}
    nlaunch = 0
    psteps = min(args.steps, 10)
    for i in range(psteps):
        b = eng.make_batch(resident[i % n_batches], args.k)
        lib.scgib_profile_enable(1)
        eng.train_step(b, world_size=world)
        torch.cuda.synchronize()
        n = lib.scgib_profile_count()
        nlaunch = n
        name, t = ctypes.c_char_p(), ctypes.c_float()
        for j in range(n):
            lib.scgib_profile_get(j, ctypes.byref(name), ctypes.byref(t))
            k_ = name.value.decode()
            cur = prof.setdefault(k_, [0.0, 0])
            cur[0] += t.value
            cur[1] += 1
        lib.scgib_profile_enable(0)
    kernels = {k_: {"ms_per_step": v[0] / psteps, "launches_per_step": v[1] // psteps,
                    "ms_per_launch": v[0] / v[1]} for k_, v in prof.items()}
    b = eng.make_batch(resident[0], args.k)
    es = 2 if bf16 else 4                 # bytes per activation element of the GIN encoders
    step_bytes = b.algorithmic_bytes(gin_layers=4, s=es, hidden=H)
    hbm, peak_src = peaks()
    # A GIN layer's backward is TWO launches here (gin_bwd_pre + gin_bwd_main): they are one roofline unit, so that the
    # SURVEY 8(d) layer-backward budget (2 x the layer's forward bytes) is counted ONCE (VERDICT r01)
    fam = {}
    for k_, v in kernels.items():
        f = "gin_bwd (pre + main)" if k_.startswith(("gin_bwd_pre", "gin_bwd_main")) else k_
        cur = fam.setdefault(f, {"ms_per_step": 0.0, "members": []})
        cur["ms_per_step"] += v["ms_per_step"]
        cur["members"].append(k_)
    dom = max(fam, key=lambda k_: fam[k_]["ms_per_step"])
    # algorithmic bytes of one layer of the dominant family (SURVEY.md 8d per-layer figures, both encoders' rows, averaged
    # over the 4 layers), and the time of that layer = the family's time per step / 4 layers
    V, D = b.N + b.Ns, b.E + b.Es
    per_layer = [(32, H), (H, H), (H, H), (H, H)]
    fwd_layer = sum(V * (di + d) * es + 4 * (V + 1 + D) for di, d in per_layer) / 4.0
    if dom.startswith("gin_bwd"):
        abytes, unit_ms = 2.0 * fwd_layer, fam[dom]["ms_per_step"] / 4.0
    elif dom.startswith("gin_fwd"):
        abytes, unit_ms = fwd_layer, fam[dom]["ms_per_step"] / 4.0
    elif dom.startswith("contrastive"):
        abytes, unit_ms = 4 * b.B * H * 4, kernels[dom]["ms_per_launch"]
    else:
        abytes, unit_ms = 3 * b.N * H * 4, kernels[dom]["ms_per_launch"]
    achieved = abytes / (unit_ms * 1e-3) / 1e9
    traffic = None                       # dram__bytes_read + write per unit, from the ncu capture of THIS build (profiles/)
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        traffic = tj.get(args.dtype, {}).get(dom, {}).get("dram_bytes_per_unit")
    except Exception:
        pass

    # the HBM-bound aggregation / pooling / segment kernels (north_star: >= 60 % of HBM peak is the target): algorithmic
    # bytes per launch (SURVEY 8d per-unit figures x this batch's sizes) / CUDA-event time per launch
    d4 = H * 4
    hbm_alg = {
        ("gin_bwd_pre_bf16.enc1+2" if bf16 else "gin_bwd_pre.enc1+2"): 3 * (b.N + b.Ns) * H * es + 4 * (b.N + b.Ns + 2 + b.E + b.Es),
        "ego_pool_fwd": (b.Ns + b.N) * d4 + 4 * (b.N + 1) + 4 * b.N,
        "graph_gate_fwd": 4 * b.N * d4 + 12 * b.N,
        "recon_bwd": 2 * b.N * d4 + 4 * (b.N + 1 + b.E),
        "input_proj_fwd": b.N * 9 * 4 + b.N * 32 * 4,
    }
    hbm_kernels = {k_: {"algorithmic_bytes_per_launch": v, "GB/s": v / (kernels[k_]["ms_per_launch"] * 1e-3) / 1e9,
                        "frac": v / (kernels[k_]["ms_per_launch"] * 1e-3) / 1e9 / hbm}
                   for k_, v in hbm_alg.items() if k_ in kernels}
    # next to the CUDA-event time (which carries ~4 us of launch + event latency per launch: a quarter of a 16 us kernel):
    # the same kernels' durations in the committed ncu launch list of this command (cold-cache, serialised), headline config only
    if not bf16 and args.batch == 4096 and args.k == 1 and H == 64 and args.recons_type == "adj":
        try:
            import csv
            ncu_names = {"gin_bwd_pre.enc1+2": "gin_bwd_pre_kernel", "ego_pool_fwd": "ego_pool_fwd", "graph_gate_fwd": "graph_gate_fwd_kernel",
                         "recon_bwd": "recon_bwd_kernel"}
            rows = list(csv.DictReader(open(os.path.join(ROOT, "profiles", "r02_ncu_launches_fp32_summary.csv"))))
            for k_, pat in ncu_names.items():
                hit = [r for r in rows if pat in r["kernel"]]
                if k_ in hbm_kernels and hit:
                    us = float(hit[0]["total_us"]) / int(hit[0]["launches"])
                    gbs = hbm_kernels[k_]["algorithmic_bytes_per_launch"] / (us * 1e-6) / 1e9
                    hbm_kernels[k_]["ncu"] = {"us_per_launch": us, "GB/s": gbs, "frac": gbs / hbm,
                                               "source": "profiles/r02_ncu_launches_fp32_summary.csv (launch list of this command)"}
        except Exception:
            pass

    if rank == 0:
        graphs = args.batch * world * args.steps
        h2d = sum(t.numel() * t.element_size() for t in (host[0].graph_ptr, host[0].indptr, host[0].indices, host[0].ndata["x"]))
        line = {
            "metric": METRIC, "value": graphs / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16" if bf16 else "f32", "data": "synthetic",
            "config": {"workload": "S-CGIB pre-training step (ego extraction + fwd + bwd + grad all-reduce + Adam), GIN-4x" + str(H) + " "
                                   "(= BASELINE's 'GIN-5x64': the published code's 5-layer GIN has 4 GINConv, SURVEY F4), "
                                   "k_transition=%d, batch %d synthetic PCQM4Mv2-shape graphs per GPU (BASELINE configs[1]%s)"
                                   % (args.k, args.batch, ", bf16 half: bf16 activations in the GIN encoders" if bf16 else ""),
                       "graphs_per_gpu": args.batch, "nodes": b.N, "edges": b.E, "ego_rows": b.Ns, "ego_edges": b.Es,
                       "parallelism": "dp%d" % world, "recons_type": args.recons_type,
                       "grad_exchange": ("fused peer-memory all-reduce + Adam kernel" if fused_dp else "NCCL all-reduce + Adam") if world > 1 else "none",
                       "l2": "no flush: per-step working set (workspace %.2f GB, 4 rotating batches) exceeds the 126 MB L2" % (eng._ws.numel() / 1e9)},
            "clocks": clocks,
            "e2e": {"value": graphs / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 16,
                    "ms_per_step": ms_e2e / args.steps},
            "e2e_resident_dataset": {"value": graphs / (ms_ids * 1e-3), "unit": UNIT, "h2d_bytes_per_step": args.batch * 4,
                                     "d2h_bytes_per_step": 16, "ms_per_step": ms_ids / args.steps,
                                     "note": "dataset shard (%d molecules, %.1f MB) resident in HBM; per step only the B molecule ids "
                                             "cross PCIe, the batch is assembled on the GPU (scgib_batch_assemble_*)"
                                             % (len(dataset), dataset.nbytes() / 1e6)},
            "e2e_dropin_module": None if ms_dropin is None else {
                "value": graphs / (ms_dropin * 1e-3), "unit": UNIT, "ms_per_step": ms_dropin / args.steps,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "note": "models.Mainmodel.forward + loss.backward() + optimizer.step() (scgib_b200.optim.FlatAdam, as the drop-in exp_pretraining.py builds it) + loss.item() per step, no "
                        "prefetch: the reference's own training loop (exp_pretraining.py:300-324) on the drop-in classes"},
            "gpu_launches": (nlaunch + 5) * args.steps,
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": hbm, "unit": "GB/s",
                         "frac": achieved / hbm, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_unit": abytes, "unit_ms": unit_ms, "members": fam[dom]["members"],
                         "note": "unit = ONE GIN layer of both encoders (layer average): forward = 1 launch, backward = "
                                 "gin_bwd_pre + gin_bwd_main (the SURVEY 8(d) layer-backward budget, 2 x forward bytes, is "
                                 "counted once over both launches); warp-specialised tcgen05 kernels, see DESIGN.md section 3"},
            "step_roofline": {"algorithmic_bytes_per_step": step_bytes, "achieved": step_bytes / (ms / args.steps * 1e-3) / 1e9,
                              "peak": hbm, "unit": "GB/s", "frac": step_bytes / (ms / args.steps * 1e-3) / 1e9 / hbm},
            "hbm_kernels": hbm_kernels,
            "kernels": kernels,
        }
        if world == 1 and not args.no_cpu_baseline:
            del eng, dm, dopt
            torch.cuda.empty_cache()
            line["torch_gpu_baseline"] = torch_gpu_reference_run(dev, k=args.k, hidden=H)
            line["cpu_baseline"], _ = cpu_reference_run(None, 3, batch=128, k=args.k, hidden=H)
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
