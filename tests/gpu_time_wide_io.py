"""Time the pre-training and fine-tuning steps over the raw feature width F and the head width C (measurement, no target):

    python tests/gpu_time_wide_io.py [--repo DIR] [--narrow-only]

Cases:
- GIN pre-training step (forward + backward + Adam of the fused engine), PCQM shape, B = 4096, k = 1, hidden 64, fp32 and
  bf16, at F in {9, 37, 89, 128}.  F = 9 uses the molecular features; wider F appends uniform random columns.  Each step
  also reports the device time of `fwd_prep`, which holds the input projection and the xagg side CTAs, and of
  `input_proj_bwd`, read from the library's profile counters.
- Fine-tuning step (features forward, Set2Set + predict head, BCE gradient, head and feature backward, Adam on both flat
  buffers), Peptides shape, B = 1024, hidden 128, at C in {10, 128, 617}.

Batches stay resident in HBM and their k-hop ego-nets are built once, outside the timed region.  Steps are timed with CUDA
events after warm-up.  ``--repo DIR`` imports the package of another checkout, for example the parent commit, and
``--narrow-only`` keeps the F = 9 / C = 10 rows, which every checkout can run.  One JSON line per measurement; the GPU name
and power limit are read in the same run."""
import argparse
import ctypes
import json
import os
import sys


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repo", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    ap.add_argument("--narrow-only", action="store_true")
    ap.add_argument("--tag", default="")
    a = ap.parse_args()
    sys.path.insert(0, os.path.abspath(a.repo))
    import torch
    from scgib_b200 import _lib
    from scgib_b200.engine import DeviceBatch, FinetuneHead, PretrainEngine
    from scgib_b200.graph import khop_ego_batch
    from scgib_b200.synth import synth_batch
    sys.path.insert(1, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from tests.gpu_time_composed_downstream import DEV, gpu_info, timed
    lib = _lib.load()
    info = dict(gpu_info(), tree=a.tag or os.path.basename(os.path.abspath(a.repo)))

    def profile(step, names):
        """device ms per step of the named library launches (profile counters, one step)"""
        step()
        torch.cuda.synchronize()
        lib.scgib_profile_enable(1)
        step()
        torch.cuda.synchronize()
        out = {}
        for i in range(lib.scgib_profile_count()):
            nm, ms = ctypes.c_char_p(), ctypes.c_float()
            if lib.scgib_profile_get(i, ctypes.byref(nm), ctypes.byref(ms)) == 0 and nm.value.decode() in names:
                out[nm.value.decode()] = round(out.get(nm.value.decode(), 0.0) + ms.value, 4)
        lib.scgib_profile_enable(0)
        return out

    B = 4096
    for F_ in ((9,) if a.narrow_only else (9, 37, 89, 128)):
        g = synth_batch(1, B, "pcqm").to(DEV)
        if F_ > 9:
            gen = torch.Generator(device=DEV).manual_seed(F_)
            g.ndata["x"] = torch.cat([g.ndata["x"], torch.rand(g.num_nodes(), F_ - 9, device=DEV, generator=gen)], 1).contiguous()
        b = DeviceBatch(g, khop_ego_batch(g, 1), g.ndata["x"])
        for dtype in ("fp32", "bf16"):
            eng = PretrainEngine(F_, gin_layers=4, hidden=64, device=DEV, seed=0, dtype=dtype)
            step = lambda: eng.train_step(b)
            runs = [timed(step, 3, 30) for _ in range(2)]
            ms = min(runs)
            print(json.dumps(dict(case="pretrain_step", in_dim=F_, dtype=dtype, batch=B, N=b.N, Ns=int(b.ego.ego_nodes.numel()),
                                  ms_per_step=round(ms, 3), runs_ms=[round(v, 3) for v in runs], graphs_per_s=round(B / ms * 1e3),
                                  kernels_ms=profile(step, ("fwd_prep", "input_proj_bwd")), **info)), flush=True)
            del eng

    B, H = 1024, 128
    g = synth_batch(2, B, "peptides").to(DEV)
    b = DeviceBatch(g, khop_ego_batch(g, 1), g.ndata["x"])
    for C in ((10,) if a.narrow_only else (10, 128, 617)):
        eng = PretrainEngine(9, gin_layers=4, hidden=H, device=DEV, seed=0)
        head = FinetuneHead(H, C, n_iters=2, sigmoid=True, device=DEV)
        head.params.copy_((torch.rand(head.total, generator=torch.Generator().manual_seed(1)) * 0.25 - 0.125).to(DEV))
        hm, hv = torch.zeros_like(head.params), torch.zeros_like(head.params)
        targets = (torch.rand(B, C, generator=torch.Generator().manual_seed(2)) < 0.1).float().to(DEV)
        n = [0]

        def step():
            Z = eng.forward_features(b)
            scores = head.forward(Z, g.graph_ptr)
            g_s = (scores - targets) / (scores * (1 - scores)).clamp_min(1e-12) / (2.0 * B * C)
            eng.extract_backward(head.backward(g_s))
            eng.adam_step(lr=1e-4, weight_decay=0.0)
            n[0] += 1
            _lib.check(lib.scgib_adam_step_f32(_lib.ptr(head.params), _lib.ptr(head.grads), _lib.ptr(hm), _lib.ptr(hv), head.total,
                                               n[0], 1e-4, 0.9, 0.999, 1e-8, 0.0, 1.0, torch.cuda.current_stream(DEV).cuda_stream), "adam")
        runs = [timed(step, 3, 30) for _ in range(2)]
        ms = min(runs)
        print(json.dumps(dict(case="finetune_step", classes=C, hidden=H, batch=B, ms_per_step=round(ms, 3),
                              runs_ms=[round(v, 3) for v in runs], graphs_per_s=round(B / ms * 1e3),
                              kernels_ms=profile(step, ("finetune_head_fwd", "finetune_head_bwd", "ft_dWp2")), **info)), flush=True)
        del eng, head


if __name__ == "__main__":
    main()
