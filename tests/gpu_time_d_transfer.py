"""Time the GIN pre-training step over the transferred feature width d_transfer (measurement, no target):

    python tests/gpu_time_d_transfer.py [--repo DIR] [--narrow-only]

Cases: PCQM shape, B = 4096, k = 1, F = 9, fp32 and bf16, at hidden 64 x d in {32, 64} and hidden 128 x d in {32, 64, 128}.
Each step (forward + backward + Adam of the fused engine) is timed with CUDA events after warm-up, twice, and the faster run
is kept.  A separate profiled step reports the device time of `fwd_prep` (input projection and the xagg side CTAs),
`input_proj_bwd`, and the layer-0 GIN launches: the first GIN forward launch and the last GIN backward launches of the step,
which serve both encoders.  ``--repo DIR`` imports the package of another checkout, for example the parent commit;
``--narrow-only`` keeps the d = 32 rows, which every checkout can run.  One JSON line per measurement; the GPU name and
power limit are read in the same run."""
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
    from scgib_b200.engine import DeviceBatch, PretrainEngine
    from scgib_b200.graph import khop_ego_batch
    from scgib_b200.synth import synth_batch
    sys.path.insert(1, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from tests.gpu_time_composed_downstream import DEV, gpu_info, timed
    lib = _lib.load()
    info = dict(gpu_info(), tree=a.tag or os.path.basename(os.path.abspath(a.repo)))

    def profile(step):
        """device ms of the named launches of one step: fwd_prep, input_proj_bwd, and the layer-0 GIN launches"""
        step()
        torch.cuda.synchronize()
        lib.scgib_profile_enable(1)
        step()
        torch.cuda.synchronize()
        launches = []
        for i in range(lib.scgib_profile_count()):
            nm, ms = ctypes.c_char_p(), ctypes.c_float()
            if lib.scgib_profile_get(i, ctypes.byref(nm), ctypes.byref(ms)) == 0:
                launches.append((nm.value.decode(), ms.value))
        lib.scgib_profile_enable(0)
        out = {n: round(ms, 4) for n, ms in launches if n in ("fwd_prep", "input_proj_bwd")}
        # layer 0 is the first GIN forward and the last GIN backward of the step: one shared launch for both encoders
        # ("...enc1+2"), or one launch per encoder (".enc1", ".enc2") on the FFMA kernels
        for prefix, first in (("gin_fwd", True), ("gin_bwd_pre", False), ("gin_bwd_main", False)):
            ls = [(n, ms) for n, ms in launches if n.startswith(prefix)]
            if ls:
                per = 1 if ls[0][0].endswith("enc1+2") else 2
                sel = ls[:per] if first else ls[-per:]
                out["layer0:" + sel[0][0].split(".")[0]] = round(sum(ms for _, ms in sel), 4)
        return out

    B = 4096
    g = synth_batch(1, B, "pcqm").to(DEV)
    b = DeviceBatch(g, khop_ego_batch(g, 1), g.ndata["x"])
    pairs = [(64, 32), (64, 64), (128, 32), (128, 64), (128, 128)]
    for H, d in pairs:
        if a.narrow_only and d != 32:
            continue
        for dtype in ("fp32", "bf16"):
            kw = {} if d == 32 else {"d_transfer": d}      # the parent checkout's engine may not take the keyword
            eng = PretrainEngine(9, gin_layers=4, hidden=H, device=DEV, seed=0, dtype=dtype, **kw)
            step = lambda: eng.train_step(b)
            runs = [timed(step, 3, 30) for _ in range(2)]
            ms = min(runs)
            print(json.dumps(dict(case="pretrain_step", hidden=H, d_transfer=d, dtype=dtype, batch=B, N=b.N,
                                  Ns=int(b.ego.ego_nodes.numel()), ms_per_step=round(ms, 3), runs_ms=[round(v, 3) for v in runs],
                                  graphs_per_s=round(B / ms * 1e3), kernels_ms=profile(step), **info)), flush=True)
            del eng


if __name__ == "__main__":
    main()
