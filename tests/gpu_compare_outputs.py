"""Compare what two checkouts compute on the default workloads, bit for bit:

    python tests/gpu_compare_outputs.py --baseline DIR [--out OUT]

Runs ``bench.py --dump-outputs`` for the pre-training and the fine-tuning workloads in this checkout and in the checkout at
DIR (each from its own tree, so each loads its own library) with the same seeds, then compares every dumped .npy array
bitwise.  Prints one JSON line per workload and array, and exits non-zero when any array differs."""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKLOADS = {"pretrain": [], "finetune": ["--workload", "finetune"]}


def dump(tree, workload, out):
    cmd = [sys.executable, "bench.py", "--gpus", "1", "--steps", "20", "--warmup", "3", "--dump-outputs", out] + WORKLOADS[workload]
    r = subprocess.run(cmd, cwd=tree, capture_output=True, text=True)
    if r.returncode != 0:
        raise SystemExit("bench.py failed in %s:\n%s" % (tree, r.stderr[-3000:]))
    return [ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline", required=True, help="checkout to compare against (built)")
    ap.add_argument("--out", default=None, help="keep the dumps here (default: a temporary directory)")
    a = ap.parse_args()
    trees = {"baseline": os.path.abspath(a.baseline), "this": ROOT}
    same = True
    with tempfile.TemporaryDirectory() as tmp:
        base = os.path.abspath(a.out or tmp)
        for wl in WORKLOADS:
            dirs = {}
            for tag, tree in trees.items():
                dirs[tag] = os.path.join(base, wl, tag)
                line = json.loads(dump(tree, wl, dirs[tag]))
                print(json.dumps(dict(workload=wl, tree=tag, metric=line.get("metric"), value=line.get("value"))), flush=True)
            for name in sorted(os.listdir(dirs["baseline"])):
                x = np.load(os.path.join(dirs["baseline"], name))
                y = np.load(os.path.join(dirs["this"], name))
                eq = x.shape == y.shape and x.tobytes() == y.tobytes()
                same &= eq
                print(json.dumps(dict(workload=wl, array=name, shape=list(x.shape), bit_identical=eq)), flush=True)
    sys.exit(0 if same else 1)


if __name__ == "__main__":
    main()
