"""Per-tile role timeline of the tc2 forward kernel (experiments): SCGIB_DBG=1024 python -m tests.gpu_tc2_trace; of the
fp16-split backward kernel gin_bwd_h: SCGIB_DBG=2048 python -m tests.gpu_tc2_trace bwdh"""
import ctypes
import numpy as np
import torch
from scgib_b200 import _lib
from scgib_b200.engine import PretrainEngine
from scgib_b200.synth import synth_batch

lib = _lib.load()
dev = torch.device("cuda:0")
import os
eng = PretrainEngine(9, gin_layers=4, device=dev, seed=0, dtype=os.environ.get("SCGIB_TRACE_DTYPE", "fp32"))
g = synth_batch(1, 4096).to(dev)
b = eng.make_batch(g, 1)
import sys
BWD = len(sys.argv) > 1 and sys.argv[1] == "bwdh"
for _ in range(3):
    eng.forward(b)
    if BWD:
        eng.backward()
torch.cuda.synchronize()
n = 160 * 16 * 12
buf = (ctypes.c_longlong * n)()
BF = os.environ.get("SCGIB_TRACE_DTYPE", "fp32") == "bf16"
(lib.scgib_debug_bwdh_trace if BWD else (lib.scgib_debug_bf16_trace if BF else lib.scgib_debug_tc2_trace))(ctypes.cast(buf, ctypes.c_void_p), n)
t = np.frombuffer(buf, dtype=np.int64).reshape(160, 16, 12).astype(np.float64)
names = (["l.start", "l.d2prev", "l.full1", "l.d1", "l.full2", "m.g13", "m.g24", "e.d1", "e.gu", "e.d2", "e.end"] if BWD else
         ["p.start", "p.landed", "p.issued", "p.gathered", "p.full", "m.g1", "m.g2", "e.d1", "e.r", "e.d2", "e.end"])
for cta in (0, 40, 100):
    t0 = t[cta, 0, 0]
    print("CTA", cta)
    for i in range(14):
        if t[cta, i, 0] == 0 and i > 0:
            break
        print("  tile %2d: " % i + " ".join("%s=%6.2f" % (names[e], (t[cta, i, e] - t0) / 1965.0) for e in range(11)))
