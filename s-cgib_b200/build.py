"""Build libscgib.so (hand-written sm_100a CUDA behind the C ABI of include/scgib.h) in-tree with nvcc.

    python s-cgib_b200/build.py [--verbose]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box with gpurun.
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libscgib.so")
SOURCES = ["api.cu", "graph_kernels.cu", "gin_kernels.cu", "head_kernels.cu", "loss_kernels.cu", "finetune_kernels.cu",
           "logm_kernels.cu", "peer_kernels.cu", "gin_tc3.cu", "gin_tc4.cu", "gin_bwd_h.cu", "contrastive_tc.cu", "head_tc.cu", "gin_bf16.cu", "gin_bwd_bf16.cu", "encoder_ops.cu",
           "encoder_bf16.cu"]
HEADERS = ["common.cuh", "kernels.cuh", "umma.cuh", "side_jobs.cuh", "scgib_private.h", os.path.join("..", "..", "include", "scgib.h")]
# hardware probes of the tcgen05 operand formats: test infrastructure, NOT linked into the product library
PROBE_DIR = os.path.join(os.path.dirname(HERE), "tests", "csrc")
PROBE_LIB = os.path.join(PROBE_DIR, "libscgib_probe.so")
PROBE_SOURCES = ["umma_test.cu", "umma_probe2.cu", "umma_probe_bf16.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr"]


def _digest():
    h = hashlib.sha256()
    for f in SOURCES + HEADERS:
        with open(os.path.join(CSRC, f), "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(FLAGS).encode())
    return h.hexdigest()


def build(verbose=False, force=False):
    os.makedirs(LIBDIR, exist_ok=True)
    stamp = os.path.join(LIBDIR, "libscgib.stamp")
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == dig:
        return LIB
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(LIBDIR, src.replace(".cu", ".o"))
        cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write("---- %s\n%s\n" % (src, out))
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    cmd = [NVCC, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    subprocess.check_call(cmd)
    with open(stamp, "w") as fh:
        fh.write(dig)
    return LIB


def build_probes(force=False):
    """tests/csrc/libscgib_probe.so (sm_100a); returns its path."""
    srcs = [os.path.join(PROBE_DIR, f) for f in PROBE_SOURCES if os.path.exists(os.path.join(PROBE_DIR, f))]
    h = hashlib.sha256()
    for f in srcs + [os.path.join(CSRC, "umma.cuh")]:
        with open(f, "rb") as fh:
            h.update(fh.read())
    stamp = os.path.join(PROBE_DIR, "libscgib_probe.stamp")
    if not force and os.path.exists(PROBE_LIB) and os.path.exists(stamp) and open(stamp).read() == h.hexdigest():
        return PROBE_LIB
    cmd = [NVCC] + FLAGS + ["-I", CSRC, "-I", os.path.join(os.path.dirname(HERE), "include"), "-shared", "-o", PROBE_LIB] + srcs + ["-lcudart"]
    subprocess.check_call(cmd)
    with open(stamp, "w") as fh:
        fh.write(h.hexdigest())
    return PROBE_LIB


if __name__ == "__main__":
    print(build(verbose="--verbose" in sys.argv, force=True))
    print(build_probes(force=True))
