"""GIN layer kernels against fp64 on non-local and dense graphs (the families of tests/test_gin_layer_edges_host.py: neighbours
beyond the 256-row gather window, tiles over the 1024 staged indices, windows clipped at row 0 and at V, row maps), and the
bf16 layer operators checked at their rounding points.

Bounds are per element, against that element's own scale, never the tensor-wide max norm (a 1500-degree hub would hide a
wrong small row behind its own magnitude):
 * fp32 aggregation a (csrc/gin_tc3.cu): |a - ref| <= (deg + 3) 2^-24 sum|terms|, ref the fp64 sum of the fp64 terms
   (recursive fp32 summation of terms that each carry one or two fp32 roundings of BN + ReLU; a BN term counts
   |(h - mean) scale| + |beta|).  Rigorous: it cannot flake, and a dropped or repeated neighbour misses it by orders of magnitude.
 * fp32 r, y (3xTF32 tcgen05 GEMMs) from the kernel's own a, r: |err| <= (K + 8) 2^-22 (|x| |W|^T + |b|).
 * bf16 a, r, y (csrc/gin_bf16.cu), each stage chained from the kernel's previous one: within one bf16 ulp of the rounded
   fp64 value plus the fp32 accumulation bound of that stage ((deg + 3) 2^-24 sum|terms| for a, (K + 2) 2^-23 (|x| |W|^T + |b|)
   for the single-pass MMAs).  Inputs are bf16 values.
 * batch statistics against fp64 statistics of the kernel's own (rounded) y: mean within 2^-17 mean|y|, rstd within 2^-16
   relative; running statistics at fp32 level.
 * bf16 backward (csrc/gin_bwd_bf16.cu) against tests/bf16_emulation.gin_bwd_ref (rounding points listed there): every output
   element's error over its fp32 accumulation magnitude (|g_u| |W1| for g_a, |g_u|^T |a| for dW1, ...).  Those bounds come from
   the values measured on a B200 (BWD_BOUND), with a 4x margin.

Every case prints its measured errors as one JSON line (shown with pytest -s)."""
import json

import numpy as np
import pytest
import torch

from tests.bf16_emulation import bf16_ulp, gin_aggregate_ref, gin_bn_act_terms, gin_bwd_ref, gin_mlp_ref
from tests.test_gin_layer_edges_host import FAMILIES, family

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U24, U23, U22 = 2.0 ** -24, 2.0 ** -23, 2.0 ** -22
BF16_INSTANCES = [(32, 64), (64, 64), (32, 128), (64, 128), (128, 128)]
# bf16 backward: the largest error over fp32 accumulation magnitude measured on a B200 (1000 W) over every case of this file;
# the bound is 4x.  g_a is the largest: a one-ulp difference of the rounded g_y / g_u operands moves it by ~2^-8 of one term.
BWD_MEASURED = {"g_a": 5.4e-3, "dW1": 7.3e-5, "db1": 2.0e-5, "dW2": 3.6e-5, "db2": 6.2e-6, "dgamma": 6.1e-8, "dbeta": 5.6e-9}
BWD_BOUND = {k: 4 * v for k, v in BWD_MEASURED.items()}
_FAM = {}


def _family(name):
    if name not in _FAM:
        f = family(name)
        src = torch.from_numpy(f["indices"].astype(np.int64))
        dst = torch.repeat_interleave(torch.arange(f["V"]), torch.from_numpy(np.diff(f["indptr"].astype(np.int64))))
        rm = None if f["row_map"] is None else torch.from_numpy(f["row_map"].astype(np.int64))
        dev = dict(indptr=torch.from_numpy(f["indptr"]).to(DEV), indices=torch.from_numpy(f["indices"]).to(DEV),
                   row_map=None if rm is None else rm.to(torch.int32).to(DEV))
        _FAM[name] = dict(f, src=src, dst=dst, rm=rm, deg=(dst.bincount(minlength=f["V"]).double())[:, None], dev=dev)
    return _FAM[name]


def _report(test, **kw):
    print(json.dumps(dict(test=test, **kw)))


def _rnd(x):
    return x.to(torch.bfloat16).double()


def _worst(err, tol):
    """largest err / tol (<= 1 passes) and where"""
    q = err / tol
    i = int(torch.argmax(q))
    return float(q.reshape(-1)[i]), np.unravel_index(i, q.shape)


def _bn_in(kin, scale, seed):
    g = torch.Generator().manual_seed(seed)
    mean = torch.randn(kin, generator=g) * 0.5 * scale
    rstd = (0.5 + 1.5 * torch.rand(kin, generator=g)) / scale
    gamma, beta = 0.5 + torch.rand(kin, generator=g), 0.6 * torch.rand(kin, generator=g) - 0.3
    return torch.stack([mean, rstd, gamma, beta]).float()


def _weights(kin, H, seed, bf16):
    g = torch.Generator().manual_seed(seed)
    W1 = torch.randn(H, kin, generator=g) / kin ** 0.5
    W2 = torch.randn(H, H, generator=g) / H ** 0.5
    b1, b2 = torch.randn(H, generator=g) * 0.1, torch.randn(H, generator=g) * 0.1
    if bf16:                     # exact bf16 values: the kernel's operand rounding is then exact, only accumulation differs
        W1, W2 = W1.bfloat16().float(), W2.bfloat16().float()
    return W1, b1, W2, b2


def _check_stats(y, bn, running0, running, V):
    """bn_out {mean, rstd} and the running-statistics update against fp64 statistics of the kernel's own y"""
    y = y.double()
    mean, var = y.mean(0), y.var(0, unbiased=False)
    scale = y.abs().mean(0)
    e_mean = _worst((bn[0].double().cpu() - mean).abs(), 2.0 ** -17 * scale + 1e-30)[0]
    rstd = 1.0 / torch.sqrt(var + 1e-5)
    e_rstd = _worst((bn[1].double().cpu() - rstd).abs(), 2.0 ** -16 * rstd)[0]
    rm = 0.9 * running0[0].double() + 0.1 * mean
    rv = 0.9 * running0[1].double() + 0.1 * var * V / max(V - 1, 1)
    e_run = max(_worst((running[0].double().cpu() - rm).abs(), 2.0 ** -20 * (running0[0].double().abs() + scale) + 1e-30)[0],
                _worst((running[1].double().cpu() - rv).abs(), 2.0 ** -20 * running0[1].double().abs() + 2.0 ** -15 * var + 1e-30)[0])
    assert e_mean <= 1 and e_rstd <= 1 and e_run <= 1, (e_mean, e_rstd, e_run)
    return e_mean, e_rstd, e_run


def _fwd_case(name, kin, H, bn_on, scale, bf16, seed):
    from scgib_b200 import ops
    f = _family(name)
    V, n_in = f["V"], f["n_in"]
    g = torch.Generator().manual_seed(seed)
    h = torch.randn(n_in, kin, generator=g) * scale
    if bf16:
        h = h.bfloat16().float()
    bn = _bn_in(kin, scale, seed + 1) if bn_on else None
    W1, b1, W2, b2 = _weights(kin, H, seed + 2, bf16)
    running0 = torch.stack([torch.randn(H, generator=g), 0.5 + torch.rand(H, generator=g)])
    running = running0.clone().to(DEV)
    d = f["dev"]
    hin = h.to(DEV).bfloat16() if bf16 else h.to(DEV)
    y, bnk, a, r = ops.gin_layer_fwd(hin, d["indptr"], d["indices"], W1.to(DEV), b1.to(DEV), W2.to(DEV), b2.to(DEV),
                                     row_map=d["row_map"], bn_in=None if bn is None else bn.to(DEV), running=running, save=True)
    torch.cuda.synchronize()
    ak, rk, yk = a.double().cpu(), r.double().cpu(), y.double().cpu()
    # aggregation: the fp64 sum of the fp64 terms, per element against its own sum|terms|
    terms, mag = gin_bn_act_terms(h, bn, bf16)
    a_ref = gin_aggregate_ref(terms, f["src"], f["dst"], f["rm"])
    a_tol = (f["deg"] + 3) * U24 * gin_aggregate_ref(mag, f["src"], f["dst"], f["rm"])
    W1d, W2d, b1d, b2d = W1.double(), W2.double(), b1.double(), b2.double()
    if bf16:
        a_ref = _rnd(a_ref)
        a_tol = a_tol + bf16_ulp(torch.maximum(a_ref.abs(), ak.abs()))
        r_ref, _ = gin_mlp_ref(ak, W1d, b1d, W2d, b2d)
        r_tol = (kin + 2) * U23 * (ak.abs() @ W1d.abs().t() + b1d.abs()) + bf16_ulp(torch.maximum(r_ref.abs(), rk.abs()))
        _, y_ref = gin_mlp_ref(None, W1d, b1d, W2d, b2d, r=rk)
        y_tol = (H + 2) * U23 * (rk.abs() @ W2d.abs().t() + b2d.abs()) + bf16_ulp(torch.maximum(y_ref.abs(), yk.abs()))
    else:
        r_ref, _ = gin_mlp_ref(ak, W1d, b1d, W2d, b2d, emulate=False)
        r_tol = (kin + 8) * U22 * (ak.abs() @ W1d.abs().t() + b1d.abs())
        _, y_ref = gin_mlp_ref(None, W1d, b1d, W2d, b2d, emulate=False, r=rk)
        y_tol = (H + 8) * U22 * (rk.abs() @ W2d.abs().t() + b2d.abs())
    res = {}
    for nm, got, ref, tol in (("a", ak, a_ref, a_tol), ("r", rk, r_ref, r_tol), ("y", yk, y_ref, y_tol)):
        q, where = _worst((got - ref).abs(), tol + 1e-300)
        res[nm] = q
        if bf16:
            res[nm + "_differs"] = float((got != ref).double().mean())
        assert q <= 1, (name, nm, q, where, float(got[where]), float(ref[where]), float(tol[where]))
    res["stats"] = _check_stats(yk, bnk, running0, running, V)
    _report("bf16_forward" if bf16 else "fp32_forward", family=name, kin=kin, H=H, bn=bn_on, scale=scale, **res)


FWD32 = [(k, bn) for k in (32, 64) for bn in (False, True) if not (bn and k == 32)]


@pytest.mark.parametrize("kin,bn_on", FWD32)
@pytest.mark.parametrize("name", FAMILIES)
def test_fp32_layer_forward_families(name, kin, bn_on):
    """scgib_gin_layer_fwd_f32 (gin_tc3) on every family: a per row against fp64, r and y from the kernel's own a and r,
    statistics of the kernel's own y."""
    _fwd_case(name, kin, 64, bn_on, 1.0, False, 11 + kin)


BF16_CASES = [(k, h, bn) for k, h in BF16_INSTANCES for bn in (False, True) if not (bn and k != h)]


@pytest.mark.parametrize("kin,H,bn_on", BF16_CASES)
@pytest.mark.parametrize("name", FAMILIES)
def test_bf16_layer_forward_families(name, kin, H, bn_on):
    """scgib_gin_layer_fwd_bf16 (gin_bf16) on every family and (kin, H) instance, each stage within one bf16 ulp of the fp64
    value computed from the kernel's previous stage."""
    _fwd_case(name, kin, H, bn_on, 1.0, True, 21 + kin + H)


@pytest.mark.parametrize("bf16", [False, True])
@pytest.mark.parametrize("scale", [1e-3, 1e2])
@pytest.mark.parametrize("name", ["macrocycles", "star", "random_map"])
def test_layer_forward_magnitudes(name, scale, bf16):
    """activations of 1e-3 and 1e2 (inputs, and the BatchNorm constants of the producing layer scaled with them)"""
    for kin, H in ((64, 64),) + (((128, 128),) if bf16 else ()):
        for bn_on in (False, True):
            _fwd_case(name, kin, H, bn_on, scale, bf16, 31 + kin)


BWD_INSTANCES = [(32, 64, True), (64, 64, True), (64, 64, False), (32, 128, True), (64, 128, True), (128, 128, True), (128, 128, False)]


def _bwd_case(name, kin, H, ga_f32, csr, scale, gscale, seed):
    from scgib_b200 import ops
    f = _family(name)
    V = f["V"]
    g = torch.Generator().manual_seed(seed)
    W1, b1, W2, b2 = _weights(kin, H, seed + 1, True)
    W1d, W2d = W1.double(), W2.double()
    # a consistent saved forward state in bf16: a, r = relu(W1 a + b1), y = W2 r + b2, bn = statistics of y
    a = _rnd(torch.randn(V, kin, generator=g, dtype=torch.float64) * scale)
    r, y = gin_mlp_ref(a, W1d, b1.double() * scale, W2d, b2.double() * scale)
    # BatchNorm constants near the statistics of y, on a coarse grid (bf16 mean, gamma, beta; power-of-two rstd): the kernel's
    # ReLU mask relu(y * scale + shift) > 0 is then exact in fp32 however the compiler contracts it, and so is the reference's
    mean, var = y.mean(0), y.var(0, unbiased=False)
    rstd = torch.pow(2.0, torch.round(-0.5 * torch.log2(var + 1e-5)))
    gamma, beta = _rnd(0.5 + torch.rand(H, generator=g, dtype=torch.float64)), _rnd(0.6 * torch.rand(H, generator=g, dtype=torch.float64) - 0.3)
    bn = torch.stack([_rnd(mean), rstd, gamma, beta]).float()
    g_next = torch.randn(V, H, generator=g, dtype=torch.float64) * gscale
    if csr:
        g_next = _rnd(g_next)
    else:
        g_next = g_next.float().double()
    out, mag = gin_bwd_ref(g_next, f["src"] if csr else None, f["dst"] if csr else None, y, r, a, bn, W1d, W2d, ga_f32)
    d = f["dev"]
    b16 = lambda t: t.to(DEV).bfloat16()
    gk = ops.gin_layer_bwd(b16(g_next) if csr else g_next.float().to(DEV), b16(y), b16(r), b16(a), bn.to(DEV), W1.to(DEV),
                           W2.to(DEV), indptr=d["indptr"] if csr else None, indices=d["indices"] if csr else None, ga_f32=ga_f32)
    torch.cuda.synchronize()
    assert (gk[0].dtype == torch.float32) == (ga_f32 or kin < H)
    res = {}
    for nm, got, ref, m in zip(("g_a", "dW1", "db1", "dW2", "db2", "dgamma", "dbeta"), gk, out, mag):
        got = got.double().cpu().reshape(ref.shape)
        q, where = _worst((got - ref).abs(), m + 1e-300)
        res[nm] = q
        assert q <= BWD_BOUND[nm], (name, nm, q, where, float(got[where]), float(ref[where]), float(m[where]))
    _report("bf16_backward", family=name, kin=kin, H=H, ga_f32=ga_f32, csr=csr, scale=scale, gscale=gscale, **res)


@pytest.mark.parametrize("csr", [False, True])
@pytest.mark.parametrize("kin,H,ga_f32", BWD_INSTANCES)
@pytest.mark.parametrize("name", ["macrocycles", "star", "dense_walk"])
def test_bf16_layer_backward(name, kin, H, ga_f32, csr):
    """scgib_gin_layer_bwd_bf16 (gin_bwd_pre_bf16 + gin_bwd_bf16) in CSR and direct mode, every ga_f32 instance, against the
    fp64 reference with the kernels' rounding points"""
    _bwd_case(name, kin, H, ga_f32, csr, 1.0, 1.0, 41 + kin + H)


@pytest.mark.parametrize("scale,gscale", [(1e-3, 1e-6), (1e2, 1e4)])
@pytest.mark.parametrize("kin,H,ga_f32", [(64, 64, False), (128, 128, True)])
def test_bf16_layer_backward_magnitudes(kin, H, ga_f32, scale, gscale):
    for csr in (False, True):
        _bwd_case("macrocycles", kin, H, ga_f32, csr, scale, gscale, 51 + kin)

