"""CPU-side checks of the bf16-mode encoder entries (csrc/encoder_bf16.cu): argument validation returns the documented
SCGIB_E_* code before anything is launched, and the workspace query sizes the partials.  No device is touched: every call
below fails validation."""
import ctypes

import pytest

E_NULL, E_SHAPE, E_ALIGN, E_WORKSPACE, E_RANGE = -1, -2, -3, -4, -5
P = ctypes.c_void_p(0x10000)          # 16-byte aligned dummy pointer (never dereferenced: validation fails first)
Q = ctypes.c_void_p(0x10008)          # 8-byte aligned only


def _lib():
    from tests.test_abi import _lib as load
    return load().load()


def test_graph_aggregate_bf16_validation():
    lib = _lib()
    f = lib.scgib_graph_aggregate_bf16
    ok = dict(i=P, W=64, rm=None, ip=P, ix=P, V=10, sn=0, dn=1, add=None, out=P, f32=0)

    def call(**kw):
        a = dict(ok, **kw)
        return f(a["i"], a["W"], a["rm"], a["ip"], a["ix"], a["V"], a["sn"], a["dn"], a["add"], a["out"], a["f32"], None)
    assert call(i=None) == E_NULL and call(ip=None) == E_NULL and call(out=None) == E_NULL
    for W in (0, 16, 48, 96, 512):
        assert call(W=W) == E_SHAPE, W
    assert call(sn=3) == E_SHAPE and call(dn=-1) == E_SHAPE
    assert call(V=0) == E_RANGE
    assert call(i=Q) == E_ALIGN and call(add=Q) == E_ALIGN and call(out=Q) == E_ALIGN


def test_linear_fwd_bf16_validation():
    lib = _lib()
    f = lib.scgib_linear_fwd_bf16
    ok = dict(X0=P, M0=None, map0=None, W0=P, K0=64, k0=0, X1=None, M1=None, W1=None, K1=0, k1=0, b=None, relu=0, V=10, O=64,
              Y=P, f32=0)

    def call(**kw):
        a = dict(ok, **kw)
        return f(a["X0"], a["M0"], a["map0"], a["W0"], a["K0"], a["k0"], a["X1"], a["M1"], a["W1"], a["K1"], a["k1"], a["b"],
                 a["relu"], a["V"], a["O"], a["Y"], a["f32"], None)
    assert call(X0=None) == E_NULL and call(W0=None) == E_NULL and call(Y=None) == E_NULL and call(X1=P) == E_NULL
    for K in (0, 16, 48, 96, 512):
        assert call(K0=K) == E_SHAPE, K
        assert call(X1=P, W1=P, K1=K) == E_SHAPE, K
    for O in (0, 16, 48, 512):
        assert call(O=O) == E_SHAPE, O
    assert call(V=0) == E_RANGE
    for k in ("X0", "M0", "W0", "X1", "M1", "W1", "b", "Y"):
        kw = {k: Q}
        if k in ("X1", "M1"):
            kw.update(W1=P, K1=64, X1=kw.get("X1", P))
        assert call(**kw) == E_ALIGN, k
    # a pair of wide operands does not fit shared memory with its row tiles
    assert call(K0=256, X1=P, W1=P, K1=256, O=256) == E_SHAPE


def test_linear_bwd_w_bf16_validation():
    lib = _lib()
    f = lib.scgib_linear_bwd_w_bf16
    need = lib.scgib_linear_bwd_w_bf16_workspace_bytes(100000, 128, 64)
    assert need >= 128 * 64 * 4 and need > lib.scgib_linear_bwd_w_bf16_workspace_bytes(1, 128, 64)
    ok = dict(G=P, M=None, X=P, mp=None, V=100000, O=128, K=64, kxo=0, acc=0, dW=P, db=None, ws=P, wsb=need)

    def call(**kw):
        a = dict(ok, **kw)
        return f(a["G"], a["M"], a["X"], a["mp"], a["V"], a["O"], a["K"], a["kxo"], a["acc"], a["dW"], a["db"], a["ws"], a["wsb"],
                 None)
    assert call(G=None) == E_NULL and call(X=None) == E_NULL and call(dW=None) == E_NULL and call(ws=None) == E_NULL
    for O in (32, 96, 192, 512):
        assert call(O=O) == E_SHAPE, O
    for K in (16, 48, 512):
        assert call(K=K) == E_SHAPE, K
    assert call(V=0) == E_RANGE
    assert call(G=Q) == E_ALIGN and call(M=Q) == E_ALIGN and call(X=Q) == E_ALIGN and call(ws=Q) == E_ALIGN
    assert call(wsb=need - 1) == E_WORKSPACE


def test_conversion_entries_validation():
    lib = _lib()
    assert lib.scgib_f32_to_bf16(None, 8, P, None) == E_NULL
    assert lib.scgib_f32_to_bf16(P, 0, P, None) == E_RANGE
    assert lib.scgib_f32_to_bf16(P, 12, P, None) == E_SHAPE
    assert lib.scgib_f32_to_bf16(Q, 8, P, None) == E_ALIGN
    assert lib.scgib_input_proj_fwd_bf16(P, P, 10, 9, 32, None, None) == E_NULL
    assert lib.scgib_input_proj_fwd_bf16(P, P, 10, 9, 64, P, None) == E_SHAPE
    assert lib.scgib_input_proj_fwd_bf16(P, P, 0, 9, 32, P, None) == E_RANGE
    assert lib.scgib_input_proj_fwd_bf16(P, P, 10, 9, 32, Q, None) == E_ALIGN


def test_encoders_follow_the_outer_dtype():
    import types
    from scgib_b200 import encoders
    import torch
    assert encoders.act_dtype(types.SimpleNamespace(act_dtype="bf16")) == torch.bfloat16
    assert encoders.act_dtype(types.SimpleNamespace(act_dtype="fp32")) == torch.float32
    assert encoders.act_dtype(types.SimpleNamespace()) == torch.float32


@pytest.mark.parametrize("encoder,hidden", [("GraphSAGE", 64), ("GCN", 64), ("GraphSAGE", 128), ("GCN", 128)])
def test_oracle_bf16_emulation_off_is_the_oracle(encoder, hidden):
    """tests/bf16_emulation.py with the switch off computes the oracle's encoder bit for bit (forward and backward); with
    it on, the result moves by bf16-sized amounts only."""
    import copy
    import numpy as np
    import torch
    from oracle.graph_ref import ego_batch_ref, synth_batch
    from oracle.scgib_oracle import make_encoder, tgraph_from_ego
    from tests.bf16_emulation import emulate
    g = synth_batch(33 + hidden, 30)
    e = ego_batch_ref(g, 1)
    tg = tgraph_from_ego(e)
    torch.manual_seed(hidden)
    ref = make_encoder(encoder, 32, hidden).double()
    t = torch.randn(int(e.sub_indptr.shape[0]) - 1, 32, dtype=torch.float64)
    outs = []
    for mode in (None, False, True):
        m = copy.deepcopy(ref)
        if mode is not None:
            emulate(m, mode)
        x = t.clone().requires_grad_(True)
        y = m(tg, x)
        (y * (0.5 + torch.rand(y.shape, dtype=torch.float64, generator=torch.Generator().manual_seed(1)))).sum().backward()
        outs.append((y.detach(), x.grad, {n: p.grad for n, p in m.named_parameters() if p.grad is not None}))
    (y0, g0, p0), (y1, g1, p1), (y2, g2, p2) = outs
    assert torch.equal(y0, y1) and torch.equal(g0, g1) and p0.keys() == p1.keys()
    assert all(torch.equal(p0[n], p1[n]) for n in p0)
    r = lambda a, b: float((a - b).abs().max() / b.abs().max())
    assert 0 < r(y2, y0) <= 2e-2 and 0 < r(g2, g0) <= 0.3      # g_t: three layers of rounded gradients
    assert np.median([r(p2[n], p0[n]) for n in p0]) <= 5e-2
