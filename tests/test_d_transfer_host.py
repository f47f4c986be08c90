"""CPU-side checks of the transferred feature width d_transfer in {32, 64, 128}, d_transfer <= hidden: the C ABI refuses every
other width with SCGIB_E_SHAPE before anything is launched and sizes its layout for the accepted ones, the module constructors
raise before any device work, and a checkpoint pre-trained at one width cannot be wrapped at another."""
import ctypes
import types

import pytest
import torch

from tests.test_abi import _lib

E_NULL, E_SHAPE, E_ALIGN, E_RANGE = -1, -2, -3, -5
P = ctypes.c_void_p(0x10000)          # 16-byte aligned dummy pointer (never dereferenced: validation fails first)
Q = ctypes.c_void_p(0x10008)          # 8-byte aligned only
ACCEPTED = [(64, 32), (64, 64), (128, 32), (128, 64), (128, 128)]     # (hidden, d_transfer)
REFUSED = [(H, d) for H in (64, 128) for d in (16, 48, 96, 256)] + [(64, 128)]


def _dims(L, d, hidden, in_dim=37, layers=4):
    return L.Dims(in_dim=in_dim, d_transfer=d, hidden=hidden, gin_layers=layers, act_dtype=0)


@pytest.mark.parametrize("hidden,d", REFUSED)
def test_layout_refuses_other_widths(hidden, d):
    L = _lib()
    lib = L.load()
    dm = _dims(L, d, hidden)
    assert lib.scgib_param_slots(ctypes.byref(dm)) == E_SHAPE
    assert lib.scgib_param_layout(ctypes.byref(dm), None, None) == E_SHAPE
    assert lib.scgib_pretrain_workspace_bytes(ctypes.byref(dm), 4, 40, 80, 120, 200) == 0
    assert lib.scgib_pretrain_forward_f32(ctypes.byref(dm), P, None, None, P, None, None, None, None, P, 1 << 20, None) == E_SHAPE


@pytest.mark.parametrize("hidden,d", ACCEPTED)
@pytest.mark.parametrize("layers", [4, 5])
def test_layout_at_accepted_widths(hidden, d, layers):
    L = _lib()
    lib = L.load()
    from scgib_b200.engine import param_names, param_shapes
    F = 37
    dm = _dims(L, d, hidden, F, layers)
    n = lib.scgib_param_slots(ctypes.byref(dm))
    off, sz = (ctypes.c_int64 * n)(), (ctypes.c_int64 * n)()
    total = lib.scgib_param_layout(ctypes.byref(dm), off, sz)
    assert total >= sum(sz) and all(o % 4 == 0 for o in off)
    assert sz[L.P_TRANSFER] == d * F                                  # transfer_d.weight [d][F]
    for e in range(2):
        base = L.P_ENC + e * layers * L.ENC_SLOTS
        assert sz[base + L.ENC_W1] == hidden * d                      # layer-0 W1 [H][d]
        for l in range(1, layers):
            assert sz[base + l * L.ENC_SLOTS + L.ENC_W1] == hidden * hidden
    shapes = param_shapes(F, layers, hidden, d)
    assert n == len(param_names(layers)) == len(shapes)
    assert [int(torch.Size(s).numel()) for s in shapes] == list(sz)
    small = lib.scgib_pretrain_workspace_bytes(ctypes.byref(_dims(L, 32, hidden, F, layers)), 128, 1920, 4100, 6000, 8200)
    wide = lib.scgib_pretrain_workspace_bytes(ctypes.byref(dm), 128, 1920, 4100, 6000, 8200)
    assert 0 < small <= wide
    if d > 32:     # t, the two layer-0 inputs a and their gradients ga0 grow with d
        assert wide - small >= (1920 * 3 + 6000 * 2) * (d - 32) * 4


def test_operator_entries_take_the_width():
    L = _lib()
    lib = L.load()
    for DT in (16, 48, 96, 256):
        assert lib.scgib_input_proj_fwd_f32(P, P, 10, 9, DT, P, None) == E_SHAPE, DT
        assert lib.scgib_input_proj_fwd_d_bf16(P, P, 10, 9, DT, P, None) == E_SHAPE, DT
        assert lib.scgib_transfer_bwd_workspace_bytes_d(10, 0, 9, DT) == 0, DT
        assert lib.scgib_transfer_bwd_d_f32(P, 9, DT, 1, P, 10, None, None, None, 0, None, None, None, P, P, 1 << 20, None) == E_SHAPE
    for DT in (32, 64, 128):
        assert lib.scgib_input_proj_fwd_f32(P, P, 0, 9, DT, P, None) == E_RANGE, DT        # accepted width: the next check fails
        assert lib.scgib_input_proj_fwd_d_bf16(P, P, 10, 9, DT, Q, None) == E_ALIGN, DT
        assert lib.scgib_transfer_bwd_d_f32(P, 9, DT, 1, P, 0, None, None, None, 0, None, None, None, P, P, 1 << 20, None) == E_RANGE
    # the partials are [grid][DT][FP]: the workspace grows by the partial rows of the wider width; DT = 32 is the old entry
    w32, w64 = lib.scgib_transfer_bwd_workspace_bytes_d(1000, 2000, 9, 32), lib.scgib_transfer_bwd_workspace_bytes_d(1000, 2000, 9, 64)
    assert w32 == lib.scgib_transfer_bwd_workspace_bytes(1000, 2000, 9)
    assert w64 - w32 >= lib.scgib_num_sms() * 32 * 32 * 4
    assert "d_transfer 32, 64 or 128" in lib.scgib_error_string(E_SHAPE).decode()


def test_bf16_projection_entries():
    """scgib_input_proj_fwd_bf16 keeps its DT = 32 contract; the *_d entry takes the wider widths and validates the rest."""
    lib = _lib().load()
    for DT in (64, 128):
        assert lib.scgib_input_proj_fwd_bf16(P, P, 10, 9, DT, P, None) == E_SHAPE, DT
        assert lib.scgib_input_proj_fwd_d_bf16(P, P, 0, 9, DT, P, None) == E_RANGE, DT
    assert lib.scgib_input_proj_fwd_d_bf16(P, P, 10, 9, 32, None, None) == E_NULL
    assert lib.scgib_input_proj_fwd_d_bf16(P, P, 10, 0, 64, P, None) == E_SHAPE
    assert lib.scgib_input_proj_fwd_d_bf16(P, P, 10, 129, 64, P, None) == E_SHAPE


def _args(**kw):
    a = types.SimpleNamespace(recons_type="adj", useAtt=1, readout_f="sum", d_transfer=32, device="cpu", batch_size=16,
                              task="graph_classification", dataset="Peptides-func", k_transition=1)
    a.__dict__.update(kw)
    return a


@pytest.mark.parametrize("hidden,d", REFUSED)
@pytest.mark.parametrize("encoder", ["GIN", "GraphSAGE"])
def test_constructors_refuse_other_widths(hidden, d, encoder, tmp_path):
    import models
    unused = str(tmp_path / "unused.pt")                 # never opened: the width check comes first
    a = _args(d_transfer=d)
    msg = r"d_transfer = %d .*allowed: 32, 64" % d
    with pytest.raises(NotImplementedError, match=msg):
        models.Mainmodel(a, 9, hidden_dim=hidden, num_layers=4, num_heads=4, k_transition=1, encoder=encoder)
    with pytest.raises(NotImplementedError, match=msg):
        models.Mainmodel_continue(a, 9, hidden, 4, 4, 1, 1, unused, encoder)
    with pytest.raises(NotImplementedError, match=msg):
        models.Mainmodel_finetuning(a, 9, hidden, 4, 4, 1, 10, unused, encoder)
    with pytest.raises(NotImplementedError, match=msg):
        models.Mainmodel_domainadapt(a, 9, hidden, 4, 4, 1, 10, unused, encoder)
    with pytest.raises(NotImplementedError, match=msg):
        models.GIN(d, hidden)


@pytest.mark.parametrize("hidden,d", ACCEPTED)
def test_constructors_build_accepted_widths(hidden, d):
    import models
    m = models.Mainmodel(_args(d_transfer=d), 37, hidden_dim=hidden, num_layers=4, num_heads=4, k_transition=1, encoder="GIN")
    assert m.transfer_d.weight.shape == (d, 37)
    assert m.Encoder1.ginlayers[0].apply_func.mlp[0].weight.shape == (hidden, d)
    s = models.Mainmodel(_args(d_transfer=d), 37, hidden_dim=hidden, num_layers=4, num_heads=4, k_transition=1, encoder="GCN")
    assert s.Encoder1.conv1.weight.shape == (d, 2 * hidden)


@pytest.mark.parametrize("encoder", ["GIN", "GraphSAGE"])
@pytest.mark.parametrize("pre,wrap", [(64, 32), (32, 64)])
def test_checkpoint_width_mismatch(encoder, pre, wrap, tmp_path):
    import models
    m = models.Mainmodel(_args(d_transfer=pre), 9, hidden_dim=64, num_layers=4, num_heads=4, k_transition=1, encoder=encoder)
    ckpt = str(tmp_path / "pre.pt")
    torch.save(m, ckpt)
    a = _args(d_transfer=wrap)
    msg = r"d_transfer = %d .*--d_transfer is %d" % (pre, wrap)
    with pytest.raises(ValueError, match=msg):
        models.Mainmodel_continue(a, 9, 64, 4, 4, 1, 1, ckpt, encoder)
    with pytest.raises(ValueError, match=msg):
        models.Mainmodel_finetuning(a, 9, 64, 4, 4, 1, 10, ckpt, encoder)
    with pytest.raises(ValueError, match=msg):
        models.Mainmodel_domainadapt(a, 9, 64, 4, 4, 1, 10, ckpt, encoder)
    ok = models.Mainmodel_continue(_args(d_transfer=pre), 9, 64, 4, 4, 1, 1, ckpt, encoder)     # the matching width loads
    assert ok.transfer_d.weight.shape == (pre, 9)


def test_cli_help_states_the_widths():
    import exp_pep_func_5
    import exp_pretraining
    for mod in (exp_pretraining, exp_pep_func_5):
        act = {a.dest: a for a in mod.build_parser()._actions}["d_transfer"]
        assert act.default == 32 and "32, 64 or 128" in act.help
