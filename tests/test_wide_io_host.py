"""CPU-side checks of the width limits 1 <= in_dim <= 128 and 0 <= C <= 1024: the C ABI refuses wider shapes with
SCGIB_E_SHAPE before anything is launched, sizes its layouts for the new widths, and the module constructors raise before
any device work."""
import ctypes
import types

import pytest

from tests.test_abi import _lib

E_SHAPE = -2


def _dims(lib_mod, in_dim, hidden=64):
    return lib_mod.Dims(in_dim=in_dim, d_transfer=32, hidden=hidden, gin_layers=4, act_dtype=0)


def test_in_dim_limit_at_the_abi():
    L = _lib()
    lib = L.load()
    buf = ctypes.create_string_buffer(1 << 12)
    P = ctypes.c_void_p(ctypes.addressof(buf))           # stands in for every device pointer: nothing is dereferenced
    for F in (1, 37, 89, 128):
        d = _dims(L, F)
        assert lib.scgib_param_slots(ctypes.byref(d)) > 0, F
        sizes = (ctypes.c_int64 * lib.scgib_param_slots(ctypes.byref(d)))()
        assert lib.scgib_param_layout(ctypes.byref(d), None, sizes) > 0
        assert 32 * F in list(sizes), F                   # transfer_d.weight [32][F]
    for F in (0, 129, 256):
        d = _dims(L, F)
        assert lib.scgib_param_slots(ctypes.byref(d)) == E_SHAPE, F
        assert lib.scgib_param_layout(ctypes.byref(d), None, None) == E_SHAPE, F
        assert lib.scgib_pretrain_workspace_bytes(ctypes.byref(d), 4, 40, 80, 120, 200) == 0, F
    for F in (0, 129):
        assert lib.scgib_input_proj_fwd_f32(P, P, 10, F, 32, P, None) == E_SHAPE, F
        assert lib.scgib_input_proj_fwd_bf16(P, P, 10, F, 32, P, None) == E_SHAPE, F
        assert lib.scgib_transfer_bwd_f32(P, F, 1, P, 10, None, None, None, 0, None, None, None, P, P, 1 << 12, None) == E_SHAPE, F
    assert "in_dim <= 128" in lib.scgib_error_string(E_SHAPE).decode()


def test_head_output_limit_at_the_abi():
    L = _lib()
    lib = L.load()
    for H in (32, 64, 128):
        for C in (0, 64, 65, 617, 1024):
            sizes = (ctypes.c_int64 * L.FT_SLOTS)()
            assert lib.scgib_finetune_head_layout(H, C, None, sizes) > 0, (H, C)
            assert sizes[L.FT_SLOTS - 2] == C * H and sizes[L.FT_SLOTS - 1] == C
        assert lib.scgib_finetune_head_layout(H, 1025, None, None) == E_SHAPE, H
        assert lib.scgib_finetune_head_layout(H, -1, None, None) == E_SHAPE, H
        assert lib.scgib_finetune_head_workspace_bytes(H, 1025, 2, 100, 1000) == 0, H
    # the weight-gradient scratch holds the 64 row-split partials of dWp2 [C][H] (B >= 8192: atb_splits(B) = 64)
    for H, C in ((32, 1024), (64, 617), (64, 1024)):
        small = lib.scgib_finetune_head_workspace_bytes(H, 64, 1, 8300, 8300)
        wide = lib.scgib_finetune_head_workspace_bytes(H, C, 1, 8300, 8300)
        assert wide - small >= 64 * (C * H - 8 * H * H) * 4, (H, C)


def _args(**kw):
    a = types.SimpleNamespace(recons_type="adj", useAtt=1, readout_f="sum", d_transfer=32, device="cpu", batch_size=16,
                              task="graph_classification", dataset="Peptides-func", k_transition=1)
    a.__dict__.update(kw)
    return a


def test_module_constructors_refuse_wide_io(tmp_path):
    import models
    unused = str(tmp_path / "unused.pt")                 # never opened: the width check comes first
    with pytest.raises(NotImplementedError, match="in_dim"):
        models.Mainmodel(_args(), 129, hidden_dim=64, num_layers=4, num_heads=4, k_transition=1, encoder="GIN")
    with pytest.raises(NotImplementedError, match="in_dim"):
        models.Mainmodel(_args(), 0, hidden_dim=64, num_layers=4, num_heads=4, k_transition=1, encoder="GCN")
    with pytest.raises(NotImplementedError, match="in_dim"):
        models.Mainmodel_continue(_args(), 129, 64, 4, 4, 1, 1, unused, "GIN")
    with pytest.raises(NotImplementedError, match="in_dim"):
        models.Mainmodel_finetuning(_args(), 129, 64, 4, 4, 1, 10, unused, "GIN")
    with pytest.raises(NotImplementedError, match="outputs"):
        models.Mainmodel_finetuning(_args(), 9, 64, 4, 4, 1, 1025, unused, "GIN")
    with pytest.raises(NotImplementedError, match="in_dim"):
        models.Mainmodel_domainadapt(_args(), 129, 64, 4, 4, 1, 10, unused, "GraphSAGE")
    with pytest.raises(FileNotFoundError):               # the widest accepted shapes get as far as loading the checkpoint
        models.Mainmodel_finetuning(_args(), 128, 64, 4, 4, 1, 1024, unused, "GIN")


def test_padded_set2set_width_choice():
    from scgib_b200.engine import PaddedSet2Set
    with pytest.raises(NotImplementedError):
        PaddedSet2Set(129, device="cpu")
    with pytest.raises(NotImplementedError):
        PaddedSet2Set(0, device="cpu")
