"""CPU-side checks of the fine-tuning / domain-adaptation surface for --encoder GraphSAGE / GCN: argument validation of the
logM loss operator and the eval-mode core gate (host code only, nothing is launched), and the wrapper construction rules
(which encoders the forward runs, the freeze rule, which path is selected)."""
import ctypes
import types

import pytest
import torch

from tests.test_abi import _lib

E_NULL, E_SHAPE, E_ALIGN, E_WORKSPACE, E_RANGE = -1, -2, -3, -4, -5


def _aligned(nbytes, align=256):
    buf = ctypes.create_string_buffer(nbytes + align)
    addr = ctypes.addressof(buf)
    return buf, ctypes.c_void_p(addr + (-addr) % align)


def test_recon_logm_argument_validation_without_gpu():
    L = _lib()
    lib = L.load()
    B, N, H = 3, 400, 64
    keep, p = _aligned(1 << 16)                       # stands in for every device pointer: nothing is dereferenced
    ws_need = lib.scgib_recon_logm_workspace_bytes(B, N, 2)
    assert ws_need > 0 and lib.scgib_recon_logm_workspace_bytes(B, N, 3) > ws_need
    for bad in ((0, N, 1), (B, 1, 1), (B, N, 0), (B, N, 9)):
        assert lib.scgib_recon_logm_workspace_bytes(*bad) == 0, bad
    ws_keep, ws = _aligned(ws_need)

    def call(Z=p, gp=p, ip=p, ix=p, B=B, N=N, H=H, k=2, loss=p, gZ=p, status=p, ws=ws, nbytes=ws_need):
        return lib.scgib_recon_logm_h_f32(Z, gp, ip, ix, B, N, H, k, 1.0, loss, gZ, status, ws, nbytes, None)

    assert call(H=96) == E_SHAPE
    assert call(H=32) == E_SHAPE
    assert call(k=0) == E_RANGE and call(k=9) == E_RANGE
    assert call(B=0) == E_RANGE and call(N=1) == E_RANGE
    for kw in ("Z", "gp", "ip", "ix", "loss", "status", "ws"):
        assert call(**{kw: None}) == E_NULL, kw
    assert call(Z=ctypes.c_void_p(p.value + 4)) == E_ALIGN
    assert call(gZ=ctypes.c_void_p(p.value + 8)) == E_ALIGN
    assert call(ws=ctypes.c_void_p(ws.value + 16)) == E_ALIGN
    assert call(nbytes=ws_need - 1) == E_WORKSPACE
    assert call(H=128, k=3, nbytes=ws_need) == E_WORKSPACE      # k = 3 needs one more [N] row of walk counts


def test_core_gate_eval_argument_validation_without_gpu():
    L = _lib()
    lib = L.load()
    B, N, H = 2, 20, 64
    keep, p = _aligned(1 << 16)
    need = lib.scgib_core_gate_workspace_bytes(H, B, N)
    assert need > 0

    def call(H=H, B=B, N=N, running=p, Hfeat=p, ws=p, nbytes=need):
        return lib.scgib_core_gate_eval_fwd_f32(Hfeat, p, B, N, H, p, p, p, p, p, p, running, p, p, p, p, p, p, p, ws, nbytes, None)

    assert call(H=96) == E_SHAPE
    assert call(B=0) == E_RANGE and call(N=1) == E_RANGE
    assert call(running=None) == E_NULL and call(Hfeat=None) == E_NULL and call(ws=None) == E_NULL
    assert call(running=ctypes.c_void_p(p.value + 4)) == E_ALIGN
    assert call(nbytes=need - 1) == E_WORKSPACE


def _args(**kw):
    a = types.SimpleNamespace(recons_type="adj", useAtt=1, readout_f="sum", d_transfer=32, device="cpu", batch_size=16,
                              task="graph_classification", dataset="Peptides-func", k_transition=1)
    a.__dict__.update(kw)
    return a


@pytest.mark.parametrize("encoder", ["GraphSAGE", "GCN"])
def test_wrappers_accept_sage_gcn_checkpoints(encoder, tmp_path):
    """Mainmodel_finetuning / Mainmodel_domainadapt around a GraphSAGE / GCN checkpoint: their own Encoder1/2 follow the
    encoder switch; the loaded module's encoders select the composed path (no GIN engine bridge); the freeze rule leaves
    no loaded parameter trainable in fine-tuning and all of them in domain adaptation."""
    import models
    pre = models.Mainmodel(_args(), 9, 64, 4, 4, 1, encoder)
    ckpt = str(tmp_path / "pre.pt")
    torch.save(pre, ckpt)
    ft = models.Mainmodel_finetuning(_args(), 9, 64, 4, 4, 1, 10, ckpt, encoder)
    assert type(ft.Encoder1).__name__ == encoder and ft.encoder_kind == encoder and ft._bridge is None
    trainable = sorted(n for n, p in ft.named_parameters() if p.requires_grad)
    assert not any(n.startswith("model.") for n in trainable)
    assert {"transfer_d.weight", "MLP.0.weight", "s2s.lstm.weight_ih_l0", "predict.2.bias"} <= set(trainable)
    da = models.Mainmodel_domainadapt(_args(), 9, 64, 4, 4, 1, 10, ckpt, encoder)
    assert da.encoder_kind == encoder and da._bridge is None
    assert all(p.requires_grad for p in da.model.parameters())
    # after domain adaptation, fine-tuning runs the adapter's own encoders (the loaded module's Encoder1 / Encoder2)
    da_ckpt = str(tmp_path / "da.pt")
    torch.save(da, da_ckpt)
    ft2 = models.Mainmodel_finetuning(_args(), 9, 64, 4, 4, 1, 10, da_ckpt, "GIN")
    assert ft2.encoder_kind == encoder and ft2._bridge is None and type(ft2.Encoder1).__name__ == "GIN"
    from scgib_b200.encoders import inner_of
    assert inner_of(ft2).Encoder1 is ft2.model.Encoder1
    # pickling round trip keeps the path
    again = pickle_roundtrip(ft, tmp_path)
    assert again._bridge is None and again.encoder_kind == encoder


def pickle_roundtrip(m, tmp_path):
    path = str(tmp_path / "rt.pt")
    torch.save(m, path)
    return torch.load(path, weights_only=False)


def test_wrappers_reject_unsupported_composed_width(tmp_path):
    import models
    with pytest.raises(NotImplementedError):
        models.Mainmodel_finetuning(_args(), 9, 96, 4, 4, 1, 10, str(tmp_path / "unused.pt"), "GraphSAGE")
