"""ctypes binding of libscgib.so (C ABI: include/scgib.h).

There is no CPU or PyTorch fallback: if the shared library is missing every entry point raises.
"""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_int64, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libscgib.so")


class Dims(ctypes.Structure):
    _fields_ = [("in_dim", c_int32), ("d_transfer", c_int32), ("hidden", c_int32), ("gin_layers", c_int32),
                ("act_dtype", c_int32)]          # ACT_F32 / ACT_BF16


class Batch(ctypes.Structure):
    _fields_ = [("struct_size", c_int32), ("B", c_int32), ("N", c_int32), ("E", c_int32), ("Ns", c_int32), ("Es", c_int32),
                ("graph_ptr", c_void_p), ("indptr", c_void_p), ("indices", c_void_p),
                ("ego_ptr", c_void_p), ("ego_nodes", c_void_p), ("ego_seed", c_void_p),
                ("sub_indptr", c_void_p), ("sub_indices", c_void_p),
                ("x", c_void_p), ("normalize_x", c_int32), ("gate_u", c_void_p), ("feat_u", c_void_p),
                ("t_override", c_void_p), ("eval_mode", c_int32), ("recon_logm_steps", c_int32)]


ACT_F32, ACT_BF16 = 0, 1
# slot enums of include/scgib.h
ENC_W1, ENC_B1, ENC_W2, ENC_B2, ENC_GAMMA, ENC_BETA, ENC_SLOTS = range(7)
(P_HEAD_W1, P_HEAD_B1, P_HEAD_W2, P_HEAD_B2, P_COMP_W1, P_COMP_B1, P_COMP_GAMMA, P_COMP_BETA, P_COMP_W2,
 P_COMP_B2, P_ATTN_W, P_ATTN_B, P_TRANSFER, P_ENC) = range(14)
EGO_CAP = 128
FT_SLOTS = 8

_SIGNATURES = {
    "scgib_version": (c_int, []),
    "scgib_error_string": (c_char_p, [c_int]),
    "scgib_num_sms": (c_int, []),
    "scgib_batch_abi_size": (c_int32, []),
    "scgib_param_layout": (c_int64, [POINTER(Dims), POINTER(c_int64), POINTER(c_int64)]),
    "scgib_param_slots": (c_int32, [POINTER(Dims)]),
    "scgib_ego_workspace_bytes": (c_size_t, [c_int32]),
    "scgib_ego_count": (c_int, [c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p,
                                c_size_t, c_void_p]),
    "scgib_ego_fill": (c_int, [c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p,
                               c_void_p, c_void_p, c_void_p]),
    "scgib_batch_workspace_bytes": (c_size_t, [c_int32]),
    "scgib_batch_assemble_count": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_size_t,
                                           c_void_p]),
    "scgib_batch_assemble_fill": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_int32, c_void_p,
                                          c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "scgib_batch_validate": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    "scgib_pretrain_workspace_bytes": (c_size_t, [POINTER(Dims), c_int32, c_int32, c_int32, c_int32, c_int32]),
    "scgib_pretrain_forward_f32": (c_int, [POINTER(Dims), c_void_p, c_void_p, POINTER(Batch), c_void_p, c_void_p,
                                           c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "scgib_pretrain_backward_f32": (c_int, [POINTER(Dims), c_void_p, POINTER(Batch), POINTER(c_float), c_void_p,
                                            c_void_p, c_size_t, c_void_p]),
    "scgib_extract_backward_f32": (c_int, [POINTER(Dims), c_void_p, POINTER(Batch), c_void_p, c_void_p, c_void_p,
                                           c_size_t, c_void_p]),
    "scgib_extract_forward_f32": (c_int, [POINTER(Dims), c_void_p, c_void_p, POINTER(Batch), c_void_p, c_void_p, c_void_p,
                                          c_void_p, c_void_p, c_size_t, c_void_p]),
    "scgib_finetune_head_layout": (c_int64, [c_int32, c_int32, POINTER(c_int64), POINTER(c_int64)]),
    "scgib_finetune_head_workspace_bytes": (c_size_t, [c_int32, c_int32, c_int32, c_int32, c_int32]),
    "scgib_finetune_head_fwd_f32": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_int32,
                                            c_int32, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "scgib_finetune_head_bwd_f32": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_int32,
                                            c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t,
                                            c_void_p]),
    "scgib_adam_step_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_float, c_float,
                                    c_float, c_float, c_float, c_float, c_void_p]),
    "scgib_peer_alloc": (c_int, [c_size_t, POINTER(c_void_p), c_char_p]),
    "scgib_peer_open": (c_int, [c_char_p, POINTER(c_void_p)]),
    "scgib_peer_close": (c_int, [c_void_p]),
    "scgib_peer_free": (c_int, [c_void_p]),
    "scgib_allreduce_adam_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, POINTER(c_void_p), POINTER(c_void_p), c_int32,
                                         c_int32, ctypes.c_uint32, c_int64, c_float, c_float, c_float, c_float, c_float,
                                         c_void_p]),
    "scgib_input_proj_fwd_f32": (c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    "scgib_gin_workspace_bytes": (c_size_t, [c_int32]),
    "scgib_gin_layer_fwd_f32": (c_int, [c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_int32,
                                        c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                        c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "scgib_gin_layer_bwd_workspace_bytes": (c_size_t, [c_int32, c_int32]),
    "scgib_gin_layer_bwd_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p,
                                        c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                        c_void_p, c_size_t, c_void_p]),
    "scgib_gin_layer_fwd_bf16_workspace_bytes": (c_size_t, [c_int32, c_int32]),
    "scgib_gin_layer_fwd_bf16": (c_int, [c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_int32,
                                         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "scgib_gin_layer_bwd_bf16_workspace_bytes": (c_size_t, [c_int32, c_int32, c_int32]),
    "scgib_gin_layer_bwd_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p,
                                         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "scgib_loss_workspace_bytes": (c_size_t, [c_int32]),
    "scgib_recon_adj_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_float, c_void_p, c_void_p, c_void_p,
                                    c_size_t, c_void_p]),
    "scgib_contrastive_f32": (c_int, [c_void_p, c_void_p, c_int32, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t,
                                      c_void_p]),
    "scgib_loss_workspace_bytes_h": (c_size_t, [c_int32, c_int32]),
    "scgib_recon_adj_h_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_float, c_void_p, c_void_p, c_void_p,
                                      c_size_t, c_void_p]),
    "scgib_contrastive_h_f32": (c_int, [c_void_p, c_void_p, c_int32, c_int32, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t,
                                        c_void_p]),
    "scgib_recon_logm_workspace_bytes": (c_size_t, [c_int32, c_int32, c_int32]),
    "scgib_recon_logm_h_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_float, c_void_p,
                                       c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "scgib_segment_sum_f32": (c_int, [c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_void_p]),
    "scgib_core_gate_workspace_bytes": (c_size_t, [c_int32, c_int32, c_int32]),
    "scgib_core_gate_fwd_f32": (c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int32] + [c_void_p] * 13 + [c_void_p, c_size_t, c_void_p]),
    "scgib_core_gate_bwd_f32": (c_int, [c_void_p, c_int32, c_int32, c_int32] + [c_void_p] * 8 + [c_float] + [c_void_p] * 7 +
                                [c_void_p, c_size_t, c_void_p]),
    "scgib_core_gate_eval_fwd_f32": (c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int32] + [c_void_p] * 14 +
                                     [c_void_p, c_size_t, c_void_p]),
    "scgib_core_gate_ema_f32": (c_int, [c_int32, c_int32, c_int32, c_void_p, c_void_p, c_size_t, c_void_p]),
    "scgib_core_cand_attn_fwd_f32": (c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p]),
    "scgib_core_cand_attn_bwd_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p,
                                             c_void_p, c_void_p, c_size_t, c_void_p]),
    "scgib_head_mlp_workspace_bytes": (c_size_t, [c_int32, c_int32]),
    "scgib_head_mlp_fwd_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int32] + [c_void_p] * 6 + [c_void_p, c_size_t, c_void_p]),
    "scgib_head_mlp_bwd_f32": (c_int, [c_void_p, c_void_p, c_int32, c_int32] + [c_void_p] * 7 + [c_void_p, c_size_t, c_void_p]),
    "scgib_segment_sum_bwd_f32": (c_int, [c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p]),
    "scgib_graph_aggregate_f32": (c_int, [c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p,
                                          c_void_p, c_void_p]),
    "scgib_segment_sum_w_f32": (c_int, [c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p]),
    "scgib_linear_fwd_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                                     c_int32, c_int32, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    "scgib_linear_bwd_w_workspace_bytes": (c_size_t, [c_int32, c_int32, c_int32]),
    "scgib_linear_bwd_w_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32,
                                       c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "scgib_transfer_bwd_workspace_bytes": (c_size_t, [c_int32, c_int32, c_int32]),
    "scgib_transfer_bwd_f32": (c_int, [c_void_p, c_int32, c_int32, c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_int32,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "scgib_transfer_bwd_workspace_bytes_d": (c_size_t, [c_int32, c_int32, c_int32, c_int32]),
    "scgib_transfer_bwd_d_f32": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_int32, c_void_p, c_void_p, c_void_p,
                                         c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "scgib_input_proj_fwd_bf16": (c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    "scgib_input_proj_fwd_d_bf16": (c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    "scgib_f32_to_bf16": (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    "scgib_graph_aggregate_bf16": (c_int, [c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p,
                                           c_void_p, c_int32, c_void_p]),
    "scgib_linear_fwd_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                                      c_int32, c_int32, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_int32, c_void_p]),
    "scgib_linear_bwd_w_bf16_workspace_bytes": (c_size_t, [c_int32, c_int32, c_int32]),
    "scgib_linear_bwd_w_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32,
                                        c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "scgib_profile_enable": (None, [c_int]),
    "scgib_profile_count": (c_int, []),
    "scgib_profile_get": (c_int, [c_int, POINTER(c_char_p), POINTER(c_float)]),
    "scgib_pretrain_workspace_offset": (c_int64, [POINTER(Dims), c_int32, c_int32, c_int32, c_int32, c_int32, c_char_p]),
}
EXPORTS = tuple(_SIGNATURES)          # exactly the entry points include/scgib.h declares (tests/test_abi.py)
# csrc/scgib_private.h: implementation selection / role-timeline dumps (tests and experiments only)
_PRIVATE_SIGNATURES = {
    "scgib_set_tensor_cores": (None, [c_int]),
    "scgib_set_tensor_cores_bwd": (None, [c_int]),
    "scgib_debug_tc2_trace": (c_int, [c_void_p, c_int]),
    "scgib_debug_bf16_trace": (c_int, [c_void_p, c_int]),
    "scgib_debug_bwdh_trace": (c_int, [c_void_p, c_int]),
}

_lib = None


def load():
    """Load libscgib.so once.  Raises (never falls back) when it is missing or incomplete."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libscgib.so not found at %s - build it with `python s-cgib_b200/build.py` "
            "(or __graft_entry__.build()).  scgib_b200 has no CPU/PyTorch fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in list(_SIGNATURES.items()) + list(_PRIVATE_SIGNATURES.items()):
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().scgib_error_string(int(rc)).decode()
        raise RuntimeError("libscgib %s failed: %s (code %d)" % (what, msg, rc))


def ptr(t):
    """Device/host pointer of a torch tensor (None -> NULL)."""
    return None if t is None else c_void_p(t.data_ptr())
