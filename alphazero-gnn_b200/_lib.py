"""ctypes binding of libazgnn_b200.so (include/azgnn_b200.h).

There is no CPU fallback: if the library is missing `lib()` raises with the build command, and
every compute entry point needs a CUDA device (the kernels are sm_100a only).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("AZG_LIBRARY") or os.path.join(_HERE, "libazgnn_b200.so")  # AZG_LIBRARY: A/B builds

OK = 0
GAME_CONNECT4, GAME_TICTACTOE, GAME_FROZENLAKE = 0, 1, 2
EVAL_STD, EVAL_GNN = 1, 2
EVAL_FOLD = 4  # tensor-core path: output_transform.2 folded into the heads (opt-in, args.b200_fold_heads)
PREC_FP32, PREC_BF16X3, PREC_BF16, PREC_F16F8 = 0, 1, 2, 3
PREC_F16F8_KS = 4  # f16f8 operands, each F x F contraction accumulated in four K-quarters (a quarter of the accumulation error)
PREC_BF16X3_KS = 5  # the same K-split on the bf16x3 operands
PREC_AUTO = -1  # wrapper-level: the fastest precision whose probe batch stays inside the fp32 contract (nets.py)
PRECISIONS = {"fp32": PREC_FP32, "bf16x3": PREC_BF16X3, "bf16": PREC_BF16, "f16f8": PREC_F16F8, "f16f8ks": PREC_F16F8_KS, "bf16x3ks": PREC_BF16X3_KS,
              "auto": PREC_AUTO}
PACKED_AS = {PREC_F16F8_KS: PREC_F16F8, PREC_BF16X3_KS: PREC_BF16X3}  # precisions that read another precision's weight images
PRECISION_NAMES = {v: k for k, v in PRECISIONS.items()}
TAG_NONE, TAG_F32, TAG_PYFLOAT, TAG_PYINT = -1, 0, 1, 2
CELL_I8, CELL_I64, CELL_F32, CELL_F64 = 0, 1, 2, 3
# search semantics of the arena (args.b200_search_semantics): the reference's backup, or Q negated before the update
SEARCH_SEMANTICS = {"reference": 0, "alphazero": 1}

_vp, _i, _i64, _sz, _d = C.c_void_p, C.c_int, C.c_int64, C.c_size_t, C.c_double


class C4Params(C.Structure):
    _fields_ = [(k, _vp) for k in ("conv1_w", "conv1_b", "conv2_w", "conv2_b", "fc_policy_w", "fc_policy_b",
                                   "fc_value_w", "fc_value_b", "ot0_w", "ot0_b", "ot2_w", "ot2_b", "ot_packed")]


class TTTParams(C.Structure):
    _fields_ = [(k, _vp) for k in ("conv1_w", "conv1_b", "conv2_w", "conv2_b", "conv3_w", "conv3_b", "fc1_w", "fc1_b",
                                   "fc_policy_w", "fc_policy_b", "fc2_w", "fc2_b", "fc_value_w", "fc_value_b",
                                   "ot0_w", "ot0_b", "ot2_w", "ot2_b")]


_GNN_LAYER_FIELDS = ("att0_w", "att0_b", "att2_w", "att2_b", "upd0_w", "upd0_b", "upd2_w", "upd2_b", "gate_w", "gate_b")


class GNNLayerParams(C.Structure):
    _fields_ = [(k, _vp) for k in _GNN_LAYER_FIELDS]


class GNNLayerGrads(C.Structure):
    _fields_ = [(k, _vp) for k in _GNN_LAYER_FIELDS]


class FLParams(C.Structure):
    _fields_ = [("fe0_w", _vp), ("fe0_b", _vp), ("fe2_w", _vp), ("fe2_b", _vp), ("gnn_w", C.POINTER(_vp)),
                ("gnn_b", C.POINTER(_vp)), ("policy_w", _vp), ("policy_b", _vp), ("value_w", _vp), ("value_b", _vp)]


class MoveParams(C.Structure):
    _fields_ = [("G", _i), ("A", _i), ("T", _i)] + [(k, _vp) for k in (
        "n0", "greedy", "u_tie", "u_sample", "roots", "player", "slot", "n1", "q1", "t1", "v0", "actions", "h_states", "h_pi",
        "h_player", "h_int", "rec_ip", "rec_iv", "rec_ep", "rec_ev", "rec_evtag", "flags")]


# name -> (restype, argtypes); mirrors include/azgnn_b200.h one to one
SIGNATURES = {
    "azg_last_error": (C.c_char_p, []),
    "azg_abi_version": (_i, []),
    "azg_device_info": (_i, [C.POINTER(_i)] * 3),
    "azg_launch_count": (C.c_ulonglong, []),
    "azg_timing_enable": (_i, [_i]),
    "azg_timing_read": (_i, [_i, C.POINTER(_d), C.POINTER(_i)]),
    "azg_pack_boards": (_i, [_vp, _i, _i, _i64, _vp, _vp]),
    "azg_encode_planes": (_i, [_vp, _i, _i64, _vp, _vp]),
    "azg_fl_encode_graph": (_i, [_vp, _i, _i64, _vp, _vp, _vp]),
    "azg_c4_workspace_bytes": (_sz, [_i, _i64, _i, _i]),
    "azg_c4_forward": (_i, [C.POINTER(C4Params), _i, _vp, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "azg_c4_forward_dyn": (_i, [C.POINTER(C4Params), _i, _vp, _i64, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "azg_c4_packed_bytes": (_sz, [_i, _i]),
    "azg_c4_pack": (_i, [C.POINTER(C4Params), _i, _i, _vp, _sz, _vp]),
    "azg_tc_linear": (_i, [_vp, _vp, _vp, _vp, _i64, _i, _i, _i, _vp, _sz, _vp]),
    "azg_ttt_workspace_bytes": (_sz, [_i, _i64, _i]),
    "azg_ttt_forward": (_i, [C.POINTER(TTTParams), _i, _vp, _i64, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "azg_ttt_packed_bytes": (_sz, [_i, _i]),
    "azg_ttt_pack": (_i, [C.POINTER(TTTParams), _i, _i, _vp, _sz, _vp]),
    "azg_ttt_tc_workspace_bytes": (_sz, [_i, _i64, _i]),
    "azg_ttt_forward_tc": (_i, [C.POINTER(TTTParams), _vp, _i, _i, _vp, _i64, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "azg_fl_forward": (_i, [C.POINTER(FLParams), _i, _i, _i, _vp, _i64, _vp, _vp, _vp]),
    "azg_linear_f32": (_i, [_vp, _vp, _vp, _vp, _i64, _i, _i, _i, _vp]),
    "azg_gemm_f32": (_i, [_i, _i, _i64, _i, _i, _vp, _i64, _vp, _i64, _vp, _i64, C.c_float, _vp]),
    "azg_mul_f32": (_i, [_vp, _vp, _vp, _i64, _vp]),
    "azg_linear_backward": (_i, [_vp, _vp, _vp, _vp, _i64, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "azg_conv3x3_relu_forward": (_i, [_vp, _vp, _vp, _vp, _i64, _i, _i, _i, _i, _i, _vp]),
    "azg_conv3x3_relu_backward": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _i, _i, _i, _vp]),
    "azg_policy_value_loss": (_i, [_vp, _vp, _vp, _vp, _i, _i, C.c_float, _vp, _vp, _vp, _vp, _vp, _vp]),
    "azg_graph_mean_relu_forward": (_i, [_vp, _vp, _i64, _i, _vp, _vp]),
    "azg_graph_mean_relu_backward": (_i, [_vp, _vp, _vp, _i64, _i, _vp, _vp]),
    "azg_grid_aggregate_relu_forward": (_i, [_vp, _i64, _i, _i, _i, _vp, _vp]),
    "azg_grid_aggregate_relu_backward": (_i, [_vp, _vp, _i64, _i, _i, _i, _vp, _vp]),
    "azg_grid_packed_bytes": (_sz, [_i]),
    "azg_grid_tc_supported": (_i, [_i, _i, _i]),
    "azg_grid_pack_weights": (_i, [_vp, _i, _i, _vp, _vp]),
    "azg_grid_layer_tc_forward": (_i, [_vp, _vp, _vp, _i64, _i, _i, _i, _i, _vp, _vp]),
    "azg_grid_layer_tc_backward_input": (_i, [_vp, _vp, _vp, _i64, _i, _i, _i, _i, _vp, _vp]),
    "azg_selfplay_move": (_i, [C.POINTER(MoveParams), _vp]),
    "azg_emit_examples": (_i, [_i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "azg_gather_examples": (_i, [_i, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "azg_grid_dw_scratch_floats": (_sz, [_i]),
    "azg_grid_layer_tc_backward_weights": (_i, [_vp, _vp, _i64, _i, _i, _vp, _vp, _vp, _vp]),
    "azg_gnn_layer_saved_floats": (_sz, [_i, _i]),
    "azg_gnn_layer_scratch_floats": (_sz, [_i, _i]),
    "azg_gnn_layer_forward": (_i, [C.POINTER(GNNLayerParams), _vp, _vp, _i, _i, _vp, _vp, _vp]),
    "azg_gnn_layer_backward": (_i, [C.POINTER(GNNLayerParams), _vp, _vp, _i, _i, _vp, _vp, _vp, C.POINTER(GNNLayerGrads), _vp, _vp]),
    "azg_arena_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "azg_arena_create": (_i, [C.POINTER(_vp), _i, _i, _i, _i, _i, _d, _vp, _sz, C.c_char_p, _vp]),
    "azg_arena_destroy": (_i, [_vp]),
    "azg_arena_copy_from": (_i, [_vp, _vp, _vp]),
    "azg_arena_set_semantics": (_i, [_vp, _i]),
    "azg_arena_set_root_noise": (_i, [_vp, _vp, _d]),
    "azg_arena_draw_root_noise": (_i, [_vp, C.c_uint64, _vp, _d, _vp, _vp]),
    "azg_philox4x64": (_i, [C.c_uint64, _vp, _i64, _vp, _vp]),
    "azg_rollout_eval": (_i, [_i, _i, _vp, _vp, _i64, _vp, _i, C.c_uint64, _vp, _vp, _vp]),
    "azg_arena_action_size": (_i, [_vp]),
    "azg_arena_reset": (_i, [_vp, _vp, _i, _vp]),
    "azg_arena_set_roots": (_i, [_vp, _vp, _vp]),
    "azg_arena_get_roots": (_i, [_vp, _vp, _vp]),
    "azg_arena_begin": (_i, [_vp, _i, _vp]),
    "azg_arena_select": (_i, [_vp, _vp, _vp, _vp]),
    "azg_arena_expand_backup": (_i, [_vp, _vp, _vp, _vp]),
    "azg_arena_select_compact": (_i, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "azg_arena_expand_backup_compact": (_i, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "azg_arena_root_stats": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "azg_arena_advance": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "azg_arena_status": (_i, [_vp, _vp, _vp]),
    "azg_arena_export": (_i, [_vp, _i, C.POINTER(_i)] + [_vp] * 11),
    "azg_rules_eval": (_i, [_i, _i, C.c_char_p, _vp, _i64, _vp, _vp, _vp, _vp, _vp]),
}

_lib = None


def bind(cdll, names=None, rename=None):
    """Attach restype/argtypes from SIGNATURES to a loaded CDLL."""
    for name, (res, args) in SIGNATURES.items():
        if names is not None and name not in names:
            continue
        fn = getattr(cdll, rename(name) if rename else name)
        fn.restype, fn.argtypes = res, args
    return cdll


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is not built; run `python alphazero-gnn_b200/build.py` "
                               "(nvcc, sm_100a). There is no CPU fallback.")
        _lib = bind(C.CDLL(LIB_PATH))
        if _lib.azg_abi_version() != 3:
            raise RuntimeError("libazgnn_b200.so ABI version mismatch; rebuild")
    return _lib


def check(rc, cdll=None, err_fn="azg_last_error"):
    if rc != OK:
        msg = getattr(cdll or lib(), err_fn)()
        raise RuntimeError(f"libazgnn_b200 error {rc}: {msg.decode() if msg else '?'}")


def require_device():
    """Raise unless a compute-10.x CUDA device is current (no fallback path exists)."""
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("azgnn_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    maj, mnr, sms = _i(), _i(), _i()
    check(lib().azg_device_info(C.byref(maj), C.byref(mnr), C.byref(sms)))
    return maj.value, mnr.value, sms.value


def stream():
    import torch
    return _vp(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    return _vp(t.data_ptr()) if t is not None else _vp(None)
