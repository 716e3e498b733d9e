"""ctypes binding of the C-ABI CUDA library (`include/gadapt.h`).

The library is built ahead of time by `g_adaptivity_b200/build.py` into
`g_adaptivity_b200/libgadapt_b200.so`.  There is no fallback: if the library is missing or a
call fails, a `RuntimeError` is raised -- the product path never computes on the CPU.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
# GAD_LIB selects another build of the same library (kernel-variant experiments, scripts/kbench.py)
LIB_PATH = os.environ.get("GAD_LIB") or os.path.join(_HERE, "libgadapt_b200.so")

_lib = None
_lock = threading.Lock()

_p = C.c_void_p
_i = C.c_int
_i64 = C.c_int64
_f = C.c_float
_sz = C.c_size_t

_i32 = C.c_int32
_fp = C.c_void_p


class TrainDesc(C.Structure):
    """`gad_train_desc` of include/gadapt.h, field by field."""
    _fields_ = [
        ("ell_in", _fp), ("ell_out", _fp), ("tile_ptr", _fp), ("N", _i64),
        ("T", _i32), ("max_tile_nodes", _i32), ("max_deg", _i32),
        ("x_comp", _fp), ("f", _fp), ("uu", _fp), ("f_scale", _fp), ("uu_scale", _fp), ("target", _fp),
        ("dim", _i32), ("CE", _i32),
        ("Mu", _fp), ("tau", _fp), ("Lw", _i32), ("L", _i32), ("C", _i32), ("inv_temp", _f),
        ("loss_kind", _i32), ("grad_scale", _f), ("loss_scale", _f),
        ("states", _fp), ("gMu", _fp), ("g_tau", _fp), ("loss", _fp), ("x_phys", _fp),
        ("workspace", _fp), ("workspace_bytes", _sz),
        ("tail", _i32), ("counter", _fp),
        ("Wq", _fp), ("bq", _fp), ("Wk", _fp), ("gWq", _fp), ("gbq", _fp), ("gWk", _fp), ("gbk", _fp),
        ("params", _fp), ("grads", _fp), ("exp_avg", _fp), ("exp_avg_sq", _fp), ("n_params", _i64),
        ("lr", _f), ("beta1", _f), ("beta2", _f), ("eps", _f), ("weight_decay", _f), ("adam_grad_scale", _f),
        ("step", _fp), ("flags", _i32), ("trace", _fp),
        ("rank", _i32), ("world", _i32), ("peers", _fp), ("peer_seq", _fp), ("peer_timeout_ms", C.c_uint32),
    ]


class PipelineSlot(C.Structure):
    """`gad_pipeline_slot` of include/gadapt.h."""
    _fields_ = [("dev_inputs", _fp), ("bytes", _sz), ("graph_exec", _fp), ("loss_dev", _fp)]


class PipelineRelay(C.Structure):
    """`gad_pipeline_relay` of include/gadapt.h."""
    _fields_ = [("device", C.c_int), ("direct_bytes", C.c_size_t), ("stream", C.c_void_p), ("staging", C.c_void_p),
                ("staging_stride", C.c_size_t)]


# name -> (restype, argtypes); mirrors include/gadapt.h declaration by declaration
SIGNATURES = {
    "gad_version": (_i, []),
    "gad_last_error": (C.c_char_p, []),
    "gad_launch_count": (C.c_longlong, []),
    "gad_device_info": (_i, [C.POINTER(_i), C.POINTER(_i), C.POINTER(_i)]),
    "gad_graph_workspace_bytes": (_sz, [_i64, _i64, _i64, _i]),
    "gad_graph_build": (_i, [_p, _i64, _p, _p, _p, _p, _i64, _i, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "gad_graph_sort_rows": (_i, [_p, _p, _i64, _p, _p]),
    "gad_graph_check_tiles": (_i, [_p, _p, _i64, _p, _i, _p, _p]),
    "gad_edge_masks": (_i, [_p, _i64, _p, _i64, _p, _p, _p, _p, _p]),
    "gad_fingerprint": (_i, [_p, _sz, C.c_uint64, _p, _p]),
    "gad_prepare_weights": (_i, [_p, _p, _p, _i, _i, _i, _f, _p, _p]),
    "gad_weight_grads": (_i, [_p, _p, _p, _p, _i, _i, _i, _f, _p, _p, _p, _p, _p]),
    "gad_pack_features": (_i, [_p, _p, _p, _p, _p, _i64, _i, _i, _p, _p]),
    "gad_deform_workspace_bytes": (_sz, [_i64, _i, _i]),
    "gad_deform_fwd": (_i, [_p, _p, _i64, _i64, _p, _i, _i, _i, _p, _i, _i, _p, _i, _p, _i, _i, _p, _p, _p, _sz, _p]),
    "gad_deform_bwd_workspace_bytes": (_sz, [_i64, _i, _i, _i]),
    "gad_deform_bwd": (_i, [_p, _p, _p, _p, _i64, _i64, _p, _i, _i, _i, _p, _p, _i, _i, _p, _i, _p, _i, _p, _p, _p,
                            _p, _sz, _p]),
    "gad_graph_build_wide": (_i, [_p, _p, _i64, _p, _p, _p]),
    "gad_deform_bwd_wide_rk4_workspace_bytes": (_sz, [_i64, _i]),
    "gad_deform_bwd_wide_rk4": (_i, [_p, _p, _i64, _i, _p, _p, _i, _i, _p, _i, _p, _i, _p, _p, _p, _sz, _p]),
    "gad_wide_persist_nodes": (_i64, [_i, _i, _i64]),
    "gad_deform_fwd_wide": (_i, [_p, _i64, _i, _i64, _p, _i, _i, _p, _i, _p, _i, _i, _p, _p, _p, _sz, _p]),
    "gad_deform_bwd_wide": (_i, [_p, _p, _i64, _i, _p, _p, _i, _i, _p, _i, _p, _i, _p, _p, _p, _p, _sz, _p]),
    "gad_graph_build_ell": (_i, [_p, _p, _i64, _p, _i, _i, _i, _p, _p, _p]),
    "gad_ell_supported": (_i, [_i, _i, _i, _i]),
    "gad_ell_workspace_bytes": (_sz, [_i, _i, _i]),
    "gad_deform_fwd_ell": (_i, [_p, _i64, _p, _i, _i, _i, _p, _i, _i, _p, _i, _p, _i, _i, _p, _p, _p]),
    "gad_deform_fwd_ell_raw": (_i, [_p, _i64, _p, _i, _i, _i, _p, _p, _p, _p, _p, _i, _i, _p, _p, _i, _p, _i, _i, _p, _p, _p]),
    "gad_deform_bwd_ell": (_i, [_p, _p, _i64, _p, _i, _i, _i, _p, _p, _i, _i, _p, _p, _i, _p, _i, _p, _p, _p, _p, _sz, _p]),
    "gad_deform_bwd_ell_rk4": (_i, [_p, _p, _i64, _p, _i, _i, _i, _p, _p, _i, _i, _p, _p, _i, _p, _i, _p, _p, _p, _sz, _p]),
    "gad_ell_rk4_bwd_supported": (_i, [_i, _i, _i]),
    "gad_train_step_ell_rk4": (_i, [C.POINTER(TrainDesc), _p]),
    "gad_ell_rk4_train_supported": (_i, [_i, _i, _i]),
    "gad_deform_train_ell": (_i, [_p, _p, _i64, _p, _i, _i, _i, _p, _p, _p, _p, _p, _p, _i, _i, _p, _i, _p, _i, _i,
                                  _f, _f, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "gad_train_step_ell": (_i, [C.POINTER(TrainDesc), _p]),
    "gad_cluster_plan": (_i, [_i, _i, _i, C.POINTER(_i), C.POINTER(_i)]),
    "gad_deform_bwd_cluster": (_i, [_p, _p, _p, _i, _i, _i, _i, _i64, _p, _p, _i, _i, _p, _i, _p, _i, _p, _p, _p, _p, _sz, _p]),
    "gad_deform_fwd_cluster": (_i, [_p, _p, _i, _i, _i, _i, _i64, _p, _p, _p, _p, _p, _i, _i, _p, _i, _p, _i, _i, _p, _p, _p]),
    "gad_graph_build_cluster": (_i, [_p, _p, _p, _i, _i, _i, _i, _p, _p, _p]),
    "gad_cluster_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "gad_cluster_occupancy": (_i, [_i, _i, _i, _i, C.POINTER(_i)]),
    "gad_train_step_cluster": (_i, [C.POINTER(TrainDesc), _i, _p]),
    "gad_conv_fwd": (_i, [_p, _p, _p, _i64, _i64, _p, _i, _p, _p, _p, _p]),
    "gad_conv_bwd": (_i, [_p, _p, _p, _p, _i64, _i64, _p, _p, _i, _p, _p, _p, _p, _sz, _p]),
    "gad_mesh_loss": (_i, [_p, _p, _i64, _i, _f, _p, _p, _p, _p]),
    "gad_mesh_loss_workspace_bytes": (_sz, [_i64]),
    "gad_adam_step": (_i, [_p, _p, _p, _p, _i64, _f, _f, _f, _f, _f, _f, _p, _p]),
    "gad_fem1d_fwd": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _i, _p, _p, _p]),
    "gad_fem1d_bwd": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p, _p]),
    "gad_fem2d_fwd": (_i, [_p, _i, _p, _i, _p, _p, _i, _p, _p, _p, _i, _i, _i, _p, _p, _i, _p, _p, _p, _p, _p]),
    "gad_fem2d_bwd": (_i, [_p, _i, _p, _i, _p, _p, _i, _p, _p, _p, _i, _i, _i, _p, _p, _i, _p, _p, _p, _p]),
    "gad_peer_exchange_bytes": (_sz, [_i, _i64]),
    "gad_peer_alloc": (_i, [_sz, C.POINTER(_p), _p]),
    "gad_peer_open": (_i, [_p, C.POINTER(_p)]),
    "gad_peer_close": (_i, [_p]),
    "gad_peer_free": (_i, [_p]),
    "gad_cnn_param_count": (_i64, [_i, _i, _i, _i]),
    "gad_cnn_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i]),
    "gad_cnn_fwd": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _i, C.POINTER(_p), C.POINTER(_p), _p, _p, _sz, _p]),
    "gad_cnn_bwd": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _i, C.POINTER(_p), C.POINTER(_p), _p, _p, _p, _sz, _p]),
    "gad_host_alloc": (_i, [_sz, _i, C.POINTER(_p)]),
    "gad_host_free": (_i, [_p]),
    "gad_pipeline_run": (_i, [C.POINTER(PipelineSlot), _i, C.POINTER(_p), _i, _i64, _p, _p, _p]),
    "gad_pipeline_run_relay": (_i, [C.POINTER(PipelineSlot), _i, C.POINTER(_p), _i, _i64, _p, _p, _p,
                                    C.POINTER(PipelineRelay)]),
    "gad_enable_peer_access": (_i, [_i, _i]),
}


def load():
    """Load the shared library (once) and declare every entry point of `include/gadapt.h`."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m g_adaptivity_b200.build` "
                "(there is no CPU or PyTorch fallback for the deformer hot path)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError here == header and library out of sync
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().gad_last_error()
        raise RuntimeError(f"{what} failed (code {rc}): {msg.decode() if msg else '?'}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL).  The tensor must be contiguous."""
    if t is None:
        return None
    assert t.is_contiguous(), "gadapt kernels take contiguous tensors"
    return t.data_ptr()
