"""ctypes loader for libaqgnn.so (the C ABI of include/aqgnn.h).

There is no CPU fallback: if the shared library is missing or a kernel launch fails this raises.
"""
import ctypes
import os

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libaqgnn.so")
ABI_VERSION = 209 # AQ_VERSION of include/aqgnn.h this table of signatures was written for

# name -> (restype, argtypes); must list every symbol declared in include/aqgnn.h
_vp, _i64, _i32, _f32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_float
_f64, _u64 = ctypes.c_double, ctypes.c_uint64
SYMBOLS = {
    "aq_version": (_i32, []),
    "aq_last_error_string": (ctypes.c_char_p, []),
    "aq_launch_count": (_i64, []),
    "aq_pack_states": (_i32, [_vp, _vp, _i64, _vp, _vp]),
    "aq_unpack_states": (_i32, [_vp, _i64, _vp, _vp, _vp]),
    "aq_legal_mask": (_i32, [_vp, _i64, _vp, _vp, _vp]),
    "aq_legal_mask_ws_bytes": (_i64, [_i64]),
    "aq_legal_mask_ws": (_i32, [_vp, _i64, _vp, _vp, _vp, _i64, _vp]),
    "aq_legal_actions_list": (_i32, [_vp, _vp, _i64, _vp, _vp, _vp]),
    "aq_state_next": (_i32, [_vp, _vp, _i64, _vp, _vp, _vp]),
    "aq_build_graph": (_i32, [_vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    "aq_build_edge_index": (_i32, [_vp, _vp, _i64, _vp, _vp, _vp]),
    "aq_edges_to_open_mask": (_i32, [_vp, _vp, _i64, _i64, _vp, _vp, _vp]),
    "aq_param_count": (_i64, []),
    "aq_gnn_saved_floats": (_i64, [_i64]),
    "aq_gnn_forward": (_i32, [_vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _i32, _vp]),
    "aq_gcn_trunk_forward": (_i32, [_vp, _vp, _vp, _i64, _vp, _i32, _vp]),
    "aq_heads_forward": (_i32, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _i32, _vp]),
    "aq_prepared_bytes": (_i64, []),
    "aq_prepare_inference": (_i32, [_vp, _vp, _vp]),
    "aq_gnn_backward_ws_floats": (_i64, [_i64]),
    "aq_gnn_backward": (_i32, [_vp, _vp, _vp, _vp, _i64, _vp, _vp, _i32, _vp]),
    "aq_loss_grad": (_i32, [_vp, _vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp]),
    "aq_adam_step": (_i32, [_vp, _vp, _vp, _vp, _i64, _i64, _f32, _f32, _f32, _f32, _f32, _vp]),
    "aq_comm_create": (_i32, [_i32, _i32, ctypes.POINTER(ctypes.c_void_p), _vp]),
    "aq_comm_open": (_i32, [_vp, _vp]),
    "aq_comm_destroy": (_i32, [_vp]),
    "aq_comm_status": (_i32, [_vp, _vp, _vp]),
    "aq_comm_set_step": (_i32, [_vp, _i64, _f32, _f32, _vp]),
    "aq_dp_adam_step": (_i32, [_vp, _vp, _vp, _vp, _vp, _f32, _f32, _f32, _f32, _vp]),
    "aq_train_backward_step": (_i32, [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _i32, _f32, _f32, _f32, _f32, _vp]),
    "aq_leaf_eval": (_i32, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _i32, _vp]),
    "aq_leaf_eval_ws_floats": (_i64, [_i64]),
    "aq_leaf_eval_host_ws_bytes": (_i64, [_i64]),
    "aq_host_ctx_create": (_i32, [ctypes.POINTER(ctypes.c_void_p)]),
    "aq_host_ctx_destroy": (_i32, [_vp]),
    "aq_leaf_eval_host": (_i32, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp]),
    "aq_compact_priors": (_i32, [_vp, _vp, _vp, _i64, _vp, _vp, _vp]),
    "aq_leaf_eval_host_compact_ws_bytes": (_i64, [_i64]),
    "aq_leaf_eval_host_compact": (_i32, [_vp, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp]),
    "aq_leaf_eval_host_compact_submit": (_i32, [_vp, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp]),
    "aq_leaf_eval_host_compact_wait": (_i32, [_vp]),
    "aq_leaf_eval_host_compact_layout": (_i32, [_i64, _vp]),
    "aq_host_ctx_stats": (_i32, [_vp, _vp]),
    "aq_mcts_ws_bytes": (_i64, [_i64, _i64]),
    "aq_mcts_reset": (_i32, [_vp, _vp, _i64, _i64, _vp]),
    "aq_mcts_advance": (_i32, [_vp, _i64, _vp, _i64, _i64, _vp, _vp, _vp, _i32, _i64, _vp, _vp, _vp]),
    "aq_mcts_select": (_i32, [_vp, _i64, _i64, _f32, _vp, _vp, _vp]),
    "aq_mcts_expand_backup": (_i32, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "aq_mcts_expand_select": (_i32, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _f32, _vp, _vp, _vp]),
    "aq_mcts_gumbel_root": (_i32, [_vp, _i64, _i64, _vp, _u64, _i32, _i32, _f32, _i32, _vp, _vp]),
    "aq_mcts_select_gumbel": (_i32, [_vp, _i64, _i64, _f32, _vp, _vp, _vp]),
    "aq_mcts_expand_select_gumbel": (_i32, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _f32, _vp, _vp, _vp]),
    "aq_mcts_gumbel_result": (_i32, [_vp, _i64, _i64, _vp, _vp, _vp]),
    "aq_mcts_root_counts": (_i32, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "aq_mcts_root_values": (_i32, [_vp, _i64, _i64, _vp, _vp, _vp, _vp]),
    "aq_mcts_root_noise": (_i32, [_vp, _i64, _i64, _vp, _u64, _i32, _f32, _f32, _vp, _vp]),
    "aq_selfplay_ws_bytes": (_i64, [_i64]),
    "aq_selfplay_advance": (_i32, [_vp, _vp, _vp, _vp, _vp, _i64, _f64, _u64, _i32, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "aq_selfplay_advance_chosen": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "aq_selfplay_advance_resign": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _f64, _u64, _i32, _vp, _i32, _vp, _vp, _vp, _f64, _f64,
                                          _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "aq_shortest_paths": (_i32, [_vp, _i64, _vp, _vp, _vp, _vp]),
    "aq_negamax_backup": (_i32, [_vp, _vp, _i64, _vp, _vp, _vp, _vp]),
}

_lib = None


class AqError(RuntimeError):
    pass


def load(build_if_missing=True):
    """Load libaqgnn.so, (re)building it with nvcc if it is absent or older than its sources.  Raises if that is
    impossible, or if the library's ABI version is not the one this table of signatures was written for."""
    global _lib
    if _lib is not None:
        return _lib
    from . import build as _build
    stale = _build.needs_build()
    if stale:
        if not build_if_missing or _build.find_nvcc() is None:
            raise AqError(f"{LIB_PATH} is {'missing' if not os.path.exists(LIB_PATH) else 'older than csrc/ or include/aqgnn.h'}; "
                          "run `python -m alphaquoridorgnn_b200.build`")
        _build.build()
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError here = header/library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.aq_version() != ABI_VERSION:
        raise AqError(f"{LIB_PATH} has ABI version {lib.aq_version()}, the loader expects {ABI_VERSION}: rebuild the library")
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().aq_last_error_string().decode()
        raise AqError(f"{what} failed (code {rc}): {msg}")


def ptr(t):
    """Device (or host) pointer of a torch tensor / None."""
    if t is None:
        return None
    assert t.is_contiguous(), "libaqgnn expects contiguous tensors"
    return ctypes.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def capture_graph(device, enqueue, what):
    """Capture enqueue(stream pointer) into a CUDA graph on a side stream; -> the graph, or None, after a warning, when capture is
    not supported (the caller then runs eagerly).  `torch.cuda.graph` is not used on purpose: on entry it empties the caching
    allocator (the 3.5 GB workspace of a finished searcher goes back to the driver and the next one pays cudaMalloc again) --
    50-350 ms per capture on the boxes measured, and self-play captures once per batch size."""
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream(device=device)
    side.wait_stream(torch.cuda.current_stream(device))
    try:
        with torch.cuda.stream(side):
            g.capture_begin(capture_error_mode="thread_local")
            try:
                enqueue(stream_ptr(device))
            finally:
                g.capture_end()
    except AqError:
        raise
    except Exception as e:
        import warnings
        warnings.warn(f"CUDA-graph capture of {what} failed ({e!r}); running eagerly")
        torch.cuda.synchronize(device)
        return None
    torch.cuda.current_stream(device).wait_stream(side)
    return g


def require_cuda(t, name):
    if not t.is_cuda:
        raise AqError(f"{name} must be a CUDA tensor: the AlphaQuoridorGNN hot path has no CPU fallback")
