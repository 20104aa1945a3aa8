"""ctypes binding of ``libgcnstring_b200.so`` (the C ABI in include/gcnstring_b200.h).

There is no CPU fallback: if the library has not been built (``__graft_entry__.build()`` /
``python gcn-string_b200/csrc/build.py``) loading raises, and every native op needs a CUDA
device.  Tensors cross the boundary as raw device pointers; anything exposing
``__dlpack__`` is unwrapped zero-copy through ``torch.from_dlpack``.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int32, c_int64, c_uint32, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgcnstring_b200.so")

GCS_OK = 0
WORKSPACE_SAMPLE_WEIGHTS = 1          # gcs_model_workspace_bytes_ex flag (GCS_WORKSPACE_SAMPLE_WEIGHTS)
_STATUS_EXC = {1: ValueError, 2: NotImplementedError, 3: MemoryError, 4: RuntimeError}


class ModelConfig(Structure):
    _fields_ = [("in_features", c_int32), ("output", c_int32), ("hidden", c_int32),
                ("message_passing", c_int32), ("pre_process", c_int32), ("post_process", c_int32),
                ("connectivity", c_int32), ("pool", c_int32), ("final_activation", c_int32),
                ("bn_momentum", c_float), ("bn_epsilon", c_float), ("aggregate", c_int32),
                ("loss", c_int32), ("huber_delta", c_float)]


class Dropout(Structure):
    """gcs_dropout: the dropout of one training-mode model call (csrc/dropout.cuh)."""
    _fields_ = [("rate", c_float), ("_pad", c_uint32), ("seed", c_uint64), ("step", c_uint64)]


class Batch(Structure):
    _fields_ = [("n_nodes", c_int64), ("nnz", c_int64), ("n_graphs", c_int32), ("rb_height", c_int32),
                ("rowptr", c_void_p), ("colidx", c_void_p), ("rowptr_t", c_void_p), ("colidx_t", c_void_p),
                ("graph_ptr", c_void_p), ("x", c_void_p), ("ldx", c_int64), ("y", c_void_p),
                ("seg_ids", c_void_p), ("rb4_blk_ptr", c_void_p), ("rb4_ent", c_void_p), ("rb4_blk_ptr_t", c_void_p), ("rb4_ent_t", c_void_p),
                ("max_graph_nodes", c_int32), ("reserved", c_int32), ("values", c_void_p), ("values_t", c_void_p),
                ("sample_weight", c_void_p)]


class GradClip(Structure):
    """gcs_grad_clip: clipping options and the device chunk table of one optimizer call."""
    _fields_ = [("mode", c_int32), ("clipvalue", c_float), ("clipnorm", c_float), ("n_chunks", c_int32),
                ("chunks", c_void_p), ("partials", c_void_p), ("chunk_base", c_int32), ("n_partials", c_int32)]


CLIP_VALUE, CLIP_NORM, CLIP_GLOBAL_NORM, CLIP_PARTIALS_READY = 1, 2, 4, 8     # gcs_clip_mode

P = c_void_p
I32, I64, F32, F64 = c_int32, c_int64, c_float, ctypes.c_double

# name -> (restype, argtypes); mirrors include/gcnstring_b200.h declaration by declaration.
PROTOTYPES = {
    "gcs_version": (c_int32, []),
    "gcs_last_error": (c_char_p, []),
    "gcs_device_sm_count": (c_int32, []),
    "gcs_set_allreduce_hook": (c_int32, [P, P, I32]),
    "gcs_batch_disjoint": (c_int32, [P, P, P, P, P, I32, I32, P, I32, I64, I64, P, P, P, P, P, P, P, P, P, P]),
    "gcs_gather_graphs": (c_int32, [P, I32, P, P, P, P, P, I32, I32, P, P, P, P, P, P, P]),
    "gcs_gather_node_rows": (c_int32, [P, I32, P, P, I32, P, P, P]),
    "gcs_coo_to_csr": (c_int32, [P, I64, I64, P, P, P, P]),
    "gcs_segment_ptr": (c_int32, [P, I64, I32, P, P, P]),
    "gcs_csr_is_symmetric": (c_int32, [P, P, I64, P, P]),
    "gcs_csr_transpose": (c_int32, [P, P, I64, I64, P, P, P, P]),
    "gcs_cast_f64_f32": (c_int32, [P, P, I64, P]),
    "gcs_linear_workspace_bytes": (c_int64, [I64, I32, I32]),
    "gcs_linear_fwd": (c_int32, [P, I64, P, P, P, I64, I64, I32, I32, P, I64, P]),
    "gcs_linear_bwd_weight_workspace_bytes": (c_int64, [I64, I32, I32]),
    "gcs_linear_bwd_weight": (c_int32, [P, I64, P, I64, P, P, I64, I32, I32, P, I64, P]),
    "gcs_linear_bwd_input": (c_int32, [P, I64, P, P, I64, I64, I32, I32, I32, P, I64, P]),
    "gcs_bn_workspace_bytes": (c_int64, [I64, I32]),
    "gcs_bn_stats": (c_int32, [P, I64, I64, I32, P, P, P, I64, P]),
    "gcs_bn_fold": (c_int32, [P, P, P, P, F32, F32, P, P, P, P, I32, P]),
    "gcs_bn_prelu_fwd": (c_int32, [P, I64, P, P, P, P, I64, I64, I32, P]),
    "gcs_bn_prelu_bwd": (c_int32, [P, I64, P, I64, P, P, P, P, P, F32, P, I64, P, P, P, P, I64, I32, P, I64, P]),
    "gcs_spmm_rb_workspace_bytes": (c_int64, [I64, I32]),
    "gcs_spmm_build_rb": (c_int32, [P, P, I64, I64, I32, P, P, P, I64, P]),
    "gcs_spmm_slab_stage_bytes": (c_int64, []),
    "gcs_spmm_sum_graphs": (c_int32, [P, I32, I32, P, P, P, P, I32, I64, P, I64, P, P, P, P, I64, P, I64, I32, P]),
    "gcs_spmm_rb4_workspace_bytes": (c_int64, [I64]),
    "gcs_spmm_build_rb4": (c_int32, [P, P, I64, I64, P, P, P, I64, P]),
    "gcs_spmm_sum": (c_int32, [P, P, P, P, I64, P, I64, P, P, P, P, I64, I32, P]),
    "gcs_contact_workspace_bytes": (I64, [I64]),
    "gcs_contact_map_rowptr": (c_int32, [P, P, I32, I64, ctypes.c_float, P, P, I64, P]),
    "gcs_contact_map_fill": (c_int32, [P, P, I32, I64, ctypes.c_float, P, P, P, P]),
    "gcs_link_pairs_offsets": (c_int32, [P, I32, P, P, I32, P, P, P, I64, P]),
    "gcs_link_pairs": (c_int32, [P, P, P, P, P, I32, P, P, P, P, I64, P, P, P, P, I64, P]),
    "gcs_spmm_aggregate_bwd": (c_int32, [P, P, P, P, P, P, I64, P, I64, I32, P, I64, P, P, P, P, I64, P, I64, P, I64, I32, P]),
    "gcs_spmm_aggregate": (c_int32, [P, P, P, P, P, I64, P, I64, P, P, P, P, I64, P, I64, I32, I32, P]),
    "gcs_segment_sum_fwd": (c_int32, [P, I64, P, I32, I32, P, I64, P]),
    "gcs_segment_sum_bwd": (c_int32, [P, I64, P, I32, I32, P, I64, P]),
    "gcs_segment_mean_fwd": (c_int32, [P, I64, P, I32, I32, P, I64, P]),
    "gcs_segment_mean_bwd": (c_int32, [P, I64, P, I32, I32, P, I64, P]),
    "gcs_attn_pool_workspace_bytes": (c_int64, [I64, I32, I32]),
    "gcs_attn_sum_pool_fwd": (c_int32, [P, I64, I64, P, P, I32, I32, P, I64, P, P, P, I64, P]),
    "gcs_attn_sum_pool_bwd": (c_int32, [P, I64, P, I64, I64, P, P, I32, I32, P, I64, P, P, P, I64, P, P, I64, P]),
    "gcs_softmax_xent": (c_int32, [P, P, I32, I32, P, P, P, F32, P]),
    "gcs_softmax_xent_workspace_bytes": (c_int64, [I64, I32]),
    "gcs_softmax_xent_ws": (c_int32, [P, P, I32, I32, P, P, P, F32, P, I64, P]),
    "gcs_sigmoid_bce_workspace_bytes": (c_int64, [I64, I32]),
    "gcs_sigmoid_bce": (c_int32, [P, P, I64, I32, P, P, P, F32, P, I64, P]),
    "gcs_regression_loss_workspace_bytes": (c_int64, [I64, I32]),
    "gcs_regression_loss": (c_int32, [I32, F32, P, P, I64, I32, P, P, P, F32, P, I64, P]),
    "gcs_weighted_loss_workspace_bytes": (c_int64, [I32, I64, I32]),
    "gcs_weighted_loss": (c_int32, [I32, I32, F32, P, P, P, I64, I32, P, P, P, F32, P, I64, P]),
    "gcs_sgd_step": (c_int32, [P, P, I64, F32, F32, P]),
    "gcs_adam_step": (c_int32, [P, P, P, P, I64, F64, F64, F64, F64, I64, F32, P]),
    "gcs_sgd_step_ex": (c_int32, [P, P, P, I64, F32, F32, I32, F32, POINTER(GradClip), P]),
    "gcs_adam_step_ex": (c_int32, [P, P, P, P, P, I64, F64, F64, F64, F64, I64, F32, POINTER(GradClip), P]),
    "gcs_grad_clip_partials": (c_int32, [P, I64, F32, POINTER(GradClip), P]),
    "gcs_comm_unique_id": (c_int32, [P]),
    "gcs_comm_init": (c_int32, [P, I32, I32, POINTER(c_void_p)]),
    "gcs_comm_destroy": (c_int32, [P]),
    "gcs_comm_rank": (c_int32, [P]),
    "gcs_comm_world_size": (c_int32, [P]),
    "gcs_allreduce_grads": (c_int32, [P, P, I64, P]),
    "gcs_allreduce_f64": (c_int32, [P, P, I64, P]),
    "gcs_model_train_step_dp": (c_int32, [POINTER(ModelConfig), P, P, POINTER(Batch), F32, P, P, P, P, I64, P, P, P, I32]),
    "gcs_model_num_params": (c_int64, [POINTER(ModelConfig)]),
    "gcs_model_num_state": (c_int64, [POINTER(ModelConfig)]),
    "gcs_model_workspace_bytes": (c_int64, [POINTER(ModelConfig), I64, I64, I32, I32]),
    "gcs_model_workspace_bytes_ex": (c_int64, [POINTER(ModelConfig), I64, I64, I32, I32, I32]),
    "gcs_model_forward": (c_int32, [POINTER(ModelConfig), P, P, POINTER(Batch), I32, P, P, I64, P]),
    "gcs_model_train_step": (c_int32, [POINTER(ModelConfig), P, P, POINTER(Batch), F32, P, P, P, P, I64, P]),
    "gcs_model_logits_offset": (c_int64, [POINTER(ModelConfig), I64, I32, I32]),
    "gcs_model_backward": (c_int32, [POINTER(ModelConfig), P, POINTER(Batch), P, P, P, I64, P]),
    "gcs_model_forward_ex": (c_int32, [POINTER(ModelConfig), P, P, POINTER(Batch), I32, P, P, I64, P, POINTER(Dropout)]),
    "gcs_model_train_step_ex": (c_int32, [POINTER(ModelConfig), P, P, POINTER(Batch), F32, P, P, P, P, I64, P,
                                          POINTER(Dropout)]),
    "gcs_model_train_step_dp_ex": (c_int32, [POINTER(ModelConfig), P, P, POINTER(Batch), F32, P, P, P, P, I64, P, P, P,
                                             I32, POINTER(Dropout)]),
    "gcs_model_backward_ex": (c_int32, [POINTER(ModelConfig), P, POINTER(Batch), P, P, P, I64, P, POINTER(Dropout)]),
    "gcs_spmm_edge_grad": (c_int32, [P, P, P, I64, P, I64, I32, P, I64, P, P, P, P, I64, P, I64, I32, P, I32, P]),
    "gcs_model_forward_attr": (c_int32, [POINTER(ModelConfig), P, P, POINTER(Batch), P, P, I64, P]),
    "gcs_model_input_grad": (c_int32, [POINTER(ModelConfig), P, POINTER(Batch), I32, P, P, I64, P, P, P, I64, P,
                                       POINTER(Dropout)]),
    "gcs_output_grad": (c_int32, [I32, P, P, I64, I32, P, P]),
}
# test/sweep hook, not part of the header
_DEBUG = {"gcs_debug_set_spmm_mode": (None, [I32]),
          "gcs_debug_set_param": (None, [I32, I32]),
          "gcs_debug_set_gemm_mode": (None, [I32]),
          "gcs_debug_launch_count": (ctypes.c_longlong, []),
          "gcs_debug_profile_begin": (None, []),
          "gcs_debug_profile_end": (c_int32, [ctypes.c_char_p, c_int32]),
          "gcs_debug_slab_timing": (None, [P]),
          "gcs_debug_prelu_branch": (c_int32, [P, I64, P, P, P, P, F32, I64, I32, P, P]),
          "gcs_debug_dropout_keep": (c_int32, [c_uint64, c_uint64, I32, I64, I32, F32, P, P]),
          "gcs_model_debug_block_buffers": (c_int32, [POINTER(ModelConfig), I64, I32, I32, POINTER(I64), POINTER(I64),
                                                      POINTER(I64), POINTER(I32)])}

_lib = None


def load() -> ctypes.CDLL:
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  gcn_string_b200 has no CPU fallback.")
    lib = ctypes.CDLL(os.environ.get("GCS_LIB_PATH", LIB_PATH))     # GCS_LIB_PATH: a kernel-variant build (scripts only)
    for table in (PROTOTYPES, _DEBUG):
        for name, (res, args) in table.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
    _lib = lib
    return lib


def check(status: int, what: str = "") -> None:
    if status != GCS_OK:
        msg = load().gcs_last_error().decode("utf-8", "replace")
        raise _STATUS_EXC.get(status, RuntimeError)(f"{what or 'gcnstring_b200'}: {msg} (status {status})")


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("gcn_string_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch


def as_tensor(obj):
    """Zero-copy view of ``obj`` as a torch tensor (torch tensor or any DLPack exporter)."""
    import torch
    if isinstance(obj, torch.Tensor):
        return obj
    if hasattr(obj, "__dlpack__"):
        return torch.from_dlpack(obj)
    raise TypeError(f"expected a torch tensor or a DLPack-capable object, got {type(obj).__name__}")


def ptr(t) -> int:
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return t.data_ptr()


def stream_ptr(stream=None) -> int:
    import torch
    s = stream if stream is not None else torch.cuda.current_stream()
    return s.cuda_stream


def model_config(cfg) -> ModelConfig:
    """params.GNNConfig -> C struct."""
    from .params import AGGREGATE, CONNECTIVITY, FINAL_ACT, POOL
    cfg.validate()
    return ModelConfig(cfg.in_features, cfg.output, cfg.hidden, cfg.message_passing, cfg.pre_process,
                       cfg.post_process, CONNECTIVITY[cfg.connectivity], POOL[cfg.pool],
                       FINAL_ACT[cfg.activation], cfg.bn_momentum, cfg.bn_epsilon, AGGREGATE[cfg.aggregate], 0, 1.0)


ALLREDUCE_FN = ctypes.CFUNCTYPE(c_int32, c_void_p, c_int64, c_void_p, c_void_p)
_hook_keepalive = {}


def set_allreduce_hook(fn, world_size: int = 1):
    """Install (or, with ``fn=None``, remove) the synchronised-BatchNorm hook of the calling thread.
    ``fn(device_ptr: int, n_doubles: int, stream: int) -> None`` must sum the fp64 buffer over all ranks in
    place, enqueued on ``stream``; exceptions are reported as a failed status of the native call."""
    import threading
    lib = load()
    key = threading.get_ident()
    if fn is None:
        check(lib.gcs_set_allreduce_hook(None, None, 1), "gcs_set_allreduce_hook")
        _hook_keepalive.pop(key, None)
        return

    def trampoline(buf, n, stream, _user):
        try:
            fn(int(buf), int(n), int(stream or 0))
            return 0
        except Exception:                          # never let an exception cross the C frames
            import traceback
            traceback.print_exc()
            return 1

    cfn = ALLREDUCE_FN(trampoline)
    _hook_keepalive[key] = cfn                     # the C side keeps a raw pointer to it
    check(lib.gcs_set_allreduce_hook(ctypes.cast(cfn, c_void_p), None, int(world_size)), "gcs_set_allreduce_hook")


def profile_begin():
    load().gcs_debug_profile_begin()


def profile_end():
    """{label: (count, total_ms)} of the ops timed since profile_begin()."""
    buf = ctypes.create_string_buffer(8192)
    load().gcs_debug_profile_end(buf, 8192)
    out = {}
    for item in buf.value.decode().split(";"):
        if item:
            label, count, ms = item.split(":")
            out[label] = (int(count), float(ms))
    return out
