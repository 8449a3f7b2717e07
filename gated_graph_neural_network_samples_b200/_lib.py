"""ctypes binding of include/ggnn_b200.h.  Fails loudly when the CUDA library is missing: there is no CPU
fallback on the product path."""
from __future__ import annotations

import ctypes as C
import os

from . import _build

c_i32p = C.POINTER(C.c_int32)
c_f32p = C.POINTER(C.c_float)


class GgnnConfig(C.Structure):
    _fields_ = [("hidden_size", C.c_int32), ("num_edge_types", C.c_int32), ("num_layers", C.c_int32),
                ("layer_timesteps", c_i32p), ("residual_offsets", c_i32p), ("residual_layers", c_i32p),
                ("use_edge_bias", C.c_int32), ("use_edge_msg_avg_aggregation", C.c_int32), ("cell", C.c_int32),
                ("activation", C.c_int32), ("precision", C.c_int32), ("device", C.c_int32),
                ("use_propagation_attention", C.c_int32)]


class GgnnLayerWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in
                ("edge_weights", "edge_biases", "gate_kernel", "gate_bias", "cand_kernel", "cand_bias", "edge_type_attention_weights",
                 "cand_hidden_bias")]


class GgnnReadoutTask(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("w_gate", "b_gate", "w_trans", "b_trans")]


class GgnnLayerGrads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in
                ("edge_weights", "edge_biases", "gate_kernel", "gate_bias", "cand_kernel", "cand_bias", "edge_type_attention_weights",
                 "cand_hidden_bias")]


# name -> (restype, argtypes): every symbol include/ggnn_b200.h declares
SYMBOLS = {
    "ggnn_create": (C.c_int, [C.POINTER(GgnnConfig), C.POINTER(C.c_void_p)]),
    "ggnn_destroy": (C.c_int, [C.c_void_p]),
    "ggnn_last_error": (C.c_char_p, [C.c_void_p]),
    "ggnn_set_weights": (C.c_int, [C.c_void_p, C.POINTER(GgnnLayerWeights), C.c_int32]),
    "ggnn_set_graph_sparse": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_void_p), c_i32p, C.c_void_p, C.c_void_p]),
    "ggnn_prepare_graph_sparse": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_void_p), c_i32p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "ggnn_set_graph_prepared": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "ggnn_free_prepared_graph": (C.c_int, [C.c_void_p]),
    "ggnn_prepared_graph_error": (C.c_char_p, [C.c_void_p]),
    "ggnn_host_prepare_graph_sparse": (C.c_int, [C.POINTER(GgnnConfig), C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_void_p), c_i32p, C.c_void_p,
                                                 C.POINTER(C.c_void_p)]),
    "ggnn_prepare_graph_dense": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.POINTER(C.c_void_p)]),
    "ggnn_host_prepare_graph_dense": (C.c_int, [C.POINTER(GgnnConfig), C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.POINTER(C.c_void_p)]),
    "ggnn_prepared_graph_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_int32), C.POINTER(C.c_int64),
                                           C.POINTER(C.c_int32), C.c_char_p, C.c_int32]),
    "ggnn_prepared_graph_arrays": (C.c_int, [C.c_void_p] + [C.c_void_p] * 6),
    "ggnn_prepared_graph_image": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "ggnn_set_graph_dense": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "ggnn_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ggnn_forward_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ggnn_run_sparse_host": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ggnn_run_dense_host": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ggnn_run_sparse_host_readout": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                               C.POINTER(GgnnReadoutTask), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ggnn_forward_host_async": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ggnn_sync_check": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ggnn_readout_set_graphs": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "ggnn_readout_forward": (C.c_int, [C.c_void_p] + [C.c_void_p] * 7 + [C.c_void_p]),
    "ggnn_readout_backward": (C.c_int, [C.c_void_p] + [C.c_void_p] * 12 + [C.c_void_p]),
    "ggnn_set_state_dropout": (C.c_int, [C.c_void_p, C.c_float, C.c_uint64]),
    "ggnn_state_dropout_mask": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_uint64, C.c_void_p]),
    "ggnn_set_save_for_backward": (C.c_int, [C.c_void_p, C.c_int32]),
    "ggnn_set_backward_precision": (C.c_int, [C.c_void_p, C.c_int32]),
    "ggnn_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(GgnnLayerGrads), C.c_int32, C.c_void_p, C.c_void_p]),
    "ggnn_num_messages": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "ggnn_get_csr": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ggnn_layer_state": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_void_p)]),
    "ggnn_copy_layer_state": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "ggnn_last_launch_count": (C.c_int, [C.c_void_p]),
    "ggnn_host_tile_plan": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_void_p), c_i32p, C.c_void_p, C.c_int32,
                                      C.c_void_p, C.c_char_p, C.c_int32]),
    "ggnn_host_target_csr": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(C.c_void_p), c_i32p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ggnn_host_stream_tables": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(C.c_void_p), c_i32p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32,
                                          C.c_void_p, C.POINTER(C.c_int32)]),
    "ggnn_debug_trace": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32]),
    "ggnn_debug_timestamps": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ggnn_plan_description": (C.c_char_p, [C.c_void_p]),
}

_lib = None


def load(build_if_missing: bool = True):
    """dlopen libggnn_b200.so (building it with nvcc first if it is absent/stale and nvcc is available)."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    if build_if_missing and _build.is_stale():
        try:
            _build.build()
        except Exception as ex:  # no nvcc on the box: use the shipped .so if there is one
            if not os.path.exists(path):
                raise RuntimeError("libggnn_b200.so is missing and could not be built: %s" % ex)
            import warnings
            warnings.warn("libggnn_b200.so is OLDER than its sources and could not be rebuilt (%s): running the stale binary" % str(ex)[:200])
    if not os.path.exists(path):
        raise RuntimeError("libggnn_b200.so not found at %s -- run `python -m gated_graph_neural_network_samples_b200._build`"
                           % path)
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
