"""ctypes binding of ``libb2e.so`` (the C ABI declared in ``include/b2e.h``).

There is no CPU fallback: if the CUDA extension is missing, loading raises, and on a
machine without a B200 ``b2e_create`` fails with the library's error message.
"""
import ctypes
import os
from typing import List

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb2e.so")

ABI_VERSION = 3  # B2E_ABI_VERSION of include/b2e.h
B2E_OK = 0
B2E_ERR_INVALID = -1
B2E_ERR_CUDA = -2
B2E_ERR_STATE = -3

MODEL_IDS = {"skipgram": 0, "cbow": 1, "glove": 2}


class B2EConfig(ctypes.Structure):
    """Mirror of ``b2e_config`` (include/b2e.h)."""
    _fields_ = [
        ("struct_size", ctypes.c_uint32),
        ("model", ctypes.c_uint32),
        ("embedding_size", ctypes.c_uint32),
        ("epochs", ctypes.c_uint32),
        ("walk_length", ctypes.c_uint32),
        ("iterations", ctypes.c_uint32),
        ("window_size", ctypes.c_uint32),
        ("number_of_negative_samples", ctypes.c_uint32),
        ("clipping_value", ctypes.c_float),
        ("return_weight", ctypes.c_float),
        ("explore_weight", ctypes.c_float),
        ("learning_rate", ctypes.c_float),
        ("learning_rate_decay", ctypes.c_float),
        ("negative_sampling_exponent", ctypes.c_float),
        ("glove_alpha", ctypes.c_float),
        ("change_node_type_weight", ctypes.c_float),
        ("change_edge_type_weight", ctypes.c_float),
        ("use_scale_free_distribution", ctypes.c_uint32),
        ("normalize_learning_rate_by_degree", ctypes.c_uint32),
        ("normalize_by_degree", ctypes.c_uint32),
        ("stochastic_downsample_by_degree", ctypes.c_uint32),
        ("scale_by_sqrt_dim", ctypes.c_uint32),
        ("walklet_scale", ctypes.c_uint32),
        ("shared_negatives", ctypes.c_uint32),
        ("deterministic", ctypes.c_uint32),
        ("chunk_walks", ctypes.c_uint32),
        ("max_concurrent_walks", ctypes.c_uint32),
        ("device", ctypes.c_int32),
    ]


class B2EPerceptronConfig(ctypes.Structure):
    """Mirror of ``b2e_perceptron_config`` (include/b2e.h)."""
    _fields_ = [
        ("struct_size", ctypes.c_uint32),
        ("n_methods", ctypes.c_uint32),
        ("methods", ctypes.c_uint32 * 12),
        ("n_edge_features", ctypes.c_uint32),
        ("edge_features", ctypes.c_uint32 * 5),
        ("number_of_epochs", ctypes.c_uint32),
        ("number_of_edges_per_mini_batch", ctypes.c_uint32),
        ("learning_rate", ctypes.c_float),
        ("first_order_decay_factor", ctypes.c_float),
        ("second_order_decay_factor", ctypes.c_float),
        ("avoid_false_negatives", ctypes.c_uint32),
        ("use_scale_free_distribution", ctypes.c_uint32),
    ]


class B2ECounters(ctypes.Structure):
    """Mirror of ``b2e_counters`` (include/b2e.h)."""
    _fields_ = [
        ("walk_steps", ctypes.c_uint64),
        ("walk_trials", ctypes.c_uint64),
        ("walk_searches", ctypes.c_uint64),
        ("walk_probes", ctypes.c_uint64),
        ("walk_filter_rejects", ctypes.c_uint64),
        ("pairs", ctypes.c_uint64),
        ("targets", ctypes.c_uint64),
        ("loss_sum", ctypes.c_double),
    ]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


# every entry point include/b2e.h declares: name -> (restype, argtypes)
_H = ctypes.c_void_p
_U64, _U32, _F32 = ctypes.c_uint64, ctypes.c_uint32, ctypes.c_float
_P = ctypes.POINTER
SIGNATURES = {
    "b2e_last_error": (ctypes.c_char_p, []),
    "b2e_abi_version": (ctypes.c_int, []),
    "b2e_device_count": (ctypes.c_int, []),
    "b2e_select_device": (ctypes.c_int, [ctypes.c_int]),
    "b2e_create": (ctypes.c_int, [_P(B2EConfig), _P(_H)]),
    "b2e_destroy": (None, [_H]),
    "b2e_load_csr": (ctypes.c_int, [_H, ctypes.c_void_p, ctypes.c_void_p, _U64, _U64]),
    "b2e_load_csr_weighted": (ctypes.c_int, [_H, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, _U64,
                                             _U64]),
    "b2e_load_types": (ctypes.c_int, [_H, ctypes.c_void_p, ctypes.c_void_p]),
    "b2e_cooccurrence": (ctypes.c_int, [_H, _U64, _U64, _U64, _U64, ctypes.c_int, _P(_U64)]),
    "b2e_cooccurrence_export": (ctypes.c_int, [_H, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "b2e_glove_train": (ctypes.c_int, [_H, _F32]),
    "b2e_glove_walk_epoch": (ctypes.c_int, [_H, _U64, _U64, _U64]),
    "b2e_glove_shard_count": (ctypes.c_int, [_H, _U32, _U32, ctypes.c_void_p, _P(_U32)]),
    "b2e_glove_shard_train": (ctypes.c_int, [_H, _F32, _U32]),
    "b2e_glove_merge": (ctypes.c_int, [_H]),
    "b2e_number_of_sources": (_U64, [_H]),
    "b2e_row_stride": (_U64, [_H]),
    "b2e_fit": (ctypes.c_int, [_H, _U64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "b2e_walks": (ctypes.c_int, [_H, _U64, _U64, _U64, _U64, ctypes.c_void_p]),
    "b2e_slot_walks": (ctypes.c_int, [_H, _U32, _U64, ctypes.c_void_p]),
    "b2e_set_streams": (ctypes.c_int, [_H, ctypes.c_void_p, ctypes.c_void_p]),
    "b2e_init_tables": (ctypes.c_int, [_H, _U64]),
    "b2e_walk_chunk": (ctypes.c_int, [_H, _U64, _U64, _U64, _U64, _U32]),
    "b2e_adopt_walks": (ctypes.c_int, [_H, _H, _U32]),
    "b2e_train_chunk": (ctypes.c_int, [_H, _U64, _U32, _F32]),
    "b2e_train_host_walks": (ctypes.c_int, [_H, _U64, ctypes.c_void_p, _U64, _U64, _U64, _F32]),
    "b2e_sync": (ctypes.c_int, [_H]),
    "b2e_device_tables": (ctypes.c_int, [_H, _P(ctypes.c_void_p), _P(ctypes.c_void_p)]),
    "b2e_host_register": (ctypes.c_int, [ctypes.c_void_p, _U64]),
    "b2e_host_unregister": (ctypes.c_int, [ctypes.c_void_p]),
    "b2e_exchange_handles": (ctypes.c_int, [_H, ctypes.c_void_p]),
    "b2e_exchange_open": (ctypes.c_int, [_H, _U32, _U32, ctypes.c_void_p]),
    "b2e_exchange_open_local": (ctypes.c_int, [_H, _U32, _U32, _P(_H)]),
    "b2e_exchange_average": (ctypes.c_int, [_H]),
    "b2e_exchange_close": (ctypes.c_int, [_H]),
    "b2e_tables_digest": (ctypes.c_int, [_H, _P(ctypes.c_double), _P(_U64)]),
    "b2e_chunk_capacity": (ctypes.c_int, [_H, _P(_U64)]),
    "b2e_export_tables": (ctypes.c_int, [_H, ctypes.c_void_p, ctypes.c_void_p]),
    "b2e_import_tables": (ctypes.c_int, [_H, ctypes.c_void_p, ctypes.c_void_p]),
    "b2e_export_alias": (ctypes.c_int, [_H, ctypes.c_void_p, ctypes.c_void_p]),
    "b2e_export_edge_alias": (ctypes.c_int, [_H, ctypes.c_void_p]),
    "b2e_counters_read": (ctypes.c_int, [_H, _P(B2ECounters)]),
    "b2e_counters_reset": (ctypes.c_int, [_H]),
    "b2e_launch_count": (_U64, [_H]),
    "b2e_features_create": (ctypes.c_int, [ctypes.c_int, ctypes.c_void_p, _U64, _U32, _P(_H)]),
    "b2e_features_from_handle": (ctypes.c_int, [_H, ctypes.c_int, _P(_H)]),
    "b2e_features_destroy": (None, [_H]),
    "b2e_edge_embedding_size": (ctypes.c_int, [_U32, ctypes.c_void_p, _U32, ctypes.c_void_p, _U32, _P(_U32)]),
    "b2e_edge_metrics": (ctypes.c_int, [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, _U64, _U64, ctypes.c_void_p,
                                        ctypes.c_void_p, _U64, ctypes.c_void_p, _U32, ctypes.c_void_p]),
    "b2e_edge_embedding": (ctypes.c_int, [_H, ctypes.c_void_p, ctypes.c_void_p, _U64, ctypes.c_void_p, _U32,
                                          ctypes.c_void_p]),
    "b2e_perceptron_fit": (ctypes.c_int, [_H, ctypes.c_void_p, ctypes.c_void_p, _U64, _U64,
                                          _P(B2EPerceptronConfig), _U64, ctypes.c_void_p, ctypes.c_void_p]),
    "b2e_perceptron_predict": (ctypes.c_int, [_H, ctypes.c_void_p, ctypes.c_void_p, _U64, _U64, ctypes.c_void_p,
                                              ctypes.c_void_p, _U64, ctypes.c_void_p, _U32, ctypes.c_void_p, _U32,
                                              ctypes.c_void_p, ctypes.c_void_p]),
    "b2e_graph_from_edges": (ctypes.c_int, [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, _U64, _U64,
                                            ctypes.c_int, _P(_H)]),
    "b2e_graph_from_edges_weighted": (ctypes.c_int, [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                                     ctypes.c_void_p, _U64, _U64, ctypes.c_int, _P(_H)]),
    "b2e_graph_synthetic": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, _U64, _U32, _U64, _U64, _U64, _U64,
                                           _U64, _P(_H)]),
    "b2e_graph_from_csr": (ctypes.c_int, [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, _U64, _U64, _P(_H)]),
    "b2e_graph_from_csr_weighted": (ctypes.c_int, [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                                   ctypes.c_void_p, _U64, _U64, _P(_H)]),
    "b2e_graph_shape": (ctypes.c_int, [_H, _P(_U64), _P(_U64)]),
    "b2e_graph_export": (ctypes.c_int, [_H, ctypes.c_void_p, ctypes.c_void_p]),
    "b2e_graph_weighted": (ctypes.c_int, [_H]),
    "b2e_graph_export_weights": (ctypes.c_int, [_H, ctypes.c_void_p]),
    "b2e_graph_destroy": (None, [_H]),
    "b2e_load_graph": (ctypes.c_int, [_H, _H]),
    "b2e_csr_from_edges": (ctypes.c_int, [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, _U64, _U64,
                                          ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, _U64, _P(_U64)]),
    "b2e_csr_from_edges_weighted": (ctypes.c_int, [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                                   ctypes.c_void_p, _U64, _U64, ctypes.c_int, ctypes.c_void_p,
                                                   ctypes.c_void_p, ctypes.c_void_p, _U64, _P(_U64)]),
    "b2e_synthetic_csr": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, _U64, _U32, _U64, _U64, _U64, _U64,
                                         _U64, ctypes.c_void_p, ctypes.c_void_p, _U64, _P(_U64)]),
}

_lib = None


def exported_symbols() -> List[str]:
    return sorted(SIGNATURES)


def load() -> ctypes.CDLL:
    """Load libb2e.so; raises if the extension has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ModuleNotFoundError(
                f"The CUDA extension {LIB_PATH} is missing and there is no CPU fallback. "
                "Build it with `python -m embiggen_b200.build` (needs nvcc, targets sm_100a)."
            )
        lib = ctypes.CDLL(LIB_PATH)
        for name, (restype, argtypes) in SIGNATURES.items():
            function = getattr(lib, name)
            function.restype = restype
            function.argtypes = argtypes
        if lib.b2e_abi_version() != ABI_VERSION:
            raise ImportError("libb2e.so ABI version mismatch; rebuild the extension.")
        _lib = lib
    return _lib


def is_built() -> bool:
    return os.path.exists(LIB_PATH)


def check(status: int) -> None:
    """Convert a b2e_status into the Python exception the reference would raise."""
    if status == B2E_OK:
        return
    message = load().b2e_last_error().decode("utf-8", "replace")
    if status == B2E_ERR_INVALID:
        raise ValueError(message)
    raise RuntimeError(message)
