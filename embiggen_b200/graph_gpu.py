"""Graph ingest on the GPU through the C ABI (SURVEY.md 8(f) row 1).

``csr_from_edges_gpu`` builds the sorted, de-duplicated CSR the reference receives from an
``ensmallen.Graph`` (/root/reference/embiggen/embedders/pecanpy_embedders/node2vec.py:139-163)
out of a plain edge list; ``erdos_renyi_gpu`` / ``rmat_gpu`` generate the synthetic graphs of the
BASELINE.json shapes and return the same graphs as the numpy generators of
:mod:`embiggen_b200.graph` (same Philox stream, same "first m distinct edges in draw order"
rule), which is how the 200 M-edge configurations become practical.

Edge weights go through both: ``weights=`` (one float32 per input edge, never negative) gives the
weighted CSR of :func:`embiggen_b200.graph.csr_from_edges`, bit for bit, and a weighted
:class:`DeviceGraph` walks by weight without its weights ever leaving HBM.
"""
import ctypes
from typing import Optional

import numpy as np

from . import _lib
from ._lib import check
from .graph import CSRGraph


def _edge_list(src, dst, weights):
    src = np.ascontiguousarray(src, dtype=np.uint32)
    dst = np.ascontiguousarray(dst, dtype=np.uint32)
    if src.shape != dst.shape or src.ndim != 1:
        raise ValueError("src and dst must be 1-d arrays of the same length.")
    if weights is not None:
        weights = np.ascontiguousarray(weights, dtype=np.float32)
        if weights.shape != src.shape:
            raise ValueError("weights must have one entry per edge.")
    return src, dst, weights


def csr_from_edges_gpu(src, dst, n: int, symmetrise: bool = True, node_names=None,
                       name: str = "graph", device: int = 0, weights=None) -> CSRGraph:
    """Sorted, de-duplicated, self-loop-free CSR, equal to :func:`embiggen_b200.graph.csr_from_edges`
    (with ``weights``: a duplicated edge keeps the weight of its first occurrence; a negative or
    NaN weight raises ValueError)."""
    src, dst, weights = _edge_list(src, dst, weights)
    capacity = max(1, src.shape[0] * (2 if symmetrise else 1))
    indptr = np.empty(n + 1, dtype=np.int64)
    indices = np.empty(capacity, dtype=np.uint32)
    out_weights = None if weights is None else np.empty(capacity, dtype=np.float32)
    nnz = ctypes.c_uint64()
    check(_lib.load().b2e_csr_from_edges_weighted(
        device, src.ctypes.data, dst.ctypes.data, None if weights is None else weights.ctypes.data, src.shape[0], n,
        int(symmetrise), indptr.ctypes.data, indices.ctypes.data,
        None if out_weights is None else out_weights.ctypes.data, capacity, ctypes.byref(nnz)))
    return CSRGraph(indptr, indices[: nnz.value].copy(), node_names=node_names, name=name,
                    directed=not symmetrise, weights=None if weights is None else out_weights[: nnz.value].copy())


class DeviceGraph:
    """A CSR that lives in HBM (``b2e_graph``): built on the GPU and handed to an engine without
    ever crossing PCIe (``Engine.load_graph``; SURVEY.md 8(f) row 1).  It offers the accessors of
    ``ensmallen.Graph`` that the embedder path calls (the same subset as
    :class:`embiggen_b200.graph.CSRGraph`), so it can be passed to ``fit_transform`` directly;
    anything that needs the arrays on the host goes through :meth:`to_host`."""

    def __init__(self, handle: ctypes.c_void_p, device: int, name: str = "graph", directed: bool = False):
        self._lib = _lib.load()
        self._handle = handle
        self.device = device
        self._name = name
        self._directed = directed
        n, nnz = ctypes.c_uint64(), ctypes.c_uint64()
        check(self._lib.b2e_graph_shape(self._handle, ctypes.byref(n), ctypes.byref(nnz)))
        self._n, self._nnz = int(n.value), int(nnz.value)
        self._weighted = bool(self._lib.b2e_graph_weighted(self._handle))
        self._host: Optional[CSRGraph] = None

    def close(self) -> None:
        if self._handle:
            self._lib.b2e_graph_destroy(self._handle)
            self._handle = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def to_host(self) -> CSRGraph:
        if self._host is None:
            indptr = np.empty(self._n + 1, dtype=np.int64)
            indices = np.empty(max(self._nnz, 1), dtype=np.uint32)
            check(self._lib.b2e_graph_export(self._handle, indptr.ctypes.data, indices.ctypes.data))
            weights = self.get_directed_edge_weights() if self._weighted else None
            self._host = CSRGraph(indptr, indices[: self._nnz], name=self._name, directed=self._directed,
                                  weights=weights)
        return self._host

    # -- accessors mirrored from ensmallen.Graph (see CSRGraph) --
    def get_name(self) -> str:
        return self._name

    def get_number_of_nodes(self) -> int:
        return self._n

    def get_number_of_directed_edges(self) -> int:
        return self._nnz

    def has_nodes(self) -> bool:
        return self._n > 0

    def has_edges(self) -> bool:
        return self._nnz > 0

    def has_edge_weights(self) -> bool:
        return self._weighted

    def get_directed_edge_weights(self) -> np.ndarray:
        """The weight of every directed edge, in CSR order (a copy from HBM)."""
        if not self._weighted:
            raise ValueError("The graph has no edge weights.")
        weights = np.empty(max(self._nnz, 1), dtype=np.float32)
        check(self._lib.b2e_graph_export_weights(self._handle, weights.ctypes.data))
        return weights[: self._nnz]

    def has_negative_edge_weights(self) -> bool:
        """Always False: graph ingest refuses negative (and NaN) weights, so a resident graph never
        holds one."""
        return False

    def has_node_types(self) -> bool:
        return False

    def has_edge_types(self) -> bool:
        return False

    def is_directed(self) -> bool:
        return self._directed

    def get_node_names(self):
        return [str(i) for i in range(self._n)]

    def get_cumulative_node_degrees(self) -> np.ndarray:
        return self.to_host().get_cumulative_node_degrees()

    def get_directed_destination_node_ids(self) -> np.ndarray:
        return self.to_host().get_directed_destination_node_ids()

    def get_number_of_disconnected_nodes(self) -> int:
        return self.to_host().get_number_of_disconnected_nodes()

    def has_disconnected_nodes(self) -> bool:
        return self.get_number_of_disconnected_nodes() > 0


def device_graph_from_csr(indptr, indices, weights=None, name: str = "graph", device: int = 0) -> DeviceGraph:
    """Upload a host CSR once (to share it between several engines), with its edge weights if given
    (one per directed edge, never negative)."""
    indptr = np.ascontiguousarray(indptr, dtype=np.int64)
    indices = np.ascontiguousarray(indices, dtype=np.uint32)
    if weights is not None:
        weights = np.ascontiguousarray(weights, dtype=np.float32)
        if weights.shape != indices.shape:
            raise ValueError("weights must have one entry per directed edge.")
    handle = ctypes.c_void_p()
    check(_lib.load().b2e_graph_from_csr_weighted(device, indptr.ctypes.data, indices.ctypes.data,
                                                  None if weights is None else weights.ctypes.data,
                                                  indptr.shape[0] - 1, indices.shape[0], ctypes.byref(handle)))
    return DeviceGraph(handle, device, name=name)


def device_graph_from_edges(src, dst, n: int, symmetrise: bool = True, name: str = "graph",
                            device: int = 0, weights=None) -> DeviceGraph:
    """:func:`csr_from_edges_gpu`, but the CSR (and its weights) stays in HBM."""
    src, dst, weights = _edge_list(src, dst, weights)
    handle = ctypes.c_void_p()
    check(_lib.load().b2e_graph_from_edges_weighted(device, src.ctypes.data, dst.ctypes.data,
                                                    None if weights is None else weights.ctypes.data,
                                                    src.shape[0], n, int(symmetrise), ctypes.byref(handle)))
    return DeviceGraph(handle, device, name=name, directed=not symmetrise)


def _synthetic_resident(kind: int, n: int, scale: int, m: int, seed: int, thresholds, name: str,
                        device: int) -> DeviceGraph:
    handle = ctypes.c_void_p()
    check(_lib.load().b2e_graph_synthetic(device, kind, n, scale, m, seed, *thresholds, ctypes.byref(handle)))
    return DeviceGraph(handle, device, name=name)


def _synthetic(kind: int, n: int, scale: int, m: int, seed: int, thresholds, name: str,
               device: int) -> CSRGraph:
    indptr = np.empty(n + 1, dtype=np.int64)
    indices = np.empty(2 * m, dtype=np.uint32)
    nnz = ctypes.c_uint64()
    check(_lib.load().b2e_synthetic_csr(device, kind, n, scale, m, seed, *thresholds,
                                        indptr.ctypes.data, indices.ctypes.data, 2 * m,
                                        ctypes.byref(nnz)))
    assert nnz.value == 2 * m
    return CSRGraph(indptr, indices, name=name)


def erdos_renyi_gpu(n: int, m: int, seed: int = 42, device: int = 0, resident: bool = False):
    """G(n, m), identical to :func:`embiggen_b200.graph.erdos_renyi`; ``resident=True`` keeps the
    CSR in HBM and returns a :class:`DeviceGraph`."""
    build = _synthetic_resident if resident else _synthetic
    return build(0, n, 0, m, seed, (0, 0, 0), f"ER_{n}_{m}", device)


def rmat_gpu(scale: int, m: int, n: Optional[int] = None, seed: int = 42,
             probabilities=(0.57, 0.19, 0.19, 0.05), device: int = 0, resident: bool = False):
    """R-MAT, identical to :func:`embiggen_b200.graph.rmat`; ``resident=True`` keeps the CSR in HBM
    and returns a :class:`DeviceGraph`."""
    n = (1 << scale) if n is None else n
    a, b, c, _ = probabilities
    thresholds = (int(a * 2 ** 32), int((a + b) * 2 ** 32), int((a + b + c) * 2 ** 32))
    build = _synthetic_resident if resident else _synthetic
    return build(1, n, scale, m, seed, thresholds, f"RMAT_{scale}_{m}", device)
