"""ctypes binding of the CPU oracle (``oracle/liboracle.so``).

TEST INFRASTRUCTURE.  Only ``tests/``, ``__graft_entry__.smoke()`` and
``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs may import this
package; ``embiggen_b200`` never does.  PARITY UNPINNED against Ensmallen, see
``oracle/oracle.h`` for what the oracle is pinned against instead.
"""
import ctypes
import os
import subprocess
from typing import Optional, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "liboracle.so")
_lib = None

PAD_TOKEN = 0xFFFFFFFF


class WalkCounters(ctypes.Structure):
    _fields_ = [
        ("steps", ctypes.c_uint64),
        ("trials", ctypes.c_uint64),
        ("first_order", ctypes.c_uint64),
        ("searches", ctypes.c_uint64),
        ("probe_sectors", ctypes.c_uint64),
        ("capped", ctypes.c_uint64),
    ]

    def as_dict(self):
        return {name: int(getattr(self, name)) for name, _ in self._fields_}


class SgnsCfg(ctypes.Structure):
    _fields_ = [
        ("model", ctypes.c_uint32),
        ("embedding_size", ctypes.c_uint32),
        ("row_stride", ctypes.c_uint32),
        ("walk_length", ctypes.c_uint32),
        ("window_size", ctypes.c_uint32),
        ("negatives", ctypes.c_uint32),
        ("clipping_value", ctypes.c_float),
        ("learning_rate", ctypes.c_float),
        ("use_alias", ctypes.c_uint32),
        ("normalize_learning_rate_by_degree", ctypes.c_uint32),
        ("scale_by_sqrt_dim", ctypes.c_uint32),
        ("downsample_bound", ctypes.c_uint32),
        ("fast_math", ctypes.c_uint32),
        ("shared_negatives", ctypes.c_uint32),
    ]


def build(force: bool = False) -> str:
    """Compile the oracle with the committed Makefile (gcc only)."""
    sources = [os.path.join(_HERE, f) for f in os.listdir(_HERE) if f.endswith((".c", ".h"))]
    stale = not os.path.exists(_LIB_PATH) or any(
        os.path.getmtime(s) > os.path.getmtime(_LIB_PATH) for s in sources
    )
    if force or stale:
        subprocess.run(["make", "-C", _HERE, "-B", "liboracle.so"], check=True,
                       stdout=subprocess.DEVNULL)
    return _LIB_PATH


def _ptr(array, ctype):
    return None if array is None else array.ctypes.data_as(ctypes.POINTER(ctype))


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        l = ctypes.CDLL(_LIB_PATH)
        u64, u32, f32 = ctypes.c_uint64, ctypes.c_uint32, ctypes.c_float
        P = ctypes.POINTER
        l.orc_philox.restype = None
        l.orc_philox.argtypes = [u64, u32, u32, u32, u32, P(u32)]
        l.orc_sources.restype = u64
        l.orc_sources.argtypes = [P(ctypes.c_int64), u64, P(u32)]
        l.orc_thresholds.restype = None
        l.orc_thresholds.argtypes = [f32, f32, P(u64)]
        l.orc_walks.restype = ctypes.c_int
        l.orc_walks.argtypes = [P(ctypes.c_int64), P(u32), u64, P(u32), u64, u64, u64, u64, u64,
                                u32, f32, f32, ctypes.c_int, P(u32), P(WalkCounters)]
        l.orc_is_undirected.restype = ctypes.c_int
        l.orc_is_undirected.argtypes = [P(ctypes.c_int64), P(u32), u64]
        l.orc_fold_thresholds.restype = None
        l.orc_fold_thresholds.argtypes = [f32, f32, P(u64), P(u64)]
        l.orc_edge_alias.restype = ctypes.c_int
        l.orc_edge_alias.argtypes = [P(ctypes.c_int64), P(f32), u64, P(u32)]
        l.orc_walks_weighted.restype = ctypes.c_int
        l.orc_walks_weighted.argtypes = [P(ctypes.c_int64), P(u32), P(u32), u64, P(u32), u64, u64, u64,
                                         u64, u64, u32, f32, f32, ctypes.c_int, P(u32), P(WalkCounters)]
        l.orc_walks_typed.restype = ctypes.c_int
        l.orc_walks_typed.argtypes = [P(ctypes.c_int64), P(u32), P(u32), P(u32), P(u32), f32, f32,
                                      u64, P(u32), u64, u64, u64, u64, u64, u32, f32, f32, ctypes.c_int,
                                      P(u32), P(WalkCounters)]
        l.orc_philox_range.restype = None
        l.orc_philox_range.argtypes = [u64, u32, u64, u32, u32, u32, P(u32)]
        l.orc_log_det.restype = f32
        l.orc_log_det.argtypes = [f32]
        l.orc_exp_det.restype = f32
        l.orc_exp_det.argtypes = [f32]
        l.orc_glove_train.restype = ctypes.c_int
        l.orc_glove_train.argtypes = [P(u32), P(u32), P(u32), u64, u32, u32, u32, f32, f32, f32,
                                      ctypes.c_int, P(f32), P(f32), P(ctypes.c_double), P(u64)]
        l.orc_alias_build.restype = ctypes.c_int
        l.orc_alias_build.argtypes = [P(ctypes.c_int64), u64, ctypes.c_double, P(u32), P(u32)]
        l.orc_set_threads.restype = None
        l.orc_set_threads.argtypes = [ctypes.c_int]
        l.orc_get_threads.restype = ctypes.c_int
        l.orc_sigmoid.restype = f32
        l.orc_sigmoid.argtypes = [f32]
        l.orc_dot.restype = f32
        l.orc_dot.argtypes = [P(f32), P(f32), u32]
        l.orc_init_tables.restype = ctypes.c_int
        l.orc_init_tables.argtypes = [u64, u32, u32, u64, P(f32), P(f32)]
        l.orc_train.restype = ctypes.c_int
        l.orc_train.argtypes = [P(SgnsCfg), P(u32), u64, u64, u64, u64, u64, P(ctypes.c_int64),
                                P(u32), P(u32), P(f32), P(f32), P(ctypes.c_double), P(u64), P(u64)]
        l.orc_synthetic_csr.restype = ctypes.c_int
        l.orc_synthetic_csr.argtypes = [ctypes.c_int, u64, u32, u64, u64, u64, u64, u64,
                                        P(ctypes.c_int64), P(u32), P(u64)]
        _lib = l
    return _lib


RMAT_PROBABILITIES = (0.57, 0.19, 0.19, 0.05)


def synthetic_csr(kind: str, n: int, m: int, scale: int = 0, seed: int = 42,
                  probabilities=RMAT_PROBABILITIES) -> Tuple[np.ndarray, np.ndarray]:
    """(indptr, indices) of the seeded Erdos-Renyi (``kind="er"``) or R-MAT (``"rmat"``) graph with
    ``m`` distinct undirected edges: the same graph as ``embiggen_b200.graph.erdos_renyi / rmat``
    and the product's GPU builder, generated by oracle/graphgen.c on ``set_threads`` host threads."""
    a, b, c, _ = probabilities
    t_a, t_ab, t_abc = int(a * 2 ** 32), int((a + b) * 2 ** 32), int((a + b + c) * 2 ** 32)
    indptr = np.empty(n + 1, dtype=np.int64)
    indices = np.empty(2 * m, dtype=np.uint32)
    nnz = ctypes.c_uint64(0)
    rc = lib().orc_synthetic_csr({"er": 0, "rmat": 1}[kind], n, scale, m, seed, t_a, t_ab, t_abc,
                                 _ptr(indptr, ctypes.c_int64), _ptr(indices, ctypes.c_uint32),
                                 ctypes.byref(nnz))
    if rc != 0:
        raise ValueError(f"orc_synthetic_csr failed with status {rc}")
    assert nnz.value == 2 * m
    return indptr, indices


def philox(seed: int, c0: int, c1: int, c2: int, c3: int) -> Tuple[int, int, int, int]:
    out = (ctypes.c_uint32 * 4)()
    lib().orc_philox(seed, c0, c1, c2, c3, out)
    return tuple(int(x) for x in out)


def philox_range(seed: int, count: int, c1: int, c2: int, c3: int, first_c0: int = 0) -> np.ndarray:
    """Blocks (c0 = first_c0 + i, c1, c2, c3), i < count, as a (count, 4) uint32 array."""
    out = np.empty((count, 4), dtype=np.uint32)
    lib().orc_philox_range(seed, first_c0, count, c1, c2, c3, _ptr(out, ctypes.c_uint32))
    return out


def set_threads(threads: int) -> None:
    lib().orc_set_threads(int(threads))


def row_stride(embedding_size: int) -> int:
    return (int(embedding_size) + 3) // 4 * 4


def _csr(indptr, indices):
    indptr = np.ascontiguousarray(indptr, dtype=np.int64)
    indices = np.ascontiguousarray(indices, dtype=np.uint32)
    return indptr, indices


def sources(indptr) -> np.ndarray:
    indptr = np.ascontiguousarray(indptr, dtype=np.int64)
    n = indptr.shape[0] - 1
    out = np.empty(n, dtype=np.uint32)
    count = lib().orc_sources(_ptr(indptr, ctypes.c_int64), n, _ptr(out, ctypes.c_uint32))
    return out[:count].copy()


def thresholds(return_weight: float, explore_weight: float) -> np.ndarray:
    out = np.zeros(3, dtype=np.uint64)
    lib().orc_thresholds(return_weight, explore_weight, _ptr(out, ctypes.c_uint64))
    return out


def edge_alias(indptr, weights) -> np.ndarray:
    """Per-row Vose alias tables of a weighted graph, shape (nnz, 2): {thr, alias index inside
    the row} (oracle/walks.c: orc_edge_alias)."""
    indptr = np.ascontiguousarray(indptr, dtype=np.int64)
    weights = np.ascontiguousarray(weights, dtype=np.float32)
    table = np.empty((weights.shape[0], 2), dtype=np.uint32)
    rc = lib().orc_edge_alias(_ptr(indptr, ctypes.c_int64), _ptr(weights, ctypes.c_float),
                              indptr.shape[0] - 1, _ptr(table, ctypes.c_uint32))
    if rc != 0:
        raise ValueError(f"orc_edge_alias failed with status {rc} (negative or NaN weight?)")
    return table


def degree_normalised_weights(indptr, indices, weights=None) -> np.ndarray:
    """normalize_by_degree (.../node2vec_skipgram.py:94-96): the weight of v -> x divided by
    max(deg(x), 1), in float32 (a single IEEE division per edge)."""
    indptr, indices = _csr(indptr, indices)
    degrees = np.maximum(np.diff(indptr), 1).astype(np.float32)
    base = np.ones(indices.shape[0], dtype=np.float32) if weights is None else \
        np.ascontiguousarray(weights, dtype=np.float32)
    return (base / degrees[indices]).astype(np.float32)


def walks(indptr, indices, seed: int, first_walk: int, n_walks: int, walk_length: int,
          return_weight: float = 1.0, explore_weight: float = 1.0, walk_id_stride: int = 1,
          srcs: Optional[np.ndarray] = None, weights=None,
          normalize_by_degree: bool = False, node_types=None, edge_types=None,
          change_node_type_weight: float = 1.0,
          change_edge_type_weight: float = 1.0,
          undirected: Optional[bool] = None) -> Tuple[np.ndarray, dict]:
    """``undirected`` (every edge mirrored) enables the folded return edge (walks.c); None =
    check the graph, as the product does at load."""
    indptr, indices = _csr(indptr, indices)
    if undirected is None:
        undirected = is_undirected(indptr, indices) if return_weight > max(1.0, explore_weight) else False
    if normalize_by_degree:
        weights = degree_normalised_weights(indptr, indices, weights)
    table = None if weights is None else edge_alias(indptr, weights)
    n = indptr.shape[0] - 1
    if srcs is None:
        srcs = sources(indptr)
    srcs = np.ascontiguousarray(srcs, dtype=np.uint32)
    out = np.empty((n_walks, walk_length), dtype=np.uint32)
    counters = WalkCounters()
    if node_types is not None:
        node_types = np.ascontiguousarray(node_types, dtype=np.uint32)
        assert node_types.shape[0] == n
    if edge_types is not None:
        edge_types = np.ascontiguousarray(edge_types, dtype=np.uint32)
        assert edge_types.shape[0] == indices.shape[0]
    rc = lib().orc_walks_typed(_ptr(indptr, ctypes.c_int64), _ptr(indices, ctypes.c_uint32),
                               _ptr(table, ctypes.c_uint32), _ptr(node_types, ctypes.c_uint32), _ptr(edge_types, ctypes.c_uint32),
                               change_node_type_weight, change_edge_type_weight, n,
                               _ptr(srcs, ctypes.c_uint32), srcs.shape[0], seed, first_walk, n_walks,
                               walk_id_stride, walk_length, return_weight, explore_weight,
                               int(bool(undirected)), _ptr(out, ctypes.c_uint32), ctypes.byref(counters))
    if rc != 0:
        raise ValueError(f"orc_walks failed with status {rc}")
    return out, counters.as_dict()


def is_undirected(indptr, indices) -> bool:
    indptr, indices = _csr(indptr, indices)
    return bool(lib().orc_is_undirected(_ptr(indptr, ctypes.c_int64), _ptr(indices, ctypes.c_uint32),
                                        indptr.shape[0] - 1))


def fold_thresholds(return_weight: float, explore_weight: float) -> Tuple[np.ndarray, int]:
    """(accept thresholds [return, common, explore], excess E) of the folded sampler (walks.c)."""
    out = np.zeros(3, dtype=np.uint64)
    excess = ctypes.c_uint64(0)
    lib().orc_fold_thresholds(return_weight, explore_weight, _ptr(out, ctypes.c_uint64), ctypes.byref(excess))
    return out, int(excess.value)


def alias_build(indptr, alpha: float = 0.75) -> Tuple[np.ndarray, np.ndarray]:
    indptr = np.ascontiguousarray(indptr, dtype=np.int64)
    n = indptr.shape[0] - 1
    thr = np.empty(n, dtype=np.uint32)
    alias = np.empty(n, dtype=np.uint32)
    rc = lib().orc_alias_build(_ptr(indptr, ctypes.c_int64), n, alpha, _ptr(thr, ctypes.c_uint32),
                               _ptr(alias, ctypes.c_uint32))
    if rc != 0:
        raise ValueError(f"orc_alias_build failed with status {rc}")
    return thr, alias


def sigmoid(x: float) -> float:
    return float(lib().orc_sigmoid(x))


def dot(a: np.ndarray, b: np.ndarray) -> float:
    a = np.ascontiguousarray(a, dtype=np.float32)
    b = np.ascontiguousarray(b, dtype=np.float32)
    return float(lib().orc_dot(_ptr(a, ctypes.c_float), _ptr(b, ctypes.c_float), a.shape[0]))


def init_tables(n: int, embedding_size: int, seed: int) -> Tuple[np.ndarray, np.ndarray]:
    stride = row_stride(embedding_size)
    t0 = np.empty((n, stride), dtype=np.float32)
    t1 = np.empty((n, stride), dtype=np.float32)
    rc = lib().orc_init_tables(n, embedding_size, stride, seed, _ptr(t0, ctypes.c_float),
                               _ptr(t1, ctypes.c_float))
    if rc != 0:
        raise ValueError(f"orc_init_tables failed with status {rc}")
    return t0, t1


def train(model: str, walk_array: np.ndarray, t0: np.ndarray, t1: np.ndarray, seed: int, n: int,
          embedding_size: int, window_size: int, negatives: int, learning_rate: float,
          clipping_value: float = 6.0, first_walk: int = 0, walk_id_stride: int = 1,
          thr: Optional[np.ndarray] = None, alias: Optional[np.ndarray] = None,
          indptr: Optional[np.ndarray] = None, normalize_learning_rate_by_degree: bool = False,
          scale_by_sqrt_dim: bool = False, stochastic_downsample_by_degree: bool = False,
          fast_math: bool = False, shared_negatives: bool = False) -> dict:
    """Train in place over row-major walks; returns loss_sum / pairs / targets.  ``fast_math``
    (vectorised dot, libm exp) is for timing the CPU baseline only, never for parity.
    ``shared_negatives`` (SkipGram): one set of negatives per centre, see sgns.c."""
    walk_array = np.ascontiguousarray(walk_array, dtype=np.uint32)
    assert t0.dtype == np.float32 and t1.dtype == np.float32
    assert t0.flags.c_contiguous and t1.flags.c_contiguous
    cfg = SgnsCfg(
        model={"skipgram": 0, "cbow": 1}[model.lower()],
        embedding_size=embedding_size,
        row_stride=t0.shape[1],
        walk_length=walk_array.shape[1],
        window_size=window_size,
        negatives=negatives,
        clipping_value=clipping_value,
        learning_rate=learning_rate,
        use_alias=int(thr is not None),
        normalize_learning_rate_by_degree=int(normalize_learning_rate_by_degree),
        scale_by_sqrt_dim=int(scale_by_sqrt_dim),
        fast_math=int(fast_math),
        shared_negatives=int(shared_negatives),
    )
    if indptr is not None:
        indptr = np.ascontiguousarray(indptr, dtype=np.int64)
    if stochastic_downsample_by_degree:
        cfg.downsample_bound = int(np.diff(indptr).max()) + 1
    loss = ctypes.c_double(0.0)
    pairs = ctypes.c_uint64(0)
    targets = ctypes.c_uint64(0)
    rc = lib().orc_train(ctypes.byref(cfg), _ptr(walk_array, ctypes.c_uint32), walk_array.shape[0],
                         first_walk, walk_id_stride, seed, n, _ptr(indptr, ctypes.c_int64),
                         _ptr(thr, ctypes.c_uint32), _ptr(alias, ctypes.c_uint32),
                         _ptr(t0, ctypes.c_float), _ptr(t1, ctypes.c_float), ctypes.byref(loss),
                         ctypes.byref(pairs), ctypes.byref(targets))
    if rc != 0:
        raise ValueError(f"orc_train failed with status {rc}")
    return {"loss_sum": loss.value, "pairs": pairs.value, "targets": targets.value}


def walklet_split(walk_array: np.ndarray, scale: int) -> np.ndarray:
    """Walklets (/root/reference/embiggen/embedders/ensmallen_embedders/walklets.py:7-149): the
    ``scale`` sub-walks made of every ``scale``-th token, as [scale][n_walks][ceil(L / scale)],
    padded with the PAD token.  Adjacent tokens of a sub-walk are exactly ``scale`` hops apart."""
    n_walks, L = walk_array.shape
    Ls = (L + scale - 1) // scale
    out = np.full((scale, n_walks, Ls), PAD_TOKEN, dtype=np.uint32)
    for r in range(scale):
        part = walk_array[:, r::scale]
        out[r, :, :part.shape[1]] = part
    return out


def train_walklets(model: str, walk_array: np.ndarray, scale: int, t0, t1, seed: int, n: int,
                   embedding_size: int, window_size: int, negatives: int, learning_rate: float,
                   first_walk: int = 0, **kwargs) -> dict:
    """``train`` over the sub-walks of scale ``scale``; sub-walk r of walk g draws its negatives
    as walk g + r * 2^48."""
    if scale < 2:
        return train(model, walk_array, t0, t1, seed, n, embedding_size, window_size, negatives,
                     learning_rate, first_walk=first_walk, **kwargs)
    total = {"loss_sum": 0.0, "pairs": 0, "targets": 0}
    for r, sub in enumerate(walklet_split(walk_array, scale)):
        stats = train(model, np.ascontiguousarray(sub), t0, t1, seed, n, embedding_size, window_size,
                      negatives, learning_rate, first_walk=first_walk + (r << 48), **kwargs)
        for key in total:
            total[key] += stats[key]
    return total


def fit(model: str, indptr, indices, seed: int, embedding_size: int, epochs: int, iterations: int,
        walk_length: int, window_size: int, negatives: int, learning_rate: float,
        learning_rate_decay: float, return_weight: float = 1.0, explore_weight: float = 1.0,
        clipping_value: float = 6.0, alpha: float = 0.75, use_scale_free_distribution: bool = True,
        normalize_learning_rate_by_degree: bool = False, chunk_walks: int = 1 << 16,
        stochastic_downsample_by_degree: bool = False, normalize_by_degree: bool = False,
        walklet_scale: int = 0, shared_negatives: bool = False):
    """Whole path: walks + SGD for ``epochs`` epochs in ascending walk-id order.

    Returns (t0, t1, epoch_mean_loss) with padded row stride.
    """
    indptr, indices = _csr(indptr, indices)
    n = indptr.shape[0] - 1
    srcs = sources(indptr)
    thr = alias = None
    if use_scale_free_distribution:
        thr, alias = alias_build(indptr, alpha)
    t0, t1 = init_tables(n, embedding_size, seed)
    walks_per_epoch = iterations * srcs.shape[0]
    lr = np.float32(learning_rate)
    losses = []
    for epoch in range(epochs):
        loss_sum, pairs = 0.0, 0
        done = 0
        while done < walks_per_epoch:
            count = min(chunk_walks, walks_per_epoch - done)
            first = epoch * walks_per_epoch + done
            w, _ = walks(indptr, indices, seed, first, count, walk_length, return_weight,
                         explore_weight, srcs=srcs, normalize_by_degree=normalize_by_degree)
            r = train_walklets(model, w, walklet_scale, t0, t1, seed, n, embedding_size, window_size,
                      negatives, float(lr), clipping_value=clipping_value,
                      first_walk=first, thr=thr, alias=alias, indptr=indptr,
                      normalize_learning_rate_by_degree=normalize_learning_rate_by_degree,
                      stochastic_downsample_by_degree=stochastic_downsample_by_degree,
                      shared_negatives=shared_negatives)
            loss_sum += r["loss_sum"]
            pairs += r["pairs"]
            done += count
        losses.append(loss_sum / max(pairs, 1))
        lr = np.float32(lr * np.float32(learning_rate_decay))
    return t0, t1, losses


# ---- GloVe on walk co-occurrences (oracle/glove.c) ----
def cooccurrence(walk_array: np.ndarray, window_size: int) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """(centre, context, count) of every ordered pair of different tokens at most ``window_size``
    positions apart (window trimmed at the borders, PAD skipped), sorted by (centre, context)."""
    walk_array = np.ascontiguousarray(walk_array, dtype=np.uint32)
    keys = []
    for d in range(1, min(window_size, walk_array.shape[1] - 1) + 1):
        a, b = walk_array[:, :-d].ravel(), walk_array[:, d:].ravel()
        ok = (a != PAD_TOKEN) & (b != PAD_TOKEN) & (a != b)
        a, b = a[ok].astype(np.uint64), b[ok].astype(np.uint64)
        keys.append((a << np.uint64(32)) | b)
        keys.append((b << np.uint64(32)) | a)
    if not keys:
        empty = np.zeros(0, dtype=np.uint32)
        return empty, empty.copy(), empty.copy()
    unique, counts = np.unique(np.concatenate(keys), return_counts=True)
    return ((unique >> np.uint64(32)).astype(np.uint32), (unique & np.uint64(0xFFFFFFFF)).astype(np.uint32),
            counts.astype(np.uint32))


def log_det(x: float) -> float:
    return float(lib().orc_log_det(x))


def glove_train(centre, context, count, t0: np.ndarray, t1: np.ndarray, embedding_size: int,
                alpha: float, learning_rate: float, clipping_value: float = 6.0,
                max_count: Optional[int] = None, tile_semantics: bool = False) -> dict:
    """One sequential pass over the triples (in place); returns loss_sum / trained.

    ``tile_semantics`` trains with the arithmetic of the production kernel (glove_tile_kernel:
    context rows updated as ``old + (-g * h)``, centre rows written back as ``row + (h - h0)``)
    instead of the specification's; see oracle/oracle.h."""
    centre = np.ascontiguousarray(centre, dtype=np.uint32)
    context = np.ascontiguousarray(context, dtype=np.uint32)
    count = np.ascontiguousarray(count, dtype=np.uint32)
    if max_count is None:
        max_count = int(count.max()) if count.shape[0] else 1
    loss = ctypes.c_double(0.0)
    trained = ctypes.c_uint64(0)
    rc = lib().orc_glove_train(_ptr(centre, ctypes.c_uint32), _ptr(context, ctypes.c_uint32),
                               _ptr(count, ctypes.c_uint32), centre.shape[0], max_count, embedding_size,
                               t0.shape[1], alpha, clipping_value, learning_rate, int(bool(tile_semantics)),
                               _ptr(t0, ctypes.c_float), _ptr(t1, ctypes.c_float), ctypes.byref(loss),
                               ctypes.byref(trained))
    if rc != 0:
        raise ValueError(f"orc_glove_train failed with status {rc}")
    return {"loss_sum": loss.value, "trained": trained.value, "max_count": max_count}


def glove_fit(indptr, indices, seed: int, embedding_size: int, epochs: int, walk_length: int,
              window_size: int, alpha: float, learning_rate: float, learning_rate_decay: float,
              return_weight: float = 1.0, explore_weight: float = 1.0, clipping_value: float = 6.0,
              iterations: int = 1):
    """Whole GloVe path: per epoch fresh walks (one per source node and iteration), their
    co-occurrence, one pass of SGD.  Returns (t0, t1, epoch_mean_loss)."""
    indptr, indices = _csr(indptr, indices)
    n = indptr.shape[0] - 1
    srcs = sources(indptr)
    t0, t1 = init_tables(n, embedding_size, seed)
    per_epoch = iterations * srcs.shape[0]
    lr = np.float32(learning_rate)
    losses = []
    for epoch in range(epochs):
        w, _ = walks(indptr, indices, seed, epoch * per_epoch, per_epoch, walk_length, return_weight,
                     explore_weight, srcs=srcs)
        centre, context, count = cooccurrence(w, window_size)
        r = glove_train(centre, context, count, t0, t1, embedding_size, alpha, float(lr), clipping_value)
        losses.append(r["loss_sum"] / max(r["trained"], 1))
        lr = np.float32(lr * np.float32(learning_rate_decay))
    return t0, t1, losses
