"""Host-side driver above the C ABI: the object that stands where the reference holds its
``ensmallen.models.SkipGram / CBOW`` instance
(/root/reference/embiggen/embedders/ensmallen_embedders/node2vec.py:65-69, used at :99).

PyTorch appears only as plumbing for the multi-GPU path (``torch.distributed`` carries the
IPC handles and the barriers around the exchange step); every kernel, the exchange kernel over
NVLink peer memory included, is in ``libb2e.so``.
"""
import ctypes
import time
from typing import List, Optional, Tuple

import numpy as np

from . import _lib
from ._lib import B2EConfig, B2ECounters, MODEL_IDS, check


class _DeviceArray:
    """Exposes a raw device pointer through ``__cuda_array_interface__``."""

    def __init__(self, pointer: int, shape: Tuple[int, ...], typestr: str = "<f4"):
        self.__cuda_array_interface__ = {
            "shape": shape, "typestr": typestr, "data": (pointer, False), "version": 2,
        }


def pairs_per_walk(walk_length: int, window_size: int) -> int:
    """P(L, w) = 2wL - w(w+1): positives of a border-trimmed window (SURVEY.md section 8)."""
    w = min(window_size, walk_length - 1)
    return 2 * w * walk_length - w * (w + 1)


def shard_chunks(walks_per_epoch: int, chunk_capacity: int, world: int, rank: int, base: int = 0):
    """Data-parallel schedule of one epoch: yields ``(first_walk_id, n_walks, stride)`` per step.

    A step covers ``chunk_capacity * world`` consecutive walk ids; rank ``r`` takes the ids
    congruent to ``r`` modulo ``world`` (strided, so R-MAT hubs spread over the ranks), i.e.
    ``first_walk_id + k * stride`` for ``k < n_walks``.  Because walks are a pure function of
    ``(seed, walk_id)`` the union over the ranks is exactly the single-GPU epoch.
    """
    step = chunk_capacity * world
    done = 0
    while done < walks_per_epoch:
        count = min(step, walks_per_epoch - done)
        mine = (count - rank + world - 1) // world if count > rank else 0
        yield base + done + rank, mine, world
        done += count


def fit_scales(engines: List["Engine"], seed: int) -> List[List[float]]:
    """Walklets in one pass: ``engines[k]`` holds the tables of scale k + 1 (all on one device,
    one graph, one walk_length); every chunk of every epoch is walked ONCE, by ``engines[0]``, and
    adopted by the others.  The schedule is b2e_fit's; returns the per-epoch losses per scale."""
    lead, cfg = engines[0], engines[0].config
    for engine in engines:
        engine.init_tables(seed)
    per_epoch, capacity = lead.walks_per_epoch, min(e.chunk_capacity for e in engines)
    lr = np.float32(cfg.learning_rate)
    losses: List[List[float]] = [[] for _ in engines]
    index = 0
    for epoch in range(cfg.epochs):
        for engine in engines:
            engine.reset_counters()
        done = 0
        while done < per_epoch:
            count = min(capacity, per_epoch - done)
            slot = index & 1
            # the adopters of two chunks ago have trained on this slot before it is walked over
            for engine in engines[1:]:
                engine.sync()
            lead.walk_chunk(seed, epoch * per_epoch + done, count, 1, slot)
            for engine in engines[1:]:
                engine.adopt_walks(lead, slot)
            for engine in engines:
                engine.train_chunk(seed, slot, float(lr))
            done += count
            index += 1
        for k, engine in enumerate(engines):
            c = engine.counters()
            losses[k].append(c["loss_sum"] / max(c["pairs"], 1))
        lr = np.float32(lr * np.float32(cfg.learning_rate_decay))
    return losses


def average_replicas(tables, process_group=None) -> None:
    """In-place average of every rank's replica of the tables (the one exchange step of the
    path).  NCCL reduces with AVG (no extra pass over HBM); gloo (CPU tests) sums then scales."""
    import torch.distributed as dist
    world = dist.get_world_size(process_group)
    average = dist.get_backend(process_group) == "nccl"
    for t in tables:
        if average:
            dist.all_reduce(t, op=dist.ReduceOp.AVG, group=process_group)
        else:
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=process_group)
            t.div_(world)


class Engine:
    """One engine = one ``b2e_handle`` on one GPU."""

    def __init__(self, model: str, embedding_size: int = 100, epochs: int = 30,
                 walk_length: int = 128, iterations: int = 10, window_size: int = 5,
                 number_of_negative_samples: int = 10, clipping_value: float = 6.0,
                 return_weight: float = 1.0, explore_weight: float = 1.0,
                 learning_rate: float = 0.01, learning_rate_decay: float = 0.9,
                 negative_sampling_exponent: float = 0.75,
                 use_scale_free_distribution: bool = True,
                 normalize_learning_rate_by_degree: bool = False,
                 normalize_by_degree: bool = False,
                 change_node_type_weight: float = 1.0, change_edge_type_weight: float = 1.0,
                 glove_alpha: float = 0.75,
                 stochastic_downsample_by_degree: bool = False,
                 scale_by_sqrt_dim: bool = False, walklet_scale: int = 0, deterministic: bool = False,
                 shared_negatives: bool = False,
                 chunk_walks: int = 0, max_concurrent_walks: int = 0, device: int = 0):
        self._lib = _lib.load()
        self._handle = ctypes.c_void_p()
        self.model = model.lower()
        if self.model not in MODEL_IDS:
            raise ValueError(f"Unknown model {model!r}; expected 'SkipGram' or 'CBOW'.")
        self.config = B2EConfig(
            struct_size=ctypes.sizeof(B2EConfig), model=MODEL_IDS[self.model],
            embedding_size=embedding_size, epochs=epochs, walk_length=walk_length,
            iterations=iterations, window_size=window_size,
            number_of_negative_samples=number_of_negative_samples,
            clipping_value=clipping_value, return_weight=return_weight,
            explore_weight=explore_weight, learning_rate=learning_rate,
            learning_rate_decay=learning_rate_decay,
            negative_sampling_exponent=negative_sampling_exponent,
            use_scale_free_distribution=int(bool(use_scale_free_distribution)),
            normalize_learning_rate_by_degree=int(bool(normalize_learning_rate_by_degree)),
            normalize_by_degree=int(bool(normalize_by_degree)),
            glove_alpha=glove_alpha,
            change_node_type_weight=change_node_type_weight,
            change_edge_type_weight=change_edge_type_weight,
            stochastic_downsample_by_degree=int(bool(stochastic_downsample_by_degree)),
            scale_by_sqrt_dim=int(bool(scale_by_sqrt_dim)), walklet_scale=int(walklet_scale),
            deterministic=int(bool(deterministic)), shared_negatives=int(bool(shared_negatives)),
            chunk_walks=chunk_walks, max_concurrent_walks=max_concurrent_walks, device=device,
        )
        check(self._lib.b2e_create(ctypes.byref(self.config), ctypes.byref(self._handle)))
        self.n = 0
        self._keepalive = None

    # ---- lifetime ----
    def close(self) -> None:
        if self._handle:
            self._lib.b2e_destroy(self._handle)
            self._handle = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *_):
        self.close()

    # ---- K1 ----
    def load_csr(self, indptr: np.ndarray, indices: np.ndarray,
                 weights: Optional[np.ndarray] = None) -> None:
        indptr = np.ascontiguousarray(indptr, dtype=np.int64)
        indices = np.ascontiguousarray(indices, dtype=np.uint32)
        if indptr.ndim != 1 or indptr.shape[0] < 2:
            raise ValueError("The provided graph is empty.")
        n, nnz = indptr.shape[0] - 1, indices.shape[0]
        pointer = None
        if weights is not None:
            weights = np.ascontiguousarray(weights, dtype=np.float32)
            if weights.shape != indices.shape:
                raise ValueError("weights must have one entry per directed edge.")
            pointer = weights.ctypes.data
        check(self._lib.b2e_load_csr_weighted(self._handle, indptr.ctypes.data, indices.ctypes.data,
                                              pointer, n, nnz))
        self.n = n
        self.nnz = nnz

    def load_graph(self, graph) -> None:
        """K1 without the copy: walk on a :class:`embiggen_b200.graph_gpu.DeviceGraph` (a CSR that
        was built on this GPU and never left HBM); a weighted one walks by its weights."""
        check(self._lib.b2e_load_graph(self._handle, graph._handle))
        self.n = graph.get_number_of_nodes()
        self.nnz = graph.get_number_of_directed_edges()

    def load_types(self, node_types: Optional[np.ndarray] = None,
                   edge_types: Optional[np.ndarray] = None) -> None:
        """Type ids of typed walks (``change_node_type_weight`` / ``change_edge_type_weight``):
        one uint32 per node / per directed edge in CSR order."""
        if node_types is not None:
            node_types = np.ascontiguousarray(node_types, dtype=np.uint32)
            if node_types.shape != (self.n,):
                raise ValueError("node_types must have one entry per node.")
        if edge_types is not None:
            edge_types = np.ascontiguousarray(edge_types, dtype=np.uint32)
            if edge_types.shape != (self.nnz,):
                raise ValueError("edge_types must have one entry per directed edge.")
        check(self._lib.b2e_load_types(self._handle,
                                       None if node_types is None else node_types.ctypes.data,
                                       None if edge_types is None else edge_types.ctypes.data))

    @property
    def number_of_sources(self) -> int:
        return int(self._lib.b2e_number_of_sources(self._handle))

    @property
    def row_stride(self) -> int:
        return int(self._lib.b2e_row_stride(self._handle))

    @property
    def chunk_capacity(self) -> int:
        out = ctypes.c_uint64()
        check(self._lib.b2e_chunk_capacity(self._handle, ctypes.byref(out)))
        return int(out.value)

    @property
    def walks_per_epoch(self) -> int:
        return self.config.iterations * self.number_of_sources

    @property
    def launch_count(self) -> int:
        return int(self._lib.b2e_launch_count(self._handle))

    # ---- whole path, host buffers (single GPU) ----
    def fit(self, seed: int, table0: Optional[np.ndarray] = None,
            table1: Optional[np.ndarray] = None) -> Tuple[np.ndarray, np.ndarray, List[float]]:
        """Returns ([central, contextual] role-ordered tables, per-epoch mean pair loss)."""
        shape = (self.n, self.config.embedding_size)
        t0 = np.empty(shape, dtype=np.float32) if table0 is None else table0
        t1 = np.empty(shape, dtype=np.float32) if table1 is None else table1
        for t in (t0, t1):
            if t.shape != shape or t.dtype != np.float32 or not t.flags.c_contiguous:
                raise ValueError(f"Output tables must be C-contiguous float32 of shape {shape}.")
        losses = np.zeros(max(1, self.config.epochs), dtype=np.float32)
        check(self._lib.b2e_fit(self._handle, seed, t0.ctypes.data, t1.ctypes.data,
                                losses.ctypes.data))
        return t0, t1, [float(x) for x in losses[: self.config.epochs]]

    # ---- GloVe pieces (model "GloVe"): co-occurrence of walks, one SGD pass over the triples ----
    def cooccurrence(self, seed: int, first_walk: int, n_walks: int, walk_id_stride: int = 1,
                     accumulate: bool = False) -> int:
        out = ctypes.c_uint64()
        check(self._lib.b2e_cooccurrence(self._handle, seed, first_walk, n_walks, walk_id_stride,
                                         int(accumulate), ctypes.byref(out)))
        self._n_triples = int(out.value)
        return self._n_triples

    def export_cooccurrence(self) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        m = getattr(self, "_n_triples", 0)
        centre, context, count = (np.empty(max(m, 1), dtype=np.uint32) for _ in range(3))
        check(self._lib.b2e_cooccurrence_export(self._handle, centre.ctypes.data, context.ctypes.data,
                                                count.ctypes.data))
        return centre[:m], context[:m], count[:m]

    def glove_train(self, learning_rate: float) -> None:
        check(self._lib.b2e_glove_train(self._handle, learning_rate))

    # ---- GloVe on several GPUs: centres sharded over the ranks, replicas merged once per epoch ----
    def glove_walk_epoch(self, seed: int, first_walk: int, n_walks: int) -> None:
        """Walk a whole epoch into HBM and take its token histogram (the same on every rank)."""
        check(self._lib.b2e_glove_walk_epoch(self._handle, seed, first_walk, n_walks))

    def glove_shard_count(self, world: int, rank: int) -> Tuple[int, np.ndarray]:
        """Count the centres this rank owns; returns (their largest count, the world + 1 owner bounds)."""
        bounds = np.zeros(world + 1, dtype=np.uint32)
        local_max = ctypes.c_uint32()
        check(self._lib.b2e_glove_shard_count(self._handle, world, rank, bounds.ctypes.data,
                                              ctypes.byref(local_max)))
        return int(local_max.value), bounds

    def glove_shard_train(self, learning_rate: float, max_count: int) -> None:
        """One SGD pass over this rank's centres, weights against the epoch's largest count."""
        check(self._lib.b2e_glove_shard_train(self._handle, learning_rate, max_count))

    def glove_merge(self) -> None:
        """Launch this rank's share of the GloVe merge (asynchronous); see :meth:`merge`."""
        check(self._lib.b2e_glove_merge(self._handle))

    def merge(self, process_group=None) -> None:
        """GloVe's exchange step: every replica takes each T0 row from the rank that owns the
        centre and the sum of all ranks' T1 changes (bit-identical replicas afterwards)."""
        import torch.distributed as dist
        self.sync()                        # my training pass is done ...
        dist.barrier(group=process_group)  # ... and so is everybody else's
        self.glove_merge()
        self.sync()
        dist.barrier(group=process_group)  # every rank has written its rows to every replica

    # ---- K2 parity/debug export ----
    def walks(self, seed: int, first_walk: int, n_walks: int, walk_id_stride: int = 1) -> np.ndarray:
        out = np.empty((n_walks, self.config.walk_length), dtype=np.uint32)
        check(self._lib.b2e_walks(self._handle, seed, first_walk, n_walks, walk_id_stride,
                                  out.ctypes.data))
        return out

    def slot_walks(self, slot: int, n_walks: int) -> np.ndarray:
        """The first ``n_walks`` walks of a walk slot, as ``train_chunk`` on that slot reads them."""
        out = np.empty((n_walks, self.config.walk_length), dtype=np.uint32)
        check(self._lib.b2e_slot_walks(self._handle, slot, n_walks, out.ctypes.data))
        return out

    # ---- stepping API ----
    def set_streams(self, walk_stream, train_stream) -> None:
        """Accepts ``torch.cuda.Stream`` objects or raw ``cudaStream_t`` integers."""
        self._keepalive = (walk_stream, train_stream)
        handles = [getattr(s, "cuda_stream", s) for s in (walk_stream, train_stream)]
        check(self._lib.b2e_set_streams(self._handle, ctypes.c_void_p(handles[0]),
                                        ctypes.c_void_p(handles[1])))

    def init_tables(self, seed: int) -> None:
        check(self._lib.b2e_init_tables(self._handle, seed))

    def walk_chunk(self, seed: int, first_walk: int, n_walks: int, walk_id_stride: int = 1,
                   slot: int = 0) -> None:
        check(self._lib.b2e_walk_chunk(self._handle, seed, first_walk, n_walks, walk_id_stride, slot))

    def adopt_walks(self, source: "Engine", slot: int) -> None:
        """Take the chunk ``source`` has just walked into ``slot`` instead of walking it again."""
        check(self._lib.b2e_adopt_walks(self._handle, source._handle, slot))

    def train_chunk(self, seed: int, slot: int, learning_rate: float) -> None:
        check(self._lib.b2e_train_chunk(self._handle, seed, slot, learning_rate))

    def train_host_walks(self, seed: int, walks: np.ndarray, learning_rate: float,
                         first_walk: int = 0, walk_id_stride: int = 1) -> None:
        walks = np.ascontiguousarray(walks, dtype=np.uint32)
        if walks.ndim != 2 or walks.shape[1] != self.config.walk_length:
            raise ValueError("walks must have shape (n_walks, walk_length).")
        check(self._lib.b2e_train_host_walks(self._handle, seed, walks.ctypes.data, first_walk,
                                             walks.shape[0], walk_id_stride, learning_rate))

    def sync(self) -> None:
        check(self._lib.b2e_sync(self._handle))

    def export_tables(self, table0: Optional[np.ndarray] = None,
                      table1: Optional[np.ndarray] = None) -> Tuple[np.ndarray, np.ndarray]:
        """Raw (input table T0, output table T1), padding stripped; into the given C-contiguous
        float32 buffers when there are any."""
        shape = (self.n, self.config.embedding_size)
        t0 = np.empty(shape, dtype=np.float32) if table0 is None else table0
        t1 = np.empty(shape, dtype=np.float32) if table1 is None else table1
        check(self._lib.b2e_export_tables(self._handle, t0.ctypes.data, t1.ctypes.data))
        return t0, t1

    def import_tables(self, t0: np.ndarray, t1: np.ndarray) -> None:
        shape = (self.n, self.config.embedding_size)
        t0 = np.ascontiguousarray(t0, dtype=np.float32)
        t1 = np.ascontiguousarray(t1, dtype=np.float32)
        if t0.shape != shape or t1.shape != shape:
            raise ValueError(f"Tables must have shape {shape}.")
        check(self._lib.b2e_import_tables(self._handle, t0.ctypes.data, t1.ctypes.data))

    def export_alias(self) -> Tuple[np.ndarray, np.ndarray]:
        thr, alias = np.empty(self.n, dtype=np.uint32), np.empty(self.n, dtype=np.uint32)
        check(self._lib.b2e_export_alias(self._handle, thr.ctypes.data, alias.ctypes.data))
        return thr, alias

    def export_edge_alias(self) -> np.ndarray:
        """The per-row alias tables of a weighted load, shape (nnz, 2): {thr, alias index inside the
        row}, the layout of ``oracle.edge_alias``."""
        table = np.empty((max(self.nnz, 1), 2), dtype=np.uint32)
        check(self._lib.b2e_export_edge_alias(self._handle, table.ctypes.data))
        return table[: self.nnz]

    def counters(self) -> dict:
        out = B2ECounters()
        check(self._lib.b2e_counters_read(self._handle, ctypes.byref(out)))
        return out.as_dict()

    def reset_counters(self) -> None:
        check(self._lib.b2e_counters_reset(self._handle))

    def device_tables(self):
        """Zero-copy torch views (n x row_stride float32) of the two device tables."""
        import torch
        p0, p1 = ctypes.c_void_p(), ctypes.c_void_p()
        check(self._lib.b2e_device_tables(self._handle, ctypes.byref(p0), ctypes.byref(p1)))
        shape = (self.n, self.row_stride)
        device = f"cuda:{self.config.device}"
        return tuple(torch.as_tensor(_DeviceArray(p.value, shape), device=device) for p in (p0, p1))

    def tables_digest(self) -> dict:
        """Sums, sums of squares, order-independent bit sums and the count of non-finite values of
        the live part of the two device tables (equal replicas give equal ``bits``)."""
        sums = (ctypes.c_double * 4)()
        words = (ctypes.c_uint64 * 3)()
        check(self._lib.b2e_tables_digest(self._handle, sums, words))
        return {"sum": (sums[0], sums[2]), "squares": (sums[1], sums[3]),
                "bits": (int(words[0]), int(words[1])), "non_finite": int(words[2])}

    # ---- the exchange step: replicas averaged by one kernel over NVLink peer memory ----
    def open_exchange(self, process_group=None) -> None:
        """Map the tables of the other ranks of the node (CUDA IPC; one process per GPU)."""
        import torch.distributed as dist
        rank, world = dist.get_rank(process_group), dist.get_world_size(process_group)
        mine = ctypes.create_string_buffer(2 * 64)
        check(self._lib.b2e_exchange_handles(self._handle, mine))
        gathered = [None] * world
        dist.all_gather_object(gathered, mine.raw, group=process_group)
        everyone = ctypes.create_string_buffer(b"".join(gathered), 2 * 64 * world)
        check(self._lib.b2e_exchange_open(self._handle, world, rank, everyone))
        self._exchange_group = process_group
        dist.barrier(group=process_group)  # nobody averages before every rank has mapped its peers

    def open_exchange_local(self, replicas: List["Engine"], rank: int) -> None:
        """Same with replicas that live in this process (tests; ``replicas[rank]`` is ignored)."""
        handles = (ctypes.c_void_p * len(replicas))(*[r._handle for r in replicas])
        check(self._lib.b2e_exchange_open_local(self._handle, len(replicas), rank, handles))

    def exchange_average(self) -> None:
        """Launch this rank's share of the averaging (asynchronous on the train stream); the
        caller brackets it with barriers, see :meth:`average`."""
        check(self._lib.b2e_exchange_average(self._handle))

    def close_exchange(self) -> None:
        check(self._lib.b2e_exchange_close(self._handle))

    def average(self, process_group=None) -> None:
        """One exchange step: every replica becomes the mean of all replicas."""
        import torch.distributed as dist
        self.sync()                        # my SGD chunk is done ...
        dist.barrier(group=process_group)  # ... and so is everybody else's
        self.exchange_average()
        self.sync()
        dist.barrier(group=process_group)  # every owner has written its rows to every replica

    # ---- data-parallel path: start nodes sharded, tables averaged at a fixed step interval ----
    def fit_distributed(self, seed: int, sync_interval: int = 4, process_group=None,
                        gather: str = "all", table0: Optional[np.ndarray] = None,
                        table1: Optional[np.ndarray] = None
                        ) -> Tuple[Optional[np.ndarray], Optional[np.ndarray], List[float]]:
        """Every rank holds the CSR and both tables; rank r walks ids = r mod world_size.

        Replicas are averaged every ``sync_interval`` chunks and at each epoch end.  Returns
        role-ordered tables like :meth:`fit`; with ``gather="rank0"`` only rank 0 copies them to
        the host (the others return ``None`` tables: at C5 a host copy is 80 GB per rank).
        A GloVe handle runs :meth:`_fit_glove_distributed` instead (``sync_interval`` does not apply).
        """
        import torch
        import torch.distributed as dist
        rank, world = dist.get_rank(process_group), dist.get_world_size(process_group)
        cfg = self.config
        if gather not in ("all", "rank0"):
            raise ValueError("gather must be 'all' or 'rank0'")
        if self.model == "glove":
            return self._fit_glove_distributed(seed, process_group, gather, table0, table1)
        self.timings = {}
        self.init_tables(seed)  # identical on every rank (counter-based init)
        opened = world == 1
        per_epoch = self.walks_per_epoch
        lr = np.float32(cfg.learning_rate)
        losses = []
        self.exchange_seconds = 0.0
        self.exchange_count = 0

        def average():
            nonlocal opened
            if world == 1:
                return
            if not opened:
                # Mapping the peers' tables costs about a second per peer (CUDA IPC over 2 x 51 GB
                # at C5).  It is done here, at the first exchange, when this rank's first chunks
                # are already queued on the device: the GPU trains while the host maps.
                begin = time.perf_counter()
                self.open_exchange(process_group)
                self.timings["open_exchange_s"] = time.perf_counter() - begin
                opened = True
            begin = time.perf_counter()
            self.average(process_group)
            self.exchange_seconds += time.perf_counter() - begin
            self.exchange_count += 1

        for epoch in range(cfg.epochs):
            self.reset_counters()
            steps = list(shard_chunks(per_epoch, self.chunk_capacity, world, rank, epoch * per_epoch))
            if steps:
                self.walk_chunk(seed, steps[0][0], steps[0][1], steps[0][2], 0)
            for index, (first, mine, stride) in enumerate(steps):
                slot = index & 1
                if index + 1 < len(steps):  # walk chunk k + 1 overlaps the SGD over chunk k
                    self.walk_chunk(seed, steps[index + 1][0], steps[index + 1][1], steps[index + 1][2], slot ^ 1)
                self.train_chunk(seed, slot, float(lr))
                if sync_interval and (index + 1) % sync_interval == 0 and index + 1 < len(steps):
                    average()
            average()
            c = self.counters()
            stats = torch.tensor([c["loss_sum"], float(c["pairs"])], dtype=torch.float64)
            if dist.get_backend(process_group) == "nccl":
                stats = stats.to(f"cuda:{cfg.device}")
            dist.all_reduce(stats, group=process_group)
            losses.append(float(stats[0] / max(float(stats[1]), 1.0)))
            lr = np.float32(lr * np.float32(cfg.learning_rate_decay))
        if world > 1 and opened:
            begin = time.perf_counter()
            dist.barrier(group=process_group)
            self.close_exchange()
            self.timings["close_exchange_s"] = time.perf_counter() - begin
        return self._gather_tables(rank, gather, table0, table1, losses)

    def _gather_tables(self, rank, gather, table0, table1, losses):
        """The end of a data-parallel fit: role-ordered tables to the host on every rank, or on
        rank 0 only (``gather="rank0"``)."""
        if gather == "rank0" and rank != 0:
            return None, None, losses
        shape = (self.n, self.config.embedding_size)
        t0 = np.empty(shape, dtype=np.float32) if table0 is None else table0
        t1 = np.empty(shape, dtype=np.float32) if table1 is None else table1
        first, second = (t1, t0) if self.model == "cbow" else (t0, t1)
        begin = time.perf_counter()
        self.export_tables(first, second)
        self.timings["export_tables_s"] = time.perf_counter() - begin
        return t0, t1, losses

    def _fit_glove_distributed(self, seed, process_group, gather, table0, table1):
        """GloVe's data-parallel epoch (DESIGN.md K7): every rank walks the whole epoch (walks
        are a pure function of (seed, walk id)), counts and trains the centres it owns -- exact
        global counts, weights against the largest count of the whole epoch, taken as a maximum
        over the ranks -- and the replicas are merged once per epoch (:meth:`merge`).
        ``timings`` holds the seconds of each phase, summed over the epochs."""
        import torch
        import torch.distributed as dist
        rank, world = dist.get_rank(process_group), dist.get_world_size(process_group)
        cfg = self.config
        on_device = dist.get_backend(process_group) == "nccl"

        def all_reduce(values, dtype, op):
            tensor = torch.tensor(values, dtype=dtype)
            if on_device:
                tensor = tensor.to(f"cuda:{cfg.device}")
            dist.all_reduce(tensor, op=op, group=process_group)
            return tensor.cpu()

        self.timings = {"walk_histogram_s": 0.0, "count_s": 0.0, "train_s": 0.0, "merge_s": 0.0}
        self.init_tables(seed)  # identical on every rank (counter-based init)
        if world > 1:
            begin = time.perf_counter()
            self.open_exchange(process_group)
            self.timings["open_exchange_s"] = time.perf_counter() - begin
        per_epoch = self.walks_per_epoch
        lr = np.float32(cfg.learning_rate)
        losses = []
        for epoch in range(cfg.epochs):
            self.reset_counters()
            begin = time.perf_counter()
            self.glove_walk_epoch(seed, epoch * per_epoch, per_epoch)
            mark = time.perf_counter()
            self.timings["walk_histogram_s"] += mark - begin
            local_max, _ = self.glove_shard_count(world, rank)
            x_max = int(all_reduce([local_max], torch.int64, dist.ReduceOp.MAX)[0])
            begin = time.perf_counter()
            self.timings["count_s"] += begin - mark
            self.glove_shard_train(float(lr), x_max)
            self.sync()
            mark = time.perf_counter()
            self.timings["train_s"] += mark - begin
            if world > 1:
                self.merge(process_group)
                self.timings["merge_s"] += time.perf_counter() - mark
            c = self.counters()
            stats = all_reduce([c["loss_sum"], float(c["pairs"])], torch.float64, dist.ReduceOp.SUM)
            losses.append(float(stats[0] / max(float(stats[1]), 1.0)))
            lr = np.float32(lr * np.float32(cfg.learning_rate_decay))
        if world > 1:
            dist.barrier(group=process_group)
            self.close_exchange()
        return self._gather_tables(rank, gather, table0, table1, losses)
