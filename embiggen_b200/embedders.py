"""Node2Vec / DeepWalk SkipGram and CBOW embedders backed by the B200 engine.

Host-side mirror of the reference's Ensmallen adapters: same constructor kwargs, defaults,
``parameters()`` / ``smoke_test_parameters()`` behaviour, capability flags and
``fit_transform(graph, return_dataframe) -> EmbeddingResult`` contract as

* ``Node2VecEnsmallen``          /root/reference/embiggen/embedders/ensmallen_embedders/node2vec.py:13-166
* ``Node2VecSkipGramEnsmallen``  .../node2vec_skipgram.py:6-165
* ``Node2VecCBOWEnsmallen``      .../node2vec_cbow.py:6-165
* ``DeepWalkSkipGramEnsmallen``  .../deepwalk_skipgram.py:6-139
* ``DeepWalkCBOWEnsmallen``      .../deepwalk_cbow.py:6-139
* ``EnsmallenEmbedder``          .../ensmallen_embedder.py:9-55

What stands where the reference holds ``ensmallen.models.SkipGram / CBOW`` is
:class:`embiggen_b200.engine.Engine` (C ABI ``include/b2e.h``, hand-written sm_100a kernels).
There is no CPU fallback: constructing an embedder without the CUDA extension and a
Blackwell GPU raises.  ``library_name()`` is ``"B200"``; with ``library_name=None`` the
registry keeps preferring "Ensmallen" (abstract_model.py:670-675), so registration is
non-breaking.
"""
import os
from typing import Any, Dict, List, Optional

import numpy as np
import pandas as pd

from . import _lib
from .embedding_api import (AbstractEmbeddingModel, AbstractModel, EmbeddingResult, abstract_class,
                            normalize_kwargs)
from .engine import Engine
from .graph import as_csr, as_types

_DTYPES = {"f16": np.float16, "f32": np.float32, "f64": np.float64}
# engine options that are not part of the reference's signature (keyword-only, defaulted)
_B200_DEFAULTS = dict(negative_sampling_exponent=0.75, scale_by_sqrt_dim=False, deterministic=False,
                      shared_negatives=False, chunk_walks=0, max_concurrent_walks=0, sync_interval=4, device=None)


@abstract_class
class B200Embedder(AbstractEmbeddingModel):
    """Counterpart of ``EnsmallenEmbedder`` (ensmallen_embedder.py:9-55)."""

    def __init__(self, random_state: Optional[int] = None, embedding_size: Optional[int] = None,
                 ring_bell: bool = False, enable_cache: bool = False):
        super().__init__(random_state=random_state, embedding_size=embedding_size,
                         ring_bell=ring_bell, enable_cache=enable_cache)

    @classmethod
    def task_name(cls) -> str:
        return "Node Embedding"

    @classmethod
    def library_name(cls) -> str:
        return "B200"

    @classmethod
    def requires_nodes_sorted_by_decreasing_node_degree(cls) -> bool:
        return False

    @classmethod
    def is_topological(cls) -> bool:
        return True

    @staticmethod
    def is_available() -> bool:
        """True when libb2e.so is built and a Blackwell device is visible."""
        try:
            return _lib.load().b2e_device_count() > 0
        except Exception:
            return False


@abstract_class
class Node2VecB200(B200Embedder):
    """Counterpart of ``Node2VecEnsmallen`` (node2vec.py:13-166)."""

    MODELS = {  # node2vec.py:16-26
        "DeepWalk CBOW": "CBOW",
        "DeepWalk SkipGram": "SkipGram",
        "DeepWalk GloVe": "GloVe",
        "Node2Vec CBOW": "CBOW",
        "Node2Vec SkipGram": "SkipGram",
        "Node2Vec GloVe": "GloVe",
    }

    def __init__(self, embedding_size: int = 100, random_state: int = 42, ring_bell: bool = False,
                 enable_cache: bool = False, **model_kwargs: Dict):
        if self.model_name() not in self.MODELS:
            raise ValueError(f"The model name {self.model_name()!r} is not in {sorted(self.MODELS)}.")
        self._model_kwargs = normalize_kwargs(
            self, {**model_kwargs, "embedding_size": embedding_size, "random_state": random_state})
        embedding_size = self._model_kwargs.pop("embedding_size")
        random_state = self._model_kwargs.pop("random_state")
        self._check_supported(self._model_kwargs)
        if self._model_kwargs.get("shared_negatives"):  # the limits b2e_create enforces, at construction
            if self.MODELS[self.model_name()] != "SkipGram":
                raise ValueError("shared_negatives is a SkipGram option (CBOW draws its negatives per centre "
                                 f"already, GloVe draws none); {self.model_name()!r} cannot use it.")
            if self._model_kwargs.get("window_size", 1) > 7 or embedding_size > 128 or \
                    self._model_kwargs.get("number_of_negative_samples", 0) > 15:
                raise ValueError("shared_negatives needs window_size <= 7, number_of_negative_samples <= 15 "
                                 "and embedding_size <= 128.")
        # Like the reference, which builds the Rust model here (node2vec.py:65-69), fail at
        # construction time when the native engine cannot run.
        _lib.load()
        self._last_losses: List[float] = []
        super().__init__(embedding_size=embedding_size, enable_cache=enable_cache,
                         ring_bell=ring_bell, random_state=random_state)

    @staticmethod
    def _check_supported(kwargs: Dict[str, Any]) -> None:
        for name in ("change_node_type_weight", "change_edge_type_weight"):
            if not kwargs.get(name, 1.0) > 0.0:
                raise ValueError(f"{name} must be strictly positive, got {kwargs.get(name)!r}.")
        if kwargs.get("dtype", "f32") not in _DTYPES:
            raise ValueError(f"dtype must be one of {sorted(_DTYPES)}, got {kwargs.get('dtype')!r}.")
        if isinstance(kwargs.get("learning_rate"), str):
            raise NotImplementedError("Only a numeric learning_rate is supported.")

    @classmethod
    def smoke_test_parameters(cls) -> Dict[str, Any]:
        """Same as node2vec.py:79-87."""
        return dict(epochs=1, embedding_size=5, window_size=1, walk_length=4, max_neighbours=10)

    def parameters(self) -> Dict[str, Any]:
        return dict(**super().parameters(), **self._model_kwargs)

    def get_losses(self) -> List[float]:
        """Mean pair loss of every epoch of the last ``fit_transform``."""
        return list(self._last_losses)

    # -- what stands where the reference calls self._model.fit_transform(graph), node2vec.py:99 --
    def _engine_kwargs(self, device: int) -> Dict[str, Any]:
        k = self._model_kwargs
        # Walklets (WalkletsB200): scale k trains window 1 on the sub-walks of every k-th token
        scale = getattr(self, "_walklet_scale", 0)
        return dict(
            model=self.MODELS[self.model_name()], embedding_size=self._embedding_size,
            epochs=k["epochs"], walk_length=k["walk_length"], iterations=k.get("iterations", 1),
            window_size=1 if scale else k["window_size"],
            number_of_negative_samples=k.get("number_of_negative_samples", 0),
            clipping_value=k.get("clipping_value", 6.0), glove_alpha=k.get("alpha", 0.75), return_weight=k.get("return_weight", 1.0),
            explore_weight=k.get("explore_weight", 1.0), learning_rate=k["learning_rate"],
            learning_rate_decay=k["learning_rate_decay"],
            negative_sampling_exponent=k["negative_sampling_exponent"],
            use_scale_free_distribution=k.get("use_scale_free_distribution", True),
            normalize_learning_rate_by_degree=k.get("normalize_learning_rate_by_degree", False),
            normalize_by_degree=k["normalize_by_degree"],
            change_node_type_weight=k.get("change_node_type_weight", 1.0),
            change_edge_type_weight=k.get("change_edge_type_weight", 1.0),
            stochastic_downsample_by_degree=bool(k.get("stochastic_downsample_by_degree", False)),
            scale_by_sqrt_dim=k["scale_by_sqrt_dim"], deterministic=k["deterministic"],
            shared_negatives=k["shared_negatives"], walklet_scale=scale,
            chunk_walks=k["chunk_walks"], max_concurrent_walks=k["max_concurrent_walks"],
            device=device)

    def _output_buffers(self, n: int, writes_files: bool = True):
        """float32 host buffers the engine writes; .npy memory maps when paths are given
        (node2vec_skipgram.py:86-93)."""
        buffers = []
        for key in ("central_nodes_embedding_path", "contextual_nodes_embedding_path"):
            path = self._model_kwargs.get(key)
            # under torch.distributed every rank returns the tables but only rank 0 owns the files
            if path is None or self._model_kwargs["dtype"] != "f32" or not writes_files:
                buffers.append(np.empty((n, self._embedding_size), dtype=np.float32))
            else:
                buffers.append(np.lib.format.open_memmap(
                    path, mode="w+", dtype=np.float32, shape=(n, self._embedding_size)))
        return buffers

    def _fit_transform(self, graph, return_dataframe: bool = True) -> EmbeddingResult:
        resident = hasattr(graph, "_handle") and hasattr(graph, "to_host")  # graph_gpu.DeviceGraph
        if resident:
            indptr, indices, weights = None, None, None
            n_nodes = graph.get_number_of_nodes()
        else:
            indptr, indices, weights = as_csr(graph)
            n_nodes = indptr.shape[0] - 1
        # max_neighbours (approximated walks for hubs) is accepted for compatibility: the walk
        # kernel always samples the exact transition distribution.
        device = self._model_kwargs["device"]
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0"))
        n = n_nodes
        world, rank = 1, 0
        try:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized():
                world, rank = dist.get_world_size(), dist.get_rank()
        except ImportError:
            pass
        # the seed is read here, not at construction: set_random_state() between holdouts takes
        # effect (abstract_classifier_model.py:711-712; SURVEY.md 8b)
        seed = int(self._random_state) & 0xFFFFFFFFFFFFFFFF
        central, contextual = self._output_buffers(n, writes_files=rank == 0)
        with Engine(**self._engine_kwargs(device)) as engine:
            if resident:
                engine.load_graph(graph)  # the CSR is in HBM already: no copy
            else:
                engine.load_csr(indptr, indices, weights)  # weighted graphs walk by weight
            if self.is_using_node_types() or self.is_using_edge_types():
                node_types, edge_types = as_types(graph)  # a graph without types walks untyped
                engine.load_types(node_types if self.is_using_node_types() else None,
                                  edge_types if self.is_using_edge_types() else None)
            if world > 1:  # GloVe shards its centres over the ranks (Engine._fit_glove_distributed)
                _, _, losses = engine.fit_distributed(seed, self._model_kwargs["sync_interval"],
                                                      table0=central, table1=contextual)
            else:
                _, _, losses = engine.fit(seed, central, contextual)
        self._last_losses = losses
        if self._model_kwargs["verbose"]:
            print(f"{self.model_name()} (B200): mean pair loss per epoch "
                  + ", ".join(f"{loss:.4f}" for loss in losses))
        dtype = _DTYPES[self._model_kwargs["dtype"]]
        node_embeddings = [central, contextual]
        if dtype is not np.float32:
            node_embeddings = [e.astype(dtype) for e in node_embeddings]
            for e, key in zip(node_embeddings, ("central_nodes_embedding_path",
                                                "contextual_nodes_embedding_path")):
                if self._model_kwargs.get(key) is not None and rank == 0:
                    # exactly the path the caller named (np.save would append ".npy" to it)
                    out = np.lib.format.open_memmap(self._model_kwargs[key], mode="w+", dtype=e.dtype,
                                                    shape=e.shape)
                    out[:] = e
                    out.flush()
        if return_dataframe:  # node2vec.py:104-109
            node_names = graph.get_node_names() if hasattr(graph, "get_node_names") else None
            node_embeddings = [pd.DataFrame(e, index=node_names) for e in node_embeddings]
        return EmbeddingResult(embedding_method_name=self.model_name(),
                               node_embeddings=node_embeddings)

    # -- capability flags, the same non-redundant subset as node2vec.py:114-166 --
    @classmethod
    def requires_edge_weights(cls) -> bool:
        return False

    @classmethod
    def requires_positive_edge_weights(cls) -> bool:
        return True

    @classmethod
    def can_use_edge_weights(cls) -> bool:
        """Returns whether the model can optionally use edge weights."""
        return True

    def is_using_edge_weights(self) -> bool:
        """Returns whether the model is parametrized to use edge weights."""
        return True

    @classmethod
    def can_use_node_types(cls) -> bool:
        """Returns whether the model can optionally use node types."""
        return True

    def is_using_node_types(self) -> bool:
        """Returns whether the model is parametrized to use node types."""
        return self._model_kwargs.get("change_node_type_weight", 1.0) != 1.0

    @classmethod
    def can_use_edge_types(cls) -> bool:
        """Returns whether the model can optionally use edge types."""
        return True

    def is_using_edge_types(self) -> bool:
        """Returns whether the model is parametrized to use edge types."""
        return self._model_kwargs.get("change_edge_type_weight", 1.0) != 1.0

    @classmethod
    def requires_node_types(cls) -> bool:
        return False

    @classmethod
    def requires_edge_types(cls) -> bool:
        return False

    @classmethod
    def is_stocastic(cls) -> bool:
        """Returns whether the model is stocastic and has therefore a random state."""
        return True


def _node2vec_init(self, embedding_size=100, epochs=30, clipping_value=6.0,
                   number_of_negative_samples=10, walk_length=128, iterations=10, window_size=5,
                   return_weight=0.25, explore_weight=4.0, change_node_type_weight=1.0,
                   change_edge_type_weight=1.0, max_neighbours=100, learning_rate=0.01,
                   learning_rate_decay=0.9, central_nodes_embedding_path=None,
                   contextual_nodes_embedding_path=None, normalize_by_degree=False,
                   stochastic_downsample_by_degree=False, normalize_learning_rate_by_degree=False,
                   use_scale_free_distribution=True, random_state=42, dtype="f32", ring_bell=False,
                   enable_cache=False, verbose=True, **b200_kwargs):
    """Signature and defaults of node2vec_skipgram.py:9-35 (identical in node2vec_cbow.py),
    plus the keyword-only B200 extras of ``_B200_DEFAULTS``."""
    Node2VecB200.__init__(
        self, embedding_size=embedding_size, epochs=epochs, clipping_value=clipping_value,
        number_of_negative_samples=number_of_negative_samples, walk_length=walk_length,
        iterations=iterations, window_size=window_size, return_weight=return_weight,
        explore_weight=explore_weight, change_node_type_weight=change_node_type_weight,
        change_edge_type_weight=change_edge_type_weight, max_neighbours=max_neighbours,
        learning_rate=learning_rate, learning_rate_decay=learning_rate_decay,
        central_nodes_embedding_path=central_nodes_embedding_path,
        contextual_nodes_embedding_path=contextual_nodes_embedding_path,
        normalize_by_degree=normalize_by_degree,
        stochastic_downsample_by_degree=stochastic_downsample_by_degree,
        normalize_learning_rate_by_degree=normalize_learning_rate_by_degree,
        use_scale_free_distribution=use_scale_free_distribution, dtype=dtype,
        random_state=random_state, ring_bell=ring_bell, enable_cache=enable_cache, verbose=verbose,
        **{**_B200_DEFAULTS, **b200_kwargs})


def _deepwalk_init(self, embedding_size=100, epochs=30, clipping_value=6.0,
                   number_of_negative_samples=10, walk_length=128, iterations=10, window_size=5,
                   max_neighbours=100, learning_rate=0.01, learning_rate_decay=0.9,
                   central_nodes_embedding_path=None, contextual_nodes_embedding_path=None,
                   normalize_by_degree=False, stochastic_downsample_by_degree=False,
                   normalize_learning_rate_by_degree=False, use_scale_free_distribution=True,
                   random_state=42, dtype="f32", ring_bell=False, enable_cache=False, verbose=True,
                   **b200_kwargs):
    """Signature and defaults of deepwalk_skipgram.py:9-31 (identical in deepwalk_cbow.py):
    no return / explore weights, i.e. p = q = 1, a first-order uniform walk."""
    Node2VecB200.__init__(
        self, embedding_size=embedding_size, epochs=epochs, clipping_value=clipping_value,
        number_of_negative_samples=number_of_negative_samples, walk_length=walk_length,
        iterations=iterations, window_size=window_size, max_neighbours=max_neighbours,
        learning_rate=learning_rate, learning_rate_decay=learning_rate_decay,
        central_nodes_embedding_path=central_nodes_embedding_path,
        contextual_nodes_embedding_path=contextual_nodes_embedding_path,
        normalize_by_degree=normalize_by_degree,
        stochastic_downsample_by_degree=stochastic_downsample_by_degree,
        normalize_learning_rate_by_degree=normalize_learning_rate_by_degree,
        use_scale_free_distribution=use_scale_free_distribution, dtype=dtype,
        random_state=random_state, ring_bell=ring_bell, enable_cache=enable_cache, verbose=verbose,
        **{**_B200_DEFAULTS, **b200_kwargs})


_NODE2VEC_HIDDEN = ("change_node_type_weight", "change_edge_type_weight", "alpha")
_DEEPWALK_HIDDEN = ("return_weight", "explore_weight") + _NODE2VEC_HIDDEN


class Node2VecSkipGramB200(Node2VecB200):
    """Node2Vec SkipGram on B200 (counterpart of node2vec_skipgram.py:6-165)."""

    __init__ = _node2vec_init

    def parameters(self) -> Dict[str, Any]:
        """Drops the same keys as node2vec_skipgram.py:148-161."""
        return {k: v for k, v in super().parameters().items() if k not in _NODE2VEC_HIDDEN}

    @classmethod
    def model_name(cls) -> str:
        return "Node2Vec SkipGram"


class Node2VecCBOWB200(Node2VecB200):
    """Node2Vec CBOW on B200 (counterpart of node2vec_cbow.py:6-165)."""

    __init__ = _node2vec_init

    def parameters(self) -> Dict[str, Any]:
        return {k: v for k, v in super().parameters().items() if k not in _NODE2VEC_HIDDEN}

    @classmethod
    def model_name(cls) -> str:
        return "Node2Vec CBOW"


class DeepWalkSkipGramB200(Node2VecB200):
    """DeepWalk SkipGram on B200 (counterpart of deepwalk_skipgram.py:6-139)."""

    __init__ = _deepwalk_init

    def parameters(self) -> Dict[str, Any]:
        """Drops the same keys as deepwalk_skipgram.py:120-135."""
        return {k: v for k, v in super().parameters().items() if k not in _DEEPWALK_HIDDEN}

    @classmethod
    def model_name(cls) -> str:
        return "DeepWalk SkipGram"


class DeepWalkCBOWB200(Node2VecB200):
    """DeepWalk CBOW on B200 (counterpart of deepwalk_cbow.py:6-139)."""

    __init__ = _deepwalk_init

    def parameters(self) -> Dict[str, Any]:
        return {k: v for k, v in super().parameters().items() if k not in _DEEPWALK_HIDDEN}

    @classmethod
    def model_name(cls) -> str:
        return "DeepWalk CBOW"


def _walklets_init(self, embedding_size=100, epochs=30, clipping_value=6.0,
                   number_of_negative_samples=10, walk_length=128, iterations=10, window_size=4,
                   return_weight=1.0, explore_weight=1.0, max_neighbours=100, learning_rate=0.01,
                   learning_rate_decay=0.9, central_nodes_embedding_path=None,
                   contextual_nodes_embedding_path=None, normalize_by_degree=False,
                   stochastic_downsample_by_degree=False, normalize_learning_rate_by_degree=False,
                   use_scale_free_distribution=True, random_state=42, dtype="f32", ring_bell=False,
                   enable_cache=False, **b200_kwargs):
    """Signature and defaults of walklets_skipgram.py:9-33 (identical in walklets_cbow.py; no
    ``verbose`` there).  Like walklets.py:112-113 the per-scale embedding size is
    ``embedding_size // window_size``."""
    if central_nodes_embedding_path is not None or contextual_nodes_embedding_path is not None:
        raise NotImplementedError("Walklets return one embedding per scale; embedding paths are not supported.")
    if "verbose" in b200_kwargs:  # the reference's Walklets constructors have no such keyword
        raise TypeError(f"{type(self).__name__}.__init__() got an unexpected keyword argument 'verbose'")
    Node2VecB200.__init__(
        self, embedding_size=embedding_size // window_size, epochs=epochs,
        clipping_value=clipping_value, number_of_negative_samples=number_of_negative_samples,
        walk_length=walk_length, iterations=iterations, window_size=window_size,
        return_weight=return_weight, explore_weight=explore_weight, max_neighbours=max_neighbours,
        learning_rate=learning_rate, learning_rate_decay=learning_rate_decay,
        normalize_by_degree=normalize_by_degree,
        stochastic_downsample_by_degree=stochastic_downsample_by_degree,
        normalize_learning_rate_by_degree=normalize_learning_rate_by_degree,
        central_nodes_embedding_path=None, contextual_nodes_embedding_path=None,
        use_scale_free_distribution=use_scale_free_distribution, dtype=dtype,
        random_state=random_state, ring_bell=ring_bell, enable_cache=enable_cache, verbose=False,
        **{**_B200_DEFAULTS, **b200_kwargs})


def _node2vec_glove_init(self, embedding_size=100, alpha=0.75, epochs=100, walk_length=512, window_size=5,
                         return_weight=0.25, explore_weight=4.0, change_node_type_weight=1.0,
                         change_edge_type_weight=1.0, max_neighbours=100, learning_rate=0.05,
                         learning_rate_decay=0.9, central_nodes_embedding_path=None,
                         contextual_nodes_embedding_path=None, normalize_by_degree=False, dtype="f32",
                         random_state=42, ring_bell=False, enable_cache=False, verbose=True, **b200_kwargs):
    """Signature and defaults of node2vec_glove.py:8-30; one walk per node and epoch (:104-106)."""
    Node2VecB200.__init__(
        self, embedding_size=embedding_size, alpha=alpha, epochs=epochs, walk_length=walk_length,
        iterations=1, window_size=window_size, return_weight=return_weight, explore_weight=explore_weight,
        change_node_type_weight=change_node_type_weight, change_edge_type_weight=change_edge_type_weight,
        max_neighbours=max_neighbours, learning_rate=learning_rate, learning_rate_decay=learning_rate_decay,
        central_nodes_embedding_path=central_nodes_embedding_path,
        contextual_nodes_embedding_path=contextual_nodes_embedding_path,
        normalize_by_degree=normalize_by_degree, dtype=dtype, random_state=random_state,
        ring_bell=ring_bell, enable_cache=enable_cache, verbose=verbose,
        **{**_B200_DEFAULTS, **b200_kwargs})


def _deepwalk_glove_init(self, embedding_size=100, alpha=0.75, epochs=100, walk_length=512, window_size=5,
                         max_neighbours=100, learning_rate=0.05, learning_rate_decay=0.99,
                         central_nodes_embedding_path=None, contextual_nodes_embedding_path=None,
                         normalize_by_degree=False, dtype="f32", random_state=42, ring_bell=False,
                         enable_cache=False, verbose=True, **b200_kwargs):
    """Signature and defaults of deepwalk_glove.py:8-26."""
    Node2VecB200.__init__(
        self, embedding_size=embedding_size, alpha=alpha, epochs=epochs, walk_length=walk_length,
        iterations=1, window_size=window_size, max_neighbours=max_neighbours,
        learning_rate=learning_rate, learning_rate_decay=learning_rate_decay,
        central_nodes_embedding_path=central_nodes_embedding_path,
        contextual_nodes_embedding_path=contextual_nodes_embedding_path,
        normalize_by_degree=normalize_by_degree, dtype=dtype, random_state=random_state,
        ring_bell=ring_bell, enable_cache=enable_cache, verbose=verbose,
        **{**_B200_DEFAULTS, **b200_kwargs})


_GLOVE_HIDDEN = ("change_node_type_weight", "change_edge_type_weight", "number_of_negative_samples",
                 "iterations")


class Node2VecGloVeB200(Node2VecB200):
    """Node2Vec GloVe on B200 (counterpart of node2vec_glove.py:5-140); not registered, like
    Walklets, so that the registry keeps the four models north_star names."""

    __init__ = _node2vec_glove_init

    def parameters(self) -> Dict[str, Any]:
        """Drops the same keys as node2vec_glove.py:124-138."""
        return {k: v for k, v in super().parameters().items() if k not in _GLOVE_HIDDEN}

    @classmethod
    def model_name(cls) -> str:
        return "Node2Vec GloVe"


class DeepWalkGloVeB200(Node2VecB200):
    """DeepWalk GloVe on B200 (counterpart of deepwalk_glove.py)."""

    __init__ = _deepwalk_glove_init

    def parameters(self) -> Dict[str, Any]:
        return {k: v for k, v in super().parameters().items()
                if k not in _GLOVE_HIDDEN + ("return_weight", "explore_weight")}

    @classmethod
    def model_name(cls) -> str:
        return "DeepWalk GloVe"


@abstract_class
class WalkletsB200(Node2VecB200):
    """Counterpart of ``WalkletsEnsmallen`` (walklets.py:7-149): one SkipGram / CBOW embedding of
    ``embedding_size // window_size`` dimensions per scale k = 1 .. window_size, scale k trained
    on the pairs exactly k hops apart (the sub-walks of every k-th token, window 1).

    ``fit_transform`` returns 2 * window_size embeddings, the [central, contextual] pair of scale
    1 first, then of scale 2, ...  Not registered, like the reference's registry expects
    (tests/test_abstract_model.py:125-126)."""

    MODELS = {"Walklets SkipGram": "SkipGram", "Walklets CBOW": "CBOW"}
    __init__ = _walklets_init

    def parameters(self) -> Dict[str, Any]:
        """walklets.py:137-141: the public embedding size is the per-scale size x window_size."""
        parameters = {k: v for k, v in super().parameters().items() if k not in _NODE2VEC_HIDDEN + ("verbose",)}
        parameters["embedding_size"] = parameters["embedding_size"] * parameters["window_size"]
        return parameters

    def _fit_transform(self, graph, return_dataframe: bool = True) -> EmbeddingResult:
        """All scales in ONE pass over the walks: the graph is uploaded once and shared, every
        chunk is walked once (by the engine of scale 1) and adopted by the engines of the other
        scales, each of which owns its pair of tables (engine.fit_scales).  A resident graph
        (graph_gpu.DeviceGraph) takes this path weighted or not: every scale builds its edge alias
        tables from the resident weights.  Weighted host graphs, typed graphs, other dtypes than
        f32 and torch.distributed runs take the scale-by-scale path."""
        from .engine import fit_scales
        from .graph_gpu import device_graph_from_csr
        window_size = self._model_kwargs["window_size"]
        distributed = False
        try:
            import torch.distributed as dist
            distributed = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        except ImportError:
            pass
        resident = hasattr(graph, "_handle") and hasattr(graph, "to_host")
        weights = None if resident else as_csr(graph)[2]
        one_pass = (weights is None and not distributed and self._model_kwargs["dtype"] == "f32"
                    and not self.is_using_node_types() and not self.is_using_edge_types())
        node_embeddings, losses = [], []
        if one_pass:
            device = self._model_kwargs["device"]
            device = int(os.environ.get("LOCAL_RANK", "0")) if device is None else device
            shared = graph if resident else device_graph_from_csr(*as_csr(graph)[:2], device=device)
            n = shared.get_number_of_nodes()
            seed = int(self._random_state) & 0xFFFFFFFFFFFFFFFF
            engines = []
            try:
                for scale in range(1, window_size + 1):
                    self._walklet_scale = scale
                    engines.append(Engine(**self._engine_kwargs(device)))
                    engines[-1].load_graph(shared)
                losses = fit_scales(engines, seed)
                for engine in engines:
                    t0, t1 = engine.export_tables()
                    node_embeddings.extend([t1, t0] if engine.model == "cbow" else [t0, t1])
            finally:
                self._walklet_scale = 0
                for engine in engines:
                    engine.close()
                if not resident:
                    shared.close()
            assert all(e.shape == (n, self._embedding_size) for e in node_embeddings)
            if return_dataframe:
                names = graph.get_node_names() if hasattr(graph, "get_node_names") else None
                node_embeddings = [pd.DataFrame(e, index=names) for e in node_embeddings]
        else:
            try:
                for scale in range(1, window_size + 1):
                    self._walklet_scale = scale
                    result = super()._fit_transform(graph, return_dataframe=return_dataframe)
                    node_embeddings.extend(result.get_all_node_embedding())
                    losses.append(self._last_losses)
            finally:
                self._walklet_scale = 0
        self._last_losses = [float(np.mean(epoch)) for epoch in zip(*losses)]
        return EmbeddingResult(embedding_method_name=self.model_name(), node_embeddings=node_embeddings)


class WalkletsSkipGramB200(WalkletsB200):
    """Walklets SkipGram on B200 (counterpart of walklets_skipgram.py)."""

    @classmethod
    def model_name(cls) -> str:
        return "Walklets SkipGram"


class WalkletsCBOWB200(WalkletsB200):
    """Walklets CBOW on B200 (counterpart of walklets_cbow.py)."""

    @classmethod
    def model_name(cls) -> str:
        return "Walklets CBOW"


B200_EMBEDDERS = (Node2VecSkipGramB200, Node2VecCBOWB200, DeepWalkSkipGramB200, DeepWalkCBOWB200)
for _model in B200_EMBEDDERS:  # abstract_model.py:721-749; Walklets are deliberately not registered
    AbstractModel.register(_model)


def embed_graph(graph, embedding_model, repository: Optional[str] = None,
                version: Optional[str] = None, library_name: Optional[str] = "B200",
                smoke_test: bool = False, return_dataframe: bool = True, **kwargs) -> EmbeddingResult:
    """Same contract as /root/reference/embiggen/embedders/graph_embedding_pipeline.py:10-106
    (model by name or instance, kwargs only with a name, smoke-test conversion, every failure
    re-raised as ValueError), defaulting to this library."""
    if isinstance(embedding_model, str):
        embedding_model = AbstractEmbeddingModel.get_model_from_library(
            model_name=embedding_model, library_name=library_name)(**kwargs)
    elif kwargs:
        raise ValueError("Please be advised that even though you have provided yourself the "
                         "embedding model, you have also provided the kwargs which would normally "
                         "be forwarded to the creation of the embedding model. It is unclear what "
                         "to do with these arguments.")
    if not isinstance(embedding_model, AbstractEmbeddingModel):
        raise ValueError("The provided object is not an embedding model, that is, it does not "
                         "extend the class `AbstractEmbeddingModel`.")
    if smoke_test:
        try:
            embedding_model = embedding_model.into_smoke_test()
        except Exception as e:
            raise ValueError(
                "An exception was raised while trying to create a smoke test version of the model "
                f"called {embedding_model.model_name()} from the library {library_name}. The body "
                f"of the exception was: {e}.") from e
    if embedding_model.requires_nodes_sorted_by_decreasing_node_degree() and \
            hasattr(graph, "sort_by_decreasing_outbound_node_degree"):  # :93-94 (none of the B200 models asks)
        graph = graph.sort_by_decreasing_outbound_node_degree()
    try:
        return embedding_model.fit_transform(graph, repository=repository, version=version,
                                             return_dataframe=return_dataframe)
    except Exception as e:
        name = graph.get_name() if hasattr(graph, "get_name") else type(graph).__name__
        raise ValueError(
            f"An exception was raised while trying to compute a node embedding on the graph {name} "
            f"using the model called {embedding_model.model_name()} from the library "
            f"{library_name}, specifically implemented in the class "
            f"{embedding_model.__class__.__name__}. The body of the exception was: {e}") from e
