"""Weighted graphs on the GPU: weighted ingest (b2e_csr_from_edges_weighted, b2e_graph_from_*_weighted)
against the numpy builder, the per-row alias tables built on the device against oracle.edge_alias,
and weighted walks and embedders on resident weighted graphs."""
import numpy as np
import pytest

import oracle
from embiggen_b200.engine import Engine
from embiggen_b200.graph import CSRGraph, csr_from_edges
from embiggen_b200.graph_gpu import csr_from_edges_gpu, device_graph_from_csr, device_graph_from_edges

pytestmark = pytest.mark.gpu


def bits(array):
    return np.ascontiguousarray(array, dtype=np.float32).view(np.uint32)


def assert_same_weighted_graph(expected, got):
    assert np.array_equal(expected.indptr, got.indptr)
    assert np.array_equal(expected.indices, got.indices)
    assert got.weights is not None and np.array_equal(bits(expected.weights), bits(got.weights))


def edge_list(graph):
    """The directed edges of a CSR graph as (src, dst, weights)."""
    src = np.repeat(np.arange(graph.get_number_of_nodes()), np.diff(graph.indptr))
    return src, graph.indices, graph.weights


def er_weighted(er_graph):
    """The ER fixture with weights spanning e^-7 .. e^7, 5 % of them exactly zero."""
    rng = np.random.default_rng(7)
    weights = np.exp(rng.uniform(-7, 7, er_graph.indices.shape[0])).astype(np.float32)
    weights[rng.random(weights.shape[0]) < 0.05] = 0.0
    return CSRGraph(er_graph.indptr, er_graph.indices, weights=weights, name="er_weighted")


def star_weighted(leaves=(1 << 17) + 5):
    """A star whose hub row has more than 2^17 edges; every leaf row has degree 1."""
    rng = np.random.default_rng(3)
    src = np.zeros(leaves, dtype=np.int64)
    dst = np.arange(1, leaves + 1)
    weights = rng.uniform(0.0, 4.0, leaves).astype(np.float32)
    weights[rng.random(leaves) < 0.1] = 0.0
    return csr_from_edges(src, dst, leaves + 1, weights=weights, name="star")


def with_zero_rows(graph):
    """Row 5 weighs nothing at all, row 6 holds one zero-weight edge."""
    weights = graph.weights.copy()
    weights[graph.indptr[5]:graph.indptr[6]] = 0.0
    weights[graph.indptr[6]] = 0.0
    return CSRGraph(graph.indptr, graph.indices, weights=weights, name=graph.get_name() + "_zero_rows")


# ---- 1. ingest ----
@pytest.mark.parametrize("symmetrise", [True, False])
def test_weighted_ingest_small_ppi(small_ppi_weighted, symmetrise):
    src, dst, weights = edge_list(small_ppi_weighted)
    expected = csr_from_edges(src, dst, 1064, symmetrise=symmetrise, weights=weights)
    assert_same_weighted_graph(expected, csr_from_edges_gpu(src, dst, 1064, symmetrise=symmetrise, weights=weights))
    resident = device_graph_from_edges(src, dst, 1064, symmetrise=symmetrise, weights=weights)
    assert resident.has_edge_weights() and not resident.has_negative_edge_weights()
    assert_same_weighted_graph(expected, resident.to_host())
    if symmetrise:
        assert_same_weighted_graph(small_ppi_weighted, resident.to_host())


@pytest.mark.parametrize("symmetrise", [True, False])
def test_weighted_ingest_random_edges(symmetrise):
    rng = np.random.default_rng(5)
    n = 5000
    src = rng.integers(0, n, 60000)
    dst = rng.integers(0, n, 60000)
    weights = np.exp(rng.uniform(-5, 5, 60000)).astype(np.float32)
    weights[rng.random(60000) < 0.03] = 0.0
    src[:100] = dst[:100]          # self-loops are dropped (their weights too)
    src[100:200] = src[200:300]    # duplicates with other weights: the first occurrence wins
    dst[100:200] = dst[200:300]
    src[300:400], dst[300:400] = dst[400:500], src[400:500]  # an edge and its reverse, weighted apart
    expected = csr_from_edges(src, dst, n, symmetrise=symmetrise, weights=weights)
    assert_same_weighted_graph(expected, csr_from_edges_gpu(src, dst, n, symmetrise=symmetrise, weights=weights))
    assert_same_weighted_graph(expected, device_graph_from_edges(src, dst, n, symmetrise=symmetrise,
                                                                 weights=weights).to_host())


@pytest.mark.parametrize("symmetrise", [True, False])
def test_weighted_ingest_first_occurrence_rule(symmetrise):
    # (0, 1) twice: its mirror (1, 0) exists only among the mirrors, where the first copy comes first;
    # (2, 3) and (3, 2) both as input edges: each key's own input edge precedes the other's mirror
    src = np.array([0, 2, 0, 3, 4, 4])
    dst = np.array([1, 3, 1, 2, 4, 5])
    weights = np.array([1.5, 2.5, 7.0, 9.0, 3.0, 0.0], dtype=np.float32)
    expected = csr_from_edges(src, dst, 6, symmetrise=symmetrise, weights=weights)
    got = csr_from_edges_gpu(src, dst, 6, symmetrise=symmetrise, weights=weights)
    assert_same_weighted_graph(expected, got)
    if symmetrise:
        row = {(int(u), int(v)): w for u in range(6) for v, w in
               zip(got.indices[got.indptr[u]:got.indptr[u + 1]], got.weights[got.indptr[u]:got.indptr[u + 1]])}
        assert row[(0, 1)] == 1.5 and row[(1, 0)] == 1.5 and row[(2, 3)] == 2.5 and row[(3, 2)] == 9.0


def test_weighted_ingest_edge_cases_and_errors():
    empty = csr_from_edges_gpu(np.zeros(0), np.zeros(0), 7, weights=np.zeros(0))
    assert empty.indices.shape[0] == 0 and not empty.indptr.any() and empty.weights.shape == (0,)
    resident = device_graph_from_edges(np.zeros(0), np.zeros(0), 7, weights=np.zeros(0))
    assert resident.has_edge_weights() and resident.get_directed_edge_weights().shape == (0,)
    src, dst = np.array([0, 1, 2]), np.array([1, 2, 3])
    for build in (csr_from_edges_gpu, device_graph_from_edges):
        with pytest.raises(ValueError, match="non-negative"):
            build(src, dst, 5, weights=np.array([1.0, -0.5, 2.0]))
        with pytest.raises(ValueError, match="non-negative"):
            build(src, dst, 5, weights=np.array([1.0, np.nan, 2.0]))
        with pytest.raises(ValueError, match="non-negative"):
            build(np.array([0, 1, 1]), np.array([1, 2, 1]), 5, weights=np.array([1.0, 1.0, -1.0]))  # a self-loop
        with pytest.raises(ValueError, match="not below the number of nodes"):
            build(np.array([0, 9]), np.array([1, 2]), 5, weights=np.array([1.0, 1.0]))
        with pytest.raises(ValueError, match="one entry per edge"):
            build(src, dst, 5, weights=np.array([1.0, 2.0]))
    unweighted = device_graph_from_edges(src, dst, 5)
    assert not unweighted.has_edge_weights() and unweighted.to_host().weights is None
    with pytest.raises(ValueError):
        unweighted.get_directed_edge_weights()


def test_device_graph_from_csr_round_trips_weights(small_ppi_weighted, er_graph):
    for graph in (small_ppi_weighted, er_weighted(er_graph)):
        resident = device_graph_from_csr(graph.indptr, graph.indices, graph.weights)
        assert resident.has_edge_weights()
        assert np.array_equal(bits(resident.get_directed_edge_weights()), bits(graph.weights))
        assert_same_weighted_graph(graph, resident.to_host())
    with pytest.raises(ValueError, match="non-negative"):
        device_graph_from_csr(graph.indptr, graph.indices, -graph.weights)
    with pytest.raises(ValueError, match="one entry per directed edge"):
        device_graph_from_csr(graph.indptr, graph.indices, graph.weights[:-1])


# ---- 2. the device alias tables == the oracle's ----
def alias_graphs(small_ppi_weighted, er_graph):
    er = er_weighted(er_graph)
    return [small_ppi_weighted, er, with_zero_rows(er), star_weighted()]


@pytest.mark.parametrize("normalize", [False, True])
def test_device_edge_alias_equals_oracle(small_ppi_weighted, er_graph, normalize):
    for graph in alias_graphs(small_ppi_weighted, er_graph):
        weights = graph.weights
        if normalize:
            weights = oracle.degree_normalised_weights(graph.indptr, graph.indices, graph.weights)
        expected = oracle.edge_alias(graph.indptr, weights)
        resident = device_graph_from_csr(graph.indptr, graph.indices, graph.weights)
        with Engine("SkipGram", walk_length=4, normalize_by_degree=normalize) as engine:
            engine.load_csr(graph.indptr, graph.indices, graph.weights)
            assert np.array_equal(engine.export_edge_alias(), expected), graph.get_name()
            engine.load_graph(resident)
            assert np.array_equal(engine.export_edge_alias(), expected), graph.get_name()
    if normalize:  # an unweighted graph with normalize_by_degree walks by 1 / deg(destination)
        graph = er_graph
        expected = oracle.edge_alias(graph.indptr, oracle.degree_normalised_weights(graph.indptr, graph.indices))
        with Engine("SkipGram", walk_length=4, normalize_by_degree=True) as engine:
            engine.load_graph(device_graph_from_csr(graph.indptr, graph.indices))
            assert np.array_equal(engine.export_edge_alias(), expected)


# ---- 3. walks ----
@pytest.mark.parametrize("rw,ew", [(1.0, 1.0), (2.0, 0.5), (0.25, 4.0)])
@pytest.mark.parametrize("normalize", [False, True])
def test_weighted_walks_on_resident_graphs(small_ppi_weighted, er_graph, rw, ew, normalize):
    for graph in (small_ppi_weighted, er_weighted(er_graph)):
        expected, _ = oracle.walks(graph.indptr, graph.indices, 42, 3, 2000, 48, rw, ew, weights=graph.weights,
                                   normalize_by_degree=normalize)
        resident = device_graph_from_csr(graph.indptr, graph.indices, graph.weights)
        with Engine("SkipGram", walk_length=48, return_weight=rw, explore_weight=ew,
                    normalize_by_degree=normalize) as engine:
            engine.load_graph(resident)
            assert np.array_equal(engine.walks(42, 3, 2000), expected), graph.get_name()
            engine.load_csr(graph.indptr, graph.indices, graph.weights)
            assert np.array_equal(engine.walks(42, 3, 2000), expected), graph.get_name()


def test_no_stale_edge_alias_between_loads(small_ppi_weighted, er_graph):
    """One engine: a weighted host graph, a weighted resident graph, then an unweighted one."""
    g = small_ppi_weighted
    other = np.random.default_rng(1).uniform(0.0, 2.0, g.indices.shape[0]).astype(np.float32)
    kw = dict(walk_length=40, return_weight=2.0, explore_weight=0.5)
    with Engine("SkipGram", **kw) as engine:
        engine.load_csr(g.indptr, g.indices, g.weights)
        want, _ = oracle.walks(g.indptr, g.indices, 5, 0, 1500, 40, 2.0, 0.5, weights=g.weights)
        assert np.array_equal(engine.walks(5, 0, 1500), want)
        engine.load_graph(device_graph_from_csr(g.indptr, g.indices, other))
        want, _ = oracle.walks(g.indptr, g.indices, 5, 0, 1500, 40, 2.0, 0.5, weights=other)
        assert np.array_equal(engine.walks(5, 0, 1500), want)
        assert np.array_equal(engine.export_edge_alias(), oracle.edge_alias(g.indptr, other))
        engine.load_graph(device_graph_from_csr(g.indptr, g.indices))
        want, _ = oracle.walks(g.indptr, g.indices, 5, 0, 1500, 40, 2.0, 0.5)
        assert np.array_equal(engine.walks(5, 0, 1500), want)
        with pytest.raises(RuntimeError, match="no edge alias table"):
            engine.export_edge_alias()


# ---- 4. embedders, deterministic ----
def test_embedders_on_a_weighted_device_graph(small_ppi_weighted):
    from embiggen_b200.embedders import DeepWalkGloVeB200, Node2VecCBOWB200, Node2VecSkipGramB200
    g = small_ppi_weighted
    resident = device_graph_from_csr(g.indptr, g.indices, g.weights)
    for cls, extra in ((Node2VecSkipGramB200, dict(iterations=1, return_weight=2.0, explore_weight=0.5)),
                       (Node2VecCBOWB200, dict(iterations=1, return_weight=0.25, explore_weight=4.0)),
                       (DeepWalkGloVeB200, {})):  # GloVe walks once per node and epoch
        kw = dict(embedding_size=16, epochs=2, walk_length=20, verbose=False, deterministic=True, **extra)
        a = cls(**kw).fit_transform(resident, return_dataframe=False).get_all_node_embedding()
        b = cls(**kw).fit_transform(g, return_dataframe=False).get_all_node_embedding()
        assert len(a) == len(b) == 2
        for x, y in zip(a, b):
            assert x.shape == (1064, 16) and np.isfinite(x).all()
            assert np.array_equal(x, y), cls.__name__


def test_walklets_on_a_weighted_device_graph(small_ppi_weighted):
    """The resident weighted graph takes the one-pass path, the host weighted graph the
    scale-by-scale path: same walks by weight, same tables in the single-warp launch."""
    from embiggen_b200.embedders import WalkletsSkipGramB200
    g = small_ppi_weighted
    resident = device_graph_from_csr(g.indptr, g.indices, g.weights)
    kw = dict(embedding_size=12, window_size=3, epochs=2, walk_length=20, iterations=1, deterministic=True,
              chunk_walks=300, return_weight=2.0, explore_weight=0.5)
    one_pass = WalkletsSkipGramB200(**kw).fit_transform(resident, return_dataframe=False).get_all_node_embedding()
    by_scale = WalkletsSkipGramB200(**kw).fit_transform(g, return_dataframe=False).get_all_node_embedding()
    assert len(one_pass) == len(by_scale) == 6
    for a, b in zip(one_pass, by_scale):
        assert np.array_equal(a, b)
