"""GPU graph ingest (C ABI b2e_csr_from_edges / b2e_synthetic_csr) against the numpy builders."""
import numpy as np
import pytest

from embiggen_b200.graph import csr_from_edges, erdos_renyi, rmat, validate_csr
from embiggen_b200.graph_gpu import csr_from_edges_gpu, erdos_renyi_gpu, rmat_gpu

pytestmark = pytest.mark.gpu


def same_graph(a, b):
    return np.array_equal(a.indptr, b.indptr) and np.array_equal(a.indices, b.indices)


@pytest.mark.parametrize("symmetrise", [True, False])
def test_csr_from_edges_matches_numpy(symmetrise):
    rng = np.random.default_rng(5)
    n = 5000
    src = rng.integers(0, n, 60000)
    dst = rng.integers(0, n, 60000)
    src[:100] = dst[:100]          # self-loops are dropped
    src[100:200] = src[200:300]    # duplicates are merged
    dst[100:200] = dst[200:300]
    expected = csr_from_edges(src, dst, n, symmetrise=symmetrise)
    got = csr_from_edges_gpu(src, dst, n, symmetrise=symmetrise)
    assert same_graph(expected, got)
    validate_csr(got.indptr, got.indices)
    assert got.is_directed() == (not symmetrise)


def test_csr_from_edges_small_ppi(small_ppi):
    """The reference's own fixture graph (tests/data/small_ppi.tsv) from its directed edge list."""
    src = np.repeat(np.arange(1064), np.diff(small_ppi.indptr))
    got = csr_from_edges_gpu(src, small_ppi.indices, 1064)
    assert same_graph(small_ppi, got)


def test_csr_from_edges_edge_cases():
    empty = csr_from_edges_gpu(np.zeros(0), np.zeros(0), 7)
    assert empty.indices.shape[0] == 0 and not empty.indptr.any()
    loops = csr_from_edges_gpu(np.arange(5), np.arange(5), 5)
    assert loops.indices.shape[0] == 0
    with pytest.raises(ValueError):
        csr_from_edges_gpu(np.array([0, 9]), np.array([1, 2]), 5)  # endpoint out of range


@pytest.mark.parametrize("n,m", [(2000, 12000), (300, 20000), (100_000, 1_000_000)])
def test_erdos_renyi_matches_numpy(n, m):
    assert same_graph(erdos_renyi(n, m, seed=7), erdos_renyi_gpu(n, m, seed=7))


@pytest.mark.parametrize("scale,m,n", [(12, 30000, 4000), (10, 5000, None), (17, 1_000_000, 100_000)])
def test_rmat_matches_numpy(scale, m, n):
    assert same_graph(rmat(scale, m, n=n, seed=11), rmat_gpu(scale, m, n=n, seed=11))


def test_full_size_shapes():
    """BASELINE C2 and C3 shapes: exact edge counts, simple, symmetric, sorted."""
    for graph, n, m in ((erdos_renyi_gpu(1_000_000, 10_000_000), 1_000_000, 10_000_000),
                        (rmat_gpu(24, 200_000_000, n=10_000_000), 10_000_000, 200_000_000)):
        assert graph.get_number_of_nodes() == n and graph.indices.shape[0] == 2 * m
        rows = np.repeat(np.arange(n, dtype=np.uint32), np.diff(graph.indptr))
        assert not (rows == graph.indices).any()                      # no self-loops
        order_ok = (graph.indices[1:] > graph.indices[:-1]) | (rows[1:] != rows[:-1])
        assert order_ok.all()                                         # sorted, no duplicates
        # symmetric: the multiset of (min, max) keys has every edge exactly twice
        lo = np.minimum(rows, graph.indices).astype(np.uint64)
        hi = np.maximum(rows, graph.indices).astype(np.uint64)
        keys = (lo << np.uint64(32)) | hi
        upper = keys[rows < graph.indices]
        lower = keys[rows > graph.indices]
        upper.sort()
        lower.sort()
        assert np.array_equal(upper, lower)


# ---- resident graphs: built on the GPU, handed to the engine without leaving HBM ----
def test_resident_graph_equals_host_graph_and_walks_identically(small_ppi):
    import oracle
    from embiggen_b200.engine import Engine
    from embiggen_b200.graph_gpu import DeviceGraph, device_graph_from_edges
    expected = rmat(12, 30000, n=4000, seed=11)
    resident = rmat_gpu(12, 30000, n=4000, seed=11, resident=True)
    assert isinstance(resident, DeviceGraph)
    assert resident.get_number_of_nodes() == 4000 and resident.get_number_of_directed_edges() == 60000
    assert same_graph(expected, resident.to_host())
    assert same_graph(erdos_renyi(2000, 12000, seed=7), erdos_renyi_gpu(2000, 12000, seed=7, resident=True).to_host())
    src = np.repeat(np.arange(1064), np.diff(small_ppi.indptr))
    assert same_graph(small_ppi, device_graph_from_edges(src, small_ppi.indices, 1064).to_host())
    # walks on the resident CSR == walks on the uploaded CSR == the oracle's
    want, _ = oracle.walks(expected.indptr, expected.indices, 3, 0, 3000, 40, 2.0, 0.5)
    kw = dict(walk_length=40, return_weight=2.0, explore_weight=0.5)
    with Engine("SkipGram", **kw) as engine:
        engine.load_csr(expected.indptr, expected.indices)  # a host graph, then the resident one
        assert np.array_equal(engine.walks(3, 0, 3000), want)
        engine.load_graph(resident)
        assert np.array_equal(engine.walks(3, 0, 3000), want)
        malformed = expected.indices.copy()
        malformed[0] = 4000  # an id out of range: found on the device, after the resident graph was let go
        with pytest.raises(ValueError):
            engine.load_csr(expected.indptr, malformed)
        with pytest.raises(RuntimeError):
            engine.walks(3, 0, 3000)  # a failed load leaves the engine without a graph
        engine.load_graph(resident)
        assert np.array_equal(engine.walks(3, 0, 3000), want)
        with Engine("SkipGram", **kw) as other:  # two engines on one resident graph
            other.load_graph(resident)
            resident.close()  # reference counted: the engines keep the arrays alive
            assert np.array_equal(other.walks(3, 0, 3000), want)
        assert np.array_equal(engine.walks(3, 0, 3000), want)  # `other` let go, this one walks on
        engine.load_csr(expected.indptr, expected.indices)  # and a host graph can replace it
        assert np.array_equal(engine.walks(3, 0, 3000), want)


def test_embedder_accepts_a_resident_graph():
    from embiggen_b200.embedders import Node2VecSkipGramB200
    resident = rmat_gpu(12, 30000, n=4000, seed=11, resident=True)
    host = resident.to_host()
    kw = dict(embedding_size=16, epochs=1, walk_length=16, iterations=1, verbose=False, deterministic=True)
    a = Node2VecSkipGramB200(**kw).fit_transform(resident, return_dataframe=False).get_all_node_embedding()
    b = Node2VecSkipGramB200(**kw).fit_transform(host, return_dataframe=False).get_all_node_embedding()
    assert a[0].shape == (4000, 16) and np.isfinite(a[0]).all() and np.isfinite(a[1]).all()
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])  # single-warp launch: same bits
