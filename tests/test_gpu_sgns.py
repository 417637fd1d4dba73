"""SkipGram / CBOW SGD kernels against the CPU oracle, through the C ABI.

Deterministic mode (one warp, ascending walk order) must reproduce the oracle's tables bit
for bit; the Hogwild production launch is compared by tolerance (update order differs).
"""
import numpy as np
import pytest

import oracle
from conftest import heldout_sgns_loss, tiny_graphs
from embiggen_b200.engine import Engine

pytestmark = pytest.mark.gpu

SEED = 42


def run_pair(graph, model, D, L, w, K, rw, ew, n_walks, lr=0.05, deterministic=True,
             use_alias=True, normalize=False, clip=6.0, alpha=0.75, scale=False, downsample=False):
    n = graph.get_number_of_nodes()
    walks, _ = oracle.walks(graph.indptr, graph.indices, SEED, 0, n_walks, L, rw, ew)
    t0, t1 = oracle.init_tables(n, D, SEED)
    thr = alias = None
    if use_alias:
        thr, alias = oracle.alias_build(graph.indptr, alpha)
    stats = oracle.train(model, walks, t0, t1, SEED, n, D, w, K, lr, clip, thr=thr, alias=alias,
                         indptr=graph.indptr, normalize_learning_rate_by_degree=normalize,
                         scale_by_sqrt_dim=scale, stochastic_downsample_by_degree=downsample)
    with Engine(model, embedding_size=D, walk_length=L, window_size=w, iterations=1,
                number_of_negative_samples=K, return_weight=rw, explore_weight=ew,
                clipping_value=clip, use_scale_free_distribution=use_alias,
                negative_sampling_exponent=alpha, normalize_learning_rate_by_degree=normalize,
                scale_by_sqrt_dim=scale, deterministic=deterministic,
                stochastic_downsample_by_degree=downsample,
                chunk_walks=n_walks) as engine:
        engine.load_csr(graph.indptr, graph.indices)
        engine.init_tables(SEED)
        init0, init1 = engine.export_tables()
        engine.walk_chunk(SEED, 0, n_walks, 1, 0)
        engine.train_chunk(SEED, 0, lr)
        g0, g1 = engine.export_tables()
        counters = engine.counters()
        gpu_alias = engine.export_alias() if use_alias else None
    return dict(o0=t0[:, :D], o1=t1[:, :D], g0=g0, g1=g1, init0=init0, init1=init1, stats=stats,
                counters=counters, alias=(thr, alias), gpu_alias=gpu_alias, n=n, D=D)


def test_init_tables_bit_exact(small_ppi):
    for D in (5, 100, 128, 200):
        t0, t1 = oracle.init_tables(1064, D, 1234)
        with Engine("SkipGram", embedding_size=D) as engine:
            engine.load_csr(small_ppi.indptr, small_ppi.indices)
            engine.init_tables(1234)
            g0, g1 = engine.export_tables()
        assert np.array_equal(g0, t0[:, :D]) and np.array_equal(g1, t1[:, :D])
        assert np.abs(g0).max() <= 0.5 / D and g0.std() > 0


@pytest.mark.parametrize("alpha", [0.0, 0.5, 0.75, 1.0, 0.6])
def test_alias_table_bit_exact(rmat_graph, alpha):
    alpha = float(np.float32(alpha))  # b2e_config carries the exponent as a C float
    thr, alias = oracle.alias_build(rmat_graph.indptr, alpha)
    with Engine("SkipGram", negative_sampling_exponent=alpha) as engine:
        engine.load_csr(rmat_graph.indptr, rmat_graph.indices)
        g_thr, g_alias = engine.export_alias()
    assert np.array_equal(g_thr, thr) and np.array_equal(g_alias, alias)


@pytest.mark.parametrize("model,D,K,w", [
    ("SkipGram", 100, 10, 4), ("CBOW", 128, 10, 4), ("SkipGram", 5, 3, 1), ("CBOW", 5, 5, 2),
    ("SkipGram", 200, 10, 5), ("CBOW", 300, 4, 3), ("SkipGram", 64, 20, 2), ("SkipGram", 128, 0, 3),
    ("SkipGram", 300, 5, 3), ("CBOW", 100, 5, 16), ("CBOW", 100, 10, 16),
])
def test_deterministic_tables_bit_exact(small_ppi, model, D, K, w):
    r = run_pair(small_ppi, model, D, 32, w, K, 0.25, 4.0, n_walks=300)
    assert r["counters"]["pairs"] == r["stats"]["pairs"]
    assert r["counters"]["targets"] == r["stats"]["targets"]
    assert np.array_equal(r["g0"], r["o0"])
    assert np.array_equal(r["g1"], r["o1"])
    assert not np.array_equal(r["g0"], r["init0"])
    assert np.isclose(r["counters"]["loss_sum"], r["stats"]["loss_sum"], rtol=1e-4)


@pytest.mark.parametrize("model", ["SkipGram", "CBOW"])
def test_deterministic_options(rmat_graph, model):
    """uniform negatives, lr / degree, dot / sqrt(D), tight clipping: still bit exact."""
    for kwargs in (dict(use_alias=False), dict(normalize=True, lr=0.5), dict(scale=True),
                   dict(clip=0.01, lr=0.5), dict(alpha=1.0), dict(downsample=True)):
        r = run_pair(rmat_graph, model, 100, 24, 3, 7, 2.0, 0.5, n_walks=200, **kwargs)
        assert np.array_equal(r["g0"], r["o0"]), kwargs
        assert np.array_equal(r["g1"], r["o1"]), kwargs
        assert r["counters"]["targets"] == r["stats"]["targets"]


@pytest.mark.parametrize("model,D,K", [("SkipGram", 100, 10), ("CBOW", 128, 10), ("SkipGram", 200, 5),
                                       ("CBOW", 300, 20)])
def test_stochastic_downsample_by_degree(small_ppi, model, D, K):
    """Pipelined and generic kernels: bit exact in the single-warp launch, the same pairs and
    targets as the oracle in the production launch, and fewer pairs than without the option."""
    r = run_pair(small_ppi, model, D, 32, 4, K, 0.25, 4.0, n_walks=300, downsample=True)
    assert np.array_equal(r["g0"], r["o0"]) and np.array_equal(r["g1"], r["o1"])
    assert r["counters"]["pairs"] == r["stats"]["pairs"]
    full = run_pair(small_ppi, model, D, 32, 4, K, 0.25, 4.0, n_walks=300, deterministic=False)
    hog = run_pair(small_ppi, model, D, 32, 4, K, 0.25, 4.0, n_walks=300, deterministic=False,
                   downsample=True)
    assert (hog["counters"]["pairs"], hog["counters"]["targets"]) == \
        (hog["stats"]["pairs"], hog["stats"]["targets"])
    assert hog["counters"]["pairs"] < full["counters"]["pairs"]


@pytest.mark.parametrize("model,D", [("SkipGram", 100), ("CBOW", 128)])
def test_hogwild_tracks_oracle(small_ppi, model, D):  # 2 iterations of 1064 start nodes
    """Production launch (concurrent walks, racy updates): same pair / target counts as the
    sequential oracle; the mean pair loss of the first pass stays within 10 % of it (updates
    of concurrently trained walks do not see each other, the staleness Hogwild accepts)."""
    r = run_pair(small_ppi, model, D, 128, 4, 10, 0.25, 4.0, n_walks=2128, deterministic=False)
    assert r["counters"]["pairs"] == r["stats"]["pairs"]
    assert r["counters"]["targets"] == r["stats"]["targets"]
    oracle_loss = r["stats"]["loss_sum"] / r["stats"]["pairs"]
    gpu_loss = r["counters"]["loss_sum"] / r["counters"]["pairs"]
    print(model, 'oracle loss', oracle_loss, 'gpu loss', gpu_loss)
    assert abs(gpu_loss - oracle_loss) <= (0.10 if model == 'SkipGram' else 0.25) * oracle_loss
    assert np.isfinite(r["g0"]).all() and np.isfinite(r["g1"]).all()
    # both runs reach the same quality: SGNS objective on a held-out sample of walks
    if model == "SkipGram":
        init = heldout_sgns_loss(small_ppi, r["init0"], r["init1"])
        oracle_quality = heldout_sgns_loss(small_ppi, r["o0"], r["o1"])
        gpu_quality = heldout_sgns_loss(small_ppi, r["g0"], r["g1"])
        print("held-out loss: init", init, "oracle", oracle_quality, "gpu", gpu_quality)
        assert gpu_quality < 0.8 * init
        assert abs(gpu_quality - oracle_quality) <= 0.10 * oracle_quality


def test_fit_matches_oracle_fit(small_ppi):
    """b2e_fit (host buffers in/out, chunked pipeline) == oracle.fit in deterministic mode."""
    kw = dict(embedding_size=20, epochs=2, iterations=1, walk_length=16, window_size=2,
              learning_rate=0.05, learning_rate_decay=0.9, return_weight=0.25, explore_weight=4.0)
    for model in ("SkipGram", "CBOW"):
        o0, o1, o_loss = oracle.fit(model, small_ppi.indptr, small_ppi.indices, SEED, negatives=5,
                                    chunk_walks=300, **kw)
        with Engine(model, number_of_negative_samples=5, deterministic=True, chunk_walks=300,
                    **kw) as engine:
            engine.load_csr(small_ppi.indptr, small_ppi.indices)
            g0, g1, g_loss = engine.fit(SEED)
        if model == "CBOW":  # role order [central, contextual]: CBOW's central table is T1
            g0, g1 = g1, g0
        assert np.array_equal(g0, o0[:, :20]) and np.array_equal(g1, o1[:, :20])
        assert np.allclose(g_loss, o_loss, rtol=1e-4)


def test_loss_decreases_over_epochs(er_graph):
    with Engine("SkipGram", embedding_size=32, epochs=4, iterations=2, walk_length=32,
                window_size=3, number_of_negative_samples=5, learning_rate=0.05) as engine:
        engine.load_csr(er_graph.indptr, er_graph.indices)
        t0, t1, losses = engine.fit(SEED)
    assert losses[-1] < losses[0]
    assert np.isfinite(t0).all() and np.isfinite(t1).all()


def test_error_paths(small_ppi):
    with pytest.raises(ValueError):
        Engine("SkipGram", embedding_size=0)
    with pytest.raises(ValueError):
        Engine("SkipGram", number_of_negative_samples=64)
    with Engine("SkipGram") as engine:
        with pytest.raises(RuntimeError):
            engine.init_tables(1)  # before load_csr
        with pytest.raises(ValueError):
            engine.load_csr(np.zeros(1, dtype=np.int64), np.zeros(0, dtype=np.uint32))
        with pytest.raises(ValueError):
            engine.load_csr(np.zeros(5, dtype=np.int64), np.zeros(0, dtype=np.uint32))


def test_baseline_config_c1(small_ppi):
    """BASELINE.json configs[0]: Node2Vec SkipGram on the reference's tests/data graph, dim=100,
    walk_length=128, window=4, 1 epoch, the reference's default p/q and iterations, through the
    embedder class; the 8-thread Hogwild oracle stands where the Ensmallen CPU run would."""
    from embiggen_b200.embedders import Node2VecSkipGramB200
    kw = dict(embedding_size=100, walk_length=128, window_size=4, epochs=1, iterations=10,
              number_of_negative_samples=10, learning_rate=0.01, learning_rate_decay=0.9)
    oracle.set_threads(8)
    try:
        o0, o1, expected = oracle.fit("SkipGram", small_ppi.indptr, small_ppi.indices, 42, negatives=10,
                                      return_weight=0.25, explore_weight=4.0,
                                      **{k: v for k, v in kw.items() if k != "number_of_negative_samples"})
    finally:
        oracle.set_threads(1)
    model = Node2VecSkipGramB200(return_weight=0.25, explore_weight=4.0, random_state=42, verbose=False, **kw)
    result = model.fit_transform(small_ppi, return_dataframe=False)
    central, contextual = result.get_all_node_embedding()
    assert central.shape == (1064, 100) and contextual.shape == (1064, 100)
    got = model.get_losses()
    print("C1 mean pair loss: oracle", expected, "gpu", got)
    assert abs(got[0] - expected[0]) <= 0.10 * expected[0]
    quality_oracle = heldout_sgns_loss(small_ppi, o0[:, :100], o1[:, :100], return_weight=0.25, explore_weight=4.0)
    quality_gpu = heldout_sgns_loss(small_ppi, central, contextual, return_weight=0.25, explore_weight=4.0)
    print("C1 held-out objective: oracle", quality_oracle, "gpu", quality_gpu)
    assert abs(quality_gpu - quality_oracle) <= 0.10 * quality_oracle


# ---- Walklets (b2e_config.walklet_scale; walklet_split_kernel) ----
@pytest.mark.parametrize("model,k,L", [("SkipGram", 2, 32), ("SkipGram", 3, 31), ("CBOW", 2, 33), ("CBOW", 5, 32)])
def test_walklets_deterministic_bit_exact(small_ppi, model, k, L):
    n, D, K, n_walks, lr = small_ppi.get_number_of_nodes(), 25, 5, 200, 0.05
    walks, _ = oracle.walks(small_ppi.indptr, small_ppi.indices, SEED, 0, n_walks, L, 0.25, 4.0)
    t0, t1 = oracle.init_tables(n, D, SEED)
    thr, alias = oracle.alias_build(small_ppi.indptr, 0.75)
    stats = oracle.train_walklets(model, walks, k, t0, t1, SEED, n, D, 1, K, lr, thr=thr, alias=alias)
    for deterministic in (True, False):
        with Engine(model, embedding_size=D, walk_length=L, window_size=1, iterations=1,
                    number_of_negative_samples=K, return_weight=0.25, explore_weight=4.0,
                    walklet_scale=k, deterministic=deterministic, chunk_walks=n_walks) as engine:
            engine.load_csr(small_ppi.indptr, small_ppi.indices)
            assert np.array_equal(engine.walks(SEED, 0, n_walks), walks)  # the export stays raw
            engine.init_tables(SEED)
            engine.reset_counters()
            engine.walk_chunk(SEED, 0, n_walks, 1, 0)
            engine.train_chunk(SEED, 0, lr)
            g0, g1 = engine.export_tables()
            counters = engine.counters()
            assert (counters["pairs"], counters["targets"]) == (stats["pairs"], stats["targets"])
            if deterministic:
                assert np.array_equal(g0, t0[:, :D]) and np.array_equal(g1, t1[:, :D])
                # host walks take the same route
                engine.init_tables(SEED)
                engine.train_host_walks(SEED, walks, lr)
                h0, h1 = engine.export_tables()
                assert np.array_equal(h0, g0) and np.array_equal(h1, g1)


def test_walklets_embedder(small_ppi):
    from embiggen_b200.embedders import WalkletsSkipGramB200, WalkletsCBOWB200
    for cls in (WalkletsSkipGramB200, WalkletsCBOWB200):
        model = cls(embedding_size=24, window_size=3, epochs=2, walk_length=32, iterations=2)
        result = model.fit_transform(small_ppi, return_dataframe=False)
        tables = result.get_all_node_embedding()
        assert len(tables) == 6 and all(t.shape == (1064, 8) and np.isfinite(t).all() for t in tables)
        assert not np.array_equal(tables[0], tables[2])  # scales differ
        losses = model.get_losses()
        assert len(losses) == 2 and losses[1] < losses[0]
        frames = model.fit_transform(small_ppi).get_all_node_embedding()
        assert list(frames[0].index) == small_ppi.get_node_names()


def test_walklets_one_pass_equals_scale_by_scale(small_ppi_weighted, small_ppi):
    """The one-pass schedule (walk a chunk once, every scale adopts it: engine.fit_scales) trains
    exactly what the scale-by-scale path trains: in the single-warp launch the tables are equal
    bit for bit.  A weighted graph takes the scale-by-scale path (same walks by weight)."""
    from embiggen_b200.embedders import WalkletsCBOWB200, WalkletsSkipGramB200
    for cls in (WalkletsSkipGramB200, WalkletsCBOWB200):
        kw = dict(embedding_size=12, window_size=3, epochs=2, walk_length=20, iterations=1,
                  deterministic=True, chunk_walks=300, return_weight=2.0, explore_weight=0.5)
        one_pass = cls(**kw).fit_transform(small_ppi, return_dataframe=False).get_all_node_embedding()
        reference = []
        model = cls(**kw)
        for scale in (1, 2, 3):  # the old path, spelled out
            model._walklet_scale = scale
            reference.extend(super(type(model).__mro__[1], model)._fit_transform(
                small_ppi, return_dataframe=False).get_all_node_embedding())
        model._walklet_scale = 0
        assert len(one_pass) == len(reference) == 6
        for a, b in zip(one_pass, reference):
            assert np.array_equal(a, b)
        weighted = cls(**kw).fit_transform(small_ppi_weighted, return_dataframe=False).get_all_node_embedding()
        assert len(weighted) == 6 and all(np.isfinite(t).all() for t in weighted)


def test_alias_table_and_start_nodes_at_scale():
    """K3 on the GPU (alias_build.cu) against the oracle's sequential sweep on a skewed graph of
    1 M nodes / 16 M edges (maximum degree ~ 10^5, a third of the nodes isolated), from host
    arrays and from a resident graph, with exact-form and libm exponents."""
    from embiggen_b200.graph_gpu import rmat_gpu
    resident = rmat_gpu(20, 16_000_000, n=1_000_000, seed=3, resident=True)
    host = resident.to_host()
    sources = np.flatnonzero(np.diff(host.indptr) > 0).astype(np.uint32)
    for alpha, graph in ((0.75, resident), (0.75, host), (1.0, host), (0.6, resident), (0.0, host)):
        thr, alias = oracle.alias_build(host.indptr, float(np.float32(alpha)))
        with Engine("SkipGram", negative_sampling_exponent=alpha, walk_length=4) as engine:
            if graph is host:
                engine.load_csr(host.indptr, host.indices)
            else:
                engine.load_graph(resident)
            g_thr, g_alias = engine.export_alias()
            assert engine.number_of_sources == len(sources)
            assert np.array_equal(engine.walks(1, 0, len(sources))[:, 0], sources)  # start-node list
        assert np.array_equal(g_thr, thr) and np.array_equal(g_alias, alias), alpha


@pytest.mark.parametrize("model", ["SkipGram", "CBOW"])
def test_sink_centre_with_degree_normalised_learning_rate_stays_finite(model):
    """A walk on a directed graph ends on a sink (out-degree 0) and that token still serves as a
    centre; with normalize_learning_rate_by_degree the rate is lr / max(deg, 1), in the kernels
    and in the oracle alike (it used to be lr / 0 = inf, poisoning the tables through the shared
    negative rows)."""
    graph = tiny_graphs()["directed_dead_end"]
    for deterministic in (True, False):
        r = run_pair(graph, model, 8, 6, 2, 3, 1.0, 1.0, 40, lr=0.5, deterministic=deterministic, normalize=True)
        assert np.isfinite(r["o0"]).all() and np.isfinite(r["o1"]).all()
        assert np.isfinite(r["g0"]).all() and np.isfinite(r["g1"]).all()
        if deterministic:
            assert np.array_equal(r["g0"], r["o0"]) and np.array_equal(r["g1"], r["o1"])
