"""SkipGram with shared negatives (`shared_negatives=True`, opt-in; north_star's shared-negative
batching): one set of K negatives per centre, shared by its pairs.  The single-warp launch of
skipgram_shared_kernel (csrc/sgns_pipe.cu) against oracle/sgns.c:train_centre_shared, bit for
bit, on graphs that force every deferred-copy case (stars, paths: repeated tokens inside the
window; hubs: a negative that is a neighbour); the production launch by counts and loss."""
import numpy as np
import pytest

import oracle
from conftest import tiny_graphs
from embiggen_b200.engine import Engine

pytestmark = pytest.mark.gpu


def run(graph, D, L, w, K, rw, ew, n_walks, seed=42, lr=0.05, deterministic=True, alias=True, normalize=False,
        scale=False, downsample=False, clip=6.0, boost=1.0, first=0):
    n = graph.get_number_of_nodes()
    walks, _ = oracle.walks(graph.indptr, graph.indices, seed, first, n_walks, L, rw, ew)
    t0, t1 = oracle.init_tables(n, D, seed)
    t0 *= np.float32(boost)
    t1 *= np.float32(boost)
    start0, start1 = t0[:, :D].copy(), t1[:, :D].copy()
    thr = table = None
    if alias:
        thr, table = oracle.alias_build(graph.indptr, 0.75)
    stats = oracle.train("SkipGram", walks, t0, t1, seed, n, D, w, K, lr, clip, first_walk=first, thr=thr,
                         alias=table, indptr=graph.indptr, normalize_learning_rate_by_degree=normalize,
                         scale_by_sqrt_dim=scale, stochastic_downsample_by_degree=downsample,
                         shared_negatives=True)
    with Engine("SkipGram", embedding_size=D, walk_length=L, window_size=w, iterations=1,
                number_of_negative_samples=K, return_weight=rw, explore_weight=ew, clipping_value=clip,
                use_scale_free_distribution=alias, normalize_learning_rate_by_degree=normalize,
                scale_by_sqrt_dim=scale, stochastic_downsample_by_degree=downsample,
                deterministic=deterministic, shared_negatives=True, chunk_walks=n_walks) as engine:
        engine.load_csr(graph.indptr, graph.indices)
        engine.import_tables(start0, start1)
        engine.reset_counters()
        engine.walk_chunk(seed, first, n_walks, 1, 0)
        engine.train_chunk(seed, 0, lr)
        g0, g1 = engine.export_tables()
        counters = engine.counters()
    return dict(o0=t0[:, :D], o1=t1[:, :D], g0=g0, g1=g1, start0=start0, stats=stats, counters=counters)


def exact(r, label=None):
    assert (r["counters"]["pairs"], r["counters"]["targets"]) == (r["stats"]["pairs"], r["stats"]["targets"]), label
    assert np.array_equal(r["g0"], r["o0"]), label
    assert np.array_equal(r["g1"], r["o1"]), label


@pytest.mark.parametrize("D,K,w", [(100, 10, 4), (128, 10, 5), (5, 3, 1), (64, 15, 7), (100, 0, 2), (32, 5, 3),
                                   (1, 1, 1), (101, 7, 6)])
def test_single_warp_launch_is_bit_exact(small_ppi, D, K, w):
    r = run(small_ppi, D, 32, w, K, 0.25, 4.0, n_walks=300)
    exact(r)
    assert r["stats"]["pairs"] > 0 and not np.array_equal(r["g0"], r["start0"])
    assert np.isclose(r["counters"]["loss_sum"], r["stats"]["loss_sum"], rtol=1e-4)


def test_options_are_bit_exact(rmat_graph):
    """uniform negatives, lr / degree, dot / sqrt(D), tight clipping, centre downsampling, rows far
    outside the linear range of the sigmoid: return_weight 2 makes a-b-a patterns (a context token
    twice in a window) common."""
    for kwargs in (dict(alias=False), dict(normalize=True, lr=0.5), dict(scale=True, boost=30.0),
                   dict(clip=0.01, lr=0.5), dict(downsample=True), dict(boost=40.0, lr=0.3),
                   dict(downsample=True, boost=25.0, normalize=True, lr=0.4)):
        exact(run(rmat_graph, 100, 24, 3, 7, 2.0, 0.5, n_walks=200, **kwargs), kwargs)


def fuzz_cases():
    rng = np.random.default_rng(20261018)
    graphs = ["star", "path", "triangle_pendant", "small_ppi", "two_components_isolated", "er", "directed_dead_end"]
    out = []
    for index in range(42):
        out.append(dict(
            graph=graphs[index % len(graphs)],
            D=int(rng.choice([1, 3, 4, 5, 17, 32, 64, 100, 101, 128])), K=int(rng.integers(0, 16)),
            w=int(rng.integers(1, 8)), L=int(rng.choice([2, 3, 5, 9, 16, 33, 40])),
            rw=float(rng.choice([1.0, 0.25, 2.0, 7.5])), ew=float(rng.choice([1.0, 4.0, 0.5])),
            lr=float(rng.choice([0.025, 0.1, 0.5])), alias=bool(rng.integers(0, 2)), scale=bool(rng.integers(0, 2)),
            normalize=bool(rng.integers(0, 2)), downsample=bool(rng.integers(0, 2)),
            seed=int(rng.integers(0, 2 ** 62))))
    return out


@pytest.mark.parametrize("case", fuzz_cases(),
                         ids=lambda c: f"{c['graph']}-D{c['D']}-K{c['K']}-w{c['w']}-L{c['L']}" + ("-S" if c["downsample"] else ""))
def test_random_shapes_are_bit_exact(case, small_ppi, er_graph):
    graph = {"small_ppi": small_ppi, "er": er_graph}.get(case["graph"]) or tiny_graphs()[case["graph"]]
    n_src = int((np.diff(graph.indptr) > 0).sum())
    r = run(graph, case["D"], case["L"], case["w"], case["K"], case["rw"], case["ew"], min(3 * n_src + 1, 160),
            seed=case["seed"], lr=case["lr"], alias=case["alias"], normalize=case["normalize"], scale=case["scale"],
            downsample=case["downsample"], boost=20.0, first=11)
    exact(r, case)


def test_production_launch_tracks_the_oracle(small_ppi):
    """Concurrent walks (Hogwild; context rows by atomic adds): the same pairs and targets as the
    sequential oracle.  The mean pair loss of the first pass is compared loosely and from one side
    mostly: measured 2.27 against the oracle's 2.87 (profiles/r02v_pytest.txt).  The gap is Hogwild
    staleness, not a defect of the kernel: on workloads where concurrent walks share no row that
    changes, this production launch (skipgram_shared_kernel<10, 4> over the persistent grid) equals
    the sequential oracle bit for bit (test_gpu_production_launch.py).  Here concurrent walks push
    a shared context row from stale copies and all their pushes are ADDED (red.global.add), which
    from the tiny initial rows acts like a larger step; the oracle run as OpenMP Hogwild
    (non-atomic rows) moves the other way by 1 %."""
    r = run(small_ppi, 100, 128, 4, 10, 0.25, 4.0, n_walks=2128, deterministic=False)
    assert (r["counters"]["pairs"], r["counters"]["targets"]) == (r["stats"]["pairs"], r["stats"]["targets"])
    expected = r["stats"]["loss_sum"] / r["stats"]["pairs"]
    got = r["counters"]["loss_sum"] / r["counters"]["pairs"]
    print("shared negatives: oracle loss per pair", expected, "gpu", got)
    assert np.isfinite(r["g0"]).all() and np.isfinite(r["g1"]).all()
    assert 0.6 * expected < got < 1.1 * expected


def test_fewer_target_rows_than_the_per_pair_draws(small_ppi):
    """What the mode is for: rows scored per pair fall from K + 1 to about 1 + K / m."""
    shared = run(small_ppi, 100, 64, 4, 10, 0.25, 4.0, n_walks=500, deterministic=False)["counters"]
    with Engine("SkipGram", embedding_size=100, walk_length=64, window_size=4, iterations=1,
                number_of_negative_samples=10, return_weight=0.25, explore_weight=4.0, chunk_walks=500) as engine:
        engine.load_csr(small_ppi.indptr, small_ppi.indices)
        engine.init_tables(42)
        engine.walk_chunk(42, 0, 500, 1, 0)
        engine.train_chunk(42, 0, 0.05)
        plain = engine.counters()
    assert shared["pairs"] == plain["pairs"]
    assert shared["targets"] / shared["pairs"] < 2.6 < 10.0 < plain["targets"] / plain["pairs"]


@pytest.mark.parametrize("kwargs", [dict(model="CBOW"), dict(window_size=8), dict(number_of_negative_samples=16),
                                    dict(embedding_size=132), dict(walk_length=1025)])
def test_unsupported_shapes_are_refused(kwargs):
    """No silent switch to the per-pair kernel: the configuration is an error at construction."""
    arguments = dict(model="SkipGram", embedding_size=100, walk_length=32, window_size=4,
                     number_of_negative_samples=10, shared_negatives=True)
    arguments.update(kwargs)
    with pytest.raises(ValueError, match="shared_negatives"):
        Engine(arguments.pop("model"), **arguments)


def test_embedder_keyword_and_link_quality(small_ppi):
    """`shared_negatives=True` on the reference-shaped class: the embedding separates held-out edges
    from non-edges about as well as the per-pair model (AUROC of the dot product; the expected
    gradient is the same, its variance is not)."""
    from embiggen_b200.embedders import Node2VecSkipGramB200
    rng = np.random.default_rng(5)
    indptr, indices = small_ppi.indptr, small_ppi.indices
    n = small_ppi.get_number_of_nodes()
    sources = np.repeat(np.arange(n), np.diff(indptr))
    edges = set(zip(sources.tolist(), indices.tolist()))
    positives = np.array([e for e in edges if e[0] < e[1]])
    negatives = []
    while len(negatives) < len(positives):
        a, b = (int(x) for x in rng.integers(0, n, 2))
        if a != b and (a, b) not in edges:
            negatives.append((a, b))
    negatives = np.array(negatives)

    def auroc(shared):
        model = Node2VecSkipGramB200(embedding_size=32, epochs=10, walk_length=32, iterations=4, window_size=4,
                                     return_weight=1.0, explore_weight=1.0, learning_rate=0.05, verbose=False,
                                     shared_negatives=shared)
        assert model.parameters()["shared_negatives"] is shared
        central, contextual = model.fit_transform(small_ppi, return_dataframe=False).get_all_node_embedding()
        score = lambda pairs: np.einsum("ij,ij->i", central[pairs[:, 0]], contextual[pairs[:, 1]]) + \
            np.einsum("ij,ij->i", central[pairs[:, 1]], contextual[pairs[:, 0]])
        p, q = score(positives), score(negatives)
        ranks = np.argsort(np.argsort(np.concatenate([p, q]))) + 1
        return (ranks[:len(p)].sum() - len(p) * (len(p) + 1) / 2) / (len(p) * len(q))

    plain, shared = auroc(False), auroc(True)
    print("AUROC of training edges vs random non-edges: per-pair negatives", plain, "shared", shared)
    assert plain > 0.7 and shared > plain - 0.05
