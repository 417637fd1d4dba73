"""Randomised parity sweep: the single-warp CUDA launch against the CPU oracle, bit for bit, over
shapes the fixed cases do not reach (odd embedding sizes, K from 0 to 15, wide windows, tiny
walks) on graphs that force repeated tokens inside a window (stars, paths, hub-and-leaf PPI) --
the cases where the asynchronous pipeline must defer a copy or add a row twice."""
import numpy as np
import pytest

import oracle
from conftest import tiny_graphs
from embiggen_b200.engine import Engine

pytestmark = pytest.mark.gpu


def cases():
    rng = np.random.default_rng(20261017)
    graphs = ["small_ppi", "star", "path", "triangle_pendant", "two_components_isolated", "er"]
    out = []
    for index in range(48):
        out.append(dict(
            graph=graphs[index % len(graphs)],
            model="SkipGram" if index % 2 == 0 else "CBOW",
            D=int(rng.choice([1, 3, 4, 5, 17, 32, 64, 100, 101, 128, 130, 200])),
            K=int(rng.integers(0, 16)),
            w=int(rng.integers(1, 9)),
            L=int(rng.choice([2, 3, 5, 9, 16, 33, 40])),
            rw=float(rng.choice([1.0, 0.25, 2.0, 7.5])),
            ew=float(rng.choice([1.0, 4.0, 0.5])),
            lr=float(rng.choice([0.025, 0.1, 0.5])),
            alias=bool(rng.integers(0, 2)),
            scale=bool(rng.integers(0, 2)),
            normalize=bool(rng.integers(0, 2)),
            seed=int(rng.integers(0, 2 ** 62)),
        ))
    # walks longer than the pipelined kernels stage (1024 tokens) take the generic SkipGram kernel
    out.append(dict(graph="small_ppi", model="SkipGram", D=100, K=5, w=3, L=1040, rw=0.25, ew=4.0, lr=0.025,
                    alias=True, scale=False, normalize=False, seed=20261021))
    return out


@pytest.mark.parametrize("case", cases(), ids=lambda c: f"{c['model']}-{c['graph']}-D{c['D']}-K{c['K']}-w{c['w']}-L{c['L']}")
def test_single_warp_launch_is_bit_exact(case, small_ppi, er_graph):
    graph = {"small_ppi": small_ppi, "er": er_graph}.get(case["graph"]) or tiny_graphs()[case["graph"]]
    n = graph.get_number_of_nodes()
    n_src = int((np.diff(graph.indptr) > 0).sum())
    n_walks = min(3 * n_src + 1, 160)
    seed, D, L = case["seed"], case["D"], case["L"]
    walks, _ = oracle.walks(graph.indptr, graph.indices, seed, 11, n_walks, L, case["rw"], case["ew"])
    t0, t1 = oracle.init_tables(n, D, seed)
    t0 *= 20.0  # leave the linear range of the sigmoid
    t1 *= 20.0
    thr = alias = None
    if case["alias"]:
        thr, alias = oracle.alias_build(graph.indptr, 0.75)
    stats = oracle.train(case["model"], walks, t0, t1, seed, n, D, case["w"], case["K"], case["lr"], 6.0,
                         first_walk=11, thr=thr, alias=alias, indptr=graph.indptr,
                         normalize_learning_rate_by_degree=case["normalize"], scale_by_sqrt_dim=case["scale"])
    with Engine(case["model"], embedding_size=D, walk_length=L, window_size=case["w"], iterations=1,
                number_of_negative_samples=case["K"], return_weight=case["rw"], explore_weight=case["ew"],
                use_scale_free_distribution=case["alias"], normalize_learning_rate_by_degree=case["normalize"],
                scale_by_sqrt_dim=case["scale"], deterministic=True, chunk_walks=n_walks) as engine:
        engine.load_csr(graph.indptr, graph.indices)
        assert np.array_equal(engine.walks(seed, 11, n_walks), walks)
        init0, init1 = oracle.init_tables(n, D, seed)
        engine.import_tables(init0[:, :D] * np.float32(20.0), init1[:, :D] * np.float32(20.0))
        engine.reset_counters()
        engine.walk_chunk(seed, 11, n_walks, 1, 0)
        engine.train_chunk(seed, 0, case["lr"])
        g0, g1 = engine.export_tables()
        counters = engine.counters()
    assert (counters["pairs"], counters["targets"]) == (stats["pairs"], stats["targets"])
    assert np.array_equal(g0, t0[:, :D])
    assert np.array_equal(g1, t1[:, :D])


def option_cases():
    rng = np.random.default_rng(777)
    graphs = ["small_ppi", "star", "directed_dead_end", "er", "triangle_pendant", "rmat"]
    out = []
    for index in range(36):
        model = ["SkipGram", "CBOW", "GloVe"][index % 3]
        out.append(dict(
            graph=graphs[index % len(graphs)], model=model,
            D=int(rng.choice([3, 16, 100, 130])), K=int(rng.integers(0, 12)), w=int(rng.integers(1, 6)),
            L=int(rng.choice([5, 9, 16, 33])),
            rw=float(rng.choice([1.0, 0.25, 2.0])), ew=float(rng.choice([1.0, 4.0, 0.5])),
            weighted=bool(rng.integers(0, 2)), normalize=bool(rng.integers(0, 2)),
            cn=float(rng.choice([1.0, 0.2, 3.0])), ce=float(rng.choice([1.0, 0.5, 4.0])),
            downsample=bool(rng.integers(0, 2)) and model != "GloVe",
            walklet=int(rng.choice([0, 0, 2, 3])) if model != "GloVe" else 0,
            alpha=float(rng.choice([0.5, 0.75, 1.0])), seed=int(rng.integers(0, 2 ** 62)),
        ))
    return out


@pytest.mark.parametrize("case", option_cases(), ids=lambda c: (
    f"{c['model']}-{c['graph']}-D{c['D']}-L{c['L']}-" + "".join(
        flag for flag, on in (("W", c["weighted"]), ("N", c["normalize"]), ("Tn", c["cn"] != 1.0),
                              ("Te", c["ce"] != 1.0), ("S", c["downsample"]), (f"k{c['walklet']}", c["walklet"]))
        if on)))
def test_options_of_the_widened_path_are_bit_exact(case, small_ppi, er_graph, rmat_graph):
    """Weights, degree normalisation, typed walks, centre downsampling, Walklets and GloVe in
    random combinations: walks bit-exact, single-warp training bit-exact."""
    graph = {"small_ppi": small_ppi, "er": er_graph, "rmat": rmat_graph}.get(case["graph"]) \
        or tiny_graphs()[case["graph"]]
    n, nnz = graph.get_number_of_nodes(), graph.indices.shape[0]
    rng = np.random.default_rng(case["seed"] % (2 ** 32))
    weights = (np.exp(rng.uniform(-3, 3, nnz))).astype(np.float32) if case["weighted"] else None
    node_types = rng.integers(0, 3, n).astype(np.uint32)
    edge_types = rng.integers(0, 3, nnz).astype(np.uint32)
    n_src = int((np.diff(graph.indptr) > 0).sum())
    n_walks = min(3 * n_src + 1, 120)
    seed, D, L, w = case["seed"], case["D"], case["L"], case["w"]
    if case["walklet"] >= L:
        case = dict(case, walklet=0)
    walks, oc = oracle.walks(graph.indptr, graph.indices, seed, 5, n_walks, L, case["rw"], case["ew"],
                             weights=weights, normalize_by_degree=case["normalize"], node_types=node_types,
                             edge_types=edge_types, change_node_type_weight=case["cn"],
                             change_edge_type_weight=case["ce"])
    t0, t1 = oracle.init_tables(n, D, seed)
    t0 *= 20.0
    t1 *= 20.0
    window = 1 if case["walklet"] else w
    kw = dict(embedding_size=D, walk_length=L, window_size=window, iterations=1,
              number_of_negative_samples=case["K"], return_weight=case["rw"], explore_weight=case["ew"],
              normalize_by_degree=case["normalize"], change_node_type_weight=case["cn"],
              change_edge_type_weight=case["ce"], stochastic_downsample_by_degree=case["downsample"],
              walklet_scale=case["walklet"], glove_alpha=case["alpha"], deterministic=True,
              chunk_walks=n_walks)
    with Engine(case["model"], **kw) as engine:
        engine.load_csr(graph.indptr, graph.indices, weights)
        engine.load_types(node_types, edge_types)
        assert np.array_equal(engine.walks(seed, 5, n_walks), walks)
        gc = engine.counters()
        assert (gc["walk_steps"], gc["walk_trials"], gc["walk_searches"]) == (oc["steps"], oc["trials"], oc["searches"])
        init0, init1 = oracle.init_tables(n, D, seed)
        engine.import_tables(init0[:, :D] * np.float32(20.0), init1[:, :D] * np.float32(20.0))
        engine.reset_counters()
        if case["model"] == "GloVe":
            centre, context, count = oracle.cooccurrence(walks, w)
            assert engine.cooccurrence(seed, 5, n_walks) == len(centre)
            for a, b in zip(engine.export_cooccurrence(), (centre, context, count)):
                assert np.array_equal(a, b)
            engine.glove_train(0.05)
            stats = oracle.glove_train(centre, context, count, t0, t1, D, case["alpha"], 0.05)
            assert engine.counters()["pairs"] == stats["trained"]
        else:
            thr, alias = oracle.alias_build(graph.indptr, 0.75)
            stats = oracle.train_walklets(case["model"], walks, case["walklet"], t0, t1, seed, n, D, window,
                                          case["K"], 0.1, first_walk=5, thr=thr, alias=alias, indptr=graph.indptr,
                                          stochastic_downsample_by_degree=case["downsample"])
            engine.walk_chunk(seed, 5, n_walks, 1, 0)
            engine.train_chunk(seed, 0, 0.1)
            counters = engine.counters()
            assert (counters["pairs"], counters["targets"]) == (stats["pairs"], stats["targets"])
        g0, g1 = engine.export_tables()
    assert np.array_equal(g0, t0[:, :D])
    assert np.array_equal(g1, t1[:, :D])
