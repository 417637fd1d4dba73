"""The production launches of the SGD and GloVe kernels against sequential references, bit for bit.

The production launch trains many walks (GloVe: tiles of 512 triples) at once, several warps to a
CTA on a persistent grid, and lets their updates race (Hogwild).  Its result depends on how the
walks interleave, so the suite used to compare it with the oracle by loss tolerances only, and
a wrong shared-memory slab in warps 1-3 or a lost write-back moves the loss by a few percent.

Here the workloads leave Hogwild nothing to race over: no two concurrently trained walks (tiles)
change a row that the other one reads.  Then the update order cannot matter, and the production
launch must give the tables of the sequential reference exactly, for every grid size.

- SkipGram / CBOW with negatives: disjoint cliques, one walk per clique in every launch, and
  tables in which a pair across cliques scores far beyond the clipping value.  Both the oracle and
  the kernels skip a clipped target entirely (no gradient, no store), so a negative drawn from
  another walk's clique is only read, and far from the clipping boundary.  Whether the tables
  really stay separated, and whether the oracle's tables really do not depend on the walk order,
  is asserted on the oracle before the GPU result is compared (``sgd_reference``).
- No negatives: walks in disjoint components cannot interact at all; a large graph of 4-cliques
  fills the whole persistent grid.
- GloVe: disjoint stars, window 1.  A leaf-centred triple always clips, so a hub-centred triple
  trains the hub's centre row and its own leaves' context rows only.  Each hub owns 16 triples,
  so no hub's run of triples straddles a tile.  The production kernel's arithmetic is not the
  specification's (see ``oracle/oracle.h``); it is compared with ``oracle.glove_train(...,
  tile_semantics=True)``.

The parametrisations name the kernel instantiation each case reaches, by the selection rules of
``launch_train_pipe`` (sgns_pipe.cu), ``launch_model`` (sgns_kernels.cu) and ``glove_train``
(glove.cu).  The checks of the constructions that need no GPU also run without one.
"""
import math

import numpy as np
import pytest

import oracle
from embiggen_b200.engine import Engine
from embiggen_b200.graph import csr_from_edges

SEED = 42
CLIP = 6.0
MARGIN = 8.0  # a cross-component score stays at least this far beyond the clipping value
PIPE_WARPS, GENERIC_WARPS = 4, 8  # warps per CTA of the pipelined kernels / of train_kernel


# ---- workload A: disjoint cliques, separated tables ----
def cliques(C, m, n=None):
    """C disjoint m-cliques on nodes a*m .. a*m+m-1; nodes from C*m to n are isolated."""
    i, j = np.triu_indices(m, 1)
    base = (np.arange(C, dtype=np.int64) * m)[:, None]
    return csr_from_edges((base + i).ravel(), (base + j).ravel(), C * m if n is None else n)


def separated_tables(C, m, D, scale, n=None, noise=0.3, seed=1):
    """T0 = s e_a + s f + noise, T1 = s e_a - s f + noise for a node of component a (e_a: unit
    vector a, f: the last coordinate): a pair inside a component scores about 0, a pair across
    components about -s^2.  Rows of isolated nodes (n > C*m) are zero."""
    assert C <= D - 1
    live = C * m
    rng = np.random.default_rng(seed)
    stride = oracle.row_stride(D)
    t0 = np.zeros((live if n is None else n, stride), dtype=np.float32)
    t1 = np.zeros_like(t0)
    component = np.arange(live) // m
    for t, sign in ((t0, 1.0), (t1, -1.0)):
        rows = noise * rng.standard_normal((live, D))
        rows[np.arange(live), component] += scale
        rows[:, D - 1] += sign * scale
        t[:live, :D] = rows.astype(np.float32)
    return t0, t1


def sgd_case(kernel, model="SkipGram", D=128, K=10, w=4, L=32, lr=0.005, C=None, m=8, rounds=4,
             shared=False, alias=True, normalize=False, scale_dot=False, downsample=False,
             walklet=0, concurrent=0, warps=PIPE_WARPS):
    """C components of m nodes; C <= D - 1 (a unit vector per component besides f)."""
    C = min(100, D - 1) if C is None else C
    concurrent = C if concurrent == "C" else concurrent
    return pytest.param(dict(model=model, D=D, K=K, w=w, L=L, lr=lr, C=C, m=m, rounds=rounds, shared=shared,
                             alias=alias, normalize=normalize, scale_dot=scale_dot, downsample=downsample,
                             walklet=walklet, concurrent=concurrent, warps=warps, kernel=kernel),
                        id=f"{kernel}-{model}-D{D}-K{K}-w{w}-L{L}" + ("-shared" if shared else "") +
                        ("" if alias else "-uniform") + ("-lr_by_degree" if normalize else "") +
                        ("-scaled_dot" if scale_dot else "") + ("-downsample" if downsample else "") +
                        (f"-walklets{walklet}" if walklet else "") + (f"-concurrent{concurrent}" if concurrent else ""))


SGD_CASES = [
    # pipelined kernels: embedding_size <= 128, walk_length <= 1024, CBOW windows of <= 31 positions
    sgd_case("skipgram_pipe_kernel<11>", K=10),
    sgd_case("skipgram_pipe_kernel<6>", K=5),
    sgd_case("skipgram_pipe_kernel<0>", K=3),
    sgd_case("cbow_pipe_kernel<11>", model="CBOW", D=100, K=10),
    sgd_case("cbow_pipe_kernel<6>", model="CBOW", D=100, K=5),
    sgd_case("cbow_pipe_kernel<0>", model="CBOW", D=100, K=3),
    sgd_case("cbow_pipe_kernel<11,true>", model="CBOW", D=128, K=10),  # 32 chunks fill the warp
    sgd_case("skipgram_shared_kernel<10,4>", K=10, shared=True),
    sgd_case("skipgram_shared_kernel<5>", K=5, shared=True),
    sgd_case("skipgram_shared_kernel<0>", K=7, shared=True),
    # generic train_kernel (8 warps per CTA): rows of more than 32 chunks, long walks, wide CBOW windows
    sgd_case("train_kernel<SkipGram,2,6,2>", D=200, C=150, warps=GENERIC_WARPS),
    sgd_case("train_kernel<SkipGram,4,3,2>", D=400, C=150, warps=GENERIC_WARPS),
    sgd_case("train_kernel<CBOW,1,11,2>", model="CBOW", D=100, w=16, L=64, lr=0.0025, warps=GENERIC_WARPS),
    sgd_case("train_kernel<SkipGram,1,11,2>", L=1040, lr=0.001, warps=GENERIC_WARPS),
]
for _model, _kernel, _D in (("SkipGram", "skipgram_pipe_kernel<11>", 128), ("CBOW", "cbow_pipe_kernel<11>", 100)):
    SGD_CASES += [
        sgd_case(_kernel, model=_model, D=_D, alias=False),
        sgd_case(_kernel, model=_model, D=_D, normalize=True, lr=0.02),
        sgd_case(_kernel, model=_model, D=_D, scale_dot=True),
        sgd_case(_kernel, model=_model, D=_D, downsample=True),
        sgd_case(_kernel, model=_model, D=_D, walklet=2),
        sgd_case(_kernel, model=_model, D=_D, walklet=3),
    ]
# walks in flight: 1 = one CTA whose warps fetch every walk; C = one walk per warp over C / 4 CTAs
for _concurrent in (1, 7, "C"):
    SGD_CASES += [
        sgd_case("skipgram_pipe_kernel<11>", K=10, concurrent=_concurrent),
        sgd_case("cbow_pipe_kernel<11>", model="CBOW", D=100, K=10, concurrent=_concurrent),
        sgd_case("skipgram_shared_kernel<10,4>", K=10, shared=True, concurrent=_concurrent),
        sgd_case("train_kernel<SkipGram,2,6,2>", D=200, C=150, concurrent=_concurrent, warps=GENERIC_WARPS),
    ]


def scale_of(case):
    """X = Y = 6: a cross-component pair starts at -36; scaled by D^(1/4) with dot / sqrt(D)."""
    return 6.0 * (case["D"] ** 0.25 if case["scale_dot"] else 1.0)


def oracle_train(case, walks, t0, t1, n, first_walk, walk_id_stride, thr, alias, indptr):
    kw = dict(clipping_value=CLIP, first_walk=first_walk, walk_id_stride=walk_id_stride, thr=thr, alias=alias,
              indptr=indptr, normalize_learning_rate_by_degree=case["normalize"], scale_by_sqrt_dim=case["scale_dot"],
              stochastic_downsample_by_degree=case["downsample"], shared_negatives=case["shared"])
    args = (t0, t1, SEED, n, case["D"], case["w"], case["K"], case["lr"])
    if case["walklet"] >= 2:
        return oracle.train_walklets(case["model"], walks, case["walklet"], *args, **kw)
    return oracle.train(case["model"], walks, *args, **kw)


def cross_component_scores(t0, t1, case, live):
    """Largest score T0[u] . T1[v] (float64, scaled like the kernels' dot) over u, v in different
    components.  Every cross score at most -(clip + margin) means the mean of several T0 rows of one
    component (CBOW) clips against another component's T1 row as well."""
    D, m = case["D"], case["m"]
    scores = t0[:live, :D].astype(np.float64) @ t1[:live, :D].astype(np.float64).T
    if case["scale_dot"]:
        scores /= math.sqrt(D)
    component = np.arange(live) // m
    return scores[component[:, None] != component[None, :]].max()


def sgd_reference(case, graph, fresh_tables, live):
    """The oracle's tables after ``rounds`` launches of C walks (walk r + k*m starts in component
    k), with the preconditions that make the production launch race-free asserted on the way:
    cross-component pairs stay clipped by a margin, training the walks one by one in a shuffled
    order gives the same tables bit for bit, and nearly every row moves."""
    C, m, D = case["C"], case["m"], case["D"]
    n = graph.get_number_of_nodes()
    thr = alias = None
    if case["alias"]:
        thr, alias = oracle.alias_build(graph.indptr, 0.75)
    t0, t1 = fresh_tables()
    s0, s1 = fresh_tables()
    start0, start1 = t0[:live].copy(), t1[:live].copy()
    bound = -(CLIP + MARGIN)
    assert cross_component_scores(t0, t1, case, live) <= bound
    stats = {"loss_sum": 0.0, "pairs": 0, "targets": 0}
    rounds = []
    order = np.random.default_rng(7)
    for r in range(case["rounds"]):
        walks, _ = oracle.walks(graph.indptr, graph.indices, SEED, r, C, case["L"], 1.0, 1.0, walk_id_stride=m)
        assert np.array_equal(walks[:, 0] // m, np.arange(C))  # one walk per component
        rounds.append(walks)
        got = oracle_train(case, walks, t0, t1, n, r, m, thr, alias, graph.indptr)
        for key in stats:
            stats[key] += got[key]
        for k in order.permutation(C):  # the same walks one by one, in another order
            oracle_train(case, walks[k:k + 1], s0, s1, n, r + k * m, 1, thr, alias, graph.indptr)
        worst = cross_component_scores(t0, t1, case, live)
        assert worst <= bound, f"round {r}: a cross-component score reached {worst}; lower the learning rate"
    assert np.array_equal(t0[:live], s0[:live]) and np.array_equal(t1[:live], s1[:live]), \
        "the oracle's tables depend on the walk order"
    moved = (t0[:live] != start0).any(axis=1) | (t1[:live] != start1).any(axis=1)
    assert stats["pairs"] > 0 and moved.mean() >= 0.95, (stats, moved.mean())
    return t0, t1, stats, rounds


def first_difference(got, want, component, what):
    """None when equal; else how many rows differ, and the first one with its component and value."""
    if np.array_equal(got, want):
        return None
    rows = np.flatnonzero((got != want).any(axis=1))
    row = rows[0]
    column = np.flatnonzero(got[row] != want[row])[0]
    return (f"{what}: {rows.size} rows differ, first row {row} (component {component[row]}) column {column}: "
            f"{got[row, column]!r} instead of {want[row, column]!r}")


def engine_for(case, **extra):
    return Engine(case["model"], embedding_size=case["D"], walk_length=case["L"], window_size=case["w"],
                  iterations=1, number_of_negative_samples=case["K"], clipping_value=CLIP,
                  return_weight=1.0, explore_weight=1.0, use_scale_free_distribution=case["alias"],
                  normalize_learning_rate_by_degree=case["normalize"], scale_by_sqrt_dim=case["scale_dot"],
                  stochastic_downsample_by_degree=case["downsample"], walklet_scale=case["walklet"],
                  shared_negatives=case["shared"], chunk_walks=case["C"],
                  max_concurrent_walks=case["concurrent"], **extra)


def train_rounds(engine, case, rounds, host_walks):
    """Every round is one launch (one per walklet scale) over the C walks of round r."""
    for r, walks in enumerate(rounds):
        before = engine.launch_count
        if host_walks:
            engine.train_host_walks(SEED, walks, case["lr"], first_walk=r, walk_id_stride=case["m"])
        else:
            engine.walk_chunk(SEED, r, case["C"], case["m"], 0)
            before = engine.launch_count
            engine.train_chunk(SEED, 0, case["lr"])
        assert engine.launch_count - before == max(1, case["walklet"])


def compare(label, got0, got1, counters, want0, want1, stats, m):
    component = np.arange(got0.shape[0]) // m
    problems = [p for p in (first_difference(got0, want0, component, "T0"),
                            first_difference(got1, want1, component, "T1")) if p]
    assert not problems, f"{label}: " + "; ".join(problems)
    assert (counters["pairs"], counters["targets"]) == (stats["pairs"], stats["targets"]), label
    assert np.isclose(counters["loss_sum"], stats["loss_sum"], rtol=1e-4), (label, counters, stats)


@pytest.mark.parametrize("case", SGD_CASES)
def test_race_free_sgd_workloads_hold_on_the_oracle(case):
    """The construction's preconditions on the CPU: a change to the oracle or to the workload that
    lets walks interact shows up here, without a GPU."""
    graph = cliques(case["C"], case["m"])
    sgd_reference(case, graph, lambda: separated_tables(case["C"], case["m"], case["D"], scale_of(case)),
                  case["C"] * case["m"])


@pytest.mark.gpu
@pytest.mark.parametrize("case", SGD_CASES)
def test_production_sgd_launch_equals_the_sequential_oracle(case):
    C, m, D = case["C"], case["m"], case["D"]
    graph = cliques(C, m)
    fresh = lambda: separated_tables(C, m, D, scale_of(case))
    want0, want1, stats, rounds = sgd_reference(case, graph, fresh, C * m)
    start0, start1 = fresh()
    with engine_for(case) as engine:
        engine.load_csr(graph.indptr, graph.indices)
        for host_walks in (False, True):
            engine.import_tables(start0[:, :D], start1[:, :D])
            engine.reset_counters()
            train_rounds(engine, case, rounds, host_walks)
            got0, got1 = engine.export_tables()
            compare(f"{case['kernel']}, {'host' if host_walks else 'GPU'} walks", got0, got1, engine.counters(),
                    want0[:, :D], want1[:, :D], stats, m)


# ---- workload B: no negatives, the whole persistent grid ----
@pytest.mark.gpu
@pytest.mark.parametrize("model,D,kernel,warps", [
    ("SkipGram", 100, "skipgram_pipe_kernel<0>", PIPE_WARPS), ("CBOW", 100, "cbow_pipe_kernel<0>", PIPE_WARPS),
    ("SkipGram", 200, "train_kernel<SkipGram,2,6,2>", GENERIC_WARPS),
    ("CBOW", 200, "train_kernel<CBOW,2,6,2>", GENERIC_WARPS)])
def test_production_launch_without_negatives_fills_the_grid(model, D, kernel, warps):
    """16 384 components of 4 nodes, all walks of a round at once: more CTAs are wanted than the
    GPU holds (at most 2048 threads per SM), so the grid is the occupancy cap sm_count * per_sm."""
    import torch
    C, m = 1 << 14, 4
    case = dict(model=model, D=D, K=0, w=4, L=32, lr=0.05, C=C, m=m, rounds=2, shared=False, alias=True,
                normalize=False, scale_dot=False, downsample=False, walklet=0, concurrent=1 << 30, kernel=kernel)
    sm_count = torch.cuda.get_device_properties(0).multi_processor_count
    assert -(-C // warps) > sm_count * (2048 // (32 * warps))
    graph = cliques(C, m)
    n = C * m
    start0, start1 = oracle.init_tables(n, D, SEED)
    start0 *= np.float32(20.0)  # out of the linear regime of the sigmoid
    start1 *= np.float32(20.0)
    t0, t1 = start0.copy(), start1.copy()
    thr, alias = oracle.alias_build(graph.indptr, 0.75)
    stats = {"loss_sum": 0.0, "pairs": 0, "targets": 0}
    rounds = []
    for r in range(case["rounds"]):
        walks, _ = oracle.walks(graph.indptr, graph.indices, SEED, r, C, case["L"], 1.0, 1.0, walk_id_stride=m)
        assert np.array_equal(walks[:, 0] // m, np.arange(C))
        rounds.append(walks)
        got = oracle_train(case, walks, t0, t1, n, r, m, thr, alias, graph.indptr)
        for key in stats:
            stats[key] += got[key]
    assert (t0 != start0).any(axis=1).mean() >= 0.95
    with engine_for(case) as engine:
        engine.load_csr(graph.indptr, graph.indices)
        for host_walks in (False, True):
            engine.import_tables(start0[:, :D], start1[:, :D])
            engine.reset_counters()
            train_rounds(engine, case, rounds, host_walks)
            got0, got1 = engine.export_tables()
            compare(f"{kernel}, {'host' if host_walks else 'GPU'} walks", got0, got1, engine.counters(),
                    t0[:, :D], t1[:, :D], stats, m)


# ---- workload C: tables of 32 GiB, skipgram_pipe_kernel<11, 3> ----
@pytest.mark.gpu
def test_skipgram_at_32_gib_of_tables():
    """Workload A on 2^25 nodes of 128 floats (2 x 16 GiB, where launch_train_pipe switches SkipGram
    K = 10 to three CTAs per SM).  All but the 800 nodes of the cliques are isolated, and an
    isolated node is never drawn as a negative (weight 0^0.75 = 0), so only the live rows train:
    they are written and read through zero-copy views of the device tables, and the oracle's
    tables are zero pages but for the rows it touches."""
    import torch
    if torch.cuda.mem_get_info()[0] < 40 << 30:
        pytest.skip("needs 40 GiB of free device memory")
    n, D = 1 << 25, 128
    case = dict(model="SkipGram", D=D, K=10, w=4, L=32, lr=0.005, C=100, m=8, rounds=4, shared=False, alias=True,
                normalize=False, scale_dot=False, downsample=False, walklet=0, concurrent=0,
                kernel="skipgram_pipe_kernel<11,3>")
    C, m = case["C"], case["m"]
    live = C * m
    assert 2 * n * oracle.row_stride(D) * 4 == 32 << 30
    graph = cliques(C, m, n)
    fresh = lambda: separated_tables(C, m, D, scale_of(case), n=n)
    want0, want1, stats, rounds = sgd_reference(case, graph, fresh, live)
    start0, start1 = separated_tables(C, m, D, scale_of(case))
    with engine_for(case) as engine:
        engine.load_csr(graph.indptr, graph.indices)
        engine.init_tables(SEED)
        d0, d1 = engine.device_tables()
        d0[:live, :D] = torch.from_numpy(start0[:, :D]).to(d0.device)
        d1[:live, :D] = torch.from_numpy(start1[:, :D]).to(d1.device)
        torch.cuda.synchronize()
        engine.reset_counters()
        train_rounds(engine, case, rounds, host_walks=False)
        engine.sync()
        got0, got1 = d0[:live, :D].cpu().numpy(), d1[:live, :D].cpu().numpy()
        compare(case["kernel"], got0, got1, engine.counters(), want0[:live, :D], want1[:live, :D], stats, m)


# ---- workload D: GloVe on disjoint stars, glove_tile_kernel ----
HUBS, LEAVES, GLOVE_L, GLOVE_LR = 2048, 16, 32, 0.05


def stars():
    """HUBS hubs (ids 0 .. HUBS-1), each with LEAVES leaves whose ids come after every hub."""
    hubs = np.repeat(np.arange(HUBS, dtype=np.int64), LEAVES)
    return csr_from_edges(hubs, HUBS + np.arange(HUBS * LEAVES), HUBS * (LEAVES + 1))


def star_triples(graph):
    """One walk per node, window 1: every triple is a hub-leaf pair, sorted by centre, and every
    hub centres exactly LEAVES triples, so the 32 hub runs of a 512-triple tile never straddle one."""
    n = graph.get_number_of_nodes()
    walks, _ = oracle.walks(graph.indptr, graph.indices, SEED, 0, n, GLOVE_L, 1.0, 1.0)
    centre, context, count = oracle.cooccurrence(walks, 1)
    per_centre = np.bincount(centre, minlength=n)
    assert (per_centre[:HUBS] == LEAVES).all(), "a hub misses a leaf: raise the walk length"
    assert (per_centre[HUBS:] == 1).all()
    assert ((centre < HUBS) != (context < HUBS)).all()
    return n, centre, context, count


def star_tables(n, D, seed=3, z=4.0):
    """Hub T1 = -z f + noise, leaf T0 = +z f + noise, hub T0 and leaf T1 small and random; noise
    orthogonal to f (the last coordinate).  A leaf-centred triple scores about -z^2 and clips."""
    rng = np.random.default_rng(seed)
    t0 = (0.1 * rng.standard_normal((n, oracle.row_stride(D)))).astype(np.float32)
    t1 = (0.1 * rng.standard_normal((n, oracle.row_stride(D)))).astype(np.float32)
    t0[:, D:] = t1[:, D:] = 0.0
    t0[:, D - 1] = t1[:, D - 1] = 0.0
    t1[:HUBS, D - 1] = -z
    t0[HUBS:, D - 1] = z
    return t0, t1


def glove_reference(triples, t0, t1, D, alpha, passes, tile_semantics=True):
    """Passes of the oracle over the star triples (in place); asserts that exactly the hub-centred
    triples trained and that the rows only leaf-centred triples touch never changed."""
    n, centre, context, count = triples
    fixed0, fixed1 = t0[HUBS:].copy(), t1[:HUBS].copy()
    trained = 0
    for _ in range(passes):
        trained += oracle.glove_train(centre, context, count, t0, t1, D, alpha, GLOVE_LR, CLIP,
                                      tile_semantics=tile_semantics)["trained"]
    assert trained == passes * HUBS * LEAVES
    assert np.array_equal(t0[HUBS:], fixed0) and np.array_equal(t1[:HUBS], fixed1)
    return trained


def test_glove_star_workload_and_tile_semantics():
    """Without a GPU: the star construction holds, and the production kernel's arithmetic stays
    within two units in the last place of max(|before|, |after|) per element of the specification
    (a rounding more in each context update; h0 + (h - h0) instead of h, exact unless h and h0 are
    more than a factor of 2 apart, by Sterbenz' lemma) without being equal to it."""
    graph = stars()
    triples = star_triples(graph)
    D = 100
    start0, start1 = star_tables(triples[0], D)
    spec0, spec1 = start0.copy(), start1.copy()
    tile0, tile1 = start0.copy(), start1.copy()
    glove_reference(triples, spec0, spec1, D, 0.75, 1, tile_semantics=False)
    glove_reference(triples, tile0, tile1, D, 0.75, 1)
    differ = 0
    for start, spec, tile in ((start0, spec0, tile0), (start1, spec1, tile1)):
        ulp = np.spacing(np.maximum(np.abs(start), np.abs(spec)))
        assert (np.abs(tile.astype(np.float64) - spec) <= 2 * ulp).all()
        differ += int((tile != spec).sum())
    assert differ > 0


@pytest.mark.gpu
@pytest.mark.parametrize("concurrent", [0, 1])
@pytest.mark.parametrize("alpha", [0.75, 0.5])
@pytest.mark.parametrize("D,kernel", [(100, "glove_tile_kernel<1,4>"), (200, "glove_tile_kernel<2,4>"),
                                      (400, "glove_tile_kernel<4,2>")])
def test_production_glove_launch_equals_the_tile_oracle(D, kernel, alpha, concurrent):
    """65 536 triples in 128 tiles over a persistent grid (concurrent = 1: one CTA of 8 warps),
    two passes, against the tile-semantics oracle bit for bit."""
    graph = stars()
    triples = star_triples(graph)
    n = triples[0]
    start0, start1 = star_tables(n, D)
    want0, want1 = start0.copy(), start1.copy()
    trained = glove_reference(triples, want0, want1, D, alpha, 2)
    with Engine("GloVe", embedding_size=D, walk_length=GLOVE_L, window_size=1, return_weight=1.0,
                explore_weight=1.0, iterations=1, clipping_value=CLIP, glove_alpha=alpha,
                max_concurrent_walks=concurrent) as engine:
        engine.load_csr(graph.indptr, graph.indices)
        engine.import_tables(start0[:, :D], start1[:, :D])
        assert engine.cooccurrence(SEED, 0, n) == triples[1].shape[0]
        assert all(np.array_equal(a, b) for a, b in zip(engine.export_cooccurrence(), triples[1:]))
        engine.reset_counters()
        for _ in range(2):
            before = engine.launch_count
            engine.glove_train(GLOVE_LR)
            assert engine.launch_count - before == 1
        got0, got1 = engine.export_tables()
        counters = engine.counters()
    star = np.concatenate([np.arange(HUBS), np.repeat(np.arange(HUBS), LEAVES)])  # a leaf's hub
    problems = [p for p in (first_difference(got0, want0[:, :D], star, "T0"),
                            first_difference(got1, want1[:, :D], star, "T1")) if p]
    assert not problems, f"{kernel}: " + "; ".join(problems)
    assert counters["pairs"] == trained
