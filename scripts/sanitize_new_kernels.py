"""Small driver for `compute-sanitizer --tool memcheck`: one tiny invocation of every kernel added
for the SURVEY 8(f) rows (general / typed walks, Walklets split, GloVe, generic SGD with the
centre skip), plus the production SkipGram / CBOW launches.  Prints 'sanitize ok' at the end."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

from embiggen_b200.engine import Engine
from embiggen_b200.graph import rmat

graph = rmat(10, 6000, n=1000, seed=3)
n = graph.get_number_of_nodes()
rng = np.random.default_rng(0)
node_types = rng.integers(0, 3, n).astype(np.uint32)
edge_types = rng.integers(0, 3, graph.indices.shape[0]).astype(np.uint32)
weights = rng.random(graph.indices.shape[0]).astype(np.float32) + 0.1

for model in ("SkipGram", "CBOW"):
    for extra in (dict(), dict(walklet_scale=3, window_size=1), dict(stochastic_downsample_by_degree=True),
                  dict(normalize_by_degree=True, change_node_type_weight=3.0, change_edge_type_weight=0.3),
                  dict(embedding_size=200)):
        kw = dict(embedding_size=100, walk_length=33, window_size=4, iterations=1, epochs=1,
                  return_weight=0.5, explore_weight=2.0)
        kw.update(extra)
        with Engine(model, **kw) as engine:
            engine.load_csr(graph.indptr, graph.indices, weights)
            engine.load_types(node_types, edge_types)
            t0, t1, losses = engine.fit(7)
            assert np.isfinite(t0).all() and np.isfinite(t1).all(), (model, extra)
# round 2: folded return edge + row filters + short-row search (unweighted, undirected), the
# CSR content check, the window-ring CBOW kernel without weights, the exchange kernel, the digest
hub = rmat(11, 20000, n=2000, seed=5)
for model in ("SkipGram", "CBOW"):
    replicas = [Engine(model, embedding_size=100, walk_length=40, window_size=4, iterations=1, epochs=1,
                       return_weight=2.0, explore_weight=0.5, chunk_walks=700) for _ in range(2)]
    for rank, engine in enumerate(replicas):
        engine.load_csr(hub.indptr, hub.indices)
        engine.init_tables(3)
        engine.walk_chunk(3, rank, 700, 2, 0)
        engine.train_chunk(3, 0, 0.05)
    for rank, engine in enumerate(replicas):
        engine.open_exchange_local(replicas, rank)
    for engine in replicas:
        engine.sync()
    for engine in replicas:
        engine.exchange_average()
    for engine in replicas:
        engine.sync()
    digests = [engine.tables_digest() for engine in replicas]
    assert digests[0]["bits"] == digests[1]["bits"] and digests[0]["non_finite"] == 0
    assert replicas[0].counters()["walk_filter_rejects"] > 0
    for engine in replicas:
        engine.close()
with Engine("GloVe", embedding_size=100, walk_length=33, window_size=4, iterations=1, epochs=2,
            chunk_walks=300) as engine:
    engine.load_csr(graph.indptr, graph.indices)
    t0, t1, losses = engine.fit(7)
    assert np.isfinite(t0).all() and np.isfinite(t1).all()
with Engine("CBOW", embedding_size=128, walk_length=40, window_size=4, iterations=1, epochs=1) as engine:  # full rows
    engine.load_csr(hub.indptr, hub.indices)
    t0, t1, losses = engine.fit(7)
    assert np.isfinite(t0).all() and np.isfinite(t1).all()
os.environ["B2E_GLOVE_SLOTS"] = "20000"  # co-occurrence by centre ranges
with Engine("GloVe", embedding_size=100, walk_length=33, window_size=4, iterations=1, epochs=2) as engine:
    engine.load_csr(graph.indptr, graph.indices)
    t0, t1, losses = engine.fit(7)
    assert np.isfinite(t0).all() and np.isfinite(t1).all()
del os.environ["B2E_GLOVE_SLOTS"]
from embiggen_b200.edge_prediction import (EdgeTransformerB200, PerceptronEdgePredictionB200,  # noqa: E402
                                           edge_metrics)
features = rng.normal(size=(n, 20)).astype(np.float32)
src, dst = rng.integers(0, n, 3000), rng.integers(0, n, 3000)
transformer = EdgeTransformerB200(["Hadamard", "Concatenate", "CosineSimilarity", "L2Distance", "Min"])
transformer.fit(features)
assert np.isfinite(transformer.transform(src, dst)).all()
assert np.isfinite(edge_metrics(graph, src, dst, ["Degree", "AdamicAdar", "JaccardCoefficient",
                                                  "ResourceAllocationIndex", "PreferentialAttachment"])).all()
for kw in (dict(), dict(edge_features=["Degree", "AdamicAdar"], edge_embeddings=["L1", "CosineSimilarity"],
                        avoid_false_negatives=True)):
    model = PerceptronEdgePredictionB200(number_of_epochs=2, number_of_edges_per_mini_batch=256, **kw)
    model.fit(graph, features)
    assert np.isfinite(model.predict_proba(src, dst, features)).all()
print("sanitize ok")
