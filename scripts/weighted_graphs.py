"""Weighted graphs on the GPU at the C3 shape (R-MAT 10 M nodes / 200 M undirected edges, generator
seed 42) with seeded log-normal weights (mu = 0, sigma = 1, numpy seed 7) on the undirected edges:

- the weighted ingest (device_graph_from_edges with weights=, symmetrised; host arrays in, a
  resident weighted graph out), timed twice;
- the load of that resident graph into a Node2Vec SkipGram engine (p = 0.5, q = 2, the C3 walk
  parameters) and of the same graph from host arrays, each with and without normalize_by_degree;
  the per-phase split comes from B2E_LOAD_TIMING=1 on stderr, which includes the device edge
  alias build and the degree of its longest row;
- oracle.edge_alias on the host for the same graph: the sequential per-row Vose loop that the
  library ran on one host thread before the tables were built on the device (a proxy for it:
  the same loop, in the oracle's C), timed once; and a bitwise comparison of the device table
  with it;
- weighted second-order walk steps/s (walk_chunk on the device, timed with a device
  synchronise), and the unweighted rate of the same graph for comparison.

    B2E_LOAD_TIMING=1 python scripts/weighted_graphs.py --out result.json 2> load_timing.txt
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {"c3": (24, 200_000_000, 10_000_000), "rmat1m": (20, 16_000_000, 1_000_000)}  # scale, edges, nodes
WALK = dict(walk_length=128, return_weight=2.0, explore_weight=0.5, iterations=1, embedding_size=100)


def stamp(what):
    print(f"[weighted_graphs] {what}", file=sys.stderr, flush=True)


def walk_rate(engine, chunks=6):
    """Walk steps per second over `chunks` full chunks after one warm-up chunk."""
    cap = engine.chunk_capacity
    engine.walk_chunk(1, 0, cap, 1, 0)
    engine.sync()
    engine.reset_counters()
    begin = time.perf_counter()
    for c in range(chunks):
        engine.walk_chunk(1, (c + 1) * cap, cap, 1, c & 1)
    engine.sync()
    seconds = time.perf_counter() - begin
    steps = engine.counters()["walk_steps"]
    return {"walks": chunks * cap, "steps": int(steps), "seconds": seconds, "steps_per_s": steps / seconds}


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--shape", default="c3", choices=sorted(SHAPES))
    parser.add_argument("--out", required=True)
    parser.add_argument("--no-oracle", action="store_true", help="skip the host oracle and the comparison")
    args = parser.parse_args()
    import torch
    import oracle
    from embiggen_b200.engine import Engine
    from embiggen_b200.graph_gpu import device_graph_from_csr, device_graph_from_edges, rmat_gpu

    scale, m, n = SHAPES[args.shape]
    result = {"shape": args.shape, "nodes": n, "undirected_edges": m, "device": torch.cuda.get_device_name(0),
              "walk": WALK}
    stamp("generating the graph")
    host = rmat_gpu(scale, m, n=n, seed=42)  # the C3 graph, as host arrays
    rows = np.repeat(np.arange(n, dtype=np.uint32), np.diff(host.indptr))
    upper = host.indices > rows
    src, dst = rows[upper], host.indices[upper]
    del rows, upper
    weights = np.random.default_rng(7).lognormal(0.0, 1.0, src.shape[0]).astype(np.float32)
    result["input_edges"] = int(src.shape[0])

    stamp("weighted ingest")
    ingest = []
    for _ in range(2):
        begin = time.perf_counter()
        graph = device_graph_from_edges(src, dst, n, weights=weights)
        torch.cuda.synchronize()
        ingest.append(time.perf_counter() - begin)
        nnz = graph.get_number_of_directed_edges()
        if len(ingest) < 2:
            graph.close()
    result["weighted_ingest_s"] = ingest
    result["nnz"] = nnz
    del src, dst, weights
    csr_weights = graph.get_directed_edge_weights()

    loads = {}
    for source in ("resident", "host"):
        for normalize in (False, True):
            key = f"{source}{'_normalized' if normalize else ''}"
            stamp(f"load {key}")
            with Engine("SkipGram", normalize_by_degree=normalize, **WALK) as engine:
                begin = time.perf_counter()
                if source == "resident":
                    engine.load_graph(graph)
                else:
                    engine.load_csr(host.indptr, host.indices, csr_weights)
                loads[key] = {"load_s": time.perf_counter() - begin}
                if key == "resident":
                    table = engine.export_edge_alias()
                    loads[key]["walk"] = walk_rate(engine)
    result["loads"] = loads

    stamp("unweighted walk rate")
    unweighted = device_graph_from_csr(host.indptr, host.indices)
    with Engine("SkipGram", **WALK) as engine:
        engine.load_graph(unweighted)
        result["unweighted_walk"] = walk_rate(engine)
    unweighted.close()
    graph.close()

    degrees = np.diff(host.indptr)
    result["longest_row"] = int(degrees.max())
    if not args.no_oracle:
        stamp("oracle.edge_alias on the host")
        begin = time.perf_counter()
        expected = oracle.edge_alias(host.indptr, csr_weights)
        result["host_oracle_edge_alias_s"] = time.perf_counter() - begin
        result["device_table_equals_oracle"] = bool(np.array_equal(expected, table))
    stamp("done")
    with open(args.out, "w") as handle:
        json.dump(result, handle, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
