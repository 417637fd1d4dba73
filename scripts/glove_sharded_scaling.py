"""Seconds per GloVe epoch at the reference's GloVe defaults (node2vec_glove.py:8-30: D = 100,
walk_length = 512, window_size = 5, alpha = 0.75, p = 4, q = 0.25) with the centre ids sharded over
G ranks (Engine.fit_distributed on a GloVe handle, DESIGN.md K7), and where the time goes:
walks + histogram (repeated on every rank), counting (incl. the all-reduce of x_max, i.e. the
wait for the slowest counter), training, merge (incl. the barriers, i.e. the wait for the slowest
trainer).  One process per rank, gloo control plane, CUDA IPC data plane; rank r on GPU r.  The
graph is built on every rank's GPU.  fit_distributed runs twice per configuration: the first
run allocates the buffers, the second is reported.

    python scripts/glove_sharded_scaling.py --graph rmat1m --world 2 --epochs 2 --out result.json
"""
import argparse
import json
import os
import socket
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GRAPHS = {"rmat1m": (20, 16_000_000, 1_000_000), "c3": (24, 200_000_000, 10_000_000)}  # scale, edges, nodes
DEFAULTS = dict(embedding_size=100, walk_length=512, window_size=5, glove_alpha=0.75, return_weight=0.25,
                explore_weight=4.0, learning_rate=0.05, learning_rate_decay=0.9, iterations=1)


def worker(rank, world, port, args):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    from embiggen_b200.engine import Engine
    from embiggen_b200.graph_gpu import rmat_gpu
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    device = rank
    scale, m, n = GRAPHS[args.graph]
    begin = time.perf_counter()
    graph = rmat_gpu(scale, m, n=n, seed=3, device=device, resident=True)
    build_s = time.perf_counter() - begin
    with Engine("GloVe", epochs=args.epochs, device=device, **DEFAULTS) as engine:
        engine.load_graph(graph)
        graph.close()
        runs = []
        for _ in range(2):
            dist.barrier()
            begin = time.perf_counter()
            _, _, losses = engine.fit_distributed(42, gather="rank0")
            runs.append((time.perf_counter() - begin, dict(engine.timings), losses))
        seconds, timings, losses = runs[-1]
        digest = engine.tables_digest()
        walks_per_epoch = engine.walks_per_epoch
    mine = {"rank": rank, "device": torch.cuda.get_device_name(device), "fit_s": seconds, "warmup_fit_s": runs[0][0],
            "graph_build_s": build_s, "per_epoch_s": {k: v / args.epochs for k, v in timings.items()
                                                      if not k.endswith(("exchange_s", "tables_s"))},
            "other_s": {k: v for k, v in timings.items() if k.endswith(("exchange_s", "tables_s"))},
            "bits": [str(b) for b in digest["bits"]], "non_finite": digest["non_finite"]}
    everyone = [None] * world
    dist.all_gather_object(everyone, mine)
    if rank == 0:
        result = {"graph": args.graph, "nodes": n, "edges": m, "world": world, "epochs": args.epochs,
                  "walks_per_epoch": walks_per_epoch,
                  "key_slots_per_epoch": 2 * walks_per_epoch * DEFAULTS["walk_length"] * DEFAULTS["window_size"],
                  "seconds_per_epoch": seconds / args.epochs, "losses": losses,
                  "replicas_identical": all(r["bits"] == everyone[0]["bits"] for r in everyone),
                  "ranks": everyone, "kwargs": DEFAULTS}
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
        print(json.dumps({k: result[k] for k in ("graph", "world", "seconds_per_epoch", "replicas_identical")}))
    dist.destroy_process_group()


def main():
    parser = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    parser.add_argument("--graph", choices=sorted(GRAPHS), default="rmat1m")
    parser.add_argument("--world", type=int, default=1)
    parser.add_argument("--epochs", type=int, default=2)
    parser.add_argument("--out", required=True)
    args = parser.parse_args()
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < args.world:
        raise SystemExit(f"--world {args.world} needs {args.world} GPUs, {torch.cuda.device_count()} are visible")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(worker, args=(args.world, port, args), nprocs=args.world, join=True)


if __name__ == "__main__":
    main()
