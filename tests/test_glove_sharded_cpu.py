"""GloVe with its centre ids sharded over several GPUs, without a GPU: the restatement of the
sharded schedule (tests/glove_sharded_oracle.py) against the one-GPU oracle, the owner rule, the
counts and the merge; then the host logic of the data-parallel driver
(Engine._fit_glove_distributed) under gloo, with the oracle standing in for the native steps."""
import os
import socket
from types import SimpleNamespace

import numpy as np
import pytest

import glove_sharded_oracle as sharded
import oracle

KW = dict(embedding_size=12, epochs=2, walk_length=24, window_size=3, alpha=0.75, learning_rate=0.05,
          learning_rate_decay=0.9, return_weight=0.5, explore_weight=2.0)


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("capacity", [None, 2_000])
def test_one_rank_is_the_one_gpu_schedule(small_ppi, capacity):
    t0, t1, losses = oracle.glove_fit(small_ppi.indptr, small_ppi.indices, 9, **KW)
    s0, s1, sharded_losses = sharded.glove_fit_sharded(small_ppi.indptr, small_ppi.indices, 9, world=1,
                                                       capacity_slots=capacity, **KW)
    assert np.array_equal(t0, s0) and np.array_equal(t1, s1)
    assert np.allclose(losses, sharded_losses, rtol=1e-12)


def epoch_walks(graph, seed=9, first=0, L=24):
    n_walks = int((np.diff(graph.indptr) > 0).sum())
    walks, _ = oracle.walks(graph.indptr, graph.indices, seed, first, n_walks, L, 0.5, 2.0)
    return walks


@pytest.mark.parametrize("world", [2, 3])
def test_owners_partition_the_centres_and_their_counts(small_ppi, rmat_graph, world):
    W = 3
    for graph in (small_ppi, rmat_graph):
        n = graph.get_number_of_nodes()
        walks = epoch_walks(graph)
        histogram = sharded.token_histogram(walks, n)
        bounds = sharded.owner_bounds(histogram, W, world)
        assert len(bounds) == world + 1 and bounds[0] == 0 and bounds[-1] == n
        assert all(a <= b for a, b in zip(bounds[:-1], bounds[1:]))  # intervals partition [0, n)
        slots = histogram.astype(np.int64) * 2 * W
        total, largest = int(slots.sum()), int(slots.max())
        for r in range(world):
            share = int(slots[bounds[r]:bounds[r + 1]].sum())
            assert abs(share - total / world) <= largest, (r, share, total / world)
        centre, context, count = oracle.cooccurrence(walks, W)
        pieces = []
        for r in range(world):
            mine = (bounds[r] <= centre) & (centre < bounds[r + 1])
            # the owner counts its centres from the walks alone: the co-occurrence of its centres
            pieces.append(tuple(a[mine] for a in (centre, context, count)))
            for lo, hi in zip(*(lambda c: (c[:-1], c[1:]))(
                    sharded.sub_ranges(histogram, W, bounds[r], bounds[r + 1], 500))):
                assert int(slots[lo:hi].sum()) <= 500 or hi - lo == 1
        for got, want in zip((np.concatenate(p) for p in zip(*pieces)), (centre, context, count)):
            assert np.array_equal(got, want)


@pytest.mark.parametrize("world", [2, 3])
def test_merge_takes_owner_rows_and_sums_the_changes(world):
    rng = np.random.default_rng(world)
    n, stride = 50, 8
    snapshot = rng.standard_normal((n, stride)).astype(np.float32)
    t0s = [rng.standard_normal((n, stride)).astype(np.float32) for _ in range(world)]
    t1s = [(snapshot + rng.standard_normal((n, stride)).astype(np.float32) * np.float32(1e-3)) for _ in range(world)]
    bounds = [0] + sorted(rng.integers(0, n, world - 1).tolist()) + [n]
    t0, t1 = sharded.merge(t0s, t1s, snapshot, bounds)
    for r in range(world):
        assert np.array_equal(t0[bounds[r]:bounds[r + 1]], t0s[r][bounds[r]:bounds[r + 1]])
    change = (t1s[0] - snapshot).astype(np.float32)
    for t in t1s[1:]:
        change = (change + (t - snapshot).astype(np.float32)).astype(np.float32)
    assert np.array_equal(t1, (snapshot + change).astype(np.float32)) and t1.dtype == np.float32
    # every replica unchanged since the snapshot: T1 stays the snapshot
    assert np.array_equal(sharded.merge(t0s, [snapshot] * world, snapshot, bounds)[1], snapshot)


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_epoch_trains_every_triple_once(small_ppi, world):
    t0, t1, losses = sharded.glove_fit_sharded(small_ppi.indptr, small_ppi.indices, 9, world=world,
                                               capacity_slots=3_000, **KW)
    _, _, single = oracle.glove_fit(small_ppi.indptr, small_ppi.indices, 9, **KW)
    assert np.isfinite(t0).all() and np.isfinite(t1).all()
    # the same triples are trained; only the staleness of T1 within an epoch differs
    assert abs(losses[0] - single[0]) <= 0.05 * single[0] and losses[-1] < losses[0]


class OracleGloveEngine:
    """Stand-in for the native steps of a GloVe engine (test code: the product has no CPU path).
    It subclasses the real Engine at run time so that Engine._fit_glove_distributed, Engine.merge
    and Engine._gather_tables run unchanged; the merge crosses the ranks with gloo all_gather."""

    @staticmethod
    def make():
        from embiggen_b200.engine import Engine

        class Stand(Engine):
            def __init__(self, model, **kwargs):
                self.model, self.config = model.lower(), SimpleNamespace(**kwargs)
                self._handle = None

            def close(self):
                pass

            def load_csr(self, indptr, indices, weights=None):
                self.indptr, self.indices, self.n = indptr, indices, indptr.shape[0] - 1

            @property
            def walks_per_epoch(self):
                return self.config.iterations * oracle.sources(self.indptr).shape[0]

            def init_tables(self, seed):
                self.t0, self.t1 = oracle.init_tables(self.n, self.config.embedding_size, seed)

            def open_exchange(self, process_group=None):
                pass

            def close_exchange(self):
                pass

            def sync(self):
                pass

            def reset_counters(self):
                self.stats = {"loss_sum": 0.0, "trained": 0}

            def glove_walk_epoch(self, seed, first_walk, n_walks):
                c = self.config
                self.walks, _ = oracle.walks(self.indptr, self.indices, seed, first_walk, n_walks, c.walk_length,
                                             c.return_weight, c.explore_weight)
                self.histogram = sharded.token_histogram(self.walks, self.n)

            def glove_shard_count(self, world, rank):
                self.bounds = sharded.owner_bounds(self.histogram, self.config.window_size, world)
                self.rank = rank
                self.triples = oracle.cooccurrence(self.walks, self.config.window_size)
                mine = (self.bounds[rank] <= self.triples[0]) & (self.triples[0] < self.bounds[rank + 1])
                return (int(self.triples[2][mine].max()) if mine.any() else 0), np.array(self.bounds)

            def glove_shard_train(self, learning_rate, max_count):
                c = self.config
                self.snapshot = self.t1.copy()
                stats = sharded.train_shard(*self.triples, self.bounds, self.rank, self.histogram, self.t0, self.t1,
                                            c.embedding_size, c.window_size, c.glove_alpha, learning_rate,
                                            c.clipping_value, max_count)
                for key in stats:
                    self.stats[key] += stats[key]

            def glove_merge(self):
                import torch
                import torch.distributed as dist
                world = dist.get_world_size()
                replicas = []
                for table in (self.t0, self.t1):
                    gathered = [torch.zeros_like(torch.from_numpy(table)) for _ in range(world)]
                    dist.all_gather(gathered, torch.from_numpy(table))
                    replicas.append([g.numpy() for g in gathered])
                self.t0, self.t1 = sharded.merge(replicas[0], replicas[1], self.snapshot, self.bounds)

            def counters(self):
                return {"loss_sum": self.stats["loss_sum"], "pairs": self.stats["trained"]}

            def export_tables(self, table0=None, table1=None):
                D = self.config.embedding_size
                table0[:] = self.t0[:, :D]
                table1[:] = self.t1[:, :D]
                return table0, table1

        return Stand


def _worker(rank, world, port, out_dir):
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    sys.path[:0] = [os.path.dirname(here), here]
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from embiggen_b200 import embedders
    from embiggen_b200.embedders import Node2VecGloVeB200
    from embiggen_b200.graph import erdos_renyi
    embedders.Engine = OracleGloveEngine.make()
    graph = erdos_renyi(300, 1500, seed=3)
    path = os.path.join(out_dir, "central.npy")
    model = Node2VecGloVeB200(embedding_size=8, epochs=2, walk_length=12, window_size=3, random_state=5,
                              verbose=False, central_nodes_embedding_path=path)
    central, contextual = model.fit_transform(graph, return_dataframe=False).get_all_node_embedding()
    np.save(os.path.join(out_dir, f"tables_{rank}.npy"), np.stack([central, contextual]))
    np.save(os.path.join(out_dir, f"losses_{rank}.npy"), np.array(model.get_losses()))
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_glove_embedder_under_gloo_runs_the_sharded_schedule(tmp_path, world):
    """Node2VecGloVeB200.fit_transform under torch.distributed no longer refuses: every rank returns
    the same tables -- those of the sharded schedule -- and rank 0 alone writes the output file."""
    import torch.multiprocessing as mp
    from embiggen_b200.graph import erdos_renyi
    mp.spawn(_worker, args=(world, free_port(), str(tmp_path)), nprocs=world, join=True)
    tables = [np.load(tmp_path / f"tables_{r}.npy") for r in range(world)]
    for r in range(1, world):
        assert np.array_equal(tables[0], tables[r])
    graph = erdos_renyi(300, 1500, seed=3)
    t0, t1, losses = sharded.glove_fit_sharded(graph.indptr, graph.indices, 5, embedding_size=8, epochs=2,
                                               walk_length=12, window_size=3, alpha=0.75, learning_rate=0.05,
                                               learning_rate_decay=0.9, return_weight=0.25, explore_weight=4.0,
                                               world=world)
    assert np.array_equal(tables[0][0], t0[:, :8]) and np.array_equal(tables[0][1], t1[:, :8])
    assert np.allclose(np.load(tmp_path / "losses_0.npy"), losses, rtol=1e-9)
    assert np.array_equal(np.load(tmp_path / "central.npy"), tables[0][0])
