"""Normative statement of GloVe with the centre ids sharded over several GPUs (DESIGN.md K7),
built from the oracle's own pieces: ``oracle.walks``, ``oracle.cooccurrence`` and
``oracle.glove_train(max_count=...)``.  Test infrastructure, like ``oracle/``.

Per epoch, with G ranks:
1. every rank walks the whole epoch (the walks of ``oracle.glove_fit``) and takes its token histogram;
2. owners: rank r owns the centres v whose key slots before them, c_v = sum_{u<v} 2 W hist[u], lie
   in [r S / G, (r + 1) S / G) (S: all slots of the epoch; nodes past the last slot go to the last
   rank) -- a pure function of the histogram;
3. each rank counts only its own centres, cut into sub-ranges of at most the sort capacity: exact
   global counts, since every key belongs to one centre; x_max is the largest count of the epoch;
4. each rank trains its own triples, centres ascending, on its replica;
5. merge: row v of T0 from the replica of owner(v); T1 = snap + ((T1_0 - snap) + (T1_1 - snap) + ...),
   float32, rank order, snap = T1 at the start of the epoch.  With one rank nothing is merged.
"""
from typing import Optional, Tuple

import numpy as np

import oracle


def token_histogram(walk_array: np.ndarray, n: int) -> np.ndarray:
    """Tokens per node over the walks (PAD skipped), uint64."""
    tokens = np.ascontiguousarray(walk_array, dtype=np.uint32).ravel()
    return np.bincount(tokens[tokens != oracle.PAD_TOKEN], minlength=n).astype(np.uint64)


def owner_bounds(histogram: np.ndarray, window_size: int, world: int) -> list:
    """``world + 1`` bounds: rank r owns the centres [bounds[r], bounds[r + 1])."""
    slots = np.asarray(histogram, dtype=np.uint64) * np.uint64(2 * window_size)
    before = np.concatenate([np.zeros(1, dtype=np.uint64), np.cumsum(slots, dtype=np.uint64)[:-1]])
    total = int(slots.sum())
    scaled = before * np.uint64(world)
    return [0] + [int(np.searchsorted(scaled, np.uint64(r * total), side="left")) for r in range(1, world)] + \
        [int(slots.shape[0])]


def sub_ranges(histogram: np.ndarray, window_size: int, lo: int, hi: int, capacity_slots: int) -> list:
    """[lo, hi) cut into ranges of at most ``capacity_slots`` key slots (one node may exceed it): a
    range closes before the node that would push it, non-empty, past the capacity.  Range bounds."""
    bounds, in_range = [lo], 0
    for v in range(lo, hi):
        s = int(histogram[v]) * 2 * window_size
        if in_range and in_range + s > capacity_slots:
            bounds.append(v)
            in_range = 0
        in_range += s
    return bounds + [hi]


def merge(t0s, t1s, snapshot: np.ndarray, bounds) -> Tuple[np.ndarray, np.ndarray]:
    """The tables every replica holds after the merge of a sharded epoch."""
    world = len(t0s)
    owner = np.searchsorted(np.asarray(bounds[1:world]), np.arange(t0s[0].shape[0]), side="right")
    t0 = t0s[0].copy()
    for r in range(1, world):
        t0[owner == r] = t0s[r][owner == r]
    change = t1s[0] - snapshot
    for t in t1s[1:]:
        change = change + (t - snapshot)
    return t0, snapshot + change


def train_shard(centre, context, count, bounds, rank, histogram, t0, t1, embedding_size, window_size, alpha,
                learning_rate, clipping_value, x_max, capacity_slots: Optional[int] = None) -> dict:
    """Step 4 for one rank, in place on its replica: its sub-ranges in ascending order of centre."""
    lo, hi = bounds[rank], bounds[rank + 1]
    cuts = [lo, hi] if capacity_slots is None else sub_ranges(histogram, window_size, lo, hi, capacity_slots)
    total = {"loss_sum": 0.0, "trained": 0}
    for a, b in zip(cuts[:-1], cuts[1:]):
        first, last = np.searchsorted(centre, [a, b])
        if last > first:
            r = oracle.glove_train(centre[first:last], context[first:last], count[first:last], t0, t1,
                                   embedding_size, alpha, learning_rate, clipping_value, max_count=x_max)
            total["loss_sum"] += r["loss_sum"]
            total["trained"] += r["trained"]
    return total


def glove_fit_sharded(indptr, indices, seed: int, embedding_size: int, epochs: int, walk_length: int,
                      window_size: int, alpha: float, learning_rate: float, learning_rate_decay: float,
                      return_weight: float = 1.0, explore_weight: float = 1.0, clipping_value: float = 6.0,
                      iterations: int = 1, world: int = 1, capacity_slots: Optional[int] = None):
    """Returns (t0, t1, epoch_mean_loss): the padded tables every replica holds at the end."""
    indptr = np.ascontiguousarray(indptr, dtype=np.int64)
    indices = np.ascontiguousarray(indices, dtype=np.uint32)
    n = indptr.shape[0] - 1
    srcs = oracle.sources(indptr)
    t0, t1 = oracle.init_tables(n, embedding_size, seed)
    per_epoch = iterations * srcs.shape[0]
    lr = np.float32(learning_rate)
    losses = []
    for epoch in range(epochs):
        w, _ = oracle.walks(indptr, indices, seed, epoch * per_epoch, per_epoch, walk_length, return_weight,
                            explore_weight, srcs=srcs)
        histogram = token_histogram(w, n)
        bounds = owner_bounds(histogram, window_size, world)
        centre, context, count = oracle.cooccurrence(w, window_size)
        x_max = int(count.max()) if count.shape[0] else 1
        snapshot = t1.copy()
        replicas, loss_sum, trained = [], 0.0, 0
        for rank in range(world):
            r0, r1 = t0.copy(), t1.copy()
            stats = train_shard(centre, context, count, bounds, rank, histogram, r0, r1, embedding_size,
                                window_size, alpha, float(lr), clipping_value, x_max, capacity_slots)
            loss_sum += stats["loss_sum"]
            trained += stats["trained"]
            replicas.append((r0, r1))
        if world == 1:
            t0, t1 = replicas[0]
        else:
            t0, t1 = merge([a for a, _ in replicas], [b for _, b in replicas], snapshot, bounds)
        losses.append(loss_sum / max(trained, 1))
        lr = np.float32(lr * np.float32(learning_rate_decay))
    return t0, t1, losses
