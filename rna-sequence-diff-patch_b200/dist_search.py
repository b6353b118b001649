"""dist_search.py — database search sharded over the GPUs of one box (SURVEY 8e, config 5).

One process per GPU (torch.distributed).  The packed database is sharded contiguously by record
index (balanced by total symbols), the query batch is the same on every rank, each rank computes
its local top-k per query with key (score desc, global index asc), and ONE all_gather of
Q x k x (fp64 score, int64 index) per rank brings the candidates together; the merge with the same
key (rsd_topk_merge) reproduces the reference's stable descending sort over the whole collection
because shards are index-contiguous.  torch is plumbing only (process group, device tensors).

There is no idf / tf-idf similarity here: a rank holds one shard and cannot know the collection's document
frequencies.  Callers that need those vector types over several GPUs use MultiEngine (one process), which runs the
document-frequency sums through its shards in order."""
from __future__ import annotations

import numpy as np

from .encoding import PackedSeqs
from .engine import Engine, topk_merge


def shard_bounds(lens: np.ndarray, world: int):
    """Contiguous [lo, hi) record ranges per rank, balanced by sum of lengths (8e: 'balance by Σ len')."""
    n = int(lens.shape[0])
    if world <= 1 or n == 0:
        return [(0, n)] + [(n, n)] * (max(world, 1) - 1)
    csum = np.concatenate([[0], np.cumsum(lens, dtype=np.int64)])
    total = int(csum[-1])
    cuts = [0]
    for r in range(1, world):
        target = total * r // world
        cuts.append(int(np.searchsorted(csum, target, side="left")))
    cuts.append(n)
    cuts = [min(max(c, 0), n) for c in cuts]
    for r in range(1, len(cuts)):
        cuts[r] = max(cuts[r], cuts[r - 1])
    return [(cuts[r], cuts[r + 1]) for r in range(world)]


def slice_packed(p: PackedSeqs, lo: int, hi: int) -> PackedSeqs:
    """Records [lo, hi) of a packed batch as a self-contained packed batch (word-aligned, so a slice)."""
    if hi <= lo:
        return PackedSeqs(np.zeros(4, np.uint32), np.zeros(0, np.int64), np.zeros(0, np.int32), p.bits, p.symmask)
    per = 32 // p.bits
    w0 = int(p.start[lo])
    w1 = int(p.start[hi - 1]) + (int(p.len[hi - 1]) + per - 1) // per
    words = np.concatenate([p.words[w0:w1], np.zeros(4, np.uint32)])
    return PackedSeqs(words, (p.start[lo:hi] - w0).astype(np.int64), p.len[lo:hi].copy(), p.bits, p.symmask,
                      canonical=p.canonical)


def gather_merge(local_idx: np.ndarray, local_score: np.ndarray, group=None, device=None):
    """all_gather the per-rank [Q, k] lists (NCCL on `device`, gloo on CPU) and merge them."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return local_idx, local_score
    world = dist.get_world_size(group)
    ti = torch.from_numpy(np.ascontiguousarray(local_idx))
    ts = torch.from_numpy(np.ascontiguousarray(local_score))
    if device is not None:
        ti, ts = ti.to(device), ts.to(device)
    gi = [torch.empty_like(ti) for _ in range(world)]
    gs = [torch.empty_like(ts) for _ in range(world)]
    dist.all_gather(gi, ti, group=group)
    dist.all_gather(gs, ts, group=group)
    idx = np.stack([t.cpu().numpy() for t in gi]); sc = np.stack([t.cpu().numpy() for t in gs])
    return topk_merge(idx, sc)


class ShardedSearch:
    """Rank-local shard on one Engine + the single collective of the search path."""

    def __init__(self, engine: Engine, db: PackedSeqs, rank: int = 0, world: int = 1, group=None, device=None):
        self.engine, self.rank, self.world, self.group, self.device = engine, rank, world, group, device
        self.bounds = shard_bounds(db.len, world)
        lo, hi = self.bounds[rank]
        self.lo, self.hi = lo, hi
        shard = slice_packed(db, lo, hi)
        shard.symmask = db.symmask
        engine.db_load(shard, global_index_base=lo)

    def search(self, Q: PackedSeqs, k: int):
        idx, sc = self.engine.db_search_topk(Q, k)
        return gather_merge(idx, sc, self.group, self.device)

    def similarity(self, query_codes: np.ndarray, method: str, k: int):
        """Top-k of one of Engine.SIM_METHODS over the sharded database: local top-k, the same all_gather + merge
        (a shard with fewer than k rankable records pads with index -1, which the merge skips)."""
        _, idx, sc = self.engine.db_similarity(query_codes, method, k=k, want_scores=False)
        return gather_merge(idx[None, :], sc[None, :], self.group, self.device)
