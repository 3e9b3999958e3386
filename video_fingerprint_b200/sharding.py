"""Multi-GPU layer: one process per GPU (torch.distributed, NCCL over NVLink/NVSwitch on the GPU box, gloo in
the CPU tests). The reference has no distributed code at all (SURVEY.md section 2); the hot path shards as
follows (SURVEY.md section 8e):

* forward: clips are independent units -> length-balanced (LPT) partition over ranks, weights replicated,
  NO collective while fingerprinting;
* join: ONE all-gather of the (n_r, dim) fp32 embedding shards, started first and overlapped with the join of the
  rank's rows against its OWN columns; the other column ranges follow once the gather has landed (`q_row0` and a column
  offset make the pair indices global);
* top-k: queries are sharded the same way, the database is the all-gathered matrix -> no merge step;
* the greedy grouping is sequential in the seed index by definition, so the per-rank pair lists are gathered
  and grouped on rank 0 (host).
"""
from __future__ import annotations

from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.distributed as dist


def partition_clips(lengths: Sequence[int], world: int) -> List[List[int]]:
    """Longest-processing-time-first assignment of clips to ranks by frame count (forward cost is ~linear
    in T). Deterministic; each rank's list is in ascending clip order."""
    order = sorted(range(len(lengths)), key=lambda i: (-int(lengths[i]), i))
    loads = [0] * world
    parts: List[List[int]] = [[] for _ in range(world)]
    for i in order:
        r = min(range(world), key=lambda k: (loads[k], k))
        parts[r].append(i)
        loads[r] += int(lengths[i])
    return [sorted(p) for p in parts]


def row_block(n: int, world: int, rank: int, align: int = 128) -> Tuple[int, int]:
    """Contiguous row block of rank `rank`; interior boundaries are multiples of the 128-row GEMM tile."""
    per = -(-n // world)
    per = -(-per // align) * align
    lo = min(n, rank * per)
    hi = min(n, lo + per)
    return lo, hi


def _world(group=None) -> Tuple[int, int]:
    if not dist.is_available() or not dist.is_initialized():
        return 1, 0
    return dist.get_world_size(group), dist.get_rank(group)


def all_gather_rows(local: torch.Tensor, group=None) -> Tuple[torch.Tensor, List[int]]:
    """All-gather row shards with possibly different row counts. Returns (concatenation in rank order, counts)."""
    world, _ = _world(group)
    if world == 1:
        return local, [local.shape[0]]
    counts_t = torch.tensor([local.shape[0]], dtype=torch.int64, device=local.device)
    all_counts = [torch.zeros_like(counts_t) for _ in range(world)]
    dist.all_gather(all_counts, counts_t, group=group)
    counts = [int(c.item()) for c in all_counts]
    width = max(counts)
    padded = torch.zeros((width,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    padded[: local.shape[0]] = local
    buf = torch.empty((world * width,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(buf, padded, group=group)
    parts = [buf[r * width : r * width + counts[r]] for r in range(world)]
    return torch.cat(parts, dim=0), counts


def sharded_fingerprint(model, clips: Sequence[torch.Tensor], group=None) -> torch.Tensor:
    """Every rank fingerprints its LPT share of `clips` (all ranks pass the same list; only the local share is
    touched), then the shards are all-gathered and put back into clip order. Returns (n, D) on every rank."""
    world, rank = _world(group)
    lengths = [int(c.shape[0]) for c in clips]
    parts = partition_clips(lengths, world)
    mine = parts[rank]
    if mine:
        local = model.fingerprint_clips([clips[i] for i in mine])
    else:
        local = torch.empty((0, model.embedding_dim), dtype=torch.float32, device=torch.device("cuda", torch.cuda.current_device()))
    gathered, counts = all_gather_rows(local, group)
    order = torch.tensor([i for p in parts for i in p], dtype=torch.int64, device=gathered.device)
    out = torch.empty_like(gathered)
    out[order] = gathered
    return out


def symmetric_block_plan(world: int, rank: int, counts: Sequence[int]) -> List[Tuple[int, int, int, int]]:
    """Blocks of the symmetric score matrix rank `rank` computes, as (local row lo, local row hi, global column lo, global
    column hi). Entry 0 is the rank's diagonal block (a self join). Every other entry is reported together with its mirror
    image, so each unordered pair of ranks appears in exactly ONE plan: rank r takes the peers r+1 .. r+(G-1)/2 (cyclically);
    for even G the block against the opposite rank is split in half between the two."""
    starts = [sum(counts[:r]) for r in range(world)]
    n_loc = counts[rank]
    plan = [(0, n_loc, starts[rank], starts[rank] + n_loc)]
    for d in range(1, (world - 1) // 2 + 1):
        peer = (rank + d) % world
        plan.append((0, n_loc, starts[peer], starts[peer] + counts[peer]))
    if world > 1 and world % 2 == 0:
        peer = (rank + world // 2) % world
        if rank < world // 2:    # my first half of rows x all of the peer's columns
            plan.append((0, n_loc // 2, starts[peer], starts[peer] + counts[peer]))
        else:                    # all my rows x the columns of the peer's rows the peer did not take
            plan.append((0, n_loc, starts[peer] + counts[peer] // 2, starts[peer] + counts[peer]))
    return plan


class _RowGather:
    """An all-gather of row shards in flight (NCCL runs it on its own stream): `wait()` returns (rows in rank order, counts).
    The returned rows live in a buffer the next gather of the same shape overwrites: use them before starting another one."""

    _bufs: dict = {}

    def __init__(self, local: torch.Tensor, group=None):
        world, _ = _world(group)
        self.local, self.world, self.work, self.buf = local, world, None, None
        if world == 1:
            self.counts = [local.shape[0]]
            return
        counts_t = torch.tensor([local.shape[0]], dtype=torch.int64, device=local.device)
        all_counts = [torch.zeros_like(counts_t) for _ in range(world)]
        dist.all_gather(all_counts, counts_t, group=group)
        self.counts = [int(c.item()) for c in all_counts]
        self.width = max(self.counts)
        if local.shape[0] == self.width:
            padded = local
        else:
            padded = torch.zeros((self.width,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
            padded[: local.shape[0]] = local
        # One receive buffer per (device, dtype, shape) is kept and reused: a fresh 0.5 - 1 GB allocation per call means a fresh
        # address for NCCL every time (and allocator churn); on shared 2-GPU boxes that showed up as sporadic ~80 ms stalls.
        # The collective is ordered after the current stream's work, i.e. after the previous call's reads of the buffer.
        shape = (world * self.width,) + tuple(local.shape[1:])
        key = (str(local.device), local.dtype, shape)
        self.buf = _RowGather._bufs.get(key)
        if self.buf is None:
            _RowGather._bufs.clear()   # keep one buffer alive, not one per size ever seen
            self.buf = _RowGather._bufs[key] = torch.empty(shape, dtype=local.dtype, device=local.device)
        self.work = dist.all_gather_into_tensor(self.buf, padded, group=group, async_op=True)

    def wait(self) -> Tuple[torch.Tensor, List[int]]:
        if self.world == 1:
            return self.local, self.counts
        self.work.wait()
        if all(c == self.width for c in self.counts):
            return self.buf, self.counts
        parts = [self.buf[r * self.width : r * self.width + self.counts[r]] for r in range(self.world)]
        return torch.cat(parts, dim=0), self.counts


def sharded_threshold_join_device(
    local_embeddings: torch.Tensor, thr: float, group=None, join_fn: Optional[Callable] = None
) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, int]:
    """Row-block sharded all-pairs join, device part. `local_embeddings` is this rank's (n_r, dim) shard, shards being
    consecutive in rank order. The all-gather of the shards is started first and runs (NCCL, NVLink) WHILE the rank joins
    its rows against its own columns - the one block that needs no remote data; the two remaining column ranges follow
    when the gather has landed. The score matrix is symmetric, so every block of it is computed by ONE rank, which also
    reports the mirrored pairs: the union of the ranks' results is the full ordered pair set, each pair exactly once,
    but a rank's list is not restricted to its own rows. Returns (i, j, s) with GLOBAL indices (device tensors,
    unordered) and the total row count. `join_fn(db, thr, q, q_row0) -> (i, j, s)` defaults to the device join; the CPU tests inject the oracle."""
    world, rank = _world(group)
    if join_fn is None:
        from .fingerprint import threshold_join_device

        def join_fn(db, thr_, q, q_row0):  # noqa: E306
            return threshold_join_device(db, thr_, q=q, q_row0=q_row0)

    local = local_embeddings.float().contiguous()
    gather = _RowGather(local, group)
    counts = gather.counts
    starts = [sum(counts[:r]) for r in range(world)]
    row0, n_loc, n_all = starts[rank], local.shape[0], sum(counts)
    out = []

    def block(db, col0, q=None, q0=0, mirror=False):
        q = local if q is None else q
        if q.shape[0] == 0 or db.shape[0] == 0:
            return
        i, j, s = (torch.as_tensor(t) for t in join_fn(db, thr, q, row0 + q0))
        i, j, s = i.to(torch.int64), j.to(torch.int64) + col0, s.to(torch.float32)
        out.append((i, j, s))
        if mirror:   # S is symmetric: the block (peer rows x my columns) is this one transposed
            out.append((j, i, s))

    block(local, row0)                       # own columns (a self join: the library screens the upper triangle only); overlaps the gather
    full, _ = gather.wait()
    for q_lo, q_hi, c_lo, c_hi in symmetric_block_plan(world, rank, counts)[1:]:
        block(full[c_lo:c_hi], c_lo, q=None if (q_lo, q_hi) == (0, n_loc) else local[q_lo:q_hi], q0=q_lo, mirror=True)
    if not out:
        z = torch.zeros(0, dtype=torch.int64, device=local.device)
        return z, z.clone(), torch.zeros(0, dtype=torch.float32, device=local.device), n_all
    return torch.cat([o[0] for o in out]), torch.cat([o[1] for o in out]), torch.cat([o[2] for o in out]), n_all


def sharded_threshold_join(
    local_embeddings: torch.Tensor,
    thr: float,
    group=None,
    join_fn: Optional[Callable] = None,
    gather_to: Optional[int] = 0,
) -> Optional[Tuple[np.ndarray, np.ndarray, np.ndarray]]:
    """`sharded_threshold_join_device` + the gather of the per-rank pair lists (as int32, int32, fp32 bits - 12 bytes a
    pair) for the sequential greedy grouping. Returns (i, j, s) sorted by (i, j) on rank `gather_to` (None elsewhere), or
    on every rank if gather_to is None."""
    world, rank = _world(group)
    i, j, s, _ = sharded_threshold_join_device(local_embeddings, thr, group, join_fn)
    dev = local_embeddings.device
    trip = torch.stack([i.to(torch.int32), j.to(torch.int32), s.contiguous().view(torch.int32)], dim=1).to(dev)
    if world > 1:
        trip, _ = all_gather_rows(trip, group)
    if gather_to is not None and rank != gather_to:
        return None
    t = trip.cpu()
    pi, pj = t[:, 0].numpy().astype(np.int64), t[:, 1].numpy().astype(np.int64)
    ps = t[:, 2].contiguous().view(torch.float32).numpy()
    order = np.lexsort((pj, pi))
    return pi[order], pj[order], ps[order]


def sharded_topk(local_queries: torch.Tensor, local_db: torch.Tensor, k: int, group=None, topk_fn: Optional[Callable] = None):
    """Query-sharded flat inner-product top-k: the database shards are all-gathered once, every rank searches its
    own queries against the full database (no merge). Returns this rank's (scores, indices)."""
    if topk_fn is None:
        from .fingerprint import topk_inner_product_device as topk_fn
    db, _ = all_gather_rows(local_db.float().contiguous(), group)
    return topk_fn(local_queries.float().contiguous(), db, k)
