"""
Multi-GPU work partitioning (one process per GPU, torch.distributed for the plumbing).

The hot path shards without any exchange inside the time loop (SURVEY.md section 8e):

  * ensemble members / scenarios  -> `partition_members`: whole members per rank;
  * calibration                   -> `partition_basins`: whole basins per rank, balanced by cell count
                                      (every basin's differential evolution is independent);
  * one scenario over several GPUs-> `BasinShard`: whole basins per rank; routing never leaves a flow
                                      component, so this is valid iff no river crosses a basin border
                                      (`basins_closed_under_flow`); Penman-Monteith needs the air
                                      temperature of the previous cell id, a one-column halo of an INPUT.

The only exchanges are a gather of small results at the end of a step (`gather_stack`, `gather_ragged_rows`) and the
rank-order fold of partial results onto rank 0 (`fold_to_rank0`, the ensemble statistics), NCCL on GPUs, gloo in the
CPU tests.
"""

import numpy as np


def lpt_partition(weights, n_parts):
    """
    Longest-processing-time-first bin packing.  Returns a list of `n_parts` index arrays (each sorted
    ascending); deterministic for equal weights (stable order, lowest-loaded / lowest-index bin wins).
    """
    weights = np.asarray(weights, dtype=np.int64)
    order = np.argsort(-weights, kind='stable')
    load = np.zeros(n_parts, dtype=np.int64)
    bins = [[] for _ in range(n_parts)]
    for i in order:
        k = int(np.argmin(load))
        bins[k].append(int(i))
        load[k] += weights[i]
    return [np.array(sorted(b), dtype=np.int64) for b in bins]


def partition_members(n_members, world_size):
    """Members of an ensemble per rank: contiguous blocks whose sizes differ by at most one."""
    base, extra = divmod(int(n_members), int(world_size))
    out, start = [], 0
    for r in range(world_size):
        n = base + (1 if r < extra else 0)
        out.append(np.arange(start, start + n))
        start += n
    return out


def partition_basins(basin_ids, world_size, basins=None):
    """
    Basin ids (1-based) per rank, balanced by cell count with `lpt_partition`.
    `basins` restricts the set (e.g. the calibration_basins of the ini file).
    """
    ids = np.asarray(basin_ids).astype(np.int64)
    counts = np.bincount(ids[ids > 0])
    cand = np.nonzero(counts)[0] if basins is None else np.asarray(sorted(int(b) for b in basins))
    parts = lpt_partition(counts[cand], world_size)
    return [cand[p] for p in parts]


def basins_closed_under_flow(dsid, basin_ids):
    """True iff every cell drains into a cell of its own basin (routing can then be sharded by basin)."""
    dsid = np.asarray(dsid)
    b = np.asarray(basin_ids)
    has = dsid > 0
    return bool(np.all(b[dsid[has] - 1] == b[has]))


class BasinShard:
    """
    The cells of a set of basins, renumbered 0..n_local-1 in ascending global order, plus what the
    kernels need to run on the shard alone.

      cells        global cell indices of the shard
      halo_cells   global indices whose `tair` must be appended as halo columns for Penman-Monteith
      prev_idx     per local cell: local index (or n_local + halo position) of global cell c - 1,
                   -1 for global cell 0 (-> xan_pm_pet's d_prev_idx)
    """

    def __init__(self, basin_ids, basins):
        ids = np.asarray(basin_ids).astype(np.int64)
        self.basins = np.asarray(basins, dtype=np.int64)
        self.cells = np.nonzero(np.isin(ids, self.basins))[0]
        n = ids.shape[0]
        local = np.full(n, -1, dtype=np.int64)
        local[self.cells] = np.arange(len(self.cells))
        prev = self.cells - 1
        need = prev[(prev >= 0)]
        need = need[local[need] < 0]
        self.halo_cells = np.unique(need)
        halo_pos = {int(g): len(self.cells) + k for k, g in enumerate(self.halo_cells)}
        self.prev_idx = np.array([(-1 if p < 0 else (local[p] if local[p] >= 0 else halo_pos[int(p)])) for p in prev],
                                 dtype=np.int32)
        self.local_of_global = local

    @property
    def n_local(self):
        return len(self.cells)

    def take(self, arr):
        """Rows of a [ncell, ...] array that belong to the shard."""
        return np.ascontiguousarray(np.asarray(arr)[self.cells])

    def take_with_halo(self, arr):
        """Shard rows followed by the halo rows (for the PM air temperature)."""
        a = np.asarray(arr)
        return np.ascontiguousarray(np.concatenate([a[self.cells], a[self.halo_cells]], axis=0))

    def local_coords(self, coords):
        """coords rows of the shard with ids renumbered 1..n_local (topology is built per shard)."""
        c = np.array(np.asarray(coords)[self.cells], dtype=float)
        c[:, 0] = np.arange(1, len(self.cells) + 1)
        return c

    def scatter(self, out_global, local_values):
        """Write shard results back into a [ncell, ...] array."""
        out_global[self.cells] = local_values
        return out_global


def gather_stack(local, group=None):
    """
    All-gather equally shaped tensors from every rank and stack them on a new leading axis
    (NCCL for cuda tensors, gloo for cpu tensors).  Single-process runs return local[None].
    """
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return local[None]
    parts = [torch.empty_like(local) for _ in range(dist.get_world_size(group))]
    dist.all_gather(parts, local.contiguous(), group=group)
    return torch.stack(parts, dim=0)


def fold_to_rank0(partial, counts, merge):
    """
    Rank-order fold of per-rank partial results onto rank 0 (point-to-point: NCCL for cuda tensors, gloo for cpu).
    partial: this rank's list of tensors (None on a rank with counts[rank] == 0); counts: items per rank;
    merge(a, na, b, nb) combines partial a of na items with partial b of nb items and returns the result.
    Rank 0 returns merge(...merge(merge(p0, c0, p1, c1), c0 + c1, p2, c2)...), skipping ranks without items (None if
    no rank has any); the other ranks send their partial and return None.  Single-process runs return `partial`.
    The order is fixed, so the result is deterministic for a given world size.
    """
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return partial
    rank = dist.get_rank()
    if rank != 0:
        if counts[rank] > 0:
            for t in partial:
                dist.send(t.contiguous(), dst=0)
        return None
    acc, n = partial, counts[0]
    for r in range(1, len(counts)):
        if counts[r] == 0:
            continue
        recv = [torch.empty_like(t) for t in acc]
        for t in recv:
            dist.recv(t, src=r)
        acc = merge(acc, n, recv, counts[r])
        n += counts[r]
    return acc


def gather_ragged_rows(local_rows, local_values, n_rows, group=None):
    """
    Every rank owns the values of some rows (e.g. calibrated parameters of its basins): returns the
    full [n_rows, ...] tensor on every rank (rows nobody owns stay NaN).
    """
    import torch
    import torch.distributed as dist
    full = torch.full((n_rows,) + tuple(local_values.shape[1:]), float('nan'), dtype=local_values.dtype,
                      device=local_values.device)
    rows = torch.as_tensor(np.asarray(local_rows), dtype=torch.long, device=local_values.device)
    if len(rows):
        full[rows] = local_values
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        mask = torch.isnan(full)
        contrib = torch.where(mask, torch.zeros_like(full), full)
        cnt = (~mask).to(full.dtype)
        dist.all_reduce(contrib, group=group)
        dist.all_reduce(cnt, group=group)
        full = torch.where(cnt > 0, contrib, torch.full_like(contrib, float('nan')))
    return full
