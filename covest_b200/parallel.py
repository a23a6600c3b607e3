"""Multi-GPU sharding of candidate sets: one process per GPU (torchrun), static slices, no
collective on the data path; one small all-gather of every rank's best rows per round
(SURVEY.md section 8(e)).  The reference's counterpart is Pool.map over candidates
(covest/grid.py:61-64, covest/covest.py:67-68).

Works with CUDA tensors over NCCL and with CPU tensors over gloo (the CPU test-suite).
"""
import numpy as np


def _dist():
    import torch.distributed as dist
    return dist


def world():
    """(rank, world_size); (0, 1) when torch.distributed is not initialised."""
    try:
        dist = _dist()
        if dist.is_available() and dist.is_initialized():
            return dist.get_rank(), dist.get_world_size()
    except ImportError:
        pass
    return 0, 1


def shard_strided(total, rank, world_size):
    """(first, stride, count) of the rank's slice: indices rank, rank + W, ...  Striding spreads
    the expensive region of a lattice (small q: many copy-number terms) over all ranks."""
    count = (total - rank + world_size - 1) // world_size if total > rank else 0
    return rank, world_size, count


def shard_blocked(total, block, rank, world_size):
    """(first, stride, block, count) of the rank's slice when it takes whole runs of `block`
    consecutive indices: runs rank, rank + W, ...  For a repeats-model lattice block is the number
    of (q1, q2, q) combinations, so that every (coverage, error_rate) group -- whose bin profiles
    the factored path computes once -- lives on one rank; all groups cost the same, so the split
    is balanced."""
    runs = (total + block - 1) // block
    mine = (runs - rank + world_size - 1) // world_size if runs > rank else 0
    count = mine * block
    if mine and (rank + (mine - 1) * world_size + 1) * block > total:
        count -= (rank + (mine - 1) * world_size + 1) * block - total
    return rank, world_size, block, count


def shard_contiguous(total, rank, world_size):
    """[lo, hi) of a balanced contiguous split."""
    base, extra = divmod(total, world_size)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def allgather_rows(rows):
    """All ranks' (K, C) row blocks stacked in rank order: (W*K, C) tensor on the same device."""
    import torch
    dist = _dist()
    if not isinstance(rows, torch.Tensor):
        rows = torch.from_numpy(np.ascontiguousarray(rows))
    rank, w = world()
    if w == 1:
        return rows
    rows = rows.contiguous()
    out = torch.empty((w * rows.shape[0], rows.shape[1]), dtype=rows.dtype, device=rows.device)
    dist.all_gather_into_tensor(out, rows)
    return out


def to_comm(array, device=None):
    """A numpy block as a tensor where the collectives of the current backend want it (`device`:
    a CUDA device under NCCL, None = host under gloo or without a process group)."""
    import torch
    t = torch.from_numpy(np.ascontiguousarray(array, dtype=np.float64))
    return t.to(device) if device is not None else t


def broadcast_rows(array, device=None, src=0):
    """Rank `src`'s float64 block on every rank (same shape everywhere); a no-op without a process
    group.  Used for the random multi-start points, which every rank draws from its own unseeded
    `random` (covest/grid.py:95-110)."""
    rank, w = world()
    if w == 1:
        return np.asarray(array, dtype=np.float64)
    t = to_comm(array, device)
    _dist().broadcast(t, src=src)
    return t.cpu().numpy()


def merge_topk(rows, k_best):
    """The k_best best rows (column 0 = log-likelihood, larger is better) of a stacked block,
    best first.  NaN and padding (-inf) sort last.  Ties are broken by the parameter columns in
    lexicographic order -- for a lattice with ascending axes that is the lattice index, i.e. the
    tie-break of the single-GPU top-K -- so the result does not depend on the number of ranks."""
    import torch
    if not isinstance(rows, torch.Tensor):
        rows = torch.from_numpy(np.ascontiguousarray(rows))
    if rows.is_cuda and rows.dtype == torch.float64 and rows.shape[0] <= 2048:
        return _merge_topk_device(rows.contiguous(), k_best)
    order = torch.arange(rows.shape[0], device=rows.device)
    for col in range(rows.shape[1] - 1, 0, -1):  # least significant key first, stable sorts
        vals = rows[order, col]
        vals = torch.where(torch.isnan(vals), torch.full_like(vals, float('inf')), vals)
        order = order[torch.sort(vals, stable=True).indices]
    key = rows[order, 0]
    key = torch.where(torch.isnan(key), torch.full_like(key, float('-inf')), key)
    order = order[torch.sort(key, descending=True, stable=True).indices]
    return rows[order[:k_best]]


def _merge_topk_device(rows, k_best):
    """merge_topk of a CUDA block in one launch (cvb_merge_rows, include/covest_b200.h): the same
    order as the torch formulation above, which stays the CPU / gloo path."""
    import ctypes

    import torch

    from . import _capi
    lib = _capi.load()
    out = torch.empty((k_best, rows.shape[1]), dtype=torch.float64, device=rows.device)
    stream = torch.cuda.current_stream(rows.device).cuda_stream
    with torch.cuda.device(rows.device):
        rc = lib.cvb_merge_rows(ctypes.c_void_p(rows.data_ptr()), int(rows.shape[0]), int(rows.shape[1]),
                                int(k_best), ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(stream or 1))
    if rc != 0:
        raise RuntimeError('cvb_merge_rows failed (%d)' % rc)
    return out[:min(int(k_best), int(rows.shape[0]))]


def merge_segments(blocks):
    """Segment by segment, the best of W per-rank (n_seg, C) row blocks (a (W, n_seg, C) array): the
    order of merge_topk -- larger column 0 first, NaN as -inf, ties by the other columns in ascending
    lexicographic order with NaN last, then the lower rank.  A segment no rank has a point of keeps
    (-inf, NaN...).  For a lattice with ascending axes the tie-break is the lattice index, so the result
    is the rows of one cvb_lattice_profile call over the whole lattice.  Vectorised over the segments."""
    blocks = np.asarray(blocks, dtype=np.float64)
    best = blocks[0].copy()
    for other in blocks[1:]:
        a = np.where(np.isnan(other[:, 0]), -np.inf, other[:, 0])
        b = np.where(np.isnan(best[:, 0]), -np.inf, best[:, 0])
        take = a > b
        undecided = a == b
        for col in range(1, blocks.shape[2]):
            u = np.where(np.isnan(other[:, col]), np.inf, other[:, col])
            v = np.where(np.isnan(best[:, col]), np.inf, best[:, col])
            take |= undecided & (u < v)
            undecided &= u == v
        best[take] = other[take]
    return best


def sharded_best_rows(evaluate_slice, total, k_best, block=1):
    """Every rank evaluates its slice (runs of `block` indices, dealt round-robin) with
    `evaluate_slice(first, stride, block, count)` -> (k_best, C) best-first rows, the row blocks
    are all-gathered and merged.  Returns the global k_best rows (identical on every rank)."""
    rank, w = world()
    first, stride, block, count = shard_blocked(total, block, rank, w)
    rows = evaluate_slice(first, stride, block, count)
    return merge_topk(allgather_rows(rows), k_best)


def split_starts(rows, rank=None, world_size=None):
    """The refinement starts this rank owns: row i goes to rank i % W."""
    r, w = world()
    rank = r if rank is None else rank
    world_size = w if world_size is None else world_size
    return rows[rank::world_size]
