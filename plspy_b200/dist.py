"""Multi-process layouts (SURVEY.md section 8e), through torch.distributed (NCCL on GPUs; the same code runs under gloo
on CPU tensors for the host-logic tests).

Resample sharding (the default): X replicated, the resample index range cut into one contiguous shard per rank
(`shard`); only the tiny permutation counters, the two p x K moment matrices and the per-resample K x K outputs cross
NVLink.  Voxel sharding (`shard="voxels"`, task methods): each rank holds the columns `voxel_shard` gives it; the
N x N Gram matrix and the N x K product X V are all-reduced and the p x K results are gathered (`gather_spans`).
"""
import torch


_LOCAL_ONLY = False


class local_only:
    """Context manager: inside it this process behaves as a single-process run (no shards, no collectives) even though
    a process group exists -- e.g. rank 0 timing the whole job on its own GPU next to the sharded run (bench.py)."""

    def __enter__(self):
        global _LOCAL_ONLY
        self._prev, _LOCAL_ONLY = _LOCAL_ONLY, True
        return self

    def __exit__(self, *exc):
        global _LOCAL_ONLY
        _LOCAL_ONLY = self._prev
        return False


def world():
    """(rank, world_size) of the default process group, (0, 1) when not initialised."""
    import torch.distributed as dist
    if _LOCAL_ONLY:
        return 0, 1
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def assert_identical_rng(what="resampling indices"):
    """Multi-process runs draw the index matrices on every rank from numpy's GLOBAL stream and each rank keeps its
    shard, which is only the reference's resample set if every rank's stream is in the same state (seed all ranks
    alike; the common `seed + rank` idiom silently mixes shards of different streams).  One tiny all-reduce of a hash
    of the state; raises on every rank when they differ."""
    rank, size = world()
    if size == 1:
        return
    import zlib
    import numpy as np
    import torch.distributed as dist
    st = np.random.get_state(legacy=True)
    h = (zlib.crc32(np.asarray(st[1], dtype=np.uint32).tobytes()) << 12) ^ int(st[2])
    dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
    t = torch.tensor([h, -h], dtype=torch.int64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    hi, lo = int(t[0].item()), -int(t[1].item())
    if hi != lo:
        raise RuntimeError(
            f"rank {rank}: numpy's global RNG state differs between the ranks, so the {what} drawn on each rank would "
            "come from different streams and the sharded run would not be the reference's resample set.  Seed every "
            "rank identically (np.random.seed(k), not k + rank) or pass perm_indices= / boot_indices= explicitly.")


def shard(n, rank=None, size=None):
    """Contiguous [lo, hi) slice of range(n) owned by `rank`; sizes differ by at most one."""
    if rank is None:
        rank, size = world()
    base, rem = divmod(int(n), int(size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def _staged(t):
    """gloo implements only some collectives for CUDA tensors: device tensors are staged through the host there (two
    processes sharing ONE GPU over gloo is how the sharded code path is tested on a single-GPU box; NCCL refuses two
    ranks on one device)."""
    import torch.distributed as dist
    return t.is_cuda and dist.get_backend() == "gloo"


def allreduce_sum_(t):
    """In-place sum over ranks (no-op for a single process). Integer counters reduce exactly."""
    import torch.distributed as dist
    if world()[1] > 1:
        if _staged(t):
            c = t.cpu()
            dist.all_reduce(c, op=dist.ReduceOp.SUM)
            t.copy_(c)
        else:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t


def allreduce_packed_(tensors):
    """ONE all-reduce for several same-dtype tensors (counts, or [sum | sumsq]): packs, reduces, unpacks."""
    if world()[1] == 1:
        return tensors
    flat = torch.cat([t.reshape(-1) for t in tensors])
    allreduce_sum_(flat)
    o = 0
    for t in tensors:
        n = t.numel()
        t.copy_(flat[o:o + n].view_as(t))
        o += n
    return tensors


VOXEL_ALIGN = 256          # voxel_shard cut points: whole pairs of 128-voxel tiles, 16-byte aligned float32 rows


def voxel_shard(p, rank=None, size=None):
    """Contiguous [v0, v1) voxel range owned by `rank` in a voxel-sharded run: every cut point is a multiple of
    VOXEL_ALIGN (the last range ends at p) and range sizes differ by at most VOXEL_ALIGN.  With p < VOXEL_ALIGN x size
    the last ranks get empty ranges."""
    if rank is None:
        rank, size = world()
    p = int(p)
    lo, hi = shard(-(-p // VOXEL_ALIGN), rank, size)
    return min(p, lo * VOXEL_ALIGN), min(p, hi * VOXEL_ALIGN)


def gather_rows(local, n_total, lo):
    """Assemble per-resample rows computed on each rank's shard into the full [n_total, ...] tensor on
    every rank with ONE all_gather (shards padded to the largest shard, then trimmed)."""
    rank, size = world()
    if size == 1:
        return local
    return gather_spans(local, [shard(n_total, r, size) for r in range(size)])


def gather_spans(local, spans):
    """Concatenate along the first axis the blocks of rows [lo, hi) that rank r holds (`spans[r]`; any sizes, empty
    ones included), on every rank, with ONE all_gather (blocks padded to the largest, then trimmed).  COLLECTIVE."""
    import torch.distributed as dist
    size = len(spans)
    if size == 1:
        return local
    mx = max(hi - l for l, hi in spans)
    tail = tuple(local.shape[1:])
    buf = local
    if local.shape[0] != mx:
        buf = torch.zeros((mx,) + tail, dtype=local.dtype, device=local.device)
        buf[:local.shape[0]] = local
    if _staged(local):
        out_h = torch.empty((size * mx,) + tail, dtype=local.dtype)
        dist.all_gather_into_tensor(out_h, buf.contiguous().cpu())
        out = out_h.to(local.device)
    else:
        out = torch.empty((size * mx,) + tail, dtype=local.dtype, device=local.device)
        dist.all_gather_into_tensor(out, buf.contiguous())
    if all(hi - l == mx for l, hi in spans):
        return out
    return torch.cat([out[r * mx:r * mx + (hi - l)] for r, (l, hi) in enumerate(spans)], dim=0)
