"""Host-side plumbing for ONE comparison partitioned over the GPUs of a box (include/rk_b200.h, rk_dist_*).

The partitioning, the exchanges (NCCL) and the kernels live in librk_b200.so (csrc/multi.cu, csrc/k7_dist.cu).  What is
left for the application — one process per GPU — is to move two small byte strings between the ranks and to decide which
slice of the file each rank loads; here that is done with torch.distributed (any backend: the strings are pickled objects).
"""
from __future__ import annotations

import numpy as np

from . import capi


def slice_bounds(n: int, rank: int, world: int) -> tuple[int, int]:
    """[lo, hi) of rank's contiguous slice of an n-record file.  Slices start on a 16-record boundary (16 x 109 bytes is a
    multiple of 16: device slices of one resident file stay 16-byte aligned); together they cover 0..n exactly."""
    def cut(r):
        if r >= world:
            return n
        b = n * r // world
        return b - b % 16
    return cut(rank), cut(rank + 1)


def csv_slice_bounds(path: str, body_pos: int, rank: int, world: int, window: int = 1 << 16) -> tuple[int, int]:
    """[lo, hi) of rank's slice of a GECKO CSV file whose body (the bytes after the 16 header lines) starts at byte
    body_pos, for rk_dist_load_csv: cut r is one byte past the first newline at or after body byte bytes * r / world, or
    the end of the file when there is none (rk_multi_load_csv's rule).  Only a window after each of the two cuts is read,
    so each process reads just the bytes around its own slice."""
    import os
    size = os.path.getsize(path)
    n = size - body_pos

    def cut(r: int, f) -> int:
        if r <= 0:
            return body_pos
        if r >= world:
            return size
        pos = body_pos + n * r // world
        while pos < size:
            f.seek(pos)
            chunk = f.read(window)
            k = chunk.find(b"\n")
            if k >= 0:
                return pos + k + 1
            pos += len(chunk)
        return size

    with open(path, "rb") as f:
        return cut(rank, f), cut(rank + 1, f)


def default_capacity(n_per_rank: int) -> int:
    """workspace rows per rank: room for an uneven partition (the cuts of the output exchange balance sort_groups work, not
    lines: a rank whose groups are small gets more lines)"""
    return int(n_per_rank * 1.5) + (1 << 16)


def bootstrap(ctx: capi.Context, cap_per_rank: int, group=None) -> None:
    """Collective over the torch.distributed group: NCCL unique id from rank 0, then the peer-memory blobs of all ranks."""
    import torch.distributed as dist
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    box = [capi.dist_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0, group=group)
    ctx.dist_init(rank, world, box[0], cap_per_rank)
    blobs = [None] * world
    dist.all_gather_object(blobs, ctx.dist_export(), group=group)
    ctx.dist_import(b"".join(blobs))


_MASK = (1 << 64) - 1


def output_checksum(order: np.ndarray, gid: np.ndarray, repval: np.ndarray, identity: np.ndarray, line_offset: int = 0) -> int:
    """Position-dependent 64-bit checksum of a range of output lines; the sum (mod 2^64) over the ranks' ranges equals the
    checksum of the whole output, so 1 GPU and N GPUs can be compared without gathering the lines."""
    with np.errstate(over="ignore"):
        pos = np.arange(line_offset, line_offset + order.shape[0], dtype=np.uint64)
        mix = (pos + np.uint64(1)) * np.uint64(0x9E3779B97F4A7C15)
        word = (order.astype(np.uint64) * np.uint64(1000003) + gid.astype(np.uint64) * np.uint64(10007)
                + repval.astype(np.uint64) * np.uint64(101) + identity.view(np.uint32).astype(np.uint64))
        return int(((word ^ mix) * np.uint64(0x2545F4914F6CDD1D)).sum(dtype=np.uint64)) & _MASK
