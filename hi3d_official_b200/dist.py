"""Multi-GPU plumbing: one process per GPU (`torchrun`), `torch.distributed` (NCCL on B200, gloo in CPU tests).

The hot path shards across GPUs in two ways (SURVEY.md 8e):
  * videos: every rank denoises its own orbital video (BASELINE configs[4]); no data-path collective, only the
    final gather of decoded frames / a max-over-ranks of the device time.  This is what bench.py --gpus N runs.
  * frames of one video (BASELINE configs[3]): rank r owns frames [r*T/R, (r+1)*T/R) of both CFG halves.
    Per-frame ops need nothing; the temporal ops need (i) an all-gather of the temporal-attention K/V rows,
    (ii) a one-frame halo for the (3,1,1) temporal conv and (iii) an all-reduce of the (sum, sumsq) GroupNorm
    partials.  The helpers below implement exactly those three exchanges on plain tensors so the same code is
    exercised under gloo on CPU (tests/test_dist_cpu.py) and NCCL on GPUs.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist


def world() -> Tuple[int, int]:
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_range(n: int, rank: int, world_size: int) -> range:
    """Contiguous, balanced split of n items (videos or frames): the first n % world ranks get one extra."""
    base, extra = divmod(n, world_size)
    start = rank * base + min(rank, extra)
    return range(start, start + base + (1 if rank < extra else 0))


def frame_owner(t: int, T: int, world_size: int) -> int:
    for r in range(world_size):
        if t in shard_range(T, r, world_size):
            return r
    raise ValueError(t)


def max_over_ranks_ms(ms: float, device) -> float:
    t = torch.tensor([ms], dtype=torch.float64, device=device)
    if world()[1] > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def gather_to_rank0(x: torch.Tensor) -> Optional[torch.Tensor]:
    """Concatenate equally-shaped per-rank tensors along dim 0 on rank 0 (decoded frames / final latents)."""
    rank, ws = world()
    if ws == 1:
        return x
    bufs = [torch.empty_like(x) for _ in range(ws)]
    dist.all_gather(bufs, x.contiguous())
    return torch.cat(bufs, 0) if rank == 0 else None


# ---- frame-sharded exchanges, NCCL / gloo form -----------------------------------------------------------------------
# Used by the launch plan (unet._Plan) when HI3D_SHARD_EXCHANGE=nccl; the default on B200 is the peer-memory form
# (peer.py + the sharded kernels), which needs no collective library on the step's path.  These operate in place on the
# plan's own buffers and are backend-agnostic, so tests/test_dist_cpu.py runs exactly this code under 2-rank gloo.
def allreduce_sum_(t: torch.Tensor, deterministic: bool = False) -> torch.Tensor:
    """[B, 32, 2] (sum, sumsq) GroupNorm partials of this rank's frames -> totals over all frames of the clip.
    deterministic: an all-gather and a sum in rank order (the order of the peer-memory exchange kernel), so that every rank
    gets the same bits run after run; an NCCL all-reduce picks its own reduction order."""
    ws = world()[1]
    if ws > 1 and deterministic:
        parts = [torch.empty_like(t) for _ in range(ws)]
        dist.all_gather(parts, t.contiguous())
        acc = parts[0].clone()
        for p in parts[1:]:
            acc += p
        t.copy_(acc)
    elif ws > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t


def halo_exchange_(g: torch.Tensor, rank: int, world_size: int) -> torch.Tensor:
    """g: [B, T_local + 2, X] haloed GroupNorm output (frames 1..T_local are local).  Frame 0 <- last local frame of
    rank-1, frame T_local+1 <- first local frame of rank+1, zeros at the clip boundaries (the Conv3d zero padding at
    t = -1 and t = T, openaimodel.py:252-261)."""
    T = g.shape[1] - 2
    ops_ = []
    for b in range(g.shape[0]):
        if rank > 0:
            ops_ += [dist.P2POp(dist.isend, g[b, 1], rank - 1), dist.P2POp(dist.irecv, g[b, 0], rank - 1)]
        else:
            g[b, 0].zero_()
        if rank + 1 < world_size:
            ops_ += [dist.P2POp(dist.isend, g[b, T], rank + 1), dist.P2POp(dist.irecv, g[b, T + 1], rank + 1)]
        else:
            g[b, T + 1].zero_()
    if ops_:
        for wk in dist.batch_isend_irecv(ops_):
            wk.wait()
    return g


def gather_frames_(local: torch.Tensor, full: torch.Tensor, B: int, rows_local: int, world_size: int) -> torch.Tensor:
    """local [B * rows_local, X] (this rank's frames of every clip) -> full [B * world * rows_local, X] in frame order:
    one all-gather per clip (the K/V all-gather before each temporal-attention block)."""
    n = rows_local
    for b in range(B):
        dist.all_gather_into_tensor(full[b * n * world_size:(b + 1) * n * world_size], local[b * n:(b + 1) * n])
    return full
