"""Frame-index partition and the single counter exchange of the multi-GPU path (SURVEY.md section 8e).

Frames are indexed f = (snr_idx*C + chan_idx)*ensemble + e (the reference's loop nest, snr outermost,
python/ofdm_utils/wofdm_simulation.py:171-177).  Rank r of W takes f = r (mod W); the device draws depend only
on the GLOBAL frame id, so the job's counters do not depend on W.  The only exchange is one sum all-reduce of
the int64 counters.  Pure host logic: importable and testable without a GPU (gloo).
"""
from __future__ import annotations

import numpy as np


def shard_count(total: int, rank: int, world: int) -> int:
    """#{f < total : f = rank (mod world)}"""
    return (total - rank + world - 1) // world if total > rank else 0


def frames_per_snr(n_snr: int, C: int, ensemble: int, shard=(0, 1)) -> np.ndarray:
    """Frames of each SNR point that fall into `shard` (mirrors wofdm_ber_run_shard's totals)."""
    r, w = shard
    per = C * int(ensemble)
    return np.array([shard_count((k + 1) * per, r, w) - shard_count(k * per, r, w) for k in range(n_snr)],
                    dtype=np.int64)


def totals(n_snr, C, ensemble, N, S, bits, shard=(0, 1)):
    """(bit_tot, sym_tot) per SNR point: frames * N*(S-1) symbols, times bits."""
    sym = frames_per_snr(n_snr, C, ensemble, shard) * N * (S - 1)
    return sym * bits, sym


def frame_ids(n_snr: int, C: int, ensemble: int, shard=(0, 1)) -> np.ndarray:
    r, w = shard
    return np.arange(r, n_snr * C * int(ensemble), w, dtype=np.int64)


def decode(f, C: int, ensemble: int):
    """global frame id -> (snr_idx, chan_idx, e)"""
    f = np.asarray(f, dtype=np.int64)
    return f // (C * ensemble), (f // ensemble) % C, f % ensemble


def allreduce_counters(counters, group=None):
    """Sum int64 counters over the process group (NCCL on GPUs, gloo on CPU).  No-op when not initialised."""
    import torch
    import torch.distributed as dist
    t = counters if isinstance(counters, torch.Tensor) else torch.as_tensor(np.asarray(counters, dtype=np.int64))
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        if dist.get_backend(group) == "nccl" and not t.is_cuda:      # NCCL reduces device tensors only
            t = t.cuda()
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t


def adaptive_allreduce(group=None):
    """reduce callable of Handle.ber_run_adaptive under torch.distributed: sums a round's int64 counts over `group` with
    allreduce_counters (one all-reduce per round).  Every rank then computes the same schedule; each passes its own shard."""
    def reduce(counts):
        return allreduce_counters(np.array(counts, dtype=np.int64), group=group)
    return reduce


def segment_frame_ids(segments, C: int, ensemble_max: int, shard=(0, 1), contiguous=False) -> np.ndarray:
    """Global frame ids of a segment list {snr_idx, e_begin, e_count} in launch order (wofdm_ber_run_segments): segments in
    the order given, channel-major then e inside a segment; `shard` keeps local indices j = shard[0] (mod shard[1]), or with
    contiguous=True the channel-mask chain's block [floor(n*k/W), floor(n*(k+1)/W)) of the n local indices
    (wofdm_ber_run_masked_segments)."""
    seg = np.asarray(segments, dtype=np.int64).reshape(-1, 3)
    parts = []
    for si, e0, ec in seg:
        c, e = np.divmod(np.arange(int(C) * int(ec), dtype=np.int64), int(ec))
        parts.append((si * C + c) * int(ensemble_max) + e0 + e)
    f = np.concatenate(parts) if parts else np.zeros(0, dtype=np.int64)
    if contiguous:
        k, w = int(shard[0]), int(shard[1])
        return f[f.size * k // w: f.size * (k + 1) // w]
    return f[shard[0]::shard[1]]


# ---- interference power: channel realisations are independent, rank r takes a contiguous block (SURVEY 8e) ----------

def channel_block(C: int, rank: int, world: int):
    """[lo, hi) of the channel realisations rank `rank` evaluates: contiguous blocks, sizes differing by at most one."""
    base, extra = divmod(int(C), int(world))
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def allgather_channel_rows(P_local, C: int, group=None):
    """Per-channel results of every rank, (C_rank, ...) rows in channel order -> (C, ...) on every rank: one
    all-gather of the padded blocks (NCCL on GPUs, gloo on CPU).  Returns P_local unchanged outside a process group."""
    import torch
    import torch.distributed as dist
    t = P_local if isinstance(P_local, torch.Tensor) else torch.as_tensor(np.asarray(P_local, dtype=np.float64))
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return t
    if dist.get_backend(group) == "nccl" and not t.is_cuda:
        t = t.cuda()
    world = dist.get_world_size(group)
    rows = max(channel_block(C, r, world)[1] - channel_block(C, r, world)[0] for r in range(world))
    pad = torch.zeros((rows,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    pad[: t.shape[0]] = t
    parts = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(parts, pad, group=group)
    return torch.cat([parts[r][: channel_block(C, r, world)[1] - channel_block(C, r, world)[0]] for r in range(world)])
