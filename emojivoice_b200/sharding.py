"""Multi-GPU partition of the synthesis path: utterances shard by batch, no collective on the data path.

SURVEY.md 8e / BASELINE.json north_star: a global utterance list is sorted by text length, cut into micro-batches of a
fixed size (bounded padding; the decoder result depends on batch composition -- SURVEY H1 -- so the micro-batch list
*is part of the input* and is the same list the oracle is run on), and the micro-batches are dealt to the ranks by
estimated work.  Each rank synthesises whole utterances and keeps its own waveforms; the only communication is an
optional reporting reduction of a few scalars.  Everything here is host logic (pure python / torch CPU tensors) and
runs unchanged under the `gloo` backend in the CPU test-suite.
"""
from __future__ import annotations

import numbers
from dataclasses import dataclass, field

SR, HOP = 22050, 256


def estimate_flops(tx: int, frames: int, n_timesteps: int) -> float:
    """Algorithmic FLOPs of one utterance (SURVEY.md 8d): encoder + n x estimator + HiFi-GAN."""
    return tx * (19_309_056 + 6_144 * tx) + n_timesteps * frames * (11_116_544 + 1_536 * frames) + frames * 614_105_088


@dataclass
class MicroBatch:
    index: int                      # position in the global micro-batch list
    items: list                     # indices into the caller's utterance list, in batch order
    tx_max: int                     # padded text length of the batch
    cost: float = 0.0               # estimated FLOPs (padding included: the batch computes on its padded extent)
    rank: int = -1


def microbatches(x_lengths, batch_size: int, n_timesteps=10, frames_per_token: float = 2.9, sort: bool = True):
    """Cut the utterance list into micro-batches of `batch_size` (the last one may be smaller).

    sort=True orders utterances by text length first (stable), which bounds padding; sort=False keeps the caller's
    order (what `matcha/cli.py:281-286`'s DataLoader does).  `frames_per_token` only feeds the cost estimate.
    n_timesteps: the Euler steps of every utterance, or a sequence with each utterance's own count (indexed like
    x_lengths); the cost of a batch sums each utterance's estimate at its own count.  The plan itself does not depend on it."""
    lens = [int(v) for v in x_lengths]
    if batch_size <= 0:
        raise ValueError("batch_size must be positive")
    per_item = not isinstance(n_timesteps, numbers.Number)
    if per_item and len(n_timesteps) != len(lens):
        raise ValueError("n_timesteps: one step count per utterance expected")
    order = sorted(range(len(lens)), key=lambda i: lens[i]) if sort else list(range(len(lens)))
    out = []
    for k in range(0, len(order), batch_size):
        items = order[k:k + batch_size]
        tx_max = max(lens[i] for i in items)
        frames = int(round(tx_max * frames_per_token))
        cost = (sum(estimate_flops(tx_max, frames, int(n_timesteps[i])) for i in items) if per_item
                else len(items) * estimate_flops(tx_max, frames, n_timesteps))
        out.append(MicroBatch(index=len(out), items=items, tx_max=tx_max, cost=cost))
    return out


def assign(batches, world_size: int):
    """Deal micro-batches to ranks: largest first onto the least loaded rank (LPT), ties to the lowest rank.
    Deterministic, so every rank derives the same plan from the same list without talking to the others.
    -> list (per rank) of micro-batch lists, each in global index order."""
    if world_size <= 0:
        raise ValueError("world_size must be positive")
    load = [0.0] * world_size
    per_rank = [[] for _ in range(world_size)]
    for mb in sorted(batches, key=lambda m: (-m.cost, m.index)):
        r = min(range(world_size), key=lambda i: (load[i], i))
        mb.rank = r
        load[r] += mb.cost
        per_rank[r].append(mb)
    for lst in per_rank:
        lst.sort(key=lambda m: m.index)
    return per_rank


def shard(x_lengths, batch_size: int, rank: int, world_size: int, **kw):
    """The micro-batches rank `rank` of `world_size` synthesises."""
    if not 0 <= rank < world_size:
        raise ValueError("rank out of range")
    return assign(microbatches(x_lengths, batch_size, **kw), world_size)[rank]


@dataclass
class ShardStats:
    utterances: int = 0
    audio_seconds: float = 0.0
    frames: int = 0
    flops: float = 0.0
    seconds: float = 0.0            # this rank's device time
    extra: dict = field(default_factory=dict)

    def add(self, mel_lengths, tx_lengths, n_timesteps, seconds):
        """n_timesteps: the step count of every utterance, or a sequence with each one's own."""
        steps = [n_timesteps] * len(tx_lengths) if isinstance(n_timesteps, numbers.Number) else list(n_timesteps)
        for t, f, n in zip(tx_lengths, mel_lengths, steps):
            self.utterances += 1
            self.frames += int(f)
            self.audio_seconds += int(f) * HOP / SR
            self.flops += estimate_flops(int(t), int(f), int(n))
        self.seconds += float(seconds)


def reduce_stats(stats: ShardStats, group=None):
    """Whole-job totals: sums over ranks, and the slowest rank's time (the job is done when the last rank is).
    Reporting only -- a handful of scalars; works on `gloo` (CPU tensors) and `nccl` (pass device=...)."""
    import torch
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return dict(utterances=stats.utterances, audio_seconds=stats.audio_seconds, frames=stats.frames, flops=stats.flops,
                    seconds=stats.seconds, world_size=1)
    dev = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
    sums = torch.tensor([stats.utterances, stats.audio_seconds, stats.frames, stats.flops], dtype=torch.float64, device=dev)
    tmax = torch.tensor([stats.seconds], dtype=torch.float64, device=dev)
    dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
    dist.all_reduce(tmax, op=dist.ReduceOp.MAX, group=group)
    return dict(utterances=int(sums[0]), audio_seconds=float(sums[1]), frames=int(sums[2]), flops=float(sums[3]),
                seconds=float(tmax[0]), world_size=dist.get_world_size(group))
