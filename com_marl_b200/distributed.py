"""Multi-GPU plumbing: one process per GPU, envs sharded contiguously, no data-path collective.

Env instances are independent (SURVEY.md §8e), so each rank steps its own slice; the RNG streams are keyed
by GLOBAL env id, which makes results independent of the sharding.  The only exchange is the all-gather of
the per-rank episode-statistics vector once per obtain_samples (NCCL over NVLink on GPUs; gloo in the CPU
tests) — a few dozen bytes, latency bound.  Grids of runs (DeviceTrainerSet, eval_policies) shard whole members the same
way (member_range) and gather their results once per round (gather_objects).
"""
import hashlib
import os
from typing import Dict, List, Tuple

import torch
import torch.distributed as dist

from .rollout import STAT_KEYS


def shard_range(n_envs_total: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous slice [lo, hi) of the global env ids owned by `rank`; sizes differ by at most one."""
    base, rem = divmod(int(n_envs_total), int(world))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def member_range(n_members: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous global member ids [lo, hi) of a training or evaluation grid that `rank` owns (shard_range's rule: sizes
    differ by at most one).  A member's random streams are keyed by its global env ids, seed and condition, so it computes
    the same thing whichever rank runs it."""
    return shard_range(n_members, rank, world)


def group_rank_world(group=None) -> Tuple[int, int]:
    """(rank, world) of this process in `group` (the default group when None); (0, 1) without torch.distributed"""
    if not (dist.is_available() and dist.is_initialized()):
        return 0, 1
    return dist.get_rank(group), dist.get_world_size(group)


def gather_objects(obj, group=None) -> List:
    """all-gather of one picklable object per rank -> [object of rank 0, object of rank 1, ...] on every rank
    (dist.all_gather_object; under NCCL the current device must be the rank's GPU, which init_from_env sets).  [obj]
    without a process group or with a group of one rank."""
    rank, world = group_rank_world(group)
    if world == 1:
        return [obj]
    out = [None] * world
    dist.all_gather_object(out, obj, group=group)
    return out


def rank_alone_group():
    """A process group holding this rank alone: what a rank's own members hand to the collectives of DevicePPO (its
    global_max / gradient all-reduce) so that they stay on this rank when a process group of several ranks exists.  Only
    this rank takes part in creating it."""
    return dist.new_group([dist.get_rank()], use_local_synchronization=True)


def check_same_on_all_ranks(what: str, value, group=None) -> None:
    """ValueError on EVERY rank when `value` (its repr, hashed) differs between the ranks of `group`: one gather of a digest,
    so that a rank given other arguments fails together with the others instead of leaving them waiting in a collective"""
    digest = hashlib.sha256(repr(value).encode()).hexdigest()
    got = gather_objects(digest, group)
    bad = [r for r, d in enumerate(got) if d != got[0]]
    if bad:
        raise ValueError(f"{what} differ between the ranks: rank(s) {bad} disagree with rank 0")


def init_from_env(backend: str = None) -> Tuple[int, int, int]:
    """(rank, local_rank, world) from torchrun's environment; initialises the default process group when
    WORLD_SIZE > 1.  Single-process runs need no process group."""
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29500")
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(local_rank)
        dist.init_process_group(backend=backend, rank=rank, world_size=world)
    return rank, local_rank, world


def gather_stats(local: torch.Tensor, group=None) -> torch.Tensor:
    """all-gather of the per-rank float64 [len(STAT_KEYS)] sums -> [world, len(STAT_KEYS)]"""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return local.reshape(1, -1).clone()
    world = dist.get_world_size(group)
    out = torch.empty((world, local.numel()), dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(out, local.contiguous().reshape(1, -1), group=group)
    return out


def summarize_stats(per_rank: torch.Tensor, scenario: str, n_agents: int) -> Dict[str, float]:
    """The per-epoch tabular keys the reference logs from `paths` (centralized_ma_ppo.py:345-372), from the
    whole-job sums: AverageReturn, SuccessRate, AverageStepCount and the per-episode count means."""
    tot = per_rank.sum(dim=0).double().cpu()
    s = dict(zip(STAT_KEYS, tot.tolist()))
    ep = max(s["episodes"], 1.0)
    n = float(n_agents)
    out = dict(NumEpisodes=s["episodes"], AverageReturn=s["return_sum"] / ep, SuccessRate=s["success_sum"] / ep,
               AverageStepCount=s["length_sum"] / ep)
    if scenario == "pp":      # capture / penalty are counts, moved / watching are per-step means over agents
        out.update(AverageCaptureCount=s["c0_sum"] / ep, AverageMovingCount=s["moved_sum"] / n / ep,
                   AveragePenaltyCount=s["c2_sum"] / ep, AverageVariable=s["c3_sum"] / n / ep, AverageVar2=0.0)
    else:                     # every Coverage detail is a per-step mean over agents
        out.update(AverageCaptureCount=s["c0_sum"] / n / ep, AverageMovingCount=s["moved_sum"] / n / ep,
                   AveragePenaltyCount=s["c2_sum"] / n / ep, AverageVariable=s["c3_sum"] / n / ep,
                   AverageVar2=s["c4_sum"] / n / ep)
    return out


def allreduce_gradients(module: torch.nn.Module, group=None) -> int:
    """Data-parallel gradient averaging for the PPO update of BASELINE config 5 (SURVEY.md §8e-2): ONE all-reduce over
    a flattened fp32 bucket of every parameter gradient (policy 46 405 + critic ~32 k floats = ~313 KB, latency bound on
    NVLink), then divide by the world size.  Returns the number of floats reduced.  A no-op without a process group.
    The reference computes `loss.backward()` in a single process (centralized_ma_ppo.py:243,251); with envs sharded
    over GPUs each rank back-propagates its own slice and calls this before `optimizer.step()`."""
    grads = [p.grad for p in module.parameters() if p.grad is not None]
    if not grads:
        return 0
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return sum(g.numel() for g in grads)
    flat = torch.cat([g.reshape(-1).float() for g in grads])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    flat /= dist.get_world_size(group)
    off = 0
    for g in grads:
        g.copy_(flat[off:off + g.numel()].view_as(g))
        off += g.numel()
    return off


def bind_to_gpu_numa(gpu_index: int) -> str:
    """Pin this process (and the pinned host arenas it allocates afterwards: first touch) to the CPU cores NVML reports as
    local to the GPU, so that a rank's host <-> device traffic stays on its own socket / memory controller when several
    ranks share a box.  Returns a short description; a no-op when NVML or the affinity call is unavailable."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(int(gpu_index))
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cores = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        allowed = cores & set(os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return f"cpus {min(allowed)}-{max(allowed)} ({len(allowed)} cores local to GPU {gpu_index})"
        return "NVML affinity mask does not intersect the allowed cores: left unchanged"
    except Exception as e:                       # NVML absent, container without the permission, ...
        return f"unchanged ({type(e).__name__})"
