"""Training and evaluation grids sharded by member over the GPUs of one box: DeviceTrainerSet(group=...) and
eval_policies(group=...) under torchrun, one process per GPU.

    torchrun --nproc-per-node W tools/grid_bench.py [--config c1 c3] [--members 64] [--envs 38] [--rounds 3]
                                                    [--eval-policies 32] [--out FILE]

One GPU per rank over NCCL (init_from_env).  With more ranks than visible GPUs the ranks share them round-robin over gloo
(NCCL takes one rank per GPU); such lines carry ranks_share_gpus = true and show that the sharded grid computes what one rank
computes, not how it scales.

Per config: a K-member grid (seeds 1 .. K, the set's own channel) of `--envs` envs per member, one warm-up round, then
`--rounds` timed rounds; a round is timed on the host from one barrier to the next after the gathered results are back, so
it is the slowest rank's round.  Then eval_policies of `--eval-policies` C3 policies x 100 greedy episodes x 200 steps (one
warm-up call, median of 3).  Each member's round-1 AverageReturn is printed and recorded: it does not depend on the number of
ranks (a member's random streams are keyed by its global env ids and seed), and neither does the digest of the evaluation's
results.  Rank 0 prints one JSON line per measurement, with the card's name and power limit read in the same run, and appends
it to --out.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {"c1": ("pp", 10, 1, 0.04, 2, 0.0), "c3": ("pp", 20, 2, 0.08, 4, 0.2)}
TIMES = ("rollout_ms", "batch_ms", "update_ms")


def gpu_info(index):
    q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def spec_of(shape):
    from com_marl_b200.scenario import ScenarioSpec
    scen, m, sen, den, cap, loss = SHAPES[shape]
    return ScenarioSpec.from_cli(scen, m, sen, den, cap=cap, loss=loss, seed=7)


def timed(fn):
    """fn() between two barriers, after a device synchronise: the slowest rank's wall time in s"""
    import torch
    import torch.distributed as dist
    if dist.is_initialized():
        dist.barrier()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    if dist.is_initialized():
        dist.barrier()
    return out, time.perf_counter() - t0


def train_grid(shape, E, K, rounds):
    import numpy as np
    from com_marl_b200.distributed import member_range
    from com_marl_b200.train import DeviceTrainerSet
    S = DeviceTrainerSet(spec_of(shape), E, list(range(1, K + 1)))
    walls, per_rank = [], []
    for r in range(rounds + 1):                # round 0: warm-up (graph capture, first launches)
        outs, wall = timed(S.train_epoch)
        if r == 0:
            ret = [o["tabular"]["AverageReturn"] for o in outs]
            continue
        walls.append(wall)
        first = {}                             # each rank's set times: those of its first member
        for o in outs:
            first.setdefault(o["rank"], {k: o[k] for k in TIMES})
        per_rank.append([first[q] for q in sorted(first)])
    med = float(np.median(walls))
    rank_ms = [{k: float(np.median([rnd[q][k] for rnd in per_rank])) for k in TIMES} for q in range(len(per_rank[0]))]
    return dict(kind="train", config=shape, members=K, envs_per_member=E, n_agents=S.spec.n_agents, rounds=rounds,
                round_s=med, round_s_all=walls, rank_set_ms=rank_ms, members_per_rank=[
                hi - lo for lo, hi in (member_range(K, q, S.world) for q in range(S.world))], round1_average_return=ret)


def value_digest(obj):
    """sha256 over the values of a nested result (structure, types, array dtypes / shapes / bytes, float bits)"""
    import numpy as np
    h = hashlib.sha256()

    def walk(x):
        h.update(type(x).__name__.encode())
        if isinstance(x, (list, tuple)):
            h.update(str(len(x)).encode())
            for y in x:
                walk(y)
        elif isinstance(x, dict):
            for k, y in x.items():
                walk(k)
                walk(y)
        elif isinstance(x, (np.ndarray, np.generic)):
            h.update(f"{x.dtype.str}{x.shape}".encode() + x.tobytes())
        elif isinstance(x, float):
            h.update(np.float64(x).tobytes())
        else:
            h.update(repr(x).encode())

    walk(obj)
    return h.hexdigest()


def eval_grid(P, episodes, steps, calls=3):
    import numpy as np
    from com_marl_b200.evaluate import eval_policies
    from com_marl_b200.rollout import make_policy
    spec = spec_of("c3")
    pols = [make_policy(spec, torch_seed=100 + i) for i in range(P)]
    run = lambda: eval_policies(spec, pols, n_eval_episodes=episodes, max_env_steps=steps)  # noqa: E731
    res, _ = timed(run)                        # warm-up
    walls = [timed(run)[1] for _ in range(calls)]
    digest = value_digest(res)
    mean_ret = [float(np.mean(r[0][2]["reward"])) for r in res]
    return dict(kind="eval_policies", config="c3", policies=P, episodes=episodes, max_env_steps=steps, calls=calls,
                call_s=float(np.median(walls)), call_s_all=walls, results_sha256=digest, mean_episode_return=mean_ret)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", nargs="+", default=["c1", "c3"], choices=sorted(SHAPES))
    ap.add_argument("--members", type=int, default=64)
    ap.add_argument("--envs", type=int, default=38)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--eval-policies", type=int, default=32)
    ap.add_argument("--eval-episodes", type=int, default=100)
    ap.add_argument("--eval-steps", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from com_marl_b200 import distributed as D
    n_gpus = torch.cuda.device_count()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # one GPU per rank over NCCL; more ranks than GPUs share them over gloo (NCCL takes one rank per GPU): that checks the
    # sharded results, not the scaling
    shared = world > n_gpus
    rank, local_rank, world = D.init_from_env(backend="gloo" if shared else None)
    gpu = local_rank % n_gpus
    torch.cuda.set_device(gpu)
    cards = D.gather_objects(gpu_info(gpu))
    common = dict(ranks=world, gpus=min(world, n_gpus), ranks_share_gpus=shared,
                  backend=("gloo" if shared else "nccl") if world > 1 else None,
                  gpu=cards[0], same_card_on_every_rank=len(set(cards)) == 1)

    def emit(rec):
        if rank == 0:
            line = json.dumps(dict(rec, **common))
            print(line, flush=True)
            if a.out:
                with open(a.out, "a") as f:
                    f.write(line + "\n")

    for shape in a.config:
        emit(train_grid(shape, a.envs, a.members, a.rounds))
    if a.eval_policies:
        emit(eval_grid(a.eval_policies, a.eval_episodes, a.eval_steps))
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
