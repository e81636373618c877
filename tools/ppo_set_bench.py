"""Training several policies in one batched run on one B200: a DeviceTrainerSet of K members against the same K members as K
standalone DeviceTrainers, round times alternated in one process after a warm-up round of each.

At the reference's batch size (bs = 60000 n / 8 agent-steps per epoch, SURVEY.md §3.2: about 38 envs x 200 steps at every team
size) a standalone round is launch-bound; E = 1024 envs per member shows where batching stops paying.  Member i of both arms
starts from the same weights (seed i) and rolls out global env ids i E .. (i + 1) E - 1, so their per-member AverageReturn of a
round must agree up to the last-bit differences of the update (printed for both).

Prints one JSON line per (config, E, K) with the card's name and power limit, read in the same run, and appends it to --out.

    python tools/ppo_set_bench.py [--config c1 c3] [--envs 38] [--members 1 4 16 64] [--rounds 2] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {"c1": ("pp", 10, 1, 0.04, 2, 0.0), "c3": ("pp", 20, 2, 0.08, 4, 0.2)}
TIMES = ("rollout_ms", "batch_ms", "update_ms")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                       timeout=30).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def spec_of(shape):
    from com_marl_b200.scenario import ScenarioSpec
    scen, m, sen, den, cap, loss = SHAPES[shape]
    return ScenarioSpec.from_cli(scen, m, sen, den, cap=cap, loss=loss, seed=7)


def run(shape, E, K, rounds):
    import numpy as np
    import torch
    from com_marl_b200.train import DeviceTrainer, DeviceTrainerSet
    seeds = list(range(1, K + 1))
    S = DeviceTrainerSet(spec_of(shape), E, seeds)
    singles = []
    for i, s in enumerate(seeds):
        t = DeviceTrainer(spec_of(shape), E, env_id0=i * E, seed=s)
        t.policy.load_state_dict(S.policies[i].state_dict())
        t.critic.load_state_dict(S.critics[i].state_dict())
        t.policy.refresh_weights(force=True)
        singles.append(t)
    set_rounds, single_rounds = [], []
    for r in range(rounds + 1):                # round 0: warm-up of both arms (graph capture, first launches)
        outs = S.train_epoch()
        sr = [t.train_epoch() for t in singles]
        if r == 0:
            ret_set = [o["tabular"]["AverageReturn"] for o in outs]
            ret_single = [o["tabular"]["AverageReturn"] for o in sr]
            continue
        set_rounds.append({k: outs[0][k] for k in TIMES})
        single_rounds.append({k: sum(o[k] for o in sr) for k in TIMES})
    med = lambda rs: {k: float(np.median([x[k] for x in rs])) for k in TIMES}  # noqa: E731
    a, b = med(set_rounds), med(single_rounds)
    tot_a, tot_b = sum(a.values()), sum(b.values())
    torch.cuda.synchronize()
    return dict(config=shape, envs_per_member=E, members=K, n_agents=S.spec.n_agents, rounds=rounds, set_ms=a, standalone_ms=b,
                set_round_ms=tot_a, standalone_round_ms=tot_b, speedup=tot_b / tot_a,
                round1_average_return_set=ret_set, round1_average_return_standalone=ret_single)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", nargs="+", default=["c1", "c3"], choices=sorted(SHAPES))
    ap.add_argument("--envs", type=int, default=38)
    ap.add_argument("--members", type=int, nargs="+", default=[1, 4, 16, 64])
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    card = gpu_info()
    for shape in a.config:
        for K in a.members:
            rec = dict(run(shape, a.envs, K, a.rounds), gpu=card)
            line = json.dumps(rec)
            print(line, flush=True)
            if a.out:
                with open(a.out, "a") as f:
                    f.write(line + "\n")


if __name__ == "__main__":
    main()
