"""Several policies in one launch on one B200: what evaluating many policies in one engine gains.

  eval    32 Comm-DP policies (8 at C5) x 100 greedy episodes x 200 steps at a bench shape as ONE eval_policies, against
          sequential eval_model calls (env_id0 = i * 100: the outputs must be identical, and are compared).  C1, C3 and C5.
  sweep   8 policies x a 12-condition grid (Ploss x Rcom) at C3: one eval_policies against 8 sequential sweeps (eval_sweep's
          loop with env_id0 = i * 12 * 100, so that every policy's outputs must be identical, and are compared).
  kernel  cm_policy_forward at C3: one PolicySet launch over P blocks against P single-policy launches of the same blocks,
          both captured in one CUDA graph and replayed, ms per replay (CUDA events), alternated in one process.

Prints one JSON line per measurement, each with the card's name and power limit, and appends them to --out
(profiles/r03c_policy_set.jsonl by default).

    python tools/policy_set_bench.py [--part eval|sweep|kernel|all] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from channel_sweep_bench import same  # noqa: E402

# bench.py's configurations (scenario, map, sen, den, cap, loss) and the policies evaluated at each: C5 (200 agents) with 8
SHAPES = {"c1": ("pp", 10, 1, 0.04, 2, 0.0), "c3": ("pp", 20, 2, 0.08, 4, 0.2), "c5": ("pp", 50, 2, 0.08, 4, 0.0)}
POLICIES = {"c1": 32, "c3": 32, "c5": 8}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def spec_of(shape, **over):
    from com_marl_b200.scenario import ScenarioSpec
    scen, m, sen, den, cap, loss = SHAPES[shape]
    return ScenarioSpec.from_cli(scen, m, sen, den, cap=cap, loss=loss, **over)


def timed(fn):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


def part_eval(args, emit):
    from com_marl_b200.evaluate import eval_model, eval_policies
    from com_marl_b200.rollout import make_policy
    for shape in args.shapes:
        spec = spec_of(shape)
        P, E, T = POLICIES[shape], args.episodes, args.max_env_steps
        pols = [make_policy(spec, torch_seed=1 + i) for i in range(P)]
        kw = dict(n_eval_episodes=E, max_env_steps=T, eval_greedy=True, seed=1)
        eval_policies(spec, pols[:2], **dict(kw, n_eval_episodes=4, max_env_steps=8))      # warm-up: library caches, allocator
        eval_model(spec, pols[0], **dict(kw, n_eval_episodes=4, max_env_steps=8))
        one, t_one = timed(lambda: eval_policies(spec, pols, **kw))
        seq, t_seq = timed(lambda: [eval_model(spec, p, env_id0=i * E, **kw) for i, p in enumerate(pols)])
        emit(dict(part="eval", shape=shape, n_agents=spec.n_agents, policies=P, episodes=E, steps=T, eval_policies_s=round(t_one, 3),
                  sequential_eval_model_s=round(t_seq, 3), speedup=round(t_seq / t_one, 2),
                  identical=all(same(list(one[i][0]), list(seq[i])) for i in range(P))))


def part_sweep(args, emit):
    from com_marl_b200.evaluate import _eval_spec, _evaluate, eval_policies, eval_sweep
    from com_marl_b200.rollout import make_policy
    spec = spec_of("c3")
    conds = [spec.with_channel(pl=pl, rcom=r) for pl in (0.0, 0.2, 0.4, 0.6) for r in (1, 3, 5)]
    P, E, T = 8, args.episodes, args.max_env_steps
    pols = [make_policy(spec, torch_seed=1 + i) for i in range(P)]
    kw = dict(n_eval_episodes=E, max_env_steps=T, eval_greedy=True, seed=1)
    eval_policies(spec, pols[:2], conditions=conds[:2], **dict(kw, n_eval_episodes=4, max_env_steps=8))
    eval_sweep(spec, pols[0], conds[:2], **dict(kw, n_eval_episodes=4, max_env_steps=8))
    one, t_one = timed(lambda: eval_policies(spec, pols, conditions=conds, **kw))
    # eval_sweep's loop (_evaluate) with policy i's envs keyed from (i C) E, the ids eval_policies gives them
    s1, c1 = _eval_spec(spec, 1), [_eval_spec(c, 1) for c in conds]
    seq, t_seq = timed(lambda: [_evaluate(s1, c1, p, E, T, True, 4, 50, False, i * len(conds) * E) for i, p in enumerate(pols)])
    emit(dict(part="sweep", shape="c3", policies=P, conditions=len(conds), episodes=E, steps=T, eval_policies_s=round(t_one, 3),
              sequential_eval_sweep_s=round(t_seq, 3), speedup=round(t_seq / t_one, 2),
              identical=all(same([list(r) for r in one[i]], [list(r) for r in seq[i]]) for i in range(P))))


def part_kernel(args, emit):
    import torch
    from com_marl_b200.envs import BatchedEnv
    from com_marl_b200.policy import PolicySet
    from com_marl_b200.rollout import make_policy
    spec = spec_of("c3")
    n = spec.n_agents
    for P, Ep in ((32, 100), (8, 1024)):
        pols = [make_policy(spec, torch_seed=1 + i) for i in range(P)]
        pset = PolicySet(pols)
        B = P * Ep
        env = BatchedEnv(spec, B)
        env.reset()
        outs = [dict(probs=torch.empty((B, n, 5), device="cuda"), actions=torch.empty((B, n), dtype=torch.int8, device="cuda"))
                for _ in range(2)]
        kw = lambda o, sl: dict(adj_bits=env.adj_bits[sl], chan_bits=env.chan_bits[sl], tick=env.tick[sl], episode=env.episode[sl],  # noqa: E731
                                greedy=False, probs=o["probs"][sl], actions=o["actions"][sl])

        def one():
            pset.act_device(env.obs, **kw(outs[0], slice(None)))

        def blocks():
            for i, p in enumerate(pols):
                sl = slice(i * Ep, (i + 1) * Ep)
                p.act_device(env.obs[sl], env_id0=i * Ep, **kw(outs[1], sl))
        graphs = []
        for fn in (one, blocks):
            fn()
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for _ in range(args.reps):
                    fn()
            graphs.append(g)
        times = [[], []]
        for _ in range(args.rounds):
            for j, g in enumerate(graphs):
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                g.replay()
                e.record()
                e.synchronize()
                times[j].append(s.elapsed_time(e) / args.reps)
        med = [sorted(t)[len(t) // 2] for t in times]
        emit(dict(part="kernel", shape="c3", policies=P, envs_per_policy=Ep, set_launch_ms=round(med[0], 4),
                  block_launches_ms=round(med[1], 4), speedup=round(med[1] / med[0], 2),
                  identical=all(torch.equal(outs[0][k], outs[1][k]) for k in outs[0])))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--part", default="all", choices=("eval", "sweep", "kernel", "all"))
    ap.add_argument("--shapes", nargs="+", default=["c1", "c3", "c5"])
    ap.add_argument("--episodes", type=int, default=100)
    ap.add_argument("--max-env-steps", type=int, default=200)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=15)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03c_policy_set.jsonl"))
    args = ap.parse_args()
    gpu = gpu_info()

    def emit(rec):
        rec["gpu"] = gpu
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")
    for part, fn in (("eval", part_eval), ("sweep", part_sweep), ("kernel", part_kernel)):
        if args.part in (part, "all"):
            fn(args, emit)


if __name__ == "__main__":
    main()
