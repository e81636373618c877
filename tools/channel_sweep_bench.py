"""Per-env channel conditions on one B200: what a sweep over channel conditions gains, and what the table instantiation
of env_kernel costs.

  sweep   A 90-condition grid at C3 (Predator-Prey map 20, sen 2, den 0.08, cap 4): Ploss in {0, 0.1, ..., 0.9} x Rcom in
          {1, ..., 9} (none collapses at map 20), 100 greedy episodes of 200 steps each, Comm-DP policy.  Wall time of ONE
          eval_sweep against the same conditions as sequential eval_model calls (env_id0 = k * 100, so the outputs must be
          identical, and are compared).
  kernel  env_kernel at C3, IID, 8192 envs per launch: the table instantiation with a one-entry table against the
          uniform IID instantiation, ms per launch (CUDA events), the two alternated in one process.

Prints one JSON line per part, with the card's name and power limit.

    python tools/channel_sweep_bench.py [--part sweep|kernel|all] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return q
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def c3(**over):
    from com_marl_b200.scenario import ScenarioSpec
    return ScenarioSpec.from_cli("pp", 20, 2, 0.08, cap=4, loss=0.2, **over)


def same(a, b):
    import numpy as np
    if isinstance(a, dict):
        return a.keys() == b.keys() and all(same(a[k], b[k]) for k in a)
    if isinstance(a, (list, tuple)):
        return len(a) == len(b) and all(same(x, y) for x, y in zip(a, b))
    if isinstance(a, np.ndarray):
        return np.array_equal(a, b)
    return a == b


def part_sweep(args):
    import torch
    from com_marl_b200.evaluate import eval_model, eval_sweep
    from com_marl_b200.rollout import make_policy
    spec = c3()
    conds = [spec.with_channel(pl=pl / 10, rcom=r) for pl in range(10) for r in range(1, 10)]
    assert all(c.rcom != 0 for c in conds)
    pol = make_policy(spec)
    E, T = args.episodes, args.max_env_steps
    kw = dict(n_eval_episodes=E, max_env_steps=T, eval_greedy=True, seed=1)
    eval_model(conds[0], pol, **kw)                                    # module loads, library caches
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    sweep = eval_sweep(spec, pol, conds, **kw)
    torch.cuda.synchronize()
    t_sweep = time.perf_counter() - t0
    t0 = time.perf_counter()
    seq = [eval_model(c, pol, env_id0=k * E, **kw) for k, c in enumerate(conds)]
    torch.cuda.synchronize()
    t_seq = time.perf_counter() - t0
    return dict(part="sweep", conditions=len(conds), episodes=E, max_env_steps=T, eval_sweep_s=round(t_sweep, 3),
                sequential_eval_model_s=round(t_seq, 3), speedup=round(t_seq / t_sweep, 2), identical=same(sweep, seq))


def part_kernel(args):
    import numpy as np
    import torch
    from com_marl_b200.envs import BatchedEnv
    spec = c3()
    B = args.envs
    uni = BatchedEnv(spec, B)
    tab = BatchedEnv(spec, B, conditions=[spec])
    acts = torch.from_numpy(np.random.default_rng(0).integers(0, 5, (B, spec.n_agents), dtype=np.int8)).cuda()
    for e in (uni, tab):
        e.reset()
        for _ in range(20):
            e.step(acts)
    torch.cuda.synchronize()
    ms = {"uniform_iid": [], "table_1_entry": []}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):
        for name, e in (("uniform_iid", uni), ("table_1_entry", tab)):
            ev0.record()
            for _ in range(args.launches):
                e.step(acts)
            ev1.record()
            ev1.synchronize()
            ms[name].append(ev0.elapsed_time(ev1) / args.launches)
    uni.check_errors()
    tab.check_errors()
    # the two kernels compute the same thing: compare the state they reached from the same start and actions
    same_state = all(torch.equal(getattr(uni, k), getattr(tab, k)) for k in ("agent_pos", "prey_pos", "obs", "chan_bits", "adj_bits"))
    med = {k: float(np.median(v)) for k, v in ms.items()}
    return dict(part="kernel", envs=B, launches_per_round=args.launches, rounds=args.rounds,
                ms_per_launch_median=med, ms_per_launch_all={k: [round(x, 5) for x in v] for k, v in ms.items()},
                table_over_uniform=round(med["table_1_entry"] / med["uniform_iid"], 4), identical=same_state)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--part", default="all", choices=["sweep", "kernel", "all"])
    ap.add_argument("--episodes", type=int, default=100)
    ap.add_argument("--max-env-steps", type=int, default=200)
    ap.add_argument("--envs", type=int, default=8192)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--out", help="also append the JSON lines to this file")
    args = ap.parse_args()
    gpu = gpu_info()
    parts = ["kernel", "sweep"] if args.part == "all" else [args.part]
    for p in parts:
        rec = dict({"sweep": part_sweep, "kernel": part_kernel}[p](args), gpu=gpu)
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
