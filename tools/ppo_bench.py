"""Rollout + PPO update rounds on N GPUs (torchrun) or one: per-round times and learning statistics.
    python tools/ppo_bench.py --config c1 --envs 2048 --epochs 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 tools/ppo_bench.py ...
Prints ONE JSON line (rank 0)."""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c1")
    ap.add_argument("--envs", type=int, default=1024, help="envs per GPU")
    ap.add_argument("--epochs", type=int, default=3)
    ap.add_argument("--mini-epochs", type=int, default=10)
    ap.add_argument("--minibatches", type=int, default=3)
    ap.add_argument("--kind", default="comm", choices=["comm", "dec", "cent"], help="runner family (DeviceTrainer kind)")
    ap.add_argument("--fused", default="auto", choices=["auto", "0", "1"], help="hand-written update kernels (cm_ppo_net) or torch autograd")
    args = ap.parse_args()
    import bench
    from com_marl_b200 import distributed as D
    from com_marl_b200.scenario import ScenarioSpec
    from com_marl_b200.train import DeviceTrainer
    rank, local_rank, world = D.init_from_env()
    torch.cuda.set_device(local_rank)
    scen, params = bench.params_for(args.config)
    spec = ScenarioSpec.from_params(scen, params, seed=1)
    tr = DeviceTrainer(spec, args.envs, device=torch.device("cuda", local_rank), env_id0=rank * args.envs, kind=args.kind,
                       optimization_mini_epochs=args.mini_epochs, optimization_n_minibatches=args.minibatches,
                       fused={"auto": "auto", "0": False, "1": True}[args.fused])
    rounds = []
    for _ in range(args.epochs):
        t0 = time.time()
        out = tr.train_epoch()
        out["wall_s"] = time.time() - t0
        rounds.append(out)
    cs = torch.tensor([tr.weights_checksum()], dtype=torch.float64, device=torch.device("cuda", local_rank))
    if world > 1:
        lst = [torch.zeros_like(cs) for _ in range(world)]
        dist.all_gather(lst, cs)
        sums = [float(x) for x in lst]
    else:
        sums = [float(cs)]
    if rank == 0:
        last = rounds[-1]
        line = dict(config=args.config, kind=args.kind, n_gpus=world, envs_per_gpu=args.envs, n_agents=spec.n_agents, horizon=spec.max_steps,
                    mini_epochs=args.mini_epochs, minibatches=args.minibatches, fused=tr.algo._fused is not None, optimizer_steps_per_round=len(last["losses"]),
                    rounds=[dict(rollout_ms=r["rollout_ms"], batch_ms=r["batch_ms"], update_ms=r["update_ms"], n_paths=r["n_paths"],
                                 loss_before=r["loss_before"], loss_after=r["loss_after"], kl=r["kl"], entropy=r["entropy"],
                                 grad_norm_mean=sum(r["grad_norms"]) / max(1, len(r["grad_norms"])),
                                 average_return=r["episode_stats"].get("AverageReturn")) for r in rounds],
                    agent_steps_per_round=last["agent_steps"] * world,
                    agent_steps_per_s_incl_update=last["agent_steps"] * world / (1e-3 * (last["rollout_ms"] + last["batch_ms"] + last["update_ms"])),
                    weights_checksum_per_rank=sums, ranks_agree=max(sums) - min(sums) == 0.0)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
