"""Kernel times of the CENT family's wide-K layers in the PPO update (cm_ppo_net kinds CM_NET_POLICY_CENT / CM_NET_BASELINE_MLP):
net_wide_fwd (Y = act(X W1 + b1)) and net_wide_dw (dW1 += X^T dZ1; the <32, 1> instance is dW4 of the policy head), from
torch.profiler over one minibatch of a round at the given config (envs x horizon / minibatches env steps), with achieved TFLOP/s
from 2 S K N per product.
    python tools/ppo_cent_kernels.py --config c3 --envs 128 --minibatches 3
Prints ONE JSON line."""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c3")
    ap.add_argument("--envs", type=int, default=128)
    ap.add_argument("--minibatches", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    import bench
    from com_marl_b200.policy import CentralizedCategoricalMLPPolicy
    from com_marl_b200.ppo import DevicePPO, GaussianMLPBaseline
    from com_marl_b200.scenario import ScenarioSpec
    from com_marl_b200.spaces import Box, Discrete, EnvSpec
    scen, params = bench.params_for(args.config)
    spec = ScenarioSpec.from_params(scen, params, seed=1)
    n, D, T = spec.n_agents, spec.obs_dim, spec.max_steps
    P = max(1, args.envs // args.minibatches)
    S, K = P * T, n * D
    es = EnvSpec(Box(np.zeros(K), np.ones(K)), Discrete(5))
    torch.manual_seed(0)
    algo = DevicePPO(CentralizedCategoricalMLPPolicy(es, n), GaussianMLPBaseline(es, hidden_sizes=(64, 64, 64)), fused=True)
    F = algo._fused
    g = torch.Generator(device="cuda").manual_seed(0)
    b = dict(obs=torch.rand(P, T, K, device="cuda", generator=g), avail=torch.ones(P, T, n * 5, device="cuda"),
             actions=torch.randint(0, 5, (P, T, n), device="cuda", generator=g), rewards=torch.rand(P, T, device="cuda", generator=g).double(),
             valids=torch.full((P,), T, dtype=torch.int32, device="cuda"))
    b = algo.finish_batch(b)
    f = b["_flat"]
    adv, ret = b["adv"].reshape(-1), b["returns"].reshape(-1)
    F.pol_map.refresh()
    F.cri_map.refresh()

    def step():
        F.critic_call(f, None, returns=ret, backward=True)
        F.policy_call(f, None, adv=adv, backward=True, inv_count=1.0 / S)

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(args.reps):
            step()
        torch.cuda.synchronize()
    # products per call: name fragment -> (K, N)
    shapes = {"net_wide_fwd_kernel<2": (K, 128), "net_wide_fwd_kernel<1": (K, 64), "net_wide_dw_kernel<128": (K, 128),
              "net_wide_dw_kernel<64": (K, 64), "net_wide_dw_kernel<32": (5 * n, 32)}
    kern = {}
    total_us = 0.0
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        total_us += t
        for frag, (k, nn) in shapes.items():
            if frag.replace("<", "") in e.key.replace("<", "").replace("cm::", "") or frag in e.key:
                per = t / args.reps
                flops = 2.0 * S * k * nn
                kern[e.key[:60]] = dict(us_per_call=per, K=k, N=nn, S=S, tflops=flops / (per * 1e-6) / 1e12)
    print(json.dumps(dict(config=args.config, envs=args.envs, n_agents=n, obs_dim=D, K=K, steps_per_minibatch=S,
                          gpu=torch.cuda.get_device_name(), kernels=kern, all_kernels_us_per_step=total_us / args.reps)), flush=True)


if __name__ == "__main__":
    main()
