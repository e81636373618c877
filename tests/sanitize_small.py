"""Smallest end-to-end exercise of every kernel, meant to run under compute-sanitizer (one tool per gpurun call):
    compute-sanitizer --tool memcheck python tests/sanitize_small.py
    compute-sanitizer --tool racecheck python tests/sanitize_small.py
"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from com_marl_b200.rollout import RolloutEngine, make_policy  # noqa: E402
from com_marl_b200.scenario import ScenarioSpec  # noqa: E402


def main():
    cases = [("pp", 10, 1, 0.04, 2, 0.3, 40, "auto", {"max_env_steps": 6}),        # lane groups of 4, tcgen05 policy, IID
             ("co", 10, 1, 0.03, 2, 0.0, 40, "auto", {"max_env_steps": 6}),        # Coverage
             ("pp", 20, 2, 0.08, 4, 0.2, 9, "auto", {"max_env_steps": 5}),         # n = 32: whole-warp groups
             ("pp", 30, 2, 0.08, 4, 0.0, 3, "auto", {"max_env_steps": 4}),         # n = 72: tc encoder -> attention kernel -> tc head
             ("pp", 50, 2, 0.08, 4, 0.0, 2, "auto", {"max_env_steps": 3})]         # n = 200: attention kernel with 13-row groups
    for scen, m, sen, den, cap, loss, B, math, over in cases:
        spec = ScenarioSpec.from_cli(scen, m, sen, den, cap=cap, loss=loss, seed=3, **over)
        pol = make_policy(spec, math=math)
        eng = RolloutEngine(spec, pol, B, ring=4, use_graph=False, record_attention=True)
        eng.reset()
        eng.run(12)
        torch.cuda.synchronize()
        eng.env.check_errors()
        pol.check_errors()
        assert np.isfinite(eng.traj["probs"].cpu().numpy()).all()
        print(scen, m, "n =", spec.n_agents, "episodes finished:", int(eng.local_stats()[0].item()))
    # Obs-DP policy (rows independent of the team) and env groups on separate streams inside a captured graph
    spec = ScenarioSpec.from_cli("co", 10, 1, 0.03, cap=2, loss=0.1, seed=3, max_env_steps=6)
    pol = make_policy(spec, kind="dec")
    eng = RolloutEngine(spec, pol, 50, ring=3, use_graph=True, groups=3)
    eng.reset()
    eng.run(9)
    torch.cuda.synchronize()
    eng.env.check_errors()
    pol.check_errors()
    print("obs-dp / env groups ok")
    # CENT policy: ragged last tile (70 envs = 64 + 6), K = n*D not a multiple of the 32-wide chunk, 2 output passes
    spec = ScenarioSpec.from_cli("pp", 20, 1, 0.05, cap=2, loss=0.0, seed=3, max_env_steps=6)
    pol = make_policy(spec, kind="cent")
    eng = RolloutEngine(spec, pol, 70, ring=3, use_graph=False, groups=2)
    eng.reset()
    eng.run(6)
    torch.cuda.synchronize()
    eng.env.check_errors()
    assert np.isfinite(eng.traj["probs"].cpu().numpy()).all()
    print("cent ok, n =", spec.n_agents)
    # Gilbert-Elliot channel + comm-only entry point + mask converters
    spec = ScenarioSpec.from_cli("pp", 10, 1, 0.08, cap=2, loss=0.2, channel_type="GE", max_env_steps=5)
    from com_marl_b200.envs import BatchedEnv
    env = BatchedEnv(spec, 17)
    env.reset()
    for _ in range(7):
        env.step(np.random.default_rng(0).integers(0, 5, size=(17, spec.n_agents)).astype(np.int8))
    env.comm_update()
    env.dist_adj(); env.channels()
    torch.cuda.synchronize()
    env.check_errors()
    # host-buffer calls (one C call = H2D + kernel + D2H, merged copies) and the PPO kernels
    spec = ScenarioSpec.from_cli("co", 10, 1, 0.03, cap=2, loss=0.1, seed=3, max_env_steps=6)
    pol = make_policy(spec)
    env = BatchedEnv(spec, 33)
    out = env.reset_host()
    for _ in range(8):
        acts, _ = pol.get_actions_host(out["pinned"]["obs"], out["pinned"]["adj_bits"], out["pinned"]["chan_bits"], return_pinned=True, inputs_arena=True)
        out = env.step_host(acts)
    env.check_errors()
    from com_marl_b200.ppo import ppo_advantages
    from com_marl_b200 import _native as N
    P, T = 11, 37
    r = torch.rand((P, T), dtype=torch.float64, device="cuda")
    b = torch.rand((P, T), device="cuda")
    v = torch.randint(1, T + 1, (P,), dtype=torch.int32, device="cuda")
    ret, raw, adv = ppo_advantages(r, b, v, 0.99, 0.97)
    assert torch.isfinite(adv).all() and torch.isfinite(ret).all()
    n = 1000
    p_, g_, m_, v_ = (torch.rand(n, device="cuda") for _ in range(4))
    N.check("cm_adam_step", N.lib().cm_adam_step(N.ptr(p_), N.ptr(g_), N.ptr(m_), N.ptr(v_), n, 3e-4, 0.9, 0.999, 1e-5, 1, 1.0, N.stream_ptr()))
    torch.cuda.synchronize()
    print("sanitize_small ok")


if __name__ == "__main__":
    main()
