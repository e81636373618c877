"""Batched evaluation driver: the reference's eval loop with every episode running in parallel on the device.

Replaces ``eval_model`` of exp_runners/predatorprey/eval_pp.py:9-104 / exp_runners/coverage/eval_co.py (same loop): the
reference plays ``n_eval_episodes`` episodes one after another — reset, then up to ``max_env_steps`` greedy policy calls
and env steps, recording per step the reward details (``VECTORS`` of exp_runners/testing.py:209; ``nodeDeg`` is
``env.ave_deg`` after the step) and ``env.success`` — and returns ``(episode_data, epi_success, epi_rewards,
bound_return)`` for the CSV / MATLAB writers of testing.py:213-367.  Here the episodes are ``n_eval_episodes``
independent envs of one RolloutEngine (no auto-reset: an env that is done is simply ignored from then on), stepped by the
fused kernels with greedy action selection; only the small per-step outputs (reward, done, counts, ave_deg, success)
ever reach the host.
"""
import copy
from typing import Dict, List, Tuple

import numpy as np
import torch

from . import distributed as D
from .policy import PolicySet
from .rollout import RolloutEngine

VECTORS = ["reward", "capture_cnt", "step_cnt", "move_cnt", "penalty_cnt", "nodeDeg", "variable", "vars2"]


def _details(scenario: str, n: int, counts: np.ndarray, reward: float, ave_deg) -> Dict[str, float]:
    """one step's reward_details (predator_prey.py:440-448, coverage.py:308-315) + nodeDeg, from the integer counts"""
    c = counts.astype(np.float64)
    nf = float(n)
    if scenario == "pp":
        return dict(reward=reward, capture_cnt=int(c[0]), step_cnt=1, move_cnt=c[1] / nf, penalty_cnt=int(c[2]),
                    nodeDeg=ave_deg, variable=c[3] / nf, vars2=0)
    return dict(reward=reward, capture_cnt=c[0] / nf, step_cnt=1, move_cnt=c[1] / nf, penalty_cnt=c[2] / nf,
                nodeDeg=ave_deg, variable=c[3] / nf, vars2=c[4] / nf)


def eval_model(env, policy, itr=0, n_eval_episodes=100, max_env_steps=200, eval_greedy=True, render=False,
               inspect_steps=False, seed=1, flag=None, groups: int = 4, chunk: int = 50, return_trajectory: bool = False,
               env_id0: int = 0):
    """``env``: a com_marl_b200 gym wrapper (or anything with ``spec_b200``) or a ScenarioSpec.  Returns the reference's
    ``(episode_data, epi_success, epi_rewards, bound_return)``: ``episode_data[i] = (step_success, {vec: [per step]})``,
    ``epi_rewards[vec][i]`` = sum over the episode's steps (mean for ``nodeDeg``), ``epi_success[i]`` = ``env.success``
    when the episode ended.  ``env_id0``: global id of the first episode's env (the random streams are keyed by it)."""
    if render:
        raise NotImplementedError("rendering is out of scope (DESIGN.md §8)")
    if flag is not None and flag[0]:
        return None, None, None, None
    spec = _eval_spec(getattr(env, "spec_b200", env), seed)
    return _evaluate(spec, None, policy, int(n_eval_episodes), max_env_steps, eval_greedy, groups, chunk, return_trajectory,
                     env_id0)[0]


def eval_sweep(env, policy, conditions, n_eval_episodes=100, max_env_steps=200, eval_greedy=True, seed=1, groups: int = 4,
               chunk: int = 50, return_trajectory: bool = False):
    """``eval_model`` over many channel conditions in ONE engine: ``conditions`` are specs that differ from ``env``'s in the
    channel fields only (``spec.with_channel(pl=..., rcom=..., channel_type=...)``).  Condition k plays its
    ``n_eval_episodes`` episodes in the envs with global ids ``k * n_eval_episodes ...``, so its result equals
    ``eval_model(conditions[k], ..., env_id0=k * n_eval_episodes)``.  Returns one ``eval_model`` tuple per condition, in
    order."""
    spec = _eval_spec(getattr(env, "spec_b200", env), seed)
    conds = [_eval_spec(c, seed) for c in conditions]
    return _evaluate(spec, conds, policy, int(n_eval_episodes), max_env_steps, eval_greedy, groups, chunk, return_trajectory, 0)


def eval_policies(env, policies, conditions=None, n_eval_episodes=100, max_env_steps=200, eval_greedy=True, seed=1,
                  groups: int = 4, chunk: int = 50, return_trajectory: bool = False, group=None):
    """``eval_model`` / ``eval_sweep`` of many policies of one class and architecture (every checkpoint of a run, the seeds
    of a configuration) in ONE engine, one policy launch per step for all of them.  ``policies``: a list or a PolicySet.
    With C conditions (C = 1 and ``env``'s own channel when ``conditions`` is None) policy i under condition k plays its
    ``n_eval_episodes`` episodes in the envs with global ids ``(i C + k) n_eval_episodes ...``, so ``results[i][k]`` equals
    ``eval_model(conditions[k], policies[i], ..., env_id0=(i C + k) n_eval_episodes)``.

    Across ranks (``group``, by default torch.distributed's default group when it is initialized): every rank passes all K
    policies and evaluates policies ``distributed.member_range(K, rank, world)`` in one engine of its own (the others are not
    touched); the ranks exchange the recorded per-step columns once, and every rank returns all K results, equal bit for bit
    to the single-rank call."""
    pols = policies.policies if isinstance(policies, PolicySet) else list(policies)
    spec = _eval_spec(getattr(env, "spec_b200", env), seed)
    conds = [_eval_spec(c, seed) for c in conditions] if conditions is not None else None
    C = len(conds) if conds else 1
    rank, world = D.group_rank_world(group)
    if world == 1:
        pset = policies if isinstance(policies, PolicySet) else PolicySet(pols)
        res = _evaluate(spec, conds, pset, int(n_eval_episodes), max_env_steps, eval_greedy, groups, chunk, return_trajectory, 0)
        return [res[i * C:(i + 1) * C] for i in range(len(pset))]
    E = int(n_eval_episodes)
    lo, hi = D.member_range(len(pols), rank, world)
    mine = None                                        # (columns, lengths) of this rank's hi - lo policies x C conditions
    if hi > lo:
        mine = _record(spec, conds, PolicySet(pols[lo:hi]), E, max_env_steps, eval_greedy, groups, chunk, return_trajectory,
                       lo * C * E, longest=lambda steps: _longest(steps, group))
    else:                                              # no policy here: still takes part in the step count's gather
        _longest(0, group)
    parts = [p for p in D.gather_objects(mine, group) if p is not None]
    cat = {k: np.concatenate([p[0][k] for p in parts], axis=1) for k in parts[0][0]}
    length = np.concatenate([p[1] for p in parts])
    res = _columns_results(conds or [spec], len(pols), cat, length, E, return_trajectory)
    return [res[i * C:(i + 1) * C] for i in range(len(pols))]


def _eval_spec(spec, seed):
    spec = copy.copy(spec)
    spec.seed = int(seed)
    spec.max_path_length = 0
    return spec


def _evaluate(spec, conditions, policy, E, max_env_steps, eval_greedy, groups, chunk, return_trajectory, env_id0):
    """the eval loop of eval_model / eval_sweep / eval_policies: E episodes per (policy, condition) (one condition: ``spec``'s own
    channel) in one RolloutEngine; -> one eval_model result per (policy, condition), policy-major"""
    cat, length = _record(spec, conditions, policy, E, max_env_steps, eval_greedy, groups, chunk, return_trajectory, env_id0)
    return _columns_results(conditions or [spec], len(policy) if isinstance(policy, PolicySet) else 1, cat, length, E,
                            return_trajectory)


def _record(spec, conditions, policy, E, max_env_steps, eval_greedy, groups, chunk, return_trajectory, env_id0, longest=None):
    """run the eval loop -> (recorded per-step columns {key: [steps, envs, ...]}, episode lengths [envs]).  ``longest`` (a
    rank's share of eval_policies across ranks: this rank's step count -> the largest of the ranks') makes the loop run on to
    the step count of the rank that ran longest, so that the recorded columns have the rows of the single-rank loop"""
    conds = (conditions or [spec]) * (len(policy) if isinstance(policy, PolicySet) else 1)
    B = E * len(conds)
    K = max(1, min(int(chunk), int(max_env_steps)))
    eng = RolloutEngine(spec, policy, B, device=policy.device, env_id0=env_id0, ring=K, greedy=bool(eval_greedy),
                        use_graph=True, groups=groups, auto_reset=False, conditions=conditions)
    eng.reset()
    length = np.zeros(B, dtype=np.int64)              # 0 = still running
    keep = {k: [] for k in ("reward", "done", "counts", "ave_deg", "success", "actions")}
    steps = 0

    def record_chunk(steps):
        eng.run_chunk()
        t = eng.traj
        m = min(K, max_env_steps - steps)
        keep["reward"].append(t["reward"][:m].cpu().numpy())
        keep["done"].append(t["done"][:m].cpu().numpy())
        keep["counts"].append(t["counts"][:m].cpu().numpy())
        keep["ave_deg"].append(t["ave_deg"][1:m + 1].cpu().numpy())        # env.ave_deg AFTER each step
        keep["success"].append(t["success"][:m].cpu().numpy())
        if return_trajectory:
            keep["actions"].append(t["actions"][:m].cpu().numpy())
        d = keep["done"][-1]
        for b in np.nonzero(length == 0)[0]:
            hit = np.nonzero(d[:, b])[0]
            if hit.size:
                length[b] = steps + int(hit[0]) + 1
        return steps + m

    while steps < max_env_steps and (length == 0).any():
        steps = record_chunk(steps)
    if longest is not None:                            # this rank's envs are done (or cut): on to the longest rank's count
        until = longest(steps)
        while steps < until:
            steps = record_chunk(steps)
    eng.env.check_errors()
    policy.check_errors()
    length[length == 0] = steps                          # cut by max_env_steps (eval_pp.py:71)
    return {k: np.concatenate(v) for k, v in keep.items() if v}, length


def _longest(steps, group):
    """the largest step count of the ranks' eval loops"""
    return max(D.gather_objects(int(steps), group))


def _columns_results(conds, n_policies, cat, length, E, return_trajectory):
    """one eval_model result per (policy, condition), policy-major, from the recorded columns of all their envs"""
    conds = list(conds) * n_policies
    return [_results(c, {k: v[:, i * E:(i + 1) * E] for k, v in cat.items()}, length[i * E:(i + 1) * E], return_trajectory)
            for i, c in enumerate(conds)]


def _results(spec, cat, length, return_trajectory):
    """eval_model's tuple for one condition's episodes (columns of the recorded steps)"""
    n, B = spec.n_agents, len(length)
    episode_data: List[Tuple[list, dict]] = []
    epi_success: List[int] = []
    epi_rewards: Dict[str, list] = {vec: [] for vec in VECTORS}
    fully = spec.rcom == 0
    for b in range(B):
        T = int(length[b])
        step_data = {vec: [] for vec in VECTORS}
        for k in range(T):
            deg = n if fully else np.float32(cat["ave_deg"][k, b])
            det = _details(spec.scenario, n, cat["counts"][k, b], float(cat["reward"][k, b]), deg)
            for vec in VECTORS:
                step_data[vec].append(det[vec])
        step_success = [int(x) for x in cat["success"][:T, b]]
        episode_data.append((step_success, step_data))
        epi_success.append(step_success[-1])
        for vec in VECTORS:
            epi_rewards[vec].append(np.mean(step_data[vec]) if vec == "nodeDeg" else np.sum(step_data[vec]))
    out = (episode_data, epi_success, epi_rewards, spec.bound_return)
    if return_trajectory:
        return out + ({k: cat[k] for k in ("actions", "reward", "done", "ave_deg", "success", "counts")}, length)
    return out
