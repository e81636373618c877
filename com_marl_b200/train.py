"""Rollout + PPO update loop on the device: what LocalRunnerWrapper.train drives in the reference
(custom_implement/local_runner_wrapper.py:41-43 obtain_samples -> CentralizedMAPPO.train_once,
centralized_ma_ppo.py:175-262), with the `paths` list skipped: the rollout engine records ``max_path_length`` steps of
every env into its device trajectory ring, ``DevicePPO.batch_from_trajectory`` pads the finished episodes, ``train_once``
updates policy and critic.  One process per GPU; every rank rolls out its own slice of the global env ids and the flat
gradient buckets are all-reduced inside the update (NCCL), so all ranks hold identical weights after every step."""
import time
from dataclasses import fields

import numpy as np
import torch

from . import distributed as D
from .policy import PolicySet
from .ppo import CommBaseCritic, DevicePPO, DevicePPOSet, GaussianMLPBaseline
from .rollout import RolloutEngine, make_policy
from .spaces import Box, Discrete, EnvSpec


class DeviceTrainer:
    def __init__(self, spec, n_envs, device="cuda", env_id0=0, seed=1, kind="comm", groups=1, **ppo_args):
        """kind: 'comm' / 'dec' (runner_*_comm.py / runner_*_obsDP.py:61: Comm-DP / Obs-DP policy + CommBaseCritic), 'cent'
        (runner_*_cent.py:60-62: CENT policy + GaussianMLPBaseline(hidden_sizes=(64, 64, 64)))"""
        self.spec, self.device, self.seed = spec, torch.device(device), int(seed)
        n, Dobs = spec.n_agents, spec.obs_dim
        spec.max_path_length = spec.max_steps
        torch.manual_seed(seed)                              # identical initial weights on every rank
        self.policy = make_policy(spec, device=self.device, kind=kind)
        env_spec = EnvSpec(Box(np.zeros(n * Dobs), np.ones(n * Dobs)), Discrete(5))
        if kind != "cent":
            self.critic = CommBaseCritic(env_spec, n, n_gcn_layers=spec.n_layers, device=self.device)
        else:
            self.critic = GaussianMLPBaseline(env_spec, hidden_sizes=(64, 64, 64), device=self.device)
        self.algo = DevicePPO(self.policy, self.critic, **ppo_args)
        # one chunk = one episode horizon: every env finishes at least one episode per round (time limit)
        # the horizon is replayed from ONE captured CUDA graph: the kernel weight blobs are persistent buffers refreshed in
        # place after every update (RolloutEngine.run_chunk -> policy.refresh_weights), so the graph stays valid
        self.engine = RolloutEngine(spec, self.policy, n_envs, device=self.device, env_id0=env_id0, ring=spec.max_steps,
                                    use_graph=True, groups=groups)
        self.epoch = 0

    def train_epoch(self):
        """one round: rollout of max_steps steps for every env, then the PPO update.  Returns timings and statistics."""
        dev = self.device
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        self.engine.reset()
        self.engine.run_chunk()
        ev[1].record()
        batch = self.algo.batch_from_trajectory(self.engine.traj)
        ev[2].record()
        # the path permutation comes from a private generator keyed by (seed, epoch): the process-global numpy stream is the
        # user's (the same permutation on every rank is not required)
        perm = np.random.default_rng([self.seed, self.epoch]).permutation(int(batch["rewards"].shape[0]))
        out = self.algo.train_once(batch=batch, shuffled_ids=perm)
        ev[3].record()
        torch.cuda.synchronize(dev)
        self.engine.env.check_errors()
        stats = D.gather_stats(self.engine.local_stats())
        self.epoch += 1
        out.update(rollout_ms=ev[0].elapsed_time(ev[1]), batch_ms=ev[1].elapsed_time(ev[2]), update_ms=ev[2].elapsed_time(ev[3]),
                   agent_steps=self.engine.K * self.engine.B * self.spec.n_agents,
                   episode_stats=D.summarize_stats(stats, self.spec.scenario, self.spec.n_agents))
        out["tabular"] = self.tabular(batch, out)
        return out

    def tabular(self, batch, out):
        """The per-epoch columns CentralizedMAPPO.train_once records in dowel's tabular (centralized_ma_ppo.py:345-372 ->
        progress.csv), from the device batch of THIS rank and the whole-job episode statistics.  Episode-count columns
        (SuccessRate, Average*Count) come from the kernels' episode accounting over every episode that finished during the
        round; return columns from the padded batch like the reference (paths that finished inside the window).
        KLBefore (KL against the policy of the previous round) and GPUMemoryMax are not reproduced."""
        return tabular_row(self.spec, self.epoch - 1, batch, out, self.engine.traj["ave_deg"][:self.engine.K])

    def weights_checksum(self):
        """float64 sum of every policy + critic parameter: equal on all ranks when the gradient all-reduce works"""
        return float(sum(p.detach().double().sum() for m in (self.policy, self.critic) for p in m.parameters()))


def tabular_row(spec, iteration, batch, out, ave_deg, record=True):
    """DeviceTrainer.tabular's row from a padded device batch, the round's output dict (episode_stats, losses, times) and the
    [K, envs] per-step mean degrees of the round's envs; recorded in dowel's tabular when it is installed and ``record``"""
    rewards, mask = batch["rewards"], batch["mask"]
    und = (rewards * mask).sum(1)
    es = out["episode_stats"]
    row = dict(Iteration=iteration, NumTrajs=int(rewards.shape[0]) * spec.n_agents,
               AverageDiscountedReturn=float(batch["returns"][:, 0].double().mean()), AverageReturn=float(und.mean()),
               SuccessRate=es["SuccessRate"], AverageCaptureCount=es["AverageCaptureCount"],
               AverageStepCount=es["AverageStepCount"], AverageMovingCount=es["AverageMovingCount"],
               AveragePenaltyCount=es["AveragePenaltyCount"], AverageVariable=es["AverageVariable"], AverageVar2=es["AverageVar2"],
               StdReturn=float(und.std(unbiased=False)), MaxReturn=float(und.max()), MinReturn=float(und.min()),
               LossBefore=out["loss_before"], LossAfter=out["loss_after"], dLoss=out["loss_before"] - out["loss_after"],
               KL=out["kl"], Entropy=out["entropy"], GradNorm=float(np.mean(out["grad_norms"])) if out["grad_norms"] else 0.0,
               EpochTime=out["update_ms"] * 1e-3)
    # AveDegree: mean over paths of the per-path mean degree (:316-318); Diameter / AveTroughput are constants of the scenario
    row["AveDegree"] = float(ave_deg.double().mean()) if spec.rcom != 0 else float(spec.n_agents)
    row["Diameter"] = float(spec.n_agents if spec.rcom == 0 else 0)
    row["AveTroughput"] = float(spec.ave_trput)
    if record:
        record_tabular(row)
    return row


def record_tabular(row):
    """a tabular row into dowel's tabular, when dowel is installed"""
    try:
        from dowel import tabular as dt
        for k, v in row.items():
            dt.record(k, v)
    except Exception:                      # dowel is optional here
        pass


class _Owned(list):
    """the per-member objects of the members a rank owns (DeviceTrainerSet across ranks), indexed by GLOBAL member id;
    iteration yields them in member order.  A member another rank owns raises KeyError."""

    def __init__(self, items, members):
        super().__init__(items)
        self.members = members

    def __getitem__(self, i):
        if isinstance(i, slice) or i not in self.members:
            raise KeyError(f"member {i!r}: this rank owns members {self.members.start} .. {self.members.stop - 1}")
        return list.__getitem__(self, i - self.members.start)


def _spec_key(spec):
    """what identifies a scenario / channel condition (every field but the ones DeviceTrainerSet sets and the derived map)"""
    return None if spec is None else tuple((f.name, getattr(spec, f.name)) for f in fields(spec)
                                           if f.name not in ("max_path_length", "wall"))


class DeviceTrainerSet:
    """K training runs of one scenario and architecture as ONE batched run — the seeds x channel conditions grids of the paper's
    experiments.  Member i is ``DeviceTrainer(conditions[i] or spec, n_envs, env_id0=env_id0 + i * n_envs, seed=seeds[i],
    kind=kind, **ppo_args)`` started from member i's initial policy and critic: global env ids i E .. (i + 1) E - 1, its own
    channel condition, path permutation ``default_rng([seeds[i], epoch])`` and initial weights drawn under
    ``torch_seed=seeds[i]``.  One RolloutEngine over a PolicySet rolls out the envs of the members; one DevicePPOSet updates
    them.  Comm-DP and Obs-DP ('comm', 'dec'); 'cent' raises.

    Across ranks (``group``, by default torch.distributed's default group when it is initialized): every rank is given the
    same seeds and conditions and runs the members ``distributed.member_range(K, rank, world)`` — ``members`` — with their
    own engine and update; nothing is exchanged on the data path, since a member computes the same thing on any rank.
    ``train_epoch`` gathers the K result dicts to every rank, ``policy_state_dicts`` the K trained policies.  ``policies``,
    ``critics``, ``batches`` and ``member_traj`` hold this rank's members, indexed by global member id (on one rank: plain
    lists of all K)."""

    def __init__(self, spec, n_envs, seeds, conditions=None, kind="comm", device="cuda", env_id0=0, groups=1, group=None,
                 **ppo_args):
        self.group = group
        self.rank, self.world = D.group_rank_world(group)
        data_parallel = ppo_args.get("process_group") is not None
        if self.world > 1:                     # first, so that every later error is raised by every rank alike
            conds = None if conditions is None else [_spec_key(c) for c in conditions]
            ppo = sorted((k, v) for k, v in ppo_args.items() if k != "process_group")    # (a group handle: only whether given)
            D.check_same_on_all_ranks("DeviceTrainerSet arguments (seeds, conditions, n_envs, kind, env_id0, spec, PPO arguments)",
                                      ([int(s) for s in seeds], conds, int(n_envs), kind, int(env_id0), _spec_key(spec), ppo,
                                       data_parallel), group)
        if kind == "cent":
            raise NotImplementedError("DeviceTrainerSet covers the Comm-DP and Obs-DP families: CENT sets are not built")
        if self.world > 1 and data_parallel:
            raise NotImplementedError("a DeviceTrainerSet member runs on one rank: members data-parallel over ranks are not built")
        self.seeds = [int(s) for s in seeds]
        K = len(self.seeds)
        if K < 1:
            raise ValueError("a DeviceTrainerSet needs at least one seed")
        if K < self.world:
            raise ValueError(f"{K} members over {self.world} ranks: every rank needs at least one member")
        conditions = [None] * K if conditions is None else list(conditions)
        if len(conditions) != K:
            raise ValueError(f"{len(conditions)} conditions for {K} members")
        self.spec, self.device, self.E, self.K = spec, torch.device(device), int(n_envs), K
        lo, hi = D.member_range(K, self.rank, self.world)
        self.members = range(lo, hi)
        spec.max_path_length = spec.max_steps
        self.specs = []
        for c in conditions:
            m = spec if c is None else c
            m.max_path_length = spec.max_steps
            self.specs.append(m)
        n, Dobs = spec.n_agents, spec.obs_dim
        env_spec = EnvSpec(Box(np.zeros(n * Dobs), np.ones(n * Dobs)), Discrete(5))
        policies, critics = [], []
        for s in self.seeds[lo:hi]:            # the critic right after its policy, from the same generator state
            policies.append(make_policy(spec, device=self.device, kind=kind, torch_seed=s))
            critics.append(CommBaseCritic(env_spec, n, n_gcn_layers=spec.n_layers, device=self.device))
        self.policies, self.critics = self._owned(policies), self._owned(critics)
        if D.group_rank_world()[1] > 1 and not data_parallel:
            # a job of several ranks (whether or not this set spans them): the members' own collectives (padded lengths,
            # minibatch plan) stay on this rank
            ppo_args = dict(ppo_args, process_group=D.rank_alone_group())
        self.algo = DevicePPOSet(policies, critics, **ppo_args)
        self.pset = PolicySet(policies)
        conds = None if all(c is None for c in conditions[lo:hi]) else self.specs[lo:hi]
        self.engine = RolloutEngine(spec, self.pset, (hi - lo) * self.E, device=self.device, env_id0=env_id0 + lo * self.E,
                                    ring=spec.max_steps, use_graph=True, groups=groups, conditions=conds,
                                    block_conditions=conds is not None)
        self.epoch = 0

    def _owned(self, items):
        return list(items) if self.world == 1 else _Owned(items, self.members)

    def _column(self, i):
        """first env column of member i in this rank's engine"""
        if i not in self.members:
            raise KeyError(f"member {i!r}: this rank owns members {self.members.start} .. {self.members.stop - 1}")
        return (i - self.members.start) * self.E

    def member_traj(self, i):
        """member i's env columns of the trajectory ring (views); i is a global member id this rank owns"""
        b = self._column(i)
        return {k: v[:, b:b + self.E] for k, v in self.engine.traj.items()}

    def train_epoch(self):
        """one round of every member; returns one dict per member, all K in member order on every rank, with the keys of
        DeviceTrainer.train_epoch (times: those of the set on the rank that ran the member) and ``rank``.  The members' tabular
        rows are recorded in dowel on rank 0."""
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        self.engine.reset()
        self.engine.run_chunk()
        ev[1].record()
        batches = [m.batch_from_trajectory(self.member_traj(i)) for i, m in zip(self.members, self.algo.members)]
        self.batches = self._owned(batches)    # (the round's padded batches, kept until the next round)
        ev[2].record()
        perms = [np.random.default_rng([self.seeds[i], self.epoch]).permutation(int(b["rewards"].shape[0]))
                 for i, b in zip(self.members, batches)]
        outs = self.algo.train_once(batches, perms)
        ev[3].record()
        torch.cuda.synchronize(self.device)
        self.engine.env.check_errors()
        self.epoch += 1
        times = dict(rollout_ms=ev[0].elapsed_time(ev[1]), batch_ms=ev[1].elapsed_time(ev[2]), update_ms=ev[2].elapsed_time(ev[3]))
        Kr = self.engine.K
        for i, out, b in zip(self.members, outs, batches):
            b0 = self._column(i)
            stats = self.engine.env.stats[b0:b0 + self.E, 7:16].sum(dim=0).reshape(1, -1)
            out.update(times, agent_steps=Kr * self.E * self.spec.n_agents, rank=self.rank,
                       episode_stats=D.summarize_stats(stats, self.spec.scenario, self.spec.n_agents))
            out["tabular"] = tabular_row(self.specs[i], self.epoch - 1, b, out, self.engine.traj["ave_deg"][:Kr, b0:b0 + self.E],
                                         record=False)
        if self.world > 1:
            outs = [o for part in D.gather_objects(outs, self.group) for o in part]
        if self.rank == 0:
            for o in outs:
                record_tabular(o["tabular"])
        return outs

    def policy_state_dicts(self):
        """every member's policy parameters as K CPU state dicts in member order, on every rank (one gather across ranks):
        what ``checkpoint.save_state_dict`` / ``load_state_dict`` and ``evaluate.eval_policies`` take"""
        mine = [{k: v.detach().cpu() for k, v in p.state_dict().items()} for p in self.policies]
        return [sd for part in D.gather_objects(mine, self.group) for sd in part]
