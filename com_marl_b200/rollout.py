"""Device-resident rollout loop: policy forward + sampling -> env step -> comm update, no host round trip.

Replaces the hot loop of CentralizedMAOnPolicyVectorizedSampler.obtain_samples
(com_marl/sampler/centralized_ma_on_policy_vectorized_sampler.py:119-231): per iteration the reference
gathers dist_adj / channels from the envs (:123-127), calls policy.get_actions (:134), steps the
VecEnvExecutor (:143) and appends to Python lists (:158-191).  Here one iteration is two kernel launches
(cm_policy_forward, cm_env_step) on one stream; K consecutive iterations write into the K slots of a
trajectory ring in HBM (the kernels write the slots directly, there is no copy) and are captured once in
a CUDA graph that is replayed; episode accounting is accumulated by the env kernel (`stats`).
"""
from typing import Dict, Optional

import numpy as np
import torch

from .envs import BatchedEnv
from .policy import CommCategoricalMLPPolicy, PolicySet
from .scenario import ScenarioSpec
from .spaces import Box, Discrete, EnvSpec

STAT_KEYS = ("episodes", "return_sum", "length_sum", "success_sum", "c0_sum", "moved_sum", "c2_sum", "c3_sum", "c4_sum")


def make_policy(spec: ScenarioSpec, device="cuda", seed: Optional[int] = None, torch_seed: int = 1,
                math: str = "auto", kind: str = "comm"):
    """Policy with the reference initialisation under torch.manual_seed(torch_seed) (SURVEY.md §8d)."""
    n, D = spec.n_agents, spec.obs_dim
    env_spec = EnvSpec(Box(np.zeros(n * D, np.float32), np.ones(n * D, np.float32)), Discrete(5))
    torch.manual_seed(torch_seed)
    if kind == "dec":      # Obs-DP: no communication (dec_categorical_mlp_policy.py)
        from .policy import DecCategoricalMLPPolicy
        return DecCategoricalMLPPolicy(env_spec, n, device=device, seed=spec.seed if seed is None else seed)
    if kind == "cent":     # CENT: one MLP over the concatenated observation (centralized_categorical_mlp_policy.py)
        from .policy import CentralizedCategoricalMLPPolicy
        return CentralizedCategoricalMLPPolicy(env_spec, n, device=device, seed=spec.seed if seed is None else seed)
    return CommCategoricalMLPPolicy(env_spec, n, n_gcn_layers=spec.n_layers, device=device,
                                    seed=spec.seed if seed is None else seed, math=math)


class RolloutEngine:
    def __init__(self, spec: ScenarioSpec, policy: CommCategoricalMLPPolicy, n_envs: int, device="cuda", env_id0: int = 0,
                 ring: int = 8, record_attention: bool = False, greedy: bool = False, use_graph: bool = True,
                 groups: int = 1, auto_reset: bool = True, conditions=None, block_conditions: bool = False):
        """``conditions``: per-env channel conditions of the envs (BatchedEnv); the env groups may cut through them.
        ``policy``: one policy, or a PolicySet of P policies: the envs are then P equal blocks in policy-major order (block i runs
        policy i and, with ``conditions``, is itself split into the conditions, or with ``block_conditions`` runs under
        ``conditions[i]`` alone); the env groups may cut through the blocks."""
        self.spec, self.policy, self.B = spec, policy, int(n_envs)
        self.device = torch.device(device)
        self._set = isinstance(policy, PolicySet)
        P = len(policy) if self._set else 1
        if self.B % P:
            raise ValueError(f"n_envs = {n_envs} does not split into {P} equal policy blocks")
        self.env = BatchedEnv(spec, n_envs, device=device, env_id0=env_id0, auto_reset=auto_reset, conditions=conditions,
                              policy_blocks=P, block_conditions=block_conditions)
        # Env groups: the envs are independent, so G contiguous groups form G independent policy -> step -> policy ...
        # chains.  Each chain runs on its own stream (forked / joined inside the captured graph): there is no device-wide
        # barrier between a step of one group and the next step of another, so partially filled waves of one launch
        # are covered by the launches of the other groups.  Results are identical for every G (global env ids key the
        # random streams).  Large teams (n > 64) hand rows between their three policy launches through a scratch buffer: every
        # group has its own (ws_slot = group index).
        G = max(1, min(int(groups), self.B))
        self.groups = G
        cuts = [self.B * g // G for g in range(G + 1)]
        self._ranges = [(cuts[g], cuts[g + 1]) for g in range(G) if cuts[g + 1] > cuts[g]]
        self._envs = [self.env] if len(self._ranges) == 1 else [self.env.slice(b0, b1) for b0, b1 in self._ranges]
        self._streams = None
        self.K, self.greedy, self.use_graph = int(ring), bool(greedy), bool(use_graph)
        e, K, B, dev = self.env, self.K, self.B, self.device
        n, L, W, D, p = e.n, e.L, e.W, e.D, max(e.p, 1)

        def z(shape, dt):
            return torch.zeros(shape, dtype=dt, device=dev)

        # trajectory ring: inputs of step k live in slot k, its outputs in slot k (+1 for obs / comm state)
        self.traj: Dict[str, torch.Tensor] = dict(
            obs=z((K + 1, B, n, D), torch.float32), adj_bits=z((K + 1, B, n, W), torch.int32),
            chan_bits=z((K + 1, B, L, n, W), torch.int32), ave_deg=z((K + 1, B), torch.float32),
            actions=z((K, B, n), torch.int8), probs=z((K, B, n, 5), torch.float32),
            reward=z((K, B), torch.float64), done=z((K, B), torch.uint8), counts=z((K, B, 6), torch.int32),
            prey_alive_out=z((K, B, p), torch.uint8), success=z((K, B), torch.uint8))
        if record_attention:
            self.traj["attention"] = z((K, B, n, n), torch.float32)
        # packed observations (24 bytes per agent): written by the env kernel next to the fp32 contract output and read by the
        # tensor-core policy kernels instead of it (Comm-DP / Obs-DP)
        self._packed = bool(getattr(policy, "_kind", 2) != 2 and policy.uses_tensor_cores())
        if self._packed:
            self.traj["obs_bits"] = z((K + 1, B, n, 6), torch.int32)
        self._graph = None
        self._warm = False
        self.steps_done = 0
        self.kernel_launches = 0
        # policy calls per iteration of each group: one, or the PolicySet segments of the group's envs
        self._pol_calls = [len(PolicySet.segments(b1 - b0, self.B // P, b0)) if self._set else 1 for b0, b1 in self._ranges]

    # ---- single iteration --------------------------------------------------------------------------
    def _iteration(self, k: int, g: int = None):
        """policy forward + sampling, then env step, for ring slot k (group g of the envs, or all groups one after another)"""
        if g is None:
            for gi in range(len(self._ranges)):
                self._iteration(k, gi)
            return
        t, e = self.traj, self._envs[g]
        b0, b1 = self._ranges[g]
        pk = dict(obs_bits=t["obs_bits"][k, b0:b1], obs_nbits=e.obs_nbits) if self._packed else {}
        if self._set:
            pk.update(envs_per_policy=self.B // len(self.policy), first_env=b0)
        self.policy.act_device(t["obs"][k, b0:b1], adj_bits=t["adj_bits"][k, b0:b1], chan_bits=t["chan_bits"][k, b0:b1], tick=e.tick, episode=e.episode,
                               greedy=self.greedy, probs=t["probs"][k, b0:b1], actions=t["actions"][k, b0:b1],
                               attention=t["attention"][k, b0:b1] if "attention" in t else None, env_id0=e.env_id0, ws_slot=g, **pk)
        out = dict(obs=t["obs"][k + 1, b0:b1], adj_bits=t["adj_bits"][k + 1, b0:b1], chan_bits=t["chan_bits"][k + 1, b0:b1],
                   ave_deg=t["ave_deg"][k + 1, b0:b1], reward=t["reward"][k, b0:b1], done=t["done"][k, b0:b1],
                   counts=t["counts"][k, b0:b1], prey_alive_out=t["prey_alive_out"][k, b0:b1],
                   success_out=t["success"][k, b0:b1])
        if self._packed:
            out["obs_bits"] = t["obs_bits"][k + 1, b0:b1]
        e.step(t["actions"][k, b0:b1], out=out)
        self.kernel_launches += 1 + self._pol_calls[g]

    def _carry(self):
        """slot K (state after the last step of a chunk) becomes slot 0 of the next chunk"""
        for k in ("obs", "adj_bits", "chan_bits", "ave_deg", "obs_bits"):
            if k in self.traj:
                self.traj[k][0].copy_(self.traj[k][self.K])

    def reset(self):
        t = self.traj
        self.env.stats.zero_()
        out = dict(obs=t["obs"][0], adj_bits=t["adj_bits"][0], chan_bits=t["chan_bits"][0], ave_deg=t["ave_deg"][0])
        if self._packed:
            out["obs_bits"] = t["obs_bits"][0]
        self.env.reset(out=out)
        self.steps_done = 0

    def _chunk_eager(self):
        if len(self._ranges) == 1:
            for k in range(self.K):
                self._iteration(k, 0)
            return
        # one chain per group, each on its own stream (fork / join on events: capturable)
        if self._streams is None:
            self._streams = [torch.cuda.Stream(device=self.device) for _ in self._ranges]
        main = torch.cuda.current_stream(self.device)
        fork = torch.cuda.Event()
        fork.record(main)
        for g, st in enumerate(self._streams):
            st.wait_event(fork)
            with torch.cuda.stream(st):
                for k in range(self.K):
                    self._iteration(k, g)
                join = torch.cuda.Event()
                join.record(st)
            main.wait_event(join)

    def _capture(self):
        g = torch.cuda.CUDAGraph()
        launches = self.kernel_launches
        with torch.cuda.graph(g):
            self._chunk_eager()          # recorded, not executed: the env state does not advance here
        self.kernel_launches = launches
        self._graph = g

    def run_chunk(self):
        """K rollout iterations (K * B * n agent-steps).  The first chunk after construction runs eagerly (it also
        warms the library's launch-geometry caches and the weight blob); later chunks replay one CUDA graph."""
        if self.steps_done:
            self._carry()
        if self.use_graph and self._warm:
            # the graph holds raw pointers to the policy's weight blobs: they are persistent buffers refreshed IN PLACE, so
            # bringing them up to date here (outside the graph) is all a parameter update needs — no re-capture
            self.policy.refresh_weights()
            if self._graph is None:
                self._capture()
            self._graph.replay()
            self.kernel_launches += self.K * (len(self._ranges) + sum(self._pol_calls))
        else:
            self._chunk_eager()
            self._warm = True
        self.steps_done += self.K

    def run(self, steps: int):
        assert steps % self.K == 0, "steps must be a multiple of the ring size"
        for _ in range(steps // self.K):
            self.run_chunk()

    # ---- episode statistics ------------------------------------------------------------------------
    def local_stats(self) -> torch.Tensor:
        """float64 [9] sums over this GPU's envs of the finished-episode accumulators (STAT_KEYS)."""
        return self.env.stats[:, 7:16].sum(dim=0)

    def agent_steps(self) -> int:
        return self.steps_done * self.B * self.env.n


class HostRollout:
    """The sampler's loop with HOST buffers, one C call per env part and step (cm_rollout_step_host): the garage-sampler
    boundary (centralized_ma_on_policy_vectorized_sampler.py:119-231) as the unit of work instead of the two step-level calls.

    Observations, masks and env state never leave the device between steps — the policy reads what the previous step left
    in HBM — so the per-step traffic is: H2D the availability bytes (the sampler's get_avail_actions(), :128-131), D2H
    everything the sampler appends to its running paths (next observation, adjacency / channel bit rows, ave_deg, reward,
    done, counts, prey_alive, success, actions, action probabilities and — ``record_attention`` — the attention weights).

    The envs are cut into ``parts`` independent batches, each with its own stream, device output arena and ``host_slots``
    pinned host arenas; one part's D2H transfers run while the other parts' kernels execute.  ``submit()`` enqueues one step
    of every part into the next host slot and returns at once; ``collect()`` waits for the oldest submitted step and returns
    its host views (valid until that slot is submitted again, i.e. for ``host_slots - 1`` further submits).  Because step
    t + 1 needs nothing from the host, a caller may keep ``host_slots - 1`` steps in flight; ``step()`` = submit + collect.
    Results are identical to RolloutEngine's (global env ids key the random streams)."""

    def __init__(self, spec: ScenarioSpec, policy, n_envs: int, device="cuda", env_id0: int = 0, parts: int = 4,
                 host_slots: int = 2, record_attention: bool = False, greedy: bool = False):
        import ctypes as C
        from . import _native as N
        self._C, self._N = C, N
        self.spec, self.policy, self.B = spec, policy, int(n_envs)
        self.device = torch.device(device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        device = self.device
        self.greedy, self.slots = bool(greedy), max(1, int(host_slots))
        P = max(1, min(int(parts), self.B))
        cuts = [self.B * g // P for g in range(P + 1)]
        self.ranges = [(cuts[g], cuts[g + 1]) for g in range(P) if cuts[g + 1] > cuts[g]]
        comm = bool(getattr(policy, "comm", False))
        self.record_attention = bool(record_attention) and comm
        self.parts = []
        n = spec.n_agents
        for g, (b0, b1) in enumerate(self.ranges):
            Bp = b1 - b0
            env = BatchedEnv(spec, Bp, device=device, env_id0=env_id0 + b0)
            pspecs = [("actions", (Bp, n), torch.int8), ("probs", (Bp, n, 5), torch.float32)]
            if self.record_attention:
                pspecs.append(("attention", (Bp, n, n), torch.float32))
            # env outputs + policy outputs in ONE arena per side (same order, same padding): a step's whole result is one
            # DMA transfer (csrc/host_abi.cu merges the neighbours of a declared arena)
            specs = env._out_specs() + pspecs
            dev_arena = N.arena(specs, device=self.device)
            for k, _, _ in env._out_specs():             # the env writes its outputs into the combined arena
                setattr(env, k, dev_arena[k])
            pdev = {k: dev_arena[k] for k, _, _ in pspecs}
            avail_dev = torch.full((Bp, n), 0x1F, dtype=torch.uint8, device=self.device)
            part = dict(env=env, range=(b0, b1), stream=torch.cuda.Stream(device=self.device), pdev=pdev, avail_dev=avail_dev,
                        env_dev=env._io(pdev["actions"]), slots=[], keep=dev_arena)
            for _ in range(self.slots):
                ha = N.arena(specs, pinned=True)
                avail = torch.full((Bp, n), 0x1F, dtype=torch.uint8).pin_memory()
                env_host, pol_host = N.StepIO(), N.PolicyIO()
                env_host.host_arena = pol_host.host_arena = 1
                for k, _, _ in env._out_specs():
                    setattr(env_host, k, ha[k].data_ptr())
                for k, _, _ in pspecs:
                    setattr(pol_host, k, ha[k].data_ptr())
                pol_host.avail_bits = avail.data_ptr()
                views = {k: v.numpy() for k, v in ha.items() if k != "_arena"}
                views["success"] = views.pop("success_out")
                views["avail_bits"] = avail.numpy()
                views["env_ids"] = (env_id0 + b0, env_id0 + b1)
                part["slots"].append(dict(env_host=env_host, pol_host=pol_host, views=views, event=torch.cuda.Event(), keep=(ha, avail)))
            self.parts.append(part)
        self._submitted = self._collected = 0
        self.kernel_launches = 0

    def _pol_structs(self, part, g):
        env, pdev = part["env"], part["pdev"]
        pol = self.policy
        if getattr(pol, "comm", False):
            return pol._call_structs(env.obs, env.adj_bits, env.chan_bits, part["avail_dev"], None, env.tick, env.episode, self.greedy,
                                     pdev["probs"], None, pdev.get("attention"), pdev["actions"], env.env_id0, g)
        return pol._call_structs(env.obs, None, None, part["avail_dev"], None, env.tick, env.episode, self.greedy, pdev["probs"], None,
                                 None, pdev["actions"], env.env_id0, g)

    def reset(self):
        """env.reset() of every env; returns the per-part host views (obs, adj_bits, chan_bits, ave_deg are meaningful)"""
        C, N = self._C, self._N
        torch.cuda.set_device(self.device)
        out = []
        for part in self.parts:
            env, sl = part["env"], part["slots"][0]
            N.check("cm_env_reset_host", N.lib().cm_env_reset_host(C.byref(env.desc), C.byref(env.state), C.byref(part["env_dev"]),
                                                                   C.byref(sl["env_host"]), part["stream"].cuda_stream))
            part["stream"].synchronize()
            out.append(sl["views"])
        self._submitted = self._collected = 0
        return out

    def submit(self):
        """enqueue one rollout step of every part (asynchronous)"""
        C, N = self._C, self._N
        assert self._submitted - self._collected < self.slots, "collect() the oldest step before submitting into its host slot"
        if torch.cuda.current_device() != (self.device.index or 0):
            torch.cuda.set_device(self.device)
        self.policy.refresh_weights()
        s = self._submitted % self.slots
        for g, part in enumerate(self.parts):
            cs = part.get("pol")
            if cs is None:
                cs = part["pol"] = self._pol_structs(part, g)
            env, sl = part["env"], part["slots"][s]
            N.check("cm_rollout_step_host", N.lib().cm_rollout_step_host(
                C.byref(cs[0]), C.byref(cs[1]), C.byref(sl["pol_host"]), C.byref(env.desc), C.byref(env.state),
                C.byref(part["env_dev"]), C.byref(sl["env_host"]), part["stream"].cuda_stream))
            sl["event"].record(part["stream"])
        self._submitted += 1
        self.kernel_launches += 2 * len(self.parts)

    def collect(self):
        """wait for the oldest submitted step; returns one dict of host views per part"""
        assert self._collected < self._submitted, "nothing in flight"
        s = self._collected % self.slots
        out = []
        for part in self.parts:
            part["slots"][s]["event"].synchronize()
            out.append(part["slots"][s]["views"])
        self._collected += 1
        return out

    def step(self):
        self.submit()
        return self.collect()

    def bytes_per_step(self):
        """(h2d, d2h) bytes one step moves"""
        h2d = d2h = 0
        for part in self.parts:
            ha, avail = part["slots"][0]["keep"]
            h2d += avail.numel()
            d2h += sum(v.numel() * v.element_size() for k, v in ha.items() if k != "_arena")
        return h2d, d2h

    def check_errors(self):
        for part in self.parts:
            part["env"].check_errors()
        self.policy.check_errors()
