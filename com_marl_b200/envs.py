"""Device-resident batched PredatorPrey / Coverage environments and their gym-contract views.

``BatchedEnv`` holds B independent instances as SoA tensors in HBM and steps them all with one
kernel launch through the C ABI (cm_env_step / cm_env_reset, include/commarl_b200.h) with the
semantics of garage's VecEnvExecutor (garage/sampler/vec_env_executor.py:19-54): env.step, time
limit, reset-on-done, observations and communication state of the post-reset state.

``PredatorPreyWrapper`` / ``CoverageWrapper`` keep the constructor signature, attributes and
``reset()/step()/get_avail_actions()`` contract of envs/predatorprey_wrapper.py:23-73 and
envs/coverage_wrapper.py:16-57 (the interface the reference's sampler and eval scripts see) over a
B = 1 ``BatchedEnv``; they exist for drop-in compatibility and parity tests, not for throughput.
"""
import ctypes as C
from typing import Optional

import numpy as np
import torch

from . import _native as N
from .scenario import ScenarioSpec
from .spaces import Box, Discrete, EnvSpec


def pack_positions(pos) -> np.ndarray:
    """(..., 2) [row, col] -> uint16 row | col << 8 (layout of agent_pos / prey_pos)"""
    pos = np.asarray(pos).astype(np.int64)
    return (pos[..., 0] | (pos[..., 1] << 8)).astype(np.uint16)


def unpack_positions(packed) -> np.ndarray:
    packed = np.asarray(packed).astype(np.uint16)
    return np.stack([packed & 0xFF, packed >> 8], axis=-1).astype(np.int8)


def check_conditions(spec: ScenarioSpec, conditions, n_envs: int, policy_blocks: int = 1, block_conditions: bool = False):
    """-> the validated list of channel conditions of a BatchedEnv (None when there are none); raises ValueError"""
    if int(policy_blocks) < 1 or int(n_envs) % int(policy_blocks):
        raise ValueError(f"n_envs = {n_envs} does not split into {policy_blocks} equal policy blocks")
    n_envs = int(n_envs) // int(policy_blocks)
    if conditions is None:
        return None
    conditions = list(conditions)
    if block_conditions:
        if len(conditions) != int(policy_blocks):
            raise ValueError(f"block_conditions needs one condition per policy block: {len(conditions)} for {policy_blocks}")
        n_envs = len(conditions)                 # (every block is whole under its condition)
    if not 1 <= len(conditions) <= N.MAX_CONDS:
        raise ValueError(f"between 1 and {N.MAX_CONDS} channel conditions are supported, got {len(conditions)}")
    if int(n_envs) % len(conditions):
        raise ValueError(f"n_envs = {n_envs} does not split evenly into {len(conditions)} conditions")
    for k, c in enumerate(conditions):
        if not spec.same_except_channel(c):
            raise ValueError(f"condition {k} differs from the spec outside the channel fields {ScenarioSpec.CHANNEL_FIELDS}")
        c.validate()
    return conditions


class BatchedEnv:
    """B environment instances of one scenario on one GPU."""

    def __init__(self, spec: ScenarioSpec, n_envs: int, device="cuda", env_id0: int = 0, auto_reset: bool = True,
                 conditions=None, policy_blocks: int = 1, block_conditions: bool = False):
        """``conditions``: optional list of specs that differ from ``spec`` in the channel fields only
        (ScenarioSpec.CHANNEL_FIELDS, e.g. ``spec.with_channel(pl=..., rcom=...)``).  The envs are then split into equal
        contiguous blocks in list order and block k communicates under ``conditions[k]`` (``spec``'s own channel is not
        used); ``cond_idx`` [B] holds each env's condition.  Everything else — and the global env ids — stays as without.
        ``policy_blocks``: the envs are that many equal blocks (one per policy of a PolicySet), each split into the conditions
        in the same way (env order policy, condition, episode).  ``block_conditions``: instead, one condition per policy block —
        block i communicates under ``conditions[i]`` (the members of a set trained each under its own channel)."""
        N.lib()  # fail loudly if the CUDA library is missing; there is no CPU path
        if not torch.cuda.is_available():
            raise RuntimeError("com_marl_b200 needs a CUDA device: the rollout engine has no CPU fallback")
        spec.validate()
        self.conditions = check_conditions(spec, conditions, n_envs, policy_blocks, block_conditions)
        self.policy_blocks = int(policy_blocks)
        self.spec, self.B, self.auto_reset = spec, int(n_envs), bool(auto_reset)
        self.device = torch.device(device)
        self.env_id0 = int(env_id0)
        n, p, G, L = spec.n_agents, spec.n_preys, spec.grid, spec.n_layers
        self.n, self.p, self.G, self.L, self.D, self.W = n, p, G, L, spec.obs_dim, (n + 31) // 32
        self.obs_nbits = spec.obs_dim - (3 if spec.scenario == "pp" else 2)     # leading 0/1 window columns of an observation row
        self.obs_bits = None                    # optional packed observation output [B, n, 6] int32 (enable_obs_bits)
        B, dev = self.B, self.device

        def z(shape, dt):
            return torch.zeros(shape, dtype=dt, device=dev)

        # ---- state (SoA, env-major; layout documented in include/commarl_b200.h) ----
        self.agent_pos = z((B, n), torch.int16)
        self.prey_pos = z((B, max(p, 1)), torch.int16)
        self.prey_alive = z((B, max(p, 1)), torch.uint8)
        self.visited = z((B, G), torch.int64)
        self.step_count = z((B,), torch.int32)
        self.total_capture = z((B,), torch.int32)
        self.success = z((B,), torch.uint8)
        self.episode = z((B,), torch.int32)
        self.tick = z((B,), torch.int32)
        chans = [c.channel for c in self.conditions] if self.conditions else [spec.channel]
        self.ge_state = z((B, n, self.W), torch.int32) if N.CH_GE in chans else None
        # ---- outputs: one arena, in the order the host-buffer call copies them (one DMA transfer, csrc/host_abi.cu) ----
        for k, v in N.arena(self._out_specs(), device=dev).items():
            setattr(self, "_out_arena" if k == "_arena" else k, v)
        self.error_flag = z((1,), torch.int32)
        self.stats = z((B, 16), torch.float64)      # episode accounting, layout in include/commarl_b200.h
        # ---- constants ----
        self._lut = torch.from_numpy(spec.lut()).to(dev)
        self._wall = torch.from_numpy(spec.wall_rows().view(np.int64)).to(dev) if spec.scenario == "co" else None
        self.cond_idx = None
        if self.conditions:
            K = len(self.conditions)
            self._conds_host = (N.ChannelCond * K)(*[c.channel_cond() for c in self.conditions])
            self._conds = torch.frombuffer(bytearray(bytes(self._conds_host)), dtype=torch.uint8).to(dev)
            P = self.policy_blocks
            if block_conditions:
                self.cond_idx = torch.arange(K, dtype=torch.uint8, device=dev).repeat_interleave(B // K)
            else:
                self.cond_idx = torch.arange(K, dtype=torch.uint8, device=dev).repeat_interleave(B // (K * P)).repeat(P)
        self.desc = self._desc()
        self.state = N.EnvState()
        self.state.n_envs = B
        for k in ("agent_pos", "prey_pos", "prey_alive", "visited", "step_count", "total_capture", "success",
                  "episode", "tick", "ge_state"):
            setattr(self.state, k, N.ptr(getattr(self, k)))
        self._spawn_agent = self._spawn_prey = None
        self._spawn_episodes = 0
        self._io_cache = {}

    def _desc(self):
        d = self.spec.to_desc(N.ptr(self._wall), N.ptr(self._lut), env_id0=self.env_id0)
        if self.cond_idx is not None:
            d.conds, d.cond_idx, d.n_conds = N.ptr(self._conds), N.ptr(self.cond_idx), len(self.conditions)
            d.conds_host = C.addressof(self._conds_host)
        return d

    def _out_specs(self):
        B, n, p, L = self.B, self.n, self.p, self.L
        return [("obs", (B, n, self.D), torch.float32), ("adj_bits", (B, n, self.W), torch.int32),
                ("chan_bits", (B, L, n, self.W), torch.int32), ("reward", (B,), torch.float64), ("done", (B,), torch.uint8),
                ("counts", (B, 6), torch.int32), ("prey_alive_out", (B, max(p, 1)), torch.uint8),
                ("success_out", (B,), torch.uint8), ("ave_deg", (B,), torch.float32)]

    def enable_obs_bits(self):
        """also write the packed observation (cm_step_io.obs_bits: window bits + scalar columns, 24 bytes per agent) — the
        form the tensor-core policy kernels read instead of the fp32 rows"""
        if self.obs_bits is None:
            self.obs_bits = torch.zeros((self.B, self.n, 6), dtype=torch.int32, device=self.device)
            self._io_cache.clear()
            self._hio = None
        return self.obs_bits

    _SLICED = ("obs_bits", "agent_pos", "prey_pos", "prey_alive", "visited", "step_count", "total_capture", "success", "episode", "tick",
               "ge_state", "obs", "reward", "done", "counts", "prey_alive_out", "success_out", "adj_bits", "chan_bits", "ave_deg",
               "stats", "_spawn_agent", "_spawn_prey", "cond_idx")

    def slice(self, b0: int, b1: int) -> "BatchedEnv":
        """View of the envs [b0, b1): shares every buffer with this object (all arrays are env-major, so the slices are
        contiguous), with its own descriptor (global env id offset) and state struct.  Independent env groups can then be
        stepped by separate launches on separate streams (RolloutEngine(groups=...)); the random streams are keyed by the
        global env id, so results do not depend on the grouping."""
        v = object.__new__(BatchedEnv)
        v.__dict__.update(self.__dict__)
        v.B, v.env_id0 = int(b1 - b0), self.env_id0 + int(b0)
        for k in self._SLICED:
            t = getattr(self, k, None)
            setattr(v, k, None if t is None else t[b0:b1])
        v.desc = v._desc()
        v.state = N.EnvState()
        v.state.n_envs = v.B
        for k in ("agent_pos", "prey_pos", "prey_alive", "visited", "step_count", "total_capture", "success",
                  "episode", "tick", "ge_state"):
            setattr(v.state, k, N.ptr(getattr(v, k)))
        v._io_cache = {}
        v._pin = v._hio = None
        return v

    # ---- injected streams (parity mode) ---------------------------------------------------------
    def set_spawn_queue(self, spawn_agent, spawn_prey=None):
        """spawn_agent int [B,E,n,2], spawn_prey int [B,E,p,2]: positions used by each env's e-th reset
        instead of the Philox spawn (SURVEY.md §8c: 'record env.agent_pos/prey_pos after each reference
        reset() and inject into the engine')."""
        sa = pack_positions(spawn_agent)
        assert sa.shape[0] == self.B and sa.shape[2] == self.n
        self._hio = None                         # the cached host-call structs carry the spawn queue pointers
        self._spawn_agent = torch.from_numpy(sa.view(np.int16)).to(self.device).contiguous()
        self._spawn_episodes = sa.shape[1]
        if self.p:
            sp = pack_positions(spawn_prey)
            assert sp.shape == (self.B, self._spawn_episodes, self.p)
            self._spawn_prey = torch.from_numpy(sp.view(np.int16)).to(self.device).contiguous()
        self._io_cache.clear()

    def _dev(self, x, dtype):
        if x is None:
            return None
        if isinstance(x, torch.Tensor):
            return x.to(device=self.device, dtype=dtype).contiguous()
        return torch.as_tensor(np.ascontiguousarray(x), dtype=dtype).to(self.device)

    def _io(self, actions=None, prey_cand=None, chan_u=None, auto_reset=None, out=None):
        io = N.StepIO()
        io.actions, io.prey_cand, io.chan_u = N.ptr(actions), N.ptr(prey_cand), N.ptr(chan_u)
        io.chan_planes = 0 if chan_u is None else int(chan_u.shape[1])
        io.spawn_agent, io.spawn_prey, io.spawn_episodes = N.ptr(self._spawn_agent), N.ptr(self._spawn_prey), self._spawn_episodes
        io.auto_reset = int(self.auto_reset if auto_reset is None else auto_reset)
        for k in ("obs", "reward", "done", "counts", "prey_alive_out", "success_out", "adj_bits", "chan_bits", "ave_deg",
                  "error_flag", "stats"):
            t = out[k] if (out is not None and k in out) else getattr(self, k)
            setattr(io, k, N.ptr(t))
        # the packed observation (24 bytes per agent, for cm_policy_forward) is written only when the caller gives a buffer
        ob = out.get("obs_bits") if out is not None else getattr(self, "obs_bits", None)
        io.obs_bits = N.ptr(ob)
        return io

    # ---- VecEnvExecutor surface -------------------------------------------------------------------
    def reset(self, mask=None, chan_u=None, out=None):
        """env.reset() for the masked envs (all when mask is None); returns the (B, n*D) observation view."""
        m = self._dev(mask, torch.uint8)
        u = self._dev(chan_u, torch.float32)
        io = self._io(chan_u=u, out=out)
        with torch.cuda.device(self.device):
            N.check("cm_env_reset", N.lib().cm_env_reset(C.byref(self.desc), C.byref(self.state), C.byref(io),
                                                        N.ptr(m), N.stream_ptr()))
        return self.obs.view(self.B, -1)

    def step(self, actions, prey_cand=None, chan_u=None, auto_reset=None, out=None):
        """One VecEnvExecutor.step for all envs.  ``actions``: int8 device tensor or array (B, n).
        Asynchronous on the current stream; returns views of the output tensors.  ``out`` may redirect any
        output (obs, reward, done, counts, prey_alive_out, adj_bits, chan_bits, ave_deg) to another tensor of the
        same shape — e.g. slot t of a trajectory buffer — so recording a trajectory costs no extra copy."""
        a = self._dev(actions, torch.int8)
        assert a.shape == (self.B, self.n), f"actions must be ({self.B}, {self.n})"
        c = self._dev(prey_cand, torch.int8)
        u = self._dev(chan_u, torch.float32)
        io = self._io(a, c, u, auto_reset, out)
        with torch.cuda.device(self.device):
            N.check("cm_env_step", N.lib().cm_env_step(C.byref(self.desc), C.byref(self.state), C.byref(io), N.stream_ptr()))
        return self.obs.view(self.B, -1), self.reward, self.done

    # ---- host-buffer surface: the drop-in call with numpy in / numpy out ------------------------------
    def _pinned(self):
        if getattr(self, "_pin", None) is None:
            pa = N.arena(self._out_specs(), pinned=True)          # mirrors the device arena: one D2H transfer per step
            self._pin = dict(actions=torch.empty((self.B, self.n), dtype=torch.int8, pin_memory=True),
                             obs=pa["obs"], reward=pa["reward"], done=pa["done"], counts=pa["counts"], adj_bits=pa["adj_bits"],
                             chan_bits=pa["chan_bits"], ave_deg=pa["ave_deg"], prey_alive_out=pa["prey_alive_out"],
                             success=pa["success_out"])
            self._pin_arena = pa["_arena"]
            self._act_dev = torch.empty((self.B, self.n), dtype=torch.int8, device=self.device)
            self._host_out = {k: v.numpy() for k, v in self._pin.items() if k != "actions"}
            self._host_out["pinned"] = self._pin   # the same buffers as torch pinned tensors (zero-copy hand-over to the policy)
        return self._pin

    _HOST_OUT = ("obs", "reward", "done", "counts", "adj_bits", "chan_bits", "ave_deg", "prey_alive_out", "success")

    def _host_io(self):
        """host-side cm_step_io (pinned buffers) + device-side cm_step_io of the host-buffer calls, built once"""
        if getattr(self, "_hio", None) is None:
            pin = self._pinned()
            hio = N.StepIO()
            hio.host_arena = 1          # the pinned outputs mirror the device output arena (_out_specs order / padding)
            hio.actions = pin["actions"].data_ptr()
            for k in self._HOST_OUT:
                setattr(hio, "success_out" if k == "success" else k, pin[k].data_ptr())
            self._hio = hio
            self._dio = self._io(self._act_dev)
            self._host_event = torch.cuda.Event()
        return self._hio, self._dio

    def step_host(self, actions, sync=True, stream=None):
        """VecEnvExecutor.step with HOST buffers: numpy actions in, numpy (views of pinned buffers) out, as ONE C call
        (cm_env_step_host): H2D actions, the step kernel, D2H obs, reward, done, counts, adj/chan bit rows, ave_deg,
        prey_alive, success (env.success as the sampler reads it at this step).
        ``sync=False`` (split phase): enqueue on the current stream and return ``(out, event)`` at once; the buffers are
        valid after ``event.synchronize()`` — lets several env batches overlap their copies on different streams."""
        hio, dio = self._host_io()
        pin = self._pin
        if actions is getattr(self, "_last_actions", None):
            pass                                                                     # the same pinned tensor as last time
        elif isinstance(actions, torch.Tensor) and actions.is_pinned() and actions.dtype == torch.int8 and actions.numel() == self.B * self.n:
            hio.actions = actions.data_ptr()                                         # already pinned: no staging copy
            self._last_actions = actions
        else:
            pin["actions"].numpy()[...] = np.asarray(actions, dtype=np.int8).reshape(self.B, self.n)
            hio.actions = pin["actions"].data_ptr()
            self._last_actions = None
        if self.device.index is not None and torch.cuda.current_device() != self.device.index:
            torch.cuda.set_device(self.device)   # the library launches on the current device
        if stream is None:
            stream = torch.cuda.current_stream(self.device)
        N.check("cm_env_step_host", N.lib().cm_env_step_host(C.byref(self.desc), C.byref(self.state), C.byref(dio), C.byref(hio),
                                                             stream.cuda_stream))
        out = self._host_out
        if not sync:
            self._host_event.record(stream)
            return out, self._host_event
        stream.synchronize()
        return out

    def reset_host(self):
        pin = self._pinned()
        hio, dio = self._host_io()
        with torch.cuda.device(self.device):
            N.check("cm_env_reset_host", N.lib().cm_env_reset_host(C.byref(self.desc), C.byref(self.state), C.byref(dio), C.byref(hio),
                                                                   N.stream_ptr()))
        torch.cuda.current_stream(self.device).synchronize()
        out = {k: pin[k].numpy() for k in ("obs", "adj_bits", "chan_bits", "ave_deg")}
        out["pinned"] = pin
        return out

    def host_step_bytes(self):
        """(h2d, d2h) bytes moved by one step_host call"""
        pin = self._pinned()
        d2h = sum(v.numel() * v.element_size() for k, v in pin.items() if k != "actions")
        return pin["actions"].numel(), d2h

    def comm_update(self, at_reset=False, chan_u=None):
        """update_communication_state alone from the current positions (env_communication.py:91-157)."""
        u = self._dev(chan_u, torch.float32)
        io = self._io(chan_u=u)
        with torch.cuda.device(self.device):
            N.check("cm_comm_update", N.lib().cm_comm_update(C.byref(self.desc), C.byref(self.state), C.byref(io),
                                                            int(at_reset), N.stream_ptr()))

    def check_errors(self):
        """Raises like the reference does on an invalid action (predator_prey.py:255); synchronises."""
        code = int(self.error_flag.item())
        if code:
            self.error_flag.zero_()
            if code == N.CM_EACTION:
                raise Exception("Action Not found!")
            raise N.NativeError("env kernel", code, N.lib().cm_strerror(code).decode())

    # ---- reference-shaped views (dense float arrays like env.dist_adj / env.channels) ---------------
    def _unpack(self, bits, rows):
        out = torch.empty((rows, self.n), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            N.check("cm_mask_unpack", N.lib().cm_mask_unpack(N.ptr(bits), N.ptr(out), rows, self.n, N.stream_ptr()))
        return out

    def dist_adj(self):
        return self._unpack(self.adj_bits, self.B * self.n).view(self.B, self.n, self.n)

    def channels(self):
        return self._unpack(self.chan_bits, self.B * self.L * self.n).view(self.B, self.L, self.n, self.n)

    def details(self) -> np.ndarray:
        """reward_details fields (capture_cnt, move_cnt, penalty_cnt, variable, vars2) as float64, rebuilt
        on the host from the integer counts exactly as the reference forms them
        (predator_prey.py:440-448/:482-490 use np.mean of 0/1 vectors; coverage.py:308-315 sum/len)."""
        c = self.counts.cpu().numpy().astype(np.float64)
        n = float(self.n)
        if self.spec.scenario == "pp":
            return np.stack([c[:, 0], c[:, 1] / n, c[:, 2], c[:, 3] / n, np.zeros(self.B)], axis=1)
        return np.stack([c[:, 0] / n, c[:, 1] / n, c[:, 2] / n, c[:, 3] / n, c[:, 4] / n], axis=1)

    def positions(self):
        """(agent_pos [B,n,2], prey_pos [B,p,2]) int8 on the host — cm_state_get of the survey's proposal"""
        a = unpack_positions(self.agent_pos.cpu().numpy().view(np.uint16))
        pp = unpack_positions(self.prey_pos.cpu().numpy().view(np.uint16)) if self.p else None
        return a, pp

    def visited_grid(self) -> np.ndarray:
        """Coverage visited map as uint8 [B,G,G]"""
        rows = self.visited.cpu().numpy().view(np.uint64)
        cols = np.arange(self.G, dtype=np.uint64)
        return ((rows[:, :, None] >> cols[None, None, :]) & np.uint64(1)).astype(np.uint8)


class _WrapperBase:
    """gym-contract view over one device env (B = 1)."""
    _scenario = None
    metadata = {"render.modes": []}

    def __init__(self, centralized, other_agent_visible=False, *args, **kwargs):
        params = kwargs["params"]
        self.params = params
        self.centralized = bool(centralized)
        self._agent_visible = other_agent_visible
        self.spec_b200 = ScenarioSpec.from_params(self._scenario, params, seed=int(params.get("seed", 1) or 1))
        if self._scenario == "co" and "max_steps" in kwargs:        # Coverage takes max_steps as a ctor kwarg (coverage.py:39)
            self.spec_b200.max_steps = int(kwargs["max_steps"])
        elif self._scenario == "co":
            self.spec_b200.max_steps = 400
        s = self.spec_b200
        self.n_agents = s.n_agents
        self.n_preys = s.n_preys
        self._max_steps = s.max_steps
        self.curriculum_learning = params.get("curriculum_learning")
        self.bound_return = s.bound_return if self._scenario == "pp" else None
        self.ave_trput = 0
        self.diameter = 0
        self.success = 0
        self.pickleable = False     # holds device memory
        self._vec = BatchedEnv(s, 1, device=kwargs.get("device", "cuda"), auto_reset=False)
        D = s.obs_dim
        w2 = s.window ** 2
        if self._scenario == "pp":
            low, high = [0.0] * D, [1.0] * D
        else:
            low, high = [-1.0] * (3 * w2) + [0.0, 0.0], [1.0] * D
        mult = s.n_agents if self.centralized else 1
        self.action_space = Discrete(5)
        self.observation_space = Box(np.array(low * mult, dtype=np.float32), np.array(high * mult, dtype=np.float32))
        self.spec = EnvSpec(self.observation_space, self.action_space)
        self.dist_adj = self.channels = None
        self.ave_deg = 0
        self._seed = None

    # -- attributes the sampler reads after every step/reset (…vectorized_sampler.py:123-127) --
    def _refresh_comm(self):
        v, s = self._vec, self.spec_b200
        if s.rcom == 0:    # env_communication.py:219-223 returns float64 ones and integer degree/diameter
            self.dist_adj = np.ones((s.n_agents, s.n_agents))
            self.ave_deg = s.n_agents
            self.diameter = s.n_agents
        else:
            self.dist_adj = v.dist_adj()[0].cpu().numpy()
            self.ave_deg = np.float32(v.ave_deg[0].item())
            self.diameter = 0
        self.channels = v.channels()[0].cpu().numpy()

    def _obs_out(self):
        o = self._vec.obs[0].cpu().numpy()
        return o.reshape(-1) if self.centralized else [o[i] for i in range(self.n_agents)]

    def inject_streams(self, prey_cand=None, chan_u=None):
        """Parity mode of the public API: pre-drawn random streams consumed one slice per call instead of the Philox streams —
        ``prey_cand`` int8 [steps, p, 5] (the np.random.choice candidates of prey_random_move, predator_prey.py:396-407; step s
        uses slice s) and ``chan_u`` float32 [steps + 1, planes, n, n] (the torch.rand draws of get_iid_channel /
        get_next_state_matrix; the first reset() uses slice 0, step s slice s + 1, and a reset() after step s re-reads slice
        s + 1 — how tests/golden/make_golden.py fed the reference).  SURVEY.md §8c's injection points."""
        self._inj_cand = None if prey_cand is None else np.asarray(prey_cand, dtype=np.int8)
        self._inj_u = None if chan_u is None else np.asarray(chan_u, dtype=np.float32)
        self._inj_t = 0

    _inj_cand = _inj_u = None
    _inj_t = 0

    def seed(self, n):
        self._seed = n
        self._vec.desc.seed = int(n)
        return [n, n]

    def get_avail_actions(self):
        avail = [[1] * self.action_space.n for _ in range(self.n_agents)]
        return np.concatenate(avail) if self.centralized else avail

    def reset(self, epoch=-1):
        self.epoch = epoch
        self._vec.reset(chan_u=None if self._inj_u is None else self._inj_u[self._inj_t][None])
        if self._scenario == "co":
            self.ave_trput = self.spec_b200.ave_trput
            self.bound_return = self.spec_b200.bound_return
        self._refresh_comm()
        return self._obs_out()

    def step(self, actions):
        v = self._vec
        a = np.asarray(actions).reshape(1, self.n_agents)
        if ((a < 0) | (a > 4)).any():
            raise Exception("Action Not found!")       # predator_prey.py:255 / coverage.py:347
        t = self._inj_t
        v.step(a.astype(np.int8), prey_cand=None if self._inj_cand is None else self._inj_cand[t][None],
               chan_u=None if self._inj_u is None else self._inj_u[t + 1][None])
        self._inj_t = t + 1
        reward = float(v.reward[0].item())
        det = v.details()[0]
        details = dict(reward=reward, capture_cnt=det[0], step_cnt=1, move_cnt=det[1], penalty_cnt=det[2],
                       variable=det[3], vars2=det[4])
        if self._scenario == "pp":
            details["capture_cnt"], details["penalty_cnt"], details["vars2"] = int(det[0]), int(det[2]), 0
        done = bool(v.done[0].item())
        self.success = int(v.success[0].item())
        self._refresh_comm()
        info = {"prey_alive": v.prey_alive_out[0].cpu().numpy().astype(bool)} if self._scenario == "pp" else {}
        if self.centralized:
            return self._obs_out(), (reward, details), done, info
        return self._obs_out(), reward, [done] * self.n_agents, info

    @property
    def agent_pos(self):
        a, _ = self._vec.positions()
        return {i: [int(a[0, i, 0]), int(a[0, i, 1])] for i in range(self.n_agents)}

    @property
    def prey_pos(self):
        _, p = self._vec.positions()
        return {i: [int(p[0, i, 0]), int(p[0, i, 1])] for i in range(self.n_preys)}

    def close(self):
        pass


class PredatorPreyWrapper(_WrapperBase):
    """Same call contract as envs/predatorprey_wrapper.py:23-73."""
    _scenario = "pp"


class CoverageWrapper(_WrapperBase):
    """Same call contract as envs/coverage_wrapper.py:16-57."""
    _scenario = "co"
