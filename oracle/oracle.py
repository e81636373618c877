"""ctypes front end of the CPU oracle (oracle/cm_oracle.c) + numpy restatement of the policy forward.

TEST INFRASTRUCTURE ONLY — see the header of cm_oracle.c.  Only tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / ``--impl reference`` legs import this module; com_marl_b200 never does.

Host-side derivations restated here (independently of com_marl_b200/scenario.py, so that parity
tests also cover the product's host logic):
  * params -> channel type / comm range            custom_implement/env_communication.py:26-75
  * Coverage obstacle layout                        envs/ma_gym/envs/coverage/coverage.py:69-80,482-500
  * observation scalar features                     predator_prey.py:195-196, coverage.py:206
  * reward coefficient signs                        predator_prey.py:66-69, coverage.py:86-92
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_build", "libcm_oracle.so")
_lib = None

PP, CO = 0, 1
CH_FC, CH_FL, CH_IID, CH_GE = 0, 1, 2, 3


def build(force=False):
    src = os.path.join(_HERE, "cm_oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s"] + (["-B"] if force else []))
    return _LIB_PATH


class _Cfg(C.Structure):
    _fields_ = [(k, C.c_int32) for k in ("scenario", "n", "p", "G", "R", "T", "load", "L", "max_path_length",
                                         "n_empty_cells", "rcom2", "chan_type", "loss_apply", "ge_init")] + \
               [(k, C.c_float) for k in ("p_loss", "pgb", "pbg", "ge_bad_rate")] + \
               [(k, C.c_double) for k in ("capture_reward", "step_cost", "moving_cost", "penalty", "lazy_penalty",
                                          "revisit_penalty", "final_reward")] + \
               [("seed", C.c_uint64), ("env_id0", C.c_int64), ("wall", C.c_void_p), ("lut_row", C.c_void_p),
                ("lut_col", C.c_void_p), ("lut_t", C.c_void_p)]


class _State(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("grid", "apos", "ppos", "alive", "visited", "t", "total_capture",
                                          "success", "episode", "tick", "ge_state")]


class _IO(C.Structure):
    _fields_ = [("actions", C.c_void_p), ("prey_cand", C.c_void_p), ("spawn_agent", C.c_void_p),
                ("spawn_prey", C.c_void_p), ("spawn_episodes", C.c_int32), ("chan_u", C.c_void_p),
                ("chan_planes", C.c_int32), ("auto_reset", C.c_int32), ("obs", C.c_void_p), ("reward", C.c_void_p),
                ("done", C.c_void_p), ("counts", C.c_void_p), ("prey_alive_out", C.c_void_p), ("adj", C.c_void_p),
                ("chan", C.c_void_p), ("ave_deg", C.c_void_p)]


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_LIB_PATH)
        _lib.orc_reset.argtypes = [C.POINTER(_Cfg), C.POINTER(_State), C.POINTER(_IO), C.c_int64, C.c_void_p]
        _lib.orc_step.argtypes = [C.POINTER(_Cfg), C.POINTER(_State), C.POINTER(_IO), C.c_int64]
        _lib.orc_sample_actions.argtypes = [C.POINTER(_Cfg), C.POINTER(_State), C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.orc_philox.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]
    return _lib


def philox(seed, c0, c1, c2, c3):
    out = np.zeros(4, dtype=np.uint32)
    lib().orc_philox(seed, c0, c1, c2, c3, out.ctypes.data)
    return out


# ------------------------------------------------------------------------------------------------
# host-side derivations
# ------------------------------------------------------------------------------------------------
def coverage_walls(map_size, obst="Easy"):
    """Wall bitmap of the (map+2)^2 Coverage grid: border + fixed obstacles scaled by r = map/10
    (coverage.py:69-80 layouts, :162-168 border, :493-500 placement)."""
    assert map_size % 10 == 0, "coverage.py:67 requires map to be a multiple of 10"
    r = map_size // 10
    G = map_size + 2
    w = np.zeros((G, G), dtype=np.uint8)
    w[[0, -1], :] = 1
    w[:, [0, -1]] = 1
    rects = [((2 * r + 1, 2 * r + 1), (6 * r, 1 * r)), ((3 * r + 1, 8 * r + 1), (4 * r, 2 * r))]
    if obst == "Hard":
        rects += [((1, 2 * r + 1), (1 * r, 3 * r)), ((1, 7 * r + 1), (2 * r, 1 * r)),
                  ((4 * r + 1, 4 * r + 1), (2 * r, 3 * r)), ((8 * r + 1, 5 * r + 1), (2 * r, 2 * r)),
                  ((8 * r + 1, 8 * r + 1), (1 * r, 1 * r))]
    for (r0, c0), (h, wd) in rects:
        for i in range(h):
            for j in range(wd):
                if 0 <= r0 + i < G and 0 <= c0 + j < G:
                    w[r0 + i, c0 + j] = 1
    return w


def spec_from_params(scenario, params, seed=0, max_path_length=None, ge=None):
    """Everything the oracle needs, derived from the reference's ``params`` dict."""
    s = {}
    s["scenario"] = PP if scenario == "pp" else CO
    m = int(params["grid_size"])
    s["map"] = m
    s["n"] = int(params["n_agents"])
    s["R"] = int(params["Rsen"])
    s["L"] = int(params["n_gcn_layers"])
    s["T"] = int(params["max_env_steps"])
    s["load"] = int(params["load"])
    s["max_path_length"] = int(max_path_length) if max_path_length else 0
    if scenario == "pp":
        s["p"] = int(params["n_preys"])
        s["G"] = m
        s["capture_reward"] = float(abs(params["capture_reward"]))
        s["step_cost"] = float(-abs(params["step_cost"]))
        s["moving_cost"] = float(-abs(params["rm"]))
        s["penalty"] = float(-abs(params["penalty"]))
        s["lazy_penalty"] = s["revisit_penalty"] = s["final_reward"] = 0.0
        s["wall"] = None
        s["n_empty_cells"] = 0
        s["lut_row"] = np.array([r / m for r in range(m)], dtype=np.float64).astype(np.float32)
        s["lut_col"] = np.array([c / (m - 1) for c in range(m)], dtype=np.float64).astype(np.float32)
        s["lut_t"] = np.array([t / s["T"] for t in range(s["T"] + 1)], dtype=np.float64).astype(np.float32)
    else:
        s["p"] = 0
        G = m + 2
        s["G"] = G
        s["capture_reward"] = float(abs(params["capture_reward"]))
        s["step_cost"] = float(-abs(params["step_cost"]))
        s["moving_cost"] = float(-abs(params["rm"]))
        s["penalty"] = float(-abs(params["penalty"]))
        s["lazy_penalty"] = float(-abs(params["lazy_penalty"]))
        s["revisit_penalty"] = float(-abs(params["revisit_penalty"]))
        s["final_reward"] = 100.0
        s["wall"] = coverage_walls(m, params.get("obstComplex", "Easy"))
        s["n_empty_cells"] = int((s["wall"] == 0).sum()) - s["n"]
        s["lut_row"] = np.array([round(r / (G - 1), 2) for r in range(G)], dtype=np.float64).astype(np.float32)
        s["lut_col"] = s["lut_row"].copy()
        s["lut_t"] = np.zeros(s["T"] + 1, dtype=np.float32)
    # communication (env_communication.py:26-75)
    pref = "tr" if params.get("mode") in ("train", "restore") else "te"
    pl = params[f"{pref}pl"]
    if pl == 0:
        ct = CH_FC
    elif 0 < pl < 1:
        ct = CH_IID
    elif pl == 1:
        ct = CH_FL
    else:
        raise ValueError("invalid Ploss")
    rcom = int(params[f"{pref}Rcom"])
    if rcom + 1 >= m:
        rcom = 0
    s["rcom2"] = -1 if rcom == 0 else 2 * rcom * rcom
    s["chan_type"] = ct
    s["p_loss"] = float(np.float32(pl))
    s["loss_apply"] = int(params.get("loss_apply", 1))
    s["pgb"] = s["pbg"] = s["ge_bad_rate"] = 0.0
    s["ge_init"] = 1
    if ge is not None:
        s["chan_type"] = CH_GE
        s["pgb"], s["pbg"] = float(np.float32(ge["Pgb"])), float(np.float32(ge["Pbg"]))
        s["ge_bad_rate"] = float(np.float32(ge["Pgb"] / (ge["Pgb"] + ge["Pbg"])))
        s["ge_init"] = int(ge["GE_INIT"])
        s["loss_apply"] = int(ge["loss_apply"])
    s["seed"] = int(seed)
    w = 2 * s["R"] + 1
    s["D"] = 2 * w * w + 3 if scenario == "pp" else 3 * w * w + 2
    return s


class OracleVecEnv:
    """B independent envs stepped by the C oracle with VecEnvExecutor semantics."""

    def __init__(self, spec, B, env_id0=0):
        self.spec, self.B = spec, B
        s = spec
        n, p, G, L = s["n"], s["p"], s["G"], s["L"]
        self.n, self.p, self.G, self.L, self.D = n, p, G, L, s["D"]
        z = np.zeros
        self.grid = z((B, G * G), np.int16)
        self.apos = z((B, n, 2), np.int8)
        self.ppos = z((B, max(p, 1), 2), np.int8)
        self.alive = z((B, max(p, 1)), np.uint8)
        self.visited = z((B, G * G), np.uint8)
        self.t = z(B, np.int32)
        self.total_capture = z(B, np.int32)
        self.success = z(B, np.uint8)
        self.episode = z(B, np.uint32)
        self.tick = z(B, np.uint32)
        self.ge_state = z((B, n, n), np.uint8)
        self.obs = z((B, n, self.D), np.float32)
        self.reward = z(B, np.float64)
        self.done = z(B, np.uint8)
        self.counts = z((B, 6), np.int32)
        self.prey_alive_out = z((B, max(p, 1)), np.uint8)
        self.adj = z((B, n, n), np.uint8)
        self.chan = z((B, L, n, n), np.uint8)
        self.ave_deg = z(B, np.float32)
        self._keep = [s["wall"], s["lut_row"], s["lut_col"], s["lut_t"]]
        self.cfg = _Cfg()
        for k in ("scenario", "n", "p", "G", "R", "T", "load", "L", "max_path_length", "n_empty_cells", "rcom2",
                  "chan_type", "loss_apply", "ge_init", "p_loss", "pgb", "pbg", "ge_bad_rate", "capture_reward",
                  "step_cost", "moving_cost", "penalty", "lazy_penalty", "revisit_penalty", "final_reward", "seed"):
            setattr(self.cfg, k, s[k])
        self.cfg.env_id0 = env_id0
        self.cfg.wall = s["wall"].ctypes.data if s["wall"] is not None else None
        self.cfg.lut_row = s["lut_row"].ctypes.data
        self.cfg.lut_col = s["lut_col"].ctypes.data
        self.cfg.lut_t = s["lut_t"].ctypes.data
        self.state = _State()
        for k in ("grid", "apos", "ppos", "alive", "visited", "t", "total_capture", "success", "episode", "tick",
                  "ge_state"):
            setattr(self.state, k, getattr(self, k).ctypes.data)
        # injected streams (None -> Philox)
        self.spawn_agent = self.spawn_prey = None

    def set_spawn_queue(self, spawn_agent, spawn_prey=None):
        """spawn_agent int8 [B,E,n,2]; spawn_prey int8 [B,E,p,2]: positions for each env's e-th reset."""
        self.spawn_agent = np.ascontiguousarray(spawn_agent, dtype=np.int8)
        self.spawn_prey = None if spawn_prey is None else np.ascontiguousarray(spawn_prey, dtype=np.int8)

    def _io(self, actions=None, prey_cand=None, chan_u=None, auto_reset=True):
        io = _IO()
        keep = []

        def ptr(a, dt):
            if a is None:
                return None
            a = np.ascontiguousarray(a, dtype=dt)
            keep.append(a)
            return a.ctypes.data

        io.actions = ptr(actions, np.int8)
        io.prey_cand = ptr(prey_cand, np.int8)
        io.spawn_agent = ptr(self.spawn_agent, np.int8)
        io.spawn_prey = ptr(self.spawn_prey, np.int8)
        io.spawn_episodes = 0 if self.spawn_agent is None else self.spawn_agent.shape[1]
        io.chan_u = ptr(chan_u, np.float32)
        io.chan_planes = 0 if chan_u is None else np.asarray(chan_u).shape[1]
        io.auto_reset = int(auto_reset)
        for k in ("obs", "reward", "done", "counts", "prey_alive_out", "adj", "chan", "ave_deg"):
            setattr(io, k, getattr(self, k).ctypes.data)
        return io, keep

    def reset(self, mask=None, chan_u=None):
        io, keep = self._io(chan_u=chan_u)
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        rc = lib().orc_reset(C.byref(self.cfg), C.byref(self.state), C.byref(io), self.B,
                             None if m is None else m.ctypes.data)
        if rc:
            raise RuntimeError(f"orc_reset failed: {rc}")
        return self.obs

    def step(self, actions, prey_cand=None, chan_u=None, auto_reset=True):
        io, keep = self._io(actions, prey_cand, chan_u, auto_reset)
        rc = lib().orc_step(C.byref(self.cfg), C.byref(self.state), C.byref(io), self.B)
        if rc:
            raise RuntimeError(f"orc_step failed: {rc}")
        return self.obs, self.reward, self.done

    def sample_actions(self, probs, u=None):
        out = np.zeros((self.B, self.n), np.int8)
        probs = np.ascontiguousarray(probs, dtype=np.float32)
        uu = None if u is None else np.ascontiguousarray(u, dtype=np.float32)
        lib().orc_sample_actions(C.byref(self.cfg), C.byref(self.state), self.B, probs.ctypes.data,
                                 None if uu is None else uu.ctypes.data, out.ctypes.data)
        return out

    def details(self):
        """The reference's reward_details dict fields rebuilt from the integer counts, float64
        (predator_prey.py:440-448 / :482-490; coverage.py:308-315)."""
        c = self.counts.astype(np.float64)
        n = float(self.n)
        if self.spec["scenario"] == PP:
            return np.stack([c[:, 0], c[:, 1] / n, c[:, 2], c[:, 3] / n, np.zeros(self.B)], axis=1)
        return np.stack([c[:, 0] / n, c[:, 1] / n, c[:, 2] / n, c[:, 3] / n, c[:, 4] / n], axis=1)


# ------------------------------------------------------------------------------------------------
# policy forward, numpy float32 (comm_categorical_mlp_policy.py:48-96, comm_base_net.py:80-108,
# attention_module.py:38-49, graph_conv_module.py:51-72, categorical_mlp_module.py:64-80)
# ------------------------------------------------------------------------------------------------
def policy_forward(w, obs, avail, adj, chan, dtype=np.float32, residual=True):
    """w: dict keyed like the reference state_dict; obs (B,n,D); avail (B,n,5) or None;
    adj (B,n,n); chan (B,L,n,n).  residual=False feeds H_L alone to the head (comm_base_net.py:105-106); a GCN layer
    without a `bias` entry has no bias.  Returns logits, masked probs, attention (unmasked softmax)."""
    f = dtype
    g = lambda k: np.asarray(w[k], dtype=f)  # noqa: E731
    x = np.asarray(obs, dtype=f)
    h = np.tanh(x @ g("encoder._layers.0.linear.weight").T + g("encoder._layers.0.linear.bias"))
    E = np.tanh(h @ g("encoder._output_layers.0.linear.weight").T + g("encoder._output_layers.0.linear.bias"))
    # attention_module.py:38-49: 'general' scores H_j^T W_a q (linear_in), 'dot' scores H_j^T q (no parameter)
    q = E @ g("attention_layer.linear_in.weight").T if "attention_layer.linear_in.weight" in w else E
    s = q @ np.swapaxes(E, -1, -2)
    s = s - s.max(axis=-1, keepdims=True)
    e = np.exp(s)
    M = (e / e.sum(axis=-1, keepdims=True)).astype(f)
    H = E
    L = chan.shape[1]
    for l in range(L):
        A = M * np.asarray(adj, dtype=f) * np.asarray(chan[:, l], dtype=f)
        A = A / (A.sum(axis=-1, keepdims=True) + f(1e-12))
        bias = g(f"gcn_layers.{l}.bias") if f"gcn_layers.{l}.bias" in w else f(0)
        H = np.tanh(A @ (H @ g(f"gcn_layers.{l}.weight")) + bias)
    X = E + H if residual else H
    for i in range(3):
        X = np.tanh(X @ g(f"categorical_output_layer._layers.{i}.linear.weight").T
                    + g(f"categorical_output_layer._layers.{i}.linear.bias"))
    logits = X @ g("categorical_output_layer._output_layers.0.linear.weight").T \
        + g("categorical_output_layer._output_layers.0.linear.bias")
    z = logits - logits.max(axis=-1, keepdims=True)
    pr = np.exp(z)
    pr = pr / pr.sum(axis=-1, keepdims=True)
    if avail is not None:
        pr = pr * np.asarray(avail, dtype=f)
    pr = pr / pr.sum(axis=-1, keepdims=True)
    return logits.astype(f), pr.astype(f), M



def policy_forward_dec(w, obs, avail, dtype=np.float32):
    """Obs-DP forward (dec_categorical_mlp_policy.py:107-124): per-agent encoder (tanh, tanh) then the categorical MLP
    (tanh, linear), softmax, availability mask, renormalisation.  w: dict keyed like the reference state_dict;
    obs (B,n,D); avail (B,n,5) or None.  Returns logits, masked probs."""
    f = dtype
    g = lambda k: np.asarray(w[k], dtype=f)  # noqa: E731
    x = np.asarray(obs, dtype=f)
    h = np.tanh(x @ g("encoder._layers.0.linear.weight").T + g("encoder._layers.0.linear.bias"))
    E = np.tanh(h @ g("encoder._output_layers.0.linear.weight").T + g("encoder._output_layers.0.linear.bias"))
    X = np.tanh(E @ g("_layers.0.linear.weight").T + g("_layers.0.linear.bias"))
    logits = X @ g("_output_layers.0.linear.weight").T + g("_output_layers.0.linear.bias")
    z = logits - logits.max(axis=-1, keepdims=True)
    pr = np.exp(z)
    pr = pr / pr.sum(axis=-1, keepdims=True)
    if avail is not None:
        pr = pr * np.asarray(avail, dtype=f)
    pr = pr / pr.sum(axis=-1, keepdims=True)
    return logits.astype(f), pr.astype(f)


def policy_forward_cent(w, obs, avail, relu=False, dtype=np.float32):
    """CENT forward (centralized_categorical_mlp_policy.py:61-97): one MLP over the concatenated observation (hidden tanh | relu,
    linear output of 5n logits), reshaped to (B,n,5), softmax per agent, availability mask, renormalisation.  w: dict keyed
    like the reference state_dict; obs (B,n*D) or (B,n,D); avail (B,n,5) or None.  Returns logits (B,n,5), masked probs."""
    f = dtype
    g = lambda k: np.asarray(w[k], dtype=f)  # noqa: E731
    x = np.asarray(obs, dtype=f)
    x = x.reshape(x.shape[0], -1)
    i = 0
    while f"_layers.{i}.linear.weight" in w:
        x = x @ g(f"_layers.{i}.linear.weight").T + g(f"_layers.{i}.linear.bias")
        x = np.maximum(x, 0) if relu else np.tanh(x)
        i += 1
    logits = x @ g("_output_layers.0.linear.weight").T + g("_output_layers.0.linear.bias")
    logits = logits.reshape(logits.shape[0], -1, 5)
    z = logits - logits.max(axis=-1, keepdims=True)
    pr = np.exp(z)
    pr = pr / pr.sum(axis=-1, keepdims=True)
    if avail is not None:
        pr = pr * np.asarray(avail, dtype=f).reshape(pr.shape)
    pr = pr / pr.sum(axis=-1, keepdims=True)
    return logits.astype(f), pr.astype(f)


# ---------------------------------------------------------------------------------------------------------------
# PPO update pieces (SURVEY.md §8f.1) — numpy restatement of the reference's tensor code, test infrastructure only
# ---------------------------------------------------------------------------------------------------------------
def discount_cumsum(x, discount):
    """tensor_utils.discount_cumsum (garage/misc/tensor_utils.py:7-23): y[t] = x[t] + discount * y[t+1], float64."""
    x = np.asarray(x, dtype=np.float64)
    y = np.zeros_like(x)
    acc = 0.0
    for t in range(len(x) - 1, -1, -1):
        acc = x[t] + float(discount) * acc
        y[t] = acc
    return y


def ppo_advantages(rewards, baselines, valids, discount, gae_lambda, center=True, eps=1e-8):
    """returns / GAE advantages / per-path normalised advantages of a padded [P, T] batch.
    rewards: zero-padded float64; baselines: float32 critic values of EVERY padded step (the reference evaluates the
    critic on the padded observations, centralized_ma_ppo.py:650-657); valids: path lengths.
    compute_advantages (garage/torch/algos/_utils.py:56-113): deltas = r + g * shift(b) - b, advantages = correlation of
    the zero-extended deltas with cumprod([1, g*lam, g*lam, ...]) over the whole row; center_adv
    (centralized_ma_ppo.py:425-429): batch_norm of each row with the mean / biased variance of its valid part."""
    r32 = np.asarray(rewards, dtype=np.float64).astype(np.float32)
    b = np.asarray(baselines, dtype=np.float32)
    P, T = r32.shape
    filt = np.cumprod(np.concatenate([[1.0], np.full(T - 1, np.float32(discount) * np.float32(gae_lambda))]).astype(np.float32),
                      dtype=np.float32)
    b_next = np.concatenate([b[:, 1:], np.zeros((P, 1), np.float32)], axis=1)
    deltas = (r32 + np.float32(discount) * b_next - b).astype(np.float32)
    raw = np.zeros((P, T), dtype=np.float32)
    for t in range(T):
        raw[:, t] = (deltas[:, t:] * filt[:T - t]).sum(axis=1, dtype=np.float32)
    returns = np.zeros((P, T), dtype=np.float32)
    adv = raw.copy()
    for p in range(P):
        v = int(valids[p])
        returns[p, :v] = discount_cumsum(np.asarray(rewards, dtype=np.float64)[p, :v], discount).astype(np.float32)
        if center:
            mean = raw[p, :v].mean(dtype=np.float32)
            var = ((raw[p, :v] - mean) ** 2).mean(dtype=np.float32)
            adv[p] = (raw[p] - mean) / np.sqrt(var + np.float32(eps))
    return returns, raw, adv
