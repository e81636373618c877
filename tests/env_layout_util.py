"""Layout matrix of env_kernel (csrc/env_kernels.cu) and the subprocess worker that replays it under a forced lane group.

env_kernel gives each env a group of 4, 8, 16 or 32 lanes (launch(), env_kernels.cu:1148-1164); the group may be smaller
than the team, and every lane-parallel loop then strides by it.  ``CM_ENV_GROUP`` forces the group, but launch() reads it
once per process, so each forced group runs in its own spawned child (``run_forced``).  The child records per-step SHA-1
digests of every output and of the whole state; tests/test_gpu_env_layouts.py compares them with the digests of the
default-group run, which it has compared with the C oracle first.

Nothing here touches CUDA at import time.
"""
import hashlib
import os
import queue
import sys
import time
import traceback

import numpy as np

TESTS = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(TESTS)
GROUPS = (4, 8, 16, 32)

# ---- launch()'s choice of the lanes per env, restated (env_kernels.cu:34-36, 71-79, 1148-1164) -------------------------
# Used to label the configs and to pick which forced groups can launch; never to predict what the kernel computes.
WARPS_PER_CTA = 8                           # kWarpsPerCta (CM_ENV_WARPS)
CONST_BYTES = 64 * 8 + 264 * 8              # kConstBytes: wall rows + the k / n table
SMEM_LIMIT = 227 * 1024                     # dynamic shared memory one CTA may opt in to on sm_100


def warp_bytes(n, p, G):
    """env_warp_bytes() rounded up to 16 bytes: the shared-memory scratch of one env (sequential-move build)"""
    n_pad, p_pad = (n + 7) & ~7, (p + 7) & ~7
    base = 2 * G * 8 + 6 * n_pad * 4 + n_pad * 2 + p_pad * 2 + p_pad + n_pad + p_pad + p_pad
    return (base + 15) & ~15


def smem_bytes(group, n, p, G):
    return CONST_BYTES + WARPS_PER_CTA * (32 // group) * warp_bytes(n, p, G)


def default_group(n, p, G):
    """the smallest group (at least 4 lanes, 8 once the team exceeds 4) that still lets three CTAs share an SM"""
    team = max(n, p)
    g = 4 if team <= 4 else 8
    while g < 32 and smem_bytes(g, n, p, G) > 225 * 1024 * WARPS_PER_CTA // 24:
        g *= 2
    return g


def group_fits(group, n, p, G):
    return smem_bytes(group, n, p, G) <= SMEM_LIMIT


# ---- the configuration matrix ------------------------------------------------------------------------------------------
GE_FAST = dict(Pgb=0.2, Pbg=0.3)            # transition rates high enough that links flip every few steps
GE_REF = dict(Pgb=0.0196, Pbg=0.282)        # the reference's defaults (bench.py's c3_ge)


def _cfg(id, scen, m, sen, den, cap, loss, over, ge, B, steps, inj=False):
    return dict(id=id, scen=scen, map=m, sen=sen, den=den, cap=cap, loss=loss, over=over, ge=ge, B=B, steps=steps, inj=inj)


CONFIGS = [
    # group 16 with IID drops, W = 3
    _cfg("g16_iid", "pp", 30, 2, 0.08, 4, 0.2, dict(max_env_steps=14), None, 192, 45),
    # multi-word GE rows (W = 2, the last word holds one link), three layers
    _cfg("ge_w2_l3", "pp", 20, 1, 0.08, 2, 0.2, dict(n_agents=33, n_preys=33, n_gcn_layers=3, max_env_steps=12),
         dict(GE_FAST, GE_INIT=1, loss_apply=1), 256, 40),
    # drawn initial GE state (plane 0, then 2 (L - 1) transition planes), W = 3, four layers, fewer preys than agents
    _cfg("ge_w3_l4_init", "pp", 20, 1, 0.08, 2, 0.2, dict(n_agents=65, n_preys=17, n_gcn_layers=4, max_env_steps=10),
         dict(GE_FAST, GE_INIT=-1, loss_apply=1), 128, 34),
    # Coverage at group 16: W = 4 with a 3-link last word, one layer (Coverage teams divide by its 3 groups)
    _cfg("co_g16_l1", "co", 40, 2, 0.03, 2, 0.1, dict(n_agents=99, n_gcn_layers=1, max_env_steps=10), None, 128, 34),
    # the preys set the team (and so the group): 4 agents, 150 preys
    _cfg("prey_team", "pp", 30, 1, 0.08, 2, 0.3, dict(n_agents=4, n_preys=150, max_env_steps=12), None, 512, 40),
    # loss_apply = 0 (every layer is the same state), all links bad at reset, W = 5
    _cfg("ge_la0_w5", "pp", 40, 1, 0.08, 2, 0.2, dict(n_agents=129, n_preys=129, max_env_steps=8),
         dict(GE_FAST, GE_INIT=0, loss_apply=0), 48, 26),
    # C5's team (n = p = 200, group 32) with channel draws
    _cfg("c5_drops", "pp", 50, 2, 0.08, 4, 0.2, dict(max_env_steps=8), None, 32, 26),
    # C3 on the Gilbert-Elliot channel (bench.py's c3_ge): one full 32-link word per row
    _cfg("c3_ge", "pp", 20, 2, 0.08, 4, 0.2, dict(max_env_steps=15), dict(GE_REF, GE_INIT=1, loss_apply=1), 1024, 50),
]
# the same configurations fed injected uniforms (chan_u): the float path of link_row_bits at W > 1
CONFIGS += [dict(c, id=c["id"] + "_inj", inj=True, B=c["B"] // 2) for c in CONFIGS
            if c["id"] in ("ge_w2_l3", "ge_w3_l4_init", "co_g16_l1")]
BY_ID = {c["id"]: c for c in CONFIGS}

SEED, ENV_ID0, ACT_SEED = 1234, 1000, 77


def params_of(cfg):
    if os.path.join(TESTS, "golden") not in sys.path:
        sys.path.insert(0, os.path.join(TESTS, "golden"))
    import ref_harness
    over = dict(cfg["over"])
    if cfg["ge"]:
        over.update(cfg["ge"])
    return ref_harness.scenario_params(cfg["scen"], cfg["map"], cfg["sen"], cfg["den"], cap=cfg["cap"], loss=cfg["loss"], **over)


def spec_of(cfg):
    from com_marl_b200.scenario import ScenarioSpec
    return ScenarioSpec.from_params(cfg["scen"], params_of(cfg), seed=SEED, channel_type="GE" if cfg["ge"] else None)


def oracle_of(cfg, B=None):
    from oracle import oracle as orc
    ospec = orc.spec_from_params(cfg["scen"], params_of(cfg), seed=SEED, ge=cfg["ge"])
    return orc.OracleVecEnv(ospec, B or cfg["B"], env_id0=ENV_ID0)


def shape_of(cfg):
    """(n, p, grid side, layers, W) of a config"""
    s = spec_of(cfg)
    return s.n_agents, s.n_preys, s.grid, s.n_layers, (s.n_agents + 31) // 32


def group_info(cfg):
    n, p, G, _, _ = shape_of(cfg)
    return default_group(n, p, G), [g for g in GROUPS if group_fits(g, n, p, G)]


def chan_planes(spec):
    from com_marl_b200 import _native as N
    return spec.n_layers if spec.channel == N.CH_IID else 2 * spec.n_layers + 1


def chan_u(cfg, spec, B, k):
    """injected uniforms of call k (0: the first reset, s + 1: step s), [B, planes, n, n] float32"""
    import streams
    return streams.uniforms_f32(9000 + k, (B, chan_planes(spec), spec.n_agents, spec.n_agents))


def actions(cfg, spec, B):
    import streams
    return streams.actions(ACT_SEED, (cfg["steps"], B, spec.n_agents))


# ---- digests --------------------------------------------------------------------------------------------------------
OUTPUTS = ("obs", "obs_bits", "adj_bits", "chan_bits", "ave_deg", "reward", "done", "counts", "prey_alive_out", "success_out")
STATE = ("agent_pos", "prey_pos", "prey_alive", "visited", "ge_state", "step_count", "total_capture", "success", "episode",
         "tick", "stats")


def digest(env):
    """{array: sha1} over every output and the whole state of a BatchedEnv"""
    out = {}
    for k in OUTPUTS + STATE:
        t = getattr(env, k)
        if t is not None:
            out[k] = hashlib.sha1(t.contiguous().cpu().numpy().tobytes()).hexdigest()
    return out


def first_difference(ref, got):
    """(step index, array) of the first digest that differs; step index 0 is the reset, k the k-th step"""
    if len(ref) != len(got):
        return (min(len(ref), len(got)), "number of steps")
    for s, (a, b) in enumerate(zip(ref, got)):
        for k in a:
            if a[k] != b.get(k):
                return (s, k)
    return None


def unpack_bits(bits, n):
    """int32 bit rows (..., W) -> uint8 (..., n)"""
    b = np.ascontiguousarray(bits).view(np.uint32)
    cols = np.arange(n)
    return ((b[..., cols >> 5] >> (cols & 31).astype(np.uint32)) & 1).astype(np.uint8)


def run(cfg, check=None):
    """Reset + cfg["steps"] auto-reset steps of a device env (default or forced group, whatever this process has).
    ``check(env, s, actions, chan_u)`` is called after the reset (s = -1, actions None) and after every step with that
    call's inputs.  Returns the per-call digests."""
    from com_marl_b200.envs import BatchedEnv
    spec = spec_of(cfg)
    B = cfg["B"]
    env = BatchedEnv(spec, B, env_id0=ENV_ID0)
    env.enable_obs_bits()
    acts = actions(cfg, spec, B)
    u = (lambda k: chan_u(cfg, spec, B, k)) if cfg["inj"] else (lambda k: None)
    u0 = u(0)
    env.reset(chan_u=u0)
    if check:
        check(env, -1, None, u0)
    dig = [digest(env)]
    for s in range(cfg["steps"]):
        us = u(s + 1)
        env.step(acts[s], chan_u=us)
        if check:
            check(env, s, acts[s], us)
        dig.append(digest(env))
    env.check_errors()
    return dig


# ---- the child process of one forced group ----------------------------------------------------------------------------
def worker(group, q):
    try:
        os.environ["CM_ENV_GROUP"] = str(group)     # before the first env launch: launch() reads it once per process
        for p in (ROOT, TESTS):
            if p not in sys.path:
                sys.path.insert(0, p)
        import torch
        torch.set_num_threads(1)
        out = {}
        for cfg in CONFIGS:
            n, p, G, _, _ = shape_of(cfg)
            if group_fits(group, n, p, G):
                out[cfg["id"]] = run(cfg)
        q.put(("ok", out))
    except BaseException:
        q.put(("error", traceback.format_exc()))


def run_forced(group, timeout=600):
    """-> {config id: digests} computed by a spawned child with CM_ENV_GROUP = group.  The child is always joined."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    proc = ctx.Process(target=worker, args=(group, q))
    proc.start()
    try:
        deadline = time.monotonic() + timeout
        while True:
            try:
                status, res = q.get(timeout=2)
                break
            except queue.Empty:
                if not proc.is_alive():
                    raise RuntimeError(f"group {group} child exited with code {proc.exitcode} before reporting")
                if time.monotonic() > deadline:
                    raise TimeoutError(f"group {group} child did not finish in {timeout} s")
        proc.join(timeout=60)
        if status != "ok":
            raise RuntimeError(f"group {group} child failed:\n{res}")
        assert proc.exitcode == 0, proc.exitcode
        return res
    finally:
        if proc.is_alive():
            proc.terminate()
            proc.join(timeout=30)
        if proc.is_alive():
            proc.kill()
            proc.join(timeout=30)
