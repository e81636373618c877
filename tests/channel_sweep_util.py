"""Channel-condition tables for tests/test_gpu_channel_sweep.py and the spawned worker that replays them under a forced
lane group.

A BatchedEnv built with ``conditions`` launches env_kernel's table instantiation: env b communicates under
conds[cond_idx[b]].  Its reference is one uniform BatchedEnv per condition (that condition's spec, env_id0 = k * E) driven
by the same actions: every output and the whole state of block k of the mixed env must equal the uniform env's, bit for
bit, after the reset and after every step.

Nothing here touches CUDA at import time.
"""
import os
import queue
import sys
import time
import traceback

import numpy as np

TESTS = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(TESTS)
SEED, ACT_SEED = 4321, 91
GE_FAST = dict(pgb=0.2, pbg=0.3)            # transition rates high enough that links flip every few steps

# (scenario, map, Rsen, density, capture load, params overrides): n = 4, 32 (W = 1), Coverage 54 (W = 2), 200 (W = 7)
SIZES = {
    "pp_n4": ("pp", 10, 1, 0.04, 2, dict(max_env_steps=10)),
    "pp_n32": ("pp", 20, 2, 0.08, 4, dict(max_env_steps=10)),
    "co_n54": ("co", 30, 1, 0.06, 2, dict(max_env_steps=10)),
    "pp_n200": ("pp", 50, 2, 0.08, 4, dict(max_env_steps=8)),
}

# with_channel arguments: FC, FL, IID at 0.05 and 0.5, IID with Rcom = 1, IID with an Rcom that collapses to fully
# connected, GE with GE_INIT 1, 0 and -1
TABLE = [dict(pl=0), dict(pl=1), dict(pl=0.05), dict(pl=0.5), dict(pl=0.2, rcom=1), dict(pl=0.2, rcom=99),
         dict(channel_type="GE", ge_init=1, **GE_FAST), dict(channel_type="GE", ge_init=0, **GE_FAST),
         dict(channel_type="GE", ge_init=-1, **GE_FAST)]
# loss_apply = 0: one GE transition per env step (GE_INIT = -1 is unsupported there)
TABLE_LA0 = [dict(pl=0), dict(pl=0.3, rcom=2), dict(channel_type="GE", ge_init=1, **GE_FAST),
             dict(channel_type="GE", ge_init=0, **GE_FAST)]

OUTPUTS = ("obs", "obs_bits", "adj_bits", "chan_bits", "ave_deg", "reward", "done", "counts", "prey_alive_out", "success_out")
STATE = ("agent_pos", "prey_pos", "prey_alive", "visited", "ge_state", "step_count", "total_capture", "success", "episode",
         "tick", "stats")


def params_of(size, **over):
    if os.path.join(TESTS, "golden") not in sys.path:
        sys.path.insert(0, os.path.join(TESTS, "golden"))
    import ref_harness
    scen, m, sen, den, cap, o = SIZES[size]
    p = dict(o, mode="test", tepl=0.2, teRcom=9)
    p.update(over)
    return ref_harness.scenario_params(scen, m, sen, den, cap=cap, **p)


def base_spec(size, **over):
    from com_marl_b200.scenario import ScenarioSpec
    return ScenarioSpec.from_params(SIZES[size][0], params_of(size, **over), seed=SEED)


def conditions(spec, table):
    return [spec.with_channel(**t) for t in table]


def max_planes(spec):
    return 2 * spec.n_layers + 1


def chan_u(spec, B, k):
    """injected uniforms of call k for every env, sized for the largest plane count of any entry (GE: 2 L + 1)"""
    import streams
    return streams.uniforms_f32(7000 + k, (B, max_planes(spec), spec.n_agents, spec.n_agents))


def arrays(env):
    """{name: host copy} of every output and the whole state of a BatchedEnv (or a slice of one)"""
    out = {}
    for k in OUTPUTS + STATE:
        t = getattr(env, k)
        if t is not None:
            out[k] = t.contiguous().cpu().numpy()
    return out


def digest(env):
    import hashlib
    return {k: hashlib.sha1(v.tobytes()).hexdigest() for k, v in arrays(env).items()}


def compare(mixed, unis, E, where):
    """block k of the mixed env == uniform env k, every array the uniform env has"""
    got = arrays(mixed)
    for k, u in enumerate(unis):
        ref = arrays(u)
        for name, r in ref.items():
            g = got[name][k * E:(k + 1) * E]
            if not np.array_equal(g, r):
                bad = tuple(int(i) for i in np.argwhere(g != r)[0]) if g.shape == r.shape else g.shape
                raise AssertionError(f"{name} of condition {k} differs from its uniform env {where}: first at {bad}")


def run_mixed(spec, conds, E, steps, inj=False, uniform=True):
    """reset + ``steps`` auto-reset steps with random actions of the mixed env (and, ``uniform``, of one uniform env per
    condition, compared after every call).  Returns (per-call digests of the mixed env, the mixed env)."""
    import streams
    from com_marl_b200.envs import BatchedEnv
    K = len(conds)
    B = K * E
    mixed = BatchedEnv(spec, B, conditions=conds)
    mixed.enable_obs_bits()
    unis = []
    if uniform:
        unis = [BatchedEnv(c, E, env_id0=k * E) for k, c in enumerate(conds)]
        for u in unis:
            u.enable_obs_bits()
    acts = streams.actions(ACT_SEED, (steps, B, spec.n_agents))
    u = (lambda k: chan_u(spec, B, k)) if inj else (lambda k: None)

    def blk(x, k):
        return None if x is None else x[k * E:(k + 1) * E]

    u0 = u(0)
    mixed.reset(chan_u=u0)
    for k, e in enumerate(unis):
        e.reset(chan_u=blk(u0, k))
    if unis:
        compare(mixed, unis, E, "after the first reset")
    dig = [digest(mixed)]
    for s in range(steps):
        us = u(s + 1)
        mixed.step(acts[s], chan_u=us)
        for k, e in enumerate(unis):
            e.step(acts[s][k * E:(k + 1) * E], chan_u=blk(us, k))
        if unis:
            compare(mixed, unis, E, f"at step {s}")
        dig.append(digest(mixed))
    mixed.check_errors()
    for e in unis:
        e.check_errors()
    return dig, mixed


# ---- forced lane groups: one spawned child per group ---------------------------------------------------------------
FORCED = [("pp_n32", False), ("co_n54", True)]      # (size, injected channel uniforms)
FORCED_E, FORCED_STEPS = 21, 24


def forced_runs():
    out = {}
    for size, inj in FORCED:
        spec = base_spec(size)
        out[f"{size}_{inj}"] = run_mixed(spec, conditions(spec, TABLE), FORCED_E, FORCED_STEPS, inj=inj, uniform=False)[0]
    return out


def worker(group, q):
    try:
        os.environ["CM_ENV_GROUP"] = str(group)     # before the first env launch: launch() reads it once per process
        for p in (ROOT, TESTS):
            if p not in sys.path:
                sys.path.insert(0, p)
        import torch
        torch.set_num_threads(1)
        q.put(("ok", forced_runs()))
    except BaseException:
        q.put(("error", traceback.format_exc()))


def run_forced(group, timeout=600):
    """-> forced_runs() computed by a spawned child with CM_ENV_GROUP = group.  The child is always joined."""
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
