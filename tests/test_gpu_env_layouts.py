"""env_kernel under every layout it chooses between, bit-exact against the C oracle.

env_kernel's lanes per env (4, 8, 16 or 32), the words per bit row (W = ceil(n / 32)), the number of channel planes
and layers, and the team that sets the group all change with the configuration.  The matrix in env_layout_util.CONFIGS
pins each of them:
  (a) every config against the oracle with generated (Philox) or injected channel streams, auto-reset, every step;
  (b) the same configs under every lane group whose shared memory fits (CM_ENV_GROUP, one spawned process per group),
      digest for digest against the default-group run of (a);
  (c) masked resets (cm_env_reset with a mask) against OracleVecEnv.reset(mask);
  (d) cm_mask_pack / cm_mask_unpack at the 32-bit word edges.
"""
import os

import numpy as np
import pytest

import env_layout_util as U

pytestmark = pytest.mark.gpu

if os.environ.get("CM_ENV_GROUP"):
    pytest.skip("CM_ENV_GROUP is set: this module forces every lane group itself and needs the default in-process",
                allow_module_level=True)

# default-group digests of (a), reused by (b)
_DEFAULT = {}


def _same(name, got, ref, where, ref_name="oracle"):
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape, f"{name}: shape {got.shape} != {ref_name} {ref.shape} {where}"
    if not np.array_equal(got, ref):
        bad = tuple(int(i) for i in np.argwhere(got != ref)[0])
        raise AssertionError(f"{name} differs from the {ref_name} {where}: first at index {bad} "
                             f"(kernel {got[bad]}, {ref_name} {ref[bad]})")


def _obs_bits_of(obs, nbits):
    """the packed observation (cm_step_io.obs_bits) of fp32 rows: bit k of words 0..2 = column k < nbits, words 3..5 the
    float bits of the remaining columns (zero where there is none)"""
    win = obs[..., :nbits]
    assert np.isin(win, (0.0, 1.0)).all()
    bits = np.zeros(obs.shape[:-1] + (96,), np.uint8)
    bits[..., :nbits] = win != 0
    words = np.packbits(bits, axis=-1, bitorder="little").view("<u4")
    scal = np.zeros(obs.shape[:-1] + (3,), np.uint32)
    rest = np.ascontiguousarray(obs[..., nbits:]).view(np.uint32)
    scal[..., :rest.shape[-1]] = rest
    return np.concatenate([words, scal], axis=-1)


class OracleCheck:
    """Steps the oracle alongside the device env and compares everything, every call.  The episode accounting the kernel
    keeps in env.stats is rebuilt from the oracle's per-step outputs in the kernel's order of float64 additions."""

    def __init__(self, cfg, oenv, auto_reset=True):
        self.cfg, self.o, self.auto_reset = cfg, oenv, auto_reset
        self.run = np.zeros((oenv.B, 7))         # running return, length, counts 0..4
        self.fin = np.zeros((oenv.B, 9))         # finished episodes, return / length / success / counts sums
        self.dones = 0

    def state(self, env, where):
        o, n, p = self.o, self.o.n, self.o.p
        _same("obs", env.obs.cpu().numpy(), o.obs, where)
        if env.obs_bits is not None:
            _same("obs_bits", env.obs_bits.cpu().numpy().view(np.uint32), _obs_bits_of(o.obs, env.obs_nbits), where)
        a, pp = env.positions()
        _same("agent_pos", a, o.apos, where)
        _same("adj_bits", U.unpack_bits(env.adj_bits.cpu().numpy(), n), o.adj, where)
        _same("chan_bits", U.unpack_bits(env.chan_bits.cpu().numpy(), n), o.chan, where)
        _same("ave_deg", env.ave_deg.cpu().numpy(), o.ave_deg, where)
        if p:
            _same("prey_pos", pp, o.ppos[:, :p], where)
            _same("prey_alive", env.prey_alive.cpu().numpy()[:, :p], o.alive[:, :p], where)
        else:
            _same("visited", env.visited_grid().reshape(env.B, -1), o.visited, where)
            _same("total_capture", env.total_capture.cpu().numpy(), o.total_capture, where)
        if env.ge_state is not None:
            _same("ge_state", U.unpack_bits(env.ge_state.cpu().numpy(), n), o.ge_state, where)
        _same("step_count", env.step_count.cpu().numpy(), o.t, where)
        _same("episode", env.episode.cpu().numpy().view(np.uint32), o.episode, where)
        _same("tick", env.tick.cpu().numpy().view(np.uint32), o.tick, where)
        _same("success", env.success.cpu().numpy(), o.success, where)

    def step(self, env, s, acts, u):
        o, p, where = self.o, self.o.p, f"at step {s}"
        o.step(acts, chan_u=u, auto_reset=self.auto_reset)
        _same("reward", env.reward.cpu().numpy(), o.reward, where)
        _same("done", env.done.cpu().numpy(), o.done, where)
        _same("counts", env.counts.cpu().numpy(), o.counts, where)
        _same("success_out", env.success_out.cpu().numpy(), o.success, where)
        if p:
            _same("prey_alive_out", env.prey_alive_out.cpu().numpy()[:, :p], o.prey_alive_out[:, :p], where)
        done = o.done.astype(bool)
        self.dones += int(done.sum())
        run = self.run + np.concatenate([o.reward[:, None], np.ones((o.B, 1)), o.counts[:, :5].astype(np.float64)], axis=1)
        f = self.fin
        f[done, 0] += 1.0
        f[done, 1] += run[done, 0]
        f[done, 2] += run[done, 1]
        f[done, 3] += o.success[done].astype(np.float64)
        f[done, 4:] += run[done, 2:]
        self.run = np.where(done[:, None], 0.0, run)
        _same("stats", env.stats.cpu().numpy(), np.concatenate([self.run, f], axis=1), where)
        self.state(env, where)

    def __call__(self, env, s, acts, u):
        if acts is None:
            self.o.reset(chan_u=u)
            self.state(env, "after the first reset")
        else:
            self.step(env, s, acts, u)


def _label(cfg):
    n, p, G, L, W = U.shape_of(cfg)
    dg, fits = U.group_info(cfg)
    ch = ("GE" if cfg["ge"] else f"IID {cfg['loss']}") + (" injected" if cfg["inj"] else "")
    return f"{cfg['id']}: {cfg['scen']} {cfg['map']} n={n} p={p} L={L} W={W} {ch}; default group {dg}, forced groups {fits}"


@pytest.mark.parametrize("cid", [c["id"] for c in U.CONFIGS])
def test_env_layout_matches_oracle(cid):
    """Every output and the whole state, every step, bit for bit, across several auto-resets per env."""
    cfg = U.BY_ID[cid]
    print(_label(cfg))
    chk = OracleCheck(cfg, U.oracle_of(cfg))
    _DEFAULT[cid] = U.run(cfg, chk)
    assert chk.dones >= 2 * cfg["B"], "the config must cross several auto-resets per env"
    assert int(chk.o.episode.min()) >= 3


def test_group_matrix_covers_every_group():
    """Across the default groups and the forced groups, every group size runs IID drops and multi-word GE rows."""
    seen = {g: set() for g in U.GROUPS}
    for cfg in U.CONFIGS:
        _, _, _, _, W = U.shape_of(cfg)
        dg, fits = U.group_info(cfg)
        print(_label(cfg))
        for g in set(fits) | {dg}:
            if cfg["ge"] and W > 1:
                seen[g].add("ge_multiword")
            if not cfg["ge"] and cfg["loss"] > 0:
                seen[g].add("iid_drops")
    for g in U.GROUPS:
        assert seen[g] == {"ge_multiword", "iid_drops"}, (g, seen[g])
    assert {U.group_info(c)[0] for c in U.CONFIGS} == set(U.GROUPS) - {4}


@pytest.mark.parametrize("group", U.GROUPS, ids=[f"group{g}" for g in U.GROUPS])
def test_forced_group_matches_default(group):
    """CM_ENV_GROUP = group in a fresh process: the per-step digests of every output, obs_bits and the whole state equal
    those of the default-group run (which (a) has compared with the oracle)."""
    forced = U.run_forced(group)
    ran, bad = [], []
    for cfg in U.CONFIGS:
        n, p, G, _, _ = U.shape_of(cfg)
        if not U.group_fits(group, n, p, G):
            assert cfg["id"] not in forced
            continue
        ref = _DEFAULT.get(cfg["id"]) or U.run(cfg)
        diff = U.first_difference(ref, forced[cfg["id"]])
        if diff is not None:
            bad.append(f"{cfg['id']}: {diff[1]} differs first at call {diff[0]} (0 = the reset)")
        ran.append(cfg["id"])
    print(f"group {group} ran {ran}")
    assert ran and not bad, f"group {group} differs from the default group: " + "; ".join(bad)


# ---- (c) masked reset ---------------------------------------------------------------------------------------------------
_KEEP = ("agent_pos", "prey_pos", "prey_alive", "visited", "ge_state", "episode", "tick", "step_count")


@pytest.mark.parametrize("cid", ["ge_w2_l3", "co_g16_l1"])
def test_masked_reset_matches_oracle(cid):
    """BatchedEnv.reset(mask) without auto-reset: the masked envs (done ones and mid-episode ones) restart exactly as the
    oracle's do, the others keep their state byte for byte, and stepping goes on in lockstep."""
    from com_marl_b200.envs import BatchedEnv
    cfg = U.BY_ID[cid]
    spec = U.spec_of(cfg)
    B, T = cfg["B"], spec.max_steps
    env = BatchedEnv(spec, B, env_id0=U.ENV_ID0, auto_reset=False)
    env.enable_obs_bits()
    chk = OracleCheck(cfg, U.oracle_of(cfg), auto_reset=False)
    acts = U.actions(cfg, spec, B)
    rng = np.random.default_rng(5)
    env.reset()
    chk(env, -1, None, None)
    # scheduled masks: random, all-one, all-zero; envs at the time limit are always reset before they step again
    sched = {3: "random", 7: "ones", 12: "zeros", 16: "random", 23: "random", 29: "random"}
    kinds = set()

    def masked_reset(mask, where):
        m, done = mask.astype(bool), chk.o.done.astype(bool)
        if (m & done).any():
            kinds.add("done")
        if (m & ~done & (chk.o.t > 0)).any():
            kinds.add("mid")
        before = {k: getattr(env, k).cpu().numpy().copy() for k in _KEEP if getattr(env, k) is not None}
        env.reset(mask=mask)
        chk.o.reset(mask=mask)
        for k, v in before.items():
            _same(f"unmasked {k}", getattr(env, k).cpu().numpy()[~m], v[~m], where, ref_name="state before the reset")
        chk.state(env, where)

    for s in range(cfg["steps"]):
        env.step(acts[s])
        chk(env, s, acts[s], None)
        expired = chk.o.t >= T
        kind = sched.get(s)
        if kind == "zeros":
            masked_reset(np.zeros(B, np.uint8), f"after the all-zero reset at step {s}")
            kinds.add("zeros")
        if kind == "ones":
            mask = np.ones(B, np.uint8)
            kinds.add("ones")
        elif kind == "random":
            mask = (expired | (rng.random(B) < 0.4)).astype(np.uint8)
        else:
            mask = expired.astype(np.uint8)
        if mask.any():
            masked_reset(mask, f"after the masked reset at step {s}")
    env.check_errors()
    assert {"zeros", "ones", "mid", "done"} <= kinds, kinds
    assert chk.dones > 0


# ---- (d) mask converters ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 31, 33, 64, 65, 255, 256])
def test_mask_pack_unpack_word_edges(n):
    """cm_mask_pack equals numpy's packing with zero padding bits; cm_mask_unpack ignores whatever the padding bits hold."""
    import torch
    from com_marl_b200.policy import CommCategoricalMLPPolicy
    from com_marl_b200.ppo import _unpack_mask
    W = (n + 31) // 32
    rng = np.random.default_rng(n)
    for rows in (1, 7, 45, 97):
        # zeros of both signs, ones and other non-zero values: pack tests != 0
        vals = np.array([0.0, -0.0, 1.0, 1.0, 0.25, -3.0], np.float32)
        dense = vals[rng.integers(0, len(vals), (rows, n))]
        bits = CommCategoricalMLPPolicy.pack_mask(torch.from_numpy(dense).cuda(), n).cpu().numpy().view(np.uint32)
        ref = np.zeros((rows, W * 32), np.uint8)
        ref[:, :n] = dense != 0
        ref = np.packbits(ref, axis=-1, bitorder="little").view("<u4")
        assert np.array_equal(bits, ref), f"pack differs at n={n}, rows={rows}"
        if n % 32:
            assert not (bits[:, -1] >> np.uint32(n % 32)).any(), "padding bits of the last word are not zero"
        # unpack rows whose padding bits hold garbage
        raw = rng.integers(0, 2 ** 32, (rows, W), dtype=np.uint64).astype(np.uint32)
        got = _unpack_mask(torch.from_numpy(raw.view(np.int32)).cuda(), n).cpu().numpy()
        cols = np.arange(n)
        want = ((raw[:, cols >> 5] >> (cols & 31).astype(np.uint32)) & 1).astype(np.float32)
        assert np.array_equal(got, want), f"unpack differs at n={n}, rows={rows}"
