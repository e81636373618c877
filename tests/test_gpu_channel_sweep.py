"""Per-env channel conditions: one launch of env_kernel's table instantiation (cm_env_desc.conds) against one uniform
launch per condition, the oracle, masked resets, forced lane groups, RolloutEngine / eval_sweep against standalone runs,
and the error paths.  The tests at the top need no GPU: ScenarioSpec.with_channel and the checks of a condition list."""
import numpy as np
import pytest

import channel_sweep_util as U

gpu = pytest.mark.gpu


# ---- host side: with_channel and the condition list ------------------------------------------------------------------
def test_with_channel_applies_init_communication_rules():
    from com_marl_b200 import _native as N
    spec = U.base_spec("pp_n32")                                 # map 20
    assert spec.with_channel(pl=0).channel == N.CH_FC
    assert spec.with_channel(pl=1).channel == N.CH_FL
    iid = spec.with_channel(pl=0.3)
    assert iid.channel == N.CH_IID and iid.p_loss == 0.3
    assert spec.with_channel(rcom=18).rcom == 18 and spec.with_channel(rcom=19).rcom == 0   # Rcom + 1 >= map collapses
    ge = spec.with_channel(pl=0.3, channel_type="GE", pgb=0.1, pbg=0.2, ge_init=-1)
    assert (ge.channel, ge.pgb, ge.pbg, ge.ge_init) == (N.CH_GE, 0.1, 0.2, -1)
    assert spec.with_channel() == spec and spec.with_channel(pl=0.3) is not spec
    with pytest.raises(ValueError):
        spec.with_channel(pl=1.5)
    with pytest.raises(ValueError):
        U.base_spec("pp_n32", loss_apply=0).with_channel(channel_type="GE", ge_init=-1)


def test_from_params_equals_with_channel():
    """from_params reads the te* parameters in test mode through with_channel"""
    from com_marl_b200.scenario import ScenarioSpec
    for over in (dict(tepl=0), dict(tepl=1), dict(tepl=0.25, teRcom=3), dict(tepl=0.25, teRcom=40), dict(GE_INIT=-1, Pgb=0.3)):
        p = U.params_of("pp_n32", **over)
        ct = "GE" if "GE_INIT" in over else None
        got = ScenarioSpec.from_params("pp", p, seed=U.SEED, channel_type=ct)
        want = U.base_spec("pp_n32").with_channel(pl=p["tepl"], rcom=p["teRcom"], channel_type=ct, pgb=p["Pgb"],
                                                    pbg=p["Pbg"], ge_init=p["GE_INIT"])
        assert got == want, over


def test_condition_list_errors():
    from com_marl_b200.envs import check_conditions
    spec = U.base_spec("pp_n32")
    conds = U.conditions(spec, U.TABLE)
    assert check_conditions(spec, conds, 9 * 5) == conds and check_conditions(spec, None, 7) is None
    other = U.base_spec("pp_n32", max_env_steps=11).with_channel(pl=0.3)
    with pytest.raises(ValueError, match="outside the channel"):
        check_conditions(spec, conds + [other], 10 * 5)
    seeded = U.conditions(spec, U.TABLE[:2])
    seeded[1].seed += 1
    with pytest.raises(ValueError, match="outside the channel"):
        check_conditions(spec, seeded, 4)
    with pytest.raises(ValueError, match="between 1 and 256"):
        check_conditions(spec, [spec.with_channel(pl=0.5)] * 257, 257)
    with pytest.raises(ValueError, match="between 1 and 256"):
        check_conditions(spec, [], 4)
    with pytest.raises(ValueError, match="evenly"):
        check_conditions(spec, conds, 9 * 5 + 1)


# ---- 1. mixed launch == uniform launches ------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("size", list(U.SIZES))
def test_mixed_equals_uniform(size):
    """Every output and the whole state of each condition's block equals a uniform env of that condition, after every
    auto-reset step, over at least three episodes per env."""
    spec = U.base_spec(size)
    _, mixed = U.run_mixed(spec, U.conditions(spec, U.TABLE), 37, 35)
    assert int(mixed.episode.min()) >= 3
    assert np.array_equal(mixed.cond_idx.cpu().numpy(), np.repeat(np.arange(len(U.TABLE)), 37))


@gpu
def test_mixed_equals_uniform_loss_apply0():
    spec = U.base_spec("pp_n32", loss_apply=0)
    _, mixed = U.run_mixed(spec, U.conditions(spec, U.TABLE_LA0), 37, 35)
    assert int(mixed.episode.min()) >= 3


# ---- 2. against the oracle ----------------------------------------------------------------------------------------------
ORACLE_TABLE = [dict(tepl=0), dict(tepl=1), dict(tepl=0.3, teRcom=2), dict(tepl=0.5, teRcom=19),
                dict(ge=dict(Pgb=0.2, Pbg=0.3, GE_INIT=-1, loss_apply=1)), dict(ge=dict(Pgb=0.2, Pbg=0.3, GE_INIT=0, loss_apply=1))]


@gpu
def test_mixed_matches_oracle():
    """Each block, every call, equals OracleVecEnv of that condition (test mode: tepl / teRcom, ge=) under the same ids."""
    import streams
    from test_gpu_env_layouts import OracleCheck
    from oracle import oracle as orc
    from com_marl_b200.envs import BatchedEnv
    from com_marl_b200.scenario import ScenarioSpec
    E, steps = 37, 30
    conds, checks = [], []
    for k, t in enumerate(ORACLE_TABLE):
        t = dict(t)
        ge = t.pop("ge", None)
        if ge:
            t.update(Pgb=ge["Pgb"], Pbg=ge["Pbg"], GE_INIT=ge["GE_INIT"])
        p = U.params_of("pp_n32", **t)
        conds.append(ScenarioSpec.from_params("pp", p, seed=U.SEED, channel_type="GE" if ge else None))
        checks.append(OracleCheck(None, orc.OracleVecEnv(orc.spec_from_params("pp", p, seed=U.SEED, ge=ge), E, env_id0=k * E)))
    env = BatchedEnv(conds[0], E * len(conds), conditions=conds)
    env.enable_obs_bits()
    views = [env.slice(k * E, (k + 1) * E) for k in range(len(conds))]
    acts = streams.actions(U.ACT_SEED, (steps, env.B, env.n))
    env.reset()
    for v, c in zip(views, checks):
        c(v, -1, None, None)
    for s in range(steps):
        env.step(acts[s])
        for k, (v, c) in enumerate(zip(views, checks)):
            c(v, s, acts[s][k * E:(k + 1) * E], None)
    env.check_errors()
    assert all(c.dones >= 2 * E for c in checks)


# ---- 3. injected uniforms, masked resets, forced lane groups ---------------------------------------------------------------
_DEFAULT = {}


@gpu
@pytest.mark.parametrize("size,inj", U.FORCED, ids=[f"{s}-{'inj' if i else 'gen'}" for s, i in U.FORCED])
def test_forced_configs_equal_uniform(size, inj):
    """The configurations the forced-group test replays, mixed == uniform in this process (co_n54: injected uniforms
    sized for the largest plane count, read by IID and GE entries alike)."""
    spec = U.base_spec(size)
    _DEFAULT[f"{size}_{inj}"] = U.run_mixed(spec, U.conditions(spec, U.TABLE), U.FORCED_E, U.FORCED_STEPS, inj=inj)[0]


@gpu
def test_injected_uniforms_pp_n200():
    spec = U.base_spec("pp_n200")
    U.run_mixed(spec, U.conditions(spec, [U.TABLE[3], U.TABLE[8], U.TABLE[0]]), 5, 10, inj=True)


@gpu
@pytest.mark.parametrize("group", [4, 16, 32])
def test_forced_group_equals_default(group):
    """CM_ENV_GROUP = group in a spawned process: the mixed env's per-call digests equal the default group's."""
    forced = U.run_forced(group)
    for size, inj in U.FORCED:
        key = f"{size}_{inj}"
        if key not in _DEFAULT:
            spec = U.base_spec(size)
            _DEFAULT[key] = U.run_mixed(spec, U.conditions(spec, U.TABLE), U.FORCED_E, U.FORCED_STEPS, inj=inj)[0]
        ref, got = _DEFAULT[key], forced[key]
        assert len(ref) == len(got)
        for s, (a, b) in enumerate(zip(ref, got)):
            assert a == b, f"{key}: group {group} differs at call {s}: {[k for k in a if a[k] != b.get(k)]}"


@gpu
def test_masked_reset_mixed():
    """reset(mask) of a mixed env: masked envs restart exactly like their uniform envs (GE initial states per entry),
    the others keep their state byte for byte."""
    import streams
    from com_marl_b200.envs import BatchedEnv
    spec = U.base_spec("pp_n32")
    conds = U.conditions(spec, U.TABLE)
    E, K = 23, len(conds)
    B = E * K
    mixed = BatchedEnv(spec, B, auto_reset=False, conditions=conds)
    unis = [BatchedEnv(c, E, env_id0=k * E, auto_reset=False) for k, c in enumerate(conds)]
    acts = streams.actions(U.ACT_SEED, (30, B, spec.n_agents))
    rng = np.random.default_rng(3)
    mixed.reset()
    for u in unis:
        u.reset()
    resets = 0
    for s in range(30):
        mixed.step(acts[s])
        for k, u in enumerate(unis):
            u.step(acts[s][k * E:(k + 1) * E])
        U.compare(mixed, unis, E, f"at step {s}")
        mask = ((mixed.step_count.cpu().numpy() >= spec.max_steps) | (rng.random(B) < 0.3)).astype(np.uint8)
        before = U.arrays(mixed)
        mixed.reset(mask=mask)
        for k, u in enumerate(unis):
            u.reset(mask=mask[k * E:(k + 1) * E])
        U.compare(mixed, unis, E, f"after the masked reset at step {s}")
        after, keep = U.arrays(mixed), mask == 0
        for name in U.STATE:
            if name in before and name != "stats":
                assert np.array_equal(after[name][keep], before[name][keep]), f"unmasked {name} changed at step {s}"
        resets += int(mask.sum())
    mixed.check_errors()
    assert resets > B


# ---- 4. rollout -----------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("kind,chunks", [("comm", 3), ("dec", 2), ("cent", 2)])
def test_rollout_groups_cut_conditions(kind, chunks):
    """RolloutEngine(conditions=..., groups=3), whose groups cut through conditions, == one standalone engine per
    condition: sampled actions, probabilities and rewards of every step."""
    from com_marl_b200.rollout import RolloutEngine, make_policy
    spec = U.base_spec("pp_n32")
    conds = U.conditions(spec, [U.TABLE[0], dict(pl=0.3, rcom=2), U.TABLE[8], U.TABLE[1]])
    E, K = 37, len(conds)
    pol = make_policy(spec, kind=kind)
    if kind == "comm":
        assert pol.uses_tensor_cores()
    eng = RolloutEngine(spec, pol, E * K, ring=8, groups=3, conditions=conds)
    cuts = [r[0] for r in eng._ranges[1:]]
    assert any(c % E for c in cuts), cuts
    alone = [RolloutEngine(c, pol, E, env_id0=k * E, ring=8) for k, c in enumerate(conds)]
    eng.reset()
    for a in alone:
        a.reset()
    for ch in range(chunks):
        eng.run_chunk()
        for a in alone:
            a.run_chunk()
        for key in ("actions", "probs", "reward", "done"):
            got = eng.traj[key].cpu().numpy()
            for k, a in enumerate(alone):
                assert np.array_equal(got[:, k * E:(k + 1) * E], a.traj[key].cpu().numpy()), f"{kind}: {key} of condition {k}, chunk {ch}"
    eng.env.check_errors()


# ---- 5. eval_sweep ------------------------------------------------------------------------------------------------------
@gpu
def test_eval_sweep_equals_eval_model():
    from com_marl_b200.evaluate import eval_model, eval_sweep
    from com_marl_b200.rollout import make_policy
    spec = U.base_spec("pp_n4", max_env_steps=40)
    conds = U.conditions(spec, [dict(pl=0.5, rcom=2), U.TABLE[5], U.TABLE[6], U.TABLE[1], dict(pl=0.1, rcom=1)])
    pol = make_policy(spec)
    E = 20
    res = eval_sweep(spec, pol, conds, n_eval_episodes=E, max_env_steps=30, seed=3, groups=2, chunk=10, return_trajectory=True)
    assert len(res) == len(conds)
    for k, c in enumerate(conds):
        want = eval_model(c, pol, n_eval_episodes=E, max_env_steps=30, seed=3, groups=1, chunk=10, return_trajectory=True,
                          env_id0=k * E)
        got = res[k]
        assert got[0] == want[0] and got[1] == want[1] and got[2] == want[2] and got[3] == want[3], f"condition {k}"
        for name in want[4]:
            assert np.array_equal(got[4][name], want[4][name]), (k, name)
        assert np.array_equal(got[5], want[5])
    fully = res[1][0][0][1]["nodeDeg"]
    assert all(x == spec.n_agents for x in fully)                  # the collapsed Rcom reports n, like the reference


# ---- 6. errors ----------------------------------------------------------------------------------------------------------
@gpu
def test_constructor_errors():
    from com_marl_b200.envs import BatchedEnv
    spec = U.base_spec("pp_n4")
    conds = U.conditions(spec, U.TABLE[:3])
    with pytest.raises(ValueError):
        BatchedEnv(spec, 10, conditions=conds)
    with pytest.raises(ValueError):
        BatchedEnv(spec, 6, conditions=conds[:1] + [U.base_spec("pp_n4", max_env_steps=11)])
    with pytest.raises(ValueError):
        BatchedEnv(spec, 257, conditions=[conds[0]] * 257)


@gpu
def test_table_entry_ge_init_minus1_with_loss_apply0_unsupported():
    from com_marl_b200 import _native as N
    from com_marl_b200.envs import BatchedEnv
    spec = U.base_spec("pp_n4", loss_apply=0)
    env = BatchedEnv(spec, 4, conditions=U.conditions(spec, [U.TABLE[0], dict(channel_type="GE", ge_init=1)]))
    env.reset()
    env._conds_host[1].ge_init = -1                                  # the host mirror the call validates
    with pytest.raises(N.NativeError) as e:
        env.step(np.zeros((4, spec.n_agents), np.int8))
    assert e.value.code == N.CM_EUNSUPPORTED


@gpu
def test_cond_idx_out_of_range_is_reported():
    from com_marl_b200 import _native as N
    from com_marl_b200.envs import BatchedEnv
    spec = U.base_spec("pp_n4")
    env = BatchedEnv(spec, 6, conditions=U.conditions(spec, U.TABLE[:3]))
    env.reset()
    env.check_errors()
    env.cond_idx[4] = 200
    env.step(np.zeros((6, spec.n_agents), np.int8))
    with pytest.raises(N.NativeError) as e:
        env.check_errors()
    assert e.value.code == N.CM_EINVAL
