"""CENT and Obs-DP forwards of cm_policy_forward against the float64 oracle at the shapes where their kernels can go wrong:
every K of the CENT first-layer walk (panel counts 1..10 continuously, every K mod 32 / K mod 4) on both maths, every team
size of both kinds, every Obs-DP width, persistent-grid walks of several tiles per CTA, the env's input value set and
all-zero rows, a misaligned observation pointer, the in-kernel random stream, production batches past 2^31 observation
elements and at the tensor-core kernel's row limit, and the tensor-core weights after parameter updates (in place, by
load_state_dict, by FlatAdam, through p.data with a forced refresh and by a fused PPO round) inside captured rollout graphs.  Helpers: tests/policy_kinds_util.py."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

import policy_kinds_util as U
from oracle import oracle as orc

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for (kind, math), r in sorted(U.REPORT.items()):
        print(f"\npolicy kinds: {kind} math={math}: largest error / tolerance {r:.3f}")


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _run_full(pol, obs, av, rng, lbl, ref=None, w=None):
    """one call with host inputs, sampling uniforms drawn here; compared on every env"""
    B, n = obs.shape[:2]
    u = rng.random((B, n), dtype=np.float32)
    got = U.host(U.forward(pol, torch.from_numpy(obs).cuda(), torch.from_numpy(U.avail_bits(av)).cuda(), torch.from_numpy(u).cuda()))
    if ref is None:
        ref = U.oracle(pol, U.state(pol) if w is None else w, obs, av)
    tol = U.cent_tc_tol(n * pol._dec_obs_dim) if U.kind_of(pol) == "cent" and U.math_of(pol) == "tc" else U.TOL
    U.check(U.label(pol, B, lbl), got, ref, u, key=(U.kind_of(pol), U.math_of(pol)), tol=tol)
    return ref


def _need(nbytes, what):
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes * 1.15:
        pytest.skip(f"{what} needs {nbytes / 2**30:.1f} GiB of device memory, {free / 2**30:.1f} GiB free")


# ---- 1. the CENT first-layer walk: every K -------------------------------------------------------------------------------
WALK = U.walk_cases()
WALK_GROUPS = 8


@pytest.mark.parametrize("group", range(WALK_GROUPS))
def test_cent_first_layer_every_K(group):
    """B = 421: 4 first-layer tiles of 128 (the last 37 rows) and 7 tiles of 64; tanh / relu and the input domains alternate"""
    B = 421
    for i in range(group, len(WALK), WALK_GROUPS):
        n, D = WALK[i]
        rng = np.random.default_rng(1000 + i)
        obs, av = U.observations(B, n, D, U.DOMAINS[i % 3], rng), U.avail(B, n, rng)
        pol = U.cent_policy(n, D, relu=bool(i % 2), math="fp32", seed=i)
        ref = _run_full(pol, obs, av, rng, f"relu={i % 2} {U.DOMAINS[i % 3]}")
        pol.math = "tc"
        _run_full(pol, obs, av, rng, f"relu={i % 2} {U.DOMAINS[i % 3]}", ref=ref)


def test_walk_covers_the_panel_pipeline():
    """the K table reaches every panel count 1..10, every K mod 32 and K mod 4, and the limits' largest K"""
    Ks = [n * D for n, D in WALK]
    assert set(range(1, 11)) <= {U.panels(K) for K in Ks}
    assert {K % 32 for K in Ks if K <= 320} == set(range(32))
    assert max(Ks) == 32768 and all(n <= 256 and D <= 128 for n, D in WALK)


# ---- 2. / 3. every team size, every Obs-DP width -----------------------------------------------------------------------------
TEAM_GROUPS = 8


@pytest.mark.parametrize("group", range(TEAM_GROUPS))
def test_cent_every_team_size(group):
    """n = 1 .. 256 at D = 53 (every n mod 16 of the output layer's passes, NO = 5n), both maths, ragged batches"""
    for n in range(1 + group, 257, TEAM_GROUPS):
        B = 131 + 7 * (n % 9)
        rng = np.random.default_rng(n)
        obs, av = U.observations(B, n, 53, U.DOMAINS[n % 3], rng), U.avail(B, n, rng)
        pol = U.cent_policy(n, 53, relu=bool(n % 2), math="tc", seed=3 * n)
        ref = _run_full(pol, obs, av, rng, U.DOMAINS[n % 3])
        pol.math = "fp32"
        _run_full(pol, obs, av, rng, U.DOMAINS[n % 3], ref=ref)


@pytest.mark.parametrize("group", range(TEAM_GROUPS))
def test_dec_every_team_size(group):
    for n in range(1 + group, 257, TEAM_GROUPS):
        B = 37 + n % 11
        rng = np.random.default_rng(5000 + n)
        obs, av = U.observations(B, n, 53, U.DOMAINS[n % 3], rng), U.avail(B, n, rng)
        _run_full(U.dec_policy(n, 53, seed=n), obs, av, rng, U.DOMAINS[n % 3])


@pytest.mark.parametrize("group", range(4))
def test_dec_every_width(group):
    """D = 1 .. 128 at n = 3: every K padding / panel count of make_tc_plan's Dec mode; 903 rows = 7 tiles + 7 rows"""
    B, n = 301, 3
    for D in range(1 + group, 129, 4):
        rng = np.random.default_rng(7000 + D)
        obs, av = U.observations(B, n, D, U.DOMAINS[D % 3], rng), U.avail(B, n, rng)
        _run_full(U.dec_policy(n, D, seed=D), obs, av, rng, U.DOMAINS[D % 3])


@pytest.mark.parametrize("n", [1, 3, 33, 200, 256])
def test_dec_persistent_walk(n):
    """every persistent CTA (2 per SM) walks at least three tiles, the last one ragged; checked on the whole first and last
    tile, the first tile of every CTA's second round and a stride sample"""
    D, sms = 53, _sms()
    B = U.rows_batch(n, sms)
    assert B * n >= 3 * 2 * sms * U.TC_ROWS
    pol = U.dec_policy(n, D, seed=n + 1)
    obs = U.device_obs(B, n, D, seed=n)
    bits = U.device_avail_bits(B, n, seed=n + 1)
    u = torch.rand((B, n), device="cuda", generator=torch.Generator(device="cuda").manual_seed(n + 2))
    out = U.forward(pol, obs, bits, u)
    envs = U.dec_sample_envs(B, n, sms)
    idx = torch.as_tensor(envs, device="cuda")
    got = U.host(out, envs)
    ref = U.oracle(pol, U.state(pol), obs.index_select(0, idx).cpu().numpy(), U.unpack_avail(bits.index_select(0, idx).cpu().numpy()))
    U.check(U.label(pol, B, f"sampled {len(envs)} envs"), got, ref, u.index_select(0, idx).cpu().numpy(), envs, key=("dec", "tc"))


# ---- 5. misaligned observation pointer ------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,n,D", [("cent", 4, 21), ("cent", 32, 53), ("cent", 7, 128), ("dec", 5, 53), ("dec", 3, 128),
                                      ("dec", 33, 7)])
def test_misaligned_obs_pointer_is_bit_identical(kind, n, D):
    """obs as a view 4 bytes into a larger buffer: for CENT with K % 4 == 0 only the pointer selects the 4-byte cp.async path,
    for Obs-DP the misaligned head of stage_obs; the outputs equal the aligned call's bit for bit (and the oracle)"""
    B = 517
    rng = np.random.default_rng(n * 131 + D)
    obs, av = U.observations(B, n, D, "env", rng), U.avail(B, n, rng)
    if kind == "cent":
        assert (n * D) % 4 == 0
    buf = torch.zeros(B * n * D + 4, device="cuda")
    aligned, shifted = buf[:B * n * D].view(B, n, D), buf[1:1 + B * n * D].view(B, n, D)
    assert aligned.data_ptr() % 16 == 0 and shifted.data_ptr() % 16 == 4
    bits = torch.from_numpy(U.avail_bits(av)).cuda()
    u = torch.from_numpy(rng.random((B, n), dtype=np.float32)).cuda()
    maths = ("tc", "fp32") if kind == "cent" else ("tc",)
    pol = U.cent_policy(n, D, math="tc", seed=n) if kind == "cent" else U.dec_policy(n, D, seed=n)
    ref = U.oracle(pol, U.state(pol), obs, av)
    for math in maths:
        pol.math = math
        aligned.copy_(torch.from_numpy(obs))
        base = U.host(U.forward(pol, aligned, bits, u))
        buf.zero_()
        shifted.copy_(torch.from_numpy(obs))
        got = U.host(U.forward(pol, shifted, bits, u))
        U.same(U.label(pol, B, "obs at a 4-byte offset"), got, base)
        U.check(U.label(pol, B, "obs at a 4-byte offset"), got, ref, u.cpu().numpy(), key=(kind, math))


# ---- 6. the in-kernel random stream ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,n", [("cent", 5), ("cent", 17), ("cent", 32), ("cent", 200), ("dec", 3), ("dec", 54), ("dec", 200)])
def test_in_kernel_draw_matches_the_stream_spec(kind, n):
    """sample_u = None: the actions are the inverse CDF of the kernel's probabilities for the draws of
    philox(seed; env_id0 + env, tick, 4 | episode << 8, il >> 2), word il & 3, u24 — with non-zero tick / episode / env_id0"""
    D, B, env_id0 = 53, 300, 987_654
    rng = np.random.default_rng(n + (0 if kind == "cent" else 99))
    obs, av = U.observations(B, n, D, "env", rng), U.avail(B, n, rng)
    tick = rng.integers(1, 2**31 - 1, B).astype(np.int32)
    episode = rng.integers(1, 2**24, B).astype(np.int32)
    pol = U.cent_policy(n, D, math="tc", seed=n) if kind == "cent" else U.dec_policy(n, D, seed=n)
    envs = U.sample_envs(B, 64, stride=40)
    ref = U.oracle(pol, U.state(pol), obs[envs], av[envs])
    u = U.action_u(pol.seed, env_id0, envs, tick, episode, n)
    for math in (("tc", "fp32") if kind == "cent" else ("tc",)):
        pol.math = math
        out = U.forward(pol, torch.from_numpy(obs).cuda(), torch.from_numpy(U.avail_bits(av)).cuda(), None,
                        torch.from_numpy(tick).cuda(), torch.from_numpy(episode).cuda(), env_id0=env_id0)
        U.check(U.label(pol, B, f"in-kernel draw, env_id0={env_id0}"), U.host(out, envs), ref, u, envs, key=(kind, math))


# ---- 7. production batches and index widths -----------------------------------------------------------------------------------
def _cent_sampled(pol, obs, bits, u, envs, lbl):
    idx = torch.as_tensor(envs, device="cuda")
    w = U.state(pol)
    ref = U.oracle(pol, w, obs.index_select(0, idx).cpu().numpy(), U.unpack_avail(bits.index_select(0, idx).cpu().numpy()))
    uh = u.index_select(0, idx).cpu().numpy()
    B = obs.shape[0]
    for math in ("fp32", "tc"):
        pol.math = math
        out = U.forward(pol, obs, bits, u)
        U.check(U.label(pol, B, lbl), U.host(out, envs), ref, uh, envs, key=("cent", math))
        del out


@pytest.mark.parametrize("n,D,B", [(32, 53, 65536), (200, 53, 2048), (200, 53, 204800)], ids=["c3", "c5", "past_2^31"])
def test_cent_production_batches(n, D, B):
    """C3 / C5 batches and n = 200, D = 53, B = 204 800: 2.17e9 observation floats (8.7 GB), sampled envs whose row * K is
    past 2^31 and the last tile included; fp32 and tc"""
    K = n * D
    _need(B * K * 4 + B * n * 5 * 8 + B * n * 5 + B * 128 * 4, f"CENT n={n} D={D} B={B}")
    pol = U.cent_policy(n, D, math="tc", seed=n)
    obs = U.device_obs(B, n, D, seed=B)
    bits = U.device_avail_bits(B, n, seed=B + 1)
    u = torch.rand((B, n), device="cuda", generator=torch.Generator(device="cuda").manual_seed(B + 2))
    envs = U.sample_envs(B, U.L1_ROWS)
    if B * K > 2**31:
        assert (envs * K > 2**31).sum() >= 128 and envs[-1] == B - 1
    _cent_sampled(pol, obs, bits, u, envs, f"sampled {len(envs)} envs")
    del obs, bits, u
    torch.cuda.empty_cache()


def _limit_case(pol, B, n, D, masks):
    """accepted and correct at n_envs * n = 2^23 (sampled, last tile included); one env more is CM_EUNSUPPORTED and leaves
    sentinel-filled outputs untouched"""
    from com_marl_b200 import _native as N
    obs = U.device_obs(B + 1, n, D, seed=n)
    bits = U.device_avail_bits(B + 1, n, seed=n + 1)
    u = torch.rand((B + 1, n), device="cuda", generator=torch.Generator(device="cuda").manual_seed(n + 2))
    adj, chan = masks(B + 1) if masks else (None, None)
    out = dict(logits=torch.full((B + 1, n, 5), -7.0, device="cuda"), probs=torch.full((B + 1, n, 5), -7.0, device="cuda"),
               actions=torch.full((B + 1, n), -7, dtype=torch.int8, device="cuda"))
    desc, io = pol._call_structs(obs, adj, chan, bits, u, None, None, False, out["probs"], out["logits"], None, out["actions"], 0, 0)
    assert N.lib().cm_policy_forward(C.byref(desc), C.byref(io), N.stream_ptr()) == N.CM_EUNSUPPORTED
    torch.cuda.synchronize()
    assert bool((out["probs"] == -7).all()) and bool((out["logits"] == -7).all()) and bool((out["actions"] == -7).all())
    kw = dict(adj_bits=adj[:B], chan_bits=chan[:B]) if masks else {}
    sl = {k: v[:B] for k, v in out.items()}
    pol.act_device(obs[:B], avail_bits=bits[:B], sample_u=u[:B], **kw, **sl)
    pol.check_errors()
    assert bool((out["probs"][B] == -7).all())
    envs = U.sample_envs(B, max(1, U.TC_ROWS // n))
    idx = torch.as_tensor(envs, device="cuda")
    ho = lambda t: t.index_select(0, idx).cpu().numpy()  # noqa: E731
    got = {k: ho(v) for k, v in sl.items()}
    return got, ho(obs), U.unpack_avail(ho(bits)), ho(u), envs, (ho(adj), ho(chan)) if masks else None


def test_tc_row_limit_dec():
    """Obs-DP at n = 32, D = 128, B = 262 144: exactly 2^23 agent rows"""
    n, D, B = 32, 128, 1 << 18
    _need((B + 1) * n * (D * 4 + 5 * 8 + 1 + 4 + 1), "Obs-DP at 2^23 rows")
    pol = U.dec_policy(n, D, seed=5)
    got, obs, av, u, envs, _ = _limit_case(pol, B, n, D, None)
    U.check(U.label(pol, B, "2^23 rows"), got, U.oracle(pol, U.state(pol), obs, av), u, envs, key=("dec", "tc"))


def test_tc_row_limit_comm():
    """Comm-DP at n = 64 (env slots of 64 tile rows), B = 131 072: exactly 2^23 agent rows, random neighbour / channel masks"""
    import policy_path_util as P
    n, D, L, B = 64, 53, 2, 1 << 17
    _need((B + 1) * n * (D * 4 + 5 * 8 + 1 + 4 + 1 + 8 * (L + 1)), "Comm-DP at 2^23 rows")
    w = P.weights(n, D, L, seed=3)
    pol = P.policy(w, n, D, L, "tc")
    self_bits = torch.zeros((n, 2), dtype=torch.int64)
    self_bits[torch.arange(n), torch.arange(n) // 32] = 1 << (torch.arange(n) % 32)
    self_bits = self_bits.to(torch.int32).cuda()

    def masks(Bm):
        g = torch.Generator(device="cuda").manual_seed(17)
        adj = torch.randint(-2**31, 2**31, (Bm, n, 2), dtype=torch.int32, device="cuda", generator=g) | self_bits
        chan = torch.randint(-2**31, 2**31, (Bm, L, n, 2), dtype=torch.int32, device="cuda", generator=g) | self_bits
        return adj, chan

    got, obs, av, u, envs, (adj, chan) = _limit_case(pol, B, n, D, masks)
    dense = lambda b: ((b.view(np.uint32)[..., np.arange(n) // 32] >> (np.arange(n) % 32).astype(np.uint32)) & 1).astype(np.uint8)  # noqa: E731
    ref = orc.policy_forward(w, obs, av, dense(adj), dense(chan), dtype=np.float64)[:2]
    U.check(f"comm math=tc n={n} D={D} L={L} B={B} 2^23 rows", got, ref, u, envs, key=("comm", "tc"))


def test_cent_env_agent_limit_rejected():
    """n_envs * n > 2^30 is CM_EUNSUPPORTED before anything else is looked at; 2^30 itself passes the check (and then meets
    the missing tensor-core operands: CM_EINVAL, still no launch)"""
    from com_marl_b200 import _native as N
    small = torch.zeros(16, device="cuda")                  # (only the pointer checks before the size check look at these)
    for n_envs, expect in (((1 << 22) + 1, N.CM_EUNSUPPORTED), (1 << 22, N.CM_EINVAL)):
        desc = N.PolicyDesc(256, 1, 1, 0, 0, 1, 1, 0, N.POLICY_CENT, 0)
        io = N.PolicyIO()
        io.n_envs, io.weights, io.obs, io.probs = n_envs, N.ptr(small), N.ptr(small), N.ptr(small)
        assert N.lib().cm_policy_forward(C.byref(desc), C.byref(io), N.stream_ptr()) == expect, n_envs


# ---- 8. the tensor-core weights after updates ------------------------------------------------------------------------------------
def _perturb(pol, how, rng):
    if how == "in place":
        with torch.no_grad():
            for p in pol.parameters():
                p.add_(torch.from_numpy(rng.normal(0, 0.05, tuple(p.shape)).astype(np.float32)).to(p.device))
    elif how == "p.data":
        # a write through .data bypasses the version counters: the caller forces the refresh
        for p in pol.parameters():
            p.data.add_(torch.from_numpy(rng.normal(0, 0.05, tuple(p.shape)).astype(np.float32)).to(p.device))
        pol.refresh_weights(force=True)
    elif how == "load_state_dict":
        pol.load_state_dict({k: v + torch.from_numpy(rng.normal(0, 0.05, tuple(v.shape)).astype(np.float32)).to(v.device)
                             for k, v in pol.state_dict().items()})
    else:
        from com_marl_b200.ppo import FlatAdam
        opt = getattr(pol, "_test_opt", None) or FlatAdam(pol, lr=0.02)
        pol._test_opt = opt
        opt.grad.copy_(torch.from_numpy(rng.normal(0, 1, opt.grad.numel()).astype(np.float32)))
        opt.step()


@pytest.mark.parametrize("kind", ["cent", "dec"])
def test_weight_refresh_in_captured_rollout(kind):
    """a RolloutEngine with one captured graph over 3 env groups; the parameters change in place, by load_state_dict, by a
    FlatAdam step and through p.data (then refresh_weights(force=True)) between chunks, and every recorded step matches the
    oracle WITH THE NEW WEIGHTS, replayed step by step on the oracle env"""
    sys.path.insert(0, GOLDEN)
    import ref_harness
    from com_marl_b200.rollout import RolloutEngine, make_policy
    from com_marl_b200.scenario import ScenarioSpec
    params = ref_harness.scenario_params("pp", 10, 1, 0.08, cap=2, loss=0.2, max_env_steps=25)
    spec = ScenarioSpec.from_params("pp", params, seed=9)
    B = 300
    pol = make_policy(spec, kind=kind)
    if kind == "cent":
        pol.math = "tc"
    assert pol.uses_tensor_cores()
    eng = RolloutEngine(spec, pol, B, ring=6, use_graph=True, groups=3)
    oenv = orc.OracleVecEnv(orc.spec_from_params("pp", params, seed=9), B)
    eng.reset(); oenv.reset()
    rng = np.random.default_rng(4)
    fwd = (lambda w, o: orc.policy_forward_cent(w, o, None, dtype=np.float64)) if kind == "cent" else \
        (lambda w, o: orc.policy_forward_dec(w, o, None, dtype=np.float64))
    for how in (None, None, "in place", "load_state_dict", "FlatAdam", "in place", "p.data"):
        if how:
            _perturb(pol, how, rng)
        w = U.state(pol)
        eng.run_chunk()
        t = {k: v.cpu().numpy() for k, v in eng.traj.items()}
        for k in range(eng.K):
            assert np.array_equal(t["obs"][k], oenv.obs)
            ref_probs = fwd(w, oenv.obs)[1]
            err = np.abs(t["probs"][k] - ref_probs).max()
            assert err <= U.TOL, f"{kind} math=tc after {how}: step {k} probs off by {err:.2e}"
            U.REPORT[(kind, "tc")] = max(U.REPORT.get((kind, "tc"), 0.0), float(err) / U.TOL)
            assert np.array_equal(t["actions"][k], oenv.sample_actions(t["probs"][k]))
            oenv.step(t["actions"][k])
            assert np.array_equal(t["reward"][k], oenv.reward) and np.array_equal(t["done"][k], oenv.done)
    eng.env.check_errors(); pol.check_errors()


def test_cent_trainer_round_then_tc_rollout():
    """DeviceTrainer(kind='cent', fused=True) on PP map 20, sensing 2, 32 agents (K = 1 696: 'auto' picks tc): after one round
    the next rollout's probabilities match the oracle on the updated state_dict"""
    from com_marl_b200.scenario import ScenarioSpec
    from com_marl_b200.train import DeviceTrainer
    spec = ScenarioSpec.from_cli("pp", 20, 2, 0.08, cap=4, loss=0.2, seed=7)
    assert spec.n_agents * spec.obs_dim == 1696
    tr = DeviceTrainer(spec, 256, kind="cent", fused=True)
    assert tr.policy.math == "tc" and tr.algo._fused is not None
    w0 = U.state(tr.policy)
    tr.train_epoch()
    w = U.state(tr.policy)
    assert max(np.abs(w[k] - w0[k]).max() for k in w) > 1e-4
    tr.engine.reset()
    tr.engine.run_chunk()
    obs, probs = tr.engine.traj["obs"], tr.engine.traj["probs"]
    for k in range(tr.engine.K):
        ref_probs = orc.policy_forward_cent(w, obs[k].cpu().numpy(), None, dtype=np.float64)[1]
        err = np.abs(probs[k].cpu().numpy() - ref_probs).max()
        assert err <= U.TOL, f"cent math=tc n=32 D=53 K=1696 B=256 after a fused PPO round: step {k} probs off by {err:.2e}"
        U.REPORT[("cent", "tc")] = max(U.REPORT.get(("cent", "tc"), 0.0), float(err) / U.TOL)
