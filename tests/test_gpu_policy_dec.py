"""Obs-DP policy (DecCategoricalMLPPolicy) on the fused tensor-core kernel: golden vectors recorded from the unmodified
reference (tests/golden/make_golden_dec.py), the float64 oracle on large ragged batches, the sampling specification,
the reference call surface, and the device rollout with the Obs-DP policy against the oracle."""
import glob
import json
import os

import numpy as np
import pytest
import torch

from oracle import oracle as orc

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
CASES = sorted(os.path.basename(p)[7:-4] for p in glob.glob(os.path.join(GOLDEN, "decpol_*.npz")))


def _policy(n, D, weights=None, seed=3):
    from com_marl_b200.policy import DecCategoricalMLPPolicy
    from com_marl_b200.spaces import Box, Discrete, EnvSpec
    pol = DecCategoricalMLPPolicy(EnvSpec(Box(np.zeros(n * D), np.ones(n * D)), Discrete(5)), n, seed=seed)
    if weights is not None:
        pol.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in weights.items()})
    return pol


@pytest.mark.parametrize("name", CASES)
def test_dec_policy_kernel_matches_reference_golden(name):
    z = np.load(os.path.join(GOLDEN, f"decpol_{name}.npz"))
    meta = json.loads(str(z["meta"]))
    n, D, B = meta["n"], meta["D"], meta["B"]
    w = {k[3:]: z[k] for k in z.files if k.startswith("w::")}
    pol = _policy(n, D, w)
    assert set(pol.state_dict().keys()) == set(w.keys())            # reference checkpoints load as they are
    obs = torch.from_numpy(z["obs"].reshape(B, n, D)).cuda()
    av = z["avail"].reshape(B, n, 5)
    bits = torch.from_numpy(((av != 0) * np.array([1, 2, 4, 8, 16])).sum(-1).astype(np.uint8)).cuda()
    probs = torch.empty((B, n, 5), device="cuda"); logits = torch.empty((B, n, 5), device="cuda")
    pol.act_device(obs, avail_bits=bits, greedy=True, probs=probs, logits=logits, actions=torch.empty((B, n), dtype=torch.int8, device="cuda"))
    pol.check_errors()
    ref_logits = z["logits"].reshape(B, n, 5)
    assert np.abs(logits.cpu().numpy() - ref_logits).max() <= 1e-5 * max(1.0, np.abs(ref_logits).max())
    assert np.abs(probs.cpu().numpy() - z["probs"].reshape(B, n, 5)).max() <= 1e-5
    # the torch training path (forward / log_likelihood / entropy) is the same formula
    with torch.no_grad():
        dist = pol.forward(torch.from_numpy(z["obs"]).cuda(), torch.from_numpy(z["avail"]).cuda())
    assert np.abs(dist.probs.cpu().numpy() - z["probs"].reshape(B, n, 5)).max() <= 1e-5


@pytest.mark.parametrize("n,D,B", [(3, 29, 16384), (4, 21, 5001), (32, 53, 2048), (54, 77, 777), (200, 53, 300), (1, 5, 100)])
def test_dec_policy_kernel_matches_oracle_batched(n, D, B):
    rng = np.random.default_rng(n * 1000 + D)
    pol = _policy(n, D)
    with torch.no_grad():
        for k, v in pol.state_dict().items():
            if k.endswith("bias"):
                v.copy_(torch.from_numpy(rng.uniform(-0.2, 0.2, size=tuple(v.shape)).astype(np.float32)))
    obs = rng.random((B, n, D), dtype=np.float32)
    avail = (rng.random((B, n, 5)) < 0.9).astype(np.float32)
    avail[..., 4] = 1.0
    bits = torch.from_numpy(((avail != 0) * np.array([1, 2, 4, 8, 16])).sum(-1).astype(np.uint8)).cuda()
    u = rng.random((B, n), dtype=np.float32)
    probs = torch.empty((B, n, 5), device="cuda"); logits = torch.empty((B, n, 5), device="cuda")
    actions = torch.empty((B, n), dtype=torch.int8, device="cuda")
    pol.act_device(torch.from_numpy(obs).cuda(), avail_bits=bits, sample_u=torch.from_numpy(u).cuda(), probs=probs, logits=logits, actions=actions)
    pol.check_errors()
    w = {k: v.cpu().numpy() for k, v in pol.state_dict().items()}
    ref_logits, ref_probs = orc.policy_forward_dec(w, obs, avail, dtype=np.float64)
    assert np.abs(logits.cpu().numpy() - ref_logits).max() <= 1e-5 * max(1.0, np.abs(ref_logits).max())
    assert np.abs(probs.cpu().numpy() - ref_probs).max() <= 1e-5
    # sampling == inverse CDF of the kernel's own probabilities (sequential fp32 cumulative sum)
    pr = probs.cpu().numpy()
    cdf = np.zeros_like(pr)
    acc = np.zeros(pr.shape[:-1], dtype=np.float32)
    for a in range(5):
        acc = (acc + pr[..., a]).astype(np.float32)
        cdf[..., a] = acc
    exp = (u[..., None] >= cdf).sum(-1)
    last = 4 - np.argmax((pr > 0)[..., ::-1], axis=-1)
    exp = np.where(exp > 4, last, exp)
    assert np.array_equal(actions.cpu().numpy(), exp)


def test_dec_get_actions_contract():
    n, D, B = 4, 21, 7
    pol = _policy(n, D)
    rng = np.random.default_rng(0)
    obs = rng.random((B, n * D), dtype=np.float32)
    acts, infos = pol.get_actions(obs, np.ones((B, n * 5), dtype=np.float32))
    assert acts.shape == (B, n) and acts.dtype == np.int64 and len(infos["action_probs"]) == B
    g, ginf = pol.get_actions(obs, np.ones((B, n * 5), dtype=np.float32), greedy=True)
    assert np.array_equal(g, np.argmax(np.stack(ginf["action_probs"]), axis=-1))
    a1, _ = pol.get_actions(obs[0], np.ones(n * 5, dtype=np.float32))
    assert a1.shape == (n,)
    assert pol.comm is False and pol.vectorized and not pol.recurrent


@pytest.mark.parametrize("scen", ["pp", "co"])
def test_dec_rollout_matches_oracle(scen):
    """device rollout with the Obs-DP policy: every step replayed on the oracle with the kernel's own actions"""
    import sys
    sys.path.insert(0, GOLDEN)
    import ref_harness
    from com_marl_b200.rollout import RolloutEngine, make_policy
    from com_marl_b200.scenario import ScenarioSpec
    over = {"max_env_steps": 25}
    params = ref_harness.scenario_params(scen, 10, 1, 0.08 if scen == "pp" else 0.03, cap=2, loss=0.2, **over)
    spec = ScenarioSpec.from_params(scen, params, seed=9)
    B, n = 300, spec.n_agents
    pol = make_policy(spec, kind="dec")
    eng = RolloutEngine(spec, pol, B, ring=6, use_graph=True, groups=3)
    oenv = orc.OracleVecEnv(orc.spec_from_params(scen, params, seed=9), B)
    eng.reset(); oenv.reset()
    w = {k: v.cpu().numpy() for k, v in pol.state_dict().items()}
    for chunk in range(6):
        eng.run_chunk()
        t = {k: v.cpu().numpy() for k, v in eng.traj.items()}
        for k in range(eng.K):
            assert np.array_equal(t["obs"][k], oenv.obs)
            _, ref_probs = orc.policy_forward_dec(w, oenv.obs, None)
            assert np.abs(t["probs"][k] - ref_probs).max() <= 1e-5
            assert np.array_equal(t["actions"][k], oenv.sample_actions(t["probs"][k]))
            oenv.step(t["actions"][k])
            assert np.array_equal(t["reward"][k], oenv.reward) and np.array_equal(t["done"][k], oenv.done)
    eng.env.check_errors(); pol.check_errors()


def test_dec_sampler_paths_contract():
    """obtain_samples with the Obs-DP policy: the reference's path dicts, attentions = None per step (no communication)"""
    import sys
    from types import SimpleNamespace
    sys.path.insert(0, GOLDEN)
    import ref_harness
    from com_marl_b200.envs import PredatorPreyWrapper
    from com_marl_b200.rollout import make_policy
    from com_marl_b200.sampler import DeviceRolloutSampler
    params = ref_harness.scenario_params("pp", 10, 1, 0.08, cap=2, loss=0.2, max_env_steps=20)
    env = PredatorPreyWrapper(centralized=True, other_agent_visible=True, params=params)
    spec = env.spec_b200
    n, D = spec.n_agents, spec.obs_dim
    algo = SimpleNamespace(policy=make_policy(spec, kind="dec"), max_path_length=20)
    sampler = DeviceRolloutSampler(algo, env, n_envs=8, chunk=10)
    sampler.start_worker()
    paths = sampler.obtain_samples(0, batch_size=8 * 20 * n)
    assert paths
    for pth in paths:
        T = len(pth["rewards"])
        assert pth["observations"].shape == (T, n * D) and pth["actions"].shape == (T, n)
        assert set(pth["agent_infos"].keys()) == {"action_probs"} and pth["agent_infos"]["action_probs"].shape == (T, n, 5)
        assert pth["attentions"].shape == (T,) and all(a is None for a in pth["attentions"])
        assert pth["dist_adjs"].shape == (T, n * n) and pth["dones"][-1]
    sampler.shutdown_worker()


def test_policy_kind_error_codes():
    """C-ABI error behaviour of the new descriptor field: unknown kinds are rejected, Comm-DP and Obs-DP need the tensor-core
    path (math = 1)."""
    import ctypes as C
    from com_marl_b200 import _native as N
    n, D, B = 3, 29, 8
    pol = _policy(n, D)
    obs = torch.zeros((B, n, D), device="cuda")
    probs = torch.empty((B, n, 5), device="cuda")
    io = N.PolicyIO()
    io.n_envs, io.weights, io.tc_weights = B, N.ptr(pol.weight_blob()), N.ptr(pol.tc_weight_blob())
    io.obs, io.probs = N.ptr(obs), N.ptr(probs)
    for kind, math, expect in ((7, 1, N.CM_EINVAL), (N.POLICY_DEC, 0, N.CM_EUNSUPPORTED), (N.POLICY_DEC, 2, N.CM_EUNSUPPORTED),
                               (N.POLICY_COMM, 0, N.CM_EUNSUPPORTED), (N.POLICY_COMM, 2, N.CM_EUNSUPPORTED), (N.POLICY_DEC, 1, N.CM_OK)):
        desc = N.PolicyDesc(n, D, 1, 0, 1, math, 1, 0, kind)
        assert N.lib().cm_policy_forward(C.byref(desc), C.byref(io), N.stream_ptr()) == expect, (kind, math)
    torch.cuda.synchronize()
    assert torch.isfinite(probs).all()


@pytest.mark.parametrize("kind", ["dec", "cent"])
def test_narrow_hidden_sizes_run_zero_padded(kind):
    """hidden_sizes below the kernels' widths (128, 64, 32) run on the same kernels, embedded in zeros: the kernel equals the
    module's own differentiable torch forward (the training path) to 1e-5"""
    from com_marl_b200.policy import CentralizedCategoricalMLPPolicy, DecCategoricalMLPPolicy
    from com_marl_b200.spaces import Box, Discrete, EnvSpec
    n, D, B = 5, 29, 97
    spec = EnvSpec(Box(np.zeros(n * D), np.ones(n * D)), Discrete(5))
    torch.manual_seed(3)
    cls = DecCategoricalMLPPolicy if kind == "dec" else CentralizedCategoricalMLPPolicy
    pol = cls(spec, n, hidden_sizes=(72, 40, 24))
    with torch.no_grad():
        for k, v in pol.state_dict().items():
            if k.endswith("bias"):
                v.uniform_(-0.1, 0.1)
    obs = torch.rand((B, n * D), device="cuda")
    avail = torch.ones((B, n * 5), device="cuda")
    probs = torch.empty((B, n, 5), device="cuda")
    pol.act_device(obs.reshape(B, n, D), probs=probs, greedy=True, actions=torch.empty((B, n), dtype=torch.int8, device="cuda"))
    pol.check_errors()
    with torch.no_grad():
        ref = pol.forward(obs, avail).probs
    assert (probs - ref).abs().max().item() <= 1e-5
    with pytest.raises(NotImplementedError):
        cls(spec, n, hidden_sizes=(256, 64, 32))
