"""GPU parity of the fused policy forward, through the C ABI (cm_policy_forward).

Tolerance (BASELINE.json north_star): logits within 1e-5 relative — measured as
max|logit - ref| <= 1e-5 * max(1, max|ref logits|) — against the reference torch forward recorded in
tests/golden/policy_*.npz; probabilities and attention within 1e-5 absolute.
"""
import numpy as np
import pytest
import torch

from golden_util import PolicyCase, policy_cases
from oracle import oracle as orc

pytestmark = pytest.mark.gpu
SMALL = policy_cases()


def _policy(n, D, L, weights=None, seed=0, math="auto", **kwargs):
    from com_marl_b200.policy import CommCategoricalMLPPolicy
    from com_marl_b200.spaces import Box, Discrete, EnvSpec
    torch.manual_seed(seed)
    pol = CommCategoricalMLPPolicy(EnvSpec(Box(np.zeros(n * D), np.ones(n * D)), Discrete(5)), n, n_gcn_layers=L, math=math, **kwargs)
    if weights is not None:
        pol.load_state_dict({k: torch.as_tensor(v) for k, v in weights.items()})   # reference checkpoints load as is
    return pol


@pytest.mark.parametrize("math", ["tc"])
@pytest.mark.parametrize("name", SMALL)
def test_policy_kernel_matches_reference_golden(name, math):
    c = PolicyCase(name)
    pol = _policy(c.n, c.D, c.L, c.weights, math=math, **c.policy_kwargs)       # (narrow / 'dot' cases: the reference's own ctor arguments)
    dist, attn = pol.forward(c.obs.reshape(c.B, -1), c.avail.reshape(c.B, -1), c.adj.astype(np.float32),
                             c.chan.astype(np.float32), get_actions=True)
    probs = dist.probs.numpy()
    assert np.abs(probs - c.probs).max() <= 1e-5
    assert np.abs(attn.numpy() - c.attn).max() <= 1e-5
    # raw logits through the device entry point
    dev = pol.device
    obs = torch.from_numpy(c.obs).to(dev)
    adj = pol.pack_mask(torch.from_numpy(c.adj.astype(np.float32)).to(dev), c.n)
    ch = pol.pack_mask(torch.from_numpy(c.chan.astype(np.float32)).to(dev), c.n)
    logits = torch.empty((c.B, c.n, 5), device=dev)
    pol.act_device(obs, adj, ch, logits=logits, greedy=True)
    pol.check_errors()
    scale = max(1.0, float(np.abs(c.logits).max()))
    err = np.abs(logits.cpu().numpy() - c.logits).max() / scale
    print(f"{name} {math}: logits rel err {err:.2e}")
    assert err <= 1e-5
    # and the differentiable torch path of the same module (used by the PPO update) agrees too
    with torch.no_grad():
        # shaped like process_samples hands them over: adj (.., n*n), channels (.., L*n, n)  (…vectorized_sampler.py:176,183)
        d2, _ = pol.forward(torch.from_numpy(c.obs.reshape(c.B, -1)).to(dev), torch.from_numpy(c.avail.reshape(c.B, -1)).to(dev),
                            torch.from_numpy(c.adj.astype(np.float32).reshape(c.B, -1)).to(dev),
                            torch.from_numpy(c.chan.astype(np.float32).reshape(c.B, c.L * c.n, c.n)).to(dev))
    assert np.abs(d2.probs.cpu().numpy() - c.probs).max() <= 1e-5


@pytest.mark.parametrize("math", ["tc"])
@pytest.mark.parametrize("n,D,B,ploss", [(3, 29, 16384, 0.0), (4, 21, 5000, 0.3), (32, 53, 2048, 0.2), (54, 77, 777, 0.1),
                                         (7, 53, 1001, 0.5), (64, 29, 64, 0.4), (1, 21, 100, 0.0),
                                         (16, 53, 333, 0.2), (17, 21, 250, 0.3), (33, 29, 203, 0.1), (40, 77, 131, 0.5),
                                         (65, 21, 70, 0.2), (72, 53, 301, 0.3), (200, 53, 97, 0.2), (256, 29, 9, 0.5),
                                         (129, 29, 33, 0.3), (96, 77, 40, 0.1), (193, 21, 5, 0.6)])
def test_policy_kernel_matches_oracle_batched(n, D, B, ploss, math):
    """Random binary observations + random masks on big ragged batches (last tile partial) vs the numpy
    restatement; sampling reproduces the inverse-CDF stream specification exactly."""
    rng = np.random.default_rng(n * 1000 + D)
    pol = _policy(n, D, 2, seed=n, math=math)
    with torch.no_grad():
        for k, v in pol.state_dict().items():
            if k.endswith("bias"):
                v.uniform_(-0.1, 0.1)
    w = {k: v.cpu().numpy() for k, v in pol.state_dict().items()}
    obs = (rng.random((B, n, D)) < 0.3).astype(np.float32)
    obs[..., -2:] = rng.random((B, n, 2)).astype(np.float32)
    adj = (rng.random((B, n, n)) < 0.7).astype(np.uint8) | np.eye(n, dtype=np.uint8)
    chan = ((rng.random((B, 2, n, n)) >= ploss).astype(np.uint8)) | np.eye(n, dtype=np.uint8)
    avail = np.ones((B, n, 5), dtype=np.uint8)
    avail[rng.random((B, n)) < 0.1, rng.integers(0, 5)] = 0
    u = rng.random((B, n)).astype(np.float32)
    dev = pol.device
    t = lambda a, dt=torch.float32: torch.as_tensor(a, dtype=dt).to(dev)  # noqa: E731
    adj_b, ch_b = pol.pack_mask(t(adj), n), pol.pack_mask(t(chan), n)
    av_b = t((avail * np.array([1, 2, 4, 8, 16], dtype=np.uint8)).sum(-1), torch.uint8)
    probs = torch.empty((B, n, 5), device=dev)
    logits = torch.empty((B, n, 5), device=dev)
    attn = torch.empty((B, n, n), device=dev)
    actions = torch.empty((B, n), dtype=torch.int8, device=dev)
    pol.act_device(t(obs), adj_b, ch_b, av_b, t(u), probs=probs, logits=logits, attention=attn, actions=actions)
    pol.check_errors()
    ref_logits, ref_probs, ref_attn = orc.policy_forward(w, obs, avail, adj, chan, dtype=np.float64)
    scale = max(1.0, float(np.abs(ref_logits).max()))
    err = np.abs(logits.cpu().numpy() - ref_logits).max() / scale
    print(f"n={n} D={D} {math}: logits rel err {err:.2e}")
    assert err <= 1e-5
    assert np.abs(probs.cpu().numpy() - ref_probs).max() <= 1e-5
    assert np.abs(attn.cpu().numpy() - ref_attn).max() <= 1e-5
    # sampling: exact against the oracle's inverse CDF evaluated on the kernel's own probabilities
    ospec = dict(n=n)
    got = actions.cpu().numpy()
    p = probs.cpu().numpy()
    c = np.zeros((B, n), dtype=np.float32)
    want = np.full((B, n), -1, dtype=np.int64)
    for a in range(5):
        c = (c + p[..., a]).astype(np.float32)
        want = np.where((want < 0) & (u < c), a, want)
    last = np.where(p > 0, np.arange(5), -1).max(-1)
    want = np.where(want < 0, last, want)
    assert np.array_equal(got, want)
    assert (np.take_along_axis(avail, got[..., None].astype(np.int64), -1) == 1).all(), "sampled a masked action"
    # greedy
    pol.act_device(t(obs), adj_b, ch_b, av_b, greedy=True, probs=probs, actions=actions)
    assert np.array_equal(actions.cpu().numpy(), probs.cpu().numpy().argmax(-1))


def test_get_actions_contract():
    """get_actions returns what the reference returns: int64 actions (B,n), lists of per-env arrays."""
    pol = _policy(4, 21, 2, math="auto")
    rng = np.random.default_rng(0)
    obs = rng.random((5, 84)).astype(np.float32)
    acts, infos = pol.get_actions(obs, np.ones((5, 20)), np.ones((5, 4, 4)), np.ones((5, 2, 4, 4)))
    assert acts.shape == (5, 4) and acts.dtype == np.int64
    assert len(infos["action_probs"]) == 5 and infos["action_probs"][0].shape == (4, 5)
    assert infos["attention_weights"][0].shape == (4, 4)
    a1, i1 = pol.get_actions(obs[0], np.ones(20), np.ones((4, 4)), np.ones((2, 4, 4)), greedy=True)
    assert a1.shape == (4,) and np.array_equal(a1, np.stack(i1["action_probs"]).argmax(-1))
    assert np.allclose(np.stack(i1["action_probs"]), infos["action_probs"][0], atol=1e-6)
