"""Training several policies in one batched run: cm_ppo_net over a set of networks (cm_net_io.n_policies), cm_adam_step_set and
DevicePPOSet, each held against what the single-network calls and a standalone DevicePPO compute."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from com_marl_b200 import _native as N

HERE = os.path.dirname(os.path.abspath(__file__))
pytestmark = pytest.mark.gpu

H1, E, C1, C2, C3, A = 128, 64, 128, 64, 32, 5


def policy_segments(D, L):
    sizes = [("enc_w1", D * H1), ("enc_b1", H1), ("enc_w2", H1 * E), ("enc_b2", E), ("att_w", E * E), ("gcn_w", L * E * E),
             ("gcn_b", L * E), ("head_w1", E * C1), ("head_b1", C1), ("head_w2", C1 * C2), ("head_b2", C2), ("head_w3", C2 * C3),
             ("head_b3", C3), ("head_w4", C3 * A), ("head_b4", A)]
    return _offsets(sizes)


def critic_segments(D, L):
    sizes = [("enc_w1", D * H1), ("enc_b1", H1), ("enc_w2", H1 * E), ("enc_b2", E), ("att_w", E * E), ("gcn_w", L * E * E),
             ("gcn_b", L * E), ("dec_w1", E * 64), ("dec_b1", 64), ("dec_w2", 64), ("dec_b2", 1), ("log_std", 1)]
    return _offsets(sizes)


def _offsets(sizes):
    out, o = [], 0
    for k, s in sizes:
        out.append((k, o, o + s))
        o += s
    return out, o


class NetSetCase:
    """K members of one kind with distinct random weights, S = K * P steps with a random tail of valid = 0 steps per member"""

    def __init__(self, kind, n, D, L, K, P, seed=0):
        self.kind, self.n, self.D, self.L, self.K, self.P = kind, n, D, L, K, P
        dev = "cuda"
        g = torch.Generator(device="cpu").manual_seed(seed)
        rnd = lambda *s: torch.rand(*s, generator=g)  # noqa: E731
        self.net = {"policy": N.NET_POLICY, "dec": N.NET_POLICY_DEC, "critic": N.NET_CRITIC}[kind]
        Lb = 1 if kind == "dec" else L
        self.segs, nb = (critic_segments if kind == "critic" else policy_segments)(D, Lb)
        lib = N.lib()
        assert nb == (lib.cm_critic_blob_floats(D, Lb) if kind == "critic" else lib.cm_policy_blob_floats(D, Lb))
        self.nb, self.stride = nb, (nb + 3) // 4 * 4 + 4                 # (a stride longer than the blob)
        w = (rnd(K, self.stride) * 2 - 1) * 0.15
        for name, a, b in self.segs:                                    # the critic's log-std near log 0.5
            if name == "log_std":
                w[:, a:b] = -0.7 + 0.1 * rnd(K, 1)
        self.weights = w.to(dev).contiguous()
        S, W = K * P, (n + 31) // 32
        self.S = S
        self.desc = N.NetDesc(self.net, n, D, Lb, 1, 0.01 if kind != "critic" else 0.0, 0.9 if kind != "critic" else 0.0,
                              1.1 if kind != "critic" else 0.0)
        self.obs = rnd(S, n, D).to(dev)
        bits = torch.randint(-2 ** 31, 2 ** 31 - 1, (S, n, W), generator=g, dtype=torch.int64).to(torch.int32)
        self.adj = bits.to(dev).contiguous()
        self.chan = torch.randint(-2 ** 31, 2 ** 31 - 1, (S, L, n, W), generator=g, dtype=torch.int64).to(torch.int32).to(dev).contiguous()
        self.actions = torch.randint(0, A, (S, n), generator=g).to(dev)
        av = torch.randint(1, 32, (S, n), generator=g) | (1 << self.actions.cpu())
        self.avail = av.to(torch.uint8).to(dev)
        self.adv = (rnd(S) * 2 - 1).to(dev)
        self.returns = (rnd(S) * 4 - 2).to(dev)
        valid = torch.ones(K, P, dtype=torch.uint8)
        self.counts = []
        for i in range(K):
            v = P - int(torch.randint(0, max(P // 3, 1) + 1, (1,), generator=g))
            valid[i, v:] = 0
            self.counts.append(max(v, 1))
        self.valid = valid.reshape(-1).to(dev).contiguous()
        self.old_ll = None

    def ws(self, chunk, K):
        need = N.lib().cm_ppo_net_workspace_floats(C.byref(self.desc), chunk, 1) + N.net_set_workspace_extra(K)
        return torch.empty(need, dtype=torch.float32, device="cuda")

    def call(self, weights, grad, s0, s1, inv, n_policies=0, chunk=None, inv_counts=None):
        """one cm_ppo_net call over steps [s0, s1); returns (rc, outputs)"""
        S = s1 - s0
        K = max(n_policies, 1)
        io = N.NetIO()
        io.n_steps = S
        io.weights, io.grad = N.ptr(weights), N.ptr(grad)
        io.obs = self.obs[s0:].data_ptr()
        if self.kind != "dec":
            io.adj_bits, io.chan_bits = self.adj[s0:].data_ptr(), self.chan[s0:].data_ptr()
        io.valid = self.valid[s0:].data_ptr()
        out = {}
        if self.kind == "critic":
            out["values"] = torch.full((S,), float("nan"), device="cuda")
            io.values, io.returns = N.ptr(out["values"]), self.returns[s0:].data_ptr()
        else:
            out["ll"], out["entropy"] = torch.full((S,), float("nan"), device="cuda"), torch.full((S,), float("nan"), device="cuda")
            out["probs"] = torch.full((S, self.n, A), float("nan"), device="cuda")
            io.ll, io.entropy, io.probs = N.ptr(out["ll"]), N.ptr(out["entropy"]), N.ptr(out["probs"])
            io.avail_bits, io.actions, io.adv = self.avail[s0:].data_ptr(), self.actions[s0:].data_ptr(), self.adv[s0:].data_ptr()
            if self.old_ll is not None:
                io.old_ll = self.old_ll[s0:].data_ptr()
        out["loss"] = torch.zeros(K, device="cuda")
        io.loss = N.ptr(out["loss"])
        io.inv_count = float(inv)
        ws = self.ws(chunk or S, K)
        io.workspace, io.workspace_floats = N.ptr(ws), ws.numel()
        if n_policies:
            io.n_policies, io.steps_per_policy, io.weights_stride, io.grad_stride = n_policies, S // n_policies, self.stride, self.stride
            io.inv_counts = N.ptr(inv_counts)
        rc = N.lib().cm_ppo_net(C.byref(self.desc), C.byref(io), N.stream_ptr())
        torch.cuda.synchronize()
        return rc, out

    def run_set(self, chunk=None):
        grad = torch.zeros_like(self.weights)
        inv = torch.tensor([1.0 / c for c in self.counts], dtype=torch.float32, device="cuda")
        rc, out = self.call(self.weights, grad, 0, self.S, 0.0, n_policies=self.K, chunk=chunk, inv_counts=inv)
        assert rc == N.CM_OK
        out["grad"] = grad
        return out

    def run_blocks(self, member_weights=None):
        """K single-network calls, member i on block i (member_weights(i): the row it reads)"""
        outs = []
        for i in range(self.K):
            wi = self.weights[member_weights(i) if member_weights else i, :self.nb].contiguous()
            grad = torch.zeros(self.nb, device="cuda")
            rc, out = self.call(wi, grad, i * self.P, (i + 1) * self.P, 1.0 / self.counts[i])
            assert rc == N.CM_OK
            out["grad"] = grad
            outs.append(out)
        return outs


def _compare(c, st, blocks):
    """largest gradient error relative to each tensor's largest magnitude, per-step outputs bit for bit, losses to 1e-6"""
    worst = 0.0
    for i, b in enumerate(blocks):
        sl = slice(i * c.P, (i + 1) * c.P)
        for k in ("ll", "entropy", "probs", "values"):
            if k in b:
                assert torch.equal(st[k][sl], b[k]), (i, k)
        # 1e-6 of the size of the mean's terms: the fp32 partial sums of the CTAs see other steps when the launch shapes
        # differ, and the policy's objective terms (advantages of both signs) cancel in the sum
        ref = float(b["loss"][0])
        scale = max(abs(ref), float((c.returns if c.kind == "critic" else c.adv)[sl].abs().mean()))
        assert abs(float(st["loss"][i]) - ref) <= 1e-6 * scale, (i, float(st["loss"][i]), ref)
        for name, a, z in c.segs:
            r = b["grad"][a:z]
            scale = float(r.abs().max())
            if scale == 0.0:
                assert not st["grad"][i, a:z].any(), (i, name)
                continue
            worst = max(worst, float((st["grad"][i, a:z] - r).abs().max()) / scale)
        assert not st["grad"][i, c.nb:].any()
    return worst


SHAPES = [("policy", 3, 20, 2), ("policy", 4, 13, 1), ("policy", 9, 30, 4), ("policy", 32, 17, 2), ("policy", 33, 21, 1),
          ("policy", 65, 9, 2), ("policy", 200, 12, 1), ("dec", 3, 20, 1), ("dec", 33, 21, 1), ("dec", 200, 12, 1),
          ("critic", 3, 20, 2), ("critic", 4, 13, 4), ("critic", 9, 30, 1), ("critic", 32, 17, 2), ("critic", 65, 9, 4),
          ("critic", 200, 12, 2)]


@pytest.mark.parametrize("kind,n,D,L", SHAPES)
@pytest.mark.parametrize("K", [2, 5])
def test_set_call_equals_block_calls(kind, n, D, L, K):
    """cm_ppo_net over K members == K single-network calls on the blocks: whole call, a workspace that holds two members and a
    bit (a chunk of whole members side by side), and one that holds less than a member (chunks cut through every block)"""
    P = max(3, 333 // n + 1)                  # P n rows per member: not a multiple of the 128-row tiles
    if (P * n) % 128 == 0:
        P += 1
    c = NetSetCase(kind, n, D, L, K, P, seed=n * 7 + K)
    if kind != "critic":                      # a frozen old policy near the current one: ratios inside and outside the clip range
        c.old_ll = c.run_set()["ll"] + 0.15 * (torch.rand(c.S, device="cuda") - 0.5)
    blocks = c.run_blocks()
    for chunk in (None, 2 * P + 1, max(1, (2 * P) // 5)):
        assert _compare(c, c.run_set(chunk), blocks) <= 2e-4
    # the test sees a wrong member: every block computed with member 0's weights is O(1) away
    if K > 1:
        wrong = c.run_blocks(member_weights=lambda i: 0)
        key = "values" if kind == "critic" else "ll"
        st = c.run_set()
        d = max(float((st[key][i * P:(i + 1) * P] - wrong[i][key]).abs().max()) for i in range(1, K))
        assert d > 1e-2


def test_set_errors():
    c = NetSetCase("policy", 5, 11, 2, 3, 7)
    inv = torch.ones(3, device="cuda")
    grad = torch.zeros_like(c.weights)

    def rc_of(**kw):
        io_kw = dict(n_policies=3, inv_counts=inv)
        io_kw.update(kw)
        return c.call(c.weights, grad, 0, c.S, 1.0, **io_kw)[0]

    assert rc_of() == N.CM_OK
    # n_steps not n_policies * steps_per_policy
    assert c.call(c.weights, grad, 0, c.S - 1, 1.0, n_policies=3, inv_counts=inv)[0] == N.CM_EINVAL
    for stride in (c.nb - 4, c.stride - 2):
        saved = c.stride
        c.stride = stride
        try:
            assert rc_of() == N.CM_EINVAL, stride
        finally:
            c.stride = saved
    assert rc_of(inv_counts=None) == N.CM_EINVAL
    for kind in (N.NET_POLICY_CENT, N.NET_BASELINE_MLP):
        saved = c.desc.kind
        c.desc.kind = kind
        try:
            assert rc_of() == N.CM_EUNSUPPORTED
        finally:
            c.desc.kind = saved


def test_adam_set_equals_single_steps():
    K, n, stride = 5, 1237, 1240
    g = torch.Generator(device="cpu").manual_seed(3)
    p = torch.randn(K, stride, generator=g).cuda()
    gr = torch.randn(K, stride, generator=g).cuda()
    m = torch.randn(K, stride, generator=g).cuda() * 0.1
    v = torch.rand(K, stride, generator=g).cuda() * 0.01
    scale = torch.rand(K, generator=g).cuda()
    steps = [3, 0, 1, 17, 0]
    ref = [t.clone() for t in (p, m, v)]
    for i, s in enumerate(steps):
        if s:
            N.check("cm_adam_step_dev", N.lib().cm_adam_step_dev(ref[0][i].data_ptr(), gr[i].data_ptr(), ref[1][i].data_ptr(),
                                                                 ref[2][i].data_ptr(), n, 3e-4, 0.9, 0.999, 1e-5, s,
                                                                 scale[i:].data_ptr(), N.stream_ptr()))
    before = [t.clone() for t in (p, m, v)]
    arr = (C.c_int32 * K)(*steps)
    N.check("cm_adam_step_set", N.lib().cm_adam_step_set(N.ptr(p), N.ptr(gr), N.ptr(m), N.ptr(v), K, n, stride, 3e-4, 0.9, 0.999, 1e-5,
                                                         arr, N.ptr(scale), N.stream_ptr()))
    torch.cuda.synchronize()
    for a, b, b0 in zip((p, m, v), ref, before):
        assert torch.equal(a, b)
        for i, s in enumerate(steps):
            if not s:
                assert torch.equal(a[i], b0[i])
        assert torch.equal(a[:, n:], b0[:, n:])                 # nothing beyond n floats of a row
    assert N.lib().cm_adam_step_set(N.ptr(p), N.ptr(gr), N.ptr(m), N.ptr(v), K, n, n - 1, 3e-4, 0.9, 0.999, 1e-5, arr, N.ptr(scale),
                                    N.stream_ptr()) == N.CM_EINVAL


# ---- DevicePPOSet ------------------------------------------------------------------------------------------------------
def _golden():
    import sys
    sys.path.insert(0, HERE)
    from test_ppo import PPOCase
    return PPOCase("pp")


def _member(c, seed, golden):
    from com_marl_b200.policy import CommCategoricalMLPPolicy
    from com_marl_b200.ppo import CommBaseCritic
    from com_marl_b200.spaces import Box, Discrete, EnvSpec
    n, D = int(c.meta["n"]), int(c.meta["D"])
    spec = EnvSpec(Box(np.zeros(n * D), np.ones(n * D)), Discrete(5))
    torch.manual_seed(seed)
    pol, cri = CommCategoricalMLPPolicy(spec, n, device="cuda"), CommBaseCritic(spec, n, device="cuda")
    if golden:
        pol.load_state_dict({k: torch.as_tensor(v) for k, v in c.sd["pol0"].items()})
        cri.load_state_dict({k: torch.as_tensor(v) for k, v in c.sd["cri0"].items()})
    return pol, cri


def _ppo_args(c):
    m = c.meta
    return dict(discount=m["discount"], gae_lambda=m["gae_lambda"], policy_ent_coeff=m["ent_coeff"], clip_grad_norm=m["clip_grad_norm"],
                optimization_n_minibatches=int(m["n_minibatches"]), optimization_mini_epochs=int(m["mini_epochs"]), policy_lr=m["lr"],
                adam_eps=m["adam_eps"])


def test_set_update_golden_anchor():
    """the reference's golden PPO round is member 1 of a 3-member set; members 0 and 2 have other weights and 4 / 5 paths (2 and
    3 minibatch slices against the golden case's own count) and match their standalone DevicePPO(fused=True)"""
    from com_marl_b200.ppo import DevicePPO, DevicePPOSet
    c = _golden()
    z = c.z
    assert len(c.paths) >= 5
    paths = [c.paths[:4], c.paths, c.paths[1:6]]
    perms = [np.random.default_rng(11).permutation(4), z["shuffled_ids"], np.random.default_rng(12).permutation(5)]
    members = [_member(c, 21, False), _member(c, 0, True), _member(c, 23, False)]
    init = [({k: v.clone() for k, v in p.state_dict().items()}, {k: v.clone() for k, v in q.state_dict().items()}) for p, q in members]
    k0 = next(iter(init[0][0]))
    assert not torch.equal(init[0][0][k0], init[2][0][k0]) and not torch.equal(init[0][0][k0], init[1][0][k0])
    S = DevicePPOSet([p for p, _ in members], [q for _, q in members], **_ppo_args(c))
    batches = [S.members[i].process_samples(paths[i]) for i in range(3)]
    outs = S.train_once(batches, perms)
    # member 1: the golden tolerances of test_train_once_matches_reference
    o = outs[1]
    assert abs(o["loss_before"] - float(z["loss_before"])) <= 2e-5
    assert np.abs(np.array(o["losses"]) - z["losses"]).max() <= 1e-4
    assert np.abs(np.array(o["baseline_losses"]) - z["baseline_losses"]).max() <= 1e-4 * max(1.0, np.abs(z["baseline_losses"]).max())
    assert np.abs(np.array(o["grad_norms"]) - z["grad_norms"]).max() <= 1e-3 * max(1.0, np.abs(z["grad_norms"]).max())
    assert abs(o["loss_after"] - float(z["loss_after"])) <= 1e-4
    assert abs(o["kl"] - float(z["kl"])) <= 1e-5
    for tag, mod in (("pol1", members[1][0]), ("cri1", members[1][1])):
        for k, v in mod.state_dict().items():
            ref, ref0 = c.sd[tag][k], c.sd[tag[:3] + "0"][k]
            assert np.abs(v.cpu().numpy() - ref).max() <= 0.02 * np.abs(ref - ref0).max() + 1e-6, (tag, k)
    # members 0 and 2 against their standalone update
    for i in (0, 2):
        pol, cri = _member(c, 99, False)
        pol.load_state_dict(init[i][0])
        cri.load_state_dict(init[i][1])
        algo = DevicePPO(pol, cri, fused=True, **_ppo_args(c))
        r = algo.train_once(paths=paths[i], shuffled_ids=perms[i])
        o = outs[i]
        assert len(o["losses"]) == len(r["losses"]) == int(c.meta["mini_epochs"]) * (2 if i == 0 else 3)
        assert abs(o["loss_before"] - r["loss_before"]) <= 2e-5
        assert np.abs(np.array(o["losses"]) - r["losses"]).max() <= 1e-4
        assert np.abs(np.array(o["baseline_losses"]) - r["baseline_losses"]).max() <= 1e-4 * max(1.0, np.abs(r["baseline_losses"]).max())
        assert np.abs(np.array(o["grad_norms"]) - r["grad_norms"]).max() <= 1e-3 * max(1.0, np.abs(r["grad_norms"]).max())
        assert abs(o["loss_after"] - r["loss_after"]) <= 1e-4 and abs(o["kl"] - r["kl"]) <= 1e-5
        assert abs(o["entropy"] - r["entropy"]) <= 1e-5
        for mod_set, mod_ref, k0 in ((members[i][0], pol, 0), (members[i][1], cri, 1)):
            for k, v in mod_set.state_dict().items():
                ref, ref0 = mod_ref.state_dict()[k].cpu().numpy(), init[i][k0][k].cpu().numpy()
                assert np.abs(v.cpu().numpy() - ref).max() <= 0.02 * np.abs(ref - ref0).max() + 1e-6, (i, k)
    # the rollout's PolicySet sees the updated rows (parameter versions bumped)
    from com_marl_b200.policy import PolicySet
    ps = PolicySet([p for p, _ in members])
    for i, (p, _) in enumerate(members):
        assert torch.equal(ps._blobs[i, :ps._n_blob], p.weight_blob())


def test_set_update_rejects():
    from com_marl_b200.policy import CentralizedCategoricalMLPPolicy, CommCategoricalMLPPolicy
    from com_marl_b200.ppo import CommBaseCritic, DevicePPOSet, GaussianMLPBaseline
    from com_marl_b200.spaces import Box, Discrete, EnvSpec
    n, D = 3, 10
    spec = EnvSpec(Box(np.zeros(n * D), np.ones(n * D)), Discrete(5))
    a = (CommCategoricalMLPPolicy(spec, n, device="cuda"), CommBaseCritic(spec, n, device="cuda"))
    b = (CommCategoricalMLPPolicy(spec, n, n_gcn_layers=1, device="cuda"), CommBaseCritic(spec, n, n_gcn_layers=1, device="cuda"))
    with pytest.raises(ValueError):
        DevicePPOSet([a[0], b[0]], [a[1], b[1]])
    cent = (CentralizedCategoricalMLPPolicy(spec, n, device="cuda"), GaussianMLPBaseline(spec, hidden_sizes=(64, 64, 64), device="cuda"))
    with pytest.raises(NotImplementedError):
        DevicePPOSet([cent[0]], [cent[1]])

    from com_marl_b200 import ppo
    orig = ppo._world
    ppo._world = lambda group=None: 2            # a process group of two ranks: sets across ranks are not built
    try:
        with pytest.raises(NotImplementedError):
            DevicePPOSet([a[0]], [a[1]], process_group=object())
    finally:
        ppo._world = orig


# ---- DeviceTrainerSet --------------------------------------------------------------------------------------------------
def _c3_shape():
    from com_marl_b200.scenario import ScenarioSpec
    return ScenarioSpec.from_cli("pp", 20, 2, 0.08, cap=4, loss=0.2, seed=5, max_env_steps=24)      # C3's team, map and channel


def test_trainer_set_equals_standalone_trainers():
    """round 1 of a 3-member DeviceTrainerSet (distinct seeds, member 1 under its own IID channel) against three standalone
    DeviceTrainers started from the members' initial weights"""
    from com_marl_b200.ppo import CommBaseCritic, DevicePPO
    from com_marl_b200.rollout import make_policy
    from com_marl_b200.spaces import Box, Discrete, EnvSpec
    from com_marl_b200.train import DeviceTrainer, DeviceTrainerSet
    E, seeds, env_id0 = 6, [3, 8, 13], 100
    args = dict(optimization_mini_epochs=2)
    spec = _c3_shape()
    conds = [None, spec.with_channel(pl=0.3), None]
    S = DeviceTrainerSet(spec, E, seeds, conditions=conds, env_id0=env_id0, **args)
    init = [({k: v.clone() for k, v in p.state_dict().items()}, {k: v.clone() for k, v in c.state_dict().items()})
            for p, c in zip(S.policies, S.critics)]
    k0 = next(iter(init[0][0]))
    assert not torch.equal(init[0][0][k0], init[1][0][k0]) and not torch.equal(init[1][0][k0], init[2][0][k0])
    outs = S.train_epoch()
    n, D = spec.n_agents, spec.obs_dim
    env_spec = EnvSpec(Box(np.zeros(n * D), np.ones(n * D)), Discrete(5))
    for i in range(3):
        t = DeviceTrainer(conds[i] or _c3_shape(), E, env_id0=env_id0 + i * E, seed=seeds[i], **args)
        t.policy.load_state_dict(init[i][0])
        t.critic.load_state_dict(init[i][1])
        t.policy.refresh_weights(force=True)
        r = t.train_epoch()
        for k, v in t.engine.traj.items():                       # the trajectory ring, bit for bit
            assert torch.equal(S.member_traj(i)[k], v), (i, k)
        # the padded batch, baselines, returns and advantages the standalone run built from the same trajectory and weights
        pol0 = make_policy(_c3_shape(), torch_seed=1)
        cri0 = CommBaseCritic(env_spec, n, n_gcn_layers=spec.n_layers)
        pol0.load_state_dict(init[i][0])
        cri0.load_state_dict(init[i][1])
        ref = DevicePPO(pol0, cri0, fused=True, **args).batch_from_trajectory(t.engine.traj)
        for k in ("obs", "actions", "rewards", "valids", "adj_bits", "chan_bits", "baselines", "returns", "adv"):
            assert torch.equal(S.batches[i][k], ref[k]), (i, k)
        o = outs[i]
        assert len(o["losses"]) == len(r["losses"])
        assert abs(o["loss_before"] - r["loss_before"]) <= 2e-5
        assert np.abs(np.array(o["losses"]) - r["losses"]).max() <= 1e-4
        assert np.abs(np.array(o["grad_norms"]) - r["grad_norms"]).max() <= 1e-3 * max(1.0, np.abs(r["grad_norms"]).max())
        assert abs(o["kl"] - r["kl"]) <= 1e-5
        for mod_set, mod_ref, j in ((S.policies[i], t.policy, 0), (S.critics[i], t.critic, 1)):
            for k, v in mod_set.state_dict().items():
                a, b, b0 = v.cpu().numpy(), mod_ref.state_dict()[k].cpu().numpy(), init[i][j][k].cpu().numpy()
                assert np.abs(a - b).max() <= 0.02 * np.abs(b - b0).max() + 1e-6, (i, k)
        for k in ("Iteration", "NumTrajs", "AverageDiscountedReturn", "AverageReturn", "StdReturn", "MaxReturn", "MinReturn",
                  "SuccessRate", "AverageCaptureCount", "AverageStepCount", "AverageMovingCount", "AveragePenaltyCount",
                  "AverageVariable", "AverageVar2", "AveDegree", "Diameter", "AveTroughput"):
            assert o["tabular"][k] == r["tabular"][k], (i, k)
        assert o["episode_stats"] == r["episode_stats"]
    # another seed for member 1 leaves the trajectories of members 0 and 2 as they were
    S2 = DeviceTrainerSet(_c3_shape(), E, [3, 99, 13], conditions=[None, _c3_shape().with_channel(pl=0.3), None], env_id0=env_id0, **args)
    S2.train_epoch()
    for i in (0, 2):
        for k, v in S.member_traj(i).items():
            assert torch.equal(S2.member_traj(i)[k], v), (i, k)
    assert not torch.equal(S2.member_traj(1)["actions"], S.member_traj(1)["actions"])


def test_trainer_set_rejects_cent():
    from com_marl_b200.train import DeviceTrainerSet
    with pytest.raises(NotImplementedError):
        DeviceTrainerSet(_c3_shape(), 4, [1, 2], kind="cent")
