"""The CENT family's PPO update on the hand-written kernels (cm_ppo_net kinds CM_NET_POLICY_CENT and CM_NET_BASELINE_MLP,
csrc/ppo_net_kernels.cu) against the torch autograd graph of the same formula (policy.py::CentralizedCategoricalMLPPolicy.forward,
ppo.py::GaussianMLPBaseline.compute_loss — themselves held against the unmodified reference by tests/test_ppo.py): per-step
outputs, losses and EVERY parameter gradient on random ragged batches with masked actions, for first-layer widths K = n*D from 65
to 32 768, tanh and relu; chunked walks; the reference golden of the co_cent runner with fused=True; whole trainer rounds."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _make(n, D, P, T, seed, relu=False, pol_sizes=(128, 64, 32), bl_sizes=(64, 64, 64), ent_coeff=0.1, positive_adv=False):
    import torch
    from com_marl_b200.policy import CentralizedCategoricalMLPPolicy
    from com_marl_b200.ppo import DevicePPO, GaussianMLPBaseline
    from com_marl_b200.spaces import Box, Discrete, EnvSpec
    torch.manual_seed(seed)
    spec = EnvSpec(Box(np.zeros(n * D), np.ones(n * D)), Discrete(5))
    mk = lambda: (CentralizedCategoricalMLPPolicy(spec, n, hidden_sizes=pol_sizes, hidden_nonlinearity="relu" if relu else "tanh"),  # noqa: E731
                  GaussianMLPBaseline(spec, hidden_sizes=bl_sizes))
    pol_a, bl_a = mk()
    pol_f, bl_f = mk()
    with torch.no_grad():                       # biases away from their zero initialisation, log-std away from 0
        for m in (pol_a, bl_a):
            for k, p in m.named_parameters():
                if k.endswith("bias") or k.endswith("_init_std"):
                    p.add_(0.1 * torch.randn_like(p))
    pol_f.load_state_dict(pol_a.state_dict())
    bl_f.load_state_dict(bl_a.state_dict())
    kw = dict(policy_ent_coeff=ent_coeff, positive_adv=positive_adv)
    auto = DevicePPO(pol_a, bl_a, fused=False, **kw)
    fused = DevicePPO(pol_f, bl_f, fused=True, **kw)
    g = torch.Generator(device="cuda").manual_seed(seed)
    rnd = lambda *s: torch.rand(*s, device="cuda", generator=g)  # noqa: E731
    valids = torch.randint(1, T + 1, (P,), device="cuda", generator=g).to(torch.int32)
    valids[0] = valids[-1] = T
    avail = (rnd(P, T, n, 5) < 0.7).float()
    avail[..., 4] = 1.0                          # one action available per agent (a fully masked agent is NaN on both paths)
    actions = torch.multinomial(avail.reshape(-1, 5), 1).reshape(P, T, n)
    b = dict(obs=rnd(P, T, n * D), avail=avail.reshape(P, T, n * 5), actions=actions, rewards=rnd(P, T).double(), valids=valids)
    t = torch.arange(T, device="cuda")[None, :] < valids[:, None]
    b["obs"] = b["obs"] * t.reshape(P, T, 1).float()
    b["rewards"] = b["rewards"] * t.double()
    return auto, fused, b


def _rel(a, ref):
    return float((a - ref).abs().max() / max(1e-12, float(ref.abs().max())))


NARROW = dict(pol_sizes=(64, 48, 16), bl_sizes=(32, 64, 16))


# (n, D): the golden shape K = 87 (rows not 16-byte aligned), K = 84, K = 65 (neither a multiple of 4 nor of the 64-wide panel),
# C3, C4, C5 and the largest K = 32 768
@pytest.mark.parametrize("n,D,P,T,kw", [
    (3, 29, 7, 9, dict()),
    (3, 29, 5, 6, dict(relu=True, ent_coeff=0.0, **NARROW)),
    (4, 21, 40, 11, dict(relu=True)),
    (5, 13, 6, 8, dict(positive_adv=True, **NARROW)),
    (32, 53, 5, 7, dict(relu=True, ent_coeff=0.0)),
    (54, 77, 3, 5, dict(**NARROW)),
    (200, 53, 2, 3, dict(relu=True)),
    (256, 128, 2, 3, dict()),
])
def test_cent_fused_outputs_and_gradients_equal_autograd(n, D, P, T, kw):
    import torch
    auto, fused, b0 = _make(n, D, P, T, seed=n + D, **kw)
    ba = auto.finish_batch(dict(b0))
    bf = fused.finish_batch(dict(b0))
    assert _rel(bf["baselines"], ba["baselines"]) <= 2e-5                  # baseline values V(s) of every padded step
    F = fused._fused
    f = bf["_flat"]
    ids = np.arange(P)[::-1].copy()[: max(1, P - 1)]
    tid = torch.as_tensor(ids, device="cuda")
    # ---- policy: per-step outputs, then loss and gradient on a minibatch with a perturbed old log-likelihood (ratios on both
    # sides of the clip range)
    with torch.no_grad():
        d = auto._dist(ba, None)
        ll_ref, ent_ref = d.log_prob(ba["actions"]).sum(-1), d.entropy().mean(-1)
        F.pol_map.refresh()
        out = F.policy_call(f, None, want_probs=True)
    assert _rel(out["ll"].reshape(P, T), ll_ref) <= 2e-5
    assert _rel(out["entropy"].reshape(P, T), ent_ref) <= 2e-5
    assert _rel(out["probs"].reshape(P, T, n, 5), d.probs) <= 2e-5
    old = ll_ref + 0.15 * torch.randn_like(ll_ref)
    old[ids[0], :3] = ll_ref[ids[0], :3] + torch.tensor([-0.3, 0.3, 0.0], device="cuda")     # (that path is T >= 3 steps long)
    auto.opt.zero_grad()
    loss_ref = auto.compute_loss(ba, tid, old)
    loss_ref.backward()
    idx = F.step_index(f, ids, valid_only=True)
    adv = ba["adv"].reshape(-1).index_select(0, idx)
    if kw.get("positive_adv"):                  # shifted by the minimum over the minibatch's padded rows, as compute_loss does
        adv = adv - ba["adv"].reshape(-1).index_select(0, F.step_index(f, ids, valid_only=False)).min()
    res = F.policy_call(f, idx, adv=adv, old_ll=old.reshape(-1).index_select(0, idx), backward=True, inv_count=1.0 / idx.numel())
    g = torch.empty_like(fused.opt.grad)
    F.pol_map.scatter_grad(g)
    tol = max(1.0, n / 32.0)                    # (the joint log-likelihood is a sum over the n agents)
    assert abs(float(res["loss"]) - float(loss_ref.detach())) <= 2e-5 * tol * max(1.0, abs(float(loss_ref.detach())))
    gref = auto.opt.grad
    o = 0
    for k, p in auto.policy.named_parameters():
        assert float(gref[o:o + p.numel()].abs().max()) > 0, ("policy", k)
        e = _rel(g[o:o + p.numel()], gref[o:o + p.numel()])
        assert e <= 2e-4 * tol, ("policy", k, e)
        o += p.numel()
    # ---- baseline: loss and gradient over every padded step of the minibatch, log_std included
    auto.baseline_opt.zero_grad()
    bl_ref = auto.baseline.compute_loss(ba["obs"][tid], ba["returns"][tid])
    bl_ref.backward()
    F.cri_map.refresh()
    idx_all = F.step_index(f, ids, valid_only=False)
    res = F.critic_call(f, idx_all, returns=ba["returns"].reshape(-1).index_select(0, idx_all), backward=True)
    assert _rel(res["values"], ba["baselines"].reshape(-1).index_select(0, idx_all)) <= 2e-5
    g = torch.empty_like(fused.baseline_opt.grad)
    F.cri_map.scatter_grad(g)
    assert abs(float(res["loss"]) - float(bl_ref.detach())) <= 2e-5 * tol * max(1.0, abs(float(bl_ref.detach())))
    gref = auto.baseline_opt.grad
    o = 0
    for k, p in auto.baseline.named_parameters():
        assert float(gref[o:o + p.numel()].abs().max()) > 0, ("baseline", k)
        e = _rel(g[o:o + p.numel()], gref[o:o + p.numel()])
        assert e <= 2e-4 * tol, ("baseline", k, e)
        o += p.numel()


def test_cent_log_std_is_not_clamped():
    """GaussianMLPBaseline has no clamp on its log-std (CommBaseCritic clamps at log 1e-6): far below the clamp the fused loss and
    the log-std gradient still follow autograd"""
    import torch
    auto, fused, b0 = _make(4, 21, 3, 4, seed=2)
    with torch.no_grad():
        for m in (auto.baseline, fused.baseline):
            m.module._init_std.fill_(-16.0)
    ba, bf = auto.finish_batch(dict(b0)), fused.finish_batch(dict(b0))
    auto.baseline_opt.zero_grad()
    bl_ref = auto.baseline.compute_loss(ba["obs"], ba["returns"])
    bl_ref.backward()
    F = fused._fused
    F.cri_map.refresh()
    res = F.critic_call(bf["_flat"], None, returns=ba["returns"].reshape(-1), backward=True)
    g = torch.empty_like(fused.baseline_opt.grad)
    F.cri_map.scatter_grad(g)
    assert abs(float(res["loss"]) - float(bl_ref.detach())) <= 2e-5 * abs(float(bl_ref.detach()))
    assert _rel(g[:1], auto.baseline_opt.grad[:1]) <= 2e-5          # (module._init_std is the first parameter)


def test_cent_chunked_walk_equals_single_chunk():
    """a workspace that holds only a few steps at a time gives the same outputs and gradients (chunks add up)"""
    import torch
    _, fused, b0 = _make(7, 13, 5, 9, seed=3, relu=True)
    bf = fused.finish_batch(dict(b0))
    F, f = fused._fused, bf["_flat"]
    F.pol_map.refresh()
    F.cri_map.refresh()
    idx = F.step_index(f, np.arange(5), valid_only=True)
    adv = bf["adv"].reshape(-1).index_select(0, idx)
    ret = bf["returns"].reshape(-1)
    p1 = F.policy_call(f, idx, adv=adv, backward=True, inv_count=1.0 / idx.numel(), want_probs=True)
    gp1 = F.pol_map.grad.clone()
    c1 = F.critic_call(f, None, returns=ret, backward=True)
    gc1 = F.cri_map.grad.clone()
    F.chunk_steps, F._ws = 4, None
    p2 = F.policy_call(f, idx, adv=adv, backward=True, inv_count=1.0 / idx.numel(), want_probs=True)
    gp2 = F.pol_map.grad.clone()
    c2 = F.critic_call(f, None, returns=ret, backward=True)
    for k in ("ll", "entropy", "probs"):
        assert torch.equal(p1[k], p2[k]), k
    assert torch.equal(c1["values"], c2["values"])
    assert _rel(gp2, gp1) <= 1e-5 and _rel(F.cri_map.grad, gc1) <= 1e-5
    assert abs(float(p1["loss"]) - float(p2["loss"])) <= 1e-6 * max(1.0, abs(float(p1["loss"])))
    assert abs(float(c1["loss"]) - float(c2["loss"])) <= 1e-6 * max(1.0, abs(float(c1["loss"])))


def test_cent_train_once_matches_reference_golden():
    """tests/golden/ppo_co_cent.npz (the unmodified reference's CENT runner: CentralizedCategoricalMLPPolicy + GaussianMLPBaseline
    (64, 64, 64)) with fused=True: every assertion of test_ppo.py::test_train_once_matches_reference"""
    import torch
    from oracle import oracle as orc
    from test_ppo import PPOCase, _build
    c = PPOCase("co_cent")
    pol, cri, algo = _build(c, fused=True)
    assert algo._fused is not None and type(algo._fused).__name__ == "FusedCentNets"
    z = c.z
    out = algo.train_once(paths=c.paths, shuffled_ids=z["shuffled_ids"])
    assert abs(out["loss_before"] - float(z["loss_before"])) <= 2e-5
    assert np.abs(np.array(out["losses"]) - z["losses"]).max() <= 1e-4
    assert np.abs(np.array(out["baseline_losses"]) - z["baseline_losses"]).max() <= 1e-4 * max(1.0, np.abs(z["baseline_losses"]).max())
    assert np.abs(np.array(out["grad_norms"]) - z["grad_norms"]).max() <= 1e-3 * max(1.0, np.abs(z["grad_norms"]).max())
    assert abs(out["loss_after"] - float(z["loss_after"])) <= 1e-4
    assert abs(out["kl"] - float(z["kl"])) <= 1e-5
    for tag, mod in (("pol1", pol), ("cri1", cri)):
        for k, v in mod.state_dict().items():
            ref, ref0 = c.sd[tag][k], c.sd[tag[:3] + "0"][k]
            step = np.abs(ref - ref0).max()
            assert np.abs(v.cpu().numpy() - ref).max() <= 0.02 * step + 1e-6, (tag, k)
    # the rollout kernels see the updated weights
    n, D = int(c.meta["n"]), int(c.meta["D"])
    obs = torch.rand((8, n, D), device="cuda")
    logits = torch.empty((8, n, 5), device="cuda")
    pol.act_device(obs, logits=logits, greedy=True)
    w = {k: v.cpu().numpy() for k, v in pol.state_dict().items()}
    ref_logits = orc.policy_forward_cent(w, obs.cpu().numpy(), None)[0]
    assert np.abs(logits.cpu().numpy() - ref_logits).max() <= 1e-5 * max(1.0, np.abs(ref_logits).max())


def _trainer(scen, fused):
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import ref_harness
    from com_marl_b200.scenario import ScenarioSpec
    from com_marl_b200.train import DeviceTrainer
    m, den, T = (10, 0.04, 12) if scen == "pp" else (10, 0.03, 14)
    params = ref_harness.scenario_params(scen, m, 1, den, cap=2, loss=0.2, max_env_steps=T)
    spec = ScenarioSpec.from_params(scen, params, seed=4)
    return DeviceTrainer(spec, 48, kind="cent", fused=fused, optimization_mini_epochs=2)


@pytest.mark.parametrize("scen", ["co", "pp"])
def test_cent_trainer_round_fused_equals_autograd(scen):
    """DeviceTrainer(kind='cent'): one round (rollout + update) on the kernels and on autograd from the same start agrees within
    the golden test's tolerances; three more fused rounds stay finite and lower the loss"""
    import torch
    ta, tf = _trainer(scen, False), _trainer(scen, True)
    assert ta.algo._fused is None and tf.algo._fused is not None
    tf.policy.load_state_dict(ta.policy.state_dict())
    tf.critic.load_state_dict(ta.critic.state_dict())
    w0 = {k: v.clone() for k, v in ta.policy.state_dict().items()}
    c0 = {k: v.clone() for k, v in ta.critic.state_dict().items()}
    torch.manual_seed(0)
    np.random.seed(0)
    oa = ta.train_epoch()
    torch.manual_seed(0)
    np.random.seed(0)
    of = tf.train_epoch()
    assert oa["n_paths"] == of["n_paths"]
    assert abs(oa["loss_before"] - of["loss_before"]) <= 2e-5 * max(1.0, abs(oa["loss_before"]))
    assert np.abs(np.array(oa["losses"]) - np.array(of["losses"])).max() <= 1e-4
    assert np.abs(np.array(oa["baseline_losses"]) - np.array(of["baseline_losses"])).max() <= 1e-4 * max(1.0, np.abs(oa["baseline_losses"]).max())
    assert abs(oa["loss_after"] - of["loss_after"]) <= 1e-4
    assert abs(oa["kl"] - of["kl"]) <= 1e-5
    for ref_mod, mod, start in ((ta.policy, tf.policy, w0), (ta.critic, tf.critic, c0)):
        for (k, ra), (_, rf) in zip(ref_mod.state_dict().items(), mod.state_dict().items()):
            step = float((ra - start[k]).abs().max())
            assert float((rf - ra).abs().max()) <= 0.02 * step + 1e-6, k
    for _ in range(3):
        o = tf.train_epoch()
        assert np.isfinite(o["loss_before"]) and np.isfinite(o["loss_after"]) and np.isfinite(o["kl"])
        assert o["loss_after"] < o["loss_before"]


def test_cent_selection_and_defaults():
    import ctypes as C

    import torch
    from com_marl_b200 import _native as N
    from com_marl_b200.policy import CentralizedCategoricalMLPPolicy
    from com_marl_b200.ppo import DevicePPO, GaussianMLPBaseline
    from com_marl_b200.spaces import Box, Discrete, EnvSpec
    n, D = 3, 29
    spec = EnvSpec(Box(np.zeros(n * D), np.ones(n * D)), Discrete(5))
    pol = CentralizedCategoricalMLPPolicy(spec, n)
    # 'auto' keeps autograd for CENT
    assert DevicePPO(pol, GaussianMLPBaseline(spec, hidden_sizes=(64, 64, 64)))._fused is None
    # the reference class default (32, 32) has two hidden layers: not a shape of the kernels
    with pytest.raises(NotImplementedError):
        DevicePPO(CentralizedCategoricalMLPPolicy(spec, n), GaussianMLPBaseline(spec, hidden_sizes=(32, 32)), fused=True)
    # the rollout blob and the update's blob map are one packing
    with torch.no_grad():
        for p in pol.parameters():
            p.add_(0.1 * torch.randn_like(p))
    assert torch.equal(pol._pack_blob(pol.state_dict()), pol.weight_blob())
    bl = GaussianMLPBaseline(spec, hidden_sizes=(64, 64, 64))
    assert bl._pack_blob(bl.state_dict()).numel() == N.lib().cm_baseline_mlp_blob_floats(n * D)
    # malformed gradient calls are rejected before any work
    buf = torch.zeros(1 << 16, device="cuda")
    for kind in (N.NET_POLICY_CENT, N.NET_BASELINE_MLP):
        desc = N.NetDesc(kind, n, D, 0, 0, 0.0, 0.9, 1.1, 0)
        io = N.NetIO()
        io.n_steps = 4
        io.weights = io.grad = io.obs = io.workspace = N.ptr(buf)
        io.workspace_floats = buf.numel()
        assert N.lib().cm_ppo_net(C.byref(desc), C.byref(io), N.stream_ptr()) == -1          # CM_EINVAL: no actions / adv, no returns
        if kind == N.NET_POLICY_CENT:
            io.actions = N.ptr(buf)
            assert N.lib().cm_ppo_net(C.byref(desc), C.byref(io), N.stream_ptr()) == -1      # adv still missing
    desc = N.NetDesc(N.NET_POLICY_CENT, 257, D, 0, 0, 0.0, 0.9, 1.1, 0)
    io = N.NetIO()
    io.n_steps, io.weights, io.obs, io.workspace, io.workspace_floats = 1, N.ptr(buf), N.ptr(buf), N.ptr(buf), buf.numel()
    assert N.lib().cm_ppo_net(C.byref(desc), C.byref(io), N.stream_ptr()) == -2               # CM_EUNSUPPORTED: n > 256
