"""Several policies in one cm_policy_forward launch (cm_policy_io.n_policies, PolicySet, eval_policies).

Every check is bit for bit against the same policies run one at a time: a PolicySet launch over P env blocks must equal P
single-policy launches, block i with env_id0 = i * envs_per_policy (probs, logits, actions, attention; greedy and sampled),
and eval_policies must equal eval_model per (policy, condition).  Each policy has distinct random weights and non-zero
biases, so a tile that reads another block's blob or a bias table left over from the previous tile's policy shows.
"""
import ctypes as C
import pickle

import pytest

import policy_set_util as U

# (kind, n, D, math, envs per policy, policies): every kVec / slot size of the Comm-DP tensor-core kernel, the large-team
# pipeline, Obs-DP (rows mode) and CENT in both maths.  Envs per policy are not multiples of the envs per tile and E n is not
# a multiple of 128.  With P = 64 the tensor-core cases have more than 296 tiles (2 CTAs x 148 SMs), so persistent CTAs walk
# tiles of several policies: the weight stream prefetches across a policy switch and the bias table is reloaded.
CASES = [("comm", n, 13, "tc", 37, 3) for n in (3, 4, 5, 6, 16, 17, 32, 33, 64)] + \
        [("comm", n, 13, "tc", 5, 3) for n in (65, 130, 200, 256)] + \
        [("dec", n, 13, "tc", E, 3) for n, E in ((4, 11), (32, 11), (200, 3))] + \
        [("cent", n, D, m, E, 3) for n, D, E in ((3, 13, 70), (32, 13, 130), (200, 5, 70)) for m in ("fp32", "tc")] + \
        [("comm", 32, 13, "tc", 37, P) for P in (1, 2, 7, 64)] + \
        [("dec", 32, 13, "tc", 20, 64), ("comm", 4, 13, "tc", 150, 64), ("comm", 65, 13, "tc", 9, 64)]


def _ids(c):
    return f"{c[0]}-n{c[1]}-D{c[2]}-{c[3]}-E{c[4]}-P{c[5]}"


def _policies(kind, n, D, math, P, base=100):
    return [U.make_policy(kind, n, D, math, seed=base + 31 * i) for i in range(P)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_ids)
def test_set_launch_equals_block_launches(case):
    from com_marl_b200.policy import PolicySet
    kind, n, D, math, Ep, P = case
    pols = _policies(kind, n, D, math, P)
    pset = PolicySet(pols)
    inp = U.inputs(kind, n, D, 2, P * Ep, seed=n * 1000 + P)
    for greedy in (True, False):
        ref = U.reference(pols, kind, n, inp, greedy)
        got = U.outputs(kind, n, P * Ep)
        U.call(pset, kind, inp, got, greedy)
        U.assert_same(f"{_ids(case)} greedy={greedy}", got, ref)


@pytest.mark.gpu
def test_group_slices_equal_whole_launch():
    """calls over slices that cut through policy blocks (what the rollout groups do) equal the whole-batch launch"""
    from com_marl_b200.policy import PolicySet
    kind, n, D, P, Ep = "comm", 32, 13, 5, 21
    pols = _policies(kind, n, D, "tc", P)
    pset = PolicySet(pols)
    inp = U.inputs(kind, n, D, 2, P * Ep, seed=5)
    ref = U.reference(pols, kind, n, inp, False)
    got = U.outputs(kind, n, P * Ep)
    for b0, b1 in ((0, 10), (10, 50), (50, 51), (51, 105)):
        U.call(pset, kind, inp, got, False, env_id0=b0, sl=slice(b0, b1), envs_per_policy=Ep, first_env=b0)
    U.assert_same("slices", got, ref)


def _raw_call(pset, kind, inp, out, **over):
    """cm_policy_forward with a hand-edited multi-policy io struct -> return code"""
    from com_marl_b200 import _native as N
    p0 = pset.policies[0]
    B = inp["obs"].shape[0]
    desc, io = p0._call_structs(inp["obs"], inp.get("adj_bits"), inp.get("chan_bits"), inp["avail_bits"], None, inp["tick"],
                                inp["episode"], True, out["probs"], out["logits"], out.get("attention"), out["actions"], 0, 0)
    io.weights, io.n_policies, io.envs_per_policy = N.ptr(pset._blobs), len(pset), B // len(pset)
    io.weights_stride, io.tc_weights_stride = pset._stride, pset._tc_stride
    if pset._tc_blobs is not None:
        io.tc_weights = N.ptr(pset._tc_blobs)
    for k, v in over.items():
        setattr(io, k, v)
    return N.lib().cm_policy_forward(C.byref(desc), C.byref(io), N.stream_ptr())


@pytest.mark.gpu
@pytest.mark.parametrize("kind,math", [("comm", "tc"), ("dec", "tc"), ("cent", "tc"), ("cent", "fp32")])
def test_invalid_blocks_and_strides(kind, math):
    import torch
    from com_marl_b200 import _native as N
    from com_marl_b200.policy import PolicySet
    n, D, P, Ep = 8, 13, 3, 10
    pset = PolicySet(_policies(kind, n, D, math, P))
    inp = U.inputs(kind, n, D, 2, P * Ep, seed=1)
    out = U.outputs(kind, n, P * Ep)
    assert _raw_call(pset, kind, inp, out) == N.CM_OK
    torch.cuda.synchronize()
    before = {k: v.clone() for k, v in out.items()}
    bad = [dict(envs_per_policy=Ep - 1), dict(envs_per_policy=0), dict(n_policies=-1), dict(n_envs=P * Ep + 1),
           dict(weights_stride=pset._stride - 4), dict(weights_stride=pset._stride + 1)]
    if pset._tc_blobs is not None:
        bad += [dict(tc_weights_stride=pset._tc_stride - 4), dict(tc_weights_stride=pset._tc_stride + 2)]
    for over in bad:
        assert _raw_call(pset, kind, inp, out, **over) == N.CM_EINVAL, over
    torch.cuda.synchronize()
    for k in out:
        assert torch.equal(out[k].nan_to_num(1.0), before[k].nan_to_num(1.0)), k


@pytest.mark.gpu
def test_host_calls_reject_policy_sets():
    from com_marl_b200 import _native as N
    L = N.lib()
    desc = N.PolicyDesc(8, 13, 2, 1, 1, 1, 1, 0, N.POLICY_COMM)
    dev, host = N.PolicyIO(), N.PolicyIO()
    dev.n_envs, dev.n_policies, dev.envs_per_policy = 6, 2, 3
    assert L.cm_policy_forward_host(C.byref(desc), C.byref(dev), C.byref(host), -1, None) == N.CM_EUNSUPPORTED
    env_desc, state, env_dev, env_host = N.EnvDesc(), N.EnvState(), N.StepIO(), N.StepIO()
    env_desc.n_agents, state.n_envs = 8, 6
    dev.actions = env_dev.actions = 64
    dev.obs = env_dev.obs = 128
    assert L.cm_rollout_step_host(C.byref(desc), C.byref(dev), C.byref(host), C.byref(env_desc), C.byref(state),
                                  C.byref(env_dev), C.byref(env_host), None) == N.CM_EUNSUPPORTED


@pytest.mark.gpu
def test_mismatched_architectures_raise():
    from com_marl_b200.policy import PolicySet
    a = U.make_policy("comm", 8, 13, "tc", seed=1)
    for other in (U.make_policy("comm", 8, 13, "tc", seed=2, L=3),
                  U.make_policy("comm", 9, 13, "tc", seed=2), U.make_policy("comm", 8, 12, "tc", seed=2),
                  U.make_policy("dec", 8, 13, "tc", seed=2), U.make_policy("cent", 8, 13, "tc", seed=2)):
        with pytest.raises(ValueError):
            PolicySet([a, other])
    with pytest.raises(ValueError):
        PolicySet([U.make_policy("cent", 8, 13, "fp32", seed=1), U.make_policy("cent", 8, 13, "fp32", seed=2, relu=True)])
    with pytest.raises(ValueError):                # the same CENT architecture on the other math
        PolicySet([U.make_policy("cent", 8, 13, "tc", seed=1), U.make_policy("cent", 8, 13, "fp32", seed=2)])


def _spec(size):
    import channel_sweep_util as CS
    return CS.base_spec(size)


def _engine_policies(spec, kind, P, base):
    from com_marl_b200.rollout import make_policy
    return [make_policy(spec, kind=kind, torch_seed=base + i) for i in range(P)]


@pytest.mark.gpu
def test_captured_graph_sees_member_updates():
    """a captured multi-policy rollout graph uses a member's new weights (load_state_dict; p.data + refresh_weights(force=True))
    for that block only: every chunk equals per-policy engines that get the same updates"""
    import torch
    from com_marl_b200.policy import PolicySet
    from com_marl_b200.rollout import RolloutEngine
    spec, P, E, K = _spec("pp_n32"), 3, 8, 4
    set_pols, ref_pols = _engine_policies(spec, "comm", P, 10), _engine_policies(spec, "comm", P, 10)
    donor = _engine_policies(spec, "comm", 1, 99)[0]
    eng = RolloutEngine(spec, PolicySet(set_pols), P * E, ring=K, groups=2)
    refs = [RolloutEngine(spec, p, E, env_id0=i * E, ring=K) for i, p in enumerate(ref_pols)]
    for e in [eng] + refs:
        e.reset()

    def update(step, pols, pset_like):
        if step == 2:
            pols[1].load_state_dict(donor.state_dict())
        if step == 3:
            with torch.no_grad():
                for p in pols[2].parameters():
                    p.data.add_(0.05)
            for p in pset_like:
                p.refresh_weights(force=True)

    for step in range(5):
        update(step, set_pols, [eng.policy])
        update(step, ref_pols, ref_pols)
        for e in [eng] + refs:
            e.run_chunk()
        torch.cuda.synchronize()
        for i, r in enumerate(refs):
            for k in ("actions", "probs", "reward", "obs"):
                assert torch.equal(eng.traj[k][:, i * E:(i + 1) * E].cpu(), r.traj[k].cpu()), (step, i, k)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["comm", "dec", "cent"])
def test_engine_groups_cut_through_blocks(kind):
    import torch
    from com_marl_b200.policy import PolicySet
    from com_marl_b200.rollout import RolloutEngine
    spec, P, E = _spec("pp_n32"), 3, 10
    pset = PolicySet(_engine_policies(spec, kind, P, 40))
    trajs = []
    for groups in (1, 4):
        eng = RolloutEngine(spec, pset, P * E, ring=4, groups=groups)
        eng.reset()
        eng.run(8)
        torch.cuda.synchronize()
        trajs.append({k: v.cpu() for k, v in eng.traj.items()})
        # per step: one env launch per group and the policy calls of each group's segments (groups of 4: 1 + 2 + 2 + 1)
        calls = sum(len(PolicySet.segments(b1 - b0, E, b0)) for b0, b1 in eng._ranges)
        assert eng.kernel_launches == 8 * (len(eng._ranges) + calls), (groups, eng.kernel_launches)
    for k in trajs[0]:
        assert torch.equal(trajs[0][k], trajs[1][k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("size,kind", [("pp_n4", "comm"), ("pp_n32", "comm"), ("pp_n32", "dec"), ("pp_n32", "cent"),
                                       ("co_n54", "comm"), ("pp_n200", "comm")])
@pytest.mark.parametrize("grid", [False, True])
def test_eval_policies_equals_eval_model(size, kind, grid):
    from com_marl_b200.evaluate import eval_model, eval_policies
    spec = _spec(size)
    P, E = 3, 6
    pols = _engine_policies(spec, kind, P, 70)
    conds = [spec.with_channel(**t) for t in U.CHANNEL_TABLE] if grid else None
    C_ = len(conds) if grid else 1
    res = eval_policies(spec, pols, conditions=conds, n_eval_episodes=E, max_env_steps=10, groups=4, chunk=4)
    assert len(res) == P and all(len(r) == C_ for r in res)
    for i, p in enumerate(pols):
        for k in range(C_):
            ref = eval_model(conds[k] if grid else spec, p, n_eval_episodes=E, max_env_steps=10, groups=1, chunk=4,
                             env_id0=(i * C_ + k) * E)
            assert pickle.dumps(res[i][k]) == pickle.dumps(ref), (i, k)


@pytest.mark.gpu
def test_member_graph_keeps_following_member():
    """a set built on a policy leaves the policy's own blobs alone: an engine captured on it still sees its updates"""
    import torch
    from com_marl_b200.evaluate import eval_policies
    from com_marl_b200.policy import PolicySet
    from com_marl_b200.rollout import RolloutEngine
    spec, E = _spec("pp_n32"), 8
    pol, ref = _engine_policies(spec, "comm", 1, 5)[0], _engine_policies(spec, "comm", 1, 5)[0]
    donor = _engine_policies(spec, "comm", 1, 99)[0]
    engs = [RolloutEngine(spec, p, E, ring=4) for p in (pol, ref)]
    for e in engs:
        e.reset()
    for step in range(4):
        if step == 2:                              # the member's graph is captured; a set and an evaluation use the member
            PolicySet([pol, donor])
            eval_policies(spec, [pol, donor], n_eval_episodes=3, max_env_steps=4, chunk=4)
            for p in (pol, ref):
                p.load_state_dict(donor.state_dict())
        for e in engs:
            e.run_chunk()
        torch.cuda.synchronize()
        for k in ("actions", "probs", "obs"):
            assert torch.equal(engs[0].traj[k].cpu(), engs[1].traj[k].cpu()), (step, k)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["comm", "cent"])
def test_repeated_policy(kind):
    """one policy object in several blocks: every block runs it"""
    from com_marl_b200.evaluate import eval_model, eval_policies
    spec, E = _spec("pp_n32"), 5
    p, q = _engine_policies(spec, kind, 2, 60)
    pols = [p, q, p, p]
    res = eval_policies(spec, pols, n_eval_episodes=E, max_env_steps=10, groups=3, chunk=4)
    for i, pol in enumerate(pols):
        ref = eval_model(spec, pol, n_eval_episodes=E, max_env_steps=10, groups=1, chunk=4, env_id0=i * E)
        assert pickle.dumps(res[i][0]) == pickle.dumps(ref), i


@pytest.mark.gpu
def test_auto_and_tc_math_share_a_set():
    """math='auto' runs the same tensor-core kernel as math='tc': one set takes both"""
    from com_marl_b200.policy import PolicySet
    n, D, Ep = 8, 13, 9
    pols = [U.make_policy("comm", n, D, "auto", seed=1), U.make_policy("comm", n, D, "tc", seed=2)]
    pset = PolicySet(pols)
    inp = U.inputs("comm", n, D, 2, 2 * Ep, seed=3)
    got = U.outputs("comm", n, 2 * Ep)
    U.call(pset, "comm", inp, got, False)
    U.assert_same("auto+tc", got, U.reference(pols, "comm", n, inp, False))


def test_policy_blocks_must_divide_envs():
    import channel_sweep_util as CS
    from com_marl_b200.envs import check_conditions
    spec = CS.base_spec("pp_n32")
    conds = [spec.with_channel(**t) for t in U.CHANNEL_TABLE]
    assert check_conditions(spec, conds, 18, policy_blocks=2) == conds
    for n_envs, blocks in ((10, 3), (19, 2), (18, 0)):
        with pytest.raises(ValueError):
            check_conditions(spec, conds, n_envs, policy_blocks=blocks)
    with pytest.raises(ValueError):
        check_conditions(spec, None, 10, policy_blocks=3)


def test_segments_cover_the_range():
    from com_marl_b200.policy import PolicySet
    for Ep in (1, 5, 18):
        for first in range(0, 3 * Ep):
            for B in range(1, 4 * Ep):
                segs = PolicySet.segments(B, Ep, first)
                assert segs[0][0] == 0 and segs[-1][1] == B
                for (s0, s1, i, whole), nxt in zip(segs, segs[1:] + [None]):
                    assert nxt is None or nxt[0] == s1
                    assert i == (first + s0) // Ep
                    if whole:
                        assert (first + s0) % Ep == 0 and s1 - s0 == whole * Ep and whole >= 2
                    else:
                        assert (first + s1 - 1) // Ep == i
