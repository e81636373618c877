"""Training and evaluation grids sharded by member over ranks (DeviceTrainerSet(group=...), eval_policies(group=...)).

Every multi-rank case runs as spawned worker processes over gloo: rank r on cuda:r when two GPUs are visible, both ranks on
cuda:0 otherwise.  The same worker run as one process is the reference, so each case compares the two-rank grid against the
single-rank set or evaluation with the same arguments.  The member plan and the result gather also run on CPU.
"""
import os
import socket
import sys
import traceback

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BATCH_KEYS = ("obs", "actions", "rewards", "valids", "adj_bits", "chan_bits", "baselines", "returns", "adv")
EPISODE_KEYS = ("Iteration", "NumTrajs", "AverageDiscountedReturn", "AverageReturn", "StdReturn", "MaxReturn", "MinReturn",
                "SuccessRate", "AverageCaptureCount", "AverageStepCount", "AverageMovingCount", "AveragePenaltyCount",
                "AverageVariable", "AverageVar2", "AveDegree", "Diameter", "AveTroughput")


# ---- process harness -------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, q, case, gpu):
    try:
        os.environ.update(RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1",
                          MASTER_PORT=str(port))
        sys.path.insert(0, ROOT)
        import torch
        import torch.distributed as dist
        torch.set_num_threads(1)
        if gpu:
            torch.cuda.set_device(rank if torch.cuda.device_count() >= 2 else 0)
        if world > 1:
            dist.init_process_group(backend="gloo", rank=rank, world_size=world)
        try:
            out = CASES[case](rank, world)
        finally:
            if world > 1:
                dist.destroy_process_group()
        q.put((rank, "ok", out))
    except BaseException:
        q.put((rank, "error", traceback.format_exc()))


def _launch(case, world, gpu=True, timeout=300):
    """{rank: what CASES[case] returned} of `world` spawned ranks; no process outlives the call"""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q, case, gpu)) for r in range(world)]
    try:
        for p in procs:
            p.start()
        res = {}
        for _ in range(world):
            r, status, out = q.get(timeout=timeout)
            assert status == "ok", f"rank {r} of {world}:\n{out}"
            res[r] = out
        for p in procs:
            p.join(timeout=120)
            assert p.exitcode == 0, p.exitcode
        return res
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
            if p.pid is not None:
                p.join(timeout=30)


# ---- cases (run inside the workers) ----------------------------------------------------------------------------------
def _c3_shape():
    from com_marl_b200.scenario import ScenarioSpec
    return ScenarioSpec.from_cli("pp", 20, 2, 0.08, cap=4, loss=0.2, seed=5, max_env_steps=24)      # C3's team, map and channel


def _c1_shape():
    from com_marl_b200.scenario import ScenarioSpec
    return ScenarioSpec.from_cli("pp", 10, 1, 0.04, cap=2, seed=7)


def _np_state(module):
    return {k: v.detach().cpu().numpy().copy() for k, v in module.state_dict().items()}


def _trainer_case(rank, world):
    """round 1 and 2 of a 3-member set: per owned member the trajectory, batch, weights before / after round 1; the K dicts;
    after round 2 whether the PolicySet rows follow the updated policies, and the gathered state dicts"""
    import torch
    from com_marl_b200.train import DeviceTrainerSet
    E, seeds, env_id0 = 6, [3, 8, 13], 100
    spec = _c3_shape()
    S = DeviceTrainerSet(spec, E, seeds, conditions=[None, spec.with_channel(pl=0.3), None], env_id0=env_id0,
                         optimization_mini_epochs=2)
    own = list(S.members)
    init = {i: (_np_state(S.policies[i]), _np_state(S.critics[i])) for i in own}
    blob0 = {i: S.policies[i].weight_blob().clone() for i in own}
    outs = S.train_epoch()
    torch.cuda.synchronize()
    blob1 = {i: S.policies[i].weight_blob().clone() for i in own}
    got = dict(members=own, init=init, outs=outs,
               traj={i: {k: v.cpu().numpy() for k, v in S.member_traj(i).items()} for i in own},
               batch={i: {k: S.batches[i][k].cpu().numpy() for k in BATCH_KEYS} for i in own},
               after={i: (_np_state(S.policies[i]), _np_state(S.critics[i])) for i in own})
    outs2 = S.train_epoch()
    torch.cuda.synchronize()
    got["round2"] = [o["tabular"]["Iteration"] for o in outs2]
    # the set's rows hold the weights round 2 rolled out with (the rollout's refresh is the only writer): the round-1 update,
    # not the initial weights; the next rollout's refresh brings in the round-2 update
    rows = S.pset._blobs[:, :S.pset._n_blob]
    got["round2_rolled_out_round1_update"] = all(torch.equal(rows[j], blob1[i]) and not torch.equal(blob1[i], blob0[i])
                                                 for j, i in enumerate(own))
    S.pset.refresh_weights()
    got["rows_follow"] = all(not torch.equal(blob1[i], S.policies[i].weight_blob()) and
                             torch.equal(rows[j], S.policies[i].weight_blob()) for j, i in enumerate(own))
    got["state_dicts"] = [{k: v.numpy() for k, v in sd.items()} for sd in S.policy_state_dicts()]
    return got


def _eval_case(rank, world):
    """eval_policies results of 4 policies x 2 conditions, 3 policies as a PolicySet and 1 policy"""
    from com_marl_b200.evaluate import eval_policies
    from com_marl_b200.policy import PolicySet
    from com_marl_b200.rollout import make_policy
    spec = _c1_shape()
    pols = [make_policy(spec, torch_seed=70 + i) for i in range(4)]
    conds = [spec.with_channel(pl=0.3), spec.with_channel(pl=0.2, rcom=1)]
    kw = dict(n_eval_episodes=20, return_trajectory=True)
    return dict(four=eval_policies(spec, pols, conditions=conds, **kw),
                three=eval_policies(spec, PolicySet(pols[:3]), conditions=conds, **kw),
                one=eval_policies(spec, pols[3:], **kw))


def _errors_case(rank, world):
    """the exception each misuse raises on this rank"""
    from com_marl_b200.train import DeviceTrainerSet
    spec = _c1_shape()
    caught = {}

    def attempt(name, fn):
        try:
            fn()
            caught[name] = None
        except Exception as e:                 # noqa: BLE001 (the type is the result)
            caught[name] = type(e).__name__

    attempt("unequal_seeds", lambda: DeviceTrainerSet(spec, 4, [1, 2 + rank]))
    attempt("unequal_envs", lambda: DeviceTrainerSet(spec, 4 + rank, [1, 2]))
    attempt("one_member", lambda: DeviceTrainerSet(spec, 4, [1]))
    attempt("cent", lambda: DeviceTrainerSet(spec, 4, [1, 2], kind="cent"))
    S = DeviceTrainerSet(spec, 4, [1, 2, 3])
    other = 2 if rank == 0 else 0
    attempt("member_traj", lambda: S.member_traj(other))
    attempt("policies", lambda: S.policies[other])
    attempt("own_member_traj", lambda: S.member_traj(S.members[0]))
    caught["members"] = list(S.members)
    # a set over a group of this rank alone inside a job of two ranks: a single-rank set, its members' collectives on the rank
    import torch.distributed as dist
    alone = dist.new_group([rank], use_local_synchronization=True)
    attempt("alone_group", lambda: DeviceTrainerSet(spec, 4, [1 + rank, 5], group=alone).train_epoch())
    attempt("data_parallel", lambda: DeviceTrainerSet(spec, 4, [1, 2], process_group=dist.group.WORLD))
    return caught


def _gather_case(rank, world):
    from com_marl_b200 import distributed as D
    got = D.gather_objects(dict(rank=rank, payload=list(range(rank + 2))))
    try:
        D.check_same_on_all_ranks("seeds", [1, 2 + rank])
        err = None
    except ValueError:
        err = "ValueError"
    D.check_same_on_all_ranks("seeds", [1, 2])                        # equal: no error
    alone = D.rank_alone_group()
    return dict(gathered=got, err=err, alone=(D.group_rank_world(alone), D.gather_objects(rank, alone)))


CASES = dict(trainer=_trainer_case, eval=_eval_case, errors=_errors_case, gather=_gather_case)


# ---- tests -----------------------------------------------------------------------------------------------------------
def _assert_same(a, b, where=()):
    """a == b bit for bit, by value: the same structure and types, arrays of the same dtype, shape and bytes, floats of the
    same bits"""
    assert type(a) is type(b), (where, type(a), type(b))
    if isinstance(a, (list, tuple)):
        assert len(a) == len(b), (where, len(a), len(b))
        for i, (x, y) in enumerate(zip(a, b)):
            _assert_same(x, y, where + (i,))
    elif isinstance(a, dict):
        assert list(a) == list(b), (where, list(a), list(b))
        for k in a:
            _assert_same(a[k], b[k], where + (k,))
    elif isinstance(a, (np.ndarray, np.generic)):
        assert a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes(), where
    elif isinstance(a, float):
        assert np.float64(a).tobytes() == np.float64(b).tobytes(), (where, a, b)
    else:
        assert a == b, (where, a, b)


@pytest.mark.gpu
def test_trainer_grid_equals_single_rank_set():
    ref = _launch("trainer", 1)[0]
    ranks = _launch("trainer", 2)
    owner = {i: r for r, g in ranks.items() for i in g["members"]}
    assert ranks[0]["members"] == [0, 1] and ranks[1]["members"] == [2]
    assert ranks[0]["outs"] == ranks[1]["outs"]                       # the same K dicts on both ranks, member order
    assert [o["rank"] for o in ranks[0]["outs"]] == [0, 0, 1] and [o["rank"] for o in ref["outs"]] == [0, 0, 0]
    assert set(ranks[0]["outs"][0]) == set(ref["outs"][0])
    for i in range(3):
        g, o, r = ranks[owner[i]], ranks[0]["outs"][i], ref["outs"][i]
        for k in ref["traj"][i]:                                      # the trajectory ring, bit for bit
            assert np.array_equal(g["traj"][i][k], ref["traj"][i][k]), (i, k)
        for k in BATCH_KEYS:                                          # the padded batch, baselines, returns, advantages
            assert np.array_equal(g["batch"][i][k], ref["batch"][i][k]), (i, k)
        for a, b in zip(g["init"][i], ref["init"][i]):
            assert all(np.array_equal(a[k], b[k]) for k in b), i
        # the update: a set of 2 (1) members instead of 3 differs only in the order of fp32 atomic sums
        assert len(o["losses"]) == len(r["losses"])
        assert abs(o["loss_before"] - r["loss_before"]) <= 2e-5
        assert np.abs(np.array(o["losses"]) - r["losses"]).max() <= 1e-4
        assert np.abs(np.array(o["grad_norms"]) - r["grad_norms"]).max() <= 1e-3 * max(1.0, np.abs(r["grad_norms"]).max())
        assert abs(o["kl"] - r["kl"]) <= 1e-5
        for j in (0, 1):
            for k, b in ref["after"][i][j].items():
                a, b0 = g["after"][i][j][k], ref["init"][i][j][k]
                assert np.abs(a - b).max() <= 0.02 * np.abs(b - b0).max() + 1e-6, (i, j, k)
        for k in EPISODE_KEYS:
            assert o["tabular"][k] == r["tabular"][k], (i, k)
        assert o["episode_stats"] == r["episode_stats"]
    # round 2 on both ranks rolled out with the round-1 update, and the next rollout takes the round-2 update; the gathered
    # weights agree on both ranks
    for g in ranks.values():
        assert g["round2_rolled_out_round1_update"] and g["rows_follow"] and g["round2"] == [1, 1, 1]
    a, b = ranks[0]["state_dicts"], ranks[1]["state_dicts"]
    assert len(a) == len(b) == 3
    assert all(set(x) == set(y) and all(np.array_equal(x[k], y[k]) for k in x) for x, y in zip(a, b))
    assert all(set(x) == set(ref["state_dicts"][0]) for x in a)


@pytest.mark.gpu
def test_eval_grid_equals_single_rank_eval_policies():
    ref = _launch("eval", 1)[0]
    ranks = _launch("eval", 2)
    for key in ("four", "three", "one"):
        for r in (0, 1):
            _assert_same(ranks[r][key], ref[key], (key, r))
    res = ref["four"]
    assert len(res) == 4 and all(len(x) == 2 for x in res) and len(res[0][0]) == 6       # return_trajectory: 6 fields


@pytest.mark.gpu
def test_grid_errors():
    ranks = _launch("errors", 2)
    for r, c in ranks.items():
        assert c["unequal_seeds"] == "ValueError" and c["unequal_envs"] == "ValueError", (r, c)
        assert c["one_member"] == "ValueError", (r, c)
        assert c["cent"] == "NotImplementedError", (r, c)
        assert c["member_traj"] == "KeyError" and c["policies"] == "KeyError", (r, c)
        assert c["own_member_traj"] is None, (r, c)
        assert c["alone_group"] is None and c["data_parallel"] == "NotImplementedError", (r, c)
    assert ranks[0]["members"] == [0, 1] and ranks[1]["members"] == [2]


def test_member_range_covers_every_member_once():
    from com_marl_b200.distributed import member_range
    for K in range(1, 71):
        for W in range(1, 9):
            spans = [member_range(K, r, W) for r in range(W)]
            assert spans[0][0] == 0 and spans[-1][1] == K
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1 and sum(sizes) == K


def test_gather_objects_rank_order_gloo():
    ranks = _launch("gather", 2, gpu=False, timeout=180)
    for r, g in ranks.items():
        assert g["gathered"] == [dict(rank=0, payload=[0, 1]), dict(rank=1, payload=[0, 1, 2])]
        assert g["err"] == "ValueError"
        assert g["alone"] == ((0, 1), [r])
    from com_marl_b200.distributed import gather_objects
    assert gather_objects({"a": 1}) == [{"a": 1}]                     # no process group: identity
