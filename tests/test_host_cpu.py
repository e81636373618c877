"""CPU-side tests: the C-ABI library loads and exports what include/commarl_b200.h declares, the product's
host logic (scenario derivation, sharding, statistics, path truncation) agrees with the oracle's independent
restatement, the N>1 plumbing works under gloo with world_size 2, and the product refuses to run without a GPU."""
import os
import re
import socket
import sys

import numpy as np
import pytest
import torch

from golden_util import EnvCase, env_cases
from oracle import oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from com_marl_b200 import _native as N
    header = open(os.path.join(ROOT, "include", "commarl_b200.h")).read()
    declared = set(re.findall(r"\b(cm_[a-z_0-9]+)\s*\(", header))
    assert declared == set(N.EXPORTS), declared ^ set(N.EXPORTS)
    lib = N.lib()
    for sym in declared:
        assert getattr(lib, sym) is not None
    assert lib.cm_abi_version() == N.ABI_VERSION
    assert lib.cm_strerror(N.CM_EACTION) == b"Action Not found!"
    assert lib.cm_policy_blob_floats(21, 2) == 42309 and lib.cm_policy_blob_floats(53, 2) == 46405   # SURVEY.md §3.3
    assert lib.cm_policy_cent_blob_floats(4, 21) == 84 * 128 + 128 + 8256 + 2080 + 33 * 20   # n*D -> 128 -> 64 -> 32 -> 5n
    assert lib.cm_policy_workspace_bytes(32, 100) == 0 and lib.cm_policy_workspace_bytes(200, 4) == 4 * 3 * 200 * 64 * 4


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback():
    from com_marl_b200 import _native as N
    from com_marl_b200.envs import BatchedEnv
    from com_marl_b200.scenario import ScenarioSpec
    assert N.lib().cm_device_count() == 0
    buf = np.zeros(64, dtype=np.float32)
    assert N.lib().cm_mask_pack(buf.ctypes.data, buf.ctypes.data, 1, 4, None) == N.CM_ENODEVICE
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        BatchedEnv(ScenarioSpec.from_cli("pp", 10, 1, 0.04), 4)


@pytest.mark.parametrize("name", env_cases())
def test_scenario_spec_matches_oracle_derivation(name):
    """com_marl_b200.scenario (product) vs oracle.spec_from_params (checker): two independent restatements of
    PredatorPrey/Coverage.__init__ + init_communication, and both match what the reference reported."""
    from com_marl_b200.scenario import ScenarioSpec
    case = EnvCase(name)
    spec = ScenarioSpec.from_params(case.scenario, case.params, max_path_length=case.max_path_length,
                                    channel_type="GE" if case.ge else None)
    o = orc.spec_from_params(case.scenario, case.params, max_path_length=case.max_path_length, ge=case.ge)
    assert (spec.n_agents, spec.n_preys, spec.grid, spec.sensing, spec.max_steps, spec.n_layers) == \
        (o["n"], o["p"], o["G"], o["R"], o["T"], o["L"])
    assert spec.obs_dim == o["D"] == case.z["obs"].shape[1] // case.n
    assert spec.rcom2 == o["rcom2"] and spec.channel == o["chan_type"]
    assert spec.rcom == case.meta["Rcom"]
    for k in ("capture_reward", "step_cost", "moving_cost", "penalty", "lazy_penalty", "revisit_penalty", "final_reward"):
        assert getattr(spec, k) == o[k], k
    assert np.array_equal(spec.lut()[:2 * spec.grid], np.concatenate([o["lut_row"], o["lut_col"]]))
    if case.scenario == "pp":
        assert np.array_equal(spec.lut()[2 * spec.grid:], o["lut_t"])
    else:
        assert np.array_equal(spec.wall, o["wall"])
        assert spec.n_empty_cells == o["n_empty_cells"] == case.meta["n_empty_cells"]
        rows = spec.wall_rows()
        back = ((rows[:, None] >> np.arange(spec.grid, dtype=np.uint64)[None, :]) & np.uint64(1)).astype(np.uint8)
        assert np.array_equal(back, spec.wall)
    assert spec.bound_return == pytest.approx(case.meta["bound_return"], rel=0, abs=1e-12)
    d = spec.to_desc(None, None)
    assert d.p_loss == np.float32(case.meta["pl"])


def test_scenario_cli_sizing_rule():
    """n_agents = int(int(den*100) * (map/10)^2) for the five BASELINE.json configs (SURVEY.md §8)"""
    from com_marl_b200.scenario import ScenarioSpec
    want = {("pp", 10, 1, 0.04): (4, 21), ("co", 10, 1, 0.03): (3, 29), ("pp", 20, 2, 0.08): (32, 53),
            ("co", 30, 2, 0.06): (54, 77), ("pp", 50, 2, 0.08): (200, 53)}
    for (scen, m, sen, den), (n, D) in want.items():
        s = ScenarioSpec.from_cli(scen, m, sen, den, cap=4 if m > 10 else 2)
        assert (s.n_agents, s.obs_dim) == (n, D)
    with pytest.raises(ValueError):
        ScenarioSpec.from_cli("pp", 10, 1, 0.04, cap=5)
    with pytest.raises(ValueError):
        ScenarioSpec.from_cli("pp", 10, 1, 0.04, loss=0.2, channel_type="GE", GE_INIT=-1, loss_apply=0)
    with pytest.raises(ValueError):
        ScenarioSpec.from_cli("co", 15, 1, 0.03)


def test_shard_range_partitions_everything():
    from com_marl_b200.distributed import shard_range
    for total in (0, 1, 7, 16384, 65537):
        for world in (1, 2, 3, 8):
            spans = [shard_range(total, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1


def test_summarize_stats():
    from com_marl_b200.distributed import summarize_stats
    per_rank = torch.tensor([[2, 30.0, 400, 1, 6, 800, 3, 120, 0], [2, 10.0, 400, 0, 2, 800, 1, 40, 0]], dtype=torch.float64)
    s = summarize_stats(per_rank, "pp", 4)
    assert s["NumEpisodes"] == 4 and s["AverageReturn"] == 10.0 and s["SuccessRate"] == 0.25
    assert s["AverageStepCount"] == 200 and s["AverageCaptureCount"] == 2 and s["AverageMovingCount"] == 100.0


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _gloo_worker(rank, world, port, q):
    os.environ.update(RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1",
                      MASTER_PORT=str(port))
    sys.path.insert(0, ROOT)
    from com_marl_b200 import distributed as D
    r, lr, w = D.init_from_env(backend="gloo")
    lo, hi = D.shard_range(1001, r, w)
    local = torch.tensor([hi - lo, 10.0 * (r + 1), 3, 1, 0, 0, 0, 0, 0], dtype=torch.float64)
    out = D.gather_stats(local)
    # gradient bucket all-reduce (config 5's PPO data parallelism): rank r holds gradient r+1 everywhere
    lin = torch.nn.Linear(4, 3)
    for p in lin.parameters():
        p.grad = torch.full_like(p, float(r + 1))
    nfl = D.allreduce_gradients(lin)
    gmean = [float(p.grad.mean()) for p in lin.parameters()]
    # the PPO update's flat gradient bucket (com_marl_b200.ppo.FlatAdam): one all-reduce, parameters' .grad are views of it
    from com_marl_b200.ppo import FlatAdam
    lin2 = torch.nn.Linear(4, 3)
    fa = FlatAdam(lin2)
    fa.grad.fill_(float(r + 1))
    fa.all_reduce()
    gmean += [float(fa.grad.mean()), float(lin2.weight.grad.mean()), float(fa.flat.numel())]
    q.put((r, (out.tolist(), nfl, gmean)))
    torch.distributed.destroy_process_group()


def test_stats_all_gather_world_size_2_gloo():
    """The only collective on the path (episode statistics all-gather), on CPU with gloo and two ranks."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert res[0] == res[1]
    stats, nfl, gmean = res[0]
    assert [row[0] for row in stats] == [501.0, 500.0] and [row[1] for row in stats] == [10.0, 20.0]
    assert nfl == 15 and gmean == [1.5, 1.5, 1.5, 1.5, 15.0]


def test_truncate_paths():
    from com_marl_b200.sampler import _truncate_paths
    mk = lambda T: dict(rewards=np.zeros(T), observations=np.zeros((T, 8)), env_infos={"prey_alive": np.zeros((T, 2))},  # noqa: E731
                        success=np.zeros(3))
    out = _truncate_paths([mk(10), mk(10), mk(10)], max_samples=4 * 14, n_agents=4)
    assert [len(p["rewards"]) for p in out] == [10, 4]
    assert out[1]["observations"].shape == (4, 8) and out[1]["env_infos"]["prey_alive"].shape == (4, 2)


def test_ppo_data_parallel_update_world_size_2_gloo():
    """The PPO update's collectives under gloo with two ranks holding 4 and 5 paths: the weighted gradient all-reduce
    reproduces the single-process update on the union batch, both ranks end with identical weights, and the unequal local
    slice counts (2 vs 3 under 3 minibatches) do not deadlock (com_marl_b200.ppo.minibatch_plan)."""
    import ppo_dp_util
    from com_marl_b200.ppo import minibatch_plan
    assert minibatch_plan(4, 3) == [(0, 2), (2, 4)] and minibatch_plan(5, 3) == [(0, 2), (2, 4), (4, 5)]   # the reference's cut
    assert minibatch_plan(0, 3) == []
    single, ranks = ppo_dp_util.run("cpu")
    ppo_dp_util.check(single, ranks)


@pytest.mark.parametrize("kw", [dict(), dict(attention_type="dot", gcn_bias=False),
                                dict(encoder_hidden_sizes=(96,), embedding_dim=48, categorical_mlp_hidden_sizes=(100, 40, 24))])
def test_fused_update_blob_maps_round_trip(kw):
    """ppo_fused._BlobMap (host logic of the hand-written PPO update): the gather map derived from the module's own packing
    function reproduces the kernel weight blob from FlatAdam's flat bucket — transposes, zero padding of narrower layers, the
    constant identity of 'dot' attention — and the inverse map returns a blob-layout gradient to the flat gradient bucket."""
    import torch
    from com_marl_b200.policy import CommCategoricalMLPPolicy
    from com_marl_b200.ppo import CommBaseCritic, FlatAdam
    from com_marl_b200.ppo_fused import _BlobMap
    from com_marl_b200.spaces import Box, Discrete, EnvSpec
    torch.manual_seed(3)
    n, D = 5, 21
    spec = EnvSpec(Box(np.zeros(n * D), np.ones(n * D)), Discrete(5))
    ckw = {k: v for k, v in kw.items() if k != "categorical_mlp_hidden_sizes"}
    if "embedding_dim" in kw:
        ckw["decoder_hidden_sizes"] = (56,)
    for mod in (CommCategoricalMLPPolicy(spec, n, device="cpu", **kw), CommBaseCritic(spec, n, device="cpu", **ckw)):
        with torch.no_grad():
            for p in mod.parameters():
                p.add_(0.1 * torch.randn_like(p))
        opt = FlatAdam(mod)
        m = _BlobMap(mod, mod._pack_blob, opt.flat)
        assert torch.equal(m.refresh(), mod._pack_blob(mod.state_dict()))
        # after an in-place update of the bucket the refreshed blob follows (the parameters are views of it)
        opt.flat.mul_(1.5)
        assert torch.equal(m.refresh(), mod._pack_blob(mod.state_dict()))
        fake = {k: torch.randn_like(p) for k, p in mod.named_parameters()}
        m.grad.copy_(mod._pack_blob(fake))
        out = torch.empty_like(opt.grad)
        m.scatter_grad(out)
        assert torch.equal(out, torch.cat([fake[k].reshape(-1) for k, _ in mod.named_parameters()]))


def test_channel_draw_integer_threshold_is_the_float_compare():
    """env_kernel compares a channel draw as an integer (csrc/env_kernels.cu link_row_bits): u = (word >> 8) * 2^-24 in fp32,
    u >= thr <=> word >= ceil(thr * 2^24) << 8 and u < thr <=> word < ceil(thr * 2^24) << 8 for every fp32 threshold with
    0 < thr * 2^24 <= 2^24 - 1.  Checked here against the float compare the oracle (and the reference, with torch.rand's 24-bit
    lattice) performs: thresholds at the ends of the range, the loss rates of the BASELINE configs, random ones; words around
    the switching point of each threshold and random ones."""
    rng = np.random.default_rng(0)
    thrs = np.concatenate([np.float32([0.2, 0.1, 0.5, 0.3, 0.0196, 0.282, 0.999, 0.999999, 1e-6, 1e-7, 2.0 ** -24, 1.0 - 2.0 ** -24]),
                           rng.random(200, dtype=np.float32), np.float32(rng.random(100) * 1e-5)]).astype(np.float32)
    for thr in thrs:
        t24 = np.float32(thr) * np.float32(16777216.0)
        assert 0.0 < t24 <= 16777215.0
        T = int(np.ceil(t24))
        tw = np.uint64(T) << np.uint64(8)
        ks = np.clip(np.arange(T - 3, T + 4), 0, (1 << 24) - 1).astype(np.uint64)
        words = np.concatenate([(ks << np.uint64(8)), (ks << np.uint64(8)) | np.uint64(0xFF), rng.integers(0, 1 << 32, 64, dtype=np.uint64)])
        u = (words >> np.uint64(8)).astype(np.float32) * np.float32(5.9604644775390625e-08)      # common.cuh::u24
        assert np.array_equal(u >= thr, words >= tw), thr
        assert np.array_equal(u < thr, words < tw), thr
        # the diagonal link: u + 1 lies in [1, 2), never below / always at or above a threshold inside (0, 1)
        assert np.all((u + np.float32(1.0)) >= thr) and not np.any((u + np.float32(1.0)) < thr)


def test_action_stream_restatement_matches_oracle_philox():
    """tests/policy_kinds_util.py restates categorical_finish's in-kernel draw for the GPU tests: its numpy Philox4x32-10 equals
    the oracle's C implementation word for word (key = both halves of a 64-bit seed, counters near 2^32), u24 is (w >> 8) 2^-24
    on [0, 1), and action_u picks word il & 3 of block il >> 2 with the stream id 4 | episode << 8"""
    import policy_kinds_util as U
    rng = np.random.default_rng(0)
    for seed in (0, 7, 0x1234_5678_9ABC_DEF0, 2**64 - 1):
        c = rng.integers(0, 2**32, (64, 4), dtype=np.uint64)
        c[0] = 2**32 - 1
        got = U.philox4x32_10(seed, c[:, 0], c[:, 1], c[:, 2], c[:, 3])
        for i in range(len(c)):
            assert np.array_equal(got[i], orc.philox(seed, *(int(x) for x in c[i]))), (seed, i)
    w = np.array([0, 255, 256, 2**31, 2**32 - 1] + rng.integers(0, 2**32, 1000).tolist(), np.uint32)
    u = U.u24(w)
    assert u.dtype == np.float32 and (u >= 0).all() and (u < 1).all()
    assert np.array_equal(u.astype(np.float64), (w >> 8).astype(np.float64) / 2**24)
    assert u[1] == 0 and u[2] == 2**-24 and u[4] == 1 - 2**-24
    seed, env_id0, n = 99, 2**32 - 3, 10
    tick, episode = np.array([5, 2**31 - 1], np.int32), np.array([3, 2**24 - 1], np.int32)
    got = U.action_u(seed, env_id0, [0, 1], tick, episode, n)
    for e in range(2):
        for il in range(n):
            blk = orc.philox(seed, (env_id0 + e) % 2**32, int(tick[e]), (4 | int(episode[e]) << 8) % 2**32, il >> 2)
            assert got[e, il] == np.float32((int(blk[il & 3]) >> 8) * 2.0**-24), (e, il)
