"""Every launch path of the PPO update kernels (cm_ppo_net) against float64 (helpers: tests/ppo_path_util.py).

A: Comm-DP at every team size 1 .. 256.  B: every observation width 1 .. 128 at n = 4 and 40, Comm-DP and Obs-DP.  C: 1 to 4
layers x residual on / off x 'general' / 'dot' attention at both sides of every band edge, narrow layers at three.  D: chunked
walks at 3 and 4 layers with W = 1, 2 and 7 mask words per row.  E: Obs-DP at every team size.  F: CENT and the MLP baseline at
every n with K = n·D over every residue of the wide kernels' chunk and panel widths.  G: a profiler trace shows that every
instantiation the launch code can select is launched, and each traced call launches exactly the predicted set.

Each case compares per-step ll / entropy / probs / values and the policy and critic losses with a float64 evaluation of the
same modules, and every policy and critic gradient with the float64 gradient at the kernels' own fp32 forward (each step's
ratio and value taken from the kernels: ppo_path_util.grads_at_kernel_forward says why), all under ppo_scale_util's
tolerances; every comparison fails on NaN.  Each test prints one
JSON line with its worst normalised errors, appended to $PPO_PATHS_REPORT when that is set."""
import json
import math
import os
import time

import pytest

import ppo_path_util as U


def _report(rec):
    line = json.dumps(rec, sort_keys=True)
    print(line)
    path = os.environ.get("PPO_PATHS_REPORT")
    if path:
        with open(path, "a") as fh:
            fh.write(line + "\n")


def _run(part, label, cases):
    import torch
    t0 = time.time()
    worst, fails = {}, []
    for c in cases:
        rec, f = U.check_case(c)
        fails += f
        for k in ("out", "loss", "critic_loss", "grad", "critic_grad", "grad_plain", "critic_grad_plain", "chunk_agree",
                  "chunked_grad", "chunked_critic_grad"):
            if k in rec:
                e = rec[k]
                worst[k] = e if (math.isnan(e) or k not in worst) else (worst[k] if math.isnan(worst[k]) else max(worst[k], e))
        worst["min_prob64"] = min(worst.get("min_prob64", 1.0), rec["min_prob64"])
        if "dot_att_blob_grad" in rec:
            worst["dot_att_blob_grad"] = max(worst.get("dot_att_blob_grad", 0.0), rec["dot_att_blob_grad"])
    torch.cuda.empty_cache()
    _report(dict(part=part, group=label, cases=len(cases), worst=worst,
                 tol=dict(out=U.TOL["out"], loss=U.TOL["loss"], critic_loss=U.TOL["critic_loss"], grad=U.TOL["grad"],
                          critic_grad=U.TOL["critic_grad"], chunk_agree=U.CHUNK_AGREE),
                 seconds=round(time.time() - t0, 2), gpu=torch.cuda.get_device_name()))
    assert not fails, fails[:20]


@pytest.mark.gpu
@pytest.mark.parametrize("band", range(len(U.BANDS)), ids=U.BAND_IDS)
def test_a_comm_every_team_size(band):
    _run("A", U.BAND_IDS[band], U.cases_a(band))


@pytest.mark.gpu
@pytest.mark.parametrize("half", [0, 1], ids=["D1-64", "D65-128"])
@pytest.mark.parametrize("n", U.B_TEAMS)
@pytest.mark.parametrize("kind", U.B_KINDS)
def test_b_every_observation_width(kind, n, half):
    _run("B", f"{kind}-n{n}-half{half}", U.cases_b(kind, n, half))


@pytest.mark.gpu
@pytest.mark.parametrize("n", U.C_TEAMS)
def test_c_architecture_matrix(n):
    _run("C", f"n{n}", U.cases_c(n))


@pytest.mark.gpu
@pytest.mark.parametrize("L", [3, 4])
@pytest.mark.parametrize("i", range(len(U.D_CASES)), ids=[f"n{d['n']}" for d in U.D_CASES])
def test_d_chunked_walk(i, L):
    _run("D", f"n{U.D_CASES[i]['n']}-L{L}", U.cases_d(i, L))


@pytest.mark.gpu
@pytest.mark.parametrize("band", range(len(U.BANDS)), ids=U.BAND_IDS)
def test_e_obs_dp_every_team_size(band):
    _run("E", U.BAND_IDS[band], U.cases_e(band))


@pytest.mark.gpu
@pytest.mark.parametrize("band", range(len(U.BANDS)), ids=U.BAND_IDS)
def test_f_cent_every_team_size(band):
    _run("F", U.BAND_IDS[band], U.cases_f(band))


@pytest.mark.gpu
def test_g_every_reachable_instantiation_is_launched(tmp_path):
    """trace the policy and critic backward calls of coverage_cases(): each launches exactly predicted_kernels, and between
    them every EXPECTED instantiation runs (the Obs-DP ones at D = 40 and 68 from the observation layer alone)"""
    import torch
    from ppo_scale_util import kernel_launches
    seen, mism = {}, []
    for c in U.coverage_cases():
        fused, _, b0, ids = U.make_case(c, seed=c["n"] + c["D"])
        bf = fused.finish_batch(dict(b0))
        F, f = fused._fused, bf["_flat"]
        idx, idx_all = F.step_index(f, ids, valid_only=True), F.step_index(f, ids, valid_only=False)
        F.pol_map.refresh()
        F.cri_map.refresh()
        runs = dict(policy=lambda: F.policy_call(f, idx, adv=bf["adv"].reshape(-1).index_select(0, idx), backward=True,
                                                 inv_count=1.0 / idx.numel()),
                    critic=lambda: F.critic_call(f, idx_all, returns=bf["returns"].reshape(-1).index_select(0, idx_all), backward=True))
        for call, run in runs.items():
            if c["kind"] == "dec" and call == "critic":
                continue
            run()
            torch.cuda.synchronize()
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                run()
                torch.cuda.synchronize()
            trace = tmp_path / f"{c['id']}_{call}.json"
            prof.export_chrome_trace(str(trace))
            got = {k for k in (U.kernel_name(nm) for nm, _ in kernel_launches(str(trace))) if k}
            want = U.predicted_kernels(c["kind"], c["n"], c["D"], call, relu=c["relu"])
            if got != want:
                mism.append((c["id"], call, sorted(got - want), sorted(want - got)))
            for k in got:
                seen.setdefault(k, []).append(f"{c['id']}/{call}")
        del fused, bf, F, f
        torch.cuda.empty_cache()
    _report(dict(part="G", launched={k: v[0] for k, v in sorted(seen.items())}, gpu=torch.cuda.get_device_name()))
    assert not mism, mism
    assert set(U.EXPECTED) <= set(seen), sorted(set(U.EXPECTED) - set(seen))
    assert not set(U.UNREACHABLE) & set(seen)
    # the bulk-copy observation layer at K not in {32, 64, 128}: Obs-DP policy calls have no other N = 128 layer
    obs_async = {"net_dense_fwd_kernel<128,1,1>": ("n40-D40", "n40-D68"), "net_dense_bwd_kernel<128,64,64,1,0>": ("n40-D40",),
                 "net_dense_bwd_kernel<128,128,64,1,0>": ("n40-D68",)}
    for k, where in obs_async.items():
        for w in where:
            assert any(s.startswith(f"B-dec-{w}-") and s.endswith("/policy") for s in seen[k]), (k, w, seen[k])
    assert any(s.startswith("A-comm-n1-") for s in seen["net_small_agg_bwd_kernel"])
    assert any(s.startswith("A-comm-n213-") for s in seen["net_agg_bwd_kernel<7,256>"])


# ---- CPU: the case tables and the restated selection -------------------------------------------------------------------------
def test_case_tables_cover_the_matrix():
    a = [c["n"] for b in range(len(U.BANDS)) for c in U.cases_a(b)]
    assert a == list(range(1, 257)) and all(c["D"] % 2 for b in range(len(U.BANDS)) for c in U.cases_a(b))
    for kind in U.B_KINDS:
        for n in U.B_TEAMS:
            assert [c["D"] for h in (0, 1) for c in U.cases_b(kind, n, h)] == list(range(1, 129))
    c = [x for n in U.C_TEAMS for x in U.cases_c(n)]
    assert {(x["n"], x["L"], x["residual"], x["att"]) for x in c if not x["sizes"]} == \
        {(n, L, r, a) for n in U.C_TEAMS for L in (1, 2, 3, 4) for r in (True, False) for a in ("general", "dot")}
    assert {x["n"] for x in c if x["sizes"]} == set(U.C_NARROW)
    e = U.cases_e
    assert sorted((x["n"], x["D"]) for b in range(len(U.BANDS)) for x in e(b)) == [(n, D) for n in range(1, 257) for D in U.E_DS]
    assert [d["n"] for d in U.D_CASES] == [7, 40, 213] and [(d["n"] + 31) // 32 for d in U.D_CASES] == [1, 2, 7]
    for i in range(len(U.D_CASES)):
        for L in (3, 4):
            (x,) = U.cases_d(i, L)
            assert x["chunk"] < x["T"] and x["T"] % x["chunk"] and x["S"] > 2 * x["chunk"]
            assert all(-(-x["S"] // G) >= 2 and (G == 1 or x["S"] % G) for G in U.block_sizes("comm", x["n"]))


def test_cent_widths_cover_every_residue():
    w = U.cent_widths()
    f = [c for b in range(len(U.BANDS)) for c in U.cases_f(b)]
    assert [c["n"] for c in f] == list(range(1, 257)) and all(c["D"] == w[c["n"]] for c in f)
    K = [n * w[n] for n in range(1, 257)]
    assert max(K) <= U.CENT_K_MAX and all(1 <= w[n] <= 128 for n in w)
    assert {k % 64 for k in K} == set(range(64)) and {k % 32 for k in K} == set(range(32))
    assert {5 * n % 64 for n in range(1, 257)} == set(range(64))
    assert {c["relu"] for c in f} == {True, False}


def test_batches_give_every_kernel_two_blocks_and_a_partial_one():
    import numpy as np
    for kind in ("comm", "dec", "cent"):
        for n in range(1, 257):
            S = U.steps_for(kind, n)
            for G in U.block_sizes(kind, n) + ([256] if kind == "cent" else []):
                assert -(-S // G) >= 2 and (G == 1 or S % G), (kind, n, S, G)
            T = U.path_len_for(S)
            lens = U.valid_lengths(S, T, np.random.RandomState(n))
            assert sum(lens) == S and 1 in lens and T in lens and max(lens) == T


def test_restated_selection():
    assert [U.kt_of(n) for n in (9, 32, 33, 64, 65, 128, 129, 224, 225, 256)] == [1, 1, 2, 2, 4, 4, 7, 7, 8, 8]
    # the 512-thread backward at KT = 7 up to cap 212, the 256-thread one beyond: n = 213 .. 224
    assert [n for n in range(129, 225) if U.nxn_threads(n, 2) == 256] == list(range(213, 225))
    assert all(U.nxn_threads(n, 1) == (512 if n > 64 else 256) for n in range(9, 257))
    assert all(U.nxn_threads(n, 2) == 256 for n in range(225, 257))
    assert U.dense_bwd_name(128, 40, True) == "net_dense_bwd_kernel<128,64,64,1,0>"
    assert U.dense_bwd_name(128, 64, True) == "net_dense_bwd_kernel<128,64,64,1,0>"
    assert U.dense_bwd_name(128, 65, False) == "net_dense_bwd_kernel<128,128,128,0,0>"
    assert U.dense_bwd_name(128, 68, True) == "net_dense_bwd_kernel<128,128,64,1,0>"
    assert U.dense_bwd_name(64, 64, True) == "net_dense_bwd_kernel<64,64,128,1,0>"
    assert U.kernel_name("void cm::net_agg_bwd_kernel<7, 256>(float const*, unsigned int const*)") == "net_agg_bwd_kernel<7,256>"
    assert U.kernel_name("cm::net_critic_head_kernel(cm::CriticHeadArgs)") == "net_critic_head_kernel"
    assert U.kernel_name("void at::native::elementwise_kernel<128, 4>(int)") is None
    # every instantiation the restated launch code can select is listed with its source line, and none is also unreachable
    assert U.all_predicted() == set(U.EXPECTED)
    assert not set(U.EXPECTED) & set(U.UNREACHABLE)
    for k in ("net_agg_bwd_kernel<7,256>", "net_softmax_bwd_kernel<7,256>", "net_dense_bwd_kernel<128,128,64,1,0>",
              "net_small_agg_bwd_kernel"):
        assert k in U.EXPECTED
    assert "net_agg_bwd_kernel<8,512>" in U.UNREACHABLE
    # the coverage cases between them are predicted to launch every expected instantiation
    pred = set()
    for c in U.coverage_cases():
        for call in (("policy",) if c["kind"] == "dec" else ("policy", "critic")):
            pred |= U.predicted_kernels(c["kind"], c["n"], c["D"], call, relu=c["relu"])
    assert pred == set(U.EXPECTED)
