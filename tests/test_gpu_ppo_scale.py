"""The PPO update kernels at production minibatch sizes, against float64 (helpers: tests/ppo_scale_util.py).

At the sizes of test_gpu_ppo_fused.py and test_gpu_ppo_cent_fused.py every persistent CTA of cm_ppo_net walks one tile or env
block.  The cases here (C1, C3, C5, Obs-DP, CENT C1 and C5 shapes, up to 10^6 agent rows) make every CTA walk several, so the
second stage of the dense kernels' bulk-copy ring, its mbarrier parity flip, the dW / db / bias accumulators carried across
tiles and the heads' block reductions are compared with a float64 evaluation of the same function on the same fp32 inputs;
test_ppo_net_cases_walk_several_units_per_cta proves from a profiler trace that they do.  cm_ppo_advantages and cm_adam_step
are held past their grid strides against float64 restatements with condition-aware bounds.  Every comparison fails on NaN."""
import ctypes as C
import json
import os
import time

import numpy as np
import pytest

import ppo_scale_util as U


def _report(rec):
    """one JSON line per case on stdout (pytest -s), appended to $PPO_SCALE_REPORT when that is set"""
    line = json.dumps(rec, sort_keys=True)
    print(line)
    path = os.environ.get("PPO_SCALE_REPORT")
    if path:
        with open(path, "a") as fh:
            fh.write(line + "\n")


def _maxabs(x):
    return float(x.abs().max()) if x.numel() else 0.0


def _grad_errors(g, ref_grads, other=None):
    """per parameter tensor: normalised error of the flat fused gradient `g` (and of `other`'s tensors) against float64"""
    out, o = {}, 0
    for i, (k, r) in enumerate(ref_grads):
        seg = g[o:o + r.numel()].double()
        scale = _maxabs(r)
        e = U.rel(_maxabs(seg - r), scale)
        e_auto = U.rel(_maxabs(other[i][1].double() - r), scale) if other is not None else None
        out[k] = (e, e_auto, scale)
        o += r.numel()
    assert o == g.numel()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("cid", U.CASE_IDS)
def test_ppo_net_matches_float64_at_scale(cid):
    """per-step ll / entropy / probs / values, the policy loss and gradient on a minibatch of valid steps, the critic loss and
    gradient on its padded steps: the kernels against float64, fp32 autograd reported beside them"""
    import torch
    case = next(c for c in U.CASES if c["id"] == cid)
    n, P, T = case["n"], case["P"], U.T_PATH
    torch.cuda.reset_peak_memory_stats()
    t0 = time.time()
    fused, auto, ref, b0 = U.make_case(case, seed=n + case["D"])
    bf = fused.finish_batch(dict(b0))                  # kernel baselines -> cm_ppo_advantages: the inputs both sides see
    F, f = fused._fused, bf["_flat"]
    with torch.no_grad():
        F.pol_map.refresh()
        out = F.policy_call(f, None, want_probs=True)
    old = out["ll"].reshape(P, T) + U.old_ll_offsets(P, T, seed=7)
    ids = np.random.RandomState(n).permutation(P - 1)             # the minibatch: every path but the last, shuffled
    tid = torch.as_tensor(ids, device="cuda")
    idx = F.step_index(f, ids, valid_only=True)
    if case.get("relu"):                                          # steps at a relu kink leave the minibatch on both sides
        kink = U.relu_kink_steps(case, ref.policy, bf)
        bf["mask"] = bf["mask"] & ~kink
        idx = idx[~kink.reshape(-1).index_select(0, idx)]
    S = int(idx.numel())
    res = F.policy_call(f, idx, adv=bf["adv"].reshape(-1).index_select(0, idx), old_ll=old.reshape(-1).index_select(0, idx),
                        backward=True, inv_count=1.0 / S)
    g = torch.empty_like(fused.opt.grad)
    F.pol_map.scatter_grad(g)
    F.cri_map.refresh()
    idx_all = F.step_index(f, ids, valid_only=False)
    resc = F.critic_call(f, idx_all, returns=bf["returns"].reshape(-1).index_select(0, idx_all), backward=True)
    gc = torch.empty_like(fused.baseline_opt.grad)
    F.cri_map.scatter_grad(gc)
    loss, closs = float(res["loss"]), float(resc["loss"])
    F._ws = None
    t_kernels = time.time() - t0

    r64 = U.evaluate(ref, case, bf, tid, old, torch.float64, outputs=True)
    r32 = U.evaluate(auto, case, bf, tid, old, torch.float32, outputs=False)
    # ---- per-step outputs over every padded step of the batch
    errs = {k: [] for k in ("ll", "entropy", "probs", "values")}
    scales = {k: [] for k in errs}
    kern = dict(ll=out["ll"].reshape(P, T), entropy=out["entropy"].reshape(P, T), probs=out["probs"].reshape(P, T, n, 5),
                values=bf["baselines"])
    min_prob, ratio_lo, ratio_hi = float("inf"), False, False
    mb = torch.zeros(P, dtype=torch.bool, device="cuda")
    mb[tid] = True
    for sl, o64 in r64["slices"]:
        for k in errs:
            errs[k].append(_maxabs(kern[k][sl].double() - o64[k]))
            scales[k].append(_maxabs(o64[k]))
        av = o64["avail"].reshape(o64["probs"].shape) > 0
        min_prob = min(min_prob, float(o64["probs"][av].min()))
        ratio = (o64["ll"] - old[sl].double()).exp()[bf["mask"][sl] & mb[sl][:, None]]
        ratio_lo |= bool((ratio < 0.9).any())
        ratio_hi |= bool((ratio > 1.1).any())
    del r64["slices"]
    assert min_prob >= U.MIN_PROB, ("an available action's float64 probability is inside Categorical's clamp", min_prob)
    assert ratio_lo and ratio_hi, "the perturbed old log-likelihood must put ratios on both sides of the clip range"
    out_err = {k: U.rel(float(np.max(errs[k])), float(np.max(scales[k]))) for k in errs}
    tm = U.team(n)
    loss_err = abs(loss - r64["loss"]) / (tm * max(1.0, abs(r64["loss"])))
    loss_err32 = abs(r32["loss"] - r64["loss"]) / (tm * max(1.0, abs(r64["loss"])))
    closs_err = abs(closs - r64["critic_loss"]) / max(1.0, abs(r64["critic_loss"]))
    closs_err32 = abs(r32["critic_loss"] - r64["critic_loss"]) / max(1.0, abs(r64["critic_loss"]))
    pg = _grad_errors(g, r64["grads"], r32["grads"])
    cg = _grad_errors(gc, r64["critic_grads"], r32["critic_grads"])
    peak = torch.cuda.max_memory_allocated()
    rec = dict(case=cid, n=n, D=case["D"], policy_steps=S, policy_rows=S * (1 if case["kind"] == "cent" else n),
               critic_steps=int(idx_all.numel()), out=out_err, out_tol=U.TOL["out"], loss=loss_err, loss_fp32_autograd=loss_err32,
               loss_tol=U.TOL["loss"], critic_loss=closs_err, critic_loss_fp32_autograd=closs_err32, critic_loss_tol=U.TOL["critic_loss"],
               grad_max=max(e for e, _, _ in pg.values()), grad_fp32_autograd_max=max(a for _, a, _ in pg.values()),
               grad_tol=U.TOL["grad"] * tm, critic_grad_max=max(e for e, _, _ in cg.values()),
               critic_grad_fp32_autograd_max=max(a for _, a, _ in cg.values()), critic_grad_tol=U.TOL["critic_grad"],
               grads={k: [e, a] for k, (e, a, _) in pg.items()}, critic_grads={k: [e, a] for k, (e, a, _) in cg.items()},
               min_prob64=min_prob, peak_gb=peak / 2 ** 30, seconds=time.time() - t0, kernel_seconds=t_kernels,
               gpu=torch.cuda.get_device_name())
    _report(rec)
    ctx = f"{cid}: fp32 autograd against the same float64 reference: loss {loss_err32:.3g}, critic loss {closs_err32:.3g}, " \
          f"policy grads {rec['grad_fp32_autograd_max']:.3g}, critic grads {rec['critic_grad_fp32_autograd_max']:.3g}"
    for k, e in out_err.items():
        assert e <= U.TOL["out"], (k, e, ctx)
    assert loss_err <= U.TOL["loss"], (loss, r64["loss"], ctx)
    assert closs_err <= U.TOL["critic_loss"], (closs, r64["critic_loss"], ctx)
    for k, (e, a, scale) in pg.items():
        assert scale > 0, ("policy", k, "no gradient in float64")
        assert e <= U.TOL["grad"] * tm, ("policy", k, e, a, ctx)
    for k, (e, a, scale) in cg.items():
        assert scale > 0, ("critic", k, "no gradient in float64")
        assert e <= U.TOL["critic_grad"], ("critic", k, e, a, ctx)
    assert peak <= U.MEM_LIMIT, peak


@pytest.mark.gpu
def test_ppo_net_cases_walk_several_units_per_cta(tmp_path):
    """every launch of the families a case declares gives each CTA >= 3 dense tiles (stage 1 of the ring and the parity
    flip run) or >= 2 env blocks; across the file every persistent family of cm_ppo_net is covered, the dense kernels in
    both their ASYNC and synchronous instantiations"""
    import torch
    from com_marl_b200 import _native as N
    lib = N.lib()
    covered, rows = set(), []
    for case in U.CASES:
        fused, _, _, b0 = U.make_case(case, seed=case["n"] + case["D"])
        del _
        bf = fused.finish_batch(dict(b0))
        F, f = fused._fused, bf["_flat"]
        P = case["P"]
        ids = np.arange(P - 1)
        idx = F.step_index(f, ids, valid_only=True)
        idx_all = F.step_index(f, ids, valid_only=False)
        F.pol_map.refresh()
        F.cri_map.refresh()
        calls = dict(policy=(F.pol_desc, idx, lambda: F.policy_call(f, idx, adv=bf["adv"].reshape(-1).index_select(0, idx), backward=True,
                                                                    inv_count=1.0 / idx.numel())),
                     critic=(F.cri_desc, idx_all, lambda: F.critic_call(f, idx_all, returns=bf["returns"].reshape(-1).index_select(0, idx_all),
                                                                        backward=True)))
        for call, (desc, ix, run) in calls.items():
            run()                                    # (workspace allocated, modules loaded: the traced call is the steady one)
            torch.cuda.synchronize()
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                run()
                torch.cuda.synchronize()
            trace = tmp_path / f"{case['id']}_{call}.json"
            prof.export_chrome_trace(str(trace))
            w1, w2 = lib.cm_ppo_net_workspace_floats(C.byref(desc), 1, 1), lib.cm_ppo_net_workspace_floats(C.byref(desc), 2, 1)
            per_step, slack = w2 - w1, 2 * w1 - w2
            chunk = (F._ws.numel() - slack) // per_step
            steps_min = min(U.chunk_sizes(int(ix.numel()), chunk))
            rep = U.launch_report(U.kernel_launches(str(trace)), case, call, steps_min)
            assert rep, (case["id"], call, "no cm_ppo_net kernel in the trace")
            for r in rep:
                if r["family"] not in case["covers"].get(call, ()):
                    continue
                rows.append(dict(case=case["id"], call=call, kernel=r["name"].split("(")[0], grid=r["grid"], units=r["units"],
                                 per_cta=r["per_cta"], steps_min_chunk=steps_min))
                assert r["per_cta"] >= U.MIN_UNITS[r["family"]], (case["id"], call, r["name"][:90], r["grid"], r["units"], steps_min)
                covered |= r["tags"]
        del fused, bf, F, f, b0
        torch.cuda.empty_cache()
    least = {}
    for r in rows:
        k = r["kernel"]
        least[k] = min(least.get(k, 1 << 30), r["per_cta"])
    _report(dict(coverage={k: v for k, v in sorted(least.items())}, gpu=torch.cuda.get_device_name()))
    assert U.REQUIRED_TAGS <= covered, sorted(U.REQUIRED_TAGS - covered)


# ---- cm_ppo_advantages past its grid stride ------------------------------------------------------------------------------
def _adv_inputs(P, T, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    valids = torch.randint(1, T + 1, (P,), device="cuda", generator=g).to(torch.int32)
    valids[0], valids[1], valids[-1] = T, 1, 1
    mask = torch.arange(T, device="cuda")[None, :] < valids[:, None]
    rewards = (torch.rand((P, T), device="cuda", generator=g, dtype=torch.float64) * 2 - 0.5) * mask
    baselines = torch.randn((P, T), device="cuda", generator=g) * 3.0
    return rewards, baselines, valids


def _call_advantages(rewards, baselines, valids, discount, lam, center, eps, outs):
    from com_marl_b200 import _native as N
    P, T = rewards.shape
    ptr = lambda x: N.ptr(x) if x is not None else None  # noqa: E731
    return N.lib().cm_ppo_advantages(N.ptr(rewards), N.ptr(baselines), N.ptr(valids), P, T, discount, lam, center, eps,
                                     ptr(outs[0]), ptr(outs[1]), ptr(outs[2]), N.stream_ptr())


def _ulp_ok(x, ref64):
    r32 = ref64.astype(np.float32)
    return np.abs(x.astype(np.float64) - r32.astype(np.float64)) <= np.spacing(np.abs(r32)).astype(np.float64)


@pytest.mark.gpu
@pytest.mark.parametrize("P,T,center,null_ret", [(20000, 200, 1, False), (5000, 8192, 1, False), (20000, 200, 0, False),
                                                 (20000, 200, 1, True)])
def test_advantages_kernel_matches_float64_past_its_grid_stride(P, T, center, null_ret):
    """P > 4 736 paths (1 184 blocks x 4 warps) runs the grid-stride loop; T = 8 192 the > 48 KB shared-memory path as well.
    Outputs start as NaN: a path the loop skips fails."""
    import torch
    from com_marl_b200 import _native as N
    rewards, baselines, valids = _adv_inputs(P, T, seed=P + T)
    discount, lam, eps = 0.99, 0.97, 1e-8
    outs = [torch.full((P, T), float("nan"), device="cuda") for _ in range(3)]
    if null_ret:
        outs[0] = outs[1] = None
    N.check("cm_ppo_advantages", _call_advantages(rewards, baselines, valids, discount, lam, center, eps, outs))
    torch.cuda.synchronize()
    ref = U.advantages64(rewards.cpu().numpy(), baselines.cpu().numpy(), valids.cpu().numpy(), discount, lam, center, eps)
    adv = outs[2].cpu().numpy()
    e_adv = np.abs(adv.astype(np.float64) - ref["adv"])
    assert (e_adv <= ref["adv_bound"]).all(), (float(np.nanmax(e_adv / np.maximum(ref["adv_bound"], 1e-300))), np.isnan(adv).sum())
    print(json.dumps(dict(P=P, T=T, center=center, null_ret=null_ret, adv_rel=float(np.max(e_adv / np.maximum(1.0, np.abs(ref["adv"])))),
                          adv_over_bound=float(np.max(e_adv / ref["adv_bound"])))))
    if null_ret:
        return
    ret, raw = outs[0].cpu().numpy(), outs[1].cpu().numpy()
    assert _ulp_ok(ret, ref["returns"]).all(), np.isnan(ret).sum()
    e_raw = np.abs(raw.astype(np.float64) - ref["raw"])
    assert (e_raw <= ref["raw_bound"]).all(), (float(np.nanmax(e_raw / ref["raw_bound"])), np.isnan(raw).sum())
    if not center:
        assert np.array_equal(adv, raw)


@pytest.mark.gpu
def test_advantages_kernel_rejects_t_beyond_8192():
    import torch
    from com_marl_b200 import _native as N
    P, T = 4, 8193
    rewards = torch.zeros((P, T), dtype=torch.float64, device="cuda")
    baselines = torch.zeros((P, T), device="cuda")
    valids = torch.full((P,), T, dtype=torch.int32, device="cuda")
    outs = [torch.full((P, T), float("nan"), device="cuda") for _ in range(3)]
    assert _call_advantages(rewards, baselines, valids, 0.99, 0.97, 1, 1e-8, outs) == N.CM_EUNSUPPORTED
    torch.cuda.synchronize()
    assert all(bool(o.isnan().all()) for o in outs)


# ---- cm_adam_step past its grid stride -----------------------------------------------------------------------------------
ADAM_N = 4194309              # ~ the CENT K = 32 768 policy bucket; 1 184 x 256 threads walk it ~14 times; not a multiple of 256


@pytest.mark.gpu
@pytest.mark.parametrize("step", [1, 2, 1000])
@pytest.mark.parametrize("dev_scale", [False, True])
def test_adam_step_kernel_matches_float64_past_its_grid_stride(step, dev_scale):
    import torch
    from com_marl_b200 import _native as N
    g = torch.Generator(device="cuda").manual_seed(step)
    n = ADAM_N
    p = torch.randn(n, device="cuda", generator=g)
    grad = torch.randn(n, device="cuda", generator=g) * 0.05
    if step == 1:
        m, v = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    else:
        m = torch.randn(n, device="cuda", generator=g) * 0.02
        v = torch.rand(n, device="cuda", generator=g) * 1e-3
    lr, b1, b2, eps, scale = 3e-4, 0.9, 0.999, 1e-5, 0.37
    state = [x.cpu().numpy() for x in (p, grad, m, v)]
    if dev_scale:
        sd = torch.tensor([scale], dtype=torch.float32, device="cuda")
        N.check("cm_adam_step_dev", N.lib().cm_adam_step_dev(N.ptr(p), N.ptr(grad), N.ptr(m), N.ptr(v), n, lr, b1, b2, eps, step,
                                                             N.ptr(sd), N.stream_ptr()))
    else:
        N.check("cm_adam_step", N.lib().cm_adam_step(N.ptr(p), N.ptr(grad), N.ptr(m), N.ptr(v), n, lr, b1, b2, eps, step, scale,
                                                     N.stream_ptr()))
    torch.cuda.synchronize()
    ref = U.adam64(*state, lr, b1, b2, eps, step, scale)
    for k, x in (("m", m), ("v", v), ("p", p)):
        e = np.abs(x.cpu().numpy().astype(np.float64) - ref[k])
        assert (e <= ref[k + "_bound"]).all(), (k, float(np.nanmax(e / np.maximum(ref[k + "_bound"], 1e-300))))
    moved = np.abs(p.cpu().numpy().astype(np.float64) - state[0].astype(np.float64))
    assert (moved > 0).mean() > 0.99            # (the step moves essentially every element)


# ---- CPU: the restatements and the work-unit arithmetic --------------------------------------------------------------------
def test_advantages64_restates_the_definition():
    rng = np.random.RandomState(0)
    P, T = 5, 9
    valids = np.array([T, 1, 4, 7, 2])
    rewards = rng.rand(P, T) * (np.arange(T)[None, :] < valids[:, None])
    baselines = rng.randn(P, T).astype(np.float32)
    ref = U.advantages64(rewards, baselines, valids, 0.99, 0.97, 1, 1e-8)
    ret, raw = U.naive_advantages64(rewards, baselines, valids, 0.99, 0.97)
    assert np.abs(ref["returns"] - ret).max() <= 1e-12 and np.abs(ref["raw"] - raw).max() <= 1e-12
    for p in range(P):                               # centring over the valid steps, applied to the whole row
        v = valids[p]
        mu, var = raw[p, :v].mean(), raw[p, :v].var()
        assert np.abs(ref["adv"][p] - (raw[p] - mu) / np.sqrt(var + float(np.float32(1e-8)))).max() <= 1e-9 * max(1.0, np.abs(ref["adv"][p]).max())
    # the bounds are positive and small: a few fp32 roundings of the magnitudes involved
    assert (ref["raw_bound"] > 0).all() and (ref["raw_bound"] <= 1e-4 * np.maximum(1.0, np.abs(ref["raw"]))).all()
    assert (ref["adv_bound"] > 0).all() and (ref["adv_bound"][valids >= 4] <= 1e-3 * np.maximum(1.0, np.abs(ref["adv"][valids >= 4]))).all()
    # the bound covers an fp32 evaluation of the same recurrence
    c = np.float32(np.float32(0.99) * np.float32(0.97))
    a = np.zeros(P, np.float32)
    r32, b32 = rewards.astype(np.float32), baselines
    for t in range(T - 1, -1, -1):
        bn = b32[:, t + 1] if t + 1 < T else np.zeros(P, np.float32)
        a = c * a + (r32[:, t] + np.float32(0.99) * bn - b32[:, t])
        assert (np.abs(a.astype(np.float64) - ref["raw"][:, t]) <= ref["raw_bound"][:, t]).all()
    unc = U.advantages64(rewards, baselines, valids, 0.99, 0.97, 0, 1e-8)
    assert np.array_equal(unc["adv"], unc["raw"])


def test_adam64_restates_torch_adam_step():
    import types

    import torch
    from ppo_dp_util import torch_adam_step
    rng = np.random.RandomState(1)
    n = 1000
    p, g, m = (rng.randn(n).astype(np.float32) for _ in range(3))
    v = rng.rand(n).astype(np.float32)
    f32 = lambda x: float(np.float32(x))  # noqa: E731
    for step in (1, 2, 1000):
        st = types.SimpleNamespace(flat=torch.tensor(p, dtype=torch.float64), grad=torch.tensor(g, dtype=torch.float64),
                                   exp_avg=torch.tensor(m, dtype=torch.float64), exp_avg_sq=torch.tensor(v, dtype=torch.float64),
                                   steps=step - 1, betas=(f32(0.9), f32(0.999)), lr=f32(3e-4), eps=f32(1e-5))
        torch_adam_step(st, grad_scale=f32(0.37))
        ref = U.adam64(p, g, m, v, 3e-4, 0.9, 0.999, 1e-5, step, 0.37)
        assert np.abs(st.flat.numpy() - ref["p"]).max() <= 1e-15
        assert np.abs(st.exp_avg.numpy() - ref["m"]).max() <= 1e-15 and np.abs(st.exp_avg_sq.numpy() - ref["v"]).max() <= 1e-15
        for k in ("p", "m", "v"):
            assert (ref[k + "_bound"] >= 0).all() and ref[k + "_bound"].max() <= 1e-5 * np.abs(ref[k]).max()


def test_work_unit_arithmetic(tmp_path):
    assert [U.env_geom_G(n) for n in (9, 32, 33, 64, 65, 200)] == [7, 2, 3, 2, 1, 1]
    assert [U.small_G(n) for n in (1, 4, 8)] == [128, 32, 16] and [U.env_group(n) for n in (1, 4, 32, 200, 256)] == [256, 64, 8, 1, 1]
    f = U.classify("void cm::net_dense_fwd_kernel<128, 1, 0>(float const*, int, float const*, float const*, float*, int, long, int)")
    assert f == ("dense", {"dense_fwd/sync"}, 128)
    assert U.classify("void cm::net_dense_bwd_kernel<64, 128, 64, 1, 1>(float const*)") == ("dense", {"dense_bwd/async", "dense_bwd/relu"}, 64)
    assert U.classify("void cm::net_dense_fwd_kernel<64, 2, 1>(float const*)")[1] == {"dense_fwd/async", "dense_fwd/relu"}
    assert U.classify("void cm::net_small_agg_bwd_kernel(float const*)")[:2] == ("small", {"small_agg_bwd"})
    assert U.classify("void cm::net_agg_bwd_kernel<7, 512>(float const*)")[:2] == ("nxn", {"agg_bwd"})
    assert U.classify("cm::net_critic_head_kernel(cm::CriticHeadArgs)")[:2] == ("head", {"critic_head"})
    assert U.classify("void cm::net_wide_dw_kernel<128, 0>(float const*)") is None and U.classify("elementwise_kernel") is None
    c1 = U.CASES[0]
    assert U.work_units("dense", 128, 4, 131072, "comm", "policy") == 4096
    assert U.work_units("head", None, 4, 131072, "cent", "critic") == 512 and U.work_units("head", None, 4, 131072, "cent", "policy") == 2048
    assert U.work_units("small", None, 4, 100, "comm", "policy") == 4 and U.work_units("nxn", None, 200, 2133, "comm", "policy") == 2133
    assert U.chunk_sizes(300000, 131072) == [131072, 131072, 37856] and U.chunk_sizes(5, 131072) == [5]
    trace = tmp_path / "t.json"
    trace.write_text(json.dumps(dict(traceEvents=[
        dict(cat="kernel", name="void cm::net_dense_bwd_kernel<128, 64, 128, 0, 0>(float const*)", args=dict(grid=[148, 1, 1])),
        dict(cat="kernel", name="void cm::net_small_scores_kernel(float const*)", args=dict(grid=[888, 1, 1])),
        dict(cat="cuda_runtime", name="cudaLaunchKernel", args=dict()),
        dict(cat="kernel", name="void at::elementwise_kernel<128, 4>()", args=dict(grid=[10, 1, 1]))])))
    rep = U.launch_report(U.kernel_launches(str(trace)), c1, "policy", 115000)
    assert [(r["family"], r["units"], r["per_cta"]) for r in rep] == [("dense", 3594, 24), ("small", 3594, 4)]
    # every required family is declared by some case
    fams = {f for c in U.CASES for v in c["covers"].values() for f in v}
    assert fams == set(U.MIN_UNITS)
