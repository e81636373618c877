"""Helpers of tests/test_gpu_ppo_scale.py: the PPO update kernels at production minibatch sizes against float64.

At the sizes of the other PPO tests every persistent CTA of cm_ppo_net (csrc/ppo_net_kernels.cu) walks one work unit, so the
second stage of the dense kernels' bulk-copy ring, its mbarrier parity flip and every accumulator carried across tiles or env
blocks never run.  The cases below are sized so that they do, and ``launch_report`` proves it from a torch.profiler trace.

What is here:
- the case table and the tolerance table (fixed; one reason each);
- the launch code's work-unit counts, restated (``work_units``) and a reader of the trace's kernel launches;
- float64 restatements of cm_ppo_advantages and cm_adam_step (csrc/ppo_kernels.cu) with error bounds from their condition;
- the batch builder and the float64 reference of the PPO losses (the same torch functions on float64 copies of the modules,
  evaluated over slices of paths so that memory stays bounded).

Nothing here touches CUDA at import time.
"""
import copy
import json
import math
import re

import numpy as np

T_PATH = 200                                   # steps per padded path, the runners' max_path_length
U32 = float(np.finfo(np.float32).eps) / 2      # unit roundoff of fp32
MEM_LIMIT = 40 << 30                           # peak device memory one case may allocate (the GPUs are shared)

# ---- cases --------------------------------------------------------------------------------------------------------------
# P = paths in the batch; the minibatch is every path but the last.  The minibatch's valid lengths are 1..T spread evenly over
# its P - 1 paths in a random order (``planned_steps``: 100.5 (P - 1) valid steps for the policy call, exactly), so that the
# chunking below does not depend on the seed; 200 (P - 1) padded steps go to the critic call.
# covers: per call, the kernel families whose every launch must give each CTA several work units (see MIN_UNITS).
CASES = [
    # Comm-DP at C1's team: 985 k agent rows in the policy call, so the default chunk_rows (524 288) walks two chunks, the
    # second 115 k steps; the critic's 490 k padded steps walk four, the last 97 k
    dict(id="c1", kind="comm", n=4, D=21, L=2, P=2451, covers=dict(policy=("dense", "small", "head"), critic=("dense", "small", "head"))),
    # C3's shape: G = 2 envs per CTA in the n x n kernels, 256 k agent rows in one chunk (the critic's 16 000 padded steps
    # stay inside one chunk of 16 384)
    dict(id="c3", kind="comm", n=32, D=53, L=2, P=81, covers=dict(policy=("dense", "nxn"), critic=("dense", "nxn", "head"))),
    # C5: one env per CTA, KT = 7, 427 k dense rows; the critic walks two chunks (2 516 + 1 684 steps)
    dict(id="c5", kind="comm", n=200, D=53, L=2, P=22, covers=dict(policy=("dense", "nxn", "head"), critic=("dense", "nxn", "head"))),
    # Obs-DP (CM_NET_POLICY_DEC): dense layers and the policy head; 10 k valid steps give the head two env blocks per CTA
    dict(id="obsdp", kind="dec", n=32, D=53, L=2, P=101, covers=dict(policy=("dense", "head"))),
    # CENT at C1's team, relu: the XRELU dense layers 2-3 over 124 k rows in one chunk (chunk_rows / n = 131 072 steps)
    dict(id="cent_c1", kind="cent", n=4, D=21, L=0, P=1241, relu=True, covers=dict(policy=("dense", "head"))),
    # CENT at C5, tanh: the K = 10 600 wide layers at their production shape; their dense layers see only ~17 tiles
    dict(id="cent_c5", kind="cent", n=200, D=53, L=0, P=22, covers=dict(policy=("head",))),
]
CASE_IDS = [c["id"] for c in CASES]

# ---- tolerances ---------------------------------------------------------------------------------------------------------
# Normalised errors max|x - x64| / max|x64| against the float64 evaluation of the same function on the same fp32 inputs.  They
# are the bounds the small-batch tests (test_gpu_ppo_fused.py, test_gpu_ppo_cent_fused.py) hold against fp32 autograd; a
# production-size batch must not need more.  `team` = max(1, n / 32) where a quantity goes through the joint log-likelihood.
TOL = {
    "out": 2e-5,            # per-step ll / entropy / probs / values: fp32 products of K <= 128 terms, no cross-row sums
    "loss": 2e-5,           # x team x max(1, |loss|): a mean over up to 250 k steps, summed per CTA, one atomic add per CTA
    "grad": 2e-4,           # x team, per parameter tensor: fp32 sums over up to 10^6 rows (register chains, then atomics)
    "critic_loss": 2e-5,    # x max(1, |loss|): as "loss" (no joint log-likelihood)
    "critic_grad": 2e-4,    # per parameter tensor, as "grad"
}
MIN_PROB = 1e-6             # smallest float64 probability of an available action: below ~1.2e-7 Categorical's clamp differs


def team(n):
    return max(1.0, n / 32.0)


def rel(err, scale):
    """normalised error; NaN stays NaN so that every `rel(...) <= tol` fails on it"""
    return float(err) / max(1e-30, float(scale)) if not (math.isnan(err) or math.isnan(scale)) else float("nan")


# ---- the launch code's work units, restated (csrc/ppo_net_kernels.cu) -------------------------------------------------------
# dense_fwd_a / dense_bwd_a (:1604-1649): tiles = ceil(R / ROWS), ROWS = 128 (forward) or the ROWS template argument of the
# backward (128, or 64 where two stages of 128-row tiles do not fit, :1655-1658); grid = min(tiles, SMs x occupancy).
# env_geom (:1716-1723): the n x n kernels own G = max(1, target / n) envs per block, target 64 up to n = 32, else 128;
# small_grid (:1824-1829): n <= kSmallN = 8 uses G = kSmallRows / n = 128 / n; env_group (:1705-1711): the heads own
# G = 1 (n >= 256) or 256 / n envs per block; the CENT baseline's head runs with n = 1 (:1986).  Units are ceil(S / G).
MIN_UNITS = {"dense": 3, "nxn": 2, "small": 2, "head": 2}     # a dense CTA needs 3 tiles for stage 1 and the parity flip


def env_geom_G(n):
    target = 64 if n <= 32 else 128
    return 1 if n >= target else target // n


def small_G(n):
    return 128 // n


def env_group(n):
    return 1 if n >= 256 else 256 // n


_DENSE_FWD = re.compile(r"net_dense_fwd_kernel<\s*(\d+),\s*(\d+),\s*(\d+)\s*>")
_DENSE_BWD = re.compile(r"net_dense_bwd_kernel<\s*(\d+),\s*(\d+),\s*(\d+),\s*(\d+),\s*(\d+)\s*>")


def classify(name):
    """kernel name -> (family, tags, ROWS or None); None for a kernel that is not one of cm_ppo_net's persistent ones"""
    m = _DENSE_FWD.search(name)
    if m:
        _, act, asy = (int(x) for x in m.groups())
        return "dense", {"dense_fwd/" + ("async" if asy else "sync")} | ({"dense_fwd/relu"} if act == 2 else set()), 128
    m = _DENSE_BWD.search(name)
    if m:
        _, _, rows, asy, xrelu = (int(x) for x in m.groups())
        return "dense", {"dense_bwd/" + ("async" if asy else "sync")} | ({"dense_bwd/relu"} if xrelu else set()), rows
    for k in ("small_scores", "small_agg_fwd", "small_agg_bwd", "small_softmax_bwd"):
        if f"net_{k}_kernel" in name:
            return "small", {k}, None
    for k in ("scores", "agg_fwd", "agg_bwd", "softmax_bwd"):
        if f"net_{k}_kernel" in name:
            return "nxn", {k}, None
    for k in ("policy_head", "critic_head", "cent_head"):
        if f"net_{k}_kernel" in name:
            return "head", {k}, None
    return None


def work_units(family, rows_per_tile, n, steps, kind, call):
    """work units of one launch over a chunk of `steps` env steps (CENT: rows = steps; the others: rows = steps x n)"""
    cent = kind == "cent"
    if family == "dense":
        R = steps if cent else steps * n
        return -(-R // rows_per_tile)
    if family == "small":
        return -(-steps // small_G(n))
    if family == "nxn":
        return -(-steps // env_geom_G(n))
    if family == "head":
        return -(-steps // env_group(1 if (cent and call == "critic") else n))
    raise ValueError(family)


def chunk_sizes(steps, chunk):
    """cm_ppo_net walks a call's steps in chunks of `chunk` (:2153-2156)"""
    return [min(chunk, steps - s0) for s0 in range(0, steps, chunk)]


def kernel_launches(trace_path):
    """[(name, gridDim.x)] of the kernel events of a torch.profiler chrome trace"""
    with open(trace_path) as fh:
        ev = json.load(fh)["traceEvents"]
    return [(e["name"], int(e["args"]["grid"][0])) for e in ev if e.get("cat") == "kernel" and "grid" in e.get("args", {})]


def launch_report(launches, case, call, steps_min):
    """per launch of a persistent family: work units per CTA, from the smallest chunk of the call (a lower bound for every
    chunk: the grid is capped at the same SMs x occupancy).  -> list of dict(name, family, tags, grid, units, per_cta)"""
    out = []
    for name, grid in launches:
        c = classify(name)
        if c is None:
            continue
        fam, tags, rows = c
        units = work_units(fam, rows, case["n"], steps_min, case["kind"], call)
        out.append(dict(name=name, family=fam, tags=tags, grid=grid, units=units, per_cta=units // max(1, grid)))
    return out


REQUIRED_TAGS = {"dense_fwd/async", "dense_fwd/sync", "dense_bwd/async", "dense_bwd/sync", "dense_fwd/relu", "dense_bwd/relu",
                 "scores", "agg_fwd", "agg_bwd", "softmax_bwd", "small_scores", "small_agg_fwd", "small_agg_bwd",
                 "small_softmax_bwd", "policy_head", "critic_head", "cent_head"}


# ---- cm_ppo_advantages in float64 (csrc/ppo_kernels.cu:13-22) ---------------------------------------------------------------
def advantages64(rewards, baselines, valids, discount, gae_lambda, center, eps):
    """float64 restatement of the kernel's specification on its fp32 inputs.  rewards float64 [P, T] (the kernel reads them as
    fp32 for delta, as float64 for the returns), baselines fp32 [P, T], valids [P]; discount, gae_lambda, eps as the fp32
    values the kernel receives.  Returns dict of float64 arrays: returns, raw, adv and the error bounds raw_bound, adv_bound.

    raw_bound: fp32 forms delta = r + g b' - b with error <= 2u (|r| + g|b'| + |b|), and each step of the recurrence
    a = fma(c, a, delta) rounds once (<= u|a|); both propagate with weight c^k, so the bound is the same recurrence run on
    m_t = 2(|r_t| + g|b_t+1| + |b_t|) + |a_t| (it follows the cancellation in delta, not |delta|), times 2 for the first-order terms.
    adv_bound: first-order propagation of raw_bound through the mean, the biased variance (fp32 sums of v terms: at most
    (ceil(v / 32) + 5) u relative for positive terms) and 1 / sqrt(var + eps), times 2."""
    P, T = rewards.shape
    g = float(np.float32(discount))
    c = float(np.float32(np.float32(discount) * np.float32(gae_lambda)))
    e32 = float(np.float32(eps))
    r32 = rewards.astype(np.float32).astype(np.float64)
    b = baselines.astype(np.float64)
    bn = np.concatenate([b[:, 1:], np.zeros((P, 1))], 1)
    delta = r32 + g * bn - b
    raw = np.empty((P, T))
    a = np.zeros(P)
    for t in range(T - 1, -1, -1):
        a = c * a + delta[:, t]
        raw[:, t] = a
    m = 2.0 * (np.abs(r32) + g * np.abs(bn) + np.abs(b)) + np.abs(raw)
    raw_bound = np.empty((P, T))
    a = np.zeros(P)
    for t in range(T - 1, -1, -1):
        a = c * a + m[:, t]
        raw_bound[:, t] = 2.0 * U32 * a
    v = np.clip(np.asarray(valids, dtype=np.int64), 0, T)
    tt = np.arange(T)[None, :]
    valid = tt < v[:, None]
    ret = np.zeros((P, T))
    y = np.zeros(P)
    for t in range(T - 1, -1, -1):
        y = np.where(t < v, rewards[:, t] + g * y, 0.0)
        ret[:, t] = y
    out = dict(returns=ret, raw=raw, raw_bound=raw_bound)
    if center:
        cnt = np.maximum(v, 1).astype(np.float64)
        mean = np.where(valid, raw, 0.0).sum(1) / cnt
        d = np.where(valid, raw - mean[:, None], 0.0)
        var = (d * d).sum(1) / cnt
        s = 1.0 / np.sqrt(var + e32)
        E = np.where(valid, raw_bound, 0.0).max(1)
        chain = (np.ceil(cnt / 32.0) + 5.0) * U32
        dmu = E + chain * np.where(valid, np.abs(raw), 0.0).sum(1) / cnt
        dvar = 2.0 * np.sqrt(var) * (E + dmu) + (E + dmu) ** 2 + chain * var
        ds = 0.5 * dvar / (var + e32) + 3.0 * U32
        adv = (raw - mean[:, None]) * s[:, None]
        out["adv"] = adv
        out["adv_bound"] = 2.0 * (s[:, None] * (raw_bound + dmu[:, None]) + np.abs(adv) * (ds[:, None] + 2.0 * U32))
    else:
        out["adv"], out["adv_bound"] = raw, raw_bound
    return out


def naive_advantages64(rewards, baselines, valids, discount, gae_lambda):
    """the definition as written (O(P T^2)), float64 throughout: returns and raw advantages, for the CPU check of advantages64"""
    P, T = rewards.shape
    g = float(np.float32(discount))
    c = float(np.float32(np.float32(discount) * np.float32(gae_lambda)))
    r = rewards.astype(np.float32).astype(np.float64)
    b = baselines.astype(np.float64)
    ret, raw = np.zeros((P, T)), np.zeros((P, T))
    for p in range(P):
        for t in range(T):
            raw[p, t] = sum(c ** k * (r[p, t + k] + g * (b[p, t + k + 1] if t + k + 1 < T else 0.0) - b[p, t + k]) for k in range(T - t))
            if t < valids[p]:
                ret[p, t] = sum(g ** k * rewards[p, t + k] for k in range(valids[p] - t))
    return ret, raw


# ---- cm_adam_step in float64 (csrc/ppo_kernels.cu:72-88; the formula of tests/ppo_dp_util.torch_adam_step) --------------------
def adam64(p, g, m, v, lr, beta1, beta2, eps, step, grad_scale):
    """one step from the fp32 state (numpy float32 arrays), in float64 with the fp32 constants the kernel receives.  Returns
    dict of float64 p, m, v and the bounds of the fp32 kernel's error: m and v round a few times relative to the magnitudes they
    are formed from; p's update carries those through m / denom, plus the rounding of step_size and 1 / sqrt(bc2)."""
    f = lambda x: float(np.float32(x))  # noqa: E731
    b1, b2, e, lr, gs = f(beta1), f(beta2), f(eps), f(lr), f(grad_scale)
    bc1, bc2 = 1.0 - b1 ** step, 1.0 - b2 ** step
    step_size, ibc2 = lr / bc1, 1.0 / math.sqrt(bc2)
    p, g, m, v = (x.astype(np.float64) for x in (p, g, m, v))
    gi = g * gs
    m1 = b1 * m + (1.0 - b1) * gi
    v1 = b2 * v + (1.0 - b2) * gi * gi
    den = np.sqrt(v1) * ibc2 + e
    p1 = p - step_size * (m1 / den)
    m_bound = 4.0 * U32 * (b1 * np.abs(m) + (1.0 - b1) * np.abs(gi))
    v_bound = 6.0 * U32 * v1
    upd = step_size * np.abs(m1) / den
    p_bound = 2.0 * (U32 * np.abs(p1) + step_size * m_bound / den + upd * (8.0 * U32 + 0.5 * v_bound / np.maximum(v1, 1e-300)))
    return dict(p=p1, m=m1, v=v1, p_bound=p_bound, m_bound=m_bound, v_bound=v_bound)


# ---- batches and the float64 reference (GPU) --------------------------------------------------------------------------------
CLIP = 0.1                  # DevicePPO.lr_clip_range
CLIP_GAP = 5e-3             # |log ratio - log(1 +- CLIP)| kept at least this far from the clip edges


def old_ll_offsets(P, T, seed):
    """old - new log-likelihood, 0.15 N(0, 1) per step: ratios exp(-offset) on both sides of the clip range, but none within
    CLIP_GAP of its edges.  The clipped objective's gradient jumps there, and the fp32 and float64 log-likelihoods (apart by up
    to ~1e-6 |ll|, 3e-4 at n = 200) would put a step on different sides: two different functions, not two precisions."""
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    d = 0.15 * torch.randn((P, T), device="cuda", generator=g, dtype=torch.float64)
    for edge in (-math.log(1.0 - CLIP), -math.log(1.0 + CLIP)):
        near = (d - edge).abs() < CLIP_GAP
        d = torch.where(near, edge + torch.where(d >= edge, CLIP_GAP, -CLIP_GAP), d)
    return d.float()


KINK_GAP = 1e-4            # |relu pre-activation| below which a step leaves the relu case's policy minibatch


def relu_kink_steps(case, pol64, b):
    """[P, T] bool: steps at which a float64 pre-activation of the relu policy's hidden layers lies within KINK_GAP of 0.  relu'
    jumps there, and the fp32 pre-activations (off by ~1e-5) would take the other side on some of 10^5 rows: two different
    functions, not two precisions.  Those steps (about 1 %) are left out of the minibatch on both sides."""
    import torch
    out = []
    with torch.no_grad():
        for sl in path_slices(case, torch.arange(b["valids"].shape[0], device="cuda")):
            x = b["obs"][sl].double()
            m = torch.full(x.shape[:-1], float("inf"), dtype=torch.float64, device=x.device)
            for layer in pol64._layers:
                z = layer(x)
                m = torch.minimum(m, z.abs().amin(-1))
                x = torch.relu(z)
            out.append(m < KINK_GAP)
    return torch.cat(out)


def planned_steps(P, T=T_PATH):
    """valid lengths of the minibatch's P - 1 paths: 1..T spread evenly (the order is drawn in make_case)"""
    m = P - 1
    return [1 + k * (T - 1) // max(1, m - 1) for k in range(m)]


def make_case(case, seed=0):
    """-> (fused DevicePPO, fp32 autograd DevicePPO, float64 DevicePPO, padded batch b0).  Random ragged paths of T = 200 steps
    (valid lengths 1..T, including 1 and T), random adjacency and channel rows with one row without any neighbour, random
    availability, biases and log-stds moved off their initial values — the construction of test_gpu_ppo_fused.py::_make."""
    import torch
    from com_marl_b200.policy import CentralizedCategoricalMLPPolicy, CommCategoricalMLPPolicy, DecCategoricalMLPPolicy
    from com_marl_b200.ppo import CommBaseCritic, DevicePPO, GaussianMLPBaseline
    from com_marl_b200.spaces import Box, Discrete, EnvSpec
    n, D, L, P, T, kind = case["n"], case["D"], case["L"], case["P"], T_PATH, case["kind"]
    torch.manual_seed(seed)
    spec = EnvSpec(Box(np.zeros(n * D), np.ones(n * D)), Discrete(5))
    if kind == "cent":
        mk = lambda: (CentralizedCategoricalMLPPolicy(spec, n, hidden_nonlinearity="relu" if case.get("relu") else "tanh"),  # noqa: E731
                      GaussianMLPBaseline(spec, hidden_sizes=(64, 64, 64)))
    elif kind == "dec":
        mk = lambda: (DecCategoricalMLPPolicy(spec, n), CommBaseCritic(spec, n, n_gcn_layers=L))  # noqa: E731
    else:
        mk = lambda: (CommCategoricalMLPPolicy(spec, n, n_gcn_layers=L), CommBaseCritic(spec, n, n_gcn_layers=L))  # noqa: E731
    pol_a, cri_a = mk()
    with torch.no_grad():
        for m in (pol_a, cri_a):
            for k, p in m.named_parameters():
                if k.endswith("bias") or k.endswith("_init_std"):
                    p.add_(0.1 * torch.randn_like(p))
    pol_64, cri_64 = copy.deepcopy(pol_a).double(), copy.deepcopy(cri_a).double()
    pol_f, cri_f = mk()
    pol_f.load_state_dict(pol_a.state_dict())
    cri_f.load_state_dict(cri_a.state_dict())
    auto = DevicePPO(pol_a, cri_a, fused=False)
    fused = DevicePPO(pol_f, cri_f, fused=True)
    ref = copy.copy(auto)                          # the same loss code (compute_loss / _dist read self.policy only)
    ref.policy, ref.baseline = pol_64, cri_64
    for m in (pol_64, cri_64):
        for p in m.parameters():
            p.grad = None
    g = torch.Generator(device="cuda").manual_seed(seed)
    rnd = lambda *s: torch.rand(*s, device="cuda", generator=g)  # noqa: E731
    lengths = torch.tensor(planned_steps(P, T), dtype=torch.int32, device="cuda")
    valids = torch.randint(1, T + 1, (P,), device="cuda", generator=g).to(torch.int32)     # (the last path: outside the minibatch)
    valids[:P - 1] = lengths[torch.randperm(P - 1, device="cuda", generator=g)]
    avail = (rnd(P, T, n, 5) < 0.8).float()
    avail[..., 4] = 1.0
    actions = torch.multinomial(avail.reshape(-1, 5), 1).reshape(P, T, n)
    b = dict(obs=rnd(P, T, n * D), avail=avail.reshape(P, T, n * 5), actions=actions, rewards=rnd(P, T).double(), valids=valids)
    if kind != "cent":
        adj = (rnd(P, T, n, n) < 0.6).float()
        adj = torch.maximum(adj, torch.eye(n, device="cuda"))
        adj[0, 0, 0, :] = 0.0                      # a row with no neighbour at all (the + 1e-12 of the renormalisation)
        chan = (rnd(P, T, L, n, n) < 0.7).float()
        chan[:, :, :, torch.arange(n), torch.arange(n)] = 1.0
        b["dist_adjs"], b["channels"] = adj.reshape(P, T, n * n), chan.reshape(P, T, L * n, n)
    t = torch.arange(T, device="cuda")[None, :] < valids[:, None]
    b["obs"] = b["obs"] * t.reshape(P, T, 1).float()
    b["rewards"] = b["rewards"] * t.double()
    return fused, auto, ref, b


def path_slices(case, ids):
    """consecutive pieces of the path list whose float64 autograd graph stays within a few GB"""
    n, L = case["n"], max(case["L"], 1)
    per_step = 8 * (2500 * n + 16 * L * n * n) if case["kind"] != "cent" else 8 * (4 * n * case["D"] + 4000 + 40 * n)
    k = max(1, int((3 << 30) // (T_PATH * per_step)))
    return [ids[i:i + k] for i in range(0, len(ids), k)]


def _sub(b, ids, dtype):
    import torch
    out = {}
    for k, v in b.items():
        if not isinstance(v, torch.Tensor) or v.dim() == 0 or v.shape[0] != b["valids"].shape[0]:
            continue
        x = v[ids]
        out[k] = x.to(dtype) if (x.is_floating_point() and k != "rewards") else x
    return out


def evaluate(ppo, case, b, ids, old, dtype, outputs=True):
    """The PPO objective of DevicePPO.compute_loss and the critic's Gaussian NLL, evaluated in `dtype` over slices of paths.
    The policy loss is a mean over the minibatch's valid steps, so each slice's loss is weighted by its share of them; the
    critic's is a mean over the padded steps.  Gradients add up in the modules' .grad.  With outputs=True also the per-step
    ll, entropy, probs and values over every path of the batch (as lists of per-slice tensors)."""
    import torch
    pol, cri = ppo.policy, ppo.baseline
    for m in (pol, cri):
        for p in m.parameters():
            p.grad = None
    nvalid = float(b["mask"][ids].sum())
    loss_p = loss_c = 0.0
    for sl in path_slices(case, ids):
        s = _sub(b, sl, dtype)
        w = float(s["mask"].sum()) / nvalid
        lp = ppo.compute_loss(s, None, old[sl].to(dtype)) * w
        lp.backward()
        loss_p += float(lp.detach())
        lc = (cri.compute_loss(s["obs"], s["returns"], s["dist_adjs"], s["channels"]) if case["kind"] != "cent"
              else cri.compute_loss(s["obs"], s["returns"])) * (len(sl) / len(ids))
        lc.backward()
        loss_c += float(lc.detach())
        del s, lp, lc
    res = dict(loss=loss_p, critic_loss=loss_c,
               grads=[(k, p.grad.detach().reshape(-1) if p.grad is not None else torch.zeros(p.numel(), dtype=dtype, device=p.device))
                      for k, p in pol.named_parameters() if p.requires_grad],
               critic_grads=[(k, p.grad.detach().reshape(-1) if p.grad is not None else torch.zeros(p.numel(), dtype=dtype, device=p.device))
                             for k, p in cri.named_parameters() if p.requires_grad])
    if outputs:
        res["slices"] = []
        all_ids = torch.arange(b["valids"].shape[0], device="cuda")
        with torch.no_grad():
            for sl in path_slices(case, all_ids):
                s = _sub(b, sl, dtype)
                d = ppo._dist(s, None)
                vals = (cri.forward(s["obs"], s["avail"], s["dist_adjs"], s["channels"]) if case["kind"] != "cent"
                        else cri.forward(s["obs"]))
                res["slices"].append((sl, dict(ll=d.log_prob(s["actions"]).sum(-1), entropy=d.entropy().mean(-1), probs=d.probs,
                                               values=vals, avail=s["avail"])))
                del s, d
    return res
