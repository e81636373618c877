"""Helpers of tests/test_gpu_policy_kinds.py: the CENT and Obs-DP forwards of cm_policy_forward against float64.

CENT (policy_cent_kernel.cu) runs the first layer (K = n*D) either in exact fp32 inside policy_cent_kernel (math 'fp32', env
tiles of 64) or on the tensor cores in policy_cent_l1_tc_kernel (math 'tc': env tiles of 128, K walked in panels of 32 through
a 6-deep fp32 ring, 2 operand stages filled by two producer teams on alternate panels and a 6-deep weight ring; 16-byte copies
when K % 4 == 0 and the observation block is 16-byte aligned, 4-byte copies otherwise).  Obs-DP runs policy_tc_kernel in rows
mode: any 128 agent rows form a tile, a persistent grid of 2 CTAs per SM walks the tiles.

What is here:
- the case tables (every K of the first-layer walk, production shapes) and batch / sample builders;
- input generators with the env's value set (0/1 window bits, up to 3 scalar columns, all-zero rows);
- a numpy Philox4x32-10 and the action-stream draw of common.cuh::categorical_finish, restated;
- one forward call on device tensors, the oracle on (sampled) envs and the comparison with a per-(kind, math) error record.

Nothing here touches CUDA at import time.
"""
import numpy as np

from policy_path_util import inverse_cdf

L1_ROWS, L1_KP = 128, 32               # policy_cent_l1_tc_kernel: envs per tile, K per panel
CENT_ROWS = 64                         # policy_cent_kernel: envs per tile
TC_ROWS = 128                          # policy_tc_kernel: agent rows per tile
TOL = 1e-5
MAX_N, MAX_D = 256, 128
REPORT = {}                            # (kind, math) -> largest error / tolerance seen


def cent_tc_tol(K):
    """CENT math 'tc' bar: TOL up to K = 16 384, then growing with K.  At K = 32 768 (n = 256, D = 128) with uniform [0, 1)
    inputs and relu the tensor-core first layer's logits measured 1.47e-5 relative on a B200: the tensor cores accumulate
    2 048 products of K = 16 in fp32 per output, so the accumulation error grows with K.  math 'fp32' keeps TOL at every K."""
    return TOL * max(1.0, K / 16384)


# ---- shapes -----------------------------------------------------------------------------------------------------------
def cent_factor(K):
    """(n, D) with n * D = K, n <= 256, D <= 128 and the largest such D; None where there is none (primes above 256 ...)"""
    for D in range(min(K, MAX_D), 0, -1):
        if K % D == 0 and K // D <= MAX_N:
            return K // D, D
    return None


def panels(K):
    return (K + L1_KP - 1) // L1_KP


def walk_cases():
    """every K = n*D from 1 to 320 that the limits allow, then the production-sized ones: [(n, D)]"""
    out = [cent_factor(K) for K in range(1, 321) if cent_factor(K)]
    out += [cent_factor(K) for K in (511, 512, 1696, 4158, 10600, 13568)]
    out += [(256, 101), (256, 128)]                    # K = 25 856 and 32 768, the largest team at two widths
    return out


def rows_batch(n, sms, tiles_per_cta=3):
    """Obs-DP batch whose agent rows give every CTA of the persistent grid (2 per SM) at least `tiles_per_cta` tiles of 128
    rows, the last tile ragged wherever n allows it"""
    grid = 2 * sms
    B = tiles_per_cta * grid * TC_ROWS // n + 1
    if (B * n) % TC_ROWS == 0 and n % TC_ROWS:
        B += 1
    return B


def sample_envs(B, tile_envs, stride=2048, extra=()):
    """sorted env indices: the whole first and last tile (tiles of `tile_envs` envs), about `stride` envs spread evenly over
    the batch, and `extra`"""
    last0 = (B - 1) // tile_envs * tile_envs
    s = set(range(min(tile_envs, B))) | set(range(last0, B)) | set(np.linspace(0, B - 1, min(B, stride)).astype(np.int64).tolist())
    s |= {int(e) for e in extra if 0 <= e < B}
    return np.array(sorted(s), np.int64)


def dec_sample_envs(B, n, sms, stride=2048):
    """Obs-DP sample: every env with a row in the first tile, the last tile and the first tile of each CTA's second round
    (tiles 2 SMs .. 4 SMs - 1), plus a stride sample"""
    grid, rows = 2 * sms, B * n
    ranges = [(0, TC_ROWS), ((rows - 1) // TC_ROWS * TC_ROWS, rows), (grid * TC_ROWS, 2 * grid * TC_ROWS)]
    extra = set()
    for r0, r1 in ranges:
        r1 = min(r1, rows)
        if r0 < r1:
            extra |= set(range(r0 // n, (r1 - 1) // n + 1))
    return sample_envs(B, 1, stride, extra)


# ---- inputs -------------------------------------------------------------------------------------------------------------
DOMAINS = ("uniform", "env", "zeros")


def observations(B, n, D, domain, rng):
    """(B, n, D) float32: 'uniform' [0, 1); 'env' the env's value set — 0/1 window bits and up to three small scalar columns
    per agent; 'zeros' the env's value set with every fifth env all zero (the padded steps of the update)"""
    if domain == "uniform":
        return rng.random((B, n, D), dtype=np.float32)
    obs = (rng.random((B, n, D)) < 0.3).astype(np.float32)
    ns = min(3, D - 1)
    if ns > 0:
        obs[..., D - ns:] = rng.integers(0, 21, (B, n, ns)).astype(np.float32) / 20.0
    if domain == "zeros":
        obs[::5] = 0.0
    return obs


def avail(B, n, rng):
    """(B, n, 5) 0/1: ~90 % of the actions available, action 4 always (the kernels' `last` rule needs one), some agents with
    action 4 alone"""
    av = (rng.random((B, n, 5)) < 0.9).astype(np.uint8)
    av[..., 4] = 1
    av[rng.random((B, n)) < 0.05, :4] = 0
    return av


def avail_bits(av):
    return (av * np.array([1, 2, 4, 8, 16], np.uint8)).sum(-1).astype(np.uint8)


def unpack_avail(bits):
    return ((bits[..., None] >> np.arange(5, dtype=np.uint8)) & 1).astype(np.uint8)


def device_obs(B, n, D, seed, device="cuda"):
    """(B, n, D) float32 generated on the device with the env's value set (no host copy of the whole batch)"""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    obs = torch.empty((B, n, D), dtype=torch.float32, device=device)
    obs.bernoulli_(0.3, generator=g)
    ns = min(3, D - 1)
    if ns > 0:
        obs[..., D - ns:].uniform_(0.0, 1.0, generator=g)
    return obs


def device_avail_bits(B, n, seed, device="cuda"):
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    return torch.randint(0, 32, (B, n), dtype=torch.uint8, device=device, generator=g) | 16


# ---- policies -----------------------------------------------------------------------------------------------------------
def _env_spec(n, D):
    from com_marl_b200.spaces import Box, Discrete, EnvSpec
    return EnvSpec(Box(np.zeros(n * D), np.ones(n * D)), Discrete(5))


def randomize_biases(pol, seed):
    """every bias redrawn in +-0.2 (the reference initialises them to zero, which hides a bias read from the wrong place)"""
    import torch
    rng = np.random.default_rng(seed)
    with torch.no_grad():
        for k, v in pol.state_dict().items():
            if k.endswith("bias"):
                v.copy_(torch.from_numpy(rng.uniform(-0.2, 0.2, tuple(v.shape)).astype(np.float32)))
    return pol


def cent_policy(n, D, relu=False, math="tc", seed=0):
    import torch
    from com_marl_b200.policy import CentralizedCategoricalMLPPolicy
    torch.manual_seed(seed)
    pol = CentralizedCategoricalMLPPolicy(_env_spec(n, D), n, hidden_nonlinearity=torch.relu if relu else torch.tanh, math=math,
                                          seed=seed + 11)
    return randomize_biases(pol, seed + 1)


def dec_policy(n, D, seed=0):
    import torch
    from com_marl_b200.policy import DecCategoricalMLPPolicy
    torch.manual_seed(seed)
    return randomize_biases(DecCategoricalMLPPolicy(_env_spec(n, D), n, seed=seed + 11), seed + 1)


def state(pol):
    return {k: v.detach().cpu().numpy() for k, v in pol.state_dict().items()}


def kind_of(pol):
    from com_marl_b200.policy import CentralizedCategoricalMLPPolicy, DecCategoricalMLPPolicy
    if isinstance(pol, CentralizedCategoricalMLPPolicy):
        return "cent"
    return "dec" if isinstance(pol, DecCategoricalMLPPolicy) else "comm"


def math_of(pol):
    return "tc" if pol.uses_tensor_cores() else "fp32"


def label(pol, B, extra=""):
    n, D = pol._n_agents, pol._dec_obs_dim
    K = n * D if kind_of(pol) == "cent" else D
    return f"{kind_of(pol)} math={math_of(pol)} n={n} D={D} K={K} panels={panels(K)} B={B}{' ' + extra if extra else ''}"


# ---- the kernel ---------------------------------------------------------------------------------------------------------
def forward(pol, obs, bits=None, u=None, tick=None, episode=None, env_id0=0, greedy=False):
    """one cm_policy_forward call on device tensors; -> device outputs {logits, probs, actions} (filled with -7 first)"""
    import torch
    assert greedy or u is not None or (tick is not None and episode is not None), "the in-kernel draw reads tick and episode"
    B, n = obs.shape[0], pol._n_agents
    out = dict(logits=torch.full((B, n, 5), -7.0, device=obs.device), probs=torch.full((B, n, 5), -7.0, device=obs.device),
               actions=torch.full((B, n), -7, dtype=torch.int8, device=obs.device))
    pol.act_device(obs, avail_bits=bits, sample_u=u, tick=tick, episode=episode, greedy=greedy, env_id0=env_id0, **out)
    pol.check_errors()
    return out


def host(out, envs=None):
    """device outputs -> numpy, only the rows of `envs` if given"""
    import torch
    if envs is None:
        return {k: v.cpu().numpy() for k, v in out.items()}
    idx = torch.as_tensor(envs, device=next(iter(out.values())).device)
    return {k: v.index_select(0, idx).cpu().numpy() for k, v in out.items()}


def oracle(pol, w, obs, av):
    """float64 oracle of the policy's kind on host arrays obs (b, n, D), av (b, n, 5) -> (logits, probs)"""
    from oracle import oracle as orc
    if kind_of(pol) == "cent":
        return orc.policy_forward_cent(w, obs.reshape(obs.shape[0], -1), av, relu=pol._relu, dtype=np.float64)
    return orc.policy_forward_dec(w, obs, av, dtype=np.float64)


# ---- comparison -----------------------------------------------------------------------------------------------------------
def _first_bad(bad, envs):
    e, a = (int(i) for i in np.argwhere(bad.reshape(bad.shape[0], bad.shape[1], -1).any(-1))[0])
    return (int(envs[e]) if envs is not None else e, a)


def check(lbl, got, ref, u, envs=None, key=None, tol=TOL):
    """logits within tol * max(1, max|ref|), probabilities within tol, actions exactly the inverse CDF of the kernel's own
    probabilities for the uniforms `u`; a failure names `lbl` and the first bad (env, agent) (`envs`: the batch index of each
    row of a sample).  The largest error / tol is recorded under `key` = (kind, math)."""
    ref_logits, ref_probs = ref
    scale = max(1.0, float(np.abs(ref_logits).max()))
    el = np.abs(got["logits"] - ref_logits)
    ep = np.abs(got["probs"] - ref_probs)
    if key is not None:
        REPORT[key] = max(REPORT.get(key, 0.0), float(el.max()) / scale / tol, float(ep.max()) / tol)
    bad = ~(el <= tol * scale)
    assert not bad.any(), f"{lbl}: logits off by {el.max() / scale:.2e} (relative) at (env, agent) {_first_bad(bad, envs)}"
    bad = ~(ep <= tol)
    assert not bad.any(), f"{lbl}: probs off by {ep.max():.2e} at (env, agent) {_first_bad(bad, envs)}"
    if u is not None and "actions" in got:
        bad = got["actions"] != inverse_cdf(got["probs"], u)
        assert not bad.any(), f"{lbl}: actions differ from the inverse CDF of the kernel's probabilities at (env, agent) {_first_bad(bad, envs)}"


def same(lbl, got, base):
    for k in got:
        a, b = got[k], base[k]
        bad = a.view(np.uint8).reshape(a.shape + (-1,)) != b.view(np.uint8).reshape(b.shape + (-1,))
        assert not bad.any(), f"{lbl}: {k} differs bitwise at (env, agent) {_first_bad(bad, None)}"


# ---- the action stream, restated --------------------------------------------------------------------------------------------
_M0, _M1, _W0, _W1, _U32 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85, 0xFFFFFFFF


def philox4x32_10(seed, c0, c1, c2, c3):
    """Philox4x32-10 (common.cuh::philox4x32_10) over numpy arrays of counters, key = (seed low word, seed high word);
    -> uint32 array (..., 4)"""
    c = [np.asarray(x, np.uint64) & _U32 for x in (c0, c1, c2, c3)]
    c = np.broadcast_arrays(*c)
    c = [x.copy() for x in c]
    k0, k1 = np.uint64(int(seed) & _U32), np.uint64((int(seed) >> 32) & _U32)
    m = np.uint64(_U32)
    for _ in range(10):
        p0 = np.uint64(_M0) * c[0]
        p1 = np.uint64(_M1) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & m, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & m]
        k0, k1 = (k0 + np.uint64(_W0)) & m, (k1 + np.uint64(_W1)) & m
    return np.stack(c, -1).astype(np.uint32)


def u24(w):
    """24 random bits -> U[0, 1) float32 on the 2^-24 lattice (common.cuh::u24)"""
    return ((np.asarray(w, np.uint32) >> 8).astype(np.float32) * np.float32(2.0 ** -24)).astype(np.float32)


def action_u(seed, env_id0, envs, tick, episode, n):
    """the uniform categorical_finish draws for agent il of env e (batch index) when no sample_u is given:
    philox(seed; env_id0 + e, tick[e], 4 | episode[e] << 8, il >> 2), word il & 3, u24.  -> (len(envs), n) float32"""
    envs = np.asarray(envs, np.int64)
    il = np.arange(n, dtype=np.int64)
    e = envs[:, None]
    blk = philox4x32_10(seed, (env_id0 + e) & _U32, np.asarray(tick, np.int64)[e] & _U32,
                        (4 | (np.asarray(episode, np.int64)[e] << 8)) & _U32, il[None, :] >> 2)
    return u24(np.take_along_axis(blk, (il & 3)[None, :, None].repeat(len(envs), 0), -1)[..., 0])
