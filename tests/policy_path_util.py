"""Kernel paths of cm_policy_forward (Comm-DP) and the helpers tests/test_gpu_policy_paths.py compares them with.

cm_policy_forward picks one of four paths by team size:
  * n <= 16: policy_tc_kernel with the exact CUDA-core attention (kVec = 4 / 2 / 1 by the team's divisibility);
  * 17 <= n <= 32 and 33 <= n <= 64: policy_tc_kernel with the tcgen05 attention in env slots of 32 / 64 tile rows;
  * n > 64: encoder and head on policy_tc_kernel, the attention on policy_attn_mma_kernel (mma.sync).

Every comparison is against the float64 oracle (oracle.policy_forward).  Nothing here touches CUDA at import time.
"""
import os

import numpy as np

TESTS = os.path.dirname(os.path.abspath(__file__))
TC_ROWS = 128                                # policy_tc_kernel: agent rows per tile


def tc_slot(n):
    """tile rows per env of policy_tc_kernel (launch_tc_mode): n itself with the CUDA-core attention, 32 / 64 with the
    tensor-core one"""
    return n if n <= 16 else (32 if n <= 32 else 64)


def path_of(n):
    if n > 64:
        return "tc + mma attention"
    if n <= 16:
        return f"tc cuda-core attention kVec={4 if n % 4 == 0 else (2 if n % 2 == 0 else 1)}"
    return f"tc tcgen05 attention slot {tc_slot(n)}"


def ragged_B(n, sms, tiles_per_cta=3):
    """a batch whose tcgen05 tiles give every CTA of the persistent grid (2 CTAs per SM) `tiles_per_cta` tiles, the
    last one ragged"""
    ept = TC_ROWS // tc_slot(n)
    return tiles_per_cta * 2 * sms * ept - max(1, ept // 2) if ept > 1 else tiles_per_cta * 2 * sms


# ---- weights and inputs ---------------------------------------------------------------------------------------------
def weights(n, D, L, residual=True, gcn_bias=True, attention="general", seed=0):
    """state dict (numpy float32) of a CommCategoricalMLPPolicy with the reference initialisation and every bias redrawn
    in +-0.1, so that each layer has its own distinct bias and swapping layers changes the result"""
    import torch
    from com_marl_b200.policy import CommCategoricalMLPPolicy
    from com_marl_b200.spaces import Box, Discrete, EnvSpec
    torch.manual_seed(seed)
    pol = CommCategoricalMLPPolicy(EnvSpec(Box(np.zeros(n * D), np.ones(n * D)), Discrete(5)), n, n_gcn_layers=L, residual=residual,
                                   gcn_bias=gcn_bias, attention_type=attention, device="cpu")
    rng = np.random.default_rng(seed + 7)
    w = {k: v.numpy().copy() for k, v in pol.state_dict().items()}
    for k in w:
        if k.endswith("bias"):
            w[k] = rng.uniform(-0.1, 0.1, w[k].shape).astype(np.float32)
    return w


def policy(w, n, D, L, math, residual=True, attention="general", device="cuda"):
    import torch
    from com_marl_b200.policy import CommCategoricalMLPPolicy
    from com_marl_b200.spaces import Box, Discrete, EnvSpec
    gcn_bias = "gcn_layers.0.bias" in w
    pol = CommCategoricalMLPPolicy(EnvSpec(Box(np.zeros(n * D), np.ones(n * D)), Discrete(5)), n, n_gcn_layers=L, residual=residual,
                                   gcn_bias=gcn_bias, attention_type=attention, device=device, math=math)
    pol.load_state_dict({k: torch.as_tensor(v) for k, v in w.items()})
    return pol


def inputs(n, D, L, B, seed, ploss=0.2, nbits=None):
    """random 0/1 observation windows (the first `nbits` columns, default D - 2) + scalar columns, random neighbour and
    channel masks with self in, a few unavailable actions, sampling uniforms"""
    rng = np.random.default_rng(seed)
    nbits = D - 2 if nbits is None else nbits
    obs = (rng.random((B, n, D)) < 0.3).astype(np.float32)
    obs[..., nbits:] = rng.random((B, n, D - nbits)).astype(np.float32)
    adj = (rng.random((B, n, n)) < 0.7).astype(np.uint8) | np.eye(n, dtype=np.uint8)
    chan = (rng.random((B, L, n, n)) >= ploss).astype(np.uint8) | np.eye(n, dtype=np.uint8)
    avail = np.ones((B, n, 5), np.uint8)
    avail[rng.random((B, n)) < 0.1, rng.integers(0, 5)] = 0
    u = rng.random((B, n)).astype(np.float32)
    return dict(obs=obs, adj=adj, chan=chan, avail=avail, u=u)


def obs_bits_of(obs, nbits):
    """the packed observation (cm_step_io.obs_bits) of fp32 rows: bit k of words 0..2 = column k < nbits, words 3..5 the
    float bits of the remaining columns (zero where there is none)"""
    win = obs[..., :nbits]
    assert np.isin(win, (0.0, 1.0)).all()
    bits = np.zeros(obs.shape[:-1] + (96,), np.uint8)
    bits[..., :nbits] = win != 0
    words = np.packbits(bits, axis=-1, bitorder="little").view("<u4")
    scal = np.zeros(obs.shape[:-1] + (3,), np.uint32)
    rest = np.ascontiguousarray(obs[..., nbits:]).view(np.uint32)
    scal[..., :rest.shape[-1]] = rest
    return np.concatenate([words, scal], axis=-1).view(np.int32)


def oracle(w, x, residual=True):
    from oracle import oracle as orc
    return orc.policy_forward(w, x["obs"], x["avail"], x["adj"], x["chan"], dtype=np.float64, residual=residual)


# ---- the kernel ---------------------------------------------------------------------------------------------------
def forward(pol, x, outputs=("logits", "probs", "attention", "actions"), packed_nbits=None):
    """one cm_policy_forward call on device copies of `x`; -> {output: numpy}.  packed_nbits: read the observation as
    obs_bits with that many window bits and pass no fp32 rows (obs = NULL)"""
    import torch
    from com_marl_b200 import _native as N
    dev = pol.device
    B, n = x["obs"].shape[:2]
    t = lambda a, dt=torch.float32: torch.as_tensor(a, dtype=dt).to(dev)  # noqa: E731
    comm = pol._kind == N.POLICY_COMM
    adj_b = pol.pack_mask(t(x["adj"]), n) if comm else None
    ch_b = pol.pack_mask(t(x["chan"]), n) if comm else None
    av_b = t((x["avail"] * np.array([1, 2, 4, 8, 16], np.uint8)).sum(-1), torch.uint8)
    shapes = dict(logits=((B, n, 5), torch.float32), probs=((B, n, 5), torch.float32), attention=((B, n, n), torch.float32),
                  actions=((B, n), torch.int8))
    out = {k: torch.full(shapes[k][0], -7, dtype=shapes[k][1], device=dev) for k in outputs}
    if packed_nbits is None and comm:
        pol.act_device(t(x["obs"]), adj_b, ch_b, av_b, t(x["u"]), **out)
    elif packed_nbits is None:
        pol.act_device(t(x["obs"]), av_b, t(x["u"]), **out)
    else:
        ob = t(obs_bits_of(x["obs"], packed_nbits), torch.int32)
        desc, io = pol._call_structs(ob, adj_b, ch_b, av_b, t(x["u"]), None, None, False, out.get("probs"), out.get("logits"),
                                     out.get("attention"), out.get("actions"), 0, 0)
        io.obs, io.obs_bits, io.obs_nbits = None, N.ptr(ob), int(packed_nbits)
        with torch.cuda.device(dev):
            N.check("cm_policy_forward", N.lib().cm_policy_forward(N.C.byref(desc), N.C.byref(io), N.stream_ptr()))
    pol.check_errors()
    return {k: v.cpu().numpy() for k, v in out.items()}


# ---- comparison -------------------------------------------------------------------------------------------------------
def inverse_cdf(p, u):
    """the sampling specification: the first action whose fp32 running sum of the probabilities exceeds u, else the last
    action of non-zero probability"""
    c = np.zeros(u.shape, np.float32)
    want = np.full(u.shape, -1, np.int64)
    for a in range(p.shape[-1]):
        c = (c + p[..., a]).astype(np.float32)
        want = np.where((want < 0) & (u < c), a, want)
    last = np.where(p > 0, np.arange(p.shape[-1]), -1).max(-1)
    return np.where(want < 0, last, want)


def _first_bad(bad):
    """(env, agent) of the first True in a (B, n, ...) array"""
    idx = np.argwhere(bad.reshape(bad.shape[0], bad.shape[1], -1).any(-1))
    return tuple(int(i) for i in idx[0])


def errors(got, ref):
    """{output: max error} of the kernel outputs against the oracle's (logits relative to max(1, max|ref|))"""
    ref_logits, ref_probs, ref_attn = ref
    e = {}
    if "logits" in got:
        e["logits"] = float(np.abs(got["logits"] - ref_logits).max()) / max(1.0, float(np.abs(ref_logits).max()))
    if "probs" in got:
        e["probs"] = float(np.abs(got["probs"] - ref_probs).max())
    if "attention" in got:
        e["attention"] = float(np.abs(got["attention"] - ref_attn).max())
    return e


def check(label, got, ref, u, tol=1e-5):
    """logits within tol * max(1, max|ref|), probabilities and attention within tol, actions exactly the inverse CDF of
    the kernel's own probabilities; a failure names `label` and the first bad (env, agent)"""
    ref_logits, ref_probs, ref_attn = ref
    if "logits" in got:
        scale = max(1.0, float(np.abs(ref_logits).max()))
        bad = np.abs(got["logits"] - ref_logits) > tol * scale
        assert not bad.any(), (f"{label}: logits off by {np.abs(got['logits'] - ref_logits).max() / scale:.2e} (relative) at "
                               f"(env, agent) {_first_bad(bad)}")
    if "probs" in got:
        bad = np.abs(got["probs"] - ref_probs) > tol
        assert not bad.any(), f"{label}: probs off by {np.abs(got['probs'] - ref_probs).max():.2e} at (env, agent) {_first_bad(bad)}"
    if "attention" in got:
        bad = np.abs(got["attention"] - ref_attn) > tol
        assert not bad.any(), f"{label}: attention off by {np.abs(got['attention'] - ref_attn).max():.2e} at (env, agent) {_first_bad(bad)}"
    if "actions" in got:
        assert "probs" in got
        bad = got["actions"] != inverse_cdf(got["probs"], u)
        assert not bad.any(), f"{label}: sampled actions differ from the inverse-CDF specification at (env, agent) {_first_bad(bad)}"


def same(label, got, base):
    """bit-identical outputs of two calls"""
    for k in got:
        a, b = got[k], base[k]
        bad = a.view(np.uint8).reshape(a.shape + (-1,)) != b.view(np.uint8).reshape(b.shape + (-1,))
        assert not bad.any(), f"{label}: {k} differs bitwise at (env, agent) {_first_bad(bad)}"


# ---- architecture matrix ------------------------------------------------------------------------------------------------
# Four architectures per kernel path: every layer count, residual on / off, GCN bias on / off and both attention types
# appear with every path.  D = 77 and D = 128 (two K panels of the encoder) are paired with L = 1 and L = 3.
ARCHS = [dict(L=1, residual=False, gcn_bias=True, attention="general", D=77),
         dict(L=2, residual=True, gcn_bias=False, attention="dot", D=53),
         dict(L=3, residual=False, gcn_bias=False, attention="general", D=128),
         dict(L=4, residual=True, gcn_bias=True, attention="dot", D=29)]
# (math, teams): one team per architecture, in ARCHS order
PATHS = {"small": ("tc", (6, 16, 14, 5)),                 # kVec 2 (teams of 2, 6, 10, 14), 4 and 1
         "slot32": ("tc", (17, 32, 24, 31)),
         "slot64": ("tc", (33, 64, 54, 40)),
         "mma": ("tc", (72, 200, 129, 256))}


def arch_cases(path):
    math, teams = PATHS[path]
    return [dict(a, n=n, math=math, id=f"{path}-n{n}-L{a['L']}") for a, n in zip(ARCHS, teams)]


def arch_label(c):
    return (f"n={c['n']} D={c['D']} L={c['L']} residual={c['residual']} gcn_bias={c['gcn_bias']} {c['attention']} "
            f"math={c['math']} [{path_of(c['n'])}]")


def arch_batch(c, sms):
    return ragged_B(c["n"], sms) if c["n"] <= 64 else 97


def arch_run(c, sms, outputs=("logits", "probs", "attention", "actions")):
    """-> (weights, inputs, kernel outputs) of one architecture case"""
    w = weights(c["n"], c["D"], c["L"], c["residual"], c["gcn_bias"], c["attention"], seed=c["n"] + 100 * c["L"])
    x = inputs(c["n"], c["D"], c["L"], arch_batch(c, sms), seed=c["n"] * 7 + c["L"])
    pol = policy(w, c["n"], c["D"], c["L"], c["math"], c["residual"], c["attention"])
    return w, x, forward(pol, x, outputs)


# ---- peaked attention -----------------------------------------------------------------------------------------------------
def peaked(w, x, scale, attention, n_empty=4, seed=0):
    """scale the score path (W_a for 'general', the encoder's output layer for 'dot') by `scale`, then replace the masks:
    each row keeps only the keys of the lower half of its float64 attention (self is not forced in), and `n_empty` rows
    keep no key at all.  -> (weights, inputs, masked-in mass of every non-empty row)"""
    from oracle import oracle as orc
    w = dict(w)
    k = "attention_layer.linear_in.weight" if attention == "general" else "encoder._output_layers.0.linear.weight"
    w[k] = (w[k].astype(np.float64) * scale).astype(np.float32)
    B, n = x["obs"].shape[:2]
    L = x["chan"].shape[1]
    _, _, M = orc.policy_forward(w, x["obs"], None, np.ones((B, n, n)), np.ones((B, L, n, n)), dtype=np.float64)
    order = np.argsort(M, axis=-1, kind="stable")
    keep = np.zeros((B, n, n), np.uint8)
    np.put_along_axis(keep, order[..., :n // 2], 1, axis=-1)
    rng = np.random.default_rng(seed)
    empty = rng.choice(B * n, size=n_empty, replace=False)
    keep.reshape(B * n, n)[empty] = 0
    mass = (M * keep).sum(-1).reshape(-1)
    mass = np.delete(mass, empty)
    return w, dict(x, adj=keep, chan=np.ones((B, L, n, n), np.uint8)), mass
