"""Helpers of tests/test_gpu_policy_set.py: policies with distinct random weights and non-zero biases, random policy inputs,
and the reference of a PolicySet launch — one single-policy launch per env block (env_id0 offset per block).

Nothing here touches CUDA at import time.
"""
import numpy as np

SEED = 2718
CHANNEL_TABLE = [dict(pl=0), dict(pl=0.3), dict(pl=0.2, rcom=1)]


def env_spec(n, D):
    from com_marl_b200.spaces import Box, Discrete, EnvSpec
    return EnvSpec(Box(np.zeros(n * D, np.float32), np.ones(n * D, np.float32)), Discrete(5))


def make_policy(kind, n, D, math, seed, L=2, relu=False):
    """kind 'comm' / 'dec' / 'cent'; every parameter drawn from its own seed so that a wrong blob or a stale bias table shows"""
    import torch
    from com_marl_b200.policy import CentralizedCategoricalMLPPolicy, CommCategoricalMLPPolicy, DecCategoricalMLPPolicy
    torch.manual_seed(seed)
    if kind == "comm":
        pol = CommCategoricalMLPPolicy(env_spec(n, D), n, n_gcn_layers=L, device="cuda", seed=SEED, math=math)
    elif kind == "dec":
        pol = DecCategoricalMLPPolicy(env_spec(n, D), n, device="cuda", seed=SEED)
    else:
        pol = CentralizedCategoricalMLPPolicy(env_spec(n, D), n, hidden_nonlinearity="relu" if relu else "tanh", device="cuda",
                                              seed=SEED, math=math)
    g = torch.Generator(device="cpu").manual_seed(seed + 17)
    with torch.no_grad():
        for name, p in pol.named_parameters():
            scale = 0.3 if name.endswith("bias") else 1.0 / max(1.0, p.shape[-1] ** 0.5)
            p.copy_((torch.rand(p.shape, generator=g) * 2 - 1) * scale)
    return pol


def inputs(kind, n, D, L, B, seed):
    """random observation rows, mask bits, availability bits and Philox keys of B envs (device tensors)"""
    import torch
    g = torch.Generator(device="cpu").manual_seed(seed)
    W = (n + 31) // 32
    d = dict(obs=torch.rand((B, n, D), generator=g).cuda(),
             avail_bits=torch.randint(1, 32, (B, n), generator=g, dtype=torch.uint8).cuda(),
             tick=torch.randint(0, 1 << 20, (B,), generator=g, dtype=torch.int32).cuda(),
             episode=torch.randint(0, 1 << 10, (B,), generator=g, dtype=torch.int32).cuda())
    if kind == "comm":
        d["adj_bits"] = torch.randint(-(1 << 31), (1 << 31) - 1, (B, n, W), generator=g, dtype=torch.int32).cuda()
        d["chan_bits"] = torch.randint(-(1 << 31), (1 << 31) - 1, (B, L, n, W), generator=g, dtype=torch.int32).cuda()
    return d


def outputs(kind, n, B):
    import torch
    o = dict(probs=torch.full((B, n, 5), float("nan"), device="cuda"), logits=torch.full((B, n, 5), float("nan"), device="cuda"),
             actions=torch.full((B, n), -7, dtype=torch.int8, device="cuda"))
    if kind == "comm":
        o["attention"] = torch.full((B, n, n), float("nan"), device="cuda")
    return o


def call(pol, kind, inp, out, greedy, env_id0=0, sl=slice(None), **extra):
    """act_device of a policy or a PolicySet on the envs `sl` of the inputs / outputs"""
    kw = dict(avail_bits=inp["avail_bits"][sl], tick=inp["tick"][sl], episode=inp["episode"][sl], greedy=greedy,
              probs=out["probs"][sl], logits=out["logits"][sl], actions=out["actions"][sl], env_id0=env_id0, **extra)
    if kind == "comm":
        kw.update(adj_bits=inp["adj_bits"][sl], chan_bits=inp["chan_bits"][sl], attention=out["attention"][sl])
    pol.act_device(inp["obs"][sl], **kw)


def reference(pols, kind, n, inp, greedy):
    """one single-policy launch per block of B / P envs, block i with env_id0 = i * B / P"""
    B = inp["obs"].shape[0]
    Ep = B // len(pols)
    out = outputs(kind, n, B)
    for i, p in enumerate(pols):
        call(p, kind, inp, out, greedy, env_id0=i * Ep, sl=slice(i * Ep, (i + 1) * Ep))
    return out


def assert_same(lbl, got, ref):
    import torch
    torch.cuda.synchronize()
    for k in ref:
        a, b = got[k].cpu(), ref[k].cpu()
        if a.dtype.is_floating_point:
            ok = torch.equal(a.nan_to_num(123.0), b.nan_to_num(123.0)) and not bool(torch.isnan(b).any())
        else:
            ok = torch.equal(a, b) and not bool((b == -7).any())
        if not ok:
            bad = (a != b).reshape(a.shape[0], -1).any(1).nonzero().flatten()
            raise AssertionError(f"{lbl}: {k} differs (first envs {bad[:8].tolist()}, of {len(bad)})")
