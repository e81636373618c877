"""Compare cm_ppo_net of two builds of libcommarl_b200.so output for output on the same seeded batches: the Comm-DP and Obs-DP
policies (policy_call) and CommBaseCritic (critic_call), forward outputs, losses and gradient blobs.  The library this checkout
built and the one given with --other (for instance one built from the parent commit) run alternately, --reps times each.  The
per-step outputs must be bit-identical.  Losses and gradients are sums of fp32 atomic adds whose order varies from run to run, so
each library's own spread over its runs is reported next to the largest difference between the two libraries; the two must
agree as closely as a library agrees with itself.
    python tools/ppo_net_ab.py --other /path/to/libcommarl_b200.so
Prints ONE JSON line; exit code 1 when any array differs."""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402


def _load_other(path):
    """only the entry points policy_call / critic_call reach (the other build may have an older ABI)"""
    from com_marl_b200 import _native as N
    L = C.CDLL(path)
    L.cm_ppo_net_workspace_floats.restype = C.c_size_t
    L.cm_ppo_net_workspace_floats.argtypes = [C.POINTER(N.NetDesc), C.c_int64, C.c_int32]
    L.cm_ppo_net.restype = C.c_int
    L.cm_ppo_net.argtypes = [C.POINTER(N.NetDesc), C.POINTER(N.NetIO), C.c_void_p]
    return L


def _calls(F, f, b, P):
    """every output of one forward and one forward + backward of both networks"""
    out = {}
    F.pol_map.refresh()
    F.cri_map.refresh()
    with torch.no_grad():
        r = F.policy_call(f, None, want_probs=True)
    out.update(fwd_ll=r["ll"], fwd_entropy=r["entropy"], fwd_probs=r["probs"])
    idx = F.step_index(f, np.arange(P), valid_only=True)
    adv = b["adv"].reshape(-1).index_select(0, idx)
    old = r["ll"].index_select(0, idx) + 0.15 * torch.randn(idx.numel(), device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
    r = F.policy_call(f, idx, adv=adv, old_ll=old, backward=True, inv_count=1.0 / idx.numel())
    out.update(pol_ll=r["ll"], pol_entropy=r["entropy"], pol_loss=r["loss"], pol_grad=F.pol_map.grad.clone())
    r = F.critic_call(f, None, returns=b["returns"].reshape(-1), backward=True)
    out.update(cri_values=r["values"], cri_loss=r["loss"], cri_grad=F.cri_map.grad.clone())
    return {k: v.clone() for k, v in out.items()}


def _cases():
    from com_marl_b200.policy import DecCategoricalMLPPolicy
    from com_marl_b200.ppo import CommBaseCritic, DevicePPO
    from com_marl_b200.spaces import Box, Discrete, EnvSpec
    from test_gpu_ppo_fused import _make
    for n, D, L, P, T in [(3, 29, 2, 7, 9), (4, 21, 2, 40, 11), (9, 53, 3, 4, 5), (32, 53, 2, 5, 7), (65, 53, 2, 2, 3), (200, 53, 2, 2, 3)]:
        _, fused, b0 = _make(n, D, L, P, T, seed=n)
        yield f"comm_n{n}_D{D}_L{L}", fused, b0, P
    for n, D in [(4, 21), (32, 53), (200, 53)]:
        _, _, b0 = _make(n, D, 2, 3, 4, seed=n + 1)
        torch.manual_seed(n)
        spec = EnvSpec(Box(np.zeros(n * D), np.ones(n * D)), Discrete(5))
        yield f"dec_n{n}_D{D}", DevicePPO(DecCategoricalMLPPolicy(spec, n), CommBaseCritic(spec, n), fused=True), b0, 3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--other", required=True, help="path of the other build of libcommarl_b200.so")
    ap.add_argument("--reps", type=int, default=4)
    args = ap.parse_args()
    from com_marl_b200 import _native as N
    mine, other = N.lib(), _load_other(args.other)
    spread = lambda xs, ys: max(float((x - y).abs().max()) for x in xs for y in ys)  # noqa: E731
    res, ok = {}, True
    for name, algo, b0, P in _cases():
        b = algo.finish_batch(dict(b0))
        F, f = algo._fused, b["_flat"]
        runs = {"mine": [], "other": []}
        for _ in range(args.reps):
            for tag, lib in (("mine", mine), ("other", other)):
                N._lib = lib
                try:
                    runs[tag].append(_calls(F, f, b, P))
                finally:
                    N._lib = mine
        case = {}
        for k in runs["mine"][0]:
            xs, ys = [r[k] for r in runs["mine"]], [r[k] for r in runs["other"]]
            cross, self_spread = spread(xs, ys), max(spread(xs, xs), spread(ys, ys))
            if k.startswith("fwd_") or k in ("pol_ll", "pol_entropy", "cri_values"):
                good = cross == 0.0 and self_spread == 0.0
            else:
                good = cross <= 2.0 * self_spread
            case[k] = dict(cross=cross, self=self_spread, ok=good)
            ok = ok and good
        res[name] = case
    print(json.dumps(dict(agree=ok, cases=res)), flush=True)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
