"""Every kernel path of the Comm-DP policy forward (cm_policy_forward) against the float64 oracle.

tests/test_gpu_policy.py checks the reference's default architecture at a handful of team sizes.  This file covers what
the kernels branch on (the paths are listed in tests/policy_path_util.py):
  (a) every team size 1 .. 256, which runs every kVec, env slot and NS / WARPS build;
  (b) an architecture matrix per path: 1 .. 4 GCN layers, residual on / off, GCN bias on / off, 'general' / 'dot'
      attention, D up to 128, with batches that give every tcgen05 CTA three tiles, the last one ragged;
  (c) packed observations (obs_bits) at the word edges of the window, for Comm-DP and Obs-DP;
  (d) probabilities and actions that do not depend on which optional outputs are requested;
  (e) peaked attention whose mass the masks remove, down to masked-in sums far below the renormalisation's 1e-12;
  (f) the device rollout at 1, 3 and 4 layers, recomputed step by step by the oracle.
Tolerances are those of tests/test_gpu_policy.py: logits within 1e-5 * max(1, max|ref|), probabilities and attention
within 1e-5, sampled actions exactly the inverse-CDF specification on the kernel's own probabilities.

test_oracle_matches_torch_float64 needs no GPU: it holds the oracle itself to the module's torch formula.
"""
import itertools

import numpy as np
import pytest
import torch

import policy_path_util as U
from oracle import oracle as orc

gpu = pytest.mark.gpu


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def test_oracle_matches_torch_float64():
    """oracle.policy_forward(float64) == CommCategoricalMLPPolicy.forward on a float64 copy of the module, for every layer
    count, residual on / off, GCN bias on / off and both attention types"""
    n, D, B = 7, 13, 4
    for L, residual, gcn_bias, attention in itertools.product((1, 2, 3, 4), (True, False), (True, False), ("general", "dot")):
        w = U.weights(n, D, L, residual, gcn_bias, attention, seed=L)
        x = U.inputs(n, D, L, B, seed=L + 10)
        pol = U.policy(w, n, D, L, "auto", residual, attention, device="cpu").double()
        assert ("gcn_layers.0.bias" in w) == gcn_bias
        with torch.no_grad():
            dist, M = pol.forward(torch.from_numpy(x["obs"].reshape(B, -1)).double(), torch.from_numpy(x["avail"].reshape(B, -1)).double(),
                                  torch.from_numpy(x["adj"]).double(), torch.from_numpy(x["chan"].reshape(B, L * n, n)).double())
        _, probs, attn = U.oracle(w, x, residual)
        label = f"L={L} residual={residual} gcn_bias={gcn_bias} {attention}"
        assert np.abs(dist.probs.numpy() - probs).max() <= 1e-12, label
        assert np.abs(M.numpy() - attn).max() <= 1e-12, label


@gpu
@pytest.mark.parametrize("math", ["tc"])
def test_every_team_size(math):
    """n = 1 .. 256 at D = 53, L = 2 and a small ragged batch"""
    D, L = 53, 2
    for n in range(1, 257):
        B = 2 * (U.TC_ROWS // U.tc_slot(n)) + 1 if n <= 64 else 3
        w = U.weights(n, D, L, seed=n)
        x = U.inputs(n, D, L, B, seed=n + 1000)
        got = U.forward(U.policy(w, n, D, L, math), x)
        U.check(f"n={n} D={D} L={L} B={B} math={math} [{U.path_of(n)}]", got, U.oracle(w, x), x["u"])


@gpu
@pytest.mark.parametrize("path", list(U.PATHS))
def test_architecture_matrix(path):
    """(b) every layer count, residual, GCN bias and attention type on each kernel path, and (e) the same probabilities
    and actions, bit for bit, when logits and attention are not requested"""
    sms = _sms()
    for c in U.arch_cases(path):
        w, x, got = U.arch_run(c, sms)
        label = f"{U.arch_label(c)} B={len(x['obs'])}"
        U.check(label, got, U.oracle(w, x, c["residual"]), x["u"])
        _, _, lean = U.arch_run(c, sms, outputs=("probs", "actions"))
        U.same(label + " without logits / attention", lean, got)


NBITS = (8, 31, 32, 33, 61, 64, 65, 90, 96)


@gpu
@pytest.mark.parametrize("team", [4, 32, 54, 72, "dec"])
def test_packed_observations(team):
    """obs_bits with obs = NULL at every word edge of the window and 0 .. 3 scalar columns: the oracle on the unpacked
    rows, and bit-identical to the call on fp32 rows"""
    from com_marl_b200.policy import DecCategoricalMLPPolicy
    from com_marl_b200.spaces import Box, Discrete, EnvSpec
    dec = team == "dec"
    n, L = (8 if dec else team), 2
    for i, nbits in enumerate(NBITS):
        ns = (i + n) % 4
        D = nbits + ns
        x = U.inputs(n, D, L, 2 * (U.TC_ROWS // U.tc_slot(n)) + 3 if n <= 64 else 5, seed=nbits * 10 + ns, nbits=nbits)
        label = f"{'Obs-DP' if dec else 'Comm-DP'} n={n} obs_nbits={nbits} scalars={ns}"
        if dec:
            torch.manual_seed(nbits)
            pol = DecCategoricalMLPPolicy(EnvSpec(Box(np.zeros(n * D), np.ones(n * D)), Discrete(5)), n)
            with torch.no_grad():
                for k, v in pol.state_dict().items():
                    if k.endswith("bias"):
                        v.uniform_(-0.1, 0.1)
            w = {k: v.cpu().numpy() for k, v in pol.state_dict().items()}
            logits, probs = orc.policy_forward_dec(w, x["obs"], x["avail"], dtype=np.float64)
            ref, outputs = (logits, probs, None), ("logits", "probs", "actions")
        else:
            w = U.weights(n, D, L, seed=nbits)
            pol = U.policy(w, n, D, L, "tc")
            ref, outputs = U.oracle(w, x), ("logits", "probs", "attention", "actions")
        got = U.forward(pol, x, outputs, packed_nbits=nbits)
        U.check(label, got, ref, x["u"])
        U.same(label + " packed vs fp32 rows", got, U.forward(pol, x, outputs))


# (path, team, math, attention, scales): the scales grow the score path geometrically until the median masked-in mass is
# far below 1e-6
PEAKED = [("small", 8, "tc", "general"), ("slot32", 32, "tc", "general"), ("slot64", 64, "tc", "general"),
          ("slot64", 48, "tc", "dot"), ("mma", 72, "tc", "general"), ("mma", 200, "tc", "dot")]
SCALES = {"general": (1.0, 2.0, 4.0, 8.0, 16.0), "dot": (1.0, 1.5, 2.25, 3.375)}


@gpu
def test_peaked_attention():
    """masks that keep only the lower half of each row's attention (and rows with no neighbour at all, where the reference
    gives tanh(b)), on attention made peaked by scaling the score path: float32 torch must agree with float64 first, then
    every path must meet the standard tolerance.  Prints the masked-in mass and the errors of every case."""
    D, L = 53, 2
    failures, lowest = [], 1.0
    print("\npath      n    attention scale  median mass  min mass   logits     probs      attention")
    for path, n, math, attention in PEAKED:
        B = 64 if n <= 64 else 12
        base_w = U.weights(n, D, L, attention=attention, seed=n + 5)
        base_x = U.inputs(n, D, L, B, seed=n + 6)
        for scale in SCALES[attention]:
            w, x, mass = U.peaked(base_w, base_x, scale, attention, seed=n)
            lowest = min(lowest, float(np.median(mass)))
            ref = U.oracle(w, x)
            label = f"peaked {path} n={n} {attention} scale={scale} math={math} [{U.path_of(n)}]"
            cpu = U.policy(w, n, D, L, "auto", attention=attention, device="cpu")
            with torch.no_grad():
                dist, _ = cpu.forward(torch.from_numpy(x["obs"].reshape(B, -1)), torch.from_numpy(x["avail"].reshape(B, -1)).float(),
                                      torch.from_numpy(x["adj"]).float(), torch.from_numpy(x["chan"].reshape(B, L * n, n)).float())
            assert np.abs(dist.probs.numpy() - ref[1]).max() <= 2e-6, f"{label}: float32 torch itself is off, the case is ill-posed"
            got = U.forward(U.policy(w, n, D, L, math, attention=attention), x)
            e = U.errors(got, ref)
            print(f"{path:9s} {n:4d} {attention:9s} {scale:6.3f} {np.median(mass):11.2e} {mass.min():10.2e} "
                  f"{e['logits']:10.2e} {e['probs']:10.2e} {e['attention']:10.2e}")
            try:
                U.check(label, got, ref, x["u"])
            except AssertionError as err:
                failures.append(str(err))
    assert lowest < 1e-6, f"the scales reach a median masked-in mass of {lowest:.2e} only"
    assert not failures, "\n".join(failures)


@gpu
@pytest.mark.parametrize("L", [1, 3, 4])
@pytest.mark.parametrize("n", [32, 72])
def test_rollout_layers(n, L):
    """RolloutEngine at n_gcn_layers = L: every recorded step's probabilities recomputed by the float64 oracle from the
    recorded observation, adjacency and channel planes (the policy read the packed observation the env kernel wrote)"""
    import os
    import sys
    sys.path.insert(0, os.path.join(U.TESTS, "golden"))
    import ref_harness
    from com_marl_b200.rollout import RolloutEngine, make_policy
    from com_marl_b200.scenario import ScenarioSpec
    params = ref_harness.scenario_params("pp", 20, 1, 0.08, cap=2, loss=0.2, n_agents=n, n_preys=n, n_gcn_layers=L, max_env_steps=5)
    spec = ScenarioSpec.from_params("pp", params, seed=11)
    pol = make_policy(spec)
    assert pol.n_gcn_layers == L and pol.uses_tensor_cores()
    B = 96
    eng = RolloutEngine(spec, pol, B, ring=4, use_graph=True)
    assert "obs_bits" in eng.traj
    eng.reset()
    w = {k: v.cpu().numpy() for k, v in pol.state_dict().items()}
    unpack = lambda bits: np.unpackbits(bits.view(np.uint8), axis=-1, count=n, bitorder="little")  # noqa: E731
    for chunk in range(2):          # eager, then the captured graph
        eng.run_chunk()
        t = {k: v.cpu().numpy() for k, v in eng.traj.items()}
        for k in range(eng.K):
            adj, chan = unpack(t["adj_bits"][k]), unpack(t["chan_bits"][k])
            assert chan.shape == (B, L, n, n)
            _, probs, _ = orc.policy_forward(w, t["obs"][k], None, adj, chan, dtype=np.float64)
            U.check(f"rollout n={n} L={L} chunk {chunk} step {k}", dict(probs=t["probs"][k]), (None, probs, None), None)
    eng.env.check_errors()
    pol.check_errors()
