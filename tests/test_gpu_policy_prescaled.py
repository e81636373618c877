"""policy_tc_kernel's tanh epilogues hand the next layer its activations pre-scaled, x' = 4096 tanh(.), and split them as
hi = 2^-12 fp16(x'), lo = fp16(x' - 4096 hi).  These cases drive every such layer (encoder, embedding E, graph
convolutions, head) to both ends of that split at once: a quarter of each layer's units saturated by a bias of +-30
(x' = +-4096, which fp16 must hold exactly), a quarter at |x| ~ 1e-5 (hi in the fp16 subnormals), a quarter at |x| ~ 1e-8
(hi = 0, the remainder in the fp16 subnormals), a quarter untouched.  Logits, probabilities and attention must stay within
the usual 1e-5 of the float64 oracle on the tensor-core attention (slots of 32 / 64 rows), the CUDA-core attention
(kVec = 4 / 1) and the large-team pipeline (encoder / head halves)."""
import numpy as np
import pytest
import torch

import policy_path_util as U

gpu = pytest.mark.gpu

# weight / bias pairs whose outputs go through a tanh epilogue into the next A operand
TANH_LAYERS = [("encoder._layers.0.linear.weight", "encoder._layers.0.linear.bias"),
               ("encoder._output_layers.0.linear.weight", "encoder._output_layers.0.linear.bias"),
               ("gcn_layers.{l}.weight", "gcn_layers.{l}.bias"),
               ("categorical_output_layer._layers.0.linear.weight", "categorical_output_layer._layers.0.linear.bias"),
               ("categorical_output_layer._layers.1.linear.weight", "categorical_output_layer._layers.1.linear.bias"),
               ("categorical_output_layer._layers.2.linear.weight", "categorical_output_layer._layers.2.linear.bias")]


def extreme_weights(n, D, L, seed):
    """U.weights with the output units of every tanh layer dealt round-robin into: saturated (bias +-30), |x| ~ 1e-5,
    |x| ~ 1e-8, unchanged"""
    w = U.weights(n, D, L, seed=seed)
    rng = np.random.default_rng(seed + 1)
    for wk, bk in TANH_LAYERS:
        for l in range(L) if "{l}" in wk else [None]:
            kw, kb = wk.format(l=l), bk.format(l=l)
            W, b = w[kw].astype(np.float64), w[kb].astype(np.float64)   # torch layout: W [out][in]
            g = np.arange(W.shape[0]) % 4
            b[g == 0] = np.where(rng.random(int((g == 0).sum())) < 0.5, -30.0, 30.0)
            for grp, s in ((1, 1e-5), (2, 1e-8)):
                W[g == grp] *= s
                b[g == grp] *= s
            w[kw], w[kb] = W.astype(np.float32), b.astype(np.float32)
    return w


@gpu
@pytest.mark.parametrize("n", [5, 8, 32, 48, 72])
def test_prescaled_activations_at_the_ends_of_fp16(n):
    D, L = 53, 2
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B = U.ragged_B(n, sms, tiles_per_cta=1) if n <= 64 else 40
    w = extreme_weights(n, D, L, seed=n)
    x = U.inputs(n, D, L, B, seed=n + 77)
    got = U.forward(U.policy(w, n, D, L, "tc"), x)
    U.check(f"n={n} saturated / subnormal activations [{U.path_of(n)}]", got, U.oracle(w, x), x["u"])
