"""CPU checks of the set update's storage: K members' flat parameter buckets moved into [K][n] rows, and the set blob maps
(ppo_fused._SetBlobMap) that turn those rows into K kernel weight blobs with one gather and K gradient blobs back into the rows
with one inverse gather."""
import numpy as np
import pytest
import torch

from com_marl_b200.policy import CommCategoricalMLPPolicy, DecCategoricalMLPPolicy
from com_marl_b200.ppo import CommBaseCritic, FlatAdam, _SetBuckets
from com_marl_b200.ppo_fused import _BlobMap, _SetBlobMap
from com_marl_b200.spaces import Box, Discrete, EnvSpec


@pytest.mark.parametrize("kind,n,D,L", [("comm", 3, 11, 2), ("comm", 5, 29, 1), ("dec", 4, 13, 1), ("critic", 6, 7, 3)])
def test_set_blob_map_round_trip(kind, n, D, L):
    K = 3
    spec = EnvSpec(Box(np.zeros(n * D), np.ones(n * D)), Discrete(5))
    mods = []
    for i in range(K):
        torch.manual_seed(100 + i)
        if kind == "comm":
            mods.append(CommCategoricalMLPPolicy(spec, n, n_gcn_layers=L, device="cpu"))
        elif kind == "dec":
            mods.append(DecCategoricalMLPPolicy(spec, n, device="cpu"))
        else:
            mods.append(CommBaseCritic(spec, n, n_gcn_layers=L, device="cpu"))
    own = [m._pack_blob(m.state_dict()).clone() for m in mods]          # each member's blob packed on its own
    opts = [FlatAdam(m) for m in mods]
    one = _BlobMap(mods[0], mods[0]._pack_blob, opts[0].flat)
    buckets = _SetBuckets(opts)
    for i, m in enumerate(mods):                                          # parameters are views of row i of the set bucket
        p = next(q for q in m.parameters() if q.requires_grad)
        assert p.data_ptr() == buckets.flat[i].data_ptr()
    sm = _SetBlobMap(one, buckets.flat)
    assert sm.stride % 4 == 0 and sm.stride >= sm.nb == own[0].numel()
    blob = sm.refresh().clone()
    assert blob.shape == (K, sm.stride)
    for i in range(K):
        assert torch.equal(blob[i, :sm.nb], own[i])
        assert not blob[i, sm.nb:].any()
    # members differ: a row offset that is wrong would copy member 0's weights
    assert not torch.equal(blob[1, :sm.nb], blob[0, :sm.nb])
    # inverse: a gradient blob holding each member's own weights comes back as that member's flat row
    sm.grad.copy_(blob)
    out = torch.full_like(buckets.flat, float("nan"))
    sm.scatter_grad(out)
    assert torch.equal(out, buckets.flat)
    # an update of row 2 moves member 2's blob only
    buckets.flat[2].add_(1.0)
    blob2 = sm.refresh().clone()
    assert torch.equal(blob2[:2], blob[:2]) and not torch.equal(blob2[2], blob[2])
