"""Hand-written forward / backward of the PPO update for the three runner families (csrc/ppo_net_kernels.cu, cm_ppo_net).

``FusedCommNets`` is what ``DevicePPO`` drives instead of torch autograd when the baseline is a ``CommBaseCritic`` and the
policy a ``CommCategoricalMLPPolicy`` (runner_*_comm.py) or a ``DecCategoricalMLPPolicy`` (runner_*_obsDP.py); ``FusedCentNets``
when the policy is a ``CentralizedCategoricalMLPPolicy`` and the baseline a ``GaussianMLPBaseline`` (runner_*_cent.py, with
``fused=True``).  Per optimizer step ONE C call per network computes the loss of centralized_ma_ppo.py:390-438 /
comm_base_critic.py / gaussian_mlp_baseline.py and the gradient of every parameter, exact fp32.  The parameters stay torch
tensors (views of FlatAdam's flat bucket): a precomputed index map turns the flat bucket into the kernels' weight blob (K-major,
zero-padded to the kernel widths) with one gather, and the gradient blob back into the flat gradient bucket with another.
"""
import ctypes as C

import numpy as np
import torch

from . import _native as N


class _BlobMap:
    """flat parameter bucket <-> kernel weight blob.  ``pack(sd)`` is the module's own packing function (transposes, zero
    padding, constants such as the identity of 'dot' attention); running it on a state dict whose tensors hold their own
    flat indices yields the gather map, running it on zeros yields the constant part."""

    def __init__(self, module, pack, flat):
        dev = flat.device
        names = [k for k, _ in module.named_parameters()]
        params = dict(module.named_parameters())
        idx_sd, zero_sd, o = {}, {}, 0
        for k in names:
            p = params[k]
            if not p.requires_grad:
                continue
            assert p.data.data_ptr() == flat.data_ptr() + 4 * o, "parameters must be views of the flat bucket, in order"
            idx_sd[k] = (torch.arange(o, o + p.numel(), device=dev, dtype=torch.float32) + 1.0).view_as(p)
            zero_sd[k] = torch.zeros_like(p)
            o += p.numel()
        assert o == flat.numel() and o < (1 << 24)
        const = pack(zero_sd)
        where = (pack(idx_sd) - const).round().to(torch.int64)            # 0 = constant / padding, i + 1 = flat[i]
        self.const = const.contiguous()
        self.mask = (where > 0).to(torch.float32)
        self.gather = (where - 1).clamp_min(0)
        pos = torch.nonzero(where > 0).reshape(-1)
        inv = torch.empty(o, dtype=torch.int64, device=dev)
        inv[where[pos] - 1] = pos
        assert pos.numel() == o, "every parameter element must appear exactly once in the blob"
        self.inverse = inv
        self.flat = flat
        self.blob = torch.empty_like(self.const)
        self.grad = torch.zeros_like(self.const)

    def refresh(self):
        torch.index_select(self.flat, 0, self.gather, out=self.blob)
        self.blob.mul_(self.mask).add_(self.const)
        return self.blob

    def scatter_grad(self, flat_grad):
        torch.index_select(self.grad, 0, self.inverse, out=flat_grad)


class _FusedNets:
    """policy + value network of one runner family on cm_ppo_net (the subclasses set the descriptors, blob maps and batch
    layout).  ``chunk_rows``: agent rows of activations kept in the workspace at a time (the kernels walk a minibatch in
    chunks; gradients add up)."""
    _obs_keys = ("obs",)                 # per-step inputs of both networks besides the policy's avail / actions / valid

    def _setup(self, policy, critic, opt, baseline_opt, chunk_rows):
        self.policy, self.critic = policy, critic
        self.device = policy.device
        self.n, self.D = policy._n_agents, policy._dec_obs_dim
        self.pol_map = _BlobMap(policy, policy._pack_blob, opt.flat)
        self.cri_map = _BlobMap(critic, critic._pack_blob, baseline_opt.flat)
        import os
        chunk_rows = int(os.environ.get("CM_PPO_CHUNK_ROWS", chunk_rows))          # (experiments)
        self.chunk_steps = max(1, int(chunk_rows) // self.n)
        self._ws = None

    def _prepare_common(self, b):
        n, D = self.n, self.D
        P, T = b["rewards"].shape
        S = P * T
        f = dict(P=P, T=T, obs=b["obs"].reshape(S, n, D).contiguous(), actions=b["actions"].reshape(S, n).contiguous())
        av = b["avail"].reshape(S, n, 5)
        wts = torch.tensor([1, 2, 4, 8, 16], dtype=torch.float32, device=av.device)
        f["avail"] = ((av != 0).to(torch.float32) * wts).sum(-1).to(torch.uint8).contiguous()
        f["valids_host"] = b["valids"].cpu().numpy().astype(np.int64)
        f["valid"] = (torch.arange(T, device=self.device)[None, :] < b["valids"][:, None]).reshape(S).to(torch.uint8).contiguous()
        return f

    # ---- batch ---------------------------------------------------------------------------------------------------
    def step_index(self, f, path_ids, valid_only):
        """flat step indices (device int64) of the given paths: every padded step, or the valid ones only"""
        T = f["T"]
        ids = np.asarray(path_ids, dtype=np.int64)
        if valid_only:
            v = f["valids_host"][ids]
            first = np.cumsum(v) - v                                     # position of each path's first step in the output
            idx = np.repeat(ids * T - first, v) + np.arange(int(v.sum()), dtype=np.int64)
        else:
            idx = (ids[:, None] * T + np.arange(T)[None, :]).reshape(-1)
        return torch.from_numpy(idx).to(self.device)

    def subset(self, f, idx, policy=True):
        """the rows `idx` of the flat batch gathered ONCE (a minibatch is walked again in every mini-epoch): a flat batch of its
        own, to be passed to policy_call / critic_call with idx = None"""
        keys = self._obs_keys + (("avail", "actions", "valid") if policy else ())
        g = {k: f[k].index_select(0, idx) for k in keys}
        g["P"], g["T"] = 1, int(idx.numel())
        return g

    # ---- one call ------------------------------------------------------------------------------------------------
    def _workspace(self, desc, steps, backward, extra=0):
        chunk = min(max(int(steps), 1), self.chunk_steps)
        need = N.lib().cm_ppo_net_workspace_floats(C.byref(desc), chunk, int(backward)) + extra
        if self._ws is None or self._ws.numel() < need:
            self._ws = None
            self._ws = torch.empty(need, dtype=torch.float32, device=self.device)
        return self._ws

    def _run(self, desc, io):
        with torch.cuda.device(self.device):
            N.check("cm_ppo_net", N.lib().cm_ppo_net(C.byref(desc), C.byref(io), N.stream_ptr()))

    def _io(self, desc, f, idx, backward, wmap):
        sel = (lambda x: x) if idx is None else (lambda x: x.index_select(0, idx))
        keep = {k: sel(f[k]) for k in self._obs_keys}
        S = keep["obs"].shape[0]
        if backward:
            (self.pol_map if desc is self.pol_desc else self.cri_map).grad.zero_()
        io = N.NetIO()
        io.n_steps = S
        io.weights = N.ptr(wmap.blob)
        io.grad = N.ptr(wmap.grad) if backward else None
        io.obs = N.ptr(keep["obs"])
        if "adj" in keep:
            io.adj_bits, io.chan_bits = N.ptr(keep["adj"]), N.ptr(keep["chan"])
        ws = self._workspace(desc, S, backward)
        io.workspace, io.workspace_floats = N.ptr(ws), ws.numel()
        return io, keep, sel, S

    def policy_call(self, f, idx=None, adv=None, old_ll=None, backward=False, want_probs=False, inv_count=None):
        """forward (+ backward) of the policy over the steps `idx` (None = all).  Returns dict(ll, entropy, probs, loss);
        with backward=True the gradient is left in the flat gradient bucket of the policy optimizer's layout
        (``pol_map.scatter_grad``)."""
        io, keep, sel, S = self._io(self.pol_desc, f, idx, backward, self.pol_map)
        keep["avail"], keep["actions"], keep["valid"] = sel(f["avail"]), sel(f["actions"]), sel(f["valid"])
        io.avail_bits, io.actions, io.valid = N.ptr(keep["avail"]), N.ptr(keep["actions"]), N.ptr(keep["valid"])
        out = dict(ll=torch.empty(S, dtype=torch.float32, device=self.device),
                   entropy=torch.empty(S, dtype=torch.float32, device=self.device))
        io.ll, io.entropy = N.ptr(out["ll"]), N.ptr(out["entropy"])
        if want_probs:
            out["probs"] = torch.empty((S, self.n, 5), dtype=torch.float32, device=self.device)
            io.probs = N.ptr(out["probs"])
        if adv is not None:
            keep["adv"] = adv.contiguous()
            io.adv = N.ptr(keep["adv"])
            if old_ll is not None:
                keep["old"] = old_ll.contiguous()
                io.old_ll = N.ptr(keep["old"])
            loss = torch.zeros(1, dtype=torch.float32, device=self.device)
            io.loss = N.ptr(loss)
            out["loss"] = loss
            if inv_count is None:
                inv_count = 1.0 / max(float(keep["valid"].sum()), 1.0)
            io.inv_count = float(inv_count)
        if S:
            self._run(self.pol_desc, io)
        return out

    def critic_call(self, f, idx=None, returns=None, backward=False):
        """values (and, with returns, the Gaussian NLL loss; with backward=True its gradient) over the steps `idx`"""
        io, keep, sel, S = self._io(self.cri_desc, f, idx, backward, self.cri_map)
        out = dict(values=torch.empty(S, dtype=torch.float32, device=self.device))
        io.values = N.ptr(out["values"])
        if returns is not None:
            keep["ret"] = returns.contiguous()
            io.returns = N.ptr(keep["ret"])
            loss = torch.zeros(1, dtype=torch.float32, device=self.device)
            io.loss = N.ptr(loss)
            out["loss"] = loss
            io.inv_count = 1.0 / max(S, 1)
        if S:
            self._run(self.cri_desc, io)
        return out


class FusedCommNets(_FusedNets):
    """policy + critic of the Comm-DP and Obs-DP runners (CommBaseCritic) on cm_ppo_net"""
    _obs_keys = ("obs", "adj", "chan")

    def __init__(self, policy, critic, opt, baseline_opt, ent_coeff, clip_range, chunk_rows=524288):
        self._setup(policy, critic, opt, baseline_opt, chunk_rows)
        # L = layers of the communication masks in the batch (the critic's; the Obs-DP policy has none of its own)
        self.L = len(critic.gcn_layers)
        self.W = (self.n + 31) // 32
        self.dec = not getattr(policy, "comm", False)
        assert self.pol_map.const.numel() == N.lib().cm_policy_blob_floats(self.D, policy.n_gcn_layers)
        assert self.cri_map.const.numel() == N.lib().cm_critic_blob_floats(self.D, self.L)
        self.pol_desc = N.NetDesc(N.NET_POLICY_DEC if self.dec else N.NET_POLICY, self.n, self.D, policy.n_gcn_layers, int(policy.residual), float(ent_coeff),
                                  1.0 - float(clip_range), 1.0 + float(clip_range))
        self.cri_desc = N.NetDesc(N.NET_CRITIC, self.n, self.D, len(critic.gcn_layers), int(critic.residual), 0.0, 0.0, 0.0)
        if self.n > 64 and self.chunk_steps > 148:        # one env per CTA in the n x n kernels: whole waves of the 148 SMs
            self.chunk_steps = self.chunk_steps // 148 * 148

    @staticmethod
    def supports(policy, critic):
        from .policy import CommCategoricalMLPPolicy, DecCategoricalMLPPolicy
        from .ppo import CommBaseCritic
        if type(critic) is not CommBaseCritic or policy._dec_obs_dim > 128 or policy._n_agents != critic._n_agents:
            return False
        if type(policy) is DecCategoricalMLPPolicy:              # Obs-DP runners: no communication in the policy
            return True
        return type(policy) is CommCategoricalMLPPolicy and len(critic.gcn_layers) == policy.n_gcn_layers

    def prepare(self, b):
        """flat (step-major) views of a padded [P, T, ...] batch; masks as bit rows, availability as bits"""
        n, L, W = self.n, self.L, self.W
        f = self._prepare_common(b)
        S = f["P"] * f["T"]
        if "adj_bits" in b:
            f["adj"], f["chan"] = b["adj_bits"].reshape(S, n, W).contiguous(), b["chan_bits"].reshape(S, L, n, W).contiguous()
        else:
            from .policy import CommCategoricalMLPPolicy
            pack = CommCategoricalMLPPolicy.pack_mask            # (static: cm_mask_pack)
            f["adj"] = pack(b["dist_adjs"].reshape(S, n, n), n)
            f["chan"] = pack(b["channels"].reshape(S, L, n, n), n)
        return f


class FusedCentNets(_FusedNets):
    """policy + baseline of the CENT runners (CentralizedCategoricalMLPPolicy + GaussianMLPBaseline) on cm_ppo_net: both
    networks read the concatenated observation of the team, one row per env step; no communication masks"""

    def __init__(self, policy, critic, opt, baseline_opt, ent_coeff, clip_range, chunk_rows=524288):
        self._setup(policy, critic, opt, baseline_opt, chunk_rows)
        assert self.pol_map.const.numel() == N.lib().cm_policy_cent_blob_floats(self.n, self.D)
        assert self.cri_map.const.numel() == N.lib().cm_baseline_mlp_blob_floats(critic.input_dim)
        self.pol_desc = N.NetDesc(N.NET_POLICY_CENT, self.n, self.D, 0, 0, float(ent_coeff), 1.0 - float(clip_range),
                                  1.0 + float(clip_range), N.NET_FLAG_RELU if policy._relu else 0)
        self.cri_desc = N.NetDesc(N.NET_BASELINE_MLP, self.n, self.D, 0, 0, 0.0, 0.0, 0.0, 0)

    @staticmethod
    def supports(policy, critic):
        from .policy import CentralizedCategoricalMLPPolicy
        from .ppo import GaussianMLPBaseline
        return (type(policy) is CentralizedCategoricalMLPPolicy and type(critic) is GaussianMLPBaseline and critic._fusable
                and policy._dec_obs_dim <= 128 and policy._n_agents <= N.MAX_AGENTS and critic.input_dim == policy._obs_dim
                and policy._obs_dim == policy._n_agents * policy._dec_obs_dim)

    def prepare(self, b):
        """flat (step-major) views of a padded [P, T, ...] batch, availability as bits (no masks)"""
        return self._prepare_common(b)


class _SetBlobMap:
    """K members' flat parameter rows ``flat [K][n]`` <-> K kernel blobs ``blob [K][stride]`` (stride = blob length rounded up to
    4 floats, the row alignment cm_ppo_net asks of a set): the gather / inverse maps of ONE member (``_BlobMap``) with a row
    offset per member, so that each direction is one index_select for all members.  Member i's single-network blob and
    gradient are ``blob[i, :nb]`` / ``grad[i, :nb]``."""

    def __init__(self, one, flat):
        K, n = flat.shape
        dev = flat.device
        self.nb = nb = one.const.numel()
        self.stride = stride = (nb + 3) // 4 * 4
        pad = lambda t: torch.cat([t, torch.zeros(stride - nb, dtype=t.dtype, device=dev)])  # noqa: E731
        rows = torch.arange(K, device=dev, dtype=torch.int64)[:, None]
        self.const, self.mask = pad(one.const)[None, :].contiguous(), pad(one.mask)[None, :].contiguous()
        self.gather = (pad(one.gather)[None, :] + rows * n).reshape(-1)
        self.inverse = (one.inverse[None, :] + rows * stride).reshape(-1)
        self.flat = flat
        self.blob = torch.zeros((K, stride), dtype=torch.float32, device=dev)
        self.grad = torch.zeros((K, stride), dtype=torch.float32, device=dev)

    def refresh(self):
        torch.index_select(self.flat.reshape(-1), 0, self.gather, out=self.blob.view(-1))
        self.blob.mul_(self.mask).add_(self.const)
        return self.blob

    def scatter_grad(self, flat_grad):
        """the gradient blobs -> flat_grad [K][n] (contiguous)"""
        torch.index_select(self.grad.view(-1), 0, self.inverse, out=flat_grad.view(-1))
