"""PPO update on the device (SURVEY.md §8f.1) — the trainer side of the rollout engine.

Mirrors, with the reference's semantics and hyper-parameter names:
  * ``CommBaseCritic``            — com_marl/torch/baselines/comm_base_critic.py:11-120 (CommBaseNet trunk + a
                                    GaussianMLPModule aggregator, ``aggregator_type='sum'``), same ``state_dict`` names;
  * ``DevicePPO.process_samples`` — CentralizedMAPPO.process_samples (centralized_ma_ppo.py:612-659): paths padded to
                                    ``[P, Tmax, ...]`` (zeros; ones for avail / dist_adj / channels), critic baselines;
  * ``DevicePPO.compute_loss``    — _compute_loss / _compute_objective (:390-438, 540-589): clipped surrogate with the
                                    HARD-CODED clip range 0.1 (:121), entropy regularisation, mean over the valid steps;
  * ``DevicePPO.train_once``      — the optimisation loop of train_once (:207-262): path ids shuffled once, cut into
                                    ``optimization_n_minibatches`` slices, ``optimization_mini_epochs`` passes, critic loss,
                                    clip_grad_norm_ on the policy, both Adam steps.
Returns, GAE advantages and their per-path normalisation run in ``cm_ppo_advantages`` and both Adam steps in
``cm_adam_step`` (hand-written CUDA over flat parameter buckets, csrc/ppo_kernels.cu).  The network forward / backward of the
Comm-DP and Obs-DP runner families (CommBaseCritic with a CommCategoricalMLPPolicy or a DecCategoricalMLPPolicy) runs on the
hand-written kernels of csrc/ppo_net_kernels.cu (``cm_ppo_net`` through ppo_fused.FusedCommNets, ``fused='auto'``); the CENT
family (CentralizedCategoricalMLPPolicy + GaussianMLPBaseline) runs on them with ``fused=True`` (ppo_fused.FusedCentNets) and on
torch autograd otherwise; ``fused=False`` (the kernels' cross-check) uses torch autograd over the policies' differentiable ``forward``.  With
more than one rank the flat gradient buckets are all-reduced (NCCL) before clipping — the only collective of the update
(SURVEY.md §8e).
"""
import ctypes as C

import numpy as np
import torch
import torch.distributed as dist
from torch import nn

from . import _native as N
from .policy import _Attention, _GraphConv, _MLP, _pad2


class _GaussianHead(nn.Module):
    """GaussianMLPModule(input_dim, 1, hidden_sizes, share_std=True) (gaussian_mlp_module.py:64-170): mean MLP +
    one learnable log-std, clamped at log(1e-6)."""

    def __init__(self, input_dim, hidden_sizes):
        super().__init__()
        self._init_std = nn.Parameter(torch.zeros(1))                      # log(init_std = 1)
        self._mean_module = _MLP(input_dim, hidden_sizes, 1, output_tanh=False)

    def forward(self, x):
        mean = self._mean_module(x)
        std = self._init_std.clamp(min=float(np.log(np.float32(1e-6)))).exp()
        return mean, std


class CommBaseCritic(nn.Module):
    """Centralised value baseline V(s) = sum_i f(E_i + H_L,i) with the policy's comm-GNN trunk."""

    def __init__(self, env_spec, n_agents, encoder_hidden_sizes=(128,), embedding_dim=64, decoder_hidden_sizes=(64,),
                 attention_type="general", n_gcn_layers=2, residual=True, gcn_bias=True, aggregator_type="sum",
                 name="base_critic", device="cuda"):
        super().__init__()
        if attention_type not in ("general", "dot") or aggregator_type != "sum":
            raise NotImplementedError("attention_type 'general' / 'dot' and aggregator_type='sum' (the runners' setting) only")
        self.name, self.device = name, torch.device(device)
        self._n_agents, self.residual, self.eps = int(n_agents), bool(residual), 1e-12
        self._dec_obs_dim = int(env_spec.observation_space.flat_dim / n_agents)
        self.encoder = _MLP(self._dec_obs_dim, tuple(encoder_hidden_sizes), embedding_dim, output_tanh=True)
        self.attention_layer = _Attention(embedding_dim, attention_type)
        self.gcn_layers = nn.ModuleList([_GraphConv(embedding_dim, gcn_bias) for _ in range(int(n_gcn_layers))])
        self.baseline_aggregator = _GaussianHead(embedding_dim, tuple(decoder_hidden_sizes))
        self._embedding_dim = int(embedding_dim)
        enc, dec = tuple(encoder_hidden_sizes), tuple(decoder_hidden_sizes)
        # shapes the hand-written update kernels hold (narrower layers run exactly, zero-padded)
        self._fusable = len(enc) == 1 and enc[0] <= 128 and embedding_dim <= 64 and len(dec) == 1 and dec[0] <= 64
        self.to(self.device)

    def _pack_blob(self, sd):
        """state dict -> the critic blob of cm_ppo_net (include/commarl_b200.h): the trunk like the policy blob, then
        dec_w1 [64][64] dec_b1 [64] dec_w2 [64] dec_b2 [1] log_std [1]"""
        E, dev = self._embedding_dim, self.device
        att = sd["attention_layer.linear_in.weight"].t() if "attention_layer.linear_in.weight" in sd else torch.eye(E, device=dev)
        parts = [_pad2(sd["encoder._layers.0.linear.weight"].t(), self._dec_obs_dim, 128), _pad2(sd["encoder._layers.0.linear.bias"], 128, 0),
                 _pad2(sd["encoder._output_layers.0.linear.weight"].t(), 128, 64), _pad2(sd["encoder._output_layers.0.linear.bias"], 64, 0),
                 _pad2(att, 64, 64)]
        L = len(self.gcn_layers)
        parts += [_pad2(sd[f"gcn_layers.{l}.weight"], 64, 64) for l in range(L)]
        parts += [_pad2(sd.get(f"gcn_layers.{l}.bias", torch.zeros(E, device=dev)), 64, 0) for l in range(L)]
        m = "baseline_aggregator._mean_module."
        parts += [_pad2(sd[m + "_layers.0.linear.weight"].t(), 64, 64), _pad2(sd[m + "_layers.0.linear.bias"], 64, 0),
                  _pad2(sd[m + "_output_layers.0.linear.weight"].t(), 64, 1), sd[m + "_output_layers.0.linear.bias"],
                  sd["baseline_aggregator._init_std"]]
        return torch.cat([p.detach().to(dev, torch.float32).contiguous().reshape(-1) for p in parts])

    def _values(self, obs_n, dist_adj, channels):
        n = self._n_agents
        obs_n = obs_n.reshape(obs_n.shape[:-1] + (n, -1))
        channels = channels.reshape(channels.shape[:-2] + (len(self.gcn_layers), n, n))
        if dist_adj.shape[-2:] != torch.Size((n, n)):
            dist_adj = dist_adj.reshape(dist_adj.shape[:-1] + (n, n))
        E = self.encoder(obs_n)
        M = self.attention_layer(E)
        H = E
        for l, gcn in enumerate(self.gcn_layers):                      # comm_base_net.py:99-104
            A = M * dist_adj * channels[..., l, :, :]
            A = A / (A.sum(dim=-1, keepdim=True) + self.eps)
            H = gcn(H, A)
        X = E + H if self.residual else H
        mean, std = self.baseline_aggregator(X)
        return mean.squeeze(-1).sum(-1), std.mean()

    def forward(self, obs_n, avail_actions_n, dist_adj, channels, get_actions=False):
        return self._values(obs_n, dist_adj, channels)[0]

    def compute_loss(self, obs_n, returns, dist_adj, channels, get_actions=False):
        mean, std = self._values(obs_n, dist_adj, channels)           # -Normal(mean, std).log_prob(returns).mean()
        return (0.5 * ((returns - mean) / std) ** 2 + std.log() + 0.5 * float(np.log(2 * np.pi))).mean()


class _GaussianMean(nn.Module):
    """parameter layout of garage's GaussianMLPModule (garage/torch/modules/gaussian_mlp_module.py:118-127,260-271):
    ``_init_std`` = log(init_std), ``_mean_module`` = MLPModule"""

    def __init__(self, input_dim, hidden_sizes, init_std):
        super().__init__()
        self._init_std = nn.Parameter(torch.tensor([float(init_std)]).log())
        self._mean_module = _MLP(input_dim, tuple(hidden_sizes), 1, output_tanh=False)


class GaussianMLPBaseline(nn.Module):
    """Value baseline of the Obs-DP and CENT runners (com_marl/torch/baselines/gaussian_mlp_baseline.py:7-117, built with
    hidden_sizes=(64, 64, 64) at runner_*_cent.py:60-62): V(s) = MLP(concatenated observation), fitted as the mean of a
    Gaussian with one learnt log-std (GaussianMLPModule, std_parameterization='exp', no clamps).  Same ``state_dict`` names
    (``module._init_std``, ``module._mean_module._layers.i.linear.*``): reference baselines load unchanged."""

    def __init__(self, env_spec, hidden_sizes=(32, 32), init_std=1.0, name="GaussianMLPBaseline", device="cuda"):
        super().__init__()
        self.name, self.device = name, torch.device(device)
        self.input_dim = int(env_spec.observation_space.flat_dim)
        self.module = _GaussianMean(self.input_dim, hidden_sizes, init_std)
        # the shape the hand-written update kernels hold (the runners' (64, 64, 64); narrower layers run exactly, zero-padded)
        self._fusable = len(tuple(hidden_sizes)) == 3 and max(hidden_sizes) <= 64
        self.to(self.device)

    def _pack_blob(self, sd):
        """state dict -> the blob of cm_ppo_net's CM_NET_BASELINE_MLP (include/commarl_b200.h): w1 [K][64] b1 w2 [64][64] b2
        w3 [64][64] b3 w4 [64] b4 [1] log_std [1], dense weights K-major, narrower layers zero-padded"""
        m = "module._mean_module."
        parts = []
        for i, k_in in enumerate((self.input_dim, 64, 64)):
            parts += [_pad2(sd[m + f"_layers.{i}.linear.weight"].t(), k_in, 64), _pad2(sd[m + f"_layers.{i}.linear.bias"], 64, 0)]
        parts += [_pad2(sd[m + "_output_layers.0.linear.weight"].t(), 64, 1), sd[m + "_output_layers.0.linear.bias"], sd["module._init_std"]]
        return torch.cat([p.detach().to(self.device, torch.float32).contiguous().reshape(-1) for p in parts])

    def forward(self, obs):
        """(P, T, O) -> (P, T) predicted values (:104-117)"""
        return self.module._mean_module(obs).flatten(-2)

    def compute_loss(self, obs, returns):
        """-mean log N(returns; V(obs), exp(log_std)) over every step of the padded batch (:83-101)"""
        mean = self.module._mean_module(obs.reshape(-1, self.input_dim))
        std = self.module._init_std.exp().expand_as(mean)
        return -torch.distributions.Normal(mean, std).log_prob(returns.reshape(-1, 1)).sum(-1).mean()


class FlatAdam:
    """The reference's Adam (my_optimizer/adam.py) over ONE flat fp32 bucket: parameters and gradients of the module are
    re-seated as views of two flat tensors, so that the gradient all-reduce is one NCCL call, the gradient norm one
    reduction and the optimizer step one kernel (cm_adam_step).

    Every element of the bucket is stepped, also those of a parameter that received no gradient in this backward pass (its
    slice of the zeroed bucket stays 0).  The reference's Adam skips parameters whose ``grad is None`` (com_marl/torch/algos/my_optimizer/adam.py:79-80).  The two
    agree as long as a parameter either always or never receives a gradient: with moments that are still zero a zero gradient
    moves nothing (0 / (0 + eps)), and that is the case for every network of the three runner families (a parameter outside the
    loss's graph — e.g. the attention weights of a policy run without communication — never gets one)."""

    def __init__(self, module, lr=3e-4, betas=(0.9, 0.999), eps=1e-5):
        self.params = [p for p in module.parameters() if p.requires_grad]
        dev = self.params[0].device
        n = sum(p.numel() for p in self.params)
        self.flat = torch.empty(n, dtype=torch.float32, device=dev)
        # gradient bucket + ONE extra slot that carries this rank's sample weight through the same all-reduce
        self._bucket = torch.zeros(n + 1, dtype=torch.float32, device=dev)
        self.grad = self._bucket[:n]
        o = 0
        for p in self.params:
            k = p.numel()
            self.flat[o:o + k].copy_(p.data.reshape(-1))
            p.data = self.flat[o:o + k].view_as(p)
            p.grad = self.grad[o:o + k].view_as(p)
            o += k
        self.exp_avg, self.exp_avg_sq = torch.zeros_like(self.flat), torch.zeros_like(self.flat)
        self.lr, self.betas, self.eps, self.steps = float(lr), betas, float(eps), 0

    def zero_grad(self):
        self._bucket.zero_()

    def all_reduce(self, group=None, weight=1.0):
        """Data-parallel gradient of the UNION minibatch: every rank's gradient is the gradient of a mean over its own
        `weight` samples (valid steps for the policy loss, batch elements for the baseline loss), so the union's gradient is
        sum_r w_r g_r / sum_r w_r.  The weight travels in the bucket's extra slot: one collective per optimizer step.  A rank
        whose slice is empty (weight 0, zero gradient) still takes part — the collective count is rank-invariant."""
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            w = float(weight)
            self.grad.mul_(w)
            self._bucket[-1] = w
            dist.all_reduce(self._bucket, group=group)
            self.grad.div_(self._bucket[-1].clamp_min(1e-30))

    def clip_coefficient(self, max_norm):
        """torch.nn.utils.clip_grad_norm_: min(1, max_norm / (||g|| + 1e-6)); returns (coefficient, norm) as 0-d tensors"""
        norm = self.grad.norm(2)
        return torch.clamp(max_norm / (norm + 1e-6), max=1.0), norm

    def step(self, grad_scale=1.0):
        """grad_scale: a float, or a 0-d / 1-element float32 DEVICE tensor (the clip coefficient as computed on the device:
        no host synchronisation between the backward pass and the step)"""
        self.steps += 1
        with torch.cuda.device(self.flat.device):
            if isinstance(grad_scale, torch.Tensor):
                self._scale = grad_scale.detach().to(torch.float32).reshape(1).contiguous()      # (kept alive until the next step)
                N.check("cm_adam_step_dev", N.lib().cm_adam_step_dev(N.ptr(self.flat), N.ptr(self.grad), N.ptr(self.exp_avg),
                                                                     N.ptr(self.exp_avg_sq), self.flat.numel(), self.lr, self.betas[0],
                                                                     self.betas[1], self.eps, self.steps, N.ptr(self._scale),
                                                                     N.stream_ptr()))
            else:
                N.check("cm_adam_step", N.lib().cm_adam_step(N.ptr(self.flat), N.ptr(self.grad), N.ptr(self.exp_avg), N.ptr(self.exp_avg_sq),
                                                             self.flat.numel(), self.lr, self.betas[0], self.betas[1], self.eps, self.steps,
                                                             float(grad_scale), N.stream_ptr()))
        for p in self.params:                 # the kernel wrote the parameters behind autograd's back: bump the version
            torch.autograd.graph.increment_version(p)      # counters, so that the policy rebuilds its kernel weight blobs


def _unpack_mask(bits, n):
    """int32 bit rows (..., n, W) -> dense float32 (..., n, n) (cm_mask_unpack)"""
    bits = bits.contiguous()
    rows = bits.numel() // bits.shape[-1]
    out = torch.empty(bits.shape[:-1] + (n,), dtype=torch.float32, device=bits.device)
    with torch.cuda.device(bits.device):
        N.check("cm_mask_unpack", N.lib().cm_mask_unpack(N.ptr(bits), N.ptr(out), rows, n, N.stream_ptr()))
    return out


def ppo_advantages(rewards, baselines, valids, discount, gae_lambda, center=True, eps=1e-8):
    """(returns, raw_adv, adv) float32 [P, T] from float64 rewards, float32 baselines [P, T] and int32 valids [P]"""
    P, T = rewards.shape
    rewards = rewards.to(torch.float64).contiguous()
    baselines = baselines.to(torch.float32).contiguous()
    valids = valids.to(torch.int32).contiguous()
    out = [torch.empty((P, T), dtype=torch.float32, device=rewards.device) for _ in range(3)]
    with torch.cuda.device(rewards.device):
        N.check("cm_ppo_advantages", N.lib().cm_ppo_advantages(N.ptr(rewards), N.ptr(baselines), N.ptr(valids), P, T, float(discount),
                                                               float(gae_lambda), int(bool(center)), float(eps), N.ptr(out[0]),
                                                               N.ptr(out[1]), N.ptr(out[2]), N.stream_ptr()))
    return out


def _world(group=None):
    return dist.get_world_size(group) if (dist.is_available() and dist.is_initialized()) else 1


def global_max(value, device, group=None):
    """max over ranks of a non-negative integer (no-op without a process group)"""
    if _world(group) == 1:
        return int(value)
    t = torch.tensor([int(value)], dtype=torch.int64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return int(t.item())


def minibatch_plan(P, n_minibatches, device="cpu", group=None):
    """[(start, stop)] slices of the shuffled path ids, one per optimizer step of a mini-epoch.  A single process cuts exactly
    like the reference (centralized_ma_ppo.py:236-241: step = ceil(P / n_minibatches), range(0, P, step)).  With several ranks
    the local path counts differ, and so would the slice counts (P = 4 gives 2 slices, P = 5 gives 3): every optimizer step
    issues collectives, so the count must not depend on the rank — it is the maximum over ranks, and a rank that has run out of
    paths appends EMPTY slices (zero gradient, weight 0) and still takes part in the all-reduces."""
    P = int(P)
    step = int(np.ceil(P / n_minibatches)) if P > 0 else 1
    plan = [(s0, min(s0 + step, P)) for s0 in range(0, P, step)]
    n_it = global_max(len(plan), device, group)
    return plan + [(P, P)] * (n_it - len(plan))


class DevicePPO:
    """CentralizedMAPPO's update (centralized_ma_ppo.py) on one GPU per rank, for the three runner families: a Comm-DP or Obs-DP
    policy with CommBaseCritic (runner_*_comm.py, runner_*_obsDP.py:61), or a CENT policy with GaussianMLPBaseline.  Like the reference, the policy call takes the
    communication masks iff the policy has them (`hasattr(policy, 'comm')`, :455-490) and the baseline call iff it is the
    'base_critic' (:229-232, :653-657)."""

    def __init__(self, policy, baseline, discount=0.99, gae_lambda=0.97, center_adv=True, positive_adv=False,
                 policy_ent_coeff=0.1, entropy_method="regularized", clip_grad_norm=7, optimization_n_minibatches=3,
                 optimization_mini_epochs=10, policy_lr=3e-4, adam_eps=1e-5, process_group=None, fused="auto"):
        if entropy_method not in ("regularized", "no_entropy"):
            raise NotImplementedError("entropy_method 'max' (entropy added to the rewards) is not implemented")
        if entropy_method == "no_entropy" and policy_ent_coeff != 0.0:
            raise ValueError("policy_ent_coeff should be zero when there is no entropy method")
        self.policy, self.baseline, self.device = policy, baseline, policy.device
        self._comm = bool(getattr(policy, "comm", False))
        self._critic_comm = getattr(baseline, "name", "") == "base_critic"
        self.discount, self.gae_lambda = float(discount), float(gae_lambda)
        self.center_adv, self.positive_adv = bool(center_adv), bool(positive_adv)
        self.ent_coeff = float(policy_ent_coeff) if entropy_method == "regularized" else 0.0
        self.lr_clip_range = 0.1                      # centralized_ma_ppo.py:121 overrides the constructor argument
        self.adv_eps = 1e-8                           # :122
        self.clip_grad_norm = clip_grad_norm
        self.n_minibatches, self.mini_epochs = int(optimization_n_minibatches), int(optimization_mini_epochs)
        self.group = process_group
        self.opt = FlatAdam(policy, lr=policy_lr, eps=adam_eps)
        self.baseline_opt = FlatAdam(baseline, lr=policy_lr, eps=adam_eps)
        # fused = hand-written forward / backward kernels (cm_ppo_net) instead of torch autograd: the Comm-DP and Obs-DP
        # families (with CommBaseCritic) and the CENT family (with GaussianMLPBaseline).  'auto' = the Comm-DP / Obs-DP kernels
        # wherever they apply; CENT stays on autograd unless fused=True: its kernels are new and opt-in, and whether the default
        # follows is decided on their measured update times against autograd (DESIGN.md §7.1 and §8 item 1,
        # profiles/r03a_ppo_cent.jsonl)
        from .ppo_fused import FusedCentNets, FusedCommNets
        cuda = self.device.type == "cuda"
        can_comm = cuda and FusedCommNets.supports(policy, baseline) and getattr(baseline, "_fusable", False)
        can_cent = cuda and FusedCentNets.supports(policy, baseline)
        if fused is True and not (can_comm or can_cent):
            raise NotImplementedError("fused=True needs, of the kernels' shapes and on a GPU, a CommCategoricalMLPPolicy or "
                                      "DecCategoricalMLPPolicy with a CommBaseCritic, or a CentralizedCategoricalMLPPolicy with a "
                                      "GaussianMLPBaseline")
        self._fused = None
        if can_comm and fused in (True, "auto"):
            self._fused = FusedCommNets(policy, baseline, self.opt, self.baseline_opt, self.ent_coeff, self.lr_clip_range)
        elif can_cent and fused is True:
            self._fused = FusedCentNets(policy, baseline, self.opt, self.baseline_opt, self.ent_coeff, self.lr_clip_range)

    # ---- process_samples ----------------------------------------------------------------------------------------
    def process_samples(self, paths):
        """paths: the sampler's list of dicts (…vectorized_sampler.py:192-224).  Returns a dict of device tensors padded to
        the longest path like the reference, plus baselines / returns / advantages."""
        dev, n = self.device, self.policy._n_agents
        P, Tmax = len(paths), global_max(max(len(p["rewards"]) for p in paths), dev, self.group)

        def pad(key, dtype, fill):
            first = np.asarray(paths[0][key])
            out = np.full((P, Tmax) + first.shape[1:], fill, dtype=dtype)
            for i, p in enumerate(paths):
                a = np.asarray(p[key])
                out[i, :len(a)] = a
            return torch.from_numpy(out).to(dev)

        b = dict(obs=pad("observations", np.float32, 0), avail=pad("avail_actions", np.float32, 1),
                 actions=pad("actions", np.int64, 0), rewards=pad("rewards", np.float64, 0),
                 dist_adjs=pad("dist_adjs", np.float32, 1), channels=pad("channels", np.float32, 1),
                 valids=torch.tensor([len(p["rewards"]) for p in paths], dtype=torch.int32, device=dev))
        return self.finish_batch(b)

    def batch_from_trajectory(self, traj, K=None):
        """The same padded batch straight from the rollout engine's device trajectory (``RolloutEngine.traj``: time-major
        slots ``obs [K+1,B,n,D]``, ``actions [K,B,n]``, ``reward [K,B]``, ``done [K,B]``, bit-row masks) without the host
        `paths` list: every episode that FINISHED inside the K recorded steps becomes one row (the reference's sampler
        only appends finished paths too, …vectorized_sampler.py:189-226), ordered env-major then by time."""
        dev, n = self.device, self.policy._n_agents
        done = traj["done"] if K is None else traj["done"][:K]
        K, B = done.shape
        done = done.to(torch.int64)
        nth = done.cumsum(0) - done                          # episodes finished before step k in env b = index of k's episode
        fin = done.sum(0)                                    # finished episodes per env
        P = int(fin.sum())
        if global_max(P, dev, self.group) == 0:              # (collective: a single rank must not bail out alone)
            raise ValueError("no episode finished inside the recorded trajectory")
        valid = nth < fin[None, :]                           # step belongs to an episode that finishes inside the window
        off = fin.cumsum(0) - fin                            # first path id of env b
        pid = off[None, :] + nth                             # [K, B] path id of every step
        ks = torch.arange(K, device=dev)[:, None].expand(K, B)
        # step inside its episode: k - (1 + the last step before k at which env b reported done)
        last_done = torch.where(done.bool(), ks, torch.full_like(ks, -1)).cummax(0).values
        prev_done = torch.cat([torch.full((1, B), -1, dtype=torch.int64, device=dev), last_done[:-1]], 0)
        t_in = ks - (prev_done + 1)
        ends = done.bool() & valid
        valids = torch.zeros(P, dtype=torch.int64, device=dev)
        valids.index_put_((pid[ends],), t_in[ends] + 1)
        # every rank pads to the job-wide longest path: the baseline loss is a mean over the PADDED batch like the
        # reference's, so the union batch of all ranks is only reproduced when the padding agrees
        Tmax = global_max(int(valids.max()) if P else 0, dev, self.group)
        src = torch.full((P * Tmax,), -1, dtype=torch.int64, device=dev)
        flat = (ks * B + torch.arange(B, device=dev)[None, :])
        src.index_put_(((pid * Tmax + t_in)[valid],), flat[valid])
        pad = src < 0
        g = src.clamp(min=0)

        def take(x, fill):
            y = x[:K].reshape((K * B,) + x.shape[2:]).index_select(0, g)
            y[pad] = fill
            return y.reshape((P, Tmax) + x.shape[2:])

        L = traj["chan_bits"].shape[2]
        adj_bits = traj["adj_bits"][:K].reshape(K * B, n, -1).index_select(0, g)
        chan_bits = traj["chan_bits"][:K].reshape(K * B, L, n, -1).index_select(0, g)
        b = dict(obs=take(traj["obs"], 0.0).reshape(P, Tmax, -1), actions=take(traj["actions"], 0).to(torch.int64),
                 rewards=take(traj["reward"], 0.0), valids=valids.to(torch.int32),
                 avail=torch.ones((P, Tmax, n * 5), dtype=torch.float32, device=dev))
        if self._fused is not None:          # the update kernels read the bit rows: no dense (P, T, n, n) masks at all
            adj_bits[pad] = -1
            chan_bits[pad] = -1
            b["adj_bits"], b["chan_bits"] = adj_bits.reshape(P, Tmax, n, -1), chan_bits.reshape(P, Tmax, L, n, -1)
        else:
            adj, chan = _unpack_mask(adj_bits, n), _unpack_mask(chan_bits, n)
            adj[pad] = 1.0
            chan[pad] = 1.0
            b["dist_adjs"], b["channels"] = adj.reshape(P, Tmax, n * n), chan.reshape(P, Tmax, L * n, n)
        return self.finish_batch(b)

    def finish_batch(self, b):
        """baselines (critic, no grad), returns and advantages for a padded device batch with the keys of process_samples"""
        with torch.no_grad():
            if self._fused is not None:
                self._fused.cri_map.refresh()
                b["_flat"] = self._fused.prepare(b)
                b["baselines"] = self._fused.critic_call(b["_flat"])["values"].reshape(b["rewards"].shape)
            elif self._critic_comm:
                b["baselines"] = self.baseline.forward(b["obs"], b["avail"], b["dist_adjs"], b["channels"]).float()
            else:
                b["baselines"] = self.baseline.forward(b["obs"]).float()
        b["returns"], b["raw_adv"], b["adv"] = ppo_advantages(b["rewards"], b["baselines"], b["valids"], self.discount,
                                                              self.gae_lambda, self.center_adv, self.adv_eps)
        T = b["rewards"].shape[1]
        b["mask"] = torch.arange(T, device=self.device)[None, :] < b["valids"][:, None]
        return b

    # ---- losses ----------------------------------------------------------------------------------------------------
    def _dist(self, b, ids):
        sel = (lambda x: x) if ids is None else (lambda x: x[ids])
        if not self._comm:
            return self.policy.forward(sel(b["obs"]), sel(b["avail"]))
        d, _ = self.policy.forward(sel(b["obs"]), sel(b["avail"]), sel(b["dist_adjs"]), sel(b["channels"]))
        return d

    def compute_loss(self, b, ids=None, old_ll=None):
        sel = (lambda x: x) if ids is None else (lambda x: x[ids])
        d = self._dist(b, ids)
        new_ll = d.log_prob(sel(b["actions"])).sum(-1)
        ent = d.entropy().mean(-1)
        old = new_ll.detach() if old_ll is None else sel(old_ll)
        adv = sel(b["adv"])
        if self.positive_adv:
            adv = adv - adv.min()
        ratio = (new_ll - old).exp()
        obj = torch.min(ratio * adv, torch.clamp(ratio, 1 - self.lr_clip_range, 1 + self.lr_clip_range) * adv)
        if self.ent_coeff:
            obj = obj + self.ent_coeff * ent
        return -obj[sel(b["mask"])].mean()

    def kl(self, b, old_probs):
        new = self._dist(b, None).probs
        t = old_probs * (old_probs.clamp_min(1e-38).log() - new.clamp_min(1e-38).log())
        return torch.where(old_probs > 0, t, torch.zeros_like(t)).sum(-1).mean()

    # ---- train_once ------------------------------------------------------------------------------------------------
    def train_once(self, paths=None, batch=None, shuffled_ids=None):
        """One policy-optimisation round.  ``paths`` (sampler output) or an already padded device ``batch``.
        ``shuffled_ids``: the path permutation (np.random.permutation in the reference)."""
        b = self.process_samples(paths) if batch is None else batch
        if self._fused is not None:
            return self._train_once_fused(b, shuffled_ids)
        P = b["rewards"].shape[0]
        with torch.no_grad():
            d0 = self._dist(b, None)
            old_probs = d0.probs
            old_ll = d0.log_prob(b["actions"]).sum(-1)              # the frozen old policy (:204) evaluated once
            loss_before = float(self.compute_loss(b, None, old_ll))
        ids_all = np.random.permutation(P) if shuffled_ids is None else np.asarray(shuffled_ids)
        plan = minibatch_plan(P, self.n_minibatches, self.device, self.group)
        T = int(b["rewards"].shape[1])
        losses, bl_losses, gnorms = [], [], []
        for _ in range(self.mini_epochs):
            for start, stop in plan:
                self.baseline_opt.zero_grad()
                self.opt.zero_grad()
                w_pol = w_bl = 0.0
                loss = bl = None
                if stop > start:
                    ids = torch.as_tensor(ids_all[start:stop], device=self.device)
                    if self._critic_comm:
                        bl = self.baseline.compute_loss(b["obs"][ids], b["returns"][ids], b["dist_adjs"][ids], b["channels"][ids])
                    else:
                        bl = self.baseline.compute_loss(b["obs"][ids], b["returns"][ids])
                    bl.backward()
                    loss = self.compute_loss(b, ids, old_ll)
                    loss.backward()
                    if _world(self.group) > 1:
                        w_pol, w_bl = float(b["mask"][ids].sum()), float((stop - start) * T)
                self.opt.all_reduce(self.group, w_pol)
                self.baseline_opt.all_reduce(self.group, w_bl)
                scale = 1.0
                if self.clip_grad_norm is not None:
                    coef, norm = self.opt.clip_coefficient(self.clip_grad_norm)
                    scale = float(coef)
                    gnorms.append(float(norm) * scale)             # policy.grad_norm() after clipping (:254-255)
                self.opt.step(scale)
                self.baseline_opt.step(1.0)
                losses.append(float(loss.detach()) if loss is not None else float("nan"))
                bl_losses.append(float(bl.detach()) if bl is not None else float("nan"))
        with torch.no_grad():
            loss_after = float(self.compute_loss(b, None, old_ll))
            kl = float(self.kl(b, old_probs))
            d1 = self._dist(b, None)
            entropy = float(d1.entropy().mean(-1).mean())
        return dict(loss_before=loss_before, loss_after=loss_after, kl=kl, entropy=entropy, losses=losses,
                    baseline_losses=bl_losses, grad_norms=gnorms, n_paths=P)

    def _train_once_fused(self, b, shuffled_ids=None):
        """train_once on the hand-written kernels (ppo_fused.FusedCommNets / FusedCentNets): the same loop, losses, clipping, all-reduces and
        Adam steps; every network forward / backward is ONE cm_ppo_net call."""
        F = self._fused
        f = b.get("_flat") or F.prepare(b)
        P, T = b["rewards"].shape
        raw_adv, ret_all = b["adv"].reshape(-1), b["returns"].reshape(-1)
        adv_all = raw_adv - raw_adv.min() if self.positive_adv else raw_adv
        n_valid_all = max(int(f["valids_host"].sum()), 1)
        with torch.no_grad():
            F.pol_map.refresh()
            F.cri_map.refresh()
            # ONE forward of the frozen old policy (:204) gives old_ll, old_probs and LossBefore: against itself the ratio is 1
            # (the kernel takes old_ll = NULL as "the new log-likelihood, detached"), the surrogate is the advantage
            old = F.policy_call(f, None, adv=adv_all, want_probs=True, inv_count=1.0 / n_valid_all)
            old_ll, old_probs, loss_before = old["ll"], old["probs"], old["loss"]
            ids_all = np.random.permutation(P) if shuffled_ids is None else np.asarray(shuffled_ids)
            plan = minibatch_plan(P, self.n_minibatches, self.device, self.group)
            losses, bl_losses, gnorms = [], [], []
            nan = torch.full((1,), float("nan"), device=self.device)
            # the minibatches are the same in every mini-epoch: their rows are gathered once, before the loop (no index upload,
            # no gather and no host synchronisation inside it)
            mbs = []
            for start, stop in plan:
                if stop <= start:
                    mbs.append(None)
                    continue
                ids = ids_all[start:stop]
                idx_all = F.step_index(f, ids, valid_only=False)
                idx = F.step_index(f, ids, valid_only=True)
                adv = raw_adv.index_select(0, idx)
                if self.positive_adv:             # shifted by the minimum over the minibatch's padded rows (centralized_ma_ppo.py:428-429)
                    adv = adv - raw_adv.index_select(0, idx_all).min()
                mbs.append(dict(cri=F.subset(f, idx_all, policy=False), ret=ret_all.index_select(0, idx_all), pol=F.subset(f, idx),
                                adv=adv, old=old_ll.index_select(0, idx), n_valid=int(idx.numel()), n_all=int(idx_all.numel())))
            for _ in range(self.mini_epochs):
                for mb in mbs:
                    self.baseline_opt.zero_grad()
                    self.opt.zero_grad()
                    w_pol = w_bl = 0.0
                    loss = bl = nan
                    if mb is not None:
                        bl = F.critic_call(mb["cri"], None, returns=mb["ret"], backward=True)["loss"]
                        F.cri_map.scatter_grad(self.baseline_opt.grad)
                        loss = F.policy_call(mb["pol"], None, adv=mb["adv"], old_ll=mb["old"], backward=True,
                                             inv_count=1.0 / max(mb["n_valid"], 1))["loss"]
                        F.pol_map.scatter_grad(self.opt.grad)
                        w_pol, w_bl = float(mb["n_valid"]), float(mb["n_all"])
                    self.opt.all_reduce(self.group, w_pol)
                    self.baseline_opt.all_reduce(self.group, w_bl)
                    scale = 1.0
                    if self.clip_grad_norm is not None:
                        coef, norm = self.opt.clip_coefficient(self.clip_grad_norm)
                        scale = coef                            # stays on the device (cm_adam_step_dev): no host round trip per step
                        gnorms.append(norm * coef)
                    self.opt.step(scale)
                    self.baseline_opt.step(1.0)
                    F.pol_map.refresh()
                    F.cri_map.refresh()
                    losses.append(loss)
                    bl_losses.append(bl)
            after = F.policy_call(f, None, adv=adv_all, old_ll=old_ll, want_probs=True, inv_count=1.0 / n_valid_all)
            new = after["probs"]
            t = old_probs * (old_probs.clamp_min(1e-38).log() - new.clamp_min(1e-38).log())
            kl = float(torch.where(old_probs > 0, t, torch.zeros_like(t)).sum(-1).mean())
            entropy = float(after["entropy"].mean())
        tolist = lambda xs: [float(x) for x in torch.cat([x.reshape(1) for x in xs]).cpu()] if xs else []  # noqa: E731
        return dict(loss_before=float(loss_before), loss_after=float(after["loss"]), kl=kl, entropy=entropy, losses=tolist(losses),
                    baseline_losses=tolist(bl_losses), grad_norms=tolist(gnorms), n_paths=P)


class DevicePPOSet:
    """K independent ``DevicePPO`` updates of one architecture and one set of hyper-parameters run side by side: every optimizer
    step is ONE ``cm_ppo_net`` call per network over all members (``cm_net_io.n_policies``) and ONE ``cm_adam_step_set`` per
    network, instead of K of each.  Member i computes what a standalone ``DevicePPO(policies[i], critics[i], fused=True)``
    computes; only the order of fp32 atomic sums differs.

    Storage: one ``[K][n]`` flat bucket per network (parameters, gradient, both moments); member i's parameters are views of row
    i, and ``members[i]`` — the member's own ``DevicePPO`` — works on those rows, so its ``process_samples`` /
    ``batch_from_trajectory`` build the member's batch.  Kernel-only: Comm-DP and Obs-DP policies with a ``CommBaseCritic`` on a
    GPU; CENT and multi-rank sets raise."""

    def __init__(self, policies, critics, **ppo_args):
        from .policy import PolicySet
        from .ppo_fused import FusedCommNets, _SetBlobMap
        policies, critics = list(policies), list(critics)
        if not policies or len(policies) != len(critics):
            raise ValueError("a DevicePPOSet needs one critic per policy")
        if _world(ppo_args.get("process_group")) > 1:
            raise NotImplementedError("DevicePPOSet runs on one rank: sets across ranks are not built")
        for p, c in zip(policies, critics):
            if p.device.type != "cuda" or not (FusedCommNets.supports(p, c) and getattr(c, "_fusable", False)):
                raise NotImplementedError("DevicePPOSet runs the update kernels of the Comm-DP / Obs-DP families only "
                                          "(CommCategoricalMLPPolicy or DecCategoricalMLPPolicy with a CommBaseCritic, on a GPU)")
        for i in range(1, len(policies)):
            if PolicySet._arch(policies[i]) != PolicySet._arch(policies[0]) or \
                    tuple((k, tuple(v.shape)) for k, v in critics[i].state_dict().items()) != \
                    tuple((k, tuple(v.shape)) for k, v in critics[0].state_dict().items()):
                raise ValueError(f"member {i} differs in architecture from member 0: one launch runs one network shape")
        ppo_args = dict(ppo_args, fused=True)
        self.members = [DevicePPO(p, c, **ppo_args) for p, c in zip(policies, critics)]
        m0 = self.members[0]
        self.K, self.device = len(policies), m0.device
        self.clip_grad_norm, self.n_minibatches, self.mini_epochs = m0.clip_grad_norm, m0.n_minibatches, m0.mini_epochs
        self.positive_adv = m0.positive_adv
        self.opt = _SetBuckets([m.opt for m in self.members])
        self.baseline_opt = _SetBuckets([m.baseline_opt for m in self.members])
        F0 = m0._fused
        self.pol = _SetBlobMap(F0.pol_map, self.opt.flat)
        self.cri = _SetBlobMap(F0.cri_map, self.baseline_opt.flat)
        for i, m in enumerate(self.members):          # the members' maps read and write the set's rows
            for mp, sm, fl in ((m._fused.pol_map, self.pol, self.opt.flat), (m._fused.cri_map, self.cri, self.baseline_opt.flat)):
                mp.flat, mp.blob, mp.grad = fl[i], sm.blob[i, :sm.nb], sm.grad[i, :sm.nb]
        self._ws = None

    # ---- one cm_ppo_net call over every member ------------------------------------------------------------------------
    def _run_set(self, desc, smap, inp, P, backward, inv_counts, policy):
        F = self.members[0]._fused
        K = self.K
        io = N.NetIO()
        io.n_steps = K * P
        io.weights, io.grad = N.ptr(smap.blob), (N.ptr(smap.grad) if backward else None)
        io.obs, io.adj_bits, io.chan_bits, io.valid = N.ptr(inp["obs"]), N.ptr(inp["adj"]), N.ptr(inp["chan"]), N.ptr(inp["valid"])
        if policy:
            io.avail_bits, io.actions, io.adv, io.old_ll = N.ptr(inp["avail"]), N.ptr(inp["actions"]), N.ptr(inp["adv"]), N.ptr(inp["old"])
        else:
            io.returns = N.ptr(inp["ret"])
        loss = torch.zeros(K, dtype=torch.float32, device=self.device)
        io.loss = N.ptr(loss)
        io.inv_counts, io.inv_count = N.ptr(inv_counts), float(inp["inv_host"][0])
        io.n_policies, io.steps_per_policy, io.weights_stride, io.grad_stride = K, P, smap.stride, smap.stride
        F._ws, ws = self._ws, None
        try:
            ws = F._workspace(desc, K * P, backward, extra=N.net_set_workspace_extra(K))
        finally:
            self._ws, F._ws = F._ws, None
        io.workspace, io.workspace_floats = N.ptr(ws), ws.numel()
        with torch.cuda.device(self.device):
            N.check("cm_ppo_net", N.lib().cm_ppo_net(C.byref(desc), C.byref(io), N.stream_ptr()))
        return loss

    @staticmethod
    def _stack(parts, P, fill, template):
        """member rows [n_i, ...] -> [K * P, ...] padded per member with `fill` to P rows"""
        out = torch.full((len(parts), P) + tuple(template.shape[1:]), fill, dtype=template.dtype, device=template.device)
        for i, t in enumerate(parts):
            if t is not None and t.shape[0]:
                out[i, :t.shape[0]] = t
        return out.reshape((len(parts) * P,) + tuple(template.shape[1:])).contiguous()

    def _slice_inputs(self, mbs, policy):
        """the set inputs of one optimizer step: member i's minibatch rows (or none), padded to the longest with finite valid = 0
        steps (zero observation, all-ones bit rows, every action available, action 0, advantage 0)"""
        key = "pol" if policy else "cri"
        rows = [mb[key]["obs"].shape[0] if mb is not None else 0 for mb in mbs]
        P = max(max(rows), 1)
        t = next(mb for mb in mbs if mb is not None)
        g = lambda k: [mb[key][k] if mb is not None else None for mb in mbs]  # noqa: E731
        inp = dict(obs=self._stack(g("obs"), P, 0, t[key]["obs"]), adj=self._stack(g("adj"), P, -1, t[key]["adj"]),
                   chan=self._stack(g("chan"), P, -1, t[key]["chan"]))
        v = torch.zeros(len(mbs), P, dtype=torch.uint8, device=self.device)
        for i, r in enumerate(rows):
            v[i, :r] = 1
        inp["valid"] = v.reshape(-1).contiguous()
        if policy:
            inp["avail"] = self._stack(g("avail"), P, 0x1F, t["pol"]["avail"])
            inp["actions"] = self._stack(g("actions"), P, 0, t["pol"]["actions"])
            inp["adv"] = self._stack([mb["adv"] if mb is not None else None for mb in mbs], P, 0.0, t["adv"])
            inp["old"] = self._stack([mb["old"] if mb is not None else None for mb in mbs], P, 0.0, t["old"])
            inv = [1.0 / max(mb["n_valid"], 1) if mb is not None else 1.0 for mb in mbs]
        else:
            inp["ret"] = self._stack([mb["ret"] if mb is not None else None for mb in mbs], P, 0.0, t["ret"])
            inv = [1.0 / max(mb["n_all"], 1) if mb is not None else 1.0 for mb in mbs]
        inp["inv_host"] = inv
        inp["inv"] = torch.tensor(inv, dtype=torch.float32, device=self.device)
        return inp, P

    # ---- train_once ---------------------------------------------------------------------------------------------------
    def train_once(self, batches, shuffled_ids=None):
        """One round of every member: ``batches[i]`` is member i's padded device batch (``members[i].process_samples`` /
        ``batch_from_trajectory``), ``shuffled_ids[i]`` its path permutation.  Returns one dict per member with the keys of
        ``DevicePPO.train_once``."""
        K = self.K
        if len(batches) != K:
            raise ValueError(f"{len(batches)} batches for {K} members")
        shuffled_ids = [None] * K if shuffled_ids is None else list(shuffled_ids)
        nan = torch.full((1,), float("nan"), device=self.device)
        with torch.no_grad():
            self.pol.refresh()
            self.cri.refresh()
            st = []                       # per member: flat batch, advantages, old policy, minibatches
            for i, (m, b) in enumerate(zip(self.members, batches)):
                F = m._fused
                f = b.get("_flat") or F.prepare(b)
                P = int(b["rewards"].shape[0])
                raw_adv, ret_all = b["adv"].reshape(-1), b["returns"].reshape(-1)
                adv_all = raw_adv - raw_adv.min() if self.positive_adv else raw_adv
                n_valid_all = max(int(f["valids_host"].sum()), 1)
                F._ws, self._ws = self._ws, None
                old = F.policy_call(f, None, adv=adv_all, want_probs=True, inv_count=1.0 / n_valid_all)
                self._ws, F._ws = F._ws, None
                ids_all = np.random.permutation(P) if shuffled_ids[i] is None else np.asarray(shuffled_ids[i])
                mbs = []
                for start, stop in minibatch_plan(P, self.n_minibatches, group=m.group):   # (a member's group: its rank alone)
                    ids = ids_all[start:stop]
                    idx_all, idx = F.step_index(f, ids, valid_only=False), F.step_index(f, ids, valid_only=True)
                    adv = raw_adv.index_select(0, idx)
                    if self.positive_adv:
                        adv = adv - raw_adv.index_select(0, idx_all).min()
                    mbs.append(dict(cri=F.subset(f, idx_all, policy=False), ret=ret_all.index_select(0, idx_all), pol=F.subset(f, idx),
                                    adv=adv, old=old["ll"].index_select(0, idx), n_valid=int(idx.numel()), n_all=int(idx_all.numel())))
                st.append(dict(f=f, P=P, adv_all=adv_all, n_valid_all=n_valid_all, old=old, mbs=mbs, losses=[], bl=[], gn=[]))
            n_slices = max(len(s["mbs"]) for s in st)
            steps = []                    # per slice: the set inputs of both networks and which members step
            for j in range(n_slices):
                mbs = [s["mbs"][j] if j < len(s["mbs"]) else None for s in st]
                steps.append((self._slice_inputs(mbs, False), self._slice_inputs(mbs, True), [mb is not None for mb in mbs]))
            F0 = self.members[0]._fused
            ones = torch.ones(K, dtype=torch.float32, device=self.device)
            for _ in range(self.mini_epochs):
                for (cri_in, Pc), (pol_in, Pp), stepped in steps:
                    self.cri.grad.zero_()
                    bl = self._run_set(F0.cri_desc, self.cri, cri_in, Pc, True, cri_in["inv"], policy=False)
                    self.cri.scatter_grad(self.baseline_opt.grad)
                    self.pol.grad.zero_()
                    loss = self._run_set(F0.pol_desc, self.pol, pol_in, Pp, True, pol_in["inv"], policy=True)
                    self.pol.scatter_grad(self.opt.grad)
                    scale = ones
                    if self.clip_grad_norm is not None:
                        coef, norm = self.opt.clip_coefficient(self.clip_grad_norm)
                        scale, gn = coef, norm * coef
                    self.opt.step(stepped, scale)
                    self.baseline_opt.step(stepped, ones)
                    self.pol.refresh()
                    self.cri.refresh()
                    for i, s in enumerate(st):
                        if stepped[i]:
                            s["losses"].append(loss[i:i + 1])
                            s["bl"].append(bl[i:i + 1])
                            if self.clip_grad_norm is not None:
                                s["gn"].append(gn[i:i + 1])
            outs = []
            for m, s in zip(self.members, st):
                F = m._fused
                F._ws, self._ws = self._ws, None
                after = F.policy_call(s["f"], None, adv=s["adv_all"], old_ll=s["old"]["ll"], want_probs=True,
                                      inv_count=1.0 / s["n_valid_all"])
                self._ws, F._ws = F._ws, None
                old_probs, new = s["old"]["probs"], after["probs"]
                t = old_probs * (old_probs.clamp_min(1e-38).log() - new.clamp_min(1e-38).log())
                kl = float(torch.where(old_probs > 0, t, torch.zeros_like(t)).sum(-1).mean())
                tolist = lambda xs: [float(x) for x in torch.cat(xs).cpu()] if xs else []  # noqa: E731
                outs.append(dict(loss_before=float(s["old"]["loss"]), loss_after=float(after["loss"]), kl=kl,
                                 entropy=float(after["entropy"].mean()), losses=tolist(s["losses"]), baseline_losses=tolist(s["bl"]),
                                 grad_norms=tolist(s["gn"]), n_paths=s["P"]))
        return outs


class _SetBuckets:
    """The flat buckets of K ``FlatAdam``s of one layout moved into ``[K][n]`` tensors (parameters, gradient, both moments):
    every member's parameters, gradient views and ``FlatAdam`` tensors become views of row i.  ``step`` is ONE
    ``cm_adam_step_set`` over the members that take a step."""

    def __init__(self, opts):
        K, o0 = len(opts), opts[0]
        n = o0.flat.numel()
        if any(o.flat.numel() != n for o in opts):
            raise ValueError("the members' parameter buckets differ in size")
        self.opts = opts
        self.flat = torch.stack([o.flat for o in opts]).contiguous()
        self.grad = torch.zeros_like(self.flat)
        self.exp_avg = torch.stack([o.exp_avg for o in opts]).contiguous()
        self.exp_avg_sq = torch.stack([o.exp_avg_sq for o in opts]).contiguous()
        for i, o in enumerate(opts):
            o.flat, o.grad, o.exp_avg, o.exp_avg_sq = self.flat[i], self.grad[i], self.exp_avg[i], self.exp_avg_sq[i]
            k0 = 0
            for p in o.params:
                k = p.numel()
                p.data = self.flat[i, k0:k0 + k].view_as(p)
                p.grad = self.grad[i, k0:k0 + k].view_as(p)
                k0 += k
        self.lr, self.betas, self.eps = o0.lr, o0.betas, o0.eps

    def clip_coefficient(self, max_norm):
        """per member: min(1, max_norm / (||g_i|| + 1e-6)) and ||g_i|| as [K] device tensors"""
        norm = self.grad.norm(2, dim=1)
        return torch.clamp(max_norm / (norm + 1e-6), max=1.0), norm

    def step(self, stepped, grad_scale):
        """one Adam step of every member i with stepped[i] (its own step count), gradient scaled by grad_scale[i] (a [K] float32
        device tensor); the other members stay bit for bit as they are"""
        K, n = self.flat.shape
        for o, s in zip(self.opts, stepped):
            o.steps += int(bool(s))
        steps = (C.c_int32 * K)(*[o.steps if s else 0 for o, s in zip(self.opts, stepped)])
        self._scale = grad_scale.detach().to(torch.float32).reshape(K).contiguous()      # (kept alive until the next step)
        with torch.cuda.device(self.flat.device):
            N.check("cm_adam_step_set", N.lib().cm_adam_step_set(N.ptr(self.flat), N.ptr(self.grad), N.ptr(self.exp_avg),
                                                                 N.ptr(self.exp_avg_sq), K, n, n, self.lr, self.betas[0], self.betas[1],
                                                                 self.eps, steps, N.ptr(self._scale), N.stream_ptr()))
        for o, s in zip(self.opts, stepped):
            if s:
                for p in o.params:
                    torch.autograd.graph.increment_version(p)
