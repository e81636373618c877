"""CommCategoricalMLPPolicy with the reference's call signature and state_dict, backed by the fused
CUDA forward (cm_policy_forward, include/commarl_b200.h).

Mirrors com_marl/torch/policies/comm_categorical_mlp_policy.py:8-140 and
com_marl/torch/modules/comm_base_net.py:11-110:
  * same constructor arguments and defaults, same ``state_dict`` parameter names/shapes (SURVEY.md §3.3),
    so reference checkpoints load with ``load_state_dict``;
  * ``get_actions(obs_n, avail_actions_n, dist_adj, channels, greedy)`` — the rollout call — runs the
    hand-written kernel (no torch ops on the hot path) and returns what the reference returns;
  * ``forward(..., get_actions=False)`` / ``entropy`` / ``log_likelihood`` — the differentiable training
    path used by the PPO update, which is outside the rollout hot path (SURVEY.md §8f-1) — is the same
    formula written with torch ops so that autograd works.
"""
import ctypes as C
import math
from collections import OrderedDict

import numpy as np
import torch
from torch import nn
from torch.distributions import Categorical

from . import _native as N


def _refresh_in_place(old, new):
    """Kernel weight blobs live in PERSISTENT device buffers: a refresh after a parameter update writes the same
    allocation, so device pointers baked into captured CUDA graphs (RolloutEngine) or cached call structs stay valid
    and the next replay reads the current weights."""
    if old is not None and old.numel() == new.numel() and old.device == new.device:
        old.copy_(new)
        return old
    return new.contiguous()


def _pad2(w, rows, cols):
    """zero-padded copy of a 2-D (or 1-D: rows only) tensor — the kernels are specialised for the reference's default layer
    widths; a narrower layer runs on them EXACTLY with its weights embedded in zeros (a padded unit computes tanh(0) = 0 and
    feeds nothing: its outgoing weights are zero too)"""
    if w.dim() == 1:
        out = w.new_zeros(rows)
        out[:w.shape[0]] = w
        return out
    out = w.new_zeros((rows, cols))
    out[:w.shape[0], :w.shape[1]] = w
    return out


class _MLP(nn.Module):
    """Parameter layout of garage's MultiHeadedMLPModule with one head
    (garage/torch/modules/multi_headed_mlp_module.py:60-100): _layers.i.linear, _output_layers.0.linear."""

    def __init__(self, input_dim, hidden_sizes, output_dim, output_tanh):
        super().__init__()
        self._layers = nn.ModuleList()
        prev = input_dim
        for size in hidden_sizes:
            lin = nn.Linear(prev, size)
            nn.init.xavier_uniform_(lin.weight)
            nn.init.zeros_(lin.bias)
            self._layers.append(nn.Sequential(OrderedDict(linear=lin)))
            prev = size
        lin = nn.Linear(prev, output_dim)
        nn.init.xavier_uniform_(lin.weight)
        nn.init.zeros_(lin.bias)
        self._output_layers = nn.ModuleList([nn.Sequential(OrderedDict(linear=lin))])
        self._output_tanh = output_tanh

    def forward(self, x):
        for layer in self._layers:
            x = torch.tanh(layer(x))
        x = self._output_layers[0](x)
        return torch.tanh(x) if self._output_tanh else x


class _Attention(nn.Module):
    """attention_module.py:15-51: 'general' (score = H_j^T W_a q, a bias-free ``linear_in``) or 'dot' (score = H_j^T q: no parameter)"""

    def __init__(self, dim, attention_type="general"):
        super().__init__()
        self.attention_type = attention_type
        if attention_type == "general":
            self.linear_in = nn.Linear(dim, dim, bias=False)

    def forward(self, query):
        context = query.transpose(-2, -1)
        q = self.linear_in(query) if self.attention_type == "general" else query
        return torch.softmax(torch.matmul(q, context), dim=-1)


class _GraphConv(nn.Module):
    """graph_conv_module.py:22-72: weight is (in, out), U(+-1/sqrt(out)) init"""

    def __init__(self, dim, bias=True):
        super().__init__()
        self.weight = nn.Parameter(torch.empty(dim, dim))
        stdv = 1.0 / math.sqrt(dim)
        self.weight.data.uniform_(-stdv, stdv)
        if bias:
            self.bias = nn.Parameter(torch.empty(dim))
            self.bias.data.uniform_(-stdv, stdv)
        else:
            self.register_parameter("bias", None)

    def forward(self, inputs, A):
        out = torch.matmul(A, torch.matmul(inputs, self.weight))
        return torch.tanh(out + self.bias) if self.bias is not None else torch.tanh(out)


class CommCategoricalMLPPolicy(nn.Module):
    _kind = N.POLICY_COMM

    def __init__(self, env_spec, n_agents, encoder_hidden_sizes=(128,), embedding_dim=64, attention_type="general",
                 n_gcn_layers=2, residual=True, gcn_bias=True, categorical_mlp_hidden_sizes=(128, 64, 32),
                 name="comm_categorical_mlp_policy", device="cuda", seed=1, math="auto"):
        super().__init__()
        if not hasattr(env_spec.action_space, "n"):
            raise AssertionError("Categorical policy only works with akro.Discrete action space.")
        enc, head = tuple(encoder_hidden_sizes), tuple(categorical_mlp_hidden_sizes)
        if len(enc) != 1 or len(head) != 3 or enc[0] > 128 or embedding_dim > 64 or head[0] > 128 or head[1] > 64 or head[2] > 32:
            raise NotImplementedError("the fused kernel holds one encoder hidden layer of <= 128 units, an embedding of <= 64 and a head "
                                      "of three hidden layers of <= (128, 64, 32) units (the reference's defaults are exactly these "
                                      "maxima; narrower layers run exactly, zero-padded)")
        if attention_type not in ("general", "dot"):
            raise NotImplementedError("attention_type must be 'general' or 'dot' (the reference's 'diff' has no forward path either: "
                                      "attention_module.py:38-51)")
        self.name, self.device = name, torch.device(device)
        self.comm, self.centralized, self.step, self.eps = True, True, 0, 1e-12
        self.residual = bool(residual)
        self._n_agents = int(n_agents)
        self._cent_obs_dim = env_spec.observation_space.flat_dim
        self._dec_obs_dim = int(self._cent_obs_dim / n_agents)
        self._action_dim = env_spec.action_space.n
        self._embedding_dim = embedding_dim
        self.n_gcn_layers = int(n_gcn_layers)
        self.seed = int(seed)
        # 'auto' = 'tc': tensor cores, error-compensated fp16 products with fp32 accumulation (fp32-level accuracy)
        if math not in ("auto", "tc"):
            raise ValueError(f"math must be 'auto' or 'tc', not {math!r}: the tensor-core kernels are the only Comm-DP forward")
        self.math = math
        self.encoder = _MLP(self._dec_obs_dim, encoder_hidden_sizes, embedding_dim, output_tanh=True)
        self.attention_layer = _Attention(embedding_dim, attention_type)
        self.gcn_layers = nn.ModuleList([_GraphConv(embedding_dim, gcn_bias) for _ in range(self.n_gcn_layers)])
        self.categorical_output_layer = _MLP(embedding_dim, categorical_mlp_hidden_sizes, self._action_dim, output_tanh=False)
        self.to(self.device)
        self._blob = None
        self._blob_sig = None
        self._tc_blob = None
        self._tc_sig = None
        self._tc_error = None
        self._workspace = None

    # ---- weight blob (layout in include/commarl_b200.h) ----------------------------------------------
    def _signature(self):
        plist = self.__dict__.get("_plist")
        if plist is None:                        # (walking the module tree costs more than the whole check)
            plist = self.__dict__["_plist"] = list(self.parameters())
        return tuple([(p.data_ptr(), p._version) for p in plist])

    def _pack_blob(self, sd):
        """state dict -> flat float32 blob in the layout of include/commarl_b200.h at the kernel's widths (128 / 64 / (128, 64,
        32)); narrower layers are embedded in zeros (_pad2), 'dot' attention is W_a = identity.  Pure tensor plumbing: also
        used with index tensors to derive the parameter <-> blob maps of the fused PPO update (ppo_fused._BlobMap)."""
        L, E, D = self.n_gcn_layers, self._embedding_dim, self._dec_obs_dim
        att = sd["attention_layer.linear_in.weight"].t() if "attention_layer.linear_in.weight" in sd \
            else torch.eye(E, device=self.device)
        parts = [_pad2(sd["encoder._layers.0.linear.weight"].t(), D, 128), _pad2(sd["encoder._layers.0.linear.bias"], 128, 0),
                 _pad2(sd["encoder._output_layers.0.linear.weight"].t(), 128, 64), _pad2(sd["encoder._output_layers.0.linear.bias"], 64, 0),
                 _pad2(att, 64, 64)]
        parts += [_pad2(sd[f"gcn_layers.{l}.weight"], 64, 64) for l in range(L)]
        parts += [_pad2(sd.get(f"gcn_layers.{l}.bias", torch.zeros(E, device=self.device)), 64, 0) for l in range(L)]
        for i, (k_in, k_out) in enumerate(((64, 128), (128, 64), (64, 32))):
            parts += [_pad2(sd[f"categorical_output_layer._layers.{i}.linear.weight"].t(), k_in, k_out),
                      _pad2(sd[f"categorical_output_layer._layers.{i}.linear.bias"], k_out, 0)]
        parts += [_pad2(sd["categorical_output_layer._output_layers.0.linear.weight"].t(), 32, self._action_dim),
                  sd["categorical_output_layer._output_layers.0.linear.bias"]]
        return torch.cat([p.detach().to(self.device, torch.float32).contiguous().reshape(-1) for p in parts])

    def weight_blob(self):
        """float32 device blob, every dense weight k-major; rebuilt when a parameter changed."""
        sig = self._signature()
        if self._blob is None or sig != self._blob_sig:
            blob = self._pack_blob(self.state_dict())
            expect = N.lib().cm_policy_blob_floats(self._dec_obs_dim, self.n_gcn_layers)
            assert blob.numel() == expect, (blob.numel(), expect)
            self._blob = _refresh_in_place(self._blob, blob)
            self._blob_sig = sig
        return self._blob

    def uses_tensor_cores(self):
        return True

    def tc_weight_blob(self):
        """pre-split (hi | lo), pre-laid-out B operands of the tcgen05 variant; rebuilt when a parameter changed"""
        blob = self.weight_blob()
        if self._tc_blob is None or self._tc_sig != self._blob_sig:
            L = self.n_gcn_layers
            n_floats = N.lib().cm_policy_tc_blob_floats(self._dec_obs_dim, L)
            # written in place from the second time on: a captured CUDA graph keeps pointing at live, current weights
            out = self._tc_blob if self._tc_blob is not None else torch.empty(n_floats, dtype=torch.float32, device=self.device)
            desc = N.PolicyDesc(self._n_agents, self._dec_obs_dim, L, int(self.residual), 0, 1, self.seed, 0, self._kind)
            with torch.cuda.device(self.device):
                N.check("cm_policy_tc_prepare", N.lib().cm_policy_tc_prepare(C.byref(desc), N.ptr(blob), N.ptr(out), N.stream_ptr()))
            self._tc_blob, self._tc_sig = out, self._blob_sig
            if self._tc_error is None:
                self._tc_error = torch.zeros(1, dtype=torch.int32, device=self.device)
        return self._tc_blob

    def refresh_weights(self, force=False):
        """bring the kernel weight blobs up to date with the parameters (in place; cheap signature check when nothing
        changed) — the rollout engine calls this before replaying a captured graph.  The signature reads the parameters'
        version counters, which every in-place op on a parameter, ``load_state_dict`` and FlatAdam bump; a write through
        ``p.data`` (``p.data.add_``, optimizers and loaders written that way) does not: call with ``force=True`` after one."""
        if force:
            self._blob_sig = self._tc_sig = None
        if self.uses_tensor_cores():
            self.tc_weight_blob()
        else:
            self.weight_blob()

    def check_errors(self):
        if self._tc_error is not None and int(self._tc_error.item()):
            self._tc_error.zero_()
            raise N.NativeError("policy_tc_kernel", N.CM_ECUDA, "a bounded device-side wait timed out")

    # ---- device fast path (no host copies) --------------------------------------------------------------
    def act_device(self, obs, adj_bits=None, chan_bits=None, avail_bits=None, sample_u=None, tick=None, episode=None,
                   greedy=False, probs=None, logits=None, attention=None, actions=None, env_id0=0, ws_slot=0, obs_bits=None,
                   obs_nbits=0):
        """Fused forward on device tensors.  obs: float32 (B, n, D) / (B, n*D).  Outputs are written into the
        given tensors (allocate once, reuse: the call is CUDA-graph capturable).  ``obs_bits`` (int32 (B, n, 6), what
        ``BatchedEnv.enable_obs_bits()`` makes the env kernel write) + ``obs_nbits``: the packed observation — the
        tensor-core kernels read it instead of ``obs`` (24 bytes per agent row instead of 4 D; identical results)."""
        desc, io = self._call_structs(obs, adj_bits, chan_bits, avail_bits, sample_u, tick, episode, greedy, probs, logits,
                                      attention, actions, env_id0, ws_slot)
        if obs_bits is not None:
            io.obs_bits, io.obs_nbits = N.ptr(obs_bits), int(obs_nbits)
        with torch.cuda.device(self.device):
            N.check("cm_policy_forward", N.lib().cm_policy_forward(C.byref(desc), C.byref(io), N.stream_ptr()))

    def _call_structs(self, obs, adj_bits, chan_bits, avail_bits, sample_u, tick, episode, greedy, probs, logits, attention,
                      actions, env_id0, ws_slot):
        """descriptor + io struct of one cm_policy_forward call on device tensors"""
        n, D, L = self._n_agents, self._dec_obs_dim, self.n_gcn_layers
        B = obs.shape[0]
        desc = N.PolicyDesc(n, D, L, int(self.residual), int(greedy), 1, self.seed, env_id0, self._kind)
        io = N.PolicyIO()
        io.n_envs = B
        io.tc_weights = N.ptr(self.tc_weight_blob())          # (refreshes the fp32 blob as well)
        io.error_flag = N.ptr(self._tc_error)
        io.weights = N.ptr(self._blob)
        for k, v in (("obs", obs), ("adj_bits", adj_bits), ("chan_bits", chan_bits), ("avail_bits", avail_bits),
                     ("sample_u", sample_u), ("tick", tick), ("episode", episode), ("probs", probs), ("logits", logits),
                     ("attention", attention), ("actions", actions)):
            setattr(io, k, N.ptr(v))
        if n > 64 and self._kind == N.POLICY_COMM:      # large teams: scratch, allocated once per concurrent caller and reused
            need = N.lib().cm_policy_workspace_bytes(n, B)
            if self._workspace is None:
                self._workspace = {}
            ws = self._workspace.get(ws_slot)
            if ws is None or ws.numel() * 4 < need:
                ws = self._workspace[ws_slot] = torch.empty((need + 3) // 4, dtype=torch.float32, device=self.device)
            io.workspace, io.workspace_bytes = N.ptr(ws), ws.numel() * 4
        return desc, io

    @staticmethod
    def pack_mask(dense, n):
        """dense float32 (..., n, n) device tensor -> int32 bit rows (..., n, ceil(n/32))"""
        dense = dense.contiguous()
        rows = dense.numel() // n
        W = (n + 31) // 32
        bits = torch.empty(dense.shape[:-1] + (W,), dtype=torch.int32, device=dense.device)
        with torch.cuda.device(dense.device):
            N.check("cm_mask_pack", N.lib().cm_mask_pack(N.ptr(dense), N.ptr(bits), rows, n, N.stream_ptr()))
        return bits

    # ---- reference call surface --------------------------------------------------------------------------
    def _run_host(self, obs_n, avail_actions_n, dist_adj, channels, greedy, want_actions):
        n, D, L, dev = self._n_agents, self._dec_obs_dim, self.n_gcn_layers, self.device
        obs = torch.as_tensor(np.asarray(obs_n), dtype=torch.float32)
        single = obs.dim() == 1
        obs = obs.reshape(-1, n, D).to(dev, non_blocking=True)
        B = obs.shape[0]
        adj = torch.as_tensor(np.asarray(dist_adj), dtype=torch.float32).reshape(B, n, n).to(dev, non_blocking=True)
        ch = torch.as_tensor(np.asarray(channels), dtype=torch.float32).reshape(B, L, n, n).to(dev, non_blocking=True)
        av = torch.as_tensor(np.asarray(avail_actions_n), dtype=torch.float32).reshape(B, n, self._action_dim)
        weights = torch.tensor([1, 2, 4, 8, 16], dtype=torch.float32)
        avail_bits = ((av != 0).float() * weights).sum(-1).to(torch.uint8).to(dev, non_blocking=True)
        probs = torch.empty((B, n, self._action_dim), dtype=torch.float32, device=dev)
        attn = torch.empty((B, n, n), dtype=torch.float32, device=dev)
        actions = torch.empty((B, n), dtype=torch.int8, device=dev) if want_actions else None
        # host-call sampling stream: keyed by the policy's own call counter (the env arrays are not visible here)
        tick = torch.full((B,), self.step & 0x7FFFFFFF, dtype=torch.int32, device=dev)
        episode = torch.full((B,), self._host_calls & 0xFFFFFF, dtype=torch.int32, device=dev)
        self._host_calls += 1
        self.act_device(obs, self.pack_mask(adj, n), self.pack_mask(ch, n), avail_bits, None, tick, episode, greedy,
                        probs, None, attn, actions)
        return single, probs, attn, actions

    _host_calls = 0

    def get_actions_host(self, obs, adj_bits, chan_bits, greedy=False, return_pinned=False, slot=0, sync=True, stream=None,
                         inputs_arena=False):
        """Batched rollout call with HOST buffers and bit-row masks (what BatchedEnv.step_host returns): numpy obs
        (B, n, D) / (B, n*D), int32 bit rows in; numpy actions (B, n) int8 and probs (B, n, 5) out.  Pinned staging
        buffers are allocated once; inputs that already are pinned torch tensors (e.g. ``step_host(...)["pinned"]``) are
        copied to the device directly.  Copies: H2D obs + masks; D2H actions + probs.

        Split-phase use (``sync=False``): everything is enqueued on the CURRENT stream and the call returns
        ``(actions, probs, event)`` at once; the outputs are valid after ``event.synchronize()``.  ``slot`` selects an
        independent set of staging buffers, so that several env batches can be in flight on different streams (the
        H2D copies of one batch then overlap the D2H copies of another: PCIe is full duplex).
        ``inputs_arena=True`` declares that pinned ``obs, adj_bits, chan_bits`` are neighbours in ONE host arena in this
        order with 256-byte padding (``BatchedEnv.step_host(...)["pinned"]`` is): the library then moves them with a single
        DMA transfer (cm_policy_io.host_arena); undeclared pinned inputs are copied one array at a time."""
        n, D, L, dev = self._n_agents, self._dec_obs_dim, self.n_gcn_layers, self.device
        B = obs.shape[0]
        stages = self.__dict__.setdefault("_stages", {})
        st = stages.get(slot)
        if st is None or st["B"] != B:
            W = (n + 31) // 32
            # inputs and outputs as arenas with the same order / padding on both sides (and as the env's host buffers):
            # the library moves each group with one DMA transfer
            ins = [("obs", (B, n, D), torch.float32), ("adj", (B, n, W), torch.int32), ("chan", (B, L, n, W), torch.int32)]
            outs = [("actions", (B, n), torch.int8), ("probs", (B, n, 5), torch.float32)]
            hi, di = N.arena(ins, pinned=True), N.arena(ins, device=dev)
            ho, do = N.arena(outs, pinned=True), N.arena(outs, device=dev)
            st = dict(B=B, tick=torch.zeros((B,), dtype=torch.int32, device=dev), episode=torch.zeros((B,), dtype=torch.int32, device=dev),
                      event=torch.cuda.Event(), _keep=(hi, di, ho, do))
            for k in ("obs", "adj", "chan"):
                st[k] = (hi[k], di[k])
            for k in ("actions", "probs"):
                st[k] = (ho[k], do[k])
            stages[slot] = st
        hio = st.get("hio")
        if hio is None:
            hio = st["hio"] = N.PolicyIO()
            hio.actions, hio.probs = st["actions"][0].data_ptr(), st["probs"][0].data_ptr()
            st["last_in"] = (None, None, None)
        if not (obs is st["last_in"][0] and adj_bits is st["last_in"][1] and chan_bits is st["last_in"][2]):
            pinned_in = True
            for k, f, src in (("obs", "obs", obs), ("adj", "adj_bits", adj_bits), ("chan", "chan_bits", chan_bits)):
                h, d = st[k]
                if isinstance(src, torch.Tensor) and src.is_pinned() and src.dtype == h.dtype and src.numel() == h.numel():
                    setattr(hio, f, src.data_ptr())                 # caller's buffer is already pinned: no staging copy
                else:
                    h.numpy()[...] = np.asarray(src).reshape(h.shape)
                    setattr(hio, f, h.data_ptr())
                    pinned_in = False
            # the same pinned tensors again (the env's persistent host buffers): nothing to re-derive next time
            st["last_in"] = (obs, adj_bits, chan_bits) if pinned_in else (None, None, None)
            hio.host_arena = int((not pinned_in) or bool(inputs_arena))     # own staging arena, or declared by the caller
        sig = self._signature()
        cs = st.get("structs")
        if cs is None or cs[0] != (sig, bool(greedy)):
            desc, dio = self._call_structs(st["obs"][1], st["adj"][1], st["chan"][1], None, None, st["tick"], st["episode"], greedy,
                                           st["probs"][1], None, None, st["actions"][1], 0, slot)
            cs = st["structs"] = ((sig, bool(greedy)), desc, dio)
        desc, dio = cs[1], cs[2]
        tick_all = self._host_calls & 0x7FFFFFFF
        self._host_calls += 1
        # ONE C call: H2D obs + masks, tick fill, the forward, D2H actions + probs (include/commarl_b200.h)
        if dev.index is not None and torch.cuda.current_device() != dev.index:
            torch.cuda.set_device(dev)           # the library launches on the current device
        if stream is None:
            stream = torch.cuda.current_stream(dev)
        N.check("cm_policy_forward_host", N.lib().cm_policy_forward_host(C.byref(desc), C.byref(dio), C.byref(hio), tick_all,
                                                                         stream.cuda_stream))
        if not sync:
            st["event"].record(stream)
            return st["actions"][0], st["probs"][0], st["event"]
        stream.synchronize()
        if return_pinned:
            return st["actions"][0], st["probs"][0]
        return st["actions"][0].numpy(), st["probs"][0].numpy()

    def host_call_bytes(self, B):
        n, D, L = self._n_agents, self._dec_obs_dim, self.n_gcn_layers
        W = (n + 31) // 32
        return B * n * D * 4 + B * n * W * 4 * (1 + L), B * n * 5 * 4 + B * n

    def forward(self, obs_n, avail_actions_n, dist_adj, channels, get_actions=False):
        """comm_categorical_mlp_policy.py:48-96.  get_actions=True: numpy in, CPU tensors out (kernel path).
        get_actions=False: torch tensors shaped (n_paths, T, ...) in, differentiable (torch ops)."""
        n = self._n_agents
        if get_actions:
            single, probs, attn, _ = self._run_host(obs_n, avail_actions_n, dist_adj, channels, False, False)
            probs, attn = probs.cpu(), attn.cpu()
            if single:
                probs, attn = probs[0], attn[0]
            return Categorical(probs=probs), attn
        obs_n = obs_n.reshape(obs_n.shape[:-1] + (n, -1))
        avail_actions_n = avail_actions_n.reshape(avail_actions_n.shape[:-1] + (n, -1))
        channels = channels.reshape(channels.shape[:-2] + (len(self.gcn_layers), n, n))
        if dist_adj.shape[-2:] != torch.Size((n, n)):
            dist_adj = dist_adj.reshape(dist_adj.shape[:-1] + (n, n))
        E = self.encoder(obs_n)
        M = self.attention_layer(E)
        H = E
        for l, gcn in enumerate(self.gcn_layers):
            A = M * dist_adj * channels[..., l, :, :]
            A = A / (A.sum(dim=-1, keepdim=True) + self.eps)
            H = gcn(H, A)
        X = E + H if self.residual else H
        dist = Categorical(logits=self.categorical_output_layer(X))
        masked = dist.probs * avail_actions_n
        masked = masked / masked.sum(dim=-1, keepdim=True)
        return Categorical(probs=masked), M

    def get_actions(self, obs_n, avail_actions_n, dist_adj, channels, greedy=False):
        """comm_categorical_mlp_policy.py:98-119: (actions int64 (B,n)|(n,), {'action_probs': [...],
        'attention_weights': [...]})"""
        with torch.no_grad():
            single, probs, attn, actions = self._run_host(obs_n, avail_actions_n, dist_adj, channels, greedy, True)
            probs, attn, actions = probs.cpu().numpy(), attn.cpu().numpy(), actions.cpu().numpy().astype(np.int64)
            if single:
                probs, attn, actions = probs[0], attn[0], actions[0]
            infos = {"action_probs": [probs[i] for i in range(len(actions))],
                     "attention_weights": [attn[i, :] for i in range(len(actions))]}
            return actions, infos

    def entropy(self, observations, avail_actions, dist_adj, channels):
        dists_n, _ = self.forward(observations, avail_actions, dist_adj, channels)
        return dists_n.entropy().mean(axis=-1)

    def log_likelihood(self, observations, avail_actions, dist_adj, channels, actions):
        dists_n, _ = self.forward(observations, avail_actions, dist_adj, channels)
        return dists_n.log_prob(actions).sum(axis=-1)

    def reset(self, dones=None):
        return

    def grad_norm(self):
        return np.sqrt(np.sum([p.grad.norm(2).item() ** 2 for p in self.parameters()]))

    @property
    def recurrent(self):
        return False



class DecCategoricalMLPPolicy(nn.Module):
    """Obs-DP policy (no communication) with the reference's call signature and state_dict, backed by the same fused
    tensor-core kernel (cm_policy_desc.kind = CM_POLICY_DEC).

    Mirrors com_marl/torch/policies/dec_categorical_mlp_policy.py:14-232: per-agent encoder D -> hidden_sizes[0] ->
    hidden_sizes[1] (tanh, MLPEncoderModule) followed by CategoricalMLPModule hidden_sizes[1] -> hidden_sizes[-1]
    (tanh) -> 5 (:76-102); the policy itself IS the categorical module, so its parameters are ``_layers.0.linear.*`` /
    ``_output_layers.0.linear.*`` next to ``encoder.*`` and reference checkpoints load with ``load_state_dict``.
    ``get_actions(observations, avail_actions, greedy)`` runs the kernel; ``forward`` / ``entropy`` / ``log_likelihood``
    (the differentiable training path, :198-226) are the same formula in torch ops."""
    _kind = N.POLICY_DEC

    def __init__(self, env_spec, n_agents, hidden_sizes=(128, 64, 32), name="DecCategoricalMLPPolicy", device="cuda", seed=1):
        super().__init__()
        if not hasattr(env_spec.action_space, "n"):
            raise AssertionError("CategoricalMLPPolicy only works with akro.Discrete action space.")
        if len(tuple(hidden_sizes)) != 3 or hidden_sizes[0] > 128 or hidden_sizes[1] > 64 or hidden_sizes[2] > 32:
            raise NotImplementedError("the fused kernel holds hidden_sizes of three layers of <= (128, 64, 32) units (the runners' "
                                      "sizes, exp_runners/env_uitils.py:188-189; narrower layers run exactly, zero-padded)")
        self.name, self.device = name, torch.device(device)
        self.comm, self.centralized, self.step = False, True, 0
        self.residual, self.math, self.n_gcn_layers = False, "tc", 1      # blob layout of one (unused) GCN layer
        self._n_agents = int(n_agents)
        self._dec_obs_dim = int(env_spec.observation_space.flat_dim / n_agents)
        self._obs_dim = self._dec_obs_dim
        self._action_dim = env_spec.action_space.n
        self._embedding_dim = hidden_sizes[1]
        self.seed = int(seed)
        head = _MLP(self._embedding_dim, (hidden_sizes[-1],), self._action_dim, output_tanh=False)   # created first, like the reference
        self._layers, self._output_layers = head._layers, head._output_layers
        self.encoder = _MLP(self._dec_obs_dim, (hidden_sizes[0],), self._embedding_dim, output_tanh=True)
        self.to(self.device)
        self._blob = self._blob_sig = self._tc_blob = self._tc_sig = self._tc_error = self._workspace = None

    _signature = CommCategoricalMLPPolicy._signature
    tc_weight_blob = CommCategoricalMLPPolicy.tc_weight_blob
    refresh_weights = CommCategoricalMLPPolicy.refresh_weights
    check_errors = CommCategoricalMLPPolicy.check_errors
    _act_device = CommCategoricalMLPPolicy.act_device
    _call_structs = CommCategoricalMLPPolicy._call_structs

    def uses_tensor_cores(self):
        return True

    def _pack_blob(self, sd):
        """the Comm-DP blob layout (include/commarl_b200.h) with the unused blocks zero: enc_w1/b1, enc_w2/b2 <- encoder,
        head_w3/b3 <- _layers.0, head_w4/b4 <- _output_layers.0"""
        dev, D = self.device, self._dec_obs_dim
        z = lambda *shape: torch.zeros(shape, device=dev)  # noqa: E731
        parts = [_pad2(sd["encoder._layers.0.linear.weight"].t(), D, 128), _pad2(sd["encoder._layers.0.linear.bias"], 128, 0),
                 _pad2(sd["encoder._output_layers.0.linear.weight"].t(), 128, 64), _pad2(sd["encoder._output_layers.0.linear.bias"], 64, 0),
                 z(64, 64), z(64, 64), z(64), z(64, 128), z(128), z(128, 64), z(64),
                 _pad2(sd["_layers.0.linear.weight"].t(), 64, 32), _pad2(sd["_layers.0.linear.bias"], 32, 0),
                 _pad2(sd["_output_layers.0.linear.weight"].t(), 32, self._action_dim), sd["_output_layers.0.linear.bias"]]
        return torch.cat([p.detach().to(dev, torch.float32).contiguous().reshape(-1) for p in parts])

    def weight_blob(self):
        sig = self._signature()
        if self._blob is None or sig != self._blob_sig:
            blob = self._pack_blob(self.state_dict())
            assert blob.numel() == N.lib().cm_policy_blob_floats(self._dec_obs_dim, 1)
            self._blob = _refresh_in_place(self._blob, blob)
            self._blob_sig = sig
        return self._blob

    def act_device(self, obs, avail_bits=None, sample_u=None, tick=None, episode=None, greedy=False, probs=None, logits=None,
                   actions=None, env_id0=0, obs_bits=None, obs_nbits=0, **_unused):
        """fused forward on device tensors (see CommCategoricalMLPPolicy.act_device); no masks, no attention output"""
        self._act_device(obs, None, None, avail_bits, sample_u, tick, episode, greedy, probs, logits, None, actions, env_id0,
                         obs_bits=obs_bits, obs_nbits=obs_nbits)

    # ---- reference call surface ----
    def forward(self, obs, avail_actions, get_actions=False):
        if get_actions:
            obs = torch.as_tensor(np.asarray(obs), dtype=torch.float32, device=self.device)
            avail_actions = torch.as_tensor(np.asarray(avail_actions), dtype=torch.float32, device=self.device)
        obs = obs.reshape(obs.shape[:-1] + (self._n_agents, -1))
        x = self.encoder(obs)
        x = torch.tanh(self._layers[0](x))
        probs = torch.softmax(self._output_layers[0](x), dim=-1)
        avail = avail_actions.reshape(avail_actions.shape[:-1] + (self._n_agents, -1))
        masked = probs * avail
        masked = masked / masked.sum(dim=-1, keepdim=True)
        return Categorical(probs=masked.cpu() if get_actions else masked)

    _host_calls = 0

    def get_actions(self, observations, avail_actions, greedy=False):
        """(B, n*D) observations, (B, n*5) availability -> (actions int64 (B, n), {'action_probs': [...]}) through the kernel"""
        n, D, dev = self._n_agents, self._dec_obs_dim, self.device
        obs = torch.as_tensor(np.asarray(observations), dtype=torch.float32)
        single = obs.dim() == 1
        obs = obs.reshape(-1, n, D).to(dev)
        B = obs.shape[0]
        av = torch.as_tensor(np.asarray(avail_actions), dtype=torch.float32).reshape(B, n, self._action_dim)
        avail_bits = ((av != 0).float() * torch.tensor([1, 2, 4, 8, 16], dtype=torch.float32)).sum(-1).to(torch.uint8).to(dev)
        probs = torch.empty((B, n, self._action_dim), dtype=torch.float32, device=dev)
        actions = torch.empty((B, n), dtype=torch.int8, device=dev)
        tick = torch.full((B,), self.step & 0x7FFFFFFF, dtype=torch.int32, device=dev)
        episode = torch.full((B,), self._host_calls & 0xFFFFFF, dtype=torch.int32, device=dev)
        self._host_calls += 1
        self.act_device(obs, avail_bits, None, tick, episode, greedy, probs, None, actions)
        self.check_errors()
        a, pr = actions.cpu().numpy().astype(np.int64), probs.cpu().numpy()
        if single:
            a, pr = a[0], pr[0]
        return a, {"action_probs": [pr[i] for i in range(len(a))]}

    def log_likelihood(self, observations, avail_actions, actions):
        return self.forward(observations, avail_actions).log_prob(actions).sum(axis=-1)

    def entropy(self, observations, avail_actions):
        return self.forward(observations, avail_actions).entropy().mean(axis=-1)

    def reset(self, dones=None):
        pass

    def grad_norm(self):
        return math.sqrt(sum(p.grad.norm(2).item() ** 2 for p in self.parameters() if p.grad is not None))

    @property
    def vectorized(self):
        return True

    @property
    def recurrent(self):
        return False


class CentralizedCategoricalMLPPolicy(nn.Module):
    """CENT policy (one MLP over the concatenated observation of the team) with the reference's call signature and
    state_dict, backed by ``policy_cent_kernel`` (cm_policy_desc.kind = CM_POLICY_CENT).

    Mirrors com_marl/torch/policies/centralized_categorical_mlp_policy.py:11-137: the policy IS garage's MLPModule
    ``n*D -> hidden_sizes -> 5n`` (xavier_uniform weights, zero biases, :16-21,43-53), so its parameters are
    ``_layers.i.linear.*`` / ``_output_layers.0.linear.*`` and reference checkpoints load with ``load_state_dict``; the
    logits are reshaped to ``(..., n, 5)``, softmax per agent, availability mask, renormalisation (:73-96).
    ``get_actions(obs_n, avail_actions_n, greedy)`` (:98-117) runs the kernel; ``forward`` / ``entropy`` /
    ``log_likelihood`` (:122-137, the differentiable training path) are the same formula in torch ops.  The runners build
    it with ``hidden_sizes=[128, 64, 32]`` and tanh or relu (runner_*_cent.py:48-58, env_uitils.py:188-189) — the sizes the
    kernel is specialised for; note that the class default ``(32, 32)`` of the reference is never used by its runners."""
    _kind = N.POLICY_CENT

    def __init__(self, env_spec, n_agents, hidden_sizes=(128, 64, 32), hidden_nonlinearity=torch.tanh,
                 name="CentralizedCategoricalMLPPolicy", device="cuda", seed=1, math="auto"):
        """math: 'fp32' = every layer in exact fp32 on the CUDA cores; 'tc' = the first layer (K = n*D) on the tcgen05 tensor
        cores with error-compensated fp16 operands (fp32-level accuracy); 'auto' = 'tc' from K = 512 inputs upwards."""
        super().__init__()
        if not hasattr(env_spec.action_space, "n"):
            raise AssertionError("Categorical policy only works with akro.Discrete action space.")
        if len(tuple(hidden_sizes)) != 3 or hidden_sizes[0] > 128 or hidden_sizes[1] > 64 or hidden_sizes[2] > 32:
            raise NotImplementedError("the kernel holds hidden_sizes of three layers of <= (128, 64, 32) units (the runners' sizes, "
                                      "exp_runners/env_uitils.py:188-189; narrower layers run exactly, zero-padded)")
        if hidden_nonlinearity in (torch.tanh, "tanh"):
            self._relu = False
        elif hidden_nonlinearity in (torch.relu, torch.nn.functional.relu, "relu"):
            self._relu = True
        else:
            raise NotImplementedError("hidden_nonlinearity must be tanh or relu (runner_*_cent.py:49)")
        if math not in ("auto", "tc", "fp32"):
            raise ValueError("math must be 'auto', 'tc' or 'fp32'")
        self.name, self.device = name, torch.device(device)
        self.centralized, self.vectorized, self.step = True, True, 0          # (no `comm` attribute: the sampler's switch)
        self._n_agents = int(n_agents)
        self._obs_dim = int(env_spec.observation_space.flat_dim)
        self._dec_obs_dim = self._obs_dim // self._n_agents
        self._action_dim = env_spec.action_space.n
        self.seed = int(seed)
        self.math = ("tc" if self._obs_dim >= 512 else "fp32") if math == "auto" else math
        mlp = _MLP(self._obs_dim, tuple(hidden_sizes), self._action_dim * self._n_agents, output_tanh=False)
        self._layers, self._output_layers = mlp._layers, mlp._output_layers
        self.layers = [self]
        self.to(self.device)
        self._blob = self._blob_sig = self._tc_blob = self._tc_sig = self._tc_error = None
        self._workspace = {}

    _signature = CommCategoricalMLPPolicy._signature
    refresh_weights = CommCategoricalMLPPolicy.refresh_weights
    check_errors = CommCategoricalMLPPolicy.check_errors

    def uses_tensor_cores(self):
        return self.math == "tc"

    def _pack_blob(self, sd):
        """state dict -> w1 [n*D][128] b1 w2 [128][64] b2 w3 [64][32] b3 w4 [32][5n] b4 (include/commarl_b200.h), narrower layers
        zero-padded; also the parameter <-> blob map of the fused PPO update (ppo_fused._BlobMap)"""
        parts = []
        for i, (k_in, k_out) in enumerate(((self._obs_dim, 128), (128, 64), (64, 32))):
            parts += [_pad2(sd[f"_layers.{i}.linear.weight"].t(), k_in, k_out), _pad2(sd[f"_layers.{i}.linear.bias"], k_out, 0)]
        parts += [_pad2(sd["_output_layers.0.linear.weight"].t(), 32, self._action_dim * self._n_agents), sd["_output_layers.0.linear.bias"]]
        return torch.cat([p.detach().to(self.device, torch.float32).contiguous().reshape(-1) for p in parts])

    def weight_blob(self):
        """the kernels' fp32 blob (_pack_blob), rebuilt when a parameter changed"""
        sig = self._signature()
        if self._blob is None or sig != self._blob_sig:
            blob = self._pack_blob(self.state_dict())
            assert blob.numel() == N.lib().cm_policy_cent_blob_floats(self._n_agents, self._dec_obs_dim)
            self._blob = _refresh_in_place(self._blob, blob)
            self._blob_sig = sig
        return self._blob

    def tc_weight_blob(self):
        """[W1_hi ; W1_lo] (256 x 32) per K panel of 32 in the tensor cores' operand layout (cm_policy_tc_prepare); rebuilt when a parameter changed"""
        blob = self.weight_blob()
        if self._tc_blob is None or self._tc_sig != self._blob_sig:
            out = self._tc_blob if self._tc_blob is not None else \
                torch.empty(N.lib().cm_policy_cent_tc_blob_floats(self._n_agents, self._dec_obs_dim), dtype=torch.float32, device=self.device)
            desc = N.PolicyDesc(self._n_agents, self._dec_obs_dim, 1, 0, 0, 1, self.seed, 0, self._kind, 0)
            with torch.cuda.device(self.device):
                N.check("cm_policy_tc_prepare", N.lib().cm_policy_tc_prepare(C.byref(desc), N.ptr(blob), N.ptr(out), N.stream_ptr()))
            self._tc_blob, self._tc_sig = out, self._blob_sig
            if self._tc_error is None:
                self._tc_error = torch.zeros(1, dtype=torch.int32, device=self.device)
        return self._tc_blob

    def act_device(self, obs, avail_bits=None, sample_u=None, tick=None, episode=None, greedy=False, probs=None, logits=None,
                   actions=None, env_id0=0, **_unused):
        """forward + sampling on device tensors (obs float32 (B, n, D) / (B, n*D)); no masks, no attention output.
        Outputs are written into the given tensors; the call is CUDA-graph capturable (with math = 'tc' after one eager call:
        the first-layer scratch is allocated once per caller, keyed by (env_id0, B) — the rollout engine's env groups run on
        parallel streams and must not share it)."""
        desc, io = self._call_structs(obs, None, None, avail_bits, sample_u, tick, episode, greedy, probs, logits, None, actions, env_id0, 0)
        with torch.cuda.device(self.device):
            N.check("cm_policy_forward", N.lib().cm_policy_forward(C.byref(desc), C.byref(io), N.stream_ptr()))

    def _call_structs(self, obs, adj_bits, chan_bits, avail_bits, sample_u, tick, episode, greedy, probs, logits, attention,
                      actions, env_id0, ws_slot):
        """descriptor + io struct of one cm_policy_forward call on device tensors (masks / attention do not exist for CENT)"""
        tc = self.math == "tc"
        B = obs.shape[0]
        desc = N.PolicyDesc(self._n_agents, self._dec_obs_dim, 1, 0, int(greedy), int(tc), self.seed, env_id0, self._kind,
                            N.POLICY_FLAG_RELU if self._relu else 0)
        io = N.PolicyIO()
        io.n_envs = B
        if tc:
            io.tc_weights = N.ptr(self.tc_weight_blob())          # (refreshes the fp32 blob as well)
            io.error_flag = N.ptr(self._tc_error)
            io.weights = N.ptr(self._blob)
            ws = self._workspace.get((env_id0, B))
            if ws is None:
                ws = self._workspace[(env_id0, B)] = torch.empty(N.lib().cm_policy_cent_workspace_bytes(B) // 4, dtype=torch.float32,
                                                                 device=self.device)
            io.workspace, io.workspace_bytes = N.ptr(ws), ws.numel() * 4
        else:
            io.weights = N.ptr(self.weight_blob())
        for k, v in (("obs", obs), ("avail_bits", avail_bits), ("sample_u", sample_u), ("tick", tick), ("episode", episode),
                     ("probs", probs), ("logits", logits), ("actions", actions)):
            setattr(io, k, N.ptr(v))
        return desc, io

    # ---- reference call surface ----
    def forward(self, obs_n, avail_actions_n, get_actions=False):
        if get_actions:
            obs_n = torch.as_tensor(np.asarray(obs_n), dtype=torch.float32, device=self.device)
            avail_actions_n = torch.as_tensor(np.asarray(avail_actions_n), dtype=torch.float32, device=self.device)
        x = obs_n
        for layer in self._layers:
            x = torch.relu(layer(x)) if self._relu else torch.tanh(layer(x))
        logits = self._output_layers[0](x)
        logits = logits.reshape(logits.shape[:-1] + (self._n_agents, -1))
        probs = torch.softmax(logits, dim=-1)
        avail = avail_actions_n.reshape(avail_actions_n.shape[:-1] + (self._n_agents, -1))
        masked = probs * avail
        masked = masked / masked.sum(dim=-1, keepdim=True)
        return Categorical(probs=masked.cpu() if get_actions else masked)

    _host_calls = 0
    get_actions = DecCategoricalMLPPolicy.get_actions

    def log_likelihood(self, observations, avail_actions_n, actions):
        return self.forward(observations, avail_actions_n).log_prob(actions).sum(axis=-1)

    def entropy(self, observations, avail_actions_n):
        return self.forward(observations, avail_actions_n).entropy().mean(axis=-1)

    def reset(self, dones=None):
        pass

    def grad_norm(self):
        return math.sqrt(sum(p.grad.norm(2).item() ** 2 for p in self.parameters() if p.grad is not None))

    @property
    def recurrent(self):
        return False


class PolicySet:
    """P policies of ONE class and architecture run by one ``cm_policy_forward`` launch per call — for evaluation (every
    checkpoint of a run, the seeds of a configuration).  The envs of a call are P equal contiguous blocks, block i runs
    ``policies[i]`` (one policy may fill several blocks).  The set owns one stacked fp32 buffer (and one stacked tensor-core
    buffer) with a row per block; ``refresh_weights`` (same signature and ``force`` semantics as the policies') copies a
    member's blobs into its rows when the member's parameters changed — in place, so a captured rollout graph over the set sees
    the update, and no other row changes.  The members' own blobs stay where they are: graphs captured on a member keep
    following it.  Equal architecture means the same class, team size, observation width, layers, residual, attention type,
    layer widths, kernel math and nonlinearity; anything else raises ValueError."""

    def __init__(self, policies):
        self.policies = list(policies)
        if not self.policies:
            raise ValueError("a PolicySet needs at least one policy")
        keys = [self._arch(p) for p in self.policies]
        for i, k in enumerate(keys[1:], 1):
            if k != keys[0]:
                raise ValueError(f"policies[{i}] differs in architecture from policies[0]: one launch runs one kernel")
        p0 = self.policies[0]
        self.device, self._kind, self.seed = p0.device, p0._kind, p0.seed
        P = len(self.policies)
        self._n_blob = p0.weight_blob().numel()
        self._stride = (self._n_blob + 3) // 4 * 4                # the bulk copies need 16-byte aligned rows
        self._blobs = torch.zeros((P, self._stride), dtype=torch.float32, device=self.device)
        self._tc_blobs, self._tc_stride, self._n_tc = None, 0, 0
        if p0.uses_tensor_cores():
            self._n_tc = p0.tc_weight_blob().numel()
            self._tc_stride = (self._n_tc + 3) // 4 * 4
            self._tc_blobs = torch.zeros((P, self._tc_stride), dtype=torch.float32, device=self.device)
        self._row_sig = [None] * P                 # member blob signature each row was copied at (None: copy pending)
        self.refresh_weights()

    @staticmethod
    def _arch(p):
        shapes = tuple((k, tuple(v.shape)) for k, v in p.state_dict().items())
        math = "tc" if p.uses_tensor_cores() else "fp32"       # CENT's two maths; 'auto' = the kernel it picked
        return (type(p), p._n_agents, p._dec_obs_dim, getattr(p, "n_gcn_layers", 0), getattr(p, "residual", False), math,
                getattr(p, "_relu", False), shapes)

    def __len__(self):
        return len(self.policies)

    def uses_tensor_cores(self):
        return self.policies[0].uses_tensor_cores()

    def _sync_row(self, i):
        """bring row i up to date with member i (its blobs refreshed first); one device copy per blob when it changed"""
        p = self.policies[i]
        if self._tc_blobs is not None:
            p.tc_weight_blob()                     # (refreshes the fp32 blob as well)
        else:
            p.weight_blob()
        if self._row_sig[i] != p._blob_sig:
            self._blobs[i, :self._n_blob].copy_(p._blob)
            if self._tc_blobs is not None:
                self._tc_blobs[i, :self._n_tc].copy_(p._tc_blob)
            self._row_sig[i] = p._blob_sig

    def refresh_weights(self, force=False):
        """the rows of every member whose parameters changed since the last refresh (``force``: every row, and every member's
        own blobs rebuilt — after a write through ``p.data``, see CommCategoricalMLPPolicy.refresh_weights)"""
        if force:
            for p in self.policies:
                p.refresh_weights(force=True)
            self._row_sig = [None] * len(self.policies)
        for i in range(len(self.policies)):
            self._sync_row(i)

    def check_errors(self):
        for p in self.policies:
            p.check_errors()

    @staticmethod
    def segments(B, envs_per_policy, first_env=0):
        """[(s0, s1, first block, whole blocks)] of a call over envs first_env .. first_env + B of a policy-major batch: runs of
        >= 2 whole blocks are one multi-policy launch (whole blocks > 0), a block the range cuts or a single block is one
        single-policy launch of its member (whole blocks = 0)"""
        Ep, out, s0 = int(envs_per_policy), [], 0
        while s0 < B:
            i, off = divmod(first_env + s0, Ep)
            if off == 0 and B - s0 >= 2 * Ep:
                s1 = s0 + (B - s0) // Ep * Ep
                out.append((s0, s1, i, (s1 - s0) // Ep))
            else:
                s1 = min(B, s0 + Ep - off)
                out.append((s0, s1, i, 0))
            s0 = s1
        return out

    def act_device(self, obs, adj_bits=None, chan_bits=None, avail_bits=None, sample_u=None, tick=None, episode=None,
                   greedy=False, probs=None, logits=None, attention=None, actions=None, env_id0=0, ws_slot=0, obs_bits=None,
                   obs_nbits=0, envs_per_policy=None, first_env=0):
        """``act_device`` of the members over policy-major envs.  By default the B envs of the call are P blocks of B / P;
        a call over a slice of a larger batch (a rollout group) gives ``envs_per_policy`` of the batch and ``first_env``,
        the slice's first env in it.  Runs of whole blocks are one multi-policy launch; a block the slice cuts runs as a
        single-policy launch of its member (PolicySet.segments).  Returns the number of cm_policy_forward calls made."""
        P, B = len(self.policies), obs.shape[0]
        Ep = B // P if envs_per_policy is None else int(envs_per_policy)
        if envs_per_policy is None and B != P * Ep:
            raise ValueError(f"{B} envs do not split into {P} equal policy blocks")
        args = dict(obs=obs, adj_bits=adj_bits, chan_bits=chan_bits, avail_bits=avail_bits, sample_u=sample_u, tick=tick,
                    episode=episode, probs=probs, logits=logits, attention=attention, actions=actions, obs_bits=obs_bits)
        segs = self.segments(B, Ep, first_env)
        for s0, s1, i, whole in segs:
            seg = {k: (v[s0:s1] if v is not None else None) for k, v in args.items()}
            if whole:
                self._launch(seg, greedy, env_id0 + s0, ws_slot, obs_nbits, whole, Ep, i)
            else:
                self._member_call(self.policies[i], seg, greedy, env_id0 + s0, ws_slot, obs_nbits)
        return len(segs)

    def _member_call(self, p, seg, greedy, env_id0, ws_slot, obs_nbits):
        kw = dict(avail_bits=seg["avail_bits"], sample_u=seg["sample_u"], tick=seg["tick"], episode=seg["episode"], greedy=greedy,
                  probs=seg["probs"], logits=seg["logits"], actions=seg["actions"], env_id0=env_id0)
        if self._kind == N.POLICY_COMM:
            p.act_device(seg["obs"], adj_bits=seg["adj_bits"], chan_bits=seg["chan_bits"], attention=seg["attention"],
                         ws_slot=ws_slot, obs_bits=seg["obs_bits"], obs_nbits=obs_nbits, **kw)
        elif self._kind == N.POLICY_DEC:
            p.act_device(seg["obs"], obs_bits=seg["obs_bits"], obs_nbits=obs_nbits, **kw)
        else:
            p.act_device(seg["obs"], **kw)

    def _launch(self, seg, greedy, env_id0, ws_slot, obs_nbits, n_blocks, Ep, first_policy):
        """one cm_policy_forward over n_blocks whole blocks of Ep envs, policies first_policy ..."""
        p0 = self.policies[first_policy]
        comm = self._kind == N.POLICY_COMM
        desc, io = p0._call_structs(seg["obs"], seg["adj_bits"] if comm else None, seg["chan_bits"] if comm else None,
                                    seg["avail_bits"], seg["sample_u"], seg["tick"], seg["episode"], greedy, seg["probs"],
                                    seg["logits"], seg["attention"] if comm else None, seg["actions"], env_id0, ws_slot)
        for i in range(first_policy, first_policy + n_blocks):
            self._sync_row(i)
        io.weights = N.ptr(self._blobs[first_policy])
        if self._tc_blobs is not None:
            io.tc_weights = N.ptr(self._tc_blobs[first_policy])
        io.n_policies, io.envs_per_policy = n_blocks, Ep
        io.weights_stride, io.tc_weights_stride = self._stride, self._tc_stride
        if seg["obs_bits"] is not None and self._kind != N.POLICY_CENT and self.uses_tensor_cores():
            io.obs_bits, io.obs_nbits = N.ptr(seg["obs_bits"]), int(obs_nbits)
        with torch.cuda.device(self.device):
            N.check("cm_policy_forward", N.lib().cm_policy_forward(C.byref(desc), C.byref(io), N.stream_ptr()))
