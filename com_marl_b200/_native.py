"""ctypes binding of the C ABI (include/commarl_b200.h) — the only way Python reaches the kernels.

There is deliberately no fallback: if ``lib/libcommarl_b200.so`` is missing or a call fails, this
module raises.  Build the library with ``python -c "import __graft_entry__ as g; g.build()"`` or
``python -m com_marl_b200.build``.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("COM_MARL_B200_LIB") or os.path.join(_HERE, "lib", "libcommarl_b200.so")

CM_OK, CM_EINVAL, CM_EUNSUPPORTED, CM_ECUDA, CM_ENODEVICE, CM_EACTION = 0, -1, -2, -3, -4, -5
PREDATOR_PREY, COVERAGE = 0, 1
CH_FC, CH_FL, CH_IID, CH_GE = 0, 1, 2, 3
POLICY_COMM, POLICY_DEC, POLICY_CENT = 0, 1, 2
POLICY_FLAG_RELU = 1
MAX_AGENTS, MAX_GRID, MAX_LAYERS = 256, 64, 4
ABI_VERSION = 8
MAX_CONDS = 256

EXPORTS = ("cm_abi_version", "cm_strerror", "cm_last_cuda_error", "cm_device_count", "cm_env_reset", "cm_env_step",
           "cm_comm_update", "cm_policy_forward", "cm_policy_blob_floats", "cm_policy_cent_blob_floats", "cm_policy_cent_tc_blob_floats", "cm_policy_cent_workspace_bytes", "cm_policy_workspace_bytes", "cm_policy_tc_blob_floats", "cm_policy_tc_prepare", "cm_mask_pack",
           "cm_mask_unpack", "cm_policy_forward_host", "cm_env_step_host", "cm_env_reset_host", "cm_rollout_step_host", "cm_ppo_advantages",
           "cm_adam_step", "cm_adam_step_dev", "cm_critic_blob_floats", "cm_baseline_mlp_blob_floats", "cm_ppo_net_workspace_floats",
           "cm_ppo_net", "cm_adam_step_set")
NET_POLICY, NET_CRITIC, NET_POLICY_DEC, NET_POLICY_CENT, NET_BASELINE_MLP = 0, 1, 2, 3, 4
NET_FLAG_RELU = 1


class EnvDesc(C.Structure):
    _fields_ = [(k, C.c_int32) for k in ("scenario", "n_agents", "n_preys", "grid", "sensing", "max_steps",
                                         "max_path_length", "load", "n_layers", "n_empty_cells", "rcom2", "channel",
                                         "loss_apply", "ge_init")] + \
               [(k, C.c_float) for k in ("p_loss", "pgb", "pbg", "ge_bad_rate")] + \
               [(k, C.c_double) for k in ("capture_reward", "step_cost", "moving_cost", "penalty", "lazy_penalty",
                                          "revisit_penalty", "final_reward")] + \
               [("seed", C.c_uint64), ("env_id0", C.c_int64), ("wall_rows", C.c_void_p), ("lut", C.c_void_p),
                ("conds", C.c_void_p), ("cond_idx", C.c_void_p), ("n_conds", C.c_int32), ("conds_host", C.c_void_p)]


class ChannelCond(C.Structure):
    _fields_ = [("channel", C.c_int32), ("rcom2", C.c_int32)] + \
               [(k, C.c_float) for k in ("p_loss", "pgb", "pbg", "ge_bad_rate")] + [("ge_init", C.c_int32)]


class EnvState(C.Structure):
    _fields_ = [("n_envs", C.c_int64)] + \
               [(k, C.c_void_p) for k in ("agent_pos", "prey_pos", "prey_alive", "visited", "step_count",
                                          "total_capture", "success", "episode", "tick", "ge_state")]


class StepIO(C.Structure):
    _fields_ = [("actions", C.c_void_p), ("prey_cand", C.c_void_p), ("spawn_agent", C.c_void_p),
                ("spawn_prey", C.c_void_p), ("spawn_episodes", C.c_int32), ("chan_u", C.c_void_p),
                ("chan_planes", C.c_int32), ("auto_reset", C.c_int32), ("obs", C.c_void_p), ("reward", C.c_void_p),
                ("done", C.c_void_p), ("counts", C.c_void_p), ("prey_alive_out", C.c_void_p),
                ("success_out", C.c_void_p), ("adj_bits", C.c_void_p), ("chan_bits", C.c_void_p), ("ave_deg", C.c_void_p),
                ("error_flag", C.c_void_p), ("stats", C.c_void_p), ("obs_bits", C.c_void_p), ("host_arena", C.c_int32)]


class PolicyDesc(C.Structure):
    _fields_ = [("n_agents", C.c_int32), ("obs_dim", C.c_int32), ("n_layers", C.c_int32), ("residual", C.c_int32),
                ("greedy", C.c_int32), ("math", C.c_int32), ("seed", C.c_uint64), ("env_id0", C.c_int64),
                ("kind", C.c_int32), ("flags", C.c_int32)]


class PolicyIO(C.Structure):
    _fields_ = [("n_envs", C.c_int64)] + \
               [(k, C.c_void_p) for k in ("weights", "obs", "adj_bits", "chan_bits", "avail_bits", "sample_u", "tick",
                                          "episode", "probs", "logits", "attention", "actions", "tc_weights",
                                          "error_flag", "workspace")] + \
               [("workspace_bytes", C.c_size_t), ("obs_bits", C.c_void_p), ("obs_nbits", C.c_int32), ("host_arena", C.c_int32)] + \
               [("n_policies", C.c_int32), ("envs_per_policy", C.c_int64), ("weights_stride", C.c_int64), ("tc_weights_stride", C.c_int64)]


class NetDesc(C.Structure):
    _fields_ = [(k, C.c_int32) for k in ("kind", "n_agents", "obs_dim", "n_layers", "residual")] + \
               [(k, C.c_float) for k in ("ent_coeff", "clip_lo", "clip_hi")] + [("flags", C.c_int32)]


class NetIO(C.Structure):
    _fields_ = [("n_steps", C.c_int64)] + \
               [(k, C.c_void_p) for k in ("weights", "grad", "obs", "adj_bits", "chan_bits", "avail_bits", "actions", "adv", "old_ll",
                                          "valid", "returns")] + \
               [("inv_count", C.c_float)] + \
               [(k, C.c_void_p) for k in ("ll", "entropy", "probs", "values", "loss", "workspace")] + \
               [("workspace_floats", C.c_size_t)] + \
               [("n_policies", C.c_int32), ("steps_per_policy", C.c_int64), ("weights_stride", C.c_int64), ("grad_stride", C.c_int64),
                ("inv_counts", C.c_void_p)]


def net_set_workspace_extra(n_policies):
    """floats a cm_ppo_net call over a set of n_policies networks needs beyond cm_ppo_net_workspace_floats (per-member loss sums)"""
    return ((2 * max(int(n_policies), 1) + 3) & ~3) - 4


class NativeError(RuntimeError):
    def __init__(self, fn, code, msg):
        super().__init__(f"{fn} failed: {code} ({msg})")
        self.code = code


_lib = None


def lib():
    """Loads the shared library (once).  Raises if it has not been built — there is no CPU path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: the CUDA library has not been built "
                          "(run __graft_entry__.build()); com_marl_b200 has no CPU fallback")
    L = C.CDLL(LIB_PATH)
    L.cm_abi_version.restype = C.c_int
    L.cm_strerror.restype = C.c_char_p
    L.cm_strerror.argtypes = [C.c_int]
    L.cm_last_cuda_error.restype = C.c_int
    L.cm_device_count.restype = C.c_int
    L.cm_env_reset.argtypes = [C.POINTER(EnvDesc), C.POINTER(EnvState), C.POINTER(StepIO), C.c_void_p, C.c_void_p]
    L.cm_env_step.argtypes = [C.POINTER(EnvDesc), C.POINTER(EnvState), C.POINTER(StepIO), C.c_void_p]
    L.cm_comm_update.argtypes = [C.POINTER(EnvDesc), C.POINTER(EnvState), C.POINTER(StepIO), C.c_int, C.c_void_p]
    L.cm_policy_forward.argtypes = [C.POINTER(PolicyDesc), C.POINTER(PolicyIO), C.c_void_p]
    L.cm_policy_blob_floats.restype = C.c_size_t
    L.cm_policy_blob_floats.argtypes = [C.c_int32, C.c_int32]
    L.cm_policy_cent_blob_floats.restype = C.c_size_t
    L.cm_policy_cent_blob_floats.argtypes = [C.c_int32, C.c_int32]
    L.cm_policy_cent_tc_blob_floats.restype = C.c_size_t
    L.cm_policy_cent_tc_blob_floats.argtypes = [C.c_int32, C.c_int32]
    L.cm_policy_cent_workspace_bytes.restype = C.c_size_t
    L.cm_policy_cent_workspace_bytes.argtypes = [C.c_int64]
    L.cm_policy_tc_blob_floats.restype = C.c_size_t
    L.cm_policy_tc_blob_floats.argtypes = [C.c_int32, C.c_int32]
    L.cm_policy_tc_prepare.restype = C.c_int
    L.cm_policy_tc_prepare.argtypes = [C.POINTER(PolicyDesc), C.c_void_p, C.c_void_p, C.c_void_p]
    L.cm_policy_workspace_bytes.restype = C.c_size_t
    L.cm_policy_workspace_bytes.argtypes = [C.c_int32, C.c_int64]
    L.cm_mask_pack.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]
    L.cm_mask_unpack.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]
    L.cm_policy_forward_host.argtypes = [C.POINTER(PolicyDesc), C.POINTER(PolicyIO), C.POINTER(PolicyIO), C.c_int64, C.c_void_p]
    L.cm_env_step_host.argtypes = [C.POINTER(EnvDesc), C.POINTER(EnvState), C.POINTER(StepIO), C.POINTER(StepIO), C.c_void_p]
    L.cm_env_reset_host.argtypes = [C.POINTER(EnvDesc), C.POINTER(EnvState), C.POINTER(StepIO), C.POINTER(StepIO), C.c_void_p]
    L.cm_rollout_step_host.argtypes = [C.POINTER(PolicyDesc), C.POINTER(PolicyIO), C.POINTER(PolicyIO), C.POINTER(EnvDesc),
                                       C.POINTER(EnvState), C.POINTER(StepIO), C.POINTER(StepIO), C.c_void_p]
    L.cm_ppo_advantages.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_float, C.c_float, C.c_int32,
                                    C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.cm_adam_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_float, C.c_float,
                               C.c_float, C.c_int32, C.c_float, C.c_void_p]
    L.cm_adam_step_dev.restype = C.c_int
    L.cm_adam_step_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_float, C.c_float,
                                   C.c_float, C.c_int32, C.c_void_p, C.c_void_p]
    L.cm_critic_blob_floats.restype = C.c_size_t
    L.cm_critic_blob_floats.argtypes = [C.c_int32, C.c_int32]
    L.cm_baseline_mlp_blob_floats.restype = C.c_size_t
    L.cm_baseline_mlp_blob_floats.argtypes = [C.c_int32]
    L.cm_ppo_net_workspace_floats.restype = C.c_size_t
    L.cm_ppo_net_workspace_floats.argtypes = [C.POINTER(NetDesc), C.c_int64, C.c_int32]
    L.cm_ppo_net.restype = C.c_int
    L.cm_ppo_net.argtypes = [C.POINTER(NetDesc), C.POINTER(NetIO), C.c_void_p]
    L.cm_adam_step_set.restype = C.c_int
    L.cm_adam_step_set.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_int64, C.c_float,
                                   C.c_float, C.c_float, C.c_float, C.POINTER(C.c_int32), C.c_void_p, C.c_void_p]
    for fn in ("cm_env_reset", "cm_env_step", "cm_comm_update", "cm_policy_forward", "cm_mask_pack", "cm_mask_unpack",
               "cm_policy_forward_host", "cm_env_step_host", "cm_env_reset_host", "cm_rollout_step_host", "cm_ppo_advantages", "cm_adam_step"):
        getattr(L, fn).restype = C.c_int
    if L.cm_abi_version() != ABI_VERSION:
        raise ImportError("libcommarl_b200.so ABI version mismatch")
    _lib = L
    return L


def check(fn, rc):
    if rc != CM_OK:
        L = lib()
        msg = L.cm_strerror(rc).decode()
        if rc == CM_ECUDA:
            msg += f", cudaError={L.cm_last_cuda_error()}"
        raise NativeError(fn, rc, msg)


def arena(specs, device=None, pinned=False, align=256):
    """Tensors carved from ONE allocation: specs = [(name, shape, dtype)] -> {name: tensor}.  Arrays that travel together
    between host and device live in arenas with the same order and padding on both sides, so the host-buffer calls of the
    library move them with a single DMA transfer (csrc/host_abi.cu merges adjacent copies)."""
    import torch
    offs, total = [], 0
    for _, shape, dt in specs:
        nbytes = int(torch.empty((), dtype=dt).element_size())
        for d in shape:
            nbytes *= int(d)
        offs.append((total, nbytes))
        total += (nbytes + align - 1) // align * align
    buf = torch.zeros(max(total, align), dtype=torch.uint8, pin_memory=True) if pinned else \
        torch.zeros(max(total, align), dtype=torch.uint8, device=device)
    out = {}
    for (name, shape, dt), (o, nbytes) in zip(specs, offs):
        out[name] = buf[o:o + nbytes].view(dt).view(tuple(int(d) for d in shape))
    out["_arena"] = buf
    return out


def ptr(t):
    """device pointer of a torch tensor (or None)"""
    return None if t is None else t.data_ptr()


def stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream
