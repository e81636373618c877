/*
 * commarl_b200.h — C ABI of the B200-native batched rollout engine for Com-MARL.
 *
 * The reference (cnuns/Com-MARL) is 100 % Python and has no FFI/plugin layer (SURVEY.md §8b); its
 * rollout path is reached through three duck-typed Python interfaces.  This header is the thin C
 * boundary underneath our Python mirror of those interfaces (com_marl_b200/).  Each entry point names
 * the reference code it replaces.  Conventions (all entry points):
 *
 *   - extern "C", plain pointers and sizes only; no torch / C++ types.
 *   - every pointer inside cm_env_state / cm_step_io / cm_policy_io is a DEVICE pointer owned by the
 *     caller (the Python side hands in torch tensor data_ptr()s); descriptors are HOST structs read at
 *     call time.  The library never allocates, never synchronises, never touches a global/default
 *     stream: work is enqueued on the given stream (a cudaStream_t) and is CUDA-graph capturable.
 *   - returns CM_OK (0) or a negative cm_error; never throws.  cm_strerror() names the code.
 *   - there is no CPU path: without a device every compute call returns CM_ENODEVICE.
 *
 * Data layout (device, SoA, env-major, one row of each array per environment instance):
 *   agent_pos  u16 [B][n]     row | col << 8            (PredatorPrey: 0..map-1, Coverage: 1..map)
 *   prey_pos   u16 [B][p]     same packing; stale for dead preys, like the reference's prey_pos dict
 *   prey_alive u8  [B][p]
 *   visited    u64 [B][G]     Coverage visited map, one 64-bit word per grid row, bit c = column c
 *   step_count i32 [B]        env._step_count
 *   total_capture i32 [B]     Coverage.total_capture_cnt
 *   success    u8  [B]        env.success, latched exactly like the reference (coverage.py:385-390 quirk)
 *   episode    u32 [B]        number of resets so far (RNG key + index into an injected spawn queue)
 *   tick       u32 [B]        steps since creation, never reset (RNG key)
 *   ge_state   u32 [B][n][W]  last Gilbert-Elliot link state, bit j of word j/32 of row i;  W = ceil(n/32)
 * Outputs of a step / reset:
 *   obs        f32 [B][n][D]  == np.concatenate(obs_n) of the wrappers (predatorprey_wrapper.py:61-66)
 *   reward     f64 [B]        fp64, reference evaluation order
 *   done       u8  [B]        np.all(dones) | time limit (vec_env_executor.py:33-35)
 *   counts     i32 [B][6]     PP: capture, moved, penalty, watching, 0, 0;  CO: capture, moved, penalty,
 *                              revisit, lazy, 0 — the integer sums the reference's reward_details are means of
 *   prey_alive_out u8 [B][p]  env_infos['prey_alive'] of the step (pre-reset)
 *   adj_bits   u32 [B][n][W]  dist_adj rows as bit masks
 *   chan_bits  u32 [B][L][n][W] channels[l] rows as bit masks
 *   ave_deg    f32 [B]
 */
#ifndef COMMARL_B200_H_
#define COMMARL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CM_ABI_VERSION 8   /* 2: host_arena / obs_bits members, cm_rollout_step_host; 3: cm_ppo_net; 4: CENT kinds of cm_ppo_net,
                              cm_net_desc.flags; 5: cm_channel_cond, per-env channel conditions (cm_env_desc.conds ...);
                              6: several policies in one cm_policy_forward (cm_policy_io.n_policies ...);
                              7: several networks in one cm_ppo_net (cm_net_io.n_policies ...), cm_adam_step_set;
                              8: Comm-DP / Obs-DP take math = 1 only */
#define CM_MAX_AGENTS 256   /* n, p */
#define CM_MAX_GRID 64      /* grid side incl. Coverage's wall border */
#define CM_MAX_LAYERS 4     /* n_gcn_layers */
#define CM_ACTIONS 5

typedef void *cm_stream_t;  /* cudaStream_t */

enum cm_scenario { CM_PREDATOR_PREY = 0, CM_COVERAGE = 1 };
enum cm_channel { CM_CH_FC = 0, CM_CH_FL = 1, CM_CH_IID = 2, CM_CH_GE = 3 };
enum cm_error {
    CM_OK = 0,
    CM_EINVAL = -1,       /* null pointer / bad size */
    CM_EUNSUPPORTED = -2, /* n > CM_MAX_AGENTS, grid > CM_MAX_GRID, load not in {2,3,4}, GE_INIT=-1 with loss_apply=0 ... */
    CM_ECUDA = -3,        /* a CUDA runtime call failed; cm_last_cuda_error() has the code */
    CM_ENODEVICE = -4,
    CM_EACTION = -5       /* an action outside 0..4 was seen ('Action Not found!', predator_prey.py:255) */
};

/* One channel condition: the members of cm_env_desc of the same names, with the same meaning and float32 rounding. */
typedef struct cm_channel_cond {
    int32_t channel;           /* cm_channel */
    int32_t rcom2;
    float p_loss;
    float pgb, pbg;
    float ge_bad_rate;
    int32_t ge_init;
} cm_channel_cond;
#define CM_MAX_CONDS 256

/* Scenario description (host).  Replaces the attribute soup PredatorPrey.__init__ / Coverage.__init__ /
 * init_communication build from `params` (predator_prey.py:51-108, coverage.py:39-109,
 * env_communication.py:10-77). */
typedef struct cm_env_desc {
    int32_t scenario;          /* cm_scenario */
    int32_t n_agents;          /* n */
    int32_t n_preys;           /* p (PredatorPrey) */
    int32_t grid;              /* G: map (PredatorPrey) or map + 2 (Coverage, wall border included) */
    int32_t sensing;           /* Rsen */
    int32_t max_steps;         /* T = env._max_steps */
    int32_t max_path_length;   /* VecEnvExecutor time limit; 0 = none */
    int32_t load;              /* PredatorPrey capture load: 2 -> reward_default, 3/4 -> reward_individual */
    int32_t n_layers;          /* L = n_gcn_layers */
    int32_t n_empty_cells;     /* Coverage: free cells - n (coverage.py:228-230) */
    int32_t rcom2;             /* 2*Rcom^2, adjacency <=> dr^2+dc^2 <= rcom2; -1 = fully connected (Rcom == 0) */
    int32_t channel;           /* cm_channel */
    int32_t loss_apply;        /* GE: 1 = a transition per GCN layer, 0 = one per env step */
    int32_t ge_init;           /* GE_INIT: 1 good, 0 bad, -1 proportional */
    float p_loss;              /* IID: float32(Ploss) */
    float pgb, pbg;            /* GE: float32(Pgb), float32(Pbg) */
    float ge_bad_rate;         /* GE: float32(Pgb / (Pgb + Pbg)) */
    double capture_reward, step_cost, moving_cost, penalty, lazy_penalty, revisit_penalty, final_reward;
                               /* signed as the reference stores them (predator_prey.py:66-69, coverage.py:86-92) */
    uint64_t seed;             /* Philox key for generated streams */
    int64_t env_id0;           /* global id of env 0 of this shard: results do not depend on the sharding */
    const uint64_t *wall_rows; /* DEVICE u64 [G]: Coverage wall bitmap rows (border + obstacles); NULL for PredatorPrey */
    const float *lut;          /* DEVICE f32 [G + G + T + 1]: obs scalar features row[r], col[c], time[t] */
    /* Per-env channel conditions (ABI 5; zero = NULL = one condition per launch, the members above).  Env b communicates
     * under conds[cond_idx[b]] instead of the descriptor's channel, rcom2, p_loss, pgb, pbg, ge_bad_rate and ge_init; every
     * other member stays uniform across the launch.  One launch may mix FC, FL, IID and GE (the reference's test-mode grid
     * of loss rate x Rcom x channel model).  Every entry is validated like the descriptor's own channel (GE_INIT = -1 with
     * loss_apply = 0 -> CM_EUNSUPPORTED; ge_state needed when an entry is GE; injected chan_u must hold the largest plane
     * count of any entry).  Validation reads conds_host, which the caller keeps equal to the device table, so that the call
     * never synchronises.  A cond_idx value >= n_conds reads entry 0 and sets io.error_flag to CM_EINVAL. */
    const cm_channel_cond *conds;      /* DEVICE [n_conds] */
    const uint8_t *cond_idx;           /* DEVICE [B] */
    int32_t n_conds;                   /* 1 .. CM_MAX_CONDS */
    const cm_channel_cond *conds_host; /* HOST copy of conds, read at call time */
} cm_env_desc;

typedef struct cm_env_state {
    int64_t n_envs;            /* B */
    uint16_t *agent_pos;
    uint16_t *prey_pos;
    uint8_t *prey_alive;
    uint64_t *visited;
    int32_t *step_count;
    int32_t *total_capture;
    uint8_t *success;
    uint32_t *episode;
    uint32_t *tick;
    uint32_t *ge_state;
} cm_env_state;

typedef struct cm_step_io {
    /* inputs */
    const int8_t *actions;     /* [B][n] (step only) */
    const int8_t *prey_cand;   /* [B][p][5] pre-drawn prey-move candidates, or NULL -> Philox */
    const uint16_t *spawn_agent; /* [B][E][n] injected spawn queue (packed like agent_pos), or NULL -> Philox */
    const uint16_t *spawn_prey;  /* [B][E][p] */
    int32_t spawn_episodes;    /* E */
    const float *chan_u;       /* [B][planes][n][n] pre-drawn channel uniforms, or NULL -> Philox */
    int32_t chan_planes;
    int32_t auto_reset;        /* 1: reset finished envs inside the step (VecEnvExecutor), obs/comm are post-reset */
    /* outputs (any may be NULL to skip, except where noted) */
    float *obs;
    double *reward;
    uint8_t *done;
    int32_t *counts;
    uint8_t *prey_alive_out;
    uint8_t *success_out;      /* [B] env.success as the sampler reads it when the step reports done */
    uint32_t *adj_bits;
    uint32_t *chan_bits;
    float *ave_deg;
    int32_t *error_flag;       /* DEVICE i32[1]: set to CM_EACTION when an invalid action is seen (optional) */
    double *stats;             /* [B][16] per-env episode accounting updated by every step (optional):
                                  running  [0] return [1] length [2..6] counts[0..4]
                                  finished [7] episodes [8] return sum [9] length sum [10] success sum [11..15] counts sums
                                  — the sums behind AverageReturn / SuccessRate / AverageCaptureCount ... that
                                  centralized_ma_ppo.py:345-372 logs from `paths` */
    uint32_t *obs_bits;        /* optional [B][n][6] u32: the same observation PACKED — words 0..2: the 0/1 window columns as bits (bit k
                                  of the 96-bit string = obs column k, k < obs_nbits = D - 3 (PredatorPrey) / D - 2 (Coverage)), words
                                  3..5: the remaining scalar columns as float bits.  24 bytes per agent instead of 4 D; cm_policy_forward
                                  reads it instead of `obs` when given (cm_policy_io.obs_bits) */
    int32_t host_arena;        /* read from the `host` struct of the *_host calls only.  Non-zero = the caller declares that the
                                  non-NULL buffers of that struct are carved from ONE host arena in the member order the call
                                  copies them, with the same padding (<= 1 KB) as the buffers of the `dev` struct: the library
                                  may then move neighbouring arrays, padding bytes included, with a single DMA transfer.
                                  0 = unrelated caller buffers: one transfer per array, nothing outside them is touched */
} cm_step_io;

/* Weight blob of CommCategoricalMLPPolicy (comm_categorical_mlp_policy.py + comm_base_net.py), float32,
 * every dense weight stored K-major ([in][out]) so that a warp reads consecutive output columns:
 *   enc_w1 [D][H1]  enc_b1 [H1]  enc_w2 [H1][E]  enc_b2 [E]  att_w [E][E]
 *   gcn_w[l] [E][E]  gcn_b[l] [E]    for l < L
 *   head_w1 [E][C1] head_b1 [C1] head_w2 [C1][C2] head_b2 [C2] head_w3 [C2][C3] head_b3 [C3] head_w4 [C3][5] head_b4 [5]
 * with the reference's default sizes H1=128, E=64, (C1,C2,C3)=(128,64,32); cm_policy_blob_floats() gives
 * the length, com_marl_b200.policy packs a reference state_dict into it. */
typedef struct cm_policy_desc {
    int32_t n_agents;          /* n */
    int32_t obs_dim;           /* D per agent */
    int32_t n_layers;          /* L */
    int32_t residual;          /* comm_categorical_mlp_policy.py:74-77 */
    int32_t greedy;            /* argmax instead of sampling (:109-112) */
    int32_t math;              /* Comm-DP / Obs-DP: 1 only (any other value: CM_EUNSUPPORTED) = tensor cores, error-compensated
                                  fp16 products (x = hi + lo) with fp32 accumulation: fp32-level accuracy; needs io.tc_weights.
                                  Teams with n <= 64: one fused tcgen05 kernel; larger teams: tcgen05 encoder -> attention /
                                  graph convolutions on mma.sync -> tcgen05 head, rows handed over through io.workspace.
                                  At most 2^23 agent rows (n_envs * n) per call; more return CM_EUNSUPPORTED.
                                  CENT: 0 or 1, see `kind` */
    uint64_t seed;
    int64_t env_id0;
    int32_t kind;              /* cm_policy_kind: 0 = Comm-DP (CommCategoricalMLPPolicy), 1 = Obs-DP (DecCategoricalMLPPolicy:
                                  per-agent encoder D -> 128 -> 64 (tanh) and head 64 -> 32 (tanh) -> 5, no communication;
                                  dec_categorical_mlp_policy.py:107-124).  Obs-DP uses the same blob layout with enc_w1/b1,
                                  enc_w2/b2, head_w3/b3, head_w4/b4 filled; tensor-core path only, any team size.
                                  2 = CENT (CentralizedCategoricalMLPPolicy, centralized_categorical_mlp_policy.py:11-97): one
                                  MLP n*D -> 128 -> 64 -> 32 -> 5n over the concatenated observation of the team, softmax per
                                  agent; its own blob (cm_policy_cent_blob_floats):
                                    w1 [n*D][128] b1 [128] w2 [128][64] b2 [64] w3 [64][32] b3 [32] w4 [32][5n] b4 [5n]
                                  math = 0: exact fp32; math = 1: the first layer (the one product whose K = n*D grows with the
                                  team) on the tcgen05 tensor cores with error-compensated fp16 operands, needs io.tc_weights
                                  (cm_policy_cent_tc_blob_floats, cm_policy_tc_prepare) and io.workspace
                                  (cm_policy_cent_workspace_bytes); n_layers / residual / masks / attention are not used */
    int32_t flags;             /* CM_POLICY_FLAG_*; CENT only */
} cm_policy_desc;

typedef enum cm_policy_kind { CM_POLICY_COMM = 0, CM_POLICY_DEC = 1, CM_POLICY_CENT = 2 } cm_policy_kind;
#define CM_POLICY_FLAG_RELU 1  /* hidden_nonlinearity = relu instead of tanh (runner_*_cent.py:49) */

typedef struct cm_policy_io {
    int64_t n_envs;            /* B */
    const float *weights;      /* blob described above */
    const float *obs;          /* [B][n][D] */
    const uint32_t *adj_bits;  /* [B][n][W] or NULL = all ones */
    const uint32_t *chan_bits; /* [B][L][n][W] or NULL = all ones */
    const uint8_t *avail_bits; /* [B][n] bit a = action a available, or NULL = all available */
    const float *sample_u;     /* [B][n] pre-drawn uniforms for action sampling, or NULL -> Philox(tick, episode) */
    const uint32_t *tick;      /* [B] RNG key words (the env state's arrays); may be NULL when sample_u or greedy */
    const uint32_t *episode;   /* [B] */
    float *probs;              /* [B][n][5] masked, renormalised action probabilities */
    float *logits;             /* [B][n][5] raw head output, or NULL */
    float *attention;          /* [B][n][n] unmasked attention softmax (agent_infos['attention_weights']), or NULL */
    int8_t *actions;           /* [B][n], or NULL */
    const float *tc_weights;   /* math == 1: blob written by cm_policy_tc_prepare() (cm_policy_tc_blob_floats() floats) */
    int32_t *error_flag;       /* DEVICE i32[1], optional: set when a bounded device-side wait times out */
    float *workspace;          /* Comm-DP teams with n > 64 only: cm_policy_workspace_bytes() bytes of scratch, 16-byte aligned:
                                  the E, Q and H_0 Wg_0 rows the large-team pipeline hands between its launches */
    size_t workspace_bytes;
    const uint32_t *obs_bits;  /* optional [B][n][6]: the packed observation cm_env_step writes (cm_step_io.obs_bits).  When given, the
                                  tensor-core kernels (math = 1) build their first operand from it — 24 bytes per agent row instead of
                                  4 D, the 0/1 columns need no low-order operand — and `obs` may be NULL; results are bit-identical */
    int32_t obs_nbits;         /* number of leading 0/1 columns in obs_bits (D - 3 / D - 2) */
    int32_t host_arena;        /* `host` struct of the *_host calls only; see cm_step_io.host_arena */
    /* Several policies of one kind and architecture in one launch (ABI 6; 0 or 1 = one policy, the members below are not read).
     * The envs are cut into n_policies contiguous blocks of envs_per_policy envs; env b runs the policy whose fp32 blob starts at
     * weights + (b / envs_per_policy) * weights_stride and whose cm_policy_tc_prepare blob (one prepare call per policy, at its
     * offset) starts at tc_weights + (b / envs_per_policy) * tc_weights_stride.  Every kernel counts its tiles per block, so no
     * tile holds rows of two policies.  Needs n_envs == n_policies * envs_per_policy, and each stride at least its blob's length
     * and a multiple of 4 floats (16-byte bulk copies); else CM_EINVAL.  The *_host calls return CM_EUNSUPPORTED. */
    int32_t n_policies;
    int64_t envs_per_policy;
    int64_t weights_stride;    /* floats */
    int64_t tc_weights_stride; /* floats; CENT with math = 0 does not read it */
} cm_policy_io;

int cm_abi_version(void);
const char *cm_strerror(int err);
int cm_last_cuda_error(void);
int cm_device_count(void);

/* env.reset() for the envs whose mask byte is non-zero (mask == NULL: all), followed by the observation
 * and update_communication_state of those envs.
 * Replaces PredatorPrey.reset / Coverage.reset (predator_prey.py:206-232, coverage.py:221-246) as
 * called by VecEnvExecutor.reset (vec_env_executor.py:47-54). */
int cm_env_reset(const cm_env_desc *desc, const cm_env_state *state, const cm_step_io *io,
                 const uint8_t *mask, cm_stream_t stream);

/* One VecEnvExecutor.step over all B envs (vec_env_executor.py:19-45): PredatorPrey.step /
 * Coverage.step (predator_prey.py:494-519, coverage.py:319-401), time limit, auto-reset, observation
 * windows (predator_prey.py:173-204, coverage.py:198-212,448-480) and update_communication_state
 * (env_communication.py:91-157: get_graph, FC/FL/IID/GE channels). */
int cm_env_step(const cm_env_desc *desc, const cm_env_state *state, const cm_step_io *io, cm_stream_t stream);

/* update_communication_state alone, from the positions currently in `state` (env_communication.py:91-157,
 * 200-243; gilbert_elliot_loss_model.py:84-87,121-150).  at_reset selects the GE (re)initialisation branch. */
int cm_comm_update(const cm_env_desc *desc, const cm_env_state *state, const cm_step_io *io, int at_reset,
                   cm_stream_t stream);

/* CommCategoricalMLPPolicy.forward(get_actions=True) + sampling for B envs in one fused kernel
 * (comm_categorical_mlp_policy.py:48-119, comm_base_net.py:80-108, attention_module.py:26-51,
 * graph_conv_module.py:51-72, categorical_mlp_module.py:64-80, multi_headed_mlp_module.py:134-149). */
int cm_policy_forward(const cm_policy_desc *desc, const cm_policy_io *io, cm_stream_t stream);
size_t cm_policy_blob_floats(int32_t obs_dim, int32_t n_layers);
/* CENT: CentralizedCategoricalMLPPolicy.forward(get_actions=True) + sampling through the same cm_policy_forward call
 * (desc.kind = CM_POLICY_CENT; centralized_categorical_mlp_policy.py:61-117); length of its weight blob in floats */
size_t cm_policy_cent_blob_floats(int32_t n_agents, int32_t obs_dim);
/* CENT with math = 1: floats of the prepared first-layer operand (cm_policy_tc_prepare with desc.kind = CM_POLICY_CENT writes it)
 * and bytes of scratch for the first layer's output rows */
size_t cm_policy_cent_tc_blob_floats(int32_t n_agents, int32_t obs_dim);
size_t cm_policy_cent_workspace_bytes(int64_t n_envs);
/* tcgen05 variant: re-lays the fp32 weight blob out as pre-split fp16 ([B_hi ; B_lo] stacked) K-major core-matrix
 * panels, one per tensor-core product, so that the kernel fetches a layer's B operand with one bulk async copy */
size_t cm_policy_tc_blob_floats(int32_t obs_dim, int32_t n_layers);
int cm_policy_tc_prepare(const cm_policy_desc *desc, const float *weights, float *tc_weights, cm_stream_t stream);
/* Comm-DP: bytes of scratch the forward needs for teams larger than one 64-row tile, 3 * n_envs * n_agents * 64 floats
 * (0 for n <= 64) */
size_t cm_policy_workspace_bytes(int32_t n_agents, int64_t n_envs);

/* ---- host-buffer calls: the reference-facing form of the three entry points above ------------------------------
 * The reference's callers hand NumPy arrays to env.step / policy.get_actions and get NumPy arrays back
 * (vec_env_executor.py:19-45, comm_categorical_mlp_policy.py:98-119).  These calls take TWO io structs of the same
 * type: `dev` exactly as for the device call (device staging buffers the kernel works on; weights / tc_weights /
 * workspace / error_flag / stats / spawn queues live only there) and `host`, whose non-NULL members are HOST buffers
 * (pinned, for the copies to be asynchronous) of the same shapes.  One call = H2D copies of the inputs named in `host`
 * -> the kernel -> D2H copies of the outputs named in `host`, all enqueued on `stream`; it never synchronises: wait
 * on the stream (or an event recorded after the call) before reading the host outputs.
 *   cm_policy_forward_host  inputs obs, adj_bits, chan_bits, avail_bits, sample_u, episode, tick; outputs actions, probs,
 *                           logits, attention.  tick_all >= 0 fills dev->tick with that value instead of copying host->tick
 *                           (the host loop's call counter as the sampling key).
 *   cm_env_step_host        input actions; outputs obs, adj_bits, chan_bits, reward, done, counts, prey_alive_out,
 *                           success_out, ave_deg.   cm_env_reset_host: the same outputs after a reset of all envs. */
int cm_policy_forward_host(const cm_policy_desc *desc, const cm_policy_io *dev, const cm_policy_io *host, int64_t tick_all,
                           cm_stream_t stream);
int cm_env_step_host(const cm_env_desc *desc, const cm_env_state *state, const cm_step_io *dev, const cm_step_io *host,
                     cm_stream_t stream);
int cm_env_reset_host(const cm_env_desc *desc, const cm_env_state *state, const cm_step_io *dev, const cm_step_io *host,
                      cm_stream_t stream);

/* One iteration of the sampler's loop for B envs as ONE call — the garage-sampler boundary
 * (CentralizedMAOnPolicyVectorizedSampler.obtain_samples, centralized_ma_on_policy_vectorized_sampler.py:119-231: read
 * dist_adj / channels / avail_actions of every env :123-131, policy.get_actions :134, vec_env.step :143, append to the
 * running paths :158-191).  Observations, masks and the env state stay on the device between calls — the policy reads
 * the observation / bit rows the previous step (or reset) left in pol_dev->obs / adj_bits / chan_bits, which must be the
 * buffers env_dev->obs / adj_bits / chan_bits point to — so NO observation travels host -> device:
 *   H2D   pol_host->avail_bits (the sampler's per-step get_avail_actions(), :128-131), when given;
 *   run   cm_policy_forward(pol_desc, pol_dev)  then  cm_env_step(env_desc, state, env_dev) with env_dev->actions ==
 *         pol_dev->actions;
 *   D2H   what the sampler appends per step, for every non-NULL member: pol_host->actions, probs, logits, attention;
 *         env_host->obs, adj_bits, chan_bits (the NEXT observation / communication state), reward, done, counts,
 *         prey_alive_out, success_out, ave_deg.
 * Asynchronous on `stream` like the other host calls. */
int cm_rollout_step_host(const cm_policy_desc *pol_desc, const cm_policy_io *pol_dev, const cm_policy_io *pol_host,
                         const cm_env_desc *env_desc, const cm_env_state *state, const cm_step_io *env_dev,
                         const cm_step_io *env_host, cm_stream_t stream);

/* ---- PPO update helpers (SURVEY.md 8f.1; the network forward / backward: cm_ppo_net below) ----
 * cm_ppo_advantages: rows of the padded [P][T] batch of CentralizedMAPPO.process_samples (centralized_ma_ppo.py:612-659):
 *   returns  = tensor_utils.discount_cumsum of the valid steps (garage/misc/tensor_utils.py:7-23; float64 recursion),
 *   raw_adv  = compute_advantages (garage/torch/algos/_utils.py:56-113) over the whole padded row, baselines of the
 *              padded tail included like the reference does,
 *   adv      = per-path normalisation with the mean / biased variance of the valid steps (center_adv,
 *              centralized_ma_ppo.py:425-429).  Any output may be NULL.
 * cm_adam_step: one step of the reference's Adam (my_optimizer/adam.py:57-120 -> functional adam; no amsgrad / weight
 *   decay) over a flat fp32 bucket, grads scaled by grad_scale (the clip_grad_norm_ coefficient) in the same pass. */
int cm_ppo_advantages(const double *rewards, const float *baselines, const int32_t *valids, int64_t n_paths, int32_t T,
                      float discount, float gae_lambda, int32_t center, float eps, float *returns, float *raw_adv, float *adv,
                      cm_stream_t stream);
int cm_adam_step(float *params, const float *grads, float *exp_avg, float *exp_avg_sq, int64_t n, float lr, float beta1,
                 float beta2, float eps, int32_t step, float grad_scale, cm_stream_t stream);
/* the same step with the gradient scale read from DEVICE memory (the clip_grad_norm_ coefficient as the norm reduction left it:
 * no host round trip between the backward pass and the optimizer step) */
int cm_adam_step_dev(float *params, const float *grads, float *exp_avg, float *exp_avg_sq, int64_t n, float lr, float beta1,
                     float beta2, float eps, int32_t step, const float *grad_scale_dev, cm_stream_t stream);
/* cm_adam_step_dev over a set of n_policies buckets in ONE launch: member i's n floats start at params / grads / exp_avg / exp_avg_sq
 * + i * stride (stride >= n floats).  steps: HOST [n_policies] step numbers (read at call time; the bias corrections are formed on
 * the host in double like cm_adam_step's); grad_scale_dev: DEVICE [n_policies] clip coefficients.  A member whose step number is 0
 * is not stepped: its parameters and moments stay bit for bit as they are.  Every stepped member's result is bit-identical to
 * cm_adam_step_dev on its row. */
int cm_adam_step_set(float *params, const float *grads, float *exp_avg, float *exp_avg_sq, int32_t n_policies, int64_t n,
                     int64_t stride, float lr, float beta1, float beta2, float eps, const int32_t *steps, const float *grad_scale_dev,
                     cm_stream_t stream);

/* ---- PPO update: hand-written forward + backward of the comm-GNN (csrc/ppo_net_kernels.cu) -----------------------------
 * cm_ppo_net runs ONE network over n_steps env steps of n agents each — the flattened (path, t) pairs of a minibatch of
 * CentralizedMAPPO.train_once (centralized_ma_ppo.py:207-262):
 *   kind = CM_NET_POLICY  CommCategoricalMLPPolicy.forward(get_actions=False) (comm_categorical_mlp_policy.py:48-96) followed by
 *                         _compute_loss / _compute_objective (centralized_ma_ppo.py:390-438, 540-589): joint log-likelihood of
 *                         the taken actions, mean entropy over the agents, ratio = exp(ll - old_ll), clipped surrogate
 *                         min(ratio adv, clip(ratio, clip_lo, clip_hi) adv) + ent_coeff entropy;  loss = -sum over the valid steps
 *                         * inv_count.  Weights / gradient in the layout of the rollout blob (cm_policy_blob_floats).
 *   kind = CM_NET_POLICY_DEC  DecCategoricalMLPPolicy.forward (dec_categorical_mlp_policy.py:107-124, 198-226: encoder D -> 128 -> 64,
 *                         head 64 -> 32 -> 5 per agent row, no masks) with the same objective; blob = the rollout blob of the Obs-DP
 *                         kind (enc_w1/b1, enc_w2/b2, head_w3/b3, head_w4/b4 filled, n_layers = 1).
 *   kind = CM_NET_CRITIC  CommBaseCritic.compute_loss (comm_base_critic.py:11-120): the same trunk, decoder 64 -> 64 (tanh) -> 1,
 *                         V(s) = sum over agents, loss = mean Gaussian negative log-likelihood of `returns` with the learnt
 *                         log-std (clamped at log 1e-6).  Blob (cm_critic_blob_floats): enc_w1 [D][128] enc_b1 enc_w2 [128][64]
 *                         enc_b2 att_w [64][64] gcn_w[l] [64][64] gcn_b[l] [64] dec_w1 [64][64] dec_b1 [64] dec_w2 [64] dec_b2 [1]
 *                         log_std [1], dense weights K-major like the policy blob.
 *   kind = CM_NET_POLICY_CENT  CentralizedCategoricalMLPPolicy.forward (centralized_categorical_mlp_policy.py:61-97, 122-137: one MLP
 *                         n*D -> 128 -> 64 -> 32 -> 5n over the concatenated observation of the team, act = tanh, or relu with
 *                         CM_NET_FLAG_RELU) followed by _compute_loss / _compute_objective: logits [S][5n] reshaped per agent, softmax,
 *                         availability mask, masked / masked.sum() (no + 1e-12), log-likelihood summed and entropy averaged over the
 *                         agents; the joint ratio and the clipped surrogate as for CM_NET_POLICY.  Blob = the rollout blob of the CENT
 *                         policy (cm_policy_cent_blob_floats).
 *   kind = CM_NET_BASELINE_MLP  GaussianMLPBaseline.compute_loss (gaussian_mlp_baseline.py:83-117): V(s) = MLP(obs[S][n*D]), three
 *                         tanh hidden layers of <= 64 units and a linear output of 1; loss = mean Gaussian negative log-likelihood over
 *                         EVERY step passed, std = exp(log_std) with no clamp.  Blob (cm_baseline_mlp_blob_floats(n*D)): w1 [n*D][64]
 *                         b1 [64] w2 [64][64] b2 [64] w3 [64][64] b3 [64] w4 [64] b4 [1] log_std [1], narrower layers zero-padded.
 *   For the two CENT kinds the rows of every product are env steps, io.obs [S][n][D] is read as [S][n*D], adj_bits / chan_bits
 *   and n_layers / residual are ignored, and n, D are limited as cm_policy_forward limits them for CM_POLICY_CENT.
 * grad == NULL: forward only (ll / entropy / probs / values / loss outputs).  grad != NULL: the parameter gradients of `loss`
 * are ADDED to grad (same layout as weights; the caller zeroes it) — exact fp32 like the autograd graph they replace.
 * Activations live in `workspace`; the steps are walked in chunks of as many steps as the workspace holds
 * (cm_ppo_net_workspace_floats(desc, chunk_steps, backward) floats hold one chunk).  Stream-ordered, capturable. */
typedef enum cm_net_kind {
    CM_NET_POLICY = 0, CM_NET_CRITIC = 1, CM_NET_POLICY_DEC = 2, CM_NET_POLICY_CENT = 3, CM_NET_BASELINE_MLP = 4
} cm_net_kind;
#define CM_NET_FLAG_RELU 1     /* CM_NET_POLICY_CENT: hidden_nonlinearity = relu instead of tanh (runner_*_cent.py:49) */
typedef struct cm_net_desc {
    int32_t kind;              /* cm_net_kind */
    int32_t n_agents, obs_dim, n_layers, residual;
    float ent_coeff;           /* policy_ent_coeff ('regularized'), 0 otherwise */
    float clip_lo, clip_hi;    /* 1 -/+ lr_clip_range (hard-coded 0.1 at centralized_ma_ppo.py:121) */
    int32_t flags;             /* CM_NET_FLAG_* */
} cm_net_desc;
typedef struct cm_net_io {
    int64_t n_steps;           /* S */
    const float *weights;      /* fp32 blob */
    float *grad;               /* or NULL */
    const float *obs;          /* [S][n][D] */
    const uint32_t *adj_bits;  /* [S][n][W] or NULL = all ones */
    const uint32_t *chan_bits; /* [S][L][n][W] or NULL = all ones */
    const uint8_t *avail_bits; /* policy: [S][n], bit a = action a available, or NULL */
    const int64_t *actions;    /* policy: [S][n] */
    const float *adv;          /* policy: [S] advantages; NULL = no objective (forward only) */
    const float *old_ll;       /* policy: [S] log-likelihood under the frozen old policy; NULL = ratio 1 */
    const uint8_t *valid;      /* [S] 0 = padded step (no contribution), or NULL = all valid; the critic reads it since ABI 7 */
    const float *returns;      /* critic: [S] */
    float inv_count;           /* 1 / (number of steps the mean of the loss runs over) */
    float *ll, *entropy;       /* policy outputs [S], optional */
    float *probs;              /* policy output [S][n][5], optional */
    float *values;             /* critic output [S], optional */
    float *loss;               /* DEVICE f32[1] (a set: [n_policies]), optional: the loss (summed in float64 over the call) is ADDED to it */
    float *workspace;
    size_t workspace_floats;
    /* Several networks of one kind and architecture in one call (ABI 7; 0 or 1 = one network, the members below are not read).  The
     * n_steps steps are n_policies contiguous blocks of steps_per_policy steps; step s runs the network whose blob starts at
     * weights + (s / steps_per_policy) * weights_stride, its gradient is ADDED at grad + (s / steps_per_policy) * grad_stride, its loss
     * is added to loss[s / steps_per_policy] (float64 sum per member) and inv_counts[s / steps_per_policy] replaces inv_count.  Every
     * kernel counts its tiles and env blocks per member, so no tile holds rows of two members; members of equal length are padded
     * with valid = 0 steps holding finite data (the critic reads `valid` too: such a step writes its value and adds nothing).  Needs
     * n_steps == n_policies * steps_per_policy, strides of at least the blob length and a multiple of 4 floats, and inv_counts when
     * a loss or gradient is asked for; else CM_EINVAL.  The workspace needs ((2 * n_policies + 3) & ~3) - 4 floats more than
     * cm_ppo_net_workspace_floats gives, for the per-member float64 loss sums.  CM_NET_POLICY_CENT / CM_NET_BASELINE_MLP:
     * CM_EUNSUPPORTED. */
    int32_t n_policies;
    int64_t steps_per_policy;
    int64_t weights_stride, grad_stride;   /* floats */
    const float *inv_counts;   /* DEVICE [n_policies] */
} cm_net_io;
size_t cm_critic_blob_floats(int32_t obs_dim, int32_t n_layers);
size_t cm_baseline_mlp_blob_floats(int32_t in_dim);
size_t cm_ppo_net_workspace_floats(const cm_net_desc *desc, int64_t chunk_steps, int32_t backward);
int cm_ppo_net(const cm_net_desc *desc, const cm_net_io *io, cm_stream_t stream);

/* dense float32 masks (the reference's dist_adj (B,n,n) / channels (B,L,n,n)) <-> bit rows */
int cm_mask_pack(const float *dense, uint32_t *bits, int64_t rows, int32_t n, cm_stream_t stream);
int cm_mask_unpack(const uint32_t *bits, float *dense, int64_t rows, int32_t n, cm_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* COMMARL_B200_H_ */
