// host_abi.cu — host-buffer entry points of the C ABI: the reference-facing calls (numpy arrays in, numpy arrays out,
// like VecEnvExecutor.step and policy.get_actions) as ONE C call each: asynchronous H2D copies of the inputs, the kernel,
// asynchronous D2H copies of the outputs, all on the caller's stream.  Nothing here synchronises or allocates: the caller
// owns pinned host buffers and device staging buffers of the same shapes and waits on the stream (or an event) before it
// reads the host outputs.
#include <cuda_runtime.h>
#include <stdint.h>

#include "commarl_b200.h"
#include "common.cuh"

namespace cm {

__global__ void fill_u32_kernel(uint32_t *__restrict__ p, int64_t n, uint32_t v)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = v;
}

// A run of copies in one direction.  When the caller has DECLARED an arena layout (host_arena != 0 in the host struct:
// the arrays are carved from one arena on both sides, same order, same alignment padding), consecutive entries whose
// source AND destination continue the previous entry with the same small gap are merged into ONE cudaMemcpyAsync: a DMA
// transfer has a fixed cost of several microseconds on the device timeline, which dominates the small arrays (reward,
// done, counts, masks of small teams ...).  The padding bytes between merged arrays are copied too — which is why
// nothing is merged for undeclared (arbitrary) caller buffers: one transfer per array, nothing outside them is touched.
struct CopyRun {
    cudaStream_t s;
    cudaMemcpyKind kind;
    bool merge;
    char *dst = nullptr;
    const char *src = nullptr;
    size_t bytes = 0;
    int rc = CM_OK;
    CopyRun(cudaStream_t s_, cudaMemcpyKind k_, bool merge_) : s(s_), kind(k_), merge(merge_) {}
    void flush()
    {
        if (bytes && rc == CM_OK) {
            const cudaError_t e = cudaMemcpyAsync(dst, src, bytes, kind, s);
            if (e != cudaSuccess) rc = set_cuda_error(e, CM_ECUDA);
        }
        bytes = 0;
    }
    void add(void *d, const void *sr, size_t n)
    {
        if (!d || !sr || n == 0) return;
        char *dc = static_cast<char *>(d);
        const char *sc = static_cast<const char *>(sr);
        if (bytes && merge) {
            const ptrdiff_t gd = dc - (dst + bytes), gs = sc - (src + bytes);
            if (gd == gs && gd >= 0 && gd <= 1024) { bytes += (size_t)gd + n; return; }
        }
        flush();
        dst = dc; src = sc; bytes = n;
    }
    int done() { flush(); return rc; }
};

static void add_policy_outputs(CopyRun &down, const cm_policy_desc *desc, size_t B, const cm_policy_io *dev, const cm_policy_io *host)
{
    const size_t n = (size_t)desc->n_agents, rows = B * n;
    down.add(host->actions, dev->actions, rows);
    down.add(host->probs, dev->probs, rows * CM_ACTIONS * 4);
    down.add(host->logits, dev->logits, rows * CM_ACTIONS * 4);
    down.add(host->attention, dev->attention, rows * n * 4);
}

static int policy_outputs_to_host(const cm_policy_desc *desc, size_t B, const cm_policy_io *dev, const cm_policy_io *host, cudaStream_t s)
{
    CopyRun down(s, cudaMemcpyDeviceToHost, host->host_arena != 0);
    add_policy_outputs(down, desc, B, dev, host);
    return down.done();
}

}  // namespace cm

#define CM_TRY(x) do { const int rc_ = (x); if (rc_ != CM_OK) return rc_; } while (0)

extern "C" int cm_policy_forward_host(const cm_policy_desc *desc, const cm_policy_io *dev, const cm_policy_io *host, int64_t tick_all,
                                      cm_stream_t stream)
{
    using namespace cm;
    if (!desc || !dev || !host) return CM_EINVAL;
    if (desc->n_agents < 1 || desc->n_agents > CM_MAX_AGENTS || desc->obs_dim < 1 || dev->n_envs < 0) return CM_EINVAL;
    if (dev->n_policies > 1 || host->n_policies > 1) return CM_EUNSUPPORTED;      // one policy per host-buffer call
    cudaStream_t s = (cudaStream_t)stream;
    const size_t B = (size_t)dev->n_envs, n = (size_t)desc->n_agents, D = (size_t)desc->obs_dim, L = (size_t)desc->n_layers;
    const size_t W = (n + 31) / 32, rows = B * n;
    if (B == 0) return CM_OK;
    CopyRun up(s, cudaMemcpyHostToDevice, host->host_arena != 0);
    up.add(const_cast<float *>(dev->obs), host->obs, rows * D * 4);
    up.add(const_cast<uint32_t *>(dev->adj_bits), host->adj_bits, rows * W * 4);
    up.add(const_cast<uint32_t *>(dev->chan_bits), host->chan_bits, rows * L * W * 4);
    up.add(const_cast<uint8_t *>(dev->avail_bits), host->avail_bits, rows);
    up.add(const_cast<float *>(dev->sample_u), host->sample_u, rows * 4);
    up.add(const_cast<uint32_t *>(dev->episode), host->episode, B * 4);
    if (tick_all < 0) up.add(const_cast<uint32_t *>(dev->tick), host->tick, B * 4);
    CM_TRY(up.done());
    if (tick_all >= 0 && dev->tick) {
        const int grid = (int)((B + 255) / 256 < 148 ? (B + 255) / 256 : 148);
        fill_u32_kernel<<<grid, 256, 0, s>>>(const_cast<uint32_t *>(dev->tick), (int64_t)B, (uint32_t)tick_all);
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return set_cuda_error(e, CM_ECUDA);
    }
    CM_TRY(cm_policy_forward(desc, dev, stream));
    return cm::policy_outputs_to_host(desc, B, dev, host, s);
}

static size_t env_obs_dim(const cm_env_desc *d)
{
    const size_t ww = (size_t)(2 * d->sensing + 1) * (size_t)(2 * d->sensing + 1);
    return d->scenario == CM_COVERAGE ? 3 * ww + 2 : 2 * ww + 3;      /* coverage.py:111-117, predator_prey.py:95-98 */
}

static void add_env_outputs(cm::CopyRun &down, const cm_env_desc *desc, size_t B, const cm_step_io *dev, const cm_step_io *host);

static int env_outputs_to_host(const cm_env_desc *desc, size_t B, const cm_step_io *dev, const cm_step_io *host, cudaStream_t s)
{
    cm::CopyRun down(s, cudaMemcpyDeviceToHost, host->host_arena != 0);
    add_env_outputs(down, desc, B, dev, host);
    return down.done();
}

static void add_env_outputs(cm::CopyRun &down, const cm_env_desc *desc, size_t B, const cm_step_io *dev, const cm_step_io *host)
{
    const size_t n = (size_t)desc->n_agents, p = (size_t)(desc->n_preys > 0 ? desc->n_preys : 1), L = (size_t)desc->n_layers;
    const size_t W = (n + 31) / 32, D = env_obs_dim(desc);
    down.add(host->obs, dev->obs, B * n * D * 4);
    down.add(host->adj_bits, dev->adj_bits, B * n * W * 4);
    down.add(host->chan_bits, dev->chan_bits, B * L * n * W * 4);
    down.add(host->reward, dev->reward, B * 8);
    down.add(host->done, dev->done, B);
    down.add(host->counts, dev->counts, B * 6 * 4);
    down.add(host->prey_alive_out, dev->prey_alive_out, B * p);
    down.add(host->success_out, dev->success_out, B);
    down.add(host->ave_deg, dev->ave_deg, B * 4);
}

extern "C" int cm_env_step_host(const cm_env_desc *desc, const cm_env_state *state, const cm_step_io *dev, const cm_step_io *host,
                                cm_stream_t stream)
{
    using namespace cm;
    if (!desc || !state || !dev || !host || !dev->actions || !host->actions) return CM_EINVAL;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t B = (size_t)state->n_envs, n = (size_t)desc->n_agents;
    if (B == 0) return CM_OK;
    CopyRun up(s, cudaMemcpyHostToDevice, false);
    up.add(const_cast<int8_t *>(dev->actions), host->actions, B * n);
    CM_TRY(up.done());
    CM_TRY(cm_env_step(desc, state, dev, stream));
    return env_outputs_to_host(desc, B, dev, host, s);
}

extern "C" int cm_env_reset_host(const cm_env_desc *desc, const cm_env_state *state, const cm_step_io *dev, const cm_step_io *host,
                                 cm_stream_t stream)
{
    if (!desc || !state || !dev || !host) return CM_EINVAL;
    if (state->n_envs == 0) return CM_OK;
    CM_TRY(cm_env_reset(desc, state, dev, nullptr, stream));
    return env_outputs_to_host(desc, (size_t)state->n_envs, dev, host, (cudaStream_t)stream);
}

extern "C" int cm_rollout_step_host(const cm_policy_desc *pol_desc, const cm_policy_io *pol_dev, const cm_policy_io *pol_host,
                                    const cm_env_desc *env_desc, const cm_env_state *state, const cm_step_io *env_dev,
                                    const cm_step_io *env_host, cm_stream_t stream)
{
    using namespace cm;
    if (!pol_desc || !pol_dev || !pol_host || !env_desc || !state || !env_dev || !env_host) return CM_EINVAL;
    if (!pol_dev->actions || pol_dev->actions != env_dev->actions) return CM_EINVAL;      // the step consumes the sampled actions
    if (!pol_dev->obs || pol_dev->obs != env_dev->obs) return CM_EINVAL;                  // ... and leaves the next observation there
    if (pol_dev->n_envs != state->n_envs || pol_desc->n_agents != env_desc->n_agents) return CM_EINVAL;
    if (pol_dev->n_policies > 1 || pol_host->n_policies > 1) return CM_EUNSUPPORTED;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t B = (size_t)state->n_envs, n = (size_t)env_desc->n_agents;
    if (B == 0) return CM_OK;
    if (pol_host->avail_bits) {
        if (!pol_dev->avail_bits) return CM_EINVAL;
        CopyRun up(s, cudaMemcpyHostToDevice, false);
        up.add(const_cast<uint8_t *>(pol_dev->avail_bits), pol_host->avail_bits, B * n);
        CM_TRY(up.done());
    }
    CM_TRY(cm_policy_forward(pol_desc, pol_dev, stream));
    CM_TRY(cm_env_step(env_desc, state, env_dev, stream));
    // everything the sampler appends, as one run of transfers: with the env outputs and the policy outputs carved from ONE
    // declared arena on both sides (HostRollout does that) the whole step result is a single DMA transfer
    CopyRun down(s, cudaMemcpyDeviceToHost, env_host->host_arena != 0 && pol_host->host_arena != 0);
    add_env_outputs(down, env_desc, B, env_dev, env_host);
    add_policy_outputs(down, pol_desc, B, pol_dev, pol_host);
    return down.done();
}
