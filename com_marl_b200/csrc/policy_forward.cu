// policy_forward.cu — the C ABI of the policy forward: argument checks, then the CENT kernels (policy_cent_kernel.cu) or
// the tensor-core kernels of Comm-DP / Obs-DP (policy_tc_kernel.cu, and for teams of more than 64 agents the pipeline
// in policy_attn_mma_kernel.cu).
#include <cuda_runtime.h>
#include <stdint.h>

#include "commarl_b200.h"
#include "policy_layout.cuh"

namespace cm {

int launch_policy_tc(const cm_policy_desc *desc, const cm_policy_io *io, cudaStream_t stream);   // policy_tc_kernel.cu
int launch_policy_cent(const cm_policy_desc *desc, const cm_policy_io *io, cudaStream_t stream); // policy_cent_kernel.cu
size_t tc_large_ws_floats(int n, int64_t n_envs);                                                // policy_attn_mma_kernel.cu

}  // namespace cm

extern "C" size_t cm_policy_blob_floats(int32_t obs_dim, int32_t n_layers)
{
    return (size_t)cm::blob_layout(obs_dim, n_layers).total;
}

extern "C" size_t cm_policy_workspace_bytes(int32_t n_agents, int64_t n_envs)
{
    if (n_agents <= 64 || n_envs <= 0) return 0;
    return cm::tc_large_ws_floats(n_agents, n_envs) * sizeof(float);
}

extern "C" int cm_policy_forward(const cm_policy_desc *desc, const cm_policy_io *io, cm_stream_t stream)
{
    using namespace cm;
    if (!desc || !io || !io->weights) return CM_EINVAL;
    // packed observations (cm_step_io.obs_bits) feed the tensor-core kernels of the Comm-DP / Obs-DP policies; CENT needs fp32 rows
    const bool packed_ok = io->obs_bits && desc->math == 1 && desc->kind != CM_POLICY_CENT;
    if (!io->obs && !packed_ok) return CM_EINVAL;
    if (io->obs_bits && (io->obs_nbits < 1 || io->obs_nbits > 96 || desc->obs_dim < io->obs_nbits || desc->obs_dim - io->obs_nbits > 3)) return CM_EINVAL;
    if (!io->probs && !io->actions && !io->logits && !io->attention) return CM_EINVAL;
    if (desc->n_agents < 1 || desc->n_agents > CM_MAX_AGENTS || desc->obs_dim < 1 || desc->obs_dim > 128) return CM_EUNSUPPORTED;
    if (desc->n_layers < 1 || desc->n_layers > CM_MAX_LAYERS) return CM_EUNSUPPORTED;
    if (io->actions && !desc->greedy && !io->sample_u && (!io->tick || !io->episode)) return CM_EINVAL;
    if (io->n_envs < 0) return CM_EINVAL;
    if (io->n_envs == 0) return CM_OK;
    if (desc->kind != CM_POLICY_COMM && desc->kind != CM_POLICY_DEC && desc->kind != CM_POLICY_CENT) return CM_EINVAL;
    if (io->n_policies < 0) return CM_EINVAL;
    if (io->n_policies > 1) {      // several policies: equal env blocks, strides that hold a blob and keep 16-byte alignment
        const bool cent = desc->kind == CM_POLICY_CENT;
        const size_t blob = cent ? cm_policy_cent_blob_floats(desc->n_agents, desc->obs_dim) : cm_policy_blob_floats(desc->obs_dim, desc->n_layers);
        if (io->envs_per_policy < 1 || io->n_envs / io->n_policies != io->envs_per_policy || io->n_envs % io->n_policies != 0) return CM_EINVAL;
        if (io->weights_stride < (int64_t)blob || (io->weights_stride & 3) != 0) return CM_EINVAL;
        if (desc->math == 1) {
            const size_t tcb = cent ? cm_policy_cent_tc_blob_floats(desc->n_agents, desc->obs_dim) : cm_policy_tc_blob_floats(desc->obs_dim, desc->n_layers);
            if (io->tc_weights_stride < (int64_t)tcb || (io->tc_weights_stride & 3) != 0) return CM_EINVAL;
        }
    }
    if (desc->kind == CM_POLICY_CENT) return launch_policy_cent(desc, io, (cudaStream_t)stream);
    if (desc->math != 1) return CM_EUNSUPPORTED;       // Comm-DP and Obs-DP run on the tensor-core kernels only
    return launch_policy_tc(desc, io, (cudaStream_t)stream);
}
