// common.cuh — small device helpers shared by the kernels of the Com-MARL B200 engine.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "commarl_b200.h"

namespace cm {

// random stream ids (generated mode); keys are (seed; env id, tick, stream | episode << 8, index)
static constexpr uint32_t kStreamSpawn = 1, kStreamPrey = 2, kStreamChan = 3, kStreamAct = 4;

int set_cuda_error(cudaError_t e, int rc);

// Philox4x32-10 (Salmon, Moraes, Dror, Shaw — SC'11), the published round function.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k)
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}

// 24 random bits -> U[0,1) float32 on the 2^-24 lattice (the lattice torch.rand(float32) uses)
__device__ __forceinline__ float u24(uint32_t w) { return (float)(w >> 8) * 5.9604644775390625e-08f; }

// 32 random bits -> prey move through the CDF of (.175,.175,.175,.175,.3) (predator_prey.py:54,401);
// thresholds are floor(cdf * 2^32)
__device__ __forceinline__ int prey_move_from_bits(uint32_t w)
{
    return (int)(w >= 751619276u) + (int)(w >= 1503238553u) + (int)(w >= 2254857830u) + (int)(w >= 3006477107u);
}

__device__ __forceinline__ int warp_sum(int v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    return v;
}

__device__ __forceinline__ float warp_max(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xFFFFFFFFu, v, o));
    return v;
}

__device__ __forceinline__ float warp_sumf(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    return v;
}

// Tail of every categorical policy: softmax of one agent's logits, availability mask, renormalisation
// (comm_categorical_mlp_policy.py:86-94, centralized_categorical_mlp_policy.py:84-96), then argmax (np.argmax: first maximum)
// or inverse-CDF sampling with a sequential fp32 cumulative sum (stream spec, DESIGN.md 3.4).  g = env * n + il.
__device__ __forceinline__ void categorical_finish(const cm_policy_desc &d, const cm_policy_io &io, const float (&lg)[CM_ACTIONS],
                                                   int64_t g, int64_t env, int il)
{
    float pr[CM_ACTIONS];
    float mx = -INFINITY;
#pragma unroll
    for (int a = 0; a < CM_ACTIONS; ++a) mx = fmaxf(mx, lg[a]);
    float sum = 0.0f;
#pragma unroll
    for (int a = 0; a < CM_ACTIONS; ++a) { pr[a] = expf(lg[a] - mx); sum += pr[a]; }
    const uint32_t av = io.avail_bits ? io.avail_bits[g] : 0x1Fu;
    float msum = 0.0f;
#pragma unroll
    for (int a = 0; a < CM_ACTIONS; ++a) { pr[a] = ((av >> a) & 1u) ? pr[a] / sum : 0.0f; msum += pr[a]; }
#pragma unroll
    for (int a = 0; a < CM_ACTIONS; ++a) pr[a] = pr[a] / msum;
    if (io.logits) for (int a = 0; a < CM_ACTIONS; ++a) io.logits[g * CM_ACTIONS + a] = lg[a];
    if (io.probs) for (int a = 0; a < CM_ACTIONS; ++a) io.probs[g * CM_ACTIONS + a] = pr[a];
    if (!io.actions) return;
    int act;
    if (d.greedy) {
        act = 0;
        for (int a = 1; a < CM_ACTIONS; ++a) if (pr[a] > pr[act]) act = a;
    } else {
        float u;
        if (io.sample_u) u = io.sample_u[g];
        else {
            const uint4 blk = philox4x32_10(
                make_uint4((uint32_t)(d.env_id0 + env), io.tick[env], kStreamAct | (io.episode[env] << 8), (uint32_t)(il >> 2)),
                make_uint2((uint32_t)d.seed, (uint32_t)(d.seed >> 32)));
            const uint32_t w = (il & 3) == 0 ? blk.x : ((il & 3) == 1 ? blk.y : ((il & 3) == 2 ? blk.z : blk.w));
            u = u24(w);
        }
        int last = 4;
        for (int a = 0; a < CM_ACTIONS; ++a) if (pr[a] > 0.0f) last = a;
        act = -1;
        float c = 0.0f;
        for (int a = 0; a < CM_ACTIONS; ++a) { c += pr[a]; if (act < 0 && u < c) act = a; }
        if (act < 0) act = last;
    }
    io.actions[g] = (int8_t)act;
}

// acc[4][4*J] += A[rows 4ty..][k0..k0+kc) * Bs[k][cols], Bs pitch = 64*J, kc a multiple of 4 (zero padded): the register-tiled fp32
// product of the CENT policy's layers (policy_cent_kernel.cu) and of the update's wide first layer (ppo_net_kernels.cu).  Thread (ty, tx)
// of a 16 x 16 grid owns rows 4ty..4ty+3 and the columns {4tx..4tx+3} + 64j
template <int J>
__device__ __forceinline__ void cent_mac(const float *__restrict__ As, int lda, const float *__restrict__ Bs, int kc, int ty, int tx,
                                         float (&acc)[4][4 * J])
{
#pragma unroll 2
    for (int k = 0; k < kc; k += 4) {
        float4 a[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = *reinterpret_cast<const float4 *>(As + (ty * 4 + i) * lda + k);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            float4 b[J];
#pragma unroll
            for (int j = 0; j < J; ++j) b[j] = *reinterpret_cast<const float4 *>(Bs + (k + kk) * (64 * J) + j * 64 + tx * 4);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float av = kk == 0 ? a[i].x : (kk == 1 ? a[i].y : (kk == 2 ? a[i].z : a[i].w));
#pragma unroll
                for (int j = 0; j < J; ++j) {
                    acc[i][4 * j + 0] = fmaf(av, b[j].x, acc[i][4 * j + 0]);
                    acc[i][4 * j + 1] = fmaf(av, b[j].y, acc[i][4 * j + 1]);
                    acc[i][4 * j + 2] = fmaf(av, b[j].z, acc[i][4 * j + 2]);
                    acc[i][4 * j + 3] = fmaf(av, b[j].w, acc[i][4 * j + 3]);
                }
            }
        }
    }
}

}  // namespace cm
