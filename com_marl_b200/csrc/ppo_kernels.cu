// ppo_kernels.cu — the two hand-written pieces of the PPO update (SURVEY.md §8f.1): per-path returns / GAE advantages /
// advantage normalisation, and the fused Adam step over a flat parameter bucket.  The network forward / backward of the
// update is csrc/ppo_net_kernels.cu (cm_ppo_net); these kernels replace the Python-side tensor plumbing around it.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "commarl_b200.h"
#include "common.cuh"

namespace cm {

// One warp per path (row of the padded [P][T] batch the reference builds in process_samples,
// centralized_ma_ppo.py:612-659).
//   returns[t]  = discounted cumulative reward over the valid steps, float64 recursion like scipy.signal.lfilter in
//                 tensor_utils.discount_cumsum (garage/misc/tensor_utils.py:7-23), stored as float32, 0 in the padding;
//   raw_adv[t]  = sum_k (discount * lambda)^k delta[t + k],  delta[t] = r[t] + discount * b[t + 1] - b[t],  b[T] = 0
//                 over the WHOLE padded row (compute_advantages, garage/torch/algos/_utils.py:56-113): the baselines of
//                 the padded tail are whatever the critic returns for an all-zero observation and DO enter the sum —
//                 that is the reference's behaviour and is reproduced;
//   adv[t]      = (raw_adv[t] - mean) / sqrt(var + eps) with the mean / biased variance of the path's VALID steps,
//                 applied to the whole row (F.batch_norm over advantages.t(), centralized_ma_ppo.py:425-429).
__global__ void ppo_advantages_kernel(const double *__restrict__ rewards, const float *__restrict__ baselines,
                                      const int32_t *__restrict__ valids, int64_t n_paths, int T, float discount, float lambda,
                                      int center, float eps, float *__restrict__ returns, float *__restrict__ raw_adv,
                                      float *__restrict__ adv)
{
    extern __shared__ float sm[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    float *buf = sm + (size_t)warp * T;
    const float c = discount * lambda;
    for (int64_t p = (int64_t)blockIdx.x * wpb + warp; p < n_paths; p += (int64_t)gridDim.x * wpb) {
        const double *r = rewards + p * T;
        const float *b = baselines + p * T;
        const int v = min(max(valids[p], 0), T);
        __syncwarp();
        for (int t = lane; t < T; t += 32) {
            const float bn = t + 1 < T ? b[t + 1] : 0.0f;
            buf[t] = (float)r[t] + discount * bn - b[t];
        }
        __syncwarp();
        if (lane == 0) {                                   // the two linear recurrences (T <= a few hundred steps)
            float a = 0.0f;
            for (int t = T - 1; t >= 0; --t) { a = fmaf(c, a, buf[t]); buf[t] = a; }
            if (returns) {
                double y = 0.0;
                for (int t = T - 1; t >= 0; --t) {
                    y = t < v ? r[t] + (double)discount * y : 0.0;
                    returns[p * T + t] = (float)y;
                }
            }
        }
        __syncwarp();
        float mean = 0.0f, inv = 1.0f;
        if (center) {
            float s = 0.0f;
            for (int t = lane; t < v; t += 32) s += buf[t];
            mean = warp_sumf(s) / (float)max(v, 1);
            float q = 0.0f;
            for (int t = lane; t < v; t += 32) { const float d = buf[t] - mean; q = fmaf(d, d, q); }
            const float var = warp_sumf(q) / (float)max(v, 1);
            inv = 1.0f / sqrtf(var + eps);
        }
        for (int t = lane; t < T; t += 32) {
            const float a = buf[t];
            if (raw_adv) raw_adv[p * T + t] = a;
            if (adv) adv[p * T + t] = center ? (a - mean) * inv : a;
        }
    }
}

// torch.optim Adam as the reference drives it (my_optimizer/adam.py:57-120 -> torch.optim._functional.adam, no amsgrad,
// no weight decay) over a flat bucket; grad_scale folds the clip_grad_norm_ coefficient into the same pass.
__global__ void adam_step_kernel(float *__restrict__ p, const float *__restrict__ g, float *__restrict__ m, float *__restrict__ v,
                                 int64_t n, float beta1, float beta2, float eps, float step_size, float inv_sqrt_bc2, float grad_scale,
                                 const float *__restrict__ grad_scale_dev)
{
    if (grad_scale_dev) grad_scale = *grad_scale_dev;       // the clip coefficient straight from the reduction that produced it
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float gi = g[i] * grad_scale;
        const float mi = beta1 * m[i] + (1.0f - beta1) * gi;
        const float vi = beta2 * v[i] + (1.0f - beta2) * gi * gi;
        m[i] = mi;
        v[i] = vi;
        const float denom = sqrtf(vi) * inv_sqrt_bc2 + eps;
        p[i] = p[i] - step_size * (mi / denom);
    }
}

// The same step over members of a set, member = blockIdx.y + the launch's first member; one that is not stepped has step_size 0 and
// is skipped whole (a zero-gradient step would still move its parameters through the moments)
static constexpr int kAdamSetMax = 256;                      // members per launch (their coefficients travel as kernel parameters)
struct AdamSetCoef { float step_size[kAdamSetMax], inv_sqrt_bc2[kAdamSetMax]; };
__global__ void adam_step_set_kernel(float *__restrict__ p, const float *__restrict__ g, float *__restrict__ m, float *__restrict__ v,
                                     int64_t n, int64_t stride, float beta1, float beta2, float eps, const AdamSetCoef c,
                                     const float *__restrict__ grad_scale_dev)
{
    const int k = blockIdx.y;
    const float step_size = c.step_size[k], inv_sqrt_bc2 = c.inv_sqrt_bc2[k];
    if (step_size == 0.0f) return;
    const float grad_scale = grad_scale_dev[k];
    const int64_t o = (int64_t)k * stride;
    p += o; g += o; m += o; v += o;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float gi = g[i] * grad_scale;
        const float mi = beta1 * m[i] + (1.0f - beta1) * gi;
        const float vi = beta2 * v[i] + (1.0f - beta2) * gi * gi;
        m[i] = mi;
        v[i] = vi;
        const float denom = sqrtf(vi) * inv_sqrt_bc2 + eps;
        p[i] = p[i] - step_size * (mi / denom);
    }
}

}  // namespace cm

extern "C" int cm_ppo_advantages(const double *rewards, const float *baselines, const int32_t *valids, int64_t n_paths, int32_t T,
                                 float discount, float gae_lambda, int32_t center, float eps, float *returns, float *raw_adv,
                                 float *adv, cm_stream_t stream)
{
    using namespace cm;
    if (!rewards || !baselines || !valids || n_paths < 0 || T < 1) return CM_EINVAL;
    if (T > 8192) return CM_EUNSUPPORTED;
    if (n_paths == 0) return CM_OK;
    const int wpb = 4;
    const size_t smem = (size_t)wpb * T * sizeof(float);
    if (smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(ppo_advantages_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return set_cuda_error(e, CM_ECUDA);
    }
    const int64_t want = (n_paths + wpb - 1) / wpb;
    const int grid = (int)(want < 148 * 8 ? want : 148 * 8);
    ppo_advantages_kernel<<<grid, wpb * 32, smem, (cudaStream_t)stream>>>(rewards, baselines, valids, n_paths, T, discount, gae_lambda,
                                                                           center, eps, returns, raw_adv, adv);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? CM_OK : set_cuda_error(e, CM_ECUDA);
}

static int adam_step_impl(float *params, const float *grads, float *exp_avg, float *exp_avg_sq, int64_t n, float lr, float beta1,
                          float beta2, float eps, int32_t step, float grad_scale, const float *grad_scale_dev, cm_stream_t stream)
{
    using namespace cm;
    if (!params || !grads || !exp_avg || !exp_avg_sq || n < 0 || step < 1) return CM_EINVAL;
    if (n == 0) return CM_OK;
    const double bc1 = 1.0 - pow((double)beta1, (double)step), bc2 = 1.0 - pow((double)beta2, (double)step);
    const float step_size = (float)((double)lr / bc1), inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
    const int64_t want = (n + 255) / 256;
    const int grid = (int)(want < 148 * 8 ? want : 148 * 8);
    adam_step_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(params, grads, exp_avg, exp_avg_sq, n, beta1, beta2, eps, step_size,
                                                            inv_sqrt_bc2, grad_scale, grad_scale_dev);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? CM_OK : set_cuda_error(e, CM_ECUDA);
}

extern "C" int cm_adam_step(float *params, const float *grads, float *exp_avg, float *exp_avg_sq, int64_t n, float lr, float beta1,
                            float beta2, float eps, int32_t step, float grad_scale, cm_stream_t stream)
{
    return adam_step_impl(params, grads, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, step, grad_scale, nullptr, stream);
}

extern "C" int cm_adam_step_dev(float *params, const float *grads, float *exp_avg, float *exp_avg_sq, int64_t n, float lr, float beta1,
                                float beta2, float eps, int32_t step, const float *grad_scale_dev, cm_stream_t stream)
{
    if (!grad_scale_dev) return CM_EINVAL;
    return adam_step_impl(params, grads, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, step, 1.0f, grad_scale_dev, stream);
}

extern "C" int cm_adam_step_set(float *params, const float *grads, float *exp_avg, float *exp_avg_sq, int32_t n_policies, int64_t n,
                                int64_t stride, float lr, float beta1, float beta2, float eps, const int32_t *steps, const float *grad_scale_dev,
                                cm_stream_t stream)
{
    using namespace cm;
    if (!params || !grads || !exp_avg || !exp_avg_sq || !steps || !grad_scale_dev || n_policies < 0 || n < 0 || stride < n) return CM_EINVAL;
    for (int32_t k = 0; k < n_policies; ++k)
        if (steps[k] < 0) return CM_EINVAL;
    if (n == 0) return CM_OK;
    for (int32_t k0 = 0; k0 < n_policies; k0 += kAdamSetMax) {
        const int cnt = n_policies - k0 < kAdamSetMax ? n_policies - k0 : kAdamSetMax;
        AdamSetCoef c;
        bool any = false;
        for (int k = 0; k < cnt; ++k) {
            const int32_t step = steps[k0 + k];
            c.step_size[k] = c.inv_sqrt_bc2[k] = 0.0f;
            if (step == 0) continue;
            const double bc1 = 1.0 - pow((double)beta1, (double)step), bc2 = 1.0 - pow((double)beta2, (double)step);
            c.step_size[k] = (float)((double)lr / bc1);
            c.inv_sqrt_bc2[k] = (float)(1.0 / sqrt(bc2));
            if (c.step_size[k] == 0.0f) return CM_EINVAL;              // (lr = 0 would read as "not stepped")
            any = true;
        }
        if (!any) continue;
        const int64_t want = (n + 255) / 256, cap = (148 * 8 + cnt - 1) / cnt;
        const dim3 grid((unsigned)(want < cap ? want : cap), (unsigned)cnt);
        const int64_t o = (int64_t)k0 * stride;
        adam_step_set_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(params + o, grads + o, exp_avg + o, exp_avg_sq + o, n, stride, beta1,
                                                                     beta2, eps, c, grad_scale_dev + k0);
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return set_cuda_error(e, CM_ECUDA);
    }
    return CM_OK;
}
