// policy_attn_kernel.cu — attention + graph convolutions of CommCategoricalMLPPolicy for LARGE teams (64 < n <= 256).
//
// Middle stage of the large-team pipeline (policy_tc_kernel.cu holds the row-wise halves on the tensor cores):
//   1. policy_tc_kernel<mode Enc> : obs rows -> E, Q = E Wa^T, H_0 Wg_0          (rows of 64 floats in global scratch)
//   2. policy_attn_kernel (here)  : per env  M = softmax_j(Q E^T),  A_l = M * Range * chan_l / (sum + 1e-12),
//                                   H_{l+1} = tanh(A_l (H_l Wg_l) + bg_l),  X = E + H_L         (comm_base_net.py:80-108,
//                                   attention_module.py:38-49, graph_conv_module.py:51-72)
//   3. policy_tc_kernel<mode Head>: X rows -> logits / probs / actions
// The n x n pieces are exact fp32 on the CUDA cores.  One CTA of 8 warps owns an environment; the keys E and the values
// H_l Wg_l of the whole team sit in shared memory (row-major, <= 256 rows), the query rows are processed in blocks of
// RT rows handed out round-robin to the warps (RT is chosen per team size so that the groups divide evenly among the 8
// warps: 13 rows for 200 agents = 16 groups), and EVERYTHING between the scores and the next layer's rows is private to a
// warp: it computes its rows' scores against all keys with an RT x KT register tile (lane = key mod 32), takes the softmax and
// the masked sums with warp shuffles, parks the un-normalised masked attention rows in its own slice of shared memory
// and multiplies them with the values (lane = 4 output columns x half of the keys).  No CTA barrier inside a layer.
// The scores are recomputed per layer (64 n^2 FMAs, as many as the aggregation) instead of keeping n x n floats per env.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "commarl_b200.h"
#include "common.cuh"
#include "policy_layout.cuh"

namespace cm {

static constexpr int kAThreads = 256, kAWarps = 8;
static constexpr int kEPitch = 68;        // floats per key row: 272 bytes, so that 8 lanes x 16 bytes touch 32 distinct banks

struct AttnArgs {
    cm_policy_desc d;
    const float *weights;                 // fp32 blob: Wg_l (l >= 1) and the graph-convolution biases
    const uint32_t *adj_bits, *chan_bits;
    float *attention;                     // [B][n][n] or NULL
    const float *scr_e;                   // [B n][64]  E
    float *scr_q;                         // [B n][64]  in: Q rows, out: X rows (in place, row by row)
    float *scr_hw;                        // [B n][64]  in: H_0 Wg_0; rewritten in place with H_l Wg_l of the later layers
    int64_t n_envs;
    int64_t envs_per_policy, weights_stride;   // several policies (kMulti): env b reads the blob at weights + (b / envs_per_policy) * weights_stride
};

template <int RT, int KT, bool kMulti>
__global__ void __launch_bounds__(kAThreads, (RT * KT <= 30) ? 2 : 1) policy_attn_kernel(const AttnArgs A)
{
    constexpr int NK = 32 * KT, AP = NK + 4;
    extern __shared__ __align__(16) float sm[];
    float *Es = sm;                              // [NK][68]   keys (rows >= n are zero)
    float *HWs = Es + NK * kEPitch;              // [NK][64]   values of the current layer (rows >= n are zero)
    float *As = HWs + NK * 64;                   // [8][RT][AP] per-warp: query rows, then attention rows, then H rows
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    float *Aw = As + warp * RT * AP;
    const int n = A.d.n_agents, L = A.d.n_layers, W = (n + 31) >> 5;
    const Blob o = blob_layout(A.d.obs_dim, L);
    const int n_groups = (n + RT - 1) / RT;      // groups of RT query rows, dealt round-robin to the warps
    const int half = lane >> 4, cl = (lane & 15) << 2;
    const int n_chunks = (n + 3) >> 2;           // key chunks of 4 (attention values / value rows beyond n are zero)

    for (int64_t env = blockIdx.x; env < A.n_envs; env += gridDim.x) {
        const size_t r_env = (size_t)env * n;
        const float *wts = kMulti ? A.weights + (env / A.envs_per_policy) * A.weights_stride : A.weights;
        __syncthreads();                         // the previous env's keys / values are dead
        for (int e = tid; e < NK * 16; e += kAThreads) {
            const int j = e >> 4, c = (e & 15) << 2;
            float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            if (j < n) v = __ldcg(reinterpret_cast<const float4 *>(A.scr_e + (r_env + j) * 64 + c));
            *reinterpret_cast<float4 *>(Es + j * kEPitch + c) = v;
        }
        for (int l = 0; l < L; ++l) {
            if (l) __syncthreads();              // every warp has written its H_l Wg_l rows and is done with the old values
            for (int e = tid; e < NK * 16; e += kAThreads) {
                const int j = e >> 4, c = (e & 15) << 2;
                float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                if (j < n) v = __ldcg(reinterpret_cast<const float4 *>(A.scr_hw + (r_env + j) * 64 + c));
                *reinterpret_cast<float4 *>(HWs + j * 64 + c) = v;
            }
            __syncthreads();
            const float *bias = wts + o.gcn_b + l * kE;
            const float4 b4 = __ldg(reinterpret_cast<const float4 *>(bias + cl));
            for (int grp = warp; grp < n_groups; grp += kAWarps) {
                const int i0 = grp * RT;                             // first query row of this group
                // ---- query rows -> the warp's slice ----
                __syncwarp();
                for (int e = lane; e < RT * 16; e += 32) {
                    const int r = e >> 4, c = (e & 15) << 2;
                    float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                    if (i0 + r < n) v = __ldcg(reinterpret_cast<const float4 *>(A.scr_q + (r_env + i0 + r) * 64 + c));
                    *reinterpret_cast<float4 *>(Aw + r * AP + c) = v;
                }
                __syncwarp();
                // neighbour masks of the rows (lane t holds word t): requested before the scores so that the L2 round trip
                // hides behind them
                uint32_t mw[RT];
#pragma unroll
                for (int r = 0; r < RT; ++r) {
                    mw[r] = 0u;
                    if (i0 + r < n && lane < W) {
                        mw[r] = 0xFFFFFFFFu;
                        if (A.adj_bits) mw[r] &= __ldg(A.adj_bits + (r_env + i0 + r) * W + lane);
                        if (A.chan_bits) mw[r] &= __ldg(A.chan_bits + (((size_t)env * L + l) * n + i0 + r) * W + lane);
                    }
                }
                // ---- scores: s[r][t] = Q[i0 + r] . E[lane + 32 t] ----
                float s[RT][KT];
#pragma unroll
                for (int r = 0; r < RT; ++r)
#pragma unroll
                    for (int t = 0; t < KT; ++t) s[r][t] = 0.0f;
#pragma unroll 2
                for (int k = 0; k < kE; k += 4) {
                    float4 q[RT];
#pragma unroll
                    for (int r = 0; r < RT; ++r) q[r] = *reinterpret_cast<const float4 *>(Aw + r * AP + k);
#pragma unroll
                    for (int t = 0; t < KT; ++t) {
                        const float4 ev = *reinterpret_cast<const float4 *>(Es + (lane + 32 * t) * kEPitch + k);
                        // (consecutive FMAs are independent: RT accumulators per k, a dependent one only RT instructions later)
#pragma unroll
                        for (int r = 0; r < RT; ++r) s[r][t] = fmaf(q[r].x, ev.x, s[r][t]);
#pragma unroll
                        for (int r = 0; r < RT; ++r) s[r][t] = fmaf(q[r].y, ev.y, s[r][t]);
#pragma unroll
                        for (int r = 0; r < RT; ++r) s[r][t] = fmaf(q[r].z, ev.z, s[r][t]);
#pragma unroll
                        for (int r = 0; r < RT; ++r) s[r][t] = fmaf(q[r].w, ev.w, s[r][t]);
                    }
                }
                __syncwarp();                                        // every lane has read the query rows
                // ---- softmax over the keys (attention_module.py:44-49), mask, un-normalised attention rows ----
                float den[RT];
#pragma unroll
                for (int r = 0; r < RT; ++r) {
                    const int i = i0 + r;
                    float mx = -INFINITY;
#pragma unroll
                    for (int t = 0; t < KT; ++t)
                        if (lane + 32 * t < n) mx = fmaxf(mx, s[r][t]);
                    mx = warp_max(mx);
                    float sum = 0.0f;
#pragma unroll
                    for (int t = 0; t < KT; ++t) {
                        s[r][t] = lane + 32 * t < n ? __expf(s[r][t] - mx) : 0.0f;
                        sum += s[r][t];
                    }
                    sum = warp_sumf(sum);
                    float dsum = 0.0f;
#pragma unroll
                    for (int t = 0; t < KT; ++t) {
                        const float p = s[r][t] / sum;
                        if (l == 0 && A.attention && i < n && lane + 32 * t < n)     // the UNMASKED softmax (comm_base_net.py:93)
                            A.attention[(r_env + i) * n + lane + 32 * t] = p;
                        const uint32_t word = __shfl_sync(0xFFFFFFFFu, mw[r], t);
                        const float a = ((word >> lane) & 1u) ? p : 0.0f;
                        dsum += a;
                        Aw[r * AP + lane + 32 * t] = a;
                    }
                    den[r] = warp_sumf(dsum);
                }
                __syncwarp();
                // ---- aggregation: out[r][cl .. cl+3] = sum_j a[r][j] HW[j][cl ..]; the two half-warps split the key chunks ----
                float acc[RT][4];
#pragma unroll
                for (int r = 0; r < RT; ++r) acc[r][0] = acc[r][1] = acc[r][2] = acc[r][3] = 0.0f;
#pragma unroll 2
                for (int c = half; c < n_chunks; c += 2) {
                    const int j = c << 2;
                    const float4 h0 = *reinterpret_cast<const float4 *>(HWs + (j + 0) * 64 + cl);
                    const float4 h1 = *reinterpret_cast<const float4 *>(HWs + (j + 1) * 64 + cl);
                    const float4 h2 = *reinterpret_cast<const float4 *>(HWs + (j + 2) * 64 + cl);
                    const float4 h3 = *reinterpret_cast<const float4 *>(HWs + (j + 3) * 64 + cl);
#pragma unroll
                    for (int r = 0; r < RT; r += 2) {              // two rows at a time: 8 independent FMAs per key
                        const float4 a0 = *reinterpret_cast<const float4 *>(Aw + r * AP + j);
                        const float4 a1 = r + 1 < RT ? *reinterpret_cast<const float4 *>(Aw + (r + 1) * AP + j) : a0;
                        const float av0[4] = {a0.x, a0.y, a0.z, a0.w}, av1[4] = {a1.x, a1.y, a1.z, a1.w};
                        const float4 hv[4] = {h0, h1, h2, h3};
#pragma unroll
                        for (int jj = 0; jj < 4; ++jj) {
                            acc[r][0] = fmaf(av0[jj], hv[jj].x, acc[r][0]);
                            acc[r][1] = fmaf(av0[jj], hv[jj].y, acc[r][1]);
                            acc[r][2] = fmaf(av0[jj], hv[jj].z, acc[r][2]);
                            acc[r][3] = fmaf(av0[jj], hv[jj].w, acc[r][3]);
                            if (r + 1 < RT) {
                                acc[r + 1][0] = fmaf(av1[jj], hv[jj].x, acc[r + 1][0]);
                                acc[r + 1][1] = fmaf(av1[jj], hv[jj].y, acc[r + 1][1]);
                                acc[r + 1][2] = fmaf(av1[jj], hv[jj].z, acc[r + 1][2]);
                                acc[r + 1][3] = fmaf(av1[jj], hv[jj].w, acc[r + 1][3]);
                            }
                        }
                    }
                }
#pragma unroll
                for (int r = 0; r < RT; ++r)
#pragma unroll
                    for (int c = 0; c < 4; ++c) acc[r][c] += __shfl_xor_sync(0xFFFFFFFFu, acc[r][c], 16);
                __syncwarp();                                        // every lane has read the attention rows
                // ---- H_{l+1} = tanh(out / (sum + 1e-12) + b)   (comm_base_net.py:103, graph_conv_module.py:66-72) ----
#pragma unroll
                for (int r = 0; r < RT; ++r) {
                    const float dn = den[r] + 1e-12f;
                    acc[r][0] = tanhf(acc[r][0] / dn + b4.x);
                    acc[r][1] = tanhf(acc[r][1] / dn + b4.y);
                    acc[r][2] = tanhf(acc[r][2] / dn + b4.z);
                    acc[r][3] = tanhf(acc[r][3] / dn + b4.w);
                }
                if (l + 1 < L) {
                    // ---- next layer's value rows: H_{l+1} Wg_{l+1} (lane = 2 output columns), written over this warp's rows ----
                    if (half == 0) {
#pragma unroll
                        for (int r = 0; r < RT; ++r)
                            *reinterpret_cast<float4 *>(Aw + r * AP + cl) = make_float4(acc[r][0], acc[r][1], acc[r][2], acc[r][3]);
                    }
                    __syncwarp();
                    const float *wg = wts + o.gcn_w + (size_t)(l + 1) * kE * kE + 2 * lane;
                    float o2[RT][2];
#pragma unroll
                    for (int r = 0; r < RT; ++r) o2[r][0] = o2[r][1] = 0.0f;
#pragma unroll 2
                    for (int k = 0; k < kE; k += 4) {
                        const float2 w0 = __ldg(reinterpret_cast<const float2 *>(wg + (k + 0) * kE));
                        const float2 w1 = __ldg(reinterpret_cast<const float2 *>(wg + (k + 1) * kE));
                        const float2 w2 = __ldg(reinterpret_cast<const float2 *>(wg + (k + 2) * kE));
                        const float2 w3 = __ldg(reinterpret_cast<const float2 *>(wg + (k + 3) * kE));
                        float4 hv[RT];
#pragma unroll
                        for (int r = 0; r < RT; ++r) hv[r] = *reinterpret_cast<const float4 *>(Aw + r * AP + k);
#pragma unroll
                        for (int r = 0; r < RT; ++r) { o2[r][0] = fmaf(hv[r].x, w0.x, o2[r][0]); o2[r][1] = fmaf(hv[r].x, w0.y, o2[r][1]); }
#pragma unroll
                        for (int r = 0; r < RT; ++r) { o2[r][0] = fmaf(hv[r].y, w1.x, o2[r][0]); o2[r][1] = fmaf(hv[r].y, w1.y, o2[r][1]); }
#pragma unroll
                        for (int r = 0; r < RT; ++r) { o2[r][0] = fmaf(hv[r].z, w2.x, o2[r][0]); o2[r][1] = fmaf(hv[r].z, w2.y, o2[r][1]); }
#pragma unroll
                        for (int r = 0; r < RT; ++r) { o2[r][0] = fmaf(hv[r].w, w3.x, o2[r][0]); o2[r][1] = fmaf(hv[r].w, w3.y, o2[r][1]); }
                    }
#pragma unroll
                    for (int r = 0; r < RT; ++r)
                        if (i0 + r < n)
                            *reinterpret_cast<float2 *>(A.scr_hw + (r_env + i0 + r) * 64 + 2 * lane) = make_float2(o2[r][0], o2[r][1]);
                } else if (half == 0) {
                    // ---- X = E + H_L (comm_base_net.py:105-106) over the query rows, which are dead ----
#pragma unroll
                    for (int r = 0; r < RT; ++r) {
                        if (i0 + r < n) {
                            float4 x = make_float4(acc[r][0], acc[r][1], acc[r][2], acc[r][3]);
                            if (A.d.residual) {
                                const float4 ev = *reinterpret_cast<const float4 *>(Es + (i0 + r) * kEPitch + cl);
                                x.x += ev.x; x.y += ev.y; x.z += ev.z; x.w += ev.w;
                            }
                            *reinterpret_cast<float4 *>(A.scr_q + (r_env + i0 + r) * 64 + cl) = x;
                        }
                    }
                }
            }
        }
    }
}

template <int RT, int KT>
static int launch_attn_t(const AttnArgs &A, cudaStream_t stream)
{
    constexpr int NK = 32 * KT;
    constexpr size_t smem = (size_t)(NK * kEPitch + NK * 64 + kAWarps * RT * (NK + 4)) * sizeof(float);
    static thread_local struct { int dev; int slots; } caches[2] = {{-1, 0}, {-1, 0}};
    const bool multi = A.weights_stride != 0;
    auto &cache = caches[multi];
    void (*kern)(const AttnArgs) = multi ? policy_attn_kernel<RT, KT, true> : policy_attn_kernel<RT, KT, false>;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return set_cuda_error(cudaGetLastError(), CM_ENODEVICE);
    if (cache.dev != dev) {
        int sms = 0, ctas = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return set_cuda_error(cudaGetLastError(), CM_ECUDA);
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return set_cuda_error(e, CM_ECUDA);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas, kern, kAThreads, smem) != cudaSuccess)
            return set_cuda_error(cudaGetLastError(), CM_ECUDA);
        cache.dev = dev;
        cache.slots = sms * (ctas < 1 ? 1 : ctas);
    }
    const int grid = (int)(A.n_envs < cache.slots ? A.n_envs : cache.slots);
    kern<<<grid, kAThreads, smem, stream>>>(A);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? CM_OK : set_cuda_error(e, CM_ECUDA);
}

static constexpr int kMaxRT = 14;
static constexpr size_t kMaxSmem = 227 * 1024;

constexpr bool attn_fits(int RT, int KT)
{
    return RT * KT <= 98 && (size_t)(32 * KT * kEPitch + 32 * KT * 64 + kAWarps * RT * (32 * KT + 4)) * 4 <= kMaxSmem;
}

// rows per group: every warp gets ceil(groups / 8) groups, a group costs its RT rows of FMAs plus a fixed part (key loads,
// query staging, softmax bookkeeping) of about three rows' worth — pick the RT with the smallest makespan that fits the
// register tile and shared memory
constexpr int attn_choose_rt(int n, int KT)
{
    int best = 5, best_cost = 1 << 30;
    for (int rt = 5; rt <= kMaxRT; ++rt) {
        if (!attn_fits(rt, KT)) continue;
        const int groups = (n + rt - 1) / rt, rounds = (groups + kAWarps - 1) / kAWarps, cost = rounds * (rt + 3);
        if (cost < best_cost) { best_cost = cost; best = rt; }
    }
    return best;
}

// only the (RT, KT) pairs some team size 65..256 actually selects are instantiated (15 kernels)
constexpr bool attn_reachable(int RT, int KT)
{
    for (int n = 32 * (KT - 1) + 1; n <= 32 * KT; ++n)
        if (n > 64 && attn_choose_rt(n, KT) == RT) return true;
    return false;
}

template <int RT, int KT>
static int launch_attn_rk(const AttnArgs &A, cudaStream_t stream)
{
    if constexpr (attn_fits(RT, KT) && attn_reachable(RT, KT)) return launch_attn_t<RT, KT>(A, stream);
    else return CM_EUNSUPPORTED;
}

template <int KT>
static int launch_attn_k(int RT, const AttnArgs &A, cudaStream_t stream)
{
    switch (RT) {
    case 5: return launch_attn_rk<5, KT>(A, stream);
    case 6: return launch_attn_rk<6, KT>(A, stream);
    case 7: return launch_attn_rk<7, KT>(A, stream);
    case 8: return launch_attn_rk<8, KT>(A, stream);
    case 9: return launch_attn_rk<9, KT>(A, stream);
    case 10: return launch_attn_rk<10, KT>(A, stream);
    case 11: return launch_attn_rk<11, KT>(A, stream);
    case 12: return launch_attn_rk<12, KT>(A, stream);
    case 13: return launch_attn_rk<13, KT>(A, stream);
    case 14: return launch_attn_rk<14, KT>(A, stream);
    }
    return CM_EUNSUPPORTED;
}

int launch_policy_tc_encode(const cm_policy_desc *desc, const cm_policy_io *io, float *scr_e, float *scr_q, float *scr_hw, cudaStream_t stream);
int launch_policy_attn_mma(const cm_policy_desc *desc, const cm_policy_io *io, const float *scr_e, float *scr_q, float *scr_hw,
                           cudaStream_t stream);                                                // policy_attn_mma_kernel.cu
int launch_policy_tc_head(const cm_policy_desc *desc, const cm_policy_io *io, const float *x_rows, cudaStream_t stream);

size_t tc_large_ws_floats(int n, int64_t n_envs) { return (size_t)3 * (size_t)n_envs * (size_t)n * kE; }

// Comm-DP forward for teams of 65..256 agents: encoder (tensor cores) -> attention / graph convolutions (here) -> head
// (tensor cores), three launches on one stream, rows handed over through the caller's workspace.
int launch_policy_tc_large(const cm_policy_desc *desc, const cm_policy_io *io, cudaStream_t stream)
{
    const int n = desc->n_agents;
    if (n <= 64 || n > CM_MAX_AGENTS) return CM_EUNSUPPORTED;
    const size_t rows = (size_t)io->n_envs * n;
    if (!io->workspace || io->workspace_bytes < tc_large_ws_floats(n, io->n_envs) * sizeof(float)) return CM_EINVAL;
    if ((reinterpret_cast<uintptr_t>(io->workspace) & 15u) != 0) return CM_EINVAL;
    float *scr_e = io->workspace, *scr_q = scr_e + rows * kE, *scr_hw = scr_q + rows * kE;
    int rc = launch_policy_tc_encode(desc, io, scr_e, scr_q, scr_hw, stream);
    if (rc) return rc;
    if (desc->math == 1) {                 // attention on the warp-level tensor path (default); math == 2: exact fp32 below
        rc = launch_policy_attn_mma(desc, io, scr_e, scr_q, scr_hw, stream);
        if (rc) return rc;
        if (!io->probs && !io->actions && !io->logits) return CM_OK;
        return launch_policy_tc_head(desc, io, scr_q, stream);
    }
    AttnArgs A;
    A.d = *desc;
    A.weights = io->weights;
    A.adj_bits = io->adj_bits;
    A.chan_bits = io->chan_bits;
    A.attention = io->attention;
    A.scr_e = scr_e; A.scr_q = scr_q; A.scr_hw = scr_hw;
    A.n_envs = io->n_envs;
    A.envs_per_policy = io->n_policies > 1 ? io->envs_per_policy : io->n_envs;
    A.weights_stride = io->n_policies > 1 ? io->weights_stride : 0;       // 0: one policy (the kMulti = false kernels)
    const int KT = (n + 31) / 32, RT = attn_choose_rt(n, KT);      // keys per lane, query rows per group
    switch (KT) {
    case 3: rc = launch_attn_k<3>(RT, A, stream); break;
    case 4: rc = launch_attn_k<4>(RT, A, stream); break;
    case 5: rc = launch_attn_k<5>(RT, A, stream); break;
    case 6: rc = launch_attn_k<6>(RT, A, stream); break;
    case 7: rc = launch_attn_k<7>(RT, A, stream); break;
    case 8: rc = launch_attn_k<8>(RT, A, stream); break;
    default: rc = CM_EUNSUPPORTED;
    }
    if (rc) return rc;
    if (!io->probs && !io->actions && !io->logits) return CM_OK;
    return launch_policy_tc_head(desc, io, scr_q, stream);
}

}  // namespace cm
