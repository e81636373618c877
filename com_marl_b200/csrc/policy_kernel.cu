// policy_kernel.cu — fused CommCategoricalMLPPolicy forward (+ action sampling) for sm_100a, fp32.
//
// Reference formula (comm_categorical_mlp_policy.py:48-119, comm_base_net.py:80-108,
// attention_module.py:38-49, graph_conv_module.py:51-72, categorical_mlp_module.py:64-80):
//   h  = tanh(obs W1^T + b1)            D   -> 128      encoder._layers.0
//   E  = tanh(h   W2^T + b2)            128 -> 64       encoder._output_layers.0 (output_nonlinearity=tanh)
//   M  = softmax_j((E Wa^T) E^T)        per env, n x n  attention_layer ('general')
//   A_l = M * Range * chan_l ; A_l /= (sum_j A_l + 1e-12)
//   H_{l+1} = tanh(A_l (H_l Wg_l) + bg_l),  H_0 = E      gcn_layers.l   (Wg is (in,out))
//   X  = E + H_L                                         residual
//   logits = head(X): tanh 64->128, tanh 128->64, tanh 64->32, linear 32->5
//   probs  = softmax(logits) * avail / sum ; action ~ Categorical(probs) | argmax
//
// One CTA (256 threads) owns a tile of 64 agent rows made of WHOLE environments (n <= 64), so the
// per-env attention / graph-convolution stay inside the tile and every activation lives in shared
// memory from the observation load to the sampled action: HBM traffic is the obs read plus the
// probs / action (and optional logits / attention) writes.  All nine matrix products run through one
// register-tiled 64-row microkernel (4 rows x N/16 columns per thread, operands k-major so that both
// operand loads are 128-bit).  The per-env n x n products are evaluated as dense 64 x 64 tile products
// whose off-env entries are exact zeros.  Weights (<= 198 KB) are read through the read-only path and
// stay L1/L2 resident.  Exact fp32 FFMA: this is the variant that meets the 1e-5 logit tolerance; a
// tcgen05 variant needs a stated tolerance (DESIGN.md §5).
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "commarl_b200.h"
#include "common.cuh"
#include "policy_layout.cuh"

namespace cm {

static constexpr int kTile = 64;        // agent rows per CTA tile
static constexpr int kPitch = 68;       // floats per k-major row (64 + 4: keeps float4 alignment, spreads banks)
static constexpr int kThreads = 256;

// ------------------------------------------------------------------------------------------------
// 64-row register-tiled product: acc[r][q] = sum_k At[k][4ty + r] * Bm[k][col(q)]
//   At : shared, k-major, pitch kPitch.      Bm : global weights (k-major, ld = N) or shared (pitch ldb)
//   thread (tx = tid & 15, ty = tid >> 4) owns rows 4ty..4ty+3 and columns
//   N=128: 4tx..4tx+3 and 64+4tx..64+4tx+3 | N=64: 4tx..4tx+3 | N=32: 2tx, 2tx+1
// ------------------------------------------------------------------------------------------------
enum { kBShared = 0, kBWeights = 1, kBScratch = 2 };   // where the B operand lives (weights: read-only path)

template <int N, int kBMode, bool kInit = true>
__device__ __forceinline__ void gemm64(const float *__restrict__ At, const float *Bm, int ldb, int K,
                                       float (&acc)[4][N / 16])
{
    constexpr int CN = N / 16;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    if constexpr (kInit) {
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int q = 0; q < CN; ++q) acc[r][q] = 0.0f;
    }
    const float *ap = At + 4 * ty;
    const float *bp = Bm + (CN == 2 ? 2 * tx : 4 * tx);
#pragma unroll 4
    for (int k = 0; k < K; ++k) {
        const float4 a4 = *reinterpret_cast<const float4 *>(ap + k * kPitch);
        const float a[4] = {a4.x, a4.y, a4.z, a4.w};
        float b[CN];
        if constexpr (CN == 2) {
            float2 v;
            if constexpr (kBMode == kBWeights) v = __ldg(reinterpret_cast<const float2 *>(bp + (size_t)k * ldb));
            else v = *reinterpret_cast<const float2 *>(bp + (size_t)k * ldb);
            b[0] = v.x; b[1] = v.y;
        } else {
#pragma unroll
            for (int h = 0; h < CN / 4; ++h) {
                float4 v;
                if constexpr (kBMode == kBWeights) v = __ldg(reinterpret_cast<const float4 *>(bp + (size_t)k * ldb + 64 * h));
                else v = *reinterpret_cast<const float4 *>(bp + (size_t)k * ldb + 64 * h);
                b[4 * h + 0] = v.x; b[4 * h + 1] = v.y; b[4 * h + 2] = v.z; b[4 * h + 3] = v.w;
            }
        }
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int q = 0; q < CN; ++q) acc[r][q] = fmaf(a[r], b[q], acc[r][q]);
    }
}

template <int N>
__device__ __forceinline__ int col_of(int q)
{
    const int tx = threadIdx.x & 15;
    if constexpr (N == 32) return 2 * tx + q;
    else return (q < 4) ? 4 * tx + q : 64 + 4 * tx + (q - 4);
}

// store the thread's 4 x CN block k-major (transposed) for the next product: outT[col][4ty..4ty+3],
// optionally adding a bias (global) and applying tanh
template <int N, bool kBias, bool kTanh>
__device__ __forceinline__ void store_kmajor(float *__restrict__ outT, const float (&acc)[4][N / 16],
                                             const float *__restrict__ bias)
{
    const int ty = threadIdx.x >> 4;
#pragma unroll
    for (int q = 0; q < N / 16; ++q) {
        const int c = col_of<N>(q);
        const float bv = kBias ? __ldg(bias + c) : 0.0f;
        float4 v = make_float4(acc[0][q] + bv, acc[1][q] + bv, acc[2][q] + bv, acc[3][q] + bv);
        if (kTanh) { v.x = tanhf(v.x); v.y = tanhf(v.y); v.z = tanhf(v.z); v.w = tanhf(v.w); }
        *reinterpret_cast<float4 *>(outT + c * kPitch + 4 * ty) = v;
    }
}

// store row-major out[row][col] (pitch kPitch) — the layout a product consumes as its B operand (N = 64)
__device__ __forceinline__ void store_rowmajor(float *__restrict__ out, const float (&acc)[4][4])
{
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
#pragma unroll
    for (int r = 0; r < 4; ++r)
        *reinterpret_cast<float4 *>(out + (4 * ty + r) * kPitch + 4 * tx) = make_float4(acc[r][0], acc[r][1], acc[r][2], acc[r][3]);
}

// categorical head on X^T (k-major, 64 rows) + softmax / availability mask / sampling for `rows` valid rows.
// Row r of the tile is agent `il` of env `env` (global row g):  n_div > 0: env = env_base + r / n_div,
// il = r % n_div (tile of whole envs);  n_div == 0: env = env_base, il = il_base + r (chunk of one env).
// (kMulti: the weights of the tile's policy are `wblk`; one policy: io.weights)
template <bool kMulti>
__device__ void head_and_sample(const PolicyArgs &A, const Blob &o, const float *wblk, const float *XT, float *bufA, float *bufB,
                                float *logit_s, int rows, int64_t g0, int64_t env_base, int il_base, int n_div)
{
    const cm_policy_desc &d = A.d;
    const cm_policy_io &io = A.io;
    const float *__restrict__ wts = kMulti ? wblk : io.weights;
    const int tid = threadIdx.x;
    {
        float acc[4][8];
        gemm64<128, kBWeights>(XT, wts + o.head_w1, kC1, kE, acc);
        store_kmajor<128, true, true>(bufA, acc, wts + o.head_b1);
    }
    __syncthreads();
    {
        float acc[4][4];
        gemm64<64, kBWeights>(bufA, wts + o.head_w2, kC2, kC1, acc);
        store_kmajor<64, true, true>(bufB, acc, wts + o.head_b2);
    }
    __syncthreads();
    {
        float acc[4][2];
        gemm64<32, kBWeights>(bufB, wts + o.head_w3, kC3, kC2, acc);
        store_kmajor<32, true, true>(bufB + 64 * kPitch, acc, wts + o.head_b3);
    }
    __syncthreads();
    // logits = x W4^T + b4
    for (int e = tid; e < kTile * CM_ACTIONS; e += kThreads) {
        const int r = e / CM_ACTIONS, a = e - r * CM_ACTIONS;
        const float *x = bufB + 64 * kPitch + r;
        float s = 0.0f;
#pragma unroll 8
        for (int k = 0; k < kC3; ++k) s = fmaf(x[k * kPitch], __ldg(wts + o.head_w4 + k * CM_ACTIONS + a), s);
        logit_s[e] = s + __ldg(wts + o.head_b4 + a);
    }
    __syncthreads();
    // softmax, availability mask, renormalise, sample
    if (tid < rows) {
        const int r = tid;
        const int64_t g = g0 + r;
        float lg[CM_ACTIONS];
#pragma unroll
        for (int a = 0; a < CM_ACTIONS; ++a) lg[a] = logit_s[r * CM_ACTIONS + a];
        categorical_finish(d, io, lg, g, n_div > 0 ? env_base + r / n_div : env_base, n_div > 0 ? r % n_div : il_base + r);
    }
}

// ------------------------------------------------------------------------------------------------
// kMulti: several policies in one launch — the tiles are counted per env block of io.envs_per_policy envs (a block may end
// in a partial tile) and a tile reads the blob of its block's policy
template <bool kMulti>
__global__ void __launch_bounds__(kThreads, 2) policy_small_kernel(const PolicyArgs A)
{
    extern __shared__ __align__(16) float sm[];
    float *bufA = sm;                              // 128 x pitch
    float *bufB = bufA + 128 * kPitch;             // 128 x pitch
    float *bufE = bufB + 128 * kPitch;             // 64 x pitch: E^T, kept for attention keys and the residual
    float *logit_s = bufE + kE * kPitch;           // 64 x 5
    const cm_policy_desc &d = A.d;
    const cm_policy_io &io = A.io;
    const int n = d.n_agents, D = d.obs_dim, L = d.n_layers, W = (n + 31) >> 5;
    const Blob o = blob_layout(D, L);
    const float *__restrict__ wts = io.weights;
    const int tid = threadIdx.x;

    for (int64_t tile = blockIdx.x; tile < A.n_tiles; tile += gridDim.x) {
        int64_t env0 = tile * A.envs_per_tile;
        int envs = (int)min((int64_t)A.envs_per_tile, io.n_envs - env0);
        if constexpr (kMulti) {
            const int64_t tpp = (io.envs_per_policy + A.envs_per_tile - 1) / A.envs_per_tile;    // tiles per block
            const int64_t p = tile / tpp, e0 = (tile - p * tpp) * A.envs_per_tile;
            wts = io.weights + p * io.weights_stride;
            env0 = p * io.envs_per_policy + e0;
            envs = (int)min((int64_t)A.envs_per_tile, io.envs_per_policy - e0);
        }
        const int rows = envs * n;                 // valid rows of this tile
        const int64_t row0 = env0 * n;             // first global agent row
        __syncthreads();
        // ---- 0. observations -> bufA as obs^T[d][r]; rows beyond `rows` are zero so that they stay finite ----
        {
            const float *src = io.obs + row0 * D;
            for (int e = tid; e < kTile * D; e += kThreads) {
                const int r = e / D, c = e - r * D;
                bufA[c * kPitch + r] = (r < rows) ? __ldg(src + e) : 0.0f;
            }
        }
        __syncthreads();
        // ---- 1. h = tanh(obs W1^T + b1) -> bufB[128] ----
        {
            float acc[4][8];
            gemm64<128, kBWeights>(bufA, wts + o.enc_w1, kH1, D, acc);
            store_kmajor<128, true, true>(bufB, acc, wts + o.enc_b1);
        }
        __syncthreads();
        // ---- 2. E = tanh(h W2^T + b2) -> bufE ----
        {
            float acc[4][4];
            gemm64<64, kBWeights>(bufB, wts + o.enc_w2, kE, kH1, acc);
            store_kmajor<64, true, true>(bufE, acc, wts + o.enc_b2);
        }
        __syncthreads();
        // ---- 3. Q = E Wa^T -> bufA[0..63] ----
        float *QT = bufA, *HW = bufA + 64 * kPitch, *MT = bufB, *HT = bufB + 64 * kPitch;
        {
            float acc[4][4];
            gemm64<64, kBWeights>(bufE, wts + o.att_w, kE, kE, acc);
            store_kmajor<64, false, false>(QT, acc, nullptr);
        }
        __syncthreads();
        // ---- 4. S = Q E^T (64 x 64 tile product; only the per-env diagonal blocks are used) -> MT[j][i] ----
        {
            float acc[4][4];
            gemm64<64, kBShared>(QT, bufE, kPitch, kE, acc);
            store_kmajor<64, false, false>(MT, acc, nullptr);
        }
        __syncthreads();
        // ---- 5. row softmax over the agents of the same env; everything else in the row becomes 0 ----
        if (tid < kTile) {
            const int i = tid;
            if (i < rows) {
                const int j0 = (i / n) * n;
                float mx = -INFINITY;
                for (int j = j0; j < j0 + n; ++j) mx = fmaxf(mx, MT[j * kPitch + i]);
                float sum = 0.0f;
                for (int j = j0; j < j0 + n; ++j) { const float e = expf(MT[j * kPitch + i] - mx); MT[j * kPitch + i] = e; sum += e; }
                for (int j = 0; j < kTile; ++j) {
                    const bool in = (j >= j0) && (j < j0 + n);
                    MT[j * kPitch + i] = in ? MT[j * kPitch + i] / sum : 0.0f;
                }
            } else {
                for (int j = 0; j < kTile; ++j) MT[j * kPitch + i] = 0.0f;
            }
        }
        __syncthreads();
        if (io.attention) {   // agent_infos['attention_weights']: the UNMASKED softmax (comm_base_net.py:93)
            float *dst = io.attention + row0 * n;
            for (int e = tid; e < rows * n; e += kThreads) {
                const int r = e / n, jl = e - r * n;
                dst[e] = MT[((r / n) * n + jl) * kPitch + r];
            }
        }
        // ---- 6. graph convolutions ----
        for (int l = 0; l < L; ++l) {
            const float *Hin = (l == 0) ? bufE : HT;
            {
                float acc[4][4];
                gemm64<64, kBWeights>(Hin, wts + o.gcn_w + l * kE * kE, kE, kE, acc);   // H_l Wg_l  (Wg is (in,out))
                store_rowmajor(HW, acc);
            }
            // A_l = M * Range * chan_l, renormalised with eps = 1e-12 (comm_base_net.py:101-103) -> QT as A^T[j][i]
            if (tid < kTile) {
                const int i = tid;
                float *AT = QT;
                if (i < rows) {
                    const int el = i / n, il = i - el * n, j0 = el * n;
                    const int64_t env = env0 + el;
                    uint32_t m0 = 0xFFFFFFFFu, m1 = 0xFFFFFFFFu;
                    if (io.adj_bits) {
                        const uint32_t *p = io.adj_bits + (env * n + il) * W;
                        m0 &= __ldg(p);
                        if (W > 1) m1 &= __ldg(p + 1);
                    }
                    if (io.chan_bits) {
                        const uint32_t *p = io.chan_bits + ((env * L + l) * n + il) * W;
                        m0 &= __ldg(p);
                        if (W > 1) m1 &= __ldg(p + 1);
                    }
                    float sum = 0.0f;
                    for (int jl = 0; jl < n; ++jl) {
                        const uint32_t bit = ((jl < 32 ? m0 : m1) >> (jl & 31)) & 1u;
                        sum += bit ? MT[(j0 + jl) * kPitch + i] : 0.0f;
                    }
                    const float den = sum + 1e-12f;
                    for (int j = 0; j < kTile; ++j) {
                        const int jl = j - j0;
                        const bool in = (jl >= 0) && (jl < n) && ((((jl < 32 ? m0 : m1) >> (jl & 31)) & 1u) != 0);
                        AT[j * kPitch + i] = in ? MT[j * kPitch + i] / den : 0.0f;
                    }
                } else {
                    for (int j = 0; j < kTile; ++j) AT[j * kPitch + i] = 0.0f;
                }
            }
            __syncthreads();
            {
                float acc[4][4];
                gemm64<64, kBShared>(QT, HW, kPitch, kTile, acc);                       // A_l (H_l Wg_l)
                store_kmajor<64, true, true>(HT, acc, wts + o.gcn_b + l * kE);       // tanh(. + b)
            }
            __syncthreads();
        }
        // ---- 7. residual X = E + H_L (comm_categorical_mlp_policy.py:74-77) ----
        if (d.residual) {
            for (int e = tid; e < kE * kTile; e += kThreads) {
                const int k = e >> 6, r = e & 63;
                HT[k * kPitch + r] += bufE[k * kPitch + r];
            }
            __syncthreads();
        }
        // ---- 8..12. categorical head, softmax, mask, sampling ----
        head_and_sample<kMulti>(A, o, wts, HT, bufA, bufB, logit_s, rows, row0, env0, 0, n);
    }
}

static size_t small_smem_bytes() { return (size_t)(2 * 128 * kPitch + kE * kPitch + kTile * CM_ACTIONS) * sizeof(float); }

// ------------------------------------------------------------------------------------------------
// Teams larger than one tile (64 < n <= 256): one CTA per environment, the team is processed in 64-row
// chunks.  E^T and the two ping-pong H_l Wg_l matrices of the whole team live in a per-CTA scratch in
// global memory (<= 192 KB per CTA, a few tens of MB in total: L2 resident); the attention is evaluated
// block by block (64 queries x 64 keys) with the row maximum / normaliser computed once (they do not
// depend on the layer) and the scores recomputed per layer instead of keeping the n x n matrix.
// A_l (H_l Wg_l) is accumulated un-normalised and divided by (sum_j A_l + 1e-12) afterwards.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void load_chunk_kmajor(float *dstT, const float *src, int ld, int col0)
{
    for (int e = threadIdx.x; e < kE * kTile; e += kThreads) {
        const int k = e >> 6, r = e & 63;
        dstT[k * kPitch + r] = src[(size_t)k * ld + col0 + r];
    }
}

template <bool kMulti>
__global__ void __launch_bounds__(kThreads, 2) policy_large_kernel(const PolicyArgs A, int np, size_t ws_floats)
{
    extern __shared__ __align__(16) float sm[];
    float *bufA = sm;
    float *bufB = bufA + 128 * kPitch;
    float *bufE = bufB + 128 * kPitch;
    float *logit_s = bufE + kE * kPitch;
    float *rowmax = logit_s + kTile * CM_ACTIONS;   // [256]
    float *rowZ = rowmax + CM_MAX_AGENTS;           // [256]
    float *den_s = rowZ + CM_MAX_AGENTS;            // [64]
    const cm_policy_desc &d = A.d;
    const cm_policy_io &io = A.io;
    const int n = d.n_agents, D = d.obs_dim, L = d.n_layers, W = (n + 31) >> 5, nc = np >> 6;
    const Blob o = blob_layout(D, L);
    const float *__restrict__ wts = io.weights;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    float *ETg = io.workspace + (size_t)blockIdx.x * ws_floats;   // [64][np]   E^T of the whole team
    float *HW0 = ETg + (size_t)kE * np;                            // [np][64]   H_l Wg_l, ping
    float *HW1 = HW0 + (size_t)np * kE;                            // [np][64]   pong
    float *QT = bufA, *AT = bufA + 64 * kPitch, *ST = bufB, *HT = bufB + 64 * kPitch;

    for (int64_t b = blockIdx.x; b < io.n_envs; b += gridDim.x) {
        if constexpr (kMulti) wts = io.weights + (b / io.envs_per_policy) * io.weights_stride;
        __syncthreads();
        // ---------------- phase 1: encoder for every chunk; E^T and H_0 Wg_0 -> scratch ----------------
        for (int c = 0; c < nc; ++c) {
            const int r0 = c * kTile, vr = min(kTile, n - r0);
            const float *src = io.obs + ((size_t)b * n + r0) * D;
            for (int e = tid; e < kTile * D; e += kThreads) {
                const int r = e / D, col = e - r * D;
                bufA[col * kPitch + r] = (r < vr) ? __ldg(src + e) : 0.0f;
            }
            __syncthreads();
            {
                float acc[4][8];
                gemm64<128, kBWeights>(bufA, wts + o.enc_w1, kH1, D, acc);
                store_kmajor<128, true, true>(bufB, acc, wts + o.enc_b1);
            }
            __syncthreads();
            {
                float acc[4][4];
                gemm64<64, kBWeights>(bufB, wts + o.enc_w2, kE, kH1, acc);
                store_kmajor<64, true, true>(bufE, acc, wts + o.enc_b2);
            }
            __syncthreads();
            for (int e = tid; e < kE * kTile; e += kThreads) {
                const int k = e >> 6, r = e & 63;
                ETg[(size_t)k * np + r0 + r] = bufE[k * kPitch + r];
            }
            {
                float acc[4][4];
                gemm64<64, kBWeights>(bufE, wts + o.gcn_w, kE, kE, acc);
#pragma unroll
                for (int r = 0; r < 4; ++r)
                    *reinterpret_cast<float4 *>(HW0 + (size_t)(r0 + 4 * ty + r) * kE + 4 * tx) =
                        make_float4(acc[r][0], acc[r][1], acc[r][2], acc[r][3]);
            }
            __syncthreads();
        }
        // ---------------- phase 2: softmax statistics of every query row (layer independent) ----------------
        for (int qc = 0; qc < nc; ++qc) {
            const int q0 = qc * kTile;
            load_chunk_kmajor(bufE, ETg, np, q0);
            __syncthreads();
            {
                float acc[4][4];
                gemm64<64, kBWeights>(bufE, wts + o.att_w, kE, kE, acc);
                store_kmajor<64, false, false>(QT, acc, nullptr);
            }
            __syncthreads();
            float m = -INFINITY, Z = 0.0f;
            for (int kc = 0; kc < nc; ++kc) {
                const int k0 = kc * kTile, vk = min(kTile, n - k0);
                {
                    float acc[4][4];
                    gemm64<64, kBScratch>(QT, ETg + k0, np, kE, acc);
                    store_kmajor<64, false, false>(ST, acc, nullptr);
                }
                __syncthreads();
                if (tid < kTile) {
                    float bm = -INFINITY;
                    for (int j = 0; j < vk; ++j) bm = fmaxf(bm, ST[j * kPitch + tid]);
                    const float mn = fmaxf(m, bm);
                    float add = 0.0f;
                    for (int j = 0; j < vk; ++j) add += expf(ST[j * kPitch + tid] - mn);
                    Z = Z * expf(m - mn) + add;
                    m = mn;
                }
                __syncthreads();
            }
            if (tid < kTile) { rowmax[q0 + tid] = m; rowZ[q0 + tid] = Z; }
        }
        __syncthreads();
        // ---------------- phase 3: graph convolutions, then the head on the last layer's output ----------------
        for (int l = 0; l < L; ++l) {
            const float *HWin = (l & 1) ? HW1 : HW0;
            float *HWout = (l & 1) ? HW0 : HW1;
            for (int qc = 0; qc < nc; ++qc) {
                const int q0 = qc * kTile, vq = min(kTile, n - q0);
                load_chunk_kmajor(bufE, ETg, np, q0);
                __syncthreads();
                {
                    float acc[4][4];
                    gemm64<64, kBWeights>(bufE, wts + o.att_w, kE, kE, acc);
                    store_kmajor<64, false, false>(QT, acc, nullptr);
                }
                __syncthreads();
                float out[4][4];
#pragma unroll
                for (int r = 0; r < 4; ++r)
#pragma unroll
                    for (int q = 0; q < 4; ++q) out[r][q] = 0.0f;
                float den = 0.0f;
                for (int kc = 0; kc < nc; ++kc) {
                    const int k0 = kc * kTile, vk = min(kTile, n - k0);
                    {
                        float acc[4][4];
                        gemm64<64, kBScratch>(QT, ETg + k0, np, kE, acc);
                        store_kmajor<64, false, false>(ST, acc, nullptr);
                    }
                    __syncthreads();
                    if (tid < kTile) {
                        const int i = tid, qi = q0 + i;
                        uint32_t m0 = 0u, m1 = 0u;
                        float mx = 0.0f, z = 1.0f;
                        if (i < vq) {
                            m0 = m1 = 0xFFFFFFFFu;
                            const int w0 = k0 >> 5;
                            if (io.adj_bits) {
                                const uint32_t *p = io.adj_bits + ((size_t)b * n + qi) * W;
                                m0 &= __ldg(p + w0);
                                m1 &= (w0 + 1 < W) ? __ldg(p + w0 + 1) : 0u;
                            }
                            if (io.chan_bits) {
                                const uint32_t *p = io.chan_bits + (((size_t)b * L + l) * n + qi) * W;
                                m0 &= __ldg(p + w0);
                                m1 &= (w0 + 1 < W) ? __ldg(p + w0 + 1) : 0u;
                            }
                            mx = rowmax[qi];
                            z = rowZ[qi];
                        }
                        for (int j = 0; j < kTile; ++j) {
                            float pj = 0.0f, aj = 0.0f;
                            if (i < vq && j < vk) {
                                pj = expf(ST[j * kPitch + i] - mx) / z;
                                aj = (((j < 32 ? m0 : m1) >> (j & 31)) & 1u) ? pj : 0.0f;
                            }
                            ST[j * kPitch + i] = pj;
                            AT[j * kPitch + i] = aj;
                            den += aj;
                        }
                    }
                    __syncthreads();
                    if (l == 0 && io.attention) {      // unmasked softmax block -> attention[b][q0+i][k0+j]
                        for (int e = tid; e < kTile * kTile; e += kThreads) {
                            const int i = e >> 6, j = e & 63;
                            if (i < vq && j < vk) io.attention[((size_t)b * n + q0 + i) * n + k0 + j] = ST[j * kPitch + i];
                        }
                    }
                    gemm64<64, kBScratch, false>(AT, HWin + (size_t)k0 * kE, kE, kTile, out);
                    __syncthreads();
                }
                if (tid < kTile) den_s[tid] = den;
                __syncthreads();
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const float dn = den_s[4 * ty + r] + 1e-12f;     // comm_base_net.py:103
#pragma unroll
                    for (int q = 0; q < 4; ++q) out[r][q] = out[r][q] / dn;
                }
                store_kmajor<64, true, true>(HT, out, wts + o.gcn_b + l * kE);
                __syncthreads();
                if (l + 1 < L) {
                    float acc[4][4];
                    gemm64<64, kBWeights>(HT, wts + o.gcn_w + (l + 1) * kE * kE, kE, kE, acc);
#pragma unroll
                    for (int r = 0; r < 4; ++r)
                        *reinterpret_cast<float4 *>(HWout + (size_t)(q0 + 4 * ty + r) * kE + 4 * tx) =
                            make_float4(acc[r][0], acc[r][1], acc[r][2], acc[r][3]);
                } else {
                    if (d.residual) {
                        for (int e = tid; e < kE * kTile; e += kThreads) {
                            const int k = e >> 6, r = e & 63;
                            HT[k * kPitch + r] += bufE[k * kPitch + r];
                        }
                        __syncthreads();
                    }
                    head_and_sample<kMulti>(A, o, wts, HT, bufA, bufB, logit_s, vq, b * n + q0, b, q0, 0);
                }
                __syncthreads();
            }
        }
    }
}

static size_t large_smem_bytes() { return small_smem_bytes() + (size_t)(2 * CM_MAX_AGENTS + kTile) * sizeof(float); }
static int round_up_tile(int n) { return (n + kTile - 1) / kTile * kTile; }
static size_t large_ws_floats(int n) { return (size_t)3 * kE * round_up_tile(n); }

int launch_policy_tc(const cm_policy_desc *desc, const cm_policy_io *io, cudaStream_t stream);   // policy_tc_kernel.cu
int launch_policy_cent(const cm_policy_desc *desc, const cm_policy_io *io, cudaStream_t stream); // policy_cent_kernel.cu
size_t tc_large_ws_floats(int n, int64_t n_envs);                                                // policy_attn_kernel.cu

struct LaunchCache { int dev; int ctas_per_sm; int sms; };

template <typename K>
static int launch_geometry(K kernel, size_t smem, LaunchCache &cache)
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return set_cuda_error(cudaGetLastError(), CM_ENODEVICE);
    if (cache.dev != dev) {
        int sms = 0, ctas = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return set_cuda_error(cudaGetLastError(), CM_ECUDA);
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return set_cuda_error(e, CM_ECUDA);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas, kernel, kThreads, smem) != cudaSuccess)
            return set_cuda_error(cudaGetLastError(), CM_ECUDA);
        cache.dev = dev; cache.ctas_per_sm = ctas < 1 ? 1 : ctas; cache.sms = sms;
    }
    return CM_OK;
}

}  // namespace cm

extern "C" size_t cm_policy_blob_floats(int32_t obs_dim, int32_t n_layers)
{
    return (size_t)cm::blob_layout(obs_dim, n_layers).total;
}

extern "C" size_t cm_policy_workspace_bytes(int32_t n_agents, int64_t n_envs)
{
    if (n_agents <= cm::kTile || n_envs <= 0) return 0;
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    else cudaGetLastError();
    const int64_t ctas = n_envs < 2 * (int64_t)sms ? n_envs : 2 * (int64_t)sms;
    const size_t ffma = (size_t)ctas * cm::large_ws_floats(n_agents), tcp = cm::tc_large_ws_floats(n_agents, n_envs);
    return (ffma > tcp ? ffma : tcp) * sizeof(float);      // whichever kernel family the caller picks with desc.math
}

extern "C" int cm_policy_forward(const cm_policy_desc *desc, const cm_policy_io *io, cm_stream_t stream)
{
    using namespace cm;
    if (!desc || !io || !io->weights) return CM_EINVAL;
    // packed observations (cm_step_io.obs_bits) feed the tensor-core kernels of the Comm-DP / Obs-DP policies; every other path needs fp32 rows
    const bool packed_ok = io->obs_bits && (desc->math == 1 || desc->math == 2) && desc->kind != CM_POLICY_CENT;
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
    const bool multi = io->n_policies > 1;
    if (multi) {                   // several policies: equal env blocks, strides that hold a blob and keep 16-byte alignment
        const bool cent = desc->kind == CM_POLICY_CENT;
        const size_t blob = cent ? cm_policy_cent_blob_floats(desc->n_agents, desc->obs_dim) : cm_policy_blob_floats(desc->obs_dim, desc->n_layers);
        if (io->envs_per_policy < 1 || io->n_envs / io->n_policies != io->envs_per_policy || io->n_envs % io->n_policies != 0) return CM_EINVAL;
        if (io->weights_stride < (int64_t)blob || (io->weights_stride & 3) != 0) return CM_EINVAL;
        if (desc->math == 1 || desc->math == 2) {
            const size_t tcb = cent ? cm_policy_cent_tc_blob_floats(desc->n_agents, desc->obs_dim) : cm_policy_tc_blob_floats(desc->obs_dim, desc->n_layers);
            if (io->tc_weights_stride < (int64_t)tcb || (io->tc_weights_stride & 3) != 0) return CM_EINVAL;
        }
    }
    if (desc->kind == CM_POLICY_CENT) return launch_policy_cent(desc, io, (cudaStream_t)stream);
    if (desc->math == 1 || desc->math == 2) return launch_policy_tc(desc, io, (cudaStream_t)stream);
    if (desc->kind == CM_POLICY_DEC) return CM_EUNSUPPORTED;       // Obs-DP runs on the tensor-core kernel only
    if (desc->math != 0) return CM_EINVAL;
    PolicyArgs A;
    A.d = *desc;
    A.io = *io;
    cudaError_t e;
    if (desc->n_agents <= kTile) {
        A.envs_per_tile = kTile / desc->n_agents;
        A.n_tiles = (io->n_envs + A.envs_per_tile - 1) / A.envs_per_tile;
        if (multi) A.n_tiles = io->n_policies * ((io->envs_per_policy + A.envs_per_tile - 1) / A.envs_per_tile);
        const size_t smem = small_smem_bytes();
        static thread_local LaunchCache cache[2] = {{-1, 0, 0}, {-1, 0, 0}};
        int rc = multi ? launch_geometry(policy_small_kernel<true>, smem, cache[1]) : launch_geometry(policy_small_kernel<false>, smem, cache[0]);
        if (rc) return rc;
        const int64_t cap = (int64_t)cache[multi].sms * cache[multi].ctas_per_sm;   // persistent: a whole number of CTAs per SM
        const int grid = (int)(A.n_tiles < cap ? A.n_tiles : cap);
        if (multi) policy_small_kernel<true><<<grid, kThreads, smem, (cudaStream_t)stream>>>(A);
        else policy_small_kernel<false><<<grid, kThreads, smem, (cudaStream_t)stream>>>(A);
    } else {
        A.envs_per_tile = 0;
        A.n_tiles = io->n_envs;
        const size_t smem = large_smem_bytes();
        static thread_local LaunchCache caches[2] = {{-1, 0, 0}, {-1, 0, 0}};
        LaunchCache &cache = caches[multi];
        int rc = multi ? launch_geometry(policy_large_kernel<true>, smem, cache) : launch_geometry(policy_large_kernel<false>, smem, cache);
        if (rc) return rc;
        const size_t ws = large_ws_floats(desc->n_agents);
        if (!io->workspace || io->workspace_bytes < ws * sizeof(float)) return CM_EINVAL;
        int64_t cap = (int64_t)cache.sms * cache.ctas_per_sm;
        const int64_t fit = (int64_t)(io->workspace_bytes / (ws * sizeof(float)));
        if (fit < cap) cap = fit;
        const int grid = (int)(io->n_envs < cap ? io->n_envs : cap);
        if (multi) policy_large_kernel<true><<<grid, kThreads, smem, (cudaStream_t)stream>>>(A, round_up_tile(desc->n_agents), ws);
        else policy_large_kernel<false><<<grid, kThreads, smem, (cudaStream_t)stream>>>(A, round_up_tile(desc->n_agents), ws);
    }
    e = cudaGetLastError();
    if (e != cudaSuccess) return set_cuda_error(e, CM_ECUDA);
    return CM_OK;
}
