// ppo_net_kernels.cu — hand-written forward + backward of the comm-GNN for the PPO update (SURVEY.md §8f.1): the policy
// network of CommCategoricalMLPPolicy (comm_categorical_mlp_policy.py:48-96, comm_base_net.py:80-108) with the clipped
// surrogate / entropy objective of CentralizedMAPPO._compute_loss (centralized_ma_ppo.py:390-438, 540-589), and the value
// network of CommBaseCritic (comm_base_critic.py:11-120) with its Gaussian negative log-likelihood loss; the same for the
// Obs-DP policy, and for the CENT family: CentralizedCategoricalMLPPolicy (centralized_categorical_mlp_policy.py:61-97) and
// GaussianMLPBaseline (gaussian_mlp_baseline.py:83-117), one MLP over the concatenated observation with rows = env steps.
// Replaces the torch autograd graph (~150 library kernels per optimizer step) by ~30 launches of these kernels, all exact fp32 (FFMA):
//
//   net_dense_fwd     Y = act(X W + b)              rows x K x N register-tiled product, K <= 128, N in {32, 64, 128}
//   net_dense_bwd     dZ = dY (1 - Y^2);  dX (+)= dZ W^T;  dW += X^T dZ;  db += sum dZ        (one pass over the rows)
//   net_scores        M = softmax(Q E^T) per env                                             (attention_module.py:38-49)
//   net_agg_fwd       H = tanh(A~ V + b),  A~ = M.adj.chan / (rowsum + 1e-12)                 (comm_base_net.py:99-104)
//   net_agg_bwd       dV = A~^T dZ,  dM (+)= d(A~)/dM applied to dZ V^T
//   net_softmax_bwd   dS = M (dM - <dM, M>);  dQ = dS E;  dE += dS^T Q
//   net_policy_head   logits = g3 W4 + b4 -> softmax -> availability mask -> log-likelihood, entropy, clipped objective,
//                     d logits -> d g3, dW4, db4      net_critic_head: V(s) = sum_i (c1_i w2 + b2), Gaussian NLL, gradients
//   net_wide_fwd      CENT first layer Y = act(X W1 + b1), K = n*D up to 32 768          net_wide_dw   dW1 += X^T dZ1, db1 (and dW4)
//   net_cent_head     CENT logits [S][5n] = h3 W4 + b4 -> the per-agent tail of net_policy_head -> d logits, db4, dh3
//
// The n x n parts work on strips of 8 query rows per warp (register tiles of 8 rows x n/32 keys per lane for the dot
// products; coefficient strips staged through shared memory for the aggregations); a CTA owns as many whole envs as fit
// into 256 rows.  Activations live in a caller-provided workspace; the batch is walked in chunks of env steps.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "commarl_b200.h"
#include "common.cuh"
#include "policy_layout.cuh"
#include "tc_common.cuh"

namespace cm {

static constexpr int kNP = 68;          // pitch (floats) of a [row][64] array in shared memory: 128-bit reads of 8 consecutive rows hit 32 banks
static constexpr int kRows = 256;       // most rows (agents) of the envs a CTA of the per-env kernels owns at a time
static constexpr int kNetThreads = 256; // head kernels: one thread per row

// Sets of networks (cm_net_io.n_policies > 1): one launch runs gridDim.y members side by side, member m = blockIdx.y.  Each kernel
// moves its row pointers by m times one member's rows and its weight / gradient pointers by m times the blob strides, so no tile or
// env block holds rows of two members, and the partial sums a persistent CTA keeps over its tiles belong to one member.  With one
// network gridDim.y = 1 and every offset is 0.
template <typename T>
__device__ __forceinline__ T *mem_off(T *p, int64_t per_member)
{
    return p ? p + (int64_t)blockIdx.y * per_member : p;
}

// ------------------------------------------------------------------------------------------------------------------
// dense layers
// ------------------------------------------------------------------------------------------------------------------
// ASYNC: the X tiles (rows of K floats, 16-byte aligned) arrive by one bulk async copy per row (cp.async.bulk, mbarrier
// complete_tx) into a two-stage ring: the next tile is in flight while the products of the current one run.  Unaligned inputs
// (the observation rows, D floats) take the synchronous load.  ACT: 0 none, 1 tanh, 2 relu.
template <int N, int ACT, int ASYNC>
__global__ void __launch_bounds__(256) net_dense_fwd_kernel(const float *__restrict__ X, int ldx, const float *__restrict__ W,
                                                            const float *__restrict__ bias, float *__restrict__ Y, int ldy, int64_t R, int K,
                                                            int64_t wstr)
{
    constexpr int TX = N >= 64 ? 16 : N / 4, TY = 256 / TX, RI = 128 / TY, CJ = N / (4 * TX);
    X = mem_off(X, R * ldx); W = mem_off(W, wstr); bias = mem_off(bias, wstr); Y = mem_off(Y, R * ldy);
    extern __shared__ float4 smem4[];
    float *sm = reinterpret_cast<float *>(smem4);
    const int K4 = (K + 3) & ~3, KP = K4 + 4;
    float *Ws = sm;                    // [K4][N]
    float *Xs0 = sm + (size_t)K4 * N;  // [stages][128][KP]
    uint64_t *bars = reinterpret_cast<uint64_t *>(Xs0 + (size_t)(ASYNC ? 2 : 1) * 128 * KP);
    const int tid = threadIdx.x, tx = tid % TX, ty = tid / TX, warp = tid >> 5, lane = tid & 31;
    for (int i = tid; i < K4 * N; i += 256) Ws[i] = i < K * N ? W[i] : 0.0f;
    float bj[CJ * 4];
#pragma unroll
    for (int j = 0; j < CJ; ++j)
#pragma unroll
        for (int q = 0; q < 4; ++q) bj[4 * j + q] = bias ? bias[4 * tx + 64 * j + q] : 0.0f;
    const int64_t tiles = (R + 127) / 128;
    if (ASYNC) {
        if (tid == 0) { tc::mbar_init(&bars[0], 1); tc::mbar_init(&bars[1], 1); tc::fence_mbar_init(); }
        __syncthreads();
    }
    auto issue = [&](int64_t tile, int stage) {
        const int64_t r0 = tile * 128;
        const int rows = (int)min((int64_t)128, R - r0);
        if (tid == 0) tc::mbar_expect_tx(&bars[stage], (uint32_t)rows * (uint32_t)K * 4u);
        if (tid < rows) tc::bulk_g2s(Xs0 + (size_t)stage * 128 * KP + tid * KP, X + (r0 + tid) * ldx, (uint32_t)K * 4u, &bars[stage]);
    };
    if (ASYNC && (int64_t)blockIdx.x < tiles) issue(blockIdx.x, 0);
    int it = 0;
    for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x, ++it) {
        const int64_t r0 = t * 128;
        const float *Xs = Xs0;
        if (ASYNC) {
            const int stage = it & 1;
            if (t + gridDim.x < tiles) issue(t + gridDim.x, stage ^ 1);     // (that stage was last read before the barrier below)
            tc::mbar_wait(&bars[stage], (uint32_t)(it >> 1) & 1u);
            Xs = Xs0 + (size_t)stage * 128 * KP;
        } else {
            __syncthreads();
            float *Xw = Xs0;
            for (int r = warp; r < 128; r += 8) {
                const int64_t gr = r0 + r;
                for (int k = lane; k < K4; k += 32) Xw[r * KP + k] = (gr < R && k < K) ? X[gr * ldx + k] : 0.0f;
            }
            __syncthreads();
        }
        float acc[RI][CJ * 4];
#pragma unroll
        for (int i = 0; i < RI; ++i)
#pragma unroll
            for (int j = 0; j < CJ * 4; ++j) acc[i][j] = 0.0f;
        for (int k4 = 0; k4 < K4; k4 += 4) {
            float4 xa[RI];
#pragma unroll
            for (int i = 0; i < RI; ++i) xa[i] = *reinterpret_cast<const float4 *>(Xs + (ty + TY * i) * KP + k4);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                float4 wb[CJ];
#pragma unroll
                for (int j = 0; j < CJ; ++j) wb[j] = *reinterpret_cast<const float4 *>(Ws + (k4 + kk) * N + 4 * tx + 64 * j);
#pragma unroll
                for (int i = 0; i < RI; ++i) {
                    const float x = kk == 0 ? xa[i].x : (kk == 1 ? xa[i].y : (kk == 2 ? xa[i].z : xa[i].w));
#pragma unroll
                    for (int j = 0; j < CJ; ++j) {
                        acc[i][4 * j + 0] = fmaf(x, wb[j].x, acc[i][4 * j + 0]);
                        acc[i][4 * j + 1] = fmaf(x, wb[j].y, acc[i][4 * j + 1]);
                        acc[i][4 * j + 2] = fmaf(x, wb[j].z, acc[i][4 * j + 2]);
                        acc[i][4 * j + 3] = fmaf(x, wb[j].w, acc[i][4 * j + 3]);
                    }
                }
            }
        }
#pragma unroll
        for (int i = 0; i < RI; ++i) {
            const int64_t gr = r0 + ty + TY * i;
            if (gr >= R) continue;
#pragma unroll
            for (int j = 0; j < CJ; ++j) {
                float4 o;
                o.x = acc[i][4 * j + 0] + bj[4 * j + 0];
                o.y = acc[i][4 * j + 1] + bj[4 * j + 1];
                o.z = acc[i][4 * j + 2] + bj[4 * j + 2];
                o.w = acc[i][4 * j + 3] + bj[4 * j + 3];
                if (ACT == 1) { o.x = tanhf(o.x); o.y = tanhf(o.y); o.z = tanhf(o.z); o.w = tanhf(o.w); }
                if (ACT == 2) { o.x = fmaxf(o.x, 0.0f); o.y = fmaxf(o.y, 0.0f); o.z = fmaxf(o.z, 0.0f); o.w = fmaxf(o.w, 0.0f); }
                *reinterpret_cast<float4 *>(Y + gr * ldy + 4 * tx + 64 * j) = o;
            }
        }
        if (ASYNC) __syncthreads();                          // every warp is done with this stage: it may be refilled
    }
}

// One pass over the rows for the three gradients of Y = X W + b given dZ = dL/d(X W + b):
//   dX[r][k] = ((accumulate ? dX[r][k] : 0) + sum_n dZ[r][n] W[k][n]) * (xact ? act'(X[r][k]) : 1),  act' = 1 - X^2 (tanh) or,
//              with XRELU, [X > 0] (relu)
//   dW[k][n] += sum_r X[r][k] dZ[r][n];   db[n] += sum_r dZ[r][n].
// xact folds the activation derivative of the layer BELOW into the hand-over (X is that layer's output and already sits in
// shared memory), so every backward layer reads plain dZ rows.  16 warps: warps 0-7 form the dX tile while warps 8-15 reduce
// dW / db over the same tile in shared memory (two independent FMA streams on one copy of the operands); dW / db stay in
// registers over the tiles of a persistent CTA and are added to global memory once.  ASYNC: dZ and X tiles arrive by one bulk
// async copy per row into a two-stage ring (the next tile is in flight during the products); unaligned X rows (the
// observations) take the synchronous load.  ROWS = rows per tile (128, or 64 where two stages of 128 do not fit).
template <int N, int KMAX, int ROWS, int ASYNC, int XRELU = 0>
__global__ void __launch_bounds__(512) net_dense_bwd_kernel(const float *__restrict__ dZ, const float *__restrict__ X, int ldx,
                                                            const float *__restrict__ W, float *__restrict__ dX, int lddx, int accumulate,
                                                            int xact, float *__restrict__ dW, float *__restrict__ db, int64_t R, int K,
                                                            int64_t wstr, int64_t gstr)
{
    constexpr int NP = N + 4, KP = KMAX + 4;
    dZ = mem_off(dZ, R * N); X = mem_off(X, R * ldx); W = mem_off(W, wstr); dX = mem_off(dX, R * lddx);
    dW = mem_off(dW, gstr); db = mem_off(db, gstr);
    constexpr int RI = ROWS / 16;                                          // dX warps: rows ty + 16 i, k = kx + 16 j
    constexpr int KJ = KMAX / 16;
    constexpr int NX = N >= 64 ? 16 : N / 4, NJ = N / (4 * NX), KY = 256 / NX;   // dW warps: n = 4 nx + 64 j, k = 4 ky + 4 KY i
    constexpr int KI = (KMAX + 4 * KY - 1) / (4 * KY);
    constexpr int NB = NJ * 4, NACC = (RI * KJ > KI * 4 * NB) ? RI * KJ : KI * 4 * NB;
    constexpr int STAGE = ROWS * (NP + KP);                               // floats per stage: dZ tile, then X tile
    extern __shared__ float4 smem4[];
    float *sm = reinterpret_cast<float *>(smem4);
    float *Ws = sm;                         // [KMAX][NP]
    float *St0 = Ws + KMAX * NP;            // [stages][ dZs [ROWS][NP] | Xs [ROWS][KP] ]
    uint64_t *bars = reinterpret_cast<uint64_t *>(St0 + (size_t)(ASYNC ? 2 : 1) * STAGE);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool role_w = tid >= 256;         // (warp-uniform)
    const int t = tid & 255;
    for (int i = tid; i < KMAX * N; i += 512) {
        const int k = i / N, n = i - k * N;
        Ws[k * NP + n] = k < K ? W[k * N + n] : 0.0f;
    }
    float acc[NACC];                        // dX warps: the tile's [RI][KJ] block; dW warps: the running [KI * 4][NB] block
#pragma unroll
    for (int a = 0; a < NACC; ++a) acc[a] = 0.0f;
    float bacc = 0.0f;
    const int kx = t & 15, ty = t >> 4;
    const int nx = t % NX, ky = t / NX;
    const int64_t tiles = (R + ROWS - 1) / ROWS;
    if (ASYNC) {
        if (tid == 0) { tc::mbar_init(&bars[0], 1); tc::mbar_init(&bars[1], 1); tc::fence_mbar_init(); }
        __syncthreads();
        if (KMAX > K)                        // (columns the copies never write)
            for (int i = tid; i < 2 * ROWS * (KMAX - K); i += 512) {
                const int st = i / (ROWS * (KMAX - K)), q = i - st * ROWS * (KMAX - K);
                St0[(size_t)st * STAGE + ROWS * NP + (q / (KMAX - K)) * KP + K + q % (KMAX - K)] = 0.0f;
            }
    }
    auto issue = [&](int64_t tile, int stage) {
        const int64_t r0 = tile * ROWS;
        const int rows = (int)min((int64_t)ROWS, R - r0);
        float *dst = St0 + (size_t)stage * STAGE;
        if (tid == 0) tc::mbar_expect_tx(&bars[stage], (uint32_t)rows * (uint32_t)(N + K) * 4u);
        if (tid < rows) tc::bulk_g2s(dst + tid * NP, dZ + (r0 + tid) * N, (uint32_t)N * 4u, &bars[stage]);
        else if (tid >= 256 && tid - 256 < rows)
            tc::bulk_g2s(dst + ROWS * NP + (tid - 256) * KP, X + (r0 + tid - 256) * ldx, (uint32_t)K * 4u, &bars[stage]);
    };
    if (ASYNC) {
        __syncthreads();
        if ((int64_t)blockIdx.x < tiles) issue(blockIdx.x, 0);
    }
    int it = 0;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++it) {
        const int64_t r0 = tile * ROWS;
        const int rows = (int)min((int64_t)ROWS, R - r0);
        const float *dZs = St0, *Xs = St0 + ROWS * NP;
        if (ASYNC) {
            const int stage = it & 1;
            if (tile + gridDim.x < tiles) issue(tile + gridDim.x, stage ^ 1);
            tc::mbar_wait(&bars[stage], (uint32_t)(it >> 1) & 1u);
            dZs = St0 + (size_t)stage * STAGE;
            Xs = dZs + ROWS * NP;
        } else {
            __syncthreads();
            float *dZw = St0, *Xw = St0 + ROWS * NP;
            for (int i = tid; i < ROWS * (N / 4); i += 512) {
                const int r = i / (N / 4), q = i - r * (N / 4);
                const int64_t gr = r0 + r;
                *reinterpret_cast<float4 *>(dZw + r * NP + 4 * q) =
                    gr < R ? *reinterpret_cast<const float4 *>(dZ + gr * N + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            for (int r = warp; r < ROWS; r += 16) {
                const int64_t gr = r0 + r;
                for (int k = lane; k < KMAX; k += 32) Xw[r * KP + k] = (gr < R && k < K) ? X[gr * ldx + k] : 0.0f;
            }
            __syncthreads();
        }
        if (!role_w) {                                       // ---- dX tile
            if (dX) {
                // the old values of an accumulating pass are requested BEFORE the products: their latency hides behind the FMAs
                float old[RI * KJ];
#pragma unroll
                for (int i = 0; i < RI; ++i)
#pragma unroll
                    for (int j = 0; j < KJ; ++j) {
                        const int r = ty + 16 * i, k = kx + 16 * j;
                        old[i * KJ + j] = (accumulate && r < rows && k < K) ? dX[(r0 + r) * lddx + k] : 0.0f;
                    }
#pragma unroll
                for (int a = 0; a < RI * KJ; ++a) acc[a] = 0.0f;
                for (int n4 = 0; n4 < N; n4 += 4) {
                    float4 w[KJ];
#pragma unroll
                    for (int j = 0; j < KJ; ++j) w[j] = *reinterpret_cast<const float4 *>(Ws + (kx + 16 * j) * NP + n4);
#pragma unroll
                    for (int i = 0; i < RI; ++i) {
                        const float4 z = *reinterpret_cast<const float4 *>(dZs + (ty + 16 * i) * NP + n4);
#pragma unroll
                        for (int j = 0; j < KJ; ++j)
                            acc[i * KJ + j] = fmaf(z.x, w[j].x, fmaf(z.y, w[j].y, fmaf(z.z, w[j].z, fmaf(z.w, w[j].w, acc[i * KJ + j]))));
                    }
                }
#pragma unroll
                for (int i = 0; i < RI; ++i) {
                    const int r = ty + 16 * i;
                    if (r >= rows) continue;
#pragma unroll
                    for (int j = 0; j < KJ; ++j) {
                        const int k = kx + 16 * j;
                        if (k < K) {
                            float v = old[i * KJ + j] + acc[i * KJ + j];
                            if (xact) { const float x = Xs[r * KP + k]; if (XRELU) v = x > 0.0f ? v : 0.0f; else v *= 1.0f - x * x; }
                            dX[(r0 + r) * lddx + k] = v;
                        }
                    }
                }
            }
        } else {                                             // ---- dW += X^T dZ, db += sum dZ over the valid rows of the tile
            if (4 * ky < KMAX) {
#pragma unroll 2
                for (int r = 0; r < rows; ++r) {
                    float4 xa[KI], za[NJ];
#pragma unroll
                    for (int i = 0; i < KI; ++i)
                        xa[i] = (4 * ky + 4 * KY * i) < KMAX ? *reinterpret_cast<const float4 *>(Xs + r * KP + 4 * ky + 4 * KY * i)
                                                             : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                    for (int j = 0; j < NJ; ++j) za[j] = *reinterpret_cast<const float4 *>(dZs + r * NP + 4 * nx + 64 * j);
#pragma unroll
                    for (int i = 0; i < KI; ++i)
#pragma unroll
                        for (int j = 0; j < NJ; ++j) {
                            const float xv[4] = {xa[i].x, xa[i].y, xa[i].z, xa[i].w};
#pragma unroll
                            for (int a = 0; a < 4; ++a) {
                                float *o = acc + (4 * i + a) * NB + 4 * j;
                                o[0] = fmaf(xv[a], za[j].x, o[0]);
                                o[1] = fmaf(xv[a], za[j].y, o[1]);
                                o[2] = fmaf(xv[a], za[j].z, o[2]);
                                o[3] = fmaf(xv[a], za[j].w, o[3]);
                            }
                        }
                }
            }
            if (db && t < N) {
                float s = 0.0f;
                for (int r = 0; r < rows; ++r) s += dZs[r * NP + t];
                bacc += s;
            }
        }
        if (ASYNC) __syncthreads();                          // every warp is done with this stage: it may be refilled
    }
    if (role_w) {
        if (4 * ky < KMAX) {
#pragma unroll
            for (int i = 0; i < KI; ++i)
#pragma unroll
                for (int a = 0; a < 4; ++a) {
                    const int k = 4 * ky + 4 * KY * i + a;
                    if (k < K) {
#pragma unroll
                        for (int j = 0; j < NJ; ++j)
#pragma unroll
                            for (int b = 0; b < 4; ++b) atomicAdd(dW + k * N + 4 * nx + 64 * j + b, acc[(4 * i + a) * NB + 4 * j + b]);
                    }
                }
        }
        if (db && t < N) atomicAdd(db + t, bacc);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// n x n parts: strips of 8 query rows per warp
// ------------------------------------------------------------------------------------------------------------------
// acc[i][j] = < A[min(i, nr-1)][:], B[min(lane + 32 j, n-1)][:] > over the 64 columns; A, B rows in shared memory (pitch kNP)
template <int KT>
__device__ __forceinline__ void strip_dots(const float *As, int nr, const float *Bs, int n, int lane, float (&acc)[8][KT])
{
    int kb[KT];
#pragma unroll
    for (int j = 0; j < KT; ++j) kb[j] = min(lane + 32 * j, n - 1) * kNP;
    int ra[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) ra[i] = min(i, nr - 1) * kNP;
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < KT; ++j) acc[i][j] = 0.0f;
#pragma unroll 1
    for (int c = 0; c < 64; c += 4) {
        float4 b[KT];
#pragma unroll
        for (int j = 0; j < KT; ++j) b[j] = *reinterpret_cast<const float4 *>(Bs + kb[j] + c);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float4 a = *reinterpret_cast<const float4 *>(As + ra[i] + c);
#pragma unroll
            for (int j = 0; j < KT; ++j) acc[i][j] = fmaf(a.x, b[j].x, fmaf(a.y, b[j].y, fmaf(a.z, b[j].z, fmaf(a.w, b[j].w, acc[i][j]))));
        }
    }
}

// res[r][0..3] = sum_k Cs[4 h + r][k] B[k][4 l + {0..3}],  k < n,  h = lane / 16, l = lane % 16:  every lane owns FOUR of the 64
// columns, the two half-warps take alternate groups of four keys (one 128-bit operand read feeds 16 FMAs, half the shared-memory
// traffic per FMA of a two-column layout) and exchange their partial sums at the end; afterwards half h holds rows 4 h .. 4 h + 3 of
// the strip.  Cs [8][CP] holds zeros from n up to the next multiple of 8.
__device__ __forceinline__ void strip_agg4(const float *Cs, int CP, const float *Bs, int n, int lane, float (&res)[4][4])
{
    const int half = lane >> 4, l16 = lane & 15;
    float out[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i) out[i][0] = out[i][1] = out[i][2] = out[i][3] = 0.0f;
    for (int k = 4 * half; k < n; k += 8) {
        float4 b[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) b[q] = *reinterpret_cast<const float4 *>(Bs + min(k + q, n - 1) * kNP + 4 * l16);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float4 c = *reinterpret_cast<const float4 *>(Cs + i * CP + k);
            out[i][0] = fmaf(c.x, b[0].x, fmaf(c.y, b[1].x, fmaf(c.z, b[2].x, fmaf(c.w, b[3].x, out[i][0]))));
            out[i][1] = fmaf(c.x, b[0].y, fmaf(c.y, b[1].y, fmaf(c.z, b[2].y, fmaf(c.w, b[3].y, out[i][1]))));
            out[i][2] = fmaf(c.x, b[0].z, fmaf(c.y, b[1].z, fmaf(c.z, b[2].z, fmaf(c.w, b[3].z, out[i][2]))));
            out[i][3] = fmaf(c.x, b[0].w, fmaf(c.y, b[1].w, fmaf(c.z, b[2].w, fmaf(c.w, b[3].w, out[i][3]))));
        }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const float other = __shfl_xor_sync(0xFFFFFFFFu, out[i][c], 16);
            if ((i >> 2) == half) res[i & 3][c] = out[i][c] + other;
        }
}

// The warp's coefficient strip Cs [8][CP] (rows j0 .. j0 + nr - 1 of an env's n x n matrix) -> the env's TRANSPOSED scratch:
// CTenv[k][j0 + i] = Cs[i][k].  One lane per key writes the strip's eight values of its key as two 128-bit stores (a whole
// 32-byte sector) — eight 4-byte stores from eight instructions to the same sector cost the L2 eight partial writes.
template <int KT>
__device__ __forceinline__ void store_strip_transposed(float *__restrict__ CTenv, const float *Cs, int CP, int n, int j0, int nr, int lane)
{
    const bool vec = nr == 8 && (n & 3) == 0;          // (j0 is a multiple of 8, the scratch 16-byte aligned: rows of n floats stay aligned)
#pragma unroll
    for (int j = 0; j < KT; ++j) {
        const int k = lane + 32 * j;
        if (k < n) {
            float v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = Cs[i * CP + k];
            float *dst = CTenv + (int64_t)k * n + j0;
            if (vec) {
                *reinterpret_cast<float4 *>(dst) = make_float4(v[0], v[1], v[2], v[3]);
                *reinterpret_cast<float4 *>(dst + 4) = make_float4(v[4], v[5], v[6], v[7]);
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) if (i < nr) dst[i] = v[i];
            }
        }
    }
}

// rows [row0, row0 + rows) x 64 floats of a global [.][64] array -> shared memory (pitch kNP); optional second array
// and the product form dZ = a (1 - b^2)
__device__ __forceinline__ void load_rows64(float *dst, const float *__restrict__ src, int64_t row0, int rows, int tid)
{
    for (int i = tid; i < rows * 16; i += blockDim.x) {
        const int r = i >> 4, q = i & 15;
        *reinterpret_cast<float4 *>(dst + r * kNP + 4 * q) = *reinterpret_cast<const float4 *>(src + (row0 + r) * 64 + 4 * q);
    }
}

struct EnvBlock { int64_t s0; int ne, rows; };
__device__ __forceinline__ EnvBlock env_block(int64_t blk, int G, int n, int64_t S)
{
    EnvBlock b;
    b.s0 = blk * G;
    b.ne = (int)min((int64_t)G, S - b.s0);
    b.rows = b.ne * n;
    return b;
}

__device__ __forceinline__ uint32_t mask_word(const uint32_t *__restrict__ bits, int64_t row, int W, int j)
{
    return bits ? (j < W ? bits[row * W + j] : 0u) : 0xFFFFFFFFu;
}

// The masked, renormalised attention rows of a strip, A~ = M . adj . chan_l / (rowsum + 1e-12)  ->  the warp's Cs [8][CP]
// (zeros beyond n and in the rows >= nr).  The strip's 8 x n values of M are requested in ONE batch before any arithmetic (one
// global round trip per strip; the mask words follow while they are in flight).  sums[i] = rowsum + 1e-12; bit j of on[i]: this
// lane's key lane + 32 j is a neighbour of row i.
template <int KT>
__device__ __forceinline__ void strip_coef(float *Cs, int CP, float (&sums)[8], uint32_t (&on)[8], const float *__restrict__ M,
                                           const uint32_t *__restrict__ adj, const uint32_t *__restrict__ chan, int64_t s, int L, int l,
                                           int n, int W, int j0, int nr, int lane)
{
    float m[8][KT];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int64_t row = s * n + j0 + min(i, nr - 1);
#pragma unroll
        for (int j = 0; j < KT; ++j) m[i][j] = lane + 32 * j < n ? M[row * n + lane + 32 * j] : 0.0f;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int ri = j0 + min(i, nr - 1);
        uint32_t bits = 0u;
        float sum = 0.0f;
#pragma unroll
        for (int j = 0; j < KT; ++j) {
            const uint32_t wd = mask_word(adj, s * n + ri, W, j) & mask_word(chan, (s * L + l) * n + ri, W, j);
            const bool o = lane + 32 * j < n && ((wd >> lane) & 1u);
            bits |= (o ? 1u : 0u) << j;
            m[i][j] = o ? m[i][j] : 0.0f;
            sum += m[i][j];
        }
        sum = warp_sumf(sum) + 1e-12f;
        sums[i] = sum;
        on[i] = bits;
#pragma unroll
        for (int j = 0; j < KT; ++j) Cs[i * CP + lane + 32 * j] = i < nr ? m[i][j] / sum : 0.0f;
    }
}

// M[s][i][:] = softmax_k < Q[s][i], E[s][k] >
template <int KT, int THREADS>
__global__ void __launch_bounds__(THREADS, THREADS == 256 ? (KT <= 2 ? 3 : 2) : 1) net_scores_kernel(const float *__restrict__ Q, const float *__restrict__ E,
                                                                 float *__restrict__ M, int n, int G, int cap, int64_t S)
{
    extern __shared__ float4 smem4[];
    float *Es = reinterpret_cast<float *>(smem4), *Qs = Es + cap * kNP;
    Q = mem_off(Q, S * n * 64); E = mem_off(E, S * n * 64); M = mem_off(M, S * n * n);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ns = (n + 7) >> 3;
    const int64_t nblk = (S + G - 1) / G;
    for (int64_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const EnvBlock eb = env_block(blk, G, n, S);
        __syncthreads();
        load_rows64(Es, E, eb.s0 * n, eb.rows, tid);
        load_rows64(Qs, Q, eb.s0 * n, eb.rows, tid);
        __syncthreads();
        for (int st = warp; st < eb.ne * ns; st += THREADS / 32) {
            const int g = st / ns, j0 = (st - g * ns) * 8, nr = min(8, n - j0);
            float acc[8][KT];
            strip_dots<KT>(Qs + (g * n + j0) * kNP, nr, Es + g * n * kNP, n, lane, acc);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                float mx = -INFINITY;
#pragma unroll
                for (int j = 0; j < KT; ++j) if (lane + 32 * j < n) mx = fmaxf(mx, acc[i][j]);
                mx = warp_max(mx);
                float sum = 0.0f;
#pragma unroll
                for (int j = 0; j < KT; ++j) { acc[i][j] = lane + 32 * j < n ? expf(acc[i][j] - mx) : 0.0f; sum += acc[i][j]; }
                sum = warp_sumf(sum);
                if (i < nr) {
                    float *mrow = M + ((eb.s0 + g) * n + j0 + i) * (int64_t)n;
#pragma unroll
                    for (int j = 0; j < KT; ++j) if (lane + 32 * j < n) mrow[lane + 32 * j] = acc[i][j] / sum;
                }
            }
        }
    }
}

// H[s][i][:] = tanh( sum_k A~[i][k] V[s][k][:] + b ),  A~ = M . adj . chan_l / (rowsum + 1e-12);  optional Xout = res + H
template <int KT, int THREADS>
__global__ void __launch_bounds__(THREADS, THREADS == 256 ? (KT <= 2 ? 3 : 2) : 1) net_agg_fwd_kernel(const float *__restrict__ M, const uint32_t *__restrict__ adj,
                                                                  const uint32_t *__restrict__ chan, int L, int l,
                                                                  const float *__restrict__ V, const float *__restrict__ bias,
                                                                  float *__restrict__ H, const float *__restrict__ res_in,
                                                                  float *__restrict__ Xout, int n, int G, int cap, int64_t S, int64_t wstr)
{
    extern __shared__ float4 smem4[];
    constexpr int CP = KT * 32 + 4;
    float *Vs = reinterpret_cast<float *>(smem4), *Call = Vs + cap * kNP;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    float *Cs = Call + warp * 8 * CP;
    const int ns = (n + 7) >> 3, W = (n + 31) >> 5;
    M = mem_off(M, S * n * n); adj = mem_off(adj, S * n * W); chan = mem_off(chan, S * L * n * W); V = mem_off(V, S * n * 64);
    bias = mem_off(bias, wstr); H = mem_off(H, S * n * 64); res_in = mem_off(res_in, S * n * 64); Xout = mem_off(Xout, S * n * 64);
    const float4 bv = *reinterpret_cast<const float4 *>(bias + 4 * (lane & 15));
    const int64_t nblk = (S + G - 1) / G;
    for (int64_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const EnvBlock eb = env_block(blk, G, n, S);
        __syncthreads();
        load_rows64(Vs, V, eb.s0 * n, eb.rows, tid);
        __syncthreads();
        for (int st = warp; st < eb.ne * ns; st += THREADS / 32) {
            const int g = st / ns, j0 = (st - g * ns) * 8, nr = min(8, n - j0);
            const int64_t s = eb.s0 + g;
            __syncwarp();
            {
                float sums[8];
                uint32_t on[8];
                strip_coef<KT>(Cs, CP, sums, on, M, adj, chan, s, L, l, n, W, j0, nr, lane);
            }
            __syncwarp();
            float res[4][4];
            strip_agg4(Cs, CP, Vs + g * n * kNP, n, lane, res);
            const int half = lane >> 4, l16 = lane & 15;
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int i = 4 * half + r;
                if (i < nr) {
                    const int64_t row = s * n + j0 + i;
                    const float4 h = make_float4(tanhf(res[r][0] + bv.x), tanhf(res[r][1] + bv.y), tanhf(res[r][2] + bv.z), tanhf(res[r][3] + bv.w));
                    *reinterpret_cast<float4 *>(H + row * 64 + 4 * l16) = h;
                    if (Xout) {
                        const float4 e = *reinterpret_cast<const float4 *>(res_in + row * 64 + 4 * l16);
                        *reinterpret_cast<float4 *>(Xout + row * 64 + 4 * l16) = make_float4(e.x + h.x, e.y + h.y, e.z + h.z, e.w + h.w);
                    }
                }
            }
        }
    }
}

// Backward of one graph-convolution layer's aggregation.  dZ = dH (1 - H^2);  dV = A~^T dZ;  db += sum dZ;
// dA~ = dZ V^T;  dM_l = mask (dA~ - <dA~, A~>) / (rowsum + 1e-12) (this layer's own array).  A~ strips are parked TRANSPOSED in CT so that the
// second pass (key strips) reads contiguous coefficient rows.
template <int KT, int THREADS>
__global__ void __launch_bounds__(THREADS, THREADS == 256 ? (KT <= 2 ? 3 : 2) : 1) net_agg_bwd_kernel(const float *__restrict__ M, const uint32_t *__restrict__ adj,
                                                                  const uint32_t *__restrict__ chan, int L, int l,
                                                                  const float *__restrict__ V, const float *__restrict__ H,
                                                                  const float *__restrict__ dH, float *__restrict__ dV,
                                                                  float *__restrict__ dM, float *__restrict__ CT,
                                                                  float *__restrict__ db, int n, int G, int cap, int64_t S, int64_t gstr)
{
    extern __shared__ float4 smem4[];
    constexpr int CP = KT * 32 + 4;
    float *Vs = reinterpret_cast<float *>(smem4), *dZs = Vs + cap * kNP, *Call = dZs + cap * kNP;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    float *Cs = Call + warp * 8 * CP;
    const int ns = (n + 7) >> 3, W = (n + 31) >> 5;
    M = mem_off(M, S * n * n); adj = mem_off(adj, S * n * W); chan = mem_off(chan, S * L * n * W); V = mem_off(V, S * n * 64);
    H = mem_off(H, S * n * 64); dH = mem_off(dH, S * n * 64); dV = mem_off(dV, S * n * 64); dM = mem_off(dM, S * n * n);
    CT = mem_off(CT, S * n * n); db = mem_off(db, gstr);
    float bacc = 0.0f;
    const int64_t nblk = (S + G - 1) / G;
    for (int64_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const EnvBlock eb = env_block(blk, G, n, S);
        __syncthreads();
        load_rows64(Vs, V, eb.s0 * n, eb.rows, tid);
        for (int i = tid; i < eb.rows * 16; i += THREADS) {
            const int r = i >> 4, q = i & 15;
            const int64_t o = (eb.s0 * n + r) * 64 + 4 * q;
            float4 g = *reinterpret_cast<const float4 *>(dH + o);
            const float4 h = *reinterpret_cast<const float4 *>(H + o);
            g.x *= 1.0f - h.x * h.x; g.y *= 1.0f - h.y * h.y; g.z *= 1.0f - h.z * h.z; g.w *= 1.0f - h.w * h.w;
            *reinterpret_cast<float4 *>(dZs + r * kNP + 4 * q) = g;
        }
        __syncthreads();
        if (tid < 64) {
            float sacc = 0.0f;
            for (int r = 0; r < eb.rows; ++r) sacc += dZs[r * kNP + tid];
            bacc += sacc;
        }
        for (int st = warp; st < eb.ne * ns; st += THREADS / 32) {          // pass 1: query strips
            const int g = st / ns, j0 = (st - g * ns) * 8, nr = min(8, n - j0);
            const int64_t s = eb.s0 + g;
            // A~ first (its global loads go out in one batch), then dA~ = dZ V^T, then dM of THIS layer (no read-modify-write: the
            // layers' contributions are summed by net_softmax_bwd)
            float sums[8];
            uint32_t on[8];
            __syncwarp();
            strip_coef<KT>(Cs, CP, sums, on, M, adj, chan, s, L, l, n, W, j0, nr, lane);
            float acc[8][KT];
            strip_dots<KT>(dZs + (g * n + j0) * kNP, nr, Vs + g * n * kNP, n, lane, acc);
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                if (i >= nr) continue;                        // (warp-uniform)
                float dot = 0.0f;
#pragma unroll
                for (int j = 0; j < KT; ++j) dot = fmaf(acc[i][j], Cs[i * CP + lane + 32 * j], dot);
                dot = warp_sumf(dot);
                float *drow = dM + (s * n + j0 + i) * (int64_t)n;
#pragma unroll
                for (int j = 0; j < KT; ++j)
                    if (lane + 32 * j < n) drow[lane + 32 * j] = ((on[i] >> j) & 1u) ? (acc[i][j] - dot) / sums[i] : 0.0f;
            }
            store_strip_transposed<KT>(CT + s * n * n, Cs, CP, n, j0, nr, lane);      // A~^T for the second pass
        }
        __syncthreads();
        for (int st = warp; st < eb.ne * ns; st += THREADS / 32) {          // pass 2: key strips
            const int g = st / ns, k0 = (st - g * ns) * 8, nk = min(8, n - k0);
            const int64_t s = eb.s0 + g;
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < KT; ++j) {
                    const int q = lane + 32 * j;
                    Cs[i * CP + q] = (i < nk && q < n) ? CT[(s * n + k0 + i) * n + q] : 0.0f;
                }
            __syncwarp();
            float res[4][4];
            strip_agg4(Cs, CP, dZs + g * n * kNP, n, lane, res);
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int i = 4 * (lane >> 4) + r;
                if (i < nk)
                    *reinterpret_cast<float4 *>(dV + (s * n + k0 + i) * 64 + 4 * (lane & 15)) = make_float4(res[r][0], res[r][1], res[r][2], res[r][3]);
            }
        }
    }
    if (db && tid < 64) atomicAdd(db + tid, bacc);
}

// dS = M (dM - <dM, M>) per query row;  dQ = dS E;  dE += dS^T Q
template <int KT, int THREADS>
__global__ void __launch_bounds__(THREADS, THREADS == 256 ? (KT <= 2 ? 3 : 2) : 1) net_softmax_bwd_kernel(const float *__restrict__ M, const float *__restrict__ dM,
                                                                      int L, int64_t dm_stride,
                                                                      const float *__restrict__ E, const float *__restrict__ Q,
                                                                      float *__restrict__ dQ, float *__restrict__ dE,
                                                                      float *__restrict__ CT, int n, int G, int cap, int64_t S)
{
    extern __shared__ float4 smem4[];
    constexpr int CP = KT * 32 + 4;
    float *Es = reinterpret_cast<float *>(smem4), *Qs = Es + cap * kNP, *Call = Qs + cap * kNP;
    M = mem_off(M, S * n * n); dM = mem_off(dM, S * n * n); E = mem_off(E, S * n * 64); Q = mem_off(Q, S * n * 64);
    dQ = mem_off(dQ, S * n * 64); dE = mem_off(dE, S * n * 64); CT = mem_off(CT, S * n * n);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    float *Cs = Call + warp * 8 * CP;
    const int ns = (n + 7) >> 3;
    const int64_t nblk = (S + G - 1) / G;
    for (int64_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const EnvBlock eb = env_block(blk, G, n, S);
        __syncthreads();
        load_rows64(Es, E, eb.s0 * n, eb.rows, tid);
        load_rows64(Qs, Q, eb.s0 * n, eb.rows, tid);
        __syncthreads();
        for (int st = warp; st < eb.ne * ns; st += THREADS / 32) {          // pass 1: query strips
            const int g = st / ns, j0 = (st - g * ns) * 8, nr = min(8, n - j0);
            const int64_t s = eb.s0 + g;
            __syncwarp();
#pragma unroll
            for (int h = 0; h < 2; ++h) {                    // four rows at a time: their loads (M and the layers' dM) in one batch
                float m[4][KT], d[4][KT];
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const int64_t row = s * n + j0 + min(4 * h + r, nr - 1);
#pragma unroll
                    for (int j = 0; j < KT; ++j) {
                        const int k = lane + 32 * j;
                        m[r][j] = k < n ? M[row * n + k] : 0.0f;
                        d[r][j] = k < n ? dM[row * n + k] : 0.0f;
                    }
                    for (int ll = 1; ll < L; ++ll)
#pragma unroll
                        for (int j = 0; j < KT; ++j) {
                            const int k = lane + 32 * j;
                            if (k < n) d[r][j] += dM[ll * dm_stride + row * n + k];
                        }
                }
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const int i = 4 * h + r;
                    float dot = 0.0f;
#pragma unroll
                    for (int j = 0; j < KT; ++j) dot = fmaf(m[r][j], d[r][j], dot);
                    dot = warp_sumf(dot);
#pragma unroll
                    for (int j = 0; j < KT; ++j) Cs[i * CP + lane + 32 * j] = i < nr ? m[r][j] * (d[r][j] - dot) : 0.0f;
                }
            }
            __syncwarp();
            store_strip_transposed<KT>(CT + s * n * n, Cs, CP, n, j0, nr, lane);      // dS^T for the second pass
            float res[4][4];
            strip_agg4(Cs, CP, Es + g * n * kNP, n, lane, res);
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int i = 4 * (lane >> 4) + r;
                if (i < nr)
                    *reinterpret_cast<float4 *>(dQ + (s * n + j0 + i) * 64 + 4 * (lane & 15)) = make_float4(res[r][0], res[r][1], res[r][2], res[r][3]);
            }
        }
        __syncthreads();
        for (int st = warp; st < eb.ne * ns; st += THREADS / 32) {          // pass 2: key strips
            const int g = st / ns, k0 = (st - g * ns) * 8, nk = min(8, n - k0);
            const int64_t s = eb.s0 + g;
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < KT; ++j) {
                    const int q = lane + 32 * j;
                    Cs[i * CP + q] = (i < nk && q < n) ? CT[(s * n + k0 + i) * n + q] : 0.0f;
                }
            __syncwarp();
            float res[4][4];
            strip_agg4(Cs, CP, Qs + g * n * kNP, n, lane, res);
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int i = 4 * (lane >> 4) + r;
                if (i < nk) {
                    float4 *p = reinterpret_cast<float4 *>(dE + (s * n + k0 + i) * 64 + 4 * (lane & 15));
                    const float4 o = *p;
                    *p = make_float4(o.x + res[r][0], o.y + res[r][1], o.z + res[r][2], o.w + res[r][3]);
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// small teams (n <= 8): one THREAD per agent row.  A strip of 8 query rows would be mostly padding here (n = 3, 4 in
// BASELINE configs 1 and 2); instead every thread keeps its row's 64 columns in registers and walks the <= 8 rows of its own
// env in shared memory.  Same formulas, same outputs as the strip kernels above.
// ------------------------------------------------------------------------------------------------------------------
static constexpr int kSmallN = 8, kSmallRows = 128;

__device__ __forceinline__ void row_load64(float (&v)[64], const float *__restrict__ src)
{
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        const float4 x = *reinterpret_cast<const float4 *>(src + 4 * q);
        v[4 * q] = x.x; v[4 * q + 1] = x.y; v[4 * q + 2] = x.z; v[4 * q + 3] = x.w;
    }
}
// out[:] = sum_k coef[k] rows[k][:], k < n (rows in shared memory, pitch kNP)
__device__ __forceinline__ void row_combine(float (&out)[64], const float (&coef)[kSmallN], const float *rows, int n)
{
#pragma unroll
    for (int c = 0; c < 64; ++c) out[c] = 0.0f;
    for (int k = 0; k < n; ++k) {
        float ck = 0.0f;
#pragma unroll
        for (int j = 0; j < kSmallN; ++j) if (j == k) ck = coef[j];
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const float4 b = *reinterpret_cast<const float4 *>(rows + k * kNP + 4 * q);
            out[4 * q] = fmaf(ck, b.x, out[4 * q]); out[4 * q + 1] = fmaf(ck, b.y, out[4 * q + 1]);
            out[4 * q + 2] = fmaf(ck, b.z, out[4 * q + 2]); out[4 * q + 3] = fmaf(ck, b.w, out[4 * q + 3]);
        }
    }
}
__device__ __forceinline__ float row_dot(const float (&v)[64], const float *row)
{
    float s0 = 0.0f, s1 = 0.0f;
#pragma unroll
    for (int q = 0; q < 16; q += 2) {
        const float4 a = *reinterpret_cast<const float4 *>(row + 4 * q), b = *reinterpret_cast<const float4 *>(row + 4 * q + 4);
        s0 = fmaf(v[4 * q], a.x, fmaf(v[4 * q + 1], a.y, fmaf(v[4 * q + 2], a.z, fmaf(v[4 * q + 3], a.w, s0))));
        s1 = fmaf(v[4 * q + 4], b.x, fmaf(v[4 * q + 5], b.y, fmaf(v[4 * q + 6], b.z, fmaf(v[4 * q + 7], b.w, s1))));
    }
    return s0 + s1;
}
__device__ __forceinline__ void row_store64(float *__restrict__ dst, const float (&v)[64])
{
#pragma unroll
    for (int q = 0; q < 16; ++q) *reinterpret_cast<float4 *>(dst + 4 * q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
}
// masked, renormalised attention row of agent `row` (global row index) in layer l: a[k], k < n; returns rowsum + 1e-12
__device__ __forceinline__ float small_coef(float (&a)[kSmallN], const float *__restrict__ M, const uint32_t *__restrict__ adj,
                                            const uint32_t *__restrict__ chan, int64_t row, int64_t chan_row, int n)
{
    const uint32_t wd = (adj ? adj[row] : 0xFFFFFFFFu) & (chan ? chan[chan_row] : 0xFFFFFFFFu);
    float sum = 0.0f;
#pragma unroll
    for (int k = 0; k < kSmallN; ++k) {
        a[k] = (k < n && ((wd >> k) & 1u)) ? M[row * n + k] : 0.0f;
        sum += a[k];
    }
    sum += 1e-12f;
#pragma unroll
    for (int k = 0; k < kSmallN; ++k) a[k] = a[k] / sum;
    return sum;
}

__global__ void __launch_bounds__(kSmallRows) net_small_scores_kernel(const float *__restrict__ Q, const float *__restrict__ E,
                                                                      float *__restrict__ M, int n, int G, int64_t S)
{
    __shared__ __align__(16) float Es[kSmallRows * kNP];
    const int tid = threadIdx.x;
    Q = mem_off(Q, S * n * 64); E = mem_off(E, S * n * 64); M = mem_off(M, S * n * n);
    const int64_t nblk = (S + G - 1) / G;
    for (int64_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const EnvBlock eb = env_block(blk, G, n, S);
        __syncthreads();
        load_rows64(Es, E, eb.s0 * n, eb.rows, tid);
        __syncthreads();
        if (tid >= eb.rows) continue;
        const int e = tid / n;
        const int64_t row = eb.s0 * n + tid;
        float q[64];
        row_load64(q, Q + row * 64);
        float sc[kSmallN];
        float mx = -INFINITY;
#pragma unroll
        for (int k = 0; k < kSmallN; ++k) {
            sc[k] = k < n ? row_dot(q, Es + (e * n + k) * kNP) : -INFINITY;
            mx = fmaxf(mx, sc[k]);
        }
        float sum = 0.0f;
#pragma unroll
        for (int k = 0; k < kSmallN; ++k) { sc[k] = k < n ? expf(sc[k] - mx) : 0.0f; sum += sc[k]; }
#pragma unroll
        for (int k = 0; k < kSmallN; ++k) if (k < n) M[row * n + k] = sc[k] / sum;
    }
}

__global__ void __launch_bounds__(kSmallRows) net_small_agg_fwd_kernel(const float *__restrict__ M, const uint32_t *__restrict__ adj,
                                                                       const uint32_t *__restrict__ chan, int L, int l,
                                                                       const float *__restrict__ V, const float *__restrict__ bias,
                                                                       float *__restrict__ H, const float *__restrict__ res,
                                                                       float *__restrict__ Xout, int n, int G, int64_t S, int64_t wstr)
{
    __shared__ __align__(16) float Vs[kSmallRows * kNP];
    __shared__ float bs[64];
    const int tid = threadIdx.x;
    M = mem_off(M, S * n * n); adj = mem_off(adj, S * n); chan = mem_off(chan, S * L * n); V = mem_off(V, S * n * 64);
    bias = mem_off(bias, wstr); H = mem_off(H, S * n * 64); res = mem_off(res, S * n * 64); Xout = mem_off(Xout, S * n * 64);
    if (tid < 64) bs[tid] = bias[tid];
    const int64_t nblk = (S + G - 1) / G;
    for (int64_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const EnvBlock eb = env_block(blk, G, n, S);
        __syncthreads();
        load_rows64(Vs, V, eb.s0 * n, eb.rows, tid);
        __syncthreads();
        if (tid >= eb.rows) continue;
        const int e = tid / n, i = tid - e * n;
        const int64_t s = eb.s0 + e, row = s * n + i;
        float a[kSmallN], out[64];
        small_coef(a, M, adj, chan, row, (s * L + l) * n + i, n);
        row_combine(out, a, Vs + e * n * kNP, n);
#pragma unroll
        for (int c = 0; c < 64; ++c) out[c] = tanhf(out[c] + bs[c]);
        row_store64(H + row * 64, out);
        if (Xout) {
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const float4 x = *reinterpret_cast<const float4 *>(res + row * 64 + 4 * q);
                *reinterpret_cast<float4 *>(Xout + row * 64 + 4 * q) =
                    make_float4(x.x + out[4 * q], x.y + out[4 * q + 1], x.z + out[4 * q + 2], x.w + out[4 * q + 3]);
            }
        }
    }
}

__global__ void __launch_bounds__(kSmallRows) net_small_agg_bwd_kernel(const float *__restrict__ M, const uint32_t *__restrict__ adj,
                                                                       const uint32_t *__restrict__ chan, int L, int l,
                                                                       const float *__restrict__ V, const float *__restrict__ H,
                                                                       const float *__restrict__ dH, float *__restrict__ dV,
                                                                       float *__restrict__ dM, float *__restrict__ db,
                                                                       int n, int G, int64_t S, int64_t gstr)
{
    extern __shared__ float4 smem4[];
    float *Vs = reinterpret_cast<float *>(smem4), *dZs = Vs + kSmallRows * kNP, *As = dZs + kSmallRows * kNP;
    const int tid = threadIdx.x;
    M = mem_off(M, S * n * n); adj = mem_off(adj, S * n); chan = mem_off(chan, S * L * n); V = mem_off(V, S * n * 64);
    H = mem_off(H, S * n * 64); dH = mem_off(dH, S * n * 64); dV = mem_off(dV, S * n * 64); dM = mem_off(dM, S * n * n);
    db = mem_off(db, gstr);
    float bacc = 0.0f;
    const int64_t nblk = (S + G - 1) / G;
    for (int64_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const EnvBlock eb = env_block(blk, G, n, S);
        __syncthreads();
        load_rows64(Vs, V, eb.s0 * n, eb.rows, tid);
        __syncthreads();
        const bool active = tid < eb.rows;
        const int e = active ? tid / n : 0, i = active ? tid - e * n : 0;
        const int64_t s = eb.s0 + e, row = s * n + i;
        if (active) {
            float dz[64];
            {
                float h[64];
                row_load64(dz, dH + row * 64);
                row_load64(h, H + row * 64);
#pragma unroll
                for (int c = 0; c < 64; ++c) dz[c] *= 1.0f - h[c] * h[c];
            }
            row_store64(dZs + tid * kNP, dz);
            float a[kSmallN];
            const float sum = small_coef(a, M, adj, chan, row, (s * L + l) * n + i, n);
            float da[kSmallN];
            float dot = 0.0f;
#pragma unroll
            for (int k = 0; k < kSmallN; ++k) {
                da[k] = k < n ? row_dot(dz, Vs + (e * n + k) * kNP) : 0.0f;
                dot = fmaf(da[k], a[k], dot);
                As[tid * kSmallN + k] = a[k];
            }
            const uint32_t wd = (adj ? adj[row] : 0xFFFFFFFFu) & (chan ? chan[(s * L + l) * n + i] : 0xFFFFFFFFu);
#pragma unroll
            for (int k = 0; k < kSmallN; ++k)
                if (k < n) {
                    const float dm = ((wd >> k) & 1u) ? (da[k] - dot) / sum : 0.0f;
                    dM[row * n + k] = dm;                 // (this layer's own array)
                }
        }
        __syncthreads();
        if (tid < 64) {
            float sacc = 0.0f;
            for (int r = 0; r < eb.rows; ++r) sacc += dZs[r * kNP + tid];
            bacc += sacc;
        }
        if (active) {                                   // dV of key row (e, i): sum over the env's query rows
            float ct[kSmallN], out[64];
#pragma unroll
            for (int q = 0; q < kSmallN; ++q) ct[q] = q < n ? As[(e * n + q) * kSmallN + i] : 0.0f;
            row_combine(out, ct, dZs + e * n * kNP, n);
            row_store64(dV + row * 64, out);
        }
    }
    if (db && tid < 64) atomicAdd(db + tid, bacc);
}

__global__ void __launch_bounds__(kSmallRows) net_small_softmax_bwd_kernel(const float *__restrict__ M, const float *__restrict__ dM, int L,
                                                                           int64_t dm_stride, const float *__restrict__ E,
                                                                           const float *__restrict__ Q, float *__restrict__ dQ,
                                                                           float *__restrict__ dE, int n, int G, int64_t S)
{
    extern __shared__ float4 smem4[];
    float *Es = reinterpret_cast<float *>(smem4), *Qs = Es + kSmallRows * kNP, *Ds = Qs + kSmallRows * kNP;
    const int tid = threadIdx.x;
    M = mem_off(M, S * n * n); dM = mem_off(dM, S * n * n); E = mem_off(E, S * n * 64); Q = mem_off(Q, S * n * 64);
    dQ = mem_off(dQ, S * n * 64); dE = mem_off(dE, S * n * 64);
    const int64_t nblk = (S + G - 1) / G;
    for (int64_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const EnvBlock eb = env_block(blk, G, n, S);
        __syncthreads();
        load_rows64(Es, E, eb.s0 * n, eb.rows, tid);
        load_rows64(Qs, Q, eb.s0 * n, eb.rows, tid);
        __syncthreads();
        const bool active = tid < eb.rows;
        const int e = active ? tid / n : 0, i = active ? tid - e * n : 0;
        const int64_t row = (eb.s0 + e) * n + i;
        if (active) {
            float ds[kSmallN], m[kSmallN];
            float dot = 0.0f;
#pragma unroll
            for (int k = 0; k < kSmallN; ++k) {
                m[k] = k < n ? M[row * n + k] : 0.0f;
                ds[k] = 0.0f;
                for (int ll = 0; ll < L; ++ll) if (k < n) ds[k] += dM[ll * dm_stride + row * n + k];
                dot = fmaf(m[k], ds[k], dot);
            }
#pragma unroll
            for (int k = 0; k < kSmallN; ++k) { ds[k] = m[k] * (ds[k] - dot); Ds[tid * kSmallN + k] = ds[k]; }
            float out[64];
            row_combine(out, ds, Es + e * n * kNP, n);
            row_store64(dQ + row * 64, out);
        }
        __syncthreads();
        if (active) {
            float ct[kSmallN], out[64];
#pragma unroll
            for (int q = 0; q < kSmallN; ++q) ct[q] = q < n ? Ds[(e * n + q) * kSmallN + i] : 0.0f;
            row_combine(out, ct, Qs + e * n * kNP, n);
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                float4 *p = reinterpret_cast<float4 *>(dE + row * 64 + 4 * q);
                const float4 o = *p;
                *p = make_float4(o.x + out[4 * q], o.y + out[4 * q + 1], o.z + out[4 * q + 2], o.w + out[4 * q + 3]);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// heads + losses
// ------------------------------------------------------------------------------------------------------------------
struct PolicyHeadArgs {
    const float *g3;             // [R][32] last hidden layer (CENT: [S][32])
    const float *w4, *b4;        // [32][5], [5]  (CENT: [32][5n], [5n])
    const uint8_t *avail_bits;   // [R] or NULL
    const int64_t *actions;      // [R] or NULL (forward only: no log-likelihood)
    const float *adv, *old_ll;   // [S]
    const uint8_t *valid;        // [S] or NULL
    float inv_count, ent_coeff, clip_lo, clip_hi;
    float *ll, *ent, *probs;
    double *loss;                // the call's loss, summed in float64 (cm_ppo_net adds it to io.loss at the end)
    float *dg3, *dw4, *db4;      // NULL: forward only; dg3 receives dZ of the last hidden layer: d g3 act'(g3)
    float *dlogits;              // CENT: [S][5n] d logits for the dW4 product
    int relu;                    // CENT: act = relu instead of tanh
    int n, G;
    int64_t S;                   // steps of one member
    const float *inv_counts;     // set: [members] 1 / count, replaces inv_count (NULL: inv_count)
    int64_t wstr, gstr;          // set: weight / gradient blob strides
};

// member blockIdx.y of a set: its rows, weights, gradient targets, loss slot and 1 / count
__device__ __forceinline__ PolicyHeadArgs policy_member(const PolicyHeadArgs &a0)
{
    PolicyHeadArgs a = a0;
    const int64_t S = a.S, R = S * a.n;
    a.g3 = mem_off(a.g3, R * 32); a.w4 = mem_off(a.w4, a.wstr); a.b4 = mem_off(a.b4, a.wstr);
    a.avail_bits = mem_off(a.avail_bits, R); a.actions = mem_off(a.actions, R);
    a.adv = mem_off(a.adv, S); a.old_ll = mem_off(a.old_ll, S); a.valid = mem_off(a.valid, S);
    a.ll = mem_off(a.ll, S); a.ent = mem_off(a.ent, S); a.probs = mem_off(a.probs, R * CM_ACTIONS);
    a.loss = mem_off(a.loss, 1); a.dg3 = mem_off(a.dg3, R * 32); a.dw4 = mem_off(a.dw4, a.gstr); a.db4 = mem_off(a.db4, a.gstr);
    if (a.inv_counts) a.inv_count = a.inv_counts[blockIdx.y];
    return a;
}

static constexpr float kProbEps = 1.1920928955078125e-07f;   // torch.finfo(float32).eps: probs_to_logits clamps to [eps, 1 - eps]

// One agent's categorical tail from its five logits z: softmax p, availability mask, renormalisation q = masked / masked.sum()
// (no + 1e-12), the clamped logs lc that Categorical(probs=q) uses, entropy and log-likelihood of `act`
__device__ __forceinline__ void head_tail_fwd(const float (&z)[CM_ACTIONS], uint32_t av, int act, float (&p)[CM_ACTIONS],
                                              float (&q)[CM_ACTIONS], float (&lc)[CM_ACTIONS], float &msum, float &ent, float &lp)
{
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < CM_ACTIONS; ++j) mx = fmaxf(mx, z[j]);
    float sum = 0.0f;
#pragma unroll
    for (int j = 0; j < CM_ACTIONS; ++j) { p[j] = expf(z[j] - mx); sum += p[j]; }
    msum = 0.0f;
#pragma unroll
    for (int j = 0; j < CM_ACTIONS; ++j) { p[j] = p[j] / sum; q[j] = ((av >> j) & 1u) ? p[j] : 0.0f; msum += q[j]; }
    ent = 0.0f;
#pragma unroll
    for (int j = 0; j < CM_ACTIONS; ++j) {
        q[j] = q[j] / msum;
        lc[j] = logf(fminf(fmaxf(q[j], kProbEps), 1.0f - kProbEps));
        ent -= q[j] * lc[j];
    }
    lp = 0.0f;
#pragma unroll
    for (int j = 0; j < CM_ACTIONS; ++j) if (j == act) lp = lc[j];
}

// d loss / d z of one agent, given gl = d loss / d ll and ge = d loss / d (its entropy term): through the clamp of probs_to_logits
// (the gradient passes inside [eps, 1 - eps]), the renormalisation and the softmax
__device__ __forceinline__ void head_tail_bwd(float gl, float ge, int act, uint32_t av, const float (&p)[CM_ACTIONS],
                                              const float (&q)[CM_ACTIONS], const float (&lc)[CM_ACTIONS], float msum,
                                              float (&gz)[CM_ACTIONS])
{
    float gq[CM_ACTIONS];
    float proj = 0.0f;
#pragma unroll
    for (int j = 0; j < CM_ACTIONS; ++j) {
        const float in = (q[j] >= kProbEps && q[j] <= 1.0f - kProbEps) ? 1.0f : 0.0f;
        gq[j] = ge * (-lc[j] - in);
        if (j == act) gq[j] += gl * (in > 0.0f ? 1.0f / q[j] : 0.0f);
        proj = fmaf(gq[j], q[j], proj);
    }
    float dot = 0.0f;
    float gp[CM_ACTIONS];
#pragma unroll
    for (int j = 0; j < CM_ACTIONS; ++j) {
        gp[j] = ((av >> j) & 1u) ? (gq[j] - proj) / msum : 0.0f;
        dot = fmaf(gp[j], p[j], dot);
    }
#pragma unroll
    for (int j = 0; j < CM_ACTIONS; ++j) gz[j] = p[j] * (gp[j] - dot);
}

// The loss terms of a CTA reach the call's sum in ONE float64 atomic add.  Added step by step into one fp32 value, 10^5 terms
// of one sign lose ~1e-3 of the sum (each rounds against the growing total with the same bias), and even one fp32 add per CTA
// loses ~1e-5: the running total must be float64 and see one term per CTA.
// Called once by every thread after its last block; *red1 was zeroed before the kernel's first barrier.
__device__ __forceinline__ void cta_loss_add(double *loss, float lsum, float *red1)
{
    const float v = warp_sumf(lsum);
    if ((threadIdx.x & 31) == 0) atomicAdd(red1, v);
    __syncthreads();
    if (threadIdx.x == 0) atomicAdd(loss, (double)*red1);
}

__global__ void net_loss_store_kernel(float *loss, const double *sum, int count)
{
    for (int i = threadIdx.x; i < count; i += blockDim.x) loss[i] += (float)sum[i];
}

// One env step s with joint log-likelihood ll and mean entropy en: outputs, the clipped surrogate added to the loss and the
// gradients gl = d loss / d ll, ge = d loss / d (one agent's entropy)
__device__ __forceinline__ void head_step_objective(const PolicyHeadArgs &a, int64_t s, float ll, float en, int n, float &gl, float &ge,
                                                    float &lsum)
{
    if (a.ll) a.ll[s] = ll;
    if (a.ent) a.ent[s] = en;
    gl = 0.0f;
    ge = 0.0f;
    const bool valid = a.valid ? a.valid[s] != 0 : true;
    if (a.adv && valid) {
        const float old = a.old_ll ? a.old_ll[s] : ll;
        const float ratio = expf(ll - old), adv = a.adv[s];
        const float rc = fminf(fmaxf(ratio, a.clip_lo), a.clip_hi);
        const float s1 = ratio * adv, s2 = rc * adv;
        const float in = (ratio >= a.clip_lo && ratio <= a.clip_hi) ? 1.0f : 0.0f;
        // torch.min's gradient goes to the smaller argument, half to each on a tie; clamp passes it inside [lo, hi]
        const float gr = s1 < s2 ? adv : (s1 > s2 ? adv * in : 0.5f * adv + 0.5f * adv * in);
        lsum += -(fminf(s1, s2) + a.ent_coeff * en) * a.inv_count;
        gl = -a.inv_count * gr * ratio;
        ge = -a.inv_count * a.ent_coeff / (float)n;
    }
}

__global__ void __launch_bounds__(kNetThreads) net_policy_head_kernel(const PolicyHeadArgs a0)
{
    const PolicyHeadArgs a = policy_member(a0);
    __shared__ float w4s[32 * CM_ACTIONS + CM_ACTIONS];
    __shared__ float ll_row[kRows], ent_row[kRows], gll_env[kRows], gent_env[kRows];
    __shared__ float red[32 * CM_ACTIONS + CM_ACTIONS], lred;
    const int tid = threadIdx.x, lane = tid & 31;
    const int n = a.n;
    float lsum = 0.0f;
    if (tid == 0) lred = 0.0f;
    for (int i = tid; i < 32 * CM_ACTIONS + CM_ACTIONS; i += kNetThreads) {
        w4s[i] = i < 32 * CM_ACTIONS ? a.w4[i] : a.b4[i - 32 * CM_ACTIONS];
        red[i] = 0.0f;
    }
    const int64_t nblk = (a.S + a.G - 1) / a.G;
    for (int64_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const EnvBlock eb = env_block(blk, a.G, n, a.S);
        __syncthreads();
        const bool active = tid < eb.rows;
        const int64_t row = eb.s0 * n + (active ? tid : 0);
        float g[32], p[CM_ACTIONS], q[CM_ACTIONS], lc[CM_ACTIONS];
        float msum = 1.0f;
        uint32_t av = 0x1Fu;
        int act = 0;
        {
            const float4 *src = reinterpret_cast<const float4 *>(a.g3 + row * 32);
#pragma unroll
            for (int k = 0; k < 8; ++k) { const float4 v = src[k]; g[4 * k] = v.x; g[4 * k + 1] = v.y; g[4 * k + 2] = v.z; g[4 * k + 3] = v.w; }
            float z[CM_ACTIONS];
#pragma unroll
            for (int j = 0; j < CM_ACTIONS; ++j) z[j] = 0.0f;
#pragma unroll
            for (int k = 0; k < 32; ++k)
#pragma unroll
                for (int j = 0; j < CM_ACTIONS; ++j) z[j] = fmaf(g[k], w4s[k * CM_ACTIONS + j], z[j]);
#pragma unroll
            for (int j = 0; j < CM_ACTIONS; ++j) z[j] += w4s[32 * CM_ACTIONS + j];
            if (a.avail_bits) av = a.avail_bits[row];
            if (a.actions) act = (int)a.actions[row];
            float ent, lp;
            head_tail_fwd(z, av, act, p, q, lc, msum, ent, lp);
            if (active) {
                ll_row[tid] = lp;
                ent_row[tid] = ent;
                if (a.probs)
#pragma unroll
                    for (int j = 0; j < CM_ACTIONS; ++j) a.probs[row * CM_ACTIONS + j] = q[j];
            }
        }
        __syncthreads();
        if (tid < eb.ne) {                                        // one thread per env: sums in agent order
            float ll = 0.0f, en = 0.0f;
            for (int i = 0; i < n; ++i) { ll += ll_row[tid * n + i]; en += ent_row[tid * n + i]; }
            en = en / (float)n;
            float gl, ge;
            head_step_objective(a, eb.s0 + tid, ll, en, n, gl, ge, lsum);
            gll_env[tid] = gl;
            gent_env[tid] = ge;
        }
        if (!a.dg3) continue;
        __syncthreads();
        float gz[CM_ACTIONS];
        {
            const int e = active ? tid / n : 0;
            const float gl = active ? gll_env[e] : 0.0f, ge = active ? gent_env[e] : 0.0f;
            float t[CM_ACTIONS];
            head_tail_bwd(gl, ge, act, av, p, q, lc, msum, t);
#pragma unroll
            for (int j = 0; j < CM_ACTIONS; ++j) gz[j] = active ? t[j] : 0.0f;
        }
        if (active) {
            float4 *dst = reinterpret_cast<float4 *>(a.dg3 + row * 32);
#pragma unroll
            for (int k4 = 0; k4 < 8; ++k4) {
                float o[4];
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    float v = 0.0f;
#pragma unroll
                    for (int j = 0; j < CM_ACTIONS; ++j) v = fmaf(gz[j], w4s[(4 * k4 + c) * CM_ACTIONS + j], v);
                    o[c] = v * (1.0f - g[4 * k4 + c] * g[4 * k4 + c]);           // dZ of the last hidden layer (tanh)
                }
                dst[k4] = make_float4(o[0], o[1], o[2], o[3]);
            }
        }
#pragma unroll
        for (int k = 0; k < 32; ++k)
#pragma unroll
            for (int j = 0; j < CM_ACTIONS; ++j) {
                const float v = warp_sumf(active ? g[k] * gz[j] : 0.0f);
                if (lane == 0) atomicAdd(&red[k * CM_ACTIONS + j], v);
            }
#pragma unroll
        for (int j = 0; j < CM_ACTIONS; ++j) {
            const float v = warp_sumf(gz[j]);
            if (lane == 0) atomicAdd(&red[32 * CM_ACTIONS + j], v);
        }
    }
    if (a.dg3) {
        __syncthreads();
        for (int i = tid; i < 32 * CM_ACTIONS + CM_ACTIONS; i += kNetThreads)
            atomicAdd(i < 32 * CM_ACTIONS ? a.dw4 + i : a.db4 + (i - 32 * CM_ACTIONS), red[i]);
    }
    if (a.loss) cta_loss_add(a.loss, lsum, &lred);
}

// CENT head: the rows are env steps, logits [S][5n] = g3 W4 + b4 with W4 [32][5n].  Thread = (step, agent), the G = 256 / n steps
// of a block with all their agents, like net_policy_head_kernel: a thread computes the five logits of its agent (the agent's W4
// columns, shared by the block's steps, come through L1), the per-agent tail and, per step, the objective.  Backward: d logits go
// to `dlogits` (dW4 is a product of its own), db4 is accumulated per thread over its blocks, and dg3 = dlogits W4^T is reduced
// over the agents of a step in agent order through shared memory, times act'(g3).
__global__ void __launch_bounds__(kNetThreads) net_cent_head_kernel(const PolicyHeadArgs a)
{
    __shared__ float ll_row[kRows], ent_row[kRows], gll_env[kRows], gent_env[kRows];
    __shared__ float dgs[kRows * 33], lred;
    const int tid = threadIdx.x;
    float lsum = 0.0f;
    if (tid == 0) lred = 0.0f;
    const int n = a.n, NO = n * CM_ACTIONS;
    const int ia = tid % n;                                       // this thread's agent (the same in every block)
    const float *__restrict__ w4 = a.w4 + ia * CM_ACTIONS;
    float dbacc[CM_ACTIONS];
#pragma unroll
    for (int j = 0; j < CM_ACTIONS; ++j) dbacc[j] = 0.0f;
    const int64_t nblk = (a.S + a.G - 1) / a.G;
    for (int64_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const EnvBlock eb = env_block(blk, a.G, n, a.S);
        __syncthreads();
        const bool active = tid < eb.rows;
        const int64_t s = eb.s0 + (active ? tid / n : 0), row = s * n + ia;
        float p[CM_ACTIONS], q[CM_ACTIONS], lc[CM_ACTIONS];
        float msum = 1.0f;
        uint32_t av = 0x1Fu;
        int act = 0;
        {
            const float4 *src = reinterpret_cast<const float4 *>(a.g3 + s * 32);
            float z[CM_ACTIONS];
#pragma unroll
            for (int j = 0; j < CM_ACTIONS; ++j) z[j] = 0.0f;
#pragma unroll
            for (int k4 = 0; k4 < 8; ++k4) {
                const float4 v = src[k4];
                const float g[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int c = 0; c < 4; ++c)
#pragma unroll
                    for (int j = 0; j < CM_ACTIONS; ++j) z[j] = fmaf(g[c], __ldg(w4 + (size_t)(4 * k4 + c) * NO + j), z[j]);
            }
#pragma unroll
            for (int j = 0; j < CM_ACTIONS; ++j) z[j] += __ldg(a.b4 + ia * CM_ACTIONS + j);
            if (a.avail_bits) av = a.avail_bits[row];
            if (a.actions) act = (int)a.actions[row];
            float ent, lp;
            head_tail_fwd(z, av, act, p, q, lc, msum, ent, lp);
            if (active) {
                ll_row[tid] = lp;
                ent_row[tid] = ent;
                if (a.probs)
#pragma unroll
                    for (int j = 0; j < CM_ACTIONS; ++j) a.probs[row * CM_ACTIONS + j] = q[j];
            }
        }
        __syncthreads();
        if (tid < eb.ne) {                                        // one thread per step: sums in agent order
            float ll = 0.0f, en = 0.0f;
            for (int i = 0; i < n; ++i) { ll += ll_row[tid * n + i]; en += ent_row[tid * n + i]; }
            en = en / (float)n;
            float gl, ge;
            head_step_objective(a, eb.s0 + tid, ll, en, n, gl, ge, lsum);
            gll_env[tid] = gl;
            gent_env[tid] = ge;
        }
        if (!a.dg3) continue;
        __syncthreads();
        if (active) {
            float gz[CM_ACTIONS];
            head_tail_bwd(gll_env[tid / n], gent_env[tid / n], act, av, p, q, lc, msum, gz);
#pragma unroll
            for (int j = 0; j < CM_ACTIONS; ++j) { a.dlogits[s * NO + ia * CM_ACTIONS + j] = gz[j]; dbacc[j] += gz[j]; }
#pragma unroll 4
            for (int k = 0; k < 32; ++k) {
                float v = 0.0f;
#pragma unroll
                for (int j = 0; j < CM_ACTIONS; ++j) v = fmaf(gz[j], __ldg(w4 + (size_t)k * NO + j), v);
                dgs[tid * 33 + k] = v;
            }
        }
        __syncthreads();
        for (int e = tid; e < eb.ne * 32; e += kNetThreads) {       // (step, k): the step's agents in order
            const int st = e >> 5, k = e & 31;
            float v = 0.0f;
            for (int i = 0; i < n; ++i) v += dgs[(st * n + i) * 33 + k];
            const int64_t o = (eb.s0 + st) * 32 + k;
            const float g = a.g3[o];
            a.dg3[o] = a.relu ? (g > 0.0f ? v : 0.0f) : v * (1.0f - g * g);
        }
    }
    if (a.dg3 && tid < a.G * n)
#pragma unroll
        for (int j = 0; j < CM_ACTIONS; ++j) atomicAdd(a.db4 + ia * CM_ACTIONS + j, dbacc[j]);
    if (a.loss) cta_loss_add(a.loss, lsum, &lred);
}

struct CriticHeadArgs {
    const float *c1;             // [R][64] decoder hidden layer
    const float *w2, *b2, *log_std;   // [64], [1], [1]
    const float *returns;        // [S] or NULL (forward only)
    float inv_count;
    float *values;
    double *loss;                // (as PolicyHeadArgs::loss)
    float *dc1, *dw2, *db2, *dlog_std;
    int unclamped;               // 1: std = exp(log_std) without CommBaseCritic's clamp at log 1e-6 (GaussianMLPBaseline)
    int n, G;
    int64_t S;                   // steps of one member
    const uint8_t *valid;        // [S] or NULL: 0 = padded step, its value is written but adds nothing to the loss or gradient
    const float *inv_counts;     // (as PolicyHeadArgs)
    int64_t wstr, gstr;
};

__device__ __forceinline__ CriticHeadArgs critic_member(const CriticHeadArgs &a0)
{
    CriticHeadArgs a = a0;
    const int64_t S = a.S, R = S * a.n;
    a.c1 = mem_off(a.c1, R * 64); a.w2 = mem_off(a.w2, a.wstr); a.b2 = mem_off(a.b2, a.wstr); a.log_std = mem_off(a.log_std, a.wstr);
    a.returns = mem_off(a.returns, S); a.values = mem_off(a.values, S); a.valid = mem_off(a.valid, S); a.loss = mem_off(a.loss, 1);
    a.dc1 = mem_off(a.dc1, R * 64); a.dw2 = mem_off(a.dw2, a.gstr); a.db2 = mem_off(a.db2, a.gstr); a.dlog_std = mem_off(a.dlog_std, a.gstr);
    if (a.inv_counts) a.inv_count = a.inv_counts[blockIdx.y];
    return a;
}

__global__ void __launch_bounds__(kNetThreads) net_critic_head_kernel(const CriticHeadArgs a0)
{
    const CriticHeadArgs a = critic_member(a0);
    __shared__ float w2s[64], v_row[kRows], gv_env[kRows], red[66], lred;
    const int tid = threadIdx.x, lane = tid & 31;
    const int n = a.n;
    float lsum = 0.0f;
    if (tid == 0) lred = 0.0f;
    if (tid < 64) w2s[tid] = a.w2[tid];
    if (tid < 66) red[tid] = 0.0f;
    const float b2 = a.b2[0];
    const float lmin = a.unclamped ? -INFINITY : logf(1e-6f);
    const float ls = a.log_std[0];
    const float lsc = fmaxf(ls, lmin), sd = expf(lsc);
    const int64_t nblk = (a.S + a.G - 1) / a.G;
    for (int64_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const EnvBlock eb = env_block(blk, a.G, n, a.S);
        __syncthreads();
        const bool active = tid < eb.rows;
        const int64_t row = eb.s0 * n + (active ? tid : 0);
        float c[64];
        {
            const float4 *src = reinterpret_cast<const float4 *>(a.c1 + row * 64);
            float v = 0.0f;
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                const float4 x = src[k];
                c[4 * k] = x.x; c[4 * k + 1] = x.y; c[4 * k + 2] = x.z; c[4 * k + 3] = x.w;
                v = fmaf(x.x, w2s[4 * k], fmaf(x.y, w2s[4 * k + 1], fmaf(x.z, w2s[4 * k + 2], fmaf(x.w, w2s[4 * k + 3], v))));
            }
            if (active) v_row[tid] = v + b2;
        }
        __syncthreads();
        if (tid < eb.ne) {
            float V = 0.0f;
            for (int i = 0; i < n; ++i) V += v_row[tid * n + i];
            const int64_t s = eb.s0 + tid;
            if (a.values) a.values[s] = V;
            float gv = 0.0f;
            if (a.returns && (!a.valid || a.valid[s])) {
                const float d = (a.returns[s] - V) / sd;
                lsum += (0.5f * d * d + logf(sd) + 0.91893853320467274178f) * a.inv_count;
                gv = -d / sd * a.inv_count;
                if (a.dlog_std && ls >= lmin) atomicAdd(&red[65], (1.0f - d * d) * a.inv_count);
            }
            gv_env[tid] = gv;
        }
        if (!a.dc1) continue;
        __syncthreads();
        const float gv = active ? gv_env[tid / n] : 0.0f;
        if (active) {
            float4 *dst = reinterpret_cast<float4 *>(a.dc1 + row * 64);
#pragma unroll
            for (int k = 0; k < 16; ++k)                  // dZ of the decoder's hidden layer (tanh)
                dst[k] = make_float4(gv * w2s[4 * k] * (1.0f - c[4 * k] * c[4 * k]), gv * w2s[4 * k + 1] * (1.0f - c[4 * k + 1] * c[4 * k + 1]),
                                     gv * w2s[4 * k + 2] * (1.0f - c[4 * k + 2] * c[4 * k + 2]),
                                     gv * w2s[4 * k + 3] * (1.0f - c[4 * k + 3] * c[4 * k + 3]));
        }
#pragma unroll
        for (int k = 0; k < 64; ++k) {
            const float v = warp_sumf(c[k] * gv);
            if (lane == 0) atomicAdd(&red[k], v);
        }
        const float v = warp_sumf(gv);
        if (lane == 0) atomicAdd(&red[64], v);
    }
    if (a.dc1) {
        __syncthreads();
        if (tid < 64) atomicAdd(a.dw2 + tid, red[tid]);
        if (tid == 64) atomicAdd(a.db2, red[64]);
        if (tid == 65 && a.dlog_std) atomicAdd(a.dlog_std, red[65]);
    }
    if (a.loss) cta_loss_add(a.loss, lsum, &lred);
}

// ------------------------------------------------------------------------------------------------------------------
// wide-K layers of the CENT family: rows are env steps, K = n*D grows with the team (87 .. 32 768)
// ------------------------------------------------------------------------------------------------------------------
static constexpr int kWRows = 64, kWK = 32, kWPA = kWK + 4;          // forward: rows per CTA, K chunk, pitch of the chunk

// Y [R][64J] = act(X [R][K] W [K][64J] + b), act: 1 tanh, 2 relu.  The fp32 first layer of policy_cent_kernel: 64 rows per CTA, K
// streamed through shared memory in chunks of 32 with the next chunk's global loads in flight (registers) while the current one
// is multiplied (cent_mac).  The rows are read with 4-byte loads, one lane per k: rows K * 4 bytes apart need no alignment.
template <int J, int ACT>
__global__ void __launch_bounds__(256) net_wide_fwd_kernel(const float *__restrict__ X, const float *__restrict__ W,
                                                           const float *__restrict__ bias, float *__restrict__ Y, int64_t R, int K)
{
    constexpr int N = 64 * J, BL = 2 * J;                            // BL: float4 of a weight chunk per thread
    __shared__ __align__(16) float Ach[kWRows * kWPA];
    __shared__ __align__(16) float Bch[kWK * N];
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15, lane = tid & 31, warp = tid >> 5;
    const int64_t row0 = (int64_t)blockIdx.x * kWRows;
    const int rows = (int)min((int64_t)kWRows, R - row0);
    const float *__restrict__ Xb = X + row0 * K;
    float acc[4][4 * J];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int c = 0; c < 4 * J; ++c) acc[i][c] = 0.0f;
    float ra[8];
    float4 rb[BL];
    auto fetch = [&](int k0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {                                // lane = k, warp + 8j = row
            const int r = warp + 8 * j;
            ra[j] = (r < rows && k0 + lane < K) ? __ldg(Xb + (size_t)r * K + k0 + lane) : 0.0f;
        }
#pragma unroll
        for (int j = 0; j < BL; ++j) {
            const int e = tid + 256 * j, kk = e / (16 * J), c4 = e - kk * (16 * J);
            rb[j] = (k0 + kk < K) ? __ldg(reinterpret_cast<const float4 *>(W + (size_t)(k0 + kk) * N + c4 * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    fetch(0);
    for (int k0 = 0; k0 < K; k0 += kWK) {
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 8; ++j) Ach[(warp + 8 * j) * kWPA + lane] = ra[j];
#pragma unroll
        for (int j = 0; j < BL; ++j) {
            const int e = tid + 256 * j, kk = e / (16 * J), c4 = e - kk * (16 * J);
            *reinterpret_cast<float4 *>(Bch + kk * N + c4 * 4) = rb[j];
        }
        __syncthreads();
        if (k0 + kWK < K) fetch(k0 + kWK);
        cent_mac<J>(Ach, kWPA, Bch, kWK, ty, tx, acc);
    }
#pragma unroll
    for (int j = 0; j < J; ++j) {
        const float4 bv = __ldg(reinterpret_cast<const float4 *>(bias + j * 64 + tx * 4));
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int r = ty * 4 + i;
            if (r >= rows) continue;
            float4 v = make_float4(acc[i][4 * j + 0] + bv.x, acc[i][4 * j + 1] + bv.y, acc[i][4 * j + 2] + bv.z, acc[i][4 * j + 3] + bv.w);
            if (ACT == 1) { v.x = tanhf(v.x); v.y = tanhf(v.y); v.z = tanhf(v.z); v.w = tanhf(v.w); }
            if (ACT == 2) { v.x = fmaxf(v.x, 0.0f); v.y = fmaxf(v.y, 0.0f); v.z = fmaxf(v.z, 0.0f); v.w = fmaxf(v.w, 0.0f); }
            *reinterpret_cast<float4 *>(Y + (row0 + r) * N + j * 64 + tx * 4) = v;
        }
    }
}

static constexpr int kWPanel = 64, kWTile = 32;                      // weight gradient: K panel per CTA, rows per staged tile

// dW += X^T dZ over the rows [blockIdx.y * rows_per_cta, ...) and K panel blockIdx.x (64 k x all N columns); db += sum dZ (the CTAs
// of panel 0).  X [R][K] (pitch ldx, rows unaligned: 4-byte loads), dZ [R][N].  X and dZ tiles of 32 rows are staged through shared
// memory with the next tile's loads in flight (registers); thread (ty, tx) owns k = ty + TY i and the columns 4 tx .. 4 tx + 3, sums
// in registers over all of the CTA's rows, and adds to global memory once.  TRANS: the result is stored transposed, dW[n][k]
// (dW4 [32][5n] of the CENT head is (d logits)^T g3 with X = d logits, dZ = g3).
template <int N, int TRANS>
__global__ void __launch_bounds__(256) net_wide_dw_kernel(const float *__restrict__ X, int ldx, const float *__restrict__ dZ,
                                                          float *__restrict__ dW, float *__restrict__ db, int64_t R, int K,
                                                          int64_t rows_per_cta)
{
    constexpr int TX = N / 4, TY = 256 / TX, KI = kWPanel / TY, ZL = kWTile * N / 4 / 256;
    __shared__ __align__(16) float Xs[kWTile * kWPanel];
    __shared__ __align__(16) float Zs[kWTile * N];
    const int tid = threadIdx.x, tx = tid % TX, ty = tid / TX, lane = tid & 31, warp = tid >> 5;
    const int k0 = blockIdx.x * kWPanel;
    const int64_t rb = (int64_t)blockIdx.y * rows_per_cta, re = min(R, rb + rows_per_cta);
    const bool do_db = db && blockIdx.x == 0 && tid < N;
    float acc[KI][4];
#pragma unroll
    for (int i = 0; i < KI; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.0f;
    float bacc = 0.0f;
    float xr[8];
    float4 zr[ZL];
    auto fetch = [&](int64_t r0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {                                // rows warp + 8 (j / 2), k = lane + 32 (j % 2)
            const int64_t r = r0 + warp + 8 * (j >> 1);
            const int k = k0 + lane + 32 * (j & 1);
            xr[j] = (r < re && k < K) ? __ldg(X + r * ldx + k) : 0.0f;
        }
#pragma unroll
        for (int j = 0; j < ZL; ++j) {
            const int e = tid + 256 * j, r = e / (N / 4), c4 = e - r * (N / 4);
            zr[j] = r0 + r < re ? __ldg(reinterpret_cast<const float4 *>(dZ + (r0 + r) * N + 4 * c4)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    if (rb < re) fetch(rb);
    for (int64_t r0 = rb; r0 < re; r0 += kWTile) {
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 8; ++j) Xs[(warp + 8 * (j >> 1)) * kWPanel + lane + 32 * (j & 1)] = xr[j];
#pragma unroll
        for (int j = 0; j < ZL; ++j) reinterpret_cast<float4 *>(Zs)[tid + 256 * j] = zr[j];
        __syncthreads();
        if (r0 + kWTile < re) fetch(r0 + kWTile);
#pragma unroll 4
        for (int r = 0; r < kWTile; ++r) {                           // (rows past the end are zeros)
            const float4 z = *reinterpret_cast<const float4 *>(Zs + r * N + 4 * tx);
#pragma unroll
            for (int i = 0; i < KI; ++i) {
                const float x = Xs[r * kWPanel + ty + TY * i];
                acc[i][0] = fmaf(x, z.x, acc[i][0]);
                acc[i][1] = fmaf(x, z.y, acc[i][1]);
                acc[i][2] = fmaf(x, z.z, acc[i][2]);
                acc[i][3] = fmaf(x, z.w, acc[i][3]);
            }
        }
        if (do_db) {
            float sacc = 0.0f;
            for (int r = 0; r < kWTile; ++r) sacc += Zs[r * N + tid];
            bacc += sacc;
        }
    }
#pragma unroll
    for (int i = 0; i < KI; ++i) {
        const int k = k0 + ty + TY * i;
        if (k < K)
#pragma unroll
            for (int c = 0; c < 4; ++c) atomicAdd(TRANS ? dW + (size_t)(4 * tx + c) * K + k : dW + (size_t)k * N + 4 * tx + c, acc[i][c]);
    }
    if (do_db) atomicAdd(db + tid, bacc);
}

// ------------------------------------------------------------------------------------------------------------------
// host side: launch helpers and the two entry points
// ------------------------------------------------------------------------------------------------------------------
struct CriticBlob { int enc_w1, enc_b1, enc_w2, enc_b2, att_w, gcn_w, gcn_b, dec_w1, dec_b1, dec_w2, dec_b2, log_std, total; };
static CriticBlob critic_blob_layout(int D, int L)
{
    CriticBlob o;
    int p = 0;
    o.enc_w1 = p; p += D * kH1;
    o.enc_b1 = p; p += kH1;
    o.enc_w2 = p; p += kH1 * kE;
    o.enc_b2 = p; p += kE;
    o.att_w = p; p += kE * kE;
    o.gcn_w = p; p += L * kE * kE;
    o.gcn_b = p; p += L * kE;
    o.dec_w1 = p; p += kE * 64;
    o.dec_b1 = p; p += 64;
    o.dec_w2 = p; p += 64;
    o.dec_b2 = p; p += 1;
    o.log_std = p; p += 1;
    o.total = p;
    return o;
}

// GaussianMLPBaseline(hidden_sizes <= (64, 64, 64)): w1 [K][64] b1 w2 [64][64] b2 w3 [64][64] b3 w4 [64] b4 [1] log_std [1]
struct BaselineBlob { int w1, b1, w2, b2, w3, b3, w4, b4, log_std, total; };
static BaselineBlob baseline_blob_layout(int K)
{
    BaselineBlob o;
    int p = 0;
    o.w1 = p; p += K * 64;
    o.b1 = p; p += 64;
    o.w2 = p; p += 64 * 64;
    o.b2 = p; p += 64;
    o.w3 = p; p += 64 * 64;
    o.b3 = p; p += 64;
    o.w4 = p; p += 64;
    o.b4 = p; p += 1;
    o.log_std = p; p += 1;
    o.total = p;
    return o;
}

static bool cent_kind(int kind) { return kind == CM_NET_POLICY_CENT || kind == CM_NET_BASELINE_MLP; }

static int g_sms = 0;
static int sm_count()
{
    if (!g_sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&g_sms, cudaDevAttrMultiProcessorCount, dev);
        if (g_sms <= 0) g_sms = 148;
    }
    return g_sms;
}

template <typename Kern>
static cudaError_t set_smem(Kern k, size_t bytes)
{
    return bytes > 48 * 1024 ? cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) : cudaSuccess;
}

#define NET_TRY(expr) do { const cudaError_t e__ = (expr); if (e__ != cudaSuccess) return e__; } while (0)

static const size_t kSmemMax = 227 * 1024;

// The members of a set one launch runs (gridDim.y = g) and their blob strides in floats; Grp() = one network
struct Grp {
    int g = 1;
    int64_t wstr = 0, gstr = 0;
};
// CTAs along x when g members of `units` work units each share about `cap` CTAs (the SMs times the occupancy)
static int grid_x(int64_t units, int64_t cap, int g)
{
    const int64_t c = (cap + g - 1) / g;
    return (int)(units < c ? units : c);
}

template <int N, int ACT, int ASYNC>
static cudaError_t dense_fwd_a(const float *X, int ldx, const float *W, const float *b, float *Y, int64_t R, int K, cudaStream_t st,
                               const Grp &q)
{
    const int K4 = (K + 3) & ~3;
    const size_t smem = ((size_t)K4 * N + (ASYNC ? 2 : 1) * 128 * (size_t)(K4 + 4)) * sizeof(float) + 16;
    NET_TRY(set_smem(net_dense_fwd_kernel<N, ACT, ASYNC>, smem));
    int per_sm = 1;
    NET_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, net_dense_fwd_kernel<N, ACT, ASYNC>, 256, smem));
    if (per_sm < 1) per_sm = 1;
    const dim3 grid(grid_x((R + 127) / 128, (int64_t)sm_count() * per_sm, q.g), q.g);
    net_dense_fwd_kernel<N, ACT, ASYNC><<<grid, 256, smem, st>>>(X, ldx, W, b, Y, N, R, K, q.wstr);
    return cudaGetLastError();
}
static bool rows_aligned(const float *X, int ldx, int K) { return (ldx & 3) == 0 && (K & 3) == 0 && (reinterpret_cast<uintptr_t>(X) & 15) == 0; }

template <int N, int ACT>
static cudaError_t dense_fwd_t(const float *X, int ldx, const float *W, const float *b, float *Y, int64_t R, int K, cudaStream_t st,
                               const Grp &q)
{
    return rows_aligned(X, ldx, K) ? dense_fwd_a<N, ACT, 1>(X, ldx, W, b, Y, R, K, st, q) : dense_fwd_a<N, ACT, 0>(X, ldx, W, b, Y, R, K, st, q);
}

// R = rows of one member (q.g members side by side, X / Y rows member-major)
static cudaError_t dense_fwd(const float *X, int ldx, const float *W, const float *b, float *Y, int64_t R, int K, int N, int act,
                             cudaStream_t st, const Grp &q = Grp())
{
    if (act == 2)                            // relu: the CENT policy's 128 -> 64 and 64 -> 32 layers
        return N == 64 ? dense_fwd_t<64, 2>(X, ldx, W, b, Y, R, K, st, q) : dense_fwd_t<32, 2>(X, ldx, W, b, Y, R, K, st, q);
    if (N == 128) return act ? dense_fwd_t<128, 1>(X, ldx, W, b, Y, R, K, st, q) : dense_fwd_t<128, 0>(X, ldx, W, b, Y, R, K, st, q);
    if (N == 64) return act ? dense_fwd_t<64, 1>(X, ldx, W, b, Y, R, K, st, q) : dense_fwd_t<64, 0>(X, ldx, W, b, Y, R, K, st, q);
    return act ? dense_fwd_t<32, 1>(X, ldx, W, b, Y, R, K, st, q) : dense_fwd_t<32, 0>(X, ldx, W, b, Y, R, K, st, q);
}

template <int N, int KMAX, int ROWS, int ASYNC, int XRELU>
static cudaError_t dense_bwd_a(const float *dZ, const float *X, int ldx, const float *W, float *dX, int accumulate, int xact, float *dW,
                               float *db, int64_t R, int K, cudaStream_t st, const Grp &q)
{
    const size_t smem = ((size_t)KMAX * (N + 4) + (ASYNC ? 2 : 1) * (size_t)ROWS * (N + 4 + KMAX + 4)) * sizeof(float) + 16;
    NET_TRY(set_smem(net_dense_bwd_kernel<N, KMAX, ROWS, ASYNC, XRELU>, smem));
    int per_sm = 1;
    NET_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, net_dense_bwd_kernel<N, KMAX, ROWS, ASYNC, XRELU>, 512, smem));
    if (per_sm < 1) per_sm = 1;
    const dim3 grid(grid_x((R + ROWS - 1) / ROWS, (int64_t)sm_count() * per_sm, q.g), q.g);
    net_dense_bwd_kernel<N, KMAX, ROWS, ASYNC, XRELU><<<grid, 512, smem, st>>>(dZ, X, ldx, W, dX, K, accumulate, xact, dW, db, R, K,
                                                                               q.wstr, q.gstr);
    return cudaGetLastError();
}

template <int N, int KMAX, int XRELU = 0>
static cudaError_t dense_bwd_t(const float *dZ, const float *X, int ldx, const float *W, float *dX, int accumulate, int xact, float *dW,
                               float *db, int64_t R, int K, cudaStream_t st, const Grp &q)
{
    // two stages of 128-row tiles where they fit into shared memory, else of 64-row tiles
    constexpr bool fits = ((size_t)KMAX * (N + 4) + 2 * (size_t)128 * (N + 4 + KMAX + 4)) * sizeof(float) + 16 <= 227 * 1024;
    if (!rows_aligned(X, ldx, K)) return dense_bwd_a<N, KMAX, 128, 0, XRELU>(dZ, X, ldx, W, dX, accumulate, xact, dW, db, R, K, st, q);
    return dense_bwd_a<N, KMAX, fits ? 128 : 64, 1, XRELU>(dZ, X, ldx, W, dX, accumulate, xact, dW, db, R, K, st, q);
}

// gradients of Y = X W + b from dZ [R][N]; dX [R][K] (lddx = K) may be NULL; xact: dX *= act'(X), 1 = tanh, 2 = relu (the CENT
// policy's 64 -> 32 and 128 -> 64 layers, the only ones built for it)
static cudaError_t dense_bwd(const float *dZ, const float *X, int ldx, const float *W, float *dX, int accumulate, int xact, float *dW,
                             float *db, int64_t R, int K, int N, cudaStream_t st, const Grp &q = Grp())
{
    if (xact == 2) return N == 32 ? dense_bwd_t<32, 64, 1>(dZ, X, ldx, W, dX, accumulate, xact, dW, db, R, K, st, q)
                                  : dense_bwd_t<64, 128, 1>(dZ, X, ldx, W, dX, accumulate, xact, dW, db, R, K, st, q);
    if (N == 128) return K <= 64 ? dense_bwd_t<128, 64>(dZ, X, ldx, W, dX, accumulate, xact, dW, db, R, K, st, q)
                                 : dense_bwd_t<128, 128>(dZ, X, ldx, W, dX, accumulate, xact, dW, db, R, K, st, q);
    if (N == 64) return K <= 64 ? dense_bwd_t<64, 64>(dZ, X, ldx, W, dX, accumulate, xact, dW, db, R, K, st, q)
                                : dense_bwd_t<64, 128>(dZ, X, ldx, W, dX, accumulate, xact, dW, db, R, K, st, q);
    return K <= 64 ? dense_bwd_t<32, 64>(dZ, X, ldx, W, dX, accumulate, xact, dW, db, R, K, st, q)
                   : dense_bwd_t<32, 128>(dZ, X, ldx, W, dX, accumulate, xact, dW, db, R, K, st, q);
}

// wide-K layers (CENT family)
template <int J, int ACT>
static cudaError_t wide_fwd_t(const float *X, const float *W, const float *b, float *Y, int64_t R, int K, cudaStream_t st)
{
    net_wide_fwd_kernel<J, ACT><<<(unsigned)((R + kWRows - 1) / kWRows), 256, 0, st>>>(X, W, b, Y, R, K);
    return cudaGetLastError();
}
// Y [R][N] = act(X [R][K] W + b), N in {64, 128}, act 1 tanh / 2 relu
static cudaError_t wide_fwd(const float *X, const float *W, const float *b, float *Y, int64_t R, int K, int N, int act, cudaStream_t st)
{
    if (N == 128) return act == 2 ? wide_fwd_t<2, 2>(X, W, b, Y, R, K, st) : wide_fwd_t<2, 1>(X, W, b, Y, R, K, st);
    return wide_fwd_t<1, 1>(X, W, b, Y, R, K, st);
}
// dW [K][N] (TRANS: [N][K]) += X^T dZ, db += sum dZ.  The rows are split across CTAs so that the K panels x row slices fill the SMs
// about four CTAs deep even when K has few panels (C3: 1 696 / 64 = 27).
template <int N, int TRANS>
static cudaError_t wide_dw_t(const float *X, int ldx, const float *dZ, float *dW, float *db, int64_t R, int K, cudaStream_t st)
{
    const int panels = (K + kWPanel - 1) / kWPanel;
    const int64_t tiles = (R + kWTile - 1) / kWTile;
    int64_t split = ((int64_t)4 * sm_count() + panels - 1) / panels;
    if (split > tiles) split = tiles;
    if (split < 1) split = 1;
    const int64_t per = (tiles + split - 1) / split * kWTile;
    const dim3 grid((unsigned)panels, (unsigned)((R + per - 1) / per));
    net_wide_dw_kernel<N, TRANS><<<grid, 256, 0, st>>>(X, ldx, dZ, dW, db, R, K, per);
    return cudaGetLastError();
}

static int env_group(int n) { return n >= kRows ? 1 : kRows / n; }          // head kernels: one thread per row, 256 rows per CTA
static dim3 env_grid(int n, int64_t S, int per_sm, int g = 1)
{
    const int G = env_group(n);
    return dim3(grid_x((S + G - 1) / G, (int64_t)sm_count() * per_sm, g), g);
}

// n x n kernels: a CTA owns G whole envs at a time, at most `cap` rows: 64 rows up to n = 32 (three or more CTAs per SM hide the
// latency of the short strips: the kernels wait on global loads), 128 up to n = 64, one env beyond
struct EnvGeom { int G, cap; };
static EnvGeom env_geom(int n)
{
    EnvGeom g;
    const int target = n <= 32 ? 64 : 128;
    g.G = n >= target ? 1 : target / n;
    g.cap = (g.G * n + 3) & ~3;
    return g;
}

struct EnvCall {
    int n, L;
    int64_t S;                   // steps of one member
    const uint32_t *adj, *chan;
    cudaStream_t st;
    Grp q;
};

template <typename Kern>
static cudaError_t env_launch_dims(Kern k, int threads, size_t smem, const EnvCall &c, dim3 *grid)
{
    NET_TRY(set_smem(k, smem));
    int per_sm = 1;
    NET_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, threads, smem));
    if (per_sm < 1) per_sm = 1;
    const EnvGeom g = env_geom(c.n);
    *grid = dim3(grid_x((c.S + g.G - 1) / g.G, (int64_t)sm_count() * per_sm, c.q.g), c.q.g);
    return cudaSuccess;
}
static size_t cs_floats(int KT, int threads) { return (size_t)(threads / 32) * 8 * (KT * 32 + 4); }

template <int KT>
static cudaError_t scores_t(const EnvCall &c, const float *Q, const float *E, float *M)
{
    const EnvGeom g = env_geom(c.n);
    const size_t smem = 2 * (size_t)g.cap * kNP * sizeof(float);
    dim3 grid;
    NET_TRY(env_launch_dims(net_scores_kernel<KT, 256>, 256, smem, c, &grid));
    net_scores_kernel<KT, 256><<<grid, 256, smem, c.st>>>(Q, E, M, c.n, g.G, g.cap, c.S);
    return cudaGetLastError();
}
template <int KT>
static cudaError_t agg_fwd_t(const EnvCall &c, int l, const float *M, const float *V, const float *bias, float *H, const float *res,
                             float *Xout)
{
    const EnvGeom g = env_geom(c.n);
    const size_t rows = (size_t)g.cap * kNP;
    const bool wide = c.n > 64 && (rows + cs_floats(KT, 512)) * sizeof(float) <= kSmemMax;      // one env per CTA: 16 warps share it
    const size_t smem = (rows + cs_floats(KT, wide ? 512 : 256)) * sizeof(float);
    dim3 grid;
    if (wide) {
        NET_TRY(env_launch_dims(net_agg_fwd_kernel<KT, 512>, 512, smem, c, &grid));
        net_agg_fwd_kernel<KT, 512><<<grid, 512, smem, c.st>>>(M, c.adj, c.chan, c.L, l, V, bias, H, res, Xout, c.n, g.G, g.cap, c.S, c.q.wstr);
    } else {
        NET_TRY(env_launch_dims(net_agg_fwd_kernel<KT, 256>, 256, smem, c, &grid));
        net_agg_fwd_kernel<KT, 256><<<grid, 256, smem, c.st>>>(M, c.adj, c.chan, c.L, l, V, bias, H, res, Xout, c.n, g.G, g.cap, c.S, c.q.wstr);
    }
    return cudaGetLastError();
}
// the two backward kernels hold two row blocks: large teams (one env per CTA, a CTA per SM) run them with 16 warps when the
// coefficient strips of 16 warps still fit
template <int KT>
static cudaError_t agg_bwd_t(const EnvCall &c, int l, const float *M, const float *V, const float *H, const float *dH, float *dV,
                             float *dM, float *CT, float *db)
{
    const EnvGeom g = env_geom(c.n);
    const size_t rows = 2 * (size_t)g.cap * kNP;
    const bool wide = c.n > 64 && (rows + cs_floats(KT, 512)) * sizeof(float) <= kSmemMax;
    const size_t smem = (rows + cs_floats(KT, wide ? 512 : 256)) * sizeof(float);
    dim3 grid;
    if (wide) {
        NET_TRY(env_launch_dims(net_agg_bwd_kernel<KT, 512>, 512, smem, c, &grid));
        net_agg_bwd_kernel<KT, 512><<<grid, 512, smem, c.st>>>(M, c.adj, c.chan, c.L, l, V, H, dH, dV, dM, CT, db, c.n, g.G, g.cap, c.S,
                                                               c.q.gstr);
    } else {
        NET_TRY(env_launch_dims(net_agg_bwd_kernel<KT, 256>, 256, smem, c, &grid));
        net_agg_bwd_kernel<KT, 256><<<grid, 256, smem, c.st>>>(M, c.adj, c.chan, c.L, l, V, H, dH, dV, dM, CT, db, c.n, g.G, g.cap, c.S,
                                                               c.q.gstr);
    }
    return cudaGetLastError();
}
template <int KT>
static cudaError_t softmax_bwd_t(const EnvCall &c, const float *M, const float *dM, int64_t dm_stride, const float *E, const float *Q,
                                 float *dQ, float *dE, float *CT)
{
    const EnvGeom g = env_geom(c.n);
    const size_t rows = 2 * (size_t)g.cap * kNP;
    const bool wide = c.n > 64 && (rows + cs_floats(KT, 512)) * sizeof(float) <= kSmemMax;
    const size_t smem = (rows + cs_floats(KT, wide ? 512 : 256)) * sizeof(float);
    dim3 grid;
    if (wide) {
        NET_TRY(env_launch_dims(net_softmax_bwd_kernel<KT, 512>, 512, smem, c, &grid));
        net_softmax_bwd_kernel<KT, 512><<<grid, 512, smem, c.st>>>(M, dM, c.L, dm_stride, E, Q, dQ, dE, CT, c.n, g.G, g.cap, c.S);
    } else {
        NET_TRY(env_launch_dims(net_softmax_bwd_kernel<KT, 256>, 256, smem, c, &grid));
        net_softmax_bwd_kernel<KT, 256><<<grid, 256, smem, c.st>>>(M, dM, c.L, dm_stride, E, Q, dQ, dE, CT, c.n, g.G, g.cap, c.S);
    }
    return cudaGetLastError();
}

#define KT_DISPATCH(fn, ...)                                              \
    do {                                                                  \
        const int kt__ = (c.n + 31) / 32;                                 \
        if (kt__ <= 1) return fn<1>(__VA_ARGS__);                         \
        if (kt__ <= 2) return fn<2>(__VA_ARGS__);                         \
        if (kt__ <= 4) return fn<4>(__VA_ARGS__);                         \
        if (kt__ <= 7) return fn<7>(__VA_ARGS__);                         \
        return fn<8>(__VA_ARGS__);                                        \
    } while (0)

static const size_t kSmallBwdSmem = (2 * (size_t)kSmallRows * kNP + (size_t)kSmallRows * kSmallN) * sizeof(float);
static dim3 small_grid(const EnvCall &c, int per_sm)
{
    const int G = kSmallRows / c.n;
    return dim3(grid_x((c.S + G - 1) / G, (int64_t)sm_count() * per_sm, c.q.g), c.q.g);
}
static cudaError_t scores(const EnvCall &c, const float *Q, const float *E, float *M)
{
    if (c.n <= kSmallN) {
        net_small_scores_kernel<<<small_grid(c, 6), kSmallRows, 0, c.st>>>(Q, E, M, c.n, kSmallRows / c.n, c.S);
        return cudaGetLastError();
    }
    KT_DISPATCH(scores_t, c, Q, E, M);
}
static cudaError_t agg_fwd(const EnvCall &c, int l, const float *M, const float *V, const float *bias, float *H, const float *res,
                           float *Xout)
{
    if (c.n <= kSmallN) {
        net_small_agg_fwd_kernel<<<small_grid(c, 6), kSmallRows, 0, c.st>>>(M, c.adj, c.chan, c.L, l, V, bias, H, res, Xout, c.n,
                                                                             kSmallRows / c.n, c.S, c.q.wstr);
        return cudaGetLastError();
    }
    KT_DISPATCH(agg_fwd_t, c, l, M, V, bias, H, res, Xout);
}
static cudaError_t agg_bwd(const EnvCall &c, int l, const float *M, const float *V, const float *H, const float *dH, float *dV, float *dM,
                           float *CT, float *db)
{
    if (c.n <= kSmallN) {
        NET_TRY(set_smem(net_small_agg_bwd_kernel, kSmallBwdSmem));
        net_small_agg_bwd_kernel<<<small_grid(c, 3), kSmallRows, kSmallBwdSmem, c.st>>>(M, c.adj, c.chan, c.L, l, V, H, dH, dV, dM, db, c.n,
                                                                             kSmallRows / c.n, c.S, c.q.gstr);
        return cudaGetLastError();
    }
    KT_DISPATCH(agg_bwd_t, c, l, M, V, H, dH, dV, dM, CT, db);
}
static cudaError_t softmax_bwd(const EnvCall &c, const float *M, const float *dM, int64_t dm_stride, const float *E, const float *Q,
                               float *dQ, float *dE, float *CT)
{
    if (c.n <= kSmallN) {
        NET_TRY(set_smem(net_small_softmax_bwd_kernel, kSmallBwdSmem));
        net_small_softmax_bwd_kernel<<<small_grid(c, 3), kSmallRows, kSmallBwdSmem, c.st>>>(M, dM, c.L, dm_stride, E, Q, dQ, dE, c.n, kSmallRows / c.n, c.S);
        return cudaGetLastError();
    }
    KT_DISPATCH(softmax_bwd_t, c, M, dM, dm_stride, E, Q, dQ, dE, CT);
}

// workspace of one chunk of `steps` env steps (floats)
static constexpr size_t kWsSlack = 164;      // alignment of the base pointer and of each of the <= 30 carved arrays; the loss sum
struct NetWs {
    float *h1, *E, *Q, *M, *V[CM_MAX_LAYERS], *H[CM_MAX_LAYERS], *X, *g1, *g2, *g3, *t32, *t64a, *t64b, *t64c, *t128, *dM, *CT;
};
static size_t ws_floats_per_step(const cm_net_desc &d, bool backward)
{
    const int n = d.n_agents, L = d.n_layers;
    if (d.kind == CM_NET_POLICY_CENT)        // h1 h2 h3; backward: d logits, dZ3 dZ2 dZ1
        return 128 + 64 + 32 + (backward ? 5 * (size_t)n + 32 + 64 + 128 : 0);
    if (d.kind == CM_NET_BASELINE_MLP) return 3 * 64 + (backward ? 3 * 64 : 0);
    size_t rows = 128 + 64 + 64 + (size_t)L * 128 + 64 + 128 + 64 + 32;
    size_t sq = 1;
    if (backward) { rows += 32 + 3 * 64 + 128; sq += 1 + (size_t)L; }          // dM: one n x n array per layer
    return (size_t)n * rows + sq * (size_t)n * n;
}
static NetWs carve(float *p, int n, int L, int64_t steps, bool backward)
{
    NetWs w;
    const size_t R = (size_t)steps * n, S2 = (size_t)steps * n * n;
    auto take = [&](size_t k) { float *q = p; p += (k + 3) & ~(size_t)3; return q; };      // every array 16-byte aligned
    w.h1 = take(R * 128); w.E = take(R * 64); w.Q = take(R * 64); w.M = take(S2);
    for (int l = 0; l < L; ++l) { w.V[l] = take(R * 64); w.H[l] = take(R * 64); }
    w.X = take(R * 64); w.g1 = take(R * 128); w.g2 = take(R * 64); w.g3 = take(R * 32);
    w.t32 = w.t64a = w.t64b = w.t64c = w.t128 = w.dM = w.CT = nullptr;
    if (backward) {
        w.t32 = take(R * 32); w.t64a = take(R * 64); w.t64b = take(R * 64); w.t64c = take(R * 64); w.t128 = take(R * 128);
        w.dM = take(S2 * L); w.CT = take(S2);
    }
    return w;
}

// the shared trunk: encoder -> attention -> graph convolutions -> X
static cudaError_t trunk_fwd(const cm_net_desc &d, const EnvCall &c, const float *wts, const Blob &o, const float *obs, const NetWs &w)
{
    const int64_t R = c.S * d.n_agents;                               // rows of one member
    NET_TRY(dense_fwd(obs, d.obs_dim, wts + o.enc_w1, wts + o.enc_b1, w.h1, R, d.obs_dim, 128, 1, c.st, c.q));
    NET_TRY(dense_fwd(w.h1, 128, wts + o.enc_w2, wts + o.enc_b2, w.E, R, 128, 64, 1, c.st, c.q));
    NET_TRY(dense_fwd(w.E, 64, wts + o.att_w, nullptr, w.Q, R, 64, 64, 0, c.st, c.q));
    NET_TRY(scores(c, w.Q, w.E, w.M));
    for (int l = 0; l < d.n_layers; ++l) {
        const float *Hin = l == 0 ? w.E : w.H[l - 1];
        NET_TRY(dense_fwd(Hin, 64, wts + o.gcn_w + l * kE * kE, nullptr, w.V[l], R, 64, 64, 0, c.st, c.q));
        const bool last = l == d.n_layers - 1;
        NET_TRY(agg_fwd(c, l, w.M, w.V[l], wts + o.gcn_b + l * kE, w.H[l], (last && d.residual) ? w.E : nullptr,
                        (last && d.residual) ? w.X : nullptr));
    }
    return cudaSuccess;
}

// dXin (gradient of the trunk's output X = E + H_L or H_L, in w.t64b) -> parameter gradients of the trunk
static cudaError_t trunk_bwd(const cm_net_desc &d, const EnvCall &c, const float *wts, float *grad, const Blob &o, const float *obs,
                             const NetWs &w)
{
    const int64_t R = c.S * d.n_agents;
    const int L = d.n_layers;
    const size_t S2 = (size_t)c.q.g * c.S * d.n_agents * d.n_agents;  // layer l's dM array starts at w.dM + l * S2 (scalar accesses only)
    float *dE = w.t64b;                       // with the residual connection the gradient of X is the first term of dE
    const float *dHl = w.t64b;
    bool dE_init = d.residual != 0;
    if (!d.residual) {                        // dX is dH_L only: park it, dE starts empty
        NET_TRY(cudaMemcpyAsync(w.t64a, w.t64b, (size_t)c.q.g * R * 64 * sizeof(float), cudaMemcpyDeviceToDevice, c.st));
        dHl = w.t64a;
    }
    for (int l = L - 1; l >= 0; --l) {
        NET_TRY(agg_bwd(c, l, w.M, w.V[l], w.H[l], dHl, w.t64c, w.dM + (size_t)l * S2, w.CT, grad + o.gcn_b + l * kE));
        const float *Hin = l == 0 ? w.E : w.H[l - 1];
        if (l == 0) {
            NET_TRY(dense_bwd(w.t64c, Hin, 64, wts + o.gcn_w, dE, dE_init ? 1 : 0, 0, grad + o.gcn_w, nullptr, R, 64, 64, c.st, c.q));
            dE_init = true;
        } else {
            NET_TRY(dense_bwd(w.t64c, Hin, 64, wts + o.gcn_w + l * kE * kE, w.t64a, 0, 0, grad + o.gcn_w + l * kE * kE, nullptr, R, 64, 64,
                              c.st, c.q));
            dHl = w.t64a;
        }
    }
    NET_TRY(softmax_bwd(c, w.M, w.dM, (int64_t)S2, w.E, w.Q, w.t64c, dE, w.CT));
    // the last term of dE (through Q = E W_a); the same pass turns the sum into dZ of the embedding layer: dE (1 - E^2)
    NET_TRY(dense_bwd(w.t64c, w.E, 64, wts + o.att_w, dE, 1, 1, grad + o.att_w, nullptr, R, 64, 64, c.st, c.q));
    NET_TRY(dense_bwd(dE, w.h1, 128, wts + o.enc_w2, w.t128, 0, 1, grad + o.enc_w2, grad + o.enc_b2, R, 128, 64, c.st, c.q));
    NET_TRY(dense_bwd(w.t128, obs, d.obs_dim, wts + o.enc_w1, nullptr, 0, 0, grad + o.enc_w1, grad + o.enc_b1, R, d.obs_dim, 128, c.st, c.q));
    return cudaSuccess;
}

static Blob trunk_of(const CriticBlob &cb)
{
    Blob o = {};
    o.enc_w1 = cb.enc_w1; o.enc_b1 = cb.enc_b1; o.enc_w2 = cb.enc_w2; o.enc_b2 = cb.enc_b2; o.att_w = cb.att_w;
    o.gcn_w = cb.gcn_w; o.gcn_b = cb.gcn_b;
    return o;
}

// the CENT family: policy (CentralizedCategoricalMLPPolicy) or baseline (GaussianMLPBaseline) over `steps` env steps, one row per step
static cudaError_t run_chunk_cent(const cm_net_desc &d, const cm_net_io &io, int64_t s0, int64_t steps, float *wsp, double *lacc,
                                  cudaStream_t st)
{
    const int n = d.n_agents, K = n * d.obs_dim, NO = n * CM_ACTIONS;
    const bool backward = io.grad != nullptr;
    const int64_t R = steps;
    const float *obs = io.obs + s0 * K;
    const float *wts = io.weights;
    float *g = io.grad;
    auto take = [&](size_t k) { float *q = wsp; wsp += (k + 3) & ~(size_t)3; return q; };      // every array 16-byte aligned
    if (d.kind == CM_NET_BASELINE_MLP) {
        const BaselineBlob o = baseline_blob_layout(K);
        float *h1 = take(R * 64), *h2 = take(R * 64), *h3 = take(R * 64);
        NET_TRY(wide_fwd(obs, wts + o.w1, wts + o.b1, h1, R, K, 64, 1, st));
        NET_TRY(dense_fwd(h1, 64, wts + o.w2, wts + o.b2, h2, R, 64, 64, 1, st));
        NET_TRY(dense_fwd(h2, 64, wts + o.w3, wts + o.b3, h3, R, 64, 64, 1, st));
        CriticHeadArgs a = {};                   // the critic head with one "agent" per step: V = h3 w4 + b4
        a.c1 = h3; a.w2 = wts + o.w4; a.b2 = wts + o.b4; a.log_std = wts + o.log_std;
        a.returns = io.returns ? io.returns + s0 : nullptr;
        a.inv_count = io.inv_count;
        a.values = io.values ? io.values + s0 : nullptr;
        a.loss = lacc;
        a.unclamped = 1;
        a.n = 1; a.G = env_group(1); a.S = steps;
        float *dz3 = nullptr, *dz2 = nullptr, *dz1 = nullptr;
        if (backward) {
            dz3 = take(R * 64); dz2 = take(R * 64); dz1 = take(R * 64);
            a.dc1 = dz3; a.dw2 = g + o.w4; a.db2 = g + o.b4; a.dlog_std = g + o.log_std;
        }
        net_critic_head_kernel<<<env_grid(1, steps, 4), kNetThreads, 0, st>>>(a);
        NET_TRY(cudaGetLastError());
        if (!backward) return cudaSuccess;
        NET_TRY(dense_bwd(dz3, h2, 64, wts + o.w3, dz2, 0, 1, g + o.w3, g + o.b3, R, 64, 64, st));
        NET_TRY(dense_bwd(dz2, h1, 64, wts + o.w2, dz1, 0, 1, g + o.w2, g + o.b2, R, 64, 64, st));
        return wide_dw_t<64, 0>(obs, K, dz1, g + o.w1, g + o.b1, R, K, st);
    }
    const CentBlob o = cent_blob_layout(n, d.obs_dim);
    const int act = (d.flags & CM_NET_FLAG_RELU) ? 2 : 1;
    float *h1 = take(R * 128), *h2 = take(R * 64), *h3 = take(R * 32);
    NET_TRY(wide_fwd(obs, wts + o.w1, wts + o.b1, h1, R, K, 128, act, st));
    NET_TRY(dense_fwd(h1, 128, wts + o.w2, wts + o.b2, h2, R, 128, 64, act, st));
    NET_TRY(dense_fwd(h2, 64, wts + o.w3, wts + o.b3, h3, R, 64, 32, act, st));
    PolicyHeadArgs a = {};
    a.g3 = h3; a.w4 = wts + o.w4; a.b4 = wts + o.b4;
    a.avail_bits = io.avail_bits ? io.avail_bits + s0 * n : nullptr;
    a.actions = io.actions ? io.actions + s0 * n : nullptr;
    a.adv = io.adv ? io.adv + s0 : nullptr;
    a.old_ll = io.old_ll ? io.old_ll + s0 : nullptr;
    a.valid = io.valid ? io.valid + s0 : nullptr;
    a.inv_count = io.inv_count; a.ent_coeff = d.ent_coeff; a.clip_lo = d.clip_lo; a.clip_hi = d.clip_hi;
    a.ll = io.ll ? io.ll + s0 : nullptr;
    a.ent = io.entropy ? io.entropy + s0 : nullptr;
    a.probs = io.probs ? io.probs + s0 * n * CM_ACTIONS : nullptr;
    a.loss = lacc;
    a.relu = act == 2;
    a.n = n; a.G = env_group(n); a.S = steps;
    float *dz3 = nullptr, *dz2 = nullptr, *dz1 = nullptr;
    if (backward) {
        a.dlogits = take(R * NO);
        dz3 = take(R * 32); dz2 = take(R * 64); dz1 = take(R * 128);
        a.dg3 = dz3; a.db4 = g + o.b4;
    }
    net_cent_head_kernel<<<env_grid(n, steps, 4), kNetThreads, 0, st>>>(a);
    NET_TRY(cudaGetLastError());
    if (!backward) return cudaSuccess;
    NET_TRY((wide_dw_t<32, 1>(a.dlogits, NO, h3, g + o.w4, nullptr, R, NO, st)));           // dW4 [32][5n] = h3^T d logits
    NET_TRY(dense_bwd(dz3, h2, 64, wts + o.w3, dz2, 0, act, g + o.w3, g + o.b3, R, 64, 32, st));
    NET_TRY(dense_bwd(dz2, h1, 128, wts + o.w2, dz1, 0, act, g + o.w2, g + o.b2, R, 128, 64, st));
    return wide_dw_t<128, 0>(obs, K, dz1, g + o.w1, g + o.b1, R, K, st);
}

// One launch sequence over steps [s0, s0 + steps) of members m0 .. m0 + g - 1 of a set, s0 = m0 * P + off (P = steps per member;
// one network: m0 = 0, ng = 1).  ng > 1 only for whole members (off = 0, steps = P), so that the inputs and the workspace both hold
// the ng members' rows `steps` steps apart.
static cudaError_t run_chunk(const cm_net_desc &d, const cm_net_io &io, int64_t P, int m0, int ng, int64_t off, int64_t steps, float *wsp,
                             double *lacc, cudaStream_t st)
{
    const int64_t s0 = m0 * P + off;
    if (cent_kind(d.kind)) return run_chunk_cent(d, io, s0, steps, wsp, lacc, st);
    const int n = d.n_agents, D = d.obs_dim, L = d.n_layers, W = (n + 31) / 32;
    const bool backward = io.grad != nullptr;
    const bool set = io.n_policies > 1;
    const NetWs w = carve(wsp, n, L, ng * steps, backward);
    const int64_t R = steps * n, r0 = s0 * n;
    EnvCall c;
    c.n = n; c.L = L; c.S = steps; c.st = st;
    c.adj = io.adj_bits ? io.adj_bits + r0 * W : nullptr;
    c.chan = io.chan_bits ? io.chan_bits + s0 * L * n * W : nullptr;
    c.q.g = ng;
    c.q.wstr = set ? io.weights_stride : 0;
    c.q.gstr = set ? io.grad_stride : 0;
    const Grp &q = c.q;
    const float *obs = io.obs + r0 * D;
    const float *wts = io.weights + m0 * q.wstr;
    float *grad = io.grad ? io.grad + m0 * q.gstr : nullptr;
    const float *inv_counts = set ? io.inv_counts + m0 : nullptr;
    if (lacc) lacc += m0;
    const int G = env_group(n);
    if (d.kind == CM_NET_POLICY || d.kind == CM_NET_POLICY_DEC) {
        const bool dec = d.kind == CM_NET_POLICY_DEC;        // Obs-DP: encoder D -> 128 -> 64 and head 64 -> 32 -> 5 per agent row, no communication
        const Blob o = blob_layout(D, L);
        const float *Xin = nullptr;
        if (dec) {
            NET_TRY(dense_fwd(obs, D, wts + o.enc_w1, wts + o.enc_b1, w.h1, R, D, 128, 1, st, q));
            NET_TRY(dense_fwd(w.h1, 128, wts + o.enc_w2, wts + o.enc_b2, w.E, R, 128, 64, 1, st, q));
            NET_TRY(dense_fwd(w.E, 64, wts + o.head_w3, wts + o.head_b3, w.g3, R, 64, 32, 1, st, q));
        } else {
            NET_TRY(trunk_fwd(d, c, wts, o, obs, w));
            Xin = d.residual ? w.X : w.H[L - 1];
            NET_TRY(dense_fwd(Xin, 64, wts + o.head_w1, wts + o.head_b1, w.g1, R, 64, 128, 1, st, q));
            NET_TRY(dense_fwd(w.g1, 128, wts + o.head_w2, wts + o.head_b2, w.g2, R, 128, 64, 1, st, q));
            NET_TRY(dense_fwd(w.g2, 64, wts + o.head_w3, wts + o.head_b3, w.g3, R, 64, 32, 1, st, q));
        }
        PolicyHeadArgs a = {};
        a.g3 = w.g3; a.w4 = wts + o.head_w4; a.b4 = wts + o.head_b4;
        a.avail_bits = io.avail_bits ? io.avail_bits + r0 : nullptr;
        a.actions = io.actions ? io.actions + r0 : nullptr;
        a.adv = io.adv ? io.adv + s0 : nullptr;
        a.old_ll = io.old_ll ? io.old_ll + s0 : nullptr;
        a.valid = io.valid ? io.valid + s0 : nullptr;
        a.inv_count = io.inv_count; a.ent_coeff = d.ent_coeff; a.clip_lo = d.clip_lo; a.clip_hi = d.clip_hi;
        a.ll = io.ll ? io.ll + s0 : nullptr;
        a.ent = io.entropy ? io.entropy + s0 : nullptr;
        a.probs = io.probs ? io.probs + r0 * CM_ACTIONS : nullptr;
        a.loss = lacc;
        a.n = n; a.G = G; a.S = steps;
        a.inv_counts = inv_counts; a.wstr = q.wstr; a.gstr = q.gstr;
        if (backward) { a.dg3 = w.t32; a.dw4 = grad + o.head_w4; a.db4 = grad + o.head_b4; }
        net_policy_head_kernel<<<env_grid(n, steps, 4, ng), kNetThreads, 0, st>>>(a);
        NET_TRY(cudaGetLastError());
        if (!backward) return cudaSuccess;
        float *g = grad;
        if (dec) {
            NET_TRY(dense_bwd(w.t32, w.E, 64, wts + o.head_w3, w.t64b, 0, 1, g + o.head_w3, g + o.head_b3, R, 64, 32, st, q));
            NET_TRY(dense_bwd(w.t64b, w.h1, 128, wts + o.enc_w2, w.t128, 0, 1, g + o.enc_w2, g + o.enc_b2, R, 128, 64, st, q));
            return dense_bwd(w.t128, obs, D, wts + o.enc_w1, nullptr, 0, 0, g + o.enc_w1, g + o.enc_b1, R, D, 128, st, q);
        }
        // (the head kernel hands over dZ of the last hidden layer; every layer's dX pass applies the tanh derivative of the one below)
        NET_TRY(dense_bwd(w.t32, w.g2, 64, wts + o.head_w3, w.t64a, 0, 1, g + o.head_w3, g + o.head_b3, R, 64, 32, st, q));
        NET_TRY(dense_bwd(w.t64a, w.g1, 128, wts + o.head_w2, w.t128, 0, 1, g + o.head_w2, g + o.head_b2, R, 128, 64, st, q));
        NET_TRY(dense_bwd(w.t128, Xin, 64, wts + o.head_w1, w.t64b, 0, 0, g + o.head_w1, g + o.head_b1, R, 64, 128, st, q));
        return trunk_bwd(d, c, wts, g, o, obs, w);
    }
    const CriticBlob cb = critic_blob_layout(D, L);
    const Blob o = trunk_of(cb);
    NET_TRY(trunk_fwd(d, c, wts, o, obs, w));
    const float *Xin = d.residual ? w.X : w.H[L - 1];
    NET_TRY(dense_fwd(Xin, 64, wts + cb.dec_w1, wts + cb.dec_b1, w.g2, R, 64, 64, 1, st, q));
    CriticHeadArgs a = {};
    a.c1 = w.g2; a.w2 = wts + cb.dec_w2; a.b2 = wts + cb.dec_b2; a.log_std = wts + cb.log_std;
    a.returns = io.returns ? io.returns + s0 : nullptr;
    a.inv_count = io.inv_count;
    a.values = io.values ? io.values + s0 : nullptr;
    a.loss = lacc;
    a.n = n; a.G = G; a.S = steps;
    a.valid = io.valid ? io.valid + s0 : nullptr;
    a.inv_counts = inv_counts; a.wstr = q.wstr; a.gstr = q.gstr;
    if (backward) { a.dc1 = w.t64a; a.dw2 = grad + cb.dec_w2; a.db2 = grad + cb.dec_b2; a.dlog_std = grad + cb.log_std; }
    net_critic_head_kernel<<<env_grid(n, steps, 4, ng), kNetThreads, 0, st>>>(a);
    NET_TRY(cudaGetLastError());
    if (!backward) return cudaSuccess;
    NET_TRY(dense_bwd(w.t64a, Xin, 64, wts + cb.dec_w1, w.t64b, 0, 0, grad + cb.dec_w1, grad + cb.dec_b1, R, 64, 64, st, q));
    return trunk_bwd(d, c, wts, grad, o, obs, w);
}

}  // namespace cm

extern "C" size_t cm_critic_blob_floats(int32_t obs_dim, int32_t n_layers)
{
    return (size_t)cm::critic_blob_layout(obs_dim, n_layers).total;
}

extern "C" size_t cm_baseline_mlp_blob_floats(int32_t in_dim)
{
    return in_dim < 1 ? 0 : (size_t)cm::baseline_blob_layout(in_dim).total;
}

extern "C" size_t cm_ppo_net_workspace_floats(const cm_net_desc *desc, int64_t chunk_steps, int32_t backward)
{
    if (!desc || chunk_steps < 1) return 0;
    return cm::ws_floats_per_step(*desc, backward != 0) * (size_t)chunk_steps + cm::kWsSlack;
}

extern "C" int cm_ppo_net(const cm_net_desc *desc, const cm_net_io *io, cm_stream_t stream)
{
    using namespace cm;
    if (!desc || !io || !io->weights || !io->obs || !io->workspace || io->n_steps < 0) return CM_EINVAL;
    const cm_net_desc &d = *desc;
    if (d.kind != CM_NET_POLICY && d.kind != CM_NET_CRITIC && d.kind != CM_NET_POLICY_DEC && !cent_kind(d.kind)) return CM_EINVAL;
    if (d.n_agents < 1 || d.n_agents > CM_MAX_AGENTS || d.obs_dim < 1 || d.obs_dim > 128 ||
        (!cent_kind(d.kind) && (d.n_layers < 1 || d.n_layers > CM_MAX_LAYERS)))
        return CM_EUNSUPPORTED;
    if (io->n_policies > 1 && cent_kind(d.kind)) return CM_EUNSUPPORTED;      // (sets: the Comm-DP / Obs-DP kinds only)
    const bool value_net = d.kind == CM_NET_CRITIC || d.kind == CM_NET_BASELINE_MLP;
    if (io->grad && !value_net && (!io->actions || !io->adv)) return CM_EINVAL;
    if (io->grad && value_net && !io->returns) return CM_EINVAL;
    if (io->n_steps == 0) return CM_OK;
    if (cm_device_count() <= 0) return CM_ENODEVICE;
    const bool backward = io->grad != nullptr;
    const bool set = io->n_policies > 1;
    const int np = set ? io->n_policies : 1;
    const int64_t P = set ? io->steps_per_policy : io->n_steps;       // steps per member
    if (set) {
        const int64_t blob = d.kind == CM_NET_CRITIC ? critic_blob_layout(d.obs_dim, d.n_layers).total
                                                     : blob_layout(d.obs_dim, d.n_layers).total;
        if (io->n_policies > 65535 || P < 1 || io->n_steps != (int64_t)np * P || io->weights_stride < blob || (io->weights_stride & 3) ||
            (backward && (io->grad_stride < blob || (io->grad_stride & 3))))
            return CM_EINVAL;
        if (!io->inv_counts && (io->loss || backward)) return CM_EINVAL;
    }
    const size_t per_step = ws_floats_per_step(d, backward);
    const size_t lacc_floats = ((size_t)2 * np + 3) & ~(size_t)3;     // one float64 loss sum per member, 16-byte aligned
    if (io->workspace_floats < per_step + kWsSlack + lacc_floats - 4) return CM_EINVAL;
    const int64_t chunk = (int64_t)((io->workspace_floats - kWsSlack - (lacc_floats - 4)) / per_step);
    float *wsp = reinterpret_cast<float *>((reinterpret_cast<uintptr_t>(io->workspace) + 15) & ~(uintptr_t)15);
    double *lacc = io->loss ? reinterpret_cast<double *>(wsp) : nullptr;      // the loss sums of every chunk (16-byte aligned)
    wsp += lacc_floats;
    const cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = lacc ? cudaMemsetAsync(lacc, 0, np * sizeof(double), st) : cudaSuccess;
    if (chunk >= P) {                    // whole members per chunk, side by side in one launch sequence
        const int per = (int)(chunk / P < np ? chunk / P : np);
        for (int m0 = 0; e == cudaSuccess && m0 < np; m0 += per)
            e = run_chunk(d, *io, P, m0, per < np - m0 ? per : np - m0, 0, P, wsp, lacc, st);
    } else {                             // a member longer than a chunk: its own chunks, one after the other
        for (int m = 0; m < np; ++m)
            for (int64_t off = 0; e == cudaSuccess && off < P; off += chunk)
                e = run_chunk(d, *io, P, m, 1, off, P - off < chunk ? P - off : chunk, wsp, lacc, st);
    }
    if (e == cudaSuccess && lacc) {
        net_loss_store_kernel<<<1, 64, 0, st>>>(io->loss, lacc, np);
        e = cudaGetLastError();
    }
    return e == cudaSuccess ? CM_OK : set_cuda_error(e, CM_ECUDA);
}
