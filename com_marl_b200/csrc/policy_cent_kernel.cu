// policy_cent_kernel.cu — CENT policy (CentralizedCategoricalMLPPolicy, centralized_categorical_mlp_policy.py:11-97):
// ONE multi-layer perceptron over the concatenated observation of the whole team,
//   logits[B][5n] = W4 act(W3 act(W2 act(W1 obs[B][n*D] + b1) + b2) + b3) + b4        (hidden sizes 128, 64, 32; act = tanh | relu)
// reshaped to [B][n][5], softmax per agent, availability mask, renormalisation, sampling (:73-96, :98-117).
//
// Rows of the product are ENVS here (not agents): a CTA of 256 threads owns a tile of 64 envs and walks the four layers
// with everything but the first layer's input in shared memory.  The first layer is the only product whose K grows with
// the team (K = n*D: 84 at C1, 1 696 at C3, 10 600 at C5): observations and W1 are streamed through shared memory in chunks
// of 32 k with the next chunk's global loads in flight (registers) while the current one is multiplied; the observation
// row block is read exactly once (the kernel's only HBM stream), W1 comes from L2.  Thread (ty, tx) of the 16 x 16 grid
// owns rows 4ty..4ty+3 and the columns {4tx..4tx+3} + 64j: every shared-memory operand read is a conflict-free 128-bit
// load, 3 loads per 32 FMAs.  The output layer is walked in passes of 16 agents (80 columns): a thread computes the five
// logits of ONE agent for its four envs, so softmax / mask / sampling finish in registers (common.cuh::categorical_finish,
// the same tail and random-stream specification as the Comm-DP / Obs-DP kernels).  Exact fp32 (FFMA, tanhf).
//
// math = 1: the first layer — the one real GEMM of the whole engine (M = envs, N = 128, K = n*D) — runs on the tcgen05 tensor
// cores in its own kernel, policy_cent_l1_tc_kernel: a CTA owns 128 envs, accumulators for all 128 outputs live in tensor
// memory (2 x 128 fp32 columns: hi*hi and the cross terms), K is walked in panels of 32 by a warp-specialised pipeline with no
// CTA barrier in the loop: two teams of 8 producer warps convert alternate panels (cp.async fp32 ring -> fp16 hi / lo operands
// in the canonical K-major core-matrix layout -> fence -> one mbarrier arrival per warp), a weight warp keeps a six-deep ring
// of the pre-split, pre-arranged [W1_hi ; W1_lo] panels (cm_policy_tc_prepare) full with bulk async copies, and an issuing
// warp only waits, issues 2 + 2 tcgen05.mma of K = 16 (A_hi x [B_hi ; B_lo] with N = 256, A_lo x B_hi with N = 128; error
// compensation x = hi + 2^-12 lo like policy_tc_kernel) and commits the stages' `empty` barriers.  The epilogue
// (acc0 + 2^-12 acc1 + b1, activation) writes h1 rows to the caller's workspace and policy_cent_kernel<.., true> runs the
// remaining layers from there.  Measurements and the experiments behind the structure: DESIGN.md 3.2.
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include "common.cuh"
#include "policy_layout.cuh"
#include "tc_common.cuh"

namespace cm {

static constexpr int kCThreads = 256, kCRows = 64, kCK = 32;
static constexpr int kPH1 = kC1 + 4, kPH2 = kC2 + 4, kPH3 = kC3 + 4, kPA = kCK + 4;      // pitches: rows stay 16-byte aligned
static constexpr int kCAgentsPerPass = 16, kCOutCols = kCAgentsPerPass * CM_ACTIONS;     // 80
static constexpr int kCentSmemFloats = kCRows * (kPH1 + kPH2 + kPH3 + kPA) + kCK * kC1;

struct CentArgs {
    cm_policy_desc d;
    cm_policy_io io;
    int K, NO, relu;
    CentBlob o;
    // several policies (MULTI): CTA t runs env tile t % tiles_per_policy of env block t / tiles_per_policy with that block's
    // blob, so the tiles are counted per block and never mix two policies
    int64_t tiles_per_policy, envs_per_policy, weights_stride;
};

// tanh(x) = 1 - 2 / (2^(2 log2(e) x) + 1) through ex2.approx / rcp.approx (|error| ~3e-7, saturates correctly): the formulation
// of the tensor-core kernels' epilogues, used on the math = 1 path; math = 0 keeps tanhf
__device__ __forceinline__ float cent_tanh_fast(float x)
{
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 2.8853900817779268f));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
    return fmaf(-2.0f, r, 1.0f);
}
template <bool RELU, bool FAST = false>
__device__ __forceinline__ float cent_act(float x) { return RELU ? fmaxf(x, 0.0f) : (FAST ? cent_tanh_fast(x) : tanhf(x)); }

// out[row][col] = act(acc + bias[col]) for the thread's 4 x 4J block
template <int J, bool RELU, bool FAST = false>
__device__ __forceinline__ void cent_store(float *__restrict__ out, int ldo, const float (&acc)[4][4 * J], const float *__restrict__ bias,
                                           int ty, int tx)
{
#pragma unroll
    for (int j = 0; j < J; ++j) {
        const float4 bv = __ldg(reinterpret_cast<const float4 *>(bias + j * 64 + tx * 4));
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            float4 v;
            v.x = cent_act<RELU, FAST>(acc[i][4 * j + 0] + bv.x);
            v.y = cent_act<RELU, FAST>(acc[i][4 * j + 1] + bv.y);
            v.z = cent_act<RELU, FAST>(acc[i][4 * j + 2] + bv.z);
            v.w = cent_act<RELU, FAST>(acc[i][4 * j + 3] + bv.w);
            *reinterpret_cast<float4 *>(out + (ty * 4 + i) * ldo + j * 64 + tx * 4) = v;
        }
    }
}

// hidden layer with its input already in shared memory: out = act(in[64][K] W[K][64*J] + b), W streamed in 32-row chunks.
// (32-wide layer: J = 1 with the upper half of the 64 columns padded by zeros — W has only N = 32 real columns.)
template <int J, bool RELU, bool FAST>
__device__ __forceinline__ void cent_hidden(const float *__restrict__ in, int ldi, int K, const float *__restrict__ W, int N,
                                            const float *__restrict__ bias, float *__restrict__ out, int ldo, float *__restrict__ Bch,
                                            int tid, int ty, int tx)
{
    float acc[4][4 * J];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int c = 0; c < 4 * J; ++c) acc[i][c] = 0.0f;
    const int NP = 64 * J;                                       // padded width of the chunk
    for (int k0 = 0; k0 < K; k0 += kCK) {
        __syncthreads();                                         // previous chunk consumed (and `in` complete on the first pass)
        for (int e = tid; e < kCK * NP / 4; e += kCThreads) {
            const int kk = e / (NP / 4), c4 = e - kk * (NP / 4);
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (c4 * 4 < N) v = __ldg(reinterpret_cast<const float4 *>(W + (size_t)(k0 + kk) * N + c4 * 4));
            *reinterpret_cast<float4 *>(Bch + kk * NP + c4 * 4) = v;
        }
        __syncthreads();
        cent_mac<J>(in + k0, ldi, Bch, kCK, ty, tx, acc);
    }
    if (tx * 4 < N || J > 1) {
        if (J == 1 && N < 64) {                                  // 32-wide layer: only tx < 8 hold real columns
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float4 bv = __ldg(reinterpret_cast<const float4 *>(bias + tx * 4));
                float4 v;
                v.x = cent_act<RELU, FAST>(acc[i][0] + bv.x); v.y = cent_act<RELU, FAST>(acc[i][1] + bv.y);
                v.z = cent_act<RELU, FAST>(acc[i][2] + bv.z); v.w = cent_act<RELU, FAST>(acc[i][3] + bv.w);
                *reinterpret_cast<float4 *>(out + (ty * 4 + i) * ldo + tx * 4) = v;
            }
        } else {
            cent_store<J, RELU, FAST>(out, ldo, acc, bias, ty, tx);
        }
    }
}

template <bool RELU, bool H1G, bool MULTI>
__global__ void __launch_bounds__(kCThreads, 2) policy_cent_kernel(const CentArgs A)
{
    extern __shared__ __align__(16) float smem[];
    float *h1 = smem;                                  // [64][132]
    float *h2 = h1 + kCRows * kPH1;                    // [64][68]
    float *h3 = h2 + kCRows * kPH2;                    // [64][36]
    float *Ach = h3 + kCRows * kPH3;                   // [64][36]   streamed observation chunk
    float *Bch = Ach + kCRows * kPA;                   // [32][128]  streamed weight chunk (also [32][80] of the output layer)
    const cm_policy_io &io = A.io;
    const float *__restrict__ wts = io.weights;
    const CentBlob &o = A.o;
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15, lane = tid & 31, warp = tid >> 5;
    const int K = A.K, n = A.d.n_agents;
    int64_t row0 = (int64_t)blockIdx.x * kCRows;
    int rows = (int)min((int64_t)kCRows, io.n_envs - row0);
    if constexpr (MULTI) {
        const int64_t pol = (int64_t)blockIdx.x / A.tiles_per_policy, e0 = ((int64_t)blockIdx.x - pol * A.tiles_per_policy) * kCRows;
        wts += pol * A.weights_stride;
        row0 = pol * A.envs_per_policy + e0;
        rows = (int)min((int64_t)kCRows, A.envs_per_policy - e0);
    }

    // ---- layer 1: h1 = act(obs W1 + b1), K streamed — or the rows the tensor-core kernel left in the workspace ----
    if (H1G) {
        const float *__restrict__ src = A.io.workspace + row0 * kC1;
        for (int e = tid; e < kCRows * kC1 / 4; e += kCThreads) {
            const int r = e >> 5, c4 = e & 31;
            const float4 v = r < rows ? __ldcg(reinterpret_cast<const float4 *>(src + (size_t)r * kC1 + c4 * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
            *reinterpret_cast<float4 *>(h1 + r * kPH1 + c4 * 4) = v;
        }
    } else {
        float acc[4][8];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int c = 0; c < 8; ++c) acc[i][c] = 0.0f;
        float ra[8];
        float4 rb[4];
        const float *__restrict__ obs = io.obs + row0 * K;
        auto fetch = [&](int k0) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {                        // lane = k, warp + 8j = row: 128-byte row segments
                const int r = warp + 8 * j;
                ra[j] = (r < rows && k0 + lane < K) ? __ldg(obs + (size_t)r * K + k0 + lane) : 0.0f;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int e = tid + kCThreads * j, kk = e >> 5, c4 = e & 31;
                rb[j] = (k0 + kk < K) ? __ldg(reinterpret_cast<const float4 *>(wts + o.w1 + (size_t)(k0 + kk) * kC1 + c4 * 4))
                                      : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        };
        fetch(0);
        for (int k0 = 0; k0 < K; k0 += kCK) {
            __syncthreads();
#pragma unroll
            for (int j = 0; j < 8; ++j) Ach[(warp + 8 * j) * kPA + lane] = ra[j];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int e = tid + kCThreads * j, kk = e >> 5, c4 = e & 31;
                *reinterpret_cast<float4 *>(Bch + kk * kC1 + c4 * 4) = rb[j];
            }
            __syncthreads();
            if (k0 + kCK < K) fetch(k0 + kCK);
            cent_mac<2>(Ach, kPA, Bch, kCK, ty, tx, acc);
        }
        cent_store<2, RELU>(h1, kPH1, acc, wts + o.b1, ty, tx);
    }
    // ---- layers 2, 3 ----
    cent_hidden<1, RELU, H1G>(h1, kPH1, kC1, wts + o.w2, kC2, wts + o.b2, h2, kPH2, Bch, tid, ty, tx);
    cent_hidden<1, RELU, H1G>(h2, kPH2, kC2, wts + o.w3, kC3, wts + o.b3, h3, kPH3, Bch, tid, ty, tx);
    // ---- output layer in passes of 16 agents; thread = one agent x four envs ----
    const int NO = A.NO;
    for (int a0 = 0; a0 < n; a0 += kCAgentsPerPass) {
        __syncthreads();                                         // h3 complete / previous pass consumed
        for (int e = tid; e < kC3 * kCOutCols; e += kCThreads) {
            const int kk = e / kCOutCols, c = e - kk * kCOutCols, col = a0 * CM_ACTIONS + c;
            Bch[e] = col < NO ? __ldg(wts + o.w4 + (size_t)kk * NO + col) : 0.0f;
        }
        __syncthreads();
        const int il = a0 + tx;
        float lg[4][CM_ACTIONS];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int a = 0; a < CM_ACTIONS; ++a) lg[i][a] = 0.0f;
#pragma unroll 2
        for (int k = 0; k < kC3; k += 4) {
            float4 x[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) x[i] = *reinterpret_cast<const float4 *>(h3 + (ty * 4 + i) * kPH3 + k);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                float w[CM_ACTIONS];
#pragma unroll
                for (int a = 0; a < CM_ACTIONS; ++a) w[a] = Bch[(k + kk) * kCOutCols + tx * CM_ACTIONS + a];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float xv = kk == 0 ? x[i].x : (kk == 1 ? x[i].y : (kk == 2 ? x[i].z : x[i].w));
#pragma unroll
                    for (int a = 0; a < CM_ACTIONS; ++a) lg[i][a] = fmaf(xv, w[a], lg[i][a]);
                }
            }
        }
        if (il < n) {
            float b4[CM_ACTIONS];
#pragma unroll
            for (int a = 0; a < CM_ACTIONS; ++a) b4[a] = __ldg(wts + o.b4 + il * CM_ACTIONS + a);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int r = ty * 4 + i;
                if (r < rows) {
                    float l5[CM_ACTIONS];
#pragma unroll
                    for (int a = 0; a < CM_ACTIONS; ++a) l5[a] = lg[i][a] + b4[a];
                    const int64_t env = row0 + r;
                    categorical_finish(A.d, io, l5, env * n + il, env, il);
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// first layer on the tensor cores (math = 1)
// ------------------------------------------------------------------------------------------------
static constexpr int kL1Producers = 256, kL1Teams = 2, kL1Threads = kL1Teams * kL1Producers + 64;   // 2 teams of 8 operand-producer warps (even / odd panels) + issuing warp + weight warp
static constexpr int kL1Rows = 128, kL1KP = 32, kL1TmemCols = 256;
static constexpr int kL1RawStages = 6, kL1AStages = 2, kL1BStages = 6;         // ring depths: fp32 panels, A operands (one stage per team), weight panels
static constexpr int kL1ABytes = kL1Rows * kL1KP * 2;                 // one of A_hi / A_lo: 8 KB
static constexpr int kL1BBytes = 2 * kC1 * kL1KP * 2;                 // [B_hi ; B_lo] stacked along N: 16 KB
static constexpr int kL1RawBytes = kL1Rows * kL1KP * 4;               // fp32 observation panel as it arrives: 16 KB
static constexpr int kL1PanelHalves = 2 * kC1 * kL1KP;                // halves per prepared W1 panel
static constexpr int kL1Groups = kL1KP / 8;                           // 8-column groups per row of a panel
static constexpr int kL1Items = kL1Rows * kL1Groups / kL1Producers;   // (row, group) items per producer thread: 2
static constexpr size_t kL1SmemBytes = (size_t)kL1AStages * 2 * kL1ABytes + (size_t)kL1BStages * kL1BBytes +
                                       (size_t)kL1RawStages * kL1RawBytes + 256;                                   // 224 KB

struct CentL1Args {
    const float *obs;
    const __half *w1tc;
    const float *b1;
    float *h1;
    int *error_flag;
    int64_t n_envs;
    int K, n_panels;
    int64_t tiles_per_policy, envs_per_policy, weights_stride, tc_weights_stride;   // as in CentArgs; tc stride in halves
};

// W1 [K][128] fp32 -> per K panel of kL1KP = 32 the stacked [W1_hi ; W1_lo] (256 rows x 32 k) in the canonical K-major core-matrix layout
__global__ void cent_l1_prepare_kernel(const float *__restrict__ w1, __half *__restrict__ out, int K, int n_panels)
{
    const int total = n_panels * kL1KP * kC1;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
        const int p = e / (kL1KP * kC1), rem = e - p * (kL1KP * kC1), k = rem / kC1, r = rem - k * kC1;
        const int kg = p * kL1KP + k;
        const float v = kg < K ? w1[(size_t)kg * kC1 + r] : 0.0f;
        const __half h = __float2half_rn(v);
        const __half l = __float2half_rn((v - __half2float(h)) * 4096.0f);
        auto idx = [&](int rr) { return (rr >> 3) * (kL1KP >> 3) * 64 + (k >> 3) * 64 + (rr & 7) * 8 + (k & 7); };
        out[(size_t)p * kL1PanelHalves + idx(r)] = h;
        out[(size_t)p * kL1PanelHalves + idx(kC1 + r)] = l;
    }
}

__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src, uint32_t src_bytes)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async4(uint32_t dst, const void *src, uint32_t src_bytes)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}

// VEC: K is a multiple of 4 and the observation block is 16-byte aligned — 16-byte copies (a chunk is then either whole or absent)
template <bool RELU, bool VEC, bool MULTI>
__global__ void __launch_bounds__(kL1Threads, 1) policy_cent_l1_tc_kernel(const CentL1Args A)
{
    using namespace tc;
    extern __shared__ __align__(1024) unsigned char l1smem[];
    unsigned char *abase = l1smem;                                                   // [2][A_hi | A_lo]
    unsigned char *bbase = abase + (size_t)kL1AStages * 2 * kL1ABytes;               // [6][B_hi ; B_lo]
    unsigned char *rawbase = bbase + (size_t)kL1BStages * kL1BBytes;                 // [6] fp32 panels
    uint64_t *full_a = reinterpret_cast<uint64_t *>(rawbase + (size_t)kL1RawStages * kL1RawBytes);
    uint64_t *empty_a = full_a + kL1AStages, *full_b = empty_a + kL1AStages, *empty_b = full_b + kL1BStages;
    uint64_t *done_bar = empty_b + kL1BStages;                                       // all products of the tile have completed
    uint32_t *tmem_s = reinterpret_cast<uint32_t *>(done_bar + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int K = A.K, NP = A.n_panels;
    int64_t row0 = (int64_t)blockIdx.x * kL1Rows;
    int rows = (int)min((int64_t)kL1Rows, A.n_envs - row0);
    const __half *w1tc = A.w1tc;
    const float *b1 = A.b1;
    if constexpr (MULTI) {                                                           // this tile's policy: W1 panels and b1
        const int64_t pol = (int64_t)blockIdx.x / A.tiles_per_policy, e0 = ((int64_t)blockIdx.x - pol * A.tiles_per_policy) * kL1Rows;
        row0 = pol * A.envs_per_policy + e0;
        rows = (int)min((int64_t)kL1Rows, A.envs_per_policy - e0);
        w1tc += pol * A.tc_weights_stride;
        b1 += pol * A.weights_stride;
    }
    constexpr int kIssuer = kL1Teams * kL1Producers / 32, kLoader = kIssuer + 1;     // warps 16, 17
    const int team = warp >> 3, ptid = tid & (kL1Producers - 1);                     // producer team (panels team, team + 2, ...) and index inside it

    if (warp == kIssuer) tmem_alloc(tmem_s, kL1TmemCols);
    if (tid == 0) {
        for (int i = 0; i < kL1AStages; ++i) { mbar_init(&full_a[i], kL1Producers / 32); mbar_init(&empty_a[i], 1); }
        for (int i = 0; i < kL1BStages; ++i) { mbar_init(&full_b[i], 1); mbar_init(&empty_b[i], 1); }
        mbar_init(done_bar, 1);
        fence_mbar_init();
    }
    fence_before_thread_sync();
    __syncthreads();
    fence_after_thread_sync();
    const uint32_t tmem = *tmem_s;
    bool ok = true;

    if (warp == kLoader) {
        // ================= weight warp: keeps the six-deep weight ring full.  A 16 KB panel that every CTA of the launch asks
        // for at about the same time takes ~2.5 k cycles to arrive, so the requests run up to six panels ahead of the products;
        // a slot is re-requested as soon as the products that read it have completed =================
        if (lane == 0) {
            for (int q = 0; q < NP; ++q) {
                const int sq = q % kL1BStages, uq = q / kL1BStages;
                if (uq > 0) ok = mbar_wait(&empty_b[sq], (uint32_t)(uq - 1) & 1u) && ok;
                mbar_expect_tx(&full_b[sq], kL1BBytes);
                bulk_g2s(bbase + (size_t)sq * kL1BBytes, w1tc + (size_t)q * kL1PanelHalves, kL1BBytes, &full_b[sq]);
            }
        }
        __syncwarp();
    } else if (warp == kIssuer) {
        // ================= issuing warp: nothing but wait -> 4 products -> commit per panel (one warp's serial instruction
        // stream paces the kernel, so everything else lives in the other warps) =================
        const uint32_t leader = elect_one() ? 1u : 0u;
        const uint32_t idesc2 = make_idesc_f16(kL1Rows, 2 * kC1), idesc1 = make_idesc_f16(kL1Rows, kC1);
        const uint64_t da0 = make_smem_desc16(smem_u32(abase), kL1KP, 0), db0 = make_smem_desc16(smem_u32(bbase), kL1KP, 0);
        int sb = 0;
        uint32_t phase_b = 0;
        for (int p = 0; p < NP; ++p) {
            const int sa = p & 1;
            ok = mbar_wait(&full_b[sb], phase_b) && ok;          // the weight panel has landed
            ok = mbar_wait(&full_a[sa], (uint32_t)(p >> 1) & 1u) && ok;     // the operands are converted and fenced
            fence_after_thread_sync();
            const uint64_t da_hi = da0 + (uint64_t)((uint32_t)sa * (2 * kL1ABytes >> 4)), da_lo = da_hi + (kL1ABytes >> 4);
            const uint64_t db = db0 + (uint64_t)((uint32_t)sb * (kL1BBytes >> 4));
#pragma unroll
            for (int j = 0; j < kL1KP / 16; ++j) mma_f16_pred(tmem, da_hi + 16 * j, db + 16 * j, idesc2, (p | j) ? 1u : 0u, leader);
#pragma unroll
            for (int j = 0; j < kL1KP / 16; ++j) mma_f16_pred(tmem + (uint32_t)kC1, da_lo + 16 * j, db + 16 * j, idesc1, 1u, leader);
            mma_commit_pred(&empty_a[sa], leader);
            mma_commit_pred(&empty_b[sb], leader);
            if (++sb == kL1BStages) { sb = 0; phase_b ^= 1u; }
        }
        mma_commit_pred(done_bar, leader);
        __syncwarp();
    } else {
        // ================= producer warps: fp32 observations -> fp16 hi / lo operands in the canonical layout =================
        // work item j of a thread: 8 consecutive k (one 16-byte core-matrix row of the fp16 operands, two 16-byte chunks of the
        // fp32 panel) of one tile row.  Consecutive lanes take consecutive rows of an 8-row group: the 16-byte operand stores of
        // a quarter warp are contiguous, and the fp32 panel is kept with its 16-byte chunks XOR-swizzled by the row
        // (chunk ^ row % 8) so that the reads are conflict free as well.  A thread converts exactly the chunks it copied itself,
        // so cp.async.wait_group is all the synchronisation the fp32 ring needs.
        int it_row[kL1Items], it_grp[kL1Items];
        uint32_t it_off[kL1Items];
#pragma unroll
        for (int j = 0; j < kL1Items; ++j) {
            const int e = ptid + kL1Producers * j, r8 = e & 7, grp = (e >> 3) % kL1Groups, rb = e / (8 * kL1Groups);
            it_row[j] = rb * 8 + r8;
            it_grp[j] = grp;
            it_off[j] = (uint32_t)(rb * kL1Groups * 128 + grp * 128 + r8 * 16);
        }
        auto raw_chunk = [&](int j, int c) {    // byte offset of chunk c (0 / 1) of item j inside an fp32 panel
            return (uint32_t)(it_row[j] * (kL1KP * 4) + (((2 * it_grp[j] + c) ^ (it_row[j] & 7)) << 4));
        };
        // everything a copy needs except the panel index is fixed per item and lives in registers: the global address of the
        // item's first column, the number of columns left in its row from there (0 for a row outside the batch) and the
        // shared-memory address of its two chunks in ring slot 0.  A chunk outside the matrix is a zero-fill copy (source size
        // 0: nothing is read, so its address needs no clamping).
        const float *it_src[kL1Items];
        int it_left[kL1Items];
        uint32_t it_dst[kL1Items][2];
#pragma unroll
        for (int j = 0; j < kL1Items; ++j) {
            const bool rv = it_row[j] < rows;
            it_src[j] = rv ? A.obs + (size_t)(row0 + it_row[j]) * K + it_grp[j] * 8 : A.obs;
            it_left[j] = rv ? K - it_grp[j] * 8 : 0;
            it_dst[j][0] = smem_u32(rawbase) + raw_chunk(j, 0);
            it_dst[j][1] = smem_u32(rawbase) + raw_chunk(j, 1);
        }
        uint32_t copy_slot = (uint32_t)team * kL1RawBytes;      // ring slot of the team's next copy: p % 6 for p = team, team + 2, ...
        auto copy_panel = [&](int p) {          // this thread's share of observation panel p -> ring slot p % 6 (zero filled outside)
            if (p < NP) {
                const int kp = p * kL1KP;
#pragma unroll
                for (int j = 0; j < kL1Items; ++j) {
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        const int left = it_left[j] - kp - 4 * c;                   // columns of the row from this chunk on
                        const uint32_t dst = it_dst[j][c] + copy_slot;
                        if (VEC) {
                            cp_async16(dst, it_src[j] + kp + 4 * c, left > 0 ? 16u : 0u);
                        } else {
#pragma unroll
                            for (int i = 0; i < 4; ++i) cp_async4(dst + 4 * i, it_src[j] + kp + 4 * c + i, left > i ? 4u : 0u);
                        }
                    }
                }
            }
            copy_slot += kL1Teams * kL1RawBytes;
            if (copy_slot >= (uint32_t)kL1RawStages * kL1RawBytes) copy_slot -= (uint32_t)kL1RawStages * kL1RawBytes;
            cp_async_commit();                  // (an empty group when p >= NP keeps the group count uniform)
        };
        // a team converts every other panel into its own operand stage, so a warp's chain (copy landed -> convert -> fence ->
        // arrive) has two panel times to complete; it keeps its current panel and the next two of its own in the fp32 ring
        copy_panel(team);
        copy_panel(team + kL1Teams);
        const int sa = team;
        uint32_t read_slot = (uint32_t)team * kL1RawBytes;
        for (int p = team; p < NP; p += kL1Teams) {
            const int ua = p >> 1;
            copy_panel(p + 2 * kL1Teams);                        // six panels of observations in flight per CTA
            cp_async_wait<2>();                                  // panel p has landed (this thread's chunks)
            if (ua > 0) ok = mbar_wait(&empty_a[sa], (uint32_t)(ua - 1) & 1u) && ok;       // products of panel p - 2 are done with the stage
            unsigned char *ah = abase + (size_t)sa * 2 * kL1ABytes, *al = ah + kL1ABytes;
            const unsigned char *rawp = rawbase + read_slot;
            read_slot += kL1Teams * kL1RawBytes;
            if (read_slot >= (uint32_t)kL1RawStages * kL1RawBytes) read_slot -= (uint32_t)kL1RawStages * kL1RawBytes;
#pragma unroll
            for (int j = 0; j < kL1Items; ++j) {
                const float4 a = *reinterpret_cast<const float4 *>(rawp + raw_chunk(j, 0));
                const float4 b = *reinterpret_cast<const float4 *>(rawp + raw_chunk(j, 1));
                const float x[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
                uint32_t h[4], l[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const __half2 hh = __floats2half2_rn(x[2 * i], x[2 * i + 1]);
                    const float2 hf = __half22float2(hh);
                    const __half2 ll = __floats2half2_rn((x[2 * i] - hf.x) * 4096.0f, (x[2 * i + 1] - hf.y) * 4096.0f);
                    h[i] = *reinterpret_cast<const uint32_t *>(&hh);
                    l[i] = *reinterpret_cast<const uint32_t *>(&ll);
                }
                *reinterpret_cast<uint4 *>(ah + it_off[j]) = make_uint4(h[0], h[1], h[2], h[3]);
                *reinterpret_cast<uint4 *>(al + it_off[j]) = make_uint4(l[0], l[1], l[2], l[3]);
            }
            fence_proxy_async();                                 // generic-proxy stores -> visible to the tensor core's async proxy
            __syncwarp();
            if (lane == 0) mbar_arrive(&full_a[sa]);             // one arrival per warp
        }
        cp_async_wait<0>();
        // ---- epilogue: every product has completed when the commit behind the last panel arrives (a barrier of its own: a
        // team that did not convert the last panel may be two phases behind on that panel's stage barrier, and a parity wait
        // cannot tell two phases apart) ----
        ok = mbar_wait(done_bar, 0u) && ok;
        fence_after_thread_sync();
        const int quad = warp & 3, sub = warp >> 2, row = quad * 32 + lane;       // TMEM lane = tile row; four warps share a quadrant
        const uint32_t lane_addr = tmem + ((uint32_t)(quad * 32) << 16);
#pragma unroll 2
        for (int c = 0; c < 32; c += 8) {
            const int col = sub * 32 + c;
            float v[8], w[8];
            tmem_ld8(lane_addr + (uint32_t)col, v);
            tmem_ld8(lane_addr + (uint32_t)(kC1 + col), w);
            tmem_ld_wait();
            const float4 bv0 = __ldg(reinterpret_cast<const float4 *>(b1 + col)), bv1 = __ldg(reinterpret_cast<const float4 *>(b1 + col + 4));
            const float bb[8] = {bv0.x, bv0.y, bv0.z, bv0.w, bv1.x, bv1.y, bv1.z, bv1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = cent_act<RELU, true>(fmaf(w[i], 1.0f / 4096.0f, v[i]) + bb[i]);
            if (row < rows) {
                float *dst = A.h1 + (size_t)(row0 + row) * kC1 + col;
                *reinterpret_cast<float4 *>(dst) = make_float4(v[0], v[1], v[2], v[3]);
                *reinterpret_cast<float4 *>(dst + 4) = make_float4(v[4], v[5], v[6], v[7]);
            }
        }
    }
    if (!ok && A.error_flag) atomicExch(A.error_flag, (int)CM_ECUDA);
    fence_before_thread_sync();
    __syncthreads();
    if (warp == kIssuer) tmem_dealloc(tmem, kL1TmemCols);
}

template <typename Kern>
static int cent_set_smem(Kern kern, size_t smem, bool &done)
{
    if (done) return CM_OK;
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return set_cuda_error(e, CM_ECUDA);
    done = true;
    return CM_OK;
}

int launch_policy_cent(const cm_policy_desc *desc, const cm_policy_io *io, cudaStream_t stream)
{
    if (desc->math != 0 && desc->math != 1) return CM_EUNSUPPORTED;
    if (io->attention) return CM_EINVAL;                         // no communication, no attention weights
    if (io->n_envs == 0) return CM_OK;
    if (io->n_envs * desc->n_agents > (int64_t)1 << 30) return CM_EUNSUPPORTED;
    const bool tcl1 = desc->math == 1;
    if (tcl1 && (!io->tc_weights || !io->workspace || io->workspace_bytes < (size_t)io->n_envs * kC1 * sizeof(float))) return CM_EINVAL;
    CentArgs A;
    A.d = *desc;
    A.io = *io;
    A.K = desc->n_agents * desc->obs_dim;
    A.NO = desc->n_agents * CM_ACTIONS;
    A.relu = desc->flags & CM_POLICY_FLAG_RELU;
    A.o = cent_blob_layout(desc->n_agents, desc->obs_dim);
    const bool multi = io->n_policies > 1;
    const int64_t epp = multi ? io->envs_per_policy : io->n_envs, n_pol = multi ? io->n_policies : 1;
    A.envs_per_policy = epp;
    A.tiles_per_policy = (epp + kCRows - 1) / kCRows;
    A.weights_stride = multi ? io->weights_stride : 0;
    const size_t smem = kCentSmemFloats * sizeof(float);
    static thread_local struct { int dev; bool set[16]; } cache = {-1, {}};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return set_cuda_error(cudaGetLastError(), CM_ENODEVICE);
    if (cache.dev != dev) { cache.dev = dev; for (bool &b : cache.set) b = false; }
    int rc;
    if (tcl1) {
        CentL1Args L;
        L.obs = io->obs;
        L.w1tc = reinterpret_cast<const __half *>(io->tc_weights);
        L.b1 = io->weights + A.o.b1;
        L.h1 = io->workspace;
        L.error_flag = io->error_flag;
        L.n_envs = io->n_envs;
        L.K = A.K;
        L.n_panels = (A.K + kL1KP - 1) / kL1KP;
        L.envs_per_policy = epp;
        L.tiles_per_policy = (epp + kL1Rows - 1) / kL1Rows;
        L.weights_stride = A.weights_stride;
        L.tc_weights_stride = multi ? 2 * io->tc_weights_stride : 0;
        const unsigned grid1 = (unsigned)(n_pol * L.tiles_per_policy);
        const bool vec = (A.K & 3) == 0 && (reinterpret_cast<uintptr_t>(io->obs) & 15) == 0;
        void (*k1)(const CentL1Args) =
            multi ? (A.relu ? (vec ? policy_cent_l1_tc_kernel<true, true, true> : policy_cent_l1_tc_kernel<true, false, true>)
                            : (vec ? policy_cent_l1_tc_kernel<false, true, true> : policy_cent_l1_tc_kernel<false, false, true>))
                  : (A.relu ? (vec ? policy_cent_l1_tc_kernel<true, true, false> : policy_cent_l1_tc_kernel<true, false, false>)
                            : (vec ? policy_cent_l1_tc_kernel<false, true, false> : policy_cent_l1_tc_kernel<false, false, false>));
        if ((rc = cent_set_smem(k1, kL1SmemBytes, cache.set[8 * multi + 4 + 2 * (A.relu ? 1 : 0) + (vec ? 1 : 0)]))) return rc;
        k1<<<grid1, kL1Threads, kL1SmemBytes, stream>>>(L);
        const cudaError_t e1 = cudaGetLastError();
        if (e1 != cudaSuccess) return set_cuda_error(e1, CM_ECUDA);
    }
    const unsigned grid = (unsigned)(n_pol * A.tiles_per_policy);
    void (*k2)(const CentArgs) =
        multi ? (A.relu ? (tcl1 ? policy_cent_kernel<true, true, true> : policy_cent_kernel<true, false, true>)
                        : (tcl1 ? policy_cent_kernel<false, true, true> : policy_cent_kernel<false, false, true>))
              : (A.relu ? (tcl1 ? policy_cent_kernel<true, true, false> : policy_cent_kernel<true, false, false>)
                        : (tcl1 ? policy_cent_kernel<false, true, false> : policy_cent_kernel<false, false, false>));
    if ((rc = cent_set_smem(k2, smem, cache.set[8 * multi + 2 * (A.relu ? 0 : 1) + (tcl1 ? 0 : 1)]))) return rc;
    k2<<<grid, kCThreads, smem, stream>>>(A);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? CM_OK : set_cuda_error(e, CM_ECUDA);
}

int cent_tc_prepare(const cm_policy_desc *desc, const float *weights, float *tc_weights, cudaStream_t stream)
{
    const int K = desc->n_agents * desc->obs_dim, NP = (K + kL1KP - 1) / kL1KP;
    const CentBlob o = cent_blob_layout(desc->n_agents, desc->obs_dim);
    cent_l1_prepare_kernel<<<256, 256, 0, stream>>>(weights + o.w1, reinterpret_cast<__half *>(tc_weights), K, NP);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? CM_OK : set_cuda_error(e, CM_ECUDA);
}

}  // namespace cm

extern "C" size_t cm_policy_cent_blob_floats(int32_t n_agents, int32_t obs_dim)
{
    if (n_agents < 1 || obs_dim < 1) return 0;
    return (size_t)cm::cent_blob_layout(n_agents, obs_dim).total;
}

extern "C" size_t cm_policy_cent_tc_blob_floats(int32_t n_agents, int32_t obs_dim)
{
    if (n_agents < 1 || obs_dim < 1) return 0;
    const int NP = (n_agents * obs_dim + cm::kL1KP - 1) / cm::kL1KP;
    return (size_t)NP * cm::kL1PanelHalves / 2;
}

extern "C" size_t cm_policy_cent_workspace_bytes(int64_t n_envs) { return n_envs > 0 ? (size_t)n_envs * cm::kC1 * sizeof(float) : 0; }
