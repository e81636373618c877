// policy_attn_mma_kernel.cu — attention + graph convolutions for large teams (64 < n <= 256) on the warp-level tensor
// path (mma.sync.m16n8k16, SASS HMMA), the middle stage of the large-team pipeline (launch_policy_tc_large at the end of
// this file):
//   1. policy_tc_kernel<mode Enc> : obs rows -> E, Q = E Wa^T, H_0 Wg_0          (rows of 64 floats in io.workspace)
//   2. policy_attn_mma_kernel     : per env  M = softmax_j(Q E^T),  A_l = M * Range * chan_l / (sum + 1e-12),
//                                   H_{l+1} = tanh(A_l (H_l Wg_l) + bg_l),  X = E + H_L         (comm_base_net.py:80-108,
//                                   attention_module.py:38-49, graph_conv_module.py:51-72)
//   3. policy_tc_kernel<mode Head>: X rows -> logits / probs / actions
//
// Why mma.sync here and not tcgen05: the unit of work is a 16-row x n-key strip of ONE environment whose softmax, masking
// and re-normalisation sit between the two products; with mma.sync the strip never leaves the warp's registers — the score
// accumulators ARE the A operand of the aggregation (the C fragment of two adjacent 8-key tiles is exactly the A fragment of
// a 16-key slice) — and there is no CTA-wide barrier, TMEM hand-over or shared-memory round trip per strip.  Measured issue
// rate on B200 (tests/native/mma_sync_probe.cu): one m16n8k16 per 8 cycles per SM sub-partition = 1019 MAC/clk/SM, against
// ~43 MAC/clk/SM an FFMA version of this stage reached (DESIGN §3.2).
//
// fp32-level accuracy comes from the same error compensation as the tcgen05 kernel: x = hi + lo, hi = fp16(x),
// lo = fp16(x - hi); a product is hi*hi + hi*lo + lo*hi accumulated in fp32 in ONE accumulator (the dropped lo*lo term is
// 2^-22 relative).  lo is NOT rescaled: below 6e-5 it is an fp16 subnormal with an absolute step of 6e-8, i.e. an absolute
// error <= 3e-8 per operand of magnitude <= 1 — two orders of magnitude below the 1e-5 tolerance.
//
// One CTA of 8 warps per env.  Shared memory: keys E as fp16 hi / lo [key][64] (B operand of the scores), values H_l Wg_l
// TRANSPOSED as fp16 hi / lo [col][key] (B operand of the aggregation), Wg_{l+1} transposed hi / lo (B operand of the next
// layer's H Wg product), and a private slice per warp (its 16 query rows in fp32, its rows' neighbour mask words).
// Strips of 16 query rows are dealt round-robin to the warps; per strip: scores (4 k-slices x NT key tiles x 3 HMMA),
// softmax / mask / masked sum in the C fragments (quad shuffles), aggregation (NK/16 key slices x 8 column tiles x 3 HMMA),
// / (sum + 1e-12) + bias, tanh, then H Wg_{l+1} (4 x 8 x 3 HMMA) -> fp32 rows for the next layer, or X = E + H_L.
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include <type_traits>

#include "commarl_b200.h"
#include "common.cuh"
#include "policy_layout.cuh"

namespace cm {

static constexpr int kEhPitch = 72;          // halves per key row of E hi / lo (144 B: 8 rows x 4 lanes hit 32 distinct banks)
static constexpr int kQhPitch = 72;          // halves per query row (hi / lo) of a warp's slice
static constexpr int kWgPitch = 72;          // halves per output column of the transposed Wg

struct AttnMmaArgs {
    cm_policy_desc d;
    const float *weights;
    const uint32_t *adj_bits, *chan_bits;
    float *attention;
    const float *scr_e;
    float *scr_q;
    float *scr_hw;
    int64_t n_envs;
};
// several policies (the kMulti kernels): env b reads the blob at weights + (b / envs_per_policy) * weights_stride.  A struct of its
// own, so that the one-policy kernels keep their parameter block
struct AttnMmaSetArgs : AttnMmaArgs {
    int64_t envs_per_policy, weights_stride;
};
template <bool kMulti>
using AttnMmaArgsOf = typename std::conditional<kMulti, AttnMmaSetArgs, AttnMmaArgs>::type;
template <bool kMulti>
__device__ __forceinline__ int64_t blob_offset(const AttnMmaArgsOf<kMulti> &A, int64_t env)
{
    if constexpr (kMulti) return (env / A.envs_per_policy) * A.weights_stride;
    else return 0;
}

__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1)
{
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// (x, y) -> packed fp16 hi pair and lo pair: hi = fp16(v), lo = fp16(v - hi)
__device__ __forceinline__ void split2(float x, float y, uint32_t &hi, uint32_t &lo)
{
    const __half2 h = __floats2half2_rn(x, y);
    const float2 hf = __half22float2(h);
    const __half2 l = __floats2half2_rn(x - hf.x, y - hf.y);
    hi = *reinterpret_cast<const uint32_t *>(&h);
    lo = *reinterpret_cast<const uint32_t *>(&l);
}

// tanh(x) = 1 - 2 / (2^(2 log2(e) x) + 1) through ex2.approx / rcp.approx (|error| ~3e-7, saturates correctly); the same
// formulation as the tcgen05 kernel's epilogues
__device__ __forceinline__ float tanh_fast(float x)
{
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 2.8853900817779268f));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
    return fmaf(-2.0f, r, 1.0f);
}

// 2^x (ex2.approx.ftz); exponentials are taken in the log2 domain: exp(s - m) = 2^(s log2(e) - m log2(e)) is ONE fused
// multiply-add and one special-function instruction (__expf costs six: subtract, scale, denormal range test and fix-up).
// The rounding of m log2(e) is common to a row's keys and to its rescaling factors, so it cancels in out / (d + 1e-12 z).
static constexpr float kLog2e = 1.4426950408889634f;
static constexpr float kLog2Eps = -39.863137138648348f;     // log2(1e-12): the renormalisation's epsilon (comm_base_net.py:102)
__device__ __forceinline__ float ex2_fast(float x)
{
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

__device__ __forceinline__ float quad_max(float v)
{
    v = fmaxf(v, __shfl_xor_sync(0xFFFFFFFFu, v, 1));
    return fmaxf(v, __shfl_xor_sync(0xFFFFFFFFu, v, 2));
}
__device__ __forceinline__ float quad_sum(float v)
{
    v += __shfl_xor_sync(0xFFFFFFFFu, v, 1);
    return v + __shfl_xor_sync(0xFFFFFFFFu, v, 2);
}

// scores of one block of U <= 8 key tiles (8 U keys) starting at tile nt0: s[u] = Q E^T; three fp16 products per tile into
// one fp32 accumulator, issued U tiles apart (an HMMA needs its accumulator back before the next one on it can start)
template <int U>
__device__ __forceinline__ void score_block(float (&s)[8][4], const __half *Qh, const __half *Ql, const __half *Eh, const __half *El,
                                            int nt0, int g, int t)
{
#pragma unroll
    for (int u = 0; u < U; ++u) s[u][0] = s[u][1] = s[u][2] = s[u][3] = 0.0f;
#pragma unroll 1
    for (int ks = 0; ks < 4; ++ks) {                            // (rolled: the body alone is 3 U HMMAs; the kernel is I-cache bound otherwise)
        const int k0 = 16 * ks + 2 * t;
        uint32_t ah[4], al[4];
        ah[0] = *reinterpret_cast<const uint32_t *>(Qh + g * kQhPitch + k0);
        ah[1] = *reinterpret_cast<const uint32_t *>(Qh + (g + 8) * kQhPitch + k0);
        ah[2] = *reinterpret_cast<const uint32_t *>(Qh + g * kQhPitch + k0 + 8);
        ah[3] = *reinterpret_cast<const uint32_t *>(Qh + (g + 8) * kQhPitch + k0 + 8);
        al[0] = *reinterpret_cast<const uint32_t *>(Ql + g * kQhPitch + k0);
        al[1] = *reinterpret_cast<const uint32_t *>(Ql + (g + 8) * kQhPitch + k0);
        al[2] = *reinterpret_cast<const uint32_t *>(Ql + g * kQhPitch + k0 + 8);
        al[3] = *reinterpret_cast<const uint32_t *>(Ql + (g + 8) * kQhPitch + k0 + 8);
        uint32_t bh[U][2], bl[U][2];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const __half *eh = Eh + (8 * (nt0 + u) + g) * kEhPitch + k0, *el = El + (8 * (nt0 + u) + g) * kEhPitch + k0;
            bh[u][0] = *reinterpret_cast<const uint32_t *>(eh); bh[u][1] = *reinterpret_cast<const uint32_t *>(eh + 8);
            bl[u][0] = *reinterpret_cast<const uint32_t *>(el); bl[u][1] = *reinterpret_cast<const uint32_t *>(el + 8);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) mma16816(s[u], ah, bh[u][0], bh[u][1]);
#pragma unroll
        for (int u = 0; u < U; ++u) mma16816(s[u], ah, bl[u][0], bl[u][1]);
#pragma unroll
        for (int u = 0; u < U; ++u) mma16816(s[u], al, bh[u][0], bh[u][1]);
    }
}

struct StripState {               // rows g (index 0) and g + 8 (index 1) of the strip
    float m0, m1;                 // running maximum of the scores times log2(e): the reference point of z
    float q0, q1;                 // running maximum of the masked-in scores times log2(e): the reference point of d and out
    float z0, z1;                 // this lane's part of sum exp(s - m)
    float d0, d1;                 // this lane's part of sum mask exp(s - q)
};

// one block of U key tiles of a strip: scores, running maximum + rescaling, exp, mask, aggregation into oacc
template <int U>
__device__ __forceinline__ void attn_block(StripState &st, float (&oacc)[8][4], const __half *Qh, const __half *Ql, const __half *Eh,
                                           const __half *El, const __half *Vh, const __half *Vl, int HWP, const uint32_t *Mw, int nt0,
                                           int n, int g, int t)
{
    float s[8][4];
    score_block<U>(s, Qh, Ql, Eh, El, nt0, g, t);
    float bm0 = -1e30f, bm1 = -1e30f, bq0 = -1e30f, bq1 = -1e30f;
    uint32_t w0[U], w1[U];                                      // mask bits of keys 2t, 2t + 1 of each tile (beyond the team: 0)
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const int nt = nt0 + u, key = 8 * nt + 2 * t;
        const uint32_t valid = key + 1 < n ? 3u : (key < n ? 1u : 0u);
        w0[u] = (Mw[g * 8 + (nt >> 2)] >> (8 * (nt & 3) + 2 * t)) & valid;
        w1[u] = (Mw[(g + 8) * 8 + (nt >> 2)] >> (8 * (nt & 3) + 2 * t)) & valid;
        if (key < n) { bm0 = fmaxf(bm0, s[u][0]); bm1 = fmaxf(bm1, s[u][2]); }
        if (key + 1 < n) { bm0 = fmaxf(bm0, s[u][1]); bm1 = fmaxf(bm1, s[u][3]); }
        if (w0[u] & 1u) bq0 = fmaxf(bq0, s[u][0]);
        if (w0[u] & 2u) bq0 = fmaxf(bq0, s[u][1]);
        if (w1[u] & 1u) bq1 = fmaxf(bq1, s[u][2]);
        if (w1[u] & 2u) bq1 = fmaxf(bq1, s[u][3]);
    }
    // the running maxima in the log2 domain (x -> fl(x log2(e)) is monotone: it commutes with the maximum)
    const float ms0 = fmaxf(st.m0, quad_max(bm0) * kLog2e), ms1 = fmaxf(st.m1, quad_max(bm1) * kLog2e);
    const float mq0 = fmaxf(st.q0, quad_max(bq0) * kLog2e), mq1 = fmaxf(st.q1, quad_max(bq1) * kLog2e);
    const float sc0 = ex2_fast(st.m0 - ms0), sc1 = ex2_fast(st.m1 - ms1);
    const float sq0 = ex2_fast(st.q0 - mq0), sq1 = ex2_fast(st.q1 - mq1);
    // exp(s - m) -> exp(s - q) for the masked-in keys; capped at 2^126 (finite): a masked-in key 2^-126 below the maximum
    // has flushed to zero already, and so then has every other masked-in key — their sum is nothing next to 1e-12
    const float f0 = ex2_fast(fminf(ms0 - mq0, 126.0f)), f1 = ex2_fast(fminf(ms1 - mq1, 126.0f));
    st.m0 = ms0; st.m1 = ms1; st.q0 = mq0; st.q1 = mq1;
    st.z0 *= sc0; st.d0 *= sq0; st.z1 *= sc1; st.d1 *= sq1;
#pragma unroll
    for (int ot = 0; ot < 8; ++ot) { oacc[ot][0] *= sq0; oacc[ot][1] *= sq0; oacc[ot][2] *= sq1; oacc[ot][3] *= sq1; }
    // exp, mask (comm_base_net.py:101): the masked, un-normalised rows stay in the accumulators
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const int key = 8 * (nt0 + u) + 2 * t;
        const float e00 = key < n ? ex2_fast(fmaf(s[u][0], kLog2e, -ms0)) : 0.0f, e01 = key + 1 < n ? ex2_fast(fmaf(s[u][1], kLog2e, -ms0)) : 0.0f;
        const float e10 = key < n ? ex2_fast(fmaf(s[u][2], kLog2e, -ms1)) : 0.0f, e11 = key + 1 < n ? ex2_fast(fmaf(s[u][3], kLog2e, -ms1)) : 0.0f;
        st.z0 += e00 + e01;
        st.z1 += e10 + e11;
        s[u][0] = (w0[u] & 1u) ? e00 * f0 : 0.0f;
        s[u][1] = (w0[u] & 2u) ? e01 * f0 : 0.0f;
        s[u][2] = (w1[u] & 1u) ? e10 * f1 : 0.0f;
        s[u][3] = (w1[u] & 2u) ? e11 * f1 : 0.0f;
        st.d0 += s[u][0] + s[u][1];
        st.d1 += s[u][2] + s[u][3];
    }
    // aggregation: out[16][64] += a (H_l Wg_l): the C fragments of tiles 2s, 2s+1 are the A fragment of key slice s
#pragma unroll
    for (int ss = 0; ss < U / 2; ++ss) {
        uint32_t ah[4], al[4];
        split2(s[2 * ss][0], s[2 * ss][1], ah[0], al[0]);
        split2(s[2 * ss][2], s[2 * ss][3], ah[1], al[1]);
        split2(s[2 * ss + 1][0], s[2 * ss + 1][1], ah[2], al[2]);
        split2(s[2 * ss + 1][2], s[2 * ss + 1][3], ah[3], al[3]);
        const int k0 = 8 * (nt0 + 2 * ss) + 2 * t;
#pragma unroll
        for (int o0 = 0; o0 < 8; o0 += 4) {
            uint32_t bh[4][2], bl[4][2];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const __half *vh = Vh + (8 * (o0 + u) + g) * HWP + k0, *vl = Vl + (8 * (o0 + u) + g) * HWP + k0;
                bh[u][0] = *reinterpret_cast<const uint32_t *>(vh); bh[u][1] = *reinterpret_cast<const uint32_t *>(vh + 8);
                bl[u][0] = *reinterpret_cast<const uint32_t *>(vl); bl[u][1] = *reinterpret_cast<const uint32_t *>(vl + 8);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) mma16816(oacc[o0 + u], ah, bh[u][0], bh[u][1]);
#pragma unroll
            for (int u = 0; u < 4; ++u) mma16816(oacc[o0 + u], ah, bl[u][0], bl[u][1]);
#pragma unroll
            for (int u = 0; u < 4; ++u) mma16816(oacc[o0 + u], al, bh[u][0], bh[u][1]);
        }
    }
}

// the UNMASKED softmax of one block of U key tiles with the final maximum and sum (agent_infos['attention_weights'])
template <int U>
__device__ __forceinline__ void attn_record_block(float *att0, float *att1, bool v0, bool v1, const StripState &st, float is0, float is1,
                                                  const __half *Qh, const __half *Ql, const __half *Eh, const __half *El, int nt0, int n,
                                                  int g, int t)
{
    float s[8][4];
    score_block<U>(s, Qh, Ql, Eh, El, nt0, g, t);
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const int key = 8 * (nt0 + u) + 2 * t;
        if (v0 && key < n) att0[key] = ex2_fast(fmaf(s[u][0], kLog2e, -st.m0)) * is0;
        if (v0 && key + 1 < n) att0[key + 1] = ex2_fast(fmaf(s[u][1], kLog2e, -st.m0)) * is0;
        if (v1 && key < n) att1[key] = ex2_fast(fmaf(s[u][2], kLog2e, -st.m1)) * is1;
        if (v1 && key + 1 < n) att1[key + 1] = ex2_fast(fmaf(s[u][3], kLog2e, -st.m1)) * is1;
    }
}

// NS = number of 16-key slices (NK = 16 NS keys >= n); WARPS = warps per CTA (16, or 8 where the operands of the largest
// teams leave no room for 16 query slices).
//
// A strip's n keys are walked in BLOCKS of 64 (flash-attention style) so that a warp holds 8 score tiles at a time instead
// of n / 8: 16 warps of <= 128 registers share an env instead of 8 warps of 248 — the strip is a dependent chain of HMMAs
// and shuffles, and the number of chains in flight is what the tensor pipe's utilisation follows.  Running per row:
// m (max), z = sum exp(s - m), q (max over the masked-in keys), d = sum mask exp(s - q), out = sum mask exp(s - q) V; a
// larger maximum rescales z, or d and out.  The reference's softmax -> mask -> renormalise (comm_base_net.py:101-103) is then
//   A~ V = out / (d + 1e-12 z 2^(m - q))        (p = exp(s - m) / z;  A~ = p mask / (sum p mask + 1e-12))
// exactly, in fp32.  Taking the masked-in weights against their own maximum keeps the largest at 1: against m they can be
// far below one once the masks remove the keys that carry the attention mass, and their fp16 hi / lo split would lose its
// relative precision (or flush to zero) before the division by their small sum.  The unmasked softmax itself (agent_infos['attention_weights']) is written, when asked for, by a second
// walk over the blocks with the final m and z.
template <int NS, int WARPS, bool kMulti>
__global__ void __launch_bounds__(WARPS * 32, 1) policy_attn_mma_kernel(const AttnMmaArgsOf<kMulti> A)
{
    constexpr int NK = 16 * NS, NT = 2 * NS, NFULL = NT / 8, TAIL = NT % 8, HWP = NK + 8, THREADS = WARPS * 32;   // key blocks of 8 tiles + a tail
    extern __shared__ __align__(16) unsigned char smraw[];
    __half *Eh = reinterpret_cast<__half *>(smraw);            // [NK][72]
    __half *El = Eh + NK * kEhPitch;
    __half *Vh = El + NK * kEhPitch;                           // [64][HWP]   (H_l Wg_l)^T hi
    __half *Vl = Vh + 64 * HWP;
    __half *Wh = Vl + 64 * HWP;                                // [64][72]    Wg_{l+1}^T hi
    __half *Wl = Wh + 64 * kWgPitch;
    __half *Qs = Wl + 64 * kWgPitch;                           // [WARPS][2][16][72] query rows hi / lo
    uint32_t *Ms = reinterpret_cast<uint32_t *>(Qs + WARPS * 2 * 16 * kQhPitch);   // [WARPS][16][8] mask words

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    __half *Qh = Qs + warp * 2 * 16 * kQhPitch, *Ql = Qh + 16 * kQhPitch;
    uint32_t *Mw = Ms + warp * 16 * 8;
    const int n = A.d.n_agents, L = A.d.n_layers, W = (n + 31) >> 5;
    const Blob o = blob_layout(A.d.obs_dim, L);
    const int n_strips = (n + 15) >> 4;

    for (int64_t env = blockIdx.x; env < A.n_envs; env += gridDim.x) {
        const size_t r_env = (size_t)env * n;
        const int64_t wofs = blob_offset<kMulti>(A, env);                                  // this env's policy blob
        __syncthreads();                                       // the previous env's operands are dead
        // ---- keys: E rows -> fp16 hi / lo ----
        // (unconditional loads from a clamped row, zeroed afterwards: predicated loads are not batched by the compiler)
#pragma unroll 4
        for (int e = tid; e < NK * 16; e += THREADS) {
            const int j = e >> 4, c = (e & 15) << 2;
            float4 v = __ldcg(reinterpret_cast<const float4 *>(A.scr_e + (r_env + min(j, n - 1)) * 64 + c));
            if (j >= n) v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            uint32_t h0, l0, h1, l1;
            split2(v.x, v.y, h0, l0);
            split2(v.z, v.w, h1, l1);
            *reinterpret_cast<uint2 *>(Eh + j * kEhPitch + c) = make_uint2(h0, h1);
            *reinterpret_cast<uint2 *>(El + j * kEhPitch + c) = make_uint2(l0, l1);
        }
        for (int l = 0; l < L; ++l) {
            if (l) __syncthreads();                            // every warp wrote its H_l Wg_l rows and is done with the old operands
            // ---- values: H_l Wg_l rows -> transposed fp16 hi / lo [col][key] ----
#pragma unroll 4
            for (int e = tid; e < NK * 16; e += THREADS) {
                const int j = e % NK, c = (e / NK) << 2;       // consecutive threads take consecutive keys: neighbouring halves
                float4 v = __ldcg(reinterpret_cast<const float4 *>(A.scr_hw + (r_env + min(j, n - 1)) * 64 + c));
                if (j >= n) v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const __half h = __float2half_rn(vv[q]);
                    Vh[(c + q) * HWP + j] = h;
                    Vl[(c + q) * HWP + j] = __float2half_rn(vv[q] - __half2float(h));
                }
            }
            // ---- Wg_{l+1} (k-major [k][c] in the blob) -> transposed fp16 hi / lo [c][k] ----
            if (l + 1 < L) {
                const float *wg = A.weights + wofs + o.gcn_w + (size_t)(l + 1) * kE * kE;
#pragma unroll 4
                for (int e = tid; e < kE * kE; e += THREADS) {
                    const int k = e >> 6, c = e & 63;
                    const float v = __ldg(wg + e);
                    const __half h = __float2half_rn(v);
                    Wh[c * kWgPitch + k] = h;
                    Wl[c * kWgPitch + k] = __float2half_rn(v - __half2float(h));
                }
            }
            __syncthreads();
            const float *bias = A.weights + wofs + o.gcn_b + l * kE;
            for (int strip = warp; strip < n_strips; strip += WARPS) {
                const int i0 = strip << 4;                     // first query row of the strip; this lane owns rows i0+g, i0+g+8
                __syncwarp();
                // ---- query rows (fp16 hi / lo) and neighbour mask words -> the warp's slice ----
                // (all 8 + 4 loads of the strip are issued before the first store: one L2 round trip per strip)
                {
                    float4 qv[8];
                    uint32_t mv[4];
#pragma unroll
                    for (int it = 0; it < 8; ++it) {
                        const int e = lane + 32 * it, r = e >> 4, c = (e & 15) << 2;
                        qv[it] = __ldcg(reinterpret_cast<const float4 *>(A.scr_q + (r_env + min(i0 + r, n - 1)) * 64 + c));
                    }
#pragma unroll
                    for (int it = 0; it < 4; ++it) {
                        const int e = lane + 32 * it, r = e >> 3, w = e & 7;
                        const size_t row = r_env + min(i0 + r, n - 1);
                        const int wc = min(w, W - 1);
                        const uint32_t ma = A.adj_bits ? __ldg(A.adj_bits + row * W + wc) : 0xFFFFFFFFu;
                        const uint32_t mc = A.chan_bits ? __ldg(A.chan_bits + (((size_t)env * L + l) * n + min(i0 + r, n - 1)) * W + wc) : 0xFFFFFFFFu;
                        mv[it] = (i0 + r < n && w < W) ? (ma & mc) : 0u;
                    }
#pragma unroll
                    for (int it = 0; it < 8; ++it) {
                        const int e = lane + 32 * it, r = e >> 4, c = (e & 15) << 2;
                        if (i0 + r >= n) qv[it] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                        uint32_t h0, l0, h1, l1;
                        split2(qv[it].x, qv[it].y, h0, l0);
                        split2(qv[it].z, qv[it].w, h1, l1);
                        *reinterpret_cast<uint2 *>(Qh + r * kQhPitch + c) = make_uint2(h0, h1);
                        *reinterpret_cast<uint2 *>(Ql + r * kQhPitch + c) = make_uint2(l0, l1);
                    }
#pragma unroll
                    for (int it = 0; it < 4; ++it) Mw[lane + 32 * it] = mv[it];
                }
                __syncwarp();
                const bool v0 = i0 + g < n, v1 = i0 + g + 8 < n;
                StripState st = {-1e30f, -1e30f, -1e30f, -1e30f, 0.0f, 0.0f, 0.0f, 0.0f};
                float oacc[8][4];
#pragma unroll
                for (int ot = 0; ot < 8; ++ot) oacc[ot][0] = oacc[ot][1] = oacc[ot][2] = oacc[ot][3] = 0.0f;
#pragma unroll 1
                for (int kb = 0; kb < NFULL; ++kb) attn_block<8>(st, oacc, Qh, Ql, Eh, El, Vh, Vl, HWP, Mw, 8 * kb, n, g, t);
                if (TAIL) attn_block<TAIL ? TAIL : 2>(st, oacc, Qh, Ql, Eh, El, Vh, Vl, HWP, Mw, 8 * NFULL, n, g, t);
                const float z0 = quad_sum(st.z0), z1 = quad_sum(st.z1);
                // 1e-12 z 2^(m - q) = z 2^(m - q + log2(1e-12)); no masked-in key at all: q = -1e30, the term is inf, den = 0
                const float den0 = 1.0f / fmaf(z0, ex2_fast(st.m0 - st.q0 + kLog2Eps), quad_sum(st.d0));
                const float den1 = 1.0f / fmaf(z1, ex2_fast(st.m1 - st.q1 + kLog2Eps), quad_sum(st.d1));
                // ---- the UNMASKED softmax (comm_base_net.py:93), when recorded: a second walk with the final m and z ----
                if (l == 0 && A.attention) {
                    const float is0 = 1.0f / z0, is1 = 1.0f / z1;
                    float *att0 = A.attention + (r_env + i0 + g) * n, *att1 = A.attention + (r_env + i0 + g + 8) * n;
#pragma unroll 1
                    for (int kb = 0; kb < NFULL; ++kb) attn_record_block<8>(att0, att1, v0, v1, st, is0, is1, Qh, Ql, Eh, El, 8 * kb, n, g, t);
                    if (TAIL) attn_record_block<TAIL ? TAIL : 2>(att0, att1, v0, v1, st, is0, is1, Qh, Ql, Eh, El, 8 * NFULL, n, g, t);
                }
                // ---- H_{l+1} = tanh(out / (sum + 1e-12) + b): rows g / g + 8, columns 8 ot + 2t, + 1 ----
#pragma unroll
                for (int ot = 0; ot < 8; ++ot) {
                    const float2 b2 = __ldg(reinterpret_cast<const float2 *>(bias + 8 * ot + 2 * t));
                    oacc[ot][0] = tanh_fast(fmaf(oacc[ot][0], den0, b2.x));
                    oacc[ot][1] = tanh_fast(fmaf(oacc[ot][1], den0, b2.y));
                    oacc[ot][2] = tanh_fast(fmaf(oacc[ot][2], den1, b2.x));
                    oacc[ot][3] = tanh_fast(fmaf(oacc[ot][3], den1, b2.y));
                }
                if (l + 1 < L) {
                    // ---- next layer's value rows: H_{l+1} Wg_{l+1}, the H fragments again being the A operand ----
                    float hacc[8][4];
#pragma unroll
                    for (int ot = 0; ot < 8; ++ot) hacc[ot][0] = hacc[ot][1] = hacc[ot][2] = hacc[ot][3] = 0.0f;
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {
                        uint32_t ah[4], al[4];
                        split2(oacc[2 * ks][0], oacc[2 * ks][1], ah[0], al[0]);
                        split2(oacc[2 * ks][2], oacc[2 * ks][3], ah[1], al[1]);
                        split2(oacc[2 * ks + 1][0], oacc[2 * ks + 1][1], ah[2], al[2]);
                        split2(oacc[2 * ks + 1][2], oacc[2 * ks + 1][3], ah[3], al[3]);
                        const int k0 = 16 * ks + 2 * t;
#pragma unroll
                        for (int o0 = 0; o0 < 8; o0 += 4) {
                            uint32_t bh[4][2], bl[4][2];
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                const __half *wh = Wh + (8 * (o0 + u) + g) * kWgPitch + k0, *wl = Wl + (8 * (o0 + u) + g) * kWgPitch + k0;
                                bh[u][0] = *reinterpret_cast<const uint32_t *>(wh); bh[u][1] = *reinterpret_cast<const uint32_t *>(wh + 8);
                                bl[u][0] = *reinterpret_cast<const uint32_t *>(wl); bl[u][1] = *reinterpret_cast<const uint32_t *>(wl + 8);
                            }
#pragma unroll
                            for (int u = 0; u < 4; ++u) mma16816(hacc[o0 + u], ah, bh[u][0], bh[u][1]);
#pragma unroll
                            for (int u = 0; u < 4; ++u) mma16816(hacc[o0 + u], ah, bl[u][0], bl[u][1]);
#pragma unroll
                            for (int u = 0; u < 4; ++u) mma16816(hacc[o0 + u], al, bh[u][0], bh[u][1]);
                        }
                    }
#pragma unroll
                    for (int ot = 0; ot < 8; ++ot) {
                        if (v0) *reinterpret_cast<float2 *>(A.scr_hw + (r_env + i0 + g) * 64 + 8 * ot + 2 * t) = make_float2(hacc[ot][0], hacc[ot][1]);
                        if (v1) *reinterpret_cast<float2 *>(A.scr_hw + (r_env + i0 + g + 8) * 64 + 8 * ot + 2 * t) = make_float2(hacc[ot][2], hacc[ot][3]);
                    }
                } else {
                    // ---- X = E + H_L (comm_base_net.py:105-106), written over the strip's query rows ----
#pragma unroll
                    for (int ot = 0; ot < 8; ++ot) {
                        const int c = 8 * ot + 2 * t;
                        if (v0) {
                            float2 x = make_float2(oacc[ot][0], oacc[ot][1]);
                            if (A.d.residual) {            // E = hi + lo from the key operand (|error| <= 3e-8)
                                const float2 eh = __half22float2(*reinterpret_cast<const __half2 *>(Eh + (i0 + g) * kEhPitch + c));
                                const float2 el = __half22float2(*reinterpret_cast<const __half2 *>(El + (i0 + g) * kEhPitch + c));
                                x.x += eh.x + el.x; x.y += eh.y + el.y;
                            }
                            *reinterpret_cast<float2 *>(A.scr_q + (r_env + i0 + g) * 64 + c) = x;
                        }
                        if (v1) {
                            float2 x = make_float2(oacc[ot][2], oacc[ot][3]);
                            if (A.d.residual) {
                                const float2 eh = __half22float2(*reinterpret_cast<const __half2 *>(Eh + (i0 + g + 8) * kEhPitch + c));
                                const float2 el = __half22float2(*reinterpret_cast<const __half2 *>(El + (i0 + g + 8) * kEhPitch + c));
                                x.x += eh.x + el.x; x.y += eh.y + el.y;
                            }
                            *reinterpret_cast<float2 *>(A.scr_q + (r_env + i0 + g + 8) * 64 + c) = x;
                        }
                    }
                }
            }
        }
    }
}

template <int NS, bool kMulti>
static int launch_attn_mma_t(const AttnMmaArgsOf<kMulti> &A, cudaStream_t stream)
{
    constexpr int NK = 16 * NS;
    constexpr size_t base = (size_t)(2 * NK * kEhPitch + 2 * 64 * (NK + 8) + 2 * 64 * kWgPitch) * sizeof(__half);
    constexpr size_t per_warp = (size_t)2 * 16 * kQhPitch * sizeof(__half) + (size_t)16 * 8 * sizeof(uint32_t);
    constexpr int WARPS = base + 16 * per_warp <= 227 * 1024 ? 16 : 8;
    constexpr size_t smem = base + WARPS * per_warp;
    static thread_local struct { int dev; int slots; } cache = {-1, 0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return set_cuda_error(cudaGetLastError(), CM_ENODEVICE);
    if (cache.dev != dev) {
        int sms = 0, ctas = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return set_cuda_error(cudaGetLastError(), CM_ECUDA);
        cudaError_t e = cudaFuncSetAttribute(policy_attn_mma_kernel<NS, WARPS, kMulti>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return set_cuda_error(e, CM_ECUDA);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas, policy_attn_mma_kernel<NS, WARPS, kMulti>, WARPS * 32, smem) != cudaSuccess)
            return set_cuda_error(cudaGetLastError(), CM_ECUDA);
        cache.dev = dev;
        cache.slots = sms * (ctas < 1 ? 1 : ctas);
    }
    const int grid = (int)(A.n_envs < cache.slots ? A.n_envs : cache.slots);
    policy_attn_mma_kernel<NS, WARPS, kMulti><<<grid, WARPS * 32, smem, stream>>>(A);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? CM_OK : set_cuda_error(e, CM_ECUDA);
}

template <bool kMulti>
static int launch_attn_mma_n(int n, const AttnMmaArgsOf<kMulti> &A, cudaStream_t stream)
{
    switch ((n + 15) / 16) {
    case 5: return launch_attn_mma_t<5, kMulti>(A, stream);
    case 6: return launch_attn_mma_t<6, kMulti>(A, stream);
    case 7: return launch_attn_mma_t<7, kMulti>(A, stream);
    case 8: return launch_attn_mma_t<8, kMulti>(A, stream);
    case 9: return launch_attn_mma_t<9, kMulti>(A, stream);
    case 10: return launch_attn_mma_t<10, kMulti>(A, stream);
    case 11: return launch_attn_mma_t<11, kMulti>(A, stream);
    case 12: return launch_attn_mma_t<12, kMulti>(A, stream);
    case 13: return launch_attn_mma_t<13, kMulti>(A, stream);
    case 14: return launch_attn_mma_t<14, kMulti>(A, stream);
    case 15: return launch_attn_mma_t<15, kMulti>(A, stream);
    case 16: return launch_attn_mma_t<16, kMulti>(A, stream);
    }
    return CM_EUNSUPPORTED;
}

int launch_policy_attn_mma(const cm_policy_desc *desc, const cm_policy_io *io, const float *scr_e, float *scr_q, float *scr_hw,
                           cudaStream_t stream)
{
    AttnMmaSetArgs A;
    A.d = *desc;
    A.weights = io->weights;
    A.adj_bits = io->adj_bits;
    A.chan_bits = io->chan_bits;
    A.attention = io->attention;
    A.scr_e = scr_e; A.scr_q = scr_q; A.scr_hw = scr_hw;
    A.n_envs = io->n_envs;
    if (io->n_policies <= 1) return launch_attn_mma_n<false>(desc->n_agents, A, stream);
    A.envs_per_policy = io->envs_per_policy;
    A.weights_stride = io->weights_stride;
    return launch_attn_mma_n<true>(desc->n_agents, A, stream);
}

int launch_policy_tc_encode(const cm_policy_desc *desc, const cm_policy_io *io, float *scr_e, float *scr_q, float *scr_hw, cudaStream_t stream);
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
    rc = launch_policy_attn_mma(desc, io, scr_e, scr_q, scr_hw, stream);
    if (rc) return rc;
    if (!io->probs && !io->actions && !io->logits) return CM_OK;
    return launch_policy_tc_head(desc, io, scr_q, stream);
}

}  // namespace cm
