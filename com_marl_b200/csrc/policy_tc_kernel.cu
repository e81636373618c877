// policy_tc_kernel.cu — fused CommCategoricalMLPPolicy forward (+ action sampling) on the 5th-generation tensor cores (tcgen05).
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
// Machine mapping: a CTA of 512 threads owns a tile of 128 agent rows (whole environments, n <= 64); TWO such CTAs are
// resident per SM (256 tensor-memory columns and ~103 KB of shared memory each), so that one tile's epilogue
// (CUDA cores) runs while the other tile's products (tensor cores) and weight copies (TMA engine) are in flight.
//   * every row-wise dense layer (encoder, attention query, H_l Wg_l, the categorical head) is a series of
//     tcgen05.mma.kind::f16 (fp16 operands, fp32 accumulators in tensor memory).  fp32-level accuracy is kept by
//     error compensation: x = x_hi + 2^-12 x_lo with x_hi = fp16(x), x_lo = fp16((x - x_hi) * 4096);
//     A_hi x [B_hi ; B_lo] (B stacked along N) gives hi*hi and hi*lo in two accumulators with one series of K/16
//     instructions, A_lo x B_hi adds the other cross term, the epilogue forms acc0 + 2^-12 acc1 (dropped term:
//     2^-24).  Measured error of one product 1-3e-7 of scale, i.e. fp32 level.  Weights are pre-split, stacked and
//     pre-arranged in the canonical K-major core-matrix layout by cm_policy_tc_prepare(), so that a product's
//     B operand is ONE bulk async copy (TMA engine, mbarrier completion) issued one to two products ahead;
//   * the per-environment pieces (n x n scores, softmax, masked renormalisation, aggregation over
//     neighbours) exactly — not as padded tile products — on the CUDA cores.  Keys (E) and values (H_l Wg_l) share
//     ONE k-major fp32 buffer in shared memory; everything that is private to a row — the query, the attention
//     row, the residual copy of E — stays in TENSOR MEMORY: the query is read straight from its accumulator by
//     all four warps of the row's lane quadrant, the attention row and E are parked in dead accumulator columns
//     with tcgen05.st and read back with tcgen05.ld.
//   * teams of 17 .. 64 agents run the n x n part on the tensor cores too (kVec = 0): an env occupies a SLOT of 32 or 64 tile
//     rows; scores = Q E^T as one 128 x 128 x 64 product over the whole tile (B operand = the E operand already in shared
//     memory; the cross-env blocks are computed and ignored) into ONE accumulator block — the cross terms first, the high-order
//     product on top through tcgen05.mma's scale-input-d form, D = A B + D 2^-12 —, softmax per row from tensor memory, and per layer the aggregation
//     TRANSPOSED per env:  out_e^T [64 x S] = (H_l Wg_l)_e^T [64 x S keys] * A_e^T [S keys x S rows]  — an M = 64 product whose
//     A operand is the value rows as written (MN-major) and whose B operand is the compact masked attention rows (K-major),
//     so nothing is padded to the tile's 128 keys; the result comes back to the row-per-thread mapping through a swizzled fp32
//     buffer.  Smaller teams keep the exact CUDA-core loops (a slot would waste most of the tile).
// TMEM lane = tile row = thread (row = 32 * (warp % 4) + lane); the four warps that share a lane quadrant
// split the accumulator columns.  Epilogues read TMEM with tcgen05.ld, apply bias + tanh, and write the next
// A operand (hi / lo) straight into the canonical layout.
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

#include "commarl_b200.h"
#include "common.cuh"
#include "policy_layout.cuh"
#include "tc_common.cuh"

#ifndef CM_TC_DEBUG
#define CM_TC_DEBUG 0   // timing experiments only: 1 skip MMAs, 2 skip tanh, 4 skip attention loops, 8 skip weight copies
#endif

namespace cm {

using namespace tc;

static constexpr int kTcRows = 128;
static constexpr int kTcThreads = 512;
static constexpr int kActBytes = 32768;                     // A operand hi | lo (128 x 64 fp16 each)
static constexpr int kSlotBytes = 16384, kWBytes = 2 * kSlotBytes;   // weight ring: 2 slots
static constexpr int kTPitch = 128;                         // floats per k-major row of the key / value buffer
static constexpr uint32_t kTmemCols = 256;                  // two accumulator blocks of 128 columns
static constexpr uint32_t kR0 = 0, kR1 = 128;               // accumulator blocks (a product's D block is 2N <= 128 columns)
static constexpr uint32_t kColM = kR0, kColE = kR0 + 64;    // scratch during the graph convolutions: attention row, residual E

struct TcArgs {
    cm_policy_desc d;
    cm_policy_io io;
    TcPlan plan;
    int envs_per_tile;
    int slot;                    // Comm-DP: tile rows per env — n (dense packing, CUDA-core attention) or 32 / 64 (tensor-core attention)
    int64_t n_tiles;
    int mode;                    // kTcModeComm / Dec / Enc / Head
    int in_dim;                  // width of the input rows (obs_dim; 64 in head mode: the rows are X = E + H_L)
    float *scr_e, *scr_q, *scr_hw;   // encoder mode: row-major [rows][64] outputs E, Q = E Wq, H_0 Wg_0 (large-team pipeline)
    int tiles_per_policy;        // several policies in one launch: tiles of each env block
};

// fp16 split of one value: hi = fp16(x), lo = fp16((x - hi) * 4096)
__device__ __forceinline__ void split16(float x, __half &hi, __half &lo)
{
    hi = __float2half_rn(x);
    lo = __float2half_rn((x - __half2float(hi)) * 4096.0f);
}
// c_i + a_i b for the two fp16 halves a_0, a_1 of a2 in fp32: fma.rn.f32.f16, ONE instruction per value (SASS FHFMA) where
// the remainder x - hi otherwise takes a half -> float conversion and a subtraction.  The product of two fp16 values is exact
// in fp32, so x - hi (exact in fp32) comes out exactly.
static constexpr uint16_t kHalfM1 = 0xBC00u, kHalf4096 = 0x6C00u, kHalfM4096 = 0xEC00u;    // -1, 4096, -4096 as fp16
__device__ __forceinline__ void fma_f32_f16x2(uint32_t a2, uint16_t b, float c0, float c1, float &d0, float &d1)
{
    asm("{.reg .f16 a0, a1;\n\tmov.b32 {a0, a1}, %2;\n\tfma.rn.f32.f16 %0, a0, %5, %3;\n\tfma.rn.f32.f16 %1, a1, %5, %4;\n\t}"
        : "=f"(d0), "=f"(d1) : "r"(a2), "f"(c0), "f"(c1), "h"(b));
}
__device__ __forceinline__ uint32_t pack_half2(float x0, float x1)
{
    const __half2 h = __floats2half2_rn(x0, x1);
    return *reinterpret_cast<const uint32_t *>(&h);
}
// split16 for two values at once: ONE packed conversion per pair (the scalar form costs a conversion and a byte permute
// per value — the conversions of the activations are the largest instruction class of the epilogues)
__device__ __forceinline__ void split16x2(float x0, float x1, uint32_t &hi, uint32_t &lo)
{
    float d0, d1;
    hi = pack_half2(x0, x1);
    fma_f32_f16x2(hi, kHalfM1, x0, x1, d0, d1);                      // x - hi
    lo = pack_half2(d0 * 4096.0f, d1 * 4096.0f);
}
// The same split of x = x' 2^-12 from the PRE-SCALED x' = 4096 x that the tanh epilogues emit (|x| <= 2): h' = fp16(x') is
// 4096 fp16(x) and 2^-12 h' = fp16(x) exactly wherever fp16(x) is normal; lo = fp16(x' - 4096 hi) with the remainder exact,
// so the operand is the one split16x2 makes, in 5 instructions per pair instead of 6.  (Below 2^-14, where fp16(x) is
// subnormal, hi may round differently from fp16(x) at a tie; lo is taken against the hi actually stored, so hi + 2^-12 lo
// still represents x to the same precision.)
__device__ __forceinline__ void split16x2_pre(float x0, float x1, uint32_t &hi, uint32_t &lo)
{
    float d0, d1;
    asm("mul.rn.f16x2 %0, %1, %2;" : "=r"(hi) : "r"(pack_half2(x0, x1)), "r"(0x0C000C00u));   // * 2^-12
    fma_f32_f16x2(hi, kHalfM4096, x0, x1, d0, d1);                   // x' - 4096 hi = 4096 (x - hi)
    lo = pack_half2(d0, d1);
}
static constexpr float kActScale = 4096.0f;                          // x' = kActScale x: the form split16x2_pre takes
// back from 8 columns of an A operand (hi, lo) to the pre-scaled x' = 4096 hi + lo
__device__ __forceinline__ void unpack_act_pre(const uint4 &hq, const uint4 &lq, float *x)
{
    const uint32_t *hw = &hq.x;
    const __half2 *ll = reinterpret_cast<const __half2 *>(&lq);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 lf = __half22float2(ll[i]);
        fma_f32_f16x2(hw[i], kHalf4096, lf.x, lf.y, x[2 * i], x[2 * i + 1]);
    }
}

// write CW (8 or 16) consecutive columns, starting at local column c0 (a multiple of 8) of a Kp-wide panel, of row `row`
// as the next A operand: hi block, then the lo block 128 * Kp halves further.  kPre: v holds kActScale x (split16x2_pre)
template <int CW, bool kPre = false>
__device__ __forceinline__ void write_act(unsigned char *act, int Kp, int row, int c0, const float (&v)[CW])
{
    const uint32_t lo_off = (uint32_t)kTcRows * Kp * 2;
#pragma unroll
    for (int g = 0; g < CW; g += 8) {
        uint4 h, l;
        if constexpr (kPre) {
            split16x2_pre(v[g + 0], v[g + 1], h.x, l.x);
            split16x2_pre(v[g + 2], v[g + 3], h.y, l.y);
            split16x2_pre(v[g + 4], v[g + 5], h.z, l.z);
            split16x2_pre(v[g + 6], v[g + 7], h.w, l.w);
        } else {
            split16x2(v[g + 0], v[g + 1], h.x, l.x);
            split16x2(v[g + 2], v[g + 3], h.y, l.y);
            split16x2(v[g + 4], v[g + 5], h.z, l.z);
            split16x2(v[g + 6], v[g + 7], h.w, l.w);
        }
        const uint32_t off = canon_off16(row, c0 + g, Kp);
        *reinterpret_cast<uint4 *>(act + off) = h;
        *reinterpret_cast<uint4 *>(act + lo_off + off) = l;
    }
}

// Operands of the transposed aggregation product.  Single accumulator, so the remainder is NOT rescaled: x' = s x,
// hi = fp16(x'), lo = fp16(x' - hi); the power-of-two scale s keeps lo out of the fp16 subnormals (values: s = 2^6, attention
// weights: s = 2^10; the product is rescaled by 2^-16 in the epilogue).  Same chunked layout as write_act.
static constexpr float kVScale = 64.0f, kPScale = 1024.0f, kPVUnscale = 1.0f / 65536.0f;
__device__ __forceinline__ void split_unscaled_x2(float x0, float x1, uint32_t &hi, uint32_t &lo)
{
    float d0, d1;
    hi = pack_half2(x0, x1);
    fma_f32_f16x2(hi, kHalfM1, x0, x1, d0, d1);
    lo = pack_half2(d0, d1);
}
template <int CW>
__device__ __forceinline__ void write_unscaled(unsigned char *buf, int Kp, uint32_t lo_off, int row, int c0, const float (&v)[CW], float scale)
{
#pragma unroll
    for (int g = 0; g < CW; g += 8) {
        uint4 h, l;
        split_unscaled_x2(v[g + 0] * scale, v[g + 1] * scale, h.x, l.x);
        split_unscaled_x2(v[g + 2] * scale, v[g + 3] * scale, h.y, l.y);
        split_unscaled_x2(v[g + 4] * scale, v[g + 5] * scale, h.z, l.z);
        split_unscaled_x2(v[g + 6] * scale, v[g + 7] * scale, h.w, l.w);
        const uint32_t off = canon_off16(row, c0 + g, Kp);
        *reinterpret_cast<uint4 *>(buf + off) = h;
        *reinterpret_cast<uint4 *>(buf + lo_off + off) = l;
    }
}

// tanh through ex2.approx / rcp.approx on a PRE-SCALED argument a = 2 log2(e) x:  tanh(x) = 1 - 2 / (2^a + 1).
// |error| <= ~3e-7 absolute (two units of fp32 rounding at 1.0), an order of magnitude below the tolerance; the scale
// is folded into the accumulator read-out (one FFMA per element does "combine hi/lo accumulators, add bias, scale"),
// and the shared-memory bias table holds 2 log2(e) * bias.  Saturates correctly: 2^a = inf -> 1, 2^a = 0 -> -1.
static constexpr float kTanhScale = 2.8853900817779268f;            // 2 log2(e)
static constexpr float kTanhScaleLo = 2.8853900817779268f / 4096.0f;
// `out` (a power of two) scales the result for free in the last FMA: out = kActScale gives the pre-scaled form of write_act
__device__ __forceinline__ float tanh_scaled(float a, float out = 1.0f)
{
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(a));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
    return fmaf(-2.0f * out, r, out);
}
// Four tanh's with ONE reciprocal: 1/A = B C D / (A B C D) ...  The special-function unit (16 lanes per clock per SM) is what
// bounds the dense epilogues locally — two MUFU per tanh occupy it for ~60 % of an epilogue — so the four reciprocals of a
// group are replaced by one plus nine multiplications on the FMA pipe: 1.25 MUFU per tanh.  Arguments are clamped at 30
// (tanh = 1 - 2^-29 rounds to 1 in fp32), so the product of four (2^a + 1) stays below 2^121.  |error| <= ~4e-7 absolute.
#ifndef CM_TANH_SHARED_RCP
#define CM_TANH_SHARED_RCP 1
#endif
__device__ __forceinline__ void tanh4_scaled(float &a0, float &a1, float &a2, float &a3, float out = 1.0f)
{
#if !CM_TANH_SHARED_RCP
    a0 = tanh_scaled(a0, out); a1 = tanh_scaled(a1, out); a2 = tanh_scaled(a2, out); a3 = tanh_scaled(a3, out);
    return;
#endif
    float e0, e1, e2, e3, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(fminf(a0, 30.0f)));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(fminf(a1, 30.0f)));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e2) : "f"(fminf(a2, 30.0f)));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e3) : "f"(fminf(a3, 30.0f)));
    const float A = e0 + 1.0f, B = e1 + 1.0f, C = e2 + 1.0f, D = e3 + 1.0f;
    const float ab = A * B, cd = C * D;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(ab * cd));
    const float rab = r * ab, rcd = r * cd;          // 1 / (C D), 1 / (A B)
    a0 = fmaf(-2.0f * out, rcd * B, out);
    a1 = fmaf(-2.0f * out, rcd * A, out);
    a2 = fmaf(-2.0f * out, rab * D, out);
    a3 = fmaf(-2.0f * out, rab * C, out);
}
// out * tanh(acc0 + 2^-12 acc1 + bias) for 4 consecutive columns, bias4 = 2 log2(e) * bias from the shared-memory table
__device__ __forceinline__ void tanh4(float *v, const float *w, const float4 b4, float out = 1.0f)
{
    v[0] = fmaf(v[0], kTanhScale, fmaf(w[0], kTanhScaleLo, b4.x));
    v[1] = fmaf(v[1], kTanhScale, fmaf(w[1], kTanhScaleLo, b4.y));
    v[2] = fmaf(v[2], kTanhScale, fmaf(w[2], kTanhScaleLo, b4.z));
    v[3] = fmaf(v[3], kTanhScale, fmaf(w[3], kTanhScaleLo, b4.w));
    tanh4_scaled(v[0], v[1], v[2], v[3], out);
}

// one converged warp: D[:, 0:N] (+)= A_hi B_hi^T, D[:, N:2N] (+)= A_hi B_lo^T + A_lo B_hi^T.  All lanes run the code
// (descriptors stay in uniform registers); the instructions are predicated on the leader lane.
// lo_from: first K slice whose A_lo is not identically zero (packed observations: only the scalar columns have a low-order part)
__device__ __forceinline__ void issue_layer(uint32_t d_tmem, const unsigned char *act, const unsigned char *wblk, int N, int Kp,
                                            uint32_t accumulate, uint32_t leader, int lo_from = 0)
{
    if (CM_TC_DEBUG & 1) return;
    const uint32_t a_hi = smem_u32(act), a_lo = a_hi + (uint32_t)kTcRows * Kp * 2, b = smem_u32(wblk);
    const int nk = Kp >> 4;                     // 1 .. 4 instructions of K = 16; the next slice starts 256 bytes (16 >> 4) further
    const uint64_t db = make_smem_desc16(b, Kp, 0);
    {   // A_hi x [B_hi ; B_lo]  (N' = 2N)
        const uint32_t idesc = make_idesc_f16(kTcRows, 2 * N);
        const uint64_t da = make_smem_desc16(a_hi, Kp, 0);
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (j < nk) mma_f16_pred(d_tmem, da + 16 * j, db + 16 * j, idesc, j ? 1u : accumulate, leader);
    }
    {   // A_lo x B_hi  (N' = N) into the cross-term accumulator
        const uint32_t idesc = make_idesc_f16(kTcRows, N);
        const uint64_t da = make_smem_desc16(a_lo, Kp, 0);
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (j < nk && j >= lo_from) mma_f16_pred(d_tmem + (uint32_t)N, da + 16 * j, db + 16 * j, idesc, 1u, leader);
    }
}

// scores of the whole tile into ONE accumulator block of 128 columns: D = Q_hi E_lo^T + Q_lo E_hi^T (remainders scaled by
// 2^12), then D = D 2^-12 + Q_hi E_hi^T (mma_f16_scale12_pred on the first K slice) — the other 128 columns of the CTA's tensor
// memory keep H_0 Wg_0, so that product shares a phase with Q = E Wa.  qbuf / ebuf: [128][64] fp16 hi, lo 16 KB further.
__device__ __forceinline__ void issue_scores(uint32_t d_tmem, const unsigned char *qbuf, const unsigned char *ebuf, uint32_t leader)
{
    if (CM_TC_DEBUG & 1) return;
    const uint32_t lo = (uint32_t)kTcRows * 64 * 2;
    const uint32_t idesc = make_idesc_f16(kTcRows, 128);
    const uint64_t q_hi = make_smem_desc16(smem_u32(qbuf), 64, 0), q_lo = make_smem_desc16(smem_u32(qbuf) + lo, 64, 0);
    const uint64_t e_hi = make_smem_desc16(smem_u32(ebuf), 64, 0), e_lo = make_smem_desc16(smem_u32(ebuf) + lo, 64, 0);
#pragma unroll
    for (int j = 0; j < 4; ++j) mma_f16_pred(d_tmem, q_hi + 16 * j, e_lo + 16 * j, idesc, j ? 1u : 0u, leader);
#pragma unroll
    for (int j = 0; j < 4; ++j) mma_f16_pred(d_tmem, q_lo + 16 * j, e_hi + 16 * j, idesc, 1u, leader);
    mma_f16_scale12_pred(d_tmem, q_hi, e_hi, idesc, leader);
#pragma unroll
    for (int j = 1; j < 4; ++j) mma_f16_pred(d_tmem, q_hi + 16 * j, e_hi + 16 * j, idesc, 1u, leader);
}

// raw accumulator read-out: acc0 -> v, acc1 -> w (the caller fuses the combination with bias and scale)
template <int CW>
__device__ __forceinline__ void ld_acc_raw(uint32_t blk, int N, int col, float (&v)[CW], float (&w)[CW])
{
#pragma unroll
    for (int c = 0; c < CW; c += 8) {
        tmem_ld8(blk + (uint32_t)(col + c), *reinterpret_cast<float(*)[8]>(&v[c]));
        tmem_ld8(blk + (uint32_t)(N + col + c), *reinterpret_cast<float(*)[8]>(&w[c]));
    }
    tmem_ld_wait();
}

// accumulator read-out: acc0 + 2^-12 acc1 for CW columns starting at column `col` of a product whose D block starts at
// TMEM address `blk` (lane quadrant included) and is 2N columns wide.  Warp-collective (tcgen05.ld is .sync.aligned).
template <int CW>
__device__ __forceinline__ void ld_acc(uint32_t blk, int N, int col, float (&v)[CW])
{
    float w[CW];
#pragma unroll
    for (int c = 0; c < CW; c += 8) {
        float t0[8], t1[8];
        tmem_ld8(blk + (uint32_t)(col + c), t0);
        tmem_ld8(blk + (uint32_t)(N + col + c), t1);
#pragma unroll
        for (int i = 0; i < 8; ++i) { v[c + i] = t0[i]; w[c + i] = t1[i]; }
    }
    tmem_ld_wait();
#pragma unroll
    for (int c = 0; c < CW; ++c) v[c] = fmaf(w[c], 1.0f / 4096.0f, v[c]);
}

// Exact per-environment attention row.  Thread (row, sub) owns the KT consecutive keys sub * KT .. of its env
// (4 * KT >= n); scores = Q[row] . E[key] with the query read from its accumulator block in tensor memory (16 columns
// at a time) and the keys from the k-major buffer.  The softmax needs ONE exchange between the four threads of a row:
// each publishes the maximum m_s and the sum l_s = sum exp(score - m_s) of its keys, after the barrier
// p = exp(score - m_s) * exp(m_s - M) / sum_s l_s exp(m_s - M).  Returns with every thread past the barrier (the
// query block and the keys are dead); the caller parks the probabilities sc[] in tensor memory.
template <int KT, int kVec>
__device__ __forceinline__ void scores_softmax(uint32_t lane_addr, const float *KV, float *red, float *attn_row, int row, int j0,
                                               int sub, int n, bool valid)
{
    const int k0 = sub * KT;
    const int nk = valid ? min(KT, n - k0) : 0;        // may be <= 0
    float sc[KT];
#pragma unroll
    for (int t = 0; t < KT; ++t) sc[t] = 0.0f;
    const float *er0 = KV + j0 + k0;
    for (int c = 0; c < 64; c += 16) {                 // warp-uniform trip count: the TMEM loads are collective
        float q[16];
        ld_acc<16>(lane_addr + kR0, 64, c, q);
        if (nk > 0 && !(CM_TC_DEBUG & 4)) {
            // the keys of a thread are consecutive floats of a k-major row: 128-bit / 64-bit shared-memory loads when the
            // team size keeps them aligned (the loop is bound by shared-memory instructions, not by the FMAs)
            if (KT >= 4 && kVec == 4) {
#pragma unroll
                for (int kk = 0; kk < 16; ++kk) {
                    const float4 *e4 = reinterpret_cast<const float4 *>(er0 + (c + kk) * kTPitch);
#pragma unroll
                    for (int t = 0; t < KT; t += 4)
                        if (t < nk) {
                            const float4 ev = e4[t >> 2];
                            sc[t] = fmaf(q[kk], ev.x, sc[t]);
                            sc[(t + 1) % KT] = fmaf(q[kk], ev.y, sc[(t + 1) % KT]);
                            sc[(t + 2) % KT] = fmaf(q[kk], ev.z, sc[(t + 2) % KT]);
                            sc[(t + 3) % KT] = fmaf(q[kk], ev.w, sc[(t + 3) % KT]);
                        }
                }
            } else if (KT >= 2 && kVec >= 2) {
#pragma unroll
                for (int kk = 0; kk < 16; ++kk) {
                    const float2 *e2 = reinterpret_cast<const float2 *>(er0 + (c + kk) * kTPitch);
#pragma unroll
                    for (int t = 0; t < KT; t += 2)
                        if (t < nk) {
                            const float2 ev = e2[t >> 1];
                            sc[t] = fmaf(q[kk], ev.x, sc[t]);
                            sc[(t + 1) % KT] = fmaf(q[kk], ev.y, sc[(t + 1) % KT]);
                        }
                }
            } else {
#pragma unroll
                for (int kk = 0; kk < 16; ++kk) {
                    const float *er = er0 + (c + kk) * kTPitch;
#pragma unroll
                    for (int t = 0; t < KT; ++t)
                        if (t < nk) sc[t] = fmaf(q[kk], er[t], sc[t]);
                }
            }
        }
    }
    float mx = -INFINITY;
#pragma unroll
    for (int t = 0; t < KT; ++t)
        if (t < nk) mx = fmaxf(mx, sc[t]);
    float sum = 0.0f;
#pragma unroll
    for (int t = 0; t < KT; ++t) {
        sc[t] = t < nk ? __expf(sc[t] - mx) : 0.0f;
        sum += sc[t];
    }
    red[sub * kTPitch + row] = mx;
    red[(4 + sub) * kTPitch + row] = sum;
    fence_before_thread_sync();
    __syncthreads();                      // every thread has read the query block and the keys
    fence_after_thread_sync();
    float gm = -INFINITY;
#pragma unroll
    for (int s = 0; s < 4; ++s) gm = fmaxf(gm, red[s * kTPitch + row]);
    float z = 0.0f;
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        const float ms = red[s * kTPitch + row];
        z += ms > -INFINITY ? red[(4 + s) * kTPitch + row] * __expf(ms - gm) : 0.0f;
    }
    const float scale = nk > 0 ? __expf(mx - gm) / z : 0.0f;
#pragma unroll
    for (int t = 0; t < KT; ++t) sc[t] *= scale;
    if (attn_row) {                       // unmasked softmax (agent_infos['attention_weights'])
#pragma unroll
        for (int t = 0; t < KT; ++t)
            if (t < nk) attn_row[k0 + t] = sc[t];
    }
    if constexpr (KT <= 8) tmem_st<KT>(lane_addr + kColM + (uint32_t)k0, sc);
    else {
        tmem_st<8>(lane_addr + kColM + (uint32_t)k0, sc);
        tmem_st<8>(lane_addr + kColM + (uint32_t)k0 + 8u, sc + 8);
    }
}

// Tensor-core attention: the scores of the whole tile are in tensor memory, columns [0, 128) (issue_scores: one accumulator
// block); the env of this row owns the key columns j0 .. j0 + n.  Thread (row, sub) takes the KT
// consecutive keys sub * KT ..; same exchange and same result placement as scores_softmax.
// e^x through ex2.approx.ftz (what __expf does, minus its denormal-range fix-up: results below 2^-126 flush to zero,
// which the sums here cannot tell from the exact value); exp_fast(-inf) = 0
__device__ __forceinline__ float exp_fast(float x)
{
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x * 1.4426950408889634f));
    return r;
}
template <int KT>
__device__ __forceinline__ void softmax_tc(uint32_t lane_addr, float *red, float *attn_row, int row, int j0, int sub, int n, bool valid)
{
    const int k0 = sub * KT;
    const int nk = valid ? max(0, min(KT, n - k0)) : 0;
    float sc[KT];
#pragma unroll
    for (int c = 0; c < KT; c += 8) tmem_ld8(lane_addr + (uint32_t)(j0 + k0 + c), *reinterpret_cast<float(*)[8]>(sc + c));
    tmem_ld_wait();
    // keys beyond the team (or every key of a padding row) score -inf once; everything below is branch-free:
    // exp_fast(-inf - m) = 0, and a thread without keys publishes max = -inf, sum = 0
    const uint32_t live = nk >= 32 ? 0xFFFFFFFFu : (1u << nk) - 1u;
    float mx = -INFINITY;
#pragma unroll
    for (int t = 0; t < KT; ++t) {
        sc[t] = (live & (1u << t)) ? sc[t] : -INFINITY;
        mx = fmaxf(mx, sc[t]);
    }
    const float mref = nk > 0 ? mx : 0.0f;             // (-inf) - (-inf) would be NaN
    float sum = 0.0f;
#pragma unroll
    for (int t = 0; t < KT; ++t) {
        sc[t] = exp_fast(sc[t] - mref);
        sum += sc[t];
    }
    red[sub * kTPitch + row] = mx;
    red[(4 + sub) * kTPitch + row] = sum;
    fence_before_thread_sync();
    __syncthreads();                      // every thread has read its scores
    fence_after_thread_sync();
    float ms[4];
#pragma unroll
    for (int s = 0; s < 4; ++s) ms[s] = red[s * kTPitch + row];
    const float gm = fmaxf(fmaxf(ms[0], ms[1]), fmaxf(ms[2], ms[3]));
    const float gref = nk > 0 ? gm : 0.0f;             // rows without keys: every maximum is -inf, the result is discarded
    float z = 0.0f;
#pragma unroll
    for (int s = 0; s < 4; ++s) z = fmaf(red[(4 + s) * kTPitch + row], exp_fast(ms[s] - gref), z);
    const float scale = nk > 0 ? __fdividef(exp_fast(mx - gm), z) : 0.0f;
#pragma unroll
    for (int t = 0; t < KT; ++t) sc[t] *= scale;
    if (attn_row) {                       // unmasked softmax (agent_infos['attention_weights'])
        if ((n & 3) == 0) {               // rows of n floats keep 16-byte alignment: whole 32-byte sectors per thread
#pragma unroll
            for (int t = 0; t < KT; t += 4)
                if (t < nk) *reinterpret_cast<float4 *>(attn_row + k0 + t) = make_float4(sc[t], sc[t + 1], sc[t + 2], sc[t + 3]);
        } else {
#pragma unroll
            for (int t = 0; t < KT; ++t)
                if (t < nk) attn_row[k0 + t] = sc[t];
        }
    }
    tmem_st<8>(lane_addr + kColM + (uint32_t)k0, sc);
    if constexpr (KT > 8) tmem_st<8>(lane_addr + kColM + (uint32_t)k0 + 8u, sc + 8);
}

// masked attention row of layer l -> B operand of the transposed aggregation (compact [128 rows][S keys], K-major), written
// as p 2^e kPScale with 2^e the power of two that brings the row's masked maximum to [1, 2): once the masks remove the keys
// that carry the attention mass, the remaining weights can be far below one, and without the rescaling their fp16 hi / lo
// split loses its relative precision (or underflows to zero) before the division by their small sum.  Leaves this
// thread's part of the row's masked sum (unscaled) in red rows 0..3 and returns 2^e in `pscale`.  Contains a CTA barrier.
template <int KT>
__device__ __forceinline__ void masked_p_operand(uint32_t lane_addr, unsigned char *pbuf, float *red, int S, int row, int sub, int n,
                                                  uint32_t m0, uint32_t m1, float &pscale)
{
    const int k0 = sub * KT;
    float p[KT];
    tmem_ld8(lane_addr + kColM + (uint32_t)k0, *reinterpret_cast<float(*)[8]>(p));
    if constexpr (KT > 8) tmem_ld8(lane_addr + kColM + (uint32_t)k0 + 8u, *reinterpret_cast<float(*)[8]>(p + 8));
    tmem_ld_wait();
    // the keys beyond the team are cleared in the mask word once (one bit test + select per key)
    const int left = n - k0;
    const uint32_t mbits = ((k0 < 32 ? m0 : m1) >> (k0 & 31)) & (left >= 32 ? 0xFFFFFFFFu : (left > 0 ? (1u << left) - 1u : 0u));
    float den = 0.0f, mx = 0.0f;
#pragma unroll
    for (int j = 0; j < KT; ++j) {
        p[j] = (mbits & (1u << j)) ? p[j] : 0.0f;
        den += p[j];
        mx = fmaxf(mx, p[j]);
    }
    red[sub * kTPitch + row] = den;
    red[(4 + sub) * kTPitch + row] = mx;
    __syncthreads();
    mx = fmaxf(fmaxf(red[4 * kTPitch + row], red[5 * kTPitch + row]), fmaxf(red[6 * kTPitch + row], red[7 * kTPitch + row]));
    // 2^(127 - exponent of mx); rows whose masked weights are all below 2^-107 (a masked sum that is nothing next to the
    // renormalisation's 1e-12) keep 2^107, so that 2^e kPScale stays finite
    pscale = mx > 0.0f ? __int_as_float((254 - max(__float_as_int(mx) >> 23, 20)) << 23) : 1.0f;
    write_unscaled<KT>(pbuf, S, (uint32_t)kTcRows * S * 2, row, k0, p, kPScale * pscale);
}

// bias offsets inside the shared-memory bias table
static constexpr int kBEnc1 = 0, kBEnc2 = 128, kBGcn = 192, kBH1 = 448, kBH2 = 576, kBH3 = 640, kBH4 = 672, kW4 = 680, kBiasFloats = 680 + kC3 * CM_ACTIONS;   // kW4: head_w4 [32][5] k-major

struct MmaOp { uint32_t dcol, acc, abuf; int lo_from; };   // accumulator block, accumulate flag, A operand buffer (0: ACT, 1: ACT2), first K slice of the A_lo pass

#ifdef CM_TC_TRACE
#define CM_TPK(slot) do { if (blockIdx.x == 0 && threadIdx.x == 0 && A.io.workspace) \
    reinterpret_cast<long long *>(A.io.workspace)[600 + (slot)] = clock64(); } while (0)
#define CM_TP(slot) do { if (blockIdx.x == 0 && threadIdx.x == 0 && io.workspace && tile == (int)blockIdx.x) \
    reinterpret_cast<long long *>(io.workspace)[600 + (slot)] = clock64(); } while (0)
#else
#define CM_TP(slot) do { } while (0)
#define CM_TPK(slot) do { } while (0)
#endif

// kVec: width (in floats) of the shared-memory loads of the attention loops — 4 when the team size is a multiple of 4,
// 2 when it is even, else 1 (the keys / values of an env start at a multiple of n floats).  One instantiation per width,
// so that small odd teams (n = 3) carry none of the vector code.  kVec = 0: the attention runs on the tensor cores (teams
// of 17 .. 64 agents, env slots of 32 / 64 rows) and the kernel carries none of the CUDA-core attention loops.
// kMode: kTcModeComm / Dec / Enc / Head as a template parameter, so that the Comm-DP kernel carries none of the other modes'
// code (the kernel is instruction-fetch sensitive: its SASS is several times the instruction cache).
// kMulti: several policies in one launch (io.n_policies > 1).  Tiles are counted per env block (A.tiles_per_policy each, the
// last one of a block may be partial), so a tile belongs to ONE policy: policy(t) = t / tiles_per_policy.  The weight stream
// prefetches across tile boundaries, so every block it requests is taken from the policy of the tile that will consume it;
// the bias table is reloaded when the CTA's next tile belongs to another policy, after the CTA barrier that ends the
// previous tile's last read of it.  A separate instantiation, so that the one-policy kernels keep their code.
template <int kVec, int kMode, bool kMulti = false>
__global__ void __launch_bounds__(kTcThreads, 2) policy_tc_kernel(const TcArgs A)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    CM_TPK(20);
#ifdef CM_TC_TRACE
    if (threadIdx.x == 0 && A.io.workspace) {
        unsigned long long gt; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt));
        reinterpret_cast<unsigned long long *>(A.io.workspace)[1024 + 2 * blockIdx.x] = gt;
    }
#endif
    unsigned char *ACT = smem;
    unsigned char *WB = smem + kActBytes;                                // weight ring: 2 slots of 16 KB
    float *KV = reinterpret_cast<float *>(smem + kActBytes + kWBytes);   // [64][128] E^T (keys), then (H_l Wg_l)^T (values)
    unsigned char *ACT2 = smem + kActBytes + kWBytes;                    // second A operand (aliases KV while it is idle)
    float *red = KV + 64 * kTPitch;                                      // [8][128] softmax max / sum exchange
    float *bias_s = red + 8 * kTPitch;                                   // [704]
    uint64_t *bars = reinterpret_cast<uint64_t *>(bias_s + kBiasFloats); // [0],[1] weight slot full, [2] MMAs done, [3] MMAs of a per-slot phase done, [4] MMAs of a two-product phase done
    uint32_t *tmem_s = reinterpret_cast<uint32_t *>(bars + 5);

    const cm_policy_desc &d = A.d;
    const cm_policy_io &io = A.io;
    const TcPlan &P = A.plan;
    const int n = d.n_agents, D = d.obs_dim, L = d.n_layers, W = (n + 31) >> 5;
    const Blob o = blob_layout(D, L);
    const float *__restrict__ wts = io.weights;
    const __half *tcw = reinterpret_cast<const __half *>(io.tc_weights);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int quad = warp & 3, sub = warp >> 2, row = quad * 32 + lane;

    if (warp == 0) tmem_alloc(tmem_s, kTmemCols);
    if (tid == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        mbar_init(&bars[2], 1);
        mbar_init(&bars[3], kVec == 0 ? (uint32_t)(kTcRows / A.slot) : 1u);      // one arrival per env slot (run_slots)
        mbar_init(&bars[4], 2);                                                  // one arrival per product of a two-product phase
        fence_mbar_init();
    }
    fence_before_thread_sync();
    __syncthreads();
    fence_after_thread_sync();
    const uint32_t tmem = *tmem_s;
    const uint32_t lane_addr = tmem + ((uint32_t)(quad * 32) << 16);
    uint32_t m_phase = 0, p_phase = 0;
    bool ok = true;

    // ---- weight stream: the stages of the plan are consumed in order, tile after tile; warp 0 keeps the
    // two ring slots full (a slot is refilled as soon as the product that read it has completed) ----
    const int n_tiles = (int)A.n_tiles, n_envs = (int)io.n_envs;
    const uint32_t my_tiles = (uint32_t)((n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x);
    const uint32_t total_blocks = my_tiles * (uint32_t)P.seq_len;
    uint32_t consumed = 0;                    // blocks consumed so far (uniform)
    uint32_t issued = 0, issued_si = 0;       // warp 0: blocks requested so far, and their stage index
    auto issue_loads = [&]() {          // warp 0, converged
        if (warp == 0) {
            while (issued < consumed + 2 && issued < total_blocks) {
                const TcStage &st = P.st[issued_si];
                const uint32_t bytes = (uint32_t)(2 * st.N * st.Kp * 2), slot = issued & 1u;
                if (elect_one()) {
                    if (CM_TC_DEBUG & 8) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&bars[slot])) : "memory"); }
                    else {
                        mbar_expect_tx(&bars[slot], bytes);
                        if constexpr (kMulti) {      // the policy of the tile this block belongs to: the CTA's (issued / seq_len)-th tile
                            const int tl = (int)blockIdx.x + (int)(issued / (uint32_t)P.seq_len) * (int)gridDim.x;
                            const __half *pw = tcw + (size_t)(tl / A.tiles_per_policy) * (size_t)io.tc_weights_stride * 2u;
                            bulk_g2s(WB + slot * (uint32_t)kSlotBytes, pw + st.w_off, bytes, &bars[slot]);
                        } else {
                            bulk_g2s(WB + slot * (uint32_t)kSlotBytes, tcw + st.w_off, bytes, &bars[slot]);
                        }
                    }
                }
                __syncwarp();
                ++issued;
                issued_si = (issued_si + 1 == (uint32_t)P.seq_len) ? 0u : issued_si + 1;
            }
        }
    };
    issue_loads();
    int si = 0;                               // stage index inside the current tile (uniform)
    // all threads: ACT is written -> warp 0 issues one product per op, each against the next weight block ->
    // everybody waits for their completion -> the freed ring slots are refilled
    auto run_mma = [&](int nops, MmaOp op0, MmaOp op1) {
#ifdef CM_TC_TRACE
        long long tr0 = clock64(), tr1, tr2 = 0, tr3, trw[2] = {0, 0};
#endif
        fence_proxy_async();
        fence_before_thread_sync();
        __syncthreads();
#ifdef CM_TC_TRACE
        tr1 = clock64();
#endif
        // A phase of two products is issued by TWO warps at once (warp i waits for weight block i and issues product i; both
        // commit on a barrier that expects two arrivals): the timeline of a tile showed 0.8 - 2.3 k cycles of issue per
        // two-product phase — one warp's instruction stream crawling through ~120 instructions while the co-resident tile's
        // epilogue owns the issue slots — against ~0.2 k of tensor latency behind the last instruction.
        // (two K panels of one product accumulate into the SAME block, in order: those stay with one warp)
        const bool par = nops == 2 && op0.dcol != op1.dcol;
        if (warp == 0 || (par && warp == 1)) {     // whole warp, converged: waits for the weights, the leader lane issues
            fence_after_thread_sync();
            const uint32_t leader = elect_one() ? 1u : 0u;
            for (int i = par ? warp : 0; i < (par ? warp + 1 : nops); ++i) {
                const uint32_t b = consumed + (uint32_t)i;
                ok = mbar_wait(&bars[b & 1u], (b >> 1) & 1u) && ok;
#ifdef CM_TC_TRACE
                trw[i & 1] = clock64();
#endif
                const TcStage &st = P.st[si + i];
                const MmaOp op = i ? op1 : op0;
                issue_layer(tmem + op.dcol, op.abuf ? ACT2 : ACT, WB + (b & 1u) * (uint32_t)kSlotBytes, st.N, st.Kp, op.acc, leader, op.lo_from);
            }
            mma_commit_pred(par ? &bars[4] : &bars[2], leader);
            __syncwarp();
#ifdef CM_TC_TRACE
            tr2 = clock64();
#endif
            // only warp 0 polls the completion barrier; the others sleep in the CTA barrier below and leave the issue slots to
            // the co-resident tile
            if (warp == 0) {
                ok = (par ? mbar_wait(&bars[4], p_phase) : mbar_wait(&bars[2], m_phase)) && ok;
                fence_before_thread_sync();
            }
        }
        if (par) p_phase ^= 1; else m_phase ^= 1;          // only the barrier that was used advances
        __syncthreads();
        fence_after_thread_sync();
#ifdef CM_TC_TRACE
        tr3 = clock64();
        if (blockIdx.x == 0 && tid == 0 && consumed < 64 && io.workspace) {
            long long *tb = reinterpret_cast<long long *>(io.workspace) + 8 * consumed;
            tb[0] = tr0; tb[1] = tr1; tb[2] = tr2; tb[3] = tr3; tb[4] = trw[0]; tb[5] = trw[1];
        }
#endif
        consumed += (uint32_t)nops;
        si += nops;
        issue_loads();
    };
    const MmaOp none = {0u, 0u, 0u, 0};
    // the same hand-shake for products whose operands are both written by the CTA (no weight stage is consumed)
    auto run_custom = [&](auto issue) {
        fence_proxy_async();
        fence_before_thread_sync();
        __syncthreads();
        if (warp == 0) {
            fence_after_thread_sync();
            const uint32_t leader = elect_one() ? 1u : 0u;
            if (!(CM_TC_DEBUG & 1)) issue(leader);
            mma_commit_pred(&bars[2], leader);
            __syncwarp();
            ok = mbar_wait(&bars[2], m_phase) && ok;
            fence_before_thread_sync();
        }
        m_phase ^= 1;
        __syncthreads();
        fence_after_thread_sync();
    };
    // products of INDEPENDENT accumulators issued by several warps at once (warp w issues the products of env slot w and commits
    // them on a barrier that expects one arrival per slot): the issue path of one thread costs ~60 cycles per instruction
    // whatever its size, so the 24 small products of an aggregation layer take a quarter of the time from four warps
    uint32_t s_phase = 0;
    auto run_slots = [&](int nw, auto issue) {
        fence_proxy_async();
        fence_before_thread_sync();
        __syncthreads();
        if (warp < nw) {
            fence_after_thread_sync();
            const uint32_t leader = elect_one() ? 1u : 0u;
            if (!(CM_TC_DEBUG & 1)) issue(warp, leader);
            mma_commit_pred(&bars[3], leader);
            __syncwarp();
        }
        if (warp == 0) {
            ok = mbar_wait(&bars[3], s_phase) && ok;
            fence_before_thread_sync();
        }
        s_phase ^= 1;
        __syncthreads();
        fence_after_thread_sync();
    };
    constexpr bool kAttnTc = kVec == 0;
    const int S = A.slot, slog = S == 64 ? 6 : 5;          // (slog is only meaningful with kAttnTc: S = 32 or 64)

    // dense epilogue of a 64-wide product: this thread's 16 columns -> bias, tanh -> next A operand (K panel of 64)
    auto epi64 = [&](uint32_t blk, int bias0, unsigned char *dst) {
        float v[16], w[16];
        ld_acc_raw<16>(lane_addr + blk, 64, 16 * sub, v, w);
        const float4 *bp = reinterpret_cast<const float4 *>(bias_s + bias0 + 16 * sub);
#pragma unroll
        for (int q = 0; q < 4; ++q) tanh4(v + 4 * q, w + 4 * q, bp[q], kActScale);
        write_act<16, true>(dst, 64, row, 16 * sub, v);
    };
    // neighbour mask of this row for layer l (dist_adj & channels[l], comm_base_net.py:101)
    uint32_t m0 = 0u, m1 = 0u;
    auto load_mask = [&](int env, int il, int l, bool valid) {
        m0 = m1 = 0u;
        if (valid) {
            m0 = m1 = 0xFFFFFFFFu;
            if (io.adj_bits) {
                const uint32_t *p = io.adj_bits + (size_t)(env * n + il) * W;
                m0 &= __ldg(p);
                if (W > 1) m1 &= __ldg(p + 1);
            }
            if (io.chan_bits) {
                const uint32_t *p = io.chan_bits + (size_t)((env * L + l) * n + il) * W;
                m0 &= __ldg(p);
                if (W > 1) m1 &= __ldg(p + 1);
            }
        }
    };

    // ---- observation staging: a tile's observations are ONE contiguous block of rows * D floats.  It is copied
    // with cp.async (no registers held, 16-byte copies where source and destination are congruent mod 16) into the
    // key/value + softmax scratch area while that area is idle (from the head of the previous tile on), and converted
    // to the fp16 hi/lo A operand when the tile starts.  Staged element i of the block lives at stage[(src & 3) + i].
    float *stage = KV;
    constexpr int kStageFloats = (64 + 8) * kTPitch - 4;
    // rows of tile tl: whole environments (Comm-DP: the attention stays inside a tile) or any 128 agent rows (Obs-DP)
    constexpr int mode = kMode;
    const int Din = A.in_dim;
    const bool dec = mode != kTcModeComm;            // every mode but Comm-DP treats the agent rows independently
    const int total_rows = n_envs * n;
    auto tile_rows = [&](int tl, int &r0, int &nr) {
        if constexpr (kMulti) {
            const int p = tl / A.tiles_per_policy, lt = tl - p * A.tiles_per_policy, epp = (int)io.envs_per_policy;
            if (dec) { const int pr = epp * n; r0 = p * pr + lt * kTcRows; nr = min(kTcRows, pr - lt * kTcRows); }
            else { const int e0 = lt * A.envs_per_tile; r0 = (p * epp + e0) * n; nr = min(A.envs_per_tile, epp - e0) * n; }
        } else {
            if (dec) { r0 = tl * kTcRows; nr = min(kTcRows, total_rows - r0); }
            else { const int e0 = tl * A.envs_per_tile; r0 = e0 * n; nr = min(A.envs_per_tile, n_envs - e0) * n; }
        }
    };
    // packed observations (io.obs_bits): a row is 6 words — 3 of window bits, 3 scalar columns as float bits — staged like 6 floats
    const bool packed = io.obs_bits != nullptr && kMode != kTcModeHead;
    const int Dst = packed ? 6 : Din;                 // words per staged row
    const float *obs_src = packed ? reinterpret_cast<const float *>(io.obs_bits) : io.obs;
    auto stage_obs = [&](int tl) {
        int r0s, rws;
        tile_rows(tl, r0s, rws);
        const float *src = obs_src + (size_t)r0s * Dst;
        const int a = (int)((reinterpret_cast<uintptr_t>(src) >> 2) & 3u);
        const int ns = min(rws * Dst, kStageFloats);
        const int nq = (a + ns + 3) >> 2;
        const uint32_t sbase = smem_u32(stage);
        for (int q = tid; q < nq; q += kTcThreads) {
            const int i0 = 4 * q - a;                   // block element of the quad's first float
            if (i0 >= 0 && i0 + 4 <= ns)
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sbase + 16u * (uint32_t)q), "l"(src + i0) : "memory");
            else {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (i0 + j >= 0 && i0 + j < ns)
                        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(sbase + 4u * (uint32_t)(4 * q + j)), "l"(src + i0 + j)
                                     : "memory");
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    if ((int)blockIdx.x < n_tiles) stage_obs((int)blockIdx.x);
    // bias table (and the last layer's weights) — after the first weight stages and the observations have been requested,
    // so that the three global round trips of the prologue overlap
    auto load_bias = [&](const float *__restrict__ w) {
        for (int i = tid; i < kBiasFloats; i += kTcThreads) {
            float v = 0.0f;
            if (i < kBEnc2) v = w[o.enc_b1 + i];
            else if (i < kBGcn) v = w[o.enc_b2 + i - kBEnc2];
            else if (i < kBH1) { if (i - kBGcn < L * 64) v = w[o.gcn_b + i - kBGcn]; }
            else if (i < kBH2) v = w[o.head_b1 + i - kBH1];
            else if (i < kBH3) v = w[o.head_b2 + i - kBH2];
            else if (i < kBH4) v = w[o.head_b3 + i - kBH3];
            else if (i < kBH4 + CM_ACTIONS) v = w[o.head_b4 + i - kBH4];
            else if (i >= kW4) v = w[o.head_w4 + i - kW4];
            bias_s[i] = i < kBH4 ? v * kTanhScale : v;        // every bias below kBH4 feeds a tanh (see tanh_scaled)
        }
    };
    int bias_policy = 0;                                 // policy whose biases bias_s holds
    if constexpr (kMulti) {
        bias_policy = (int)blockIdx.x / A.tiles_per_policy;
        load_bias(wts + (size_t)bias_policy * (size_t)io.weights_stride);
    } else {
        load_bias(wts);
    }
    __syncthreads();

    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        int row0, rows;
        tile_rows(tile, row0, rows);
        bool valid = row < rows;
        int g = row0 + row;
        // Comm-DP: env index inside the tile / agent index / first row of the env; Obs-DP rows are independent
        int el = valid ? (dec ? g / n : row / n) : 0;
        int il = valid ? (dec ? g - el * n : row - el * n) : 0, j0 = dec ? 0 : el * n;
        if constexpr (kAttnTc) {            // env slots of S tile rows: slot el holds agents 0 .. n - 1, the rest of the slot is padding
            el = row >> slog; il = row & (S - 1); j0 = el << slog;
            valid = il < n && el * n < rows;
            g = row0 + el * n + il;
            if (!valid) { el = 0; il = 0; }
        }
        const int env = dec ? el : row0 / n + el;
        const bool next_has = tile + (int)gridDim.x < n_tiles;
        si = 0;

        // ---------------- encoder layer 1: obs panels -> h[:, 0:64] in R0, h[:, 64:128] in R1 ----------------
        CM_TP(18);
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();                                   // the staged observations of this tile are visible
        if constexpr (kMulti) {
            // every thread is past the previous tile's last read of the bias table; the first product phase below (a CTA
            // barrier) orders these writes before the first epilogue that reads them
            const int p = tile / A.tiles_per_policy;
            if (p != bias_policy) { bias_policy = p; load_bias(wts + (size_t)p * (size_t)io.weights_stride); }
        }
        CM_TP(19);
        {
            const float *src = obs_src + (size_t)row0 * Dst;
            const int a = (int)((reinterpret_cast<uintptr_t>(src) >> 2) & 3u);
            const int total_f = rows * Dst, ns = min(total_f, kStageFloats);
            const int nbits = io.obs_nbits;
            for (int pnl = 0; pnl < P.l1_panels; ++pnl) {
                const int Kp = P.st[si].Kp, kofs = 64 * pnl, kg = Kp >> 3;          // kg = 2, 4, 6 or 8 groups of 8 columns
                const uint32_t lo_off = (uint32_t)kTcRows * Kp * 2, inv = packed ? 0u : (65536u + (uint32_t)kg - 1u) / (uint32_t)kg;   // (a run-time division: only where it is used)
                for (int e8 = tid; e8 < kTcRows * kg; e8 += kTcThreads) {           // one group of 8 columns of one row
                    // fp32 rows: consecutive threads take consecutive column groups of a row (consecutive floats); packed rows:
                    // consecutive threads take the SAME column group of consecutive rows, so that only the warps that own the
                    // group with the scalar columns run the float path (no divergence inside a warp)
                    const int r = packed ? (e8 & (kTcRows - 1)) : (int)(((uint32_t)e8 * inv) >> 16);
                    const int k8 = packed ? (e8 >> 7) << 3 : (e8 - r * kg) << 3;
                    uint4 hq, lq;
                    uint32_t *hw = &hq.x, *lw = &lq.x;
                    int rr = r;                                  // row of the tile's observation block behind tile row r
                    if constexpr (kAttnTc) { const int e_ = r >> slog, i_ = r & (S - 1); rr = i_ < n ? e_ * n + i_ : rows; }
                    if (packed) {
                        const int kb = kofs + k8;
                        const bool okr = rr < rows;
                        const uint32_t *wrow = reinterpret_cast<const uint32_t *>(stage + a) + rr * 6;     // (a packed tile is always staged whole)
                        if (kb + 8 <= nbits || kb >= Din) {
                            // window bits expand to 0 / 1: exact in fp16, no low-order part
                            const uint32_t b8 = (okr && kb < nbits) ? (wrow[kb >> 5] >> (kb & 31)) & 0xFFu : 0u;   // (8 | 32: one word)
#pragma unroll
                            for (int j2 = 0; j2 < 4; ++j2) {
                                hw[j2] = (((b8 >> (2 * j2)) & 1u) ? 0x3C00u : 0u) | (((b8 >> (2 * j2 + 1)) & 1u) ? 0x3C000000u : 0u);
                                lw[j2] = 0u;
                            }
                        } else {
                            // the group with the scalar columns (float bits in words 3..5): split like any float
                            float x[8];
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                const int k = kb + j;
                                x[j] = 0.0f;
                                if (okr && k < Din) x[j] = k < nbits ? (float)((wrow[k >> 5] >> (k & 31)) & 1u) : __uint_as_float(wrow[3 + k - nbits]);
                            }
#pragma unroll
                            for (int j2 = 0; j2 < 4; ++j2) split16x2(x[2 * j2], x[2 * j2 + 1], hw[j2], lw[j2]);
                        }
                    } else {
                        float x[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const int k = kofs + k8 + j, i = rr * Din + k;
                            x[j] = 0.0f;
                            if (rr < rows && k < Din) x[j] = i < ns ? stage[a + i] : __ldg(src + i);
                        }
#pragma unroll
                        for (int j2 = 0; j2 < 4; ++j2) split16x2(x[2 * j2], x[2 * j2 + 1], hw[j2], lw[j2]);
                    }
                    const uint32_t off = canon_off16(r, k8, Kp);
                    *reinterpret_cast<uint4 *>(ACT + off) = hq;
                    *reinterpret_cast<uint4 *>(ACT + lo_off + off) = lq;
                }
                // packed rows: A_lo is zero before the K slice that holds the first scalar column
                const int lo_from = packed ? max(0, min(Kp >> 4, (nbits - kofs) >> 4)) : 0;
                run_mma(2, MmaOp{kR0, (uint32_t)pnl, 0u, lo_from}, MmaOp{kR1, (uint32_t)pnl, 0u, lo_from});
            }
        }
        // ---------------- encoder layer 2 (K = 128 as the two panels of h) -> R0 ----------------
        if (mode != kTcModeHead) {          // head mode: the two products above already were the first head layer
        // (the second K panel of the A operand lives in the idle key / value buffer, so both products issue together)
        epi64(kR0, kBEnc1, ACT);
        epi64(kR1, kBEnc1 + 64, ACT2);
        run_mma(2, MmaOp{kR0, 0u, 0u}, MmaOp{kR0, 1u, 1u});
        // ---------------- E = tanh(. + b2): keys (k-major fp32) + A operand; Q -> R0, H_0 Wg_0 -> R1 ----------------
        {
            // E is also wanted unscaled as fp32 (the CUDA-core attention's keys, the large-team pipeline's rows): those
            // instantiations split it from the unscaled value
            constexpr bool e_pre = !((kMode == kTcModeComm && !kAttnTc) || kMode == kTcModeEnc);
            float v[16], w[16];
            ld_acc_raw<16>(lane_addr + kR0, 64, 16 * sub, v, w);
            const float4 *bp = reinterpret_cast<const float4 *>(bias_s + kBEnc2 + 16 * sub);
#pragma unroll
            for (int q = 0; q < 4; ++q) tanh4(v + 4 * q, w + 4 * q, bp[q], e_pre ? kActScale : 1.0f);
            if (!dec && !kAttnTc) {
#pragma unroll
                for (int c = 0; c < 16; ++c) KV[(16 * sub + c) * kTPitch + row] = v[c];
            }
            if (mode == kTcModeEnc && valid) {                        // E rows for the attention kernel (keys, residual)
#pragma unroll
                for (int c = 0; c < 16; c += 4)
                    *reinterpret_cast<float4 *>(A.scr_e + (size_t)g * kE + 16 * sub + c) = make_float4(v[c], v[c + 1], v[c + 2], v[c + 3]);
            }
            write_act<16, e_pre>(ACT, 64, row, 16 * sub, v);
        }
        }   // mode != head
        uint32_t tk = 0u, ep = 0u;                                                // sampling keys: latency hidden by the head
        if (mode != kTcModeEnc && sub == 0 && valid && io.actions && !d.greedy && !io.sample_u) { tk = __ldg(io.tick + env); ep = __ldg(io.episode + env); }
        if (mode == kTcModeEnc) {
            // large-team pipeline, first half: Q = E Wq and H_0 Wg_0 as rows in global scratch; the attention kernel takes over
            if (next_has) stage_obs(tile + (int)gridDim.x);
            run_mma(2, MmaOp{kR0, 0u, 0u}, MmaOp{kR1, 0u, 0u});
            float q[16], hw[16];
            ld_acc<16>(lane_addr + kR0, 64, 16 * sub, q);
            ld_acc<16>(lane_addr + kR1, 64, 16 * sub, hw);
            if (valid) {
#pragma unroll
                for (int c = 0; c < 16; c += 4) {
                    *reinterpret_cast<float4 *>(A.scr_q + (size_t)g * kE + 16 * sub + c) = make_float4(q[c], q[c + 1], q[c + 2], q[c + 3]);
                    *reinterpret_cast<float4 *>(A.scr_hw + (size_t)g * kE + 16 * sub + c) = make_float4(hw[c], hw[c + 1], hw[c + 2], hw[c + 3]);
                }
            }
            continue;
        }
        if (mode == kTcModeDec) {
            // Obs-DP (dec_categorical_mlp_policy.py:107-124): the embedding is the input of the 64 -> 32 layer
            if (next_has) stage_obs(tile + (int)gridDim.x);                           // the second-operand / key-value area is idle
            run_mma(1, MmaOp{kR1, 0u, 0u}, none);
        } else {
        if (mode == kTcModeComm) {
        if constexpr (kAttnTc) {
        // ================= tensor-core attention (17 <= n <= 64; env slots of S = 32 / 64 rows) =================
        load_mask(env, il, 0, valid);
        run_mma(2, MmaOp{kR0, 0u, 0u}, MmaOp{kR1, 0u, 0u});                // Q = E Wa -> R0, H_0 Wg_0 -> R1 (one phase, two issuing warps)
        {   // the query rows become the A operand of the score product (the second operand buffer is idle)
            float q[16];
            ld_acc<16>(lane_addr + kR0, 64, 16 * sub, q);
            write_act<16>(ACT2, 64, row, 16 * sub, q);
        }
        // scores of the whole tile: [128 rows] x [128 keys] = Q E^T; the B operand [E_hi ; E_lo] IS the A operand the encoder
        // epilogue left in ACT (same K-major core-matrix layout, lo block 128 rows further).  One accumulator block, columns
        // [0, 128) (issue_scores); H_0 Wg_0 waits in R1 until the softmax is done.
        CM_TP(0);
        run_custom([&](uint32_t leader) { issue_scores(tmem + kR0, ACT2, ACT, leader); });
        {
            float *attn_row = (io.attention && valid) ? io.attention + (size_t)g * n : nullptr;
            if (S == 32) softmax_tc<8>(lane_addr, red, attn_row, row, j0, sub, n, valid);
            else softmax_tc<16>(lane_addr, red, attn_row, row, j0, sub, n, valid);
        }
        const uint32_t v_lo = (uint32_t)kTcRows * 64 * 2;                  // lo block of the value operand / of a 64-wide A operand
        {   // E (this thread's 16 columns of the A operand) -> tensor memory, for the residual: ACT becomes the attention operand.
            // (the barrier below separates these reads from the first attention rows written into ACT)
            if (d.residual) {
                float ev[16];
#pragma unroll
                for (int g8 = 0; g8 < 16; g8 += 8) {
                    const uint32_t off = canon_off16(row, 16 * sub + g8, 64);
                    const uint4 hq = *reinterpret_cast<const uint4 *>(ACT + off);
                    const uint4 lq = *reinterpret_cast<const uint4 *>(ACT + v_lo + off);
                    unpack_act_pre(hq, lq, ev + g8);
                }
                tmem_st<8>(lane_addr + kColE + (uint32_t)(16 * sub), ev);
                tmem_st<8>(lane_addr + kColE + (uint32_t)(16 * sub + 8), ev + 8);
                tmem_st_wait();
            }
            tmem_st_wait();
        }
        CM_TP(1);
        {   // values (H_0 Wg_0, in R1 since the phase of the query product) -> A operand of the transposed aggregation (as
            // written: [key][64], i.e. MN-major); the score product has read the query rows out of this buffer
            // (barrier: every thread has read its E columns out of ACT and the softmax exchange out of `red` before the first
            // layer's attention rows and masked sums are written there — the product phase that used to sit here did that)
            __syncthreads();
            float v[16];
            ld_acc<16>(lane_addr + kR1, 64, 16 * sub, v);
            write_unscaled<16>(ACT2, 64, v_lo, row, 16 * sub, v, kVScale);
        }
        CM_TP(2);
        const int n_slots = kTcRows >> slog;                                // envs per tile
        for (int l = 0; l < L; ++l) {
            // A_l = M * Range * chan_l (comm_base_net.py:101): this thread's keys -> B operand rows in ACT (E / H_l are dead
            // there); the row's masked sum and maximum through one exchange
            float pscale;
            if (S == 32) masked_p_operand<8>(lane_addr, ACT, red, S, row, sub, n, m0, m1, pscale);
            else masked_p_operand<16>(lane_addr, ACT, red, S, row, sub, n, m0, m1, pscale);
            // out_e^T [64 x S] = V_e^T [64 x S keys] A_e^T [S keys x S rows] for every env slot e, three fp16 products each
            // into ONE accumulator (columns e S .. of R1; row c of the result = lane 32 (c / 16) + c % 16)
            run_slots(n_slots, [&](int e, uint32_t leader) {
                const uint32_t idesc = make_idesc_f16(64, S) | kIdescAMajorMN;
                const uint32_t a0 = smem_u32(ACT2), b0 = smem_u32(ACT), p_lo = (uint32_t)kTcRows * S * 2;
                const uint32_t dcol = tmem + kR1 + (uint32_t)(e << slog);
                const uint32_t ae = a0 + (uint32_t)e * (uint32_t)S * 128u;                       // key rows e S ..: 128 bytes per key
                const uint32_t be = b0 + (uint32_t)e * (uint32_t)(S >> 3) * (uint32_t)(S >> 3) * 128u;   // query rows e S ..
                for (int j = 0; j < (S >> 4); ++j) {
                    const uint64_t da_hi = make_smem_desc16_mn(ae + (uint32_t)j * 2048u, 64), da_lo = make_smem_desc16_mn(ae + v_lo + (uint32_t)j * 2048u, 64);
                    const uint64_t db_hi = make_smem_desc16(be, S, j), db_lo = make_smem_desc16(be + p_lo, S, j);
                    mma_f16_pred(dcol, da_hi, db_hi, idesc, j ? 1u : 0u, leader);
                    mma_f16_pred(dcol, da_hi, db_lo, idesc, 1u, leader);
                    mma_f16_pred(dcol, da_lo, db_hi, idesc, 1u, leader);
                }
            });
            const float den = ((red[row] + red[kTPitch + row]) + red[2 * kTPitch + row]) + red[3 * kTPitch + row];
            CM_TP(3 + 4 * l);
            {   // out^T (tensor memory: lane = column c, columns = tile rows) -> T[row][64] fp32, the 16-byte chunk index
                // XOR-swizzled by t_key(row): the warp reads its 32 tile rows in ONE load, the half-warp h taking rows
                // 32 sub + 16 h + k (k = 0 .. 15) of the 16 columns c of its quadrant, and stores them as scalars.  The key
                // (row & 7) ^ 4 (row / 16 % 2) keeps such a store conflict-free (the 16 lanes of a half-warp hit 16 banks, the
                // other half the other 16), a thread reads its 16 columns back as four 128-bit loads (8 lanes = 8 chunks).
                // t_key(row) = (k & 7) ^ 4 h is a compile-time constant per store up to the half-warp term.
                const int c = 16 * quad + (lane & 15), h = lane >> 4;
                float o[16];
                tmem_ld16x32(lane_addr + kR1 + (uint32_t)(32 * sub), o);
                // word index of (row 32 sub + 16 h, chunk (c / 4) ^ 4 h); the chunk occupies bits 2..5 alone, so the swizzle of
                // row + j (j < 8) is an XOR of j << 2
                const int t0 = (32 * sub + 16 * h) * 64 + ((((c >> 2) ^ (h << 2))) << 2) + (c & 3);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    float *tj = KV + (t0 ^ (j << 2));
                    tj[j * 64] = o[j];
                    tj[(8 + j) * 64] = o[8 + j];
                }
                fence_before_thread_sync();
                __syncthreads();
                fence_after_thread_sync();
            }
            // H_{l+1} = tanh(out / (sum + 1e-12) + b) for this thread's 16 columns (graph_conv_module.py:51-72); out carries
            // the row's scale 2^e, the sum does not (an exact power-of-two factor: (sum + 1e-12) 2^e <= 2 n + 2^107 1e-12)
            const float inv = __fdividef(kTanhScale * kPVUnscale, (den + 1e-12f) * pscale);
            float v[16];
            const float4 *bp = reinterpret_cast<const float4 *>(bias_s + kBGcn + l * 64 + 16 * sub);
            const float4 *Tr = reinterpret_cast<const float4 *>(KV + row * 64);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float4 b4 = bp[q];
                const float4 t4 = Tr[(4 * sub + q) ^ ((row & 7) ^ ((row >> 2) & 4))];   // t_key(row)
                v[4 * q + 0] = fmaf(t4.x, inv, b4.x);
                v[4 * q + 1] = fmaf(t4.y, inv, b4.y);
                v[4 * q + 2] = fmaf(t4.z, inv, b4.z);
                v[4 * q + 3] = fmaf(t4.w, inv, b4.w);
                tanh4_scaled(v[4 * q + 0], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3], kActScale);
            }
            if (d.residual && l + 1 == L) {               // X = E + H_L (comm_base_net.py:105-106), both pre-scaled
                float ev[16];
                tmem_ld8(lane_addr + kColE + (uint32_t)(16 * sub), *reinterpret_cast<float(*)[8]>(ev));
                tmem_ld8(lane_addr + kColE + (uint32_t)(16 * sub + 8), *reinterpret_cast<float(*)[8]>(ev + 8));
                tmem_ld_wait();
#pragma unroll
                for (int c = 0; c < 16; ++c) v[c] += ev[c];
            }
            write_act<16, true>(ACT, 64, row, 16 * sub, v);
            CM_TP(4 + 4 * l);
            if (l + 1 < L) {
                load_mask(env, il, l + 1, valid);
                run_mma(1, MmaOp{kR1, 0u, 0u}, none);         // H_{l+1} Wg_{l+1} -> R1 (the transposed result has been read)
                CM_TP(5 + 4 * l);
                float hv[16];
                ld_acc<16>(lane_addr + kR1, 64, 16 * sub, hv);
                write_unscaled<16>(ACT2, 64, v_lo, row, 16 * sub, hv, kVScale);
            }
        }
        } else {
        // ================= exact CUDA-core attention (n <= 16) =================
        load_mask(env, il, 0, valid);
        run_mma(2, MmaOp{kR0, 0u, 0u}, MmaOp{kR1, 0u, 0u});
        // ---------------- scores, softmax (exact per environment, CUDA cores); attention row -> TMEM ----------------
        CM_TP(0);
        {
            float *attn_row = (io.attention && valid) ? io.attention + (size_t)g * n : nullptr;
            switch (n <= 4 ? 1 : (n <= 8 ? 2 : (n <= 16 ? 4 : (n <= 32 ? 8 : 16)))) {
            case 1: scores_softmax<1, kVec>(lane_addr, KV, red, attn_row, row, j0, sub, n, valid); break;
            case 2: scores_softmax<2, kVec>(lane_addr, KV, red, attn_row, row, j0, sub, n, valid); break;
            case 4: scores_softmax<4, kVec>(lane_addr, KV, red, attn_row, row, j0, sub, n, valid); break;
            case 8: scores_softmax<8, kVec>(lane_addr, KV, red, attn_row, row, j0, sub, n, valid); break;
            default: scores_softmax<16, kVec>(lane_addr, KV, red, attn_row, row, j0, sub, n, valid); break;
            }
        }
        // H_0 Wg_0 replaces the keys (everybody is past the softmax barrier)
        CM_TP(1);
        {
            float v[16];
            ld_acc<16>(lane_addr + kR1, 64, 16 * sub, v);
#pragma unroll
            for (int c = 0; c < 16; ++c) KV[(16 * sub + c) * kTPitch + row] = v[c];
            tmem_st_wait();
            fence_before_thread_sync();
            __syncthreads();              // values and attention rows (TMEM scratch) are visible
            fence_after_thread_sync();
        }
        // ---------------- graph convolutions ----------------
        CM_TP(2);
        for (int l = 0; l < L; ++l) {
            // A_l = M * Range * chan_l / (sum + 1e-12); out = A_l (H_l Wg_l)   (comm_base_net.py:101-103, graph_conv_module.py:51-72)
            float acc[16];
#pragma unroll
            for (int c = 0; c < 16; ++c) acc[c] = 0.0f;
            float den = 0.0f;
            const float *hw0 = KV + (16 * sub) * kTPitch + j0;
            for (int c0 = 0; c0 < n; c0 += 8) {          // warp-uniform: the TMEM loads are collective
                float a8[8];
                tmem_ld8(lane_addr + kColM + (uint32_t)c0, a8);
                tmem_ld_wait();
                if (!(CM_TC_DEBUG & 4)) {
                    // mask the chunk's attention values (same key order as the scalar loop: the sums are bit-identical)
                    const uint32_t mbits = (c0 < 32 ? m0 : m1) >> (c0 & 31);
#pragma unroll
                    for (int j = 0; j < 8; ++j) a8[j] = (c0 + j < n && ((mbits >> j) & 1u)) ? a8[j] : 0.0f;
                    // the values of consecutive keys are consecutive floats of a k-major row: vector loads when aligned
                    if (kVec == 4) {
#pragma unroll
                        for (int j = 0; j < 8; j += 4)
                            if (c0 + j < n) {
                                den += a8[j]; den += a8[j + 1]; den += a8[j + 2]; den += a8[j + 3];
#pragma unroll
                                for (int c = 0; c < 16; ++c) {
                                    const float4 h = *reinterpret_cast<const float4 *>(hw0 + c * kTPitch + c0 + j);
                                    acc[c] = fmaf(a8[j + 3], h.w, fmaf(a8[j + 2], h.z, fmaf(a8[j + 1], h.y, fmaf(a8[j], h.x, acc[c]))));
                                }
                            }
                    } else if (kVec == 2) {
#pragma unroll
                        for (int j = 0; j < 8; j += 2)
                            if (c0 + j < n) {
                                den += a8[j]; den += a8[j + 1];
#pragma unroll
                                for (int c = 0; c < 16; ++c) {
                                    const float2 h = *reinterpret_cast<const float2 *>(hw0 + c * kTPitch + c0 + j);
                                    acc[c] = fmaf(a8[j + 1], h.y, fmaf(a8[j], h.x, acc[c]));
                                }
                            }
                    } else {
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            if (c0 + j < n) {
                                den += a8[j];
                                const float *hw = hw0 + c0 + j;
#pragma unroll
                                for (int c = 0; c < 16; ++c) acc[c] = fmaf(a8[j], hw[c * kTPitch], acc[c]);
                            }
                    }
                }
            }
            CM_TP(3 + 4 * l);
            const float inv = kTanhScale / (den + 1e-12f);            // scale of tanh_scaled folded into the normalisation
            float v[16];
            const float4 *bp = reinterpret_cast<const float4 *>(bias_s + kBGcn + l * 64 + 16 * sub);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float4 b4 = bp[q];
                v[4 * q + 0] = fmaf(acc[4 * q + 0], inv, b4.x);
                v[4 * q + 1] = fmaf(acc[4 * q + 1], inv, b4.y);
                v[4 * q + 2] = fmaf(acc[4 * q + 2], inv, b4.z);
                v[4 * q + 3] = fmaf(acc[4 * q + 3], inv, b4.w);
                tanh4_scaled(v[4 * q + 0], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3], kActScale);
            }
            if (d.residual) {                             // X = E + H_L (comm_base_net.py:105-106), both pre-scaled
                // E is still in the A operand buffer (this thread wrote these 16 columns itself) until the first layer's
                // output replaces it; with more than one layer it is parked in tensor memory meanwhile
                if (l == 0) {
                    float ev[16];
#pragma unroll
                    for (int g8 = 0; g8 < 16; g8 += 8) {
                        const uint32_t off = canon_off16(row, 16 * sub + g8, 64);
                        const uint4 hq = *reinterpret_cast<const uint4 *>(ACT + off);
                        const uint4 lq = *reinterpret_cast<const uint4 *>(ACT + (uint32_t)kTcRows * 64 * 2 + off);
                        unpack_act_pre(hq, lq, ev + g8);
                    }
                    if (L == 1) {
#pragma unroll
                        for (int c = 0; c < 16; ++c) v[c] += ev[c];
                    } else {
                        tmem_st<8>(lane_addr + kColE + (uint32_t)(16 * sub), ev);
                        tmem_st<8>(lane_addr + kColE + (uint32_t)(16 * sub + 8), ev + 8);
                        tmem_st_wait();
                    }
                } else if (l + 1 == L) {
                    float ev[16];
                    tmem_ld8(lane_addr + kColE + (uint32_t)(16 * sub), *reinterpret_cast<float(*)[8]>(ev));
                    tmem_ld8(lane_addr + kColE + (uint32_t)(16 * sub + 8), *reinterpret_cast<float(*)[8]>(ev + 8));
                    tmem_ld_wait();
#pragma unroll
                    for (int c = 0; c < 16; ++c) v[c] += ev[c];
                }
            }
            write_act<16, true>(ACT, 64, row, 16 * sub, v);
            CM_TP(4 + 4 * l);
            if (l + 1 < L) {
                load_mask(env, il, l + 1, valid);
                run_mma(1, MmaOp{kR1, 0u, 0u}, none);         // every thread is done with the values of layer l here
                CM_TP(5 + 4 * l);
                float hv[16];
                ld_acc<16>(lane_addr + kR1, 64, 16 * sub, hv);
#pragma unroll
                for (int c = 0; c < 16; ++c) KV[(16 * sub + c) * kTPitch + row] = hv[c];
                __syncthreads();
            }
        }
        }   // CUDA-core attention
        // ---------------- categorical head ----------------
        run_mma(2, MmaOp{kR0, 0u, 0u}, MmaOp{kR1, 0u, 0u});                       // 64 -> 128 as two output halves
        }   // Comm-DP only (head mode enters here: its first two products came with the input rows)
        epi64(kR0, kBH1, ACT);                                                    // 128 -> 64: two K panels, issued together
        epi64(kR1, kBH1 + 64, ACT2);
        run_mma(2, MmaOp{kR0, 0u, 0u}, MmaOp{kR0, 1u, 1u});
        if (next_has) stage_obs(tile + (int)gridDim.x);                           // keys / values / ACT2 are dead: next tile's obs
        epi64(kR0, kBH2, ACT);                                                    // 64 -> 32
        run_mma(1, MmaOp{kR1, 0u, 0u}, none);
        }   // Comm-DP / head
        {   // 32 -> 5 on the CUDA cores (exact fp32): this thread's 8 inputs -> 5 partial logits, parked in tensor memory
            float v[8], w[8], part[8];
            ld_acc_raw<8>(lane_addr + kR1, 32, 8 * sub, v, w);
            const float4 *bp = reinterpret_cast<const float4 *>(bias_s + kBH3 + 8 * sub);
            tanh4(v, w, bp[0]);
            tanh4(v + 4, w + 4, bp[1]);
#pragma unroll
            for (int a = 0; a < 8; ++a) part[a] = 0.0f;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const float *w4 = bias_s + kW4 + (8 * sub + c) * CM_ACTIONS;
#pragma unroll
                for (int a = 0; a < CM_ACTIONS; ++a) part[a] = fmaf(v[c], w4[a], part[a]);
            }
            tmem_st<8>(lane_addr + kR0 + (uint32_t)(8 * sub), part);
            tmem_st_wait();
            fence_before_thread_sync();
            __syncthreads();
            fence_after_thread_sync();
        }
        // ---------------- softmax, availability mask, renormalise, sample ----------------
        CM_TP(16);
        if (sub == 0) {
            float lg8[8];
#pragma unroll
            for (int a = 0; a < 8; ++a) lg8[a] = a < CM_ACTIONS ? bias_s[kBH4 + a] : 0.0f;
#pragma unroll
            for (int s4 = 0; s4 < 4; ++s4) {
                float pq[8];
                tmem_ld8(lane_addr + kR0 + (uint32_t)(8 * s4), pq);
                tmem_ld_wait();
#pragma unroll
                for (int a = 0; a < 8; ++a) lg8[a] += pq[a];
            }
            if (valid) {
                float lg[CM_ACTIONS], pr[CM_ACTIONS];
                float mx = -INFINITY;
#pragma unroll
                for (int a = 0; a < CM_ACTIONS; ++a) { lg[a] = lg8[a]; mx = fmaxf(mx, lg[a]); }
                float sum = 0.0f;
#pragma unroll
                for (int a = 0; a < CM_ACTIONS; ++a) { pr[a] = expf(lg[a] - mx); sum += pr[a]; }
                const uint32_t av = io.avail_bits ? io.avail_bits[g] : 0x1Fu;
                float msum = 0.0f;
#pragma unroll
                for (int a = 0; a < CM_ACTIONS; ++a) { pr[a] = ((av >> a) & 1u) ? pr[a] / sum : 0.0f; msum += pr[a]; }
#pragma unroll
                for (int a = 0; a < CM_ACTIONS; ++a) pr[a] = pr[a] / msum;
                if (io.logits) for (int a = 0; a < CM_ACTIONS; ++a) io.logits[(size_t)g * CM_ACTIONS + a] = lg[a];
                if (io.probs) for (int a = 0; a < CM_ACTIONS; ++a) io.probs[(size_t)g * CM_ACTIONS + a] = pr[a];
                if (io.actions) {
                    int act;
                    if (d.greedy) {
                        act = 0;
                        for (int a = 1; a < CM_ACTIONS; ++a) if (pr[a] > pr[act]) act = a;
                    } else {
                        float u;
                        if (io.sample_u) u = io.sample_u[g];
                        else {
                            const uint4 blk = philox4x32_10(
                                make_uint4((uint32_t)(d.env_id0 + env), tk, kStreamAct | (ep << 8), (uint32_t)(il >> 2)),
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
            }
        }
        CM_TP(17);
        // the next tile's first products overwrite R0 / R1 only after the barrier inside run_mma, which the threads that
        // are still reading the logits have not reached yet
    }
    if (!ok && io.error_flag) atomicExch(io.error_flag, (int)CM_ECUDA);
    fence_before_thread_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, kTmemCols);
    CM_TPK(21);
#ifdef CM_TC_TRACE
    if (threadIdx.x == 0 && A.io.workspace) {
        unsigned long long gt; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt));
        reinterpret_cast<unsigned long long *>(A.io.workspace)[1024 + 2 * blockIdx.x + 1] = gt;
    }
#endif
}

// ------------------------------------------------------------------------------------------------
// weight preparation: fp32 k-major blob -> per-stage canonical hi | lo panels
// ------------------------------------------------------------------------------------------------
__global__ void tc_prepare_kernel(const float *__restrict__ w, __half *__restrict__ out, const TcPlan P)
{
    for (int s = 0; s < P.n_stages; ++s) {
        const TcStage st = P.st[s];
        const int total = st.N * st.Kp;
        for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
            const int r = e / st.Kp, k = e - r * st.Kp;
            float v = 0.0f;
            if (st.n0 + r < st.Nsrc && st.k0 + k < st.Ksrc) v = w[st.src_off + (size_t)(st.k0 + k) * st.Nsrc + st.n0 + r];
            const __half h = __float2half_rn(v);
            const __half l = __float2half_rn((v - __half2float(h)) * 4096.0f);
            // canonical K-major layout over the stacked 2N rows: hi rows [0, N), lo rows [N, 2N)
            auto idx = [&](int rr) { return (rr >> 3) * (st.Kp >> 3) * 64 + (k >> 3) * 64 + (rr & 7) * 8 + (k & 7); };
            out[st.w_off + idx(r)] = h;
            out[st.w_off + idx(st.N + r)] = l;
        }
    }
}

static size_t tc_smem_bytes() { return (size_t)kActBytes + kWBytes + (64 + 8) * kTPitch * 4 + kBiasFloats * 4 + 64; }   // (4 mbarriers + the TMEM base)

static int launch_tc_mode(const cm_policy_desc *desc, const cm_policy_io *io, int mode, int in_dim, float *scr_e, float *scr_q,
                          float *scr_hw, cudaStream_t stream)
{
    if (!io->tc_weights) return CM_EINVAL;
    const bool rows_mode = mode != kTcModeComm;
    if ((!rows_mode && desc->n_agents > 64) || desc->obs_dim > 128) return CM_EUNSUPPORTED;
    if (io->n_envs * desc->n_agents > (int64_t)1 << 23) return CM_EUNSUPPORTED;      // 32-bit element indices inside the kernel
    TcArgs A;
    A.d = *desc;
    A.io = *io;
    A.mode = mode;
    A.in_dim = in_dim;
    A.scr_e = scr_e; A.scr_q = scr_q; A.scr_hw = scr_hw;
    A.plan = make_tc_plan(desc->obs_dim, desc->n_layers, mode);
    // Comm-DP teams of 17 .. 64 agents: attention on the tensor cores, an env per slot of 32 / 64 tile rows (a slot is a
    // multiple of the warp size, so a warp's rows share their env's key columns); smaller teams: dense packing, CUDA cores
    const bool attn_tc = !rows_mode && desc->n_agents > 16;
    A.slot = rows_mode ? 0 : (attn_tc ? (desc->n_agents <= 32 ? 32 : 64) : desc->n_agents);
    A.envs_per_tile = rows_mode ? 0 : kTcRows / A.slot;
    A.n_tiles = rows_mode ? (io->n_envs * desc->n_agents + kTcRows - 1) / kTcRows : (io->n_envs + A.envs_per_tile - 1) / A.envs_per_tile;
    const bool multi = io->n_policies > 1;
    A.tiles_per_policy = (int)A.n_tiles;
    if (multi) {            // tiles counted per env block: no tile holds rows of two policies
        A.tiles_per_policy = (int)(rows_mode ? (io->envs_per_policy * desc->n_agents + kTcRows - 1) / kTcRows
                                             : (io->envs_per_policy + A.envs_per_tile - 1) / A.envs_per_tile);
        A.n_tiles = (int64_t)io->n_policies * A.tiles_per_policy;
    }
    const size_t smem = tc_smem_bytes();
    const int vec = rows_mode ? 1 : (attn_tc ? 0 : ((desc->n_agents & 3) == 0 ? 4 : ((desc->n_agents & 1) == 0 ? 2 : 1)));
    void (*kernel)(const TcArgs) =
        !multi ? (mode == kTcModeDec ? policy_tc_kernel<1, kTcModeDec>
                  : mode == kTcModeEnc ? policy_tc_kernel<1, kTcModeEnc>
                  : mode == kTcModeHead ? policy_tc_kernel<1, kTcModeHead>
                  : vec == 0 ? policy_tc_kernel<0, kTcModeComm>
                  : vec == 4 ? policy_tc_kernel<4, kTcModeComm> : (vec == 2 ? policy_tc_kernel<2, kTcModeComm> : policy_tc_kernel<1, kTcModeComm>))
               : (mode == kTcModeDec ? policy_tc_kernel<1, kTcModeDec, true>
                  : mode == kTcModeEnc ? policy_tc_kernel<1, kTcModeEnc, true>
                  : mode == kTcModeHead ? policy_tc_kernel<1, kTcModeHead, true>
                  : vec == 0 ? policy_tc_kernel<0, kTcModeComm, true>
                  : vec == 4 ? policy_tc_kernel<4, kTcModeComm, true>
                  : (vec == 2 ? policy_tc_kernel<2, kTcModeComm, true> : policy_tc_kernel<1, kTcModeComm, true>));
    static thread_local struct { int dev; int sms; } cache[2][7] = {{{-1, 0}, {-1, 0}, {-1, 0}, {-1, 0}, {-1, 0}, {-1, 0}, {-1, 0}},
                                                                    {{-1, 0}, {-1, 0}, {-1, 0}, {-1, 0}, {-1, 0}, {-1, 0}, {-1, 0}}};
    auto &cc = cache[multi][mode == kTcModeComm ? (vec == 0 ? 6 : (vec >> 1)) : 2 + mode];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return set_cuda_error(cudaGetLastError(), CM_ENODEVICE);
    if (cc.dev != dev) {
        int sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return set_cuda_error(cudaGetLastError(), CM_ECUDA);
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return set_cuda_error(e, CM_ECUDA);
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return set_cuda_error(e, CM_ECUDA);
        cc.dev = dev; cc.sms = sms;
    }
    int slots = 2 * cc.sms;                                                   // persistent: two CTAs per SM
#ifdef CM_TC_TRACE
    if (const char *ev = getenv("CM_TC_SLOTS")) slots = atoi(ev) * cc.sms;      // experiments only
#endif
    const int grid = (int)(A.n_tiles < slots ? A.n_tiles : slots);
    kernel<<<grid, kTcThreads, smem, stream>>>(A);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_cuda_error(e, CM_ECUDA);
    return CM_OK;
}

int launch_policy_tc_large(const cm_policy_desc *desc, const cm_policy_io *io, cudaStream_t stream);   // policy_attn_mma_kernel.cu

int launch_policy_tc(const cm_policy_desc *desc, const cm_policy_io *io, cudaStream_t stream)
{
    if (desc->kind == CM_POLICY_COMM && desc->n_agents > 64) return launch_policy_tc_large(desc, io, stream);
    const int mode = desc->kind == CM_POLICY_DEC ? kTcModeDec : kTcModeComm;
    return launch_tc_mode(desc, io, mode, desc->obs_dim, nullptr, nullptr, nullptr, stream);
}

// large-team pipeline halves (launch_policy_tc_large drives them): rows -> E, Q, H_0 Wg_0 ; X rows -> logits / actions
int launch_policy_tc_encode(const cm_policy_desc *desc, const cm_policy_io *io, float *scr_e, float *scr_q, float *scr_hw, cudaStream_t stream)
{
    return launch_tc_mode(desc, io, kTcModeEnc, desc->obs_dim, scr_e, scr_q, scr_hw, stream);
}
int launch_policy_tc_head(const cm_policy_desc *desc, const cm_policy_io *io, const float *x_rows, cudaStream_t stream)
{
    cm_policy_io io2 = *io;
    io2.obs = x_rows;
    return launch_tc_mode(desc, &io2, kTcModeHead, kE, nullptr, nullptr, nullptr, stream);
}

}  // namespace cm

extern "C" size_t cm_policy_tc_blob_floats(int32_t obs_dim, int32_t n_layers)
{
    return (size_t)(cm::make_tc_plan(obs_dim, n_layers).total_halves + 1) / 2;
}

namespace cm { int cent_tc_prepare(const cm_policy_desc *desc, const float *weights, float *tc_weights, cudaStream_t stream); }   // policy_cent_kernel.cu

extern "C" int cm_policy_tc_prepare(const cm_policy_desc *desc, const float *weights, float *tc_weights, cm_stream_t stream)
{
    if (!desc || !weights || !tc_weights) return CM_EINVAL;
    if (desc->kind == CM_POLICY_CENT) {
        if (desc->n_agents < 1 || desc->n_agents > CM_MAX_AGENTS || desc->obs_dim < 1 || desc->obs_dim > 128) return CM_EUNSUPPORTED;
        if (cm_device_count() < 1) return CM_ENODEVICE;
        return cm::cent_tc_prepare(desc, weights, tc_weights, (cudaStream_t)stream);
    }
    if (desc->n_layers < 1 || desc->n_layers > CM_MAX_LAYERS || desc->obs_dim < 1 || desc->obs_dim > 128) return CM_EUNSUPPORTED;
    if (cm_device_count() < 1) return CM_ENODEVICE;
    const cm::TcPlan P = cm::make_tc_plan(desc->obs_dim, desc->n_layers, cm::kTcModeComm);   // every mode reads this blob
    cm::tc_prepare_kernel<<<64, 256, 0, (cudaStream_t)stream>>>(weights, reinterpret_cast<__half *>(tc_weights), P);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? CM_OK : cm::set_cuda_error(e, CM_ECUDA);
}
