// policy_layout.cuh — weight-blob layouts shared by the policy kernels.
#pragma once
#include <stdint.h>

#include "commarl_b200.h"

namespace cm {

static constexpr int kH1 = 128, kE = 64, kC1 = 128, kC2 = 64, kC3 = 32;

struct Blob {   // float offsets into the weight blob (commarl_b200.h)
    int enc_w1, enc_b1, enc_w2, enc_b2, att_w, gcn_w, gcn_b, head_w1, head_b1, head_w2, head_b2, head_w3, head_b3,
        head_w4, head_b4, total;
};

__host__ __device__ inline Blob blob_layout(int D, int L)
{
    Blob o;
    int p = 0;
    o.enc_w1 = p; p += D * kH1;
    o.enc_b1 = p; p += kH1;
    o.enc_w2 = p; p += kH1 * kE;
    o.enc_b2 = p; p += kE;
    o.att_w = p; p += kE * kE;
    o.gcn_w = p; p += L * kE * kE;
    o.gcn_b = p; p += L * kE;
    o.head_w1 = p; p += kE * kC1;
    o.head_b1 = p; p += kC1;
    o.head_w2 = p; p += kC1 * kC2;
    o.head_b2 = p; p += kC2;
    o.head_w3 = p; p += kC2 * kC3;
    o.head_b3 = p; p += kC3;
    o.head_w4 = p; p += kC3 * CM_ACTIONS;
    o.head_b4 = p; p += CM_ACTIONS;
    o.total = p;
    return o;
}

// CENT policy blob (CentralizedCategoricalMLPPolicy: one MLP over the concatenated observation, K = n*D inputs, 5n outputs),
// every dense weight K-major like the Comm-DP blob:  w1 [n*D][128] b1 [128] w2 [128][64] b2 [64] w3 [64][32] b3 [32] w4 [32][5n] b4 [5n]
struct CentBlob { int w1, b1, w2, b2, w3, b3, w4, b4, total; };

__host__ __device__ inline CentBlob cent_blob_layout(int n, int D)
{
    CentBlob o;
    int p = 0;
    o.w1 = p; p += n * D * kC1;
    o.b1 = p; p += kC1;
    o.w2 = p; p += kC1 * kC2;
    o.b2 = p; p += kC2;
    o.w3 = p; p += kC2 * kC3;
    o.b3 = p; p += kC3;
    o.w4 = p; p += kC3 * n * CM_ACTIONS;
    o.b4 = p; p += n * CM_ACTIONS;
    o.total = p;
    return o;
}

// ---- tcgen05 variant.  Every dense product runs on the tensor cores in fp16 with error compensation:
//   x = x_hi + 2^-12 x_lo,   x_hi = fp16(x),   x_lo = fp16((x - x_hi) * 4096)        (22+ significant bits)
//   D[:, 0:N]  = A_hi B_hi^T                     (one accumulator)
//   D[:, N:2N] = A_hi B_lo^T + A_lo B_hi^T       (second accumulator, weight 2^-12 in the epilogue)
// One "stage" = the B operand of one product: [B_hi ; B_lo] stacked along N (2N rows x Kp fp16) in the canonical
// K-major core-matrix layout, so that A_hi x stage yields both accumulators with ONE series of K/16 instructions and
// A_lo x (first N rows) adds the remaining cross term with another K/16.  Every product has N <= 64 (the two 128-wide
// layers are split into output halves, n0 = 0 / 64) and K <= 64 (wide inputs are split into K panels, k0 = 0 / 64), so
// a stage is at most 16 KB (a slot of the kernel's weight ring) and an accumulator block at most 128 tensor-memory
// columns: a CTA needs 256 columns and ~103 KB of shared memory, and TWO tiles stay resident per SM.  Stages are
// stored in the order in which a tile consumes them.  Offsets are in halves. ----
struct TcStage { int w_off, src_off, N, Kp, k0, n0, Ksrc, Nsrc; };
static constexpr int kTcMaxStages = 20;
struct TcPlan {
    int n_stages, total_halves, seq_len;
    int l1_panels;                          // obs K panels (1 or 2)
    TcStage st[kTcMaxStages];
};

// Kernel modes.  COMM and DEC are the public policy kinds; ENC and HEAD are the row-wise halves of the large-team
// pipeline (teams of more than 64 agents: encoder + first value projection, then the attention kernel, then the head).
// All of them read the SAME prepared blob: the stage list of COMM contains every product, the other modes use a
// sub-list of it with the original offsets.
enum { kTcModeComm = 0, kTcModeDec = 1, kTcModeEnc = 2, kTcModeHead = 3 };

__host__ __device__ inline TcPlan make_tc_plan(int D, int L, int mode = kTcModeComm)
{
    const Blob o = blob_layout(D, L);
    TcPlan F;                                 // the full (COMM) list
    int s = 0, off = 0;
    auto add = [&](int src_off, int N, int Kp, int k0, int n0, int Ksrc, int Nsrc) {
        F.st[s].w_off = off; F.st[s].src_off = src_off; F.st[s].N = N; F.st[s].Kp = Kp; F.st[s].k0 = k0; F.st[s].n0 = n0;
        F.st[s].Ksrc = Ksrc; F.st[s].Nsrc = Nsrc;
        off += 2 * N * Kp;
        return s++;
    };
    const int Dp = (D + 15) / 16 * 16;
    const int panels = Dp > 64 ? 2 : 1;
    for (int pnl = 0; pnl < panels; ++pnl) {
        const int Kp = pnl == 0 ? (Dp <= 64 ? Dp : 64) : Dp - 64;
        add(o.enc_w1, 64, Kp, 64 * pnl, 0, D, kH1);                      // h[:, 0:64]
        add(o.enc_w1, 64, Kp, 64 * pnl, 64, D, kH1);                     // h[:, 64:128]
    }
    add(o.enc_w2, kE, 64, 0, 0, kH1, kE);
    add(o.enc_w2, kE, 64, 64, 0, kH1, kE);
    const int i_att = s;
    add(o.att_w, kE, 64, 0, 0, kE, kE);
    for (int l = 0; l < L; ++l) add(o.gcn_w + l * kE * kE, kE, 64, 0, 0, kE, kE);
    const int i_head = s;
    add(o.head_w1, 64, 64, 0, 0, kE, kC1);
    add(o.head_w1, 64, 64, 0, 64, kE, kC1);
    add(o.head_w2, kC2, 64, 0, 0, kC1, kC2);
    add(o.head_w2, kC2, 64, 64, 0, kC1, kC2);
    const int i_head3 = s;
    add(o.head_w3, kC3, 64, 0, 0, kC2, kC3);
    // (the last layer, 32 -> 5, runs on the CUDA cores in exact fp32)
    F.n_stages = s;
    F.total_halves = off;
    // sub-list of the mode
    TcPlan P;
    P.total_halves = off;
    P.l1_panels = mode == kTcModeHead ? 1 : panels;
    int t = 0;
    auto take = [&](int a, int b) { for (int i = a; i < b; ++i) P.st[t++] = F.st[i]; };
    if (mode == kTcModeComm) take(0, s);
    else if (mode == kTcModeDec) { take(0, i_att); take(i_head3, s); }        // Obs-DP: the embedding feeds the 64 -> 32 layer
    else if (mode == kTcModeEnc) take(0, i_att + 2);                          // ... attention query, H_0 Wg_0
    else take(i_head, s);                                                     // head on X = E + H_L
    P.n_stages = t;
    P.seq_len = t;
    return P;
}

// offset (in halves) of the graph-convolution weight stage of layer l inside the prepared blob
__host__ __device__ inline TcStage tc_gcn_stage(int D, int L, int l)
{
    const TcPlan F = make_tc_plan(D, L, kTcModeComm);
    const int panels = ((D + 15) / 16 * 16) > 64 ? 2 : 1;
    return F.st[2 * panels + 2 + 1 + l];
}

}  // namespace cm
