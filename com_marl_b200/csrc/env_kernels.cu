// env_kernels.cu — batched PredatorPrey / Coverage step, reset, observation windows and communication
// state for sm_100a.  A group of 4, 8, 16 or 32 lanes owns one environment instance (8 lanes for teams of up
// to ~56 agents: a warp then walks 4 envs at once and their order-dependent loops share its instructions).
//
// B200 mapping (DESIGN.md §3): state lives in HBM as SoA rows (positions u16, flags u8, bit rows u64);
// a lane group stages its env in shared memory, rebuilds the occupancy of the grid as 64-bit ROW BITMAPS
// (agents / preys or visited / walls) instead of the reference's grid of strings, runs the two
// order-dependent loops (agent moves, prey capture+walk) on one lane over those bitmaps while all the
// order-independent work (neighbour counts, candidate screening, watching flags, window extraction,
// adjacency, channel draws) is done lane-parallel, and streams the fp32 observation block out with
// fully coalesced 128-bit stores.  Everything here is integer/bit work bound by HBM traffic and issue slots;
// no tensor cores are involved on purpose.
//
// Semantics follow the reference exactly (file:line cited at each step); the data model does not.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "commarl_b200.h"
#include "common.cuh"

namespace cm {

typedef unsigned long long u64;

// 1: exact parallel move resolution (resolve_agents / resolve_preys); 0: the order-dependent loops on the group's lane 0.
// Both are bit-exact against the reference; which one is compiled in is a measured choice (DESIGN.md 3.1).
#ifndef CM_ENV_PARALLEL_MOVES
#define CM_ENV_PARALLEL_MOVES 0
#endif
#ifndef CM_ENV_WARPS
#define CM_ENV_WARPS 8
#endif
static constexpr int kWarpsPerCta = CM_ENV_WARPS;   // 24 warps per SM either way (80 registers)
// per-CTA constants in shared memory: wall rows [64] u64 | k / n as IEEE doubles for k = 0 .. n (<= 256) [257] f64
static constexpr int kConstBytes = 64 * 8 + 264 * 8;

struct EnvArgs {
    cm_env_desc d;
    cm_env_state s;
    cm_step_io io;
    const uint8_t *mask;
    int mode;        // 0 step, 1 reset, 2 comm only
    int at_reset;    // comm-only: GE branch selector
    int n_pad, p_pad;
    int warp_bytes;  // dynamic shared memory per environment group
    int group;       // lanes per environment: 4, 8, 16 or 32
};

// per-warp scratch carved out of dynamic shared memory
struct Scratch {
    u64 *occA;       // [G] agent rows
    u64 *occB;       // [G] prey rows (PredatorPrey) / visited rows (Coverage)
    uint32_t *win;   // [6][n_pad] per agent: 3 words of packed window bits, 3 scalar features (float bits)
    uint16_t *posA;  // [n_pad]
    uint16_t *posP;  // [p_pad]
    uint8_t *alive;  // [p_pad]
    int8_t *act;     // [n_pad]
    uint8_t *kcnt;   // [p_pad] agents around prey j
    int8_t *mv;      // [p_pad] screened random move of prey j
    // parallel move resolution (resolve_agents / resolve_preys)
    u64 *x1, *x2, *x3;   // [G] each: cells that may change / cells targeted once / cells targeted more than once
    uint16_t *tgtA;  // [n_pad] target cell of agent i (0xFFFF: does not try to move)
    uint16_t *finA;  // [n_pad] position of agent i after its turn
    uint16_t *tgtP;  // [p_pad]
    uint16_t *finP;  // [p_pad]
    uint8_t *alvF;   // [p_pad] prey j alive after its turn
    uint8_t *slow;   // [max(n_pad, p_pad)] entity must be resolved in index order
};

__host__ __device__ inline int env_warp_bytes(int n_pad, int p_pad, int G)
{
    const int base = 2 * G * 8 + 6 * n_pad * 4 + n_pad * 2 + p_pad * 2 + p_pad + n_pad + p_pad + p_pad;
#if CM_ENV_PARALLEL_MOVES
    return base + 3 * G * 8 + 2 * n_pad * 2 + 2 * p_pad * 2 + p_pad + (n_pad > p_pad ? n_pad : p_pad);
#else
    return base;                                   // the scratch of the parallel move resolution is not carved out
#endif
}

__device__ __forceinline__ Scratch carve(unsigned char *base, int n_pad, int p_pad, int G)
{
    Scratch s;
    s.occA = reinterpret_cast<u64 *>(base);
    s.occB = s.occA + G;
#if CM_ENV_PARALLEL_MOVES
    s.x1 = s.occB + G;
    s.x2 = s.x1 + G;
    s.x3 = s.x2 + G;
    s.win = reinterpret_cast<uint32_t *>(s.x3 + G);
    s.posA = reinterpret_cast<uint16_t *>(s.win + 6 * n_pad);
    s.tgtA = s.posA + n_pad;
    s.finA = s.tgtA + n_pad;
    s.posP = s.finA + n_pad;
    s.tgtP = s.posP + p_pad;
    s.finP = s.tgtP + p_pad;
    s.alive = reinterpret_cast<uint8_t *>(s.finP + p_pad);
#else
    s.x1 = s.x2 = s.x3 = nullptr;
    s.tgtA = s.finA = s.tgtP = s.finP = nullptr;
    s.win = reinterpret_cast<uint32_t *>(s.occB + G);
    s.posA = reinterpret_cast<uint16_t *>(s.win + 6 * n_pad);
    s.posP = s.posA + n_pad;
    s.alive = reinterpret_cast<uint8_t *>(s.posP + p_pad);
#endif
    s.act = reinterpret_cast<int8_t *>(s.alive + p_pad);
    s.kcnt = reinterpret_cast<uint8_t *>(s.act + n_pad);
    s.mv = reinterpret_cast<int8_t *>(s.kcnt + p_pad);
#if CM_ENV_PARALLEL_MOVES
    s.alvF = reinterpret_cast<uint8_t *>(s.mv + p_pad);
    s.slow = s.alvF + p_pad;
#else
    s.alvF = s.slow = nullptr;
#endif
    return s;
}

// set bit c of row r from several lanes at once: native 32-bit shared-memory atomics on the row's halves
__device__ __forceinline__ void set_bit(u64 *rows, int r, int c)
{
    atomicOr(reinterpret_cast<unsigned int *>(rows + r) + (c >> 5), 1u << (c & 31));
}

// action -> displacement: 0 down(+row) 1 left(-col) 2 up(-row) 3 right(+col) 4 noop
// (predator_prey.py:240-253,640-646; coverage.py:336-345)
__device__ __forceinline__ int d_row(int a) { return a == 0 ? 1 : (a == 2 ? -1 : 0); }
__device__ __forceinline__ int d_col(int a) { return a == 3 ? 1 : (a == 1 ? -1 : 0); }

__device__ __forceinline__ int bit_at(const u64 *rows, int r, int c, int G)
{
    return (r >= 0 && r < G && c >= 0 && c < G) ? (int)((rows[r] >> c) & 1ull) : 0;
}

// entities of `rows` in the 4-neighbourhood of (r,c); (r,c) itself may lie outside the grid, each
// neighbour is bounds-checked on its own (predator_prey.py:309-329).
__device__ __forceinline__ int count4(const u64 *rows, int r, int c, int G)
{
    return bit_at(rows, r + 1, c, G) + bit_at(rows, r - 1, c, G) + bit_at(rows, r, c + 1, G) + bit_at(rows, r, c - 1, G);
}

// (2R+1) bits of row `r` centred on column c, LSB = column c-R; cells outside the grid read `oob`.
__device__ __forceinline__ uint32_t window_row(const u64 *rows, int r, int c, int R, int G, int oob)
{
    const uint32_t mask = (1u << (2 * R + 1)) - 1u;
    if (r < 0 || r >= G) return oob ? mask : 0u;
    u64 v = rows[r];
    if (oob) v |= ~((G >= 64) ? ~0ull : ((1ull << G) - 1ull));  // columns >= G
    int sh = c - R;
    uint32_t seg;
    if (sh >= 0) seg = (uint32_t)(v >> sh);
    else {
        seg = (uint32_t)(v << (-sh));
        if (oob) seg |= (1u << (-sh)) - 1u;                      // columns < 0
    }
    return seg & mask;
}

__device__ __forceinline__ uint32_t window_bits(const u64 *rows, int r, int c, int R, int G, int oob)
{
    const int w = 2 * R + 1;
    uint32_t bits = 0;
    for (int dr = 0; dr < w; ++dr) bits |= window_row(rows, r - R + dr, c, R, G, oob) << (dr * w);
    return bits;
}

// ------------------------------------------------------------------------------------------------
// random streams (generated mode): Philox4x32-10 keyed by (seed; env id, tick, stream|episode<<8, index)
// ------------------------------------------------------------------------------------------------
struct RngKey {
    uint32_t env, tick, episode;
    uint2 key;
};

__device__ __forceinline__ uint4 rng_block(const RngKey &k, uint32_t stream, uint32_t index)
{
    return philox4x32_10(make_uint4(k.env, k.tick, stream | (k.episode << 8), index), k.key);
}

// A group of `gs` consecutive lanes (4, 8, 16 or 32) owns one environment: small teams pack several envs into a warp.
// Groups of the same warp follow different control flow (different trip counts, resets), so every warp-level
// primitive below is restricted to the group's own lanes.
struct Grp {
    int gs, gl;          // group size, lane index inside the group
    unsigned mask;       // the group's lanes
    __device__ __forceinline__ void sync() const { __syncwarp(mask); }
    __device__ __forceinline__ int sum(int v) const
    {
        for (int o = gs >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o);
        return v;
    }
    __device__ __forceinline__ int any(int pred) const { return __any_sync(mask, pred); }
    // bit k = predicate of the group's lane k
    __device__ __forceinline__ unsigned ballot(int pred) const { return (__ballot_sync(mask, pred) & mask) >> (__ffs(mask) - 1); }
    __device__ __forceinline__ int bcast0(int v) const { return __shfl_sync(mask, v, 0, gs); }
};

struct ChanSrc {
    const float *u;  // injected planes of this env, or nullptr
    RngKey key;
    int n;
    uint32_t cached_idx;
    uint4 cached;
    __device__ __forceinline__ float draw(int plane, int i, int j)
    {
        if (u) return __ldg(u + ((size_t)plane * n + i) * n + j);
        uint32_t q = (uint32_t)((plane * n + i) * n + j);
        if ((q >> 2) != cached_idx) {
            cached_idx = q >> 2;
            cached = rng_block(key, kStreamChan, cached_idx);
        }
        uint32_t w = (q & 3) == 0 ? cached.x : ((q & 3) == 1 ? cached.y : ((q & 3) == 2 ? cached.z : cached.w));
        return u24(w);
    }
};

// 32 links of one row: bit jj = ((u(plane, i, 32 w + jj) + [i == j]) < thr) if kLess else (... >= thr).  Generated mode
// walks the Philox blocks that cover the row (4 draws per block) instead of testing a block cache per draw.
template <bool kLess>
__device__ __forceinline__ uint32_t link_row_bits(ChanSrc &src, int plane, int i, int w, int jn, float thr)
{
    uint32_t bits = 0;
    const int n = src.n;
    if (src.u) {
        for (int jj = 0; jj < jn; ++jj) {
            const int j = w * 32 + jj;
            const float v = __fadd_rn(__ldg(src.u + ((size_t)plane * n + i) * n + j), (i == j) ? 1.0f : 0.0f);
            bits |= (uint32_t)(kLess ? (v < thr) : (v >= thr)) << jj;
        }
        return bits;
    }
    const uint32_t q0 = (uint32_t)((plane * n + i) * n + w * 32), q1 = q0 + (uint32_t)jn;   // draw indices [q0, q1)
    // Thresholds inside (0, 1) — every probability but the degenerate ones — compare as INTEGERS: a draw is u = k 2^-24 with
    // k = word >> 8 (exact in fp32), so u >= thr <=> k >= ceil(thr 2^24) =: T <=> word >= T << 8, and u < thr <=> word < T << 8;
    // the diagonal's u + 1 lies in [1, 2): never below such a threshold, always at or above it.  One compare + select per link
    // instead of convert / scale / add / compare / select; blocks that lie inside the row take four links at once.
    const float t24 = thr * 16777216.0f;
    if (t24 > 0.0f && t24 <= 16777215.0f) {
        const uint32_t tw = (uint32_t)ceilf(t24) << 8;
        for (uint32_t blk = q0 >> 2; blk <= (q1 - 1u) >> 2; ++blk) {
            const uint4 r4 = rng_block(src.key, kStreamChan, blk);
            const uint32_t b4 = (kLess ? (uint32_t)(r4.x < tw) : (uint32_t)(r4.x >= tw)) | (kLess ? (uint32_t)(r4.y < tw) : (uint32_t)(r4.y >= tw)) << 1 |
                                (kLess ? (uint32_t)(r4.z < tw) : (uint32_t)(r4.z >= tw)) << 2 | (kLess ? (uint32_t)(r4.w < tw) : (uint32_t)(r4.w >= tw)) << 3;
            const int sft = (int)(blk * 4u) - (int)q0;                         // position of the block's first draw in the row
            if (sft >= 0 && sft + 4 <= jn) bits |= b4 << sft;
            else {
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (sft + k >= 0 && sft + k < jn) bits |= ((b4 >> k) & 1u) << (sft + k);
            }
        }
        if ((i >> 5) == w) bits = kLess ? bits & ~(1u << (i & 31)) : bits | (1u << (i & 31));
        return bits;
    }
    for (uint32_t blk = q0 >> 2; blk <= (q1 - 1u) >> 2; ++blk) {
        const uint4 r4 = rng_block(src.key, kStreamChan, blk);
        const uint32_t ws[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t q = blk * 4u + (uint32_t)k;
            if (q >= q0 && q < q1) {
                const int jj = (int)(q - q0);
                const float v = __fadd_rn(u24(ws[k]), (i == w * 32 + jj) ? 1.0f : 0.0f);
                bits |= (uint32_t)(kLess ? (v < thr) : (v >= thr)) << jj;
            }
        }
    }
    return bits;
}

// ------------------------------------------------------------------------------------------------
// communication state: get_graph + channels (env_communication.py:91-157,200-243)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void comm_update(const EnvArgs &A, const Scratch &S, int64_t b, const Grp &G, const RngKey &key, bool at_reset)
{
    const cm_env_desc &d = A.d;
    const int n = d.n_agents, L = d.n_layers, W = (n + 31) >> 5;
    // adjacency rows: dr^2 + dc^2 <= 2 Rcom^2 (== cdist <= sqrt(2 Rcom^2) on integer coordinates, :230);
    // Rcom == 0 means fully connected (:219-223)
    int deg = 0;
    for (int item = G.gl; item < n * W; item += G.gs) {
        const int i = item / W, w = item - i * W;
        uint32_t bits = 0;
        const int jn = min(32, n - w * 32);
        if (d.rcom2 < 0) bits = jn == 32 ? 0xFFFFFFFFu : ((1u << jn) - 1u);
        else {
            const int ri = S.posA[i] & 0xFF, ci = S.posA[i] >> 8;
            for (int jj = 0; jj < jn; ++jj) {
                const uint16_t pj = S.posA[w * 32 + jj];
                const int dr = ri - (pj & 0xFF), dc = ci - (pj >> 8);
                bits |= (uint32_t)(dr * dr + dc * dc <= d.rcom2) << jj;
            }
        }
        deg += __popc(bits);
        if (A.io.adj_bits) A.io.adj_bits[(b * n + i) * W + w] = bits;
    }
    if (A.io.ave_deg) {
        deg = G.sum(deg);
        // float32 dist_adj.sum(axis=1).mean(axis=0) (:232); the fully connected branch returns n (:221)
        if (G.gl == 0) A.io.ave_deg[b] = d.rcom2 < 0 ? (float)n : __fdiv_rn((float)deg, (float)n);
    }
    if (!A.io.chan_bits && d.channel != CM_CH_GE) return;
    uint32_t *out = A.io.chan_bits ? A.io.chan_bits + (size_t)b * L * n * W : nullptr;
    ChanSrc src;
    src.u = A.io.chan_u ? A.io.chan_u + (size_t)b * A.io.chan_planes * n * n : nullptr;
    src.key = key;
    src.n = n;
    src.cached_idx = 0xFFFFFFFFu;
    if (d.channel == CM_CH_FC || d.channel == CM_CH_FL) {                    // :93-100
        for (int item = G.gl; item < L * n * W; item += G.gs) {
            const int w = item % W, i = (item / W) % n;
            const int jn = min(32, n - w * 32);
            uint32_t bits = jn == 32 ? 0xFFFFFFFFu : ((1u << jn) - 1u);
            if (d.channel == CM_CH_FL) bits = ((i >> 5) == w) ? (1u << (i & 31)) : 0u;
            out[item] = bits;
        }
    } else if (d.channel == CM_CH_IID) {                                      // get_iid_channel :200-214
        for (int item = G.gl; item < L * n * W; item += G.gs) {
            const int w = item % W, i = (item / W) % n, l = item / (W * n);
            const int jn = min(32, n - w * 32);
            out[item] = link_row_bits<false>(src, l, i, w, jn, d.p_loss);
        }
    } else {                                                                   // GE :106-157
        uint32_t *state = A.s.ge_state + (size_t)b * n * W;
        for (int item = G.gl; item < n * W; item += G.gs) {
            const int i = item / W, w = item - i * W;
            const int jn = min(32, n - w * 32);
            const uint32_t full = jn == 32 ? 0xFFFFFFFFu : ((1u << jn) - 1u);
            uint32_t st;
            int plane = 0, first_layer = 0;
            if (at_reset) {
                if (d.ge_init == 1) st = full;
                else if (d.ge_init == 0) st = 0u;
                else {                                  // get_init_state, gilbert_elliot_loss_model.py:84-87
                    st = 0u;
                    for (int jj = 0; jj < jn; ++jj) st |= (uint32_t)(src.draw(0, i, w * 32 + jj) >= d.ge_bad_rate) << jj;
                    plane = 1;
                }
                if (d.loss_apply == 0) {
                    if (out) for (int l = 0; l < L; ++l) out[(l * n + i) * W + w] = st;
                    state[item] = st;
                    continue;
                }
                if (out) out[(0 * n + i) * W + w] = st;  // include_prev=True: layer 0 is the initial state
                first_layer = 1;
            } else {
                st = state[item];
            }
            const int n_trans = d.loss_apply == 0 ? 1 : L - first_layer;
            for (int tr = 0; tr < n_trans; ++tr) {      // get_next_state_matrix :137-148: g2b draw, then b2g draw
                const uint32_t g2b = link_row_bits<true>(src, plane, i, w, jn, d.pgb);
                const uint32_t b2g = link_row_bits<true>(src, plane + 1, i, w, jn, d.pbg);
                plane += 2;
                st = (st & ~(st & g2b)) | (~st & b2g & full);
                if (out) {
                    if (d.loss_apply == 0) for (int l = 0; l < L; ++l) out[(l * n + i) * W + w] = st;
                    else out[((first_layer + tr) * n + i) * W + w] = st;
                }
            }
            state[item] = st;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// reset / spawn (predator_prey.py:150-171,206-232; coverage.py:172-196,221-246)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void reset_env(const EnvArgs &A, const Scratch &S, const u64 *wall, int64_t b, const Grp &G,
                          RngKey &key, int &t, int &total_capture)
{
    const cm_env_desc &d = A.d;
    const int n = d.n_agents, p = d.n_preys, Gd = d.grid;
    const bool co = d.scenario == CM_COVERAGE;
    for (int r = G.gl; r < Gd; r += G.gs) { S.occA[r] = 0ull; S.occB[r] = 0ull; }
    G.sync();
    if (A.io.spawn_agent) {
        int ep = (int)key.episode;
        if (ep >= A.io.spawn_episodes) {          // queue exhausted: flag it, reuse the last entry
            if (G.gl == 0 && A.io.error_flag) atomicExch(A.io.error_flag, (int)CM_EINVAL);
            ep = A.io.spawn_episodes - 1;
        }
        for (int i = G.gl; i < n; i += G.gs) {
            const uint16_t q = A.io.spawn_agent[((size_t)b * A.io.spawn_episodes + ep) * n + i];
            S.posA[i] = q;
            set_bit(S.occA, q & 0xFF, q >> 8);
            if (co) set_bit(S.occB, q & 0xFF, q >> 8);                // coverage.py:188 start cells are visited
        }
        for (int j = G.gl; j < p; j += G.gs) {
            const uint16_t q = A.io.spawn_prey[((size_t)b * A.io.spawn_episodes + ep) * p + j];
            S.posP[j] = q;
            S.alive[j] = 1;
            set_bit(S.occB, q & 0xFF, q >> 8);
        }
    } else if (G.gl == 0) {
        // sequential rejection sampling on one lane; a reset happens once per episode, not per step
        const int lo = co ? 1 : 0, span = co ? Gd - 2 : Gd;
        uint32_t ctr = 0;
        uint4 blk = make_uint4(0, 0, 0, 0);
        auto draw = [&](int &r, int &c) {
            if ((ctr & 1u) == 0) blk = rng_block(key, kStreamSpawn, ctr >> 1);
            const uint32_t wr = (ctr & 1u) ? blk.z : blk.x, wc = (ctr & 1u) ? blk.w : blk.y;
            ++ctr;
            r = lo + (int)__umulhi(wr, (uint32_t)span);
            c = lo + (int)__umulhi(wc, (uint32_t)span);
        };
        for (int i = 0; i < n; ++i) {
            int r = 0, c = 0;
            for (int tries = 0; tries <= (1 << 20); ++tries) {
                draw(r, c);
                const u64 busy = S.occA[r] | (co ? wall[r] : 0ull);
                if (!((busy >> c) & 1ull)) break;
            }
            S.posA[i] = (uint16_t)(r | (c << 8));
            S.occA[r] |= 1ull << c;
            if (co) S.occB[r] |= 1ull << c;
        }
        for (int j = 0; j < p; ++j) {
            int r = 0, c = 0;
            for (int tries = 0; tries <= (1 << 20); ++tries) {
                draw(r, c);
                // vacant and no agent in the 4-neighbourhood (predator_prey.py:166)
                if (!(((S.occA[r] | S.occB[r]) >> c) & 1ull) && count4(S.occA, r, c, Gd) == 0) break;
            }
            S.posP[j] = (uint16_t)(r | (c << 8));
            S.alive[j] = 1;
            S.occB[r] |= 1ull << c;
        }
    }
    G.sync();
    t = 0;
    total_capture = 0;
    key.episode += 1;
}

// ------------------------------------------------------------------------------------------------
// observations (predator_prey.py:173-204; coverage.py:198-212,448-480)
// ------------------------------------------------------------------------------------------------
// Phase 1, one lane per agent: the windows are extracted into registers and packed into ONE bit string per agent
// (window after window, <= 75 bits -> 3 words) next to the agent's 3 scalar features.  Phase 2: the env's [n][D] block is
// contiguous, so the group streams it out flat — consecutive lanes store consecutive floats (fully coalesced), one
// shift + mask + convert per float, no divergent select chain.
__device__ __forceinline__ void write_obs(const EnvArgs &A, const Scratch &S, const u64 *wall, int64_t b, const Grp &G, int t)
{
    const cm_env_desc &d = A.d;
    if (!A.io.obs && !A.io.obs_bits) return;
    const int n = d.n_agents, Gd = d.grid, R = d.sensing, w = 2 * R + 1, ww = w * w, np_ = A.n_pad;
    const bool co = d.scenario == CM_COVERAGE;
    const int nbits = (co ? 3 : 2) * ww, D = nbits + (co ? 2 : 3);
    const float *lut_row = d.lut, *lut_col = d.lut + Gd, *lut_t = d.lut + 2 * Gd;
    const float ft = co ? 0.0f : __ldg(lut_t + t);
    for (int i = G.gl; i < n; i += G.gs) {
        const int r = S.posA[i] & 0xFF, c = S.posA[i] >> 8;
        const float fr = __ldg(lut_row + r), fc = __ldg(lut_col + c);      // in flight while the windows are extracted
        u64 lo;
        uint32_t hi = 0u;
        if (co) {
            const uint32_t w0 = window_bits(wall, r, c, R, Gd, 1);          // wall channel, out-of-grid = wall (:464-466)
            const uint32_t w1 = window_bits(S.occA, r, c, R, Gd, 0);        // agents, self included
            const uint32_t w2 = window_bits(S.occB, r, c, R, Gd, 0);        // visited
            lo = (u64)w0 | ((u64)w1 << ww) | ((u64)w2 << (2 * ww));
            if (3 * ww > 64) hi = w2 >> (64 - 2 * ww);
        } else {
            const uint32_t w0 = window_bits(S.occA, r, c, R, Gd, 0);        // agents, self included
            const uint32_t w1 = window_bits(S.occB, r, c, R, Gd, 0);        // preys
            lo = (u64)w0 | ((u64)w1 << ww);
        }
        S.win[0 * np_ + i] = (uint32_t)lo;
        S.win[1 * np_ + i] = (uint32_t)(lo >> 32);
        S.win[2 * np_ + i] = hi;
        S.win[3 * np_ + i] = __float_as_uint(fr);
        S.win[4 * np_ + i] = __float_as_uint(fc);
        S.win[5 * np_ + i] = __float_as_uint(ft);
    }
    G.sync();
    if (A.io.obs_bits) {                          // the packed form (24 bytes per agent), for cm_policy_forward
        uint32_t *ob = A.io.obs_bits + (size_t)b * n * 6;
        for (int e = G.gl; e < n * 6; e += G.gs) {
            const int i = e / 6, wd = e - i * 6;
            ob[e] = S.win[wd * np_ + i];
        }
    }
    if (!A.io.obs) return;
    float *out = A.io.obs + (size_t)b * n * D;
    const int total = n * D;
    const uint32_t magic = (uint32_t)((0x100000000ull + (u64)D - 1ull) / (u64)D);   // e / D == umulhi(e, magic) for e < 2^25
    auto value = [&](int i, int k) -> float {                                 // column k of agent i's row
        const int kk = k < nbits ? k : 96 + 32 * (k - nbits);                 // bit index, or the word of the scalar feature
        const uint32_t word = S.win[(kk >> 5) * np_ + i];
        return k < nbits ? (float)((word >> (kk & 31)) & 1u) : __uint_as_float(word);
    };
    // the block is streamed out as 128-bit stores: a lane builds four consecutive floats (agent / column advanced
    // incrementally: one division per four floats), the lanes of a group store consecutive 16-byte pieces; the <= 3 floats
    // before the first 16-byte boundary and after the last one go out as scalars
    const int head = min(total, (int)((4u - (uint32_t)((reinterpret_cast<uintptr_t>(out) >> 2) & 3u)) & 3u));
    const int nv = (total - head) >> 2;
    for (int e = G.gl; e < head; e += G.gs) out[e] = value(0, e);             // (head <= 3 < D)
#pragma unroll 2
    for (int v = G.gl; v < nv; v += G.gs) {
        const int e = head + 4 * v;
        int i = (int)__umulhi((uint32_t)e, magic), k = e - i * D;
        float4 f;
        f.x = value(i, k); if (++k == D) { k = 0; ++i; }
        f.y = value(i, k); if (++k == D) { k = 0; ++i; }
        f.z = value(i, k); if (++k == D) { k = 0; ++i; }
        f.w = value(i, k);
        *reinterpret_cast<float4 *>(out + e) = f;
    }
    for (int e = head + 4 * nv + G.gl; e < total; e += G.gs) {
        const int i = (int)__umulhi((uint32_t)e, magic);
        out[e] = value(i, e - i * D);
    }
}

// ------------------------------------------------------------------------------------------------
// Parallel move resolution.  The reference moves entities ONE AFTER ANOTHER in index order (agents:
// predator_prey.py:497-500,240-261 / coverage.py:330-375; preys: predator_prey.py:417-432 / :460-478), so an entity sees
// its predecessors where they ended up and its successors where they started.  Almost all moves of a step do not interact:
// an entity takes the FAST path — its outcome is read off the occupancy at the start of the loop, all lanes in parallel —
// unless a cell it depends on may change during the loop (it is the position of another entity that may move or vanish,
// or somebody else targets it too); those few are resolved in index order afterwards, each by the whole lane group (every
// lane compares its own entities' positions "at that turn": final for lower indices, initial for higher ones).  The
// interaction test may over-approximate (it ignores index order); the slow path is always exact.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool test_bit(const u64 *rows, uint16_t cell) { return (rows[cell & 0xFF] >> (cell >> 8)) & 1ull; }
// atomically sets the cell's bit, returns whether it was set before
__device__ __forceinline__ bool test_and_set(u64 *rows, uint16_t cell)
{
    const int c = cell >> 8;
    const unsigned bit = 1u << (c & 31);
    return atomicOr(reinterpret_cast<unsigned int *>(rows + (cell & 0xFF)) + (c >> 5), bit) & bit;
}
__device__ __forceinline__ bool adjacent4(uint16_t a, uint16_t b)
{
    const int dr = (int)(a & 0xFF) - (int)(b & 0xFF), dc = (int)(a >> 8) - (int)(b >> 8);
    return dr * dr + dc * dc == 1;
}

// entities in the 4-neighbourhood of the IN-GRID cell (r, c), counted on rows combined on the fly (kOr: a | b, else a & ~b);
// rows carry no bits at columns >= G
template <bool kOr>
__device__ __forceinline__ int count4_in(const u64 *a, const u64 *b, int r, int c, int G)
{
    auto row = [&](int rr) { return kOr ? (a[rr] | b[rr]) : (a[rr] & ~b[rr]); };
    int cnt = __popcll(((row(r) << 1) >> c) & 5ull);
    if (r > 0) cnt += (int)((row(r - 1) >> c) & 1ull);
    if (r + 1 < G) cnt += (int)((row(r + 1) >> c) & 1ull);
    return cnt;
}

// Agents of one env.  `fixed` = rows of the cells that block a move and do not change while agents move (PredatorPrey: the
// preys; Coverage: the walls).  On return S.finA holds every agent's position after the loop (S.posA still the initial one)
// and S.tgtA its target (0xFFFF: NOOP, or a move off the grid when !count_oob).  Returns this lane's number of movers that were blocked
// (Coverage's penalty count; moves off the grid included).
__device__ __forceinline__ int resolve_agents(const Scratch &S, const Grp &G, int n, int Gd, const u64 *fixed)
{
    for (int r = G.gl; r < Gd; r += G.gs) { S.x1[r] = 0ull; S.x2[r] = 0ull; S.x3[r] = 0ull; }
    G.sync();
    int blocked = 0;
#pragma unroll 1
    for (int i = G.gl; i < n; i += G.gs) {
        const int a = S.act[i];
        const uint16_t q = S.posA[i];
        uint16_t tg = 0xFFFF;
        if (a != 4) {
            const int nr = (q & 0xFF) + d_row(a), nc = (q >> 8) + d_col(a);
            if (nr >= 0 && nr < Gd && nc >= 0 && nc < Gd) tg = (uint16_t)(nr | (nc << 8));
            else ++blocked;
        }
        S.tgtA[i] = tg;
        S.finA[i] = q;
        if (tg != 0xFFFF) {
            set_bit(S.x1, q & 0xFF, q >> 8);                       // a mover's cell may become free
            if (test_and_set(S.x2, tg)) set_bit(S.x3, tg & 0xFF, tg >> 8);   // targeted more than once
        }
    }
    G.sync();
#pragma unroll 1
    for (int i = G.gl; i < n; i += G.gs) {
        const uint16_t tg = S.tgtA[i];
        bool slow = false;
        if (tg != 0xFFFF) {
            slow = test_bit(S.x1, tg) || test_bit(S.x3, tg);
            if (!slow) {                                           // nobody else touches the target: the initial occupancy decides
                if (test_bit(S.occA, tg) || test_bit(fixed, tg)) ++blocked;
                else S.finA[i] = tg;
            }
        }
        S.slow[i] = slow;
    }
    G.sync();
#pragma unroll 1
    for (int base = 0; base < n; base += G.gs) {
        unsigned m = G.ballot(base + G.gl < n && S.slow[base + G.gl]);
        while (m) {
            const int is = base + __ffs(m) - 1;
            m &= m - 1;
            const uint16_t tg = S.tgtA[is];
            int hit = 0;
#pragma unroll 1
            for (int k = G.gl; k < n; k += G.gs)
                if (k != is) hit |= (k > is ? S.posA[k] : S.finA[k]) == tg;
            const bool free = !G.any(hit) && !test_bit(fixed, tg);
            if (G.gl == (is & (G.gs - 1))) {
                if (free) S.finA[is] = tg;
                else ++blocked;
            }
            G.sync();
        }
    }
    return blocked;
}

// Preys of one env (PredatorPrey), after the agents have moved (S.occA final) and S.kcnt / S.mv have been computed.  On
// return S.finP / S.alvF hold every prey's position / alive flag after the loop.  Returns this lane's (captures | penalties << 16).
__device__ __forceinline__ int resolve_preys(const Scratch &S, const Grp &G, int p, int Gd, int load)
{
    for (int r = G.gl; r < Gd; r += G.gs) { S.x1[r] = 0ull; S.x2[r] = 0ull; S.x3[r] = 0ull; }
    G.sync();
#pragma unroll 1
    for (int j = G.gl; j < p; j += G.gs) {
        const uint16_t q = S.posP[j];
        uint16_t tg = 0xFFFF;
        const int al = S.alive[j];
        if (al) {
            const int mv = S.mv[j];
            if (mv != 4) {
                const int nr = (q & 0xFF) + d_row(mv), nc = (q >> 8) + d_col(mv);
                if (nr >= 0 && nr < Gd && nc >= 0 && nc < Gd) tg = (uint16_t)(nr | (nc << 8));
            }
            if (S.kcnt[j] >= 1 || tg != 0xFFFF) set_bit(S.x1, q & 0xFF, q >> 8);     // may be captured or walk away
            if (tg != 0xFFFF && test_and_set(S.x2, tg)) set_bit(S.x3, tg & 0xFF, tg >> 8);
        }
        S.tgtP[j] = tg;
        S.finP[j] = q;
        S.alvF[j] = (uint8_t)al;
    }
    G.sync();
    // capture rule of one prey given the preys around it (:419-431 / :462-477; edges dict :123-144)
    auto need_of = [&](int r, int c, int prey_nb) {
        if (load == 2) return load;
        const int re = (r == 0 || r == Gd - 1), ce = (c == 0 || c == Gd - 1);
        const int nadj = (re && ce) ? 2 : ((re || ce) ? 3 : load);
        return min(load, nadj - prey_nb);
    };
    int capture = 0, penalty = 0;
#pragma unroll 1
    for (int j = G.gl; j < p; j += G.gs) {
        bool slow = false;
        if (S.alive[j]) {
            const uint16_t q = S.posP[j], tg = S.tgtP[j];
            const int r = q & 0xFF, c = q >> 8, k = S.kcnt[j];
            // Captured or not (only preys next to an agent are tested)?  The rule of reward_individual looks at the preys
            // around this one, which may change during the loop; its outcome is fixed anyway when it is the same for the
            // FEWEST preys that can be around (those that surely stay) and for the MOST (every cell a prey stands on or walks
            // to — its own target, one of the four cells, does not count unless it is somebody else's too)
            int state = 0;                                         // 0 stays, 1 captured, 2 depends on the order
            if (k >= 1) {
                if (load == 2) state = 1;                          // reward_default: need = load = 2 <= k ... see below
                else {
                    const int own = (tg != 0xFFFF && !test_bit(S.occB, tg) && !test_bit(S.x3, tg)) ? 1 : 0;
                    const int most = count4_in<true>(S.occB, S.x2, r, c, Gd) - own, fewest = count4_in<false>(S.occB, S.x1, r, c, Gd);
                    const bool cap_most = need_of(r, c, most) <= k, cap_fewest = need_of(r, c, fewest) <= k;
                    state = cap_most == cap_fewest ? (int)cap_most : 2;
                }
                if (load == 2) state = load <= k;
            }
            const bool walk_slow = tg != 0xFFFF && (test_bit(S.x1, tg) || test_bit(S.x3, tg));
            slow = state == 2 || (state == 0 && walk_slow);
            if (!slow) {
                if (state == 1) { ++capture; S.alvF[j] = 0; }
                else {
                    penalty += k >= 1;
                    if (tg != 0xFFFF && !test_bit(S.occA, tg) && !test_bit(S.occB, tg)) S.finP[j] = tg;
                }
            }
        }
        S.slow[j] = slow;
    }
    G.sync();
#pragma unroll 1
    for (int base = 0; base < p; base += G.gs) {
        unsigned m = G.ballot(base + G.gl < p && S.slow[base + G.gl]);
        while (m) {
            const int js = base + __ffs(m) - 1;
            m &= m - 1;
            const uint16_t q = S.posP[js], tg = S.tgtP[js];
            const int r = q & 0xFF, c = q >> 8, k = S.kcnt[js];
            int around = 0, hit = 0;
#pragma unroll 1
            for (int o = G.gl; o < p; o += G.gs) {
                if (o == js) continue;
                const bool al = o > js ? S.alive[o] != 0 : S.alvF[o] != 0;
                const uint16_t po = o > js ? S.posP[o] : S.finP[o];
                around += al && adjacent4(po, q);
                hit |= al && po == tg;
            }
            const bool owner = G.gl == (js & (G.gs - 1));
            bool gone = false;
            if (k >= 1) {
                const int prey_nb = load != 2 ? G.sum(around) : 0;
                if (need_of(r, c, prey_nb) <= k) { gone = true; if (owner) { ++capture; S.alvF[js] = 0; } }
                else if (owner) ++penalty;
            }
            const bool blocked = G.any(hit) || tg == 0xFFFF || test_bit(S.occA, tg);
            if (owner && !gone && !blocked) S.finP[js] = tg;
            G.sync();
        }
    }
    return capture | (penalty << 16);
}

// ------------------------------------------------------------------------------------------------
// the kernel: mode 0 = VecEnvExecutor.step, 1 = reset(mask), 2 = comm only
// ------------------------------------------------------------------------------------------------
#ifdef CM_ENV_TRACE
#define CM_ETP(k) do { if (blockIdx.x == 0 && threadIdx.x == 0) trace_t[k] = clock64(); } while (0)
#else
#define CM_ETP(k) do { } while (0)
#endif

// Specialised on the scenario, the channel family and whether pre-drawn streams are injected: the kernel is bound by
// instruction FETCH (ncu: 1-3 warps per issue slot wait for instructions; every warp walks a long, divergent path through
// the code of one env), so an instantiation carries only the code of its own scenario / channel / stream source — the
// descriptor fields are overwritten with the template constants and the branches on them fold after inlining.
// kChan: 0 = FC / FL (told apart at run time), CM_CH_IID, CM_CH_GE, or kChanTable: every env reads its own channel condition
// (cm_env_desc.conds) and comm_update branches on its channel at run time; that code lives in its own instantiations only.
static constexpr int kChanTable = 4;
template <int kScen, int kChan, bool kInj>
__global__ void __launch_bounds__(kWarpsPerCta * 32, 24 / kWarpsPerCta) env_kernel(const EnvArgs A_in)
{
    EnvArgs A = A_in;
    A.d.scenario = kScen;
    if (kChan == 0) { if (A.d.channel != CM_CH_FL) A.d.channel = CM_CH_FC; }
    else if (kChan != kChanTable) A.d.channel = kChan;
    if (kScen == CM_COVERAGE) { A.d.n_preys = 0; A.s.prey_pos = nullptr; A.s.prey_alive = nullptr; }
    if (!kInj) { A.io.prey_cand = nullptr; A.io.chan_u = nullptr; A.io.spawn_agent = nullptr; A.io.spawn_prey = nullptr; }
#ifdef CM_ENV_TRACE
    long long trace_t[12] = {0};
#endif
    CM_ETP(0);
    extern __shared__ __align__(16) unsigned char smem[];
    const cm_env_desc &d = A.d;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    Grp G;
    G.gs = A.group;
    G.gl = lane & (A.group - 1);
    G.mask = A.group == 32 ? 0xFFFFFFFFu : (((1u << A.group) - 1u) << (lane - G.gl));
    const int epw = 32 / A.group, grp = lane / A.group;          // envs per warp, this lane's group
    const int n = d.n_agents, p = d.n_preys, Gd = d.grid;
    const bool co = d.scenario == CM_COVERAGE;
    u64 *wall = reinterpret_cast<u64 *>(smem);               // [Gd] shared by the CTA (Coverage)
    double *mean_lut = reinterpret_cast<double *>(smem + 64 * 8);   // k / n, correctly rounded: mean(x) = sum / len (coverage.py:601-602)
    if (co) {
        for (int r = threadIdx.x; r < Gd; r += blockDim.x) wall[r] = d.wall_rows[r];
        for (int k = threadIdx.x; k <= n; k += blockDim.x) mean_lut[k] = __ddiv_rn((double)k, (double)n);
    }
    __syncthreads();
    CM_ETP(1);
    const Scratch S = carve(smem + kConstBytes + (size_t)(warp * epw + grp) * A.warp_bytes, A.n_pad, A.p_pad, Gd);
    const int64_t stride = (int64_t)gridDim.x * kWarpsPerCta * epw;
    for (int64_t b = ((int64_t)blockIdx.x * kWarpsPerCta + warp) * epw + grp; b < A.s.n_envs; b += stride) {
        if (A.mode == 1 && A.mask && !A.mask[b]) continue;
        G.sync();
        RngKey key;
        key.env = (uint32_t)(d.env_id0 + b);
        key.key = make_uint2((uint32_t)d.seed, (uint32_t)(d.seed >> 32));
        key.tick = A.s.tick[b];
        key.episode = A.s.episode[b];
        int t = A.s.step_count[b];
        int total_capture = co ? A.s.total_capture[b] : 0;
        bool did_reset = false;
        // every global read of this env is issued here, in one batch: the state, the actions, the success latch and the
        // running episode accumulators (used only at the end of the step) — one memory round trip instead of four
        uint8_t success = 0;
        double run7[7] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        int moved = 0, bad = 0;
        CM_ETP(2);

        bool do_reset = A.mode == 1;              // (reset_env has ONE call site, after the step logic: code size)
        if (!do_reset) {
            // ---- stage the env in shared memory and rebuild the row bitmaps from the positions ----
            for (int r = G.gl; r < Gd; r += G.gs) { S.occA[r] = 0ull; S.occB[r] = co ? A.s.visited[b * Gd + r] : 0ull; }
            for (int i = G.gl; i < n; i += G.gs) S.posA[i] = A.s.agent_pos[b * n + i];
            for (int j = G.gl; j < p; j += G.gs) { S.posP[j] = A.s.prey_pos[b * p + j]; S.alive[j] = A.s.prey_alive[b * p + j]; }
            if (A.mode == 0) {
                success = A.s.success[b];
                if (G.gl == 0 && A.io.stats) {
#pragma unroll
                    for (int k = 0; k < 7; ++k) run7[k] = A.io.stats[b * 16 + k];
                }
                for (int i = G.gl; i < n; i += G.gs) {
                    int a = A.io.actions[b * n + i];
                    if (a < 0 || a > 4) { bad = 1; a = 4; }
                    S.act[i] = (int8_t)a;
                    moved += (a != 4);
                }
            }
            G.sync();
            for (int i = G.gl; i < n; i += G.gs) set_bit(S.occA, S.posA[i] & 0xFF, S.posA[i] >> 8);
            for (int j = G.gl; j < p; j += G.gs)
                if (S.alive[j]) set_bit(S.occB, S.posP[j] & 0xFF, S.posP[j] >> 8);
            G.sync();
        }

        CM_ETP(3);
        if (A.mode == 0) {
            // =================================== env.step ===================================
            t += 1;
            key.tick += 1;                        // every draw of this step is keyed with the new tick
            moved = G.sum(moved);
            if (G.any(bad) && G.gl == 0 && A.io.error_flag) atomicExch(A.io.error_flag, (int)CM_EACTION);
            CM_ETP(4);
            int c0 = 0, c2 = 0, c3 = 0, c4 = 0;   // counts (see commarl_b200.h)
            double reward = 0.0;
            int env_done = 0;
#if CM_ENV_PARALLEL_MOVES
            // ---- agents move one after another, lower index first (predator_prey.py:497-500,240-261; coverage.py:330-375):
            // resolved in parallel, exactly (resolve_agents); PredatorPrey's preys stand still meanwhile, Coverage's walls always ----
            const int blocked_moves = resolve_agents(S, G, n, Gd, co ? wall : S.occB);
#endif
            if (!co) {
#if CM_ENV_PARALLEL_MOVES
                for (int r = G.gl; r < Gd; r += G.gs) S.occA[r] = 0ull;
                G.sync();
                for (int i = G.gl; i < n; i += G.gs) {
                    const uint16_t q = S.finA[i];
                    S.posA[i] = q;
                    set_bit(S.occA, q & 0xFF, q >> 8);
                }
                G.sync();
#else
                // ---- agents move one after another, lower index first (predator_prey.py:497-500,240-261) ----
                if (G.gl == 0) {
                    // the action and position of agent i + 1 are loaded while agent i is resolved: the only loop-carried
                    // dependency left is the occupancy rows themselves
                    int a_nx = S.act[0];
                    uint16_t q_nx = S.posA[0];
                    for (int i = 0; i < n; ++i) {
                        const int a = a_nx;
                        const uint16_t q = q_nx;
                        if (i + 1 < n) { a_nx = S.act[i + 1]; q_nx = S.posA[i + 1]; }
                        if (a == 4) continue;
                        const int r = q & 0xFF, c = q >> 8;
                        const int nr = r + d_row(a), nc = c + d_col(a);
                        if (nr < 0 || nr >= Gd || nc < 0 || nc >= Gd) continue;
                        if (((S.occA[nr] | S.occB[nr]) >> nc) & 1ull) continue;
                        S.occA[r] &= ~(1ull << c);
                        S.occA[nr] |= 1ull << nc;
                        S.posA[i] = (uint16_t)(nr | (nc << 8));
                    }
                }
                G.sync();
#endif
                // ---- order-independent part of the prey loop, lane-parallel ----
                // Agents stand still while preys are processed, and prey j's own position / alive flag only
                // change in its own turn, so: the agent count around prey j (:419/:462), the screening of its
                // <= 5 move candidates against agent neighbourhoods (:400-404) and the prey_watching flags
                // (:421-422) do not depend on the processing order.
                for (int j = G.gl; j < p; j += G.gs) {
                    if (!S.alive[j]) continue;
                    const int r = S.posP[j] & 0xFF, c = S.posP[j] >> 8;
                    S.kcnt[j] = (uint8_t)count4(S.occA, r, c, Gd);
                    uint32_t words[5];
                    if (!A.io.prey_cand) {
                        const uint4 q0 = rng_block(key, kStreamPrey, 2 * j), q1 = rng_block(key, kStreamPrey, 2 * j + 1);
                        words[0] = q0.x; words[1] = q0.y; words[2] = q0.z; words[3] = q0.w; words[4] = q1.x;
                    }
                    int mv = 4;
                    for (int tr = 0; tr < 5; ++tr) {
                        const int cnd = A.io.prey_cand ? (int)A.io.prey_cand[((size_t)b * p + j) * 5 + tr]
                                                       : prey_move_from_bits(words[tr]);
                        if (count4(S.occA, r + d_row(cnd), c + d_col(cnd), Gd) == 0) { mv = cnd; break; }
                    }
                    S.mv[j] = (int8_t)mv;
                }
                int watching = 0;
                for (int i = G.gl; i < n; i += G.gs)
                    watching += count4(S.occB, S.posA[i] & 0xFF, S.posA[i] >> 8, Gd) > 0;
                c3 = G.sum(watching);
                G.sync();
#if CM_ENV_PARALLEL_MOVES
                // ---- order-dependent part: capture test against the preys still standing, then the walk — resolved in
                // parallel, exactly (resolve_preys) ----
                {
                    const int cp = resolve_preys(S, G, p, Gd, d.load);
                    const int capture = G.sum(cp & 0xFFFF), penalty = G.sum(cp >> 16);
                    c0 = capture;
                    c2 = penalty;
                    for (int r = G.gl; r < Gd; r += G.gs) S.occB[r] = 0ull;
                    G.sync();
                    for (int j = G.gl; j < p; j += G.gs) {
                        const uint16_t q = S.finP[j];
                        const uint8_t al = S.alvF[j];
                        S.posP[j] = q;
                        S.alive[j] = al;
                        if (al) set_bit(S.occB, q & 0xFF, q >> 8);
                    }
                    if (G.gl == 0) {
                        // :434 / :480, fixed left-to-right fp64 evaluation, no contraction
                        reward = __dadd_rn(__dadd_rn(d.step_cost, __dmul_rn(d.capture_reward, (double)capture)),
                                           __ddiv_rn(__dmul_rn(d.moving_cost, (double)moved), (double)n));
                        if (d.load == 2) reward = __dadd_rn(reward, __dmul_rn(d.penalty, (double)penalty));
                    }
                }
                G.sync();
#else
                // ---- order-dependent part: capture test against the preys still standing, then the walk ----
                if (G.gl == 0) {
                    int capture = 0, penalty = 0;
                    // prey j + 1's flags are loaded while prey j is resolved (a prey only changes its own entries)
                    int al_nx = S.alive[0], k_nx = S.kcnt[0], mv_nx = S.mv[0];
                    uint16_t q_nx = S.posP[0];
                    for (int j = 0; j < p; ++j) {
                        const int al = al_nx, k = k_nx, mvj = mv_nx;
                        const uint16_t q = q_nx;
                        if (j + 1 < p) { al_nx = S.alive[j + 1]; k_nx = S.kcnt[j + 1]; mv_nx = S.mv[j + 1]; q_nx = S.posP[j + 1]; }
                        if (!al) continue;
                        const int r = q & 0xFF, c = q >> 8;
                        if (k >= 1) {
                            int need = d.load;
                            if (d.load != 2) {   // reward_individual :469-470; edges dict :123-144 (corner 2, border 3, else load)
                                const int re = (r == 0 || r == Gd - 1), ce = (c == 0 || c == Gd - 1);
                                const int nadj = (re && ce) ? 2 : ((re || ce) ? 3 : d.load);
                                need = min(d.load, nadj - count4(S.occB, r, c, Gd));
                            }
                            if (need <= k) {     // captured: leaves the grid at once (:301)
                                ++capture;
                                S.alive[j] = 0;
                                S.occB[r] &= ~(1ull << c);
                                continue;
                            }
                            ++penalty;
                        }
                        const int mv = mvj;
                        if (mv != 4) {           // __update_prey_pos :276-299
                            const int nr = r + d_row(mv), nc = c + d_col(mv);
                            if (nr >= 0 && nr < Gd && nc >= 0 && nc < Gd && !(((S.occA[nr] | S.occB[nr]) >> nc) & 1ull)) {
                                S.occB[r] &= ~(1ull << c);
                                S.occB[nr] |= 1ull << nc;
                                S.posP[j] = (uint16_t)(nr | (nc << 8));
                            }
                        }
                    }
                    c0 = capture;
                    c2 = penalty;
                    // :434 / :480, fixed left-to-right fp64 evaluation, no contraction
                    reward = __dadd_rn(__dadd_rn(d.step_cost, __dmul_rn(d.capture_reward, (double)capture)),
                                       __ddiv_rn(__dmul_rn(d.moving_cost, (double)moved), (double)n));
                    if (d.load == 2) reward = __dadd_rn(reward, __dmul_rn(d.penalty, (double)penalty));
                }
                G.sync();
#endif
                int any_alive = 0;
                for (int j = G.gl; j < p; j += G.gs) {
                    any_alive |= S.alive[j];
                    if (A.io.prey_alive_out) A.io.prey_alive_out[b * p + j] = S.alive[j];
                }
                any_alive = G.any(any_alive);
                if (t >= d.max_steps || !any_alive) {            // :511-517
                    success = any_alive ? 0 : 1;
                    env_done = 1;
                }
            } else {
#if CM_ENV_PARALLEL_MOVES
                // ---- Coverage.step (coverage.py:319-401): sequential moves over wall | agent rows, resolved in parallel,
                // exactly (resolve_agents).  A cell is entered by at most one agent per step (the first one blocks it), so
                // "new cell or revisit" is read off the visited map as it was before the step ----
                {
                    int pen = blocked_moves, cap = 0, rev = 0;
                    for (int i = G.gl; i < n; i += G.gs) {
                        const uint16_t q = S.finA[i];
                        if (q != S.posA[i]) { if (test_bit(S.occB, q)) ++rev; else ++cap; }
                    }
                    pen = G.sum(pen); cap = G.sum(cap); rev = G.sum(rev);
                    for (int r = G.gl; r < Gd; r += G.gs) S.occA[r] = 0ull;
                    G.sync();                                     // every lane has read the old visited map / agent rows
                    for (int i = G.gl; i < n; i += G.gs) {
                        const uint16_t q = S.finA[i];
                        if (q != S.posA[i]) set_bit(S.occB, q & 0xFF, q >> 8);
                        S.posA[i] = q;
                        set_bit(S.occA, q & 0xFF, q >> 8);
                    }
                    if (G.gl == 0) {
                    const int lazy = n - moved;
                    c0 = cap; c2 = pen; c3 = rev; c4 = lazy;
                    total_capture += cap;
                    double final_reward = 0.0;
                    if (total_capture == d.n_empty_cells) { final_reward = d.final_reward; env_done = 1; }   // :378-382
                    if (t >= d.max_steps) { success = env_done ? 1 : 0; env_done = 1; }                       // :385-390
                    // get_reward :300-306; mean(x) = sum / n comes from the table of correctly rounded k / n
                    reward = __dadd_rn(d.step_cost, __dmul_rn(d.capture_reward, mean_lut[cap]));
                    reward = __dadd_rn(reward, __dmul_rn(d.moving_cost, mean_lut[moved]));
                    reward = __dadd_rn(reward, __dmul_rn(d.penalty, mean_lut[pen]));
                    reward = __dadd_rn(reward, __dmul_rn(d.lazy_penalty, mean_lut[lazy]));
                    reward = __dadd_rn(reward, __dmul_rn(d.revisit_penalty, mean_lut[rev]));
                    reward = __dadd_rn(reward, final_reward);
                    }
                }
#else
                // ---- Coverage.step (coverage.py:319-401): sequential moves over wall | agent rows ----
                if (G.gl == 0) {
                    int cap = 0, pen = 0, rev = 0;
                    int a_nx = S.act[0];
                    uint16_t q_nx = S.posA[0];
                    for (int i = 0; i < n; ++i) {
                        const int a = a_nx;
                        const uint16_t q = q_nx;
                        if (i + 1 < n) { a_nx = S.act[i + 1]; q_nx = S.posA[i + 1]; }
                        if (a == 4) continue;                    // lazy, counted below
                        const int r = q & 0xFF, c = q >> 8;
                        const int nr = r + d_row(a), nc = c + d_col(a);
                        if (nr < 0 || nr >= Gd || nc < 0 || nc >= Gd || (((S.occA[nr] | wall[nr]) >> nc) & 1ull)) { ++pen; continue; }
                        if ((S.occB[nr] >> nc) & 1ull) ++rev;
                        else { S.occB[nr] |= 1ull << nc; ++cap; }
                        S.occA[r] &= ~(1ull << c);
                        S.occA[nr] |= 1ull << nc;
                        S.posA[i] = (uint16_t)(nr | (nc << 8));
                    }
                    const int lazy = n - moved;
                    c0 = cap; c2 = pen; c3 = rev; c4 = lazy;
                    total_capture += cap;
                    double final_reward = 0.0;
                    if (total_capture == d.n_empty_cells) { final_reward = d.final_reward; env_done = 1; }   // :378-382
                    if (t >= d.max_steps) { success = env_done ? 1 : 0; env_done = 1; }                       // :385-390
                    // get_reward :300-306; mean(x) = sum / n comes from the table of correctly rounded k / n
                    reward = __dadd_rn(d.step_cost, __dmul_rn(d.capture_reward, mean_lut[cap]));
                    reward = __dadd_rn(reward, __dmul_rn(d.moving_cost, mean_lut[moved]));
                    reward = __dadd_rn(reward, __dmul_rn(d.penalty, mean_lut[pen]));
                    reward = __dadd_rn(reward, __dmul_rn(d.lazy_penalty, mean_lut[lazy]));
                    reward = __dadd_rn(reward, __dmul_rn(d.revisit_penalty, mean_lut[rev]));
                    reward = __dadd_rn(reward, final_reward);
                }
#endif
                G.sync();
                env_done = G.bcast0(env_done);
                total_capture = G.bcast0(total_capture);
                success = (uint8_t)G.bcast0((int)success);
            }
            CM_ETP(5);
            int done = env_done;
            if (d.max_path_length > 0 && t >= d.max_path_length) done = 1;   // vec_env_executor.py:33-35
            if (G.gl == 0) {
                if (A.io.reward) A.io.reward[b] = reward;
                if (A.io.done) A.io.done[b] = (uint8_t)done;
                if (A.io.counts) {
                    int32_t *cn = A.io.counts + b * 6;
                    cn[0] = c0; cn[1] = moved; cn[2] = c2; cn[3] = c3; cn[4] = c4; cn[5] = 0;
                }
                A.s.success[b] = success;
                if (A.io.success_out) A.io.success_out[b] = success;
                if (A.io.stats) {                 // episode accounting (sampler bookkeeping, ...vectorized_sampler.py:158-227)
                    double *st = A.io.stats + b * 16;
                    const double run[7] = {run7[0] + reward, run7[1] + 1.0, run7[2] + c0, run7[3] + moved, run7[4] + c2, run7[5] + c3, run7[6] + c4};
                    if (done) {
                        st[7] += 1.0; st[8] += run[0]; st[9] += run[1]; st[10] += (double)success;
                        for (int k = 0; k < 5; ++k) st[11 + k] += run[2 + k];
                        for (int k = 0; k < 7; ++k) st[k] = 0.0;
                    } else {
                        for (int k = 0; k < 7; ++k) st[k] = run[k];
                    }
                }
            }
            CM_ETP(6);
            do_reset = done && A.io.auto_reset;   // vec_env_executor.py:36-43
        }
        if (do_reset) {
            reset_env(A, S, wall, b, G, key, t, total_capture);
            did_reset = true;
        }

        CM_ETP(7);
        if (A.mode != 2) {
            // ---- write the state back ----
            for (int i = G.gl; i < n; i += G.gs) A.s.agent_pos[b * n + i] = S.posA[i];
            for (int j = G.gl; j < p; j += G.gs) { A.s.prey_pos[b * p + j] = S.posP[j]; A.s.prey_alive[b * p + j] = S.alive[j]; }
            if (co) for (int r = G.gl; r < Gd; r += G.gs) A.s.visited[b * Gd + r] = S.occB[r];
            if (G.gl == 0) {
                A.s.step_count[b] = t;
                A.s.tick[b] = key.tick;
                A.s.episode[b] = key.episode;
                if (co) A.s.total_capture[b] = total_capture;
            }
            CM_ETP(8);
            write_obs(A, S, wall, b, G, t);
        }
        CM_ETP(9);
        if (kChan == kChanTable) {                // this env's channel condition, loaded once
            int k = A.d.cond_idx[b];
            if (k >= A.d.n_conds) {
                if (G.gl == 0 && A.io.error_flag) atomicExch(A.io.error_flag, (int)CM_EINVAL);
                k = 0;
            }
            const cm_channel_cond c = A.d.conds[k];
            A.d.channel = c.channel;
            A.d.rcom2 = c.rcom2;
            A.d.p_loss = c.p_loss;
            A.d.pgb = c.pgb;
            A.d.pbg = c.pbg;
            A.d.ge_bad_rate = c.ge_bad_rate;
            A.d.ge_init = c.ge_init;
        }
        comm_update(A, S, b, G, key, A.mode == 2 ? (A.at_reset != 0) : did_reset);
        CM_ETP(10);
#ifdef CM_ENV_TRACE
        if (blockIdx.x == 0 && threadIdx.x == 0 && A.io.stats && A.mode == 0) {
            long long *tb = reinterpret_cast<long long *>(A.io.stats);
            for (int k = 0; k < 11; ++k) tb[k] = trace_t[k];
        }
#endif
    }
}

typedef void (*env_kernel_fn)(const EnvArgs);
template <int kScen>
static env_kernel_fn pick_env_kernel_s(int channel, bool inj)
{
    switch (channel) {
    case kChanTable: return inj ? env_kernel<kScen, kChanTable, true> : env_kernel<kScen, kChanTable, false>;
    case CM_CH_IID: return inj ? env_kernel<kScen, CM_CH_IID, true> : env_kernel<kScen, CM_CH_IID, false>;
    case CM_CH_GE: return inj ? env_kernel<kScen, CM_CH_GE, true> : env_kernel<kScen, CM_CH_GE, false>;
    default: return inj ? env_kernel<kScen, 0, true> : env_kernel<kScen, 0, false>;
    }
}
static env_kernel_fn pick_env_kernel(int scenario, int channel, bool inj)
{
    return scenario == CM_COVERAGE ? pick_env_kernel_s<CM_COVERAGE>(channel, inj) : pick_env_kernel_s<CM_PREDATOR_PREY>(channel, inj);
}

// checks of one channel condition; *planes = injected channel planes it draws
static int validate_channel(int channel, int ge_init, int loss_apply, int n_layers, const cm_env_state *s, int *planes)
{
    if (channel < CM_CH_FC || channel > CM_CH_GE) return CM_EINVAL;
    if (channel == CM_CH_GE) {
        if (ge_init == -1 && loss_apply == 0) return CM_EUNSUPPORTED;  // broken in the reference (env_communication.py:121)
        if (!s->ge_state) return CM_EINVAL;
    }
    *planes = channel == CM_CH_IID ? n_layers : (channel == CM_CH_GE ? 2 * n_layers + 1 : 0);
    return CM_OK;
}

static int validate(const cm_env_desc *d, const cm_env_state *s, const cm_step_io *io, int mode)
{
    if (!d || !s || !io) return CM_EINVAL;
    if (s->n_envs < 0) return CM_EINVAL;
    if (d->n_agents < 1 || d->n_agents > CM_MAX_AGENTS || d->n_preys < 0 || d->n_preys > CM_MAX_AGENTS) return CM_EUNSUPPORTED;
    if (d->grid < 2 || d->grid > CM_MAX_GRID || d->sensing < 0 || d->sensing > 2) return CM_EUNSUPPORTED;
    if (d->n_layers < 1 || d->n_layers > CM_MAX_LAYERS) return CM_EUNSUPPORTED;
    if (d->scenario == CM_PREDATOR_PREY) {
        if (d->load < 2 || d->load > 4) return CM_EUNSUPPORTED;          // capv undefined otherwise (predator_prey.py:77-79)
        if (!s->prey_pos || !s->prey_alive) return CM_EINVAL;
    } else if (d->scenario == CM_COVERAGE) {
        if (d->n_preys != 0) return CM_EINVAL;
        if (!d->wall_rows || !s->visited || !s->total_capture) return CM_EINVAL;
    } else return CM_EINVAL;
    int need = 0;   // channel planes an injected chan_u must hold
    if (d->conds) {
        if (!d->conds_host || !d->cond_idx || d->n_conds < 1 || d->n_conds > CM_MAX_CONDS) return CM_EINVAL;
        for (int k = 0; k < d->n_conds; ++k) {
            const cm_channel_cond &c = d->conds_host[k];
            int planes = 0;
            const int rc = validate_channel(c.channel, c.ge_init, d->loss_apply, d->n_layers, s, &planes);
            if (rc) return rc;
            need = planes > need ? planes : need;
        }
    } else {
        const int rc = validate_channel(d->channel, d->ge_init, d->loss_apply, d->n_layers, s, &need);
        if (rc) return rc;
    }
    if (!s->agent_pos || !s->step_count || !s->success || !s->episode || !s->tick) return CM_EINVAL;
    if (!d->lut && (io->obs || io->obs_bits)) return CM_EINVAL;
    if (mode == 0 && !io->actions) return CM_EINVAL;
    if (io->spawn_agent && (io->spawn_episodes < 1 || (d->n_preys > 0 && !io->spawn_prey))) return CM_EINVAL;
    if (io->chan_u && io->chan_planes < need) return CM_EINVAL;
    return CM_OK;
}

static int launch(const cm_env_desc *d, const cm_env_state *s, const cm_step_io *io, const uint8_t *mask, int mode,
                  int at_reset, cudaStream_t stream)
{
    int rc = validate(d, s, io, mode);
    if (rc) return rc;
    if (s->n_envs == 0) return CM_OK;
    EnvArgs A;
    A.d = *d; A.s = *s; A.io = *io; A.mask = mask; A.mode = mode; A.at_reset = at_reset;
    A.n_pad = (d->n_agents + 7) & ~7;
    A.p_pad = (d->n_preys + 7) & ~7;
    A.warp_bytes = (env_warp_bytes(A.n_pad, A.p_pad, d->grid) + 15) & ~15;
    const int team = d->n_agents > d->n_preys ? d->n_agents : d->n_preys;
    // Lanes per env.  Small teams: the smallest power of two >= the team.  Larger teams: every loop strides by the group size, so
    // a group may be SMALLER than the team — the lane-parallel loops then cost the same warp instructions per env, while the
    // order-dependent loops of the group's lane 0 (45 % of the warp instructions at n = 32 with one env per warp) are shared
    // by the 2 or 4 envs of a warp.  Measured at C3 (n = 32): 0.085 / 0.067 / 0.056 ms per 8192 envs with 32 / 16 / 8 lanes.
    // The smallest group whose shared memory still lets three CTAs share an SM wins (C5, n = 200: 32 lanes).
    A.group = team <= 4 ? 4 : 8;
    while (A.group < 32 && kConstBytes + (size_t)kWarpsPerCta * (32 / A.group) * A.warp_bytes > (size_t)225 * 1024 * kWarpsPerCta / 24) A.group *= 2;
    {   // experiments only: CM_ENV_GROUP=4|8|16|32 overrides the lanes per env
        static const int forced = [] { const char *e = getenv("CM_ENV_GROUP"); return e ? atoi(e) : 0; }();
        if (forced == 4 || forced == 8 || forced == 16 || forced == 32) A.group = forced;
    }
    const int envs_per_cta = kWarpsPerCta * (32 / A.group);
    const size_t smem = kConstBytes + (size_t)envs_per_cta * A.warp_bytes;
    // launch geometry is cached per (device, smem) so that steady-state calls issue nothing but the launch
    // (keeps the call CUDA-graph capturable)
    static thread_local struct { int dev; size_t smem; const void *kernel; int ctas_per_sm; int sms; } cache = {-1, 0, nullptr, 0, 0};
    const bool inj = io->prey_cand || io->chan_u || io->spawn_agent || io->spawn_prey;
    void (*kernel)(const EnvArgs) = pick_env_kernel(d->scenario, d->conds ? kChanTable : d->channel, inj);
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return set_cuda_error(cudaGetLastError(), CM_ENODEVICE);
    if (cache.dev != dev || cache.smem != smem || cache.kernel != (const void *)kernel) {
        int sms = 0, ctas = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return set_cuda_error(cudaGetLastError(), CM_ECUDA);
        if (smem > 48 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return set_cuda_error(e, CM_ECUDA);
        }
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas, kernel, kWarpsPerCta * 32, smem) != cudaSuccess)
            return set_cuda_error(cudaGetLastError(), CM_ECUDA);
        cache.dev = dev; cache.smem = smem; cache.kernel = (const void *)kernel; cache.ctas_per_sm = ctas < 1 ? 1 : ctas; cache.sms = sms;
    }
    // persistent grid: a whole number of CTAs per SM, warps stride over the envs
    int64_t want = (s->n_envs + envs_per_cta - 1) / envs_per_cta;
    int64_t cap = (int64_t)cache.sms * cache.ctas_per_sm;
    int grid = (int)(want < cap ? want : cap);
    kernel<<<grid, kWarpsPerCta * 32, smem, stream>>>(A);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_cuda_error(e, CM_ECUDA);
    return CM_OK;
}

}  // namespace cm

extern "C" int cm_env_reset(const cm_env_desc *desc, const cm_env_state *state, const cm_step_io *io,
                            const uint8_t *mask, cm_stream_t stream)
{
    return cm::launch(desc, state, io, mask, 1, 1, (cudaStream_t)stream);
}

extern "C" int cm_env_step(const cm_env_desc *desc, const cm_env_state *state, const cm_step_io *io, cm_stream_t stream)
{
    return cm::launch(desc, state, io, nullptr, 0, 0, (cudaStream_t)stream);
}

extern "C" int cm_comm_update(const cm_env_desc *desc, const cm_env_state *state, const cm_step_io *io, int at_reset,
                              cm_stream_t stream)
{
    return cm::launch(desc, state, io, nullptr, 2, at_reset, (cudaStream_t)stream);
}
