"""Helpers of tests/test_gpu_ppo_paths.py: every launch path of the PPO update kernels (cm_ppo_net, csrc/ppo_net_kernels.cu)
against float64, at small batches.

tests/test_gpu_ppo_scale.py holds six production shapes; this file walks the shapes at which the launch code branches: every
team size 1 .. 256 (the n x n kernels' KT = ceil(n / 32) template, their 256- or 512-thread variant, group sizes that do not
divide 64, 128 or 256), every observation width 1 .. 128 (the synchronous and the bulk-copy first layer, KMAX 64 / 128),
1 to 4 layers, residual on / off, 'general' / 'dot' attention, narrow layers, chunked walks, and the CENT wide kernels at
every K = n·D residue of their chunk and panel widths.

What is here:
- the case tables of parts A-F (``cases_*``) and the batch sizing that gives every n x n and head kernel at least two env
  blocks, the last one partial;
- the case builder (a generalisation of ppo_scale_util.make_case) and the comparison of one case against float64
  (``check_case``), with ppo_scale_util's tolerances;
- the launch code's template selection, restated (``predicted_kernels``), the list of instantiations it can reach
  (``EXPECTED``, with the source line that selects each) and of those it cannot (``UNREACHABLE``, with the reason).

Nothing here touches CUDA at import time.
"""
import copy
import math
import re

import numpy as np

import ppo_scale_util as SU

TOL = SU.TOL
MIN_PROB = SU.MIN_PROB
team = SU.team
rel = SU.rel
CHUNK_AGREE = 1e-5          # chunked against single-chunk gradient, per tensor, normalised by the float64 tensor's max

# ---- batch sizing ---------------------------------------------------------------------------------------------------------
# Env-block sizes the kernels use (ppo_scale_util restates the launch code): the heads G = env_group(n) (the CENT baseline's
# head runs with n = 1), the small n x n kernels (n <= 8) G = 128 / n, the others G = env_geom_G(n).  A call over S steps
# gives each kernel ceil(S / G) >= 2 blocks, the last one partial, when S > G and S % G != 0 for every G > 1.
MIN_STEPS = 256             # valid steps of every policy minibatch at least: ratios on both sides of the clip range


def block_sizes(kind, n):
    """env-block sizes of the kernels a policy call of this kind runs (the critic's n x n kernels are the policy's)"""
    gs = [SU.env_group(n)]
    if kind in ("comm", "dec"):                    # (Obs-DP: the n x n kernels run in its CommBaseCritic)
        gs.append(SU.small_G(n) if n <= 8 else SU.env_geom_G(n))
    return gs


def steps_for(kind, n):
    """valid steps of the policy minibatch: > every block size, a multiple of none; CENT: > 256 for the baseline head too"""
    gs = block_sizes(kind, n) + ([256] if kind == "cent" else [])
    S = max(MIN_STEPS, max(gs) + 1)
    while any(g > 1 and S % g == 0 for g in gs):
        S += 1
    return S


def path_len_for(S):
    """an odd path length, about S / 2 capped at 41: several paths, each a few chunks long in part D"""
    return 2 * (min(S, 80) // 4) + 1


def valid_lengths(S, T, rng):
    """lengths of the minibatch's paths: 1 and T among them, summing to exactly S, in a random order"""
    assert S >= T + 1
    out, rem = [1, T], S - 1 - T
    while rem > 0:
        k = min(int(rng.randint(1, T + 1)), rem)
        out.append(k)
        rem -= k
    rng.shuffle(out)
    return out


# ---- the case tables --------------------------------------------------------------------------------------------------------
def case(part, kind, n, D, L=2, residual=True, att="general", sizes=None, relu=False, chunk=None, S=None):
    S = steps_for(kind, n) if S is None else S
    c = dict(part=part, kind=kind, n=n, D=D, L=L if kind != "cent" else 0, residual=residual, att=att, sizes=sizes, relu=relu,
             chunk=chunk, S=S, T=path_len_for(S))
    c["id"] = f"{part}-{kind}-n{n}-D{D}-L{c['L']}" + ("" if residual else "-nores") + ("-dot" if att == "dot" else "") + \
              ("-narrow" if sizes else "") + ("-relu" if relu else "") + (f"-chunk{chunk}" if chunk else "")
    return c


# launch bands of the n x n kernels: small kernels (n <= 8), KT = 1, 2, 4, 7 (512 threads in the backward), 7 (256), 8
BANDS = [(1, 8), (9, 32), (33, 64), (65, 128), (129, 170), (171, 212), (213, 224), (225, 256)]
BAND_IDS = [f"n{a}-{b}" for a, b in BANDS]
ODD_DS = (13, 21, 29, 53, 77, 1, 127)


def cases_a(band):
    """A: Comm-DP, every n of the band, L = 2, residual, 'general'; D alternates among odd widths"""
    a, b = BANDS[band]
    return [case("A", "comm", n, ODD_DS[n % len(ODD_DS)]) for n in range(a, b + 1)]


B_TEAMS = (4, 40)           # the small n x n kernels; KT = 2 (G = 3, cap 120)
B_KINDS = ("comm", "dec")


def cases_b(kind, n, half):
    """B: every observation width 1 .. 128 (half 0: 1 .. 64, half 1: 65 .. 128): the synchronous first layer at D % 4 != 0,
    the bulk-copy one at D % 4 == 0 with KMAX 64 up to D = 64 and 128 from D = 65"""
    return [case("B", kind, n, D) for D in range(1 + 64 * half, 65 + 64 * half)]


C_TEAMS = (1, 3, 8, 9, 32, 33, 64, 65, 128, 129, 212, 213, 224, 225, 256)     # both sides of every band edge
C_NARROW = (3, 65, 213)
NARROW = ((96,), 48, (100, 40, 24), (56,))      # encoder, embedding, head, critic decoder: zero-padded into (128, 64, .., 64)


def cases_c(n):
    """C: L = 1 .. 4 x residual on / off x 'general' / 'dot' at one team size; narrow layers at three of them"""
    D = ODD_DS[n % len(ODD_DS)]
    out = [case("C", "comm", n, D, L=L, residual=r, att=a) for L in (1, 2, 3, 4) for r in (True, False) for a in ("general", "dot")]
    if n in C_NARROW:
        out += [case("C", "comm", n, D, L=L, sizes=NARROW) for L in (1, 3)]
    return out


# D: chunked walks at W = 1, 2, 7 words per mask row; chunk_steps below the path length, so boundaries fall inside paths
D_CASES = [dict(n=7, D=21, chunk=5), dict(n=40, D=44, chunk=4), dict(n=213, D=29, chunk=2)]


D_STEPS = 67                # > every block size of n = 7, 40, 213 (36, 18, 6, 3, 1) and a multiple of none: the chunked and
                            # single-chunk sums differ by summation order, which grows with the steps summed (8.7e-6 of
                            # CHUNK_AGREE's 1e-5 at 256 steps)


def cases_d(i, L):
    d = D_CASES[i]
    return [case("D", "comm", d["n"], d["D"], L=L, chunk=d["chunk"], S=D_STEPS)]


E_DS = (29, 68)             # one odd width (synchronous first layer) and one D % 4 == 0 past 64 (bulk copy, KMAX 128)


def cases_e(band):
    """E: Obs-DP (CM_NET_POLICY_DEC) with CommBaseCritic, every n of the band at both widths"""
    a, b = BANDS[band]
    return [case("E", "dec", n, D) for n in range(a, b + 1) for D in E_DS]


CENT_K_MAX = 32768
CENT_FILL = (21, 53, 8, 128, 77, 3, 64, 100)


def cent_widths():
    """D per n = 1 .. 256 such that K = n·D takes every residue mod 64 (so mod 32 too) and K <= 32 768.  Odd n reach every
    residue: D = r n^-1 mod 64; the rest cycle through CENT_FILL.  5n mod 64 takes every residue over n = 1 .. 64 (5 is odd)."""
    out, todo = {}, list(range(64))
    for n in range(1, 257):
        if n % 2 and todo:
            r = todo.pop(0)
            D = (r * pow(n, -1, 64)) % 64 or 64
            if D + 64 <= 128 and n * (D + 64) <= CENT_K_MAX and n % 4 == 1:
                D += 64
        else:
            D = CENT_FILL[n % len(CENT_FILL)]
        while n * D > CENT_K_MAX:
            D //= 2
        out[n] = D
    return out


def cases_f(band):
    """F: CENT policy (tanh and relu alternating) with the GaussianMLPBaseline, every n of the band"""
    a, b = BANDS[band]
    w = cent_widths()
    return [case("F", "cent", n, w[n], relu=bool(n % 2 == 0)) for n in range(a, b + 1)]


# ---- the launch code's template selection, restated (csrc/ppo_net_kernels.cu) ------------------------------------------------
SMEM_MAX = 227 * 1024       # kSmemMax (:1602)
KNP = 68                    # kNP (:34)


def kt_of(n):
    """KT_DISPATCH (:1813-1821)"""
    kt = (n + 31) // 32
    return next(k for k in (1, 2, 4, 7, 8) if kt <= k)


def env_cap(n):
    """env_geom's cap (:1716-1723)"""
    return (SU.env_geom_G(n) * n + 3) & ~3


def cs_floats(KT, threads):
    """:1744"""
    return threads // 32 * 8 * (KT * 32 + 4)


def nxn_threads(n, blocks):
    """agg_fwd_t (:1762, one row block) and agg_bwd_t / softmax_bwd_t (:1782, :1800, two): 512 threads when n > 64 and the
    coefficient strips of 16 warps fit beside the row blocks"""
    KT = kt_of(n)
    return 512 if n > 64 and (blocks * env_cap(n) * KNP + cs_floats(KT, 512)) * 4 <= SMEM_MAX else 256


def dense_fwd_name(N, act, aligned):
    """dense_fwd / dense_fwd_t (:1620-1634): ASYNC iff the rows are 16-byte aligned (ldx % 4 == 0 and K % 4 == 0)"""
    return f"net_dense_fwd_kernel<{N},{act},{int(aligned)}>"


def dense_bwd_name(N, K, aligned, xrelu=False):
    """dense_bwd / dense_bwd_t (:1651-1674): KMAX = 64 for K <= 64 else 128 (the relu layers: KMAX 64 at N = 32, 128 at N = 64);
    synchronous rows: ROWS 128; bulk copy: ROWS 128 when two stages fit (:1656), else 64"""
    KMAX = (64 if N == 32 else 128) if xrelu else (64 if K <= 64 else 128)
    if not aligned:
        return f"net_dense_bwd_kernel<{N},{KMAX},128,0,{int(xrelu)}>"
    fits = (KMAX * (N + 4) + 2 * 128 * (N + 4 + KMAX + 4)) * 4 + 16 <= SMEM_MAX
    return f"net_dense_bwd_kernel<{N},{KMAX},{128 if fits else 64},1,{int(xrelu)}>"


def nxn_names(n, backward):
    if n <= 8:                                     # kSmallN (:1832, :1841, :1851, :1862)
        s = {"net_small_scores_kernel", "net_small_agg_fwd_kernel"}
        return s | ({"net_small_agg_bwd_kernel", "net_small_softmax_bwd_kernel"} if backward else set())
    KT = kt_of(n)
    s = {f"net_scores_kernel<{KT},256>", f"net_agg_fwd_kernel<{KT},{nxn_threads(n, 1)}>"}
    if backward:
        t = nxn_threads(n, 2)
        s |= {f"net_agg_bwd_kernel<{KT},{t}>", f"net_softmax_bwd_kernel<{KT},{t}>"}
    return s


def predicted_kernels(kind, n, D, call, backward=True, relu=False):
    """cm_ppo_net kernels one call launches (names as ``kernel_name`` normalises them).  kind comm / dec / cent; call
    policy / critic; the observation rows are aligned iff D % 4 == 0 (torch allocations, chunk offsets r0·D)."""
    al = D % 4 == 0
    s = {"net_loss_store_kernel"}                  # (:2158; the calls traced here all pass a loss)
    if kind == "cent":
        act = 2 if relu else 1
        if call == "policy":                       # run_chunk_cent (:1999-2031)
            s |= {f"net_wide_fwd_kernel<2,{act}>", dense_fwd_name(64, act, True), dense_fwd_name(32, act, True), "net_cent_head_kernel"}
            if backward:
                s |= {"net_wide_dw_kernel<32,1>", dense_bwd_name(32, 64, True, relu), dense_bwd_name(64, 128, True, relu),
                      "net_wide_dw_kernel<128,0>"}
        else:                                      # the baseline (:1973-1997)
            s |= {"net_wide_fwd_kernel<1,1>", dense_fwd_name(64, 1, True), "net_critic_head_kernel"}
            if backward:
                s |= {dense_bwd_name(64, 64, True), "net_wide_dw_kernel<64,0>"}
        return s
    trunk_f = {dense_fwd_name(128, 1, al), dense_fwd_name(64, 1, True), dense_fwd_name(64, 0, True)} | nxn_names(n, False)
    trunk_b = {dense_bwd_name(64, 64, True), dense_bwd_name(64, 128, True), dense_bwd_name(128, D, al)} | nxn_names(n, True)
    if call == "critic":                           # (:2092-2109)
        s |= trunk_f | {dense_fwd_name(64, 1, True), "net_critic_head_kernel"}
        return s | (trunk_b | {dense_bwd_name(64, 64, True)} if backward else set())
    s.add("net_policy_head_kernel")
    if kind == "dec":                              # (:2052-2055, :2081-2085)
        s |= {dense_fwd_name(128, 1, al), dense_fwd_name(64, 1, True), dense_fwd_name(32, 1, True)}
        return s | ({dense_bwd_name(32, 64, True), dense_bwd_name(64, 128, True), dense_bwd_name(128, D, al)} if backward else set())
    s |= trunk_f | {dense_fwd_name(128, 1, True), dense_fwd_name(64, 1, True), dense_fwd_name(32, 1, True)}      # (:2057-2061)
    if backward:                                   # (:2087-2090)
        s |= trunk_b | {dense_bwd_name(32, 64, True), dense_bwd_name(64, 128, True), dense_bwd_name(128, 64, True)}
    return s


def all_predicted():
    """every name predicted_kernels gives over every supported (kind, n, D, nonlinearity)"""
    out = set()
    for n in range(1, 257):
        for D in range(1, 129):
            for call in ("policy", "critic"):
                out |= predicted_kernels("comm", n, D, call) | predicted_kernels("dec", n, D, "policy")
        out |= predicted_kernels("cent", n, 21, "policy", relu=False) | predicted_kernels("cent", n, 21, "policy", relu=True)
        out |= predicted_kernels("cent", n, 21, "critic")
    return out


# Every instantiation the launch code can select, with the source line (csrc/ppo_net_kernels.cu) that selects it.
EXPECTED = {
    "net_dense_fwd_kernel<128,1,0>": ":1623 dense_fwd_t, !rows_aligned: the observation layer at D % 4 != 0 (:1906, :2053)",
    "net_dense_fwd_kernel<128,1,1>": ":1623 rows_aligned: the observation layer at D % 4 == 0; the policy head's 64 -> 128 (:2059)",
    "net_dense_fwd_kernel<64,1,1>": ":1632 N == 64, tanh: 128 -> 64 embedding (:1907), head (:2060), critic decoder (:2096), "
                                    "baseline (:1977)",
    "net_dense_fwd_kernel<64,0,1>": ":1632 N == 64, linear: Q = E W_a (:1908) and V = H W_l (:1912)",
    "net_dense_fwd_kernel<32,1,1>": ":1633 N == 32, tanh: the policy head's 64 -> 32 (:2055, :2061); CENT tanh (:2004)",
    "net_dense_fwd_kernel<64,2,1>": ":1630 act == 2, N == 64: CENT relu 128 -> 64 (:2003)",
    "net_dense_fwd_kernel<32,2,1>": ":1630 act == 2, N == 32: CENT relu 64 -> 32 (:2004)",
    "net_dense_bwd_kernel<64,64,128,1,0>": ":1670 N == 64, K <= 64; two 128-row stages fit (:1656): GCN / attention / critic "
                                           "decoder / baseline layers",
    "net_dense_bwd_kernel<64,128,64,1,0>": ":1671 N == 64, K = 128; 64-row stages (:1656): 128 -> 64 layers",
    "net_dense_bwd_kernel<128,64,64,1,0>": ":1668 N == 128, K <= 64, aligned: the head's 64 -> 128 (:2089) and the observation "
                                           "layer at D % 4 == 0, D <= 64 (:1950, :2084)",
    "net_dense_bwd_kernel<128,128,64,1,0>": ":1669 N == 128, K > 64, aligned: the observation layer at D % 4 == 0, D >= 68",
    "net_dense_bwd_kernel<128,64,128,0,0>": ":1657 !rows_aligned, K <= 64: the observation layer at odd D <= 63",
    "net_dense_bwd_kernel<128,128,128,0,0>": ":1657 !rows_aligned, K > 64: the observation layer at D % 4 != 0, D >= 65",
    "net_dense_bwd_kernel<32,64,128,1,0>": ":1672 N == 32: the policy head's 64 -> 32 (:2082, :2087); CENT tanh (:2029)",
    "net_dense_bwd_kernel<32,64,128,1,1>": ":1666 xact == 2, N == 32: CENT relu 64 -> 32 (:2029)",
    "net_dense_bwd_kernel<64,128,64,1,1>": ":1667 xact == 2, N == 64: CENT relu 128 -> 64 (:2030)",
    "net_small_scores_kernel": ":1832 n <= kSmallN",
    "net_small_agg_fwd_kernel": ":1841 n <= kSmallN",
    "net_small_agg_bwd_kernel": ":1851 n <= kSmallN",
    "net_small_softmax_bwd_kernel": ":1862 n <= kSmallN",
    **{f"net_scores_kernel<{k},256>": f":1836 KT_DISPATCH -> {k}" for k in (1, 2, 4, 7, 8)},
    "net_agg_fwd_kernel<1,256>": ":1762 n <= 64: 256 threads (n 9 .. 32)",
    "net_agg_fwd_kernel<2,256>": ":1762 n <= 64: 256 threads (n 33 .. 64)",
    "net_agg_fwd_kernel<4,512>": ":1762 wide (n 65 .. 128)",
    "net_agg_fwd_kernel<7,512>": ":1762 wide (n 129 .. 224)",
    "net_agg_fwd_kernel<8,512>": ":1762 wide (n 225 .. 256: 256·68 + 33 280 floats fit)",
    **{f"net_{k}_kernel<1,256>": f":{ln} n <= 64: 256 threads (n 9 .. 32)" for k, ln in (("agg_bwd", 1782), ("softmax_bwd", 1800))},
    **{f"net_{k}_kernel<2,256>": f":{ln} n <= 64: 256 threads (n 33 .. 64)" for k, ln in (("agg_bwd", 1782), ("softmax_bwd", 1800))},
    **{f"net_{k}_kernel<4,512>": f":{ln} wide (n 65 .. 128)" for k, ln in (("agg_bwd", 1782), ("softmax_bwd", 1800))},
    **{f"net_{k}_kernel<7,512>": f":{ln} wide: 2·cap·68 + 29 184 floats fit up to cap = 212 (n 129 .. 212)"
       for k, ln in (("agg_bwd", 1782), ("softmax_bwd", 1800))},
    **{f"net_{k}_kernel<7,256>": f":{ln} not wide: cap 216 .. 224 (n 213 .. 224)" for k, ln in (("agg_bwd", 1782), ("softmax_bwd", 1800))},
    **{f"net_{k}_kernel<8,256>": f":{ln} not wide: cap >= 228 (n 225 .. 256)" for k, ln in (("agg_bwd", 1782), ("softmax_bwd", 1800))},
    "net_wide_fwd_kernel<1,1>": ":1687 N == 64: the baseline's first layer (:1976)",
    "net_wide_fwd_kernel<2,1>": ":1686 N == 128, tanh: the CENT first layer (:2002)",
    "net_wide_fwd_kernel<2,2>": ":1686 N == 128, relu: the CENT first layer (:2002)",
    "net_wide_dw_kernel<64,0>": ":1997 the baseline's dW1",
    "net_wide_dw_kernel<128,0>": ":2031 the CENT policy's dW1",
    "net_wide_dw_kernel<32,1>": ":2028 the CENT policy's transposed dW4 [32][5n]",
    "net_policy_head_kernel": ":2077 Comm-DP and Obs-DP policy",
    "net_critic_head_kernel": ":2105 CommBaseCritic; :1992 the baseline (n = 1 per step)",
    "net_cent_head_kernel": ":2025 CENT policy",
    "net_loss_store_kernel": ":2158 a call with a loss",
}

# Instantiations that are compiled (every template the dispatchers name) but that no input can select.
UNREACHABLE = {
    **{f"net_agg_fwd_kernel<{k},512>": "wide needs n > 64 (:1762); KT <= 2 means n <= 64" for k in (1, 2)},
    **{f"net_agg_fwd_kernel<{k},256>": "the row block and 16 warps' strips always fit (largest: KT 8, cap 256: 198 KB)" for k in (4, 7, 8)},
    **{f"net_{f}_kernel<{k},512>": "wide needs n > 64 (:1782, :1800)" for f in ("agg_bwd", "softmax_bwd") for k in (1, 2)},
    **{f"net_{f}_kernel<4,256>": "two row blocks of cap <= 128 and 16 warps' strips fit (134 KB)" for f in ("agg_bwd", "softmax_bwd")},
    **{f"net_{f}_kernel<8,512>": "2·cap·68 + 33 280 floats > 227 KB for every cap >= 228" for f in ("agg_bwd", "softmax_bwd")},
    **{dense_fwd_name(128, 0, a): "no layer is linear with 128 outputs" for a in (0, 1)},
    **{dense_fwd_name(32, 0, a): "no layer is linear with 32 outputs" for a in (0, 1)},
    **{dense_fwd_name(N, act, False): "the input is a workspace array: 16-byte aligned, ldx = K in {64, 128}"
       for N, act in ((64, 1), (64, 0), (32, 1), (64, 2), (32, 2))},
    **{f"net_dense_bwd_kernel<{N},{KM},128,0,{x}>": "the input is a workspace array: 16-byte aligned, ldx = K in {64, 128}"
       for N, KM, x in ((64, 64, 0), (64, 128, 0), (32, 64, 0), (32, 64, 1), (64, 128, 1))},
    "net_dense_bwd_kernel<32,128,128,0,0>": "no layer has 32 outputs and more than 64 inputs",
    "net_dense_bwd_kernel<32,128,128,1,0>": "no layer has 32 outputs and more than 64 inputs",
}


def kernel_name(raw):
    """'void cm::net_dense_fwd_kernel<128, 1, 0>(float const*, ...)' -> 'net_dense_fwd_kernel<128,1,0>'; None for a kernel that
    is not cm_ppo_net's"""
    m = re.search(r"cm::(net_\w+)(<[^>]*>)?\(", raw)
    return None if m is None else m.group(1) + (m.group(2) or "").replace(" ", "")


# Cases of the sweep whose launches the coverage test traces: between them every EXPECTED entry, n = 1, the 256-thread
# backward at KT = 7 and the bulk-copy observation layer at K = 40 (KMAX 64) and K = 68 (KMAX 128) in Obs-DP calls, where the
# policy has no other N = 128 layer (so the trace attributes those instantiations to the observation layer alone).
def coverage_cases():
    f = cent_widths()
    return ([case("A", "comm", n, ODD_DS[n % len(ODD_DS)]) for n in (1, 3, 9, 33, 65, 129, 213, 225)] +
            [case("B", "dec", 40, D) for D in (21, 40, 68, 77)] + [case("B", "comm", 4, 64), case("B", "comm", 4, 68)] +
            [case("F", "cent", n, f[n], relu=r) for n, r in ((5, False), (32, True))])


# ---- the case builder (GPU) -----------------------------------------------------------------------------------------------
def make_case(c, seed=0):
    """-> (fused DevicePPO, float64 DevicePPO, padded batch b0, minibatch path ids).  The construction of
    ppo_scale_util.make_case with the case's T, L, residual, attention, layer sizes and kind: ragged valid lengths that include
    1 and T and sum to c['S'] over the minibatch, random adjacency and channel rows with one row without a neighbour, random
    availability with action 4 always available, biases and log-stds moved off their initial values."""
    import torch
    from com_marl_b200.policy import CentralizedCategoricalMLPPolicy, CommCategoricalMLPPolicy, DecCategoricalMLPPolicy
    from com_marl_b200.ppo import CommBaseCritic, DevicePPO, GaussianMLPBaseline
    from com_marl_b200.spaces import Box, Discrete, EnvSpec
    n, D, L, T, kind, sizes = c["n"], c["D"], c["L"], c["T"], c["kind"], c["sizes"]
    rng = np.random.RandomState(seed)
    lengths = valid_lengths(c["S"], T, rng)
    P = len(lengths) + 1
    torch.manual_seed(seed)
    spec = EnvSpec(Box(np.zeros(n * D), np.ones(n * D)), Discrete(5))
    if kind == "cent":
        pol = CentralizedCategoricalMLPPolicy(spec, n, hidden_nonlinearity="relu" if c["relu"] else "tanh",
                                              **({} if sizes is None else dict(hidden_sizes=sizes[2])))
        cri = GaussianMLPBaseline(spec, hidden_sizes=(64, 64, 64) if sizes is None else (sizes[1],) * 3)
    else:
        ckw = {} if sizes is None else dict(encoder_hidden_sizes=sizes[0], embedding_dim=sizes[1], decoder_hidden_sizes=sizes[3])
        cri = CommBaseCritic(spec, n, n_gcn_layers=L, residual=c["residual"], attention_type=c["att"], **ckw)
        if kind == "dec":
            pol = DecCategoricalMLPPolicy(spec, n, **({} if sizes is None else dict(hidden_sizes=(sizes[0][0], sizes[1], sizes[2][2]))))
        else:
            kw = {} if sizes is None else dict(encoder_hidden_sizes=sizes[0], embedding_dim=sizes[1], categorical_mlp_hidden_sizes=sizes[2])
            pol = CommCategoricalMLPPolicy(spec, n, n_gcn_layers=L, residual=c["residual"], attention_type=c["att"], **kw)
    with torch.no_grad():
        for m in (pol, cri):
            for k, p in m.named_parameters():
                if k.endswith("bias") or k.endswith("_init_std"):
                    p.add_(0.1 * torch.randn_like(p))
    pol64, cri64 = copy.deepcopy(pol).double(), copy.deepcopy(cri).double()
    fused = DevicePPO(pol, cri, fused=True)
    assert fused._fused is not None
    ref = copy.copy(fused)                         # the same loss code (compute_loss / _dist read self.policy only)
    ref._fused, ref.policy, ref.baseline = None, pol64, cri64
    g = torch.Generator(device="cuda").manual_seed(seed)
    rnd = lambda *s: torch.rand(*s, device="cuda", generator=g)  # noqa: E731
    valids = torch.tensor(lengths + [int(rng.randint(1, T + 1))], dtype=torch.int32, device="cuda")
    avail = (rnd(P, T, n, 5) < 0.8).float()
    avail[..., 4] = 1.0
    actions = torch.multinomial(avail.reshape(-1, 5), 1).reshape(P, T, n)
    b = dict(obs=rnd(P, T, n * D), avail=avail.reshape(P, T, n * 5), actions=actions, rewards=rnd(P, T).double(), valids=valids)
    if kind != "cent":
        adj = (rnd(P, T, n, n) < 0.6).float()
        adj = torch.maximum(adj, torch.eye(n, device="cuda"))
        adj[0, 0, 0, :] = 0.0                      # a row with no neighbour at all (the + 1e-12 of the renormalisation)
        chan = (rnd(P, T, L, n, n) < 0.7).float()
        chan[:, :, :, torch.arange(n), torch.arange(n)] = 1.0
        b["dist_adjs"], b["channels"] = adj.reshape(P, T, n * n), chan.reshape(P, T, L * n, n)
    t = torch.arange(T, device="cuda")[None, :] < valids[:, None]
    b["obs"] = b["obs"] * t.reshape(P, T, 1).float()
    b["rewards"] = b["rewards"] * t.double()
    ids = rng.permutation(P - 1)                   # the minibatch: every path but the last, shuffled
    return fused, ref, b, ids


def old_ll_offsets(P, T, ids, seed):
    """ppo_scale_util.old_ll_offsets (ratios on both sides of the clip range, none within CLIP_GAP of its edges), with the first
    step of the minibatch's first two paths set to +-0.25 so that a small minibatch has ratios on both sides for certain"""
    d = SU.old_ll_offsets(P, T, seed)
    d[int(ids[0]), 0], d[int(ids[1]), 0] = 0.25, -0.25
    return d


def _maxabs(x):
    return float(x.abs().max()) if x.numel() else 0.0


def _zero_ok(c, k):
    """a float64 gradient that is exactly zero by construction: at n = 1 every softmax has one key, so nothing reaches W_a"""
    return c["n"] == 1 and k.startswith("attention_layer.")


def grad_errors(c, g, ref_grads):
    """per parameter tensor: normalised error of the flat kernel gradient `g` against float64; a tensor whose float64
    gradient is exactly zero must be exactly zero (and may be so only where _zero_ok says why)"""
    out, o = {}, 0
    for k, r in ref_grads:
        seg = g[o:o + r.numel()].double()
        scale = _maxabs(r)
        if scale == 0:
            out[k] = 0.0 if (_zero_ok(c, k) and _maxabs(seg) == 0) else float("nan")
        else:
            out[k] = rel(_maxabs(seg - r), scale)
        o += r.numel()
    assert o == g.numel()
    return out


def grads_at_kernel_forward(ppo, c, b, ids, old, ll, values):
    """float64 gradients of the policy and critic losses of ppo_scale_util.evaluate, with each step's ratio exp(ll - old)
    formed from the kernel's fp32 log-likelihood `ll` [P, T] and each step's value from the kernel's fp32 `values` [P, T]
    (as constants: the derivatives are the float64 ones at that point).

    Why the gradients are held against this and not against the float64 forward: the kernels' ll and values are fp32 sums
    over n agents, within TOL["out"] of float64 (up to |dll| ~ 3e-4 at |ll| ~ 300, n = 250), and that error moves each
    step's ratio by as much, relative, and each critic residual R - V by |dV|.  The minibatch gradient is a sum of such
    terms whose centred advantages (residuals) cancel, so the relative error of a bias gradient is that per-step error times
    sum|terms| / |sum terms| — past TOL["grad"]·team(n) at some cases (n = 72, 216, 249, 250; a larger minibatch does not
    remove it, the errors are per step).  With the kernel's own forward fed in, the same cases agree to 2e-6 .. 2e-5: the
    backward pass is held exactly, and the forward is held by the per-step comparison under TOL["out"]."""
    import torch
    pol, cri = ppo.policy, ppo.baseline
    for m in (pol, cri):
        for p in m.parameters():
            p.grad = None
    nvalid = float(b["mask"][ids].sum())
    for sl in SU.path_slices(c, ids):
        s = SU._sub(b, sl, torch.float64)
        d = ppo._dist(s, None)
        new = d.log_prob(s["actions"]).sum(-1)
        new = new + (ll[sl].double() - new).detach()
        ratio = (new - old[sl].double()).exp()
        obj = torch.min(ratio * s["adv"], torch.clamp(ratio, 1 - ppo.lr_clip_range, 1 + ppo.lr_clip_range) * s["adv"])
        if ppo.ent_coeff:
            obj = obj + ppo.ent_coeff * d.entropy().mean(-1)
        (-obj[s["mask"]].sum() / nvalid).backward()
        v = values[sl].double()
        if c["kind"] == "cent":                    # GaussianMLPBaseline.compute_loss
            mean = cri.module._mean_module(s["obs"].reshape(-1, cri.input_dim))
            mean = mean + (v.reshape(-1, 1) - mean).detach()
            std = cri.module._init_std.exp().expand_as(mean)
            lc = -torch.distributions.Normal(mean, std).log_prob(s["returns"].reshape(-1, 1)).sum(-1).mean()
        else:                                      # CommBaseCritic.compute_loss
            mean, std = cri._values(s["obs"], s["dist_adjs"], s["channels"])
            mean = mean + (v - mean).detach()
            lc = (0.5 * ((s["returns"] - mean) / std) ** 2 + std.log() + 0.5 * float(np.log(2 * np.pi))).mean()
        (lc * (len(sl) / len(ids))).backward()
        del s, d
    grad = lambda m: [(k, p.grad.detach().reshape(-1) if p.grad is not None else torch.zeros(p.numel(), dtype=torch.float64, device=p.device))  # noqa: E731
                      for k, p in m.named_parameters() if p.requires_grad]
    return dict(grads=grad(pol), critic_grads=grad(cri))


def check_case(c, seed=None):
    """Run one case on the kernels and in float64; -> record of normalised errors (NaN where a value is NaN) and the list of
    failures (empty when every comparison holds).  Compared: per-step ll, entropy, probs and values over every padded step; the
    policy loss and every policy gradient on the minibatch's valid steps with old_ll perturbed across the clip range; the
    critic loss and every critic gradient on the minibatch's padded steps.  Part D cases also run the chunked walk."""
    import torch
    seed = (c["n"] * 1009 + c["D"] * 31 + c["L"] * 7 + len(c["id"])) if seed is None else seed
    fused, ref, b0, ids = make_case(c, seed)
    P, T, n = b0["valids"].shape[0], c["T"], c["n"]
    bf = fused.finish_batch(dict(b0))              # kernel baselines -> cm_ppo_advantages: the inputs both sides see
    F, f = fused._fused, bf["_flat"]
    F.chunk_steps = 1 << 30                        # one chunk (part D walks its own below)
    F._ws = None
    with torch.no_grad():
        F.pol_map.refresh()
        out = F.policy_call(f, None, want_probs=True)
    old = out["ll"].reshape(P, T) + old_ll_offsets(P, T, ids, seed)
    tid = torch.as_tensor(ids, device="cuda")
    idx = F.step_index(f, ids, valid_only=True)
    if c["relu"]:                                  # steps at a relu kink leave the minibatch on both sides
        kink = SU.relu_kink_steps(c, ref.policy, bf)
        bf["mask"] = bf["mask"] & ~kink
        idx = idx[~kink.reshape(-1).index_select(0, idx)]
    S = int(idx.numel())
    idx_all = F.step_index(f, ids, valid_only=False)
    adv_i, old_i = bf["adv"].reshape(-1).index_select(0, idx), old.reshape(-1).index_select(0, idx)
    ret_i = bf["returns"].reshape(-1).index_select(0, idx_all)

    def grads(chunk):
        F.chunk_steps, F._ws = chunk, None
        F.pol_map.refresh()
        res = F.policy_call(f, idx, adv=adv_i, old_ll=old_i, backward=True, inv_count=1.0 / S)
        g = torch.empty_like(fused.opt.grad)
        F.pol_map.scatter_grad(g)
        blob_g = F.pol_map.grad.clone()
        F.cri_map.refresh()
        resc = F.critic_call(f, idx_all, returns=ret_i, backward=True)
        gc = torch.empty_like(fused.baseline_opt.grad)
        F.cri_map.scatter_grad(gc)
        return float(res["loss"]), g, float(resc["loss"]), gc, blob_g

    loss, g, closs, gc, blob_g = grads(1 << 30)
    chunked = grads(c["chunk"]) if c["chunk"] else None
    F._ws = None

    r64 = SU.evaluate(ref, c, bf, tid, old, torch.float64, outputs=True)
    rk = grads_at_kernel_forward(ref, c, bf, tid, old, out["ll"].reshape(P, T), bf["baselines"])
    kern = dict(ll=out["ll"].reshape(P, T), entropy=out["entropy"].reshape(P, T), probs=out["probs"].reshape(P, T, n, 5),
                values=bf["baselines"])
    errs, scales = {k: 0.0 for k in kern}, {k: 0.0 for k in kern}
    min_prob, ratio_lo, ratio_hi = float("inf"), False, False
    mb = torch.zeros(P, dtype=torch.bool, device="cuda")
    mb[tid] = True
    nan = False
    for sl, o64 in r64["slices"]:
        for k in kern:
            d = kern[k][sl].double() - o64[k]
            nan |= bool(d.isnan().any())
            errs[k] = max(errs[k], _maxabs(d))
            scales[k] = max(scales[k], _maxabs(o64[k]))
        av = o64["avail"].reshape(o64["probs"].shape) > 0
        min_prob = min(min_prob, float(o64["probs"][av].min()))
        ratio = (o64["ll"] - old[sl].double()).exp()[bf["mask"][sl] & mb[sl][:, None]]
        ratio_lo |= bool((ratio < 1.0 - SU.CLIP).any())
        ratio_hi |= bool((ratio > 1.0 + SU.CLIP).any())
    out_err = {k: float("nan") if nan else rel(errs[k], scales[k]) for k in kern}
    tm = team(n)
    rec = dict(id=c["id"], part=c["part"], n=n, D=c["D"], L=c["L"], policy_steps=S, critic_steps=int(idx_all.numel()),
               out=max(out_err.values(), key=lambda e: (math.isnan(e), e)),
               loss=abs(loss - r64["loss"]) / (tm * max(1.0, abs(r64["loss"]))),
               critic_loss=abs(closs - r64["critic_loss"]) / max(1.0, abs(r64["critic_loss"])),
               min_prob64=min_prob)
    pg, cg = grad_errors(c, g, rk["grads"]), grad_errors(c, gc, rk["critic_grads"])
    worst = lambda d: max(d.values(), key=lambda e: (math.isnan(e), e))  # noqa: E731
    rec["grad"] = worst(pg) / tm                   # (in units of TOL["grad"]: divided by team(n))
    rec["critic_grad"] = worst(cg)
    # (reported: the same gradients against the float64 forward; the gap is the forward's rounding, grads_at_kernel_forward)
    rec["grad_plain"] = worst(grad_errors(c, g, r64["grads"])) / tm
    rec["critic_grad_plain"] = worst(grad_errors(c, gc, r64["critic_grads"]))
    fails = []
    ok = lambda e, tol: e <= tol  # noqa: E731   (False on NaN)
    for k, e in out_err.items():
        if not ok(e, TOL["out"]):
            fails.append((c["id"], k, e))
    if not ok(rec["loss"], TOL["loss"]):
        fails.append((c["id"], "loss", loss, r64["loss"]))
    if not ok(rec["critic_loss"], TOL["critic_loss"]):
        fails.append((c["id"], "critic_loss", closs, r64["critic_loss"]))
    fails += [(c["id"], "policy grad", k, e) for k, e in pg.items() if not ok(e, TOL["grad"] * tm)]
    fails += [(c["id"], "critic grad", k, e) for k, e in cg.items() if not ok(e, TOL["critic_grad"])]
    if not min_prob >= MIN_PROB:
        fails.append((c["id"], "an available action's float64 probability is inside Categorical's clamp", min_prob))
    if not (ratio_lo and ratio_hi):
        fails.append((c["id"], "ratios on one side of the clip range only"))
    if c["kind"] == "comm" and c["att"] == "dot":
        # no W_a parameter: the blob's W_a slice is the constant identity, and the kernel's gradient of that slice (E^T dQ,
        # :1948) is not a gradient of any parameter — no flat index may read it (blob layout: policy_layout.cuh)
        att0 = c["D"] * 128 + 128 + 128 * 64 + 64
        touched = ((F.pol_map.inverse >= att0) & (F.pol_map.inverse < att0 + 64 * 64)).any()
        if bool(touched) or any(k.startswith("attention_layer.") for k, _ in r64["grads"]):
            fails.append((c["id"], "dot attention: a parameter maps into the W_a slice of the blob"))
        rec["dot_att_blob_grad"] = _maxabs(blob_g[att0:att0 + 64 * 64])
    if chunked is not None:
        closs_c = chunked[2]
        pgc, cgc = grad_errors(c, chunked[1], rk["grads"]), grad_errors(c, chunked[3], rk["critic_grads"])
        rec["chunked_grad"] = worst(pgc) / tm
        rec["chunked_critic_grad"] = worst(cgc)
        agree = max(rel(_maxabs(chunked[1][o0:o0 + r.numel()].double() - g[o0:o0 + r.numel()].double()), _maxabs(r))
                    for o0, r in _offsets(rk["grads"]))
        agree_c = max(rel(_maxabs(chunked[3][o0:o0 + r.numel()].double() - gc[o0:o0 + r.numel()].double()), _maxabs(r))
                      for o0, r in _offsets(rk["critic_grads"]))
        rec["chunk_agree"] = max(agree, agree_c)
        fails += [(c["id"], "chunked policy grad", k, e) for k, e in pgc.items() if not ok(e, TOL["grad"] * tm)]
        fails += [(c["id"], "chunked critic grad", k, e) for k, e in cgc.items() if not ok(e, TOL["critic_grad"])]
        if not ok(abs(closs_c - r64["critic_loss"]) / max(1.0, abs(r64["critic_loss"])), TOL["critic_loss"]):
            fails.append((c["id"], "chunked critic loss", closs_c, r64["critic_loss"]))
        if not ok(abs(chunked[0] - r64["loss"]) / (tm * max(1.0, abs(r64["loss"]))), TOL["loss"]):
            fails.append((c["id"], "chunked loss", chunked[0], r64["loss"]))
        if not ok(rec["chunk_agree"], CHUNK_AGREE):
            fails.append((c["id"], "chunked against single-chunk gradient", rec["chunk_agree"]))
        # a chunk boundary inside a path, for both calls
        ends = set(np.cumsum([int(x) for x in b0["valids"][torch.as_tensor(ids)].cpu()]).tolist())
        inside = [k for k in range(c["chunk"], S, c["chunk"]) if k not in ends]
        if not inside or T % c["chunk"] == 0:
            fails.append((c["id"], "no chunk boundary falls inside a path"))
    del r64, rk, fused, ref, bf, F, f
    return rec, fails


def _offsets(ref_grads):
    o = 0
    for _, r in ref_grads:
        yield o, r
        o += r.numel()
