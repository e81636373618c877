#!/usr/bin/env python
"""bench.py — agent-steps/s of the batched rollout hot path (env step + comm + comm-GNN policy forward).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c3] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one rollout iteration over the whole batch: cm_policy_forward (forward + action sampling) followed by
cm_env_step (PredatorPrey/Coverage step, auto-reset, observation windows, adjacency + channel masks).  The default
workload is the configuration BASELINE.json's metric is quoted on, configs[2]: Predator-Prey --map 20 --sen 2 --den 0.08
--cap 4 --loss 0.2 (comm graph d^2 <= 162, IID packet drops, prey random walk), 65536 envs per B200 (weak scaling: every
GPU steps its own 65536 envs; the only collective of the rollout is the episode-statistics all-gather after the timed
region).  One JSON line is printed by rank 0:

  value      device-resident rollout: inputs live in HBM, steps replayed from one CUDA graph of `ring` iterations.  The
             timed region is exactly --steps steps: the graph holds the largest divisor of --steps that is not above --ring.
             The configs of the sweep have no step count of their own and are timed for at least --min-seconds.
  e2e        the same loop through the sampler-level host-buffer call (HostRollout = cm_rollout_step_host): one C call per
             env part and step runs policy -> env on device-resident state, copies the availability bytes host -> device
             and everything the sampler appends per step (next observation, masks, reward, done, counts, actions,
             probabilities ...) device -> pinned host memory.  `e2e.step_api` is the step-level pair of calls
             (policy.get_actions_host + BatchedEnv.step_host: observations travel both ways) kept as a secondary figure.
  roofline   the dominant kernel (policy forward) against the measured bf16 tensor peak, plus the env kernel against the
             measured HBM copy bandwidth (kernel durations from CUDA events around graphs of launches of ONE kernel).
  configs    a bounded sweep over the other BASELINE configs (c1..c5) with the same measurements, and `c5_ppo`: rollout +
             PPO update of config 5 (with N > 1: gradient all-reduces over NCCL inside the timed region).  With N > 1 the
             sweep is c4 + c5_ppo (the configs BASELINE shards over GPUs).
  cpu_baseline  the oracle port (C env oracle + numpy policy) on the box's host cores, bounded sample; next to it the
             survey-time figure of the real (pure Python) reference, labelled as measured elsewhere.

`--impl reference` times that CPU port on all host cores (the reference itself is pure Python and is not present
on the GPU box; oracle/ is its pinned restatement).

`--dump-outputs DIR` writes what the timed loop of `value` handed back for its last step to DIR/<name>.npy (see
dump_last_step), so that two builds run with the same arguments, hence the same inputs, can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: (scenario, map, sen, den, cap, loss, envs per GPU)  — BASELINE.json configs[0..4]
    "c1": ("pp", 10, 1, 0.04, 2, 0.0, 16384),
    "c2": ("co", 10, 1, 0.03, 2, 0.0, 16384),
    "c3": ("pp", 20, 2, 0.08, 4, 0.2, 65536),
    "c4": ("co", 30, 2, 0.06, 2, 0.1, 16384),
    "c5": ("pp", 50, 2, 0.08, 4, 0.0, 2048),
}
# sweep-only variants: BASELINE configs[2] names "Gilbert-Elliot drops" although `--loss 0.2` on the reference's command line
# reaches the IID channel only (init_communication forces FC / IID / FL, env_communication.py:35-43; the GE branch needs
# env.channelType set by hand): c3 is the CLI's IID reading, c3_ge the same workload on the Gilbert-Elliot Markov channel
# (Pgb = 0.0196, Pbg = 0.282: the reference's defaults, one transition per GCN layer)
VARIANTS = {"c3_ge": ("c3", dict(channel_type="GE"))}
WORKLOAD_TEXT = {
    "c1": "Predator-Prey --map 10 --sen 1 --den 0.04 --cap 2 --loss 0, 16384 envs per B200",
    "c2": "Coverage --map 10 --sen 1 --den 0.03 --loss 0, 16384 batched envs per B200",
    "c3": "Predator-Prey --map 20 --sen 2 --den 0.08 --cap 4 --loss 0.2 (IID drops), 65536 envs per B200",
    "c4": "Coverage --map 30 --sen 2 --den 0.06 --loss 0.1, 16384 envs per B200",
    "c5": "Predator-Prey --map 50 --sen 2 --den 0.08 --cap 4, 2048 envs per B200",
    "c3_ge": "Predator-Prey --map 20 --sen 2 --den 0.08 --cap 4, Gilbert-Elliot drops (Pgb 0.0196, Pbg 0.282, a transition per GCN layer), "
             "65536 envs per B200",
}
# BASELINE.md §2: the unmodified pure-Python reference (garage sampler + ma_gym env + CPU torch policy), one core,
# measured while the survey was written — NOT on this box; the reference cannot travel to the GPU box.
REFERENCE_PYTHON = {"c1": 1.6e3, "c2": 1.7e3, "c3": 5.3e3, "c4": 6.0e3, "c5": 7.2e3}
METRIC = "agent-steps/sec, batched PP/Coverage step+comm+policy rollout"
UNIT = "agent-steps/s"


def params_for(cfg):
    scen, m, sen, den, cap, loss, _ = CONFIGS[cfg]
    n = int(int(den * 100) * (m / 10) ** 2)
    p = dict(grid_size=m, Rsen=sen, n_agents=n, n_gcn_layers=2, loss_apply=1, mode="train", trpl=loss, trRcom=9, rm=0)
    if scen == "pp":
        p.update(n_preys=n, load=cap, max_env_steps=200, capture_reward=10, step_cost=0.1, penalty=0)
    else:
        p.update(n_groups=3, obstComplex="Easy", load=2, capture_reward=2, step_cost=0, penalty=1, revisit_penalty=0.5,
                 lazy_penalty=1, max_env_steps=400)
    return scen, p


def policy_flops_per_agent(D, n, L):
    return 2 * (D * 128 + 128 * 64) + 2 * 64 * 64 + 2 * 64 * n + L * (2 * 64 * 64 + 2 * n * 64) + \
        2 * (64 * 128 + 128 * 64 + 64 * 32 + 32 * 5)


def env_bytes_per_agent_step(spec):
    """SURVEY.md §8(d): 4 D [obs write] + S [state r/w] + (1+L) ceil(n/32) 4 [adj + channel rows] + E/n"""
    n, L, G = spec.n_agents, spec.n_layers, spec.grid
    S = 11.0 if spec.scenario == "pp" else 5.0 + 2.0 * ((G * G + 7) // 8) / n
    masks = (1 + L) * ((n + 31) // 32) * 4
    if spec.channel == 3:
        masks += 2 * L * ((n + 31) // 32) * 4
    return 4.0 * spec.obs_dim + S + masks + 16.0 / n


# ------------------------------------------------------------------------------------------------
# CPU port (oracle): the reference arm and the cpu_baseline leg
# ------------------------------------------------------------------------------------------------
def _cpu_worker(args):
    cfg, B, steps, seed, env_id0 = args
    os.environ["OMP_NUM_THREADS"] = os.environ["OPENBLAS_NUM_THREADS"] = os.environ["MKL_NUM_THREADS"] = "1"
    from oracle import oracle as orc
    scen, params = params_for(cfg)
    ospec = orc.spec_from_params(scen, params, seed=seed)
    env = orc.OracleVecEnv(ospec, B, env_id0=env_id0)
    rng = np.random.default_rng(seed)
    n, D, L = ospec["n"], ospec["D"], ospec["L"]
    w = _random_weights(D, L, rng)
    env.reset()
    # one untimed iteration, then the timed sample
    t0 = None
    for s in range(steps + 1):
        if s == 1:
            t0 = time.perf_counter()
        _, probs, _ = orc.policy_forward(w, env.obs, None, env.adj, env.chan)
        acts = env.sample_actions(probs)
        env.step(acts)
    return B * n * steps, time.perf_counter() - t0


def _random_weights(D, L, rng):
    def xav(o, i):
        lim = np.sqrt(6.0 / (i + o))
        return rng.uniform(-lim, lim, size=(o, i)).astype(np.float32)
    w = {"encoder._layers.0.linear.weight": xav(128, D), "encoder._layers.0.linear.bias": np.zeros(128, np.float32),
         "encoder._output_layers.0.linear.weight": xav(64, 128), "encoder._output_layers.0.linear.bias": np.zeros(64, np.float32),
         "attention_layer.linear_in.weight": xav(64, 64)}
    for l in range(L):
        w[f"gcn_layers.{l}.weight"] = rng.uniform(-0.125, 0.125, size=(64, 64)).astype(np.float32)
        w[f"gcn_layers.{l}.bias"] = rng.uniform(-0.125, 0.125, size=64).astype(np.float32)
    for i, (o, k) in enumerate(((128, 64), (64, 128), (32, 64))):
        w[f"categorical_output_layer._layers.{i}.linear.weight"] = xav(o, k)
        w[f"categorical_output_layer._layers.{i}.linear.bias"] = np.zeros(o, np.float32)
    w["categorical_output_layer._output_layers.0.linear.weight"] = xav(5, 32)
    w["categorical_output_layer._output_layers.0.linear.bias"] = np.zeros(5, np.float32)
    return w


def cpu_port_throughput(cfg, procs, envs_per_proc, steps):
    """P independent processes, each a single-threaded oracle rollout of its own envs; rates are summed
    (the reference cannot use more than one env per core either, SURVEY.md §2a)."""
    import multiprocessing as mp
    from oracle import oracle as orc
    orc.build()
    jobs = [(cfg, envs_per_proc, steps, 1 + i, i * envs_per_proc) for i in range(procs)]
    if procs == 1:
        from threadpoolctl import threadpool_limits
        with threadpool_limits(1):               # "cores": 1 means one thread, BLAS included
            res = [_cpu_worker(jobs[0])]
    else:
        for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
            os.environ[k] = "1"                  # inherited by the spawned workers before they import numpy
        with mp.get_context("spawn").Pool(procs) as pool:
            res = pool.map(_cpu_worker, jobs)
    return sum(a / t for a, t in res), sum(a for a, _ in res)


def reference_python_note(cfg):
    return {"value": REFERENCE_PYTHON[cfg], "unit": UNIT, "cores": 1,
            "where": "survey container (8-vCPU Xeon, Sapphire Rapids), NOT this box — BASELINE.md §2; the unmodified pure-Python "
                     "reference (garage sampler + ma_gym env + CPU torch policy) cannot travel to the GPU box"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    scen, params = params_for(args.config)
    n = params["n_agents"]
    # bounded sample: every "step" of this arm is one policy+env iteration over envs_per_proc envs on every core
    envs_per_proc = max(4, min(256, 20000 // max(n, 1)))
    # bounded: a single-process pilot fixes the step count so that every core works for ~15 s (the run stays within minutes)
    pilot_rate, _ = cpu_port_throughput(args.config, 1, envs_per_proc, 10)
    steps_cpu = int(max(10, min(200000, 15.0 * pilot_rate / (envs_per_proc * n))))
    t0 = time.perf_counter()
    rate, agent_steps = cpu_port_throughput(args.config, cores, envs_per_proc, steps_cpu)
    wall = time.perf_counter() - t0
    line = {"metric": METRIC, "value": rate, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * cores * envs_per_proc * n / rate,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+int", "data": "synthetic",
            "config": {"workload": WORKLOAD_TEXT[args.config], "config": args.config},
            "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{cores} processes x {envs_per_proc} envs x {steps_cpu} steps of the oracle port "
                                       f"(C env oracle + numpy fp32 policy, 1 thread each), wall {wall:.1f}s",
                             "reference_python": reference_python_note(args.config)},
            "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), file=args.out, flush=True)


# ------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md recipe)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.lines, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def close(self):
        """ends the sampling loop: nvidia-smi -lms would otherwise outlive a run that fails before stop()"""
        if self.proc is not None and self.proc.poll() is None:
            self.proc.terminate()
            self.proc.wait()

    def stop(self, t_lo, t_hi):
        """median SM clock and throttle reasons of the samples taken INSIDE [t_lo, t_hi] (the timed region)"""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        time.sleep(0.1)
        self.close()
        sm, mx, reasons, power = [], None, set(), []
        for ts, ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                clk, mxc = float(f[1]), float(f[2])
            except ValueError:
                continue
            mx = mxc
            if t_lo <= ts <= t_hi + 0.05:
                sm.append(clk)
                try:
                    power.append(float(f[3]))
                except ValueError:
                    pass
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm),
                "power_w_max": max(power) if power else None, "region_s": t_hi - t_lo}


# ------------------------------------------------------------------------------------------------
# one configuration on this rank's GPU
# ------------------------------------------------------------------------------------------------
class Ctx:
    def __init__(self, args):
        import torch
        import torch.distributed as dist
        from com_marl_b200 import distributed as D
        self.torch, self.dist, self.D = torch, dist, D
        self.rank, self.local_rank, self.world = D.init_from_env()
        if not torch.cuda.is_available():
            raise SystemExit("bench.py --impl b200 needs a GPU: the engine has no CPU path")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.numa = D.bind_to_gpu_numa(self.local_rank)
        self.args = args
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        self.hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        self.tc_peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0)))
        self.peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
        try:
            self.traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        except Exception:
            self.traffic = {}

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def max_over_ranks(self, *vals):
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t]


DUMP_BYTES = 64 << 20
DUMP_MAX_ENVS = 512


def dump_last_step(eng, out_dir):
    """Writes what RolloutEngine handed its caller for the last step it ran, as DIR/<name>.npy: the policy's actions and
    probabilities and the env's reward, done, counts, prey_alive_out, success (ring slot K - 1), the next observation,
    adjacency / channel bit rows and ave_deg (slot K), plus the episode-statistics sums of the whole run (episode_stats).
    Rows are a fixed seeded sample of at most DUMP_MAX_ENVS envs (their indices in env_index), fewer if the files would pass
    DUMP_BYTES.  float32 arrays stay float32; integers (bit rows included) become float64, which holds them exactly."""
    import torch
    t, K = eng.traj, eng.K
    rows = {k: t[k][K - 1] for k in ("actions", "probs", "reward", "done", "counts", "prey_alive_out", "success")}
    rows.update({k: t[k][K] for k in ("obs", "adj_bits", "chan_bits", "ave_deg")})
    per_env = sum(v[0].numel() * (4 if v.dtype == torch.float32 else 8) for v in rows.values())
    count = min(eng.B, DUMP_MAX_ENVS, (DUMP_BYTES - (1 << 20)) // per_env)
    idx = np.sort(np.random.default_rng(0).choice(eng.B, size=count, replace=False))
    sel = torch.as_tensor(idx, device=eng.device)
    arrays = {k: v.index_select(0, sel).cpu().numpy() for k, v in rows.items()}
    arrays["env_index"] = idx
    arrays["episode_stats"] = eng.local_stats().cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a.astype(np.float32 if a.dtype == np.float32 else np.float64))


def measure_config(cx, cfg, steps_req, warm_req, min_seconds, full, clocks=None, e2e_seconds=0.5, dump_dir=None):
    """rollout value / kernel rooflines / e2e of one BASELINE config on this rank's GPU; every rank runs it, all return the
    same record (times are max over ranks).  steps_req > 0 times exactly that many steps, 0 at least min_seconds."""
    torch, args, dev = cx.torch, cx.args, cx.dev
    from com_marl_b200.rollout import HostRollout, RolloutEngine, make_policy
    from com_marl_b200.scenario import ScenarioSpec
    base_cfg, spec_over = VARIANTS.get(cfg, (cfg, {}))
    scen, params = params_for(base_cfg)
    spec = ScenarioSpec.from_params(scen, params, seed=1, **spec_over)
    B = (args.envs if (args.envs and cfg == args.config) else CONFIGS[base_cfg][6])
    n, Dobs, L = spec.n_agents, spec.obs_dim, spec.n_layers
    # the engine runs whole graphs of `ring` steps: a ring that divides the requested count times exactly that count
    ring = max(k for k in range(1, min(args.ring, steps_req) + 1) if steps_req % k == 0) if steps_req > 0 else args.ring
    pol = make_policy(spec, device=dev)
    # independent env groups: 4 chains for teams up to 64 (8 when a chain still gets ~2000 policy tiles per launch — C3: measured
    # 849 -> 864 M agent-steps/s; smaller batches lose with 8), two chains for the three-launch pipeline of large teams (C5: 315 -> 320 M)
    groups = args.groups if args.groups > 0 else ((8 if B * n >= (1 << 21) else 4) if n <= 64 else 2)
    eng = RolloutEngine(spec, pol, B, device=dev, env_id0=cx.rank * B, ring=ring, use_graph=True, groups=groups)
    eng.reset()
    warm = max(3 * ring, ((warm_req + ring - 1) // ring) * ring)
    eng.run(warm - ring)                            # untimed: first chunk eager, graph captured on the second
    torch.cuda.synchronize(dev)
    # pilot (still warm-up): one replay, to size the timed region
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(); eng.run(ring); ev1.record()
    torch.cuda.synchronize(dev)
    pilot_ms, = cx.max_over_ranks(ev0.elapsed_time(ev1) / ring)
    steps = steps_req if steps_req > 0 else max(ring, int(np.ceil(min_seconds * 1e3 / max(pilot_ms, 1e-6) / ring)) * ring)
    # ---------------- value: device-resident rollout ----------------
    launches0 = eng.kernel_launches
    cx.barrier(); torch.cuda.synchronize(dev)
    t_lo = time.time()
    ev0.record()
    eng.run(steps)
    ev1.record()
    torch.cuda.synchronize(dev); cx.barrier()
    t_hi = time.time()
    ms = ev0.elapsed_time(ev1)
    launches = eng.kernel_launches - launches0
    eng.env.check_errors()
    pol.check_errors()
    if dump_dir is not None and cx.rank == 0:
        dump_last_step(eng, dump_dir)               # before the kernel timings below overwrite the ring
    clock_info = clocks.stop(t_lo, t_hi) if clocks is not None else None
    stats = cx.D.gather_stats(eng.local_stats())          # the rollout's only collective (NCCL over NVLink)
    # ---------------- per-kernel durations: CUDA events around a CUDA graph of launches of ONE kernel ----------------
    # (events around single eager launches would include the host's launch gaps, which are of the order of these kernels)
    eng._carry()
    t = eng.traj
    reps = 32 if full else 16
    gb0, gb1 = eng._ranges[0]
    Bk, ek = gb1 - gb0, eng._envs[0]

    packed = "obs_bits" in t            # the env kernel also writes the packed observation and the policy kernel reads it (as in the timed region)

    def policy_call(k, e, b0, b1):
        pk = dict(obs_bits=t["obs_bits"][k, b0:b1], obs_nbits=e.obs_nbits) if packed else {}
        pol.act_device(t["obs"][k, b0:b1], t["adj_bits"][k, b0:b1], t["chan_bits"][k, b0:b1], tick=e.tick, episode=e.episode,
                       probs=t["probs"][k, b0:b1], actions=t["actions"][k, b0:b1], env_id0=e.env_id0,
                       ws_slot=eng._envs.index(e) if e in eng._envs else 0, **pk)

    def env_call(k, e, b0, b1):
        out = dict(obs=t["obs"][k + 1, b0:b1], adj_bits=t["adj_bits"][k + 1, b0:b1], chan_bits=t["chan_bits"][k + 1, b0:b1],
                   ave_deg=t["ave_deg"][k + 1, b0:b1], reward=t["reward"][k, b0:b1], done=t["done"][k, b0:b1],
                   counts=t["counts"][k, b0:b1], prey_alive_out=t["prey_alive_out"][k, b0:b1], success_out=t["success"][k, b0:b1])
        if packed:
            out["obs_bits"] = t["obs_bits"][k + 1, b0:b1]
        e.step(t["actions"][k, b0:b1], out=out)

    def replay_ms(g, per):
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g.replay()
        a.record()
        for _ in range(3):
            g.replay()
        b.record()
        torch.cuda.synchronize(dev)
        return a.elapsed_time(b) / (3 * per)

    def time_alone(fn):
        for k in range(2):
            fn(k, ek, gb0, gb1)                     # warm (also keeps the ring consistent: slot k feeds slot k + 1)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for k in range(reps):
                fn(k % ring, ek, gb0, gb1)
        return replay_ms(g, reps)

    def time_groups(fn, alone):
        """all env groups' launches of one kernel, concurrently on the groups' streams like in the timed region: the
        wall time of one such round / number of groups = the launch duration under the concurrency it really runs at"""
        G = len(eng._ranges)
        if G == 1:
            return alone
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            main = torch.cuda.current_stream(dev)
            fork = torch.cuda.Event(); fork.record(main)
            for st in eng._streams:
                st.wait_event(fork)
            for k in range(reps):
                for g, (b0, b1) in enumerate(eng._ranges):
                    with torch.cuda.stream(eng._streams[g]):
                        fn(k % ring, eng._envs[g], b0, b1)
            for st in eng._streams:
                j = torch.cuda.Event(); j.record(st); main.wait_event(j)
        return replay_ms(gr, reps * G)

    pol_alone_ms = time_alone(policy_call)
    env_alone_ms = time_alone(env_call)
    pol_ms = time_groups(policy_call, pol_alone_ms)
    env_ms = time_groups(env_call, env_alone_ms)
    n_groups = len(eng._ranges)
    episode_stats = cx.D.summarize_stats(stats, spec.scenario, n)
    tc = pol.uses_tensor_cores()
    # ---------------- value with the attention weights recorded (the reference returns them every step) ----------------
    att = None
    del eng, t, ek
    torch.cuda.empty_cache()
    if full and getattr(pol, "comm", False):
        ring_a = min(ring, 16)
        eng = RolloutEngine(spec, pol, B, device=dev, env_id0=cx.rank * B, ring=ring_a, use_graph=True, groups=groups, record_attention=True)
        eng.reset()
        eng.run(3 * ring_a)
        torch.cuda.synchronize(dev)
        sa = max(ring_a, int(np.ceil(0.5 * steps / ring_a)) * ring_a)
        cx.barrier(); torch.cuda.synchronize(dev)
        ev0.record(); eng.run(sa); ev1.record()
        torch.cuda.synchronize(dev); cx.barrier()
        ms_a, = cx.max_over_ranks(ev0.elapsed_time(ev1))
        att = {"value": sa * B * n * cx.world / (ms_a * 1e-3), "unit": UNIT, "steps": sa, "ms_per_step": ms_a / sa,
               "attention_bytes_per_step": B * n * n * 4,
               "note": "the same device-resident loop with agent_infos['attention_weights'] (B x n x n fp32) written into the "
                       "trajectory ring by the policy kernel every step"}
        del eng
        torch.cuda.empty_cache()
    # ---------------- e2e: host buffers through the sampler-level call ----------------
    NB = args.e2e_batches if (args.e2e_batches > 0 and B % max(1, args.e2e_batches) == 0) else 1
    hr = HostRollout(spec, pol, B, device=dev, env_id0=cx.rank * B, parts=NB, host_slots=2)
    hr.reset()
    checksum = [0.0]

    def e2e_loop(k):
        """k steps, one step in flight ahead of the one whose host buffers are read"""
        hr.submit()
        for i in range(k):
            if i + 1 < k:
                hr.submit()
            outs = hr.collect()
            checksum[0] += float(outs[0]["reward"][0])         # the host really reads the step's result
    e2e_loop(4)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter(); e2e_loop(4); pilot = (time.perf_counter() - t0) / 4
    pilot, = cx.max_over_ranks(pilot)
    e2e_steps = int(max(8, min(args.e2e_steps, np.ceil(e2e_seconds / max(pilot, 1e-6)))))
    cx.barrier(); torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    e2e_loop(e2e_steps)
    torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - t0
    cx.barrier()
    hr.check_errors()
    h2d, d2h = hr.bytes_per_step()
    del hr
    torch.cuda.empty_cache()
    step_api = None
    if full:
        step_api = measure_e2e_step_api(cx, spec, pol, B, NB, e2e_seconds)
    ms_max, e2e_max = cx.max_over_ranks(ms, e2e_s)
    agent_steps = steps * B * n * cx.world
    value = agent_steps / (ms_max * 1e-3)
    flops = policy_flops_per_agent(Dobs, n, L) * Bk * n               # per launch (one env group)
    env_bytes = env_bytes_per_agent_step(spec) * Bk * n
    kname = ("policy_tc_kernel<comm>" if n <= 64 else "policy_tc_kernel<enc> + policy_attn_mma_kernel + policy_tc_kernel<head>") if tc \
        else ("policy_small_kernel" if n <= 64 else "policy_large_kernel")
    traffic = cx.traffic.get(cfg, {}) if (cfg in CONFIGS and B == CONFIGS[cfg][6]) else {}
    if n <= 64:
        pol_traffic = traffic.get(kname, traffic.get("policy_tc_kernel"))
    else:
        parts = [traffic.get(k) for k in ("policy_tc_kernel<enc>", "policy_attn_mma_kernel", "policy_tc_kernel<head>")]
        pol_traffic = sum(parts) if all(p is not None for p in parts) else None
    # what the tensor pipe actually executes per 128-row tile: 3 passes over the padded dense layers
    Dp = (Dobs + 15) // 16 * 16
    dense_mac = Dp * 128 + 128 * 64 + 64 * 64 * (1 + L) + 64 * 128 + 128 * 64 + 64 * 32 + 32 * 16
    rows_per_tile = (128 // n) * n if n <= 64 else 128            # whole envs per tile (n <= 64) / any 128 rows (large teams)
    tc_flops = (3 * 2 * dense_mac * 128 * ((Bk * n + rows_per_tile - 1) // rows_per_tile)) if tc else 0
    pol_tflops = flops / (pol_ms * 1e-3) / 1e12
    env_gbs = env_bytes / (env_ms * 1e-3) / 1e9
    rec = {
        "value": value, "unit": UNIT, "steps": steps, "warmup": warm, "ms_per_step": ms_max / steps, "timed_region_s": ms_max * 1e-3,
        "gpu_launches": launches * cx.world,
        "config": {"workload": WORKLOAD_TEXT[cfg], "config": cfg, "envs_per_gpu": B, "n_agents": n,
                   "obs_dim": Dobs, "ring_slots": ring, "env_groups": n_groups,
                   "attention": ("not recorded in `value` (RolloutEngine(record_attention=False)); `value_with_attention` times the "
                                 "loop that writes it") if full else "not recorded",
                   "l2": f"inputs are produced by the previous step; the trajectory ring ({ring + 1} slots, "
                         f"{(ring + 1) * B * n * Dobs * 4 / 2**20:.0f} MiB of observations) is larger than the 126 MB L2, "
                         "so no slot survives a ring cycle in cache",
                   "observations": "the env kernel writes the fp32 contract rows (4 D bytes per agent) into the trajectory ring AND a packed copy "
                                   "(window bits + scalar columns, 24 bytes per agent) that the policy kernel reads instead; roofline_env counts "
                                   "the SURVEY 8(d) bytes (fp32 rows), the extra 24 bytes per agent are not credited",
                   "streams": "on-device Philox4x32-10 (spawn, prey walk, channel draws, action sampling)"},
        "e2e": {"value": e2e_steps * B * n * cx.world / e2e_max, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": e2e_steps, "batches": NB, "ms_per_step": 1e3 * e2e_max / e2e_steps,
                "api": "HostRollout.submit/collect = cm_rollout_step_host, the sampler-level boundary (one C call per env part and step: "
                       "H2D availability bytes, policy forward -> env step on device-resident state, D2H next observation + masks + "
                       "ave_deg + reward + done + counts + prey_alive + success + actions + probabilities into pinned host memory); "
                       f"{NB} env parts on their own streams, one step in flight ahead of the one the host reads",
                "step_api": step_api},
        "roofline": {"bound": "tensor", "kernel": kname,
                     "achieved": pol_tflops, "peak": cx.tc_peak, "unit": "TFLOP/s", "frac": pol_tflops / cx.tc_peak, "traffic": pol_traffic,
                     "peak_source": cx.peak_src + ", bf16 dense sustained; the kernel issues A_hi x [B_hi;B_lo] and A_lo x B_hi in fp16 per "
                                    "algorithmic product (error compensation) on padded K, so the tensor pipe executes ~3.3x the algorithmic FLOPs counted here",
                     "flop_per_launch": flops, "tensor_flop_issued_per_launch": tc_flops, "ms_per_launch": pol_ms,
                     "share_of_step": pol_ms / (pol_ms + env_ms), "envs_per_launch": Bk, "launches_per_step": n_groups,
                     "ms_per_launch_alone": pol_alone_ms,
                     "note": "one launch = one env group; ms_per_launch = wall time of the groups' concurrent launches (separate streams, as in "
                             "the timed region; CUDA graph, CUDA events) / number of groups; ms_per_launch_alone = the same launch with the GPU to itself"},
        "roofline_env": {"bound": "hbm", "kernel": "env_kernel", "achieved": env_gbs, "peak": cx.hbm_peak, "unit": "GB/s",
                         "frac": env_gbs / cx.hbm_peak, "traffic": traffic.get("env_kernel"), "bytes_per_launch": env_bytes, "ms_per_launch": env_ms,
                         "bytes_per_agent_step": env_bytes_per_agent_step(spec), "peak_source": cx.peak_src, "envs_per_launch": Bk,
                         "launches_per_step": n_groups, "ms_per_launch_alone": env_alone_ms},
        "episode_stats": episode_stats,
    }
    if att is not None:
        rec["value_with_attention"] = att
    if clock_info is not None:
        rec["clocks"] = clock_info
    rec["_tc"] = tc
    return rec


def measure_e2e_step_api(cx, spec, pol, B, NB, seconds):
    """the step-level pair of host calls (round 1's e2e): policy.get_actions_host + BatchedEnv.step_host — observations +
    masks + actions go H2D and every result D2H each step; event-driven antiphase over NB env parts"""
    torch, dev = cx.torch, cx.dev
    from com_marl_b200.envs import BatchedEnv
    n = spec.n_agents
    Bh = B // NB
    henvs = [BatchedEnv(spec, Bh, device=dev, env_id0=cx.rank * B + h * Bh) for h in range(NB)]
    hstreams = [torch.cuda.Stream(dev) for _ in range(NB)]
    outs = [e.reset_host() for e in henvs]
    torch.cuda.synchronize(dev)

    def pol_phase(h):
        pin = outs[h]["pinned"]            # host (pinned) buffers filled by the previous step of this part
        a, _, ev = pol.get_actions_host(pin["obs"], pin["adj_bits"], pin["chan_bits"], inputs_arena=True, slot=100 + h, sync=False,
                                        stream=hstreams[h])
        return a, ev

    def env_phase(h, acts):
        return henvs[h].step_host(acts, sync=False, stream=hstreams[h])

    phase, pend, evs = {}, {}, {}
    for h in range(NB):
        pend[h], evs[h] = pol_phase(h)
        phase[h] = "pol"
        if h % 2 == 1:
            evs[h].synchronize()
            outs[h], evs[h] = env_phase(h, pend[h])
            phase[h] = "env"

    def iteration():                   # every part advances by one full step (one policy call + one env step)
        for _ in range(2):
            for h in range(NB):
                evs[h].synchronize()
                if phase[h] == "pol":
                    outs[h], evs[h] = env_phase(h, pend[h])
                    phase[h] = "env"
                else:
                    pend[h], evs[h] = pol_phase(h)
                    phase[h] = "pol"

    for _ in range(3):
        iteration()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter(); iteration(); iteration(); pilot = (time.perf_counter() - t0) / 2
    pilot, = cx.max_over_ranks(pilot)
    k = int(max(5, min(cx.args.e2e_steps, np.ceil(seconds / max(pilot, 1e-6)))))
    cx.barrier(); torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for _ in range(k):
        iteration()
    torch.cuda.synchronize(dev)
    s = time.perf_counter() - t0
    cx.barrier()
    for e in henvs:
        e.check_errors()
    ph2d, pd2h = pol.host_call_bytes(B)
    eh2d, ed2h = [sum(x) for x in zip(*[e.host_step_bytes() for e in henvs])]
    s_max, = cx.max_over_ranks(s)
    del henvs
    pol.__dict__.pop("_stages", None)
    torch.cuda.empty_cache()
    return {"value": k * B * n * cx.world / s_max, "unit": UNIT, "h2d_bytes_per_step": ph2d + eh2d, "d2h_bytes_per_step": pd2h + ed2h,
            "steps": k, "api": "policy.get_actions_host + BatchedEnv.step_host = cm_policy_forward_host + cm_env_step_host"}


def measure_c5_ppo(cx, envs, rounds=2):
    """BASELINE configs[4]: PP 50/2/.08 cap 4, comm-GNN rollout + PPO update; with N > 1 every optimizer step all-reduces the
    flat policy and critic gradient buckets over NCCL inside the timed region (SURVEY.md 8e-2)."""
    torch, dev = cx.torch, cx.dev
    from com_marl_b200.scenario import ScenarioSpec
    from com_marl_b200.train import DeviceTrainer
    scen, params = params_for("c5")
    spec = ScenarioSpec.from_params(scen, params, seed=1)
    tr = DeviceTrainer(spec, envs, device=dev, env_id0=cx.rank * envs, optimization_mini_epochs=2)
    tr.train_epoch()                         # warm-up rounds: allocations, cuBLAS handles, NCCL communicator (first, eager chunk) ...
    tr.train_epoch()                         # ... and the capture of the rollout graph (second chunk)
    torch.cuda.synchronize(dev)
    cx.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    outs = [tr.train_epoch() for _ in range(rounds)]
    ev1.record()
    torch.cuda.synchronize(dev); cx.barrier()
    ms, = cx.max_over_ranks(ev0.elapsed_time(ev1))
    o = outs[-1]
    steps_opt = len(o["losses"])
    csum = torch.tensor([tr.weights_checksum()], dtype=torch.float64, device=dev)
    lo, hi = csum.clone(), csum.clone()
    if cx.world > 1:
        cx.dist.all_reduce(lo, op=cx.dist.ReduceOp.MIN); cx.dist.all_reduce(hi, op=cx.dist.ReduceOp.MAX)
    agent_steps = rounds * o["agent_steps"] * cx.world
    rec = {"value": agent_steps / (ms * 1e-3), "unit": UNIT, "what": "rollout of one 200-step horizon for every env + PPO update "
           f"({steps_opt} optimizer steps = 2 mini-epochs x 3 minibatches; policy and critic gradient buckets "
           + ("all-reduced over NCCL every step" if cx.world > 1 else "no all-reduce at N = 1") + "), per round",
           "workload": WORKLOAD_TEXT["c5"].replace("2048", str(envs)), "envs_per_gpu": envs, "rounds": rounds, "ms_per_round": ms / rounds,
           "rollout_ms": o["rollout_ms"], "batch_ms": o["batch_ms"], "update_ms": o["update_ms"], "optimizer_steps_per_round": steps_opt,
           "allreduce_calls_per_round": (2 * steps_opt) if cx.world > 1 else 0, "n_paths_per_rank": o["n_paths"],
           "loss_before": o["loss_before"], "loss_after": o["loss_after"], "kl": o["kl"],
           "update_path": ("hand-written forward + backward kernels (cm_ppo_net: exact fp32, csrc/ppo_net_kernels.cu) + cm_adam_step"
                           if tr.algo._fused is not None else "torch autograd + cm_adam_step"),
           "weights_identical_on_all_ranks": bool(float(lo) == float(hi))}
    del tr
    torch.cuda.empty_cache()
    return rec


def run_b200_arm(args):
    cx = Ctx(args)
    clocks = ClockSampler(cx.local_rank) if cx.rank == 0 else None
    if clocks is not None:
        clocks.start()
        time.sleep(0.2)
    try:
        main = measure_config(cx, args.config, args.steps, args.warmup, args.min_seconds, True, clocks, dump_dir=args.dump_outputs)
    finally:
        if clocks is not None:
            clocks.close()
    sweep = {}
    if not args.no_sweep:
        names = [c for c in (("c4",) if cx.world > 1 else ("c1", "c2", "c3", "c3_ge", "c4", "c5")) if c != args.config]
        for c in names:
            r = measure_config(cx, c, 0, 0, args.min_seconds, False, None, e2e_seconds=0.3)
            sweep[c] = {k: r[k] for k in ("value", "ms_per_step", "steps", "timed_region_s", "e2e", "roofline", "roofline_env")}
            sweep[c]["workload"] = r["config"]["workload"]
            for k in ("api", "step_api"):
                sweep[c]["e2e"].pop(k, None)
        sweep["c5_ppo"] = measure_c5_ppo(cx, args.ppo_envs)
    if cx.rank != 0:
        if cx.world > 1:
            cx.dist.destroy_process_group()
        return
    tc = main.pop("_tc")
    line = {
        "metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": cx.world, "steps": main["steps"], "warmup": main["warmup"],
        "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": ("f32-equivalent: error-compensated fp16-split tcgen05 products (x = hi + 2^-12 lo) with fp32 accumulation in TMEM (policy)"
                  if tc else "f32 FFMA (policy)") + " + u8/u16/u64 bit rows (env, comm)",
        "data": "synthetic", "timed_region_s": main["timed_region_s"],
        "steps_note": f"the timed region is exactly --steps {args.steps} steps, replays of a {main['config']['ring_slots']}-step graph; "
                      f"--warmup {args.warmup} was rounded up to whole replays (at least 3)",
        "config": main["config"], "e2e": main["e2e"], "gpu_launches": main["gpu_launches"],
        "roofline": main["roofline"], "roofline_env": main["roofline_env"], "clocks": main.get("clocks"),
        "episode_stats": main["episode_stats"], "host_affinity": cx.numa,
    }
    if "value_with_attention" in main:
        line["value_with_attention"] = main["value_with_attention"]
    if sweep:
        line["configs"] = sweep
    if cx.world == 1 and not args.no_cpu_baseline:
        t0 = time.perf_counter()
        n = main["config"]["n_agents"]
        Bc = max(8, min(512, 40000 // n))
        pilot_rate, _ = cpu_port_throughput(args.config, 1, Bc, 10)
        Sc = int(max(10, min(200000, 10.0 * pilot_rate / (Bc * n))))      # ~10 s of single-thread CPU work
        rate, _ = cpu_port_throughput(args.config, 1, Bc, Sc)
        line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": 1, "kind": "port",
                                "sample": f"{Bc} envs x {Sc} steps of the oracle port (C env oracle + numpy fp32 policy), "
                                          f"1 thread, {time.perf_counter() - t0:.1f}s",
                                "reference_python": reference_python_note(args.config)}
    print(json.dumps(line), file=args.out, flush=True)
    if cx.world > 1:
        cx.dist.destroy_process_group()


def _quiet_stdout():
    """Libraries (NCCL's version banner, torchrun notices) print to fd 1; the contract is ONE JSON line on stdout.
    Route fd 1 to stderr for the whole run and hand back a handle on the real stdout for the final line."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = os.fdopen(os.dup(2), "w")
    return real


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=256)
    ap.add_argument("--warmup", type=int, default=192)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c3", choices=sorted(CONFIGS))
    ap.add_argument("--envs", type=int, default=0, help="envs per GPU of --config (default: the config's)")
    ap.add_argument("--ring", type=int, default=64, help="trajectory ring slots = steps per CUDA graph (at most; see `value`)")
    ap.add_argument("--min-seconds", type=float, default=0.25, help="floor on the timed region of each config of the sweep")
    ap.add_argument("--e2e-steps", type=int, default=2000, help="cap on the steps of an e2e (host-buffer) loop")
    ap.add_argument("--e2e-batches", type=int, default=4, help="independent env parts of the e2e (host-buffer) loops")
    ap.add_argument("--groups", type=int, default=0, help="independent env groups, each a policy->step chain on its own stream (0: 4 or 8 for teams <= 64, else 2)")
    ap.add_argument("--ppo-envs", type=int, default=128, help="envs per GPU of the c5_ppo sub-record")
    ap.add_argument("--no-sweep", action="store_true", help="skip the configs sweep and the c5_ppo sub-record")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    args.out = _quiet_stdout()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
