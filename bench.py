#!/usr/bin/env python3
"""
bench.py -- env-steps/sec of the gym-fx env.step() hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2|cfg3|cfg4|cfg5]
                  [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" = one env.step() of every env of the workload.  Default
workload = BASELINE configs[1]: 4096 envs/GPU, feature_window_preprocessor (window=128, 5 OHLCV features, rolling
z-score over 256 bars), direct_fixed_sltp, pnl_reward, synthetic EURUSD 1-min candles (2^19 bars, SURVEY 8d).

ours:       K steps through fxenv_step_many in batches of <= 500 (actions pre-generated on the device, observation rows
            rotating through a ring LARGER than L2 so every step's stores reach HBM).  The library runs a batch either
            as ONE persistent launch whose warps pull (step, env) tickets and honour per-env dependencies, or as a CUDA
            graph of single-step launches (include/fxenv.h: fxenv_step_many_engine) -- `config.engine` says which.
            `value` = whole-job env-steps/s (inputs resident in HBM), max-over-ranks device time.
            `single_step_graph` = the same K steps forced through the graph of grid-serialised single steps.
            `e2e`   = same metric through the reference-facing host-buffer call (fxenv_step_host): per step H2D of
            the actions from pinned memory, the kernel, D2H of obs/reward/terminated, host sync.
            `roofline` = algorithmic bytes per launch / average launch duration vs measured HBM peak.
            `cpu_baseline` = the C oracle port timed on this box's host cores (rank 0, N=1, bounded sample).
            `closed_loop` = BASELINE configs[3] shape with the policy IN the loop (fused tcgen05 actor-critic kernel <->
            env step, VecFxEnv.rollout) and one PPO update with its NCCL all-reduces (time per update and share).
            `other_workloads` (N=1) = short runs of BASELINE configs[2] and configs[4] (cfg3 / cfg5 shapes).
            --dump-outputs DIR: after the timed steps, rank 0 writes what the last timed step handed back (see
            dump_outputs) as DIR/<name>.npy.  Inputs are seeded, so two builds run with the same arguments can be
            compared output for output.
reference:  the CPU arm: the oracle port (oracle/fxenv_oracle.c; the Python reference cannot travel to the GPU box)
            stepping the SAME workload with all host threads.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

OHLCV = ["OPEN", "HIGH", "LOW", "CLOSE", "VOLUME"]
DEFAULTS = {"initial_cash": 10000.0, "position_size": 1.0, "commission": 0.0, "slippage": 0.0, "price_column": "CLOSE"}
WORKLOADS = {
    # name: (envs/GPU, window, strategy, reward, pairs, R = reward-state bytes per env-step (SURVEY 8d))
    "cfg2": (4096, 128, "direct_fixed_sltp", "pnl_reward", 1, 0),
    "cfg3": (16384, 256, "direct_atr_sltp", "dd_penalized_reward", 1, 16),
    "cfg4": (4096, 128, "direct_fixed_sltp", "sharpe_reward", 1, 520),
    "cfg5": (8192, 512, "direct_atr_sltp", "sharpe_reward", 4, 520),
}
T_BARS = 1 << 19
L2_BYTES = 126 * 1024 * 1024
ORDER_CAP = int(os.environ.get("FXENV_ORDER_CAP", "256"))  # order-table entries per env (overflowing envs are reported)


def build_workload(name, envs_per_gpu=None, n_shards=1):
    """-> (cfg for envs_per_gpu * n_shards envs, candles, minutes, envs_per_gpu, obs_dim, algorithmic bytes per env-step,
    description).  n_shards > 1 only for the CPU arm, which steps the envs of all N GPUs in one process."""
    from gym_fx_b200.config import lower_config
    from gym_fx_b200.plugin_loader import DEFAULT_PLUGINS, build_plugins
    from gym_fx_b200.synth import PAIR_PIP, synth_candles, synth_minutes

    envs, W, strat, rew, pairs, R = WORKLOADS[name]
    W = int(os.environ.get("FXENV_BENCH_WINDOW", W))  # experiments only
    if envs_per_gpu:
        envs = envs_per_gpu
    cfgd = {**DEFAULTS, "window_size": W, "feature_columns": list(OHLCV)}
    pl = build_plugins(cfgd, {**DEFAULT_PLUGINS, "strategy": strat, "reward": rew,
                              "preprocessor": "feature_window_preprocessor"})
    cfg = lower_config(cfgd, broker_plugin=pl["broker"], strategy_plugin=pl["strategy"],
                       preprocessor_plugin=pl["preprocessor"], reward_plugin=pl["reward"], columns=OHLCV,
                       num_envs=envs * n_shards, num_pairs=pairs, order_capacity=ORDER_CAP,
                       pair_pip_size=list(PAIR_PIP[:pairs]) if pairs > 1 else None)
    cfg.auto_reset = 1   # SURVEY 8d: auto-reset on (episodes span the table, so `terminated_frac` stays 0 in a run)
    candles = [synth_candles(T_BARS, p) for p in range(pairs)]
    minutes = [synth_minutes(T_BARS) for _ in range(pairs)]
    D = W * 5 + 2 * W + 4
    algo_bytes = 4 * D + 4 + 1 + 4 + R  # per env-step (SURVEY 8d)
    desc = (f"{name}: {envs} envs/GPU, feature_window W={W} F=5 rolling_zscore S=256, {strat}, {rew}, "
            f"{pairs} pair(s), synthetic 1-min candles T=2^19")
    return cfg, candles, minutes, envs, D, algo_bytes, desc


def preroll_steps(cfg):
    """Untimed steps every episode is advanced by before the warm-up, so that the measured steps are the ones an episode
    consists of (the tables hold 2^19 bars): windows full, z-score statistics from the full rolling window.  The first
    max(window, scaling_window) steps of an episode run the padded-window / running-statistics paths instead."""
    return int(max(cfg.window_size, cfg.scaling_window if cfg.scaling != 0 else 0)) + 16


def common_config(desc, envs_per_gpu, D, world, preroll):
    """The `config` object of the JSON line: identical for both arms (`--impl ours` / `--impl reference`) of one run."""
    return {"workload": desc, "envs_per_gpu": envs_per_gpu, "obs_dim": D, "parallelism": f"env-shard x{world}",
            "actions": "uniform {0,1,2}, i.i.d. per env-step, seeded", "auto_reset": True,
            "episode_phase": f"steady state: every episode advanced {preroll} untimed steps (> window, scaling window) "
                             "before the warm-up steps"}


def pin_to_gpu_numa_node(local_rank):
    """Bind this process (and therefore the pinned host buffers it allocates afterwards: first touch) to the CPU cores
    of the NUMA node its GPU hangs off, so that host<->device copies of different ranks do not cross the socket link."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = torch.cuda.get_device_properties(local_rank).pci_domain_id
        dev = torch.cuda.get_device_properties(local_rank).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.extend(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return {"numa_node": node, "cpus": len(allowed)}
    except Exception:
        return None
    return None


class ClockSampler:
    """SM clock / throttle-reason sampler running DURING the timed region (B200_PROFILING.md).  NVML polled every ~2 ms
    from a thread (the timed region is tens of milliseconds, too short for `nvidia-smi -lms`); falls back to nvidia-smi."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.nvml, self._stop = [], None, None, False
        self.sm, self.mx, self.bits = [], None, 0
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            try:
                uuid = "GPU-" + str(torch.cuda.get_device_properties(index).uuid)   # robust to CUDA_VISIBLE_DEVICES
                try:
                    self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
                except Exception:
                    self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.nvml = pynvml
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(index)], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        while not self._stop:
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
                self.bits |= int(n.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                try:
                    self.bits |= int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                except Exception:
                    pass
            time.sleep(0.002)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self._stop = True
            self.th.join(timeout=1)
            n = self.nvml
            names = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))
            reasons = sorted(nm for nm, bit in names if self.bits & bit)
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.mx, "reasons": reasons,
                    "samples": len(self.sm), "source": "nvml, 2 ms polling during the timed region"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "source": "nvidia-smi -lms 50"}


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def cpu_port_rate(workload, total_envs, steps, warmup, threads, budget_s=None):
    """env-steps/s of the oracle port on the host: every env stepped `steps` times by `threads` host threads, each
    thread running its env slice through the steps without a per-step barrier (envs are independent)."""
    from gym_fx_b200.synth import start_offsets
    from oracle.c_oracle import OracleVec, ParallelStepper

    cfg, candles, minutes, envs, D, _, desc = build_workload(workload, total_envs)
    vec = OracleVec(cfg, candles, minutes)
    pre = preroll_steps(cfg)
    vec.reset(start_offsets(total_envs, T_BARS, steps + warmup + pre + 64, 256))
    ps = ParallelStepper(vec, threads)
    rng = np.random.default_rng(1234)
    chunk = 8
    acts = rng.integers(0, 3, (chunk, total_envs)).astype(np.int32)
    for _ in range(-(-pre // chunk)):        # same episode phase as the GPU arm (preroll_steps)
        ps.run(acts)
    if warmup:
        ps.run(acts[:min(warmup, chunk)])
    t0 = time.perf_counter()
    done = 0
    while done < steps:
        k = min(chunk, steps - done)
        ps.run(acts[:k])
        done += k
        if budget_s is not None and time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    vec.close()
    return total_envs * done / dt, done, dt, ps.threads, desc, pre


def run_reference(args, rank, world):
    """--impl reference: the CPU arm (oracle port, all host threads), rank 0 only."""
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    envs_per_gpu = args.envs or WORKLOADS[args.workload][0]
    total = envs_per_gpu * args.gpus
    rate, done, dt, used, _, pre = cpu_port_rate(args.workload, total, args.steps, args.warmup, threads)
    _, _, _, _, D, _, desc = build_workload(args.workload, envs_per_gpu)
    line = {
        "impl": "reference", "metric": "env-steps/sec", "value": rate, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": done, "warmup": args.warmup, "ms_per_step": dt / done * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": common_config(desc, envs_per_gpu, D, args.gpus, pre),
        "details": {"total_envs": total,
                    "note": "CPU arm: C port of the reference path (oracle/fxenv_oracle.c) stepping the envs of all "
                            f"{args.gpus} GPU shard(s) on this host; the Python reference (measured in the build container "
                            "over the backtrader shim: 676 steps/s/process at this shape, "
                            "profiles/r1_reference_python_rate.json) cannot travel to the GPU box"},
        "cpu_baseline": {"value": rate, "unit": "env-steps/s", "cores": used, "kind": "port",
                         "sample": f"{total} envs x {done} steps, {used} host threads (pthreads), each thread runs its env slice without a per-step barrier"},
        "e2e": {"value": rate, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit_json(line)


def single_step_graph_rate(args, cfg, candles, minutes, N, starts, acts, ring, rews, terms, chunk):
    """The same steps through the other fxenv_step_many engine (CUDA graph of grid-serialised single-step launches),
    which is also what a policy-in-the-loop caller of fxenv_step gets: reported next to `value` for transparency."""
    import torch
    from gym_fx_b200.vec_env import VecFxEnv

    os.environ["FXENV_ENGINE"] = "graph"
    try:
        env = VecFxEnv(cfg, candles, minutes, device=ring.device)
    finally:
        del os.environ["FXENV_ENGINE"]
    env.reset(starts)
    K = min(args.steps, 2 * chunk)
    reps = max(1, K // chunk)
    for _ in range(2):
        env.step_many(acts, ring, rews, terms)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(reps):
        env.step_many(acts, ring, rews, terms)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    env.close()
    return {"value": N * reps * chunk / (ms * 1e-3), "unit": "env-steps/s", "ms_per_step": ms / (reps * chunk), "steps": reps * chunk,
            "note": "CUDA graph of single-step launches (grid-wide dependency between steps, programmatic dependent launch)"}


def short_workload_rate(name, K, dev):
    """`other_workloads`: a short device-resident run (K steps after 3 warm-up steps, same rules as the main measurement)
    of another BASELINE shape on this GPU: value / us per step / roofline fraction / engine."""
    import torch
    from gym_fx_b200.sharding import shard_starts
    from gym_fx_b200.vec_env import VecFxEnv

    cfg, candles, minutes, N, D, algo_bytes, desc = build_workload(name)
    env = VecFxEnv(cfg, candles, minutes, device=dev)
    pre = preroll_steps(cfg)
    env.reset(torch.as_tensor(shard_starts(N, 0, 1, T_BARS, 2 * K + pre + K + 64, 256)))
    gen = torch.Generator(device=dev)
    gen.manual_seed(4321)
    acts = torch.randint(0, 3, (K, N), generator=gen, device=dev, dtype=torch.int32)
    slots = max(2, -(-int(L2_BYTES * 1.8) // (N * D * 4)))
    ring = torch.empty((slots, N, D), dtype=torch.float32, device=dev)
    rews = torch.empty((K, N), dtype=torch.float32, device=dev)
    terms = torch.empty((K, N), dtype=torch.uint8, device=dev)
    plan = env.plan_step_many(acts, ring, rews, terms)
    for _ in range(-(-pre // K) + 1):       # episodes into steady state, then the warm-up: K >= 3 steps
        plan()
    torch.cuda.synchronize(dev)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    plan()
    ev1.record()
    torch.cuda.synchronize(dev)
    ms = ev0.elapsed_time(ev1)
    peak, _ = measured_peak_gbs()
    out = {"workload": desc, "value": N * K / (ms * 1e-3), "unit": "env-steps/s", "ms_per_step": ms / K, "steps": K,
           "engine": env.step_many_engine(K), "roofline_frac": N * algo_bytes / (ms * 1e-3 / K) / 1e9 / peak,
           "order_overflow_envs": int((env.info()["flags"] & 16).ne(0).sum().item())}
    env.close()
    del ring
    torch.cuda.empty_cache()
    return out


def closed_loop_block(K, rank, world, dev, dist):
    """BASELINE configs[3]: 4096 envs/GPU (W=128, fixed SL/TP, sharpe_reward) with a PPO actor-critic MLP(256,256) IN the
    loop -- the fused tcgen05 policy kernel between the env steps (VecFxEnv.rollout) -- followed by one PPO update whose
    gradients / advantage statistics cross the ranks by NCCL all-reduce.  Device time, max over ranks."""
    import torch
    from gym_fx_b200.learner import ActorCritic, ppo_update
    from gym_fx_b200.sharding import shard_starts
    from gym_fx_b200.vec_env import VecFxEnv

    cfg, candles, minutes, N, D, _, desc = build_workload("cfg4")
    env = VecFxEnv(cfg, candles, minutes, device=dev)
    H = 32 if K >= 8 else max(2, K)                          # rollout horizon (not tied to --steps: a PPO-sized chunk)
    reps = max(1, min(8, K // H))
    pre = preroll_steps(cfg)
    env.reset(torch.as_tensor(shard_starts(N, rank, world, T_BARS, (reps + 3) * H + pre + 128, 256)))
    gen = torch.Generator(device=dev)
    gen.manual_seed(77 + rank)
    pa = torch.randint(0, 3, (64, N), generator=gen, device=dev, dtype=torch.int32)
    pring = torch.empty((2, N, D), dtype=torch.float32, device=dev)
    prew, pterm = torch.empty((64, N), dtype=torch.float32, device=dev), torch.empty((64, N), dtype=torch.uint8, device=dev)
    for _ in range(-(-pre // 64)):                           # episodes into steady state (preroll_steps), random actions
        env.step_many(pa, pring, prew, pterm)
    del pring
    torch.manual_seed(0)                                     # identical replicas on every rank
    torch.backends.cuda.matmul.allow_tf32 = True
    net = ActorCritic(D).to(dev)
    opt = torch.optim.Adam(net.parameters(), lr=3e-4, eps=1e-5)
    pol = env.make_policy(net)
    buf = env.rollout(pol, H, seed=rank)                     # warm-up (instantiates the graph), also the learner's batch
    env.rollout(pol, H, buffers=buf, seed=rank + 1000)
    if dist:
        dist.barrier()
    torch.cuda.synchronize(dev)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for r in range(reps):
        env.rollout(pol, H, buffers=buf, seed=rank + 2000 + r)
    ev1.record()
    torch.cuda.synchronize(dev)
    roll_ms = ev0.elapsed_time(ev1) / reps
    prev_done = torch.zeros(N, dtype=torch.uint8, device=dev)
    ppo_update(net, opt, buf, prev_done, dist, epochs=1, minibatches=4)      # warm-up (cuBLAS handles, NCCL channels)
    timers = {}
    if dist:
        dist.barrier()
    torch.cuda.synchronize(dev)
    u0, u1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    u0.record()
    stats = ppo_update(net, opt, buf, prev_done, dist, epochs=1, minibatches=4, timers=timers)
    pol.set_weights(net)                                     # new parameters for the next rollout (bf16 repack)
    u1.record()
    torch.cuda.synchronize(dev)
    upd_ms = u0.elapsed_time(u1)
    ar_ms = sum(a.elapsed_time(b) for a, b in timers.get("allreduce", []))
    t = torch.tensor([roll_ms, upd_ms, ar_ms], dtype=torch.float64, device=dev)
    if dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    roll_ms, upd_ms, ar_ms = (float(x) for x in t)
    n_params = sum(p.numel() for p in net.parameters())
    env.close()
    return {
        "workload": desc, "policy": f"actor-critic MLP({D},256,256)+3 logits+value, fused tcgen05 kernel (bf16 x bf16 -> fp32), Gumbel-max sampling in-kernel",
        "horizon": H, "rollouts_timed": reps, "value": N * world * H / (roll_ms * 1e-3), "unit": "env-steps/s",
        "ms_per_step": roll_ms / H, "kernels_per_step": 2,
        "learner": {"update": "PPO, 1 epoch x 4 minibatches, torch autograd (tf32), Adam", "update_ms": upd_ms,
                    "allreduce_ms_per_update": ar_ms, "allreduce_share_of_update": ar_ms / upd_ms if upd_ms > 0 else None,
                    "allreduce_calls_per_update": len(timers.get("allreduce", [])),
                    "grad_bucket_bytes": n_params * 4, "advantage_stats_bytes": 24,
                    "collective": "NCCL all-reduce (flat gradient bucket per minibatch + [sum, sumsq, count] once)" if dist else "none (1 GPU)",
                    "train_value": N * world * H / ((roll_ms + upd_ms) * 1e-3), **stats},
    }


DUMP_BUDGET = 60 << 20   # array bytes of one --dump-outputs: the files, .npy headers included, stay under 64 MB


def dump_outputs(path, env, ring, rews, terms, last):
    """--dump-outputs: what the last timed step (index `last` of its fxenv_step_many batch) handed its caller -- every
    env's observation row, reward and terminated flag -- and the equity of every env after it, as <path>/<name>.npy
    (float32 / float64).  `env_index` holds the env ids of the rows; when the full arrays would exceed DUMP_BUDGET,
    the rows are a fixed seeded sample of the envs."""
    N = ring.shape[1]
    out = {"obs": ring[last % ring.shape[0]], "reward": rews[last], "terminated": terms[last].float(),
           "equity": env.info()["equity"]}
    per_env = sum(v[0].numel() * v.element_size() for v in out.values()) + 8   # + 8: env_index
    idx = np.arange(N)
    if per_env * N > DUMP_BUDGET:
        idx = np.sort(np.random.default_rng(0).choice(N, DUMP_BUDGET // per_env, replace=False))
    os.makedirs(path, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(path, name + ".npy"), v.cpu().numpy()[idx])
    np.save(os.path.join(path, "env_index.npy"), idx.astype(np.float64))


def run_ours(args, rank, world, local_rank):
    import torch
    from gym_fx_b200.sharding import check_pair_alignment, shard_starts
    from gym_fx_b200.vec_env import VecFxEnv

    assert torch.cuda.is_available(), "bench.py needs a CUDA device for --impl ours"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=dev)
    numa = pin_to_gpu_numa_node(local_rank)
    cfg, candles, minutes, N, D, algo_bytes, desc = build_workload(args.workload, args.envs)
    K, Wm = args.steps, max(3, args.warmup)
    env = VecFxEnv(cfg, candles, minutes, device=dev)
    # envs are sharded by rank: global env id = rank * N + i (SURVEY 8e: no collective in the data path)
    check_pair_alignment(N, cfg.num_pairs)
    pre = preroll_steps(cfg)
    chunk = min(K, 500)                      # steps per fxenv_step_many batch; K = full batches + one remainder batch
    starts = torch.as_tensor(shard_starts(N, rank, world, T_BARS, K + Wm + pre + 3 * chunk + 464, 256))
    env.reset(starts)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    acts = torch.randint(0, 3, (chunk, N), generator=gen, device=dev, dtype=torch.int32)
    slots = max(2, -(-int(L2_BYTES * 1.8) // (N * D * 4)))  # ring > 1.8x L2 so stores cannot just sit in L2
    ring = torch.empty((slots, N, D), dtype=torch.float32, device=dev)
    rews = torch.empty((chunk, N), dtype=torch.float32, device=dev)
    terms = torch.empty((chunk, N), dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev)

    # the argument sets are validated once; a launch is then a single C call (VecFxEnv.plan_step_many)
    full = env.plan_step_many(acts, ring, rews, terms)
    rem = K % chunk
    tail = env.plan_step_many(acts[:rem], ring, rews[:rem], terms[:rem]) if rem else None

    # episodes into steady state (preroll_steps), then the warm-up (also instantiates the graph)
    for _ in range(-(-pre // chunk)):
        full()
    wchunks = -(-Wm // chunk)
    for _ in range(max(1, wchunks)):
        full()
    if tail:                                 # the remainder batch has its own launch sequence: instantiate it now too
        tail()
    torch.cuda.synchronize(dev)

    sampler = ClockSampler(local_rank) if rank == 0 else None
    launches0 = env.launch_count()
    if dist:
        dist.barrier()
    torch.cuda.synchronize(dev)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    nfull = K // chunk
    # the device spins ~0.3 ms while the host enqueues the start event and the launches: the timed region starts with
    # the first launch already queued, as it is for every launch after the first in a training loop (host launch latency
    # is not device time of the K steps; without this a 20-step run carries ~10 us of it, more when 8 ranks share a host)
    torch.cuda._sleep(600_000)
    ev0.record(stream)
    for _ in range(nfull):
        full()
    if tail:
        tail()
    ev1.record(stream)
    torch.cuda.synchronize(dev)
    if dist:
        dist.barrier()
    ms = ev0.elapsed_time(ev1)
    launches = env.launch_count() - launches0
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    clocks = sampler.stop() if sampler else None
    engine = env.step_many_engine(chunk)
    overflow = int((env.info()["flags"] & 16).ne(0).sum().item())
    term_frac = float(terms.float().mean().item())
    if args.dump_outputs and rank == 0:      # before anything below reuses the buffers or steps the envs further
        dump_outputs(args.dump_outputs, env, ring, rews, terms, (rem or chunk) - 1)

    # ---- e2e: reference-facing host-buffer call, copies inside the timed region; median of 5 repeats of K steps
    Ke, reps = min(K, 400), 5
    h_act = torch.empty(N, dtype=torch.int32).pin_memory()
    h_acts_all = acts[:min(chunk, Ke)].cpu()
    h_obs = torch.empty((N, D), dtype=torch.float32).pin_memory()
    h_rew = torch.empty(N, dtype=torch.float32).pin_memory()
    h_term = torch.empty(N, dtype=torch.uint8).pin_memory()
    for k in range(3):
        h_act.copy_(h_acts_all[k % h_acts_all.shape[0]])
        env.step_host(h_act, h_obs, h_rew, h_term)
    e2e_times = []
    for _ in range(reps):
        if dist:
            dist.barrier()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for k in range(Ke):
            h_act.copy_(h_acts_all[k % h_acts_all.shape[0]])
            env.step_host(h_act, h_obs, h_rew, h_term)   # synchronous: returns when the results are in host memory
        e2e_times.append(time.perf_counter() - t0)
    te = torch.tensor(e2e_times, dtype=torch.float64, device=dev)
    if dist:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)      # per repeat: the slowest rank
    e2e_s = float(te.median().item())
    e2e_rate = N * world * Ke / e2e_s

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        per_launch_s = ms_max * 1e-3 / K
        achieved = N * algo_bytes / per_launch_s / 1e9
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
                per_step = json.load(fh).get(args.workload + "_per_step")
                traffic = per_step * K / max(1, int(launches)) if per_step and args.envs is None else None
        except Exception:
            pass
        line = {
            "metric": "env-steps/sec", "value": N * world * K / (ms_max * 1e-3), "unit": "env-steps/s",
            "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": ms_max / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": common_config(desc, N, D, world, pre),
            "details": {"actions": "torch.Generator(seed=1234+rank), pre-generated on device",
                        "l2": f"obs rows rotate through a {slots}-slot ring ({slots * N * D * 4 / 2**20:.0f} MiB > 126 MiB L2)",
                        "engine": (f"persistent launch: {chunk} steps per launch, warps pull (round of steps, env) tickets, per-env dependencies"
                                   if engine == "persistent" else f"CUDA graph of {chunk} single-step launches (programmatic dependent launch)"),
                        "order_overflow_envs": overflow, "terminated_frac": term_frac, "numa": numa},
            "clocks": clocks,
            "e2e": {"value": e2e_rate, "unit": "env-steps/s", "h2d_bytes_per_step": N * 4,
                    "d2h_bytes_per_step": N * (D * 4 + 4 + 1), "steps": Ke, "repeats": reps,
                    "note": "fxenv_step_host: pinned host buffers, synchronous per step (PCIe-bound); median of the "
                            "repeats, each the slowest rank"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "frac_of_nominal_8TBs": achieved / 8000.0,
                         "traffic": traffic, "peak_source": peak_src,
                         "kernel": "fx_rollout_kernel" if engine == "persistent" else "fx_step_kernel",
                         "algorithmic_bytes_per_launch": N * algo_bytes * K / max(1, int(launches)),
                         "avg_launch_us": ms_max * 1e3 / max(1, int(launches)),
                         "note": "achieved = algorithmic bytes of the timed region / its CUDA-event duration (the "
                                 "region is back-to-back launches of this one kernel); traffic = ncu dram bytes per env-step x envs"},
        }
        if world == 1 and engine == "persistent" and not args.no_single_step:
            line["single_step_graph"] = single_step_graph_rate(args, cfg, candles, minutes, N, starts, acts, ring, rews, terms, chunk)
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            sample_envs = min(N, 4096)
            rate, done, dt, used, _, _ = cpu_port_rate(args.workload, sample_envs, 100000, 3, threads, budget_s=8.0)
            line["cpu_baseline"] = {"value": rate, "unit": "env-steps/s", "cores": used, "kind": "port",
                                    "sample": f"{sample_envs} envs x {done} steps ({dt:.1f} s), C oracle port, {used} host threads, "
                                              f"no per-step barrier"}
    env.close()
    del ring
    torch.cuda.empty_cache()
    extra = {}
    if not args.no_closed_loop:
        try:
            extra["closed_loop"] = closed_loop_block(K, rank, world, dev, dist)
        except Exception as exc:   # the headline line must survive a failure of an auxiliary block -- but say so
            extra["closed_loop"] = {"error": f"{type(exc).__name__}: {exc}"}
    if rank == 0:
        if world == 1 and not args.no_other_workloads:
            extra["other_workloads"] = {}
            for name in ("cfg3", "cfg5"):
                try:
                    extra["other_workloads"][name] = short_workload_rate(name, max(3, min(K, 100)), dev)
                except Exception as exc:
                    extra["other_workloads"][name] = {"error": f"{type(exc).__name__}: {exc}"}
        line.update(extra)
        emit_json(line)
    if dist:
        dist.barrier()
        dist.destroy_process_group()


_REAL_STDOUT = None


def quiet_stdout():
    """Library chatter (e.g. NCCL's version banner) must not land on stdout: the contract is ONE JSON line there."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit_json(line):
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(line), flush=True)
    if _REAL_STDOUT is not None:
        os.dup2(2, 1)


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--envs", type=int, default=None, help="envs per GPU (default: the workload's)")
    ap.add_argument("--no-single-step", action="store_true", help="skip the single-step-graph reference measurement")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-closed-loop", action="store_true", help="skip the policy-in-the-loop (cfg4) block")
    ap.add_argument("--no-other-workloads", action="store_true", help="skip the short cfg3 / cfg5 runs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (--impl ours)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
        run_reference(args, rank, world)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit(f"--gpus {args.gpus} needs torchrun (python -m torch.distributed.run --nproc-per-node {args.gpus} ...)")
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
