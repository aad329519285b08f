#!/usr/bin/env python
"""bench.py -- env-steps/s INCLUDING Q-updates (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    (N > 1: one process per GPU, as  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...)

Workload (BASELINE.json configs[4], one GPU's shard; named in config.workload): independent agent
populations (seed x platform-speed x learning-rate sweep), x axis, curriculum step 0, ~1M envs per GPU,
every population with its own Q-table pair; weak scaling over GPUs with NO data-path collective.

A bench "step" = ONE global step of every env on the GPU = one launch of train_kernel (select -> dynamics ->
discretise -> check -> reward -> alpha -> Q update -> auto-reset).  `value` = env-steps/s summed over all
ranks, timed with CUDA events on the launching stream, L2 flushed (untimed) between timed launches, max over
ranks.  `e2e` = the same metric through the C-ABI host-buffer entry point dqlb200_train_host (pinned host
env-state + tables + trainer state copied in, E2E_CHUNK global steps, everything copied back, every call).
`cpu_baseline` = the reference's single-env Python loop (oracle port) on one host core, bounded sample.
`--impl reference` = that loop on every host core.
`--dump-outputs DIR` = after the timed steps, what they left to the caller as DIR/<name>.npy (see dump_outputs); the inputs
are fixed by the arguments, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import pathlib
import subprocess
import sys
import threading
import time

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "env_steps_per_sec_incl_q_updates"
UNIT = "env-steps/s"
POPULATIONS_PER_GPU = 888          # 6 CTAs per SM x 148 SMs (shared-memory limit of train_kernel<4>: 35 KB per population)
ENVS_PER_POPULATION = 1280         # 10 full slots of 128 threads; 888 * 1280 = 1,136,640 envs per GPU  (BASELINE config 5: "1M envs per GPU")
THREADS_PER_BLOCK = 128
E2E_CHUNK = 64                     # global steps per host-buffer call (about one episode, the reference's save interval)
E2E_TABLE_LEVELS = 2               # curriculum step 0 with promotions off: levels 0 (live) and 1 (next) of the tables travel, checked by the library
ALGORITHMIC_BYTES_PER_ENV_STEP = 96   # SURVEY.md 8(d): 48 B env state read + 48 B written, one step per launch
RAMP_LAUNCHES = 356                # untimed clock ramp, 32 global steps each: 0.3 s on a B200 at 1,965 MHz, 1,000 W power limit
DUMP_ENVS = 65536                  # --dump-outputs: env states of this many envs, a fixed seeded sample
DUMP_MAX_BYTES = 64 << 20


SHARED_SYNC_EVERY = 16             # global steps between two shared-table all-reduces (N > 1 only)
CONFIG4_SYNC_EVERY = 16            # config 4 on N GPUs: global steps between two merges / exchanges of an axis' tables


def envs_per_gpu_shared(P: int, n_p: int) -> int:
    return P * n_p


def workload_config(n_gpus: int) -> dict:
    return {
        "workload": "BASELINE configs[4] per-GPU shard: independent populations (seed x platform-speed x learning-rate "
                    "sweep), x axis, curriculum step 0, training incl. Q-updates",
        "populations_per_gpu": POPULATIONS_PER_GPU, "envs_per_population": ENVS_PER_POPULATION,
        "envs_per_gpu": POPULATIONS_PER_GPU * ENVS_PER_POPULATION, "n_gpus": n_gpus,
        "global_steps_per_launch": 1, "e2e_global_steps_per_call": E2E_CHUNK,
        "threads_per_block": THREADS_PER_BLOCK, "parallelism": f"population-partitioned x{n_gpus}, no collective",
        "l2": "flushed (256 MiB write) between timed launches; env state 51 MB < L2",
        "rng": "Philox4x32-10, key = seed (5 seeds per sweep point), counter word 3 = global population id", "platform_speeds": [0.4, 0.8, 1.2, 1.6],
        "alpha_variants": [[0.02949, 0.51], [0.05, 0.6]],
    }


def dump_outputs(eng, out: pathlib.Path, np):
    """What the timed training steps leave to their caller, read back after the last one and written as out/<name>.npy:
    the Q-table pair and visit counts of every population (all curriculum levels), the trainer state of every population, and the
    env state of DUMP_ENVS envs drawn with a fixed seed (the whole env state is 54 MB of packed words; the sample keeps the dump
    small).  Everything is float32 (what the kernel holds as float32) or float64 (exact for the integers and the float64 sums)."""
    t = eng.tables.cpu().numpy().view(np.uint32)                    # [population][q_a, q_b, count][MAX_CELLS]
    arrays = {"q_a": t[:, 0].view(np.float32), "q_b": t[:, 1].view(np.float32), "count": t[:, 2].astype(np.float64)}
    ps = eng.population_state()
    for f in ps.dtype.names:
        arrays["population_" + f] = ps[f].astype(np.float64)
    # env layout [population][tile of 32 envs][vector A, B, C][env in tile][4 words]; fields as in env_unpack (csrc/env_state.cuh)
    w = eng.env_state.view(eng.P, eng.tiles_per_population, 3, 32, 4).cpu().numpy().view(np.uint32)
    pick = np.sort(np.random.default_rng(0).choice(eng.n_total, min(DUMP_ENVS, eng.n_total), replace=False))
    pop, env = pick // eng.n_p, pick % eng.n_p
    e = w[pop, env // 32, :, env % 32]                              # [n][A, B, C][4 words]
    arrays["env_index"] = pick.astype(np.float64)                   # population * envs_per_population + env
    arrays["env_body"] = e[:, 0, :3].view(np.float32)               # x_d, v_d, theta
    arrays["env_prev_rel"] = e[:, 1, 2:].view(np.float32)           # previous rel_p, rel_v (reward shaping)
    # platform phase, set-point index, packed word (state id, step count, curriculum check, flags, position bin), episode
    arrays["env_words"] = np.stack([e[:, 0, 3], e[:, 1, 0], e[:, 2, 0], e[:, 2, 1]], axis=1).astype(np.float64)
    arrays["env_cum_reward"] = np.ascontiguousarray(e[:, 2, 2:]).view(np.float64)[:, 0]
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte limit")
    out.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out / f"{name}.npy", np.ascontiguousarray(a))


# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md): NVML polled every 10 ms from a thread
    (the timed region of the headline is a few milliseconds; nvidia-smi -lms cannot sample that fast), nvidia-smi as the
    fallback.  stop() raises when not a single sample was taken: a bench line without clocks is not a measurement."""
    REASONS = (("hw_slowdown", "HwSlowdown"), ("hw_thermal_slowdown", "HwThermalSlowdown"), ("sw_thermal_slowdown", "SwThermalSlowdown"),
               ("sw_power_cap", "SwPowerCap"), ("hw_power_brake", "HwPowerBrakeSlowdown"))

    def __init__(self, gpu_index: int):
        self.idx, self.samples, self.max_mhz, self.reasons, self.power = gpu_index, [], None, set(), []
        self._stop = threading.Event()
        self._thread, self._nvml, self._h, self.source = None, None, None, None

    def _visible_index(self) -> int:
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[self.idx])
            except (ValueError, IndexError):
                pass
        return self.idx

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml, self._h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(self._visible_index())
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
            self.source = "nvml, 10 ms period"
            self._thread = threading.Thread(target=self._poll_nvml, daemon=True)
        except Exception:
            self._nvml, self.source = None, "nvidia-smi -lms 50"
            self._thread = threading.Thread(target=self._poll_smi, daemon=True)
        self._thread.start()

    def _poll_nvml(self):
        n = self._nvml
        get_reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self._stop.is_set():
            try:
                self.samples.append(float(n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM)))
                mask = int(get_reasons(self._h))
                for name, suffix in self.REASONS:
                    bit = getattr(n, "nvmlClocksEventReason" + suffix, None) or getattr(n, "nvmlClocksThrottleReason" + suffix, 0)
                    if mask & bit:
                        self.reasons.add(name)
                self.power.append(n.nvmlDeviceGetPowerUsage(self._h) / 1000.0)
            except Exception:
                pass
            self._stop.wait(0.010)

    def _poll_smi(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            proc = subprocess.Popen(["nvidia-smi", f"--id={self._visible_index()}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                    stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            return
        for line in proc.stdout:
            r = [c.strip() for c in line.split(",")]
            try:
                self.samples.append(float(r[0])); self.max_mhz = float(r[1]); self.power.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    self.reasons.add(name)
            if self._stop.is_set():
                break
        proc.terminate()

    def stop(self) -> dict:
        self._stop.set()
        if self._thread is not None:
            self._thread.join(timeout=2.0)
        if not self.samples:
            raise RuntimeError("clock sampler took no sample (NVML and nvidia-smi both unavailable?): the bench line would carry no clocks")
        sm = sorted(self.samples)
        return {"sm_mhz": sm[len(sm) // 2], "sm_mhz_min": sm[0], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(sm), "power_w_max": max(self.power) if self.power else None, "source": self.source,
                "window": "from before the warm-up launches to the end of the e2e calls"}


def measured_peak_hbm():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def cpu_baseline(seconds: float = 12.0) -> dict:
    from oracle.cpu_loop import run_single_env
    steps, t = 0, 0.0
    while t < seconds:                       # bounded sample of the same workload: curriculum step 0, one env
        n, _, s = run_single_env(50000, seed=42 + steps)
        steps += n
        t += s
    c_port = None
    try:          # the same loop restated in plain C (oracle/c/loop.c): what an optimised CPU implementation would reach per core
        from oracle.c_loop import run_single_env_c
        n_c, _, s_c = run_single_env_c(4_000_000)
        c_port = {"value": n_c / s_c, "unit": UNIT, "cores": 1, "sample": f"{n_c} env-steps in {s_c:.2f} s",
                  "what": "oracle/c/loop.c: the single-env trainer loop in plain C (float32 tables, Philox contract, fp32 stand-in), "
                          "bit-identical to the reference fixtures (tests/test_oracle_c.py)"}
    except Exception as exc:
        c_port = {"error": str(exc)}
    flat = {}
    if c_port and "value" in c_port:      # scalar copies at the top level of cpu_baseline (a parser that keeps only scalars keeps them)
        flat = {"c_port_value": c_port["value"], "c_port_cores": c_port["cores"], "c_port_sample": c_port["sample"]}
    return {"value": steps / t, "unit": UNIT, "cores": 1, "kind": "port", **flat, "c_port": c_port,
            "sample": f"{steps} env-steps of the single-env reference loop (oracle port, float64 tables, analytic stand-in), "
                      f"{t:.1f} s on 1 of {os.cpu_count()} host cores",
            "context": "the unmodified reference loop measures 6.9-7.5e3 env-steps/s per core on the same stand-in (BASELINE.md section 2); "
                       "the reference's own Gazebo-locked training ran at 20.3 env-steps/s"}


# ----------------------------------------------------------------------------------------------------
def run_reference(args, rank: int, world: int):
    """The reference's own CPU implementation of the path (oracle port: /root/reference is Python and cannot
    travel to the GPU box) on every host core; rank 0 only."""
    if rank != 0:
        return
    import multiprocessing as mp
    from oracle.cpu_loop import run_all_cores
    cores = os.cpu_count() or 1
    steps_per_proc = 4000                     # one bench step = cores x 4000 env-steps (bounded sample)
    pool = mp.get_context("fork").Pool(cores)
    try:
        for w in range(args.warmup):
            run_all_cores(steps_per_proc, cores, seed0=1000 * w, pool=pool)
        total, wall = 0, 0.0
        for k in range(args.steps):
            n, s = run_all_cores(steps_per_proc, cores, seed0=7919 * (k + 1), pool=pool)
            total += n
            wall += s
    finally:
        pool.close()
        pool.join()
    v = total / wall
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(args.gpus),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{args.steps} steps x {cores} processes x {steps_per_proc} env-steps of the single-env reference loop"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------
def run_ours(args, rank: int, local_rank: int, world: int):
    import numpy as np
    import torch
    import torch.distributed as dist
    from dql_multirotor_landing_b200 import constants as K
    from dql_multirotor_landing_b200.engine import Engine, greedy_policy

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL prints its version banner on stdout when the communicator is created: send fd 1 to stderr meanwhile, so that
        # stdout carries the ONE JSON line and nothing else
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize(dev)
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    from dql_multirotor_landing_b200 import parallel
    numa_node = parallel.bind_to_gpu_numa_node(local_rank) if world > 1 else None     # pinned e2e buffers next to the GPU
    P, n_p = POPULATIONS_PER_GPU, ENVS_PER_POPULATION
    speeds = [0.4, 0.8, 1.2, 1.6]
    variants = [(0.02949, 0.51), (0.05, 0.6)]
    mine = parallel.partition_populations(P * world, world, rank)          # global population ids of this rank
    seeds, v_mp, alpha_index = parallel.sweep_axes(mine, 5, speeds, len(variants))
    eng = Engine(P, n_p, device=local_rank, threads_per_block=THREADS_PER_BLOCK, seeds=seeds, population_ids=list(mine),
                 v_mp=v_mp, alpha_variants=variants, alpha_index=alpha_index,
                 tp=K.TrainerParameters(max_num_episodes=10 ** 12, success_rate=2.0))   # stay in curriculum step 0 while timing
    eng.reset(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev)

    # clock ramp (untimed, not counted as warm-up steps): a fixed number of launches of the same kernel, so that the timed steps
    # start from the same state in every run with the same arguments
    for _ in range(0 if os.environ.get("DQL_BENCH_NO_RAMP") else RAMP_LAUNCHES):
        eng.train(32)
        torch.cuda.synchronize(dev)
    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(args.warmup):
        flush.zero_()
        eng.train(1)
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    launches = 0
    for k in range(args.steps):
        flush.zero_()                          # untimed L2 flush
        ev[k][0].record(stream)
        eng.train(1)
        ev[k][1].record(stream)
        launches += 1
    barrier()
    ms = sum(a.elapsed_time(b) for a, b in ev)
    eng.check_errors()
    if args.dump_outputs and rank == 0:
        dump_outputs(eng, pathlib.Path(args.dump_outputs), np)

    # ---- e2e: host buffers through dqlb200_train_host ----------------------------------------------
    env_h = torch.empty_like(eng.env_state, device="cpu").pin_memory()
    tab_h = torch.empty_like(eng.tables, device="cpu").pin_memory()
    ps_h = torch.empty_like(eng.pop_state, device="cpu").pin_memory()
    env_h.copy_(eng.env_state); tab_h.copy_(eng.tables); ps_h.copy_(eng.pop_state)
    torch.cuda.synchronize(dev)
    e2e_calls = max(3, min(args.steps, 20))
    for _ in range(2):
        eng.train_host(E2E_CHUNK, env_h, tab_h, ps_h, table_levels=E2E_TABLE_LEVELS)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_calls):
        eng.train_host(E2E_CHUNK, env_h, tab_h, ps_h, table_levels=E2E_TABLE_LEVELS)          # synchronises inside
        launches += min(8, P)                                   # one train_kernel launch per pipelined chunk of populations
    barrier()
    e2e_s = time.perf_counter() - t0
    clocks = sampler.stop()
    # The ceiling of any host-buffer API on this box: the same pinned buffers copied in and out (one cudaMemcpyAsync per buffer and
    # direction, both directions at once on two streams), every rank at the same time -- what the host memory system and the PCIe
    # links give N ranks, without a single kernel.  e2e's own copy rate (h2d/d2h_gb_per_s_per_rank) is to be read against it.
    copy_ceiling = None
    try:
        s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        env_d2 = torch.empty_like(eng.env_state)
        reps_c = 6
        def copies(h2d_on, d2h_on):
            barrier()
            t0c = time.perf_counter()
            for _ in range(reps_c):
                if h2d_on:
                    with torch.cuda.stream(s_in):
                        env_d2.copy_(env_h, non_blocking=True)
                if d2h_on:
                    with torch.cuda.stream(s_out):
                        env_h.copy_(eng.env_state, non_blocking=True)
            barrier()
            return time.perf_counter() - t0c
        copies(True, True)
        nbytes = env_h.numel() * env_h.element_size()
        t_in, t_out, t_both = copies(True, False), copies(False, True), copies(True, True)
        tc = torch.tensor([t_in, t_out, t_both], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tc, op=dist.ReduceOp.MAX)
        copy_ceiling = {"bytes_per_copy": nbytes, "h2d_alone_gb_per_s_per_rank": nbytes * reps_c / float(tc[0]) / 1e9,
                        "d2h_alone_gb_per_s_per_rank": nbytes * reps_c / float(tc[1]) / 1e9,
                        "both_directions_gb_per_s_per_rank_and_direction": nbytes * reps_c / float(tc[2]) / 1e9,
                        "ranks_copying_at_once": world, "timing": "host wall clock between barriers, max over ranks"}
        del env_d2
    except Exception as exc:
        copy_ceiling = {"error": str(exc)}
    # bytes that cross PCIe per call and direction: env state + E2E_TABLE_LEVELS of 5 table levels (+ the last level on the way in,
    # which quirk Q7 reads at the end of step 0) + trainer state
    tab_level = tab_h.numel() * 4 // K.MAX_CURRICULUM
    d2h = env_h.numel() * 4 + E2E_TABLE_LEVELS * tab_level + ps_h.numel()
    h2d = d2h + tab_level
    steps_done = int(np.frombuffer(ps_h.numpy().tobytes(), dtype=K.POPULATION_STATE_DTYPE)["total_steps"].sum())

    t_ms = torch.tensor([ms, e2e_s * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_max, e2e_ms_max = float(t_ms[0]), float(t_ms[1])
    envs_gpu = P * n_p
    value = world * envs_gpu * args.steps / (ms_max * 1e-3)
    e2e_value = world * envs_gpu * E2E_CHUNK * e2e_calls / (e2e_ms_max * 1e-3)

    # ---- N > 1: shared-table mode (BASELINE config 5): ONE agent, ~1M envs per GPU, replicas merged on each GPU and then
    # across GPUs by one NCCL all-reduce of the packed Q-delta/count buffer every SHARED_SYNC_EVERY global steps ------------
    shared = None
    if world > 1 and not args.no_extra:
        from dql_multirotor_landing_b200.parallel import SharedTableSync
        es = Engine(P, n_p, device=local_rank, threads_per_block=THREADS_PER_BLOCK, seeds=[42] * P,
                    population_ids=[rank * P + p for p in range(P)], replicas_per_population=P,
                    tp=K.TrainerParameters(max_num_episodes=10 ** 12, success_rate=2.0))
        es.reset(0)
        sync = SharedTableSync(es, pooled_promotion=True)
        rounds = 8
        for _ in range(2):
            es.train(SHARED_SYNC_EVERY); sync.sync()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(rounds):
            es.train(SHARED_SYNC_EVERY)
            sync.sync()
            launches += 4
        b.record(stream)
        barrier()
        es.check_errors()
        t_sh = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
        dist.all_reduce(t_sh, op=dist.ReduceOp.MAX)
        agree = torch.stack([es.tables[0, 0].float().sum(), es.tables[0, 2].float().sum()]).double()
        lo, hi = agree.clone(), agree.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        shared = {"env_steps_per_s": world * envs_per_gpu_shared(P, n_p) * SHARED_SYNC_EVERY * rounds / (float(t_sh[0]) * 1e-3),
                  "sync_every_global_steps": SHARED_SYNC_EVERY, "envs_sharing_one_table_pair": world * P * n_p,
                  "allgather_bytes_per_rank_and_sync": int(sync.packed.numel() * 4), "replicas_per_gpu": P,
                  "tables_identical_on_all_ranks": bool(torch.equal(lo, hi)), "timing": "CUDA events, max over ranks"}
        es.close()

    config4 = None
    if world > 1 and not args.no_extra:
        try:
            config4 = config4_multi_gpu(rank, local_rank, world, dev, barrier, torch, dist, K)
        except Exception as exc:
            config4 = {"error": f"{type(exc).__name__}: {exc}"}

    line = None
    if rank == 0:
        peak, peak_src = measured_peak_hbm()
        launch_s = ms_max * 1e-3 / args.steps
        achieved = ALGORITHMIC_BYTES_PER_ENV_STEP * envs_gpu / launch_s / 1e9
        traffic, traffic_src = None, None
        prof = ROOT / "profiles" / "train_kernel_traffic.json"
        if prof.exists():      # DRAM bytes per launch cannot be measured outside a profiler: the committed ncu figure of the same launch shape
            try:
                tj = json.loads(prof.read_text())
                traffic, traffic_src = tj.get("dram_bytes_per_launch"), "static: " + str(tj.get("source", "profiles/train_kernel_traffic.json")) + " (ncu --set full of this launch shape, not measured in this run)"
            except Exception:
                traffic = None
        extra = {}
        if not args.no_extra:
            extra = extra_measurements(eng, dev, np, torch, greedy_policy)
        if shared is not None:
            extra["config5_shared_table_mode"] = shared
        if config4 is not None:
            extra["config4_x_and_y_agents_262144_envs_each_multi_gpu"] = config4
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(world),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "kernel": "dql::train_kernel<4, false, 3>  (4 warps per CTA, no trace, production instance for full slots)",
                         "algorithmic_bytes_per_launch": ALGORITHMIC_BYTES_PER_ENV_STEP * envs_gpu,
                         "note": "instruction-issue bound, not HBM bound: see DESIGN.md section 6 and profiles/"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "h2d_gb_per_s_per_rank": h2d * e2e_calls / e2e_s / 1e9, "d2h_gb_per_s_per_rank": d2h * e2e_calls / e2e_s / 1e9,
                    "global_steps_per_call": E2E_CHUNK, "calls": e2e_calls, "api": "dqlb200_train_host (pinned host buffers)",
                    "host_numa_node_rank0": numa_node, "host_numa_binding_note": parallel.last_bind_note,
                    "pinned_copy_ceiling": copy_ceiling,
                    "step": "one e2e step = one dqlb200_train_host call: env state + tables + trainer state copied in, 64 global steps, all copied back"},
            "gpu_launches": launches, "clocks": clocks, "total_env_steps_counted_on_device": steps_done,
            "cpu_baseline": cpu_baseline() if not args.no_cpu else None,
            "extra": extra,
        }
        # SURVEY 8d: "two candidate roofs; report both, the lower one binds": the measured unordered-atomic RMW roof next to HBM
        rmw = extra.get("table_rmw_roof") if isinstance(extra, dict) else None
        if isinstance(rmw, dict) and "visits_per_s" in rmw:
            per_gpu = value / world
            line["roofline_rmw"] = {"bound": "smem-atomics", "achieved": per_gpu, "peak": rmw["visits_per_s"], "unit": "table visits/s (1 visit = count + Q_a read-modify-write)",
                                    "frac": per_gpu / rmw["visits_per_s"], "peak_source": "measured in this run: dqlb200_bench_table_rmw on the recorded cell sequence of a traced run",
                                    "binding_roof": "hbm" if line["roofline"]["frac"] >= per_gpu / rmw["visits_per_s"] else "smem-atomics",
                                    "note": "headline launch shape (one global step per launch); the HBM roof is the lower (binding) one for independent populations"}
    eng.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if line is not None:
        print(json.dumps(line), flush=True)


def config4_multi_gpu(rank, local_rank, world, dev, barrier, torch, dist, K) -> dict:
    """BASELINE configs[3] on N >= 2 GPUs (training_x.sh / training_y.sh run concurrently): ranks [0, N/2) train the x agent, ranks
    [N/2, N) the y agent, 262,144 envs per agent.  N = 2: one axis per GPU, no collective.  N >= 4: an axis is shared by G = N/2
    ranks (262,144 / G envs each as replicas of 512 envs), kept identical by the shared-table exchange inside the axis' process
    group every CONFIG4_SYNC_EVERY global steps.  Device-timed (CUDA events), max over ranks."""
    from dql_multirotor_landing_b200.engine import Engine
    from dql_multirotor_landing_b200.parallel import SharedTableSync
    half = world // 2
    axis = "x" if rank < half else "y"
    g_rank = rank % half
    groups = [dist.new_group(ranks=list(range(0, half))), dist.new_group(ranks=list(range(half, world)))]      # created by every rank
    group = groups[0 if rank < half else 1]
    n_r, total_per_agent, M, rounds = 512, 262144, CONFIG4_SYNC_EVERY, 32          # 32 exchange rounds: a timed region of a few ms is at the mercy of one late rank
    R = total_per_agent // n_r // half                     # replicas of this rank
    e4 = Engine(R, n_r, device=local_rank, threads_per_block=128, seeds=[42] * R, population_ids=[g_rank * R + p for p in range(R)],
                replicas_per_population=R, axes=[axis] * R, tp=K.TrainerParameters(success_rate=2.0, max_num_episodes=10 ** 12))
    e4.reset(0)
    sync = SharedTableSync(e4, pooled_promotion=True, group=group) if half > 1 else None
    stream = torch.cuda.current_stream(dev)

    def interval():
        if sync is not None:          # M fused global steps on this rank's replicas, then local merge + exchange inside the axis group
            e4.train(M)
            sync.sync()
        else:                         # one GPU per axis: (train, replica merge) graphs, merged every M steps like the 1-GPU leg
            e4.train_merged(M, M)
    for _ in range(2):
        interval()
    barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(rounds):
        interval()
    b.record(stream)
    barrier()
    e4.check_errors()
    t = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    out = {"env_steps_per_s": 2 * total_per_agent * M * rounds / (float(t[0]) * 1e-3), "n_gpus": world,
           "split": (f"ranks 0..{half - 1}: x agent, ranks {half}..{world - 1}: y agent; " +
                     ("one axis per GPU, no collective" if half == 1 else
                      f"each axis shared by {half} ranks ({R} replicas x {n_r} envs per rank), shared-table exchange inside the axis group")),
           "envs_per_agent": total_per_agent, "replicas_per_rank": R, "envs_per_replica": n_r, "merge_every_steps": M,
           "timing": "CUDA events, max over ranks"}
    if sync is not None:
        agree = torch.stack([e4.tables[0, 0].float().sum(), e4.tables[0, 2].float().sum()]).double()
        lo, hi = agree.clone(), agree.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN, group=group); dist.all_reduce(hi, op=dist.ReduceOp.MAX, group=group)
        same = torch.tensor([1.0 if torch.equal(lo, hi) else 0.0], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        out["tables_identical_on_all_ranks_of_an_axis"] = bool(same.item() == 1.0)
    e4.close()
    return out


def config3_with_promotion(dev, np, torch, K, Engine, timed_events) -> dict:
    """BASELINE configs[2] as stated (SURVEY 8d item 3): ONE agent, 65,536 envs, promotion ENABLED, from scratch.
    (a) the reference thresholds (0.96 of the last 100 episodes, transfer as written) at merge_every 1 (the Trainer default) and 16:
        env-steps/s, wall time, and the success rate reached after a fixed budget of global steps -- speed and learning quality side
        by side (the reference algorithm plateaus below 0.96 on the analytic stand-in, DESIGN.md section 3, so this is time to plateau);
    (b) the curriculum walk with the threshold at 0.80 and transfer_mode "paper": wall time to every promotion."""
    from dql_multirotor_landing_b200.trainer import replica_shape
    envs = 65536
    out = {"envs": envs, "timing": "CUDA events around every chunk of global steps",
           "replica_shape": "Trainer default per merge interval (trainer.replica_shape): 128 replicas x 512 envs in 256-thread blocks when merging after every "
                            "step, 512 x 128 in 128-thread blocks when merging every 16 steps; the learning curve does not depend on the split"}

    def run(tp, merge_every, budget_steps, chunk):
        n_r = replica_shape(envs, merge_every)
        R = envs // n_r
        e = Engine(R, n_r, device=dev.index or 0, threads_per_block=256 if n_r >= 256 else 128, seeds=[42] * R, population_ids=list(range(R)), replicas_per_population=R, tp=tp)
        e.reset(0)
        e.train_merged(merge_every, merge_every); torch.cuda.synchronize(dev)       # graph instantiation outside the timed region
        wall, done, rows, prev = 0.0, 0, [], e.population_state()
        w_prev, promoted = 0, []
        while done < budget_steps:
            wall += timed_events(lambda: e.train_merged(chunk, merge_every))
            done += chunk
            ps = e.population_state()
            d_ep = int(ps["total_episodes"].sum() - prev["total_episodes"].sum())
            d_su = int(ps["total_successes"].sum() - prev["total_successes"].sum())
            w = int(ps[0]["working_step"])
            rows.append({"global_steps": done, "wall_s": wall, "working_step": w, "success_rate_in_chunk": d_su / max(d_ep, 1),
                         "window_success_rate": float(ps["window_sum"].sum()) / max(float(ps["window_count"].sum()), 1.0)})
            if w != w_prev or int(ps[0]["finished"]):
                promoted.append({"to_working_step": w, "finished": int(ps[0]["finished"]), "global_steps": done, "wall_s": wall,
                                 "promoted_at_global_step": [int(x) for x in ps[0]["promoted_at"]]})
                w_prev = w
            prev = ps
            if int(ps[0]["finished"]):
                break
        e.check_errors()
        e.close()
        return {"merge_every": merge_every, "replicas": R, "envs_per_replica": n_r, "global_steps": done, "env_steps": envs * done, "wall_s": wall, "env_steps_per_s": envs * done / wall,
                "success_rate_last_chunk": rows[-1]["success_rate_in_chunk"], "window_success_rate_at_end": rows[-1]["window_success_rate"],
                "working_step_at_end": rows[-1]["working_step"], "promotions": promoted,
                "curve": [{k: (round(v, 4) if isinstance(v, float) else v) for k, v in r.items()} for r in rows[:: max(len(rows) // 8, 1)]]}

    ref_tp = K.TrainerParameters(max_num_episodes=50000 * envs)          # reference thresholds; the episode budget is per env (trainer.py)
    out["reference_thresholds"] = {f"merge_every_{M}": run(ref_tp, M, 131072, 8192) for M in (1, 16)}
    out["reference_thresholds"]["note"] = ("success_rate 0.96 / 100 episodes as in PKG/trainer.py:34-36: not reached on the analytic stand-in (plateau 0.80-0.87), "
                                           "so no promotion happens and the figures are time-to-plateau; merge_every 1 is the Trainer default")
    walk_tp = K.TrainerParameters(success_rate=0.8, transfer_mode="paper", max_num_episodes=50000 * envs)
    out["curriculum_walk_threshold_0.80_paper_transfer"] = run(walk_tp, 1, 196608, 8192)
    return out


def extra_measurements(eng, dev, np, torch, greedy_policy) -> dict:
    """Other BASELINE configs, device-timed, for context (not the headline)."""
    out = {}

    def timed(fn, reps=3):
        best = 1e30
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); torch.cuda.synchronize(dev)
            best = min(best, a.elapsed_time(b))
        return best * 1e-3

    eng.train(64); torch.cuda.synchronize(dev)
    s = timed(lambda: eng.train(64))
    out["fused_64_steps_per_launch_env_steps_per_s"] = eng.n_total * 64 / s
    # config 2: greedy evaluation of the committed policy, 1,048,576 episodes
    qa, qb = np.load(ROOT / "assets" / "Q_table_a.npy"), np.load(ROOT / "assets" / "Q_table_b.npy")
    pol = greedy_policy(qa, qb)
    n_ep = 1 << 20
    eng.eval_greedy(pol, 4096)
    t0 = time.perf_counter()
    res = eng.eval_greedy(pol, n_ep)
    s = time.perf_counter() - t0
    # config 2, both axes: the same policy on x, its mirror image on y, "eight" platform (PKG/moving_platform.py:92-111)
    try:
        from dql_multirotor_landing_b200 import constants as K2
        from dql_multirotor_landing_b200.engine import mirrored_policy
        ta = K2.TwoAxisParameters(trajectory=K2.TRAJ_EIGHT, r_x=3.0, v_x=0.8, r_y=3.0, y_action_enabled=True, y_init_enabled=True)
        eng.eval_greedy_2d(pol, mirrored_policy(pol), 4096, two_axis=ta)
        t0 = time.perf_counter()
        r2 = eng.eval_greedy_2d(pol, mirrored_policy(pol), n_ep, two_axis=ta)
        s2 = time.perf_counter() - t0
        out["config2_two_axis_eval_eight_trajectory"] = {"episodes": r2["episodes"], "env_steps": r2["steps"], "env_steps_per_s": r2["steps"] / s2,
                                                         "landing_rate": r2["termination_hist"][3] / max(r2["episodes"], 1),
                                                         "termination_hist": r2["termination_hist"], "timing": "host wall clock incl. launch+sync"}
    except Exception as exc:
        out["config2_two_axis_eval_eight_trajectory"] = {"error": str(exc)}
    # config 3: ONE agent, 65,536 envs sharing one Q-table pair (replica-merge mode: 512 replicas x 128 envs, merged every 16 steps)
    try:
        from dql_multirotor_landing_b200 import constants as K
        from dql_multirotor_landing_b200.engine import Engine
        from dql_multirotor_landing_b200.trainer import replica_shape
        steps = 256
        res3 = {"timing": "CUDA events, best of 3; (train launch, replica merge) pairs replayed as one CUDA graph"}

        def agent3(M):          # the Trainer's replica split for this merge interval (trainer.replica_shape)
            n_r = replica_shape(65536, M)
            R = 65536 // n_r
            e = Engine(R, n_r, device=dev.index or 0, threads_per_block=256 if n_r >= 256 else 128, seeds=[42] * R, population_ids=list(range(R)),
                       replicas_per_population=R, tp=K.TrainerParameters(success_rate=2.0, max_num_episodes=10 ** 12))
            e.reset(0)
            return e, R, n_r

        for M in (1, 16):          # merge after every step (closest to one shared table) / every 16 steps (throughput)
            e3, R, n_r = agent3(M)
            e3.train_merged(2 * M, M); torch.cuda.synchronize(dev)
            s3 = timed(lambda: e3.train_merged(steps, M))
            res3[f"env_steps_per_s_merge_every_{M}"] = R * n_r * steps / s3
            res3[f"replicas_x_envs_merge_every_{M}"] = [R, n_r]
            if M == 1:
                e3.close()
        # the config's own figure is the one at the Trainer default (merge after EVERY step: the setting that learns, see
        # config3_promotion_enabled); every 16 steps is the throughput end of the trade-off
        res3["env_steps_per_s"] = res3["env_steps_per_s_merge_every_1"]
        res3["merge_every_of_env_steps_per_s"] = 1
        # per curriculum step (SURVEY 8d config 3): the same agent started at working step w from the committed tables
        # (more live levels to stage, snapshot and discretise; no exploration draws for w > 0), merged every 16 steps
        try:
            cnt = np.load(ROOT / "assets" / "state_action_count.npy")
            per_w = {}
            for w in range(5):
                e3.set_group_tables(0, qa, qb, cnt)
                e3.reset(w)
                e3.train_merged(32, 16); torch.cuda.synchronize(dev)
                per_w[str(w)] = R * n_r * steps / timed(lambda: e3.train_merged(steps, 16))
            res3["env_steps_per_s_by_working_step_merge_every_16"] = per_w
            res3["promotion"] = ("the reference algorithm plateaus at a success rate of 0.80-0.87 on the analytic stand-in at step 0, below "
                                 "the 0.96 threshold (DESIGN.md section 3); tools/train_demo.py walks the curriculum with the threshold at 0.8")
        except Exception as exc:
            res3["env_steps_per_s_by_working_step_merge_every_16"] = {"error": str(exc)}
        out["config3_one_agent_65536_envs"] = res3
        e3.close()
        try:
            def timed_events(fn):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); fn(); b.record(); torch.cuda.synchronize(dev)
                return a.elapsed_time(b) * 1e-3
            out["config3_promotion_enabled"] = config3_with_promotion(dev, np, torch, K, Engine, timed_events)
        except Exception as exc:
            out["config3_promotion_enabled"] = {"error": f"{type(exc).__name__}: {exc}"}
    except Exception as exc:      # never let a context measurement break the headline line
        out["config3_one_agent_65536_envs"] = {"error": str(exc)}
    # config 4: decoupled x- and y-axis agents trained concurrently, 262,144 envs each (2 agents x 512 replicas x 512 envs)
    try:
        R, n_r, M, steps = 512, 512, 16, 128
        e4 = Engine(2 * R, n_r, device=dev.index or 0, threads_per_block=128, seeds=[42] * (2 * R), population_ids=list(range(2 * R)),
                    replicas_per_population=R, axes=["x"] * R + ["y"] * R,
                    tp=K.TrainerParameters(success_rate=2.0, max_num_episodes=10 ** 12))
        e4.reset(0)
        e4.train_merged(2 * M, M); torch.cuda.synchronize(dev)
        s4 = timed(lambda: e4.train_merged(steps, M))
        out["config4_x_and_y_agents_262144_envs_each"] = {"env_steps_per_s": 2 * R * n_r * steps / s4, "replicas_per_agent": R,
                                                         "envs_per_replica": n_r, "merge_every_steps": M, "timing": "CUDA events, best of 3"}
        e4.close()
    except Exception as exc:
        out["config4_x_and_y_agents_262144_envs_each"] = {"error": str(exc)}
    # SURVEY 8d streaming case: env state far larger than L2 (888 x 5,120 envs = 218 MB), ONE global step per launch, launches
    # back to back without any flush (every launch has to stream the whole state from and to HBM)
    try:
        n_big = 5120
        eb = Engine(POPULATIONS_PER_GPU, n_big, device=dev.index or 0, threads_per_block=THREADS_PER_BLOCK, seeds=list(range(POPULATIONS_PER_GPU)),
                    tp=K.TrainerParameters(success_rate=2.0, max_num_episodes=10 ** 12))
        eb.reset(0)
        eb.train(64); torch.cuda.synchronize(dev)
        reps = 40
        def many():
            for _ in range(reps):
                eb.train(1)
        sb = timed(many)
        rate = eb.n_total * reps / sb
        peak, _src = measured_peak_hbm()
        out["streaming_case_state_larger_than_l2"] = {
            "envs_per_gpu": eb.n_total, "env_state_bytes": eb.n_total * 48, "global_steps_per_launch": 1, "launches_timed_back_to_back": reps,
            "env_steps_per_s": rate, "algorithmic_gb_per_s": rate * ALGORITHMIC_BYTES_PER_ENV_STEP / 1e9,
            "frac_of_measured_hbm_peak": rate * ALGORITHMIC_BYTES_PER_ENV_STEP / 1e9 / peak, "l2": "no flush needed: 218 MB of state per launch vs 126 MB of L2",
            "timing": "CUDA events around 40 launches, best of 3"}
        eb.close()
    except Exception as exc:
        out["streaming_case_state_larger_than_l2"] = {"error": str(exc)}
    # SURVEY 8d "atomic roof": the visited cells of a real run (traced), replayed with unordered shared-memory atomics
    try:
        et = Engine(64, 256, device=dev.index or 0, threads_per_block=128, seeds=list(range(64)),
                    tp=K.TrainerParameters(success_rate=2.0, max_num_episodes=10 ** 12))
        et.reset(0)
        et.train(2500)                                           # past the pure-exploration phase of the first episodes
        tr = et.train(64, trace=True)
        cells = (tr["state"].astype(np.int64) * 3 + tr["action"]).astype(np.uint16).reshape(-1)
        rmw = et.bench_table_rmw(cells)
        hot = np.bincount(cells, minlength=2835)
        out["table_rmw_roof"] = {"visits_per_s": rmw["visits_per_s"], "rmw_per_s": rmw["rmw_per_s"],
                                 "distinct_cells": int((hot > 0).sum()), "hottest_cell_share": float(hot.max() / hot.sum()),
                                 "what": "2 unordered shared-memory atomics (red.shared.add.f32 + .u32) per recorded visit, 888 CTAs x 128 "
                                         "threads, tables in shared memory; an upper bound for the table update alone, NOT deterministic"}
        et.close()
        # SURVEY 8d: the shared-table configurations against the measured RMW roof (one visit = count + Q_a update = 2 RMW):
        # frac = env-steps/s of the WHOLE step (dynamics, reward, select, ordered update) / visits/s of the unordered atomics alone
        roof = rmw["visits_per_s"]
        fr = {"fused_independent_populations": out["fused_64_steps_per_launch_env_steps_per_s"] / roof}
        for key in ("config3_one_agent_65536_envs", "config4_x_and_y_agents_262144_envs_each"):
            if isinstance(out.get(key), dict) and "env_steps_per_s" in out[key]:
                fr[key] = out[key]["env_steps_per_s"] / roof
        out["table_rmw_roof"]["frac_of_rmw_roof"] = fr
    except Exception as exc:
        out["table_rmw_roof"] = {"error": str(exc)}
    out["config2_greedy_eval"] = {"episodes": res["episodes"], "env_steps": res["steps"], "env_steps_per_s": res["steps"] / s,
                                  "landing_rate": res["termination_hist"][3] / max(res["episodes"], 1),
                                  "termination_hist": res["termination_hist"], "timing": "host wall clock incl. launch+sync"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extra", action="store_true", help="skip the other-config measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (rank 0's populations)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        # not under torchrun: relaunch as one process per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 2000), __file__,
               "--gpus", str(args.gpus), "--steps", str(args.steps), "--warmup", str(args.warmup)]
        cmd += ["--no-cpu"] if args.no_cpu else []
        cmd += ["--no-extra"] if args.no_extra else []
        cmd += ["--dump-outputs", os.path.abspath(args.dump_outputs)] if args.dump_outputs else []
        sys.exit(subprocess.call(cmd))
    run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
