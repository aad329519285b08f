"""Greedy evaluation of many agents (development aid, not the bench): 888 populations x 1,280 envs, the committed assets/ tables
loaded into every population, seeds and population ids varied, working step 4 (the tables' last level).  One call measures:

  a  one Engine.eval_agents(1024) launch: every agent's LUT built on the device from its tables, 909,312 episodes
  b  the per-agent host path: 888 x (get_tables -> greedy_policy -> eval_greedy(1024)), host clock around synchronised work
  c  eval_greedy of the same 909,312 episodes under one policy: the per-episode ceiling of (a)
  ab eval_greedy of 1,048,576 episodes with this build and with --baseline-lib (another build of the library, e.g. of an earlier
     commit, loaded through its bare C-ABI so that its ABI version may differ), alternating

(a), (c) and (ab) are CUDA-event times of the launch alone; the tables (30 MB) stay L2-resident.  The GPU's name and power limit
are read in the same call.
usage: python tools/perf_probe_eval.py [--baseline-lib build_variants/libdqlb200_parent.so] [--reps 9] [--out FILE]"""
import argparse
import ctypes as C
import json
import pathlib
import statistics
import subprocess
import sys
import time

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import numpy as np
import torch
from dql_multirotor_landing_b200 import _ffi
from dql_multirotor_landing_b200 import constants as K
from dql_multirotor_landing_b200.engine import Engine, greedy_policy

P, N_P, E, W = 888, 1280, 1024, 4
N_STATES = K.MAX_CURRICULUM * K.STATES_PER_LEVEL


def gpu_info():
    info = dict(name=torch.cuda.get_device_name(0))
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in out.split(",")]
    except Exception as e:          # reported, never guessed
        info["power_limit"] = f"not read: {e}"
    return info


def events_ms(fn, reps):
    """CUDA-event time of fn() (one launch) after one warm-up: (min, median) in ms."""
    fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return min(times), statistics.median(times)


def stats_of(buf, n):
    st = buf.cpu().numpy().view(np.uint64).reshape(n, 11)
    return int(st[:, 0].sum()), int(st[:, 1].sum()), int(st[:, 4].sum() + st[:, 5].sum())      # episodes, steps, successes (codes 2, 3)


class RawEval:
    """dqlb200_eval_greedy of one library build through its bare C-ABI (a one-population handle, nothing bound)."""

    def __init__(self, path, policy):
        self.lib = lib = C.CDLL(str(path))
        vp = C.c_void_p
        lib.dqlb200_create.argtypes = [C.POINTER(K.Config), C.POINTER(C.c_float), C.POINTER(K.PopulationParams), C.c_int, C.POINTER(vp)]
        lib.dqlb200_destroy.argtypes = [vp]
        lib.dqlb200_eval_greedy.argtypes = [vp, C.c_int, vp, C.c_int64, C.c_int64, C.c_int, vp, vp, C.c_int, vp]
        lib.dqlb200_config_bytes.restype = C.c_size_t
        if lib.dqlb200_config_bytes() != C.sizeof(K.Config):
            raise RuntimeError(f"{path}: dqlb200_config layout differs from this tree's")
        cfg = K.build_config(1, 32, 32)
        cfg.abi_version = lib.dqlb200_abi_version()
        dp = K.DynamicsParameters()
        dphase, r, rw, rw2 = K.platform_constants(dp.r_mp, dp.v_mp, K.MdpParameters().f_ag, dp.n_sub)
        pps = (K.PopulationParams * 1)(K.PopulationParams(42, 0, 0, dphase, r, rw, rw2, 0, np.float32(dp.g), 0))
        lut = K.alpha_lut().astype(np.float32)
        self.h = vp()
        if lib.dqlb200_create(C.byref(cfg), lut.ctypes.data_as(C.POINTER(C.c_float)), pps, 0, C.byref(self.h)):
            raise RuntimeError(f"{path}: dqlb200_create failed")
        self.pol = torch.as_tensor(np.asarray(policy, np.uint8), device="cuda")
        self.stats = torch.zeros(C.sizeof(K.EvalStats), dtype=torch.uint8, device="cuda")

    def __call__(self, n):
        if self.lib.dqlb200_eval_greedy(self.h, 0, self.pol.data_ptr(), 0, n, W, self.stats.data_ptr(), None, 0,
                                        torch.cuda.current_stream().cuda_stream):
            raise RuntimeError("dqlb200_eval_greedy failed")

    def close(self):
        self.lib.dqlb200_destroy(self.h)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline-lib", default=None, help="another build of libdqlb200.so for the eval_kernel A/B")
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("perf_probe_eval needs a CUDA device")
    res = dict(gpu=gpu_info(), shape=dict(populations=P, envs_per_population=N_P, episodes_per_agent=E, working_step=W))
    qa, qb, cnt = (np.load(ROOT / "assets" / f) for f in ("Q_table_a.npy", "Q_table_b.npy", "state_action_count.npy"))
    eng = Engine(P, N_P, threads_per_block=128, seeds=[1000 + p for p in range(P)], population_ids=list(range(P)))
    for p in range(P):
        eng.set_tables(p, qa, qb, cnt)
    eng.reset(0)
    stream = lambda: eng._stream()
    total = P * E

    # (a) one eval_agents launch
    buf_a = torch.zeros(P * C.sizeof(K.EvalStats), dtype=torch.uint8, device=eng.device)
    run_a = lambda: _ffi.check(eng.lib.dqlb200_eval_agents(eng.handle, W, 0, E, buf_a.data_ptr(), None, stream()))
    t_min, t_med = events_ms(run_a, a.reps)
    buf_a.zero_(); run_a()
    eps, steps, successes = stats_of(buf_a, P)
    assert eps == total
    t0 = time.perf_counter()
    ev = eng.eval_agents(E, working_step=W)
    wall = time.perf_counter() - t0
    res["a_eval_agents"] = dict(ms_min=round(t_min, 3), ms_med=round(t_med, 3), env_steps=steps, env_steps_per_s=f"{steps / (t_med * 1e-3):.4e}",
                                episodes_per_s=f"{total / (t_med * 1e-3):.4e}", wall_ms_engine_call=round(wall * 1e3, 3),
                                success_rate=round(successes / eps, 4), success_rate_min_agent=round(float(ev["success_rate"].min()), 4))

    # (b) the per-agent host path of the parent API: tables to the host, float64 argmax, one eval_greedy per agent
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    steps_b, succ_b = 0, 0
    for p in range(P):
        tqa, tqb, _ = eng.get_tables(p)
        r = eng.eval_greedy(greedy_policy(tqa, tqb), E, population=p, working_step=W)
        steps_b += r["steps"]
        succ_b += r["termination_hist"][2] + r["termination_hist"][3]
    torch.cuda.synchronize()
    wall_b = time.perf_counter() - t0
    res["b_host_loop"] = dict(ms=round(wall_b * 1e3, 2), env_steps=steps_b, env_steps_per_s=f"{steps_b / wall_b:.4e}",
                              success_rate=round(succ_b / total, 4))

    # (c) the same number of episodes under one policy
    pol = np.zeros(N_STATES, np.uint8)
    pol[:] = greedy_policy(qa, qb)
    raw = RawEval(_ffi.LIB_PATH, pol)
    t_min_c, t_med_c = events_ms(lambda: raw(total), a.reps)
    raw.stats.zero_(); raw(total)
    _, steps_c, _ = stats_of(raw.stats, 1)
    res["c_eval_greedy_one_policy"] = dict(ms_min=round(t_min_c, 3), ms_med=round(t_med_c, 3), env_steps=steps_c,
                                           env_steps_per_s=f"{steps_c / (t_med_c * 1e-3):.4e}")
    res["a_over_c_env_steps_per_s"] = round((steps / t_med) / (steps_c / t_med_c), 4)
    res["a_speedup_over_b"] = round(wall_b / (t_med * 1e-3), 1)

    # (ab) eval_kernel of this build against another build, alternating
    if a.baseline_lib:
        n_ab = 1 << 20
        base = RawEval(a.baseline_lib, pol)
        runs = {"this": [], "baseline": []}
        for name, fn in (("this", raw), ("baseline", base)):
            fn(n_ab)                   # warm-up
        torch.cuda.synchronize()
        for _ in range(a.reps):
            for name, fn in (("this", raw), ("baseline", base)):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); fn(n_ab); e1.record()
                torch.cuda.synchronize()
                runs[name].append(e0.elapsed_time(e1))
        for fn in (raw, base):
            fn.stats.zero_(); fn(n_ab)
        same = bool(torch.equal(raw.stats, base.stats))
        res["ab_eval_greedy_1M"] = dict(baseline=str(a.baseline_lib), identical_stats=same,
                                        **{f"{k}_ms_min": round(min(v), 3) for k, v in runs.items()},
                                        **{f"{k}_ms_med": round(statistics.median(v), 3) for k, v in runs.items()})
        base.close()
    raw.close()
    eng.check_errors()
    eng.close()
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        pathlib.Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        pathlib.Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
