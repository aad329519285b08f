"""Two-axis greedy evaluation of many x/y agent pairs (development aid, not the bench): 888 populations x 1,280 envs, 444 x agents
holding the committed assets/ tables and 444 y agents holding the same tables mirrored into the y frame (angle index reversed,
increase / decrease swapped, so that they land on y), seeds and population ids varied; pair k = (x agent k, y agent 444 + k), the
"eight" platform (r = 3, v = 0.8) with the y action and the y start offset on, working step 4.  One call measures:

  a  one Engine.eval_pairs launch over 444 pairs x 1,024 episodes = 454,656 episodes, both LUTs of every pair built on the device
  b  the per-pair host path: 444 x (get_tables -> greedy_policy of both members -> eval_greedy_2d(1024)), host clock around
     synchronised work (a y agent flies its own LUT, so no mirror is taken)
  c  eval_greedy_2d of the same 454,656 episodes under one LUT pair (the float32 LUTs of the x and the y tables): the per-episode
     ceiling of (a)
  ab eval_greedy_2d of 1,048,576 episodes with this build and with --baseline-lib (another build of the library, e.g. of an earlier
     commit, loaded through its bare C-ABI so that its ABI version may differ), alternating

Every row of (a) is checked against eval_greedy_2d(1,024) under the same LUTs, and (ab) compares the two builds' statistics.
(a), (c) and (ab) are CUDA-event times of the call alone ((a) includes the 3.5 KB upload of the pair list); the tables (30 MB)
stay L2-resident.  The GPU's name and power limit are read in the same call.
usage: python tools/perf_probe_eval2d.py [--baseline-lib build_variants/libdqlb200_parent.so] [--reps 9] [--out FILE]"""
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

H, N_P, E, W = 444, 1280, 1024, 4
P = 2 * H
N_STATES = K.MAX_CURRICULUM * K.STATES_PER_LEVEL
EIGHT = K.TwoAxisParameters(trajectory=K.TRAJ_EIGHT, r_x=3.0, v_x=0.8, r_y=3.0, y_action_enabled=True, y_init_enabled=True)


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


def y_frame(q):
    """A table of the x frame as a y agent holds it: q_y[.., theta, a] = q[.., 6 - theta, {1,0,2}[a]] (engine.mirrored_policy)."""
    return np.ascontiguousarray(q[..., ::-1, :][..., [1, 0, 2]])


def f32_lut(qa, qb):
    """The float32 first-max LUT the library builds: (Q_a + Q_b) * 0.5f per operation, first maximum."""
    avg = (qa.astype(np.float32) + qb.astype(np.float32)) * np.float32(0.5)
    lut = np.zeros(N_STATES, np.uint8)
    lut[: avg.size // 3] = np.argmax(avg.reshape(-1, 3), axis=1)
    return lut


class RawEval2D:
    """dqlb200_eval_greedy_2d of one library build through its bare C-ABI (a one-population handle, nothing bound)."""

    def __init__(self, path, lut_x, lut_y):
        self.lib = lib = C.CDLL(str(path))
        vp = C.c_void_p
        lib.dqlb200_create.argtypes = [C.POINTER(K.Config), C.POINTER(C.c_float), C.POINTER(K.PopulationParams), C.c_int, C.POINTER(vp)]
        lib.dqlb200_destroy.argtypes = [vp]
        lib.dqlb200_eval_greedy_2d.argtypes = [vp, C.POINTER(K.Eval2DParams), vp, vp, C.c_int64, C.c_int64, vp, vp, C.c_int, vp]
        lib.dqlb200_config_bytes.restype = C.c_size_t
        lib.dqlb200_eval2d_params_bytes.restype = C.c_size_t
        if lib.dqlb200_config_bytes() != C.sizeof(K.Config) or lib.dqlb200_eval2d_params_bytes() != C.sizeof(K.Eval2DParams):
            raise RuntimeError(f"{path}: dqlb200_config / dqlb200_eval2d_params layout differs from this tree's")
        cfg = K.build_config(1, 32, 32)
        cfg.abi_version = lib.dqlb200_abi_version()
        dp = K.DynamicsParameters()
        pps = (K.PopulationParams * 1)(K.PopulationParams(42, 0, 0, 0, 0.0, 0.0, 0.0, 0, np.float32(dp.g), 0))
        alpha = K.alpha_lut().astype(np.float32)
        self.h = vp()
        if lib.dqlb200_create(C.byref(cfg), alpha.ctypes.data_as(C.POINTER(C.c_float)), pps, 0, C.byref(self.h)):
            raise RuntimeError(f"{path}: dqlb200_create failed")
        self.prm = K.eval2d_params(EIGHT, dp, K.MdpParameters().f_ag, 42, 0, W)
        self.px = torch.as_tensor(lut_x, device="cuda")
        self.py = torch.as_tensor(lut_y, device="cuda")
        self.stats = torch.zeros(C.sizeof(K.EvalStats), dtype=torch.uint8, device="cuda")

    def __call__(self, n):
        if self.lib.dqlb200_eval_greedy_2d(self.h, C.byref(self.prm), self.px.data_ptr(), self.py.data_ptr(), 0, n, self.stats.data_ptr(),
                                           None, 0, torch.cuda.current_stream().cuda_stream):
            raise RuntimeError("dqlb200_eval_greedy_2d failed")

    def close(self):
        self.lib.dqlb200_destroy(self.h)


def stats_of(buf, n):
    st = buf.cpu().numpy().view(np.uint64).reshape(n, 11)
    return int(st[:, 0].sum()), int(st[:, 1].sum()), int(st[:, 4].sum() + st[:, 5].sum()), st      # episodes, steps, successes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline-lib", default=None, help="another build of libdqlb200.so for the eval2d_kernel A/B")
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("perf_probe_eval2d needs a CUDA device")
    res = dict(gpu=gpu_info(), shape=dict(x_agents=H, y_agents=H, pairs=H, envs_per_population=N_P, episodes_per_pair=E,
                                          working_step=W, platform="eight, r 3, v 0.8, y action and y offset on"))
    qa, qb, cnt = (np.load(ROOT / "assets" / f) for f in ("Q_table_a.npy", "Q_table_b.npy", "state_action_count.npy"))
    eng = Engine(P, N_P, threads_per_block=128, seeds=[1000 + p for p in range(P)], population_ids=list(range(P)),
                 axes=["x"] * H + ["y"] * H)
    for p in range(H):
        eng.set_tables(p, qa, qb, cnt)
        eng.set_tables(H + p, y_frame(qa), y_frame(qb), y_frame(cnt))
    eng.reset(0)
    total = H * E
    pairs = np.asarray([(k, H + k) for k in range(H)], np.int32)

    # (a) one eval_pairs call
    prm = K.eval2d_params(EIGHT, eng.dp, eng.mp.f_ag, 42, 0, W)
    buf_a = torch.zeros(H * C.sizeof(K.EvalStats), dtype=torch.uint8, device=eng.device)
    run_a = lambda: _ffi.check(eng.lib.dqlb200_eval_pairs(eng.handle, C.byref(prm), pairs.ctypes.data, H, 0, E, buf_a.data_ptr(),
                                                          eng._stream()))
    t_min, t_med = events_ms(run_a, a.reps)
    buf_a.zero_(); run_a()
    eps, steps, successes, st = stats_of(buf_a, H)
    assert eps == total and (st == st[0]).all()          # identical LUTs, one key: identical rows
    t0 = time.perf_counter()
    ev = eng.eval_pairs(E, pairs, two_axis=EIGHT, working_step=W)
    wall = time.perf_counter() - t0
    res["a_eval_pairs"] = dict(ms_min=round(t_min, 3), ms_med=round(t_med, 3), env_steps=steps, env_steps_per_s=f"{steps / (t_med * 1e-3):.4e}",
                               episodes_per_s=f"{total / (t_med * 1e-3):.4e}", wall_ms_engine_call=round(wall * 1e3, 3),
                               success_rate=round(successes / eps, 4), success_rate_min_pair=round(float(ev["success_rate"].min()), 4))

    # (b) the per-pair host path of the parent API: both members' tables to the host, float64 argmax, one eval_greedy_2d per pair
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    steps_b, succ_b = 0, 0
    for gx, gy in pairs:
        pol_x = greedy_policy(*eng.get_tables(int(gx))[:2])
        pol_y = greedy_policy(*eng.get_tables(int(gy))[:2])      # a y agent: its own LUT (an x agent would take mirrored_policy)
        r = eng.eval_greedy_2d(pol_x, pol_y, E, two_axis=EIGHT, working_step=W)
        steps_b += r["steps"]
        succ_b += r["termination_hist"][2] + r["termination_hist"][3]
    torch.cuda.synchronize()
    wall_b = time.perf_counter() - t0
    res["b_host_loop"] = dict(ms=round(wall_b * 1e3, 2), env_steps=steps_b, env_steps_per_s=f"{steps_b / wall_b:.4e}",
                              success_rate=round(succ_b / total, 4))

    # (c) the same number of episodes under one LUT pair
    lut_x, lut_y = f32_lut(qa, qb), f32_lut(y_frame(qa), y_frame(qb))
    raw = RawEval2D(_ffi.LIB_PATH, lut_x, lut_y)
    t_min_c, t_med_c = events_ms(lambda: raw(total), a.reps)
    raw.stats.zero_(); raw(total)
    _, steps_c, _, _ = stats_of(raw.stats, 1)
    # (a) flies episodes 0 .. E-1 once per pair, (c) episodes 0 .. total-1: every row of (a) must equal eval_greedy_2d(E)
    raw.stats.zero_(); raw(E)
    assert (stats_of(raw.stats, 1)[3][0] == st[0]).all(), "eval_pairs row differs from eval_greedy_2d under the same LUTs"
    res["a_rows_equal_eval_greedy_2d"] = True
    res["c_eval_greedy_2d_one_lut_pair"] = dict(ms_min=round(t_min_c, 3), ms_med=round(t_med_c, 3), env_steps=steps_c,
                                                env_steps_per_s=f"{steps_c / (t_med_c * 1e-3):.4e}")
    res["a_over_c_env_steps_per_s"] = round((steps / t_med) / (steps_c / t_med_c), 4)
    res["a_speedup_over_b"] = round(wall_b / (t_med * 1e-3), 1)

    # (ab) eval2d_kernel of this build against another build, alternating
    if a.baseline_lib:
        n_ab = 1 << 20
        base = RawEval2D(a.baseline_lib, lut_x, lut_y)
        runs = {"this": [], "baseline": []}
        for fn in (raw, base):
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
        res["ab_eval_greedy_2d_1M"] = dict(baseline=str(a.baseline_lib), identical_stats=same, env_steps=stats_of(raw.stats, 1)[1],
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
