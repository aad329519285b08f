"""Greedy evaluation of many agents under a list of platform motions (development aid, not the bench): 888 agents holding the
committed assets/ tables, seeds and population ids varied, r_mp = 2 and v_mp in {0.4, 0.8, 1.2, 1.6}, 1,024 episodes per
(agent, platform), working step 4.  One call measures:

  a  one Engine.eval_platforms launch: 888 x 4 cells, 3,637,248 episodes
  b  the host path it replaces: one Engine per platform (same seeds, population ids, axes), every agent's float32 LUT taken from
     its tables on the host, one eval_greedy per (agent, platform); host clock around synchronised work, Engine set-up excluded
  c  one eval_agents launch of as many episodes (4,096 per agent under its own platform): the per-episode ceiling of (a)
  ab eval_agents of this build against --baseline-lib (another build of the library, e.g. of an earlier commit, bound through its
     bare C-ABI to the same device buffers), alternating

Every row of (a) must equal the matching row of (b), episode counts, env-steps and termination histograms.  (a), (c) and (ab)
are CUDA-event times of the launch alone; the tables (30 MB) stay L2-resident.  The GPU's name and power limit are read in the
same call.
usage: python tools/perf_probe_eval_platforms.py [--baseline-lib build_variants/libdqlb200_parent.so] [--reps 9] [--out FILE]"""
import argparse
import ctypes as C
import json
import pathlib
import statistics
import sys
import time

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import numpy as np
import torch
from dql_multirotor_landing_b200 import _ffi
from dql_multirotor_landing_b200 import constants as K
from dql_multirotor_landing_b200.engine import Engine
from perf_probe_eval import events_ms, gpu_info

P, N_P, E, W = 888, 32, 1024, 4
R_MP, SPEEDS = 2.0, (0.4, 0.8, 1.2, 1.6)
N_STATES = K.MAX_CURRICULUM * K.STATES_PER_LEVEL
SEEDS, PIDS = [1000 + p for p in range(P)], list(range(P))


def f32_lut(tables_u32):
    """Float32 first-max LUT of [3][MAX_CELLS] table words: (Q_a + Q_b) * 0.5f, rounded per operation (eval_agents' policy)."""
    n = K.MAX_CURRICULUM * K.CELLS_PER_LEVEL
    qa, qb = tables_u32[0, :n].view(np.float32).reshape(-1, 3), tables_u32[1, :n].view(np.float32).reshape(-1, 3)
    return np.argmax((qa + qb) * np.float32(0.5), axis=1).astype(np.uint8)


def stats_rows(buf, n):
    return buf.cpu().numpy().view(np.uint64).reshape(n, 11).astype(np.int64)


class RawAgents:
    """dqlb200_eval_agents of one library build through its bare C-ABI, bound to an Engine's device buffers (read only)."""

    def __init__(self, path, eng):
        self.lib = lib = C.CDLL(str(path))
        vp = C.c_void_p
        lib.dqlb200_create.argtypes = [C.POINTER(K.Config), C.POINTER(C.c_float), C.POINTER(K.PopulationParams), C.c_int, C.POINTER(vp)]
        lib.dqlb200_destroy.argtypes = [vp]
        lib.dqlb200_bind.argtypes = [vp, vp, vp, vp]
        lib.dqlb200_eval_agents.argtypes = [vp, C.c_int, C.c_int64, C.c_int64, vp, vp, vp]
        lib.dqlb200_config_bytes.restype = C.c_size_t
        if lib.dqlb200_config_bytes() != C.sizeof(K.Config):
            raise RuntimeError(f"{path}: dqlb200_config layout differs from this tree's")
        cfg = K.Config.from_buffer_copy(eng.cfg)
        cfg.abi_version = lib.dqlb200_abi_version()
        dphase, r, rw, rw2 = K.platform_constants(eng.dp.r_mp, eng.dp.v_mp, eng.mp.f_ag, eng.dp.n_sub)
        pps = (K.PopulationParams * P)(*[K.PopulationParams(SEEDS[p], 0, PIDS[p], dphase, r, rw, rw2, 0, np.float32(eng.dp.g), 0)
                                         for p in range(P)])
        lut = K.alpha_lut().astype(np.float32)
        self.h = vp()
        if lib.dqlb200_create(C.byref(cfg), lut.ctypes.data_as(C.POINTER(C.c_float)), pps, 0, C.byref(self.h)):
            raise RuntimeError(f"{path}: dqlb200_create failed")
        if lib.dqlb200_bind(self.h, eng.env_state.data_ptr(), eng.tables.data_ptr(), eng.pop_state.data_ptr()):
            raise RuntimeError(f"{path}: dqlb200_bind failed")
        self.stats = torch.zeros(P * C.sizeof(K.EvalStats), dtype=torch.uint8, device="cuda")

    def __call__(self, n):
        if self.lib.dqlb200_eval_agents(self.h, W, 0, n, self.stats.data_ptr(), None, torch.cuda.current_stream().cuda_stream):
            raise RuntimeError("dqlb200_eval_agents failed")

    def close(self):
        self.lib.dqlb200_destroy(self.h)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline-lib", default=None, help="another build of libdqlb200.so for the eval_agents A/B")
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("perf_probe_eval_platforms needs a CUDA device")
    platforms = [(R_MP, v) for v in SPEEDS]
    n_c = len(platforms)
    res = dict(gpu=gpu_info(), shape=dict(agents=P, platforms=platforms, episodes_per_cell=E, working_step=W))
    qa, qb, cnt = (np.load(ROOT / "assets" / f) for f in ("Q_table_a.npy", "Q_table_b.npy", "state_action_count.npy"))
    eng = Engine(P, N_P, threads_per_block=32, seeds=SEEDS, population_ids=PIDS)
    eng.set_tables(0, qa, qb, cnt)
    eng.tables[1:].copy_(eng.tables[0:1].expand(P - 1, -1, -1))
    eng.reset(0)
    total = P * n_c * E

    # (a) one eval_platforms launch
    host_pl = (K.Platform * n_c)(*[K.Platform(*K.platform_constants(r, v, eng.mp.f_ag, eng.dp.n_sub)) for r, v in platforms])
    buf_a = torch.zeros(P * n_c * C.sizeof(K.EvalStats), dtype=torch.uint8, device=eng.device)
    run_a = lambda: _ffi.check(eng.lib.dqlb200_eval_agents_platforms(eng.handle, W, 0, E, host_pl, n_c, buf_a.data_ptr(), eng._stream()))
    t_min, t_med = events_ms(run_a, a.reps)
    t0 = time.perf_counter()
    ev = eng.eval_platforms(E, platforms, working_step=W)
    wall = time.perf_counter() - t0
    steps = int(ev["steps"].sum())
    assert int(ev["episodes"].sum()) == total
    rate_by_platform = (ev["termination_hist"][:, :, 2] + ev["termination_hist"][:, :, 3]).sum(axis=0) / (P * E)
    res["a_eval_platforms"] = dict(ms_min=round(t_min, 3), ms_med=round(t_med, 3), env_steps=steps,
                                   env_steps_per_s=f"{steps / (t_med * 1e-3):.4e}", episodes_per_s=f"{total / (t_med * 1e-3):.4e}",
                                   wall_ms_engine_call=round(wall * 1e3, 3),
                                   success_rate_by_platform=[round(float(x), 4) for x in rate_by_platform])

    # (b) the host path: one Engine per platform, float32 LUT per agent from its tables, one eval_greedy per (agent, platform)
    t0 = time.perf_counter()
    per_platform = []
    for r, v in platforms:
        e = Engine(P, N_P, threads_per_block=32, seeds=SEEDS, population_ids=PIDS, r_mp=[r] * P, v_mp=[v] * P)
        e.tables.copy_(eng.tables)
        per_platform.append(e)
    torch.cuda.synchronize()
    setup_b = time.perf_counter() - t0
    t0 = time.perf_counter()
    rows_b = np.zeros((P, n_c, 11), np.int64)
    for g in range(P):
        lut = f32_lut(eng.tables[g].cpu().numpy().view(np.uint32))
        for c, e in enumerate(per_platform):
            rb = e.eval_greedy(lut, E, population=g, working_step=W)
            rows_b[g, c] = [rb["episodes"], rb["steps"], *rb["termination_hist"]]
    torch.cuda.synchronize()
    wall_b = time.perf_counter() - t0
    rows_a = np.concatenate([ev["episodes"][..., None], ev["steps"][..., None], ev["termination_hist"]], axis=2)
    mismatched = int((rows_a != rows_b).any(axis=2).sum())
    res["b_host_path"] = dict(ms=round(wall_b * 1e3, 2), setup_ms=round(setup_b * 1e3, 2), env_steps=int(rows_b[:, :, 1].sum()),
                              env_steps_per_s=f"{rows_b[:, :, 1].sum() / wall_b:.4e}")
    res["row_check"] = dict(rows=P * n_c, mismatched=mismatched, ok=mismatched == 0)
    for e in per_platform:
        e.close()

    # (c) eval_agents over as many episodes, each agent under its own platform
    e_c = E * n_c
    buf_c = torch.zeros(P * C.sizeof(K.EvalStats), dtype=torch.uint8, device=eng.device)
    run_c = lambda: _ffi.check(eng.lib.dqlb200_eval_agents(eng.handle, W, 0, e_c, buf_c.data_ptr(), None, eng._stream()))
    t_min_c, t_med_c = events_ms(run_c, a.reps)
    buf_c.zero_(); run_c()
    steps_c = int(stats_rows(buf_c, P)[:, 1].sum())
    res["c_eval_agents"] = dict(episodes_per_agent=e_c, ms_min=round(t_min_c, 3), ms_med=round(t_med_c, 3), env_steps=steps_c,
                                env_steps_per_s=f"{steps_c / (t_med_c * 1e-3):.4e}")
    res["a_over_c_env_steps_per_s"] = round((steps / t_med) / (steps_c / t_med_c), 4)
    res["a_speedup_over_b"] = round(wall_b / (t_med * 1e-3), 1)

    # (ab) eval_agents of this build against another build on the same bound buffers, alternating
    if a.baseline_lib:
        this, base = RawAgents(_ffi.LIB_PATH, eng), RawAgents(a.baseline_lib, eng)
        runs = {"this": [], "baseline": []}
        for fn in (this, base):
            fn(E)                      # warm-up
        torch.cuda.synchronize()
        for _ in range(a.reps):
            for name, fn in (("this", this), ("baseline", base)):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); fn(E); e1.record()
                torch.cuda.synchronize()
                runs[name].append(e0.elapsed_time(e1))
        for fn in (this, base):
            fn.stats.zero_(); fn(E)
        res["ab_eval_agents"] = dict(baseline=str(a.baseline_lib), identical_stats=bool(torch.equal(this.stats, base.stats)),
                                     **{f"{k}_ms_min": round(min(v), 3) for k, v in runs.items()},
                                     **{f"{k}_ms_med": round(statistics.median(v), 3) for k, v in runs.items()},
                                     **{f"{k}_ms_all": [round(x, 3) for x in v] for k, v in runs.items()})
        this.close()
        base.close()
    eng.check_errors()
    eng.close()
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        pathlib.Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        pathlib.Path(a.out).write_text(line + "\n")
    if mismatched:
        raise SystemExit(f"row check failed: {mismatched} of {P * n_c} rows differ from the host path")


if __name__ == "__main__":
    main()
