"""TEST/BENCH INFRASTRUCTURE ONLY -- never imported by the product package.

ctypes driver of oracle/c/loop.c: the reference trainer loop for one environment in plain C (float32 tables, the Philox draw
contract, the deterministic stand-in).  tests/test_oracle_c.py holds it identical to the fixtures of the unmodified reference;
bench.py times it as a second, much stricter CPU baseline next to the Python port."""
from __future__ import annotations

import ctypes as C
import pathlib
import subprocess
import time

import numpy as np

from .dynamics import StandInDet, StandInParams, derive

CDIR = pathlib.Path(__file__).resolve().parent / "c"


class Params(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("h", "half_h2", "k_theta", "g", "c_d", "r", "rw", "rw2")] + [
        ("dphase", C.c_uint32), ("n_sub", C.c_int32), ("accel_mode", C.c_int32), ("kf_q", C.c_float), ("kf_r", C.c_float),
        ("second_order", C.c_int32), ("pid_ticks", C.c_int32)] + [(n, C.c_float) for n in (
            "att_kr", "att_kw", "inv_m", "inv_mg", "g_abs", "pid_kp", "pid_ki", "pid_lo", "pid_hi", "pid_windup", "pid_dt",
            "bw_inv_denom", "bw_k2", "z_init")]


class LoopParams(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("dz", "z_touch", "half_platform", "p_max_f", "two_p_max_f", "sigma_x")] + [
        (n, C.c_double) for n in ("f_ag", "t_max", "p_max", "alpha_min", "omega", "gamma")]


def load() -> C.CDLL:
    so = CDIR / "libstandin_oracle.so"
    if not so.exists():
        subprocess.run(["make", "-C", str(CDIR)], check=True, capture_output=True)
    lib = C.CDLL(str(so))
    lib.mdp_sizeof.restype = C.c_size_t
    lib.oracle_single_env_loop.argtypes = [C.c_void_p] * 3 + [C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 11
    return lib


def run_single_env_c(n_steps: int, seed: int = 42, w: int = 0):
    """n_steps env-steps incl. Q-updates of one env at curriculum step w; returns (steps, episodes, seconds)."""
    lib = load()
    sp = StandInParams()
    d = derive(sp)
    p = Params(h=d.h, half_h2=d.half_h2, k_theta=d.k_theta, g=d.g, c_d=d.c_d, r=d.r, rw=d.rw, rw2=d.rw2, dphase=d.dphase, n_sub=d.n_sub,
               z_init=d.z_init)
    lp = LoopParams(dz=d.dz, z_touch=d.z_touch, half_platform=d.half_platform, p_max_f=d.p_max, two_p_max_f=d.two_p_max, sigma_x=d.sigma_x,
                    f_ag=sp.f_ag, t_max=20.0, p_max=sp.p_max, alpha_min=0.02949, omega=0.51, gamma=0.99)
    qa, qb, count = np.zeros(2835, np.float32), np.zeros(2835, np.float32), np.zeros(2835, np.float64)
    obs = np.zeros((n_steps, 5), np.float32)
    ints = [np.zeros(n_steps, np.int32) for _ in range(6)]
    reward = np.zeros(n_steps, np.float64)
    buf = C.create_string_buffer(lib.mdp_sizeof())
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    t0 = time.perf_counter()
    episodes = lib.oracle_single_env_loop(C.byref(p), C.byref(lp), C.cast(buf, C.c_void_p), seed, 0, w, 0, n_steps, ptr(qa), ptr(qb), ptr(count),
                                          ptr(obs), *[ptr(a) for a in ints[:5]], ptr(reward), ptr(ints[5]))
    return n_steps, int(episodes), time.perf_counter() - t0


class TrainerParamsC(C.Structure):
    _fields_ = [("curriculum_steps", C.c_int32), ("window_len", C.c_int32), ("transfer_mode", C.c_int32), ("success_rate", C.c_double),
                ("max_num_episodes", C.c_int64), ("transfer_ratio", C.c_float * 5)]


class PopulationResult(C.Structure):
    _fields_ = [("w", C.c_int32), ("finished", C.c_int32), ("window_count", C.c_int32), ("window_sum", C.c_int32), ("t", C.c_int64),
                ("episodes_done", C.c_int64), ("total_steps", C.c_int64), ("total_episodes", C.c_int64), ("total_successes", C.c_int64),
                ("term_hist", C.c_int64 * 9), ("n_promotions", C.c_int32)]


def run_population_c(n_envs: int, n_steps: int, seed: int = 42, population: int = 0, w0: int = 0, tp=None, sp: StandInParams = None,
                     qa0=None, qb0=None, trace: bool = False):
    """oracle/c/population.c: PopulationOracle (batched semantics S1, float32 tables) in C.  Returns dict(qa, qb, count, result[, traces])."""
    from .agent_oracle import transfer_ratio
    from .loop import TrainerParams
    lib = load()
    tp = tp or TrainerParams()
    sp = sp or StandInParams(f_ag=tp.f_ag, p_max=tp.p_max)
    d = derive(sp)
    p = Params(h=d.h, half_h2=d.half_h2, k_theta=d.k_theta, g=d.g, c_d=d.c_d, r=d.r, rw=d.rw, rw2=d.rw2, dphase=d.dphase, n_sub=d.n_sub,
               z_init=d.z_init, accel_mode={"exact": 0, "kalman_reference": 1, "kalman": 2}[sp.accel_mode],
               kf_q=np.float32(sp.kf_process_variance), kf_r=np.float32(sp.kf_measurement_sd ** 2),
               second_order=int(sp.dynamics_model == "second_order"))
    lp = LoopParams(dz=d.dz, z_touch=d.z_touch, half_platform=d.half_platform, p_max_f=d.p_max, two_p_max_f=d.two_p_max, sigma_x=d.sigma_x,
                    f_ag=tp.f_ag, t_max=tp.t_max, p_max=tp.p_max, alpha_min=tp.alpha_min, omega=tp.omega, gamma=tp.gamma)
    tpc = TrainerParamsC(tp.curriculum_steps, tp.successive_successful_episodes, {"reference": 0, "paper": 1}[tp.transfer_mode],
                         tp.success_rate, tp.max_num_episodes, (C.c_float * 5)(*[np.float32(transfer_ratio(k, tp.scale_modification_value)) for k in range(5)]))
    qa = np.zeros(2835, np.float32) if qa0 is None else np.ascontiguousarray(qa0, np.float32).reshape(-1).copy()
    qb = np.zeros(2835, np.float32) if qb0 is None else np.ascontiguousarray(qb0, np.float32).reshape(-1).copy()
    count = np.zeros(2835, np.float64)
    res = PopulationResult()
    ptr = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
    tr = dict(action=np.zeros((n_steps, n_envs), np.uint8), next_state=np.zeros((n_steps, n_envs), np.uint16),
              code=np.zeros((n_steps, n_envs), np.uint8), reward=np.zeros((n_steps, n_envs), np.float64)) if trace else {}
    lib.oracle_population_run.argtypes = [C.c_void_p] * 3 + [C.c_int, C.c_uint64, C.c_uint32, C.c_int, C.c_int] + [C.c_void_p] * 8
    rc = lib.oracle_population_run(C.byref(p), C.byref(lp), C.byref(tpc), n_envs, seed, population, w0, n_steps, ptr(qa), ptr(qb), ptr(count),
                                   C.byref(res), ptr(tr.get("action")), ptr(tr.get("next_state")), ptr(tr.get("code")), ptr(tr.get("reward")))
    if rc:
        raise RuntimeError(f"oracle_population_run failed ({rc})")
    shape = (5, 3, 3, 3, 7, 3)
    return dict(qa=qa.reshape(shape), qb=qb.reshape(shape), count=count.reshape(shape), result=res, **tr)
