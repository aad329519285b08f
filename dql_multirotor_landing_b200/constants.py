"""Host-side constant tables for the CUDA kernels (packed into ``dqlb200_config``, include/dqlb200.h).

Everything here is evaluated ONCE on the host, in float64, with the same expressions the reference
uses, and uploaded; the kernels never re-derive a threshold.  Reference sources:

  * discretisation limits / goal widths / angles      PKG/mdp.py:42-65, 145, 149-170, 257-333
  * terminal checks                                   PKG/mdp.py:335-439
  * reward constants                                  PKG/mdp.py:441-541
  * learning-rate, exploration, transfer schedules    PKG/trainer.py:88-138
  * promotion rule                                    PKG/trainer.py:219-236

(PKG = src/dql_multirotor_landing/src/dql_multirotor_landing in the reference tree.)

The key trick ("cut points"): every float64 comparison the reference makes on
``clip(x / x_max, -1, 1)`` is monotone in x.  The kernels hold x in fp32, so each comparison is
equivalent to ``x >= cut`` for one fp32 number ``cut`` -- found here by bisection over the fp32
number line, evaluating the reference's float64 expression.  The device then discretises with a
handful of fp32 compares and is bit-exact by construction.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass, field
from typing import Callable, List, Optional, Sequence

import numpy as np

MAX_CURRICULUM = 5
STATES_PER_LEVEL = 189
CELLS_PER_LEVEL = 567
MAX_CELLS = MAX_CURRICULUM * CELLS_PER_LEVEL
ALPHA_LUT = 1003
EPS_LUT = 2002
MAX_SETPOINTS = 64              # DQLB200_MAX_SETPOINTS
MAX_WINDOW = 128
ENV_STATE_BYTES = 48
ABI_VERSION = 11

LIMITS_POSITION = [1.0, 0.64, 0.4096, 0.262144, 0.16777216]   # PKG/mdp.py:45-47
LIMITS_VELOCITY = [1.0, 0.8, 0.64, 0.512, 0.4096]              # PKG/mdp.py:48-50
LIMITS_ACCELERATION = [1.0, 1.0, 1.0, 1.0, 1.0]                # PKG/mdp.py:51-53

TERMINATION_STRINGS = {   # CheckResult values, PKG/mdp.py:69-75
    2: "SUCCESS: Goal state reached",
    3: "SUCCESS: Touched platform",
    4: "FAILURE: Drone moved too far from platform in x direction",
    5: "FAILURE: Drone moved too far from platform in y direction",
    6: "FAILURE: Drone moved too far from platform in z direction",
    7: "FAILURE: Reached minimum altitude",
    8: "FAILURE: Maximum episode duration",
}


# ------------------------------------------------------------------------------------------------
# ctypes mirrors of include/dqlb200.h
# ------------------------------------------------------------------------------------------------
class Cuts(C.Structure):
    _fields_ = [("lvl_lo", (C.c_float * 4) * 2), ("lvl_hi", (C.c_float * 4) * 2),
                ("bin1", (C.c_float * 5) * 3), ("bin2", (C.c_float * 5) * 3)]


class RewardLevel(C.Structure):
    _fields_ = [("lim_v", C.c_double), ("r_p_max", C.c_double), ("r_v_max", C.c_double),
                ("r_dur", C.c_double), ("r_term_succ", C.c_double), ("r_term_fail", C.c_double)]


class SetpointNext(C.Structure):
    _fields_ = [("next", C.c_uint32), ("value_f32", C.c_float)]


class Config(C.Structure):
    _fields_ = [
        ("struct_bytes", C.c_uint32), ("abi_version", C.c_uint32),
        ("n_populations", C.c_int32), ("envs_per_population", C.c_int32),
        ("curriculum_steps", C.c_int32), ("threads_per_block", C.c_int32),
        ("cuts", Cuts * MAX_CURRICULUM), ("angle_cut", C.c_float * 6),
        ("fz_lo", C.c_float), ("fz_hi", C.c_float), ("z_min_cut", C.c_float), ("z_max_cut", C.c_float),
        ("timeout_steps", C.c_int32), ("success_steps", C.c_int32),
        ("reward", RewardLevel * MAX_CURRICULUM),
        ("p_max", C.c_double), ("v_max", C.c_double), ("theta_max", C.c_double), ("delta_theta", C.c_double),
        ("w_p", C.c_double), ("w_v", C.c_double), ("w_theta", C.c_double),
        ("a_max", C.c_double), ("minimum_altitude", C.c_double), ("timeout_threshold", C.c_double), ("f_ag", C.c_double),
        ("limits", (C.c_double * MAX_CURRICULUM) * 3),
        ("goal_width", ((C.c_double * MAX_CURRICULUM) * 3) * MAX_CURRICULUM),
        ("angles", C.c_double * 7),
        ("h", C.c_float), ("half_h2", C.c_float), ("k_theta", C.c_float), ("g", C.c_float), ("c_d", C.c_float),
        ("dz_train", C.c_float), ("dz_sim", C.c_float), ("z_init", C.c_float), ("z_touch", C.c_float),
        ("half_platform", C.c_float), ("p_max_f", C.c_float), ("two_p_max_f", C.c_float), ("sigma_x", C.c_float),
        ("n_sub", C.c_int32),
        ("gamma", C.c_float), ("transfer_ratio", C.c_float * MAX_CURRICULUM), ("transfer_mode", C.c_int32),
        ("window_len", C.c_int32), ("promote_successes", C.c_int32), ("max_num_episodes", C.c_int64),
        ("n_alpha_luts", C.c_int32), ("replicas_per_population", C.c_int32),
        ("noise_pos_sd", C.c_float), ("noise_vel_sd", C.c_float),
        ("accel_mode", C.c_int32), ("kf_q", C.c_float), ("kf_r", C.c_float),
        ("dynamics_model", C.c_int32), ("pid_ticks", C.c_int32),
        ("att_kr", C.c_float), ("att_kw", C.c_float), ("inv_m", C.c_float), ("inv_mg", C.c_float), ("g_abs", C.c_float),
        ("pid_kp", C.c_float), ("pid_ki", C.c_float), ("pid_lo", C.c_float), ("pid_hi", C.c_float), ("pid_windup", C.c_float),
        ("pid_dt", C.c_float), ("pid_i0", C.c_float), ("bw_inv_denom", C.c_float), ("bw_k2", C.c_float),
        ("vz_train", C.c_float), ("vz_sim", C.c_float),
        ("eps_threshold", C.c_uint32 * EPS_LUT),
        ("n_setpoints", C.c_int32), ("setpoint_zero", C.c_int32),
        ("setpoint_value", C.c_double * MAX_SETPOINTS),
        ("setpoint_next", (SetpointNext * 3) * MAX_SETPOINTS),
        ("setpoint_rtheta", ((C.c_double * 3) * MAX_SETPOINTS) * 2),
    ]


class PopulationParams(C.Structure):
    _fields_ = [("seed_lo", C.c_uint32), ("seed_hi", C.c_uint32), ("population_id", C.c_uint32),
                ("dphase", C.c_uint32), ("r", C.c_float), ("rw", C.c_float), ("rw2", C.c_float),
                ("alpha_lut", C.c_int32), ("g", C.c_float), ("axis", C.c_int32)]


class PopulationState(C.Structure):
    _fields_ = [
        ("working_step", C.c_int32), ("finished", C.c_int32), ("t", C.c_uint32), ("error_flags", C.c_uint32),
        ("episodes_in_step", C.c_int64),
        ("window_head", C.c_int32), ("window_count", C.c_int32), ("window_sum", C.c_int32), ("pending_advance", C.c_int32),
        ("window", C.c_uint8 * MAX_WINDOW),
        ("total_steps", C.c_uint64), ("total_episodes", C.c_uint64), ("total_successes", C.c_uint64),
        ("termination_hist", C.c_uint64 * 9),
        ("return_sum", C.c_double), ("episode_steps_sum", C.c_uint64),
        ("promoted_at", C.c_uint32 * MAX_CURRICULUM),
        ("last_code", C.c_int32), ("last_steps", C.c_int32), ("last_cumulative", C.c_double),
    ]


POPULATION_STATE_DTYPE = np.dtype([
    ("working_step", "<i4"), ("finished", "<i4"), ("t", "<u4"), ("error_flags", "<u4"),
    ("episodes_in_step", "<i8"),
    ("window_head", "<i4"), ("window_count", "<i4"), ("window_sum", "<i4"), ("pending_advance", "<i4"),
    ("window", "u1", (MAX_WINDOW,)),
    ("total_steps", "<u8"), ("total_episodes", "<u8"), ("total_successes", "<u8"),
    ("termination_hist", "<u8", (9,)),
    ("return_sum", "<f8"), ("episode_steps_sum", "<u8"),
    ("promoted_at", "<u4", (MAX_CURRICULUM,)),
    ("last_code", "<i4"), ("last_steps", "<i4"), ("last_cumulative", "<f8"),
], align=True)
assert POPULATION_STATE_DTYPE.itemsize == C.sizeof(PopulationState)


class Trace(C.Structure):
    _fields_ = [("obs", C.c_void_p), ("reward", C.c_void_p), ("action", C.c_void_p), ("code", C.c_void_p),
                ("done", C.c_void_p), ("contact", C.c_void_p), ("state", C.c_void_p), ("next_state", C.c_void_p),
                ("episode", C.c_void_p), ("action_override", C.c_void_p)]


class EvalStats(C.Structure):
    _fields_ = [("episodes", C.c_uint64), ("steps", C.c_uint64), ("termination_hist", C.c_uint64 * 9)]


class Platform(C.Structure):
    """dqlb200_platform (include/dqlb200.h): one platform motion of dqlb200_eval_agents_platforms, the fields of
    PopulationParams with the same names (platform_constants)."""
    _fields_ = [("dphase", C.c_uint32), ("r", C.c_float), ("rw", C.c_float), ("rw2", C.c_float)]


class Eval2DParams(C.Structure):
    """dqlb200_eval2d_params (include/dqlb200.h)."""
    _fields_ = [("seed_lo", C.c_uint32), ("seed_hi", C.c_uint32), ("stream_id", C.c_uint32), ("trajectory", C.c_int32),
                ("dphase_x", C.c_uint32), ("dphase_y", C.c_uint32),
                ("r_x", C.c_float), ("rw_x", C.c_float), ("rw2_x", C.c_float), ("r_y", C.c_float), ("rw_y", C.c_float), ("rw2_y", C.c_float),
                ("g_x", C.c_float), ("g_y", C.c_float), ("y_action_enabled", C.c_int32), ("y_init_enabled", C.c_int32),
                ("working_step", C.c_int32), ("reserved", C.c_int32)]


class Trace2D(C.Structure):
    _fields_ = [("obs", C.c_void_p), ("action_x", C.c_void_p), ("action_y", C.c_void_p), ("code", C.c_void_p), ("done", C.c_void_p),
                ("contact", C.c_void_p), ("state_x", C.c_void_p), ("state_y", C.c_void_p)]


TRAJ_RECTILINEAR_X, TRAJ_RECTILINEAR_XY, TRAJ_EIGHT = 0, 1, 2
SHARED_WORDS = 2 * MAX_CELLS + 4              # DQLB200_SHARED_WORDS: 32-bit words per agent and rank in the shared-table exchange


# ------------------------------------------------------------------------------------------------
# parameters (defaults = the reference's)
# ------------------------------------------------------------------------------------------------
@dataclass
class MdpParameters:
    """TrainingMdp / SimulationMdp keyword defaults (PKG/mdp.py:214-235, 582-603)."""
    f_ag: float = 22.92
    t_max: float = 20
    p_max: float = 4.5
    w_p: float = -100.0
    w_v: float = -10.0
    w_theta: float = -1.55
    w_dur: float = -6.0
    w_fail: float = -2.6
    w_succ: float = 2.6
    n_theta: int = 3
    v_max: float = 3.39411
    a_max: float = 1.28
    theta_max: float = float(np.deg2rad(21.37723))
    delta_theta: float = float(np.deg2rad(7.12574))
    beta: float = 1 / 3
    sigma_a: float = 0.416
    minimum_altitude: float = 0.2


ACCEL_MODES = {"exact": 0, "kalman_reference": 1, "kalman": 2}
DYNAMICS_MODELS = {"first_order": 0, "second_order": 1}


@dataclass
class DynamicsParameters:
    """Analytic stand-in for the Gazebo/RotorS path (DESIGN.md; parameters traced in SURVEY.md A.3)."""
    tau_theta: float = 1.0 / 7.0     # k_omega / k_R          PKG/attitude_controller.py:86-87
    c_d: float = 0.2                 # rotor drag / mass       gazebo_motor_model.cpp:464-466
    g: float = 9.81                  #                         PKG/attitude_controller.py:59
    r_mp: float = 2.0                # platform amplitude      PKG/moving_platform.py (r_x)
    v_mp: float = 1.6                # platform max speed      launch/environment.launch:62-64
    z_init: float = 4.0              #                         PKG/trainer.py:41
    v_z_train: float = -0.1          #                         PKG/mdp.py:212
    v_z_sim: float = -0.4            #                         PKG/mdp.py:580
    z_touch: float = 0.515           # bumper top + body       urdf/moving_platform.urdf:16,38,51,58
    half_platform: float = 0.5
    n_sub: int = 1
    noise_pos_sd: float = 0.0        # Gaussian noise on the observed rel. position   PKG/observation_utils.py:127-129 (launch: 0)
    noise_vel_sd: float = 0.0        # ... and velocity (manager_node defaults 0.25 / 0.1, launch/environment.launch:56-57 sets 0)
    # relative acceleration seen by the MDP: "exact" (analytic), "kalman_reference" (PKG/filters.py:4-80 over the finite
    # difference against the FIRST sample, as PKG/observation_utils.py:137-150 is written), "kalman" (consecutive samples)
    accel_mode: str = "exact"
    kf_process_variance: float = 1e-4      # scripts/manager_node.py:96-98
    kf_measurement_sd: float = 0.1         # manager_node passes noise_vel_sd (default 0.1); R = sd ** 2 (PKG/filters.py:50-52)
    # "first_order" (the stand-in of SURVEY A.3) or "second_order": attitude as torque on inertia under the geometric controller
    # (PKG/attitude_controller.py:86-87,124-156) + the vertical PID node (PKG/pid.py:62-104, launch/drone.launch:33-46)
    dynamics_model: str = "first_order"
    mass: float = 0.68                     # PKG/attitude_controller.py:57, hummingbird.xacro:29
    inertia: float = 0.007                 # PKG/attitude_controller.py:59 (Ixx = Iyy)
    k_R: float = 0.7                       # PKG/attitude_controller.py:86
    k_omega: float = 0.1                   # PKG/attitude_controller.py:87
    pid_kp: float = 5.0                    # launch/drone.launch:35-40
    pid_ki: float = 10.0
    pid_lower: float = 0.0
    pid_upper: float = 10.0
    pid_windup: float = 10.0
    pid_ticks: int = 10                    # PID node iterations per sub-step (rate_hz 1000 against the 100 Hz state topic, PKG/pid.py:14)


@dataclass
class TwoAxisParameters:
    """Platform and axis conventions of the two-axis evaluator (dqlb200_eval_greedy_2d).  Defaults = the reference:
    rectilinear periodic platform along x only (PKG/moving_platform.py:113-125), y action and y start offset disabled
    (PKG/mdp.py:863-876, PKG/landing_simulation_env.py:336-340).  `eight` uses r = 3, v = 0.8 (PKG/moving_platform.py:92-96)."""
    trajectory: int = 0
    r_x: float = 2.0
    v_x: float = 1.6
    r_y: float = 2.0
    v_y: float = 1.0
    g_y_sign: float = -1.0           # a_y = -g tan(roll) in the reference's ENU frame
    y_action_enabled: bool = False
    y_init_enabled: bool = False


def eval2d_params(ta: "TwoAxisParameters", dp: "DynamicsParameters", f_ag: float, seed: int, stream_id: int, working_step: int) -> Eval2DParams:
    h = (1.0 / f_ag) / dp.n_sub
    wx = ta.v_x / ta.r_x
    turns = lambda w: int(round(w * h / (2.0 * math.pi) * 2.0 ** 32)) & 0xFFFFFFFF
    f = np.float32
    if ta.trajectory == TRAJ_EIGHT:
        dpy, ry, rwy, rw2y = turns(wx), f(ta.r_y), f(ta.r_y * wx), f(4.0 * ta.r_y * wx * wx)
    elif ta.trajectory == TRAJ_RECTILINEAR_XY:
        wy = ta.v_y / ta.r_y
        dpy, ry, rwy, rw2y = turns(wy), f(ta.r_y), f(ta.r_y * wy), f(ta.r_y * wy * wy)
    else:
        dpy, ry, rwy, rw2y = 0, f(0.0), f(0.0), f(0.0)
    return Eval2DParams(seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF, stream_id, ta.trajectory, turns(wx), dpy,
                        f(ta.r_x), f(ta.r_x * wx), f(ta.r_x * wx * wx), ry, rwy, rw2y, f(dp.g), f(ta.g_y_sign * dp.g),
                        int(ta.y_action_enabled), int(ta.y_init_enabled), working_step, 0)


@dataclass
class TrainerParameters:
    """Trainer keyword defaults (PKG/trainer.py:20-44)."""
    curriculum_steps: int = 5
    successive_successful_episodes: int = 100
    success_rate: float = 0.96
    max_num_episodes: int = 50000
    alpha_min: float = 0.02949
    omega: float = 0.51
    gamma: float = 0.99
    scale_modification_value: Sequence[float] = (0.8172650252856599, 0.8211253690681617,
                                                 0.8257273369742982, 0.8311571820651724)
    transfer_mode: str = "reference"   # "reference": quirk Q7 (PKG/trainer.py:238-243); "paper": scale k-1 -> k before step k


# ------------------------------------------------------------------------------------------------
# schedules (PKG/trainer.py:88-138)
# ------------------------------------------------------------------------------------------------
def alpha_value(count: float, alpha_min: float, omega: float) -> float:
    if count == 0:
        return alpha_min
    return float(np.max([np.float_power(1 / count, omega), alpha_min]))


def alpha_lut(alpha_min: float = 0.02949, omega: float = 0.51) -> np.ndarray:
    """float32(alpha(count)) for count 0..1002.  The last entry must be the saturated value."""
    lut = np.asarray([alpha_value(c, alpha_min, omega) for c in range(ALPHA_LUT)], np.float64)
    for c in (ALPHA_LUT - 1, ALPHA_LUT, 5 * ALPHA_LUT, 10 ** 7):
        if alpha_value(c, alpha_min, omega) != alpha_min:
            raise ValueError(f"alpha schedule (alpha_min={alpha_min}, omega={omega}) does not saturate by count "
                             f"{ALPHA_LUT - 1}; the device LUT cannot represent it")
    return lut.astype(np.float32)


def exploration_rate(episode: int, working_step: int) -> float:
    if working_step > 0:
        return 0.0
    if 0 <= episode <= 800:
        return 1.0
    return max(1 + (0.01 - 1) * (episode - 800) / (2000 - 800), 0.01)


def explore_threshold(eps: float) -> int:
    """uniform = u24 * 2**-24 (exact);  uniform < eps  <=>  u24 < ceil(eps * 2**24)."""
    return int(math.ceil(eps * 2.0 ** 24))


def transfer_learning_ratio(step: int, scale: Sequence[float]) -> float:
    if step < 1:
        return 1.0
    if step < len(scale) + 1:
        return scale[step - 1]
    raise ValueError(f"Transfer learning can be done up to he 5th curiculum_step, {step} is invalid")


# ------------------------------------------------------------------------------------------------
# fp32 cut points
# ------------------------------------------------------------------------------------------------
def _key_to_f32(k: int) -> np.float32:
    """Order-preserving map: integer k in [0, 2**32) -> fp32 (-inf .. +inf, NaNs at the ends)."""
    b = (k ^ 0x80000000) if (k & 0x80000000) else (~k & 0xFFFFFFFF)
    return np.array([b], np.uint32).view(np.float32)[0]


def _f32_to_key(x) -> int:
    b = int(np.array([x], np.float32).view(np.uint32)[0])
    return (b ^ 0x80000000) if not (b & 0x80000000) else (~b & 0xFFFFFFFF)


_KEY_NEG_INF = _f32_to_key(np.float32(-np.inf))
_KEY_POS_INF = _f32_to_key(np.float32(np.inf))


def first_true(pred: Callable[[float], bool]) -> np.float32:
    """Smallest fp32 x (in -inf..+inf) with pred(float(x)) True, for pred monotone False->True.
    Returns NaN when pred is never true (then `x >= cut` is false for every x, as required)."""
    lo, hi = _KEY_NEG_INF, _KEY_POS_INF
    if pred(float(_key_to_f32(lo))):
        return np.float32(-np.inf)
    if not pred(float(_key_to_f32(hi))):
        return np.float32(np.nan)
    while hi - lo > 1:          # invariant: pred(lo) False, pred(hi) True
        mid = (lo + hi) // 2
        if pred(float(_key_to_f32(mid))):
            hi = mid
        else:
            lo = mid
    return _key_to_f32(hi)


def _clip(x: float, lo: float, hi: float) -> float:
    return float(np.clip(x, lo, hi))


def goal_width(q: int, level: int, w: int, mp: MdpParameters) -> float:
    """limit[level] * contraction, exactly as PKG/mdp.py:285-317 forms it."""
    if q == 2:
        contraction = mp.sigma_a
        if level == w:
            contraction *= mp.beta
        return LIMITS_ACCELERATION[level] * contraction
    lim = LIMITS_POSITION if q == 0 else LIMITS_VELOCITY
    contraction = mp.beta
    if level < w:
        contraction = lim[level + 1] / lim[level]
    return lim[level] * contraction


def build_cuts(w: int, mp: MdpParameters) -> Cuts:
    cuts = Cuts()
    norm = [mp.p_max, mp.v_max, mp.a_max]
    lims = [LIMITS_POSITION, LIMITS_VELOCITY, LIMITS_ACCELERATION]
    nan = float("nan")
    for q in range(3):
        v = lambda x, q=q: _clip(x / norm[q], -1, 1)
        if q < 2:
            for idx in range(1, 5):
                if idx <= w:
                    lim = lims[q][idx]
                    cuts.lvl_lo[q][idx - 1] = first_true(lambda x: not (v(x) < -lim))
                    cuts.lvl_hi[q][idx - 1] = first_true(lambda x: v(x) > lim)
                else:   # level idx does not exist at this working step: never "inside"
                    cuts.lvl_lo[q][idx - 1] = nan
                    cuts.lvl_hi[q][idx - 1] = nan
        for level in range(5):
            if level <= w:
                goal = goal_width(q, level, w, mp)
                cuts.bin1[q][level] = first_true(lambda x: not (v(x) < -goal))
                cuts.bin2[q][level] = first_true(lambda x: v(x) > goal)
            else:
                cuts.bin1[q][level] = nan
                cuts.bin2[q][level] = nan
    return cuts


def build_angle_cuts(mp: MdpParameters) -> List[np.float32]:
    angles = np.linspace(-mp.theta_max, mp.theta_max, (mp.n_theta * 2) + 1)   # PKG/mdp.py:145

    def index(x: float) -> int:
        return int(np.argmin(np.abs(angles - np.clip(x, -mp.theta_max, mp.theta_max))))   # PKG/mdp.py:318-323

    return [first_true(lambda x, i=i: index(x) >= i + 1) for i in range(6)]


def build_reward_levels(mp: MdpParameters) -> List[RewardLevel]:
    dt = 1 / mp.f_ag
    out = []
    for level in range(MAX_CURRICULUM):
        lv, la = LIMITS_VELOCITY[level], LIMITS_ACCELERATION[level]
        r_p_max = np.abs(mp.w_p) * lv * dt
        r_v_max = np.abs(mp.w_v) * la * dt
        r_theta_max = np.abs(mp.w_theta) * (mp.delta_theta / mp.theta_max) * lv
        r_dur_max = mp.w_dur * lv * dt
        r_max = r_p_max + r_v_max + r_theta_max + r_dur_max
        out.append(RewardLevel(lv, float(r_p_max), float(r_v_max), float(mp.w_dur * lv * dt),
                               float(mp.w_succ * r_max), float(mp.w_fail * r_max)))
    return out


def build_setpoints(mp: MdpParameters):
    """Closure of the pitch set-point under TrainingMdp.continuous_action (PKG/mdp.py:543-560) starting from 0.0, with the
    reference's own float64 operations (min / max of Python floats after one add).  Returns (values sorted, index of 0.0,
    next[i][a], rtheta[fresh][prev][a]) -- rtheta is the set-point part of the reward in the reference's operation order:
    w_theta * (|phi(next)| - |phi(prev)|) / theta_max with phi(i) = w_theta * |value[i] / theta_max| (PKG/mdp.py:463-474, 506-514)."""
    tm, d = float(mp.theta_max), float(mp.delta_theta)
    seen, frontier = {0.0}, [0.0]
    while frontier:
        v = frontier.pop()
        for nv in (min((v + d, tm)), max((v - d, -tm))):
            if nv not in seen:
                if len(seen) >= MAX_SETPOINTS:
                    raise ValueError(f"more than {MAX_SETPOINTS} reachable pitch set-points for theta_max={tm}, delta_theta={d}")
                seen.add(nv)
                frontier.append(nv)
    values = sorted(seen)
    index = {v: i for i, v in enumerate(values)}
    zero = index[0.0]
    nxt = [[index[min((v + d, tm))], index[max((v - d, -tm))], i] for i, v in enumerate(values)]
    phi = [mp.w_theta * np.abs(v / mp.theta_max) for v in values]
    rtheta = [[[float(mp.w_theta * (np.abs(phi[nxt[zero if fresh else p][a]]) - np.abs(phi[p])) / mp.theta_max) for a in range(3)]
               for p in range(len(values))] for fresh in (0, 1)]
    return values, zero, nxt, rtheta


def first_int_at_least(x: float) -> int:
    n = max(int(x) - 1, 0)
    while not (n >= x):
        n += 1
    return n


def promote_threshold(window_len: int, success_rate: float) -> int:
    """First integer s with s / window_len > success_rate (PKG/trainer.py:222-232); window_len+1 if none."""
    for s in range(window_len + 1):
        if s / window_len > success_rate:
            return s
    return window_len + 1


def platform_constants(r_mp: float, v_mp: float, f_ag: float, n_sub: int):
    """(dphase, r, r*w, r*w^2): platform x = r sin(w t), w = v/r (PKG/moving_platform.py:116-125)."""
    h = (1.0 / f_ag) / n_sub
    w = v_mp / r_mp
    dphase = int(round(w * h / (2.0 * math.pi) * 2.0 ** 32)) & 0xFFFFFFFF
    return dphase, np.float32(r_mp), np.float32(r_mp * w), np.float32(r_mp * w * w)


def platform_motions(platforms) -> np.ndarray:
    """A list of platform motions (r_mp, v_mp) as float64 [C, 2]; ValueError for an empty list, a wrong shape, a non-finite value,
    r_mp <= 0 or v_mp < 0."""
    try:
        pl = np.asarray(platforms, dtype=np.float64)
    except (TypeError, ValueError) as e:
        raise ValueError(f"platforms must be a sequence of (r_mp, v_mp) pairs: {e}") from None
    if pl.ndim != 2 or pl.shape[1] != 2 or len(pl) < 1:
        raise ValueError(f"platforms must be a non-empty sequence of (r_mp, v_mp) pairs, got shape {pl.shape}")
    if not np.isfinite(pl).all():
        raise ValueError("platforms: r_mp and v_mp must be finite")
    if not (pl[:, 0] > 0).all() or not (pl[:, 1] >= 0).all():
        raise ValueError("platforms: r_mp must be > 0 and v_mp >= 0")
    return pl


def build_config(n_populations: int, envs_per_population: int, threads_per_block: int = 256,
                 mp: Optional[MdpParameters] = None, dp: Optional[DynamicsParameters] = None,
                 tp: Optional[TrainerParameters] = None, n_alpha_luts: int = 1, replicas_per_population: int = 1) -> Config:
    mp, dp, tp = mp or MdpParameters(), dp or DynamicsParameters(), tp or TrainerParameters()
    if not (1 <= tp.curriculum_steps <= MAX_CURRICULUM):
        raise ValueError("curriculum_steps must be in 1..5 (the reference's Limits hold 5 levels)")
    if not (1 <= tp.successive_successful_episodes <= MAX_WINDOW):
        raise ValueError(f"successive_successful_episodes must be in 1..{MAX_WINDOW}")
    cfg = Config()
    cfg.struct_bytes, cfg.abi_version = C.sizeof(Config), ABI_VERSION
    cfg.n_populations, cfg.envs_per_population = n_populations, envs_per_population
    cfg.curriculum_steps, cfg.threads_per_block = tp.curriculum_steps, threads_per_block
    for w in range(MAX_CURRICULUM):
        cfg.cuts[w] = build_cuts(w, mp)
    for i, c in enumerate(build_angle_cuts(mp)):
        cfg.angle_cut[i] = c
    cfg.fz_lo = first_true(lambda x: not (x < -mp.p_max))       # PKG/mdp.py:365-368
    cfg.fz_hi = first_true(lambda x: x > mp.p_max)
    cfg.z_min_cut = first_true(lambda z: not (z < mp.minimum_altitude))   # PKG/mdp.py:383
    cfg.z_max_cut = first_true(lambda z: z > mp.p_max)                    # PKG/mdp.py:389
    cfg.timeout_steps = first_int_at_least(mp.t_max * mp.f_ag)            # PKG/mdp.py:395
    cfg.success_steps = first_int_at_least(mp.f_ag)                       # PKG/mdp.py:415
    for level, rl in enumerate(build_reward_levels(mp)):
        cfg.reward[level] = rl
    cfg.p_max, cfg.v_max, cfg.theta_max, cfg.delta_theta = mp.p_max, mp.v_max, mp.theta_max, mp.delta_theta
    cfg.w_p, cfg.w_v, cfg.w_theta = mp.w_p, mp.w_v, mp.w_theta
    cfg.a_max, cfg.minimum_altitude, cfg.f_ag = mp.a_max, mp.minimum_altitude, mp.f_ag
    cfg.timeout_threshold = mp.t_max * mp.f_ag
    for q, lim in enumerate((LIMITS_POSITION, LIMITS_VELOCITY, LIMITS_ACCELERATION)):
        for level in range(MAX_CURRICULUM):
            cfg.limits[q][level] = lim[level]
    for w in range(MAX_CURRICULUM):
        for q in range(3):
            for level in range(MAX_CURRICULUM):
                cfg.goal_width[w][q][level] = goal_width(q, level, w, mp) if level <= w else float("nan")
    for i, a in enumerate(np.linspace(-mp.theta_max, mp.theta_max, (mp.n_theta * 2) + 1)):
        cfg.angles[i] = a
    h = (1.0 / mp.f_ag) / dp.n_sub
    cfg.h, cfg.half_h2 = h, 0.5 * h * h
    cfg.k_theta = -math.expm1(-h / dp.tau_theta)
    cfg.g, cfg.c_d = dp.g, dp.c_d
    cfg.dz_train, cfg.dz_sim = dp.v_z_train * (1.0 / mp.f_ag), dp.v_z_sim * (1.0 / mp.f_ag)
    cfg.z_init, cfg.z_touch, cfg.half_platform = dp.z_init, dp.z_touch, dp.half_platform
    cfg.p_max_f, cfg.two_p_max_f, cfg.sigma_x = mp.p_max, 2.0 * mp.p_max, mp.p_max / 3.0
    cfg.n_sub = dp.n_sub
    cfg.noise_pos_sd, cfg.noise_vel_sd = dp.noise_pos_sd, dp.noise_vel_sd
    cfg.accel_mode = ACCEL_MODES[dp.accel_mode]
    cfg.kf_q, cfg.kf_r = dp.kf_process_variance, dp.kf_measurement_sd ** 2
    cfg.dynamics_model = DYNAMICS_MODELS[dp.dynamics_model]
    cfg.pid_ticks = dp.pid_ticks
    g_abs = abs(dp.g)
    cfg.att_kr, cfg.att_kw = dp.k_R / dp.inertia, dp.k_omega / dp.inertia
    cfg.inv_m, cfg.inv_mg, cfg.g_abs = 1.0 / dp.mass, 1.0 / (dp.mass * g_abs), g_abs
    cfg.pid_kp, cfg.pid_ki, cfg.pid_lo, cfg.pid_hi, cfg.pid_windup = dp.pid_kp, dp.pid_ki, dp.pid_lower, dp.pid_upper, dp.pid_windup
    cfg.pid_dt = h / max(dp.pid_ticks, 1)
    cfg.pid_i0 = dp.mass * g_abs / dp.pid_ki if dp.pid_ki else 0.0
    cfg.bw_inv_denom, cfg.bw_k2 = 1.0 / (1 + 1.0 ** 2 + 1.414 * 1.0), 1.0 ** 2 - 1.414 * 1.0 + 1      # PKG/filters.py:92-93,103 with c = 1
    cfg.vz_train, cfg.vz_sim = dp.v_z_train, dp.v_z_sim
    cfg.gamma = tp.gamma
    for k in range(MAX_CURRICULUM):
        cfg.transfer_ratio[k] = transfer_learning_ratio(k, tp.scale_modification_value)
    cfg.transfer_mode = {"reference": 0, "paper": 1}[tp.transfer_mode]
    cfg.window_len = tp.successive_successful_episodes
    cfg.promote_successes = promote_threshold(tp.successive_successful_episodes, tp.success_rate)
    cfg.max_num_episodes = tp.max_num_episodes
    cfg.n_alpha_luts = n_alpha_luts
    if replicas_per_population < 1 or n_populations % replicas_per_population:
        raise ValueError("n_populations must be a multiple of replicas_per_population")
    cfg.replicas_per_population = replicas_per_population
    for e in range(EPS_LUT):
        cfg.eps_threshold[e] = explore_threshold(exploration_rate(e, 0))
    values, zero, nxt, rtheta = build_setpoints(mp)
    cfg.n_setpoints, cfg.setpoint_zero = len(values), zero
    for i, v in enumerate(values):
        cfg.setpoint_value[i] = v
        for a in range(3):
            cfg.setpoint_next[i][a].next = nxt[i][a]
            cfg.setpoint_next[i][a].value_f32 = np.float32(values[nxt[i][a]])
            for fresh in (0, 1):
                cfg.setpoint_rtheta[fresh][i][a] = rtheta[fresh][i][a]
    return cfg
