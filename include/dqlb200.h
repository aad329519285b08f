/*
 * dqlb200.h -- C-ABI of libdqlb200.so: the B200 (sm_100a) implementation of the batched
 * landing-MDP step + tabular Double-Q update.
 *
 * The reference (valerio98-lab/DQL_multirotor_landing) has NO FFI for this path: its boundary is the
 * Python class API in src/dql_multirotor_landing/src/dql_multirotor_landing/{mdp,double_q_learning,
 * trainer}.py ("PKG/" below).  Each entry point names the reference code it replaces.  The Python
 * side of this repo (dql_multirotor_landing_b200/) binds these symbols with ctypes and mirrors the
 * reference classes on top; INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success, a negative dqlb200_status otherwise; the message of the
 *     last error of the calling thread is dqlb200_last_error();
 *   - device buffers are BORROWED (caller-owned, e.g. torch tensors; they must outlive the calls);
 *   - all work is enqueued on the caller's cudaStream_t (passed as void*); nothing synchronises
 *     unless the name says so (`_host` entry points copy and synchronise);
 *   - one host thread per handle; no global mutable state besides the thread-local error string.
 */
#ifndef DQLB200_H
#define DQLB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DQLB200_ABI_VERSION 11
#define DQLB200_MAX_CURRICULUM 5
#define DQLB200_STATES_PER_LEVEL 189          /* 3*3*3*7      (PKG/double_q_learning.py:38-40) */
#define DQLB200_CELLS_PER_LEVEL 567           /* 189 * 3 actions */
#define DQLB200_MAX_CELLS (DQLB200_MAX_CURRICULUM * DQLB200_CELLS_PER_LEVEL)   /* 2835 */
#define DQLB200_ALPHA_LUT 1003                /* count 0..1002; alpha(count >= 1002) == alpha_min */
#define DQLB200_EPS_LUT 2002                  /* episode 0..2000, [2001] = every later episode */
#define DQLB200_MAX_SETPOINTS 64              /* reachable pitch set-points (33 for the reference defaults) */
#define DQLB200_MAX_WINDOW 128                /* success window (Trainer successive_successful_episodes) */
#define DQLB200_SHARED_WORDS (2 * DQLB200_MAX_CELLS + 4)   /* 32-bit words per agent and rank in the shared-table exchange buffer */
#define DQLB200_ENV_STATE_BYTES 48            /* 3 x 16 B per environment, in tiles of 32 envs: [population][tile][3][32][16 B] */
#define DQLB200_ENV_TILE_BYTES 1536           /* one tile = 32 envs of one population = three contiguous 512-byte runs */

typedef enum dqlb200_status {
  DQLB200_OK = 0,
  DQLB200_ERR_ARG = -1,
  DQLB200_ERR_CUDA = -2,
  DQLB200_ERR_STATE = -3,
  DQLB200_ERR_DEVICE_FLAG = -4                /* a kernel raised an error flag (e.g. NaN observation) */
} dqlb200_status;

/* CheckResult codes (PKG/mdp.py:68-77); the strings are returned by dqlb200_termination_string(). */
enum {
  DQLB200_NON_TERMINAL = 0, DQLB200_NON_TERMINAL_SUCCESS = 1, DQLB200_TERMINAL_SUCCESS = 2,
  DQLB200_TERMINAL_CONTACT = 3, DQLB200_TERMINAL_FLYZONE_X = 4, DQLB200_TERMINAL_FLYZONE_Y = 5,
  DQLB200_TERMINAL_FLYZONE_Z = 6, DQLB200_TERMINAL_MINIMUM_ALTITUDE = 7, DQLB200_TERMINAL_TIMEOUT = 8
};

/* fp32 cut points of the discretisation for ONE working curriculum step w.  Every comparison the
 * reference makes in float64 on clip(x / x_max, -1, 1) (PKG/mdp.py:149-170, 263-317) is monotone in
 * the fp32 observation x, so it equals "x >= cut" for a cut found on the host by bisection over the
 * fp32 number line with the reference's own float64 expression (constants.py).  q: 0 = position,
 * 1 = velocity, 2 = acceleration. */
typedef struct dqlb200_cuts {
  float lvl_lo[2][4];   /* [q][idx-1]: first x with NOT (v < -limit[idx])      idx = 1..4 */
  float lvl_hi[2][4];   /* [q][idx-1]: first x with      v >  limit[idx]                  */
  float bin1[3][5];     /* [q][level]: first x whose bin is >= 1  (v >= -goal)            */
  float bin2[3][5];     /* [q][level]: first x whose bin is == 2  (v >   goal)            */
} dqlb200_cuts;

/* float64 reward constants for one discretisation level (PKG/mdp.py:476-536). */
typedef struct dqlb200_reward_level {
  double lim_v;         /* Limits.velocity[level]                                          */
  double r_p_max;       /* |w_p| * lim_v * dt                                              */
  double r_v_max;       /* |w_v| * lim_a * dt                                              */
  double r_dur;         /* w_dur * lim_v * dt                                              */
  double r_term_succ;   /* w_succ * r_max                                                  */
  double r_term_fail;   /* w_fail * r_max   (also for plain NON_TERMINAL, quirk Q8)         */
} dqlb200_reward_level;

/* Everything the kernels need that does not change during a run.  Built by constants.py with the
 * reference's own expressions; POD, copied to the device by dqlb200_create(). */
typedef struct dqlb200_config {
  uint32_t struct_bytes;            /* = sizeof(dqlb200_config), checked */
  uint32_t abi_version;
  /* ---- layout ---- */
  int32_t n_populations;            /* independent agents (Q-table pairs) on this device */
  int32_t envs_per_population;
  int32_t curriculum_steps;         /* 1..5 (DoubleQLearningAgent(curriculum_steps)) */
  int32_t threads_per_block;        /* 32, 64, 128 or 256: one block per population */
  /* ---- MDP (PKG/mdp.py) ---- */
  dqlb200_cuts cuts[DQLB200_MAX_CURRICULUM];         /* indexed by working step w */
  float angle_cut[6];               /* first pitch whose argmin index is >= i+1 (PKG/mdp.py:318-323) */
  float fz_lo, fz_hi;               /* fly zone x: out  <=>  !(x >= fz_lo) || (x >= fz_hi)  (PKG/mdp.py:365-368) */
  float z_min_cut, z_max_cut;       /* z < minimum_altitude <=> !(z >= z_min_cut); z > p_max <=> z >= z_max_cut */
  int32_t timeout_steps;            /* first integer n with n >= t_max * f_ag   (459); <= 511 to bind an env state */
  int32_t success_steps;            /* first integer n with n >= f_ag           (23);  <= 31 to bind an env state  */
  /* The env state packs the step count into 9 bits and the goal-step count into 5 (csrc/env_state.cuh): dqlb200_bind refuses
   * (DQLB200_ERR_ARG) a configuration whose counts would overflow them.  The facade kernels count in float64 and have no limit. */
  dqlb200_reward_level reward[DQLB200_MAX_CURRICULUM];
  double p_max, v_max, theta_max, delta_theta, w_p, w_v, w_theta;
  /* float64 tables for the facade kernel, which discretises arbitrary float64 observations with the
   * reference's own comparisons (PKG/mdp.py:149-170, 285-323, 383-395) */
  double a_max, minimum_altitude, timeout_threshold /* t_max * f_ag */, f_ag;
  double limits[3][DQLB200_MAX_CURRICULUM];          /* Limits.position / velocity / acceleration */
  double goal_width[DQLB200_MAX_CURRICULUM][3][DQLB200_MAX_CURRICULUM];   /* [w][q][level] */
  double angles[7];                                   /* np.linspace(-theta_max, theta_max, 7) */
  /* ---- stand-in dynamics, fp32, one rounding each (DESIGN.md "dynamics") ---- */
  float h, half_h2, k_theta, g, c_d, dz_train, dz_sim, z_init, z_touch, half_platform;
  float p_max_f, two_p_max_f, sigma_x;
  int32_t n_sub;
  /* ---- agent / trainer schedules (PKG/trainer.py:88-138, PKG/double_q_learning.py) ---- */
  float gamma;
  float transfer_ratio[DQLB200_MAX_CURRICULUM];      /* float32(transfer_learning_ratio(k)) */
  int32_t transfer_mode;            /* 0 = reference (quirk Q7), 1 = paper */
  int32_t window_len;               /* successive_successful_episodes (<= DQLB200_MAX_WINDOW) */
  int32_t promote_successes;        /* first integer s with s / window_len > success_rate */
  int64_t max_num_episodes;
  int32_t n_alpha_luts;             /* learning-rate variants for sweeps (>= 1) */
  int32_t replicas_per_population;  /* 1 = every population is one agent; R > 1 = R consecutive populations are
                                     * replicas of one agent merged by dqlb200_replica_merge (they never promote alone) */
  /* ---- observation realism (SURVEY.md 8f-3): Gaussian noise on the observed relative position / velocity
   * (PKG/observation_utils.py:127-129, manager_node parameters noise_pos_sd / noise_vel_sd; launch default 0 = off).
   * Applied to what the MDP sees (discretisation, fly-zone check, shaping); the physical state and `contact` stay exact. */
  float noise_pos_sd, noise_vel_sd;
  /* ---- observation realism (SURVEY.md 8f-3): the relative acceleration the MDP sees.
   *   0 = exact (the stand-in's analytic acceleration, default)
   *   1 = the reference's estimator as written: a scalar Kalman filter (PKG/filters.py:4-37, Q = kf_q, R = kf_r) over the
   *       finite difference (v_now - v_first) / (t_now - t_first), the anchor sample being the FIRST observation the node ever
   *       made (PKG/observation_utils.py:137-150 never refreshes last_velocity / last_timestep) -- one update per sub-step
   *       (n_sub = 4 is the 100 Hz publish rate of manager_node, scripts/manager_node.py:78-80); the filter and its anchor
   *       live as long as the simulator: they survive episode resets and curriculum steps
   *   2 = the estimator as evidently intended: the same filter over consecutive samples (v_now - v_prev) / h
   * Needs dqlb200_bind_filter_state(). */
  int32_t accel_mode;
  float kf_q, kf_r;                 /* process variance (1e-4), measurement variance (noise_vel_sd^2, scripts/manager_node.py:96-98) */
  /* ---- higher-fidelity per-env model (SURVEY.md 8f-4); 0 = the first-order stand-in (default), 1 = second order:
   *   attitude: the geometric controller of PKG/attitude_controller.py:124-156 reduced to one axis, torque M = -k_R sin(theta -
   *     theta_sp) - k_w omega on the inertia J (att_kr = k_R / J = 0.7 / 0.007, att_kw = k_w / J = 0.1 / 0.007)
   *   vertical: the v_z PID node (PKG/pid.py:62-104, gains launch/drone.launch:33-46: Kp 5, Ki 10, Kd 0, effort in [0, 10] N,
   *     wind-up 10) with its Butterworth error filter (PKG/filters.py:83-108), `pid_ticks` (2..64) node iterations per sub-step;
   *     thrust along the body axis: a_x = sign * (T / m) sin(theta) - c_d v, a_z = (T / m) cos(theta) - g  (m = 0.68)
   * Altitude becomes state (the first-order model derives it from the step count).  Needs dqlb200_bind_dynamics_state(). */
  int32_t dynamics_model, pid_ticks;
  float att_kr, att_kw, inv_m, inv_mg, g_abs;
  float pid_kp, pid_ki, pid_lo, pid_hi, pid_windup, pid_dt, pid_i0 /* m g / Ki: the integral of a hovering simulator */;
  float bw_inv_denom, bw_k2;        /* 1 / (1 + c^2 + 1.414 c), c^2 - 1.414 c + 1 with c = 1 (PKG/filters.py:92-93,103) */
  float vz_train, vz_sim;           /* v_z set-points -0.1 / -0.4 (PKG/mdp.py:212, 580) */
  uint32_t eps_threshold[DQLB200_EPS_LUT];           /* ceil(eps(episode) * 2^24) for working step 0 */
  /* ---- pitch set-point as an index (R3).  TrainingMdp.continuous_action (PKG/mdp.py:543-560) only ever adds / subtracts
   * delta_theta and clamps to +-theta_max, starting from 0 at every reset: the float64 values it can reach form a small closed
   * set (33 for the defaults -- three interleaved lattices, because 3 delta_theta < theta_max by 1.4e-6 delta_theta),
   * enumerated on the host with the reference's own float64 operations (constants.py: build_setpoints).  The env state
   * stores the INDEX; the kernels read, per (index, action), the next index and the float32 set-point for the dynamics, and
   * per (fresh episode?, previous index, action) the set-point term of the reward, w_theta * (|phi(next)| - |phi(prev)|) /
   * theta_max with phi(i) = w_theta * |value[i] / theta_max| (PKG/mdp.py:463-474, 506-514), evaluated on the host in the
   * reference's operation order.  A memoisation of exact arithmetic: identical bits, ~35 instructions per env-step fewer. */
  int32_t n_setpoints, setpoint_zero;                /* size of the set (<= DQLB200_MAX_SETPOINTS), index of 0.0 */
  double setpoint_value[DQLB200_MAX_SETPOINTS];
  struct { uint32_t next; float value_f32; } setpoint_next[DQLB200_MAX_SETPOINTS][3];      /* [index][action] */
  double setpoint_rtheta[2][DQLB200_MAX_SETPOINTS][3];                                      /* [fresh][previous index][action] */
} dqlb200_config;

/* Per-population constants (sweep axes: seed x platform speed x learning-rate schedule). */
typedef struct dqlb200_population_params {
  uint32_t seed_lo, seed_hi;        /* Philox key */
  uint32_t population_id;           /* Philox counter word 3 */
  uint32_t dphase;                  /* platform phase advance per sub-step, uint32 turns */
  float r, rw, rw2;                 /* platform amplitude, r*w, r*w^2 */
  int32_t alpha_lut;                /* index into the alpha LUT array */
  float g;                          /* SIGNED gravity of the agent's axis: a_d = g tan(angle) - c_d v_d.  x agents (pitch): +g;
                                     * y agents (roll, training_y.sh / `direction:=y`): -g in the reference's ENU frame */
  int32_t axis;                     /* 0 = x, 1 = y (informational) */
} dqlb200_population_params;

/* Per-population mutable trainer state (device resident, 320 B).  Mirrors the Trainer fields the
 * reference pickles (PKG/trainer.py:83-86) plus counters replacing its per-episode log. */
typedef struct dqlb200_population_state {
  int32_t working_step;             /* Trainer._working_curriculum_step */
  int32_t finished;                 /* 1 after the last curriculum step ended */
  uint32_t t;                       /* global step index (Philox counter word 1) */
  uint32_t error_flags;             /* bit 0: NaN observation */
  int64_t episodes_in_step;         /* completed episodes in this curriculum step */
  int32_t window_head, window_count, window_sum;
  int32_t pending_advance;          /* set by dqlb200_replica_merge: 1 = promoted, 2 = max_num_episodes reached */
  uint8_t window[DQLB200_MAX_WINDOW];
  uint64_t total_steps, total_episodes, total_successes;
  uint64_t termination_hist[9];
  double return_sum;                /* sum of "Cumulative reward" of finished episodes (quirk Q12) */
  uint64_t episode_steps_sum;
  uint32_t promoted_at[DQLB200_MAX_CURRICULUM];      /* t at which step k ended (0 = not yet) */
  int32_t last_code, last_steps;    /* last finished episode, in env order */
  double last_cumulative;
} dqlb200_population_state;

/* Optional per-step trace for parity tests: arrays of [n_steps][n_envs_total], any may be NULL. */
typedef struct dqlb200_trace {
  float* obs;                       /* [..][5] rel_p, rel_v, rel_a, pitch, z */
  double* reward;
  uint8_t* action; uint8_t* code; uint8_t* done; uint8_t* contact;
  uint16_t* state; uint16_t* next_state;
  int32_t* episode;
  const int8_t* action_override;    /* [n_steps][n_envs_total], < 0 = use the agent */
} dqlb200_trace;

/* Result of dqlb200_eval_greedy (scripts/simulation.py loop, N episodes at once). */
typedef struct dqlb200_eval_stats {
  uint64_t episodes, steps;
  uint64_t termination_hist[9];
} dqlb200_eval_stats;

/* One platform motion x = r sin(w t) of dqlb200_eval_agents_platforms (16 B): the fields of dqlb200_population_params with the
 * same names and meaning, computed on the host the same way (constants.platform_constants(r_mp, v_mp, f_ag, n_sub)). */
typedef struct dqlb200_platform {
  uint32_t dphase;                  /* platform phase advance per sub-step, uint32 turns */
  float r, rw, rw2;                 /* platform amplitude, r*w, r*w^2 */
} dqlb200_platform;

/* Two-axis greedy evaluation (SURVEY.md 8f-2): pitch drives x, roll drives y, one platform under both.
 * trajectory 0: x = r_x sin(w_x t), y = 0                     (PKG/moving_platform.py:113-125 with omega_y = 0)
 *            1: x = r_x sin(w_x t), y = r_y sin(w_y t)        (the "future extension" kept in :113-125)
 *            2: x = r_x cos(w t),  y = r_y sin(w t) cos(w t)  ("eight", PKG/moving_platform.py:92-111; rw2_y holds 4 r_y w^2)
 * g_x / g_y are SIGNED: a = g tan(angle) - c_d v; in the reference's ENU frame g_y = -g.
 * y_action_enabled = 0 reproduces the reference, whose roll branch is dead code (PKG/mdp.py:863-876);
 * y_init_enabled = 0 reproduces `0 * clip(...)` (PKG/landing_simulation_env.py:336-340). */
typedef struct dqlb200_eval2d_params {
  uint32_t seed_lo, seed_hi, stream_id;     /* Philox key and counter word 3 */
  int32_t trajectory;
  uint32_t dphase_x, dphase_y;              /* platform phase advance per sub-step, uint32 turns */
  float r_x, rw_x, rw2_x, r_y, rw_y, rw2_y;
  float g_x, g_y;
  int32_t y_action_enabled, y_init_enabled;
  int32_t working_step;
  int32_t reserved;
} dqlb200_eval2d_params;

/* Optional per-step trace of dqlb200_eval_greedy_2d: arrays [trace_steps][n_episodes], any may be NULL. */
typedef struct dqlb200_trace2d {
  float* obs;                       /* [..][9] rel_p_x, rel_v_x, rel_a_x, pitch, z, rel_p_y, rel_v_y, rel_a_y, roll */
  uint8_t* action_x; uint8_t* action_y; uint8_t* code; uint8_t* done; uint8_t* contact;
  uint16_t* state_x; uint16_t* state_y;     /* states AFTER the step */
} dqlb200_trace2d;

typedef struct dqlb200_handle dqlb200_handle;

int dqlb200_abi_version(void);
size_t dqlb200_config_bytes(void);
size_t dqlb200_population_state_bytes(void);
size_t dqlb200_eval2d_params_bytes(void);
size_t dqlb200_platform_bytes(void);
/* Bytes of the env-state buffer for a layout: n_populations * ceil(envs_per_population / 32) * DQLB200_ENV_TILE_BYTES. */
size_t dqlb200_env_state_bytes(int n_populations, int envs_per_population);
const char* dqlb200_last_error(void);
/* CheckResult.value strings (PKG/mdp.py:69-75); NULL for non-terminal codes. */
const char* dqlb200_termination_string(int code);

/* Replaces: Trainer.__init__ / gym.make("Landing-Training-v0") (PKG/trainer.py:20-86,176-183).
 * alpha_luts: n_alpha_luts x DQLB200_ALPHA_LUT floats (host); pop_params: n_populations entries (host). */
int dqlb200_create(const dqlb200_config* cfg, const float* alpha_luts,
                   const dqlb200_population_params* pop_params, int device, dqlb200_handle** out);
int dqlb200_destroy(dqlb200_handle* h);
/* 1 when the handle's configuration equals the reference-default configuration bit for bit, so that dqlb200_train runs the
 * production instance whose MDP / dynamics constants are compile-time literals; 0: the generic instance (run-time constants,
 * observation noise, any divisor).  Both instances produce identical results for the default configuration. */
int dqlb200_uses_default_instance(dqlb200_handle* h);
/* The same test on a configuration, host only (no device needed): 1 / 0, negative on a malformed struct. */
int dqlb200_config_is_default(const dqlb200_config* cfg);

/* Borrow device buffers.
 *   env_state : dqlb200_env_state_bytes() bytes, 16-B aligned: [population][tile][3][32][16 B] -- a tile holds 32 consecutive
 *               envs of one population as three 512-byte runs (vectors A, B, C); the last tile of a population is padded, so
 *               a population (and any range of populations) is one contiguous block
 *   tables    : [n_populations][3][DQLB200_MAX_CELLS] 32-bit words: Q_a (f32), Q_b (f32), count (u32)
 *               == DoubleQLearningAgent.Q_table_a / Q_table_b / state_action_counter, row-major
 *               (curriculum, p, v, a, theta, action) like the .npy files (PKG/double_q_learning.py:38-53)
 *   pop_state : n_populations x dqlb200_population_state
 * Refused (DQLB200_ERR_ARG) when timeout_steps > 511 or success_steps > 31: the env state cannot count such episodes. */
int dqlb200_bind(dqlb200_handle* h, void* env_state, void* tables, void* pop_state);

/* Borrow the per-env state of the acceleration estimator (accel_mode != 0): n_populations * envs_per_population x 16 bytes
 * {x (f32 estimate), P (f32 variance), v_ref (f32 anchor / previous velocity), n (u32 samples seen)}, 16-B aligned.
 * Replaces: ObservationUtils.filter / last_velocity / last_timestep (PKG/observation_utils.py:44-50).  dqlb200_reset()
 * initialises it (x = 0, P = 1, PKG/filters.py:15-16); nothing else ever clears it. */
int dqlb200_bind_filter_state(dqlb200_handle* h, void* filter_state);

/* Borrow the per-env state of the second-order model (dynamics_model != 0): 32 bytes per env as [2][n] 16-byte vectors
 * {omega, z, v_z, PID integral}, {e1, f1, f2, f3 (Butterworth memory: previous input, three previous outputs)}, 16-B aligned.  Replaces: the Gazebo body state the
 * first-order model does not carry and the memory of the pid_v_z node (PKG/pid.py:14-23).  dqlb200_reset() initialises it. */
int dqlb200_bind_dynamics_state(dqlb200_handle* h, void* dynamics_state);

/* Replaces: env.reset() for every env + a fresh TrainingMdp (PKG/landing_simulation_env.py:167-243,
 * PKG/trainer.py:176-189).  Sets every population to working step `initial_step`, t = 0. */
int dqlb200_reset(dqlb200_handle* h, int initial_step, void* stream);

/* Replaces: the `while not done` body of Trainer.curriculum_training for every env, k_steps times
 * (PKG/trainer.py:191-245): guess -> continuous_action -> [stand-in physics] -> discrete_state ->
 * check -> reward -> alpha -> update -> auto-reset -> success window / promotion / transfer.
 * trace may be NULL. */
int dqlb200_train(dqlb200_handle* h, int k_steps, const dqlb200_trace* trace, void* stream);

/* Same with HOST buffers (pinned): copies env_state / tables / pop_state in, runs k_steps, copies them back and synchronises.
 * This is the end-to-end call bench.py times as `e2e`.  The call is pipelined over 8 chunks of populations (DQLB200_HOST_CHUNKS overrides: measurement aid) on internal
 * streams (copy-in of chunk c+1 and copy-out of chunk c-1 overlap the training of chunk c).
 * table_levels: 0 = transfer every table level; L > 0 = only levels 0 .. L-1 of every table row travel (both directions, plus
 * -- in reference transfer mode -- the last level on the way in for populations at step 0, which quirk Q7 reads): the caller's
 * promise that no population needs more (working step w touches levels 0 .. w, a promotion inside the call w + 1).  Refused
 * up front when a working step already exceeds it, reported (DQLB200_ERR_STATE) when a promotion inside the call broke it.
 * Configurations with accel_mode != 0 or dynamics_model != 0 have per-env extension state that must travel too: they are
 * refused here (DQLB200_ERR_ARG) and served by dqlb200_train_host_ext. */
int dqlb200_train_host(dqlb200_handle* h, int k_steps, void* env_state_host, void* tables_host,
                       void* pop_state_host, int table_levels, void* stream);

/* dqlb200_train_host with the per-env extension state of the options (SURVEY.md 8f-3 / 8f-4) travelling beside the env state,
 * chunk by chunk: filter_state_host = [n_envs] x 16 B (accel_mode != 0, the layout of dqlb200_bind_filter_state),
 * dynamics_state_host = [2][n_envs] x 16 B (dynamics_model != 0, the layout of dqlb200_bind_dynamics_state); either may be NULL
 * when its option is off (both NULL: exactly dqlb200_train_host).  The device buffers bound with dqlb200_bind_filter_state /
 * dqlb200_bind_dynamics_state are the staging buffers. */
int dqlb200_train_host_ext(dqlb200_handle* h, int k_steps, void* env_state_host, void* tables_host, void* pop_state_host,
                           void* filter_state_host, void* dynamics_state_host, int table_levels, void* stream);

/* Replaces: scripts/simulation.py:48-63 (+ SimulationLandingEnv.reset/step, SimulationMdp):
 * n_episodes greedy episodes of population `population`'s policy, episode i uses reset draws
 * (env = first_episode + i).  policy: 945-byte action LUT (device) = argmax((Q_a+Q_b)/2) per state.
 * stats_out: device pointer to dqlb200_eval_stats (accumulated, caller zeroes).  trace may be NULL
 * (arrays [max_steps][n_episodes]). */
int dqlb200_eval_greedy(dqlb200_handle* h, int population, const uint8_t* policy, int64_t first_episode,
                        int64_t n_episodes, int working_step, void* stats_out, const dqlb200_trace* trace,
                        int trace_steps, void* stream);

/* Greedy SimulationMdp episodes of EVERY agent's current policy, built on the device from the bound float32 tables, in one
 * launch and without a host round trip per agent.
 *   agents       : agent g is the replica group g*R .. g*R+R-1 (R = replicas_per_population; R = 1: every population is an
 *                  agent), n_agents = n_populations / R.  The group is read through replica g*R: its tables, its
 *                  dqlb200_population_params (Philox key, population_id, platform, axis) and its trainer state.
 *                  dqlb200_train_merged and dqlb200_replica_merge leave all replicas of a group identical; between merges the
 *                  other replicas are not looked at.
 *   policy       : for every state s < curriculum_steps * 189 the FIRST maximum over a of float32 (Q_a[s,a] + Q_b[s,a]) * 0.5f,
 *                  each operation rounded to nearest (the arithmetic of the greedy action in dqlb200_train and
 *                  dqlb200_agent_select, i.e. the policy the agent follows at epsilon = 0); states at and above
 *                  curriculum_steps * 189 act 0.
 *   working_step : w >= 0 evaluates every agent under the cut table of step w; -1 uses each agent's live
 *                  dqlb200_population_state.working_step (read on the device; a finished agent holds curriculum_steps - 1).
 *   episodes     : episode i of agent g uses the reset draw (first_episode + i, 0, reset, population_id) under the Philox key of
 *                  replica g*R, so agent g's episodes are, one for one, those of dqlb200_eval_greedy(population = g*R, policy =
 *                  its float32 LUT, first_episode, n_episodes = episodes_per_agent, working_step = w).  With accel_mode /
 *                  dynamics_model every episode starts a fresh simulator, as there.
 *   stats_out    : device dqlb200_eval_stats[n_agents], accumulated (the caller zeroes), exact integer counts.
 *   policy_out   : nullable, device uint8 [n_agents][DQLB200_MAX_CURRICULUM * DQLB200_STATES_PER_LEVEL]: the LUT evaluated.
 * Nothing bound is written: env state, tables, trainer state and the option buffers are only read (or not read at all).
 * Refused: working_step < -1 or >= curriculum_steps, stats_out NULL (DQLB200_ERR_ARG); tables or trainer state not bound, an
 * option without its bound buffer (DQLB200_ERR_STATE).  episodes_per_agent <= 0 does nothing. */
int dqlb200_eval_agents(dqlb200_handle* h, int working_step, int64_t first_episode, int64_t episodes_per_agent,
                        void* stats_out, uint8_t* policy_out, void* stream);

/* dqlb200_eval_agents under each of a LIST of platform motions, in one launch: agents x platforms x episodes from the live
 * float32 tables, for how an agent lands at platform speeds and amplitudes it was not trained on.
 *   platforms_host : host dqlb200_platform[n_platforms].  Copied into a library-owned host buffer and from there to a
 *                    library-owned device buffer on `stream`: the list (pageable or pinned) is never read after the call
 *                    returns, so the caller may rewrite it at once.
 *   cell (g, c)    : agent g (as in dqlb200_eval_agents: replica g*R, its tables, Philox key, population_id, signed g / axis and
 *                    live or given working step) flying platform c: only dphase, r, rw, rw2 of its dqlb200_population_params
 *                    are replaced.  Row (g, c) is, episode for episode, dqlb200_eval_greedy(population = g*R, <g's float32
 *                    first-max LUT>, first_episode, episodes_per_agent, working_step) on a handle whose population g*R has
 *                    platform c.  The reset draw does not depend on the platform, so episode i starts from the same x offset
 *                    and platform phase (in turns) under every platform: differences between columns are differences of
 *                    platform motion alone.  With accel_mode / dynamics_model every episode starts a fresh simulator.
 *   stats_out      : device dqlb200_eval_stats[n_agents][n_platforms], agent-major, accumulated (the caller zeroes).
 * Nothing bound is written.  dqlb200_eval_agents is this call with each agent's own platform.
 * Refused (DQLB200_ERR_ARG): a NULL handle, platforms_host or stats_out; n_platforms < 1; a platform whose r is not finite or
 * <= 0, or whose rw / rw2 is not finite or < 0; working_step outside -1 .. curriculum_steps - 1; more than 0x7FFFFFFF blocks
 * (ceil(episodes_per_agent / 256) * n_agents * n_platforms).  Tables or trainer state not bound, an option without its bound
 * buffer: DQLB200_ERR_STATE.  episodes_per_agent <= 0 does nothing. */
int dqlb200_eval_agents_platforms(dqlb200_handle* h, int working_step, int64_t first_episode, int64_t episodes_per_agent,
                                  const dqlb200_platform* platforms_host, int n_platforms, void* stats_out, void* stream);

/* Un-fused environment entry points: the gym surface of the reference with caller-supplied actions, no agent, no table.
 *   dqlb200_env_reset  replaces TrainingLandingEnv.reset / SimulationLandingEnv.reset (PKG/landing_simulation_env.py:167-243,
 *                      327-400) + mdp.reset() for the envs whose mask byte is non-zero (mask NULL = all).  fresh_mdp != 0 also
 *                      clears what only a NEW TrainingMdp clears (shaping memory, quirk Q11; episode index).  birth = Philox
 *                      counter word 1 of the reset draws.  out_state (nullable): the state of EVERY env after the call.
 *   dqlb200_env_step   replaces TrainingLandingEnv.step (PKG/landing_simulation_env.py:245-282: continuous_action -> physics
 *                      -> discrete_state -> check -> reward) for every env; actions: int8 [n_envs_total].  auto_reset != 0 starts
 *                      the next episode of a finished env inside the call (birth t + 1, like dqlb200_train); simulation != 0
 *                      selects SimulationMdp semantics (v_z = -0.4, no goal logic, reward 0, PKG/mdp.py:784-877).  Outputs
 *                      (all nullable, device, [n_envs_total]): state after the step (auto_reset: of a finished env the first state of
 *                      its next episode), float64 reward, CheckResult code, done,
 *                      obs [..][5], "Number of steps", "Cumulative reward" (without this step's reward, quirk Q12), and
 *                      out_next_state: the state the step ENDED in (differs from out_state only for an auto-reset env).
 * Both work on the bound env_state; they neither read nor write tables or trainer state. */
int dqlb200_env_reset(dqlb200_handle* h, int working_step, uint32_t birth, const uint8_t* mask, int fresh_mdp, int simulation,
                      uint16_t* out_state, void* stream);
int dqlb200_env_step(dqlb200_handle* h, int working_step, uint32_t t, const int8_t* actions, int auto_reset, int simulation,
                     uint16_t* out_state, double* out_reward, uint8_t* out_code, uint8_t* out_done, float* out_obs,
                     uint32_t* out_steps, double* out_cumulative, uint16_t* out_next_state, void* stream);

/* Un-fused agent entry points on the bound float32 tables (batched DoubleQLearningAgent.guess / update with the trainer's
 * schedules; PKG/double_q_learning.py:91-146, PKG/trainer.py:88-126, 191-209):
 *   dqlb200_agent_select  for every env: epsilon-greedy action of its CURRENT state (read from the bound env state, like its
 *                         per-curriculum-step episode index that drives epsilon): greedy = first max of (Q_a + Q_b) / 2; both
 *                         draws of guess() come from Philox (env, t, step, population) -- the draws dqlb200_train uses at global
 *                         step t.  out_actions uint8 [n_envs_total]; out_states (nullable) the states acted on.
 *   dqlb200_agent_update  count[sa] += 1; Q_a[sa] += alpha(count before) * (r + (gamma * max_a' Q_a[s'][a']) * [p-bin changed]
 *                         - Q_a[sa]) for every env, applied per population in env-index order against the bootstrap values of the
 *                         tables as they were when the call started (the "S1" semantics of dqlb200_train, DESIGN.md section 3).
 * A loop of agent_select -> env_step(auto_reset) -> agent_update leaves tables and env state bit-identical to dqlb200_train
 * (tests/test_gpu_facade.py); promotion / transfer stay with the caller (dqlb200_transfer). */
int dqlb200_agent_select(dqlb200_handle* h, int working_step, uint32_t t, uint8_t* out_actions, uint16_t* out_states, void* stream);
int dqlb200_agent_update(dqlb200_handle* h, const uint16_t* states, const uint8_t* actions, const uint16_t* next_states,
                         const double* rewards, void* stream);

/* Replaces: scripts/simulation.py:48-63 with BOTH agents acting (agent_x.predict / agent_y.predict,
 * SimulationMdp.discrete_state_x/_y PKG/mdp.py:634-782, check :784-845 incl. FLYZONE_Y and contact on both axes).
 * policy_x / policy_y: 945-byte action LUTs (device).  Episode i uses the reset draws of (env = first_episode + i,
 * stream p->stream_id).  stats_out: device dqlb200_eval_stats (accumulated, caller zeroes). */
int dqlb200_eval_greedy_2d(dqlb200_handle* h, const dqlb200_eval2d_params* p, const uint8_t* policy_x,
                           const uint8_t* policy_y, int64_t first_episode, int64_t n_episodes, void* stats_out,
                           const dqlb200_trace2d* trace, int trace_steps, void* stream);

/* dqlb200_eval_greedy_2d for MANY (x agent, y agent) pairs at once, each pair's two LUTs built on the device from the bound
 * float32 tables: one launch, no host round trip per pair.
 *   pairs_host   : host int32 [n_pairs][2] = (gx, gy), agent indices 0 .. n_populations / R - 1 (R = replicas_per_population;
 *                  agent g is the replica group g*R .. g*R+R-1, read through replica g*R: its tables, its axis, its trainer
 *                  state).  The list is validated on the host, copied into a library-owned host buffer and from there to a
 *                  library-owned device buffer on `stream`: pairs_host (pageable or pinned) is never read after the call
 *                  returns, so the caller may reuse it at once.  An agent may appear in any number of pairs.
 *   x LUT        : for every state s < curriculum_steps * 189 the FIRST maximum over a of float32 (Q_a[s,a] + Q_b[s,a]) * 0.5f
 *                  of agent gx, each operation rounded to nearest (the policy dqlb200_eval_agents evaluates); gx must be an
 *                  x-axis agent (dqlb200_population_params.axis 0).
 *   y LUT        : gy a y-axis agent (axis 1): its own float32 first-max LUT.  gy an x-axis agent: the mirror image of its
 *                  float32 LUT, lut_y[s] = {1,0,2}[lut(rest*7 + 6 - theta)] with rest, theta = divmod(s, 7) (the rule of
 *                  engine.mirrored_policy: the state with the mirrored angle index, increase and decrease swapped), so one
 *                  agent trained on x flies both axes as the reference's scripts/simulation.py does.
 *                  States at and above curriculum_steps * 189 act 0 on both axes.
 *   p            : platform, gravity signs, y options and the Philox key (seed, stream_id) of the whole launch: every pair
 *                  sees the same episodes' initial conditions, so differences between pairs are differences of policy.
 *                  p->working_step >= 0 evaluates every pair under the cut table of that step; -1 (allowed here only) takes
 *                  the lower of the two members' live dqlb200_population_state.working_step, read on the device and clamped
 *                  to 0 .. curriculum_steps - 1.
 *   episodes     : episode i of pair k is, one for one, episode first_episode + i of dqlb200_eval_greedy_2d(p, lut_x, lut_y)
 *                  with that pair's LUTs and working step.
 *   stats_out    : device dqlb200_eval_stats[n_pairs], accumulated (the caller zeroes), exact integer counts.
 * Nothing bound is written: env state, tables and trainer state are only read.
 * Refused (DQLB200_ERR_ARG): a NULL handle, p, pairs_host or stats_out; n_pairs < 1; an agent index out of range; an x member
 * that is a y-axis agent; trajectory outside 0..2; working_step outside -1 .. curriculum_steps - 1; accel_mode != 0 or
 * dynamics_model != 0 (as dqlb200_eval_greedy_2d); more than 0x7FFFFFFF blocks.  Tables or trainer state not bound:
 * DQLB200_ERR_STATE.  episodes_per_pair <= 0 does nothing. */
int dqlb200_eval_pairs(dqlb200_handle* h, const dqlb200_eval2d_params* p, const int32_t* pairs_host, int n_pairs,
                       int64_t first_episode, int64_t episodes_per_pair, void* stats_out, void* stream);

/* Replaces: DoubleQLearningAgent.transfer_learning (PKG/double_q_learning.py:77-89) on the bound
 * tables of every population. */
int dqlb200_transfer(dqlb200_handle* h, int step, float ratio, void* stream);

/* Checks the error flags the kernels raise where the reference raises ValueError (NaN observation PKG/mdp.py:170, empty state
 * :353, missing previous state :442-452): ONE reduction launch over the populations' flags and ONE 12-byte copy, then a stream
 * synchronisation.  DQLB200_ERR_DEVICE_FLAG names the first offending population. */
int dqlb200_check_errors(dqlb200_handle* h, void* stream);

/* Shared-table mode (one agent replicated on G devices; one NCCL collective between them).  An "agent" is a group of
 * R = cfg.replicas_per_population consecutive populations (R = 1: one population; R > 1: call dqlb200_replica_merge first, so
 * that the R local copies agree).  snapshot holds ONE [3][DQLB200_MAX_CELLS] entry per agent (the tables of the last sync),
 * packed ONE entry of DQLB200_SHARED_WORDS 32-bit words per agent.
 *   pack  : packed <- [ Q_a bits | count | successes in the windows, finished episodes (lo, hi), alive ]   (raw words, integers)
 *   ...   the caller ALL-GATHERS packed over the ranks (torch.distributed.all_gather_into_tensor / ncclAllGather) into
 *         gathered[n_ranks][n_agents][DQLB200_SHARED_WORDS] ...
 *   apply : the all-reduce proper, in RANK ORDER: dcount_g = count_g - count_snap; Q_a <- Q_snap + sum_g (Q_g - Q_snap) * dcount_g
 *           / sum_g dcount_g (float32, one defined order), count <- count_snap + sum_g dcount_g (exact 64-bit sum, saturating
 *           at 2^32 - 1) in every local replica, the shared snapshot and the bound merge snapshot; a cell ONE rank visited takes
 *           that rank's value bit for bit on every rank (so G = 1 never alters a table).  The result is identical on every
 *           rank and from run to run, for any number of visits per sync.  With pooled_promote_successes > 0 the promotion /
 *           max_num_episodes decision (PKG/trainer.py:219-245) is taken from the integer counters summed over all ranks and
 *           armed in every local replica (it takes effect at the next dqlb200_train); pass the threshold for G * R * window_len
 *           episodes, and 0 to dqlb200_replica_merge so that no rank decides alone.
 * Replaces nothing in the reference (it has one process); the merge rule is the replica-merge rule below with ranks as replicas. */
int dqlb200_shared_pack(dqlb200_handle* h, void* packed, void* stream);
int dqlb200_shared_apply(dqlb200_handle* h, void* snapshot, const void* gathered, int n_ranks, int pooled_promote_successes, void* stream);
/* The whole exchange as ONE call for a caller that holds an NCCL communicator (SURVEY.md 8b: allreduce_tables(h, ncclComm_t,
 * stream)): dqlb200_replica_merge on the bound merge snapshot (R > 1 only; with replica_promote_successes, or 0 when a pooled
 * threshold is given: no rank decides alone) -> dqlb200_shared_pack -> ncclAllGather(packed -> gathered, n_agents *
 * DQLB200_SHARED_WORDS int32 per rank) on `stream` -> dqlb200_shared_apply.  nccl_comm is the caller's ncclComm_t (passed as
 * void*: this header does not include nccl.h), n_ranks its size; packed: [n_agents][DQLB200_SHARED_WORDS] words, gathered:
 * n_ranks times that.  NCCL is resolved at run time (dlsym on the process, then libnccl.so.2): the library itself does not link
 * against it, and the call fails with DQLB200_ERR_STATE when it cannot be found.  In Python the same sequence is
 * parallel.SharedTableSync.sync (torch.distributed all-gather between the two C calls). */
int dqlb200_shared_sync_nccl(dqlb200_handle* h, void* snapshot, void* packed, void* gathered, void* nccl_comm, int n_ranks,
                             int replica_promote_successes, int pooled_promote_successes, void* stream);

/* Replica-merge mode (one agent with more envs than one CTA can hold: BASELINE configs 2-3, "N envs sharing one
 * Q-table pair").  The agent's envs are split over R = cfg.replicas_per_population consecutive populations (replicas),
 * each running the S1 semantics on its own table copy; this call merges the R copies of every group into one table
 * and writes it back to all replicas and to `snapshot` ([n_groups][3][DQLB200_MAX_CELLS] words, the merged tables of
 * the previous call; initialise it with the starting tables):
 *     dcount_r = count_r - count_snap,  Q <- Q_snap + sum_r (Q_r - Q_snap) * dcount_r / sum_r dcount_r  (replica order,
 *     fp32),  count <- count_snap + sum_r dcount_r;  a cell only one replica visited keeps that replica's value.
 * It also pools the replicas' success windows: when sum(window_sum) >= pooled_promote_successes or the group's finished
 * episodes reach max_num_episodes, every replica gets pending_advance set and performs transfer + fresh restart at
 * the start of its next dqlb200_train launch (PKG/trainer.py:232-245).  With R = 1 the tables are left untouched.
 * The curriculum transfer (PKG/double_q_learning.py:77-89) acts on the merged table: every replica applies it to its copy
 * and the first replica of a group applies it to the bound snapshot, which therefore has to be registered with
 * dqlb200_bind_merge_snapshot before the first dqlb200_train launch of a replicated layout (NULL unbinds). */
int dqlb200_bind_merge_snapshot(dqlb200_handle* h, void* snapshot);
int dqlb200_replica_merge(dqlb200_handle* h, void* snapshot, int pooled_promote_successes, void* stream);
/* total_steps global steps with a replica merge after every `merge_every` of them (the loop Trainer.curriculum_training runs
 * in replica-merge mode), submitted from C: the (train launch, merge) pair is captured ONCE as a CUDA graph and replayed on
 * an internal stream that is ordered after / before `stream` by events.  Equivalent to alternating dqlb200_train(h,
 * merge_every) and dqlb200_replica_merge on the bound merge snapshot. */
int dqlb200_train_merged(dqlb200_handle* h, int total_steps, int merge_every, int pooled_promote_successes, void* stream);

/* Facade kernels behind TrainingMdp / SimulationMdp / DoubleQLearningAgent single-object calls
 * (float64 observations from the host, reference comparisons in float64; PKG/mdp.py:257-541).
 * obs: [n][6] doubles rel_p, rel_v, rel_a, pitch, z, rel_p_y; contact [n]; action [n];
 * mdp_state: [n] records of 12 doubles {theta_sp, phi_p, phi_v, phi_theta, cumulative_reward,
 * step_count, curriculum_check, result_code, cur_state(-1 none), prev_state(-1 none), rel_p, rel_v};
 * out_state [n] uint16; out_code [n] uint8; out_reward [n] double.  `ops` is an OR of DQLB200_OP_*,
 * applied in the order RESET, ACTION, OBSERVE, CHECK, REWARD.  All pointers are device pointers. */
#define DQLB200_OP_ACTION 1    /* continuous_action   (PKG/mdp.py:543-560) */
#define DQLB200_OP_OBSERVE 2   /* discrete_state      (PKG/mdp.py:257-333) */
#define DQLB200_OP_CHECK 4     /* check               (PKG/mdp.py:335-439 / 784-845) */
#define DQLB200_OP_REWARD 8    /* reward              (PKG/mdp.py:441-541) */
#define DQLB200_OP_RESET 16    /* reset               (PKG/mdp.py:562-569 / 879-886) */
#define DQLB200_OP_SIMULATION 256   /* SimulationMdp semantics instead of TrainingMdp */
int dqlb200_mdp_facade_step(dqlb200_handle* h, int working_step, int ops, int64_t n,
                            const double* obs, const uint8_t* contact, const int8_t* action,
                            double* mdp_state, uint16_t* out_state, uint8_t* out_code, double* out_reward,
                            void* stream);

/* Measurement aid (SURVEY.md 8d, "atomic roof"): replays a recorded sequence of visited table cells with UNORDERED
 * shared-memory atomics -- per visit one red.shared.add.f32 on Q_a[cell] and one red.shared.add.u32 on count[cell], i.e.
 * the two read-modify-writes of one Q update (PKG/double_q_learning.py:100,145) -- from `blocks` CTAs of `threads`
 * threads, each thread `visits_per_thread` visits, tables in shared memory like train_kernel.  cells: device uint16
 * [n_cells] (cell = state id * 3 + action, exported from a traced training run).  checksum_out: device uint64 (keeps the
 * work alive).  The caller times the launch with CUDA events: visits / time = the rate an unordered-atomics design could
 * not exceed for the table update alone; train_kernel's ordered commit is compared against it in bench.py. */
int dqlb200_bench_table_rmw(dqlb200_handle* h, const uint16_t* cells, int64_t n_cells, int visits_per_thread, int threads,
                            int blocks, void* checksum_out, void* stream);

/* Measurement aid: launches an empty kernel with train_kernel's launch shape (grid, block, dynamic shared memory, by-value
 * parameter block); timed by the caller to separate the cost of launching from the cost of the work. */
int dqlb200_bench_launch_floor(dqlb200_handle* h, int blocks, int threads, int smem_bytes, void* stream);

/* Device self-test: the 3-instruction float64 division used for fp32 numerators (x / p_max, x / v_max) against
 * the IEEE division for every finite fp32 bit pattern; mismatches_out[0] = wrong quotients of the production
 * routine (must be 0), [1] = of the one-correction-step variant (diagnostic), [2] = of the float64-numerator
 * routine used for x / theta_max on 2^32 pseudo-random numerators (must be 0).  Synchronises. */
int dqlb200_selftest_division(dqlb200_handle* h, uint64_t* mismatches_out, void* stream);

/* Device self-test of the fp32 cut-table discretisation (R5: PKG/mdp.py:149-170, 257-333) on caller-supplied observations.
 * obs: device float [n][4] = rel_p, rel_v, rel_a, pitch; out_state: device uint16 [n] state ids for working step `working_step`.
 * variant selects the instantiation the production kernels use: 0 = run-time constants, level loop bounded by the working step
 * (generic train_kernel, env_step_kernel); 1 = compile-time constants + cut table in shared memory (production train_kernel;
 * needs the reference-default configuration); 2 / 3 = the same two with every level index probed (eval kernels, env reset).
 * tests/test_gpu_parity.py feeds it every probe of tests/golden/discretise.npz (+-3 ulp around every threshold). */
int dqlb200_selftest_discretise(dqlb200_handle* h, int working_step, int variant, int64_t n, const float* obs, uint16_t* out_state,
                                void* stream);

/* Facade kernel behind single-object DoubleQLearningAgent calls, float64 like the reference's tables
 * (PKG/double_q_learning.py:38-40).  tables_f64: device [3][DQLB200_MAX_CELLS] doubles (Q_a, Q_b, count).
 *   DQLB200_AGENT_PREDICT : out_action[i] = argmax((Q_a[s_i] + Q_b[s_i]) / 2)          (PKG/double_q_learning.py:119-124)
 *   DQLB200_AGENT_UPDATE  : for i in order: count[sa_i] += 1; Q_a[sa_i] += alpha_i * (reward_i + (gamma * max Q_a[s'_i])
 *                           * [p-bin changed] - Q_a[sa_i])                               (PKG/double_q_learning.py:91-108,126-146)
 *   DQLB200_AGENT_TRANSFER: Q_{a,b}[step] = Q_{a,b}[src] * ratio  (step = state[0], ratio = alpha[0], src = next_state[0] = (step - 1)
 *                           modulo the AGENT's curriculum_steps, so that step 0 reads its last slot like Q[-1]; :77-89)
 * state / next_state are state ids (< 945), action in 0..2; all pointers are device pointers. */
#define DQLB200_AGENT_PREDICT 1
#define DQLB200_AGENT_UPDATE 2
#define DQLB200_AGENT_TRANSFER 4
int dqlb200_agent_facade(dqlb200_handle* h, int op, int64_t n, double* tables_f64, const int32_t* state,
                         const int32_t* action, const int32_t* next_state, const double* alpha,
                         const double* reward, double gamma, int32_t* out_action, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DQLB200_H */
