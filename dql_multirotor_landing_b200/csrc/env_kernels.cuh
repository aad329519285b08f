// env_kernels.cuh -- reset, greedy evaluation (one and two axes) and the un-fused gym-surface kernels
// Part of libdqlb200 (see dqlb200.cu for the kernel inventory and the C-ABI).
#pragma once
#include "train_kernel.cuh"

namespace dql {

// -------------------------------------------------------------------------------------------------
__global__ void reset_kernel(const __grid_constant__ KC kc, EnvPtrs env, dqlb200_population_state* pop_state,
                             const dqlb200_population_params* pop_params, int initial_step) {
  const int pop = blockIdx.y;
  const int env_i = blockIdx.x * blockDim.x + threadIdx.x;
  __shared__ dqlb200_cuts cuts;
  if (threadIdx.x == 0) cuts = kc.cuts[initial_step];
  __syncthreads();
  if (env_i < kc.envs_per_population) {
    const dqlb200_population_params pp = pop_params[pop];
    Env e;
    Kf kf = kf_initial();       // a new simulator: the only place the estimator and the PID memory are ever cleared
    Ext ex = ext_initial(kc);
    env_reset(kc, pp, cuts, kc.angle_cut, e, (uint32_t)env_i, 0u, initial_step, /*fresh_mdp=*/true, (uint32_t)env.sp_zero, env.d ? &kf : nullptr, env.e ? &ex : nullptr);
    env_store(env, (size_t)pop * kc.envs_per_population + env_i, e);
    if (kc.accel_mode != 0 && env.d) kf_store(env, (size_t)pop * kc.envs_per_population + env_i, kf);
    if (kc.dynamics_model != 0 && env.e) ext_store(env, (size_t)pop * kc.envs_per_population + env_i, ex);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    dqlb200_population_state ps;
    memset(&ps, 0, sizeof(ps));
    ps.working_step = initial_step;
    pop_state[pop] = ps;
  }
}

// -------------------------------------------------------------------------------------------------
// R15: greedy evaluation, SimulationMdp semantics (PKG/mdp.py:784-886, scripts/simulation.py:48-63)
// -------------------------------------------------------------------------------------------------
// One greedy episode of `policy` (a shared-memory LUT): the reset draw of episode `ep`, the SimulationMdp check chain, and the
// optional per-step trace (row `i` of arrays [trace_steps][n_episodes]).  Returns the termination code; `step` = its length.
template <bool GENERIC, class KT>
__device__ __forceinline__ int greedy_episode(const KT& kk, const dqlb200_population_params& pp, const dqlb200_cuts& cuts,
                                              const uint8_t* s_policy, unsigned long long ep, const dqlb200_trace& trace,
                                              int trace_steps, long long i, long long n_episodes, int& step) {
  const uint4 d = philox4x32_10(make_uint4((uint32_t)ep, 0u, PURPOSE_RESET, pp.population_id), pp.seed_lo, pp.seed_hi);
  Body b;
  Kf kf = kf_initial();       // accel_mode != 0: every evaluation episode runs on a freshly started simulator
  Kf* const kfp = (GENERIC && kk.accel_mode != 0) ? &kf : nullptr;
  Ext ex = ext_initial(kk);
  Ext* const exp_ = (GENERIC && kk.dynamics_model != 0) ? &ex : nullptr;
  Obs o = dyn_reset(kk, pp, b, d, /*normal_init=*/false, /*simulation=*/true, kk.dz_sim, kfp, exp_);
  uint32_t sid = (uint32_t)discretise_cuts(cuts, kk.angle_cut, o).id();
  double sp = 0.0;
  int code = DQLB200_NON_TERMINAL;
  step = 0;
  while (code < DQLB200_TERMINAL_SUCCESS) {
    const int a = s_policy[sid];
    sp = apply_action(kk, sp, a);
    dyn_advance(kk, pp, b, (float)sp, kfp, exp_, kk.vz_sim);
    step += 1;
    o = dyn_observe(kk, pp, b, step, kk.dz_sim, kfp, exp_);
    const uint32_t sid2 = (uint32_t)discretise_cuts(cuts, kk.angle_cut, o).id();
    if (o.contact) code = DQLB200_TERMINAL_CONTACT;
    else if (!(o.rel_p >= kk.fz_lo) || (o.rel_p >= kk.fz_hi)) code = DQLB200_TERMINAL_FLYZONE_X;
    else if (!(o.z >= kk.z_min_cut)) code = DQLB200_TERMINAL_MINIMUM_ALTITUDE;
    else if (o.z >= kk.z_max_cut) code = DQLB200_TERMINAL_FLYZONE_Z;
    else if (step >= kk.timeout_steps) code = DQLB200_TERMINAL_TIMEOUT;
    if (step <= trace_steps) {
      const size_t ti = (size_t)(step - 1) * (size_t)n_episodes + (size_t)i;
      if (trace.obs) {
        float* po = trace.obs + ti * 5;
        po[0] = o.rel_p; po[1] = o.rel_v; po[2] = o.rel_a; po[3] = o.pitch; po[4] = o.z;
      }
      if (trace.action) trace.action[ti] = (uint8_t)a;
      if (trace.code) trace.code[ti] = (uint8_t)code;
      if (trace.done) trace.done[ti] = (uint8_t)(code >= DQLB200_TERMINAL_SUCCESS);
      if (trace.contact) trace.contact[ti] = (uint8_t)o.contact;
      if (trace.state) trace.state[ti] = (uint16_t)sid;
      if (trace.next_state) trace.next_state[ti] = (uint16_t)sid2;
    }
    sid = sid2;
  }
  return code;
}

template <bool GENERIC>
__global__ void __launch_bounds__(256) eval_kernel(const __grid_constant__ KC kc, const dqlb200_population_params* pop_params,
                                                   int population, const uint8_t* __restrict__ policy,
                                                   long long first_episode, long long n_episodes, int w,
                                                   dqlb200_eval_stats* stats, dqlb200_trace trace, int trace_steps) {
  const auto& kk = ConstsOf<GENERIC>::get(kc);
  __shared__ uint8_t s_policy[DQLB200_MAX_CURRICULUM * DQLB200_STATES_PER_LEVEL];
  __shared__ dqlb200_cuts cuts;
  __shared__ unsigned int s_hist[9], s_steps, s_eps;      // per-block totals fit 32 bits (256 episodes x 459 steps): native shared atomics, not 64-bit CAS loops
  for (int i = threadIdx.x; i < DQLB200_MAX_CURRICULUM * DQLB200_STATES_PER_LEVEL; i += blockDim.x) s_policy[i] = policy[i];
  if (threadIdx.x == 0) { cuts = kc.cuts[w]; s_steps = s_eps = 0u; }
  if (threadIdx.x < 9) s_hist[threadIdx.x] = 0u;
  __syncthreads();
  const dqlb200_population_params pp = pop_params[population];
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_episodes) {
    int step;
    const int code = greedy_episode<GENERIC>(kk, pp, cuts, s_policy, (unsigned long long)(first_episode + i), trace, trace_steps, i, n_episodes, step);
    atomicAdd(&s_hist[code], 1u);
    atomicAdd(&s_steps, (unsigned int)step);
    atomicAdd(&s_eps, 1u);
  }
  __syncthreads();
  if (threadIdx.x < 9 && s_hist[threadIdx.x]) atomicAdd((unsigned long long*)&stats->termination_hist[threadIdx.x], (unsigned long long)s_hist[threadIdx.x]);
  if (threadIdx.x == 0) {
    atomicAdd((unsigned long long*)&stats->steps, (unsigned long long)s_steps);
    atomicAdd((unsigned long long*)&stats->episodes, (unsigned long long)s_eps);
  }
}

// Greedy action of state s from float32 tables: the first maximum of (Q_a + Q_b) * 0.5f over the actions in order, each operation
// rounded to nearest -- the arithmetic of build_snapshot (train_kernel) and agent_select_kernel.
__device__ __forceinline__ uint8_t greedy_action_f32(const float* __restrict__ qa, const float* __restrict__ qb, int s) {
  const float p0 = fmul(fadd(qa[s * 3 + 0], qb[s * 3 + 0]), 0.5f);
  const float p1 = fmul(fadd(qa[s * 3 + 1], qb[s * 3 + 1]), 0.5f);
  const float p2 = fmul(fadd(qa[s * 3 + 2], qb[s * 3 + 2]), 0.5f);
  int a = 0;
  float best = p0;
  if (p1 > best) { best = p1; a = 1; }
  if (p2 > best) { a = 2; }
  return (uint8_t)a;
}

// Every agent's greedy policy in one launch: blocks_per_agent blocks of 256 episodes per agent on a flat 1-D grid (agent =
// blockIdx.x / blocks_per_agent).  Agent g reads replica g * replicas: its tables (the LUT is built per block in shared memory),
// Philox key, platform and -- for w < 0 -- its live working step.  Episode i of agent g is episode first_episode + i of
// eval_kernel for population g * replicas under the same LUT.  Reads the tables and trainer state, writes only stats / policy_out.
template <bool GENERIC>
__global__ void __launch_bounds__(256) eval_agents_kernel(const __grid_constant__ KC kc, const dqlb200_population_params* pop_params,
                                                          const uint32_t* __restrict__ tables, const dqlb200_population_state* __restrict__ pop_state,
                                                          int replicas, int blocks_per_agent, long long first_episode,
                                                          long long episodes_per_agent, int w, dqlb200_eval_stats* stats,
                                                          uint8_t* __restrict__ policy_out) {
  const auto& kk = ConstsOf<GENERIC>::get(kc);
  constexpr int N_STATES = DQLB200_MAX_CURRICULUM * DQLB200_STATES_PER_LEVEL;
  __shared__ uint8_t s_policy[N_STATES];
  __shared__ dqlb200_cuts cuts;
  __shared__ unsigned int s_hist[9], s_steps, s_eps;
  const int agent = (int)(blockIdx.x / (unsigned)blocks_per_agent);
  const int block_in_agent = (int)(blockIdx.x - (unsigned)agent * (unsigned)blocks_per_agent);
  const int pop = agent * replicas;
  const float* qa = reinterpret_cast<const float*>(tables + (size_t)pop * 3 * DQLB200_MAX_CELLS);
  const float* qb = qa + DQLB200_MAX_CELLS;
  const int live_states = kc.curriculum_steps * DQLB200_STATES_PER_LEVEL;
  for (int s = threadIdx.x; s < N_STATES; s += blockDim.x) s_policy[s] = s < live_states ? greedy_action_f32(qa, qb, s) : (uint8_t)0;
  if (threadIdx.x == 0) {
    const int wl = w >= 0 ? w : min(max(pop_state[pop].working_step, 0), kc.curriculum_steps - 1);      // clamped: never index past cuts[]
    cuts = kc.cuts[wl];
    s_steps = s_eps = 0u;
  }
  if (threadIdx.x < 9) s_hist[threadIdx.x] = 0u;
  __syncthreads();
  if (policy_out && block_in_agent == 0)
    for (int s = threadIdx.x; s < N_STATES; s += blockDim.x) policy_out[(size_t)agent * N_STATES + s] = s_policy[s];
  const dqlb200_population_params pp = pop_params[pop];
  const long long i = (long long)block_in_agent * blockDim.x + threadIdx.x;
  if (i < episodes_per_agent) {
    int step;
    const dqlb200_trace no_trace = {};
    const int code = greedy_episode<GENERIC>(kk, pp, cuts, s_policy, (unsigned long long)(first_episode + i), no_trace, 0, i, episodes_per_agent, step);
    atomicAdd(&s_hist[code], 1u);
    atomicAdd(&s_steps, (unsigned int)step);
    atomicAdd(&s_eps, 1u);
  }
  __syncthreads();
  dqlb200_eval_stats* st = stats + agent;
  if (threadIdx.x < 9 && s_hist[threadIdx.x]) atomicAdd((unsigned long long*)&st->termination_hist[threadIdx.x], (unsigned long long)s_hist[threadIdx.x]);
  if (threadIdx.x == 0) {
    atomicAdd((unsigned long long*)&st->steps, (unsigned long long)s_steps);
    atomicAdd((unsigned long long*)&st->episodes, (unsigned long long)s_eps);
  }
}

// -------------------------------------------------------------------------------------------------
// Un-fused environment entry points (the gym surface of the reference: TrainingLandingEnv / SimulationLandingEnv reset()
// and step(), PKG/landing_simulation_env.py:167-282, 327-400): the caller supplies the actions, no agent, no table.  Same
// device functions and the same operation order as phase A of train_kernel; tests/test_gpu_facade.py holds the two
// bit-identical (a traced train launch with forced actions == a sequence of env steps).
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) env_reset_kernel(const __grid_constant__ KC kc, EnvPtrs env, const dqlb200_population_params* pop_params,
                                                        int w, uint32_t birth, const uint8_t* __restrict__ mask, int fresh_mdp, int simulation,
                                                        uint16_t* out_state) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long n_total = (long long)kc.n_populations * kc.envs_per_population;
  if (i >= n_total) return;
  Env e;
  env_load(env, (size_t)i, e);
  const bool filt = kc.accel_mode != 0 && env.d;
  const bool so = kc.dynamics_model != 0 && env.e;
  Kf kf;
  Ext ex;
  if (filt) kf = kf_load(env, (size_t)i);
  if (so) ex = ext_load(env, (size_t)i);
  if (!mask || mask[i]) {
    const int pop = (int)(i / kc.envs_per_population);
    const uint32_t env_i = (uint32_t)(i % kc.envs_per_population);
    const dqlb200_population_params pp = pop_params[pop];
    if (simulation) {      // SimulationLandingEnv.reset (PKG/landing_simulation_env.py:327-340) + SimulationMdp.reset (PKG/mdp.py:879-886)
      const uint4 d = philox4x32_10(make_uint4(env_i, birth, PURPOSE_RESET, pp.population_id), pp.seed_lo, pp.seed_hi);
      const Obs o = dyn_reset(kc, pp, e.b, d, /*normal_init=*/false, /*simulation=*/true, kc.dz_sim, filt ? &kf : nullptr, so ? &ex : nullptr);
      const DState ds = discretise_cuts(kc.cuts[w], kc.angle_cut, o);
      e.sid = (uint32_t)ds.id(); e.bp = (uint32_t)ds.bp;
      e.step_count = 0; e.curriculum_check = 0; e.sticky_success = false; e.fresh = true; e.cum_reward = 0.0;
      e.sp_idx = (uint32_t)env.sp_zero; e.prev_rel_p = 0.0f; e.prev_rel_v = 0.0f;
      if (fresh_mdp) e.episode = 0;
    } else {
      env_reset(kc, pp, kc.cuts[w], kc.angle_cut, e, env_i, birth, w, fresh_mdp != 0, (uint32_t)env.sp_zero, filt ? &kf : nullptr, so ? &ex : nullptr);
    }
    env_store(env, (size_t)i, e);
    if (filt) kf_store(env, (size_t)i, kf);
    if (so) ext_store(env, (size_t)i, ex);
  }
  if (out_state) out_state[i] = (uint16_t)e.sid;
}

template <bool DIV2>
__global__ void __launch_bounds__(128) env_step_kernel(const __grid_constant__ KC kc, EnvPtrs env, const dqlb200_population_params* pop_params,
                                                       int w, uint32_t t, const int8_t* __restrict__ actions, int auto_reset, int simulation,
                                                       uint16_t* out_state, double* out_reward, uint8_t* out_code, uint8_t* out_done,
                                                       float* out_obs, uint32_t* out_steps, double* out_cumulative, uint16_t* out_next_state, uint32_t* error_flag) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long n_total = (long long)kc.n_populations * kc.envs_per_population;
  if (i >= n_total) return;
  const int pop = (int)(i / kc.envs_per_population);
  const uint32_t env_i = (uint32_t)(i % kc.envs_per_population);
  const dqlb200_population_params pp = pop_params[pop];
  const dqlb200_cuts& cuts = kc.cuts[w];
  Env e;
  env_load(env, (size_t)i, e);
  const bool filt = kc.accel_mode != 0 && env.d;
  const bool so = kc.dynamics_model != 0 && env.e;
  Kf kf;
  Ext ex;
  if (filt) kf = kf_load(env, (size_t)i);
  if (so) ex = ext_load(env, (size_t)i);
  const int a = actions[i];
  // R3 .. R8 in the order of TrainingLandingEnv.step (PKG/landing_simulation_env.py:245-282)
  // R3 through the set-point tables (the memoised float64 arithmetic of continuous_action, see dqlb200_config)
  const double prev_sp = env.sp_value[e.sp_idx];
  const uint32_t sp_new = env.sp_next[(e.fresh ? (uint32_t)env.sp_zero : e.sp_idx) * 3u + (uint32_t)a].x;
  const double sp = env.sp_value[sp_new];
  dyn_advance(kc, pp, e.b, (float)sp, filt ? &kf : nullptr, so ? &ex : nullptr, simulation ? kc.vz_sim : kc.vz_train);
  const uint32_t step_count = e.step_count + 1u;
  Obs o = dyn_observe(kc, pp, e.b, (int)step_count, simulation ? kc.dz_sim : kc.dz_train, filt ? &kf : nullptr, so ? &ex : nullptr);
  if (kc.noise_enabled && !simulation) {      // the words the fused kernel uses at global step t
    const uint4 d = philox4x32_10(make_uint4(env_i, t, PURPOSE_STEP, pp.population_id), pp.seed_lo, pp.seed_hi);
    add_observation_noise(kc, o, d.z, d.w);
  }
  const DState ds = discretise_cuts(cuts, kc.angle_cut, o, w);
  const uint32_t sid2 = (uint32_t)ds.id();
  const bool t_fx = !(o.rel_p >= kc.fz_lo) || (o.rel_p >= kc.fz_hi);
  const bool t_zmin = !(o.z >= kc.z_min_cut), t_zmax = o.z >= kc.z_max_cut;
  const bool t_time = (int)step_count >= kc.timeout_steps;
  const bool goal_bins = !simulation && !(o.contact || t_fx || t_zmin || t_zmax || t_time) && ds.bp == 1 && ds.bv == 1;
  const bool at_level = e.sid >= (uint32_t)(w * DQLB200_STATES_PER_LEVEL) && ds.level == w;
  const uint32_t cc = goal_bins ? (at_level ? e.curriculum_check + 1u : 0u) : e.curriculum_check;
  int code = e.sticky_success ? DQLB200_NON_TERMINAL_SUCCESS : DQLB200_NON_TERMINAL;
  if (goal_bins && at_level) code = ((int)cc >= kc.success_steps) ? DQLB200_TERMINAL_SUCCESS : DQLB200_NON_TERMINAL_SUCCESS;
  code = t_time ? DQLB200_TERMINAL_TIMEOUT : code;
  code = t_zmax ? DQLB200_TERMINAL_FLYZONE_Z : code;
  code = t_zmin ? DQLB200_TERMINAL_MINIMUM_ALTITUDE : code;
  code = t_fx ? DQLB200_TERMINAL_FLYZONE_X : code;
  code = o.contact ? DQLB200_TERMINAL_CONTACT : code;
  const bool done = code >= DQLB200_TERMINAL_SUCCESS;
  if (!(fabsf(o.rel_p) <= 3.4028234664e38f) || !(fabsf(o.rel_v) <= 3.4028234664e38f) || !(fabsf(o.rel_a) <= 3.4028234664e38f))
    atomicOr(error_flag, 1u);
  double r = 0.0;
  if (!simulation) {
    const double phi_p = shaping(kc.w_p, o.rel_p, kc.p_max, kc.rcp_p_max, kc.clip_p_f, DIV2);
    const double phi_v = shaping(kc.w_v, o.rel_v, kc.v_max, kc.rcp_v_max, kc.clip_v_f, DIV2);
    const double phi_t = __dmul_rn(kc.w_theta, fabs(div_f64_by_const(sp, kc.theta_max, kc.rcp_theta_max)));
    const double prev_p = shaping(kc.w_p, e.prev_rel_p, kc.p_max, kc.rcp_p_max, kc.clip_p_f, DIV2);
    const double prev_v = shaping(kc.w_v, e.prev_rel_v, kc.v_max, kc.rcp_v_max, kc.clip_v_f, DIV2);
    const double prev_t = __dmul_rn(kc.w_theta, fabs(div_f64_by_const(prev_sp, kc.theta_max, kc.rcp_theta_max)));
    const bool succ_reward = code == DQLB200_NON_TERMINAL_SUCCESS || code == DQLB200_TERMINAL_SUCCESS;
    r = reward_f64(kc, kc.reward[ds.level], phi_p, phi_v, phi_t, prev_p, prev_v, prev_t, succ_reward);
  }
  if (out_reward) out_reward[i] = r;
  if (out_next_state) out_next_state[i] = (uint16_t)sid2;
  if (out_code) out_code[i] = (uint8_t)code;
  if (out_done) out_done[i] = (uint8_t)done;
  if (out_obs) { float* po = out_obs + i * 5; po[0] = o.rel_p; po[1] = o.rel_v; po[2] = o.rel_a; po[3] = o.pitch; po[4] = o.z; }
  if (out_steps) out_steps[i] = step_count;
  if (out_cumulative) out_cumulative[i] = e.cum_reward;          // quirk Q12: without this step's reward
  e.sp_idx = sp_new;
  e.prev_rel_p = o.rel_p;
  e.prev_rel_v = o.rel_v;
  e.episode += done ? 1u : 0u;
  e.sid = sid2;
  e.bp = (uint32_t)ds.bp;
  e.step_count = step_count;
  e.curriculum_check = cc;
  e.sticky_success = (code == DQLB200_NON_TERMINAL_SUCCESS);
  e.fresh = false;
  e.cum_reward = __dadd_rn(e.cum_reward, r);
  if (done && auto_reset && !simulation) env_reset(kc, pp, cuts, kc.angle_cut, e, env_i, t + 1u, w, /*fresh_mdp=*/false, (uint32_t)env.sp_zero, filt ? &kf : nullptr, so ? &ex : nullptr);
  if (out_state) out_state[i] = (uint16_t)e.sid;       // of a finished env with auto_reset: the first state of its next episode
  env_store(env, (size_t)i, e);
  if (filt) kf_store(env, (size_t)i, kf);
  if (so) ext_store(env, (size_t)i, ex);
}

// -------------------------------------------------------------------------------------------------
// SURVEY 8f-2: two-axis greedy evaluation.  One thread per episode; pitch drives x, roll drives y (signed gravity per
// axis), one platform under both (three trajectories).  Same operation order as oracle/dynamics.py: StandIn2D.
// -------------------------------------------------------------------------------------------------
struct Axis {
  float pos, vel, ang, acc;
};
template <class KT>
__device__ __forceinline__ void axis_advance(const KT& kc, Axis& b, float sp, float g) {
  b.ang = fadd(b.ang, fmul(fsub(sp, b.ang), kc.k_theta));
  b.acc = fsub(fmul(g, det_tan(b.ang)), fmul(kc.c_d, b.vel));
  b.pos = fadd(fadd(b.pos, fmul(b.vel, kc.h)), fmul(b.acc, kc.half_h2));
  b.vel = fadd(b.vel, fmul(b.acc, kc.h));
}
struct Platform2D {
  float xm, um, axm, ym, vm, aym;
};
__device__ __forceinline__ Platform2D platform_2d(const dqlb200_eval2d_params& p, uint32_t phase_x, uint32_t phase_y) {
  Platform2D m;
  float sx, cx;
  det_sincos_turns(phase_x, sx, cx);
  if (p.trajectory == 2) {
    const float sc = fmul(sx, cx);
    m.xm = fmul(p.r_x, cx); m.um = -fmul(p.rw_x, sx); m.axm = -fmul(p.rw2_x, cx);
    m.ym = fmul(p.r_y, sc); m.vm = fmul(p.rw_y, fsub(fmul(cx, cx), fmul(sx, sx))); m.aym = -fmul(p.rw2_y, sc);
  } else {
    float sy, cy;
    det_sincos_turns(phase_y, sy, cy);
    m.xm = fmul(p.r_x, sx); m.um = fmul(p.rw_x, cx); m.axm = -fmul(p.rw2_x, sx);
    m.ym = fmul(p.r_y, sy); m.vm = fmul(p.rw_y, cy); m.aym = -fmul(p.rw2_y, sy);
  }
  return m;
}

// One greedy two-axis episode of the shared-memory LUTs s_pol_x / s_pol_y: the reset draw of episode `ep` under p's key, the
// hover step, the sub-step loop, both discretisations, the check chain and the optional per-step trace (row `i` of arrays
// [trace_steps][n_episodes]).  Returns the termination code; `step` = its length.
template <class KT>
__device__ __forceinline__ int greedy_episode_2d(const KT& kk, const dqlb200_eval2d_params& p, const dqlb200_cuts& cuts,
                                                 const uint8_t* s_pol_x, const uint8_t* s_pol_y, unsigned long long ep,
                                                 const dqlb200_trace2d& trace, int trace_steps, long long i, long long n_episodes,
                                                 int& step) {
  const uint4 d = philox4x32_10(make_uint4((uint32_t)ep, 0u, PURPOSE_RESET, p.stream_id), p.seed_lo, p.seed_hi);
  // PKG/landing_simulation_env.py:327-340: uniform offsets inside the fly zone, absolute clip, random platform phase
  const float x_init = fadd(-kk.p_max_f, fmul(kk.two_p_max_f, fmul(__uint2float_rn(d.x >> 8), (float)(1.0 / 16777216.0))));
  const float y_init = fadd(-kk.p_max_f, fmul(kk.two_p_max_f, fmul(__uint2float_rn(d.y >> 8), (float)(1.0 / 16777216.0))));
  uint32_t phase_x = d.z, phase_y = (p.trajectory == 2) ? d.z : d.w;
  Platform2D m = platform_2d(p, phase_x, phase_y);
  Axis bx, by;
  bx.pos = clipf(fsub(m.xm, x_init), -kk.p_max_f, kk.p_max_f);
  by.pos = p.y_init_enabled ? clipf(fsub(m.ym, y_init), -kk.p_max_f, kk.p_max_f) : 0.0f;
  bx.vel = bx.ang = bx.acc = by.vel = by.ang = by.acc = 0.0f;
  double sp_x = 0.0, sp_y = 0.0;
  int code = DQLB200_NON_TERMINAL;
  step = -1;
  uint32_t sid_x = 0, sid_y = 0;
  while (code < DQLB200_TERMINAL_SUCCESS) {
    int ax = 255, ay = 255;
    if (step >= 0) {          // step == -1: the hover period after the reset (PKG/landing_simulation_env.py:222-224)
      ax = s_pol_x[sid_x];
      ay = s_pol_y[sid_y];
      sp_x = apply_action(kk, sp_x, ax);
      if (p.y_action_enabled) sp_y = apply_action(kk, sp_y, ay);
    }
    for (int k = 0; k < kk.n_sub; ++k) {
      axis_advance(kk, bx, (float)sp_x, p.g_x);
      axis_advance(kk, by, (float)sp_y, p.g_y);
      phase_x += p.dphase_x;
      phase_y += p.dphase_y;
    }
    step += 1;
    m = platform_2d(p, phase_x, phase_y);
    Obs ox, oy;
    ox.rel_p = fsub(m.xm, bx.pos); ox.rel_v = fsub(m.um, bx.vel); ox.rel_a = fsub(m.axm, bx.acc); ox.pitch = bx.ang;
    oy.rel_p = fsub(m.ym, by.pos); oy.rel_v = fsub(m.vm, by.vel); oy.rel_a = fsub(m.aym, by.acc); oy.pitch = by.ang;
    const float z = fadd(kk.z_init, fmul(__int2float_rn(step), kk.dz_sim));
    const bool contact = (z <= kk.z_touch) && (fabsf(ox.rel_p) <= kk.half_platform) && (fabsf(oy.rel_p) <= kk.half_platform);
    sid_x = (uint32_t)discretise_cuts(cuts, kk.angle_cut, ox).id();
    sid_y = (uint32_t)discretise_cuts(cuts, kk.angle_cut, oy).id();
    if (step == 0) continue;          // the reset only observes (no check, PKG/landing_simulation_env.py:236-243)
    if (contact) code = DQLB200_TERMINAL_CONTACT;
    else if (!(ox.rel_p >= kk.fz_lo) || (ox.rel_p >= kk.fz_hi)) code = DQLB200_TERMINAL_FLYZONE_X;
    else if (!(oy.rel_p >= kk.fz_lo) || (oy.rel_p >= kk.fz_hi)) code = DQLB200_TERMINAL_FLYZONE_Y;
    else if (!(z >= kk.z_min_cut)) code = DQLB200_TERMINAL_MINIMUM_ALTITUDE;
    else if (z >= kk.z_max_cut) code = DQLB200_TERMINAL_FLYZONE_Z;
    else if (step >= kk.timeout_steps) code = DQLB200_TERMINAL_TIMEOUT;
    if (step <= trace_steps) {
      const size_t ti = (size_t)(step - 1) * (size_t)n_episodes + (size_t)i;
      if (trace.obs) {
        float* po = trace.obs + ti * 9;
        po[0] = ox.rel_p; po[1] = ox.rel_v; po[2] = ox.rel_a; po[3] = ox.pitch; po[4] = z;
        po[5] = oy.rel_p; po[6] = oy.rel_v; po[7] = oy.rel_a; po[8] = oy.pitch;
      }
      if (trace.action_x) trace.action_x[ti] = (uint8_t)ax;
      if (trace.action_y) trace.action_y[ti] = (uint8_t)ay;
      if (trace.code) trace.code[ti] = (uint8_t)code;
      if (trace.done) trace.done[ti] = (uint8_t)(code >= DQLB200_TERMINAL_SUCCESS);
      if (trace.contact) trace.contact[ti] = (uint8_t)contact;
      if (trace.state_x) trace.state_x[ti] = (uint16_t)sid_x;
      if (trace.state_y) trace.state_y[ti] = (uint16_t)sid_y;
    }
  }
  return code;
}

template <bool GENERIC>
__global__ void __launch_bounds__(256) eval2d_kernel(const __grid_constant__ KC kc, const __grid_constant__ dqlb200_eval2d_params p,
                                                     const uint8_t* __restrict__ policy_x, const uint8_t* __restrict__ policy_y,
                                                     long long first_episode, long long n_episodes, dqlb200_eval_stats* stats,
                                                     dqlb200_trace2d trace, int trace_steps) {
  const auto& kk = ConstsOf<GENERIC>::get(kc);
  __shared__ uint8_t s_pol_x[DQLB200_MAX_CURRICULUM * DQLB200_STATES_PER_LEVEL], s_pol_y[DQLB200_MAX_CURRICULUM * DQLB200_STATES_PER_LEVEL];
  __shared__ dqlb200_cuts cuts;
  __shared__ unsigned int s_hist[9], s_steps, s_eps;      // per-block totals fit 32 bits (256 episodes x 459 steps): native shared atomics, not 64-bit CAS loops
  for (int i = threadIdx.x; i < DQLB200_MAX_CURRICULUM * DQLB200_STATES_PER_LEVEL; i += blockDim.x) {
    s_pol_x[i] = policy_x[i];
    s_pol_y[i] = policy_y[i];
  }
  if (threadIdx.x == 0) { cuts = kc.cuts[p.working_step]; s_steps = s_eps = 0u; }
  if (threadIdx.x < 9) s_hist[threadIdx.x] = 0u;
  __syncthreads();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_episodes) {
    int step;
    const int code = greedy_episode_2d(kk, p, cuts, s_pol_x, s_pol_y, (unsigned long long)(first_episode + i), trace, trace_steps, i,
                                       n_episodes, step);
    atomicAdd(&s_hist[code], 1u);
    atomicAdd(&s_steps, (unsigned int)step);
    atomicAdd(&s_eps, 1u);
  }
  __syncthreads();
  if (threadIdx.x < 9 && s_hist[threadIdx.x]) atomicAdd((unsigned long long*)&stats->termination_hist[threadIdx.x], (unsigned long long)s_hist[threadIdx.x]);
  if (threadIdx.x == 0) {
    atomicAdd((unsigned long long*)&stats->steps, (unsigned long long)s_steps);
    atomicAdd((unsigned long long*)&stats->episodes, (unsigned long long)s_eps);
  }
}

// Every (x agent, y agent) pair's two-axis greedy landing in one launch: blocks_per_pair blocks of 256 episodes per pair on a
// flat 1-D grid (pair = blockIdx.x / blocks_per_pair).  Pair k = (gx, gy) = pairs[2k], pairs[2k + 1]; agent g reads replica
// g * replicas.  Each block builds both LUTs in shared memory from the live tables: x from gx's float32 first-max; y from gy's
// own float32 first-max when gy is a y-axis agent (population axis 1), else the mirror image of gy's x policy
// (lut_y[s] = {1,0,2}[lut(rest * 7 + 6 - theta)], rest, theta = divmod(s, 7): engine.mirrored_policy).  States at and above
// curriculum_steps * 189 act 0 on both axes.  Platform, gravity signs, y options and Philox key come from p for every pair, so
// episode i of every pair starts from the same draw: episode first_episode + i of eval2d_kernel under the two LUTs.  p.working_step
// < 0: the lower of the two members' live working steps.  Reads tables and trainer state, writes only stats.
template <bool GENERIC>
__global__ void __launch_bounds__(256) eval_pairs_kernel(const __grid_constant__ KC kc, const __grid_constant__ dqlb200_eval2d_params p,
                                                         const dqlb200_population_params* pop_params, const uint32_t* __restrict__ tables,
                                                         const dqlb200_population_state* __restrict__ pop_state,
                                                         const int32_t* __restrict__ pairs, int replicas, int blocks_per_pair,
                                                         long long first_episode, long long episodes_per_pair, dqlb200_eval_stats* stats) {
  const auto& kk = ConstsOf<GENERIC>::get(kc);
  constexpr int N_STATES = DQLB200_MAX_CURRICULUM * DQLB200_STATES_PER_LEVEL;
  __shared__ uint8_t s_pol_x[N_STATES], s_pol_y[N_STATES];
  __shared__ dqlb200_cuts cuts;
  __shared__ unsigned int s_hist[9], s_steps, s_eps;
  const int pair = (int)(blockIdx.x / (unsigned)blocks_per_pair);
  const int block_in_pair = (int)(blockIdx.x - (unsigned)pair * (unsigned)blocks_per_pair);
  const int pop_x = pairs[2 * pair] * replicas, pop_y = pairs[2 * pair + 1] * replicas;
  const float* qax = reinterpret_cast<const float*>(tables + (size_t)pop_x * 3 * DQLB200_MAX_CELLS);
  const float* qbx = qax + DQLB200_MAX_CELLS;
  const float* qay = reinterpret_cast<const float*>(tables + (size_t)pop_y * 3 * DQLB200_MAX_CELLS);
  const float* qby = qay + DQLB200_MAX_CELLS;
  const bool y_own = pop_params[pop_y].axis == 1;
  const int live_states = kc.curriculum_steps * DQLB200_STATES_PER_LEVEL;
  for (int s = threadIdx.x; s < N_STATES; s += blockDim.x) {
    uint8_t ax = 0, ay = 0;
    if (s < live_states) {
      ax = greedy_action_f32(qax, qbx, s);
      if (y_own) {
        ay = greedy_action_f32(qay, qby, s);
      } else {
        const int rest = s / 7, theta = s - rest * 7;
        const uint8_t a = greedy_action_f32(qay, qby, rest * 7 + 6 - theta);
        ay = a == 2 ? (uint8_t)2 : (uint8_t)(1 - a);      // {1, 0, 2}[a]: increase and decrease swap
      }
    }
    s_pol_x[s] = ax;
    s_pol_y[s] = ay;
  }
  if (threadIdx.x == 0) {
    int w = p.working_step;
    if (w < 0) w = min(max(min(pop_state[pop_x].working_step, pop_state[pop_y].working_step), 0), kc.curriculum_steps - 1);
    cuts = kc.cuts[w];
    s_steps = s_eps = 0u;
  }
  if (threadIdx.x < 9) s_hist[threadIdx.x] = 0u;
  __syncthreads();
  const long long i = (long long)block_in_pair * blockDim.x + threadIdx.x;
  if (i < episodes_per_pair) {
    int step;
    const dqlb200_trace2d no_trace = {};
    const int code = greedy_episode_2d(kk, p, cuts, s_pol_x, s_pol_y, (unsigned long long)(first_episode + i), no_trace, 0, i,
                                       episodes_per_pair, step);
    atomicAdd(&s_hist[code], 1u);
    atomicAdd(&s_steps, (unsigned int)step);
    atomicAdd(&s_eps, 1u);
  }
  __syncthreads();
  dqlb200_eval_stats* st = stats + pair;
  if (threadIdx.x < 9 && s_hist[threadIdx.x]) atomicAdd((unsigned long long*)&st->termination_hist[threadIdx.x], (unsigned long long)s_hist[threadIdx.x]);
  if (threadIdx.x == 0) {
    atomicAdd((unsigned long long*)&st->steps, (unsigned long long)s_steps);
    atomicAdd((unsigned long long*)&st->episodes, (unsigned long long)s_eps);
  }
}


}  // namespace dql
