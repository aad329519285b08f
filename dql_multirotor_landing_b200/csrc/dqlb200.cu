// libdqlb200: kernels + C-ABI (include/dqlb200.h).  Compile for sm_100a only:
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -Xcompiler -fPIC -shared
//
// Kernel inventory (this file holds the C-ABI; the kernels live in the headers it includes)
//   dqlb200_device.cuh   Philox4x32-10, deterministic fp32 math, stand-in dynamics (R4), cut-table discretisation (R5),
//                        set-point (R3), exact float64 divisions, reward (R7)
//   env_state.cuh        the 48-byte env state: pack/unpack, reset law (R1/R8), cp.async prefetch
//   train_kernel.cuh     train_kernel<WARPS, TRACE, VARIANT>: one CTA per population (agent), K fused global steps per launch.
//                        Per step and env: epsilon-greedy select (R9/R10), set-point, dynamics, discretise, check (R6),
//                        reward, learning rate (R11), table update (R12), auto-reset, success window / promotion /
//                        transfer (R13/R14).  Q_a / count live in shared memory for the whole launch.
//   env_kernels.cuh      reset_kernel (R1 + R8 for every env), eval_kernel / eval2d_kernel (R15: greedy SimulationMdp
//                        episodes, one thread per episode, one or two axes), eval_agents_kernel (every agent's greedy policy
//                        from its live tables, one launch, under its own platform or a list of platform motions),
//                        eval_pairs_kernel (every x/y agent pair's two-axis landing from
//                        the live tables, one launch), env_reset_kernel / env_step_kernel (gym surface)
//   facade_kernels.cuh   float64 single-object TrainingMdp / SimulationMdp / DoubleQLearningAgent calls, division self-test
//   table_kernels.cuh    transfer (R13), shared-table pack/apply, replica merge, atomic-roof micro-benchmark
//
// Same-cell update semantics ("S1", DESIGN.md): all envs of a population select and bootstrap from the
// tables as of the START of the global step; the updates are then applied one by one in env-index order
// to the live table, each with the learning rate of the live pre-increment count.  Implementation: env
// index = slot * blockDim + thread; the commit of (slot, warp) chunks is serialised by a baton passed
// between warps with named barriers; inside a chunk, lanes hitting the same cell are found with
// __match_any_sync and applied sequentially in lane order by shuffles.  Bit-exact vs the sequential
// oracle for any number of envs.
#include <cuda_runtime.h>

#include <cstdio>
#include <cmath>
#include <cstring>
#include <new>
#include <string>
#include <vector>
#include <dlfcn.h>


#include "env_state.cuh"
#include "train_kernel.cuh"
#include "env_kernels.cuh"
#include "facade_kernels.cuh"
#include "table_kernels.cuh"


// =================================================================================================
// C-ABI
// =================================================================================================
struct dqlb200_handle {
  dqlb200_config cfg;
  dql::KC kc;
  int device;
  dqlb200_config* d_cfg;
  float* d_alpha;
  dqlb200_population_params* d_pop_params;
  uint32_t* d_error;
  void* env_state;
  void* tables;
  void* pop_state;
  void* merge_snapshot;
  void* filter_state;       // accel_mode != 0: [n_total] x 16 B estimator state (dqlb200_bind_filter_state)
  void* dynamics_state;     // dynamics_model != 0: [2][n_total] x 16 B second-order model state (dqlb200_bind_dynamics_state)
  bool kc_default;              // the configuration equals the compile-time defaults: the production instance may run
  std::vector<int32_t> pop_axis;    // host copy of every population's axis (dqlb200_eval_pairs validates pairs without a device read)
  std::vector<int32_t> pairs_stage;  // dqlb200_eval_pairs: the caller's pair list, copied here before the (staged) upload
  int32_t* d_pairs;                 // dqlb200_eval_pairs: the uploaded pair list, grown on demand
  int d_pairs_cap;
  cudaEvent_t pairs_read;           // recorded after the launch that reads d_pairs; the next upload waits for it
  std::vector<dqlb200_platform> platforms_stage;   // dqlb200_eval_agents_platforms: the caller's list, staged as pairs_stage
  dqlb200_platform* d_platforms;                   // the uploaded list, grown on demand
  int d_platforms_cap;
  cudaEvent_t platforms_read;                      // recorded after the launch that reads d_platforms
  size_t smem_bytes;
  // dqlb200_train_host pipelines the populations in chunks over these streams (copy-in / train / copy-out overlap)
  static constexpr int MAX_HOST_CHUNKS = 64;
  cudaStream_t chunk_stream[MAX_HOST_CHUNKS];
  cudaEvent_t chunk_done[MAX_HOST_CHUNKS];
  cudaEvent_t host_start;
  bool chunk_ready;
  // dqlb200_train_merged replays ONE captured CUDA graph (train launch of `merged_k` steps + replica merge) on its own stream
  cudaStream_t merged_stream;
  cudaEvent_t merged_in, merged_out;
  cudaGraphExec_t merged_exec, merged_exec_multi;      // one (train, merge) pair / MERGED_GRAPH_PAIRS pairs
  int merged_k, merged_promote;
  bool merged_ready;
};

static thread_local std::string g_last_error;
static int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}
#define CUDA_TRY(expr)                                                                                      \
  do {                                                                                                      \
    cudaError_t _e = (expr);                                                                                \
    if (_e != cudaSuccess) return fail(DQLB200_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
  } while (0)

extern "C" {

int dqlb200_abi_version(void) { return DQLB200_ABI_VERSION; }
size_t dqlb200_config_bytes(void) { return sizeof(dqlb200_config); }
size_t dqlb200_population_state_bytes(void) { return sizeof(dqlb200_population_state); }
size_t dqlb200_eval2d_params_bytes(void) { return sizeof(dqlb200_eval2d_params); }
size_t dqlb200_platform_bytes(void) { return sizeof(dqlb200_platform); }
size_t dqlb200_env_state_bytes(int n_populations, int envs_per_population) {
  if (n_populations < 0 || envs_per_population < 0) return 0;
  return (size_t)n_populations * (((size_t)envs_per_population + 31) / 32) * dql::ENV_TILE_BYTES;
}
const char* dqlb200_last_error(void) { return g_last_error.c_str(); }

const char* dqlb200_termination_string(int code) {
  switch (code) {
    case DQLB200_TERMINAL_SUCCESS: return "SUCCESS: Goal state reached";
    case DQLB200_TERMINAL_CONTACT: return "SUCCESS: Touched platform";
    case DQLB200_TERMINAL_FLYZONE_X: return "FAILURE: Drone moved too far from platform in x direction";
    case DQLB200_TERMINAL_FLYZONE_Y: return "FAILURE: Drone moved too far from platform in y direction";
    case DQLB200_TERMINAL_FLYZONE_Z: return "FAILURE: Drone moved too far from platform in z direction";
    case DQLB200_TERMINAL_MINIMUM_ALTITUDE: return "FAILURE: Reached minimum altitude";
    case DQLB200_TERMINAL_TIMEOUT: return "FAILURE: Maximum episode duration";
    default: return nullptr;
  }
}

// Smallest non-negative fp32 x with RN((double)x / d) >= 1.0: np.clip(x / d, -1, 1) saturates exactly for |x| >= this cut
// (the correctly rounded quotient is monotone in x), so the shaping potentials clip on the fp32 observation.
static float first_f32_with_unit_quotient(double d) {
  float x = (float)d;
  while ((double)x / d >= 1.0) x = nextafterf(x, 0.0f);
  while (!((double)x / d >= 1.0)) x = nextafterf(x, INFINITY);
  return x;
}

static void fill_kc(const dqlb200_config& c, dql::KC& k) {
  memcpy(k.cuts, c.cuts, sizeof(k.cuts));
  memcpy(k.reward, c.reward, sizeof(k.reward));
  k.p_max = c.p_max; k.v_max = c.v_max; k.theta_max = c.theta_max; k.delta_theta = c.delta_theta;
  k.w_p = c.w_p; k.w_v = c.w_v; k.w_theta = c.w_theta;
  k.rcp_p_max = 1.0 / c.p_max; k.rcp_v_max = 1.0 / c.v_max; k.rcp_theta_max = 1.0 / c.theta_max;
  k.div_two_steps = (c.p_max == 4.5 && c.v_max == 3.39411) ? 0 : 1;
  k.clip_p_f = first_f32_with_unit_quotient(c.p_max);
  k.clip_v_f = first_f32_with_unit_quotient(c.v_max);
  memcpy(k.angle_cut, c.angle_cut, sizeof(k.angle_cut));
  k.fz_lo = c.fz_lo; k.fz_hi = c.fz_hi; k.z_min_cut = c.z_min_cut; k.z_max_cut = c.z_max_cut;
  k.h = c.h; k.half_h2 = c.half_h2; k.k_theta = c.k_theta; k.g = c.g; k.c_d = c.c_d;
  k.dz_train = c.dz_train; k.dz_sim = c.dz_sim; k.z_init = c.z_init; k.z_touch = c.z_touch;
  k.half_platform = c.half_platform; k.p_max_f = c.p_max_f; k.two_p_max_f = c.two_p_max_f; k.sigma_x = c.sigma_x;
  k.gamma = c.gamma;
  k.noise_pos_sd = c.noise_pos_sd; k.noise_vel_sd = c.noise_vel_sd;
  k.noise_enabled = (c.noise_pos_sd != 0.0f || c.noise_vel_sd != 0.0f) ? 1 : 0;
  k.accel_mode = c.accel_mode; k.kf_q = c.kf_q; k.kf_r = c.kf_r;
  k.dynamics_model = c.dynamics_model; k.pid_ticks = c.pid_ticks;
  k.att_kr = c.att_kr; k.att_kw = c.att_kw; k.inv_m = c.inv_m; k.inv_mg = c.inv_mg; k.g_abs = c.g_abs;
  k.pid_kp = c.pid_kp; k.pid_ki = c.pid_ki; k.pid_lo = c.pid_lo; k.pid_hi = c.pid_hi; k.pid_windup = c.pid_windup;
  k.pid_dt = c.pid_dt; k.pid_i0 = c.pid_i0; k.bw_inv_denom = c.bw_inv_denom; k.bw_k2 = c.bw_k2;
  k.vz_train = c.vz_train; k.vz_sim = c.vz_sim;
  memcpy(k.transfer_ratio, c.transfer_ratio, sizeof(k.transfer_ratio));
  k.timeout_steps = c.timeout_steps; k.success_steps = c.success_steps; k.n_sub = c.n_sub;
  k.transfer_mode = c.transfer_mode; k.window_len = c.window_len; k.promote_successes = c.promote_successes;
  k.curriculum_steps = c.curriculum_steps; k.envs_per_population = c.envs_per_population;
  k.n_populations = c.n_populations; k.max_num_episodes = c.max_num_episodes;
  k.replicas = c.replicas_per_population;
}

int dqlb200_create(const dqlb200_config* cfg, const float* alpha_luts, const dqlb200_population_params* pop_params,
                   int device, dqlb200_handle** out) {
  if (!cfg || !alpha_luts || !pop_params || !out) return fail(DQLB200_ERR_ARG, "null argument");
  if (cfg->struct_bytes != sizeof(dqlb200_config) || cfg->abi_version != DQLB200_ABI_VERSION)
    return fail(DQLB200_ERR_ARG, "dqlb200_config size/ABI mismatch: host " + std::to_string(cfg->struct_bytes) +
                                     " vs library " + std::to_string(sizeof(dqlb200_config)));
  if (cfg->n_populations < 1 || cfg->envs_per_population < 1) return fail(DQLB200_ERR_ARG, "empty layout");
  if (cfg->curriculum_steps < 1 || cfg->curriculum_steps > DQLB200_MAX_CURRICULUM) return fail(DQLB200_ERR_ARG, "curriculum_steps out of range");
  const int tpb = cfg->threads_per_block;
  if (tpb != 32 && tpb != 64 && tpb != 128 && tpb != 256) return fail(DQLB200_ERR_ARG, "threads_per_block must be 32, 64, 128 or 256");
  if (cfg->window_len < 1 || cfg->window_len > DQLB200_MAX_WINDOW) return fail(DQLB200_ERR_ARG, "window_len out of range");
  if (cfg->n_alpha_luts < 1 || cfg->n_sub < 1) return fail(DQLB200_ERR_ARG, "n_alpha_luts / n_sub must be >= 1");
  if (cfg->n_setpoints < 1 || cfg->n_setpoints > DQLB200_MAX_SETPOINTS || cfg->setpoint_zero < 0 || cfg->setpoint_zero >= cfg->n_setpoints)
    return fail(DQLB200_ERR_ARG, "set-point tables missing or too large (constants.py: build_setpoints)");
  if (cfg->accel_mode < 0 || cfg->accel_mode > 2) return fail(DQLB200_ERR_ARG, "accel_mode must be 0 (exact), 1 (reference filter) or 2 (consecutive-sample filter)");
  if (cfg->dynamics_model < 0 || cfg->dynamics_model > 1) return fail(DQLB200_ERR_ARG, "dynamics_model must be 0 (first order) or 1 (second order)");
  if (cfg->dynamics_model != 0 && (cfg->pid_ticks < 2 || cfg->pid_ticks > 64 || !(cfg->inv_m > 0.0f) || !(cfg->pid_hi >= cfg->pid_lo)))
    return fail(DQLB200_ERR_ARG, "second-order model: pid_ticks in 2..64, positive mass and pid_hi >= pid_lo required");
  if (cfg->accel_mode != 0 && (!(cfg->kf_q >= 0.0f) || !(cfg->kf_r >= 0.0f) || !(cfg->kf_q + cfg->kf_r > 0.0f)))
    return fail(DQLB200_ERR_ARG, "acceleration filter needs non-negative variances, not both zero");
  if (cfg->replicas_per_population < 1 || cfg->n_populations % cfg->replicas_per_population)
    return fail(DQLB200_ERR_ARG, "n_populations must be a multiple of replicas_per_population (>= 1)");
  for (int p = 0; p < cfg->n_populations; ++p)
    if (pop_params[p].alpha_lut < 0 || pop_params[p].alpha_lut >= cfg->n_alpha_luts) return fail(DQLB200_ERR_ARG, "population alpha_lut index out of range");
  int count = 0;
  CUDA_TRY(cudaGetDeviceCount(&count));
  if (device < 0 || device >= count) return fail(DQLB200_ERR_ARG, "no such CUDA device");
  CUDA_TRY(cudaSetDevice(device));
  dqlb200_handle* h = new (std::nothrow) dqlb200_handle();
  if (!h) return fail(DQLB200_ERR_STATE, "out of host memory");
  struct Guard {       // every early return below releases what has been allocated so far
    dqlb200_handle* h;
    ~Guard() { if (h) dqlb200_destroy(h); }
  } guard{h};
  h->cfg = *cfg;
  fill_kc(*cfg, h->kc);
  h->kc_default = dql::kdef_matches(h->kc);
  h->device = device;
  h->env_state = h->tables = h->pop_state = h->merge_snapshot = h->filter_state = h->dynamics_state = nullptr;
  h->chunk_ready = false;
  h->merged_ready = false;
  h->merged_exec = h->merged_exec_multi = nullptr;
  h->merged_k = 0;
  h->merged_promote = 0;
  try {
    h->pop_axis.assign(cfg->n_populations, 0);
  } catch (...) {
    return fail(DQLB200_ERR_STATE, "out of host memory");
  }
  for (int p = 0; p < cfg->n_populations; ++p) h->pop_axis[p] = pop_params[p].axis;
  h->d_pairs = nullptr;
  h->d_pairs_cap = 0;
  h->pairs_read = nullptr;
  h->d_platforms = nullptr;
  h->d_platforms_cap = 0;
  h->platforms_read = nullptr;
  CUDA_TRY(cudaMalloc(&h->d_cfg, sizeof(dqlb200_config)));
  CUDA_TRY(cudaMemcpy(h->d_cfg, cfg, sizeof(dqlb200_config), cudaMemcpyHostToDevice));
  const size_t lut_bytes = (size_t)cfg->n_alpha_luts * DQLB200_ALPHA_LUT * sizeof(float);
  CUDA_TRY(cudaMalloc(&h->d_alpha, lut_bytes));
  CUDA_TRY(cudaMemcpy(h->d_alpha, alpha_luts, lut_bytes, cudaMemcpyHostToDevice));
  const size_t pp_bytes = (size_t)cfg->n_populations * sizeof(dqlb200_population_params);
  CUDA_TRY(cudaMalloc(&h->d_pop_params, pp_bytes));
  CUDA_TRY(cudaMemcpy(h->d_pop_params, pop_params, pp_bytes, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMalloc(&h->d_error, 4 * sizeof(uint32_t)));
  CUDA_TRY(cudaMemset(h->d_error, 0, 4 * sizeof(uint32_t)));
  {
    const int tpb_ = cfg->threads_per_block;
    const int n_slots = (cfg->envs_per_population + tpb_ - 1) / tpb_;
    if (n_slots > 2047) return fail(DQLB200_ERR_ARG, "envs_per_population too large for threads_per_block (max 2047 slots per thread)");
    h->smem_bytes = dql::train_smem_bytes(tpb_, true, cfg->n_setpoints);      // the largest instance (extended / trace): tables + snapshot + set-point table + reset queues + staging slots
    if (h->smem_bytes > 227 * 1024) return fail(DQLB200_ERR_ARG, "population does not fit in shared memory: lower envs_per_population");
  }
#define DQL_SET_SMEM1(W, T, D)                                                                                            \
  CUDA_TRY(cudaFuncSetAttribute(dql::train_kernel<W, T, D>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared)); \
  CUDA_TRY(cudaFuncSetAttribute(dql::train_kernel<W, T, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dql::train_smem_bytes(W * 32, T || D == 2, cfg->n_setpoints)));
#define DQL_SET_SMEM(W) DQL_SET_SMEM1(W, false, 0) DQL_SET_SMEM1(W, false, 1) DQL_SET_SMEM1(W, false, 2) DQL_SET_SMEM1(W, false, 3) DQL_SET_SMEM1(W, true, 2)
  DQL_SET_SMEM(1) DQL_SET_SMEM(2) DQL_SET_SMEM(4) DQL_SET_SMEM(8)
  CUDA_TRY(cudaFuncSetAttribute(dql::replica_merge_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dql::merge_smem_bytes(32)));
#undef DQL_SET_SMEM
#undef DQL_SET_SMEM1
  guard.h = nullptr;
  *out = h;
  return DQLB200_OK;
}

int dqlb200_uses_default_instance(dqlb200_handle* h) { return (h && h->kc_default) ? 1 : 0; }

int dqlb200_config_is_default(const dqlb200_config* cfg) {
  if (!cfg || cfg->struct_bytes != sizeof(dqlb200_config)) return fail(DQLB200_ERR_ARG, "dqlb200_config size mismatch");
  dql::KC k;
  fill_kc(*cfg, k);
  return dql::kdef_matches(k) ? 1 : 0;
}

int dqlb200_destroy(dqlb200_handle* h) {
  if (!h) return DQLB200_OK;
  cudaSetDevice(h->device);
  cudaFree(h->d_cfg);
  cudaFree(h->d_alpha);
  cudaFree(h->d_pop_params);
  cudaFree(h->d_error);
  cudaFree(h->d_pairs);
  if (h->pairs_read) cudaEventDestroy(h->pairs_read);
  cudaFree(h->d_platforms);
  if (h->platforms_read) cudaEventDestroy(h->platforms_read);
  if (h->chunk_ready) {
    for (int c = 0; c < dqlb200_handle::MAX_HOST_CHUNKS; ++c) {
      cudaStreamDestroy(h->chunk_stream[c]);
      cudaEventDestroy(h->chunk_done[c]);
    }
    cudaEventDestroy(h->host_start);
  }
  if (h->merged_exec) cudaGraphExecDestroy(h->merged_exec);
  if (h->merged_exec_multi) cudaGraphExecDestroy(h->merged_exec_multi);
  if (h->merged_ready) {
    cudaStreamDestroy(h->merged_stream);
    cudaEventDestroy(h->merged_in);
    cudaEventDestroy(h->merged_out);
  }
  delete h;
  return DQLB200_OK;
}

int dqlb200_bind(dqlb200_handle* h, void* env_state, void* tables, void* pop_state) {
  if (!h || !env_state || !tables || !pop_state) return fail(DQLB200_ERR_ARG, "null argument");
  if (((uintptr_t)env_state & 15u) || ((uintptr_t)tables & 3u) || ((uintptr_t)pop_state & 7u))
    return fail(DQLB200_ERR_ARG, "misaligned buffer (env_state needs 16 B, pop_state 8 B)");
  // The packed env state counts an episode's steps in STEP_BITS bits and the goal steps in CC_BITS bits (env_state.cuh); a count
  // that reaches the limit ends the episode and is never stored, so the limit itself may be the largest field value.  (The
  // single-object facade kernels keep their counts in float64 and never bind an env state: any t_max * f_ag works there.)
  constexpr int max_steps = (1 << dql::STEP_BITS) - 1, max_goal = (1 << dql::CC_BITS) - 1;
  if (h->cfg.timeout_steps > max_steps)
    return fail(DQLB200_ERR_ARG, "episode length timeout_steps = " + std::to_string(h->cfg.timeout_steps) + " (t_max * f_ag = " +
                                     std::to_string(h->cfg.timeout_threshold) + ") exceeds " + std::to_string(max_steps) +
                                     ", the largest step count the env state holds");
  if (h->cfg.success_steps > max_goal)
    return fail(DQLB200_ERR_ARG, "goal length success_steps = " + std::to_string(h->cfg.success_steps) + " (f_ag = " +
                                     std::to_string(h->cfg.f_ag) + ") exceeds " + std::to_string(max_goal) +
                                     ", the largest goal-step count the env state holds");
  h->env_state = env_state;
  h->tables = tables;
  h->pop_state = pop_state;
  h->merged_k = 0;                 // a captured graph holds the old pointers
  return DQLB200_OK;
}

int dqlb200_bind_filter_state(dqlb200_handle* h, void* filter_state) {
  if (!h) return fail(DQLB200_ERR_ARG, "null handle");
  if ((uintptr_t)filter_state & 15u) return fail(DQLB200_ERR_ARG, "misaligned filter_state (needs 16 B)");
  h->filter_state = filter_state;
  h->merged_k = 0;                 // a captured graph holds the old pointer
  return DQLB200_OK;
}

int dqlb200_bind_dynamics_state(dqlb200_handle* h, void* dynamics_state) {
  if (!h) return fail(DQLB200_ERR_ARG, "null handle");
  if ((uintptr_t)dynamics_state & 15u) return fail(DQLB200_ERR_ARG, "misaligned dynamics_state (needs 16 B)");
  h->dynamics_state = dynamics_state;
  h->merged_k = 0;
  return DQLB200_OK;
}

// an option that needs its own per-env buffer and has none bound: refuse instead of computing with the default model
#define DQL_NEED_FILTER(h)                                                                                                          \
  if ((h)->cfg.accel_mode != 0 && !(h)->filter_state) return fail(DQLB200_ERR_STATE, "accel_mode != 0 needs dqlb200_bind_filter_state()"); \
  if ((h)->cfg.dynamics_model != 0 && !(h)->dynamics_state) return fail(DQLB200_ERR_STATE, "dynamics_model != 0 needs dqlb200_bind_dynamics_state()")

static size_t env_tiles_per_pop(const dqlb200_config& c) { return ((size_t)c.envs_per_population + 31) / 32; }
static size_t env_state_bytes(const dqlb200_config& c, size_t n_pop) { return n_pop * env_tiles_per_pop(c) * dql::ENV_TILE_BYTES; }

static dql::EnvPtrs env_ptrs(const dqlb200_handle* h, void* base) {
  const size_t n = (size_t)h->cfg.n_populations * h->cfg.envs_per_population;
  dql::EnvPtrs p;
  p.base = reinterpret_cast<unsigned char*>(base);
  p.n_p = h->cfg.envs_per_population;
  p.tiles_per_pop = (int)env_tiles_per_pop(h->cfg);
  p.d = h->cfg.accel_mode != 0 ? reinterpret_cast<uint4*>(h->filter_state) : nullptr;
  p.e = h->cfg.dynamics_model != 0 ? reinterpret_cast<uint4*>(h->dynamics_state) : nullptr;
  p.n = n;
  p.sp_value = h->d_cfg->setpoint_value;            // device addresses inside the device copy of the configuration
  p.sp_next = reinterpret_cast<const uint2*>(&h->d_cfg->setpoint_next[0][0]);
  p.sp_rtheta = &h->d_cfg->setpoint_rtheta[0][0][0];
  p.sp_zero = h->cfg.setpoint_zero;
  p.n_sp = h->cfg.n_setpoints;
  return p;
}

int dqlb200_reset(dqlb200_handle* h, int initial_step, void* stream) {
  if (!h || !h->env_state) return fail(DQLB200_ERR_STATE, "buffers not bound");
  if (initial_step < 0 || initial_step >= h->cfg.curriculum_steps) return fail(DQLB200_ERR_ARG, "initial_step out of range");
  DQL_NEED_FILTER(h);
  CUDA_TRY(cudaSetDevice(h->device));
  const dim3 grid((h->cfg.envs_per_population + 255) / 256, h->cfg.n_populations);
  dql::reset_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(h->kc, env_ptrs(h, h->env_state),
                                                           (dqlb200_population_state*)h->pop_state, h->d_pop_params, initial_step);
  CUDA_TRY(cudaGetLastError());
  return DQLB200_OK;
}

static int launch_train(dqlb200_handle* h, int k_steps, const dqlb200_trace* trace, void* env_state, void* tables,
                        void* pop_state, cudaStream_t stream, int pop_offset = 0, int pop_count = -1) {
  dql::TrainArgs a;
  a.env = env_ptrs(h, env_state);
  a.tables = (uint32_t*)tables;
  a.pop_state = (dqlb200_population_state*)pop_state;
  a.pop_params = h->d_pop_params;
  a.alpha_luts = h->d_alpha;
  a.eps_threshold = h->d_cfg->eps_threshold;
  if (trace) a.trace = *trace; else memset(&a.trace, 0, sizeof(a.trace));
  a.merge_snapshot = (h->cfg.replicas_per_population > 1) ? (uint32_t*)h->merge_snapshot : nullptr;
  a.k_steps = k_steps;
  a.pop_offset = pop_offset;
  a.n_total = (long long)h->cfg.n_populations * h->cfg.envs_per_population;
  const int grid = pop_count < 0 ? h->cfg.n_populations : pop_count;
  const bool tracing = trace != nullptr;
  const bool extended = h->cfg.accel_mode != 0 || h->cfg.dynamics_model != 0;      // options with extra per-env state
  const size_t smem = dql::train_smem_bytes(h->cfg.threads_per_block, tracing || extended, h->cfg.n_setpoints);      // the trace instances are extended ones
  const bool full_slots = h->cfg.envs_per_population % h->cfg.threads_per_block == 0;
#define DQL_LAUNCH(W)                                                                        \
  if (tracing) dql::train_kernel<W, true, 2><<<grid, W * 32, smem, stream>>>(h->kc, a);                     \
  else if (extended) dql::train_kernel<W, false, 2><<<grid, W * 32, smem, stream>>>(h->kc, a);            \
  else if (!h->kc_default) dql::train_kernel<W, false, 1><<<grid, W * 32, smem, stream>>>(h->kc, a);      \
  else if (full_slots) dql::train_kernel<W, false, 3><<<grid, W * 32, smem, stream>>>(h->kc, a);          \
  else dql::train_kernel<W, false, 0><<<grid, W * 32, smem, stream>>>(h->kc, a);
  switch (h->cfg.threads_per_block) {
    case 32: DQL_LAUNCH(1) break;
    case 64: DQL_LAUNCH(2) break;
    case 128: DQL_LAUNCH(4) break;
    default: DQL_LAUNCH(8) break;
  }
#undef DQL_LAUNCH
  CUDA_TRY(cudaGetLastError());
  return DQLB200_OK;
}

int dqlb200_train(dqlb200_handle* h, int k_steps, const dqlb200_trace* trace, void* stream) {
  if (!h || !h->env_state) return fail(DQLB200_ERR_STATE, "buffers not bound");
  if (k_steps < 0) return fail(DQLB200_ERR_ARG, "k_steps < 0");
  if (k_steps == 0) return DQLB200_OK;
  DQL_NEED_FILTER(h);
  CUDA_TRY(cudaSetDevice(h->device));
  return launch_train(h, k_steps, trace, h->env_state, h->tables, h->pop_state, (cudaStream_t)stream);
}

int dqlb200_train_host(dqlb200_handle* h, int k_steps, void* env_state_host, void* tables_host, void* pop_state_host,
                       int table_levels, void* stream) {
  return dqlb200_train_host_ext(h, k_steps, env_state_host, tables_host, pop_state_host, nullptr, nullptr, table_levels, stream);
}

int dqlb200_train_host_ext(dqlb200_handle* h, int k_steps, void* env_state_host, void* tables_host, void* pop_state_host,
                           void* filter_state_host, void* dynamics_state_host, int table_levels, void* stream) {
  if (!h || !h->env_state) return fail(DQLB200_ERR_STATE, "buffers not bound (device staging buffers are the bound ones)");
  if (!env_state_host || !tables_host || !pop_state_host) return fail(DQLB200_ERR_ARG, "null host buffer");
  // the per-env extension state of the options travels like the env state (never computed with a default model instead)
  if (h->cfg.accel_mode != 0 && !filter_state_host)
    return fail(DQLB200_ERR_ARG, "accel_mode != 0: the estimator state must travel too (dqlb200_train_host_ext with filter_state_host)");
  if (h->cfg.dynamics_model != 0 && !dynamics_state_host)
    return fail(DQLB200_ERR_ARG, "dynamics_model != 0: the second-order state must travel too (dqlb200_train_host_ext with dynamics_state_host)");
  DQL_NEED_FILTER(h);
  const bool with_filter = h->cfg.accel_mode != 0, with_dyn = h->cfg.dynamics_model != 0;
  if (k_steps < 0) return fail(DQLB200_ERR_ARG, "k_steps < 0");
  if (table_levels < 0 || table_levels > h->cfg.curriculum_steps) return fail(DQLB200_ERR_ARG, "table_levels must be 0 (all) .. curriculum_steps");
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  if (!h->chunk_ready) {
    for (int c = 0; c < dqlb200_handle::MAX_HOST_CHUNKS; ++c) {
      CUDA_TRY(cudaStreamCreateWithFlags(&h->chunk_stream[c], cudaStreamNonBlocking));
      CUDA_TRY(cudaEventCreateWithFlags(&h->chunk_done[c], cudaEventDisableTiming));
    }
    CUDA_TRY(cudaEventCreateWithFlags(&h->host_start, cudaEventDisableTiming));
    h->chunk_ready = true;
  }
  // Populations are independent within a launch, so the call is pipelined over chunks of populations: while chunk c
  // trains, chunk c+1 is copied in and chunk c-1 is copied out (PCIe is full duplex, the copy engines run beside the SMs).
  // Tables: `table_levels` = L > 0 transfers only levels 0 .. L-1 of every table row (one strided copy per chunk and
  // direction) -- the caller's promise that no population reaches working step L - 1 + 1 inside the call (a launch touches
  // the levels 0 .. w of its working step w, and w + 1 when it is promoted); checked after the call.  L = 0: all levels.
  const int P = h->cfg.n_populations, cs_levels = h->cfg.curriculum_steps;
  // Chunk count: measured on one B200 (tools/perf_probe_e2e.py, 888 x 1,280 envs, 64 steps): 1 chunk 4.25 ms, 4: 3.05, 8: 2.93, 16: 3.03,
  // 32: 3.40, 64: 4.06 -- every chunk costs ~11 API calls of host time, and the call cannot end before the copy-in of everything
  // plus the 64 sequential steps of the last chunk.  DQLB200_HOST_CHUNKS overrides the default (measurement aid).
  int want_chunks = 8;
  if (const char* e = getenv("DQLB200_HOST_CHUNKS")) want_chunks = atoi(e);
  want_chunks = want_chunks < 1 ? 1 : (want_chunks > dqlb200_handle::MAX_HOST_CHUNKS ? dqlb200_handle::MAX_HOST_CHUNKS : want_chunks);
  const int n_chunks = P < want_chunks ? P : want_chunks;
  const size_t row_bytes = (size_t)DQLB200_MAX_CELLS * 4, tab_stride = 3 * row_bytes, ps_stride = sizeof(dqlb200_population_state);
  const size_t level_bytes = (size_t)DQLB200_CELLS_PER_LEVEL * 4;
  const dqlb200_population_state* ps_h = reinterpret_cast<const dqlb200_population_state*>(pop_state_host);
  CUDA_TRY(cudaEventRecord(h->host_start, s));
  for (int c = 0; c < n_chunks; ++c) {
    const int p0 = (int)((long long)P * c / n_chunks), p1 = (int)((long long)P * (c + 1) / n_chunks);
    if (p1 == p0) continue;
    int w_max = 0, w_min = cs_levels;
    for (int p = p0; p < p1; ++p) {
      w_max = ps_h[p].working_step > w_max ? ps_h[p].working_step : w_max;
      w_min = ps_h[p].working_step < w_min ? ps_h[p].working_step : w_min;
    }
    const int levels = table_levels > 0 ? table_levels : cs_levels;
    if (w_max + 1 > levels) return fail(DQLB200_ERR_ARG, "table_levels is smaller than the live levels of a population's working step");
    cudaStream_t cs = h->chunk_stream[c];
    CUDA_TRY(cudaStreamWaitEvent(cs, h->host_start, 0));
    const size_t e0 = env_state_bytes(h->cfg, (size_t)p0), eb = env_state_bytes(h->cfg, (size_t)(p1 - p0));      // a range of populations is one block
    CUDA_TRY(cudaMemcpyAsync((char*)h->env_state + e0, (const char*)env_state_host + e0, eb, cudaMemcpyHostToDevice, cs));
    CUDA_TRY(cudaMemcpy2DAsync((char*)h->tables + p0 * tab_stride, row_bytes, (const char*)tables_host + p0 * tab_stride, row_bytes,
                               levels * level_bytes, (size_t)3 * (p1 - p0), cudaMemcpyHostToDevice, cs));
    if (h->cfg.transfer_mode == 0 && w_min == 0 && levels < cs_levels)      // quirk Q7: ending step 0 reads the LAST level (slot -1)
      CUDA_TRY(cudaMemcpy2DAsync((char*)h->tables + p0 * tab_stride + (cs_levels - 1) * level_bytes, row_bytes,
                                 (const char*)tables_host + p0 * tab_stride + (cs_levels - 1) * level_bytes, row_bytes, level_bytes,
                                 (size_t)3 * (p1 - p0), cudaMemcpyHostToDevice, cs));
    CUDA_TRY(cudaMemcpyAsync((char*)h->pop_state + p0 * ps_stride, (const char*)pop_state_host + p0 * ps_stride, (p1 - p0) * ps_stride, cudaMemcpyHostToDevice, cs));
    // extension state of the chunk's envs: [n] x 16 B (estimator) and [2][n] x 16 B (second-order model: two planes, one 2-D copy)
    const size_t x0 = (size_t)p0 * h->cfg.envs_per_population * 16, xb = (size_t)(p1 - p0) * h->cfg.envs_per_population * 16;
    const size_t plane = (size_t)P * h->cfg.envs_per_population * 16;
    if (with_filter) CUDA_TRY(cudaMemcpyAsync((char*)h->filter_state + x0, (const char*)filter_state_host + x0, xb, cudaMemcpyHostToDevice, cs));
    if (with_dyn) CUDA_TRY(cudaMemcpy2DAsync((char*)h->dynamics_state + x0, plane, (const char*)dynamics_state_host + x0, plane, xb, 2, cudaMemcpyHostToDevice, cs));
    if (k_steps > 0) {
      const int rc = launch_train(h, k_steps, nullptr, h->env_state, h->tables, h->pop_state, cs, p0, p1 - p0);
      if (rc) return rc;
    }
    CUDA_TRY(cudaMemcpyAsync((char*)env_state_host + e0, (const char*)h->env_state + e0, eb, cudaMemcpyDeviceToHost, cs));
    CUDA_TRY(cudaMemcpy2DAsync((char*)tables_host + p0 * tab_stride, row_bytes, (const char*)h->tables + p0 * tab_stride, row_bytes,
                               levels * level_bytes, (size_t)3 * (p1 - p0), cudaMemcpyDeviceToHost, cs));
    CUDA_TRY(cudaMemcpyAsync((char*)pop_state_host + p0 * ps_stride, (const char*)h->pop_state + p0 * ps_stride, (p1 - p0) * ps_stride, cudaMemcpyDeviceToHost, cs));
    if (with_filter) CUDA_TRY(cudaMemcpyAsync((char*)filter_state_host + x0, (const char*)h->filter_state + x0, xb, cudaMemcpyDeviceToHost, cs));
    if (with_dyn) CUDA_TRY(cudaMemcpy2DAsync((char*)dynamics_state_host + x0, plane, (const char*)h->dynamics_state + x0, plane, xb, 2, cudaMemcpyDeviceToHost, cs));
    CUDA_TRY(cudaEventRecord(h->chunk_done[c], cs));
    CUDA_TRY(cudaStreamWaitEvent(s, h->chunk_done[c], 0));
  }
  CUDA_TRY(cudaStreamSynchronize(s));
  // the promise behind table_levels: nobody went beyond the transferred levels
  for (int p = 0; p < P && table_levels > 0 && table_levels < cs_levels; ++p)
    if (ps_h[p].working_step + 1 > table_levels && !ps_h[p].finished)
      return fail(DQLB200_ERR_STATE, "population " + std::to_string(p) + " was promoted beyond the transferred table levels: repeat the call with table_levels = 0");
  return DQLB200_OK;
}

int dqlb200_eval_greedy(dqlb200_handle* h, int population, const uint8_t* policy, int64_t first_episode, int64_t n_episodes,
                        int working_step, void* stats_out, const dqlb200_trace* trace, int trace_steps, void* stream) {
  if (!h || !policy || !stats_out) return fail(DQLB200_ERR_ARG, "null argument");
  if (population < 0 || population >= h->cfg.n_populations) return fail(DQLB200_ERR_ARG, "population out of range");
  if (working_step < 0 || working_step >= DQLB200_MAX_CURRICULUM) return fail(DQLB200_ERR_ARG, "working_step out of range");
  if (n_episodes <= 0) return DQLB200_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  dqlb200_trace tr;
  if (trace) tr = *trace; else memset(&tr, 0, sizeof(tr));
  const long long blocks = (n_episodes + 255) / 256;
  if (h->kc_default)
    dql::eval_kernel<false><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(h->kc, h->d_pop_params, population, policy, first_episode, n_episodes,
                                                                              working_step, (dqlb200_eval_stats*)stats_out, tr, trace ? trace_steps : 0);
  else
    dql::eval_kernel<true><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(h->kc, h->d_pop_params, population, policy, first_episode, n_episodes,
                                                                             working_step, (dqlb200_eval_stats*)stats_out, tr, trace ? trace_steps : 0);
  CUDA_TRY(cudaGetLastError());
  return DQLB200_OK;
}

// ceil(episodes_per_agent / 256) blocks per cell x n_agents x n_platforms cells fit one launch's 1-D grid (episodes_per_agent >= 1;
// n_agents and n_platforms are below 2^31, so their product does not overflow)
static bool eval_agents_grid_fits(const dqlb200_handle* h, int64_t episodes_per_agent, int n_platforms) {
  const long long cells = (long long)(h->cfg.n_populations / h->cfg.replicas_per_population) * n_platforms;
  return (episodes_per_agent - 1) / 256 + 1 <= 0x7FFFFFFFLL / cells;
}

// One eval_agents_kernel launch over n_agents x n_platforms cells (d_platforms nullptr: each agent's own platform, n_platforms 1).
// The caller has checked every argument.
static int launch_eval_agents(dqlb200_handle* h, int working_step, int64_t first_episode, int64_t episodes_per_agent,
                              const dqlb200_platform* d_platforms, int n_platforms, void* stats_out, uint8_t* policy_out, cudaStream_t s) {
  const long long blocks_per_agent = (episodes_per_agent - 1) / 256 + 1;
  const int R = h->cfg.replicas_per_population, n_agents = h->cfg.n_populations / R;
  CUDA_TRY(cudaSetDevice(h->device));
  const unsigned grid = (unsigned)(blocks_per_agent * n_agents * n_platforms);
  const auto* ps = (const dqlb200_population_state*)h->pop_state;
  if (h->kc_default)
    dql::eval_agents_kernel<false><<<grid, 256, 0, s>>>(h->kc, h->d_pop_params, (const uint32_t*)h->tables, ps, R, (int)blocks_per_agent,
                                                       first_episode, episodes_per_agent, working_step, d_platforms, n_platforms,
                                                       (dqlb200_eval_stats*)stats_out, policy_out);
  else
    dql::eval_agents_kernel<true><<<grid, 256, 0, s>>>(h->kc, h->d_pop_params, (const uint32_t*)h->tables, ps, R, (int)blocks_per_agent,
                                                      first_episode, episodes_per_agent, working_step, d_platforms, n_platforms,
                                                      (dqlb200_eval_stats*)stats_out, policy_out);
  CUDA_TRY(cudaGetLastError());
  return DQLB200_OK;
}

int dqlb200_eval_agents(dqlb200_handle* h, int working_step, int64_t first_episode, int64_t episodes_per_agent, void* stats_out,
                        uint8_t* policy_out, void* stream) {
  if (!h) return fail(DQLB200_ERR_ARG, "null handle");
  if (!stats_out) return fail(DQLB200_ERR_ARG, "stats_out required");
  if (working_step < -1 || working_step >= h->cfg.curriculum_steps)
    return fail(DQLB200_ERR_ARG, "working_step must be -1 (each agent's live step) or 0 .. curriculum_steps - 1");
  if (!h->tables || !h->pop_state) return fail(DQLB200_ERR_STATE, "tables / trainer state not bound");
  DQL_NEED_FILTER(h);
  if (episodes_per_agent <= 0) return DQLB200_OK;
  if (!eval_agents_grid_fits(h, episodes_per_agent, 1)) return fail(DQLB200_ERR_ARG, "episodes_per_agent * n_agents exceeds one launch's grid");
  return launch_eval_agents(h, working_step, first_episode, episodes_per_agent, nullptr, 1, stats_out, policy_out, (cudaStream_t)stream);
}

int dqlb200_eval_agents_platforms(dqlb200_handle* h, int working_step, int64_t first_episode, int64_t episodes_per_agent,
                                  const dqlb200_platform* platforms_host, int n_platforms, void* stats_out, void* stream) {
  if (!h) return fail(DQLB200_ERR_ARG, "null handle");
  if (!platforms_host || !stats_out) return fail(DQLB200_ERR_ARG, "platforms_host and stats_out are required");
  if (n_platforms < 1) return fail(DQLB200_ERR_ARG, "n_platforms must be >= 1");
  for (int c = 0; c < n_platforms; ++c) {
    const dqlb200_platform& pl = platforms_host[c];
    if (!std::isfinite(pl.r) || !(pl.r > 0.0f))
      return fail(DQLB200_ERR_ARG, "platform " + std::to_string(c) + ": r must be finite and > 0");
    if (!std::isfinite(pl.rw) || !std::isfinite(pl.rw2) || !(pl.rw >= 0.0f) || !(pl.rw2 >= 0.0f))
      return fail(DQLB200_ERR_ARG, "platform " + std::to_string(c) + ": rw and rw2 must be finite and >= 0");
  }
  if (working_step < -1 || working_step >= h->cfg.curriculum_steps)
    return fail(DQLB200_ERR_ARG, "working_step must be -1 (each agent's live step) or 0 .. curriculum_steps - 1");
  if (!h->tables || !h->pop_state) return fail(DQLB200_ERR_STATE, "tables / trainer state not bound");
  DQL_NEED_FILTER(h);
  if (episodes_per_agent <= 0) return DQLB200_OK;
  if (!eval_agents_grid_fits(h, episodes_per_agent, n_platforms))
    return fail(DQLB200_ERR_ARG, "episodes_per_agent * n_agents * n_platforms exceeds one launch's grid");
  try {
    h->platforms_stage.assign(platforms_host, platforms_host + n_platforms);
  } catch (...) {
    return fail(DQLB200_ERR_STATE, "out of host memory");
  }
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  if (!h->platforms_read) CUDA_TRY(cudaEventCreateWithFlags(&h->platforms_read, cudaEventDisableTiming));
  if (n_platforms > h->d_platforms_cap) {
    CUDA_TRY(cudaEventSynchronize(h->platforms_read));      // the previous launch has read the old list
    CUDA_TRY(cudaFree(h->d_platforms));
    h->d_platforms = nullptr;
    h->d_platforms_cap = 0;
    CUDA_TRY(cudaMalloc(&h->d_platforms, (size_t)n_platforms * sizeof(dqlb200_platform)));
    h->d_platforms_cap = n_platforms;
  }
  CUDA_TRY(cudaStreamWaitEvent(s, h->platforms_read, 0));      // a launch on another stream may still read the list
  // from pageable memory the copy is staged before cudaMemcpyAsync returns, so neither platforms_host nor platforms_stage is read later
  CUDA_TRY(cudaMemcpyAsync(h->d_platforms, h->platforms_stage.data(), (size_t)n_platforms * sizeof(dqlb200_platform), cudaMemcpyHostToDevice, s));
  const int rc = launch_eval_agents(h, working_step, first_episode, episodes_per_agent, h->d_platforms, n_platforms, stats_out, nullptr, s);
  if (rc) return rc;
  CUDA_TRY(cudaEventRecord(h->platforms_read, s));
  return DQLB200_OK;
}

int dqlb200_env_reset(dqlb200_handle* h, int working_step, uint32_t birth, const uint8_t* mask, int fresh_mdp, int simulation,
                      uint16_t* out_state, void* stream) {
  if (!h || !h->env_state) return fail(DQLB200_ERR_STATE, "buffers not bound");
  if (working_step < 0 || working_step >= DQLB200_MAX_CURRICULUM) return fail(DQLB200_ERR_ARG, "working_step out of range");
  DQL_NEED_FILTER(h);
  CUDA_TRY(cudaSetDevice(h->device));
  const long long n = (long long)h->cfg.n_populations * h->cfg.envs_per_population;
  dql::env_reset_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(h->kc, env_ptrs(h, h->env_state), h->d_pop_params, working_step,
                                                                                     birth, mask, fresh_mdp, simulation, out_state);
  CUDA_TRY(cudaGetLastError());
  return DQLB200_OK;
}

int dqlb200_env_step(dqlb200_handle* h, int working_step, uint32_t t, const int8_t* actions, int auto_reset, int simulation,
                     uint16_t* out_state, double* out_reward, uint8_t* out_code, uint8_t* out_done, float* out_obs, uint32_t* out_steps,
                     double* out_cumulative, uint16_t* out_next_state, void* stream) {
  if (!h || !h->env_state) return fail(DQLB200_ERR_STATE, "buffers not bound");
  if (!actions) return fail(DQLB200_ERR_ARG, "actions required");
  if (working_step < 0 || working_step >= DQLB200_MAX_CURRICULUM) return fail(DQLB200_ERR_ARG, "working_step out of range");
  DQL_NEED_FILTER(h);
  CUDA_TRY(cudaSetDevice(h->device));
  const long long n = (long long)h->cfg.n_populations * h->cfg.envs_per_population;
  const unsigned blocks = (unsigned)((n + 127) / 128);
  if (h->kc.div_two_steps)
    dql::env_step_kernel<true><<<blocks, 128, 0, (cudaStream_t)stream>>>(h->kc, env_ptrs(h, h->env_state), h->d_pop_params, working_step, t, actions, auto_reset,
                                                                       simulation, out_state, out_reward, out_code, out_done, out_obs, out_steps, out_cumulative, out_next_state, h->d_error);
  else
    dql::env_step_kernel<false><<<blocks, 128, 0, (cudaStream_t)stream>>>(h->kc, env_ptrs(h, h->env_state), h->d_pop_params, working_step, t, actions, auto_reset,
                                                                        simulation, out_state, out_reward, out_code, out_done, out_obs, out_steps, out_cumulative, out_next_state, h->d_error);
  CUDA_TRY(cudaGetLastError());
  return DQLB200_OK;
}

int dqlb200_agent_select(dqlb200_handle* h, int working_step, uint32_t t, uint8_t* out_actions, uint16_t* out_states, void* stream) {
  if (!h || !h->env_state || !h->tables) return fail(DQLB200_ERR_STATE, "buffers not bound");
  if (!out_actions) return fail(DQLB200_ERR_ARG, "out_actions required");
  if (working_step < 0 || working_step >= DQLB200_MAX_CURRICULUM) return fail(DQLB200_ERR_ARG, "working_step out of range");
  CUDA_TRY(cudaSetDevice(h->device));
  const long long n = (long long)h->cfg.n_populations * h->cfg.envs_per_population;
  dql::agent_select_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(h->kc, env_ptrs(h, h->env_state), (const uint32_t*)h->tables,
                                                                                        h->d_pop_params, h->d_cfg->eps_threshold, working_step, t,
                                                                                        out_actions, out_states);
  CUDA_TRY(cudaGetLastError());
  return DQLB200_OK;
}

int dqlb200_agent_update(dqlb200_handle* h, const uint16_t* states, const uint8_t* actions, const uint16_t* next_states, const double* rewards,
                         void* stream) {
  if (!h || !h->tables) return fail(DQLB200_ERR_STATE, "buffers not bound");
  if (!states || !actions || !next_states || !rewards) return fail(DQLB200_ERR_ARG, "null argument");
  CUDA_TRY(cudaSetDevice(h->device));
  dql::agent_update_kernel<<<h->cfg.n_populations, 32, 0, (cudaStream_t)stream>>>(h->kc, (uint32_t*)h->tables, h->d_pop_params, h->d_alpha, states, actions,
                                                                                next_states, rewards);
  CUDA_TRY(cudaGetLastError());
  return DQLB200_OK;
}

int dqlb200_eval_greedy_2d(dqlb200_handle* h, const dqlb200_eval2d_params* p, const uint8_t* policy_x, const uint8_t* policy_y,
                           int64_t first_episode, int64_t n_episodes, void* stats_out, const dqlb200_trace2d* trace, int trace_steps,
                           void* stream) {
  if (!h || !p || !policy_x || !policy_y || !stats_out) return fail(DQLB200_ERR_ARG, "null argument");
  if (p->trajectory < 0 || p->trajectory > 2) return fail(DQLB200_ERR_ARG, "trajectory must be 0 (rectilinear x), 1 (rectilinear x and y) or 2 (eight)");
  if (p->working_step < 0 || p->working_step >= DQLB200_MAX_CURRICULUM) return fail(DQLB200_ERR_ARG, "working_step out of range");
  if (h->cfg.accel_mode != 0 || h->cfg.dynamics_model != 0)      // refuse rather than silently evaluate on the default model
    return fail(DQLB200_ERR_ARG, "the two-axis evaluator runs the first-order model with the analytic acceleration only (accel_mode = dynamics_model = 0)");
  if (n_episodes <= 0) return DQLB200_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  dqlb200_trace2d tr;
  if (trace) tr = *trace; else memset(&tr, 0, sizeof(tr));
  const long long blocks = (n_episodes + 255) / 256;
  if (h->kc_default)
    dql::eval2d_kernel<false><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(h->kc, *p, policy_x, policy_y, first_episode, n_episodes,
                                                                                (dqlb200_eval_stats*)stats_out, tr, trace ? trace_steps : 0);
  else
    dql::eval2d_kernel<true><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(h->kc, *p, policy_x, policy_y, first_episode, n_episodes,
                                                                               (dqlb200_eval_stats*)stats_out, tr, trace ? trace_steps : 0);
  CUDA_TRY(cudaGetLastError());
  return DQLB200_OK;
}

int dqlb200_eval_pairs(dqlb200_handle* h, const dqlb200_eval2d_params* p, const int32_t* pairs_host, int n_pairs, int64_t first_episode,
                       int64_t episodes_per_pair, void* stats_out, void* stream) {
  if (!h) return fail(DQLB200_ERR_ARG, "null handle");
  if (!p || !pairs_host || !stats_out) return fail(DQLB200_ERR_ARG, "params, pairs and stats_out are required");
  if (n_pairs < 1) return fail(DQLB200_ERR_ARG, "n_pairs must be >= 1");
  if (p->trajectory < 0 || p->trajectory > 2) return fail(DQLB200_ERR_ARG, "trajectory must be 0 (rectilinear x), 1 (rectilinear x and y) or 2 (eight)");
  if (p->working_step < -1 || p->working_step >= h->cfg.curriculum_steps)
    return fail(DQLB200_ERR_ARG, "working_step must be -1 (the lower live step of each pair) or 0 .. curriculum_steps - 1");
  const int R = h->cfg.replicas_per_population, n_agents = h->cfg.n_populations / R;
  for (int k = 0; k < n_pairs; ++k) {
    const int gx = pairs_host[2 * k], gy = pairs_host[2 * k + 1];
    if (gx < 0 || gx >= n_agents || gy < 0 || gy >= n_agents)
      return fail(DQLB200_ERR_ARG, "pair " + std::to_string(k) + ": agent index outside 0 .. " + std::to_string(n_agents - 1));
    if (h->pop_axis[(size_t)gx * R] == 1)
      return fail(DQLB200_ERR_ARG, "pair " + std::to_string(k) + ": x member " + std::to_string(gx) + " is a y-axis agent");
  }
  if (!h->tables || !h->pop_state) return fail(DQLB200_ERR_STATE, "tables / trainer state not bound");
  if (h->cfg.accel_mode != 0 || h->cfg.dynamics_model != 0)      // refuse rather than silently evaluate on the default model
    return fail(DQLB200_ERR_ARG, "the two-axis evaluator runs the first-order model with the analytic acceleration only (accel_mode = dynamics_model = 0)");
  if (episodes_per_pair <= 0) return DQLB200_OK;
  const long long blocks_per_pair = (episodes_per_pair + 255) / 256;
  if (blocks_per_pair * n_pairs > 0x7FFFFFFFLL) return fail(DQLB200_ERR_ARG, "episodes_per_pair * n_pairs exceeds one launch's grid");
  try {
    h->pairs_stage.assign(pairs_host, pairs_host + (size_t)n_pairs * 2);
  } catch (...) {
    return fail(DQLB200_ERR_STATE, "out of host memory");
  }
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  if (!h->pairs_read) CUDA_TRY(cudaEventCreateWithFlags(&h->pairs_read, cudaEventDisableTiming));
  if (n_pairs > h->d_pairs_cap) {
    CUDA_TRY(cudaEventSynchronize(h->pairs_read));      // the previous launch has read the old list
    CUDA_TRY(cudaFree(h->d_pairs));
    h->d_pairs = nullptr;
    h->d_pairs_cap = 0;
    CUDA_TRY(cudaMalloc(&h->d_pairs, (size_t)n_pairs * 2 * sizeof(int32_t)));
    h->d_pairs_cap = n_pairs;
  }
  CUDA_TRY(cudaStreamWaitEvent(s, h->pairs_read, 0));      // a launch on another stream may still read the list
  // from pageable memory the copy is staged before cudaMemcpyAsync returns, so neither pairs_host nor pairs_stage is read later
  CUDA_TRY(cudaMemcpyAsync(h->d_pairs, h->pairs_stage.data(), (size_t)n_pairs * 2 * sizeof(int32_t), cudaMemcpyHostToDevice, s));
  const unsigned grid = (unsigned)(blocks_per_pair * n_pairs);
  const auto* ps = (const dqlb200_population_state*)h->pop_state;
  if (h->kc_default)
    dql::eval_pairs_kernel<false><<<grid, 256, 0, s>>>(h->kc, *p, h->d_pop_params, (const uint32_t*)h->tables, ps, h->d_pairs, R,
                                                      (int)blocks_per_pair, first_episode, episodes_per_pair, (dqlb200_eval_stats*)stats_out);
  else
    dql::eval_pairs_kernel<true><<<grid, 256, 0, s>>>(h->kc, *p, h->d_pop_params, (const uint32_t*)h->tables, ps, h->d_pairs, R,
                                                     (int)blocks_per_pair, first_episode, episodes_per_pair, (dqlb200_eval_stats*)stats_out);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaEventRecord(h->pairs_read, s));
  return DQLB200_OK;
}

int dqlb200_transfer(dqlb200_handle* h, int step, float ratio, void* stream) {
  if (!h || !h->tables) return fail(DQLB200_ERR_STATE, "buffers not bound");
  if (step < 0 || step >= h->cfg.curriculum_steps) return fail(DQLB200_ERR_ARG, "step out of range");
  CUDA_TRY(cudaSetDevice(h->device));
  dql::transfer_kernel<<<h->cfg.n_populations, 256, 0, (cudaStream_t)stream>>>((uint32_t*)h->tables, h->cfg.n_populations,
                                                                             h->cfg.curriculum_steps, step, ratio);
  CUDA_TRY(cudaGetLastError());
  return DQLB200_OK;
}

int dqlb200_check_errors(dqlb200_handle* h, void* stream) {
  if (!h) return fail(DQLB200_ERR_ARG, "null handle");
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  // d_error: [0] facade kernels' flag, [1] OR of the populations' flags, [2] first offending population -- ONE reduction
  // launch and ONE 12-byte copy, whatever the number of populations
  if (h->pop_state) {
    const uint32_t init[2] = {0u, 0xFFFFFFFFu};
    CUDA_TRY(cudaMemcpyAsync(h->d_error + 1, init, sizeof(init), cudaMemcpyHostToDevice, s));
    dql::error_reduce_kernel<<<(h->cfg.n_populations + 255) / 256, 256, 0, s>>>((const dqlb200_population_state*)h->pop_state, h->cfg.n_populations,
                                                                                 h->d_error + 1);
    CUDA_TRY(cudaGetLastError());
  }
  uint32_t e[3] = {0u, 0u, 0u};
  CUDA_TRY(cudaMemcpyAsync(e, h->d_error, h->pop_state ? sizeof(e) : sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  if (e[0]) {
    CUDA_TRY(cudaMemsetAsync(h->d_error, 0, sizeof(uint32_t), s));
    return fail(DQLB200_ERR_DEVICE_FLAG, e[0] & 1u ? "Unexpected discretization case: NaN observation"
                                                   : (e[0] & 2u ? "Cannot check an empty state" : "Previous state missing"));
  }
  if (e[1]) return fail(DQLB200_ERR_DEVICE_FLAG, "population " + std::to_string(e[2]) + ": NaN observation (error_flags=" + std::to_string(e[1]) + ")");
  return DQLB200_OK;
}

int dqlb200_selftest_discretise(dqlb200_handle* h, int working_step, int variant, int64_t n, const float* obs, uint16_t* out_state, void* stream) {
  if (!h || !obs || !out_state) return fail(DQLB200_ERR_ARG, "null argument");
  if (working_step < 0 || working_step >= DQLB200_MAX_CURRICULUM) return fail(DQLB200_ERR_ARG, "working_step out of range");
  if (variant < 0 || variant > 3) return fail(DQLB200_ERR_ARG, "variant must be 0..3");
  if ((variant & 1) && !h->kc_default) return fail(DQLB200_ERR_STATE, "the compile-time-constant variants need the reference-default configuration");
  if (n <= 0) return DQLB200_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  const unsigned blocks = (unsigned)((n + 127) / 128);
  cudaStream_t s = (cudaStream_t)stream;
  switch (variant) {
    case 0: dql::selftest_discretise_kernel<false, true><<<blocks, 128, 0, s>>>(h->kc, working_step, n, obs, out_state); break;
    case 1: dql::selftest_discretise_kernel<true, true><<<blocks, 128, 0, s>>>(h->kc, working_step, n, obs, out_state); break;
    case 2: dql::selftest_discretise_kernel<false, false><<<blocks, 128, 0, s>>>(h->kc, working_step, n, obs, out_state); break;
    default: dql::selftest_discretise_kernel<true, false><<<blocks, 128, 0, s>>>(h->kc, working_step, n, obs, out_state); break;
  }
  CUDA_TRY(cudaGetLastError());
  return DQLB200_OK;
}

int dqlb200_shared_pack(dqlb200_handle* h, void* packed, void* stream) {
  if (!h || !h->tables || !h->pop_state || !packed) return fail(DQLB200_ERR_ARG, "null argument / not bound");
  CUDA_TRY(cudaSetDevice(h->device));
  const int R = h->cfg.replicas_per_population, n_agents = h->cfg.n_populations / R;
  const long long n = (long long)n_agents * DQLB200_MAX_CELLS;
  dql::shared_pack_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>((const uint32_t*)h->tables, (uint32_t*)packed,
                                                                                       (const dqlb200_population_state*)h->pop_state, n_agents, R);
  CUDA_TRY(cudaGetLastError());
  return DQLB200_OK;
}

int dqlb200_shared_apply(dqlb200_handle* h, void* snapshot, const void* gathered, int n_ranks, int pooled_promote_successes, void* stream) {
  if (!h || !h->tables || !h->pop_state || !snapshot || !gathered) return fail(DQLB200_ERR_ARG, "null argument / not bound");
  if (n_ranks < 1) return fail(DQLB200_ERR_ARG, "n_ranks < 1");
  CUDA_TRY(cudaSetDevice(h->device));
  const int R = h->cfg.replicas_per_population, n_agents = h->cfg.n_populations / R;
  if (R > 1 && !h->merge_snapshot) return fail(DQLB200_ERR_STATE, "replicated layout: bind the merge snapshot first (dqlb200_bind_merge_snapshot)");
  const long long n = (long long)n_agents * DQLB200_MAX_CELLS;
  dql::shared_apply_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>((uint32_t*)h->tables, (uint32_t*)snapshot,
                                                                                        R > 1 ? (uint32_t*)h->merge_snapshot : nullptr,
                                                                                        (const uint32_t*)gathered, n_ranks, (dqlb200_population_state*)h->pop_state,
                                                                                        n_agents, R, pooled_promote_successes, h->cfg.max_num_episodes);
  CUDA_TRY(cudaGetLastError());
  return DQLB200_OK;
}

// ---------------------------------------------------------------------------------------------
// The shared-table exchange as ONE call under the C-ABI (SURVEY.md 8b: allreduce_tables(h, ncclComm_t, stream)).  NCCL is not a
// link-time dependency of the library: ncclAllGather is looked up at run time, first among the symbols already loaded into the
// process (a caller that created a communicator has NCCL loaded -- PyTorch's bundled copy, or the system's), then in libnccl.so.2.
namespace {
typedef int (*nccl_all_gather_fn)(const void*, void*, size_t, int /*ncclDataType_t*/, void* /*ncclComm_t*/, cudaStream_t);
nccl_all_gather_fn find_nccl_all_gather() {
  static nccl_all_gather_fn fn = nullptr;
  if (fn) return fn;
  void* sym = dlsym(RTLD_DEFAULT, "ncclAllGather");
  if (!sym) {
    if (void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL)) sym = dlsym(lib, "ncclAllGather");
  }
  fn = reinterpret_cast<nccl_all_gather_fn>(sym);
  return fn;
}
}  // namespace

int dqlb200_shared_sync_nccl(dqlb200_handle* h, void* snapshot, void* packed, void* gathered, void* nccl_comm, int n_ranks,
                             int replica_promote_successes, int pooled_promote_successes, void* stream) {
  if (!h || !snapshot || !packed || !gathered || !nccl_comm) return fail(DQLB200_ERR_ARG, "null argument");
  if (n_ranks < 1) return fail(DQLB200_ERR_ARG, "n_ranks < 1");
  nccl_all_gather_fn all_gather = find_nccl_all_gather();
  if (!all_gather) return fail(DQLB200_ERR_STATE, "ncclAllGather not found: load NCCL (libnccl.so.2) into the process first");
  const int R = h->cfg.replicas_per_population, n_agents = h->cfg.n_populations / R;
  int rc;
  if (R > 1) {      // the local copies agree first; with a pooled promotion no rank decides alone
    if (!h->merge_snapshot) return fail(DQLB200_ERR_STATE, "replicated layout: bind the merge snapshot first (dqlb200_bind_merge_snapshot)");
    if ((rc = dqlb200_replica_merge(h, h->merge_snapshot, pooled_promote_successes > 0 ? 0 : replica_promote_successes, stream))) return rc;
  }
  if ((rc = dqlb200_shared_pack(h, packed, stream))) return rc;
  const size_t words = (size_t)n_agents * DQLB200_SHARED_WORDS;
  const int nccl_rc = all_gather(packed, gathered, words, /*ncclInt32*/ 2, nccl_comm, (cudaStream_t)stream);
  if (nccl_rc != 0) return fail(DQLB200_ERR_CUDA, "ncclAllGather failed with ncclResult_t " + std::to_string(nccl_rc));
  return dqlb200_shared_apply(h, snapshot, gathered, n_ranks, pooled_promote_successes, stream);
}

int dqlb200_mdp_facade_step(dqlb200_handle* h, int working_step, int ops, int64_t n, const double* obs, const uint8_t* contact,
                            const int8_t* action, double* mdp_state, uint16_t* out_state, uint8_t* out_code, double* out_reward,
                            void* stream) {
  if (!h || !mdp_state) return fail(DQLB200_ERR_ARG, "null argument");
  if (working_step < 0 || working_step >= DQLB200_MAX_CURRICULUM) return fail(DQLB200_ERR_ARG, "working_step out of range");
  if ((ops & (DQLB200_OP_OBSERVE | DQLB200_OP_CHECK)) && !obs) return fail(DQLB200_ERR_ARG, "obs required");
  if ((ops & DQLB200_OP_CHECK) && !contact) return fail(DQLB200_ERR_ARG, "contact required");
  if ((ops & DQLB200_OP_ACTION) && !action) return fail(DQLB200_ERR_ARG, "action required");
  if (n <= 0) return DQLB200_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  dql::facade_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(h->d_cfg, working_step, ops, n, obs, contact, action,
                                                                                   mdp_state, out_state, out_code, out_reward, h->d_error);
  CUDA_TRY(cudaGetLastError());
  return DQLB200_OK;
}

int dqlb200_bind_merge_snapshot(dqlb200_handle* h, void* snapshot) {
  if (!h) return fail(DQLB200_ERR_ARG, "null handle");
  if ((uintptr_t)snapshot & 3u) return fail(DQLB200_ERR_ARG, "misaligned snapshot");
  h->merge_snapshot = snapshot;
  h->merged_k = 0;
  return DQLB200_OK;
}

static int launch_merge(dqlb200_handle* h, void* snapshot, int pooled_promote_successes, cudaStream_t stream) {
  const int R = h->cfg.replicas_per_population;
  const dim3 grid((DQLB200_MAX_CELLS + 31) / 32 + 1, h->cfg.n_populations / R);     // one CTA per tile of 32 cells + one for the pooled counters
  if (R > 128) {      // 32 warps: 512 replicas per round trip
    const size_t smem = dql::merge_smem_bytes(32);      // > 48 KB: the attribute is set in dqlb200_create
    dql::replica_merge_kernel<32><<<grid, 1024, smem, stream>>>((uint32_t*)h->tables, (uint32_t*)snapshot, (dqlb200_population_state*)h->pop_state,
                                                              R, pooled_promote_successes, h->cfg.max_num_episodes);
  } else {
    dql::replica_merge_kernel<8><<<grid, 256, dql::merge_smem_bytes(8), stream>>>((uint32_t*)h->tables, (uint32_t*)snapshot,
                                                                                 (dqlb200_population_state*)h->pop_state, R,
                                                                                 pooled_promote_successes, h->cfg.max_num_episodes);
  }
  CUDA_TRY(cudaGetLastError());
  return DQLB200_OK;
}

int dqlb200_replica_merge(dqlb200_handle* h, void* snapshot, int pooled_promote_successes, void* stream) {
  if (!h || !h->tables || !h->pop_state || !snapshot) return fail(DQLB200_ERR_ARG, "null argument / not bound");
  if (h->cfg.replicas_per_population > 1 && snapshot != h->merge_snapshot)
    return fail(DQLB200_ERR_STATE, "snapshot is not the one bound with dqlb200_bind_merge_snapshot (train launches keep it current across transfers)");
  const int R = h->cfg.replicas_per_population;
  if (R < 1 || h->cfg.n_populations % R) return fail(DQLB200_ERR_STATE, "n_populations is not a multiple of replicas_per_population");
  CUDA_TRY(cudaSetDevice(h->device));
  return launch_merge(h, snapshot, pooled_promote_successes, (cudaStream_t)stream);
}

int dqlb200_train_merged(dqlb200_handle* h, int total_steps, int merge_every, int pooled_promote_successes, void* stream) {
  if (!h || !h->env_state || !h->tables || !h->pop_state) return fail(DQLB200_ERR_STATE, "buffers not bound");
  if (!h->merge_snapshot) return fail(DQLB200_ERR_STATE, "bind the merge snapshot first (dqlb200_bind_merge_snapshot)");
  if (total_steps < 0 || merge_every < 1) return fail(DQLB200_ERR_ARG, "total_steps >= 0 and merge_every >= 1 required");
  if (total_steps == 0) return DQLB200_OK;
  DQL_NEED_FILTER(h);
  CUDA_TRY(cudaSetDevice(h->device));
  if (!h->merged_ready) {
    CUDA_TRY(cudaStreamCreateWithFlags(&h->merged_stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreateWithFlags(&h->merged_in, cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&h->merged_out, cudaEventDisableTiming));
    h->merged_ready = true;
  }
  cudaStream_t ms = h->merged_stream, cs = (cudaStream_t)stream;
  const int n_full = total_steps / merge_every, rem = total_steps % merge_every;
  constexpr int MERGED_GRAPH_PAIRS = 16;
  if (n_full > 0 && (h->merged_k != merge_every || h->merged_promote != pooled_promote_successes || !h->merged_exec)) {
    // (train launch of merge_every steps, replica merge) pairs captured once and replayed: a pair is launch-bound for
    // populations of a few hundred CTAs (two ~5 us launches around ~20 us of work).  Two graphs: one pair, and
    // MERGED_GRAPH_PAIRS pairs back to back (one submission per 16 pairs; the kernels of a graph follow each other without
    // a host round trip).
    if (h->merged_exec) { cudaGraphExecDestroy(h->merged_exec); h->merged_exec = nullptr; }
    if (h->merged_exec_multi) { cudaGraphExecDestroy(h->merged_exec_multi); h->merged_exec_multi = nullptr; }
    for (int pairs : {1, MERGED_GRAPH_PAIRS}) {
      cudaGraph_t graph = nullptr;
      CUDA_TRY(cudaStreamBeginCapture(ms, cudaStreamCaptureModeThreadLocal));
      int rc = 0;
      for (int p = 0; p < pairs && !rc; ++p) {
        rc = launch_train(h, merge_every, nullptr, h->env_state, h->tables, h->pop_state, ms);
        if (!rc) rc = launch_merge(h, h->merge_snapshot, pooled_promote_successes, ms);
      }
      const cudaError_t ce = cudaStreamEndCapture(ms, &graph);
      if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
      CUDA_TRY(ce);
      CUDA_TRY(cudaGraphInstantiate(pairs == 1 ? &h->merged_exec : &h->merged_exec_multi, graph, 0));
      CUDA_TRY(cudaGraphDestroy(graph));
    }
    h->merged_k = merge_every;
    h->merged_promote = pooled_promote_successes;
  }
  CUDA_TRY(cudaEventRecord(h->merged_in, cs));
  CUDA_TRY(cudaStreamWaitEvent(ms, h->merged_in, 0));
  for (int i = 0; i < n_full / MERGED_GRAPH_PAIRS; ++i) CUDA_TRY(cudaGraphLaunch(h->merged_exec_multi, ms));
  for (int i = 0; i < n_full % MERGED_GRAPH_PAIRS; ++i) CUDA_TRY(cudaGraphLaunch(h->merged_exec, ms));
  if (rem) {
    int rc = launch_train(h, rem, nullptr, h->env_state, h->tables, h->pop_state, ms);
    if (!rc) rc = launch_merge(h, h->merge_snapshot, pooled_promote_successes, ms);
    if (rc) return rc;
  }
  CUDA_TRY(cudaEventRecord(h->merged_out, ms));
  CUDA_TRY(cudaStreamWaitEvent(cs, h->merged_out, 0));
  return DQLB200_OK;
}

int dqlb200_bench_table_rmw(dqlb200_handle* h, const uint16_t* cells, int64_t n_cells, int visits_per_thread, int threads, int blocks,
                            void* checksum_out, void* stream) {
  if (!h || !cells || !checksum_out) return fail(DQLB200_ERR_ARG, "null argument");
  if (n_cells < 1 || visits_per_thread < 1 || threads < 32 || threads > 1024 || blocks < 1) return fail(DQLB200_ERR_ARG, "bad launch shape");
  CUDA_TRY(cudaSetDevice(h->device));
  dql::table_rmw_roof_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(cells, n_cells, visits_per_thread, (unsigned long long*)checksum_out);
  CUDA_TRY(cudaGetLastError());
  return DQLB200_OK;
}

#ifdef DQL_TIMING
// probe builds only (tools/perf_probe_timeline.py): the %globaltimer stamps of the last train_kernel launch, [4096][8]
int dqlb200_debug_timing(unsigned long long* out, int n_words) {
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(cudaMemcpyFromSymbol(out, dql::dql_timing, (size_t)n_words * sizeof(unsigned long long)));
  return DQLB200_OK;
}
#endif

int dqlb200_bench_launch_floor(dqlb200_handle* h, int blocks, int threads, int smem_bytes, void* stream) {
  if (!h || blocks < 1 || threads < 32 || threads > 1024 || smem_bytes < 0 || smem_bytes > 227 * 1024) return fail(DQLB200_ERR_ARG, "bad launch shape");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaFuncSetAttribute(dql::launch_floor_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
  dql::launch_floor_kernel<<<blocks, threads, smem_bytes, (cudaStream_t)stream>>>(h->kc, (int*)h->d_error);
  CUDA_TRY(cudaGetLastError());
  return DQLB200_OK;
}

int dqlb200_selftest_division(dqlb200_handle* h, uint64_t* mismatches_out, void* stream) {
  if (!h || !mismatches_out) return fail(DQLB200_ERR_ARG, "null argument");
  CUDA_TRY(cudaSetDevice(h->device));
  unsigned long long* d = nullptr;
  CUDA_TRY(cudaMalloc(&d, 3 * sizeof(unsigned long long)));
  CUDA_TRY(cudaMemsetAsync(d, 0, 3 * sizeof(unsigned long long), (cudaStream_t)stream));
  dql::selftest_division_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(h->kc, d);
  CUDA_TRY(cudaGetLastError());
  unsigned long long v[3] = {0, 0, 0};
  CUDA_TRY(cudaMemcpyAsync(v, d, sizeof(v), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  CUDA_TRY(cudaFree(d));
  mismatches_out[0] = v[0];
  mismatches_out[1] = v[1];
  mismatches_out[2] = v[2];
  return DQLB200_OK;
}

int dqlb200_agent_facade(dqlb200_handle* h, int op, int64_t n, double* tables_f64, const int32_t* state, const int32_t* action,
                         const int32_t* next_state, const double* alpha, const double* reward, double gamma, int32_t* out_action,
                         void* stream) {
  if (!h || !tables_f64 || !state) return fail(DQLB200_ERR_ARG, "null argument");
  if (op == DQLB200_AGENT_PREDICT && !out_action) return fail(DQLB200_ERR_ARG, "out_action required");
  if (op == DQLB200_AGENT_UPDATE && (!action || !next_state || !alpha || !reward)) return fail(DQLB200_ERR_ARG, "update operands required");
  if (op == DQLB200_AGENT_TRANSFER && !alpha) return fail(DQLB200_ERR_ARG, "ratio required");
  if (op != DQLB200_AGENT_PREDICT && op != DQLB200_AGENT_UPDATE && op != DQLB200_AGENT_TRANSFER) return fail(DQLB200_ERR_ARG, "unknown op");
  if (n <= 0) return DQLB200_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  dql::agent_facade_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(op, n, tables_f64, h->cfg.curriculum_steps, state, action, next_state,
                                                            alpha, reward, gamma, out_action);
  CUDA_TRY(cudaGetLastError());
  return DQLB200_OK;
}

}  // extern "C"
