"""Batched device driver: owns the torch tensors (device memory handles) and calls the C-ABI.

One ``Engine`` = one CUDA device = ``n_populations`` independent agents (Q-table pairs), each with
``envs_per_population`` environments; one CTA per population (csrc/train_kernel.cuh: train_kernel).
This replaces the `while not done` loop of Trainer.curriculum_training (PKG/trainer.py:187-245)."""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np
import torch

from . import _ffi
from . import constants as K


class Engine:
    def __init__(self, n_populations: int, envs_per_population: int, *, device: int = 0, threads_per_block: int = 256,
                 seeds: Optional[Sequence[int]] = None, population_ids: Optional[Sequence[int]] = None,
                 v_mp: Optional[Sequence[float]] = None, alpha_variants: Optional[Sequence[tuple]] = None,
                 alpha_index: Optional[Sequence[int]] = None, replicas_per_population: int = 1,
                 axes: Optional[Sequence[str]] = None, r_mp: Optional[Sequence[float]] = None,
                 mp: Optional[K.MdpParameters] = None, dp: Optional[K.DynamicsParameters] = None,
                 tp: Optional[K.TrainerParameters] = None):
        if not torch.cuda.is_available():
            raise _ffi.Dqlb200Error("no CUDA device: dql_multirotor_landing_b200 has no CPU fallback")
        self.lib = _ffi.load()
        self.mp, self.dp, self.tp = mp or K.MdpParameters(), dp or K.DynamicsParameters(), tp or K.TrainerParameters()
        self.P, self.n_p, self.device_index = n_populations, envs_per_population, device
        self.device = torch.device("cuda", device)
        alpha_variants = list(alpha_variants or [(self.tp.alpha_min, self.tp.omega)])
        self.R = replicas_per_population
        self.cfg = K.build_config(n_populations, envs_per_population, threads_per_block, self.mp, self.dp, self.tp,
                                  n_alpha_luts=len(alpha_variants), replicas_per_population=replicas_per_population)
        luts = np.concatenate([K.alpha_lut(a, o) for a, o in alpha_variants]).astype(np.float32)
        seeds = list(seeds) if seeds is not None else [42] * n_populations
        population_ids = list(population_ids) if population_ids is not None else list(range(n_populations))
        v_mp = list(v_mp) if v_mp is not None else [self.dp.v_mp] * n_populations
        # platform amplitude per population (default: DynamicsParameters.r_mp).  Decoupled per-axis training under the
        # reference's "eight" trajectory (PKG/moving_platform.py:92-111: x = r cos wt, y = r sin wt cos wt = (r/2) sin 2wt)
        # is a parameter choice: x agent (r, v), y agent (r / 2, v) -- see eight_axis_platforms().
        r_mp = list(r_mp) if r_mp is not None else [self.dp.r_mp] * n_populations
        alpha_index = list(alpha_index) if alpha_index is not None else [0] * n_populations
        # axis of every agent: "x" (pitch, a = +g tan) or "y" (roll, a = -g tan in the reference's ENU frame; training_y.sh)
        axes = list(axes) if axes is not None else ["x"] * n_populations
        if any(a not in ("x", "y") for a in axes):
            raise ValueError("axes entries must be 'x' or 'y'")
        self.axes = axes
        pps = (K.PopulationParams * n_populations)()
        for p in range(n_populations):
            dphase, r, rw, rw2 = K.platform_constants(r_mp[p], v_mp[p], self.mp.f_ag, self.dp.n_sub)
            pps[p] = K.PopulationParams(seeds[p] & 0xFFFFFFFF, (seeds[p] >> 32) & 0xFFFFFFFF, population_ids[p], dphase,
                                        r, rw, rw2, alpha_index[p], np.float32(self.dp.g if axes[p] == "x" else -self.dp.g),
                                        0 if axes[p] == "x" else 1)
        self.handle = C.c_void_p()
        _ffi.check(self.lib.dqlb200_create(C.byref(self.cfg), luts.ctypes.data_as(C.POINTER(C.c_float)), pps, device,
                                           C.byref(self.handle)))
        n = n_populations * envs_per_population
        self.n_total = n
        with torch.cuda.device(self.device):
            # [population][tile][3][32 envs][16 B]: tiles of 32 envs, 1536 contiguous bytes each (csrc/env_state.cuh)
            self.tiles_per_population = (envs_per_population + 31) // 32
            self.env_state = torch.zeros(self.lib.dqlb200_env_state_bytes(n_populations, envs_per_population) // 4, dtype=torch.int32, device=self.device)
            self.tables = torch.zeros((n_populations, 3, K.MAX_CELLS), dtype=torch.int32, device=self.device)
            self.pop_state = torch.zeros(n_populations * C.sizeof(K.PopulationState), dtype=torch.uint8, device=self.device)
        _ffi.check(self.lib.dqlb200_bind(self.handle, self.env_state.data_ptr(), self.tables.data_ptr(), self.pop_state.data_ptr()))
        self.filter_state = None
        if self.cfg.accel_mode != 0:      # SURVEY 8f-3: per-env state of the acceleration estimator {x, P, v_ref, n}, 16 B/env
            with torch.cuda.device(self.device):
                fs = torch.zeros((n, 4), dtype=torch.int32, device=self.device)
                fs[:, 1] = 0x3F800000     # P = 1.0f (PKG/filters.py:16): a simulator that has not published yet
            self.filter_state = fs
            _ffi.check(self.lib.dqlb200_bind_filter_state(self.handle, fs.data_ptr()))
        self.dynamics_state = None
        if self.cfg.dynamics_model != 0:  # SURVEY 8f-4: [2][n] x 16 B {omega, z, v_z, integral}, {e1, f1, f2, f3}; dqlb200_reset initialises it
            with torch.cuda.device(self.device):
                self.dynamics_state = torch.zeros((2, n, 4), dtype=torch.float32, device=self.device)
                self.dynamics_state[0, :, 1] = float(self.cfg.z_init)
                self.dynamics_state[0, :, 3] = float(self.cfg.pid_i0)
            _ffi.check(self.lib.dqlb200_bind_dynamics_state(self.handle, self.dynamics_state.data_ptr()))
        self._trace_keep = None
        self.merge_snapshot = None       # replica-merge mode: [n_groups][3][MAX_CELLS] merged tables of the last merge
        self.pooled_promote = K.promote_threshold(self.tp.successive_successful_episodes * self.R, self.tp.success_rate)

    def close(self):
        if getattr(self, "handle", None):
            self.lib.dqlb200_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------------------------------
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def reset(self, initial_step: int = 0):
        _ffi.check(self.lib.dqlb200_reset(self.handle, initial_step, self._stream()))

    def train(self, k_steps: int, trace: bool = False, action_override: Optional[np.ndarray] = None):
        """k_steps fused global steps for every population.  With trace=True returns per-step arrays [k][n_total]."""
        tr = None
        out = None
        if trace or action_override is not None:
            n, dev = self.n_total, self.device
            out = dict(
                obs=torch.zeros((k_steps, n, 5), dtype=torch.float32, device=dev),
                reward=torch.zeros((k_steps, n), dtype=torch.float64, device=dev),
                action=torch.zeros((k_steps, n), dtype=torch.uint8, device=dev),
                code=torch.zeros((k_steps, n), dtype=torch.uint8, device=dev),
                done=torch.zeros((k_steps, n), dtype=torch.uint8, device=dev),
                contact=torch.zeros((k_steps, n), dtype=torch.uint8, device=dev),
                state=torch.zeros((k_steps, n), dtype=torch.int16, device=dev),
                next_state=torch.zeros((k_steps, n), dtype=torch.int16, device=dev),
                episode=torch.zeros((k_steps, n), dtype=torch.int32, device=dev),
            )
            ov = None
            if action_override is not None:
                ov = torch.as_tensor(np.ascontiguousarray(action_override, dtype=np.int8).reshape(k_steps, n), device=dev)
            tr = K.Trace(*[out[k].data_ptr() for k in ("obs", "reward", "action", "code", "done", "contact", "state",
                                                       "next_state", "episode")], ov.data_ptr() if ov is not None else None)
            self._trace_keep = (out, ov)
        _ffi.check(self.lib.dqlb200_train(self.handle, k_steps, C.byref(tr) if tr is not None else None, self._stream()))
        if out is not None:
            torch.cuda.synchronize(self.device)
            return {k: v.cpu().numpy() for k, v in out.items()}
        return None

    def train_host(self, k_steps: int, env_state_host: torch.Tensor, tables_host: torch.Tensor, pop_state_host: torch.Tensor,
                   table_levels: int = 0, filter_state_host: Optional[torch.Tensor] = None,
                   dynamics_state_host: Optional[torch.Tensor] = None):
        """End-to-end call with pinned HOST buffers (copies in, k_steps, copies out, synchronises).  table_levels = L > 0: only
        the table levels 0 .. L-1 travel (the caller's promise that no population is promoted beyond them inside the call; the
        library checks it afterwards); 0 = every level.  With accel_mode / dynamics_model the per-env extension state travels too
        (filter_state_host [n, 4], dynamics_state_host [2, n, 4] float32, the layouts of the bound device buffers)."""
        if filter_state_host is None and dynamics_state_host is None:
            _ffi.check(self.lib.dqlb200_train_host(self.handle, k_steps, env_state_host.data_ptr(), tables_host.data_ptr(),
                                                   pop_state_host.data_ptr(), int(table_levels), self._stream()))
            return
        ptr = lambda t: t.data_ptr() if t is not None else None
        _ffi.check(self.lib.dqlb200_train_host_ext(self.handle, k_steps, env_state_host.data_ptr(), tables_host.data_ptr(),
                                                   pop_state_host.data_ptr(), ptr(filter_state_host), ptr(dynamics_state_host),
                                                   int(table_levels), self._stream()))

    # ------------------------------------------------------------------------------------------
    # replica-merge mode: R consecutive populations are replicas of one agent (more envs than one CTA holds)
    def _ensure_merge_snapshot(self):
        if self.merge_snapshot is None:
            self.merge_snapshot = self.tables[:: self.R].clone().contiguous()
            _ffi.check(self.lib.dqlb200_bind_merge_snapshot(self.handle, self.merge_snapshot.data_ptr()))

    def replica_merge(self):
        self._ensure_merge_snapshot()
        _ffi.check(self.lib.dqlb200_replica_merge(self.handle, self.merge_snapshot.data_ptr(), self.pooled_promote, self._stream()))

    def train_merged(self, total_steps: int, merge_every: int = 1, graph: bool = True):
        """total_steps global steps, merging the replicas of every agent after each `merge_every` steps.  graph=True submits
        the whole loop from C as replays of one captured CUDA graph (dqlb200_train_merged); graph=False alternates the two
        entry points from Python (same result, one ctypes call per launch)."""
        self._ensure_merge_snapshot()
        if graph:
            _ffi.check(self.lib.dqlb200_train_merged(self.handle, total_steps, merge_every, self.pooled_promote, self._stream()))
            return
        done = 0
        while done < total_steps:
            k = min(merge_every, total_steps - done)
            self.train(k)
            self.replica_merge()
            done += k

    def set_group_tables(self, group: int, qa: np.ndarray, qb: np.ndarray, count: np.ndarray):
        for r in range(self.R):
            self.set_tables(group * self.R + r, qa, qb, count)
        self.merge_snapshot = None
        _ffi.check(self.lib.dqlb200_bind_merge_snapshot(self.handle, None))

    def bench_table_rmw(self, cells: np.ndarray, visits_per_thread: int = 256, threads: int = 128, blocks: int = 888, reps: int = 5) -> dict:
        """Measurement aid (SURVEY 8d): rate of UNORDERED shared-memory read-modify-writes on a recorded sequence of visited
        cells (uint16, cell = state * 3 + action), two RMW per visit.  Returns visits/s (CUDA events, best of reps)."""
        dev = self.device
        d_cells = torch.as_tensor(np.ascontiguousarray(cells, np.uint16).view(np.int16), device=dev)
        chk = torch.zeros(1, dtype=torch.int64, device=dev)
        best = float("inf")
        for _ in range(reps + 1):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            _ffi.check(self.lib.dqlb200_bench_table_rmw(self.handle, d_cells.data_ptr(), d_cells.numel(), visits_per_thread, threads, blocks,
                                                        chk.data_ptr(), self._stream()))
            b.record()
            torch.cuda.synchronize(dev)
            best = min(best, a.elapsed_time(b) * 1e-3)
        visits = visits_per_thread * threads * blocks
        return {"visits_per_s": visits / best, "rmw_per_s": 2 * visits / best, "visits": visits, "seconds": best,
                "threads": threads, "blocks": blocks}

    # ------------------------------------------------------------------------------------------
    # un-fused entry points: the reference's loop body as separate operators (PKG/trainer.py:191-212)
    def env_reset(self, working_step: int = 0, birth: int = 0, fresh_mdp: bool = True):
        """env.reset() for every env (dqlb200_env_reset); returns the states (int16 tensor)."""
        st = torch.zeros(self.n_total, dtype=torch.int16, device=self.device)
        _ffi.check(self.lib.dqlb200_env_reset(self.handle, working_step, birth, None, int(fresh_mdp), 0, st.data_ptr(), self._stream()))
        return st

    def agent_select(self, working_step: int, t: int):
        """agent.guess(state, exploration_rate(episode, step)) for every env; returns (actions uint8, states int16)."""
        act = torch.zeros(self.n_total, dtype=torch.uint8, device=self.device)
        st = torch.zeros(self.n_total, dtype=torch.int16, device=self.device)
        _ffi.check(self.lib.dqlb200_agent_select(self.handle, working_step, t, act.data_ptr(), st.data_ptr(), self._stream()))
        return act, st

    def env_step(self, working_step: int, t: int, actions: torch.Tensor, auto_reset: bool = True):
        """env.step(action) for every env (dqlb200_env_step); returns dict(state, next_state, reward, code, done) of tensors."""
        dev, n = self.device, self.n_total
        out = dict(state=torch.zeros(n, dtype=torch.int16, device=dev), next_state=torch.zeros(n, dtype=torch.int16, device=dev),
                   reward=torch.zeros(n, dtype=torch.float64, device=dev), code=torch.zeros(n, dtype=torch.uint8, device=dev),
                   done=torch.zeros(n, dtype=torch.uint8, device=dev))
        a8 = actions.to(torch.int8)
        _ffi.check(self.lib.dqlb200_env_step(self.handle, working_step, t, a8.data_ptr(), int(auto_reset), 0, out["state"].data_ptr(),
                                             out["reward"].data_ptr(), out["code"].data_ptr(), out["done"].data_ptr(), None, None, None,
                                             out["next_state"].data_ptr(), self._stream()))
        self._keep = a8
        return out

    def agent_update(self, states: torch.Tensor, actions: torch.Tensor, next_states: torch.Tensor, rewards: torch.Tensor):
        """agent.update(state + (action,), next_state, alpha(count), gamma, reward) for every env, S1 order (dqlb200_agent_update)."""
        _ffi.check(self.lib.dqlb200_agent_update(self.handle, states.data_ptr(), actions.data_ptr(), next_states.data_ptr(), rewards.data_ptr(),
                                                 self._stream()))

    def selftest_division(self) -> int:
        """Exhaustive device check of the fast float64 division (all fp32 numerators); returns the mismatch count."""
        out = (C.c_uint64 * 3)()
        _ffi.check(self.lib.dqlb200_selftest_division(self.handle, out, self._stream()))
        self.selftest_one_step_mismatches = int(out[1])
        return int(out[0]) + int(out[2])

    def check_errors(self):
        _ffi.check(self.lib.dqlb200_check_errors(self.handle, self._stream()))

    # ------------------------------------------------------------------------------------------
    # tables <-> DoubleQLearningAgent arrays (float64, shape (cs,3,3,3,7,3); PKG/double_q_learning.py:38-40)
    def set_tables(self, population: int, qa: np.ndarray, qb: np.ndarray, count: np.ndarray):
        cs = self.tp.curriculum_steps
        host = np.zeros((3, K.MAX_CELLS), np.uint32)
        host[0, : cs * K.CELLS_PER_LEVEL] = np.asarray(qa, np.float64).astype(np.float32).reshape(-1).view(np.uint32)
        host[1, : cs * K.CELLS_PER_LEVEL] = np.asarray(qb, np.float64).astype(np.float32).reshape(-1).view(np.uint32)
        host[2, : cs * K.CELLS_PER_LEVEL] = np.asarray(count, np.float64).reshape(-1).astype(np.uint32)
        self.tables[population].copy_(torch.from_numpy(host.view(np.int32)))

    def get_tables(self, population: int, dtype=np.float64):
        cs = self.tp.curriculum_steps
        host = self.tables[population].cpu().numpy().view(np.uint32)
        shape = (cs, 3, 3, 3, 7, 3)
        n = cs * K.CELLS_PER_LEVEL
        qa = host[0, :n].view(np.float32).astype(dtype).reshape(shape)
        qb = host[1, :n].view(np.float32).astype(dtype).reshape(shape)
        count = host[2, :n].astype(np.float64).reshape(shape)
        return qa, qb, count

    def population_state(self) -> np.ndarray:
        raw = self.pop_state.cpu().numpy()
        return raw.view(K.POPULATION_STATE_DTYPE).copy()

    def selftest_discretise(self, obs: np.ndarray, working_step: int, variant: int = 0) -> np.ndarray:
        """Device discretisation (csrc/dqlb200_device.cuh: discretise_cuts) of fp32 observations [n][4] = rel_p, rel_v, rel_a, pitch
        -> state ids; variant: see dqlb200_selftest_discretise (include/dqlb200.h)."""
        o = torch.as_tensor(np.ascontiguousarray(obs, np.float32).reshape(-1, 4), device=self.device)
        out = torch.zeros(o.shape[0], dtype=torch.int16, device=self.device)
        _ffi.check(self.lib.dqlb200_selftest_discretise(self.handle, int(working_step), int(variant), o.shape[0], o.data_ptr(), out.data_ptr(),
                                                        self._stream()))
        return out.cpu().numpy().astype(np.uint16)

    def set_episode_index(self, episode: int):
        """Test hook: set every env's per-curriculum-step episode index (word C.y of the state)."""
        v = self.env_state.view(self.P, self.tiles_per_population, 3, 32, 4)
        v[:, :, 2, :, 1] = int(episode)

    # ------------------------------------------------------------------------------------------
    def eval_greedy(self, policy: np.ndarray, n_episodes: int, *, population: int = 0, first_episode: int = 0,
                    working_step: int = 4, trace_steps: int = 0):
        """Greedy SimulationMdp episodes (scripts/simulation.py:48-63).  policy: uint8 action per state id (945)."""
        dev = self.device
        pol = np.zeros(K.MAX_CURRICULUM * K.STATES_PER_LEVEL, np.uint8)
        pol[: len(policy)] = policy
        d_pol = torch.as_tensor(pol, device=dev)
        stats = torch.zeros(C.sizeof(K.EvalStats), dtype=torch.uint8, device=dev)
        tr, out = None, None
        if trace_steps > 0:
            out = dict(
                obs=torch.zeros((trace_steps, n_episodes, 5), dtype=torch.float32, device=dev),
                action=torch.zeros((trace_steps, n_episodes), dtype=torch.uint8, device=dev),
                code=torch.zeros((trace_steps, n_episodes), dtype=torch.uint8, device=dev),
                done=torch.zeros((trace_steps, n_episodes), dtype=torch.uint8, device=dev),
                contact=torch.zeros((trace_steps, n_episodes), dtype=torch.uint8, device=dev),
                state=torch.zeros((trace_steps, n_episodes), dtype=torch.int16, device=dev),
                next_state=torch.zeros((trace_steps, n_episodes), dtype=torch.int16, device=dev),
            )
            tr = K.Trace(out["obs"].data_ptr(), None, out["action"].data_ptr(), out["code"].data_ptr(), out["done"].data_ptr(),
                         out["contact"].data_ptr(), out["state"].data_ptr(), out["next_state"].data_ptr(), None, None)
        _ffi.check(self.lib.dqlb200_eval_greedy(self.handle, population, d_pol.data_ptr(), first_episode, n_episodes, working_step,
                                                stats.data_ptr(), C.byref(tr) if tr is not None else None, trace_steps, self._stream()))
        torch.cuda.synchronize(dev)
        return _eval_result(K.EvalStats.from_buffer_copy(stats.cpu().numpy().tobytes()), out)

    def eval_agents(self, episodes_per_agent: int, *, working_step: Optional[int] = None, first_episode: int = 0,
                    return_policies: bool = False) -> dict:
        """Greedy SimulationMdp episodes of every agent's current policy, built on the device from the live float32 tables
        (dqlb200_eval_agents): one launch, one copy back, one synchronisation.  Agent g is replica group g (population g * R);
        working_step None = each agent's live working step.  Agent g's episodes are those of
        eval_greedy(<its float32 greedy LUT>, episodes_per_agent, population=g * R, first_episode=..., working_step=...).
        Returns NumPy arrays over the agents: episodes [A], steps [A], termination_hist [A, 9], success_rate [A] (goal or
        contact, the reference's two "SUCCESS" codes) and, with return_policies, policy [A, 945] uint8."""
        A = self.P // self.R
        stats_bytes, n_states = A * C.sizeof(K.EvalStats), K.MAX_CURRICULUM * K.STATES_PER_LEVEL
        buf = torch.zeros(stats_bytes + (A * n_states if return_policies else 0), dtype=torch.uint8, device=self.device)
        w = -1 if working_step is None else int(working_step)
        _ffi.check(self.lib.dqlb200_eval_agents(self.handle, w, int(first_episode), int(episodes_per_agent), buf.data_ptr(),
                                                buf.data_ptr() + stats_bytes if return_policies else None, self._stream()))
        host = buf.cpu().numpy()          # synchronises the stream
        st = host[:stats_bytes].view(np.uint64).reshape(A, 11).astype(np.int64)
        res = dict(episodes=st[:, 0], steps=st[:, 1], termination_hist=st[:, 2:])
        hist = res["termination_hist"]            # codes 2 (goal) and 3 (contact); a SimulationMdp episode only ends in 3
        res["success_rate"] = (hist[:, 2] + hist[:, 3]) / np.maximum(res["episodes"], 1)
        if return_policies:
            res["policy"] = host[stats_bytes:].reshape(A, n_states).copy()
        return res

    def eval_platforms(self, episodes_per_agent: int, platforms: Sequence[Sequence[float]], *, working_step: Optional[int] = None,
                       first_episode: int = 0) -> dict:
        """eval_agents under each of a list of platform motions (dqlb200_eval_agents_platforms): every agent x every platform x
        episodes_per_agent greedy SimulationMdp episodes from the live float32 tables, one launch, one copy back, one
        synchronisation.  platforms: (r_mp, v_mp) pairs, converted as the Engine converts its own (platform_constants).  Cell
        (g, c) is eval_greedy(<g's float32 LUT>, episodes_per_agent, population=g * R, first_episode=..., working_step=...) on an
        Engine whose population g * R flies platform c; episode i starts from the same offset and platform phase under every
        platform.  working_step None = each agent's live working step.  Returns NumPy arrays: platforms [C, 2], episodes [A, C],
        steps [A, C], termination_hist [A, C, 9], success_rate [A, C] (goal or contact, as eval_agents)."""
        pl = K.platform_motions(platforms)
        n = len(pl)
        host = (K.Platform * n)()
        for c, (r, v) in enumerate(pl):
            host[c] = K.Platform(*K.platform_constants(r, v, self.mp.f_ag, self.dp.n_sub))
            if not all(np.isfinite([host[c].r, host[c].rw, host[c].rw2])) or not host[c].r > 0:
                raise ValueError(f"platform {c} (r_mp={r}, v_mp={v}) does not fit float32")
        A = self.P // self.R
        stats_bytes = A * n * C.sizeof(K.EvalStats)
        buf = torch.zeros(stats_bytes, dtype=torch.uint8, device=self.device)
        w = -1 if working_step is None else int(working_step)
        _ffi.check(self.lib.dqlb200_eval_agents_platforms(self.handle, w, int(first_episode), int(episodes_per_agent), host, n,
                                                          buf.data_ptr(), self._stream()))
        st = buf.cpu().numpy().view(np.uint64).reshape(A, n, 11).astype(np.int64)      # the copy synchronises the stream
        res = dict(platforms=pl, episodes=st[:, :, 0], steps=st[:, :, 1], termination_hist=st[:, :, 2:])
        hist = res["termination_hist"]
        res["success_rate"] = (hist[:, :, 2] + hist[:, :, 3]) / np.maximum(res["episodes"], 1)
        return res

    def eval_greedy_2d(self, policy_x: np.ndarray, policy_y: np.ndarray, n_episodes: int, *, two_axis: Optional[K.TwoAxisParameters] = None,
                       seed: int = 42, stream_id: int = 0, first_episode: int = 0, working_step: int = 4, trace_steps: int = 0):
        """Greedy two-axis SimulationMdp episodes: agent_x and agent_y both predict every step (scripts/simulation.py:48-63).
        policy_x / policy_y: uint8 action per state id.  Defaults reproduce the reference (y action disabled)."""
        dev = self.device
        ta = two_axis or K.TwoAxisParameters()
        prm = K.eval2d_params(ta, self.dp, self.mp.f_ag, seed, stream_id, working_step)

        def lut(p):
            full = np.zeros(K.MAX_CURRICULUM * K.STATES_PER_LEVEL, np.uint8)
            full[: len(p)] = p
            return torch.as_tensor(full, device=dev)

        d_px, d_py = lut(policy_x), lut(policy_y)
        stats = torch.zeros(C.sizeof(K.EvalStats), dtype=torch.uint8, device=dev)
        tr, out = None, None
        if trace_steps > 0:
            u8 = lambda: torch.zeros((trace_steps, n_episodes), dtype=torch.uint8, device=dev)
            i16 = lambda: torch.zeros((trace_steps, n_episodes), dtype=torch.int16, device=dev)
            out = dict(obs=torch.zeros((trace_steps, n_episodes, 9), dtype=torch.float32, device=dev), action_x=u8(), action_y=u8(),
                       code=u8(), done=u8(), contact=u8(), state_x=i16(), state_y=i16())
            tr = K.Trace2D(*[out[k].data_ptr() for k in ("obs", "action_x", "action_y", "code", "done", "contact", "state_x", "state_y")])
        _ffi.check(self.lib.dqlb200_eval_greedy_2d(self.handle, C.byref(prm), d_px.data_ptr(), d_py.data_ptr(), first_episode, n_episodes,
                                                   stats.data_ptr(), C.byref(tr) if tr is not None else None, trace_steps, self._stream()))
        torch.cuda.synchronize(dev)
        return _eval_result(K.EvalStats.from_buffer_copy(stats.cpu().numpy().tobytes()), out)

    def eval_pairs(self, episodes_per_pair: int, pairs: Sequence[Sequence[int]], *, two_axis: Optional[K.TwoAxisParameters] = None,
                   seed: int = 42, stream_id: int = 0, first_episode: int = 0, working_step: Optional[int] = None) -> dict:
        """Greedy two-axis SimulationMdp episodes of every (x agent, y agent) pair, both LUTs built on the device from the live
        float32 tables (dqlb200_eval_pairs): one launch, one copy back, one synchronisation.  pairs: (gx, gy) agent indices
        (agent g = replica group g, population g * R); gx must be an x agent.  gy a y agent flies y with its own policy, gy an
        x agent with the mirror image of its policy (mirrored_policy).  working_step None = the lower of the two members' live
        working steps.  Pair k's episodes are those of eval_greedy_2d(<lut_x>, <lut_y>, episodes_per_pair, two_axis=...,
        seed=..., stream_id=..., first_episode=..., working_step=...), the same initial conditions for every pair.  Returns
        NumPy arrays over the pairs: pairs [K, 2], episodes [K], steps [K], termination_hist [K, 9], success_rate [K] (goal or
        contact)."""
        pr = np.asarray(pairs, dtype=np.int64)
        if pr.size == 0:
            pr = pr.reshape(0, 2)
        if pr.ndim != 2 or pr.shape[1] != 2:
            raise ValueError("pairs must be a sequence of (gx, gy) agent indices")
        if pr.size and (pr.min() < np.iinfo(np.int32).min or pr.max() > np.iinfo(np.int32).max):
            raise ValueError("agent index out of range")
        host_pairs = np.ascontiguousarray(pr, dtype=np.int32)
        n = len(host_pairs)
        w = -1 if working_step is None else int(working_step)
        prm = K.eval2d_params(two_axis or K.TwoAxisParameters(), self.dp, self.mp.f_ag, seed, stream_id, w)
        stats_bytes = n * C.sizeof(K.EvalStats)
        buf = torch.zeros(max(stats_bytes, 1), dtype=torch.uint8, device=self.device)
        _ffi.check(self.lib.dqlb200_eval_pairs(self.handle, C.byref(prm), host_pairs.ctypes.data, n, int(first_episode),
                                               int(episodes_per_pair), buf.data_ptr(), self._stream()))
        host = buf.cpu().numpy()          # synchronises the stream
        st = host[:stats_bytes].view(np.uint64).reshape(n, 11).astype(np.int64)
        res = dict(pairs=pr, episodes=st[:, 0], steps=st[:, 1], termination_hist=st[:, 2:])
        hist = res["termination_hist"]            # codes 2 (goal) and 3 (contact), as eval_agents
        res["success_rate"] = (hist[:, 2] + hist[:, 3]) / np.maximum(res["episodes"], 1)
        return res


def eight_axis_platforms(r: float = 3.0, v: float = 0.8):
    """(r_mp, v_mp) of the x and the y agent for decoupled training under the reference's "eight" platform trajectory
    (PKG/moving_platform.py:92-111, r_x = r_y = 3, t_x = 0.8): each axis sees a sinusoid -- x: amplitude r, peak speed
    v = r w; y: r sin(wt) cos(wt) = (r / 2) sin(2 w t), amplitude r / 2, peak speed (r / 2)(2 w) = v.  The start phase is
    random per episode, so cos versus sin makes no difference."""
    return (r, v), (r / 2.0, v)


def _eval_result(st, out):
    res = dict(episodes=int(st.episodes), steps=int(st.steps), termination_hist=[int(x) for x in st.termination_hist])
    if out is not None:
        res["trace"] = {k: v.cpu().numpy() for k, v in out.items()}
    return res


def mirrored_policy(policy: np.ndarray) -> np.ndarray:
    """y-axis policy derived from an x policy by symmetry (a_y = -g tan(roll)): act as the x policy would in the state with
    the mirrored angle index and swap increase/decrease.  For a y agent trained on its own (BASELINE config 4) use its own
    greedy_policy instead."""
    lut = np.asarray(policy, np.uint8).reshape(-1, 7)
    return np.asarray([1, 0, 2], np.uint8)[lut[:, ::-1]].reshape(-1)


def greedy_policy(qa: np.ndarray, qb: np.ndarray) -> np.ndarray:
    """DoubleQLearningAgent.predict for every state (PKG/double_q_learning.py:119-124), evaluated in the
    tables' own precision (float64 for the committed .npy files) -> uint8 action LUT indexed by state id."""
    avg = np.add(qa, qb) / 2
    return np.argmax(avg.reshape(-1, 3), axis=1).astype(np.uint8)
