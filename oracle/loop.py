"""TEST INFRASTRUCTURE ONLY -- never imported by the product package.

The trainer hot loop (PKG/trainer.py:169-245 with PKG/landing_simulation_env.py
:167-282 ordering) re-hosted on the analytic stand-in, for ONE population of
``n_envs`` environments sharing one Q-table pair.  With n_envs == 1 it is the
reference loop step for step (SURVEY.md A.10); for n_envs > 1 it DEFINES the
batched semantics the CUDA kernel must reproduce ("S1", DESIGN.md):

  * every env selects its action and reads its bootstrap value from the tables
    as they were at the START of the global step (snapshot);
  * the Q/count updates are applied one after the other in env-index order on
    the live table, each with the learning rate of the live (pre-increment)
    count -- exactly as if the envs took turns in the reference loop;
  * finished episodes are appended to the success window in env order, the
    promotion test runs after every append (PKG/trainer.py:219-236) and takes
    effect at the end of the global step (all envs restart with a fresh MDP).

Pure Python / NumPy: use small n_envs * steps (seconds); the full-size runs are
checked through size-independent properties (tests/test_gpu_parity.py).
"""
from __future__ import annotations

from collections import deque
from dataclasses import dataclass, field
from typing import Optional, Tuple

import numpy as np

from . import philox
from .agent_oracle import SCALE_MODIFICATION, AgentOracle, exploration_rate, explore_threshold, state_id, transfer_ratio
from .dynamics import StandInDet, StandInParams, add_observation_noise
from .mdp_oracle import (MdpParams, TERMINAL_SUCCESS, TrainingMdpOracle)


@dataclass
class TrainerParams:
    """Defaults of Trainer.__init__ (PKG/trainer.py:20-44)."""
    curriculum_steps: int = 5
    successive_successful_episodes: int = 100
    success_rate: float = 0.96
    max_num_episodes: int = 50000
    alpha_min: float = 0.02949
    omega: float = 0.51
    gamma: float = 0.99
    t_max: float = 20
    f_ag: float = 22.92
    p_max: float = 4.5
    transfer_mode: str = "reference"      # "reference" (quirk Q7) | "paper"
    scale_modification_value: Tuple[float, ...] = SCALE_MODIFICATION     # transfer ratios of steps 1..4


class PopulationOracle:
    def __init__(self, n_envs: int, seed: int = 42, population: int = 0, w0: int = 0,
                 tp: Optional[TrainerParams] = None, mp: Optional[MdpParams] = None,
                 sp: Optional[StandInParams] = None, dtype=np.float32, agent: Optional[AgentOracle] = None,
                 self_promote: bool = True):
        self.self_promote = self_promote        # False: replica of a larger population (ReplicatedPopulationOracle decides)
        self.n, self.seed, self.pop = n_envs, seed, population
        self.tp = tp or TrainerParams()
        self.mp = mp or MdpParams()
        self.sp = sp or StandInParams(f_ag=self.tp.f_ag, p_max=self.tp.p_max)
        self.agent = agent or AgentOracle(self.tp.curriculum_steps, dtype, self.tp.alpha_min, self.tp.omega, self.tp.gamma)
        self.dyn = StandInDet(self.sp, n_envs)
        self.w = w0
        self.t = 0                      # global step index (Philox counter word 1)
        self.finished = False
        self.window = deque([], maxlen=self.tp.successive_successful_episodes)
        self.episodes_done = 0          # completed episodes in this curriculum step
        self.total_steps = 0
        self.total_episodes = 0
        self.total_successes = 0
        self.term_hist = np.zeros(9, np.int64)
        self.promotions = []            # (t, w) log
        self._fresh_mdps()
        self._reset_envs(range(self.n), birth=self.t)

    # -- helpers -------------------------------------------------------------------------------
    def _fresh_mdps(self):
        tp = self.tp
        self.mdps = [TrainingMdpOracle(self.w, tp.f_ag, tp.t_max, tp.p_max, self.mp, self.sp.v_z) for _ in range(self.n)]
        self.ep = np.zeros(self.n, np.int64)
        self.state = [None] * self.n

    def _reset_envs(self, idx, birth: int):
        """R1 + one hover period + first discrete_state (PKG/landing_simulation_env.py:167-243)."""
        idx = np.asarray(list(idx), dtype=np.int64)
        if idx.size == 0:
            return
        w0, w1, w2, _ = philox.draws(self.seed, self.pop, idx, birth, philox.PURPOSE_RESET)
        self.dyn.reset(idx, w0, w1, w2, normal_init=(self.w == 0))
        self.dyn.advance(np.zeros(idx.size, np.float32), idx, hover=True)
        rel_p, rel_v, rel_a, pitch, z, contact = self.dyn.observe(np.zeros(idx.size), idx)
        if self.sp.noise_pos_sd or self.sp.noise_vel_sd:
            n0, n1, _, _ = philox.draws(self.seed, self.pop, idx, birth, philox.PURPOSE_RESET_NOISE)
            rel_p, rel_v = add_observation_noise(self.sp, rel_p, rel_v, n0, n1)
        for k, i in enumerate(idx):
            m = self.mdps[i]
            m.reset()
            self.state[i] = m.observe(rel_p[k], rel_v[k], rel_a[k], pitch[k], z[k], contact[k])

    # -- one global step -----------------------------------------------------------------------
    def step(self, actions_override=None):
        """Advance every env by one agent step.  Returns a trace dict of per-env arrays."""
        n, tp, ag = self.n, self.tp, self.agent
        tr = dict(
            obs=np.zeros((n, 5), np.float32), contact=np.zeros(n, np.uint8), action=np.zeros(n, np.uint8),
            state=np.zeros(n, np.uint16), next_state=np.zeros(n, np.uint16), code=np.zeros(n, np.uint8),
            done=np.zeros(n, np.uint8), reward=np.zeros(n, np.float64), episode=np.zeros(n, np.int64),
        )
        if self.finished:
            return tr
        env = np.arange(n)
        d0, d1, d2, d3 = philox.draws(self.seed, self.pop, env, self.t, philox.PURPOSE_STEP)
        noisy = bool(self.sp.noise_pos_sd or self.sp.noise_vel_sd)
        snap_a, snap_b = ag.qa.copy(), ag.qb.copy()
        promote = advance = False
        finished_envs = []
        for i in range(n):
            m, s = self.mdps[i], self.state[i]
            eps = exploration_rate(int(self.ep[i]), self.w)
            explore = (int(d0[i]) >> 8) < explore_threshold(eps)
            greedy = int(np.argmax(np.add(snap_a[s], snap_b[s]) / 2))
            a = int((int(d1[i]) * 3) >> 32) if explore else greedy
            if actions_override is not None:
                a = int(actions_override[i])
            th_sp = m.act(a)
            self.dyn.advance(np.asarray([th_sp], np.float32), np.asarray([i]))
            rel_p, rel_v, rel_a, pitch, z, contact = (x[0] for x in self.dyn.observe(np.asarray([m.step_count + 1]), np.asarray([i])))
            if noisy:       # words z, w of the step draw (the table-pick draw of update() is consumed and ignored, quirk Q1)
                rel_p, rel_v = (x[0] for x in add_observation_noise(self.sp, rel_p, rel_v, d2[i:i + 1], d3[i:i + 1]))
            s2 = m.observe(rel_p, rel_v, rel_a, pitch, z, contact)
            code, done = m.check()
            r = m.reward()
            sa = s + (a,)
            ag.update(sa, s2, ag.alpha(sa), r, q_snapshot=snap_a)
            tr["obs"][i] = (rel_p, rel_v, rel_a, pitch, z)
            tr["contact"][i], tr["action"][i], tr["code"][i], tr["done"][i] = contact, a, code, done
            tr["state"][i], tr["next_state"][i], tr["reward"][i], tr["episode"][i] = state_id(s), state_id(s2), r, self.ep[i]
            self.total_steps += 1
            if done:
                ok = int(code == TERMINAL_SUCCESS)          # PKG/trainer.py:219-221
                self.window.append(ok)
                self.total_episodes += 1
                self.total_successes += ok
                self.term_hist[code] += 1
                self.episodes_done += 1
                if self.self_promote and sum(self.window) / tp.successive_successful_episodes > tp.success_rate:
                    promote = True
                if self.self_promote and self.episodes_done >= tp.max_num_episodes:
                    advance = True
                self.ep[i] += 1
                finished_envs.append(i)
            else:
                self.state[i] = s2
        self._reset_envs(finished_envs, birth=self.t + 1)
        if promote or advance:
            self._advance_curriculum(promote)
        self.t += 1
        return tr

    def _advance_curriculum(self, promoted: bool):
        """PKG/trainer.py:232-245: clear the window on promotion, transfer, next working step."""
        tp, ag = self.tp, self.agent
        if promoted:
            self.window.clear()
        self.promotions.append((self.t, self.w, promoted))
        if tp.transfer_mode == "reference":
            ag.transfer(self.w, transfer_ratio(self.w, tp.scale_modification_value))
        elif self.w + 1 < tp.curriculum_steps:
            ag.transfer(self.w + 1, transfer_ratio(self.w + 1, tp.scale_modification_value))
        self.w += 1
        self.episodes_done = 0
        if self.w >= tp.curriculum_steps:
            self.finished = True
            self.w = tp.curriculum_steps - 1
            return
        self._fresh_mdps()
        self._reset_envs(range(self.n), birth=self.t + 1)


class ReplicatedPopulationOracle:
    """Replica-merge mode (DESIGN.md section 3): ONE agent whose envs are split over R replicas.  Every replica runs
    the S1 semantics on its own copy of the tables; after every `merge_every` global steps the copies are merged:
    Q <- Q_snap + sum_r (Q_r - Q_snap) * dcount_r / sum_r dcount_r  (replica order, float32), count <- count_snap +
    sum_r dcount_r; a cell visited by one replica only keeps that replica's value.  The success windows are pooled:
    promotion when sum_r window_sum_r / (R * window_len) > success_rate, advance when the pooled finished episodes reach
    max_num_episodes; both take effect before the next global step.  With R = 1 the tables are never altered."""

    def __init__(self, replicas: int, envs_per_replica: int, seed: int = 42, first_population: int = 0, w0: int = 0,
                 tp: Optional[TrainerParams] = None, sp: Optional[StandInParams] = None, merge_every: int = 1):
        self.R, self.merge_every = replicas, merge_every
        self.tp = tp or TrainerParams()
        self.reps = [PopulationOracle(envs_per_replica, seed=seed, population=first_population + r, w0=w0, tp=self.tp, sp=sp,
                                      dtype=np.float32, self_promote=False) for r in range(replicas)]
        self.snap_q = self.reps[0].agent.qa.copy()
        self.snap_c = self.reps[0].agent.count.copy()
        self.steps = 0
        self.pending = 0

    def step(self):
        if self.pending:
            for rep in self.reps:
                if not rep.finished:
                    rep.t -= 1                       # _advance_curriculum uses birth = t + 1 = the next step index
                    rep._advance_curriculum(self.pending == 1)
                    rep.t += 1
            # the transfer acts on the merged table (all copies are identical here): the snapshot follows it
            self.snap_q = self.reps[0].agent.qa.copy()
            self.pending = 0
        out = [rep.step() for rep in self.reps]
        self.steps += 1
        if self.steps % self.merge_every == 0:
            self.merge()
        return out

    def merge(self):
        f32 = np.float32
        R = self.R
        dcs = [rep.agent.count - self.snap_c for rep in self.reps]
        tot = sum(dcs)
        visitors = sum((d > 0).astype(np.int64) for d in dcs)
        num = np.zeros(self.snap_q.shape, f32)
        single = self.snap_q.copy()
        for rep, d in zip(self.reps, dcs):
            hit = d > 0
            contrib = ((rep.agent.qa - self.snap_q).astype(f32) * d.astype(f32)).astype(f32)
            num = np.where(hit, (num + contrib).astype(f32), num)
            single = np.where(hit, rep.agent.qa, single)
        with np.errstate(invalid="ignore", divide="ignore"):
            mean = (self.snap_q + (num / tot.astype(f32)).astype(f32)).astype(f32)
        q_new = np.where(visitors == 1, single, np.where(visitors > 1, mean, self.snap_q)).astype(f32)
        c_new = self.snap_c + tot
        for rep in self.reps:
            rep.agent.qa[...] = q_new
            rep.agent.count[...] = c_new
        self.snap_q, self.snap_c = q_new.copy(), c_new.copy()
        live = all((not rep.finished) for rep in self.reps)
        if live and not self.pending:
            successes = sum(sum(rep.window) for rep in self.reps)
            episodes = sum(rep.episodes_done for rep in self.reps)
            if successes / (R * self.tp.successive_successful_episodes) > self.tp.success_rate:
                self.pending = 1
            elif episodes >= self.tp.max_num_episodes:
                self.pending = 2


def eval_episode(policy, seed: int, population: int, episode_id: int, sp: StandInParams,
                 tp: Optional[TrainerParams] = None, mp: Optional[MdpParams] = None, w: int = 4):
    """One greedy SimulationMdp episode (scripts/simulation.py:48-63 + PKG/landing_simulation_env.py:327-340).
    ``policy`` maps a 5-tuple state to an action.  Returns a list of per-step dict rows (row 0 = reset)."""
    from .mdp_oracle import SimulationMdpOracle
    tp = tp or TrainerParams()
    mdp = SimulationMdpOracle(w, tp.f_ag, tp.t_max, tp.p_max, mp)
    dyn = StandInDet(sp, 1)
    idx = np.asarray([0])
    w0, w1, w2, _ = philox.draws(seed, population, np.asarray([episode_id]), 0, philox.PURPOSE_RESET)
    dyn.reset(idx, w0, w1, w2, normal_init=False, simulation=True)
    dyn.advance(np.zeros(1, np.float32), hover=True)
    rp, rv, ra, pit, z, c = (x[0] for x in dyn.observe(np.zeros(1)))
    sx, _ = mdp.observe(rp, rv, ra, pit, z, c)
    rows = [dict(obs=(rp, rv, ra, pit, z), contact=c, action=255, state=state_id(sx), code=0, done=0)]
    done, k = False, 0
    while not done:
        a = policy(sx)
        th = mdp.act(a)
        dyn.advance(np.asarray([th], np.float32))
        k += 1
        rp, rv, ra, pit, z, c = (x[0] for x in dyn.observe(np.asarray([k])))
        sx, _ = mdp.observe(rp, rv, ra, pit, z, c)
        code, done = mdp.check()
        rows.append(dict(obs=(rp, rv, ra, pit, z), contact=c, action=a, state=state_id(sx), code=code, done=int(done)))
    return rows


def mirrored_policy(policy_lut):
    """Policy of the y agent derived from an x policy by symmetry (roll convention a_y = -g tan(roll)): with roll' = -roll
    the y axis obeys the x dynamics, so act as the x policy would in the state with the mirrored angle index and swap the
    increase/decrease actions.  policy_lut: uint8[945] indexed by state id."""
    lut = np.asarray(policy_lut, np.uint8)
    out = np.empty_like(lut)
    swap = np.asarray([1, 0, 2], np.uint8)
    for sid in range(len(lut)):
        rest, th = divmod(sid, 7)
        out[sid] = swap[lut[rest * 7 + (6 - th)]]
    return out


def eval_episode_2d(policy_x, policy_y, seed: int, stream: int, episode_id: int, p2, tp: Optional[TrainerParams] = None,
                    mp: Optional[MdpParams] = None, w: int = 4):
    """One greedy two-axis SimulationMdp episode (scripts/simulation.py:48-63): both agents predict every step
    (PKG/double_q_learning.py:119-124); the y action moves the roll set-point only if p2.y_action_enabled (the reference
    has that branch disabled, PKG/mdp.py:863-876).  policy_x / policy_y: uint8[945] LUTs by state id.  Rows: per-step dicts
    (row 0 = reset)."""
    from .dynamics import StandIn2D
    from .mdp_oracle import SimulationMdpOracle
    tp = tp or TrainerParams()
    mdp = SimulationMdpOracle(w, tp.f_ag, tp.t_max, tp.p_max, mp)
    dyn = StandIn2D(p2, 1)
    w0, w1, w2, w3 = philox.draws(seed, stream, np.asarray([episode_id]), 0, philox.PURPOSE_RESET)
    dyn.reset(w0, w1, w2, w3)
    dyn.advance(np.zeros(1, np.float32), np.zeros(1, np.float32))

    def look(k):
        o = {kk: v[0] for kk, v in dyn.observe(np.asarray([k])).items()}
        sx, sy = mdp.observe(o["rel_p_x"], o["rel_v_x"], o["rel_a_x"], o["pitch"], o["z"], o["contact"],
                             o["rel_p_y"], o["rel_v_y"], o["rel_a_y"], o["roll"])
        return o, sx, sy

    o, sx, sy = look(0)
    rows = [dict(obs=o, action_x=255, action_y=255, state_x=state_id(sx), state_y=state_id(sy), code=0, done=0)]
    sp_y, done, k = 0.0, False, 0
    prm = mdp.prm
    while not done:
        ax, ay = int(policy_x[state_id(sx)]), int(policy_y[state_id(sy)])
        sp_x = mdp.act(ax)
        if p2.y_action_enabled:
            if ay == 0:
                sp_y = min(sp_y + prm.delta_theta, prm.theta_max)
            elif ay == 1:
                sp_y = max(sp_y - prm.delta_theta, -prm.theta_max)
        dyn.advance(np.asarray([sp_x], np.float32), np.asarray([sp_y], np.float32))
        k += 1
        o, sx, sy = look(k)
        code, done = mdp.check()
        rows.append(dict(obs=o, action_x=ax, action_y=ay, state_x=state_id(sx), state_y=state_id(sy), code=code, done=int(done)))
    return rows
