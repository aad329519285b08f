"""GPU parity (-m gpu) at NON-default parameters.  Every other parity test runs the reference-default MDP constants; here the
divisors, reward weights, set-point lattice, production-compatible trainer constants, discount, a three-step curriculum and the
episode-length limits of the packed env state are each held to the oracle bit for bit (traces, tables, counters), and the fast
division and the cut-table discretisation are checked exhaustively / at their edges under the same parameters."""
import dataclasses

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from dql_multirotor_landing_b200 import constants as K
from oracle.agent_oracle import AgentOracle, state_id
from oracle.dynamics import StandInParams, derive
from oracle.loop import PopulationOracle, ReplicatedPopulationOracle, TrainerParams
from oracle.mdp_oracle import (TERMINAL_SUCCESS, TERMINAL_TIMEOUT, TERMINATION_STRINGS, MdpParams, TrainingMdpOracle,
                               discretise, linspace7)

PROMOTING = dict(success_rate=0.15, successive_successful_episodes=6, max_num_episodes=90)
NO_PROMOTION = dict(success_rate=2.0, max_num_episodes=10 ** 12)


def oracle_params(mp: K.MdpParameters, tp: K.TrainerParameters, dp: K.DynamicsParameters):
    """(TrainerParams, MdpParams, StandInParams) of the oracle for the library's parameter objects.  Every field is carried over
    by name, so a field one side does not know raises here instead of letting the oracle run other dynamics."""
    otp = TrainerParams(**{**dataclasses.asdict(tp), "scale_modification_value": tuple(tp.scale_modification_value)},
                        t_max=mp.t_max, f_ag=mp.f_ag, p_max=mp.p_max)
    omp = MdpParams(**{k: v for k, v in dataclasses.asdict(mp).items() if k not in ("f_ag", "t_max", "p_max")})
    d = dataclasses.asdict(dp)
    d["v_z"] = d.pop("v_z_train")
    d.pop("v_z_sim")                     # the greedy evaluation's set-point; training never reads it
    osp = StandInParams(f_ag=mp.f_ag, p_max=mp.p_max, **d)
    return otp, omp, osp


def _assert_same_constants(cfg, otp, omp, osp):
    """The configuration the kernels got and the oracle's parameters describe the same MDP and stand-in."""
    d = derive(osp)
    for name in ("h", "half_h2", "k_theta", "c_d", "z_init", "z_touch", "half_platform", "sigma_x"):
        assert getattr(cfg, name) == float(getattr(d, name)), name
    assert (cfg.p_max_f, cfg.two_p_max_f, cfg.dz_train, cfg.n_sub) == (float(d.p_max), float(d.two_p_max), float(d.dz), d.n_sub)
    assert (cfg.p_max, cfg.v_max, cfg.a_max, cfg.theta_max, cfg.delta_theta) == (otp.p_max, omp.v_max, omp.a_max, omp.theta_max, omp.delta_theta)
    assert (cfg.w_p, cfg.w_v, cfg.w_theta, cfg.minimum_altitude) == (omp.w_p, omp.w_v, omp.w_theta, omp.minimum_altitude)
    assert cfg.timeout_threshold == otp.t_max * otp.f_ag and cfg.f_ag == otp.f_ag and cfg.gamma == np.float32(otp.gamma)
    assert [cfg.transfer_ratio[k] for k in range(1, 5)] == [float(np.float32(r)) for r in otp.scale_modification_value]


def _engine(P, n_p, mp, tp, dp=None, **kw):
    from dql_multirotor_landing_b200.engine import Engine
    return Engine(P, n_p, mp=mp, tp=tp, dp=dp or K.DynamicsParameters(), **kw)


def _assert_trace_step(tr, t, o, sl, where):
    assert np.array_equal(tr["obs"][t, sl].view(np.uint32), o["obs"].view(np.uint32)), where
    for key in ("action", "code", "done"):
        assert np.array_equal(tr[key][t, sl], o[key]), (where, key)
    assert np.array_equal(tr["next_state"][t, sl].astype(np.uint16), o["next_state"]), where
    assert np.array_equal(tr["reward"][t, sl], o["reward"]), where          # float64, bit for bit


def _assert_tables_and_counters(eng, p, pop):
    qa, qb, cnt = eng.get_tables(p, np.float32)
    assert np.array_equal(qa.view(np.uint32), pop.agent.qa.view(np.uint32))
    assert np.array_equal(qb.view(np.uint32), pop.agent.qb.view(np.uint32))
    assert np.array_equal(cnt, pop.agent.count)
    ps = eng.population_state()[p]
    promoted_at = [0] * K.MAX_CURRICULUM
    for t, w, _ in pop.promotions:
        promoted_at[w] = t + 1
    assert (int(ps["working_step"]), int(ps["finished"]), int(ps["total_episodes"])) == (pop.w, int(pop.finished), pop.total_episodes)
    assert list(ps["termination_hist"]) == list(pop.term_hist)
    assert [int(x) for x in ps["promoted_at"]] == promoted_at


def _random_tables(seed):
    """[3][MAX_CELLS] uint32: Q_a, Q_b (float32 bits) and counts, non-zero at every level."""
    rng = np.random.default_rng(seed)
    t = np.empty((3, K.MAX_CELLS), np.uint32)
    t[0] = rng.standard_normal(K.MAX_CELLS).astype(np.float32).view(np.uint32)
    t[1] = rng.standard_normal(K.MAX_CELLS).astype(np.float32).view(np.uint32)
    t[2] = rng.integers(1, 2000, size=K.MAX_CELLS)
    return t


def _load_agent(agent, t):
    n = agent.qa.size
    agent.qa[...] = t[0, :n].view(np.float32).reshape(agent.qa.shape)
    agent.qb[...] = t[1, :n].view(np.float32).reshape(agent.qb.shape)
    agent.count[...] = t[2, :n].astype(np.float64).reshape(agent.count.shape)


def run_parity(mp, tp, *, default_instance, n_envs=70, tpb=64, seed=3, chunks=(1, 63, 200, 136), min_w=2,
               tables=None, dp=None, action_override=None):
    """The trace instance against PopulationOracle step by step, then tables and trainer counters, then the non-trace instance
    (production or generic, as `default_instance` says) from the same start must leave the same tables, env and trainer state."""
    dp = dp or K.DynamicsParameters()
    otp, omp, osp = oracle_params(mp, tp, dp)
    eng = _engine(1, n_envs, mp, tp, dp, threads_per_block=tpb, seeds=[seed])
    _assert_same_constants(eng.cfg, otp, omp, osp)
    assert eng.lib.dqlb200_uses_default_instance(eng.handle) == int(default_instance)
    agent = AgentOracle(otp.curriculum_steps, np.float32, otp.alpha_min, otp.omega, otp.gamma)
    if tables is not None:
        eng.tables[0].copy_(torch.from_numpy(tables.view(np.int32)))
        _load_agent(agent, tables)
    eng.reset(0)
    pop = PopulationOracle(n_envs, seed=seed, population=0, w0=0, dtype=np.float32, tp=otp, mp=omp, sp=osp, agent=agent)
    t0, rows = 0, []
    for chunk in chunks:
        ov = None if action_override is None else action_override[t0:t0 + chunk]
        tr = eng.train(chunk, trace=True, action_override=ov)
        for t in range(chunk):
            if pop.finished:
                break
            o = pop.step(None if ov is None else ov[t])
            _assert_trace_step(tr, t, o, slice(None), t0 + t)
            rows.append(o)
        t0 += chunk
    eng.check_errors()
    _assert_tables_and_counters(eng, 0, pop)
    assert pop.w >= min_w, "the run should cross the promotions it is meant to test"
    eng2 = _engine(1, n_envs, mp, tp, dp, threads_per_block=tpb, seeds=[seed])
    if tables is not None:
        eng2.tables[0].copy_(torch.from_numpy(tables.view(np.int32)))
    eng2.reset(0)
    t0 = 0
    for chunk in chunks:
        if action_override is None:
            eng2.train(chunk)
        else:      # forced actions need the trace instance; it is the same instance the first run used
            eng2.train(chunk, action_override=action_override[t0:t0 + chunk])
        t0 += chunk
    eng2.check_errors()
    torch.cuda.synchronize()
    assert torch.equal(eng2.tables, eng.tables) and torch.equal(eng2.env_state, eng.env_state)
    assert torch.equal(eng2.pop_state, eng.pop_state)
    return eng, pop, rows


# ------------------------------------------------------------------------------------------------------------------------------
# (a) - (e): one parameter group at a time away from the defaults
# ------------------------------------------------------------------------------------------------------------------------------
CASES = {
    # divisors: the generic instance, the two-step division, sigma_x and the fly-zone cuts of the reset law
    "divisors": (dict(p_max=5.0, v_max=3.0), {}, False, 64),
    # shaping weights and the altitude cut
    "weights": (dict(w_p=-80.0, w_v=-12.0, w_theta=-2.0, minimum_altitude=0.3), {}, False, 64),
    # 63 reachable set-points (the default lattice has 33): the largest shared-memory set-point table
    "setpoints": (dict(theta_max=0.3, delta_theta=0.047), {}, False, 256),
    # constants the production instance reads from run-time tables
    "production": (dict(beta=0.3, sigma_a=0.5, a_max=1.5, w_dur=-5.0, w_succ=3.0, w_fail=-2.0),
                   dict(alpha_min=0.05, omega=0.6, scale_modification_value=(0.9, 0.7, 1.1, 0.6)), True, 64),
    "discount": ({}, dict(gamma=0.9), False, 64),
}


@pytest.mark.parametrize("case", list(CASES))
def test_nondefault_parameters_vs_oracle(case):
    mp_kw, tp_kw, default_instance, tpb = CASES[case]
    mp = K.MdpParameters(**mp_kw)
    tp = K.TrainerParameters(**PROMOTING, **tp_kw)
    if case == "setpoints":
        assert K.build_config(1, 70, tpb, mp).n_setpoints == 63
    run_parity(mp, tp, default_instance=default_instance, tpb=tpb)


# ------------------------------------------------------------------------------------------------------------------------------
# (f) three curriculum steps: the in-kernel transfer reads slot (w - 1 + 3) % 3, never a level beyond the curriculum
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["reference", "paper"])
def test_three_curriculum_steps_from_loaded_tables(mode):
    t0 = _random_tables(11)
    tp = K.TrainerParameters(curriculum_steps=3, transfer_mode=mode, **PROMOTING)
    eng, pop, _ = run_parity(K.MdpParameters(), tp, default_instance=True, chunks=(1, 40, 100), tables=t0)
    assert pop.finished and int(eng.population_state()[0]["finished"]) == 1
    assert [w for _, w, _ in pop.promotions] == [0, 1, 2]
    after = eng.tables.cpu().numpy().view(np.uint32)[0]
    assert np.array_equal(after[:, 3 * K.CELLS_PER_LEVEL:], t0[:, 3 * K.CELLS_PER_LEVEL:])    # levels 3 and 4: untouched


def test_three_curriculum_steps_replica_merge():
    """Replica-merge mode (R = 3 CTAs of one agent, merged after every step) with three curriculum steps from loaded tables."""
    R, n_r, steps = 3, 40, 200
    t0 = _random_tables(12)
    tp = K.TrainerParameters(curriculum_steps=3, **PROMOTING)
    eng = _engine(R, n_r, K.MdpParameters(), tp, threads_per_block=32, seeds=[5] * R, population_ids=list(range(R)), replicas_per_population=R)
    assert eng.lib.dqlb200_uses_default_instance(eng.handle) == 1
    for r in range(R):
        eng.tables[r].copy_(torch.from_numpy(t0.view(np.int32)))
    eng.reset(0)
    otp, _, osp = oracle_params(K.MdpParameters(), tp, K.DynamicsParameters())
    ora = ReplicatedPopulationOracle(R, n_r, seed=5, tp=otp, sp=osp, merge_every=1)
    for rep in ora.reps:
        _load_agent(rep.agent, t0)
    ora.snap_q, ora.snap_c = ora.reps[0].agent.qa.copy(), ora.reps[0].agent.count.copy()
    eng.train_merged(60, 1)
    eng.train_merged(steps - 60, 1)
    eng.check_errors()
    for _ in range(steps):
        ora.step()
    assert all(rep.finished for rep in ora.reps), "the run should reach the end of the curriculum"
    ps = eng.population_state()
    t = eng.tables.cpu().numpy().view(np.uint32)
    for r in range(R):
        qa, qb, cnt = eng.get_tables(r, np.float32)
        rep = ora.reps[r]
        assert np.array_equal(cnt, rep.agent.count), r
        assert np.array_equal(qa.view(np.uint32), rep.agent.qa.view(np.uint32)), r
        assert np.array_equal(qb.view(np.uint32), rep.agent.qb.view(np.uint32)), r
        assert (ps[r]["working_step"], ps[r]["finished"], ps[r]["total_episodes"]) == (rep.w, 1, rep.total_episodes)
        assert np.array_equal(t[r, :, 3 * K.CELLS_PER_LEVEL:], t0[:, 3 * K.CELLS_PER_LEVEL:]), r


# ------------------------------------------------------------------------------------------------------------------------------
# (g) episode lengths at the limits of the packed env state (9-bit step counter, 5-bit goal counter)
# ------------------------------------------------------------------------------------------------------------------------------
def _episode_lengths(rows, code):
    """Lengths of the episodes that ended with `code` (rows: the oracle's per-step dicts)."""
    n = len(rows[0]["done"])
    since, out = np.zeros(n, np.int64), []
    for o in rows:
        since += 1
        for i in np.nonzero(o["done"])[0]:
            if o["code"][i] == code:
                out.append(int(since[i]))
            since[i] = 0
    return out


def test_longest_countable_episode_times_out_like_the_oracle():
    """t_max * f_ag = 510.9: timeout_steps = 511, the largest count the 9-bit field holds.  Some hovering envs live that long."""
    mp = K.MdpParameters(t_max=22.29)
    assert K.build_config(1, 1, 32, mp).timeout_steps == 511
    n_envs, steps = 64, 530
    acts = np.full((steps, n_envs), 2, np.int8)
    _, _, rows = run_parity(mp, K.TrainerParameters(**NO_PROMOTION), default_instance=False, n_envs=n_envs, chunks=(1, 300, 229),
                            min_w=0, action_override=acts)
    lengths = _episode_lengths(rows, TERMINAL_TIMEOUT)
    assert lengths and all(n == 511 for n in lengths), lengths


def test_longest_countable_goal_succeeds_like_the_oracle():
    """f_ag = 31: success_steps = 31, the largest count the 5-bit goal counter holds (t_max = 16: 496 steps)."""
    mp = K.MdpParameters(f_ag=31.0, t_max=16)
    cfg = K.build_config(1, 1, 32, mp)
    assert (cfg.success_steps, cfg.timeout_steps) == (31, 496)
    _, _, rows = run_parity(mp, K.TrainerParameters(**NO_PROMOTION), default_instance=False, chunks=(1, 99, 100), min_w=0)
    assert _episode_lengths(rows, TERMINAL_SUCCESS), "no goal success in the run"


@pytest.mark.parametrize("mp_kw,limit", [(dict(t_max=22.33), "exceeds 511,"), (dict(f_ag=32.0, t_max=15), "exceeds 31,")])
def test_episode_lengths_the_env_state_cannot_count_are_refused(tmp_path, mp_kw, limit):
    """timeout_steps = 512 (t_max * f_ag = 511.8) and success_steps = 32 (f_ag = 32, 480 steps) would overflow the packed counters;
    binding an env state to such a configuration fails, so neither an Engine nor a Trainer runs it."""
    from dql_multirotor_landing_b200 import _ffi
    from dql_multirotor_landing_b200.trainer import Trainer
    mp = K.MdpParameters(**mp_kw)
    with pytest.raises(_ffi.Dqlb200Error, match=limit):
        _engine(1, 32, mp, K.TrainerParameters(), threads_per_block=32)
    trainer = Trainer(num_envs=32, threads_per_block=32, save_path=tmp_path / "run", verbose=False, **mp_kw)
    with pytest.raises(_ffi.Dqlb200Error, match=limit):
        trainer.curriculum_training()


def test_facade_counts_episodes_past_the_packed_limit():
    """The single-object TrainingMdp keeps its step count in float64, not in the packed env state: t_max = 25 (573 steps) works
    and times out at step 573 exactly like the oracle, every state and float64 reward equal on the way."""
    from dql_multirotor_landing_b200.mdp import ContinuousObservation, TrainingMdp, state_id as sid
    from dql_multirotor_landing_b200.msg import Observation
    m = TrainingMdp(0, 22.92, 25)
    ref = TrainingMdpOracle(0, 22.92, 25, 4.5, MdpParams())
    rng = np.random.default_rng(2)
    obs = np.stack([rng.uniform(2.0, 4.0, 600), rng.uniform(-0.5, 0.5, 600), rng.uniform(-0.5, 0.5, 600),
                    rng.uniform(-0.3, 0.3, 600), rng.uniform(1.0, 4.0, 600)], axis=1).astype(np.float32).astype(np.float64)
    acts = rng.integers(0, 3, 600)

    def look(k):
        p, v, a, th, z = obs[k]
        return ContinuousObservation(Observation(rel_p_x=p, rel_v_x=v, rel_a_x=a), th, 0.0, z)

    m.reset()
    ref.reset()
    assert sid(m.discrete_state(look(0))) == state_id(ref.observe(*obs[0][:4], obs[0][4], False))
    for k in range(1, 600):
        assert m.continuous_action(int(acts[k])).pitch == ref.act(int(acts[k]))
        assert sid(m.discrete_state(look(k))) == state_id(ref.observe(*obs[k][:4], obs[k][4], False)), k
        info = m.check()
        code, done = ref.check()
        assert m.reward() == ref.reward(), k
        assert ("Termination condition" in info) == done, k
        if done:
            break
    assert k == 573 and code == TERMINAL_TIMEOUT
    assert info["Termination condition"] == TERMINATION_STRINGS[TERMINAL_TIMEOUT] and info["Number of steps"] == 573


# ------------------------------------------------------------------------------------------------------------------------------
# the fast division and the discretisation cuts at other divisors, against float64 directly
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mp_kw", [dict(p_max=5.0, v_max=3.0), dict(p_max=3.7, v_max=4.1), dict(p_max=6.3, v_max=2.9, theta_max=0.33)])
def test_two_step_division_is_exact_for_every_fp32_numerator(mp_kw):
    """div_f32_by_const with the second correction step (any divisor but the defaults) == IEEE float64 division for every finite fp32
    numerator and both divisors; div_f64_by_const by theta_max on 2^32 float64 numerators."""
    eng = _engine(1, 1, K.MdpParameters(**mp_kw), K.TrainerParameters(), threads_per_block=32)
    assert eng.lib.dqlb200_uses_default_instance(eng.handle) == 0
    assert eng.selftest_division() == 0


def _probe_rows(cfg, w, scale, rng):
    """fp32 observations [n][4]: every finite cut of working step w and every angle cut with +-3 ulp around it in its own
    coordinate (the others random), plus random values over several magnitudes."""
    cuts = cfg.cuts[w]
    per_q = [[cuts.lvl_lo[q][i] for i in range(4)] + [cuts.lvl_hi[q][i] for i in range(4)] for q in range(2)] + [[]]
    for q in range(3):
        per_q[q] += [cuts.bin1[q][lv] for lv in range(5)] + [cuts.bin2[q][lv] for lv in range(5)]
    per_q.append([cfg.angle_cut[i] for i in range(6)])
    rows = []
    for q, values in enumerate(per_q):
        for c in {np.float32(v) for v in values if np.isfinite(v)}:
            x = np.float32(c)
            probes = [x]
            lo = hi = x
            for _ in range(3):
                lo, hi = np.nextafter(lo, np.float32(-np.inf)), np.nextafter(hi, np.float32(np.inf))
                probes += [lo, hi]
            base = (rng.standard_normal((len(probes), 4)) * scale).astype(np.float32)
            base[:, q] = probes
            rows.append(base)
    rnd = rng.standard_normal((3000, 4)) * scale * 10.0 ** rng.uniform(-3, 0.5, size=(3000, 1))
    rows.append(rnd.astype(np.float32))
    return np.concatenate(rows)


@pytest.mark.parametrize("case", ["divisors", "setpoints", "production"])
def test_discretisation_edges_at_nondefault_cuts(case):
    """The cut tables the host derives for other parameters, on the device (run-time cuts, bounded and unbounded level loop), against
    the reference's float64 discretisation (oracle.mdp_oracle.discretise) under the same parameters, working steps 0..4."""
    mp = K.MdpParameters(**CASES[case][0])
    otp, omp, _ = oracle_params(mp, K.TrainerParameters(), K.DynamicsParameters())
    eng = _engine(1, 1, mp, K.TrainerParameters(), threads_per_block=32)
    # the production-compatible case also runs the production instances' variants (compile-time angle cuts, staged cut table)
    default_instance = eng.lib.dqlb200_uses_default_instance(eng.handle) == 1
    assert default_instance == CASES[case][2]
    angles = linspace7(omp.theta_max, omp.n_theta)
    scale = np.asarray([mp.p_max, mp.v_max, mp.a_max, mp.theta_max]) * 0.6
    rng = np.random.default_rng(7)
    for w in range(5):
        obs = _probe_rows(eng.cfg, w, scale, rng)
        want = np.asarray([state_id(discretise(w, omp, otp.p_max, angles, *(float(x) for x in row))) for row in obs], np.uint16)
        for variant in ((0, 1, 2, 3) if default_instance else (0, 2)):
            got = eng.selftest_discretise(obs, w, variant)
            bad = np.nonzero(got != want)[0]
            assert bad.size == 0, (w, variant, obs[bad[:4]], got[bad[:4]], want[bad[:4]])
