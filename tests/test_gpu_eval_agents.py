"""GPU tests (-m gpu) of Engine.eval_agents / dqlb200_eval_agents: every agent's greedy policy, built on the device from its live
float32 tables, evaluated in one launch.  The main contract: agent g's episodes are those of eval_greedy for population g * R
under the float32 first-max LUT of its tables, episode for episode."""
import ctypes as C
import pathlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from dql_multirotor_landing_b200 import _ffi
from dql_multirotor_landing_b200 import constants as K

ROOT = pathlib.Path(__file__).resolve().parent.parent
N_STATES = K.MAX_CURRICULUM * K.STATES_PER_LEVEL


def _engine(P, n_p=32, **kw):
    from dql_multirotor_landing_b200.engine import Engine
    kw.setdefault("threads_per_block", 32)
    return Engine(P, n_p, **kw)


def _random_tables(seed):
    """[3][MAX_CELLS] uint32: Q_a, Q_b (float32 bits) and counts at every level."""
    rng = np.random.default_rng(seed)
    t = np.empty((3, K.MAX_CELLS), np.uint32)
    t[0] = rng.standard_normal(K.MAX_CELLS).astype(np.float32).view(np.uint32)
    t[1] = rng.standard_normal(K.MAX_CELLS).astype(np.float32).view(np.uint32)
    t[2] = rng.integers(1, 2000, size=K.MAX_CELLS)
    return t


def _assets_tables():
    qa, qb, cnt = (np.load(ROOT / "assets" / f) for f in ("Q_table_a.npy", "Q_table_b.npy", "state_action_count.npy"))
    t = np.zeros((3, K.MAX_CELLS), np.uint32)
    t[0] = qa.astype(np.float32).reshape(-1).view(np.uint32)
    t[1] = qb.astype(np.float32).reshape(-1).view(np.uint32)
    t[2] = cnt.reshape(-1).astype(np.uint32)
    return t


def _put(eng, p, t):
    eng.tables[p].copy_(torch.from_numpy(t.view(np.int32)))


def f32_lut(t, cs=K.MAX_CURRICULUM):
    """NumPy float32 first-max greedy LUT of [3][MAX_CELLS] table words: (Q_a + Q_b) * 0.5f, rounded per operation."""
    n = cs * K.CELLS_PER_LEVEL
    qa, qb = t[0, :n].view(np.float32).reshape(-1, 3), t[1, :n].view(np.float32).reshape(-1, 3)
    avg = (qa + qb) * np.float32(0.5)
    assert avg.dtype == np.float32
    lut = np.zeros(N_STATES, np.uint8)
    lut[: cs * K.STATES_PER_LEVEL] = np.argmax(avg, axis=1)          # argmax: the first maximum
    return lut


def _row(res, g):
    return (int(res["episodes"][g]), int(res["steps"][g]), [int(x) for x in res["termination_hist"][g]])


def _single(eng, lut, n, p, first, w):
    r = eng.eval_greedy(lut, n, population=p, first_episode=first, working_step=w)
    return (r["episodes"], r["steps"], r["termination_hist"])


SWEEP = dict(seeds=[3, 17, 42, 99, 2 ** 33 + 5, 1234], population_ids=[0, 7, 2, 11, 4, 5], v_mp=[1.6, 0.8, 1.2, 0.4, 1.6, 1.0],
             r_mp=[2.0, 3.0, 1.5, 2.0, 2.5, 1.0], axes=["x", "y", "x", "y", "y", "x"])


@pytest.mark.parametrize("generic", [False, True])
@pytest.mark.parametrize("w", [0, 4])
def test_every_agent_equals_eval_greedy_of_its_float32_lut(generic, w):
    mp = K.MdpParameters(p_max=4.0) if generic else None
    eng = _engine(6, mp=mp, **SWEEP)
    assert eng.lib.dqlb200_uses_default_instance(eng.handle) == (0 if generic else 1)
    tabs = [_random_tables(100 + p) for p in range(6)]
    for p, t in enumerate(tabs):
        _put(eng, p, t)
    res = eng.eval_agents(300, first_episode=57, working_step=w)
    assert res["termination_hist"].shape == (6, 9)
    for p in range(6):
        assert _row(res, p) == _single(eng, f32_lut(tabs[p]), 300, p, 57, w), p
    assert np.array_equal(res["success_rate"], (res["termination_hist"][:, 2] + res["termination_hist"][:, 3]) / 300)


def test_policy_is_the_float32_first_max():
    from dql_multirotor_landing_b200.engine import greedy_policy
    eng = _engine(2, seeds=[1, 2])
    t0, t1 = _random_tables(5), _random_tables(6)
    s = 10                                   # planted: float32 rounds actions 0 and 1 to a tie, float64 does not
    qa, qb = t1[0].view(np.float32), t1[1].view(np.float32)
    qa[3 * s: 3 * s + 3] = [1.0, 1.0, 0.0]
    qb[3 * s: 3 * s + 3] = [0.0, 2.0 ** -25, 0.0]
    _put(eng, 0, t0)
    _put(eng, 1, t1)
    res = eng.eval_agents(64, working_step=4, return_policies=True)
    pol = res["policy"]
    assert pol.shape == (2, N_STATES) and pol.dtype == np.uint8
    assert np.array_equal(pol[0], f32_lut(t0)) and np.array_equal(pol[1], f32_lut(t1))
    assert pol[1, s] == 0
    assert greedy_policy(*eng.get_tables(1)[:2])[s] == 1       # the float64-widened host LUT picks the other action
    # levels beyond curriculum_steps act 0, whatever the table words hold there
    eng3 = _engine(2, seeds=[1, 2], tp=K.TrainerParameters(curriculum_steps=3))
    _put(eng3, 0, t0)
    _put(eng3, 1, t1)
    pol3 = eng3.eval_agents(16, working_step=2, return_policies=True)["policy"]
    assert np.array_equal(pol3[0], f32_lut(t0, 3)) and np.array_equal(pol3[1], f32_lut(t1, 3))
    assert not pol3[:, 3 * K.STATES_PER_LEVEL:].any() and f32_lut(t0)[3 * K.STATES_PER_LEVEL:].any()


def test_against_the_oracle():
    from oracle.agent_oracle import state_id
    from oracle.dynamics import StandInParams
    from oracle.loop import eval_episode
    seeds, pids, v_mp, r_mp, axes = [5, 77, 123], [0, 9, 3], [1.6, 0.8, 1.2], [2.0, 3.0, 1.5], ["x", "y", "x"]
    eng = _engine(3, seeds=seeds, population_ids=pids, v_mp=v_mp, r_mp=r_mp, axes=axes)
    t = _assets_tables()
    for p in range(3):
        _put(eng, p, t)
    lut = f32_lut(t)
    n, first, w = 16, 200, 4
    res = eng.eval_agents(n, first_episode=first, working_step=w)
    for g in range(3):
        sp = StandInParams(v_z=-0.4, v_mp=v_mp[g], r_mp=r_mp[g], g=9.81 if axes[g] == "x" else -9.81)
        hist, steps = np.zeros(9, np.int64), 0
        for ep in range(n):
            rows = eval_episode(lambda s: int(lut[state_id(s)]), seeds[g], pids[g], first + ep, sp, w=w)[1:]
            hist[rows[-1]["code"]] += 1
            steps += len(rows)
        assert _row(res, g) == (n, steps, list(hist)), g


def _set_live_steps(eng, working_step, finished=None):
    v = eng.pop_state.view(torch.int32).view(eng.P, C.sizeof(K.PopulationState) // 4)
    v[:, 0] = torch.tensor(working_step, dtype=torch.int32, device=eng.device)
    if finished is not None:
        v[:, 1] = torch.tensor(finished, dtype=torch.int32, device=eng.device)


def test_live_working_steps():
    eng = _engine(5, seeds=[11, 12, 13, 14, 15])
    tabs = [_random_tables(200 + p) for p in range(5)]
    for p, t in enumerate(tabs):
        _put(eng, p, t)
    eng.reset(0)
    ws = [0, 3, 1, 2, 4]
    _set_live_steps(eng, ws, finished=[0, 0, 0, 0, 1])           # a finished agent holds curriculum_steps - 1
    assert [int(x) for x in eng.population_state()["working_step"]] == ws
    live = eng.eval_agents(128, first_episode=9)
    for p, w in enumerate(ws):
        fixed = eng.eval_agents(128, first_episode=9, working_step=w)
        assert _row(live, p) == _row(fixed, p), p
        assert _row(live, p) == _single(eng, f32_lut(tabs[p]), 128, p, 9, w), p


def test_replica_groups_read_replica_zero():
    R = 4
    eng = _engine(2 * R, seeds=[11] * R + [22] * R, population_ids=list(range(2 * R)), replicas_per_population=R)
    rng = np.random.default_rng(8)
    for g in range(2):
        eng.set_group_tables(g, rng.standard_normal(K.MAX_CELLS), rng.standard_normal(K.MAX_CELLS),
                             rng.integers(0, 50, K.MAX_CELLS))
    eng.reset(0)
    eng.train_merged(64, merge_every=4)
    tabs = eng.tables.cpu().numpy().view(np.uint32)
    for g in range(2):                        # the merge leaves every replica of a group identical
        for r in range(1, R):
            assert np.array_equal(tabs[g * R + r], tabs[g * R])
    ws = eng.population_state()["working_step"]
    res = eng.eval_agents(200, first_episode=3, return_policies=True)
    assert res["episodes"].shape == (2,)
    for g in range(2):
        assert np.array_equal(res["policy"][g], f32_lut(tabs[g * R]))
        assert _row(res, g) == _single(eng, f32_lut(tabs[g * R]), 200, g * R, 3, int(ws[g * R])), g


def _snapshot(eng):
    bufs = dict(env=eng.env_state, tables=eng.tables, pop=eng.pop_state, filt=eng.filter_state, dyn=eng.dynamics_state)
    return {k: v.clone() for k, v in bufs.items() if v is not None}


@pytest.mark.parametrize("dp", [dict(dynamics_model="second_order", n_sub=4), dict(accel_mode="kalman", n_sub=4)])
def test_options_read_only_and_deterministic(dp):
    eng = _engine(3, seeds=[4, 5, 6], dp=K.DynamicsParameters(**dp))
    tabs = [_random_tables(300 + p) for p in range(3)]
    for p, t in enumerate(tabs):
        _put(eng, p, t)
    eng.reset(2)
    eng.train(40)
    torch.cuda.synchronize()
    before = _snapshot(eng)
    assert len(before) == 4
    a = eng.eval_agents(100, first_episode=1)
    b = eng.eval_agents(100, first_episode=1)
    after = _snapshot(eng)
    for k in before:
        assert torch.equal(before[k], after[k]), k
    for key in ("episodes", "steps", "termination_hist"):
        assert np.array_equal(a[key], b[key]), key
    tabs = eng.tables.cpu().numpy().view(np.uint32)
    for p in range(3):
        assert _row(a, p) == _single(eng, f32_lut(tabs[p]), 100, p, 1, 2), p
    # the option without its bound buffer is refused, not evaluated on the default model
    bind, name = ((eng.lib.dqlb200_bind_filter_state, "dqlb200_bind_filter_state") if dp.get("accel_mode")
                  else (eng.lib.dqlb200_bind_dynamics_state, "dqlb200_bind_dynamics_state"))
    _ffi.check(bind(eng.handle, None))
    with pytest.raises(RuntimeError, match=name):
        eng.eval_agents(10)


def test_refusals_and_empty_call():
    eng = _engine(2, seeds=[1, 2])
    for w in (K.TrainerParameters().curriculum_steps, -2):
        with pytest.raises(RuntimeError, match="working_step"):
            eng.eval_agents(10, working_step=w)
    stats = torch.zeros(2 * C.sizeof(K.EvalStats), dtype=torch.uint8, device=eng.device)
    assert eng.lib.dqlb200_eval_agents(eng.handle, 0, 0, 10, None, None, None) == -1          # DQLB200_ERR_ARG: no stats_out
    assert eng.lib.dqlb200_eval_agents(eng.handle, 0, 0, 0, stats.data_ptr(), None, None) == 0
    torch.cuda.synchronize()
    assert not stats.any()
    res = eng.eval_agents(0)
    assert not res["episodes"].any() and not res["termination_hist"].any()


def test_at_size_with_the_committed_tables():
    P = 888
    eng = _engine(P, seeds=[1000 + p for p in range(P)], population_ids=list(range(P)))
    t = _assets_tables()
    eng.tables.copy_(torch.from_numpy(np.broadcast_to(t, (P,) + t.shape).copy().view(np.int32)))
    res = eng.eval_agents(1024, working_step=4)
    assert int(res["episodes"].sum()) == P * 1024 and int(res["termination_hist"].sum()) == P * 1024
    lut = f32_lut(t)
    for p in (0, 1, 137, 400, 511, 700, 886, 887):
        assert _row(res, p) == _single(eng, lut, 1024, p, 0, 4), p
    pooled = (res["termination_hist"][:, 2].sum() + res["termination_hist"][:, 3].sum()) / res["episodes"].sum()
    assert pooled > 0.85, pooled


def _trainer(tmp_path, **kw):
    from dql_multirotor_landing_b200.trainer import Trainer
    return Trainer(num_envs=64, chunk_steps=32, threads_per_block=32, verbose=False, save_path=tmp_path, **kw)


def test_trainer_greedy_curve(tmp_path):
    tr = _trainer(tmp_path / "a", num_populations=3, max_global_steps=32 * 6, eval_every=2, eval_episodes=256)
    info = tr.curriculum_training()
    assert len(tr.history) == 6
    for i, h in enumerate(tr.history):
        if i % 2 == 1:
            assert 0.0 <= h["Greedy success rate"] <= 1.0
            assert len(h["Greedy success rates"]) == 3 and h["Greedy success rate"] == h["Greedy success rates"][0]
        else:
            assert "Greedy success rate" not in h and "Greedy success rates" not in h
    assert "Greedy success rate" in info
    # the evaluation leaves training untouched
    ref = _trainer(tmp_path / "b", num_populations=3, max_global_steps=32 * 6)
    ref.curriculum_training()
    for name in ("tables", "pop_state", "env_state"):
        assert torch.equal(getattr(tr._engine, name), getattr(ref._engine, name)), name
    # a default Trainer's log and pickle are as before
    assert set(ref.history[0]) == {"Termination condition", "Number of steps", "Cumulative reward", "Mean reward", "Curent episode",
                                   "Remaining episodes", "Exploration rate", "Learning rate", "Success rate", "Global steps",
                                   "Env steps", "Episodes in chunk", "Pooled episodes", "working_step"}
    assert "_eval_every" not in ref.__getstate__() and "_eval_episodes" not in ref.__getstate__()


def test_trainer_tensorboard_tag(tmp_path):
    pytest.importorskip("tensorboard")
    tr = _trainer(tmp_path, max_global_steps=32, eval_every=1, eval_episodes=64, tensorboard=True)
    info = tr.curriculum_training()
    tr.log(info)
    events = list((tmp_path / "logs").glob("events.out.tfevents.*"))
    assert events and any(b"Episode/Greedy Success Rate" in e.read_bytes() for e in events)
