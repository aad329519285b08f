"""Tests of Engine.eval_platforms / dqlb200_eval_agents_platforms: every agent's greedy policy, built on the device from its live
float32 tables, under each of a list of platform motions in one launch.  The main contract: cell (g, c) is, episode for episode,
eval_greedy for population g * R under the float32 first-max LUT of g's tables, on an Engine whose population g * R flies
platform c (same seeds, population ids and axes).  Tests marked gpu need a CUDA device; the rest run anywhere."""
import ctypes as C
import pathlib

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from dql_multirotor_landing_b200 import _ffi
from dql_multirotor_landing_b200 import constants as K

gpu = pytest.mark.gpu
ROOT = pathlib.Path(__file__).resolve().parent.parent
N_STATES = K.MAX_CURRICULUM * K.STATES_PER_LEVEL
SPEEDS = [(2.0, 0.4), (2.0, 0.8), (2.0, 1.2), (2.0, 1.6)]
MIXED = [(3.0, 1.0), (1.5, 0.0), (2.0, 1.6)]          # other amplitudes, a resting platform, the default


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
    lut = np.zeros(N_STATES, np.uint8)
    lut[: cs * K.STATES_PER_LEVEL] = np.argmax((qa + qb) * np.float32(0.5), axis=1)
    return lut


def _cell(res, g, c):
    return (int(res["episodes"][g, c]), int(res["steps"][g, c]), [int(x) for x in res["termination_hist"][g, c]])


def _single(eng, lut, n, p, first, w):
    r = eng.eval_greedy(lut, n, population=p, first_episode=first, working_step=w)
    return (r["episodes"], r["steps"], r["termination_hist"])


def _per_platform_engines(P, platforms, **kw):
    """One Engine per platform with the same seeds, population ids and axes: the host path eval_platforms replaces."""
    return [_engine(P, r_mp=[r] * P, v_mp=[v] * P, **kw) for r, v in platforms]


SWEEP = dict(seeds=[3, 17, 42, 99, 2 ** 33 + 5, 1234], population_ids=[0, 7, 2, 11, 4, 5], axes=["x", "y", "x", "y", "y", "x"])


@gpu
@pytest.mark.parametrize("generic", [False, True])
@pytest.mark.parametrize("w", [0, 4])
def test_every_cell_equals_eval_greedy_on_a_per_platform_engine(generic, w):
    mp = K.MdpParameters(p_max=4.0) if generic else None
    eng = _engine(6, mp=mp, v_mp=[1.6, 0.8, 1.2, 0.4, 1.6, 1.0], r_mp=[2.0, 3.0, 1.5, 2.0, 2.5, 1.0], **SWEEP)
    assert eng.lib.dqlb200_uses_default_instance(eng.handle) == (0 if generic else 1)
    tabs = [_random_tables(100 + p) for p in range(6)]
    for p, t in enumerate(tabs):
        _put(eng, p, t)
    platforms = SPEEDS + MIXED
    res = eng.eval_platforms(300, platforms, first_episode=57, working_step=w)
    assert res["episodes"].shape == (6, 7) and res["termination_hist"].shape == (6, 7, 9)
    assert np.array_equal(res["platforms"], np.asarray(platforms, np.float64))
    for c, e in enumerate(_per_platform_engines(6, platforms, mp=mp, **SWEEP)):
        for p in range(6):
            assert _cell(res, p, c) == _single(e, f32_lut(tabs[p]), 300, p, 57, w), (p, c)
        e.close()
    hist = res["termination_hist"]
    assert np.array_equal(res["success_rate"], (hist[:, :, 2] + hist[:, :, 3]) / 300)
    # the platform changes the outcome: the columns are not all alike
    assert len({tuple(res["steps"][:, c]) for c in range(7)}) > 1


@gpu
def test_own_platform_reproduces_eval_agents():
    v_mp, r_mp = [1.6, 0.8, 1.2], [2.0, 3.0, 1.5]
    eng = _engine(3, seeds=[5, 6, 7], population_ids=[4, 1, 9], v_mp=v_mp, r_mp=r_mp, axes=["x", "y", "x"])
    for p in range(3):
        _put(eng, p, _random_tables(40 + p))
    own = eng.eval_agents(400, first_episode=11, working_step=3)
    res = eng.eval_platforms(400, list(zip(r_mp, v_mp)), first_episode=11, working_step=3)
    for g in range(3):         # agent g's own platform is column g
        assert _cell(res, g, g) == (int(own["episodes"][g]), int(own["steps"][g]), [int(x) for x in own["termination_hist"][g]]), g


@gpu
def test_episode_starts_do_not_depend_on_the_platform():
    """Episode i starts from the same x offset and platform phase (in turns) under every platform: the reset draw (Philox words
    0 and 2) ignores the platform.  Read from device traces under one constant action, so the drone's own motion is the same
    in every column: a resting platform gives its velocity, the phase then follows from rel_v = r w cos(phase) - v_d."""
    from oracle import philox
    seed, pid, first, n, k_max = 77, 3, 5, 256, 3
    lut = np.zeros(N_STATES, np.uint8)                  # one constant action everywhere
    rest = [(1.0, 0.0), (2.0, 0.0), (3.0, 0.0)]
    moving = [(2.0, 0.4), (1.0, 0.8), (3.0, 1.2), (2.0, 1.6)]
    traces = {}
    for (r, v), e in zip(rest + moving, _per_platform_engines(1, rest + moving, seeds=[seed], population_ids=[pid])):
        traces[(r, v)] = e.eval_greedy(lut, n, first_episode=first, working_step=4, trace_steps=k_max)["trace"]
        dphase, n_sub = K.platform_constants(r, v, e.mp.f_ag, e.dp.n_sub)[0], e.dp.n_sub
        traces[(r, v)]["dphase"] = dphase
        p_max = e.mp.p_max
        e.close()
    w0, _, w2, _ = philox.draws(seed, pid, np.arange(first, first + n), 0, philox.PURPOSE_RESET)
    phase0 = w2.astype(np.float64)
    x_init = -p_max + 2 * p_max * (w0 >> 8).astype(np.float64) / 2 ** 24
    alive = np.ones(n, bool)                            # episodes still running after k_max steps under every platform
    for tr in traces.values():
        alive &= ~tr["done"][: k_max - 1].any(axis=0)
    # x offset: under a resting platform x_d0 = r sin(phase0) - x_init unless clipped, so rel_p = x_init - drift, whatever r is
    unclipped = np.all([np.abs(r * np.sin(2 * np.pi * phase0 / 2 ** 32) - x_init) < p_max - 1e-3 for r, _ in rest], axis=0)
    sel = alive & unclipped
    assert sel.sum() > n // 4, sel.sum()
    rel_p = [traces[pl]["obs"][:, sel, 0] for pl in rest]
    for other in rel_p[1:]:
        np.testing.assert_allclose(other, rel_p[0], atol=1e-4)
    # phase: cos(phase after k steps) from rel_v, against the Philox start phase advanced by (hover + k) * n_sub * dphase
    v_d = -traces[rest[0]]["obs"][:, alive, 1]
    for r, v in moving:
        tr = traces[(r, v)]
        rw = float(K.platform_constants(r, v, 22.92, n_sub)[2])
        for k in range(1, k_max + 1):
            ph = (phase0[alive] + (k + 1) * n_sub * tr["dphase"]) % 2 ** 32
            np.testing.assert_allclose((tr["obs"][k - 1, alive, 1] + v_d[k - 1]) / rw, np.cos(2 * np.pi * ph / 2 ** 32), atol=1e-4)


@gpu
def test_against_the_oracle():
    from oracle.agent_oracle import state_id
    from oracle.dynamics import StandInParams
    from oracle.loop import eval_episode
    seeds, pids, axes = [5, 77, 123], [0, 9, 3], ["x", "y", "x"]
    eng = _engine(3, seeds=seeds, population_ids=pids, axes=axes)
    t = _assets_tables()
    for p in range(3):
        _put(eng, p, t)
    lut = f32_lut(t)
    platforms = [(2.0, 0.4), (3.0, 1.2), (1.0, 0.8)]
    n, first, w = 8, 200, 4
    res = eng.eval_platforms(n, platforms, first_episode=first, working_step=w)
    for g in range(3):
        for c, (r, v) in enumerate(platforms):
            sp = StandInParams(v_z=-0.4, v_mp=v, r_mp=r, g=9.81 if axes[g] == "x" else -9.81)
            hist, steps = np.zeros(9, np.int64), 0
            for ep in range(n):
                rows = eval_episode(lambda s: int(lut[state_id(s)]), seeds[g], pids[g], first + ep, sp, w=w)[1:]
                hist[rows[-1]["code"]] += 1
                steps += len(rows)
            assert _cell(res, g, c) == (n, steps, list(hist)), (g, c)


def _set_live_steps(eng, working_step, finished=None):
    v = eng.pop_state.view(torch.int32).view(eng.P, C.sizeof(K.PopulationState) // 4)
    v[:, 0] = torch.tensor(working_step, dtype=torch.int32, device=eng.device)
    if finished is not None:
        v[:, 1] = torch.tensor(finished, dtype=torch.int32, device=eng.device)


@gpu
def test_live_working_steps():
    eng = _engine(5, seeds=[11, 12, 13, 14, 15])
    tabs = [_random_tables(200 + p) for p in range(5)]
    for p, t in enumerate(tabs):
        _put(eng, p, t)
    eng.reset(0)
    ws = [0, 3, 1, 2, 4]
    _set_live_steps(eng, ws, finished=[0, 0, 0, 0, 1])
    live = eng.eval_platforms(128, MIXED, first_episode=9)
    for p, w in enumerate(ws):
        fixed = eng.eval_platforms(128, MIXED, first_episode=9, working_step=w)
        for c in range(len(MIXED)):
            assert _cell(live, p, c) == _cell(fixed, p, c), (p, c)
    e = _per_platform_engines(5, MIXED[:1], seeds=[11, 12, 13, 14, 15])[0]
    for p, w in enumerate(ws):
        assert _cell(live, p, 0) == _single(e, f32_lut(tabs[p]), 128, p, 9, w), p


@gpu
def test_replica_groups_read_replica_zero():
    R = 4
    kw = dict(seeds=[11] * R + [22] * R, population_ids=list(range(2 * R)))
    eng = _engine(2 * R, replicas_per_population=R, **kw)
    rng = np.random.default_rng(8)
    for g in range(2):
        eng.set_group_tables(g, rng.standard_normal(K.MAX_CELLS), rng.standard_normal(K.MAX_CELLS), rng.integers(0, 50, K.MAX_CELLS))
    eng.reset(0)
    eng.train_merged(64, merge_every=4)
    tabs = eng.tables.cpu().numpy().view(np.uint32)
    ws = eng.population_state()["working_step"]
    res = eng.eval_platforms(200, SPEEDS, first_episode=3)
    assert res["episodes"].shape == (2, 4)
    for c, e in enumerate(_per_platform_engines(2 * R, SPEEDS, **kw)):
        for g in range(2):
            assert _cell(res, g, c) == _single(e, f32_lut(tabs[g * R]), 200, g * R, 3, int(ws[g * R])), (g, c)
        e.close()


def _snapshot(eng):
    bufs = dict(env=eng.env_state, tables=eng.tables, pop=eng.pop_state, filt=eng.filter_state, dyn=eng.dynamics_state)
    return {k: v.clone() for k, v in bufs.items() if v is not None}


@gpu
@pytest.mark.parametrize("dp", [dict(dynamics_model="second_order", n_sub=4), dict(accel_mode="kalman", n_sub=4)])
def test_options_read_only_deterministic_and_additive(dp):
    dyn = K.DynamicsParameters(**dp)
    eng = _engine(3, seeds=[4, 5, 6], dp=dyn)
    for p in range(3):
        _put(eng, p, _random_tables(300 + p))
    eng.reset(2)
    eng.train(40)
    torch.cuda.synchronize()
    before = _snapshot(eng)
    assert len(before) == 4
    a = eng.eval_platforms(200, MIXED, first_episode=1)
    b = eng.eval_platforms(200, MIXED, first_episode=1)
    lo = eng.eval_platforms(100, MIXED, first_episode=1)
    hi = eng.eval_platforms(100, MIXED, first_episode=101)
    after = _snapshot(eng)
    for k in before:
        assert torch.equal(before[k], after[k]), k
    for key in ("episodes", "steps", "termination_hist"):
        assert np.array_equal(a[key], b[key]), key
        assert np.array_equal(a[key], lo[key] + hi[key]), key
    tabs = eng.tables.cpu().numpy().view(np.uint32)
    for c, e in enumerate(_per_platform_engines(3, MIXED, seeds=[4, 5, 6], dp=dyn)):
        for p in range(3):
            assert _cell(a, p, c) == _single(e, f32_lut(tabs[p]), 200, p, 1, 2), (p, c)
        e.close()
    # the option without its bound buffer is refused, not evaluated on the default model
    bind, name = ((eng.lib.dqlb200_bind_filter_state, "dqlb200_bind_filter_state") if dp.get("accel_mode")
                  else (eng.lib.dqlb200_bind_dynamics_state, "dqlb200_bind_dynamics_state"))
    _ffi.check(bind(eng.handle, None))
    with pytest.raises(RuntimeError, match=name):
        eng.eval_platforms(10, MIXED)


def _host_platforms(eng, platforms, pinned=False):
    arr = np.zeros((len(platforms), 4), np.uint32)
    for c, (r, v) in enumerate(platforms):
        dphase, pr, rw, rw2 = K.platform_constants(r, v, eng.mp.f_ag, eng.dp.n_sub)
        arr[c] = [dphase, *np.asarray([pr, rw, rw2], np.float32).view(np.uint32)]
    t = torch.from_numpy(arr.view(np.int32))
    return t.pin_memory() if pinned else t


@gpu
@pytest.mark.parametrize("pinned", [False, True])
def test_platform_list_may_be_rewritten_when_the_call_returns(pinned):
    eng = _engine(3, seeds=[7, 8, 9])
    for p in range(3):
        _put(eng, p, _random_tables(500 + p))
    want = eng.eval_platforms(256, SPEEDS, working_step=3)
    lst = _host_platforms(eng, SPEEDS, pinned)
    other = _host_platforms(eng, [(1.0, 0.0)] * 4)
    stats = torch.zeros(3 * 4 * C.sizeof(K.EvalStats), dtype=torch.uint8, device=eng.device)
    torch.cuda._sleep(100_000_000)            # the stream is still busy when the call returns ...
    _ffi.check(eng.lib.dqlb200_eval_agents_platforms(eng.handle, 3, 0, 256, C.cast(lst.data_ptr(), C.POINTER(K.Platform)), 4,
                                                     stats.data_ptr(), eng._stream()))
    lst.copy_(other)                          # ... and the caller rewrites its list at once
    st = stats.cpu().numpy().view(np.uint64).reshape(3, 4, 11).astype(np.int64)
    assert np.array_equal(st[:, :, 0], want["episodes"]) and np.array_equal(st[:, :, 1], want["steps"])
    assert np.array_equal(st[:, :, 2:], want["termination_hist"])


@gpu
def test_refusals_and_empty_call():
    eng = _engine(2, seeds=[1, 2])
    for bad in ([], [(2.0, 0.8, 1.0)], [(2.0, float("nan"))], [(0.0, 0.8)], [(2.0, -0.5)], [(float("inf"), 0.8)]):
        with pytest.raises(ValueError):
            eng.eval_platforms(10, bad)
    err = _ffi.Dqlb200Error
    for w in (K.TrainerParameters().curriculum_steps, -2):
        with pytest.raises(err, match="working_step"):
            eng.eval_platforms(10, SPEEDS, working_step=w)
    with pytest.raises(err, match="grid"):
        eng.eval_platforms(256 << 28, SPEEDS)
    # raw calls: the library's own checks, and calls with no episodes leave stats untouched
    call = eng.lib.dqlb200_eval_agents_platforms
    stats = torch.zeros(2 * 4 * C.sizeof(K.EvalStats), dtype=torch.uint8, device=eng.device)
    good = (K.Platform * 4)(*[K.Platform(*K.platform_constants(r, v, eng.mp.f_ag, eng.dp.n_sub)) for r, v in SPEEDS])
    assert call(None, 4, 0, 10, good, 4, stats.data_ptr(), None) == -1
    assert call(eng.handle, 4, 0, 10, None, 4, stats.data_ptr(), None) == -1
    assert call(eng.handle, 4, 0, 10, good, 4, None, None) == -1
    for n in (0, -3):
        assert call(eng.handle, 4, 0, 10, good, n, stats.data_ptr(), None) == -1
        assert b"n_platforms" in eng.lib.dqlb200_last_error()
    for fields, msg in (((0, 0.0, 0.0, 0.0), b"r must be"), ((0, -1.0, 0.0, 0.0), b"r must be"), ((0, float("inf"), 0.0, 0.0), b"r must be"),
                        ((0, float("nan"), 0.0, 0.0), b"r must be"), ((0, 2.0, -0.1, 0.0), b"rw and rw2"),
                        ((0, 2.0, 0.1, float("nan")), b"rw and rw2"), ((0, 2.0, float("inf"), 0.0), b"rw and rw2"),
                        ((0, 2.0, 0.1, -1.0), b"rw and rw2")):
        bad = (K.Platform * 2)(good[0], K.Platform(*fields))
        assert call(eng.handle, 4, 0, 10, bad, 2, stats.data_ptr(), None) == -1, fields
        assert msg in eng.lib.dqlb200_last_error() and b"platform 1" in eng.lib.dqlb200_last_error()
    for w in (5, -2):
        assert call(eng.handle, w, 0, 10, good, 4, stats.data_ptr(), None) == -1
    # blocks x agents x platforms is computed without overflow: 2^62 episodes and 2^30 platforms are refused, not wrapped
    assert call(eng.handle, 4, 0, 1 << 62, good, 4, stats.data_ptr(), None) == -1 and b"grid" in eng.lib.dqlb200_last_error()
    many = (K.Platform * (1 << 12))(*([good[0]] * (1 << 12)))
    assert call(eng.handle, 4, 0, 256 << 18, many, 1 << 12, stats.data_ptr(), None) == -1
    assert call(eng.handle, 4, 0, 0, good, 4, stats.data_ptr(), None) == 0
    assert call(eng.handle, 4, 0, -5, good, 4, stats.data_ptr(), None) == 0
    torch.cuda.synchronize()
    assert not stats.any()
    res = eng.eval_platforms(0, SPEEDS)
    assert res["episodes"].shape == (2, 4) and not res["episodes"].any() and not res["termination_hist"].any()
    assert not res["success_rate"].any()
    # the estimator option without its buffer, and a handle with nothing bound
    opt = _engine(2, seeds=[1, 2], dp=K.DynamicsParameters(accel_mode="kalman", n_sub=4))
    _ffi.check(opt.lib.dqlb200_bind_filter_state(opt.handle, None))
    assert call(opt.handle, 4, 0, 10, good, 4, stats.data_ptr(), None) == -3                     # DQLB200_ERR_STATE
    raw = C.c_void_p()
    cfg = K.build_config(2, 32, 32)
    pps = (K.PopulationParams * 2)(*[K.PopulationParams(1, 0, p, 0, 1.0, 0.0, 0.0, 0, np.float32(9.81), 0) for p in range(2)])
    _ffi.check(eng.lib.dqlb200_create(C.byref(cfg), K.alpha_lut().astype(np.float32).ctypes.data_as(C.POINTER(C.c_float)), pps, 0,
                                      C.byref(raw)))
    try:
        assert call(raw, 4, 0, 10, good, 4, stats.data_ptr(), None) == -3
        assert b"not bound" in eng.lib.dqlb200_last_error()
    finally:
        eng.lib.dqlb200_destroy(raw)
    torch.cuda.synchronize()
    assert not stats.any()


@gpu
def test_at_size_with_the_committed_tables():
    P = 888
    kw = dict(seeds=[1000 + p for p in range(P)], population_ids=list(range(P)))
    eng = _engine(P, **kw)
    t = _assets_tables()
    eng.tables.copy_(torch.from_numpy(np.broadcast_to(t, (P,) + t.shape).copy().view(np.int32)))
    res = eng.eval_platforms(1024, SPEEDS, working_step=4)
    assert res["episodes"].shape == (P, 4)
    assert int(res["episodes"].sum()) == P * 4 * 1024 and int(res["termination_hist"].sum()) == P * 4 * 1024
    lut = f32_lut(t)
    for c, e in enumerate(_per_platform_engines(P, SPEEDS, **kw)):
        for p in (0, 1, 137, 400, 511, 700, 886, 887):
            assert _cell(res, p, c) == _single(e, lut, 1024, p, 0, 4), (p, c)
        e.close()
    # the committed agent was trained at v = 1.6 (r = 2): it lands there
    hist = res["termination_hist"]
    pooled = (hist[:, 3, 2].sum() + hist[:, 3, 3].sum()) / res["episodes"][:, 3].sum()
    assert pooled > 0.85, pooled


def _trainer(tmp_path, **kw):
    from dql_multirotor_landing_b200.trainer import Trainer
    return Trainer(num_envs=64, chunk_steps=32, threads_per_block=32, verbose=False, save_path=tmp_path, **kw)


@gpu
def test_trainer_curve_by_platform(tmp_path):
    tr = _trainer(tmp_path / "a", num_populations=3, max_global_steps=32 * 4, eval_every=2, eval_episodes=256, eval_platforms=SPEEDS)
    info = tr.curriculum_training()
    assert len(tr.history) == 4
    for i, h in enumerate(tr.history):
        if i % 2 == 1:
            rows = h["Greedy success rates by platform"]
            assert len(rows) == 3 and all(len(row) == 4 for row in rows)
            assert all(0.0 <= x <= 1.0 for row in rows for x in row)
        else:
            assert "Greedy success rates by platform" not in h and "Greedy success rate by platform" not in h
    assert info["Greedy success rate by platform"] == tr.history[-1]["Greedy success rates by platform"][0]
    again = tr._engine.eval_platforms(256, SPEEDS)["success_rate"]
    assert [[float(x) for x in row] for row in again] == tr.history[-1]["Greedy success rates by platform"]
    # the evaluation leaves training untouched, and a default Trainer logs and pickles as before
    ref = _trainer(tmp_path / "b", num_populations=3, max_global_steps=32 * 4)
    ref.curriculum_training()
    for name in ("tables", "pop_state", "env_state"):
        assert torch.equal(getattr(tr._engine, name), getattr(ref._engine, name)), name
    assert set(ref.history[0]) == {"Termination condition", "Number of steps", "Cumulative reward", "Mean reward", "Curent episode",
                                   "Remaining episodes", "Exploration rate", "Learning rate", "Success rate", "Global steps",
                                   "Env steps", "Episodes in chunk", "Pooled episodes", "working_step"}
    assert "_eval_platforms" not in ref.__getstate__()


@gpu
def test_trainer_tensorboard_tags(tmp_path):
    pytest.importorskip("tensorboard")
    tr = _trainer(tmp_path, max_global_steps=32, eval_every=1, eval_episodes=64, eval_platforms=[(2.0, 0.4), (3.0, 1.2)],
                  tensorboard=True)
    info = tr.curriculum_training()
    tr.log(info)
    events = list((tmp_path / "logs").glob("events.out.tfevents.*"))
    data = b"".join(e.read_bytes() for e in events)
    assert b"Episode/Greedy Success Rate (r=2, v=0.4)" in data and b"Episode/Greedy Success Rate (r=3, v=1.2)" in data


def test_trainer_platform_arguments(tmp_path):
    with pytest.raises(ValueError, match="eval_every"):
        _trainer(tmp_path, eval_platforms=SPEEDS)
    for bad in ([], [(2.0,)], [(0.0, 0.8)], [(2.0, -1.0)], [(2.0, float("inf"))]):
        with pytest.raises(ValueError):
            _trainer(tmp_path, eval_every=1, eval_platforms=bad)
    tr = _trainer(tmp_path, eval_every=1, eval_platforms=np.asarray(SPEEDS))
    assert tr._eval_platforms == SPEEDS and all(type(x) is float for p in tr._eval_platforms for x in p)
    assert "_eval_platforms" not in _trainer(tmp_path).__getstate__()
    assert "_eval_platforms" not in _trainer(tmp_path, eval_every=2).__getstate__()
