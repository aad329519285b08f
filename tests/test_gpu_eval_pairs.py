"""Tests of Engine.eval_pairs / dqlb200_eval_pairs: every (x agent, y agent) pair's two-axis greedy landing, both LUTs built on
the device from the live float32 tables, in one launch.  The main contract: pair k's episodes are those of eval_greedy_2d under
the float32 first-max LUT of gx on x and, on y, gy's own LUT (a y agent) or the mirror image of it (an x agent), episode for
episode.  The GPU tests are marked; the Trainer's argument checks run anywhere."""
import ctypes as C
import pathlib

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from dql_multirotor_landing_b200 import _ffi
from dql_multirotor_landing_b200 import constants as K

ROOT = pathlib.Path(__file__).resolve().parent.parent
N_STATES = K.MAX_CURRICULUM * K.STATES_PER_LEVEL
gpu = pytest.mark.gpu

XY = K.TwoAxisParameters(trajectory=K.TRAJ_RECTILINEAR_XY, y_action_enabled=True, y_init_enabled=True)
EIGHT = K.TwoAxisParameters(trajectory=K.TRAJ_EIGHT, r_x=3.0, v_x=0.8, r_y=3.0, y_action_enabled=True, y_init_enabled=True)


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


def _luts(tabs, axes, gx, gy):
    """The LUT pair the library must fly for pair (gx, gy): gy's own on y when it is a y agent, else its mirror image."""
    from dql_multirotor_landing_b200.engine import mirrored_policy
    ly = f32_lut(tabs[gy])
    return f32_lut(tabs[gx]), (ly if axes[gy] == "y" else mirrored_policy(ly))


def _row(res, k):
    return (int(res["episodes"][k]), int(res["steps"][k]), [int(x) for x in res["termination_hist"][k]])


def _single(eng, lut_x, lut_y, n, first, w, ta, seed=42, stream_id=0):
    r = eng.eval_greedy_2d(lut_x, lut_y, n, two_axis=ta, seed=seed, stream_id=stream_id, first_episode=first, working_step=w)
    return (r["episodes"], r["steps"], r["termination_hist"])


def _set_live_steps(eng, working_step):
    v = eng.pop_state.view(torch.int32).view(eng.P, C.sizeof(K.PopulationState) // 4)
    v[:, 0] = torch.tensor(working_step, dtype=torch.int32, device=eng.device)


SWEEP = dict(seeds=[3, 17, 42, 99, 2 ** 33 + 5, 1234], population_ids=[0, 7, 2, 11, 4, 5], v_mp=[1.6, 0.8, 1.2, 0.4, 1.6, 1.0],
             r_mp=[2.0, 3.0, 1.5, 2.0, 2.5, 1.0], axes=["x", "y", "x", "y", "y", "x"])
PAIRS = [(0, 1), (2, 3), (5, 4), (0, 0), (2, 5), (0, 3)]      # y agents, mirrored x agents, repeated agents
PLATFORMS = {f"{name}-{'y' if y else 'noy'}": K.TwoAxisParameters(trajectory=traj, r_x=r, v_x=v, r_y=r, v_y=1.0,
                                                                   y_action_enabled=y, y_init_enabled=y)
             for name, traj, r, v in (("x", K.TRAJ_RECTILINEAR_X, 2.0, 1.6), ("xy", K.TRAJ_RECTILINEAR_XY, 2.0, 1.6),
                                      ("eight", K.TRAJ_EIGHT, 3.0, 0.8))
             for y in (False, True)}


@gpu
@pytest.mark.parametrize("platform", sorted(PLATFORMS))
@pytest.mark.parametrize("generic", [False, True])
@pytest.mark.parametrize("w", [0, 4])
def test_every_pair_equals_eval_greedy_2d_of_its_float32_luts(platform, generic, w):
    ta = PLATFORMS[platform]
    mp = K.MdpParameters(p_max=4.0) if generic else None
    eng = _engine(6, mp=mp, **SWEEP)
    assert eng.lib.dqlb200_uses_default_instance(eng.handle) == (0 if generic else 1)
    tabs = [_random_tables(100 + p) for p in range(6)]
    for p, t in enumerate(tabs):
        _put(eng, p, t)
    res = eng.eval_pairs(300, PAIRS, two_axis=ta, seed=1234, stream_id=5, first_episode=57, working_step=w)
    assert res["termination_hist"].shape == (6, 9) and np.array_equal(res["pairs"], PAIRS)
    for k, (gx, gy) in enumerate(PAIRS):
        assert _row(res, k) == _single(eng, *_luts(tabs, SWEEP["axes"], gx, gy), 300, 57, w, ta, 1234, 5), (k, gx, gy)
    assert np.array_equal(res["success_rate"], (res["termination_hist"][:, 2] + res["termination_hist"][:, 3]) / 300)


@gpu
def test_both_members_follow_the_float32_first_max():
    """Every state planted with a tie that float32 resolves to action 0 and float64 to action 1, once on an x member and once
    on a y member (own LUT and mirrored): the pair flies the float32 choice."""
    from dql_multirotor_landing_b200.engine import greedy_policy, mirrored_policy
    axes = ["x", "y", "x", "y"]
    eng = _engine(4, seeds=[1, 2, 3, 4], axes=axes)
    tabs = [_random_tables(10 + p) for p in range(4)]
    for g in (0, 1):
        qa, qb = tabs[g][0].view(np.float32), tabs[g][1].view(np.float32)
        qa[:] = np.tile(np.float32([1.0, 1.0, 0.0]), K.MAX_CELLS // 3)
        qb[:] = np.tile(np.float32([0.0, 2.0 ** -25, 0.0]), K.MAX_CELLS // 3)
    for p, t in enumerate(tabs):
        _put(eng, p, t)
    for g in (0, 1):
        assert not f32_lut(tabs[g]).any() and (greedy_policy(*eng.get_tables(g)[:2]) == 1).all()
    pairs = [(0, 3), (2, 1), (2, 0)]          # planted x member; planted y member (own LUT); planted x agent mirrored on y
    res = eng.eval_pairs(512, pairs, two_axis=XY, working_step=4)
    for k, (gx, gy) in enumerate(pairs):
        lx, ly = _luts(tabs, axes, gx, gy)
        assert _row(res, k) == _single(eng, lx, ly, 512, 0, 4, XY), k
        f64 = lambda g: greedy_policy(*eng.get_tables(g)[:2])
        lx64 = f64(gx)
        ly64 = f64(gy) if axes[gy] == "y" else mirrored_policy(f64(gy))
        assert _row(res, k) != _single(eng, lx64, ly64, 512, 0, 4, XY), k       # the float64 LUTs fly differently


@gpu
def test_against_the_oracle():
    from oracle.dynamics import sim2d_cases
    from oracle.loop import eval_episode_2d, mirrored_policy
    p2 = sim2d_cases()["eight"]
    ta = K.TwoAxisParameters(trajectory=p2.trajectory, r_x=p2.base.r_mp, v_x=p2.base.v_mp, r_y=p2.r_y, v_y=p2.v_y,
                             y_action_enabled=p2.y_action_enabled, y_init_enabled=p2.y_init_enabled)
    eng = _engine(2, seeds=[5, 6], axes=["x", "y"])
    tabs = [_assets_tables(), _random_tables(77)]
    for p, t in enumerate(tabs):
        _put(eng, p, t)
    n, first, w = 24, 300, 4
    res = eng.eval_pairs(n, [(0, 1), (0, 0)], two_axis=ta, seed=77, stream_id=3, first_episode=first, working_step=w)
    lx = f32_lut(tabs[0])
    for k, ly in enumerate((f32_lut(tabs[1]), mirrored_policy(lx))):
        hist, steps = np.zeros(9, np.int64), 0
        for ep in range(n):
            rows = eval_episode_2d(lx, ly, 77, 3, first + ep, p2, w=w)[1:]
            hist[rows[-1]["code"]] += 1
            steps += len(rows)
        assert _row(res, k) == (n, steps, list(hist)), k


@gpu
def test_live_working_step_is_the_lower_of_the_pair():
    axes = ["x", "y", "x", "x"]
    eng = _engine(4, seeds=[11, 12, 13, 14], axes=axes)
    tabs = [_random_tables(200 + p) for p in range(4)]
    for p, t in enumerate(tabs):
        _put(eng, p, t)
    eng.reset(0)
    ws = [3, 1, 0, 4]
    _set_live_steps(eng, ws)
    assert [int(x) for x in eng.population_state()["working_step"]] == ws
    pairs = [(0, 1), (0, 0), (3, 1), (2, 3), (3, 3), (3, 0)]
    live = eng.eval_pairs(128, pairs, two_axis=XY, first_episode=9)
    for k, (gx, gy) in enumerate(pairs):
        w = min(ws[gx], ws[gy])
        fixed = eng.eval_pairs(128, [(gx, gy)], two_axis=XY, first_episode=9, working_step=w)
        assert _row(live, k) == _row(fixed, 0), k
        assert _row(live, k) == _single(eng, *_luts(tabs, axes, gx, gy), 128, 9, w, XY), k


@gpu
def test_replica_groups_read_replica_zero():
    R = 3
    axes = ["x"] * R + ["y"] * R
    eng = _engine(2 * R, seeds=[11] * R + [22] * R, population_ids=list(range(2 * R)), replicas_per_population=R, axes=axes)
    tabs = [_random_tables(400 + p) for p in range(2 * R)]          # every replica different: only replica g * R may count
    for p, t in enumerate(tabs):
        _put(eng, p, t)
    res = eng.eval_pairs(200, [(0, 1), (0, 0)], two_axis=EIGHT, first_episode=3, working_step=2)
    assert res["episodes"].shape == (2,)
    for k, (gx, gy) in enumerate([(0, 1), (0, 0)]):
        assert _row(res, k) == _single(eng, *_luts(tabs, axes, gx * R, gy * R), 200, 3, 2, EIGHT), k
    with pytest.raises(_ffi.Dqlb200Error, match="agent index"):
        eng.eval_pairs(10, [(0, 2)])                # two agents, not six populations


def _snapshot(eng):
    return {k: getattr(eng, k).clone() for k in ("env_state", "tables", "pop_state")}


@gpu
def test_read_only_deterministic_and_additive():
    axes = ["x", "y", "x"]
    eng = _engine(3, seeds=[4, 5, 6], axes=axes)
    for p in range(3):
        _put(eng, p, _random_tables(300 + p))
    eng.reset(2)
    eng.train(40)
    torch.cuda.synchronize()
    before = _snapshot(eng)
    pairs = [(0, 1), (2, 0), (0, 2)]
    a = eng.eval_pairs(300, pairs, two_axis=EIGHT, first_episode=1)
    b = eng.eval_pairs(300, pairs, two_axis=EIGHT, first_episode=1)
    lo = eng.eval_pairs(150, pairs, two_axis=EIGHT, first_episode=1)
    hi = eng.eval_pairs(150, pairs, two_axis=EIGHT, first_episode=151)
    after = _snapshot(eng)
    for k in before:
        assert torch.equal(before[k], after[k]), k
    for key in ("episodes", "steps", "termination_hist"):
        assert np.array_equal(a[key], b[key]), key
        assert np.array_equal(a[key], lo[key] + hi[key]), key
    tabs = eng.tables.cpu().numpy().view(np.uint32)
    ws = eng.population_state()["working_step"]
    for k, (gx, gy) in enumerate(pairs):
        assert _row(a, k) == _single(eng, *_luts(tabs, axes, gx, gy), 300, 1, int(min(ws[gx], ws[gy])), EIGHT), k


@gpu
def test_pinned_pair_list_may_be_reused_when_the_call_returns():
    axes = ["x", "y", "x"]
    eng = _engine(3, seeds=[7, 8, 9], axes=axes)
    for p in range(3):
        _put(eng, p, _random_tables(500 + p))
    want = eng.eval_pairs(256, [(0, 1), (2, 0)], two_axis=XY, working_step=3)
    pinned = torch.tensor([[0, 1], [2, 0]], dtype=torch.int32).pin_memory()
    prm = K.eval2d_params(XY, eng.dp, eng.mp.f_ag, 42, 0, 3)
    stats = torch.zeros(2 * C.sizeof(K.EvalStats), dtype=torch.uint8, device=eng.device)
    torch.cuda._sleep(100_000_000)            # the stream is still busy when the call returns ...
    _ffi.check(eng.lib.dqlb200_eval_pairs(eng.handle, C.byref(prm), pinned.data_ptr(), 2, 0, 256, stats.data_ptr(), eng._stream()))
    pinned.copy_(torch.tensor([[2, 2], [0, 0]], dtype=torch.int32))      # ... and the caller rewrites its list at once
    st = stats.cpu().numpy().view(np.uint64).reshape(2, 11).astype(np.int64)
    assert np.array_equal(st[:, 0], want["episodes"]) and np.array_equal(st[:, 1], want["steps"])
    assert np.array_equal(st[:, 2:], want["termination_hist"])


@gpu
def test_refusals_and_empty_call():
    eng = _engine(3, seeds=[1, 2, 3], axes=["x", "y", "x"])
    err = _ffi.Dqlb200Error
    with pytest.raises(err, match="n_pairs"):
        eng.eval_pairs(10, [])
    for bad in ([(0, 3)], [(-1, 1)], [(3, 1)], [(0, -1)]):
        with pytest.raises(err, match="agent index"):
            eng.eval_pairs(10, bad)
    with pytest.raises(err, match="y-axis agent"):
        eng.eval_pairs(10, [(0, 1), (1, 0)])
    with pytest.raises(err, match="trajectory"):
        eng.eval_pairs(10, [(0, 1)], two_axis=K.TwoAxisParameters(trajectory=3))
    for w in (K.TrainerParameters().curriculum_steps, -2):
        with pytest.raises(err, match="working_step"):
            eng.eval_pairs(10, [(0, 1)], working_step=w)
    with pytest.raises(err, match="grid"):
        eng.eval_pairs(256 << 31, [(0, 1)])
    # raw calls: null arguments, and a call with no episodes leaves stats untouched
    prm = K.eval2d_params(K.TwoAxisParameters(), eng.dp, eng.mp.f_ag, 42, 0, 4)
    pairs = np.asarray([[0, 1], [2, 2]], np.int32)
    stats = torch.zeros(2 * C.sizeof(K.EvalStats), dtype=torch.uint8, device=eng.device)
    call = eng.lib.dqlb200_eval_pairs
    assert call(None, C.byref(prm), pairs.ctypes.data, 2, 0, 10, stats.data_ptr(), None) == -1
    assert call(eng.handle, None, pairs.ctypes.data, 2, 0, 10, stats.data_ptr(), None) == -1
    assert call(eng.handle, C.byref(prm), None, 2, 0, 10, stats.data_ptr(), None) == -1
    assert call(eng.handle, C.byref(prm), pairs.ctypes.data, 2, 0, 10, None, None) == -1
    assert call(eng.handle, C.byref(prm), pairs.ctypes.data, 0, 0, 10, stats.data_ptr(), None) == -1
    assert call(eng.handle, C.byref(prm), pairs.ctypes.data, 2, 0, 0, stats.data_ptr(), None) == 0
    assert call(eng.handle, C.byref(prm), pairs.ctypes.data, 2, 0, -5, stats.data_ptr(), None) == 0
    torch.cuda.synchronize()
    assert not stats.any()
    res = eng.eval_pairs(0, [(0, 1), (2, 0)])
    assert not res["episodes"].any() and not res["steps"].any() and not res["termination_hist"].any()
    assert np.array_equal(res["success_rate"], [0.0, 0.0])
    # the estimator / second-order options are refused, as by eval_greedy_2d
    opt = _engine(2, seeds=[1, 2], axes=["x", "y"], dp=K.DynamicsParameters(accel_mode="kalman", n_sub=4))
    with pytest.raises(err, match="two-axis evaluator"):
        opt.eval_pairs(10, [(0, 1)])
    # a handle with nothing bound
    raw = C.c_void_p()
    cfg = K.build_config(2, 32, 32)
    pps = (K.PopulationParams * 2)(*[K.PopulationParams(1, 0, p, 0, 0.0, 0.0, 0.0, 0, np.float32(9.81), 0) for p in range(2)])
    _ffi.check(eng.lib.dqlb200_create(C.byref(cfg), K.alpha_lut().astype(np.float32).ctypes.data_as(C.POINTER(C.c_float)), pps, 0,
                                      C.byref(raw)))
    try:
        assert call(raw, C.byref(prm), pairs[:1].ctypes.data, 1, 0, 10, stats.data_ptr(), None) == -3      # DQLB200_ERR_STATE
        assert b"not bound" in eng.lib.dqlb200_last_error()
    finally:
        eng.lib.dqlb200_destroy(raw)


@gpu
def test_at_size_with_the_committed_tables():
    P, H = 888, 444
    axes = ["x"] * H + ["y"] * H
    eng = _engine(P, seeds=[1000 + p for p in range(P)], population_ids=list(range(P)), axes=axes)
    t = _assets_tables()
    eng.tables.copy_(torch.from_numpy(np.broadcast_to(t, (P,) + t.shape).copy().view(np.int32)))
    pairs = [(k, H + k) for k in range(H)]
    res = eng.eval_pairs(1024, pairs, two_axis=EIGHT, working_step=4)
    assert int(res["episodes"].sum()) == H * 1024 and int(res["termination_hist"].sum()) == H * 1024
    for k in range(1, H):            # identical LUTs, one key: identical rows
        assert _row(res, k) == _row(res, 0), k
    lut = f32_lut(t)
    for k in (0, 211, 443):
        assert _row(res, k) == _single(eng, lut, lut, 1024, 0, 4, EIGHT), k


def _trainer(tmp_path, **kw):
    from dql_multirotor_landing_b200.trainer import Trainer
    return Trainer(num_envs=64, chunk_steps=32, threads_per_block=32, verbose=False, save_path=tmp_path, **kw)


@gpu
def test_trainer_two_axis_curve(tmp_path):
    tr = _trainer(tmp_path / "a", num_populations=3, max_global_steps=32 * 3, eval_every=1, eval_episodes=256, eval_two_axis=EIGHT)
    info = tr.curriculum_training()
    assert info["Greedy two-axis success rate"] == tr.history[-1]["Greedy two-axis success rate"]
    assert len(tr.history) == 3
    for h in tr.history:
        assert 0.0 <= h["Greedy two-axis success rate"] <= 1.0
        assert len(h["Greedy two-axis success rates"]) == 3
        assert h["Greedy two-axis success rate"] == h["Greedy two-axis success rates"][0]
        assert len(h["Greedy success rates"]) == 3
    # every agent flies its own policy on x and its mirror image on y, at its live working step
    again = tr._engine.eval_pairs(256, [(g, g) for g in range(3)], two_axis=EIGHT)["success_rate"]
    assert [float(r) for r in again] == tr.history[-1]["Greedy two-axis success rates"]
    # the evaluation leaves training untouched
    ref = _trainer(tmp_path / "b", num_populations=3, max_global_steps=32 * 3)
    ref.curriculum_training()
    for name in ("tables", "pop_state", "env_state"):
        assert torch.equal(getattr(tr._engine, name), getattr(ref._engine, name)), name
    assert "Greedy two-axis success rate" not in ref.history[-1]


@gpu
def test_trainer_two_axis_tensorboard_tag(tmp_path):
    pytest.importorskip("tensorboard")
    tr = _trainer(tmp_path, max_global_steps=32, eval_every=1, eval_episodes=64, eval_two_axis=XY, tensorboard=True)
    info = tr.curriculum_training()
    tr.log(info)
    events = list((tmp_path / "logs").glob("events.out.tfevents.*"))
    assert events and any(b"Episode/Greedy Two-Axis Success Rate" in e.read_bytes() for e in events)


def test_trainer_two_axis_arguments(tmp_path):
    with pytest.raises(ValueError, match="eval_every"):
        _trainer(tmp_path, eval_two_axis=EIGHT)
    with pytest.raises(ValueError, match="direction"):
        _trainer(tmp_path, eval_every=1, eval_two_axis=EIGHT, direction="y")
    with pytest.raises(ValueError, match="first-order"):
        _trainer(tmp_path, eval_every=1, eval_two_axis=EIGHT, dynamics=K.DynamicsParameters(dynamics_model="second_order", n_sub=4))
    assert "_eval_two_axis" not in _trainer(tmp_path).__getstate__()
    assert "_eval_two_axis" not in _trainer(tmp_path, eval_every=2).__getstate__()
    assert _trainer(tmp_path, eval_every=2, eval_two_axis=EIGHT).__getstate__()["_eval_two_axis"] == EIGHT
