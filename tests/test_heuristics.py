"""The reference's hand-written policies (SURVEY.md 8f row 4) as the in-kernel action source of the rollout
kernels (madrl_ww_rollout_heuristic / madrl_pursuit_rollout_heuristic):

  * the oracle restatement (oracle/heuristics_oracle.py) is pinned to the REAL classes
    (heuristics/waterworld.py, heuristics/pursuit.py; their actions recorded, tests/reference_record.py);
  * the kernel source, run on the CPU by the warp emulator (tests/emu), closes the loop exactly as the
    oracle policy driving the oracle env does.  The same checks run on the GPU in
    tests/test_heuristics_gpu.py.
"""
import os
import shutil
import types

import numpy as np
import pytest

from conftest import ROOT
from oracle import refshim
from oracle.heuristics_oracle import (pursuit_action, pursuit_action_table, policy_draw, waterworld_action)
from oracle.philox import Stream
from oracle.pursuit_oracle import PursuitOracle
from oracle.waterworld_oracle import WaterworldOracle
from reference_record import recorded

needs_cxx = pytest.mark.skipif(shutil.which(os.environ.get("CXX", "g++")) is None, reason="no host C++ compiler")


def f32(x):
    return np.asarray(x, dtype=np.float64).astype(np.float32)


# ------------------------------------------------------------------------------ oracle == reference
def test_waterworld_policy_oracle_equals_reference_bitwise():
    """The reference policy's actions (recorded) on 600 random observations, bit for bit."""
    rs = np.random.RandomState(0)
    cases = []
    for K in (30, 7):
        D = 7 * K + 3
        for i in range(300):
            o = rs.rand(D) * (rs.rand(D) < 0.2)
            o[7 * K:7 * K + 2] = rs.rand(2) < 0.3
            if i == 5:
                o[:] = 0
            cases.append((K, i, o))

    def reference():
        pol = refshim.load_reference_heuristics()[0](None, None)
        return dict(actions=np.array([pol.sample_actions(o[None])[0][0] for _, _, o in cases]))
    ref = recorded("heuristics_waterworld", reference)["actions"]
    for (K, i, o), a in zip(cases, ref):
        assert np.array_equal(a, waterworld_action(o)), (K, i)


class _Space(object):
    def __init__(self, draws):
        self.draws = draws

    def sample(self):
        return self.draws.pop(0)


@pytest.mark.parametrize("py2", [False, True])
def test_pursuit_policy_oracle_equals_reference(py2):
    """py2=False: heuristics/pursuit.py executed as is (Python 3: `xs / 2` is a true division).
    py2=True: the same source with line 23's two divisions spelt `//`, what they mean in Python 2.
    The reference policy's actions on 1600 random windows are recorded; 77 stands for a sampled action."""
    rs = np.random.RandomState(1)
    cases = []
    for R in (7, 4, 5, 9):
        for i in range(400):
            o = np.zeros((R, R, 4))
            o[..., 2] = (rs.rand(R, R) < 0.06) * 0.1
            cases.append((R, i, o))

    def reference():
        _, P, src = refshim.load_reference_heuristics()
        if py2:
            ported = src.replace("x, y = xs / 2, ys / 2", "x, y = xs // 2, ys // 2")
            assert ported != src
            mod = types.ModuleType("_ref_heuristics_pursuit_py2")
            exec(compile(ported.split("if __name__")[0], "heuristics/pursuit.py[py2 division]", "exec"), mod.__dict__)
            P = mod.PursuitHeuristicPolicy
        return dict(actions=np.array([P(None, _Space([77])).sample_actions(o)[0] for _, _, o in cases]))
    ref = recorded("heuristics_pursuit_py%d" % (2 if py2 else 3), reference)["actions"]
    tabs = {R: pursuit_action_table(R, py2) for R in (7, 4, 5, 9)}
    for (R, i, o), a in zip(cases, ref):
        assert a == pursuit_action(o, lambda: 77, py2), (R, i)
        if a != 77:   # the tabulated form the CUDA host code uses
            xev, yev = np.nonzero(o[..., 2])
            c = float(R // 2) if py2 else R / 2
            k = np.argmin((xev - c) ** 2 + (yev - c) ** 2)
            assert tabs[R][xev[k] * R + yev[k]] == a


# ------------------------------------------------------------------------------ emulated kernels
WW = {
    "c2": dict(n_pursuers=5, n_evaders=5),
    "dense": dict(n_pursuers=5, n_evaders=5, n_coop=1, radius=0.04, sensor_range=0.3),
    "c4": dict(n_pursuers=20, n_evaders=50, n_poison=50),
    "k40_randobst": dict(n_pursuers=4, n_evaders=40, n_poison=3, n_sensors=40, n_coop=2, radius=0.03, obstacle_loc=None,
                         addid=False),
}


def check_waterworld_closed_loop(eng, cfg, seed, base, obs0, act, obs, rew, done, info, mpl, tol, min_norm):
    """The engine's actions are the oracle policy's on the previous observation; the env they drive is the oracle env."""
    T, E = act.shape[:2]
    checked = skipped = 0
    for e in range(E):
        o = WaterworldOracle(rng=Stream(seed, base + e), **cfg)
        prev = np.array(o.reset())
        assert np.abs(prev - obs0[e]).max() < tol
        prev, ts = obs0[e].astype(np.float64), 0
        for t in range(T):
            for i in range(cfg['n_pursuers']):
                want, n = waterworld_action(prev[i], return_norm=True)
                if 0 < n < min_norm:
                    skipped += 1
                    continue
                checked += 1
                assert np.abs(want - act[t, e, i]).max() < tol, (t, e, i)
            oo, rr, dd, ii = o.step(act[t, e].astype(np.float64))
            ts += 1
            dd = dd or (mpl and ts >= mpl)
            assert bool(done[t, e]) == dd and [ii['evcatches'], ii['pocatches']] == list(info[t, e]), (t, e)
            assert np.abs(rr - rew[t, e]).max() < tol
            if dd:
                oo, ts = o.reset(), 0
            assert np.abs(np.array(oo) - obs[t, e]).max() < tol, (t, e)
            prev = obs[t, e].astype(np.float64)
    return checked, skipped


@needs_cxx
@pytest.mark.parametrize("name,E,T", [("c2", 4, 50), ("dense", 4, 60), ("c4", 2, 6), ("k40_randobst", 2, 20)])
def test_emulated_waterworld_policy_closes_the_loop_fp64(name, E, T):
    from emu.driver import EmuWaterworld
    cfg, seed, base, mpl = WW[name], 11, 300, 17
    eng = EmuWaterworld(E, seed=seed, env_id_base=base, max_path_length=mpl, **cfg)
    obs0 = eng.reset()
    act, obs, rew, done, info = eng.rollout_heuristic(T, obs0, auto_reset=True)
    assert np.all(np.abs(np.linalg.norm(act, axis=-1) - 1) < 1e-12 + (np.linalg.norm(act, axis=-1) == 0))
    checked, _ = check_waterworld_closed_loop(eng, cfg, seed, base, obs0, act, obs, rew, done, info, mpl, 1e-9, 0.0)
    assert checked == T * E * cfg['n_pursuers']
    assert done.any() == (T >= mpl)      # the horizon cut-off + in-place reset is part of the loop
    # chunk invariance: two launches chained through the last observation == one launch
    eng2 = EmuWaterworld(E, seed=seed, env_id_base=base, max_path_length=mpl, **cfg)
    o0 = eng2.reset()
    a1 = eng2.rollout_heuristic(T // 2, o0, auto_reset=True)
    a2 = eng2.rollout_heuristic(T - T // 2, a1[1][-1], auto_reset=True)
    for x, y1, y2 in zip((act, obs, rew, done, info), a1, a2):
        assert np.array_equal(x, np.concatenate([y1, y2]))


@needs_cxx
def test_emulated_waterworld_policy_fp32():
    from emu.driver import EmuWaterworld
    cfg, seed, base, E, T = WW["c2"], 5, 40, 6, 40
    eng = EmuWaterworld(E, seed=seed, env_id_base=base, fp64=False, **cfg)
    obs0 = eng.reset()
    act, obs, rew, done, info = eng.rollout_heuristic(T, obs0, auto_reset=False)
    checked = 0
    for e in range(E):
        prev = obs0[e].astype(np.float64)
        for t in range(T):
            for i in range(cfg['n_pursuers']):
                want, n = waterworld_action(prev[i], return_norm=True)
                if n == 0:
                    assert not act[t, e, i].any()
                elif n > 1e-2:
                    checked += 1
                    assert np.abs(want - act[t, e, i]).max() < 1e-5, (t, e, i)
            prev = obs[t, e].astype(np.float64)
    assert checked > 0.5 * T * E * cfg['n_pursuers']


def test_waterworld_policy_needs_the_speed_feature_layout():
    if shutil.which(os.environ.get("CXX", "g++")) is None:
        pytest.skip("no host C++ compiler")
    from emu.driver import EmuWaterworld
    eng = EmuWaterworld(2, n_pursuers=3, n_evaders=3, speed_features=False)
    with pytest.raises(RuntimeError, match="speed_features"):
        eng.rollout_heuristic(2, eng.reset())


def pool16():
    return np.load(os.path.join(ROOT, "maps", "map_pool16.npy"))


def small_map():
    m = np.zeros((1, 5, 5), dtype=np.int32)
    m[0, 2, 2] = -1
    return m


C3 = dict(n_evaders=30, n_pursuers=8, obs_range=7, surround=True, n_catch=2, flatten=True, reward_mech='local',
          catchr=0.1, term_pursuit=5.0, sample_maps=True, include_id=True)
PE = {
    "c3": (pool16, C3),
    "sparse_conv": (pool16, dict(C3, n_evaders=3, n_pursuers=6, obs_range=5, flatten=False, surround=False, n_catch=1)),
    "even_r4": (small_map, dict(n_evaders=2, n_pursuers=5, obs_range=4, surround=False, n_catch=1, reward_mech='global')),
    "r9_global": (pool16, dict(C3, n_evaders=4, n_pursuers=10, obs_range=9, reward_mech='global', include_id=False)),
}


def evader_window(o, R, flatten):
    """(R, R) evader channel of one agent's observation in either layout (pursuit_evade.py:440-449)."""
    o = np.asarray(o)
    return o.reshape(-1)[2 * R * R:3 * R * R].reshape(R, R) if flatten else o.reshape(R, R, 4)[..., 2]


def check_pursuit_closed_loop(maps, cfg, seed, base, obs0, act, obs, rew, done, removed, mpl, py2):
    T, E = act.shape[:2]
    R, flat, Np = cfg['obs_range'], cfg.get('flatten', True), cfg['n_pursuers']
    n_random = 0
    for e in range(E):
        o = PursuitOracle(maps, rng=Stream(seed, base + e), **cfg)
        first = o.reset()
        assert np.array_equal(f32(first).reshape(obs0[e].shape), obs0[e])
        prev, ts = obs0[e], 0
        for t in range(T):
            ctr = o.rng.counter     # the env's draw counter when `prev` was produced
            for q in range(Np):
                win = np.zeros((R, R, 4))
                win[..., 2] = evader_window(prev[q], R, flat)
                drew = []
                want = pursuit_action(win, lambda: drew.append(1) or policy_draw(seed, base + e, ctr, q), py2)
                n_random += len(drew)
                assert want == act[t, e, q], (t, e, q)
            oo, rr, dd, ii = o.step(act[t, e])
            ts += 1
            dd = dd or (mpl and ts >= mpl)
            assert bool(done[t, e]) == dd and ii['removed'] == removed[t, e], (t, e)
            assert np.array_equal(f32(rr), rew[t, e])
            if dd:
                oo, ts = o.reset(), 0
            assert np.array_equal(f32(oo).reshape(obs[t, e].shape), obs[t, e]), (t, e)
            prev = obs[t, e]
    return n_random


@needs_cxx
@pytest.mark.parametrize("py2", [True, False])
@pytest.mark.parametrize("name,E,T", [("c3", 3, 30), ("sparse_conv", 4, 50), ("even_r4", 5, 60), ("r9_global", 3, 30)])
def test_emulated_pursuit_policy_closes_the_loop(name, E, T, py2):
    from emu.driver import EmuPursuit
    mk, cfg = PE[name]
    maps, seed, base, mpl = mk(), 21, 900, 13
    eng = EmuPursuit(E, maps, seed=seed, env_id_base=base, max_path_length=mpl, **cfg)
    obs0 = eng.reset()
    act, obs, rew, done, removed = eng.rollout_heuristic(T, obs0, auto_reset=True, py2_division=py2)
    assert act.min() >= 0 and act.max() <= 4
    n_random = check_pursuit_closed_loop(maps, cfg, seed, base, obs0, act, obs, rew, done, removed, mpl, py2)
    if name != "c3":
        assert n_random > 0          # the injected sampler stream was exercised
    assert done.any()
    eng2 = EmuPursuit(E, maps, seed=seed, env_id_base=base, max_path_length=mpl, **cfg)
    o0 = eng2.reset()
    a1 = eng2.rollout_heuristic(T // 3, o0, auto_reset=True, py2_division=py2)
    a2 = eng2.rollout_heuristic(T - T // 3, a1[1][-1], auto_reset=True, py2_division=py2)
    for x, y1, y2 in zip((act, obs, rew, done, removed), a1, a2):
        assert np.array_equal(x, np.concatenate([y1, y2]))


# ------------------------------------------------------------------------------ stand-alone generators
@needs_cxx
@pytest.mark.parametrize("dtype,tol", [(np.float64, 1e-12), (np.float32, 1e-5)])
def test_emulated_waterworld_generator_matches_oracle(dtype, tol):
    from emu.driver import ww_heuristic_actions
    rs = np.random.RandomState(3)
    for K, D in ((30, 213), (7, 51), (40, 282)):
        obs = (rs.rand(37, D) * (rs.rand(37, D) < 0.2)).astype(dtype)
        obs[:, 7 * K:7 * K + 2] = rs.rand(37, 2) < 0.3
        obs[4] = 0
        got = ww_heuristic_actions(obs, K)
        for i in range(37):
            want, n = waterworld_action(obs[i].astype(np.float64), return_norm=True)
            if n == 0 or n > 1e-2 or dtype == np.float64:
                assert np.abs(got[i] - want).max() < tol, (K, i)


@needs_cxx
@pytest.mark.parametrize("py2", [True, False])
def test_emulated_pursuit_generator_matches_oracle(py2):
    from emu.driver import pursuit_heuristic_actions
    rs = np.random.RandomState(4)
    for R in (7, 4, 11):
        n = 150
        win = (rs.rand(n, R, R) < 0.04) * 0.1
        fb = rs.randint(0, 5, n)
        conv = np.zeros((n, R, R, 4), np.float32)
        conv[..., 2] = win
        conv[..., 1] = 0.3      # other channels must not matter
        flat = np.concatenate([np.full((n, R * R), 0.1), np.full((n, R * R), 0.2), win.reshape(n, -1), np.ones((n, 1))], 1)
        want = [pursuit_action(conv[i], lambda i=i: int(fb[i]), py2) for i in range(n)]
        assert list(pursuit_heuristic_actions(conv.reshape(n, -1), R, False, fb, py2)) == want
        assert list(pursuit_heuristic_actions(flat, R, True, fb, py2)) == want
        assert any(w == f and not win[i].any() for i, (w, f) in enumerate(zip(want, fb)))


# ------------------------------------------------------------------------------ closed-loop goldens
# tests/golden/cl_*.npz: the REAL reference env stepped by the REAL reference policy (oracle/make_golden.py
# gen_closed_loop).  The engine's in-kernel policy rollout must reproduce the whole trajectory.
import json  # noqa: E402

from conftest import GOLDEN_DIR  # noqa: E402

CL_WW = ["cl_ww_c2", "cl_ww_dense"]
CL_PE = ["cl_pe_conv_py2", "cl_pe_conv_py3", "cl_pe_sparse_py2"]


def check_closed_loop_golden_ww(g, reset, rollout, tol):
    obs0 = reset()
    assert np.abs(obs0[0] - g["obs0"]).max() < tol
    act, obs, rew, done, info = rollout(len(g["actions"]), obs0)
    assert np.abs(act[:, 0] - g["actions"]).max() < tol
    assert np.abs(obs[:, 0] - g["obs"]).max() < tol and np.abs(rew[:, 0] - g["rew"]).max() < tol
    assert np.array_equal(info[:, 0], g["info"]) and not done.any()


def check_closed_loop_golden_pe(g, reset, rollout):
    obs0 = reset()
    assert np.array_equal(obs0[0], f32(g["obs0"]).reshape(obs0[0].shape))
    T = len(g["actions"])
    act, obs, rew, done, removed = rollout(T, obs0)
    assert np.array_equal(act[:, 0], g["actions"])
    assert np.array_equal(obs[:, 0], f32(g["obs"]).reshape(obs[:, 0].shape))
    assert np.array_equal(rew[:, 0], f32(g["rew"]))
    assert np.array_equal(done[:, 0].astype(bool), g["done"]) and np.array_equal(removed[:, 0], g["removed"])


@needs_cxx
@pytest.mark.parametrize("name", CL_WW)
def test_emulated_waterworld_policy_reproduces_reference_closed_loop(name):
    from emu.driver import EmuWaterworld
    g = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    eng = EmuWaterworld(1, seed=int(g["seed"]), env_id_base=int(g["env_id"]), **json.loads(str(g["config"])))
    check_closed_loop_golden_ww(g, eng.reset, lambda T, o: eng.rollout_heuristic(T, o, auto_reset=False), 1e-9)
    assert eng.state(0)["counter"] == int(g["counter"])


@needs_cxx
@pytest.mark.parametrize("name", CL_PE)
def test_emulated_pursuit_policy_reproduces_reference_closed_loop(name):
    from emu.driver import EmuPursuit
    g = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    maps = pool16() if str(g["maps"]) == "pool16" else small_map()
    eng = EmuPursuit(1, maps, seed=int(g["seed"]), env_id_base=int(g["env_id"]), **json.loads(str(g["config"])))
    check_closed_loop_golden_pe(g, eng.reset, lambda T, o: eng.rollout_heuristic(T, o, auto_reset=False,
                                                                                py2_division=bool(g["py2"])))
    assert eng.state(0)["counter"] == int(g["counter"])


# ------------------------------------------------------------------------------ random configurations
@needs_cxx
@pytest.mark.parametrize("case", range(6))
def test_emulated_waterworld_policy_random_configurations(case):
    """Every template shape of the POLICY instantiation (1-8 objects per lane, 1-2 sensors per lane, compile-time and
    run-time K, global / local reward, random obstacle, horizon resets) closes the loop like the oracle does."""
    from emu.driver import EmuWaterworld
    rs = np.random.RandomState(1000 + case)
    Np = int(rs.choice([1, 2, 3, 7, 12, 32]))
    shape = [(3, 2), (20, 9), (60, 40), (120, 100), (4, 4), (1, 1)][case]
    cfg = dict(n_pursuers=Np, n_evaders=int(shape[0]), n_poison=int(shape[1]), n_sensors=int(rs.choice([1, 5, 30, 33, 64])),
               n_coop=int(rs.choice([1, 2])), radius=float(rs.choice([0.015, 0.04])), sensor_range=float(rs.choice([0.2, 0.35])),
               reward_mech=str(rs.choice(['local', 'global'])), addid=bool(rs.randint(2)),
               obstacle_loc=None if rs.randint(2) else np.array([0.5, 0.5]))
    if Np + shape[0] + shape[1] > 256:
        cfg['n_pursuers'] = Np = 8
    E, T, seed, base, mpl = 2, 7, 77 + case, 10 * case, 5
    eng = EmuWaterworld(E, seed=seed, env_id_base=base, max_path_length=mpl, **cfg)
    obs0 = eng.reset()
    act, obs, rew, done, info = eng.rollout_heuristic(T, obs0, auto_reset=True)
    # a sum that cancels to rounding noise is normalised to a noise-determined direction (see DESIGN.md section 5):
    # such decisions (norm < 1e-9) are not comparable, everything downstream of one is skipped
    for e in range(E):
        o = WaterworldOracle(rng=Stream(seed, base + e), **cfg)
        o.reset()
        prev, ts = obs0[e].astype(np.float64), 0
        for t in range(T):
            norms = [waterworld_action(prev[i], return_norm=True) for i in range(Np)]
            if any(0 < n_ < 1e-9 for _, n_ in norms):
                break
            for i, (want, _) in enumerate(norms):
                assert np.abs(want - act[t, e, i]).max() < 1e-9, (t, e, i)
            oo, rr, dd, ii = o.step(act[t, e].astype(np.float64))
            ts += 1
            dd = dd or ts >= mpl
            assert bool(done[t, e]) == dd and [ii['evcatches'], ii['pocatches']] == list(info[t, e])
            if dd:
                oo, ts = o.reset(), 0
            assert np.abs(np.array(oo) - obs[t, e]).max() < 1e-9 and np.abs(rr - rew[t, e]).max() < 1e-9
            prev = obs[t, e].astype(np.float64)


@needs_cxx
@pytest.mark.parametrize("case", range(5))
def test_emulated_pursuit_policy_random_configurations(case):
    from emu.driver import EmuPursuit
    rs = np.random.RandomState(2000 + case)
    R = int(rs.choice([1, 2, 3, 6, 11]))
    cfg = dict(n_evaders=int(rs.choice([1, 5, 33, 64])), n_pursuers=int(rs.choice([1, 4, 9, 32])), obs_range=R,
               surround=bool(rs.randint(2)), n_catch=int(rs.choice([1, 2])), flatten=bool(rs.randint(2)),
               reward_mech=str(rs.choice(['local', 'global'])), catchr=0.1, sample_maps=True, include_id=bool(rs.randint(2)))
    maps = pool16() if case % 2 == 0 else small_map()
    E, T, seed, base, mpl = 2, 12, 55 + case, 7 * case, 5
    py2 = bool(case % 2)
    eng = EmuPursuit(E, maps, seed=seed, env_id_base=base, max_path_length=mpl, **cfg)
    obs0 = eng.reset()
    act, obs, rew, done, removed = eng.rollout_heuristic(T, obs0, auto_reset=True, py2_division=py2)
    check_pursuit_closed_loop(maps, cfg, seed, base, obs0, act, obs, rew, done, removed, mpl, py2)
