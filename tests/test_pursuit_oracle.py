"""Pin the PursuitEvade oracle: golden vectors recorded from the real reference and long bit-exact
differential runs against it (its side recorded, tests/reference_record.py)."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN_DIR, ROOT
from oracle.philox import Stream
from oracle.pursuit_oracle import PursuitOracle
from reference_record import assert_same_trace, recorded, trace

PE_GOLDEN = ["pe_c3", "pe_c3_global", "pe_ncatch", "pe_window", "pe_small", "pe_even_range", "pe_crowd", "pe_random_opp"]


def small_map():
    m = np.zeros((1, 5, 5), dtype=np.int32)
    m[0, 2, 2] = -1
    return m


def load_pe_golden(name):
    g = np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False)
    cfg = json.loads(str(g["config"]))
    maps = np.load(os.path.join(ROOT, "maps", "map_pool16.npy")) if str(g["maps"]) == "pool16" else small_map()
    return g, cfg, maps


def test_map_pool_fixture():
    mp = np.load(os.path.join(ROOT, "maps", "map_pool16.npy"))
    assert mp.shape == (10, 16, 16) and mp.dtype == np.int32 and set(np.unique(mp)) == {-1, 0}
    assert 60 <= (mp[0] == -1).sum() <= 88


@pytest.mark.parametrize("name", PE_GOLDEN)
def test_oracle_reproduces_golden(name):
    g, cfg, maps = load_pe_golden(name)
    o = PursuitOracle(maps, rng=Stream(int(g["seed"]), int(g["env_id"])), **cfg)
    assert np.array_equal(np.array(o.reset()), g["obs0"])
    resets = list(g["reset_at"])
    k = 0
    for t in range(g["actions"].shape[0]):
        obs, rew, done, info = o.step(g["actions"][t])
        assert np.array_equal(np.array(obs), g["obs"][t]), t
        assert np.array_equal(np.asarray(rew, dtype=np.float64), g["rew"][t]), t
        assert done == bool(g["done"][t]) and info["removed"] == int(g["removed"][t])
        if k < len(resets) and resets[k] == t:
            assert np.array_equal(np.array(o.reset()), g["reset_obs"][k])
            k += 1
    assert o.rng.counter == int(g["counter"])


@pytest.mark.parametrize("kw,steps,seed,small", [
    (dict(n_evaders=30, n_pursuers=8, obs_range=7, surround=True, n_catch=2, flatten=True,
          reward_mech='local', catchr=0.1, term_pursuit=5.0, sample_maps=True, include_id=True), 500, 1, False),
    (dict(n_evaders=20, n_pursuers=12, obs_range=5, surround=False, reward_mech='global', catchr=0.1,
          sample_maps=True, urgency_reward=-0.1), 400, 3, False),
    (dict(n_evaders=2, n_pursuers=4, obs_range=3, surround=True, reward_mech='local', catchr=0.1), 1500, 5, True),
    (dict(n_evaders=3, n_pursuers=3, obs_range=4, surround=False, n_catch=1, reward_mech='global',
          flatten=False), 300, 6, True),
    # random_opponents (pursuit_evade.py:81-82,177-181): 1..max_opponents-1 evaders per episode
    (dict(n_evaders=5, n_pursuers=6, obs_range=3, surround=False, n_catch=1, reward_mech='local', catchr=0.1,
          random_opponents=True, max_opponents=6), 600, 8, True),
])
def test_oracle_equals_reference_bitwise(kw, steps, seed, small):
    """The oracle and the reference class, same stream and actions, reset after a done step and every 97 steps:
    every observation, reward, done, info and reset identical and the same number of draws (reference side
    recorded)."""
    maps = small_map() if small else np.load(os.path.join(ROOT, "maps", "map_pool16.npy"))
    ar = np.random.RandomState(seed)
    actions = [ar.randint(0, 5, size=kw['n_pursuers']) for _ in range(steps)]
    every97 = lambda t: t % 97 == 96                                       # noqa: E731

    def reference():
        from oracle.refshim import make_reference_pursuit
        ref = make_reference_pursuit(maps, Stream(seed, 5), **kw)
        return dict(trace(ref, actions, every97), counter=ref.evader_controller.rng.counter)
    orc = PursuitOracle(maps, rng=Stream(seed, 5), **kw)
    got = dict(trace(orc, actions, every97), counter=orc.rng.counter)
    assert_same_trace(got, recorded("pe_oracle_s%d" % seed, reference))


def test_scripted_quirks():
    """Known answers for the reference quirks of SURVEY.md 8a (values derived by hand from the code)."""
    m = np.zeros((1, 6, 6), dtype=np.int32)
    m[0, 0, 3] = -1
    o = PursuitOracle(m, n_evaders=1, n_pursuers=4, obs_range=3, catchr=0.1, reward_mech='local',
                      rng=Stream(1, 0))
    o.reset()
    # need_to_surround ignores buildings in row/column 0: (1,3) next to building (0,3) still needs 4
    assert o._need_to_surround(1, 3) == 4
    assert o._need_to_surround(0, 0) == 2 and o._need_to_surround(0, 2) == 3
    # a corner pursuer counts its own (clipped) cell: 3 * catchr with one evader on (0,0)... (pe:374-380)
    o.ppos[:] = [[0, 0], [5, 5], [5, 4], [4, 5]]
    o.epos[:] = [[0, 0]]
    r = o._reward()
    assert r[0] == pytest.approx(0.2) and r[1] == 0.0     # clip(-1)->0 twice => own cell counted twice
    # a captured evader is still visible in the observation of the capturing step (pe:244-251)
    o.ppos[:] = [[1, 2], [3, 2], [2, 1], [2, 4]]
    o.epos[:] = [[2, 2]]
    o.rng = type("Stay", (), {"randint": lambda self, *a: 4, "counter": 0})()
    obs, rew, done, info = o.step([4, 4, 4, 3])            # 4th pursuer moves (2,4)->(2,3): surrounded
    assert info["removed"] == 1 and done
    assert obs[0][2 * 9 + 2 * 3 + 1] == np.float32(0.1)   # channel 2, window cell (2,1) = map (2,2)
    assert np.all(rew >= 5.0)
