"""Pin the Waterworld oracle: golden vectors (from the real reference) and long differential runs
against the reference classes themselves (their side recorded, tests/reference_record.py)."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN_DIR
from oracle.philox import Stream
from reference_record import assert_same_trace, recorded, trace
from oracle.waterworld_oracle import WaterworldOracle

WW_GOLDEN = ["ww_c2", "ww_dense", "ww_c4", "ww_global_nospeed"]


def load_golden(name):
    g = np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False)
    cfg = json.loads(str(g["config"]))
    if "obstacle_loc" in cfg and cfg["obstacle_loc"] is not None:
        cfg["obstacle_loc"] = np.array(cfg["obstacle_loc"])
    return g, cfg


@pytest.mark.parametrize("name", WW_GOLDEN)
def test_oracle_reproduces_golden(name):
    g, cfg = load_golden(name)
    o = WaterworldOracle(rng=Stream(int(g["seed"]), int(g["env_id"])), **cfg)
    assert np.array_equal(np.array(o.reset()), g["obs0"])
    for t in range(g["actions"].shape[0]):
        obs, rew, done, info = o.step(g["actions"][t])
        assert np.array_equal(np.array(obs), g["obs"][t]), t
        assert np.array_equal(rew, g["rew"][t]), t
        assert done == bool(g["done"][t])
        assert [info["evcatches"], info["pocatches"]] == list(g["info"][t])
    assert np.array_equal(o.px, g["final_px"]) and np.array_equal(o.ex, g["final_ex"])
    assert np.array_equal(o.ov, g["final_ov"])
    assert o.np_random.counter == int(g["counter"])


@pytest.mark.parametrize("cfg,steps,seed", [
    (dict(n_pursuers=5, n_evaders=5), 1200, 1),
    (dict(n_pursuers=5, n_evaders=5, n_coop=1, obstacle_loc=None, reward_mech='global'), 1100, 2),
    (dict(n_pursuers=20, n_evaders=50, n_poison=50), 120, 3),
    (dict(n_pursuers=3, n_evaders=4, n_poison=2, n_sensors=7, speed_features=False, addid=False,
          n_coop=1, radius=0.05), 1100, 4),
])
def test_oracle_equals_reference_bitwise(cfg, steps, seed):
    """The oracle and the reference class, same stream and actions: every observation, reward, done, info and
    reset identical, the same number of draws, the same final evader positions (reference side recorded)."""
    ar = np.random.RandomState(seed)
    actions = [ar.randn(cfg['n_pursuers'] * 2) * 0.5 for _ in range(steps)]

    def reference():
        from oracle.refshim import load_reference
        ref = load_reference()[0](**cfg)
        ref.np_random = Stream(seed, 7)
        return dict(trace(ref, actions), counter=ref.np_random.counter,
                    final_ex=np.array([p.position for p in ref._evaders]))
    orc = WaterworldOracle(rng=Stream(seed, 7), **cfg)
    got = dict(trace(orc, actions), counter=orc.np_random.counter, final_ex=orc.ex)
    assert_same_trace(got, recorded("ww_oracle_s%d" % seed, reference))


def test_reset_consumes_one_step_and_quirks():
    """Scripted known answers for the reference quirks listed in SURVEY.md 8a."""
    o = WaterworldOracle(2, 2, n_poison=1, n_coop=1, rng=Stream(3, 0))
    o.reset()
    assert o.t == 1                                   # reset() returns step(zeros)[0]  (ww:172)
    # one pursuer catching two evaders at once is credited food_reward only once (ww:383)
    s = o.get_state()
    s['px'][:] = [[0.2, 0.2], [0.8, 0.8]]; s['pv'][:] = 0
    s['ex'][:] = [[0.2, 0.21], [0.21, 0.2]]; s['ev'][:] = 0
    s['ox'][:] = [[0.9, 0.1]]; s['ov'][:] = 0
    o.set_state(s)
    obs, rew, done, info = o.step(np.zeros((2, 2)))
    assert info['evcatches'] == 2
    assert rew[0] == pytest.approx(1.0 + 0.05) and rew[1] == 0.0
    # an evader leaving through ONE wall is not bounced and not clipped (ww:401)
    s = o.get_state()
    s['ex'][0] = [0.999, 0.5]; s['ev'][0] = [0.01, 0.0]
    o.set_state(s)
    o.step(np.zeros((2, 2)))
    assert o.ex[0, 0] > 1.0 and o.ev[0, 0] == 0.01
