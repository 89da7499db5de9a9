"""Pin the ContinuousHostageWorld oracle against golden vectors recorded from the real reference
and against long runs of the reference classes themselves (their side recorded, tests/reference_record.py)."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN_DIR
from oracle.hostage_oracle import HostageOracle
from oracle.philox import Stream
from reference_record import assert_same_trace, recorded, trace

HW_GOLDEN = ["hw_c5", "hw_c5_local", "hw_dense", "hw_k12"]


def load_hw_golden(name):
    g = np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False)
    kw = json.loads(str(g["config"]))
    if 'key_loc' in kw:
        kw['key_loc'] = np.array(kw['key_loc'])
    return g, tuple(int(a) for a in g["args"]), kw


@pytest.mark.parametrize("name", HW_GOLDEN)
def test_oracle_reproduces_golden(name):
    g, args, kw = load_hw_golden(name)
    o = HostageOracle(*args, rng=Stream(int(g["seed"]), int(g["env_id"])), **kw)
    assert np.array_equal(np.array(o.reset()), g["obs0"])
    resets, k = list(g["reset_at"]), 0
    for t in range(g["actions"].shape[0]):
        obs, rew, done, info = o.step(g["actions"][t])
        assert np.array_equal(np.array(obs), g["obs"][t]), t
        assert np.array_equal(rew, g["rew"][t]), t
        assert done == bool(g["done"][t]) and [info["ho_saved"], info["cr_encs"]] == list(g["info"][t])
        if k < len(resets) and resets[k] == t:
            assert np.array_equal(np.array(o.reset()), g["reset_obs"][k])
            k += 1
    assert o.np_random.counter == int(g["counter"])


@pytest.mark.parametrize("args,kw,steps,seed,std", [
    ((10, 16, 16, 4, 2), {}, 700, 1, 0.5),
    ((10, 16, 16, 4, 2), dict(reward_mech='local'), 700, 2, 2.0),
    ((3, 10, 5, 1, 2), dict(radius=0.05, sensor_range=0.35, key_radius=0.06, reward_mech='local', addid=False), 1500, 3, 3.0),
    ((4, 6, 8, 2, 1), dict(radius=0.04, n_sensors=12, key_radius=0.05, bomb_radius=0.02), 1500, 4, 3.0),
])
def test_oracle_equals_reference_bitwise(args, kw, steps, seed, std):
    """The oracle and the reference class, same stream and actions: every observation, reward, done, info and
    reset identical and the same number of draws (reference side recorded)."""
    ar = np.random.RandomState(seed)
    actions = [ar.randn(args[0] * 2) * std for _ in range(steps)]

    def reference():
        from oracle.refshim import load_reference
        ref = load_reference()[2](*args, **kw)
        ref.np_random = Stream(seed, 3)
        return dict(trace(ref, actions), counter=ref.np_random.counter)
    orc = HostageOracle(*args, rng=Stream(seed, 3), **kw)
    got = dict(trace(orc, actions), counter=orc.np_random.counter)
    assert_same_trace(got, recorded("hw_oracle_s%d" % seed, reference))


def test_scripted_quirks():
    o = HostageOracle(2, 2, 1, 1, 1, rng=Stream(4, 0), reward_mech='local')
    o.reset()
    key0 = o.key_loc.copy()
    o.reset()
    assert np.array_equal(o.key_loc, key0)                 # key location persists across resets (hw:148)
    assert o.t == 1                                        # reset consumes one step (hw:179)
    assert np.all(o.rx >= 0.5 + o.radius)                  # closed gate confines rescuers (hw:255-261)
    # an already-saved hostage is "saved" (and rewarded) again every step a rescuer sits on it
    s = o.get_state()
    s['gate_open'] = True
    s['rx'][:] = [[0.3, 0.2], [0.9, 0.9]]; s['rv'][:] = 0
    s['hx'][:] = [[0.3, 0.21], [0.8, 0.1]]
    s['cx'][:] = [[0.1, 0.9]]; s['cv'][:] = 0
    s['bomb'] = np.array([[0.01, 0.01]])
    s['saved'][:] = [True, False]
    o.set_state(s)
    obs, rew, done, info = o.step(np.zeros((2, 2)))
    assert info['ho_saved'] == 1 and rew[0] == pytest.approx(5.0 + 0.01)
