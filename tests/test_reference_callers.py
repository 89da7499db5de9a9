"""The drop-in boundary as the REFERENCE'S OWN callers exercise it (CPU).

INTEGRATION.md claims that the existing runners / samplers run unchanged on the drop-in classes.  The
callers below were run, unmodified (``oracle/refshim.py``), over the reference env wrapped in ``CallLog``,
which recorded every reset() / step(action) they made and what the env returned
(tests/reference_record.py, tests/golden/ref_callers_*.npz).  Here the drop-in class receives exactly
those calls, on the same injected Philox stream, and must return what the reference env returned; a
caller only sees what the env returns, so it produces the same over either:

  * the env wrappers ``ObservationBuffer`` / ``StandardizedEnv`` / ``DiagnosticsWrapper``
    (madrl_environments/__init__.py:143-389),
  * rltools ``decrollout`` (rltools/rltools/samplers/__init__.py:148-190),
  * ``RLLabEnv`` + rllab ``dec_rollout`` (rllabwrapper/__init__.py:29-90, rllab/rllab/sampler/ma_sampler.py:52-100),
  * rllab ``VecEnvExecutor`` (rllab/sandbox/rocky/tf/envs/vec_env_executor.py:6-48): its recorded outputs
    against those of the ``env.vec_env_executor(n_envs, max_path_length)`` hook.

The drop-in classes run on the emulator build of the kernels here (tests/emu ``emulated_dropins``:
only the engine object is swapped, the class code is the product's); under ``-m gpu`` the same
classes are covered on the real library by tests/test_*_gpu.py::test_dropin_env_surface.
"""
import json

import numpy as np
import pytest
import torch

from oracle.philox import Stream
from reference_record import recorded

WW_KW = dict(n_pursuers=3, n_evaders=4, n_poison=3, n_sensors=8, n_coop=1, radius=0.05, sensor_range=0.3)
HW_ARGS, HW_KW = (3, 5, 4, 1, 1), dict(radius=0.05, n_sensors=8, sensor_range=0.3, key_radius=0.06)
PE_MAPS_KW = dict(n_evaders=3, n_pursuers=4, obs_range=3, surround=False, n_catch=1, reward_mech='local', catchr=0.1,
                  sample_maps=False)
SEED = 31


def pe_maps():
    maps = np.zeros((1, 6, 6), dtype=np.int32)
    maps[0, 2, 3] = -1
    return maps


@pytest.fixture()
def world():
    """The drop-in classes, on the emulator build of the kernels."""
    import madrl_b200
    from emu.driver import emulated_dropins
    with emulated_dropins():
        yield dict(ours=(madrl_b200.MAWaterWorld, madrl_b200.PursuitEvade, madrl_b200.ContinuousHostageWorld))


def make_ref(family, env_id=0):
    """The reference env of one family on the stream key (SEED, env_id) (recording only)."""
    from oracle.refshim import load_reference, make_reference_pursuit
    RefWW, _, RefHW = load_reference()
    if family == "pe":
        return make_reference_pursuit(pe_maps(), Stream(SEED, 5), **PE_MAPS_KW)
    ref = RefWW(**WW_KW) if family == "ww" else RefHW(*HW_ARGS, **HW_KW)
    ref.np_random = Stream(SEED, env_id)
    return ref


def make_ours(world, family, env_id=0):
    """The drop-in env of one family on the same stream key as make_ref."""
    OurWW, OurPE, OurHW = world["ours"]
    if family == "pe":
        return OurPE(pe_maps(), seed=SEED, env_id=5, **PE_MAPS_KW)
    if family == "ww":
        return OurWW(seed=SEED, env_id=env_id, dtype=torch.float64, **WW_KW)
    return OurHW(*HW_ARGS, seed=SEED, env_id=env_id, dtype=torch.float64, **HW_KW)


def same(a, b, tol=1e-9):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and (a.size == 0 or float(np.abs(a - b).max()) <= tol)


def plain(x):
    """JSON-comparable form of an info dict (NumPy scalars and arrays as Python values)."""
    return json.loads(json.dumps(x, default=lambda v: v.tolist()))


class CallLog(object):
    """Stands in for an env: forwards everything to it and records each reset() / step(action) with its result."""

    def __init__(self, env):
        self.__dict__.update(env_=env, calls=[])

    def __getattr__(self, k):
        return getattr(self.env_, k)

    def __setattr__(self, k, v):
        setattr(self.env_, k, v)

    def reset(self):
        o = self.env_.reset()
        self.calls.append((None, o))
        return o

    def step(self, a):
        out = self.env_.step(a)
        self.calls.append((np.array(a),) + tuple(out))
        return out

    def arrays(self, p):
        """The calls as arrays named p + '_*'; `reset` marks the reset() calls, the step results are in call order."""
        steps = [c for c in self.calls if c[0] is not None]
        return {p + "_reset": np.array([c[0] is None for c in self.calls]),
                p + "_obs": np.array([np.asarray(c[1], dtype=np.float64) for c in self.calls]),
                p + "_act": np.array([c[0] for c in steps]),
                p + "_rew": np.array([np.asarray(c[2], dtype=np.float64) for c in steps]),
                p + "_done": np.array([bool(c[3]) for c in steps]),
                p + "_info": json.dumps([plain(c[4]) for c in steps])}


def replay(env, g, p, cast=lambda x: x, obs_tol=1e-9):
    """Makes the recorded calls p on `env`: every result must be what the reference env returned.  Returns the
    number of step() calls."""
    infos, k = json.loads(str(g[p + "_info"])), 0
    for n, is_reset in enumerate(g[p + "_reset"]):
        if is_reset:
            o = env.reset()
        else:
            o, r, d, i = env.step(g[p + "_act"][k])
            assert same(cast(r), cast(g[p + "_rew"][k])) and d == bool(g[p + "_done"][k]), (p, n)
            assert plain(i) == infos[k], (p, n, i, infos[k])
            k += 1
        assert same(cast(o), cast(g[p + "_obs"][n]), obs_tol), (p, n)
    return k


def surface(env):
    """What the callers read from an env besides reset() / step()."""
    return dict(n_agents=len(env.agents), reward_mech=env.reward_mech,
                timestep_limit=getattr(env, "timestep_limit", -1),
                obs_shape=np.array([ag.observation_space.shape for ag in env.agents]),
                act_dims=np.array([getattr(ag.action_space, "shape", None) or (ag.action_space.n,)
                                   for ag in env.agents]),
                obs_low=np.array([ag.observation_space.low for ag in env.agents]))


def assert_same_surface(ours, g):
    s = surface(ours)
    for k, v in s.items():
        assert np.array_equal(np.asarray(v), g[k]), k


# ------------------------------------------------------------------------------------ wrappers
@pytest.mark.parametrize("family", ["ww", "hw"])
def test_reference_wrappers_around_dropin_equal_wrappers_around_reference(world, family):
    def reference():
        from oracle.refshim import install
        install()
        import madrl_environments as me

        def stack(env):
            # ObservationBuffer.__init__ assigns to its own read-only `reward_mech` property
            # (madrl_environments/__init__.py:151 vs :171) and raises for ANY env, the reference's included;
            # the runners never enable it (buffer_size 1).  Its step/reset logic is exercised by building the
            # object the way its __init__ would have.
            with pytest.raises(AttributeError):
                me.ObservationBuffer(env, 3)
            ob = me.ObservationBuffer.__new__(me.ObservationBuffer)
            ob._unwrapped, ob._buffer_size = env, 3
            ob._buffer = [np.zeros(tuple(ag.observation_space.shape) + (3,)) for ag in env.agents]
            std = me.StandardizedEnv(env, scale_reward=0.5, enable_obsnorm=True, enable_rewnorm=True, obs_alpha=0.05,
                                     rew_alpha=0.02)
            return ob, std, me.DiagnosticsWrapper(std, discount=0.9, max_traj_len=20, log_interval=10 ** 9)

        # two independent envs: ObservationBuffer and the StandardizedEnv/Diagnostics chain both step the env
        ref, ref2 = CallLog(make_ref(family)), CallLog(make_ref(family))
        ob, _, _ = stack(ref)
        _, _, dg = stack(ref2)
        ob.reset(), dg.reset()
        rs = np.random.RandomState(1)
        logs = 0
        for t in range(50):
            act = rs.randn(len(ref.agents), 2) * 2.0
            ob.step(act)
            _, _, d, log = dg.step(act)
            logs += bool(log)
            if d:
                dg.reset(), ob.reset()
        return dict(surface(ref.env_), logs=logs, **ref.arrays("buffer"), **ref2.arrays("diagnostics"))
    g = recorded("callers_wrappers_" + family, reference)
    ours, ours2 = make_ours(world, family), make_ours(world, family)
    assert_same_surface(ours, g)
    assert replay(ours, g, "buffer") == replay(ours2, g, "diagnostics") == 50
    assert g["logs"] >= 2


# ------------------------------------------------------------------------------------ rltools
class ScriptedPolicy(object):
    """What decrollout / dec_rollout need from a policy: per-agent actions from a seeded stream."""

    def __init__(self, n_agents, discrete, seed=3):
        self.n, self.discrete, self.seed = n_agents, discrete, seed

    def reset(self, dones=None):
        self.rs = np.random.RandomState(self.seed)

    def _draw(self):
        if self.discrete:
            return self.rs.randint(0, 5, size=(self.n, 1))
        return self.rs.randn(self.n, 2) * 2.0

    def sample_actions(self, obs):                  # rltools
        assert np.asarray(obs).shape[0] == self.n
        a = self._draw()
        return list(a), list(a.astype(np.float64))

    def get_actions(self, olist):                   # rllab
        assert len(olist) == self.n
        a = self._draw()
        return (list(a[:, 0]) if self.discrete else list(a)), dict(mean=a.astype(np.float64))


@pytest.mark.parametrize("family", ["ww", "hw", "pe"])
def test_rltools_decrollout_over_dropin_equals_over_reference(world, family):
    def reference():
        from oracle.refshim import load_rltools_samplers
        samplers = load_rltools_samplers()
        env = CallLog(make_ref(family))
        pol = ScriptedPolicy(len(env.agents), discrete=(family == "pe"))
        trajs = samplers.decrollout(env, pol, 40, env.agents[0].action_space)
        return dict(traj_lens=np.array([len(t) for t in trajs]), **env.arrays("decrollout"))
    g = recorded("callers_decrollout_" + family, reference)
    ours = make_ours(world, family)
    # Pursuit contract (SURVEY.md 8a): observations identical after casting the reference's float64 to
    # float32 -- the reference mixes float64 0.1 (out-of-bounds fill) with widened float32(0.1) cells
    cast = (lambda x: np.asarray(x, np.float64).astype(np.float32)) if family == "pe" else (lambda x: x)
    n = replay(ours, g, "decrollout", cast, 0.0 if family == "pe" else 1e-9)
    assert len(g["traj_lens"]) == len(ours.agents) >= 3 and all(g["traj_lens"] == n) and n >= 10


# ------------------------------------------------------------------------------------ rllab
@pytest.mark.parametrize("family", ["ww", "hw"])
def test_rllab_dec_rollout_through_rllabenv(world, family):
    def reference():
        from oracle.refshim import load_rllab_callers
        RLLabEnv, ma_sampler, _ = load_rllab_callers()
        env = CallLog(make_ref(family))
        wrapped = RLLabEnv(env, ma_mode='decentralized')          # reads agents[0] spaces, timestep_limit
        path = ma_sampler.dec_rollout(wrapped, ScriptedPolicy(len(env.agents), discrete=False), max_path_length=30)
        return dict(surface(env.env_), horizon=wrapped.horizon, flat_dim=wrapped.observation_space.flat_dim,
                    path_lens=np.array([p['observations'].shape[0] for p in path]), **env.arrays("dec_rollout"))
    g = recorded("callers_dec_rollout_" + family, reference)
    ours = make_ours(world, family)
    assert_same_surface(ours, g)
    assert g["horizon"] == ours.timestep_limit == 1000 and g["flat_dim"] == ours.agents[0].observation_space.shape[0]
    assert replay(ours, g, "dec_rollout") == 30 and all(g["path_lens"] == 30)


@pytest.mark.parametrize("family", ["ww", "hw"])
def test_vec_env_executor_hook_equals_reference_vec_env_executor(world, family):
    """rllab's VecEnvExecutor over n reference envs (stream keys (SEED, 0..n-1)) against the batched
    executor the drop-in class hands out through `env.vec_env_executor(n, max_path_length)`: same
    obs lists, rewards, dones (horizon cut-off + reset in place) and stacked env_infos."""
    n, mpl, T = 3, 7, 20
    rs = np.random.RandomState(2)
    acts = [rs.randn(n, (WW_KW["n_pursuers"] if family == "ww" else HW_ARGS[0]), 2) * 2.0 for _ in range(T)]

    def reference():
        from oracle.refshim import load_rllab_callers
        RLLabEnv, _, VecEnvExecutor = load_rllab_callers()
        ref_ex = VecEnvExecutor([RLLabEnv(make_ref(family, env_id=i), ma_mode='decentralized') for i in range(n)], mpl)
        out = dict(num_envs=ref_ex.num_envs, obs0=np.asarray(ref_ex.reset(), dtype=np.float64))
        steps = [ref_ex.step(list(a)) for a in acts]
        keys = sorted(steps[0][3])
        out.update(obs=np.array([np.asarray(s[0], dtype=np.float64) for s in steps]),
                   rew=np.array([np.asarray(s[1], dtype=np.float64) for s in steps]),
                   done=np.array([np.asarray(s[2]) for s in steps]), info_keys=json.dumps(keys))
        return dict(out, **{"info_" + k: np.array([s[3][k] for s in steps]) for k in keys})
    g = recorded("callers_vec_env_executor_" + family, reference)
    ours = make_ours(world, family)
    assert ours.vectorized is True
    our_ex = ours.vec_env_executor(n_envs=n, max_path_length=mpl)
    assert our_ex.num_envs == g["num_envs"] == n
    assert our_ex.observation_space.shape == ours.agents[0].observation_space.shape
    assert same(g["obs0"], our_ex.reset())
    keys = json.loads(str(g["info_keys"]))
    for t in range(T):
        o2, r2, d2, i2 = our_ex.step(acts[t])
        assert same(g["obs"][t], o2) and same(g["rew"][t], r2) and np.array_equal(g["done"][t], d2), t
        assert keys == sorted(i2) and all(np.array_equal(g["info_" + k][t], i2[k]) for k in keys), t
    assert int(np.sum(g["done"])) >= 2 * n


# ------------------------------------------------------------------------------------ heuristic policies
def test_reference_policies_drive_the_dropin_envs(world):
    """The reference's hand-written policies (heuristics/waterworld.py, heuristics/pursuit.py, as restated in
    oracle/heuristics_oracle.py and pinned to the reference classes in tests/test_heuristics.py) stepping the
    drop-in env classes per agent, as the reference's Visualizer does, reproduce the closed-loop goldens that the
    same policies produced on the reference envs (tests/golden/cl_*.npz)."""
    import os
    from conftest import GOLDEN_DIR, ROOT
    from oracle.heuristics_oracle import policy_draw, pursuit_action, waterworld_action
    OurWW, OurPE, _ = world["ours"]
    g = np.load(os.path.join(GOLDEN_DIR, "cl_ww_c2.npz"))
    env = OurWW(seed=int(g["seed"]), env_id=int(g["env_id"]), dtype=torch.float64, **json.loads(str(g["config"])))
    o = env.reset()
    assert np.abs(np.array(o) - g["obs0"]).max() < 1e-9
    for t in range(60):
        a = np.array([waterworld_action(np.asarray(oi)) for oi in o])
        assert np.abs(a - g["actions"][t]).max() < 1e-9, t
        o, r, d, i = env.step(a)
        assert np.abs(np.array(o) - g["obs"][t]).max() < 1e-9 and np.abs(r - g["rew"][t]).max() < 1e-9
        assert [i['evcatches'], i['pocatches']] == list(g["info"][t])
    # Pursuit (heuristics/pursuit.py as it runs under Python 3: true division)
    g = np.load(os.path.join(GOLDEN_DIR, "cl_pe_conv_py3.npz"))
    maps = np.load(os.path.join(ROOT, "maps", "map_pool16.npy"))
    seed, env_id = int(g["seed"]), int(g["env_id"])
    env = OurPE(maps, seed=seed, env_id=env_id, **json.loads(str(g["config"])))

    def sample():
        raise AssertionError("every pursuer of this golden sees an evader")

    o = env.reset()
    assert np.array_equal(np.array(o, dtype=np.float32), np.asarray(g["obs0"], dtype=np.float32))
    for t in range(40):
        a = [int(pursuit_action(np.asarray(oq), sample, False)) for oq in o]
        assert a == list(g["actions"][t]), t
        o, r, d, i = env.step(a)
        assert np.array_equal(np.array(o, dtype=np.float32), np.asarray(g["obs"][t], dtype=np.float32))
        assert i['removed'] == g["removed"][t] and d == bool(g["done"][t])
    assert policy_draw(seed, env_id, 0, 0) in range(5)
