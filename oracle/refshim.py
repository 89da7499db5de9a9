"""Import shim for the REAL sisl/MADRL reference classes (test infrastructure only).

TEST INFRASTRUCTURE -- never imported by the product package ``madrl_b200``.

The reference (``/root/reference``) is pure Python but cannot be imported unmodified on this
image: ``rltools/rltools/util.py`` is a SyntaxError on Python >= 3.7 and ``gym`` / ``matplotlib``
are not installed (SURVEY.md section 8c).  This module registers *stub modules* for exactly those
imports in ``sys.modules`` and puts the reference root on ``sys.path`` so that

    madrl_environments.pursuit.waterworld.MAWaterWorld
    madrl_environments.pursuit.pursuit_evade.PursuitEvade
    madrl_environments.hostage.ContinuousHostageWorld

can be imported and executed UNMODIFIED.  No reference file is copied or edited.  Only recording
uses this shim (``oracle/make_golden.py`` and ``MADRL_RECORD_REFERENCE=1`` runs of the tests,
tests/reference_record.py); the tests compare with the golden vectors it produced (``tests/golden``).

Stub behaviour follows the originals:
  * ``rltools.util.EzPickle``      -- pickle by constructor args (rltools/rltools/util.py:261-288)
  * ``rltools.util.stack_dict_list`` -- (rltools/rltools/util.py:125-138)
  * ``gym.spaces.Box/Discrete``    -- shape/low/high/n holders
  * ``gym.utils.seeding.np_random``-- returns (numpy RandomState, seed)
"""
import os
import sys
import types

import numpy as np

REFERENCE_ROOT = os.environ.get("MADRL_REFERENCE_ROOT", "/root/reference")


def reference_available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "madrl_environments"))


class _EzPickle(object):
    def __init__(self, *args, **kwargs):
        self._ezpickle_args = args
        self._ezpickle_kwargs = kwargs

    def __getstate__(self):
        return {"_ezpickle_args": self._ezpickle_args, "_ezpickle_kwargs": self._ezpickle_kwargs}

    def __setstate__(self, d):
        out = type(self)(*d["_ezpickle_args"], **d["_ezpickle_kwargs"])
        self.__dict__.update(out.__dict__)


def _stack_dict_list(dict_list):
    ret = dict()
    if not dict_list:
        return ret
    for k in dict_list[0].keys():
        eg = dict_list[0][k]
        if isinstance(eg, dict):
            ret[k] = _stack_dict_list([x[k] for x in dict_list])
        else:
            ret[k] = np.array([x[k] for x in dict_list])
    return ret


class _Box(object):
    def __init__(self, low, high, shape=None):
        if shape is None:
            self.low = np.asarray(low, dtype=np.float64)
            self.high = np.asarray(high, dtype=np.float64)
        else:
            self.low = np.full(shape, low, dtype=np.float64)
            self.high = np.full(shape, high, dtype=np.float64)

    @property
    def shape(self):
        return self.low.shape


class _Discrete(object):
    def __init__(self, n):
        self.n = n


def _np_random(seed=None):
    return np.random.RandomState(seed), seed


def _module(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


_installed = False


def install():
    """Register the stubs and make the reference importable.  Idempotent."""
    global _installed
    if _installed:
        return
    if not reference_available():
        raise RuntimeError("reference tree not found at %s" % REFERENCE_ROOT)
    if not hasattr(np, "bool"):
        np.bool = bool  # pursuit_evade.py:476 uses the alias removed in NumPy >= 1.24
    # rltools.util (the real file does not parse on py3.7+)
    rl = _module("rltools")
    rl.util = _module("rltools.util", EzPickle=_EzPickle, stack_dict_list=_stack_dict_list)
    # gym
    if "gym" not in sys.modules:
        gym = _module("gym")
        gym.spaces = _module("gym.spaces", Box=_Box, Discrete=_Discrete)
        gym.utils = _module("gym.utils")
        gym.utils.seeding = _module("gym.utils.seeding", np_random=_np_random)
        gym.error = _module("gym.error", InvalidFrame=type("InvalidFrame", (Exception,), {}))
        gym.monitoring = _module("gym.monitoring")
        gym.monitoring.video_recorder = _module("gym.monitoring.video_recorder",
                                                ImageEncoder=type("ImageEncoder", (object,), {}))
    # matplotlib (render/animate only)
    try:
        import matplotlib.pyplot  # noqa: F401
        import matplotlib.animation  # noqa: F401
    except Exception:
        mpl = _module("matplotlib")
        mpl.animation = _module("matplotlib.animation")
        mpl.pyplot = _module("matplotlib.pyplot")
        mpl.patches = _module("matplotlib.patches", Rectangle=type("Rectangle", (object,), {}))
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    _installed = True


def load_reference():
    """Returns (MAWaterWorld, PursuitEvade, ContinuousHostageWorld) -- the real reference classes."""
    install()
    from madrl_environments.pursuit.waterworld import MAWaterWorld
    from madrl_environments.pursuit.pursuit_evade import PursuitEvade
    from madrl_environments.hostage import ContinuousHostageWorld
    return MAWaterWorld, PursuitEvade, ContinuousHostageWorld


def load_rllab_numeric():
    """(rllab.algos.util, rllab.misc.special) loaded from their files with the theano / rllab
    package imports stubbed out -- only their NumPy functions are used (center_advantages,
    shift_advantages_to_positive, explained_variance_1d, discount_cumsum)."""
    import importlib.util
    if not reference_available():
        raise RuntimeError("reference tree not found at %s" % REFERENCE_ROOT)
    saved = dict(sys.modules)
    try:
        for name in ("theano", "theano.tensor", "theano.tensor.nnet", "theano.tensor.extra_ops", "rllab",
                     "rllab.core", "rllab.misc"):
            _module(name)
        sys.modules["theano"].tensor = sys.modules["theano.tensor"]
        sys.modules["theano.tensor"].nnet = sys.modules["theano.tensor.nnet"]
        sys.modules["theano.tensor"].extra_ops = sys.modules["theano.tensor.extra_ops"]
        _module("rllab.core.serializable", Serializable=type("Serializable", (object,), {}))
        _module("rllab.misc.ext", extract=lambda *a, **k: None)
        out = []
        for rel, name in (("rllab/rllab/algos/util.py", "_ref_rllab_algos_util"),
                          ("rllab/rllab/misc/special.py", "_ref_rllab_misc_special")):
            spec = importlib.util.spec_from_file_location(name, os.path.join(REFERENCE_ROOT, rel))
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
            out.append(mod)
        return tuple(out)
    finally:
        for k in list(sys.modules):
            if k not in saved:
                del sys.modules[k]
        sys.modules.update(saved)


class _NumpyProxy(object):
    """Stands in for the ``np`` global of a reference module: ``.random`` is the injected stream,
    everything else is the real numpy."""

    def __init__(self, stream):
        self.random = stream

    def __getattr__(self, name):
        return getattr(np, name)


def make_reference_pursuit(map_pool, stream, **kwargs):
    """Real ``PursuitEvade`` whose every random draw (``np.random.randint/uniform`` in
    pursuit_evade.py:183-186 and utils/agent_utils.py:39-45, evader ``controller.act`` at
    pursuit_evade.py:240) comes from ``stream``.  The module-level ``np`` of the two reference
    modules is swapped for a proxy while the returned env is in use (single env at a time)."""
    install()
    from madrl_environments.pursuit import pursuit_evade as pe_mod
    from madrl_environments.pursuit.utils import agent_utils as au_mod
    from oracle.philox import StreamController
    proxy = _NumpyProxy(stream)
    pe_mod.np = proxy
    au_mod.np = proxy
    env = pe_mod.PursuitEvade(map_pool, evader_controller=StreamController(5, stream), **kwargs)
    env.np_random = stream      # pursuit_evade.py:179 (random_opponents) draws from self.np_random
    return env


def load_rllab_callers():
    """The reference's OWN callers of the env boundary, imported unmodified:
    ``(RLLabEnv, ma_sampler module, VecEnvExecutor)`` --
    rllabwrapper/__init__.py:29-90, rllab/rllab/sampler/ma_sampler.py (dec_rollout :52-100),
    rllab/sandbox/rocky/tf/envs/vec_env_executor.py:6-48.  theano / path.py / the process-pool modules
    are stubbed (none of them is touched by the code paths used); everything else is the real file."""
    install()
    import inspect
    if not hasattr(inspect, "getargspec"):      # removed in Python 3.11; rllab/core/serializable.py:13 uses it
        import collections
        _AS = collections.namedtuple("ArgSpec", "args varargs keywords defaults")

        def getargspec(f):
            fs = inspect.getfullargspec(f)
            return _AS(fs.args, fs.varargs, fs.varkw, fs.defaults)
        inspect.getargspec = getargspec
    for p in (os.path.join(REFERENCE_ROOT, "rllab"), REFERENCE_ROOT):
        if p not in sys.path:
            sys.path.insert(0, p)
    if "theano" not in sys.modules:
        th = _module("theano")
        th.tensor = _module("theano.tensor")
        th.tensor.nnet = _module("theano.tensor.nnet")
        th.tensor.extra_ops = _module("theano.tensor.extra_ops")
        th.config = types.SimpleNamespace(floatX="float32")
    if "path" not in sys.modules:
        _module("path", Path=type("Path", (str,), {}))
    import gym
    if not hasattr(gym, "envs"):
        gym.envs = _module("gym.envs")
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        import rllab.sampler  # noqa: F401  (the real package)
        for name in ("rllab.sampler.parallel_sampler", "rllab.sampler.stateful_pool"):
            if name not in sys.modules:
                _module(name, _get_scoped_G=None, _worker_set_env_params=None, singleton_pool=None)
        from rllab.sampler import ma_sampler
        from rllabwrapper import RLLabEnv
        # sandbox.rocky.tf.misc.tensor_utils is the only import of vec_env_executor.py besides numpy/pickle
        from rllab.misc import tensor_utils as _tu
        for name in ("sandbox", "sandbox.rocky", "sandbox.rocky.tf", "sandbox.rocky.tf.misc"):
            if name not in sys.modules:
                _module(name)
        import importlib.util
        spec = importlib.util.spec_from_file_location(
            "sandbox.rocky.tf.misc.tensor_utils",
            os.path.join(REFERENCE_ROOT, "rllab", "sandbox", "rocky", "tf", "misc", "tensor_utils.py"))
        try:
            tu = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(tu)
        except Exception:            # needs tensorflow: the stacking helpers are the same functions in rllab.misc
            tu = _tu
        sys.modules["sandbox.rocky.tf.misc.tensor_utils"] = tu
        sys.modules["sandbox.rocky.tf.misc"].tensor_utils = tu
        spec = importlib.util.spec_from_file_location(
            "_ref_vec_env_executor",
            os.path.join(REFERENCE_ROOT, "rllab", "sandbox", "rocky", "tf", "envs", "vec_env_executor.py"))
        vee = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(vee)
    return RLLabEnv, ma_sampler, vee.VecEnvExecutor


def load_rltools_samplers():
    """rltools/rltools/samplers/__init__.py (centrollout / decrollout / concrollout, :98-235) and
    trajutil.py loaded from their files; ``rltools.nn`` (TensorFlow) is a stub -- only the Sampler base
    class, which the rollout functions do not use, refers to it."""
    install()
    import importlib.util
    rl = sys.modules["rltools"]
    if "rltools.nn" not in sys.modules:
        rl.nn = _module("rltools.nn", Standardizer=object, NoOpStandardizer=object)
    if "rltools.trajutil" not in sys.modules:
        spec = importlib.util.spec_from_file_location(
            "rltools.trajutil", os.path.join(REFERENCE_ROOT, "rltools", "rltools", "trajutil.py"))
        tj = importlib.util.module_from_spec(spec)
        sys.modules["rltools.trajutil"] = tj
        spec.loader.exec_module(tj)
        rl.trajutil = tj
    spec = importlib.util.spec_from_file_location(
        "_ref_rltools_samplers", os.path.join(REFERENCE_ROOT, "rltools", "rltools", "samplers", "__init__.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def load_reference_heuristics():
    """heuristics/waterworld.py and heuristics/pursuit.py loaded from their files, with ``rltools.policy.Policy``
    (a TensorFlow ``nn.Model`` subclass, rltools/rltools/policy/__init__.py:4-22) replaced by a stub that keeps
    the two spaces.  Returns (WaterworldHeuristicPolicy, PursuitHeuristicPolicy, pursuit_source) -- the source
    text lets a test re-evaluate heuristics/pursuit.py:23 `xs / 2` with Python 2's integer division."""
    install()
    import importlib.util
    rl = sys.modules["rltools"]

    class Policy(object):
        def __init__(self, observation_space, action_space):
            self._observation_space, self._action_space = observation_space, action_space

        @property
        def observation_space(self):
            return self._observation_space

        @property
        def action_space(self):
            return self._action_space

    rl.policy = _module("rltools.policy", Policy=Policy)
    out = []
    for name in ("waterworld", "pursuit"):
        path = os.path.join(REFERENCE_ROOT, "heuristics", name + ".py")
        spec = importlib.util.spec_from_file_location("_ref_heuristics_" + name, path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        out.append(mod)
    with open(os.path.join(REFERENCE_ROOT, "heuristics", "pursuit.py")) as f:
        src = f.read()
    return out[0].WaterworldHeuristicPolicy, out[1].PursuitHeuristicPolicy, src
