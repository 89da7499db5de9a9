"""PursuitEvade on the B200 engine (integer path, bit-exact with the reference).

``BatchedPursuitEvade`` is the batched tensor API; ``PursuitEvade`` is the drop-in for
``madrl_environments.pursuit.pursuit_evade.PursuitEvade`` (constructor ``PursuitEvade(map_pool,
**kwargs)`` with the reference's keyword names, pursuit_evade.py:28-152) backed by a one-env
engine, including the curriculum attributes that survive pickling (pursuit_evade.py:397-411).
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._engine import _BatchedEngine, _HeuristicRollout
from .core import AbstractMAEnv, Agent, EzPickle
from .spaces import Box, Discrete


class DiscreteAgent(Agent):
    """Per-pursuer descriptor (utils/DiscreteAgent.py:11-62): spaces only."""

    def __init__(self, obs_range=3, n_channels=3, flatten=False):
        self._obs_range = obs_range
        if flatten:
            self._obs_shape = (n_channels * obs_range ** 2 + 1,)
        else:
            self._obs_shape = (obs_range, obs_range, 4)

    @property
    def observation_space(self):
        return Box(low=-np.inf, high=np.inf, shape=self._obs_shape)

    @property
    def action_space(self):
        return Discrete(5)


class BatchedPursuitEvade(_HeuristicRollout, _BatchedEngine):
    """E lockstep PursuitEvade instances resident in HBM.

    Keyword names follow pursuit_evade.py:49-148.  Evader motion uses the env's counter-based
    stream (the reference's default controller is an unseeded RandomState shared by every
    instance, utils/Controllers.py:11, so there is no reference stream to reproduce).
    Actions int32 [T, E, Np]; obs / rew float32; info [T, E] int32 = evaders removed;
    rollout_heuristic runs heuristics/pursuit.py:18-50 (walk towards the nearest visible evader, a
    random move when none is visible).
    """

    _prefix, _Layout, _agents_attr = "pursuit", _lib.PELayout, "n_pursuers"
    _dtypes, _action_dtype, _info_keys = (torch.float32,), torch.int32, ("removed",)

    def __init__(self, n_envs, map_pool, n_evaders=1, n_pursuers=1, obs_range=3, flatten=True,
                 layer_norm=10, n_catch=2, catchr=0.01, term_pursuit=5.0, urgency_reward=0.0,
                 include_id=True, surround=True, constraint_window=1.0, sample_maps=False,
                 reward_mech='global', random_opponents=False, max_opponents=10, device=None, seed=0,
                 env_id_base=0, max_path_length=0):
        mp = np.ascontiguousarray(np.asarray(map_pool), dtype=np.int32)
        if mp.ndim == 2:
            mp = mp[None]
        self.map_pool = mp
        self.n_envs, self.n_pursuers, self.n_evaders = n_envs, n_pursuers, n_evaders
        self.obs_range, self.reward_mech, self.flatten = obs_range, reward_mech, bool(flatten)
        cfg = _lib.PEConfig(
            n_envs=n_envs, env_id_base=env_id_base, n_pursuers=n_pursuers, n_evaders=n_evaders,
            xs=mp.shape[1], ys=mp.shape[2], n_maps=mp.shape[0], obs_range=obs_range,
            flatten=int(bool(flatten)), n_catch=n_catch, surround=int(bool(surround)),
            reward_global=int(reward_mech == 'global'), include_id=int(bool(include_id)),
            sample_maps=int(bool(sample_maps)), max_path_length=int(max_path_length or 0),
            max_opponents=int(max_opponents) if random_opponents else 0,   # pursuit_evade.py:81-82,177-181
            layer_norm=float(layer_norm), catchr=float(catchr), term_pursuit=float(term_pursuit),
            urgency_reward=float(urgency_reward), constraint_window=float(constraint_window),
            seed=int(seed))
        _BatchedEngine.__init__(self, cfg, device, torch.float32, create_args=(C.c_void_p(mp.ctypes.data),))
        self.n_agents = int(self.layout.n_agents)

    @property
    def state(self):
        L, E, Np, A, RR = self.layout, self.n_envs, self.n_pursuers, self.n_agents, self.obs_range ** 2
        pos = self._view(L.pos, torch.uint8, (E, 2, A))
        return dict(pursuer_x=pos[:, 0, :Np], pursuer_y=pos[:, 1, :Np], evader_x=pos[:, 0, Np:],
                    evader_y=pos[:, 1, Np:], gone=self._view(L.gone, torch.int64, (E,)),
                    map_id=self._view(L.map_id, torch.int32, (E,)),
                    path_len=self._view(L.path_len, torch.int32, (E,)),
                    rng_counter=self._view(L.rng_counter, torch.int64, (E,)),
                    stale=self._view(L.stale, torch.int16, (E, Np, RR)))

    def set_params(self, catchr=None, constraint_window=None):
        """Curriculum updates (pursuit_evade.py:264-272)."""
        if catchr is not None:
            self.cfg.catchr = float(catchr)
        if constraint_window is not None:
            self.cfg.constraint_window = float(constraint_window)
        _lib.check(self._L.madrl_pursuit_set_params(self._h, self.cfg.catchr, self.cfg.constraint_window))

    def _policy_args(self, py2_division=True):
        """`py2_division` (rollout_heuristic keyword): the window centre `xs / 2` (heuristics/pursuit.py:23)
        as Python 2 -- the reference's language -- computes it (R // 2); False = Python 3 true division."""
        return (int(bool(py2_division)),)


class PursuitEvade(AbstractMAEnv, EzPickle):
    """Drop-in for the reference class: ``PursuitEvade(map_pool, **kwargs)``."""

    vectorized = True

    def __init__(self, map_pool, **kwargs):
        EzPickle.__init__(self, map_pool, **kwargs)
        kw = dict(kwargs)
        self.sample_maps = kw.pop('sample_maps', False)
        self.map_pool = map_pool
        self.map_matrix = np.asarray(map_pool)[0]
        self.xs, self.ys = self.map_matrix.shape
        self._reward_mech = kw.pop('reward_mech', 'global')
        self.n_evaders = kw.pop('n_evaders', 1)
        self.n_pursuers = kw.pop('n_pursuers', 1)
        self.obs_range = kw.pop('obs_range', 3)
        self.obs_offset = int((self.obs_range - 1) / 2)
        self.flatten = kw.pop('flatten', True)
        self.layer_norm = kw.pop('layer_norm', 10)
        self.n_catch = kw.pop('n_catch', 2)
        self.random_opponents = kw.pop('random_opponents', False)      # pursuit_evade.py:81-82
        self.max_opponents = kw.pop('max_opponents', 10)
        self.catchr = kw.pop('catchr', 0.01)
        self.caughtr = kw.pop('caughtr', -0.01)
        self.term_pursuit = kw.pop('term_pursuit', 5.0)
        self.term_evade = kw.pop('term_evade', -5.0)
        self.urgency_reward = kw.pop('urgency_reward', 0.0)
        self.include_id = kw.pop('include_id', True)
        if not kw.pop('train_pursuit', True):
            raise NotImplementedError("train_pursuit=False is not supported by the batched engine")
        self.surround = kw.pop('surround', True)
        self.constraint_window = kw.pop('constraint_window', 1.0)
        self.curriculum_remove_every = kw.pop('curriculum_remove_every', 500)
        self.curriculum_constrain_rate = kw.pop('curriculum_constrain_rate', 0.0)
        self.curriculum_turn_off_shaping = kw.pop('curriculum_turn_off_shaping', np.inf)
        self._engine_kwargs = dict(device=kw.pop('device', None))
        self._seed_value = kw.pop('seed', 0)
        self._env_id = kw.pop('env_id', 0)
        for k in ('ally_layer', 'opponent_layer', 'evader_controller', 'pursuer_controller', 'initial_config'):
            if kw.pop(k, None) is not None:
                raise NotImplementedError("%s cannot be injected into the batched engine" % k)
        n = 3 * self.obs_range ** 2 + (1 if self.include_id else 0)
        self.low, self.high = np.zeros(n), np.ones(n)
        self.action_space = Discrete(5)
        if self.flatten:
            self.observation_space = Box(self.low, self.high)
        else:
            self.observation_space = Box(low=-np.inf, high=np.inf, shape=(4, self.obs_range, self.obs_range))
        self.act_dims = [5 for _ in range(self.n_pursuers)]
        self.setup()

    def _ctor_params(self):
        return dict(n_evaders=self.n_evaders, n_pursuers=self.n_pursuers, obs_range=self.obs_range,
                    flatten=self.flatten, layer_norm=self.layer_norm, n_catch=self.n_catch,
                    catchr=self.catchr, term_pursuit=self.term_pursuit,
                    urgency_reward=self.urgency_reward, include_id=self.include_id,
                    surround=self.surround, constraint_window=self.constraint_window,
                    sample_maps=self.sample_maps, reward_mech=self._reward_mech,
                    random_opponents=self.random_opponents, max_opponents=self.max_opponents)

    def setup(self):
        self.pursuers = [DiscreteAgent(self.obs_range, flatten=self.flatten) for _ in range(self.n_pursuers)]
        self._engine = BatchedPursuitEvade(1, self.map_pool, seed=self._seed_value,
                                           env_id_base=self._env_id, **self._ctor_params(),
                                           **self._engine_kwargs)
        self._n_live = self.n_evaders

    @property
    def agents(self):
        return self.pursuers

    @property
    def reward_mech(self):
        return self._reward_mech

    def seed(self, seed=None):
        self._seed_value = 0 if seed is None else int(seed)
        self._engine.seed(self._seed_value)
        return [seed]

    def get_param_values(self):
        return self.__dict__

    def n_agents(self):
        return self.n_pursuers

    def reset(self):
        self._engine.set_params(self.catchr, self.constraint_window)
        obs = self._engine.reset().cpu().numpy().astype(np.float64)
        self._n_live = self.n_evaders
        if self.random_opponents:      # this episode's evader count was drawn on the device (pursuit_evade.py:179)
            gone = int(self._engine.state['gone'][0].item()) & ((1 << self.n_evaders) - 1)
            self._n_live = self.n_evaders - bin(gone).count("1")
        return [self._shape(obs[0, i]) for i in range(self.n_pursuers)]

    def _shape(self, o):
        return o if self.flatten else o.reshape(self.obs_range, self.obs_range, 4)

    @property
    def is_terminal(self):
        return self._n_live == 0

    def step(self, actions):
        if isinstance(actions, (list, np.ndarray)):
            acts = np.asarray(actions).reshape(-1)[:self.n_pursuers]
        else:  # one joint action, pursuit_evade.py:233
            acts = np.array(np.unravel_index(actions, self.act_dims))
        obs, rew, done, info = self._engine.step(acts.astype(np.int32)[None], auto_reset=False)
        obs = obs.cpu().numpy().astype(np.float64)
        rew = rew[0].cpu().numpy().astype(np.float64)
        removed = int(info['removed'][0].item())
        self._n_live -= removed
        obslist = [self._shape(obs[0, i]) for i in range(self.n_pursuers)]
        if self._reward_mech == 'global':
            return obslist, [rew[0]] * self.n_pursuers, bool(done[0].item()), {'removed': removed}
        return obslist, rew, bool(done[0].item()), {'removed': removed}

    def update_curriculum(self, itr):
        self.constraint_window += self.curriculum_constrain_rate
        self.constraint_window = np.clip(self.constraint_window, 0.0, 1.0)
        if itr != 0 and itr % self.curriculum_remove_every == 0 and self.n_pursuers > 4:
            self.n_evaders -= 1
            self.n_pursuers -= 1
            self.setup()
        if itr > self.curriculum_turn_off_shaping:
            self.catchr = 0.0

    def __getstate__(self):
        d = EzPickle.__getstate__(self)
        d['constraint_window'] = self.constraint_window
        d['n_evaders'] = self.n_evaders
        d['n_pursuers'] = self.n_pursuers
        d['catchr'] = self.catchr
        return d

    def __setstate__(self, d):
        EzPickle.__setstate__(self, d)
        self.constraint_window = d['constraint_window']
        self.n_evaders = d['n_evaders']
        self.n_pursuers = d['n_pursuers']
        self.catchr = d['catchr']
        self.setup()

    def vec_env_executor(self, n_envs, max_path_length):
        from .vec_executor import PursuitVecExecutor
        return PursuitVecExecutor(self, n_envs, max_path_length)
