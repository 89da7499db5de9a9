"""MAWaterWorld on the B200 engine.

``BatchedMAWaterWorld`` is the batched tensor API (E envs, torch CUDA tensors in and out).
``MAWaterWorld`` is the drop-in for ``madrl_environments.pursuit.waterworld.MAWaterWorld``
(same constructor, ``reset/step/seed/agents/reward_mech/timestep_limit/is_terminal/
get_param_values/set_param_values``; waterworld.py:75-436) backed by a one-env engine, and it
advertises rllab's batched plug-in hook (``vectorized`` / ``vec_env_executor``;
rllab/sandbox/rocky/tf/envs/base.py:97-103) so that ``VectorizedSampler`` gets a GPU batch.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._engine import _BatchedEngine, _HeuristicRollout
from .core import AbstractMAEnv, Agent, EzPickle
from .spaces import Box


class Archea(Agent):
    """Per-pursuer descriptor (waterworld.py:10-39): spaces only; state lives on the GPU."""

    def __init__(self, idx, radius, n_sensors, sensor_range, addid=True, speed_features=True):
        self._idx = idx
        self._radius = radius
        self._n_sensors = n_sensors
        self._sensor_range = sensor_range
        self._sensor_obscoord = 4 + (3 if speed_features else 0)
        self._obs_dim = n_sensors * self._sensor_obscoord + 2 + (1 if addid else 0)

    @property
    def observation_space(self):
        return Box(low=-10, high=10, shape=(self._obs_dim,))

    @property
    def action_space(self):
        return Box(low=-1, high=1, shape=(2,))


class BatchedMAWaterWorld(_HeuristicRollout, _BatchedEngine):
    """E lockstep MAWaterWorld instances resident in HBM.

    Parameters mirror waterworld.py:77-81 plus the batch/engine arguments:
    ``n_envs``; ``device``; ``seed`` and ``env_id_base`` (RNG key = (seed, env_id_base + e), so a
    sharded batch reproduces the unsharded one); ``max_path_length`` (VecEnvExecutor horizon);
    ``dtype`` torch.float32 (production) or torch.float64 (verification build).
    Actions [T, E, Np, 2]; info [T, E, 2] = (evcatches, pocatches); rollout_heuristic runs
    heuristics/waterworld.py:11-53.
    """

    timestep_limit = 1000
    _prefix, _Layout, _agents_attr = "ww", _lib.WWLayout, "n_pursuers"
    _action_tail, _info_tail, _info_keys = (2,), (2,), ("evcatches", "pocatches")

    def __init__(self, n_envs, n_pursuers, n_evaders, n_coop=2, n_poison=10, radius=0.015,
                 obstacle_radius=0.2, obstacle_loc=np.array([0.5, 0.5]), ev_speed=0.01,
                 poison_speed=0.01, n_sensors=30, sensor_range=0.2, action_scale=0.01,
                 poison_reward=-1., food_reward=1., encounter_reward=.05, control_penalty=-.5,
                 reward_mech='local', addid=True, speed_features=True, device=None, seed=0,
                 env_id_base=0, max_path_length=0, dtype=torch.float32):
        self.n_envs, self.n_pursuers, self.n_evaders, self.n_poison = n_envs, n_pursuers, n_evaders, n_poison
        self.n_sensors = n_sensors
        self.reward_mech = reward_mech
        rand_obst = obstacle_loc is None
        ox, oy = (0.0, 0.0) if rand_obst else (float(obstacle_loc[0]), float(obstacle_loc[1]))
        cfg = _lib.WWConfig(
            n_envs=n_envs, env_id_base=env_id_base, n_pursuers=n_pursuers, n_evaders=n_evaders,
            n_poison=n_poison, n_sensors=n_sensors, n_coop=n_coop,
            reward_global=int(reward_mech == 'global'), addid=int(bool(addid)),
            speed_features=int(bool(speed_features)), random_obstacle=int(rand_obst),
            timestep_limit=self.timestep_limit, max_path_length=int(max_path_length or 0),
            fp64=int(dtype == torch.float64), radius=radius, obstacle_radius=obstacle_radius,
            obstacle_x=ox, obstacle_y=oy, ev_speed=ev_speed, poison_speed=poison_speed,
            sensor_range=sensor_range, action_scale=action_scale, poison_reward=poison_reward,
            food_reward=food_reward, encounter_reward=encounter_reward,
            control_penalty=control_penalty, seed=int(seed))
        _BatchedEngine.__init__(self, cfg, device, dtype)
        self.n_obj = int(self.layout.n_obj)

    @property
    def state(self):
        """Named views into the HBM state blob (one record per env)."""
        L, E, N, dt = self.layout, self.n_envs, self.n_obj, self.dtype
        objs = self._view(L.objs, dt, (E, 4, N))
        obst = self._view(L.obst, dt, (E, 2))
        return dict(
            pos_x=objs[:, 0], pos_y=objs[:, 1], vel_x=objs[:, 2], vel_y=objs[:, 3],
            obst_x=obst[:, 0], obst_y=obst[:, 1],
            timestep=self._view(L.timestep, torch.int32, (E,)),
            path_len=self._view(L.path_len, torch.int32, (E,)),
            rng_counter=self._view(L.rng_counter, torch.int64, (E,)),
            sensors=self._view(L.sensors, dt, (2, self.n_sensors)))

    def set_peers(self, rank, t_max, rew_peers, done_peers, info_peers):
        """Enable the fused exchange: `*_peers` are lists (one per DESTINATION rank) of tensors
        aliasing the destination gather buffers; this rank writes slot `rank` of each
        (see madrl_b200.dist.PeerGather)."""
        n = len(rew_peers)
        arr = lambda ts: (C.c_void_p * n)(*[t.data_ptr() for t in ts])
        self._peer_keepalive = (rew_peers, done_peers, info_peers)
        _lib.check(self._L.madrl_ww_set_peers(self._h, n, rank, t_max, arr(rew_peers), arr(done_peers),
                                              arr(info_peers)))

    def clear_peers(self):
        self._peer_keepalive = None
        _lib.check(self._L.madrl_ww_set_peers(self._h, 0, 0, 0, None, None, None))


class MAWaterWorld(AbstractMAEnv, EzPickle):
    """Drop-in for the reference class (same constructor, waterworld.py:77-81)."""

    vectorized = True  # rllab batched plug-in hook (tf/envs/base.py:97-103)

    def __init__(self, n_pursuers, n_evaders, n_coop=2, n_poison=10, radius=0.015,
                 obstacle_radius=0.2, obstacle_loc=np.array([0.5, 0.5]), ev_speed=0.01,
                 poison_speed=0.01, n_sensors=30, sensor_range=0.2, action_scale=0.01,
                 poison_reward=-1., food_reward=1., encounter_reward=.05, control_penalty=-.5,
                 reward_mech='local', addid=True, speed_features=True, **kwargs):
        EzPickle.__init__(self, n_pursuers, n_evaders, n_coop, n_poison, radius, obstacle_radius,
                          obstacle_loc, ev_speed, poison_speed, n_sensors, sensor_range,
                          action_scale, poison_reward, food_reward, encounter_reward,
                          control_penalty, reward_mech, addid, speed_features, **kwargs)
        self.n_pursuers, self.n_evaders, self.n_coop, self.n_poison = n_pursuers, n_evaders, n_coop, n_poison
        self.radius, self.obstacle_radius, self.obstacle_loc = radius, obstacle_radius, obstacle_loc
        self.ev_speed, self.poison_speed = ev_speed, poison_speed
        self.n_sensors, self.sensor_range, self.action_scale = n_sensors, sensor_range, action_scale
        self.poison_reward, self.food_reward = poison_reward, food_reward
        self.encounter_reward, self.control_penalty = encounter_reward, control_penalty
        self._reward_mech, self._addid, self._speed_features = reward_mech, addid, speed_features
        self._engine_kwargs = dict(device=kwargs.pop('device', None), dtype=kwargs.pop('dtype', torch.float32))
        self._seed_value = kwargs.pop('seed', 0)
        self._env_id = kwargs.pop('env_id', 0)
        self._pursuers = [Archea(i + 1, radius, n_sensors, sensor_range, addid, speed_features)
                          for i in range(n_pursuers)]
        self._timesteps = 0
        self.setup()

    def _ctor_params(self):
        return dict(n_pursuers=self.n_pursuers, n_evaders=self.n_evaders, n_coop=self.n_coop,
                    n_poison=self.n_poison, radius=self.radius, obstacle_radius=self.obstacle_radius,
                    obstacle_loc=self.obstacle_loc, ev_speed=self.ev_speed,
                    poison_speed=self.poison_speed, n_sensors=self.n_sensors,
                    sensor_range=self.sensor_range, action_scale=self.action_scale,
                    poison_reward=self.poison_reward, food_reward=self.food_reward,
                    encounter_reward=self.encounter_reward, control_penalty=self.control_penalty,
                    reward_mech=self._reward_mech, addid=self._addid,
                    speed_features=self._speed_features)

    def setup(self):
        """(Re)build the engine from the current attributes (set_param_values contract)."""
        self._engine = BatchedMAWaterWorld(1, seed=self._seed_value, env_id_base=self._env_id,
                                           **self._ctor_params(), **self._engine_kwargs)

    @property
    def reward_mech(self):
        return self._reward_mech

    @property
    def timestep_limit(self):
        return 1000

    @property
    def agents(self):
        return self._pursuers

    def get_param_values(self):
        return self.__dict__

    def seed(self, seed=None):
        self._seed_value = 0 if seed is None else int(seed)
        self._engine.seed(self._seed_value)
        return [seed]

    def reset(self):
        obs = self._engine.reset().cpu().numpy().astype(np.float64)
        self._timesteps = 1  # reset consumes one internal step (waterworld.py:172)
        return [obs[0, i] for i in range(self.n_pursuers)]

    @property
    def is_terminal(self):
        return self._timesteps >= self.timestep_limit

    def step(self, action_Np2):
        a = np.asarray(action_Np2, dtype=np.float64).reshape((self.n_pursuers, 2))  # waterworld.py:221-222
        obs, rew, done, info = self._engine.step(a[None], auto_reset=False)
        obs = obs.cpu().numpy().astype(np.float64)
        self._timesteps += 1
        return ([obs[0, i] for i in range(self.n_pursuers)], rew[0].cpu().numpy().astype(np.float64),
                bool(done[0].item()),
                dict(evcatches=int(info['evcatches'][0].item()), pocatches=int(info['pocatches'][0].item())))

    def vec_env_executor(self, n_envs, max_path_length):
        from .vec_executor import WaterworldVecExecutor
        return WaterworldVecExecutor(self, n_envs, max_path_length)
