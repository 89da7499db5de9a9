"""ContinuousHostageWorld on the B200 engine.

``BatchedHostageWorld`` is the batched tensor API; ``ContinuousHostageWorld`` is the drop-in for
``madrl_environments.hostage.ContinuousHostageWorld`` (same constructor, hostage.py:75-79).
"""
import numpy as np
import torch

from . import _lib
from ._engine import _BatchedEngine
from .core import AbstractMAEnv, Agent, EzPickle
from .spaces import Box


class CircAgent(Agent):
    """Per-rescuer descriptor (hostage.py:10-37): spaces only."""

    def __init__(self, idx, radius, n_sensors, sensor_range, addid=True):
        self._idx, self._radius, self._n_sensors, self._sensor_range = idx, radius, n_sensors, sensor_range
        self._obs_dim = n_sensors * 5 + 5 + (1 if addid else 0)

    @property
    def observation_space(self):
        return Box(low=-np.inf, high=np.inf, shape=(self._obs_dim,))

    @property
    def action_space(self):
        return Box(low=-10, high=10, shape=(2,))


class BatchedHostageWorld(_BatchedEngine):
    """E lockstep ContinuousHostageWorld instances resident in HBM (arguments: hostage.py:75-79).
    Actions [T, E, n_good, 2]; info [T, E, 2] = (ho_saved, cr_encs)."""

    timestep_limit = 1000
    _prefix, _Layout, _agents_attr = "hostage", _lib.HWLayout, "n_good"
    _action_tail, _info_tail, _info_keys = (2,), (2,), ("ho_saved", "cr_encs")

    def __init__(self, n_envs, n_good, n_hostages, n_bad, n_coop_save, n_coop_avoid, radius=0.015,
                 key_loc=None, bad_speed=0.01, n_sensors=30, sensor_range=0.2, action_scale=0.01,
                 save_reward=5., hit_reward=-1., encounter_reward=0.01, not_saved_reward=-3,
                 bomb_reward=-5., bomb_radius=0.05, key_radius=0.0075, control_penalty=-.1,
                 reward_mech='global', addid=True, device=None, seed=0, env_id_base=0,
                 max_path_length=0, dtype=torch.float32):
        self.n_envs, self.n_good, self.n_hostages, self.n_bad = n_envs, n_good, n_hostages, n_bad
        self.n_sensors, self.reward_mech = n_sensors, reward_mech
        rand_key = key_loc is None
        kx, ky = (0.0, 0.0) if rand_key else [float(v) for v in np.asarray(key_loc).reshape(-1)[:2]]
        cfg = _lib.HWConfig(
            n_envs=n_envs, env_id_base=env_id_base, n_good=n_good, n_hostages=n_hostages, n_bad=n_bad,
            n_coop_save=n_coop_save, n_coop_avoid=n_coop_avoid, n_sensors=n_sensors,
            reward_global=int(reward_mech == 'global'), addid=int(bool(addid)),
            random_key=int(rand_key), timestep_limit=self.timestep_limit,
            max_path_length=int(max_path_length or 0), fp64=int(dtype == torch.float64),
            radius=radius, key_x=kx, key_y=ky, bad_speed=bad_speed, sensor_range=float(sensor_range),
            action_scale=action_scale, save_reward=save_reward, hit_reward=hit_reward,
            encounter_reward=encounter_reward, not_saved_reward=float(not_saved_reward),
            bomb_reward=bomb_reward, bomb_radius=bomb_radius, key_radius=key_radius,
            control_penalty=control_penalty, seed=int(seed))
        _BatchedEngine.__init__(self, cfg, device, dtype)
        self.n_obj = int(self.layout.n_obj)

    @property
    def state(self):
        L, E, N, dt = self.layout, self.n_envs, self.n_obj, self.dtype
        objs = self._view(L.objs, dt, (E, 4, N))
        fixed = self._view(L.fixed, dt, (E, 4))
        return dict(pos_x=objs[:, 0], pos_y=objs[:, 1], vel_x=objs[:, 2], vel_y=objs[:, 3],
                    key=fixed[:, 0:2], bomb=fixed[:, 2:4],
                    saved=self._view(L.saved, torch.uint8, (E, self.n_hostages)),
                    flags=self._view(L.flags, torch.int32, (E,)),
                    timestep=self._view(L.timestep, torch.int32, (E,)),
                    path_len=self._view(L.path_len, torch.int32, (E,)),
                    rng_counter=self._view(L.rng_counter, torch.int64, (E,)))


class ContinuousHostageWorld(AbstractMAEnv, EzPickle):
    """Drop-in for the reference class (same constructor, hostage.py:75-79)."""

    vectorized = True

    def __init__(self, n_good, n_hostages, n_bad, n_coop_save, n_coop_avoid, radius=0.015,
                 key_loc=None, bad_speed=0.01, n_sensors=30, sensor_range=0.2, action_scale=0.01,
                 save_reward=5., hit_reward=-1., encounter_reward=0.01, not_saved_reward=-3,
                 bomb_reward=-5., bomb_radius=0.05, key_radius=0.0075, control_penalty=-.1,
                 reward_mech='global', addid=True, **kwargs):
        EzPickle.__init__(self, n_good, n_hostages, n_bad, n_coop_save, n_coop_avoid, radius,
                          key_loc, bad_speed, n_sensors, sensor_range, action_scale, save_reward,
                          hit_reward, encounter_reward, not_saved_reward, bomb_reward, bomb_radius,
                          key_radius, control_penalty, reward_mech, addid, **kwargs)
        self.n_good, self.n_hostages, self.n_bad = n_good, n_hostages, n_bad
        self.n_coop_save, self.n_coop_avoid = n_coop_save, n_coop_avoid
        self.radius, self.key_loc, self.key_radius, self.bad_speed = radius, key_loc, key_radius, bad_speed
        self.n_sensors, self.sensor_range, self.action_scale = n_sensors, sensor_range, action_scale
        self.save_reward, self.hit_reward, self.encounter_reward = save_reward, hit_reward, encounter_reward
        self.not_saved_reward, self.bomb_reward, self.bomb_radius = not_saved_reward, bomb_reward, bomb_radius
        self.control_penalty, self._reward_mech, self._addid = control_penalty, reward_mech, addid
        self._engine_kwargs = dict(device=kwargs.pop('device', None), dtype=kwargs.pop('dtype', torch.float32))
        self._seed_value = kwargs.pop('seed', 0)
        self._env_id = kwargs.pop('env_id', 0)
        self._rescuers = [CircAgent(i + 1, radius, n_sensors, sensor_range, addid) for i in range(n_good)]
        self._done = False
        self.setup()

    def _ctor_params(self):
        return dict(n_good=self.n_good, n_hostages=self.n_hostages, n_bad=self.n_bad,
                    n_coop_save=self.n_coop_save, n_coop_avoid=self.n_coop_avoid, radius=self.radius,
                    key_loc=self.key_loc, bad_speed=self.bad_speed, n_sensors=self.n_sensors,
                    sensor_range=self.sensor_range, action_scale=self.action_scale,
                    save_reward=self.save_reward, hit_reward=self.hit_reward,
                    encounter_reward=self.encounter_reward, not_saved_reward=self.not_saved_reward,
                    bomb_reward=self.bomb_reward, bomb_radius=self.bomb_radius,
                    key_radius=self.key_radius, control_penalty=self.control_penalty,
                    reward_mech=self._reward_mech, addid=self._addid)

    def setup(self):
        self._engine = BatchedHostageWorld(1, seed=self._seed_value, env_id_base=self._env_id,
                                           **self._ctor_params(), **self._engine_kwargs)

    @property
    def reward_mech(self):
        return self._reward_mech

    @property
    def timestep_limit(self):
        return 1000

    @property
    def agents(self):
        return self._rescuers

    @property
    def is_gate_open(self):
        return bool(int(self._engine.state['flags'][0].item()) & 1)

    def get_param_values(self):
        return self.__dict__

    def seed(self, seed=None):
        self._seed_value = 0 if seed is None else int(seed)
        self._engine.seed(self._seed_value)
        return [seed]

    def reset(self):
        obs = self._engine.reset().cpu().numpy().astype(np.float64)
        self._done = False
        return [obs[0, i] for i in range(self.n_good)]

    @property
    def is_terminal(self):
        return self._done

    def step(self, action_Nr2):
        a = np.asarray(action_Nr2, dtype=np.float64).reshape((self.n_good, 2))   # hostage.py:229-230
        obs, rew, done, info = self._engine.step(a[None], auto_reset=False)
        obs = obs.cpu().numpy().astype(np.float64)
        self._done = bool(done[0].item())
        return ([obs[0, i] for i in range(self.n_good)], rew[0].cpu().numpy().astype(np.float64), self._done,
                dict(ho_saved=int(info['ho_saved'][0].item()), cr_encs=int(info['cr_encs'][0].item())))

    def vec_env_executor(self, n_envs, max_path_length):
        from .vec_executor import HostageVecExecutor
        return HostageVecExecutor(self, n_envs, max_path_length)
