"""The batched tensor API shared by the three env families.

``_BatchedEngine`` owns one ``madrl_<prefix>_*`` handle of the C ABI (include/madrl_b200.h) and its
HBM state blob, and moves torch tensors across that ABI: every caller-supplied tensor is checked
(dtype, shape, contiguity, device) before its pointer crosses.  A family subclass builds its config,
calls ``_BatchedEngine.__init__`` and sets the class attributes below.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class _BatchedEngine(object):
    """E lockstep envs of one family resident in HBM."""

    _prefix = None                 # C prefix: madrl_<prefix>_create, ...
    _Layout = None                 # ctypes struct filled by madrl_<prefix>_state_layout
    _agents_attr = None            # attribute holding the agents per obs row ("n_pursuers", "n_good")
    _dtypes = (torch.float32, torch.float64)   # obs / reward dtypes the family's kernels are built for
    _action_dtype = None           # None: the obs dtype
    _action_tail = ()              # action shape after [T, E, agents]
    _info_tail = ()                # info shape after [T, E]
    _info_keys = ()                # step(): info dict keys, one per column of the info tail

    def __init__(self, cfg, device=None, dtype=torch.float32, create_args=()):
        if dtype not in self._dtypes:
            raise TypeError("%s supports dtype %s, got %s" % (
                type(self).__name__, " or ".join(str(d) for d in self._dtypes), dtype))
        if not torch.cuda.is_available():
            raise _lib.EngineError("madrl_b200 needs a CUDA device (there is no CPU fallback)")
        self._L = _lib.lib()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None \
            else torch.device(device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.dtype = dtype
        self.cfg = cfg
        self.layout = self._Layout()
        _lib.check(self._fn("state_layout")(C.byref(cfg), C.byref(self.layout)))
        self.obs_dim = int(self.layout.obs_dim)
        self._term_obs = None
        with torch.cuda.device(self.device):
            self._blob = torch.zeros(int(self.layout.total_bytes), dtype=torch.uint8, device=self.device)
            h = C.c_void_p()
            _lib.check(self._fn("create")(C.byref(cfg), *create_args, _ptr(self._blob), C.byref(h)))
        self._h = h

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            self._fn("destroy")(h)

    def _fn(self, name):
        return getattr(self._L, "madrl_%s_%s" % (self._prefix, name))

    @property
    def _n_rows(self):
        return getattr(self, self._agents_attr)

    # ------------------------------------------------------------------ state views
    def _view(self, off, dtype, shape):
        n = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
        return self._blob[off:off + n].view(dtype).view(*shape)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ------------------------------------------------------------------ settings
    def set_terminal_obs(self, term_obs):
        """Keep the terminal observations of done steps: `term_obs` (same shape / dtype as the obs tensor
        of the following auto-reset rollouts) receives, at the [t, e] slots where `done` is set, the
        observation the env returned BEFORE it was reset in place (StandardizedEnv needs it,
        madrl_environments/__init__.py:283-291).  None switches it off."""
        if term_obs is not None:
            _lib.require_tensor(term_obs, "term_obs", self.dtype, None, self.device)
        self._term_obs = term_obs
        _lib.check(self._fn("set_terminal_obs")(self._h, _ptr(term_obs)))

    def set_launch(self, warps_per_block=0, blocks_per_sm=0):
        _lib.check(self._fn("set_launch")(self._h, warps_per_block, blocks_per_sm))

    # ------------------------------------------------------------------ env surface (batched)
    def seed(self, seed=None):
        with torch.cuda.device(self.device):
            _lib.check(self._fn("seed")(self._h, 0 if seed is None else int(seed), self._stream()))
        return [seed]

    def reset(self, mask=None, out=None):
        """reset() of the masked envs (all if None) -> obs [E, agents, D]."""
        shape = (self.n_envs, self._n_rows, self.obs_dim)
        if out is not None:
            obs = _lib.require_tensor(out, "out", self.dtype, shape, self.device)
        else:
            obs = torch.zeros(shape, dtype=self.dtype, device=self.device)
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        with torch.cuda.device(self.device):
            _lib.check(self._fn("reset")(self._h, _ptr(mask), _ptr(obs), self._stream()))
        return obs

    def _require_outputs(self, T, out, device, obs_last=False):
        """dtype / shape / contiguity / placement of caller-supplied trajectory buffers."""
        obs, rew, done, info = out
        E, A, D = self.n_envs, self._n_rows, self.obs_dim
        _lib.require_tensor(obs, "obs", self.dtype, (E, A, D) if obs_last else (T, E, A, D), device)
        _lib.require_tensor(rew, "rew", self.dtype, (T, E, A), device)
        _lib.require_tensor(done, "done", torch.uint8, (T, E), device)
        _lib.require_tensor(info, "info", torch.int32, (T, E) + self._info_tail, device)
        return obs, rew, done, info

    def _device_outputs(self, T, out, auto_reset):
        """The trajectory tensors of a device rollout (allocated when `out` is None), after checking that
        an attached terminal-obs tensor, which the kernel writes only under auto-reset, has their shape."""
        E, A, D = self.n_envs, self._n_rows, self.obs_dim
        if out is None:
            out = (torch.empty((T, E, A, D), dtype=self.dtype, device=self.device),
                   torch.empty((T, E, A), dtype=self.dtype, device=self.device),
                   torch.empty((T, E), dtype=torch.uint8, device=self.device),
                   torch.empty((T, E) + self._info_tail, dtype=torch.int32, device=self.device))
        else:
            out = self._require_outputs(T, out, self.device)
        if auto_reset and self._term_obs is not None:
            _lib.require_tensor(self._term_obs, "term_obs", self.dtype, (T, E, A, D), self.device)
        return out

    def _actions_shape(self, T):
        return (T, self.n_envs, self._n_rows) + self._action_tail

    def rollout(self, actions, auto_reset=True, out=None):
        """T lockstep steps in one kernel launch.  actions [T, E, agents, *action tail] ->
        (obs [T,E,agents,D], rew [T,E,agents], done [T,E] uint8, info [T,E,*info tail] int32)."""
        actions = actions.to(device=self.device, dtype=self._action_dtype or self.dtype).contiguous()
        T = actions.shape[0]
        _lib.require_tensor(actions, "actions", actions.dtype, self._actions_shape(T), self.device)
        obs, rew, done, info = self._device_outputs(T, out, auto_reset)
        with torch.cuda.device(self.device):
            _lib.check(self._fn("rollout")(self._h, T, _ptr(actions), _ptr(obs), _ptr(rew), _ptr(done), _ptr(info),
                                           int(auto_reset), self._stream()))
        return obs, rew, done, info

    def step(self, actions, auto_reset=False):
        """One lockstep step.  actions [E, agents, *action tail] (or anything reshapeable to it)."""
        a = torch.as_tensor(actions, device=self.device, dtype=self._action_dtype or self.dtype).reshape(
            self._actions_shape(1))
        obs, rew, done, info = self.rollout(a, auto_reset=auto_reset)
        if not self._info_tail:
            return obs[0], rew[0], done[0], {self._info_keys[0]: info[0]}
        return obs[0], rew[0], done[0], {k: info[0, :, i] for i, k in enumerate(self._info_keys)}

    def rollout_host(self, actions, obs, rew, done, info, auto_reset=True, obs_last=False):
        """rollout() with HOST tensors (pinned for full PCIe speed); the copies are inside the call,
        chunked and overlapped with the compute (csrc/host_pipeline.cuh).  `obs_last=True`: only the last
        step's observations come back (obs is [E, A, D]) -- the policy-on-device mode."""
        T = actions.shape[0]
        _lib.require_tensor(actions, "actions", self._action_dtype or self.dtype, self._actions_shape(T), 'cpu')
        self._require_outputs(T, (obs, rew, done, info), 'cpu', obs_last)
        with torch.cuda.device(self.device):
            _lib.check(self._fn("rollout_host2")(self._h, T, _ptr(actions), _ptr(obs), _ptr(rew), _ptr(done),
                                                 _ptr(info), int(auto_reset), 1 if obs_last else 0))
        return obs, rew, done, info


class _HeuristicRollout(object):
    """rollout_heuristic() of the families whose kernel can evaluate the reference's hand-written policy."""

    def _policy_args(self):
        """Extra arguments of madrl_<prefix>_rollout_heuristic, from rollout_heuristic's keywords."""
        return ()

    def rollout_heuristic(self, T, obs0, auto_reset=True, out=None, record_actions=True, actions_out=None,
                          **policy):
        """T lockstep steps in one launch with the reference's hand-written policy (heuristics/<family>.py)
        evaluated inside the kernel: closed loop, no action tensor, no per-step launch.  obs0 [E, agents, D]
        = the observation the first action is computed from (`reset()`'s, or `obs[-1]` of the previous
        rollout).  `actions_out`: caller-owned buffer for the actions taken (no allocation in a rollout
        loop).  Returns (actions [T,E,agents,*action tail] or None, obs, rew, done, info)."""
        extra = self._policy_args(**policy)
        _lib.require_tensor(obs0, "obs0", self.dtype, (self.n_envs, self._n_rows, self.obs_dim), self.device)
        obs, rew, done, info = self._device_outputs(T, out, auto_reset)
        act_dtype = self._action_dtype or self.dtype
        if actions_out is not None:
            act = _lib.require_tensor(actions_out, "actions_out", act_dtype, self._actions_shape(T), self.device)
        else:
            act = torch.empty(self._actions_shape(T), dtype=act_dtype, device=self.device) if record_actions else None
        with torch.cuda.device(self.device):
            _lib.check(self._fn("rollout_heuristic")(self._h, T, _ptr(obs0), _ptr(act), _ptr(obs), _ptr(rew),
                                                     _ptr(done), _ptr(info), int(auto_reset), *extra,
                                                     self._stream()))
        return act, obs, rew, done, info
