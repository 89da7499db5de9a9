"""API-level behaviour of the engines through the C ABI (needs a GPU): host-buffer entry points,
masked reset, seed(), error codes."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from conftest import ROOT

pytestmark = pytest.mark.gpu


def engines():
    from madrl_b200 import BatchedHostageWorld, BatchedMAWaterWorld, BatchedPursuitEvade
    maps = np.load(os.path.join(ROOT, "maps", "map_pool16.npy"))
    ww = lambda **k: BatchedMAWaterWorld(64, 5, 5, seed=3, **k)
    pe = lambda **k: BatchedPursuitEvade(64, maps, n_evaders=30, n_pursuers=8, obs_range=7, catchr=0.1,
                                         sample_maps=True, reward_mech='local', seed=3, **k)
    hw = lambda **k: BatchedHostageWorld(64, 10, 16, 16, 4, 2, seed=3, **k)
    return dict(ww=ww, pe=pe, hw=hw)


def actions_for(name, T, eng, gen):
    if name == "pe":
        return torch.randint(0, 5, (T, eng.n_envs, eng.n_pursuers), dtype=torch.int32, generator=gen)
    n = eng.n_pursuers if name == "ww" else eng.n_good
    return torch.randn(T, eng.n_envs, n, 2, generator=gen) * 0.5


@pytest.mark.parametrize("name", ["ww", "pe", "hw"])
def test_host_rollout_equals_device_rollout(name):
    mk = engines()[name]
    gen = torch.Generator().manual_seed(0)
    a, b = mk(), mk()
    oa, ob = a.reset(), b.reset()
    assert torch.equal(oa, ob)
    T = 9
    act = actions_for(name, T, a, gen)
    dev_out = [x.cpu() for x in a.rollout(act.cuda(), auto_reset=True)]
    host_out = (torch.empty_like(dev_out[0]).pin_memory(), torch.empty_like(dev_out[1]).pin_memory(),
                torch.empty_like(dev_out[2]).pin_memory(), torch.empty_like(dev_out[3]).pin_memory())
    b.rollout_host(act.contiguous().pin_memory(), *host_out, auto_reset=True)
    for x, y in zip(dev_out, host_out):
        assert torch.equal(x, y)


@pytest.mark.parametrize("name", ["ww", "pe", "hw"])
def test_masked_reset_and_seed(name):
    mk = engines()[name]
    eng = mk()
    obs0 = eng.reset().clone()
    pos0 = {k: v.clone() for k, v in eng.state.items() if k.endswith(('_x', '_y'))}
    gen = torch.Generator().manual_seed(1)
    eng.rollout(actions_for(name, 5, eng, gen).cuda(), auto_reset=False)
    state_before = {k: v.clone() for k, v in eng.state.items()}
    mask = torch.zeros(eng.n_envs, dtype=torch.uint8)
    mask[::4] = 1
    out = torch.full_like(obs0, -7.0)
    eng.reset(mask=mask, out=out)
    keep = ~mask.bool().cuda()
    assert (out[keep] == -7.0).all() and (out[mask.bool().cuda()] != -7.0).any()
    for k, v in eng.state.items():          # unmasked envs untouched
        if v.shape[0] == eng.n_envs:
            assert torch.equal(v[keep], state_before[k][keep]), k
    # seed(s) re-keys and restarts every stream: same seed => same reset observations again
    eng.seed(3)
    again = eng.reset()
    if name == "ww":
        assert torch.equal(again, obs0)
    elif name == "pe":                      # same spawns; obs may differ in the never-cleared
        for k, v in pos0.items():           # out-of-bounds window cells (pursuit_evade.py:119,438)
            assert torch.equal(eng.state[k], v), k
    # (hostage keeps its key location across resets, hostage.py:148, so its stream shifts by two draws)
    eng.seed(4)
    assert not torch.equal(eng.reset(), again)


def test_error_codes_and_messages():
    from madrl_b200 import BatchedHostageWorld, BatchedMAWaterWorld, EngineError, _lib
    with pytest.raises(EngineError, match="n_pursuers"):
        BatchedMAWaterWorld(4, 40, 5)
    with pytest.raises(EngineError, match="n_sensors"):
        BatchedMAWaterWorld(4, 5, 5, n_sensors=100)
    with pytest.raises(TypeError, match="dtype"):       # no fp16 kernel: would write 4-byte values into 2-byte rows
        BatchedHostageWorld(4, 2, 2, 2, 1, 1, dtype=torch.float16)
    eng = BatchedMAWaterWorld(4, 5, 5)
    lib = _lib.lib()
    assert lib.madrl_ww_rollout(eng._h, 0, None, None, None, None, None, 0, None) == -1
    assert b"T must be" in lib.madrl_last_error()
    assert lib.madrl_ww_reset(None, None, None, None) == -1
    with pytest.raises(EngineError):
        eng.set_launch(warps_per_block=9)
    # the terminal-obs side tensor is written at the [t, e] slots of every later auto-reset rollout
    T, shape = 6, (6, 4, 5, eng.obs_dim)
    with pytest.raises(TypeError, match="term_obs"):
        eng.set_terminal_obs(torch.zeros(shape, dtype=torch.float64, device=eng.device))
    eng.set_terminal_obs(torch.zeros((T - 1,) + shape[1:], dtype=torch.float32, device=eng.device))
    eng.reset()
    n = _lib.launch_count()
    with pytest.raises(ValueError, match="term_obs"):
        eng.rollout(torch.zeros(T, 4, 5, 2, device=eng.device), auto_reset=True)
    assert _lib.launch_count() == n                      # refused before the launch
