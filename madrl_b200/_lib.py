"""ctypes binding of the C ABI declared in ``include/madrl_b200.h``.

The CUDA library is the product: if it cannot be loaded there is NO fallback -- importing an
engine class raises.  PyTorch is used only to own device memory and streams.
"""
import ctypes as C
import os

from . import build as _build

_lib = None


class EngineError(RuntimeError):
    pass


class WWConfig(C.Structure):
    _fields_ = [
        ("n_envs", C.c_int32), ("env_id_base", C.c_int32),
        ("n_pursuers", C.c_int32), ("n_evaders", C.c_int32), ("n_poison", C.c_int32),
        ("n_sensors", C.c_int32), ("n_coop", C.c_int32),
        ("reward_global", C.c_int32), ("addid", C.c_int32), ("speed_features", C.c_int32),
        ("random_obstacle", C.c_int32), ("timestep_limit", C.c_int32),
        ("max_path_length", C.c_int32), ("fp64", C.c_int32),
        ("radius", C.c_double), ("obstacle_radius", C.c_double), ("obstacle_x", C.c_double),
        ("obstacle_y", C.c_double), ("ev_speed", C.c_double), ("poison_speed", C.c_double),
        ("sensor_range", C.c_double), ("action_scale", C.c_double), ("poison_reward", C.c_double),
        ("food_reward", C.c_double), ("encounter_reward", C.c_double),
        ("control_penalty", C.c_double), ("seed", C.c_uint64),
    ]


class WWLayout(C.Structure):
    _fields_ = [
        ("total_bytes", C.c_size_t), ("objs", C.c_size_t), ("obst", C.c_size_t),
        ("timestep", C.c_size_t), ("path_len", C.c_size_t), ("rng_counter", C.c_size_t),
        ("sensors", C.c_size_t),
        ("n_obj", C.c_int32), ("obs_dim", C.c_int32), ("real_bytes", C.c_int32), ("_pad", C.c_int32),
    ]


class PEConfig(C.Structure):
    _fields_ = [
        ("n_envs", C.c_int32), ("env_id_base", C.c_int32), ("n_pursuers", C.c_int32),
        ("n_evaders", C.c_int32), ("xs", C.c_int32), ("ys", C.c_int32), ("n_maps", C.c_int32),
        ("obs_range", C.c_int32), ("flatten", C.c_int32), ("n_catch", C.c_int32),
        ("surround", C.c_int32), ("reward_global", C.c_int32), ("include_id", C.c_int32),
        ("sample_maps", C.c_int32), ("max_path_length", C.c_int32), ("max_opponents", C.c_int32),
        ("layer_norm", C.c_double), ("catchr", C.c_double), ("term_pursuit", C.c_double),
        ("urgency_reward", C.c_double), ("constraint_window", C.c_double), ("seed", C.c_uint64),
    ]


class PELayout(C.Structure):
    _fields_ = [
        ("total_bytes", C.c_size_t), ("pos", C.c_size_t), ("gone", C.c_size_t),
        ("map_id", C.c_size_t), ("path_len", C.c_size_t), ("rng_counter", C.c_size_t),
        ("stale", C.c_size_t), ("maps", C.c_size_t), ("lut", C.c_size_t), ("idv", C.c_size_t),
        ("n_agents", C.c_int32), ("obs_dim", C.c_int32),
    ]


class HWConfig(C.Structure):
    _fields_ = [
        ("n_envs", C.c_int32), ("env_id_base", C.c_int32), ("n_good", C.c_int32),
        ("n_hostages", C.c_int32), ("n_bad", C.c_int32), ("n_coop_save", C.c_int32),
        ("n_coop_avoid", C.c_int32), ("n_sensors", C.c_int32), ("reward_global", C.c_int32),
        ("addid", C.c_int32), ("random_key", C.c_int32), ("timestep_limit", C.c_int32),
        ("max_path_length", C.c_int32), ("fp64", C.c_int32),
        ("radius", C.c_double), ("key_x", C.c_double), ("key_y", C.c_double),
        ("bad_speed", C.c_double), ("sensor_range", C.c_double), ("action_scale", C.c_double),
        ("save_reward", C.c_double), ("hit_reward", C.c_double), ("encounter_reward", C.c_double),
        ("not_saved_reward", C.c_double), ("bomb_reward", C.c_double), ("bomb_radius", C.c_double),
        ("key_radius", C.c_double), ("control_penalty", C.c_double), ("seed", C.c_uint64),
    ]


class HWLayout(C.Structure):
    _fields_ = [
        ("total_bytes", C.c_size_t), ("objs", C.c_size_t), ("fixed", C.c_size_t),
        ("saved", C.c_size_t), ("flags", C.c_size_t), ("timestep", C.c_size_t),
        ("path_len", C.c_size_t), ("rng_counter", C.c_size_t), ("sensors", C.c_size_t),
        ("n_obj", C.c_int32), ("obs_dim", C.c_int32), ("real_bytes", C.c_int32), ("_pad", C.c_int32),
    ]


def _declare(lib):
    vp, i32, u64 = C.c_void_p, C.c_int, C.c_uint64
    lib.madrl_last_error.restype = C.c_char_p
    lib.madrl_version.restype = C.c_int
    lib.madrl_abi_sizes.argtypes = [C.POINTER(C.c_int32)]
    lib.madrl_abi_sizes.restype = None
    lib.madrl_launch_count.restype = C.c_uint64
    lib.madrl_set_host_chunk_bytes.argtypes = [C.c_size_t]
    lib.madrl_set_host_chunk_bytes.restype = None
    lib.madrl_ipc_alloc.argtypes = [C.c_size_t, C.POINTER(vp), C.c_char_p]
    lib.madrl_ipc_open.argtypes = [C.c_char_p, C.POINTER(vp)]
    lib.madrl_ipc_close.argtypes = [vp]
    lib.madrl_ipc_free.argtypes = [vp]
    lib.madrl_stream_memops_available.restype = C.c_int
    lib.madrl_copy_async.argtypes = [vp, vp, C.c_size_t, vp]
    lib.madrl_stream_write32.argtypes = [vp, vp, C.c_uint32]
    lib.madrl_stream_wait_geq32.argtypes = [vp, vp, C.c_uint32]
    lib.madrl_ww_heuristic_actions.argtypes = [i32, C.c_size_t, i32, i32, vp, vp, vp]
    lib.madrl_pursuit_heuristic_actions.argtypes = [C.c_size_t, i32, i32, i32, i32, vp, vp, vp, vp, vp]
    lib.madrl_gae_f32.argtypes = [i32, i32, i32, vp, vp, vp, vp, C.c_double, C.c_double, vp, vp, vp]
    lib.madrl_frame_stack_f32.argtypes = [i32, i32, i32, i32, i32, vp, vp, vp, vp, vp]
    lib.madrl_standardize_f32.argtypes = [i32, C.c_size_t, vp, vp, vp, C.c_double, C.c_double, i32,
                                          C.c_double, i32, vp]
    lib.madrl_episode_stats_f32.argtypes = [i32, i32, i32, vp, vp, C.c_double, i32, vp, vp, vp, vp, vp, vp]
    lib.madrl_standardize_obs_terminal_f32.argtypes = [i32, i32, C.c_size_t, vp, vp, vp, vp, vp, C.c_double, C.c_double, vp]
    lib.madrl_paths_plan.argtypes = [i32, i32, i32, vp, vp, vp, vp, vp, vp]
    lib.madrl_paths_pack_u32.argtypes = [i32, i32, i32, i32, vp, vp, vp, vp, vp, vp]
    lib.madrl_moments_f32.argtypes = [C.c_size_t, vp, vp, vp, vp, vp]
    lib.madrl_center_advantages_f32.argtypes = [C.c_size_t, vp, i32, i32, vp, vp, vp]
    for fam, cfg, lay in (("ww", WWConfig, WWLayout), ("pursuit", PEConfig, PELayout),
                          ("hostage", HWConfig, HWLayout)):
        f = lambda name: getattr(lib, "madrl_%s_%s" % (fam, name))   # noqa: E731
        f("state_layout").argtypes = [C.POINTER(cfg), C.POINTER(lay)]
        f("create").argtypes = [C.POINTER(cfg), vp, C.POINTER(vp)]
        f("destroy").argtypes = [vp]
        f("state_ptr").argtypes = [vp]
        f("state_ptr").restype = vp
        f("seed").argtypes = [vp, u64, vp]
        f("set_launch").argtypes = [vp, i32, i32]
        f("set_terminal_obs").argtypes = [vp, vp]
        f("reset").argtypes = [vp, vp, vp, vp]
        f("rollout").argtypes = [vp, i32, vp, vp, vp, vp, vp, i32, vp]
        f("step").argtypes = [vp, vp, vp, vp, vp, vp, i32, vp]
        f("reset_host").argtypes = [vp, vp, vp]
        f("rollout_host").argtypes = [vp, i32, vp, vp, vp, vp, vp, i32]
        f("rollout_host2").argtypes = [vp, i32, vp, vp, vp, vp, vp, i32, i32]
    lib.madrl_pursuit_create.argtypes = [C.POINTER(PEConfig), vp, vp, C.POINTER(vp)]   # + the map pool
    lib.madrl_pursuit_set_params.argtypes = [vp, C.c_double, C.c_double]
    lib.madrl_ww_set_peers.argtypes = [vp, i32, i32, i32, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]
    lib.madrl_ww_rollout_heuristic.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, i32, vp]
    lib.madrl_pursuit_rollout_heuristic.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, i32, i32, vp]


def lib():
    """Load (building if needed) the CUDA library.  Raises EngineError on failure."""
    global _lib
    if _lib is None:
        path = os.environ.get("MADRL_B200_LIB")            # override: kernel-variant experiments
        if path is None:
            # build() is a no-op when the library was built from exactly the sources in the tree
            # (content hash); a stale git-ignored .so left over from other sources is rebuilt, not loaded
            try:
                path = _build.build(force=bool(os.environ.get("MADRL_B200_REBUILD")))
            except Exception as e:  # no nvcc / compile error: there is no CPU fallback
                raise EngineError("madrl_b200 CUDA library is missing or stale and could not be built: %s" % e)
        try:
            lib_ = C.CDLL(path)
        except OSError as e:
            raise EngineError("cannot load %s: %s" % (path, e))
        _declare(lib_)
        sizes = (C.c_int32 * 6)()
        lib_.madrl_abi_sizes(sizes)
        want = [C.sizeof(t) for t in (WWConfig, WWLayout, PEConfig, PELayout, HWConfig, HWLayout)]
        if list(sizes) != want:
            raise EngineError("%s was built against another include/madrl_b200.h: struct sizes %s, this "
                              "binding expects %s" % (path, list(sizes), want))
        _lib = lib_
    return _lib


def require_tensor(t, name, dtype, shape, device):
    """Validate a caller-supplied tensor before its data_ptr() crosses the C ABI (a wrong dtype,
    a non-contiguous view or a short buffer would otherwise be silent garbage or an out-of-bounds
    device write).  `shape` None: any shape.  `device`: a torch.device for device buffers, 'cpu' for
    host buffers."""
    import torch
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor, got %r" % (name, type(t)))
    if t.dtype != dtype:
        raise TypeError("%s must be %s, got %s" % (name, dtype, t.dtype))
    if shape is not None and tuple(t.shape) != tuple(shape):
        raise ValueError("%s must have shape %s, got %s" % (name, tuple(shape), tuple(t.shape)))
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % name)
    if device == 'cpu':
        if t.device.type != 'cpu':
            raise ValueError("%s must be a host tensor, got %s" % (name, t.device))
    elif t.device != device:
        raise ValueError("%s must live on %s, got %s" % (name, device, t.device))
    return t


def check(rc):
    if rc != 0:
        raise EngineError("madrl_b200 error %d: %s" % (rc, lib().madrl_last_error().decode()))


def launch_count():
    return int(lib().madrl_launch_count())
