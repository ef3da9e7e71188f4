"""ctypes binding of libcgl_b200.so (the C ABI declared in include/cgl_b200.h).

PyTorch is used by the callers for device memory and streams only; no torch type crosses this
boundary -- every call passes raw device pointers, sizes and a cudaStream_t.

There is NO CPU fallback: if the CUDA library cannot be loaded (or built), importing the
product fails loudly with `CglNativeError`.
"""
from __future__ import annotations

import ctypes
import os

_PKG_DIR = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.environ.get("CGL_B200_LIB") or os.path.join(_PKG_DIR, "libcgl_b200.so")      # (override: tuning builds)

E_BADARG, E_BADINDEX, E_NOMEM = -1, -2, -3
ABI_VERSION = 2                         # CGL_B200_ABI_VERSION


class CglNativeError(RuntimeError):
    """Raised when libcgl_b200.so is missing or one of its entry points reports an error."""


_vp, _u64, _u32, _i = ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int

# name -> (restype, argtypes); mirrors include/cgl_b200.h one to one
SIGNATURES = {
    "cgl_abi_version": (_i, []),
    "cgl_last_error": (ctypes.c_char_p, []),
    "cgl_alarm_words": (_i, [ctypes.POINTER(ctypes.POINTER(ctypes.c_int))]),
    "cgl_set_wait_timeout_ms": (_i, [_u32]),
    "cgl_test_fault": (_i, [_i]),
    "cgl_device_count": (_i, [ctypes.POINTER(_i)]),
    "cgl_device_info": (_i, [_i, ctypes.c_char_p, _i, ctypes.POINTER(_i), ctypes.POINTER(_i),
                             ctypes.POINTER(_i), ctypes.POINTER(_u64)]),
    "cgl_words_per_row": (_u32, [_u32]),
    "cgl_pack": (_i, [_vp, _vp, _u64, _u32, _u32, _vp]),
    "cgl_unpack": (_i, [_vp, _vp, _u64, _u32, _u32, _vp]),
    "cgl_init_stable": (_i, [_vp, _vp, _u64, _u32, _i, _vp]),
    "cgl_toggle": (_i, [_vp, _vp, _u64, _u32, _vp, _u32, _i, _vp, _vp]),
    "cgl_env_step": (_i, [_vp, _vp, _vp, _u64, _u32, _vp, _i, _i, _vp, _vp, _vp, _vp]),
    "cgl_env_step_chained": (_i, [_vp, _vp, _vp, _u64, _u32, _vp, _i, _i, _vp, _vp, _vp, _vp, _u32, _u32, _vp]),
    "cgl_env_run": (_i, [_vp, _vp, _vp, _u64, _u32, _u32, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "cgl_env_run_rule": (_i, [_vp, _vp, _vp, _u64, _u32, _u32, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "cgl_breakdown_stable": (_i, [_vp, _u64, _u64, _vp, _vp]),
    "cgl_env_step_rule": (_i, [_vp, _vp, _vp, _vp, _u64, _u32, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _u32, _u32, _vp]),
    "cgl_toggle_rule": (_i, [_vp, _vp, _u64, _u32, _vp, _u32, _i, _i, _vp, _vp]),
    "cgl_init_stable_rule": (_i, [_vp, _vp, _u64, _u32, _i, _i, _vp]),
    "cgl_env_step_io": (_i, [_vp, _vp, _vp, _vp, _u64, _u32, _vp, _i, _i, _vp, _vp, _vp, _vp, _u32, _u32, _vp]),
    "cgl_sim_step": (_i, [_vp, _vp, _vp, _u32, ctypes.c_int32, _i, _i, _i, _i, _i, _i, _vp, _vp, _u32, _vp]),
    "cgl_sim_step_max_side": (_u32, []),
    "cgl_env_step_is_fused": (_i, [_u32]),
    "cgl_env_step_launches": (_i, [_u32, _i]),
    "cgl_life_step": (_i, [_vp, _vp, _u64, _u32, _u32, _i, _vp, _vp]),
    "cgl_life_run": (_i, [_vp, _vp, _u32, _u32, _i, _u32, _u32, ctypes.POINTER(_i), _vp]),
    "cgl_life_run_pop": (_i, [_vp, _vp, _u32, _u32, _i, _u32, _u32, _u32, _u32, _vp, ctypes.POINTER(_i), _vp]),
    "cgl_life_tune": (_i, [_vp, _vp, _u32, _u32, _i, _u32, _vp]),
    "cgl_reward": (_i, [_vp, _u64, _u64, _vp, _vp]),
    "cgl_alive": (_i, [_vp, _u64, _u64, _vp, _vp]),
    "cgl_match": (_i, [_vp, _vp, _u64, _vp, _vp]),
    "cgl_step_state_gpu": (_i, [_vp, _vp, _u32, _i, _i]),
    "cgl_env_step_host": (_i, [_vp, _vp, _vp, _u64, _u32, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp]),
    "cgl_env_step_host_async": (_i, [_vp, _vp, _vp, _u64, _u32, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp]),
    "cgl_stream_wait": (_i, [_vp]),
    "cgl_ipc_get_handle": (_i, [_vp, _vp]),
    "cgl_ipc_open_handle": (_i, [_vp, ctypes.POINTER(_vp)]),
    "cgl_ipc_close_handle": (_i, [_vp]),
    "cgl_halo_exchange": (_i, [_vp] * 12 + [_u64, _u32, _vp]),
    "cgl_dev_alloc": (_i, [_u64, ctypes.POINTER(_vp)]),
    "cgl_dev_free": (_i, [_vp]),
    "cgl_dev_memset": (_i, [_vp, _i, _u64, _vp]),
    "cgl_state_granularity": (ctypes.c_size_t, [_i]),
    "cgl_state_alloc": (_vp, [ctypes.c_size_t, _i, _vp]),
    "cgl_state_free": (None, [_vp, ctypes.c_size_t, _i, _vp]),
    "cgl_state_compressed": (_i, [_vp]),
}

class EnvStepArgs(ctypes.Structure):
    """cgl_env_step_args_t (include/cgl_b200.h)."""
    _fields_ = [("world_in", _vp), ("world_out", _vp), ("stable_in", _vp), ("stable_out", _vp), ("n_envs", _u64),
                ("side", _u32), ("spawn", ctypes.c_int32), ("stable_max", ctypes.c_int32), ("dead_rule", ctypes.c_int32),
                ("empty", ctypes.c_int32), ("empty_min", ctypes.c_int32), ("masked_toggle", ctypes.c_int32),
                ("actions", _vp), ("reward_out", _vp), ("alive_out", _vp), ("err_flag", _vp), ("token", _vp),
                ("want", _u32), ("publish", _u32), ("chain_mode", _u32), ("seq_counter", ctypes.POINTER(_u32))]


CHAIN_NONE, CHAIN_IDS, CHAIN_SEQ = 0, 1, 2

class EnvRunArgs(ctypes.Structure):
    """cgl_env_run_args_t (include/cgl_b200.h)."""
    _fields_ = [("world_in", _vp), ("world_out", _vp), ("stable", _vp), ("n_envs", _u64), ("side", _u32),
                ("max_steps", _u32), ("stop_when_fixed", ctypes.c_int32), ("spawn", ctypes.c_int32),
                ("stable_max", ctypes.c_int32), ("dead_rule", ctypes.c_int32), ("empty", ctypes.c_int32),
                ("empty_min", ctypes.c_int32), ("masked_toggle", ctypes.c_int32), ("actions", _vp),
                ("reward_trace", _vp), ("alive_trace", _vp), ("steps_out", _vp), ("reward_out", _vp),
                ("alive_out", _vp), ("err_flag", _vp)]


class EnvRunObsArgs(ctypes.Structure):
    """cgl_env_run_obs_args_t (include/cgl_b200.h)."""
    _fields_ = [("run", EnvRunArgs), ("obs_trace", _vp)]


SIGNATURES["cgl_env_run_ex"] = (_i, [ctypes.POINTER(EnvRunArgs), _vp])
SIGNATURES["cgl_env_run_obs"] = (_i, [ctypes.POINTER(EnvRunObsArgs), _vp])
SIGNATURES["cgl_env_run_cycle"] = (_i, [ctypes.POINTER(EnvRunArgs), _u32, _vp, _vp])
RUN_MAX_PERIOD = 8                      # CGL_RUN_MAX_PERIOD
SIGNATURES["cgl_env_run_settle"] = (_i, [ctypes.POINTER(EnvRunArgs), _vp, _vp])


class EnvActionRewardsArgs(ctypes.Structure):
    """cgl_env_action_rewards_args_t (include/cgl_b200.h)."""
    _fields_ = [("world", _vp), ("stable", _vp), ("n_envs", _u64), ("side", _u32), ("spawn", ctypes.c_int32),
                ("stable_max", ctypes.c_int32), ("dead_rule", ctypes.c_int32), ("empty", ctypes.c_int32),
                ("empty_min", ctypes.c_int32), ("masked_toggle", ctypes.c_int32), ("rewards_out", _vp),
                ("best_action_out", _vp), ("best_reward_out", _vp)]


SIGNATURES["cgl_env_action_rewards"] = (_i, [ctypes.POINTER(EnvActionRewardsArgs), _vp])
SIGNATURES["cgl_env_step_ex"] = (_i, [ctypes.POINTER(EnvStepArgs), _vp])
SIGNATURES["cgl_env_step_seq"] = (_i, [ctypes.POINTER(EnvStepArgs), _u32, _u64, _u64, _vp])
SIGNATURES["cgl_env_step_seq_timed"] = (_i, [ctypes.POINTER(EnvStepArgs), _u32, _u64, _u64, _vp, _vp, _vp])

class SimStepArgs(ctypes.Structure):
    """cgl_sim_step_args_t (include/cgl_b200.h)."""
    _fields_ = [("world_a", _vp), ("world_b", _vp), ("stable", _vp), ("side", _u32), ("spawn", ctypes.c_int32),
                ("stable_max", ctypes.c_int32), ("dead_rule", ctypes.c_int32), ("empty", ctypes.c_int32),
                ("empty_min", ctypes.c_int32), ("masked_toggle", ctypes.c_int32), ("obs_mirror", _vp), ("result", _vp),
                ("flip_planes", ctypes.POINTER(_u32))]


SIGNATURES["cgl_sim_step_ex"] = (_i, [ctypes.POINTER(SimStepArgs), ctypes.c_int32, _u32, _vp])
SIGNATURES["cgl_sim_serve"] = (_i, [ctypes.POINTER(SimStepArgs), _vp, _u32, _u32, _u32, _vp])
SIGNATURES["cgl_sim_serve_max_side"] = (_u32, [])
SIM_QUIT = 0xFFFFFFFE

POLICY_FN = ctypes.CFUNCTYPE(None, _vp, _u32, _u64, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32))
SIGNATURES["cgl_rollout_create"] = (_i, [ctypes.POINTER(_vp), _u32, _u32, ctypes.POINTER(_vp), ctypes.POINTER(_vp),
                                         ctypes.POINTER(_vp), _u64, _u32, _i, _i, ctypes.POINTER(_vp), _u32])
SIGNATURES["cgl_rollout_buffers"] = (_i, [_vp, _u32, ctypes.POINTER(ctypes.POINTER(ctypes.c_int32)),
                                          ctypes.POINTER(ctypes.POINTER(ctypes.c_int32))])
SIGNATURES["cgl_rollout_run"] = (_i, [_vp, _u64, _vp, _vp])
SIGNATURES["cgl_rollout_parity"] = (_i, [_vp, _u32, _u32])
SIGNATURES["cgl_rollout_destroy"] = (_i, [_vp])

_lib = None


def load(build_if_missing: bool = True) -> ctypes.CDLL:
    """Load (building first if the .so is absent and nvcc is available) and type the library."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH) and build_if_missing:
        try:
            import importlib.util
            spec = importlib.util.spec_from_file_location("_cgl_b200_build", os.path.join(_PKG_DIR, "build.py"))
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
            mod.build()
        except Exception as exc:  # noqa: BLE001
            raise CglNativeError(f"libcgl_b200.so is missing and could not be built: {exc}") from exc
    if not os.path.exists(LIB_PATH):
        raise CglNativeError(f"{LIB_PATH} not found: build it with `python {_PKG_DIR}/build.py` "
                             "(there is no CPU fallback)")
    try:
        lib = ctypes.CDLL(LIB_PATH)
    except OSError as exc:
        raise CglNativeError(f"cannot load {LIB_PATH}: {exc}") from exc
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here == header/library mismatch
        fn.restype, fn.argtypes = res, args
    if lib.cgl_abi_version() != ABI_VERSION:
        raise CglNativeError("libcgl_b200.so ABI version mismatch")
    _lib = lib
    return lib


_ext = None


def ext():
    """The thin PyTorch C++ extension (csrc_ext/cgl_torch_ext.cpp -> cgl_b200/_cgl_ext.so): torch-typed entry points
    over the same C ABI.  Built by build.py (build_ext); a missing extension raises -- nothing falls back."""
    global _ext
    if _ext is None:
        load()                                  # libcgl_b200.so first: the extension links against it
        try:
            from . import _cgl_ext as mod
        except ImportError as exc:
            raise CglNativeError(f"cgl_b200/_cgl_ext.so is missing or does not load ({exc}): build it with "
                                 f"`python {_PKG_DIR}/build.py --ext`") from exc
        if mod.abi_version() != ABI_VERSION:
            raise CglNativeError("_cgl_ext.so was built against another ABI version")
        _ext = mod
    return _ext


_state_allocator = None
_state_pools = {}


def state_pool(device_index: int):
    """The torch.cuda.MemPool of `device_index` over cgl_state_alloc / cgl_state_free (hardware-compressed device
    memory, see include/cgl_b200.h), or None if the device offers no compression.  One pool per device, kept for the
    life of the process."""
    global _state_allocator
    if device_index in _state_pools:
        return _state_pools[device_index]
    import torch
    pool = None
    if load().cgl_state_granularity(device_index):
        if _state_allocator is None:
            _state_allocator = torch.cuda.memory.CUDAPluggableAllocator(LIB_PATH, "cgl_state_alloc", "cgl_state_free")
        with torch.cuda.device(device_index):
            pool = torch.cuda.MemPool(_state_allocator.allocator())
    _state_pools[device_index] = pool
    return pool


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().cgl_last_error().decode("utf-8", "replace")
        raise CglNativeError(f"{what or 'libcgl_b200'} failed (rc={rc}): {msg}")


ALARM_NAMES = ("an action / toggle index outside [0, size] was ignored",
               "chained env step: a plane token never arrived (state planes out of sync)",
               "life mode: a strip token of the previous launch never arrived",
               "halo exchange: a ring neighbour never delivered its rows")
_alarm = None


def alarm():
    """The library's alarm words as a live numpy view (int32[4], host-mapped pinned memory; see cgl_alarm_words in
    include/cgl_b200.h).  Also installs them on the current CUDA device.  Reading costs no synchronisation."""
    global _alarm
    import numpy as np
    p = ctypes.POINTER(ctypes.c_int)()
    check(load().cgl_alarm_words(ctypes.byref(p)), "cgl_alarm_words")
    if _alarm is None:
        _alarm = np.ctypeslib.as_array(p, shape=(4,))
    return _alarm


def check_alarm(clear: bool = True) -> None:
    """Raise if a kernel gave up on a device-side wait (words 1..3).  Word 0 (invalid action) is left to
    BatchedSim.check_actions, which turns it into the reference's ValueError."""
    a = _alarm if _alarm is not None else alarm()
    if a[1] or a[2] or a[3]:
        msgs = [ALARM_NAMES[i] for i in (1, 2, 3) if a[i]]
        if clear:
            a[1:] = 0
        raise CglNativeError("; ".join(msgs))


def dptr(t) -> ctypes.c_void_p:
    """Raw device (or host) pointer of a torch tensor / None."""
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def current_stream() -> ctypes.c_void_p:
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
