"""ctypes loader of the CUDA extension (predpreygrass_b200/libppg_b200.so).

There is no CPU fallback: if the library is missing or does not export the C-ABI of include/ppg.h
the import of anything that computes fails loudly.
"""
import ctypes as C
import os

from .config import PpgBuffers, PpgConfig, PpgReturns, PpgTape

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PPG_LIB") or os.path.join(HERE, "libppg_b200.so")  # PPG_LIB: an experimental build of the same ABI

# every symbol include/ppg.h declares
SYMBOLS = [
    "ppg_abi_version", "ppg_default_config", "ppg_create", "ppg_destroy", "ppg_load_tape", "ppg_reset", "ppg_step",
    "ppg_step_ordered", "ppg_step_host", "ppg_random_actions", "ppg_get_buffers", "ppg_snapshot_size", "ppg_snapshot", "ppg_restore",
    "ppg_read_env", "ppg_read_env_eco", "ppg_read_env_stag", "ppg_stats", "ppg_stats_device", "ppg_stats_clear", "ppg_launch_count", "ppg_last_error",
    "ppg_profile_begin", "ppg_profile_end", "ppg_profile_env_cycles", "ppg_rollout_random", "ppg_selftest_pow", "ppg_read_episode_eco", "ppg_read_episode_events_eco", "ppg_read_env_acc", "ppg_set_pdl_chain",
    "ppg_world_state", "ppg_track_returns", "ppg_get_returns", "ppg_episode_stats_device", "ppg_episode_stats_clear",
]

_lib = None


class PpgError(RuntimeError):
    pass


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PpgError(
            f"{LIB_PATH} is missing: build it with `python -m predpreygrass_b200.build` "
            "(there is no CPU fallback for the environment step)"
        )
    L = C.CDLL(LIB_PATH)
    missing = [s for s in SYMBOLS if not hasattr(L, s)]
    if missing:
        raise PpgError(f"{LIB_PATH} does not export {missing}")
    vp, i32, u64 = C.c_void_p, C.c_int32, C.c_uint64
    L.ppg_abi_version.restype = C.c_int
    L.ppg_default_config.argtypes = [C.POINTER(PpgConfig)]
    L.ppg_default_config.restype = None
    L.ppg_create.argtypes = [C.POINTER(PpgConfig), i32, i32, C.POINTER(vp)]
    L.ppg_destroy.argtypes = [vp]
    L.ppg_load_tape.argtypes = [vp, C.POINTER(PpgTape)]
    L.ppg_reset.argtypes = [vp, vp, vp, vp]
    L.ppg_step.argtypes = [vp, vp, vp, vp]
    L.ppg_step_ordered.argtypes = [vp, vp, vp, vp, vp, vp]
    L.ppg_step_host.argtypes = [vp, vp, vp, C.POINTER(PpgBuffers), vp, vp]
    L.ppg_random_actions.argtypes = [vp, u64, vp, vp, vp]
    L.ppg_get_buffers.argtypes = [vp, C.POINTER(PpgBuffers)]
    L.ppg_selftest_pow.argtypes = [vp, vp, vp, C.c_int64, i32]
    L.ppg_rollout_random.argtypes = [C.POINTER(vp), i32, C.POINTER(vp), i32, u64]
    L.ppg_set_pdl_chain.argtypes = [i32]
    L.ppg_snapshot_size.argtypes = [vp]
    L.ppg_snapshot_size.restype = C.c_size_t
    L.ppg_snapshot.argtypes = [vp, vp, C.c_size_t, vp]
    L.ppg_restore.argtypes = [vp, vp, C.c_size_t, vp]
    L.ppg_read_env.argtypes = [vp, i32] + [vp] * 9
    L.ppg_read_env_eco.argtypes = [vp, i32] + [vp] * 6
    L.ppg_read_env_stag.argtypes = [vp, i32] + [vp] * 6
    L.ppg_read_episode_eco.argtypes = [vp, i32, vp, vp]
    L.ppg_read_episode_events_eco.argtypes = [vp, i32, vp]
    L.ppg_read_env_acc.argtypes = [vp, i32, vp, vp]
    L.ppg_world_state.argtypes = [vp, i32, i32, vp, vp]
    L.ppg_track_returns.argtypes = [vp, i32, vp]
    L.ppg_get_returns.argtypes = [vp, C.POINTER(PpgReturns)]
    L.ppg_episode_stats_device.argtypes = [vp, C.POINTER(vp), vp]
    L.ppg_episode_stats_clear.argtypes = [vp, vp]
    L.ppg_stats.argtypes = [vp, vp, vp]
    L.ppg_stats_device.argtypes = [vp, C.POINTER(vp), vp]
    L.ppg_stats_clear.argtypes = [vp, vp]
    L.ppg_launch_count.argtypes = [vp]
    L.ppg_launch_count.restype = C.c_int64
    L.ppg_profile_begin.argtypes = [vp]
    L.ppg_profile_env_cycles.argtypes = [vp, vp, vp, vp, vp, vp]
    L.ppg_profile_end.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(i32)]
    L.ppg_last_error.argtypes = [vp]
    L.ppg_last_error.restype = C.c_char_p
    _lib = L
    return L


def check(rc, handle=None):
    if rc != 0:
        msg = load().ppg_last_error(handle)
        raise PpgError(f"ppg error {rc}: {msg.decode() if msg else ''}")
