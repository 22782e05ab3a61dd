"""ctypes binding of libcrl_b200.so (include/crl_b200.h).

There is deliberately no fallback: if the CUDA library has not been built or
cannot be loaded, importing the simulator fails loudly.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcrl_b200.so")

CRL_OK = 0
CRL_E_INVALID, CRL_E_CUDA, CRL_E_STATE, CRL_E_SERVES = -1, -2, -3, -4   # include/crl_b200.h
ATLAS_SHAPE = (22, 22, 34, 160, 3)
DEFAULT_ATLAS = os.path.join(_HERE, "data", "scoreboard_atlas.npz")

EXPORTS = [
    "crl_abi_version", "crl_last_error", "crl_pong_create", "crl_pong_destroy", "crl_pong_load_atlas",
    "crl_pong_inject_serves", "crl_pong_seed", "crl_pong_reset", "crl_pong_step", "crl_pong_step_state",
    "crl_pong_render_obs", "crl_pong_render_obs_generic", "crl_pong_terminal_obs", "crl_pong_step_host",
    "crl_pong_get_state", "crl_pong_set_state", "crl_pong_render_raw", "crl_pong_random_actions",
    "crl_launch_count", "crl_pong_check", "crl_pong_get_stats", "crl_pong_ring_phase", "crl_pong_render_obs_f32", "crl_pong_reset_state",
    "crl_pong_set_obs_buffers", "crl_pong_forget_obs",
    "crl_car_create", "crl_car_destroy", "crl_car_load_glyphs", "crl_car_inject_tracks", "crl_car_load_tracks", "crl_car_reset",
    "crl_car_step", "crl_car_step_state", "crl_car_render_obs", "crl_car_get_state", "crl_car_get_track",
    "crl_car_random_actions", "crl_car_get_stats", "crl_car_get_contacts", "crl_car_check",
    "crl_car_seed", "crl_car_step_host", "crl_car_set_elapsed", "crl_car_set_state", "crl_car_ring_phase", "crl_car_render_state", "crl_car_set_obs_rotation",
    "crl_obs_alloc", "crl_obs_free",
]


class PongConfig(ctypes.Structure):
    _fields_ = [
        ("num_envs", ctypes.c_int32), ("n_agents", ctypes.c_int32), ("resized_dim", ctypes.c_int32),
        ("frame_stack", ctypes.c_int32), ("max_num_rounds", ctypes.c_int32), ("device", ctypes.c_int32),
        ("stack_mode", ctypes.c_int32), ("zero_on_done", ctypes.c_int32),
        ("seed", ctypes.c_uint64), ("first_env", ctypes.c_int64),
    ]


class CarConfig(ctypes.Structure):
    _fields_ = [
        ("num_envs", ctypes.c_int32), ("num_players", ctypes.c_int32), ("frame_stack", ctypes.c_int32),
        ("action_repeat", ctypes.c_int32), ("max_episode_steps", ctypes.c_int32), ("device", ctypes.c_int32),
        ("done_mode", ctypes.c_int32), ("stack_mode", ctypes.c_int32),
        ("seed", ctypes.c_uint64), ("first_env", ctypes.c_int64),
    ]


DEFAULT_CAR_GLYPHS = os.path.join(_HERE, "data", "car_hud_glyphs.npz")


_lib = None
_ext = None
EXT_PATH = os.path.join(_HERE, "_crl_torch.so")


def ext():
    """The torch C++ extension of the host layer (csrc/crl_torch.cpp, built in-tree by build.py).  The vec-envs call the
    library only through it; there is no ctypes or CPU fallback behind them: a missing extension is an ImportError."""
    global _ext
    if _ext is None:
        if not os.path.exists(EXT_PATH) or not os.path.exists(LIB_PATH):
            raise ImportError(
                "%s not found: the CUDA extension is not built. Run `python competitive-rl_b200/build.py` "
                "(there is no CPU fallback)." % (EXT_PATH if os.path.exists(LIB_PATH) else LIB_PATH))
        import importlib.util
        import sys
        import torch  # noqa: F401  (loads libc10 / libtorch before the extension)
        name = (__name__.rsplit(".", 1)[0] + "._crl_torch") if "." in __name__ else "_crl_torch"
        spec = importlib.util.spec_from_file_location(name, EXT_PATH)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        sys.modules[name] = mod
        _ext = mod
    return _ext


try:                      # one exception type whichever way the library was called
    CrlError = ext().CrlError
except ImportError:       # not built yet; the ctypes path below still reports errors

    class CrlError(RuntimeError):
        pass


def load():
    """Load the C-ABI library; raises if it is missing (build with build.py / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "%s not found: the CUDA extension is not built. Run `python competitive-rl_b200/build.py` "
            "(there is no CPU fallback)." % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    vp, i32, u64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_uint64
    L.crl_abi_version.restype = ctypes.c_int
    L.crl_last_error.restype = ctypes.c_char_p
    L.crl_launch_count.restype = u64
    L.crl_pong_create.argtypes = [ctypes.POINTER(PongConfig), ctypes.POINTER(vp)]
    L.crl_pong_destroy.argtypes = [vp]
    L.crl_pong_load_atlas.argtypes = [vp, vp, ctypes.c_size_t, vp]
    L.crl_pong_inject_serves.argtypes = [vp, vp, i32, vp]
    L.crl_pong_seed.argtypes = [vp, u64]
    L.crl_pong_reset.argtypes = [vp, vp, vp, vp]
    L.crl_pong_step.argtypes = [vp] * 9
    L.crl_pong_step_state.argtypes = [vp] * 7
    L.crl_pong_render_obs.argtypes = [vp] * 4
    L.crl_pong_render_obs_generic.argtypes = [vp] * 4
    L.crl_pong_terminal_obs.argtypes = [vp] * 5
    L.crl_pong_step_host.argtypes = [vp] * 11
    L.crl_pong_get_state.argtypes = [vp, vp, vp]
    L.crl_pong_set_state.argtypes = [vp, vp, vp]
    L.crl_pong_render_raw.argtypes = [vp, i32, vp, vp, vp]
    L.crl_pong_random_actions.argtypes = [vp, i32, u64, u64, vp]
    L.crl_pong_check.argtypes = [vp, vp]
    L.crl_pong_ring_phase.argtypes = [vp]
    L.crl_pong_render_obs_f32.argtypes = [vp, i32, vp, vp, vp, vp]
    L.crl_pong_reset_state.argtypes = [vp, vp]
    L.crl_pong_get_stats.argtypes = [vp, vp, vp]
    L.crl_pong_set_obs_buffers.argtypes = [vp, ctypes.POINTER(vp), ctypes.POINTER(vp), i32, vp]
    L.crl_pong_forget_obs.argtypes = [vp]
    L.crl_obs_alloc.argtypes = [i32, ctypes.c_size_t, ctypes.POINTER(vp), ctypes.POINTER(i32)]
    L.crl_obs_free.argtypes = [vp]
    L.crl_car_create.argtypes = [ctypes.POINTER(CarConfig), ctypes.POINTER(vp)]
    L.crl_car_destroy.argtypes = [vp]
    L.crl_car_load_glyphs.argtypes = [vp, vp, ctypes.c_size_t, vp]
    L.crl_car_inject_tracks.argtypes = [vp, vp, i32, vp, i32, vp]
    L.crl_car_load_tracks.argtypes = [vp, vp, vp, i32, vp]
    L.crl_car_reset.argtypes = [vp, vp, vp]
    L.crl_car_step.argtypes = [vp] * 9
    L.crl_car_step_state.argtypes = [vp] * 7
    L.crl_car_seed.argtypes = [vp, u64, vp]
    L.crl_car_step_host.argtypes = [vp] * 10
    L.crl_car_set_elapsed.argtypes = [vp, vp, vp]
    L.crl_car_set_state.argtypes = [vp, vp, vp]
    L.crl_car_ring_phase.argtypes = [vp]
    L.crl_car_set_obs_rotation.argtypes = [vp, ctypes.POINTER(vp), i32, vp]
    L.crl_car_render_state.argtypes = [vp, vp, vp]
    L.crl_car_render_obs.argtypes = [vp] * 4
    L.crl_car_get_state.argtypes = [vp, vp, vp]
    L.crl_car_get_track.argtypes = [vp, i32, ctypes.POINTER(i32), vp, i32, vp]
    L.crl_car_random_actions.argtypes = [vp, i32, u64, u64, vp]
    L.crl_car_get_stats.argtypes = [vp, vp, vp]
    L.crl_car_get_contacts.argtypes = [vp, vp, vp, vp]
    L.crl_car_check.argtypes = [vp, vp]
    for name in EXPORTS:
        fn = getattr(L, name)
        if name not in ("crl_last_error", "crl_launch_count"):
            fn.restype = ctypes.c_int
    _lib = L
    return L


def check(rc):
    if rc != CRL_OK:
        raise CrlError("crl error %d: %s" % (rc, load().crl_last_error().decode()))


def launch_count():
    return int(load().crl_launch_count())
