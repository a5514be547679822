"""ctypes binding of the batched C ABI (include/mfmarl_batched.h).  A missing library is a hard error."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.normpath(os.path.join(_HERE, "..", "..", "build", "libmagent.so"))


class MfbConfig(ctypes.Structure):
    _fields_ = [
        ("n_envs", ctypes.c_int), ("map_width", ctypes.c_int), ("map_height", ctypes.c_int),
        ("capacity", ctypes.c_int), ("embedding_size", ctypes.c_int), ("rng_mode", ctypes.c_int),
        ("seed", ctypes.c_uint), ("env_base", ctypes.c_int), ("max_steps", ctypes.c_int),
        ("auto_reset", ctypes.c_int), ("device", ctypes.c_int), ("step_threads", ctypes.c_int),
        ("obs_tile_agents", ctypes.c_int), ("obs_record", ctypes.c_int), ("concurrent_step_envs", ctypes.c_int),
        ("random_sides", ctypes.c_int),
        ("hp", ctypes.c_float), ("speed", ctypes.c_float), ("view_radius", ctypes.c_float),
        ("attack_radius", ctypes.c_float), ("damage", ctypes.c_float), ("step_recover", ctypes.c_float),
        ("kill_supply", ctypes.c_float), ("step_reward", ctypes.c_float), ("kill_reward", ctypes.c_float),
        ("dead_penalty", ctypes.c_float), ("attack_penalty", ctypes.c_float),
        ("attack_bonus", ctypes.c_float * 2),
    ]


_lib = None


def load_library(path=None):
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or os.environ.get("MAGENT_LIB") or LIB_PATH
    if not os.path.exists(path):
        raise OSError("CUDA engine library not found at %s -- build it with `python __graft_entry__.py`; "
                      "there is no CPU fallback" % path)
    lib = ctypes.CDLL(path, ctypes.RTLD_GLOBAL)
    vp, ci, cp = ctypes.c_void_p, ctypes.c_int, ctypes.c_char_p
    sig = {
        "mfb_default_config": [ctypes.POINTER(MfbConfig)],
        "mfb_create": [ctypes.POINTER(MfbConfig), ctypes.POINTER(vp)],
        "mfb_destroy": [vp],
        "mfb_reset": [vp],
        "mfb_add_walls": [vp, ci, vp, vp],
        "mfb_add_agents": [vp, ci, ci, vp, vp, ctypes.POINTER(ci)],
        "mfb_add_agents_per_env": [vp, ci, ci, vp, vp, vp],
        "mfb_add_agents_random": [vp, ci, ci, ci, ci, ci, ci],
        "mfb_set_seed": [vp, ctypes.c_ulong],
        "mfb_query": [vp, cp, ctypes.POINTER(ci)],
        "mfb_observe": [vp, vp, vp, ci, vp],
        "mfb_observe_groups": [vp, vp, vp, vp, vp, vp],
        "mfb_observe_groups_bf16": [vp, vp, vp, vp, vp, vp],
        "mfb_state_device_ptr": [vp, cp, ctypes.POINTER(vp)],
        "mfb_step": [vp, vp, vp, vp, vp, vp, vp, ci, vp],
        "mfb_clear_dead": [vp, vp],
        "mfb_mean_action": [vp, vp, vp, ci, ci, ci, vp],
        "mfb_local_mean_action": [vp, ctypes.c_double, vp, vp, vp],
        "mfb_get": [vp, cp, vp, vp],
        "mfb_num_device_ptr": [vp, ctypes.POINTER(vp)],
        "mfb_save_envs": [vp, ci, vp, vp, vp],
        "mfb_load_envs": [vp, ci, vp, vp, vp],
        "mfb_render_observations": [vp, ci, vp, ci, vp, vp, vp, vp, vp],
        "mfb_step_host": [vp, vp, vp, vp, vp, vp, vp],
        "mfb_step_host_async": [vp, vp, vp, vp, vp, vp, vp, ctypes.POINTER(ci)],
        "mfb_host_wait": [vp, ci],
        "mfb_alloc_device": [ctypes.c_ulong, ci, ctypes.POINTER(vp), ctypes.POINTER(ci)],
        "mfb_free_device": [vp],
        "mfi_step_lattices": [ci, ci, ci, vp, vp, vp, ctypes.c_double, vp, vp, ctypes.c_uint, ctypes.c_uint,
                              ctypes.c_uint, vp, vp, vp, vp],
        "mfi_run_lattices": [ci, ci, ci, ci, vp, vp, vp, ctypes.c_double, vp, vp, ctypes.c_uint, ctypes.c_uint,
                             ctypes.c_uint, vp, vp, vp],
        "mfi_metropolis": [ci, ci, ci, vp, vp, ctypes.c_uint, ctypes.c_uint, ctypes.c_uint, vp, vp, vp],
        "mfi_swendsen_wang": [ci, ci, ci, vp, vp, ctypes.c_uint, ctypes.c_uint, ctypes.c_uint, vp, vp, vp],
    }
    for name, argtypes in sig.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = ci
    lib.mfb_last_error.restype = cp
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise RuntimeError(load_library().mfb_last_error().decode("utf-8", "replace"))
