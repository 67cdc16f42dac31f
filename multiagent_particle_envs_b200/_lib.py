"""ctypes binding of libmpe_b200.so (the C ABI declared in include/mpe_b200.h).

There is no CPU fallback: if the CUDA extension has not been built, or a call fails, this module
raises.  Build with `python -c "import __graft_entry__ as g; g.build()"` (or `make -C
multiagent_particle_envs_b200/csrc`).
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MPE_B200_LIB") or os.path.join(_HERE, "csrc", "libmpe_b200.so")   # override: kernel A/B experiments

MPE_ABI_VERSION = 1
MPE_MAX_AGENTS = 8
MPE_MAX_LANDMARKS = 8

# enum mpe_scenario
SCN_SIMPLE, SCN_SPREAD, SCN_TAG, SCN_WORLD_COMM, SCN_ADVERSARY, SCN_PUSH, SCN_SPEAKER_LISTENER, \
    SCN_REFERENCE, SCN_CRYPTO, SCN_CUSTOM = range(10)

# enum mpe_step_flags
FLAG_SHARED_REWARD = 1
FLAG_FORCE_DISCRETE_ACTION = 2
FLAG_DISCRETE_ACTION_INPUT = 4
FLAG_HOST_SLAB = 8
FLAG_SAMPLE_ACTIONS = 16

ERR_BAD_ARG = -1
ERR_UNSUPPORTED = -3
ERR_NO_DEVICE = -5


class MpeDesc(ctypes.Structure):
    """mirror of `struct mpe_desc` (include/mpe_b200.h)"""
    _fields_ = [
        ("abi_version", ctypes.c_int32),
        ("scenario", ctypes.c_int32),
        ("n_agents", ctypes.c_int32),
        ("n_landmarks", ctypes.c_int32),
        ("dim_c", ctypes.c_int32),
        ("n_adversaries", ctypes.c_int32),
        ("n_obstacles", ctypes.c_int32),
        ("n_food", ctypes.c_int32),
        ("n_forests", ctypes.c_int32),
        ("reserved_i", ctypes.c_int32 * 7),
        ("dt", ctypes.c_double),
        ("damping", ctypes.c_double),
        ("contact_force", ctypes.c_double),
        ("contact_margin", ctypes.c_double),
        ("agent_size", ctypes.c_double * MPE_MAX_AGENTS),
        ("agent_mass", ctypes.c_double * MPE_MAX_AGENTS),
        ("agent_sens", ctypes.c_double * MPE_MAX_AGENTS),
        ("agent_max_speed", ctypes.c_double * MPE_MAX_AGENTS),
        ("landmark_size", ctypes.c_double * MPE_MAX_LANDMARKS),
        ("agent_movable", ctypes.c_uint8 * MPE_MAX_AGENTS),
        ("agent_collide", ctypes.c_uint8 * MPE_MAX_AGENTS),
        ("agent_silent", ctypes.c_uint8 * MPE_MAX_AGENTS),
        ("agent_adversary", ctypes.c_uint8 * MPE_MAX_AGENTS),
        ("agent_leader", ctypes.c_uint8 * MPE_MAX_AGENTS),
        ("landmark_collide", ctypes.c_uint8 * MPE_MAX_LANDMARKS),
        ("reserved_b", ctypes.c_uint8 * 16),
    ]


class MpeError(RuntimeError):
    pass


_P = ctypes.c_void_p
_PP = ctypes.POINTER(ctypes.c_void_p)
_SIGNATURES = {
    # name: (restype, argtypes)
    "mpe_create": (ctypes.c_int, [ctypes.POINTER(MpeDesc), ctypes.c_int64, ctypes.c_int, ctypes.POINTER(_P)]),
    "mpe_destroy": (ctypes.c_int, [_P]),
    "mpe_num_agents": (ctypes.c_int, [_P]),
    "mpe_num_envs": (ctypes.c_int64, [_P]),
    "mpe_obs_dim": (ctypes.c_int, [_P, ctypes.c_int]),
    "mpe_act_dim": (ctypes.c_int, [_P, ctypes.c_int]),
    "mpe_num_speakers": (ctypes.c_int, [_P]),
    "mpe_num_goals": (ctypes.c_int, [_P]),
    "mpe_info_dim": (ctypes.c_int, [_P]),
    "mpe_bytes_per_env_step": (ctypes.c_int64, [_P]),
    "mpe_reset": (ctypes.c_int, [_P, _P, _P, _P, _P, _P, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64, _P]),
    "mpe_reset_dev_epoch": (ctypes.c_int, [_P, _P, _P, _P, _P, _P, ctypes.c_uint64, ctypes.c_uint64, _P, _P]),
    "mpe_set_action": (ctypes.c_int, [_P, _PP, _P, _P, ctypes.c_uint32, _P]),
    "mpe_world_step": (ctypes.c_int, [_P, _P, _P, _P, _P, _P, _P]),
    "mpe_observe": (ctypes.c_int, [_P, _P, _P, _P, _P, _PP, _P, _P, _P, ctypes.c_uint32, _P]),
    "mpe_step": (ctypes.c_int, [_P, _P, _P, _P, _P, _PP, _PP, _P, _P, _P, ctypes.c_uint32, _P]),
    "mpe_rollout": (ctypes.c_int, [_P, _P, _P, _P, _P, _PP, ctypes.c_int32, _PP, _P, _P, _P, ctypes.c_uint32, _P]),
    "mpe_rollout_policy": (ctypes.c_int, [_P, _P, _P, _P, _P, _PP, _PP, _PP, _PP, ctypes.c_int32, ctypes.c_int32, _PP, _P, _P,
                                          _PP, _P, ctypes.c_uint32, _P]),
    "mpe_collect": (ctypes.c_int, [_P, _P, _P, _P, _P, ctypes.c_int32, ctypes.c_int32, _PP, _PP, _PP, _PP, _PP, _PP,
                                   ctypes.c_int32, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_uint64, _PP, _P, _P, _PP, _PP,
                                   _P, ctypes.c_uint32, _P]),
    "mpe_collect_supported": (ctypes.c_int, [_P, ctypes.c_int32, ctypes.c_int32]),
    "mpe_step_host": (ctypes.c_int, [_P, _P, _P, _P, _P, _PP, _PP, _PP, _P, _P, _P, _PP, _P, _P, _P,
                                     ctypes.c_uint32, _P]),
    "mpe_strerror": (ctypes.c_char_p, [ctypes.c_int]),
    "mpe_last_cuda_error": (ctypes.c_char_p, []),
    "mpe_abi_version": (ctypes.c_int, []),
    "mpe_kernel_launches": (ctypes.c_int64, []),
    "mpe_probe_stream": (ctypes.c_int, [ctypes.c_int, _P, ctypes.c_int64, _P, ctypes.c_int64, ctypes.c_int64, _P]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def load():
    """Load libmpe_b200.so; raises ImportError (loudly) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "multiagent_particle_envs_b200: CUDA extension %s is missing. There is no CPU fallback. "
            "Build it with `python -c \"import __graft_entry__ as g; g.build()\"`." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.mpe_abi_version() != MPE_ABI_VERSION:
        raise ImportError("libmpe_b200.so ABI %d != binding ABI %d" % (lib.mpe_abi_version(), MPE_ABI_VERSION))
    _lib = lib
    return lib


def check(rc, what=""):
    if rc >= 0:
        return rc
    lib = load()
    msg = lib.mpe_strerror(rc).decode()
    if rc == -4:
        msg += ": " + lib.mpe_last_cuda_error().decode()
    raise MpeError("%s failed: %s" % (what or "libmpe_b200 call", msg))


def ptr_array(ptrs):
    arr = (ctypes.c_void_p * len(ptrs))(*ptrs)
    return arr
