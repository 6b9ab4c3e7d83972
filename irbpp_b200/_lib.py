"""ctypes binding of the C ABI declared in ``include/irbpp.h``.

There is deliberately no fallback: if ``lib/libirbpp.so`` is missing this raises, and if no CUDA
device is present ``irbpp_create`` fails with ``IRBPP_ECUDA``."""
import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("IRBPP_LIB") or os.path.join(HERE, "lib", "libirbpp.so")   # IRBPP_LIB: build-variant experiments

c_i32, c_i64, c_f64 = ctypes.c_int32, ctypes.c_int64, ctypes.c_double
c_void_p, c_char_p = ctypes.c_void_p, ctypes.c_char_p

IRBPP_OK, IRBPP_EINVAL, IRBPP_ECUDA, IRBPP_ESTATE, IRBPP_EDEVICE = 0, -1, -2, -3, -4
ABI_VERSION = 2


class IrbppConfig(ctypes.Structure):
    _fields_ = [("num_envs", c_i32), ("num_rotations", c_i32), ("selected_action", c_i32),
                ("buffer_size", c_i32), ("bin_dimension", c_f64 * 3), ("resolution_act", c_f64),
                ("resolution_h", c_f64), ("resolution_z", c_f64), ("device", c_i32), ("approx_legacy", c_i32)]


class IrbppStepResult(ctypes.Structure):
    _fields_ = [("reward", c_void_p), ("done", c_void_p), ("valid", c_void_p), ("error", c_void_p),
                ("counter", c_void_p), ("ep_len", c_void_p), ("ratio", c_void_p), ("ep_reward", c_void_p)]


# The block the pointers of IrbppStepResult point into: one array of N per field, in this order
# (csrc/irbpp_kernels.cuh carve_results states the same layout).
RESULT_FIELDS = (("ratio", np.dtype(np.float64)), ("ep_reward", np.dtype(np.float64)), ("reward", np.dtype(np.float32)),
                 ("counter", np.dtype(np.int32)), ("ep_len", np.dtype(np.int32)), ("done", np.dtype(np.uint8)),
                 ("valid", np.dtype(np.uint8)), ("error", np.dtype(np.uint8)))


def result_offsets(n):
    """Byte offset of every array in the result block of n bins, and the size of the block."""
    offsets, size = {}, 0
    for name, dt in RESULT_FIELDS:
        offsets[name] = size
        size += n * dt.itemsize
    return offsets, size


class IrbppReplayBanks(ctypes.Structure):
    _fields_ = [("num_banks", c_i32), ("capacity", c_i32), ("obs_len", c_i32), ("row_stride", c_i32),
                ("tree", c_void_p), ("states", c_void_p), ("actions", c_void_p), ("rewards", c_void_p),
                ("nonterminals", c_void_p), ("index", c_void_p), ("full", c_void_p), ("max_priority", c_void_p),
                ("timestep", c_void_p)]


REPLAY_MAX_STEPS = 16


class IrbppReplaySampleArgs(ctypes.Structure):
    _fields_ = [("batch", c_i32), ("multi_step", c_i32), ("n_step_scaling", ctypes.c_float * REPLAY_MAX_STEPS),
                ("priority_weight", c_f64), ("seed", ctypes.c_uint64), ("counter", ctypes.c_uint64),
                ("u_table", c_void_p), ("max_attempts", c_i32), ("banks", c_void_p), ("tree_index", c_void_p),
                ("states", c_void_p), ("actions", c_void_p), ("returns", c_void_p), ("next_states", c_void_p),
                ("nonterminals", c_void_p), ("weights", c_void_p), ("error", c_void_p)]


# symbol -> (restype, argtypes); every symbol of include/irbpp.h appears here (checked by the tests)
SIGNATURES = {
    "irbpp_abi_version": (c_i32, []),
    "irbpp_create": (c_i32, [ctypes.POINTER(IrbppConfig), ctypes.POINTER(c_void_p)]),
    "irbpp_destroy": (c_i32, [c_void_p]),
    "irbpp_last_error": (c_char_p, [c_void_p]),
    "irbpp_obs_len": (c_i32, [c_void_p, ctypes.POINTER(c_i32), ctypes.POINTER(c_i32), ctypes.POINTER(c_i32)]),
    "irbpp_load_shapes": (c_i32, [c_void_p, c_i32, c_i32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_i64]),
    "irbpp_set_sequences": (c_i32, [c_void_p, c_void_p, c_i32]),
    "irbpp_set_item_rng": (c_i32, [c_void_p, ctypes.c_uint64]),
    "irbpp_reset": (c_i32, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "irbpp_step_async": (c_i32, [c_void_p, c_void_p, c_i32, c_void_p, c_void_p]),
    "irbpp_step_wait": (c_i32, [c_void_p, ctypes.POINTER(IrbppStepResult)]),
    "irbpp_step_wait_device": (c_i32, [c_void_p, ctypes.POINTER(IrbppStepResult)]),
    "irbpp_device_results": (c_i32, [c_void_p, ctypes.POINTER(IrbppStepResult)]),
    "irbpp_get_action_candidates": (c_i32, [c_void_p, c_void_p, c_i32, c_void_p, c_void_p]),
    "irbpp_get_all_possible_observation": (c_i32, [c_void_p, c_void_p, c_void_p]),
    "irbpp_heuristic_actions": (c_i32, [c_void_p, c_i32, c_i32, c_void_p, c_void_p, c_i32, c_void_p]),
    "irbpp_step_poses_async": (c_i32, [c_void_p, c_void_p, c_i32, c_void_p, c_void_p]),
    "irbpp_debug_state": (c_i32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "irbpp_debug_set_heightmap": (c_i32, [c_void_p, c_void_p]),
    "irbpp_debug_scan": (c_i32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "irbpp_debug_hulls": (c_i32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "irbpp_launch_count": (c_i64, [c_void_p]),
    "irbpp_packed_obs_bytes": (c_i32, [c_i32]),
    "irbpp_pack_observations": (c_i32, [c_void_p, c_i64, c_i32, c_i32, c_void_p, c_void_p]),
    "irbpp_unpack_observations": (c_i32, [c_void_p, c_i32, c_i32, c_void_p, c_i64, c_void_p]),
    "irbpp_sample_point_clouds": (c_i32, [c_void_p, c_i32, c_i32, c_void_p, c_i64, c_i32, c_void_p, c_i32, ctypes.c_uint64,
                                          ctypes.c_uint64, c_i32, c_void_p, c_void_p, c_void_p]),
    "irbpp_shape_features": (c_i32, [c_void_p, c_i32, c_i32, c_void_p, c_i64, c_i32, c_void_p, c_i32, ctypes.c_uint64,
                                     ctypes.c_uint64, c_i32, c_void_p, c_void_p, c_void_p, c_void_p, ctypes.c_float,
                                     c_void_p, c_void_p, c_void_p]),
    "irbpp_debug_phase_cycles": (c_i32, [c_void_p, c_i32, c_void_p]),
    "irbpp_replay_append": (c_i32, [ctypes.POINTER(IrbppReplayBanks), c_void_p, c_i64, c_void_p, c_void_p, c_void_p,
                                    c_void_p, ctypes.c_float, c_void_p]),
    "irbpp_replay_sample": (c_i32, [ctypes.POINTER(IrbppReplayBanks), ctypes.POINTER(IrbppReplaySampleArgs), c_void_p]),
    "irbpp_replay_update_priorities": (c_i32, [ctypes.POINTER(IrbppReplayBanks), c_void_p, c_void_p, c_i32, c_void_p]),
}

_LIB = None


class IrbppError(RuntimeError):
    def __init__(self, code, message):
        RuntimeError.__init__(self, "irbpp error %d: %s" % (code, message))
        self.code = code


def load():
    """Load ``libirbpp.so`` (built by ``irbpp_b200.build``); fails loudly when it is missing."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("CUDA library %s not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the library does not export the symbol
        fn.restype = res
        fn.argtypes = args
    if lib.irbpp_abi_version() != ABI_VERSION:
        raise RuntimeError("libirbpp ABI %d != binding %d" % (lib.irbpp_abi_version(), ABI_VERSION))
    _LIB = lib
    return lib


def check(lib, handle, rc):
    if rc != IRBPP_OK:
        msg = lib.irbpp_last_error(handle)
        raise IrbppError(rc, msg.decode() if msg else "?")
