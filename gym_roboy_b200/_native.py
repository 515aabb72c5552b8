"""ctypes binding of include/roboy_b200.h -- the only door into the CUDA library.

There is no CPU fallback: if libroboy_b200.so is missing this raises, and if there is no CUDA
device `roboy_create` fails (ROBOY_E_CUDA) and `check()` raises.
"""
import ctypes
import os

from . import build as _build

ABI_VERSION = 2
DIM_JOINT, DIM_ACTION, DIM_OBS = 3, 8, 9          # the MSJ robot; other robots: RoboyCfg.dim_joint / dim_action
MAX_JOINT, JOINT_PAD, MAX_ACTION = 15, 16, 64    # ROBOY_MAX_JOINT, ROBOY_JOINT_PAD, ROBOY_MAX_ACTION

STEP_MASK = 0x00FFFFFF
F_HELD_ZERO64 = 1 << 24
F_HELD_INFEASIBLE = 1 << 25
ERR_ACTION, ERR_REWARD_RANGE, ERR_GOAL_BOUNDS, ERR_STATE_BOUNDS = 1, 2, 4, 8
REWARD_RANGE_PROBE = 2   # roboy_compute_reward(check_range=ROBOY_REWARD_RANGE_PROBE)
STAT_NAMES = ("steps", "episodes", "successes", "timeouts", "sum_reward", "sum_episode_len", "holds", "violations")
# layout of the packed policy image of roboy_policy_rollout (ROBOY_POLICY_* in include/roboy_b200.h), in floats
POLICY_HIDDEN = 64
POLICY_OFF_W1, POLICY_OFF_B1, POLICY_OFF_W2, POLICY_OFF_B2, POLICY_OFF_W3, POLICY_OFF_B3 = 0, 576, 640, 4736, 4800, 5312
POLICY_NET_FLOATS = 5320
POLICY_OFF_VF, POLICY_OFF_PI, POLICY_OFF_STD, POLICY_OFF_LOGNORM, POLICY_IMAGE_FLOATS = 0, 5320, 10640, 10648, 10652
# indices into the offsets roboy_policy_layout returns for any robot (ROBOY_POLICY_LAYOUT_*)
(POLICY_LAYOUT_W1, POLICY_LAYOUT_B1, POLICY_LAYOUT_W2, POLICY_LAYOUT_B2, POLICY_LAYOUT_W3, POLICY_LAYOUT_VF_B3, POLICY_LAYOUT_PI_B3,
 POLICY_LAYOUT_VF, POLICY_LAYOUT_PI, POLICY_LAYOUT_STD, POLICY_LAYOUT_LOGNORM, POLICY_LAYOUT_FLOATS) = range(12)
POLICY_LAYOUT_WORDS = 12
# roboy_ppo_grad's statistics vector (ROBOY_PPO_STAT_*)
PPO_STAT_NAMES = ("loss", "pg_loss", "vf_loss", "entropy", "approxkl", "clipfrac", "adv_mean", "adv_std", "bad_indices")
# ... and of the tensor-core variant's image (ROBOY_TC_*): float16 element offsets, then byte offsets
TC_K_HIDDEN = 80
TC_OFF_W1, TC_OFF_W2, TC_OFF_W3, TC_NET_HALVES, TC_OFF_VF, TC_OFF_PI = 0, 1024, 6144, 7424, 0, 7424
TC_OFF_LO_BYTES, TC_OFF_STD_BYTES, TC_BIAS32_NET_FLOATS, TC_IMAGE_BYTES = 29696, 59392, 80, 60080
(BUF_GOAL, BUF_STEP_FLAGS, BUF_HELD, BUF_OBS, BUF_REWARD, BUF_DONE, BUF_STATS, BUF_TERMINAL_OBS, BUF_DONE_BITS) = range(9)
HOST_STAGED, HOST_MAPPED_OUT, HOST_MAPPED_ALL = 0, 1, 2


class RoboyCfg(ctypes.Structure):
    """struct roboy_cfg (include/roboy_b200.h); field order is ABI."""
    _fields_ = [
        ("n_envs", ctypes.c_uint64), ("env_id_base", ctypes.c_uint64), ("seed", ctypes.c_uint64),
        ("angle_low", ctypes.c_float), ("angle_high", ctypes.c_float),
        ("vel_low", ctypes.c_float), ("vel_high", ctypes.c_float),
        ("act_low", ctypes.c_float), ("act_high", ctypes.c_float),
        ("max_episode_len", ctypes.c_int32), ("joint_vel_penalty", ctypes.c_int32),
        ("bonus_for_goal", ctypes.c_int32), ("auto_reset", ctypes.c_int32),
        ("penalty_boundary", ctypes.c_float), ("bonus_goal", ctypes.c_float),
        ("reward_lo", ctypes.c_double), ("reward_hi", ctypes.c_double),
        ("dim_joint", ctypes.c_int32), ("dim_action", ctypes.c_int32),
        ("per_component_bounds", ctypes.c_int32), ("reserved", ctypes.c_int32),
        ("angle_low_v", ctypes.c_float * JOINT_PAD), ("angle_high_v", ctypes.c_float * JOINT_PAD),
        ("vel_low_v", ctypes.c_float * JOINT_PAD), ("vel_high_v", ctypes.c_float * JOINT_PAD),
        ("act_low_v", ctypes.c_float * MAX_ACTION), ("act_high_v", ctypes.c_float * MAX_ACTION),
    ]


_vp, _u64, _i32, _int = ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int32, ctypes.c_int
_cfgp = ctypes.POINTER(RoboyCfg)

# name -> (restype, argtypes); every symbol include/roboy_b200.h declares
SIGNATURES = {
    "roboy_abi_version": (_int, []),
    "roboy_last_error": (ctypes.c_char_p, []),
    "roboy_cfg_msj": (_int, [_cfgp]),
    "roboy_hold_interval": (_int, [_cfgp, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float)]),
    "roboy_hold_intervals": (_int, [_cfgp, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float)]),
    "roboy_robot_dims": (_int, [_vp, ctypes.POINTER(_int), ctypes.POINTER(_int), ctypes.POINTER(_int), ctypes.POINTER(_int)]),
    "roboy_fast_division": (_int, [_vp, ctypes.POINTER(_int)]),
    "roboy_penalty_float32": (_int, [_vp, ctypes.POINTER(_int)]),
    "roboy_create": (_int, [_cfgp, _int, ctypes.POINTER(_vp)]),
    "roboy_destroy": (_int, [_vp]),
    "roboy_set_reward_range": (_int, [_vp, ctypes.c_double, ctypes.c_double]),
    "roboy_reset": (_int, [_vp, _vp, _vp, _vp]),
    "roboy_step": (_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "roboy_step_many": (_int, [_vp, ctypes.c_uint32, _vp, _vp, _vp, _vp, _vp]),
    "roboy_step_host": (_int, [_vp, _vp, _vp, _vp, _vp]),
    "roboy_set_host_pipeline": (_int, [_vp, _u64, _int]),
    "roboy_set_host_ramp": (_int, [_vp, _int]),
    "roboy_set_host_pattern": (_int, [_vp, _int]),
    "roboy_set_host_autotune": (_int, [_vp, _int]),
    "roboy_get_host_pipeline": (_int, [_vp, ctypes.POINTER(_u64), ctypes.POINTER(_int), ctypes.POINTER(_int)]),
    "roboy_set_host_mode": (_int, [_vp, _int]),
    "roboy_host_alloc": (_int, [_u64, _int, ctypes.POINTER(_vp)]),
    "roboy_host_free": (_int, [_vp]),
    "roboy_host_copy_probe": (_int, [_vp, _vp, _vp, _vp, _vp, _int, _int, _int, ctypes.POINTER(ctypes.c_double)]),
    "roboy_enable_done_index": (_int, [_vp, _int]),
    "roboy_done_indices": (_int, [_vp, _vp, _u64, _vp, _vp, _vp]),
    "roboy_reseed": (_int, [_vp, _u64]),
    "roboy_set_terminal_obs": (_int, [_vp, _vp]),
    "roboy_compute_reward": (_int, [_vp, _u64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _int, _vp]),
    "roboy_set_goal": (_int, [_vp, _u64, _vp, _vp, _vp]),
    "roboy_set_state": (_int, [_vp, _u64, _vp, _vp, _vp, _vp, _vp]),
    "roboy_set_step_num": (_int, [_vp, _u64, _vp, _vp, _vp]),
    "roboy_read_state": (_int, [_vp, _u64, _vp, _vp, _vp, _vp, _vp]),
    "roboy_sim_step": (_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "roboy_sim_reset": (_int, [_vp, _vp, _vp]),
    "roboy_new_goal": (_int, [_vp, _vp, _vp]),
    "roboy_set_flags": (_int, [_vp, _int, _int, _int]),
    "roboy_set_seed": (_int, [_vp, _u64]),
    "roboy_buffer": (_int, [_vp, _int, ctypes.POINTER(_vp), ctypes.POINTER(_u64)]),
    "roboy_export_dlpack": (_vp, [_vp, _int]),
    "roboy_get_counter": (_int, [_vp, ctypes.POINTER(_u64)]),
    "roboy_set_counter": (_int, [_vp, _u64]),
    "roboy_stats": (_int, [_vp, ctypes.POINTER(ctypes.c_double), _vp]),
    "roboy_clear_stats": (_int, [_vp, _vp]),
    "roboy_clear_errors": (_int, [_vp, _vp]),
    "roboy_errors": (_int, [_vp, ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(_u64), _vp]),
    "roboy_step_external": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "roboy_reset_external": (_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "roboy_gae": (_int, [_u64, _u64, _vp, _vp, _vp, _vp, ctypes.c_float, ctypes.c_float, _vp, _vp, _vp]),
    "roboy_policy_rollout": (_int, [_vp, ctypes.c_uint32, _vp, _u64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _int, _vp]),
    "roboy_policy_rollout_tc": (_int, [_vp, ctypes.c_uint32, _vp, _u64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _int, _int, _vp]),
    "roboy_policy_evaluate": (_int, [_vp, ctypes.c_uint32, _vp, _vp, ctypes.c_uint32, _vp, _vp, _vp, _vp, _vp]),
    "roboy_policy_tc_geometry": (_int, [_vp, _int, _int, ctypes.POINTER(_int), ctypes.POINTER(_int), ctypes.POINTER(_int),
                                        ctypes.POINTER(_int)]),
    "roboy_policy_layout": (_int, [_int, _int, ctypes.POINTER(ctypes.c_uint32)]),
    "roboy_ppo_workspace_bytes": (_int, [_int, _int, _u64, ctypes.POINTER(_u64)]),
    "roboy_ppo_grad": (_int, [_int, _int, _vp, _u64, _vp, _u64, _vp, _vp, _vp, _vp, _vp, ctypes.c_float, ctypes.c_float,
                              ctypes.c_float, ctypes.c_float, _vp, _vp, _vp, _vp]),
    "roboy_policy_geometry": (_int, [_vp, _int, ctypes.POINTER(_int), ctypes.POINTER(_int), ctypes.POINTER(_int),
                                     ctypes.POINTER(_int)]),
    "roboy_launch_count": (_int, [_vp, ctypes.POINTER(_u64)]),
    "roboy_null_step": (_int, [_vp, _vp]),
    "roboy_step_geometry": (_int, [_vp, ctypes.POINTER(_int), ctypes.POINTER(_int), ctypes.POINTER(_int)]),
}

_lib = None


class RoboyNativeError(RuntimeError):
    pass


def lib_path():
    # ROBOY_B200_LIB: load another build of the same library, e.g. another checkout's, to time two versions side by side
    # (the compile-time kernel experiments it used to load are in commit aa5e1cc, removed afterwards)
    return os.environ.get("ROBOY_B200_LIB") or _build.LIB_PATH


def load():
    """Load libroboy_b200.so (building is NOT attempted here: see gym_roboy_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise RoboyNativeError(
            "CUDA library not built: {} is missing. Build it with `python -m gym_roboy_b200.build` "
            "(or __graft_entry__.build()). There is no CPU fallback.".format(path))
    L = ctypes.CDLL(path)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(L, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = restype
        fn.argtypes = argtypes
    if L.roboy_abi_version() != ABI_VERSION:
        raise RoboyNativeError("ABI mismatch: library {} vs binding {}".format(L.roboy_abi_version(), ABI_VERSION))
    _lib = L
    return L


def check(code):
    if code != 0:
        msg = load().roboy_last_error()
        raise RoboyNativeError("roboy_b200 call failed ({}): {}".format(code, (msg or b"").decode()))


def dlpack_capsule(managed_tensor_ptr):
    """Wrap a DLManagedTensor* in the PyCapsule torch.from_dlpack() consumes."""
    if not managed_tensor_ptr:
        check(-1)
    new_capsule = ctypes.pythonapi.PyCapsule_New
    new_capsule.restype = ctypes.py_object
    new_capsule.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_void_p]
    return new_capsule(managed_tensor_ptr, b"dltensor", None)


def policy_layout(dim_obs, dim_action):
    """roboy_policy_layout: the section offsets (indexed by POLICY_LAYOUT_*) of the policy image for these dims, in floats."""
    off = (ctypes.c_uint32 * POLICY_LAYOUT_WORDS)()
    check(load().roboy_policy_layout(int(dim_obs), int(dim_action), off))
    return list(off)
