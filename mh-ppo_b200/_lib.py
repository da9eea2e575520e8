"""ctypes binding of libmhppo_b200.so (the C ABI of include/mhppo.h).  Fails loudly if the library
has not been built (`python mh-ppo_b200/build.py`) -- there is no fallback path."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MHPPO_LIB", os.path.join(_HERE, "libmhppo_b200.so"))  # override: kernel-tuning experiments only


class LibraryMissing(RuntimeError):
    pass


class MhppoError(RuntimeError):
    pass


class EnvCfg(C.Structure):
    _fields_ = [("variant", C.c_int32), ("nb_car", C.c_int32), ("nb_ped", C.c_int32), ("nb_lines", C.c_int32),
                ("max_episode", C.c_int32), ("sin_model", C.c_int32), ("device", C.c_int32), ("reserved", C.c_int32),
                ("dt", C.c_double), ("car_b", C.c_double * 4), ("ped_b", C.c_double * 8), ("cross_b", C.c_double * 2),
                ("seed", C.c_uint64), ("n_envs", C.c_int64), ("env_id0", C.c_int64)]


class EnvDims(C.Structure):
    _fields_ = [("n_slots", C.c_int32), ("n_lead", C.c_int32), ("n_action", C.c_int32), ("n_obs", C.c_int32),
                ("n_ped", C.c_int32), ("done_step", C.c_int32), ("reserved", C.c_int32 * 2)]


class RolloutCfg(C.Structure):
    _fields_ = [("nb_ped", C.c_int32), ("nb_lines", C.c_int32), ("T", C.c_int32), ("legacy_nb_car", C.c_int32),
                ("n_envs", C.c_int64), ("seed", C.c_uint64), ("env_id0", C.c_int64)]


class View(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("env_stride", C.c_int64), ("comp_stride", C.c_int64)]


# every symbol include/mhppo.h declares (tests/test_abi.py checks the list against the header)
SYMBOLS = {
    "mhppo_abi_version": (C.c_int, []),
    "mhppo_last_error": (C.c_char_p, []),
    "mhppo_device_count": (C.c_int, []),
    "mhppo_env_create": (C.c_int, [C.POINTER(EnvCfg), C.POINTER(C.c_void_p)]),
    "mhppo_env_destroy": (C.c_int, [C.c_void_p]),
    "mhppo_env_get_dims": (C.c_int, [C.c_void_p, C.POINTER(EnvDims)]),
    "mhppo_env_reset": (C.c_int, [C.c_void_p, C.c_void_p, View, C.c_void_p]),
    "mhppo_env_step": (C.c_int, [C.c_void_p, View, View, View, View, C.c_void_p, C.c_int, View, C.c_void_p]),
    "mhppo_env_reset_pedestrian": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mhppo_env_reset_cars": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mhppo_env_observe": (C.c_int, [C.c_void_p, View, C.c_void_p]),
    "mhppo_env_step_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_int, C.c_void_p]),
    "mhppo_env_reset_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "mhppo_env_export_state": (C.c_int, [C.c_void_p] * 8),
    "mhppo_env_import_state": (C.c_int, [C.c_void_p] * 8),
    "mhppo_env_state_bytes_per_env": (C.c_int64, [C.c_void_p]),
    "mhppo_launch_count": (C.c_int64, []),
    "mhppo_net_padded_in": (C.c_int, [C.c_int32]),
    "mhppo_net_param_count": (C.c_int, [C.c_int32]),
    "mhppo_choice_act": (C.c_int, [C.POINTER(RolloutCfg), C.c_void_p, C.c_void_p, C.c_uint32] + [C.c_void_p] * 6),
    "mhppo_choice_eval": (C.c_int, [C.POINTER(RolloutCfg), C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "mhppo_policy_eval": (C.c_int, [C.POINTER(RolloutCfg)] + [C.c_void_p] * 4 + [C.c_float] * 4 + [C.c_void_p] * 3),
    "mhppo_policy_act": (C.c_int, [C.POINTER(RolloutCfg)] + [C.c_void_p] * 5 + [C.c_int32, C.c_uint32] + [C.c_void_p] * 5),
    "mhppo_rollout_steps": (C.c_int, [C.c_void_p, C.POINTER(RolloutCfg)] + [C.c_void_p] * 5 + [C.c_uint32] + [C.c_void_p] * 7 + [C.c_int32, C.c_void_p]),
    "mhppo_episode_stats": (C.c_int, [C.c_void_p] + [C.c_int32] * 6 + [C.c_int64, C.c_float] + [C.c_void_p] * 5),
    "mhppo_returns": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mhppo_update_workspace_bytes": (C.c_int64, [C.c_int32]),
    "mhppo_value_stats": (C.c_int, [C.c_int32, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_int64, C.c_int64] + [C.c_void_p] * 6),
    "mhppo_critic_grad_stats": (C.c_int, [C.c_int32, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p,
                                          C.c_float] + [C.c_void_p] * 6),
    "mhppo_ppo_grad": (C.c_int, [C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_int64, C.c_int64]
                       + [C.c_void_p] * 5 + [C.c_float] * 5 + [C.c_void_p] * 4),
    "mhppo_ppo_grad_dev": (C.c_int, [C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_int64, C.c_int64]
                           + [C.c_void_p] * 6 + [C.c_float] * 3 + [C.c_void_p] * 4),
    "mhppo_ppo_grad_ent": (C.c_int, [C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_int64, C.c_int64]
                           + [C.c_void_p] * 6 + [C.c_float] * 4 + [C.c_void_p] * 4),
    "mhppo_gae": (C.c_int, [C.c_void_p] * 3 + [C.c_int32, C.c_int64, C.c_double, C.c_double] + [C.c_void_p] * 4),
    "mhppo_minibatch_plan": (C.c_int, [C.POINTER(RolloutCfg)] + [C.c_void_p] * 3 + [C.c_uint32, C.c_int32, C.c_int32] + [C.c_void_p] * 5),
    "mhppo_adam2": (C.c_int, [C.c_void_p] * 4 + [C.c_int32, C.c_float, C.c_int32] + [C.c_void_p] * 4 + [C.c_int32, C.c_float, C.c_int32]
                    + [C.c_float] * 3 + [C.c_void_p]),
    "mhppo_critic_grad_diag": (C.c_int, [C.c_int32, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p,
                                         C.c_float] + [C.c_void_p] * 7),
    "mhppo_ppo_grad_diag": (C.c_int, [C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_int64, C.c_int64]
                            + [C.c_void_p] * 6 + [C.c_float] * 4 + [C.c_void_p] * 6),
    "mhppo_adam2_halt": (C.c_int, [C.c_void_p] * 4 + [C.c_int32, C.c_float, C.c_int32] + [C.c_void_p] * 4 + [C.c_int32, C.c_float, C.c_int32]
                         + [C.c_float] * 3 + [C.c_void_p, C.c_double] + [C.c_void_p] * 3),
    "mhppo_adam2_clip": (C.c_int, [C.c_void_p] * 4 + [C.c_int32, C.c_float, C.c_int32] + [C.c_void_p] * 4 + [C.c_int32, C.c_float, C.c_int32]
                         + [C.c_float] * 3 + [C.c_double, C.c_void_p, C.c_void_p, C.c_double] + [C.c_void_p] * 3),
    "mhppo_adam2_sched": (C.c_int, [C.c_void_p] * 4 + [C.c_int32, C.c_float, C.c_int32] + [C.c_void_p] * 4 + [C.c_int32, C.c_float, C.c_int32]
                          + [C.c_float] * 3 + [C.c_double, C.c_void_p, C.c_void_p, C.c_double] + [C.c_void_p] * 2
                          + [C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_void_p, C.c_void_p]),
    "mhppo_tc_failures": (C.c_int, []),
    "mhppo_set_mlp_mode": (C.c_int, [C.c_int32]),
    "mhppo_set_gaussian_head": (C.c_int, [C.c_float, C.c_float, C.c_float, C.c_float]),
    "mhppo_gap_selftest": (C.c_int, [C.c_int64] + [C.c_void_p] * 8 + [C.c_uint64, C.c_uint32, C.c_uint32] + [C.c_void_p] * 5),
    "mhppo_tc_selftest": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "mhppo_adam": (C.c_int, [C.c_void_p] * 4 + [C.c_int32] + [C.c_float] * 4 + [C.c_int32, C.c_float, C.c_void_p]),
}

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LibraryMissing("%s not built: run `python mh-ppo_b200/build.py` (nvcc, sm_100a). "
                                 "mhppo_b200 has no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        if L.mhppo_abi_version() != 1:
            raise MhppoError("ABI version mismatch")
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise MhppoError("mhppo error %d: %s" % (rc, lib().mhppo_last_error().decode()))


def launch_count():
    return int(lib().mhppo_launch_count())
