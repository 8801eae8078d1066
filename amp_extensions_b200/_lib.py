"""ctypes binding of libsimstep.so (include/simstep.h).

There is no fallback: if the shared library is missing or does not load, importing a compute entry
point raises.  The CPU oracle under oracle/ is test infrastructure and is never imported from here.
"""
import ctypes as C
import os

from . import build as _build

_c_float_p = C.POINTER(C.c_float)
_c_void_p = C.c_void_p

MAX_HIDDEN = 8
MAX_BODIES = 32
MAX_JOINTS = 32
ABI_VERSION = 1

PREC = {"tf32": 0, "fp16": 1, "bf16": 2}
ACT = {"relu": 0, "tanh": 1}
SHAPE = {"sphere": 0, "capsule": 1, "box": 2}
RFF_INPUT = {None: 0, "s": 1, "sa": 2, "ss": 3, "sas": 4}  # SIMSTEP_RFF_INPUT_*; None: inferred from in_dim


class SimstepConfig(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32),
        ("state_dim", C.c_int32),
        ("action_dim", C.c_int32),
        ("n_models", C.c_int32),
        ("n_hidden", C.c_int32),
        ("hidden", C.c_int32 * MAX_HIDDEN),
        ("dense_connect", C.c_int32),
        ("activation", C.c_int32),
        ("transform", C.c_int32),
        ("precision", C.c_int32),
        ("max_chunk_envs", C.c_int32),
        ("reserved", C.c_int32 * 7),
    ]


class SimstepTermination(C.Structure):
    _fields_ = [
        ("horizon", C.c_int32),
        ("enable_velocity_check", C.c_int32),
        ("vel_offset", C.c_int32),
        ("vel_threshold", C.c_float),
        ("vel_divisor", C.c_float),
        ("record_all_world", C.c_int32),
        ("record_world_root_pos", C.c_int32),
        ("n_bodies", C.c_int32),
        ("body_offset", C.c_int32 * MAX_BODIES),
        ("body_shape", C.c_int32 * MAX_BODIES),
        ("body_param0", C.c_float * MAX_BODIES),
        ("body_param1", C.c_float * MAX_BODIES),
        ("pos_dim", C.c_int32),
    ]


class SimstepCharacter(C.Structure):
    _fields_ = [
        ("n_joints", C.c_int32),
        ("joint_type", C.c_int32 * MAX_JOINTS),
        ("parent", C.c_int32 * MAX_JOINTS),
        ("attach", (C.c_float * 3) * MAX_JOINTS),
        ("param_offset", C.c_int32 * MAX_JOINTS),
        ("is_end_eff", C.c_int32 * MAX_JOINTS),
        ("diff_weight", C.c_float * MAX_JOINTS),
        ("body_mass", C.c_float * MAX_JOINTS),
        ("body_attach", (C.c_float * 3) * MAX_JOINTS),
        ("dof", C.c_int32),
    ]


_SIGNATURES = {
    # name: (restype, argtypes)
    "simstep_abi_version": (C.c_int, []),
    "simstep_last_error": (C.c_char_p, [_c_void_p]),
    "simstep_create": (C.c_int, [C.POINTER(SimstepConfig), C.POINTER(_c_void_p)]),
    "simstep_destroy": (C.c_int, [_c_void_p]),
    "simstep_query": (C.c_int, [_c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "simstep_load_ensemble": (C.c_int, [_c_void_p, C.POINTER(_c_void_p), C.POINTER(_c_void_p), C.POINTER(_c_void_p)]),
    "simstep_set_termination": (C.c_int, [_c_void_p, C.POINTER(SimstepTermination)]),
    "simstep_load_rff": (C.c_int, [_c_void_p, C.c_int32, C.c_int32, _c_void_p, _c_void_p, C.c_int32]),
    "simstep_load_rff_typed": (C.c_int, [_c_void_p, C.c_int32, C.c_int32, C.c_int32, _c_void_p, _c_void_p, C.c_int32]),
    "simstep_set_rff_split": (C.c_int, [_c_void_p, C.c_int32]),
    "simstep_saturation_count": (C.c_int, [_c_void_p, C.POINTER(C.c_int64), C.c_int32]),
    "simstep_forward_launches": (C.c_int, [_c_void_p, C.c_int64, C.POINTER(C.c_int32)]),
    "simstep_debug_check_guards": (C.c_int, [_c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "simstep_debug_chain_schedule": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32),
                                               C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "simstep_forward": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, C.c_int64, _c_void_p, _c_void_p]),
    "simstep_discrepancy": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, C.c_int64, _c_void_p, _c_void_p]),
    "simstep_step": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p, C.c_int64, _c_void_p,
                               _c_void_p, _c_void_p, _c_void_p]),
    "simstep_step_cost": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p, C.c_int64, _c_void_p,
                                    _c_void_p, _c_void_p, _c_void_p, C.c_float, C.c_float, C.c_float, C.c_float,
                                    C.c_int32, _c_void_p, _c_void_p, _c_void_p, _c_void_p]),
    "simstep_rff_features": (C.c_int, [_c_void_p, _c_void_p, C.c_int64, _c_void_p, _c_void_p, _c_void_p]),
    "simstep_rff_dot": (C.c_int, [_c_void_p, _c_void_p, C.c_int64, _c_void_p, _c_void_p, _c_void_p]),
    "simstep_bonus_cost": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, C.c_int64, _c_void_p, C.c_float, C.c_float,
                                     C.c_float, C.c_float, C.c_int32, _c_void_p, _c_void_p, _c_void_p, _c_void_p]),
    "simstep_load_clip": (C.c_int, [_c_void_p, C.POINTER(SimstepCharacter), C.c_int32, _c_void_p, _c_void_p,
                                    _c_void_p, C.c_float, C.c_int32, _c_void_p]),
    "simstep_imitation_reward": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p, C.c_int64,
                                           _c_void_p, _c_void_p, _c_void_p]),
    "simstep_clip_sample": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, C.c_int64, _c_void_p, _c_void_p, _c_void_p]),
    "simstep_record_state": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
                                       C.c_float, _c_void_p, _c_void_p]),
    "simstep_load_feature_net": (C.c_int, [_c_void_p, C.POINTER(_c_void_p), C.POINTER(_c_void_p), C.c_int32, _c_void_p,
                                           _c_void_p, C.c_int32]),
    "simstep_set_cost_transform": (C.c_int, [_c_void_p, C.c_int32]),
    "simstep_load_policy": (C.c_int, [_c_void_p, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                      C.POINTER(_c_void_p), C.POINTER(_c_void_p), C.c_int32, _c_void_p, _c_void_p,
                                      _c_void_p, _c_void_p, _c_void_p]),
    "simstep_policy_act": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, C.c_int64, _c_void_p, _c_void_p, _c_void_p]),
    "simstep_discount": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p, C.c_int32,
                                   C.c_int64, C.c_float, C.c_float, _c_void_p, _c_void_p, _c_void_p]),
    "simstep_auto_reset": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p, C.c_int32, C.c_int64,
                                     _c_void_p, _c_void_p, _c_void_p, _c_void_p]),
    "simstep_moments": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, C.c_int64, _c_void_p, _c_void_p]),
    "simstep_whiten": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, C.c_int64, _c_void_p, C.c_float, _c_void_p,
                                 _c_void_p]),
    "simstep_train_init": (C.c_int, [_c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_float, C.c_float, C.c_float]),
    "simstep_train_step": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, _c_void_p, C.c_int32, C.c_float, _c_void_p,
                                     _c_void_p]),
    "simstep_train_loss": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, _c_void_p, C.c_int32, _c_void_p, _c_void_p]),
    "simstep_train_grads": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, _c_void_p, C.c_int32, _c_void_p, _c_void_p]),
    "simstep_train_export": (C.c_int, [_c_void_p, C.c_int32, C.POINTER(_c_void_p), C.POINTER(_c_void_p)]),
    "simstep_npg_init": (C.c_int, [_c_void_p, C.c_float, C.POINTER(C.c_int64)]),
    "simstep_npg_params": (C.c_int, [_c_void_p, C.c_int32, _c_void_p, _c_void_p]),
    "simstep_npg_grad": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p, C.c_int64, _c_void_p, _c_void_p]),
    "simstep_npg_prepare": (C.c_int, [_c_void_p, _c_void_p, C.c_int64, _c_void_p, C.c_int64, _c_void_p]),
    "simstep_npg_fvp": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, C.c_int64, _c_void_p, C.c_int64, _c_void_p, _c_void_p,
                                  _c_void_p]),
    "simstep_npg_cg": (C.c_int, [_c_void_p, C.c_int32, _c_void_p, C.c_double, _c_void_p]),
    "simstep_npg_apply": (C.c_int, [_c_void_p, C.c_double, C.c_int32, _c_void_p]),
    "simstep_npg_diag": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p, C.c_int64, _c_void_p, _c_void_p]),
    "simstep_npg_scalars": (C.c_int, [_c_void_p, _c_void_p, _c_void_p]),
    "simstep_baseline_init": (C.c_int, [_c_void_p, C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.c_float, C.c_float,
                                        C.c_float, C.c_float, C.c_float, _c_void_p, _c_void_p, _c_void_p, C.c_int64]),
    "simstep_baseline_state": (C.c_int, [_c_void_p, C.c_int32, _c_void_p, _c_void_p, _c_void_p, _c_void_p,
                                         C.POINTER(C.c_int64)]),
    "simstep_baseline_predict": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, C.c_int64, _c_void_p, _c_void_p]),
    "simstep_baseline_fit": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, _c_void_p, C.c_int64, _c_void_p, C.c_int64,
                                       C.c_int32, C.c_int32, _c_void_p]),
    "simstep_bc_init": (C.c_int, [_c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_float, C.c_float, C.c_float,
                                  C.c_float, C.c_float, _c_void_p, _c_void_p, _c_void_p, C.c_int64,
                                  C.POINTER(C.c_int64)]),
    "simstep_bc_state": (C.c_int, [_c_void_p, C.c_int32, _c_void_p, _c_void_p, _c_void_p, _c_void_p,
                                   C.POINTER(C.c_int64)]),
    "simstep_bc_loss": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, C.c_int64, _c_void_p, _c_void_p]),
    "simstep_bc_fit": (C.c_int, [_c_void_p, _c_void_p, _c_void_p, C.c_int64, _c_void_p, C.c_int64, C.c_int32,
                                 C.c_int32, _c_void_p]),
    "simstep_bc_commit": (C.c_int, [_c_void_p, _c_void_p]),
    "simstep_histogram": (C.c_int, [_c_void_p, _c_void_p, C.c_int64, C.c_double, C.c_double, C.c_int32, _c_void_p,
                                    _c_void_p]),
    "simstep_quantile_op": (C.c_int, [_c_void_p, C.c_int32, _c_void_p, C.c_int64, C.c_int32, _c_void_p, _c_void_p,
                                      _c_void_p, _c_void_p]),
    "simstep_reduce_max_sum": (C.c_int, [_c_void_p, _c_void_p, C.c_int64, _c_void_p, _c_void_p]),
    "simstep_profile_enable": (C.c_int, [_c_void_p, C.c_int32]),
    "simstep_profile_read": (C.c_int, [_c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.c_int32]),
    "simstep_debug_gemm": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_int32, _c_void_p, _c_void_p,
                                     _c_void_p, _c_void_p, _c_void_p]),
    "simstep_launch_count": (C.c_int64, []),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


class SimstepError(RuntimeError):
    pass


def lib_path():
    return _build.LIB


def load(build_if_missing=True):
    """Load libsimstep.so (building it in-tree with nvcc when absent). Raises if that is impossible."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if not os.path.exists(path):
        if not build_if_missing:
            raise SimstepError(f"{path} is missing; run `python -m amp_extensions_b200.build`")
        _build.build()
    elif build_if_missing and os.path.exists(_build.STAMP) and _build.needs_build() and _build.have_nvcc():
        _build.build()   # the sources changed since the library was built: never run stale kernels silently
    lib = C.CDLL(path, mode=C.RTLD_GLOBAL)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here means the .so does not match simstep.h
        fn.restype = res
        fn.argtypes = args
    got = lib.simstep_abi_version()
    if got != ABI_VERSION:
        raise SimstepError(f"libsimstep ABI {got} != binding ABI {ABI_VERSION}")
    _lib = lib
    return lib


def check(rc, handle=None):
    if rc != 0:
        msg = load().simstep_last_error(handle)
        raise SimstepError(f"libsimstep error {rc}: {msg.decode() if msg else '?'}")


PROF_CATEGORIES = ("prep", "ensemble_gemm", "post", "rff_pack", "rff_gemm", "combine", "imitation", "reserved")


def launch_count():
    return int(load().simstep_launch_count())
