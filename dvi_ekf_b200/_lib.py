"""ctypes binding of libeskf_b200.so (the C ABI declared in include/eskf.h).

There is deliberately no CPU fallback: if the CUDA library is missing or no
CUDA device is usable, every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ESKF_B200_LIB") or os.path.join(HERE, "libeskf_b200.so")

MEM_HOST, MEM_DEVICE = 0, 1
FLAG_ZERO_FROZEN = 1
STATUS_UPDATE_SKIPPED, STATUS_ASIN_DOMAIN = 1, 2
NSTAT = 16
NCONS = 8
NDOFSUM = 80
NCARRY = 4

EXPORTS = (
    "eskf_create", "eskf_destroy", "eskf_set_state", "eskf_set_noise", "eskf_propagate", "eskf_update",
    "eskf_run", "eskf_get_state", "eskf_sync", "eskf_launch_count", "eskf_set_tuning", "eskf_last_error",
    "eskf_version", "eskf_fp64_peak", "eskf_set_variant", "eskf_noise_dump", "eskf_prepass", "eskf_prepass_last_error",
    "eskf_set_prepass_budget", "eskf_keep_jacobians", "eskf_get_jacobians", "eskf_keep_consistency", "eskf_get_consistency",
    "eskf_get_dof_history", "eskf_get_dof_envelope", "eskf_run_epochs", "eskf_set_groups", "eskf_get_group_sums",
    "eskf_set_meas_dropout", "eskf_set_meas_outliers", "eskf_set_innovation_gate",
)


class EskfModel(C.Structure):
    _fields_ = [
        ("scope_length", C.c_double),
        ("cam_angle_rad", C.c_double),
        ("frozen_mask", C.c_int32),
        ("flags", C.c_int32),
    ]


class EskfStreams(C.Structure):
    _fields_ = [
        ("n_steps", C.c_int64),
        ("n_epochs", C.c_int64),
        ("n_traj", C.c_int32),
        ("mem", C.c_int32),
        ("filters_per_traj", C.c_int64),
        ("dt", C.c_void_p),
        ("om_acc", C.c_void_p),
        ("n_prop", C.c_void_p),
        ("cam", C.c_void_p),
        ("notch", C.c_void_p),
        ("cam_ref", C.c_void_p),
        ("imu_ref", C.c_void_p),
        ("gt_dofs", C.c_double * 6),
        ("seed", C.c_uint64),
        ("filter_id0", C.c_int64),
        ("imu_noise_std", C.c_double * 6),
        ("cam_noise_std", C.c_double * 7),
        ("noise_free_filter0", C.c_int32),
        ("noise_id_modulus", C.c_int32),
        ("trace_x", C.c_void_p),
    ]


class EskfPrepassIn(C.Structure):
    _fields_ = [
        ("n_frames", C.c_int64),
        ("interframe_vals", C.c_int32),
        ("euler_mode", C.c_int32),
        ("scale", C.c_double),
        ("gt_dofs", C.c_double * 6),
        ("ic_dofs", C.c_double * 6),
        ("t", C.c_void_p),
        ("xyz", C.c_void_p),
        ("q_xyzw", C.c_void_p),
        ("notch3", C.c_void_p),
    ]


class EskfPrepassOut(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("x0", "u0", "dt", "om_acc", "t_imu", "n_prop", "cam", "notch", "cam_ref", "imu_ref",
                                          "imu_ref_rows")]


class EskfError(RuntimeError):
    pass


_lib = None


def load():
    """Loads the shared library (once) and declares the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise EskfError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback)"
        )
    lib = C.CDLL(LIB_PATH)
    vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int
    lib.eskf_create.argtypes = [C.POINTER(EskfModel), i64, i32, vp, C.POINTER(vp)]
    lib.eskf_destroy.argtypes = [vp]
    lib.eskf_set_state.argtypes = [vp, vp, i64, vp, i64, vp, i64, vp, i64, i32]
    lib.eskf_set_noise.argtypes = [vp, vp, i64, vp, i64, vp, i64, i32]
    lib.eskf_propagate.argtypes = [vp, vp, vp, i64, i32, i32]
    lib.eskf_update.argtypes = [vp, vp, vp, i32, vp, i32]
    lib.eskf_run.argtypes = [vp, C.POINTER(EskfStreams), vp, vp, i32]
    lib.eskf_run_epochs.argtypes = [vp, C.POINTER(EskfStreams), i64, i64, vp, vp, vp, vp, i32]
    lib.eskf_get_state.argtypes = [vp, vp, vp, vp, vp, vp, i32]
    lib.eskf_sync.argtypes = [vp]
    lib.eskf_launch_count.argtypes = [vp]
    lib.eskf_launch_count.restype = i64
    lib.eskf_set_tuning.argtypes = [vp, i32]
    lib.eskf_set_variant.argtypes = [vp, i32]
    lib.eskf_set_prepass_budget.argtypes = [vp, i64]
    lib.eskf_keep_jacobians.argtypes = [vp, i32]
    lib.eskf_get_jacobians.argtypes = [vp, vp, vp, i32]
    lib.eskf_keep_consistency.argtypes = [vp, i32]
    lib.eskf_get_consistency.argtypes = [vp, vp, vp, vp, C.POINTER(i64), i32]
    lib.eskf_get_dof_history.argtypes = [vp, vp, vp, C.POINTER(i64), i32]
    lib.eskf_get_dof_envelope.argtypes = [vp, vp, C.POINTER(i64), i32]
    lib.eskf_set_groups.argtypes = [vp, i64]
    lib.eskf_set_meas_dropout.argtypes = [vp, vp, i64, i64, i32]
    lib.eskf_set_meas_outliers.argtypes = [vp, vp, i64, i64, vp, i32]
    lib.eskf_set_innovation_gate.argtypes = [vp, vp, i64, i32]
    lib.eskf_get_group_sums.argtypes = [vp, vp, vp, vp, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), i32]
    lib.eskf_fp64_peak.argtypes = [i32, vp, i32, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.eskf_noise_dump.argtypes = [i32, vp, C.c_uint64, i64, i64, i64, i64, i32, vp, i32]
    lib.eskf_prepass.argtypes = [i32, vp, C.POINTER(EskfModel), C.POINTER(EskfPrepassIn), C.POINTER(EskfPrepassOut),
                                 C.POINTER(C.c_int64)]
    lib.eskf_prepass_last_error.restype = C.c_char_p
    lib.eskf_last_error.restype = C.c_char_p
    lib.eskf_version.restype = C.c_char_p
    for name in EXPORTS:
        if name not in ("eskf_launch_count", "eskf_last_error", "eskf_version", "eskf_prepass_last_error"):
            getattr(lib, name).restype = i32
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().eskf_last_error().decode(errors="replace")
        raise EskfError(f"{what} failed (code {rc}): {msg}")
