"""ctypes binding of ``libocd_b200.so`` -- the C ABI declared in ``include/ocd_b200.h``.

There is no CPU fallback: if the shared library is missing this module raises at import, and on a
machine without a CUDA device every compute entry point returns ``OCD_ECUDA`` which is raised as
:class:`OcdCudaError`.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import os

_HERE = Path(__file__).resolve().parent
# OCD_B200_LIB: a variant build of the same library (scripts/tuning/build_variants.sh) for A/B measurements
LIB_PATH = Path(os.environ["OCD_B200_LIB"]).resolve() if os.environ.get("OCD_B200_LIB") else _HERE / "libocd_b200.so"

ABI_VERSION = 3
MAX_LANES, MAX_OTHER, MAX_PLAN, MAX_H, MAX_STARTS = 4, 7, 16, 64, 6
LBFGS_MAX_H = 16
OK, EINVAL, EUNSUP, ECUDA, ENOMEM = 0, -1, -2, -3, -4
SMOOTH_F, SMOOTH_THRESHOLD, SMOOTH_BUMP = 0, 1, 2
FORM_THROUGHPUT, FORM_LATENCY, FORM_WIDE, FORM_TIME_PARALLEL = 0, 1, 2, 3


class OcdError(RuntimeError):
    """Any non-zero status from the engine."""


class OcdCudaError(OcdError):
    """OCD_ECUDA: no CUDA device, or a launch/copy failed."""


class ocd_params(C.Structure):
    """Mirror of ``ocd_params`` (include/ocd_b200.h)."""
    _fields_ = [
        ("H", C.c_int32), ("C", C.c_int32), ("L", C.c_int32), ("n_iter", C.c_int32),
        ("num_lanes", C.c_int32), ("other_mode", C.c_int32), ("extra_inits", C.c_int32),
        ("math_mode", C.c_int32), ("optimizer", C.c_int32), ("reserved", C.c_int32),
        ("lr", C.c_double), ("dt", C.c_double), ("friction", C.c_double), ("target_speed", C.c_double),
        ("lane_x", C.c_double * MAX_LANES),
    ]


class ocd_scenario(C.Structure):
    """Mirror of ``ocd_scenario`` (include/ocd_b200.h)."""
    _fields_ = [
        ("n_other", C.c_int32), ("critical_t", C.c_int32),
        ("kind", C.c_int32 * MAX_OTHER), ("plan_len", C.c_int32 * MAX_OTHER),
        ("init_state", (C.c_float * 4) * MAX_OTHER),
        ("friction", C.c_float * MAX_OTHER),
        ("control", (C.c_float * 2) * MAX_OTHER),
        ("plan", ((C.c_float * 2) * MAX_PLAN) * MAX_OTHER),
        ("teleport_state", C.c_float * 4),
    ]


_P, _I64, _I32 = C.c_void_p, C.c_int64, C.c_int32
_PROTOTYPES = {
    # name: (restype, argtypes)
    "ocd_abi_version": (C.c_int, []),
    "ocd_strerror": (C.c_char_p, [C.c_int]),
    "ocd_num_starts": (C.c_int, [_P]),
    "ocd_device_count": (C.c_int, []),
    "ocd_dynamics_step_batch": (C.c_int, [_P, _P, C.c_float, C.c_float, _P, _P, _I64, _P]),
    "ocd_smooth_batch": (C.c_int, [C.c_int, _P, C.c_double, C.c_double, _P, _I64, _P]),
    "ocd_features_batch": (C.c_int, [_P, _P, _P, _I64, _P]),
    "ocd_reward_grad_batch": (C.c_int, [_P, _P, _P, _P, _I64, _P, _I64, _P, _P, _P, _I64, _P]),
    "ocd_kernel_form": (C.c_int, [_P, _I64, C.c_int]),
    "ocd_feature_jacobian_batch": (C.c_int, [_P, _P, _P, _P, _I64, _P, _P, _I64, _P]),
    "ocd_feature_hessian_batch": (C.c_int, [_P, _P, _P, _P, _I64, _P, _I64, _P]),
    "ocd_solve_batch": (C.c_int, [_P, _P, _P, _I64, _P, _I64, _P, _P, _P, _P, _P, _P, _I64, _P]),
    "ocd_solve_vjp_workspace_bytes": (C.c_int, [_P, _I64, C.POINTER(C.c_size_t)]),
    "ocd_solve_vjp_batch": (C.c_int, [_P, _P, _P, _I64, _P, _I64, _P, _P, _P, _P, _P, _P, _P, C.c_size_t, _I64, _P]),
    "ocd_episode_batch": (C.c_int, [_P, _P, _P, _P, _P, _I64, _P, _P, _P, _I32, _I32,
                                    _P, _P, _P, _P, _P, _I64, _P]),
    "ocd_episode_vjp_workspace_bytes": (C.c_int, [_P, _I32, _I64, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "ocd_episode_vjp_batch": (C.c_int, [_P, _P, _P, _I64, _P, _P, _I32, _P, _P, _P, _P, _P, _P, _P, _P, C.c_size_t,
                                        _I64, _P]),
    "ocd_ctx_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "ocd_ctx_destroy": (None, [_P]),
    "ocd_host_register": (C.c_int, [_P, C.c_size_t]),
    "ocd_host_unregister": (C.c_int, [_P]),
    "ocd_solve_batch_host": (C.c_int, [_P, _P, _P, _P, _I64, _P, _I64, _P, _P, _P, _P, _P, _I64]),
    "ocd_solve_first_host": (C.c_int, [_P, _P, _P, _P, _I64, _P, _I64, _P, _P, _P, _P, _P, _I64]),
    "ocd_episode_batch_host": (C.c_int, [_P, _P, _P, _P, _P, _P, _I64, _P, _P, _P, _I32, _I32, _P, _P, _I64]),
    "ocd_fp32_peak": (C.c_int, [C.c_int, C.POINTER(C.c_double), _P]),
}
EXPORTS = tuple(_PROTOTYPES)


def _load() -> C.CDLL:
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C l4dc-mpc-ocd_b200/csrc`). The engine has no CPU fallback.")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in _PROTOTYPES.items():
        fn = getattr(lib, name)      # AttributeError here == header/library mismatch
        fn.restype, fn.argtypes = res, args
    if lib.ocd_abi_version() != ABI_VERSION:
        raise ImportError(f"libocd_b200.so ABI {lib.ocd_abi_version()} != binding ABI {ABI_VERSION}")
    return lib


lib = _load()


def strerror(code: int) -> str:
    return lib.ocd_strerror(int(code)).decode()


def check(code: int, what: str = "") -> None:
    """Raise the Python exception the reference would: ValueError for bad arguments/shapes
    (interact_drive/simulation_utils.py:110-115), OcdCudaError / OcdError otherwise."""
    if code == OK:
        return
    msg = f"{what}: {strerror(code)} (code {code})" if what else f"{strerror(code)} (code {code})"
    if code in (EINVAL, EUNSUP):
        raise ValueError(msg)
    if code == ECUDA:
        raise OcdCudaError(msg)
    if code == ENOMEM:
        raise MemoryError(msg)
    raise OcdError(msg)
