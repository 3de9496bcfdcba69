"""ctypes binding of the C-ABI in include/pioneer_b200.h (libpioneer_b200.so, sm_100a).

This is the only place the shared library is opened.  There is no CPU fallback: if the library is
missing and cannot be built with nvcc, importing the env classes raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

from . import build as _build

PNR_ABI_VERSION = 4
PNR_DOF = 6
PNR_OBS_DIM = 137
PNR_MAX_CAPSULES = 8
PNR_MAX_OBSTACLES = 4
PNR_STATS_LEN = 8
PNR_FILTER_DELTA_LEN = 1 + 2 * PNR_OBS_DIM

PNR_OK = 0
PNR_ARITH_F32, PNR_ARITH_LEGACY64 = 0, 1
PNR_OBS_TERMINAL, PNR_OBS_AUTORESET = 0, 1
PNR_MODE_KINEMATIC, PNR_MODE_DYNAMIC = 0, 1
PNR_DONE, PNR_TRUNCATED = 1, 2
PNR_OBSTACLE_NONE, PNR_OBSTACLE_PLANE, PNR_OBSTACLE_BOX, PNR_OBSTACLE_SPHERE = 0, 1, 2, 3
PNR_STEPPING_EXPLICIT, PNR_STEPPING_BULLET = 0, 1
PNR_HOST_FULL, PNR_HOST_COMPACT = 0, 1
PNR_OBS_COMPACT_DIM, PNR_OBS_CONST_BEGIN, PNR_OBS_CONST_END = 101, 18, 54
PNR_SYNC_MAX_PEERS, PNR_SYNC_WINDOW_BYTES, PNR_SYNC_IPC_BYTES = 16, 73984, 64

_d3 = C.c_double * 3
_d9 = C.c_double * 9


class pnr_model(C.Structure):
    _fields_ = [
        ("dof", C.c_int32), ("n_capsules", C.c_int32),
        ("axis", _d3 * PNR_DOF), ("origin_xyz", _d3 * PNR_DOF), ("origin_rot", _d9 * PNR_DOF),
        ("tip_xyz", _d3),
        ("lower", C.c_double * PNR_DOF), ("upper", C.c_double * PNR_DOF),
        ("effort", C.c_double * PNR_DOF), ("damping", C.c_double * PNR_DOF),
        ("body_mass", C.c_double * PNR_DOF), ("body_com", _d3 * PNR_DOF), ("body_inertia", _d9 * PNR_DOF),
        ("capsule_body", C.c_int32 * PNR_MAX_CAPSULES), ("capsule_radius", C.c_double * PNR_MAX_CAPSULES),
        ("capsule_p0", _d3 * PNR_MAX_CAPSULES), ("capsule_p1", _d3 * PNR_MAX_CAPSULES),
    ]


class pnr_config(C.Structure):
    _fields_ = [
        ("max_v_to_r", C.c_double), ("max_a_to_v", C.c_double),
        ("done_distance", C.c_double),
        ("award_max", C.c_double), ("award_done", C.c_double),
        ("award_potential_slope", C.c_double), ("penalty_step", C.c_double),
        ("target_lo", _d3), ("target_hi", _d3),
        ("timestep", C.c_double), ("frame_skip", C.c_int32),
        ("gravity", C.c_double),
        ("max_episode_steps", C.c_int32), ("arith", C.c_int32), ("obs_mode", C.c_int32),
        ("auto_reset", C.c_int32), ("mode", C.c_int32),
        ("kp", C.c_double), ("kd", C.c_double), ("torque_scale", C.c_double),
        ("n_obstacles", C.c_int32), ("obstacle_type", C.c_int32 * PNR_MAX_OBSTACLES),
        ("obstacle_p", _d3 * PNR_MAX_OBSTACLES), ("obstacle_e", _d3 * PNR_MAX_OBSTACLES),
        ("contact_penalty", C.c_double),
        ("random_box", C.c_int32),
        ("box_pos_lo", C.c_double * 2), ("box_pos_hi", C.c_double * 2), ("box_size_lo", _d3), ("box_size_hi", _d3),
        ("stepping", C.c_int32),
        ("link_damping", C.c_double), ("max_velocity", C.c_double),
        ("motor_kp", C.c_double), ("motor_kd", C.c_double), ("motor_max_force", C.c_double),
    ]


_H = C.c_void_p          # pnr_handle*
_P = C.c_void_p          # raw device / host data pointer
_S = C.c_void_p          # cudaStream_t

# name -> (restype, argtypes); kept in one table so tests can check it against the header
SIGNATURES = {
    "pnr_abi_version": (C.c_int, []),
    "pnr_last_error": (C.c_char_p, []),
    "pnr_default_config": (None, [C.POINTER(pnr_config)]),
    "pnr_create": (C.c_int, [C.POINTER(pnr_model), C.POINTER(pnr_config), C.c_int64, C.c_int64, C.c_int,
                             C.c_uint64, C.POINTER(_H)]),
    "pnr_destroy": (None, [_H]),
    "pnr_num_envs": (C.c_int64, [_H]),
    "pnr_get_bounds": (C.c_int, [_H, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float),
                                 C.POINTER(C.c_float)]),
    "pnr_get_obs_constants": (C.c_int, [_H, C.POINTER(C.c_float)]),
    "pnr_seed": (C.c_int, [_H, C.c_uint64]),
    "pnr_get_counters": (C.c_int, [_H, C.POINTER(C.c_uint32), C.POINTER(C.c_double), C.POINTER(C.c_uint64)]),
    "pnr_set_counters": (C.c_int, [_H, C.c_uint32, C.c_double]),
    "pnr_tick_advance": (C.c_int, [_H, C.c_uint32, _S]),
    "pnr_reset": (C.c_int, [_H, _P, C.c_int64, _P, _P, _P, _S]),
    "pnr_step": (C.c_int, [_H, _P, _P, _P, _P, _S]),
    "pnr_step_many": (C.c_int, [_H, C.c_int32, _P, C.c_int64, _P, C.c_int64, _P, _P, _S]),
    "pnr_step_host": (C.c_int, [_H, _P, _P, _P, _P]),
    "pnr_step_host_begin": (C.c_int, [_H, _P, _P, _P, _P, C.c_int]),
    "pnr_step_host_end": (C.c_int, [_H]),
    "pnr_expand_obs_host": (C.c_int, [_H, _P, _P, C.c_int64]),
    "pnr_observe": (C.c_int, [_H, _P, C.c_int64, _P, _S]),
    "pnr_observe_done": (C.c_int, [_H, _P, _P, _P, _S]),
    "pnr_get_state": (C.c_int, [_H, _P, _P, _P, _P, _P, _P, _P, _S]),
    "pnr_set_state": (C.c_int, [_H, _P, _P, _P, _P, _P, _P, _P, _S]),
    "pnr_get_boxes": (C.c_int, [_H, _P, _S]),
    "pnr_set_boxes": (C.c_int, [_H, _P, _S]),
    "pnr_stats": (C.c_int, [_H, C.POINTER(C.c_double), C.c_int, _S]),
    "pnr_set_stats": (C.c_int, [_H, C.POINTER(C.c_double)]),
    "pnr_stats_merge_device": (C.c_int, [_P, C.c_int, C.c_int, _P, _S]),
    "pnr_stats_device": (C.c_int, [_H, _P, C.c_int, _S]),
    "pnr_sync_window_create": (C.c_int, [_H, C.POINTER(C.c_ubyte)]),
    "pnr_sync_window_ptr": (C.c_int, [_H, C.POINTER(C.c_void_p)]),
    "pnr_sync_window_connect": (C.c_int, [_H, C.POINTER(C.c_ubyte), C.c_int, C.c_int]),
    "pnr_sync_window_connect_ptrs": (C.c_int, [_H, C.POINTER(C.c_void_p), C.c_int, C.c_int]),
    "pnr_iteration_sync": (C.c_int, [_H, C.c_int, C.c_int, _P, C.c_int, _S]),
    "pnr_sync_status": (C.c_int, [_H, C.POINTER(C.c_int)]),
    "pnr_filter_configure": (C.c_int, [_H, C.c_double, C.c_int, C.c_int]),
    "pnr_filter_apply": (C.c_int, [_H, _P, _P, C.c_int64, C.c_int, C.c_int, _S]),
    "pnr_filter_fuse": (C.c_int, [_H, C.c_int, C.c_int]),
    "pnr_filter_delta_device": (C.c_int, [_H, _P, _S]),
    "pnr_filter_sync": (C.c_int, [_H, C.POINTER(C.c_double), _S]),
    "pnr_filter_sync_device": (C.c_int, [_H, _P, _S]),
    "pnr_filter_get": (C.c_int, [_H, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "pnr_filter_set": (C.c_int, [_H, C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_double), _S]),
    "pnr_launch_count": (C.c_int64, [_H]),
}

_lib: Optional[C.CDLL] = None


class PioneerB200Error(RuntimeError):
    pass


def load(build_if_missing: bool = True) -> C.CDLL:
    """Open libpioneer_b200.so (building it in-tree with nvcc first if it is missing or stale)."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    override = os.environ.get("PIONEER_B200_LIB")        # another build of the library (A/B comparisons)
    if override:
        path, build_if_missing = override, False
    if build_if_missing:
        try:
            path = _build.build()
        except Exception as exc:  # no nvcc on this machine: use the shipped library if there is one
            if not os.path.exists(path):
                raise ImportError("pioneer_b200: the CUDA library is not built and nvcc failed "
                                  f"(there is no CPU fallback): {exc}") from exc
    if not os.path.exists(path):
        raise ImportError(f"pioneer_b200: {path} not found; run `python -m pioneer_b200.build` "
                          "(there is no CPU fallback)")
    lib = C.CDLL(path)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = header and library disagree
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.pnr_abi_version() != PNR_ABI_VERSION:
        raise ImportError(f"pioneer_b200: ABI version {lib.pnr_abi_version()} != {PNR_ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != PNR_OK:
        msg = load().pnr_last_error()
        raise PioneerB200Error(f"{what or 'pioneer_b200'} failed ({rc}): {msg.decode() if msg else ''}")


def _fill(dst, src):
    """Copy a (nested) numpy array into a (nested) ctypes array."""
    import numpy as np
    flat = np.ascontiguousarray(src, dtype=np.float64).ravel()
    C.memmove(dst, flat.ctypes.data, flat.nbytes)


def model_from_chain(chain) -> pnr_model:
    """pioneer_b200.urdf.ChainModel -> pnr_model.  The static base transform must be identity
    (it is for the Pioneer arm; a general one would be folded into origin[0] here)."""
    import numpy as np
    assert chain.dof == PNR_DOF, f"the CUDA path is built for {PNR_DOF} DoF, the URDF has {chain.dof}"
    assert np.allclose(chain.base_rot, np.eye(3)) and np.allclose(chain.base_xyz, 0.0)
    m = pnr_model()
    m.dof = chain.dof
    _fill(m.axis, chain.axis); _fill(m.origin_xyz, chain.origin_xyz); _fill(m.origin_rot, chain.origin_rot)
    _fill(m.tip_xyz, chain.tip_xyz)
    _fill(m.lower, chain.lower); _fill(m.upper, chain.upper)
    _fill(m.effort, chain.effort); _fill(m.damping, chain.damping)
    _fill(m.body_mass, chain.body_mass); _fill(m.body_com, chain.body_com); _fill(m.body_inertia, chain.body_inertia)
    caps = chain.capsules[:PNR_MAX_CAPSULES]
    assert len(chain.capsules) <= PNR_MAX_CAPSULES, "too many collision capsules"
    m.n_capsules = len(caps)
    for i, (body, radius, p0, p1) in enumerate(caps):
        m.capsule_body[i] = int(body)
        m.capsule_radius[i] = float(radius)
        for k in range(3):
            m.capsule_p0[i][k] = float(p0[k])
            m.capsule_p1[i][k] = float(p1[k])
    return m
