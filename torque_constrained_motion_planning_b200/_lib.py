"""ctypes loader for libtcmp.so (include/tcmp.h).  No torch types cross this boundary: callers
pass integer addresses (``tensor.data_ptr()`` / ``ndarray.ctypes.data``) and sizes.

The loader FAILS LOUDLY when the CUDA library is missing or cannot be loaded: there is no CPU
fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# TCMP_LIB selects an experimental build (libtcmp<suffix>.so of build.build(suffix=...)) for A/B scripts; still a
# libtcmp CUDA library or nothing -- there is no CPU fallback either way
LIB_PATH = os.environ.get("TCMP_LIB") or os.path.join(_HERE, "libtcmp.so")

OK = 0
MODE = {"rne": 0, "nov": 1, "dyn": 2, "base": 3}
DTYPE = {"f64": 0, "f32": 1}
PAYLOAD_THRESHOLD_TEST = 0.01  # panda_primitives.py:139,178
PAYLOAD_THRESHOLD_RAW = 0.0    # rne.py:184

_vp = ctypes.c_void_p
_i64 = ctypes.c_int64
_i32 = ctypes.c_int
_f64 = ctypes.c_double

# name -> (restype, argtypes); every symbol include/tcmp.h declares
SIGNATURES = {
    "tcmp_abi_version": (_i32, []),
    "tcmp_last_error": (ctypes.c_char_p, []),
    "tcmp_device_count": (_i32, []),
    "tcmp_rne_batch": (_i32, [_i32, _i32, _i64, _vp, _vp, _vp, _vp, _f64, _f64, _vp, _vp, _vp]),
    "tcmp_model_default": (_i32, [_vp]),
    "tcmp_rne_batch_model": (_i32, [_vp, _i32, _i32, _i64, _vp, _vp, _vp, _vp, _f64, _f64, _vp, _vp, _vp]),
    "tcmp_dynamics_batch": (_i32, [_vp, _i64, _vp, _vp, _vp, _f64, _vp, _vp, _vp, _vp, _vp]),
    "tcmp_forward_dynamics_batch": (_i32, [_vp, _i32, _i64, _vp, _vp, _vp, _vp, _f64, _vp, _vp, _vp]),
    "tcmp_rollout_batch": (_i32, [_vp, _i32, _i64, _i32, _f64, _vp, _vp, _vp, _i32, _vp, _f64, _vp, _vp, _vp, _vp, _vp, _vp,
                                  _vp, _vp, _vp]),
    "tcmp_track_batch": (_i32, [_vp, _i32, _i64, _i32, _f64, _i32, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _f64, _vp, _f64,
                                _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "tcmp_payload_interval_batch": (_i32, [_vp, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "tcmp_edge_payload_interval": (_i32, [_vp, _i32, _i64, _i32, _vp, _vp, _i32, _vp, _vp, _vp, _vp]),
    "tcmp_edge_feasibility_model": (_i32, [_vp, _i32, _i32, _i64, _i32, _vp, _vp, _f64, _f64, _i32, _vp, _vp]),
    "tcmp_traj_feasibility_model": (_i32, [_vp, _i32, _i32, _i32, _i32, _vp, _f64, _f64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "tcmp_ik_select_model": (_i32, [_vp, _i64, _vp, _vp, _vp, _i32, _i32, _vp, _i32, _vp, _vp, _i32, _f64, _f64, _i32, _vp, _vp,
                              _vp, _vp]),
    "tcmp_extend_prefix_model": (_i32, [_vp, _i32, _i64, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _f64, _f64, _f64, _vp, _vp, _vp]),
    "tcmp_rne_batch_scatter": (_i32, [_i32, _i32, _i64, _vp, _vp, _vp, _vp, _f64, _f64, _vp, _i32,
                                      ctypes.POINTER(_vp), _i64, _vp]),
    "tcmp_rne_batch_scatter_mc": (_i32, [_i32, _i32, _i64, _vp, _vp, _vp, _vp, _f64, _f64, _vp, _i32,
                                         ctypes.POINTER(_vp), _vp, _i64, _vp]),
    "tcmp_peer_push": (_i32, [_vp, _i64, _i32, ctypes.POINTER(_vp), _i64, _vp]),
    "tcmp_peer_signal": (_i32, [_i32, _i32, ctypes.POINTER(_vp), _vp]),
    "tcmp_peer_wait": (_i32, [_vp, _i32, _vp]),
    "tcmp_peer_alloc": (_i32, [ctypes.POINTER(_vp), _i64, ctypes.c_char_p]),
    "tcmp_peer_free": (_i32, [_vp]),
    "tcmp_peer_open": (_i32, [ctypes.c_char_p, ctypes.POINTER(_vp)]),
    "tcmp_peer_close": (_i32, [_vp]),
    "tcmp_edge_feasibility": (_i32, [_i32, _i32, _i64, _i32, _vp, _vp, _f64, _f64, _i32, _vp, _vp]),
    "tcmp_edge_feasibility_scatter": (_i32, [_i32, _i64, _i32, _vp, _vp, _f64, _f64, _i32, _i32, ctypes.POINTER(_vp),
                                             _i64, _vp]),
    "tcmp_traj_feasibility": (_i32, [_i32, _i32, _i32, _i32, _vp, _f64, _f64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "tcmp_ik_batch": (_i32, [_i64, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp]),
    "tcmp_ik_select": (_i32, [_i64, _vp, _vp, _vp, _i32, _i32, _vp, _i32, _vp, _vp, _i32, _f64, _f64, _i32, _vp, _vp,
                              _vp, _vp]),
    "tcmp_collision_batch": (_i32, [_i64, _vp, _i32, _vp, _vp, _vp, _f64, _vp, _vp]),
    "tcmp_extend_prefix": (_i32, [_i32, _i64, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _f64, _f64, _f64, _vp, _vp, _vp]),
    "tcmp_fk_batch": (_i32, [_i64, _vp, _vp, _vp, _vp]),
    "tcmp_workspace_create": (_i32, [ctypes.POINTER(_vp), _i64]),
    "tcmp_workspace_destroy": (_i32, [_vp]),
    "tcmp_rne_batch_host": (_i32, [_vp, _i32, _i32, _i64, _vp, _vp, _vp, _vp, _f64, _f64, _vp, _vp]),
    "tcmp_rne_batch_host_async": (_i32, [_vp, _i32, _i32, _i64, _vp, _vp, _vp, _vp, _f64, _f64, _vp, _vp]),
    "tcmp_workspace_sync": (_i32, [_vp]),
    "tcmp_edge_feasibility_host": (_i32, [_vp, _i32, _i32, _i64, _i32, _vp, _vp, _f64, _f64, _i32, _vp]),
    "tcmp_ik_batch_host": (_i32, [_vp, _i64, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp]),
    "tcmp_host_alloc": (_i32, [ctypes.POINTER(_vp), _i64]),
    "tcmp_host_free": (_i32, [_vp]),
    "tcmp_fp64_peak": (_i32, [_i32, ctypes.POINTER(_f64), _vp]),
    "tcmp_get_limits": (_i32, [_vp, _vp, _vp, _vp]),
}


class TcmpError(RuntimeError):
    pass


_lib = None


def load():
    """Load libtcmp.so once.  Raises TcmpError (never falls back) if it is absent or unloadable."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise TcmpError(
            "libtcmp.so is not built (%s). Build it with `python -m torque_constrained_motion_planning_b200.build` "
            "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
    try:
        lib = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)
    except OSError as e:  # pragma: no cover
        raise TcmpError("cannot load %s: %s" % (LIB_PATH, e)) from e
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.tcmp_abi_version() != 1:
        raise TcmpError("libtcmp.so ABI version %d != 1" % lib.tcmp_abi_version())
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != OK:
        msg = load().tcmp_last_error()
        raise TcmpError("libtcmp call failed (%d): %s" % (rc, msg.decode() if msg else "?"))
