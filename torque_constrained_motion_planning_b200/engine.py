"""Batched Python entry points over the C-ABI (include/tcmp.h).

Two calling conventions, chosen by the type of the first array argument:

* **device**: ``torch`` CUDA tensors in, ``torch`` CUDA tensors out.  Zero-copy: only
  ``data_ptr()`` and the current stream cross into libtcmp.so.
* **host**: NumPy arrays (or CPU tensors) in, NumPy arrays out, staged through a
  :class:`Workspace` (pinned-or-pageable host memory -> chunked H2D / kernel / D2H pipeline).

All state arrays are structure-of-arrays ``[7][n]`` (joint-major), the layout the kernels read
coalesced.  Nothing here computes torques on the CPU; without a B200 and libtcmp.so every call
raises.
"""
from __future__ import annotations

import ctypes
import threading
from typing import Optional

import numpy as np

from . import _lib
from ._lib import DTYPE, MODE, PAYLOAD_THRESHOLD_TEST, TcmpError, check, load

_NP = {"f64": np.float64, "f32": np.float32}


def _is_cuda_tensor(x) -> bool:
    return hasattr(x, "is_cuda") and bool(x.is_cuda)


def _torch():
    import torch
    return torch


def _tdtype(dtype):
    torch = _torch()
    return {"f64": torch.float64, "f32": torch.float32}[dtype]


def _ptr(t) -> Optional[int]:
    return None if t is None else int(t.data_ptr())


def _nptr(a) -> Optional[int]:
    return None if a is None else int(a.ctypes.data)


def _stream_ptr() -> int:
    return int(_torch().cuda.current_stream().cuda_stream)


def _as_dev(x, dtype, shape, device):
    torch = _torch()
    if x is None:
        return None
    if torch.is_tensor(x) and x.dtype == _tdtype(dtype) and x.device == device and x.is_contiguous() \
            and tuple(x.shape) == tuple(shape):
        return x          # hot path: already a usable buffer, no dispatcher round trips
    if not torch.is_tensor(x):
        x = torch.as_tensor(np.asarray(x), device=device)
    x = x.to(device=device, dtype=_tdtype(dtype)).contiguous()
    if tuple(x.shape) != tuple(shape):
        raise ValueError("expected shape %s, got %s" % (tuple(shape), tuple(x.shape)))
    return x


def _as_host(x, dtype, shape):
    if x is None:
        return None
    if hasattr(x, "numpy") and not isinstance(x, np.ndarray):
        x = x.numpy()
    a = np.ascontiguousarray(x, dtype=_NP[dtype])
    if a.shape != tuple(shape):
        raise ValueError("expected shape %s, got %s" % (tuple(shape), a.shape))
    return a


class Workspace:
    """Device staging buffers + streams for the host-array entry points (tcmp_workspace)."""

    def __init__(self, chunk_states: int = 0):
        self._h = ctypes.c_void_p()
        # a tcmp_workspace serialises nothing itself: one host call at a time per workspace (the shared default
        # workspace is what concurrent Python threads would otherwise collide on)
        self.lock = threading.Lock()
        check(load().tcmp_workspace_create(ctypes.byref(self._h), int(chunk_states)))

    @property
    def handle(self):
        return self._h

    def close(self):
        if self._h:
            load().tcmp_workspace_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass


_default_ws: Optional[Workspace] = None


def default_workspace() -> Workspace:
    global _default_ws
    if _default_ws is None:
        _default_ws = Workspace()
    return _default_ws


def device_count() -> int:
    n = load().tcmp_device_count()
    if n < 0:
        raise TcmpError("no CUDA device: %s" % load().tcmp_last_error().decode())
    return n


class InertialModel:
    """``tcmp_model`` (include/tcmp.h): the masses, centres of mass, inertias, payload lever, tool height and torque
    limits the torque test uses -- what the reference keeps in rne.py's module-level lists ``ms`` / ``cs`` /
    ``inertia_matrices`` (rne.py:102,119,138).  One flat float64[99] record; the attributes are writable views::

        m = InertialModel.default(); m.mass[8] = 1.1; m.com[8] = [0, 0, 0.06]      # another hand
        tau, ok = torque_test_batch(q, qd, qdd, 1.0, model=m)
    """
    DOUBLES = 9 + 27 + 54 + 1 + 1 + 7

    def __init__(self, record=None):
        if record is None:
            record = np.empty(self.DOUBLES)
            check(load().tcmp_model_default(record.ctypes.data))
        self.record = np.ascontiguousarray(record, dtype=np.float64).reshape(self.DOUBLES).copy()

    @classmethod
    def default(cls) -> "InertialModel":
        return cls()

    mass = property(lambda self: self.record[0:9])
    com = property(lambda self: self.record[9:36].reshape(9, 3))
    inertia = property(lambda self: self.record[36:90].reshape(9, 6))
    torque_limit = property(lambda self: self.record[92:99])

    @property
    def payload_radius(self) -> float:
        return float(self.record[90])

    @payload_radius.setter
    def payload_radius(self, v: float) -> None:
        self.record[90] = v

    @property
    def tool_z(self) -> float:
        return float(self.record[91])

    @tool_z.setter
    def tool_z(self, v: float) -> None:
        self.record[91] = v


def _mptr(model) -> Optional[int]:
    """Host pointer of an InertialModel's record for the tcmp_*_model entry points (None -> NULL = stock Panda)."""
    return None if model is None else int(model.record.ctypes.data)


def torque_test_batch(q, qd=None, qdd=None, payload_mass=0.0, mode: str = "rne", dtype: str = "f64",
                      payload_threshold: float = PAYLOAD_THRESHOLD_TEST, want_tau: bool = True,
                      want_mask: bool = True, workspace: Optional[Workspace] = None, out_tau=None, out_mask=None,
                      model: Optional[InertialModel] = None):
    """Batched torque test (tcmp_rne_batch).  q/qd/qdd ``[7][n]``; payload_mass scalar or ``[n]``.
    Returns ``(tau [7][n] or None, feasible uint8 [n] or None)``.  Device path only: ``out_tau`` / ``out_mask``
    are optional preallocated CUDA tensors to write into (no allocation on the call).  ``model``: another inertial
    set than the compiled-in Panda (tcmp_rne_batch_model); host arrays are then staged through torch."""
    lib = load()
    if not (want_tau or want_mask):
        raise ValueError("nothing to compute")
    n = int(q.shape[1])
    scalar = 0.0
    pm = None
    if np.ndim(payload_mass) == 0:
        scalar = float(payload_mass)
    else:
        pm = payload_mass
    if model is not None and not _is_cuda_tensor(q):
        torch = _torch()
        dev = torch.device("cuda", torch.cuda.current_device())
        up = lambda a: None if a is None else torch.as_tensor(_as_host(a, dtype, np.shape(a)), device=dev)
        tau, mask = torque_test_batch(up(q), up(qd), up(qdd), scalar if pm is None else up(pm), mode, dtype,
                                      payload_threshold, want_tau, want_mask, model=model)
        return (None if tau is None else tau.cpu().numpy()), (None if mask is None else mask.cpu().numpy())
    if _is_cuda_tensor(q):
        torch = _torch()
        dev = q.device
        with torch.cuda.device(dev):
            qt = _as_dev(q, dtype, (7, n), dev)
            qdt = _as_dev(qd, dtype, (7, n), dev)
            qddt = _as_dev(qdd, dtype, (7, n), dev)
            pmt = _as_dev(pm, dtype, (n,), dev)
            tau = (out_tau if out_tau is not None else torch.empty((7, n), dtype=_tdtype(dtype), device=dev)) \
                if want_tau else None
            mask = (out_mask if out_mask is not None else torch.empty((n,), dtype=torch.uint8, device=dev)) \
                if want_mask else None
            if model is None:
                check(lib.tcmp_rne_batch(MODE[mode], DTYPE[dtype], n, _ptr(qt), _ptr(qdt), _ptr(qddt), _ptr(pmt),
                                         scalar, float(payload_threshold), _ptr(tau), _ptr(mask), _stream_ptr()))
            else:
                check(lib.tcmp_rne_batch_model(model.record.ctypes.data, MODE[mode], DTYPE[dtype], n, _ptr(qt),
                                               _ptr(qdt), _ptr(qddt), _ptr(pmt), scalar, float(payload_threshold),
                                               _ptr(tau), _ptr(mask), _stream_ptr()))
        return tau, mask
    ws = workspace or default_workspace()
    qa = _as_host(q, dtype, (7, n))
    qda = _as_host(qd, dtype, (7, n))
    qdda = _as_host(qdd, dtype, (7, n))
    pma = _as_host(pm, dtype, (n,))
    tau = np.empty((7, n), dtype=_NP[dtype]) if want_tau else None
    mask = np.empty((n,), dtype=np.uint8) if want_mask else None
    with ws.lock:
        check(lib.tcmp_rne_batch_host(ws.handle, MODE[mode], DTYPE[dtype], n, _nptr(qa), _nptr(qda), _nptr(qdda),
                                      _nptr(pma), scalar, float(payload_threshold), _nptr(tau), _nptr(mask)))
    return tau, mask


def torque_test_batch_host_into(ws: Workspace, mode, dtype, q, qd, qdd, payload_mass, payload_scalar,
                                payload_threshold, tau_out, mask_out) -> None:
    """Allocation-free host call for benchmarking: every array is a preallocated (pinned) ndarray."""
    n = int(q.shape[1])
    with ws.lock:
        check(load().tcmp_rne_batch_host(ws.handle, MODE[mode], DTYPE[dtype], n, _nptr(q), _nptr(qd), _nptr(qdd),
                                         _nptr(payload_mass), float(payload_scalar), float(payload_threshold),
                                         _nptr(tau_out), _nptr(mask_out)))


def torque_test_batch_host_async(ws: Workspace, mode, dtype, q, qd, qdd, payload_mass, payload_scalar,
                                 payload_threshold, tau_out, mask_out) -> None:
    """tcmp_rne_batch_host_async: enqueue one batch of pinned host arrays and return; consecutive batches pipeline on the
    workspace's streams.  Outputs are complete (and inputs reusable) after ``workspace_sync(ws)``."""
    n = int(q.shape[1])
    with ws.lock:
        check(load().tcmp_rne_batch_host_async(ws.handle, MODE[mode], DTYPE[dtype], n, _nptr(q), _nptr(qd), _nptr(qdd),
                                               _nptr(payload_mass), float(payload_scalar), float(payload_threshold),
                                               _nptr(tau_out), _nptr(mask_out)))


def workspace_sync(ws: Workspace) -> None:
    with ws.lock:
        check(load().tcmp_workspace_sync(ws.handle))


def edge_feasibility(qa, qb, n_waypoints: int = 64, payload_mass: float = 0.0, mode: str = "rne",
                     dtype: str = "f64", payload_threshold: float = PAYLOAD_THRESHOLD_TEST,
                     static_only: bool = False, workspace: Optional[Workspace] = None,
                     model: Optional[InertialModel] = None):
    """RRT* edge check (tcmp_edge_feasibility): first infeasible min-jerk waypoint per edge
    (== n_waypoints when the edge is feasible).  qa/qb ``[7][n_edges]``.  ``model``: another inertial set
    (tcmp_edge_feasibility_model; host arrays are then staged through torch)."""
    lib = load()
    n = int(qa.shape[1])
    if model is not None and not _is_cuda_tensor(qa):
        torch = _torch()
        dev = torch.device("cuda", torch.cuda.current_device())
        up = lambda x: torch.as_tensor(_as_host(x, dtype, (7, n)), device=dev)
        return edge_feasibility(up(qa), up(qb), n_waypoints, payload_mass, mode, dtype, payload_threshold,
                                static_only, model=model).cpu().numpy()
    if _is_cuda_tensor(qa):
        torch = _torch()
        dev = qa.device
        with torch.cuda.device(dev):
            a = _as_dev(qa, dtype, (7, n), dev)
            b = _as_dev(qb, dtype, (7, n), dev)
            ff = torch.empty((n,), dtype=torch.int32, device=dev)
            check(lib.tcmp_edge_feasibility_model(_mptr(model), MODE[mode], DTYPE[dtype], n, int(n_waypoints), _ptr(a),
                                                  _ptr(b), float(payload_mass), float(payload_threshold),
                                                  int(static_only), _ptr(ff), _stream_ptr()))
        return ff
    ws = workspace or default_workspace()
    a = _as_host(qa, dtype, (7, n))
    b = _as_host(qb, dtype, (7, n))
    ff = np.empty((n,), dtype=np.int32)
    with ws.lock:
        check(lib.tcmp_edge_feasibility_host(ws.handle, MODE[mode], DTYPE[dtype], n, int(n_waypoints), _nptr(a),
                                             _nptr(b), float(payload_mass), float(payload_threshold),
                                             int(static_only), _nptr(ff)))
    return ff


def traj_feasibility(coeffs, samples_per_segment: int, payload_mass: float = 0.0, mode: str = "rne",
                     dtype: str = "f64", payload_threshold: float = PAYLOAD_THRESHOLD_TEST,
                     want_samples: bool = True, want_tau: bool = True, device=None,
                     model: Optional[InertialModel] = None):
    """Final-trajectory check (tcmp_traj_feasibility[_model]) on min-jerk coefficients ``[n_seg][7][6]``.
    Returns dict(q, qd, qdd, tau  [7][n] tensors or None, feasible uint8 [n], first_fail int)."""
    torch = _torch()
    lib = load()
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    c = np.ascontiguousarray(coeffs, dtype=np.float64)
    n_seg = c.shape[0]
    if c.shape != (n_seg, 7, 6):
        raise ValueError("coeffs must be [n_seg][7][6]")
    S = int(samples_per_segment)
    n = n_seg * S
    with torch.cuda.device(dev):
        ct = torch.as_tensor(c, device=dev)
        td = _tdtype(dtype)
        mk = (lambda: torch.empty((7, n), dtype=td, device=dev))
        q = mk() if want_samples else None
        qd = mk() if want_samples else None
        qdd = mk() if want_samples else None
        tau = mk() if want_tau else None
        mask = torch.empty((n,), dtype=torch.uint8, device=dev)
        ff = torch.full((1,), n, dtype=torch.int32, device=dev)
        check(lib.tcmp_traj_feasibility_model(_mptr(model), MODE[mode], DTYPE[dtype], n_seg, S, _ptr(ct),
                                              float(payload_mass), float(payload_threshold), _ptr(q), _ptr(qd),
                                              _ptr(qdd), _ptr(tau), _ptr(mask), _ptr(ff), _stream_ptr()))
        first = int(ff.item())
    return {"q": q, "qd": qd, "qdd": qdd, "tau": tau, "feasible": mask, "first_fail": first}


def ik_batch(rot9, trans3, free, want_sols: bool = True, want_status: bool = True,
             workspace: Optional[Workspace] = None):
    """Batched IK (tcmp_ik_batch).  rot9 ``[9][n]``, trans3 ``[3][n]``, free ``[n_free][n]`` or
    ``[n_free]`` (broadcast).  Returns ``(sols [n*n_free][8][7] or None, counts int32, status uint8 or None)``
    with solve index ``pose*n_free + f``."""
    lib = load()
    n = int(rot9.shape[1])
    bcast = int(len(free.shape) == 1)
    n_free = int(free.shape[0])
    fshape = (n_free,) if bcast else (n_free, n)
    if _is_cuda_tensor(rot9):
        torch = _torch()
        dev = rot9.device
        with torch.cuda.device(dev):
            r = _as_dev(rot9, "f64", (9, n), dev)
            t = _as_dev(trans3, "f64", (3, n), dev)
            f = _as_dev(free, "f64", fshape, dev)
            sols = torch.empty((n * n_free, 8, 7), dtype=torch.float64, device=dev) if want_sols else None
            counts = torch.empty((n * n_free,), dtype=torch.int32, device=dev)
            status = torch.empty((n * n_free,), dtype=torch.uint8, device=dev) if want_status else None
            check(lib.tcmp_ik_batch(n, _ptr(r), _ptr(t), _ptr(f), n_free, bcast, _ptr(sols), _ptr(counts),
                                    _ptr(status), _stream_ptr()))
        return sols, counts, status
    ws = workspace or default_workspace()
    r = _as_host(rot9, "f64", (9, n))
    t = _as_host(trans3, "f64", (3, n))
    f = _as_host(free, "f64", fshape)
    sols = np.empty((n * n_free, 8, 7), dtype=np.float64) if want_sols else None
    counts = np.empty((n * n_free,), dtype=np.int32)
    status = np.empty((n * n_free,), dtype=np.uint8) if want_status else None
    with ws.lock:
        check(lib.tcmp_ik_batch_host(ws.handle, n, _nptr(r), _nptr(t), _nptr(f), n_free, bcast, _nptr(sols),
                                     _nptr(counts), _nptr(status)))
    return sols, counts, status


def ik_select(rot9, trans3, free, q_ref, payload_mass: float = 0.0, mode: str = "rne", q_lo=None, q_hi=None,
              payload_threshold: float = PAYLOAD_THRESHOLD_TEST, norm: str = "inf",
              model: Optional[InertialModel] = None):
    """Goal-IK selection (tcmp_ik_select): per pose, the IK solution of the free-joint sweep that is inside the
    joint limits, passes the static torque test ``mode`` and is nearest to ``q_ref`` ([7][n] or [7]).
    Returns (best_q [7][n], best_cost [n] (+inf = none), n_valid int32 [n]); CUDA tensors in -> CUDA tensors out,
    NumPy in -> NumPy out.  Ties keep the first solution in (free value, solver order); a NaN cost ranks after every
    number, so a NaN joint in ``q_ref`` returns the first surviving solution with ``best_cost`` NaN (``n_valid``
    unchanged), and a +-inf joint the first survivor with ``best_cost`` +inf.  With no survivor: zeros, +inf, 0.  A NaN
    limit in ``q_lo`` / ``q_hi`` bounds nothing."""
    torch = _torch()
    lib = load()
    lim = get_limits()
    lo = np.ascontiguousarray(lim["q_lo"] if q_lo is None else q_lo, dtype=np.float64)
    hi = np.ascontiguousarray(lim["q_hi"] if q_hi is None else q_hi, dtype=np.float64)
    host = not _is_cuda_tensor(rot9)
    dev = torch.device("cuda", torch.cuda.current_device()) if host else rot9.device
    n = int(rot9.shape[1])
    bcast = int(len(free.shape) == 1)
    n_free = int(free.shape[0])
    rb = int(len(q_ref.shape) == 1)
    with torch.cuda.device(dev):
        r = _as_dev(rot9, "f64", (9, n), dev)
        t = _as_dev(trans3, "f64", (3, n), dev)
        f = _as_dev(free, "f64", (n_free,) if bcast else (n_free, n), dev)
        ref = _as_dev(q_ref, "f64", (7,) if rb else (7, n), dev)
        best = torch.empty((7, n), dtype=torch.float64, device=dev)
        cost = torch.empty((n,), dtype=torch.float64, device=dev)
        nv = torch.empty((n,), dtype=torch.int32, device=dev)
        check(lib.tcmp_ik_select_model(_mptr(model), n, _ptr(r), _ptr(t), _ptr(f), n_free, bcast, _ptr(ref), rb,
                                       _nptr(lo), _nptr(hi), MODE[mode], float(payload_mass),
                                       float(payload_threshold), int(norm in ("inf", "max")), _ptr(best),
                                       _ptr(cost), _ptr(nv), _stream_ptr()))
    if host:
        return best.cpu().numpy(), cost.cpu().numpy(), nv.cpu().numpy()
    return best, cost, nv


class _Obstacle(ctypes.Structure):   # tcmp_obstacle (include/tcmp.h)
    _fields_ = [("kind", ctypes.c_int32), ("reserved", ctypes.c_int32), ("center", ctypes.c_double * 3),
                ("half", ctypes.c_double * 3)]


class PackedScene:
    """Obstacles + joint limits marshalled once (ctypes array of tcmp_obstacle, contiguous limit arrays) so that
    per-edge calls do not rebuild them (that was half of a 200 us collision call in the planner)."""

    def __init__(self, obstacles, q_lo=None, q_hi=None, payload_radius=0.0):
        self.n = len(obstacles)
        self.obs = pack_obstacles(obstacles)
        self.lo, self.hi = _limits_arrays(q_lo, q_hi)
        self.payload_radius = float(payload_radius)


def pack_obstacles(obstacles):
    """collision.Box / collision.Sphere objects -> ctypes array of tcmp_obstacle."""
    arr = (_Obstacle * max(len(obstacles), 1))()
    for i, ob in enumerate(obstacles):
        if hasattr(ob, "radius"):
            arr[i].kind = 1
            arr[i].half[0] = float(ob.radius)
        else:
            arr[i].kind = 0
            for r in range(3):
                arr[i].half[r] = float(ob.half[r])
        for r in range(3):
            arr[i].center[r] = float(ob.center[r])
    return arr


def _limits_arrays(q_lo, q_hi):
    lim = get_limits()
    lo = np.ascontiguousarray(lim["q_lo"] if q_lo is None else q_lo, dtype=np.float64)
    hi = np.ascontiguousarray(lim["q_hi"] if q_hi is None else q_hi, dtype=np.float64)
    return lo, hi


def collision_batch(q, obstacles, q_lo=None, q_hi=None, payload_radius: float = 0.0):
    """Synthetic-scene collision predicate (tcmp_collision_batch): q ``[7][n]`` -> hit uint8 ``[n]``.
    ``obstacles`` is a list of collision.Box / Sphere or a :class:`PackedScene` (then the other arguments are
    taken from it)."""
    torch = _torch()
    lib = load()
    sc = obstacles if isinstance(obstacles, PackedScene) else PackedScene(obstacles, q_lo, q_hi, payload_radius)
    host = not _is_cuda_tensor(q)
    dev = torch.device("cuda", torch.cuda.current_device()) if host else q.device
    n = int(q.shape[1])
    with torch.cuda.device(dev):
        qt = _as_dev(q, "f64", (7, n), dev)
        hit = torch.empty((n,), dtype=torch.uint8, device=dev)
        check(lib.tcmp_collision_batch(n, _ptr(qt), sc.n, ctypes.addressof(sc.obs), _nptr(sc.lo), _nptr(sc.hi),
                                       sc.payload_radius, _ptr(hit), _stream_ptr()))
    return hit.cpu().numpy() if host else hit


def extend_prefix(q1, q2, resolution, obstacles, payload_mass: float = 0.0, mode: str = "rne", q_lo=None,
                  q_hi=None, payload_radius: float = 0.0, payload_threshold: float = PAYLOAD_THRESHOLD_TEST,
                  model: Optional[InertialModel] = None):
    """Safe-prefix length of every candidate RRT* edge q1 -> q2 (tcmp_extend_prefix): extend steps generated,
    collision-checked and (if collision-free) statically torque-tested on the device.
    q1/q2 ``[7][n_edges]`` -> (n_steps int32 [n_edges], prefix int32 [n_edges])."""
    torch = _torch()
    lib = load()
    sc = obstacles if isinstance(obstacles, PackedScene) else PackedScene(obstacles, q_lo, q_hi, payload_radius)
    res = np.ascontiguousarray(resolution, dtype=np.float64)
    host = not _is_cuda_tensor(q1)
    dev = torch.device("cuda", torch.cuda.current_device()) if host else q1.device
    n = int(q1.shape[1])
    with torch.cuda.device(dev):
        a = _as_dev(q1, "f64", (7, n), dev)
        b = _as_dev(q2, "f64", (7, n), dev)
        ns = torch.empty((n,), dtype=torch.int32, device=dev)
        pre = torch.empty((n,), dtype=torch.int32, device=dev)
        check(lib.tcmp_extend_prefix_model(_mptr(model), MODE[mode], n, _ptr(a), _ptr(b), _nptr(res), sc.n,
                                           ctypes.addressof(sc.obs), _nptr(sc.lo), _nptr(sc.hi), sc.payload_radius,
                                           float(payload_mass), float(payload_threshold), _ptr(ns), _ptr(pre),
                                           _stream_ptr()))
    if host:
        return ns.cpu().numpy(), pre.cpu().numpy()
    return ns, pre


def fk_batch(q):
    """Batched FK (tcmp_fk_batch): q ``[7][n]`` -> (trans3 ``[3][n]``, rot9 ``[9][n]``)."""
    torch = _torch()
    lib = load()
    host = not _is_cuda_tensor(q)
    dev = torch.device("cuda", torch.cuda.current_device()) if host else q.device
    n = int(q.shape[1])
    with torch.cuda.device(dev):
        qt = _as_dev(q, "f64", (7, n), dev)
        trans = torch.empty((3, n), dtype=torch.float64, device=dev)
        rot = torch.empty((9, n), dtype=torch.float64, device=dev)
        check(lib.tcmp_fk_batch(n, _ptr(qt), _ptr(trans), _ptr(rot), _stream_ptr()))
    if host:
        return trans.cpu().numpy(), rot.cpu().numpy()
    return trans, rot


def dynamics_batch(q, qd=None, payload_mass=0.0, mass_matrix: bool = True, coriolis: bool = False,
                   gravity: bool = True, jacobian: bool = False, model: Optional[InertialModel] = None):
    """Joint-space dynamics terms per state (tcmp_dynamics_batch), fp64: q ``[7][n]``, qd ``[7][n]`` (needed for the
    Coriolis matrix), payload_mass scalar or ``[n]`` (a rigid body on the flange iff m > 0; 0 = the arm alone).
    Returns ``{"M": [7][7][n], "C": [7][7][n], "g": [7][n], "J": [6][7][n]}`` with None for the terms not requested;
    M qdd + C qd + g equals the rne torques.  J is the geometric Jacobian [linear; angular] of the grasp-target point
    in the base frame.  CUDA tensors in -> CUDA tensors out, NumPy in -> NumPy out."""
    if not (mass_matrix or coriolis or gravity or jacobian):
        raise ValueError("nothing to compute")
    if coriolis and qd is None:
        raise ValueError("the Coriolis matrix needs qd")
    torch = _torch()
    lib = load()
    host = not _is_cuda_tensor(q)
    dev = torch.device("cuda", torch.cuda.current_device()) if host else q.device
    n = int(q.shape[1])
    scalar, pm = (float(payload_mass), None) if np.ndim(payload_mass) == 0 else (0.0, payload_mass)
    with torch.cuda.device(dev):
        qt = _as_dev(q, "f64", (7, n), dev)
        qdt = _as_dev(qd, "f64", (7, n), dev) if coriolis else None
        pmt = _as_dev(pm, "f64", (n,), dev)
        mk = lambda want, shape: torch.empty(shape, dtype=torch.float64, device=dev) if want else None
        out = {"M": mk(mass_matrix, (7, 7, n)), "C": mk(coriolis, (7, 7, n)), "g": mk(gravity, (7, n)),
               "J": mk(jacobian, (6, 7, n))}
        check(lib.tcmp_dynamics_batch(_mptr(model), n, _ptr(qt), _ptr(qdt), _ptr(pmt), scalar, _ptr(out["M"]),
                                      _ptr(out["C"]), _ptr(out["g"]), _ptr(out["J"]), _stream_ptr()))
    if host:
        return {k: None if v is None else v.cpu().numpy() for k, v in out.items()}
    return out


def forward_dynamics_batch(q, qd=None, tau=None, payload_mass=0.0, mode: str = "rne", qdd: bool = True,
                           minv: bool = False, model: Optional[InertialModel] = None):
    """Forward dynamics per state (tcmp_forward_dynamics_batch), fp64: the joint accelerations
    qdd = M(q)^-1 (tau - h(q, qd)) that the torques tau produce, and the inverse mass matrix M^-1.
    q ``[7][n]``; qd, tau ``[7][n]`` or None (zeros); payload_mass scalar or ``[n]``.  mode "rne": the payload is a
    rigid body on the flange iff m > 0; "dyn": M is the arm alone and the payload a tool-point force m g.  The result
    inverts the torque test: torque_test_batch(q, qd, qdd, m, mode=mode, payload_threshold=0) returns tau.
    Returns ``{"qdd": [7][n], "Minv": [7][7][n]}`` with None for what was not requested.  A non-finite q or mass makes
    the state's outputs NaN, a non-finite qd or tau its qdd (include/tcmp.h).  CUDA tensors in -> CUDA tensors out,
    NumPy in -> NumPy out."""
    if not (qdd or minv):
        raise ValueError("nothing to compute")
    torch = _torch()
    lib = load()
    host = not _is_cuda_tensor(q)
    dev = torch.device("cuda", torch.cuda.current_device()) if host else q.device
    n = int(q.shape[1])
    scalar, pm = (float(payload_mass), None) if np.ndim(payload_mass) == 0 else (0.0, payload_mass)
    with torch.cuda.device(dev):
        qt = _as_dev(q, "f64", (7, n), dev)
        qdt = _as_dev(qd, "f64", (7, n), dev)
        taut = _as_dev(tau, "f64", (7, n), dev)
        pmt = _as_dev(pm, "f64", (n,), dev)
        out = {"qdd": torch.empty((7, n), dtype=torch.float64, device=dev) if qdd else None,
               "Minv": torch.empty((7, 7, n), dtype=torch.float64, device=dev) if minv else None}
        check(lib.tcmp_forward_dynamics_batch(_mptr(model), MODE[mode], n, _ptr(qt), _ptr(qdt), _ptr(taut), _ptr(pmt),
                                              scalar, _ptr(out["qdd"]), _ptr(out["Minv"]), _stream_ptr()))
    if host:
        return {k: None if v is None else v.cpu().numpy() for k, v in out.items()}
    return out


def _interval_outputs(torch, n, dev):
    return (torch.empty((n,), dtype=torch.float64, device=dev), torch.empty((n,), dtype=torch.float64, device=dev),
            torch.empty((n,), dtype=torch.uint8, device=dev))


def payload_interval_batch(q, qd=None, qdd=None, mode: str = "rne", model: Optional[InertialModel] = None):
    """Payload masses each state can carry within the torque limits (tcmp_payload_interval_batch), fp64.
    q/qd/qdd ``[7][n]`` (qd/qdd both or neither; ignored in nov).  Returns ``(m_lo [n], m_hi [n], unloaded_ok uint8
    [n])``: the torque test at an attached mass m passes iff m_lo < m < m_hi, and with no payload attached iff
    unloaded_ok (see :func:`payload_passes`, :func:`max_payload`).  CUDA tensors in -> CUDA tensors out, NumPy in ->
    NumPy out."""
    if (qd is None) != (qdd is None):
        raise ValueError("qd and qdd must both be given or both be None")
    torch = _torch()
    lib = load()
    host = not _is_cuda_tensor(q)
    dev = torch.device("cuda", torch.cuda.current_device()) if host else q.device
    n = int(q.shape[1])
    dynamic = mode != "nov" and qd is not None
    with torch.cuda.device(dev):
        qt = _as_dev(q, "f64", (7, n), dev)
        qdt = _as_dev(qd, "f64", (7, n), dev) if dynamic else None
        qddt = _as_dev(qdd, "f64", (7, n), dev) if dynamic else None
        lo, hi, ok = _interval_outputs(torch, n, dev)
        check(lib.tcmp_payload_interval_batch(_mptr(model), MODE[mode], n, _ptr(qt), _ptr(qdt), _ptr(qddt), _ptr(lo),
                                              _ptr(hi), _ptr(ok), _stream_ptr()))
    if host:
        return lo.cpu().numpy(), hi.cpu().numpy(), ok.cpu().numpy()
    return lo, hi, ok


def edge_payload_interval(qa, qb, n_waypoints: int = 64, mode: str = "rne", static_only: bool = False,
                          model: Optional[InertialModel] = None):
    """Payload masses each RRT* edge qa -> qb can carry at every one of its min-jerk waypoints (the samples of
    :func:`edge_feasibility`), per edge (tcmp_edge_payload_interval).  qa/qb ``[7][n_edges]``.  Returns
    ``(m_lo, m_hi, unloaded_ok)`` as :func:`payload_interval_batch`; edge_feasibility at an attached mass m returns
    n_waypoints iff m_lo < m < m_hi."""
    torch = _torch()
    lib = load()
    host = not _is_cuda_tensor(qa)
    dev = torch.device("cuda", torch.cuda.current_device()) if host else qa.device
    n = int(qa.shape[1])
    with torch.cuda.device(dev):
        a = _as_dev(qa, "f64", (7, n), dev)
        b = _as_dev(qb, "f64", (7, n), dev)
        lo, hi, ok = _interval_outputs(torch, n, dev)
        check(lib.tcmp_edge_payload_interval(_mptr(model), MODE[mode], n, int(n_waypoints), _ptr(a), _ptr(b),
                                             int(static_only), _ptr(lo), _ptr(hi), _ptr(ok), _stream_ptr()))
    if host:
        return lo.cpu().numpy(), hi.cpu().numpy(), ok.cpu().numpy()
    return lo, hi, ok


def traj_payload_interval(coeffs, samples_per_segment: int, mode: str = "rne", model: Optional[InertialModel] = None,
                          device=None):
    """Payload masses a whole piecewise min-jerk trajectory (coefficients ``[n_seg][7][6]``) can carry: the
    intersection over the samples :func:`traj_feasibility` tests.  Returns ``(m_lo, m_hi, unloaded_ok)`` as Python
    float, float, int; traj_feasibility at an attached mass m finds no failure iff m_lo < m < m_hi."""
    torch = _torch()
    if mode == "base":
        return -float("inf"), float("inf"), 1
    s = traj_feasibility(coeffs, samples_per_segment, mode="base", want_tau=False, device=device, model=model)
    lo, hi, ok = payload_interval_batch(s["q"], s["qd"], s["qdd"], mode=mode, model=model)
    if lo.numel() == 0:
        return -float("inf"), float("inf"), 1
    r = torch.stack([lo.max(), hi.min(), ok.min().to(torch.float64)]).cpu().tolist()
    return r[0], r[1], int(r[2])


def _xp(x):
    """torch for tensors, NumPy for everything else (the interval helpers work on either)."""
    import sys
    torch = sys.modules.get("torch")
    return torch if torch is not None and torch.is_tensor(x) else np


def max_payload(m_lo, m_hi, unloaded_ok, mode: str, payload_threshold: float = PAYLOAD_THRESHOLD_TEST):
    """Elementwise: the largest M such that the torque test passes at every mass in [0, M), from the intervals of
    :func:`payload_interval_batch` / :func:`edge_payload_interval` (torch tensors or NumPy arrays).
      rne / nov: masses up to the threshold are not attached, so 0 if the unloaded arm fails, else m_hi when
                 m_lo <= threshold < m_hi and the threshold otherwise;
      dyn:       the tool force applies at every mass: max(m_hi, 0) when unloaded_ok and m_lo <= 0, else 0;
      base:      +inf."""
    xp = _xp(m_lo)
    hi = m_hi if xp is not np else np.asarray(m_hi, dtype=np.float64)
    lo = m_lo if xp is not np else np.asarray(m_lo, dtype=np.float64)
    ok = (unloaded_ok if xp is not np else np.asarray(unloaded_ok)) != 0
    zero = xp.zeros_like(hi)
    if mode == "base":
        return xp.full_like(hi, float("inf"))
    if mode == "dyn":
        return xp.where(ok & (lo <= 0), xp.where(hi > 0, hi, zero), zero)
    t = float(payload_threshold)
    return xp.where(ok, xp.where((lo <= t) & (t < hi), hi, xp.full_like(hi, t)), zero)


def payload_passes(m_lo, m_hi, unloaded_ok, mass, mode: str, payload_threshold: float = PAYLOAD_THRESHOLD_TEST):
    """Elementwise: the torque test's verdict at payload mass ``mass`` (scalar or per element), reproduced from the
    intervals -- m_lo < mass < m_hi where the test attaches the mass (mass > threshold in rne / nov, every mass in dyn),
    unloaded_ok where it does not, always True in base."""
    xp = _xp(m_lo)
    lo = m_lo if xp is not np else np.asarray(m_lo, dtype=np.float64)
    hi = m_hi if xp is not np else np.asarray(m_hi, dtype=np.float64)
    ok = (unloaded_ok if xp is not np else np.asarray(unloaded_ok)) != 0
    if mode == "base":
        return xp.ones_like(ok)
    inside = (lo < mass) & (hi > mass)
    if mode == "dyn":
        return inside
    t = float(payload_threshold)
    if np.ndim(mass) == 0:
        return inside if float(mass) > t else ok
    return xp.where(mass > t, inside, ok)


def fp64_peak(iters: int = 4096) -> float:
    """Measured FP64 FMA throughput of the current device in FLOP/s (tcmp_fp64_peak)."""
    out = ctypes.c_double(0.0)
    check(load().tcmp_fp64_peak(int(iters), ctypes.byref(out), None))
    return float(out.value)


def get_limits():
    tq, lo, hi, vm = (np.empty(7) for _ in range(4))
    check(load().tcmp_get_limits(_nptr(tq), _nptr(lo), _nptr(hi), _nptr(vm)))
    return {"torque": tq, "q_lo": lo, "q_hi": hi, "qd_max": vm}
