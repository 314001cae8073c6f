"""Reference data of the IKFast solver for the IK tests, stored in the repository.

The compiled, unmodified reference solver (ikfast_panda_arm.cpp, built by oracle/Makefile as oracle/_ref) is not part
of this repository.  What the IK tests compare with is stored under tests/golden/ instead, per named input set:

* ``ik_reference.json``: the SHA-256 of the reference's solution COUNTS (int32, solve order pose * n_free + f) and,
  for the one test that asserts bit-for-bit solutions, of the solutions too; plus where the data came from.
* ``ik_reference_sols.npz``: the reference's solutions on a seeded sample of solves (``<name>_idx``,
  ``<name>_sols``), compared with a tolerance, so a last-bit change of the solver does not fail them.

``check(name, counts, sols, ...)`` compares a solver's output with the stored data.  ``ik_batch(name, ...)`` returns
the reference's full output for tests that need every solve (for example to allow mismatches only on flagged
solves): it is computed by the compiled reference when oracle/_ref is present, by the host build of
csrc/ik_core.cuh otherwise, and is accepted only if it matches the stored data.  ``fk_batch`` builds the poses the
tests solve (host build, glibc sin / cos): it agrees with the reference's ComputeFk to 1e-15, not bit for bit, and the
stored data were recorded on exactly these poses.

IK_REFERENCE_RECORD=1 records the data of this run instead of checking it.  It takes the compiled reference when
present; without it, the host build only after it has reproduced the reference's golden set ik_cfg3.npz (counts
exactly, solutions to 1e-9), and the file then says so.
"""
import ctypes
import hashlib
import json
import os
import shutil
import subprocess

import numpy as np

import oracle
from conftest import GOLDEN, ROOT, load_golden

NATIVE = os.path.join(ROOT, "tests", "native")
PINS = os.path.join(GOLDEN, "ik_reference.json")
SOLS = os.path.join(GOLDEN, "ik_reference_sols.npz")
SAMPLE = 16          # solves per input set whose solutions are stored
_dp = ctypes.POINTER(ctypes.c_double)


def build_host_ik(name, defines=()):
    so = os.path.join(NATIVE, name)
    src = os.path.join(NATIVE, "ik_host.cpp")
    core = os.path.join(ROOT, "torque_constrained_motion_planning_b200", "csrc", "ik_core.cuh")
    tab = os.path.join(ROOT, "torque_constrained_motion_planning_b200", "csrc", "sincos_table.inc")
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in (src, core, tab)):
        subprocess.check_call([shutil.which("g++"), "-O2", "-fPIC", "-shared", "-fopenmp", "-ffp-contract=off"] +
                              ["-D" + d for d in defines] + ["-o", so, src])
    return ctypes.CDLL(so)


def wrap_host_ik(L):
    """(rot9 [9][n], trans3 [3][n], free [n_free][n] or [n_free]) -> (sols [n*n_free][8][7], counts, status)."""

    def fn(rot, trans, free, want_sols=True):
        rot, trans, free = (np.ascontiguousarray(a, dtype=np.float64) for a in (rot, trans, free))
        n, nf, b = rot.shape[1], free.shape[0], int(free.ndim == 1)
        sols = np.zeros((n * nf, 8, 7)) if want_sols else None
        c = np.zeros(n * nf, np.int32)
        st = np.zeros(n * nf, np.uint8)
        L.host_ik_batch(ctypes.c_int64(n), rot.ctypes.data_as(_dp), trans.ctypes.data_as(_dp),
                        free.ctypes.data_as(_dp), nf, b, None if sols is None else sols.ctypes.data_as(_dp),
                        c.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
                        st.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)))
        return sols, c, st
    return fn


_lib = None


def _host():
    global _lib
    if _lib is None:
        _lib = build_host_ik("libik_host.so")
    return _lib


def host_ik(rot9, trans3, free, want_sols=True):
    """The host build of csrc/ik_core.cuh: (sols or None, counts, status)."""
    return wrap_host_ik(_host())(rot9, trans3, free, want_sols)


def fk_batch(q):
    """q [7][n] -> (trans [3][n], rot [9][n]): the flange pose of ComputeFk's convention (to 1e-15)."""
    q = np.ascontiguousarray(q, dtype=np.float64)
    n = q.shape[1]
    trans, rot = np.empty((3, n)), np.empty((9, n))
    _host().host_fk_batch(ctypes.c_int64(n), q.ctypes.data_as(_dp), trans.ctypes.data_as(_dp),
                          rot.ctypes.data_as(_dp))
    return trans, rot


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _angle_err(a, b):
    return np.abs((a - b + np.pi) % (2 * np.pi) - np.pi)


_source = None


def _reference(rot9, trans3, free, want_sols=True):
    """The reference solver's output and its name: the compiled original, or the host build once it has reproduced
    the original's golden set."""
    global _source
    if oracle.have_ref():
        sols, counts = oracle.ref_ik_batch(rot9, trans3, free, want_sols=want_sols)
        return sols, counts, "compiled reference IKFast (oracle/_ref)"
    if _source is None:
        g = load_golden("ik_cfg3.npz")
        s, c, _ = host_ik(g["rot"], g["trans"], g["free"])
        valid = np.arange(8)[None, :, None] < c[:, None, None]
        assert np.array_equal(c, g["counts"]) and (_angle_err(s, g["sols"]) * valid).max() < 1e-9, \
            "the host build does not reproduce the reference's golden set: not a reference"
        _source = "host build of csrc/ik_core.cuh, checked against the reference's ik_cfg3.npz"
    sols, counts, _ = host_ik(rot9, trans3, free, want_sols)
    return sols, counts, _source


def _record(name, counts, sols, bitwise):
    pins = json.load(open(PINS)) if os.path.exists(PINS) else {}
    data = dict(np.load(SOLS)) if os.path.exists(SOLS) else {}
    pins[name] = {"counts_sha256": _sha(counts.astype(np.int32))}
    if sols is not None:
        nz = np.nonzero(counts > 0)[0]
        idx = np.sort(np.random.default_rng(0).choice(nz, size=min(SAMPLE, len(nz)), replace=False))
        data[name + "_idx"], data[name + "_sols"] = idx, sols[idx]
        if bitwise:
            pins[name]["sols_sha256"] = _sha(sols)
    with open(PINS, "w") as f:
        json.dump(pins, f, indent=1, sort_keys=True)
        f.write("\n")
    np.savez_compressed(SOLS, **data)


def _record_source(source):
    pins = json.load(open(PINS)) if os.path.exists(PINS) else {}
    if pins.get("_source") != source:
        pins["_source"] = source
        with open(PINS, "w") as f:
            json.dump(pins, f, indent=1, sort_keys=True)
            f.write("\n")


def check(name, counts, sols=None, inputs=None, tol=1e-6, bitwise=False):
    """Assert that `counts` [n_solves] (and `sols` [n_solves][8][7], same order, angles modulo 2 pi within `tol` on
    the stored sample; bit for bit everywhere when `bitwise`) are the reference's on the input set `name`.  `inputs`
    = (rot9, trans3, free) are only used to record."""
    if os.environ.get("IK_REFERENCE_RECORD") == "1":
        rs, rc, source = _reference(*inputs, want_sols=sols is not None)
        _record(name, np.asarray(rc, dtype=np.int32), rs, bitwise)
        _record_source(source)
    _verify(name, counts, sols, tol, bitwise)


def _verify(name, counts, sols, tol, bitwise):
    counts = np.asarray(counts).astype(np.int32)
    pin = json.load(open(PINS))[name]
    assert _sha(counts) == pin["counts_sha256"], "solution counts differ from the reference's on %r" % name
    if sols is not None:
        data = np.load(SOLS)
        idx, want = data[name + "_idx"], data[name + "_sols"]
        valid = np.arange(8)[None, :, None] < counts[idx][:, None, None]
        worst = (_angle_err(np.asarray(sols)[idx], want) * valid).max()
        assert worst <= tol, (name, worst)
        if bitwise:
            assert _sha(np.asarray(sols)) == pin["sols_sha256"], "solutions differ in the last bit on %r" % name


def ik_batch(name, rot9, trans3, free, want_sols=True):
    """The reference's (sols [n*n_free][8][7] or None, counts int32 [n*n_free]) on the input set `name`, checked
    against the stored data; solve index = pose * n_free + f."""
    sols, counts, source = _reference(rot9, trans3, free, want_sols)
    counts = np.asarray(counts, dtype=np.int32)
    if os.environ.get("IK_REFERENCE_RECORD") == "1":
        _record(name, counts, sols, False)
        _record_source(source)
    _verify(name, counts, sols, 1e-12, False)
    return sols, counts
