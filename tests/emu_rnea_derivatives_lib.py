"""ctypes binding to the inverse-dynamics derivatives' per-state routine compiled for the host (tests/emu/emu_rnea_derivatives.cpp).
Test infrastructure only, like emu_lib."""
import ctypes
import os
import subprocess

import numpy as np

import emu_lib as el

_HERE = os.path.dirname(os.path.abspath(__file__))
_EMU = os.path.join(_HERE, "emu")
_CSRC = os.path.join(os.path.dirname(_HERE), "mecano_b200", "csrc")
_OUT = os.path.join(_EMU, "libmecano_emu_rnea_derivatives.so")
_DEPS = [os.path.join(_EMU, f) for f in ("emu_rnea_derivatives.cpp", "emu.cpp")] + [os.path.join(_CSRC, f) for f in (
    "flatten.cpp", "flatten.h", "program.h", "spatial.cuh", "algorithms.cuh", "jointmath.cuh", "multidof.cuh", "multidof_aba.cuh", "rnea.cuh",
    "aba.cuh", "crba.cuh", "coriolis.cuh", "rnea_derivatives.cuh")] + [os.path.join(os.path.dirname(_HERE), "include", "mecano_b200.h")]
_LIB = None
_dp = ctypes.POINTER(ctypes.c_double)


def build():
    src = [os.path.join(_EMU, "emu_rnea_derivatives.cpp"), os.path.join(_CSRC, "flatten.cpp")]
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-x", "c++"] + src + ["-o", _OUT])


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(_OUT) or any(os.path.getmtime(_OUT) < os.path.getmtime(f) for f in _DEPS):
            build()
        _LIB = ctypes.CDLL(_OUT)
    return _LIB


def _d(a):
    return None if a is None else a.ctypes.data_as(_dp)


def rnea_derivatives(tree, gravity, q, qd, qdd, fext=None):
    """(tau [nv, n], dtau_dq [nv, nv, n], dtau_dqd [nv, nv, n]) of `tree` (a tests.treedesc.TreeDesc), all NaN-prefilled before the
    call.  fext: [nb, 6, n] in the order of the tree (rows of body b = its CoM-frame wrench), or None."""
    d, keep, order = el.tree_desc_c(tree)
    n = q.shape[1]
    nv = tree.nv
    tau = np.full((nv, n), np.nan)
    dq = np.full((nv * nv, n), np.nan)
    dqd = np.full((nv * nv, n), np.nan)
    g = np.ascontiguousarray(gravity, dtype=np.float64)
    q, qd, qdd = (np.ascontiguousarray(x, dtype=np.float64) for x in (q, qd, qdd))
    f = None if fext is None else np.ascontiguousarray(np.asarray(fext)[order].reshape(6 * tree.nb, n), dtype=np.float64)
    err = ctypes.create_string_buffer(256)
    rc = lib().emu_rnea_derivatives(ctypes.byref(d), _d(g), ctypes.c_long(n), ctypes.c_long(n), _d(q), _d(qd), _d(qdd), _d(f), _d(tau), _d(dq),
                                    _d(dqd), err, 256)
    if rc != 0:
        raise RuntimeError("emu_rnea_derivatives rc=%d: %s" % (rc, err.value.decode()))
    return tau, dq.reshape(nv, nv, n), dqd.reshape(nv, nv, n)


def count_flops(tree, q, qd, qdd):
    """Operation counts of one state (the first columns of q, qd, qdd), as emu_lib.Emu.count_flops."""
    d, keep, _ = el.tree_desc_c(tree)
    out = (ctypes.c_long * 5)()
    q1, qd1, qdd1 = (np.ascontiguousarray(x[:, :1], dtype=np.float64) for x in (q, qd, qdd))
    rc = lib().emu_count_flops_rnea_derivatives(ctypes.byref(d), _d(q1), _d(qd1), _d(qdd1), out)
    assert rc == 0
    return dict(zip(("add", "mul", "div", "sincos", "flops"), list(out)))
