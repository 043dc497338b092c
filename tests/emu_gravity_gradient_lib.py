"""ctypes binding to the gravity gradient's per-state routine compiled for the host (tests/emu/emu_gravity_gradient.cpp).  Test
infrastructure only, like emu_lib."""
import ctypes
import os
import subprocess

import numpy as np

import emu_lib as el

_HERE = os.path.dirname(os.path.abspath(__file__))
_EMU = os.path.join(_HERE, "emu")
_CSRC = os.path.join(os.path.dirname(_HERE), "mecano_b200", "csrc")
_OUT = os.path.join(_EMU, "libmecano_emu_gravity_gradient.so")
_DEPS = [os.path.join(_EMU, f) for f in ("emu_gravity_gradient.cpp", "emu.cpp")] + [os.path.join(_CSRC, f) for f in (
    "flatten.cpp", "flatten.h", "program.h", "spatial.cuh", "algorithms.cuh", "jointmath.cuh", "multidof.cuh", "multidof_aba.cuh", "rnea.cuh",
    "aba.cuh", "crba.cuh", "coriolis.cuh", "gravity_gradient.cuh")] + [os.path.join(os.path.dirname(_HERE), "include", "mecano_b200.h")]
_LIB = None
_dp = ctypes.POINTER(ctypes.c_double)


def build():
    src = [os.path.join(_EMU, "emu_gravity_gradient.cpp"), os.path.join(_CSRC, "flatten.cpp")]
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


def gravity_gradient(tree, gravity, q, fext=None):
    """(tau [nv, n], G [nv, nv, n]) of `tree` (a tests.treedesc.TreeDesc), both NaN-prefilled before the call.  fext: [nb, 6, n] in the
    order of the tree (rows of body b = its CoM-frame wrench), or None."""
    d, keep, order = el.tree_desc_c(tree)
    n = q.shape[1]
    tau = np.full((tree.nv, n), np.nan)
    G = np.full((tree.nv * tree.nv, n), np.nan)
    g = np.ascontiguousarray(gravity, dtype=np.float64)
    q = np.ascontiguousarray(q, dtype=np.float64)
    f = None if fext is None else np.ascontiguousarray(np.asarray(fext)[order].reshape(6 * tree.nb, n), dtype=np.float64)
    err = ctypes.create_string_buffer(256)
    rc = lib().emu_gravity_gradient(ctypes.byref(d), _d(g), ctypes.c_long(n), ctypes.c_long(n), _d(q), _d(f), _d(tau), _d(G), err, 256)
    if rc != 0:
        raise RuntimeError("emu_gravity_gradient rc=%d: %s" % (rc, err.value.decode()))
    return tau, G.reshape(tree.nv, tree.nv, n)


def count_flops(tree, q):
    """Operation counts of one state (the first column of q), as emu_lib.Emu.count_flops."""
    d, keep, _ = el.tree_desc_c(tree)
    out = (ctypes.c_long * 5)()
    q1 = np.ascontiguousarray(q[:, :1], dtype=np.float64)
    rc = lib().emu_count_flops_gravity_gradient(ctypes.byref(d), _d(q1), out)
    assert rc == 0
    return dict(zip(("add", "mul", "div", "sincos", "flops"), list(out)))
