"""ctypes binding to the joint-torque regressor's per-state routine compiled for the host (tests/emu/emu_regressor.cpp).  Test
infrastructure only, like emu_lib."""
import ctypes
import os
import subprocess

import numpy as np

import emu_lib as el

_HERE = os.path.dirname(os.path.abspath(__file__))
_EMU = os.path.join(_HERE, "emu")
_CSRC = os.path.join(os.path.dirname(_HERE), "mecano_b200", "csrc")
_OUT = os.path.join(_EMU, "libmecano_emu_regressor.so")
_DEPS = [os.path.join(_EMU, f) for f in ("emu_regressor.cpp", "emu.cpp")] + [os.path.join(_CSRC, f) for f in (
    "flatten.cpp", "flatten.h", "program.h", "spatial.cuh", "algorithms.cuh", "jointmath.cuh", "multidof.cuh", "multidof_aba.cuh", "rnea.cuh",
    "aba.cuh", "crba.cuh", "coriolis.cuh", "regressor.cuh")] + [os.path.join(os.path.dirname(_HERE), "include", "mecano_b200.h")]
_LIB = None
_dp = ctypes.POINTER(ctypes.c_double)


def build():
    src = [os.path.join(_EMU, "emu_regressor.cpp"), os.path.join(_CSRC, "flatten.cpp")]
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-x", "c++"] + src + ["-o", _OUT])


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(_OUT) or any(os.path.getmtime(_OUT) < os.path.getmtime(f) for f in _DEPS):
            build()
        _LIB = ctypes.CDLL(_OUT)
    return _LIB


def _d(a):
    return np.ascontiguousarray(a, dtype=np.float64).ctypes.data_as(_dp)


def regressor(tree, gravity, q, qd, qdd):
    """Y [nv, 10 nb, n] with column blocks in the order of `tree` (a tests.treedesc.TreeDesc), NaN-prefilled before the call.  The C
    description is level ordered, so block w of the routine's output belongs to body order[w] of the tree: the block convention is
    exercised too."""
    d, keep, order = el.tree_desc_c(tree)
    n = q.shape[1]
    Y = np.full((tree.nv * 10 * tree.nb, n), np.nan)
    g = np.ascontiguousarray(gravity, dtype=np.float64)
    q, qd, qdd = (np.ascontiguousarray(a, dtype=np.float64) for a in (q, qd, qdd))
    err = ctypes.create_string_buffer(256)
    rc = lib().emu_joint_torque_regressor(ctypes.byref(d), _d(g), ctypes.c_long(n), ctypes.c_long(n), _d(q), _d(qd), _d(qdd), Y.ctypes.data_as(_dp),
                                          err, 256)
    if rc != 0:
        raise RuntimeError("emu_joint_torque_regressor rc=%d: %s" % (rc, err.value.decode()))
    Yc = Y.reshape(tree.nv, tree.nb, 10, n)
    out = np.empty_like(Yc)
    out[:, order] = Yc
    return out.reshape(tree.nv, 10 * tree.nb, n)


def count_flops(tree, q, qd, qdd):
    """Operation counts of one state (the first column of q, qd, qdd), as emu_lib.Emu.count_flops."""
    d, keep, _ = el.tree_desc_c(tree)
    out = (ctypes.c_long * 5)()
    q1, qd1, qdd1 = (np.ascontiguousarray(a[:, :1], dtype=np.float64) for a in (q, qd, qdd))
    rc = lib().emu_count_flops_regressor(ctypes.byref(d), _d(q1), _d(qd1), _d(qdd1), out)
    assert rc == 0
    return dict(zip(("add", "mul", "div", "sincos", "flops"), list(out)))
