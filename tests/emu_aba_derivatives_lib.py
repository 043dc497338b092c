"""ctypes binding to the forward-dynamics derivatives' per-state linear algebra compiled for the host
(tests/emu/emu_aba_derivatives.cpp), and the emulated composition of mecano_b200_aba_derivatives: ABA, the inverse-dynamics
derivatives at its qdd and CRBA (each emulated by its own harness), then the L^T D L routine.  Test infrastructure only, like
emu_lib."""
import ctypes
import os
import subprocess

import numpy as np

import emu_lib as el
import emu_rnea_derivatives_lib as erl

_HERE = os.path.dirname(os.path.abspath(__file__))
_EMU = os.path.join(_HERE, "emu")
_CSRC = os.path.join(os.path.dirname(_HERE), "mecano_b200", "csrc")
_OUT = os.path.join(_EMU, "libmecano_emu_aba_derivatives.so")
_DEPS = [os.path.join(_EMU, "emu_aba_derivatives.cpp")] + [os.path.join(_CSRC, f) for f in (
    "flatten.cpp", "flatten.h", "program.h", "spatial.cuh", "ltdl_solve.cuh")] + [os.path.join(os.path.dirname(_HERE), "include", "mecano_b200.h")]
_LIB = None
_dp = ctypes.POINTER(ctypes.c_double)
_ip = ctypes.POINTER(ctypes.c_int)


def build():
    src = [os.path.join(_EMU, "emu_aba_derivatives.cpp"), os.path.join(_CSRC, "flatten.cpp")]
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-x", "c++"] + src + ["-o", _OUT])


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(_OUT) or any(os.path.getmtime(_OUT) < os.path.getmtime(f) for f in _DEPS):
            build()
        _LIB = ctypes.CDLL(_OUT)
    return _LIB


def _d(a):
    return a.ctypes.data_as(_dp)


def _check(rc, err, what):
    if rc != 0:
        raise RuntimeError("%s rc=%d: %s" % (what, rc, err.value.decode()))


def ltdl_tree(tree):
    """(dof [nv], lam [nv]): DoF k of the factor is row dof[k] of the matrices, its DoF parent lam[k] < k (-1 at a root joint)."""
    d, keep, _ = el.tree_desc_c(tree)
    dof, lam = np.zeros(tree.nv, np.int32), np.zeros(tree.nv, np.int32)
    err = ctypes.create_string_buffer(256)
    _check(lib().emu_ltdl_tree(ctypes.byref(d), dof.ctypes.data_as(_ip), lam.ctypes.data_as(_ip), err, 256), err, "emu_ltdl_tree")
    return dof, lam


def factor(tree, M):
    """The factor of M [nv, nv, n] in place of a copy (ltdl_factor): unit L below the diagonal in the factor's DoF order, 1 / D on
    the diagonal, every other entry as it was."""
    d, keep, _ = el.tree_desc_c(tree)
    n = M.shape[2]
    F = np.ascontiguousarray(M, dtype=np.float64).copy()
    err = ctypes.create_string_buffer(256)
    _check(lib().emu_ltdl_factor(ctypes.byref(d), ctypes.c_long(n), ctypes.c_long(n), _d(F), err, 256), err, "emu_ltdl_factor")
    return F


def solve(tree, M, dtau_dq, dtau_dqd):
    """(M^-1, -M^-1 dtau_dq, -M^-1 dtau_dqd), each [nv, nv, n], from the whole routine (ltdl_solve_state) on copies."""
    d, keep, _ = el.tree_desc_c(tree)
    n = M.shape[2]
    Mi, A, B = (np.ascontiguousarray(x, dtype=np.float64).copy() for x in (M, dtau_dq, dtau_dqd))
    err = ctypes.create_string_buffer(256)
    _check(lib().emu_ltdl_solve(ctypes.byref(d), ctypes.c_long(n), ctypes.c_long(n), _d(Mi), _d(A), _d(B), err, 256), err, "emu_ltdl_solve")
    return Mi, A, B


def aba_derivatives(tree, gravity, q, qd, tau, fext=None):
    """(qdd [nv, n], dqdd_dq, dqdd_dqd, minv [nv, nv, n]): the four launches of mecano_b200_aba_derivatives, emulated.  fext: [nb, 6, n]
    in the order of the tree, or None."""
    e = el.Emu(tree, gravity=gravity)
    qdd = e.aba(q, qd, tau, fext)
    _, dq, dqd = erl.rnea_derivatives(tree, gravity, q, qd, qdd, fext)
    minv, A, B = solve(tree, e.crba(q), dq, dqd)
    return qdd, A, B, minv
