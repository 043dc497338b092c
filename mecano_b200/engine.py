"""Low-level engine: one handle = one flattened tree on one device.  Thin, allocation-free wrapper
over the C ABI for torch CUDA tensors (device entry points) and numpy / pinned arrays (host entry
points).  Buffers are [rows, n_states] float64 with unit stride along states (ld = stride of rows)."""
import ctypes

import numpy as np

from . import _capi
from ._capi import check, lib


def _dev_ptr_ld(t, rows, n, device=None):
    """(pointer, ld) of a torch CUDA tensor [rows, n] float64 with contiguous states (on `device`, if given)."""
    import torch

    if t is None:
        return None, None
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float64):
        raise TypeError("expected a float64 CUDA tensor")
    if device is not None and t.device.index != device:
        raise ValueError("tensor lives on cuda:%s, the engine on cuda:%d" % (t.device.index, device))
    if t.dim() != 2 or t.shape[0] != rows or t.shape[1] != n:
        raise ValueError("expected shape [%d, %d], got %s" % (rows, n, tuple(t.shape)))
    if n > 1 and t.stride(1) != 1:
        raise ValueError("states must be contiguous (stride 1 along dim 1)")
    return t.data_ptr(), (t.stride(0) if rows > 1 else max(n, t.stride(0)))


def _host_ptr_ld(a, rows, n):
    if a is None:
        return None, None
    if not (isinstance(a, np.ndarray) and a.dtype == np.float64):
        raise TypeError("expected a float64 numpy array")
    if a.ndim != 2 or a.shape[0] != rows or a.shape[1] != n:
        raise ValueError("expected shape [%d, %d], got %s" % (rows, n, a.shape))
    if n > 1 and a.strides[1] != 8:
        raise ValueError("states must be contiguous")
    return a.ctypes.data, (a.strides[0] // 8 if rows > 1 else max(n, a.strides[0] // 8))


def _same_ld(lds):
    lds = [l for l in lds if l is not None]
    if any(l != lds[0] for l in lds):
        raise ValueError("all buffers of one call must share the same leading dimension")
    return lds[0]


class Engine:
    def __init__(self, desc, device=0, keepalive=None):
        """desc: _capi.TreeDesc (level-ordered tables)."""
        self._h = ctypes.c_void_p()
        self._keep = keepalive
        rc = lib.mecano_b200_create(ctypes.byref(desc), int(device), ctypes.byref(self._h))
        if rc != 0:
            msg = lib.mecano_b200_last_error(None)
            raise _capi.MecanoB200Error(rc, msg.decode() if msg else "")
        self.device = int(device)
        self.nv = lib.mecano_b200_n_dofs(self._h)
        self.nq = lib.mecano_b200_n_cfg(self._h)
        self.nb = lib.mecano_b200_n_bodies(self._h)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            lib.mecano_b200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_gravity(self, gx, gy, gz):
        check(lib.mecano_b200_set_gravity(self._h, float(gx), float(gy), float(gz)), self._h)

    def set_variant(self, variant):
        """0 = auto (by batch size), 1 = one thread per state, 2 = one warp per state (trees of up to 32 bodies)."""
        check(lib.mecano_b200_set_variant(self._h, int(variant)), self._h)

    def set_precision(self, precision):
        """"fp64" (default) or "fp32": the optional single-precision variant of the plain RNEA / ABA / CRBA calls."""
        check(lib.mecano_b200_set_precision(self._h, {"fp64": 0, "fp32": 1}[precision]), self._h)

    def set_grid_limit(self, algo, max_blocks):
        """Cap the persistent grid of one algorithm (0 = whole device): leaves SMs to kernels running concurrently on other streams."""
        check(lib.mecano_b200_set_grid_limit(self._h, int(algo), int(max_blocks)), self._h)

    def specialize(self, algos=("rnea", "aba", "crba"), force=False):
        """Compile tree-specialised kernels (mecano_b200_specialize): seconds per algorithm, cached on disk.  Algorithms whose
        unrolled code would not fit the instruction caches keep the generic kernel unless force=True."""
        mask = 0x100 if force else 0
        for a in algos:
            mask |= 1 << {"rnea": 0, "aba": 1, "crba": 2}[a] if isinstance(a, str) else 1 << int(a)
        check(lib.mecano_b200_specialize(self._h, mask), self._h)

    def kernel_info(self, algo, n_states=0):
        info = _capi.KernelInfo()
        check(lib.mecano_b200_kernel_info_get(self._h, int(algo), int(n_states), ctypes.byref(info)), self._h)
        return info.as_dict()

    def _dp(self, t, rows, n):
        return _dev_ptr_ld(t, rows, n, self.device)

    def _stream(self):
        """torch's current stream ON THE ENGINE'S DEVICE (not on torch's current device)."""
        import torch

        return torch.cuda.current_stream(self.device).cuda_stream

    # ---- device entry points (asynchronous on torch's current stream)
    def rnea(self, q, qd, qdd, tau, fext=None, flags=0, body_acc=None, joint_wrench=None):
        """body_acc / joint_wrench ([6 * nb, n], optional): the by-products of mecano_b200_rnea_full."""
        n = q.shape[1]
        pq, l0 = self._dp(q, self.nq, n)
        pqd, l1 = self._dp(qd, self.nv, n)
        pqdd, l2 = self._dp(qdd, self.nv, n)
        pt, l3 = self._dp(tau, self.nv, n)
        pf, l4 = self._dp(fext, 6 * self.nb, n)
        if body_acc is None and joint_wrench is None:
            check(lib.mecano_b200_rnea(self._h, n, _same_ld([l0, l1, l2, l3, l4]), pq, pqd, pqdd, pf, pt, flags, self._stream()), self._h)
            return tau
        pa, l5 = self._dp(body_acc, 6 * self.nb, n)
        pw, l6 = self._dp(joint_wrench, 6 * self.nb, n)
        check(lib.mecano_b200_rnea_full(self._h, n, _same_ld([l0, l1, l2, l3, l4, l5, l6]), pq, pqd, pqdd, pf, pt, pa, pw, flags, self._stream()), self._h)
        return tau

    def aba(self, q, qd, tau, qdd, fext=None, flags=0):
        n = q.shape[1]
        pq, l0 = self._dp(q, self.nq, n)
        pqd, l1 = self._dp(qd, self.nv, n)
        pt, l2 = self._dp(tau, self.nv, n)
        pqdd, l3 = self._dp(qdd, self.nv, n)
        pf, l4 = self._dp(fext, 6 * self.nb, n)
        check(lib.mecano_b200_aba(self._h, n, _same_ld([l0, l1, l2, l3, l4]), pq, pqd, pt, pf, pqdd, flags, self._stream()), self._h)
        return qdd

    def set_joint_source_modes(self, accel_source):
        """accel_source: [n_bodies] ints in the order of the tree description (non-zero = ACCELERATION_SOURCE), or None to reset."""
        if accel_source is None:
            check(lib.mecano_b200_set_joint_source_modes(self._h, None), self._h)
            return
        src = np.ascontiguousarray(accel_source, dtype=np.int32)
        if src.shape != (self.nb,):
            raise ValueError("expected %d source modes" % self.nb)
        check(lib.mecano_b200_set_joint_source_modes(self._h, src.ctypes.data), self._h)

    def aba_sources(self, q, qd, tau, qdd_in, qdd, tau_out=None, fext=None):
        n = q.shape[1]
        pq, l0 = self._dp(q, self.nq, n)
        pqd, l1 = self._dp(qd, self.nv, n)
        pt, l2 = self._dp(tau, self.nv, n)
        pi, l3 = self._dp(qdd_in, self.nv, n)
        pqdd, l4 = self._dp(qdd, self.nv, n)
        pto, l5 = self._dp(tau_out, self.nv, n)
        pf, l6 = self._dp(fext, 6 * self.nb, n)
        check(lib.mecano_b200_aba_sources(self._h, n, _same_ld([l0, l1, l2, l3, l4, l5, l6]), pq, pqd, pt, pi, pf, pqdd, pto, self._stream()), self._h)
        return qdd

    def aba_sources_host(self, q, qd, tau, qdd_in, qdd, tau_out=None, fext=None):
        n = q.shape[1]
        pq, l0 = _host_ptr_ld(q, self.nq, n)
        pqd, l1 = _host_ptr_ld(qd, self.nv, n)
        pt, l2 = _host_ptr_ld(tau, self.nv, n)
        pi, l3 = _host_ptr_ld(qdd_in, self.nv, n)
        pqdd, l4 = _host_ptr_ld(qdd, self.nv, n)
        pto, l5 = _host_ptr_ld(tau_out, self.nv, n)
        pf, l6 = _host_ptr_ld(fext, 6 * self.nb, n)
        check(lib.mecano_b200_aba_sources_host(self._h, n, _same_ld([l0, l1, l2, l3, l4, l5, l6]), pq, pqd, pt, pi, pf, pqdd, pto), self._h)
        return qdd

    def packed_size(self):
        """Rows of the packed mass-matrix layout (CRBA_PACKED): unique entries that are not structurally zero."""
        return lib.mecano_b200_crba_packed_size(self._h)

    def packed_index(self):
        """(row, col) int32 arrays: packed row p holds M[row[p], col[p]] (= M[col[p], row[p]])."""
        n = self.packed_size()
        row, col = np.zeros(n, np.int32), np.zeros(n, np.int32)
        check(lib.mecano_b200_crba_packed_index(self._h, row.ctypes.data, col.ctypes.data), self._h)
        return row, col

    def mass_matrix_rows(self, layout):
        return self.packed_size() if (layout & _capi.CRBA_PACKED) else self.nv * self.nv

    def crba(self, q, M, layout=_capi.CRBA_ENTRY_MAJOR):
        """M: [nv*nv, n] (entry-major), [packed_size, n] (packed) or [n, nv*nv] (state-major) float64 CUDA tensor."""
        n = q.shape[1]
        pq, ld = self._dp(q, self.nq, n)
        if not (layout & _capi.CRBA_STATE_MAJOR):
            pm, lm = self._dp(M, self.mass_matrix_rows(layout), n)
            ld = _same_ld([ld, lm])
        else:
            if tuple(M.shape) != (n, self.nv * self.nv) or not M.is_contiguous():
                raise ValueError("state-major mass matrix must be a contiguous [n, nv*nv] tensor")
            pm = M.data_ptr()
        check(lib.mecano_b200_crba(self._h, n, ld, pq, pm, layout, self._stream()), self._h)
        return M

    def coriolis(self, q, qd, M, C):
        """M, C [nv*nv, n] entry-major; torch CUDA tensors or numpy arrays (host path)."""
        n = q.shape[1]
        host = isinstance(q, np.ndarray)
        f = _host_ptr_ld if host else self._dp
        pq, l0 = f(q, self.nq, n)
        pqd, l1 = f(qd, self.nv, n)
        pm, l2 = f(M, self.nv * self.nv, n)
        pc, l3 = f(C, self.nv * self.nv, n)
        ld = _same_ld([l0, l1, l2, l3])
        if host:
            check(lib.mecano_b200_coriolis_host(self._h, n, ld, pq, pqd, pm, pc), self._h)
        else:
            check(lib.mecano_b200_coriolis(self._h, n, ld, pq, pqd, pm, pc, self._stream()), self._h)

    def joint_torque_regressor(self, q, qd, qdd, Y):
        """Y [nv * 10 nb, n] entry-major (mecano_b200_joint_torque_regressor); torch CUDA tensors or numpy arrays (host path)."""
        n = q.shape[1]
        host = isinstance(q, np.ndarray)
        f = _host_ptr_ld if host else self._dp
        pq, l0 = f(q, self.nq, n)
        pqd, l1 = f(qd, self.nv, n)
        pqdd, l2 = f(qdd, self.nv, n)
        py, l3 = f(Y, self.nv * 10 * self.nb, n)
        ld = _same_ld([l0, l1, l2, l3])
        if host:
            check(lib.mecano_b200_joint_torque_regressor_host(self._h, n, ld, pq, pqd, pqdd, py), self._h)
        else:
            check(lib.mecano_b200_joint_torque_regressor(self._h, n, ld, pq, pqd, pqdd, py, self._stream()), self._h)
        return Y

    def gravity_gradient(self, q, tau, G, fext=None):
        """tau [nv, n], G [nv * nv, n] entry-major (mecano_b200_gravity_gradient), fext [6 * nb, n] or None; torch CUDA tensors or
        numpy arrays (host path)."""
        n = q.shape[1]
        host = isinstance(q, np.ndarray)
        f = _host_ptr_ld if host else self._dp
        pq, l0 = f(q, self.nq, n)
        pf, l1 = f(fext, 6 * self.nb, n)
        pt, l2 = f(tau, self.nv, n)
        pg, l3 = f(G, self.nv * self.nv, n)
        ld = _same_ld([l0, l1, l2, l3])
        if host:
            check(lib.mecano_b200_gravity_gradient_host(self._h, n, ld, pq, pf, pt, pg), self._h)
        else:
            check(lib.mecano_b200_gravity_gradient(self._h, n, ld, pq, pf, pt, pg, self._stream()), self._h)
        return G

    def rnea_derivatives(self, q, qd, qdd, tau, dq, dqd, fext=None):
        """tau [nv, n], dq and dqd [nv * nv, n] entry-major (mecano_b200_rnea_derivatives), fext [6 * nb, n] or None; torch CUDA
        tensors or numpy arrays (host path)."""
        n = q.shape[1]
        host = isinstance(q, np.ndarray)
        f = _host_ptr_ld if host else self._dp
        pq, l0 = f(q, self.nq, n)
        pv, l1 = f(qd, self.nv, n)
        pa, l2 = f(qdd, self.nv, n)
        pf, l3 = f(fext, 6 * self.nb, n)
        pt, l4 = f(tau, self.nv, n)
        pdq, l5 = f(dq, self.nv * self.nv, n)
        pdv, l6 = f(dqd, self.nv * self.nv, n)
        ld = _same_ld([l0, l1, l2, l3, l4, l5, l6])
        if host:
            check(lib.mecano_b200_rnea_derivatives_host(self._h, n, ld, pq, pv, pa, pf, pt, pdq, pdv), self._h)
        else:
            check(lib.mecano_b200_rnea_derivatives(self._h, n, ld, pq, pv, pa, pf, pt, pdq, pdv, self._stream()), self._h)
        return dq

    def aba_derivatives(self, q, qd, tau, qdd, dq, dqd, minv, fext=None):
        """qdd [nv, n], dq, dqd and minv [nv * nv, n] entry-major (mecano_b200_aba_derivatives), fext [6 * nb, n] or None; torch CUDA
        tensors or numpy arrays (host path)."""
        n = q.shape[1]
        host = isinstance(q, np.ndarray)
        f = _host_ptr_ld if host else self._dp
        pq, l0 = f(q, self.nq, n)
        pv, l1 = f(qd, self.nv, n)
        pt, l2 = f(tau, self.nv, n)
        pf, l3 = f(fext, 6 * self.nb, n)
        pa, l4 = f(qdd, self.nv, n)
        pdq, l5 = f(dq, self.nv * self.nv, n)
        pdv, l6 = f(dqd, self.nv * self.nv, n)
        pmi, l7 = f(minv, self.nv * self.nv, n)
        ld = _same_ld([l0, l1, l2, l3, l4, l5, l6, l7])
        if host:
            check(lib.mecano_b200_aba_derivatives_host(self._h, n, ld, pq, pv, pt, pf, pa, pdq, pdv, pmi), self._h)
        else:
            check(lib.mecano_b200_aba_derivatives(self._h, n, ld, pq, pv, pt, pf, pa, pdq, pdv, pmi, self._stream()), self._h)
        return dq

    def crba_centroidal(self, q, M, cmm, com, frame=_capi.FRAME_WORLD):
        """M [nv*nv, n] entry-major, cmm [6*nv, n], com [4, n]; torch CUDA tensors or numpy arrays (host path)."""
        n = q.shape[1]
        host = isinstance(q, np.ndarray)
        f = _host_ptr_ld if host else self._dp
        pq, l0 = f(q, self.nq, n)
        pm, l1 = f(M, self.nv * self.nv, n)
        pa, l2 = f(cmm, 6 * self.nv, n)
        pc, l3 = f(com, 4, n)
        ld = _same_ld([l0, l1, l2, l3])
        if host:
            check(lib.mecano_b200_crba_centroidal_host(self._h, n, ld, pq, pm, pa, pc, int(frame)), self._h)
        else:
            check(lib.mecano_b200_crba_centroidal(self._h, n, ld, pq, pm, pa, pc, int(frame), self._stream()), self._h)

    def center_of_mass(self, q, com):
        """com [4, n]: centre of mass in the root frame and total mass per state, without a matrix (the com rows of crba_centroidal)."""
        n = q.shape[1]
        host = isinstance(q, np.ndarray)
        f = _host_ptr_ld if host else self._dp
        pq, l0 = f(q, self.nq, n)
        pc, l1 = f(com, 4, n)
        ld = _same_ld([l0, l1])
        if host:
            check(lib.mecano_b200_center_of_mass_host(self._h, n, ld, pq, pc), self._h)
        else:
            check(lib.mecano_b200_center_of_mass(self._h, n, ld, pq, pc, self._stream()), self._h)

    def centroidal_convective_term(self, q, qd, com, out, frame=_capi.FRAME_WORLD):
        """out [6, n]; com [4, n] as written by crba_centroidal (None allowed for the world frame)."""
        n = q.shape[1]
        host = isinstance(q, np.ndarray)
        f = _host_ptr_ld if host else self._dp
        pq, l0 = f(q, self.nq, n)
        pqd, l1 = f(qd, self.nv, n)
        pc, l2 = f(com, 4, n)
        po, l3 = f(out, 6, n)
        ld = _same_ld([l0, l1, l2, l3])
        if host:
            check(lib.mecano_b200_centroidal_convective_term_host(self._h, n, ld, pq, pqd, pc, po, int(frame)), self._h)
        else:
            check(lib.mecano_b200_centroidal_convective_term(self._h, n, ld, pq, pqd, pc, po, int(frame), self._stream()), self._h)

    def integrate(self, dt, q, qd, qdd):
        """doubleIntegrateFromAcceleration on device matrices, in place."""
        n = q.shape[1]
        pq, l0 = self._dp(q, self.nq, n)
        pqd, l1 = self._dp(qd, self.nv, n)
        pqdd, l2 = self._dp(qdd, self.nv, n)
        check(lib.mecano_b200_integrate(self._h, n, _same_ld([l0, l1, l2]), float(dt), pq, pqd, pqdd, self._stream()), self._h)

    def integrate_host(self, dt, q, qd, qdd):
        n = q.shape[1]
        pq, l0 = _host_ptr_ld(q, self.nq, n)
        pqd, l1 = _host_ptr_ld(qd, self.nv, n)
        pqdd, l2 = _host_ptr_ld(qdd, self.nv, n)
        check(lib.mecano_b200_integrate_host(self._h, n, _same_ld([l0, l1, l2]), float(dt), pq, pqd, pqdd), self._h)

    # ---- host entry points (synchronous; inputs/outputs in host memory, pinned for full speed)
    def rnea_host(self, q, qd, qdd, tau, fext=None, flags=0, body_acc=None, joint_wrench=None):
        n = q.shape[1]
        pq, l0 = _host_ptr_ld(q, self.nq, n)
        pqd, l1 = _host_ptr_ld(qd, self.nv, n)
        pqdd, l2 = _host_ptr_ld(qdd, self.nv, n)
        pt, l3 = _host_ptr_ld(tau, self.nv, n)
        pf, l4 = _host_ptr_ld(fext, 6 * self.nb, n)
        if body_acc is None and joint_wrench is None:
            check(lib.mecano_b200_rnea_host(self._h, n, _same_ld([l0, l1, l2, l3, l4]), pq, pqd, pqdd, pf, pt, flags), self._h)
            return tau
        pa, l5 = _host_ptr_ld(body_acc, 6 * self.nb, n)
        pw, l6 = _host_ptr_ld(joint_wrench, 6 * self.nb, n)
        check(lib.mecano_b200_rnea_full_host(self._h, n, _same_ld([l0, l1, l2, l3, l4, l5, l6]), pq, pqd, pqdd, pf, pt, pa, pw, flags), self._h)
        return tau

    def aba_host(self, q, qd, tau, qdd, fext=None, flags=0):
        n = q.shape[1]
        pq, l0 = _host_ptr_ld(q, self.nq, n)
        pqd, l1 = _host_ptr_ld(qd, self.nv, n)
        pt, l2 = _host_ptr_ld(tau, self.nv, n)
        pqdd, l3 = _host_ptr_ld(qdd, self.nv, n)
        pf, l4 = _host_ptr_ld(fext, 6 * self.nb, n)
        check(lib.mecano_b200_aba_host(self._h, n, _same_ld([l0, l1, l2, l3, l4]), pq, pqd, pt, pf, pqdd, flags), self._h)
        return qdd

    def crba_host(self, q, M, layout=_capi.CRBA_ENTRY_MAJOR):
        n = q.shape[1]
        pq, ld = _host_ptr_ld(q, self.nq, n)
        pm, ld = self._host_mass_matrix(M, layout, n, ld)
        check(lib.mecano_b200_crba_host(self._h, n, ld, pq, pm, layout), self._h)
        return M

    def _host_mass_matrix(self, M, layout, n, ld):
        if M is None:
            return None, ld
        if not (layout & _capi.CRBA_STATE_MAJOR):
            pm, lm = _host_ptr_ld(M, self.mass_matrix_rows(layout), n)
            return pm, _same_ld([ld, lm])
        if M.shape != (n, self.nv * self.nv) or not M.flags.c_contiguous:
            raise ValueError("state-major mass matrix must be a contiguous [n, nv*nv] array")
        return M.ctypes.data, ld

    def _step_args(self, q, qd, qdd_in, tau_in, tau_out, qdd_out, M, layout, fext):
        n = q.shape[1]
        pq, l0 = _host_ptr_ld(q, self.nq, n)
        ptrs = [_host_ptr_ld(a, self.nv, n) for a in (qd, qdd_in, tau_in, tau_out, qdd_out)]
        pf, lf = _host_ptr_ld(fext, 6 * self.nb, n)
        ld = _same_ld([l0, lf] + [l for _, l in ptrs])
        pm, ld = self._host_mass_matrix(M, layout, n, ld)
        (pqd, _), (pqdd, _), (ptin, _), (ptout, _), (pqo, _) = ptrs
        return n, ld, pq, pqd, pqdd, ptin, pf, ptout, pqo, pm

    def step_host(self, q, qd, qdd_in=None, tau_in=None, tau_out=None, qdd_out=None, M=None, layout=_capi.CRBA_ENTRY_MAJOR, fext=None):
        """mecano_b200_step_host: inverse dynamics (qdd_in -> tau_out), forward dynamics (tau_in -> qdd_out) and the mass matrix of
        the same states in one host call; q / qd cross PCIe once.  Any calculator is skipped by leaving its buffers None."""
        n, ld, pq, pqd, pqdd, ptin, pf, ptout, pqo, pm = self._step_args(q, qd, qdd_in, tau_in, tau_out, qdd_out, M, layout, fext)
        check(lib.mecano_b200_step_host(self._h, n, ld, pq, pqd, pqdd, ptin, pf, ptout, pqo, pm, layout), self._h)


class _BorrowedEngine(Engine):
    """View of one handle of a multi-device engine (not owned: never destroyed through this object)."""

    def __init__(self, handle, device):
        self._h = ctypes.c_void_p(handle)
        self._keep = None
        self.device = int(device)
        self.nv = lib.mecano_b200_n_dofs(self._h)
        self.nq = lib.mecano_b200_n_cfg(self._h)
        self.nb = lib.mecano_b200_n_bodies(self._h)

    def close(self):
        self._h = None


class MultiDeviceEngine:
    """mecano_b200_multi_*: one tree on several GPUs of one box behind one host call.  The batch is cut into disjoint contiguous
    slices of the state index, one per listed device (a device may be listed more than once); no collective, results
    bit-identical to the single-device call.  Host (numpy / pinned) matrices only: a device matrix lives on one GPU."""

    def __init__(self, desc, devices, keepalive=None):
        self.devices = [int(d) for d in devices]
        self._m = ctypes.c_void_p()
        self._keep = keepalive
        dev = np.ascontiguousarray(self.devices, dtype=np.int32)
        rc = lib.mecano_b200_multi_create(ctypes.byref(desc), dev.ctypes.data, len(self.devices), ctypes.byref(self._m))
        if rc != 0:
            msg = lib.mecano_b200_last_error(None)
            raise _capi.MecanoB200Error(rc, msg.decode() if msg else "")
        self.lanes = [_BorrowedEngine(lib.mecano_b200_multi_handle(self._m, i), d) for i, d in enumerate(self.devices)]
        self.device = self.devices[0]
        self.nv, self.nq, self.nb = self.lanes[0].nv, self.lanes[0].nq, self.lanes[0].nb

    def close(self):
        if getattr(self, "_m", None) is not None and self._m:
            for lane in self.lanes:
                lane.close()
            lib.mecano_b200_multi_destroy(self._m)
            self._m = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            msg = lib.mecano_b200_multi_last_error(self._m)
            raise _capi.MecanoB200Error(rc, msg.decode() if msg else "")

    def slices(self, n_states):
        """[(start, count)] per listed device for a batch of n_states."""
        out = []
        for i in range(len(self.devices)):
            s, c = ctypes.c_int64(), ctypes.c_int64()
            self._check(lib.mecano_b200_multi_slice(self._m, int(n_states), i, ctypes.byref(s), ctypes.byref(c)))
            out.append((s.value, c.value))
        return out

    # setters that are properties of every handle
    def set_gravity(self, gx, gy, gz):
        self._check(lib.mecano_b200_multi_set_gravity(self._m, float(gx), float(gy), float(gz)))

    def set_variant(self, variant):
        for lane in self.lanes:
            lane.set_variant(variant)

    def set_precision(self, precision):
        for lane in self.lanes:
            lane.set_precision(precision)

    def set_grid_limit(self, algo, max_blocks):
        for lane in self.lanes:
            lane.set_grid_limit(algo, max_blocks)

    def specialize(self, algos=("rnea", "aba", "crba"), force=False):
        for lane in self.lanes:
            lane.specialize(algos, force)

    def kernel_info(self, algo, n_states=0):
        return self.lanes[0].kernel_info(algo, n_states)

    def packed_size(self):
        return self.lanes[0].packed_size()

    def packed_index(self):
        return self.lanes[0].packed_index()

    def mass_matrix_rows(self, layout):
        return self.lanes[0].mass_matrix_rows(layout)

    @staticmethod
    def _no_byproducts(body_acc, joint_wrench):
        if body_acc is not None or joint_wrench is not None:
            raise NotImplementedError("per-body by-products are served per device (use the engine of one device)")

    def rnea_host(self, q, qd, qdd, tau, fext=None, flags=0, body_acc=None, joint_wrench=None):
        self._no_byproducts(body_acc, joint_wrench)
        n = q.shape[1]
        pq, l0 = _host_ptr_ld(q, self.nq, n)
        pqd, l1 = _host_ptr_ld(qd, self.nv, n)
        pqdd, l2 = _host_ptr_ld(qdd, self.nv, n)
        pt, l3 = _host_ptr_ld(tau, self.nv, n)
        pf, l4 = _host_ptr_ld(fext, 6 * self.nb, n)
        self._check(lib.mecano_b200_multi_rnea_host(self._m, n, _same_ld([l0, l1, l2, l3, l4]), pq, pqd, pqdd, pf, pt, flags))
        return tau

    def aba_host(self, q, qd, tau, qdd, fext=None, flags=0):
        n = q.shape[1]
        pq, l0 = _host_ptr_ld(q, self.nq, n)
        pqd, l1 = _host_ptr_ld(qd, self.nv, n)
        pt, l2 = _host_ptr_ld(tau, self.nv, n)
        pqdd, l3 = _host_ptr_ld(qdd, self.nv, n)
        pf, l4 = _host_ptr_ld(fext, 6 * self.nb, n)
        self._check(lib.mecano_b200_multi_aba_host(self._m, n, _same_ld([l0, l1, l2, l3, l4]), pq, pqd, pt, pf, pqdd, flags))
        return qdd

    def crba_host(self, q, M, layout=_capi.CRBA_ENTRY_MAJOR):
        n = q.shape[1]
        pq, ld = _host_ptr_ld(q, self.nq, n)
        pm, ld = Engine._host_mass_matrix(self.lanes[0], M, layout, n, ld)
        self._check(lib.mecano_b200_multi_crba_host(self._m, n, ld, pq, pm, layout))
        return M

    def step_host(self, q, qd, qdd_in=None, tau_in=None, tau_out=None, qdd_out=None, M=None, layout=_capi.CRBA_ENTRY_MAJOR, fext=None):
        n, ld, pq, pqd, pqdd, ptin, pf, ptout, pqo, pm = Engine._step_args(self.lanes[0], q, qd, qdd_in, tau_in, tau_out, qdd_out, M, layout, fext)
        self._check(lib.mecano_b200_multi_step_host(self._m, n, ld, pq, pqd, pqdd, ptin, pf, ptout, pqo, pm, layout))

    def _device_only(self, *a, **k):
        raise TypeError("a multi-device engine takes host (numpy) matrices: a device tensor lives on one GPU")

    rnea = aba = crba = aba_sources = integrate = _device_only

    def _single_device_only(self, *a, **k):
        raise NotImplementedError("this entry point is served per device: build the calculator on one device")

    aba_sources_host = coriolis = crba_centroidal = centroidal_convective_term = center_of_mass = integrate_host = set_joint_source_modes = _single_device_only
    joint_torque_regressor = gravity_gradient = rnea_derivatives = aba_derivatives = _single_device_only


def measure_fp64_peak(device=0):
    v = ctypes.c_double()
    check(lib.mecano_b200_measure_fp64_peak(device, ctypes.byref(v)))
    return v.value


def measure_fp64_sustained(device=0, seconds=1.0):
    """FP64 FMA chain back to back for `seconds`: TFLOP/s over the second half (the board's power management has settled)."""
    v = ctypes.c_double()
    check(lib.mecano_b200_measure_fp64_sustained(device, float(seconds), ctypes.byref(v)))
    return v.value


def measure_hbm_peak(device=0):
    v = ctypes.c_double()
    check(lib.mecano_b200_measure_hbm_peak(device, ctypes.byref(v)))
    return v.value
