"""Exact reference for the analytic derivative kernels (rnea_derivatives.cuh, gravity_gradient.cuh) by complex-step differentiation.

RNEA is real-analytic in q and qd.  Evaluated in complex arithmetic at q + i h t_j, where t_j is the state integrator's tangent for
velocity column j, Im tau / h is the directional derivative d tau / dq e_j to rounding error: no subtraction, so no step-size
trade-off (h = 1e-30 leaves every second-order term below 1e-60).  The recursion is the textbook body-frame RNEA of
featherstone_np (Featherstone, "Rigid Body Dynamics Algorithms", table 5.1), written once more here so that it runs in any dtype
and over a batch axis: it shares no code with the kernels or the C oracle, only featherstone_np.Model's constant per-body tables
(S, I, Xcom).  Everything stays complex-analytic: no abs, norm, maximum or conjugate (quaternions are normalised with
sqrt(sum x^2)).  Test infrastructure only."""
import numpy as np

import featherstone_np as fn

H = 1e-30
NDOF = {fn.REVOLUTE: 1, fn.PRISMATIC: 1, fn.SPHERICAL: 3, fn.PLANAR: 3, fn.SIXDOF: 6}


def _skew(u):
    return np.array([[0.0, -u[2], u[1]], [u[2], 0.0, -u[0]], [-u[1], u[0], 0.0]])


def _cross(a, b):
    """[3, B] x [3, B] (np.cross conjugates nothing either, but this keeps the arithmetic explicit)."""
    return np.stack([a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]])


def _rot_axis(u, a):
    """[3, 3, B]: rotation by the angles a [B] about the unit axis u (Rodrigues)."""
    u = np.asarray(u, dtype=float)
    K = _skew(u / np.sqrt(u @ u))
    return np.eye(3)[:, :, None] + K[:, :, None] * np.sin(a) + (K @ K)[:, :, None] * (1.0 - np.cos(a))


def _rot_quat(x, y, z, s):
    return np.asarray(fn.rot_quat(x, y, z, s))


def joint_pose(t, i, q):
    """(R [3, 3, B], p [3, B]): the child frame of joint i in its parent's frame, p_parent = R p_child + p (featherstone_np.joint_X)."""
    qi = q[t.cfg_off[i]:]
    jt = t.jtype[i]
    B = q.shape[1]
    zero = 0.0 * qi[0]
    if jt == fn.REVOLUTE:
        RJ, tJ = _rot_axis(t.axis[i], qi[0]), np.zeros((3, B), dtype=q.dtype)
    elif jt == fn.PRISMATIC:
        RJ, tJ = np.broadcast_to(np.eye(3)[:, :, None], (3, 3, B)), np.asarray(t.axis[i])[:, None] * qi[0]
    elif jt == fn.SPHERICAL:
        RJ, tJ = _rot_quat(*qi[:4]), np.zeros((3, B), dtype=q.dtype)
    elif jt == fn.PLANAR:  # rotation about y by the pitch, translation in the x-z plane
        RJ, tJ = _rot_axis([0.0, 1.0, 0.0], qi[0]), np.stack([qi[1], zero, qi[2]])
    else:
        RJ, tJ = _rot_quat(*qi[:4]), qi[4:7]
    R = np.einsum("ij,jkb->ikb", t.off_R[i], RJ)
    p = np.einsum("ij,jb->ib", t.off_R[i], tJ) + np.asarray(t.off_p[i])[:, None]
    return R, p


def _xm(R, p, v):
    """X v for the motion transform X of the pose (R, p): (E w, E (l - p x w)) with E = R^T."""
    w, l = v[:3], v[3:]
    return np.concatenate([np.einsum("jib,jb->ib", R, w), np.einsum("jib,jb->ib", R, l - _cross(p, w))])


def _xf(R, p, f):
    """X^T f for a force f = (n, f) in child coordinates: (R n + p x (R f), R f)."""
    n, fl = np.einsum("ijb,jb->ib", R, f[:3]), np.einsum("ijb,jb->ib", R, f[3:])
    return np.concatenate([n + _cross(p, fl), fl])


def _crm(v, u):
    """v x u (motion): (w x uw, w x ul + vl x uw)."""
    w, l = v[:3], v[3:]
    return np.concatenate([_cross(w, u[:3]), _cross(w, u[3:]) + _cross(l, u[:3])])


def _crf(v, f):
    """v x* f (force): (w x n + vl x f, w x f)."""
    w, l = v[:3], v[3:]
    return np.concatenate([_cross(w, f[:3]) + _cross(l, f[3:]), _cross(w, f[3:])])


def rnea(m, q, qd, qdd, gravity, fext=None):
    """tau [nv, B] of RNEA over a batch, in the dtype of the inputs.  m: featherstone_np.Model; q [nq, B], qd and qdd [nv, B];
    fext: [nb, 6, B] wrenches in each body's centre-of-mass frame, or None."""
    t = m.t
    B = q.shape[1]
    dt = np.result_type(q, qd, qdd)
    a0 = np.zeros((6, B), dtype=dt)
    a0[3:] = -np.asarray(gravity, dtype=float)[:, None]
    pose, v, a, f = [None] * t.nb, [None] * t.nb, [None] * t.nb, [None] * t.nb
    for i in range(t.nb):
        p, d, nd = t.parent[i], t.dof_off[i], m._nd(i)
        R, pp = pose[i] = joint_pose(t, i, q)
        vJ = m.S[i] @ qd[d:d + nd]
        v[i] = (_xm(R, pp, v[p]) if p >= 0 else 0.0) + vJ
        a[i] = _xm(R, pp, a[p] if p >= 0 else a0) + m.S[i] @ qdd[d:d + nd] + _crm(v[i], vJ)
        f[i] = m.I[i] @ a[i] + _crf(v[i], m.I[i] @ v[i])
        if fext is not None:
            f[i] = f[i] - m.Xcom[i].T @ fext[i]
    tau = np.zeros((t.nv, B), dtype=dt)
    for i in range(t.nb - 1, -1, -1):
        d, nd = t.dof_off[i], m._nd(i)
        tau[d:d + nd] = m.S[i].T @ f[i]
        if t.parent[i] >= 0:
            f[t.parent[i]] = f[t.parent[i]] + _xf(*pose[i], f[i])
    return tau


def _qmul(a, b):
    """Hamilton product of quaternions stored (x, y, z, s)."""
    ax, ay, az, as_ = a
    bx, by, bz, bs = b
    return np.stack([as_ * bx + ax * bs + ay * bz - az * by, as_ * by - ax * bz + ay * bs + az * bx,
                     as_ * bz + ax * by - ay * bx + az * bs, as_ * bs - ax * bx - ay * by - az * bz])


def tangent(t, q, j):
    """[nq, B]: dq/dt of the state integrator's step (mo_integrate, mecano_b200_integrate) at dt = 0 with qd = e_j, qdd = 0.  Its
    second-order terms do not enter the first derivative."""
    B = q.shape[1]
    dq = np.zeros((t.nq, B), dtype=q.dtype)
    for i in range(t.nb):
        c, d, jt = t.cfg_off[i], t.dof_off[i], t.jtype[i]
        if not d <= j < d + NDOF[jt]:
            continue
        k = j - d
        if jt in (fn.REVOLUTE, fn.PRISMATIC):
            dq[c] = 1.0
        elif jt == fn.PLANAR:  # (pitch rate, body-frame x and z velocities) -> (pitch, x, z) of the parent frame
            th, e = q[c], np.eye(3)[k]
            dq[c] = e[0]
            dq[c + 1] = np.cos(th) * e[1] + np.sin(th) * e[2]
            dq[c + 2] = -np.sin(th) * e[1] + np.cos(th) * e[2]
        elif k < 3:  # spherical, or the angular part of a six-DoF joint: body-frame angular velocity
            w = np.zeros((4, 1))
            w[k] = 1.0
            dq[c:c + 4] = 0.5 * _qmul(q[c:c + 4], w)
        else:  # six-DoF linear velocity in the body frame, position in the parent frame
            dq[c + 4:c + 7] = _rot_quat(*q[c:c + 4])[:, k - 3]
        break
    return dq


def derivatives(t, g, q, qd, qdd, fext=None, h=H):
    """(tau [nv, n], d tau / dq [nv, nv, n], d tau / dqd [nv, nv, n]) by complex steps: all 2 nv + 1 evaluations of all n states in
    one batch.  Column j of d tau / dq is the derivative along tangent(t, q, j).  The gravity gradient G is d tau / dq at
    qd = qdd = 0."""
    m = fn.Model(t)
    nv, n = t.nv, q.shape[1]
    k = 2 * nv + 1
    Q = np.repeat(q[:, None, :], k, axis=1).astype(complex)
    V = np.repeat(qd[:, None, :], k, axis=1).astype(complex)
    for j in range(nv):
        Q[:, 1 + j] += 1j * h * tangent(t, q, j)
        V[j, 1 + nv + j] += 1j * h
    A = np.repeat(qdd[:, None, :], k, axis=1).astype(complex)
    F = None if fext is None else np.repeat(np.asarray(fext)[:, :, None, :], k, axis=2).reshape(t.nb, 6, k * n)
    tau = rnea(m, Q.reshape(t.nq, k * n), V.reshape(nv, k * n), A.reshape(nv, k * n), g, F).reshape(nv, k, n)
    return tau[:, 0].real.copy(), tau[:, 1:1 + nv].imag / h, tau[:, 1 + nv:].imag / h
