"""Forward-dynamics derivatives (mecano_b200_aba_derivatives, ForwardDynamicsDerivativesCalculator): qdd(q, qd, tau) of ABA with
d qdd / dq (column j along the step the state integrator takes with qd = e_j), d qdd / dqd and M^-1 = d qdd / d tau.  The call
composes ABA, the inverse-dynamics derivatives and CRBA with one new routine, the tree-sparse L^T D L factor and solve
(mecano_b200/csrc/ltdl_solve.cuh).

CPU tests run that routine compiled for the host (tests/emu/emu_aba_derivatives.cpp), alone and composed with the emulated ABA,
inverse-dynamics derivatives and CRBA.  The exact reference is complex-step differentiation of forward dynamics built from the
independent complex RNEA of complex_step.py: M from RNEA columns, the bias from RNEA at zero acceleration, solved in complex
arithmetic at q + i h t_j.  GPU tests run the sm_100a kernels.

The host entry point is compared with the device entry point across chunks in a child process (this file run as a script), since
the staging budget (MECANO_B200_HOST_CHUNK_MB) is read once per process."""
import os
import subprocess
import sys

import numpy as np
import pytest

import complex_step as cs
import emu_aba_derivatives_lib as eal
import emu_gravity_gradient_lib as egl
import emu_lib as el
import featherstone_np as fn
import oracle_lib as ol
import treedesc as td
from test_emulation import trees
from test_gravity_gradient import engine_of, planar_chain, rel, welded_systems

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
EPS = 1e-5
EXACT_TOL = 1e-10  # against the complex-step reference, relative to the largest entry of the matrix
FD_TOL = 1e-6      # against central differences, per state, relative to max(1, max |D|)


def fd_ok(D, Dfd):
    """[nv, nv, n] each: the finite-difference error, state by state, relative to max(1, max |D|) of the state."""
    scale = np.maximum(1.0, np.abs(D).max(axis=(0, 1)))
    return float(np.max(np.abs(D - Dfd).max(axis=(0, 1)) / scale))


def case(idx, n=3):
    rng = np.random.default_rng(2300 + idx)
    t = trees(rng)[idx]
    g = (rng.uniform(-1, 1), rng.uniform(-1, 1), -rng.uniform(1, 10))
    q, qd, _, tau = td.random_states(rng, t, n)
    fext = rng.uniform(-1, 1, size=(t.nb, 6, n))
    return t, g, q, qd, tau, fext


def exact_reference(t, g, q, qd, tau, fext=None, h=cs.H):
    """(qdd [nv, n], dqdd_dq, dqdd_dqd, minv [nv, nv, n]) by complex steps through forward dynamics qdd = M^-1 (tau - c): at each of the
    2 nv + 1 points (the state, q + i h t_j, qd + i h e_j) M is formed from nv RNEA columns (no velocity, gravity or wrench) and the
    bias c from RNEA at zero acceleration, all in one complex batch, then solved in complex arithmetic; Im qdd / h is the column."""
    m = fn.Model(t)
    nv, nq, n = t.nv, t.nq, q.shape[1]
    P = 2 * nv + 1
    Q = np.repeat(q[:, None, :], P, axis=1).astype(complex)
    V = np.repeat(qd[:, None, :], P, axis=1).astype(complex)
    for j in range(nv):
        Q[:, 1 + j] += 1j * h * cs.tangent(t, q, j)
        V[j, 1 + nv + j] += 1j * h
    Q, V = Q.reshape(nq, P * n), V.reshape(nv, P * n)
    Qm = np.repeat(Q[:, None, :], nv, axis=1).reshape(nq, nv * P * n)
    E = np.repeat(np.eye(nv)[:, :, None], P * n, axis=2).reshape(nv, nv * P * n)
    M = cs.rnea(m, Qm, np.zeros((nv, nv * P * n), complex), E.astype(complex), (0.0, 0.0, 0.0)).reshape(nv, nv, P * n)
    F = None if fext is None else np.repeat(np.asarray(fext)[:, :, None, :], P, axis=2).reshape(t.nb, 6, P * n)
    c = cs.rnea(m, Q, V, np.zeros((nv, P * n), complex), g, F)
    rhs = np.repeat(tau[:, None, :], P, axis=1).reshape(nv, P * n) - c
    qdd = np.linalg.solve(M.transpose(2, 0, 1), rhs.T[:, :, None])[:, :, 0].T.reshape(nv, P, n)
    minv = np.linalg.inv(M.reshape(nv, nv, P, n)[:, :, 0].real.transpose(2, 0, 1)).transpose(1, 2, 0)
    return qdd[:, 0].real.copy(), qdd[:, 1:1 + nv].imag / h, qdd[:, 1 + nv:].imag / h, minv


def oracle_central_differences(t, g, q, qd, tau, fext=None):
    """(qdd, dqdd_dq, dqdd_dqd, minv) from the C oracle's aba_batch: at q moved by integrate_batch with dt = +-EPS, qd = e_j, qdd = 0;
    at qd +- EPS e_j; and at tau +- e_j (ABA is linear in tau, so that difference is exact to rounding)."""
    o = ol.Oracle(t, gravity=g)
    n, nv = q.shape[1], t.nv
    z = np.zeros((nv, n))
    f = None if fext is None else np.ascontiguousarray(np.asarray(fext).reshape(6 * t.nb, n))
    dq, dqd, mi = (np.zeros((nv, nv, n)) for _ in range(3))
    for j in range(nv):
        e = np.zeros((nv, n))
        e[j] = 1.0
        qp, _, _ = o.integrate_batch(EPS, q, e, z)
        qm, _, _ = o.integrate_batch(-EPS, q, e, z)
        dq[:, j] = (o.aba_batch(qp, qd, tau, f) - o.aba_batch(qm, qd, tau, f)) / (2 * EPS)
        dqd[:, j] = (o.aba_batch(q, qd + EPS * e, tau, f) - o.aba_batch(q, qd - EPS * e, tau, f)) / (2 * EPS)
        mi[:, j] = (o.aba_batch(q, qd, tau + e, f) - o.aba_batch(q, qd, tau - e, f)) / 2.0
    return o.aba_batch(q, qd, tau, f), dq, dqd, mi


def ancestors_or_self(lam):
    """Boolean [nv, nv] in the factor's DoF order: entry (k, i) is set when i is k or one of its DoF ancestors."""
    nv = len(lam)
    A = np.zeros((nv, nv), bool)
    for k in range(nv):
        i = k
        while i >= 0:
            A[k, i] = True
            i = lam[i]
    return A


# ---------------------------------------------------------------------------------------------------------------- CPU


@pytest.mark.parametrize("idx", range(16))
def test_dof_tree_is_a_preorder(idx):
    t = case(idx)[0]
    dof, lam = eal.ltdl_tree(t)
    assert sorted(dof) == list(range(t.nv))
    assert all(lam[k] < k for k in range(t.nv))
    assert (lam < 0).sum() == sum(1 for b in range(t.nb) if t.parent[b] < 0), "one DoF tree root per root joint"


@pytest.mark.parametrize("idx", range(16))
def test_factor_reproduces_the_mass_matrix_and_touches_nothing_else(idx):
    """L^T D L = M to 1e-12, and no entry outside M's lower pattern (in the factor's DoF order) changes."""
    t, g, q, qd, tau, fext = case(idx)
    M = el.Emu(t, gravity=g).crba(q)
    F = eal.factor(t, M)
    dof, lam = eal.ltdl_tree(t)
    pat = ancestors_or_self(lam)
    Fp, Mp = F[dof][:, dof], M[dof][:, dof]
    assert np.array_equal(Fp[~pat], Mp[~pat]), "entries outside the pattern must be left as they were"
    for s in range(q.shape[1]):
        L = np.where(pat & ~np.eye(t.nv, dtype=bool), Fp[:, :, s], 0.0) + np.eye(t.nv)
        D = 1.0 / np.diag(Fp[:, :, s])
        assert rel(L.T @ np.diag(D) @ L, Mp[:, :, s]) < 1e-12


@pytest.mark.parametrize("idx", range(16))
def test_solve_against_numpy(idx):
    """The routine on M and two random right-hand-side matrices against numpy.linalg.solve on dense M (bound: cond(M) times the
    rounding unit); M^-1 M = I and M^-1 symmetric to rounding; every entry written."""
    t, g, q, qd, tau, fext = case(idx)
    n, nv = q.shape[1], t.nv
    M = el.Emu(t, gravity=g).crba(q)
    rng = np.random.default_rng(idx)
    X, Y = rng.uniform(-1, 1, size=(nv, nv, n)), rng.uniform(-1, 1, size=(nv, nv, n))
    Mi, A, B = eal.solve(t, M, X, Y)
    assert not (np.isnan(Mi).any() or np.isnan(A).any() or np.isnan(B).any())
    for s in range(n):
        Ms = M[:, :, s]
        bound = 1e-15 * np.linalg.cond(Ms) * 8
        assert rel(A[:, :, s], -np.linalg.solve(Ms, X[:, :, s])) < bound
        assert rel(B[:, :, s], -np.linalg.solve(Ms, Y[:, :, s])) < bound
        assert np.max(np.abs(Mi[:, :, s] @ Ms - np.eye(nv))) < bound
        assert np.max(np.abs(Mi[:, :, s] - Mi[:, :, s].T)) <= 1e-14 * np.max(np.abs(Mi[:, :, s]))


@pytest.mark.parametrize("with_fext", [False, True])
@pytest.mark.parametrize("idx", range(16))
def test_emulated_composition_against_exact_and_central_differences(idx, with_fext):
    """All five joint types, floating bases, a 100-body tree, random gravity and state, with and without external wrenches: the
    emulated four launches against the complex-step reference (1e-10) and against central differences of the oracle's ABA
    through its integrator (1e-6); qdd against the oracle's ABA."""
    t, g, q, qd, tau, fext = case(idx)
    f = fext if with_fext else None
    qdd, dq, dqd, minv = eal.aba_derivatives(t, g, q, qd, tau, f)
    for x in (qdd, dq, dqd, minv):
        assert not np.isnan(x).any(), "every entry must be written"
    x_qdd, x_dq, x_dqd, x_minv = exact_reference(t, g, q, qd, tau, f)
    assert rel(qdd, x_qdd) < 1e-11
    assert rel(dq, x_dq) < EXACT_TOL
    assert rel(dqd, x_dqd) < EXACT_TOL
    assert rel(minv, x_minv) < EXACT_TOL
    o_qdd, o_dq, o_dqd, o_minv = oracle_central_differences(t, g, q, qd, tau, f)
    assert rel(qdd, o_qdd) < 1e-11
    assert fd_ok(dq, o_dq) < FD_TOL
    assert fd_ok(dqd, o_dqd) < FD_TOL
    assert fd_ok(minv, o_minv) < 1e-11


@pytest.mark.parametrize("idx", range(16))
def test_emulated_identities_at_rest(idx):
    """At qd = 0, d qdd / dqd = 0; with tau = the gravity torques there, qdd = 0 (to rounding) and d qdd / dq = -M^-1 G with the
    gravity gradient's G."""
    t, g, q, _, _, fext = case(idx)
    z = np.zeros((t.nv, q.shape[1]))
    tau_g, G = egl.gravity_gradient(t, g, q)
    qdd, dq, dqd, minv = eal.aba_derivatives(t, g, q, z, tau_g)
    assert np.all(dqd == 0.0)
    assert np.max(np.abs(qdd)) < 1e-10 * max(1.0, np.max(np.abs(tau_g)))
    assert rel(dq, -np.einsum("ijs,jks->iks", minv, G)) < 1e-10


def test_planar_two_link_arm_closed_form():
    """qdd = M^-1 (tau - c - g) of the two-link arm, and its partials -M^-1 d(tau_ID)/dx with the closed-form d tau / dq, d tau / dqd at
    that qdd (h = m2 l1 l2c sin q2)."""
    m1, m2, l1, l1c, l2c, g0 = 1.3, 0.8, 0.9, 0.4, 0.35, 9.81
    Izz = 0.03
    t = planar_chain([l1], [l1c, l2c], [m1, m2])
    rng = np.random.default_rng(4)
    n = 17
    q, qd, tau = (rng.uniform(-np.pi, np.pi, size=(2, n)) for _ in range(3))
    qdd, dq, dqd, minv = eal.aba_derivatives(t, (0.0, -g0, 0.0), q, qd, tau)
    s1, c1, s2, c2 = np.sin(q[0]), np.cos(q[0]), np.sin(q[1]), np.cos(q[1])
    s12, c12 = np.sin(q[0] + q[1]), np.cos(q[0] + q[1])
    k = m2 * l1 * l2c
    h = k * s2
    M11 = 2 * Izz + m1 * l1c ** 2 + m2 * (l1 ** 2 + l2c ** 2) + 2 * k * c2
    M12 = Izz + m2 * l2c ** 2 + k * c2
    M22 = np.full(n, Izz + m2 * l2c ** 2)
    det = M11 * M22 - M12 ** 2
    Mi = np.array([[M22, -M12], [-M12, M11]]) / det
    grav = g0 * np.array([m1 * l1c * c1 + m2 * (l1 * c1 + l2c * c12), m2 * l2c * c12])
    bias = np.array([-h * (2 * qd[0] * qd[1] + qd[1] ** 2), h * qd[0] ** 2]) + grav
    a = np.einsum("ijs,js->is", Mi, tau - bias)
    dg1 = -g0 * m2 * l2c * s12
    dtau_dq = np.array([
        [-g0 * (m1 * l1c * s1 + m2 * (l1 * s1 + l2c * s12)), -2 * k * s2 * a[0] - k * s2 * a[1] - k * c2 * (2 * qd[0] * qd[1] + qd[1] ** 2) + dg1],
        [dg1, -k * s2 * a[0] + k * c2 * qd[0] ** 2 + dg1]])
    dtau_dqd = np.array([[-2 * h * qd[1], -2 * h * (qd[0] + qd[1])], [2 * h * qd[0], np.zeros(n)]])
    assert rel(qdd, a) < 1e-13
    assert rel(minv, Mi) < 1e-13
    assert rel(dq, -np.einsum("ijs,jks->iks", Mi, dtau_dq)) < 1e-12
    assert rel(dqd, -np.einsum("ijs,jks->iks", Mi, dtau_dqd)) < 1e-12


def test_null_handle_is_refused():
    from mecano_b200 import _capi

    lib = _capi.lib
    assert lib.mecano_b200_aba_derivatives(None, 1, 1, *([None] * 8), None) == -1
    assert lib.mecano_b200_aba_derivatives_host(None, 1, 1, *([None] * 8)) == -1


def test_cpp_host_mirror_links_the_forward_derivatives(tmp_path):
    src = tmp_path / "fd.cpp"
    src.write_text('#include "%s"\nint main() { auto a = &mecano::ForwardDynamicsDerivativesCalculator::compute; return a ? 0 : 1; }\n'
                   % os.path.join(ROOT, "mecano_b200", "csrc", "host", "calculators.hpp"))
    exe = str(tmp_path / "fd")
    libdir = os.path.join(ROOT, "mecano_b200")
    subprocess.check_call(["g++", "-std=c++17", "-Wall", str(src), "-o", exe, "-L" + libdir, "-lmecano_b200", "-Wl,-rpath," + libdir])


# ---------------------------------------------------------------------------------------------------------------- GPU


@pytest.fixture(scope="module")
def torch_dev():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device; the product has no CPU fallback"
    return torch, torch.device("cuda:0")


@pytest.mark.gpu
@pytest.mark.parametrize("idx", range(16))
def test_device_and_host_entry_points_match_the_emulated_composition(torch_dev, idx):
    """ld = n + 11 with NaN padding that must stay NaN; qdd bit-identical to mecano_b200_aba; both entry points bit-identical to
    each other and within 1e-12 of the emulated composition."""
    torch, dev = torch_dev
    t, g, q, qd, tau, fext = case(idx, n=37)
    e, order = engine_of(t, g)
    n, ld = q.shape[1], q.shape[1] + 11
    nv = t.nv
    pad = lambda a: np.ascontiguousarray(np.pad(a, ((0, 0), (0, ld - n))))  # noqa: E731
    hq, hv, ht = pad(q), pad(qd), pad(tau)
    tq, tv, tt = (torch.from_numpy(x).to(dev)[:, :n] for x in (hq, hv, ht))
    for f in (None, fext):
        hf = None if f is None else pad(f[order].reshape(6 * t.nb, n))
        hout = [np.full((rows, ld), np.nan) for rows in (nv, nv * nv, nv * nv, nv * nv)]
        e.aba_derivatives(hq[:, :n], hv[:, :n], ht[:, :n], *[x[:, :n] for x in hout], fext=None if hf is None else hf[:, :n])
        tf = None if hf is None else torch.from_numpy(hf).to(dev)[:, :n]
        dout = [torch.full((rows, ld), float("nan"), dtype=torch.float64, device=dev) for rows in (nv, nv * nv, nv * nv, nv * nv)]
        e.aba_derivatives(tq, tv, tt, *[x[:, :n] for x in dout], fext=tf)
        qdd_aba = torch.full((nv, ld), float("nan"), dtype=torch.float64, device=dev)
        e.aba(tq, tv, tt, qdd_aba[:, :n], fext=tf)
        emu = eal.aba_derivatives(t, g, q, qd, tau, f)
        assert torch.equal(dout[0][:, :n], qdd_aba[:, :n]), "qdd must be what mecano_b200_aba computes"
        for h_, d_, em in zip(hout, dout, emu):
            d_ = d_.cpu().numpy()
            assert np.array_equal(d_, h_, equal_nan=True), "device and host must agree bit for bit"
            assert np.isnan(d_[:, n:]).all(), "nothing written beyond n"
            assert not np.isnan(d_[:, :n]).any(), "every entry written"
            assert rel(d_[:, :n].reshape(em.shape), em) < 1e-12


@pytest.mark.gpu
def test_h37_2e18_states_against_device_central_differences(torch_dev):
    """2^18 humanoid states: every column of the three matrices against central differences of mecano_b200_aba on the device
    (through mecano_b200_integrate for d qdd / dq; at tau +- e_j, exact for ABA's linearity, for M^-1)."""
    torch, dev = torch_dev
    rng = np.random.default_rng(38)
    t = td.humanoid(rng, 2)
    g = (0.3, -0.2, -9.81)
    n = 1 << 18
    nv = t.nv
    assert (t.nb, nv, t.nq) == (32, 37, 38)
    q, qd, _, tau = (torch.from_numpy(x).to(dev) for x in td.random_states(rng, t, n))
    e, _ = engine_of(t, g)
    new = lambda rows: torch.empty((rows, n), dtype=torch.float64, device=dev)  # noqa: E731
    qdd, dq, dqd, minv = new(nv), new(nv * nv), new(nv * nv), new(nv * nv)
    e.aba_derivatives(q, qd, tau, qdd, dq, dqd, minv)
    tp, tm = new(nv), new(nv)
    zero = torch.zeros((nv, n), dtype=torch.float64, device=dev)
    worst = {}
    for D, wrt, step in ((dq.view(nv, nv, n), "q", EPS), (dqd.view(nv, nv, n), "qd", EPS), (minv.view(nv, nv, n), "tau", 1.0)):
        scale = D.abs().amax(dim=(0, 1)).clamp(min=1.0)
        for j in range(nv):
            for dt, out in ((step, tp), (-step, tm)):
                if wrt == "q":
                    qj, vj = q.clone(), zero.clone()
                    vj[j] = 1.0
                    e.integrate(dt, qj, vj, zero.clone())
                    e.aba(qj, qd, tau, out)
                elif wrt == "qd":
                    vj = qd.clone()
                    vj[j] += dt
                    e.aba(q, vj, tau, out)
                else:
                    tj = tau.clone()
                    tj[j] += dt
                    e.aba(q, qd, tj, out)
            err = ((D[:, j] - (tp - tm) / (2 * step)).abs().amax(dim=0) / scale).max().item()
            worst[wrt] = max(worst.get(wrt, 0.0), err)
    print("worst central-difference error", worst)
    assert worst["q"] < FD_TOL and worst["qd"] < FD_TOL, worst
    assert worst["tau"] < 1e-11, worst


@pytest.mark.gpu
def test_calculator_on_systems_with_fixed_and_ignored_joints(torch_dev):
    """Against central differences of ForwardDynamicsCalculator, host and device paths; external wrenches on such systems are
    refused."""
    import mecano_b200 as mb

    torch, dev = torch_dev
    grav = (0.2, 0.1, -9.81)
    for system in welded_systems():
        assert system.hasWeldedBodies()
        rng = np.random.default_rng(6)
        n = 200
        q, qd, _, tau = mb.MultiBodySystemRandomTools.nextState(rng, system, n)
        nv = system.getNumberOfDoFs()
        integ = mb.MultiBodySystemStateIntegrator(system)
        fdyn = mb.ForwardDynamicsCalculator(system)
        fdyn.setGravitationalAcceleration(*grav)
        qdd_r = fdyn.compute(q, qd, tau).copy()
        Dq, Dv, Dt = np.zeros((nv, nv, n)), np.zeros((nv, nv, n)), np.zeros((nv, nv, n))
        for j in range(nv):
            cq, cv, ct = [], [], []
            for dt in (EPS, -EPS):
                qj, vj = q.copy(), np.zeros((nv, n))
                vj[j] = 1.0
                integ.setIntegrationDT(dt)
                integ.doubleIntegrateFromAcceleration(qj, vj, np.zeros((nv, n)))
                cq.append(fdyn.compute(qj, qd, tau).copy())
                vd = qd.copy()
                vd[j] += dt
                cv.append(fdyn.compute(q, vd, tau).copy())
                td_ = tau.copy()
                td_[j] += dt / EPS
                ct.append(fdyn.compute(q, qd, td_).copy())
            Dq[:, j] = (cq[0] - cq[1]) / (2 * EPS)
            Dv[:, j] = (cv[0] - cv[1]) / (2 * EPS)
            Dt[:, j] = (ct[0] - ct[1]) / 2.0
        calc = mb.ForwardDynamicsDerivativesCalculator(system)
        calc.setGravitationalAcceleration(*grav)
        for dev_path in (True, False):
            args = [torch.from_numpy(np.ascontiguousarray(x)).to(dev) if dev_path else x for x in (q, qd, tau)]
            dq = calc.compute(*args)
            out = [dq, calc.getAccelerationConfigurationGradientMatrix(), calc.getAccelerationVelocityGradientMatrix(),
                   calc.getInverseMassMatrix(), calc.getJointAccelerationMatrix()]
            dq, dq2, dqd, minv, qdd = (x.cpu().numpy() if dev_path else np.asarray(x) for x in out)
            assert np.array_equal(dq, dq2)
            assert dq.shape == (nv * nv, n) and dqd.shape == (nv * nv, n) and minv.shape == (nv * nv, n) and qdd.shape == (nv, n)
            assert np.array_equal(qdd, qdd_r), "qdd must be what ForwardDynamicsCalculator computes"
            assert fd_ok(dq.reshape(nv, nv, n), Dq) < FD_TOL
            assert fd_ok(dqd.reshape(nv, nv, n), Dv) < FD_TOL
            assert fd_ok(minv.reshape(nv, nv, n), Dt) < 1e-11
        calc.setExternalWrenches(np.zeros((6 * system.getNumberOfJoints(), n)))
        with pytest.raises(NotImplementedError):
            calc.compute(q, qd, tau)


@pytest.mark.gpu
def test_refusals(torch_dev):
    import mecano_b200 as mb
    from mecano_b200 import _capi

    torch, dev = torch_dev
    rng = np.random.default_rng(3)
    t = td.humanoid(rng, 2)
    e, _ = engine_of(t, (0.0, 0.0, -9.81))
    lib = _capi.lib
    n, nv = 64, t.nv
    z = lambda rows: torch.zeros((rows, n), dtype=torch.float64, device=dev)  # noqa: E731
    q, v, tau, qdd, dq, dqd, minv = z(t.nq), z(nv), z(nv), z(nv), z(nv * nv), z(nv * nv), z(nv * nv)
    bufs = [x.data_ptr() for x in (q, v, tau)] + [None] + [x.data_ptr() for x in (qdd, dq, dqd, minv)]
    for i in (0, 1, 2, 4, 5, 6, 7):  # every buffer but fext is required
        b = list(bufs)
        b[i] = None
        assert lib.mecano_b200_aba_derivatives(e._h, n, n, *b, None) == -1
    assert lib.mecano_b200_aba_derivatives(e._h, n, n - 1, *bufs, None) == -3
    assert lib.mecano_b200_aba_derivatives_host(e._h, n, n - 1, *([None] * 8)) == -3
    assert lib.mecano_b200_aba_derivatives_host(e._h, n, n, *([None] * 8)) == -1
    minv.fill_(7.0)
    assert lib.mecano_b200_aba_derivatives(e._h, 0, 0, *([None] * 8), None) == 0  # n = 0: a no-op
    assert lib.mecano_b200_aba_derivatives_host(e._h, 0, 0, *([None] * 8)) == 0
    torch.cuda.synchronize()
    assert bool((minv == 7.0).all())
    hb = [np.zeros((r, n)) for r in (t.nq, nv, nv)] + [None] + [np.zeros((r, n)) for r in (nv, nv * nv, nv * nv, nv * nv)]
    hp = [None if x is None else x.ctypes.data for x in hb]
    e.set_precision("fp32")
    assert lib.mecano_b200_aba_derivatives(e._h, n, n, *bufs, None) == -2
    assert lib.mecano_b200_aba_derivatives_host(e._h, n, n, *hp) == -2
    e.set_precision("fp64")
    src = np.zeros(t.nb, np.int32)
    src[3] = 1
    e.set_joint_source_modes(src)
    assert lib.mecano_b200_aba_derivatives(e._h, n, n, *bufs, None) == -1
    assert lib.mecano_b200_aba_derivatives_host(e._h, n, n, *hp) == -1
    e.set_joint_source_modes(None)
    assert lib.mecano_b200_aba_derivatives(e._h, n, n, *bufs, None) == 0
    # a welded system's handle with external wrenches: its wrench ranks count the fixed joints, beyond the 6 n_bodies rows of fext
    welded = welded_systems()[0]
    ew = mb.Engine(welded.tables().contents, 0, keepalive=welded)
    wz = lambda rows: torch.zeros((rows, n), dtype=torch.float64, device=dev)  # noqa: E731
    wb = [wz(welded.getConfigurationMatrixSize()), wz(ew.nv), wz(ew.nv), wz(6 * ew.nb), wz(ew.nv)] + [wz(ew.nv * ew.nv) for _ in range(3)]
    wp = [x.data_ptr() for x in wb]
    assert lib.mecano_b200_aba_derivatives(ew._h, n, n, *wp, None) == -3
    wp[3] = None
    assert lib.mecano_b200_aba_derivatives(ew._h, n, n, *wp, None) == 0
    # a tree the inverse-dynamics derivatives kernel does not fit: refused like mecano_b200_rnea_derivatives
    deep = None
    for depth in (60, 90, 120, 127):
        c = td.chain(np.random.default_rng(depth), depth)
        try:
            ec, _ = engine_of(c, (0.0, 0.0, -9.81))
        except Exception:
            continue  # the handle itself refuses the tree
        if ec.kernel_info(_capi.ALGO_RNEA_DERIVATIVES, 1024)["block_threads"] == 0:
            deep = (c, ec)
            break
    if deep is not None:
        print("refused as too large for the inverse-dynamics derivatives kernel: a chain of", deep[0].nb)
        c, ec = deep
        cb = [z(c.nq), z(c.nv), z(c.nv)] + [None] + [z(c.nv)] + [z(c.nv * c.nv) for _ in range(3)]
        assert lib.mecano_b200_aba_derivatives(ec._h, n, n, *[None if x is None else x.data_ptr() for x in cb], None) == -5
    with pytest.raises(NotImplementedError):
        w = np.zeros((welded.getNumberOfDoFs(), 4))
        mb.ForwardDynamicsDerivativesCalculator(welded, device=[0, 0]).compute(np.zeros((welded.getConfigurationMatrixSize(), 4)), w, w)
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_host_entry_point_matches_the_device_across_chunks():
    env = dict(os.environ, MECANO_B200_HOST_CHUNK_MB="1", PYTHONPATH=os.pathsep.join([ROOT, HERE] + sys.path))
    r = subprocess.run([sys.executable, os.path.abspath(__file__)], env=env, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "forward-dynamics derivatives host entry point matches" in r.stdout


def _compare_host_and_device():
    """With a 1 MB staging budget: 13001 H37 states span many chunks (256 states each) and end on a ragged one; pinned and pageable
    ld > n host views whose columns beyond n must stay NaN."""
    import torch

    import mecano_b200 as mb
    from test_gpu_parity import build

    dev = torch.device("cuda:0")
    s, t = build(kind="humanoid", seed=7, n_joints=2)
    nq, nv, nb = t.nq, t.nv, t.nb
    e = mb.InverseDynamicsCalculator(s)._engine
    e.set_gravity(0.3, -0.2, -9.81)
    rng = np.random.default_rng(18)
    n, ld = 13001, 13001 + 37
    q, qd, _, tau = mb.MultiBodySystemRandomTools.nextState(rng, s, n)
    fext = rng.uniform(-1, 1, size=(6 * nb, n))
    dv = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    dnew = lambda rows: torch.full((rows, n), float("nan"), dtype=torch.float64, device=dev)  # noqa: E731
    for pinned in (True, False):
        for f in (None, fext):
            bufs = []

            def host(rows, fill=None):
                b = torch.empty((rows, ld), dtype=torch.float64).pin_memory().numpy() if pinned else np.empty((rows, ld))
                b[:] = np.nan
                if fill is not None:
                    b[:, :n] = fill
                bufs.append(b)
                return b[:, :n]

            hq, hv, ht = host(nq, q), host(nv, qd), host(nv, tau)
            hout = [host(nv), host(nv * nv), host(nv * nv), host(nv * nv)]
            hf = None if f is None else host(6 * nb, f)
            e.aba_derivatives(hq, hv, ht, *hout, fext=hf)
            dout = [dnew(nv), dnew(nv * nv), dnew(nv * nv), dnew(nv * nv)]
            e.aba_derivatives(dv(q), dv(qd), dv(tau), *dout, fext=None if f is None else dv(f))
            for h_, d_, what in zip(hout, dout, ("qdd", "dqdd_dq", "dqdd_dqd", "minv")):
                assert np.array_equal(h_, d_.cpu().numpy()), "%s (pinned=%s, fext=%s)" % (what, pinned, f is not None)
            for b in bufs:
                assert np.isnan(b[:, n:]).all(), "columns beyond n were written (pinned=%s)" % pinned
    print("forward-dynamics derivatives host entry point matches")


if __name__ == "__main__":
    _compare_host_and_device()
