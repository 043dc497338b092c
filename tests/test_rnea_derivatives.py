"""Inverse-dynamics derivatives (mecano_b200_rnea_derivatives, InverseDynamicsDerivativesCalculator): tau(q, qd, qdd) of RNEA with
d tau / dq (column j along the step the state integrator takes with qd = e_j) and d tau / dqd.  The reference is built from entry
points that already exist: central differences of the C oracle's integrator and RNEA (CPU), of mecano_b200_integrate and
mecano_b200_rnea (GPU), and of InverseDynamicsCalculator (the calculator on welded systems).  CPU tests run the kernel's per-state
routine compiled for the host (tests/emu/emu_rnea_derivatives.cpp); the GPU tests run the sm_100a kernel.

The host entry point is compared with the device entry point across chunks in a child process (this file run as a script), since
the staging budget (MECANO_B200_HOST_CHUNK_MB) is read once per process."""
import os
import subprocess
import sys

import numpy as np
import pytest

import emu_gravity_gradient_lib as egl
import emu_rnea_derivatives_lib as erl
import oracle_lib as ol
import treedesc as td
from test_emulation import trees
from test_gravity_gradient import engine_of, planar_chain, rel, structural_zeros, welded_systems

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
EPS = 1e-5
FD_TOL = 1e-6   # d tau / dq against central differences, per state, relative to max(1, max |D|) (measured on the CPU trees: <= 5e-9)
FDV_TOL = 1e-8  # d tau / dqd: tau is quadratic in qd, so its central differences are exact to round-off (measured: <= 3e-10)
TAU_TOL = 1e-12


def fd_ok(D, Dfd):
    """[nv, nv, n] each: the finite-difference error, state by state, relative to max(1, max |D|) of the state."""
    scale = np.maximum(1.0, np.abs(D).max(axis=(0, 1)))
    return float(np.max(np.abs(D - Dfd).max(axis=(0, 1)) / scale))


def oracle_central_differences(t, g, q, qd, qdd, fext=None):
    """(tau [nv, n], dq [nv, nv, n], dqd [nv, nv, n]) from the C oracle: integrate_batch with dt = +-EPS, qd = e_j, qdd = 0 then
    rnea_batch at the moved q for dq; rnea_batch at qd +- EPS e_j for dqd."""
    o = ol.Oracle(t, gravity=g)
    n = q.shape[1]
    z = np.zeros((t.nv, n))
    f = None if fext is None else np.ascontiguousarray(np.asarray(fext).reshape(6 * t.nb, n))
    dq, dqd = np.zeros((t.nv, t.nv, n)), np.zeros((t.nv, t.nv, n))
    for j in range(t.nv):
        e = np.zeros((t.nv, n))
        e[j] = 1.0
        qp, _, _ = o.integrate_batch(EPS, q, e, z)
        qm, _, _ = o.integrate_batch(-EPS, q, e, z)
        dq[:, j] = (o.rnea_batch(qp, qd, qdd, f) - o.rnea_batch(qm, qd, qdd, f)) / (2 * EPS)
        dqd[:, j] = (o.rnea_batch(q, qd + EPS * e, qdd, f) - o.rnea_batch(q, qd - EPS * e, qdd, f)) / (2 * EPS)
    return o.rnea_batch(q, qd, qdd, f), dq, dqd


def case(idx, n=3):
    rng = np.random.default_rng(1900 + idx)
    t = trees(rng)[idx]
    g = (rng.uniform(-1, 1), rng.uniform(-1, 1), -rng.uniform(1, 10))
    q, qd, qdd, _ = td.random_states(rng, t, n)
    fext = rng.uniform(-1, 1, size=(t.nb, 6, n))
    return t, g, q, qd, qdd, fext


# ---------------------------------------------------------------------------------------------------------------- CPU


@pytest.mark.parametrize("with_fext", [False, True])
@pytest.mark.parametrize("idx", range(16))
def test_emulated_derivatives_match_oracle_central_differences(idx, with_fext):
    """All five joint types, floating bases, a 100-body tree, random gravity and state, with and without external wrenches: both
    matrices against central differences, tau against RNEA, every entry written, the structural zeros +0.0 in both."""
    t, g, q, qd, qdd, fext = case(idx)
    f = fext if with_fext else None
    tau, dq, dqd = erl.rnea_derivatives(t, g, q, qd, qdd, f)
    assert not np.isnan(tau).any() and not np.isnan(dq).any() and not np.isnan(dqd).any(), "every entry must be written"
    tau_o, dq_o, dqd_o = oracle_central_differences(t, g, q, qd, qdd, f)
    assert rel(tau, tau_o) < TAU_TOL
    assert fd_ok(dq, dq_o) < FD_TOL
    assert fd_ok(dqd, dqd_o) < FDV_TOL
    z = structural_zeros(t)
    for D in (dq, dqd):
        assert np.all((D[z] == 0.0) & ~np.signbit(D[z])), "structural zeros are +0.0"


@pytest.mark.parametrize("with_fext", [False, True])
@pytest.mark.parametrize("idx", range(16))
def test_emulated_derivatives_at_rest_reduce_to_the_gravity_gradient(idx, with_fext):
    """At qd = qdd = 0, d tau / dq is the gravity gradient's G and d tau / dqd vanishes."""
    t, g, q, _, _, fext = case(idx)
    f = fext if with_fext else None
    z = np.zeros((t.nv, q.shape[1]))
    tau, dq, dqd = erl.rnea_derivatives(t, g, q, z, z, f)
    tau_g, G = egl.gravity_gradient(t, g, q, f)
    assert rel(tau, tau_g) < TAU_TOL
    assert rel(dq, G) < 1e-12
    assert np.all(dqd == 0.0)


@pytest.mark.parametrize("idx", range(16))
def test_emulated_velocity_derivative_identities(idx):
    """tau is quadratic in qd: dqd . qd = 2 (tau(q, qd, qdd) - tau(q, 0, qdd)) (Euler), and d tau / dqd does not depend on qdd."""
    t, g, q, qd, qdd, fext = case(idx, n=4)
    tau, _, dqd = erl.rnea_derivatives(t, g, q, qd, qdd, fext)
    tau0, _, _ = erl.rnea_derivatives(t, g, q, np.zeros_like(qd), qdd, fext)
    lhs = np.einsum("ijs,js->is", dqd, qd)
    assert rel(lhs, 2 * (tau - tau0)) < 1e-12
    qdd2 = np.random.default_rng(idx).uniform(-3, 3, size=qdd.shape)
    _, _, dqd2 = erl.rnea_derivatives(t, g, q, qd, qdd2, fext)
    assert rel(dqd2, dqd) < 1e-13


def test_planar_two_link_arm_closed_form():
    """With h = m2 l1 l2c sin q2: d tau1 / dqd = (-2 h qd2, -2 h (qd1 + qd2)), d tau2 / dqd = (2 h qd1, 0); d tau / dq is the
    derivative of tau = M(q2) qdd + (-h (2 qd1 qd2 + qd2^2), h qd1^2) + g(q)."""
    m1, m2, l1, l1c, l2c, g0 = 1.3, 0.8, 0.9, 0.4, 0.35, 9.81
    Izz = 0.03  # planar_chain: J = diag(0.01, 0.02, 0.03) about the centre of mass
    t = planar_chain([l1], [l1c, l2c], [m1, m2])
    rng = np.random.default_rng(3)
    n = 17
    q, qd, qdd = (rng.uniform(-np.pi, np.pi, size=(2, n)) for _ in range(3))
    tau, dq, dqd = erl.rnea_derivatives(t, (0.0, -g0, 0.0), q, qd, qdd)
    s1, c1, s2, c2 = np.sin(q[0]), np.cos(q[0]), np.sin(q[1]), np.cos(q[1])
    s12, c12 = np.sin(q[0] + q[1]), np.cos(q[0] + q[1])
    k = m2 * l1 * l2c
    h = k * s2
    M11 = 2 * Izz + m1 * l1c ** 2 + m2 * (l1 ** 2 + l2c ** 2) + 2 * k * c2
    M12 = Izz + m2 * l2c ** 2 + k * c2
    M22 = Izz + m2 * l2c ** 2
    grav = g0 * np.array([m1 * l1c * c1 + m2 * (l1 * c1 + l2c * c12), m2 * l2c * c12])
    tau_ref = np.array([M11 * qdd[0] + M12 * qdd[1] - h * (2 * qd[0] * qd[1] + qd[1] ** 2), M12 * qdd[0] + M22 * qdd[1] + h * qd[0] ** 2]) + grav
    dqd_ref = np.array([[-2 * h * qd[1], -2 * h * (qd[0] + qd[1])], [2 * h * qd[0], np.zeros(n)]])
    dg1 = -g0 * m2 * l2c * s12
    dq_ref = np.array([
        [-g0 * (m1 * l1c * s1 + m2 * (l1 * s1 + l2c * s12)), -2 * k * s2 * qdd[0] - k * s2 * qdd[1] - k * c2 * (2 * qd[0] * qd[1] + qd[1] ** 2) + dg1],
        [dg1, -k * s2 * qdd[0] + k * c2 * qd[0] ** 2 + dg1]])
    assert rel(tau, tau_ref) < 1e-13
    assert rel(dqd, dqd_ref) < 1e-13
    assert rel(dq, dq_ref) < 1e-13


def test_cpp_host_mirror_links_the_derivatives(tmp_path):
    src = tmp_path / "rd.cpp"
    src.write_text('#include "%s"\nint main() { auto a = &mecano::InverseDynamicsDerivativesCalculator::compute; return a ? 0 : 1; }\n'
                   % os.path.join(ROOT, "mecano_b200", "csrc", "host", "calculators.hpp"))
    exe = str(tmp_path / "rd")
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
def test_device_and_host_entry_points_match_the_emulated_routine(torch_dev, idx):
    torch, dev = torch_dev
    t, g, q, qd, qdd, fext = case(idx, n=37)
    e, order = engine_of(t, g)
    n, ld = q.shape[1], q.shape[1] + 11
    nv = t.nv
    pad = lambda a: np.ascontiguousarray(np.pad(a, ((0, 0), (0, ld - n))))  # noqa: E731
    hq, hv, ha = pad(q), pad(qd), pad(qdd)
    tq, tv, ta = (torch.from_numpy(x).to(dev)[:, :n] for x in (hq, hv, ha))
    for f in (None, fext):
        # fext rows in the order of the handle's description (wrench_index defaults to that order)
        hf = None if f is None else pad(f[order].reshape(6 * t.nb, n))
        htau, hdq, hdqd = np.full((nv, ld), np.nan), np.full((nv * nv, ld), np.nan), np.full((nv * nv, ld), np.nan)
        e.rnea_derivatives(hq[:, :n], hv[:, :n], ha[:, :n], htau[:, :n], hdq[:, :n], hdqd[:, :n], fext=None if hf is None else hf[:, :n])
        tf = None if hf is None else torch.from_numpy(hf).to(dev)[:, :n]
        ttau = torch.full((nv, ld), float("nan"), dtype=torch.float64, device=dev)
        tdq = torch.full((nv * nv, ld), float("nan"), dtype=torch.float64, device=dev)
        tdqd = torch.full((nv * nv, ld), float("nan"), dtype=torch.float64, device=dev)
        e.rnea_derivatives(tq, tv, ta, ttau[:, :n], tdq[:, :n], tdqd[:, :n], fext=tf)
        etau, edq, edqd = erl.rnea_derivatives(t, g, q, qd, qdd, f)
        z = structural_zeros(t)
        for h_, d_, em in ((htau, ttau, etau), (hdq, tdq, edq), (hdqd, tdqd, edqd)):
            d_ = d_.cpu().numpy()
            assert np.array_equal(d_, h_, equal_nan=True), "device and host must agree bit for bit"
            assert np.isnan(d_[:, n:]).all(), "nothing written beyond n"
            assert rel(d_[:, :n].reshape(em.shape), em) < 1e-12
            if em.ndim == 3:
                assert np.all(d_[:, :n].reshape(em.shape)[z] == 0.0)


@pytest.mark.gpu
def test_h37_2e18_states_against_device_central_differences(torch_dev):
    """2^18 humanoid states: both matrices against central differences taken on the device with mecano_b200_integrate +
    mecano_b200_rnea for all 37 columns; tau against mecano_b200_rnea; at rest, d tau / dq against mecano_b200_gravity_gradient."""
    torch, dev = torch_dev
    rng = np.random.default_rng(37)
    t = td.humanoid(rng, 2)
    g = (0.3, -0.2, -9.81)
    n = 1 << 18
    nv, nq = t.nv, t.nq
    assert (t.nb, nv, nq) == (32, 37, 38)
    q, qd, qdd = (torch.from_numpy(x).to(dev) for x in td.random_states(rng, t, n)[:3])
    e, _ = engine_of(t, g)
    new = lambda rows: torch.empty((rows, n), dtype=torch.float64, device=dev)  # noqa: E731
    tau, dq, dqd = new(nv), new(nv * nv), new(nv * nv)
    e.rnea_derivatives(q, qd, qdd, tau, dq, dqd)
    tau_r = new(nv)
    e.rnea(q, qd, qdd, tau_r)
    assert ((tau - tau_r).abs().max() / tau_r.abs().max().clamp(min=1.0)).item() < TAU_TOL
    worst_q = worst_v = 0.0
    tp, tm = new(nv), new(nv)
    zero = torch.zeros((nv, n), dtype=torch.float64, device=dev)
    for D, wrt in ((dq.view(nv, nv, n), "q"), (dqd.view(nv, nv, n), "qd")):
        scale = D.abs().amax(dim=(0, 1)).clamp(min=1.0)
        for j in range(nv):
            for dt, out in ((EPS, tp), (-EPS, tm)):
                if wrt == "q":
                    qj, vj = q.clone(), zero.clone()
                    vj[j] = 1.0
                    e.integrate(dt, qj, vj, zero.clone())
                    e.rnea(qj, qd, qdd, out)
                else:
                    vj = qd.clone()
                    vj[j] += dt
                    e.rnea(q, vj, qdd, out)
            err = ((D[:, j] - (tp - tm) / (2 * EPS)).abs().amax(dim=0) / scale).max().item()
            if wrt == "q":
                worst_q = max(worst_q, err)
            else:
                worst_v = max(worst_v, err)
    assert worst_q < FD_TOL, worst_q
    assert worst_v < FDV_TOL, worst_v
    G, tau_g = new(nv * nv), new(nv)
    e.gravity_gradient(q, tau_g, G)
    e.rnea_derivatives(q, zero, zero, tau, dq, dqd)
    assert ((dq - G).abs().max() / G.abs().max()).item() < 1e-12
    assert bool((dqd == 0).all())


@pytest.mark.gpu
def test_calculator_on_systems_with_fixed_and_ignored_joints(torch_dev):
    """Against central differences of InverseDynamicsCalculator, with and without external wrenches, host and device paths."""
    import mecano_b200 as mb

    torch, dev = torch_dev
    grav = (0.2, 0.1, -9.81)
    for system in welded_systems():
        assert system.hasWeldedBodies()
        rng = np.random.default_rng(5)
        n = 200
        q, qd, qdd, _ = mb.MultiBodySystemRandomTools.nextState(rng, system, n)
        nv, nj = system.getNumberOfDoFs(), system.getNumberOfJoints()
        fext = rng.uniform(-1, 1, size=(6 * nj, n))
        integ = mb.MultiBodySystemStateIntegrator(system)
        ident = mb.InverseDynamicsCalculator(system)
        ident.setGravitationalAcceleration(*grav)
        calc = mb.InverseDynamicsDerivativesCalculator(system)
        calc.setGravitationalAcceleration(*grav)
        for f in (None, fext):
            if f is None:
                ident.setExternalWrenchesToZero()
            else:
                ident.setExternalWrenches(f)
            tau_r = ident.compute(q, qd, qdd).copy()
            Dq, Dv = np.zeros((nv, nv, n)), np.zeros((nv, nv, n))
            for j in range(nv):
                cq, cv = [], []
                for dt in (EPS, -EPS):
                    qj, vj = q.copy(), np.zeros((nv, n))
                    vj[j] = 1.0
                    integ.setIntegrationDT(dt)
                    integ.doubleIntegrateFromAcceleration(qj, vj, np.zeros((nv, n)))
                    cq.append(ident.compute(qj, qd, qdd).copy())
                    vd = qd.copy()
                    vd[j] += dt
                    cv.append(ident.compute(q, vd, qdd).copy())
                Dq[:, j] = (cq[0] - cq[1]) / (2 * EPS)
                Dv[:, j] = (cv[0] - cv[1]) / (2 * EPS)
            for dev_path in (True, False):
                if f is None:
                    calc.setExternalWrenchesToZero()
                else:
                    calc.setExternalWrenches(torch.from_numpy(f).to(dev) if dev_path else f)
                args = [torch.from_numpy(np.ascontiguousarray(x)).to(dev) if dev_path else x for x in (q, qd, qdd)]
                dq = calc.compute(*args)
                out = [dq, calc.getTauConfigurationGradientMatrix(), calc.getTauVelocityGradientMatrix(), calc.getJointTauMatrix()]
                dq, dq2, dqd, tau = (x.cpu().numpy() if dev_path else np.asarray(x) for x in out)
                assert np.array_equal(dq, dq2)
                assert dq.shape == (nv * nv, n) and dqd.shape == (nv * nv, n) and tau.shape == (nv, n)
                assert rel(tau, tau_r) < TAU_TOL
                assert fd_ok(dq.reshape(nv, nv, n), Dq) < FD_TOL
                assert fd_ok(dqd.reshape(nv, nv, n), Dv) < FDV_TOL


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
    q, v, a, tau, dq, dqd = z(t.nq), z(nv), z(nv), z(nv), z(nv * nv), z(nv * nv)
    bufs = [x.data_ptr() for x in (q, v, a)] + [None] + [x.data_ptr() for x in (tau, dq, dqd)]
    for i in (0, 1, 2, 4, 5, 6):  # every buffer but fext is required
        b = list(bufs)
        b[i] = None
        assert lib.mecano_b200_rnea_derivatives(e._h, n, n, *b, None) == -1
    assert lib.mecano_b200_rnea_derivatives(e._h, n, n - 1, *bufs, None) == -3
    assert lib.mecano_b200_rnea_derivatives_host(e._h, n, n - 1, *([None] * 7)) == -3
    assert lib.mecano_b200_rnea_derivatives_host(e._h, n, n, *([None] * 7)) == -1
    dq.fill_(7.0)
    assert lib.mecano_b200_rnea_derivatives(e._h, 0, 0, *([None] * 7), None) == 0  # n = 0: a no-op
    assert lib.mecano_b200_rnea_derivatives_host(e._h, 0, 0, *([None] * 7)) == 0
    torch.cuda.synchronize()
    assert bool((dq == 7.0).all())
    e.set_precision("fp32")
    assert lib.mecano_b200_rnea_derivatives(e._h, n, n, *bufs, None) == -2
    h = [np.zeros((r, n)) for r in (t.nq, nv, nv)] + [None] + [np.zeros((r, n)) for r in (nv, nv * nv, nv * nv)]
    assert lib.mecano_b200_rnea_derivatives_host(e._h, n, n, *[None if x is None else x.ctypes.data for x in h]) == -2
    e.set_precision("fp64")
    # a welded system's handle with external wrenches: its wrench ranks count the fixed joints, beyond the 6 n_bodies rows of fext
    welded = welded_systems()[0]
    ew = mb.Engine(welded.tables().contents, 0, keepalive=welded)
    wz = lambda rows: torch.zeros((rows, n), dtype=torch.float64, device=dev)  # noqa: E731
    wb = [wz(welded.getConfigurationMatrixSize()), wz(ew.nv), wz(ew.nv), wz(6 * ew.nb), wz(ew.nv), wz(ew.nv * ew.nv), wz(ew.nv * ew.nv)]
    wp = [x.data_ptr() for x in wb]
    assert lib.mecano_b200_rnea_derivatives(ew._h, n, n, *wp, None) == -3
    wp[3] = None
    assert lib.mecano_b200_rnea_derivatives(ew._h, n, n, *wp, None) == 0
    with pytest.raises(NotImplementedError):
        w = np.zeros((welded.getNumberOfDoFs(), 4))
        mb.InverseDynamicsDerivativesCalculator(welded, device=[0, 0]).compute(np.zeros((welded.getConfigurationMatrixSize(), 4)), w, w)
    info = e.kernel_info(_capi.ALGO_RNEA_DERIVATIVES, 1 << 18)
    assert info["variant"] == 1 and info["bytes_per_state"] == 8.0 * (t.nq + 3 * t.nv + 2 * t.nv * t.nv)
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_host_entry_point_matches_the_device_across_chunks():
    env = dict(os.environ, MECANO_B200_HOST_CHUNK_MB="1", PYTHONPATH=os.pathsep.join([ROOT, HERE] + sys.path))
    r = subprocess.run([sys.executable, os.path.abspath(__file__)], env=env, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "inverse-dynamics derivatives host entry point matches" in r.stdout


def _compare_host_and_device():
    """With a 1 MB staging budget: 13001 H37 states span many chunks (256 states each: 2,888 rows per state without fext) and end on
    a ragged one; pinned and pageable ld > n host views whose columns beyond n must stay NaN."""
    import torch

    import mecano_b200 as mb
    from test_gpu_parity import build

    dev = torch.device("cuda:0")
    s, t = build(kind="humanoid", seed=7, n_joints=2)
    nq, nv, nb = t.nq, t.nv, t.nb
    e = mb.InverseDynamicsCalculator(s)._engine
    e.set_gravity(0.3, -0.2, -9.81)
    rng = np.random.default_rng(17)
    n, ld = 13001, 13001 + 37
    q, qd, qdd, _ = mb.MultiBodySystemRandomTools.nextState(rng, s, n)
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

            hq, hv, ha, htau, hdq, hdqd = host(nq, q), host(nv, qd), host(nv, qdd), host(nv), host(nv * nv), host(nv * nv)
            hf = None if f is None else host(6 * nb, f)
            e.rnea_derivatives(hq, hv, ha, htau, hdq, hdqd, fext=hf)
            dtau, ddq, ddqd = dnew(nv), dnew(nv * nv), dnew(nv * nv)
            e.rnea_derivatives(dv(q), dv(qd), dv(qdd), dtau, ddq, ddqd, fext=None if f is None else dv(f))
            for h_, d_, what in ((htau, dtau, "tau"), (hdq, ddq, "dtau_dq"), (hdqd, ddqd, "dtau_dqd")):
                assert np.array_equal(h_, d_.cpu().numpy()), "%s (pinned=%s, fext=%s)" % (what, pinned, f is not None)
            for b in bufs:
                assert np.isnan(b[:, n:]).all(), "columns beyond n were written (pinned=%s)" % pinned
    print("inverse-dynamics derivatives host entry point matches")


if __name__ == "__main__":
    _compare_host_and_device()
