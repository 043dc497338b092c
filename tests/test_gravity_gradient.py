"""Gravity gradient (mecano_b200_gravity_gradient, MultiBodyGravityGradientCalculator): tau_g(q) = RNEA(q, 0, 0, fext) and its
configuration gradient G = d tau_g / dq, column j along the step the state integrator takes with qd = e_j.  The reference is built
from entry points that already exist: central differences of the C oracle's integrator and RNEA (CPU), of mecano_b200_integrate and
mecano_b200_rnea (GPU), and of InverseDynamicsCalculator (the calculator on welded systems).  CPU tests run the kernel's per-state
routine compiled for the host (tests/emu/emu_gravity_gradient.cpp); the GPU tests run the sm_100a kernel.

The host entry point is compared with the device entry point across chunks in a child process (this file run as a script), since
the staging budget (MECANO_B200_HOST_CHUNK_MB) is read once per process."""
import os
import subprocess
import sys

import numpy as np
import pytest

import emu_gravity_gradient_lib as egl
import oracle_lib as ol
import treedesc as td
from test_emulation import trees

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
EPS = 1e-5
FD_TOL = 1e-6  # |G - central difference| <= FD_TOL * max(1, max |G|) per state (measured on the CPU trees: <= 6e-9)
TAU_TOL = 1e-12
ONE_DOF_FIXED_BASE = (0, 1, 2, 3, 11)  # indices of test_emulation.trees without a floating base or three-DoF joints


def rel(a, b):
    return float(np.max(np.abs(a - b)) / max(1.0, np.max(np.abs(b))))


def fd_ok(G, Gfd):
    """[nv, nv, n] each: the finite-difference bound, state by state."""
    scale = np.maximum(1.0, np.abs(G).max(axis=(0, 1)))
    return float(np.max(np.abs(G - Gfd).max(axis=(0, 1)) / scale))


def oracle_central_differences(t, g, q, fext=None):
    """(tau [nv, n], G [nv, nv, n]) from the C oracle: integrate_batch with dt = +-EPS, qd = e_j, qdd = 0, then rnea_batch at rest."""
    o = ol.Oracle(t, gravity=g)
    n = q.shape[1]
    z = np.zeros((t.nv, n))
    f = None if fext is None else np.ascontiguousarray(np.asarray(fext).reshape(6 * t.nb, n))
    G = np.zeros((t.nv, t.nv, n))
    for j in range(t.nv):
        e = np.zeros((t.nv, n))
        e[j] = 1.0
        qp, _, _ = o.integrate_batch(EPS, q, e, z)
        qm, _, _ = o.integrate_batch(-EPS, q, e, z)
        G[:, j] = (o.rnea_batch(qp, z, z, f) - o.rnea_batch(qm, z, z, f)) / (2 * EPS)
    return o.rnea_batch(q, z, z, f), G


def structural_zeros(t):
    """Boolean [nv, nv]: the DoFs of rows and columns on no common root path (the mass matrix's structural zeros)."""
    body = np.empty(t.nv, dtype=np.int64)
    for b in range(t.nb):
        body[t.dof_off[b]:t.dof_off[b] + td.NDOF[int(t.jtype[b])]] = b

    def ancestors(b):
        out = set()
        while b >= 0:
            out.add(b)
            b = int(t.parent[b])
        return out

    anc = [ancestors(b) for b in range(t.nb)]
    return np.array([[not (body[i] in anc[body[j]] or body[j] in anc[body[i]]) for j in range(t.nv)] for i in range(t.nv)])


def case(idx, n=3):
    rng = np.random.default_rng(900 + idx)
    t = trees(rng)[idx]
    g = (rng.uniform(-1, 1), rng.uniform(-1, 1), -rng.uniform(1, 10))
    q, _, _, _ = td.random_states(rng, t, n)
    fext = rng.uniform(-1, 1, size=(t.nb, 6, n))
    return t, g, q, fext


# ---------------------------------------------------------------------------------------------------------------- CPU


@pytest.mark.parametrize("with_fext", [False, True])
@pytest.mark.parametrize("idx", range(16))
def test_emulated_gradient_matches_oracle_central_differences(idx, with_fext):
    """All five joint types, floating bases, a 100-body tree, random gravity, with and without external wrenches: G against central
    differences, tau against RNEA at rest, every entry written, the structural zeros exactly 0.0."""
    t, g, q, fext = case(idx)
    f = fext if with_fext else None
    tau, G = egl.gravity_gradient(t, g, q, f)
    assert not np.isnan(tau).any() and not np.isnan(G).any(), "every entry must be written (structural zeros included)"
    tau_o, G_o = oracle_central_differences(t, g, q, f)
    assert rel(tau, tau_o) < TAU_TOL
    assert fd_ok(G, G_o) < FD_TOL
    z = structural_zeros(t)
    assert np.all(G[z] == 0.0)
    assert np.all((G[z] == 0.0) & ~np.signbit(G[z])), "structural zeros are +0.0"


@pytest.mark.parametrize("idx", ONE_DOF_FIXED_BASE)
def test_emulated_gradient_is_symmetric_on_one_dof_trees(idx):
    """Without external wrenches, on a fixed-base tree of one-DoF joints G is the Hessian of the potential energy."""
    t, g, q, _ = case(idx, n=5)
    assert all(int(j) in (td.REVOLUTE, td.PRISMATIC) for j in t.jtype)
    _, G = egl.gravity_gradient(t, g, q)
    assert rel(G, np.swapaxes(G, 0, 1)) < 1e-12


def planar_chain(lengths, coms, masses):
    """Revolute joints about z, link k from joint k to joint k + 1 along its x axis, centre of mass at coms[k] along x."""
    nb = len(masses)
    t = td.TreeDesc(
        nb=nb, nv=nb, nq=nb, parent=np.arange(-1, nb - 1, dtype=np.int32), jtype=np.zeros(nb, np.int32),
        axis=np.tile([0.0, 0.0, 1.0], (nb, 1)), off_R=np.tile(np.eye(3), (nb, 1, 1)),
        off_p=np.array([[0.0 if k == 0 else lengths[k - 1], 0.0, 0.0] for k in range(nb)]), com_R=np.tile(np.eye(3), (nb, 1, 1)),
        com_p=np.array([[c, 0.0, 0.0] for c in coms]), J=np.tile(np.diag([0.01, 0.02, 0.03]), (nb, 1, 1)), mass=np.asarray(masses, float),
        dof_off=np.arange(nb, dtype=np.int32), cfg_off=np.arange(nb, dtype=np.int32))
    return t.contiguous()


def test_pendulum_closed_form():
    """m l about z, gravity along -y: V = m g l sin q, tau = m g l cos q, G = -m g l sin q."""
    m, l, g0 = 1.7, 0.6, 9.81
    t = planar_chain([], [l], [m])
    q = np.linspace(-3.0, 3.0, 13)[None, :]
    tau, G = egl.gravity_gradient(t, (0.0, -g0, 0.0), q)
    assert rel(tau[0], m * g0 * l * np.cos(q[0])) < 1e-14
    assert rel(G[0, 0], -m * g0 * l * np.sin(q[0])) < 1e-14


def test_planar_two_link_arm_closed_form():
    """V = g (m1 l1c s1 + m2 (l1 s1 + l2c s12)); tau = grad V, G = the Hessian of V."""
    m1, m2, l1, l1c, l2c, g0 = 1.3, 0.8, 0.9, 0.4, 0.35, 9.81
    t = planar_chain([l1], [l1c, l2c], [m1, m2])
    rng = np.random.default_rng(2)
    q = rng.uniform(-np.pi, np.pi, size=(2, 17))
    tau, G = egl.gravity_gradient(t, (0.0, -g0, 0.0), q)
    s1, c1, s12, c12 = np.sin(q[0]), np.cos(q[0]), np.sin(q[0] + q[1]), np.cos(q[0] + q[1])
    tau_ref = g0 * np.array([m1 * l1c * c1 + m2 * (l1 * c1 + l2c * c12), m2 * l2c * c12])
    h12 = -g0 * m2 * l2c * s12
    G_ref = np.array([[-g0 * (m1 * l1c * s1 + m2 * (l1 * s1 + l2c * s12)), h12], [h12, h12]])
    assert rel(tau, tau_ref) < 1e-14
    assert rel(G, G_ref) < 1e-14


def test_cpp_host_mirror_links_the_gravity_gradient(tmp_path):
    src = tmp_path / "gg.cpp"
    src.write_text('#include "%s"\nint main() { auto a = &mecano::MultiBodyGravityGradientCalculator::compute; return a ? 0 : 1; }\n'
                   % os.path.join(ROOT, "mecano_b200", "csrc", "host", "calculators.hpp"))
    exe = str(tmp_path / "gg")
    libdir = os.path.join(ROOT, "mecano_b200")
    subprocess.check_call(["g++", "-std=c++17", "-Wall", str(src), "-o", exe, "-L" + libdir, "-lmecano_b200", "-Wl,-rpath," + libdir])


# ---------------------------------------------------------------------------------------------------------------- GPU


@pytest.fixture(scope="module")
def torch_dev():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device; the product has no CPU fallback"
    return torch, torch.device("cuda:0")


def engine_of(t, gravity):
    import emu_lib as el
    import mecano_b200 as mb
    from mecano_b200 import _capi

    d, keep, order = el.tree_desc_c(t)
    e = mb.Engine(_capi.TreeDesc.from_buffer_copy(bytes(d)), 0, keepalive=keep)
    e.set_gravity(*gravity)
    return e, order


@pytest.mark.gpu
@pytest.mark.parametrize("idx", range(16))
def test_device_and_host_entry_points_match_the_emulated_routine(torch_dev, idx):
    torch, dev = torch_dev
    t, g, q, fext = case(idx, n=37)
    e, order = engine_of(t, g)
    n, ld = q.shape[1], q.shape[1] + 11
    nv = t.nv
    pad = lambda a: np.ascontiguousarray(np.pad(a, ((0, 0), (0, ld - n))))  # noqa: E731
    for f in (None, fext):
        # fext rows in the order of the handle's description (wrench_index defaults to that order)
        hf = None if f is None else pad(f[order].reshape(6 * t.nb, n))
        hq = pad(q)
        htau, hG = np.full((nv, ld), np.nan), np.full((nv * nv, ld), np.nan)
        e.gravity_gradient(hq[:, :n], htau[:, :n], hG[:, :n], fext=None if hf is None else hf[:, :n])
        tq = torch.from_numpy(hq).to(dev)[:, :n]
        tf = None if hf is None else torch.from_numpy(hf).to(dev)[:, :n]
        ttau = torch.full((nv, ld), float("nan"), dtype=torch.float64, device=dev)
        tG = torch.full((nv * nv, ld), float("nan"), dtype=torch.float64, device=dev)
        e.gravity_gradient(tq, ttau[:, :n], tG[:, :n], fext=tf)
        dtau, dG = ttau.cpu().numpy(), tG.cpu().numpy()
        assert np.array_equal(dtau, htau, equal_nan=True) and np.array_equal(dG, hG, equal_nan=True), "device and host must agree bit for bit"
        assert np.isnan(dtau[:, n:]).all() and np.isnan(dG[:, n:]).all(), "nothing written beyond n"
        etau, eG = egl.gravity_gradient(t, g, q, f)
        assert rel(dtau[:, :n], etau) < 1e-12
        assert rel(dG[:, :n].reshape(nv, nv, n), eG) < 1e-12
        assert np.all(dG[:, :n].reshape(nv, nv, n)[structural_zeros(t)] == 0.0)


@pytest.mark.gpu
def test_h37_2e18_states_against_device_central_differences(torch_dev):
    """2^18 humanoid states: G against central differences taken on the device with mecano_b200_integrate + mecano_b200_rnea for all
    37 columns; tau against mecano_b200_rnea at rest."""
    torch, dev = torch_dev
    rng = np.random.default_rng(37)
    t = td.humanoid(rng, 2)
    g = (0.3, -0.2, -9.81)
    n = 1 << 18
    nv, nq = t.nv, t.nq
    assert (t.nb, nv, nq) == (32, 37, 38)
    q = torch.from_numpy(td.random_states(rng, t, n)[0]).to(dev)
    e, _ = engine_of(t, g)
    tau = torch.empty((nv, n), dtype=torch.float64, device=dev)
    G = torch.empty((nv * nv, n), dtype=torch.float64, device=dev)
    e.gravity_gradient(q, tau, G)
    z = torch.zeros((nv, n), dtype=torch.float64, device=dev)
    tau_r = torch.empty_like(tau)
    e.rnea(q, z, z, tau_r)
    assert ((tau - tau_r).abs().max() / tau_r.abs().max().clamp(min=1.0)).item() < TAU_TOL
    G3 = G.view(nv, nv, n)
    scale = G3.abs().amax(dim=(0, 1)).clamp(min=1.0)
    worst = 0.0
    tp, tm = torch.empty_like(tau), torch.empty_like(tau)
    for j in range(nv):
        for dt, out in ((EPS, tp), (-EPS, tm)):
            qj, vj, aj = q.clone(), torch.zeros((nv, n), dtype=torch.float64, device=dev), torch.zeros((nv, n), dtype=torch.float64, device=dev)
            vj[j] = 1.0
            e.integrate(dt, qj, vj, aj)
            e.rnea(qj, z, z, out)
        fd = (tp - tm) / (2 * EPS)
        worst = max(worst, ((G3[:, j] - fd).abs().amax(dim=0) / scale).max().item())
    assert worst < FD_TOL, worst


def welded_systems():
    """A floating base with a one-DoF tree below it; the same with FixedJoints, and with one subtree ignored."""
    from test_regressor import welded_systems as ws

    return ws()


@pytest.mark.gpu
def test_calculator_on_systems_with_fixed_and_ignored_joints(torch_dev):
    """Against central differences of InverseDynamicsCalculator at rest, with and without external wrenches, host and device paths."""
    import mecano_b200 as mb

    torch, dev = torch_dev
    grav = (0.2, 0.1, -9.81)
    for system in welded_systems():
        assert system.hasWeldedBodies()
        rng = np.random.default_rng(5)
        n = 200
        q, _, _, _ = mb.MultiBodySystemRandomTools.nextState(rng, system, n)
        nv, nj = system.getNumberOfDoFs(), system.getNumberOfJoints()
        fext = rng.uniform(-1, 1, size=(6 * nj, n))
        integ = mb.MultiBodySystemStateIntegrator(system)
        ident = mb.InverseDynamicsCalculator(system)
        ident.setGravitationalAcceleration(*grav)
        calc = mb.MultiBodyGravityGradientCalculator(system)
        calc.setGravitationalAcceleration(*grav)
        z = np.zeros((nv, n))
        for f in (None, fext):
            if f is None:
                ident.setExternalWrenchesToZero()
            else:
                ident.setExternalWrenches(f)
            tau_r = ident.compute(q, z, z).copy()
            Gfd = np.zeros((nv, nv, n))
            for j in range(nv):
                cols = []
                for dt in (EPS, -EPS):
                    qj, vj = q.copy(), np.zeros((nv, n))
                    vj[j] = 1.0
                    integ.setIntegrationDT(dt)
                    integ.doubleIntegrateFromAcceleration(qj, vj, np.zeros((nv, n)))
                    cols.append(ident.compute(qj, z, z).copy())
                Gfd[:, j] = (cols[0] - cols[1]) / (2 * EPS)
            for dev_path in (True, False):
                if f is None:
                    calc.setExternalWrenchesToZero()
                else:
                    calc.setExternalWrenches(torch.from_numpy(f).to(dev) if dev_path else f)
                G = calc.compute(torch.from_numpy(q).to(dev) if dev_path else q)
                tau = calc.getTauMatrix()
                G, tau = (x.cpu().numpy() if dev_path else np.asarray(x) for x in (G, tau))
                assert G.shape == (nv * nv, n) and tau.shape == (nv, n)
                assert rel(tau, tau_r) < TAU_TOL
                assert fd_ok(G.reshape(nv, nv, n), Gfd) < FD_TOL


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
    q = torch.zeros((t.nq, n), dtype=torch.float64, device=dev)
    tau = torch.zeros((nv, n), dtype=torch.float64, device=dev)
    G = torch.zeros((nv * nv, n), dtype=torch.float64, device=dev)
    p = lambda x: x.data_ptr()  # noqa: E731
    assert lib.mecano_b200_gravity_gradient(e._h, n, n, None, None, p(tau), p(G), None) == -1
    assert lib.mecano_b200_gravity_gradient(e._h, n, n, p(q), None, None, p(G), None) == -1
    assert lib.mecano_b200_gravity_gradient(e._h, n, n, p(q), None, p(tau), None, None) == -1
    assert lib.mecano_b200_gravity_gradient(e._h, n, n - 1, p(q), None, p(tau), p(G), None) == -3
    assert lib.mecano_b200_gravity_gradient_host(e._h, n, n - 1, None, None, None, None) == -3
    assert lib.mecano_b200_gravity_gradient_host(e._h, n, n, None, None, None, None) == -1
    G.fill_(7.0)
    assert lib.mecano_b200_gravity_gradient(e._h, 0, 0, None, None, None, None, None) == 0  # n = 0: a no-op
    assert lib.mecano_b200_gravity_gradient_host(e._h, 0, 0, None, None, None, None) == 0
    torch.cuda.synchronize()
    assert bool((G == 7.0).all())
    e.set_precision("fp32")
    assert lib.mecano_b200_gravity_gradient(e._h, n, n, p(q), None, p(tau), p(G), None) == -2
    hq, htau, hG = np.zeros((t.nq, n)), np.zeros((nv, n)), np.zeros((nv * nv, n))
    assert lib.mecano_b200_gravity_gradient_host(e._h, n, n, hq.ctypes.data, None, htau.ctypes.data, hG.ctypes.data) == -2
    e.set_precision("fp64")
    # a welded system's handle with external wrenches: its wrench ranks count the fixed joints, beyond the 6 n_bodies rows of fext
    welded = welded_systems()[0]
    ew = mb.Engine(welded.tables().contents, 0, keepalive=welded)
    wq = torch.zeros((welded.getConfigurationMatrixSize(), n), dtype=torch.float64, device=dev)
    wf = torch.zeros((6 * ew.nb, n), dtype=torch.float64, device=dev)
    wt = torch.zeros((ew.nv, n), dtype=torch.float64, device=dev)
    wG = torch.zeros((ew.nv * ew.nv, n), dtype=torch.float64, device=dev)
    assert lib.mecano_b200_gravity_gradient(ew._h, n, n, p(wq), p(wf), p(wt), p(wG), None) == -3
    assert lib.mecano_b200_gravity_gradient(ew._h, n, n, p(wq), None, p(wt), p(wG), None) == 0
    with pytest.raises(NotImplementedError):
        mb.MultiBodyGravityGradientCalculator(welded, device=[0, 0]).compute(np.zeros((welded.getConfigurationMatrixSize(), 4)))
    info = e.kernel_info(_capi.ALGO_GRAVITY_GRADIENT, 1 << 18)
    assert info["variant"] == 1 and info["bytes_per_state"] == 8.0 * (t.nq + t.nv + t.nv * t.nv)
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_host_entry_point_matches_the_device_across_chunks():
    env = dict(os.environ, MECANO_B200_HOST_CHUNK_MB="1", PYTHONPATH=os.pathsep.join([ROOT, HERE] + sys.path))
    r = subprocess.run([sys.executable, os.path.abspath(__file__)], env=env, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "gravity gradient host entry point matches" in r.stdout


def _compare_host_and_device():
    """With a 1 MB staging budget: 13001 H37 states span at least four chunks (256 states each: 1,444 rows per state without fext) and end on a
    ragged one; pinned and pageable ld > n host views whose columns beyond n must stay NaN."""
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
    q, _, _, _ = mb.MultiBodySystemRandomTools.nextState(rng, s, n)
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

            hq, htau, hG = host(nq, q), host(nv), host(nv * nv)
            hf = None if f is None else host(6 * nb, f)
            e.gravity_gradient(hq, htau, hG, fext=hf)
            dtau, dG = dnew(nv), dnew(nv * nv)
            e.gravity_gradient(dv(q), dtau, dG, fext=None if f is None else dv(f))
            for h_, d_, what in ((htau, dtau, "tau"), (hG, dG, "G")):
                assert np.array_equal(h_, d_.cpu().numpy()), "%s (pinned=%s, fext=%s)" % (what, pinned, f is not None)
            for b in bufs:
                assert np.isnan(b[:, n:]).all(), "columns beyond n were written (pinned=%s)" % pinned
    print("gravity gradient host entry point matches")


if __name__ == "__main__":
    _compare_host_and_device()
