"""Joint-torque regressor Y(q, qd, qdd) (mecano_b200_joint_torque_regressor, JointTorqueRegressorCalculator): tau = Y pi for ANY
inertial parameters pi.  The reference is built here from the existing RNEA oracle alone, by linearity (regressor_oracle): it
depends only on the definition in include/mecano_b200.h, not on how the kernel is written.  CPU tests run the kernel's per-state
routine compiled for the host (tests/emu/emu_regressor.cpp); the GPU tests run the sm_100a kernel."""
import dataclasses
import os

import numpy as np
import pytest

import emu_lib as el
import emu_regressor_lib as erl
import oracle_lib as ol
import treedesc as td
from test_emulation import trees

TOL = 1e-9
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

# column order of a body's ten parameters (include/mecano_b200.h: MECANO_B200_REGRESSOR_*, mirrored by mecano_b200._capi)
COL_M, COL_MC, COL_I = 0, 1, 4
SYM = ((0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2))  # xx xy xz yy yz zz


def rel(a, b):
    return float(np.max(np.abs(a - b)) / max(1.0, np.max(np.abs(b))))


def unit_sym(k):
    U = np.zeros((3, 3))
    i, j = SYM[k]
    U[i, j] = U[j, i] = 1.0
    return U


def with_params(t, b, m, c, I):
    """Copy of tree t in which body b has mass m, centre of mass c and moment of inertia I about the origin, both in its CoM frame
    (bodyFixedFrame: com_R, com_p), converted to the tree description's (mass, com_p, J about the CoM) by the parallel-axis rule."""
    u = dataclasses.replace(t, com_p=t.com_p.copy(), J=t.J.copy(), mass=t.mass.copy())
    u.mass[b] = m
    u.com_p[b] = t.com_p[b] + t.com_R[b] @ c
    u.J[b] = I - m * (np.dot(c, c) * np.eye(3) - np.outer(c, c))  # (need not be positive definite for RNEA)
    return u.contiguous()


def massless(t):
    return dataclasses.replace(t, mass=np.zeros(t.nb), J=np.zeros((t.nb, 3, 3))).contiguous()


def regressor_oracle(t, gravity, q, qd, qdd):
    """Y [nv, 10 nb, n] column by column from mo_rnea: every body massless except body b with a unit parameter set (m = 1 in every
    set, so that no conversion divides by a zero mass); first moments and inertias minus the mass column."""
    base = massless(t)
    tau = lambda u: ol.Oracle(u, gravity=gravity).rnea_batch(q, qd, qdd)  # noqa: E731
    Y = np.zeros((t.nv, 10 * t.nb, q.shape[1]))
    zero3 = np.zeros(3)
    for b in range(t.nb):
        ym = tau(with_params(base, b, 1.0, zero3, np.zeros((3, 3))))
        Y[:, 10 * b + COL_M] = ym
        for j in range(3):
            Y[:, 10 * b + COL_MC + j] = tau(with_params(base, b, 1.0, np.eye(3)[j], np.zeros((3, 3)))) - ym
        for k in range(6):
            Y[:, 10 * b + COL_I + k] = tau(with_params(base, b, 1.0, zero3, unit_sym(k))) - ym
    return Y


def model_params(t):
    """The model's own pi: [m, 0, 0, 0, J_xx, J_xy, J_xz, J_yy, J_yz, J_zz] per body (tree order)."""
    pi = np.zeros(10 * t.nb)
    for b in range(t.nb):
        pi[10 * b + COL_M] = t.mass[b]
        pi[10 * b + COL_I:10 * b + COL_I + 6] = [t.J[b][i, j] for i, j in SYM]
    return pi


def random_params(rng, t):
    """A random physical parameter set pi' (positive masses, CoM offsets, inertias about the CoM positive definite) and the
    tree that carries it."""
    u = t
    pi = np.zeros(10 * t.nb)
    for b in range(t.nb):
        m, c = 0.1 + rng.uniform(), rng.uniform(-0.5, 0.5, size=3)
        I = td.random_spd_inertia(rng) + m * (np.dot(c, c) * np.eye(3) - np.outer(c, c))
        u = with_params(u, b, m, c, I)
        pi[10 * b + COL_M] = m
        pi[10 * b + COL_MC:10 * b + COL_MC + 3] = m * c
        pi[10 * b + COL_I:10 * b + COL_I + 6] = [I[i, j] for i, j in SYM]
    return u, pi


def structural_zeros(t):
    """Boolean [nv, nb]: DoF row i is off the path from the root to body b."""
    z = np.ones((t.nv, t.nb), dtype=bool)
    for b in range(t.nb):
        a = b
        while a >= 0:
            z[t.dof_off[a]:t.dof_off[a] + td.NDOF[int(t.jtype[a])], b] = False
            a = t.parent[a]
    return z


def emu_regressor(t, gravity, q, qd, qdd):
    """Y [nv, 10 nb, n] in tree order from the kernel routine compiled for the host (tests/emu/emu_regressor.cpp), NaN-prefilled."""
    return erl.regressor(t, gravity, q, qd, qdd)


def case(idx, n=4):
    rng = np.random.default_rng(700 + idx)
    t = trees(rng)[idx]
    g = (rng.uniform(-1, 1), rng.uniform(-1, 1), -rng.uniform(1, 10))
    q, qd, qdd, _ = td.random_states(rng, t, n)
    return rng, t, g, q, qd, qdd


# ---------------------------------------------------------------------------------------------------------------- CPU


def test_column_order_table_matches_the_bindings():
    from mecano_b200 import _capi

    assert (_capi.REGRESSOR_M, _capi.REGRESSOR_MC, _capi.REGRESSOR_I) == (COL_M, COL_MC, COL_I)
    text = open(os.path.join(ROOT, "include", "mecano_b200.h")).read()
    for name, v in (("M", COL_M), ("MC", COL_MC), ("I", COL_I)):
        assert "#define MECANO_B200_REGRESSOR_%s %d\n" % (name, v) in text


@pytest.mark.parametrize("idx", range(16))
def test_emulated_regressor_matches_oracle_helper(idx):
    """All five joint types, floating bases, a 100-body tree, random gravity; every entry written, the structural zeros exactly 0."""
    rng, t, g, q, qd, qdd = case(idx)
    Y = emu_regressor(t, g, q, qd, qdd)
    assert not np.isnan(Y).any(), "every entry of Y must be written (structural zeros included)"
    assert rel(Y, regressor_oracle(t, g, q, qd, qdd)) < TOL
    z = np.repeat(structural_zeros(t), 10, axis=1)
    assert np.all(Y[z] == 0.0)


@pytest.mark.parametrize("idx", [0, 5, 8, 13, 15])
def test_oracle_helper_reproduces_rnea(idx):
    """The helper against mo_rnea on the model's own parameters, and the kernel routine with a random physical parameter set."""
    rng, t, g, q, qd, qdd = case(idx)
    Yo = regressor_oracle(t, g, q, qd, qdd)
    tau = ol.Oracle(t, gravity=g).rnea_batch(q, qd, qdd)
    assert rel(np.einsum("icn,c->in", Yo, model_params(t)), tau) < TOL
    u, pi = random_params(rng, t)
    tau2 = ol.Oracle(u, gravity=g).rnea_batch(q, qd, qdd)
    assert rel(np.einsum("icn,c->in", Yo, pi), tau2) < TOL
    Ye = emu_regressor(t, g, q, qd, qdd)  # Y depends on the kinematics only
    assert rel(np.einsum("icn,c->in", Ye, pi), tau2) < TOL


def test_cpp_host_mirror_links_the_regressor(tmp_path):
    import subprocess

    src = tmp_path / "reg.cpp"
    src.write_text('#include "%s"\nint main() { auto a = &mecano::JointTorqueRegressorCalculator::compute; '
                   'auto b = &mecano::JointTorqueRegressorCalculator::getInertialParameterVector; return (a && b) ? 0 : 1; }\n'
                   % os.path.join(ROOT, "mecano_b200", "csrc", "host", "calculators.hpp"))
    exe = str(tmp_path / "reg")
    libdir = os.path.join(ROOT, "mecano_b200")
    subprocess.check_call(["g++", "-std=c++17", "-Wall", str(src), "-o", exe, "-L" + libdir, "-lmecano_b200", "-Wl,-rpath," + libdir])


# ---------------------------------------------------------------------------------------------------------------- GPU


@pytest.fixture(scope="module")
def torch_dev():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device; the product has no CPU fallback"
    return torch, torch.device("cuda:0")


def engine_of(t, gravity):
    import mecano_b200 as mb
    from mecano_b200 import _capi

    d, keep, order = el.tree_desc_c(t)
    e = mb.Engine(_capi.TreeDesc.from_buffer_copy(bytes(d)), 0, keepalive=keep)
    e.set_gravity(*gravity)
    return e, order


def to_tree_order(Y, t, order):
    n = Y.shape[-1]
    Yc = Y.reshape(t.nv, t.nb, 10, n)
    out = np.empty_like(Yc)
    out[:, order] = Yc
    return out.reshape(t.nv, 10 * t.nb, n)


@pytest.mark.gpu
@pytest.mark.parametrize("idx", range(16))
def test_device_and_host_entry_points_match_oracle_helper(torch_dev, idx):
    torch, dev = torch_dev
    rng, t, g, q, qd, qdd = case(idx, n=37)
    e, order = engine_of(t, g)
    n, ld = q.shape[1], q.shape[1] + 11
    rows = t.nv * 10 * t.nb
    pad = lambda a: np.ascontiguousarray(np.pad(a, ((0, 0), (0, ld - n))))  # noqa: E731
    hq, hqd, hqdd = (pad(a) for a in (q, qd, qdd))
    hY = np.full((rows, ld), np.nan)
    e.joint_torque_regressor(hq[:, :n], hqd[:, :n], hqdd[:, :n], hY[:, :n])
    tq, tqd, tqdd = (torch.from_numpy(a).to(dev)[:, :n] for a in (hq, hqd, hqdd))
    tY = torch.full((rows, ld), float("nan"), dtype=torch.float64, device=dev)
    e.joint_torque_regressor(tq, tqd, tqdd, tY[:, :n])
    dY = tY.cpu().numpy()
    assert np.array_equal(dY[:, :n], hY[:, :n]), "device and host entry points must agree bit for bit"
    assert np.isnan(dY[:, n:]).all() and np.isnan(hY[:, n:]).all(), "nothing written beyond n"
    Y = to_tree_order(dY[:, :n], t, order)
    assert rel(Y, regressor_oracle(t, g, q, qd, qdd)) < TOL
    assert np.all(Y[np.repeat(structural_zeros(t), 10, axis=1)] == 0.0)


@pytest.mark.gpu
def test_h37_2e18_states_on_device(torch_dev):
    """2^18 humanoid states: Y pi_model against mecano_b200_rnea, and Y pi' against RNEA on a second handle built with a random
    physical parameter set -- pins the frame and the column order on the device."""
    torch, dev = torch_dev
    rng = np.random.default_rng(37)
    t = td.humanoid(rng, 2)
    g = (0.1, -0.2, -9.81)
    n = 1 << 18
    assert (t.nb, t.nv, t.nq) == (32, 37, 38)
    q, qd, qdd, _ = (torch.from_numpy(a).to(dev) for a in td.random_states(rng, t, n))
    e, order = engine_of(t, g)
    Y = torch.empty((t.nv * 10 * t.nb, n), dtype=torch.float64, device=dev)
    e.joint_torque_regressor(q, qd, qdd, Y)
    Y3 = Y.view(t.nv, 10 * t.nb, n)

    def check(tree, pi_tree_order):
        pi = np.asarray(pi_tree_order).reshape(t.nb, 10)[order].reshape(-1)  # to the handle's column blocks
        tau_y = torch.einsum("icn,c->in", Y3, torch.from_numpy(pi).to(dev))
        e2, _ = engine_of(tree, g)
        tau = torch.empty((t.nv, n), dtype=torch.float64, device=dev)
        e2.rnea(q, qd, qdd, tau)
        err = ((tau_y - tau).abs().amax(dim=0) / tau.abs().amax(dim=0).clamp(min=1.0)).max().item()
        assert err < TOL, err

    check(t, model_params(t))
    u, pi = random_params(rng, t)
    check(u, pi)


def welded_systems():
    """A floating base with a one-DoF tree below it; the same with a FixedJoint, and with one subtree ignored."""
    import mecano_b200 as mb

    out = []
    for mode in ("fixed", "ignore"):
        rng = np.random.default_rng(11)
        root = mb.RigidBody("elevator")
        body = lambda name, j: mb.RigidBody(name, j, td.random_spd_inertia(rng), 0.1 + rng.uniform(),  # noqa: E731
                                            mb.RigidBodyTransform(td.random_rotation(rng), rng.uniform(-0.5, 0.5, size=3)))
        bodies = [body("pelvis", mb.SixDoFJoint("floating", root))]
        ignore = []
        for k in range(9):
            pred = bodies[rng.integers(len(bodies))]
            T = mb.RigidBodyTransform(td.random_rotation(rng), rng.uniform(-1, 1, size=3))
            if k in (3, 6) and mode == "fixed":
                j = mb.FixedJoint("j%d" % k, pred, T)
            else:
                j = mb.RevoluteJoint("j%d" % k, pred, T, rng.normal(size=3))
                if k == 4 and mode == "ignore":
                    j.setQ(0.7)
                    ignore.append(j)
            bodies.append(body("b%d" % k, j))
        out.append(mb.MultiBodySystem.toMultiBodySystemBasics(root, ignore or None))
    return out


@pytest.mark.gpu
def test_calculator_on_systems_with_fixed_and_ignored_joints(torch_dev):
    import mecano_b200 as mb

    torch, dev = torch_dev
    for system in welded_systems():
        assert system.hasWeldedBodies()
        q, qd, qdd, _ = mb.MultiBodySystemRandomTools.nextState(np.random.default_rng(5), system, 300)
        reg = mb.JointTorqueRegressorCalculator(system)
        reg.setGravitationalAcceleration(0.2, 0.1, -9.81)
        ident = mb.InverseDynamicsCalculator(system)
        ident.setGravitationalAcceleration(0.2, 0.1, -9.81)
        pi = reg.getInertialParameterVector()
        nv = system.getNumberOfDoFs()
        for dev_path in (True, False):
            a = [torch.from_numpy(x).to(dev) for x in (q, qd, qdd)] if dev_path else [q, qd, qdd]
            Y = reg.compute(*a)
            Yn = Y.cpu().numpy() if dev_path else np.asarray(Y)
            assert Yn.shape == (nv * pi.size, q.shape[1])
            tau = ident.compute(*a)
            tau = tau.cpu().numpy() if dev_path else tau
            assert rel(np.einsum("icn,c->in", Yn.reshape(nv, pi.size, -1), pi), tau) < TOL


@pytest.mark.gpu
def test_refusals(torch_dev):
    import mecano_b200 as mb
    from mecano_b200 import _capi

    torch, dev = torch_dev
    rng = np.random.default_rng(3)
    t = td.humanoid(rng, 2)
    e, _ = engine_of(t, (0.0, 0.0, -9.81))
    lib = _capi.lib
    n = 64
    rows = t.nv * 10 * t.nb
    q, qd, qdd = (torch.zeros((r, n), dtype=torch.float64, device=dev) for r in (t.nq, t.nv, t.nv))
    Y = torch.zeros((rows, n), dtype=torch.float64, device=dev)
    p = lambda x: x.data_ptr()  # noqa: E731
    assert lib.mecano_b200_joint_torque_regressor(e._h, n, n, None, p(qd), p(qdd), p(Y), None) == -1
    assert lib.mecano_b200_joint_torque_regressor(e._h, n, n, p(q), p(qd), p(qdd), None, None) == -1
    assert lib.mecano_b200_joint_torque_regressor(e._h, n, n - 1, p(q), p(qd), p(qdd), p(Y), None) == -3
    assert lib.mecano_b200_joint_torque_regressor_host(e._h, n, n - 1, None, None, None, None) == -3
    Y.fill_(7.0)
    assert lib.mecano_b200_joint_torque_regressor(e._h, 0, 0, None, None, None, None, None) == 0  # n = 0: a no-op
    assert lib.mecano_b200_joint_torque_regressor_host(e._h, 0, 0, None, None, None, None) == 0
    torch.cuda.synchronize()
    assert bool((Y == 7.0).all())
    e.set_precision("fp32")
    assert lib.mecano_b200_joint_torque_regressor(e._h, n, n, p(q), p(qd), p(qdd), p(Y), None) == -2
    assert lib.mecano_b200_joint_torque_regressor_host(e._h, n, n, q.cpu().numpy().ctypes.data, qd.cpu().numpy().ctypes.data,
                                                       qdd.cpu().numpy().ctypes.data, np.zeros((rows, n)).ctypes.data) == -2
    e.set_precision("fp64")
    # a welded system's handle: its wrench ranks count the fixed joints, no ten-column block per rank
    welded = welded_systems()[0]
    ew = mb.Engine(welded.tables().contents, 0, keepalive=welded)
    nq, nv = welded.getConfigurationMatrixSize(), welded.getNumberOfDoFs()
    a = [torch.zeros((r, n), dtype=torch.float64, device=dev) for r in (nq, nv, nv, nv * 10 * ew.nb)]
    assert lib.mecano_b200_joint_torque_regressor(ew._h, n, n, *(p(x) for x in a), None) == -3
    info = e.kernel_info(_capi.ALGO_REGRESSOR, 1 << 18)
    assert info["variant"] == 1 and info["bytes_per_state"] == 8.0 * (t.nq + 2 * t.nv + 10 * t.nb * t.nv)
