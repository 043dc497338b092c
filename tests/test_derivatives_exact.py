"""The analytic derivative kernels (rnea_derivatives.cuh: tau, d tau / dq, d tau / dqd; gravity_gradient.cuh: tau_g, G) against an
exact reference: complex-step differentiation of an independent RNEA (tests/complex_step.py), which agrees with the true derivative
to rounding error.  test_rnea_derivatives.py and test_gravity_gradient.py check the definition through the state integrator with
central differences (1e-6), and the device against the same source compiled for the host; here the mathematics itself is held to
1e-12 on the CPU and the device kernels to 1e-11 at every launch configuration the planner can pick for them.

The CPU tests check the reference (against the C oracle's RNEA and integrator, a closed form, and its own step size) and the kernels'
per-state routines compiled for the host (tests/emu).  The GPU tests run the sm_100a kernels at every configuration of kCfg
(thread_kernels.cuh) forced with MECANO_B200_CFG, at batch sizes around the block and across more than two waves of the grid."""
import os
import re

import numpy as np
import pytest

import complex_step as cs
import emu_gravity_gradient_lib as egl
import emu_rnea_derivatives_lib as erl
import oracle_lib as ol
import treedesc as td
from test_emulation import trees
from test_gravity_gradient import engine_of, planar_chain, structural_zeros

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
N_TREES = 16
TOL = 1e-12      # the kernels' per-state routines against the complex-step reference, per state (measured: <= 2.5e-13, edge states included)
DEV_TOL = 1e-11  # the device kernels against the complex-step reference, per state (measured on a B200 over every configuration: <= 6.7e-14)
# revolute angles around the fast sin/cos limit (|q| = 1e5, jointmath.cuh: MB_SINCOS_FAST_LIMIT) and far beyond it
LARGE_ANGLES = (1e5, np.nextafter(1e5, 0.0), -1e5, -np.nextafter(1e5, 0.0), 1e6, -1e7, 1e8, -1e9, 1e9)
GRAVITY = ("random", "zero", "x")


def per_state(D, R):
    """Worst |D - R| of each state relative to max(1, max |R|) of that state; D and R [..., n]."""
    ax = tuple(range(R.ndim - 1))
    return float(np.max(np.abs(D - R).max(axis=ax) / np.maximum(1.0, np.abs(R).max(axis=ax))))


def gravity_of(rng, kind):
    if kind == "zero":
        return (0.0, 0.0, 0.0)
    if kind == "x":
        return (rng.uniform(1, 10), 0.0, 0.0)
    return (rng.uniform(-1, 1), rng.uniform(-1, 1), -rng.uniform(1, 10))


def edge_states(rng, t, n_random=4):
    """Random states, then: qd = 0 with qdd != 0; qdd = 0; one state per LARGE_ANGLES value with every other revolute joint at that
    angle (the trees with revolute joints); one with every prismatic displacement at +-1e5 (the trees with prismatic joints)."""
    rev = [int(t.cfg_off[i]) for i in range(t.nb) if t.jtype[i] == td.REVOLUTE]
    pris = [int(t.cfg_off[i]) for i in range(t.nb) if t.jtype[i] == td.PRISMATIC]
    n = n_random + 2 + (len(LARGE_ANGLES) if rev else 0) + (1 if pris else 0)
    q, qd, qdd, _ = td.random_states(rng, t, n)
    s = n_random
    qd[:, s] = 0.0
    qdd[:, s + 1] = 0.0
    s += 2
    if rev:
        for k, a in enumerate(LARGE_ANGLES):
            for r in rev[k % 2::2] or rev:
                q[r, s] = a
            s += 1
    if pris:
        q[pris, s] = 1e5 * rng.choice([-1.0, 1.0], size=len(pris))
    return q, qd, qdd


def case(idx, kind="random", n_random=4):
    rng = np.random.default_rng(6100 + idx)
    t = trees(rng)[idx]
    g = gravity_of(rng, kind)
    q, qd, qdd = edge_states(rng, t, n_random)
    fext = rng.uniform(-1, 1, size=(t.nb, 6, q.shape[1]))
    return t, g, q, qd, qdd, fext


def assert_plus_zeros(t, *mats):
    z = structural_zeros(t)
    for D in mats:
        assert np.all((D[z] == 0.0) & ~np.signbit(D[z])), "structural zeros are +0.0"


# ---------------------------------------------------------------------------------------------------------------- CPU: the reference


@pytest.mark.parametrize("idx", range(N_TREES))
def test_reference_tau_matches_the_oracle(idx):
    """Re tau of the complex-step evaluation is RNEA: against the C oracle, with and without external wrenches."""
    t, g, q, qd, qdd, fext = case(idx)
    o = ol.Oracle(t, gravity=g)
    for f in (None, fext):
        tau, _, _ = cs.derivatives(t, g, q, qd, qdd, f)
        fo = None if f is None else np.ascontiguousarray(f.reshape(6 * t.nb, -1))
        assert per_state(tau, o.rnea_batch(q, qd, qdd, fo)) < 1e-12


@pytest.mark.parametrize("idx", range(N_TREES))
def test_tangent_is_the_derivative_of_the_integrator_step(idx):
    """tangent(t, q, j) against central differences of the oracle's integrator (the step mecano_b200_integrate takes) with qd = e_j,
    qdd = 0, dt = +-1e-6: every column, every joint type (at angles of order one: a step of 1e-6 is below the spacing of 1e9)."""
    rng = np.random.default_rng(6200 + idx)
    t = trees(rng)[idx]
    q = td.random_states(rng, t, 8)[0]
    o = ol.Oracle(t)
    n = q.shape[1]
    z = np.zeros((t.nv, n))
    dt = 1e-6
    for j in range(t.nv):
        e = np.zeros((t.nv, n))
        e[j] = 1.0
        qp, _, _ = o.integrate_batch(dt, q, e, z)
        qm, _, _ = o.integrate_batch(-dt, q, e, z)
        assert np.max(np.abs(cs.tangent(t, q, j) - (qp - qm) / (2 * dt))) < 1e-9, j


@pytest.mark.parametrize("idx", [3, 8, 10, 13, 14, 15])
def test_reference_does_not_depend_on_the_step(idx):
    """No subtraction, so no step-size trade-off: h = 1e-20 and 1e-40 give what h = 1e-30 gives, up to the rounding of h t_j and of
    the division by h (measured: <= 1.1e-15)."""
    t, g, q, qd, qdd, fext = case(idx)
    ref = cs.derivatives(t, g, q, qd, qdd, fext)
    for h in (1e-20, 1e-40):
        for a, b in zip(cs.derivatives(t, g, q, qd, qdd, fext, h=h), ref):
            assert per_state(a, b) < 1e-14, h


def test_reference_planar_two_link_arm_closed_form():
    """test_rnea_derivatives.test_planar_two_link_arm_closed_form, with the complex-step reference in place of the kernel routine."""
    m1, m2, l1, l1c, l2c, g0 = 1.3, 0.8, 0.9, 0.4, 0.35, 9.81
    Izz = 0.03
    t = planar_chain([l1], [l1c, l2c], [m1, m2])
    rng = np.random.default_rng(3)
    n = 17
    q, qd, qdd = (rng.uniform(-np.pi, np.pi, size=(2, n)) for _ in range(3))
    tau, dq, dqd = cs.derivatives(t, (0.0, -g0, 0.0), q, qd, qdd)
    s1, s2, c2 = np.sin(q[0]), np.sin(q[1]), np.cos(q[1])
    c1, s12, c12 = np.cos(q[0]), np.sin(q[0] + q[1]), np.cos(q[0] + q[1])
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
    assert per_state(tau, tau_ref) < 1e-13
    assert per_state(dqd, dqd_ref) < 1e-13
    assert per_state(dq, dq_ref) < 1e-13


# ---------------------------------------------------------------------------------------------------------------- CPU: the kernels' routines


@pytest.mark.parametrize("kind", GRAVITY)
@pytest.mark.parametrize("with_fext", [False, True])
@pytest.mark.parametrize("idx", range(N_TREES))
def test_emulated_derivatives_match_the_complex_step_reference(idx, with_fext, kind):
    """Both kernels' per-state routines, every tree, random / zero / x-only gravity, at random and edge states (qd = 0, qdd = 0,
    revolute angles at and beyond the fast sin/cos limit, prismatic displacements of 1e5): tau, d tau / dq, d tau / dqd and G
    per state to 1e-12; every entry written; the structural zeros +0.0."""
    t, g, q, qd, qdd, fext = case(idx, kind)
    f = fext if with_fext else None
    tau, dq, dqd = erl.rnea_derivatives(t, g, q, qd, qdd, f)
    ctau, cdq, cdqd = cs.derivatives(t, g, q, qd, qdd, f)
    for D, R in ((tau, ctau), (dq, cdq), (dqd, cdqd)):
        assert not np.isnan(D).any(), "every entry must be written"
        assert per_state(D, R) < TOL
    z = np.zeros_like(qd)
    tau_g, G = egl.gravity_gradient(t, g, q, f)
    ctau_g, cG, _ = cs.derivatives(t, g, q, z, z, f)
    assert not np.isnan(tau_g).any() and not np.isnan(G).any()
    assert per_state(tau_g, ctau_g) < TOL
    assert per_state(G, cG) < TOL
    assert_plus_zeros(t, dq, dqd, G)


# ---------------------------------------------------------------------------------------------------------------- GPU


def cfg_table():
    """[(block, work-area class, TMEM stack slots)] of kCfg in thread_kernels.cuh, in index order."""
    text = open(os.path.join(ROOT, "mecano_b200", "csrc", "thread_kernels.cuh")).read()
    n = int(re.search(r"constexpr int kNumCfg = (\d+);", text).group(1))
    body = re.search(r"constexpr Cfg kCfg\[kNumCfg\] = \{(.*?)\};", text, re.S).group(1)
    table = [tuple(int(x) for x in m) for m in re.findall(r"\{\s*(\d+)\s*,\s*(\d+)\s*,\s*(\d+)\s*\}", body)]
    assert len(table) == n
    return table


def test_configuration_table_parses():
    table = cfg_table()
    assert len(table) >= 14 and all(b % 32 == 0 and c in (0, 1) and tm >= 0 for b, c, tm in table)


@pytest.fixture(scope="module")
def torch_dev():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device; the product has no CPU fallback"
    return torch, torch.device("cuda:0")


P = 257  # distinct states of a device batch: state s of the batch is base state s % P (prime: no tile size divides it)


class Kernel:
    """One of the two kernels on a handle: runs a tiled batch at ld = n + 11 with NaN-filled buffers and returns its outputs
    [rows, ld] on the device, for the comparisons of check()."""

    def __init__(self, name, t, torch, dev):
        from mecano_b200 import _capi

        self.name, self.t, self.torch, self.dev = name, t, torch, dev
        self.algo = _capi.ALGO_RNEA_DERIVATIVES if name == "rd" else _capi.ALGO_GRAVITY_GRADIENT
        nv = t.nv
        self.rows = (nv, nv * nv, nv * nv) if name == "rd" else (nv, nv * nv)

    def run(self, e, base, n, fext_rows):
        torch, dev = self.torch, self.dev
        ld = n + 11
        cols = torch.arange(n, device=dev) % P

        def tiled(x):
            out = torch.full((x.shape[0], ld), float("nan"), dtype=torch.float64, device=dev)
            out[:, :n] = x[:, cols]
            return out

        q, qd, qdd = (tiled(x) for x in base)
        f = None if fext_rows is None else tiled(fext_rows)[:, :n]
        outs = [torch.full((r, ld), float("nan"), dtype=torch.float64, device=dev) for r in self.rows]
        if self.name == "rd":
            e.rnea_derivatives(q[:, :n], qd[:, :n], qdd[:, :n], *(o[:, :n] for o in outs), fext=f)
        else:
            e.gravity_gradient(q[:, :n], *(o[:, :n] for o in outs), fext=f)
        return outs, cols

    def check(self, outs, cols, n, refs):
        """Every entry written, nothing beyond n, the structural zeros +0.0; the worst per-state error against each reference
        ([rows, P] device tensors), in the order given."""
        torch = self.torch
        nv = self.t.nv
        zrows = torch.from_numpy(np.flatnonzero(structural_zeros(self.t).ravel())).to(self.dev)
        worst = []
        for k, o in enumerate(outs):
            assert bool(torch.isnan(o[:, n:]).all()), "%s: columns beyond n were written" % self.name
            d = o[:, :n]
            assert not bool(torch.isnan(d).any()), "%s: every entry must be written" % self.name
            if d.shape[0] == nv * nv and zrows.numel():
                zs = d[zrows]
                assert bool(((zs == 0) & ~torch.signbit(zs)).all()), "%s: structural zeros are +0.0" % self.name
        for ref in refs:
            w = 0.0
            for o, r in zip(outs, ref):
                scale = r.abs().amax(dim=0).clamp(min=1.0)[cols]
                w = max(w, ((o[:, :n] - r[:, cols]).abs().amax(dim=0) / scale).max().item())
            worst.append(w)
        return worst


def references(t, g, q, qd, qdd, fext, torch, dev):
    """{(kernel, with fext): ([emulated outputs], [complex-step outputs])}, each a list of [rows, P] device tensors."""
    to = lambda a: torch.from_numpy(np.ascontiguousarray(a.reshape(a.shape[0] if a.ndim == 2 else a.shape[0] * a.shape[1], -1))).to(dev)  # noqa: E731
    z = np.zeros_like(qd)
    out = {}
    for f in (None, fext):
        out[("rd", f is not None)] = ([to(x) for x in erl.rnea_derivatives(t, g, q, qd, qdd, f)], [to(x) for x in cs.derivatives(t, g, q, qd, qdd, f)])
        out[("gg", f is not None)] = ([to(x) for x in egl.gravity_gradient(t, g, q, f)], [to(x) for x in cs.derivatives(t, g, q, z, z, f)[:2]])
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("idx", range(N_TREES))
def test_device_kernels_at_every_launch_configuration(torch_dev, monkeypatch, idx):
    """For each configuration of kCfg forced on a new handle: either the entry point refuses (the configuration does not fit the
    tree: a TMEM stack these kernels do not have, a work-area class too small, or too much shared memory for its block), or it runs
    with exactly the forced block size.  Each run: n = 1, block - 1, block + 1 and a multi-tile batch (more than two waves of the
    whole device for trees of up to 40 DoFs, two tiles and a ragged one beyond), with and without external wrenches, ld = n + 11
    with the columns beyond n left NaN; the whole batch against the emulated routine (1e-12) and the complex-step reference
    (1e-11)."""
    import mecano_b200 as mb

    torch, dev = torch_dev
    table = cfg_table()
    rng = np.random.default_rng(7100 + idx)
    t = trees(rng)[idx]
    g = gravity_of(rng, GRAVITY[idx % 3])
    q, qd, qdd, _ = td.random_states(rng, t, P)
    qd[:, 1] = 0.0
    qdd[:, 2] = 0.0
    fext = rng.uniform(-1, 1, size=(t.nb, 6, P))
    refs = references(t, g, q, qd, qdd, fext, torch, dev)
    kernels = [Kernel(name, t, torch, dev) for name in ("rd", "gg")]
    ran = {k.name: {} for k in kernels}
    refused = {k.name: [] for k in kernels}
    worst = {"emulated": 0.0, "complex step": 0.0}
    order = None
    for i, (block, cls, tm) in enumerate(table):
        monkeypatch.setenv("MECANO_B200_CFG", "rd=%d,gg=%d" % (i, i))
        e, order = engine_of(t, g)
        monkeypatch.delenv("MECANO_B200_CFG")
        fo = np.ascontiguousarray(fext[order].reshape(6 * t.nb, P))
        base = [torch.from_numpy(x).to(dev) for x in (q, qd, qdd)]
        for k in kernels:
            info = e.kernel_info(k.algo, 1 << 16)
            if info["block_threads"] == 0:
                with pytest.raises(mb._capi.MecanoB200Error) as err:
                    k.run(e, base, 64, None)
                assert err.value.code == -5, (k.name, i)  # MECANO_B200_ERR_TOO_LARGE
                refused[k.name].append(i)
                continue
            assert info["block_threads"] == block and info["tmem_stack_slots"] == 0, (k.name, i, info)
            ran[k.name][i] = info
            sizes = [1, block - 1, block + 1]
            sizes.append(2 * info["sm_count"] * info["blocks_per_sm"] * block + 37 if t.nv <= 40 else 2 * block + (block + 1) // 2)
            for n in sizes:
                for with_f in (False, True):
                    outs, cols = k.run(e, base, n, torch.from_numpy(fo).to(dev) if with_f else None)
                    emu, ref = refs[(k.name, with_f)]
                    w_emu, w_cs = k.check(outs, cols, n, [emu, ref])
                    assert w_emu < 1e-12, (k.name, i, n, with_f, w_emu)
                    assert w_cs < DEV_TOL, (k.name, i, n, with_f, w_cs)
                    worst["emulated"] = max(worst["emulated"], w_emu)
                    worst["complex step"] = max(worst["complex step"], w_cs)
                    del outs
        e.close()
    # the refusals are the configurations that cannot fit, and the planner's own choice is one that runs
    e, _ = engine_of(t, g)
    for k in kernels:
        assert ran[k.name], "%s: no configuration runs" % k.name
        for i in refused[k.name]:
            block, cls, tm = table[i]
            if tm > 0:
                continue  # these kernels keep their stack in shared memory only
            # within one work-area class, shared memory and registers per block grow with the block: the refused block is larger
            # than every block of its class that ran
            same_class = [table[j][0] for j in ran[k.name] if table[j][1] == cls]
            assert all(b < block for b in same_class), (k.name, i, same_class)
            # a class-0 block refused while a class-1 block at least as large runs (same shared memory) is refused for its work
            # areas: then the tree needs class 1 and no class-0 configuration runs at all
            if cls == 0 and any(table[j][1] == 1 and table[j][0] >= block for j in ran[k.name]):
                assert not same_class, (k.name, i)
        for i in ran[k.name]:
            assert table[i][2] == 0, (k.name, i)
        default = e.kernel_info(k.algo, 1 << 16)
        keys = ("block_threads", "blocks_per_sm", "regs_per_thread", "local_bytes_per_thread", "dynamic_smem_bytes")
        assert any(all(default[x] == info[x] for x in keys) for info in ran[k.name].values()), (k.name, default)
    e.close()
    print("\ntree %d (nb %d, nv %d): ran rd %s gg %s; refused rd %s gg %s; worst against the emulated routine %.1e, against the "
          "complex-step reference %.1e" % (idx, t.nb, t.nv, sorted(ran["rd"]), sorted(ran["gg"]), refused["rd"], refused["gg"],
                                           worst["emulated"], worst["complex step"]))


@pytest.mark.gpu
@pytest.mark.parametrize("idx", [1, 2, 3, 8, 11, 13])
def test_device_kernels_at_large_angles(torch_dev, idx):
    """The edge states of the CPU tests (revolute angles at and beyond the fast sin/cos limit, prismatic displacements of 1e5, qd = 0,
    qdd = 0) through both device kernels at the planner's configuration, against the emulated routine and the complex-step
    reference."""
    torch, dev = torch_dev
    t, g, q, qd, qdd, fext = case(idx, n_random=2)
    n = q.shape[1]
    e, order = engine_of(t, g)
    base = [torch.from_numpy(np.ascontiguousarray(np.tile(x, (1, -(-P // n)))[:, :P])).to(dev) for x in (q, qd, qdd)]
    fx = np.tile(fext, (1, 1, -(-P // n)))[:, :, :P]
    refs = references(t, g, *(x.cpu().numpy() for x in base), fx, torch, dev)
    fo = torch.from_numpy(np.ascontiguousarray(fx[order].reshape(6 * t.nb, P))).to(dev)
    for name in ("rd", "gg"):
        k = Kernel(name, t, torch, dev)
        for with_f in (False, True):
            outs, cols = k.run(e, base, P, fo if with_f else None)
            w_emu, w_cs = k.check(outs, cols, P, refs[(name, with_f)])
            assert w_emu < 1e-12, (name, with_f, w_emu)
            assert w_cs < DEV_TOL, (name, with_f, w_cs)


@pytest.mark.gpu
def test_h37_2e18_states_against_the_complex_step_reference(torch_dev):
    """512 strided states of a 2^18-state humanoid batch, both kernels, against the complex-step reference."""
    torch, dev = torch_dev
    rng = np.random.default_rng(37)
    t = td.humanoid(rng, 2)
    g = (0.3, -0.2, -9.81)
    n, stride = 1 << 18, 512
    nv = t.nv
    q, qd, qdd, _ = td.random_states(rng, t, n)
    e, _ = engine_of(t, g)
    tq, tqd, tqdd = (torch.from_numpy(x).to(dev) for x in (q, qd, qdd))
    new = lambda rows: torch.full((rows, n), float("nan"), dtype=torch.float64, device=dev)  # noqa: E731
    tau, dq, dqd = new(nv), new(nv * nv), new(nv * nv)
    e.rnea_derivatives(tq, tqd, tqdd, tau, dq, dqd)
    tau_g, G = new(nv), new(nv * nv)
    e.gravity_gradient(tq, tau_g, G)
    s = slice(stride // 2, n, stride)
    qs, qds, qdds = q[:, s], qd[:, s], qdd[:, s]
    assert qs.shape[1] == n // stride
    host = lambda x: x[:, s].cpu().numpy()  # noqa: E731
    ref = cs.derivatives(t, g, qs, qds, qdds)
    for D, R in zip((host(tau), host(dq).reshape(nv, nv, -1), host(dqd).reshape(nv, nv, -1)), ref):
        assert per_state(D, R) < DEV_TOL
    z = np.zeros_like(qds)
    ref_g = cs.derivatives(t, g, qs, z, z)
    assert per_state(host(tau_g), ref_g[0]) < DEV_TOL
    assert per_state(host(G).reshape(nv, nv, -1), ref_g[1]) < DEV_TOL
