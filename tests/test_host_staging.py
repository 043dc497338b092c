"""GPU test of the chunked staging behind every *_host entry point: with a 1 MB staging budget every call spans at least four
chunks over the handle's three slots and ends on a ragged chunk.  Each host entry point must return exactly what its device entry
point returns for the same states, bit for bit, and leave the columns of an ld > n buffer beyond n untouched; host buffers are
pinned and pageable.

The budget is read once per process (MECANO_B200_HOST_CHUNK_MB), so the comparisons run in a child process: this file run as a
script."""
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


@pytest.mark.gpu
def test_host_entry_points_match_the_device_across_chunks():
    env = dict(os.environ, MECANO_B200_HOST_CHUNK_MB="1", PYTHONPATH=os.pathsep.join([ROOT, HERE] + sys.path))
    r = subprocess.run([sys.executable, os.path.abspath(__file__)], env=env, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "all host entry points match" in r.stdout


def _compare_all():
    import torch

    import mecano_b200 as mb
    from mecano_b200 import _capi
    from test_gpu_parity import build

    dev = torch.device("cuda:0")
    s, t = build(kind="humanoid", seed=7, n_joints=2)
    nq, nv, nb = t.nq, t.nv, t.nb
    e = mb.InverseDynamicsCalculator(s)._engine
    e.set_gravity(0.3, -0.2, -9.81)
    rng = np.random.default_rng(17)
    # 13001 states: four full chunks and a ragged one for the narrowest job (the centre of mass, 3072 states per chunk)
    n, ld = 13001, 13001 + 37
    q, qd, qdd, tau = mb.MultiBodySystemRandomTools.nextState(rng, s, n)
    fext = rng.uniform(-1, 1, size=(6 * nb, n))
    dv = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    dnew = lambda rows: torch.full((rows, n), float("nan"), dtype=torch.float64, device=dev)  # noqa: E731

    for pinned in (True, False):
        tail = {}  # id of a host view -> the columns of its buffer beyond n

        def host(rows, fill=None):
            """[rows, n] view of a [rows, ld] buffer holding NaN beyond n (and `fill`, if given, before)."""
            b = torch.empty((rows, ld), dtype=torch.float64).pin_memory().numpy() if pinned else np.empty((rows, ld))
            b[:] = np.nan
            if fill is not None:
                b[:, :n] = fill
            v = b[:, :n]
            tail[id(v)] = b[:, n:]
            return v

        def same(h, d, what):
            assert np.array_equal(h, d.cpu().numpy() if isinstance(d, torch.Tensor) else d), "%s (pinned=%s)" % (what, pinned)
            assert np.isnan(tail[id(h)]).all(), "%s: columns beyond n were written (pinned=%s)" % (what, pinned)

        hq, hqd, hqdd, htau, hf = host(nq, q), host(nv, qd), host(nv, qdd), host(nv, tau), host(6 * nb, fext)
        tq, tqd, tqdd, ttau, tf = dv(q), dv(qd), dv(qdd), dv(tau), dv(fext)

        # inverse dynamics: plain with external wrenches, with a flag, with the by-products
        same(e.rnea_host(hq, hqd, hqdd, host(nv), fext=hf), e.rnea(tq, tqd, tqdd, dnew(nv), fext=tf), "rnea_host")
        flags = _capi.RNEA_NO_CORIOLIS
        same(e.rnea_host(hq, hqd, hqdd, host(nv), flags=flags), e.rnea(tq, tqd, tqdd, dnew(nv), flags=flags), "rnea_host NO_CORIOLIS")
        ha, hw, da, dw = host(6 * nb), host(6 * nb), dnew(6 * nb), dnew(6 * nb)
        same(e.rnea_host(hq, hqd, hqdd, host(nv), fext=hf, body_acc=ha, joint_wrench=hw), e.rnea(tq, tqd, tqdd, dnew(nv), fext=tf, body_acc=da, joint_wrench=dw),
             "rnea_full_host tau")
        same(ha, da, "rnea_full_host body_acc")
        same(hw, dw, "rnea_full_host joint_wrench")

        # forward dynamics, plain and with joints in ACCELERATION_SOURCE mode
        same(e.aba_host(hq, hqd, htau, host(nv), fext=hf), e.aba(tq, tqd, ttau, dnew(nv), fext=tf), "aba_host")
        modes = np.zeros(nb, np.int32)
        modes[3::4] = 1
        e.set_joint_source_modes(modes)
        hto, dto = host(nv), dnew(nv)
        same(e.aba_sources_host(hq, hqd, htau, hqdd, host(nv), tau_out=hto, fext=hf), e.aba_sources(tq, tqd, ttau, tqdd, dnew(nv), tau_out=dto, fext=tf),
             "aba_sources_host qdd")
        same(hto, dto, "aba_sources_host tau_out")
        e.set_joint_source_modes(None)

        # mass matrix in every layout and copy-back case
        M = e.crba(tq, dnew(nv * nv)).cpu().numpy()
        same(e.crba_host(hq, host(nv * nv)), M, "crba_host entry-major")
        zero = ~M.any(axis=1)
        assert zero.any()
        kept = host(nv * nv, np.where(zero[:, None], 0.0, np.nan))
        same(e.crba_host(hq, kept, _capi.CRBA_ZEROS_PRESENT), M, "crba_host ZEROS_PRESENT")
        sm = np.full((n + 3, nv * nv), np.nan)
        if pinned:
            sm = torch.full((n + 3, nv * nv), float("nan"), dtype=torch.float64).pin_memory().numpy()
        e.crba_host(hq, sm[:n], _capi.CRBA_STATE_MAJOR)
        assert np.array_equal(sm[:n], M.T) and np.isnan(sm[n:]).all(), "crba_host state-major (pinned=%s)" % pinned
        rows = e.packed_size()
        same(e.crba_host(hq, host(rows), _capi.CRBA_PACKED), e.crba(tq, dnew(rows), _capi.CRBA_PACKED), "crba_host packed")

        # the fused step
        ht, hqo, hM = host(nv), host(nv), host(nv * nv)
        e.step_host(hq, hqd, qdd_in=hqdd, tau_in=htau, tau_out=ht, qdd_out=hqo, M=hM)
        same(ht, e.rnea(tq, tqd, tqdd, dnew(nv)), "step_host tau")
        same(hqo, e.aba(tq, tqd, ttau, dnew(nv)), "step_host qdd")
        same(hM, M, "step_host M")

        # the calls that used to stage synchronously
        hM, hC, dM, dC = host(nv * nv), host(nv * nv), dnew(nv * nv), dnew(nv * nv)
        e.coriolis(hq, hqd, hM, hC)
        e.coriolis(tq, tqd, dM, dC)
        same(hM, dM, "coriolis_host M")
        same(hC, dC, "coriolis_host C")
        ny = nv * 10 * nb
        same(e.joint_torque_regressor(hq, hqd, hqdd, host(ny)), e.joint_torque_regressor(tq, tqd, tqdd, dnew(ny)), "joint_torque_regressor_host")
        for frame in (_capi.FRAME_WORLD, _capi.FRAME_CENTER_OF_MASS):
            hM, hA, hc, dM, dA, dc = host(nv * nv), host(6 * nv), host(4), dnew(nv * nv), dnew(6 * nv), dnew(4)
            e.crba_centroidal(hq, hM, hA, hc, frame)
            e.crba_centroidal(tq, dM, dA, dc, frame)
            for h_, d_, what in ((hM, dM, "M"), (hA, dA, "cmm"), (hc, dc, "com")):
                same(h_, d_, "crba_centroidal_host %s frame %d" % (what, frame))
            ho, do = host(6), dnew(6)
            e.centroidal_convective_term(hq, hqd, hc, ho, frame)
            e.centroidal_convective_term(tq, tqd, dc, do, frame)
            same(ho, do, "centroidal_convective_term_host frame %d" % frame)
        hc, dc = host(4), dnew(4)
        e.center_of_mass(hq, hc)
        e.center_of_mass(tq, dc)
        same(hc, dc, "center_of_mass_host")

        # integration, in place
        iq, iqd, iqdd = host(nq, q), host(nv, qd), host(nv, qdd)
        # device matrices with an even ld: the integrator takes its paired-column path there (integrate.cu: vec2), as it does on
        # every chunk of the host path (a multiple of 256 states wide)
        jq, jqd, jqdd = (torch.zeros((x.shape[0], n + 1), dtype=torch.float64, device=dev) for x in (q, qd, qdd))
        for j_, x in ((jq, q), (jqd, qd), (jqdd, qdd)):
            j_[:, :n] = dv(x)
        jq, jqd, jqdd = jq[:, :n], jqd[:, :n], jqdd[:, :n]
        e.integrate_host(1e-3, iq, iqd, iqdd)
        e.integrate(1e-3, jq, jqd, jqdd)
        for h_, d_, what in ((iq, jq, "q"), (iqd, jqd, "qd"), (iqdd, jqdd, "qdd")):
            same(h_, d_, "integrate_host %s" % what)
    print("all host entry points match")


if __name__ == "__main__":
    _compare_all()
