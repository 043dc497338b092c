"""GPU test of the refusals of every device / host entry-point pair of the C ABI, on real handles of the H37 humanoid: the return
code and mecano_b200_last_error of bad shapes, NULL buffers, empty batches, unknown frames, a NaN step, fp32 handles on the
fp64-only calls, joints in ACCELERATION_SOURCE mode, an aliased tau_out and wrench ranks beyond the body count.  Both entry
points of a pair must refuse the same input in the same way, apart from the two differences stated below.

Every pointer a call receives is a real buffer of the call's shape (device memory for a device entry point, host memory for a
host one) or NULL; a call that passes its checks runs on those buffers."""
import ctypes

import numpy as np
import pytest

from mecano_b200 import _capi

pytestmark = pytest.mark.gpu

OK, INVALID, UNSUPPORTED, SHAPE = 0, -1, -2, -3
N_NEGATIVE = (SHAPE, "n_states must be >= 0")
LD_SHORT = (SHAPE, "ld must be >= n_states")
NULL_BUFFER = (INVALID, "NULL buffer")
NO_QDD_IN = (INVALID, "NULL buffer (qdd_in) with joints in ACCELERATION_SOURCE mode")
UNKNOWN_FRAME = (INVALID, "unknown centroidal momentum frame")
NO_COM = (INVALID, "the centre-of-mass frame needs the com rows of mecano_b200_crba_centroidal")
NAN_DT = (INVALID, "dt is NaN")
ABA_NEEDS_SOURCES = (INVALID, "joints in ACCELERATION_SOURCE mode need their accelerations: call mecano_b200_aba_sources")
FD_NEEDS_EFFORTS = (INVALID, "the forward-dynamics derivatives need every joint in EFFORT_SOURCE mode (mecano_b200_set_joint_source_modes)")
TAU_OUT_ALIAS = (INVALID, "tau_out must not alias tau when joints are in ACCELERATION_SOURCE mode")
FP64_ONLY = {
    "joint_torque_regressor": (UNSUPPORTED, "the joint-torque regressor is computed in fp64 only (mecano_b200_set_precision)"),
    "gravity_gradient": (UNSUPPORTED, "the gravity gradient is computed in fp64 only (mecano_b200_set_precision)"),
    "rnea_derivatives": (UNSUPPORTED, "the inverse-dynamics derivatives are computed in fp64 only (mecano_b200_set_precision)"),
    "aba_derivatives": (UNSUPPORTED, "the forward-dynamics derivatives are computed in fp64 only (mecano_b200_set_precision)"),
}
RANKS = {
    "joint_torque_regressor": (SHAPE, "joint-torque regressor: wrench_index ranks must be below n_bodies (one ten-column block per body)"),
    "gravity_gradient": (SHAPE, "gravity gradient: with external wrenches the wrench_index ranks must be below n_bodies (fext has 6 n_bodies rows)"),
    "rnea_derivatives": (SHAPE, "inverse-dynamics derivatives: with external wrenches the wrench_index ranks must be below n_bodies (fext has 6 n_bodies rows)"),
    "aba_derivatives": (SHAPE, "forward-dynamics derivatives: with external wrenches the wrench_index ranks must be below n_bodies (fext has 6 n_bodies rows)"),
}

# name: (host entry point, arguments after (handle, n, ld), required buffers); the device entry point is mecano_b200_<name> with
# the stream last.  flags / layout / frame / dt are scalars, every other argument a buffer.
CALLS = {
    "rnea": ("rnea_host", "q qd qdd fext tau flags", "q qd qdd tau"),
    "rnea_full": ("rnea_full_host", "q qd qdd fext tau body_acc joint_wrench flags", "q qd qdd tau"),
    "aba": ("aba_host", "q qd tau fext qdd flags", "q qd tau qdd"),
    "aba_sources": ("aba_sources_host", "q qd tau qdd_in fext qdd tau_out", "q qd tau qdd"),
    "crba": ("crba_host", "q M layout", "q M"),
    "crba_centroidal": ("crba_centroidal_host", "q M cmm com frame", "q M cmm com"),
    "center_of_mass": ("center_of_mass_host", "q com", "q com"),
    "centroidal_convective_term": ("centroidal_convective_term_host", "q qd com out frame", "q qd out"),
    "coriolis": ("coriolis_host", "q qd M C", "q qd M C"),
    "joint_torque_regressor": ("joint_torque_regressor_host", "q qd qdd Y", "q qd qdd Y"),
    "gravity_gradient": ("gravity_gradient_host", "q fext tau G", "q tau G"),
    "rnea_derivatives": ("rnea_derivatives_host", "q qd qdd fext tau dq dqd", "q qd qdd tau dq dqd"),
    "aba_derivatives": ("aba_derivatives_host", "q qd tau fext qdd dq dqd minv", "q qd tau qdd dq dqd minv"),
    "integrate": ("integrate_host", "dt q qd qdd", "q qd qdd"),
}
SIDES = ("device", "host")
N = 4


@pytest.fixture(scope="module")
def env():
    import torch

    import mecano_b200 as mb
    from test_gpu_parity import build

    assert torch.cuda.is_available(), "GPU tests need a CUDA device; the product has no CPU fallback"
    s, t = build(kind="humanoid", seed=7, n_joints=2)
    nq, nv, nb = t.nq, t.nv, t.nb
    lib = _capi.lib
    handles = []

    def create(desc_ref):
        h = ctypes.c_void_p()
        assert lib.mecano_b200_create(desc_ref, 0, ctypes.byref(h)) == 0, lib.mecano_b200_last_error(None)
        handles.append(h)
        return h

    plain = create(s.tables())
    fp32 = create(s.tables())
    assert lib.mecano_b200_set_precision(fp32, 1) == 0
    sources = create(s.tables())
    modes = np.zeros(nb, np.int32)
    modes[3::4] = 1
    assert lib.mecano_b200_set_joint_source_modes(sources, modes.ctypes.data) == 0
    # the body of rank nb - 1 takes rank nb: the ranks stay distinct, one of them is >= n_bodies
    desc = _capi.TreeDesc.from_buffer_copy(s.tables().contents)
    ranks = np.array([desc.wrench_index[i] for i in range(nb)], np.int32)
    ranks[ranks == nb - 1] = nb
    desc.wrench_index = ranks.ctypes.data_as(_capi.c_ip)
    wide = create(ctypes.byref(desc))

    rows = {"q": nq, "qd": nv, "qdd": nv, "tau": nv, "qdd_in": nv, "tau_out": nv, "fext": 6 * (nb + 1), "body_acc": 6 * nb,
            "joint_wrench": 6 * nb, "M": nv * nv, "C": nv * nv, "cmm": 6 * nv, "com": 4, "out": 6, "Y": 10 * nb * nv, "G": nv * nv,
            "dq": nv * nv, "dqd": nv * nv, "minv": nv * nv}
    q, qd, qdd, tau = mb.MultiBodySystemRandomTools.nextState(np.random.default_rng(3), s, N)
    state = {"q": q, "qd": qd, "qdd": qdd, "tau": tau, "qdd_in": qdd}
    bufs = {"host": {}, "device": {}}
    for name, r in rows.items():
        a = np.array(state[name]) if name in state else np.zeros((r, N))
        if name == "com":
            a[3] = 1.0  # a positive mass
        bufs["host"][name] = a
        bufs["device"][name] = torch.from_numpy(a.copy()).cuda()
    yield dict(torch=torch, lib=lib, plain=plain, fp32=fp32, sources=sources, wide=wide, bufs=bufs, keep=(s, ranks))
    torch.cuda.synchronize()
    for h in handles:
        lib.mecano_b200_destroy(h)


def call(env, name, side, handle="plain", n=N, ld=N, null=(), frame=0, dt=0.01, alias=None):
    """rc and last error of one entry point; `null`: buffers passed as NULL (every other one is real), `alias`: (a, b) passes
    buffer b's pointer for argument a."""
    lib, h = env["lib"], env[handle]
    host_name, params, _ = CALLS[name]
    null = null.split() if isinstance(null, str) else null
    bufs = env["bufs"][side]

    def ptr(p):
        if alias and p == alias[0]:
            p = alias[1]
        if p in null:
            return None
        b = bufs[p]
        return b.ctypes.data if side == "host" else b.data_ptr()

    scalars = {"flags": 0, "layout": 0, "frame": frame, "dt": dt}
    args = [scalars[p] if p in scalars else ptr(p) for p in params.split()]
    if side == "device":
        rc = getattr(lib, "mecano_b200_" + name)(h, n, ld, *args, None)
    else:
        rc = getattr(lib, "mecano_b200_" + host_name)(h, n, ld, *args)
    if rc == OK:
        return OK
    msg = lib.mecano_b200_last_error(h)
    return rc, msg.decode() if msg else None


def every_buffer(name):
    return CALLS[name][1].split()


def test_null_handle():
    for name, (host_name, params, _) in CALLS.items():
        scalars = {"flags": 0, "layout": 0, "frame": 0, "dt": 0.01}
        args = [scalars.get(p) for p in params.split()]
        assert getattr(_capi.lib, "mecano_b200_" + name)(None, 1, 1, *args, None) == INVALID, name
        assert getattr(_capi.lib, "mecano_b200_" + host_name)(None, 1, 1, *args) == INVALID, name


@pytest.mark.parametrize("name", list(CALLS))
def test_shapes_empty_batches_and_null_buffers(env, name):
    required = CALLS[name][2].split()
    for side in SIDES:
        assert call(env, name, side, n=-1, ld=N) == N_NEGATIVE, side
        assert call(env, name, side, n=N, ld=N - 1) == LD_SHORT, side
        assert call(env, name, side, n=0, ld=0, null=every_buffer(name)) == OK, side
        assert call(env, name, side) == OK, side
        for b in required:
            assert call(env, name, side, null=b) == NULL_BUFFER, (side, b)
    env["torch"].cuda.synchronize()


@pytest.mark.parametrize("side", SIDES)
def test_frames_and_dt(env, side):
    for name in ("crba_centroidal", "centroidal_convective_term"):
        assert call(env, name, side, frame=_capi.FRAME_CENTER_OF_MASS) == OK
        assert call(env, name, side, frame=2) == UNKNOWN_FRAME
        assert call(env, name, side, n=0, ld=0, null=every_buffer(name), frame=2) == OK
    assert call(env, "centroidal_convective_term", side, frame=_capi.FRAME_CENTER_OF_MASS, null="com") == NO_COM
    assert call(env, "centroidal_convective_term", side, frame=_capi.FRAME_WORLD, null="com") == OK
    # the NULL checks come first
    assert call(env, "crba_centroidal", side, frame=2, null="cmm") == NULL_BUFFER
    assert call(env, "centroidal_convective_term", side, frame=_capi.FRAME_CENTER_OF_MASS, null="com out") == NULL_BUFFER
    assert call(env, "integrate", side, dt=float("nan")) == NAN_DT
    assert call(env, "integrate", side, dt=float("nan"), null="qd") == NULL_BUFFER
    assert call(env, "integrate", side, n=0, ld=0, null=every_buffer("integrate"), dt=float("nan")) == OK
    env["torch"].cuda.synchronize()


@pytest.mark.parametrize("side", SIDES)
@pytest.mark.parametrize("name", list(FP64_ONLY))
def test_fp32_handle_on_fp64_only_calls(env, name, side):
    # refused before the empty-batch return and before the NULL checks
    assert call(env, name, side, handle="fp32") == FP64_ONLY[name]
    assert call(env, name, side, handle="fp32", n=0, ld=0, null=every_buffer(name)) == FP64_ONLY[name]
    assert call(env, name, side, handle="fp32", null="q") == FP64_ONLY[name]
    assert call(env, name, side, handle="fp32", n=-1) == N_NEGATIVE


def test_acceleration_sources(env):
    every = every_buffer("aba_sources")
    # the host entry point checks qdd_in ahead of everything else; the device entry point when it launches
    assert call(env, "aba_sources", "host", handle="sources", n=0, ld=0, null=every) == NO_QDD_IN
    assert call(env, "aba_sources", "device", handle="sources", n=0, ld=0, null=every) == OK
    assert call(env, "aba_sources", "host", handle="sources", n=-1, null="qdd_in") == NO_QDD_IN
    assert call(env, "aba_sources", "device", handle="sources", n=-1, null="qdd_in") == N_NEGATIVE
    assert call(env, "aba_sources", "host", handle="sources", null="q qdd_in") == NO_QDD_IN
    assert call(env, "aba_sources", "device", handle="sources", null="q qdd_in") == NULL_BUFFER
    for side in SIDES:
        assert call(env, "aba_sources", side, handle="sources", null="qdd_in") == NO_QDD_IN, side
        assert call(env, "aba_sources", side, handle="sources") == OK, side
        assert call(env, "aba_sources", side, handle="sources", null="tau_out") == OK, side
        assert call(env, "aba", side, handle="sources") == ABA_NEEDS_SOURCES, side
        assert call(env, "aba", side, handle="sources", n=0, ld=0, null=every_buffer("aba")) == OK, side
        assert call(env, "aba_derivatives", side, handle="sources") == FD_NEEDS_EFFORTS, side
        assert call(env, "aba_derivatives", side, handle="sources", n=0, ld=0, null=every_buffer("aba_derivatives")) == FD_NEEDS_EFFORTS, side
    # on the device tau_out may not be tau itself (the host stages them in different rows)
    assert call(env, "aba_sources", "device", handle="sources", alias=("tau_out", "tau")) == TAU_OUT_ALIAS
    assert call(env, "aba_sources", "device", alias=("tau_out", "tau")) == OK
    env["torch"].cuda.synchronize()


@pytest.mark.parametrize("side", SIDES)
def test_wrench_ranks_beyond_the_bodies(env, side):
    # the regressor has one ten-column block per rank: refused whatever the batch
    name = "joint_torque_regressor"
    assert call(env, name, side, handle="wide") == RANKS[name]
    assert call(env, name, side, handle="wide", n=0, ld=0, null=every_buffer(name)) == RANKS[name]
    # the others only with external wrenches, also on an empty batch, after the NULL checks
    for name in ("gravity_gradient", "rnea_derivatives", "aba_derivatives"):
        assert call(env, name, side, handle="wide") == RANKS[name], name
        assert call(env, name, side, handle="wide", null="fext") == OK, name
        assert call(env, name, side, handle="wide", n=0, ld=0, null=[b for b in every_buffer(name) if b != "fext"]) == RANKS[name], name
        assert call(env, name, side, handle="wide", n=0, ld=0, null=every_buffer(name)) == OK, name
        assert call(env, name, side, handle="wide", null="q") == NULL_BUFFER, name
    env["torch"].cuda.synchronize()
