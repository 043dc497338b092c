"""RNEA, ABA, CRBA, the Coriolis matrix and the joint-torque regressor at every launch configuration they can run, and the
body-parallel kernels (warp_kernels.cu, team_kernels.cu) at every team size.

The planner (kernels.cu: plan_thread_kernel) picks one entry of kCfg (thread_kernels.cuh) per tree and algorithm, so the suite
elsewhere sees only the configurations its trees happen to produce.  Here every entry is forced through MECANO_B200_CFG on the
16 trees of test_emulation: a configuration either is refused for a reason the table explains, or runs at exactly its block and
tensor-memory stack, at batch sizes around the block and across a persistent grid, and gives bit for bit what the planner's own
configuration gives (where the stack lives does not change the arithmetic; the Coriolis kernel only to rounding, ROUNDING_ONLY).  The planner's results are held to the kernels'
routines compiled for the host (tests/emu, 1e-12; ABA 1e-13 cond(M)) and to the C oracle (1e-9; ABA through its
equation-of-motion residual, the regressor through Y pi = tau).

The body-parallel kernels run a warp per state up to 32 bodies and a team of 32 ceil(nb / 32) threads up to 128; the trees below
give every team size, a last warp with one body and full teams, as a chain (deepest exchange) and as a floating base with a wide
tree (sibling rounds across warps).  Every batch is P base states tiled (state s is base state s % P), so the CPU reference work
does not grow with the batch."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

import emu_lib as el
import emu_regressor_lib as erl
import oracle_lib as ol
import treedesc as td
from test_derivatives_exact import P, cfg_table, per_state, torch_dev  # noqa: F401  (torch_dev: fixture)
from test_emulation import trees
from test_gravity_gradient import engine_of, structural_zeros
from test_regressor import model_params

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(HERE), "mecano_b200", "csrc")
N_TREES = 16
EMU_TOL = 1e-12      # against the kernels' routines compiled for the host (FMA contraction differs), per state
ABA_EMU_TOL = 1e-13  # ABA against the same, times cond2(M) of the state: deep chains amplify the contraction differences
ORACLE_TOL = 1e-9    # against the C oracle, per state (the suite's tolerance)
# ABA: |ID_oracle(q, qd, qdd) - tau| / max(1, |tau|, |M qdd|), the backward error, which does not depend on the conditioning (a
# state of the 60-body chain with cond2(M) = 6e4: 1.5e-8 relative to |tau| alone, 2.2e-12 as here)
RESIDUAL_TOL = 1e-10
PAD = 11             # ld = n + PAD; the columns beyond n start NaN and must stay NaN
ALGOS = ("rnea", "aba", "crba", "cor", "reg")
ALGO_ID = {"rnea": 0, "aba": 1, "crba": 2, "cor": 3, "reg": 4}  # program.h: MbAlgo
CALLS = {
    "rnea": ("rnea", "rnea_fext", "rnea_no_coriolis", "rnea_no_accelerations", "rnea_full"),
    "aba": ("aba", "aba_fext"),
    "crba": ("crba", "crba_state_major", "crba_packed", "crba_centroidal"),
    "cor": ("cor",),
    "reg": ("reg",),
}
RNEA_FLAGS = {"rnea": 0, "rnea_fext": 0, "rnea_no_coriolis": 1, "rnea_no_accelerations": 2}
# Every configuration gives the planner's bits, except the Coriolis kernel (coriolis.cuh: 255 registers, spilling): ptxas contracts
# its multiplies and adds into FMAs differently under the register budget of each block (cuobjdump -sass: the 192-thread
# instantiation holds 1347 DFMA, the 320- and 384-thread ones 1379, those of 32 to 256 threads 1350).  Measured on a B200: up to
# 1.4e-13 apart.  Its configurations must agree with the planner's per state to EMU_TOL instead.
ROUNDING_ONLY = ("cor",)


def algo_table():
    """{MECANO_B200_CFG key: (wide_stack, thread_only)} of mb_algo in program.h."""
    text = open(os.path.join(CSRC, "program.h")).read()
    return {k: (w == "true", o == "true") for k, w, o in re.findall(r'return \{"(\w+)", \d+, (true|false), (true|false)', text)}


def partial_tm_block():
    return int(re.search(r"#define MB_PARTIAL_TM_BLOCK (\d+)", open(os.path.join(CSRC, "program.h")).read()).group(1))


def counter_ring():
    return int(re.search(r"#define MB_COUNTERS (\d+)", open(os.path.join(CSRC, "api.cu")).read()).group(1))


def wide_stack_slots(t, algo):
    """The wide stack area (double2 slots per state) of one algorithm's flattened program (tests/emu/emu_layout.cpp)."""
    out = os.path.join(HERE, "emu", "libmecano_emu_layout.so")
    deps = [os.path.join(HERE, "emu", "emu_layout.cpp")] + [os.path.join(CSRC, f) for f in ("flatten.cpp", "flatten.h", "program.h")]
    if not os.path.exists(out) or any(os.path.getmtime(out) < os.path.getmtime(f) for f in deps):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-x", "c++", deps[0], deps[1], "-o", out])
    d, keep, _ = el.tree_desc_c(t)  # keep: the arrays d points into
    wide, narrow = ctypes.c_int(), ctypes.c_int()
    assert ctypes.CDLL(out).emu_stack_areas(ctypes.byref(d), algo, ctypes.byref(wide), ctypes.byref(narrow)) == 0
    return wide.value


def tm_fits(wide, wstack2, block, tm):
    """program.h: mb_tm_fits -- the wide stack area fits the tensor-memory slots, or the block keeps the deeper slots in shared
    memory."""
    return tm == 0 or (wide and (wstack2 <= tm or block == partial_tm_block()))


def check_refusals(table, ran, refused, wide, wstack2):
    """The refusals are the configurations that cannot fit.  Shared memory and registers per block grow with the block and, for
    the tensor-memory configurations, shrink with the slots held in tensor memory: a configuration j that ran 'covers' i when it
    needs at least as much of both (same stack kind, block_j >= block_i, tm_j <= tm_i)."""
    for j in ran:
        assert tm_fits(wide, wstack2, *[table[j][k] for k in (0, 2)]), ("ran without fitting the tensor-memory stack", j)

    def covers(j, i):
        (bi, _, ti), (bj, _, tj) = table[i], table[j]
        return bj >= bi and (tj > 0) == (ti > 0) and tj <= ti

    for i in refused:
        block, cls, tm = table[i]
        if not tm_fits(wide, wstack2, block, tm):
            continue  # no wide stack, or a wide area deeper than the tensor-memory slots of that block
        # within one work-area class the refused configuration needs more than every one that ran
        assert not [j for j in ran if table[j][1] == cls and covers(j, i)], ("refused, but a larger one of its class ran", i)
        # a class-0 configuration refused while a class-1 one that needs as much runs is refused for its work areas: then no
        # class-0 configuration runs at all
        if cls == 0 and any(table[j][1] == 1 and covers(j, i) for j in ran):
            assert not [j for j in ran if table[j][1] == 0], ("class 0 refused for its work areas, yet one ran", i)


# ---------------------------------------------------------------------------------------------------------------- states and references


def thread_case(idx):
    rng = np.random.default_rng(8100 + idx)
    t = trees(rng)[idx]
    g = (rng.uniform(-1, 1), rng.uniform(-1, 1), -rng.uniform(1, 10))
    q, qd, qdd, tau = td.random_states(rng, t, P)
    qd[:, 1] = 0.0
    qdd[:, 2] = 0.0
    fext = rng.uniform(-1, 1, size=(t.nb, 6, P))
    return t, g, (q, qd, qdd, tau, fext)


def regressor_zeros(t):
    """Boolean [nv, nb]: joint row i does not support body b (b is not in the subtree of the joint's body)."""
    body = np.empty(t.nv, dtype=np.int64)
    for b in range(t.nb):
        body[t.dof_off[b]:t.dof_off[b] + td.NDOF[int(t.jtype[b])]] = b
    z = np.ones((t.nv, t.nb), bool)
    for b in range(t.nb):
        a = b
        while a >= 0:
            z[body == a, b] = False
            a = int(t.parent[a])
    return z


def residual(o, Mo, q, qd, qdd, tau, fext_rows):
    """Worst equation-of-motion residual of forward dynamics over the states: |ID_oracle(q, qd, qdd) - tau| relative to the
    larger of the terms that cancel in it (max(1, |tau|, |M qdd|))."""
    qdd = np.ascontiguousarray(qdd)
    r = np.abs(o.rnea_batch(q, qd, qdd, fext_rows) - tau).max(axis=0)
    scale = np.maximum(np.maximum(1.0, np.abs(tau).max(axis=0)), np.abs(np.einsum("ijs,js->is", Mo, qdd)).max(axis=0))
    return float(np.max(r / scale))


class References:
    """Per call, on the P base states and in the row order of the device outputs: the emulated routines and the oracle."""

    def __init__(self, t, g, states, order):
        q, qd, qdd, tau, fext = states
        nv, nb = t.nv, t.nb
        self.t, self.g, self.states, self.order = t, g, states, order
        emu, o = el.Emu(t, gravity=g), ol.Oracle(t, gravity=g)
        self.oracle = o
        fo = np.ascontiguousarray(fext.reshape(6 * nb, P))  # tree order (oracle)
        desc = lambda a: np.ascontiguousarray(a[order].reshape(6 * nb, P))  # noqa: E731  (bodies of the C description)
        self.Mo = o.crba_batch(q)
        self.cond = np.array([np.linalg.cond(self.Mo[:, :, s]) for s in range(P)])
        self.emu = {name: [emu.rnea(q, qd, qdd, fext if name == "rnea_fext" else None, flags=f)] for name, f in RNEA_FLAGS.items()}
        self.oracle_ref = {name: [o.rnea_batch(q, qd, qdd, fo if name == "rnea_fext" else None, flags=f)] for name, f in RNEA_FLAGS.items()}
        tau_f, acc, wr = emu.rnea_full(q, qd, qdd, fext)
        self.emu["rnea_full"] = [tau_f, desc(acc), desc(wr)]
        full = [o.rnea_full(q[:, s], qd[:, s], qdd[:, s], np.ascontiguousarray(fext[:, :, s])) for s in range(P)]
        self.oracle_ref["rnea_full"] = [np.stack([f[0] for f in full], -1), desc(np.stack([f[1] for f in full], -1)), desc(np.stack([f[2] for f in full], -1))]
        self.emu["aba"] = [emu.aba(q, qd, tau)]
        self.emu["aba_fext"] = [emu.aba(q, qd, tau, fext)]
        M = emu.crba(q).reshape(nv * nv, P)
        self.emu["crba"] = self.emu["crba_state_major"] = [M]
        self.oracle_ref["crba"] = self.oracle_ref["crba_state_major"] = [self.Mo.reshape(nv * nv, P)]
        self.emu["crba_packed"] = [emu.crba_packed(q)]
        self.packed = emu.packed_index()
        self.oracle_ref["crba_packed"] = [self.Mo[self.packed[0], self.packed[1]]]
        Mc, cmm, com = emu.crba_centroidal(q)
        self.emu["crba_centroidal"] = [Mc.reshape(nv * nv, P), cmm.reshape(6 * nv, P), np.vstack([com[:3] / com[3], com[3:]])]
        cen = [o.crba_centroidal(q[:, s], 0) for s in range(P)]
        self.oracle_ref["crba_centroidal"] = [self.Mo.reshape(nv * nv, P), np.stack([c[1] for c in cen], -1).reshape(6 * nv, P),
                                              np.stack([np.append(c[2], c[3]) for c in cen], -1)]
        Mk, Ck = emu.coriolis(q, qd)
        self.emu["cor"] = [Mk.reshape(nv * nv, P), Ck.reshape(nv * nv, P)]
        cor = [o.coriolis(q[:, s], qd[:, s]) for s in range(P)]
        self.oracle_ref["cor"] = [np.stack([c[0] for c in cor], -1).reshape(nv * nv, P), np.stack([c[1] for c in cor], -1).reshape(nv * nv, P)]
        Y = erl.regressor(t, g, q, qd, qdd)
        self.emu["reg"] = [np.ascontiguousarray(Y.reshape(nv, nb, 10, P)[:, order].reshape(nv * 10 * nb, P))]
        self.pi_desc = model_params(t).reshape(nb, 10)[order].ravel()
        self.tau_plain = self.oracle_ref["rnea"][0]
        self.mzero = structural_zeros(t).ravel()
        self.yzero = np.repeat(regressor_zeros(t)[:, order], 10, axis=1).ravel()

    def check(self, name, outs):
        """The outputs of one call on the P base states (numpy [rows, P]) against both references; returns the worst error
        against (emulated routine, oracle)."""
        nv = self.t.nv
        for D in outs:
            assert not np.isnan(D).any(), "%s: every entry must be written" % name
        zeros = {"crba": [self.mzero], "crba_state_major": [self.mzero], "crba_centroidal": [self.mzero, None, None],
                 "cor": [self.mzero, self.mzero], "reg": [self.yzero]}.get(name, [])
        for D, z in zip(outs, zeros):
            if z is not None:
                assert np.all((D[z] == 0.0) & ~np.signbit(D[z])), "%s: structural zeros are +0.0" % name
        q, qd, _, tau, fext = self.states
        if name.startswith("aba"):
            err = np.abs(outs[0] - self.emu[name][0]).max(axis=0) / np.maximum(1.0, np.abs(self.emu[name][0]).max(axis=0))
            assert np.all(err <= ABA_EMU_TOL * self.cond), (name, float(np.max(err / self.cond)))
            fo = np.ascontiguousarray(fext.reshape(6 * self.t.nb, P)) if name == "aba_fext" else None
            res = residual(self.oracle, self.Mo, q, qd, outs[0], tau, fo)
            assert res < RESIDUAL_TOL, (name, res)
            return float(np.max(err / self.cond)), res
        w_emu = max(per_state(D, R) for D, R in zip(outs, self.emu[name]))
        assert w_emu < EMU_TOL, (name, w_emu)
        if name == "reg":
            Ypi = np.einsum("icn,c->in", outs[0].reshape(nv, -1, P), self.pi_desc)
            w_o = per_state(Ypi, self.tau_plain)
        else:
            w_o = max(per_state(D, R) for D, R in zip(outs, self.oracle_ref[name]))
        assert w_o < ORACLE_TOL, (name, w_o)
        return w_emu, w_o


# ---------------------------------------------------------------------------------------------------------------- device helpers


def tiled_inputs(torch, dev, base, n):
    """The base states ([rows, P] device tensors) tiled to n states, as [rows, n] views of NaN-padded [rows, n + PAD] buffers."""
    cols = torch.arange(n, device=dev) % P
    out = {}
    for k, v in base.items():
        buf = torch.full((v.shape[0], n + PAD), float("nan"), dtype=torch.float64, device=dev)
        buf[:, :n] = v[:, cols]
        out[k] = buf[:, :n]
    return out, cols


def run_call(name, e, t, x, n, torch, dev):
    """One call on tiled inputs; its outputs as [rows, n] views, after checking that nothing beyond n was written."""
    from mecano_b200 import _capi

    nv, nb = t.nv, t.nb
    new = lambda rows: torch.full((rows, n + PAD), float("nan"), dtype=torch.float64, device=dev)  # noqa: E731
    if name == "crba_state_major":
        M = torch.full((n + PAD, nv * nv), float("nan"), dtype=torch.float64, device=dev)
        e.crba(x["q"], M[:n], _capi.CRBA_STATE_MAJOR)
        assert bool(torch.isnan(M[n:]).all()), "%s: states beyond n were written" % name
        return [M[:n].t()]
    if name in RNEA_FLAGS:
        outs = [new(nv)]
        e.rnea(x["q"], x["qd"], x["qdd"], outs[0][:, :n], fext=x["fext"] if name == "rnea_fext" else None, flags=RNEA_FLAGS[name])
    elif name == "rnea_full":
        outs = [new(nv), new(6 * nb), new(6 * nb)]
        e.rnea(x["q"], x["qd"], x["qdd"], outs[0][:, :n], fext=x["fext"], body_acc=outs[1][:, :n], joint_wrench=outs[2][:, :n])
    elif name in ("aba", "aba_fext"):
        outs = [new(nv)]
        e.aba(x["q"], x["qd"], x["tau"], outs[0][:, :n], fext=x["fext"] if name == "aba_fext" else None)
    elif name == "crba":
        outs = [new(nv * nv)]
        e.crba(x["q"], outs[0][:, :n])
    elif name == "crba_packed":
        outs = [new(e.packed_size())]
        e.crba(x["q"], outs[0][:, :n], _capi.CRBA_PACKED)
    elif name == "crba_centroidal":
        outs = [new(nv * nv), new(6 * nv), new(4)]
        e.crba_centroidal(x["q"], *(o[:, :n] for o in outs))
    elif name == "cor":
        outs = [new(nv * nv), new(nv * nv)]
        e.coriolis(x["q"], x["qd"], *(o[:, :n] for o in outs))
    else:
        outs = [new(nv * 10 * nb)]
        e.joint_torque_regressor(x["q"], x["qd"], x["qdd"], outs[0][:, :n])
    for o in outs:
        assert bool(torch.isnan(o[:, n:]).all()), "%s: columns beyond n were written" % name
    return [o[:, :n] for o in outs]


def device_base(torch, dev, states, order):
    q, qd, qdd, tau, fext = states
    nb = fext.shape[0]
    fo = np.ascontiguousarray(fext[order].reshape(6 * nb, P))
    return {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in (("q", q), ("qd", qd), ("qdd", qdd), ("tau", tau), ("fext", fo))}


def open_forced(monkeypatch, t, g, setting):
    """A handle with MECANO_B200_CFG = setting (None: the planner's choice), thread-per-state; None if creation is refused with
    MECANO_B200_ERR_TOO_LARGE."""
    import mecano_b200 as mb

    if setting is not None:
        monkeypatch.setenv("MECANO_B200_CFG", setting)
    try:
        e, _ = engine_of(t, g)
    except mb._capi.MecanoB200Error as err:
        assert err.code == -5, (setting, str(err))  # MECANO_B200_ERR_TOO_LARGE
        return None
    finally:
        monkeypatch.delenv("MECANO_B200_CFG", raising=False)
    e.set_variant(1)
    return e


# ---------------------------------------------------------------------------------------------------------------- CPU


def test_tables_parse():
    table = cfg_table()
    algos = algo_table()
    assert set(ALGOS) <= set(algos)
    assert [k for k in ALGOS if algos[k][0]] == ["rnea", "aba"], "RNEA and ABA are the algorithms with a wide (TMEM-capable) stack"
    assert [k for k in ALGOS if algos[k][1]] == ["cor", "reg"]
    assert any(b == partial_tm_block() and tm > 0 for b, _, tm in table), "the partial-TMEM configuration is compiled"
    assert counter_ring() >= 2
    # the spill-over of the partial-TMEM block is reached: some test trees have a wide area deeper than its tensor-memory slots
    rng_trees = [trees(np.random.default_rng(8100 + i))[i] for i in range(N_TREES)]
    partial_tm = [tm for b, _, tm in table if b == partial_tm_block()][0]
    assert sum(wide_stack_slots(t, 0) > partial_tm for t in rng_trees) >= 2


@pytest.mark.parametrize("idx", range(N_TREES))
def test_references_of_every_call_agree(idx):
    """The two references agree with each other on the states the GPU tests use (so a GPU failure is the kernel's), and the
    structural zeros of the mass matrix, the Coriolis matrix and the regressor are +0.0 in the emulated routines."""
    t, g, states = thread_case(idx)
    _, _, order = el.tree_desc_c(t)
    ref = References(t, g, states, order)
    for name in sum(CALLS.values(), ()):
        ref.check(name, ref.emu[name])


# ---------------------------------------------------------------------------------------------------------------- GPU: thread per state


@pytest.mark.gpu
@pytest.mark.parametrize("idx", range(N_TREES))
def test_thread_kernels_at_every_launch_configuration(torch_dev, monkeypatch, idx):
    """For each kCfg entry forced for RNEA, ABA, CRBA, Coriolis and regressor: refused with MECANO_B200_ERR_TOO_LARGE for a
    reason the table gives (check_refusals), or run at exactly its block and tensor-memory slots.  Each configuration that runs:
    n = 1, block - 1, block + 1 and a large batch (RNEA / ABA: beyond one wave of the grid, so that the persistent grid draws
    from its counter; the others: two tiles and a ragged one), every call of CALLS, ld = n + 11 with the tail left NaN; every
    output bit for bit what the planner's configuration gives on the same base state (Coriolis: to rounding, ROUNDING_ONLY), and
    that checked against the emulated routines and the oracle."""
    import mecano_b200 as mb

    torch, dev = torch_dev
    table = cfg_table()
    algos = algo_table()
    t, g, states = thread_case(idx)
    _, _, order = el.tree_desc_c(t)
    ref = References(t, g, states, order)
    wstack2 = {k: wide_stack_slots(t, ALGO_ID[k]) for k in ("rnea", "aba")}
    base = device_base(torch, dev, states, order)

    # the planner's configuration: the results every forced configuration must reproduce
    e = open_forced(monkeypatch, t, g, None)
    assert e is not None
    planned = {k: e.kernel_info(ALGO_ID[k], 1 << 16) for k in ALGOS}
    x, _ = tiled_inputs(torch, dev, base, P)
    canon, worst = {}, {}
    for k in ALGOS:
        for name in CALLS[k]:
            outs = run_call(name, e, t, x, P, torch, dev)
            canon[name] = [o.clone() for o in outs]
            worst[name] = ref.check(name, [o.cpu().numpy() for o in outs])
    assert np.array_equal(np.stack(e.packed_index()), np.stack(ref.packed))
    e.close()

    ran = {k: {} for k in ALGOS}
    refused = {k: [] for k in ALGOS}
    differ = []
    rounding = 0.0  # worst per-state difference of a ROUNDING_ONLY kernel from the planner's configuration
    for i, (block, cls, tm) in enumerate(table):
        handles = {}
        every = ",".join("%s=%d" % (k, i) for k in ALGOS)
        e = open_forced(monkeypatch, t, g, every)
        if e is not None:
            handles = {k: e for k in ALGOS}
        else:
            # one of the algorithms with a generic form refuses at handle creation: find which, one handle each
            for k in ("rnea", "aba", "crba"):
                h = open_forced(monkeypatch, t, g, "%s=%d" % (k, i))
                if h is None:
                    refused[k].append(i)
                else:
                    handles[k] = h
            h = open_forced(monkeypatch, t, g, "cor=%d,reg=%d" % (i, i))
            assert h is not None
            handles["cor"] = handles["reg"] = h
        for k, h in handles.items():
            info = h.kernel_info(ALGO_ID[k], 1 << 16)
            if info["block_threads"] == 0:
                assert algos[k][1], (k, i, "only a thread-only kernel may be refused after handle creation")
                with pytest.raises(mb._capi.MecanoB200Error) as err:
                    run_call(CALLS[k][0], h, t, tiled_inputs(torch, dev, base, 64)[0], 64, torch, dev)
                assert err.value.code == -5, (k, i, str(err.value))  # MECANO_B200_ERR_TOO_LARGE
                refused[k].append(i)
                continue
            assert info["variant"] == 1 and info["block_threads"] == block, (k, i, info)
            assert info["tmem_stack_slots"] == (tm if algos[k][0] else 0), (k, i, info)
            ran[k][i] = info
        sizes = {}
        for k in ran:
            if i not in ran[k]:
                continue
            info = ran[k][i]
            big = info["sm_count"] * info["blocks_per_sm"] * block + 37 if k in ("rnea", "aba") else 2 * block + (block + 1) // 2
            for n in (1, block - 1, block + 1, big):
                sizes.setdefault(n, []).append(k)
        for n, ks in sorted(sizes.items()):
            x, cols = tiled_inputs(torch, dev, base, n)
            for k in ks:
                for name in CALLS[k]:
                    outs = run_call(name, handles[k], t, x, n, torch, dev)
                    for o, c in zip(outs, canon[name]):
                        if name in ROUNDING_ONLY and not bool(torch.isnan(o).any()):
                            r = c[:, cols]
                            w = ((o - r).abs().amax(dim=0) / r.abs().amax(dim=0).clamp(min=1.0)).max().item()
                            rounding = max(rounding, w)
                            if w <= EMU_TOL:
                                continue
                        if not torch.equal(o, c[:, cols]):
                            d = (o - c[:, cols]).abs()
                            differ.append((name, i, n, float(d[~torch.isnan(d)].max()) if bool((~torch.isnan(d)).any()) else float("nan"),
                                           int(torch.isnan(o).sum())))
                    del outs
            del x
        for h in {id(h): h for h in handles.values()}.values():
            h.close()

    for k in ALGOS:
        assert ran[k], "%s: no configuration runs" % k
        check_refusals(table, ran[k], refused[k], algos[k][0], wstack2.get(k, 0))
        keys = ("block_threads", "blocks_per_sm", "regs_per_thread", "local_bytes_per_thread", "dynamic_smem_bytes", "tmem_stack_slots")
        assert any(all(planned[k][x] == info[x] for x in keys) for info in ran[k].values()), (k, planned[k])
    print("\ntree %d (nb %d, nv %d, wide stack rnea %d / aba %d slots)" % (idx, t.nb, t.nv, wstack2["rnea"], wstack2["aba"]))
    for k in ALGOS:
        print("  %-4s ran %s refused %s" % (k, sorted(ran[k]), sorted(refused[k])))
    print("  worst against the emulated routines %.1e (ABA, per cond2(M): %.1e), against the oracle %.1e (ABA residual %.1e)" % (
        max(v[0] for n, v in worst.items() if not n.startswith("aba")), max(worst["aba"][0], worst["aba_fext"][0]),
        max(v[1] for n, v in worst.items() if not n.startswith("aba")), max(worst["aba"][1], worst["aba_fext"][1])))
    print("  every other configuration bit for bit the planner's, Coriolis within %.1e" % rounding)
    assert not differ, "outputs that differ from the planner's configuration (call, cfg, n, max |diff|, NaNs): %s" % differ[:20]


@pytest.mark.gpu
def test_persistent_work_counters_across_the_ring(torch_dev):
    """The warps of a persistent grid draw their states from a counter pair that the last warp to run dry re-arms for the next
    launch that uses it (gpu_ctx.cuh: thread_block_run); a handle cycles through a ring of MB_COUNTERS pairs.  Every pair is used
    at least three times here -- first from the zeroed allocation, then twice after a re-arm -- by RNEA and ABA on persistent
    grids: each launch bit for bit the first, into a NaN-filled buffer."""
    torch, dev = torch_dev
    rng = np.random.default_rng(37)
    t = td.humanoid(rng, 2)
    g = (0.3, -0.2, -9.81)
    e, order = engine_of(t, g)
    e.set_variant(1)
    launches = 2 * counter_ring() + 1
    q, qd, qdd, tau = td.random_states(rng, t, P)
    base = {k: torch.from_numpy(v).to(dev) for k, v in (("q", q), ("qd", qd), ("qdd", qdd), ("tau", tau))}
    n = None
    for k in ("rnea", "aba"):
        info = e.kernel_info(ALGO_ID[k], 1 << 16)
        assert info["tmem_stack_slots"] > 0, (k, info)  # a persistent grid that draws from the counters
        size = info["sm_count"] * info["blocks_per_sm"] * info["block_threads"] + 37
        n = size if n is None else max(n, size)
    x, _ = tiled_inputs(torch, dev, base, n)
    x["fext"] = None
    first = {}
    for it in range(launches):
        for name in ("rnea", "aba"):
            out = run_call(name, e, t, x, n, torch, dev)[0]
            if it == 0:
                assert not bool(torch.isnan(out).any()), name
                first[name] = out
            else:
                assert torch.equal(out, first[name]), (name, it, int(torch.isnan(out).sum()))
    e.close()


# ---------------------------------------------------------------------------------------------------------------- body-parallel kernels

BODY_COUNTS = (1, 2, 31, 32, 33, 63, 64, 65, 95, 96, 97, 127, 128)
SHAPES = ("chain", "floating")
# A handle also plans the thread-per-state kernels and refuses a tree whose stack does not fit a 32-state block in shared memory
# (MECANO_B200_ERR_TOO_LARGE): a single chain of 95 bodies already, although the team kernels take 128 bodies of any depth
CHAIN_DEPTH = 64


def body_parallel_tree(shape, nb):
    """One-DoF and SixDoF joints only (warp_variant_supports).  chain: revolute / prismatic joints in series, the deepest
    exchange: one chain up to CHAIN_DEPTH bodies, beyond that a second chain from the fixed base.  floating: a SixDoF
    root; half of the other bodies hang off the root, each of the rest off one of those -- a root with nb // 2 children spread
    over the warps of the team."""
    rng = np.random.default_rng(9100 + 2 * nb + (shape == "floating"))
    one_dof = lambda m: [td.PRISMATIC if rng.uniform() < 0.3 else td.REVOLUTE for _ in range(m)]  # noqa: E731
    if shape == "chain":
        parent = [b - 1 for b in range(min(nb, CHAIN_DEPTH))] + [-1 if b == CHAIN_DEPTH else b - 1 for b in range(CHAIN_DEPTH, nb)]
        return td.make_tree(rng, parent, one_dof(nb))
    first = nb // 2  # children of the root
    parent = [-1] + [0] * first + [1 + k for k in range(nb - 1 - first)]
    return td.make_tree(rng, parent, [td.SIXDOF] + one_dof(nb - 1))


def team_threads(nb):
    return 128 if nb <= 32 else 32 * -(-nb // 32)  # warp kernels: four states of a warp each per 128-thread block


def test_body_parallel_trees_cover_every_team_size():
    """The builders give the body counts, team sizes, joint types and shapes that the GPU tests are meant to cover."""
    teams = set()
    for shape in SHAPES:
        for nb in BODY_COUNTS:
            t = body_parallel_tree(shape, nb)
            assert t.nb == nb and set(t.jtype.tolist()) <= {td.REVOLUTE, td.PRISMATIC, td.SIXDOF}
            children = np.bincount(t.parent[t.parent >= 0], minlength=nb)
            depth = np.zeros(nb, int)
            for b in range(nb):
                depth[b] = 0 if t.parent[b] < 0 else depth[t.parent[b]] + 1
            if shape == "chain":
                assert depth.max() == min(nb, CHAIN_DEPTH) - 1 and children.max() <= 2 and (t.jtype != td.SIXDOF).all()
            else:
                assert t.jtype[0] == td.SIXDOF and (t.jtype[1:] != td.SIXDOF).all() and depth.max() <= 2
                assert children.max() == nb // 2
            if nb > 32:
                teams.add((team_threads(nb), nb % 32))
    assert {T for T, _ in teams} == {64, 96, 128}
    assert {T for T, r in teams if r == 1} == {64, 96, 128}, "a last warp holding one body, in every team size"
    assert {T for T, r in teams if r == 0} == {64, 96, 128}, "full teams"
    assert max(BODY_COUNTS) == 128  # MB_MAX_BODIES


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("nb", BODY_COUNTS)
def test_body_parallel_trees_emulated(shape, nb):
    """The kernels' routines on these trees against the oracle (the trees are well posed for the GPU tests' bounds)."""
    t = body_parallel_tree(shape, nb)
    rng = np.random.default_rng(nb)
    q, qd, qdd, tau = td.random_states(rng, t, 4)
    e, o = el.Emu(t), ol.Oracle(t)
    assert per_state(e.rnea(q, qd, qdd), o.rnea_batch(q, qd, qdd)) < ORACLE_TOL
    assert per_state(e.aba(q, qd, tau), o.aba_batch(q, qd, tau)) < ORACLE_TOL
    assert per_state(e.crba(q).reshape(t.nv ** 2, -1), o.crba_batch(q).reshape(t.nv ** 2, -1)) < ORACLE_TOL


WARP_CALLS = ("rnea", "rnea_fext", "rnea_no_coriolis", "aba", "aba_fext", "crba", "crba_state_major")


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("nb", BODY_COUNTS)
def test_body_parallel_kernels_at_every_team_size(torch_dev, shape, nb):
    """The warp variant at n = 1, 2, 333 and a batch larger than the grid of warps / teams (so that they loop), ld = n + 11 with
    the tail left NaN: every state bit for bit its base state's result, which is held to the oracle (ABA by its residual) and to
    the thread-per-state kernel of the same handle (1e-12, ABA 1e-13 cond2(M)); the dense mass matrix again with ZEROS_PRESENT
    into the same buffer with every structurally non-zero entry poisoned.  Then AUTO on both sides of its threshold: warp below,
    thread from it on, each bit for bit its variant's results."""
    from mecano_b200 import _capi

    torch, dev = torch_dev
    t = body_parallel_tree(shape, nb)
    rng = np.random.default_rng(9300 + nb)
    g = (rng.uniform(-1, 1), rng.uniform(-1, 1), -rng.uniform(1, 10))
    q, qd, qdd, tau = td.random_states(rng, t, P)
    fext = rng.uniform(-1, 1, size=(t.nb, 6, P))
    states = (q, qd, qdd, tau, fext)
    e, order = engine_of(t, g)
    base = device_base(torch, dev, states, order)
    o = ol.Oracle(t, gravity=g)
    fo = np.ascontiguousarray(fext.reshape(6 * nb, P))
    Mo = o.crba_batch(q)
    cond = np.array([np.linalg.cond(Mo[:, :, s]) for s in range(P)])
    nv = t.nv

    def results(variant):
        e.set_variant(variant)
        x, _ = tiled_inputs(torch, dev, base, P)
        return {name: run_call(name, e, t, x, P, torch, dev)[0].clone() for name in WARP_CALLS}

    thread, warp = results(1), results(2)
    for k in ("rnea", "aba", "crba"):
        info = e.kernel_info(ALGO_ID[k], 1 << 16)
        assert info["variant"] == 2 and info["block_threads"] == team_threads(nb), (k, info)
    worst = [0.0, 0.0]
    for name in WARP_CALLS:
        W, T = warp[name].cpu().numpy(), thread[name].cpu().numpy()
        assert not np.isnan(W).any(), name
        if name.startswith("aba"):
            err = np.abs(W - T).max(axis=0) / np.maximum(1.0, np.abs(T).max(axis=0))
            assert np.all(err <= ABA_EMU_TOL * cond), (name, float(np.max(err / cond)))
            res = residual(o, Mo, q, qd, W, tau, fo if name == "aba_fext" else None)
            assert res < RESIDUAL_TOL, (name, res)
            worst = [max(worst[0], float(np.max(err / cond))), max(worst[1], res)]
            continue
        if name.startswith("crba"):
            R = Mo.reshape(nv * nv, P)
            z = structural_zeros(t).ravel()
            assert np.all((W[z] == 0.0) & ~np.signbit(W[z])), name
        else:
            R = o.rnea_batch(q, qd, qdd, fo if name == "rnea_fext" else None, flags=RNEA_FLAGS[name])
        w_t, w_o = per_state(W, T), per_state(W, R)
        assert w_t < EMU_TOL and w_o < ORACLE_TOL, (name, w_t, w_o)
        worst = [max(worst[0], w_t), max(worst[1], w_o)]

    e.set_variant(2)
    info = e.kernel_info(0, 1 << 16)
    grid_states = info["sm_count"] * 64  # more than either body-parallel grid holds at once (warps: 16 blocks of 4 per SM)
    for n in (1, 2, 333, grid_states + 37):
        x, cols = tiled_inputs(torch, dev, base, n)
        for name in WARP_CALLS:
            out = run_call(name, e, t, x, n, torch, dev)[0]
            assert torch.equal(out, warp[name][:, cols]), (name, n, int(torch.isnan(out).sum()))
        # ZEROS_PRESENT: the structural zeros of the previous call stay, everything else is written again
        M = torch.full((nv * nv, n + PAD), float("nan"), dtype=torch.float64, device=dev)
        e.crba(x["q"], M[:, :n])
        z = torch.from_numpy(structural_zeros(t).ravel()).to(dev)
        M[~z, :n] = float("nan")
        e.crba(x["q"], M[:, :n], _capi.CRBA_ZEROS_PRESENT)
        assert bool(torch.isnan(M[:, n:]).all()) and torch.equal(M[:, :n], warp["crba"][:, cols]), ("zeros present", n)
        del x

    # AUTO: warp-per-state below the threshold, thread-per-state from it on
    e.set_variant(0)
    for k, name in (("rnea", "rnea"), ("aba", "aba"), ("crba", "crba")):
        lo, hi = 1, 1 << 24
        assert e.kernel_info(ALGO_ID[k], lo)["variant"] == 2 and e.kernel_info(ALGO_ID[k], hi)["variant"] == 1
        while hi - lo > 1:
            mid = (lo + hi) // 2
            lo, hi = (mid, hi) if e.kernel_info(ALGO_ID[k], mid)["variant"] == 2 else (lo, mid)
        for n, ref in ((lo, warp), (hi, thread)):
            x, cols = tiled_inputs(torch, dev, base, n)
            out = run_call(name, e, t, x, n, torch, dev)[0]
            assert torch.equal(out, ref[name][:, cols]), (k, n)
    e.close()
    print("\n%s %d bodies (team %d): worst against the thread kernel %.1e (ABA per cond2(M)), against the oracle %.1e (ABA residual)"
          % (shape, nb, team_threads(nb), worst[0], worst[1]))


@pytest.mark.gpu
def test_129_bodies_never_run_on_the_warp_variant(torch_dev):
    """One body beyond MB_MAX_BODIES: the handle may refuse the tree, or build it for the thread-per-state kernels; either way
    the warp variant raises and writes nothing."""
    import mecano_b200 as mb

    torch, dev = torch_dev
    t = body_parallel_tree("chain", 129)
    try:
        e, _ = engine_of(t, (0.0, 0.0, -9.81))
    except mb._capi.MecanoB200Error:
        return
    rng = np.random.default_rng(129)
    q, qd, qdd, _ = (torch.from_numpy(v).to(dev) for v in td.random_states(rng, t, 64))
    out = torch.full((t.nv, 64), float("nan"), dtype=torch.float64, device=dev)
    with pytest.raises(mb._capi.MecanoB200Error):
        e.set_variant(2)
        e.rnea(q, qd, qdd, out)
    assert bool(torch.isnan(out).all())
    e.close()
