#!/usr/bin/env python
"""bench.py -- batched RNEA / ABA / CRBA states/sec on the 37-DoF humanoid (fp64), the metric of BASELINE.json.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched under torch.distributed.run)
    python bench.py --impl reference --gpus N --steps K --warmup W

One "step" evaluates all three calculators (InverseDynamicsCalculator, ForwardDynamicsCalculator,
CompositeRigidBodyMassMatrixCalculator) once on a batch of synthetic random states of the H37 humanoid tree
(SixDoF + 31 revolute joints: 32 bodies, 37 DoF, 38 configuration rows); a state counts as processed when all
three have been evaluated.  `value` = states of all ranks / (max-over-ranks time per step), inputs resident in HBM.
Per-GPU work is fixed (weak scaling); ranks own disjoint slices and there is no collective on the data path.

Rank 0 prints ONE JSON line (see the task contract): metric/value/unit/..., `roofline` for the dominant kernel
(CRBA, HBM-bound) plus per-kernel details under `kernels`, `cpu_baseline` (the C oracle port timed on the host
cores on a bounded sample), `e2e` (the same step through the host-pointer C-ABI entry points: pinned host buffers,
H2D + kernels + D2H inside the timed region) and `clocks`.  `extras` (rank 0, outside the timed step; `--no-extras` skips
them) times the rows next to the path: state integrator, calculator-owned mass matrix, RNEA by-products, forward dynamics with
joint source modes, centroidal momentum matrix / centre of mass alone / convective term, Coriolis matrix, the optional fp32 variant
with its error, BASELINE configs 1 and 2, and the end-to-end step with the packed mass matrix (`e2e_packed`) and with the dense matrix kept
in one host buffer from step to step (`e2e_dense_kept`).

`--dump-outputs DIR` writes what the last timed step returned -- mass_matrix.npy (entry-major [nv*nv][S]), qdd.npy (forward
dynamics, [nv][S]) and tau.npy (inverse dynamics, [nv][S]), all fp64 -- for a fixed, seeded sample of S <= 2048 of the states.
The states are generated on the device from fixed seeds, so two builds run with the same arguments see the same inputs.

`--impl reference`: Mecano itself is Java and no JVM exists on these boxes (SURVEY.md 8c), so the reference arm
times the reference-faithful C restatement (oracle/, "port") multithreaded on all host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HUMANOID_SEED = 20251017
STATE_SEED = 1234
DUMP_SEED = 4321
DUMP_STATES = 2048  # states in the --dump-outputs sample over all ranks: ~24 MB for H37, the dense mass matrix being most of it
GRAVITY = (0.0, 0.0, -9.81)
FP64_NOMINAL_TFLOPS = 37.2  # 148 SMs x 64 DFMA/clk x 2 flop x 1.965 GHz (SURVEY.md section 6); the measured DFMA-chain figure is ~93 % of it
METRIC = "RNEA+ABA+CRBA states/sec (37-DoF humanoid, fp64)"
UNIT = "states/s"


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--states", type=int, default=1 << 20, help="states per GPU (weak scaling)")
    p.add_argument("--neck", type=int, default=2, help="2 -> H37 (37 DoF), 1 -> H36 (36 DoF)")
    p.add_argument("--cpu-sample", type=int, default=0, help="states in the bounded CPU-baseline sample (0: sized from --cpu-budget)")
    p.add_argument("--cpu-budget", type=float, default=60.0, help="seconds of CPU work the reference arm's timed steps may take in total")
    p.add_argument("--e2e-steps", type=int, default=5)
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-cpu", action="store_true")
    p.add_argument("--no-extras", action="store_true", help="skip the kernels timed outside the step (ncu launch lists of the step alone)")
    p.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed, for a fixed sample of the states, "
                                                         "as DIR/<name>.npy (fp64)")
    args = p.parse_args()
    if args.steps < 1 or args.warmup < 0:
        p.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        p.error("--dump-outputs writes the outputs of the GPU step; the reference arm times other states")
    return args


def workload_name(neck, n):
    return "H%d humanoid (SixDoF + %d revolute, %d bodies), %d states/GPU, RNEA+ABA+CRBA per step" % (36 + (neck == 2), 29 + neck, 30 + neck, n)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
                power.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def build_system(neck):
    import mecano_b200 as mb

    elevator = mb.RigidBody("elevator")
    mb.MultiBodySystemRandomTools.nextHumanoid(HUMANOID_SEED, elevator, neck)
    return mb.MultiBodySystem.toMultiBodySystemBasics(elevator)


def bench_tree(neck):
    """The humanoid of the benchmark as neutral tables (tests/golden/bench_tree_H*.npz, written by tests/golden/make_bench_tree.py
    from the host model with HUMANOID_SEED): what the CPU legs build the oracle from, without importing the product package."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import treedesc

    z = np.load(os.path.join(ROOT, "tests", "golden", "bench_tree_H%d.npz" % (35 + neck)))
    assert int(z["seed"]) == HUMANOID_SEED, "tests/golden/bench_tree_*.npz is stale: run tests/golden/make_bench_tree.py"
    fields = {k: (int(z[k]) if z[k].ndim == 0 else z[k]) for k in z.files if k != "seed"}
    return treedesc.TreeDesc(**fields).contiguous()


def oracle_for_tree(tree):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib

    return oracle_lib.Oracle(tree, gravity=GRAVITY), oracle_lib


def same_tree(system, tree):
    """The GPU arm's generated system equals the committed tables the CPU arm uses (both arms on the same multi-body system)."""
    d = system.describe()
    return all(np.array_equal(np.asarray(d[k]), getattr(tree, k)) for k in ("parent", "jtype", "axis", "off_R", "off_p", "com_R", "com_p", "J", "mass", "dof_off", "cfg_off"))


def cpu_step(oracle, q, qd, qdd, tau, nthreads=0):
    """The reference path for one batch: ID, FD and the mass matrix, one calculator instance per thread."""
    oracle.rnea_batch(q, qd, qdd, nthreads=nthreads)
    oracle.aba_batch(q, qd, tau, nthreads=nthreads)
    oracle.crba_batch(q, nthreads=nthreads)


def run_reference(args, rank, world):
    """The reference arm: the CPU implementation of the path on the host cores.  Imports nothing of the product (no
    mecano_b200, no CUDA library): tree from the committed tables, states from numpy, compute in oracle/."""
    if rank != 0:
        return
    tree = bench_tree(args.neck)  # puts tests/ on the path
    oracle, oracle_lib = oracle_for_tree(tree)
    import treedesc

    cores = oracle_lib.lib().mo_max_threads()
    rng = np.random.default_rng(STATE_SEED)
    # warm-up doubles as a rate probe: the sample of each timed step is sized so that the K timed steps take about
    # --cpu-budget seconds in total (at most the full batch); throughput is per state and states are independent, so the
    # rate does not depend on the sample size
    probe = 4096
    q, qd, qdd, tau = treedesc.random_states(rng, tree, probe)
    cpu_step(oracle, q, qd, qdd, tau)
    t0 = time.perf_counter()
    for _ in range(max(1, min(args.warmup, 3))):
        cpu_step(oracle, q, qd, qdd, tau)
    rate = probe * max(1, min(args.warmup, 3)) / (time.perf_counter() - t0)
    n = args.cpu_sample if args.cpu_sample > 0 else int(min(args.states, max(8192, rate * args.cpu_budget / max(1, args.steps))))
    n = max(256, n // 256 * 256)
    q, qd, qdd, tau = treedesc.random_states(rng, tree, n)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_step(oracle, q, qd, qdd, tau)
    dt = (time.perf_counter() - t0) / args.steps
    value = n / dt
    sample = "%d states of the same workload per step (bounded sample), C restatement of Mecano (oracle/), %d threads" % (n, cores)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.neck, args.states), "sample_states_per_step": n,
                   "sample_note": "a full %d-state step takes ~%.0f s on these cores; each step is a bounded sample sized for ~%.0f s of CPU work over the "
                                  "%d timed steps (states are independent: the per-state rate does not depend on the sample size)"
                                  % (args.states, args.states / value, args.cpu_budget, args.steps),
                   "note": "Mecano is Java; no JVM on this box: reference arm = reference-faithful C port on host cores (-O2, -ffp-contract=off)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def owned_zero_entries(system):
    """Mass-matrix entries (i * nv + j) that couple joints of unrelated branches: zero for every state."""
    joints = system.getJointsToConsider()
    prov = system.getJointMatrixIndexProvider()
    nv = system.getNumberOfDoFs()

    def ancestors(j):
        out = set()
        while j is not None:
            out.add(j)
            j = j.getPredecessor().getParentJoint()
        return out

    anc = {j: ancestors(j) for j in joints}
    zeros = []
    for a in joints:
        for b in joints:
            if a is b or a in anc[b] or b in anc[a]:
                continue
            for r in prov.getJointDoFIndices(a):
                for c in prov.getJointDoFIndices(b):
                    zeros.append(r * nv + c)
    return zeros


def a7_configs(mb, torch, dev, device_index):
    """BASELINE.json configs 1 and 2 on the 7-DoF revolute arm (MultiBodySystemRandomTools.nextRevoluteJointChain look-alike):
    config 1 = InverseDynamicsCalculator on ONE state on the CPU (the C port, one thread; the latency a Mecano user sees per call),
    next to the GPU's single-state latency (warp-per-state kernel); config 2 = batched RNEA of 65,536 random states on one B200,
    every state verified against the oracle."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    import treedesc

    elevator = mb.RigidBody("elevator")
    mb.MultiBodySystemRandomTools.nextRevoluteJointChain(7, elevator, 7)
    arm = mb.MultiBodySystem.toMultiBodySystemBasics(elevator)
    oracle = oracle_lib.Oracle(treedesc.TreeDesc(**arm.describe()).contiguous(), gravity=GRAVITY)
    rng = np.random.default_rng(STATE_SEED)
    n2 = 65536
    q, qd, qdd, _ = mb.MultiBodySystemRandomTools.nextState(rng, arm, n2)
    out = {}
    # config 1: one state per call, single thread
    q1, qd1, qdd1 = (np.ascontiguousarray(a[:, :1]) for a in (q, qd, qdd))
    for _ in range(2000):
        oracle.rnea_batch(q1, qd1, qdd1, nthreads=1)
    reps = 20000
    t0 = time.perf_counter()
    for _ in range(reps):
        oracle.rnea_batch(q1, qd1, qdd1, nthreads=1)
    cpu_call_us = (time.perf_counter() - t0) / reps * 1e6
    t0 = time.perf_counter()
    oracle.rnea_batch(q, qd, qdd, nthreads=1)
    cpu_state_us = (time.perf_counter() - t0) / n2 * 1e6
    ident = mb.InverseDynamicsCalculator(arm, device=device_index)
    ident.setGravitationalAcceleration(*GRAVITY)
    tq, tqd, tqdd = (torch.from_numpy(a).to(dev) for a in (q, qd, qdd))
    tau = torch.empty((7, n2), dtype=torch.float64, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, reps):
        for _ in range(5):
            fn()
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    one = timed(lambda: ident.compute(tq[:, :1], tqd[:, :1], tqdd[:, :1], tau[:, :1]), 200)
    out["config1_a7_single_state"] = {
        "cpu_us_per_call": cpu_call_us, "cpu_us_per_state_in_a_loop": cpu_state_us, "cpu_kind": "port (C restatement, 1 thread; per call includes the ctypes call)",
        "gpu_us_per_call_device_resident": one * 1e3, "gpu_variant": ident.kernelInfo(1)["variant"],
        "what": "BASELINE config 1: InverseDynamicsCalculator, 7-DoF revolute chain, a single state"}
    ms = timed(lambda: ident.compute(tq, tqd, tqdd, tau), 50)
    ref = oracle.rnea_batch(q, qd, qdd)
    got = ident.compute(tq, tqd, tqdd, tau).cpu().numpy()
    err = np.abs(got - ref).max(axis=0) / np.maximum(1.0, np.abs(ref).max(axis=0))
    out["config2_a7_rnea_65536"] = {
        "ms": ms, "states_per_s": n2 / (ms * 1e-3), "algorithmic_bytes_per_state": 224, "achieved_gbs": 224.0 * n2 / (ms * 1e-3) / 1e9,
        "max_rel_error_vs_oracle_per_state": float(err.max()), "states_verified": n2, "tolerance": 1e-9, "variant": ident.kernelInfo(n2)["variant"],
        "what": "BASELINE config 2: batched RNEA, 7-DoF revolute arm, 65,536 random states on one B200, every state compared with the oracle "
                "(launch-latency regime: ~15 MB of traffic)"}
    assert err.max() < 1e-9
    return out


_JSON_FD = None


def bind_to_gpu_numa_node(index):
    """Pin this process to the CPUs next to its GPU (NVML's ideal CPU affinity) before any pinned host buffer is allocated, so
    that the end-to-end path's staging memory is first touched on the GPU's own NUMA node: with several ranks on a two-socket
    box the host <-> device copies otherwise cross the socket interconnect.  Returns the number of CPUs bound to, or None."""
    try:
        import pynvml

        pynvml.nvmlInit()
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(visible.split(",")[index]) if visible and visible.split(",")[index].isdigit() else index
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def claim_stdout():
    """stdout carries the one JSON line and nothing else: libraries that chat on file descriptor 1 (NCCL prints its version
    there) are sent to stderr for the duration of the run, and the line itself goes to the original descriptor."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_JSON_FD, data)


def dump_outputs(path, outputs, n, world, rank):
    """--dump-outputs: the same DUMP_STATES / world states (columns, drawn with DUMP_SEED) of every output on every rank,
    concatenated rank after rank along the state axis; rank 0 writes path/<name>.npy.  The inputs are seeded, so two builds
    run with the same arguments can be compared output for output."""
    import torch
    import torch.distributed as dist

    k = max(1, min(n, DUMP_STATES // world))
    idx = torch.from_numpy(np.sort(np.random.default_rng(DUMP_SEED).choice(n, k, replace=False)))
    for name, out in outputs.items():
        part = out.index_select(1, idx.to(out.device))
        if world > 1:
            parts = [torch.empty_like(part) for _ in range(world)]
            dist.all_gather(parts, part)
            part = torch.cat(parts, dim=1)
        if rank == 0:
            os.makedirs(path, exist_ok=True)
            np.save(os.path.join(path, name + ".npy"), part.cpu().numpy())


def main():
    args = parse_args()
    claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    import mecano_b200 as mb
    from mecano_b200 import sharding

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None  # N = 1 keeps every host core for the CPU baseline
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    system = build_system(args.neck)
    nv, nq, nb = system.getNumberOfDoFs(), system.getConfigurationMatrixSize(), system.getNumberOfJoints()
    n = args.states
    ident = mb.InverseDynamicsCalculator(system, device=local_rank)
    fdyn = mb.ForwardDynamicsCalculator(system, device=local_rank)
    crba = mb.CompositeRigidBodyMassMatrixCalculator(system, device=local_rank)
    for c in (ident, fdyn):
        c.setGravitationalAcceleration(*GRAVITY)

    # synthetic states generated on the device for the device-resident measurement (seed differs per rank: disjoint slices)
    gen = torch.Generator(device=dev).manual_seed(STATE_SEED + rank)
    q = (torch.rand((nq, n), dtype=torch.float64, device=dev, generator=gen) * 2 - 1) * np.pi
    quat = torch.randn((4, n), dtype=torch.float64, device=dev, generator=gen)
    q[0:4] = quat / quat.norm(dim=0, keepdim=True)
    q[4:7] = torch.rand((3, n), dtype=torch.float64, device=dev, generator=gen) * 2 - 1
    qd = torch.rand((nv, n), dtype=torch.float64, device=dev, generator=gen) * 2 - 1
    qdd = torch.rand((nv, n), dtype=torch.float64, device=dev, generator=gen) * 2 - 1
    tau_in = torch.rand((nv, n), dtype=torch.float64, device=dev, generator=gen) * 2 - 1
    tau = torch.empty((nv, n), dtype=torch.float64, device=dev)
    qdd_out = torch.empty((nv, n), dtype=torch.float64, device=dev)
    M = torch.empty((nv * nv, n), dtype=torch.float64, device=dev)

    # One step = the three calculators on the same batch, in the order of a controller tick: mass matrix, forward dynamics, inverse
    # dynamics.  (The kernel that follows CRBA also absorbs the write-back of the ~100 MB of mass-matrix lines still dirty in L2,
    # about 15 us: forward dynamics, the longest of the three, rather than inverse dynamics, the shortest.)
    STEP_ORDER = ("crba", "aba", "rnea")

    def step(events=None):
        if events is not None:
            events[0].record()
        crba.getMassMatrix(q, M)
        if events is not None:
            events[1].record()
        fdyn.compute(q, qd, tau_in, qdd_out)
        if events is not None:
            events[2].record()
        ident.compute(q, qd, qdd, tau)
        if events is not None:
            events[3].record()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(args.steps)]
    barrier()
    t_start = torch.cuda.Event(enable_timing=True)
    t_stop = torch.cuda.Event(enable_timing=True)
    t_start.record()
    for k in range(args.steps):
        step(evs[k])
    t_stop.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:  # before the extras below reuse the output buffers
        dump_outputs(args.dump_outputs, {"mass_matrix": M, "qdd": qdd_out, "tau": tau}, n, world, rank)

    ms_total = t_start.elapsed_time(t_stop)
    ms_step = sharding.max_over_ranks(ms_total / args.steps, dev)
    per_kernel_ms = {name: float(np.mean([evs[k][i].elapsed_time(evs[k][i + 1]) for k in range(args.steps)]))
                     for i, name in enumerate(STEP_ORDER)}
    per_kernel_ms = {k: sharding.max_over_ranks(v, dev) for k, v in per_kernel_ms.items()}
    value = n * world / (ms_step * 1e-3)

    # ---- roofline (rank 0 numbers; every rank runs the same kernels on the same amount of work)
    peaks, peak_src = measured_peaks()
    hbm_peak = float(peaks["hbm_gbs"])
    # FP64 denominators, measured right after the timed region: the burst figure (best of five 4.6 ms launches of an FMA chain) and
    # the sustained one (the same chain back to back for as long as the timed region, at least 0.25 s, rate over the second half).
    # They agree (34.8 TFLOP/s, profiles/r06zm): the FMA chain alone does not reach the board's power cap.  The step does -- CRBA
    # writing at 6 TB/s next to two FP64-bound kernels: over 100 steps the SM clock settles at ~1830 of 1965 MHz (sw_power_cap) and
    # every FP64-bound time stretches with it -- so each kernel's fraction is also given against the peak scaled to the SM clock
    # sampled during the timed region (fp64_frac_at_sampled_clock).
    fp64_sustained = mb.measure_fp64_sustained(local_rank, max(0.25, min(2.0, ms_total * 1e-3))) if rank == 0 else 0.0
    fp64_peak = mb.measure_fp64_peak(local_rank) if rank == 0 else 0.0
    flops_path = os.path.join(ROOT, "profiles", "algorithmic_flops.json")
    flops = json.load(open(flops_path)) if os.path.exists(flops_path) else {}
    exec_path = os.path.join(ROOT, "profiles", "executed_flops.json")
    exec_flops = json.load(open(exec_path)) if os.path.exists(exec_path) else {}
    key = "H%d" % nv
    kernels = {}
    for name, calc in (("rnea", ident), ("aba", fdyn), ("crba", crba)):
        info = calc.kernelInfo(n)
        ms = per_kernel_ms[name]
        gbs = info["bytes_per_state"] * n / (ms * 1e-3) / 1e9
        entry = {"ms": ms, "states_per_s": n / (ms * 1e-3), "algorithmic_bytes_per_state": info["bytes_per_state"], "achieved_gbs": gbs,
                 "hbm_frac": gbs / hbm_peak, "block_threads": info["block_threads"], "regs": info["regs_per_thread"],
                 "smem_bytes": info["dynamic_smem_bytes"], "blocks_per_sm": info["blocks_per_sm"],
                 "tmem_stack_slots": info["tmem_stack_slots"], "specialized": info["specialized"]}
        fl = flops.get(key, {}).get(name)
        if fl and fp64_peak:
            tf = fl * n / (ms * 1e-3) / 1e12
            entry.update({"algorithmic_flops_per_state": fl, "achieved_tflops": tf, "fp64_frac": tf / fp64_peak,
                          "fp64_frac_of_sustained_peak": tf / fp64_sustained if fp64_sustained else None,
                          "fp64_frac_at_sampled_clock": (tf / (fp64_peak * clocks["sm_mhz"] / clocks["sm_max_mhz"])
                                                         if clocks and clocks.get("sm_mhz") and clocks.get("sm_max_mhz") else None),
                          "fp64_frac_of_nominal": tf / FP64_NOMINAL_TFLOPS})
            fe = exec_flops.get(key, {}).get(name)
            if fe:  # what the current routines execute for the same result (fewer: profiles/executed_flops.json)
                entry.update({"executed_flops_per_state": fe, "executed_tflops": fe * n / (ms * 1e-3) / 1e12,
                              "fp64_frac_executed": fe * n / (ms * 1e-3) / 1e12 / fp64_peak})
        kernels[name] = entry
    # ---- next-row kernels (SURVEY.md 8f), timed outside the step: the state integrator that follows ABA in a roll-out
    extras = {}
    if rank == 0 and not args.no_extras:
        integ = mb.MultiBodySystemStateIntegrator(system, 1.0e-3, engine=fdyn._engine)
        iq, iqd, iqdd = q.clone(), qd.clone(), qdd_out.clone()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(3):
            integ.doubleIntegrateFromAcceleration(iq, iqd, iqdd)
        reps = 10
        e0.record()
        for _ in range(reps):
            integ.doubleIntegrateFromAcceleration(iq, iqd, iqdd)
        e1.record()
        torch.cuda.synchronize()
        ims = e0.elapsed_time(e1) / reps
        n6 = sum(1 for j in system.getJointsToConsider() if j.getDegreesOfFreedom() == 6)
        ibytes = 8.0 * (5 * (nb - n6) + 35 * n6)  # one-DoF: read q, qd, qdd, write q, qd; SixDoF: read 19 rows, write 16
        extras["integrate"] = {"ms": ims, "states_per_s": n / (ims * 1e-3), "algorithmic_bytes_per_state": ibytes,
                               "achieved_gbs": ibytes * n / (ims * 1e-3) / 1e9, "hbm_frac": ibytes * n / (ims * 1e-3) / 1e9 / hbm_peak,
                               "what": "MultiBodySystemStateIntegrator.doubleIntegrateFromAcceleration, in place, %d states" % n}
        del iq, iqd, iqdd
        # the calculator-owned mass matrix (getMassMatrix(q) without an output argument): structurally zero entries are
        # written by the first call only
        owned = mb.CompositeRigidBodyMassMatrixCalculator(system, device=local_rank)
        for _ in range(3):
            owned.getMassMatrix(q)
        e0.record()
        for _ in range(reps):
            owned.getMassMatrix(q)
        e1.record()
        torch.cuda.synchronize()
        oms = e0.elapsed_time(e1) / reps
        nnz = nv * nv - len(set(owned_zero_entries(system)))
        obytes = 8.0 * (nq + nnz)
        extras["crba_owned_buffer"] = {"ms": oms, "states_per_s": n / (oms * 1e-3), "algorithmic_bytes_per_state": obytes,
                                       "achieved_gbs": obytes * n / (oms * 1e-3) / 1e9, "hbm_frac": obytes * n / (oms * 1e-3) / 1e9 / hbm_peak,
                                       "nonzero_entries": nnz, "entries": nv * nv,
                                       "what": "CompositeRigidBodyMassMatrixCalculator.getMassMatrix(q) into the calculator's own matrix: the "
                                               "%d structurally zero entries are written once, not per call (MECANO_B200_CRBA_ZEROS_PRESENT)" % (nv * nv - nnz)}
        del owned
        # the packed layout on the device (the end-to-end number with it is extras.e2e_packed)
        pk = mb.CompositeRigidBodyMassMatrixCalculator(system, device=local_rank)
        prow, _ = pk.getMassMatrixPackedIndex()
        Pk = torch.empty((len(prow), n), dtype=torch.float64, device=dev)
        for _ in range(3):
            pk.getMassMatrix(q, Pk, packed=True)
        e0.record()
        for _ in range(reps):
            pk.getMassMatrix(q, Pk, packed=True)
        e1.record()
        torch.cuda.synchronize()
        pms = e0.elapsed_time(e1) / reps
        pbytes = 8.0 * (nq + len(prow))
        extras["crba_packed"] = {"ms": pms, "states_per_s": n / (pms * 1e-3), "algorithmic_bytes_per_state": pbytes,
                                 "achieved_gbs": pbytes * n / (pms * 1e-3) / 1e9, "hbm_frac": pbytes * n / (pms * 1e-3) / 1e9 / hbm_peak,
                                 "packed_rows": len(prow), "entries": nv * nv,
                                 "what": "getMassMatrix(q, packed=True): the unique entries that are not structurally zero (MECANO_B200_CRBA_PACKED), "
                                         "bit-identical to the dense matrix's entries"}
        del pk, Pk

        def timed(fn):
            for _ in range(3):
                fn()
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / reps

        def hbm_entry(ms, nbytes, what):
            return {"ms": ms, "states_per_s": n / (ms * 1e-3), "algorithmic_bytes_per_state": nbytes,
                    "achieved_gbs": nbytes * n / (ms * 1e-3) / 1e9, "hbm_frac": nbytes * n / (ms * 1e-3) / 1e9 / hbm_peak, "what": what}

        # RNEA with its by-products (getBodyAcceleration / getComputedJointWrench for every body): 12 nb more rows written
        full = mb.InverseDynamicsCalculator(system, device=local_rank).setComputeByProducts()
        full.setGravitationalAcceleration(*GRAVITY)
        extras["rnea_byproducts"] = hbm_entry(timed(lambda: full.compute(q, qd, qdd, tau)), 8.0 * (nq + 3 * nv + 12 * nb),
                                              "InverseDynamicsCalculator.compute + body accelerations + joint wrenches (mecano_b200_rnea_full)")
        del full
        # forward dynamics with every second one-DoF joint an ACCELERATION_SOURCE, efforts of those joints included (pass four)
        locked = [j for i, j in enumerate(system.getJointsToConsider()) if j.getDegreesOfFreedom() == 1 and i % 2 == 0]
        mixed = mb.ForwardDynamicsCalculator(system, device=local_rank)
        mixed.setGravitationalAcceleration(*GRAVITY)
        mixed.setJointSourceModes(lambda j: mb.JointSourceMode.ACCELERATION_SOURCE if j in locked else None)
        extras["aba_source_modes"] = hbm_entry(timed(lambda: mixed.compute(q, qd, tau_in, qdd_out, jointAccelerationInput=qdd)),
                                               8.0 * (2 * nq + 8 * nv),
                                               "ForwardDynamicsCalculator.compute(tau, qdd) with %d of %d joints in ACCELERATION_SOURCE mode + getJointTauMatrix "
                                               "(ABA launch + RNEA launch + row copies; mecano_b200_aba_sources)" % (len(locked), nb))
        del mixed
        # mass matrix + centroidal momentum matrix + centre of mass, then the convective term, in the centre-of-mass frame
        cen = mb.CompositeRigidBodyMassMatrixCalculator(system, "centerOfMassFrame", device=local_rank)
        extras["crba_centroidal"] = hbm_entry(timed(lambda: cen.getCentroidalMomentumMatrix(q)), 8.0 * (nq + nv * nv + 6 * nv + 4),
                                              "getMassMatrix + getCentroidalMomentumMatrix + centre of mass (mecano_b200_crba_centroidal; the "
                                              "centre-of-mass shift re-reads and re-writes 9 nv rows, not counted)")
        extras["center_of_mass"] = hbm_entry(timed(lambda: cen.getCenterOfMass(q)), 8.0 * (nq + 4),
                                             "CenterOfMassCalculator.getCenterOfMass + getTotalMass (mecano_b200_center_of_mass: the by-product "
                                             "mass-matrix kernel launched without a matrix -- composite inertias only, no unit momenta, no stores)")
        extras["centroidal_convective_term"] = hbm_entry(timed(lambda: cen.getCentroidalConvectiveTermMatrix(q, qd)), 8.0 * (2 * nq + nv + 2 * 4 + 6),
                                                         "getCentroidalConvectiveTermMatrix in the centre-of-mass frame (mecano_b200_center_of_mass for the q "
                                                         "passed + mecano_b200_centroidal_convective_term: one RNEA launch whose joint efforts go to a scratch "
                                                         "buffer, + the shift)")
        cen.setEnableCoriolisMatrixCalculation(True)
        extras["coriolis_matrix"] = hbm_entry(timed(lambda: cen.getCoriolisMatrix(q, qd)), 8.0 * (nq + nv + 2 * nv * nv),
                                              "getMassMatrix + getCoriolisMatrix, both dense nv x nv (mecano_b200_coriolis)")
        del cen
        # the optional fp32 variant of the three kernels (arithmetic in float, buffers fp64), reported separately with its error
        f32 = {}
        M32 = torch.empty_like(M)
        for name, calc32, run32, ref_out in (
                ("rnea", mb.InverseDynamicsCalculator(system, device=local_rank), lambda c: c.compute(q, qd, qdd), ident.compute(q, qd, qdd)),
                ("aba", mb.ForwardDynamicsCalculator(system, device=local_rank), lambda c: c.compute(q, qd, tau_in), fdyn.compute(q, qd, tau_in)),
                ("crba", mb.CompositeRigidBodyMassMatrixCalculator(system, device=local_rank), lambda c: c.getMassMatrix(q, M32), crba.getMassMatrix(q, M))):
            calc32.setKernelVariant("thread").setPrecision("fp32")
            if name != "crba":
                calc32.setGravitationalAcceleration(*GRAVITY)
            ms32 = timed(lambda: run32(calc32))
            out32 = run32(calc32)
            # per state: max |fp32 - fp64| over the outputs of the state / max(1, max |fp64| of the state)
            per_state = (out32 - ref_out).abs().amax(dim=0) / ref_out.abs().amax(dim=0).clamp(min=1.0)
            srt = per_state.sort().values
            f32[name] = {"ms": ms32, "states_per_s": n / (ms32 * 1e-3), "speedup_vs_fp64": kernels[name]["ms"] / ms32,
                         "rel_error_vs_fp64": {"median": float(srt[n // 2]), "p99": float(srt[int(n * 0.99)]), "p99.9": float(srt[int(n * 0.999)]),
                                               "max": float(srt[-1])}}
            del per_state, srt
            del calc32, out32
        del M32
        extras["fp32_variant"] = dict(f32, what="optional single-precision variant (mecano_b200_set_precision): arithmetic in float, all buffers fp64; "
                                                "error per state = max |fp32 - fp64| / max(1, max |fp64|), quantiles over the batch")
    if rank == 0 and world == 1 and not args.no_extras and not args.no_cpu:
        extras.update(a7_configs(mb, torch, dev, local_rank))
    dom = max(kernels, key=lambda k: kernels[k]["ms"])
    # The dominant kernel is reported against the roofline that binds it (SURVEY.md 8d): RNEA / ABA sit above the machine
    # balance (FP64 pipe), CRBA below it (HBM, write-dominated).  MEASURED_PEAKS.json has no FP64 figure, so the FP64
    # denominator is the DFMA-chain microbenchmark of this library measured in this run (mecano_b200_measure_fp64_peak).
    kd = kernels[dom]
    balance = fp64_peak * 1e12 / (hbm_peak * 1e9) if fp64_peak else 0.0
    intensity = kd.get("algorithmic_flops_per_state", 0.0) / kd["algorithmic_bytes_per_state"]
    if fp64_peak and intensity > balance:
        roofline = {"kernel": dom, "bound": "fp64", "achieved": kd["achieved_tflops"], "peak": fp64_peak, "unit": "TFLOP/s",
                    "frac": kd["fp64_frac"], "traffic": None, "peak_source": "FP64 DFMA chain measured live in this run (no FP64 figure in MEASURED_PEAKS.json)",
                    "hbm": {"achieved": kd["achieved_gbs"], "peak": hbm_peak, "unit": "GB/s", "frac": kd["hbm_frac"], "peak_source": peak_src}}
    else:
        roofline = {"kernel": dom, "bound": "hbm", "achieved": kd["achieved_gbs"], "peak": hbm_peak, "unit": "GB/s",
                    "frac": kd["hbm_frac"], "traffic": None, "peak_source": peak_src, "fp64_peak_tflops_measured_live": fp64_peak,
                    "fp64_peak_tflops_sustained_live": fp64_sustained,
                    "fp64_note": "kernels[*].fp64_frac is against the burst figure (best of five 4.6 ms launches of an FMA chain), "
                                 "fp64_frac_of_sustained_peak against the same chain run back to back for the length of the timed region, "
                                 "fp64_frac_at_sampled_clock against the burst figure scaled by clocks.sm_mhz / clocks.sm_max_mhz (the step, "
                                 "unlike the FMA chain, reaches the power cap when it runs for long)"}
    roofline["flop_per_byte"] = intensity
    roofline["machine_balance_flop_per_byte"] = balance
    traffic_path = os.path.join(ROOT, "profiles", "dram_traffic.json")
    if os.path.exists(traffic_path):
        tr_all = json.load(open(traffic_path))
        for name in kernels:
            if name in tr_all:
                kernels[name]["dram_traffic_bytes_per_state_ncu"] = tr_all[name]["bytes_per_state"]
        tr = tr_all.get(dom)
        if tr:
            roofline["traffic"] = tr["bytes_per_state"] * n
            roofline["traffic_note"] = "NOT measured in this run: dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu capture (profiles/dram_traffic.json: %s)" % tr.get("note")

    line = None
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(args.neck, n), "states_per_gpu": n, "n_dofs": nv, "n_cfg": nq, "n_bodies": nb,
                       "parallelism": "disjoint state slices per GPU, no collective", "cpus_bound_per_rank": numa, "l2": "inputs (%.2f GB/step) and outputs larger than L2; no explicit flush"
                       % (8.0 * (3 * nq + 4 * nv) * n / 1e9), "humanoid_seed": HUMANOID_SEED, "mass_matrix_layout": "entry-major [nv*nv][N]",
                       "step_order": ", ".join(STEP_ORDER)},
            "roofline": roofline, "kernels": kernels, "extras": extras, "gpu_launches": 3 * args.steps, "clocks": clocks,
        }

    # ---- CPU baseline: the oracle port on the host cores, bounded sample of the same workload (rank 0, N = 1 only)
    if rank == 0 and world == 1 and not args.no_cpu:
        tree = bench_tree(args.neck)
        assert same_tree(system, tree), "tests/golden/bench_tree_*.npz does not match the generated humanoid: run tests/golden/make_bench_tree.py"
        oracle, oracle_lib = oracle_for_tree(tree)
        cores = oracle_lib.lib().mo_max_threads()
        ns = args.cpu_sample if args.cpu_sample > 0 else 32768
        hq, hqd, hqdd, htau = (x[:, :ns].cpu().numpy().copy() for x in (q, qd, qdd, tau_in))
        cpu_step(oracle, hq[:, :1024].copy(), hqd[:, :1024].copy(), hqdd[:, :1024].copy(), htau[:, :1024].copy())
        t0 = time.perf_counter()
        cpu_step(oracle, hq, hqd, hqdd, htau)
        dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": ns / dt, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": "first %d states of the same batch, one pass of RNEA+ABA+CRBA, C restatement of Mecano (oracle/), one instance per thread" % ns}
    elif rank == 0:
        line["cpu_baseline"] = None

    # ---- end to end: the same step through the public host API with pinned host matrices, host <-> device copies inside the
    # timed region.  ONE call per step (MultiBodyDynamicsStep.compute -> mecano_b200_step_host: q / qd cross PCIe once); with
    # N > 1 rank 0 drives all N GPUs through one multi-device call (mecano_b200_multi_step_host slices the state-minor batch)
    # while the other ranks wait at the barrier.  The headline `e2e` returns the dense mass matrix as Mecano does; the packed
    # layout (unique non-zero entries) is reported next to it under extras.
    if not args.no_e2e:
        if rank == 0:
            devices = list(range(world)) if world > 1 else local_rank
            stepc = mb.MultiBodyDynamicsStep(system, device=devices)
            stepc.setGravitationalAcceleration(*GRAVITY)
            hn = n * world
            rows_dense, rows_packed = nv * nv, stepc.getMassMatrixRows(packed=True)

            def pin(rows, cols):
                return torch.empty((rows, cols), dtype=torch.float64).pin_memory()

            # pinned host memory for the whole job; if the box cannot pin that much, halve the states per GPU and say so
            while True:
                try:
                    hq, hqd, hqdd, htau_in, htau, hqdd_out, hM = pin(nq, hn), pin(nv, hn), pin(nv, hn), pin(nv, hn), pin(nv, hn), pin(nv, hn), pin(rows_dense, hn)
                    break
                except RuntimeError:
                    hq = hqd = hqdd = htau_in = htau = hqdd_out = hM = None
                    hn //= 2
                    if hn < 65536 * world:
                        raise
            per = hn // world
            for g in range(world):  # every GPU's slice holds the same synthetic states as the device-resident run of rank 0
                sl = slice(g * per, (g + 1) * per)
                hq[:, sl].copy_(q[:, :per]); hqd[:, sl].copy_(qd[:, :per]); hqdd[:, sl].copy_(qdd[:, :per]); htau_in[:, sl].copy_(tau_in[:, :per])
            nq_, nqd_, nqdd_, ntau_in, ntau, nqdd_out, nM = (t_.numpy() for t_ in (hq, hqd, hqdd, htau_in, htau, hqdd_out, hM))

            def host_step(packed, zeros_present=False):
                Mv = nM[:rows_packed] if packed else nM
                stepc.compute(nq_, nqd_, qdd=nqdd_, tau=ntau_in, tauOut=ntau, qddOut=nqdd_out, massMatrix=Mv, packed=packed,
                              massMatrixZerosPresent=zeros_present)

            def timed_host(packed, zeros_present=False):
                host_step(packed)  # warm-up (allocates the staging buffers; dense: writes every entry, structural zeros included)
                t0 = time.perf_counter()
                for _ in range(args.e2e_steps):
                    host_step(packed, zeros_present)
                return (time.perf_counter() - t0) / args.e2e_steps  # the call returns when the outputs are complete on the host

            # PCIe denominators measured live: one large pinned copy each way on device 0
            pcie = {}
            probe = torch.empty(1 << 27, dtype=torch.float64, device=dev)  # 1 GiB
            hprobe = torch.empty(1 << 27, dtype=torch.float64).pin_memory()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for name, (dst, src) in (("d2h", (hprobe, probe)), ("h2d", (probe, hprobe))):
                best = 0.0
                for _ in range(3):
                    ev0.record(); dst.copy_(src, non_blocking=True); ev1.record(); torch.cuda.synchronize()
                    best = max(best, 8.0 * (1 << 27) / (ev0.elapsed_time(ev1) * 1e-3) / 1e9)
                pcie[name + "_gbs_peak"] = best
            del probe, hprobe
        if world > 1:
            dist.barrier()
        if rank == 0:
            h2d = int(8 * (nq + 3 * nv) * hn)
            dt = timed_host(False)
            d2h = int(8 * (2 * nv + rows_dense) * hn)
            api = ("MultiBodyDynamicsStep.compute (one call: inverse dynamics, forward dynamics, mass matrix) on pinned host matrices -> "
                   + ("mecano_b200_multi_step_host over %d GPUs from one thread" % world if world > 1 else "mecano_b200_step_host"))
            line["e2e"] = {"value": hn / dt, "unit": UNIT, "ms_per_step": dt * 1e3, "steps": args.e2e_steps, "states_per_gpu": per,
                           "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "mass_matrix_layout": "dense entry-major [nv*nv][N] (Mecano's symmetric matrix, zeros included)",
                           "api": api, "check": float(np.abs(ntau).max()), "clock": "host wall clock around the blocking call",
                           "roofline": {"bound": "pcie", "achieved": d2h / dt / 1e9 / world, "peak": pcie["d2h_gbs_peak"], "unit": "GB/s per GPU, device -> host",
                                        "frac": d2h / dt / 1e9 / world / pcie["d2h_gbs_peak"], "h2d_gbs_peak": pcie["h2d_gbs_peak"],
                                        "peak_source": "1 GiB pinned cudaMemcpy each way on GPU 0, measured in this run"}}
            # the dense matrix kept in one host buffer across steps, as Mecano's calculator keeps its own: structurally zero
            # entries written (and transferred) by the warm-up call only
            nnz_rows = rows_dense - len(set(owned_zero_entries(system)))
            dto = timed_host(False, True)
            d2ho = int(8 * (2 * nv + nnz_rows) * hn)
            line["extras"]["e2e_dense_kept"] = {
                "value": hn / dto, "unit": UNIT, "ms_per_step": dto * 1e3, "steps": args.e2e_steps, "states_per_gpu": per, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2ho, "check": float(np.abs(nM).max()), "zero_entries_still_zero": bool(not nM[sorted(set(owned_zero_entries(system)))[:8]].any()),
                "pcie_d2h_frac": d2ho / dto / 1e9 / world / pcie["d2h_gbs_peak"],
                "what": "as e2e, the dense entry-major matrix kept in the same host buffer from step to step (what Mecano's calculator-owned "
                        "DMatrixRMaj is): the %d of %d entries that are structurally zero are written by the first call and neither recomputed nor "
                        "transferred again (MECANO_B200_CRBA_ZEROS_PRESENT through MultiBodyDynamicsStep.compute(massMatrixZerosPresent=True)); the "
                        "result in host memory is the same dense matrix bit for bit" % (rows_dense - nnz_rows, rows_dense)}
            dtp = timed_host(True)
            d2hp = int(8 * (2 * nv + rows_packed) * hn)
            line["extras"]["e2e_packed"] = {
                "value": hn / dtp, "unit": UNIT, "ms_per_step": dtp * 1e3, "steps": args.e2e_steps, "states_per_gpu": per, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2hp, "check": float(np.abs(nM[:rows_packed]).max()),
                "pcie_d2h_frac": d2hp / dtp / 1e9 / world / pcie["d2h_gbs_peak"],
                "what": "as e2e, mass matrix in the packed layout (MECANO_B200_CRBA_PACKED): the %d unique entries that are not structurally zero "
                        "instead of %d, with the index map exported for scattering into a DMatrixRMaj" % (rows_packed, rows_dense)}
        if world > 1:
            dist.barrier()
    elif rank == 0:
        line["e2e"] = None

    if rank == 0:
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
