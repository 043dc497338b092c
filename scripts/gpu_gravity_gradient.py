"""Gravity gradient on the benchmark humanoid (H37: 32 bodies, 37 DoFs): the device call at 2^20 states timed with CUDA events
after warm-up, the mass-matrix call on the same batch (same output size) for comparison, the finite-difference route a user had
before (2 nv calls each of mecano_b200_integrate and mecano_b200_rnea, assembled into the same G) timed on the same batch, and the
host-pointer call end to end at 2^18.  Bytes are computed from shapes (kernel_info bytes_per_state: q read, tau and G written); the
HBM fraction is against the read+write copy peak measured in the same run.  Device name, power limit and the kernel's registers,
local memory and launch configuration are read in the same call.  Writes one JSON line to <out>/gravity_gradient.jsonl.

    python scripts/gpu_gravity_gradient.py [--out DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
import mecano_b200 as mb  # noqa: E402


def timed(fn, reps=10):
    """Median, min and max of `reps` calls in ms, CUDA events, after one warm-up call.  G (12 GB at 2^20 states) is far beyond L2."""
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), float(np.min(ts)), float(np.max(ts))


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30)
        return float(out.stdout.strip().splitlines()[0])
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=".", help="directory that receives gravity_gradient.jsonl")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    assert torch.cuda.is_available(), "needs a CUDA device"
    system = bench.build_system(2)
    nv, nq = system.getNumberOfDoFs(), system.getConfigurationMatrixSize()
    gg = mb.MultiBodyGravityGradientCalculator(system)
    gg.setGravitationalAcceleration(-9.81)
    eng = gg._engine
    crba = mb.CompositeRigidBodyMassMatrixCalculator(system)
    hbm_gbs = mb.measure_hbm_peak(0)
    res = {"tree": "H37", "nv": nv, "nq": nq, "device": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(), "hbm_peak_copy_gbs": hbm_gbs}
    rng = np.random.default_rng(1)

    n = 1 << 20
    q = torch.from_numpy(mb.MultiBodySystemRandomTools.nextState(rng, system, n)[0]).cuda()
    tau = torch.empty((nv, n), dtype=torch.float64, device="cuda")
    G = torch.empty((nv * nv, n), dtype=torch.float64, device="cuda")
    info = gg.kernelInfo(n)
    ms, lo, hi = timed(lambda: eng.gravity_gradient(q, tau, G))
    bps = info["bytes_per_state"]
    res["kernel"] = {"n": n, "ms": ms, "ms_min": lo, "ms_max": hi, "states_per_s": n / (ms * 1e-3), "bytes": bps * n, "gbs": bps * n / (ms * 1e-3) / 1e9,
                     "hbm_fraction": bps * n / (ms * 1e-3) / 1e9 / hbm_gbs, "regs": info["regs_per_thread"], "local_bytes": info["local_bytes_per_thread"],
                     "block": info["block_threads"], "blocks_per_sm": info["blocks_per_sm"], "dynamic_smem": info["dynamic_smem_bytes"],
                     "stack_doubles": info["stack_doubles"]}
    G_ref = G.clone()

    # the mass matrix of the same states: the same nv^2 doubles written per state
    M = torch.empty((nv * nv, n), dtype=torch.float64, device="cuda")
    mms, mlo, mhi = timed(lambda: crba.getMassMatrix(q, massMatrix=M))
    minfo = crba.kernelInfo(n)
    res["mass_matrix"] = {"ms": mms, "ms_min": mlo, "ms_max": mhi, "gbs": minfo["bytes_per_state"] * n / (mms * 1e-3) / 1e9,
                          "hbm_fraction": minfo["bytes_per_state"] * n / (mms * 1e-3) / 1e9 / hbm_gbs,
                          "block": minfo["block_threads"], "blocks_per_sm": minfo["blocks_per_sm"], "regs": minfo["regs_per_thread"]}
    del M
    torch.cuda.empty_cache()

    # the route without this calculator: central differences, column by column, through the integrator and inverse dynamics
    eps = 1e-5
    z = torch.zeros((nv, n), dtype=torch.float64, device="cuda")
    qj = torch.empty_like(q)
    vj, aj = torch.empty((nv, n), dtype=torch.float64, device="cuda"), torch.empty((nv, n), dtype=torch.float64, device="cuda")
    tp, tm = torch.empty((nv, n), dtype=torch.float64, device="cuda"), torch.empty((nv, n), dtype=torch.float64, device="cuda")
    G3 = G.view(nv, nv, n)

    def fd_route():
        for j in range(nv):
            for dt, out in ((eps, tp), (-eps, tm)):
                qj.copy_(q)
                vj.zero_()
                vj[j] = 1.0
                aj.zero_()
                eng.integrate(dt, qj, vj, aj)
                eng.rnea(qj, z, z, out)
            G3[:, j] = (tp - tm) / (2 * eps)

    fms, flo, fhi = timed(fd_route, reps=3)
    scale = G_ref.view(nv, nv, n).abs().amax(dim=(0, 1)).clamp(min=1.0)
    fd_err = ((G_ref.view(nv, nv, n) - G3).abs().amax(dim=(0, 1)) / scale).max().item()
    res["finite_differences"] = {"ms": fms, "ms_min": flo, "ms_max": fhi, "calls": {"integrate": 2 * nv, "rnea": 2 * nv},
                                 "speedup": fms / ms, "max_rel_difference_to_kernel": fd_err}
    del G, G_ref, qj, vj, aj, tp, tm, z
    torch.cuda.empty_cache()

    # the host-pointer call end to end at 2^18 (PCIe both ways, pageable numpy buffers), one call after a small warm-up
    nh = 1 << 18
    hq = q[:, :nh].cpu().numpy().copy()
    htau, hG = np.empty((nv, nh)), np.empty((nv * nv, nh))
    eng.gravity_gradient(hq[:, :1024].copy(), np.empty((nv, 1024)), np.empty((nv * nv, 1024)))
    t0 = time.perf_counter()
    eng.gravity_gradient(hq, htau, hG)
    hs = time.perf_counter() - t0
    dtau, dG = torch.empty((nv, 4096), dtype=torch.float64, device="cuda"), torch.empty((nv * nv, 4096), dtype=torch.float64, device="cuda")
    eng.gravity_gradient(q[:, :4096].contiguous(), dtau, dG)
    res["host"] = {"n": nh, "s": hs, "states_per_s": nh / hs, "bytes": bps * nh, "gbs": bps * nh / hs / 1e9,
                   "bit_identical_to_device_first_4096": bool(np.array_equal(hG[:, :4096], dG.cpu().numpy()))}
    line = json.dumps(res)
    print(line)
    with open(os.path.join(args.out, "gravity_gradient.jsonl"), "a") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
