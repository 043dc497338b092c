"""Inverse-dynamics derivatives on the benchmark humanoid (H37: 32 bodies, 37 DoFs): the device call at 2^20 states timed with CUDA
events after warm-up, the Coriolis-matrix call on the same batch (two nv x nv matrices written per state as well) for comparison, the
finite-difference route a user had before (per column 2 calls each of mecano_b200_integrate and mecano_b200_rnea for d tau / dq and 2
calls of mecano_b200_rnea for d tau / dqd, assembled into the same matrices) timed on the same batch, and the host-pointer call end to
end at 2^18.  Bytes are computed from shapes (kernel_info bytes_per_state: q, qd, qdd read, tau and both matrices written); the HBM
fraction is against the read+write copy peak measured in the same run.  Device name, power limit and the kernel's registers, local
memory and launch configuration are read in the same call.  Writes one JSON line to <out>/rnea_derivatives.jsonl.

    python scripts/gpu_rnea_derivatives.py [--out DIR]
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
    """Median, min and max of `reps` calls in ms, CUDA events, after one warm-up call.  The matrices (23 GB at 2^20 states) are far beyond L2."""
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
    ap.add_argument("--out", default=".", help="directory that receives rnea_derivatives.jsonl")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    assert torch.cuda.is_available(), "needs a CUDA device"
    system = bench.build_system(2)
    nv, nq = system.getNumberOfDoFs(), system.getConfigurationMatrixSize()
    calc = mb.InverseDynamicsDerivativesCalculator(system)
    calc.setGravitationalAcceleration(-9.81)
    eng = calc._engine
    hbm_gbs = mb.measure_hbm_peak(0)
    res = {"tree": "H37", "nv": nv, "nq": nq, "device": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(), "hbm_peak_copy_gbs": hbm_gbs}
    rng = np.random.default_rng(1)

    n = 1 << 20
    q, qd, qdd = (torch.from_numpy(x).cuda() for x in mb.MultiBodySystemRandomTools.nextState(rng, system, n)[:3])
    new = lambda rows: torch.empty((rows, n), dtype=torch.float64, device="cuda")  # noqa: E731
    tau, dq, dqd = new(nv), new(nv * nv), new(nv * nv)
    info = calc.kernelInfo(n)
    ms, lo, hi = timed(lambda: eng.rnea_derivatives(q, qd, qdd, tau, dq, dqd))
    bps = info["bytes_per_state"]
    res["kernel"] = {"n": n, "ms": ms, "ms_min": lo, "ms_max": hi, "states_per_s": n / (ms * 1e-3), "bytes": bps * n, "gbs": bps * n / (ms * 1e-3) / 1e9,
                     "hbm_fraction": bps * n / (ms * 1e-3) / 1e9 / hbm_gbs, "regs": info["regs_per_thread"], "local_bytes": info["local_bytes_per_thread"],
                     "block": info["block_threads"], "blocks_per_sm": info["blocks_per_sm"], "dynamic_smem": info["dynamic_smem_bytes"],
                     "stack_doubles": info["stack_doubles"]}
    dq_ref, dqd_ref = dq.clone(), dqd.clone()

    # the mass and Coriolis matrices of the same states (mecano_b200_coriolis): two nv^2 matrices written per state as well
    cms, clo, chi = timed(lambda: eng.coriolis(q, qd, dq, dqd))
    cinfo = eng.kernel_info(3, n)
    res["coriolis"] = {"ms": cms, "ms_min": clo, "ms_max": chi, "gbs": cinfo["bytes_per_state"] * n / (cms * 1e-3) / 1e9,
                       "hbm_fraction": cinfo["bytes_per_state"] * n / (cms * 1e-3) / 1e9 / hbm_gbs,
                       "block": cinfo["block_threads"], "blocks_per_sm": cinfo["blocks_per_sm"], "regs": cinfo["regs_per_thread"]}

    # the route without this calculator: central differences, column by column, through the integrator and inverse dynamics
    eps = 1e-5
    z = torch.zeros((nv, n), dtype=torch.float64, device="cuda")
    qj, vj, aj = torch.empty_like(q), new(nv), new(nv)
    tp, tm = new(nv), new(nv)
    D3q, D3v = dq.view(nv, nv, n), dqd.view(nv, nv, n)

    def fd_route():
        for j in range(nv):
            for dt, out in ((eps, tp), (-eps, tm)):
                qj.copy_(q)
                vj.zero_()
                vj[j] = 1.0
                aj.zero_()
                eng.integrate(dt, qj, vj, aj)
                eng.rnea(qj, qd, qdd, out)
            D3q[:, j] = (tp - tm) / (2 * eps)
            for dt, out in ((eps, tp), (-eps, tm)):
                vj.copy_(qd)
                vj[j] += dt
                eng.rnea(q, vj, qdd, out)
            D3v[:, j] = (tp - tm) / (2 * eps)

    fms, flo, fhi = timed(fd_route, reps=3)
    errs = {}
    for name, ref, D in (("dtau_dq", dq_ref, D3q), ("dtau_dqd", dqd_ref, D3v)):
        r3 = ref.view(nv, nv, n)
        scale = r3.abs().amax(dim=(0, 1)).clamp(min=1.0)
        errs[name] = ((r3 - D).abs().amax(dim=(0, 1)) / scale).max().item()
    res["finite_differences"] = {"ms": fms, "ms_min": flo, "ms_max": fhi, "calls": {"integrate": 2 * nv, "rnea": 4 * nv},
                                 "speedup": fms / ms, "max_rel_difference_to_kernel": errs}
    del dq, dqd, dq_ref, dqd_ref, qj, vj, aj, tp, tm, z
    torch.cuda.empty_cache()

    # the host-pointer call end to end at 2^18 (PCIe both ways, pageable numpy buffers), one call after a small warm-up
    nh = 1 << 18
    hq, hv, ha = (x[:, :nh].cpu().numpy().copy() for x in (q, qd, qdd))
    htau, hdq, hdqd = np.empty((nv, nh)), np.empty((nv * nv, nh)), np.empty((nv * nv, nh))
    eng.rnea_derivatives(hq[:, :1024].copy(), hv[:, :1024].copy(), ha[:, :1024].copy(), np.empty((nv, 1024)), np.empty((nv * nv, 1024)),
                         np.empty((nv * nv, 1024)))
    t0 = time.perf_counter()
    eng.rnea_derivatives(hq, hv, ha, htau, hdq, hdqd)
    hs = time.perf_counter() - t0
    m = 4096
    dtau, ddq, ddqd = (torch.empty((r, m), dtype=torch.float64, device="cuda") for r in (nv, nv * nv, nv * nv))
    eng.rnea_derivatives(q[:, :m].contiguous(), qd[:, :m].contiguous(), qdd[:, :m].contiguous(), dtau, ddq, ddqd)
    res["host"] = {"n": nh, "s": hs, "states_per_s": nh / hs, "bytes": bps * nh, "gbs": bps * nh / hs / 1e9,
                   "bit_identical_to_device_first_4096": bool(np.array_equal(hdq[:, :m], ddq.cpu().numpy()) and np.array_equal(hdqd[:, :m], ddqd.cpu().numpy()))}
    line = json.dumps(res)
    print(line)
    with open(os.path.join(args.out, "rnea_derivatives.jsonl"), "a") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
