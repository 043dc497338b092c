"""Joint-torque regressor on the benchmark humanoid (H37: 32 bodies, 37 DoFs): the device call at 2^16 and 2^18 states timed with
CUDA events after warm-up, the mass-matrix call on the same batch for comparison, and the host-pointer call end to end at 2^18.
Bytes are computed from shapes (kernel_info bytes_per_state: q, qd, qdd read, Y written); the HBM fraction is against the
read+write copy peak measured in the same run.  Device name, power limit and the kernel's registers / local memory are read in
the same call.  Writes one JSON line to <out>/regressor.jsonl.

    python scripts/gpu_regressor.py [--out DIR]
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
    """Median of `reps` launches in ms, CUDA events, after one warm-up launch.  Y (>= 6 GB) is far beyond L2."""
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
    ap.add_argument("--out", default=".", help="directory that receives regressor.jsonl")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    assert torch.cuda.is_available(), "needs a CUDA device"
    system = bench.build_system(2)
    nv, nq = system.getNumberOfDoFs(), system.getConfigurationMatrixSize()
    reg = mb.JointTorqueRegressorCalculator(system)
    reg.setGravitationalAcceleration(-9.81)
    crba = mb.CompositeRigidBodyMassMatrixCalculator(system)
    nb = reg._engine.nb
    hbm_gbs = mb.measure_hbm_peak(0)
    res = {"tree": "H37", "nb": nb, "nv": nv, "nq": nq, "device": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(),
           "hbm_peak_copy_gbs": hbm_gbs, "runs": []}
    rng = np.random.default_rng(1)
    for log2n in (16, 18):
        n = 1 << log2n
        q, qd, qdd, _ = mb.MultiBodySystemRandomTools.nextState(rng, system, n)
        tq, tqd, tqdd = (torch.from_numpy(x).cuda() for x in (q, qd, qdd))
        Y = torch.empty((nv * 10 * nb, n), dtype=torch.float64, device="cuda")
        M = torch.empty((nv * nv, n), dtype=torch.float64, device="cuda")
        info = reg.kernelInfo(n)
        ms, lo, hi = timed(lambda: reg._engine.joint_torque_regressor(tq, tqd, tqdd, Y))
        mms, mlo, mhi = timed(lambda: crba.getMassMatrix(tq, massMatrix=M))
        minfo = crba.kernelInfo(n)
        run = {"n": n,
               "regressor": {"ms": ms, "ms_min": lo, "ms_max": hi, "states_per_s": n / (ms * 1e-3), "bytes": info["bytes_per_state"] * n,
                             "gbs": info["bytes_per_state"] * n / (ms * 1e-3) / 1e9, "hbm_fraction": info["bytes_per_state"] * n / (ms * 1e-3) / 1e9 / hbm_gbs,
                             "regs": info["regs_per_thread"], "local_bytes": info["local_bytes_per_thread"], "block": info["block_threads"],
                             "blocks_per_sm": info["blocks_per_sm"]},
               "mass_matrix": {"ms": mms, "ms_min": mlo, "ms_max": mhi, "states_per_s": n / (mms * 1e-3), "bytes": minfo["bytes_per_state"] * n,
                               "gbs": minfo["bytes_per_state"] * n / (mms * 1e-3) / 1e9, "hbm_fraction": minfo["bytes_per_state"] * n / (mms * 1e-3) / 1e9 / hbm_gbs}}
        if log2n == 18:
            # the host-pointer call end to end (PCIe both ways, pageable numpy buffers), one call after a small warm-up
            hY = np.empty((nv * 10 * nb, n))
            reg._engine.joint_torque_regressor(q[:, :1024].copy(), qd[:, :1024].copy(), qdd[:, :1024].copy(), np.empty((nv * 10 * nb, 1024)))
            t0 = time.perf_counter()
            reg._engine.joint_torque_regressor(q, qd, qdd, hY)
            hs = time.perf_counter() - t0
            run["host"] = {"s": hs, "states_per_s": n / hs, "bytes": info["bytes_per_state"] * n, "gbs": info["bytes_per_state"] * n / hs / 1e9,
                           "bit_identical_to_device_first_4096": bool(np.array_equal(hY[:, :4096], Y[:, :4096].cpu().numpy()))}
            del hY
        res["runs"].append(run)
        del Y, M, tq, tqd, tqdd
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    with open(os.path.join(args.out, "regressor.jsonl"), "a") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
