"""Forward-dynamics derivatives on the benchmark humanoid (H37: 32 bodies, 37 DoFs), all in one run:
  * the whole device call at 2^20 states, CUDA events after warm-up;
  * its three reused launches alone on the same batch (mecano_b200_aba, mecano_b200_rnea_derivatives, mecano_b200_crba), their sum,
    and the new L^T D L solve kernel alone from a torch.profiler trace of the whole call taken afterwards (profiler off for every
    other timing); the solve's bytes (M read, both partials read and written, M^-1 written: 6 nv^2 doubles per state) over its
    time, against the read+write copy peak measured in the same run;
  * the finite-difference route a user had before: per column 2 calls each of mecano_b200_integrate and mecano_b200_aba for
    d qdd / dq, 2 calls of mecano_b200_aba for d qdd / dqd and 2 for M^-1, assembled into the same matrices, timed on the same batch,
    with the largest difference to the analytic result;
  * the host-pointer call end to end at 2^18 states (pageable numpy buffers).
Device name and power limit are read in the same call.  Writes one JSON line to <out>/aba_derivatives.jsonl.

    python scripts/gpu_aba_derivatives.py [--out DIR]
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
    """Median, min and max of `reps` calls in ms, CUDA events, after one warm-up call.  The matrices (11.5 GB each at 2^20 states)
    are far beyond L2."""
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


def kernel_times_ms(fn, reps=5):
    """{kernel name: mean device time per call in ms} from a torch.profiler trace of `reps` calls."""
    from torch.profiler import ProfilerActivity, profile

    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if ev.device_type.name == "CUDA" or getattr(ev, "self_device_time_total", 0) > 0:
            t = getattr(ev, "self_device_time_total", None)
            if t is None:
                t = ev.self_cuda_time_total
            out[ev.key] = out.get(ev.key, 0.0) + t / 1e3 / reps
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=".", help="directory that receives aba_derivatives.jsonl")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    assert torch.cuda.is_available(), "needs a CUDA device"
    system = bench.build_system(2)
    nv, nq = system.getNumberOfDoFs(), system.getConfigurationMatrixSize()
    calc = mb.ForwardDynamicsDerivativesCalculator(system)
    calc.setGravitationalAcceleration(-9.81)
    eng = calc._engine
    hbm_gbs = mb.measure_hbm_peak(0)
    res = {"tree": "H37", "nv": nv, "nq": nq, "device": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(), "hbm_peak_copy_gbs": hbm_gbs}
    rng = np.random.default_rng(1)

    n = 1 << 20
    q, qd, _, tau = (torch.from_numpy(x).cuda() for x in mb.MultiBodySystemRandomTools.nextState(rng, system, n))
    new = lambda rows: torch.empty((rows, n), dtype=torch.float64, device="cuda")  # noqa: E731
    qdd, dq, dqd, minv = new(nv), new(nv * nv), new(nv * nv), new(nv * nv)
    call = lambda: eng.aba_derivatives(q, qd, tau, qdd, dq, dqd, minv)  # noqa: E731
    ms, lo, hi = timed(call)
    res["call"] = {"n": n, "ms": ms, "ms_min": lo, "ms_max": hi, "states_per_s": n / (ms * 1e-3)}

    # the three reused launches alone, on the same batch and buffers
    qdd2, tau2 = new(nv), new(nv)
    parts = {"aba": timed(lambda: eng.aba(q, qd, tau, qdd2)),
             "rnea_derivatives": timed(lambda: eng.rnea_derivatives(q, qd, qdd2, tau2, dq, dqd)),
             "crba": timed(lambda: eng.crba(q, minv))}
    res["reused"] = {k: {"ms": v[0], "ms_min": v[1], "ms_max": v[2]} for k, v in parts.items()}
    res["reused_sum_ms"] = sum(v[0] for v in parts.values())
    call()
    torch.cuda.synchronize()
    ref = [x.clone() for x in (qdd, dq, dqd, minv)]
    res["qdd_bit_identical_to_aba"] = bool(torch.equal(ref[0], qdd2))

    # the solve kernel alone, from a profiler trace of the whole call
    kt = kernel_times_ms(call)
    solve = [v for k, v in kt.items() if "ltdl_solve_kernel" in k]
    solve_ms = solve[0] if solve else None
    solve_bytes = 6.0 * nv * nv * 8 * n
    res["solve_kernel"] = {"ms_profiler": solve_ms, "bytes": solve_bytes, "bytes_per_state": solve_bytes / n,
                           "gbs": solve_bytes / (solve_ms * 1e-3) / 1e9 if solve_ms else None,
                           "hbm_fraction": solve_bytes / (solve_ms * 1e-3) / 1e9 / hbm_gbs if solve_ms else None,
                           "ms_call_minus_reused": ms - res["reused_sum_ms"]}
    res["profiler_kernels_ms"] = {k[:120]: v for k, v in sorted(kt.items(), key=lambda kv: -kv[1])[:8]}

    # the route without this call: central differences, column by column, through the integrator and forward dynamics
    eps = 1e-5
    qj, vj, aj = torch.empty_like(q), new(nv), new(nv)
    tj = new(nv)
    ap_, am_ = new(nv), new(nv)
    Dq, Dv, Dt = dq.view(nv, nv, n), dqd.view(nv, nv, n), minv.view(nv, nv, n)

    def fd_route():
        for j in range(nv):
            for dt, out in ((eps, ap_), (-eps, am_)):
                qj.copy_(q)
                vj.zero_()
                vj[j] = 1.0
                aj.zero_()
                eng.integrate(dt, qj, vj, aj)
                eng.aba(qj, qd, tau, out)
            Dq[:, j] = (ap_ - am_) / (2 * eps)
            for dt, out in ((eps, ap_), (-eps, am_)):
                vj.copy_(qd)
                vj[j] += dt
                eng.aba(q, vj, tau, out)
            Dv[:, j] = (ap_ - am_) / (2 * eps)
            for dt, out in ((1.0, ap_), (-1.0, am_)):
                tj.copy_(tau)
                tj[j] += dt
                eng.aba(q, qd, tj, out)
            Dt[:, j] = (ap_ - am_) / 2.0

    fms, flo, fhi = timed(fd_route, reps=3)
    errs = {}
    for name, r, D in (("dqdd_dq", ref[1], Dq), ("dqdd_dqd", ref[2], Dv), ("minv", ref[3], Dt)):
        r3 = r.view(nv, nv, n)
        scale = r3.abs().amax(dim=(0, 1)).clamp(min=1.0)
        errs[name] = ((r3 - D).abs().amax(dim=(0, 1)) / scale).max().item()
    res["finite_differences"] = {"ms": fms, "ms_min": flo, "ms_max": fhi, "calls": {"integrate": 2 * nv, "aba": 6 * nv},
                                 "speedup": fms / ms, "max_rel_difference_to_call": errs}
    del dq, dqd, minv, ref, qj, vj, aj, tj, ap_, am_, Dq, Dv, Dt
    torch.cuda.empty_cache()

    # the host-pointer call end to end at 2^18 (PCIe both ways, pageable numpy buffers), one call after a small warm-up
    nh = 1 << 18
    hq, hv, ht = (x[:, :nh].cpu().numpy().copy() for x in (q, qd, tau))
    hout = [np.empty((nv, nh)), np.empty((nv * nv, nh)), np.empty((nv * nv, nh)), np.empty((nv * nv, nh))]
    eng.aba_derivatives(hq[:, :1024].copy(), hv[:, :1024].copy(), ht[:, :1024].copy(), np.empty((nv, 1024)), *[np.empty((nv * nv, 1024)) for _ in range(3)])
    t0 = time.perf_counter()
    eng.aba_derivatives(hq, hv, ht, *hout)
    hs = time.perf_counter() - t0
    res["host"] = {"n": nh, "s": hs, "states_per_s": nh / hs}
    line = json.dumps(res)
    print(line)
    with open(os.path.join(args.out, "aba_derivatives.jsonl"), "a") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
