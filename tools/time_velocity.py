"""Device time of pcb_band_velocity against the A apply on the same seeded columns: python tools/time_velocity.py [reps]

Cases: N = 120 fcc chiral (whole planes), N = 160 bcc_dg cross-DoF (half planes), N = 150 sc_curv chiral (five-pass), each at 10
and 16 columns.  The velocity call, the A apply and the E^ apply (PCB_APPLY_EFOURIER) alternate so that they see the same clocks;
each call is timed with CUDA events on the context's stream (medians).  A second, separate phase runs torch.profiler over the
velocity calls for k_band_velocity's own time.  Counts of the reduction: 48 n^2 N^3 FP64 flops (6 n^2 complex FMAs per point)
and 2 n 48 N^3 bytes (X and E^ read once); floors at the measured FP64 rate (profiles/r01_fp64_peak.log, 37.2 TFLOP/s) and
6538.6 GB/s.  Prints one JSON line."""
import importlib
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ.setdefault("PCB200_QUIET", "1")
pcb = importlib.import_module("linear-eigenvalue-problems-in-photonic-crystals_b200")
mfd, ne, L = pcb.discretization, pcb.numerical_experiments, pcb._lib

CASES = [(120, "fcc", "chiral"), (160, "bcc_dg", "pseudochiral_crossdof"), (150, "sc_curv", "chiral")]
WIDTHS = (10, 16)
ALPHA = np.array([0.3, 0.2, 0.1]) * np.pi
FP64_TFLOPS, HBM_GBPS = 37.2, 6538.6


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(pcb.devarray.default_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"device": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:      # the timings stand without it, but say so
        return {"device": "unknown", "power_limit": f"not read: {e}"}


def kernel_ms(op, X, calls=20):
    """Mean device time of k_band_velocity per velocity call, from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            op.band_velocity(X)
    tot = 0.0
    for ev in prof.key_averages():
        if "k_band_velocity" in ev.key:
            t = getattr(ev, "device_time_total", None)
            tot += (t if t is not None else ev.cuda_time_total) / 1e3
    return tot / calls


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 40
    res = {"reps": reps, **device_info(), "cases": []}
    for N, d_flag, typ in CASES:
        relax, pnt = mfd.set_relaxation(ALPHA)
        a_fft, b_fft = mfd.fft_blocks(N, 1, pcb.dielectric.diel_info(d_flag, option="ct"), alpha=ALPHA)
        inv_fft = mfd.inverse_3_times_3_B(b_fft, pnt, relax[0])
        Diels = getattr(mfd, typ + "_handle")(N, d_flag)
        A = ne.pc_mfd_handle(a_fft, (pnt * b_fft[0], pnt * b_fft[1]), Diels, inv_fft, relax[0])[0]
        op, ctx = A.op, pcb.get_context(N)
        for m in WIDTHS:
            X, Y = ctx.random_block(m, 2024), ctx.empty(m)
            for _ in range(3):
                op.band_velocity(X)
                op.apply_into(L.APPLY_A, X, Y)
                op.apply_into(L.APPLY_EFOURIER, X, Y)
            ctx.sync()
            t_v, t_a, t_e = [], [], []
            for _ in range(reps):
                for mode, acc in ((None, t_v), (L.APPLY_A, t_a), (L.APPLY_EFOURIER, t_e)):
                    ctx.timer_start()
                    if mode is None:
                        op.band_velocity(X)
                    else:
                        op.apply_into(mode, X, Y)
                    acc.append(ctx.timer_stop())
            nn = N ** 3
            flops, nbytes = 48.0 * m * m * nn, 2.0 * m * 48 * nn
            floor_f, floor_b = flops / (FP64_TFLOPS * 1e12) * 1e3, nbytes / (HBM_GBPS * 1e9) * 1e3
            k_ms = kernel_ms(op, X)
            v_med, a_med = float(np.median(t_v)), float(np.median(t_a))
            res["cases"].append({
                "N": N, "lattice": d_flag, "type": typ, "cols": m,
                "velocity_ms": v_med, "velocity_ms_min": float(np.min(t_v)), "apply_A_ms": a_med,
                "ratio_velocity_over_A": v_med / a_med, "efourier_ms": float(np.median(t_e)),
                "kernel_ms": k_ms, "kernel_GFLOPs": flops / (k_ms * 1e-3) / 1e9 if k_ms > 0 else None,
                "kernel_GBps": nbytes / (k_ms * 1e-3) / 1e9 if k_ms > 0 else None,
                "floor_fp64_ms": floor_f, "floor_hbm_ms": floor_b,
                "share_of_larger_floor": max(floor_f, floor_b) / k_ms if k_ms > 0 else None,
            })
            del X, Y
        del A, op, Diels
        pcb.devarray.drop_contexts()
        ctx.trim()
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
