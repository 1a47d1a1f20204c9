"""Device time of pcb_field_energy against the A apply on the same seeded columns: python tools/time_energy.py [cols] [reps]

Cases: N = 120 fcc chiral (whole planes), N = 160 bcc_dg cross-DoF (half planes), N = 150 sc_curv chiral (natural layout).
The two calls alternate (energy, A, energy, A, ...) so that both see the same clocks; each call is timed with CUDA events on the
context's stream.  A second, separate phase runs torch.profiler over the energy calls for the reduction kernel's own time.
Bytes: the energy call moves 5C + N^3 per column (x read, x-forward store, plane / y, z passes read + store, reduction read;
C = 48 N^3 = one column), the reduction kernel 1C + N^3 (the field and the mask byte).  Prints one JSON line."""
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
ALPHA = np.array([0.3, 0.2, 0.1]) * np.pi


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(pcb.devarray.default_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"device": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:      # the timings stand without it, but say so
        return {"device": "unknown", "power_limit": f"not read: {e}"}


def kernel_ms(op, X, calls=20):
    """Mean device time of the reduction kernel (k_field_energy*) per energy call, from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            op.field_energy(X)
    tot, names = 0.0, set()
    for ev in prof.key_averages():
        if "k_field_energy" in ev.key:
            t = getattr(ev, "device_time_total", None)
            tot += (t if t is not None else ev.cuda_time_total) / 1e3
            names.add(ev.key.split("(")[0])
    return tot / calls, sorted(names)


def main():
    m = int(sys.argv[1]) if len(sys.argv) > 1 else 16
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 60
    res = {"cols": m, "reps": reps, **device_info(), "cases": []}
    for N, d_flag, typ in CASES:
        relax, pnt = mfd.set_relaxation(ALPHA)
        a_fft, b_fft = mfd.fft_blocks(N, 1, pcb.dielectric.diel_info(d_flag, option="ct"), alpha=ALPHA)
        inv_fft = mfd.inverse_3_times_3_B(b_fft, pnt, relax[0])
        Diels = getattr(mfd, typ + "_handle")(N, d_flag)
        A = ne.pc_mfd_handle(a_fft, (pnt * b_fft[0], pnt * b_fft[1]), Diels, inv_fft, relax[0])[0]
        op, ctx = A.op, pcb.get_context(N)
        X, Y = ctx.random_block(m, 2024), ctx.empty(m)
        for _ in range(3):
            op.field_energy(X)
            op.apply_into(L.APPLY_A, X, Y)
        ctx.sync()
        t_e, t_a = [], []
        for _ in range(reps):
            ctx.timer_start()
            op.field_energy(X)
            t_e.append(ctx.timer_stop())
            ctx.timer_start()
            op.apply_into(L.APPLY_A, X, Y)
            t_a.append(ctx.timer_stop())
        nn = N ** 3
        C = 48 * nn
        k_ms, k_names = kernel_ms(op, X)
        e_med, a_med = float(np.median(t_e)), float(np.median(t_a))
        res["cases"].append({
            "N": N, "lattice": d_flag, "type": typ,
            "layout": "plane" if (N % 8 == 0 and N <= 160) else "natural",
            "energy_ms": e_med, "energy_ms_min": float(np.min(t_e)), "energy_ms_mean": float(np.mean(t_e)),
            "apply_A_ms": a_med, "apply_A_ms_min": float(np.min(t_a)), "ratio_energy_over_A": e_med / a_med,
            "bytes_per_col_call": 5 * C + nn, "call_GBps": m * (5 * C + nn) / (e_med * 1e-3) / 1e9,
            "reduction_kernels": k_names, "reduction_ms": k_ms, "bytes_per_col_reduction": C + nn,
            "reduction_GBps": m * (C + nn) / (k_ms * 1e-3) / 1e9 if k_ms > 0 else None,
        })
        del X, Y, A, op, Diels
        pcb.devarray.drop_contexts()
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
