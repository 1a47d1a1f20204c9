"""Device time of the H apply with the materials dielectric against the chiral one on the same structure:
python tools/time_materials.py [cols] [reps]

Cases: N = 120 fcc (whole planes), N = 160 fcc (z-split half planes), N = 150 sc_curv (five-pass operator).  The lattice's Omega_1
is split into 8 materials at random (eps 4 ... 13) on a background of eps = 2.  Three operators alternate call by call, so that
all see the same clocks: the materials H, the chiral H with the seven-sweep plane pass ("mid_five" 0, the pass structure the
materials H runs) and the chiral H with the default options (the five-sweep k_mid2 at N = 120).  Each call is timed with CUDA
events on the context's stream; the medians are reported.  Bytes: the index bytes add 3 N^3 per column to the 336 N^3 an apply
moves.  Prints one JSON line, with the card name and power limit read in the same run."""
import importlib
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
os.environ.setdefault("PCB200_QUIET", "1")
pcb = importlib.import_module("linear-eigenvalue-problems-in-photonic-crystals_b200")
mfd, ne, L = pcb.discretization, pcb.numerical_experiments, pcb._lib
from time_energy import device_info  # noqa: E402

CASES = [(120, "fcc"), (160, "fcc"), (150, "sc_curv")]
ALPHA = np.array([0.3, 0.2, 0.1]) * np.pi
N_MAT, BACKGROUND = 8, 2.0


def materials_map(N, d_flag, seed=7):
    """Omega_1 of the lattice split into N_MAT materials at random: (mat, inv_eps)."""
    rng = np.random.default_rng(seed)
    mat = np.zeros(3 * N ** 3, dtype=np.uint8)
    ind = pcb.dielectric.diel_io_index(N, d_flag, dofs="edge")
    mat[ind] = rng.integers(1, N_MAT + 1, size=ind.size)
    eps = np.linspace(4.0, 13.0, N_MAT)
    return mat, np.concatenate(([1.0 / BACKGROUND], 1.0 / eps))


def main():
    m = int(sys.argv[1]) if len(sys.argv) > 1 else 16
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 60
    res = {"cols": m, "reps": reps, **device_info(), "n_mat": N_MAT, "cases": []}
    for N, d_flag in CASES:
        relax, pnt = mfd.set_relaxation(ALPHA)
        a_fft, b_fft = mfd.fft_blocks(N, 1, pcb.dielectric.diel_info(d_flag, option="ct"), alpha=ALPHA)
        inv_fft = mfd.inverse_3_times_3_B(b_fft, pnt, relax[0])
        b = (pnt * b_fft[0], pnt * b_fft[1])
        ctx = pcb.get_context(N)
        mat, inv_eps = materials_map(N, d_flag)
        ops = {}
        ops["materials"] = ne.pc_mfd_handle(a_fft, b, mfd.DielHandle.materials(N, mat, inv_eps), inv_fft, relax[0])[1].op
        ctx.option("mid_five", 0)
        ops["chiral_seven_sweep"] = ne.pc_mfd_handle(a_fft, b, mfd.chiral_handle(N, d_flag), inv_fft, relax[0])[1].op
        ctx.option("mid_five", -1)
        ops["chiral_default"] = ne.pc_mfd_handle(a_fft, b, mfd.chiral_handle(N, d_flag), inv_fft, relax[0])[1].op
        X, Y = ctx.random_block(m, 2024), ctx.empty(m)
        for _ in range(3):
            for op in ops.values():
                op.apply_into(L.APPLY_H, X, Y)
        ctx.sync()
        t = {k: [] for k in ops}
        for _ in range(reps):
            for k, op in ops.items():
                ctx.timer_start()
                op.apply_into(L.APPLY_H, X, Y)
                t[k].append(ctx.timer_stop())
        med = {k: float(np.median(v)) for k, v in t.items()}
        res["cases"].append({
            "N": N, "lattice": d_flag, "structure": "natural (five-pass)" if N % 8 else ("z-split planes" if N > 120 else "whole planes"),
            **{f"H_{k}_ms": v for k, v in med.items()},
            **{f"H_{k}_ms_min": float(np.min(v)) for k, v in t.items()},
            "materials_over_chiral_same_structure": med["materials"] / med["chiral_seven_sweep"],
            "materials_over_chiral_default": med["materials"] / med["chiral_default"],
        })
        del X, Y, ops
        pcb.devarray.drop_contexts()
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
