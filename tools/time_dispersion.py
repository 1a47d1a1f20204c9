"""Per-material energy and dispersive band structures on one GPU: python tools/time_dispersion.py [cols] [reps] [k_points]

Phase 1, pcb_material_energy against pcb_field_energy: the same seeded columns and the same materials dielectric (Omega_1 split
into 8 materials at random on a background of eps = 2, as tools/time_materials.py: n_mat = 9, the register-bin kernels), the two
calls alternated call by call and timed with CUDA events on the context's stream; medians.  Cases: N = 120 fcc (whole planes),
N = 160 fcc (z-split half planes), N = 150 sc_curv (natural layout); and N = 120 fcc with Omega_1 split into 255 materials
(n_mat = 256, the match path).  Both calls run the same forward passes; the difference is the reduction kernel.
Phase 2, in a phase of its own (the profiler off elsewhere): torch.profiler's CUDA time of k_material_energy[_t] and k_field_energy[_t] per call.
Phase 3, a dispersive band structure: bcc_dg at N = 120, 10 bands, one gyroid network eps = 16, the other Lorentz (eps_inf = 12,
sigma = 2, f0 = 2.0) on the branch below its resonance (window (0, 2.0): above it that network's eps -> 0 expels the field and the
bands have no root), on the first k_points points of the path: seconds, LOBPCG solves and iterations per point (the first point
cold, the others warm-started in vectors and frequencies), and the same run with eps = (16, 12) for comparison.
Prints one JSON line, with the card name and power limit read in the same run."""
import importlib
import json
import os
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
os.environ.setdefault("PCB200_QUIET", "1")
pcb = importlib.import_module("linear-eigenvalue-problems-in-photonic-crystals_b200")
mfd, ne, L, dsp = pcb.discretization, pcb.numerical_experiments, pcb._lib, pcb.dispersion
from time_energy import device_info  # noqa: E402
from time_materials import ALPHA, materials_map  # noqa: E402

CASES = [(120, "fcc", "whole planes", 8), (160, "fcc", "z-split half planes", 8), (150, "sc_curv", "natural layout", 8),
         (120, "fcc", "whole planes", 255)]


def many_map(N, d_flag, n, seed=7):
    """Omega_1 split into n materials at random (eps 4 ... 13) on a background of eps = 2."""
    rng = np.random.default_rng(seed)
    mat = np.zeros(3 * N ** 3, dtype=np.uint8)
    ind = pcb.dielectric.diel_io_index(N, d_flag, dofs="edge")
    mat[ind] = rng.integers(1, n + 1, size=ind.size)
    return mat, np.concatenate(([0.5], 1.0 / np.linspace(4.0, 13.0, n)))


def energy_op(N, d_flag, n):
    relax, pnt = mfd.set_relaxation(ALPHA)
    a_fft, b_fft = mfd.fft_blocks(N, 1, pcb.dielectric.diel_info(d_flag, option="ct"), alpha=ALPHA)
    inv_fft = mfd.inverse_3_times_3_B(b_fft, pnt, relax[0])
    mat, inv_eps = materials_map(N, d_flag) if n == 8 else many_map(N, d_flag, n)
    return ne.pc_mfd_handle(a_fft, (pnt * b_fft[0], pnt * b_fft[1]), mfd.DielHandle.materials(N, mat, inv_eps), inv_fft,
                            relax[0])[0].op


def phase_calls(m, reps):
    out = []
    for N, d_flag, structure, n in CASES:
        ctx = pcb.get_context(N)
        op = energy_op(N, d_flag, n)
        X = ctx.random_block(m, 2024)
        calls = {"material_energy": lambda: op.material_energy(X), "field_energy": lambda: op.field_energy(X)}
        for _ in range(3):
            for f in calls.values():
                f()
        t = {k: [] for k in calls}
        for _ in range(reps):
            for k, f in calls.items():
                ctx.timer_start()
                f()
                t[k].append(ctx.timer_stop())
        med = {k: float(np.median(v)) for k, v in t.items()}
        e = op.material_energy(X)
        e_in, e_tot = op.field_energy(X)
        out.append({"N": N, "lattice": d_flag, "structure": structure, "n_mat": n + 1, **{f"{k}_ms": v for k, v in med.items()},
                    **{f"{k}_ms_min": float(np.min(v)) for k, v in t.items()},
                    "ratio": med["material_energy"] / med["field_energy"],
                    "max_rel_sum_vs_e_tot": float(np.max(np.abs(e.sum(axis=1) - e_tot) / e_tot))})
        del X, op
        pcb.devarray.drop_contexts()
    return out


def phase_profile(m):
    import torch
    from torch.profiler import ProfilerActivity, profile
    out = []
    for N, d_flag, structure, n in CASES:
        ctx = pcb.get_context(N)
        op = energy_op(N, d_flag, n)
        X = ctx.random_block(m, 2024)
        op.material_energy(X), op.field_energy(X)
        ctx.sync()
        calls = 10
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(calls):
                op.material_energy(X)
                op.field_energy(X)
            ctx.sync()
            torch.cuda.synchronize()
        k = {}
        for ev in prof.key_averages():
            if "k_material_energy" in ev.key or "k_field_energy" in ev.key:
                name = "k_material_energy" if "material" in ev.key else "k_field_energy"
                k[name + "_ms_per_call"] = k.get(name + "_ms_per_call", 0.0) + ev.device_time_total / 1e3 / calls
        out.append({"N": N, "structure": structure, "n_mat": n + 1, **k})
        del X, op
        pcb.devarray.drop_contexts()
    return out


def phase_bands(k_points):
    out = {}
    N, d_flag, nev = 120, "bcc_dg", 10
    lor = dsp.Lorentz(12.0, [(2.0, 2.0)])
    for tag, eps, window in (("dispersive", [16.0, lor], (0.0, 2.0)), ("fixed_eps", [16.0, 12.0], None)):
        solves = {}

        def counting(H, *a, **kw):      # LOBPCG solves per k-point (the operator's alpha)
            key = tuple(np.round(np.asarray(H.op.a_fft.alpha, dtype=float), 12))
            solves[key] = solves.get(key, 0) + 1
            return pcb.lobpcg.lobpcg_sep_softlock(H, *a, **kw)

        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "bands.json")
            t0 = time.time()
            ne.bandgap(N, d_flag, solver=counting, type="materials", eps_opt=eps, indices=list(range(k_points)), nev=nev,
                       seed=1000, path=path, window=window)
            wall = time.time() - t0
            lib = json.load(open(path))
        its = lib[f"{d_flag}_{N}_iterations"][:k_points]
        fq = lib[f"{d_flag}_{N}_frequencies"][:k_points]
        n_s = list(solves.values())
        out[tag] = {"wall_s": wall, "phase_seconds": {k: round(v, 3) for k, v in ne.bandgap.last_timing.items()},
                    "points": [{"lobpcg_solves": n_s[i] if i < len(n_s) else None,
                                "solves_per_band": n_s[i] / nev if i < len(n_s) else None,
                                "lobpcg_iterations": its[i][0], "lobpcg_seconds": its[i][1], "frequencies": fq[i]}
                               for i in range(k_points)]}
    return out


def main():
    m = int(sys.argv[1]) if len(sys.argv) > 1 else 16
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 40
    k_points = int(sys.argv[3]) if len(sys.argv) > 3 else 3
    res = {"cols": m, "reps": reps, **device_info()}
    res["calls"] = phase_calls(m, reps)
    res["profile"] = phase_profile(m)
    res["bands"] = phase_bands(k_points)
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
