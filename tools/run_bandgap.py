"""Full band-structure runs (BASELINE configs 2-4): [torchrun ...] tools/run_bandgap.py N d_flag type [nev] [max_k] [--energy] [--velocity]
    [--eps e1,e2,...] [--window lo,hi]

Single process: numerical_experiments.bandgap over the whole k-path on one GPU.  Under torch.distributed.run: bandgap_sharded,
one contiguous k-chunk per GPU, rank 0 merges the rows into the reference-format JSON (output/<type>/bandgap_<d_flag>.json
under --out).  Prints one JSON line with the wall time, per-k seconds and iteration statistics.  --energy also records, per k-point,
the fraction of each band's electric energy inside the dielectric ("<d_flag>_<N>_energy_fraction" in the JSON); --velocity the group
velocity of each band along the path ("<d_flag>_<N>_group_velocity", null for the zero modes at Gamma).  --eps sets eps_opt: one
permittivity per region for type materials (bcc_dg: its two gyroid networks, e.g. --eps 16,12), else one value.  For type materials
an entry may also be dispersive, drude:EPS_INF:FP or lorentz:EPS_INF:SIGMA:F0 (e.g. --eps 16,lorentz:12:2:2.0): the frequency rows
then hold the self-consistent frequencies, in the highest admissible window or in --window lo,hi (e.g. --window 0,2.0, the branch
below the Lorentz resonance)."""
import importlib
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ.setdefault("PCB200_QUIET", "1")


def parse_eps(item, dsp):
    """One --eps entry: a number, drude:EPS_INF:FP or lorentz:EPS_INF:SIGMA:F0."""
    parts = item.split(":")
    if parts[0] == "drude" and len(parts) == 3:
        return dsp.Drude(float(parts[1]), float(parts[2]))
    if parts[0] == "lorentz" and len(parts) == 4:
        return dsp.Lorentz(float(parts[1]), [(float(parts[2]), float(parts[3]))])
    if len(parts) != 1:
        raise SystemExit(f"--eps entry {item!r}: expected a number, drude:EPS_INF:FP or lorentz:EPS_INF:SIGMA:F0")
    return float(item)


def main():
    energy = "--energy" in sys.argv[1:]
    velocity = "--velocity" in sys.argv[1:]
    args = sys.argv[1:]
    eps, window = None, None
    if "--eps" in args:
        i = args.index("--eps")
        eps = args[i + 1].split(",")
        del args[i:i + 2]
    if "--window" in args:
        i = args.index("--window")
        window = tuple(float(v) for v in args[i + 1].split(","))
        del args[i:i + 2]
    argv = [sys.argv[0]] + [a for a in args if a not in ("--energy", "--velocity")]
    N, d_flag, typ = int(argv[1]), argv[2], argv[3]
    pcb = importlib.import_module("linear-eigenvalue-problems-in-photonic-crystals_b200")
    if eps is not None:
        eps = [parse_eps(v, pcb.dispersion) if typ == "materials" else float(v) for v in eps]
    eps_opt = 0 if eps is None else (eps if typ == "materials" else eps[0])
    nev = int(argv[4]) if len(argv) > 4 else 10
    max_k = int(argv[5]) if len(argv) > 5 else 0
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    gather = None
    if world > 1:
        import torch.distributed as td
        td.init_process_group(backend="gloo")

        def gather(obj):
            out = [None] * world if rank == 0 else None
            td.gather_object(obj, out, dst=0)
            return out
    pcb.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    ne = pcb.numerical_experiments
    n_k = pcb.dielectric.kpath(d_flag).shape[0]
    indices = list(range(n_k if max_k <= 0 else min(max_k, n_k)))
    out_dir = os.path.join("gpurun_out", "bands", typ) + "/"
    os.makedirs(out_dir, exist_ok=True)
    final = os.path.join(out_dir, f"bandgap_{d_flag}.json")
    if rank == 0 and os.path.exists(final):
        os.remove(final)
    if world > 1:
        td.barrier()
    t0 = time.time()
    rows = ne.bandgap_sharded(N, d_flag, rank, world, type=typ, eps_opt=eps_opt, nev=nev, seed=1000, out_dir=out_dir,
                              indices=indices, gather=gather if world > 1 else (lambda o: [o]), energy=energy,
                              velocity=velocity, window=window)
    wall = time.time() - t0
    if world > 1:
        td.barrier()
        wall = time.time() - t0
    if rank == 0:
        lib = json.load(open(final))
        its = np.array(lib[f"{d_flag}_{N}_iterations"])[indices]
        ok = its[:, 0] > 0
        print(json.dumps({"N": N, "lattice": d_flag, "type": typ, "nev": nev, "gpus": world, "k_points": len(indices),
                          "failed": int((~ok).sum()), "wall_s_incl_setup": wall, "sum_solver_s": float(its[ok, 1].sum()),
                          "mean_s_per_k": float(its[ok, 1].mean()), "mean_iterations": float(its[ok, 0].mean()),
                          "std_iterations": float(its[ok, 0].std()), "json": final,
                          "rank0_phase_seconds": {k: round(v, 3) for k, v in getattr(ne.bandgap, "last_timing", {}).items()}}), flush=True)
    if world > 1:
        td.destroy_process_group()


if __name__ == "__main__":
    main()
