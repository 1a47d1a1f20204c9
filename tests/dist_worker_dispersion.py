"""Worker for tests/test_dispersion.py: one rank of a world-size-2 gloo job on the CPU (host-emulation build of the kernels).
Runs numerical_experiments.bandgap_sharded with a dispersive material (a Drude network of the double gyroid) on a 4-point slice
of the k-path; rank 0 writes the merged JSON."""
import importlib
import os
import sys

import torch.distributed as td

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ["PCB200_QUIET"] = "1"


def main():
    out_dir, lib = sys.argv[1], sys.argv[2]
    td.init_process_group(backend="gloo")
    rank, world = td.get_rank(), td.get_world_size()
    pcb = importlib.import_module("linear-eigenvalue-problems-in-photonic-crystals_b200")
    pcb._lib.use_library(lib)
    pcb.set_device(0)

    def gather(obj):
        out = [None] * world if rank == 0 else None
        td.gather_object(obj, out, dst=0)
        return out

    eps = [16.0, pcb.dispersion.Drude(12.0, 0.5)]
    pcb.numerical_experiments.bandgap_sharded(8, "bcc_dg", rank, world, type="materials", eps_opt=eps, nev=4, seed=1000,
                                              out_dir=out_dir + "/", indices=[1, 2, 3, 4], gather=gather, energy=True)
    td.barrier()
    td.destroy_process_group()


if __name__ == "__main__":
    main()
