#!/usr/bin/env python3
"""Benchmark of the hot path (BASELINE.json metric: op-applies/s and seconds-to-10-bands per k-point at N=120).

    python bench.py [--gpus N --steps K --warmup W]                 # this repo's CUDA path
    python bench.py --impl reference [--gpus N --steps K --warmup W] # the reference algorithm on the host CPU

One STEP = one block application of H = A M A^H + gamma B^H B + shift to m = 16 columns (16 op-applies) of the
workload "fcc, isotropic eps=13, N=120" (BASELINE configs[1]) at one k-point of the FCC path; with N GPUs every
rank works on its own k-point of the path (k-path sharding: no data-path collective -> "weak" scaling).
Timed with CUDA events on the library's stream (pcb_timer_*), max over ranks, inputs resident in HBM
(1.33 GB per block >> 126 MB L2, so every step streams from DRAM).  Extra legs, all reported in the single JSON line:
  e2e         the same step through the reference-facing callable H_func(x) with HOST (pinned) buffers:
              upload + apply + download inside the timed region
  lobpcg      seconds to converge the lowest 10 bands (tol 1e-4) for the rank's k-points, warm-started like bandgap()
  passes      device time of each of the five kernels of one block apply (pcb_apply_timed)
  cpu_baseline the oracle's NumPy/pocketfft restatement of the same apply on the host cores (bounded sample)
With --dump-outputs DIR, rank 0 also writes the result of the last timed step to DIR (see dump_outputs): the inputs are
seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = "linear-eigenvalue-problems-in-photonic-crystals_b200"
sys.path.insert(0, ROOT)
os.environ.setdefault("PCB200_QUIET", "1")

N_GRID, NEV, M_BLOCK, LATTICE, DTYPE_TYPE = 120, 10, 16, "fcc", "chiral"
B_OP_PER_N3 = 336.0   # algorithmic bytes per op-apply / N^3 (SURVEY.md 8d, DESIGN.md "Roofline")


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.proc, self.path = None, os.path.join("/tmp", f"pcb_clocks_{os.getpid()}.csv")
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(device), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        for line in open(self.path):
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            busy = sorted(sm)[len(sm) // 2:]          # upper half = samples under load
            out.update(sm_mhz=statistics.median(busy), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        try:
            os.remove(self.path)
        except OSError:
            pass
        return out


class Dist:
    """torch.distributed plumbing for N > 1 (barrier + max-reduce of timings); nothing for N = 1."""

    def __init__(self, n_gpus):
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.td = None
        if self.world > 1:
            import torch
            import torch.distributed as td
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            use_nccl = torch.cuda.is_available()
            if use_nccl:
                torch.cuda.set_device(self.local)
            td.init_process_group(backend="nccl" if use_nccl else "gloo")
            self.td, self.torch = td, torch
            self.dev = torch.device("cuda", self.local) if use_nccl else torch.device("cpu")

    def barrier(self):
        if self.td is not None:
            self.td.barrier()

    def max(self, v):
        if self.td is None:
            return float(v)
        t = self.torch.tensor([float(v)], dtype=self.torch.float64, device=self.dev)
        self.td.all_reduce(t, op=self.td.ReduceOp.MAX)
        return float(t.item())

    def gather(self, obj):
        if self.td is None:
            return [obj]
        out = [None] * self.world if self.rank == 0 else None
        self.td.gather_object(obj, out, dst=0)
        return out

    def close(self):
        if self.td is not None:
            self.td.destroy_process_group()


def ncu_traffic(n, m, npass):
    """DRAM bytes of one launch (one m-column block apply: dram__bytes_read.sum + dram__bytes_write.sum over its passes) from the
    newest committed `ncu --set full` summary of exactly this shape, profiles/*_ncu.json (written by tools/ncu_summary.py next to
    the .md table).  A STATIC figure from that capture, not measured by this run: (value, "file @ commit") or (None, reason)."""
    import glob
    best = None
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_ncu.json"))):
        try:
            with open(path) as f:
                d = json.load(f)
        except Exception:
            continue
        if d.get("N") == n and d.get("cols") == m and d.get("passes") == npass and d.get("dram_bytes_per_apply"):
            best = (float(d["dram_bytes_per_apply"]), f"static, from {os.path.basename(path)} (commit {d.get('commit', '?')}): ncu dram__bytes_read.sum + dram__bytes_write.sum")
    return best if best else (None, "no committed ncu capture of this shape")


def fcc_alpha(pcb, rank, world):
    """k-point of this rank: first point of its contiguous chunk of the 120-point FCC path (numerical_experiments.kpath_chunks)."""
    ne = pcb.numerical_experiments
    alphas = pcb.dielectric.kpath(LATTICE)
    chunk = ne.kpath_chunks(alphas.shape[0], world)[rank]
    # rank 0's chunk starts at index 0 = first interior point of X-U; use the chunk's own k-points
    return alphas, chunk


def build_ops(pcb, n, alpha, Diels):
    mfd, ne = pcb.discretization, pcb.numerical_experiments
    relax, pnt = mfd.set_relaxation(alpha)
    ct = pcb.dielectric.diel_info(LATTICE, option="ct")
    a_fft, b_fft = mfd.fft_blocks(n, 1, ct, alpha=alpha)
    inv_fft = mfd.inverse_3_times_3_B(b_fft, pnt, relax[0])
    b_fft = (pnt * b_fft[0], pnt * b_fft[1])
    return ne.pc_mfd_handle(a_fft, b_fft, Diels, inv_fft, relax[0]), relax[0]


def host_threads():
    """Host threads the CPU legs use: every core of the box, set EXPLICITLY (torchrun exports OMP_NUM_THREADS=1 for N > 1, which
    would otherwise change the BLAS pool between the N = 1 and N > 1 runs of the reference arm)."""
    cores = os.cpu_count() or 1
    info = {"cores": cores, "scipy_fft_workers": cores, "blas_threads": None}
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        threadpool_limits(limits=cores)
        info["blas_threads"] = max([t.get("num_threads", 1) for t in threadpool_info() if t.get("user_api") == "blas"] or [1])
    except Exception:
        pass
    return info


def cpu_apply_rate(n, alpha, cols, reps, warm, workers):
    """Oracle port of AMA_BB (oracle/pc_oracle.py) on the host: op-applies/s on `cols` columns."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pc_oracle as oc
    pcb = importlib.import_module(PKG)
    oc.FFT_WORKERS = workers
    a_fft, b_fft, inv_fft, shift, _ = oc.assemble_symbols(n, LATTICE, alpha)
    ind_e = pcb.dielectric.compute_index(n, LATTICE, "edge")     # geometry only (chunked; same index set as the oracle's)
    A, H, P = oc.pc_mfd_handle(a_fft, b_fft, oc.chiral_handle(n, LATTICE, ind_e=ind_e), inv_fft, shift)
    x = oc.random_x0(3 * n ** 3, cols, 1)
    for _ in range(warm):
        H(x)
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        H(x)
        times.append(time.perf_counter() - t0)
    return cols / (sum(times) / len(times)), times


def build_ops_for(pcb, n, lattice, alpha, Diels):
    mfd, ne = pcb.discretization, pcb.numerical_experiments
    relax, pnt = mfd.set_relaxation(alpha)
    ct = pcb.dielectric.diel_info(lattice, option="ct")
    a_fft, b_fft = mfd.fft_blocks(n, 1, ct, alpha=alpha)
    inv_fft = mfd.inverse_3_times_3_B(b_fft, pnt, relax[0])
    b_fft = (pnt * b_fft[0], pnt * b_fft[1])
    return (a_fft, b_fft, inv_fft, relax[0])


def timed_passes(pcb, op, X, Y, m, reps=5):
    import ctypes as C
    L = pcb._lib
    buf, npass = (C.c_float * 8)(), C.c_int()
    acc = np.zeros(8)
    for _ in range(reps):
        L.check(L.lib().pcb_apply_timed(op.h, L.APPLY_H, m, L.ptr_array(X.ptrs), L.ptr_array(Y.ptrs), buf, C.byref(npass)), "pcb_apply_timed")
        acc += np.array(buf[:8])
    return [float(v) / reps for v in acc[:npass.value]]


def dump_outputs(out_dir, Y, seed=0):
    """Writes the result of the last timed step, Y = H X (R x m complex128 on the device), as float64 .npy files:
      H_X_sample.npy        (rows, m, 2) real and imaginary parts of Y at `rows` sorted row indices drawn with a fixed seed
                            (32 MiB: 131072 rows at m = 16), the same rows for the same N and m in every run
      H_X_column_norms.npy  (m,) the 2-norm of every column of the whole of Y"""
    Yh = Y.get()
    R, m = Yh.shape
    rows = min(R, (32 << 20) // (16 * m))
    idx = np.sort(np.random.default_rng(seed).choice(R, size=rows, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "H_X_sample.npy"), np.ascontiguousarray(Yh[idx]).view(np.float64).reshape(rows, m, 2))
    np.save(os.path.join(out_dir, "H_X_column_norms.npy"), np.linalg.norm(Yh, axis=0))


def paper2_dielectric_leg(pcb, ctx, n, m, steps, warmup, peak):
    """Extra keys: the same 16-column H block apply with the Paper-2 dielectrics (BASELINE configs[2]: bcc single gyroid,
    pseudochiral) -- the coupled 3x3 M (clusters of three CTAs in the plane pass) and the cross-DoF M (plane halves around the
    stencil kernel).  Roofline against 336 N^3 (and 432 N^3 for the cross-DoF M, whose stencil is a pass of its own)."""
    return dielectric_leg(pcb, ctx, n, m, steps, warmup, peak, "bcc_sg", ("pseudochiral_trivial", "pseudochiral_crossdof"))


def larger_grid_leg(pcb, m, steps, warmup, peak, n=160):
    """Extra key `larger_grids`: the 16-column H block apply at N = 160 (BASELINE configs[3] shape: bcc double gyroid, both
    pseudochiral discretisations; and the isotropic FCC operator) -- the z-split plane mode (half planes) instead of five passes."""
    ctx = pcb.get_context(n)
    try:
        return (dielectric_leg(pcb, ctx, n, m, steps, warmup, peak, "fcc", ("chiral",))
                + dielectric_leg(pcb, ctx, n, m, steps, warmup, peak, "bcc_dg", ("pseudochiral_trivial", "pseudochiral_crossdof")))
    finally:
        ctx.trim()


def dielectric_leg(pcb, ctx, n, m, steps, warmup, peak, lattice, types):
    mfd, ne, L = pcb.discretization, pcb.numerical_experiments, pcb._lib
    out = []
    alpha = pcb.dielectric.kpath(lattice)[0]
    sym = build_ops_for(pcb, n, lattice, alpha, None)
    X, Y = ctx.random_block(m, 4321), ctx.empty(m)
    for typ in types:
        Diels = getattr(mfd, typ + "_handle")(n, lattice)
        A, H, P = ne.pc_mfd_handle(sym[0], sym[1], Diels, sym[2], sym[3])
        for _ in range(warmup):
            H.op.apply_into(L.APPLY_H, X, Y)
        ctx.sync()
        ctx.timer_start()
        for _ in range(steps):
            H.op.apply_into(L.APPLY_H, X, Y)
        ms = ctx.timer_stop() / steps
        row = {"workload": f"{lattice} {typ} N={n} m={m} H block apply", "ms_per_step": ms, "op_applies_per_sec": m / ms * 1e3,
               "pass_ms": timed_passes(pcb, H.op, X, Y, m, 3),
               "roofline_frac_336N3": 336.0 * n ** 3 * m / (ms * 1e-3) / 1e9 / peak}
        if typ.endswith("crossdof"):
            row["roofline_frac_432N3"] = 432.0 * n ** 3 * m / (ms * 1e-3) / 1e9 / peak
        out.append(row)
        del A, H, P, Diels
    return out


def large_grid_leg(dist, pcb, n, nev, lattice="sc_curv", typ="chiral", check=True, apply_steps=5):
    """Large-grid mode (SURVEY 8e-ii, BASELINE configs[4]) on all ranks of this job: ONE eigenproblem, dense phase row-sharded
    (slab contexts), Gram pair all-reduced with NCCL, operator on whole columns through the slab exchange.  Reports the LOBPCG
    iteration time, the exchange bandwidth over NVLink, the all-reduce latency and the agreement with a one-GPU solve."""
    import ctypes as C
    sh, mfd, ne, L = pcb.sharded, pcb.discretization, pcb.numerical_experiments, pcb._lib
    uid = [sh.new_unique_id() if dist.rank == 0 else None]
    dist.td.broadcast_object_list(uid, src=0)
    comm = sh.SlabComm(n, dist.rank, dist.world, unique_id=uid[0])
    alpha = np.array([np.pi, np.pi, np.pi])
    m = nev + round(0.6 * nev)
    sym = build_ops_for(pcb, n, lattice, alpha, None)
    Diels = getattr(mfd, typ + "_handle")(n, lattice)
    A, H, P = sh.pc_mfd_handle_sharded(comm, sym[0], sym[1], Diels, sym[2], sym[3])
    col_bytes = 48.0 * n ** 3
    x0 = comm.slab.random_block(m, 99)
    # operator applies on m columns spread over all ranks, device-timed on the slab stream.  Blocks from work_block() are mapped
    # into every rank (CUDA IPC), so this takes the peer-memory path: the x passes read / write the slabs of all ranks over NVLink.
    # The same applies through the NCCL slab exchange (blocks that are not shared) are timed next to it.
    xs, ys = comm.slab.work_block("bench.x", m), comm.slab.work_block("bench.y", m)
    xs.assign(x0)
    y0 = comm.slab.empty(m)

    def time_applies(src, dstb):
        for _ in range(2):
            H.op.apply_into(L.APPLY_H, src, dstb)
        comm.slab.sync(); comm.full.sync()
        dist.barrier()
        comm.slab.timer_start()
        for _ in range(apply_steps):
            H.op.apply_into(L.APPLY_H, src, dstb)
        return dist.max(comm.slab.timer_stop() / apply_steps)

    ms_apply = time_applies(xs, ys)
    ms_apply_exch = time_applies(x0, y0)
    # the exchange alone: slabs -> whole columns on their owners
    owners = [j % dist.world for j in range(m)]
    win, _ = comm.work_blocks((m + dist.world - 1) // dist.world)
    pin = [win.ptrs[j // dist.world] if owners[j] == dist.rank else 0 for j in range(m)]
    comm.exchange(True, owners, x0, pin)
    comm.slab.sync()
    dist.barrier()
    comm.slab.timer_start()
    for _ in range(apply_steps):
        comm.exchange(True, owners, x0, pin)
    ms_exch = dist.max(comm.slab.timer_stop() / apply_steps)
    moved = m * col_bytes * (dist.world - 1) / dist.world        # bytes that cross NVLink per exchange (all ranks together)
    ar = C.c_float()
    L.check(L.lib().pcb_comm_allreduce_timed(comm.slab.h, 2 * 96 * 96 * 2, 20, C.byref(ar)), "pcb_comm_allreduce_timed")
    del y0
    dist.barrier()
    t0 = time.perf_counter()
    lam, x, info = pcb.lobpcg.lobpcg_sep_softlock(H, P, x0, nev)
    wall = dist.max(time.perf_counter() - t0)
    out = {"N": n, "world": dist.world, "nev": nev, "m": m, "lattice": lattice, "type": typ,
           "iterations": int(info[0]) if lam is not None else -1,
           "solver_s": dist.max(float(info[1])) if lam is not None else None, "wall_s": wall,
           "ms_per_iteration": 1e3 * float(info[1]) / max(1, int(info[0])) if lam is not None else None,
           "H_apply_ms_per_block": ms_apply, "op_applies_per_sec": m / ms_apply * 1e3,
           "H_apply_path": {0: "NCCL slab exchange both ways", 1: "peer memory: both x passes read / write the slabs of all ranks over NVLink (pcb_apply_dist)",
                            2: "NCCL gather (pipelined) + scatter fused into the last FFT pass over peer memory (pcb_apply_dist)"}[comm.p2p_mode if comm.p2p else 0],
           "H_apply_ms_per_block_exchange_path": ms_apply_exch,
           "H_apply_nvlink_GBps_aggregate": 2 * m * col_bytes * (dist.world - 1) / dist.world / (ms_apply * 1e-3) / 1e9,
           "exchange_ms": ms_exch, "exchange_GBps_aggregate": moved / (ms_exch * 1e-3) / 1e9,
           "exchange_GBps_per_gpu_each_direction": moved / dist.world / (ms_exch * 1e-3) / 1e9,
           "gram_allreduce_us": 1e3 * float(ar.value), "collective": "ncclAllReduce (Gram pair, norms) + grouped ncclSend/ncclRecv (slab exchange)",
           "pipeline_chunks": sh.LG_CHUNKS}
    if check and dist.rank == 0 and lam is not None:
        A1, H1, P1 = ne.pc_mfd_handle(sym[0], sym[1], Diels, sym[2], sym[3])
        x1 = comm.full.random_block(m, 99)
        lam1, xs1, info1 = pcb.lobpcg.lobpcg_sep_softlock(H1, P1, x1, nev)
        out["single_gpu"] = {"iterations": int(info1[0]), "solver_s": float(info1[1]),
                             "max_rel_eig_diff": float(np.max(np.abs(lam[:nev] - lam1[:nev]) / np.abs(lam1[:nev])))}
        del x1, xs1
    dist.barrier()
    del x0, x
    comm.close()
    return out


def run_large_grid(args):
    """--mode large-grid: BASELINE configs[4] shape (sc_curv, N = 256, 20 bands on 8 GPUs; pass --n / --nev for smaller boxes)."""
    dist = Dist(args.gpus)
    if dist.world < 2:
        raise SystemExit("--mode large-grid needs torchrun with >= 2 ranks")
    pcb = importlib.import_module(PKG)
    pcb.set_device(dist.local)
    sampler = ClockSampler(dist.local) if dist.rank == 0 else None
    res = large_grid_leg(dist, pcb, args.n, args.nev, check=args.n <= 160, apply_steps=max(3, args.steps))
    clocks = sampler.stop() if sampler else None
    if dist.rank == 0:
        line = {"metric": "op_applies_per_sec", "value": res["op_applies_per_sec"], "unit": "op-applies/s", "n_gpus": dist.world,
                "steps": max(3, args.steps), "warmup": 2, "ms_per_step": res["H_apply_ms_per_block"], "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "mode": "large-grid",
                "config": {"workload": f"sc_curv chiral N={args.n} m={res['m']}: ONE eigenproblem over {dist.world} GPUs (configs[4] shape), "
                                       "H block apply through the slab exchange", "parallelism": f"rows of S/HS sharded x{dist.world}, NCCL all-reduce of the Gram pair"},
                "large_grid": res, "clocks": clocks}
        print(json.dumps(line), flush=True)
    dist.close()


def cpu_full_baseline(n, alpha, cores):
    """SURVEY 8(d) CPU yard-stick on the oracle port: the C1 solve (sc_curv, chiral, N = 48, 10 bands, rng(0) x0) and three LOBPCG
    iterations at N = `n` (fcc, chiral) -- minutes of host time, so only with --cpu-full."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pc_oracle as oc
    pcb = importlib.import_module(PKG)
    oc.FFT_WORKERS = cores
    out = {}
    x0 = oc.random_x0(3 * 48 ** 3, 16, 0)
    t0 = time.perf_counter()
    o = oc.eigen_1p(48, "sc_curv", np.array([np.pi, np.pi, np.pi]), type="chiral", nev=10, x0=x0)
    out["c1_solve_s"] = time.perf_counter() - t0
    out["c1_iterations"] = int(o["info"][0])
    # the same solve (same x0) on the GPU, for the record next to it
    mfd, ne = pcb.discretization, pcb.numerical_experiments
    al = np.array([np.pi, np.pi, np.pi])
    relax, pnt = mfd.set_relaxation(al)
    af, bf = mfd.fft_blocks(48, 1, pcb.dielectric.diel_info("sc_curv", option="ct"), alpha=al)
    iv = mfd.inverse_3_times_3_B(bf, pnt, relax[0])
    A1, H1, P1 = ne.pc_mfd_handle(af, (pnt * bf[0], pnt * bf[1]), mfd.chiral_handle(48, "sc_curv"), iv, relax[0])
    lam_g, _, info_g = pcb.lobpcg.lobpcg_sep_softlock(H1, P1, x0, 10)
    out["c1_gpu_solve_s"] = float(info_g[1])
    out["c1_gpu_iterations"] = int(info_g[0])
    out["c1_max_rel_eig_diff_gpu_vs_cpu"] = float(np.max(np.abs(lam_g[:10] - o["lambdas"][:10]) / np.abs(o["lambdas"][:10])))
    a_fft, b_fft, inv_fft, shift, _ = oc.assemble_symbols(n, LATTICE, alpha)
    ind_e = pcb.dielectric.compute_index(n, LATTICE, "edge")
    A, H, P = oc.pc_mfd_handle(a_fft, b_fft, oc.chiral_handle(n, LATTICE, ind_e=ind_e), inv_fft, shift)
    x0 = oc.random_x0(3 * n ** 3, 16, 1)
    t0 = time.perf_counter()
    oc.lobpcg_sep_softlock(H, P, x0, 10, maxiter=3)
    out["lobpcg_3_iterations_s"] = time.perf_counter() - t0
    out["s_per_iteration"] = out["lobpcg_3_iterations_s"] / 3
    return out


def run_reference(args):
    """--impl reference: the reference algorithm's CPU implementation (oracle port; the reference itself is Python+CuPy and
    cannot be imported on the GPU box) on this arm's config, all host threads, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    th = host_threads()
    cores = th["cores"]
    n = args.n
    pcb = importlib.import_module(PKG)
    alphas = pcb.dielectric.kpath(LATTICE)
    alpha = alphas[0]
    cols = args.cols          # the same 16-column block apply per step as the CUDA arm (same_config)
    t0 = time.perf_counter()
    rate, times = cpu_apply_rate(n, alpha, cols, args.steps, args.warmup, cores)
    ms = 1e3 * sum(times) / len(times)
    sample = (f"the full {cols}-column block per step (H apply, N={n}; oracle port of pcfft.AMA_BB, scipy.fft workers={cores}, "
              f"BLAS threads={th['blas_threads']}); the reference itself is Python + CuPy and cannot run on this box")
    line = {"impl": "reference", "metric": "op_applies_per_sec", "value": rate, "unit": "op-applies/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{LATTICE} {DTYPE_TYPE} eps=13 N={n} m={M_BLOCK} H block apply (configs[1])", "N": n,
                       "lattice": LATTICE, "type": DTYPE_TYPE, "cols_per_step": cols},
            "cpu_baseline": {"value": rate, "unit": "op-applies/s", "cores": cores, "kind": "port", "sample": sample, "threads": th},
            "e2e": {"value": rate, "unit": "op-applies/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "wall_s": time.perf_counter() - t0}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="pcb200", choices=["pcb200", "reference"])
    ap.add_argument("--n", "--grid", dest="n", type=int, default=N_GRID, help="grid size N (use --grid under torchrun, whose parser trips over --n)")
    ap.add_argument("--cols", type=int, default=M_BLOCK, help="block width m (16 for 10 bands, 32 for 20 bands)")
    ap.add_argument("--kpoints", type=int, default=3, help="k-points per rank for the LOBPCG leg (0 = skip)")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--no-blocks", action="store_true", help="skip the LOBPCG block-kernel micro-timings")
    ap.add_argument("--mode", default="kpath", choices=["kpath", "large-grid"],
                    help="kpath: the headline (one k-point per GPU, no collective); large-grid: one eigenproblem over all ranks (NCCL)")
    ap.add_argument("--nev", type=int, default=NEV, help="bands (large-grid mode)")
    ap.add_argument("--no-paper2", action="store_true", help="skip the Paper-2 dielectric legs")
    ap.add_argument("--no-large-grid", action="store_true", help="N > 1: skip the large-grid (NCCL) leg")
    ap.add_argument("--cpu-full", action="store_true", help="CPU baseline per SURVEY 8(d): also the C1 solve (N=48) and 3 LOBPCG iterations at N=120 on the host")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the output of the last timed step (seeded row sample + column norms, float64 .npy) to DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.mode == "large-grid"):
        ap.error("--dump-outputs applies to the CUDA k-path benchmark only")
    if args.impl == "reference":
        return run_reference(args)
    if args.mode == "large-grid":
        return run_large_grid(args)
    args.warmup = max(args.warmup, 3)

    dist = Dist(args.gpus)
    pcb = importlib.import_module(PKG)
    pcb.set_device(dist.local)
    if pcb.backend() != "cuda-sm_100a":
        raise SystemExit("bench.py requires the CUDA build of libpcb200.so")
    n, m = args.n, args.cols
    ne, mfd = pcb.numerical_experiments, pcb.discretization
    ctx = pcb.get_context(n)
    alphas, chunk = fcc_alpha(pcb, dist.rank, dist.world)
    Diels = mfd.chiral_handle(n, LATTICE)
    (A, H, P), shift = build_ops(pcb, n, alphas[chunk[0]], Diels)
    op = H.op
    X, Y = ctx.random_block(m, 1234 + dist.rank), ctx.empty(m)
    ctx.sync()

    # ---- device-resident block applies ---------------------------------------------------------------------
    sampler = ClockSampler(dist.local) if dist.rank == 0 else None
    for _ in range(args.warmup):
        op.apply_into(pcb._lib.APPLY_H, X, Y)
    ctx.sync()
    dist.barrier()
    l0 = ctx.launches()
    ctx.timer_start()
    for _ in range(args.steps):
        op.apply_into(pcb._lib.APPLY_H, X, Y)
    ms_total = ctx.timer_stop()
    launches = ctx.launches() - l0
    dist.barrier()
    ms_total = dist.max(ms_total)
    if args.dump_outputs and dist.rank == 0:
        dump_outputs(args.dump_outputs, Y)
    if sampler:      # keep the identical load running so that nvidia-smi (50 ms period) gets enough samples of this workload
        t_end = time.perf_counter() + 0.6
        while time.perf_counter() < t_end:
            for _ in range(20):
                op.apply_into(pcb._lib.APPLY_H, X, Y)
            ctx.sync()
    clocks = sampler.stop() if sampler else None
    ms_step = ms_total / args.steps
    value = dist.world * m * args.steps / (ms_total * 1e-3)

    # ---- per-pass device times -------------------------------------------------------------------------------
    pass_ms = np.array(timed_passes(pcb, op, X, Y, m, 5))

    class _NP:
        value = len(pass_ms)
    npass = _NP()
    col_bytes = 48.0 * n ** 3            # one column, one direction
    if npass.value == 3:                  # plane mode: x forward (transposed store), fused y/z/M/z/y plane pass, x inverse
        pass_cols, names = [2, 2, 3], ["x_fwd+KAh -> W'", "y,z fwd + M + z,y inv on (i1,i2) planes", "x_inv+KA+gKB+shift"]
        kernel_desc = "op-apply = 3 passes (k_xfwd<T>, k_mid2 [five-sweep plane pass; k_mid where N != 8 x odd], k_xinv<T>)"
    else:
        pass_cols, names = [2, 2, 2, 2, 3], ["x_fwd+KAh", "y_fwd", "z_fwd+M+z_inv", "y_inv", "x_inv+KA+gKB+shift"]
        kernel_desc = "op-apply = 5 passes (k_xfwd, k_line, k_zmid, k_line, k_xinv)"
    pass_bytes = np.array(pass_cols) * col_bytes * m
    passes = [{"name": nm, "ms": float(t), "GBps": float(b / (t * 1e-3) / 1e9)} for nm, t, b in zip(names, pass_ms, pass_bytes)]

    peak, peak_src = measured_peak()
    achieved = B_OP_PER_N3 * n ** 3 * m / (ms_step * 1e-3) / 1e9 * 1.0     # per rank: every rank runs the same step
    # DRAM bytes of one launch (= one 16-column block apply) from ncu --set full captures of exactly these kernels and this
    # shape (dram__bytes_read.sum + dram__bytes_write.sum summed over the passes): plane mode profiles/r01_f_final_ncu.md
    # (5.487 GB read + 3.864 GB written), five-pass profiles/r01_c_final_ncu.md; null for other shapes
    traffic, traffic_src = ncu_traffic(n, m, npass.value)
    roofline = {"bound": "hbm", "kernel": kernel_desc,
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": traffic_src,
                "peak_source": peak_src, "algorithmic_bytes_per_launch": B_OP_PER_N3 * n ** 3 * m,
                "moved_bytes_per_launch": float(pass_bytes.sum()), "moved_GBps": float(pass_bytes.sum() / (ms_step * 1e-3) / 1e9)}

    # ---- LOBPCG block kernels on the same shapes (m = 16 active columns, n_loc = 48) --------------------------------
    blocks = []
    if not args.no_blocks:
        L = pcb._lib
        S, HS = ctx.random_block(3 * m, 77), ctx.random_block(3 * m, 78)
        lam = np.linspace(1.0, 2.0, m)
        Rb = 16.0 * ctx.R        # bytes of one column

        def timed(fn, reps=10):
            fn(); ctx.sync(); ctx.timer_start()
            for _ in range(reps):
                fn()
            return ctx.timer_stop() / reps

        t = timed(lambda: op.residual(S[:, :m], HS[:, :m], S[:, m:2 * m], lam, precond=True))
        blocks.append({"name": f"residual+norms+precond (m={m})", "ms": t, "GBps": 3 * m * Rb / t / 1e6})
        G = np.empty((3 * m, 3 * m), dtype=np.complex128); T = np.empty_like(G)
        t = timed(lambda: L.check(L.lib().pcb_gram2(ctx.h, 3 * m, L.ptr_array(S.ptrs), L.ptr_array(HS.ptrs), G.ctypes.data, T.ctypes.data), "gram2"))
        nl = 3 * m
        blocks.append({"name": f"gram pair (n_loc={3 * m})", "ms": t, "GBps": 2 * nl * Rb / t / 1e6,
                       "GFLOPs": 8.0 * ctx.R * nl * (nl + 1) / t / 1e6})
        t = timed(lambda: L.check(L.lib().pcb_gram2_top(ctx.h, nl, m, L.ptr_array(S.ptrs), L.ptr_array(HS.ptrs), G.ctypes.data, T.ctypes.data), "gram2_top"))
        blocks.append({"name": f"gram pair, rows of W only (n_loc={nl}, n_act={m}; 7 of 8 iterations)", "ms": t,
                       "GBps": (nl + m) * Rb / t / 1e6, "GFLOPs": 16.0 * ctx.R * m * nl / t / 1e6})
        E = np.ascontiguousarray(np.random.default_rng(0).standard_normal((nl, m)) + 0j) / nl
        t = timed(lambda: L.check(L.lib().pcb_update(ctx.h, m, nl, L.ptr_array(S.ptrs), L.ptr_array(HS.ptrs), L.ptr_array(S[:, 2 * m:].ptrs),
                                                     L.ptr_array(HS[:, 2 * m:].ptrs), E.ctypes.data), "update"))
        blocks.append({"name": f"fused update (m={m}, n_loc={3 * m})", "ms": t, "GBps": (2 * nl + 4 * m) * Rb / t / 1e6,
                       "GFLOPs": 16.0 * ctx.R * m * nl / t / 1e6})
        t = timed(lambda: op.update_resid(m, nl, S, HS, S[:, 2 * m:], HS[:, 2 * m:], E, lam, S[:, m:2 * m]))
        blocks.append({"name": f"fused update + next residual/norms/precond (m={m}, n_loc={3 * m}; replaces the two kernels above it and the residual)",
                       "ms": t, "GBps": (2 * nl + 5 * m) * Rb / t / 1e6, "GFLOPs": 16.0 * ctx.R * m * nl / t / 1e6})
        t = timed(lambda: op.apply_into(L.APPLY_H, S[:, :m], HS[:, :m]))
        blocks.append({"name": f"H apply ({m} columns)", "ms": t, "GBps": B_OP_PER_N3 * n ** 3 * m / t / 1e6})
        del S, HS

    # ---- end to end: host (pinned) buffers through the reference-facing callable ---------------------------------
    xh, yh = pcb.pinned_empty((ctx.R, m)), pcb.pinned_empty((ctx.R, m))
    X.get(out=xh)
    for _ in range(2):
        H(xh, out=yh)
    ctx.sync()
    dist.barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        H(xh, out=yh)
    ctx.sync()
    e2e_s = dist.max(time.perf_counter() - t0)
    e2e = {"value": dist.world * m * args.e2e_steps / e2e_s, "unit": "op-applies/s", "h2d_bytes_per_step": int(xh.nbytes),
           "d2h_bytes_per_step": int(yh.nbytes), "ms_per_step": 1e3 * e2e_s / args.e2e_steps, "steps": args.e2e_steps,
           "api": "H_func(x_host, out=y_host) from numerical_experiments.pc_mfd_handle"}
    pcb.devarray.pinned_free(xh)
    pcb.devarray.pinned_free(yh)
    del X, Y

    # ---- LOBPCG: seconds to 10 bands for this rank's k-points (warm-started chain, as bandgap()) -----------------
    lob = None
    if args.kpoints > 0:
        secs, iters, x = [], [], None
        for j, idx in enumerate(chunk[:args.kpoints]):
            (A, H, P), shift = build_ops(pcb, n, alphas[idx], Diels)
            x0 = ctx.random_block(m, 1000 + idx) if x is None else x
            lam, x, info = pcb.lobpcg.lobpcg_sep_softlock(H, P, x0, NEV, tol=1e-4)
            if lam is None:
                secs.append(float("nan")); iters.append(-1); x = None
                continue
            secs.append(float(info[1])); iters.append(int(info[0]))
        allr = dist.gather({"rank": dist.rank, "k_indices": [int(i) for i in chunk[:args.kpoints]], "sec": secs, "iters": iters})
        if dist.rank == 0:
            flat_s = [s for r in allr for s in r["sec"]]
            flat_i = [i for r in allr for i in r["iters"]]
            lob = {"sec_to_10_bands_mean": float(np.mean(flat_s)), "sec_to_10_bands": flat_s, "iterations": flat_i,
                   "ms_per_iteration": float(1e3 * np.sum(flat_s) / max(1, np.sum(flat_i))), "tol": 1e-4,
                   "k_indices": [r["k_indices"] for r in allr], "first_of_chunk": "random start (seed 1000+idx), rest warm-started"}

    # ---- CPU baseline (rank 0, N=1 only) --------------------------------------------------------------------------
    # ---- Paper-2 dielectrics (extra keys) and, for N > 1, the large-grid mode with its NCCL collectives ----------------
    paper2 = None
    if not args.no_paper2 and n == N_GRID:
        paper2 = paper2_dielectric_leg(pcb, ctx, n, m, max(5, min(args.steps, 20)), 3, peak)
    larger = None
    if not args.no_paper2 and n == N_GRID and dist.world == 1:
        larger = larger_grid_leg(pcb, m, 5, 2, peak)
    large = None
    if dist.world > 1 and not args.no_large_grid:
        large = large_grid_leg(dist, pcb, n, NEV, check=True)

    cpu = None
    if dist.rank == 0 and dist.world == 1 and not args.no_cpu:
        th = host_threads()
        cores = th["cores"]
        cols = 2
        rate, times = cpu_apply_rate(n, alphas[chunk[0]], cols, 3, 1, cores)
        cpu = {"value": rate, "unit": "op-applies/s", "cores": cores, "kind": "port", "threads": th,
               "sample": f"{cols} of the {m} columns of one step, 3 timed reps after 1 warm-up (oracle AMA_BB, scipy.fft workers={cores})"}
        if args.cpu_full:
            cpu["survey_8d"] = cpu_full_baseline(n, alphas[chunk[0]], cores)

    if dist.rank == 0:
        line = {"metric": "op_applies_per_sec", "value": value, "unit": "op-applies/s", "n_gpus": dist.world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": f"{LATTICE} {DTYPE_TYPE} eps=13 N={n} m={m} H block apply (configs[1]); one k-point of the FCC path per GPU",
                           "N": n, "lattice": LATTICE, "type": DTYPE_TYPE, "cols_per_step": m, "l2": "inputs exceed L2 (1.33 GB per block)",
                           "parallelism": f"k-path sharding x{dist.world}, no collective"},
                "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
                "passes": passes, "block_kernels": blocks, "lobpcg": lob, "paper2_dielectrics": paper2, "larger_grids": larger, "large_grid": large}
        print(json.dumps(line), flush=True)
    dist.close()


if __name__ == "__main__":
    main()
