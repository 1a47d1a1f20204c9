"""Lattice geometry on the host: k-path data, DoF meshes and the index sets of Omega_1.

Mirrors the public surface of paper_2/dielectric.py (diel_info :20-35, diel_alpha :37-49,
diel_io_index :58-97, mesh3d_*_dofs :104-130, FLAG_* :157-261).  Runs once per lattice in NumPy
(SURVEY.md 2.2: host set-up, < 1 s at N = 120 once cached); the GPU only ever sees the resulting
int64 index lists, which the C ABI packs into a per-cell bit mask.  The ``.bin`` wire format
(raw little-endian int64) and directory layout are the reference's.
"""
import os
import tempfile
import time

import numpy as np
from numpy import pi

from .environment import (CHIRAL_EPS_EG, DIEL_LIB, DIEL_PATH, GAP, GREEN, PSEUDOCHIRAL_EPS_LOC, RED, RESET, say)


def diel_info(d_flag, option=None):
    """Coordinate transform `ct`, symmetry points `sym`, or both (dielectric.py:20-35)."""
    name = d_flag.split("_")[0]
    ct = np.array(DIEL_LIB["CT_" + name])
    sym = np.array(DIEL_LIB["sym_" + name])
    if option == "ct":
        return ct
    if option == "sym":
        return sym
    return ct, sym


def diel_alpha(d_flag, no, gap=GAP):
    """Translation vector number `no` of the path (dielectric.py:37-49)."""
    sym = np.array(DIEL_LIB["sym_" + d_flag.split("_")[0]])
    seg, pos = divmod(no, gap)
    if pos == 0:
        return sym[seg, :]
    return (pos * sym[seg + 1, :] + (gap - pos) * sym[seg, :]) / gap


def kpath(d_flag, gap=GAP):
    """All translation vectors of the band path, in the order of bandgap()
    (numerical_experiments.py:342-346): `gap` points per segment, end point included."""
    sym = diel_info(d_flag, "sym").astype(float)
    nseg = sym.shape[0] - 1
    alphas = np.zeros((nseg * gap, 3))
    for s in range(nseg):
        alphas[(s + 1) * gap - 1, :] = sym[s + 1, :]
        for j in range(gap - 1):
            alphas[s * gap + j, :] = ((j + 1) * sym[s + 1, :] + (gap - j - 1) * sym[s, :]) / gap
    return alphas


def diel_chiral_const(d_flag="sc_curv"):
    return CHIRAL_EPS_EG[d_flag]


def diel_pseudochiral_const(no=0):
    return PSEUDOCHIRAL_EPS_LOC[no]


# ---------------------------------------------------------------------------------------------
# DoF meshes (dielectric.py:104-130): row r = c*N^3 + i0 + N*i1 + N^2*i2
# ---------------------------------------------------------------------------------------------
def _grid(N):
    ax = np.arange(N)
    return np.tile(ax, N * N), np.tile(np.repeat(ax, N), N), np.repeat(ax, N * N)


def mesh3d_edge_dofs(N):
    """(3 N^3, 3) coordinates of the edge DoFs: component c sits half a cell along axis c."""
    i0, i1, i2 = _grid(N)
    blocks = []
    for c in range(3):
        cols = [i0 / N, i1 / N, i2 / N]
        cols[c] = ((i0, i1, i2)[c] + 0.5) / N
        blocks.append(np.column_stack(cols))
    return np.vstack(blocks)


def mesh3d_volume_dofs(N):
    """(N^3, 3) coordinates of the cell centres."""
    i0, i1, i2 = _grid(N)
    return np.column_stack(((i0 + 0.5) / N, (i1 + 0.5) / N, (i2 + 0.5) / N))


# ---------------------------------------------------------------------------------------------
# Flag functions (dielectric.py:157-261): indices of the points inside the dielectric
# ---------------------------------------------------------------------------------------------
def FLAG_sc_flat1(coo):
    x, y, z = coo[:, 0], coo[:, 1], coo[:, 2]
    q = 0.25
    return np.where((x <= q) & (y <= q) | (x <= q) & (z <= q) | (y <= q) & (z <= q))[0]


def FLAG_sc_flat2(coo):
    x, y, z = coo[:, 0], coo[:, 1], coo[:, 2]
    return np.where((x <= 0.25) & (y <= 0.25)
                    | (x <= 0.25) & (z >= 0.25) & (z <= 0.5)
                    | (y >= 0.5) & (y <= 0.75) & (z >= 0.5) & (z <= 0.75)
                    | (x >= 0.5) & (x <= 0.75) & (z >= 0.75))[0]


def FLAG_sc_curv(coo_in):
    """Sphere of radius 0.345 joined by three axis-parallel rods of radius 0.11 (cell centre)."""
    rod, ball = 0.11, 0.345
    p = coo_in - 0.5
    xx, yy, zz = p[:, 0] ** 2, p[:, 1] ** 2, p[:, 2] ** 2
    return np.where((xx + yy + zz <= ball ** 2) | (xx + yy <= rod ** 2) | (xx + zz <= rod ** 2) | (yy + zz <= rod ** 2))[0]


def FLAG_bcc_gyroid(coo, double_flag=False):
    r = coo.T
    g = np.sin(2 * pi * r[0]) * np.cos(2 * pi * r[1]) + np.sin(2 * pi * r[1]) * np.cos(2 * pi * r[2]) + \
        np.sin(2 * pi * r[2]) * np.cos(2 * pi * r[0])
    return np.where((np.abs(g) if double_flag else g) > 1.1)[0]


def FLAG_bcc_sg(coo):
    return FLAG_bcc_gyroid(coo, double_flag=False)


def FLAG_bcc_dg(coo):
    return FLAG_bcc_gyroid(coo, double_flag=True)


def FLAG_fcc(coo_in, chunk=1 << 16):
    """Diamond network: 18 spheres (r = 0.12) at the lattice sites plus 16 prolate spheroids
    (semi-minor axis 0.11) along the four bonds leaving each of the four basis sites."""
    r_sph, b_ell = 0.12, 0.11
    pts = np.array(coo_in, dtype=float)
    if pts.ndim == 1:
        pts = pts.reshape(3, 1)
    elif pts.shape[0] != 3:
        pts = pts.T
    basis = np.array([[0, 0, 0.5, 0.5], [0, 0.5, 0, 0.5], [0, 0.5, 0.5, 0]], dtype=float)
    quarter = np.ones(3) * 0.25
    sites = np.hstack((np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [0, 1, 1], [1, 0, 1], [1, 1, 0],
                                 [1, 1, 1], [0, 0.5, 0.5], [0.5, 0, 0.5], [0.5, 0.5, 0], [1, 0.5, 0.5],
                                 [0.5, 1, 0.5], [0.5, 0.5, 1]], dtype=float).T, quarter[:, None] + basis))
    bonds = []
    for i in range(4):
        mid = (basis[:, i] + quarter) / 2
        half = (basis[:, i] - quarter) / 2
        length = np.linalg.norm(half)
        bonds.append((mid, length, half / length))
    inside = np.zeros(pts.shape[1], dtype=bool)

    def one_chunk(s):
        x = pts[:, s:s + chunk]
        hit = np.any(np.sum((x[:, :, None] - sites[:, None, :]) ** 2, axis=0) < r_sph * r_sph, axis=1)
        for mid, length, direction in bonds:
            X = x[:, None, :] - (mid[:, None] + basis)[:, :, None]
            major = np.hypot(b_ell, length)
            along = np.tensordot(direction, X, axes=([0], [0])) ** 2
            across = np.sum(X ** 2, axis=0) - along
            hit |= np.any((along / major ** 2) + (across / b_ell ** 2) < 1, axis=0)
        inside[s:s + chunk] = hit

    # the chunks are independent and NumPy releases the GIL inside its loops: a few host threads cut the one-off set-up of an
    # N = 120 band-structure run from ~7 s to ~1 s without touching the arithmetic (the index sets stay bit-identical)
    starts = list(range(0, pts.shape[1], chunk))
    workers = min(8, os.cpu_count() or 1, len(starts))
    if workers > 1:
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(workers) as pool:
            list(pool.map(one_chunk, starts))
    else:
        for s in starts:
            one_chunk(s)
    return np.where(inside)[0]


_FLAGS = {"sc_flat1": FLAG_sc_flat1, "sc_flat2": FLAG_sc_flat2, "sc_curv": FLAG_sc_curv,
          "bcc_sg": FLAG_bcc_sg, "bcc_dg": FLAG_bcc_dg, "fcc": FLAG_fcc}


_index_cache = {}     # (N, d_flag, dofs) -> int64 indices (in-process complement of the on-disk .bin cache)
_geom_digest = []


def _geometry_digest():
    """Short digest of this module's source (the FLAG_* / mesh definitions): versions the private on-disk index cache."""
    if not _geom_digest:
        import hashlib
        with open(__file__, "rb") as f:
            _geom_digest.append(hashlib.sha256(f.read()).hexdigest()[:12])
    return _geom_digest[0]


def _cache_dir_is_private(root):
    """True when the cache root belongs to this user and nobody else may write to it."""
    try:
        st = os.stat(root)
    except OSError:
        return False
    return st.st_uid == os.getuid() and (st.st_mode & 0o022) == 0


def compute_index(N, d_flag, dofs="edge"):
    """Index set of Omega_1 computed from the geometry (the compute branch of diel_io_index)."""
    ct = diel_info(d_flag, option="ct")
    mesh = mesh3d_edge_dofs(N) if dofs == "edge" else mesh3d_volume_dofs(N)
    return np.asarray(_FLAGS[d_flag](mesh @ np.linalg.inv(ct.T)), dtype=np.int64)


_GEOM_KIND = {"sc_flat1": 0, "sc_flat2": 1, "sc_curv": 2, "bcc_sg": 3, "bcc_dg": 4, "fcc": 5}
geometry_stats = {}      # last device evaluation: {"seconds", "ambiguous"} (set-up timing for the runners / bench)


def device_index_sets(N, d_flag, ctx=None):
    """(edge indices, volume indices) of Omega_1 with the O(N^3) classification on the GPU (pcb_geometry_mask).

    The kernel evaluates FLAG_<d_flag> for the 3 N^3 edge and N^3 volume DoF points and reports every point whose deciding
    inequality has a margin below 1e-10 (exact ties of the flat lattices, last-bit differences to NumPy's arithmetic); only
    those are re-evaluated here with the NumPy expression of compute_index, so the result is bit-identical to it
    (tests: every lattice at N = 12 ... 48, FCC / gyroid at N = 120) at a fraction of a second instead of 5-8 s at N = 120."""
    from . import _lib as L
    from . import devarray
    t0 = time.time()
    ctx = ctx if ctx is not None else devarray.get_context(N)
    nn = N ** 3
    minv = np.ascontiguousarray(np.linalg.inv(diel_info(d_flag, option="ct").T), dtype=np.float64)
    mask, amb = np.empty(nn, dtype=np.uint8), np.empty(nn, dtype=np.uint8)
    L.check(L.lib().pcb_geometry_mask(ctx.h, _GEOM_KIND[d_flag], minv.ctypes.data_as(L.c_double_p), mask.ctypes.data, amb.ctypes.data),
            "pcb_geometry_mask")
    n_amb = 0
    for d in range(4):
        cells = np.flatnonzero((amb >> d) & 1)
        if cells.size == 0:
            continue
        n_amb += cells.size
        i = [cells % N, (cells // N) % N, cells // (N * N)]
        cols = [(i[ax] + 0.5) / N if (d == 3 or d == ax) else i[ax] / N for ax in range(3)]
        pts = np.column_stack(cols)
        if pts.shape[0] == 3:          # FLAG_fcc reads a (3, 3) array as (axis, point): avoid the ambiguous shape
            pts = np.vstack((pts, pts[:1]))
        hit = np.zeros(pts.shape[0], dtype=bool)
        hit[_FLAGS[d_flag](pts @ minv)] = True
        inside = hit[:cells.size]
        bit = np.uint8(1 << d)
        mask[cells] = np.where(inside, mask[cells] | bit, mask[cells] & np.uint8(~bit & 0xFF))
    ind_e = np.concatenate([c * nn + np.flatnonzero((mask >> c) & 1) for c in range(3)]).astype(np.int64)
    ind_v = np.flatnonzero((mask >> 3) & 1).astype(np.int64)
    geometry_stats.update(seconds=time.time() - t0, ambiguous=int(n_amb), N=N, d_flag=d_flag)
    return ind_e, ind_v


def material_regions(N, d_flag):
    """Edge-DoF index sets of the materials of a lattice (discretization.materials_handle): for bcc_dg its two gyroid networks,
    g > 1.1 (= bcc_sg) and g < -1.1 -- the inversion r -> -r swaps them --, for every other lattice the one set Omega_1."""
    ind = diel_io_index(N, d_flag, dofs="edge")
    if d_flag != "bcc_dg":
        return [ind]
    sg = diel_io_index(N, "bcc_sg", dofs="edge")
    return [sg, np.setdiff1d(ind, sg, assume_unique=True)]


def diel_io_index(N, d_flag, dofs="edge", gpu=True, cache=True):
    """Indices of the dielectric edge / volume DoFs (dielectric.py:58-97).

    Loads ``DIEL_PATH/<dofs>_dofs/<d_flag>_<N>.bin`` (raw int64) when present, otherwise computes
    the set from the geometry and -- like the reference -- stores it there if the directory exists.
    Always returns a host int64 array (`gpu` is accepted for signature compatibility: the device
    representation is a bit mask owned by the dielectric handle)."""
    if d_flag is None:
        rng = np.random.default_rng()
        return rng.integers(0, 3 * N ** 3 - 1, size=int(0.372 * 3 * N ** 3)).astype(np.int64)
    t0 = time.time()
    path = os.path.join(DIEL_PATH, dofs + "_dofs", f"{d_flag}_{N}.bin")
    if not os.path.isdir(os.path.dirname(path)):
        # no reference-style directory in the working directory: keep the same raw-int64 files in a per-user cache so that
        # the geometry (seconds of NumPy at N = 120, per process) is evaluated once per machine, not once per run and rank
        # (directory private to the user, file name keyed by a digest of this module's geometry code: a stale file from an
        # older FLAG_* definition or one planted by another user is never picked up)
        root = os.environ.get("PCB200_CACHE", os.path.join(tempfile.gettempdir(), f"pcb200_index_cache_{os.getuid()}"))
        path = os.path.join(root, dofs + "_dofs", f"{d_flag}_{N}_{_geometry_digest()}.bin")
        private = True
    else:
        private = False
    ind = None
    if (N, d_flag, dofs) in _index_cache:
        ind = _index_cache[(N, d_flag, dofs)]
    elif os.path.exists(path) and (not private or _cache_dir_is_private(os.path.dirname(os.path.dirname(path)))):
        ind = np.fromfile(path, dtype=np.int64)
        limit = 3 * N ** 3 if dofs == "edge" else N ** 3
        if ind.size == 0 or ind.size > limit or ind.min() < 0 or ind.max() >= limit or np.any(np.diff(ind) <= 0):
            ind = None            # truncated / foreign file: recompute
        else:
            say(f"{GREEN}Index file already exists.{RESET}")
    if ind is None:
        if gpu and d_flag in _GEOM_KIND and os.environ.get("PCB200_HOST_GEOMETRY", "0") != "1":
            # geometry on the device: both index sets come out of one kernel launch (the other one is kept for the next call)
            ind_e, ind_v = device_index_sets(N, d_flag)
            _index_cache[(N, d_flag, "edge")], _index_cache[(N, d_flag, "volume")] = ind_e, ind_v
            ind = ind_e if dofs == "edge" else ind_v
        else:
            ind = compute_index(N, d_flag, dofs)
        if cache:
            say(f"{RED}New lattice type {d_flag} or size {N} isn't computed.{RESET}")
            try:
                os.makedirs(os.path.dirname(path), mode=0o700, exist_ok=True)
                tmp = f"{path}.{os.getpid()}.tmp"
                ind.tofile(tmp)
                os.replace(tmp, path)          # atomic: concurrent ranks may race for the same file
            except OSError:
                pass
    _index_cache[(N, d_flag, dofs)] = ind
    say(f"Dielectric {dofs} indices for {d_flag} with N = {N} loaded, {time.time() - t0:<6.3f}s elapsed.")
    return ind
