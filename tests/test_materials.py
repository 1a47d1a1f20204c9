"""Dielectrics of several isotropic materials: pcb_diel_create_materials, DielHandle.materials, materials_handle and the runners.

Each edge DoF r carries a material index mat[r]; M is diagonal with (M x)_r = inv_eps[mat[r]] x_r (index 0: the background).  The
oracle restates that M on the host (x * inv_eps[mat]) inside the NumPy operator of oracle/pc_oracle.py.  The ``emu`` tests run at
small N on the host-emulation build (whole planes at N = 8, 16, 24, half planes at 16, natural layout at 6 and 12); the ``gpu``
tests run the sizes users run on the B200.
"""
import json
import os

import numpy as np
import pytest

from test_field_energy import _GENERIC, _check_widths, _same, emu, field_energy, gpu  # noqa: F401
from test_group_velocity import _mode, efourier, velocity_matrices

_OPTIONS = {"plane": 1, "plane_split": 0, "mid_five": -1}


def oracle_materials(mat, inv_eps):
    """Oracle M: x * inv_eps[mat] row by row."""
    d = np.asarray(inv_eps)[np.asarray(mat)]
    return lambda x: x * (d if x.ndim == 1 else d[:, None])


def random_map(N, n_mat, seed, background=2.0):
    rng = np.random.default_rng(seed)
    mat = rng.integers(0, n_mat, size=3 * N ** 3).astype(np.uint8)
    inv_eps = 1.0 / rng.uniform(1.5, 16.0, size=n_mat)
    inv_eps[0] = 1.0 / background
    return mat, inv_eps


def _with_options(pkg, N, options, fn):
    ctx = pkg.get_context(N)
    try:
        for k, v in options.items():
            ctx.option(k, v)
        return fn(ctx)
    finally:
        for k in options:
            ctx.option(k, _OPTIONS[k])


def _ops(pkg, N, d_flag, Diels, alpha=_GENERIC):
    """(A_func, H_func) of the device operator for a dielectric handle (None: vacuum)."""
    mfd, ne = pkg.discretization, pkg.numerical_experiments
    alpha = np.asarray(alpha, dtype=float)
    relax, pnt = mfd.set_relaxation(alpha)
    a_fft, b_fft = mfd.fft_blocks(N, 1, pkg.dielectric.diel_info(d_flag, option="ct"), alpha=alpha)
    inv_fft = mfd.inverse_3_times_3_B(b_fft, pnt, relax[0])
    return ne.pc_mfd_handle(a_fft, (pnt * b_fft[0], pnt * b_fft[1]), Diels, inv_fft, relax[0])[:2]


def _colerr(got, want):
    return np.linalg.norm(got - want, axis=0) / np.linalg.norm(want, axis=0)


# ---- 1, 5: operator, fields, energy and velocity against the oracle --------------------------------------------------------
def _check_case(pkg, oc, case, width=16):
    N, d_flag, n_mat, options = case

    def run(ctx):
        L = pkg._lib
        mat, inv_eps = random_map(N, n_mat, 100 + N + n_mat)
        Diels = pkg.discretization.DielHandle.materials(N, mat, inv_eps)
        A_func, H_func = _ops(pkg, N, d_flag, Diels)
        op = A_func.op
        diel = oracle_materials(mat, inv_eps)
        a, b, inv, shift, _ = oc.assemble_symbols(N, d_flag, np.asarray(_GENERIC))
        X = ctx.random_block(width, 31 + N)
        chk = [0, width - 1] if width > 1 else [0]
        x = X.get()[:, chk]
        # A, H against the oracle; every column of the wide call equals the column applied alone and within a 3-column call
        for fn, want in ((A_func, oc.AMA(x, a, diel)), (H_func, oc.AMA_BB(x, a, b, diel, shift))):
            Y = fn(X)
            assert np.all(_colerr(Y.get()[:, chk], want) < 1e-12)
            for sel in ([0], [width - 1], list(range(min(3, width)))):
                assert _same(pkg, Y.cols(sel), fn(X.cols(sel))).all(), sel
        # M, D / E fields and E^ against the oracle; M in place equals M out of place
        xs = X.cols(chk)
        assert np.all(_colerr(Diels(xs).get(), diel(x)) < 1e-12)
        D, E, w_in, w_tot = field_energy(x, a, diel, np.flatnonzero(mat))
        for mode, want in ((L.APPLY_DFIELD, D), (L.APPLY_EFIELD, E), (L.APPLY_EFOURIER, efourier(x, a, diel))):
            assert np.all(_colerr(op.apply(mode, xs).get(), want) < 1e-12), mode
        Z = xs.copy()
        assert L.lib().pcb_apply(op.h, L.APPLY_M, Z.k, L.ptr_array(Z.ptrs), L.ptr_array(Z.ptrs)) == 0
        assert _same(pkg, Diels(xs), Z).all()
        # energy: e_in over the rows outside the background, the same bits at any width
        e_in, e_tot = op.field_energy(xs)
        assert np.all(np.abs(e_tot - w_tot) < 1e-11 * np.abs(w_tot)), (e_tot, w_tot)
        assert np.all(np.abs(e_in - w_in) < 1e-11 * np.abs(w_tot)), (e_in, w_in)
        _check_widths(pkg, op, ctx, k=max(9, width + 1))
        # velocity matrices through the A passes of this kind (tolerance as in test_group_velocity)
        V, xx, xax = op.band_velocity(xs)
        Vo, Bo = velocity_matrices(x, op.apply(L.APPLY_EFOURIER, xs).get(), op.a_fft.dtables, N)
        for d in range(3):
            err = np.abs(V[d] - Vo[d])
            assert np.all(err <= np.maximum(1e-12 * np.abs(Vo[d]).max(), 1e-14 * Bo[d])), (d, err.max())

    _with_options(pkg, N, options, run)


def _case_id(c):
    return f"N{c[0]}-{c[1]}-mat{c[2]}" + "".join(f"-{k}{v}" for k, v in c[3].items())


EMU_CASES = [(N, "bcc_dg", n_mat, opt) for N, opt in [(8, {}), (16, {}), (24, {}), (16, {"plane_split": 1}), (6, {}), (12, {})]
             for n_mat in (2, 8, 256)]
GPU_CASES = [
    (96, "fcc", 8, {}),                          # whole planes
    (120, "fcc", 256, {}),
    (120, "bcc_dg", 2, {}),
    (128, "sc_curv", 8, {}),                     # z-split half planes
    (144, "bcc_dg", 2, {}),
    (160, "fcc", 256, {}),
    (100, "bcc_dg", 8, {}),                      # five-pass operator
    (150, "sc_curv", 256, {}),
    (120, "fcc", 8, {"plane": 0}),
]


@pytest.mark.parametrize("case", EMU_CASES, ids=_case_id)
def test_operator_vs_oracle_emu(emu, oracle, case):
    _check_case(emu, oracle, case, width=5)


@pytest.mark.gpu
@pytest.mark.parametrize("case", GPU_CASES, ids=_case_id)
def test_operator_vs_oracle(gpu, oracle, case):
    _check_case(gpu, oracle, case)


@pytest.mark.gpu
def test_operator_vs_oracle_n256(gpu, oracle):
    _check_case(gpu, oracle, (256, "sc_curv", 8, {}), width=3)


# ---- 2: the chiral M as a materials map ------------------------------------------------------------------------------------
def _chiral_equal(pkg, N, d_flag, options, exact=True):
    def run(ctx):
        mfd = pkg.discretization
        X = ctx.random_block(3, 5)
        ch = _ops(pkg, N, d_flag, mfd.chiral_handle(N, d_flag))
        ma = _ops(pkg, N, d_flag, mfd.materials_handle(N, d_flag))
        for f_ch, f_ma in zip(ch, ma):
            if exact:
                assert _same(pkg, f_ch(X), f_ma(X)).all()
            else:
                assert np.all(_colerr(f_ma(X).get(), f_ch(X).get()) < 1e-13)

    _with_options(pkg, N, options, run)


_SAME_STRUCTURE = [{"mid_five": 0}, {"plane_split": 1}, {"plane": 0}]


@pytest.mark.parametrize("d_flag", ["fcc", "sc_curv", "bcc_dg"])
@pytest.mark.parametrize("N,options", [(24, _SAME_STRUCTURE[0]), (16, _SAME_STRUCTURE[1]), (16, _SAME_STRUCTURE[2]), (12, {})])
def test_chiral_as_materials_emu(emu, N, d_flag, options):
    _chiral_equal(emu, N, d_flag, options)


@pytest.mark.gpu
@pytest.mark.parametrize("d_flag", ["fcc", "sc_curv", "bcc_dg"])
@pytest.mark.parametrize("N,options", [(120, _SAME_STRUCTURE[0]), (160, {}), (120, _SAME_STRUCTURE[2]), (150, {})])
def test_chiral_as_materials(gpu, N, d_flag, options):
    _chiral_equal(gpu, N, d_flag, options)


@pytest.mark.gpu
def test_chiral_as_materials_default_n120(gpu):
    _chiral_equal(gpu, 120, "fcc", {}, exact=False)      # chiral runs the five-sweep k_mid2 here, materials the seven-sweep k_mid


def test_material_regions(emu):
    dl = emu.dielectric
    sg, dg = dl.diel_io_index(12, "bcc_sg"), dl.diel_io_index(12, "bcc_dg")
    r = dl.material_regions(12, "bcc_dg")
    assert len(r) == 2 and np.array_equal(r[0], sg) and np.array_equal(np.union1d(r[0], r[1]), dg)
    assert np.intersect1d(r[0], r[1]).size == 0 and r[1].size > 0
    assert [np.array_equal(a, dl.diel_io_index(12, "fcc")) for a in dl.material_regions(12, "fcc")] == [True]
    with pytest.raises(ValueError, match="regions"):
        emu.discretization.materials_handle(12, "bcc_dg", eps_opt=[16.0])
    # later regions override earlier ones
    h = emu.discretization.materials_handle(6, "sc_curv", eps_opt=[2.0, 4.0], regions=[np.arange(10), np.arange(5, 12)])
    assert np.array_equal(h.mat[:13], [1] * 5 + [2] * 7 + [0]) and np.array_equal(h.inv_eps, [1.0, 0.5, 0.25])


# ---- 3: uniform medium ---------------------------------------------------------------------------------------------------
def _uniform(pkg, oc, N, options):
    def run(ctx):
        mfd = pkg.discretization
        X = ctx.random_block(3, 8)
        A_mat = _ops(pkg, N, "sc_curv", mfd.materials_handle(N, "sc_curv", regions=[], background=4.0))[0]
        A_vac = _ops(pkg, N, "sc_curv", None)[0]
        assert np.array_equal(A_mat(X).get(), 0.25 * A_vac(X).get())
        T = A_mat.op.a_fft.tables
        for q, w in (((1, 2, 0), [0.3, -1.0, 0.5]), ((N - 1, 0, 3 % N), [1.0, 0.2, -0.7])):
            x, K, _ = _mode(N, T, q, w)
            want = np.vdot(K, K).real / 4 * x
            got = np.asarray(A_mat(x[:, None])).ravel()
            assert np.linalg.norm(got - want) <= 1e-13 * np.linalg.norm(want)

    _with_options(pkg, N, options, run)


@pytest.mark.parametrize("N,options", [(8, {}), (24, {"mid_five": 0}), (16, {"plane_split": 1}), (6, {}), (12, {})])
def test_uniform_medium_emu(emu, oracle, N, options):
    _uniform(emu, oracle, N, options)


@pytest.mark.gpu
@pytest.mark.parametrize("N,options", [(120, {"mid_five": 0}), (160, {}), (150, {})])
def test_uniform_medium(gpu, oracle, N, options):
    _uniform(gpu, oracle, N, options)


# ---- 4: solve parity ------------------------------------------------------------------------------------------------------
def _solve(pkg, oc, N, nev):
    alpha = np.array([0.3, 0.2, 0.1]) * np.pi
    eps = [16.0, 12.0]
    regions = pkg.dielectric.material_regions(N, "bcc_dg")
    mat = np.zeros(3 * N ** 3, dtype=np.uint8)
    for i, r in enumerate(regions):
        mat[r] = i + 1
    x0 = oc.random_x0(3 * N ** 3, oc.block_width(nev), 17)
    res = pkg.numerical_experiments.eigen_1p(N, "bcc_dg", alpha, type="materials", eps_opt=eps, nev=nev, x0=x0.copy())
    a, b, inv, shift, _ = oc.assemble_symbols(N, "bcc_dg", alpha)
    H, P = oc.pc_mfd_handle(a, b, oracle_materials(mat, [1.0, 1 / 16.0, 1 / 12.0]), inv, shift)[1:]
    lam, _, info = oc.lobpcg_sep_softlock(H, P, x0, nev)
    assert int(res["info"][0]) == int(info[0])
    assert np.all(np.abs(res["lambdas"][:nev] - lam[:nev]) <= 1e-10 * np.abs(lam[:nev]))


@pytest.mark.parametrize("N", [12, 16])
def test_solve_parity_emu(emu, oracle, N):
    _solve(emu, oracle, N, 6)


@pytest.mark.gpu
def test_solve_parity(gpu, oracle):
    _solve(gpu, oracle, 48, 10)


# ---- 6: refusals ----------------------------------------------------------------------------------------------------------
def _refusals(pkg):
    import ctypes as C
    L = pkg._lib
    N = 6
    ctx = pkg.get_context(N)
    good_mat, good_eps = np.zeros(3 * N ** 3, dtype=np.uint8), np.array([1.0, 0.5])

    def create(c, mat, inv_eps, n=None, n_mat=None):
        h = C.c_void_p()
        inv_eps = np.ascontiguousarray(inv_eps, dtype=np.float64)
        rc = L.lib().pcb_diel_create_materials(c.h, mat.ctypes.data, mat.size if n is None else n,
                                               inv_eps.ctypes.data_as(L.c_double_p), len(inv_eps) if n_mat is None else n_mat, C.byref(h))
        return rc, h.value

    assert create(ctx, good_mat, good_eps)[0] == 0
    bad_index = good_mat.copy()
    bad_index[77] = 2
    big = np.full(257, 0.5)
    for args, what in [((bad_index, good_eps), b"mat[77]"), ((good_mat, good_eps, None, 0), b"n_mat"),
                       ((good_mat, big), b"n_mat"), ((good_mat, [1.0, -0.5]), b"inv_eps[1]"), ((good_mat, [1.0, 0.0]), b"inv_eps[1]"),
                       ((good_mat, [np.inf, 0.5]), b"inv_eps[0]"), ((good_mat, [1.0, np.nan]), b"inv_eps[1]"),
                       ((good_mat, good_eps, 3 * N ** 3 - 1), b"n = ")]:
        rc, h = create(ctx, *args)
        assert rc == -1 and h is None, what
        assert what in L.lib().pcb_last_error(), (what, L.lib().pcb_last_error())
    slab = pkg.devarray.Context(N, pkg.devarray.default_device(), slab=(0, 3))
    rc, h = create(slab, good_mat, good_eps)
    assert rc == -2 and h is None and b"slab" in L.lib().pcb_last_error()
    with pytest.raises(ValueError, match="0 ... 255"):
        pkg.discretization.DielHandle.materials(N, np.full(3 * N ** 3, 300), good_eps)


def test_refusals_emu(emu):
    _refusals(emu)


@pytest.mark.gpu
def test_refusals(gpu):
    _refusals(gpu)


# ---- 7: runners -----------------------------------------------------------------------------------------------------------
def _runners(pkg, N, tmp_path):
    ne = pkg.numerical_experiments
    d_flag, nev = "bcc_dg", 4
    n_k = pkg.dielectric.kpath(d_flag, ne.GAP).shape[0]
    idx = [0, 1]
    keys = [f"{d_flag}_{N}_iterations", f"{d_flag}_{N}_frequencies"]
    p_mat, p_ch, p_two = (str(tmp_path / f) for f in ("mat.json", "chiral.json", "two.json"))
    # with the defaults the materials M is the chiral M: the same pass structure gives the same rows
    assert ne.bandgap(N, d_flag, type="materials", indices=idx, nev=nev, seed=3, path=p_mat) == []
    assert ne.bandgap(N, d_flag, type="chiral", indices=idx, nev=nev, seed=3, path=p_ch) == []
    mat, ch = json.load(open(p_mat)), json.load(open(p_ch))
    assert set(mat) == set(keys) and len(mat[keys[0]]) == n_k
    assert mat[keys[1]][:2] == ch[keys[1]][:2]
    # two networks, with energy and velocity rows
    assert ne.bandgap(N, d_flag, type="materials", eps_opt=[16.0, 12.0], indices=idx, nev=nev, seed=3, path=p_two,
                      energy=True, velocity=True) == []
    two = json.load(open(p_two))
    for i in idx:
        assert all(0.0 < f < 1.0 for f in two[f"{d_flag}_{N}_energy_fraction"][i])
        assert len(two[f"{d_flag}_{N}_group_velocity"][i]) == nev
        assert two[keys[1]][i] != mat[keys[1]][i]
    r = ne.eigen_1p(N, d_flag, [0.3, 0.2, 0.1], type="materials", eps_opt=[16.0, 12.0], nev=nev, seed=3, energy=True, velocity=True)
    assert r["energy_fraction"].shape == (nev,) and r["group_velocity"].shape == (nev, 3)


def test_runners_emu(emu, tmp_path):
    _runners(emu, 8, tmp_path)


@pytest.mark.gpu
def test_runners(gpu, tmp_path):
    _runners(gpu, 48, tmp_path)


@pytest.mark.gpu
def test_run_bandgap_cli(tmp_path):
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PCB200_QUIET="1", PYTHONPATH=root)
    out = subprocess.run([sys.executable, os.path.join(root, "tools", "run_bandgap.py"), "16", "bcc_dg", "materials", "4", "2",
                          "--eps", "16,12", "--energy", "--velocity"], cwd=str(tmp_path), env=env, capture_output=True, text=True,
                         timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    fin = json.load(open(os.path.join(str(tmp_path), line["json"])))
    for i in (0, 1):
        assert all(v is not None for v in fin["bcc_dg_16_group_velocity"][i])
        assert all(0.0 < f < 1.0 for f in fin["bcc_dg_16_energy_fraction"][i])
