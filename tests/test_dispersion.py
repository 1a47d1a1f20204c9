"""Dispersive materials: pcb_material_energy, pcb_diel_set_inv_eps, the permittivity models and the self-consistent band iteration.

For a column x, D = FFT3(K_A^H x), E = M D, rows r = c N^3 + p of a materials dielectric (E_r = D_r / eps_{mat[r]}):
    e_m = Re sum_{r: mat[r] = m} conj(D_r) E_r / N^3,   sum_m e_m = e_tot,   sum_{m != 0} e_m = e_in (pcb_field_energy).
The test restates e_m from the NumPy oracle's D (oracle/pc_oracle.py: a_block, scipy.fft.fftn) binned by material.  A band of a
crystal with eps_m(f) is self-consistent where f = F_j(eps(f)), F_j the plain solve's frequency; in a homogeneous medium the roots
are known in closed form.  The ``emu`` tests run at small N on the host-emulation build (whole planes at N = 8, 16, half planes at
16, natural layout at 6 and 12); the ``gpu`` tests run the kernels at N = 120 (whole planes), 160 (half planes) and 150 (natural
layout) on the B200, and the solves at the sizes of the other solver tests.
"""
import json
import math
import os

import numpy as np
import pytest

from test_field_energy import _GENERIC, _same, emu, field_energy, gpu  # noqa: F401
from test_materials import _ops, _with_options, oracle_materials, random_map

_LAYOUTS_EMU = [(8, {}), (16, {}), (16, {"plane_split": 1}), (6, {}), (12, {})]
_LAYOUTS_GPU = [(120, {}), (160, {}), (150, {})]


def _raw_energy(pkg, op, X, n_mat, out):
    L = pkg._lib
    return L.lib().pcb_material_energy(op.h, X.k, L.ptr_array(X.ptrs), n_mat, out.ctypes.data_as(L.c_double_p))


# ---- 1: per-material energy against the oracle --------------------------------------------------------------------------
def _check_energy(pkg, oc, N, options, n_mat, widths=(1, 3, 16, 33)):
    def run(ctx):
        mat, inv_eps = random_map(N, n_mat, 300 + N + n_mat)
        Diels = pkg.discretization.DielHandle.materials(N, mat, inv_eps)
        A_func = _ops(pkg, N, "bcc_dg", Diels)[0]
        op = A_func.op
        a = oc.assemble_symbols(N, "bcc_dg", np.asarray(_GENERIC))[0]
        k = max(widths)
        X = ctx.random_block(k, 77 + N)
        chk = [0, k - 1]
        x = X.get()[:, chk]
        D, E, _, _ = field_energy(x, a, oracle_materials(mat, inv_eps), np.flatnonzero(mat))
        t = (D.conj() * E).real / N ** 3
        want = np.array([np.bincount(mat, weights=t[:, j], minlength=n_mat) for j in range(len(chk))])
        n0 = ctx.launches()
        e = op.material_energy(X)
        # the forward half of A's layout and the two reduction kernels, per launch of 32 columns
        fwd = 2 if options.get("plane", 1) and N % 8 == 0 and N <= 160 else 3
        assert ctx.launches() - n0 == ((k + 31) // 32) * (fwd + 2)
        got = e[chk]
        assert got.shape == want.shape
        nz = want > 0
        assert np.all(np.abs(got[nz] - want[nz]) <= 1e-12 * want[nz]), np.max(np.abs(got[nz] - want[nz]) / want[nz])
        assert np.all(got[~nz] == 0.0)
        # sums: e_tot and e_in of pcb_field_energy, to rounding
        e_in, e_tot = op.field_energy(X)
        assert np.all(np.abs(e.sum(axis=1) - e_tot) <= 1e-13 * e_tot)
        assert np.all(np.abs(e[:, 1:].sum(axis=1) - e_in) <= 1e-13 * e_tot)
        # a row has the same bits at every width and on every call
        for w in widths:
            assert np.array_equal(op.material_energy(X.cols(range(w))), e[:w]), w
        for j in (1, k // 2, k - 1):
            assert np.array_equal(op.material_energy(X.cols([j])), e[j:j + 1]), j
        assert np.array_equal(op.material_energy(X), e)
        # a host array is uploaded
        assert np.array_equal(op.material_energy(X.get()[:, :1]), e[:1])

    _with_options(pkg, N, options, run)


# n_mat <= 16: bins in registers; 17 and 256: the match path
@pytest.mark.parametrize("n_mat", [1, 2, 8, 16, 17, 256])
@pytest.mark.parametrize("N,options", _LAYOUTS_EMU, ids=lambda v: str(v))
def test_material_energy_emu(emu, oracle, N, options, n_mat):
    _check_energy(emu, oracle, N, options, n_mat)


@pytest.mark.gpu
@pytest.mark.parametrize("n_mat", [1, 2, 8, 16, 17, 256])
@pytest.mark.parametrize("N,options", _LAYOUTS_GPU + [(120, {"plane": 0})], ids=lambda v: str(v))
def test_material_energy(gpu, oracle, N, options, n_mat):
    _check_energy(gpu, oracle, N, options, n_mat)


def _default_map(pkg, N, d_flag, options):
    """On materials_handle's default map, sum_{m != 0} f_m is energy_fraction of the same operator."""
    def run(ctx):
        ne = pkg.numerical_experiments
        A_func = _ops(pkg, N, d_flag, pkg.discretization.materials_handle(N, d_flag))[0]
        X = ctx.random_block(5, 9)
        f = ne.material_energy(X, A_func)
        assert f.shape == (5, 3 if d_flag == "bcc_dg" else 2)
        assert np.all(np.abs(f.sum(axis=1) - 1.0) <= 1e-14)
        assert np.all(np.abs(f[:, 1:].sum(axis=1) - ne.energy_fraction(X, A_func)) <= 1e-13)
        if d_flag == "bcc_dg":
            assert np.all(f[:, 1] > 0) and np.all(f[:, 2] > 0)

    _with_options(pkg, N, options, run)


@pytest.mark.parametrize("d_flag", ["bcc_dg", "fcc"])
@pytest.mark.parametrize("N,options", [(8, {}), (16, {"plane_split": 1}), (12, {})], ids=lambda v: str(v))
def test_default_map_emu(emu, N, options, d_flag):
    _default_map(emu, N, d_flag, options)


@pytest.mark.gpu
@pytest.mark.parametrize("N,options", _LAYOUTS_GPU, ids=lambda v: str(v))
def test_default_map(gpu, N, options):
    _default_map(gpu, N, "bcc_dg", options)


# ---- 2: refusals ------------------------------------------------------------------------------------------------------------
def _refusals(pkg):
    import ctypes as C
    L = pkg._lib
    mfd = pkg.discretization
    N = 8
    ctx = pkg.get_context(N)
    X = ctx.random_block(2, 3)
    mat, inv_eps = random_map(N, 3, 5)
    Diels = mfd.DielHandle.materials(N, mat, inv_eps)
    A_mat = _ops(pkg, N, "bcc_dg", Diels)[0]
    out = np.full((2, 4), 7.0)
    for A_func, n_mat, what in ((_ops(pkg, N, "bcc_dg", mfd.chiral_handle(N, "bcc_dg"))[0], 2, b"materials"),
                                (_ops(pkg, N, "bcc_dg", None)[0], 1, b"materials"),
                                (A_mat, 4, b"n_mat = 4"), (A_mat, 2, b"n_mat = 2")):
        assert _raw_energy(pkg, A_func.op, X, n_mat, out) == -1, what
        assert what in L.lib().pcb_last_error(), L.lib().pcb_last_error()
        assert np.all(out == 7.0)
    with pytest.raises(L.PcbError, match="materials"):
        _ops(pkg, N, "bcc_dg", None)[0].op.material_energy(X)
    slab = pkg.devarray.Context(N, pkg.devarray.default_device(), slab=(0, 4))
    a_fft, _ = mfd.fft_blocks(N, 1, pkg.dielectric.diel_info("bcc_dg", option="ct"), alpha=np.array(_GENERIC))
    op = pkg.pcfft.Operator(a_fft, 0.0, 0.0, 0.0, None, ctx=slab)
    Xs = slab.random_block(2, 5)
    assert _raw_energy(pkg, op, Xs, 3, out) == -2 and b"slab" in L.lib().pcb_last_error()
    assert np.all(out == 7.0)
    # pcb_diel_set_inv_eps: wrong length, eps <= 0, NaN, another kind; A keeps its bits
    before = A_mat(X).get()
    for t, what in (([0.5, 0.25], b"n_mat = 2"), ([0.5, 0.25, 0.1, 0.1], b"n_mat = 4"), ([0.5, -0.25, 0.1], b"inv_eps[1]"),
                    ([0.5, 0.0, 0.1], b"inv_eps[1]"), ([0.5, 0.25, np.nan], b"inv_eps[2]"), ([np.inf, 0.25, 0.1], b"inv_eps[0]")):
        t = np.asarray(t, dtype=np.float64)
        assert L.lib().pcb_diel_set_inv_eps(Diels.h, t.ctypes.data_as(L.c_double_p), len(t)) == -1, what
        assert what in L.lib().pcb_last_error(), (what, L.lib().pcb_last_error())
        with pytest.raises(L.PcbError):
            Diels.set_inv_eps(t)
        assert np.array_equal(A_mat(X).get(), before)
    assert np.array_equal(Diels.inv_eps, inv_eps)
    ch = mfd.chiral_handle(N, "bcc_dg")
    t = np.array([1.0, 0.5])
    assert L.lib().pcb_diel_set_inv_eps(ch.h, t.ctypes.data_as(L.c_double_p), 2) == -1
    assert b"MATERIALS" in L.lib().pcb_last_error()
    with pytest.raises(ValueError):
        ch.set_inv_eps(t)
    # at_frequency refuses an eps that is not > 0 (below the Drude window) and keeps the table
    h = mfd.materials_handle(N, "bcc_dg", eps_opt=[16.0, pkg.dispersion.Drude(4.0, 1.0)])
    t0 = h.inv_eps.copy()
    with pytest.raises(ValueError, match="finite and > 0"):
        h.at_frequency(0.4)
    assert np.array_equal(h.inv_eps, t0)
    del C


def test_refusals_emu(emu):
    _refusals(emu)


@pytest.mark.gpu
def test_refusals(gpu):
    _refusals(gpu)


# ---- 3: table update ----------------------------------------------------------------------------------------------------------
def _table_update(pkg, N, options):
    def run(ctx):
        mfd = pkg.discretization
        mat, t0 = random_map(N, 8, 11)
        t1 = 1.0 / np.random.default_rng(12).uniform(1.5, 16.0, size=8)
        h = mfd.DielHandle.materials(N, mat, t0)
        A_old, H_old = _ops(pkg, N, "bcc_dg", h)
        X = ctx.random_block(3, 21)
        A_old(X), H_old(X)
        h.set_inv_eps(t1)
        assert np.array_equal(h.inv_eps, t1)
        A_new, H_new = _ops(pkg, N, "bcc_dg", mfd.DielHandle.materials(N, mat, t1))
        assert _same(pkg, A_old(X), A_new(X)).all()
        assert _same(pkg, H_old(X), H_new(X)).all()
        assert np.array_equal(A_old.op.material_energy(X), A_new.op.material_energy(X))

    _with_options(pkg, N, options, run)


@pytest.mark.parametrize("N,options", [(8, {}), (16, {"plane_split": 1}), (12, {})], ids=lambda v: str(v))
def test_table_update_emu(emu, N, options):
    _table_update(emu, N, options)


@pytest.mark.gpu
@pytest.mark.parametrize("N,options", _LAYOUTS_GPU, ids=lambda v: str(v))
def test_table_update(gpu, N, options):
    _table_update(gpu, N, options)


# ---- 4: Hellmann-Feynman per material -----------------------------------------------------------------------------------------
def _hellmann_feynman(pkg, N):
    """Two-network double gyroid at eps = (16, 12): dlambda/deps_2 = -lambda f_2 / eps_2, against a central difference of
    warm-started solves in eps_2 (tolerance of test_field_energy's Hellmann-Feynman test)."""
    ne, mfd = pkg.numerical_experiments, pkg.discretization
    d_flag, alpha, nev, eps = "bcc_dg", np.array(_GENERIC), 6, [16.0, 12.0]
    res = ne.eigen_1p(N, d_flag, alpha, type="materials", nev=nev, seed=11, tol=1e-7, eps_opt=eps)
    a_fft, b_fft, inv_fft, _, shift = ne.uniform_initialization(N, d_flag, alpha, nev=nev, seed=11)
    A_func = ne.pc_mfd_handle(a_fft, b_fft, mfd.materials_handle(N, d_flag, eps_opt=eps), inv_fft, shift)[0]
    f2 = ne.material_energy(res["x"][:, :nev], A_func)[:, 2]
    lam = (2 * np.pi * np.asarray(res["omega_re"])) ** 2
    h = 1e-3 * eps[1]
    lp, lm = [(2 * np.pi * np.asarray(ne.eigen_1p(N, d_flag, alpha, type="materials", nev=nev, x0=res["x"].copy(), tol=1e-7,
                                                    eps_opt=[eps[0], e])["omega_re"])) ** 2 for e in (eps[1] + h, eps[1] - h)]
    fd = (lp - lm) / (2 * h)
    hf = -lam * f2 / eps[1]
    gaps = np.diff(lam)
    checked = 0
    for i in range(nev):
        lo = gaps[i - 1] if i > 0 else np.inf
        hi = gaps[i] if i < nev - 1 else np.inf
        if min(lo, hi) > 1e-2 * lam[i] and lam[i] > 1e-6:
            assert abs(fd[i] - hf[i]) <= 1e-4 * abs(hf[i]), (i, fd[i], hf[i])
            checked += 1
    assert checked >= 2, (lam, f2)


def test_hellmann_feynman_per_material_emu(emu):
    _hellmann_feynman(emu, 8)


@pytest.mark.gpu
def test_hellmann_feynman_per_material(gpu):
    _hellmann_feynman(gpu, 48)


# ---- 5: exact answers in a homogeneous dispersive medium ----------------------------------------------------------------------
def _homogeneous(pkg, N, nev):
    ne, dsp = pkg.numerical_experiments, pkg.dispersion
    d_flag, alpha = "sc_curv", np.array(_GENERIC)
    kw = dict(nev=nev, seed=7, tol=1e-8)
    vac = np.asarray(ne.eigen_1p(N, d_flag, alpha, type=None, **kw)["omega_re"])
    # Drude: eps_inf f^2 - f_p^2 = f_vac^2
    eps_inf, f_p = 2.0, 0.4
    r = ne.eigen_1p(N, d_flag, alpha, type="materials", diel_kw={"regions": [], "background": dsp.Drude(eps_inf, f_p)}, **kw)
    want = np.sqrt((vac ** 2 + f_p ** 2) / eps_inf)
    assert np.all(np.abs(r["omega_re"] - want) <= 1e-7 * want), (r["omega_re"], want)
    assert r["eps"].shape == (nev, 1) and np.all(r["newton_steps"] >= 1)
    assert np.allclose(r["eps"][:, 0], eps_inf - f_p ** 2 / want ** 2, rtol=1e-6)
    labels = dsp._clusters(vac, 1e-6)
    assert len(set(labels)) < nev          # the plane-wave pairs: the cluster path
    # Lorentz: -eps_inf x^2 + (eps_inf f0^2 + sigma f0^2 + f_vac^2) x - f_vac^2 f0^2 = 0, x = f^2
    eps_inf, sigma, f0 = 2.0, 1.5, float(np.mean(vac))
    lor = dsp.Lorentz(eps_inf, [(sigma, f0)])
    b = eps_inf * f0 ** 2 + sigma * f0 ** 2 + vac ** 2
    disc = np.sqrt(b * b - 4 * eps_inf * vac ** 2 * f0 ** 2)
    upper, lower = np.sqrt((b + disc) / (2 * eps_inf)), np.sqrt((b - disc) / (2 * eps_inf))
    diel_kw = {"regions": [], "background": lor}
    r_up = ne.eigen_1p(N, d_flag, alpha, type="materials", diel_kw=diel_kw, **kw)
    assert np.all(np.abs(r_up["omega_re"] - upper) <= 1e-7 * upper), (r_up["omega_re"], upper)
    r_lo = ne.eigen_1p(N, d_flag, alpha, type="materials", diel_kw=diel_kw, window=(0.0, f0), **kw)
    assert np.all(np.abs(r_lo["omega_re"] - lower) <= 1e-7 * lower), (r_lo["omega_re"], lower)
    # constant models are not dispersive: exactly the plain result
    c = ne.eigen_1p(N, d_flag, alpha, type="materials", diel_kw={"regions": [], "background": dsp.Constant(4.0)}, **kw)
    p = ne.eigen_1p(N, d_flag, alpha, type="materials", diel_kw={"regions": [], "background": 4.0}, **kw)
    assert np.array_equal(c["omega_re"], p["omega_re"]) and "newton_steps" not in c


def test_homogeneous_emu(emu):
    _homogeneous(emu, 8, 6)


@pytest.mark.gpu
def test_homogeneous(gpu):
    _homogeneous(gpu, 48, 10)


# ---- 6: self-consistency in a crystal -----------------------------------------------------------------------------------------
def _crystal(pkg, N, nev):
    ne, dsp = pkg.numerical_experiments, pkg.dispersion
    alpha = np.array(_GENERIC)
    lor = dsp.Lorentz(12.0, [(2.0, 2.0)])
    # the bands lie below the resonance (above it, in the highest window, the network at eps -> 0 expels the field: no root)
    r = ne.eigen_1p(N, "bcc_dg", alpha, type="materials", eps_opt=[16.0, lor], nev=nev, seed=5, tol=1e-8, window=(0.0, 2.0))
    f = np.asarray(r["omega_re"])
    assert np.all(np.isfinite(f)) and np.all(r["newton_steps"] <= 8), (f, r["newton_steps"])
    assert np.allclose(r["eps"][:, 2], lor.eps(f)) and np.all(r["eps"][:, 1] == 16.0)
    for j in range(nev):
        p = ne.eigen_1p(N, "bcc_dg", alpha, type="materials", eps_opt=[16.0, float(lor.eps(f[j]))], nev=nev, seed=6, tol=1e-8)
        assert abs(p["omega_re"][j] - f[j]) <= 1e-7 * f[j], (j, p["omega_re"][j], f[j])


def test_crystal_emu(emu):
    _crystal(emu, 8, 4)


@pytest.mark.gpu
def test_crystal(gpu):
    _crystal(gpu, 32, 6)


# ---- 7: CPU only: the models and the iteration --------------------------------------------------------------------------------
def test_models():
    import importlib
    dsp = importlib.import_module("linear-eigenvalue-problems-in-photonic-crystals_b200.dispersion")
    dr, lo = dsp.Drude(2.0, 0.5), dsp.Lorentz(3.0, [(1.0, 1.0), (0.5, 2.0)])
    for m, fs in ((dr, [0.5, 0.9, 3.0]), (lo, [0.3, 1.5, 2.5])):
        for f in fs:
            h = 1e-6 * f
            assert abs(m.deps(f) - (m.eps(f + h) - m.eps(f - h)) / (2 * h)) <= 1e-6 * abs(m.deps(f)), (m, f)
            assert m.deps(f) > 0
    assert dr.windows() == [(0.5 / math.sqrt(2.0), math.inf)]
    w = lo.windows()
    assert len(w) == 3 and w[0] == (0.0, 1.0) and w[1][1] == 2.0 and w[2][1] == math.inf
    for a, b in w[1:]:
        assert abs(lo.eps(a)) < 1e-9 and lo.eps(a * (1 + 1e-6)) > 0
        assert lo.eps(0.5 * (a + min(b, 10.0))) > 0
    assert lo.eps(0.999) > 0 and lo.eps(0.0) == 3.0 + 1.0 + 0.5
    assert dsp.windows([dr, 4.0, lo]) == [(0.5 / math.sqrt(2.0), 1.0), w[1], w[2]]
    assert dsp.is_dispersive([1.0, dr]) and not dsp.is_dispersive([1.0, dsp.Constant(2.0)])
    for bad in (lambda: dsp.Drude(0.0, 1.0), lambda: dsp.Lorentz(1.0, []), lambda: dsp.Lorentz(1.0, [(-1.0, 1.0)])):
        with pytest.raises(ValueError):
            bad()


def _synthetic(dsp, c, models, calls=None):
    """solve(f, x) of a synthetic crystal: lambda_j = sum_m c[j, m] / eps_m(f) (monotone), fractions f_jm = c_jm / eps_m / lambda_j;
    F = sqrt(lambda) (s = 1)."""
    models = [dsp.as_model(m) for m in models]

    def solve(f, x):
        if calls is not None:
            calls.append(f)
        inv = np.array([1.0 / float(m.eps(f)) for m in models])
        e = c * inv[None, :]
        lam = e.sum(axis=1)
        return np.sqrt(lam), e / lam[:, None], (x or 0) + 1
    return solve


def test_self_consistent_synthetic():
    import importlib
    from scipy.optimize import brentq
    dsp = importlib.import_module("linear-eigenvalue-problems-in-photonic-crystals_b200.dispersion")
    models = [1.0, dsp.Drude(4.0, 0.8), dsp.Lorentz(6.0, [(1.0, 3.0)])]
    c = np.array([[0.2, 1.0, 0.5], [0.2, 1.0, 0.5], [0.1, 3.0, 2.0], [1.0, 2.0, 6.0]])
    solve = _synthetic(dsp, c, models)
    lo, hi = dsp.windows(models)[-1]
    assert hi == math.inf and lo > 3.0

    def root(j, a, b):
        return brentq(lambda f: f * f - sum(c[j, m] / float(dsp.as_model(models[m]).eps(f)) for m in range(3)), a, b, xtol=1e-15)
    want = np.array([root(j, lo * (1 + 1e-9), 100.0) for j in range(4)])
    res = dsp.self_consistent(solve, models, np.full(4, 1.0))
    assert np.all(np.abs(res["freq"] - want) <= 1e-9 * want), (res["freq"], want)
    # bands 0 and 1 coincide: one shared iteration
    assert res["steps"][0] == res["steps"][1] and res["solves"] == res["steps"][0] + res["steps"][2] + res["steps"][3]
    assert res["x"] == res["solves"] and np.all(res["steps"] <= 6)
    # a start far above the roots
    far = dsp.self_consistent(solve, models, np.full(4, 20.0), max_steps=20)
    assert np.all(np.abs(far["freq"] - want) <= 1e-9 * want), far["freq"]
    # fractions that hide the eps term of g': every Newton step overshoots, and leaves the bracket from the second one on;
    # the bisection fallback still converges
    calls = []
    inner = _synthetic(dsp, c, models, calls)

    def wrong(f, x):
        F, frac, x = inner(f, x)
        return F, 0.0 * frac, x
    bis = dsp.self_consistent(wrong, models, np.full(4, 1.0), max_steps=80)
    assert np.all(np.abs(bis["freq"] - want) <= 1e-6 * want), bis["freq"]      # linear convergence: the step-size stop
    assert np.any(np.diff(np.sign(np.array(calls[:bis["steps"][0]]) - want[0])) != 0)      # iterates on both sides of the root
    # the window below the Lorentz resonance (its own roots), and a cap on the solves that leaves NaN
    w0 = dsp.windows(models)
    low = [w for w in w0 if w[1] == 3.0][0]
    want_lo = np.array([root(j, low[0] * (1 + 1e-12), 3.0 * (1 - 1e-12)) for j in range(4)])
    res_lo = dsp.self_consistent(solve, models, np.full(4, 1.0), window=low)
    assert np.all(np.abs(res_lo["freq"] - want_lo) <= 1e-9 * want_lo), (res_lo["freq"], want_lo)
    capped = dsp.self_consistent(solve, models, np.full(4, 20.0), max_steps=2)
    assert np.all(np.isnan(capped["freq"])) and np.all(capped["steps"] == 2)
    # no root: a band with F = 0 at every eps (a zero mode) gets NaN after one solve
    c0 = c.copy()
    c0[3] = 0.0
    z = dsp.self_consistent(_synthetic(dsp, c0, models), models, np.full(4, 1.0), zero=1e-4)
    assert np.isnan(z["freq"][3]) and z["steps"][3] == 1 and np.all(np.isfinite(z["freq"][:3]))
    with pytest.raises(ValueError):
        dsp.self_consistent(solve, models, np.full(4, 1.0), window=(2.0, 1.0))


# ---- 8: runners ---------------------------------------------------------------------------------------------------------------
def _runners(pkg, N, tmp_path, idx):
    ne, dsp = pkg.numerical_experiments, pkg.dispersion
    d_flag, nev = "bcc_dg", 4
    key_it, key_fq, key_en = (f"{d_flag}_{N}_{s}" for s in ("iterations", "frequencies", "energy_fraction"))
    n_k = pkg.dielectric.kpath(d_flag, ne.GAP).shape[0]
    a, b, c = idx
    eps = [16.0, dsp.Drude(12.0, 0.5)]
    p_all, p_part = str(tmp_path / "all.json"), str(tmp_path / "part.json")
    assert ne.bandgap(N, d_flag, type="materials", eps_opt=eps, indices=idx, nev=nev, seed=3, path=p_all, energy=True) == []
    rec = json.load(open(p_all))
    assert set(rec) == {key_it, key_fq, key_en} and len(rec[key_fq]) == n_k
    for i in idx:
        fq = rec[key_fq][i]
        assert len(fq) == nev and rec[key_it][i][0] > 0 and rec[key_it][i][1] > 0
        # a band that stays below the plasma edge at every eps (near Gamma) has no root: null; so have the zero modes at Gamma
        assert all(v is None or v > 0.5 / math.sqrt(12.0) for v in fq) and fq[-1] is not None
        if not np.any(pkg.dielectric.kpath(d_flag, ne.GAP)[i]):
            assert fq[:2] == [None, None]
        assert all(v is None or 0.0 < v < 1.0 for v in rec[key_en][i])
    # the frequency rows are self-consistent: a plain solve at eps(f) at the last point returns f
    alpha = pkg.dielectric.kpath(d_flag, ne.GAP)[c]
    f = rec[key_fq][c][-1]
    p = ne.eigen_1p(N, d_flag, alpha, type="materials", eps_opt=[16.0, float(eps[1].eps(f))], nev=nev, seed=4, tol=1e-8)
    assert abs(p["omega_re"][-1] - f) <= 1e-5 * f
    # resume: a file with the rows of the first two points only gets the third
    assert ne.bandgap(N, d_flag, type="materials", eps_opt=eps, indices=[a, b], nev=nev, seed=3, path=p_part) == []
    assert ne.bandgap(N, d_flag, type="materials", eps_opt=eps, nev=nev, seed=3, path=p_part, only=idx) == []
    part = json.load(open(p_part))
    assert part[key_fq][a:c] == rec[key_fq][a:c]
    assert [v is None for v in part[key_fq][c]] == [v is None for v in rec[key_fq][c]]
    assert all(abs(u - v) <= 1e-6 * v for u, v in zip(part[key_fq][c], rec[key_fq][c]) if v is not None)
    # velocity=True is refused with a dispersive material
    with pytest.raises(ValueError, match="d eps / d omega"):
        ne.bandgap(N, d_flag, type="materials", eps_opt=eps, indices=idx, nev=nev, path=str(tmp_path / "v.json"), velocity=True)
    with pytest.raises(ValueError, match="d eps / d omega"):
        ne.eigen_1p(N, d_flag, _GENERIC, type="materials", eps_opt=eps, nev=nev, velocity=True)


def test_runners_emu(emu, tmp_path):
    _runners(emu, 8, tmp_path, [0, 1, 2])      # away from Gamma: at N = 8 many bands near it have no root and spend 12 solves each


@pytest.mark.gpu
def test_runners(gpu, tmp_path):
    _runners(gpu, 32, tmp_path, [18, 19, 20])    # across Gamma (19)


def test_sharded_two_ranks_emu(emu_lib, tmp_path):
    """bandgap_sharded over two gloo processes with a Drude network: the merged rows equal those of single-process runs of the
    same chunks."""
    import subprocess
    import sys
    from conftest import ROOT
    out2, out1 = tmp_path / "w2", tmp_path / "w1"
    out2.mkdir()
    out1.mkdir()
    env = dict(os.environ, PCB200_QUIET="1", OMP_NUM_THREADS="1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29573", os.path.join(ROOT, "tests", "dist_worker_dispersion.py"), str(out2), emu_lib]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    merged = json.load(open(out2 / "bandgap_bcc_dg.json"))
    import importlib
    pcb = importlib.import_module("linear-eigenvalue-problems-in-photonic-crystals_b200")
    pcb._lib.use_library(emu_lib)
    ne = pcb.numerical_experiments
    eps = [16.0, pcb.dispersion.Drude(12.0, 0.5)]
    for rank in (0, 1):
        ne.bandgap_sharded(8, "bcc_dg", rank, 2, type="materials", eps_opt=eps, nev=4, seed=1000, out_dir=str(out1) + "/",
                           indices=[1, 2, 3, 4], energy=True)
    for rank, ks in ((0, [1, 2]), (1, [3, 4])):
        part = json.load(open(out1 / f"bandgap_bcc_dg.rank{rank}.json"))
        for k in ks:
            for key in ("frequencies", "energy_fraction"):
                assert merged[f"bcc_dg_8_{key}"][k] == part[f"bcc_dg_8_{key}"][k], (k, key)
            assert merged["bcc_dg_8_iterations"][k][0] == part["bcc_dg_8_iterations"][k][0]
            assert all(v is not None and v > 0 for v in merged["bcc_dg_8_frequencies"][k])
    assert merged["bcc_dg_8_iterations"][0] == [0, 0]
    pcb.devarray.drop_contexts()


def test_parse_eps():
    """--eps entries of tools/run_bandgap.py: numbers, drude:EPS_INF:FP, lorentz:EPS_INF:SIGMA:F0; anything else is refused."""
    import importlib.util
    from conftest import ROOT
    spec = importlib.util.spec_from_file_location("run_bandgap", os.path.join(ROOT, "tools", "run_bandgap.py"))
    rb = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(rb)
    dsp = importlib.import_module("linear-eigenvalue-problems-in-photonic-crystals_b200.dispersion")
    assert rb.parse_eps("16", dsp) == 16.0
    d = rb.parse_eps("drude:12:0.5", dsp)
    assert isinstance(d, dsp.Drude) and (d.eps_inf, d.f_p) == (12.0, 0.5)
    lo = rb.parse_eps("lorentz:12:2:2.0", dsp)
    assert isinstance(lo, dsp.Lorentz) and lo.eps_inf == 12.0 and lo.terms == [(2.0, 2.0)]
    for bad in ("drude:12", "lorentz:12:2", "debye:1:2", "drude:12:0.5:1"):
        with pytest.raises(SystemExit, match="expected a number"):
            rb.parse_eps(bad, dsp)


@pytest.mark.gpu
def test_run_bandgap_cli_drude(tmp_path):
    """The CLI with a Drude network in the default window: self-consistent rows above the plasma edge, or null."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PCB200_QUIET="1", PYTHONPATH=root)
    out = subprocess.run([sys.executable, os.path.join(root, "tools", "run_bandgap.py"), "16", "bcc_dg", "materials", "4", "2",
                          "--eps", "16,drude:12:0.5", "--energy"], cwd=str(tmp_path), env=env, capture_output=True, text=True,
                         timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    fin = json.load(open(os.path.join(str(tmp_path), line["json"])))
    for i in (0, 1):
        fq = fin["bcc_dg_16_frequencies"][i]
        assert len(fq) == 4 and fq[-1] is not None and all(v is None or v > 0.5 / math.sqrt(12.0) for v in fq)
        assert len(fin["bcc_dg_16_energy_fraction"][i]) == 4


@pytest.mark.gpu
def test_run_bandgap_cli(tmp_path):
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PCB200_QUIET="1", PYTHONPATH=root)
    out = subprocess.run([sys.executable, os.path.join(root, "tools", "run_bandgap.py"), "16", "bcc_dg", "materials", "4", "2",
                          "--eps", "16,lorentz:12:2:2.0", "--window", "0,2.0"], cwd=str(tmp_path), env=env, capture_output=True,
                         text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    fin = json.load(open(os.path.join(str(tmp_path), line["json"])))
    fq = fin["bcc_dg_16_frequencies"][1]
    assert all(v is not None and 0.0 < v < 2.0 for v in fq)
