"""Electric energy of modes in the dielectric: pcb_field_energy, the D / E field modes of pcb_apply and the runners' opt-in output.

For a column x, D = FFT3(K_A^H x) (unnormalised), E = M D, rows r = c N^3 + p:
    e_tot = Re sum_r conj(D_r) E_r / N^3 (= x^H A x),   e_in = the same sum over the rows of ind_e (edge DoFs in Omega_1),
and f = e_in / e_tot.  References: the NumPy oracle (oracle/pc_oracle.py: a_block, scipy.fft.fftn, the *_handle M's) and host
sums.  The ``emu`` tests run every check at small N on the host-emulation build (plane layout at N = 8, 16 and in the z-split
form at 16, natural layout at 6 and 12); the ``gpu`` tests run the sizes users run on the B200.
"""
import ctypes as C
import importlib
import os

import numpy as np
import pytest
import scipy.fft as sfft

from conftest import PKG

_GENERIC = [0.3 * np.pi, 0.2 * np.pi, 0.1 * np.pi]
_NEAR_GAMMA = [np.pi / 20, 0.0, 0.0]
_DEFAULT_OPTIONS = {"plane": 1, "plane_cross": 1, "plane_split": 0}


def _bind(request, which):
    pkg = importlib.import_module(PKG)
    pkg._lib.use_library(request.getfixturevalue("emu_lib" if which == "emu" else "cuda_lib"))
    if which == "cuda":
        assert pkg.backend() == "cuda-sm_100a"
    pkg.backend_name = which
    return pkg


@pytest.fixture
def emu(request):
    pkg = _bind(request, "emu")
    yield pkg
    pkg.devarray.drop_contexts()
    pkg.lobpcg._helpers.clear()


@pytest.fixture
def gpu(request):
    pkg = _bind(request, "cuda")
    yield pkg
    pkg.devarray.drop_contexts()
    pkg.lobpcg._helpers.clear()
    import gc
    gc.collect()
    for ctx in list(pkg.devarray._contexts.values()):
        ctx.trim()


# ---- oracle -------------------------------------------------------------------------------------------------------------
def field_energy(X, D_A, diel, ind_e):
    """Oracle: (D, E, e_in, e_tot) of the columns of X by the definitions (host NumPy / scipy)."""
    import pc_oracle as oc
    nn3, m = X.shape
    n = round((nn3 // 3) ** (1 / 3))
    D = oc.a_block(X, -D_A.conj()).reshape(n, n, n, 3 * m, order="F")
    D = sfft.fftn(D, axes=(0, 1, 2), workers=os.cpu_count() or 1).reshape(nn3, m, order="F")
    E = diel(D)
    t = (D.conj() * E).real / n ** 3
    return D, E, t[ind_e].sum(axis=0), t.sum(axis=0)


def _setup(pkg, oc, N, d_flag, typ, alpha, k=1):
    """Device operator (the A_func of pc_mfd_handle) and the oracle's (a_fft, M, ind_e) for one case."""
    mfd, ne = pkg.discretization, pkg.numerical_experiments
    alpha = np.asarray(alpha, dtype=float)
    relax, pnt = mfd.set_relaxation(alpha)
    a_fft, b_fft = mfd.fft_blocks(N, 1, pkg.dielectric.diel_info(d_flag, option="ct"), alpha=alpha)
    inv_fft = mfd.inverse_3_times_3_B(b_fft, pnt, relax[0])
    kw = {"k": k} if typ == "pseudochiral_crossdof" else {}
    Diels = None if typ is None else getattr(mfd, typ + "_handle")(N, d_flag, **kw)
    A_func = ne.pc_mfd_handle(a_fft, (pnt * b_fft[0], pnt * b_fft[1]), Diels, inv_fft, relax[0])[0]
    a, _, _, _, _ = oc.assemble_symbols(N, d_flag, alpha)
    if typ is None:
        return A_func, a, (lambda v: v), np.zeros(0, dtype=np.int64)
    ind_e = pkg.dielectric.compute_index(N, d_flag, "edge")
    okw = {"ind_e": ind_e}
    if typ == "pseudochiral_trivial":
        okw["ind_v"] = pkg.dielectric.compute_index(N, d_flag, "volume")
    if typ == "pseudochiral_crossdof":
        okw["k"] = k
    return A_func, a, oc.HANDLES[typ](N, d_flag, **okw), ind_e


def _energy_rc(pkg, op, X, e_in, e_tot):
    return pkg._lib.lib().pcb_field_energy(op.h, X.k, pkg._lib.ptr_array(X.ptrs), e_in.ctypes.data_as(pkg._lib.c_double_p),
                                           e_tot.ctypes.data_as(pkg._lib.c_double_p))


def _same(pkg, A, B):
    """Per column: A_j == B_j bit for bit; B is overwritten with A - B."""
    L = pkg._lib
    L.check(L.lib().pcb_axpby(A.ctx.h, A.k, L.ptr_array(A.ptrs), L.ptr_array(B.ptrs), 1.0, -1.0), "pcb_axpby")
    return pkg.pcfft.column_norms(B) == 0.0


def _rel(got, want, floor):
    return np.abs(got - want) / np.maximum(np.abs(want), floor)


def _plane_layout(N, options):
    """A / H run on the plane layout: N % 8 == 0 up to N = 160 (whole or half planes), unless the plane mode is switched off."""
    return options.get("plane", 1) != 0 and N % 8 == 0 and N <= 160


def _with_options(pkg, N, options, fn):
    ctx = pkg.get_context(N)
    try:
        for k, v in options.items():
            ctx.option(k, v)
        return fn(ctx)
    finally:
        for k in options:
            ctx.option(k, _DEFAULT_OPTIONS[k])


# ---- parity, field modes and identities ------------------------------------------------------------------------------------
def _check_case(pkg, oc, case, ncols=3, widths=True):
    N, d_flag, typ, k, alpha, options = case

    def run(ctx):
        L = pkg._lib
        A_func, a, diel, ind_e = _setup(pkg, oc, N, d_flag, typ, alpha, k)
        op = A_func.op
        X = ctx.random_block(ncols, 4242 + N)
        x = X.get()
        e_in, e_tot = op.field_energy(X)
        D, E, w_in, w_tot = field_energy(x, a, diel, ind_e)
        scale = np.abs(w_tot)
        # 1. parity with the oracle
        assert np.all(_rel(e_tot, w_tot, 0) < 1e-11), (e_tot, w_tot)
        assert np.all(np.abs(e_in - w_in) / scale < 1e-11), (e_in, w_in)
        # 2. field modes D / E vs the oracle; in place equals out of place (no mode refuses an aliased column)
        Y = ctx.empty(ncols)
        for mode, want, tag in ((L.APPLY_DFIELD, D, "D"), (L.APPLY_EFIELD, E, "E")):
            op.apply_into(mode, X, Y)
            got = Y.get()
            err = np.linalg.norm(got - want, axis=0) / np.linalg.norm(want, axis=0)
            assert np.all(err < 1e-12), (tag, err)
            field = pkg.numerical_experiments.mode_fields(X, A_func, which=tag).get()
            assert np.array_equal(field, got), tag
            Z = X.copy()
            assert pkg._lib.lib().pcb_apply(op.h, mode, ncols, L.ptr_array(Z.ptrs), L.ptr_array(Z.ptrs)) == 0, tag
            assert _same(pkg, Y, Z).all(), (tag, "in place")
            if tag == "D":
                d_host = got
            else:
                e_host = got
        # 3. identities: e_tot = Re x^H A x, e_in = host sum over ind_e of the downloaded fields, e_in = 0 in vacuum, 0 <= f <= 1
        ax = A_func(X)
        xax = pkg.pcfft.column_dots(X, ax).real
        assert np.all(_rel(e_tot, xax, 0) < 1e-11), (e_tot, xax)
        host_in = (d_host[ind_e].conj() * e_host[ind_e]).real.sum(axis=0) / N ** 3
        assert np.all(np.abs(e_in - host_in) / scale < 1e-11), (e_in, host_in)
        if typ is None:
            assert np.all(e_in == 0.0)
        f = pkg.numerical_experiments.energy_fraction(X, A_func)
        assert np.array_equal(f, e_in / e_tot)
        if typ in (None, "chiral"):
            assert np.all((f >= 0.0) & (f <= 1.0)), f
        # 4. x is read only; a repeated call gives the same bits; a host array is uploaded
        assert np.array_equal(X.get(), x)
        n0 = ctx.launches()
        again = op.field_energy(X)
        assert np.array_equal(again[0], e_in) and np.array_equal(again[1], e_tot)
        # the forward half of A's layout (x forward + forward plane half, or x, y and z forward), the energy kernel, the sum
        assert ctx.launches() - n0 == (2 if _plane_layout(N, options) else 3) + 2, ctx.launches() - n0
        host = op.field_energy(x[:, :1])
        assert host[0][0] == e_in[0] and host[1][0] == e_tot[0]
        if widths:
            _check_widths(pkg, op, ctx)

    _with_options(pkg, N, options, run)


def _check_widths(pkg, op, ctx, k=33):
    """A 33-column call (two launch chunks) gives every column the bits of its single-column call."""
    X = ctx.random_block(k, 99)
    e_in, e_tot = op.field_energy(X)
    for j in range(k):
        s_in, s_tot = op.field_energy(X.cols([j]))
        assert s_in[0] == e_in[j] and s_tot[0] == e_tot[j], j
    part = op.field_energy(X.cols(range(5, 9)))
    assert np.array_equal(part[0], e_in[5:9]) and np.array_equal(part[1], e_tot[5:9])


_KINDS = [(None, 1), ("chiral", 1), ("pseudochiral_trivial", 1), ("pseudochiral_crossdof", 1), ("pseudochiral_crossdof", 2)]
_EMU_LAYOUTS = [(8, {}), (16, {}), (16, {"plane_split": 1}), (6, {}), (12, {})]
EMU_CASES = [(N, "bcc_sg", typ, k, alpha, opt) for N, opt in _EMU_LAYOUTS for typ, k in _KINDS for alpha in (_GENERIC, _NEAR_GAMMA)]
GPU_CASES = [
    (120, "fcc", "chiral", 1, _GENERIC, {}),                                   # whole planes
    (120, "bcc_sg", "pseudochiral_trivial", 1, _NEAR_GAMMA, {}),               # slot mask of the cluster form
    (120, "bcc_sg", "pseudochiral_crossdof", 1, _GENERIC, {"plane_cross": 1}),
    (120, "bcc_sg", "pseudochiral_crossdof", 1, _GENERIC, {"plane_cross": 2}),
    (120, "fcc", "chiral", 1, _GENERIC, {"plane": 0}),                         # natural layout at 120
    (96, "sc_curv", "chiral", 1, _GENERIC, {"plane_split": 0}),
    (96, "sc_curv", "chiral", 1, _GENERIC, {"plane_split": 1}),                # half planes
    (128, "bcc_dg", "pseudochiral_crossdof", 1, _GENERIC, {}),
    (160, "bcc_dg", "pseudochiral_crossdof", 1, _GENERIC, {}),
    (160, "bcc_dg", "chiral", 1, _GENERIC, {}),
    (150, "sc_curv", "chiral", 1, _GENERIC, {}),                              # natural layout
    (150, "bcc_sg", "pseudochiral_crossdof", 1, _GENERIC, {}),
    (120, "sc_curv", None, 1, _GENERIC, {}),
]


def _case_id(c):
    opt = "".join(f"-{k}{v}" for k, v in c[5].items())
    kk = f"-k{c[3]}" if c[2] == "pseudochiral_crossdof" else ""
    al = "-nearG" if c[4] is _NEAR_GAMMA else ""
    return f"N{c[0]}-{c[1]}-{c[2] or 'vacuum'}{kk}{al}{opt}"


@pytest.mark.parametrize("case", EMU_CASES, ids=_case_id)
def test_field_energy_emu(emu, oracle, case):
    _check_case(emu, oracle, case, widths=(case[4] is _GENERIC))


@pytest.mark.gpu
@pytest.mark.parametrize("case", GPU_CASES, ids=_case_id)
def test_field_energy(gpu, oracle, case):
    _check_case(gpu, oracle, case, widths=case[0] in (120, 150, 160) and case[5].get("plane_cross") != 2)


@pytest.mark.gpu
def test_field_energy_n256(gpu, oracle):
    _check_case(gpu, oracle, (256, "sc_curv", "chiral", 1, _GENERIC, {}), ncols=1, widths=False)


def _slab_refused(pkg):
    mfd = pkg.discretization
    a_fft, _ = mfd.fft_blocks(8, 1, pkg.dielectric.diel_info("sc_curv", option="ct"), alpha=np.array(_GENERIC))
    slab = pkg.devarray.Context(8, pkg.devarray.default_device(), slab=(0, 4))
    op = pkg.pcfft.Operator(a_fft, 0.0, 0.0, 0.0, None, ctx=slab)
    X = slab.random_block(2, 5)
    e_in, e_tot = np.full(2, 7.0), np.full(2, 7.0)
    assert _energy_rc(pkg, op, X, e_in, e_tot) == -2
    assert b"slab" in pkg._lib.lib().pcb_last_error()
    assert np.all(e_in == 7.0) and np.all(e_tot == 7.0)


def test_slab_context_refused_emu(emu):
    _slab_refused(emu)


@pytest.mark.gpu
def test_slab_context_refused(gpu):
    _slab_refused(gpu)


def test_non_operator_callable_rejected_emu(emu):
    ne = emu.numerical_experiments
    x = emu.get_context(8).random_block(1, 1)
    with pytest.raises(TypeError, match="pc_mfd_handle"):
        ne.energy_fraction(x, lambda v: v)
    with pytest.raises(TypeError, match="pc_mfd_handle"):
        ne.mode_fields(x, lambda v: v)


# ---- physics: Hellmann-Feynman --------------------------------------------------------------------------------------------
def _hellmann_feynman(pkg, N):
    """Chiral M = 1/eps on Omega_1: dlambda/deps = -lambda f / eps.  Central difference of lambda_re over eps (1 +- 1e-3), the
    +- solves warm-started from the eps solution, against -lambda_re f / eps for every band separated from its neighbours."""
    ne = pkg.numerical_experiments
    d_flag, alpha, nev = "sc_curv", np.array(_GENERIC), 6
    eps = pkg.dielectric.diel_chiral_const(d_flag)
    res = ne.eigen_1p(N, d_flag, alpha, type="chiral", nev=nev, seed=11, tol=1e-7, eps_opt=eps, energy=True)
    lam = (2 * np.pi * np.asarray(res["omega_re"])) ** 2
    f = res["energy_fraction"]
    h = 1e-3 * eps
    lp, lm = [(2 * np.pi * np.asarray(ne.eigen_1p(N, d_flag, alpha, type="chiral", nev=nev, x0=res["x"].copy(), tol=1e-7,
                                                    eps_opt=e)["omega_re"])) ** 2 for e in (eps + h, eps - h)]
    fd = (lp - lm) / (2 * h)
    hf = -lam * f / eps
    gaps = np.diff(lam)
    checked = 0
    for i in range(nev):
        lo = gaps[i - 1] if i > 0 else np.inf
        hi = gaps[i] if i < nev - 1 else np.inf
        if min(lo, hi) > 1e-2 * lam[i] and lam[i] > 1e-6:
            assert abs(fd[i] - hf[i]) <= 1e-4 * abs(hf[i]), (i, fd[i], hf[i])
            checked += 1
    assert checked >= 2, (lam, f)


def test_hellmann_feynman_emu(emu):
    _hellmann_feynman(emu, 8)


@pytest.mark.gpu
def test_hellmann_feynman(gpu):
    _hellmann_feynman(gpu, 48)


# ---- runners ---------------------------------------------------------------------------------------------------------------
def _runners(pkg, N, tmp_path):
    import json
    ne = pkg.numerical_experiments
    d_flag, nev, idx = "sc_curv", 5, [0, 1, 2]
    key_it, key_fq, key_en = f"{d_flag}_{N}_iterations", f"{d_flag}_{N}_frequencies", f"{d_flag}_{N}_energy_fraction"
    p_on, p_off = str(tmp_path / "on.json"), str(tmp_path / "off.json")
    assert ne.bandgap(N, d_flag, type="chiral", indices=idx, nev=nev, seed=31, path=p_on, energy=True) == []
    assert "energy" in ne.bandgap.last_timing
    assert ne.bandgap(N, d_flag, type="chiral", indices=idx, nev=nev, seed=31, path=p_off) == []
    assert "energy" not in ne.bandgap.last_timing
    on, off = json.load(open(p_on)), json.load(open(p_off))
    assert key_en not in off and set(off) == {key_it, key_fq}
    for i in idx:
        assert on[key_fq][i] == off[key_fq][i]
        assert on[key_it][i][0] == off[key_it][i][0]
        assert len(on[key_en][i]) == nev and all(0.0 < v < 1.0 for v in on[key_en][i])
    n_k = len(on[key_it])
    assert all(on[key_en][i] == [0] * nev for i in range(n_k) if i not in idx)
    # resume: rows written without energies are recomputed and get them
    assert ne.bandgap(N, d_flag, type="chiral", nev=nev, seed=31, path=p_off, only=idx, energy=True) == []
    res = json.load(open(p_off))
    for i in idx:
        assert res[key_en][i] == on[key_en][i]
        assert res[key_fq][i] == on[key_fq][i]
    # k-path sharding (world size 1): the energy rows are merged into the final file
    out_dir = str(tmp_path / "sharded") + "/"
    rows = ne.bandgap_sharded(N, d_flag, 0, 1, type="chiral", nev=nev, seed=31, out_dir=out_dir, indices=idx,
                              gather=lambda o: [o], energy=True)
    assert set(rows["energy_fraction"]) == set(idx)
    fin = json.load(open(os.path.join(out_dir, f"bandgap_{d_flag}.json")))
    for i in idx:
        assert fin[key_en][i] == rows["energy_fraction"][i]
    merged = ne.merge_records([{"iterations": {}, "frequencies": {}}], n_k, nev)
    assert len(merged) == 2
    # eigen_1p(energy=True): the fractions of energy_fraction on its x
    alpha = np.array(_GENERIC)
    r = ne.eigen_1p(N, d_flag, alpha, type="chiral", nev=nev, seed=5, energy=True)
    mfd = pkg.discretization
    a_fft, b_fft, inv_fft, _, shift = ne.uniform_initialization(N, d_flag, alpha, nev=nev, seed=5)
    A_func = ne.pc_mfd_handle(a_fft, b_fft, mfd.chiral_handle(N, d_flag), inv_fft, shift)[0]
    assert np.array_equal(r["energy_fraction"], ne.energy_fraction(r["x"][:, :nev], A_func))
    assert "energy_fraction" not in ne.eigen_1p(N, d_flag, alpha, type="chiral", nev=nev, seed=5)


def test_runners_emu(emu, tmp_path):
    _runners(emu, 8, tmp_path)


@pytest.mark.gpu
def test_runners(gpu, tmp_path):
    _runners(gpu, 48, tmp_path)
