"""Band group velocities by Hellmann-Feynman: PCB_APPLY_EFOURIER, pcb_band_velocity, group_velocity and the runners' opt-in output.

E^ = IFFT3(M FFT3(K_A^H x)) is AMA before its last K_A (A x = K_A E^).  For d, a, b cyclic and tau_d = dK_d/dalpha_d
(FourierSymbols.dtables), W_d = X^H ((tau_d e_d) x E^) and V_d = W_d + W_d^H = X^H (dA/dalpha_d) X.  References: the NumPy oracle
(oracle/pc_oracle.py: a_block, scipy.fft, the *_handle M's), exact plane-wave eigenvectors of the vacuum operator, and central
differences of solved eigenvalues.  The ``emu`` tests run at small N on the host-emulation build (plane layout at N = 8, 16 and
in the z-split form at 16, natural layout at 6 and 12); the ``gpu`` tests run the sizes users run on the B200.
"""
import os

import numpy as np
import pytest
import scipy.fft as sfft

from test_field_energy import GPU_CASES, _GENERIC, _case_id, _same, _setup, _with_options, emu, gpu  # noqa: F401

_KINDS = [(None, 1), ("chiral", 1), ("pseudochiral_trivial", 1), ("pseudochiral_crossdof", 1), ("pseudochiral_crossdof", 2)]
_EMU_LAYOUTS = [(8, {}), (16, {}), (16, {"plane_split": 1}), (6, {}), (12, {})]
EMU_CASES = [(N, "bcc_sg", typ, k, _GENERIC, opt) for N, opt in _EMU_LAYOUTS for typ, k in _KINDS]


# ---- oracle -------------------------------------------------------------------------------------------------------------
def efourier(X, D_A, diel):
    """Oracle: E^ = ifftn(M(fftn(a_block(X, -conj a)))) of the columns of X."""
    import pc_oracle as oc
    nn3, m = X.shape
    n = round((nn3 // 3) ** (1 / 3))
    w = os.cpu_count() or 1
    D = oc.a_block(X, -D_A.conj()).reshape(n, n, n, 3 * m, order="F")
    D = sfft.fftn(D, axes=(0, 1, 2), workers=w).reshape(nn3, m, order="F")
    E = diel(D).reshape(n, n, n, 3 * m, order="F")
    return sfft.ifftn(E, axes=(0, 1, 2), workers=w).reshape(nn3, m, order="F")


def dsymbol(dtables, N, d):
    """dD/dalpha_d as a symbol vector of a_block: component d holds tau_d[i_d], the others are zero."""
    p = np.arange(N ** 3)
    idx = (p % N, (p // N) % N, p // (N * N))
    out = np.zeros(3 * N ** 3, dtype=np.complex128)
    out[d * N ** 3:(d + 1) * N ** 3] = dtables[d][idx[d]]
    return out


def velocity_matrices(X, Eh, dtables, N):
    """Oracle V_d = W_d + W_d^H, and B_d = 2 sum_q |tau_d| (|x_i,b| |E^_j,a| + |x_i,a| |E^_j,b|), the sum of the magnitudes of
    the terms an entry adds up (its rounding error scale)."""
    import pc_oracle as oc
    V, B = [], []
    for d in range(3):
        ds = dsymbol(dtables, N, d)
        W = X.conj().T @ oc.a_block(Eh, ds)
        V.append(W + W.conj().T)
        n3 = N ** 3
        a, b = (d + 1) % 3, (d + 2) % 3
        t = np.abs(ds[d * n3:(d + 1) * n3])[:, None]
        ax, ae = np.abs(X), np.abs(Eh)
        sl = lambda A, c: A[c * n3:(c + 1) * n3]      # noqa: E731
        B.append(2 * ((sl(ax, b) * t).T @ sl(ae, a) + (sl(ax, a) * t).T @ sl(ae, b)))
    return np.array(V), np.array(B)


def _velocity_rc(pkg, op, X, V, xx, xax):
    L = pkg._lib
    dt = np.ascontiguousarray(op.a_fft.dtables)
    return L.lib().pcb_band_velocity(op.h, X.k, L.ptr_array(X.ptrs), dt.view(np.float64).ctypes.data_as(L.c_double_p),
                                     V.ctypes.data, xx.ctypes.data_as(L.c_double_p), xax.ctypes.data_as(L.c_double_p))


# ---- 1-3: E^ parity, velocity matrices vs the oracle, determinism -------------------------------------------------------
def _check_case(pkg, oc, case, widths=(1, 5, 17, 32)):
    N, d_flag, typ, k, alpha, options = case

    def run(ctx):
        L = pkg._lib
        A_func, a, diel, _ = _setup(pkg, oc, N, d_flag, typ, alpha, k)
        op = A_func.op
        m = max(widths)
        X = ctx.random_block(m, 777 + N)
        x = X.get()
        # 1. E^ vs the oracle; K_A(E^) is A bit for bit; in place refused exactly where A refuses it
        Eh = op.apply(L.APPLY_EFOURIER, X)
        k3, k2 = min(3, m), min(2, m)
        want = efourier(x[:, :k3], a, diel)
        got = Eh.get()
        err = np.linalg.norm(got[:, :k3] - want, axis=0) / np.linalg.norm(want, axis=0)
        assert np.all(err < 1e-12), err
        ka = op.apply(L.APPLY_KA, Eh)
        ax = op.apply(L.APPLY_A, X)
        assert _same(pkg, ax, ka).all()
        ax = op.apply(L.APPLY_A, X)
        for mode in (L.APPLY_A, L.APPLY_EFOURIER):
            Z = X.cols(range(k2)).copy()
            rc = L.lib().pcb_apply(op.h, mode, k2, L.ptr_array(Z.ptrs), L.ptr_array(Z.ptrs))
            if mode == L.APPLY_A:
                rc_a = rc
            else:
                assert rc == rc_a, (rc, rc_a)
                if rc == 0:
                    assert _same(pkg, Eh.cols(range(k2)), Z).all()
                else:
                    assert np.array_equal(Z.get(), x[:, :k2])
        # 2. velocity matrices vs the oracle, xx and xax vs host values.  The oracle runs on columns in every 16 x 16 block
        #    pair of the kernel (0, 15 | 16, 17, 31) -- host memory at N = 160 -- and the widths below tie the rest to them.
        #    Both sides add 2 N^3 terms in FP64 in different orders: beyond 1e-12 max|V_d| (met at the emulated sizes), an entry
        #    may differ by 1e-14 of the sum of its terms' magnitudes B (about 45 eps; measured up to 2.4e-12 max|V_d|, i.e.
        #    ~1e-15 B, at N = 120 ... 256, where B / max|V_d| ~ N^1.5).  One wrong term in N^3 would be ~N^-3 B.
        V, xx, xax = op.band_velocity(X)
        oc_cols = [j for j in (0, 1, 5, 15, 16, 17, 30, 31) if j < m]
        Vo, Bo = velocity_matrices(x[:, oc_cols], got[:, oc_cols], op.a_fft.dtables, N)
        for d in range(3):
            err = np.abs(V[d][oc_cols][:, oc_cols] - Vo[d])
            assert np.all(err <= np.maximum(1e-12 * np.abs(Vo[d]).max(), 1e-14 * Bo[d])), (d, err.max(), np.abs(Vo[d]).max())
            assert np.array_equal(V[d], V[d].conj().T)
        assert np.all(np.abs(xx - (np.abs(x) ** 2).sum(axis=0)) <= 1e-12 * xx)
        xax_host = pkg.pcfft.column_dots(X, ax).real
        assert np.all(np.abs(xax - xax_host) <= 1e-11 * np.abs(xax_host)), (xax, xax_host)
        # 3. widths: a subset's V is the sub-block of the wide call, bit for bit; repeated calls are identical; x is read only
        for w in widths:
            sel = list(range(m - w, m)) if w > 1 else [m // 2]
            Vs, xs, xas = op.band_velocity(X.cols(sel))
            assert np.array_equal(Vs, V[:, sel][:, :, sel]), w
            assert np.array_equal(xs, xx[sel]) and np.array_equal(xas, xax[sel]), w
        again = op.band_velocity(X)
        assert all(np.array_equal(p, q) for p, q in zip(again, (V, xx, xax)))
        assert np.array_equal(X.get(), x)
        hc = [0, m - 1]
        host = op.band_velocity(x[:, hc])
        assert np.array_equal(host[0], V[:, hc][:, :, hc])

    _with_options(pkg, N, options, run)


@pytest.mark.parametrize("case", EMU_CASES, ids=_case_id)
def test_velocity_matrices_emu(emu, oracle, case):
    _check_case(emu, oracle, case)


def test_velocity_matrices_one_column_emu(emu, oracle):
    _check_case(emu, oracle, (16, "sc_curv", "chiral", 1, _GENERIC, {}), widths=(1,))


@pytest.mark.gpu
@pytest.mark.parametrize("case", GPU_CASES, ids=_case_id)
def test_velocity_matrices(gpu, oracle, case):
    _check_case(gpu, oracle, case)


@pytest.mark.gpu
def test_velocity_matrices_n256(gpu, oracle):
    _check_case(gpu, oracle, (256, "sc_curv", "chiral", 1, _GENERIC, {}), widths=(1,))


def _refusals(pkg):
    ctx = pkg.get_context(8)
    mfd = pkg.discretization
    a_fft, _ = mfd.fft_blocks(8, 1, pkg.dielectric.diel_info("sc_curv", option="ct"), alpha=np.array(_GENERIC))
    op = pkg.pcfft.Operator(a_fft, 0.0, 0.0, 0.0, None, ctx=ctx)
    X = ctx.random_block(33, 3)
    V, xx, xax = np.full((3, 33, 33), 7.0 + 7.0j), np.full(33, 7.0), np.full(33, 7.0)
    assert _velocity_rc(pkg, op, X, V, xx, xax) == -2
    assert np.all(V == 7.0 + 7.0j) and np.all(xx == 7.0) and np.all(xax == 7.0)
    slab = pkg.devarray.Context(8, pkg.devarray.default_device(), slab=(0, 4))
    op_s = pkg.pcfft.Operator(a_fft, 0.0, 0.0, 0.0, None, ctx=slab)
    Xs = slab.random_block(2, 5)
    V, xx, xax = np.full((3, 2, 2), 7.0 + 7.0j), np.full(2, 7.0), np.full(2, 7.0)
    assert _velocity_rc(pkg, op_s, Xs, V, xx, xax) == -2
    assert b"slab" in pkg._lib.lib().pcb_last_error()
    assert np.all(V == 7.0 + 7.0j) and np.all(xx == 7.0) and np.all(xax == 7.0)
    with pytest.raises(TypeError, match="pc_mfd_handle"):
        pkg.numerical_experiments.group_velocity(X.cols([0]), lambda v: v)
    # the cached E^ columns are released by trim
    op.band_velocity(X.cols(range(4)))
    assert ctx.trim() >= 4 * ctx.R * 16


def test_refusals_emu(emu):
    _refusals(emu)


@pytest.mark.gpu
def test_refusals(gpu):
    _refusals(gpu)


# ---- 4-5: exact vacuum answers -------------------------------------------------------------------------------------------
def _vacuum(pkg, oc, N, alpha):
    A_func, _, _, _ = _setup(pkg, oc, N, "sc_curv", None, alpha)
    return A_func, A_func.op.a_fft.tables, A_func.op.a_fft.dtables


def _mode(N, tables, q, w):
    """Column with one Fourier coefficient at q and polarisation v = K(q) x w (an exact eigenvector in vacuum, lambda = |K|^2)."""
    K = np.array([tables[c][0][q[0]] + tables[c][1][q[1]] + tables[c][2][q[2]] for c in range(3)])
    v = np.cross(K, np.asarray(w, dtype=np.complex128))
    x = np.zeros(3 * N ** 3, dtype=np.complex128)
    p = q[0] + N * q[1] + N * N * q[2]
    for c in range(3):
        x[c * N ** 3 + p] = v[c]
    return x, K, v


def _exact_vacuum(pkg, oc, N):
    A_func, T, dt = _vacuum(pkg, oc, N, _GENERIC)
    op = A_func.op
    qs = [(1, 2, 0), (N - 1, 0, 3 % N), (2, N - 2, 1)]
    cols, want, lam = [], [], []
    for q, w in zip(qs, ([0.3, -1.0, 0.5], [1.0, 0.2, -0.7], [-0.4, 0.9, 1.1])):
        x, K, v = _mode(N, T, q, w)
        cols.append(x)
        lam.append(np.vdot(K, K).real)
        want.append([2 * (np.conj(K[d]) * dt[d][q[d]]).real * np.vdot(v, v).real for d in range(3)])
    X = np.stack(cols, axis=1)
    V, xx, xax = op.band_velocity(X)
    want = np.array(want)
    for j in range(len(qs)):
        for d in range(3):
            assert abs(V[d, j, j].real - want[j, d]) <= 1e-12 * np.abs(want[j]).max(), (j, d)
    off = np.abs(V - V * np.eye(len(qs))[None]).max()
    assert off <= 1e-12 * np.abs(V).max()
    lam = np.array(lam)
    assert np.allclose(xax / xx, lam, rtol=1e-12, atol=0)
    # group_velocity without a direction: the analytic gradients of the modes
    g = pkg.numerical_experiments.group_velocity(X, A_func)
    assert np.allclose(g, want / xx[:, None] / (2 * np.sqrt(lam))[:, None], rtol=1e-10, atol=1e-14)


@pytest.mark.parametrize("N", [8, 16, 6, 12])
def test_exact_vacuum_emu(emu, oracle, N):
    _exact_vacuum(emu, oracle, N)


def test_exact_vacuum_split_emu(emu, oracle):
    _with_options(emu, 16, {"plane_split": 1}, lambda ctx: _exact_vacuum(emu, oracle, 16))


@pytest.mark.gpu
@pytest.mark.parametrize("N", [120, 160, 256])
def test_exact_vacuum(gpu, oracle, N):
    _exact_vacuum(gpu, oracle, N)


def _degenerate(pkg, oc, N):
    """Vacuum sc at alpha = (0.3 pi, 0, 0): the modes +-e_y and +-e_z, two polarisations each, are one degenerate cluster of 8;
    along u = e_y it splits into +v (2), -v (2) and 0 (4)."""
    ne = pkg.numerical_experiments
    A_func, T, dt = _vacuum(pkg, oc, N, [0.3 * np.pi, 0.0, 0.0])
    qs = [(0, 1, 0), (0, N - 1, 0), (0, 0, 1), (0, 0, N - 1)]
    cols, vel = [], []
    for q in qs:
        for w in ([1.0, 0.0, 0.0], [0.0, 0.3, 1.0] if q[1] else [0.0, 1.0, 0.3]):
            x, K, v = _mode(N, T, q, w)
            cols.append(x)
            lam = np.vdot(K, K).real
            vel.append(2 * (np.conj(K[1]) * dt[1][q[1]]).real / (2 * np.sqrt(lam)))
    X0 = np.stack(cols, axis=1)
    rng = np.random.default_rng(3)
    Q, _ = np.linalg.qr(rng.standard_normal((8, 8)) + 1j * rng.standard_normal((8, 8)))
    X = X0 @ Q                                  # a basis of the cluster that is not the modes
    vel = np.sort(vel)
    assert vel[-1] > 1e-3 and abs(vel[3]) < 1e-12
    up = ne.group_velocity(X, A_func, direction=[0.0, 2.0, 0.0], side=+1)
    down = ne.group_velocity(X, A_func, direction=[0.0, 1.0, 0.0], side=-1)
    scale = np.abs(vel).max()
    assert np.abs(up - vel).max() <= 1e-10 * scale, (up, vel)
    assert np.abs(down - vel[::-1]).max() <= 1e-10 * scale, (down, vel)
    # without a direction the cluster reports its trace average (basis independent)
    g = ne.group_velocity(X, A_func)
    g0 = ne.group_velocity(X0, A_func)
    assert np.allclose(g, g[0]) and np.allclose(g, g0, rtol=1e-10, atol=1e-14)
    # at a generic k-point every band's vector is the analytic gradient of its mode
    A_func, T, dt = _vacuum(pkg, oc, N, _GENERIC)
    cols, want = [], []
    for q in [(1, 0, 0), (0, 2, 1), (N - 1, 1, 2)]:
        x, K, v = _mode(N, T, q, [0.2, -0.5, 1.0])
        cols.append(x)
        lam = np.vdot(K, K).real
        want.append([2 * (np.conj(K[d]) * dt[d][q[d]]).real / (2 * np.sqrt(lam)) for d in range(3)])
    g = ne.group_velocity(np.stack(cols, axis=1), A_func)
    assert np.allclose(g, np.array(want), rtol=1e-10, atol=1e-14)


def test_degenerate_clusters_emu(emu, oracle):
    _degenerate(emu, oracle, 8)


@pytest.mark.gpu
def test_degenerate_clusters(gpu, oracle):
    _degenerate(gpu, oracle, 120)


# ---- 6: Hellmann-Feynman against finite differences ---------------------------------------------------------------------
def _hf_fd(pkg, N, d_flag, typ, tol):
    ne, mfd = pkg.numerical_experiments, pkg.discretization
    alpha, nev, h = np.array(_GENERIC), 6, 1e-3
    u = np.array([0.6, -0.8, 0.0])
    res = ne.eigen_1p(N, d_flag, alpha, type=typ, nev=nev, seed=11, tol=tol)
    a_fft, b_fft, inv_fft, _, shift = ne.uniform_initialization(N, d_flag, alpha, nev=nev, seed=11)
    A_func = ne.pc_mfd_handle(a_fft, b_fft, ne._handle(typ, N, d_flag), inv_fft, shift)[0]
    vel = ne.group_velocity(res["x"][:, :nev], A_func, direction=u)
    om = 2 * np.pi * np.asarray(res["omega_re"])
    wp, wm = [2 * np.pi * np.asarray(ne.eigen_1p(N, d_flag, alpha + s * h * u, type=typ, nev=nev, x0=res["x"].copy(),
                                                  tol=tol)["omega_re"]) for s in (1, -1)]
    fd = (wp - wm) / (2 * h)
    lam = om ** 2
    gaps = np.diff(lam)
    checked = 0
    for i in range(nev):
        lo = gaps[i - 1] if i > 0 else np.inf
        hi = gaps[i] if i < nev - 1 else np.inf
        if min(lo, hi) > 1e-2 * lam[i] and lam[i] > 1e-6:
            assert abs(fd[i] - vel[i]) <= max(1e-4 * abs(vel[i]), 1e-6 * lam[i]), (i, fd[i], vel[i])
            checked += 1
    assert checked >= 2, (lam, vel)


@pytest.mark.parametrize("d_flag,typ", [("sc_curv", "chiral"), ("bcc_sg", "pseudochiral_crossdof")])
def test_hellmann_feynman_emu(emu, d_flag, typ):
    _hf_fd(emu, 8, d_flag, typ, 1e-9)


@pytest.mark.gpu
@pytest.mark.parametrize("d_flag,typ", [("sc_curv", "chiral"), ("bcc_sg", "pseudochiral_crossdof")])
def test_hellmann_feynman(gpu, d_flag, typ):
    _hf_fd(gpu, 48, d_flag, typ, 1e-8)


# ---- 7: runners ------------------------------------------------------------------------------------------------------------
def _runners(pkg, N, tmp_path):
    import json
    ne = pkg.numerical_experiments
    d_flag, nev = "sc_curv", 5
    n_k = pkg.dielectric.kpath(d_flag, ne.GAP).shape[0]
    idx = [0, 1, n_k - 1]                       # the sc path ends at Gamma
    key_it, key_fq, key_v = f"{d_flag}_{N}_iterations", f"{d_flag}_{N}_frequencies", f"{d_flag}_{N}_group_velocity"
    p_on, p_off = str(tmp_path / "on.json"), str(tmp_path / "off.json")
    assert ne.bandgap(N, d_flag, type="chiral", indices=idx, nev=nev, seed=31, path=p_on, velocity=True) == []
    assert "velocity" in ne.bandgap.last_timing
    assert ne.bandgap(N, d_flag, type="chiral", indices=idx, nev=nev, seed=31, path=p_off) == []
    assert "velocity" not in ne.bandgap.last_timing
    on, off = json.load(open(p_on)), json.load(open(p_off))
    assert key_v not in off and set(off) == {key_it, key_fq}
    for i in idx:
        assert on[key_fq][i] == off[key_fq][i]
        assert len(on[key_v][i]) == nev
    assert on[key_v][n_k - 1][:2] == [None, None]          # the zero modes at Gamma
    assert all(v is not None for v in on[key_v][0]) and all(v is not None for v in on[key_v][1])
    assert all(on[key_v][i] == [0] * nev for i in range(n_k) if i not in idx)
    # the row of a point is group_velocity along its segment, from the segment's start side
    sym = pkg.dielectric.diel_info(d_flag, "sym").astype(float)
    alpha = pkg.dielectric.kpath(d_flag, ne.GAP)[1]
    r = ne.eigen_1p(N, d_flag, alpha, type="chiral", nev=nev, seed=5, velocity=True)
    a_fft, b_fft, inv_fft, _, shift = ne.uniform_initialization(N, d_flag, alpha, nev=nev, seed=5)
    A_func = ne.pc_mfd_handle(a_fft, b_fft, pkg.discretization.chiral_handle(N, d_flag), inv_fft, shift)[0]
    assert np.array_equal(r["group_velocity"], ne.group_velocity(r["x"][:, :nev], A_func), equal_nan=True)
    assert r["velocity_cluster"].shape == (nev,)
    assert "group_velocity" not in ne.eigen_1p(N, d_flag, alpha, type="chiral", nev=nev, seed=5)
    along = ne.group_velocity(r["x"][:, :nev], A_func, direction=sym[1] - sym[0], side=-1)
    assert np.allclose(along, on[key_v][1], rtol=1e-4, atol=1e-6)
    # resume: rows written without velocities are recomputed and get them
    assert ne.bandgap(N, d_flag, type="chiral", nev=nev, seed=31, path=p_off, only=idx, velocity=True) == []
    res = json.load(open(p_off))
    for i in idx:
        assert res[key_v][i] == on[key_v][i]
        assert res[key_fq][i] == on[key_fq][i]
    # k-path sharding (world size 1): the velocity rows are merged into the final file
    out_dir = str(tmp_path / "sharded") + "/"
    rows = ne.bandgap_sharded(N, d_flag, 0, 1, type="chiral", nev=nev, seed=31, out_dir=out_dir, indices=idx,
                              gather=lambda o: [o], velocity=True)
    assert set(rows["group_velocity"]) == set(idx)
    fin = json.load(open(os.path.join(out_dir, f"bandgap_{d_flag}.json")))
    for i in idx:
        assert fin[key_v][i] == rows["group_velocity"][i]
    assert len(ne.merge_records([{"iterations": {}, "frequencies": {}}], n_k, nev)) == 2
    merged = ne.merge_records([{"iterations": {}, "frequencies": {}, "group_velocity": {1: [0.5] * nev}}], n_k, nev)
    assert len(merged) == 4 and merged[2] is None and merged[3][1] == [0.5] * nev


def test_runners_emu(emu, tmp_path):
    _runners(emu, 8, tmp_path)


@pytest.mark.gpu
def test_runners(gpu, tmp_path):
    _runners(gpu, 48, tmp_path)


@pytest.mark.gpu
def test_run_bandgap_cli(tmp_path):
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PCB200_QUIET="1", PYTHONPATH=root)
    out = subprocess.run([sys.executable, os.path.join(root, "tools", "run_bandgap.py"), "16", "sc_curv", "chiral", "4", "2",
                          "--velocity"], cwd=str(tmp_path), env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    fin = json.load(open(os.path.join(str(tmp_path), line["json"])))
    assert all(v is not None for v in fin["sc_curv_16_group_velocity"][0])
