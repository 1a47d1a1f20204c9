"""The operator and the block kernels at the block widths and row counts the solver produces.

The solver applies H to m = nev + round(0.6 nev) columns and to W_act of any width 1..m, and the dense phase runs on
slabs of any height in the large-grid mode.  The kernels split work by width and by rows in ways the narrow, tile-aligned
shapes of the other tests never reach:

  * pcb_apply splits a call into launches of PCB_MAXC = 32 columns, and the persistent plane / z-mid / cluster kernels deal
    (column, component, line[, half]) items over a fixed grid, so what a CTA gets depends on the width;
  * the block kernels have pipeline prologues (k_update: 2-3 stages, k_update_res: a named-barrier handshake that starts
    waiting at the third tile of a CTA) that behave differently when a CTA gets 1, 2 or 3 row tiles, and partial last
    tiles whenever R is not a multiple of the tile height (N = 150: 22 500 cells per plane, = 4 mod 16);
  * pcb_apply_host moves a block in chunks of 8 columns through two staging slots that are reused behind events.

References: the NumPy oracle (oracle/pc_oracle.py), scipy.fft and complex128 NumPy products.  The ``emu`` tests run the
same checks at small N on the host-emulation build; the ``gpu`` tests run the sizes the solver uses on the B200.
"""
import ctypes as C
import importlib
import os

import numpy as np
import pytest

from conftest import PKG

STRUCT_PLANE, STRUCT_CROSS_PLANE, STRUCT_FIVE, STRUCT_CROSS7 = "plane", "cross-plane", "five", "cross7"


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
        ctx.trim()          # hand GB-sized cached blocks back between the tests (shared device)


def _sms(pkg):
    if pkg.backend_name == "emu":
        return 2                                    # pcb_ctx_create of the emulation build
    import torch
    return torch.cuda.get_device_properties(pkg.devarray.default_device()).multi_processor_count


# ---- device-side helpers ----------------------------------------------------------------------------------------------
def _axpby(pkg, X, Y, a, b):
    L = pkg._lib
    L.check(L.lib().pcb_axpby(X.ctx.h, X.k, L.ptr_array(X.ptrs), L.ptr_array(Y.ptrs), float(a), float(b)), "pcb_axpby")


def _same(pkg, A, B):
    """Per column: A_j == B_j bit for bit (up to the sign of zeros).  B <- A - B on the device (B is overwritten), and a
    difference of finite doubles is exactly zero only for equal operands; NaN / Inf give a non-zero (NaN) norm."""
    _axpby(pkg, A, B, 1.0, -1.0)
    return pkg.pcfft.column_norms(B) == 0.0


def _apply_rc(pkg, op, mode, X, Y):
    return pkg._lib.lib().pcb_apply(op.h, mode, X.k, pkg._lib.ptr_array(X.ptrs), pkg._lib.ptr_array(Y.ptrs))


def _apply_timed(pkg, op, mode, X, Y):
    """pcb_apply_timed: (return code, number of kernels timed)."""
    ms, n = (C.c_float * 8)(), C.c_int()
    rc = pkg._lib.lib().pcb_apply_timed(op.h, mode, X.k, pkg._lib.ptr_array(X.ptrs), pkg._lib.ptr_array(Y.ptrs), ms, C.byref(n))
    return rc, n.value


def _colerr(got, want):
    return np.linalg.norm(got - want, axis=0) / np.linalg.norm(want, axis=0)


# ---- operators ----------------------------------------------------------------------------------------------------
def _ops(pkg, N, d_flag, alpha, typ, eps_opt=0):
    mfd, ne = pkg.discretization, pkg.numerical_experiments
    relax, pnt = mfd.set_relaxation(alpha)
    a_fft, b_fft = mfd.fft_blocks(N, 1, pkg.dielectric.diel_info(d_flag, option="ct"), alpha=alpha)
    inv_fft = mfd.inverse_3_times_3_B(b_fft, pnt, relax[0])
    Diels = None if typ is None else getattr(mfd, typ + "_handle")(N, d_flag, eps_opt=eps_opt)
    return ne.pc_mfd_handle(a_fft, (pnt * b_fft[0], pnt * b_fft[1]), Diels, inv_fft, relax[0])[1].op


def _oracle(pkg, oc, N, d_flag, alpha, typ, eps_opt=0):
    """(symbols a, b, inv, shift, M) of the oracle; index sets from the product's geometry code, which equals the oracle's
    dense evaluation bit for bit (test_index_sets_n120, test_device_geometry_matches_host) and is much faster at large N."""
    oc.FFT_WORKERS = os.cpu_count() or 1
    a, b, inv, shift, _ = oc.assemble_symbols(N, d_flag, alpha)
    if typ is None:
        diel = lambda v: v      # noqa: E731
    else:
        kw = {"ind_e": pkg.dielectric.compute_index(N, d_flag, "edge")}
        if typ == "pseudochiral_trivial":
            kw["ind_v"] = pkg.dielectric.compute_index(N, d_flag, "volume")
        diel = oc.HANDLES[typ](N, d_flag, eps_opt=eps_opt, **kw)
    return a, b, inv, shift, diel


def _oracle_AH(oc, sym, x):
    a, b, inv, shift, diel = sym
    ax = oc.AMA(x, a, diel)
    return ax, ax + oc.h_block(x, b) + shift * x       # = oc.AMA_BB without a second AMA


# (N, lattice, dielectric, alpha, context options, pass structure of A / H)
_ALPHA_FCC = [0.3 * np.pi, 2 * np.pi, 0.0]
GPU_CASES = [
    (120, "fcc", None, _ALPHA_FCC, {}, STRUCT_PLANE),
    (120, "fcc", "chiral", _ALPHA_FCC, {}, STRUCT_PLANE),                               # five-sweep plane pass k_mid2
    (120, "fcc", "chiral", _ALPHA_FCC, {"mid_five": 0}, STRUCT_PLANE),                  # seven-sweep TMA plane pass
    (120, "bcc_sg", "pseudochiral_trivial", [np.pi / 20, 0.0, 0.0], {}, STRUCT_PLANE),  # coupled M on clusters of 3 CTAs
    (120, "bcc_sg", "pseudochiral_crossdof", [np.pi, 0.5 * np.pi, 0.0], {"plane_cross": 1}, STRUCT_CROSS_PLANE),
    (120, "bcc_sg", "pseudochiral_crossdof", [np.pi, 0.5 * np.pi, 0.0], {"plane_cross": 2}, STRUCT_CROSS_PLANE),
    (160, "sc_curv", None, [np.pi, 0.4, 0.0], {}, STRUCT_PLANE),                        # z-split half planes
    (160, "fcc", "chiral", _ALPHA_FCC, {}, STRUCT_PLANE),
    (160, "bcc_dg", "pseudochiral_trivial", [np.pi, 0.0, np.pi], {}, STRUCT_PLANE),     # half-plane clusters
    (160, "bcc_dg", "pseudochiral_crossdof", [np.pi, 0.0, np.pi], {}, STRUCT_CROSS_PLANE),
    (150, "fcc", "chiral", _ALPHA_FCC, {}, STRUCT_FIVE),                                # five passes, k_zmid
    (150, "bcc_sg", "pseudochiral_trivial", [np.pi / 20, 0.0, 0.0], {}, STRUCT_FIVE),
    (150, "bcc_sg", "pseudochiral_crossdof", [np.pi, 0.5 * np.pi, 0.0], {}, STRUCT_CROSS7),
    (256, "sc_curv", "chiral", [np.pi, np.pi, np.pi], {}, STRUCT_FIVE),                 # single-stage k_zmid
    (256, "bcc_dg", "pseudochiral_crossdof", [np.pi, 0.0, np.pi], {}, STRUCT_CROSS7),
]
# the same structures at sizes the emulation runs (no clusters there: the coupled M takes the five-pass path)
EMU_CASES = [
    (16, "sc_curv", None, _ALPHA_FCC, {}, STRUCT_PLANE),
    (24, "fcc", "chiral", _ALPHA_FCC, {"mid_five": 1}, STRUCT_PLANE),
    (16, "fcc", "chiral", _ALPHA_FCC, {}, STRUCT_PLANE),
    (16, "bcc_dg", "pseudochiral_crossdof", [np.pi, 0.0, np.pi], {"plane_cross": 1}, STRUCT_CROSS_PLANE),
    (16, "bcc_dg", "pseudochiral_crossdof", [np.pi, 0.0, np.pi], {"plane_cross": 2}, STRUCT_CROSS_PLANE),
    (16, "fcc", "chiral", _ALPHA_FCC, {"plane_split": 1}, STRUCT_PLANE),                # z-split half planes
    (16, "bcc_dg", "pseudochiral_crossdof", [np.pi, 0.0, np.pi], {"plane_split": 1, "plane_cross": 2}, STRUCT_CROSS_PLANE),
    (12, "fcc", "chiral", _ALPHA_FCC, {}, STRUCT_FIVE),
    (12, "sc_curv", "pseudochiral_trivial", [np.pi, 0.0, 0.0], {}, STRUCT_FIVE),
    (12, "bcc_sg", "pseudochiral_crossdof", [np.pi, 0.5 * np.pi, 0.0], {}, STRUCT_CROSS7),
]
_DEFAULT_OPTIONS = {"mid_five": -1, "plane_cross": 1, "plane_split": 0}


def _kernels(struct, N, options):
    """Kernels of one A / H apply of at most 32 columns, the cross-DoF stencil kernel included."""
    if struct == STRUCT_CROSS_PLANE:      # stencil fused into the inverse plane half (4), or its own kernel between the halves (5):
        return 5 if options.get("plane_cross", 2 if N >= 160 else 1) == 2 else 4      # the default of the z-split sizes N >= 160
    return {STRUCT_PLANE: 3, STRUCT_FIVE: 5, STRUCT_CROSS7: 7}[struct]


def _case_id(c):
    opt = "".join(f"-{k}{v}" for k, v in c[4].items())
    return f"N{c[0]}-{c[1]}-{c[2] or 'vacuum'}{opt}"


def _operator_widths(pkg, oc, case, widths, timed_width):
    """H and A at every width: each column bit-identical to the single-column apply of that column, the first and the last
    column of the widest call against the oracle, pcb_apply_timed == pcb_apply, and in-place calls: equal to the
    out-of-place result where the structure allows them, else refused with every output column untouched."""
    ctx, options = pkg.get_context(case[0]), case[4]
    try:      # (plane_cross and plane_split are read at apply time: kept for the whole case)
        for k, v in options.items():
            ctx.option(k, v)
        _operator_widths_on(pkg, oc, ctx, case, widths, timed_width)
    finally:
        for k in options:
            ctx.option(k, _DEFAULT_OPTIONS[k])


def _operator_widths_on(pkg, oc, ctx, case, widths, timed_width):
    N, d_flag, typ, alpha, options, struct = case
    alpha = np.array(alpha, dtype=float)
    L = pkg._lib
    op = _ops(pkg, N, d_flag, alpha, typ)
    kmax = max(widths)
    X = ctx.random_block(kmax, 1000 + N)
    Y1, Y = ctx.empty(kmax), ctx.empty(kmax)
    sym = _oracle(pkg, oc, N, d_flag, alpha, typ)
    ends = [0, kmax - 1]
    want_a, want_h = _oracle_AH(oc, sym, X.cols(ends).get())
    inplace_ok = {L.APPLY_H: struct == STRUCT_PLANE, L.APPLY_A: struct != STRUCT_CROSS_PLANE}
    for mode, want in ((L.APPLY_H, want_h), (L.APPLY_A, want_a)):
        name = "H" if mode == L.APPLY_H else "A"
        for j in range(kmax):
            op.apply_into(mode, X.cols([j]), Y1.cols([j]))
        assert np.all(_colerr(Y1.cols(ends).get(), want) < 1e-12), (name, "oracle")
        for w in widths:
            op.apply_into(mode, X.cols(range(w)), Y.cols(range(w)))
            eq = _same(pkg, Y1.cols(range(w)), Y.cols(range(w)))
            assert eq.all(), (name, w, np.flatnonzero(~eq))
        # pcb_apply_timed runs the kernels bench.py's per-pass table reports: the same kernels and numbers as pcb_apply
        kernels = _kernels(struct, N, options)
        n0 = ctx.launches()
        L.check(_apply_rc(pkg, op, mode, X.cols(range(timed_width)), Y.cols(range(timed_width))), "pcb_apply")
        assert ctx.launches() - n0 == kernels, (name, "pcb_apply launches", ctx.launches() - n0)
        n0 = ctx.launches()
        rc, npass = _apply_timed(pkg, op, mode, X.cols(range(timed_width)), Y.cols(range(timed_width)))
        L.check(rc, "pcb_apply_timed")
        assert npass == kernels and ctx.launches() - n0 == kernels, (name, "pcb_apply_timed", npass, ctx.launches() - n0)
        assert _same(pkg, Y1.cols(range(timed_width)), Y.cols(range(timed_width))).all(), (name, "timed")
        Y.assign(X)
        rc = _apply_rc(pkg, op, mode, Y, Y)
        if inplace_ok[mode]:
            assert rc == 0, (name, pkg._lib.lib().pcb_last_error())
            assert _same(pkg, Y1, Y).all(), (name, "in place")
        else:
            assert rc == -2, (name, "in place must be refused")
            _refused_alias_leaves_outputs(pkg, op, mode, X, Y, kmax - 1)
            if timed_width > 1:
                _refused_alias_leaves_outputs(pkg, op, mode, X, Y, timed_width - 1, timed=timed_width)


def _refused_alias_leaves_outputs(pkg, op, mode, X, Y, j_alias, timed=0):
    """out[j_alias] = in[j_alias] where the structure refuses in-place columns: -2, and no output column is written -- also
    when the aliased column is in a later launch chunk than columns already processed (j_alias >= PCB_MAXC = 32).  The outputs
    hold a copy of X before the call, which differs from op(X) everywhere: a column written before the refusal shows."""
    k = timed or X.k
    Y.assign(X)                                          # snapshot: Y_j = X_j, not op(X_j)
    probe = (pkg.pcfft.column_norms(X.cols([j_alias])), pkg.pcfft.column_dots(X.cols([j_alias]), X.cols([0])))
    out = pkg.devarray.DeviceBlock(Y.ctx, _owners=Y._owners, _ptrs=Y.ptrs[:k])
    out.ptrs[j_alias] = X.ptrs[j_alias]
    rc = _apply_timed(pkg, op, mode, X.cols(range(k)), out)[0] if timed else _apply_rc(pkg, op, mode, X.cols(range(k)), out)
    assert rc == -2, ("aliased column", j_alias, rc)
    assert b"in[" in pkg._lib.lib().pcb_last_error()
    Y.ctx.sync()
    others = [j for j in range(k) if j != j_alias]
    eq = _same(pkg, X.cols(others), Y.cols(others))
    assert eq.all(), ("output written before the refusal", j_alias, [others[i] for i in np.flatnonzero(~eq)])
    assert (pkg.pcfft.column_norms(X.cols([j_alias])), pkg.pcfft.column_dots(X.cols([j_alias]), X.cols([0]))) == probe


@pytest.mark.parametrize("case", EMU_CASES, ids=_case_id)
def test_operator_widths_emu(emu, oracle, case):
    _operator_widths(emu, oracle, case, (1, 2, 5, 33), 16)


@pytest.mark.gpu
@pytest.mark.parametrize("case", GPU_CASES, ids=_case_id)
def test_operator_widths(gpu, oracle, case):
    if case[0] == 256:
        _operator_widths(gpu, oracle, case, (1, 3, 9), 9)          # one column is 805 MB
    else:
        _operator_widths(gpu, oracle, case, (1, 2, 5, 17, 32, 33), 16)


def _pointwise_and_fft(pkg, oc, N, d_flag, typ, alpha):
    """P, M, K_A, K_A^H, gamma K_B, FFT and IFFT on 33 columns (two launches where a mode launches per chunk) vs the oracle /
    scipy on the first and the last two columns; in place (allowed for all but the cross-DoF M) equals out of place, and the
    cross-DoF M refuses an aliased column in its second launch without writing any output column."""
    import scipy.fft as sf
    L = pkg._lib
    alpha = np.array(alpha, dtype=float)
    ctx = pkg.get_context(N)
    op = _ops(pkg, N, d_flag, alpha, typ)
    a, b, inv, shift, diel = _oracle(pkg, oc, N, d_flag, alpha, typ)
    k = 33
    X = ctx.random_block(k, 7 + N)
    Y, Z = ctx.empty(k), ctx.empty(k)
    probe = [0, 31, 32]
    x = X.cols(probe).get()
    fft = lambda v, f: f(v.reshape(3, N, N, N), axes=(1, 2, 3), workers=oc.FFT_WORKERS).reshape(v.shape)  # noqa: E731
    refs = {L.APPLY_P: lambda: oc.h_block(x, inv), L.APPLY_M: lambda: diel(x), L.APPLY_KA: lambda: oc.a_block(x, a),
            L.APPLY_KAH: lambda: oc.a_block(x, -a.conj()), L.APPLY_KB: lambda: oc.h_block(x, b),
            L.APPLY_FFT: lambda: np.stack([fft(x[:, j], sf.fftn) for j in range(len(probe))], axis=1),
            L.APPLY_IFFT: lambda: np.stack([fft(x[:, j], sf.ifftn) for j in range(len(probe))], axis=1)}
    for mode, ref in refs.items():
        op.apply_into(mode, X, Y)
        tol = 1e-13 if mode in (L.APPLY_FFT, L.APPLY_IFFT) else 1e-14
        assert np.all(_colerr(Y.cols(probe).get(), ref()) < tol), mode
        Z.assign(X)
        rc = _apply_rc(pkg, op, mode, Z, Z)
        if mode == L.APPLY_M and typ == "pseudochiral_crossdof":
            assert rc == -2
            _refused_alias_leaves_outputs(pkg, op, mode, X, Z, k - 1)      # aliased column in the second launch
            continue
        assert rc == 0, pkg._lib.lib().pcb_last_error()
        assert _same(pkg, Y, Z).all(), ("in place", mode)


@pytest.mark.parametrize("N,typ", [(16, "chiral"), (12, "chiral"), (12, "pseudochiral_crossdof")])
def test_pointwise_and_fft_modes_width33_emu(emu, oracle, N, typ):
    _pointwise_and_fft(emu, oracle, N, "bcc_sg", typ, [np.pi, 0.5 * np.pi, 0.0])


@pytest.mark.gpu
@pytest.mark.parametrize("N,typ", [(120, "chiral"), (150, "chiral"), (150, "pseudochiral_crossdof")])
def test_pointwise_and_fft_modes_width33(gpu, oracle, N, typ):
    _pointwise_and_fft(gpu, oracle, N, "bcc_sg", typ, [np.pi, 0.5 * np.pi, 0.0])


# ---- block kernels on slabs: ragged row counts and 1, 2, 3, 4, many row tiles per CTA -------------------------------------
def _update_variant(m, nl):
    """The k_update instantiation update_impl (pcb_capi.cu) selects for (m, n_loc), its rows per tile and CTAs per SM."""
    MP = 8 * ((m + 7) // 8)
    MPp, JT = MP + 2, MP // 4
    nlp = ((m + 1) & ~1) + ((nl - m + 1) & ~1)
    smem = lambda tr, stages: 16 * (2 * nlp * MPp + 2 * stages * nlp * (tr + 4))   # noqa: E731
    cap = 224 * 1024
    if JT == 4 and smem(32, 3) <= cap:
        name, tr, sm = "k_update<32,1,3>", 32, smem(32, 3)
    elif JT == 4 and smem(48, 2) <= cap:
        name, tr, sm = "k_update<48,1>", 48, smem(48, 2)
    elif smem(32, 2) <= cap:
        name, tr, sm = ("k_update<32,1>" if 4 * JT <= 16 else "k_update<32,2>"), 32, smem(32, 2)
    else:
        name, tr, sm = "k_update<16,1>", 16, smem(16, 2)      # (<16,2> needs 2 JT > 16: m > 32, never)
    fused = JT == 4 and m <= 16 and smem(48, 2) + 16 * 2 * 48 * 17 <= 226 * 1024
    return name, tr, max(1, min(4, cap // (sm + 1024))), fused


# (m, n_loc) pairs covering every k_update instantiation the solver can select (nev 5..20: m = 8..32, n_loc <= 3 m)
UPDATE_PAIRS = [(8, 24), (16, 42), (16, 58), (16, 64), (20, 60), (32, 64), (16, 96), (32, 96)]
FUSED_M, TWO_KERNEL_M = (9, 13, 16), (4, 8, 20, 32)


def _gram_ctas_per_sm(n):
    """CTAs per SM pcb_gram2 plans for n columns (before the occupancy query, which can only lower it)."""
    nt = (n + 7) // 8
    npairs = nt * (nt + 1) // 2
    nlaunch = -(-npairs // 40)
    np_ = -(-npairs // nlaunch)
    W = 0
    for ppw in (1, 2):
        w = -(-np_ // ppw)
        if W == 0 and w <= 20 and ((w * ppw - np_) * 8 <= np_ or ppw == 2):
            W = w
    W = max(W, 4)
    smem = 16 * 4 * 8 * nt * 36
    return max(1, min(4, 224 * 1024 // (smem + 1024), 2048 // (32 * W)))


def _tiles_per_cta(ntiles, grid):
    return -(-ntiles // max(1, min(grid, ntiles)))


def _tile_counts(N, h, sms):
    """Row tiles per CTA the three tiled kernels are expected to get on a slab of h planes -- a copy of the launch planning,
    used only to choose the slabs; the counts reported and asserted are the ones the library reports (pcb_block_launch_info)."""
    nloc = h * N * N
    R = 3 * nloc
    out = {"k_gram2(n=24)": _tiles_per_cta(-(-R // 32), sms * _gram_ctas_per_sm(24)),
           "k_update_res": _tiles_per_cta(-(-nloc // 16), sms)}
    for m, nl in ((8, 24), (16, 42)):
        name, tr, per_sm, _ = _update_variant(m, nl)
        out[name] = _tiles_per_cta(-(-R // tr), sms * per_sm)
    return out


def _sweep_slabs(pkg, sms):
    """The smallest slabs (N, z0, z1) on which every tiled kernel gets 1, 2, 3 and 4 row tiles per CTA, plus the ragged ones
    (cells per plane = 4 mod 16, z0 > 0), which give every kernel many tiles per CTA."""
    sizes = (6, 8, 12, 16) if pkg.backend_name == "emu" else (24, 48)
    want = {}
    for N in sizes:
        for h in range(1, N + 1):
            for kern, t in _tile_counts(N, h, sms).items():
                key = (kern, t)
                if t <= 4 and (key not in want or h * N * N < want[key][1] * want[key][0] ** 2):
                    want[key] = (N, h)
    slabs = sorted({(N, N - h, N) if i % 2 else (N, 0, h) for i, (N, h) in enumerate(sorted(set(want.values())))})
    ragged = [(6, 2, 5), (6, 0, 1)] if pkg.backend_name == "emu" else [(150, 37, 40), (150, 0, 7)]
    targets = {}
    for kern, t in want:
        targets.setdefault(kern, set()).add(t)
    return slabs + ragged, targets


def _slab_rows(N, z0, z1):
    nn, pl = N ** 3, N * N
    return np.concatenate([c * nn + np.arange(z0 * pl, z1 * pl) for c in range(3)])


def _hot_rows(R, nloc):
    """Rows that carry large values: the first and the last row, both sides of the last tile boundary of every tile height
    (16 / 32 / 48 rows, 16 cells), the component boundaries and all of the last partial tiles."""
    rows = {0, R - 1}
    for t in (16, 32, 48):
        b = (R // t) * t
        rows |= {b - 1, min(b, R - 1)} | set(range(b, R))
        rows |= {t - 1, min(t, R - 1)}
    for c in range(3):
        for cell in (0, 15, 16, nloc - 16 - (nloc % 16), nloc - 1):
            if 0 <= cell < nloc:
                rows.add(c * nloc + cell)
    return np.array(sorted(rows))


def _block(rng, R, nloc, k):
    """k columns of different scales (1e-3 .. 1e3) with large entries on the hot rows."""
    a = rng.standard_normal((R, k)) + 1j * rng.standard_normal((R, k))
    a[_hot_rows(R, nloc)] *= 1e3
    return a * np.logspace(-3, 3, k)[rng.permutation(k)]


def _check_gram(G, ref, sa, sb, R, c=16):
    """Entry by entry against the Cauchy-Schwarz scale of its two columns: |G_ab - ref_ab| <= c 1e-15 sqrt(R) |s_a| |s_b|."""
    bound = c * 1e-15 * np.sqrt(R) * np.outer(sa, sb)
    bad = np.abs(G - ref) > bound
    assert not bad.any(), (np.argwhere(bad)[:5], np.max(np.abs(G - ref) / bound))


# K_P^-1 is inverted per cell on the device from the symbol tables; where the 3 x 3 block is ill-conditioned (the cells near
# k = 0, which _hot_rows weights by 1e3) its entries are a few 1e-12 off the oracle's inverse.  A wrong plane (z0) or a wrong
# lambda is an O(1) error.
PRECOND_TOL = 1e-11


def _slab_op(pkg, ctx, N, d_flag="fcc", alpha=(0.3, 0.0, 0.1)):
    mfd = pkg.discretization
    alpha = np.array(alpha, dtype=float)
    relax, pnt = mfd.set_relaxation(alpha)
    a_fft, b_fft = mfd.fft_blocks(N, 1, pkg.dielectric.diel_info(d_flag, option="ct"), alpha=alpha)
    inv_fft = mfd.inverse_3_times_3_B(b_fft, pnt, relax[0])
    gamma, pshift = pkg.pcfft._sym_consistency(a_fft, (pnt * b_fft[0], pnt * b_fft[1]), inv_fft)
    return pkg.pcfft.Operator(a_fft, gamma, relax[0], pshift, None, ctx=ctx), alpha


def _launched(pkg, ctx):
    """(name, row tiles per CTA) of the last tiled block kernel the library planned on this context."""
    L = pkg._lib
    name, grid, tiles = C.create_string_buffer(32), C.c_longlong(), C.c_longlong()
    L.check(L.lib().pcb_block_launch_info(ctx.h, name, 32, C.byref(grid), C.byref(tiles)), "pcb_block_launch_info")
    return name.value.decode(), -(-tiles.value // grid.value)


def _block_kernels_on_slab(pkg, oc, N, z0, z1, counts):
    L = pkg._lib
    lib = L.lib()
    P = L.ptr_array
    ctx = pkg.devarray.Context(N, slab=(z0, z1))
    R, nloc = ctx.R, ctx.nloc
    seen = counts.setdefault((N, z0, z1), {})      # kernel -> row tiles per CTA, as launched
    rng = np.random.default_rng(N * 1000 + z0 * 37 + z1)
    s = _block(rng, R, nloc, 96)
    d = rng.standard_normal((R, 1))
    hs = d * s                                  # S^H HS Hermitian, like S^H (H S)
    S, HS = ctx.from_host(s), ctx.from_host(hs)
    ns, nh = np.linalg.norm(s, axis=0), np.linalg.norm(hs, axis=0)
    # Gram pair: every width class (one 8-column tile, padding, several launches)
    for n in (5, 24, 48, 96):
        G, T = pkg.orthogonalization.gram_pair(S.cols(range(n)), HS.cols(range(n)))
        g, t = s[:, :n].conj().T @ s[:, :n], s[:, :n].conj().T @ hs[:, :n]
        _check_gram(G, (g + g.conj().T) / 2, ns[:n], ns[:n], R)
        _check_gram(T, (t + t.conj().T) / 2, np.maximum(ns[:n], nh[:n]), np.maximum(ns[:n], nh[:n]), R)
        if n == 24:
            name, seen["k_gram2(n=24)"] = _launched(pkg, ctx)
            assert name == "k_gram2"
    for ntop in (3, 8, 20):
        n = 48
        G, T = pkg.orthogonalization.gram_pair_top(S.cols(range(n)), HS.cols(range(n)), ntop)
        g, t = s[:, :ntop].conj().T @ s[:, :n], hs[:, :ntop].conj().T @ s[:, :n]
        _check_gram(G[:ntop], g, ns[:ntop], ns[:n], R)
        _check_gram(T[:ntop], t, nh[:ntop], ns[:n], R)
    # column dots over 96 columns
    dots = pkg.pcfft.column_dots(S, HS)
    assert np.all(np.abs(dots - np.einsum("ij,ij->j", s.conj(), hs)) <= 16e-15 * np.sqrt(R) * ns * nh)
    # axpby
    Y = ctx.from_host(hs[:, :5])
    _axpby(pkg, S.cols(range(5)), Y, 0.75, -1.5)
    ref = 0.75 * s[:, :5] - 1.5 * hs[:, :5]
    assert np.all(np.abs(Y.get() - ref) <= 4e-16 * (np.abs(0.75 * s[:, :5]) + np.abs(1.5 * hs[:, :5])))
    # residual (+ preconditioner), 7 and 33 columns: one 8-column group, and a second launch (PCB_MAXC_RP = 32)
    op, alpha = _slab_op(pkg, ctx, N)
    io = oc.assemble_symbols(N, "fcc", alpha)[2]
    rows = _slab_rows(N, z0, z1)
    io_slab = (io[0][rows], io[1][rows])
    for k in (7, 33):
        lam = np.linspace(-2.0, 3.0, k)
        r = s[:, :k] * lam - hs[:, :k]
        for precond in range(4):
            W = ctx.empty(k)
            norms2 = np.empty(k)
            L.check(lib.pcb_residual(op.h, precond, k, P(S.ptrs[:k]), P(HS.ptrs[:k]), P(W.ptrs), lam.ctypes.data_as(L.c_double_p),
                                     norms2.ctypes.data_as(L.c_double_p)), "pcb_residual")
            assert np.allclose(norms2, np.linalg.norm(r, axis=0) ** 2, rtol=1e-13, atol=0), (k, precond)
            want = oc.h_block(r, io_slab) if precond in (1, 2) else r
            err = _colerr(W.get(), want)
            if precond < 2:
                assert np.all(err < (1e-14 if precond == 0 else PRECOND_TOL)), (k, precond, err)
            else:      # rounded to complex64 before K_P^-1: off by that rounding, and not less
                assert np.all(err < 1e-7) and np.all(err > 1e-10), (k, precond, err)
    # update, every k_update instantiation
    for m, nl in UPDATE_PAIRS:
        name, tpc = _check_update(pkg, ctx, s, hs, m, nl, rng)
        counts.setdefault(("variants",), set()).add(name)
        if (m, nl) in ((8, 24), (16, 42)):
            seen[name] = tpc
    # update + residual: fused (k_update_res) and two kernels, direct and through _start / _wait
    for m in FUSED_M + TWO_KERNEL_M:
        for split in (False, True):
            name, tpc = _check_update_resid(pkg, oc, ctx, op, io_slab, s, hs, m, 3 * m, rng, split)
            assert (name == "k_update_res") == (m in FUSED_M), (m, name)
            if name == "k_update_res":
                seen[name] = tpc


def _check_update(pkg, ctx, s, hs, m, nl, rng):
    """pcb_update vs NumPy; returns the instantiation the library ran and its row tiles per CTA."""
    L = pkg._lib
    P = L.ptr_array
    S, HS = ctx.from_host(s[:, :nl]), ctx.from_host(hs[:, :nl])
    Pd, HPd = ctx.empty(m), ctx.empty(m)
    E = np.ascontiguousarray(rng.standard_normal((nl, m)) + 1j * rng.standard_normal((nl, m)))
    L.check(L.lib().pcb_update(ctx.h, m, nl, P(S.ptrs), P(HS.ptrs), P(Pd.ptrs), P(HPd.ptrs), E.ctypes.data), "pcb_update")
    for a, A, Pb in ((s, S, Pd), (hs, HS, HPd)):
        pn = a[:, m:nl] @ E[m:]
        xn = a[:, :m] @ E[:m] + pn
        scale = np.abs(a[:, :nl]).max(axis=0) @ np.abs(E)            # per output column: sum_k |a_k|_inf |E_kj|
        got = A.get()
        assert np.all(np.abs(got[:, :m] - xn) <= 1e-14 * scale), (m, nl, _update_variant(m, nl)[0])
        assert np.all(np.abs(Pb.get() - pn) <= 1e-14 * scale), (m, nl, _update_variant(m, nl)[0])
        assert np.array_equal(got[:, m:], a[:, m:nl]), "W / P inputs must stay untouched"
    launched = _launched(pkg, ctx)
    assert launched[0] == _update_variant(m, nl)[0], (m, nl, launched)      # the case names the variant it runs
    return launched


def _check_update_resid(pkg, oc, ctx, op, io_slab, s, hs, m, nl, rng, split):
    L = pkg._lib
    P = L.ptr_array
    S, HS = ctx.from_host(s[:, :nl]), ctx.from_host(hs[:, :nl])
    Pd, HPd, W = ctx.empty(m), ctx.empty(m), ctx.empty(m)
    E = np.ascontiguousarray(rng.standard_normal((nl, m)) + 1j * rng.standard_normal((nl, m)))
    lam = np.linspace(0.5, 3.0, m)
    lp = lam.ctypes.data_as(L.c_double_p)
    norms2 = np.empty(m)
    args = (op.h, m, nl, P(S.ptrs), P(HS.ptrs), P(Pd.ptrs), P(HPd.ptrs), E.ctypes.data, lp, P(W.ptrs))
    if split:
        L.check(L.lib().pcb_update_resid_start(*args), "pcb_update_resid_start")
        L.check(L.lib().pcb_update_resid_wait(op.h, m, norms2.ctypes.data_as(L.c_double_p)), "pcb_update_resid_wait")
    else:
        L.check(L.lib().pcb_update_resid(*args, norms2.ctypes.data_as(L.c_double_p)), "pcb_update_resid")
    launched = _launched(pkg, ctx)
    xn = s[:, :nl] @ E
    hxn = hs[:, :nl] @ E
    sc_x = np.abs(s[:, :nl]).max(axis=0) @ np.abs(E)
    sc_h = np.abs(hs[:, :nl]).max(axis=0) @ np.abs(E)
    got_x, got_hx = S.get()[:, :m], HS.get()[:, :m]
    assert np.all(np.abs(got_x - xn) <= 1e-14 * sc_x) and np.all(np.abs(got_hx - hxn) <= 1e-14 * sc_h), (m, split)
    # the residual of the updated columns, its norms and W = K_P^-1 r on the slab rows (symbols at i2 = z0 + plane; a wrong
    # plane or a wrong lambda is an O(1) error)
    r = got_x * lam - got_hx
    assert np.allclose(norms2, np.linalg.norm(r, axis=0) ** 2, rtol=1e-12, atol=0), (m, split)
    assert np.all(_colerr(W.get(), oc.h_block(r, io_slab)) < PRECOND_TOL), (m, split)
    return launched


def _report(counts, sms):
    lines = [f"row tiles per CTA on {sms} SMs, as launched (slab N, z0, z1 -> kernel: tiles):"]
    reached = {}
    for key, c in sorted((k, v) for k, v in counts.items() if k != ("variants",)):
        lines.append(f"  {key}: " + ", ".join(f"{n} {t}" for n, t in c.items()))
        for n, t in c.items():
            reached.setdefault(n, set()).add(t)
    for n, ts in reached.items():
        lines.append(f"  reached {n}: {sorted(ts)}")
    lines.append(f"  k_update instantiations launched: {sorted(counts.get(('variants',), ()))}")
    print("\n".join(lines))
    return reached


def _block_sweep(pkg, oc):
    sms = _sms(pkg)
    counts = {}
    slabs, targets = _sweep_slabs(pkg, sms)
    for N, z0, z1 in slabs:
        _block_kernels_on_slab(pkg, oc, N, z0, z1, counts)
    reached = _report(counts, sms)
    for kern, ts in reached.items():
        assert targets[kern] <= ts, (kern, ts)
        if pkg.backend_name == "cuda":      # (the emulation has 2 "SMs": one tile per CTA is out of reach for k_update_res)
            assert {1, 2, 3, 4} <= ts and max(ts) >= 6, (kern, ts)
    assert counts[("variants",)] == {"k_update<32,1,3>", "k_update<48,1>", "k_update<32,1>", "k_update<32,2>", "k_update<16,1>"}


def test_block_kernels_tile_counts_and_ragged_slabs_emu(emu, oracle):
    _block_sweep(emu, oracle)


@pytest.mark.gpu
def test_block_kernels_tile_counts_and_ragged_slabs(gpu, oracle):
    _block_sweep(gpu, oracle)


@pytest.mark.gpu
def test_block_kernels_whole_n150(gpu, oracle):
    """One whole N = 150 context (R = 10 125 000 rows: a partial last tile of every height) at m = 8, n_loc = 24."""
    N, m, nl = 150, 8, 24
    ctx = gpu.get_context(N)
    rng = np.random.default_rng(150)
    S0 = ctx.random_block(nl, 150)
    s = S0.get()
    del S0
    s[_hot_rows(ctx.R, ctx.nloc)] *= 1e3
    s *= np.logspace(-2, 2, nl)
    d = rng.standard_normal((ctx.R, 1))
    hs = d * s
    S, HS = ctx.from_host(s), ctx.from_host(hs)
    ns, nh = np.linalg.norm(s, axis=0), np.linalg.norm(hs, axis=0)
    G, T = gpu.orthogonalization.gram_pair(S, HS)
    g, t = s.conj().T @ s, s.conj().T @ hs
    _check_gram(G, (g + g.conj().T) / 2, ns, ns, ctx.R)
    _check_gram(T, (t + t.conj().T) / 2, np.maximum(ns, nh), np.maximum(ns, nh), ctx.R)
    del S, HS
    _check_update(gpu, ctx, s, hs, m, nl, rng)
    op, alpha = _slab_op(gpu, ctx, N)
    io = oracle.assemble_symbols(N, "fcc", alpha)[2]
    _check_update_resid(gpu, oracle, ctx, op, io, s, hs, m, nl, rng, True)


def _fill_uniform_on_slabs(pkg, N, slabs):
    full = pkg.get_context(N).random_block(3, 77).get()
    for z0, z1 in slabs:
        ctx = pkg.devarray.Context(N, slab=(z0, z1))
        assert np.array_equal(ctx.random_block(3, 77).get(), full[_slab_rows(N, z0, z1)]), (z0, z1)


def test_fill_uniform_slab_matches_full_context_emu(emu):
    _fill_uniform_on_slabs(emu, 12, [(0, 1), (5, 7), (3, 12), (0, 12)])


@pytest.mark.gpu
def test_fill_uniform_slab_matches_full_context(gpu):
    _fill_uniform_on_slabs(gpu, 150, [(0, 7), (37, 40), (149, 150)])


# ---- host pipeline ------------------------------------------------------------------------------------------------------
def _wide(pkg, shape, pinned):
    return pkg.devarray.pinned_empty(shape) if pinned else np.empty(shape, dtype=np.complex128)


def _host_pipeline(pkg, N, widths):
    """pcb_apply_host (chunks of 8 columns, two staging slots reused from chunk 2 on, ragged last chunk, staging re-sized
    when the width changes) on views into wider row-major arrays (ldx, ldy > k): bit-identical to pcb_apply on the device,
    and the columns outside the views are never touched.  Pinned and pageable host memory alternate."""
    L = pkg._lib
    lib = L.lib()
    alpha = np.array([0.3 * np.pi, 2 * np.pi, 0.0])
    op = _ops(pkg, N, "fcc", alpha, "chiral")
    ctx = op.ctx
    R = ctx.R
    rng = np.random.default_rng(N)
    for i, k in enumerate(widths):
        pinned = i % 2 == 0
        ldx, ldy, off = k + 3, k + 2, 1
        xw = _wide(pkg, (R, ldx), pinned)
        xw[:] = rng.standard_normal((R, ldx)) + 1j * rng.standard_normal((R, ldx))
        x_keep = xw.copy()
        yw = _wide(pkg, (R, ldy), not pinned)
        X = ctx.from_host(np.ascontiguousarray(xw[:, off:off + k]))
        Y = ctx.empty(k)
        for mode in (L.APPLY_H, L.APPLY_A, L.APPLY_P):
            yw[:] = complex(np.nan, np.inf)                             # sentinel
            L.check(lib.pcb_apply_host(op.h, mode, k, xw[:, off:].ctypes.data, ldx, yw[:, off:].ctypes.data, ldy), "pcb_apply_host")
            op.apply_into(mode, X, Y)
            assert np.array_equal(yw[:, off:off + k], Y.get()), (k, mode)
            sent = np.delete(yw, np.arange(off, off + k), axis=1)
            assert np.all(np.isnan(sent.real)) and np.all(np.isinf(sent.imag)), (k, mode, "wrote outside the view")
            assert np.array_equal(xw, x_keep, equal_nan=True)
        # the same layouts through pcb_block_upload / pcb_block_download
        B = ctx.empty(k)
        L.check(lib.pcb_block_upload(ctx.h, xw[:, off:].ctypes.data, ldx, k, L.ptr_array(B.ptrs)), "pcb_block_upload")
        assert np.array_equal(B.get(), xw[:, off:off + k])
        yw[:] = complex(np.nan, np.inf)
        L.check(lib.pcb_block_download(ctx.h, yw[:, off:].ctypes.data, ldy, k, L.ptr_array(B.ptrs)), "pcb_block_download")
        assert np.array_equal(yw[:, off:off + k], xw[:, off:off + k])
        sent = np.delete(yw, np.arange(off, off + k), axis=1)
        assert np.all(np.isnan(sent.real)) and np.all(np.isinf(sent.imag))
        pkg.devarray.pinned_free(xw if pinned else yw)


def test_host_pipeline_widths_and_strides_emu(emu):
    _host_pipeline(emu, 8, (3, 20, 1, 8, 9, 17))


@pytest.mark.gpu
def test_host_pipeline_widths_and_strides(gpu):
    _host_pipeline(gpu, 120, (3, 20, 1, 9))        # 3 -> 20 -> 1: staging re-sized; 20 = 8 + 8 + 4 and 9 = 8 + 1: ragged last chunks
