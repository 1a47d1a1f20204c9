"""Mimetic finite-difference symbols and dielectric handles (public surface of paper_2/discretization.py).

What the reference materialises as O(N^3) CuPy arrays -- ``a_fft`` (3 N^3 complex), ``b_fft`` and
``inv_fft`` (3 N^3 real + 3 N^3 complex each; README.md:115 "192 N^3 bytes") -- is kept here as
*descriptors*: nine 1-D tables of length N from which the kernels regenerate the Fourier symbol
K_c(i0,i1,i2) = T[c][0][i0] + T[c][1][i1] + T[c][2][i2] on the fly (SURVEY.md A.2-A.3).  The
functions keep the reference's names, arguments and return arity, so `numerical_experiments`
code reads the same; ``.toarray()`` materialises the reference array where a test wants it.
"""
from fractions import Fraction
from time import time

import numpy as np
from numpy import pi

from . import _lib as L
from . import dielectric as diel
from . import devarray
from .environment import K, SC_C, SCAL, say


# ---------------------------------------------------------------------------------------------
# Relaxation (discretization.py:31-49)
# ---------------------------------------------------------------------------------------------
def set_relaxation(alpha, scal=SCAL):
    """((shift, deflation ratio), penalty gamma) for a translation vector."""
    nu = np.linalg.norm(np.asarray(alpha, dtype=float) / scal)
    if nu > 1:
        return (0, 0.6), 4 * pi * pi
    if nu == 0:
        return (1.0 / pi, 0.6), 4 * pi * pi
    return (nu, 0.6), (2 * pi / nu) ** 2


# ---------------------------------------------------------------------------------------------
# Stencils and 1-D symbols (discretization.py:152-222)
# ---------------------------------------------------------------------------------------------
def mfd_stencil(k, deriv_order):
    """2k-point symmetric stencil on the staggered points {2(j-k)+1}: interpolation (order 0) or
    first derivative (order 1, per half-cell pair => factor 2) at the origin.

    The reference solves the moment system with sympy (:152-193); the same rational numbers are
    obtained here from the Lagrange basis: c_j = (order+1)! / order! ... evaluated exactly in
    fractions (order 0: L_j(0); order 1: 2 L_j'(0))."""
    npts = 2 * k
    if deriv_order >= npts:
        raise ValueError(f"Derivative order ({deriv_order}) must be less than the number of stencil points ({npts}).")
    if deriv_order > 1:
        return _moment_stencil(k, deriv_order)
    pts = [Fraction(2 * (j - k) + 1) for j in range(npts)]
    out = []
    for j, pj in enumerate(pts):
        others = [p for i, p in enumerate(pts) if i != j]
        denom = Fraction(1)
        for p in others:
            denom *= (pj - p)
        if deriv_order == 0:
            num = Fraction(1)
            for p in others:
                num *= -p
        else:
            num = Fraction(0)
            for skip in range(len(others)):
                term = Fraction(1)
                for i, p in enumerate(others):
                    if i != skip:
                        term *= -p
                num += term
            num *= 2
        out.append(float(num / denom))
    return np.array(out)


def _moment_stencil(k, deriv_order):
    """General order: exact rational solve of sum_j c_j p_j^i = (order+1) [i == order]."""
    n = 2 * k
    pts = [Fraction(2 * (j - k) + 1) for j in range(n)]
    rows = [[p ** i for p in pts] + [Fraction(deriv_order + 1 if i == deriv_order else 0)] for i in range(n)]
    for col in range(n):
        piv = next(r for r in range(col, n) if rows[r][col] != 0)
        rows[col], rows[piv] = rows[piv], rows[col]
        rows[col] = [v / rows[col][col] for v in rows[col]]
        for r in range(n):
            if r != col and rows[r][col] != 0:
                f = rows[r][col]
                rows[r] = [a - f * b for a, b in zip(rows[r], rows[col])]
    return np.array([float(rows[r][n]) for r in range(n)])


def diag_circulant_complex(sten, Lw, ind, N):
    """Eigenvalues of the periodic (circulant) stencil operator = N * ifft(first row) (:195-222)."""
    first = np.zeros(N, dtype=complex)
    first[0:Lw - (ind - 1)] = sten[ind - 1:Lw]
    if ind > 1:
        first[N - (ind - 1):N] = sten[0:ind - 1]
    return np.fft.ifft(first) * N


class FourierSymbols:
    """Descriptor of the curl symbol a_fft = (K_0, K_1, K_2) (fft_blocks, discretization.py:301-346).

    K_c = sum_j CT[c][j] D1[i_j] + 1j alpha_c/scal D0[i_c];  `tables[c][j]` holds the i_j-dependent
    summand, so K_c(i0,i1,i2) = tables[c][0][i0] + tables[c][1][i1] + tables[c][2][i2]."""

    def __init__(self, N, k, ct, alpha=None, scal=SCAL, factor=1.0):
        self.N, self.k, self.scal = int(N), int(k), scal
        self.ct = np.array(ct, dtype=float)
        self.alpha = None if alpha is None else np.asarray(alpha, dtype=float)
        self.factor = factor           # a_fft /= SCAL in the runners
        h = scal / N
        self.D1 = diag_circulant_complex(mfd_stencil(k, 1) / h, 2 * k, k, N)
        self.D0 = diag_circulant_complex(mfd_stencil(k, 0), 2 * k, k, N)

    def with_alpha(self, alpha, factor=None):
        s = FourierSymbols.__new__(FourierSymbols)
        s.__dict__.update(self.__dict__)
        s.alpha = None if alpha is None else np.asarray(alpha, dtype=float)
        if factor is not None:
            s.factor = factor
        return s

    def __truediv__(self, c):
        return self.with_alpha(self.alpha, factor=self.factor / c)

    __itruediv__ = __truediv__

    # -conj(a_fft) is how the reference spells K_A^H (pcfft.py:148); track it symbolically
    adjoint = False

    def conj(self):
        s = self.with_alpha(self.alpha)
        s._conj = not getattr(self, "_conj", False)
        s._neg = getattr(self, "_neg", False)
        return s

    def __neg__(self):
        s = self.with_alpha(self.alpha)
        s._neg = not getattr(self, "_neg", False)
        s._conj = getattr(self, "_conj", False)
        return s

    def kind(self):
        """'KA' for a_fft, 'KAH' for -conj(a_fft)."""
        c, n = getattr(self, "_conj", False), getattr(self, "_neg", False)
        if c == n:
            return "KAH" if c else "KA"
        raise ValueError("only a_fft and -conj(a_fft) are supported symbol forms")

    @property
    def tables(self):
        t = np.zeros((3, 3, self.N), dtype=np.complex128)
        for c in range(3):
            for j in range(3):
                t[c, j] = self.ct[c][j] * self.D1
            if self.alpha is not None:
                t[c, c] = t[c, c] + 1j * (self.alpha[c] / self.scal) * self.D0
        return t * self.factor

    @property
    def dtables(self):
        """(3, N) derivatives of the tables by the k-point: dK_c/dalpha_d = delta_cd dtables[d][i_d].  alpha enters only the
        Bloch term of the diagonal tables, so dtables[d] = 1j factor / scal D0 for every d and does not depend on alpha."""
        return np.tile(1j * (self.factor / self.scal) * np.asarray(self.D0, dtype=np.complex128), (3, 1))

    def toarray(self):
        """The reference's dense a_fft (3 N^3,) -- tests / interoperability only."""
        t, N = self.tables, self.N
        return np.concatenate([(t[c, 2][:, None, None] + t[c, 1][None, :, None] + t[c, 0][None, None, :]).ravel()
                               for c in range(3)])


class PenaltySymbols:
    """Descriptor of b_fft = (|K_c|^2, (conj(K_0)K_1, conj(K_0)K_2, conj(K_1)K_2)) times a scalar
    (fft_blocks :343-344; scaled by pnt in numerical_experiments.py:62,445)."""

    def __init__(self, a_sym, scale=1.0):
        self.a, self.scale = a_sym, scale

    def __getitem__(self, i):          # b_fft[0], b_fft[1] as in the reference tuple
        return _PenaltyPart(self, i)

    def __iter__(self):
        return iter((self[0], self[1]))

    def toarray(self):
        A = self.a.toarray()
        n = self.a.N ** 3
        a0, a1, a2 = A[:n], A[n:2 * n], A[2 * n:]
        return (self.scale * np.concatenate(((a0 * a0.conj()).real, (a1 * a1.conj()).real, (a2 * a2.conj()).real)),
                self.scale * np.concatenate((a0.conj() * a1, a0.conj() * a2, a1.conj() * a2)))


class _PenaltyPart:
    """b_fft[i] with scalar arithmetic (pnt * b_fft[0] / SCAL / SCAL keeps working)."""

    def __init__(self, parent, i, scale=1.0):
        self.parent, self.i, self.scale = parent, i, scale

    def __mul__(self, c):
        return _PenaltyPart(self.parent, self.i, self.scale * c)

    __rmul__ = __mul__

    def __truediv__(self, c):
        return _PenaltyPart(self.parent, self.i, self.scale / c)

    def toarray(self):
        return self.scale * self.parent.toarray()[self.i]


def penalty_scale(b_fft):
    """gamma carried by a b_fft given either as PenaltySymbols or as the (part0, part1) tuple."""
    if isinstance(b_fft, PenaltySymbols):
        return b_fft.scale
    p0 = b_fft[0]
    return p0.scale * p0.parent.scale


class PrecondSymbols:
    """Descriptor of inv_fft = symbols of (K_A K_A^H + pnt K_B + shift)^-1 (inverse_3_times_3_B :284-295);
    the 3x3 cofactor inverse is evaluated inside the kernels."""

    def __init__(self, a_sym, pnt, shift, scale=1.0):
        self.a, self.pnt, self.shift, self.scale = a_sym, pnt, shift, scale

    def __getitem__(self, i):
        return _PrecondPart(self, i)

    def __iter__(self):
        return iter((self[0], self[1]))


class _PrecondPart:
    def __init__(self, parent, i, scale=1.0):
        self.parent, self.i, self.scale = parent, i, scale

    def __mul__(self, c):
        return _PrecondPart(self.parent, self.i, self.scale * c)

    __rmul__ = __mul__


def fft_blocks(N, k, CT, alpha=None, scal=SCAL):
    """alpha None -> (D, Di) alpha-independent descriptors; else (A, B) (discretization.py:301-346)."""
    base = FourierSymbols(N, k, CT, None, scal)
    if alpha is None:
        return base, base
    a = base.with_alpha(alpha)
    return a, PenaltySymbols(a)


def inverse_3_times_3_B(B, pnt, shift=0.0):
    a = B.a if isinstance(B, PenaltySymbols) else B[0].parent.a
    return PrecondSymbols(a, pnt, shift)


# ---------------------------------------------------------------------------------------------
# Dielectric handles (discretization.py:352-453)
# ---------------------------------------------------------------------------------------------
class DielHandle:
    """Callable ``Diels(x)`` = M x in real space, and the object the fused operator consumes."""

    def __init__(self, n, kind, ind_e, ind_v, ediag, eoff, k=1, device=None):
        self.n, self.kind = int(n), kind
        self.ctx = devarray.get_context(n, device)
        self.ediag = np.asarray(ediag, dtype=np.float64).copy()
        self.eoff = np.asarray(eoff, dtype=np.complex128).copy()
        self.k = int(k) if k else 1
        sten = np.ascontiguousarray(mfd_stencil(self.k, 0), dtype=np.float64)
        ind_e = np.ascontiguousarray(ind_e, dtype=np.int64)
        ind_v = np.ascontiguousarray(ind_v if ind_v is not None else np.zeros(0), dtype=np.int64)
        self.n_e, self.n_v = len(ind_e), len(ind_v)
        import ctypes as C
        h = C.c_void_p()
        eo = np.ascontiguousarray(self.eoff).view(np.float64)
        lib = L.lib()
        L.check(lib.pcb_diel_create(self.ctx.h, kind, ind_e.ctypes.data_as(L.c_int64_p), len(ind_e),
                                    ind_v.ctypes.data_as(L.c_int64_p), len(ind_v),
                                    self.ediag.ctypes.data_as(L.c_double_p), eo.ctypes.data_as(L.c_double_p),
                                    self.k, sten.ctypes.data_as(L.c_double_p), C.byref(h)), "pcb_diel_create")
        self.h = h
        import weakref
        self._fin = weakref.finalize(self, lib.pcb_diel_destroy, h)
        self._ident_op = None

    @classmethod
    def materials(cls, n, mat, inv_eps, device=None):
        """Several isotropic materials (pcb_diel_create_materials): (M x)_r = inv_eps[mat[r]] x_r, with `mat` the material index
        of each of the 3 n^3 edge DoFs (row order r = c n^3 + p; index 0 is the background) and `inv_eps` one 1 / eps per
        material (at most 256)."""
        mat = np.asarray(mat)
        if mat.dtype != np.uint8 and mat.size and (mat.min() < 0 or mat.max() > 255):
            raise ValueError("material indices must lie in 0 ... 255")
        self = cls.__new__(cls)
        self.n, self.kind = int(n), L.DIEL_MATERIALS
        self.ctx = devarray.get_context(n, device)
        self.mat = np.ascontiguousarray(mat, dtype=np.uint8)
        self.inv_eps = np.ascontiguousarray(inv_eps, dtype=np.float64).ravel()
        import ctypes as C
        h = C.c_void_p()
        lib = L.lib()
        L.check(lib.pcb_diel_create_materials(self.ctx.h, self.mat.ctypes.data, self.mat.size,
                                              self.inv_eps.ctypes.data_as(L.c_double_p), len(self.inv_eps), C.byref(h)),
                "pcb_diel_create_materials")
        self.h = h
        import weakref
        self._fin = weakref.finalize(self, lib.pcb_diel_destroy, h)
        self._ident_op = None
        return self

    def set_inv_eps(self, inv_eps):
        """Replace the 1 / eps table of a materials dielectric in place (pcb_diel_set_inv_eps): every operator built on this
        handle applies the new values from its next launch.  Refused, with the old table kept, for another kind, a wrong length
        or a value that is not finite and > 0."""
        if self.kind != L.DIEL_MATERIALS:
            raise ValueError("set_inv_eps: only a materials dielectric has a table of 1 / eps")
        t = np.ascontiguousarray(inv_eps, dtype=np.float64).ravel()
        L.check(L.lib().pcb_diel_set_inv_eps(self.h, t.ctypes.data_as(L.c_double_p), len(t)), "pcb_diel_set_inv_eps")
        self.inv_eps = t.copy()

    def at_frequency(self, f):
        """Set every material's eps to its model's value at frequency f (models: dispersion.Drude / Lorentz / Constant, kept by
        materials_handle) and return the eps.  Raises ValueError, the table unchanged, when some eps is not finite and > 0 there."""
        models = getattr(self, "models", None)
        if models is None:
            raise ValueError("at_frequency: this handle has no permittivity models (materials_handle keeps them)")
        eps = np.array([float(m.eps(f)) for m in models])
        if not np.all(np.isfinite(eps) & (eps > 0.0)):
            raise ValueError(f"at_frequency({f}): eps = {eps} is not finite and > 0 for every material")
        self.set_inv_eps(1.0 / eps)
        return eps

    def __call__(self, x):
        from . import pcfft
        return pcfft.diel_apply(self, x)


def chiral_handle(n, d_flag, eps_opt=0, k=None, device=None):
    """Isotropic medium: rows in Omega_1 divided by eps (discretization.py:352-366)."""
    ind_e = diel.diel_io_index(n, d_flag, dofs="edge")
    eps1 = diel.diel_chiral_const(d_flag) if (eps_opt is None or eps_opt == 0) else eps_opt
    inv = 1.0 / eps1
    return DielHandle(n, L.DIEL_CHIRAL, ind_e, None, [inv, inv, inv], [0, 0, 0], device=device)


def materials_handle(n, d_flag, eps_opt=None, regions=None, background=1.0, device=None):
    """Several isotropic materials: the edge DoFs of regions[i] (index arrays into the 3 n^3 rows; later regions override earlier
    ones where they overlap) are divided by eps_opt[i], every other row by `background`.  Defaults: the regions of
    dielectric.material_regions (bcc_dg: its two gyroid networks; every other lattice: Omega_1) and the lattice's chiral eps for
    each of them -- the same M as chiral_handle(n, d_flag).

    Every entry of eps_opt and `background` may be a number or a dispersion model (dispersion.Drude / Lorentz); the handle keeps
    one model per material in `models` (index 0: the background) and starts from eps_inf of each; `at_frequency(f)` sets the
    table to eps(f)."""
    from . import dispersion as dsp
    regions = diel.material_regions(n, d_flag) if regions is None else list(regions)
    if len(regions) > 255:
        raise ValueError(f"{len(regions)} regions: at most 255 besides the background")
    if eps_opt is None or (np.isscalar(eps_opt) and eps_opt == 0):
        eps = [float(diel.diel_chiral_const(d_flag))] * len(regions)
    else:
        eps = np.atleast_1d(np.asarray(eps_opt, dtype=object))      # numbers (0-d arrays too) or models
        if eps.ndim != 1:
            raise ValueError(f"eps_opt has shape {eps.shape}: expected one value per region")
        eps = eps.tolist()
        if len(eps) != len(regions):
            raise ValueError(f"eps_opt has {len(eps)} values for {len(regions)} regions")
    models = [dsp.as_model(background)] + [dsp.as_model(e) for e in eps]
    mat = np.zeros(3 * n ** 3, dtype=np.uint8)
    for i, reg in enumerate(regions):
        mat[np.asarray(reg, dtype=np.int64)] = i + 1
    inv_eps = 1.0 / np.array([m.eps_inf for m in models])
    h = DielHandle.materials(n, mat, inv_eps, device=device)
    h.models = models
    return h


def _eps_loc(d_flag, eps_opt, eps_mat):
    if eps_mat is not None:
        return np.asarray(eps_mat, dtype=complex)
    return diel.diel_pseudochiral_const(eps_opt) / diel.diel_chiral_const(d_flag)


def pseudochiral_trivial_handle(n, d_flag=SC_C, eps_opt=0, eps_mat=None, k=None, flag_mat=False, device=None):
    """M_Trivial (discretization.py:368-401): eps_cc on the edge DoFs of Omega_1 and the off-diagonal
    eps_ab coupling the three components of a cell whose volume DoF lies in Omega_1."""
    if flag_mat:
        raise NotImplementedError("flag_mat=True (explicit CSR matrix) is a set-up/debug path of the reference; "
                                  "the device operator is matrix-free")
    t0 = time()
    eps = _eps_loc(d_flag, eps_opt, eps_mat)
    ind_e = diel.diel_io_index(n, d_flag, dofs="edge")
    ind_v = diel.diel_io_index(n, d_flag, dofs="volume")
    h = DielHandle(n, L.DIEL_TRIVIAL, ind_e, ind_v, [eps[0].real, eps[1].real, eps[2].real], eps[3:6], device=device)
    say(f"D-matrix is generated, runtime = {time() - t0:<6.3f}s.")
    return h


def pseudochiral_crossdof_handle(n, d_flag=SC_C, eps_opt=0, eps_mat=None, k=1, flag_mat=False, device=None):
    """M_CrossDoF (discretization.py:403-453): same diagonal; off-diagonal blocks eps_ab S_ab with the
    2k-point averaging stencils between the staggered edge DoFs (applied as a stencil kernel)."""
    if flag_mat:
        raise NotImplementedError("flag_mat=True (explicit CSR matrix) is a set-up/debug path of the reference; "
                                  "the device operator is matrix-free")
    t0 = time()
    eps = _eps_loc(d_flag, eps_opt, eps_mat)
    ind_e = diel.diel_io_index(n, d_flag, dofs="edge")
    h = DielHandle(n, L.DIEL_CROSSDOF, ind_e, None, [eps[0].real, eps[1].real, eps[2].real], eps[3:6], k=k, device=device)
    say(f"D-matrix (her) is generated, runtime = {time() - t0:<6.3f}s.")
    return h
