"""The matrix-free operator on the GPU (public surface of paper_2/pcfft.py).

    AMA(x, a_fft, Diels)                  = K_A IFFT3( M FFT3( K_A^H x ) )           pcfft.py:130-158
    AMA_BB(x, a_fft, b_fft, Diels, shift) = AMA + gamma K_B x + shift x               pcfft.py:160-181
    H_block(x, inv_fft)                   = K_P^-1 x  (preconditioner)                pcfft.py:50-70
    A_block / A_block_kernel, H_block_kernel: the point-wise symbol multiplies        pcfft.py:18-43,91-108

x may be a NumPy array of shape (3n^3, k) / (3n^3,) (uploaded, result downloaded -- the
reference-facing path with host buffers) or a DeviceBlock (stays on the device).  All O(N^3) work
happens in libpcb200.so; see csrc/pcb_operator.cuh for the pass structure.
"""
import ctypes as C
import weakref

import numpy as np

from . import _lib as L
from . import devarray
from .devarray import DeviceBlock
from .discretization import (DielHandle, FourierSymbols, PenaltySymbols, PrecondSymbols, _PenaltyPart, _PrecondPart,
                             penalty_scale)


class Operator:
    """One k-point's operator on one GPU (pcb_op): symbol tables + gamma/shift + dielectric."""

    def __init__(self, a_fft, gamma=0.0, shift=0.0, pshift=None, diel=None, device=None, ctx=None):
        if not isinstance(a_fft, FourierSymbols):
            raise TypeError("a_fft must come from discretization.fft_blocks (FourierSymbols descriptor)")
        if diel is not None and not isinstance(diel, DielHandle):
            raise TypeError("Diels must be a handle from discretization.*_handle, or None for the identity")
        self.a_fft, self.diel = a_fft, diel
        self.N = a_fft.N
        self.ctx = ctx if ctx is not None else (diel.ctx if diel is not None else devarray.get_context(self.N, device))
        if diel is not None and diel.ctx is not self.ctx:
            raise ValueError("dielectric handle lives on another context")
        if diel is not None and diel.n != self.N:
            raise ValueError(f"dielectric handle is for n = {diel.n}, symbols for n = {self.N}")
        self.gamma, self.shift = float(gamma), float(shift)
        self.pshift = float(shift if pshift is None else pshift)
        self._lib = L.lib()
        t = np.ascontiguousarray(a_fft.tables, dtype=np.complex128)
        h = C.c_void_p()
        L.check(self._lib.pcb_op_create(self.ctx.h, t.view(np.float64).ctypes.data_as(L.c_double_p), self.gamma, self.shift,
                                        self.pshift, diel.h if diel is not None else None, C.byref(h)), "pcb_op_create")
        self.h = h
        self._fin = weakref.finalize(self, self._lib.pcb_op_destroy, h)

    def update(self, a_fft, gamma, shift, pshift=None):
        """Re-target the operator to another k-point (same grid and dielectric) without reallocating."""
        self.a_fft, self.gamma, self.shift = a_fft, float(gamma), float(shift)
        self.pshift = float(shift if pshift is None else pshift)
        t = np.ascontiguousarray(a_fft.tables, dtype=np.complex128)
        L.check(self._lib.pcb_op_update(self.h, t.view(np.float64).ctypes.data_as(L.c_double_p), self.gamma, self.shift,
                                        self.pshift, self.diel.h if self.diel is not None else None), "pcb_op_update")

    # -- device-level calls ---------------------------------------------------------------
    def apply_into(self, mode, src, dst):
        """dst_j = op(src_j) on DeviceBlocks (column views welcome)."""
        if src.k != dst.k:
            raise ValueError("column count mismatch")
        if src.k == 0:
            return dst
        L.check(self._lib.pcb_apply(self.h, mode, src.k, L.ptr_array(src.ptrs), L.ptr_array(dst.ptrs)), "pcb_apply")
        return dst

    def apply(self, mode, x, out=None):
        """Functional form used by the drop-in callables: returns a new array of x's kind
        (`out`: optional preallocated host array -- e.g. pinned -- receiving the result of a host-array call).
        Host-array calls stage through cached device blocks (no cudaMalloc/cudaFree of GB-sized blocks per call)."""
        if isinstance(x, DeviceBlock):
            blk, _ = devarray.as_block(self.ctx, x)
            res = DeviceBlock(self.ctx, blk.k, vec=blk.vec)
            self.apply_into(mode, blk, res)
            return res
        x = np.ascontiguousarray(x, dtype=np.complex128)
        vec = x.ndim == 1
        k = 1 if vec else x.shape[1]
        if x.shape[0] != self.ctx.R:
            raise ValueError(f"expected {self.ctx.R} rows, got {x.shape[0]}")
        if self.ctx.slab is not None:
            raise ValueError("host-array calls need a full (non-slab) context")
        y = out if out is not None else np.empty((self.ctx.R, k), dtype=np.complex128)
        y2 = y.reshape(self.ctx.R, k)
        if not y2.flags.c_contiguous or y2.dtype != np.complex128:
            raise ValueError("out must be a C-contiguous complex128 array")
        # H2D / compute / D2H pipeline over column chunks inside the C ABI
        rc = self._lib.pcb_apply_host(self.h, mode, k, x.ctypes.data, k, y2.ctypes.data, k)
        if rc != 0 and b"memory" in self._lib.pcb_last_error().lower() and self.ctx.trim():
            # the staging of the pipeline is a plain cudaMalloc: give the context's cached blocks back and try once more
            rc = self._lib.pcb_apply_host(self.h, mode, k, x.ctypes.data, k, y2.ctypes.data, k)
        L.check(rc, "pcb_apply_host")
        return y.reshape(-1) if (vec and out is None) else y

    def residual(self, x, hx, w, lambdas, precond=True, single=False):
        """w_j = [K_P^-1] (lambda_j x_j - hx_j); returns ||lambda_j x_j - hx_j||_2 (lobpcg.py:394-397,442).
        ``single``: the residual is rounded to complex64 before the preconditioner (lobpcg.py:574-577)."""
        k = x.k
        lam = np.ascontiguousarray(lambdas, dtype=np.float64)
        out = np.empty(k, dtype=np.float64)
        L.check(self._lib.pcb_residual(self.h, (2 if precond else 3) if single else (1 if precond else 0), k, L.ptr_array(x.ptrs), L.ptr_array(hx.ptrs),
                                       L.ptr_array(w.ptrs), lam.ctypes.data_as(L.c_double_p),
                                       out.ctypes.data_as(L.c_double_p)), "pcb_residual")
        return np.sqrt(out)


    def field_energy(self, X):
        """(e_in, e_tot) per column, NumPy arrays: e_tot = Re D^H M D / N^3 = x^H A x and e_in the same sum over the rows in
        Omega_1 (the edge DoFs of the dielectric), with D = FFT3(K_A^H x) -- see pcb_field_energy in include/pcb200.h.
        X: a DeviceBlock on this operator's context (column views welcome) or a host array (3n^3, k) / (3n^3,), uploaded."""
        X, _ = devarray.as_block(self.ctx, X)
        e_in, e_tot = np.zeros(X.k), np.zeros(X.k)
        if X.k:
            L.check(self._lib.pcb_field_energy(self.h, X.k, L.ptr_array(X.ptrs), e_in.ctypes.data_as(L.c_double_p),
                                               e_tot.ctypes.data_as(L.c_double_p)), "pcb_field_energy")
        return e_in, e_tot

    def material_energy(self, X):
        """(k, n_mat) NumPy array: e_m = Re sum over the rows of material m of conj(D_r) E_r / N^3 per column, for an operator
        on a materials dielectric -- see pcb_material_energy in include/pcb200.h.  Row sums are e_tot of field_energy.  X: a
        DeviceBlock on this operator's context (column views welcome) or a host array (3n^3, k) / (3n^3,), uploaded."""
        X, _ = devarray.as_block(self.ctx, X)
        n_mat = len(self.diel.inv_eps) if self.diel is not None and hasattr(self.diel, "inv_eps") else 0
        e = np.zeros((X.k, n_mat))
        if X.k:
            L.check(self._lib.pcb_material_energy(self.h, X.k, L.ptr_array(X.ptrs), n_mat, e.ctypes.data_as(L.c_double_p)),
                    "pcb_material_energy")
        return e

    def band_velocity(self, X):
        """(V, xx, xax) of the columns of X (n <= 32): V (3, n, n) complex, V[d] = X^H (dA/dalpha_d) X (Hermitian), xx[j] =
        x_j^H x_j, xax[j] = Re x_j^H A x_j -- see pcb_band_velocity in include/pcb200.h.  dA/dalpha_d comes from
        FourierSymbols.dtables of this operator's symbols.  X: a DeviceBlock on this operator's context (column views welcome)
        or a host array (3n^3, k) / (3n^3,), uploaded."""
        X, _ = devarray.as_block(self.ctx, X)
        n = X.k
        V = np.zeros((3, n, n), dtype=np.complex128)
        xx, xax = np.zeros(n), np.zeros(n)
        if n:
            dt = np.ascontiguousarray(self.a_fft.dtables, dtype=np.complex128)
            L.check(self._lib.pcb_band_velocity(self.h, n, L.ptr_array(X.ptrs), dt.view(np.float64).ctypes.data_as(L.c_double_p),
                                                V.ctypes.data, xx.ctypes.data_as(L.c_double_p),
                                                xax.ctypes.data_as(L.c_double_p)), "pcb_band_velocity")
        return V, xx, xax

    def update_resid(self, m, n_loc, s_loc, hs_loc, P, HP, E, lambdas, W):
        """_sep_update_after_rr (lobpcg.py:1248-1270) fused with the next iteration's residual, norms and preconditioner
        (:394-397,442): returns ||lambda_j x_j - hx_j||_2 of the UPDATED X, HX; W receives K_P^-1 of those residuals."""
        lam = np.ascontiguousarray(lambdas, dtype=np.float64)
        out = np.empty(m, dtype=np.float64)
        L.check(self._lib.pcb_update_resid(self.h, m, n_loc, L.ptr_array(s_loc.ptrs), L.ptr_array(hs_loc.ptrs), L.ptr_array(P.ptrs),
                                           L.ptr_array(HP.ptrs), E.ctypes.data, lam.ctypes.data_as(L.c_double_p), L.ptr_array(W.ptrs),
                                           out.ctypes.data_as(L.c_double_p)), "pcb_update_resid")
        return np.sqrt(out)


    def update_resid_start(self, m, n_loc, s_loc, hs_loc, P, HP, E, lambdas, W):
        """update_resid without waiting for the result: returns a callable that delivers the norms (host work overlaps the GPU)."""
        lam = np.ascontiguousarray(lambdas, dtype=np.float64)
        keep = (E, lam, s_loc, hs_loc)      # alive until the kernels have been enqueued (the C side stages E synchronously)
        L.check(self._lib.pcb_update_resid_start(self.h, m, n_loc, L.ptr_array(s_loc.ptrs), L.ptr_array(hs_loc.ptrs), L.ptr_array(P.ptrs),
                                                 L.ptr_array(HP.ptrs), E.ctypes.data, lam.ctypes.data_as(L.c_double_p),
                                                 L.ptr_array(W.ptrs)), "pcb_update_resid_start")

        def wait():
            out = np.empty(m, dtype=np.float64)
            L.check(self._lib.pcb_update_resid_wait(self.h, m, out.ctypes.data_as(L.c_double_p)), "pcb_update_resid_wait")
            return np.sqrt(out)
        return wait


class OperatorCallable:
    """What pc_mfd_handle returns instead of a lambda: callable like the reference's closures, and
    recognisable by the solver so that it can run the fused device path."""

    def __init__(self, op, mode):
        self.op, self.mode = op, mode

    def __call__(self, x, out=None):
        return self.op.apply(self.mode, x, out=out)


def _sym_consistency(a_fft, b_fft=None, inv_fft=None):
    """gamma and the preconditioner shift implied by descriptor scalings (see discretization.py)."""
    fa = a_fft.factor
    gamma = 0.0
    if b_fft is not None:
        if isinstance(b_fft, PenaltySymbols):
            sb, fb = b_fft.scale, b_fft.a.factor
        else:
            sb, fb = penalty_scale(b_fft), b_fft[0].parent.a.factor
            if abs(b_fft[1].scale * b_fft[1].parent.scale - sb) > 1e-15 * abs(sb):
                raise ValueError("b_fft[0] and b_fft[1] carry different scalings")
        gamma = sb * (fb / fa) ** 2
    pshift = None
    if inv_fft is not None:
        if isinstance(inv_fft, PrecondSymbols):
            par, si = inv_fft, inv_fft.scale
        else:
            par, si = inv_fft[0].parent, inv_fft[0].scale * inv_fft[0].parent.scale
        r = (fa / par.a.factor) ** 2
        if abs(si * r - 1.0) > 1e-12:
            raise ValueError("inv_fft scaling is inconsistent with a_fft (expected inv_fft * SCAL^2 with a_fft / SCAL)")
        pshift = par.shift * r
        gamma_p = par.pnt
        if b_fft is not None and abs(gamma_p - gamma) > 1e-12 * max(1.0, abs(gamma)):
            raise ValueError("inv_fft was built with a different penalty than b_fft")
        if b_fft is None:
            gamma = gamma_p
    return gamma, pshift


def build_operator(a_fft, b_fft, Diels, inv_fft, shift=0.0, device=None):
    gamma, pshift = _sym_consistency(a_fft, b_fft, inv_fft)
    return Operator(a_fft, gamma, shift, pshift if pshift is not None else shift, Diels, device=device)


# ---------------------------------------------------------------------------------------------
# Reference-named functions
# ---------------------------------------------------------------------------------------------
def AMA(x_in, D_A, Diels, h_handle=None, a_handle=None):
    """K_A IFFT3( M FFT3( K_A^H x ) )  (pcfft.py:130-158)."""
    return Operator(D_A, 0.0, 0.0, 0.0, Diels).apply(L.APPLY_A, x_in)


def AMA_BB(x_in, D_A, D_B, Diels, shift=0, h_handle=None, a_handle=None):
    """(A M A^H + gamma B^H B + shift) x  (pcfft.py:160-181)."""
    gamma, _ = _sym_consistency(D_A, D_B, None)
    return Operator(D_A, gamma, shift, shift, Diels).apply(L.APPLY_H, x_in)


def H_block(x, DIAG):
    """Hermitian 3x3 block multiply (pcfft.py:50-70): DIAG = inv_fft -> K_P^-1 x; DIAG = b_fft -> gamma K_B x."""
    first = DIAG if isinstance(DIAG, (PrecondSymbols, PenaltySymbols)) else DIAG[0]
    if isinstance(first, (PrecondSymbols, _PrecondPart)):
        par = first if isinstance(first, PrecondSymbols) else first.parent
        gamma, pshift = _sym_consistency(par.a, None, DIAG)
        return Operator(par.a, gamma, 0.0, pshift).apply(L.APPLY_P, x)
    if isinstance(first, (PenaltySymbols, _PenaltyPart)):
        par = first if isinstance(first, PenaltySymbols) else first.parent
        gamma, _ = _sym_consistency(par.a, DIAG, None)
        return Operator(par.a, gamma, 0.0, 0.0).apply(L.APPLY_KB, x)
    raise TypeError("H_block expects b_fft or inv_fft descriptors")


H_block_kernel = H_block


def A_block(x, D):
    """Cross product with the symbol vector (pcfft.py:91-108): D = a_fft -> K_A x; D = -conj(a_fft) -> K_A^H x."""
    mode = L.APPLY_KA if D.kind() == "KA" else L.APPLY_KAH
    base = D.with_alpha(D.alpha)      # strip the conj/neg markers
    return Operator(base, 0.0, 0.0, 0.0).apply(mode, x)


A_block_kernel = A_block
A_block_dim1 = A_block      # the reference's 1-D twins (pcfft.py:72-89,110-124): vectors keep their shape here
H_block_dim1 = H_block


def diel_apply(handle, x):
    """Diels(x): M x in real space (discretization.py:352-453)."""
    if handle._ident_op is None:
        from .discretization import FourierSymbols as FS
        handle._ident_op = Operator(FS(handle.n, 1, np.eye(3)), 0.0, 0.0, 0.0, handle)
    return handle._ident_op.apply(L.APPLY_M, x)


def fftn3(x, n=None, inverse=False, device=None):
    """Batched 3-D DFT of every component/column (cupyx.scipy.fft.fftn/ifftn over axes (0,1,2), pcfft.py:149,151)."""
    if isinstance(x, DeviceBlock):
        ctx = x.ctx
    else:
        n = n or round((np.asarray(x).shape[0] // 3) ** (1 / 3))
        ctx = devarray.get_context(n, device)
    from .discretization import FourierSymbols as FS
    op = Operator(FS(ctx.N, 1, np.eye(3)), 0.0, 0.0, 0.0, None)
    return op.apply(L.APPLY_IFFT if inverse else L.APPLY_FFT, x)


# ---------------------------------------------------------------------------------------------
# Column reductions used by environment.norms / dots and the post-processing
# ---------------------------------------------------------------------------------------------
def _to_device(X):
    if isinstance(X, DeviceBlock):
        return X
    X = np.asarray(X)
    n = round((X.shape[0] // 3) ** (1 / 3))
    if 3 * n ** 3 != X.shape[0]:
        raise ValueError("expected 3 n^3 rows")
    return DeviceBlock.from_host(devarray.get_context(n), X)


def column_dots(X, Y):
    """diag(X^H Y) (environment.dots, environment.py:145-157), reduced on the device."""
    X, Y = _to_device(X), _to_device(Y)
    out = np.empty(X.k, dtype=np.complex128)
    L.check(L.lib().pcb_coldots(X.ctx.h, X.k, L.ptr_array(X.ptrs), L.ptr_array(Y.ptrs), out.ctypes.data), "pcb_coldots")
    return out


def column_norms(X):
    """Column 2-norms (environment.norms, environment.py:131-143)."""
    X = _to_device(X)
    return np.sqrt(column_dots(X, X).real)
