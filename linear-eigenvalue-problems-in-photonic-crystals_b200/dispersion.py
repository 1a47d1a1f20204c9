"""Dispersive materials: lossless permittivity models eps(f) and the self-consistent band iteration.

Frequencies f are those the runners print and record, f = sqrt(lambda) scal / 2 pi (units a / lambda_0).  For band j of a crystal
whose materials have eps_m(f), the self-consistent frequency is the root of

    g_j(f) = f^2 - F_j(f)^2,    F_j(f) = s sqrt(lambda_j(eps_1(f), ..., eps_n(f))),  s = scal / 2 pi,

F_j(f) being the plain solve at the permittivities of f.  By Hellmann-Feynman on the per-material energies (pcb_material_energy),
dlambda_j / deps_m = -lambda_j f_jm / eps_m with f_jm = e_m / e_tot, so

    g_j'(f) = 2 f + F_j^2 sum_m f_jm eps_m'(f) / eps_m(f).

Each lambda_j is non-increasing in every eps_m (Courant-Fischer: M decreases in the Loewner order), and eps_m' > 0 for the lossless
Drude and Lorentz models, so g_j is strictly increasing on an admissible window -- an interval on which every eps_m is finite and
> 0 -- and band j has at most one self-consistent frequency there.  ``self_consistent`` keeps a bracket from the sign of g at
every solve and falls back to bisection when a Newton step leaves it.  The Newton steps are taken on

    h_j(f) = g_j(f) / (f^2 F_j^2) = 1 / F_j^2 - 1 / f^2,    h_j'(f) = sum_m f_jm eps_m'(f) / eps_m(f) / F_j^2 + 2 / f^3,

which has the same root and sign: 1 / F_j^2 ~ eps is smooth at the lower edge of a window above a Drude plasma frequency or a
Lorentz resonance, where eps -> 0 and g has a pole (Newton on g converges only linearly near such an edge).  It takes the solves
as a callback, so a test can drive it with a synthetic lambda(eps).
"""
import math

import numpy as np

__all__ = ["Constant", "Drude", "Lorentz", "as_model", "is_dispersive", "windows", "default_window", "predict", "self_consistent"]


def _positive(name, v):
    v = float(v)
    if not (math.isfinite(v) and v > 0.0):
        raise ValueError(f"{name} = {v} must be finite and > 0")
    return v


class Constant:
    """eps(f) = eps: a material without dispersion."""

    def __init__(self, eps):
        self.eps_inf = _positive("eps", eps)

    def eps(self, f):
        return self.eps_inf + 0.0 * np.asarray(f, dtype=float)

    def deps(self, f):
        return 0.0 * np.asarray(f, dtype=float)

    def windows(self):
        return [(0.0, math.inf)]

    def __repr__(self):
        return f"Constant({self.eps_inf})"


class Drude:
    """Lossless Drude model eps(f) = eps_inf - f_p^2 / f^2 (a metal or plasma above its plasma frequency); eps' = 2 f_p^2 / f^3.
    Admissible for f > f_p / sqrt(eps_inf), where eps > 0."""

    def __init__(self, eps_inf, f_p):
        self.eps_inf, self.f_p = _positive("eps_inf", eps_inf), _positive("f_p", f_p)

    def eps(self, f):
        f = np.asarray(f, dtype=float)
        return self.eps_inf - self.f_p ** 2 / f ** 2

    def deps(self, f):
        f = np.asarray(f, dtype=float)
        return 2.0 * self.f_p ** 2 / f ** 3

    def windows(self):
        return [(self.f_p / math.sqrt(self.eps_inf), math.inf)]

    def __repr__(self):
        return f"Drude({self.eps_inf}, {self.f_p})"


class Lorentz:
    """Lossless Lorentz model eps(f) = eps_inf + sum_k sigma_k f_k^2 / (f_k^2 - f^2) (a polar dielectric near its resonances
    f_k, strengths sigma_k > 0); eps' = sum_k 2 sigma_k f_k^2 f / (f_k^2 - f^2)^2.  eps increases between consecutive poles, so
    the admissible windows are [0, f_1) and, above each pole f_k, the interval from the zero of eps to the next pole (to infinity
    above the last one)."""

    def __init__(self, eps_inf, terms):
        self.eps_inf = _positive("eps_inf", eps_inf)
        self.terms = sorted(((_positive("sigma", s), _positive("f0", f0)) for s, f0 in terms), key=lambda t: t[1])
        if not self.terms:
            raise ValueError("Lorentz needs at least one (sigma, f0) term")
        if len({f0 for _, f0 in self.terms}) != len(self.terms):
            raise ValueError("Lorentz resonances must be distinct")

    def eps(self, f):
        f = np.asarray(f, dtype=float)
        return self.eps_inf + sum(s * f0 ** 2 / (f0 ** 2 - f ** 2) for s, f0 in self.terms)

    def deps(self, f):
        f = np.asarray(f, dtype=float)
        return sum(2.0 * s * f0 ** 2 * f / (f0 ** 2 - f ** 2) ** 2 for s, f0 in self.terms)

    def _zero(self, lo, hi):
        """The zero of eps on (lo, hi), where eps rises from -inf to a positive value (bisection to the last bit)."""
        a, b = lo, hi
        for _ in range(200):
            m = 0.5 * (a + b)
            if m <= a or m >= b:
                break
            if self.eps(m) > 0.0:
                b = m
            else:
                a = m
        return b

    def windows(self):
        poles = [f0 for _, f0 in self.terms]
        out = [(0.0, poles[0])]
        for k, p in enumerate(poles):
            nxt = poles[k + 1] if k + 1 < len(poles) else math.inf
            top = nxt if math.isfinite(nxt) else 2.0 * p
            while not math.isfinite(nxt) and self.eps(top) <= 0.0:
                top *= 2.0
            # just above the pole eps -> -inf; eps > 0 somewhere below the next pole (or as f -> inf, eps -> eps_inf > 0)
            lo = p * (1.0 + 1e-15)
            hi = nxt * (1.0 - 1e-15) if math.isfinite(nxt) else top
            out.append((self._zero(lo, hi), nxt))
        return out

    def __repr__(self):
        return f"Lorentz({self.eps_inf}, {self.terms})"


def as_model(v):
    """A number becomes Constant(v); a model is returned as it is."""
    if isinstance(v, (Constant, Drude, Lorentz)):
        return v
    if hasattr(v, "eps") and hasattr(v, "deps") and hasattr(v, "windows") and hasattr(v, "eps_inf"):
        return v
    return Constant(v)


def is_dispersive(models):
    return any(not isinstance(as_model(m), Constant) for m in models)


def windows(models):
    """Admissible windows of several materials: the intervals on which every model is finite and > 0 (intersections of the
    models' windows), ascending."""
    cur = [(0.0, math.inf)]
    for m in models:
        nxt = []
        for a, b in cur:
            for c, d in as_model(m).windows():
                lo, hi = max(a, c), min(b, d)
                if lo < hi:
                    nxt.append((lo, hi))
        cur = sorted(nxt)
    return cur


def default_window(models):
    """The highest admissible window: above every Drude plasma frequency and Lorentz resonance, where eps < eps_inf."""
    ws = windows(models)
    if not ws:
        raise ValueError("the materials have no common frequency window in which every eps is finite and > 0")
    return ws[-1]


def predict(F, frac, eps_ref, models, window):
    """Start frequencies from one solve at the permittivities eps_ref: with the fields held fixed, lambda scales as
    sum_m f_m eps_ref_m / eps_m, so band j is predicted at the root of f^2 = F_j^2 sum_m f_jm eps_ref_m / eps_m(f) in the window
    (bisection on the models alone; exact in a homogeneous medium).  NaN where F_j is 0 or the prediction has no root there."""
    models = [as_model(m) for m in models]
    lo, hi = float(window[0]), float(window[1])
    top = hi if math.isfinite(hi) else 2.0 * max(lo, 1.0)
    out = np.full(len(F), np.nan)
    for j, (Fj, fj) in enumerate(zip(np.asarray(F, dtype=float), np.asarray(frac, dtype=float))):
        if not (Fj > 0.0) or not np.all(np.isfinite(fj)):
            continue

        def h(f):
            eps = np.array([float(m.eps(f)) for m in models])
            return 1.0 / (Fj * Fj * float(np.sum(fj * eps_ref / eps))) - 1.0 / (f * f)
        a, b = lo + 1e-12 * max(top - lo, 1.0), top * (1.0 - 1e-12) if math.isfinite(hi) else top
        while not math.isfinite(hi) and h(b) < 0.0 and b < 1e12:
            b *= 2.0
        if not (h(a) < 0.0 < h(b)):
            continue
        for _ in range(200):
            m = 0.5 * (a + b)
            if m <= a or m >= b:
                break
            if h(m) < 0.0:
                a = m
            else:
                b = m
        out[j] = 0.5 * (a + b)
    return out


def _clusters(F, degen_tol):
    """Cluster label per band: frequencies agreeing to a relative degen_tol in F^2 (lambda), grouped transitively."""
    lam = np.asarray(F, dtype=float) ** 2
    order = np.argsort(lam, kind="stable")
    labels = np.empty(len(lam), dtype=int)
    cur = 0
    for r, j in enumerate(order):
        if r > 0:
            prev = lam[order[r - 1]]
            if abs(lam[j] - prev) > degen_tol * max(abs(lam[j]), abs(prev)):
                cur += 1
        labels[j] = cur
    return labels


def _inside(f, lo, hi):
    """f moved strictly inside (lo, hi): at the window's edges some eps is 0 or infinite."""
    span = (hi - lo) if math.isfinite(hi) else max(lo, 1.0)
    return min(max(f, lo + 1e-3 * span), hi - 1e-3 * span) if math.isfinite(hi) else max(f, lo + 1e-3 * span)


def self_consistent(solve, models, start, window=None, ftol=1e-7, max_steps=12, degen_tol=1e-6, x0=None, zero=0.0):
    """Self-consistent frequencies of nev bands, g_j(f) = f^2 - F_j(f)^2 = 0, by safeguarded Newton on h_j = 1 / F_j^2 - 1 / f^2
    (see the module docstring).

    solve(f, x0) -> (F, frac, x): F (nev,) the frequencies of a plain solve at eps_m(f) of every material, frac (nev, n_mat) the
    per-material energy fractions e_m / e_tot of those bands, x whatever the next call takes as its warm start (x0 first).
    models: one model (or number) per material, in the order of frac's columns.  start: (nev,) initial frequencies, clamped into
    the window (NaN: its lower edge).  window: (lo, hi), default the highest admissible window of the models.

    Band by band from the lowest: the bands whose F agree with the current band's to a relative degen_tol (in lambda) form a
    cluster that shares one iteration, with the cluster means of 1 / F^2 and of the derivative term (both basis-independent).
    The bracket [lo, hi] shrinks with the sign of g at every solve; a Newton step outside it is replaced by bisection (doubling while
    hi is infinite).  A band stops when |delta f| <= ftol f; one without a bracketed root within max_steps solves gets NaN, and so
    does a band whose F is <= zero at a solve (F = 0 at every eps: the zero modes at Gamma, g = f^2 > 0 has no root).
    Returns a dict: "freq" (nev,), "steps" (nev,) solves spent on each band's cluster, "solves" in all, "x" the last warm start,
    "F" / "frac" of the last solve of each band's cluster (at its own frequency)."""
    models = [as_model(m) for m in models]
    start = np.asarray(start, dtype=float)
    nev = len(start)
    if window is None:
        window = default_window(models)
    wlo, whi = float(window[0]), float(window[1])
    if not wlo < whi:
        raise ValueError(f"window {window} is empty")
    freq = np.full(nev, np.nan)
    steps = np.zeros(nev, dtype=int)
    F_last, frac_last = np.full(nev, np.nan), None
    done = np.zeros(nev, dtype=bool)
    x = x0
    solves = 0
    j = 0
    while j < nev:
        if done[j]:
            j += 1
            continue
        lo, hi = wlo, whi
        f = _inside(lo if np.isnan(start[j]) else start[j], lo, hi)
        cluster = [j]
        conv = False
        for _ in range(max_steps):
            F, frac, x = solve(f, x)
            solves += 1
            F, frac = np.asarray(F, dtype=float), np.asarray(frac, dtype=float)
            if frac_last is None:
                frac_last = np.full((nev, frac.shape[1]), np.nan)
            lab = _clusters(F, degen_tol)
            cluster = [k for k in range(j, nev) if lab[k] == lab[j] and not done[k]]
            for k in cluster:
                steps[k] += 1
            eps = np.array([float(m.eps(f)) for m in models])
            deps = np.array([float(m.deps(f)) for m in models])
            if np.all(F[cluster] <= zero):
                F_last[cluster], frac_last[cluster] = F[cluster], frac[cluster]
                break
            # Newton on h = g / (f^2 F^2) = 1 / F^2 - 1 / f^2 (same root and sign): 1 / F^2 is nearly linear in eps, also at a
            # window edge where eps -> 0 and g has a pole
            iF2 = 1.0 / F[cluster] ** 2
            g = float(iF2.mean()) - 1.0 / (f * f)
            dg = float(np.mean(iF2 * (frac[cluster] @ (deps / eps)))) + 2.0 / f ** 3
            if g < 0.0:
                lo = f
            else:
                hi = f
            fn = f - g / dg if dg > 0.0 else math.nan
            F_last[cluster], frac_last[cluster] = F[cluster], frac[cluster]
            if abs(fn - f) <= ftol * f:              # also a step below one ulp (fn == f: on the root)
                conv = True
                f = fn
                break
            if not (lo < fn < hi):
                fn = 0.5 * (lo + hi) if math.isfinite(hi) else 2.0 * max(f, lo)
            f = _inside(fn, wlo, whi) if not (wlo < fn < whi) else fn
        for k in cluster:
            freq[k] = f if conv else np.nan
            done[k] = True
        j += 1
    return {"freq": freq, "steps": steps, "solves": solves, "x": x, "F": F_last, "frac": frac_last}
