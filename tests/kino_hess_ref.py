"""tests/kino_hess_ref.py -- TEST INFRASTRUCTURE ONLY (CPU oracle of the kino-dynamic Lagrangian Hessian).

The exact Hessian of lam_f f(x) + lam_g' g(x) for the kino-dynamic NLP restated in oracle/kino_ref.py: second
derivatives of oracle/kino_ref.py:knot_rows (closed-form kinematics, literal=False) by forward-mode dual numbers with
complex components, which share no code with the product's second-order type (kino_knot.cuh: Dual2)."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
import kino_ref as kr  # noqa: E402


class _HyperDual:
    """Forward-mode dual number with complex components, for second derivatives without subtractive cancellation: the
    value v[j] carries a complex step i h e_j on input j, the dual part d[j, i] the tangent of input i.  Every direction
    j and every tangent i are carried at once (v [n], d [n, n]), so one pass of knot_rows(..., literal=False) over an
    object array of these gives Im d[j, i] / h = d2 / dz_j dz_i.  Operators return NotImplemented for ndarray operands,
    so that numpy broadcasts down to the elements."""
    __slots__ = ("v", "d")

    def __init__(self, v, d):
        self.v, self.d = v, d

    def __add__(self, o):
        if isinstance(o, np.ndarray):
            return NotImplemented
        if isinstance(o, _HyperDual):
            return _HyperDual(self.v + o.v, self.d + o.d)
        return _HyperDual(self.v + o, self.d)

    __radd__ = __add__

    def __neg__(self):
        return _HyperDual(-self.v, -self.d)

    def __sub__(self, o):
        if isinstance(o, np.ndarray):
            return NotImplemented
        return self + (-o)

    def __rsub__(self, o):
        if isinstance(o, np.ndarray):
            return NotImplemented
        return (-self) + o

    def __mul__(self, o):
        if isinstance(o, np.ndarray):
            return NotImplemented
        if isinstance(o, _HyperDual):
            return _HyperDual(self.v * o.v, self.d * o.v[:, None] + self.v[:, None] * o.d)
        return _HyperDual(self.v * o, self.d * o)

    __rmul__ = __mul__

    def __truediv__(self, o):
        if isinstance(o, np.ndarray):
            return NotImplemented
        if isinstance(o, _HyperDual):
            q = self.v / o.v
            return _HyperDual(q, (self.d - q[:, None] * o.d) / o.v[:, None])
        return _HyperDual(self.v / o, self.d / o)

    def __rtruediv__(self, o):
        if isinstance(o, np.ndarray):
            return NotImplemented
        q = o / self.v
        return _HyperDual(q, -(q / self.v)[:, None] * self.d)

    def sin(self):
        return _HyperDual(np.sin(self.v), np.cos(self.v)[:, None] * self.d)

    def cos(self):
        return _HyperDual(np.cos(self.v), -np.sin(self.v)[:, None] * self.d)

    def tan(self):
        t = np.tan(self.v)
        return _HyperDual(t, (1.0 + t * t)[:, None] * self.d)


def knot_hess(pb, k, z, lam, last, h=1e-30):
    """Exact Hessian [n, n] of lam' (rows of knot k) in the knot-local inputs z (72; 60 for the last knot): a dual
    number seeded on input i, a complex step on input j (_HyperDual)."""
    z = np.asarray(z, dtype=np.float64)
    n = z.size
    zz = np.empty(n, dtype=object)
    for e in range(n):
        v = np.full(n, z[e], dtype=np.complex128)
        v[e] += 1j * h
        d = np.zeros((n, n), dtype=np.complex128)
        d[:, e] = 1.0
        zz[e] = _HyperDual(v, d)
    rows = kr.knot_rows(pb, k, zz[0:12], zz[48:60], zz[12:24], zz[24:48], None if last else zz[60:72], literal=False)
    L = sum(float(l) * r for l, r in zip(lam, rows) if l != 0.0)
    if not isinstance(L, _HyperDual):
        return np.zeros((n, n))
    return L.d.imag / h


def hess_exact(pb, x, lam_f, lam_g, QN, Xref, pattern=None):
    """Exact Hessian of the Lagrangian lam_f f(x) + lam_g' g(x) (tests only), f = (X_N - Xref)' QN (X_N - Xref) the
    terminal cost (Xref does not enter the Hessian), from the 72 x 72 (60 x 60 for the last knot) knot-local blocks of
    knot_hess plus 2 lam_f QN on the diagonal of X_{N-1}.  Dense [nx, nx], or with pattern = (colind, row) (CCS, upper
    triangle) the value array at that pattern.  lam_f / lam_g None: zero."""
    N = pb["N"]
    d = kr.dims(N)
    x = np.asarray(x, dtype=np.float64)
    H = np.zeros((d["nx"], d["nx"]))
    if lam_g is not None:
        lam_g = np.asarray(lam_g, dtype=np.float64)
        for k in range(N - 1):
            last = k == N - 2
            cols = [kr.knot_col(N, k, v) for v in range(60 if last else 72)]
            base = 48 + 141 * k
            H[np.ix_(cols, cols)] += knot_hess(pb, k, x[cols], lam_g[base:base + (117 if last else 141)], last)
    if lam_f is not None:
        xo = 12 * (N - 1)
        H[np.arange(xo, xo + 12), np.arange(xo, xo + 12)] += 2.0 * float(lam_f) * np.asarray(QN, dtype=np.float64)
    if pattern is None:
        return H
    colind, row = pattern
    col = np.repeat(np.arange(d["nx"]), np.diff(colind))
    return H[row, col]
