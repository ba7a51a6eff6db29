"""Independent numpy restatement of the two variant NLPs that the solver poses besides landingCtrller_IPOPT.
TEST INFRASTRUCTURE.

Written from the reference's formulation, not from oracle/ip_ref.c or the CUDA code:
 * formulation 1, the fixed contact schedule of quadruped_SRBM_NLP.m:84-176: running cost
   sum_k dt_k ((X_k - Xref_k)' QX (X_k - Xref_k) + f_k' Qf f_k) (:85-92), f_z <= cs f_max (:148), cs c_z = 0 (:154),
   cs (c+ - c) = 0 (:155-158), no terminal rows (:105-108 are commented out);
 * the "CCC" problem of generate_quadruped_SRBM_CCC.m: formulation 0's rows with the running GRF cost (:80-91) and a
   kinematic box of other half-widths (:169-176).
The rows shared with formulation 0 come from the oracle (oracle/srb_ref.c, pinned to the reference C).  Rows keep
formulation 0's layout.  A row that is not a constraint of the variant ("free": the terminal rows and the unused rows of
formulation 1, and a schedule row whose cs is 0, which reads 0 = 0) has g = 0, a zero Jacobian row, infinite bounds,
and its multiplier must be 0.
"""
import numpy as np

from oracle_lib import Oracle

EQ, INEQ, FREE = 0, 1, 2

_ORACLES = {}


def oracle(N):
    if N not in _ORACLES:
        _ORACLES[N] = Oracle(N)
    return _ORACLES[N]


def leg_row(N, k, l):
    """first row of leg l in knot k's block: c_z (formulation 0) / cs c_z (formulation 1)"""
    return 36 + 104 * k + 16 + (6 if k == N - 2 else 12) * l


def kin_row(N, k, l):
    """first of the three kinematic-box rows of leg l in knot k"""
    return leg_row(N, k, l) + (2 if k == N - 2 else 8)


def c_var(N, k, i):
    return 12 * N + 24 * k + i


def f_var(N, k, i):
    return 12 * N + 24 * k + 12 + i


class VariantNLP:
    """The NLP at parameter vector p (built by the oracle's build_p_x0).  cs [N-1, 4] of 0 / 1 selects formulation 1,
    None formulation 0.  Qf [3] per force component, QX [12] per state, kin_box = (kx, ky, kz) half-widths."""

    def __init__(self, N, p, cs=None, Qf=(0.0, 0.0, 0.0), QX=None, kin_box=(0.15, 0.15, 0.30)):
        self.N = N
        self.o = o = oracle(N)
        self.p = np.ascontiguousarray(p, dtype=np.float64)
        self.cs = None if cs is None else np.asarray(cs, dtype=np.float64).reshape(N - 1, 4)
        self.Qf = np.tile(np.asarray(Qf, dtype=np.float64), 4)
        self.QX = np.zeros(12) if QX is None else np.asarray(QX, dtype=np.float64)
        self.kin_box = tuple(float(v) for v in kin_box)
        self.dt = self.p[o.off["o_dt"]:o.off["o_dt"] + N - 1]
        self.Xref = self.p[:12 * (N - 1)].reshape(N - 1, 12)
        self.lb, self.ub = self._bounds()
        self.kind = np.where(self.lb == self.ub, EQ, np.where(np.isinf(self.lb) & np.isinf(self.ub), FREE, INEQ))

    # ---- rows
    def _replaced_rows(self):
        """(row, what, k, l, a) of every row that formulation 1 restates: what = 'cz' (cs c_z of knot k, leg l), 'ns'
        (cs (c+ - c) of axis a) or 'free'"""
        N, out = self.N, [(r, "free", 0, 0, 0) for r in range(12, 36)]
        for k in range(N - 1):
            for l in range(4):
                L = leg_row(N, k, l)
                out.append((L, "cz", k, l, 0))
                out.append((L + 1, "free", k, l, 0))
                if k < N - 2:
                    for a in range(3):
                        out.append((L + 2 + a, "ns", k, l, a))
                        out.append((L + 5 + a, "free", k, l, a))
        return out

    def _bounds(self):
        N, o = self.N, self.o
        lb, ub = o.bounds(self.p)
        kx, ky, kz = self.kin_box
        for k in range(N - 1):
            for l in range(4):
                K = kin_row(N, k, l)
                lb[K:K + 3] = (-kx, -ky, -kz)
                ub[K:K + 3] = (kx, ky, 0.0)
        if self.cs is not None:
            f_max = self.p[o.off["o_fmax"]]
            for k in range(N - 1):
                ub[36 + 104 * k + 12:36 + 104 * k + 16] = self.cs[k] * f_max
            for r, what, k, l, _ in self._replaced_rows():
                on = what != "free" and self.cs[k, l] != 0
                lb[r], ub[r] = (0.0, 0.0) if on else (-np.inf, np.inf)
        return lb, ub

    def g(self, x):
        _, g = self.o.g(x, self.p)
        if self.cs is not None:
            N = self.N
            for r, what, k, l, a in self._replaced_rows():
                if what == "cz":
                    g[r] = self.cs[k, l] * x[c_var(N, k, 3 * l + 2)]
                elif what == "ns":
                    g[r] = self.cs[k, l] * (x[c_var(N, k + 1, 3 * l + a)] - x[c_var(N, k, 3 * l + a)])
                else:
                    g[r] = 0.0
        return g

    def jac(self, x):
        """dense [m, nx]"""
        o, N = self.o, self.N
        _, _, J = o.jac_g(x, self.p)
        colind, row = o.spJ[2:2 + o.nx + 1], o.spJ[2 + o.nx + 1:]
        D = np.zeros((o.m, o.nx))
        for c in range(o.nx):
            D[row[colind[c]:colind[c + 1]], c] = J[colind[c]:colind[c + 1]]
        if self.cs is not None:
            for r, what, k, l, a in self._replaced_rows():
                D[r] = 0.0
                if what == "cz":
                    D[r, c_var(N, k, 3 * l + 2)] = self.cs[k, l]
                elif what == "ns":
                    D[r, c_var(N, k, 3 * l + a)] = -self.cs[k, l]
                    D[r, c_var(N, k + 1, 3 * l + a)] = self.cs[k, l]
        D[self.kind == FREE] = 0.0
        return D

    # ---- cost
    def cost(self, x):
        """(f, grad f): the oracle's terminal cost plus sum_k dt_k (sum_j Qf[j%3] f_kj^2 + sum_i QX_i (X_ki - Xref_ki)^2)"""
        N = self.N
        _, f, gr = self.o.grad_f(x, self.p)
        gr = gr.copy()
        F = x[12 * N:].reshape(N - 1, 24)[:, 12:]
        E = x[:12 * (N - 1)].reshape(N - 1, 12) - self.Xref
        h = self.dt[:, None]
        f = f + float(np.sum(h * (self.Qf * F * F))) + float(np.sum(h * (self.QX * E * E)))
        gr[12 * N:].reshape(N - 1, 24)[:, 12:] += 2.0 * h * self.Qf * F
        gr[:12 * (N - 1)] += (2.0 * h * self.QX * E).ravel()
        return f, gr

    # ---- certificate
    def kkt(self, x, lam):
        """(f, viol, stat, comp, max |lam| on free rows) at (x, lam), with the definitions of
        test_gpu_solve.py::_kkt_certificate: viol = max over the rows that are constraints of max(lb - g, g - ub);
        stat = max |grad f + J' lam|; comp = max over inequality rows of min(|lam| dist(g, nearest finite bound), |lam|)."""
        f, gf = self.cost(x)
        g = self.g(x)
        J = self.jac(x)
        on = self.kind != FREE
        viol = float(np.max(np.maximum(self.lb - g, g - self.ub)[on]))
        stat = float(np.max(np.abs(gf + J.T @ lam)))
        ineq = self.kind == INEQ
        dl = np.where(np.isfinite(self.lb), g - self.lb, np.inf)
        du = np.where(np.isfinite(self.ub), self.ub - g, np.inf)
        with np.errstate(invalid="ignore"):
            c = np.minimum(np.abs(lam) * np.minimum(dl, du), np.abs(lam))
        comp = float(np.max(np.where(ineq, c, 0.0)))
        free = float(np.max(np.abs(lam[~on]), initial=0.0))
        return f, viol, stat, comp, free


def from_drop(N, pb, drop, **kw):
    """VariantNLP of the scenario `drop` [12] under the oracle problem `pb` (p built as the reference's callers build it)"""
    p, _ = oracle(N).build_p_x0(pb, drop[:6], drop[6:])
    return VariantNLP(N, p, **kw)


def ballistic_schedule_dt(dt, z0, z_touch=0.28):
    """landing_controller_b200.ballistic_schedule on the knot spacings dt [N-1]: all legs in flight while the body,
    falling freely from z0 (explicit Euler steps), is above z_touch, then stance.  [N-1, 4]"""
    z, v = float(z0), 0.0
    cs = np.ones((len(dt), 4), dtype=np.int32)
    for k, h in enumerate(dt):
        if z > z_touch:
            cs[k] = 0
        z, v = z + v * h, v - 9.81 * h
    return cs


def alternating_dt(N, T):
    """short / long knot spacings (1 : 3) summing to T: the running-cost weight dt_k then differs from dt_(k+1) by a
    factor 3 at every knot, so a running-cost term weighted with the wrong step is visible"""
    w = np.where(np.arange(N - 1) % 2 == 0, 1.0, 3.0)
    return T * w / w.sum()
