"""CPU restatement of the interior-point solve of the kino-dynamic NLP (tests only; the library's
landing_kino_solve_batch), written from oracle/ip_ref.c:ip_solve_ws -- not from the CUDA driver.

Functions come from the oracle: g = oracle/kino_ref.py:eval_g, J = kino_ref.jac_exact (complex step), W =
tests/kino_hess_ref.py:hess_exact, the terminal cost in numpy.  The Newton direction and delta_w come from the host build
of landing_controller_b200/csrc/kino_step.cuh (tests/hostcheck/kino_step_host.cpp), which tests/test_kino_step_host.py
certifies against a dense solve of the full, unreduced system.  Everything else -- relaxed bounds, init_slacks, IPOPT's
scaled error E0, the termination test, the monotone barrier update, tau, the filter with switching condition and
Armijo test, the jamming watchdog, re-centring, the accept step with the kappa_sigma clamp -- is restated here.

`certificate` checks a returned point against the oracle alone: violation of the original bounds, the scaled
stationarity error of grad f + J' y, and complementarity."""
import ctypes
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import kino_ref as kr  # noqa: E402
from kino_hess_ref import hess_exact  # noqa: E402

_dp = ctypes.POINTER(ctypes.c_double)
_lp = ctypes.POINTER(ctypes.c_longlong)
QN = np.array([0, 0, 100, 10, 10, 0, 10, 10, 10, 10, 10, 10.0])
XREF = np.array([0, 0, 0.25, 0, 0, 0, 0, 0, 0, 0, 0, 0.0])
MAXFILTER = 64
CONVERGED, MAX_ITER, LINESEARCH_FAIL, NAN, FACTOR_FAIL = 0, 1, 2, 3, 4


def build_harness(tmpdir):
    so = os.path.join(str(tmpdir), "libkino_step_host.so")
    src = os.path.join(ROOT, "tests", "hostcheck", "kino_step_host.cpp")
    subprocess.check_call(["/usr/bin/g++", "-O1", "-std=c++17", "-fPIC", "-shared", src, "-o", so])
    return ctypes.CDLL(so)


def options(**kw):
    """landing_options_default (include/landing_b200.h) as a dict."""
    o = dict(max_iter=3000, tol=1e-4, constr_viol_tol=1e-3, dual_inf_tol=1.0, compl_inf_tol=1e-4, mu_init=0.1,
             bound_push=0.5, bound_frac=0.5, bound_relax_factor=1e-6, jam_iters=5, jam_alpha=0.02, max_restarts=8,
             restart_mu=0.0)
    o.update(kw)
    return o


def eq_rows(N):
    r = np.arange(kr.dims(N)["m"])
    return (r < 24) | ((r >= 48) & ((r - 48) % 141 < 12))


def drop_problem(N, drop):
    """The oracle problem, bounds and reference-trajectory guess of one drop (generate_landingCtrller_KNITRO.m:232-286,
    as landing_kino_setup_batch computes them with x_srb = NULL)."""
    pb = kr.default_problem(N)
    q0, qd0 = drop[:6], drop[6:]
    R = kr.rpy_to_rot_xyz(q0[3:6])
    vb = R.T @ qd0[3:6]
    pb["kin_box"] = np.array([kr.kin_box_limits(vb[0], "x"), kr.kin_box_limits(vb[1], "y")])
    ss = np.array([[1, -1, 1], [1, 1, 1], [-1, -1, 1], [-1, 1, 1.0]])
    c_init = np.concatenate([q0[:3] + R @ (ss[l] * np.array([0.2, 0.15, -0.3])) for l in range(4)])
    lbg, ubg = kr.bounds(pb, q0, qd0, c_init)
    q_ref = np.array([0, 0, 0.25, 0, 0, 0.0])
    X = np.zeros((N, 12))
    for k in range(N):
        t = k / (N - 1)
        X[k, :6] = q0 + (q_ref - q0) * t
        X[k, 6:] = qd0 * (1 - t)
    U = np.zeros((N - 1, 24))
    for k in range(N - 1):
        Rk = kr.rpy_to_rot_xyz(X[k, 3:6])
        U[k, :12] = np.concatenate([X[k, :3] + Rk @ (ss[l] * np.array([0.2, 0.2, -0.3])) for l in range(4)])
    jg = np.tile([0.0, -np.pi / 4, np.pi / 2], 4 * (N - 1))
    return pb, lbg, ubg, np.concatenate([X.ravel(), jg, U.ravel()])


def cost(x, N):
    d = x[12 * (N - 1):12 * N] - XREF
    gf = np.zeros_like(x)
    gf[12 * (N - 1):12 * N] = 2.0 * QN * d
    return float(np.sum(QN * d * d)), gf


class Problem:
    """Oracle evaluations at the library's CCS patterns (jsp, hsp: the full CasADi CCS arrays)."""

    def __init__(self, pb, jsp, hsp):
        self.pb, self.N = pb, pb["N"]
        self.jsp, self.hsp = np.ascontiguousarray(jsp, np.int64), np.ascontiguousarray(hsp, np.int64)
        nx = int(jsp[1])
        self.jpat = (jsp[2:2 + nx + 1], jsp[2 + nx + 1:])
        self.hpat = (hsp[2:2 + nx + 1], hsp[2 + nx + 1:])

    def g(self, x):
        return kr.eval_g(self.pb, x)

    def jac(self, x):
        return kr.jac_exact(self.pb, x, self.jpat)

    def hess(self, x, y):
        return hess_exact(self.pb, x, 1.0, y, QN, XREF, self.hpat)


def host_step(h, P, jv, hv, gf, g, s, y, zL, zU, lb, ub, mu, dw_last):
    N = P.N
    nx, m = kr.dims(N)["nx"], kr.dims(N)["m"]
    vec = [np.ascontiguousarray(v, dtype=np.float64) for v in (g, s, y, zL, zU, lb, ub)]
    outs = [np.full(nx, np.nan)] + [np.full(m, np.nan) for _ in range(4)]
    res = np.full(5, np.nan)
    vp = (_dp * 7)(*[v.ctypes.data_as(_dp) for v in vec])
    op = (_dp * 5)(*[o.ctypes.data_as(_dp) for o in outs])
    jv, hv, gf = (np.ascontiguousarray(a, np.float64) for a in (jv, hv, gf))
    rc = h.kino_step_host(ctypes.c_int(N), P.jsp.ctypes.data_as(_lp), P.hsp.ctypes.data_as(_lp), jv.ctypes.data_as(_dp),
                          hv.ctypes.data_as(_dp), gf.ctypes.data_as(_dp), vp, ctypes.c_double(mu),
                          ctypes.c_double(dw_last), ctypes.c_double(0.5), op, res.ctypes.data_as(_dp))
    assert rc == 0
    return outs, res[0], int(res[2])


def init_slacks(g, lb, ub, eq, o, mu):
    """ip_ref.c init_slacks."""
    m = g.size
    s, y, zL, zU = np.zeros(m), np.zeros(m), np.zeros(m), np.zeros(m)
    for i in range(m):
        if eq[i]:
            continue
        lo, up = lb[i], ub[i]
        sv = g[i]
        if np.isfinite(lo) and np.isfinite(up):
            pL = min(o["bound_push"] * max(1.0, abs(lo)), o["bound_frac"] * (up - lo))
            pU = min(o["bound_push"] * max(1.0, abs(up)), o["bound_frac"] * (up - lo))
            sv = min(max(sv, lo + pL), up - pU)
        elif np.isfinite(lo):
            sv = max(sv, lo + o["bound_push"] * max(1.0, abs(lo)))
        elif np.isfinite(up):
            sv = min(sv, up - o["bound_push"] * max(1.0, abs(up)))
        s[i] = sv
        if np.isfinite(lo):
            zL[i] = mu / (sv - lo)
        if np.isfinite(up):
            zU[i] = mu / (up - sv)
        y[i] = zU[i] - zL[i]
    return s, y, zL, zU


def solve(h, P, lbo, ubo, x0, o, log=None):
    """ip_ref.c ip_solve_ws on the kino-dynamic NLP.  Returns a dict: x, y, f, status, iters, restarts.  log (a list):
    one dict per accepted trial (mu, alpha, the current theta / phi / dphi, theta_min / theta_max, the trial's theta /
    phi, a copy of the filter it was tested against, ftype) and one per re-centring."""
    N = P.N
    m = lbo.size
    eq = eq_rows(N)
    fl, fu = np.isfinite(lbo) & ~eq, np.isfinite(ubo) & ~eq
    lb, ub = lbo.copy(), ubo.copy()
    lb[fl] -= o["bound_relax_factor"] * np.maximum(1.0, np.abs(lbo[fl]))
    ub[fu] += o["bound_relax_factor"] * np.maximum(1.0, np.abs(ubo[fu]))
    x = np.array(x0, dtype=np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        g = P.g(x)
    f, _ = cost(x, N)
    mu = o["mu_init"]
    s, y, zL, zU = init_slacks(g, lb, ub, eq, o, mu)
    filt = []
    theta0, dw_last = -1.0, 0.0
    status, it, restarts, tiny = MAX_ITER, 0, 0, 0
    ineq = ~eq
    while True:
        with np.errstate(invalid="ignore", over="ignore"):
            jv, hv = P.jac(x), P.hess(x, y)
            _, gf = cost(x, N)
            col = np.repeat(np.arange(x.size), np.diff(P.jpat[0]))
            gradL = gf.copy()
            np.add.at(gradL, col, jv * y[P.jpat[1]])
        # assemble's error pieces
        nb = int(fl.sum() + fu.sum())
        rs = np.where(ineq, -y, 0.0) - np.where(fl, zL, 0.0) + np.where(fu, zU, 0.0)
        dL, dU = np.where(fl, s - lb, 0.0), np.where(fu, ub - s, 0.0)
        c0 = max(np.max(np.where(fl, np.abs(zL * dL), 0.0)), np.max(np.where(fu, np.abs(zU * dU), 0.0)))
        zsum = float(np.sum(np.where(fl, zL, 0.0)) + np.sum(np.where(fu, zU, 0.0)))
        ysum = float(np.sum(np.abs(y)))
        prim = max(np.max(np.abs(g[eq] - lb[eq])), np.max(np.abs(g[ineq] - s[ineq])))
        dual = max(np.max(np.abs(rs[ineq])), np.max(np.abs(gradL)))
        with np.errstate(invalid="ignore"):
            viol = max(0.0, float(np.max(np.maximum(lbo - g, g - ubo))))
        nan = (np.isnan(f) or np.isnan(g).any() or np.isnan(y).any() or np.isnan(lbo).any() or np.isnan(ubo).any()
               or np.isnan(s[ineq]).any() or np.isnan(zL[fl]).any() or np.isnan(zU[fu]).any() or np.isnan(gradL).any())
        s_d = max(100.0, (ysum + zsum) / (m + nb)) / 100.0
        s_c = max(100.0, zsum / max(nb, 1)) / 100.0
        E0 = max(dual / s_d, prim, c0 / s_c)
        if nan or not np.isfinite(E0) or not np.isfinite(f):
            status = NAN
            break
        if E0 <= o["tol"] and dual <= o["dual_inf_tol"] and viol <= o["constr_viol_tol"] and c0 <= o["compl_inf_tol"]:
            status = CONVERGED
            break
        if it == o["max_iter"]:
            status = MAX_ITER
            break

        def cmu_at(mu_):
            return max(np.max(np.where(fl, np.abs(zL * dL - mu_), 0.0)), np.max(np.where(fu, np.abs(zU * dU - mu_), 0.0)))
        cmu = cmu_at(mu)
        changed = False
        while True:
            Emu = max(dual / s_d, prim, cmu / s_c)
            if not (Emu <= 10.0 * mu) or mu <= o["tol"] / 10.0 * 1.0000001:
                break
            mu = max(o["tol"] / 10.0, min(0.2 * mu, mu ** 1.5))
            changed = True
            cmu = cmu_at(mu)
        if changed:
            filt = []
        tau = max(0.99, 1.0 - mu)
        (dx, ds, dy, dzL, dzU), dw, st = host_step(h, P, jv, hv, gf, g, s, y, zL, zU, lb, ub, mu, dw_last)
        if st != 0:
            status = NAN if st == 5 else FACTOR_FAIL
            break
        dw_last = dw
        # fraction to the boundary
        a_pr, a_du = 1.0, 1.0
        for i in np.flatnonzero(fl):
            if ds[i] < 0:
                a_pr = min(a_pr, -tau * (s[i] - lb[i]) / ds[i])
            if dzL[i] < 0:
                a_du = min(a_du, -tau * zL[i] / dzL[i])
        for i in np.flatnonzero(fu):
            if ds[i] > 0:
                a_pr = min(a_pr, tau * (ub[i] - s[i]) / ds[i])
            if dzU[i] < 0:
                a_du = min(a_du, -tau * zU[i] / dzU[i])

        def merit(f_, g_, s_):
            th = float(np.sum(np.abs(g_[eq] - lb[eq])) + np.sum(np.abs(g_[ineq] - s_[ineq])))
            with np.errstate(invalid="ignore", divide="ignore"):
                ph = f_ - mu * float(np.sum(np.log(s_[fl] - lb[fl]))) - mu * float(np.sum(np.log(ub[fu] - s_[fu])))
            return ph, th
        phi, theta = merit(f, g, s)
        if theta0 < 0:
            theta0 = theta
        theta_max, theta_min = 1e4 * max(1.0, theta0), 1e-4 * max(1.0, theta0)
        xo = 12 * (N - 1)
        dphi = float(np.dot(gf[xo:xo + 12], dx[xo:xo + 12])) - mu * float(np.sum(ds[fl] / (s[fl] - lb[fl]))) + \
            mu * float(np.sum(ds[fu] / (ub[fu] - s[fu])))
        alpha, accepted, ftype, ls = a_pr, False, 0, 0
        while alpha > 1e-12 * a_pr and ls < 40:
            xt = x + alpha * dx
            stt = np.where(ineq, s + alpha * ds, s)
            with np.errstate(invalid="ignore", over="ignore"):
                gt = P.g(xt)
            ft, _ = cost(xt, N)
            pht, tht = merit(ft, gt, stt)
            fok = all(not (tht >= a and pht >= b) for a, b in filt)
            if np.isfinite(pht) and np.isfinite(tht) and tht <= theta_max and fok:
                sw = theta <= theta_min and dphi < 0 and alpha * (-dphi) ** 2.3 > theta ** 1.1
                if sw:
                    if pht <= phi + 1e-8 * alpha * dphi:
                        accepted, ftype = True, 1
                elif tht <= (1.0 - 1e-5) * theta or pht <= phi - 1e-5 * theta:
                    accepted = True
            if accepted:
                break
            alpha *= 0.5
            ls += 1
        if accepted:
            tiny = tiny + 1 if alpha < o["jam_alpha"] else 0
            if log is not None:
                log.append(dict(it=it, mu=mu, alpha=alpha, restart=False, theta=theta, phi=phi, dphi=dphi,
                                theta_min=theta_min, theta_max=theta_max, theta_trial=tht, phi_trial=pht,
                                filter=list(filt), ftype=ftype))
        if accepted and o["jam_iters"] > 0 and tiny >= o["jam_iters"] and restarts < o["max_restarts"]:
            accepted = False
        if not accepted:
            tiny = 0
            if restarts < o["max_restarts"]:
                restarts += 1
                mu = o["restart_mu"] if o["restart_mu"] > 0 else o["mu_init"]
                s, y, zL, zU = init_slacks(g, lb, ub, eq, o, mu)
                filt = []
                theta0 = -1.0
                if log is not None:
                    log.append(dict(it=it, mu=mu, alpha=None, restart=True))
                it += 1
                continue
            status = LINESEARCH_FAIL
            break
        if not ftype:
            if len(filt) == MAXFILTER:
                filt.pop(0)
            filt.append(((1.0 - 1e-5) * theta, phi - 1e-5 * theta))
        x, g, f = xt, gt, ft
        s = np.where(ineq, s + alpha * ds, s)
        y = y + alpha * dy
        with np.errstate(divide="ignore", invalid="ignore"):
            d = s - lb
            z = zL + a_du * dzL
            zL = np.where(fl, np.maximum(np.minimum(z, 1e10 * mu / d), mu / (1e10 * d)), zL)
            d = ub - s
            z = zU + a_du * dzU
            zU = np.where(fu, np.maximum(np.minimum(z, 1e10 * mu / d), mu / (1e10 * d)), zU)
        it += 1
    return dict(x=x, y=y, f=f, status=status, iters=it, restarts=restarts)


def certificate(pb, x, y, lbo, ubo):
    """KKT measures of (x, y) from the oracle alone: violation of the original bounds, IPOPT's scaled stationarity error
    max|grad f + J' y| / s_d, and scaled complementarity: over the inequality rows, |y_i| times the distance to the bound
    its sign selects (y the multiplier of L = f + y' g), or |y_i| itself when that bound is infinite (a multiplier of the
    wrong sign), divided by s_c = max(100, mean |y_i|) / 100 as IPOPT scales it."""
    N = pb["N"]
    g = kr.eval_g(pb, x)
    J = kr.jac_exact(pb, x)
    _, gf = cost(x, N)
    viol = max(0.0, float(np.max(np.maximum(lbo - g, g - ubo))))
    m = g.size
    s_d = max(100.0, float(np.sum(np.abs(y))) / m) / 100.0
    stat = float(np.max(np.abs(gf + J.T @ y))) / s_d
    ineq = ~eq_rows(N)
    with np.errstate(invalid="ignore"):
        up = np.where(np.isfinite(ubo), y * np.abs(ubo - g), y)
        lo = np.where(np.isfinite(lbo), -y * np.abs(g - lbo), -y)
        c = np.where(y > 0, up, np.where(y < 0, lo, 0.0))
    s_c = max(100.0, float(np.mean(np.abs(y[ineq])))) / 100.0
    compl = float(np.max(np.where(ineq, c, 0.0))) / s_c
    return dict(viol=viol, stat=stat, compl=compl, g=g)


def check_filter_acceptance(e, gamma_theta=1e-5, gamma_phi=1e-5, eta_phi=1e-8, s_theta=1.1, s_phi=2.3, delta=1.0):
    """The acceptance rule of the filter line search (Waechter & Biegler 2006, as oracle/ip_ref.c states it), rechecked on
    one logged accepted trial: finite and below theta_max, not dominated by any filter entry, and either the switching
    condition with the Armijo test (ftype 1) or sufficient decrease in theta or phi (ftype 0).  Returns the failed clause
    or None."""
    tht, pht = e["theta_trial"], e["phi_trial"]
    if not (np.isfinite(tht) and np.isfinite(pht)):
        return "not finite"
    if tht > e["theta_max"]:
        return "theta above theta_max"
    for th_f, ph_f in e["filter"]:
        if tht >= th_f and pht >= ph_f:
            return "dominated by the filter entry (%g, %g)" % (th_f, ph_f)
    switching = e["theta"] <= e["theta_min"] and e["dphi"] < 0 and \
        e["alpha"] * (-e["dphi"]) ** s_phi > delta * e["theta"] ** s_theta
    if switching != (e["ftype"] == 1):
        return "ftype %d but switching condition %s" % (e["ftype"], switching)
    if switching:
        return None if pht <= e["phi"] + eta_phi * e["alpha"] * e["dphi"] else "Armijo test"
    if tht <= (1 - gamma_theta) * e["theta"] or pht <= e["phi"] - gamma_phi * e["theta"]:
        return None
    return "no sufficient decrease"
