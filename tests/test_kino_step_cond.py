"""Interior-point Newton step of the kino-dynamic NLP (landing_controller_b200/csrc/kino_step.cuh, host build) at
near-converged, ill-conditioned iterates: the stored KNITRO solutions of the N = 21 problem with slacks mu / (|lam| + mu)
from their active bounds and perfectly centred bound multipliers, so that sigma = z / (s - lbg) grows like lam^2 / mu
as it does in the last iterations of an interior-point loop.  Against the refined solve of the full, unreduced system:
the backward error of the host direction, its forward error bounded through a 1-norm condition estimate, and the inertia
decision against numpy eigenvalues of the reduced Hessian.  near_converged() is also the input of the GPU check in
tests/test_kino_step_scale.py."""
import os
import sys

import numpy as np
import pytest
import scipy.linalg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import kino_ref as kr  # noqa: E402
from kino_hess_ref import hess_exact  # noqa: E402
from test_kino import stored  # noqa: E402
from test_kino_step_host import (harness, patterns, ccs, eq_rows, full_system, reduced_hessian,  # noqa: E402,F401
                                 dw_trials, run_host, QN_DEFAULT, REF_DEFAULT)

N = 21
MUS = (1e-2, 1e-5, 1e-8, 1e-10)
TAGS = ("ms", "gs")
EPS = np.finfo(np.float64).eps


def near_converged(pb, x, lam, N, mu):
    """g, bounds and an iterate (s, y, zL, zU) at x that is complementary as a converging loop's is: on an inequality
    row whose multiplier marks an active side (lam < 0 with finite lbg, lam > 0 with finite ubg) the slack sits
    mu / (|lam| + mu) from that bound (at most half the bound gap), elsewhere at g pushed at least 1e-3 inside its bounds
    (mid-gap for narrower gaps); zL = mu / (s - lbg), zU = mu / (ubg - s) on the finite bounds, y = lam.  Then sigma is
    about lam^2 / mu on the active rows.  NaN where a quantity does not exist (equality rows, infinite bounds)."""
    g = kr.eval_g(pb, x, literal=False)
    lbg, ubg = kr.bounds(pb, x[:6], x[6:12], x[24 * N - 12:24 * N])
    m = g.size
    ineq = ~eq_rows(N)
    fl, fu = ineq & np.isfinite(lbg), ineq & np.isfinite(ubg)
    gap = ubg - lbg
    push = np.minimum(1e-3, 0.5 * gap)
    with np.errstate(invalid="ignore"):
        s = np.clip(g, np.where(fl, lbg + push, -np.inf), np.where(fu, ubg - push, np.inf))
        dist = np.minimum(mu / (np.abs(lam) + mu), 0.5 * gap)
    lo = fl & (lam < 0)
    up = fu & (lam > 0)
    s[lo] = lbg[lo] + dist[lo]
    s[up] = ubg[up] - dist[up]
    s[~ineq] = np.nan
    zL = np.full(m, np.nan)
    zU = np.full(m, np.nan)
    zL[fl] = mu / (s[fl] - lbg[fl])
    zU[fu] = mu / (ubg[fu] - s[fu])
    assert np.all(s[fl] - lbg[fl] > 0) and np.all(ubg[fu] - s[fu] > 0), "iterate not strictly interior"
    assert np.all(zL[fl] > 0) and np.all(zU[fu] > 0) and np.all(np.isfinite(zL[fl])) and np.all(np.isfinite(zU[fu]))
    return dict(g=g, lbg=lbg, ubg=ubg, s=s, y=np.asarray(lam, dtype=np.float64).copy(), zL=zL, zU=zU)


def sigma(it):
    """sigma of every inequality row (0 elsewhere)."""
    sg = np.zeros(it["g"].size)
    fl, fu = np.isfinite(it["zL"]), np.isfinite(it["zU"])
    sg[fl] += it["zL"][fl] / (it["s"][fl] - it["lbg"][fl])
    sg[fu] += it["zU"][fu] / (it["ubg"][fu] - it["s"][fu])
    return sg


def scenario_at(tag, mu, jsp, hsp):
    """A stored point as a host-build scenario: the near-converged iterate, J (dense and CCS values) from the oracle's
    complex-step Jacobian, W = hess_exact(lam_f = 1, lam_g = y) (dense and CCS values), grad f of the terminal cost."""
    pb, x, lam, _ = stored(tag)
    sc = near_converged(pb, x, lam, N, mu)
    sc.update(J=kr.jac_exact(pb, x), jv=kr.jac_exact(pb, x, ccs(jsp)),
              W=hess_exact(pb, x, 1.0, sc["y"], QN_DEFAULT, REF_DEFAULT),
              hv=hess_exact(pb, x, 1.0, sc["y"], QN_DEFAULT, REF_DEFAULT, ccs(hsp)))
    gf = np.zeros_like(x)
    xo = 12 * (N - 1)
    gf[xo:xo + 12] = 2.0 * QN_DEFAULT * (x[xo:xo + 12] - REF_DEFAULT)
    sc["gf"] = gf
    return sc


def cond1(A):
    """1-norm condition estimate of the sparse matrix A from its sparse LU factors."""
    import scipy.sparse.linalg as spl
    if A.shape[0] < 6000:
        return float(np.linalg.cond(A.toarray(), 1))
    lu = spl.splu(A.tocsc())
    inv = spl.LinearOperator(A.shape, matvec=lu.solve, rmatvec=lambda v: lu.solve(v, trans="T"), dtype=np.float64)
    return float(spl.onenormest(A) * spl.onenormest(inv))


def errors(sc, mu, outs, dw):
    """(backward error of the direction outs in the unreduced system, forward error against its refined solve
    (max over dx, ds, dy, dzL, dzU of |.|inf relative to max(1, |ref|inf)), the reference, (A, b, pack))."""
    args = [sc[k] for k in ("gf", "g", "s", "y", "zL", "zU", "lbg", "ubg")]
    ref, (A, b, pack) = full_system(N, sc["J"], sc["W"], *args, mu, dw, want_system=True)
    z = pack(*outs)
    back = float(np.max(np.abs(A @ z - b)) / (abs(A).max() * np.max(np.abs(z)) + np.max(np.abs(b))))
    fwd = max(float(np.max(np.abs(o - r)) / max(1.0, float(np.max(np.abs(r))))) for o, r in zip(outs, ref))
    return back, fwd, ref, (A, b, pack)


@pytest.fixture(scope="module")
def pats():
    return patterns(N)


@pytest.mark.parametrize("tag", TAGS)
def test_near_converged_iterate_is_centred_and_ill_conditioned(tag):
    """The helper's iterate: strictly interior, z (s - bound) = mu on every finite bound, sigma growing to lam^2 / mu."""
    pb, x, lam, _ = stored(tag)
    top = []
    for mu in MUS:
        it = near_converged(pb, x, lam, N, mu)
        fl, fu = np.isfinite(it["zL"]), np.isfinite(it["zU"])
        assert np.allclose(it["zL"][fl] * (it["s"][fl] - it["lbg"][fl]), mu, rtol=1e-12, atol=0)
        assert np.allclose(it["zU"][fu] * (it["ubg"][fu] - it["s"][fu]), mu, rtol=1e-12, atol=0)
        top.append(sigma(it).max())
    assert all(b > a for a, b in zip(top, top[1:])), top
    assert top[-1] > 90 * top[-2] and top[-1] > 1e6, top  # lam^2 / mu once the active rows dominate
    print("%s: max sigma %s at mu %s" % (tag, ["%.1e" % t for t in top], list(MUS)))


@pytest.mark.parametrize("tag", TAGS)
def test_host_step_at_near_converged_iterates(harness, pats, tag):  # noqa: F811
    """The host build from dw_last = 0 at mu = 1e-2 .. 1e-10: backward error <= 1e-13 in the unreduced system; forward
    error against its refined solve <= 1e-9 at mu = 1e-2 and <= 1e3 eps kappa elsewhere (kappa: 1-norm condition estimate
    of the unreduced system -- at small mu the forward error is governed by conditioning, not by the elimination); the
    inertia decision against numpy eigenvalues of the reduced Hessian: positive definite with the reported delta_w, and
    with delta_w > 0 not clearly positive definite (lambda_min <= 1e-10 |H|) at the schedule's previous trial value."""
    jsp, hsp = pats
    for mu in MUS:
        sc = scenario_at(tag, mu, jsp, hsp)
        outs, res = run_host(harness, N, jsp, hsp, sc, mu, 0.0)
        assert res[2] == 0, (tag, mu, res)
        dw, nf = float(res[0]), int(res[1])
        back, fwd, _, (A, _, _) = errors(sc, mu, outs, dw)
        kappa = cond1(A)
        lam_min = []
        for d in ([dw] if dw == 0 else [dw, dw_trials(0.0, nf)[-2]]):
            H = reduced_hessian(N, sc["J"], sc["W"], sc["s"], sc["zL"], sc["zU"], sc["lbg"], sc["ubg"], d)
            ev = np.linalg.eigvalsh(H)
            lam_min.append((ev.min(), np.abs(ev).max()))
        print("%s mu=%.0e: max sigma %.1e, delta_w %g (%d factorisations), backward %.1e, forward %.1e, kappa %.1e, "
              "lambda_min %s" % (tag, mu, sigma(sc).max(), dw, nf, back, fwd, kappa,
                                 ["%.2e (|H| %.1e)" % t for t in lam_min]))
        assert back <= 1e-13, (tag, mu, back)
        assert fwd <= (1e-9 if mu == 1e-2 else 1e3 * EPS * kappa), (tag, mu, fwd, kappa)
        assert dw_trials(0.0, nf)[-1] == dw
        assert lam_min[0][0] > 0, (tag, mu, dw, lam_min)
        if dw > 0:
            assert lam_min[1][0] <= 1e-10 * lam_min[1][1], (tag, mu, dw, lam_min)
