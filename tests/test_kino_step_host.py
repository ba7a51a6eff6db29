"""Interior-point Newton step of the kino-dynamic NLP on the CPU: the plan, the Riccati sweeps, the recovery and the
inertia schedule of landing_controller_b200/csrc/kino_step.cuh compiled for the host, against a dense solve of the full,
unreduced primal-dual system (dx, ds, dy, dzL, dzU) assembled from the oracle's exact Jacobian (oracle/kino_ref.py:
jac_exact) and exact Hessian (tests/kino_hess_ref.py:hess_exact).  Also the numpy restatement of the system, of the
inertia schedule and of the fraction-to-boundary rule that tests/test_kino_step.py holds the GPU to."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.linalg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import kino_ref as kr  # noqa: E402
from kino_hess_ref import hess_exact  # noqa: E402
from test_kino_exact import random_problem, random_x  # noqa: E402

_dp = ctypes.POINTER(ctypes.c_double)
_ip = ctypes.POINTER(ctypes.c_int)
_lp = ctypes.POINTER(ctypes.c_longlong)
QN_DEFAULT = np.array([0, 0, 100, 10, 10, 0, 10, 10, 10, 10, 10, 10.0])
REF_DEFAULT = np.array([0, 0, 0.25, 0, 0, 0, 0, 0, 0, 0, 0, 0.0])


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    """tests/hostcheck/kino_step_host.cpp, built into a temporary directory (the checkout may be read-only)."""
    so = str(tmp_path_factory.mktemp("kino_step_host") / "libkino_step_host.so")
    src = os.path.join(ROOT, "tests", "hostcheck", "kino_step_host.cpp")
    subprocess.check_call(["/usr/bin/g++", "-O1", "-std=c++17", "-fPIC", "-shared", src, "-o", so])
    return ctypes.CDLL(so)


def patterns(N):
    """The library's CCS patterns of J and of the upper triangle of W (host logic, no GPU)."""
    import landing_controller_b200 as lc
    lib = lc.load_library()
    lib.landing_kino_sparsity.restype = _lp
    lib.landing_kino_hess_sparsity.restype = _lp
    out = []
    for sp in (lib.landing_kino_sparsity(N), lib.landing_kino_hess_sparsity(N)):
        nx = sp[1]
        nnz = sp[2 + nx]
        out.append(np.ctypeslib.as_array(sp, shape=(2 + nx + 1 + nnz,)).copy())
    return out


def ccs(sp):
    nx = int(sp[1])
    return sp[2:2 + nx + 1], sp[2 + nx + 1:]


def eq_rows(N):
    m = kr.dims(N)["m"]
    r = np.arange(m)
    return (r < 24) | ((r >= 48) & ((r - 48) % 141 < 12))


def interior_point(rng, N, g, lbg, ubg, y_scale=1.0):
    """Random interior slacks and bound multipliers for bounds lbg / ubg (NaN where they must be ignored: equality rows,
    infinite bounds), and random y."""
    m = g.size
    eq = eq_rows(N)
    fl, fu = np.isfinite(lbg) & ~eq, np.isfinite(ubg) & ~eq
    s = g + rng.normal(size=m) * 0.1
    both = fl & fu
    s[both] = lbg[both] + (ubg[both] - lbg[both]) * rng.uniform(0.1, 0.9, both.sum())
    s[fl & ~fu] = lbg[fl & ~fu] + rng.uniform(0.01, 2.0, (fl & ~fu).sum())
    s[fu & ~fl] = ubg[fu & ~fl] - rng.uniform(0.01, 2.0, (fu & ~fl).sum())
    s[eq] = np.nan
    zL = np.where(fl, rng.uniform(0.05, 5.0, m), np.nan)
    zU = np.where(fu, rng.uniform(0.05, 5.0, m), np.nan)
    y = rng.normal(size=m) * y_scale
    return s, y, zL, zU


def full_system(N, J, W, gf, g, s, y, zL, zU, lbg, ubg, mu, dw, want_system=False):
    """The unreduced Newton system of IPOPT's form (include/landing_b200.h: landing_kino_step_batch), assembled sparse, and
    its solution dx, ds, dy, dzL, dzU (0 where a quantity does not exist, as the library writes them).  J, W: dense or
    scipy.sparse (W symmetric).  want_system: also (A, b, pack) with pack(dx, ds, dy, dzL, dzU) -> z."""
    import scipy.sparse as sps
    J, W = sps.csr_matrix(J), sps.csr_matrix(W)
    m, nx = J.shape
    eq = eq_rows(N)
    I, E = np.flatnonzero(~eq), np.flatnonzero(eq)
    L = np.flatnonzero(~eq & np.isfinite(lbg))
    U = np.flatnonzero(~eq & np.isfinite(ubg))
    nI, nL, nU = I.size, L.size, U.size
    oS, oY, oL, oU = nx, nx + nI, nx + nI + m, nx + nI + m + nL
    n = oU + nU
    zl = np.zeros(m); zl[L] = zL[L]
    zu = np.zeros(m); zu[U] = zU[U]
    posI = -np.ones(m, dtype=int); posI[I] = np.arange(nI)
    posL = -np.ones(m, dtype=int); posL[L] = np.arange(nL)
    posU = -np.ones(m, dtype=int); posU[U] = np.arange(nU)
    Sel = lambda rows, cols, vals, nr, nc: sps.csr_matrix((vals, (rows, cols)), shape=(nr, nc))  # noqa: E731
    eyeI = Sel(np.arange(nI), I, np.ones(nI), nI, m)  # picks the inequality rows
    Lm = Sel(np.arange(nI)[posL[I] >= 0], posL[I][posL[I] >= 0], np.ones(nL), nI, nL)
    Um = Sel(np.arange(nI)[posU[I] >= 0], posU[I][posU[I] >= 0], np.ones(nU), nI, nU)
    dL, dU = s[L] - lbg[L], ubg[U] - s[U]
    Z = None
    A = sps.bmat([
        [W + dw * sps.identity(nx), Z, J.T, Z, Z],
        [Z, Z, -eyeI, -Lm, Um],
        [J[E], Z, Z, Z, Z],
        [J[I], -sps.identity(nI), Z, Z, Z],
        [Z, Sel(np.arange(nL), posI[L], zL[L], nL, nI), Z, sps.diags(dL), Z],
        [Z, Sel(np.arange(nU), posI[U], -zU[U], nU, nI), Z, Z, sps.diags(dU)]], format="csc", dtype=np.float64)
    b = np.concatenate([-(gf + J.T @ y), y[I] + zl[I] - zu[I], -(g[E] - lbg[E]), -(g[I] - s[I]),
                        mu - zL[L] * dL, mu - zU[U] * dU])
    assert A.shape == (n, n) and b.size == n
    if n <= 6000:  # dense LU, refined with residuals in extended precision: accurate to about the working precision
        Ad = A.toarray()
        lu = scipy.linalg.lu_factor(Ad)
        z = scipy.linalg.lu_solve(lu, b)
        Al, bl = Ad.astype(np.longdouble), b.astype(np.longdouble)
        for _ in range(3):
            z = z + scipy.linalg.lu_solve(lu, (bl - Al @ z.astype(np.longdouble)).astype(np.float64))
    else:  # sparse LU with refinement
        import scipy.sparse.linalg as spl
        lu = spl.splu(A)
        z = lu.solve(b)
        for _ in range(3):
            z = z + lu.solve(b - A @ z)
    dx = z[:nx]
    ds = np.zeros(m); ds[I] = z[oS:oS + nI]
    dy = z[oY:oY + m]
    dzL = np.zeros(m); dzL[L] = z[oL:oL + nL]
    dzU = np.zeros(m); dzU[U] = z[oU:oU + nU]
    if not want_system:
        return dx, ds, dy, dzL, dzU

    def pack(dx_, ds_, dy_, dzL_, dzU_):
        return np.concatenate([dx_, ds_[I], dy_, dzL_[L], dzU_[U]])
    return (dx, ds, dy, dzL, dzU), (A, b, pack)


def reduced_hessian(N, J, W, s, zL, zU, lbg, ubg, dw):
    """Z' (W + J_I' Sigma J_I + dw I) Z, Z a basis of the null space of J_E."""
    eq = eq_rows(N)
    sig = np.zeros(J.shape[0])
    fl, fu = ~eq & np.isfinite(lbg), ~eq & np.isfinite(ubg)
    sig[fl] += zL[fl] / (s[fl] - lbg[fl])
    sig[fu] += zU[fu] / (ubg[fu] - s[fu])
    H = W + J.T @ (sig[:, None] * J) + dw * np.eye(J.shape[1])
    Z = scipy.linalg.null_space(J[eq])
    return Z.T @ H @ Z


def dw_trials(dw_last, n):
    """The first n values of the inertia-correction schedule (oracle/ip_ref.c ip_solve_ws) from dw_last."""
    dw = dw_last / 3.0 if dw_last > 0 else 0.0
    if dw_last > 0 and dw < 1e-7:
        dw = 0.0
    out = []
    for tries in range(n):
        out.append(dw)
        if dw == 0:
            dw = 1e-4 if dw_last == 0 else max(1e-20, dw_last / 3.0)
        else:
            dw *= 100.0 if (dw_last == 0 and tries < 8) else 8.0
    return out


def fraction_to_boundary(N, s, ds, zL, dzL, zU, dzU, lbg, ubg, tau):
    """alpha_pr, alpha_du of oracle/ip_ref.c (ip_solve_ws), in the same operation order as the library."""
    eq = eq_rows(N)
    apr = adu = 1.0
    for i in np.flatnonzero(~eq):
        if np.isfinite(lbg[i]):
            if ds[i] < 0: apr = min(apr, -tau * (s[i] - lbg[i]) / ds[i])
            if dzL[i] < 0: adu = min(adu, -tau * zL[i] / dzL[i])
        if np.isfinite(ubg[i]):
            if ds[i] > 0: apr = min(apr, tau * (ubg[i] - s[i]) / ds[i])
            if dzU[i] < 0: adu = min(adu, -tau * zU[i] / dzU[i])
    return apr, adu


def scenario(rng, N, jsp, hsp, y_scale=1.0):
    """Inputs built without the library: pb, x, J (dense and CCS values), W (dense and CCS values), grad f, g, bounds and
    an interior iterate."""
    pb = random_problem(rng, N)
    x = random_x(rng, N, 1)[0]
    g = kr.eval_g(pb, x, literal=False)
    Jd = kr.jac_exact(pb, x)
    jv = kr.jac_exact(pb, x, ccs(jsp))
    drop = np.concatenate([x[:6], x[6:12]])
    lbg, ubg = kr.bounds(pb, drop[:6], drop[6:], x[24 * N - 12:24 * N])
    s, y, zL, zU = interior_point(rng, N, g, lbg, ubg, y_scale)
    Wd = hess_exact(pb, x, 1.0, y, QN_DEFAULT, REF_DEFAULT)
    hv = hess_exact(pb, x, 1.0, y, QN_DEFAULT, REF_DEFAULT, ccs(hsp))
    gf = np.zeros_like(x)
    xo = 12 * (N - 1)
    gf[xo:xo + 12] = 2.0 * QN_DEFAULT * (x[xo:xo + 12] - REF_DEFAULT)
    return dict(pb=pb, x=x, g=g, J=Jd, jv=jv, W=Wd, hv=hv, gf=gf, lbg=lbg, ubg=ubg, s=s, y=y, zL=zL, zU=zU)


def run_host(h, N, jsp, hsp, sc, mu, dw_last, tau=0.99):
    nx, m = kr.dims(N)["nx"], kr.dims(N)["m"]
    vec = [np.ascontiguousarray(sc[k], dtype=np.float64) for k in ("g", "s", "y", "zL", "zU", "lbg", "ubg")]
    outs = [np.full(nx, np.nan)] + [np.full(m, np.nan) for _ in range(4)]
    res = np.full(5, np.nan)
    vp = (_dp * 7)(*[v.ctypes.data_as(_dp) for v in vec])
    op = (_dp * 5)(*[o.ctypes.data_as(_dp) for o in outs])
    rc = h.kino_step_host(ctypes.c_int(N), jsp.ctypes.data_as(_lp), hsp.ctypes.data_as(_lp),
                          sc["jv"].ctypes.data_as(_dp), sc["hv"].ctypes.data_as(_dp), sc["gf"].ctypes.data_as(_dp), vp,
                          ctypes.c_double(mu), ctypes.c_double(dw_last), ctypes.c_double(tau), op,
                          res.ctypes.data_as(_dp))
    assert rc == 0
    return outs, res


def rel(a, b):
    return float(np.max(np.abs(a - b)) / max(1.0, float(np.max(np.abs(b)))))


@pytest.mark.parametrize("N", [3, 4, 6])
def test_host_step_solves_the_full_system(harness, N):
    """dx, ds, dy, dzL, dzU of the host build agree with a dense solve of the unreduced system (same dw) to 1e-10
    relative to max(1, |.|inf), from dw_last = 0 and from a previous regularisation."""
    rng = np.random.default_rng(100 + N)
    jsp, hsp = patterns(N)
    worst = 0.0
    for rep, dw_last in enumerate((0.0, 0.0, 3e-3, 1e-9)):
        sc = scenario(rng, N, jsp, hsp, y_scale=1.0 if rep % 2 == 0 else 30.0)
        mu = 10.0 ** rng.uniform(-3, 0)
        outs, res = run_host(harness, N, jsp, hsp, sc, mu, dw_last)
        assert res[2] == 0, res
        ref = full_system(N, sc["J"], sc["W"], sc["gf"], sc["g"], sc["s"], sc["y"], sc["zL"], sc["zU"], sc["lbg"],
                          sc["ubg"], mu, res[0])
        for name, a, b in zip(("dx", "ds", "dy", "dzL", "dzU"), outs, ref):
            e = rel(a, b)
            worst = max(worst, e)
            assert e < 1e-10, (N, rep, name, e)
    print("N=%d host step vs full system: worst %.2e" % (N, worst))


@pytest.mark.parametrize("N", [3, 4, 6])
def test_host_step_inertia_correction(harness, N):
    """With the reported dw the reduced Hessian is positive definite; with the schedule's previous trial value it is not;
    a positive-definite scenario from dw_last = 0 gives dw = 0 in one factorisation."""
    rng = np.random.default_rng(200 + N)
    jsp, hsp = patterns(N)
    seen_reg = False
    for rep in range(4):
        y_scale = 0.0 if rep == 0 else 100.0
        sc = scenario(rng, N, jsp, hsp, y_scale=y_scale)
        outs, res = run_host(harness, N, jsp, hsp, sc, 0.1, 0.0)
        assert res[2] == 0
        dw, nf = res[0], int(res[1])
        trials = dw_trials(0.0, nf)
        assert trials[-1] == dw
        red = lambda d: np.linalg.eigvalsh(reduced_hessian(N, sc["J"], sc["W"], sc["s"], sc["zL"], sc["zU"],  # noqa
                                                           sc["lbg"], sc["ubg"], d))
        assert red(dw).min() > 0, (rep, dw)
        if rep == 0:
            assert dw == 0.0 and nf == 1
        if dw > 0:
            seen_reg = True
            assert red(trials[-2]).min() <= 0, (rep, trials[-2])
    assert seen_reg


def test_dw_schedule_restates_ip_ref():
    assert dw_trials(0.0, 4) == [0.0, 1e-4, 1e-2, 1.0]
    assert dw_trials(3e-3, 3) == [1e-3, 8e-3, 6.4e-2]
    assert dw_trials(1e-7, 3)[:2] == [0.0, max(1e-20, 1e-7 / 3.0)]


@pytest.mark.parametrize("N", [3, 4, 6])
def test_plan_contracts_every_nonzero_once(harness, N):
    """Through an instrumented source: one factorisation's assembly reads every Hessian entry and every grad f column
    exactly once; a Jacobian entry of an inequality row with n entries n + 2 times (the row's outer product and its
    gradient term), one of a dynamics row once (G), and the identities (boundary rows, X_{k+1} in the dynamics rows)
    never -- each is in the plan under exactly one role."""
    rng = np.random.default_rng(300 + N)
    jsp, hsp = patterns(N)
    sc = scenario(rng, N, jsp, hsp)
    nx, m = kr.dims(N)["nx"], kr.dims(N)["m"]
    colind, row = ccs(jsp)
    nnzJ, nnzH = row.size, ccs(hsp)[1].size
    jc, hc, gc, role = (np.zeros(nnzJ, np.int32), np.zeros(nnzH, np.int32), np.zeros(nx, np.int32),
                        np.full(nnzJ, -7, np.int32))
    vec = [np.ascontiguousarray(sc[k]) for k in ("g", "s", "y", "zL", "zU", "lbg", "ubg")]
    vp = (_dp * 7)(*[v.ctypes.data_as(_dp) for v in vec])
    assert harness.kino_step_cover(ctypes.c_int(N), jsp.ctypes.data_as(_lp), hsp.ctypes.data_as(_lp),
                                   sc["jv"].ctypes.data_as(_dp), sc["hv"].ctypes.data_as(_dp),
                                   sc["gf"].ctypes.data_as(_dp), vp, ctypes.c_double(0.1), jc.ctypes.data_as(_ip),
                                   hc.ctypes.data_as(_ip), gc.ctypes.data_as(_ip), role.ctypes.data_as(_ip)) == 0
    assert np.all(hc == 1) and np.all(gc == 1)
    col = np.repeat(np.arange(nx), np.diff(colind))
    eq = eq_rows(N)
    per_row = np.bincount(row, minlength=m)
    expect_role = np.where(row < 24, 0, np.where(eq[row], 2, 3))
    for e in np.flatnonzero(eq[row] & (row >= 48)):  # X_{k+1} identity of a dynamics row
        k, rho = (row[e] - 48) // 141, (row[e] - 48) % 141
        st = 9 + rho if rho < 3 else (3 + rho if rho < 6 else rho - 6)
        if col[e] == 12 * (k + 1) + st:
            expect_role[e] = 1
    assert np.array_equal(role, expect_role)
    expect = np.select([role == 3, role == 2], [per_row[row] + 2, 1], 0)
    assert np.array_equal(jc, expect)


def test_plan_refuses_an_entry_outside_every_stage(harness):
    """A Hessian entry coupling two knots that share no stage (X_0, X_2) is refused; the library's patterns are accepted."""
    N = 4
    jsp, hsp = patterns(N)
    assert harness.kino_step_plan_ok(ctypes.c_int(N), jsp.ctypes.data_as(_lp), hsp.ctypes.data_as(_lp)) == 0
    nx = int(hsp[1])
    colind, row = ccs(hsp)
    c = 24  # X_2[0]: add the entry (row 0, col 24)
    rows = list(row)
    ins = int(colind[c])
    rows.insert(ins, 0)
    ci = colind.copy()
    ci[c + 1:] += 1
    bad = np.concatenate([hsp[:2], ci, np.array(rows, dtype=np.int64)]).astype(np.int64)
    assert harness.kino_step_plan_ok(ctypes.c_int(N), jsp.ctypes.data_as(_lp), bad.ctypes.data_as(_lp)) == -1
    assert nx == kr.dims(N)["nx"]


def test_host_step_refuses_a_non_interior_iterate(harness):
    N = 3
    rng = np.random.default_rng(5)
    jsp, hsp = patterns(N)
    sc = scenario(rng, N, jsp, hsp)
    i = np.flatnonzero(~eq_rows(N) & np.isfinite(sc["lbg"]))[3]
    sc["s"][i] = sc["lbg"][i]
    _, res = run_host(harness, N, jsp, hsp, sc, 0.1, 0.0)
    assert res[2] == 5
