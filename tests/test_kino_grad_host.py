"""Lagrangian gradient of the kino-dynamic NLP on the CPU: the owner contraction of the gradient kernels
(landing_controller_b200/csrc/kino_grad.cuh) compiled for the host against lam_f grad f + J' lam_g with the oracle's exact
Jacobian (oracle/kino_ref.py:jac_exact), and its coverage: every non-zero of J is contracted exactly once, and nothing
else.  Also the numpy reference of the KKT residuals that tests/test_kino_kkt.py holds the GPU to."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import kino_ref as kr  # noqa: E402
from test_kino_host import random_params, _prm  # noqa: E402

_dp = ctypes.POINTER(ctypes.c_double)
_ip = ctypes.POINTER(ctypes.c_int)
QN_DEFAULT = np.array([0, 0, 100, 10, 10, 0, 10, 10, 10, 10, 10, 10.0])   # generate_landingCtrller_KNITRO.m:260
REF_DEFAULT = np.array([0, 0, 0.25, 0, 0, 0, 0, 0, 0, 0, 0, 0.0])         # :236-237


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    """tests/hostcheck/kino_grad_host.cpp, built into a temporary directory (the checkout may be read-only)."""
    so = str(tmp_path_factory.mktemp("kino_grad_host") / "libkino_grad_host.so")
    src = os.path.join(ROOT, "tests", "hostcheck", "kino_grad_host.cpp")
    subprocess.check_call(["/usr/bin/g++", "-O1", "-std=c++17", "-fPIC", "-shared", src, "-o", so])
    return ctypes.CDLL(so)


def _ptr(a, typ=_dp):
    return a.ctypes.data_as(typ)


def random_point(rng, N):
    """Random parameters and knot spacings, x at landing magnitudes (forces up to 300 N), lam_g, lam_f, QN, ref."""
    pb = dict(kr.default_problem(N), **random_params(rng))
    pb["dt"] = rng.uniform(0.005, 0.1, N - 1)
    X, Jp, U = kr.split(rng.uniform(-0.5, 0.5, kr.dims(N)["nx"]), N)
    X[:, 3:6] = rng.uniform(-1, 1, (N, 3))
    X[:, 6:12] = rng.uniform(-3, 3, (N, 6))
    Jp[:] = rng.uniform(-1, 1, Jp.shape)
    U[:, 12:] = rng.uniform(-100, 100, (N - 1, 12))
    U[:, 14::3] = rng.uniform(0, 300, (N - 1, 4))
    x = np.concatenate([X.ravel(), Jp.ravel(), U.ravel()])
    return pb, x, rng.normal(size=kr.dims(N)["m"]), rng.uniform(0.1, 3.0), rng.uniform(0, 100, 12), \
        rng.uniform(-0.5, 0.5, 12)


def grad_reference(pb, x, lam_f, lam_g, QN, ref):
    """lam_f grad f + J' lam_g with the exact Jacobian, and the per-column scale sum_i |J_ij lam_i| + |lam_f df/dx_j|."""
    N = pb["N"]
    J = kr.jac_exact(pb, x)
    gf = np.zeros_like(x)
    lf = 0.0 if lam_f is None else lam_f
    gf[12 * (N - 1):12 * N] = lf * 2.0 * QN * (x[12 * (N - 1):12 * N] - ref)
    lg = np.zeros(J.shape[0]) if lam_g is None else lam_g
    return gf + J.T @ lg, np.abs(J * lg[:, None]).sum(0) + np.abs(gf)


def kkt_reference(g, lbg, ubg, lam_g, grad_x):
    """viol, dual_inf, compl_inf of one scenario, as include/landing_b200.h defines them (NaN anywhere -> all NaN)."""
    lam = np.zeros_like(g) if lam_g is None else lam_g
    if np.isnan(np.concatenate([g, lbg, ubg, lam, grad_x])).any():
        return np.nan, np.nan, np.nan
    with np.errstate(invalid="ignore"):
        viol = max(0.0, np.where(np.isfinite(lbg), lbg - g, 0.0).max(), np.where(np.isfinite(ubg), g - ubg, 0.0).max())
        ineq = lbg < ubg
        c = np.zeros_like(g)
        up, lo = ineq & (lam > 0), ineq & (lam < 0)
        c[up] = lam[up] * np.abs(ubg[up] - g[up])
        c[lo] = -lam[lo] * np.abs(g[lo] - lbg[lo])
    return viol, float(np.abs(grad_x).max()), float(c.max())


@pytest.mark.parametrize("N", [3, 4])
def test_owner_contraction_on_host_matches_the_exact_gradient(harness, N):
    """Every column of the owners' gradient against lam_f grad f + J' lam_g at 1e-13 relative to the column's scale,
    at random parameters, spacings and forces up to 300 N; N = 3 and 4 hold both knot classes."""
    rng = np.random.default_rng(40 + N)
    worst = 0.0
    for _ in range(4):
        pb, x, lam_g, lam_f, QN, ref = random_point(rng, N)
        out = np.full(x.size, np.nan)
        harness.kino_grad_host(N, _ptr(x), _ptr(pb["dt"]), _ptr(_prm(pb)), _ptr(lam_g), ctypes.c_double(lam_f),
                               _ptr(QN), _ptr(ref), _ptr(out))
        r, scale = grad_reference(pb, x, lam_f, lam_g, QN, ref)
        e = np.abs(out - r) / np.maximum(1.0, scale)
        assert e.max() <= 1e-13, (e.max(), int(e.argmax()))
        worst = max(worst, e.max())
    print("kino grad owners N=%d vs exact: worst rel. error %.2e" % (N, worst))


@pytest.mark.parametrize("N", [3, 4])
def test_owner_contraction_touches_every_jacobian_nonzero_exactly_once(harness, N):
    """Instrumented contraction: no (row, column) pair is contracted twice, and the pairs contracted with a non-zero
    tangent are exactly the non-zeros of the exact Jacobian (boundary identities included)."""
    rng = np.random.default_rng(50 + N)
    d = kr.dims(N)
    for _ in range(3):
        pb, x, _, _, _, _ = random_point(rng, N)
        cnt = np.zeros((d["m"], d["nx"]), dtype=np.int32)
        nz = np.zeros_like(cnt)
        harness.kino_grad_cover(N, _ptr(x), _ptr(pb["dt"]), _ptr(_prm(pb)), _ptr(cnt, _ip), _ptr(nz, _ip))
        J = kr.jac_exact(pb, x)
        assert cnt.max() <= 1, np.argwhere(cnt > 1)[:5]
        missing = np.argwhere((J != 0) & (nz == 0))
        assert missing.size == 0, ("Jacobian non-zero (row, col) never contracted", missing[:5])
        extra = np.argwhere((J == 0) & (nz != 0))
        assert extra.size == 0, ("(row, col) contracted with a non-zero tangent outside J", extra[:5])


def test_stored_knitro_points_kkt_residuals_on_host():
    """The residuals of the two stored KNITRO points (tests/golden/kino_n21.npz) with the oracle's bounds and lam_f = 1,
    measured here as the reference of the GPU test: the main_scripts point is stationary to 1e-4 of max |J_ij lam_i|;
    both carry wrong-sign multipliers of at most 6e-8 on inequality rows whose violated side is an infinite bound, which
    makes compl_inf = +inf by its definition; without those rows it is below 1e-6."""
    from test_kino import stored
    for tag, viol_tol in (("ms", 1e-6), ("gs", 5e-5)):
        pb, x, lam, (q0, qd0, c0) = stored(tag)
        g = kr.eval_g(pb, x, literal=False)
        lbg, ubg = kr.bounds(pb, q0, qd0, c0)
        grad, _ = grad_reference(pb, x, 1.0, lam, QN_DEFAULT, REF_DEFAULT)
        viol, dual, compl = kkt_reference(g, lbg, ubg, lam, grad)
        scale = np.abs(kr.jac_exact(pb, x) * lam[:, None]).max()
        ineq = lbg < ubg
        wrong = ineq & (((lam > 0) & np.isinf(ubg)) | ((lam < 0) & np.isinf(lbg)))
        rest = kkt_reference(g, np.where(wrong, -np.inf, lbg), np.where(wrong, np.inf, ubg), np.where(wrong, 0, lam),
                             grad)[2]
        print("%s: viol %.3g dual_inf %.3g (%.3g of max|J_ij lam_i|) compl_inf %g, %d wrong-sign rows (max |lam| %.2g), "
              "compl_inf without them %.3g" % (tag, viol, dual, dual / scale, compl, wrong.sum(),
                                               np.abs(lam[wrong]).max(), rest))
        assert viol <= viol_tol
        assert compl == np.inf and 0 < wrong.sum() <= 20 and np.abs(lam[wrong]).max() <= 6e-8 and rest <= 1e-6
        if tag == "ms":
            assert dual <= 1e-4 * scale
