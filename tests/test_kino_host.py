"""Kino-dynamic NLP on the CPU: the exact (complex-step) Jacobian of the oracle, oracle/kino_ref.py:jac_exact, against
finite differences and the stored KNITRO solution; the product's knot template and Jacobian pass table (kino_knot.cuh)
compiled for the host against that exact Jacobian; and the library's CCS pattern against every exact non-zero."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import kino_ref as kr  # noqa: E402

NIN = 72
_dp = ctypes.POINTER(ctypes.c_double)


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    """tests/hostcheck/kino_host.cpp, built into a temporary directory (the checkout may be read-only)."""
    so = str(tmp_path_factory.mktemp("kino_host") / "libkino_host.so")
    src = os.path.join(ROOT, "tests", "hostcheck", "kino_host.cpp")
    subprocess.check_call(["/usr/bin/g++", "-O1", "-std=c++17", "-fPIC", "-shared", src, "-o", so])
    return ctypes.CDLL(so)


def _ptr(a, typ=_dp):
    return a.ctypes.data_as(typ)


def random_params(rng):
    """mu, mass, Ib, and an Ib_inv that is deliberately not 1 / Ib (a swapped or ignored field shows)."""
    return {"mu": rng.uniform(0.3, 1.2), "mass": rng.uniform(5.0, 12.0), "Ib": rng.uniform(0.03, 0.4, 3),
            "Ib_inv": rng.uniform(2.0, 25.0, 3)}


def random_knot(rng):
    """Knot-local inputs at landing magnitudes: positions within 0.5 m, angles within 1 rad, rates within 3, forces up
    to 300 N."""
    z = rng.uniform(-0.5, 0.5, NIN)
    for o in (0, 48):  # X_k, X_{k+1}: r, rpy, omega, v
        z[o + 3:o + 6] = rng.uniform(-1, 1, 3)
        z[o + 6:o + 12] = rng.uniform(-3, 3, 6)
    z[12:24] = rng.uniform(-1, 1, 12)
    z[36:48] = rng.uniform(-100, 100, 12)
    z[38:48:3] = rng.uniform(0, 300, 4)
    return z


def _prm(p):
    return np.concatenate([[p["mu"], p["mass"]], p["Ib"], p["Ib_inv"]])


@pytest.mark.parametrize("last", [False, True])
def test_knot_template_on_host_matches_the_exact_jacobian(harness, last):
    """kino_knot.cuh compiled for the host: rows and every Dual1 Jacobian column of one knot against the complex step of
    the oracle, at random points with random parameters and knot spacing."""
    rng = np.random.default_rng(7 + last)
    nin, nrow = (60, 117) if last else (72, 141)
    worst = 0.0
    for _ in range(20):
        z = random_knot(rng)
        pb = dict(random_params(rng), dt=[rng.uniform(0.005, 0.2)])
        g, J = np.zeros(141), np.zeros((141, NIN))
        harness.kino_host_knot(int(last), _ptr(z), ctypes.c_double(pb["dt"][0]), _ptr(_prm(pb)), _ptr(g), _ptr(J))
        go, Jo = kr.knot_jac(pb, 0, z[:nin], last)
        assert np.max(np.abs(g[:nrow] - go) / np.maximum(1.0, np.abs(go))) <= 1e-13
        assert not np.any(g[nrow:]) and not np.any(J[nrow:]) and not np.any(J[:, nin:])
        err = np.max(np.abs(J[:nrow, :nin] - Jo) / np.maximum(1.0, np.abs(Jo)))
        worst = max(worst, err)
        assert err <= 1e-13, err
    print("knot template (last=%d) vs complex step: worst rel. error %.2e" % (last, worst))


@pytest.mark.parametrize("last", [False, True])
def test_jacobian_passes_emit_every_nonzero_exactly_once(harness, last):
    """The pass table of the Jacobian kernels (kino::PassOf masks, kino::jac_pass seeding, the last-knot skip): the union
    of all passes reproduces every non-zero of the full Dual1 Jacobian, emits no entry twice, and agrees in value."""
    rng = np.random.default_rng(17 + last)
    for _ in range(5):
        z = random_knot(rng)
        prm, h = _prm(random_params(rng)), rng.uniform(0.005, 0.2)
        g, Jf = np.zeros(141), np.zeros((141, NIN))
        harness.kino_host_knot(int(last), _ptr(z), ctypes.c_double(h), _ptr(prm), _ptr(g), _ptr(Jf))
        Jp, cnt = np.zeros((141, NIN)), np.zeros((141, NIN), dtype=np.int32)
        harness.kino_host_passes(int(last), _ptr(z), ctypes.c_double(h), _ptr(prm), _ptr(Jp),
                                 _ptr(cnt, ctypes.POINTER(ctypes.c_int)))
        assert cnt.max() <= 1, np.argwhere(cnt > 1)[:5]
        missing = np.argwhere((Jf != 0) & (cnt == 0))
        assert missing.size == 0, ("(row, input) not covered by any pass", missing[:5])
        assert np.max(np.abs(Jp - Jf) / np.maximum(1.0, np.abs(Jf))) <= 1e-14


def test_exact_jacobian_agrees_with_finite_differences():
    N = 4
    rng = np.random.default_rng(3)
    pb = dict(kr.default_problem(N), **random_params(rng))
    pb["dt"] = rng.uniform(0.01, 0.1, N - 1)
    for _ in range(2):
        x = rng.uniform(-0.7, 0.7, kr.dims(N)["nx"])
        Je, Jf = kr.jac_exact(pb, x), kr.jac_fd(pb, x, literal=False)
        assert np.max(np.abs(Je - Jf)) <= 1e-7 * max(1.0, np.abs(Je).max())
        assert np.array_equal(Je != 0, Jf != 0)  # same pattern (a row that does not read a column has an exact 0 in both)


def test_stored_knitro_point_is_stationary_for_the_exact_jacobian():
    d = np.load(os.path.join(ROOT, "tests", "golden", "kino_n21.npz"))
    x, lam = d["ms_x"], d["ms_lam_g"]
    J = kr.jac_exact(kr.default_problem(21), x)
    r = J.T @ lam
    QN = np.array([0, 0, 100, 10, 10, 0, 10, 10, 10, 10, 10, 10.0])         # generate_landingCtrller_KNITRO.m:260
    ref = np.array([0, 0, 0.25, 0, 0, 0, 0, 0, 0, 0, 0, 0.0])              # :236-237
    r[240:252] += 2 * QN * (x[240:252] - ref)
    scale = np.abs(J.T * lam).max()
    assert scale > 1e-2 and np.abs(r).max() <= 1e-4 * scale, (np.abs(r).max(), scale)


@pytest.mark.parametrize("N", [3, 4, 21])
def test_library_kino_pattern_holds_every_exact_nonzero(N):
    """landing_kino_sparsity(N) (host logic of the product library, no GPU needed) contains every entry that is non-zero
    in the exact Jacobian, on every column, at random points with random parameters (threshold 0)."""
    import landing_controller_b200 as lc
    lib = lc.load_library()
    d = (ctypes.c_longlong * 4)()
    assert lib.landing_kino_dims(N, d) == 0
    nx, m, nnz = int(d[1]), int(d[2]), int(d[3])
    assert (nx, m) == (kr.dims(N)["nx"], kr.dims(N)["m"])
    sp = np.ctypeslib.as_array(lib.landing_kino_sparsity(N), shape=(2 + nx + 1 + nnz,))
    colind, row = sp[2:2 + nx + 1], sp[2 + nx + 1:]
    inpat = np.zeros((m, nx), dtype=bool)
    inpat[row, np.repeat(np.arange(nx), np.diff(colind))] = True
    rng = np.random.default_rng(N)
    for _ in range(3 if N == 21 else 6):
        pb = dict(kr.default_problem(N), **random_params(rng))
        pb["dt"] = rng.uniform(0.01, 0.1, N - 1)
        X, Jp, U = kr.split(rng.uniform(-1, 1, nx), N)
        U[:, 12:] *= 300.0
        x = np.concatenate([X.ravel(), Jp.ravel(), U.ravel()])
        out = np.argwhere((kr.jac_exact(pb, x) != 0) & ~inpat)
        assert out.size == 0, ("(row, col) non-zero outside the pattern", out[:5])
