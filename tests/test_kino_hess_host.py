"""Lagrangian Hessian of the kino-dynamic NLP on the CPU: the exact (dual x complex-step) Hessian of the oracle,
tests/kino_hess_ref.py:hess_exact, against finite differences of the exact gradient; the product's knot template under the
second-order type and its Hessian pass table (kino_knot.cuh) compiled for the host against that exact Hessian; and the
library's upper-triangle CCS pattern against every exact non-zero, with one writer per entry."""
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
import kino_hess_ref as kh  # noqa: E402

NIN = 72
_dp = ctypes.POINTER(ctypes.c_double)
_ip = ctypes.POINTER(ctypes.c_int)


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    """tests/hostcheck/kino_hess_host.cpp, built into a temporary directory (the checkout may be read-only)."""
    so = str(tmp_path_factory.mktemp("kino_hess_host") / "libkino_hess_host.so")
    src = os.path.join(ROOT, "tests", "hostcheck", "kino_hess_host.cpp")
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
    for o in (0, 48):
        z[o + 3:o + 6] = rng.uniform(-1, 1, 3)
        z[o + 6:o + 12] = rng.uniform(-3, 3, 6)
    z[12:24] = rng.uniform(-1, 1, 12)
    z[36:48] = rng.uniform(-100, 100, 12)
    z[38:48:3] = rng.uniform(0, 300, 4)
    return z


def random_x(rng, N):
    X, J, U = kr.split(rng.uniform(-1, 1, kr.dims(N)["nx"]), N)
    U[:, 12:] *= 300.0
    return np.concatenate([X.ravel(), J.ravel(), U.ravel()])


def _prm(p):
    return np.concatenate([[p["mu"], p["mass"]], p["Ib"], p["Ib_inv"]])


def pass_table(harness):
    a, b, in_last = (np.zeros(64, dtype=np.int32) for _ in range(3))
    n = harness.kino_hess_host_table(_ptr(a, _ip), _ptr(b, _ip), _ptr(in_last, _ip))
    return a[:n], b[:n], in_last[:n]


def test_exact_hessian_agrees_with_finite_differences_of_the_exact_gradient():
    """Every column of hess_exact against the central difference of lam_f grad f + J' lam_g (jac_exact), N = 3 and 4,
    random parameters, knot spacings and multipliers; the dense result is symmetric."""
    rng = np.random.default_rng(11)
    for N in (3, 4):
        pb = dict(kr.default_problem(N), **random_params(rng))
        pb["dt"] = rng.uniform(0.01, 0.1, N - 1)
        d = kr.dims(N)
        x = random_x(rng, N) * 0.5
        lam, lam_f, QN = rng.normal(size=d["m"]), rng.uniform(0.5, 2.0), rng.uniform(0, 100, 12)
        xo = 12 * (N - 1)

        def grad(xx):
            gf = np.zeros(d["nx"])
            gf[xo:xo + 12] = 2 * QN * xx[xo:xo + 12]
            return lam_f * gf + kr.jac_exact(pb, xx).T @ lam

        H = kh.hess_exact(pb, x, lam_f, lam, QN, np.zeros(12))
        scale = np.abs(H).max()
        assert np.abs(H - H.T).max() <= 1e-13 * scale
        eps = 1e-6
        for c in range(d["nx"]):
            e = np.zeros(d["nx"])
            e[c] = eps
            fd = (grad(x + e) - grad(x - e)) / (2 * eps)
            assert np.abs(fd - H[:, c]).max() <= 1e-6 * max(1.0, np.abs(H[:, c]).max()), (N, c)


@pytest.mark.parametrize("last", [False, True])
def test_hessian_passes_match_the_exact_knot_hessian_and_cover_it_once(harness, last):
    """kino_knot.cuh compiled for the host: every pass of the Hessian table (second-order type, masks, seeding, the
    last-knot skip), contracted with random multipliers, against the exact knot-local Hessian of the oracle at random
    points, parameters and knot spacings; the union of the passes covers every exact non-zero of the upper triangle
    exactly once."""
    rng = np.random.default_rng(23 + last)
    nin, nrow = (60, 117) if last else (72, 141)
    worst = 0.0
    for _ in range(12):
        z = random_knot(rng)
        pb = dict(random_params(rng), dt=[rng.uniform(0.005, 0.2)])
        lam = np.zeros(141)
        lam[:nrow] = rng.normal(size=nrow)
        Hp, cnt = np.zeros((NIN, NIN)), np.zeros((NIN, NIN), dtype=np.int32)
        harness.kino_hess_host_passes(int(last), _ptr(z), ctypes.c_double(pb["dt"][0]), _ptr(_prm(pb)), _ptr(lam),
                                      _ptr(Hp), _ptr(cnt, _ip))
        He = np.triu(kh.knot_hess(pb, 0, z[:nin], lam[:nrow], last))
        assert cnt.max() <= 1, np.argwhere(cnt > 1)[:5]
        assert not np.any(cnt[nin:]) and not np.any(cnt[:, nin:])
        missing = np.argwhere((He != 0) & (cnt[:nin, :nin] == 0))
        assert missing.size == 0, ("exact non-zero not covered by any pass", missing[:5])
        err = np.max(np.abs(Hp[:nin, :nin] - He) / np.maximum(1.0, np.abs(He)))
        worst = max(worst, err)
        assert err <= 1e-12, err
    print("Hessian passes (last=%d) vs exact: worst rel. error %.2e" % (last, worst))


@pytest.mark.parametrize("N", [3, 4, 21])
def test_library_kino_hess_pattern_holds_every_exact_nonzero_with_one_writer(harness, N):
    """landing_kino_hess_sparsity(N) (host logic, no GPU): upper triangular, rows sorted within each column, consistent
    colind; contains every non-zero of the exact Hessian at random points, parameters and multipliers; and each of its
    entries is reached by exactly one writer -- one (knot, pass, block entry) of the pass table or the terminal-cost
    diagonal of the last knot."""
    import landing_controller_b200 as lc
    lib = lc.load_library()
    nx = kr.dims(N)["nx"]
    sp = lib.landing_kino_hess_sparsity(N)
    assert sp, lib.landing_last_error()
    assert sp[0] == nx and sp[1] == nx
    colind = np.ctypeslib.as_array(sp, shape=(2 + nx + 1,))[2:].copy()
    nnz = int(colind[-1])
    row = np.ctypeslib.as_array(sp, shape=(2 + nx + 1 + nnz,))[2 + nx + 1:].copy()
    assert colind[0] == 0 and np.all(np.diff(colind) >= 0)
    col = np.repeat(np.arange(nx), np.diff(colind))
    assert np.all(row <= col) and np.all(row >= 0)
    for c in range(nx):
        assert np.all(np.diff(row[colind[c]:colind[c + 1]]) > 0)
    inpat = np.zeros((nx, nx), dtype=bool)
    inpat[row, col] = True
    assert not lib.landing_kino_hess_sparsity(2)
    # every exact non-zero
    rng = np.random.default_rng(100 + N)
    m = kr.dims(N)["m"]
    for _ in range(2 if N == 21 else 4):
        pb = dict(kr.default_problem(N), **random_params(rng))
        pb["dt"] = rng.uniform(0.01, 0.1, N - 1)
        H = np.triu(kh.hess_exact(pb, random_x(rng, N), rng.uniform(0.5, 2), rng.normal(size=m),
                                  rng.uniform(1, 100, 12), np.zeros(12)))
        out = np.argwhere((H != 0) & ~inpat)
        assert out.size == 0, ("(row, col) non-zero outside the pattern", out[:5])
    # writers: every block entry of every pass in every knot, and the cost diagonal
    a, b, in_last = pass_table(harness)
    assert len(set(zip(a.tolist(), b.tolist()))) == len(a) and np.all(a <= b)
    writers = np.zeros((nx, nx), dtype=np.int32)
    for k in range(N - 1):
        last = k == N - 2
        for P in range(len(a)):
            if last and not in_last[P]:
                continue
            for i in range(3):
                for j in range(i if a[P] == b[P] else 0, 3):
                    ci, cj = kr.knot_col(N, k, 3 * a[P] + i), kr.knot_col(N, k, 3 * b[P] + j)
                    writers[min(ci, cj), max(ci, cj)] += 1
    xo = 12 * (N - 1)
    writers[np.arange(xo, xo + 12), np.arange(xo, xo + 12)] += 1
    assert np.all(writers[row, col] == 1), np.argwhere(inpat & (writers != 1))[:5]
