"""Lagrangian Hessian of the kino-dynamic NLP on the GPU (landing_kino_hess_batch): every CCS entry of sampled scenarios
against the exact Hessian of the oracle (tests/kino_hess_ref.py:hess_exact) over knot counts, ragged batches, both layouts,
both memory spaces, random parameters, knot spacings and a different lam_f per scenario; NULL multipliers; that every
output entry is written on every call; the literal launch count of each call; refused arguments; and, at the two stored
KNITRO solutions, H d against central differences of the library's own grad f + J' lam_g."""
import ctypes
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import kino_ref as kr  # noqa: E402
import kino_hess_ref as kh  # noqa: E402
from test_kino_exact import random_problem, random_x, sample, kino_problem  # noqa: E402

pytestmark = pytest.mark.gpu


def random_setup(rng, s):
    """landing_kino_setup with random QN and terminal references (the references do not enter the Hessian)."""
    ks = s.kino_setup_data()
    QN, ref = rng.uniform(0, 100, 12), rng.uniform(-0.5, 0.5, 12)
    for i in range(12):
        ks.QN[i] = QN[i]
    for i in range(6):
        ks.q_term_ref[i], ks.qd_term_ref[i] = ref[i], ref[6 + i]
    return ks, QN, ref


def expected_launches(B, layout, lam_g):
    """Three Hessian kernels; AoS batches of 64 or more add the transposes of x, lam_g (when given) and hess."""
    return 3 + ((2 + (lam_g is not None)) if layout == "AOS" and B >= 64 else 0)


def hessian(s, lc, x, pb, lam_f, lam_g, ks, layout, memspace):
    """hess [B, nnzH] (AoS numpy) from one call in the given layout and memory space; asserts the literal launch count.
    Device outputs are pre-filled with NaN, so an entry that no kernel writes shows."""
    B = x.shape[0]
    lay = getattr(lc, layout)
    tr = (lambda a: a) if layout == "AOS" else (lambda a: None if a is None else np.ascontiguousarray(a.T))
    xin, lgin = tr(x), tr(lam_g)
    l0 = s.launches
    if memspace == "HOST":
        h = s.kino_hess_host(xin, pb, lam_f=lam_f, lam_g=lgin, ks=ks, layout=lay)
    else:
        import torch
        dev = torch.device("cuda:0")
        nnz = len(s.kino_hess_sparsity()[1])
        ht = torch.full((B, nnz) if layout == "AOS" else (nnz, B), float("nan"), dtype=torch.float64, device=dev)
        t = (lambda a: None if a is None else torch.tensor(a, device=dev))
        args = [t(xin), t(lam_f), t(lgin)]
        torch.cuda.synchronize()
        s.kino_hess_device(args[0], pb, ht, lam_f=args[1], lam_g=args[2], ks=ks, layout=lay)
        s.synchronize()
        h = ht.cpu().numpy()
        assert not np.isnan(h).any(), "an output entry was not written"
    assert s.launches - l0 == expected_launches(B, layout, lam_g)
    return h if layout == "AOS" else np.ascontiguousarray(h.T)


def check_against_exact(s, pbo, x, lam_f, lam_g, QN, h, bs):
    pattern = s.kino_hess_sparsity()
    worst = 0.0
    for b in bs:
        He = kh.hess_exact(pbo, x[b], None if lam_f is None else lam_f[b], None if lam_g is None else lam_g[b], QN,
                           None, pattern)
        e = np.abs(h[b] - He) / np.maximum(1.0, np.abs(He))
        assert e.max() <= 1e-12, (b, e.max(), int(e.argmax()))
        worst = max(worst, e.max())
    return worst


# (N, B, layout, memory space): every N, B in {1, 63, 64, 129, 257} (direct AoS below 64, the transposed AoS path from
# 64, partial CTAs of 128 threads), both layouts, host and device buffers
CASES = [(3, 1, "AOS", "HOST"), (3, 257, "SOA", "DEVICE"), (4, 63, "AOS", "HOST"), (4, 129, "AOS", "DEVICE"),
         (21, 64, "AOS", "HOST"), (21, 257, "SOA", "HOST"), (21, 1, "SOA", "DEVICE"), (30, 129, "SOA", "HOST"),
         (30, 64, "AOS", "DEVICE"), (30, 63, "AOS", "DEVICE")]


@pytest.mark.parametrize("N,B,layout,memspace", CASES)
def test_gpu_kino_hess_matches_the_exact_hessian(N, B, layout, memspace):
    import landing_controller_b200 as lc
    rng = np.random.default_rng(2000 * N + B)
    s = lc.LandingSolver(N=N, device=0)
    pbo = random_problem(rng, N)
    x = random_x(rng, N, B)
    lam_f = rng.uniform(0.1, 3.0, B)
    lam_g = rng.normal(size=(B, kr.dims(N)["m"]))
    ks, QN, _ = random_setup(rng, s)
    h = hessian(s, lc, x, kino_problem(s, pbo), lam_f, lam_g, ks, layout, memspace)
    w = check_against_exact(s, pbo, x, lam_f, lam_g, QN, h, sample(rng, B))
    print("kino hess N=%d B=%d %s %s: worst rel. error %.2e" % (N, B, layout, memspace, w))
    s.close()


@pytest.mark.parametrize("layout,memspace", [("AOS", "DEVICE"), ("SOA", "HOST")])
def test_gpu_kino_hess_null_multipliers(layout, memspace):
    """lam_f NULL, lam_g NULL, and both NULL (an all-zero result, every entry written)."""
    import landing_controller_b200 as lc
    N, B = 4, 65
    rng = np.random.default_rng(31)
    s = lc.LandingSolver(N=N, device=0)
    pbo = random_problem(rng, N)
    pb = kino_problem(s, pbo)
    x = random_x(rng, N, B)
    lam_f, lam_g = rng.uniform(0.1, 3.0, B), rng.normal(size=(B, kr.dims(N)["m"]))
    ks, QN, _ = random_setup(rng, s)
    for lf, lg in ((None, lam_g), (lam_f, None)):
        h = hessian(s, lc, x, pb, lf, lg, ks if lf is not None else None, layout, memspace)
        check_against_exact(s, pbo, x, lf, lg, QN, h, [0, 64])
    h = hessian(s, lc, x, pb, None, None, None, layout, memspace)
    assert not np.any(h)
    s.close()


def test_gpu_kino_hess_second_call_sees_new_inputs():
    """One context, host buffers, the transposed AoS path: (x1, pb1, lam1) and then (x2, pb2, lam2); the second
    result must be that of the second inputs (no stale staging, no cached parameters or spacings)."""
    import landing_controller_b200 as lc
    N, B = 21, 129
    rng = np.random.default_rng(6)
    s = lc.LandingSolver(N=N, device=0)
    m = kr.dims(N)["m"]
    p1, p2 = random_problem(rng, N), random_problem(rng, N)
    x1, x2 = random_x(rng, N, B), random_x(rng, N, B)
    lf1, lf2 = rng.uniform(0.1, 3, B), rng.uniform(0.1, 3, B)
    lg1, lg2 = rng.normal(size=(B, m)), rng.normal(size=(B, m))
    (ks1, QN1, _), (ks2, QN2, _) = random_setup(rng, s), random_setup(rng, s)
    h1 = s.kino_hess_host(x1, kino_problem(s, p1), lam_f=lf1, lam_g=lg1, ks=ks1)
    h2 = s.kino_hess_host(x2, kino_problem(s, p2), lam_f=lf2, lam_g=lg2, ks=ks2)
    check_against_exact(s, p1, x1, lf1, lg1, QN1, h1, [0])
    w = check_against_exact(s, p2, x2, lf2, lg2, QN2, h2, [0, 77, B - 1])
    print("kino hess second call: worst rel. error %.2e" % w)
    s.close()


def test_gpu_kino_hess_refused_arguments_leave_the_context_usable():
    """Each refused call returns LANDING_ERR_ARG and is followed by a good call with the same result as before; B = 0
    succeeds and launches nothing."""
    import landing_controller_b200 as lc
    from landing_controller_b200.api import _ptr
    N, B = 4, 5
    rng = np.random.default_rng(8)
    s = lc.LandingSolver(N=N, device=0)
    lib = s.lib
    pbo = random_problem(rng, N)
    pb = kino_problem(s, pbo)
    nnz = len(s.kino_hess_sparsity()[1])
    x = random_x(rng, N, B)
    lam_f, lam_g = rng.uniform(0.1, 3, B), rng.normal(size=(B, kr.dims(N)["m"]))
    ks, _, _ = random_setup(rng, s)
    ref = s.kino_hess_host(x, pb, lam_f=lam_f, lam_g=lam_g, ks=ks)
    no_dt = lc.api.KinoProblem()
    no_dt.mu, no_dt.mass = pb.mu, pb.mass
    out = np.zeros((B, nnz))

    def call(ctx=s.ctx, B_=B, pb_=pb, ks_=ks, x_=x, lf=lam_f, hs=out):
        return lib.landing_kino_hess_batch(ctx, B_, lc.HOST, lc.AOS, None if pb_ is None else ctypes.byref(pb_),
                                           None if ks_ is None else ctypes.byref(ks_), _ptr(x_), _ptr(lf),
                                           _ptr(lam_g), _ptr(hs))

    bad = [dict(ctx=None), dict(pb_=None), dict(pb_=no_dt), dict(x_=None), dict(hs=None), dict(B_=-1), dict(ks_=None)]
    for kw in bad:
        l0 = s.launches
        assert call(**kw) == 1, kw
        assert s.launches == l0
        out[:] = np.nan
        assert call() == 0
        assert np.array_equal(out, ref), kw
    l0 = s.launches
    assert call(B_=0) == 0 and s.launches == l0
    assert call(ks_=None, lf=None) == 0  # lam_f NULL: ks may be NULL
    s.close()


def test_gpu_kino_hess_is_the_derivative_of_the_library_gradient_at_the_stored_solutions():
    """At both stored KNITRO points (tests/golden/kino_n21.npz) with their stored lam_g and lam_f = 1, H d equals the
    central difference of the library's own grad f + J' lam_g (landing_kino_cost_batch, landing_kino_eval_batch) along
    random directions d."""
    import landing_controller_b200 as lc
    N = 21
    d = np.load(os.path.join(ROOT, "tests", "golden", "kino_n21.npz"))
    s = lc.LandingSolver(N=N, device=0)
    pb = s.kino_problem(kr.DT_VAL)
    ks = s.kino_setup_data()
    colJ, rowJ = s.kino_sparsity()
    colJ_of = np.repeat(np.arange(len(colJ) - 1), np.diff(colJ))
    colH, rowH = s.kino_hess_sparsity()
    colH_of = np.repeat(np.arange(len(colH) - 1), np.diff(colH))
    rng = np.random.default_rng(21)
    for key in ("gs", "ms"):
        x, lam = d[key + "_x"], d[key + "_lam_g"]
        nx = x.size

        def grad(xs):  # [B, nx] -> [B, nx]
            _, gf = s.kino_cost_host(xs, ks=ks)
            _, jac = s.kino_eval_host(xs, pb, want_g=False)
            out = gf.copy()
            for b in range(xs.shape[0]):
                np.add.at(out[b], colJ_of, jac[b] * lam[rowJ])
            return out

        h = s.kino_hess_host(x[None], pb, lam_f=np.ones(1), lam_g=lam[None], ks=ks)[0]
        eps = 1e-4
        dirs = rng.normal(size=(4, nx))
        g = grad(np.concatenate([x + eps * dirs, x - eps * dirs]))
        for i, dv in enumerate(dirs):
            Hd = np.zeros(nx)
            np.add.at(Hd, rowH, h * dv[colH_of])
            off = rowH != colH_of
            np.add.at(Hd, colH_of[off], h[off] * dv[rowH[off]])
            fd = (g[i] - g[4 + i]) / (2 * eps)
            err = np.abs(fd - Hd).max() / np.abs(Hd).max()
            assert err <= 1e-6, (key, i, err)
    s.close()
