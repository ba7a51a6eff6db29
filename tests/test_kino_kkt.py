"""Lagrangian gradient and KKT residuals of the kino-dynamic NLP on the GPU (landing_kino_kkt_batch): every grad_x entry
of sampled scenarios against lam_f grad f + J' lam_g with the oracle's exact Jacobian over knot counts, ragged batches,
both layouts, both memory spaces, random parameters and knot spacings; NULL multipliers; that every output entry is
written on every call; the literal launch count of each call; bit-identical results across layouts and memory spaces;
refused arguments; the residuals against numpy, with infinite bounds, equality rows, wrong-sign multipliers and a NaN in
one scenario; and the two stored KNITRO points."""
import ctypes
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import kino_ref as kr  # noqa: E402
from test_kino_exact import random_problem, random_x, sample, kino_problem  # noqa: E402
from test_kino_hess import random_setup  # noqa: E402
from test_kino_grad_host import grad_reference, kkt_reference, QN_DEFAULT, REF_DEFAULT  # noqa: E402

pytestmark = pytest.mark.gpu
ALL = ("grad_x", "viol", "dual_inf", "compl_inf")


def expected_launches(B, layout, want, lam_g, bounds):
    """The launch count documented by landing_kino_kkt_batch in capi.cu."""
    if not want:
        return 0
    n = 6 * ("grad_x" in want or "dual_inf" in want) + ("viol" in want or "compl_inf" in want)
    n += any(w in want for w in ("viol", "dual_inf", "compl_inf"))
    if layout == "AOS" and B >= 64:
        n += 1 + (lam_g is not None) + 2 * bounds + ("grad_x" in want)
    return n


def kkt(s, lc, x, pb, lam_f=None, lam_g=None, lbg=None, ubg=None, ks=None, want=ALL, layout="AOS", memspace="HOST"):
    """The wanted outputs (AoS numpy) of one call in the given layout and memory space; asserts the literal launch count.
    Device outputs are pre-filled with NaN, so an entry that no kernel writes shows."""
    B, nx = x.shape
    lay = getattr(lc, layout)
    tr = (lambda a: a) if layout == "AOS" else (lambda a: None if a is None else np.ascontiguousarray(a.T))
    xin, lgin, lbin, ubin = tr(x), tr(lam_g), tr(lbg), tr(ubg)
    if lam_f is not None and ks is None:
        ks = s.kino_setup_data()
    l0 = s.launches
    if memspace == "HOST":
        out = s.kino_kkt_host(xin, pb, lam_f=lam_f, lam_g=lgin, lbg=lbin, ubg=ubin, ks=ks, want=want, layout=lay)
    else:
        import torch
        dev = torch.device("cuda:0")
        t = (lambda a: None if a is None else torch.tensor(a, device=dev))
        outs = {k: torch.full((B,), float("nan"), dtype=torch.float64, device=dev) for k in want if k != "grad_x"}
        if "grad_x" in want:
            outs["grad_x"] = torch.full((B, nx) if layout == "AOS" else (nx, B), float("nan"), dtype=torch.float64,
                                        device=dev)
        args = dict(x=t(xin), lam_f=t(lam_f), lam_g=t(lgin), lbg=t(lbin), ubg=t(ubin))
        torch.cuda.synchronize()
        s.kino_kkt_device(args["x"], pb, lam_f=args["lam_f"], lam_g=args["lam_g"], lbg=args["lbg"], ubg=args["ubg"],
                          ks=ks, layout=lay, **outs)
        s.synchronize()
        out = {k: v.cpu().numpy() for k, v in outs.items()}
        finite = all(a is None or np.isfinite(a).all() for a in (x, lam_f, lam_g))  # (NaN inputs give NaN entries)
        if "grad_x" in out and finite:
            assert not np.isnan(out["grad_x"]).any(), "an output entry was not written"
    assert s.launches - l0 == expected_launches(B, layout, want, lam_g, lbg is not None)
    if "grad_x" in out and layout == "SOA":
        out["grad_x"] = np.ascontiguousarray(out["grad_x"].T)
    return out


def check_grad(pbo, x, lam_f, lam_g, QN, ref, grad, bs):
    worst = 0.0
    for b in bs:
        r, scale = grad_reference(pbo, x[b], None if lam_f is None else lam_f[b], None if lam_g is None else lam_g[b],
                                  QN, ref)
        e = np.abs(grad[b] - r) / np.maximum(1.0, scale)
        assert e.max() <= 1e-12, (b, e.max(), int(e.argmax()))
        worst = max(worst, e.max())
    return worst


# (N, B, layout, memory space): every N, B in {1, 63, 64, 129, 257} (direct AoS below 64, the transposed AoS path from
# 64, partial CTAs of 128 threads), both layouts, host and device buffers
CASES = [(3, 1, "AOS", "HOST"), (3, 257, "SOA", "DEVICE"), (4, 63, "AOS", "HOST"), (4, 129, "AOS", "DEVICE"),
         (21, 64, "AOS", "HOST"), (21, 257, "SOA", "HOST"), (21, 1, "SOA", "DEVICE"), (30, 129, "SOA", "HOST"),
         (30, 64, "AOS", "DEVICE"), (30, 63, "AOS", "DEVICE")]


@pytest.mark.parametrize("N,B,layout,memspace", CASES)
def test_gpu_kino_grad_matches_the_exact_reference(N, B, layout, memspace):
    import landing_controller_b200 as lc
    rng = np.random.default_rng(3000 * N + B)
    s = lc.LandingSolver(N=N, device=0)
    pbo = random_problem(rng, N)
    x = random_x(rng, N, B)
    lam_f = rng.uniform(0.1, 3.0, B)
    lam_g = rng.normal(size=(B, kr.dims(N)["m"]))
    ks, QN, ref = random_setup(rng, s)
    out = kkt(s, lc, x, kino_problem(s, pbo), lam_f=lam_f, lam_g=lam_g, ks=ks, want=("grad_x",), layout=layout,
              memspace=memspace)
    w = check_grad(pbo, x, lam_f, lam_g, QN, ref, out["grad_x"], sample(rng, B))
    print("kino grad N=%d B=%d %s %s: worst rel. error %.2e" % (N, B, layout, memspace, w))
    s.close()


@pytest.mark.parametrize("layout,memspace", [("AOS", "DEVICE"), ("SOA", "HOST")])
def test_gpu_kino_grad_null_multipliers(layout, memspace):
    """lam_f NULL, lam_g NULL, and both NULL (an all-zero result, every entry written)."""
    import landing_controller_b200 as lc
    N, B = 4, 65
    rng = np.random.default_rng(32)
    s = lc.LandingSolver(N=N, device=0)
    pbo = random_problem(rng, N)
    pb = kino_problem(s, pbo)
    x = random_x(rng, N, B)
    lam_f, lam_g = rng.uniform(0.1, 3.0, B), rng.normal(size=(B, kr.dims(N)["m"]))
    ks, QN, ref = random_setup(rng, s)
    for lf, lg in ((None, lam_g), (lam_f, None)):
        out = kkt(s, lc, x, pb, lam_f=lf, lam_g=lg, ks=ks if lf is not None else None, want=("grad_x", "dual_inf"),
                  layout=layout, memspace=memspace)
        check_grad(pbo, x, lf, lg, QN, ref, out["grad_x"], [0, 64])
        assert np.array_equal(out["dual_inf"], np.abs(out["grad_x"]).max(1))
    out = kkt(s, lc, x, pb, want=("grad_x", "dual_inf"), layout=layout, memspace=memspace)
    assert not np.any(out["grad_x"]) and not np.any(out["dual_inf"])
    s.close()


def test_gpu_kino_kkt_second_call_sees_new_inputs():
    """One context, host buffers, the transposed AoS path: (x1, pb1, lam1) and then (x2, pb2, lam2); the second result
    must be that of the second inputs (no stale staging, scratch, parameters or spacings)."""
    import landing_controller_b200 as lc
    N, B = 21, 129
    rng = np.random.default_rng(7)
    s = lc.LandingSolver(N=N, device=0)
    m = kr.dims(N)["m"]
    p1, p2 = random_problem(rng, N), random_problem(rng, N)
    x1, x2 = random_x(rng, N, B), random_x(rng, N, B)
    lf1, lf2 = rng.uniform(0.1, 3, B), rng.uniform(0.1, 3, B)
    lg1, lg2 = rng.normal(size=(B, m)), rng.normal(size=(B, m))
    (ks1, QN1, r1), (ks2, QN2, r2) = random_setup(rng, s), random_setup(rng, s)
    o1 = kkt(s, lc, x1, kino_problem(s, p1), lam_f=lf1, lam_g=lg1, ks=ks1, want=("grad_x",))
    o2 = kkt(s, lc, x2, kino_problem(s, p2), lam_f=lf2, lam_g=lg2, ks=ks2, want=("grad_x",))
    check_grad(p1, x1, lf1, lg1, QN1, r1, o1["grad_x"], [0])
    w = check_grad(p2, x2, lf2, lg2, QN2, r2, o2["grad_x"], [0, 77, B - 1])
    print("kino grad second call: worst rel. error %.2e" % w)
    s.close()


def random_bounds(rng, B, N):
    """lbg / ubg of the oracle's row layout (equality rows, one-sided rows with an infinite bound, boxes) at random
    drops and random boxes."""
    lb, ub = [], []
    for _ in range(B):
        pbo = kr.default_problem(N)
        pbo["kin_box"] = rng.uniform(0, 0.2, 2)
        lo, up = kr.bounds(pbo, rng.normal(size=6), rng.normal(size=6), rng.normal(size=12))
        lb.append(lo), ub.append(up)
    return np.array(lb), np.array(ub)


def kkt_point(rng, N, B):
    """A random primal-dual point with bounds: lam_g with wrong-sign multipliers on infinite bounds in the odd scenarios
    only (compl_inf = +inf there), zero multipliers elsewhere on those rows."""
    pbo = random_problem(rng, N)
    x = random_x(rng, N, B)
    lbg, ubg = random_bounds(rng, B, N)
    lam_g = rng.normal(size=lbg.shape)
    wrong = ((lam_g > 0) & np.isinf(ubg)) | ((lam_g < 0) & np.isinf(lbg))
    lam_g[::2][wrong[::2]] = 0.0
    return pbo, x, lbg, ubg, lam_g, rng.uniform(0.1, 3.0, B)


def test_gpu_kino_kkt_scalars_match_numpy_and_nan_stays_in_its_scenario():
    import landing_controller_b200 as lc
    N, B = 4, 70
    rng = np.random.default_rng(11)
    s = lc.LandingSolver(N=N, device=0)
    pbo, x, lbg, ubg, lam_g, lam_f = kkt_point(rng, N, B)
    ks, QN, ref = random_setup(rng, s)
    x[3, 17] = np.nan        # x of scenario 3
    lam_g[5, 50] = np.nan    # lam_g of scenario 5 (on a dynamics row, an equality row)
    lbg[8, 300] = np.nan     # a bound of scenario 8
    lam_f[9] = np.nan        # lam_f of scenario 9
    bad = {3, 5, 8, 9}
    pb = kino_problem(s, pbo)
    for layout, memspace in (("AOS", "HOST"), ("SOA", "DEVICE")):
        out = kkt(s, lc, x, pb, lam_f=lam_f, lam_g=lam_g, lbg=lbg, ubg=ubg, ks=ks, layout=layout, memspace=memspace)
        for b in range(B):
            if b in bad:
                assert np.isnan([out["viol"][b], out["dual_inf"][b], out["compl_inf"][b]]).all(), b
                continue
            g = kr.eval_g(pbo, x[b], literal=False)
            gr, scale = grad_reference(pbo, x[b], lam_f[b], lam_g[b], QN, ref)
            viol, dual, compl = kkt_reference(g, lbg[b], ubg[b], lam_g[b], gr)
            assert not np.isnan(out["grad_x"][b]).any()
            assert abs(out["viol"][b] - viol) <= 1e-12 * max(1.0, np.abs(g).max()), (b, out["viol"][b], viol)
            assert abs(out["dual_inf"][b] - dual) <= 1e-12 * max(1.0, scale.max()), (b, out["dual_inf"][b], dual)
            if np.isinf(compl):
                assert out["compl_inf"][b] == np.inf and b % 2 == 1, b
            else:
                e = np.abs(g).max() + np.abs(np.where(np.isfinite(lbg[b]), lbg[b], 0)).max() + np.abs(ubg[b][np.isfinite(ubg[b])]).max()
                assert abs(out["compl_inf"][b] - compl) <= 1e-12 * max(1.0, np.abs(lam_g[b]).max() * e), (b, compl)
        assert np.isinf(out["compl_inf"][1::2][[b not in bad for b in range(1, B, 2)]]).all()
    s.close()


def test_gpu_kino_kkt_is_bit_identical_across_layouts_and_memory_spaces():
    """All four outputs, every combination of layout and memory space, direct (B = 63) and transposed (B = 129) AoS."""
    import landing_controller_b200 as lc
    N = 21
    rng = np.random.default_rng(12)
    s = lc.LandingSolver(N=N, device=0)
    for B in (63, 129):
        pbo, x, lbg, ubg, lam_g, lam_f = kkt_point(rng, N, B)
        pb = kino_problem(s, pbo)
        ks, _, _ = random_setup(rng, s)
        res = [kkt(s, lc, x, pb, lam_f=lam_f, lam_g=lam_g, lbg=lbg, ubg=ubg, ks=ks, layout=lay, memspace=mem)
               for lay in ("AOS", "SOA") for mem in ("HOST", "DEVICE")]
        res.append(kkt(s, lc, x, pb, lam_f=lam_f, lam_g=lam_g, lbg=lbg, ubg=ubg, ks=ks))  # run to run
        for r in res[1:]:
            for k in ALL:
                assert np.array_equal(r[k], res[0][k]), (B, k)
    s.close()


def test_gpu_kino_kkt_launch_counts_of_every_output_combination():
    import itertools
    import landing_controller_b200 as lc
    N = 3
    rng = np.random.default_rng(13)
    s = lc.LandingSolver(N=N, device=0)
    pb = kino_problem(s, random_problem(rng, N))
    for B in (5, 64):
        _, x, lbg, ubg, lam_g, lam_f = kkt_point(rng, N, B)
        for r in range(1, 5):
            for want in itertools.combinations(ALL, r):
                for lg in (None, lam_g):
                    kkt(s, lc, x, pb, lam_f=lam_f, lam_g=lg, lbg=lbg, ubg=ubg, want=want)  # asserts the count
                if "viol" not in want and "compl_inf" not in want:
                    kkt(s, lc, x, pb, lam_g=lam_g, want=want)
    l0 = s.launches
    kkt(s, lc, x, pb, want=())
    assert s.launches == l0
    s.close()


def test_gpu_kino_kkt_refused_arguments_leave_the_context_usable():
    """Each refused call returns LANDING_ERR_ARG and launches nothing, and is followed by a good call with the same
    result as before; B = 0 succeeds and launches nothing."""
    import landing_controller_b200 as lc
    from landing_controller_b200.api import _ptr, KinoKktIO
    N, B = 4, 5
    rng = np.random.default_rng(9)
    s = lc.LandingSolver(N=N, device=0)
    lib = s.lib
    pbo, x, lbg, ubg, lam_g, lam_f = kkt_point(rng, N, B)
    pb = kino_problem(s, pbo)
    ks, _, _ = random_setup(rng, s)
    ref = s.kino_kkt_host(x, pb, lam_f=lam_f, lam_g=lam_g, lbg=lbg, ubg=ubg, ks=ks)
    no_dt = lc.api.KinoProblem()
    no_dt.mu, no_dt.mass = pb.mu, pb.mass
    out = {k: np.zeros((B, x.shape[1])) if k == "grad_x" else np.zeros(B) for k in ALL}

    def call(ctx=s.ctx, B_=B, pb_=pb, ks_=ks, io_=True, x_=x, lf=lam_f, lb=lbg, ub=ubg, viol=True, compl=True):
        io = KinoKktIO(_ptr(x_), _ptr(lf), _ptr(lam_g), _ptr(lb), _ptr(ub), _ptr(out["grad_x"]),
                       _ptr(out["viol"]) if viol else None, _ptr(out["dual_inf"]),
                       _ptr(out["compl_inf"]) if compl else None)
        return lib.landing_kino_kkt_batch(ctx, B_, lc.HOST, lc.AOS, None if pb_ is None else ctypes.byref(pb_),
                                          None if ks_ is None else ctypes.byref(ks_), ctypes.byref(io) if io_ else None)

    bad = [dict(ctx=None), dict(pb_=None), dict(pb_=no_dt), dict(io_=False), dict(x_=None), dict(B_=-1),
           dict(ks_=None), dict(lb=None), dict(ub=None), dict(lb=None, ub=None), dict(lb=None, ub=None, compl=False),
           dict(lb=None, ub=None, viol=False)]
    for kw in bad:
        l0 = s.launches
        assert call(**kw) == 1, kw
        assert s.launches == l0, kw
        for v in out.values():
            v[:] = np.nan
        assert call() == 0
        for k in ALL:
            assert np.array_equal(out[k], ref[k]), (kw, k)
    l0 = s.launches
    assert call(B_=0) == 0 and s.launches == l0
    assert call(ks_=None, lf=None) == 0  # lam_f NULL: ks may be NULL
    assert call(lb=None, ub=None, viol=False, compl=False) == 0  # no bounds: grad_x and dual_inf
    s.close()


@pytest.mark.parametrize("tag,viol_tol", [("ms", 1e-6), ("gs", 5e-5)])
def test_gpu_kino_kkt_at_the_stored_knitro_points(tag, viol_tol):
    """tests/golden/kino_n21.npz with lam_f = 1 and the bounds of landing_kino_setup_batch for the stored drop: viol
    within the tolerance of the stored points' feasibility test, dual_inf and compl_inf equal to the host values
    (tests/test_kino_grad_host.py); dual_inf within 1e-4 of max |J_ij lam_i| at the main_scripts point.  compl_inf is
    +inf at both: the stored multipliers have the wrong sign on a few inequality rows whose violated side is an infinite
    bound (|lam| <= 6e-8)."""
    import landing_controller_b200 as lc
    from test_kino import stored
    N = 21
    s = lc.LandingSolver(N=N, device=0)
    pbo, x, lam, _ = stored(tag)
    X = x[:12 * N].reshape(N, 12)
    lbg, ubg, _ = s.kino_setup_host(X[0][None], want_x0=False)
    pb = kino_problem(s, pbo)
    out = kkt(s, lc, x[None], pb, lam_f=np.ones(1), lam_g=lam[None], lbg=lbg, ubg=ubg)
    g = kr.eval_g(pbo, x, literal=False)
    grad, _ = grad_reference(pbo, x, 1.0, lam, QN_DEFAULT, REF_DEFAULT)
    viol, dual, compl = kkt_reference(g, lbg[0], ubg[0], lam, grad)
    scale = np.abs(kr.jac_exact(pbo, x) * lam[:, None]).max()
    print("%s: viol %.3g dual_inf %.3g (%.3g of max|J_ij lam_i|) compl_inf %g" % (
        tag, out["viol"][0], out["dual_inf"][0], out["dual_inf"][0] / scale, out["compl_inf"][0]))
    assert out["viol"][0] <= viol_tol and abs(out["viol"][0] - viol) <= 1e-12
    assert abs(out["dual_inf"][0] - dual) <= 1e-12 * scale
    assert out["compl_inf"][0] == compl == np.inf
    if tag == "ms":
        assert out["dual_inf"][0] <= 1e-4 * scale
    s.close()
