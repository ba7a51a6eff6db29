"""Interior-point Newton step of the kino-dynamic NLP on the GPU (landing_kino_step_batch), with inputs composed from the
library's own calls (landing_kino_eval_batch, landing_kino_hess_batch, landing_kino_cost_batch): dx, ds, dy, dzL, dzU
against a sparse solve of the full, unreduced system and the linearised residuals of the GPU's own direction, over knot
counts, ragged batches, both layouts and both memory spaces; bit identity across them; the literal launch count; the
fraction-to-boundary step lengths against numpy; inertia correction against the host build; the first iteration from
landing_kino_setup_batch's SRB-based initial guess; failure isolation; refused arguments and B = 0."""
import ctypes
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import kino_ref as kr  # noqa: E402
from test_kino_exact import random_problem, random_x, kino_problem  # noqa: E402
from test_kino_step_host import (harness, patterns, interior_point, full_system, fraction_to_boundary,  # noqa: E402,F401
                                 run_host, ccs, eq_rows, dw_trials)

pytestmark = pytest.mark.gpu
IN = ("g", "jac", "hess", "grad_f", "s", "y", "zL", "zU", "lbg", "ubg")
OUT = ("dx", "ds", "dy", "dzL", "dzU")


def make_inputs(s, rng, N, B, y_scale=1.0):
    """AoS numpy inputs of B scenarios: g / jac from landing_kino_eval_batch, hess with lam_f = 1 and lam_g = y from
    landing_kino_hess_batch, grad_f from landing_kino_cost_batch, the bounds of the drop, an interior iterate."""
    pbo = random_problem(rng, N)
    pb = kino_problem(s, pbo)
    x = random_x(rng, N, B)
    g, jac = s.kino_eval_host(x, pb)
    ks = s.kino_setup_data()
    _, gf = s.kino_cost_host(x, ks)
    cols = {k: [] for k in ("lbg", "ubg", "s", "y", "zL", "zU")}
    for b in range(B):
        lbg, ubg = kr.bounds(pbo, x[b, :6], x[b, 6:12], x[b, 24 * N - 12:24 * N])
        sl, y, zL, zU = interior_point(rng, N, g[b], lbg, ubg, y_scale)
        for k, v in zip(("lbg", "ubg", "s", "y", "zL", "zU"), (lbg, ubg, sl, y, zL, zU)):
            cols[k].append(v)
    inp = {k: np.array(v) for k, v in cols.items()}
    hess = s.kino_hess_host(x, pb, lam_f=np.ones(B), lam_g=inp["y"], ks=ks)
    inp.update(g=g, jac=jac, hess=hess, grad_f=gf, mu=10.0 ** rng.uniform(-3, 0, B), dw_last=np.zeros(B))
    return inp


def step(s, lc, inp, layout, memspace, tau=0.99):
    """One call; AoS numpy outputs.  Device outputs are pre-filled with NaN / -7 so an unwritten entry shows; asserts the
    launch count documented in capi.cu."""
    B = inp["mu"].shape[0]
    tr = (lambda a: a) if layout == "AOS" else (lambda a: np.ascontiguousarray(a.T))
    lay = getattr(lc, layout)
    l0 = s.launches
    if memspace == "HOST":
        out = s.kino_step_host(*[tr(inp[k]) for k in IN], inp["mu"], inp["dw_last"], tau=tau, layout=lay)
    else:
        import torch
        dev = torch.device("cuda:0")
        t = {k: torch.tensor(tr(inp[k]), device=dev) for k in IN}
        t["mu"], t["dw_last"] = torch.tensor(inp["mu"], device=dev), torch.tensor(inp["dw_last"], device=dev)
        d = s.kino_dims()
        shp = lambda n: (B, n) if layout == "AOS" else (n, B)  # noqa: E731
        o = {"dx": torch.full(shp(d["nx"]), float("nan"), dtype=torch.float64, device=dev)}
        for k in OUT[1:]:
            o[k] = torch.full(shp(d["m"]), float("nan"), dtype=torch.float64, device=dev)
        for k in ("delta_w", "alpha_pr", "alpha_du"):
            o[k] = torch.full((B,), float("nan"), dtype=torch.float64, device=dev)
        for k in ("n_factor", "status"):
            o[k] = torch.full((B,), -7, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        s.kino_step_device(t, o, tau=tau, layout=lay)
        s.synchronize()
        out = {k: v.cpu().numpy() for k, v in o.items()}
    assert s.launches - l0 == (16 if layout == "AOS" and B >= 64 else 1)
    if layout == "SOA":
        for k in OUT:
            out[k] = np.ascontiguousarray(out[k].T)
    return out


def dense(sp, vals, sym=False):
    import scipy.sparse as sps
    colind, row = ccs(sp)
    n = int(sp[1])
    col = np.repeat(np.arange(n), np.diff(colind))
    A = sps.csr_matrix((vals, (row, col)), shape=(int(sp[0]), n))
    return A + sps.triu(A, 1).T if sym else A


@pytest.mark.parametrize("N,B", [(3, 67), (5, 5), (21, 65)])
def test_gpu_step_solves_the_full_system(N, B):
    """Sampled scenarios against a sparse solve of the unreduced system (1e-9 relative), the GPU direction's own
    linearised residuals, alpha_pr / alpha_du against numpy exactly; the same bits in both layouts and memory spaces."""
    import landing_controller_b200 as lc
    s = lc.LandingSolver(N=N, device=0)
    rng = np.random.default_rng(N * 7 + B)
    inp = make_inputs(s, rng, N, B)
    inp["dw_last"][1::3] = 3e-3
    res = {}
    for layout in ("AOS", "SOA"):
        for memspace in ("HOST", "DEVICE"):
            res[(layout, memspace)] = step(s, lc, inp, layout, memspace)
    ref = res[("AOS", "HOST")]
    for key, o in res.items():
        for k in OUT + ("delta_w", "n_factor", "status", "alpha_pr", "alpha_du"):
            assert np.array_equal(o[k], ref[k], equal_nan=True), (key, k)
    assert np.all(ref["status"] == 0)
    jsp, hsp = patterns(N)
    worst = worst_res = 0.0
    for b in sorted({0, B - 1} | set(rng.choice(B, size=min(3, B), replace=False).tolist())):
        J, W = dense(jsp, inp["jac"][b]), dense(hsp, inp["hess"][b], sym=True)
        args = [inp[k][b] for k in ("grad_f", "g", "s", "y", "zL", "zU", "lbg", "ubg")]
        exact, (A, rhs, pack) = full_system(N, J, W, *args, inp["mu"][b], ref["delta_w"][b], want_system=True)
        for name, e in zip(OUT, exact):
            err = float(np.max(np.abs(ref[name][b] - e)) / max(1.0, float(np.max(np.abs(e)))))
            worst = max(worst, err)
            assert err < 1e-9, (b, name, err)
        z = pack(*[ref[k][b] for k in OUT])
        r = np.max(np.abs(A @ z - rhs)) / (abs(A).max() * np.max(np.abs(z)) + np.max(np.abs(rhs)))
        worst_res = max(worst_res, r)
        assert r < 1e-13, (b, r)
        apr, adu = fraction_to_boundary(N, inp["s"][b], ref["ds"][b], inp["zL"][b], ref["dzL"][b], inp["zU"][b],
                                        ref["dzU"][b], inp["lbg"][b], inp["ubg"][b], 0.99)
        assert apr == ref["alpha_pr"][b] and adu == ref["alpha_du"][b]
    print("N=%d B=%d: worst %.2e vs full system, residual %.2e, delta_w %s" %
          (N, B, worst, worst_res, np.unique(ref["delta_w"]).tolist()))


def test_gpu_step_inertia_correction_matches_the_host_build(harness):  # noqa: F811
    """Large random y: scenarios need delta_w > 0; delta_w and n_factor equal the host build's exactly."""
    import landing_controller_b200 as lc
    N, B = 5, 8
    s = lc.LandingSolver(N=N, device=0)
    rng = np.random.default_rng(11)
    inp = make_inputs(s, rng, N, B, y_scale=100.0)
    inp["dw_last"][4:] = rng.uniform(1e-6, 1.0, 4)
    out = step(s, lc, inp, "SOA", "DEVICE")
    jsp, hsp = patterns(N)
    for b in range(B):
        sc = {k: inp[k][b] for k in ("g", "s", "y", "zL", "zU", "lbg", "ubg")}
        sc.update(jv=inp["jac"][b], hv=inp["hess"][b], gf=inp["grad_f"][b])
        _, r = run_host(harness, N, jsp, hsp, sc, inp["mu"][b], inp["dw_last"][b])
        assert r[0] == out["delta_w"][b] and r[1] == out["n_factor"][b] and r[2] == out["status"][b] == 0, (b, r)
    assert (out["delta_w"] > 0).sum() >= 4
    print("delta_w", out["delta_w"].tolist(), "n_factor", out["n_factor"].tolist())


def test_gpu_step_first_iteration_from_the_srb_initial_guess():
    """Drops through landing_kino_setup_batch (x0 from SRB solutions), s = g(x0) pushed inside the bounds (IPOPT's
    bound_push = bound_frac = 0.01), z = mu / distance, y = 0, mu = 0.1: status 0 and finite directions for every drop."""
    import landing_controller_b200 as lc
    N, B = 21, 32
    srb = lc.LandingSolver(N=N, device=0)
    drops = lc.grid_sweep(B)
    x_srb = srb.solve(drops)["x"]
    s = lc.LandingSolver(N=N, device=0)
    lbg, ubg, x0 = s.kino_setup_host(drops, x_srb=x_srb)
    pb = s.kino_problem(kr.DT_VAL)
    ks = s.kino_setup_data()
    g, jac = s.kino_eval_host(x0, pb)
    _, gf = s.kino_cost_host(x0, ks)
    hess = s.kino_hess_host(x0, pb, lam_f=np.ones(B), lam_g=np.zeros_like(g), ks=ks)
    eq = eq_rows(N)
    with np.errstate(invalid="ignore"):
        pL = np.minimum(0.01 * np.maximum(1.0, np.abs(lbg)), 0.01 * (ubg - lbg))
        pU = np.minimum(0.01 * np.maximum(1.0, np.abs(ubg)), 0.01 * (ubg - lbg))
        sl = np.clip(g, np.where(np.isfinite(lbg), lbg + pL, -np.inf), np.where(np.isfinite(ubg), ubg - pU, np.inf))
        zL = np.where(np.isfinite(lbg) & ~eq, 0.1 / (sl - lbg), 0.0)
        zU = np.where(np.isfinite(ubg) & ~eq, 0.1 / (ubg - sl), 0.0)
    inp = dict(g=g, jac=jac, hess=hess, grad_f=gf, s=sl, y=np.zeros_like(g), zL=zL, zU=zU, lbg=lbg, ubg=ubg,
               mu=np.full(B, 0.1), dw_last=np.zeros(B))
    out = step(s, lc, inp, "AOS", "HOST")
    assert np.all(out["status"] == 0), out["status"]
    for k in OUT:
        assert np.all(np.isfinite(out[k])), k
    vals, counts = np.unique(out["delta_w"], return_counts=True)
    print("first iteration, %d drops: delta_w distribution %s, n_factor mean %.2f" %
          (B, dict(zip(vals.tolist(), counts.tolist())), out["n_factor"].mean()))


def test_gpu_step_failures_stay_in_their_scenario():
    """A NaN in one scenario's Jacobian and a slack on its bound in another change nothing elsewhere (bit for bit).  The
    NaN is on an inequality row's entry in a control column of stage 1, so it reaches that stage's control block: the
    first reports LANDING_ST_FACTOR_FAIL after the whole inertia schedule, the second LANDING_ST_NOT_INTERIOR; both
    with NaN outputs."""
    import landing_controller_b200 as lc
    N, B = 4, 6
    s = lc.LandingSolver(N=N, device=0)
    rng = np.random.default_rng(3)
    inp = make_inputs(s, rng, N, B)
    clean = step(s, lc, inp, "SOA", "DEVICE")
    bad = {k: v.copy() for k, v in inp.items()}
    colind, row = ccs(patterns(N)[0])
    c = 12 * N + 12  # jpos_1[0], a control of stage 1
    e = next(e for e in range(colind[c], colind[c + 1]) if not eq_rows(N)[row[e]])
    bad["jac"][1, e] = np.nan
    i = np.flatnonzero(~eq_rows(N) & np.isfinite(inp["lbg"][4]))[5]
    bad["s"][4, i] = bad["lbg"][4, i]
    out = step(s, lc, bad, "SOA", "DEVICE")
    for b in (0, 2, 3, 5):
        for k in OUT + ("delta_w", "n_factor", "status", "alpha_pr", "alpha_du"):
            assert np.array_equal(out[k][b], clean[k][b]), (b, k)
    assert out["status"][4] == 5  # LANDING_ST_NOT_INTERIOR
    assert out["n_factor"][4] == 0 and np.isnan(out["delta_w"][4])
    for k in OUT:
        assert np.all(np.isnan(out[k][4])), k
    trials = dw_trials(0.0, 100)
    nf = next(i for i, d in enumerate(trials) if d > 1e40)
    assert out["status"][1] == 4  # LANDING_ST_FACTOR_FAIL
    assert out["n_factor"][1] == nf and out["delta_w"][1] == trials[nf]
    for k in OUT + ("alpha_pr", "alpha_du"):
        assert np.all(np.isnan(out[k][1])), k


def test_gpu_step_refused_arguments_and_empty_batch():
    import landing_controller_b200 as lc
    from landing_controller_b200.api import KinoStepIO, _ptr
    N, B = 3, 2
    s = lc.LandingSolver(N=N, device=0)
    rng = np.random.default_rng(4)
    inp = make_inputs(s, rng, N, B)
    d = s.kino_dims()
    outs = {k: np.zeros((B, d["nx"] if k == "dx" else d["m"])) for k in OUT}
    scal = {k: np.zeros(B) for k in ("delta_w", "alpha_pr", "alpha_du")}
    ints = {k: np.zeros(B, np.int32) for k in ("n_factor", "status")}

    def io(drop=None, tau=0.5, alpha=2):
        p = {k: _ptr(np.ascontiguousarray(inp[k])) for k in IN + ("mu", "dw_last")}
        p.update({k: _ptr(v) for k, v in outs.items()})
        if drop:
            p[drop] = None
        return KinoStepIO(*[p[k] for k in IN], p["mu"], p["dw_last"], *[p[k] for k in OUT], _ptr(scal["delta_w"]),
                          _ptr(ints["n_factor"], ctypes.POINTER(ctypes.c_int)),
                          _ptr(ints["status"], ctypes.POINTER(ctypes.c_int)), tau,
                          _ptr(scal["alpha_pr"]) if alpha >= 1 else None, _ptr(scal["alpha_du"]) if alpha >= 2 else None)
    call = lambda B_, x: s.lib.landing_kino_step_batch(s.ctx, B_, lc.HOST, lc.AOS, ctypes.byref(x))  # noqa: E731
    l0 = s.launches
    for bad in [(B, io("jac")), (B, io("mu")), (B, io("dx")), (-1, io()), (B, io(tau=1.0)), (B, io(tau=0.0)),
                (B, io(alpha=1))]:
        assert call(*bad) == 1
    assert s.lib.landing_kino_step_batch(s.ctx, B, lc.HOST, lc.AOS, None) == 1
    assert call(0, io()) == 0
    assert s.launches == l0
    assert call(B, io(tau=1.0, alpha=0)) == 0  # (tau is not read without the alpha outputs)
    assert s.launches == l0 + 1 and np.all(ints["status"] == 0)
    ref = step(s, lc, inp, "AOS", "HOST", tau=0.5)
    for k in OUT:
        assert np.array_equal(outs[k], ref[k]), k
