"""Interior-point solve of the kino-dynamic NLP on the GPU (landing_kino_solve_batch): iterates against the CPU
restatement tests/kino_ip_ref.py (written from oracle/ip_ref.c), converged points certified by the oracle, bit identity
across batches, orders, memory spaces and calls, statuses, refused arguments and the documented launch count."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import kino_ref as kr  # noqa: E402
import kino_ip_ref as ki  # noqa: E402
from test_kino_exact import kino_problem  # noqa: E402
from test_kino_step_host import patterns  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    return ki.build_harness(tmp_path_factory.mktemp("kino_solve_host"))


def solver(N):
    import landing_controller_b200 as lc
    s = lc.LandingSolver(N=N, device=0)
    return s, kino_problem(s, kr.default_problem(N))


def srb_guess(N, drops):
    import landing_controller_b200 as lc
    srb = lc.LandingSolver(N=N, device=0)
    if N == 21:
        srb.set_dt(kr.DT_VAL)
    x = srb.solve(drops)["x"]
    srb.close()
    return x


def set_opt(s, **kw):
    import landing_controller_b200 as lc
    o = lc.api.Options()
    s.lib.landing_options_default(o)
    for k, v in kw.items():
        setattr(o, k, v)
    return o


def launches_formula(stats, with_x0):
    R, S, C = (int(v) for v in stats)
    return 25 * R + 5 * S + 3 * C - 14 + (1 if with_x0 else 0)


@pytest.mark.parametrize("N", [3, 5, 21])
def test_iterates_match_the_cpu_restatement(harness, N):
    """max_iter = 1, 3, 6 from SRB-based guesses: status and iters equal the CPU restatement's, x / y / f agree to 1e-9
    relative."""
    import landing_controller_b200 as lc
    drops = lc.grid_sweep(16)[[0, 7, 13]]
    x_srb = srb_guess(N, drops)
    s, pb = solver(N)
    lbo, ubo, x0 = s.kino_setup_host(drops, x_srb=x_srb)
    jsp, hsp = patterns(N)
    P = ki.Problem(kr.default_problem(N), jsp, hsp)
    worst = 0.0
    for mi in (1, 3, 6):
        out = s.kino_solve_host(drops, x_srb=x_srb, pb=pb, options=set_opt(s, max_iter=mi))
        for b in range(len(drops)):
            r = ki.solve(harness, P, lbo[b], ubo[b], x0[b], ki.options(max_iter=mi))
            assert (out["status"][b], out["iters"][b]) == (r["status"], r["iters"]), (mi, b, out["status"][b], r)
            for a, e in ((out["x"][b], r["x"]), (out["lam_g"][b], r["y"]), (out["f"][b:b + 1], np.array([r["f"]]))):
                err = float(np.max(np.abs(a - e)) / max(1.0, float(np.max(np.abs(e)))))
                worst = max(worst, err)
                assert err <= 1e-9, (mi, b, err)
    print("N=%d worst relative difference %.2e" % (N, worst))


def test_recentring_watchdog_and_linesearch_failure_match_the_cpu_restatement(harness):
    """Parity where the re-centring path runs: the watchdog fires after every accepted step shorter than 0.9
    (jam_iters = 1), at most two re-centrings, 20 iterations, N = 3.  status, iters, restarts, x, y and f equal the CPU
    restatement's (1e-9 relative); at least one scenario re-centres."""
    import landing_controller_b200 as lc
    N = 3
    drops = lc.grid_sweep(16)[[0, 5, 10, 15]]
    s, pb = solver(N)
    lbo, ubo, x0 = s.kino_setup_host(drops)
    jsp, hsp = patterns(N)
    P = ki.Problem(kr.default_problem(N), jsp, hsp)
    kw = dict(max_iter=20, jam_iters=1, jam_alpha=0.9, max_restarts=2)
    out = s.kino_solve_host(drops, pb=pb, options=set_opt(s, **kw))
    restarted = 0
    for b in range(len(drops)):
        r = ki.solve(harness, P, lbo[b], ubo[b], x0[b], ki.options(**kw))
        got = (out["status"][b], out["iters"][b], out["restarts"][b])
        assert got == (r["status"], r["iters"], r["restarts"]), (b, got, r["status"], r["iters"], r["restarts"])
        restarted += r["restarts"] > 0
        for a, e in ((out["x"][b], r["x"]), (out["lam_g"][b], r["y"]), (out["f"][b:b + 1], np.array([r["f"]]))):
            err = float(np.max(np.abs(a - e)) / max(1.0, float(np.max(np.abs(e)))))
            assert err <= 1e-9, (b, err)
    assert restarted >= 1
    print("re-centring parity: statuses", out["status"].tolist(), "restarts", out["restarts"].tolist())


def certify(s, pb, out, lbo, ubo, N):
    ks = s.kino_setup_data()
    conv = np.flatnonzero(out["status"] == 0)
    if conv.size == 0:
        return 0
    kkt = s.kino_kkt_host(out["x"][conv], pb, ks=ks, lam_f=np.ones(conv.size), lam_g=out["lam_g"][conv],
                          lbg=lbo[conv], ubg=ubo[conv])
    worst = {}
    for i, b in enumerate(conv):
        c = ki.certificate(kr.default_problem(N), out["x"][b], out["lam_g"][b], lbo[b], ubo[b])
        assert c["viol"] <= 1e-3, (b, c["viol"])       # constr_viol_tol
        assert c["stat"] <= 1e-3, (b, c["stat"])
        assert c["compl"] <= 1e-3, (b, c["compl"])
        worst = {k: max(worst.get(k, 0.0), c[k]) for k in ("viol", "stat", "compl")}
        f_ref, _ = ki.cost(out["x"][b], N)
        assert abs(out["f"][b] - f_ref) <= 1e-12 * max(1.0, abs(f_ref))
        for k in ("viol", "dual_inf", "compl_inf"):
            assert np.array_equal(out[k][b], kkt[k][i]) or (np.isinf(out[k][b]) and np.isinf(kkt[k][i])), (k, b)
    print("certificate, worst over the converged points:", worst)
    return conv.size


def test_converged_points_are_certified_by_the_oracle():
    """Every CONVERGED scenario of a 64-drop grid and a 16-drop random sweep at N = 21: violation and scaled
    stationarity from the oracle's g and exact J, f_star against the oracle cost, and the returned measures equal to
    landing_kino_kkt_batch at (x_star, 1, lam_g)."""
    import landing_controller_b200 as lc
    N = 21
    # at least: measured 44 of 64 and 15 of 16 (DESIGN.md 3.2), with headroom
    for drops, least in ((lc.grid_sweep(64), 36), (lc.random_sweep(16, seed=5), 12)):
        x_srb = srb_guess(N, drops)
        s, pb = solver(N)
        lbo, ubo, _ = s.kino_setup_host(drops, x_srb=x_srb)
        out = s.kino_solve_host(drops, x_srb=x_srb, pb=pb)
        n = certify(s, pb, out, lbo, ubo, N)
        assert n >= least, (n, least, np.bincount(out["status"], minlength=5).tolist())
        print("%d drops: %d converged, iters mean %.1f max %d, restarts mean %.2f, statuses %s" % (
            len(drops), n, out["iters"].mean(), out["iters"].max(), out["restarts"].mean(),
            np.bincount(out["status"], minlength=5).tolist()))


def test_stored_knitro_points():
    """At the two stored drops: the solve from the SRB-based guess (reported beside the stored cost), and from the
    stored point itself with a small mu_init and bound_push, which must converge to a cost no more than 1e-8 above the
    stored one (measured: 3.2e-9 against 2.1e-11 for ms, 3.5e-9 against 3.5e-15 for gs; the costs are at the level
    tol = 1e-4 resolves, DESIGN.md 3.2)."""
    from test_kino import stored
    N = 21
    s, pb = solver(N)
    for tag in ("ms", "gs"):
        pbo, xs, _, (q0, qd0, _) = stored(tag)
        drop = np.concatenate([q0, qd0])[None, :]
        f_stored, _ = ki.cost(xs, N)
        x_srb = srb_guess(N, drop)
        out = s.kino_solve_host(drop, x_srb=x_srb, pb=pb)
        print("%s: from SRB status %d iters %d f %.6g (stored %.6g) |x - x_stored|inf %.3g" % (
            tag, out["status"][0], out["iters"][0], out["f"][0], f_stored, np.max(np.abs(out["x"][0] - xs))))
        out2 = s.kino_solve_host(drop, x0=xs[None, :], pb=pb, options=set_opt(s, mu_init=1e-4, bound_push=1e-4,
                                                                                 bound_frac=1e-4))
        print("%s: from the stored point status %d iters %d f %.6g" % (tag, out2["status"][0], out2["iters"][0],
                                                                        out2["f"][0]))
        assert out2["status"][0] == 0, (tag, out2["status"][0])
        assert out2["f"][0] <= f_stored + 1e-8, (tag, out2["f"][0], f_stored)


def test_bit_identity_batches_orders_memory_and_calls():
    """8 x SMs + 37 drops with one NaN drop: bit-identical to chunks of at most SMs, reversed and permuted, device
    buffers and a second call; the NaN drop gives LANDING_ST_NAN."""
    import torch
    import landing_controller_b200 as lc
    N = 5
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B = 8 * sms + 37
    drops = lc.random_sweep(B, seed=11)
    inan = 101
    drops[inan, 4] = np.nan
    s, pb = solver(N)
    opt = set_opt(s, max_iter=40)
    ref = s.kino_solve_host(drops, pb=pb, options=opt)
    assert ref["status"][inan] == 3
    keys = ("x", "f", "status", "iters", "lam_g", "viol", "dual_inf", "compl_inf", "restarts")

    def same(a, b, idx=None):
        for k in keys:
            va = a[k] if idx is None else a[k][idx]
            assert np.array_equal(va, b[k], equal_nan=True) if va.dtype.kind == "f" else np.array_equal(va, b[k]), k
    parts = [s.kino_solve_host(drops[i:i + sms], pb=pb, options=opt) for i in range(0, B, sms)]
    same(ref, {k: np.concatenate([p[k] for p in parts]) for k in keys})
    for perm in (np.arange(B)[::-1], np.random.default_rng(3).permutation(B)):
        o = s.kino_solve_host(drops[perm], pb=pb, options=opt)
        same({k: ref[k][perm] for k in keys}, o)
    same(ref, s.kino_solve_host(drops, pb=pb, options=opt))
    dev = torch.device("cuda:0")
    d = s.kino_dims()
    t = dict(x=torch.zeros(B, d["nx"], dtype=torch.float64, device=dev), f=torch.zeros(B, dtype=torch.float64, device=dev),
             status=torch.zeros(B, dtype=torch.int32, device=dev), iters=torch.zeros(B, dtype=torch.int32, device=dev),
             lam_g=torch.zeros(B, d["m"], dtype=torch.float64, device=dev),
             restarts=torch.zeros(B, dtype=torch.int32, device=dev))
    for k in ("viol", "dual_inf", "compl_inf"):
        t[k] = torch.zeros(B, dtype=torch.float64, device=dev)
    dT = torch.tensor(drops, device=dev)
    torch.cuda.synchronize()
    s.kino_solve_device(dT, t["x"], t["f"], t["status"], t["iters"], lam_g=t["lam_g"], viol=t["viol"],
                        dual_inf=t["dual_inf"], compl_inf=t["compl_inf"], restarts=t["restarts"], pb=pb, options=opt)
    s.synchronize()
    same(ref, {k: v.cpu().numpy() for k, v in t.items()})
    print("B=%d statuses %s" % (B, np.bincount(ref["status"], minlength=5).tolist()))


def test_statuses_arguments_and_launches():
    import landing_controller_b200 as lc
    import ctypes
    N = 4
    drops = lc.grid_sweep(16)
    s, pb = solver(N)
    # MAX_ITER
    out = s.kino_solve_host(drops, pb=pb, options=set_opt(s, max_iter=2))
    assert np.all((out["status"] == 1) | (out["status"] == 0) | (out["status"] == 4)), out["status"]
    assert np.all(out["iters"][out["status"] == 1] == 2)
    # launch count = the documented formula, with and without x0
    for x0 in (None, s.kino_setup_host(drops, want_bounds=False)[2]):
        l0 = s.launches
        out = s.kino_solve_host(drops, x0=x0, pb=pb, options=set_opt(s, max_iter=30))
        assert s.launches - l0 == launches_formula(out["stats"], x0 is not None), (s.launches - l0, out["stats"])
    # the watchdog off through max_restarts = 0 changes only the scenarios that re-centre
    a = s.kino_solve_host(drops, pb=pb, options=set_opt(s, max_iter=60))
    b = s.kino_solve_host(drops, pb=pb, options=set_opt(s, max_iter=60, max_restarts=0))
    same = a["restarts"] == 0
    assert np.array_equal(a["x"][same], b["x"][same]) and np.array_equal(a["iters"][same], b["iters"][same])
    assert np.all(b["restarts"] == 0)
    # optional outputs may be NULL
    c = s.kino_solve_host(drops, pb=pb, options=set_opt(s, max_iter=60), want=())
    assert np.array_equal(c["x"], a["x"]) and np.array_equal(c["status"], a["status"])
    # B = 0 launches nothing
    l0 = s.launches
    e = s.kino_solve_host(np.zeros((0, 12)), pb=pb)
    assert s.launches == l0 and list(e["stats"]) == [0, 0, 0]
    # refused arguments leave the context usable
    ks = s.kino_setup_data()
    io = lc.api.KinoSolveIO()
    opt = set_opt(s)
    assert s.lib.landing_kino_solve_batch(s.ctx, 1, lc.HOST, ctypes.byref(pb), ctypes.byref(ks), ctypes.byref(opt),
                                          ctypes.byref(io)) == 1
    assert s.lib.landing_kino_solve_batch(s.ctx, 1, lc.HOST, ctypes.byref(pb), None, ctypes.byref(opt),
                                          ctypes.byref(io)) == 1
    for bad in (dict(max_iter=-1), dict(tol=0.0), dict(mu_init=-1.0), dict(bound_frac=0.7), dict(max_restarts=-2)):
        with pytest.raises(RuntimeError):
            s.kino_solve_host(drops[:2], pb=pb, options=set_opt(s, **bad))
    assert s.lib.landing_kino_solve_batch(s.ctx, -1, lc.HOST, ctypes.byref(pb), ctypes.byref(ks), ctypes.byref(opt),
                                          ctypes.byref(io)) == 1
    again = s.kino_solve_host(drops, pb=pb, options=set_opt(s, max_iter=60))
    assert np.array_equal(again["x"], a["x"])
