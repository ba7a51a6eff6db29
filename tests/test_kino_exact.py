"""Kino-dynamic NLP on the GPU against exact references: g against the oracle on every scenario, and EVERY CCS entry of
the Jacobian against the complex-step Jacobian of the oracle (oracle/kino_ref.py:jac_exact) on sampled scenarios, at
non-default parameters and knot spacings, over knot counts, ragged batches, both layouts and both memory spaces; that
every output entry is written on every call; and the bounds, initial guess and cost at a randomised landing_kino_setup."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import kino_ref as kr  # noqa: E402

pytestmark = pytest.mark.gpu


def random_problem(rng, N):
    """Oracle problem with random mu, mass, Ib, an Ib_inv deliberately not 1 / Ib, and a random spacing per knot."""
    pb = kr.default_problem(N)
    pb.update(mu=rng.uniform(0.3, 1.2), mass=rng.uniform(5.0, 12.0), Ib=rng.uniform(0.03, 0.4, 3),
              Ib_inv=rng.uniform(2.0, 25.0, 3), dt=rng.uniform(0.005, 0.1, N - 1))
    return pb


def random_x(rng, N, B):
    """x = [X; jpos; U] at landing magnitudes: body within 0.5 m, angles within 1 rad, rates within 3, feet near the body,
    forces up to 300 N."""
    X = rng.uniform(-0.5, 0.5, (B, N, 12))
    X[..., 3:6] = rng.uniform(-1, 1, (B, N, 3))
    X[..., 6:12] = rng.uniform(-3, 3, (B, N, 6))
    J = rng.uniform(-1, 1, (B, N - 1, 12))
    U = rng.uniform(-0.5, 0.5, (B, N - 1, 24))
    U[..., 12:] = rng.uniform(-100, 100, (B, N - 1, 12))
    U[..., 14::3] = rng.uniform(0, 300, (B, N - 1, 4))
    return np.concatenate([X.reshape(B, -1), J.reshape(B, -1), U.reshape(B, -1)], axis=1)


def sample(rng, B):
    """b = 0, the last scenario, 127 and 128 (either side of a 128-thread CTA) where B allows, and four random ones."""
    fixed = {0, B - 1} | {b for b in (127, 128) if b < B}
    return sorted(fixed | set(rng.choice(B, size=min(4, B), replace=False).tolist()))


def kino_problem(s, pbo):
    return s.kino_problem(pbo["dt"], mu=pbo["mu"], mass=pbo["mass"], Ib=pbo["Ib"], Ib_inv=pbo["Ib_inv"])


def evaluate(s, lc, x, pb, layout, memspace):
    """g [B, m] and jac [B, nnz] (AoS numpy) from a call in the given layout and memory space.  Device outputs are
    pre-filled with NaN, so an entry that no kernel writes shows."""
    d = s.kino_dims()
    xin = x if layout == lc.AOS else np.ascontiguousarray(x.T)
    if memspace == lc.HOST:
        g, jac = s.kino_eval_host(xin, pb, layout=layout)
    else:
        import torch
        dev = torch.device("cuda:0")
        B = x.shape[0]
        shp = (lambda n: (B, n)) if layout == lc.AOS else (lambda n: (n, B))
        xt = torch.tensor(xin, device=dev)
        gt = torch.full(shp(d["m"]), float("nan"), dtype=torch.float64, device=dev)
        jt = torch.full(shp(d["nnzJ"]), float("nan"), dtype=torch.float64, device=dev)
        s.kino_eval_device(xt, pb, g=gt, jac=jt, layout=layout)
        s.synchronize()
        g, jac = gt.cpu().numpy(), jt.cpu().numpy()
        assert not np.isnan(g).any() and not np.isnan(jac).any(), "an output entry was not written"
    if layout == lc.SOA:
        g, jac = np.ascontiguousarray(g.T), np.ascontiguousarray(jac.T)
    return g, jac


def check_against_exact(s, pbo, x, g, jac, bs):
    """g of every scenario against the oracle, every CCS entry of the scenarios bs against the exact Jacobian;
    returns the worst relative errors."""
    wg = 0.0
    for b in range(x.shape[0]):
        go = kr.eval_g(pbo, x[b], literal=False)
        e = np.max(np.abs(g[b] - go) / np.maximum(1.0, np.abs(go)))
        assert e <= 1e-12, (b, e)
        wg = max(wg, e)
    pattern = s.kino_sparsity()
    wj = 0.0
    for b in bs:
        Je = kr.jac_exact(pbo, x[b], pattern)
        e = np.abs(jac[b] - Je) / np.maximum(1.0, np.abs(Je))
        assert e.max() <= 1e-12, (b, e.max(), int(e.argmax()))
        wj = max(wj, e.max())
    return wg, wj


# (N, B, layout, memory space): every N, B in {1, 63, 64, 129, 257} (direct AoS below 64, the transposed AoS path from
# 64, partial CTAs of 128 threads), both layouts, host and device buffers
CASES = [(3, 1, "AOS", "HOST"), (3, 257, "SOA", "DEVICE"), (4, 63, "AOS", "HOST"), (4, 129, "AOS", "DEVICE"),
         (21, 64, "AOS", "HOST"), (21, 257, "SOA", "HOST"), (21, 1, "SOA", "DEVICE"), (30, 129, "SOA", "HOST"),
         (30, 64, "AOS", "DEVICE")]


@pytest.mark.parametrize("N,B,layout,memspace", CASES)
def test_gpu_kino_eval_matches_the_exact_jacobian(N, B, layout, memspace):
    import landing_controller_b200 as lc
    rng = np.random.default_rng(1000 * N + B)
    s = lc.LandingSolver(N=N, device=0)
    pbo = random_problem(rng, N)
    x = random_x(rng, N, B)
    g, jac = evaluate(s, lc, x, kino_problem(s, pbo), getattr(lc, layout), getattr(lc, memspace))
    wg, wj = check_against_exact(s, pbo, x, g, jac, sample(rng, B))
    print("kino N=%d B=%d %s %s: worst rel. error g %.2e, jac %.2e" % (N, B, layout, memspace, wg, wj))
    s.close()


def test_gpu_kino_eval_second_call_sees_new_inputs_and_parameters():
    """One context, host buffers, the transposed AoS path: (x1, pb1) and then (x2, pb2) with a different dt and different
    parameters; the second result must be that of (x2, pb2) (no stale staging, no cached parameters or spacings)."""
    import landing_controller_b200 as lc
    N, B = 21, 129
    rng = np.random.default_rng(5)
    s = lc.LandingSolver(N=N, device=0)
    p1, p2 = random_problem(rng, N), random_problem(rng, N)
    x1, x2 = random_x(rng, N, B), random_x(rng, N, B)
    g1, j1 = s.kino_eval_host(x1, kino_problem(s, p1))
    g2, j2 = s.kino_eval_host(x2, kino_problem(s, p2))
    check_against_exact(s, p1, x1, g1, j1, [0])
    wg, wj = check_against_exact(s, p2, x2, g2, j2, [0, 77, B - 1])
    print("kino second call: worst rel. error g %.2e, jac %.2e" % (wg, wj))
    s.close()


def test_gpu_kino_problems_keep_their_own_knot_spacings():
    """Two KinoProblem built from temporaries (lists), both alive, then both evaluated: each call reads the spacings of
    its own problem, also after the memory of a released temporary has been reused."""
    import landing_controller_b200 as lc
    N, B = 4, 3
    rng = np.random.default_rng(9)
    s = lc.LandingSolver(N=N, device=0)
    p1, p2 = random_problem(rng, N), random_problem(rng, N)
    pb1 = s.kino_problem(list(p1["dt"]), mu=p1["mu"], mass=p1["mass"], Ib=list(p1["Ib"]), Ib_inv=list(p1["Ib_inv"]))
    pb2 = s.kino_problem(list(p2["dt"]), mu=p2["mu"], mass=p2["mass"], Ib=list(p2["Ib"]), Ib_inv=list(p2["Ib_inv"]))
    junk = [np.full(N - 1, -1.0) for _ in range(8)]  # takes the blocks of any array released above
    assert np.array_equal(np.ctypeslib.as_array(pb1.dt, shape=(N - 1,)), p1["dt"])
    x = random_x(rng, N, B)
    for pb, po in ((pb1, p1), (pb2, p2), (pb1, p1)):
        g, jac = s.kino_eval_host(x, pb)
        check_against_exact(s, po, x, g, jac, [1])
    del junk
    s.close()


def random_setup(rng, s):
    """Every field of landing_kino_setup randomised."""
    ks = s.kino_setup_data()
    u = rng.uniform
    fields = {"q_term_min": u(-1, 0.1, 6), "qd_term_min": u(-2, -0.1, 6), "z_min": u(0.02, 0.2),
              "l_leg_max": u(0.3, 0.5), "jpos_min": u(-2, -0.1, 12), "jpos_max": u(0.1, 2.5, 12), "tau_max": u(10, 40, 3),
              "QN": u(0, 100, 12), "q_term_ref": u(-0.5, 0.5, 6), "qd_term_ref": u(-0.5, 0.5, 6), "jpos_guess": u(-1, 1, 3)}
    fields["q_term_max"] = fields["q_term_min"] + u(0.1, 2, 6)
    fields["qd_term_max"] = fields["qd_term_min"] + u(0.1, 2, 6)
    for k, v in fields.items():
        if np.ndim(v):
            for i, vi in enumerate(v):
                getattr(ks, k)[i] = vi
        else:
            setattr(ks, k, v)
    return ks, fields


@pytest.mark.parametrize("N,with_srb", [(3, True), (21, False), (21, True), (30, False)])
def test_gpu_kino_setup_and_cost_follow_a_random_setup(N, with_srb):
    import landing_controller_b200 as lc
    B = 67
    rng = np.random.default_rng(N + 100 * with_srb)
    s = lc.LandingSolver(N=N, device=0)
    d = s.kino_dims()
    ks, fs = random_setup(rng, s)
    drops = lc.random_sweep(B, seed=N)
    x_srb = rng.normal(size=(B, 36 * N - 24)) if with_srb else None
    lb, ub, x0 = s.kino_setup_host(drops, x_srb=x_srb, ks=ks)
    ss = np.array([[1, -1, 1], [1, 1, 1], [-1, -1, 1], [-1, 1, 1.0]])
    qref = np.concatenate([fs["q_term_ref"], fs["qd_term_ref"]])
    for b in range(B):
        pbo = kr.default_problem(N)
        pbo.update({k: fs[k] for k in ("q_term_min", "q_term_max", "qd_term_min", "qd_term_max", "z_min", "l_leg_max",
                                       "jpos_min", "jpos_max", "tau_max")})
        R = kr.rpy_to_rot_xyz(drops[b, 3:6])
        vb = R.T @ drops[b, 9:12]
        pbo["kin_box"] = np.array([kr.kin_box_limits(vb[0], "x"), kr.kin_box_limits(vb[1], "y")])
        c_init = np.concatenate([drops[b, :3] + R @ (ss[l] * np.array([0.2, 0.15, -0.3])) for l in range(4)])
        lo, uo = kr.bounds(pbo, drops[b, :6], drops[b, 6:], c_init)
        fl, fu = np.isfinite(lo), np.isfinite(uo)
        assert np.array_equal(fl, np.isfinite(lb[b])) and np.array_equal(fu, np.isfinite(ub[b]))
        assert np.array_equal(lb[b][~fl], lo[~fl]) and np.array_equal(ub[b][~fu], uo[~fu])  # the same infinities
        assert np.max(np.abs(lb[b][fl] - lo[fl])) <= 1e-15 and np.max(np.abs(ub[b][fu] - uo[fu])) <= 1e-15
        # initial guess: jpos_guess on every knot, X / U from the SRB solution or the reference trajectories
        X, J, U = kr.split(x0[b], N)
        assert np.array_equal(J, np.tile(fs["jpos_guess"], (N - 1, 4)))
        if with_srb:
            assert np.array_equal(X.ravel(), x_srb[b, :12 * N]) and np.array_equal(U.ravel(), x_srb[b, 12 * N:])
        else:
            t = np.arange(N)[:, None] / (N - 1)
            assert np.allclose(X, drops[b] + (qref - drops[b]) * t, rtol=0, atol=1e-14)
            for k in range(N - 1):
                Rk = kr.rpy_to_rot_xyz(X[k, 3:6])
                cref = np.concatenate([X[k, :3] + Rk @ (ss[l] * np.array([0.2, 0.2, -0.3])) for l in range(4)])
                assert np.allclose(U[k, :12], cref, rtol=0, atol=1e-14) and np.all(U[k, 12:] == 0)
    # terminal cost and its gradient: QN and the terminal references of the setup
    xx = rng.normal(size=(B, d["nx"]))
    f, gf = s.kino_cost_host(xx, ks=ks)
    e = xx[:, 12 * (N - 1):12 * N] - qref
    assert np.allclose(f, (fs["QN"] * e * e).sum(1), rtol=1e-14, atol=0)
    go = np.zeros_like(xx)
    go[:, 12 * (N - 1):12 * N] = 2 * fs["QN"] * e
    assert np.allclose(gf, go, rtol=1e-14, atol=0)
    s.close()
