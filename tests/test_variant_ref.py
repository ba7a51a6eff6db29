"""CPU tests of the restatement of the fixed-schedule and CCC problems (tests/variant_ref.py): its own derivatives, its
reduction to the oracle, the product's SCHED knot template compiled for the host against it, and the CPU
interior-point solutions (oracle/ip_ref.c) certified as KKT points of it."""
import ctypes
import os

import numpy as np
import pytest

import ccc_problem as ccc
import landing_controller_b200 as lc
import variant_ref as vr
from oracle_ip import default_options, default_problem, solve_cpu
from oracle_lib import _dp

# tolerances of test_gpu_solve.py::_kkt_certificate: constr_viol_tol (+ bound_relax_factor), dual infeasibility with
# s_d <= 100, complementarity
VIOL, STAT, COMP = 1e-3 + 2e-6, 1e-2, 2e-3


def _random_point(N, seed):
    """a random (x, p, cs) with a non-uniform dt, a perturbed Xref and both contact states on every leg"""
    rng = np.random.default_rng(seed)
    o = vr.oracle(N)
    pb = lc.apply_schedule_parameters(default_problem())
    p, x0 = o.build_p_x0(pb, lc.single_drop()[0, :6], lc.single_drop()[0, 6:])
    p[o.off["o_dt"]:o.off["o_dt"] + N - 1] = rng.uniform(0.01, 0.05, N - 1)
    p[:12 * N] += 0.1 * rng.normal(size=12 * N)
    x = x0 + 0.2 * rng.normal(size=o.nx)
    cs = rng.integers(0, 2, size=(N - 1, 4)).astype(np.int32)
    cs[0], cs[-1] = 0, 1
    return x, p, cs


@pytest.mark.parametrize("N", [5, 16, 30])
def test_cost_gradient_and_replaced_rows_against_central_differences(N):
    x, p, cs = _random_point(N, N)
    QX = np.linspace(1.0, 12.0, 12)
    v = vr.VariantNLP(N, p, cs, Qf=(1e-2, 2e-2, 3e-2), QX=QX, kin_box=lc.SCHED_KIN_BOX)
    f, gf = v.cost(x)
    J = v.jac(x)
    replaced = np.array([r for r, *_ in v._replaced_rows()])
    eps = 1e-6
    for c in range(v.o.nx):
        xp, xm = x.copy(), x.copy()
        xp[c] += eps
        xm[c] -= eps
        d = (v.cost(xp)[0] - v.cost(xm)[0]) / (2 * eps)
        assert abs(d - gf[c]) <= 1e-6 * max(1.0, abs(gf[c])), c
        dg = (v.g(xp) - v.g(xm)) / (2 * eps)
        assert np.max(np.abs(dg[replaced] - J[replaced, c])) <= 1e-9, c  # linear rows: exact up to rounding
        assert np.max(np.abs(dg - J[:, c])) <= 1e-6, c


def test_reduces_to_the_oracle_outside_the_replaced_rows():
    """cs = 1 everywhere, Qf = QX = 0, default box: cost, gradient, rows, Jacobian and bounds are the oracle's bit for
    bit except on the rows formulation 1 restates; formulation 0 with the default box is the oracle everywhere."""
    N = 16
    x, p, _ = _random_point(N, 3)
    o = vr.oracle(N)
    _, f0, gf0 = o.grad_f(x, p)
    _, g0 = o.g(x, p)
    lb0, ub0 = o.bounds(p)
    J0 = vr.VariantNLP(N, p).jac(x)
    v0 = vr.VariantNLP(N, p)
    assert np.array_equal(v0.g(x), g0) and np.array_equal(v0.lb, lb0) and np.array_equal(v0.ub, ub0)
    assert (v0.kind != vr.FREE).all()
    v = vr.VariantNLP(N, p, np.ones((N - 1, 4)))
    f, gf = v.cost(x)
    assert f == f0 and np.array_equal(gf, gf0)
    rep = np.zeros(o.m, dtype=bool)
    rep[[r for r, *_ in v._replaced_rows()]] = True
    J = v.jac(x)
    assert np.array_equal(v.g(x)[~rep], g0[~rep]) and np.array_equal(J[~rep], J0[~rep])
    assert np.array_equal(v.lb[~rep], lb0[~rep]) and np.array_equal(v.ub[~rep], ub0[~rep])
    # the restated rows: 24 free terminal rows, per knot and leg one free and (but the last knot) three free rows,
    # and cs c_z = 0, cs (c+ - c) = 0 as equalities
    assert (v.kind[12:36] == vr.FREE).all()
    assert np.sum(rep & (v.kind == vr.FREE)) == 24 + 4 * (N - 1) + 12 * (N - 2)
    assert np.sum(rep & (v.kind == vr.EQ)) == 4 * (N - 1) + 12 * (N - 2)
    k, l = 3, 2
    L = vr.leg_row(N, k, l)
    assert np.flatnonzero(J[L]).tolist() == [vr.c_var(N, k, 3 * l + 2)]
    assert J[L + 3, vr.c_var(N, k, 3 * l + 1)] == -1.0 and J[L + 3, vr.c_var(N, k + 1, 3 * l + 1)] == 1.0
    assert np.count_nonzero(J[L + 3]) == 2


def test_bounds_of_the_schedule_and_the_kinematic_box():
    N = 6
    x, p, cs = _random_point(N, 1)
    v = vr.VariantNLP(N, p, cs, kin_box=(0.05, 0.04, 0.27))
    f_max = p[v.o.off["o_fmax"]]
    for k in range(N - 1):
        for l in range(4):
            fz = 36 + 104 * k + 12 + l
            assert (v.lb[fz], v.ub[fz]) == (0.0, cs[k, l] * f_max)
            K = vr.kin_row(N, k, l)
            assert v.lb[K:K + 3].tolist() == [-0.05, -0.04, -0.27] and v.ub[K:K + 3].tolist() == [0.05, 0.04, 0.0]
            L = vr.leg_row(N, k, l)
            assert v.kind[L] == (vr.EQ if cs[k, l] else vr.FREE) and v.kind[L + 1] == vr.FREE
            if k < N - 2:
                assert (v.kind[L + 2:L + 5] == (vr.EQ if cs[k, l] else vr.FREE)).all()
                assert (v.kind[L + 5:L + 8] == vr.FREE).all()


# ---------------------------------------------------------------- the SCHED knot template compiled for the host
@pytest.mark.parametrize("N", [5, 16, 30])
def test_sched_knot_template_on_host_matches_the_restatement(N):
    """knot_eval<..., SCHED = true> against the restatement: every g entry and every Jacobian entry of the knot rows at
    1e-13 relative; the Hessian equals the oracle's with the multipliers of the restated rows zeroed (those rows are
    linear or absent)."""
    from test_oracle_eval import _host_harness
    h = _host_harness()
    o = vr.oracle(N)
    colind, row = o.spJ[2:2 + o.nx + 1], o.spJ[2 + o.nx + 1:]
    col = np.repeat(np.arange(o.nx), np.diff(colind))
    knot = row >= 36
    in_pattern = np.zeros((o.m, o.nx), dtype=bool)
    in_pattern[row, col] = True
    for seed in range(5):
        x, p, cs = _random_point(N, 100 * N + seed)
        lam = np.random.default_rng(seed).normal(size=o.m)
        v = vr.VariantNLP(N, p, cs)
        g, J, H = np.zeros(o.m), np.zeros(o.nnzJ), np.zeros(o.nnzH)
        csi = np.ascontiguousarray(cs, dtype=np.int32)
        h.hostcheck_eval_sched(N, _dp(x), _dp(p), ctypes.c_double(0.3), _dp(lam),
                               csi.ctypes.data_as(ctypes.POINTER(ctypes.c_int)), _dp(g), _dp(J), _dp(H))
        gr, Jr = v.g(x), v.jac(x)
        assert np.max(np.abs(g[36:] - gr[36:]) / np.maximum(1.0, np.abs(gr[36:]))) <= 1e-13
        Jv = Jr[row, col]
        assert np.max(np.abs(J[knot] - Jv[knot]) / np.maximum(1.0, np.abs(Jv[knot]))) <= 1e-13
        assert not Jr[~in_pattern].any()  # every non-zero of the restated rows has a place in the CCS pattern
        lam0 = lam.copy()
        lam0[[r for r, *_ in v._replaced_rows() if r >= 36]] = 0.0
        _, H0 = o.hess_l(x, p, 0.3, lam0)
        assert np.max(np.abs(H - H0) / np.maximum(1.0, np.abs(H0))) <= 1e-13


# ---------------------------------------------------------------- CPU interior-point solutions certified
def sched_problem(N, T, cs, dt=None, z_max=1.0):
    """(oracle problem, ip options) of formulation 1 with the parameter set of quadruped_SRBM_NLP.m"""
    pb = lc.apply_schedule_parameters(default_problem(), z_max=z_max)
    pb.T = T
    if dt is not None:
        pb.set_dt(dt)
    opt = default_options(run_Qf=lc.SCHED_QF, kin_box=lc.SCHED_KIN_BOX).set_schedule(cs, lc.SCHED_QX)
    return pb, opt


def sched_cases():
    """name -> (N, T, cs, dt, z_max, drops) of the formulation-1 problems the certificates cover"""
    ref = np.zeros((1, 12))
    ref[0, 2], ref[0, 11] = 0.35, -1.0        # quadruped_SRBM_NLP.m:29-33
    cfg0 = np.repeat(lc.single_drop(), 4, axis=0)  # BASELINE configs[0] and three variants of it
    cfg0[1, 9] = 0.0; cfg0[2, 4] = 0.15; cfg0[3, 10] = 0.4; cfg0[3, 3] = -0.1
    dt = vr.alternating_dt(30, 0.6)
    return {"reference16": (16, 0.5, lc.reference_schedule(16), None, 0.4, ref),
            "config0": (30, 0.6, lc.ballistic_schedule(30, 0.6, 0.5), None, 1.0, cfg0),
            "alternating_dt": (30, 0.6, vr.ballistic_schedule_dt(dt, 0.5), dt, 1.0, cfg0[:2]),
            "n50": (50, 0.6, lc.ballistic_schedule(50, 0.6, 0.5), None, 1.0, cfg0[:2])}


def certify(v, x, lam, f_ret, viol_ret):
    """asserts the certificate of one converged point and returns (stat, max |lam|)"""
    f, viol, stat, comp, free = v.kkt(x, lam)
    assert viol <= VIOL and stat <= STAT and comp <= COMP, (viol, stat, comp)
    assert free == 0.0
    assert abs(f - f_ret) <= 1e-12 * max(1.0, abs(f))
    assert abs(max(viol, 0.0) - viol_ret) <= 1e-9
    return stat, float(np.max(np.abs(lam)))


@pytest.mark.parametrize("case", ["reference16", "config0", "alternating_dt", "n50"])
def test_cpu_fixed_schedule_solutions_are_kkt_points_of_the_restatement(case):
    N, T, cs, dt, z_max, drops = sched_cases()[case]
    pb, opt = sched_problem(N, T, cs, dt, z_max)
    r = solve_cpu(N, drops, opt, pb, want_lam=True)
    assert (r["status"] == 0).all()
    out = []
    for b in range(len(drops)):
        v = vr.from_drop(N, pb, drops[b], cs=cs, Qf=lc.SCHED_QF, QX=lc.SCHED_QX, kin_box=lc.SCHED_KIN_BOX)
        out.append(certify(v, r["x"][b], r["lam_g"][b], r["f"][b], r["viol"][b]))
    print("%s: max stationarity %.1e, max |lam| %.1e" % (case, max(s for s, _ in out), max(m for _, m in out)))


def test_cpu_ccc_solutions_are_kkt_points_of_the_restatement():
    d = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ccc_n41.npz"))
    drops = np.ascontiguousarray(d["X"][:, :, 0])
    pb = ccc.fill_problem(default_problem())
    r = solve_cpu(ccc.N, drops, default_options(run_Qf=list(ccc.QF), kin_box=list(ccc.KIN_BOX)), pb, want_lam=True)
    assert (r["status"] == 0).mean() >= 0.9
    out = [certify(vr.from_drop(ccc.N, pb, drops[b], Qf=ccc.QF, kin_box=ccc.KIN_BOX), r["x"][b], r["lam_g"][b],
                   r["f"][b], r["viol"][b]) for b in np.flatnonzero(r["status"] == 0)]
    print("CCC: %d of %d converged, max stationarity %.1e, max |lam| %.1e"
          % (len(out), len(drops), max(s for s, _ in out), max(m for _, m in out)))


def test_solve_cpu_with_multipliers_takes_the_same_path_as_the_batch():
    N, T, cs, dt, z_max, drops = sched_cases()["alternating_dt"]
    pb, opt = sched_problem(N, T, cs, dt, z_max)
    opt.max_iter = 6
    a = solve_cpu(N, drops, opt, pb)
    b = solve_cpu(N, drops, opt, pb, want_lam=True)
    assert np.array_equal(a["x"], b["x"]) and np.array_equal(a["iters"], b["iters"]) and np.array_equal(a["f"], b["f"])
