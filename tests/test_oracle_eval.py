"""CPU tests: the oracle (oracle/srb_ref.c) against the reference's golden vectors, and the
product's knot template compiled for the host against the oracle."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle_lib import CasadiLib, Oracle, REF_SO, _dp, c_llp, have_ref

TOL = 1e-10  # north_star: function, Jacobian and Hessian values within 1e-10 relative


def rel(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b)) / np.maximum(1.0, np.abs(b))))


@pytest.fixture(scope="module")
def o21():
    return Oracle(21)


def test_sizes_match_reference(o21):
    assert (o21.nx, o21.np_, o21.m, o21.nnzJ, o21.nnzH) == (732, 354, 2092, 7664, 3780)
    for N, dims in ((30, (1056, 471, 3028, 11129, 5481)), (50, (1776, 731, 5108, 18829, 9261))):
        o = Oracle(N)
        assert (o.nx, o.np_, o.m, o.nnzJ, o.nnzH) == dims


def test_sparsity_integer_equal_to_reference(o21, golden):
    # casadi_s5 / casadi_s4 of landingCtrller_IPOPT.c:63-64
    assert np.array_equal(o21.spJ, golden["spJ"])
    assert np.array_equal(o21.spH, golden["spH"])


def test_parameter_offsets(o21):
    # SURVEY 8a, verified against the generated C
    exp = dict(o_dt=252, o_qmin=272, o_qmax=278, o_qdmin=284, o_qdmax=290, o_qinit=296, o_qdinit=302,
               o_qtmin=308, o_qtmax=314, o_qdtmin=320, o_qdtmax=326, o_QN=332, o_mu=344, o_lleg=345,
               o_fmax=346, o_mass=347, o_Ib=348, o_Ibinv=351)
    assert o21.off == exp


def test_golden_vectors(o21, golden):
    for i in range(int(golden["n_cases"])):
        c = {k: golden["c%d_%s" % (i, k)] for k in ("x", "p", "lam_f", "lam_g", "f", "g", "J", "H", "gf", "gx", "gp")}
        lf = float(c["lam_f"][0])
        _, f = o21.f(c["x"], c["p"])
        _, g, J = o21.jac_g(c["x"], c["p"])
        _, H = o21.hess_l(c["x"], c["p"], lf, c["lam_g"])
        _, f2, gf = o21.grad_f(c["x"], c["p"])
        _, f3, g3, gx, gp = o21.grad(c["x"], c["p"], lf, c["lam_g"])
        assert rel([f], c["f"]) < TOL and rel([f2], c["f"]) < TOL
        assert rel(g, c["g"]) < TOL and rel(g3, c["g"]) < TOL
        assert rel(J, c["J"]) < TOL
        assert rel(H, c["H"]) < TOL
        assert rel(gf, c["gf"]) < TOL
        assert rel(gx, c["gx"]) < TOL
        assert rel(gp, c["gp"]) < TOL


def test_kat0_from_survey(o21, golden):
    # SURVEY.md appendix B.3 (values printed from the compiled reference C)
    x, p = golden["c0_x"], golden["c0_p"]
    _, g, J = o21.jac_g(x, p)
    _, H = o21.hess_l(x, p, 1.0, np.ones(o21.m))
    exp = [0, 0, -0.5, 0, 0, 0, -0.00363548230731944, -0.00181774115365972, 0.2870290353853611, -0.0522, 0.02562, 0]
    assert np.allclose(g[36:48], exp, rtol=0, atol=1e-14)
    assert np.allclose(g[100:116], [-0.42, 0, 0, 0, -2.42, 0, 0, 0, -0.92, 0, 0, 0, -1.92, 0, 0, 0], atol=1e-14)
    assert abs(J.sum() - 446.8217242462433) < 1e-9 and abs(np.abs(J).sum() - 2374.3204157537566) < 1e-9
    assert abs(H.sum() - 560.1979584000001) < 1e-9 and abs(np.abs(H).sum() - 2607.579796) < 1e-9


@pytest.mark.skipif(not have_ref(), reason="compiled reference C not present (oracle/_ref, built by `make -C oracle ref` "
                                           "from the reference's own landingCtrller_IPOPT.c)")
def test_live_reference_random(o21):
    ref = CasadiLib(REF_SO)
    rng = np.random.default_rng(7)
    worst = 0.0
    for _ in range(300):
        x = rng.normal(size=o21.nx) * rng.choice([0.05, 0.3, 0.8])
        p = rng.uniform(0.5, 1.5, size=o21.np_)
        lam = rng.normal(size=o21.m)
        lf = np.array([rng.normal()])
        _, (g_r, J_r) = ref.call("nlp_jac_g", [x, p])
        _, (H_r,) = ref.call("nlp_hess_l", [x, p, lf, lam])
        _, g, J = o21.jac_g(x, p)
        _, H = o21.hess_l(x, p, float(lf[0]), lam)
        worst = max(worst, rel(g, g_r), rel(J, J_r), rel(H, H_r))
    assert worst < TOL


@pytest.mark.parametrize("N", [5, 30])
def test_generic_n_finite_differences(N):
    """No reference C exists for N != 21: derivative self-consistency by central differences."""
    o = Oracle(N)
    rng = np.random.default_rng(N)
    x = rng.normal(size=o.nx) * 0.3
    p = rng.uniform(0.5, 1.5, size=o.np_)
    lam = rng.normal(size=o.m)
    _, g, J = o.jac_g(x, p)
    _, H = o.hess_l(x, p, 0.7, lam)
    colind, row = o.spJ[2:2 + o.nx + 1], o.spJ[2 + o.nx + 1:]
    hcol, hrow = o.spH[2:2 + o.nx + 1], o.spH[2 + o.nx + 1:]
    Jd = np.zeros((o.m, o.nx))
    Hd = np.zeros((o.nx, o.nx))
    for c in range(o.nx):
        Jd[row[colind[c]:colind[c + 1]], c] = J[colind[c]:colind[c + 1]]
        Hd[hrow[hcol[c]:hcol[c + 1]], c] = H[hcol[c]:hcol[c + 1]]
    Hd = Hd + np.triu(Hd, 1).T
    eps = 1e-6
    for c in rng.choice(o.nx, size=40, replace=False):
        xp, xm = x.copy(), x.copy()
        xp[c] += eps
        xm[c] -= eps
        _, gp_ = o.g(xp, p)
        _, gm_ = o.g(xm, p)
        assert np.max(np.abs((gp_ - gm_) / (2 * eps) - Jd[:, c])) < 1e-6
        _, _, _, gxp, _ = o.grad(xp, p, 0.7, lam)
        _, _, _, gxm, _ = o.grad(xm, p, 0.7, lam)
        assert np.max(np.abs((gxp - gxm) / (2 * eps) - Hd[:, c])) < 1e-5


def test_bounds_and_initial_guess(o21):
    pb = o21.default_problem()
    q0 = np.array([0, 0, 0.6, 0, np.pi / 4, -np.pi / 6])
    qd0 = np.array([0, 4, 5, 1.3, -2, -2.0])
    p, x0 = o21.build_p_x0(pb, q0, qd0)
    lb, ub = o21.bounds(p)
    assert np.array_equal(lb[:6], q0) and np.array_equal(ub[6:12], qd0)
    assert np.all(lb[36:48] == 0) and np.all(ub[36:48] == 0)
    # counts of the bound constants decoded from the reference's .casadi (SURVEY 8a): 0.001 x80 rows ...
    assert np.sum(ub == 0.001) == 4 * 20 and np.sum(ub == 0.01) == 12 * 19 and np.sum(lb == -0.01) == 12 * 19
    assert np.sum(lb == -0.30) == 80 and np.sum(ub == 0.15) == 160
    assert np.sum(np.isfinite(lb) & np.isfinite(ub) & (lb < ub)) == 16 * 20  # two-sided rows
    assert np.sum(lb == ub) == 12 * 21
    # x0 = [Xref(:); Uref(:)], Xref endpoints exact
    assert np.array_equal(x0[:6], q0) and np.array_equal(x0[12 * 20:12 * 20 + 6], [0, 0, 0.275, 0, 0, 0])
    assert np.allclose(x0[12 * 21:12 * 21 + 3], q0[:3] + [0.2, -0.1, -0.2])
    assert np.all(x0[12 * 21 + 12:12 * 21 + 24] == 0)
    # gradient-based NLP scaling (nlp_scaling_max_gradient = 50) is the identity at x0
    _, g, J = o21.jac_g(x0, p)
    assert np.max(np.abs(J)) <= 50.0


def _host_harness():
    d = os.path.join(os.path.dirname(__file__), "hostcheck")
    so = os.path.join(d, "libknot_host.so")
    src = os.path.join(d, "knot_host.cpp")
    hdr = os.path.join(d, "..", "..", "landing_controller_b200", "csrc", "srb_knot.cuh")
    if (not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(src), os.path.getmtime(hdr))):
        subprocess.check_call(["/usr/bin/g++", "-O1", "-std=c++17", "-fPIC", "-shared", src, "-o", so])
    h = ctypes.CDLL(so)
    h.hostcheck_sparsity.restype = c_llp
    return h


@pytest.mark.parametrize("N", [21, 30, 50])
def test_kernel_template_on_host_matches_oracle(N):
    """The device knot template (srb_knot.cuh) compiled for the host: values and CCS maps."""
    h = _host_harness()
    o = Oracle(N)
    sj = np.ctypeslib.as_array(h.hostcheck_sparsity(N, 0), shape=(len(o.spJ),))
    sh = np.ctypeslib.as_array(h.hostcheck_sparsity(N, 1), shape=(len(o.spH),))
    assert np.array_equal(sj, o.spJ) and np.array_equal(sh, o.spH)
    rng = np.random.default_rng(N)
    for _ in range(20):
        x = rng.normal(size=o.nx) * 0.4
        p = rng.uniform(0.5, 1.5, size=o.np_)
        lam = rng.normal(size=o.m)
        g, J, H = np.zeros(o.m), np.zeros(o.nnzJ), np.zeros(o.nnzH)
        h.hostcheck_eval(N, _dp(x), _dp(p), ctypes.c_double(0.3), _dp(lam), _dp(g), _dp(J), _dp(H))
        _, g0, J0 = o.jac_g(x, p)
        _, H0 = o.hess_l(x, p, 0.3, lam)
        assert rel(g, g0) < TOL and rel(J, J0) < TOL and rel(H, H0) < TOL
