"""Time-varying LQR pass (quadruped_SRBM_NLP.m:428-497): the numpy restatement (oracle/tvlqr_ref.py) against its defining
properties on CPU, the CUDA kernel against the restatement on GPU.  The reference keeps no output of this pass."""
import os
import sys

import numpy as np
import pytest

import landing_controller_b200 as lc

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
from crba_constants import zero_configuration  # noqa: E402
import tvlqr_ref  # noqa: E402

FIX = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ccc_n41.npz")


def _stored(b):
    d = np.load(FIX)
    return d["X"][b], np.vstack([d["c"][b], d["f"][b]])


def test_inertia_at_the_zero_configuration():
    z = zero_configuration()
    assert z["mass"] == 8.251999999999999            # same links, same total mass as at q_home
    assert np.allclose(z["Ib3"], z["Ib3"].T) and np.all(np.linalg.eigvalsh(z["Ib3"]) > 0)
    assert np.allclose(np.diag(z["Ib3"]), [0.082057376, 0.246291, 0.267475776], rtol=1e-9)


def test_variational_dynamics_structure_and_limits():
    z = zero_configuration()
    rng = np.random.default_rng(0)
    xd, ud = rng.normal(size=24) * 0.3, rng.normal(size=12) * 20
    A, B = tvlqr_ref.variational_AB(xd, ud, z["Ib3"], z["mass"])
    # kinematics rows and the linear-momentum row are exact, whatever the reference point
    assert np.array_equal(A[0:3, 9:12], np.eye(3)) and np.count_nonzero(A[0:3]) == 3
    assert np.array_equal(A[3:6, 6:9], np.eye(3)) and np.allclose(A[3:6, 3:6], -tvlqr_ref.skew(xd[6:9]))
    assert np.allclose(B[9:12], np.tile(np.eye(3), 4) / z["mass"]) and np.count_nonzero(A[9:12]) == 0
    # the angular row is the derivative of Ib^-1 (R' sum (pf - p) x f - omega x Ib omega) w.r.t. forces, feet and p
    def wdot(p, pf, f, om):
        Rt = tvlqr_ref.rpy_to_rot(xd[3:6])
        tau = sum(np.cross(pf[3 * l:3 * l + 3] - p, f[3 * l:3 * l + 3]) for l in range(4))
        return np.linalg.solve(z["Ib3"], Rt @ tau - np.cross(om, z["Ib3"] @ om))
    eps = 1e-6
    for j in range(12):
        e = np.zeros(12); e[j] = eps
        fd = (wdot(xd[0:3], xd[12:24], ud + e, xd[6:9]) - wdot(xd[0:3], xd[12:24], ud - e, xd[6:9])) / (2 * eps)
        assert np.allclose(B[6:9, j], fd, atol=1e-6)
        fd = (wdot(xd[0:3], xd[12:24] + e, ud, xd[6:9]) - wdot(xd[0:3], xd[12:24] - e, ud, xd[6:9])) / (2 * eps)
        assert np.allclose(A[6:9, 12 + j], fd, atol=1e-5)
    for j in range(3):
        e = np.zeros(3); e[j] = eps
        fd = (wdot(xd[0:3] + e, xd[12:24], ud, xd[6:9]) - wdot(xd[0:3] - e, xd[12:24], ud, xd[6:9])) / (2 * eps)
        assert np.allclose(A[6:9, j], fd, atol=1e-5)
    # gyroscopic block: Ib^-1 (skew(Ib om) - skew(om) Ib) = -d/d om [Ib^-1 (om x Ib om)]
    om = xd[6:9]
    for j in range(3):
        e = np.zeros(3); e[j] = eps
        g = lambda o: np.linalg.solve(z["Ib3"], -np.cross(o, z["Ib3"] @ o))
        assert np.allclose(A[6:9, 6 + j], (g(om + e) - g(om - e)) / (2 * eps), atol=1e-6)


def test_riccati_pass_properties_on_a_stored_trajectory():
    z = zero_configuration()
    X, U = _stored(2)  # drop_vZ
    Q, R, F, dt = tvlqr_ref.default_weights()
    n = int(round(0.6 / dt)) + 1
    P, K = tvlqr_ref.riccati_backward(X, U, 0.6, Q, R, F, dt, n, z["Ib3"], z["mass"])
    assert np.array_equal(P[-1], F)
    for k in range(n):
        assert np.allclose(P[k], P[k].T, atol=1e-9 * max(1.0, np.abs(P[k]).max()))
    # explicit Euler (what the reference integrates with, generateRiccatiIntegrator.m:53) does not keep P positive
    # semi-definite at dt = 0.022 on a 250 N landing; the defect is first order in dt and vanishes with it
    def defect(step):
        m = int(round(0.6 / step)) + 1
        Pm, _ = tvlqr_ref.riccati_backward(X, U, 0.6, Q, R, F, step, m, z["Ib3"], z["mass"])
        return -min(np.linalg.eigvalsh(0.5 * (p + p.T)).min() for p in Pm) / np.abs(Pm).max()
    d1, d2, d3 = defect(0.022), defect(0.005), defect(0.001)
    assert d1 > d2 > d3 and d3 < 1e-4
    # one step re-derived independently: P[k-1] - P[k] = dt (A'P + PA - P B R^-1 B'P + Q)
    k = n // 2
    t_star = np.arange(41) * 0.6 / 40
    xd, ud = tvlqr_ref.sample_reference(X, U, t_star, k * dt)
    A, B = tvlqr_ref.variational_AB(xd, ud, z["Ib3"], z["mass"])
    rhs = A.T @ P[k] + P[k] @ A - P[k] @ B @ np.diag(1 / R) @ B.T @ P[k] + Q
    assert np.allclose((P[k - 1] - P[k]) / dt, rhs, rtol=1e-9, atol=1e-9)
    assert np.allclose(K[k], np.diag(1 / R) @ B.T @ P[k])


@pytest.mark.gpu
def test_gpu_tvlqr_matches_restatement():
    z = zero_configuration()
    d = np.load(FIX)
    idx = [0, 2, 7, 17, 35]
    xs = np.array([np.concatenate([d["X"][b].T.ravel(), np.hstack([d["c"][b].T, d["f"][b].T]).ravel()]) for b in idx])
    s = lc.LandingSolver(N=41)
    par = s.tvlqr_default()
    assert par.n_steps == 28 and abs(par.mass - z["mass"]) < 1e-15 and np.allclose(list(par.Ib), z["Ib3"].ravel(), rtol=1e-12)
    P, K = s.tvlqr(xs, par)
    s.close()
    Q, R, F, dt = tvlqr_ref.default_weights()
    for i, b in enumerate(idx):
        U = np.vstack([d["c"][b], d["f"][b]])
        Pr, Kr = tvlqr_ref.riccati_backward(d["X"][b], U, 0.6, Q, R, F, dt, par.n_steps, z["Ib3"], z["mass"])
        assert np.max(np.abs(P[i] - Pr)) <= 1e-10 * max(1.0, np.abs(Pr).max())
        assert np.max(np.abs(K[i] - Kr)) <= 1e-10 * max(1.0, np.abs(Kr).max())


def _spd(rng, n, lo, hi):
    """Random symmetric positive definite n x n with eigenvalues in [lo, hi], exactly symmetric (the kernel forms
    A'P + PA as W + W', which needs a symmetric P)."""
    V, _ = np.linalg.qr(rng.normal(size=(n, n)))
    S = (V * rng.uniform(lo, hi, n)) @ V.T
    return 0.5 * (S + S.T)


def _weights(rng):
    """Full (non-diagonal) SPD Q and F over all 24 states, a non-uniform R, a full SPD body inertia with off-diagonal
    entries and a non-default mass."""
    z = zero_configuration()
    Ib = z["Ib3"] + 0.01 * _spd(rng, 3, 0.2, 1.0) + 0.004 * (np.ones((3, 3)) - np.eye(3))
    return dict(Q=_spd(rng, 24, 0.05, 2.0), F=_spd(rng, 24, 0.5, 6.0), R=rng.uniform(40.0, 150.0, 12), Ib=Ib,
                mass=rng.uniform(6.0, 11.0))


def _random_trajectories(rng, N, B):
    """Landing-like trajectories X [B, 12, N], U [B, 24, N-1]: feet near their nominal place under the hips, forces up
    to 100 N per leg."""
    X = np.empty((B, 12, N))
    X[:, 0:2], X[:, 2] = rng.uniform(-0.1, 0.1, (B, 2, N)), rng.uniform(0.2, 0.4, (B, N))
    X[:, 3:6], X[:, 6:12] = rng.uniform(-0.3, 0.3, (B, 3, N)), rng.uniform(-1, 1, (B, 6, N))
    feet = np.array([[0.2, -0.15, -0.3], [0.2, 0.15, -0.3], [-0.2, -0.15, -0.3], [-0.2, 0.15, -0.3]]).ravel()
    U = np.empty((B, 24, N - 1))
    U[:, 0:12] = np.tile(X[:, 0:3, :-1], (1, 4, 1)) + feet[None, :, None] + rng.uniform(-0.05, 0.05, (B, 12, N - 1))
    U[:, 12:24] = rng.uniform(-20, 20, (B, 12, N - 1))
    U[:, 14::3] = rng.uniform(0, 100, (B, 4, N - 1))
    return X, U


def _stored_trajectories(idx):
    d = np.load(FIX)
    return np.array([d["X"][b] for b in idx]), np.array([np.vstack([d["c"][b], d["f"][b]]) for b in idx])


def _par(s, T, dt, n_steps, w):
    par = s.tvlqr_default()
    par.T, par.dt, par.n_steps, par.mass = T, dt, n_steps, w["mass"]
    par.Q[:], par.F[:], par.R[:], par.Ib[:] = (w[k].ravel().tolist() for k in ("Q", "F", "R", "Ib"))
    return par


def _check(P, K, X, U, T, dt, n_steps, w, which):
    """P [n_steps, 24, 24] and K [n_steps, 12, 24] of the trajectories `which` against the restatement; worst errors."""
    wp = wk = 0.0
    for i in which:
        Pr, Kr = tvlqr_ref.riccati_backward(X[i], U[i], T, w["Q"], w["R"], w["F"], dt, n_steps, w["Ib"], w["mass"])
        if P is not None:
            e = np.max(np.abs(P[i] - Pr)) / max(1.0, np.abs(Pr).max())
            assert e <= 1e-10, (i, e)
            wp = max(wp, e)
        if K is not None:
            e = np.max(np.abs(K[i] - Kr)) / max(1.0, np.abs(Kr).max())
            assert e <= 1e-10, (i, e)
            wk = max(wk, e)
    return wp, wk


def _xs(X, U):
    return np.array([np.concatenate([x.T.ravel(), u.T.ravel()]) for x, u in zip(X, U)])


# (N, T, dt, n_steps, trajectories): every time point on a knot (dt = T/(N-1) and 2T/(N-1)), the reference's step on
# another horizon, one time point only, a long pass of 301 steps
TVLQR_CASES = [(21, 0.5, 0.5 / 20, 21, "random"), (30, 0.3, 2 * 0.3 / 29, 15, "random"), (41, 0.45, 0.022, 21, "random"),
               (41, 0.6, 0.022, 1, "stored"), (41, 0.6, 0.002, 301, "stored")]


@pytest.mark.gpu
@pytest.mark.parametrize("N,T,dt,n_steps,traj", TVLQR_CASES)
def test_gpu_tvlqr_full_weights_and_other_grids(N, T, dt, n_steps, traj):
    rng = np.random.default_rng(N * 1000 + n_steps)
    w = _weights(rng)
    X, U = _random_trajectories(rng, N, 4) if traj == "random" else _stored_trajectories([0, 2, 17])
    s = lc.LandingSolver(N=N)
    P, K = s.tvlqr(_xs(X, U), _par(s, T, dt, n_steps, w))
    s.close()
    wp, wk = _check(P, K, X, U, T, dt, n_steps, w, range(len(X)))
    print("tvlqr N=%d T=%g dt=%g n_steps=%d: worst rel. error P %.2e, K %.2e" % (N, T, dt, n_steps, wp, wk))


@pytest.mark.gpu
def test_gpu_tvlqr_single_outputs_device_buffers_and_a_large_batch():
    """P_out or K_out NULL (each alone) through the C ABI, device buffers, and B = 300 CTAs checked on a sample."""
    import ctypes
    import torch
    N, B, T, dt, n_steps = 21, 300, 0.6, 0.022, 28
    rng = np.random.default_rng(300)
    w = _weights(rng)
    X, U = _random_trajectories(rng, N, B)
    xs = _xs(X, U)
    s = lc.LandingSolver(N=N)
    par = _par(s, T, dt, n_steps, w)
    P, K = s.tvlqr(xs, par)
    wp, wk = _check(P, K, X, U, T, dt, n_steps, w, [0, 1, 127, 128, 255, 299])
    print("tvlqr B=%d: worst rel. error P %.2e, K %.2e" % (B, wp, wk))
    dp = ctypes.POINTER(ctypes.c_double)
    Ponly, Konly = np.zeros_like(P[:3]), np.zeros_like(K[:3])
    x3 = np.ascontiguousarray(xs[:3])
    for Pp, Kp in ((Ponly, None), (None, Konly)):
        rc = s.lib.landing_tvlqr_batch(s.ctx, 3, lc.HOST, ctypes.byref(par), x3.ctypes.data_as(dp),
                                       None if Pp is None else Pp.ctypes.data_as(dp),
                                       None if Kp is None else Kp.ctypes.data_as(dp))
        assert rc == 0, s.lib.landing_last_error()
    assert np.array_equal(Ponly, P[:3]) and np.array_equal(Konly, K[:3])
    dev = torch.device("cuda:0")
    xt = torch.tensor(xs[:5], device=dev)
    Pt = torch.full((5, n_steps, 24, 24), float("nan"), dtype=torch.float64, device=dev)
    Kt = torch.full((5, n_steps, 12, 24), float("nan"), dtype=torch.float64, device=dev)
    rc = s.lib.landing_tvlqr_batch(s.ctx, 5, lc.DEVICE, ctypes.byref(par), ctypes.cast(xt.data_ptr(), dp),
                                   ctypes.cast(Pt.data_ptr(), dp), ctypes.cast(Kt.data_ptr(), dp))
    assert rc == 0, s.lib.landing_last_error()
    s.synchronize()
    assert np.array_equal(Pt.cpu().numpy(), P[:5]) and np.array_equal(Kt.cpu().numpy(), K[:5])
    s.close()
