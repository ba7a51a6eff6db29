"""GPU tests of the solver on its two variant problems, certified with the independent restatement (tests/variant_ref.py):
the fixed contact schedule (formulation 1, quadruped_SRBM_NLP.m) and the "CCC" problem (formulation 0 with a running
GRF cost and a tighter kinematic box, generate_quadruped_SRBM_CCC.m).  Also formulation 1 beyond the four-scenario
parity test: more scenarios than resident CTA slots, device buffers, a non-uniform dt, an initial guess, a context
that changes its problem between calls, and the multi-GPU entry point."""
import ctypes
import os

import numpy as np
import pytest

import ccc_problem as ccc
import landing_controller_b200 as lc
import variant_ref as vr
from oracle_ip import default_options, default_problem, solve_cpu, solve_cpu_x0
from test_variant_ref import certify, sched_cases, sched_problem

pytestmark = pytest.mark.gpu


def sched_solver(N, T, cs, dt=None, z_max=1.0, QX=lc.SCHED_QX):
    s = lc.LandingSolver(N=N)
    lc.apply_schedule_parameters(s.problem, z_max=z_max)
    s.problem.T = T
    if dt is not None:
        s.set_dt(dt)
    s.set_schedule(cs, QX)
    return s


def _check_against_cpu(r, c, conv):
    """where the GPU and CPU solutions agree to 1e-6, their multipliers agree to 5e-5 relative to max(1, |lam|)
    (measured: up to 8.2e-6 at N = 50, where max |lam| is 1.9e3 and some active rows are nearly dependent, so the
    multipliers are less well determined than x*); returns how many scenarios that covered"""
    n = 0
    for b in np.flatnonzero(conv & (c["status"] == 0)):
        dx = np.max(np.abs(r["x"][b] - c["x"][b]))
        lam = c["lam_g"][b]
        dl = np.max(np.abs(r["lam_g"][b] - lam) / np.maximum(1.0, np.abs(lam)))
        print("  scenario %d: max |dx| %.1e, max |dlam| / max(1, |lam|) %.1e" % (b, dx, dl))
        if dx <= 1e-6:
            assert dl <= 5e-5
            n += 1
    return n


@pytest.mark.parametrize("case", ["reference16", "config0", "alternating_dt", "n50"])
def test_fixed_schedule_solutions_are_kkt_points_of_the_restatement(case):
    N, T, cs, dt, z_max, drops = sched_cases()[case]
    s = sched_solver(N, T, cs, dt, z_max)
    r = s.solve(drops, want_lam=True)
    s.close()
    pb, opt = sched_problem(N, T, cs, dt, z_max)
    c = solve_cpu(N, drops, opt, pb, want_lam=True)
    conv = r["status"] == 0
    assert conv.all()
    out = [certify(vr.from_drop(N, pb, drops[b], cs=cs, Qf=lc.SCHED_QF, QX=lc.SCHED_QX, kin_box=lc.SCHED_KIN_BOX),
                   r["x"][b], r["lam_g"][b], r["f"][b], r["viol"][b]) for b in range(len(drops))]
    n = _check_against_cpu(r, c, conv)
    print("%s (GPU): max stationarity %.1e, max |lam| %.1e, multipliers checked against the CPU on %d of %d"
          % (case, max(a for a, _ in out), max(m for _, m in out), n, len(drops)))
    # (on the reference's own N = 16 problem the GPU and CPU x* differ by more than 1e-6; both are certified above)
    assert n >= 1 or case == "reference16"


def test_ccc_solutions_are_kkt_points_of_the_restatement():
    d = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ccc_n41.npz"))
    drops = np.ascontiguousarray(d["X"][:, :, 0])
    s = lc.LandingSolver(N=ccc.N)
    ccc.fill_problem(s.problem)
    r = s.solve(drops, want_lam=True)
    s.close()
    pb = ccc.fill_problem(default_problem())
    c = solve_cpu(ccc.N, drops, default_options(run_Qf=list(ccc.QF), kin_box=list(ccc.KIN_BOX)), pb, want_lam=True)
    conv = r["status"] == 0
    assert conv.mean() >= 0.9
    out = [certify(vr.from_drop(ccc.N, pb, drops[b], Qf=ccc.QF, kin_box=ccc.KIN_BOX), r["x"][b], r["lam_g"][b],
                   r["f"][b], r["viol"][b]) for b in np.flatnonzero(conv)]
    n = _check_against_cpu(r, c, conv)
    print("CCC (GPU): %d of %d converged, max stationarity %.1e, max |lam| %.1e, multipliers checked against the CPU "
          "on %d" % (conv.sum(), len(drops), max(a for a, _ in out), max(m for _, m in out), n))
    assert n >= 10


def _drop_family(B):
    """configs[0] with the forward speed and the pitch varied (the CPU restatement converges on all 297)"""
    d = np.repeat(lc.single_drop(), B, axis=0)
    t = np.linspace(0.0, 1.0, B)
    d[:, 9] = 0.5 + t
    d[:, 4] = 0.05 * np.cos(5.0 * t)
    return d


@pytest.mark.parametrize("B", [1, 297])
def test_fixed_schedule_beyond_the_resident_slots_host_and_device(B):
    """297 scenarios = one more than the 2 x 148 resident CTA slots of a B200: every scenario is bit-identical to a
    singleton solve, with host and with device buffers, and the first iterates equal the CPU restatement's."""
    import torch
    N, T = 30, 0.6
    cs = lc.ballistic_schedule(N, T, 0.5)
    drops = _drop_family(B)
    s = sched_solver(N, T, cs)
    r = s.solve(drops, want_lam=True)
    m, nx = s.dims["m"], s.dims["nx"]
    dev = torch.device("cuda:0")
    t = dict(x=torch.zeros(B, nx, dtype=torch.float64, device=dev), f=torch.zeros(B, dtype=torch.float64, device=dev),
             st=torch.full((B,), 9, dtype=torch.int32, device=dev), it=torch.zeros(B, dtype=torch.int32, device=dev),
             viol=torch.zeros(B, dtype=torch.float64, device=dev),
             lam=torch.zeros(B, m, dtype=torch.float64, device=dev))
    s.solve_device(torch.tensor(drops, device=dev), t["x"], t["f"], t["st"], t["it"], viol=t["viol"], lam_g=t["lam"])
    torch.cuda.synchronize()
    for key, name in (("x", "x"), ("f", "f"), ("st", "status"), ("it", "iters"), ("viol", "viol"), ("lam", "lam_g")):
        assert np.array_equal(t[key].cpu().numpy(), r[name]), name
    assert (r["status"] == 0).mean() >= 0.95
    for b in range(B):
        one = s.solve(drops[b:b + 1], want_lam=True)
        for k in ("x", "f", "lam_g", "viol", "status", "iters"):
            assert np.array_equal(one[k][0], r[k][b]), (b, k)
    s.options.max_iter = 2
    r2 = s.solve(drops)
    s.close()
    pb, opt = sched_problem(N, T, cs)
    opt.max_iter = 2
    c2 = solve_cpu(N, drops, opt, pb)
    assert np.array_equal(r2["iters"], c2["iters"])
    assert np.max(np.abs(r2["x"] - c2["x"])) <= 1e-8


def test_fixed_schedule_nonuniform_dt_from_an_initial_guess():
    """alternating knot spacings with a schedule built for them, solved from a caller's initial guess (the converged
    solution of a neighbouring drop): the first iterates equal the CPU restatement's from the same guess, and the
    converged points are KKT points of the restatement."""
    N, T, cs, dt, z_max, drops = sched_cases()["alternating_dt"]
    s = sched_solver(N, T, cs, dt)
    base = s.solve(drops)
    assert (base["status"] == 0).all()
    near = drops.copy()
    near[:, 9] += 0.05
    x0 = base["x"].copy()
    x0[:, :12] = near
    pb, opt = sched_problem(N, T, cs, dt)
    for iters in (1, 4):
        s.options.max_iter = iters
        opt.max_iter = iters
        g = s.solve(near, x0=x0)
        c = solve_cpu_x0(N, near, x0, opt, pb)
        assert np.array_equal(g["iters"], c["iters"])
        assert np.max(np.abs(g["x"] - c["x"])) <= 1e-8
    s.options.max_iter = 3000
    w = s.solve(near, x0=x0, want_lam=True)
    s.close()
    assert (w["status"] == 0).all()
    for b in range(len(near)):
        v = vr.from_drop(N, pb, near[b], cs=cs, Qf=lc.SCHED_QF, QX=lc.SCHED_QX, kin_box=lc.SCHED_KIN_BOX)
        certify(v, w["x"][b], w["lam_g"][b], w["f"][b], w["viol"][b])


def test_context_that_changes_schedule_weights_and_formulation_matches_fresh_contexts():
    """One context solves schedule 1, then schedule 2 with other running weights, then formulation 0; each result is
    bit-identical to a fresh context's (a stale schedule or stale QX on the device would show here)."""
    N, T = 30, 0.6
    drops = _drop_family(5)
    cs1 = lc.ballistic_schedule(N, T, 0.5)
    cs2 = cs1.copy()
    cs2[6:9, :2] = 0  # the front legs touch down later
    QX2 = 0.5 * np.asarray(lc.SCHED_QX)
    steps = [(cs1, lc.SCHED_QX), (cs2, QX2), (None, None)]
    s = sched_solver(N, T, cs1)
    seq = []
    for cs, QX in steps:
        s.set_schedule(cs, QX)
        seq.append(s.solve(drops, want_lam=True))
    s.close()
    for (cs, QX), got in zip(steps, seq):
        f = sched_solver(N, T, cs1)
        f.set_schedule(cs, QX)
        ref = f.solve(drops, want_lam=True)
        f.close()
        for k in ("x", "f", "lam_g", "viol", "status", "iters"):
            assert np.array_equal(got[k], ref[k]), k
    assert not np.array_equal(seq[0]["x"], seq[1]["x"]) and not np.array_equal(seq[1]["x"], seq[2]["x"])


def test_multi_gpu_entry_point_gathers_the_fixed_schedule_solutions():
    """landing_solve_batch_multi with formulation 1 (the same GPU listed more than once on a one-GPU machine) gathers
    the single-context bits, multipliers included."""
    import torch
    N, T = 30, 0.6
    cs = np.ascontiguousarray(lc.ballistic_schedule(N, T, 0.5), dtype=np.int32)
    drops = _drop_family(13)
    devices = [0, 1] if torch.cuda.device_count() >= 2 else [0, 0]
    m = lc.MultiGpuSolver(N, devices + [0])
    lc.apply_schedule_parameters(m.problem)
    m.problem.T = T
    m.problem.cs = cs.ctypes.data_as(ctypes.POINTER(ctypes.c_int))
    m.problem.formulation = 1
    for i in range(12):
        m.problem.QX[i] = lc.SCHED_QX[i]
    r = m.solve(drops, want_lam=True)
    m.close()
    s = sched_solver(N, T, cs)
    ref = s.solve(drops, want_lam=True)
    s.close()
    assert (ref["status"] == 0).all()
    for k in ("x", "f", "lam_g", "viol", "status", "iters"):
        assert np.array_equal(r[k], ref[k]), k
