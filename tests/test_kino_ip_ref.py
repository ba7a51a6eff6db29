"""CPU checks of the interior-point restatement of the kino-dynamic solve (tests/kino_ip_ref.py), which the GPU solve
(tests/test_kino_solve.py) is held to iterate by iterate.

The restatement converges at N = 21 from the stored KNITRO point of the `ms` drop (tests/golden/kino_n21.npz) with
mu_init = bound_push = bound_frac = 1e-4, and the oracle certifies the point it returns.  Measured on the CPU: 33
iterations in about 32 s (about 1 s per iteration at N = 21, most of it in the oracle's exact Hessian); 62 iterations for
the `gs` drop, which is left to the GPU tests.  At N = 3 and 4 the grid drops do not converge from the reference
trajectories or from SRB solutions (neither does the CPU SRB solve there: the horizons are too coarse for those drops),
so at those sizes a short run checks every accepted trial against the filter's acceptance rule, restated separately
(check_filter_acceptance)."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import kino_ip_ref as ki  # noqa: E402
from test_kino_step_host import patterns  # noqa: E402


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    return ki.build_harness(tmp_path_factory.mktemp("kino_ip_ref"))


def check_log(log, mu_init):
    """Every accepted trial satisfies the acceptance rule; mu is IPOPT's monotone sequence: each logged value is either
    the restart value after a re-centring or the previous value times powers of the Fiacco-McCormick update."""
    assert log
    prev = mu_init
    for e in log:
        if e["restart"]:
            prev = e["mu"]
            continue
        bad = ki.check_filter_acceptance(e)
        assert bad is None, (bad, e["it"])
        mu, m = prev, prev
        ok = mu == e["mu"]
        while not ok and m > 1e-5 * 1.0000001:
            m = max(1e-5, min(0.2 * m, m ** 1.5))
            ok = m == e["mu"]
        assert ok, (e["it"], prev, e["mu"])
        prev = e["mu"]


@pytest.mark.parametrize("N", [3, 4])
def test_accepted_trials_pass_the_filter_rule(harness, N):
    from landing_controller_b200.sweeps import grid_sweep
    jsp, hsp = patterns(N)
    pb, lbo, ubo, x0 = ki.drop_problem(N, grid_sweep(16)[5])
    log = []
    r = ki.solve(harness, ki.Problem(pb, jsp, hsp), lbo, ubo, x0, ki.options(max_iter=12), log)
    assert r["status"] in (ki.CONVERGED, ki.MAX_ITER, ki.LINESEARCH_FAIL, ki.FACTOR_FAIL)
    check_log(log, 0.1)
    assert np.all(np.isfinite(r["x"]))


def test_converges_from_the_stored_knitro_point_and_is_certified(harness):
    from test_kino import stored
    N = 21
    _, xs, _, (q0, qd0, _) = stored("ms")
    pb, lbo, ubo, _ = ki.drop_problem(N, np.concatenate([q0, qd0]))
    jsp, hsp = patterns(N)
    log = []
    o = ki.options(mu_init=1e-4, bound_push=1e-4, bound_frac=1e-4)
    r = ki.solve(harness, ki.Problem(pb, jsp, hsp), lbo, ubo, xs, o, log)
    assert r["status"] == ki.CONVERGED, r["status"]
    check_log(log, 1e-4)
    c = ki.certificate(pb, r["x"], r["y"], lbo, ubo)
    assert c["viol"] <= o["constr_viol_tol"] and c["stat"] <= o["tol"] and c["compl"] <= o["compl_inf_tol"], c
    f_stored, _ = ki.cost(xs, N)
    assert r["f"] <= f_stored + 1e-8, (r["f"], f_stored)
