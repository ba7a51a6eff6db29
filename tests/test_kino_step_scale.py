"""Interior-point Newton step of the kino-dynamic NLP on the GPU (landing_kino_step_batch) where one CTA serves several
scenarios, at more knot counts and at near-converged iterates.

k_kino_step runs a persistent grid of at most the resident CTAs; each CTA takes scenario ids from a counter and reuses
its shared stage matrix, its reduction slots and its scratch slot for the next one.  An SM holds at most 2048 threads,
8 CTAs of 256, so a batch of more than 8 x SMs scenarios makes some CTA take at least two, whatever the occupancy.  Such a
batch, mixing inertia corrections of different lengths, factorisation failures and non-interior iterates, is checked bit
for bit against the same scenarios in calls of at most SMs scenarios (one per CTA) and under permutation, against the
host build and the full unreduced system, and across a context whose scratch grows between calls.  Then the full-system
check at N = 4, 30 and 50, and the near-converged iterates of tests/test_kino_step_cond.py as a batch."""
import os
import sys
import time

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
from test_kino_step import make_inputs, step, dense, OUT  # noqa: E402
from test_kino_step_host import (harness, patterns, ccs, eq_rows, full_system, fraction_to_boundary,  # noqa: E402,F401
                                 dw_trials, run_host, rel)
from test_kino_step_cond import MUS, TAGS, scenario_at, sigma, errors  # noqa: E402

pytestmark = pytest.mark.gpu
ALL = OUT + ("delta_w", "n_factor", "status", "alpha_pr", "alpha_du")
ST_FACTOR_FAIL, ST_NOT_INTERIOR = 4, 5  # include/landing_b200.h


def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def take(inp, idx):
    return {k: v[idx] for k, v in inp.items()}


def chunked(s, lc, inp, layout, memspace, size):
    """The batch in consecutive calls of at most `size` scenarios, outputs concatenated."""
    B = inp["mu"].shape[0]
    parts = [step(s, lc, take(inp, slice(a, min(a + size, B))), layout, memspace) for a in range(0, B, size)]
    return {k: np.concatenate([p[k] for p in parts]) for k in ALL}


def assert_same(out, ref, idx=slice(None), what=""):
    for k in ALL:
        assert np.array_equal(out[k], ref[k][idx], equal_nan=True), (what, k)


def host_scenario(inp, b):
    sc = {k: inp[k][b] for k in ("g", "s", "y", "zL", "zU", "lbg", "ubg")}
    sc.update(jv=inp["jac"][b], hv=inp["hess"][b], gf=inp["grad_f"][b])
    return sc


def host_matches(h, N, inp, out, idx):
    """status of the host build equals the GPU's on the scenarios idx, and so do delta_w and n_factor wherever the host
    build reports them (not for a non-interior iterate)."""
    jsp, hsp = patterns(N)
    for b in idx:
        _, r = run_host(h, N, jsp, hsp, host_scenario(inp, b), inp["mu"][b], inp["dw_last"][b])
        assert r[2] == out["status"][b], (b, r)
        if r[2] != ST_NOT_INTERIOR:
            assert r[1] == out["n_factor"][b] and r[0] == out["delta_w"][b], (b, r)


def against_full_system(N, inp, out, idx):
    """Sampled scenarios against the refined solve of the unreduced system (1e-9 relative), the normalised residual of
    the GPU direction in that system (1e-13) and alpha_pr / alpha_du against numpy (exactly).  Returns the worst
    forward error and residual."""
    jsp, hsp = patterns(N)
    worst = worst_res = 0.0
    for b in idx:
        J, W = dense(jsp, inp["jac"][b]), dense(hsp, inp["hess"][b], sym=True)
        args = [inp[k][b] for k in ("grad_f", "g", "s", "y", "zL", "zU", "lbg", "ubg")]
        exact, (A, rhs, pack) = full_system(N, J, W, *args, inp["mu"][b], out["delta_w"][b], want_system=True)
        for name, e in zip(OUT, exact):
            err = rel(out[name][b], e)
            worst = max(worst, err)
            assert err < 1e-9, (N, b, name, err)
        z = pack(*[out[k][b] for k in OUT])
        r = np.max(np.abs(A @ z - rhs)) / (abs(A).max() * np.max(np.abs(z)) + np.max(np.abs(rhs)))
        worst_res = max(worst_res, r)
        assert r < 1e-13, (N, b, r)
        apr, adu = fraction_to_boundary(N, inp["s"][b], out["ds"][b], inp["zL"][b], out["dzL"][b], inp["zU"][b],
                                        out["dzU"][b], inp["lbg"][b], inp["ubg"][b], 0.99)
        assert apr == out["alpha_pr"][b] and adu == out["alpha_du"][b], b
    return worst, worst_res


def control_diag(N, hsp, k):
    """CCS position of a diagonal Hessian entry of a control variable of stage k (jpos_k)."""
    colind, row = ccs(hsp)
    for c in range(12 * N + 12 * k, 12 * N + 12 * k + 12):
        e = np.flatnonzero(row[colind[c]:colind[c + 1]] == c)
        if e.size:
            return int(colind[c] + e[0])
    raise AssertionError("no diagonal Hessian entry on a control of stage %d" % k)


def mixed_batch(s, N, B, seed):
    """B scenarios whose CTAs get out of step: every third with y_scale = 100 (delta_w > 0, several factorisations),
    dw_last from {0, 1e-9, 3e-3, 0.5}, a NaN on a control's Hessian diagonal in the middle stage every 97th
    (LANDING_ST_FACTOR_FAIL after the whole schedule) and a slack on its lower bound every 89th
    (LANDING_ST_NOT_INTERIOR).  Returns the inputs and the indices of the two kinds of failure."""
    rng = np.random.default_rng(seed)
    nbig = len(range(2, B, 3))
    small = make_inputs(s, rng, N, B - nbig)
    big = make_inputs(s, rng, N, nbig, y_scale=100.0)
    isbig = np.arange(B) % 3 == 2
    inp = {}
    for k in small:
        v = np.empty((B,) + small[k].shape[1:], dtype=small[k].dtype)
        v[~isbig], v[isbig] = small[k], big[k]
        inp[k] = v
    inp["dw_last"] = rng.choice([0.0, 1e-9, 3e-3, 0.5], size=B)
    _, hsp = patterns(N)
    nan_b = np.arange(96, B, 97)
    inp["hess"][nan_b, control_diag(N, hsp, (N - 1) // 2)] = np.nan
    ni_b = np.arange(88, B, 89)
    for b in ni_b:
        i = np.flatnonzero(~eq_rows(N) & np.isfinite(inp["lbg"][b]))[7]
        inp["s"][b, i] = inp["lbg"][b, i]
    return inp, nan_b, ni_b


@pytest.fixture(scope="module")
def grid_batch():
    """The mixed batch at N = 21 with B = 8 SMs + 37, and its outputs from one call on a fresh context (SoA, device)."""
    import landing_controller_b200 as lc
    N = 21
    sms = sm_count()
    B = 8 * sms + 37
    s = lc.LandingSolver(N=N, device=0)
    inp, nan_b, ni_b = mixed_batch(s, N, B, 2100)
    out = step(s, lc, inp, "SOA", "DEVICE")
    print("\npersistent grid: B = %d scenarios at N = %d on %d SMs; B > 8 x SMs = %d, so some CTA served at least two"
          % (B, N, sms, 8 * sms))
    return dict(N=N, B=B, sms=sms, inp=inp, out=out, nan_b=nan_b, ni_b=ni_b)


def test_gpu_step_persistent_grid_equals_one_scenario_per_cta(grid_batch):
    """The whole batch in one call equals, bit for bit, the same scenarios in calls of at most SMs scenarios (one per
    CTA), in SoA / device and AoS / host (AoS with B >= 64 on the transposed path, the chunks too)."""
    import landing_controller_b200 as lc
    g = grid_batch
    s = lc.LandingSolver(N=g["N"], device=0)
    assert_same(chunked(s, lc, g["inp"], "SOA", "DEVICE", g["sms"]), g["out"], what="SOA chunks")
    aos = step(s, lc, g["inp"], "AOS", "HOST")
    assert_same(aos, g["out"], what="AOS whole")
    assert_same(chunked(s, lc, g["inp"], "AOS", "HOST", g["sms"]), aos, what="AOS chunks")


def test_gpu_step_persistent_grid_is_order_invariant(grid_batch):
    """Reversed and randomly permuted, every scenario's outputs are unchanged bit for bit."""
    import landing_controller_b200 as lc
    g = grid_batch
    s = lc.LandingSolver(N=g["N"], device=0)
    for perm in (np.arange(g["B"])[::-1], np.random.default_rng(7).permutation(g["B"])):
        out = step(s, lc, take(g["inp"], perm), "SOA", "DEVICE")
        assert_same(out, g["out"], perm, what="permuted")


def test_gpu_step_persistent_grid_failures(grid_batch, harness):  # noqa: F811
    """A NaN on a control's Hessian diagonal: LANDING_ST_FACTOR_FAIL with n_factor and delta_w of the whole schedule (as
    the host build and dw_trials) and NaN outputs; a slack on its bound: LANDING_ST_NOT_INTERIOR, n_factor 0, NaN
    delta_w and outputs; every other scenario status 0 with delta_w and n_factor equal to the host build's."""
    g = grid_batch
    inp, out = g["inp"], g["out"]
    bad = np.zeros(g["B"], dtype=bool)
    bad[g["nan_b"]] = bad[g["ni_b"]] = True
    assert np.all(out["status"][~bad] == 0)
    assert np.all(out["status"][g["nan_b"]] == ST_FACTOR_FAIL)
    assert np.all(out["status"][g["ni_b"]] == ST_NOT_INTERIOR)
    assert np.all(out["n_factor"][g["ni_b"]] == 0) and np.all(np.isnan(out["delta_w"][g["ni_b"]]))
    for b in g["nan_b"]:
        trials = dw_trials(inp["dw_last"][b], 200)
        nf = next(i for i, d in enumerate(trials) if d > 1e40)
        assert out["n_factor"][b] == nf and out["delta_w"][b] == trials[nf], (b, out["n_factor"][b], nf)
    for k in OUT + ("alpha_pr", "alpha_du"):
        assert np.all(np.isnan(out[k][bad])), k
        assert np.all(np.isfinite(out[k][~bad])), k
    t0 = time.time()
    host_matches(harness, g["N"], inp, out, range(g["B"]))
    print("failures: %d factorisation failures (n_factor %s), %d non-interior; host build on all %d scenarios in %.0f s"
          % (len(g["nan_b"]), sorted(set(out["n_factor"][g["nan_b"]].tolist())), len(g["ni_b"]), g["B"],
             time.time() - t0))


def test_gpu_step_persistent_grid_against_the_full_system(grid_batch):
    """About 12 good scenarios spread over the batch, some among the last SMs ids (reached only after an earlier
    scenario on the same CTA), against the full unreduced system."""
    g = grid_batch
    good = np.flatnonzero(g["out"]["status"] == 0)
    rng = np.random.default_rng(12)
    late = good[good >= g["B"] - g["sms"]]
    idx = sorted(set(rng.choice(good, 9, replace=False).tolist()) | set(rng.choice(late, 3, replace=False).tolist()))
    worst, worst_res = against_full_system(g["N"], g["inp"], g["out"], idx)
    print("persistent grid N=%d, scenarios %s: worst %.2e vs full system, residual %.2e, delta_w %s" %
          (g["N"], idx, worst, worst_res, np.unique(g["out"]["delta_w"][good]).tolist()))


def test_gpu_step_scratch_grows_on_one_context(grid_batch):
    """One context called with B = 5, then the large batch (the scratch grows to the resident CTAs), then the first 5
    again: each call equals a fresh context's bit for bit."""
    import landing_controller_b200 as lc
    g = grid_batch
    first = take(g["inp"], slice(0, 5))
    fresh5 = step(lc.LandingSolver(N=g["N"], device=0), lc, first, "SOA", "DEVICE")
    s = lc.LandingSolver(N=g["N"], device=0)
    assert_same(step(s, lc, first, "SOA", "DEVICE"), fresh5, what="B=5 first")
    assert_same(step(s, lc, g["inp"], "SOA", "DEVICE"), g["out"], what="large batch after B=5")
    assert_same(step(s, lc, first, "SOA", "DEVICE"), fresh5, what="B=5 after the large batch")


@pytest.mark.parametrize("N,B,layout,memspace,nsample", [(4, 1, "AOS", "HOST", 1), (4, 64, "AOS", "HOST", 4),
                                                         (30, 65, "SOA", "DEVICE", 4), (50, 33, "SOA", "DEVICE", 3)])
def test_gpu_step_at_more_knot_counts(harness, N, B, layout, memspace, nsample):  # noqa: F811
    """N = 4 (the smallest problem with a control stage that is neither the first nor the last), N = 30 and N = 50 (the
    benchmark's largest): sampled scenarios against the full system, delta_w / n_factor of every scenario against the
    host build."""
    import landing_controller_b200 as lc
    s = lc.LandingSolver(N=N, device=0)
    rng = np.random.default_rng(300 + N + B)
    inp = make_inputs(s, rng, N, B)
    inp["dw_last"][1::3] = 3e-3
    out = step(s, lc, inp, layout, memspace)
    assert np.all(out["status"] == 0)
    host_matches(harness, N, inp, out, range(B))
    idx = sorted({B - 1} | set(rng.choice(B - 1, size=min(nsample - 1, B - 1), replace=False).tolist()))
    t0 = time.time()
    worst, worst_res = against_full_system(N, inp, out, idx)
    print("N=%d B=%d %s/%s, %d scenarios: worst %.2e vs full system, residual %.2e (%.1f s), delta_w %s" %
          (N, B, layout, memspace, len(idx), worst, worst_res, time.time() - t0, np.unique(out["delta_w"]).tolist()))


def test_gpu_step_persistent_grid_at_n50(harness):  # noqa: F811
    """N = 50 with B = 8 SMs + 37: bit for bit against calls of at most SMs scenarios, and delta_w / n_factor / status
    of every scenario against the host build."""
    import landing_controller_b200 as lc
    N = 50
    sms = sm_count()
    B = 8 * sms + 37
    s = lc.LandingSolver(N=N, device=0)
    inp, _, _ = mixed_batch(s, N, B, 5000)
    out = step(s, lc, inp, "SOA", "DEVICE")
    assert_same(chunked(s, lc, inp, "SOA", "DEVICE", sms), out, what="N=50 chunks")
    host_matches(harness, N, inp, out, range(B))
    print("N=50: B = %d on %d SMs bit-identical to one scenario per CTA; status counts %s" %
          (B, sms, np.unique(out["status"], return_counts=True)))


def test_gpu_step_at_near_converged_iterates(harness):  # noqa: F811
    """The near-converged iterates of the stored KNITRO points (tests/test_kino_step_cond.py), each (point, mu) pair
    with dw_last 0 and 1e-4, repeated over a batch larger than 8 x SMs: status 0; every copy of a pair identical bit
    for bit; backward error <= 1e-13 in the unreduced system; delta_w / n_factor equal to the host build; dx within
    1e-9 of the host build's at mu = 1e-2 and elsewhere within 10x the host build's own forward error against the
    refined full-system solve (the GPU and host builds differ in FMA contraction)."""
    import landing_controller_b200 as lc
    N = 21
    jsp, hsp = patterns(N)
    combos = [(tag, mu, dwl) for tag in TAGS for mu in MUS for dwl in (0.0, 1e-4)]
    scs = {(tag, mu): scenario_at(tag, mu, jsp, hsp) for tag in TAGS for mu in MUS}
    sms = sm_count()
    B = 8 * sms + 37
    which = np.arange(B) % len(combos)
    rows = {"g": "g", "jac": "jv", "hess": "hv", "grad_f": "gf", "s": "s", "y": "y", "zL": "zL", "zU": "zU",
            "lbg": "lbg", "ubg": "ubg"}
    stack = {k: np.array([scs[c[:2]][v] for c in combos]) for k, v in rows.items()}
    inp = {k: v[which] for k, v in stack.items()}
    inp["mu"] = np.array([c[1] for c in combos])[which]
    inp["dw_last"] = np.array([c[2] for c in combos])[which]
    s = lc.LandingSolver(N=N, device=0)
    out = step(s, lc, inp, "SOA", "DEVICE")
    assert np.all(out["status"] == 0), np.unique(out["status"])
    for j, (tag, mu, dwl) in enumerate(combos):
        idx = np.flatnonzero(which == j)
        for k in ALL:
            assert np.all(out[k][idx] == out[k][idx[0]]), (tag, mu, dwl, k)
        b = idx[0]
        sc = scs[(tag, mu)]
        houts, r = run_host(harness, N, jsp, hsp, sc, mu, dwl)
        assert r[0] == out["delta_w"][b] and r[1] == out["n_factor"][b], (tag, mu, dwl, r)
        gouts = [out[k][b] for k in OUT]
        back, fwd, _, _ = errors(sc, mu, gouts, r[0])
        hback, hfwd, _, _ = errors(sc, mu, houts, r[0])
        diff = rel(gouts[0], houts[0])
        print("%s mu=%.0e dw_last=%g: max sigma %.1e, delta_w %g (%d), GPU backward %.1e forward %.1e, host forward "
              "%.1e, |dx_gpu - dx_host| %.1e" % (tag, mu, dwl, sigma(sc).max(), r[0], r[1], back, fwd, hfwd, diff))
        assert back <= 1e-13, (tag, mu, dwl, back)
        assert diff <= (1e-9 if mu == 1e-2 else 10 * hfwd), (tag, mu, dwl, diff, hfwd)
    print("near-converged batch: B = %d on %d SMs (> 8 x SMs)" % (B, sms))
