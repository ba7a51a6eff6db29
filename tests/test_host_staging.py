"""Host staging of the batched C ABI.

Every batched entry point must return the same bits whether the caller's buffers are in host memory (staged copies,
or zero-copy for small evaluations) or in device memory, in AoS or SoA layout, for batch sizes on both sides of the
zero-copy (B < 64) and AoS-via-SoA (B >= 64) thresholds, and must issue the number of kernel launches listed here.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import landing_controller_b200 as lc
from landing_controller_b200.api import AOS, DEVICE, HOST, SOA, EvalIO, SolveIO, _ip, _ptr

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N = 21
SIZES = (1, 63, 64, 257)
BMAX = max(SIZES)
MAX_ITER = 5


@pytest.fixture(scope="module")
def s():
    solver = lc.LandingSolver(N=N, device=0)
    solver.options.max_iter = MAX_ITER
    yield solver
    solver.close()


@pytest.fixture(scope="module")
def data(s):
    """Seeded inputs of every entry point for BMAX scenarios (AoS); smaller batches take the first B rows."""
    rng = np.random.default_rng(7)
    d = s.dims
    drops = lc.random_sweep(BMAX, seed=3)
    p, x0 = s.build_host(drops)
    kd = s.kino_dims()
    _, _, kx0 = s.kino_setup_host(drops)
    return dict(
        drops=drops, p=p,
        x=x0 + 0.05 * rng.normal(size=x0.shape),
        x0=x0 + 0.01 * rng.normal(size=x0.shape),
        lam_f=rng.uniform(0.5, 1.5, size=(BMAX, 1)),
        lam_g=rng.normal(size=(BMAX, d["m"])),
        x_star=x0 + 0.02 * rng.normal(size=x0.shape),
        kx=kx0 + 0.05 * rng.normal(size=(BMAX, kd["nx"])),
    )


def call(s, memspace, layout, B, ins, outs, fn, aos_only=()):
    """Runs fn(B, pointers) with the inputs ins {name: AoS array or None} (transposed for SoA unless named in
    aos_only) and zeroed outputs outs {name: (n, dtype)}; returns the outputs as AoS numpy arrays and the change of
    the context's launch count."""
    tr = (lambda a: np.ascontiguousarray(a.T)) if layout == SOA else np.ascontiguousarray
    host_in = {k: None if a is None else (np.ascontiguousarray(a) if k in aos_only else tr(a)) for k, a in ins.items()}
    host_out = {k: tr(np.zeros((B, n), dtype=dt)) for k, (n, dt) in outs.items()}
    if memspace == DEVICE:
        import torch
        bufs = {k: None if a is None else torch.from_numpy(a).cuda() for k, a in {**host_in, **host_out}.items()}
        torch.cuda.synchronize()  # the library stream does not wait for torch's
    else:
        bufs = {**host_in, **host_out}
    before = s.launches
    rc = fn(B, {k: _ptr_of(a) for k, a in bufs.items()})
    assert rc == 0, s.lib.landing_last_error().decode()
    if memspace == DEVICE:
        s.synchronize()
        res = {k: bufs[k].cpu().numpy() for k in outs}
    else:
        res = host_out
    return {k: tr(a) if layout == SOA else a for k, a in res.items()}, s.launches - before


def _ptr_of(a):
    """C pointer of a numpy array or torch tensor, typed by its dtype."""
    if a is None:
        return None
    return _ptr(a, _ip) if "int32" in str(a.dtype) else _ptr(a)


def combos(layouts=(AOS, SOA)):
    return [(B, mem, lay) for B in SIZES for mem in (HOST, DEVICE) for lay in layouts]


def check_same(results, atomic=None):
    """All results of one batch size are bit-identical to the first (host, AoS) one.  atomic: {name: columns} that
    are sums accumulated with atomics (summation order varies between runs), compared to rounding instead."""
    ref = results[0][1]
    for key, r in results[1:]:
        assert set(r) == set(ref), key
        for k in ref:
            a, b = r[k], ref[k]
            cols = (atomic or {}).get(k)
            if cols is not None:
                np.testing.assert_allclose(a[:, cols], b[:, cols], rtol=1e-9, atol=1e-12, err_msg="%s %s" % (key, k))
                a, b = np.delete(a, cols, axis=1), np.delete(b, cols, axis=1)
            assert np.array_equal(a, b), "%s: %s differs" % (key, k)


def run_matrix(run, layouts=(AOS, SOA), atomic=None):
    """run(B, memspace, layout) -> (outputs, launches, expected launches) over all combinations."""
    by_b = {}
    for B, mem, lay in combos(layouts):
        out, n, want = run(B, mem, lay)
        assert n == want, "B=%d memspace=%d layout=%d: %d launches, expected %d" % (B, mem, lay, n, want)
        by_b.setdefault(B, []).append(((B, mem, lay), out))
    for B, res in by_b.items():
        check_same(res, atomic)


# ---------------------------------------------------------------- landing_eval_batch
# (outputs, status requested, inputs, launches when the kernels read the caller's layout, launches for an AoS batch
# with B >= 64, which runs on transposed copies: one transpose per present input and output)
EVAL_CASES = [
    (("f",), True, ("x", "p"), 1, 4),
    (("g",), True, ("x", "p"), 1, 4),
    (("g", "jac"), True, ("x", "p"), 1, 5),
    (("g", "jac"), False, ("x", "p"), 1, 5),
    (("hess",), True, ("x", "p", "lam_f", "lam_g"), 1, 6),
    (("f", "grad_f"), True, ("x", "p"), 1, 5),
    (("grad_x", "grad_p"), True, ("x", "p", "lam_f", "lam_g"), 1, 7),
    (("f", "g", "grad_f", "jac", "hess", "grad_x", "grad_p"), True, ("x", "p", "lam_f", "lam_g"), 2, 13),
    ((), True, ("x", "p"), 0, 2),
]
EVAL_IN = ("x", "p", "lam_f", "lam_g")
EVAL_OUT = ("f", "g", "grad_f", "jac", "hess", "grad_x", "grad_p")


def eval_sizes(s):
    d = s.dims
    return dict(f=1, g=d["m"], grad_f=d["nx"], jac=d["nnzJ"], hess=d["nnzH"], grad_x=d["nx"], grad_p=d["np"])


def eval_call(s, data, B, mem, lay, outs, status, ins):
    size = eval_sizes(s)
    o = {k: (size[k], np.float64) for k in outs}
    if status:
        o["status"] = (1, np.int32)
    i = {k: data[k][:B] for k in ins}

    def fn(B, ptr):
        io = EvalIO(*[ptr.get(k) for k in EVAL_IN + EVAL_OUT], ptr.get("status"))
        return s.lib.landing_eval_batch(s.ctx, B, mem, lay, ctypes.byref(io))

    return call(s, mem, lay, B, i, o, fn)


@pytest.mark.parametrize("case", range(len(EVAL_CASES)))
def test_eval_batch(s, data, case):
    outs, status, ins, direct, via_soa = EVAL_CASES[case]
    npar = s.dims["np"]
    # the shared scalar parameters mu, mass, Ib, Ib_inv (the last ten entries of p bar l_leg_max, f_max) are summed
    # over the knots with atomics
    atomic = {"grad_p": [npar - 10] + list(range(npar - 7, npar))}

    def run(B, mem, lay):
        out, n = eval_call(s, data, B, mem, lay, outs, status, ins)
        return out, n, via_soa if (lay == AOS and B >= 64) else direct

    run_matrix(run, atomic=atomic)


# ---------------------------------------------------------------- landing_bounds_batch / landing_build_batch
def test_bounds_batch(s, data):
    m = s.dims["m"]

    def run(B, mem, lay):
        out, n = call(s, mem, lay, B, {"p": data["p"][:B]}, {"lbg": (m, np.float64), "ubg": (m, np.float64)},
                      lambda B, q: s.lib.landing_bounds_batch(s.ctx, B, mem, lay, q["p"], q["lbg"], q["ubg"]))
        return out, n, 1

    run_matrix(run)


@pytest.mark.parametrize("outs", [("p", "x0"), ("p",), ("x0",)])
def test_build_batch(s, data, outs):
    d = s.dims
    size = dict(p=d["np"], x0=d["nx"])

    def run(B, mem, lay):
        def fn(B, q):
            return s.lib.landing_build_batch(s.ctx, B, mem, lay, ctypes.byref(s.problem), q["drops"], q.get("p"),
                                             q.get("x0"))
        # drops is AoS whatever the layout
        out, n = call(s, mem, lay, B, {"drops": data["drops"][:B]}, {k: (size[k], np.float64) for k in outs}, fn,
                      aos_only=("drops",))
        return out, n, 1

    run_matrix(run)


# ---------------------------------------------------------------- landing_solve_batch
def solve_call(s, data, B, mem, x0, lam, viol):
    d = s.dims
    o = {"x_star": (d["nx"], np.float64), "f_star": (1, np.float64), "status": (1, np.int32),
         "iters": (1, np.int32)}
    if lam:
        o["lam_g"] = (d["m"], np.float64)
    if viol:
        o["viol"] = (1, np.float64)

    def fn(B, q):
        io = SolveIO(q["drops"], q.get("x0"), q["x_star"], q["f_star"], q.get("lam_g"), q.get("viol"), q["status"],
                     q["iters"])
        return s.lib.landing_solve_batch(s.ctx, B, mem, ctypes.byref(s.problem), ctypes.byref(s.options),
                                         ctypes.byref(io))

    return call(s, mem, AOS, B, {"drops": data["drops"][:B], "x0": data["x0"][:B] if x0 else None}, o, fn)


@pytest.mark.parametrize("x0", [False, True])
@pytest.mark.parametrize("lam", [False, True])
@pytest.mark.parametrize("viol", [False, True])
def test_solve_batch(s, data, x0, lam, viol):
    def run(B, mem, lay):
        out, n = solve_call(s, data, B, mem, x0, lam, viol)
        return out, n, 2 if B == 1 else 3  # k_kinds + k_solve, and the work-queue order when B > 1

    run_matrix(run, layouts=(AOS,))


# ---------------------------------------------------------------- landing_tvlqr_batch
@pytest.mark.parametrize("want_K", [False, True])
def test_tvlqr_batch(s, data, want_K):
    par = s.tvlqr_default()
    ns = par.n_steps
    o = {"P": (576 * ns, np.float64)}
    if want_K:
        o["K"] = (288 * ns, np.float64)

    def run(B, mem, lay):
        out, n = call(s, mem, AOS, B, {"x": data["x_star"][:B]}, o,
                      lambda B, q: s.lib.landing_tvlqr_batch(s.ctx, B, mem, ctypes.byref(par), q["x"], q["P"],
                                                             q.get("K")))
        return out, n, 1

    run_matrix(run, layouts=(AOS,))


# ---------------------------------------------------------------- kino-dynamic NLP
@pytest.fixture(scope="module")
def kpb(s):
    return s.kino_problem(lc.SWEEP_DT)  # non-uniform knot spacings of the sweep callers (N = 21)


# (outputs, launches when the kernels read the caller's layout, launches for an AoS batch with B >= 64)
KINO_EVAL_CASES = [(("g",), 1, 3), (("jac",), 8, 10), (("g", "jac"), 9, 12)]


@pytest.mark.parametrize("case", range(len(KINO_EVAL_CASES)))
def test_kino_eval_batch(s, data, kpb, case):
    outs, direct, via_soa = KINO_EVAL_CASES[case]
    kd = s.kino_dims()
    size = dict(g=kd["m"], jac=kd["nnzJ"])

    def run(B, mem, lay):
        out, n = call(s, mem, lay, B, {"x": data["kx"][:B]}, {k: (size[k], np.float64) for k in outs},
                      lambda B, q: s.lib.landing_kino_eval_batch(s.ctx, B, mem, lay, ctypes.byref(kpb), q["x"],
                                                                 q.get("g"), q.get("jac")))
        return out, n, via_soa if (lay == AOS and B >= 64) else direct

    run_matrix(run)


@pytest.mark.parametrize("outs", [("lbg",), ("ubg",), ("x0",), ("lbg", "ubg"), ("lbg", "ubg", "x0")])
@pytest.mark.parametrize("with_srb", [False, True])
def test_kino_setup_batch(s, data, outs, with_srb):
    kd = s.kino_dims()
    size = dict(lbg=kd["m"], ubg=kd["m"], x0=kd["nx"])
    ks = s.kino_setup_data()

    def run(B, mem, lay):
        ins = {"drops": data["drops"][:B], "x_srb": data["x_star"][:B] if with_srb else None}
        out, n = call(s, mem, lay, B, ins, {k: (size[k], np.float64) for k in outs},
                      lambda B, q: s.lib.landing_kino_setup_batch(s.ctx, B, mem, lay, ctypes.byref(ks), q["drops"],
                                                                  q.get("x_srb"), q.get("lbg"), q.get("ubg"),
                                                                  q.get("x0")))
        return out, n, 1

    run_matrix(run)


@pytest.mark.parametrize("outs", [("f",), ("grad_f",), ("f", "grad_f")])
def test_kino_cost_batch(s, data, outs):
    kd = s.kino_dims()
    size = dict(f=1, grad_f=kd["nx"])
    ks = s.kino_setup_data()

    def run(B, mem, lay):
        out, n = call(s, mem, lay, B, {"x": data["kx"][:B]}, {k: (size[k], np.float64) for k in outs},
                      lambda B, q: s.lib.landing_kino_cost_batch(s.ctx, B, mem, lay, ctypes.byref(ks), q["x"],
                                                                 q.get("f"), q.get("grad_f")))
        return out, n, 1

    run_matrix(run)


# ---------------------------------------------------------------- buffer reuse, refused calls, LANDING_NO_ZEROCOPY
def test_large_small_large_on_one_context(data):
    """The grow-only buffers of one context serve a large, a small and again a large call: each gives the bits of the
    same call on a fresh context."""
    outs = ("f", "g", "grad_f", "jac", "hess")
    ins = EVAL_IN

    def fresh(fn):
        t = lc.LandingSolver(N=N, device=0)
        t.options.max_iter = MAX_ITER
        try:
            return fn(t)
        finally:
            t.close()

    reused = lc.LandingSolver(N=N, device=0)
    reused.options.max_iter = MAX_ITER
    try:
        for B in (BMAX, 1, BMAX, 3, BMAX):
            for mem in (HOST, DEVICE):
                got, _ = eval_call(reused, data, B, mem, AOS, outs, True, ins)
                want, _ = fresh(lambda t: eval_call(t, data, B, mem, AOS, outs, True, ins))
                check_same([("fresh", want), (("reused", B, mem), got)])
                got, _ = solve_call(reused, data, B, mem, True, True, True)
                want, _ = fresh(lambda t: solve_call(t, data, B, mem, True, True, True))
                check_same([("fresh", want), (("reused", B, mem), got)])
    finally:
        reused.close()


def test_refused_calls_then_a_good_call(s, data):
    lib, ctx = s.lib, s.ctx
    want, _ = solve_call(s, data, 8, HOST, False, True, True)
    want_eval, _ = eval_call(s, data, 8, HOST, AOS, ("g", "jac"), True, ("x", "p"))

    def refused(rc_want, msg, fn):
        before = s.launches
        assert fn() == rc_want
        assert lib.landing_last_error().decode() == msg
        assert s.launches == before

    B = 8
    d = s.dims
    drops = np.ascontiguousarray(data["drops"][:B])
    x = np.zeros((B, d["nx"]))
    f = np.zeros(B)
    st, it = np.zeros(B, np.int32), np.zeros(B, np.int32)
    io = SolveIO(_ptr(drops), None, None, _ptr(f), None, None, _ptr(st, _ip), _ptr(it, _ip))
    refused(1, "landing_solve_batch: x_star, f_star, status and iters are required",
            lambda: lib.landing_solve_batch(ctx, B, HOST, ctypes.byref(s.problem), ctypes.byref(s.options),
                                            ctypes.byref(io)))
    io = SolveIO(None, None, _ptr(x), _ptr(f), None, None, _ptr(st, _ip), _ptr(it, _ip))
    refused(1, "landing_solve_batch: drops is NULL",
            lambda: lib.landing_solve_batch(ctx, B, HOST, ctypes.byref(s.problem), ctypes.byref(s.options),
                                            ctypes.byref(io)))
    refused(1, "landing_eval_batch: bad arguments",
            lambda: lib.landing_eval_batch(ctx, -1, HOST, AOS, ctypes.byref(EvalIO())))
    p = np.zeros((B, d["np"]))
    lb, ub = np.zeros((B, d["m"])), np.zeros((B, d["m"]))
    refused(1, "landing_bounds_batch: bad arguments",
            lambda: lib.landing_bounds_batch(ctx, 0, HOST, AOS, _ptr(p), _ptr(lb), _ptr(ub)))
    refused(1, "landing_build_batch: bad arguments",
            lambda: lib.landing_build_batch(ctx, 0, HOST, AOS, ctypes.byref(s.problem), _ptr(drops), _ptr(p), None))
    bad = lc.api.Problem.from_buffer_copy(s.problem)
    bad.formulation = 2
    refused(1, "landing_problem: formulation must be 0 or 1",
            lambda: lib.landing_build_batch(ctx, B, HOST, AOS, ctypes.byref(bad), _ptr(drops), _ptr(p), None))
    neg = np.full(N - 1, -0.03)
    bad.formulation = 0
    bad.dt = neg.ctypes.data_as(lc.api._dp)
    refused(1, "landing_problem: knot spacings must be positive",
            lambda: lib.landing_solve_batch(ctx, B, HOST, ctypes.byref(bad), ctypes.byref(s.options),
                                            ctypes.byref(SolveIO(_ptr(drops), None, _ptr(x), _ptr(f), None, None,
                                                                 _ptr(st, _ip), _ptr(it, _ip)))))
    kpb = s.kino_problem(neg)
    kx = np.zeros((B, s.kino_dims()["nx"]))
    g = np.zeros((B, s.kino_dims()["m"]))
    refused(1, "landing_problem: knot spacings must be positive",
            lambda: lib.landing_kino_eval_batch(ctx, B, HOST, AOS, ctypes.byref(kpb), _ptr(kx), _ptr(g), None))
    refused(1, "landing_tvlqr_batch: bad arguments",
            lambda: lib.landing_tvlqr_batch(ctx, B, HOST, None, _ptr(x), None, None))
    # empty batches are no-ops where the ABI allows them
    for fn in (lambda: lib.landing_eval_batch(ctx, 0, HOST, AOS, ctypes.byref(EvalIO())),
               lambda: lib.landing_solve_batch(ctx, 0, HOST, ctypes.byref(s.problem), None, ctypes.byref(SolveIO()))):
        before = s.launches
        assert fn() == 0 and s.launches == before
    got, _ = solve_call(s, data, 8, HOST, False, True, True)
    check_same([("before", want), ("after", got)])
    got, _ = eval_call(s, data, 8, HOST, AOS, ("g", "jac"), True, ("x", "p"))
    check_same([("before", want_eval), ("after", got)])


NO_ZC_SCRIPT = r"""
import sys
sys.path.insert(0, sys.argv[1])
sys.path.insert(0, sys.argv[1] + "/tests")
import numpy as np
import landing_controller_b200 as lc
import test_host_staging as t
data = dict(np.load(sys.argv[2]))
s = lc.LandingSolver(N=t.N, device=0)
out = {}
for B in t.NO_ZC_SIZES:
    for j, (outs, ins) in enumerate(t.NO_ZC_CASES):
        r, n = t.eval_call(s, data, B, lc.HOST, lc.AOS, outs, True, ins)
        out.update({"%d_%d_%s" % (B, j, k): a for k, a in r.items()})
        out["%d_%d_launches" % (B, j)] = np.array(n)
np.savez(sys.argv[3], **out)
"""
NO_ZC_SIZES = (1, 3)  # all outputs but grad_x / grad_p of B = 3 fit the 512 KB of the zero-copy path
NO_ZC_CASES = [(("g", "jac"), ("x", "p")), (("hess",), EVAL_IN), (("f", "g", "grad_f", "jac", "hess"), EVAL_IN),
               ((), ("x", "p"))]


def test_staged_copies_under_no_zerocopy_give_the_zero_copy_bits(s, data, tmp_path):
    """LANDING_NO_ZEROCOPY=1 (read once per process) makes small host evaluations use the staged copies."""
    if os.environ.get("LANDING_NO_ZEROCOPY"):
        pytest.skip("this process already runs without zero-copy")
    inp, res = tmp_path / "in.npz", tmp_path / "out.npz"
    np.savez(inp, **{k: data[k][:max(NO_ZC_SIZES)] for k in EVAL_IN})
    env = dict(os.environ, LANDING_NO_ZEROCOPY="1")
    subprocess.run([sys.executable, "-c", NO_ZC_SCRIPT, ROOT, str(inp), str(res)], env=env, check=True, timeout=600)
    staged = np.load(res)
    for B in NO_ZC_SIZES:
        for j, (outs, ins) in enumerate(NO_ZC_CASES):
            r, n = eval_call(s, data, B, HOST, AOS, outs, True, ins)
            assert int(staged["%d_%d_launches" % (B, j)]) == n
            for k, a in r.items():
                assert np.array_equal(staged["%d_%d_%s" % (B, j, k)], a), (B, outs, k)
