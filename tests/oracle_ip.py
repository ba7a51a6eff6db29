"""ctypes binding of the CPU interior-point reference (oracle/ip_ref.c). TEST INFRASTRUCTURE."""
import ctypes
import os

import numpy as np

from oracle_lib import Problem, _dp, build_oracle


class IpOptions(ctypes.Structure):
    _fields_ = [("max_iter", ctypes.c_int), ("tol", ctypes.c_double), ("constr_viol_tol", ctypes.c_double),
                ("dual_inf_tol", ctypes.c_double), ("compl_inf_tol", ctypes.c_double),
                ("mu_init", ctypes.c_double), ("bound_push", ctypes.c_double), ("bound_frac", ctypes.c_double),
                ("bound_relax_factor", ctypes.c_double), ("max_soc", ctypes.c_int), ("verbose", ctypes.c_int),
                ("jam_alpha", ctypes.c_double), ("jam_iters", ctypes.c_int), ("max_restarts", ctypes.c_int),
                ("run_Qf", ctypes.c_double * 3), ("kin_box", ctypes.c_double * 3),
                ("formulation", ctypes.c_int), ("cs", ctypes.POINTER(ctypes.c_int)), ("QX", ctypes.c_double * 12),
                ("delta_c", ctypes.c_double), ("acceptable_tol", ctypes.c_double), ("acceptable_iter", ctypes.c_int),
                ("restart_mu", ctypes.c_double)]

    def set_schedule(self, cs, QX):
        """fixed-contact-schedule formulation: cs [N-1, 4] of 0/1 (kept alive), running state weights QX [12]"""
        self._cs = np.ascontiguousarray(cs, dtype=np.int32)
        self.cs = self._cs.ctypes.data_as(ctypes.POINTER(ctypes.c_int))
        self.formulation = 1
        for i in range(12):
            self.QX[i] = QX[i]
        return self


class IpResult(ctypes.Structure):
    _fields_ = [("status", ctypes.c_int), ("iters", ctypes.c_int), ("n_factor", ctypes.c_int),
                ("f", ctypes.c_double), ("viol", ctypes.c_double), ("dual_inf", ctypes.c_double),
                ("compl_inf", ctypes.c_double), ("mu", ctypes.c_double), ("restarts", ctypes.c_int)]


_FAST = {}


def _lib(fast=False):
    if fast:
        if "lib" not in _FAST:
            from oracle_lib import build_oracle_fast
            path, how = build_oracle_fast()
            _FAST["lib"], _FAST["how"] = ctypes.CDLL(path), how
        return _FAST["lib"]
    lib = ctypes.CDLL(build_oracle())
    return lib


def fast_build_flags():
    _lib(fast=True)
    return _FAST["how"]


def default_options(**kw):
    o = IpOptions()
    _lib().ip_options_default(ctypes.byref(o))
    for k, v in kw.items():
        if k in ("run_Qf", "kin_box", "QX"):
            for i in range(len(v)):
                getattr(o, k)[i] = v[i]
        else:
            setattr(o, k, v)
    return o


def default_problem(**kw):
    pb = Problem()
    _lib().srb_problem_default(ctypes.byref(pb))
    for k, v in kw.items():
        setattr(pb, k, v)
    return pb


def solve_cpu(N, drops, opt=None, pb=None, threads=0, fast=False, want_lam=False):
    """drops [B,12] -> dict(x [B,nx], status, iters, f, viol, n_factor).  fast: the -O3 -march=native build (timing only).
    want_lam: also lam_g [B,m]; the scenarios then go one at a time through ip_solve (which returns the multipliers) on
    a pool of host threads, from the same initial guess as ip_solve_batch."""
    lib = _lib(fast)
    drops = np.ascontiguousarray(drops, dtype=np.float64)
    B = drops.shape[0]
    nx = 36 * N - 24
    opt = opt or default_options()
    pb = pb or default_problem()
    x = np.zeros((B, nx))
    res = (IpResult * B)()
    threads = min(threads or (os.cpu_count() or 1), max(B, 1))
    out = {}
    if want_lam:
        from concurrent.futures import ThreadPoolExecutor
        from oracle_lib import Oracle
        o = Oracle(N)
        lam = np.zeros((B, o.m))

        def one(b):  # (ctypes releases the GIL during the call)
            p, x0 = o.build_p_x0(pb, drops[b, :6], drops[b, 6:])
            lib.ip_solve(o.plan, _dp(p), _dp(x0), ctypes.byref(opt), _dp(x[b]), _dp(lam[b]), ctypes.byref(res[b]))

        with ThreadPoolExecutor(threads) as ex:
            list(ex.map(one, range(B)))
        out["lam_g"] = lam
    else:
        rc = lib.ip_solve_batch(N, B, _dp(drops), ctypes.byref(pb), ctypes.byref(opt), _dp(x), res, threads)
        assert rc == 0
    out.update(x=x, status=np.array([r.status for r in res]), iters=np.array([r.iters for r in res]),
               f=np.array([r.f for r in res]), viol=np.array([r.viol for r in res]),
               n_factor=np.array([r.n_factor for r in res]), mu=np.array([r.mu for r in res]),
               dual_inf=np.array([r.dual_inf for r in res]), compl_inf=np.array([r.compl_inf for r in res]),
               restarts=np.array([r.restarts for r in res]))
    return out


def solve_cpu_x0(N, drops, x0, opt=None, pb=None):
    """Like solve_cpu, but from the caller's initial guess x0 [B,nx] (the `_ws` flavour of the reference is called with a
    previous solution: generate_landingCtrller_IPOPT_warmstart.m:227-230). One scenario at a time through ip_solve."""
    from oracle_lib import Oracle
    lib = _lib()
    o = Oracle(N)
    opt = opt or default_options()
    pb = pb or default_problem()
    drops = np.ascontiguousarray(drops, dtype=np.float64)
    x0 = np.ascontiguousarray(x0, dtype=np.float64)
    B, nx = drops.shape[0], 36 * N - 24
    x = np.zeros((B, nx))
    res = (IpResult * B)()
    for b in range(B):
        p, _ = o.build_p_x0(pb, drops[b, :6], drops[b, 6:])
        p = np.ascontiguousarray(p)
        lib.ip_solve(o.plan, _dp(p), _dp(x0[b]), ctypes.byref(opt), _dp(x[b]), None, ctypes.byref(res[b]))  # returns the status
    return dict(x=x, status=np.array([r.status for r in res]), iters=np.array([r.iters for r in res]),
                f=np.array([r.f for r in res]), viol=np.array([r.viol for r in res]))
