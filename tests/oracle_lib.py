"""ctypes bindings for the CPU oracle (oracle/liboracle.so) and, when it has been built,
the compiled reference C (oracle/_ref/landingCtrller_IPOPT.so).

TEST INFRASTRUCTURE: imported only by tests/, bench.py's cpu_baseline/reference legs and
__graft_entry__.smoke().  The product package never imports this module.
"""
import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_SO = os.path.join(ORACLE_DIR, "liboracle.so")
REF_SO = os.path.join(ORACLE_DIR, "_ref", "landingCtrller_IPOPT.so")

c_dp = ctypes.POINTER(ctypes.c_double)
c_llp = ctypes.POINTER(ctypes.c_longlong)


def _dp(a):
    return None if a is None else a.ctypes.data_as(c_dp)


def build_oracle(force=False):
    srcs = [os.path.join(ORACLE_DIR, f) for f in os.listdir(ORACLE_DIR) if f.endswith((".c", ".h"))]
    if force or not os.path.exists(ORACLE_SO) or any(
            os.path.getmtime(s) > os.path.getmtime(ORACLE_SO) for s in srcs):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "liboracle.so"], stdout=subprocess.DEVNULL)
    return ORACLE_SO


def build_oracle_fast():
    """The -O3 -march=native build used by the TIMED CPU arm of bench.py (never by the parity tests): always rebuilt on
    the host that runs the bench, because -march=native code from another machine may not run here.  It goes to a
    temporary directory (removed at exit), so that the bench writes nothing into the checkout, which may be read-only.
    When that build fails, falls back to the bit-reproducible build and says so, with the error, in the returned label."""
    try:
        tmp = tempfile.mkdtemp(prefix="landing_oracle_")
        atexit.register(shutil.rmtree, tmp, True)
        fast_so = os.path.join(tmp, "liboracle_fast.so")
        subprocess.run(["make", "-C", ORACLE_DIR, "fast", "FAST_SO=" + fast_so], check=True, capture_output=True,
                       text=True)
        return fast_so, "gcc -O3 -march=native -fopenmp (built on this host)"
    except (OSError, subprocess.CalledProcessError) as e:
        why = (getattr(e, "stderr", None) or "").strip().splitlines() or [str(e)]
        return build_oracle(), "gcc -O2 -ffp-contract=off -fopenmp (the -O3 build failed: %s)" % why[-1]


class Plan(ctypes.Structure):
    _fields_ = [("N", ctypes.c_int), ("nx", ctypes.c_int), ("np", ctypes.c_int), ("m", ctypes.c_int),
                ("nnzJ", ctypes.c_int), ("nnzH", ctypes.c_int),
                ("spJ", c_llp), ("spH", c_llp),
                ("jmap", ctypes.POINTER(ctypes.c_int)), ("hmap", ctypes.POINTER(ctypes.c_int)),
                ("jbnd", ctypes.c_int * 36), ("hterm", ctypes.c_int * 12),
                ("o_dt", ctypes.c_int), ("o_qmin", ctypes.c_int), ("o_qmax", ctypes.c_int),
                ("o_qdmin", ctypes.c_int), ("o_qdmax", ctypes.c_int), ("o_qinit", ctypes.c_int),
                ("o_qdinit", ctypes.c_int), ("o_qtmin", ctypes.c_int), ("o_qtmax", ctypes.c_int),
                ("o_qdtmin", ctypes.c_int), ("o_qdtmax", ctypes.c_int), ("o_QN", ctypes.c_int),
                ("o_mu", ctypes.c_int), ("o_lleg", ctypes.c_int), ("o_fmax", ctypes.c_int),
                ("o_mass", ctypes.c_int), ("o_Ib", ctypes.c_int), ("o_Ibinv", ctypes.c_int)]


class Problem(ctypes.Structure):
    _fields_ = [("T", ctypes.c_double)] + [(n, ctypes.c_double * 6) for n in (
        "q_min", "q_max", "qd_min", "qd_max", "q_term_min", "q_term_max", "qd_term_min",
        "qd_term_max", "q_term_ref", "qd_term_ref")] + [
        ("c_ref", ctypes.c_double * 12), ("QN", ctypes.c_double * 12),
        ("mu", ctypes.c_double), ("l_leg_max", ctypes.c_double), ("f_max", ctypes.c_double),
        ("mass", ctypes.c_double), ("Ib", ctypes.c_double * 3), ("Ib_inv", ctypes.c_double * 3),
        ("dt", c_dp)]

    def set_dt(self, dt):
        """knot spacings (keeps the array alive); None = uniform"""
        if dt is None:
            self._dt, self.dt = None, None
        else:
            self._dt = np.ascontiguousarray(dt, dtype=np.float64)
            self.dt = self._dt.ctypes.data_as(c_dp)
            self.T = float(self._dt.sum())
        return self


class Oracle:
    """Generic-N CPU restatement (oracle/srb_ref.c)."""

    def __init__(self, N):
        self.lib = ctypes.CDLL(build_oracle())
        L = self.lib
        L.srb_plan_create.restype = ctypes.POINTER(Plan)
        L.srb_plan_create.argtypes = [ctypes.c_int]
        L.srb_plan_free.argtypes = [ctypes.POINTER(Plan)]
        self.plan = L.srb_plan_create(N)
        pl = self.plan.contents
        self.N, self.nx, self.np_, self.m = pl.N, pl.nx, pl.np, pl.m
        self.nnzJ, self.nnzH = pl.nnzJ, pl.nnzH
        self.spJ = np.ctypeslib.as_array(pl.spJ, shape=(2 + self.nx + 1 + self.nnzJ,)).copy()
        self.spH = np.ctypeslib.as_array(pl.spH, shape=(2 + self.nx + 1 + self.nnzH,)).copy()
        self.off = {n: getattr(pl, n) for n, _ in Plan._fields_ if n.startswith("o_")}

    def __del__(self):
        try:
            self.lib.srb_plan_free(self.plan)
        except Exception:
            pass

    def f(self, x, p):
        f = np.zeros(1)
        rc = self.lib.srb_f(self.plan, _dp(x), _dp(p), _dp(f))
        return rc, f[0]

    def g(self, x, p):
        g = np.zeros(self.m)
        rc = self.lib.srb_g(self.plan, _dp(x), _dp(p), _dp(g))
        return rc, g

    def grad_f(self, x, p):
        f = np.zeros(1)
        gr = np.zeros(self.nx)
        rc = self.lib.srb_grad_f(self.plan, _dp(x), _dp(p), _dp(f), _dp(gr))
        return rc, f[0], gr

    def jac_g(self, x, p):
        g = np.zeros(self.m)
        J = np.zeros(self.nnzJ)
        rc = self.lib.srb_jac_g(self.plan, _dp(x), _dp(p), _dp(g), _dp(J))
        return rc, g, J

    def hess_l(self, x, p, lam_f, lam_g):
        H = np.zeros(self.nnzH)
        rc = self.lib.srb_hess_l(self.plan, _dp(x), _dp(p), ctypes.c_double(lam_f), _dp(lam_g), _dp(H))
        return rc, H

    def grad(self, x, p, lam_f, lam_g):
        f = np.zeros(1)
        g = np.zeros(self.m)
        gx = np.zeros(self.nx)
        gp = np.zeros(self.np_)
        rc = self.lib.srb_grad(self.plan, _dp(x), _dp(p), ctypes.c_double(lam_f), _dp(lam_g),
                               _dp(f), _dp(g), _dp(gx), _dp(gp))
        return rc, f[0], g, gx, gp

    def bounds(self, p):
        lb = np.zeros(self.m)
        ub = np.zeros(self.m)
        self.lib.srb_bounds(self.plan, _dp(p), _dp(lb), _dp(ub))
        return lb, ub

    def default_problem(self):
        pb = Problem()
        self.lib.srb_problem_default(ctypes.byref(pb))
        return pb

    def build_p_x0(self, pb, q_init, qd_init):
        p = np.zeros(self.np_)
        x0 = np.zeros(self.nx)
        qi = np.ascontiguousarray(q_init, dtype=np.float64)
        qd = np.ascontiguousarray(qd_init, dtype=np.float64)
        self.lib.srb_build_p_x0(self.plan, ctypes.byref(pb), _dp(qi), _dp(qd), _dp(p), _dp(x0))
        return p, x0


class CasadiLib:
    """Any shared library exporting the CasADi-generated symbol set of landingCtrller_IPOPT.c
    (the compiled reference, or the product's drop-in library)."""
    FUNCS = ("nlp", "nlp_f", "nlp_g", "nlp_grad", "nlp_grad_f", "nlp_hess_l", "nlp_jac_g")

    def __init__(self, path):
        self.lib = ctypes.CDLL(path)
        for fn in self.FUNCS:
            for suf, res, args in (("_n_in", ctypes.c_longlong, []), ("_n_out", ctypes.c_longlong, []),
                                   ("_sparsity_in", c_llp, [ctypes.c_longlong]),
                                   ("_sparsity_out", c_llp, [ctypes.c_longlong]),
                                   ("_name_in", ctypes.c_char_p, [ctypes.c_longlong]),
                                   ("_name_out", ctypes.c_char_p, [ctypes.c_longlong]),
                                   ("_default_in", ctypes.c_double, [ctypes.c_longlong])):
                h = getattr(self.lib, fn + suf)
                h.restype = res
                h.argtypes = args
            getattr(self.lib, fn).restype = ctypes.c_int

    def sparsity(self, fn, i, out=True):
        s = getattr(self.lib, fn + ("_sparsity_out" if out else "_sparsity_in"))(i)
        nrow, ncol = s[0], s[1]
        nnz = s[2 + ncol]
        return np.array([s[j] for j in range(2 + ncol + 1 + nnz)], dtype=np.int64)

    def nnz_out(self, fn, i):
        s = getattr(self.lib, fn + "_sparsity_out")(i)
        return s[2 + s[1]]

    def call(self, fn, args, skip=(), mem=0):
        """args: list of arrays (or None).  Returns (rc, [outputs]).  mem: memory object from F_checkout."""
        n_in = getattr(self.lib, fn + "_n_in")()
        n_out = getattr(self.lib, fn + "_n_out")()
        assert len(args) == n_in
        keep = [None if a is None else np.ascontiguousarray(a, dtype=np.float64).ravel() for a in args]
        argv = (c_dp * n_in)(*[_dp(a) for a in keep])
        outs = [None if i in skip else np.zeros(self.nnz_out(fn, i)) for i in range(n_out)]
        resv = (c_dp * n_out)(*[_dp(o) for o in outs])
        szs = [ctypes.c_longlong() for _ in range(4)]
        getattr(self.lib, fn + "_work")(*[ctypes.byref(s) for s in szs])
        iw = (ctypes.c_longlong * max(1, szs[2].value))()
        w = (ctypes.c_double * max(1, szs[3].value))()
        rc = getattr(self.lib, fn)(argv, resv, iw, w, mem)
        return rc, outs


def have_ref():
    return os.path.exists(REF_SO)
