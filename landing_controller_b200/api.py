"""Host-side Python mirror of the reference's solver interface for the landing hot path.

The reference's callers (MATLAB) do

    f = Function.load('landingCtrller_IPOPT.casadi')
    [x, cost] = f(Xref, Uref, dt, q_min, ..., x0, mu, l_leg_max, f_max, mass, Ib, Ib_inv)

(optimizations/landing/main_scripts/landing_optimization.m:300-311,
 generate_data/generate_training_data_automated.m:130-136) one drop condition at a time.  Here
`LandingSolver.solve(drops)` does the same for a batch of drop conditions through the C ABI of
liblanding_b200.so (include/landing_b200.h).  PyTorch only provides device memory / streams.

There is no CPU path: if the CUDA library is missing or no GPU is present, construction fails.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblanding_b200.so")
DROPIN_PATH = os.path.join(_HERE, "dropin", "landingCtrller_IPOPT.so")

HOST, DEVICE = 0, 1
AOS, SOA = 0, 1

STATUS = {0: "converged", 1: "max_iter", 2: "linesearch_fail", 3: "nan", 4: "factor_fail", 9: "running"}

_dp = ctypes.POINTER(ctypes.c_double)
_ip = ctypes.POINTER(ctypes.c_int)


class EvalIO(ctypes.Structure):
    _fields_ = [(n, _dp) for n in ("x", "p", "lam_f", "lam_g", "f", "g", "grad_f", "jac", "hess",
                                   "grad_x", "grad_p")] + [("status", _ip)]


class Problem(ctypes.Structure):
    _fields_ = [("T", ctypes.c_double)] + [(n, ctypes.c_double * 6) for n in (
        "q_min", "q_max", "qd_min", "qd_max", "q_term_min", "q_term_max", "qd_term_min",
        "qd_term_max", "q_term_ref", "qd_term_ref")] + [
        ("c_ref", ctypes.c_double * 12), ("QN", ctypes.c_double * 12),
        ("mu", ctypes.c_double), ("l_leg_max", ctypes.c_double), ("f_max", ctypes.c_double),
        ("mass", ctypes.c_double), ("Ib", ctypes.c_double * 3), ("Ib_inv", ctypes.c_double * 3),
        ("Qf", ctypes.c_double * 3), ("kin_box", ctypes.c_double * 3), ("dt", _dp),
        ("formulation", ctypes.c_int), ("cs", _ip), ("QX", ctypes.c_double * 12), ("delta_c", ctypes.c_double)]


class Options(ctypes.Structure):
    _fields_ = [("max_iter", ctypes.c_int), ("tol", ctypes.c_double), ("constr_viol_tol", ctypes.c_double),
                ("dual_inf_tol", ctypes.c_double), ("compl_inf_tol", ctypes.c_double),
                ("mu_init", ctypes.c_double), ("bound_push", ctypes.c_double),
                ("bound_frac", ctypes.c_double), ("bound_relax_factor", ctypes.c_double),
                ("max_soc", ctypes.c_int), ("jam_iters", ctypes.c_int), ("jam_alpha", ctypes.c_double),
                ("max_restarts", ctypes.c_int), ("reserved", ctypes.c_int * 5), ("restart_mu", ctypes.c_double)]


class Tvlqr(ctypes.Structure):
    _fields_ = [("T", ctypes.c_double), ("dt", ctypes.c_double), ("n_steps", ctypes.c_int),
                ("Q", ctypes.c_double * 576), ("F", ctypes.c_double * 576), ("R", ctypes.c_double * 12),
                ("Ib", ctypes.c_double * 9), ("mass", ctypes.c_double)]


class KinoProblem(ctypes.Structure):
    """landing_kino_problem: shared numeric data of the kino-dynamic NLP (generate_landingCtrller_KNITRO.m:224-262)."""
    _fields_ = [("mu", ctypes.c_double), ("mass", ctypes.c_double), ("Ib", ctypes.c_double * 3),
                ("Ib_inv", ctypes.c_double * 3), ("dt", _dp)]


class KinoSetup(ctypes.Structure):
    """landing_kino_setup: bounds / initial-guess / cost data of the kino-dynamic NLP
    (generate_landingCtrller_KNITRO.m:214-262,325)."""
    _fields_ = [("q_term_min", ctypes.c_double * 6), ("q_term_max", ctypes.c_double * 6),
                ("qd_term_min", ctypes.c_double * 6), ("qd_term_max", ctypes.c_double * 6),
                ("z_min", ctypes.c_double), ("l_leg_max", ctypes.c_double),
                ("jpos_min", ctypes.c_double * 12), ("jpos_max", ctypes.c_double * 12), ("tau_max", ctypes.c_double * 3),
                ("QN", ctypes.c_double * 12), ("q_term_ref", ctypes.c_double * 6), ("qd_term_ref", ctypes.c_double * 6),
                ("jpos_guess", ctypes.c_double * 3)]


class SolveIO(ctypes.Structure):
    _fields_ = [("drops", _dp), ("x0", _dp), ("x_star", _dp), ("f_star", _dp), ("lam_g", _dp),
                ("viol", _dp), ("status", _ip), ("iters", _ip)]


def load_library(path=LIB_PATH):
    if not os.path.exists(path):
        raise RuntimeError(
            "landing_controller_b200: %s is missing -- build it with __graft_entry__.build() "
            "(there is no CPU fallback)" % path)
    lib = ctypes.CDLL(path)
    lib.landing_last_error.restype = ctypes.c_char_p
    lib.landing_sparsity_for.restype = ctypes.POINTER(ctypes.c_longlong)
    lib.landing_sparsity_for.argtypes = [ctypes.c_int, ctypes.c_int]
    lib.landing_create.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]
    lib.landing_destroy.argtypes = [ctypes.c_void_p]
    lib.landing_eval_batch.argtypes = [ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_int,
                                       ctypes.POINTER(EvalIO)]
    lib.landing_bounds_batch.argtypes = [ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_int,
                                         _dp, _dp, _dp]
    lib.landing_build_batch.argtypes = [ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_int,
                                        ctypes.POINTER(Problem), _dp, _dp, _dp]
    lib.landing_solve_batch.argtypes = [ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int,
                                        ctypes.POINTER(Problem), ctypes.POINTER(Options),
                                        ctypes.POINTER(SolveIO)]
    if hasattr(lib, "landing_kino_eval_batch"):
        lib.landing_kino_dims.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_longlong)]
        lib.landing_kino_sparsity.restype = ctypes.POINTER(ctypes.c_longlong)
        lib.landing_kino_sparsity.argtypes = [ctypes.c_int]
        lib.landing_kino_eval_batch.argtypes = [ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_int,
                                                ctypes.POINTER(KinoProblem), _dp, _dp, _dp]
    if hasattr(lib, "landing_kino_setup_batch"):
        lib.landing_kino_setup_default.argtypes = [ctypes.POINTER(KinoSetup)]
        lib.landing_kino_setup_default.restype = None
        lib.landing_kino_setup_batch.argtypes = [ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_int,
                                                 ctypes.POINTER(KinoSetup), _dp, _dp, _dp, _dp, _dp]
        lib.landing_kino_cost_batch.argtypes = [ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_int,
                                                ctypes.POINTER(KinoSetup), _dp, _dp, _dp]
    if hasattr(lib, "landing_kino_hess_batch"):
        lib.landing_kino_hess_sparsity.restype = ctypes.POINTER(ctypes.c_longlong)
        lib.landing_kino_hess_sparsity.argtypes = [ctypes.c_int]
        lib.landing_kino_hess_batch.argtypes = [ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_int,
                                                ctypes.POINTER(KinoProblem), ctypes.POINTER(KinoSetup), _dp, _dp, _dp,
                                                _dp]
    lib.landing_launch_count.restype = ctypes.c_longlong
    lib.landing_launch_count.argtypes = [ctypes.c_void_p]
    if hasattr(lib, "landing_fp64_peak"):
        lib.landing_fp64_peak.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_double)]
    lib.landing_stream.restype = ctypes.c_void_p
    lib.landing_stream.argtypes = [ctypes.c_void_p]
    lib.landing_dims_for.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_longlong)]
    lib.landing_problem_default.argtypes = [ctypes.POINTER(Problem)]
    lib.landing_problem_default.restype = None
    lib.landing_options_default.argtypes = [ctypes.POINTER(Options)]
    lib.landing_options_default.restype = None
    lib.landing_tvlqr_default.argtypes = [ctypes.POINTER(Tvlqr)]
    lib.landing_tvlqr_default.restype = None
    lib.landing_tvlqr_batch.argtypes = [ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.POINTER(Tvlqr),
                                        _dp, _dp, _dp]
    lib.landing_synchronize.argtypes = [ctypes.c_void_p]
    lib.landing_multi_create.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int),
                                         ctypes.POINTER(ctypes.c_void_p)]
    lib.landing_multi_destroy.argtypes = [ctypes.c_void_p]
    lib.landing_solve_batch_multi.argtypes = [ctypes.c_void_p, ctypes.c_longlong, ctypes.POINTER(Problem),
                                              ctypes.POINTER(Options), ctypes.POINTER(SolveIO)]
    return lib


def dims_for(N, lib=None):
    lib = lib or load_library()
    d = (ctypes.c_longlong * 6)()
    if lib.landing_dims_for(N, d) != 0:
        raise ValueError(lib.landing_last_error().decode())
    return dict(N=d[0], nx=d[1], np=d[2], m=d[3], nnzJ=d[4], nnzH=d[5])


def sparsity_for(N, which, lib=None):
    """CasADi CCS array of which = 0 jac_g, 1 hess_l (upper), 2 x, 3 p, 4 scalar, 5 g. No GPU needed."""
    lib = lib or load_library()
    s = lib.landing_sparsity_for(N, which)
    if not s:
        raise ValueError("landing_sparsity_for(N=%d, which=%d): need N >= 3 and which in 0..5" % (N, which))
    ncol = s[1]
    nnz = s[2 + ncol]
    return np.ctypeslib.as_array(s, shape=(2 + ncol + 1 + nnz,)).copy()


def _ptr(a, typ=_dp):
    """numpy array (host) or torch tensor (host/device) -> C pointer."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        assert a.flags["C_CONTIGUOUS"]
        return a.ctypes.data_as(typ)
    assert a.is_contiguous()
    return ctypes.cast(a.data_ptr(), typ)


class LandingSolver:
    """Batched GPU solver / evaluator for the N-knot SRB landing NLP."""

    def __init__(self, N=21, device=0, lib_path=LIB_PATH):
        self.lib = load_library(lib_path)
        self.ctx = ctypes.c_void_p()
        rc = self.lib.landing_create(N, device, ctypes.byref(self.ctx))
        if rc != 0:
            raise RuntimeError("landing_create failed (%d): %s" % (rc, self.lib.landing_last_error().decode()))
        self.N, self.device = N, device
        self.dims = dims_for(N, self.lib)
        self.problem = Problem()
        self.lib.landing_problem_default(ctypes.byref(self.problem))
        self.options = Options()
        self.lib.landing_options_default(ctypes.byref(self.options))

    def set_dt(self, dt=None):
        """Knot spacings dt[0..N-2] (non-uniform grids of the reference's sweep / MPC callers,
        generate_training_data_automated.m:28), or None for the uniform T/(N-1).  Also sets T = sum(dt)."""
        if dt is None:
            self._dt = None
            self.problem.dt = None
            return self
        dt = np.ascontiguousarray(dt, dtype=np.float64)
        if dt.shape != (self.N - 1,):
            raise ValueError("dt must have N-1 = %d entries" % (self.N - 1))
        self._dt = dt  # keeps the host array alive: the library reads it during each call
        self.problem.dt = dt.ctypes.data_as(_dp)
        self.problem.T = float(dt.sum())
        return self

    def set_schedule(self, cs=None, QX=None):
        """Fixed-contact-schedule formulation (quadruped_SRBM_NLP.m; BASELINE configs[0]): cs [N-1, 4] of 0 / 1 and the
        running state weights QX [12]; None switches back to the contact-implicit formulation."""
        if cs is None:
            self._cs, self.problem.cs, self.problem.formulation = None, None, 0
            for i in range(12):
                self.problem.QX[i] = 0.0
            return self
        cs = np.ascontiguousarray(cs, dtype=np.int32)
        if cs.shape != (self.N - 1, 4):
            raise ValueError("cs must have shape (N-1, 4)")
        self._cs = cs  # keeps the host array alive: the library reads it during each call
        self.problem.cs = cs.ctypes.data_as(_ip)
        self.problem.formulation = 1
        for i in range(12):
            self.problem.QX[i] = 0.0 if QX is None else float(QX[i])
        return self

    def close(self):
        if getattr(self, "ctx", None):
            self.lib.landing_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise RuntimeError("%s failed (%d): %s" % (what, rc, self.lib.landing_last_error().decode()))

    @property
    def launches(self):
        return self.lib.landing_launch_count(self.ctx)

    def fp64_peak_tflops(self):
        """Measured FP64 FMA throughput of this device (TFLOP/s)."""
        v = ctypes.c_double()
        self._check(self.lib.landing_fp64_peak(self.ctx, ctypes.byref(v)), "landing_fp64_peak")
        return v.value

    @property
    def stream_ptr(self):
        return self.lib.landing_stream(self.ctx)

    # ---- batched evaluation of the generated functions ------------------------------------
    def eval(self, B, memspace, layout, x=None, p=None, lam_f=None, lam_g=None, f=None, g=None,
             grad_f=None, jac=None, hess=None, grad_x=None, grad_p=None, status=None):
        io = EvalIO(_ptr(x), _ptr(p), _ptr(lam_f), _ptr(lam_g), _ptr(f), _ptr(g), _ptr(grad_f),
                    _ptr(jac), _ptr(hess), _ptr(grad_x), _ptr(grad_p), _ptr(status, _ip))
        self._check(self.lib.landing_eval_batch(self.ctx, B, memspace, layout, ctypes.byref(io)),
                    "landing_eval_batch")

    def eval_host(self, x, p, lam_f=None, lam_g=None, want=("f", "g", "grad_f", "jac", "hess"), layout=AOS):
        """Convenience: host numpy AoS [B, n] in -> dict of host numpy outputs."""
        d = self.dims
        x = np.ascontiguousarray(x, dtype=np.float64)
        B = x.shape[0] if layout == AOS else x.shape[1]
        sizes = dict(f=1, g=d["m"], grad_f=d["nx"], jac=d["nnzJ"], hess=d["nnzH"], grad_x=d["nx"], grad_p=d["np"])
        outs = {k: np.zeros((B, sizes[k]) if layout == AOS else (sizes[k], B)) for k in want}
        status = np.zeros(B, dtype=np.int32)
        self.eval(B, HOST, layout, x=x, p=np.ascontiguousarray(p, dtype=np.float64),
                  lam_f=None if lam_f is None else np.ascontiguousarray(lam_f, dtype=np.float64),
                  lam_g=None if lam_g is None else np.ascontiguousarray(lam_g, dtype=np.float64),
                  status=status, **outs)
        outs["status"] = status
        return outs

    def bounds_host(self, p, layout=AOS):
        p = np.ascontiguousarray(p, dtype=np.float64)
        B = p.shape[0] if layout == AOS else p.shape[1]
        shape = (B, self.dims["m"]) if layout == AOS else (self.dims["m"], B)
        lb, ub = np.zeros(shape), np.zeros(shape)
        self._check(self.lib.landing_bounds_batch(self.ctx, B, HOST, layout, _ptr(p), _ptr(lb), _ptr(ub)),
                    "landing_bounds_batch")
        return lb, ub

    def build_host(self, drops, layout=AOS):
        """drops [B,12] -> (p [B,np], x0 [B,nx]) as the reference's callers build them."""
        drops = np.ascontiguousarray(drops, dtype=np.float64)
        B = drops.shape[0]
        p = np.zeros((B, self.dims["np"]) if layout == AOS else (self.dims["np"], B))
        x0 = np.zeros((B, self.dims["nx"]) if layout == AOS else (self.dims["nx"], B))
        self._check(self.lib.landing_build_batch(self.ctx, B, HOST, layout, ctypes.byref(self.problem),
                                                 _ptr(drops), _ptr(p), _ptr(x0)), "landing_build_batch")
        return p, x0

    # ---- the solve: one NLP per drop condition ----------------------------------------------
    def set_flavour(self, name):
        """Option set of the reference's two serialized solvers: "cold" = landingCtrller_IPOPT
        (generate_landingCtrller_IPOPT.m:241-242: bound_push = bound_frac = 0.5), "ws" = landingCtrller_IPOPT_ws
        (generate_landingCtrller_IPOPT_warmstart.m:246-247: 5e-3, called with a previous solution as x0 (:227-230));
        everything else is identical in the two generators."""
        v = {"cold": 0.5, "ws": 5e-3}[name]
        self.options.bound_push = v
        self.options.bound_frac = v
        return self

    def solve(self, drops, x0=None, want_lam=False, want_lam_p=False):
        """drops: host numpy [B,12] (q_init[6], qd_init[6]). Returns dict of host arrays.

        want_lam: also return lam_g [B,m].  want_lam_p: also return lam_x [B,nx] and lam_p [B,np], obtained as CasADi's
        Nlpsol does after the solve (nlpsol.cpp:609-625): one nlp_grad evaluation at (x*, lam_f = 1, lam_g*);
        lam_x = -grad_gamma_x is ~0 here (the reference passes no variable bounds), lam_p = -grad_gamma_p."""
        want_lam = want_lam or want_lam_p
        if want_lam_p and any(self.problem.Qf[i] != 0.0 for i in range(3)):
            # lam_x / lam_p come from nlp_grad of the landingCtrller_IPOPT functions, which have no running GRF cost
            raise ValueError("want_lam_p is defined for the landingCtrller_IPOPT problem only (problem.Qf must be 0): "
                             "the generated functions behind nlp_grad do not contain the running cost of the CCC variant")
        drops = np.ascontiguousarray(drops, dtype=np.float64)
        B = drops.shape[0]
        d = self.dims
        out = dict(x=np.zeros((B, d["nx"])), f=np.zeros(B), viol=np.zeros(B),
                   status=np.full(B, 9, dtype=np.int32), iters=np.zeros(B, dtype=np.int32))
        if want_lam:
            out["lam_g"] = np.zeros((B, d["m"]))
        x0c = None if x0 is None else np.ascontiguousarray(x0, dtype=np.float64)
        io = SolveIO(_ptr(drops), _ptr(x0c), _ptr(out["x"]), _ptr(out["f"]), _ptr(out.get("lam_g")),
                     _ptr(out["viol"]), _ptr(out["status"], _ip), _ptr(out["iters"], _ip))
        self._check(self.lib.landing_solve_batch(self.ctx, B, HOST, ctypes.byref(self.problem),
                                                 ctypes.byref(self.options), ctypes.byref(io)),
                    "landing_solve_batch")
        if want_lam_p:
            p, _ = self.build_host(drops)
            g = self.eval_host(out["x"], p, lam_f=np.ones(B), lam_g=out["lam_g"], want=("grad_x", "grad_p"))
            out["lam_x"], out["lam_p"] = -g["grad_x"], -g["grad_p"]
        return out

    def tvlqr_default(self):
        par = Tvlqr()
        self.lib.landing_tvlqr_default(ctypes.byref(par))
        par.T = self.problem.T
        par.n_steps = int(round(par.T / par.dt)) + 1
        return par

    def tvlqr(self, x_star, par=None, want_K=True):
        """Time-varying LQR pass along solved trajectories x_star [B, nx] (quadruped_SRBM_NLP.m:428-497):
        P [B, n_steps, 24, 24] and, if asked, the gains K [B, n_steps, 12, 24]."""
        par = par or self.tvlqr_default()
        x = np.ascontiguousarray(x_star, dtype=np.float64)
        B = x.shape[0]
        P = np.zeros((B, par.n_steps, 24, 24))
        K = np.zeros((B, par.n_steps, 12, 24)) if want_K else None
        self._check(self.lib.landing_tvlqr_batch(self.ctx, B, HOST, ctypes.byref(par), _ptr(x), _ptr(P), _ptr(K)),
                    "landing_tvlqr_batch")
        return (P, K) if want_K else P

    # ---- kino-dynamic ("full-body") NLP of the reference's KNITRO variant (SURVEY 8 f-2)
    def kino_dims(self):
        d = (ctypes.c_longlong * 4)()
        self._check(self.lib.landing_kino_dims(self.N, d), "landing_kino_dims")
        return {"N": int(d[0]), "nx": int(d[1]), "m": int(d[2]), "nnzJ": int(d[3])}

    def kino_sparsity(self):
        """CCS pattern of dg/dx: (colind [nx + 1], row [nnz])."""
        d = self.kino_dims()
        sp = self.lib.landing_kino_sparsity(self.N)
        a = np.ctypeslib.as_array(sp, shape=(2 + d["nx"] + 1 + d["nnzJ"],))
        return a[2:2 + d["nx"] + 1].copy(), a[2 + d["nx"] + 1:].copy()

    def kino_problem(self, dt, mu=0.75, mass=None, Ib=None, Ib_inv=None):
        """Parameter values of generate_landingCtrller_KNITRO.m:224-262 (mass / inertia as in landing_problem)."""
        pb = KinoProblem()
        pb.mu = mu
        pb.mass = self.problem.mass if mass is None else mass
        for i in range(3):
            pb.Ib[i] = self.problem.Ib[i] if Ib is None else Ib[i]
            pb.Ib_inv[i] = self.problem.Ib_inv[i] if Ib_inv is None else Ib_inv[i]
        dt = np.ascontiguousarray(dt, dtype=np.float64)
        if dt.shape != (self.N - 1,):
            raise ValueError("dt must have N-1 = %d entries" % (self.N - 1))
        pb._dt = dt  # keeps the host array alive as long as this problem: the library reads it during each call
        pb.dt = dt.ctypes.data_as(_dp)
        return pb

    def kino_eval_host(self, x, pb, want_g=True, want_jac=True, layout=AOS):
        """g [B, m] and the CCS value array of dg/dx [B, nnz] of the kino-dynamic NLP for a batch of
        x = [X(:); jpos(:); U(:)] (host arrays; layout SOA: [n, B])."""
        d = self.kino_dims()
        x = np.ascontiguousarray(x, dtype=np.float64)
        B = x.shape[0] if layout == AOS else x.shape[1]
        shp = (lambda n: (B, n)) if layout == AOS else (lambda n: (n, B))
        g = np.zeros(shp(d["m"])) if want_g else None
        jac = np.zeros(shp(d["nnzJ"])) if want_jac else None
        self._check(self.lib.landing_kino_eval_batch(self.ctx, B, HOST, layout, ctypes.byref(pb), _ptr(x), _ptr(g), _ptr(jac)),
                    "landing_kino_eval_batch")
        return g, jac

    def kino_eval_device(self, x, pb, g=None, jac=None, layout=SOA):
        """Same with CUDA torch tensors already in HBM (enqueued on the library stream)."""
        B = x.shape[0] if layout == AOS else x.shape[1]
        self._check(self.lib.landing_kino_eval_batch(self.ctx, B, DEVICE, layout, ctypes.byref(pb), _ptr(x), _ptr(g), _ptr(jac)),
                    "landing_kino_eval_batch")

    def kino_setup_data(self):
        """landing_kino_setup with the reference's values (generate_landingCtrller_KNITRO.m:214-262,325)."""
        ks = KinoSetup()
        self.lib.landing_kino_setup_default(ctypes.byref(ks))
        return ks

    def kino_setup_host(self, drops, x_srb=None, ks=None, want_bounds=True, want_x0=True):
        """lbg, ubg [B, m] and the initial guess x0 [B, n_x] = [X; jpos_guess; U] of the kino-dynamic NLP for a batch of
        drop conditions [B, 12]; x_srb [B, 36N-24]: SRB solutions (landing_solve_batch) to start from, None: the
        reference trajectories (generate_landingCtrller_KNITRO.m:272-286,302-325).  Host arrays, AoS."""
        d = self.kino_dims()
        ks = ks or self.kino_setup_data()
        drops = np.ascontiguousarray(drops, dtype=np.float64)
        B = drops.shape[0]
        if x_srb is not None:
            x_srb = np.ascontiguousarray(x_srb, dtype=np.float64)
            if x_srb.shape != (B, 36 * self.N - 24):
                raise ValueError("x_srb must be [B, 36N-24]")
        lb = np.zeros((B, d["m"])) if want_bounds else None
        ub = np.zeros((B, d["m"])) if want_bounds else None
        x0 = np.zeros((B, d["nx"])) if want_x0 else None
        self._check(self.lib.landing_kino_setup_batch(self.ctx, B, HOST, AOS, ctypes.byref(ks), _ptr(drops), _ptr(x_srb),
                                                      _ptr(lb), _ptr(ub), _ptr(x0)), "landing_kino_setup_batch")
        return lb, ub, x0

    def kino_setup_device(self, drops, x_srb=None, lbg=None, ubg=None, x0=None, ks=None, layout=AOS):
        """Same with CUDA torch tensors already in HBM (enqueued on the library stream); any output may be None."""
        ks = ks or self.kino_setup_data()
        B = drops.shape[0] if layout == AOS else drops.shape[1]
        self._check(self.lib.landing_kino_setup_batch(self.ctx, B, DEVICE, layout, ctypes.byref(ks), _ptr(drops), _ptr(x_srb),
                                                      _ptr(lbg), _ptr(ubg), _ptr(x0)), "landing_kino_setup_batch")

    def kino_cost_host(self, x, ks=None):
        """Terminal cost f [B] and its gradient [B, n_x] of the kino-dynamic NLP (generate_landingCtrller_KNITRO.m:86-88)."""
        d = self.kino_dims()
        ks = ks or self.kino_setup_data()
        x = np.ascontiguousarray(x, dtype=np.float64)
        B = x.shape[0]
        f, gf = np.zeros(B), np.zeros((B, d["nx"]))
        self._check(self.lib.landing_kino_cost_batch(self.ctx, B, HOST, AOS, ctypes.byref(ks), _ptr(x), _ptr(f), _ptr(gf)),
                    "landing_kino_cost_batch")
        return f, gf

    def kino_hess_sparsity(self):
        """Upper-triangle CCS pattern of the Lagrangian Hessian of the kino-dynamic NLP: (colind [nx + 1], row [nnz])."""
        sp = self.lib.landing_kino_hess_sparsity(self.N)
        if not sp:
            raise RuntimeError("landing_kino_hess_sparsity: %s" % self.lib.landing_last_error().decode())
        nx = sp[1]
        a = np.ctypeslib.as_array(sp, shape=(2 + nx + 1 + sp[2 + nx],))
        return a[2:2 + nx + 1].copy(), a[2 + nx + 1:].copy()

    def kino_hess_host(self, x, pb, lam_f=None, lam_g=None, ks=None, layout=AOS):
        """CCS value array [B, nnzH] of the upper triangle of d2/dx2 (lam_f f + lam_g' g) of the kino-dynamic NLP
        (host arrays; layout SOA: [n, B]).  lam_f [B], lam_g [B, m]: None = zero; ks: QN of the terminal cost (default
        landing_kino_setup when lam_f is given)."""
        x = np.ascontiguousarray(x, dtype=np.float64)
        B = x.shape[0] if layout == AOS else x.shape[1]
        nnz = len(self.kino_hess_sparsity()[1])
        if lam_f is not None:
            lam_f = np.ascontiguousarray(lam_f, dtype=np.float64)
            ks = ks or self.kino_setup_data()
        if lam_g is not None:
            lam_g = np.ascontiguousarray(lam_g, dtype=np.float64)
        hess = np.zeros((B, nnz) if layout == AOS else (nnz, B))
        self._check(self.lib.landing_kino_hess_batch(self.ctx, B, HOST, layout, ctypes.byref(pb),
                                                     None if ks is None else ctypes.byref(ks), _ptr(x), _ptr(lam_f),
                                                     _ptr(lam_g), _ptr(hess)), "landing_kino_hess_batch")
        return hess

    def kino_hess_device(self, x, pb, hess, lam_f=None, lam_g=None, ks=None, layout=SOA):
        """Same with CUDA torch tensors already in HBM (enqueued on the library stream)."""
        B = x.shape[0] if layout == AOS else x.shape[1]
        if lam_f is not None:
            ks = ks or self.kino_setup_data()
        self._check(self.lib.landing_kino_hess_batch(self.ctx, B, DEVICE, layout, ctypes.byref(pb),
                                                     None if ks is None else ctypes.byref(ks), _ptr(x), _ptr(lam_f),
                                                     _ptr(lam_g), _ptr(hess)), "landing_kino_hess_batch")

    def synchronize(self):
        self._check(self.lib.landing_synchronize(self.ctx), "landing_synchronize")

    def solve_device(self, drops, x_star, f_star, status, iters, viol=None, lam_g=None, x0=None, order_streams=True):
        """All arguments are CUDA torch tensors already resident in HBM (no copies).  The library only ENQUEUES on its
        own stream (include/landing_b200.h, stream contract): with order_streams the library stream first waits for the
        caller's current torch stream (the producers of the inputs) and the caller's stream then waits for the library
        stream, so that the call behaves like any other op on the current stream."""
        B = drops.shape[0]
        if order_streams:
            import torch
            lib_stream = torch.cuda.ExternalStream(self.stream_ptr, device=drops.device)
            cur = torch.cuda.current_stream(drops.device)
            lib_stream.wait_stream(cur)
        io = SolveIO(_ptr(drops), _ptr(x0), _ptr(x_star), _ptr(f_star), _ptr(lam_g), _ptr(viol),
                     _ptr(status, _ip), _ptr(iters, _ip))
        self._check(self.lib.landing_solve_batch(self.ctx, B, DEVICE, ctypes.byref(self.problem),
                                                 ctypes.byref(self.options), ctypes.byref(io)),
                    "landing_solve_batch")
        if order_streams:
            cur.wait_stream(lib_stream)


class MultiGpuSolver:
    """One sweep on several GPUs of this process (landing_solve_batch_multi): interleaved shards, one host thread per
    device, results gathered in global scenario order in host memory."""

    def __init__(self, N, devices, lib_path=LIB_PATH):
        self.lib = load_library(lib_path)
        self.N, self.devices = N, list(devices)
        self.handle = ctypes.c_void_p()
        arr = (ctypes.c_int * len(self.devices))(*self.devices)
        rc = self.lib.landing_multi_create(N, len(self.devices), arr, ctypes.byref(self.handle))
        if rc != 0:
            raise RuntimeError("landing_multi_create failed (%d): %s" % (rc, self.lib.landing_last_error().decode()))
        self.dims = dims_for(N, self.lib)
        self.problem, self.options = Problem(), Options()
        self.lib.landing_problem_default(ctypes.byref(self.problem))
        self.lib.landing_options_default(ctypes.byref(self.options))

    def solve(self, drops, want_lam=False):
        drops = np.ascontiguousarray(drops, dtype=np.float64)
        B, d = drops.shape[0], self.dims
        out = dict(x=np.zeros((B, d["nx"])), f=np.zeros(B), viol=np.zeros(B),
                   status=np.full(B, 9, dtype=np.int32), iters=np.zeros(B, dtype=np.int32))
        if want_lam:
            out["lam_g"] = np.zeros((B, d["m"]))
        io = SolveIO(_ptr(drops), None, _ptr(out["x"]), _ptr(out["f"]), _ptr(out.get("lam_g")), _ptr(out["viol"]),
                     _ptr(out["status"], _ip), _ptr(out["iters"], _ip))
        rc = self.lib.landing_solve_batch_multi(self.handle, B, ctypes.byref(self.problem), ctypes.byref(self.options),
                                                ctypes.byref(io))
        if rc != 0:
            raise RuntimeError("landing_solve_batch_multi failed (%d): %s" % (rc, self.lib.landing_last_error().decode()))
        return out

    def close(self):
        if getattr(self, "handle", None):
            self.lib.landing_multi_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def contact_set(x, N, thresh=1.0):
    """cs[leg,k] = f_z > 1  (optimizations/landing/codegen_casadi/test_loadCasadi_ws.m:144-147)."""
    x = np.asarray(x)
    U = x[..., 12 * N:].reshape(x.shape[:-1] + (N - 1, 24))
    return U[..., 12 + 2::3][..., :4] > thresh
