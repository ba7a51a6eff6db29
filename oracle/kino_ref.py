"""oracle/kino_ref.py -- TEST INFRASTRUCTURE ONLY (CPU oracle).

numpy restatement of the constraint function of the reference's kino-dynamic ("full-body") landing NLP, the KNITRO
variant (SURVEY 8 f-2): /root/reference/optimizations/landing/generate_solver/generate_landingCtrller_KNITRO.m:34-193.
The generated C of that variant is absent from the reference (.MISSING_LARGE_BLOBS: landingCtrller_KNITRO.c/.so), so
the functions are restated from the generator script and the utilities it calls, each cited below, and pinned by the
one solution of this NLP that the reference stores (generate_solver/prevSoln.mat: X_star, jpos_star, U_star,
lam_g_star[2844]): tests/test_kino.py checks that the stored point is feasible for the restated rows and stationary
for the restated Jacobian with the stored multipliers.

Variables (Opti creation order, :45-51):  x = [X(:) (12 N); jpos(:) (12 (N-1)); U(:) (24 (N-1))], column-major,
X_k = (r, rpy, omega_body, v_world), U_k = (c[4x3], f[4x3]).  Rows (Opti canonical form, optistack_internal.cpp:742-870:
`a == b` -> a - b = 0, one- and two-sided inequalities keep the variable expression as g):
  0..23   q_0, qd_0, c_0 (= q_init, qd_init, c_init)                 :93-95
  24..47  q_{N-1} (twice), qd_{N-1} (twice)                          :98-101
  per knot k (141 rows, 117 for the last knot: no no-slip rows):
    v+ - v - rddot dt | om+ - om - omdot dt | r+ - r - v dt | rpy+ - rpy - Binv (R om) dt       :128-131
    f_z (4)                                                                                    :134
    per leg: c_z | f_z c_z | [f_z (c+ - c) (3) twice] | p_x | p_y | p_z | p.p | tau (3)        :139-174
    friction (16) | z_k | c - FK (12) twice | jpos (12) twice                                  :177-193
"""
import numpy as np

# ---- robot constants (utilities_general/dynamics-utilities/get_robot_params.m:50-115, 'mc3D')
ABAD_LOC = np.array([0.19, 0.049, 0.0])           # abadLocation = [bodyLength, bodyWidth, 0] / 2   (:86)
L1, L2, L3, L4 = 0.062, 0.209, 0.195, 0.004       # abad / hip / knee link lengths (:56-58); l_4 get_foot_jacobians_mc.m:8
HIP_SRBM = np.array([[0.19, -0.1, 0], [0.19, 0.1, 0], [-0.19, -0.1, 0], [-0.19, 0.1, 0]])  # (:90-91)
SIDE_SIGN = np.array([[1, 1, -1, -1], [-1, 1, -1, 1], [1, 1, 1, 1]])   # get_robot_model.m:194 (columns = legs)
TAU_MAX = np.array([18.0, 18.0, 27.99])           # gear ratios (6, 6, 9.33) x 3 Nm   (get_robot_model.m:237-241)
GRAVITY = np.array([0.0, 0.0, -9.81])             # get_robot_model.m:140
JPOS_MIN = np.tile([-np.pi / 3, -np.pi / 2, 0.0], 4)          # generate_landingCtrller_KNITRO.m:252-253
JPOS_MAX = np.tile([np.pi / 3, np.pi / 2, 3 * np.pi / 4], 4)
DT_VAL = np.array([0.05] + [0.02] * 15 + [0.05, 0.05, 0.1, 0.2])   # :30


def rx(t):  # coordinate transforms of spatial_v2/3D/rx.m, ry.m, rz.m:8-13
    c, s = np.cos(t), np.sin(t)
    return np.array([[1, 0, 0], [0, c, s], [0, -s, c]])


def ry(t):
    c, s = np.cos(t), np.sin(t)
    return np.array([[c, 0, -s], [0, 1, 0], [s, 0, c]])


def rz(t):
    c, s = np.cos(t), np.sin(t)
    return np.array([[c, s, 0], [-s, c, 0], [0, 0, 1]])


def rpy_to_rot_xyz(rpy):  # rpyToRotMat_xyz.m:2  (body -> world)
    return rx(rpy[0]).T @ ry(rpy[1]).T @ rz(rpy[2]).T


def binv(rpy):  # Binv.m:13-17
    psi, th = rpy[2], rpy[1]
    return np.array([[np.cos(psi) / np.cos(th), np.sin(psi) / np.cos(th), 0],
                     [-np.sin(psi), np.cos(psi), 0],
                     [np.cos(psi) * np.tan(th), np.sin(psi) * np.tan(th), 1]])


def _skew(v):
    return np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]])


def _plux(E, r):  # spatial_v2/spatial/plux.m: E, r -> X
    X = np.zeros((6, 6))
    X[:3, :3] = E
    X[3:, :3] = -E @ _skew(r)
    X[3:, 3:] = E
    return X


def _plux_r(X):  # plux_2.m: translation of a Pluecker transform
    E = X[:3, :3]
    M = -E.T @ X[3:, :3]
    return 0.5 * np.array([M[2, 1] - M[1, 2], M[0, 2] - M[2, 0], M[1, 0] - M[0, 1]])


def _jcalc(jt, q):  # spatial_v2/dynamics/jcalc.m:19-40
    if jt == "Rx": return _plux(rx(q), np.zeros(3))
    if jt == "Ry": return _plux(ry(q), np.zeros(3))
    if jt == "Rz": return _plux(rz(q), np.zeros(3))
    r = np.zeros(3)
    r["xyz".index(jt[1])] = q
    return _plux(np.eye(3), r)


def forward_kin_foot_literal(q18):
    """get_forward_kin_foot.m:4-25 on the 18-body model of get_robot_model.m:134-244 (literal: 6x6 transforms)."""
    jtype = ["Px", "Py", "Pz", "Rx", "Ry", "Rz"]
    parent = [0, 1, 2, 3, 4, 5]
    xtree = [np.eye(6)] * 6
    xfoot, bfoot = [], []
    for leg in range(4):
        ss = SIDE_SIGN[:, leg]
        jtype += ["Rx", "Ry", "Ry"]
        nb = len(parent)
        parent += [6, nb + 1, nb + 2]
        xtree += [_plux(np.eye(3), ss * ABAD_LOC),
                  _plux(rz(np.pi), np.zeros(3)) @ _plux(np.eye(3), ss * np.array([0, L1, 0])),
                  _plux(np.eye(3), ss * np.array([0, 0, -L2]))]
        xfoot.append(_plux(np.eye(3), ss * np.array([0, 0, -L3])))
        bfoot.append(nb + 3)
    X0 = []
    for i in range(18):
        Xup = _jcalc(jtype[i], q18[i]) @ xtree[i]
        X0.append(Xup if parent[i] == 0 else Xup @ X0[parent[i] - 1])
    return [_plux_r(xfoot[l] @ X0[bfoot[l] - 1]) for l in range(4)]


def leg_fk_body(leg, ql):
    """Closed form of the same chain: foot position relative to the body origin, body frame (what the CUDA kernel uses;
    tests/test_kino.py checks it against forward_kin_foot_literal)."""
    s1, c1 = np.sin(ql[0]), np.cos(ql[0])
    s2, c2 = np.sin(ql[1]), np.cos(ql[1])
    s23, c23 = np.sin(ql[1] + ql[2]), np.cos(ql[1] + ql[2])
    sy = SIDE_SIGN[1, leg]
    a = L2 * c2 + L3 * c23          # leg extension along the (rotated) -z axis
    b = L2 * s2 + L3 * s23
    return SIDE_SIGN[:, leg] * ABAD_LOC + np.array([b, sy * L1 * c1 + a * s1, sy * L1 * s1 - a * c1])


def foot_jacobian_mc(leg, ql):  # get_foot_jacobians_mc.m:3-24
    ss = [-1, 1, -1, 1][leg]
    s1, s2, s3 = np.sin(ql)
    c1, c2, c3 = np.cos(ql)
    c23 = c2 * c3 - s2 * s3
    s23 = s2 * c3 + c2 * s3
    return np.array([[0, L3 * c23 + L2 * c2, L3 * c23],
                     [L3 * c1 * c23 + L2 * c1 * c2 - (L1 + L4) * s1 * ss, -L3 * s1 * s23 - L2 * s1 * s2, -L3 * s1 * s23],
                     [L3 * s1 * c23 + L2 * c2 * s1 + (L1 + L4) * ss * c1, L3 * c1 * s23 + L2 * c1 * s2, L3 * c1 * s23]])


def kin_box_limits(v, d):  # utilities_landing/kin_box_limits.m
    bmax = 0.15 if d == "x" else 0.25
    return abs(v * bmax / 2.0) if abs(v) < 2.0 else bmax


def dims(N):
    return {"N": N, "nx": 12 * N + 36 * (N - 1), "m": 48 + 141 * (N - 2) + 117}


def split(x, N):
    X = x[:12 * N].reshape(N, 12)
    J = x[12 * N:12 * N + 12 * (N - 1)].reshape(N - 1, 12)
    U = x[12 * N + 12 * (N - 1):].reshape(N - 1, 24)
    return X, J, U


def default_problem(N=21):
    """Shared numeric data of generate_landingCtrller_KNITRO.m:224-262 (mass / Ib: oracle/crba_constants.py values)."""
    return {"N": N, "dt": DT_VAL.copy() if N == 21 else np.full(N - 1, 0.6 / (N - 1)), "mu": 0.75, "l_leg_max": 0.4,
            "mass": 8.252, "Ib": np.array([0.0575772985, 0.2340089948, 0.2796738483]),
            "Ib_inv": np.array([17.3774688889, 4.2733400093, 3.5775519238]),
            "q_term_min": np.array([-10, -10, 0.15, -0.1, -0.1, -10.0]), "q_term_max": np.array([10, 10, 5, 0.1, 0.1, 10.0]),
            "qd_term_min": np.array([-10, -10, -10, -.5, -.5, -.5]), "qd_term_max": np.array([10, 10, 10, .5, .5, .5]),
            "z_min": 0.075, "kin_box": np.zeros(2), "jpos_min": JPOS_MIN.copy(), "jpos_max": JPOS_MAX.copy()}


def knot_rows(pb, k, Xk, Xn, jk, Uk, cn, literal=True):
    """The rows of knot k (0-based), generate_landingCtrller_KNITRO.m:107-193.  cn = c_{k+1} or None for the last knot.
    literal: forward kinematics through the 6x6 spatial transforms as the reference does, else the closed form."""
    h = pb["dt"][k]
    r, rpy, om, v = Xk[0:3], Xk[3:6], Xk[6:9], Xk[9:12]
    c, f = Uk[:12].reshape(4, 3), Uk[12:].reshape(4, 3)
    R = rpy_to_rot_xyz(rpy)
    rdd = f.sum(0) / pb["mass"] + GRAVITY
    tq = sum(np.cross(c[l] - r, f[l]) for l in range(4))
    omd = pb["Ib_inv"] * (R.T @ tq - np.cross(om, pb["Ib"] * om))
    g = [Xn[9:12] - v - rdd * h, Xn[6:9] - om - omd * h, Xn[0:3] - r - v * h, Xn[3:6] - rpy - binv(rpy) @ (R @ om) * h]
    g.append(f[:, 2].copy())
    if literal:
        feet = forward_kin_foot_literal(np.concatenate([Xk[:6], jk]))
    else:
        feet = [r + R @ leg_fk_body(l, jk[3 * l:3 * l + 3]) for l in range(4)]
    for l in range(4):
        rows = [c[l, 2], f[l, 2] * c[l, 2]]
        if cn is not None:
            d = f[l, 2] * (cn[3 * l:3 * l + 3] - c[l])
            rows += list(d) + list(d)
        p = c[l] - (r + R @ HIP_SRBM[l])
        rows += [p[0], p[1], p[2], p @ p]
        tau = foot_jacobian_mc(l, jk[3 * l:3 * l + 3]).T @ (-R.T @ f[l])
        rows += list(tau)
        g.append(np.array(rows))
    mu = pb["mu"]
    g.append(f[:, 0] - 0.71 * mu * f[:, 2])     # f_x <= 0.71 mu f_z   -> a - b <= 0
    g.append(-0.71 * mu * f[:, 2] - f[:, 0])    # f_x >= -0.71 mu f_z  -> b - a <= 0
    g.append(f[:, 1] - 0.71 * mu * f[:, 2])
    g.append(-0.71 * mu * f[:, 2] - f[:, 1])
    g.append(np.array([r[2]]))
    d = c.reshape(12) - np.concatenate(feet)
    g += [d, d, jk, jk]
    return np.concatenate(g)


def eval_g(pb, x, literal=True):
    N = pb["N"]
    X, J, U = split(np.asarray(x, dtype=np.float64), N)
    g = [X[0, 0:6], X[0, 6:12], U[0, :12], X[N - 1, 0:6], X[N - 1, 0:6], X[N - 1, 6:12], X[N - 1, 6:12]]
    for k in range(N - 1):
        g.append(knot_rows(pb, k, X[k], X[k + 1], J[k], U[k], U[k + 1, :12] if k + 1 < N - 1 else None, literal))
    return np.concatenate(g)


def bounds(pb, q_init, qd_init, c_init):
    """lbg, ubg in row order (Opti canonical form)."""
    N = pb["N"]
    INF = np.inf
    lb = [q_init, qd_init, c_init, pb["q_term_min"], np.full(6, -INF), pb["qd_term_min"], np.full(6, -INF)]
    ub = [q_init, qd_init, c_init, np.full(6, INF), pb["q_term_max"], np.full(6, INF), pb["qd_term_max"]]
    kx, ky = 0.125 + pb["kin_box"][0], 0.125 + pb["kin_box"][1]
    for k in range(N - 1):
        last = k == N - 2
        lb.append(np.zeros(12)); ub.append(np.zeros(12))
        lb.append(np.zeros(4)); ub.append(np.full(4, INF))
        for l in range(4):
            l_, u_ = [0.0, -INF], [INF, 0.001]
            if not last:
                l_ += [-INF] * 3 + [-0.001] * 3
                u_ += [0.001] * 3 + [INF] * 3
            ss = [-1, 1, -1, 1][l]
            l_ += [-kx, (-ky if l in (0, 2) else -0.05 * ss), -0.4, -INF]
            u_ += [kx, (-0.05 * ss if l in (0, 2) else ky), -0.075, pb["l_leg_max"] ** 2]
            tau_max = np.asarray(pb.get("tau_max", TAU_MAX))
            l_ += list(-tau_max); u_ += list(tau_max)
            lb.append(np.array(l_)); ub.append(np.array(u_))
        lb.append(np.full(16, -INF)); ub.append(np.zeros(16))
        lb.append(np.array([pb["z_min"]])); ub.append(np.array([INF]))
        lb += [np.full(12, -0.01), np.full(12, -INF), pb["jpos_min"], np.full(12, -INF)]
        ub += [np.full(12, INF), np.full(12, 0.01), np.full(12, INF), pb["jpos_max"]]
    return np.concatenate(lb), np.concatenate(ub)


def knot_col(N, k, v):
    """Knot-local input v of knot k (X_k 0..11 | jpos_k 12..23 | U_k 24..47 | X_{k+1} 48..59 | c_{k+1} 60..71) -> column
    of x."""
    if v < 12: return 12 * k + v
    if v < 24: return 12 * N + 12 * k + (v - 12)
    if v < 48: return 24 * N - 12 + 24 * k + (v - 24)
    if v < 60: return 12 * (k + 1) + (v - 48)
    return 24 * N - 12 + 24 * (k + 1) + (v - 60)


def knot_jac(pb, k, z, last, h=1e-30):
    """Rows of knot k and their exact Jacobian [rows, len(z)] in the knot-local inputs z (72; 60 for the last knot), by
    the complex step: d g / d z_j = Im g(z + i h e_j) / h has no subtractive cancellation, so it is exact to rounding.
    The closed-form kinematics (literal=False) are complex-safe."""
    z = np.asarray(z, dtype=np.complex128)

    def rows(zz):
        return knot_rows(pb, k, zz[0:12], zz[48:60], zz[12:24], zz[24:48], None if last else zz[60:72], literal=False)

    J = np.zeros((117 if last else 141, z.size))
    for j in range(z.size):
        zz = z.copy()
        zz[j] += 1j * h
        J[:, j] = rows(zz).imag / h
    return rows(z).real, J


def jac_exact(pb, x, pattern=None):
    """Exact dg/dx (tests only): the complex-step Jacobian of every knot (knot_jac) plus the 48 identity entries of the
    boundary rows.  Dense [m, nx], or with pattern = (colind, row) (CCS) the value array at that pattern."""
    N = pb["N"]
    d = dims(N)
    x = np.asarray(x, dtype=np.float64)
    Jm = np.zeros((d["m"], d["nx"]))
    nu = 24 * N - 12  # first column of U
    bcols = list(range(12)) + [nu + i for i in range(12)] + [12 * (N - 1) + i for i in (0, 1, 2, 3, 4, 5) * 2] + \
        [12 * (N - 1) + 6 + i for i in (0, 1, 2, 3, 4, 5) * 2]
    Jm[np.arange(48), bcols] = 1.0
    for k in range(N - 1):
        last = k == N - 2
        cols = [knot_col(N, k, v) for v in range(60 if last else 72)]
        _, Jk = knot_jac(pb, k, x[cols], last)
        base = 48 + 141 * k
        Jm[base:base + Jk.shape[0], cols] = Jk
    if pattern is None:
        return Jm
    colind, row = pattern
    col = np.repeat(np.arange(d["nx"]), np.diff(colind))
    return Jm[row, col]


def jac_fd(pb, x, h=1e-6, cols=None, literal=True):
    """Dense central-difference Jacobian (tests only; 2844 x 972 at N = 21); cols: only these columns are filled."""
    x = np.asarray(x, dtype=np.float64)
    m = dims(pb["N"])["m"]
    Jm = np.zeros((m, x.size))
    for i in (range(x.size) if cols is None else cols):
        e = np.zeros_like(x); e[i] = h
        Jm[:, i] = (eval_g(pb, x + e, literal) - eval_g(pb, x - e, literal)) / (2 * h)
    return Jm
