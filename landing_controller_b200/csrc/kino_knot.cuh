// kino_knot.cuh -- one knot of the kino-dynamic ("full-body") landing NLP, the reference's KNITRO variant
// (SURVEY 8 f-2): generate_solver/generate_landingCtrller_KNITRO.m:107-193 with get_forward_kin_foot.m:4-25 on the
// 18-body model of get_robot_model.m:134-244 (closed form of that chain), get_foot_jacobians_mc.m:3-24,
// rpyToRotMat_xyz.m:2, Binv.m:13-17.  Templated on the scalar type of every input block: double for the constraint values, DualN
// (value + tangents) on the seeded block for the Jacobian columns, Dual2 (second order) on two seeded triples for the
// blocks of the Lagrangian Hessian -- exact derivatives, no hand-derived entries.  Host and device.
//
// Knot-local inputs (72): X_k 0..11 (r, rpy, omega_body, v_world) | jpos_k 12..23 | U_k 24..47 (c[4x3], f[4x3]) |
// X_{k+1} 48..59 | c_{k+1} 60..71 (unused by the last knot).  Knot-local rows (141; 117 for the last knot, whose 24
// no-slip rows are absent): see the row map in oracle/kino_ref.py.
#pragma once
#include <cmath>
#include <type_traits>

namespace srb {
namespace kino {

#ifdef __CUDACC__
#define KHD __host__ __device__ __forceinline__
#else
#define KHD inline
#endif

constexpr int NIN = 72, ROWS_INT = 141, ROWS_LAST = 117;
constexpr double L1 = 0.062, L2 = 0.209, L3 = 0.195, L4 = 0.004;  // get_robot_params.m:56-58, get_foot_jacobians_mc.m:8
constexpr double ABAD_X = 0.19, ABAD_Y = 0.049;                    // abadLocation, get_robot_params.m:86

// Value + K tangents.  The knot function below is generic in the scalar type of every input block separately, so a
// Jacobian pass seeds one block (three tangents) and leaves the others plain doubles: whatever does not depend on the
// seeded block stays ordinary double arithmetic, and a row whose value comes out as a plain double has no entry in the
// columns of that pass -- exact block sparsity at compile time.
template <int K> struct DualN {
  double v, d[K];
  KHD DualN() : v(0.0) {
#pragma unroll
    for (int j = 0; j < K; j++) d[j] = 0.0;
  }
  KHD DualN(double a) : v(a) {
#pragma unroll
    for (int j = 0; j < K; j++) d[j] = 0.0;
  }
  KHD DualN(double a, double t0) : v(a) {  // first tangent t0
#pragma unroll
    for (int j = 0; j < K; j++) d[j] = 0.0;
    d[0] = t0;
  }
};
template <int K> KHD DualN<K> seeded(double a, int j) { DualN<K> r(a); r.d[j] = 1.0; return r; }  // unit tangent j
template <int K> KHD DualN<K> operator+(const DualN<K>& a, const DualN<K>& b) {
  DualN<K> r; r.v = a.v + b.v;
#pragma unroll
  for (int j = 0; j < K; j++) r.d[j] = a.d[j] + b.d[j];
  return r;
}
template <int K> KHD DualN<K> operator-(const DualN<K>& a, const DualN<K>& b) {
  DualN<K> r; r.v = a.v - b.v;
#pragma unroll
  for (int j = 0; j < K; j++) r.d[j] = a.d[j] - b.d[j];
  return r;
}
template <int K> KHD DualN<K> operator-(const DualN<K>& a) {
  DualN<K> r; r.v = -a.v;
#pragma unroll
  for (int j = 0; j < K; j++) r.d[j] = -a.d[j];
  return r;
}
template <int K> KHD DualN<K> operator*(const DualN<K>& a, const DualN<K>& b) {
  DualN<K> r; r.v = a.v * b.v;
#pragma unroll
  for (int j = 0; j < K; j++) r.d[j] = a.d[j] * b.v + a.v * b.d[j];
  return r;
}
template <int K> KHD DualN<K> operator/(const DualN<K>& a, const DualN<K>& b) {
  DualN<K> r; const double q = a.v / b.v; r.v = q;
#pragma unroll
  for (int j = 0; j < K; j++) r.d[j] = (a.d[j] - q * b.d[j]) / b.v;
  return r;
}
// mixed with plain doubles
template <int K> KHD DualN<K> operator+(const DualN<K>& a, double b) { DualN<K> r = a; r.v = a.v + b; return r; }
template <int K> KHD DualN<K> operator+(double a, const DualN<K>& b) { DualN<K> r = b; r.v = a + b.v; return r; }
template <int K> KHD DualN<K> operator-(const DualN<K>& a, double b) { DualN<K> r = a; r.v = a.v - b; return r; }
template <int K> KHD DualN<K> operator-(double a, const DualN<K>& b) { DualN<K> r = -b; r.v = a - b.v; return r; }
template <int K> KHD DualN<K> operator*(const DualN<K>& a, double b) {
  DualN<K> r; r.v = a.v * b;
#pragma unroll
  for (int j = 0; j < K; j++) r.d[j] = a.d[j] * b;
  return r;
}
template <int K> KHD DualN<K> operator*(double a, const DualN<K>& b) { return b * a; }
template <int K> KHD DualN<K> operator/(const DualN<K>& a, double b) { return a * (1.0 / b); }
template <int K> KHD DualN<K> operator/(double a, const DualN<K>& b) {
  DualN<K> r; const double q = a / b.v; r.v = q;
#pragma unroll
  for (int j = 0; j < K; j++) r.d[j] = -(q * b.d[j]) / b.v;
  return r;
}
template <int K> KHD void sincos_s(const DualN<K>& a, DualN<K>& s, DualN<K>& c) {
  const double sv = sin(a.v), cv = cos(a.v);
  s.v = sv; c.v = cv;
#pragma unroll
  for (int j = 0; j < K; j++) { s.d[j] = cv * a.d[j]; c.d[j] = -sv * a.d[j]; }
}
KHD void sincos_s(double a, double& s, double& c) { s = sin(a); c = cos(a); }
using Dual1 = DualN<1>;  // one tangent (host-side pattern probing)

// Second order, forward over forward: value, three tangents in seed set A, three in seed set B and the 3 x 3 block of
// mixed second derivatives h[i][j] = d2 / dA_i dB_j.  A Hessian pass types the block(s) of two input triples this way
// (seeds A on one triple, B on the other; both on the same triple for a diagonal block) and every other block a plain
// double, so the knot function above runs unchanged and whatever does not depend on either triple stays ordinary double
// arithmetic.
struct Dual2 {
  double v, a[3], b[3], h[3][3];
  KHD Dual2() : Dual2(0.0) {}
  KHD Dual2(double x) : v(x) {
#pragma unroll
    for (int i = 0; i < 3; i++) {
      a[i] = 0.0; b[i] = 0.0;
#pragma unroll
      for (int j = 0; j < 3; j++) h[i][j] = 0.0;
    }
  }
};
KHD Dual2 operator+(const Dual2& x, const Dual2& y) {
  Dual2 r; r.v = x.v + y.v;
#pragma unroll
  for (int i = 0; i < 3; i++) {
    r.a[i] = x.a[i] + y.a[i]; r.b[i] = x.b[i] + y.b[i];
#pragma unroll
    for (int j = 0; j < 3; j++) r.h[i][j] = x.h[i][j] + y.h[i][j];
  }
  return r;
}
KHD Dual2 operator-(const Dual2& x) {
  Dual2 r; r.v = -x.v;
#pragma unroll
  for (int i = 0; i < 3; i++) {
    r.a[i] = -x.a[i]; r.b[i] = -x.b[i];
#pragma unroll
    for (int j = 0; j < 3; j++) r.h[i][j] = -x.h[i][j];
  }
  return r;
}
KHD Dual2 operator-(const Dual2& x, const Dual2& y) {
  Dual2 r; r.v = x.v - y.v;
#pragma unroll
  for (int i = 0; i < 3; i++) {
    r.a[i] = x.a[i] - y.a[i]; r.b[i] = x.b[i] - y.b[i];
#pragma unroll
    for (int j = 0; j < 3; j++) r.h[i][j] = x.h[i][j] - y.h[i][j];
  }
  return r;
}
KHD Dual2 operator*(const Dual2& x, const Dual2& y) {
  Dual2 r; r.v = x.v * y.v;
#pragma unroll
  for (int i = 0; i < 3; i++) {
    r.a[i] = x.a[i] * y.v + x.v * y.a[i];
    r.b[i] = x.b[i] * y.v + x.v * y.b[i];
  }
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int j = 0; j < 3; j++)
      r.h[i][j] = x.h[i][j] * y.v + x.v * y.h[i][j] + x.a[i] * y.b[j] + y.a[i] * x.b[j];
  return r;
}
KHD Dual2 operator/(const Dual2& x, const Dual2& y) {  // q = x / y from x = q y
  Dual2 r; const double iy = 1.0 / y.v; r.v = x.v * iy;
#pragma unroll
  for (int i = 0; i < 3; i++) {
    r.a[i] = (x.a[i] - r.v * y.a[i]) * iy;
    r.b[i] = (x.b[i] - r.v * y.b[i]) * iy;
  }
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int j = 0; j < 3; j++)
      r.h[i][j] = (x.h[i][j] - r.v * y.h[i][j] - r.a[i] * y.b[j] - y.a[i] * r.b[j]) * iy;
  return r;
}
// mixed with plain doubles
KHD Dual2 operator*(const Dual2& x, double y) {
  Dual2 r; r.v = x.v * y;
#pragma unroll
  for (int i = 0; i < 3; i++) {
    r.a[i] = x.a[i] * y; r.b[i] = x.b[i] * y;
#pragma unroll
    for (int j = 0; j < 3; j++) r.h[i][j] = x.h[i][j] * y;
  }
  return r;
}
KHD Dual2 operator*(double x, const Dual2& y) { return y * x; }
KHD Dual2 operator+(const Dual2& x, double y) { Dual2 r = x; r.v = x.v + y; return r; }
KHD Dual2 operator+(double x, const Dual2& y) { Dual2 r = y; r.v = x + y.v; return r; }
KHD Dual2 operator-(const Dual2& x, double y) { Dual2 r = x; r.v = x.v - y; return r; }
KHD Dual2 operator-(double x, const Dual2& y) { Dual2 r = -y; r.v = x - y.v; return r; }
KHD Dual2 operator/(const Dual2& x, double y) { return x * (1.0 / y); }
KHD Dual2 operator/(double x, const Dual2& y) { return Dual2(x) / y; }
KHD void sincos_s(const Dual2& x, Dual2& s, Dual2& c) {
  const double sv = sin(x.v), cv = cos(x.v);
  s.v = sv; c.v = cv;
#pragma unroll
  for (int i = 0; i < 3; i++) {
    s.a[i] = cv * x.a[i]; s.b[i] = cv * x.b[i];
    c.a[i] = -sv * x.a[i]; c.b[i] = -sv * x.b[i];
  }
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int j = 0; j < 3; j++) {
      const double ab = x.a[i] * x.b[j];
      s.h[i][j] = cv * x.h[i][j] - sv * ab;
      c.h[i][j] = -sv * x.h[i][j] - cv * ab;
    }
}

// result type of an arithmetic expression of two scalar types
template <class A, class B> struct Promote { using type = A; };
template <int K> struct Promote<double, DualN<K>> { using type = DualN<K>; };
template <> struct Promote<double, Dual2> { using type = Dual2; };
template <class A, class B> using Pr = typename Promote<A, B>::type;

struct Params {
  double mu, mass, Ib[3], Ib_inv[3];
};

// knot-local input v of knot k -> column of x = [X(:) (12 N); jpos(:) (12 (N-1)); U(:) (24 (N-1))]
KHD long long knot_col(int N, int k, int v) {
  if (v < 12) return 12LL * k + v;
  if (v < 24) return 12LL * N + 12LL * k + (v - 12);
  if (v < 48) return 12LL * N + 12LL * (N - 1) + 24LL * k + (v - 24);
  if (v < 60) return 12LL * (k + 1) + (v - 48);
  return 12LL * N + 12LL * (N - 1) + 24LL * (k + 1) + (v - 60);
}

KHD double hip_x(int l) { return l < 2 ? 0.19 : -0.19; }      // hipSrbmLocation, get_robot_params.m:90-91
KHD double hip_y(int l) { return (l & 1) ? 0.1 : -0.1; }
KHD double side_y(int l) { return (l & 1) ? 1.0 : -1.0; }     // side_sign(2, leg) = sideSign of get_foot_jacobians_mc.m:3

// Row groups (what an input can reach): the Jacobian passes evaluate only the groups that depend on their input.
enum : unsigned { G_DYN = 1u, G_LEG0 = 2u, G_FRIC = 32u, G_Z = 64u, G_JPOS = 128u, G_ALL = 255u };
KHD constexpr unsigned reach(int v) {  // knot-local input -> row groups
  if (v < 6) return G_DYN | (15u * G_LEG0) | G_Z;          // r, rpy: dynamics, every leg's hip / torque / FK rows, z_k
  if (v < 12) return G_DYN;                                // omega, v
  if (v < 24) return (G_LEG0 << ((v - 12) / 3)) | G_JPOS;  // joint angles of one leg
  if (v < 36) return G_DYN | (G_LEG0 << ((v - 24) / 3));   // foot position of one leg
  if (v < 48) return G_DYN | (G_LEG0 << ((v - 36) / 3)) | G_FRIC;  // GRF of one leg
  if (v < 60) return G_DYN;                                // next state (identity entries of the dynamics rows)
  return G_LEG0 << ((v - 60) / 3);                         // next foot position: no-slip rows of one leg
}

// rows of one knot into out(rho, value).  Inputs by block, each with its own scalar type: r, e (rpy), w (omega_body),
// v | jp | c | f | Xn (next state) | cn (next foot positions); h = dt_k; only the row groups in mask are evaluated.
template <bool LAST, class Tr, class Te, class Tw, class Tv, class TJ, class TC, class TF, class TXn, class TCn, class Sink>
KHD void knot_rows_h(const Tr* r, const Te* e, const Tw* om, const Tv* vel, const TJ* jp, const TC* c, const TF* f,
                     const TXn* Xn, const TCn* cn, double h, const Params& pr, Sink& out, unsigned mask) {
  constexpr bool last = LAST;
  Te sr, cr, sp, cp, sy, cy;
  sincos_s(e[0], sr, cr);
  sincos_s(e[1], sp, cp);
  sincos_s(e[2], sy, cy);
  // body -> world, rpyToRotMat_xyz.m:2: R = rx(roll)' ry(pitch)' rz(yaw)'
  const Te R[9] = {cp * cy, -(cp * sy), sp,
                   cr * sy + sr * sp * cy, cr * cy - sr * sp * sy, -(sr * cp),
                   sr * sy - cr * sp * cy, sr * cy + cr * sp * sy, cr * cp};
  if (mask & G_DYN) {
    // dynamics (:119-131)
    using Td = Pr<TC, Tr>;            // c - r
    using Tq = Pr<Td, TF>;            // (c - r) x f
    TF fs[3] = {TF(0.0), TF(0.0), TF(0.0)};
    Tq tq[3] = {Tq(0.0), Tq(0.0), Tq(0.0)};
#pragma unroll
    for (int l = 0; l < 4; l++) {
      const Td d0 = c[3 * l] - r[0], d1 = c[3 * l + 1] - r[1], d2 = c[3 * l + 2] - r[2];
      const TF f0 = f[3 * l], f1 = f[3 * l + 1], f2 = f[3 * l + 2];
      fs[0] = fs[0] + f0; fs[1] = fs[1] + f1; fs[2] = fs[2] + f2;
      tq[0] = tq[0] + (d1 * f2 - d2 * f1);
      tq[1] = tq[1] + (d2 * f0 - d0 * f2);
      tq[2] = tq[2] + (d0 * f1 - d1 * f0);
    }
    const double grav[3] = {0.0, 0.0, -9.81};
#pragma unroll
    for (int i = 0; i < 3; i++) out(i, Xn[9 + i] - vel[i] - (fs[i] * (1.0 / pr.mass) + grav[i]) * h);
    {
      const Tw om0 = om[0], om1 = om[1], om2 = om[2];
      const Tw io0 = om0 * pr.Ib[0], io1 = om1 * pr.Ib[1], io2 = om2 * pr.Ib[2];
      const Tw cx[3] = {om1 * io2 - om2 * io1, om2 * io0 - om0 * io2, om0 * io1 - om1 * io0};
#pragma unroll
      for (int i = 0; i < 3; i++) {
        const auto rt = R[i] * tq[0] + R[3 + i] * tq[1] + R[6 + i] * tq[2];  // (R' tq)_i
        out(3 + i, Xn[6 + i] - om[i] - pr.Ib_inv[i] * (rt - cx[i]) * h);
      }
#pragma unroll
      for (int i = 0; i < 3; i++) out(6 + i, Xn[i] - r[i] - vel[i] * h);
      // Euler rates: Binv(rpy) (R omega), Binv.m:13-17 with psi = rpy(3), theta = rpy(2)
      const auto w0 = R[0] * om0 + R[1] * om1 + R[2] * om2, w1 = R[3] * om0 + R[4] * om1 + R[5] * om2,
                 w2 = R[6] * om0 + R[7] * om1 + R[8] * om2;
      const Te tanp = sp / cp;
      const auto e0 = (cy * w0 + sy * w1) / cp, e1 = cy * w1 - sy * w0, e2 = (cy * w0 + sy * w1) * tanp + w2;
      out(9, Xn[3] - e[0] - e0 * h);
      out(10, Xn[4] - e[1] - e1 * h);
      out(11, Xn[5] - e[2] - e2 * h);
    }
  }
  if (mask & G_FRIC) {
#pragma unroll
    for (int l = 0; l < 4; l++) out(12 + l, f[3 * l + 2]);
  }
  constexpr int per_leg = last ? 9 : 15;
  using Tfoot = Pr<Pr<Tr, Te>, TJ>;
  Tfoot foot[12];
#pragma unroll
  for (int l = 0; l < 4; l++) {
    if (!(mask & (G_LEG0 << l))) continue;
    int rho = 16 + per_leg * l;
    const TF fz = f[3 * l + 2];
    out(rho++, c[3 * l + 2]);
    out(rho++, fz * c[3 * l + 2]);
    if (!last) {
#pragma unroll
      for (int rep = 0; rep < 2; rep++)
#pragma unroll
        for (int i = 0; i < 3; i++) out(rho++, fz * (cn[3 * l + i] - c[3 * l + i]));
    }
    const double hx = hip_x(l), hy = hip_y(l);
    Pr<Pr<TC, Tr>, Te> p[3];
#pragma unroll
    for (int i = 0; i < 3; i++) p[i] = c[3 * l + i] - (r[i] + R[3 * i] * hx + R[3 * i + 1] * hy);
    out(rho++, p[0]);
    out(rho++, p[1]);
    out(rho++, p[2]);
    out(rho++, p[0] * p[0] + p[1] * p[1] + p[2] * p[2]);
    // leg kinematics
    TJ s1, c1, s2, c2, s3, c3;
    sincos_s(jp[3 * l], s1, c1);
    sincos_s(jp[3 * l + 1], s2, c2);
    sincos_s(jp[3 * l + 2], s3, c3);
    const TJ c23 = c2 * c3 - s2 * s3, s23 = s2 * c3 + c2 * s3;
    const double ss = side_y(l);
    // torque rows: tau = J_f' (-R' f)   (:168-173; J_f of get_foot_jacobians_mc.m:17-19, with its l_4 offset)
    {
      const auto fb0 = -(R[0] * f[3 * l] + R[3] * f[3 * l + 1] + R[6] * f[3 * l + 2]);
      const auto fb1 = -(R[1] * f[3 * l] + R[4] * f[3 * l + 1] + R[7] * f[3 * l + 2]);
      const auto fb2 = -(R[2] * f[3 * l] + R[5] * f[3 * l + 1] + R[8] * f[3 * l + 2]);
      const TJ a = L3 * c23 + L2 * c2, b = L3 * s23 + L2 * s2;
      const double l14 = (L1 + L4) * ss;
      const TJ J10 = c1 * a - s1 * l14, J20 = s1 * a + c1 * l14;
      const TJ J11 = -(s1 * b), J21 = c1 * b;
      const TJ J02 = L3 * c23, J12 = -(s1 * s23) * L3, J22 = c1 * s23 * L3;
      out(rho++, J10 * fb1 + J20 * fb2);            // (J(1,1) = 0)
      out(rho++, a * fb0 + J11 * fb1 + J21 * fb2);
      out(rho++, J02 * fb0 + J12 * fb1 + J22 * fb2);
    }
    // foot position by forward kinematics (get_forward_kin_foot.m:4-25, closed form; oracle/kino_ref.py: leg_fk_body)
    {
      const TJ a = L2 * c2 + L3 * c23, b = L2 * s2 + L3 * s23;
      const TJ pb0 = (l < 2 ? ABAD_X : -ABAD_X) + b;
      const TJ pb1 = (ss * ABAD_Y) + (ss * L1) * c1 + a * s1;
      const TJ pb2 = (ss * L1) * s1 - a * c1;
#pragma unroll
      for (int i = 0; i < 3; i++) foot[3 * l + i] = r[i] + R[3 * i] * pb0 + R[3 * i + 1] * pb1 + R[3 * i + 2] * pb2;
    }
  }
  int rho = 16 + 4 * per_leg;
  const double km = 0.71 * pr.mu;
  if (mask & G_FRIC) {
#pragma unroll
    for (int l = 0; l < 4; l++) out(rho + l, f[3 * l] - km * f[3 * l + 2]);
#pragma unroll
    for (int l = 0; l < 4; l++) out(rho + 4 + l, -(km * f[3 * l + 2]) - f[3 * l]);
#pragma unroll
    for (int l = 0; l < 4; l++) out(rho + 8 + l, f[3 * l + 1] - km * f[3 * l + 2]);
#pragma unroll
    for (int l = 0; l < 4; l++) out(rho + 12 + l, -(km * f[3 * l + 2]) - f[3 * l + 1]);
  }
  rho += 16;
  if (mask & G_Z) out(rho, r[2]);
  rho++;
#pragma unroll
  for (int i = 0; i < 12; i++) {
    if (!(mask & (G_LEG0 << (i / 3)))) continue;
    const auto d = c[i] - foot[i];
    out(rho + i, d);
    out(rho + 12 + i, d);
  }
  rho += 24;
  if (mask & G_JPOS) {
#pragma unroll
    for (int i = 0; i < 12; i++) {
      out(rho + i, jp[i]);
      out(rho + 12 + i, jp[i]);
    }
  }
}

// one scalar type for all 72 knot-local inputs
template <bool LAST, class S, class Sink>
KHD void knot_rows_t(const S* in, double h, const Params& pr, Sink& out, unsigned mask = G_ALL) {
  knot_rows_h<LAST>(in, in + 3, in + 6, in + 9, in + 12, in + 24, in + 36, in + 48, in + 60, h, pr, out, mask);
}

// run-time knot class
template <class S, class Sink>
KHD void knot_rows(const S* in, double h, const Params& pr, bool last, Sink& out, unsigned mask = G_ALL) {
  if (last) knot_rows_t<true, S, Sink>(in, h, pr, out, mask);
  else knot_rows_t<false, S, Sink>(in, h, pr, out, mask);
}

// Jacobian passes.  A pass seeds one triple of knot-local inputs (three tangents: r | rpy | omega | v | the
// joint angles, foot position, force, next foot position of one leg | a triple of the next state) and runs the knot
// function with that block typed DualN<3> and every other block a plain double, restricted to the row groups the triple
// can reach; the rpy triple, which reaches every leg's rows through R, is split into five passes (dynamics, four legs).
// Together the passes emit every non-zero of dg/dz exactly once (tests/test_kino_host.py checks this on the host).
constexpr int JAC_PASSES = 28;
template <int G> struct PassOf {  // pass -> (first seeded input, row groups)
  static constexpr int v0 = G < 24 ? 3 * G : 3;
  static constexpr unsigned mask = G == 1 ? G_DYN : G >= 24 ? (G_LEG0 << (G - 24)) : reach(3 * G);
};
KHD constexpr bool pass_in_knot(bool last, int G) { return !(last && G >= 20 && G < 24); }  // (no c_{k+1} in the last knot)

// Pass G on the knot-local inputs x: out(rho, DualN<3>) gets d row / d x[v0 + j] as tangent j (out(rho, double): a row
// that does not depend on the triple).
template <bool LAST, int G, class Sink>
KHD void jac_pass(const double* x, double h, const Params& pr, Sink& s) {
  using D = DualN<3>;
  constexpr int v0 = PassOf<G>::v0, blk = v0 < 12 ? v0 / 3 : v0 < 24 ? 4 : v0 < 36 ? 5 : v0 < 48 ? 6 : v0 < 60 ? 7 : 8;
  constexpr unsigned mask = PassOf<G>::mask;
  if constexpr (blk < 4) {  // a triple of X_k
    D t[3];
#pragma unroll
    for (int j = 0; j < 3; j++) t[j] = seeded<3>(x[v0 + j], j);
    if constexpr (blk == 0) knot_rows_h<LAST>(t, x + 3, x + 6, x + 9, x + 12, x + 24, x + 36, x + 48, x + 60, h, pr, s, mask);
    if constexpr (blk == 1) knot_rows_h<LAST>(x, t, x + 6, x + 9, x + 12, x + 24, x + 36, x + 48, x + 60, h, pr, s, mask);
    if constexpr (blk == 2) knot_rows_h<LAST>(x, x + 3, t, x + 9, x + 12, x + 24, x + 36, x + 48, x + 60, h, pr, s, mask);
    if constexpr (blk == 3) knot_rows_h<LAST>(x, x + 3, x + 6, t, x + 12, x + 24, x + 36, x + 48, x + 60, h, pr, s, mask);
  } else {  // a triple of a 12-block: the block as duals, tangents on the triple
    constexpr int base = 12 * (blk - 3), off = v0 - base;
    D t[12];
#pragma unroll
    for (int i = 0; i < 12; i++) t[i] = (i >= off && i < off + 3) ? seeded<3>(x[base + i], i - off) : D(x[base + i]);
    if constexpr (blk == 4) knot_rows_h<LAST>(x, x + 3, x + 6, x + 9, t, x + 24, x + 36, x + 48, x + 60, h, pr, s, mask);
    if constexpr (blk == 5) knot_rows_h<LAST>(x, x + 3, x + 6, x + 9, x + 12, t, x + 36, x + 48, x + 60, h, pr, s, mask);
    if constexpr (blk == 6) knot_rows_h<LAST>(x, x + 3, x + 6, x + 9, x + 12, x + 24, t, x + 48, x + 60, h, pr, s, mask);
    if constexpr (blk == 7) knot_rows_h<LAST>(x, x + 3, x + 6, x + 9, x + 12, x + 24, x + 36, t, x + 60, h, pr, s, mask);
    if constexpr (blk == 8) knot_rows_h<LAST>(x, x + 3, x + 6, x + 9, x + 12, x + 24, x + 36, x + 48, t, h, pr, s, mask);
  }
}

// Hessian passes.  Triples of knot-local inputs: 0 r | 1 rpy | 2 omega | 3 v | 4 + l joint angles, 8 + l foot position,
// 12 + l force of leg l | 16..19 next state | 20 + l next foot position.  A pass is an ordered pair of triples (a <= b)
// whose cross block d2 L / dz_a dz_b is non-zero somewhere: it runs the knot function with the block(s) of the two
// triples typed Dual2 (seeds A on a, B on b), restricted to the row groups both triples reach, and owns the 3 x 3 block
// (its upper triangle when a == b).  The table is grouped by weight (the kernels of kino_hess.cu): the pairs with rpy,
// whose rotation matrix makes every row second order; the joint-angle pairs; the rest.  The host plan derives the
// non-zero pairs by probing every one of the 300 triple pairs and refuses a table that misses one.
constexpr int HESS_PASSES = 45, HESS_RPY_END = 15, HESS_JPOS_END = 23;
KHD constexpr int hess_pair(int P) {  // pass -> 32 a + b
  constexpr int t[HESS_PASSES] = {
      // [0, 15): with rpy -- r, rpy, omega, and the joint angles, foot position and force of each leg
      0 * 32 + 1, 1 * 32 + 1, 1 * 32 + 2, 1 * 32 + 4, 1 * 32 + 5, 1 * 32 + 6, 1 * 32 + 7, 1 * 32 + 8, 1 * 32 + 9,
      1 * 32 + 10, 1 * 32 + 11, 1 * 32 + 12, 1 * 32 + 13, 1 * 32 + 14, 1 * 32 + 15,
      // [15, 23): joint angles x joint angles, joint angles x force, by leg
      4 * 32 + 4, 4 * 32 + 12, 5 * 32 + 5, 5 * 32 + 13, 6 * 32 + 6, 6 * 32 + 14, 7 * 32 + 7, 7 * 32 + 15,
      // [23, 45): r x r, r x foot position, r x force, omega x omega, and per leg foot position x foot position,
      // foot position x force, force x next foot position
      0 * 32 + 0, 0 * 32 + 8, 0 * 32 + 9, 0 * 32 + 10, 0 * 32 + 11, 0 * 32 + 12, 0 * 32 + 13, 0 * 32 + 14, 0 * 32 + 15,
      2 * 32 + 2, 8 * 32 + 8, 8 * 32 + 12, 9 * 32 + 9, 9 * 32 + 13, 10 * 32 + 10, 10 * 32 + 14, 11 * 32 + 11,
      11 * 32 + 15, 12 * 32 + 20, 13 * 32 + 21, 14 * 32 + 22, 15 * 32 + 23};
  return t[P];
}
KHD constexpr int tri_block(int t) { return t < 4 ? t : t < 8 ? 4 : t < 12 ? 5 : t < 16 ? 6 : t < 20 ? 7 : 8; }
KHD constexpr int block_base(int blk) { return blk < 4 ? 3 * blk : 12 * (blk - 3); }
template <int P> struct HessPassOf {  // pass -> (triples a <= b, row groups both reach)
  static constexpr int a = hess_pair(P) / 32, b = hess_pair(P) % 32;
  static constexpr unsigned mask = reach(3 * a) & reach(3 * b);
};
KHD constexpr bool hess_pass_in_knot(bool last, int P) { return !(last && hess_pair(P) % 32 >= 20); }  // (no c_{k+1})

// One input block of a Hessian pass: the caller's doubles, or -- if the block holds triple a or b -- a Dual2 copy seeded
// with tangent A_i on element i of triple a and B_j on element j of triple b.
template <int BLK, int TA, int TB> struct HessBlock {
  static constexpr bool typed = tri_block(TA) == BLK || tri_block(TB) == BLK;
  static constexpr int base = block_base(BLK), len = BLK < 4 ? 3 : 12;
  using T = typename std::conditional<typed, Dual2, double>::type;
  T buf[typed ? len : 1];
  const T* p;
  KHD explicit HessBlock(const double* x) {
    if constexpr (typed) {
#pragma unroll
      for (int i = 0; i < len; i++) {
        buf[i] = Dual2(x[base + i]);
        if ((base + i) / 3 == TA) buf[i].a[(base + i) % 3] = 1.0;
        if ((base + i) / 3 == TB) buf[i].b[(base + i) % 3] = 1.0;
      }
      p = buf;
    } else {
      p = x + base;
    }
  }
};

// Pass P on the knot-local inputs x: out(rho, Dual2) gets d2 row / dz_{3a+i} dz_{3b+j} as h[i][j] (out(rho, double): a
// row that depends on neither triple).
template <bool LAST, int P, class Sink>
KHD void hess_pass(const double* x, double h, const Params& pr, Sink& s) {
  constexpr int A = HessPassOf<P>::a, B = HessPassOf<P>::b;
  const HessBlock<0, A, B> b0(x);
  const HessBlock<1, A, B> b1(x);
  const HessBlock<2, A, B> b2(x);
  const HessBlock<3, A, B> b3(x);
  const HessBlock<4, A, B> b4(x);
  const HessBlock<5, A, B> b5(x);
  const HessBlock<6, A, B> b6(x);
  const HessBlock<7, A, B> b7(x);
  const HessBlock<8, A, B> b8(x);
  knot_rows_h<LAST>(b0.p, b1.p, b2.p, b3.p, b4.p, b5.p, b6.p, b7.p, b8.p, h, pr, s, HessPassOf<P>::mask);
}

// Which thread of a (scenario, knot) quadruple owns row rho when the knot is split by leg (k_kino_g): the rows of leg l
// (contact, hip box, leg length, torques, foot kinematics, joint limits of that leg) belong to part l, everything else
// (dynamics, f_z, friction, z) to part 0.  constexpr: behind a filtering sink the compiler drops what a part never emits.
template <bool LAST> KHD constexpr int row_owner(int rho) {
  constexpr int per_leg = LAST ? 9 : 15, legs_end = 16 + 4 * per_leg, fk = legs_end + 17;
  if (rho < 16) return 0;
  if (rho < legs_end) return (rho - 16) / per_leg;
  if (rho < fk) return 0;                                   // friction, z
  if (rho < fk + 24) return ((rho - fk) % 12) / 3;          // c - FK (12, twice)
  return ((rho - fk - 24) % 12) / 3;                        // joint angles (12, twice)
}

}  // namespace kino
}  // namespace srb
