// pn_problems.cuh -- the reference's IVP zoo (src/odecheckpts/ivps.py) as device functors.
//
// The reference hands JAX-traceable Python callables to probdiffeq, which differentiates them
// (Jacobian for correction_ts1: experiments/1_van_der_pol/vdp.py:64; Taylor-mode jets for
// taylor.odejet_padded_scan: src/odecheckpts/ivpsolvers.py:63-67).  Here each problem is a
// struct with
//   D, Q, P           ODE dimension, ODE order, number of parameters
//   vf(u, par, f)     u = (u, u', ...)[Q*D]  ->  f[D]
//   jac(u, par, J)    J[D][Q*D]  (HAS_JAC)
//   vf_jet<N>(U, par, F)  the same expression on truncated power series (normalised Taylor
//                     coefficients), used once per member for the initial state.
//   TIME              optional, false when absent: the problem is time-dependent and its functions take
//                     the time after the state: vf(u, t, par, f), jac(u, t, par, J) and vf_jet<N>(U, Tc, par, F)
//                     with Tc[N] the time's normalised Taylor coefficients.  The kernels call the three through
//                     vf_at / jac_at / taylor_init, which pass the time to a time-dependent problem only.
// Fixed-size problems only; the Brusselator (d = 2N) lives in the CTA-per-IVP kernel.
#pragma once
#include "pn_math.cuh"

namespace pn {

PN_DEV double inv_pow32(double s) { return rcp(s * dsqrt(s)); }  // s^(-3/2)

// ---- truncated power series of length N -------------------------------------------------
template <int N>
PN_DEV void jet_mul(const double* a, const double* b, double* out) {
#pragma unroll
  for (int k = 0; k < N; ++k) {
    double acc = a[0] * b[k];
#pragma unroll
    for (int j = 1; j <= k; ++j) acc = fma(a[j], b[k - j], acc);
    out[k] = acc;
  }
}
template <int N>
PN_DEV void jet_inv_pow32(const double* s, double* out) {
  out[0] = inv_pow32(s[0]);
#pragma unroll
  for (int k = 1; k < N; ++k) {
    double acc = 0.0;
#pragma unroll
    for (int j = 1; j <= k; ++j) {
      double coef = -1.5 * (double)j - (double)(k - j);
      acc = fma(coef * s[j], out[k - j], acc);
    }
    out[k] = acc / ((double)k * s[0]);
  }
}

// ---- logistic: u' = a u (1 - b u)   (ivps.py:8-17) --------------------------------------
struct Logistic {
  static constexpr int D = 1, Q = 1, P = 2, ID = 0;
  static constexpr bool HAS_JAC = true;
  PN_DEV static void vf(const double* u, const double* par, double* f) {
    f[0] = (par[0] * u[0]) * fma(-par[1], u[0], 1.0);
  }
  PN_DEV static void jac(const double* u, const double* par, double* J) {
    J[0] = par[0] * fma(-2.0 * par[1], u[0], 1.0);
  }
  template <int N>
  PN_DEV static void vf_jet(const double* U, const double* par, double* F) {
    double au[N], w[N];
#pragma unroll
    for (int k = 0; k < N; ++k) {
      au[k] = par[0] * U[k];
      w[k] = fma(-par[1], U[k], (k == 0) ? 1.0 : 0.0);
    }
    jet_mul<N>(au, w, F);
  }
};

// ---- rigid body (ivps.py:20-29; diffeqzoo) ------------------------------------------------
struct RigidBody {
  static constexpr int D = 3, Q = 1, P = 3, ID = 1;
  static constexpr bool HAS_JAC = true;
  PN_DEV static void vf(const double* u, const double* par, double* f) {
    f[0] = par[0] * (u[1] * u[2]);
    f[1] = par[1] * (u[0] * u[2]);
    f[2] = par[2] * (u[0] * u[1]);
  }
  PN_DEV static void jac(const double* u, const double* par, double* J) {
    J[0] = 0.0;             J[1] = par[0] * u[2];   J[2] = par[0] * u[1];
    J[3] = par[1] * u[2];   J[4] = 0.0;             J[5] = par[1] * u[0];
    J[6] = par[2] * u[1];   J[7] = par[2] * u[0];   J[8] = 0.0;
  }
  template <int N>
  PN_DEV static void vf_jet(const double* U, const double* par, double* F) {
    double pr[N];
    jet_mul<N>(U + 1 * N, U + 2 * N, pr);
#pragma unroll
    for (int k = 0; k < N; ++k) F[0 * N + k] = par[0] * pr[k];
    jet_mul<N>(U + 0 * N, U + 2 * N, pr);
#pragma unroll
    for (int k = 0; k < N; ++k) F[1 * N + k] = par[1] * pr[k];
    jet_mul<N>(U + 0 * N, U + 1 * N, pr);
#pragma unroll
    for (int k = 0; k < N; ++k) F[2 * N + k] = par[2] * pr[k];
  }
};

// ---- Lotka-Volterra (diffeqzoo) --------------------------------------------------------------
struct LotkaVolterra {
  static constexpr int D = 2, Q = 1, P = 4, ID = 6;
  static constexpr bool HAS_JAC = true;
  PN_DEV static void vf(const double* u, const double* par, double* f) {
    double uv = u[0] * u[1];
    f[0] = fma(-par[1], uv, par[0] * u[0]);
    f[1] = fma(par[3], uv, -(par[2] * u[1]));
  }
  PN_DEV static void jac(const double* u, const double* par, double* J) {
    J[0] = fma(-par[1], u[1], par[0]);  J[1] = -(par[1] * u[0]);
    J[2] = par[3] * u[1];               J[3] = fma(par[3], u[0], -par[2]);
  }
  template <int N>
  PN_DEV static void vf_jet(const double* U, const double* par, double* F) {
    double uv[N];
    jet_mul<N>(U, U + N, uv);
#pragma unroll
    for (int k = 0; k < N; ++k) {
      F[k] = fma(-par[1], uv[k], par[0] * U[k]);
      F[N + k] = fma(par[3], uv[k], -(par[2] * U[N + k]));
    }
  }
};

// ---- Van der Pol, second order: u'' = mu (u' (1 - u^2) - u)   (ivps.py:159-167) ---------
struct VanDerPol {
  static constexpr int D = 1, Q = 2, P = 1, ID = 5;
  static constexpr bool HAS_JAC = true;
  PN_DEV static void vf(const double* u, const double* par, double* f) {
    double y = u[0], yd = u[1];
    f[0] = par[0] * fma(yd, fma(-y, y, 1.0), -y);
  }
  PN_DEV static void jac(const double* u, const double* par, double* J) {
    double y = u[0], yd = u[1];
    J[0] = par[0] * fma(-2.0 * y, yd, -1.0);
    J[1] = par[0] * fma(-y, y, 1.0);
  }
  template <int N>
  PN_DEV static void vf_jet(const double* U, const double* par, double* F) {
    const double* y = U;
    const double* yd = U + N;
    double yy[N], w[N], pr[N];
    jet_mul<N>(y, y, yy);
    w[0] = fma(-y[0], y[0], 1.0);
#pragma unroll
    for (int k = 1; k < N; ++k) w[k] = -yy[k];
    jet_mul<N>(yd, w, pr);
    F[0] = par[0] * fma(yd[0], w[0], -y[0]);
#pragma unroll
    for (int k = 1; k < N; ++k) F[k] = par[0] * (pr[k] - y[k]);
  }
};

// ---- restricted three-body problem, second order (ivps.py:32-41; diffeqzoo) -------------
struct ThreeBody {
  static constexpr int D = 2, Q = 2, P = 1, ID = 2;
  static constexpr bool HAS_JAC = true;
  PN_DEV static void vf(const double* u, const double* par, double* f) {
    double mu = par[0], mp = 1.0 - mu;
    double x = u[0], y = u[1], xd = u[2], yd = u[3];
    double a = x + mu, b = x - mp;
    double p1 = inv_pow32(fma(y, y, a * a));
    double p2 = inv_pow32(fma(y, y, b * b));
    f[0] = fma(-mu, b * p2, fma(-mp, a * p1, fma(2.0, yd, x)));
    f[1] = fma(-mu, y * p2, fma(-mp, y * p1, fma(-2.0, xd, y)));
  }
  // columns (x, y, x', y'); p = s^(-3/2), dp/d(a or y) = q (a or y) with q = -3 p / s
  PN_DEV static void jac(const double* u, const double* par, double* J) {
    double mu = par[0], mp = 1.0 - mu;
    double x = u[0], y = u[1];
    double a = x + mu, b = x - mp;
    double s1 = fma(y, y, a * a), s2 = fma(y, y, b * b);
    double p1 = inv_pow32(s1), p2 = inv_pow32(s2);
    double q1 = (-3.0 * p1) * rcp(s1), q2 = (-3.0 * p2) * rcp(s2);
    J[0] = 1.0 - fma(mu, fma(b * b, q2, p2), mp * fma(a * a, q1, p1));
    J[1] = -fma(mu, (b * y) * q2, mp * ((a * y) * q1));
    J[2] = 0.0;
    J[3] = 2.0;
    J[4] = J[1];
    J[5] = 1.0 - fma(mu, fma(y * y, q2, p2), mp * fma(y * y, q1, p1));
    J[6] = -2.0;
    J[7] = 0.0;
  }
  template <int N>
  PN_DEV static void vf_jet(const double* U, const double* par, double* F) {
    double mu = par[0], mp = 1.0 - mu;
    const double *x = U, *y = U + N, *xd = U + 2 * N, *yd = U + 3 * N;
    double a[N], b[N], s1[N], s2[N], p1[N], p2[N], t1[N], t2[N], yy[N];
#pragma unroll
    for (int k = 0; k < N; ++k) {
      a[k] = (k == 0) ? x[0] + mu : x[k];
      b[k] = (k == 0) ? x[0] - mp : x[k];
    }
    jet_mul<N>(y, y, yy);
    jet_mul<N>(a, a, t1);
    jet_mul<N>(b, b, t2);
    s1[0] = fma(y[0], y[0], a[0] * a[0]);
    s2[0] = fma(y[0], y[0], b[0] * b[0]);
#pragma unroll
    for (int k = 1; k < N; ++k) {
      s1[k] = yy[k] + t1[k];
      s2[k] = yy[k] + t2[k];
    }
    jet_inv_pow32<N>(s1, p1);
    jet_inv_pow32<N>(s2, p2);
    jet_mul<N>(a, p1, t1);
    jet_mul<N>(b, p2, t2);
#pragma unroll
    for (int k = 0; k < N; ++k) F[k] = fma(-mu, t2[k], fma(-mp, t1[k], fma(2.0, yd[k], x[k])));
    jet_mul<N>(y, p1, t1);
    jet_mul<N>(y, p2, t2);
#pragma unroll
    for (int k = 0; k < N; ++k) F[N + k] = fma(-mu, t2[k], fma(-mp, t1[k], fma(-2.0, xd[k], y[k])));
  }
};

// ---- Pleiades, second order: 7 bodies, masses 1..7 (ivps.py:59-99) ------------------------
// u = (x[7], y[7]);  a_i = sum_{j != i} m_j (r_j - r_i) / |r_j - r_i|^3
struct Pleiades {
  static constexpr int D = 14, Q = 2, P = 0, ID = 3;
  static constexpr bool HAS_JAC = false;
  PN_DEV static void vf(const double* u, const double*, double* f) {
    const double *x = u, *y = u + 7;
#pragma unroll
    for (int i = 0; i < 7; ++i) {
      double ax = 0.0, ay = 0.0;
#pragma unroll
      for (int j = 0; j < 7; ++j) {
        if (j == i) continue;
        double dx = x[j] - x[i], dy = y[j] - y[i];
        double p = inv_pow32(fma(dy, dy, dx * dx));
        ax = fma((double)(j + 1), p * dx, ax);
        ay = fma((double)(j + 1), p * dy, ay);
      }
      f[i] = ax;
      f[7 + i] = ay;
    }
  }
  PN_DEV static void jac(const double*, const double*, double*) {}
  template <int N>
  PN_DEV static void vf_jet(const double* U, const double*, double* F) {
    const double *x = U, *y = U + 7 * N;
    for (int i = 0; i < 7; ++i) {
      double* ax = F + i * N;
      double* ay = F + (7 + i) * N;
      for (int k = 0; k < N; ++k) ax[k] = ay[k] = 0.0;
      for (int j = 0; j < 7; ++j) {
        if (j == i) continue;
        double dx[N], dy[N], s[N], p[N], t1[N], t2[N];
        const double mj = (double)(j + 1);
        for (int k = 0; k < N; ++k) {
          dx[k] = x[j * N + k] - x[i * N + k];
          dy[k] = y[j * N + k] - y[i * N + k];
        }
        jet_mul<N>(dx, dx, t1);
        jet_mul<N>(dy, dy, t2);
        s[0] = fma(dy[0], dy[0], dx[0] * dx[0]);
        for (int k = 1; k < N; ++k) s[k] = t2[k] + t1[k];
        jet_inv_pow32<N>(s, p);
        jet_mul<N>(p, dx, t1);
        jet_mul<N>(p, dy, t2);
        for (int k = 0; k < N; ++k) {
          ax[k] = fma(mj, t1[k], ax[k]);
          ay[k] = fma(mj, t2[k], ay[k]);
        }
      }
    }
  }
};

// ---- Brusselator with N grid points, d = 2N (ivps.py:124-156); params (alpha) ---------------
// u = (u[N], v[N]); boundary pads u = 1, v = 3; c = alpha (N+1)^2.  Fixed small N only (lane per
// dimension); large N runs in the warp-per-IVP kernel (pn_wide_kernel.cuh).
template <int NPTS>
struct Brusselator {
  static constexpr int D = 2 * NPTS, Q = 1, P = 1, ID = 4;
  static constexpr bool HAS_JAC = true;
  PN_DEV static void vf(const double* u, const double* par, double* f) {
    const double c = par[0] * (double)((NPTS + 1) * (NPTS + 1));
    const double *uu = u, *vv = u + NPTS;
#pragma unroll
    for (int i = 0; i < NPTS; ++i) {
      double ul = (i == 0) ? 1.0 : uu[i - 1], ur = (i == NPTS - 1) ? 1.0 : uu[i + 1];
      double vl = (i == 0) ? 3.0 : vv[i - 1], vr = (i == NPTS - 1) ? 3.0 : vv[i + 1];
      double uuv = (uu[i] * uu[i]) * vv[i];
      double lap_u = fma(-2.0, uu[i], ul + ur);
      double lap_v = fma(-2.0, vv[i], vl + vr);
      f[i] = fma(c, lap_u, fma(-4.0, uu[i], 1.0 + uuv));
      f[NPTS + i] = fma(c, lap_v, fma(3.0, uu[i], -uuv));
    }
  }
  PN_DEV static void jac(const double* u, const double* par, double* J) {
    const double c = par[0] * (double)((NPTS + 1) * (NPTS + 1));
    const double *uu = u, *vv = u + NPTS;
    for (int e = 0; e < D * D; ++e) J[e] = 0.0;
    for (int i = 0; i < NPTS; ++i) {
      const double two_uv = (2.0 * uu[i]) * vv[i];
      const double u2 = uu[i] * uu[i];
      J[i * D + i] = fma(-2.0, c, two_uv - 4.0);
      J[i * D + NPTS + i] = u2;
      J[(NPTS + i) * D + i] = 3.0 - two_uv;
      J[(NPTS + i) * D + NPTS + i] = fma(-2.0, c, -u2);
      if (i > 0) {
        J[i * D + i - 1] = c;
        J[(NPTS + i) * D + NPTS + i - 1] = c;
      }
      if (i < NPTS - 1) {
        J[i * D + i + 1] = c;
        J[(NPTS + i) * D + NPTS + i + 1] = c;
      }
    }
  }
  template <int N>
  PN_DEV static void vf_jet(const double* U, const double* par, double* F) {
    const double c = par[0] * (double)((NPTS + 1) * (NPTS + 1));
    for (int i = 0; i < NPTS; ++i) {
      const double* ui = U + i * N;
      const double* vi = U + (NPTS + i) * N;
      double u2[N], uuv[N];
      jet_mul<N>(ui, ui, u2);
      jet_mul<N>(u2, vi, uuv);
      for (int k = 0; k < N; ++k) {
        double padu = (k == 0) ? 1.0 : 0.0, padv = (k == 0) ? 3.0 : 0.0;
        double ul = (i == 0) ? padu : U[(i - 1) * N + k];
        double ur = (i == NPTS - 1) ? padu : U[(i + 1) * N + k];
        double vl = (i == 0) ? padv : U[(NPTS + i - 1) * N + k];
        double vr = (i == NPTS - 1) ? padv : U[(NPTS + i + 1) * N + k];
        double lap_u = fma(-2.0, ui[k], ul + ur);
        double lap_v = fma(-2.0, vi[k], vl + vr);
        F[i * N + k] = fma(c, lap_u, fma(-4.0, ui[k], padu + uuv[k]));
        F[(NPTS + i) * N + k] = fma(c, lap_v, fma(3.0, ui[k], -uuv[k]));
      }
    }
  }
};

// Brusselator with a RUNTIME grid size (CTA-per-IVP "wide" kernel): the vector field and the Taylor
// initialisation are written out inside the kernel (they need the CTA's shared staging buffers);
// this tag only carries the compile-time facts.  D is a dummy register column.
struct BrusselatorWide {
  static constexpr int D = 1, Q = 1, P = 1, ID = 4;
  static constexpr bool HAS_JAC = false;
  PN_DEV static void vf(const double*, const double*, double* f) { f[0] = 0.0; }
  PN_DEV static void jac(const double*, const double*, double*) {}
  template <int N>
  PN_DEV static void vf_jet(const double*, const double*, double* F) {
#pragma unroll
    for (int k = 0; k < N; ++k) F[k] = 0.0;
  }
};

// ---- time-dependent problems (TIME) ------------------------------------------------------
template <class Prob, class = void>
struct TimeDependent {
  static constexpr bool value = false;
};
template <class Prob>
struct TimeDependent<Prob, decltype(void(Prob::TIME))> {
  static constexpr bool value = Prob::TIME;
};
template <class Prob>
PN_DEV void vf_at(const double* u, double t, const double* par, double* f) {
  if constexpr (TimeDependent<Prob>::value)
    Prob::vf(u, t, par, f);
  else
    Prob::vf(u, par, f);
}
template <class Prob>
PN_DEV void jac_at(const double* u, double t, const double* par, double* J) {
  if constexpr (TimeDependent<Prob>::value)
    Prob::jac(u, t, par, J);
  else
    Prob::jac(u, par, J);
}

// taylor.odejet_padded_scan replacement: tc[k][l] = u_l^{(k)}(t0), k = 0..NU.  A time-dependent field sees the
// time as the series t0 + (t - t0), coefficients (t0, 1, 0, ...): the recursion then yields the exact derivatives
// of a non-autonomous ODE, where a time frozen at t0 would leave all but the first derivative wrong.
template <class Prob, int NU>
PN_DEV void taylor_init(const double* u0 /*[Q*D]*/, double t0, const double* par, double (&tc)[NU + 1][Prob::D]) {
  constexpr int N = NU + 1, D = Prob::D, Q = Prob::Q;
  double C[D * N], U[Q * D * N], F[D * N];
#pragma unroll
  for (int i = 0; i < D * N; ++i) C[i] = 0.0;
#pragma unroll
  for (int l = 0; l < D; ++l) {
    C[l * N] = u0[l];
    if (Q == 2) C[l * N + 1] = u0[D + l];
  }
#pragma unroll
  for (int k = 0; k + Q <= NU; ++k) {
#pragma unroll
    for (int l = 0; l < D; ++l) {
#pragma unroll
      for (int i = 0; i < N; ++i) U[l * N + i] = C[l * N + i];
      if (Q == 2) {
#pragma unroll
        for (int i = 0; i < N; ++i) U[(D + l) * N + i] = (i + 1 < N) ? (double)(i + 1) * C[l * N + i + 1] : 0.0;
      }
    }
    if constexpr (TimeDependent<Prob>::value) {
      double Tc[N];
#pragma unroll
      for (int i = 0; i < N; ++i) Tc[i] = (i == 0) ? t0 : ((i == 1) ? 1.0 : 0.0);
      Prob::template vf_jet<N>(U, Tc, par, F);
    } else {
      Prob::template vf_jet<N>(U, par, F);
    }
#pragma unroll
    for (int l = 0; l < D; ++l) {
      if (Q == 1)
        C[l * N + k + 1] = F[l * N + k] / (double)(k + 1);
      else
        C[l * N + k + 2] = F[l * N + k] / (double)((k + 2) * (k + 1));
    }
  }
  double fact = 1.0;
#pragma unroll
  for (int k = 0; k <= NU; ++k) {
    if (k > 0) fact *= (double)k;
#pragma unroll
    for (int l = 0; l < D; ++l) tc[k][l] = fact * C[l * N + k];
  }
}

}  // namespace pn
