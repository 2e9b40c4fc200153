// pn_user_problem.cuh -- user-defined vector fields, compiled at run time (pn_jit.cu) into the same kernel
// templates the built-in problems of pn_problems.cuh use.
//
// A user writes the vector field once, templated on the number type:
//   template <class T> PN_DEV void vf(const T* u, const double* p, T* f)     u = (u, u', ...)[Q*D] -> f[D]
// and optionally  PN_DEV void jac(const double* u, const double* p, double* J)   J[D][Q*D].
// A time-dependent field (registered with PN_B200_FORM_TIME_DEPENDENT) takes the time after the state:
//   template <class T> PN_DEV void vf(const T* u, const T& t, const double* p, T* f)
//   PN_DEV void jac(const double* u, double t, const double* p, double* J)
// UserProblem evaluates it on doubles for the step, on truncated Taylor series (Jet<N>) for the Taylor-mode
// initialisation, and -- when the user gives no Jacobian -- on Jet<2> once per state column for the Jacobian.
//
// Jet<N> holds normalised Taylor coefficients c[k] = x^(k)(t0) / k!, the layout vf_jet uses.  Every recurrence
// keeps the built-ins' style: explicit fma, coefficient 0 computed exactly as the scalar function would be.
#pragma once
#include "pn_problems.cuh"

namespace pn {
namespace jet {

template <int N>
struct Jet {
  double c[N];
  Jet() = default;
  PN_DEV Jet(double v) {
    c[0] = v;
#pragma unroll
    for (int k = 1; k < N; ++k) c[k] = 0.0;
  }
};

template <class T>
struct JetOrder {
  static constexpr int value = 0;
};
template <int N>
struct JetOrder<Jet<N>> {
  static constexpr int value = N;
};
template <class A, class B, class C>
struct JetResult {
  static constexpr int NA = JetOrder<A>::value, NB = JetOrder<B>::value, NC = JetOrder<C>::value;
  static constexpr int N = NA > NB ? (NA > NC ? NA : NC) : (NB > NC ? NB : NC);
};
template <class A, class B>
struct IsSame {
  static constexpr bool value = false;
};
template <class A>
struct IsSame<A, A> {
  static constexpr bool value = true;
};
template <bool B, class T>
struct EnableIf {};
template <class T>
struct EnableIf<true, T> {
  using type = T;
};

template <int N>
PN_DEV double coef(const Jet<N>& x, int k) { return x.c[k]; }
PN_DEV double coef(double x, int k) { return k == 0 ? x : 0.0; }

// ---- + - ------------------------------------------------------------------------------------------------------
template <int N>
PN_DEV Jet<N> operator+(const Jet<N>& a, const Jet<N>& b) {
  Jet<N> r;
#pragma unroll
  for (int k = 0; k < N; ++k) r.c[k] = a.c[k] + b.c[k];
  return r;
}
template <int N>
PN_DEV Jet<N> operator+(const Jet<N>& a, double b) {
  Jet<N> r = a;
  r.c[0] = a.c[0] + b;
  return r;
}
template <int N>
PN_DEV Jet<N> operator+(double a, const Jet<N>& b) {
  Jet<N> r = b;
  r.c[0] = a + b.c[0];
  return r;
}
template <int N>
PN_DEV Jet<N> operator-(const Jet<N>& a) {
  Jet<N> r;
#pragma unroll
  for (int k = 0; k < N; ++k) r.c[k] = -a.c[k];
  return r;
}
template <int N>
PN_DEV Jet<N> operator-(const Jet<N>& a, const Jet<N>& b) {
  Jet<N> r;
#pragma unroll
  for (int k = 0; k < N; ++k) r.c[k] = a.c[k] - b.c[k];
  return r;
}
template <int N>
PN_DEV Jet<N> operator-(const Jet<N>& a, double b) {
  Jet<N> r = a;
  r.c[0] = a.c[0] - b;
  return r;
}
template <int N>
PN_DEV Jet<N> operator-(double a, const Jet<N>& b) {
  Jet<N> r = -b;
  r.c[0] = a - b.c[0];
  return r;
}

// ---- * / ------------------------------------------------------------------------------------------------------
template <int N>
PN_DEV Jet<N> operator*(const Jet<N>& a, const Jet<N>& b) {
  Jet<N> r;
  jet_mul<N>(a.c, b.c, r.c);
  return r;
}
template <int N>
PN_DEV Jet<N> operator*(const Jet<N>& a, double b) {
  Jet<N> r;
#pragma unroll
  for (int k = 0; k < N; ++k) r.c[k] = a.c[k] * b;
  return r;
}
template <int N>
PN_DEV Jet<N> operator*(double a, const Jet<N>& b) {
  Jet<N> r;
#pragma unroll
  for (int k = 0; k < N; ++k) r.c[k] = a * b.c[k];
  return r;
}
// q = a / b:  q_k = (a_k - sum_{j=1..k} b_j q_{k-j}) / b_0
template <int N>
PN_DEV Jet<N> operator/(const Jet<N>& a, const Jet<N>& b) {
  Jet<N> q;
  q.c[0] = a.c[0] / b.c[0];
#pragma unroll
  for (int k = 1; k < N; ++k) {
    double acc = a.c[k];
#pragma unroll
    for (int j = 1; j <= k; ++j) acc = ::fma(-b.c[j], q.c[k - j], acc);
    q.c[k] = acc / b.c[0];
  }
  return q;
}
template <int N>
PN_DEV Jet<N> operator/(const Jet<N>& a, double b) {
  Jet<N> r;
#pragma unroll
  for (int k = 0; k < N; ++k) r.c[k] = a.c[k] / b;
  return r;
}
template <int N>
PN_DEV Jet<N> operator/(double a, const Jet<N>& b) { return Jet<N>(a) / b; }

template <int N, class B>
PN_DEV Jet<N>& operator+=(Jet<N>& a, const B& b) { return a = a + b; }
template <int N, class B>
PN_DEV Jet<N>& operator-=(Jet<N>& a, const B& b) { return a = a - b; }
template <int N, class B>
PN_DEV Jet<N>& operator*=(Jet<N>& a, const B& b) { return a = a * b; }
template <int N, class B>
PN_DEV Jet<N>& operator/=(Jet<N>& a, const B& b) { return a = a / b; }

// fma(a, b, c) with at least one jet operand: coefficient k is c_k + (a b)_k, accumulated with fma in the order of
// jet_mul; a product with a double operand is one fma per coefficient
template <class A, class B, class C>
PN_DEV typename EnableIf<(JetResult<A, B, C>::N > 0), Jet<JetResult<A, B, C>::N>>::type fma(const A& a, const B& b, const C& c) {
  constexpr int N = JetResult<A, B, C>::N;
  constexpr bool JA = JetOrder<A>::value > 0, JB = JetOrder<B>::value > 0;
  Jet<N> r;
#pragma unroll
  for (int k = 0; k < N; ++k) {
    double acc = coef(c, k);
    if (JA && JB) {
#pragma unroll
      for (int j = 0; j <= k; ++j) acc = ::fma(coef(a, j), coef(b, k - j), acc);
    } else if (JA) {
      acc = ::fma(coef(a, k), coef(b, 0), acc);
    } else if (JB) {
      acc = ::fma(coef(a, 0), coef(b, k), acc);
    } else if (k == 0) {
      acc = ::fma(coef(a, 0), coef(b, 0), acc);
    }
    r.c[k] = acc;
  }
  return r;
}

// ---- elementary functions -------------------------------------------------------------------------------------
// the double overloads are the kernels' branch-free IEEE ones; exp / log / sin / cos / sqrt / pow on doubles are
// CUDA's (the user's unqualified call finds them next to these templates)
PN_DEV double rcp(double x) { return ::pn::rcp(x); }
template <int N>
PN_DEV Jet<N> rcp(const Jet<N>& b) {
  Jet<N> q;
  q.c[0] = ::pn::rcp(b.c[0]);
#pragma unroll
  for (int k = 1; k < N; ++k) {
    double acc = 0.0;
#pragma unroll
    for (int j = 1; j <= k; ++j) acc = ::fma(-b.c[j], q.c[k - j], acc);
    q.c[k] = acc * q.c[0];
  }
  return q;
}
// r^2 = a:  r_k = (a_k - sum_{j=1..k-1} r_j r_{k-j}) / (2 r_0)
template <int N>
PN_DEV Jet<N> sqrt(const Jet<N>& a) {
  Jet<N> r;
  r.c[0] = ::sqrt(a.c[0]);
#pragma unroll
  for (int k = 1; k < N; ++k) {
    double acc = a.c[k];
#pragma unroll
    for (int j = 1; j < k; ++j) acc = ::fma(-r.c[j], r.c[k - j], acc);
    r.c[k] = acc / (2.0 * r.c[0]);
  }
  return r;
}
// e' = a' e:  e_k = sum_{j=1..k} j a_j e_{k-j} / k
template <int N>
PN_DEV Jet<N> exp(const Jet<N>& a) {
  Jet<N> e;
  e.c[0] = ::exp(a.c[0]);
#pragma unroll
  for (int k = 1; k < N; ++k) {
    double acc = 0.0;
#pragma unroll
    for (int j = 1; j <= k; ++j) acc = ::fma((double)j * a.c[j], e.c[k - j], acc);
    e.c[k] = acc / (double)k;
  }
  return e;
}
// a l' = a':  l_k = (a_k - sum_{j=1..k-1} j l_j a_{k-j} / k) / a_0
template <int N>
PN_DEV Jet<N> log(const Jet<N>& a) {
  Jet<N> l;
  l.c[0] = ::log(a.c[0]);
#pragma unroll
  for (int k = 1; k < N; ++k) {
    double acc = 0.0;
#pragma unroll
    for (int j = 1; j < k; ++j) acc = ::fma((double)j * l.c[j], a.c[k - j], acc);
    l.c[k] = (a.c[k] - acc / (double)k) / a.c[0];
  }
  return l;
}
// s' = a' c, c' = -a' s
template <int N>
PN_DEV void sincos(const Jet<N>& a, Jet<N>* s, Jet<N>* c) {
  s->c[0] = ::sin(a.c[0]);
  c->c[0] = ::cos(a.c[0]);
#pragma unroll
  for (int k = 1; k < N; ++k) {
    double as = 0.0, ac = 0.0;
#pragma unroll
    for (int j = 1; j <= k; ++j) {
      as = ::fma((double)j * a.c[j], c->c[k - j], as);
      ac = ::fma((double)j * a.c[j], s->c[k - j], ac);
    }
    s->c[k] = as / (double)k;
    c->c[k] = -ac / (double)k;
  }
}
template <int N>
PN_DEV Jet<N> sin(const Jet<N>& a) {
  Jet<N> s, c;
  sincos(a, &s, &c);
  return s;
}
template <int N>
PN_DEV Jet<N> cos(const Jet<N>& a) {
  Jet<N> s, c;
  sincos(a, &s, &c);
  return c;
}
// y = a^p, a y' = p a' y:  y_k = sum_{j=1..k} (p j - (k - j)) a_j y_{k-j} / (k a_0)   (jet_inv_pow32 for any p)
template <int N>
PN_DEV Jet<N> pow(const Jet<N>& a, double p) {
  Jet<N> y;
  y.c[0] = ::pow(a.c[0], p);
#pragma unroll
  for (int k = 1; k < N; ++k) {
    double acc = 0.0;
#pragma unroll
    for (int j = 1; j <= k; ++j) {
      const double cf = p * (double)j - (double)(k - j);
      acc = ::fma(cf * a.c[j], y.c[k - j], acc);
    }
    y.c[k] = acc / ((double)k * a.c[0]);
  }
  return y;
}
// integer powers by repeated products (defined at a_0 = 0 too)
template <int N>
PN_DEV Jet<N> pow(const Jet<N>& a, int n) {
  const int m = n < 0 ? -n : n;
  Jet<N> r(1.0);
  for (int i = 0; i < m; ++i) r = r * a;
  return n < 0 ? rcp(r) : r;
}

}  // namespace jet

using jet::Jet;

// Problem functor over a user source `Src` with Src::vf<T> (and Src::jac when HAS_SRC_JAC): the interface of the
// functors in pn_problems.cuh.  ID is not read by any kernel; the registry keys user problems by their own id.
// TIME_: Src::vf<T>(u, t, p, f) and Src::jac(u, t, p, J) take the time, as a number of type T (a Jet<N> in the
// Taylor-mode initialisation, the constant (t, 0) in the derived Jacobian); an autonomous source never sees it.
template <class Src, int D_, int Q_, int P_, bool HAS_SRC_JAC, bool TIME_ = false>
struct UserProblem {
  static constexpr int D = D_, Q = Q_, P = P_, ID = -1;
  static constexpr bool HAS_JAC = true, TIME = TIME_;
  template <class T>
  PN_DEV static void src_vf(const T* u, const T& t, const double* par, T* f) {
    if constexpr (TIME)
      Src::template vf<T>(u, t, par, f);
    else
      Src::template vf<T>(u, par, f);
  }
  PN_DEV static void vf(const double* u, const double* par, double* f) { src_vf<double>(u, 0.0, par, f); }
  PN_DEV static void vf(const double* u, double t, const double* par, double* f) { src_vf<double>(u, t, par, f); }
  PN_DEV static void jac(const double* u, const double* par, double* J) { jac(u, 0.0, par, J); }
  // without a user Jacobian: column j is the first-order coefficient of vf at u + eps e_j
  PN_DEV static void jac(const double* u, double t, const double* par, double* J) {
    if constexpr (HAS_SRC_JAC) {
      if constexpr (TIME)
        Src::jac(u, t, par, J);
      else
        Src::jac(u, par, J);
    } else {
      const Jet<2> tj(t);
      for (int j = 0; j < Q * D; ++j) {
        Jet<2> x[Q * D], f[D];
#pragma unroll
        for (int i = 0; i < Q * D; ++i) {
          x[i].c[0] = u[i];
          x[i].c[1] = (i == j) ? 1.0 : 0.0;
        }
        src_vf<Jet<2>>(x, tj, par, f);
#pragma unroll
        for (int l = 0; l < D; ++l) J[l * Q * D + j] = f[l].c[1];
      }
    }
  }
  template <int N>
  PN_DEV static void vf_jet(const double* U, const double* par, double* F) {
    vf_jet<N>(U, nullptr, par, F);
  }
  template <int N>
  PN_DEV static void vf_jet(const double* U, const double* Tc, const double* par, double* F) {
    Jet<N> x[Q * D], f[D], tj(0.0);
#pragma unroll
    for (int i = 0; i < Q * D; ++i)
#pragma unroll
      for (int k = 0; k < N; ++k) x[i].c[k] = U[i * N + k];
    if constexpr (TIME) {
#pragma unroll
      for (int k = 0; k < N; ++k) tj.c[k] = Tc[k];
    }
    src_vf<Jet<N>>(x, tj, par, f);
#pragma unroll
    for (int l = 0; l < D; ++l)
#pragma unroll
      for (int k = 0; k < N; ++k) F[l * N + k] = f[l].c[k];
  }
};

// Problem functor over a user's `struct Problem` with the interface of pn_problems.cuh (TIME included).  Its own
// Jacobian when it has one, else column j is the first-order coefficient of vf_jet<2> at u + eps e_j, with the time
// held constant.
template <class Pr>
struct FullProblem {
  static constexpr int D = Pr::D, Q = Pr::Q, P = Pr::P, ID = -1;
  static constexpr bool HAS_JAC = true, TIME = TimeDependent<Pr>::value;
  PN_DEV static void vf(const double* u, const double* par, double* f) { Pr::vf(u, par, f); }
  PN_DEV static void vf(const double* u, double t, const double* par, double* f) { Pr::vf(u, t, par, f); }
  PN_DEV static void jac(const double* u, const double* par, double* J) { jac(u, 0.0, par, J); }
  PN_DEV static void jac(const double* u, double t, const double* par, double* J) {
    if constexpr (Pr::HAS_JAC) {
      jac_at<Pr>(u, t, par, J);
    } else {
      const double Tc[2] = {t, 0.0};
      for (int j = 0; j < Q * D; ++j) {
        double U[Q * D * 2], F[D * 2];
#pragma unroll
        for (int i = 0; i < Q * D; ++i) {
          U[2 * i] = u[i];
          U[2 * i + 1] = (i == j) ? 1.0 : 0.0;
        }
        vf_jet<2>(U, Tc, par, F);
#pragma unroll
        for (int l = 0; l < D; ++l) J[l * Q * D + j] = F[2 * l + 1];
      }
    }
  }
  template <int N>
  PN_DEV static void vf_jet(const double* U, const double* par, double* F) {
    Pr::template vf_jet<N>(U, par, F);
  }
  template <int N>
  PN_DEV static void vf_jet(const double* U, const double* Tc, const double* par, double* F) {
    if constexpr (TIME)
      Pr::template vf_jet<N>(U, Tc, par, F);
    else
      Pr::template vf_jet<N>(U, par, F);
  }
};

// ---- evaluation of a problem for users and tests (pn_b200_problem_evaluate[_at]) ---------------------------------
// per state b, at the time t0 = t[b] (0 without t): f = vf(u0, t0, p), tc = taylor_init (the Taylor coefficients
// u^(k)(t0), k = 0..NU), J = jac(u0, t0, p)
template <class Prob, int NU>
__global__ void __launch_bounds__(128) pn_problem_eval_kernel(long long n, int num_params, const double* t, const double* u0,
                                                              const double* params, double* f, double* tc, double* J) {
  constexpr int D = Prob::D, Q = Prob::Q, P = (Prob::P > 0 ? Prob::P : 1);
  const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n) return;
  double u[Q * D], par[P];
  for (int i = 0; i < Q * D; ++i) u[i] = u0[b * Q * D + i];
  for (int i = 0; i < P; ++i) par[i] = (i < num_params) ? params[b * num_params + i] : 0.0;
  const double t0 = t ? t[b] : 0.0;
  if (f) {
    double fb[D];
    vf_at<Prob>(u, t0, par, fb);
    for (int l = 0; l < D; ++l) f[b * D + l] = fb[l];
  }
  if (tc) {
    double c[NU + 1][D];
    taylor_init<Prob, NU>(u, t0, par, c);
    for (int k = 0; k <= NU; ++k)
      for (int l = 0; l < D; ++l) tc[(b * (NU + 1) + k) * D + l] = c[k][l];
  }
  if (J && Prob::HAS_JAC) {
    double Jb[D * Q * D];
    jac_at<Prob>(u, t0, par, Jb);
    for (int e = 0; e < D * Q * D; ++e) J[b * D * Q * D + e] = Jb[e];
  }
}

}  // namespace pn
