// pn_dense_kernel.cuh -- warp-per-IVP solver kernel for the DENSE factorisation with d > 1 (sm_100a).
//
// impl.select("dense", ode_shape=(d,)) (experiments/1_van_der_pol/vdp.py:61 for d = 1; BASELINE
// configs 3 and 5 ask for dense EKF1 on the rigid body and the Brusselator): mean in R^D, one
// D x D square-root factor, D = (nu+1) d, EKF0 or EKF1 with a d x D observation matrix
// (SURVEY App. A.3 "EKF1 (dense)"), filter or fixed-point strategy, dynamic or no calibration.
//
// One warp owns one IVP and runs the same "uber step" state machine as pn_scalar_kernel.cuh
// (attempt / checkpoint prediction A / checkpoint prediction B), but the D x D matrices live in
// shared memory and the linear algebra is warp-cooperative:
//   * matrix products: one output element per lane, inner index ascending;
//   * Householder QR (R only): every lane forms the reflector of column j redundantly from
//     broadcast shared-memory reads, then lane c updates column c;
//   * triangular solves: one right-hand-side column per lane.
// Every output element is therefore produced by ONE lane in exactly the order of the CPU oracle's
// generic dense engine (oracle/pn_solver.c), so results are bit-identical to it.
// State-space ordering: derivative-major, index i*d + l.
#pragma once
#include "pn_scalar_kernel.cuh"
#include "pn_smooth_kernel.cuh"

namespace pn {

// The dense kernels take the same argument blocks as the thread-per-IVP family (SolveArgs /
// SmoothArgs); only the workspace layout differs: member-major [B][K][SLOT].

// ---- warp-cooperative dense helpers (shared memory operands, leading dimension explicit) ------
namespace wc {

// C[r x c] = A[r x k] B[k x c]; one element per lane, inner index ascending from the k = 0 product
PN_DEV void matmul(const double* A, int lda, const double* B, int ldb, double* C, int ldc, int r, int k, int c, int lane) {
  for (int e = lane; e < r * c; e += 32) {
    const int i = e / c, j = e - i * c;
    double acc = A[i * lda] * B[j];
#pragma unroll 4
    for (int l = 1; l < k; ++l) acc = fma(A[i * lda + l], B[l * ldb + j], acc);
    C[i * ldc + j] = acc;
  }
  __syncwarp();
}

// Householder QR, R only (oracle/pn_linalg.c: pn_qr_r / pn_qr_r_partial).  M is rows x cols with
// leading dimension ld.  `shape` names the structural zeros of the stacked matrix so that the
// loops skip them (exact: a zero entry contributes fma(0, x, acc) = acc in the oracle's full loops):
//   QR_FULL            no structure
//   QR_TOPTRI_BOTFULL  top nb x . block upper triangular (zero below its diagonal), bottom block full
//   QR_TOPFULL_BOTTRI  top nb x . block full, bottom block upper triangular
enum : int { QR_FULL = 0, QR_TOPTRI_BOTFULL = 1, QR_TOPFULL_BOTTRI = 2 };
PN_DEV void qr_r(double* M, int ld, int rows, int cols, int lane, int ncols = 1 << 30, int shape = QR_FULL, int nb = 0) {
  int kmax = rows < cols ? rows : cols;
  if (ncols < kmax) kmax = ncols;  // triangularise only the first ncols columns (pn_qr_r_partial)
  for (int j = 0; j < kmax; ++j) {
    // rows below the diagonal that can be non-zero in column j: [a0, a1) and [b0, b1)
    int a0 = j + 1, a1 = rows, b0 = rows, b1 = rows;
    if (shape == QR_TOPTRI_BOTFULL && j < nb) { a0 = nb; a1 = rows; }
    if (shape == QR_TOPFULL_BOTTRI) { a0 = j + 1; a1 = nb; b0 = nb; b1 = nb + j + 1; }
    double sigma2 = 0.0;
#pragma unroll 4
    for (int i = a0; i < a1; ++i) {
      const double x = M[i * ld + j];
      sigma2 = fma(x, x, sigma2);
    }
#pragma unroll 4
    for (int i = b0; i < b1; ++i) {
      const double x = M[i * ld + j];
      sigma2 = fma(x, x, sigma2);
    }
    if (!(sigma2 > 0.0)) continue;  // warp-uniform: every lane read the same column
    const double alpha = M[j * ld + j];
    const double norm = dsqrt(fma(alpha, alpha, sigma2));
    const double v0 = (alpha >= 0.0) ? (alpha + norm) : (alpha - norm);
    const double beta = (alpha >= 0.0) ? -norm : norm;
    const double g = rcp(norm * (fabs(alpha) + norm));
    for (int c = j + 1 + lane; c < cols; c += 32) {
      double w = 0.0;
#pragma unroll 4
      for (int i = a0; i < a1; ++i) w = fma(M[i * ld + j], M[i * ld + c], w);
#pragma unroll 4
      for (int i = b0; i < b1; ++i) w = fma(M[i * ld + j], M[i * ld + c], w);
      w = fma(v0, M[j * ld + c], w);
      const double f = w * g;
      M[j * ld + c] = fma(-f, v0, M[j * ld + c]);
#pragma unroll 4
      for (int i = a0; i < a1; ++i) M[i * ld + c] = fma(-f, M[i * ld + j], M[i * ld + c]);
#pragma unroll 4
      for (int i = b0; i < b1; ++i) M[i * ld + c] = fma(-f, M[i * ld + j], M[i * ld + c]);
    }
    __syncwarp();
    if (lane == 0) M[j * ld + j] = beta;
    for (int i = a0 + lane; i < a1; i += 32) M[i * ld + j] = 0.0;
    for (int i = b0 + lane; i < b1; i += 32) M[i * ld + j] = 0.0;
    __syncwarp();
  }
}

// R X = B (R n x n upper, B n x c): back substitution, one column per lane
PN_DEV void solve_upper(const double* R, int ldr, const double* Bm, int ldb, double* X, int ldx, int n, int c, int lane) {
  for (int j = lane; j < c; j += 32) {
    for (int i = n - 1; i >= 0; --i) {
      const double inv = rcp(R[i * ldr + i]);
      double acc = Bm[i * ldb + j];
      for (int k = i + 1; k < n; ++k) acc = fma(-R[i * ldr + k], X[k * ldx + j], acc);
      X[i * ldx + j] = acc * inv;
    }
  }
  __syncwarp();
}

// R^T X = B: forward substitution, one column per lane
PN_DEV void solve_upper_transposed(const double* R, int ldr, const double* Bm, int ldb, double* X, int ldx, int n, int c, int lane) {
  for (int j = lane; j < c; j += 32) {
    for (int i = 0; i < n; ++i) {
      const double inv = rcp(R[i * ldr + i]);
      double acc = Bm[i * ldb + j];
      for (int k = 0; k < i; ++k) acc = fma(-R[k * ldr + i], X[k * ldx + j], acc);
      X[i * ldx + j] = acc * inv;
    }
  }
  __syncwarp();
}

PN_DEV void copy(double* dst, const double* src, int count, int lane) {
  for (int e = lane; e < count; e += 32) dst[e] = src[e];
  __syncwarp();
}

PN_DEV void set_identity(double* G, double* g, double* Lam, int Dn, int lane) {
  for (int e = lane; e < Dn * Dn; e += 32) {
    const int i = e / Dn, j = e - i * Dn;
    G[e] = (i == j) ? 1.0 : 0.0;
    Lam[e] = 0.0;
  }
  for (int e = lane; e < Dn; e += 32) g[e] = 0.0;
  __syncwarp();
}

}  // namespace wc

template <int N, int DD>
struct DenseLayout {
  static constexpr int Dn = N * DD;
  static constexpr int MAT = Dn * Dn;
  static constexpr int BW = 2 * MAT + Dn;        // G, g, Lam (full storage)
  static constexpr int MARG = Dn + MAT;          // mean, chol
  static constexpr int SLOT_FIX = BW + MARG;
  static constexpr int SLOT_FILT = MARG;
  // shared memory per warp (doubles)
  static constexpr int SMEM = 16 * MAT + 12 * Dn + 5 * DD * Dn + 4 * DD + 8;
  static constexpr int SMEM_SMOOTH = 5 * MAT + 4 * Dn;
};

template <class Prob, int NU, int STRAT, int WARPS>
__global__ void __launch_bounds__(32 * WARPS) pn_dense_kernel(const __grid_constant__ SolveArgs a) {
  constexpr int N = NU + 1, d = Prob::D, Q = Prob::Q, P = (Prob::P > 0 ? Prob::P : 1);
  using Lay = DenseLayout<N, d>;
  constexpr int Dn = Lay::Dn, MAT = Lay::MAT;
  constexpr bool FIX = (STRAT == 1);
  constexpr int SLOT = FIX ? Lay::SLOT_FIX : Lay::SLOT_FILT;
  constexpr double TIME_EPS = 10.0 * 2.220446049250313e-16;
  constexpr int W2 = 2 * Dn;

  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double* sp = smem + (size_t)warp * Lay::SMEM;
  auto take = [&](int count) { double* r = sp; sp += count; return r; };
  // state
  double* S_m = take(Dn);   double* S_L = take(MAT);
  double* S_G = take(MAT);  double* S_g = take(Dn);  double* S_Lam = take(MAT);
  // accepted-but-uncommitted state while a checkpoint is interpolated
  double* P_m = take(Dn);   double* P_L = take(MAT);
  // step outputs
  double* m_ext = take(Dn); double* m_new = take(Dn);
  double* L_ext = take(MAT); double* L_new = take(MAT);
  double* Gm = take(MAT);   double* gm = take(Dn);   double* Lm = take(MAT);
  // work
  double* m_p = take(Dn);   double* m_ext_p = take(Dn);
  double* M = take(4 * MAT);
  double* X = take(MAT);    // X = RY^{-1} R12, later T = G1 Ln
  double* Gn = take(MAT);   double* gn = take(Dn);   double* Ln = take(MAT);
  double* L_p = take(MAT);  // also AL
  double* H = take(d * Dn); double* Rs = take(Dn * d); double* HL = take(d * Dn);
  double* Wt = take(d * Dn);  // also Y / gain^T chain
  double* gainT = take(d * Dn);
  double* pv = take(Dn);    double* pinvv = take(Dn);
  double* zv = take(d);     double* errv = take(d);  double* yv = take(d);

  const double* LQ = a.lq;
  const double inv_sqrt_d = rcp(dsqrt((double)d));
  auto lqfull = [&](int i, int j) -> double {  // (LQ kron I_d)[i][j]
    return ((i % d) == (j % d)) ? LQ[(i / d) * N + (j / d)] : 0.0;
  };

  for (;;) {
    // ---- fetch a member (one per warp) ----------------------------------------------------
    unsigned long long tk = 0;
    if (lane == 0) tk = atomicAdd(a.ticket, 1ULL);
    tk = __shfl_sync(0xffffffffu, tk, 0);
    if (tk >= (unsigned long long)a.B) break;
    const long long b = a.order ? a.order[tk] : (long long)tk;
    double par[P];
#pragma unroll
    for (int i = 0; i < P; ++i) par[i] = (i < a.num_params) ? a.params[b * a.num_params + i] : 0.0;
    const double atol = a.tol ? a.tol[2 * b] : a.atol, rtol = a.tol ? a.tol[2 * b + 1] : a.rtol;
    const double sigma0 = a.sigma0 ? a.sigma0[b] : 1.0;
    {
      double u0[Q * d], tc[N][d];
#pragma unroll
      for (int i = 0; i < Q * d; ++i) u0[i] = a.u0[b * (Q * d) + i];
      taylor_init<Prob, NU>(u0, grid_row(a, b)[0], par, tc);
      if (lane == 0) {
#pragma unroll
        for (int i = 0; i < N; ++i)
#pragma unroll
          for (int l = 0; l < d; ++l) S_m[i * d + l] = tc[i][l];
      }
      for (int e = lane; e < MAT; e += 32) S_L[e] = 0.0;
      __syncwarp();
      wc::set_identity(S_G, S_g, S_Lam, Dn, lane);
    }
    double* slot_base = a.cond + (size_t)b * a.K * SLOT;
    if (!FIX) {  // filter: slot 0 = initial marginal
      for (int e = lane; e < Dn; e += 32) slot_base[e] = S_m[e];
      for (int e = lane; e < MAT; e += 32) slot_base[Dn + e] = 0.0;
    }
    double t = grid_row(a, b)[0], dt_next = a.dt0, le_prev = 0.0;
    double pend_t = 0.0, pend_sigma = 1.0, sigma_state = sigma0;
    int mode = MODE_STEP;
    long long k_next = 1, n_acc = 0, n_rej = 0, n_att = 0;
    if (lane == 0) a.n_accepted[b * a.K] = 0;
    if (lane == 0 && a.out_scale) a.out_scale[b * a.K] = sigma0;
    bool finished = false;
    int st = 0;

    while (!finished) {
      const double t_ck = grid_row(a, b)[k_next < a.K ? k_next : a.K - 1];
      double dt, sigma_given;
      if (mode == MODE_STEP) {
        dt = (a.flags & FLAG_FIXED_GRID) ? (t_ck - t) : dt_next;
        sigma_given = sigma0;
      } else if (mode == MODE_INTERP_A) {
        dt = t_ck - t;
        sigma_given = pend_sigma;
      } else {
        dt = pend_t - t;
        sigma_given = pend_sigma;
      }
      // ================= uber step =====================================================
      {
        const double adt = fabs(dt);
        const double sq = dsqrt(adt);
        const double isq = rcp(sq), idt = rcp(adt);
        double dtp = 1.0, idtp = 1.0;
        double pn_[N], pinvn[N];
#pragma unroll
        for (int k = 0; k <= NU; ++k) {
          const int i = NU - k;
          pn_[i] = (sq * dtp) * (1.0 / factorial(k));
          pinvn[i] = (isq * idtp) * factorial(k);
          dtp *= adt;
          idtp *= idt;
        }
        if (lane == 0) {
#pragma unroll
          for (int i = 0; i < N; ++i)
#pragma unroll
            for (int l = 0; l < d; ++l) {
              pv[i * d + l] = pn_[i];
              pinvv[i * d + l] = pinvn[i];
            }
        }
        __syncwarp();
      }
      // predicted mean (A = A1 kron I_d, applied structurally: zero terms are exact no-ops)
      for (int e = lane; e < Dn; e += 32) m_p[e] = pinvv[e] * S_m[e];
      __syncwarp();
      for (int e = lane; e < Dn; e += 32) {
        const int i = e / d, l = e - i * d;
        double acc = m_p[e];
        for (int j = i + 1; j < N; ++j) acc = fma(Binom<N>::at(i, j), m_p[j * d + l], acc);
        m_ext_p[e] = acc;
        m_ext[e] = pv[e] * acc;
      }
      __syncwarp();
      // linearise: every lane evaluates the (tiny) vector field redundantly in registers
      {
        double uarg[Q * d], f[d];
#pragma unroll
        for (int k = 0; k < Q * d; ++k) uarg[k] = m_ext[k];
        Prob::vf(uarg, par, f);
        if (lane == 0) {
#pragma unroll
          for (int l = 0; l < d; ++l) zv[l] = m_ext[Q * d + l] - f[l];
        }
        for (int e = lane; e < d * Dn; e += 32) H[e] = 0.0;
        __syncwarp();
        if (lane == 0) {
#pragma unroll
          for (int l = 0; l < d; ++l) H[l * Dn + Q * d + l] = 1.0;
        }
        if (Prob::HAS_JAC && a.correction == 1) {
          double J[d * Q * d];
          Prob::jac(uarg, par, J);
          if (lane == 0) {
#pragma unroll
            for (int l = 0; l < d; ++l)
#pragma unroll
              for (int k = 0; k < Q * d; ++k) H[l * Dn + k] = -J[l * (Q * d) + k];
          }
        }
        __syncwarp();
      }
      // calibration + local error (App. A.3, dense): S_Q = (H p LQ)(H p LQ)^T through a QR
      double sigma_hat, sigma;
      {
        for (int e = lane; e < Dn * d; e += 32) {
          const int j = e / d, l = e - j * d;
          double acc = 0.0;
          for (int i = 0; i < Dn; ++i) acc = fma(H[l * Dn + i] * pv[i], lqfull(i, j), acc);
          Rs[j * d + l] = acc;
        }
        __syncwarp();
        wc::qr_r(Rs, d, Dn, d, lane);
        if (lane == 0) {
          // y = R^{-T} z (forward substitution), sequential
          for (int i = 0; i < d; ++i) {
            const double inv = rcp(Rs[i * d + i]);
            double acc = zv[i];
            for (int k = 0; k < i; ++k) acc = fma(-Rs[k * d + i], yv[k], acc);
            yv[i] = acc * inv;
          }
        }
        __syncwarp();
        double yy = 0.0;
        for (int l = 0; l < d; ++l) yy = fma(yv[l], yv[l], yy);
        sigma_hat = dsqrt(yy) * inv_sqrt_d;
        if (lane == 0) {
          for (int l = 0; l < d; ++l) {
            double cc = 0.0;
            for (int i = 0; i <= l; ++i) cc = fma(Rs[i * d + l], Rs[i * d + l], cc);
            errv[l] = (fabs(dt) * sigma_hat) * dsqrt(cc);
          }
        }
        __syncwarp();
        sigma = (mode == MODE_STEP) ? ((a.calibration == 1) ? sigma_hat : sigma_given) : sigma_given;
      }
      // predict covariance
      {
        for (int e = lane; e < MAT; e += 32) L_p[e] = pinvv[e / Dn] * S_L[e];
        __syncwarp();
        double* AL = X;  // X is free until the triangular solve
        for (int e = lane; e < MAT; e += 32) {
          const int r = e / Dn, c = e - r * Dn;
          const int i = r / d, l = r - i * d;
          // generic product A L_p restricted to the non-zeros of A1 kron I (order preserved)
          double acc = 0.0;
          bool first = true;
          for (int j = 0; j < N; ++j) {
            const double aij = Binom<N>::at(i, j);
            if (j < i) continue;
            const double x = L_p[(j * d + l) * Dn + c];
            acc = first ? (aij * x) : fma(aij, x, acc);
            first = false;
          }
          AL[e] = acc;
        }
        __syncwarp();
        if (!FIX) {
          for (int e = lane; e < MAT; e += 32) {
            const int i = e / Dn, j = e - i * Dn;
            M[i * Dn + j] = sigma * lqfull(j, i);
            M[(Dn + i) * Dn + j] = AL[j * Dn + i];
          }
          __syncwarp();
          wc::qr_r(M, Dn, W2, Dn, lane, 1 << 30, wc::QR_TOPTRI_BOTFULL, Dn);
          for (int e = lane; e < MAT; e += 32) {
            const int i = e / Dn, j = e - i * Dn;
            L_ext[e] = (j <= i) ? pv[i] * M[j * Dn + i] : 0.0;
          }
          __syncwarp();
        } else {
          for (int e = lane; e < MAT; e += 32) {
            const int i = e / Dn, j = e - i * Dn;
            M[i * W2 + j] = sigma * lqfull(j, i);
            M[i * W2 + Dn + j] = 0.0;
            M[(Dn + i) * W2 + j] = AL[j * Dn + i];
            M[(Dn + i) * W2 + Dn + j] = L_p[j * Dn + i];
          }
          __syncwarp();
          wc::qr_r(M, W2, W2, W2, lane, Dn, wc::QR_TOPTRI_BOTFULL, Dn);  // lower-right block stays full: see pn_scalar_kernel.cuh
          // X = RY^{-1} R12
          wc::solve_upper(M, W2, M + Dn, W2, X, Dn, Dn, Dn, lane);
          for (int e = lane; e < MAT; e += 32) {
            const int i = e / Dn, j = e - i * Dn;
            Gn[e] = (pv[i] * X[j * Dn + i]) * pinvv[j];
            Ln[e] = pv[i] * M[(Dn + j) * W2 + Dn + i];
            L_ext[e] = (j <= i) ? pv[i] * M[j * W2 + i] : 0.0;
          }
          for (int i = lane; i < Dn; i += 32) {
            double acc = m_p[i];
            for (int k = 0; k < Dn; ++k) acc = fma(-X[k * Dn + i], m_ext_p[k], acc);
            gn[i] = pv[i] * acc;
          }
          __syncwarp();
          // merge with the running conditional (App. A.4)
          wc::matmul(S_G, Dn, Gn, Dn, Gm, Dn, Dn, Dn, Dn, lane);
          for (int i = lane; i < Dn; i += 32) {
            double acc = S_g[i];
            for (int k = 0; k < Dn; ++k) acc = fma(S_G[i * Dn + k], gn[k], acc);
            gm[i] = acc;
          }
          double* T = X;
          wc::matmul(S_G, Dn, Ln, Dn, T, Dn, Dn, Dn, Dn, lane);
          for (int e = lane; e < MAT; e += 32) {
            const int i = e / Dn, j = e - i * Dn;
            M[i * Dn + j] = T[j * Dn + i];
            M[(Dn + i) * Dn + j] = S_Lam[j * Dn + i];
          }
          __syncwarp();
          wc::qr_r(M, Dn, W2, Dn, lane, 1 << 30, wc::QR_TOPFULL_BOTTRI, Dn);
          for (int e = lane; e < MAT; e += 32) {
            const int i = e / Dn, j = e - i * Dn;
            Lm[e] = (j <= i) ? M[j * Dn + i] : 0.0;
          }
          __syncwarp();
        }
      }
      // correction (matrix observation, App. A.3 "EKF1 (dense)")
      double e_norm;
      {
        wc::matmul(H, Dn, L_ext, Dn, HL, Dn, d, Dn, Dn, lane);
        double* Rm = Rs;  // Dn x d
        for (int e = lane; e < Dn * d; e += 32) {
          const int j = e / d, l = e - j * d;
          Rm[e] = HL[l * Dn + j];
        }
        __syncwarp();
        wc::qr_r(Rm, d, Dn, d, lane);
        for (int e = lane; e < d * Dn; e += 32) {
          const int l = e / Dn, i = e - l * Dn;
          double acc = 0.0;
          for (int j = 0; j < Dn; ++j) acc = fma(L_ext[i * Dn + j], HL[l * Dn + j], acc);
          Wt[e] = acc;
        }
        __syncwarp();
        double* Y = M;  // d x Dn scratch
        wc::solve_upper_transposed(Rm, d, Wt, Dn, Y, Dn, d, Dn, lane);
        wc::solve_upper(Rm, d, Y, Dn, gainT, Dn, d, Dn, lane);
        double* Mc = M + d * Dn;
        for (int e = lane; e < MAT; e += 32) {
          const int j = e / Dn, i = e - j * Dn;
          double acc = L_ext[i * Dn + j];
          for (int l = 0; l < d; ++l) acc = fma(-HL[l * Dn + j], gainT[l * Dn + i], acc);
          Mc[j * Dn + i] = acc;
        }
        __syncwarp();
        wc::qr_r(Mc, Dn, Dn, Dn, lane);
        for (int e = lane; e < MAT; e += 32) {
          const int i = e / Dn, j = e - i * Dn;
          L_new[e] = (j <= i) ? Mc[j * Dn + i] : 0.0;
        }
        for (int i = lane; i < Dn; i += 32) {
          double acc = m_ext[i];
          for (int l = 0; l < d; ++l) acc = fma(-gainT[l * Dn + i], zv[l], acc);
          m_new[i] = acc;
        }
        __syncwarp();
        double acc = 0.0;
        for (int l = 0; l < d; ++l) {
          const double ratio = errv[l] * rcp(fma(rtol, fabs(m_new[l]), atol));
          acc = fma(ratio, ratio, acc);
        }
        e_norm = dsqrt(acc) * inv_sqrt_d;
      }
      double fac, le_now;
      {
        le_now = det_log(e_norm < 2.2250738585072014e-308 ? 2.2250738585072014e-308 : e_norm);
        le_now = (e_norm == 0.0) ? -745.0 : le_now;
        fac = a.safety * det_exp(fma(a.pow_p, le_prev, -((a.pow_i + a.pow_p) * le_now)));
        fac = (e_norm == 0.0) ? a.factor_max : fac;
        fac = (e_norm != e_norm) ? e_norm : fac;
        fac = (fac < a.factor_max) ? fac : a.factor_max;
        fac = (fac > a.factor_min) ? fac : a.factor_min;
      }
      // ================= bookkeeping (warp-uniform) =====================================
      auto emit_cond = [&](double* dst, const double* G_, const double* g_, const double* L_) {
        for (int e = lane; e < MAT; e += 32) {
          dst[e] = G_[e];
          dst[MAT + Dn + e] = L_[e];
        }
        for (int e = lane; e < Dn; e += 32) dst[MAT + e] = g_[e];
      };
      auto emit_identity_cond = [&](double* dst) {
        for (int e = lane; e < MAT; e += 32) {
          dst[e] = ((e / Dn) == (e % Dn)) ? 1.0 : 0.0;
          dst[MAT + Dn + e] = 0.0;
        }
        for (int e = lane; e < Dn; e += 32) dst[MAT + e] = 0.0;
      };
      auto emit_marg = [&](double* dst, const double* m_, const double* L_) {
        for (int e = lane; e < Dn; e += 32) dst[e] = m_[e];
        for (int e = lane; e < MAT; e += 32) dst[Dn + e] = L_[e];
      };
      auto resolve_hits = [&]() {
        while (k_next < a.K && !(t + TIME_EPS < grid_row(a, b)[k_next])) {
          double* slot = slot_base + (size_t)k_next * SLOT;
          if (FIX) {
            emit_cond(slot, S_G, S_g, S_Lam);
            if (k_next == a.K - 1) {
              emit_identity_cond(slot_base);
              emit_marg(slot_base + Lay::BW, S_m, S_L);
            }
            __syncwarp();
            wc::set_identity(S_G, S_g, S_Lam, Dn, lane);
          } else {
            emit_marg(slot, S_m, S_L);
          }
          if (lane == 0) a.n_accepted[b * a.K + k_next] = n_acc;
          if (lane == 0 && a.out_scale) a.out_scale[b * a.K + k_next] = sigma_state;
          k_next += 1;
        }
        if (k_next >= a.K) finished = true;
      };
      auto after_checkpoint = [&]() {
        if (k_next < a.K && pend_t > grid_row(a, b)[k_next] + TIME_EPS) {
          mode = MODE_INTERP_A;
        } else {
          t = pend_t;
          sigma_state = pend_sigma;
          wc::copy(S_m, P_m, Dn, lane);
          wc::copy(S_L, P_L, MAT, lane);
          if (FIX) {
            wc::copy(S_G, Gm, MAT, lane);
            wc::copy(S_g, gm, Dn, lane);
            wc::copy(S_Lam, Lm, MAT, lane);
          }
          mode = MODE_STEP;
          resolve_hits();
        }
      };
      const bool fixed_grid = (a.flags & FLAG_FIXED_GRID) != 0;
      if (mode == MODE_STEP) {
        n_att += 1;
        if (e_norm != e_norm && !fixed_grid) {
          finished = true;
          st = 1;
        } else {
          dt_next = fac * dt;
          if (e_norm <= 1.0 || fixed_grid) {
            if (!fixed_grid) {
              le_prev = le_now;
            }
            n_acc += 1;
            const double t1 = fixed_grid ? t_ck : (t + dt);
            const bool overshoot = (k_next < a.K) && (t1 > t_ck + TIME_EPS);
            if (overshoot) {
              pend_t = t1;
              pend_sigma = sigma;
              wc::copy(P_m, m_new, Dn, lane);
              wc::copy(P_L, L_new, MAT, lane);
              mode = MODE_INTERP_A;
            } else {
              t = t1;
              sigma_state = sigma;
              wc::copy(S_m, m_new, Dn, lane);
              wc::copy(S_L, L_new, MAT, lane);
              if (FIX) {
                wc::copy(S_G, Gm, MAT, lane);
                wc::copy(S_g, gm, Dn, lane);
                wc::copy(S_Lam, Lm, MAT, lane);
              }
              resolve_hits();
            }
          } else {
            n_rej += 1;
          }
          if (!finished && mode == MODE_STEP && a.max_attempts > 0 && n_att >= a.max_attempts) {
            finished = true;
            st = 2;
          }
        }
      } else if (mode == MODE_INTERP_A) {
        double* slot = slot_base + (size_t)k_next * SLOT;
        if (FIX) {
          emit_cond(slot, Gm, gm, Lm);
          __syncwarp();
          wc::set_identity(S_G, S_g, S_Lam, Dn, lane);
        } else {
          emit_marg(slot, m_ext, L_ext);
        }
        t = t_ck;
        wc::copy(S_m, m_ext, Dn, lane);
        wc::copy(S_L, L_ext, MAT, lane);
        if (lane == 0) a.n_accepted[b * a.K + k_next] = n_acc;
        if (lane == 0 && a.out_scale) a.out_scale[b * a.K + k_next] = pend_sigma;
        if (FIX) {
          mode = MODE_INTERP_B;
        } else {
          k_next += 1;
          after_checkpoint();
        }
      } else {
        if (k_next == a.K - 1) {
          emit_cond(slot_base, Gm, gm, Lm);
          emit_marg(slot_base + Lay::BW, P_m, P_L);
        }
        k_next += 1;
        after_checkpoint();
      }
    }
    if (lane == 0) {
      a.n_rejected[b] = n_rej;
      a.status[b] = st;
      if (st != 0)
        for (long long kk = k_next; kk < a.K; ++kk) a.n_accepted[b * a.K + kk] = n_acc;
    }
    __syncwarp();
  }
}

// ---- backward marginalisation for the dense factorisation: one warp per member ----------------
template <int N, int DD, int STRAT, int WARPS>
__global__ void __launch_bounds__(32 * WARPS) pn_dense_smooth_kernel(const SmoothArgs a) {
  using Lay = DenseLayout<N, DD>;
  constexpr int Dn = Lay::Dn, MAT = Lay::MAT, d = DD;
  constexpr bool FIX = (STRAT == 1);
  constexpr int SLOT = FIX ? Lay::SLOT_FIX : Lay::SLOT_FILT;
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long b = (long long)blockIdx.x * WARPS + warp;
  if (b >= a.B) return;
  double* sp = smem + (size_t)warp * Lay::SMEM_SMOOTH;
  double* m = sp;            double* L = m + Dn;
  double* mo = L + MAT;      double* T = mo + Dn;
  double* M = T + MAT;       // 2 Dn x Dn
  double* G = M + 2 * MAT;   double* g = G + MAT;   // staged conditional (Lam is read straight from global)
  const bool ok = (a.status[b] == 0);
  const double* base = a.cond + (size_t)b * a.K * SLOT;
  const double nanv = __longlong_as_double(0x7ff8000000000000LL);

  auto marginalise = [&](const double* c) {
    wc::copy(G, c, MAT, lane);
    wc::copy(g, c + MAT, Dn, lane);
    const double* Lam = c + MAT + Dn;
    for (int i = lane; i < Dn; i += 32) {
      double acc = g[i];
      for (int k = 0; k < Dn; ++k) acc = fma(G[i * Dn + k], m[k], acc);
      mo[i] = acc;
    }
    wc::matmul(G, Dn, L, Dn, T, Dn, Dn, Dn, Dn, lane);
    for (int e = lane; e < MAT; e += 32) {
      const int i = e / Dn, j = e - i * Dn;
      M[i * Dn + j] = T[j * Dn + i];
      M[(Dn + i) * Dn + j] = Lam[j * Dn + i];
    }
    __syncwarp();
    wc::qr_r(M, Dn, 2 * Dn, Dn, lane, 1 << 30, wc::QR_TOPFULL_BOTTRI, Dn);
    for (int e = lane; e < MAT; e += 32) {
      const int i = e / Dn, j = e - i * Dn;
      L[e] = (j <= i) ? M[j * Dn + i] : 0.0;
    }
    wc::copy(m, mo, Dn, lane);
  };
  if (FIX) {
    wc::copy(m, base + Lay::BW, Dn, lane);
    wc::copy(L, base + Lay::BW + Dn, MAT, lane);
    marginalise(base);
  }
  for (long long k = a.K - 1; k >= 0; --k) {
    if (!FIX) {
      wc::copy(m, base + (size_t)k * SLOT, Dn, lane);
      wc::copy(L, base + (size_t)k * SLOT + Dn, MAT, lane);
    }
    for (int l = lane; l < d; l += 32) {
      double acc = 0.0;
      for (int j = 0; j < Dn; ++j) acc = fma(L[l * Dn + j], L[l * Dn + j], acc);
      a.u[(b * a.K + k) * d + l] = ok ? m[l] : nanv;
      a.u_std[(b * a.K + k) * d + l] = ok ? dsqrt(acc) : nanv;
    }
    if (a.marg_mean)
      for (int e = lane; e < Dn; e += 32) a.marg_mean[(b * a.K + k) * Dn + e] = ok ? m[e] : nanv;
    if (a.marg_chol)
      for (int e = lane; e < MAT; e += 32) a.marg_chol[(b * a.K + k) * MAT + e] = ok ? L[e] : nanv;
    __syncwarp();
    if (k == 0) break;
    if (FIX) marginalise(base + (size_t)k * SLOT);
  }
}

}  // namespace pn
