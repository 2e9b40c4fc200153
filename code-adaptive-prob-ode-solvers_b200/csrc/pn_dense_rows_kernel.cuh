// pn_dense_rows_kernel.cuh -- dense factorisation, d > 1, D = (nu+1) d <= 32: register-resident
// Householder columns, LANES (16 or 32) lanes per IVP (sm_100a).
//
// Same solver as pn_dense_kernel.cuh (impl.select("dense", ode_shape=(d,)), EKF0 / EKF1 with a
// d x D observation matrix, filter or fixed-point strategy; SURVEY App. A.3/A.4) and the same
// "uber step" state machine, but the linear algebra is laid out so that every long dependent
// chain runs in registers:
//
//   * lane c owns ROW c of every D x D factor (L, G, Lam, L_ext, ...), which is COLUMN c of the
//     transposed, stacked matrices the square-root updates triangularise.  A Householder step j
//     is: lane j publishes its column to a small shared buffer, every lane reads it back as a
//     broadcast, forms the reflector redundantly (same operations, same order -> same bits) and
//     updates its own column in registers.  No shared-memory round trip sits inside a dot product.
//   * the 2D x 2D block QR of the fixed-point predict gives lane c the two columns c and D + c;
//     its pivot rows never need a register index (the top-left block is sigma L_Q^T (x) I, known
//     in closed form; the top-right block starts at zero), so that loop stays rolled.
//   * matrix products are row-per-lane with the right operand broadcast from shared memory;
//     triangular solves are column-per-lane with the reciprocal diagonal computed once.
//   * D <= 16 packs TWO IVPs per warp (LANES = 16): the heavy step is straight-line and identical
//     for both halves, only the bookkeeping between steps diverges.
//
// Every output element is produced by one lane with exactly the operation order of the CPU
// oracle's generic dense engine (oracle/pn_solver.c, pn_linalg.c: pn_qr_r / pn_qr_r_partial);
// loops skip structural zeros only (fma(0, x, acc) == acc), so results are bit-identical to it
// and to pn_dense_kernel.cuh.  Workspace slot layout and smoothing kernel are the dense family's.
#pragma once
#include "pn_dense_kernel.cuh"

namespace pn {

template <int N, int DD>
struct DenseRowsLayout {
  static constexpr int Dn = N * DD;
  static constexpr int MAT = Dn * Dn;
  static constexpr int VB = 2 * Dn + 2;  // one reflector broadcast buffer (even: it is read and written as 16-byte pairs)
  static constexpr int TABLES = 2 * N * N;  // L_Q and the flipped Pascal matrix, once per CTA
  static constexpr int TRI = Dn * (Dn + 1) / 2;  // a packed lower-triangular factor (row i at i (i + 1) / 2)
  // shared memory per IVP slot (doubles): 6 full matrices, the running Lam packed (it is only read as one row per
  // lane by the merge and copied / emitted between steps: packing it is what lets an eighth warp fit on an SM at
  // D = 15) + vectors, see the take() list in the kernel; rounded up to an even count so that the broadcast buffers
  // at the front of every slot stay 16-byte aligned
  static constexpr int SMEM_SLOT = (6 * MAT + TRI + 9 * Dn + 2 * DD * Dn + DD * DD + 2 * VB + 1) & ~1;
};

template <class Prob, int NU, int STRAT, int LANES, int WARPS>
__global__ void __launch_bounds__(32 * WARPS) pn_dense_rows_kernel(const __grid_constant__ SolveArgs a) {
  constexpr int N = NU + 1, d = Prob::D, Q = Prob::Q, P = (Prob::P > 0 ? Prob::P : 1);
  using Lay = DenseLayout<N, d>;
  using RL = DenseRowsLayout<N, d>;
  constexpr int Dn = Lay::Dn, MAT = Lay::MAT, VB = RL::VB;
  constexpr bool FIX = (STRAT == 1);
  constexpr int SLOT = FIX ? Lay::SLOT_FIX : Lay::SLOT_FILT;
  constexpr double TIME_EPS = 10.0 * 2.220446049250313e-16;
  constexpr int GPW = 32 / LANES;  // IVPs per warp
  static_assert(LANES == 16 || LANES == 32, "LANES must be 16 or 32");
  static_assert(Dn <= LANES, "one lane per state row");
  // The observation matrix H = E_q - J only touches the derivatives 0 .. q, and L_Q (x) I and L_ext are lower
  // triangular: H p (L_Q (x) I) and H L_ext are exactly zero from column LIM = (q+1) d on.  The matrices the
  // calibration, the innovation and the corrected factor triangularise therefore have their sub-diagonal
  // non-zeros in the first LIM rows only, and the generic QR leaves a column with an all-zero sub-diagonal
  // untouched: the loops below stop at LIM (exact -- same bits as the full loops, 9 of 14 reflectors of the
  // corrected factor and 60 % of every inner product of the two d-column QRs skipped at D = 15).
  constexpr int LIM = ((Q + 1) * d < Dn) ? (Q + 1) * d : Dn;

  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = lane / LANES, c = lane - sub * LANES;  // c: the row (= transposed column) this lane owns
  const unsigned gmask = (LANES == 32) ? 0xffffffffu : (0xffffu << (16 * sub));
  const int lead = sub * LANES;
  const bool act = c < Dn;
  const int cr = act ? c : (Dn - 1);     // clamped: inactive lanes shadow the last row and never store
  const int ci = cr / d, cl = cr - ci * d;  // derivative index, ODE dimension of row cr

  double* LQs = smem;
  double* A1s = smem + N * N;
  for (int e = threadIdx.x; e < N * N; e += blockDim.x) {
    LQs[e] = a.lq[e];
    A1s[e] = Binom<N>::at(e / N, e % N);
  }
  __syncthreads();

  double* sp = smem + RL::TABLES + (size_t)(warp * GPW + sub) * RL::SMEM_SLOT;
  auto take = [&](int count) { double* r = sp; sp += count; return r; };
  double* vb = take(2 * VB);  // first: 16-byte aligned (reflector broadcasts move as double2)
  // state
  double* S_m = take(Dn);   double* S_L = take(MAT);
  double* S_G = take(MAT);  double* S_g = take(Dn);  double* S_Lam = take(RL::TRI);  // (packed lower triangle)
  // step outputs.  (m_new, L_new) is only written by an attempted step (MODE_STEP), so it doubles
  // as the accepted-but-uncommitted state while the checkpoints inside that step are interpolated.
  double* m_ext = take(Dn); double* m_new = take(Dn);
  double* L_ext = take(MAT); double* L_new = take(MAT);
  double* gm = take(Dn);
  // work
  double* m_p = take(Dn);   double* m_ext_p = take(Dn);
  double* W1 = take(MAT);   // R11 of the block QR, then G of this step (rows), then the merged G
  double* W2 = take(MAT);   // R12 of the block QR, then Lam of this step (rows), then the merged Lam
  double* Gm = W1;
  double* Lm = W2;
  double* P_m = m_new;
  double* P_L = L_new;
  double* gn_s = take(Dn);  double* dinv = take(Dn);
  double* H = take(d * Dn); double* HLs = take(d * Dn);
  double* Rs = take(d * d);

  double a1row[N];  // row ci of the flipped Pascal matrix
#pragma unroll
  for (int j = 0; j < N; ++j) a1row[j] = A1s[ci * N + j];
  const double inv_sqrt_d = rcp(dsqrt((double)d));
  const int tri_cr = cr * (cr + 1) / 2;  // row cr of a packed lower-triangular factor

  // Reflector broadcast as 16-byte pairs: lane `owner` stores the pairs that cover elements [e0, e1) of `src`
  // (a register array indexed like the buffer), every lane reads them back into `dst`.  Elements outside [e0, e1)
  // that share a pair are stored / loaded as well and simply not used.
  auto publish_pairs = [&](double* buf, bool owner, const double* src, int e0, int e1) {
    if (owner) {
      double2* b2 = reinterpret_cast<double2*>(buf);
#pragma unroll
      for (int pp = 0; pp < VB / 2; ++pp)
        if (pp >= (e0 >> 1) && pp <= ((e1 - 1) >> 1)) b2[pp] = make_double2(src[2 * pp], src[2 * pp + 1]);
    }
  };
  auto fetch_pairs = [&](const double* buf, double* dst, int e0, int e1) {
    const double2* b2 = reinterpret_cast<const double2*>(buf);
#pragma unroll
    for (int pp = 0; pp < VB / 2; ++pp)
      if (pp >= (e0 >> 1) && pp <= ((e1 - 1) >> 1)) {
        const double2 t = b2[pp];
        dst[2 * pp] = t.x;
        dst[2 * pp + 1] = t.y;
      }
  };
  auto gsync = [&]() { __syncwarp(gmask); };
  auto gcopy = [&](double* dst, const double* src, int count) {
    for (int e = c; e < count; e += LANES) dst[e] = src[e];
    __syncwarp(gmask);
  };
  // running Lam <- merged Lam of this step (W2, full rows): every lane packs its own row
  auto pack_lam = [&]() {
    if (act) {
#pragma unroll
      for (int k = 0; k < Dn; ++k)
        if (k <= c) S_Lam[tri_cr + k] = W2[c * Dn + k];
    }
    __syncwarp(gmask);
  };
  auto set_identity = [&]() {
    for (int e = c; e < MAT; e += LANES) {
      const int i = e / Dn, j = e - i * Dn;
      S_G[e] = (i == j) ? 1.0 : 0.0;
    }
    for (int e = c; e < RL::TRI; e += LANES) S_Lam[e] = 0.0;
    for (int e = c; e < Dn; e += LANES) S_g[e] = 0.0;
    __syncwarp(gmask);
  };

  // D x d Householder QR (R only, no structure) with one column per lane: lanes l < d hold column
  // l of X^T where X is d x Dn row-major in shared memory.  Publishes the d x d factor to Rs.
  auto small_qr = [&](const double* X) {
    const int lr = (c < d) ? c : (d - 1);
    double rm[LIM];
#pragma unroll
    for (int i = 0; i < LIM; ++i) rm[i] = X[lr * Dn + i];
#pragma unroll
    for (int j = 0; j < d; ++j) {
      double* vbj = vb + (j & 1) * VB;
      double src[VB], v[VB];
#pragma unroll
      for (int i = 0; i < VB; ++i) src[i] = (i < LIM) ? rm[i] : 0.0;
      publish_pairs(vbj, c == j, src, j, LIM);
      __syncwarp();
      fetch_pairs(vbj, v, j, LIM);
      const double alpha = v[j];
      double sigma2 = 0.0;
#pragma unroll
      for (int i = j + 1; i < LIM; ++i) sigma2 = fma(v[i], v[i], sigma2);
      const Reflector R = make_reflector(alpha, sigma2);
      double w = 0.0;
#pragma unroll
      for (int i = j + 1; i < LIM; ++i) w = fma(v[i], rm[i], w);
      w = fma(R.v0, rm[j], w);
      const double f = w * R.ng;
      const double nj = fma(f, R.v0, rm[j]);
#pragma unroll
      for (int i = j + 1; i < LIM; ++i) rm[i] = fma(f, v[i], rm[i]);
      rm[j] = (c == j) ? R.beta : nj;
    }
    if (c < d) {
#pragma unroll
      for (int i = 0; i < d; ++i)
        if (i <= c) Rs[i * d + c] = rm[i];
    }
    __syncwarp();
  };

  // per-IVP control state (uniform within a lane group)
  bool have = false, drained = false;
  long long b = 0;
  double par[P];
  double atol = 0.0, rtol = 0.0, sigma0 = 1.0;
  double* slot_base = nullptr;
  double t = 0.0, dt_next = 0.0, le_prev = 0.0, pend_t = 0.0, pend_sigma = 1.0, sigma_state = 1.0;
  int mode = MODE_STEP, st = 0;
  long long k_next = 1, n_acc = 0, n_rej = 0, n_att = 0;
#pragma unroll
  for (int i = 0; i < P; ++i) par[i] = 0.0;

  for (;;) {
    // ---- fetch a member (one per lane group) ----------------------------------------------
    if (!have && !drained) {
      unsigned long long tk = 0;
      if (c == 0) tk = atomicAdd(a.ticket, 1ULL);
      tk = __shfl_sync(gmask, tk, lead);
      if (tk >= (unsigned long long)a.B) {
        drained = true;
      } else {
        have = true;
        b = a.order ? a.order[tk] : (long long)tk;
#pragma unroll
        for (int i = 0; i < P; ++i) par[i] = (i < a.num_params) ? a.params[b * a.num_params + i] : 0.0;
        atol = a.tol ? a.tol[2 * b] : a.atol;
        rtol = a.tol ? a.tol[2 * b + 1] : a.rtol;
        sigma0 = a.sigma0 ? a.sigma0[b] : 1.0;
        {
          double u0[Q * d], tc[N][d];
#pragma unroll
          for (int i = 0; i < Q * d; ++i) u0[i] = a.u0[b * (Q * d) + i];
          taylor_init<Prob, NU>(u0, grid_row(a, b)[0], par, tc);
          if (c == 0) {
#pragma unroll
            for (int i = 0; i < N; ++i)
#pragma unroll
              for (int l = 0; l < d; ++l) S_m[i * d + l] = tc[i][l];
          }
          for (int e = c; e < MAT; e += LANES) S_L[e] = 0.0;
          __syncwarp(gmask);
          set_identity();
        }
        slot_base = a.cond + (size_t)b * a.K * SLOT;
        if (!FIX) {  // filter: slot 0 = initial marginal
          for (int e = c; e < Dn; e += LANES) slot_base[e] = S_m[e];
          for (int e = c; e < MAT; e += LANES) slot_base[Dn + e] = 0.0;
        }
        t = grid_row(a, b)[0];
        dt_next = a.dt0;
        le_prev = 0.0;
        pend_t = 0.0;
        pend_sigma = 1.0;
        sigma_state = sigma0;
        mode = MODE_STEP;
        k_next = 1;
        n_acc = n_rej = n_att = 0;
        st = 0;
        if (c == 0) a.n_accepted[b * a.K] = 0;
        if (c == 0 && a.out_scale) a.out_scale[b * a.K] = sigma0;
        if constexpr (!FIX) {
          // trajectory: traj_t [cap][B], traj_u and traj_std [cap][d][B]; lane l < d writes component l, lane 0 the
          // time.  The initial point has a zero factor.
          if (a.flags & FLAG_RECORD) {
            if (c == 0) a.traj_t[b] = t;
            if (c < d) {
              a.traj_u[(long long)c * a.B + b] = S_m[c];
              a.traj_std[(long long)c * a.B + b] = 0.0;
            }
          }
        }
      }
    }
    if (__all_sync(0xffffffffu, !have)) break;
    __syncwarp();

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
    // ================= uber step (straight-line, identical for every lane group) =============
    double pn_[N], pinvn[N];
    {
      const double adt = fabs(dt);
      // |dt| is a positive normal number: the unguarded fast paths are exact (as in pn_scalar_kernel.cuh)
      const double sq = dsqrt_raw(adt);
      const double isq = rcp_raw(sq), idt = rcp_raw(adt);
      double dtp = 1.0, idtp = 1.0;
#pragma unroll
      for (int k = 0; k <= NU; ++k) {
        const int i = NU - k;
        pn_[i] = (sq * dtp) * (1.0 / factorial(k));
        pinvn[i] = (isq * idtp) * factorial(k);
        dtp *= adt;
        idtp *= idt;
      }
    }
    double pc = pn_[0], pic = pinvn[0];  // preconditioner entries of the lane's own row
#pragma unroll
    for (int i = 1; i < N; ++i) {
      pc = (ci == i) ? pn_[i] : pc;
      pic = (ci == i) ? pinvn[i] : pic;
    }
    // predicted mean (A = A1 kron I_d applied structurally)
    if (act) m_p[c] = pic * S_m[c];
    __syncwarp();
    {
      double acc = m_p[cr];
#pragma unroll
      for (int j = 1; j < N; ++j) {
        const double nx = fma(a1row[j], m_p[j * d + cl], acc);
        acc = (j > ci) ? nx : acc;
      }
      if (act) {
        m_ext_p[c] = acc;
        m_ext[c] = pc * acc;
      }
    }
    __syncwarp();
    // linearise: every lane evaluates the (tiny) vector field redundantly in registers; a time-dependent problem at
    // the time the prediction reaches (the same double an accepted step or a checkpoint commits as the new time)
    double zv[d];
    {
      double t_vf = 0.0;
      if constexpr (TimeDependent<Prob>::value) {
        if (mode == MODE_STEP)
          t_vf = (a.flags & FLAG_FIXED_GRID) ? t_ck : (t + dt);
        else
          t_vf = (mode == MODE_INTERP_A) ? t_ck : pend_t;
      }
      double uarg[Q * d], f[d];
#pragma unroll
      for (int k = 0; k < Q * d; ++k) uarg[k] = m_ext[k];
      vf_at<Prob>(uarg, t_vf, par, f);
#pragma unroll
      for (int l = 0; l < d; ++l) zv[l] = m_ext[Q * d + l] - f[l];
      for (int e = c; e < d * Dn; e += LANES) H[e] = 0.0;
      __syncwarp();
      if (c == 0) {
#pragma unroll
        for (int l = 0; l < d; ++l) H[l * Dn + Q * d + l] = 1.0;
      }
      if (Prob::HAS_JAC && a.correction == 1) {
        double J[d * Q * d];
        jac_at<Prob>(uarg, t_vf, par, J);
        if (c == 0) {
#pragma unroll
          for (int l = 0; l < d; ++l)
#pragma unroll
            for (int k = 0; k < Q * d; ++k) H[l * Dn + k] = -J[l * (Q * d) + k];
        }
      }
      __syncwarp();
    }
    // calibration + local error (App. A.3, dense): S_Q = (H p LQ)(H p LQ)^T through a QR
    double sigma_hat, sigma, errv[d];
    {
      // row cr of (H p (LQ kron I))^T; only i = a d + cl meets a non-zero of LQ kron I
#pragma unroll
      for (int l = 0; l < d; ++l) {
        double acc = 0.0;
#pragma unroll
        for (int q = 0; q < N; ++q) acc = fma(H[l * Dn + q * d + cl] * pn_[q], LQs[q * N + ci], acc);
        if (act) HLs[l * Dn + c] = acc;
      }
      __syncwarp();
      small_qr(HLs);
      double yv[d];
#pragma unroll
      for (int i = 0; i < d; ++i) {
        const double inv = rcp_raw(Rs[i * d + i]);
        double acc = zv[i];
#pragma unroll
        for (int k = 0; k < i; ++k) acc = fma(-Rs[k * d + i], yv[k], acc);
        yv[i] = acc * inv;
      }
      double yy = 0.0;
#pragma unroll
      for (int l = 0; l < d; ++l) yy = fma(yv[l], yv[l], yy);
      sigma_hat = dsqrt(yy) * inv_sqrt_d;
#pragma unroll
      for (int l = 0; l < d; ++l) {
        double cc = 0.0;
#pragma unroll
        for (int i = 0; i <= l; ++i) cc = fma(Rs[i * d + l], Rs[i * d + l], cc);
        errv[l] = (fabs(dt) * sigma_hat) * dsqrt(cc);
      }
      sigma = (mode == MODE_STEP) ? ((a.calibration == 1) ? sigma_hat : sigma_given) : sigma_given;
      __syncwarp();  // Rs is rewritten by the correction
    }
    // predict covariance: columns of [sigma LQ^T (x) I | 0 ; (A L_p)^T | L_p^T]
    {
      double lb[Dn], rb[Dn];  // bottom halves of the lane's left / right column
      // (A L_p)[cr][k] = sum_j A1[ci][j] pinv_j L[j d + cl][k]: A1[ci][j] = 0 for j < ci, so those terms only add
      // exact zeros in front of the first product (fma(a, x, +-0) = a x rounded): no lane-dependent selects
#pragma unroll
      for (int k = 0; k < Dn; ++k) {
        double acc = a1row[0] * (pinvn[0] * S_L[cl * Dn + k]);
#pragma unroll
        for (int j = 1; j < N; ++j) acc = fma(a1row[j], pinvn[j] * S_L[(j * d + cl) * Dn + k], acc);
        lb[k] = acc;
        if (FIX) rb[k] = pic * S_L[cr * Dn + k];
      }
      for (int j = 0; j < Dn; ++j) {
        const int jq = j / d, jr = j - jq * d;
        const double top_l = sigma * ((cl == jr) ? LQs[ci * N + jq] : 0.0);
        double* vbj = vb + (j & 1) * VB;
        double src[VB], v[VB];
#pragma unroll
        for (int k = 0; k < VB; ++k) src[k] = (k < Dn) ? lb[k] : ((k == Dn) ? top_l : 0.0);
        publish_pairs(vbj, c == j, src, 0, Dn + 1);
        __syncwarp();
        fetch_pairs(vbj, v, 0, Dn + 1);
        double sigma2 = 0.0;
#pragma unroll
        for (int k = 0; k < Dn; ++k) sigma2 = fma(v[k], v[k], sigma2);
        const Reflector R = make_reflector(v[Dn], sigma2);
        double wl = 0.0, wr = 0.0;
#pragma unroll
        for (int k = 0; k < Dn; ++k) {
          wl = fma(v[k], lb[k], wl);
          if (FIX) wr = fma(v[k], rb[k], wr);
        }
        wl = fma(R.v0, top_l, wl);
        const double fl = wl * R.ng;
        const double ntop = fma(fl, R.v0, top_l);
#pragma unroll
        for (int k = 0; k < Dn; ++k) lb[k] = fma(fl, v[k], lb[k]);
        const double r11 = (c == j) ? R.beta : ((c > j) ? ntop : 0.0);
        if (act) L_ext[c * Dn + j] = (c >= j) ? (pc * r11) : 0.0;
        if (FIX) {
          wr = fma(R.v0, 0.0, wr);
          const double fr = wr * R.ng;
          const double rtop = fma(fr, R.v0, 0.0);
#pragma unroll
          for (int k = 0; k < Dn; ++k) rb[k] = fma(fr, v[k], rb[k]);
          if (act) {
            W1[j * Dn + c] = r11;
            W2[j * Dn + c] = rtop;
          }
        }
      }
      if (FIX) {
        __syncwarp();
        if (act) dinv[c] = rcp_raw(W1[c * Dn + c]);  // a zero pivot poisons the solve with NaN either way
        __syncwarp();
        // X = R11^{-1} R12, column cr
        double x[Dn];
#pragma unroll
        for (int i = Dn - 1; i >= 0; --i) {
          double acc = W2[i * Dn + cr];
#pragma unroll
          for (int k = i + 1; k < Dn; ++k) acc = fma(-W1[i * Dn + k], x[k], acc);
          x[i] = acc * dinv[i];
        }
        double gnc;
        {
          double acc = m_p[cr];
#pragma unroll
          for (int k = 0; k < Dn; ++k) acc = fma(-x[k], m_ext_p[k], acc);
          gnc = pc * acc;
        }
        __syncwarp();  // every lane is done with R11 / R12
        if (act) {
#pragma unroll
          for (int j = 0; j < Dn; ++j) {
            W1[c * Dn + j] = (pc * x[j]) * pinvn[j / d];  // G of this step, row c
            W2[c * Dn + j] = pc * rb[j];                  // Lam of this step, row c
          }
          gn_s[c] = gnc;
        }
        __syncwarp();
        // merge with the running conditional (App. A.4): rows of S_G W1, S_G W2
        double tt[Dn], bl[Dn];
        {
          double accG[Dn];
          double gacc = S_g[cr];
          {
            const double s = S_G[cr * Dn];
#pragma unroll
            for (int j = 0; j < Dn; ++j) {
              accG[j] = s * W1[j];
              tt[j] = s * W2[j];
            }
            gacc = fma(s, gn_s[0], gacc);
          }
          for (int l = 1; l < Dn; ++l) {
            const double s = S_G[cr * Dn + l];
#pragma unroll
            for (int j = 0; j < Dn; ++j) {
              accG[j] = fma(s, W1[l * Dn + j], accG[j]);
              tt[j] = fma(s, W2[l * Dn + j], tt[j]);
            }
            gacc = fma(s, gn_s[l], gacc);
          }
          __syncwarp();  // every lane is done with this step's G and Lam: W1 / W2 take the merged ones
          if (act) {
#pragma unroll
            for (int j = 0; j < Dn; ++j) Gm[c * Dn + j] = accG[j];
            gm[c] = gacc;
          }
        }
#pragma unroll
        for (int k = 0; k < Dn; ++k) bl[k] = (k <= cr) ? S_Lam[tri_cr + k] : 0.0;
        // QR of [T^T ; Lam_run^T]: top block full, bottom block upper triangular
#pragma unroll
        for (int j = 0; j < Dn; ++j) {
          double* vbj = vb + (j & 1) * VB;
          double src[VB], rd[VB];
#pragma unroll
          for (int e = 0; e < VB; ++e) src[e] = (e < Dn) ? tt[e] : ((e < 2 * Dn) ? bl[e - Dn] : 0.0);
          publish_pairs(vbj, c == j, src, j, Dn + j + 1);
          __syncwarp();
          fetch_pairs(vbj, rd, j, Dn + j + 1);
          const double alpha = rd[j];
          double vt[Dn], vl[Dn];
          double sigma2 = 0.0;
#pragma unroll
          for (int i = j + 1; i < Dn; ++i) {
            vt[i] = rd[i];
            sigma2 = fma(vt[i], vt[i], sigma2);
          }
#pragma unroll
          for (int k = 0; k <= j; ++k) {
            vl[k] = rd[Dn + k];
            sigma2 = fma(vl[k], vl[k], sigma2);
          }
          const Reflector R = make_reflector(alpha, sigma2);
          double w = 0.0;
#pragma unroll
          for (int i = j + 1; i < Dn; ++i) w = fma(vt[i], tt[i], w);
#pragma unroll
          for (int k = 0; k <= j; ++k) w = fma(vl[k], bl[k], w);
          w = fma(R.v0, tt[j], w);
          const double f = w * R.ng;
          const double nj = fma(f, R.v0, tt[j]);
#pragma unroll
          for (int i = j + 1; i < Dn; ++i) tt[i] = fma(f, vt[i], tt[i]);
#pragma unroll
          for (int k = 0; k <= j; ++k) bl[k] = fma(f, vl[k], bl[k]);
          tt[j] = (c == j) ? R.beta : nj;
        }
        if (act) {
#pragma unroll
          for (int j = 0; j < Dn; ++j) Lm[c * Dn + j] = (j <= c) ? tt[j] : 0.0;
        }
      }
      __syncwarp();  // L_ext (and the merged conditional) complete
    }
    // correction (matrix observation, App. A.3 "EKF1 (dense)")
    double e_norm;
    {
#pragma unroll
      for (int l = 0; l < d; ++l) {
        double acc = H[l * Dn] * L_ext[cr];
#pragma unroll
        for (int i = 1; i < LIM; ++i) acc = fma(H[l * Dn + i], L_ext[i * Dn + cr], acc);  // H is zero from column LIM on
        if (act) HLs[l * Dn + c] = acc;
      }
      __syncwarp();
      small_qr(HLs);
      double le[Dn], gt[d];
#pragma unroll
      for (int j = 0; j < Dn; ++j) le[j] = L_ext[cr * Dn + j];
      {
        double wt[d], y[d];
#pragma unroll
        for (int l = 0; l < d; ++l) {
          double acc = 0.0;
#pragma unroll
          for (int j = 0; j < LIM; ++j) acc = fma(le[j], HLs[l * Dn + j], acc);
          wt[l] = acc;
        }
#pragma unroll
        for (int i = 0; i < d; ++i) {
          const double inv = rcp_raw(Rs[i * d + i]);
          double acc = wt[i];
#pragma unroll
          for (int k = 0; k < i; ++k) acc = fma(-Rs[k * d + i], y[k], acc);
          y[i] = acc * inv;
        }
#pragma unroll
        for (int i = d - 1; i >= 0; --i) {
          const double inv = rcp_raw(Rs[i * d + i]);
          double acc = y[i];
#pragma unroll
          for (int k = i + 1; k < d; ++k) acc = fma(-Rs[i * d + k], gt[k], acc);
          gt[i] = acc * inv;
        }
      }
      double mc[Dn];  // column cr of (L_ext - gain HL)^T; rows >= LIM are those of L_ext^T and never change
#pragma unroll
      for (int j = 0; j < Dn; ++j) {
        double acc = le[j];
        if (j < LIM) {
#pragma unroll
          for (int l = 0; l < d; ++l) acc = fma(-HLs[l * Dn + j], gt[l], acc);
        }
        mc[j] = acc;
      }
#pragma unroll
      for (int j = 0; j < LIM - 1; ++j) {
        double* vbj = vb + (j & 1) * VB;
        double src[VB], v[VB];
#pragma unroll
        for (int i = 0; i < VB; ++i) src[i] = (i < LIM) ? mc[i] : 0.0;
        publish_pairs(vbj, c == j, src, j, LIM);
        __syncwarp();
        fetch_pairs(vbj, v, j, LIM);
        const double alpha = v[j];
        double sigma2 = 0.0;
#pragma unroll
        for (int i = j + 1; i < LIM; ++i) sigma2 = fma(v[i], v[i], sigma2);
        const Reflector R = make_reflector(alpha, sigma2);
        double w = 0.0;
#pragma unroll
        for (int i = j + 1; i < LIM; ++i) w = fma(v[i], mc[i], w);
        w = fma(R.v0, mc[j], w);
        const double f = w * R.ng;
        const double nj = fma(f, R.v0, mc[j]);
#pragma unroll
        for (int i = j + 1; i < LIM; ++i) mc[i] = fma(f, v[i], mc[i]);
        mc[j] = (c == j) ? R.beta : nj;
      }
      if (act && mode == MODE_STEP) {
#pragma unroll
        for (int j = 0; j < Dn; ++j) L_new[c * Dn + j] = (j <= c) ? mc[j] : 0.0;
        double acc = m_ext[c];
#pragma unroll
        for (int l = 0; l < d; ++l) acc = fma(-gt[l], zv[l], acc);
        m_new[c] = acc;
      }
      __syncwarp();
      double acc = 0.0;
#pragma unroll
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
    // ================= bookkeeping (uniform within a lane group, divergent between groups) ====
    if (!have) continue;
    bool finished = false;
    auto emit_cond = [&](double* dst, const double* G_, const double* g_, const double* L_) {
      for (int e = c; e < MAT; e += LANES) {
        dst[e] = G_[e];
        dst[MAT + Dn + e] = L_[e];
      }
      for (int e = c; e < Dn; e += LANES) dst[MAT + e] = g_[e];
    };
    auto emit_running_cond = [&](double* dst) {  // (S_G, S_g, S_Lam): Lam is packed
      for (int e = c; e < MAT; e += LANES) {
        const int i = e / Dn, j = e - i * Dn;
        dst[e] = S_G[e];
        dst[MAT + Dn + e] = (j <= i) ? S_Lam[i * (i + 1) / 2 + j] : 0.0;
      }
      for (int e = c; e < Dn; e += LANES) dst[MAT + e] = S_g[e];
    };
    auto emit_identity_cond = [&](double* dst) {
      for (int e = c; e < MAT; e += LANES) {
        dst[e] = ((e / Dn) == (e % Dn)) ? 1.0 : 0.0;
        dst[MAT + Dn + e] = 0.0;
      }
      for (int e = c; e < Dn; e += LANES) dst[MAT + e] = 0.0;
    };
    auto emit_marg = [&](double* dst, const double* m_, const double* L_) {
      for (int e = c; e < Dn; e += LANES) dst[e] = m_[e];
      for (int e = c; e < MAT; e += LANES) dst[Dn + e] = L_[e];
    };
    // filter: record the committed point (m_, L_) as trajectory point n_acc.  Lane l < d owns row l of L_: the std
    // of component l is sqrt((L L^T)_ll), its row's sum of squares in ascending order (the zeros right of the
    // diagonal add nothing)
    auto record = [&](double tt, const double* m_, const double* L_) {
      if ((a.flags & FLAG_RECORD) && n_acc < a.traj_cap) {
        if (c == 0) a.traj_t[n_acc * a.B + b] = tt;
        if (c < d) {
          double acc = 0.0;
          for (int j = 0; j <= c; ++j) acc = fma(L_[c * Dn + j], L_[c * Dn + j], acc);
          a.traj_u[(n_acc * d + c) * a.B + b] = m_[c];
          a.traj_std[(n_acc * d + c) * a.B + b] = dsqrt(acc);
        }
      }
    };
    auto resolve_hits = [&]() {
      while (k_next < a.K && !(t + TIME_EPS < grid_row(a, b)[k_next])) {
        double* slot = slot_base + (size_t)k_next * SLOT;
        if (FIX) {
          emit_running_cond(slot);
          if (k_next == a.K - 1) {
            emit_identity_cond(slot_base);
            emit_marg(slot_base + Lay::BW, S_m, S_L);
          }
          gsync();
          set_identity();
        } else {
          emit_marg(slot, S_m, S_L);
        }
        if (c == 0) a.n_accepted[b * a.K + k_next] = n_acc;
        if (c == 0 && a.out_scale) a.out_scale[b * a.K + k_next] = sigma_state;
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
        gcopy(S_m, P_m, Dn);
        gcopy(S_L, P_L, MAT);
        if (FIX) {
          gcopy(S_G, Gm, MAT);
          gcopy(S_g, gm, Dn);
          pack_lam();
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
          if (!fixed_grid) le_prev = le_now;
          n_acc += 1;
          const double t1 = fixed_grid ? t_ck : (t + dt);
          const bool overshoot = (k_next < a.K) && (t1 > t_ck + TIME_EPS);
          if (overshoot) {
            pend_t = t1;
            pend_sigma = sigma;  // the accepted state stays in (m_new, L_new) = (P_m, P_L)
            mode = MODE_INTERP_A;
          } else {
            t = t1;
            sigma_state = sigma;
            gcopy(S_m, m_new, Dn);
            gcopy(S_L, L_new, MAT);
            if (FIX) {
              gcopy(S_G, Gm, MAT);
              gcopy(S_g, gm, Dn);
              pack_lam();
            }
            if constexpr (!FIX) record(t1, m_new, L_new);
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
        gsync();
        set_identity();
      } else {
        emit_marg(slot, m_ext, L_ext);
        if constexpr (!FIX) record(t_ck, m_ext, L_ext);
      }
      t = t_ck;
      gcopy(S_m, m_ext, Dn);
      gcopy(S_L, L_ext, MAT);
      if (c == 0) a.n_accepted[b * a.K + k_next] = n_acc;
      if (c == 0 && a.out_scale) a.out_scale[b * a.K + k_next] = pend_sigma;
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
    if (finished) {
      if (c == 0) {
        a.n_rejected[b] = n_rej;
        a.status[b] = st;
        if (st != 0)
          for (long long kk = k_next; kk < a.K; ++kk) a.n_accepted[b * a.K + kk] = n_acc;
      }
      if constexpr (!FIX) {
        if (c == 0 && (a.flags & FLAG_RECORD)) a.traj_len[b] = (n_acc + 1 < a.traj_cap) ? (n_acc + 1) : a.traj_cap;
      }
      have = false;
    }
  }
}

}  // namespace pn
