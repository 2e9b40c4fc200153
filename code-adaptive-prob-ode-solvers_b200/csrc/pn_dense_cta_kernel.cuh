// pn_dense_cta_kernel.cuh -- CTA-per-IVP solver kernel for the DENSE factorisation with a LARGE state
// dimension D = (nu+1) d (sm_100a, fp64, FP64 tensor path).
//
// impl.select("dense", ode_shape=(d,)) with correction_ts1 / correction_ts0 (experiments/1_van_der_pol/
// vdp.py:61-66 for d = 1) on the Brusselator (src/odecheckpts/ivps.py:124-156, driver shape
// experiments/4_brusselator/run.py:51-61): BASELINE config 5 "dense sqrt-EKF1 factorisation,
// checkpointed smoother, ensemble over the diffusion parameter".  One CTA (256 threads) owns one IVP
// and runs the same state machine as the other families (attempt / checkpoint prediction A / B), but
// the D x D factors live in global memory (a per-CTA scratch region that stays L2-resident for small
// ensembles) and the O(D^3) work is BLOCKED so that it runs on the FP64 tensor path:
//   * Householder QR of the stacked square-root factors as panel factorisation (panel of NB columns in
//     shared memory, one pass + one CTA reduction per column) + compact-WY update of the trailing
//     columns, W = V^T C, Y = T^T W, C <- C - V Y, with mma.sync.m8n8k4.f64 (SASS: DMMA.8x8x4), V read
//     from the shared panel, C streamed from global memory as tensor fragments;
//   * the products of the conditional algebra (G1 G2, G1 Lam2, L H^T, H^T gain) as shared-memory-tiled
//     DMMA GEMMs (64 x 64 CTA tile, register-prefetched 16-deep stages);
//   * the triangular solve for the smoothing gain as blocked back substitution (DMMA update + in-block
//     substitution, one right-hand-side column per thread).
// The structure of the stacked matrices is used to pick the ACTIVE rows of every panel (upper
// triangular top or bottom blocks), which is exact.
//
// Arithmetic order: measured on B200 (scripts/micro/dmma_probe.cu), DMMA.8x8x4 is per output element
// exactly the ascending-k chain of four fma's.  So every blocked product here is an ascending-index
// fma chain per element, every reduction has a fixed order, and oracle/pn_blocked.c restates the whole
// blocked algorithm on the CPU: results are compared with it bit for bit (tests/test_gpu_dense_cta.py).
// Internally the factors are stored TRANSPOSED (U = L^T upper triangular, GT = G^T, LamU = Lam^T) so
// that no product or stacked matrix needs a transposed copy; the element arithmetic is unchanged.
#pragma once
#include "pn_scalar_kernel.cuh"
#include "pn_smooth_kernel.cuh"

namespace pn {
namespace cta {

constexpr int T = 256;                 // threads per CTA
constexpr int WARPS = T / 32;
constexpr int TRSM_BLOCK = 64;         // block rows of the blocked back substitution (oracle: pn_solve_upper_blocked)
constexpr int GEMM_SMEM = 16 * 68 + 64 * 20;  // doubles: B tile [16][68] + A tile max([64][20], [16][68])
enum : int { QR_FULL = 0, QR_TOPTRI_BOTFULL = 1, QR_TOPFULL_BOTTRI = 2 };

PN_DEV void dmma(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1},{%2},{%3},{%0,%1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

// CTA-order sum (oracle: cta_reduce): butterfly over the 32 lanes, then the warps in ascending order.
// red: [WARPS] doubles of shared memory.  Every thread gets the total.  Two barriers.
PN_DEV double cta_sum(double v, int red_off) {
  extern __shared__ double cta_sh[];
  double* red = cta_sh + red_off;
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) v = v + __shfl_xor_sync(0xffffffffu, v, off);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double r = red[0];
#pragma unroll
  for (int w = 1; w < WARPS; ++w) r = r + red[w];
  __syncthreads();
  return r;
}

// sum of squares of v[0..k) in the oracle's reduction_group = 256 order
PN_DEV double cta_sum_squares(const double* v, int k, int red) {
  double acc = 0.0;
  for (int c = threadIdx.x; c < k; c += T) acc = fma(v[c], v[c], acc);
  return cta_sum(acc, red);
}

// ------------------------------------------------------------------------------------------------
// C[M x N] = (C0 ? C0 : 0) -/+ A B  with DMMA.  A(i,k) = a_kmajor ? A[k*lda + i] : A[i*lda + k];
// B(k,j) = B[k*ldb + j]; C / C0 row-major.  Per element: ascending-k fma chain starting from the
// initial value (NEG: fma(-a, b, acc)).  C0 may alias C.  smem: GEMM_SMEM doubles.
// ------------------------------------------------------------------------------------------------
template <bool NEG>
__device__ __noinline__ void gemm(double* C, int ldc, const double* A, int lda, bool a_kmajor, const double* B, int ldb,
                                  int M, int N, int K, const double* C0, int ldc0) {
  extern __shared__ double cta_sh[];
  double* Bs = cta_sh;             // [16][68]
  double* As = cta_sh + 16 * 68;   // m-major: [64][20]; k-major: [16][68]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
  const int wm = (warp >> 2) * 32, wn = (warp & 3) * 16;  // warp tile 32 x 16 inside the 64 x 64 CTA tile
  for (int i0 = 0; i0 < M; i0 += 64) {
    for (int j0 = 0; j0 < N; j0 += 64) {
      double acc[4][2][2];
#pragma unroll
      for (int mt = 0; mt < 4; ++mt)
#pragma unroll
        for (int nt = 0; nt < 2; ++nt)
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int i = i0 + wm + mt * 8 + g, j = j0 + wn + nt * 8 + 2 * t + h;
            acc[mt][nt][h] = (C0 && i < M && j < N) ? C0[(size_t)i * ldc0 + j] : 0.0;
          }
      double ra[4], rb[4];
      auto load_stage = [&](int k0) {
#pragma unroll
        for (int s = 0; s < 4; ++s) {
          const int e = tid + T * s;  // 0..1023
          {
            const int k = k0 + (e >> 6), j = j0 + (e & 63);
            rb[s] = (k < K && j < N) ? B[(size_t)k * ldb + j] : 0.0;
          }
          if (a_kmajor) {
            const int k = k0 + (e >> 6), i = i0 + (e & 63);
            ra[s] = (k < K && i < M) ? A[(size_t)k * lda + i] : 0.0;
          } else {
            const int i = i0 + (e >> 4), k = k0 + (e & 15);
            ra[s] = (k < K && i < M) ? A[(size_t)i * lda + k] : 0.0;
          }
        }
      };
      auto store_stage = [&]() {
#pragma unroll
        for (int s = 0; s < 4; ++s) {
          const int e = tid + T * s;
          Bs[(e >> 6) * 68 + (e & 63)] = rb[s];
          if (a_kmajor)
            As[(e >> 6) * 68 + (e & 63)] = NEG ? -ra[s] : ra[s];
          else
            As[(e >> 4) * 20 + (e & 15)] = NEG ? -ra[s] : ra[s];
        }
      };
      load_stage(0);
      for (int k0 = 0; k0 < K; k0 += 16) {
        __syncthreads();  // previous stage's fragment reads are done
        store_stage();
        __syncthreads();
        if (k0 + 16 < K) load_stage(k0 + 16);  // in flight while this stage computes
#pragma unroll
        for (int k4 = 0; k4 < 16; k4 += 4) {
          double fa[4], fb[2];
#pragma unroll
          for (int mt = 0; mt < 4; ++mt)
            fa[mt] = a_kmajor ? As[(k4 + t) * 68 + wm + mt * 8 + g] : As[(wm + mt * 8 + g) * 20 + k4 + t];
#pragma unroll
          for (int nt = 0; nt < 2; ++nt) fb[nt] = Bs[(k4 + t) * 68 + wn + nt * 8 + g];
#pragma unroll
          for (int mt = 0; mt < 4; ++mt)
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) dmma(acc[mt][nt][0], acc[mt][nt][1], fa[mt], fb[nt]);
        }
      }
#pragma unroll
      for (int mt = 0; mt < 4; ++mt)
#pragma unroll
        for (int nt = 0; nt < 2; ++nt)
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int i = i0 + wm + mt * 8 + g, j = j0 + wn + nt * 8 + 2 * t + h;
            if (i < M && j < N) C[(size_t)i * ldc + j] = acc[mt][nt][h];
          }
    }
  }
  __syncthreads();
}

// ------------------------------------------------------------------------------------------------
// Blocked Householder QR, R only (oracle/pn_blocked.c: pn_qr_blocked).  M: rows x cols, leading
// dimension ld, in global memory; only the first ncols columns are triangularised, all columns get
// the reflectors.  On exit the upper triangle holds R; entries below the diagonal are NOT cleared
// (nobody reads them).
// ------------------------------------------------------------------------------------------------
// Shared-memory layout of the QR (offsets in doubles from the start of the dynamic shared memory; the
// functions below address it through the extern array so that the compiler emits LDS / STS, not generic
// loads).  The panel sits at offset 0 and is aliased by the GEMM tiles (never live at the same time).
template <int NB>
struct QrSmem {
  static constexpr int LDP = NB + 4;  // (LDP mod 16) == 4: conflict-free tensor fragment reads
  int P;     // [hmax4][LDP] panel / V
  int Tm;    // [NB][NB]
  int red;   // [WARPS][NB]
  int v0;    // [NB]
  int beta;  // [NB]
  int wf;    // [WARPS][NB]   per warp: f (columns right of the pivot) / Gram entries S (columns left of it)
  int wy;    // [WARPS][2][NB][16]
  __host__ __device__ static constexpr int fixed_doubles() { return NB * NB + 2 * WARPS * NB + 2 * NB + WARPS * 2 * NB * 16; }
  __host__ __device__ static int panel_doubles(int hmax) { return ((hmax + 7) / 8 * 8) * LDP; }
  __host__ __device__ void layout(int hmax) {
    const int panel = panel_doubles(hmax);
    int o = panel > GEMM_SMEM ? panel : GEMM_SMEM;
    P = 0;
    Tm = o;   o += NB * NB;
    red = o;  o += WARPS * NB;
    v0 = o;   o += NB;
    beta = o; o += NB;
    wf = o;   o += WARPS * NB;
    wy = o;
  }
};

// Warp sum of NB per-lane partial values by a TRANSPOSED butterfly: level by level a lane keeps half of its
// values and sends the other half to its xor partner, so the tree of additions per value is exactly the
// plain butterfly's (xor 16, 8, 4, 2, 1; a + b is commutative) at NB - 1 instead of 5 NB exchanges.
// On return the lane holds the warp total of value `cidx`.
template <int NB>
PN_DEV double warp_sum_transposed(const double (&part)[NB], int lane, int& cidx) {
  double q[NB];
#pragma unroll
  for (int i = 0; i < NB; ++i) q[i] = part[i];
  cidx = 0;
#pragma unroll
  for (int lvl = 0; lvl < 5; ++lvl) {
    const int off = 16 >> lvl;
    const int n = (NB >> lvl) > 0 ? (NB >> lvl) : 1;
    if (n > 1) {
      const int half = n / 2;
      const bool hi = (lane & off) != 0;
#pragma unroll
      for (int i = 0; i < half; ++i) {
        const double send = hi ? q[i] : q[i + half];
        const double keep = hi ? q[i + half] : q[i];
        q[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
      }
      cidx = (cidx << 1) | (hi ? 1 : 0);
    } else {
      q[0] = q[0] + __shfl_xor_sync(0xffffffffu, q[0], off);
    }
  }
  return q[0];
}

template <int NB>
__device__ __noinline__ void qr_blocked(double* M, int ld, int rows, int cols, int ncols, int shape, int ntop, const QrSmem<NB>& s) {
  constexpr int LDP = QrSmem<NB>::LDP;
  extern __shared__ double cta_sh[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
  int kmax = rows < cols ? rows : cols;
  if (ncols < kmax) kmax = ncols;
  double* P = cta_sh + s.P;
  double* Tm = cta_sh + s.Tm;
  double* red = cta_sh + s.red;
  double* wf = cta_sh + s.wf + warp * NB;
  for (int j0 = 0; j0 < kmax; j0 += NB) {
    const int w = (kmax - j0 < NB) ? (kmax - j0) : NB;
    // gathered row r of the panel  ->  row of M
    int h, split, base2;
    if (shape == QR_TOPTRI_BOTFULL) {
      h = w + (rows - ntop);
      split = w;
      base2 = ntop - w;
    } else if (shape == QR_TOPFULL_BOTTRI) {
      int end = ntop + j0 + w;
      if (end > rows) end = rows;
      h = end - j0;
      split = h;
      base2 = j0;
    } else {
      h = rows - j0;
      split = h;
      base2 = j0;
    }
    auto grow = [&](int r) -> int { return (r < split) ? (j0 + r) : (base2 + r); };
    const int h8 = (h + 7) / 8 * 8;
    __syncthreads();
    for (int e = tid; e < h8 * NB; e += T) {
      const int r = e / NB, c = e - r * NB;
      P[r * LDP + c] = (r < h && c < w) ? M[(size_t)grow(r) * ld + j0 + c] : 0.0;
    }
    for (int e = tid; e < NB * NB; e += T) Tm[e] = 0.0;
    __syncthreads();
    // ---- panel factorisation: one pass + one CTA reduction per column ------------------------------
    for (int jj = 0; jj < w; ++jj) {
      double part[NB];
#pragma unroll
      for (int c = 0; c < NB; ++c) part[c] = 0.0;
      for (int r = tid; r < h; r += T) {
        if (r > jj) {
          const double x = P[r * LDP + jj];
#pragma unroll
          for (int c = 0; c < NB; ++c) part[c] = fma(x, P[r * LDP + c], part[c]);
        }
      }
      int cidx;
      const double wtot = warp_sum_transposed<NB>(part, lane, cidx);
      red[warp * NB + cidx] = wtot;
      __syncthreads();
      // lane c < NB of every warp: CTA total of column c (warps in ascending order), pivot-row entry
      const int cl = lane & (NB - 1);
      double tot = red[cl];
#pragma unroll
      for (int ww = 1; ww < WARPS; ++ww) tot = tot + red[ww * NB + cl];
      const double prow = P[jj * LDP + cl];
      const double sigma2 = __shfl_sync(0xffffffffu, tot, jj);
      const double alpha = __shfl_sync(0xffffffffu, prow, jj);
      const Reflector rf = make_reflector(alpha, sigma2);
      const double fS = fma(rf.v0, prow, tot);  // right of the pivot: v^T column; left of it: Gram entry S
      if (lane < NB) wf[cl] = (cl > jj) ? fS * rf.g : fS;
      __syncthreads();  // pivot row and red[] have been read by everybody; wf is complete
      double f[NB];
#pragma unroll
      for (int c = 0; c < NB; ++c) f[c] = wf[c];
      for (int r = tid; r < h; r += T) {
        if (r > jj) {
          const double x = P[r * LDP + jj];
#pragma unroll
          for (int c = 0; c < NB; ++c)
            if (c > jj) P[r * LDP + c] = fma(-f[c], x, P[r * LDP + c]);
        }
      }
      if (tid == (jj % T)) {  // owner of the pivot row
#pragma unroll
        for (int c = 0; c < NB; ++c)
          if (c > jj) P[jj * LDP + c] = fma(-f[c], rf.v0, P[jj * LDP + c]);
        P[jj * LDP + jj] = rf.v0;
        cta_sh[s.v0 + jj] = rf.v0;
        cta_sh[s.beta + jj] = rf.beta;
        Tm[jj * NB + jj] = rf.g;
      }
      if (tid < jj) {  // T[0:jj, jj] = -g T[0:jj, 0:jj] S   (warp 0: its wf holds S[k] for k < jj)
        double acc = 0.0;
        for (int k = tid; k < jj; ++k) acc = fma(Tm[tid * NB + k], wf[k], acc);
        Tm[tid * NB + jj] = (-rf.g) * acc;
      }
    }
    __syncthreads();
    // ---- R entries of the panel back to M; V = panel with the entries above the pivots cleared -----
    for (int e = tid; e < w * w; e += T) {
      const int r = e / w, c = e - r * w;
      double val = 0.0;
      if (r < c) val = P[r * LDP + c];
      if (r == c) val = cta_sh[s.beta + c];
      M[(size_t)(j0 + r) * ld + j0 + c] = val;
    }
    __syncthreads();
    for (int e = tid; e < w * w; e += T) {
      const int r = e / w, c = e - r * w;
      if (r < c) P[r * LDP + c] = 0.0;
    }
    __syncthreads();
    // ---- trailing columns: 16 columns per warp at a time, as two interleaved 8-column tensor tiles ----
    // (tile 0 = even columns, tile 1 = odd columns: a lane's two B-fragment entries are adjacent in memory)
    const int c_first = j0 + w;
    const int ntiles = (cols - c_first + 15) / 16;
    const bool vec_ok = ((ld & 1) == 0) && ((c_first & 1) == 0) && ((((size_t)M) & 15) == 0);
    double* w0s = cta_sh + s.wy + (size_t)warp * 2 * NB * 16;
    double* ys = w0s + NB * 16;
    const int nchunk = (h + 3) / 4;
    constexpr int U = 8;
    for (int tile = warp; tile < ntiles; tile += WARPS) {
      const int c0 = c_first + tile * 16;
      const int cA = c0 + 2 * g;
      auto loadB = [&](int chunk, double& b0, double& b1) {
        const int r = chunk * 4 + t;
        b0 = 0.0;
        b1 = 0.0;
        if (chunk < nchunk && r < h) {
          const double* rowp = M + (size_t)grow(r) * ld;
          if (vec_ok && cA + 1 < cols) {
            const double2 v = *reinterpret_cast<const double2*>(rowp + cA);
            b0 = v.x;
            b1 = v.y;
          } else {
            if (cA < cols) b0 = rowp[cA];
            if (cA + 1 < cols) b1 = rowp[cA + 1];
          }
        }
      };
      // W0 = V^T C  (NB x 16): chain over the gathered rows, ascending
      double acc[NB / 8][2][2];
#pragma unroll
      for (int mt = 0; mt < NB / 8; ++mt) acc[mt][0][0] = acc[mt][0][1] = acc[mt][1][0] = acc[mt][1][1] = 0.0;
      double bc0[U], bc1[U];
#pragma unroll
      for (int u = 0; u < U; ++u) loadB(u, bc0[u], bc1[u]);
      for (int blk = 0; blk * U < nchunk; ++blk) {
        double bn0[U], bn1[U];
#pragma unroll
        for (int u = 0; u < U; ++u) loadB((blk + 1) * U + u, bn0[u], bn1[u]);  // in flight while this block computes
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int chunk = blk * U + u;
          if (chunk < nchunk) {
            const int r = chunk * 4 + t;
#pragma unroll
            for (int mt = 0; mt < NB / 8; ++mt) {
              const double a = P[r * LDP + mt * 8 + g];
              dmma(acc[mt][0][0], acc[mt][0][1], a, bc0[u]);
              dmma(acc[mt][1][0], acc[mt][1][1], a, bc1[u]);
            }
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          bc0[u] = bn0[u];
          bc1[u] = bn1[u];
        }
      }
      // C fragment (row g, column index 2t + hh of tile tau) -> column offset 2 (2t + hh) + tau of the 16
#pragma unroll
      for (int mt = 0; mt < NB / 8; ++mt)
#pragma unroll
        for (int tau = 0; tau < 2; ++tau)
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) w0s[(mt * 8 + g) * 16 + 4 * t + 2 * hh + tau] = acc[mt][tau][hh];
      __syncwarp();
      // Y = T^T W0: Y[a][col] = sum_{i <= a} T[i][a] W0[i][col], ascending i
      {
        const int col = lane & 15;
#pragma unroll
        for (int q = 0; q < NB / 2; ++q) {
          const int a = (lane >> 4) + 2 * q;
          double y = 0.0;
          for (int i = 0; i <= a; ++i) y = fma(Tm[i * NB + a], w0s[i * 16 + col], y);
          ys[a * 16 + col] = y;
        }
      }
      __syncwarp();
      double yb[2][NB / 4];
#pragma unroll
      for (int kk = 0; kk < NB / 4; ++kk) {
        yb[0][kk] = -ys[(4 * kk + t) * 16 + 2 * g];  // C - V Y = C + V (-Y): fma(v, -y, c) == fma(-v, y, c) bit for bit
        yb[1][kk] = -ys[(4 * kk + t) * 16 + 2 * g + 1];
      }
      // C <- C - V Y: chain over the panel columns, ascending, starting from C.  A lane owns 4 adjacent
      // columns c0 + 4t .. c0 + 4t + 3 of row g of every 8-row tile.
      const int cX = c0 + 4 * t;
      const bool vec4 = vec_ok && (cX + 3 < cols);
      const int nm = (h + 7) / 8;
      constexpr int UM = 4;
      auto loadX = [&](int mtile, double (&x)[4]) {
        const int r = mtile * 8 + g;
        x[0] = x[1] = x[2] = x[3] = 0.0;
        if (mtile < nm && r < h) {
          const double* rowp = M + (size_t)grow(r) * ld;
          if (vec4) {
            const double2 v0 = *reinterpret_cast<const double2*>(rowp + cX);
            const double2 v1 = *reinterpret_cast<const double2*>(rowp + cX + 2);
            x[0] = v0.x; x[1] = v0.y; x[2] = v1.x; x[3] = v1.y;
          } else {
#pragma unroll
            for (int e = 0; e < 4; ++e)
              if (cX + e < cols) x[e] = rowp[cX + e];
          }
        }
      };
      double xc[UM][4];
#pragma unroll
      for (int u = 0; u < UM; ++u) loadX(u, xc[u]);
      for (int mb = 0; mb < nm; mb += UM) {
        double xn[UM][4];
#pragma unroll
        for (int u = 0; u < UM; ++u) loadX(mb + UM + u, xn[u]);
#pragma unroll
        for (int u = 0; u < UM; ++u) {
          const int mtile = mb + u;
          const int r = mtile * 8 + g;
          if (mtile < nm) {
            const bool rv = r < h;
#pragma unroll
            for (int kk = 0; kk < NB / 4; ++kk) {
              const double a = rv ? P[r * LDP + 4 * kk + t] : 0.0;
              dmma(xc[u][0], xc[u][2], a, yb[0][kk]);
              dmma(xc[u][1], xc[u][3], a, yb[1][kk]);
            }
            if (rv) {
              double* rowp = M + (size_t)grow(r) * ld;
              if (vec4) {
                *reinterpret_cast<double2*>(rowp + cX) = make_double2(xc[u][0], xc[u][1]);
                *reinterpret_cast<double2*>(rowp + cX + 2) = make_double2(xc[u][2], xc[u][3]);
              } else {
#pragma unroll
                for (int e = 0; e < 4; ++e)
                  if (cX + e < cols) rowp[cX + e] = xc[u][e];
              }
            }
          }
        }
#pragma unroll
        for (int u = 0; u < UM; ++u)
#pragma unroll
          for (int e = 0; e < 4; ++e) xc[u][e] = xn[u][e];
      }
      __syncwarp();
    }
  }
  __syncthreads();
}

// R X = B (R n x n upper, ld ldr; B n x c; X n x c), blocked back substitution
// (oracle/pn_blocked.c: pn_solve_upper_blocked with nb = TRSM_BLOCK).
static __device__ __noinline__ void solve_upper_blocked(const double* R, int ldr, const double* B, int ldb, double* X, int ldx,
                                                 int n, int c) {
  const int nblk = (n + TRSM_BLOCK - 1) / TRSM_BLOCK;
  for (int bi = nblk - 1; bi >= 0; --bi) {
    const int i0 = bi * TRSM_BLOCK, i1 = (i0 + TRSM_BLOCK < n) ? i0 + TRSM_BLOCK : n;
    if (i1 < n) {
      gemm<true>(X + (size_t)i0 * ldx, ldx, R + (size_t)i0 * ldr + i1, ldr, false, X + (size_t)i1 * ldx, ldx, i1 - i0, c,
                 n - i1, B + (size_t)i0 * ldb, ldb);
    } else {
      for (int e = threadIdx.x; e < (i1 - i0) * c; e += T) {
        const int i = i0 + e / c, j = e % c;
        X[(size_t)i * ldx + j] = B[(size_t)i * ldb + j];
      }
      __syncthreads();
    }
    for (int j = threadIdx.x; j < c; j += T) {
      for (int i = i1 - 1; i >= i0; --i) {
        double a = X[(size_t)i * ldx + j];
        for (int k = i + 1; k < i1; ++k) a = fma(-R[(size_t)i * ldr + k], X[(size_t)k * ldx + j], a);
        X[(size_t)i * ldx + j] = a * rcp(R[(size_t)i * ldr + i]);
      }
    }
    __syncthreads();
  }
}

// Unblocked substitutions with a small d x d factor (oracle/pn_linalg.c order), one column per thread.
// R^T X = B (forward):  X[i] = (B[i] - sum_{k<i} R[k][i] X[k]) / R[i][i], k ascending
PN_DEV void solve_upper_transposed_cols(const double* R, int ldr, const double* B, int ldb, double* X, int ldx, int n, int c) {
  for (int j = threadIdx.x; j < c; j += T) {
    for (int i = 0; i < n; ++i) {
      double a = B[(size_t)i * ldb + j];
      for (int k = 0; k < i; ++k) a = fma(-R[(size_t)k * ldr + i], X[(size_t)k * ldx + j], a);
      X[(size_t)i * ldx + j] = a * rcp(R[(size_t)i * ldr + i]);
    }
  }
  __syncthreads();
}
// R X = B (backward): X[i] = (B[i] - sum_{k>i} R[i][k] X[k]) / R[i][i], k ascending
PN_DEV void solve_upper_cols(const double* R, int ldr, const double* B, int ldb, double* X, int ldx, int n, int c) {
  for (int j = threadIdx.x; j < c; j += T) {
    for (int i = n - 1; i >= 0; --i) {
      double a = B[(size_t)i * ldb + j];
      for (int k = i + 1; k < n; ++k) a = fma(-R[(size_t)i * ldr + k], X[(size_t)k * ldx + j], a);
      X[(size_t)i * ldx + j] = a * rcp(R[(size_t)i * ldr + i]);
    }
  }
  __syncthreads();
}

// ---- problems with a runtime dimension ---------------------------------------------------------
// Interface: vf(u, par, f, d) cooperative over the CTA (caller synchronises); h_row(l, ...) the sparse
// row l of H = E_q - J E_{0..q-1} restricted to its structural non-zeros, columns ascending.
constexpr int H_MAX = 6;
struct BrusselatorRt {
  static constexpr int Q = 1, P = 1, ID = 4;
  static constexpr bool HAS_JAC = true;
  PN_DEV static void vf(const double* u, const double* par, double* f, int d) {
    const int Np = d / 2;
    const double c = par[0] * (double)((Np + 1) * (Np + 1));
    const double *uu = u, *vv = u + Np;
    for (int i = threadIdx.x; i < Np; i += T) {
      const double ul = (i == 0) ? 1.0 : uu[i - 1], ur = (i == Np - 1) ? 1.0 : uu[i + 1];
      const double vl = (i == 0) ? 3.0 : vv[i - 1], vr = (i == Np - 1) ? 3.0 : vv[i + 1];
      const double uuv = (uu[i] * uu[i]) * vv[i];
      const double lap_u = fma(-2.0, uu[i], ul + ur);
      const double lap_v = fma(-2.0, vv[i], vl + vr);
      f[i] = fma(c, lap_u, fma(-4.0, uu[i], 1.0 + uuv));
      f[Np + i] = fma(c, lap_v, fma(3.0, uu[i], -uuv));
    }
  }
  // non-zeros of row l of the Jacobian d f / d u (d x d), columns ascending; returns their number
  PN_DEV static int jac_row(int l, const double* u, const double* par, int d, int* cols, double* vals) {
    const int Np = d / 2;
    const double c = par[0] * (double)((Np + 1) * (Np + 1));
    const int i = (l < Np) ? l : l - Np;
    const double ui = u[i], vi = u[Np + i];
    const double two_uv = (2.0 * ui) * vi, u2 = ui * ui;
    int k = 0;
    if (l < Np) {
      if (i > 0) { cols[k] = i - 1; vals[k++] = c; }
      cols[k] = i; vals[k++] = fma(-2.0, c, two_uv - 4.0);
      if (i < Np - 1) { cols[k] = i + 1; vals[k++] = c; }
      cols[k] = Np + i; vals[k++] = u2;
    } else {
      cols[k] = i; vals[k++] = 3.0 - two_uv;
      if (i > 0) { cols[k] = Np + i - 1; vals[k++] = c; }
      cols[k] = Np + i; vals[k++] = fma(-2.0, c, -u2);
      if (i < Np - 1) { cols[k] = Np + i + 1; vals[k++] = c; }
    }
    return k;
  }
  // Taylor-mode initialisation (taylor.odejet_padded_scan, ivpsolvers.py:63-67): m[k*d + l] = u_l^{(k)}(t0)
  template <int N>
  PN_DEV static void taylor(const double* u0, const double* par, double* m, int d) {
    const int Np = d / 2, tid = threadIdx.x;
    const double cc = par[0] * (double)((Np + 1) * (Np + 1));
    for (int c = tid; c < d; c += T) {
      m[c] = u0[c];
      for (int i = 1; i < N; ++i) m[(size_t)i * d + c] = 0.0;
    }
    __syncthreads();
    for (int k = 0; k < N - 1; ++k) {
      for (int gi = tid; gi < Np; gi += T) {
        double uj[N], vj[N], u2[N];
        for (int j = 0; j <= k; ++j) {
          uj[j] = m[(size_t)j * d + gi];
          vj[j] = m[(size_t)j * d + Np + gi];
        }
        for (int kk = 0; kk <= k; ++kk) {
          double acc = uj[0] * uj[kk];
          for (int j = 1; j <= kk; ++j) acc = fma(uj[j], uj[kk - j], acc);
          u2[kk] = acc;
        }
        double uuv = u2[0] * vj[k];
        for (int j = 1; j <= k; ++j) uuv = fma(u2[j], vj[k - j], uuv);
        const double padu = (k == 0) ? 1.0 : 0.0, padv = (k == 0) ? 3.0 : 0.0;
        const double ul = (gi == 0) ? padu : m[(size_t)k * d + gi - 1];
        const double ur = (gi == Np - 1) ? padu : m[(size_t)k * d + gi + 1];
        const double vl = (gi == 0) ? padv : m[(size_t)k * d + Np + gi - 1];
        const double vr = (gi == Np - 1) ? padv : m[(size_t)k * d + Np + gi + 1];
        const double lap_u = fma(-2.0, uj[k], ul + ur);
        const double lap_v = fma(-2.0, vj[k], vl + vr);
        const double fu = fma(cc, lap_u, fma(-4.0, uj[k], padu + uuv));
        const double fv = fma(cc, lap_v, fma(3.0, uj[k], -uuv));
        m[(size_t)(k + 1) * d + gi] = fu / (double)(k + 1);
        m[(size_t)(k + 1) * d + Np + gi] = fv / (double)(k + 1);
      }
      __syncthreads();
    }
    double fact = 1.0;
    for (int k = 0; k < N; ++k) {
      if (k > 0) fact *= (double)k;
      for (int c = tid; c < d; c += T) m[(size_t)k * d + c] = fact * m[(size_t)k * d + c];
    }
    __syncthreads();
  }
};

// ---- workspace layout ----------------------------------------------------------------------------
// slot (per member and checkpoint): [GT | g | LamU] + [m | U]  (kernel-native transposed storage)
__host__ __device__ inline size_t slot_doubles(int Dn, bool fix) {
  const size_t MAT = (size_t)Dn * Dn;
  return fix ? (2 * MAT + Dn) + (Dn + MAT) : (Dn + MAT);
}
// per-CTA scratch (doubles)
__host__ __device__ inline size_t scratch_doubles(int Dn, int d, int q) {
  const size_t MAT = (size_t)Dn * Dn;
  return 17 * MAT                       // S_U S_GT S_LamU P_U M(4) X GnT LnT U_ext GmT M2(2) Mc
         + 12 * (size_t)Dn              // S_m S_g P_m m_ext m_new m_p m_ext_p pv pinvv gn gm spare
         + 5 * (size_t)d * Dn           // HLt Rm Wt Yt gainT
         + (size_t)(q + 1) * d * d      // Rs
         + 6 * (size_t)d                // zv errv yv fv ratio spare
         + 2 * (size_t)d * H_MAX        // Hv, Hc (ints, in double-sized cells)
         + (size_t)d                    // Hn (ints, in double-sized cells)
         + 64;
}
template <int NB>
__host__ __device__ inline size_t smem_doubles(int Dn) {
  const int panel = QrSmem<NB>::panel_doubles(Dn + NB);
  return (size_t)(panel > GEMM_SMEM ? panel : GEMM_SMEM) + QrSmem<NB>::fixed_doubles() + 64;
}

// MINB = 2: compiled for two resident CTAs per SM (128 registers; chosen by the host when two CTAs' shared
// memory fits, i.e. for D up to ~400: twice the warps to hide the latency of the panel and the streamed tiles)
template <class Prob, int NU, int STRAT, int NB, int MINB>
__global__ void __launch_bounds__(T, MINB) pn_dense_cta_kernel(const __grid_constant__ SolveArgs a) {
  constexpr int N = NU + 1, Q = Prob::Q, P = (Prob::P > 0 ? Prob::P : 1);
  constexpr bool FIX = (STRAT == 1);
  constexpr double TIME_EPS = 10.0 * 2.220446049250313e-16;
  const int d = a.wide_d, Dn = N * d, W2 = 2 * Dn;
  const size_t MAT = (size_t)Dn * Dn;
  const size_t SLOT = slot_doubles(Dn, FIX), BW = 2 * MAT + Dn;
  const int tid = threadIdx.x;

  extern __shared__ double smem[];
  QrSmem<NB> qs;
  qs.layout(Dn + NB);
  const int red = qs.red;  // [WARPS] for scalar CTA sums (never live at the same time as a QR)
  __shared__ unsigned long long s_ticket;
  __shared__ double s_bcast[4];

  // per-CTA scratch
  double* sp = a.wide_mean + (size_t)blockIdx.x * scratch_doubles(Dn, d, Q);
  auto take = [&](size_t count) { double* r = sp; sp += count; return r; };
  double* S_U = take(MAT);   double* S_GT = take(MAT);  double* S_LamU = take(MAT);  double* P_U = take(MAT);
  double* M = take(4 * MAT); double* X = take(MAT);     double* GnT = take(MAT);     double* LnT = take(MAT);
  double* U_ext = take(MAT); double* GmT = take(MAT);   double* M2 = take(2 * MAT);  double* Mc = take(MAT);
  double* S_m = take(Dn);    double* S_g = take(Dn);    double* P_m = take(Dn);      double* m_ext = take(Dn);
  double* m_new = take(Dn);  double* m_p = take(Dn);    double* m_ext_p = take(Dn);  double* pv = take(Dn);
  double* pinvv = take(Dn);  double* gn = take(Dn);     double* gm = take(Dn);       take(Dn);
  double* HLt = take((size_t)d * Dn);  double* Rm = take((size_t)d * Dn);  double* Wt = take((size_t)d * Dn);
  double* Yt = take((size_t)d * Dn);   double* gainT = take((size_t)d * Dn);
  double* Rs = take((size_t)(Q + 1) * d * d);
  double* zv = take(d);      double* errv = take(d);    double* yv = take(d);        double* fv = take(d);
  double* ratio = take(d);   take(d);
  double* Hv = take((size_t)d * H_MAX);
  int* Hc = (int*)take((size_t)d * H_MAX);
  int* Hn = (int*)take(d);

  const double* LQ = a.lq;
  const double inv_sqrt_d = rcp(dsqrt((double)d));

  for (;;) {
    __syncthreads();
    if (tid == 0) s_ticket = atomicAdd(a.ticket, 1ULL);
    __syncthreads();
    const unsigned long long tk = s_ticket;
    if (tk >= (unsigned long long)a.B) break;
    const long long b = a.order ? a.order[tk] : (long long)tk;
    double par[P];
#pragma unroll
    for (int i = 0; i < P; ++i) par[i] = (i < a.num_params) ? a.params[b * a.num_params + i] : 0.0;
    const double atol = a.tol ? a.tol[2 * b] : a.atol, rtol = a.tol ? a.tol[2 * b + 1] : a.rtol;
    const double sigma0 = a.sigma0 ? a.sigma0[b] : 1.0;
    Prob::template taylor<N>(a.u0 + (size_t)b * Q * d, par, S_m, d);
    for (size_t e = tid; e < MAT; e += T) {
      const int i = (int)(e / Dn), j = (int)(e - (size_t)i * Dn);
      S_U[e] = 0.0;
      S_GT[e] = (i == j) ? 1.0 : 0.0;
      S_LamU[e] = 0.0;
    }
    for (int e = tid; e < Dn; e += T) S_g[e] = 0.0;
    double* slot_base = a.cond + (size_t)b * a.K * SLOT;
    if (!FIX) {
      for (int e = tid; e < Dn; e += T) slot_base[e] = S_m[e];
      for (size_t e = tid; e < MAT; e += T) slot_base[Dn + e] = 0.0;
    }
    __syncthreads();
    double t = grid_row(a, b)[0], dt_next = a.dt0, le_prev = 0.0;
    double pend_t = 0.0, pend_sigma = 1.0, sigma_state = sigma0;
    int mode = MODE_STEP;
    long long k_next = 1, n_acc = 0, n_rej = 0, n_att = 0;
    if (tid == 0) a.n_accepted[b * a.K] = 0;
    if (tid == 0 && a.out_scale) a.out_scale[b * a.K] = sigma0;
    if constexpr (!FIX) {
      // trajectory: traj_t [cap][B], traj_u and traj_std [cap][d][B]; thread l writes component l (and l + T, ...),
      // thread 0 the time.  The initial point has a zero factor.
      if (a.flags & FLAG_RECORD) {
        if (tid == 0) a.traj_t[b] = t;
        for (int l = tid; l < d; l += T) {
          a.traj_u[(long long)l * a.B + b] = S_m[l];
          a.traj_std[(long long)l * a.B + b] = 0.0;
        }
      }
    }
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
      const bool stepping = (mode == MODE_STEP);
      // ---- preconditioner and predicted mean ------------------------------------------------------
      double pn_[N], pinvn[N];
      {
        const double adt = fabs(dt);
        const double sq = dsqrt(adt);
        const double isq = rcp(sq), idt = rcp(adt);
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
      for (int e = tid; e < Dn; e += T) {
        const int i = e / d;
        double p = pn_[0], pi = pinvn[0];
#pragma unroll
        for (int k = 1; k < N; ++k) {
          p = (i == k) ? pn_[k] : p;
          pi = (i == k) ? pinvn[k] : pi;
        }
        pv[e] = p;
        pinvv[e] = pi;
        m_p[e] = pi * S_m[e];
      }
      __syncthreads();
      for (int e = tid; e < Dn; e += T) {
        const int i = e / d, l = e - i * d;
        double acc = m_p[e];
        for (int j = i + 1; j < N; ++j) acc = fma(Binom<N>::at(i, j), m_p[j * d + l], acc);
        m_ext_p[e] = acc;
        m_ext[e] = pv[e] * acc;
      }
      __syncthreads();
      // ---- linearise, calibrate, local error (attempted steps only) ---------------------------------
      double sigma = sigma_given, sigma_hat = 0.0;
      if (stepping) {
        Prob::vf(m_ext, par, fv, d);
        __syncthreads();
        for (int l = tid; l < d; l += T) {
          zv[l] = m_ext[Q * d + l] - fv[l];
          int cols[H_MAX];
          double vals[H_MAX];
          int k = 0;
          if (Prob::HAS_JAC && a.correction == 1) {
            k = Prob::jac_row(l, m_ext, par, d, cols, vals);
            for (int s = 0; s < k; ++s) vals[s] = -vals[s];
          }
          cols[k] = Q * d + l;
          vals[k++] = 1.0;
          Hn[l] = k;
          for (int s = 0; s < k; ++s) {
            Hc[l * H_MAX + s] = cols[s];
            Hv[l * H_MAX + s] = vals[s];
          }
        }
        for (int e = tid; e < (Q + 1) * d * d; e += T) Rs[e] = 0.0;
        __syncthreads();
        // Rs[(jb d + jl)][l] = sum_{ib >= jb} (H[l][ib d + jl] p_ib) lq[ib][jb]   (ascending ib)
        for (int l = tid; l < d; l += T) {
          const int k = Hn[l];
          for (int s = 0; s < k; ++s) {
            const int c = Hc[l * H_MAX + s];
            const int ib = c / d, jl = c - ib * d;
            const double hp = Hv[l * H_MAX + s] * pv[ib * d];
            for (int jb = 0; jb <= ib; ++jb) {
              double* dst = Rs + ((size_t)(jb * d + jl) * d + l);
              *dst = fma(hp, LQ[ib * N + jb], *dst);
            }
          }
        }
        __syncthreads();
        qr_blocked<NB>(Rs, d, (Q + 1) * d, d, d, QR_FULL, 0, qs);
        // y = R^{-T} z: column-oriented forward substitution (ascending-k chain per element)
        for (int l = tid; l < d; l += T) yv[l] = zv[l];
        __syncthreads();
        for (int k = 0; k < d; ++k) {
          if (tid == (k % T)) yv[k] = yv[k] * rcp(Rs[(size_t)k * d + k]);
          __syncthreads();
          const double yk = yv[k];
          for (int i = k + 1 + tid; i < d; i += T) yv[i] = fma(-Rs[(size_t)k * d + i], yk, yv[i]);
          __syncthreads();
        }
        if (tid == 0) {
          double yy = 0.0;
          for (int l = 0; l < d; ++l) yy = fma(yv[l], yv[l], yy);
          s_bcast[0] = dsqrt(yy) * inv_sqrt_d;
        }
        __syncthreads();
        sigma_hat = s_bcast[0];
        for (int l = tid; l < d; l += T) {
          double cc = 0.0;
          for (int i = 0; i <= l; ++i) cc = fma(Rs[(size_t)i * d + l], Rs[(size_t)i * d + l], cc);
          errv[l] = (fabs(dt) * sigma_hat) * dsqrt(cc);
        }
        sigma = (a.calibration == 1) ? sigma_hat : sigma_given;
        __syncthreads();
      }
      // ---- predict the covariance -----------------------------------------------------------------------
      // stacked matrix rows D.. : [ (A L_p)^T | L_p^T ] = [ U_p A^T | U_p ],  U_p = U diag(pinv)
      {
        const int ldM = FIX ? W2 : Dn;
        for (size_t e = tid; e < MAT; e += T) {
          const int i = (int)(e / Dn), j = (int)(e - (size_t)i * Dn);
          const int jb = j / d, l = j - jb * d;
          // top: sigma LQ^T  (LQ = lq kron I)
          const int ib = i / d;
          M[(size_t)i * ldM + j] = ((i - ib * d) == l) ? sigma * LQ[jb * N + ib] : 0.0;
          // bottom-left: AL[j][i] = sum_{jb' >= jb} A1[jb][jb'] L_p[jb' d + l][i]
          double acc = pinvv[j] * S_U[(size_t)i * Dn + j];
          for (int k = jb + 1; k < N; ++k) acc = fma(Binom<N>::at(jb, k), pinvv[k * d + l] * S_U[(size_t)i * Dn + k * d + l], acc);
          M[(size_t)(Dn + i) * ldM + j] = acc;
          if (FIX) {
            M[(size_t)i * ldM + Dn + j] = 0.0;
            M[(size_t)(Dn + i) * ldM + Dn + j] = pinvv[j] * S_U[(size_t)i * Dn + j];
          }
        }
        __syncthreads();
        qr_blocked<NB>(M, ldM, W2, ldM, Dn, QR_TOPTRI_BOTFULL, Dn, qs);
        if (FIX) {
          solve_upper_blocked(M, W2, M + Dn, W2, X, Dn, Dn, Dn);
          for (size_t e = tid; e < MAT; e += T) {
            const int r = (int)(e / Dn), c = (int)(e - (size_t)r * Dn);
            GnT[e] = (pv[c] * X[e]) * pinvv[r];
            LnT[e] = pv[c] * M[(size_t)(Dn + r) * W2 + Dn + c];
            U_ext[e] = (c >= r) ? pv[c] * M[(size_t)r * W2 + c] : 0.0;
          }
          for (int i = tid; i < Dn; i += T) {
            double acc = m_p[i];
            for (int k = 0; k < Dn; ++k) acc = fma(-X[(size_t)k * Dn + i], m_ext_p[k], acc);
            gn[i] = pv[i] * acc;
          }
          __syncthreads();
          // merge with the running conditional (App. A.4), transposed storage
          gemm<false>(GmT, Dn, GnT, Dn, false, S_GT, Dn, Dn, Dn, Dn, nullptr, 0);
          for (int i = tid; i < Dn; i += T) {
            double acc = S_g[i];
            for (int k = 0; k < Dn; ++k) acc = fma(S_GT[(size_t)k * Dn + i], gn[k], acc);
            gm[i] = acc;
          }
          gemm<false>(M2, Dn, LnT, Dn, false, S_GT, Dn, Dn, Dn, Dn, nullptr, 0);
          for (size_t e = tid; e < MAT; e += T) M2[MAT + e] = S_LamU[e];
          __syncthreads();
          qr_blocked<NB>(M2, Dn, W2, Dn, Dn, QR_TOPFULL_BOTTRI, Dn, qs);
        } else {
          for (size_t e = tid; e < MAT; e += T) {
            const int r = (int)(e / Dn), c = (int)(e - (size_t)r * Dn);
            U_ext[e] = (c >= r) ? pv[c] * M[(size_t)r * Dn + c] : 0.0;
          }
          __syncthreads();
        }
      }
      // ---- correction (matrix observation, App. A.3 "EKF1 (dense)") ----------------------------------
      double e_norm = 0.0, fac = 1.0, le_now = 0.0;
      if (stepping) {
        // HLt[r][l] = sum_i H[l][i] L_ext[i][r] = sum_i H[l][i] U_ext[r][i]  (ascending i)
        for (size_t e = tid; e < (size_t)Dn * d; e += T) {
          const int r = (int)(e / d), l = (int)(e - (size_t)r * d);
          const int k = Hn[l];
          double acc = 0.0;
          for (int s = 0; s < k; ++s) acc = fma(Hv[l * H_MAX + s], U_ext[(size_t)r * Dn + Hc[l * H_MAX + s]], acc);
          HLt[e] = acc;
          Rm[e] = acc;
        }
        __syncthreads();
        qr_blocked<NB>(Rm, d, Dn, d, d, QR_FULL, 0, qs);
        // Wt[l][i] = sum_j L_ext[i][j] HL[l][j] = sum_j HLt[j][l] U_ext[j][i]
        gemm<false>(Wt, Dn, HLt, d, true, U_ext, Dn, d, Dn, Dn, nullptr, 0);
        solve_upper_transposed_cols(Rm, d, Wt, Dn, Yt, Dn, d, Dn);
        solve_upper_cols(Rm, d, Yt, Dn, gainT, Dn, d, Dn);
        // Mc = L_ext^T - HL^T gain^T = U_ext - HLt gainT
        gemm<true>(Mc, Dn, HLt, d, false, gainT, Dn, Dn, Dn, d, U_ext, Dn);
        qr_blocked<NB>(Mc, Dn, Dn, Dn, Dn, QR_FULL, 0, qs);
        for (int i = tid; i < Dn; i += T) {
          double acc = m_ext[i];
          for (int l = 0; l < d; ++l) acc = fma(-gainT[(size_t)l * Dn + i], zv[l], acc);
          m_new[i] = acc;
        }
        __syncthreads();
        for (int l = tid; l < d; l += T) ratio[l] = errv[l] * rcp(fma(rtol, fabs(m_new[l]), atol));
        __syncthreads();
        e_norm = dsqrt(cta_sum_squares(ratio, d, red)) * inv_sqrt_d;
        le_now = det_log(e_norm < 2.2250738585072014e-308 ? 2.2250738585072014e-308 : e_norm);
        le_now = (e_norm == 0.0) ? -745.0 : le_now;
        fac = a.safety * det_exp(fma(a.pow_p, le_prev, -((a.pow_i + a.pow_p) * le_now)));
        fac = (e_norm == 0.0) ? a.factor_max : fac;
        fac = (e_norm != e_norm) ? e_norm : fac;
        fac = (fac < a.factor_max) ? fac : a.factor_max;
        fac = (fac > a.factor_min) ? fac : a.factor_min;
      }
      // ================= bookkeeping (CTA-uniform) ======================================================
      auto copy_vec = [&](double* dst, const double* src, size_t count) {
        for (size_t e = tid; e < count; e += T) dst[e] = src[e];
      };
      auto copy_upper = [&](double* dst, const double* src, int lds) {  // D x D upper triangle, zeros below
        for (size_t e = tid; e < MAT; e += T) {
          const int r = (int)(e / Dn), c = (int)(e - (size_t)r * Dn);
          dst[e] = (c >= r) ? src[(size_t)r * lds + c] : 0.0;
        }
      };
      auto set_identity = [&]() {
        for (size_t e = tid; e < MAT; e += T) {
          const int i = (int)(e / Dn), j = (int)(e - (size_t)i * Dn);
          S_GT[e] = (i == j) ? 1.0 : 0.0;
          S_LamU[e] = 0.0;
        }
        for (int e = tid; e < Dn; e += T) S_g[e] = 0.0;
      };
      auto emit_cond = [&](double* dst, const double* GT_, const double* g_, const double* LamU_, int ldl) {
        for (size_t e = tid; e < MAT; e += T) {
          const int r = (int)(e / Dn), c = (int)(e - (size_t)r * Dn);
          dst[e] = GT_[e];
          dst[MAT + Dn + e] = (c >= r) ? LamU_[(size_t)r * ldl + c] : 0.0;
        }
        for (int e = tid; e < Dn; e += T) dst[MAT + e] = g_[e];
      };
      auto emit_identity_cond = [&](double* dst) {
        for (size_t e = tid; e < MAT; e += T) {
          dst[e] = ((e / Dn) == (e % Dn)) ? 1.0 : 0.0;
          dst[MAT + Dn + e] = 0.0;
        }
        for (int e = tid; e < Dn; e += T) dst[MAT + e] = 0.0;
      };
      auto emit_marg = [&](double* dst, const double* m_, const double* U_) {
        for (int e = tid; e < Dn; e += T) dst[e] = m_[e];
        for (size_t e = tid; e < MAT; e += T) dst[Dn + e] = U_[e];
      };
      auto commit_merged = [&]() {  // running conditional <- merged conditional of this step
        copy_vec(S_GT, GmT, MAT);
        copy_vec(S_g, gm, Dn);
        copy_upper(S_LamU, M2, Dn);
      };
      // filter: record the committed point (m_, U_ = L^T) as trajectory point n_acc.  The std of component l is
      // sqrt((L L^T)_ll), the sum of squares of column l of U in ascending row order (the zeros below the diagonal
      // add nothing); consecutive threads read consecutive columns
      auto record = [&](double tt, const double* m_, const double* U_) {
        if ((a.flags & FLAG_RECORD) && n_acc < a.traj_cap) {
          if (tid == 0) a.traj_t[n_acc * a.B + b] = tt;
          for (int l = tid; l < d; l += T) {
            double acc = 0.0;
            for (int j = 0; j <= l; ++j) acc = fma(U_[(size_t)j * Dn + l], U_[(size_t)j * Dn + l], acc);
            a.traj_u[(n_acc * d + l) * a.B + b] = m_[l];
            a.traj_std[(n_acc * d + l) * a.B + b] = dsqrt(acc);
          }
        }
      };
      auto resolve_hits = [&]() {
        while (k_next < a.K && !(t + TIME_EPS < grid_row(a, b)[k_next])) {
          double* slot = slot_base + (size_t)k_next * SLOT;
          __syncthreads();
          if (FIX) {
            emit_cond(slot, S_GT, S_g, S_LamU, Dn);
            if (k_next == a.K - 1) {
              emit_identity_cond(slot_base);
              emit_marg(slot_base + BW, S_m, S_U);
            }
            __syncthreads();
            set_identity();
          } else {
            emit_marg(slot, S_m, S_U);
          }
          if (tid == 0) a.n_accepted[b * a.K + k_next] = n_acc;
          if (tid == 0 && a.out_scale) a.out_scale[b * a.K + k_next] = sigma_state;
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
          copy_vec(S_m, P_m, Dn);
          copy_vec(S_U, P_U, MAT);
          if (FIX) commit_merged();
          mode = MODE_STEP;
          resolve_hits();
        }
      };
      __syncthreads();
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
              pend_sigma = sigma;
              copy_vec(P_m, m_new, Dn);
              copy_upper(P_U, Mc, Dn);
              mode = MODE_INTERP_A;
            } else {
              t = t1;
              sigma_state = sigma;
              copy_vec(S_m, m_new, Dn);
              copy_upper(S_U, Mc, Dn);
              if (FIX) commit_merged();
              if constexpr (!FIX) record(t1, m_new, Mc);  // only the upper triangle of Mc is the factor
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
          emit_cond(slot, GmT, gm, M2, Dn);
          __syncthreads();
          set_identity();
        } else {
          emit_marg(slot, m_ext, U_ext);
          if constexpr (!FIX) record(t_ck, m_ext, U_ext);
        }
        t = t_ck;
        copy_vec(S_m, m_ext, Dn);
        copy_vec(S_U, U_ext, MAT);
        if (tid == 0) a.n_accepted[b * a.K + k_next] = n_acc;
        if (tid == 0 && a.out_scale) a.out_scale[b * a.K + k_next] = pend_sigma;
        if (FIX) {
          mode = MODE_INTERP_B;
        } else {
          k_next += 1;
          after_checkpoint();
        }
      } else {
        if (k_next == a.K - 1) {
          emit_cond(slot_base, GmT, gm, M2, Dn);
          emit_marg(slot_base + BW, P_m, P_U);
        }
        k_next += 1;
        after_checkpoint();
      }
      __syncthreads();
    }
    if (tid == 0) {
      a.n_rejected[b] = n_rej;
      a.status[b] = st;
      if (st != 0)
        for (long long kk = k_next; kk < a.K; ++kk) a.n_accepted[b * a.K + kk] = n_acc;
      if constexpr (!FIX) {
        if (a.flags & FLAG_RECORD) a.traj_len[b] = (n_acc + 1 < a.traj_cap) ? (n_acc + 1) : a.traj_cap;
      }
    }
  }
}

// ---- backward marginalisation for the CTA-per-IVP dense family: one CTA per member -----------------
// rv_{k-1} = ( G_k m_k + g_k , R(QR([ (G_k L_k)^T ; Lam_k^T ]))^T )  (ivpsolvers.py:80-81, App. A.4/A.6)
struct CtaSmoothArgs {
  long long B, K;
  int d, n;
  const double* cond;
  double* scratch;  // per CTA: m, mo [D] + U [D*D] + M2 [2 D*D]
  const int32_t* status;
  double *u, *u_std, *marg_mean, *marg_chol;
};
__host__ __device__ inline size_t smooth_scratch_doubles(int Dn) { return 3 * (size_t)Dn * Dn + 2 * (size_t)Dn + 16; }

template <int STRAT, int NB>
__global__ void __launch_bounds__(T, 1) pn_dense_cta_smooth_kernel(const CtaSmoothArgs a) {
  constexpr bool FIX = (STRAT == 1);
  const int d = a.d, Dn = a.n * d, tid = threadIdx.x;
  const size_t MAT = (size_t)Dn * Dn, SLOT = slot_doubles(Dn, FIX), BW = 2 * MAT + Dn;
  extern __shared__ double smem[];
  QrSmem<NB> qs;
  qs.layout(Dn + NB);
  double* sc = a.scratch + (size_t)blockIdx.x * smooth_scratch_doubles(Dn);
  double* m = sc;          double* mo = m + Dn;
  double* U = mo + Dn;     double* M2 = U + MAT;
  const double nanv = __longlong_as_double(0x7ff8000000000000LL);
  for (long long b = blockIdx.x; b < a.B; b += gridDim.x) {
    const bool ok = (a.status[b] == 0);
    const double* base = a.cond + (size_t)b * a.K * SLOT;
    auto marginalise = [&](const double* c) {
      const double* GT = c;
      const double* gvec = c + MAT;
      const double* LamU = c + MAT + Dn;
      for (int i = tid; i < Dn; i += T) {
        double acc = gvec[i];
        for (int k = 0; k < Dn; ++k) acc = fma(GT[(size_t)k * Dn + i], m[k], acc);
        mo[i] = acc;
      }
      // M2 top = (G L)^T = U GT
      gemm<false>(M2, Dn, U, Dn, false, GT, Dn, Dn, Dn, Dn, nullptr, 0);
      for (size_t e = tid; e < MAT; e += T) M2[MAT + e] = LamU[e];
      __syncthreads();
      qr_blocked<NB>(M2, Dn, 2 * Dn, Dn, Dn, QR_TOPFULL_BOTTRI, Dn, qs);
      for (size_t e = tid; e < MAT; e += T) {
        const int r = (int)(e / Dn), cc = (int)(e - (size_t)r * Dn);
        U[e] = (cc >= r) ? M2[e] : 0.0;
      }
      for (int i = tid; i < Dn; i += T) m[i] = mo[i];
      __syncthreads();
    };
    __syncthreads();
    if (FIX) {
      for (int e = tid; e < Dn; e += T) m[e] = base[BW + e];
      for (size_t e = tid; e < MAT; e += T) U[e] = base[BW + Dn + e];
      __syncthreads();
      marginalise(base);
    }
    for (long long k = a.K - 1; k >= 0; --k) {
      if (!FIX) {
        for (int e = tid; e < Dn; e += T) m[e] = base[(size_t)k * SLOT + e];
        for (size_t e = tid; e < MAT; e += T) U[e] = base[(size_t)k * SLOT + Dn + e];
        __syncthreads();
      }
      for (int l = tid; l < d; l += T) {
        double acc = 0.0;  // row l of L = column l of U
        for (int j = 0; j < Dn; ++j) acc = fma(U[(size_t)j * Dn + l], U[(size_t)j * Dn + l], acc);
        a.u[((size_t)b * a.K + k) * d + l] = ok ? m[l] : nanv;
        a.u_std[((size_t)b * a.K + k) * d + l] = ok ? dsqrt(acc) : nanv;
      }
      if (a.marg_mean)
        for (int e = tid; e < Dn; e += T) a.marg_mean[((size_t)b * a.K + k) * Dn + e] = ok ? m[e] : nanv;
      if (a.marg_chol)
        for (size_t e = tid; e < MAT; e += T) {
          const int i = (int)(e / Dn), j = (int)(e - (size_t)i * Dn);  // L[i][j] = U[j][i]
          a.marg_chol[((size_t)b * a.K + k) * MAT + e] = ok ? U[(size_t)j * Dn + i] : nanv;
        }
      __syncthreads();
      if (k == 0) break;
      if (FIX) marginalise(base + (size_t)k * SLOT);
    }
  }
}

}  // namespace cta
}  // namespace pn
