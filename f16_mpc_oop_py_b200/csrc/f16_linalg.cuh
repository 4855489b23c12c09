// f16_linalg.cuh -- per-system bodies of the small dense algebra in f16_linalg.cu (one thread per system there).
//
//   reduce_one   element k of the 9-state / 3-input model gathered from an 18 x 18 forward Jacobian
//   zoh_one      cont2discrete(method='zoh'): expm([[A, B], [0, 0]] dt) -> Ad, Bd
//   dlqr_one     K = (B'PB + R)^-1 B'PA with P from the discrete algebraic Riccati equation (structured doubling)
//
// The same header compiles for the host (a development aid of the test-suite, as f16_model.cuh does), so the CPU tests check
// this arithmetic against mpmath and scipy too; the product library never contains a host path.  linalg.o is built with FMA contraction (-fmad=true) and
// the host build without it, so the two agree to rounding, not bit for bit.
#pragma once
#include <math.h>

#include "f16_model.cuh"  // F16_HD

namespace f16 {
namespace linalg {

constexpr int MAXD = 22;  // 18 states + 4 inputs

// dlqr_one's info[0] (include/f16_b200.h, dlqr_batch)
enum DlqrStatus {
  DLQR_OK = 0,
  DLQR_NOT_CONVERGED = 1,    // the tolerance was not met within max_doublings
  DLQR_R_SINGULAR = -1,
  DLQR_IGH_SINGULAR = -2,    // I + G H singular in a doubling
  DLQR_NONFINITE = -3,       // NaN or Inf in the data or in an iterate
  DLQR_RBPB_SINGULAR = -4,   // R + B'PB singular
  DLQR_NOT_STABILISING = -5, // converged to a solution P for which A - BK is not stable
  DLQR_NOT_A_SOLUTION = -6   // the doubling broke down: the P it converged to fails the Riccati residual test
};

F16_HD double la_nan() {
#if defined(__CUDA_ARCH__)
  return __longlong_as_double(0x7ff8000000000000LL);
#else
  return __builtin_nan("");
#endif
}

F16_HD void matmul(const double* X, const double* Y, double* Z, int n) {  // Z = X Y, n x n, ld MAXD
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++) {
      double a = 0;
      for (int k = 0; k < n; k++) a = fma(X[i * MAXD + k], Y[k * MAXD + j], a);
      Z[i * MAXD + j] = a;
    }
}

// exp(M) for an n x n matrix (ld MAXD), in place; T1, T2 scratch
F16_HD void expm(double* M, double* T1, double* T2, int n) {
  double norm = 0;
  for (int j = 0; j < n; j++) {
    double c = 0;
    for (int i = 0; i < n; i++) c += fabs(M[i * MAXD + j]);
    norm = fmax(norm, c);
  }
  int s = 0;
  if (norm > 0.5) {
    frexp(norm, &s);  // norm = f 2^s, f in [0.5, 1)
    s += 1;
    if (s < 0) s = 0;
    if (s > 60) s = 60;
  }
  const double sc = ldexp(1.0, -s);
  for (int i = 0; i < n * MAXD; i++) M[i] *= sc;
  // Horner form of sum_k M^k / k!, degree 14: T1 = I + M/14; T1 = I + (M/13) T1; ...
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++) T1[i * MAXD + j] = (i == j ? 1.0 : 0.0) + M[i * MAXD + j] * (1.0 / 14);
  for (int k = 13; k >= 1; k--) {
    matmul(M, T1, T2, n);
    const double inv = 1.0 / k;
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) T1[i * MAXD + j] = (i == j ? 1.0 : 0.0) + T2[i * MAXD + j] * inv;
  }
  for (int q = 0; q < s; q++) {
    matmul(T1, T1, T2, n);
    for (int i = 0; i < n * MAXD; i++) T1[i] = T2[i];
  }
  for (int i = 0; i < n * MAXD; i++) M[i] = T1[i];
}

// system p of a stack: A [N][n][n], B [N][n][m] -> Ad [N][n][n], Bd [N][n][m]; M, T1, T2 scratch of MAXD x MAXD
F16_HD void zoh_one(const double* A, const double* B, int n, int m, long long p, double dt, double* Ad, double* Bd, double* M,
                    double* T1, double* T2) {
  const int d = n + m;
  for (int i = 0; i < d; i++)
    for (int j = 0; j < d; j++) {
      double v = 0;
      if (i < n) v = (j < n ? A[p * n * n + i * n + j] : B[p * n * m + i * m + (j - n)]) * dt;
      M[i * MAXD + j] = v;
    }
  expm(M, T1, T2, d);
  for (int i = 0; i < n; i++) {
    for (int j = 0; j < n; j++) Ad[p * n * n + i * n + j] = M[i * MAXD + j];
    for (int j = 0; j < m; j++) Bd[p * n * m + i * m + j] = M[i * MAXD + n + j];
  }
}

// Z = X^-1 by Gauss-Jordan with partial pivoting (n <= 18, ld MAXD); returns false when singular
F16_HD bool invert(const double* X, double* Z, double* W, int n) {
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++) {
      W[i * MAXD + j] = X[i * MAXD + j];
      Z[i * MAXD + j] = i == j ? 1.0 : 0.0;
    }
  for (int c = 0; c < n; c++) {
    int piv = c;
    double best = fabs(W[c * MAXD + c]);
    for (int r = c + 1; r < n; r++)
      if (fabs(W[r * MAXD + c]) > best) { best = fabs(W[r * MAXD + c]); piv = r; }
    if (!(best > 0)) return false;
    if (piv != c)
      for (int j = 0; j < n; j++) {
        double t = W[c * MAXD + j]; W[c * MAXD + j] = W[piv * MAXD + j]; W[piv * MAXD + j] = t;
        t = Z[c * MAXD + j]; Z[c * MAXD + j] = Z[piv * MAXD + j]; Z[piv * MAXD + j] = t;
      }
    const double inv = 1.0 / W[c * MAXD + c];
    for (int j = 0; j < n; j++) { W[c * MAXD + j] *= inv; Z[c * MAXD + j] *= inv; }
    for (int r = 0; r < n; r++) {
      if (r == c) continue;
      const double f = W[r * MAXD + c];
      if (f == 0) continue;
      for (int j = 0; j < n; j++) {
        W[r * MAXD + j] = fma(-f, W[c * MAXD + j], W[r * MAXD + j]);
        Z[r * MAXD + j] = fma(-f, Z[c * MAXD + j], Z[r * MAXD + j]);
      }
    }
  }
  return true;
}

// Structured doubling for  P = A'PA - A'PB (R + B'PB)^-1 B'PA + Q:
//   A0 = A, G0 = B R^-1 B', H0 = Q;  W = (I + G H)^-1;  A+ = A W A;  G+ = G + A W G A';  H+ = H + A' H W A;  H -> P
// Started from H0 = Q, H converges to the smallest positive semi-definite solution.  That is the stabilising one when
// (A, Q) is detectable; when it is not (an unstable mode Q does not weigh), H still converges, to a P that leaves the
// mode unstable.  So a converged P passes two checks before it is reported (status 0):
//   it solves the equation: max|A'PA - P + Q - (B'PA)'K| <= 1e-5 (max|Q| + max|P| (1 + ||A||_1^2)), the right side an
//     upper bound of the terms' size.  A doubling can break down numerically (an undetectable mode growing A_k and G past
//     1e90, I + GH ill-conditioned beyond 1e50) and converge to an H that is not a solution: -6.
//   A - BK is stable: F = A - BK squared until ||F^(2^j)||_inf <= 1/2 (then rho(F) < 1), at most 64 times; F^(2^j)
//     overflowing or never getting there is -5.  The doubled matrix A_k is not the test: H can meet its tolerance
//     while A_k is still large (a slow stable mode Q does not weigh carries no P).
// System p of a stack; Q [n][n], R [m][m] shared.  Ak, G, H, W, T1, T2, T3: scratch of MAXD x MAXD.
F16_HD void dlqr_one(const double* Ad, const double* Bd, const double* Q, const double* R, int n, int m, long long p,
                     int max_doublings, double tol, double* K, double* P_out, int* info, double* Ak, double* G, double* H,
                     double* W, double* T1, double* T2, double* T3) {
  const double* A0 = Ad + p * n * n;
  const double* B0 = Bd + p * n * m;
  int status = DLQR_OK;
  // R^-1 (m x m) -> T1;  G = B R^-1 B'
  bool finite = true;  // an Inf in R or B can vanish from R^-1 and G: screen them as given
  for (int i = 0; i < m; i++)
    for (int j = 0; j < m; j++) {
      T2[i * MAXD + j] = R[i * m + j];
      finite &= (bool)isfinite(R[i * m + j]);
    }
  if (!invert(T2, T1, T3, m)) status = DLQR_R_SINGULAR;
  for (int i = 0; i < n; i++)
    for (int j = 0; j < m; j++) {  // T2 = B R^-1  (n x m)
      double a = 0;
      for (int k = 0; k < m; k++) a = fma(B0[i * m + k], T1[k * MAXD + j], a);
      T2[i * MAXD + j] = a;
      finite &= (bool)isfinite(B0[i * m + j]);
    }
  double a0norm1 = 0;  // ||A0||_1
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++) {
      double a = 0;
      for (int k = 0; k < m; k++) a = fma(T2[i * MAXD + k], B0[j * m + k], a);
      G[i * MAXD + j] = a;
      Ak[i * MAXD + j] = A0[i * n + j];
      H[i * MAXD + j] = Q[i * n + j];
      finite &= isfinite(a) && isfinite(A0[i * n + j]) && isfinite(Q[i * n + j]);
    }
  for (int j = 0; j < n; j++) {
    double c = 0;
    for (int i = 0; i < n; i++) c += fabs(A0[i * n + j]);
    a0norm1 = fmax(a0norm1, c);
  }
  if (status == DLQR_OK && !finite) status = DLQR_NONFINITE;
  bool converged = false;
  int it = 0;
  for (; it < max_doublings && status == DLQR_OK; it++) {
    matmul(G, H, T1, n);  // T1 = I + G H
    for (int i = 0; i < n; i++) T1[i * MAXD + i] += 1.0;
    if (!invert(T1, W, T2, n)) { status = DLQR_IGH_SINGULAR; break; }
    matmul(Ak, W, T1, n);                       // T1 = A W
    matmul(T1, G, T2, n);                       // T2 = A W G
    for (int i = 0; i < n; i++)                 // G += A W G A'
      for (int j = 0; j < n; j++) {
        double a = 0;
        for (int k = 0; k < n; k++) a = fma(T2[i * MAXD + k], Ak[j * MAXD + k], a);
        T3[i * MAXD + j] = a;
      }
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) {
        G[i * MAXD + j] += T3[i * MAXD + j];
        finite &= (bool)isfinite(G[i * MAXD + j]);
      }
    matmul(W, Ak, T2, n);                       // T2 = W A
    matmul(H, T2, T3, n);                       // T3 = H W A
    bool h_finite = true;
    double dmax = 0, hmax = 0;
    for (int i = 0; i < n; i++)                 // H += A' H W A
      for (int j = 0; j < n; j++) {
        double a = 0;
        for (int k = 0; k < n; k++) a = fma(Ak[k * MAXD + i], T3[k * MAXD + j], a);
        T2[i * MAXD + j] = a;
      }
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) {
        H[i * MAXD + j] += T2[i * MAXD + j];
        h_finite &= (bool)isfinite(H[i * MAXD + j]);
        dmax = fmax(dmax, fabs(T2[i * MAXD + j]));
        hmax = fmax(hmax, fabs(H[i * MAXD + j]));
      }
    matmul(T1, Ak, T2, n);                      // A <- A W A
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) {
        Ak[i * MAXD + j] = T2[i * MAXD + j];
        finite &= (bool)isfinite(T2[i * MAXD + j]);
      }
    // fmax skips NaN, so dmax and hmax cannot carry the divergence test: every update is screened above.  A_k or G
    // overflowing in the doubling where H converges is the non-stabilising case, not a divergence of P.
    if (!h_finite) { status = DLQR_NONFINITE; it++; break; }
    if (dmax <= tol * hmax) { converged = true; status = finite ? DLQR_OK : DLQR_NOT_STABILISING; it++; break; }
    if (!finite) { status = DLQR_NONFINITE; it++; break; }
  }
  if (status == DLQR_OK && !converged) status = DLQR_NOT_CONVERGED;
  // symmetrise P, K = (R + B'PB)^-1 B'PA
  for (int i = 0; i < n; i++)
    for (int j = i + 1; j < n; j++) {
      const double v = 0.5 * (H[i * MAXD + j] + H[j * MAXD + i]);
      H[i * MAXD + j] = v;
      H[j * MAXD + i] = v;
    }
  for (int i = 0; i < m; i++)                   // T1 = B'P  (m x n)
    for (int j = 0; j < n; j++) {
      double a = 0;
      for (int k = 0; k < n; k++) a = fma(B0[k * m + i], H[k * MAXD + j], a);
      T1[i * MAXD + j] = a;
    }
  for (int i = 0; i < m; i++)                   // T2 = R + B'PB (m x m)
    for (int j = 0; j < m; j++) {
      double a = R[i * m + j];
      for (int k = 0; k < n; k++) a = fma(T1[i * MAXD + k], B0[k * m + j], a);
      T2[i * MAXD + j] = a;
    }
  if (!invert(T2, W, T3, m) && status == DLQR_OK) status = DLQR_RBPB_SINGULAR;
  for (int i = 0; i < m; i++)                   // T3 = B'PA (m x n)
    for (int j = 0; j < n; j++) {
      double a = 0;
      for (int k = 0; k < n; k++) a = fma(T1[i * MAXD + k], A0[k * n + j], a);
      T3[i * MAXD + j] = a;
    }
  for (int i = 0; i < m; i++)                   // G = K (m x n)
    for (int j = 0; j < n; j++) {
      double a = 0;
      for (int k = 0; k < m; k++) a = fma(W[i * MAXD + k], T3[k * MAXD + j], a);
      G[i * MAXD + j] = a;
    }
  if (status == DLQR_OK) {  // the Riccati residual A'PA - P + Q - (B'PA)'K against the size of its terms
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) Ak[i * MAXD + j] = A0[i * n + j];
    matmul(H, Ak, T2, n);                       // T2 = P A
    double rmax = 0, pmax = 0, qmax = 0;
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) {
        double a = Q[i * n + j] - H[i * MAXD + j];
        for (int k = 0; k < n; k++) a = fma(Ak[k * MAXD + i], T2[k * MAXD + j], a);
        for (int k = 0; k < m; k++) a = fma(-T3[k * MAXD + i], G[k * MAXD + j], a);
        rmax = fmax(rmax, fabs(a));
        pmax = fmax(pmax, fabs(H[i * MAXD + j]));
        qmax = fmax(qmax, fabs(Q[i * n + j]));
      }
    if (!(rmax <= 1e-5 * (qmax + pmax * (1.0 + a0norm1 * a0norm1)))) status = DLQR_NOT_A_SOLUTION;
  }
  if (status == DLQR_OK) {  // A - BK stable: ||(A - BK)^(2^j)||_inf <= 1/2 for some j <= 64, so rho^(2^j) <= 1/2
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) {
        double a = A0[i * n + j];
        for (int k = 0; k < m; k++) a = fma(-B0[i * m + k], G[k * MAXD + j], a);
        Ak[i * MAXD + j] = a;
      }
    bool stable = false;
    for (int q = 0; q <= 64; q++) {
      double fnorm = 0;
      bool fin = true;
      for (int i = 0; i < n; i++) {
        double r = 0;
        for (int j = 0; j < n; j++) r += fabs(Ak[i * MAXD + j]);
        fin &= (bool)isfinite(r);
        fnorm = fmax(fnorm, r);
      }
      if (!fin) break;  // grown past the double range: unstable
      if (fnorm <= 0.5) { stable = true; break; }
      if (q == 64) break;
      matmul(Ak, Ak, T2, n);
      for (int i = 0; i < n; i++)
        for (int j = 0; j < n; j++) Ak[i * MAXD + j] = T2[i * MAXD + j];
    }
    if (!stable) status = DLQR_NOT_STABILISING;
  }
  for (int i = 0; i < m; i++)
    for (int j = 0; j < n; j++) K[p * m * n + i * n + j] = status < 0 ? la_nan() : G[i * MAXD + j];
  if (P_out)
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) P_out[p * n * n + i * n + j] = H[i * MAXD + j];
  if (info) {
    info[2 * p] = status;
    info[2 * p + 1] = it;
  }
}

// element k in [0, 108) of system p: A [N][18][18] -> A_na [N][9][9] (k % 12 < 9) or B_na [N][9][3]
// rows of the reduced model in full-state numbering (lf2dot, lf1dot swapped as env.py:184,189 does);
// columns: mpc_states = {phi, theta, alpha, beta, p, q, r, lf1, lf2} (parameters.py:135), inputs -> actuator states 13..15
F16_HD void reduce_one(const double* A, long long p, int k, double* A_na, double* B_na) {
  const int rows[9] = {3, 4, 7, 8, 9, 10, 11, 16, 17};
  const int cols[12] = {3, 4, 7, 8, 9, 10, 11, 17, 16, 13, 14, 15};
  const int i = k / 12, j = k - i * 12;
  const double v = A[p * 324 + rows[i] * 18 + cols[j]];
  if (j < 9) A_na[p * 81 + i * 9 + j] = v;
  else B_na[p * 27 + i * 3 + (j - 9)] = v;
}

}  // namespace linalg
}  // namespace f16
