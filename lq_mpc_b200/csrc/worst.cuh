// worst.cuh — exact gradient of the unconstrained law's closed-loop cost J_inf in the model error (dA, dB), and a
// projected ascent over the error set {||dA|| <= e_A, ||dB|| <= e_B}. One sample per thread.
//
// Forward pass (riccati.cuh's recursion on A^ = A + dA, B^ = B + dB): P(0) = Pt, for k = 1..N
//   G_k = R + B^'P(k-1)B^,  K(k) = -G_k^-1 B^'P(k-1)A^,  P(k) = Q + A^'(P(k-1) - P(k-1)B^ G_k^-1 B^'P(k-1))A^  (k < N),
// K0 = K(N). Closed loop on the TRUE plant: A_cl = A + B K0, W = Q + K0'R K0, S = W + A_cl'S A_cl, J = x0'S x0.
//
// Adjoint. With Lambda = x0 x0' + A_cl Lambda A_cl' (the state Gramian sum_k x_k x_k'), dJ/dK0 = 2(R K0 + B'S A_cl)
// Lambda = Kbar. K0 = -G^-1 B^'P A^ with P = P(N-1), G = G_N, F = A^ + B^ K0 and Z = G^-1 Kbar give
//   dJ/dA^ = -P B^ Z,  dJ/dB^ = -P F Z' - P B^ Z K0',  and dJ/dP = Pbar = -(F Z'B^' + B^ Z F')/2.
// P(k) written in Joseph form, Q + K'R K + (A^ + B^K)'P(k-1)(A^ + B^K), is stationary in K at the optimal gain K(k)
// (envelope theorem), so the reverse sweep k = N-1..1 needs no derivative of the gains: with F_k = A^ + B^ K(k),
//   X = 2 P(k-1) F_k Pbar,  dJ/dA^ += X,  dJ/dB^ += X K(k)',  Pbar <- F_k Pbar F_k'.
// The sweep reads the pairs (P(k-1), K(k)), k = 1..N-1, that the forward pass stores in the strided workspace.
//
// Sup over the initial state (SUP = true). The performance ratio J / V_expert = x0'S x0 / x0'P_exp x0 is a Rayleigh
// quotient, so its worst case over x0 is gamma = lambda_max(L^-1 S L^-T), P_exp = L L', attained at x* = L^-T w (w the
// top eigenvector). J := gamma replaces x0'S x0, and where lambda_max is simple dgamma = x*'dS x*: the adjoint above
// with x0 = x*. Where it is repeated gamma has an upward kink, which an ascent is not trapped by.
#pragma once
#include "clqr.cuh"

namespace lq {

constexpr int FLAG_ASCENT_MAXITER = 2048;   // the ascent's iteration budget ran out before the stationarity test held
// flags after which a value or gradient is not usable
constexpr int kWorstFail = FLAG_CHOL_FAIL | FLAG_LYAP_NOCONV | FLAG_EIG_NOCONV | FLAG_NONFINITE;
constexpr int kWorstMaxBacktrack = 60;      // step shrinks by 4^60 ~ 1e36 before the line search gives up

// stage records of one sample: the upper triangle of P(k-1) and the gain K(k), k = 1..N-1
template <int n, int m>
LQ_HD int64_t worst_ws_doubles(int N) {
  return (int64_t)(N > 1 ? N - 1 : 0) * (n * (n + 1) / 2 + m * n);
}

// out (R x C) = A (R x K) * B' with B (C x K)
template <int R, int K, int C>
LQ_HD void mmt(const double* A, const double* B, double* out) {
  LQ_UNROLL for (int i = 0; i < R; ++i)
    LQ_UNROLL for (int j = 0; j < C; ++j) {
      double acc = A[i * K] * B[j * K];
      LQ_UNROLL for (int k = 1; k < K; ++k) acc = fma(A[i * K + k], B[j * K + k], acc);
      out[i * C + j] = acc;
    }
}

// Solve L Y = X (forward) with the reciprocal diagonal of chol_inv; X is (m x c), overwritten.
template <int m, int c>
LQ_HD void solve_l_inv(const double* L, const double* dinv, double* X) {
  LQ_UNROLL for (int j = 0; j < c; ++j)
    LQ_UNROLL for (int i = 0; i < m; ++i) {
      double s = X[i * c + j];
      LQ_UNROLL for (int k = 0; k < i; ++k) s = fma(-L[i * m + k], X[k * c + j], s);
      X[i * c + j] = s * dinv[i];
    }
}

// The Cholesky factor of the constant expert matrix, P_exp = L L' (chol_inv: reciprocal diagonal in Li), formed once
// per thread for the SUP mode.
template <int n>
struct ExpertFactor {
  double L[n * n], Li[n];
  bool ok;
};

template <int n, int m>
LQ_HD ExpertFactor<n> expert_factor(const Problem<n, m>& pb) {
  ExpertFactor<n> f;
  LQ_UNROLL for (int i = 0; i < n * n; ++i) f.L[i] = pb.Pexp[i];
  f.ok = chol_inv<n>(f.L, f.Li);
  return f;
}

// gamma = lambda_max(L^-1 S L^-T), the worst state x* = L^-T w (normalised to x*'P_exp x* = 1, its entry of largest
// magnitude positive, ties to the lowest index) and the relative eigengap (lambda_1 - lambda_2) / lambda_1 (1 at n = 1).
// Returns CHOL_FAIL (P_exp not positive definite; all outputs NaN) or EIG_NOCONV (Jacobi off its tolerance).
template <int n>
LQ_HD int sup_ratio(const ExpertFactor<n>& ef, const double* S, double* gamma, double* xs, double* gap) {
  if (!ef.ok) {
    *gamma = *gap = NAN;
    LQ_UNROLL for (int i = 0; i < n; ++i) xs[i] = NAN;
    return FLAG_CHOL_FAIL;
  }
  double T[n * n], M[n * n];
  LQ_UNROLL for (int i = 0; i < n * n; ++i) T[i] = S[i];
  solve_l_inv<n, n>(ef.L, ef.Li, T);             // L^-1 S
  LQ_UNROLL for (int i = 0; i < n; ++i)
    LQ_UNROLL for (int j = 0; j < n; ++j) M[i * n + j] = T[j * n + i];
  solve_l_inv<n, n>(ef.L, ef.Li, M);             // L^-1 (L^-1 S)' = L^-1 S L^-T
  LQ_UNROLL for (int i = 0; i < n; ++i)
    LQ_UNROLL for (int j = i + 1; j < n; ++j) M[i * n + j] = M[j * n + i] = 0.5 * (M[i * n + j] + M[j * n + i]);
  double w[n], V[n * n];
  const bool conv = sym_eig_jacobi<n>(M, w, V);
  // the top eigenpair by selects (no dynamic index into registers)
  double l1 = w[0], l2 = -HUGE_VAL, v[n];
  LQ_UNROLL for (int i = 0; i < n; ++i) v[i] = V[i * n];
  LQ_UNROLL for (int j = 1; j < n; ++j) {
    const bool top = w[j] > l1;
    l2 = dmax(l2, top ? l1 : w[j]);
    l1 = top ? w[j] : l1;
    LQ_UNROLL for (int i = 0; i < n; ++i) v[i] = top ? V[i * n + j] : v[i];
  }
  double vv = 0.0;
  LQ_UNROLL for (int i = 0; i < n; ++i) vv = fma(v[i], v[i], vv);
  vv = 1.0 / sqrt(vv);
  LQ_UNROLL for (int i = 0; i < n; ++i) v[i] *= vv;
  solve_lt_inv<n, 1>(ef.L, ef.Li, v);
  double big = v[0];
  LQ_UNROLL for (int i = 1; i < n; ++i) big = (fabs(v[i]) > fabs(big)) ? v[i] : big;
  LQ_UNROLL for (int i = 0; i < n; ++i) xs[i] = (big < 0.0) ? -v[i] : v[i];
  *gamma = l1;
  *gap = (n == 1) ? 1.0 : (l1 - l2) / l1;
  return conv ? 0 : FLAG_EIG_NOCONV;
}

// J (and rho) at the model error (dA, dB); with gA / gB non-null also dJ/d(dA) [n*n] and dJ/d(dB) [n*m] (NaN where the
// value is unstable or failed). Returns the flags: CHOL_FAIL of any stage, EIG_NOCONV, UNSTABLE (J = +inf),
// LYAP_NOCONV, NONFINITE. ws holds worst_ws_doubles<n, m>(N) doubles and is written only for the gradient.
// SUP: J is gamma (x0 is not read); the factor ef of P_exp is an input, x* [n] and the eigengap go to xs and gap (NaN
// where the loop is unstable or P_exp has no Cholesky factor), and the gradient is that of gamma.
template <int n, int m, bool SUP = false>
LQ_HD int worst_eval(const Problem<n, m>& pb, const double* dA, const double* dB, const double* x0, int N,
                     const WsView& ws, double* J_out, double* rho_out, double* gA, double* gB,
                     const ExpertFactor<n>* ef = nullptr, double* xs = nullptr, double* gap = nullptr) {
  constexpr int ps = n * (n + 1) / 2, rs = ps + m * n;
  const bool grad = gA != nullptr;
  double Ah[n * n], Bh[n * m], P[n * n], K0[m * n];
  LQ_UNROLL for (int i = 0; i < n * n; ++i) { Ah[i] = pb.A[i] + dA[i]; P[i] = pb.Pt[i]; }
  LQ_UNROLL for (int i = 0; i < n * m; ++i) Bh[i] = pb.B[i] + dB[i];
  RicStage<n, m> st;
  int flags = 0;
  for (int k = 1; k < N; ++k) {
    riccati_factor<n, m>(P, Bh, pb.R, st);
    if (!st.ok) flags |= FLAG_CHOL_FAIL;
    if (grad) {
      const int64_t o = (int64_t)(k - 1) * rs;
      int e = 0;
      LQ_UNROLL for (int i = 0; i < n; ++i)
        LQ_UNROLL for (int j = i; j < n; ++j) ws[o + e++] = P[i * n + j];
      riccati_gain<n, m>(st, Ah, K0);
      LQ_UNROLL for (int i = 0; i < m * n; ++i) ws[o + ps + i] = K0[i];
    }
    riccati_update<n, m>(st, Ah, pb.Q, P);
  }
  riccati_factor<n, m>(P, Bh, pb.R, st);        // horizon N: P = P(N-1), st holds G_N = L L'
  if (!st.ok) flags |= FLAG_CHOL_FAIL;
  riccati_gain<n, m>(st, Ah, K0);

  double Acl[n * n], W[n * n], RK[m * n], S[n * n];
  LQ_UNROLL for (int i = 0; i < n; ++i)
    LQ_UNROLL for (int j = 0; j < n; ++j) {
      double acc = pb.A[i * n + j];
      LQ_UNROLL for (int k = 0; k < m; ++k) acc = fma(pb.B[i * m + k], K0[k * n + j], acc);
      Acl[i * n + j] = acc;
    }
  mm<m, m, n>(pb.R, K0, RK);
  sym_add_mtm<m, n>(pb.Q, K0, RK, W);
  bool ok;
  const double rho = spectral_radius<n>(Acl, &ok);
  if (!ok) flags |= FLAG_EIG_NOCONV;
  *rho_out = rho;
  if (grad) {
    LQ_UNROLL for (int i = 0; i < n * n; ++i) gA[i] = NAN;
    LQ_UNROLL for (int i = 0; i < n * m; ++i) gB[i] = NAN;
  }
  if (!(rho < 1.0)) {
    *J_out = HUGE_VAL;
    if constexpr (SUP) {
      *gap = NAN;
      LQ_UNROLL for (int i = 0; i < n; ++i) xs[i] = NAN;
    }
    return flags | FLAG_UNSTABLE;
  }
  if (!lyapunov_doubling<n>(Acl, W, S)) flags |= FLAG_LYAP_NOCONV;
  double J;
  if constexpr (SUP) {
    flags |= sup_ratio<n>(*ef, S, &J, xs, gap);
    x0 = xs;                                     // the Gramian below is seeded with x* x*'
  } else {
    J = quad<n>(x0, S, x0);
  }
  if (!(fabs(J) <= 1.79e308)) flags |= FLAG_NONFINITE;
  *J_out = J;
  if (!grad || (flags & kWorstFail)) return flags;

  double Lam[n * n];
  {
    double AclT[n * n], X0[n * n];
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = 0; j < n; ++j) { AclT[i * n + j] = Acl[j * n + i]; X0[i * n + j] = x0[i] * x0[j]; }
    if (!lyapunov_doubling<n>(AclT, X0, Lam)) return flags | FLAG_LYAP_NOCONV;
  }
  double Z[m * n];                               // Z = G^-1 Kbar, Kbar = 2 (R K0 + B'S A_cl) Lambda
  {
    double SA[n * n], T[m * n];
    mm<n, n, n>(S, Acl, SA);
    mtm<n, m, n>(pb.B, SA, T);
    LQ_UNROLL for (int i = 0; i < m * n; ++i) T[i] = 2.0 * (T[i] + RK[i]);
    mm<m, n, n>(T, Lam, Z);
  }
  solve_l_inv<m, n>(st.L, st.Li, Z);
  solve_lt_inv<m, n>(st.L, st.Li, Z);
  double F[n * n], PB[n * m], Pbar[n * n];
  LQ_UNROLL for (int i = 0; i < n; ++i)
    LQ_UNROLL for (int j = 0; j < n; ++j) {
      double acc = Ah[i * n + j];
      LQ_UNROLL for (int k = 0; k < m; ++k) acc = fma(Bh[i * m + k], K0[k * n + j], acc);
      F[i * n + j] = acc;
    }
  mm<n, n, m>(P, Bh, PB);
  {
    double T[n * n], ZK[m * m], U[n * m];
    mm<n, m, n>(PB, Z, T);
    LQ_UNROLL for (int i = 0; i < n * n; ++i) gA[i] = -T[i];
    mm<n, n, n>(P, F, T);                        // P F
    mmt<n, n, m>(T, Z, U);                       // P F Z'
    mmt<m, n, m>(Z, K0, ZK);                     // Z K0'
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = 0; j < m; ++j) {
        double acc = U[i * m + j];
        LQ_UNROLL for (int k = 0; k < m; ++k) acc = fma(PB[i * m + k], ZK[k * m + j], acc);
        gB[i * m + j] = -acc;
      }
    mmt<n, n, m>(F, Z, U);                       // U = F Z'
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = i; j < n; ++j) {
        double acc = 0.0;
        LQ_UNROLL for (int k = 0; k < m; ++k) acc = fma(U[i * m + k], Bh[j * m + k], fma(Bh[i * m + k], U[j * m + k], acc));
        Pbar[i * n + j] = Pbar[j * n + i] = -0.5 * acc;
      }
  }
  for (int k = N - 1; k >= 1; --k) {
    const int64_t o = (int64_t)(k - 1) * rs;
    double Pk[n * n], Kk[m * n], Fk[n * n], T[n * n], X[n * n];
    int e = 0;
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = i; j < n; ++j) { const double v = ws[o + e++]; Pk[i * n + j] = v; Pk[j * n + i] = v; }
    LQ_UNROLL for (int i = 0; i < m * n; ++i) Kk[i] = ws[o + ps + i];
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = 0; j < n; ++j) {
        double acc = Ah[i * n + j];
        LQ_UNROLL for (int l = 0; l < m; ++l) acc = fma(Bh[i * m + l], Kk[l * n + j], acc);
        Fk[i * n + j] = acc;
      }
    mm<n, n, n>(Pk, Fk, T);
    mm<n, n, n>(T, Pbar, X);
    LQ_UNROLL for (int i = 0; i < n * n; ++i) gA[i] = fma(2.0, X[i], gA[i]);
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = 0; j < m; ++j) {
        double acc = 0.0;
        LQ_UNROLL for (int l = 0; l < n; ++l) acc = fma(X[i * n + l], Kk[j * n + l], acc);
        gB[i * m + j] = fma(2.0, acc, gB[i * m + j]);
      }
    mm<n, n, n>(Fk, Pbar, T);
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = i; j < n; ++j) {
        double acc = 0.0;
        LQ_UNROLL for (int l = 0; l < n; ++l) acc = fma(T[i * n + l], Fk[j * n + l], acc);
        Pbar[i * n + j] = Pbar[j * n + i] = acc;
      }
  }
  return flags;
}

// ---- the error set. norm: 0 = Frobenius, 1 = spectral, 2 = entrywise max (K6's codes, then lqmpc_eval_seeded's box)

template <int len>
LQ_HD double fro2(const double* M) {
  double s = 0.0;
  LQ_UNROLL for (int i = 0; i < len; ++i) s = fma(M[i], M[i], s);
  return s;
}

// Rescale the (r x c) block M until the norm measured by `nrm` is <= e (rounding of the first rescale only).
template <int len, class Norm>
LQ_HD void shrink_to(double* M, double e, Norm nrm) {
  for (int it = 0; it < 8; ++it) {
    const double v = nrm(M);
    if (v <= e) return;
    const double c = (e / v) * (1.0 - 0x1p-52);
    LQ_UNROLL for (int i = 0; i < len; ++i) M[i] *= c;
  }
}

// Euclidean projection of the (r x c) block M onto {||M|| <= e}; a point inside is returned unchanged.
template <int r, int c>
LQ_HD void worst_project(double* M, double e, int norm) {
  constexpr int len = r * c;
  if (!(e > 0.0)) {
    LQ_UNROLL for (int i = 0; i < len; ++i) M[i] = 0.0;
    return;
  }
  if (norm == 2) {
    LQ_UNROLL for (int i = 0; i < len; ++i) M[i] = dmin(dmax(M[i], -e), e);
  } else if (norm == 0) {
    shrink_to<len>(M, e, [](const double* X) { return sqrt(fro2<len>(X)); });
  } else {
    if (norm2<r, c>(M) <= e) return;
    // M'M = V Sigma^2 V':  M <- M V diag(min(1, e / sigma_i)) V'
    double G[c * c], w[c], V[c * c], T[c * c];
    LQ_UNROLL for (int i = 0; i < c; ++i)
      LQ_UNROLL for (int j = i; j < c; ++j) {
        double s = 0.0;
        LQ_UNROLL for (int k = 0; k < r; ++k) s = fma(M[k * c + i], M[k * c + j], s);
        G[i * c + j] = G[j * c + i] = s;
      }
    sym_eig_jacobi<c>(G, w, V);
    LQ_UNROLL for (int k = 0; k < c; ++k) w[k] = (w[k] > e * e) ? e / sqrt(w[k]) : 1.0;
    LQ_UNROLL for (int i = 0; i < c; ++i)
      LQ_UNROLL for (int j = 0; j < c; ++j) {
        double s = 0.0;
        LQ_UNROLL for (int k = 0; k < c; ++k) s = fma(V[i * c + k] * w[k], V[j * c + k], s);
        T[i * c + j] = s;
      }
    double out[len];
    mm<r, c, c>(M, T, out);
    LQ_UNROLL for (int i = 0; i < len; ++i) M[i] = out[i];
    shrink_to<len>(M, e, [](const double* X) { return norm2<r, c>(X); });
  }
}

// out = Proj(M + h g) for one block; returns ||out - M||^2 / e^2 (0 for an e = 0 block)
template <int r, int c>
LQ_HD double worst_step(const double* M, const double* g, double h, double e, int norm, double* out) {
  if (!(e > 0.0)) {
    LQ_UNROLL for (int i = 0; i < r * c; ++i) out[i] = 0.0;
    return 0.0;
  }
  LQ_UNROLL for (int i = 0; i < r * c; ++i) out[i] = fma(h, g[i], M[i]);
  worst_project<r, c>(out, e, norm);
  double s = 0.0;
  LQ_UNROLL for (int i = 0; i < r * c; ++i) { const double d = out[i] - M[i]; s = fma(d, d, s); }
  return s / (e * e);
}

struct AscentSettings {
  double eA, eB, tol;
  int norm, max_iter;
};

// Projected ascent of J over the error set from (dA, dB), both overwritten with the result. The iteration runs in the
// normalised coordinates u = (dA / e_A, dB / e_B) with gradient g^ = (e_A dJ/d(dA), e_B dJ/d(dB)):
//   * project the start; at every accepted point the stationarity residual is r = ||Proj(u + g^/||g^||) - u||_2
//     (0 when g^ = 0) and the ascent stops when r <= tol;
//   * trial u+ = Proj(u + t g^), the first t = 0.5 / ||g^||, then Barzilai-Borwein t = s's / (-s'y) when s'y < 0 and
//     10 t otherwise; accepted when J(u+) >= J(u) + 1e-4 g^.(u+ - u), else t <- t / 4;
//   * trials take the value only, the gradient is computed at accepted points;
//   * an unstable trial lies in the set and destabilises the loop: it is the result (J = +inf, UNSTABLE);
//   * a trial with another failure flag is rejected; a start with one ends the ascent there;
//   * the budget of max_iter accepted steps (or a line search that shrinks t by 4^60) ends it with ASCENT_MAXITER.
// Returns the flags of the final point; J, rho and the accepted-step count go to the outputs.
// SUP: the ascent of gamma (worst_eval's SUP mode; x0 is not read) with x* of the final point in xs [n].
template <int n, int m, bool SUP = false>
LQ_HD int worst_ascent(const Problem<n, m>& pb, double* dA, double* dB, const double* x0, int N,
                       const AscentSettings& as, const WsView& ws, double* J_out, double* rho_out, int* iters,
                       const ExpertFactor<n>* ef = nullptr, double* xs = nullptr) {
  const double eA2 = as.eA * as.eA, eB2 = as.eB * as.eB;
  worst_project<n, n>(dA, as.eA, as.norm);
  worst_project<n, m>(dB, as.eB, as.norm);
  double gA[n * n], gB[n * m], J, rho, gap, xt[n];
  int flags = worst_eval<n, m, SUP>(pb, dA, dB, x0, N, ws, &J, &rho, gA, gB, ef, xs, &gap);
  int it = 0;
  double t = 0.0;
  while (!(flags & (kWorstFail | FLAG_UNSTABLE))) {
    const double gn2 = eA2 * fro2<n * n>(gA) + eB2 * fro2<n * m>(gB);
    if (!(gn2 > 0.0)) break;                              // g^ = 0: r = 0
    const double gn = sqrt(gn2);
    double tA[n * n], tB[n * m];
    const double r2 = worst_step<n, n>(dA, gA, eA2 / gn, as.eA, as.norm, tA) +
                      worst_step<n, m>(dB, gB, eB2 / gn, as.eB, as.norm, tB);
    if (sqrt(r2) <= as.tol) break;
    if (it >= as.max_iter) { flags |= FLAG_ASCENT_MAXITER; break; }
    if (it == 0) t = 0.5 / gn;
    double Jt = 0.0, rt = 0.0, ss = 0.0;
    int ft = 0;
    bool accepted = false;
    for (int bt = 0; bt < kWorstMaxBacktrack; ++bt) {
      ss = worst_step<n, n>(dA, gA, t * eA2, as.eA, as.norm, tA) + worst_step<n, m>(dB, gB, t * eB2, as.eB, as.norm, tB);
      double dot = 0.0;
      LQ_UNROLL for (int i = 0; i < n * n; ++i) dot = fma(gA[i], tA[i] - dA[i], dot);
      LQ_UNROLL for (int i = 0; i < n * m; ++i) dot = fma(gB[i], tB[i] - dB[i], dot);
      ft = worst_eval<n, m, SUP>(pb, tA, tB, x0, N, ws, &Jt, &rt, nullptr, nullptr, ef, xt, &gap);
      if ((ft & FLAG_UNSTABLE) || (!(ft & kWorstFail) && Jt >= J + 1e-4 * dmax(dot, 0.0))) { accepted = true; break; }
      t *= 0.25;
    }
    if (!accepted) { flags |= FLAG_ASCENT_MAXITER; break; }
    ++it;
    if (ft & FLAG_UNSTABLE) {
      LQ_UNROLL for (int i = 0; i < n * n; ++i) dA[i] = tA[i];
      LQ_UNROLL for (int i = 0; i < n * m; ++i) dB[i] = tB[i];
      if constexpr (SUP) { LQ_UNROLL for (int i = 0; i < n; ++i) xs[i] = xt[i]; }
      J = Jt; rho = rt; flags = ft;
      break;
    }
    // the gradient at the accepted point (its value repeats the trial's bit for bit). With s = u+ - u and
    // y = g^+ - g^, s'y = (dA+ - dA).(gA+ - gA) + (dB+ - dB).(gB+ - gB): the scales e cancel.
    double nA[n * n], nB[n * m], sy = 0.0;
    flags = worst_eval<n, m, SUP>(pb, tA, tB, x0, N, ws, &J, &rho, nA, nB, ef, xs, &gap);
    LQ_UNROLL for (int i = 0; i < n * n; ++i) {
      sy = fma(tA[i] - dA[i], nA[i] - gA[i], sy);
      dA[i] = tA[i]; gA[i] = nA[i];
    }
    LQ_UNROLL for (int i = 0; i < n * m; ++i) {
      sy = fma(tB[i] - dB[i], nB[i] - gB[i], sy);
      dB[i] = tB[i]; gB[i] = nB[i];
    }
    t = (sy < 0.0) ? ss / -sy : 10.0 * t;
  }
  *J_out = J;
  *rho_out = rho;
  *iters = it;
  return flags;
}

// ---- the same steps as shared functions, for the objectives of other headers (worst_inf.cuh). worst_eval and
// worst_ascent above keep their own inline copies: routing them through these functions changes the generated code
// of 21 of the 44 kernels of k_worst.cu (same operations, different register allocation and spills).

// worst_eval's forward recursion on (Ah, Bh) from P = P(0) (set by the caller): K0 = K(N), P left at P(N-1) and st
// holding the factor of G_N. With `grad` the pairs (P(k-1), K(k)), k = 1..N-1, go to ws. Returns CHOL_FAIL of any stage.
template <int n, int m>
LQ_HD int riccati_records(const Problem<n, m>& pb, const double* Ah, const double* Bh, int N, const WsView& ws,
                          bool grad, double* P, RicStage<n, m>& st, double* K0) {
  constexpr int ps = n * (n + 1) / 2, rs = ps + m * n;
  int flags = 0;
  for (int k = 1; k < N; ++k) {
    riccati_factor<n, m>(P, Bh, pb.R, st);
    if (!st.ok) flags |= FLAG_CHOL_FAIL;
    if (grad) {
      const int64_t o = (int64_t)(k - 1) * rs;
      int e = 0;
      LQ_UNROLL for (int i = 0; i < n; ++i)
        LQ_UNROLL for (int j = i; j < n; ++j) ws[o + e++] = P[i * n + j];
      riccati_gain<n, m>(st, Ah, K0);
      LQ_UNROLL for (int i = 0; i < m * n; ++i) ws[o + ps + i] = K0[i];
    }
    riccati_update<n, m>(st, Ah, pb.Q, P);
  }
  riccati_factor<n, m>(P, Bh, pb.R, st);        // horizon N: P = P(N-1), st holds G_N = L L'
  if (!st.ok) flags |= FLAG_CHOL_FAIL;
  riccati_gain<n, m>(st, Ah, K0);
  return flags;
}

// worst_eval's reverse sweep: from Kbar = dJ/dK0 (in Z, overwritten) to gA = dJ/d(dA), gB = dJ/d(dB) (written), with
// K0, P = P(N-1) and the factor st of riccati_records and its stage records in ws.
template <int n, int m>
LQ_HD void riccati_adjoint(const double* Ah, const double* Bh, const double* K0, const double* P,
                           const RicStage<n, m>& st, double* Z, int N, const WsView& ws, double* gA, double* gB) {
  constexpr int ps = n * (n + 1) / 2, rs = ps + m * n;
  solve_l_inv<m, n>(st.L, st.Li, Z);
  solve_lt_inv<m, n>(st.L, st.Li, Z);
  double F[n * n], PB[n * m], Pbar[n * n];
  LQ_UNROLL for (int i = 0; i < n; ++i)
    LQ_UNROLL for (int j = 0; j < n; ++j) {
      double acc = Ah[i * n + j];
      LQ_UNROLL for (int k = 0; k < m; ++k) acc = fma(Bh[i * m + k], K0[k * n + j], acc);
      F[i * n + j] = acc;
    }
  mm<n, n, m>(P, Bh, PB);
  {
    double T[n * n], ZK[m * m], U[n * m];
    mm<n, m, n>(PB, Z, T);
    LQ_UNROLL for (int i = 0; i < n * n; ++i) gA[i] = -T[i];
    mm<n, n, n>(P, F, T);                        // P F
    mmt<n, n, m>(T, Z, U);                       // P F Z'
    mmt<m, n, m>(Z, K0, ZK);                     // Z K0'
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = 0; j < m; ++j) {
        double acc = U[i * m + j];
        LQ_UNROLL for (int k = 0; k < m; ++k) acc = fma(PB[i * m + k], ZK[k * m + j], acc);
        gB[i * m + j] = -acc;
      }
    mmt<n, n, m>(F, Z, U);                       // U = F Z'
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = i; j < n; ++j) {
        double acc = 0.0;
        LQ_UNROLL for (int k = 0; k < m; ++k) acc = fma(U[i * m + k], Bh[j * m + k], fma(Bh[i * m + k], U[j * m + k], acc));
        Pbar[i * n + j] = Pbar[j * n + i] = -0.5 * acc;
      }
  }
  for (int k = N - 1; k >= 1; --k) {
    const int64_t o = (int64_t)(k - 1) * rs;
    double Pk[n * n], Kk[m * n], Fk[n * n], T[n * n], X[n * n];
    int e = 0;
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = i; j < n; ++j) { const double v = ws[o + e++]; Pk[i * n + j] = v; Pk[j * n + i] = v; }
    LQ_UNROLL for (int i = 0; i < m * n; ++i) Kk[i] = ws[o + ps + i];
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = 0; j < n; ++j) {
        double acc = Ah[i * n + j];
        LQ_UNROLL for (int l = 0; l < m; ++l) acc = fma(Bh[i * m + l], Kk[l * n + j], acc);
        Fk[i * n + j] = acc;
      }
    mm<n, n, n>(Pk, Fk, T);
    mm<n, n, n>(T, Pbar, X);
    LQ_UNROLL for (int i = 0; i < n * n; ++i) gA[i] = fma(2.0, X[i], gA[i]);
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = 0; j < m; ++j) {
        double acc = 0.0;
        LQ_UNROLL for (int l = 0; l < n; ++l) acc = fma(X[i * n + l], Kk[j * n + l], acc);
        gB[i * m + j] = fma(2.0, acc, gB[i * m + j]);
      }
    mm<n, n, n>(Fk, Pbar, T);
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = i; j < n; ++j) {
        double acc = 0.0;
        LQ_UNROLL for (int l = 0; l < n; ++l) acc = fma(T[i * n + l], Fk[j * n + l], acc);
        Pbar[i * n + j] = Pbar[j * n + i] = acc;
      }
  }
}

// worst_ascent for any objective: the projected ascent over the error set from (dA, dB), both overwritten with the
// result, in the normalised coordinates u = (dA / e_A, dB / e_B) with gradient g^ = (e_A dJ/d(dA), e_B dJ/d(dB)):
//   * project the start; at every accepted point the stationarity residual is r = ||Proj(u + g^/||g^||) - u||_2
//     (0 when g^ = 0) and the ascent stops when r <= tol;
//   * trial u+ = Proj(u + t g^), the first t = 0.5 / ||g^||, then Barzilai-Borwein t = s's / (-s'y) when s'y < 0 and
//     10 t otherwise; accepted when J(u+) >= J(u) + 1e-4 g^.(u+ - u), else t <- t / 4;
//   * trials take the value only, the gradient is computed at accepted points;
//   * an unstable trial lies in the set and destabilises the loop: it is the result (J = +inf, UNSTABLE);
//   * a trial with a flag of kFail is rejected; a start with one ends the ascent there;
//   * the budget of max_iter accepted steps (or a line search that shrinks t by 4^60) ends it with ASCENT_MAXITER.
// The objective is `eval(dA, dB, &J, &rho, gA, gB)` -> flags, a trial when gA is null; `keep_trial()` is called when
// an unstable trial becomes the result, so that the objective can keep that trial's other outputs. Returns the flags of
// the final point; J, rho and the accepted-step count go to the outputs.
template <int n, int m, int kFail, class Eval, class KeepTrial>
LQ_HD int ascent_run(double* dA, double* dB, const AscentSettings& as, Eval eval, KeepTrial keep_trial,
                     double* J_out, double* rho_out, int* iters) {
  const double eA2 = as.eA * as.eA, eB2 = as.eB * as.eB;
  worst_project<n, n>(dA, as.eA, as.norm);
  worst_project<n, m>(dB, as.eB, as.norm);
  double gA[n * n], gB[n * m], J, rho;
  int flags = eval(dA, dB, &J, &rho, gA, gB);
  int it = 0;
  double t = 0.0;
  while (!(flags & (kFail | FLAG_UNSTABLE))) {
    const double gn2 = eA2 * fro2<n * n>(gA) + eB2 * fro2<n * m>(gB);
    if (!(gn2 > 0.0)) break;                              // g^ = 0: r = 0
    const double gn = sqrt(gn2);
    double tA[n * n], tB[n * m];
    const double r2 = worst_step<n, n>(dA, gA, eA2 / gn, as.eA, as.norm, tA) +
                      worst_step<n, m>(dB, gB, eB2 / gn, as.eB, as.norm, tB);
    if (sqrt(r2) <= as.tol) break;
    if (it >= as.max_iter) { flags |= FLAG_ASCENT_MAXITER; break; }
    if (it == 0) t = 0.5 / gn;
    double Jt = 0.0, rt = 0.0, ss = 0.0;
    int ft = 0;
    bool accepted = false;
    for (int bt = 0; bt < kWorstMaxBacktrack; ++bt) {
      ss = worst_step<n, n>(dA, gA, t * eA2, as.eA, as.norm, tA) + worst_step<n, m>(dB, gB, t * eB2, as.eB, as.norm, tB);
      double dot = 0.0;
      LQ_UNROLL for (int i = 0; i < n * n; ++i) dot = fma(gA[i], tA[i] - dA[i], dot);
      LQ_UNROLL for (int i = 0; i < n * m; ++i) dot = fma(gB[i], tB[i] - dB[i], dot);
      ft = eval(tA, tB, &Jt, &rt, nullptr, nullptr);
      if ((ft & FLAG_UNSTABLE) || (!(ft & kFail) && Jt >= J + 1e-4 * dmax(dot, 0.0))) { accepted = true; break; }
      t *= 0.25;
    }
    if (!accepted) { flags |= FLAG_ASCENT_MAXITER; break; }
    ++it;
    if (ft & FLAG_UNSTABLE) {
      LQ_UNROLL for (int i = 0; i < n * n; ++i) dA[i] = tA[i];
      LQ_UNROLL for (int i = 0; i < n * m; ++i) dB[i] = tB[i];
      keep_trial();
      J = Jt; rho = rt; flags = ft;
      break;
    }
    // the gradient at the accepted point (its value repeats the trial's bit for bit). With s = u+ - u and
    // y = g^+ - g^, s'y = (dA+ - dA).(gA+ - gA) + (dB+ - dB).(gB+ - gB): the scales e cancel.
    double nA[n * n], nB[n * m], sy = 0.0;
    flags = eval(tA, tB, &J, &rho, nA, nB);
    LQ_UNROLL for (int i = 0; i < n * n; ++i) {
      sy = fma(tA[i] - dA[i], nA[i] - gA[i], sy);
      dA[i] = tA[i]; gA[i] = nA[i];
    }
    LQ_UNROLL for (int i = 0; i < n * m; ++i) {
      sy = fma(tB[i] - dB[i], nB[i] - gB[i], sy);
      dB[i] = tB[i]; gB[i] = nB[i];
    }
    t = (sy < 0.0) ? ss / -sy : 10.0 * t;
  }
  *J_out = J;
  *rho_out = rho;
  *iters = it;
  return flags;
}

}  // namespace lq
