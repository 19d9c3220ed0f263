// riccati.cuh — per-sample certainty-equivalent LQ-MPC evaluation (unconstrained law), one sample per thread.
//
// Reference semantics restated (citations into /root/reference):
//   * MPC gain of horizon N on the ESTIMATED model (A^,B^) = (A+dA, B+dB): the minimiser of the cost built in
//     LQ_MPC_Controller.solve (utils_class.py:59-75, zero references, terminal weight P) is u_0 = K_0 x with K_0
//     from the finite-horizon Riccati recursion started at P (when no input bound is active).
//   * closed loop on the TRUE plant (utils_class.py:277): x+ = (A + B K_0) x, cost accumulated as in
//     utils_class.py:261,282-283; its T -> infinity limit is x0' S x0 with S the solution of the discrete Lyapunov
//     equation S = W + Acl' S Acl, W = Q + K0' R K0. For n = 3, 4 the scalar x0' S x0 comes from the characteristic
//     polynomial of Acl (lyapunov_cost_poly), elsewhere and where that is not accepted S is obtained by squared doubling.
//   * stability check: spectral radius of the closed loop (utils.py:358 style eigvals + max|.|).
//   * performance ratio: J / V_expert(x0), V_expert = x0' Pexp x0 the expert (true-model) optimal cost
//     (utils_class.py:786) — Pexp is prepared once per problem on the device (prep kernel).
// Horizons N_min..N_max share ONE recursion: the Riccati iterates are nested in N.
#pragma once
#include "eig.cuh"
#include "small_la.cuh"

namespace lq {

enum Flags : int {
  FLAG_UNSTABLE = 1,       // rho(A_cl) >= 1  -> J_inf = +inf
  FLAG_QP_ACTIVE = 2,      // some planned input hit its bound (exact active-set solve was needed)
  FLAG_QP_MAXITER = 4,     // active-set iteration budget exhausted
  FLAG_DARE_NOCONV = 8,    // doubling iteration for the DARE did not converge
  FLAG_NONFINITE = 16,     // NaN/Inf produced
  FLAG_BOUND_INVALID = 32, // 1 - xi - eta <= 0: the performance bound is void (the reference still computes it)
  FLAG_LYAP_NOCONV = 64,   // Lyapunov doubling hit its iteration cap
  FLAG_EIG_NOCONV = 128,   // QR iteration did not converge
  FLAG_CHOL_FAIL = 256,    // R + B'PB not positive definite
  FLAG_DOMAIN_ERROR = 512  // math.log / math.sqrt domain error (the reference raises ValueError, utils.py:506-507,514)
};

template <int n, int m>
struct Problem {
  double A[n * n];     // true plant
  double B[n * m];
  double Q[n * n];
  double R[m * m];
  double Pt[n * n];    // terminal weight (every reference caller passes P = Q)
  double Pexp[n * n];  // expert cost matrix: V_expert(x0) = x0' Pexp x0
  double Qinv[n * n];
  double ulo[m], uhi[m];
  double maxQ, minQ, maxR, minR;
  int has_bounds;
  int qr_scalar;       // Q = q I and R = r I (then the literal kron ordering of utils.py:317-318 is immaterial)
};

// One Riccati "half step" from the current cost-to-go P (of horizon k-1):
//   PB = P B^, G = R + B^' PB = L L', Y = PB L^-T.  Then
//   gain of horizon k:  K = -L^-T (Y' A^)
//   next cost-to-go:    P+ = Q + A^' (P - Y Y') A^
template <int n, int m>
struct RicStage {
  double Y[n * m];
  double L[m * m];
  double Li[m];        // reciprocals of L's diagonal
  bool ok;
};

template <int n, int m>
LQ_HD void riccati_factor(const double* P, const double* Bh, const double* R, RicStage<n, m>& st) {
  mm<n, n, m>(P, Bh, st.Y);                       // PB
  LQ_UNROLL for (int i = 0; i < m; ++i)           // G = R + B^' PB  (lower triangle is all chol needs)
    LQ_UNROLL for (int j = 0; j <= i; ++j) {
      double acc = R[i * m + j];
      LQ_UNROLL for (int k = 0; k < n; ++k) acc = fma(Bh[k * m + i], st.Y[k * m + j], acc);
      st.L[i * m + j] = acc;
      st.L[j * m + i] = acc;
    }
  st.ok = chol_inv<m>(st.L, st.Li);
  solve_right_lt_inv<n, m>(st.L, st.Li, st.Y);    // Y = PB L^-T
}

template <int n, int m>
LQ_HD void riccati_gain(const RicStage<n, m>& st, const double* Ah, double* K) {
  mtm<n, m, n>(st.Y, Ah, K);                      // Y' A^   (m x n)
  solve_lt_inv<m, n>(st.L, st.Li, K);             // L^-T (.)
  LQ_UNROLL for (int i = 0; i < m * n; ++i) K[i] = -K[i];
}

template <int n, int m>
LQ_HD void riccati_update(const RicStage<n, m>& st, const double* Ah, const double* Q, double* P) {
  double Mx[n * n], MA[n * n];
  sym_sub_yyt<n, m>(P, st.Y, Mx);                 // M = P - Y Y'
  mm<n, n, n>(Mx, Ah, MA);
  sym_add_mtm<n, n>(Q, Ah, MA, P);                // P+ = Q + A^' M A^
}

// Infinite-horizon cost matrix of x+ = Acl x with stage weight W by squared doubling:
//   S_{j+1} = S_j + M_j' S_j M_j,  M_{j+1} = M_j^2,  S_0 = W, M_0 = Acl.
template <int n>
LQ_HD bool lyapunov_doubling(const double* Acl, const double* W, double* S) {
  double M[n * n], SM[n * n], T[n * n];
  LQ_UNROLL for (int i = 0; i < n * n; ++i) { S[i] = W[i]; M[i] = Acl[i]; }
  const double zero[1] = {0.0};
  (void)zero;
  for (int it = 0; it < 64; ++it) {
    mm<n, n, n>(S, M, SM);
    uint32_t thi = 0, shi = 0;                         // max |increment|, max |S| as exponent words (abs_hi)
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = i; j < n; ++j) {
        double acc = 0.0;
        LQ_UNROLL for (int k = 0; k < n; ++k) acc = fma(M[k * n + i], SM[k * n + j], acc);
        T[i * n + j] = acc;
        thi = umax32(thi, abs_hi(acc));
      }
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = i; j < n; ++j) {
        const double v = S[i * n + j] + T[i * n + j];
        S[i * n + j] = v; S[j * n + i] = v;
        shi = umax32(shi, abs_hi(v));
      }
    if ((thi >> 20) == 0x7ffu || (shi >> 20) == 0x7ffu) return false;             // NaN / Inf
    if (!(from_abs_hi(thi) > 1e-18 * from_abs_hi(shi))) return true;              // converged
    mm<n, n, n>(M, M, SM);
    uint32_t mhi = 0;
    LQ_UNROLL for (int i = 0; i < n * n; ++i) { M[i] = SM[i]; mhi = umax32(mhi, abs_hi(SM[i])); }
    // the next increment is bounded entrywise by n^2 max|M|^2 max|S| (S is PSD and non-decreasing, its largest entry
    // sits on the diagonal): once that is below the threshold the iteration that would only confirm it is skipped
    const double mb = from_abs_hi(mhi) * 1.000002;                       // abs_hi truncates the mantissa by < 2^-20
    if ((double)(n * n) * mb * mb <= 1e-18) return true;
  }
  return false;
}

// Smallest elimination pivot lyapunov_cost_poly accepts. Small pivots come with clustered or strongly non-normal
// spectra and with rho near 1; calibrated on the host against a 50-digit Stein solve: with 1e-3 the worst accepted
// relative error over those families is ~2.5e-12, without a threshold 1.2e-10 (tests/test_k1_closed_loop_cost.py).
constexpr double kLyapPolyMinPivot = 1e-3;

// J = x0' S x0 with S = W + Acl' S Acl (rho(Acl) < 1) from the characteristic polynomial of Acl, n = 3, 4, without S.
// With x_k = Acl^k x0, c_ij = x_i' W x_j and gamma_d = sum_{k>=0} x_k' W x_{k+d} (J = gamma_0), Cayley-Hamilton gives
// x_{k+n} = -sum_{r=1..n} a_r x_{k+n-r} (a_0 = 1); its inner product with x_{k+j} summed over k, j = 0..n, is
//   sum_r a_r gamma_{|n-r-j|} = sum_r a_r sum_{i < min(j, n-r)} c_{i, i+|n-r-j|},
// n + 1 equations in gamma_0..gamma_n that need only x_0..x_{n-1}. Taken in the order j = n..0 their first pivot is
// a_0 = 1 and elimination needs no row swaps (in the order j = 0..n it would be det(Acl)). The result is accepted only
// if every pivot exceeds kLyapPolyMinPivot in magnitude, J is finite and J >= c_00 + ... + c_{n-1,n-1}, the partial
// sum S >= sum_{k<n} (Acl')^k W Acl^k guarantees; otherwise the caller runs lyapunov_doubling.
template <int n>
LQ_HD bool lyapunov_cost_poly(const CharPoly& cp, const double* Acl, const double* W, const double* x0, double* J) {
  static_assert(n == 3 || n == 4, "characteristic-polynomial route is for n = 3, 4");
  constexpr int n1 = n + 1;
  const double f2 = cp.fro * cp.fro;
  double al[n1];                                        // coefficients of the polynomial of Acl itself (unscaled)
  al[0] = 1.0;
  al[1] = cp.a * cp.fro;
  al[2] = cp.b * f2;
  al[3] = cp.c * (f2 * cp.fro);
  if constexpr (n == 4) al[n] = cp.d * (f2 * f2);
  double x[n * n], wx[n * n];                           // x[k*n + i] = (Acl^k x0)_i, wx[k*n + i] = (W x_k)_i
  LQ_UNROLL for (int i = 0; i < n; ++i) x[i] = x0[i];
  LQ_UNROLL for (int k = 1; k < n; ++k) mv<n, n>(Acl, x + (k - 1) * n, x + k * n);
  LQ_UNROLL for (int k = 0; k < n; ++k) mv<n, n>(W, x + k * n, wx + k * n);
  double c[n * n];                                      // c[i*n + j] = x_i' W x_j, i <= j
  LQ_UNROLL for (int i = 0; i < n; ++i)
    LQ_UNROLL for (int j = i; j < n; ++j) {
      double acc = x[i * n] * wx[j * n];
      LQ_UNROLL for (int e = 1; e < n; ++e) acc = fma(x[i * n + e], wx[j * n + e], acc);
      c[i * n + j] = acc;
    }
  // row t is the equation j = n - t; columns are gamma_0..gamma_n. -0.0 is the additive identity the compiler folds.
  double G[n1 * n1], h[n1];
  LQ_UNROLL for (int t = 0; t < n1; ++t) {
    const int j = n - t;
    LQ_UNROLL for (int d = 0; d < n1; ++d) G[t * n1 + d] = -0.0;
    h[t] = -0.0;
    LQ_UNROLL for (int r = 0; r < n1; ++r) {
      const int d = (n - r - j) < 0 ? (j + r - n) : (n - r - j);
      G[t * n1 + d] += al[r];
      const int lim = j < n - r ? j : n - r;
      if (lim > 0) {
        double s = c[d];
        LQ_UNROLL for (int i = 1; i < lim; ++i) s += c[i * n + i + d];
        h[t] = fma(al[r], s, h[t]);
      }
    }
  }
  double ip[n1];
  bool piv_ok = true;
  LQ_UNROLL for (int k = 0; k < n1; ++k) {
    const double p = G[k * n1 + k];
    piv_ok = piv_ok && (fabs(p) > kLyapPolyMinPivot);
    ip[k] = rcp(p);
    LQ_UNROLL for (int i = k + 1; i < n1; ++i) {
      const double f = G[i * n1 + k] * ip[k];
      LQ_UNROLL for (int col = k + 1; col < n1; ++col) G[i * n1 + col] = fma(-f, G[k * n1 + col], G[i * n1 + col]);
      h[i] = fma(-f, h[k], h[i]);
    }
  }
  double g[n1];
  LQ_UNROLL for (int k = n1 - 1; k >= 0; --k) {
    double s = h[k];
    LQ_UNROLL for (int col = k + 1; col < n1; ++col) s = fma(-G[k * n1 + col], g[col], s);
    g[k] = s * ip[k];
  }
  double psum = c[0];
  LQ_UNROLL for (int i = 1; i < n; ++i) psum += c[i * n + i];
  *J = g[0];
  return piv_ok && fabs(g[0]) <= 1.79e308 && g[0] >= psum;
}

// Closed-loop figures for one gain K on the true plant. kLyapPoly (n = 3, 4): J from lyapunov_cost_poly where it is
// accepted; false runs the doubling for every sample (the earlier path, kept as an A/B reference).
template <int n, int m, bool kLyapPoly = true>
LQ_HD void closed_loop_eval(const Problem<n, m>& pb, const double* K, const double* x0, int T,
                            double* J_inf, double* rho_out, double* J_T, int* flags) {
  double Acl[n * n], W[n * n], RK[m * n];
  LQ_UNROLL for (int i = 0; i < n; ++i)
    LQ_UNROLL for (int j = 0; j < n; ++j) {
      double acc = pb.A[i * n + j];
      LQ_UNROLL for (int k = 0; k < m; ++k) acc = fma(pb.B[i * m + k], K[k * n + j], acc);
      Acl[i * n + j] = acc;
    }
  mm<m, m, n>(pb.R, K, RK);
  sym_add_mtm<m, n>(pb.Q, K, RK, W);
  bool ok, cp_ok;
  CharPoly cp;
  const double rho = spectral_radius<n>(Acl, &ok, &cp, &cp_ok);
  if (!ok) *flags |= FLAG_EIG_NOCONV;
  *rho_out = rho;
  if (!(rho < 1.0)) {
    *flags |= FLAG_UNSTABLE;
    *J_inf = HUGE_VAL;
  } else {
    double J;
    bool fast = false;
    if constexpr (kLyapPoly && (n == 3 || n == 4)) fast = cp_ok && lyapunov_cost_poly<n>(cp, Acl, W, x0, &J);
    if (!fast) {
      double S[n * n];
      if (!lyapunov_doubling<n>(Acl, W, S)) *flags |= FLAG_LYAP_NOCONV;
      J = quad<n>(x0, S, x0);
      if (!(fabs(J) <= 1.79e308)) *flags |= FLAG_NONFINITE;
    }
    *J_inf = J;
  }
  if (T > 0) {  // finite-T cost exactly as accumulated by utils_class.py:261,282-283
    double x[n], xn[n], u[m];
    LQ_UNROLL for (int i = 0; i < n; ++i) x[i] = x0[i];
    double cost = quad<n>(x, pb.Q, x);
    for (int t = 0; t < T; ++t) {
      mv<m, n>(K, x, u);
      LQ_UNROLL for (int i = 0; i < n; ++i) {
        double acc = 0.0;
        LQ_UNROLL for (int j = 0; j < n; ++j) acc = fma(pb.A[i * n + j], x[j], acc);
        LQ_UNROLL for (int j = 0; j < m; ++j) acc = fma(pb.B[i * m + j], u[j], acc);
        xn[i] = acc;
      }
      cost += quad<n>(xn, pb.Q, xn);
      cost += quad<m>(u, pb.R, u);
      LQ_UNROLL for (int i = 0; i < n; ++i) x[i] = xn[i];
    }
    *J_T = cost;
  }
}

// Full per-sample evaluation over the nested horizons N_min..N_max. `sink(h, ...)` receives column h = N - N_min.
template <int n, int m, class Sink, bool kLyapPoly = true>
LQ_HD void eval_sample(const Problem<n, m>& pb, const double* dA, const double* dB, const double* x0,
                       int N_min, int N_max, int T, bool want_vn, Sink& sink) {
  double Ah[n * n], Bh[n * m], P[n * n];
  LQ_UNROLL for (int i = 0; i < n * n; ++i) { Ah[i] = pb.A[i] + dA[i]; P[i] = pb.Pt[i]; }
  LQ_UNROLL for (int i = 0; i < n * m; ++i) Bh[i] = pb.B[i] + dB[i];
  const double v_exp = quad<n>(x0, pb.Pexp, x0);
  RicStage<n, m> st;
  int sticky = 0;
  for (int k = 1; k <= N_max; ++k) {
    riccati_factor<n, m>(P, Bh, pb.R, st);
    if (!st.ok) sticky |= FLAG_CHOL_FAIL;
    const bool emit = (k >= N_min);
    double K[m * n];
    if (emit) riccati_gain<n, m>(st, Ah, K);
    if (k < N_max || want_vn) riccati_update<n, m>(st, Ah, pb.Q, P);   // P is now the horizon-k cost-to-go
    if (emit) {
      int flags = sticky;
      double J, rho, JT = 0.0;
      closed_loop_eval<n, m, kLyapPoly>(pb, K, x0, T, &J, &rho, &JT, &flags);
      const double vn = want_vn ? quad<n>(x0, P, x0) : 0.0;
      sink(k - N_min, J, rho, J / v_exp, vn, JT, flags, K);
    }
  }
}

// Problem preparation (device, one thread): Qinv, extremal eigenvalues of Q and R, the scalar-weights flag and the
// expert cost matrix Pexp = N_opc-step Riccati cost-to-go of the TRUE model (utils_class.py:757,786), or the DARE
// limit when N_opc <= 0 (iterated to a fixed point).
template <int n, int m>
LQ_HD void prepare_problem(Problem<n, m>& pb, int N_opc) {
  inverse<n>(pb.Q, pb.Qinv);
  sym_eig_minmax<n>(pb.Q, &pb.minQ, &pb.maxQ);
  sym_eig_minmax<m>(pb.R, &pb.minR, &pb.maxR);
  bool scal = true;
  LQ_UNROLL for (int i = 0; i < n; ++i)
    LQ_UNROLL for (int j = 0; j < n; ++j)
      scal = scal && (pb.Q[i * n + j] == ((i == j) ? pb.Q[0] : 0.0));
  LQ_UNROLL for (int i = 0; i < m; ++i)
    LQ_UNROLL for (int j = 0; j < m; ++j)
      scal = scal && (pb.R[i * m + j] == ((i == j) ? pb.R[0] : 0.0));
  pb.qr_scalar = scal ? 1 : 0;
  double P[n * n];
  LQ_UNROLL for (int i = 0; i < n * n; ++i) P[i] = pb.Pt[i];
  RicStage<n, m> st;
  const int iters = (N_opc > 0) ? N_opc : 100000;
  for (int k = 0; k < iters; ++k) {
    double Pold[n * n];
    LQ_UNROLL for (int i = 0; i < n * n; ++i) Pold[i] = P[i];
    riccati_factor<n, m>(P, pb.B, pb.R, st);
    riccati_update<n, m>(st, pb.A, pb.Q, P);
    if (N_opc <= 0) {
      double d = 0.0;
      LQ_UNROLL for (int i = 0; i < n * n; ++i) d = dmax(d, fabs(P[i] - Pold[i]));
      if (d <= 1e-16 * max_abs<n * n>(P)) break;
    }
  }
  LQ_UNROLL for (int i = 0; i < n * n; ++i) pb.Pexp[i] = P[i];
}

}  // namespace lq
