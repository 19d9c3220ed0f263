// pclqr.cuh — exact solution of the finite-horizon LQ problem with a GENERAL input polytope, one sample per thread.
//
// Reference semantics: LQ_MPC_Controller.solve (utils_class.py:48-91) constrains every planned input by
// `F_u @ u_i <= 1` (utils_class.py:81) for an arbitrary F_u (p x m). clqr.cuh covers the case every caller in the
// reference uses (one non-zero per row: a box); this header covers the rest of the interface (SURVEY 8f.3).
//
// Method: the same primal active-set iteration as clqr.cuh, with the working set a set of (stage, row) pairs. The
// equality-constrained sub-problem is again ONE affine Riccati sweep: at stage k the unconstrained minimiser of
// u'Gu + 2u'h is projected onto {F_W u = 1} in the G-metric,
//     u = u_unc - G^-1 F_W' (F_W G^-1 F_W')^-1 (F_W u_unc - 1),
// which keeps the law affine in x (gain and offset), so the cost-to-go recursion is unchanged. Rows join the working
// set by the ratio test along z* - z (a blocking row is never a combination of the rows already active at its stage:
// those have F_W dz = 0), rows leave by the sign of their KKT multiplier, recovered stage by stage from the costate
// sweep as mu = -(F_W F_W')^-1 F_W dJ/du_k. Working sets are 256-bit masks: N * p <= 256.
#pragma once
#include "clqr.cuh"

namespace lq {

constexpr int kPolyMaxRows = 12;

// rows of F_u, row-major p x m (a pointer every thread reads uniformly: device global memory / host memory)
struct Poly {
  const double* F = nullptr;
  int p = 0;
  LQ_HD double f(int i, int j, int m) const { return F[i * m + j]; }
};

// F_i u for row i
template <int m>
LQ_HD double poly_row(const Poly& py, int i, const double* u) {
  double acc = 0.0;
  LQ_UNROLL for (int j = 0; j < m; ++j) acc = fma(py.f(i, j, m), u[j], acc);
  return acc;
}

// Rows of stage k in the working set, gathered into FW (m x m, zero rows beyond the count). Returns the count (<= m).
template <int m>
LQ_HD int poly_gather(const Poly& py, const Mask128& W, int k, double* FW) {
  LQ_UNROLL for (int e = 0; e < m * m; ++e) FW[e] = 0.0;
  int c = 0;
  for (int i = 0; i < py.p; ++i) {
    if (c < m && W.test(k * py.p + i)) {
      LQ_UNROLL for (int r = 0; r < m; ++r)
        if (r == c) { LQ_UNROLL for (int j = 0; j < m; ++j) FW[r * m + j] = py.f(i, j, m); }
      ++c;
    }
  }
  return c;
}

// Backward affine Riccati sweep for the working set W: stores K_k (m x n) and k_k (m), u_k = K_k x_k + k_k.
template <int n, int m>
LQ_HD bool pclqr_backward(const Problem<n, m>& pb, const Plan<n, m>& pl, int N, const Mask128& W, const Poly& py,
                          const WsView& ws, const Refs& rf) {
  const ClqrLayout<n, m> L(N);
  double S[n * n], s[n];
  LQ_UNROLL for (int i = 0; i < n * n; ++i) S[i] = pb.Pt[i];
  LQ_UNROLL for (int i = 0; i < n; ++i) {
    double acc = 0.0;
    LQ_UNROLL for (int j = 0; j < n; ++j) acc = fma(-pb.Pt[i * n + j], rf.x(j, N - 1), acc);
    s[i] = acc;
  }
  bool ok = true;
  for (int k = N - 1; k >= 0; --k) {
    double SB[n * m], G[m * m], Hx[m * (n + 1)];
    mm<n, n, m>(S, pl.Bh, SB);
    LQ_UNROLL for (int i = 0; i < m; ++i)
      LQ_UNROLL for (int j = 0; j <= i; ++j) {
        double acc = pb.R[i * m + j];
        LQ_UNROLL for (int r = 0; r < n; ++r) acc = fma(pl.Bh[r * m + i], SB[r * m + j], acc);
        G[i * m + j] = acc; G[j * m + i] = acc;
      }
    LQ_UNROLL for (int i = 0; i < m; ++i) {
      LQ_UNROLL for (int j = 0; j < n; ++j) {
        double acc = 0.0;
        LQ_UNROLL for (int r = 0; r < n; ++r) acc = fma(SB[r * m + i], pl.Ah[r * n + j], acc);
        Hx[i * (n + 1) + j] = acc;
      }
      double acc = 0.0;
      LQ_UNROLL for (int r = 0; r < n; ++r) acc = fma(pl.Bh[r * m + i], s[r], acc);
      LQ_UNROLL for (int r = 0; r < m; ++r) acc = fma(-pb.R[i * m + r], rf.u(r, k), acc);
      Hx[i * (n + 1) + n] = acc;
    }
    // unconstrained stage law u = -Hx [x; 1]
    ok = chol<m>(G) && ok;
    solve_l<m, n + 1>(G, Hx);
    solve_lt<m, n + 1>(G, Hx);
    double FW[m * m];
    const int c = poly_gather<m>(py, W, k, FW);
    if (c > 0) {
      double Y[m * m], M[m * m], Lam[m * (n + 1)];
      LQ_UNROLL for (int j = 0; j < m; ++j)
        LQ_UNROLL for (int r = 0; r < m; ++r) Y[j * m + r] = FW[r * m + j];
      solve_l<m, m>(G, Y);
      solve_lt<m, m>(G, Y);                                   // Y = G^-1 F_W'   (columns >= c are zero)
      LQ_UNROLL for (int i = 0; i < m; ++i)
        LQ_UNROLL for (int r = 0; r < m; ++r) {
          double acc = 0.0;
          LQ_UNROLL for (int j = 0; j < m; ++j) acc = fma(FW[i * m + j], Y[j * m + r], acc);
          M[i * m + r] = acc;
        }
      LQ_UNROLL for (int i = 0; i < m; ++i)
        if (i >= c) M[i * m + i] = 1.0;                       // identity padding keeps the factorisation size static
      ok = chol<m>(M) && ok;
      LQ_UNROLL for (int i = 0; i < m; ++i)
        LQ_UNROLL for (int col = 0; col <= n; ++col) {
          double acc = 0.0;
          LQ_UNROLL for (int j = 0; j < m; ++j) acc = fma(FW[i * m + j], Hx[j * (n + 1) + col], acc);
          Lam[i * (n + 1) + col] = -acc;
        }
      LQ_UNROLL for (int i = 0; i < m; ++i)
        if (i < c) Lam[i * (n + 1) + n] -= 1.0;               // F_W u_unc - 1
      solve_l<m, n + 1>(M, Lam);
      solve_lt<m, n + 1>(M, Lam);
      LQ_UNROLL for (int j = 0; j < m; ++j)
        LQ_UNROLL for (int col = 0; col <= n; ++col) {
          double acc = Hx[j * (n + 1) + col];
          LQ_UNROLL for (int r = 0; r < m; ++r) acc = fma(Y[j * m + r], Lam[r * (n + 1) + col], acc);
          Hx[j * (n + 1) + col] = acc;
        }
    }
    double K[m * n], kv[m];
    LQ_UNROLL for (int i = 0; i < m; ++i) {
      LQ_UNROLL for (int j = 0; j < n; ++j) K[i * n + j] = -Hx[i * (n + 1) + j];
      kv[i] = -Hx[i * (n + 1) + n];
    }
    LQ_UNROLL for (int e = 0; e < m * n; ++e) ws[L.oKc + (int64_t)k * (m * n) + e] = K[e];
    LQ_UNROLL for (int e = 0; e < m; ++e) ws[L.okc + (int64_t)k * m + e] = kv[e];
    if (k > 0) {
      // S_k = Q + K'RK + Acl' S Acl ;  s_k = -Q r_{k-1} + K'R (kv - u_ref_k) + Acl'(S B kv + s)
      double Acl[n * n], SA[n * n], RK[m * n], bk[n], t[n], Rk[m];
      LQ_UNROLL for (int i = 0; i < n; ++i)
        LQ_UNROLL for (int j = 0; j < n; ++j) {
          double acc = pl.Ah[i * n + j];
          LQ_UNROLL for (int r = 0; r < m; ++r) acc = fma(pl.Bh[i * m + r], K[r * n + j], acc);
          Acl[i * n + j] = acc;
        }
      mv<n, m>(pl.Bh, kv, bk);
      LQ_UNROLL for (int i = 0; i < n; ++i) {
        double acc = s[i];
        LQ_UNROLL for (int j = 0; j < n; ++j) acc = fma(S[i * n + j], bk[j], acc);
        t[i] = acc;
      }
      mm<m, m, n>(pb.R, K, RK);
      double kw[m];
      LQ_UNROLL for (int j = 0; j < m; ++j) kw[j] = kv[j] - rf.u(j, k);
      mv<m, m>(pb.R, kw, Rk);
      LQ_UNROLL for (int i = 0; i < n; ++i) {
        double acc = 0.0;
        LQ_UNROLL for (int r = 0; r < n; ++r) acc = fma(-pb.Q[i * n + r], rf.x(r, k - 1), acc);
        LQ_UNROLL for (int r = 0; r < m; ++r) acc = fma(K[r * n + i], Rk[r], acc);
        LQ_UNROLL for (int r = 0; r < n; ++r) acc = fma(Acl[r * n + i], t[r], acc);
        s[i] = acc;
      }
      mm<n, n, n>(S, Acl, SA);
      double Sn[n * n];
      sym_add_mtm<m, n>(pb.Q, K, RK, Sn);
      sym_add_mtm<n, n>(Sn, Acl, SA, S);
    }
  }
  return ok;
}

// Exact constrained solve from state x0. Returns flags; writes u0[m] and V (= optimum + x0'Qx0).
template <int n, int m>
LQ_HD int pclqr_solve(const Problem<n, m>& pb, const Plan<n, m>& pl, int N, const double* x0, const Poly& py,
                      const WsView& ws, double* u0, double* V, const Refs& rf = Refs()) {
  const ClqrLayout<n, m> L(N);
  const int p = py.p;
  double x[n], xn[n], u[m];
  const bool trk = rf.any();
  int flags = 0;
  Mask128 W;
  // ---- 1. unconstrained plan; feasible => optimal
  if (trk && !pclqr_backward<n, m>(pb, pl, N, W, py, ws, rf)) flags |= FLAG_CHOL_FAIL;
  const int64_t oK = trk ? L.oKc : L.oKu;
  bool feas = true;
  LQ_UNROLL for (int i = 0; i < n; ++i) x[i] = x0[i];
  double cost_u = quad<n>(x0, pb.Q, x0);
  for (int k = 0; k < N; ++k) {
    double K[m * n];
    LQ_UNROLL for (int e = 0; e < m * n; ++e) K[e] = ws[oK + (int64_t)k * (m * n) + e];
    mv<m, n>(K, x, u);
    LQ_UNROLL for (int j = 0; j < m; ++j) {
      if (trk) u[j] += ws[L.okc + (int64_t)k * m + j];
      if (k == 0) u0[j] = u[j];
    }
    for (int i = 0; i < p; ++i)
      if (poly_row<m>(py, i, u) > 1.0) feas = false;
    if (!feas) break;
    step_model<n, m>(pl.Ah, pl.Bh, x, u, xn);
    if (trk) {
      double du[m], dx[n];
      LQ_UNROLL for (int j = 0; j < m; ++j) du[j] = u[j] - rf.u(j, k);
      LQ_UNROLL for (int i = 0; i < n; ++i) dx[i] = xn[i] - rf.x(i, k);
      cost_u += quad<m>(du, pb.R, du);
      cost_u += (k == N - 1) ? quad<n>(dx, pb.Pt, dx) : quad<n>(dx, pb.Q, dx);
    }
    LQ_UNROLL for (int i = 0; i < n; ++i) x[i] = xn[i];
  }
  if (feas) {
    *V = trk ? cost_u : quad<n>(x0, pl.P0, x0);
    return flags;
  }
  flags |= FLAG_QP_ACTIVE;
  if (N * p > kMaskBits || p > kPolyMaxRows) {   // beyond the working-set mask: V = NaN, u0 shrunk onto the polytope, flagged
    double worst = 1.0;
    for (int i = 0; i < p; ++i) worst = dmax(worst, poly_row<m>(py, i, u0));
    LQ_UNROLL for (int j = 0; j < m; ++j) u0[j] /= worst;
    *V = NAN;
    return flags | FLAG_QP_MAXITER;
  }
  // ---- 2. feasible start: roll the unconstrained law out, shrinking each infeasible input radially onto the polytope
  //         (the origin is interior: F_u 0 = 0 < 1); the row that stops it enters the working set
  LQ_UNROLL for (int i = 0; i < n; ++i) x[i] = x0[i];
  for (int k = 0; k < N; ++k) {
    double K[m * n];
    LQ_UNROLL for (int e = 0; e < m * n; ++e) K[e] = ws[oK + (int64_t)k * (m * n) + e];
    mv<m, n>(K, x, u);
    LQ_UNROLL for (int j = 0; j < m; ++j)
      if (trk) u[j] += ws[L.okc + (int64_t)k * m + j];
    double worst = 1.0;
    int row = -1;
    for (int i = 0; i < p; ++i) {
      const double fu = poly_row<m>(py, i, u);
      if (fu > worst) { worst = fu; row = i; }
    }
    if (row >= 0) {
      const double sc = 1.0 / worst;
      LQ_UNROLL for (int j = 0; j < m; ++j) u[j] *= sc;
      W.set(k * p + row);
    }
    LQ_UNROLL for (int j = 0; j < m; ++j) ws[L.oz + (int64_t)k * m + j] = u[j];
    step_model<n, m>(pl.Ah, pl.Bh, x, u, xn);
    LQ_UNROLL for (int i = 0; i < n; ++i) x[i] = xn[i];
  }
  // ---- 3. primal active-set iterations
  const int maxit = 8 * N * p + 32;
  bool done = false;
  for (int it = 0; it < maxit && !done; ++it) {
    if (!pclqr_backward<n, m>(pb, pl, N, W, py, ws, rf)) flags |= FLAG_CHOL_FAIL;
    // forward sweep: candidate z* (zs), its trajectory (xs), largest feasible step along z* - z
    double alpha = 1.0;
    int block = -1;
    LQ_UNROLL for (int i = 0; i < n; ++i) { x[i] = x0[i]; ws[L.oxs + i] = x0[i]; }
    for (int k = 0; k < N; ++k) {
      double K[m * n], zc[m];
      LQ_UNROLL for (int e = 0; e < m * n; ++e) K[e] = ws[L.oKc + (int64_t)k * (m * n) + e];
      mv<m, n>(K, x, u);
      LQ_UNROLL for (int j = 0; j < m; ++j) {
        u[j] += ws[L.okc + (int64_t)k * m + j];
        ws[L.ozs + (int64_t)k * m + j] = u[j];
        zc[j] = ws[L.oz + (int64_t)k * m + j];
      }
      for (int i = 0; i < p; ++i) {
        if (W.test(k * p + i)) continue;
        const double fs = poly_row<m>(py, i, u);
        if (fs > 1.0 + 1e-13) {                            // (rows meeting at a degenerate vertex sit at 1 +- rounding)
          const double fc = poly_row<m>(py, i, zc);
          const double a = (1.0 - fc) / (fs - fc);
          if (a < alpha) { alpha = a; block = k * p + i; }
        }
      }
      step_model<n, m>(pl.Ah, pl.Bh, x, u, xn);
      LQ_UNROLL for (int i = 0; i < n; ++i) { x[i] = xn[i]; ws[L.oxs + (int64_t)(k + 1) * n + i] = xn[i]; }
    }
    if (block >= 0) {
      if (alpha < 0.0) alpha = 0.0;
      for (int e = 0; e < N * m; ++e) {
        const double zc = ws[L.oz + e];
        ws[L.oz + e] = fma(alpha, ws[L.ozs + e] - zc, zc);
      }
      W.set(block);
      continue;
    }
    // full step: z = z*; multipliers of the active rows from the costate sweep over the stored trajectory
    for (int e = 0; e < N * m; ++e) ws[L.oz + e] = ws[L.ozs + e];
    double lam[n];
    {
      double xe[n];
      LQ_UNROLL for (int i = 0; i < n; ++i) xe[i] = ws[L.oxs + (int64_t)N * n + i] - rf.x(i, N - 1);
      mv<n, n>(pb.Pt, xe, lam);
      LQ_UNROLL for (int i = 0; i < n; ++i) lam[i] *= 2.0;
    }
    double worst = 0.0;
    int rel = -1;
    for (int k = N - 1; k >= 0; --k) {
      double FW[m * m];
      const int c = poly_gather<m>(py, W, k, FW);
      if (c > 0) {
        double uk[m], g[m], gs = 0.0;
        LQ_UNROLL for (int j = 0; j < m; ++j) uk[j] = ws[L.oz + (int64_t)k * m + j] - rf.u(j, k);
        mv<m, m>(pb.R, uk, g);
        LQ_UNROLL for (int j = 0; j < m; ++j) {
          double acc = 2.0 * g[j];
          gs += fabs(acc);
          double a2 = 0.0;
          LQ_UNROLL for (int r = 0; r < n; ++r) a2 = fma(pl.Bh[r * m + j], lam[r], a2);
          gs += fabs(a2);
          g[j] = acc + a2;                                   // dJ/du_{k,j}
        }
        // mu = -(F_W F_W')^-1 F_W g  (identity-padded to m x m)
        double M[m * m], mu[m];
        LQ_UNROLL for (int i = 0; i < m; ++i) {
          LQ_UNROLL for (int r = 0; r < m; ++r) {
            double acc = 0.0;
            LQ_UNROLL for (int j = 0; j < m; ++j) acc = fma(FW[i * m + j], FW[r * m + j], acc);
            M[i * m + r] = acc;
          }
          double acc = 0.0;
          LQ_UNROLL for (int j = 0; j < m; ++j) acc = fma(FW[i * m + j], g[j], acc);
          mu[i] = -acc;
        }
        LQ_UNROLL for (int i = 0; i < m; ++i)
          if (i >= c) M[i * m + i] = 1.0;
        if (!chol<m>(M)) flags |= FLAG_CHOL_FAIL;
        solve_l<m, 1>(M, mu);
        solve_lt<m, 1>(M, mu);
        // the i-th gathered row is the i-th set bit of stage k
        int idx = 0;
        for (int i = 0; i < p; ++i) {
          if (idx < m && W.test(k * p + i)) {
            double mui = 0.0, fn = 0.0;
            LQ_UNROLL for (int r = 0; r < m; ++r)
              if (r == idx) {
                mui = mu[r];
                LQ_UNROLL for (int j = 0; j < m; ++j) fn += fabs(FW[r * m + j]);
              }
            const double tol = 1e-11 * gs / (fn + 1e-300) + 1e-300;
            if (-mui > tol && -mui > worst) { worst = -mui; rel = k * p + i; }
            ++idx;
          }
        }
      }
      if (k > 0) {
        double xk[n], qx[n], atl[n];
        LQ_UNROLL for (int i = 0; i < n; ++i) xk[i] = ws[L.oxs + (int64_t)k * n + i] - rf.x(i, k - 1);
        mv<n, n>(pb.Q, xk, qx);
        LQ_UNROLL for (int i = 0; i < n; ++i) {
          double acc = 2.0 * qx[i];
          LQ_UNROLL for (int r = 0; r < n; ++r) acc = fma(pl.Ah[r * n + i], lam[r], acc);
          atl[i] = acc;
        }
        LQ_UNROLL for (int i = 0; i < n; ++i) lam[i] = atl[i];
      }
    }
    if (rel < 0) done = true;
    else W.clear(rel);
  }
  if (!done) flags |= FLAG_QP_MAXITER;
  // ---- 4. objective along z
  LQ_UNROLL for (int i = 0; i < n; ++i) x[i] = x0[i];
  double cost = quad<n>(x0, pb.Q, x0);
  for (int k = 0; k < N; ++k) {
    LQ_UNROLL for (int j = 0; j < m; ++j) {
      u[j] = ws[L.oz + (int64_t)k * m + j];
      if (k == 0) u0[j] = u[j];
    }
    step_model<n, m>(pl.Ah, pl.Bh, x, u, xn);
    double du[m], dx[n];
    LQ_UNROLL for (int j = 0; j < m; ++j) du[j] = u[j] - rf.u(j, k);
    LQ_UNROLL for (int i = 0; i < n; ++i) dx[i] = xn[i] - rf.x(i, k);
    cost += quad<m>(du, pb.R, du);
    cost += (k == N - 1) ? quad<n>(dx, pb.Pt, dx) : quad<n>(dx, pb.Q, dx);
    LQ_UNROLL for (int i = 0; i < n; ++i) x[i] = xn[i];
  }
  *V = cost;
  return flags;
}

// Closed-loop simulation (utils_class.py:245-285) with the polytope-constrained controller.
template <int n, int m, class Traj>
LQ_HD int psimulate_sample(const Problem<n, m>& pb, const Plan<n, m>& pl, int N, int T, const double* x0,
                           const Poly& py, const WsView& ws, double* J_T, int* n_active, Traj& traj,
                           const Refs& rf = Refs()) {
  double x[n], xn[n], u[m];
  LQ_UNROLL for (int i = 0; i < n; ++i) x[i] = x0[i];
  traj.state(0, x);
  double cost = quad<n>(x, pb.Q, x);
  int flags = 0, act = 0;
  for (int t = 0; t < T; ++t) {
    double V;
    const int f = pclqr_solve<n, m>(pb, pl, N, x, py, ws, u, &V, rf);
    flags |= f;
    act += (f & FLAG_QP_ACTIVE) ? 1 : 0;
    step_model<n, m>(pb.A, pb.B, x, u, xn);
    cost += quad<n>(xn, pb.Q, xn);
    cost += quad<m>(u, pb.R, u);
    traj.input(t, u);
    traj.state(t + 1, xn);
    LQ_UNROLL for (int i = 0; i < n; ++i) x[i] = xn[i];
  }
  *J_T = cost;
  *n_active = act;
  return flags;
}

// Feasibility certificate of the unconstrained plan for the polytope (plan_prepare's argument with rows F_i instead of
// box components): the planned input is u_k = g_k x_0, g_k = K_k Phi_k, so by Cauchy-Schwarz in the P0 metric
//     F_i u_k <= sqrt(F_i g_k P0^-1 g_k' F_i') sqrt(x_0' P0 x_0),
// and x_0' P0 x_0 <= cstar := min_{k,i} 1 / (F_i g_k P0^-1 g_k' F_i') keeps every planned input inside F_u u <= 1.
// Reads the gains plan_prepare stored (ws.Ku). Returns cstar with the 1 - 1e-9 margin, -1 when P0 is not positive
// definite.
template <int n, int m>
LQ_HD double poly_certificate(const Plan<n, m>& pl, int N, const Poly& py, const WsView& ws) {
  const ClqrLayout<n, m> L(N);
  double Lc[n * n], Lci[n], Phi[n * n];
  LQ_UNROLL for (int i = 0; i < n * n; ++i) Lc[i] = pl.P0[i];
  if (!chol_inv<n>(Lc, Lci)) return -1.0;
  LQ_UNROLL for (int i = 0; i < n; ++i)
    LQ_UNROLL for (int j = 0; j < n; ++j) Phi[i * n + j] = (i == j) ? 1.0 : 0.0;
  double cs = HUGE_VAL;
  for (int k = 0; k < N; ++k) {
    double K[m * n], g[m * n];
    LQ_UNROLL for (int e = 0; e < m * n; ++e) K[e] = ws[L.oKu + (int64_t)k * (m * n) + e];
    mm<m, n, n>(K, Phi, g);
    for (int r = 0; r < py.p; ++r) {
      double y[n], q = 0.0;                                  // y = L^-1 (F_r g)', q = y'y
      LQ_UNROLL for (int i = 0; i < n; ++i) {
        double acc = 0.0;
        LQ_UNROLL for (int j = 0; j < m; ++j) acc = fma(py.f(r, j, m), g[j * n + i], acc);
        LQ_UNROLL for (int c = 0; c < i; ++c) acc = fma(-Lc[i * n + c], y[c], acc);
        y[i] = acc * Lci[i];
        q = fma(y[i], y[i], q);
      }
      if (q > 0.0) cs = dmin(cs, 1.0 / q);
    }
    if (k + 1 < N) {
      double Acl[n * n], Pn[n * n];
      LQ_UNROLL for (int i = 0; i < n; ++i)
        LQ_UNROLL for (int j = 0; j < n; ++j) {
          double acc = pl.Ah[i * n + j];
          LQ_UNROLL for (int r = 0; r < m; ++r) acc = fma(pl.Bh[i * m + r], K[r * n + j], acc);
          Acl[i * n + j] = acc;
        }
      mm<n, n, n>(Acl, Phi, Pn);
      LQ_UNROLL for (int i = 0; i < n * n; ++i) Phi[i] = Pn[i];
    }
  }
  return (cs == cs) ? cs * (1.0 - 1e-9) : -1.0;
}

// Infinite-horizon closed loop with the input polytope (clqr.cuh: certified_closed_loop): the unconstrained plan of
// plan_prepare, the polytope certificate above, pclqr_solve for the steps before the certificate.
template <int n, int m>
LQ_HD int psimulate_inf_sample(const Problem<n, m>& pb, Plan<n, m>& pl, int N, int T_max, const double* x0,
                               const Poly& py, const WsView& ws, double* J_inf, int* T_cert) {
  const int pf = plan_prepare<n, m>(pb, pl, N, ws, /*certificate=*/false);
  const double cstar = poly_certificate<n, m>(pl, N, py, ws);
  return pf | certified_closed_loop<n, m>(pb, pl, N, cstar, T_max, x0, ws, [&](const double* x, double* u) {
    double V;
    return pclqr_solve<n, m>(pb, pl, N, x, py, ws, u, &V);
  }, J_inf, T_cert);
}

}  // namespace lq
