// worst_inf.cuh — exact gradient of the input-constrained closed loop's certified J_inf (K2c, clqr.cuh:
// certified_closed_loop) in the model error (dA, dB), and the projected ascent of worst.cuh on it. Box only, regulation
// only, one sample per thread.
//
//   J_inf = sum_{t<tau} (x_t'Q x_t + u_t'R u_t) + x_tau'S x_tau,  u_t = QP_N(x_t; A^, B^)_0,  x_{t+1} = A x_t + B u_t,
//
// S = W + A_cl'S A_cl with A_cl = A + B K0, K0 the unconstrained horizon-N gain of (A^, B^). J_inf is continuous in
// (dA, dB): the QP minimiser is continuous in its data (strictly convex, fixed constraints), and the certified step tau
// makes no jump, because a state just outside the S-level set still gets u = K0 x (the level set lies strictly inside
// the feasibility ellipsoid), where x'S x = x'Q x + u'R u + x+'S x+ holds exactly. It is smooth wherever every
// pre-certificate QP is strictly complementary, and there its gradient is one reverse pass over the steps t < tau.
// With lambda the cotangent of x_{t+1}, lambda_tau = 2 S x_tau, and c = 2 R u_t + B'lambda that of u_t:
//   * the step took the unconstrained law (the certificate's fast path or a feasible rollout): u_t = K0 x_t, so
//     Kbar += c x_t' and lambda <- 2 Q x_t + A'lambda + K0'c;
//   * a bound was active: with the final working set fixed u_t = Kc0 x_t + kc0 (Kc0 the stage-0 gain of the last affine
//     sweep), so lambda <- 2 Q x_t + A'lambda + Kc0'c, plus the vector-Jacobian product of c'u_t in (A^, B^) (qp_vjp).
// The tail adds Kbar += 2 (R K0 + B'S A_cl) Lambda with Lambda = x_tau x_tau' + A_cl Lambda A_cl' (worst_eval's adjoint
// with x0 := x_tau), and riccati_adjoint maps the summed Kbar to (gA, gB). At tau = 0 this is worst_eval's gradient.
//
// The reverse pass needs x_t for t <= tau: the forward pass stores them (the states region of the workspace) and each
// step's QP is solved again from its stored state, which regenerates its working set, gains and plan bit for bit.
#pragma once
#include "worst.cuh"

namespace lq {

// the objective's failure flags: a value or gradient with one of them is not used
constexpr int kInfFail = kWorstFail | FLAG_QP_MAXITER | FLAG_TAIL_UNCERTIFIED;

// doubles of qp_vjp's plan records: the plan x^ [N+1][n], u [N][m] and the adjoint plan xb [N+1][n], ub [N][m]
template <int n, int m>
LQ_HD int64_t vjp_ws_doubles(int N) {
  return 2 * ((int64_t)(N + 1) * n + (int64_t)N * m);
}

// Per-sample workspace of inf_grad_eval: clqr.cuh's solve region first (all a value-only call touches), then the
// Riccati stage records, the VJP's plan records and the closed-loop states x_0..x_tau.
template <int n, int m>
struct InfGradLayout {
  int64_t oW, oV, oX, total;
  LQ_HD InfGradLayout(int N, int T_max) {
    oW = clqr_ws_doubles<n, m>(N);
    oV = oW + worst_ws_doubles<n, m>(N);
    oX = oV + vjp_ws_doubles<n, m>(N);
    total = oX + (int64_t)(T_max + 1) * n;
  }
};

LQ_HD WsView ws_at(const WsView& ws, int64_t off) { return WsView{ws.p + off * ws.stride, ws.stride}; }

// Vector-Jacobian product of the QP's first input: qA += d(c'u_0)/dA^, qB += d(c'u_0)/dB^ for the solve from x0 that
// clqr_solve just finished (its workspace `ws` and final working set `aset`), by the implicit-function theorem on the
// equality-constrained LQ of that working set. The adjoint LQ has the same (A^, B^, Q, R, P), xb_0 = 0, the clamped
// inputs fixed at 0, ub_0 = G~^-1 c / 2 on the free inputs (G~ = R + B^'S_1 B^, S_1 the working set's cost-to-go at
// stage 1) and ub_k = Kc_k xb_k beyond. With the costates p_N = 2 P x^_N, p_k = 2 Q x^_k + A^'p_{k+1} (and pb alike):
//   d(c'u_0)/dA^ = -sum_{k<N} (pb_{k+1} x^_k' + p_{k+1} xb_k'),   d(c'u_0)/dB^ = -sum_{k<N} (pb_{k+1} u_k' + p_{k+1} ub_k').
// The stage-0 gain of the working set goes to Kc0. rec holds vjp_ws_doubles(N) doubles.
template <int n, int m>
LQ_HD void qp_vjp(const Problem<n, m>& pb, const Plan<n, m>& pl, int N, const double* x0, const double* c,
                  const ClqrActiveSet& aset, const WsView& ws, const WsView& rec, double* qA, double* qB,
                  double* Kc0) {
  const ClqrLayout<n, m> L(N);
  const int64_t ou = (int64_t)(N + 1) * n, oxb = ou + (int64_t)N * m, oub = oxb + (int64_t)(N + 1) * n;
  auto gain = [&](int k, double* K, double* kv) {
    const bool tail = k > aset.klast;
    const int64_t og = tail ? L.oKu : L.oKc;
    LQ_UNROLL for (int e = 0; e < m * n; ++e) K[e] = ws[og + (int64_t)k * (m * n) + e];
    LQ_UNROLL for (int j = 0; j < m; ++j) kv[j] = tail ? 0.0 : ws[L.okc + (int64_t)k * m + j];
  };
  // 1. the plan of the working set
  double x[n], xn[n], u[m];
  LQ_UNROLL for (int i = 0; i < n; ++i) { x[i] = x0[i]; rec[i] = x0[i]; }
  for (int k = 0; k < N; ++k) {
    double K[m * n], kv[m];
    gain(k, K, kv);
    if (k == 0) { LQ_UNROLL for (int e = 0; e < m * n; ++e) Kc0[e] = K[e]; }
    mv<m, n>(K, x, u);
    LQ_UNROLL for (int j = 0; j < m; ++j) { u[j] += kv[j]; rec[ou + (int64_t)k * m + j] = u[j]; }
    step_model<n, m>(pl.Ah, pl.Bh, x, u, xn);
    LQ_UNROLL for (int i = 0; i < n; ++i) { x[i] = xn[i]; rec[(int64_t)(k + 1) * n + i] = xn[i]; }
  }
  // 2. S_1: S_N = P, S_k = Q + K_k'R K_k + (A^ + B^ K_k)'S_{k+1}(A^ + B^ K_k) with the working set's gains
  double S[n * n];
  LQ_UNROLL for (int i = 0; i < n * n; ++i) S[i] = pb.Pt[i];
  for (int k = N - 1; k >= 1; --k) {
    double K[m * n], kv[m], Acl[n * n], SA[n * n], RK[m * n], Sn[n * n];
    gain(k, K, kv);
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = 0; j < n; ++j) {
        double acc = pl.Ah[i * n + j];
        LQ_UNROLL for (int r = 0; r < m; ++r) acc = fma(pl.Bh[i * m + r], K[r * n + j], acc);
        Acl[i * n + j] = acc;
      }
    mm<m, m, n>(pb.R, K, RK);
    mm<n, n, n>(S, Acl, SA);
    sym_add_mtm<m, n>(pb.Q, K, RK, Sn);
    sym_add_mtm<n, n>(Sn, Acl, SA, S);
  }
  // 3. ub_0 = G~^-1 c / 2 on the free inputs of stage 0
  double ub[m];
  {
    double SB[n * m], G[m * m];
    bool fx[m];
    mm<n, n, m>(S, pl.Bh, SB);
    LQ_UNROLL for (int i = 0; i < m; ++i) {
      fx[i] = aset.fixed.test(i);
      LQ_UNROLL for (int j = 0; j < m; ++j) {
        double acc = pb.R[i * m + j];
        LQ_UNROLL for (int r = 0; r < n; ++r) acc = fma(pl.Bh[r * m + i], SB[r * m + j], acc);
        G[i * m + j] = acc;
      }
    }
    LQ_UNROLL for (int i = 0; i < m; ++i) {
      ub[i] = fx[i] ? 0.0 : 0.5 * c[i];
      LQ_UNROLL for (int j = 0; j < m; ++j)
        if (fx[i] || fx[j]) G[i * m + j] = (i == j) ? 1.0 : 0.0;
    }
    chol<m>(G);
    solve_l<m, 1>(G, ub);
    solve_lt<m, 1>(G, ub);
  }
  // 4. the adjoint plan
  double xb[n];
  LQ_UNROLL for (int i = 0; i < n; ++i) { xb[i] = 0.0; rec[oxb + i] = 0.0; }
  for (int k = 0; k < N; ++k) {
    if (k > 0) {
      double K[m * n], kv[m];
      gain(k, K, kv);
      mv<m, n>(K, xb, ub);
    }
    LQ_UNROLL for (int j = 0; j < m; ++j) rec[oub + (int64_t)k * m + j] = ub[j];
    step_model<n, m>(pl.Ah, pl.Bh, xb, ub, xn);
    LQ_UNROLL for (int i = 0; i < n; ++i) { xb[i] = xn[i]; rec[oxb + (int64_t)(k + 1) * n + i] = xn[i]; }
  }
  // 5. both costates backward, and the sums
  double p[n], pq[n];
  mv<n, n>(pb.Pt, x, p);
  mv<n, n>(pb.Pt, xb, pq);
  LQ_UNROLL for (int i = 0; i < n; ++i) { p[i] *= 2.0; pq[i] *= 2.0; }
  for (int k = N - 1; k >= 0; --k) {
    double xk[n], uk[m], xbk[n], ubk[m];
    LQ_UNROLL for (int i = 0; i < n; ++i) { xk[i] = rec[(int64_t)k * n + i]; xbk[i] = rec[oxb + (int64_t)k * n + i]; }
    LQ_UNROLL for (int j = 0; j < m; ++j) { uk[j] = rec[ou + (int64_t)k * m + j]; ubk[j] = rec[oub + (int64_t)k * m + j]; }
    LQ_UNROLL for (int i = 0; i < n; ++i) {
      LQ_UNROLL for (int j = 0; j < n; ++j) qA[i * n + j] -= fma(pq[i], xk[j], p[i] * xbk[j]);
      LQ_UNROLL for (int j = 0; j < m; ++j) qB[i * m + j] -= fma(pq[i], uk[j], p[i] * ubk[j]);
    }
    if (k > 0) {
      double a[n], b[n];
      mv<n, n>(pb.Q, xk, a);
      mv<n, n>(pb.Q, xbk, b);
      LQ_UNROLL for (int i = 0; i < n; ++i) {
        double s1 = 2.0 * a[i], s2 = 2.0 * b[i];
        LQ_UNROLL for (int r = 0; r < n; ++r) { s1 = fma(pl.Ah[r * n + i], p[r], s1); s2 = fma(pl.Ah[r * n + i], pq[r], s2); }
        a[i] = s1; b[i] = s2;
      }
      LQ_UNROLL for (int i = 0; i < n; ++i) { p[i] = a[i]; pq[i] = b[i]; }
    }
  }
}

// K2c's J_inf, T_cert and flags at the model error (dA, dB) from x0, computed by plan_prepare + certified_closed_loop
// exactly as simulate_inf_sample, and rho(A + B K0). With gA / gB non-null also dJ_inf/d(dA) [n*n] and dJ_inf/d(dB)
// [n*m]: NaN where J_inf is +inf or NaN or a flag of kInfFail is set. ws holds InfGradLayout(N, T_max).total doubles
// (clqr_ws_doubles(N) for a value-only call, which writes nothing beyond them).
template <int n, int m>
LQ_HD int inf_grad_eval(const Problem<n, m>& pb, const double* dA, const double* dB, const double* x0, int N,
                        int T_max, const WsView& ws, double* J_out, int* T_cert, double* rho_out, double* gA,
                        double* gB) {
  const bool grad = gA != nullptr;
  const InfGradLayout<n, m> lay(N, T_max);
  const WsView wx = ws_at(ws, lay.oX);
  Plan<n, m> pl;
  LQ_UNROLL for (int i = 0; i < n * n; ++i) pl.Ah[i] = pb.A[i] + dA[i];
  LQ_UNROLL for (int i = 0; i < n * m; ++i) pl.Bh[i] = pb.B[i] + dB[i];
  int flags = plan_prepare<n, m>(pb, pl, N, ws, /*certificate=*/true);
  if (grad) { LQ_UNROLL for (int i = 0; i < n; ++i) wx[i] = x0[i]; }
  int t = 0;
  flags |= certified_closed_loop<n, m>(pb, pl, N, pl.cstar, T_max, x0, ws, [&](const double* x, double* u) {
    double V;
    const int f = clqr_solve<n, m>(pb, pl, N, x, ws, u, &V);
    if (grad) {                                   // x_{t+1}, as certified_closed_loop forms it
      double xn[n];
      step_model<n, m>(pb.A, pb.B, x, u, xn);
      ++t;
      LQ_UNROLL for (int i = 0; i < n; ++i) wx[(int64_t)t * n + i] = xn[i];
    }
    return f;
  }, J_out, T_cert);
  double K0[m * n], Acl[n * n];
  LQ_UNROLL for (int e = 0; e < m * n; ++e) K0[e] = Plan<n, m>::kHoldK0 ? pl.K0[Plan<n, m>::kHoldK0 ? e : 0]
                                                                         : ws[ClqrLayout<n, m>(N).oKu + e];
  LQ_UNROLL for (int i = 0; i < n; ++i)
    LQ_UNROLL for (int j = 0; j < n; ++j) {
      double acc = pb.A[i * n + j];
      LQ_UNROLL for (int k = 0; k < m; ++k) acc = fma(pb.B[i * m + k], K0[k * n + j], acc);
      Acl[i * n + j] = acc;
    }
  {
    bool ok;
    *rho_out = spectral_radius<n>(Acl, &ok);
  }
  if (!grad) return flags;
  LQ_UNROLL for (int i = 0; i < n * n; ++i) gA[i] = NAN;
  LQ_UNROLL for (int i = 0; i < n * m; ++i) gB[i] = NAN;
  if ((flags & (kInfFail | FLAG_UNSTABLE)) || !(fabs(*J_out) <= 1.79e308)) return flags;

  // the Riccati records of the adjoint; K0 and S as the value path formed them (same recursion, same operations)
  const WsView ww = ws_at(ws, lay.oW);
  double P[n * n], W[n * n], RK[m * n], S[n * n];
  LQ_UNROLL for (int i = 0; i < n * n; ++i) P[i] = pb.Pt[i];
  RicStage<n, m> st;
  riccati_records<n, m>(pb, pl.Ah, pl.Bh, N, ww, true, P, st, K0);
  LQ_UNROLL for (int i = 0; i < n; ++i)
    LQ_UNROLL for (int j = 0; j < n; ++j) {
      double acc = pb.A[i * n + j];
      LQ_UNROLL for (int k = 0; k < m; ++k) acc = fma(pb.B[i * m + k], K0[k * n + j], acc);
      Acl[i * n + j] = acc;
    }
  mm<m, m, n>(pb.R, K0, RK);
  sym_add_mtm<m, n>(pb.Q, K0, RK, W);
  if (!lyapunov_doubling<n>(Acl, W, S)) return flags | FLAG_LYAP_NOCONV;

  const int tau = *T_cert;
  double xt[n], lam[n], Kbar[m * n], qA[n * n], qB[n * m];
  LQ_UNROLL for (int i = 0; i < n; ++i) xt[i] = wx[(int64_t)tau * n + i];
  mv<n, n>(S, xt, lam);
  LQ_UNROLL for (int i = 0; i < n; ++i) lam[i] *= 2.0;
  LQ_UNROLL for (int i = 0; i < m * n; ++i) Kbar[i] = 0.0;
  LQ_UNROLL for (int i = 0; i < n * n; ++i) qA[i] = 0.0;
  LQ_UNROLL for (int i = 0; i < n * m; ++i) qB[i] = 0.0;
  const WsView wv = ws_at(ws, lay.oV);
  for (int s = tau - 1; s >= 0; --s) {
    double x[n], u[m], V, c[m], Ks[m * n];
    LQ_UNROLL for (int i = 0; i < n; ++i) x[i] = wx[(int64_t)s * n + i];
    ClqrActiveSet aset;
    const int f = clqr_solve<n, m>(pb, pl, N, x, ws, u, &V, Refs(), 0, &aset);
    mv<m, m>(pb.R, u, c);
    LQ_UNROLL for (int j = 0; j < m; ++j) {
      double acc = 2.0 * c[j];
      LQ_UNROLL for (int r = 0; r < n; ++r) acc = fma(pb.B[r * m + j], lam[r], acc);
      c[j] = acc;
    }
    if (f & FLAG_QP_ACTIVE) {
      qp_vjp<n, m>(pb, pl, N, x, c, aset, ws, wv, qA, qB, Ks);
    } else {
      LQ_UNROLL for (int e = 0; e < m * n; ++e) Ks[e] = K0[e];
      LQ_UNROLL for (int j = 0; j < m; ++j)
        LQ_UNROLL for (int i = 0; i < n; ++i) Kbar[j * n + i] = fma(c[j], x[i], Kbar[j * n + i]);
    }
    double nl[n], qx[n];
    mv<n, n>(pb.Q, x, qx);
    LQ_UNROLL for (int i = 0; i < n; ++i) {
      double acc = 2.0 * qx[i];
      LQ_UNROLL for (int r = 0; r < n; ++r) acc = fma(pb.A[r * n + i], lam[r], acc);
      LQ_UNROLL for (int j = 0; j < m; ++j) acc = fma(Ks[j * n + i], c[j], acc);
      nl[i] = acc;
    }
    LQ_UNROLL for (int i = 0; i < n; ++i) lam[i] = nl[i];
  }
  // the tail: Kbar += 2 (R K0 + B'S A_cl) Lambda, Lambda the Gramian of the closed loop from x_tau
  {
    double AclT[n * n], X0[n * n], Lam[n * n], SA[n * n], T[m * n], TL[m * n];
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = 0; j < n; ++j) { AclT[i * n + j] = Acl[j * n + i]; X0[i * n + j] = xt[i] * xt[j]; }
    if (!lyapunov_doubling<n>(AclT, X0, Lam)) return flags | FLAG_LYAP_NOCONV;
    mm<n, n, n>(S, Acl, SA);
    mtm<n, m, n>(pb.B, SA, T);
    LQ_UNROLL for (int i = 0; i < m * n; ++i) T[i] = 2.0 * (T[i] + RK[i]);
    mm<m, n, n>(T, Lam, TL);
    LQ_UNROLL for (int i = 0; i < m * n; ++i) Kbar[i] += TL[i];
  }
  riccati_adjoint<n, m>(pl.Ah, pl.Bh, K0, P, st, Kbar, N, ww, gA, gB);
  LQ_UNROLL for (int i = 0; i < n * n; ++i) gA[i] += qA[i];
  LQ_UNROLL for (int i = 0; i < n * m; ++i) gB[i] += qB[i];
  return flags;
}

// The ascent of worst.cuh (ascent_run) on inf_grad_eval's J_inf, rejecting trials with a flag of kInfFail. T_cert of
// the final point goes to *T_cert.
template <int n, int m>
LQ_HD int inf_ascent(const Problem<n, m>& pb, double* dA, double* dB, const double* x0, int N, int T_max,
                     const AscentSettings& as, const WsView& ws, double* J_out, int* T_cert, double* rho_out,
                     int* iters) {
  int tc_trial = -1;
  return ascent_run<n, m, kInfFail>(dA, dB, as, [&](const double* a, const double* b, double* J, double* rho,
                                                    double* ga, double* gb) {
    return inf_grad_eval<n, m>(pb, a, b, x0, N, T_max, ws, J, ga ? T_cert : &tc_trial, rho, ga, gb);
  }, [&]() { *T_cert = tc_trial; }, J_out, rho_out, iters);
}

}  // namespace lq
