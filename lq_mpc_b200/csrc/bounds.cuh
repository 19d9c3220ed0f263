// bounds.cuh — K3: per-sample bound coefficients alpha, beta (energy_bound) and xi, eta (energy_decreasing).
//
// Restates (citations into /root/reference):
//   ct.dlqr                         utils_class.py:761,840,923  -> DARE by structure-preserving doubling (SDA)
//   local_radius                    utils.py:548-564
//   ex_stability_lq                 utils.py:343-380   (closed loop taken as A + B K; the reference's `A + B * K`
//                                                        is element-wise and equals it exactly when m = 1)
//   ex_stability_bounds             utils.py:567-584
//   geo_M, fc_omega_eta, fc_ec_h    utils.py:393-409, 469-523, 526-538
//   fc_ec_g_x/g_u, bar_g_x/bar_g_u  utils.py:78-117, 186-223
//   sl_syn_Phi / sl_syn_Gamma       utils.py:126-174   (never materialised: only G_d = A^d B and Gram matrices)
//   fc_ec_theta, fc_ec_E            utils.py:226-334
//   energy_bound / energy_decreasing  utils_class.py:308-373 ; J_bound  utils_class.py:858-859
//
// ||Gamma||_2 and lambda_min(H^) need extreme eigenvalues of (N m) x (N m) symmetric matrices. They are obtained
// MATRIX-FREE (gramspec.cuh): Gamma is a simulation operator, so "H^ - x I is positive definite" is decided by an
// N-stage Riccati-type elimination on n x n blocks and the extremes follow by bisection — O(N n^3) per probe, no
// scratch memory. Only the literal kron(Q, I) weight ordering of utils.py:317-318 with NON-scalar Q, R (not a stage-wise
// cost) still takes the dense route: Gram matrix by a block recurrence (O(N^2 m^2 n)), Householder tridiagonalisation
// inside the strided per-thread workspace, Sturm bisection (also reachable with LQMPC_K3_DENSE=1 for A/B tests).
#pragma once
#include "clqr.cuh"
#include "gramspec.cuh"

namespace lq {

enum BoundField : int {
  BF_ALPHA = 0, BF_BETA, BF_XI, BF_ETA, BF_BOUND, BF_E_PSI, BF_E_U, BF_E_PSI_U, BF_THETA_U, BF_THETA_X_U,
  BF_C_K, BF_RHO_K, BF_GAMMA, BF_RHO_GAMMA, BF_L_V, BF_N_0, BF_OMEGA_N1, BF_OMEGA_N0D5, BF_ERR_TH, BF_N_MIN,
  BF_H, BF_EPSILON_K, BF_NORM_A, BF_NORM_B, BF_NORM_K, BF_NORM_GAMMA, BF_NORM_PHI, BF_MIN_H, BF_RHO_CL,
  BF_BAR_U, BF_BAR_D_U, BF_COUNT
};

// ---- DARE: X = A'X(I + G X)^-1 A + Q, G = B R^-1 B', by the structure-preserving doubling algorithm.
template <int n, int m>
LQ_HD bool dare_sda(const double* A, const double* B, const double* Q, const double* R, double* X) {
  double Ak[n * n], G[n * n], H[n * n];
  {
    double L[m * m], Y[n * m];
    LQ_UNROLL for (int i = 0; i < m * m; ++i) L[i] = R[i];
    chol<m>(L);
    LQ_UNROLL for (int i = 0; i < n * m; ++i) Y[i] = B[i];
    solve_right_lt<n, m>(L, Y);
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = i; j < n; ++j) {
        double acc = 0.0;
        LQ_UNROLL for (int k = 0; k < m; ++k) acc = fma(Y[i * m + k], Y[j * m + k], acc);
        G[i * n + j] = acc; G[j * n + i] = acc;
      }
  }
  LQ_UNROLL for (int i = 0; i < n * n; ++i) { Ak[i] = A[i]; H[i] = Q[i]; }
  bool conv = false;
  for (int it = 0; it < 60 && !conv; ++it) {
    double W[n * n], V[n * 2 * n];   // V = W^-1 [A | G]
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = 0; j < n; ++j) {
        double acc = (i == j) ? 1.0 : 0.0;
        LQ_UNROLL for (int k = 0; k < n; ++k) acc = fma(G[i * n + k], H[k * n + j], acc);
        W[i * n + j] = acc;
        V[i * 2 * n + j] = Ak[i * n + j];
        V[i * 2 * n + n + j] = G[i * n + j];
      }
    if (!lu_solve<n, 2 * n>(W, V)) return false;
    double V1[n * n], V2[n * n], T1[n * n], An[n * n];
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = 0; j < n; ++j) { V1[i * n + j] = V[i * 2 * n + j]; V2[i * n + j] = V[i * 2 * n + n + j]; }
    mm<n, n, n>(Ak, V1, An);                    // A+ = A W^-1 A
    // G+ = G + A (W^-1 G) A'
    mm<n, n, n>(Ak, V2, T1);
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = i; j < n; ++j) {
        double acc = 0.0;
        LQ_UNROLL for (int k = 0; k < n; ++k) acc = fma(T1[i * n + k], Ak[j * n + k], acc);
        double acc2 = 0.0;
        LQ_UNROLL for (int k = 0; k < n; ++k) acc2 = fma(T1[j * n + k], Ak[i * n + k], acc2);
        const double v = G[i * n + j] + 0.5 * (acc + acc2);
        G[i * n + j] = v; G[j * n + i] = v;
      }
    // H+ = H + A' H (W^-1 A)
    double HV[n * n];
    mm<n, n, n>(H, V1, HV);
    double dmaxv = 0.0, hmax = 0.0;
    double Hn[n * n];
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = i; j < n; ++j) {
        double acc = 0.0, acc2 = 0.0;
        LQ_UNROLL for (int k = 0; k < n; ++k) acc = fma(Ak[k * n + i], HV[k * n + j], acc);
        LQ_UNROLL for (int k = 0; k < n; ++k) acc2 = fma(Ak[k * n + j], HV[k * n + i], acc2);
        const double inc = 0.5 * (acc + acc2);
        const double v = H[i * n + j] + inc;
        Hn[i * n + j] = v; Hn[j * n + i] = v;
        dmaxv = dmax(dmaxv, fabs(inc));
        hmax = dmax(hmax, fabs(v));
      }
    LQ_UNROLL for (int i = 0; i < n * n; ++i) { H[i] = Hn[i]; Ak[i] = An[i]; }
    if (!(dmaxv > 1e-17 * hmax)) conv = (dmaxv == dmaxv);
  }
  LQ_UNROLL for (int i = 0; i < n * n; ++i) X[i] = H[i];
  return conv;
}

// K = (R + B'XB)^-1 B'XA  (python-control convention u = -Kx)
template <int n, int m>
LQ_HD void dlqr_gain(const double* A, const double* B, const double* R, const double* X, double* K) {
  RicStage<n, m> st;
  riccati_factor<n, m>(X, B, R, st);
  riccati_gain<n, m>(st, A, K);
  LQ_UNROLL for (int i = 0; i < m * n; ++i) K[i] = -K[i];
}

// ---- extreme eigenvalues of a k x k symmetric matrix stored (lower triangle used) in the strided workspace.
// a: k*k doubles at offset oa (row-major), d/e: k doubles each.
LQ_HD_NOINLINE void ws_tridiagonalize(const WsView& ws, int64_t oa, int64_t od, int64_t oe, int k) {
#define A_(i, j) ws[oa + (int64_t)(i)*k + (j)]
  for (int i = k - 1; i >= 1; --i) {
    const int l = i - 1;
    double h = 0.0, scale = 0.0;
    if (l > 0) {
      for (int j = 0; j <= l; ++j) scale += fabs(A_(i, j));
      if (scale == 0.0) {
        ws[oe + i] = A_(i, l);
      } else {
        for (int j = 0; j <= l; ++j) {
          const double v = A_(i, j) / scale;
          A_(i, j) = v;
          h = fma(v, v, h);
        }
        double f = A_(i, l);
        double g = (f >= 0.0) ? -sqrt(h) : sqrt(h);
        ws[oe + i] = scale * g;
        h -= f * g;
        A_(i, l) = f - g;
        f = 0.0;
        for (int j = 0; j <= l; ++j) {
          g = 0.0;
          for (int kk = 0; kk <= j; ++kk) g = fma(A_(j, kk), A_(i, kk), g);
          for (int kk = j + 1; kk <= l; ++kk) g = fma(A_(kk, j), A_(i, kk), g);
          const double ej = g / h;
          ws[oe + j] = ej;
          f = fma(ej, A_(i, j), f);
        }
        const double hh = f / (h + h);
        for (int j = 0; j <= l; ++j) {
          f = A_(i, j);
          g = ws[oe + j] - hh * f;
          ws[oe + j] = g;
          for (int kk = 0; kk <= j; ++kk) A_(j, kk) -= f * ws[oe + kk] + g * A_(i, kk);
        }
      }
    } else {
      ws[oe + i] = A_(i, l);
    }
  }
  ws[oe + 0] = 0.0;
  for (int i = 0; i < k; ++i) ws[od + i] = A_(i, i);
#undef A_
}

// number of eigenvalues of the tridiagonal (d, e) that are < x  (Sturm count)
LQ_HD int sturm_count(const WsView& ws, int64_t od, int64_t oe, int k, double x, double pivmin) {
  int cnt = 0;
  double q = ws[od] - x;
  if (fabs(q) < pivmin) q = -pivmin;
  cnt += (q < 0.0);
  for (int i = 1; i < k; ++i) {
    const double e = ws[oe + i];
    q = ws[od + i] - x - e * e / q;
    if (fabs(q) < pivmin) q = -pivmin;
    cnt += (q < 0.0);
  }
  return cnt;
}

// Smallest and largest eigenvalue of the tridiagonal (d, e) by Sturm counts. Both searches advance together and each
// pass over the matrix evaluates THREE shifts per search (quarter points: 2 bits per pass): one load of (d_i, e_i)
// feeds six independent pivot recurrences, so the workspace is streamed ~26 times instead of ~104 and the reciprocal
// chains overlap (the one-shift-per-pass version was bound by the latency of its divisions and of the strided loads).
LQ_HD_NOINLINE void ws_tridiag_extremes(const WsView& ws, int64_t od, int64_t oe, int k, double* lmin, double* lmax) {
  double gl = ws[od], gu = ws[od], emax = 0.0;
  for (int i = 0; i < k; ++i) {
    const double e0 = fabs(ws[oe + i]);
    const double e1 = (i + 1 < k) ? fabs(ws[oe + i + 1]) : 0.0;
    const double di = ws[od + i];
    gl = dmin(gl, di - e0 - e1);
    gu = dmax(gu, di + e0 + e1);
    emax = dmax(emax, e0);
  }
  const double span = dmax(fabs(gl), fabs(gu));
  gl -= 2.2e-16 * span * k + 1e-300;
  gu += 2.2e-16 * span * k + 1e-300;
  const double pivmin = dmax(1e-300, 2.3e-308 * dmax(1.0, emax * emax));
  // search 0: smallest eigenvalue = largest x with count(x) == 0   (target count 1)
  // search 1: largest eigenvalue  = smallest x with count(x) == k  (target count k)
  double lo[2] = {gl, gl}, hi[2] = {gu, gu};
  bool live[2] = {true, true};
  for (int it = 0; it < 200 && (live[0] || live[1]); ++it) {
    double x[2][3], q[2][3];
    int cnt[2][3];
    LQ_UNROLL for (int s = 0; s < 2; ++s) {
      const double w = hi[s] - lo[s];
      LQ_UNROLL for (int j = 0; j < 3; ++j) {
        x[s][j] = fma(w, 0.25 * (j + 1), lo[s]);
        double q0 = ws[od] - x[s][j];
        if (fabs(q0) < pivmin) q0 = -pivmin;
        q[s][j] = q0;
        cnt[s][j] = (q0 < 0.0);
      }
    }
    for (int i = 1; i < k; ++i) {
      const double e = ws[oe + i], di = ws[od + i];
      const double e2 = e * e;
      LQ_UNROLL for (int s = 0; s < 2; ++s)
        LQ_UNROLL for (int j = 0; j < 3; ++j) {
          double qn = fma(-e2, rcp(q[s][j]), di - x[s][j]);
          if (fabs(qn) < pivmin) qn = -pivmin;
          q[s][j] = qn;
          cnt[s][j] += (qn < 0.0);
        }
    }
    LQ_UNROLL for (int s = 0; s < 2; ++s) {
      if (!live[s]) continue;
      const int target = (s == 0) ? 1 : k;
      // counts are non-decreasing in x: the first quarter point that reaches the target bounds the eigenvalue above
      double nlo = lo[s], nhi = hi[s];
      if (cnt[s][0] >= target) nhi = x[s][0];
      else if (cnt[s][1] >= target) { nlo = x[s][0]; nhi = x[s][1]; }
      else if (cnt[s][2] >= target) { nlo = x[s][1]; nhi = x[s][2]; }
      else nlo = x[s][2];
      if (!(nlo > lo[s] || nhi < hi[s])) live[s] = false;            // the quarter points no longer separate lo / hi
      lo[s] = nlo; hi[s] = nhi;
      if (hi[s] - lo[s] <= 4.5e-16 * dmax(fabs(lo[s]), fabs(hi[s]))) live[s] = false;
    }
  }
  *lmin = 0.5 * (lo[0] + hi[0]);
  *lmax = 0.5 * (lo[1] + hi[1]);
}

template <int n, int m>
LQ_HD_NOINLINE_T GramSpectrum gram_spectrum_call(const double* Ah, const double* Bh, const double* Q, const double* R,
                                                 double minR, int N) {
  return gram_spectrum<n, m>(Ah, Bh, Q, R, minR, N);
}

template <int n, int m>
struct BoundsLayout {
  int N, k;
  int64_t oG, oC, od, oe, total;
  LQ_HD explicit BoundsLayout(int N_) : N(N_), k(N_ * m) {
    oG = 0;
    oC = oG + (int64_t)N * n * m;
    od = oC + (int64_t)k * k;
    oe = od + k;
    total = oe + k;
  }
};

// per-thread scratch of the DENSE route only (the matrix-free route needs none)
template <int n, int m>
LQ_HD int64_t bounds_ws_doubles(int N) {
  return BoundsLayout<n, m>(N).total;
}

// which route a problem takes (host and device agree through this one predicate)
LQ_HD bool bounds_matrix_free(int qr_scalar, int strict_reference, int force_dense) {
  return (qr_scalar || !strict_reference) && !force_dense;
}

struct BoundsScalars {
  int N;
  double e_A, e_B, M_V;
  double p[3];
  double V_expert;
  double bar_u, bar_d_u;   // < 0: derive from the input box
  int strict_reference;    // literal kron ordering of utils.py:317-318 (only matters when Q, R are not scalar)
  int force_dense = 0;     // take the dense Householder route even where the matrix-free one applies (A/B tests)
  const double* polyF = nullptr;   // general input polytope rows [p][m] (then bar_u / bar_d_u must be supplied), or NULL
  int polyP = 0;
};

// Everything of the bound computation that is scalar arithmetic on the norms / eigenvalue extremes the matrix part
// produced (shared by the thread-per-sample kernel below and the run-time-dimension warp route, dyn.cuh).
struct BoundsNorms {
  double fA, fB, nK;        // ||A^||_2, ||B^||_2, ||K||_2
  double eps_K;             // local_radius (utils.py:548-564)
  double rho_cl;            // rho(A^ + B^ K)
  double nPhi;              // ||Phi||_2
  double cmax, min_H;       // lambda_max(Gamma'Gamma), lambda_min(H^)
  double bu, bdu;           // max ||u||^2, max ||u1 - u2||^2 over the input set
  double nx2;               // ||x||^2
};

// Error-consistent sums of fc_ec_g_x / fc_ec_g_u (utils.py:78-117, 186-223, 296-305) over i = 0..N (bgu: i < N).
struct EcSums {
  double s_in, s_out, bgx, bgu;
};

LQ_HD EcSums ec_sums(int N, double fA, double fB, double e_A, double e_B, double nx, double bu) {
  const double eAfA = e_A + fA, eBfB = e_B + fB;
  double s_in = 0.0, s_out = 0.0, bgx = 0.0, bgu = 0.0, bgu_in = 0.0;
  for (int i = 0; i <= N; ++i) {
    const double fpi = pow(fA, (double)i);
    const double gx1 = pow(eAfA, (double)i) - fpi;
    const double gu1 = eBfB * gx1 + e_B * fpi;
    s_out += (s_in + gx1 * gx1) * (nx * nx + i * bu);
    s_in += gu1 * gu1;
    if (i >= 1) bgx += gx1;
    if (i < N) { bgu_in += gu1; bgu += bgu_in; }
  }
  EcSums r;
  r.s_in = s_in; r.s_out = s_out; r.bgx = bgx; r.bgu = bgu;
  return r;
}

// The same sums extended one horizon at a time (horizon range): each new term is computed exactly as ec_sums computes
// it (pow, not running products: (e_A + fA)^i - fA^i cancels, and running products would carry their accumulated
// rounding into the difference) and accumulated in the same order, so every horizon's sums equal ec_sums(N).
// at(N) must be called with N = N_min, N_min + 1, ...
struct EcRunning {
  double fA, fB, e_A, e_B, nx, bu;
  double s_in = 0.0, s_out = 0.0, bgx = 0.0, bgu = 0.0, bgu_in = 0.0, gu_pend = 0.0;
  int i = 0;
  bool pend = false;                     // gu_pend: the term i - 1 of bgu, owed once the horizon exceeds i - 1
  LQ_HD EcSums at(int N) {
    const double eAfA = e_A + fA, eBfB = e_B + fB;
    if (pend && i - 1 < N) { bgu_in += gu_pend; bgu += bgu_in; pend = false; }
    for (; i <= N; ++i) {
      const double fpi = pow(fA, (double)i);
      const double gx1 = pow(eAfA, (double)i) - fpi;
      const double gu1 = eBfB * gx1 + e_B * fpi;
      s_out += (s_in + gx1 * gx1) * (nx * nx + i * bu);
      s_in += gu1 * gu1;
      if (i >= 1) bgx += gx1;
      if (i < N) { bgu_in += gu1; bgu += bgu_in; } else { gu_pend = gu1; pend = true; }
    }
    EcSums r;
    r.s_in = s_in; r.s_out = s_out; r.bgx = bgx; r.bgu = bgu;
    return r;
  }
};

// es: the error-consistent sums of horizon sc.N when the caller carries them (horizon range), else computed here.
LQ_HD int bounds_formulas(double maxQ, double minQ, double maxR, double minR, const BoundsScalars& sc,
                          const BoundsNorms& q, double* out, const EcSums* es = nullptr) {
  int flags = 0;
  const int N = sc.N;
  const double fA = q.fA, fB = q.fB, nK = q.nK, eps_K = q.eps_K, rho_cl = q.rho_cl, bu = q.bu, bdu = q.bdu;
  const double ratioQ = maxQ / minQ;
  out[BF_BAR_U] = bu; out[BF_BAR_D_U] = bdu;
  out[BF_NORM_A] = fA; out[BF_NORM_B] = fB; out[BF_NORM_K] = nK;
  out[BF_EPSILON_K] = eps_K;
  out[BF_RHO_CL] = rho_cl;
  out[BF_NORM_PHI] = q.nPhi;
  const double nG = sqrt(dmax(q.cmax, 0.0));
  out[BF_NORM_GAMMA] = nG;
  const double min_H = q.min_H;
  out[BF_MIN_H] = min_H;
  const double nx2 = q.nx2;
  const double rho_K = (rho_cl + 0.4) * (rho_cl + 0.4);
  const double C_K = (1.0 + maxR * nK * nK / minQ) * dmax(1.0, ratioQ * 1.21);
  const double gam = C_K / (1.0 - rho_K);
  const double rho_g = (gam - 1.0) / gam;
  out[BF_C_K] = C_K; out[BF_RHO_K] = rho_K; out[BF_GAMMA] = gam; out[BF_RHO_GAMMA] = rho_g;
  // ---------------- ex_stability_bounds (utils.py:567-584)
  const double L_V = dmax(gam, sc.M_V / eps_K);
  const double N_0 = ceil(dmax(0.0, sc.M_V / eps_K - gam));
  out[BF_L_V] = L_V; out[BF_N_0] = N_0;
  // ---------------- fc_omega_eta (utils.py:469-523)
  const double fA2 = fA * fA;
  const double G_A = (fA == 1.0) ? (double)(N - 1) : (1.0 - pow(fA, 2.0 * (N - 1))) / (1.0 - fA2);
  const double term = 1.0 + fA2 * ratioQ;
  const double arg1 = fA2 * ratioQ * gam;
  if (!(arg1 > 0.0) || !(rho_g > 0.0)) flags |= FLAG_DOMAIN_ERROR;   // math.log raises ValueError in the reference
  const double N_min = ceil(N_0 - log(arg1) / log(rho_g));
  const double fApow = pow(fA, (double)(2 * N - 2));
  const double rg_pow = pow(rho_g, (double)N - N_0);
  const double w1 = maxQ * (term * fApow + G_A);
  const double decay = maxQ * fApow * gam * rg_pow;
  const double w05_a = maxQ * (L_V - 1.0) * G_A;
  if (w05_a < 0.0 || decay < 0.0) flags |= FLAG_DOMAIN_ERROR;        // math.sqrt domain error
  const double w05 = sqrt(w05_a) + 0.5 * term * sqrt(decay);
  const double eta = (term - 1.0) * gam * rg_pow;
  const double disc = w05 * w05 + w1 * (1.0 - eta);
  if (disc < 0.0) flags |= FLAG_DOMAIN_ERROR;
  const double err_th_r = (sqrt(disc) - w05) / w1;
  out[BF_OMEGA_N1] = w1; out[BF_OMEGA_N0D5] = w05; out[BF_ETA] = eta; out[BF_ERR_TH] = err_th_r * err_th_r;
  out[BF_N_MIN] = N_min;
  // ---------------- fc_ec_h and xi (utils.py:526-538, utils_class.py:371)
  const double h = sc.e_A * sc.e_A / minQ + sc.e_B * sc.e_B / minR;
  const double xi = h * w1 + 2.0 * sqrt(h) * w05;
  out[BF_H] = h; out[BF_XI] = xi;
  // ---------------- error-consistent sums (utils.py:78-117, 186-223, 296-305)
  const double nx = sqrt(nx2);
  const EcSums ec = es ? *es : ec_sums(N, fA, fB, sc.e_A, sc.e_B, nx, bu);
  const double s_out = ec.s_out, bgx = ec.bgx, bgu = ec.bgu;
  const double E_psi = maxQ * s_out;
  const double theta_u = maxQ * (2.0 * nG * bgu + bgu * bgu);
  const double theta_xu = maxQ * (nG * bgx + out[BF_NORM_PHI] * bgu + bgx * bgu);
  const double bar_theta = sqrt(N * bu) * theta_u + nx * theta_xu;
  const double cand = dmin(sqrt(N * bdu), bar_theta / min_H);
  const double E_u = maxR * cand * cand;
  const double E_psi_u = maxQ / maxR * (nG + bgu) * (nG + bgu) * E_u;
  out[BF_E_PSI] = E_psi; out[BF_E_U] = E_u; out[BF_E_PSI_U] = E_psi_u;
  out[BF_THETA_U] = theta_u; out[BF_THETA_X_U] = theta_xu;
  // ---------------- alpha, beta (utils_class.py:329-340), J_bound (utils_class.py:858-859)
  const double sp = sqrt(E_psi), su = sqrt(E_u), spu = sqrt(E_psi_u);
  const double p0 = sc.p[0], p1 = sc.p[1], p2 = sc.p[2];
  const double alpha = dmax(p0 * sp + p2 * spu + p0 * sp * p2 * spu, p1 * su);
  const double beta = (1.0 + p0 * sp) * ((1.0 / p2) * spu + E_psi_u) + (1.0 / p1) * su + E_u + (1.0 / p0) * sp + E_psi;
  out[BF_ALPHA] = alpha; out[BF_BETA] = beta;
  const double den = 1.0 - xi - eta;
  if (!(den > 0.0)) flags |= FLAG_BOUND_INVALID;
  out[BF_BOUND] = (alpha * sc.V_expert + beta) / den;
  return flags;
}

// Gamma[(t, r), (j, s)] for t = 0..N, j = 0..N-1 from the stored G_d = A^d B.
template <int n, int m>
LQ_HD double gamma_entry(const WsView& ws, const BoundsLayout<n, m>& L, int t, int r, int j, int s) {
  return (t > j) ? ws[L.oG + (int64_t)(t - 1 - j) * (n * m) + r * m + s] : 0.0;
}

// ---- the horizon-independent part of the per-sample bound computation: input-set constants, ||A^||, ||B^||, ||K||,
// local_radius and rho(A^ + B^ K). K is the terminal gain in the u = +Kx convention (callers pass -K_dlqr).
struct BoundsPrefix {
  double bu, bdu;           // max ||u||^2, max ||u1 - u2||^2 over the input set
  double fA, fB, nK;        // ||A^||_2, ||B^||_2, ||K||_2
  double eps_K;             // local_radius (utils.py:548-564)
  double rho_cl;            // rho(A^ + B^ K)
  int flags;
};

template <int n, int m>
LQ_HD BoundsPrefix bounds_prefix(const Problem<n, m>& pb, const double* Ah, const double* Bh, const double* K,
                                 const BoundsScalars& sc) {
  BoundsPrefix pr;
  pr.flags = 0;
  // ---------------- input-set constants (utils.py:592-650 for a box: attained at vertices)
  double bu = sc.bar_u, bdu = sc.bar_d_u;
  if (bu < 0.0) {
    bu = 0.0;
    LQ_UNROLL for (int j = 0; j < m; ++j) bu += dmax(pb.ulo[j] * pb.ulo[j], pb.uhi[j] * pb.uhi[j]);
  }
  if (bdu < 0.0) {
    bdu = 0.0;
    LQ_UNROLL for (int j = 0; j < m; ++j) bdu += (pb.uhi[j] - pb.ulo[j]) * (pb.uhi[j] - pb.ulo[j]);
  }
  pr.bu = bu;
  pr.bdu = bdu;
  // ---------------- norms
  pr.fA = norm2<n, n>(Ah); pr.fB = norm2<n, m>(Bh); pr.nK = norm2<m, n>(K);
  // ---------------- local_radius (utils.py:548-564): max_i ||(F_u K)_i||^2 in the Q^-1 metric — box rows, or the
  //                  rows of a general polytope
  double amax = 0.0;
  if (sc.polyP > 0) {
    for (int i = 0; i < sc.polyP; ++i) {
      double fk[n];
      LQ_UNROLL for (int c = 0; c < n; ++c) {
        double acc = 0.0;
        LQ_UNROLL for (int j = 0; j < m; ++j) acc = fma(sc.polyF[i * m + j], K[j * n + c], acc);
        fk[c] = acc;
      }
      amax = dmax(amax, quad<n>(fk, pb.Qinv, fk));
    }
  } else {
    LQ_UNROLL for (int j = 0; j < m; ++j) {
      const double kq = quad<n>(K + j * n, pb.Qinv, K + j * n);
      if (pb.ulo[j] > -1e300) amax = dmax(amax, kq / (pb.ulo[j] * pb.ulo[j]));
      if (pb.uhi[j] < 1e300) amax = dmax(amax, kq / (pb.uhi[j] * pb.uhi[j]));
    }
  }
  pr.eps_K = 1.0 / amax;
  // ---------------- ex_stability_lq (utils.py:343-380)
  double Acl[n * n];
  LQ_UNROLL for (int i = 0; i < n; ++i)
    LQ_UNROLL for (int j = 0; j < n; ++j) {
      double acc = Ah[i * n + j];
      LQ_UNROLL for (int r = 0; r < m; ++r) acc = fma(Bh[i * m + r], K[r * n + j], acc);
      Acl[i * n + j] = acc;
    }
  bool eig_ok;
  pr.rho_cl = spectral_radius<n>(Acl, &eig_ok);
  if (!eig_ok) pr.flags |= FLAG_EIG_NOCONV;
  return pr;
}

// ||Phi||_2 of utils.py:126-144: Phi'Phi = sum_{t=0..N} (A^t)'A^t, one term per horizon. Extending the sum from N to
// N + 1 adds the next term to the same accumulator, so every horizon of a range gets the single-horizon value exactly.
template <int n>
struct PhiGram {
  double Mt[n * n], acc[n * n];
  int t;
  LQ_HD PhiGram() : t(0) {
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = 0; j < n; ++j) { Mt[i * n + j] = (i == j) ? 1.0 : 0.0; acc[i * n + j] = Mt[i * n + j]; }
  }
  LQ_HD void extend_to(const double* Ah, int N) {
    for (; t < N; ++t) {
      double Mn[n * n];
      mm<n, n, n>(Ah, Mt, Mn);
      LQ_UNROLL for (int i = 0; i < n * n; ++i) Mt[i] = Mn[i];
      sym_add_mtm<n, n>(acc, Mt, Mt, Mn);
      LQ_UNROLL for (int i = 0; i < n * n; ++i) acc[i] = Mn[i];
    }
  }
  LQ_HD double norm() const {
    double lo, hi;
    sym_eig_minmax<n>(acc, &lo, &hi);
    return sqrt(dmax(hi, 0.0));
  }
};

// running error-consistent sums of one sample (horizon range): the constants of bounds_formulas
template <int n>
LQ_HD EcRunning ec_running(const BoundsPrefix& pr, const BoundsScalars& sc, const double* x) {
  EcRunning r;
  double nx2 = 0.0;
  LQ_UNROLL for (int i = 0; i < n; ++i) nx2 = fma(x[i], x[i], nx2);
  r.fA = pr.fA; r.fB = pr.fB; r.e_A = sc.e_A; r.e_B = sc.e_B; r.nx = sqrt(nx2); r.bu = pr.bu;
  return r;
}

// ---- the per-horizon part: the scalar formulas on the prefix, ||Phi|| and the two Gram-spectrum extremes of horizon
// sc.N. out[BF_COUNT] receives every intermediate the reference's helper functions return.
template <int n, int m>
LQ_HD int bounds_horizon(const Problem<n, m>& pb, const BoundsPrefix& pr, double nPhi, double cmax, double min_H,
                         const double* x, const BoundsScalars& sc, double* out, const EcSums* es = nullptr) {
  BoundsNorms q;
  q.fA = pr.fA; q.fB = pr.fB; q.nK = pr.nK; q.eps_K = pr.eps_K; q.rho_cl = pr.rho_cl; q.nPhi = nPhi; q.cmax = cmax;
  q.min_H = min_H;
  q.bu = pr.bu; q.bdu = pr.bdu;
  q.nx2 = 0.0;
  LQ_UNROLL for (int i = 0; i < n; ++i) q.nx2 = fma(x[i], x[i], q.nx2);
  int flags = pr.flags | bounds_formulas(pb.maxQ, pb.minQ, pb.maxR, pb.minR, sc, q, out, es);
  LQ_UNROLL for (int i = 0; i < BF_COUNT; ++i)
    if (!(fabs(out[i]) <= 1.79e308)) flags |= FLAG_NONFINITE;
  return flags;
}

// Per-sample bound computation of one horizon: bounds_prefix + bounds_horizon with ||Gamma||, lambda_min(H^) from
// the matrix-free bisection (or the dense route).
template <int n, int m>
LQ_HD int bounds_sample(const Problem<n, m>& pb, const double* Ah, const double* Bh, const double* K,
                        const double* x, const BoundsScalars& sc, const WsView& ws, double* out) {
  const BoundsLayout<n, m> L(sc.N);
  const int N = sc.N, k = L.k;
  const bool matrix_free = bounds_matrix_free(pb.qr_scalar, sc.strict_reference, sc.force_dense);
  LQ_UNROLL for (int i = 0; i < BF_COUNT; ++i) out[i] = 0.0;
  const BoundsPrefix pr = bounds_prefix<n, m>(pb, Ah, Bh, K, sc);
  const double minR = pb.minR;
  // ---------------- G_d = A^d B (dense route), ||Phi||_2
  if (!matrix_free) {
    double Gd[n * m];
    LQ_UNROLL for (int i = 0; i < n * m; ++i) Gd[i] = Bh[i];
    for (int d = 0; d < N; ++d) {
      LQ_UNROLL for (int e = 0; e < n * m; ++e) ws[L.oG + (int64_t)d * (n * m) + e] = Gd[e];
      double Gn[n * m];
      mm<n, n, m>(Ah, Gd, Gn);
      LQ_UNROLL for (int i = 0; i < n * m; ++i) Gd[i] = Gn[i];
    }
  }
  double nPhi;
  {
    PhiGram<n> phi;
    phi.extend_to(Ah, N);
    nPhi = phi.norm();
  }
  double cmin = 0.0, cmax = 0.0, min_H;
  if (matrix_free) {
    // ---------------- matrix-free: bisection on the N-stage elimination (gramspec.cuh); Q, R enter stage-wise
    // (n >= 5: a separate, non-inlined function — inlined into this body the register allocator gave up at n = 8)
    const GramSpectrum gs = (n <= 4) ? gram_spectrum<n, m>(Ah, Bh, pb.Q, pb.R, minR, N)
                                     : gram_spectrum_call<n, m>(Ah, Bh, pb.Q, pb.R, minR, N);
    cmax = gs.cmax;
    min_H = gs.min_H;
  } else {
  // ---------------- dense: Gamma'Gamma by the block recurrence C[j][j'] = C[j+1][j'+1] + G_{N-1-j}' G_{N-1-j'}
  for (int j = N - 1; j >= 0; --j)
    for (int jp = j; jp >= 0; --jp) {
      double ga[n * m], gb[n * m];
      LQ_UNROLL for (int e = 0; e < n * m; ++e) {
        ga[e] = ws[L.oG + (int64_t)(N - 1 - j) * (n * m) + e];
        gb[e] = ws[L.oG + (int64_t)(N - 1 - jp) * (n * m) + e];
      }
      LQ_UNROLL for (int a = 0; a < m; ++a)
        LQ_UNROLL for (int b = 0; b < m; ++b) {
          double acc = (j + 1 < N) ? ws[L.oC + (int64_t)((j + 1) * m + a) * k + ((jp + 1) * m + b)] : 0.0;
          LQ_UNROLL for (int r = 0; r < n; ++r) acc = fma(ga[r * m + a], gb[r * m + b], acc);
          ws[L.oC + (int64_t)(j * m + a) * k + (jp * m + b)] = acc;
          if (j == jp) ws[L.oC + (int64_t)(jp * m + b) * k + (j * m + a)] = acc;
        }
    }
  ws_tridiagonalize(ws, L.oC, L.od, L.oe, k);
  ws_tridiag_extremes(ws, L.od, L.oe, k, &cmin, &cmax);
  if (pb.qr_scalar) {
    min_H = pb.R[0] + pb.Q[0] * cmin;
  } else {
    // general weights: H^ = barR + Gamma' barQ Gamma with the literal kron(Q, I_{N+1}), kron(R, I_N) of
    // utils.py:317-318 (strict_reference) or the time-major block-diagonal weights
    for (int c = 0; c < k; ++c)
      for (int d = 0; d <= c; ++d) {
        double acc;
        if (sc.strict_reference) acc = ((c % N) == (d % N)) ? pb.R[(c / N) * m + (d / N)] : 0.0;
        else acc = ((c / m) == (d / m)) ? pb.R[(c % m) * m + (d % m)] : 0.0;
        const int jc = c / m, sc_ = c % m, jd = d / m, sd = d % m;
        const int rows = (N + 1) * n;
        for (int a = 0; a < rows; ++a) {
          const int ta = a / n, ra = a % n;
          const double gac = gamma_entry<n, m>(ws, L, ta, ra, jc, sc_);
          if (gac != 0.0) {
            double inner = 0.0;
            if (sc.strict_reference) {
              const int ia = a / (N + 1), sa = a % (N + 1);
              for (int jb = 0; jb < n; ++jb) {
                const int b = jb * (N + 1) + sa;
                inner = fma(pb.Q[ia * n + jb], gamma_entry<n, m>(ws, L, b / n, b % n, jd, sd), inner);
              }
            } else {
              for (int jb = 0; jb < n; ++jb)
                inner = fma(pb.Q[ra * n + jb], gamma_entry<n, m>(ws, L, ta, jb, jd, sd), inner);
            }
            acc = fma(gac, inner, acc);
          }
        }
        ws[L.oC + (int64_t)c * k + d] = acc;
      }
    double hmax;
    ws_tridiagonalize(ws, L.oC, L.od, L.oe, k);
    ws_tridiag_extremes(ws, L.od, L.oe, k, &min_H, &hmax);
  }
  }
  // ---------------- scalar formulas (shared with the run-time-dimension route)
  return bounds_horizon<n, m>(pb, pr, nPhi, cmax, min_H, x, sc, out);
}

}  // namespace lq
