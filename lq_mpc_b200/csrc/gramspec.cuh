// gramspec.cuh — extreme eigenvalues of the horizon-N Gram operators WITHOUT forming them (matrix-free, O(N n^3) per probe).
//
// energy_bound needs ||Gamma||_2 = sqrt(lambda_max(Gamma'Gamma)) and lambda_min(H^), H^ = barR + Gamma' barQ Gamma
// (reference utils.py:248-258: np.linalg.norm(Gamma, 2); utils.py:316-322: np.min(np.linalg.eigvals(hatH))) where
// Gamma (utils.py:145-174) is the block lower-triangular Toeplitz map from the stacked inputs u_0..u_{N-1} to the
// stacked states x_0..x_N of x+ = A x + B u, x_0 = 0. Both matrices are (N m) x (N m); round 1 assembled the Gram
// matrix and reduced it by Householder reflections ((N m)^3 flops, (N m)^2 doubles of scratch per sample).
//
// Gamma is a SIMULATION OPERATOR, so the quadratic form it induces is an N-stage LQ cost,
//     u' (barR - x I + Gamma' barQ Gamma) u  =  sum_t  x_t' Q x_t + u_t' (R - x I) u_t ,   x_{t+1} = A x_t + B u_t, x_0 = 0,
// and dynamic programming from the last stage eliminates u_{N-1}, ..., u_0 one block at a time:
//     G_s = (R - x I) + B' P B,     P <- Q + A' (P - P B G_s^-1 B' P) A,     P_0 = Q        (s = 1..N)
// This IS the block LDL' factorisation of the (N m) x (N m) matrix in that elimination order (Sylvester: its inertia is
// the sum of the inertias of the G_s). Hence
//     H^ - x I  positive definite   <=>   every G_s is positive definite              (lambda_min(H^) > x)
//     x I - Gamma'Gamma  pos. def.  <=>   every G'_s = x I - B' P B is pos. def. with P <- I + A'(P + P B G'_s^-1 B' P) A
// Each probe is a Cholesky factorisation in disguise: when every pivot is positive the computed factors are the exact
// factors of a matrix within a few ulps ||.|| of the probed one, so the yes/no answer is reliable down to the same
// backward error LAPACK's eigvals has on the assembled matrix. The two extremes are located by bisection on these
// one-sided predicates: ~52 probes x N stages x O(n^3) flops, all in registers, no scratch memory, one sample per
// thread with two independent recursions (the two searches) interleaved for instruction-level parallelism.
// General (non-scalar) weights in the time-major convention cost nothing extra: Q and R simply enter the recursion.
// (The literal kron(Q, I) ordering of utils.py:317-318 with non-scalar Q is NOT a stage-wise cost; it stays on the
// dense path of bounds.cuh.)
#pragma once
#include "riccati.cuh"

namespace lq {

// Square-root-free factorisation test of a small symmetric matrix: G = L D L' (unit lower L left below the diagonal),
// reciprocals of the pivots in dinv (MUFU.RCP64H + 2 Newton steps instead of the ~30-instruction FP64 rsqrt of a
// Cholesky: ncu showed 8 % of the kernel's instructions there). Returns "every pivot is positive" (a positive normal
// number: a denormal pivot counts as zero); a non-positive or NaN pivot is replaced by 1 so that nothing downstream overflows (the probe has failed anyway).
template <int m>
LQ_HD bool ldl_pos(double* G, double* dinv) {
  bool ok = true;
  double dv[m];
  LQ_UNROLL for (int j = 0; j < m; ++j) {
    double w[m];
    double d = G[j * m + j];
    LQ_UNROLL for (int k = 0; k < j; ++k) {
      w[k] = G[j * m + k] * dv[k];
      d = fma(-G[j * m + k], w[k], d);
    }
    const bool pos = is_pos_normal(d);           // integer pipe: the probes are FP64-pipe bound
    ok = ok && pos;
    d = pos ? d : 1.0;
    dv[j] = d;
    dinv[j] = rcp(d);
    LQ_UNROLL for (int i = j + 1; i < m; ++i) {
      double s = G[i * m + j];
      LQ_UNROLL for (int k = 0; k < j; ++k) s = fma(-G[i * m + k], w[k], s);
      G[i * m + j] = s * dinv[j];
    }
  }
  return ok;
}

// One elimination stage. G = Rd + sigma B'PB (Rd already carries the shift), positivity test, and unless `last`
// P <- Qw + A' (P - sigma (P B) G^-1 (P B)') A. Returns "G is positive definite".
template <int n, int m>
LQ_HD bool gs_stage(const double* Ah, const double* Bh, const double* Qw, const double* Rd, double sigma, bool last,
                    double* P) {
  double Y[n * m], L[m * m], Di[m];
  mm<n, n, m>(P, Bh, Y);
  LQ_UNROLL for (int i = 0; i < m; ++i)
    LQ_UNROLL for (int j = 0; j <= i; ++j) {
      double acc = 0.0;
      LQ_UNROLL for (int k = 0; k < n; ++k) acc = fma(Bh[k * m + i], Y[k * m + j], acc);
      L[i * m + j] = fma(sigma, acc, Rd[i * m + j]);
    }
  const bool ok = ldl_pos<m>(L, Di);
  if (last) return ok;
  // Z = P B L^-T (unit triangular: no divisions), then P - sigma Z D^-1 Z'
  LQ_UNROLL for (int i = 0; i < n; ++i)
    LQ_UNROLL for (int j = 1; j < m; ++j) {
      double s = Y[i * m + j];
      LQ_UNROLL for (int k = 0; k < j; ++k) s = fma(-Y[i * m + k], L[j * m + k], s);
      Y[i * m + j] = s;
    }
  double Mx[n * n], MA[n * n];
  LQ_UNROLL for (int i = 0; i < n; ++i) {
    double yd[m];
    LQ_UNROLL for (int k = 0; k < m; ++k) yd[k] = Y[i * m + k] * Di[k];
    LQ_UNROLL for (int j = i; j < n; ++j) {
      double acc = 0.0;
      LQ_UNROLL for (int k = 0; k < m; ++k) acc = fma(yd[k], Y[j * m + k], acc);
      const double v = fma(-sigma, acc, P[i * n + j]);
      Mx[i * n + j] = v;
      Mx[j * n + i] = v;
    }
  }
  mm<n, n, n>(Mx, Ah, MA);
  sym_add_mtm<n, n>(Qw, Ah, MA, P);
  return ok;
}

// n = 2 (the shipped example and every sweep of the reference): the congruence P -> A' P A acts on the three unique
// entries (p00, p01, p11) of a symmetric 2 x 2 matrix as ONE 3 x 3 map that depends on A^ only,
//     M3 = [ a^2, 2ac, c^2 ; ab, ad + bc, cd ; b^2, 2bd, d^2 ],   A^ = [a b; c d],
// formed once per sample: 9 FMAs per stage instead of the 14 of the two 2 x 2 products (the stage drops from ~35 to
// ~28 FP64 instructions at m = 1; the probes are FP64-pipe bound). Same elimination as gs_stage; P is read and written
// through its full 2 x 2 storage so that callers do not change.
LQ_HD void gs_congruence2(const double* Ah, double* M3) {
  const double a = Ah[0], b = Ah[1], c = Ah[2], d = Ah[3];
  M3[0] = a * a; M3[1] = 2.0 * a * c; M3[2] = c * c;
  M3[3] = a * b; M3[4] = fma(a, d, b * c); M3[5] = c * d;
  M3[6] = b * b; M3[7] = 2.0 * b * d; M3[8] = d * d;
}

template <int m, bool LAST>
LQ_HD bool gs_stage2(const double* M3, const double* Bh, const double* Qw, const double* Rd, double sigma, double* P) {
  constexpr int n = 2;
  double Y[n * m], L[m * m], Di[m];
  LQ_UNROLL for (int j = 0; j < m; ++j) {
    Y[j] = fma(P[1], Bh[m + j], P[0] * Bh[j]);
    Y[m + j] = fma(P[3], Bh[m + j], P[1] * Bh[j]);
  }
  LQ_UNROLL for (int i = 0; i < m; ++i)
    LQ_UNROLL for (int j = 0; j <= i; ++j) {
      const double acc = fma(Bh[m + i], Y[m + j], Bh[i] * Y[j]);
      L[i * m + j] = fma(sigma, acc, Rd[i * m + j]);
    }
  const bool ok = ldl_pos<m>(L, Di);
  if (LAST) return ok;                     // the last stage only decides its pivot (compile-time: the loop is peeled)
  LQ_UNROLL for (int i = 0; i < n; ++i)
    LQ_UNROLL for (int j = 1; j < m; ++j) {
      double sacc = Y[i * m + j];
      LQ_UNROLL for (int k = 0; k < j; ++k) sacc = fma(-Y[i * m + k], L[j * m + k], sacc);
      Y[i * m + j] = sacc;
    }
  double p0 = P[0], p1 = P[1], p2 = P[3];
  LQ_UNROLL for (int k = 0; k < m; ++k) {
    const double w0 = sigma * (Y[k] * Di[k]), w1 = sigma * (Y[m + k] * Di[k]);
    p0 = fma(-w0, Y[k], p0);
    p1 = fma(-w0, Y[m + k], p1);
    p2 = fma(-w1, Y[m + k], p2);
  }
  const double t0 = fma(M3[2], p2, fma(M3[1], p1, fma(M3[0], p0, Qw[0])));
  const double t1 = fma(M3[5], p2, fma(M3[4], p1, fma(M3[3], p0, Qw[1])));
  const double t2 = fma(M3[8], p2, fma(M3[7], p1, fma(M3[6], p0, Qw[3])));
  P[0] = t0; P[1] = t1; P[2] = t1; P[3] = t2;
  return ok;
}

// Relative width at which a bisection stops: 2^-42. The spectrum enters alpha / beta / J_bound, which are compared at
// 1e-9 (north_star); 2.3e-13 leaves three orders of margin and saves a fifth of the probes of a full-precision search.
constexpr double kGramSpectrumTol = 2.2737367544323206e-13;

struct GramSpectrum {
  double min_H;    // lambda_min(barR + Gamma' barQ Gamma), time-major weights (== R[0] + Q[0] lambda_min(Gamma'Gamma) for scalar weights)
  double cmax;     // lambda_max(Gamma'Gamma)
  int probes;      // bisection passes used (diagnostics)
};

// Both extremes for the estimated model (Ah, Bh) and horizon N. Q, R: stage weights (R positive definite, Q >= 0);
// minR = lambda_min(R).
template <int n, int m>
LQ_HD GramSpectrum gram_spectrum(const double* Ah, const double* Bh, const double* Q, const double* R, double minR,
                                 int N) {
  double eye[n * n];
  LQ_UNROLL for (int i = 0; i < n; ++i)
    LQ_UNROLL for (int j = 0; j < n; ++j) eye[i * n + j] = (i == j) ? 1.0 : 0.0;
  // ---- brackets. lambda_max(Gamma'Gamma): Rayleigh quotients of the unit inputs at stage 0 from below, the l1 bound
  //      on a Toeplitz operator norm (sum of the impulse-response norms) from above.
  double colsq[m], sumF = 0.0;
  LQ_UNROLL for (int j = 0; j < m; ++j) colsq[j] = 0.0;
  {
    double Gd[n * m];
    LQ_UNROLL for (int e = 0; e < n * m; ++e) Gd[e] = Bh[e];
    for (int d = 0; d < N; ++d) {
      double fro = 0.0;
      LQ_UNROLL for (int r = 0; r < n; ++r)
        LQ_UNROLL for (int j = 0; j < m; ++j) {
          const double g = Gd[r * m + j];
          colsq[j] = fma(g, g, colsq[j]);
          fro = fma(g, g, fro);
        }
      sumF += sqrt(fro);
      double Gn[n * m];
      mm<n, n, m>(Ah, Gd, Gn);
      LQ_UNROLL for (int e = 0; e < n * m; ++e) Gd[e] = Gn[e];
    }
  }
  double loC = 0.0;
  LQ_UNROLL for (int j = 0; j < m; ++j) loC = dmax(loC, colsq[j]);
  loC *= (1.0 - 1e-14);
  double hiC = sumF * sumF * (1.0 + 1e-14);
  // lambda_min(H^): H^ >= barR from below; the Rayleigh quotient of a unit input at the LAST stage (it only moves x_N)
  // from above: min_j (R + B'QB)_jj.
  double loH = minR * (1.0 - 1e-15), hiH = HUGE_VAL;
  {
    double QB[n * m];
    mm<n, n, m>(Q, Bh, QB);
    LQ_UNROLL for (int j = 0; j < m; ++j) {
      double acc = R[j * m + j];
      LQ_UNROLL for (int k = 0; k < n; ++k) acc = fma(Bh[k * m + j], QB[k * m + j], acc);
      hiH = dmin(hiH, acc);
    }
    hiH *= (1.0 + 1e-14);
  }
  GramSpectrum out;
  bool liveH = (hiH > loH), liveC = (hiC > loC) && (hiC == hiC) && (hiC < 1.7e308);
  if (!(hiC == hiC) || !(hiC < 1.7e308)) { loC = hiC = sumF * sumF; }      // overflow / NaN operands: propagate
  // Plain bisection on the two predicates. (Safeguarded regula falsi on the last pivot — a smooth monotone function
  // of the shift whose zero is the eigenvalue — was measured on the host harness: 14-32 probes per sample on average
  // instead of 43, but its slow tail, samples whose next pole sits within ~1e-6 of the root, puts the MAXIMUM over the
  // 32 samples of a warp at 33-48 probes: no gain in SIMT, so the simpler search stays.)
  double M3[9];
  if (n == 2) gs_congruence2(Ah, M3);
  int pass = 0;
  for (; pass < 128 && (liveH || liveC); ++pass) {
    const double xH = 0.5 * (loH + hiH), xC = 0.5 * (loC + hiC);
    double RdH[m * m], RdC[m * m], PH[n * n], PC[n * n];
    LQ_UNROLL for (int i = 0; i < m; ++i)
      LQ_UNROLL for (int j = 0; j < m; ++j) {
        RdH[i * m + j] = R[i * m + j] - ((i == j) ? xH : 0.0);
        RdC[i * m + j] = (i == j) ? xC : 0.0;
      }
    LQ_UNROLL for (int e = 0; e < n * n; ++e) { PH[e] = Q[e]; PC[e] = eye[e]; }
    bool okH = true, okC = true;
    if (n == 2) {                         // as below, with the 3 x 3 congruence map
      for (int s = 1; s < N; ++s) {
        okH = gs_stage2<m, false>(M3, Bh, Q, RdH, 1.0, PH) && okH;
        okC = gs_stage2<m, false>(M3, Bh, eye, RdC, -1.0, PC) && okC;
        if (!okH && !okC) break;
      }
      if (okH || okC) {                   // stage N (peeled): pivots only
        okH = gs_stage2<m, true>(M3, Bh, Q, RdH, 1.0, PH) && okH;
        okC = gs_stage2<m, true>(M3, Bh, eye, RdC, -1.0, PC) && okC;
      }
    } else if (n <= 4) {                  // two independent recursions interleaved: instruction-level parallelism
      for (int s = 1; s <= N; ++s) {
        const bool last = (s == N);
        okH = gs_stage<n, m>(Ah, Bh, Q, RdH, 1.0, last, PH) && okH;
        okC = gs_stage<n, m>(Ah, Bh, eye, RdC, -1.0, last, PC) && okC;
        if (!okH && !okC) break;          // both probes already decided
      }
    } else {                              // n >= 5: one recursion at a time (an n x n block is 2 n^2 registers)
      for (int s = 1; s <= N && okH; ++s) okH = gs_stage<n, m>(Ah, Bh, Q, RdH, 1.0, s == N, PH);
      for (int s = 1; s <= N && okC; ++s) okC = gs_stage<n, m>(Ah, Bh, eye, RdC, -1.0, s == N, PC);
    }
    if (liveH) {
      if (okH) loH = xH; else hiH = xH;
      const double mid = 0.5 * (loH + hiH);
      liveH = (hiH - loH > kGramSpectrumTol * hiH) && (mid > loH) && (mid < hiH);
    }
    if (liveC) {
      if (okC) hiC = xC; else loC = xC;
      const double mid = 0.5 * (loC + hiC);
      liveC = (hiC - loC > kGramSpectrumTol * hiC) && (mid > loC) && (mid < hiC);
    }
  }
  out.min_H = 0.5 * (loH + hiH);
  out.cmax = 0.5 * (loC + hiC);
  out.probes = pass;
  return out;
}

// Stopping rule of the bisections: the bracket is narrower than kGramSpectrumTol relative, or its midpoint no longer
// separates the ends.
LQ_HD bool gs_live(double lo, double hi) {
  const double mid = 0.5 * (lo + hi);
  return (hi - lo > kGramSpectrumTol * hi) && (mid > lo) && (mid < hi);
}

// Both extremes for every horizon N_min..N_max; emit(N, GramSpectrum) is called for each N in increasing order, with
// `probes` = the bisection passes spent on that horizon. Returns the elimination stages run in total.
//
// The elimination runs from the last stage (PH starts at Q, PC at I), so the pivot at s stages to go is the same for
// every horizon: "H^_N - x I > 0" iff G_1..G_N(x) are positive, and likewise for x I - Gamma_N'Gamma_N. Hence
//   * a probe that runs one stage beyond N also answers the predicate of horizon N + 1 — bit for bit the probe a
//     search of horizon N + 1 would make at that shift — and the probes of horizon N leave N + 1 a bracket;
//   * lambda_min(H^_N) is non-increasing and lambda_max(Gamma_N'Gamma_N) non-decreasing in N: the fail side of
//     horizon N (a shift whose pivots fail within N stages) is a fail side of N + 1;
//   * a horizon whose inherited bracket is already converged spends one probe at its pass side, which certifies that
//     side for N + 1 (where the extremes have converged in N, every later horizon costs this one probe);
//   * otherwise the first two probes certify a guess: the extreme extrapolated from the previous horizons (a polynomial
//     in N for lambda_min(H^), which settles to a limit; through the ratio of successive values for
//     lambda_max(Gamma'Gamma), which grows like rho(A^)^2N when A^ is unstable; second order from three horizons,
//     first order from two), +- a relative margin of twice the previous extrapolation error (2^-40 .. 2^-6). Both probes
//     inside the bracket shrink it to twice the margin; a miss still moves one end.
// Each horizon then bisects with the one-sided predicates and the stopping rule of gram_spectrum. The first searched
// horizon starts from gram_spectrum's brackets, so N_min == N_max IS gram_spectrum(N_max).
// State of the range search between horizons; next() searches the next horizon. The n >= 5 kernels call it through
// the non-inlined gram_range_next_call (as gram_spectrum_call: inlined there, the register allocator gives up).
template <int n, int m>
struct GramRange {
  const double *Ah, *Bh, *Q, *R;
  int N, N_max;                                  // N: the last horizon searched (or N_min - 1)
  double colsq[m], sumF, Gd[n * m], loH0, hiH0, M3[9];
  // what the probes so far say about the NEXT horizon: H pass / fail sides, C fail / pass sides
  double nLoH, nHiH, nLoC, nHiC;
  bool inhH, inhC;
  double vH1, vH2, vH3, vC1, vC2, vC3;           // results of the previous horizons
  double errH, errC;                             // relative errors of their guesses
  int hist;                                      // consecutive searched horizons behind N (for the extrapolation)
  int stages;

  LQ_HD void init(const double* Ah_, const double* Bh_, const double* Q_, const double* R_, double minR, int N_min,
                  int N_max_) {
    Ah = Ah_; Bh = Bh_; Q = Q_; R = R_; N_max = N_max_; N = 0;
    // brackets of gram_spectrum: the impulse-response sums colsq / sumF grow by one term per horizon; the H side does
    // not depend on N
    sumF = 0.0;
    LQ_UNROLL for (int j = 0; j < m; ++j) colsq[j] = 0.0;
    LQ_UNROLL for (int e = 0; e < n * m; ++e) Gd[e] = Bh[e];
    loH0 = minR * (1.0 - 1e-15);
    hiH0 = HUGE_VAL;
    {
      double QB[n * m];
      mm<n, n, m>(Q, Bh, QB);
      LQ_UNROLL for (int j = 0; j < m; ++j) {
        double acc = R[j * m + j];
        LQ_UNROLL for (int k = 0; k < n; ++k) acc = fma(Bh[k * m + j], QB[k * m + j], acc);
        hiH0 = dmin(hiH0, acc);
      }
      hiH0 *= (1.0 + 1e-14);
    }
    if (n == 2) gs_congruence2(Ah, M3);
    nLoH = -HUGE_VAL; nHiH = HUGE_VAL; nLoC = -HUGE_VAL; nHiC = HUGE_VAL;
    inhH = inhC = false;
    vH1 = vH2 = vH3 = vC1 = vC2 = vC3 = 0.0;
    errH = errC = 0x1p-6;
    hist = 0;
    stages = 0;
    while (N + 1 < N_min) extend();
  }

  LQ_HD void extend() {                          // impulse-response term of horizon N + 1
    ++N;
    double fro = 0.0;
    LQ_UNROLL for (int r = 0; r < n; ++r)
      LQ_UNROLL for (int j = 0; j < m; ++j) {
        const double g = Gd[r * m + j];
        colsq[j] = fma(g, g, colsq[j]);
        fro = fma(g, g, fro);
      }
    sumF += sqrt(fro);
    double Gn[n * m];
    mm<n, n, m>(Ah, Gd, Gn);
    LQ_UNROLL for (int e = 0; e < n * m; ++e) Gd[e] = Gn[e];
  }

  LQ_HD GramSpectrum next() {
    extend();
    double eye[n * n];
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = 0; j < n; ++j) eye[i * n + j] = (i == j) ? 1.0 : 0.0;
    double loC = 0.0;
    LQ_UNROLL for (int j = 0; j < m; ++j) loC = dmax(loC, colsq[j]);
    loC *= (1.0 - 1e-14);
    double hiC = sumF * sumF * (1.0 + 1e-14);
    double loH = loH0, hiH = hiH0;
    bool liveH = (hiH > loH), liveC = (hiC > loC) && (hiC == hiC) && (hiC < 1.7e308);
    if (!(hiC == hiC) || !(hiC < 1.7e308)) { loC = hiC = sumF * sumF; }      // overflow / NaN operands: propagate
    const bool srchH = liveH, srchC = liveC;     // valid brackets: their probes inform horizon N + 1
    if (inhH && liveH) { loH = dmax(loH, nLoH); hiH = dmin(hiH, nHiH); liveH = gs_live(loH, hiH); }
    if (inhC && liveC) { loC = dmax(loC, nLoC); hiC = dmin(hiC, nHiC); liveC = gs_live(loC, hiC); }
    const int L = (N < N_max) ? N + 1 : N;      // probes look one stage ahead
    nLoH = -HUGE_VAL; nHiH = HUGE_VAL; nLoC = -HUGE_VAL; nHiC = HUGE_VAL;
    bool cert = !liveH && !liveC && (L > N) && (srchH || srchC);
    double gH[2] = {0.0, 0.0}, gC[2] = {0.0, 0.0}, guessH = 0.0, guessC = 0.0;
    int kH = 2, kC = 2;                          // next certification point of the guess (2: none left)
    if (hist >= 2 && liveH && vH2 > 0.0) {
      guessH = (hist >= 3) ? fma(3.0, vH1 - vH2, vH3) : 2.0 * vH1 - vH2;
      const double d = dmin(dmax(2.0 * errH, 0x1p-40), 0x1p-6);
      gH[0] = guessH * (1.0 - d); gH[1] = guessH * (1.0 + d); kH = 0;   // pass side (lo) first
    }
    if (hist >= 2 && liveC && vC2 > 0.0) {
      const double r1 = vC1 / vC2;
      guessC = vC1 * ((hist >= 3 && vC3 > 0.0) ? 2.0 * r1 - vC2 / vC3 : r1);
      const double d = dmin(dmax(2.0 * errC, 0x1p-40), 0x1p-6);
      gC[0] = guessC * (1.0 + d); gC[1] = guessC * (1.0 - d); kC = 0;   // pass side (hi) first
    }
    int pass = 0;
    for (; pass < 128 && (liveH || liveC || cert); ++pass) {
      double xH = cert ? loH : 0.5 * (loH + hiH), xC = cert ? hiC : 0.5 * (loC + hiC);
      while (kH < 2 && !(gH[kH] > loH && gH[kH] < hiH)) ++kH;
      if (kH < 2 && liveH) xH = gH[kH++];
      while (kC < 2 && !(gC[kC] > loC && gC[kC] < hiC)) ++kC;
      if (kC < 2 && liveC) xC = gC[kC++];
      double RdH[m * m], RdC[m * m], PH[n * n], PC[n * n];
      LQ_UNROLL for (int i = 0; i < m; ++i)
        LQ_UNROLL for (int j = 0; j < m; ++j) {
          RdH[i * m + j] = R[i * m + j] - ((i == j) ? xH : 0.0);
          RdC[i * m + j] = (i == j) ? xC : 0.0;
        }
      LQ_UNROLL for (int e = 0; e < n * n; ++e) { PH[e] = Q[e]; PC[e] = eye[e]; }
      bool okH = true, okC = true, hN = false, cN = false;   // ok*: pivots 1..s positive; *N: pivots 1..N positive
      if (n <= 4) {                       // the two recursions interleaved, as in gram_spectrum
        for (int s = 1; s < L; ++s) {
          if (n == 2) {
            okH = gs_stage2<m, false>(M3, Bh, Q, RdH, 1.0, PH) && okH;
            okC = gs_stage2<m, false>(M3, Bh, eye, RdC, -1.0, PC) && okC;
          } else {
            okH = gs_stage<n, m>(Ah, Bh, Q, RdH, 1.0, false, PH) && okH;
            okC = gs_stage<n, m>(Ah, Bh, eye, RdC, -1.0, false, PC) && okC;
          }
          ++stages;
          if (s == N) { hN = okH; cN = okC; }
          if (!okH && !okC) break;
        }
        if (okH || okC) {                 // stage L (peeled): pivots only
          if (n == 2) {
            okH = gs_stage2<m, true>(M3, Bh, Q, RdH, 1.0, PH) && okH;
            okC = gs_stage2<m, true>(M3, Bh, eye, RdC, -1.0, PC) && okC;
          } else {
            okH = gs_stage<n, m>(Ah, Bh, Q, RdH, 1.0, true, PH) && okH;
            okC = gs_stage<n, m>(Ah, Bh, eye, RdC, -1.0, true, PC) && okC;
          }
          ++stages;
        }
        if (L == N) { hN = okH; cN = okC; }
      } else {                            // n >= 5: one recursion at a time
        for (int s = 1; s <= L && okH; ++s) {
          okH = gs_stage<n, m>(Ah, Bh, Q, RdH, 1.0, s == L, PH);
          ++stages;
          if (s == N) hN = okH;
        }
        for (int s = 1; s <= L && okC; ++s) {
          okC = gs_stage<n, m>(Ah, Bh, eye, RdC, -1.0, s == L, PC);
          ++stages;
          if (s == N) cN = okC;
        }
      }
      if (liveH) {
        if (hN) loH = xH; else hiH = xH;
        liveH = gs_live(loH, hiH);
      }
      if (liveC) {
        if (cN) hiC = xC; else loC = xC;
        liveC = gs_live(loC, hiC);
      }
      if (L > N) {                        // pivots 1..N+1: the predicate of horizon N + 1 at these shifts
        if (srchH) { if (okH) nLoH = dmax(nLoH, xH); else nHiH = dmin(nHiH, xH); }
        if (srchC) { if (okC) nHiC = dmin(nHiC, xC); else nLoC = dmax(nLoC, xC); }
      }
      cert = false;
    }
    GramSpectrum out;
    out.min_H = 0.5 * (loH + hiH);
    out.cmax = 0.5 * (loC + hiC);
    out.probes = pass;
    // the fail sides of horizon N fail within N stages, hence for N + 1 as well
    nHiH = dmin(nHiH, hiH);
    nLoC = dmax(nLoC, loC);
    inhH = srchH;
    inhC = srchC;
    if (guessH > 0.0) errH = fabs(guessH - out.min_H) / out.min_H;
    if (guessC > 0.0) errC = fabs(guessC - out.cmax) / out.cmax;
    if (!(errH < 0x1p-6)) errH = 0x1p-6;
    if (!(errC < 0x1p-6)) errC = 0x1p-6;
    vH3 = vH2; vH2 = vH1; vH1 = out.min_H;
    vC3 = vC2; vC2 = vC1; vC1 = out.cmax;
    hist = (srchH && srchC) ? hist + 1 : 0;
    return out;
  }
};

template <int n, int m>
LQ_HD_NOINLINE_T GramSpectrum gram_range_next_call(GramRange<n, m>& g) {
  return g.next();
}

template <int n, int m, class Emit>
LQ_HD int gram_spectrum_range(const double* Ah, const double* Bh, const double* Q, const double* R, double minR,
                              int N_min, int N_max, Emit emit) {
  GramRange<n, m> g;
  g.init(Ah, Bh, Q, R, minR, N_min, N_max);
  for (int N = N_min; N <= N_max; ++N) emit(N, (n <= 4) ? g.next() : gram_range_next_call<n, m>(g));
  return g.stages;
}

}  // namespace lq
