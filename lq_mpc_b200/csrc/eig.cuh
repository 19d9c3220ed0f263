// eig.cuh — spectral radius of a small general (non-symmetric) real matrix, one matrix per thread.
//
// Replaces `np.max(np.abs(np.linalg.eigvals(A_cl)))` (reference utils.py:358 and the stability check of the
// closed loop).  Algorithm: Householder reduction to upper Hessenberg form followed by the Francis implicit
// double-shift QR iteration with deflation (the classical EISPACK "hqr" scheme), written here for tiny fixed n
// with every loop bound a compile-time constant and run-time *predicates* selecting the active window, so that
// after unrolling all indices are static and the matrix stays in registers on the device.
#pragma once
#include "small_la.cuh"

namespace lq {

// Householder reduction to upper Hessenberg form (similarity transform; eigenvalues preserved).
template <int n>
LQ_HD void hessenberg(double* a) {
  LQ_UNROLL for (int k = 0; k < n - 2; ++k) {
    double alpha = 0.0;
    LQ_UNROLL for (int i = k + 1; i < n; ++i) alpha = fma(a[i * n + k], a[i * n + k], alpha);
    double tail = alpha - a[(k + 1) * n + k] * a[(k + 1) * n + k];
    if (tail > 0.0) {  // something below the sub-diagonal to annihilate
      const double x0 = a[(k + 1) * n + k];
      const double nrm = sqrt(alpha);
      const double beta = (x0 >= 0.0) ? -nrm : nrm;
      double v[n];
      LQ_UNROLL for (int i = 0; i < n; ++i) v[i] = (i > k) ? a[i * n + k] : 0.0;
      v[k + 1] = x0 - beta;
      double vv = 0.0;
      LQ_UNROLL for (int i = k + 1; i < n; ++i) vv = fma(v[i], v[i], vv);
      const double tau = 2.0 / vv;
      // A <- (I - tau v v^T) A
      LQ_UNROLL for (int j = 0; j < n; ++j) {
        double s = 0.0;
        LQ_UNROLL for (int i = k + 1; i < n; ++i) s = fma(v[i], a[i * n + j], s);
        s *= tau;
        LQ_UNROLL for (int i = k + 1; i < n; ++i) a[i * n + j] = fma(-s, v[i], a[i * n + j]);
      }
      // A <- A (I - tau v v^T)
      LQ_UNROLL for (int i = 0; i < n; ++i) {
        double s = 0.0;
        LQ_UNROLL for (int j = k + 1; j < n; ++j) s = fma(a[i * n + j], v[j], s);
        s *= tau;
        LQ_UNROLL for (int j = k + 1; j < n; ++j) a[i * n + j] = fma(-s, v[j], a[i * n + j]);
      }
      LQ_UNROLL for (int i = k + 2; i < n; ++i) a[i * n + k] = 0.0;
    }
  }
}

// moduli of the two eigenvalues of the 2x2 block [[y, b],[c, x]] (w = b*c), max of them.
LQ_HD double block2_rho(double y, double x, double w) {
  const double p = 0.5 * (y - x);
  const double q = fma(p, p, w);
  const double z = sqrt(fabs(q));
  if (q >= 0.0) {
    const double zz = p + dsign(z, p);
    const double r1 = x + zz;
    const double r2 = (zz != 0.0) ? x - w / zz : r1;
    return dmax(fabs(r1), fabs(r2));
  }
  const double re = x + p;
  return sqrt(fma(re, re, z * z));
}

// Get/set with a run-time index over a register array, resolved by predicated selects (n is tiny).
template <int len>
LQ_HD double rget(const double* a, int idx) {
  double r = 0.0;
  LQ_UNROLL for (int i = 0; i < len; ++i) r = (i == idx) ? a[i] : r;
  return r;
}

// Spectral radius by Hessenberg + Francis QR; *ok=false if the iteration did not converge within its budget.
template <int n>
LQ_HD double spectral_radius_qr(const double* Ain, bool* ok) {
  *ok = true;
  if (n == 1) return fabs(Ain[0]);
  if (n == 2) return block2_rho(Ain[0], Ain[3], Ain[1] * Ain[2]);
  double a[n * n];
  LQ_UNROLL for (int i = 0; i < n * n; ++i) a[i] = Ain[i];
  hessenberg<n>(a);
  double anorm = 0.0;
  LQ_UNROLL for (int i = 0; i < n; ++i)
    LQ_UNROLL for (int j = 0; j < n; ++j)
      if (j >= i - 1) anorm += fabs(a[i * n + j]);
  double rho = 0.0;
  double t = 0.0;       // accumulated exceptional shifts
  int nn = n - 1;       // active block is rows/cols l..nn
  int its = 0;
  int guard = 0;
  while (nn >= 0 && guard < 150 * n) {
    ++guard;
    // ---- find the start l of the active unreduced block (small sub-diagonal test)
    int l = 0;
    LQ_UNROLL for (int i = n - 1; i >= 1; --i) {
      if (i <= nn && l == 0) {
        double s = fabs(a[(i - 1) * n + (i - 1)]) + fabs(a[i * n + i]);
        if (s == 0.0) s = anorm;
        if (fabs(a[i * n + (i - 1)]) + s == s) { a[i * n + (i - 1)] = 0.0; l = i; }
      }
    }
    // x = a[nn][nn], y = a[nn-1][nn-1], w = a[nn][nn-1]*a[nn-1][nn]
    double x = 0.0, y = 0.0, w = 0.0;
    LQ_UNROLL for (int i = 0; i < n; ++i)
      if (i == nn) {
        x = a[i * n + i];
        if (i >= 1) { y = a[(i - 1) * n + (i - 1)]; w = a[i * n + (i - 1)] * a[(i - 1) * n + i]; }
      }
    if (l == nn) {  // one real root
      rho = dmax(rho, fabs(x + t));
      nn -= 1; its = 0;
      continue;
    }
    if (l == nn - 1) {  // a 2x2 block: two roots
      rho = dmax(rho, block2_rho(y + t, x + t, w));
      nn -= 2; its = 0;
      continue;
    }
    // ---- no deflation: one Francis double-shift sweep on rows/cols l..nn  (nn - l >= 2)
    if (its >= 120) { *ok = false; break; }
    if (its == 10 || its == 20) {  // exceptional shift (EISPACK schedule)
      t += x;
      LQ_UNROLL for (int i = 0; i < n; ++i) if (i <= nn) a[i * n + i] -= x;
      double s = 0.0;
      LQ_UNROLL for (int i = 2; i < n; ++i)
        if (i == nn) s = fabs(a[i * n + (i - 1)]) + fabs(a[(i - 1) * n + (i - 2)]);
      x = y = 0.75 * s;
      w = -0.4375 * s * s;
    }
    ++its;
    // choose the start row mst of the bulge (two consecutive small sub-diagonals), scanning up from nn-2
    int mst = l;
    double p = 0.0, q = 0.0, r = 0.0;
    {
      bool done = false;
      LQ_UNROLL for (int mm = n - 3; mm >= 0; --mm) {
        if (mm <= nn - 2 && mm >= l && !done) {
          const double z = a[mm * n + mm];
          const double rr = x - z, ss = y - z;
          double pp = (rr * ss - w) / a[(mm + 1) * n + mm] + a[mm * n + (mm + 1)];
          double qq = a[(mm + 1) * n + (mm + 1)] - z - rr - ss;
          double r3 = a[(mm + 2) * n + (mm + 1)];
          const double sc = fabs(pp) + fabs(qq) + fabs(r3);
          const double isc = 1.0 / sc;
          pp *= isc; qq *= isc; r3 *= isc;
          p = pp; q = qq; r = r3; mst = mm;
          if (mm == l) {
            done = true;
          } else {
            const double u = fabs(a[mm * n + (mm - 1)]) * (fabs(qq) + fabs(r3));
            const double v = fabs(pp) * (fabs(a[(mm - 1) * n + (mm - 1)]) + fabs(z) +
                                         fabs(a[(mm + 1) * n + (mm + 1)]));
            if (u + v == v) done = true;
          }
        }
      }
    }
    LQ_UNROLL for (int i = 2; i < n; ++i)
      if (i >= mst + 2 && i <= nn) {
        a[i * n + (i - 2)] = 0.0;
        if (i >= 3 && i != mst + 2) a[i * n + (i - 3)] = 0.0;
      }
    // bulge chase
    LQ_UNROLL for (int k = 0; k < n - 1; ++k) {
      if (k >= mst && k <= nn - 1) {
        const bool last = (k == nn - 1);
        double xs = 0.0;
        if (k != mst) {
          p = a[k * n + (k - 1 < 0 ? 0 : k - 1)];
          q = a[(k + 1) * n + (k - 1 < 0 ? 0 : k - 1)];
          r = 0.0;
          if (!last && k + 2 < n) r = a[(k + 2 < n ? k + 2 : n - 1) * n + (k - 1 < 0 ? 0 : k - 1)];
          xs = fabs(p) + fabs(q) + fabs(r);
          if (xs != 0.0) { const double ixs = 1.0 / xs; p *= ixs; q *= ixs; r *= ixs; }
        }
        const double s = dsign(sqrt(p * p + q * q + r * r), p);
        if (s != 0.0) {
          if (k == mst) {
            if (l != mst && k >= 1) a[k * n + (k - 1)] = -a[k * n + (k - 1)];
          } else if (k >= 1) {
            a[k * n + (k - 1)] = -s * xs;
          }
          p += s;
          const double is = 1.0 / s, ip = 1.0 / p;
          const double hx = p * is, hy = q * is, hz = r * is;
          q *= ip; r *= ip;
          // row modification (columns k..nn)
          LQ_UNROLL for (int j = 0; j < n; ++j)
            if (j >= k && j <= nn) {
              double pp = a[k * n + j] + q * a[(k + 1) * n + j];
              if (!last && k + 2 < n) {
                pp += r * a[(k + 2 < n ? k + 2 : n - 1) * n + j];
                a[(k + 2 < n ? k + 2 : n - 1) * n + j] -= pp * hz;
              }
              a[(k + 1) * n + j] -= pp * hy;
              a[k * n + j] -= pp * hx;
            }
          // column modification (rows l..min(nn, k+3))
          LQ_UNROLL for (int i = 0; i < n; ++i)
            if (i >= l && i <= nn && i <= k + 3) {
              double pp = hx * a[i * n + k] + hy * a[i * n + (k + 1)];
              if (!last && k + 2 < n) {
                pp += hz * a[i * n + (k + 2 < n ? k + 2 : n - 1)];
                a[i * n + (k + 2 < n ? k + 2 : n - 1)] -= pp * r;
              }
              a[i * n + (k + 1)] -= pp * q;
              a[i * n + k] -= pp;
            }
        }
      }
    }
  }
  if (nn >= 0) *ok = false;
  return rho;
}

// ---------------------------------------------------------------------------------------------------------------
// Fast path for n = 3, 4: characteristic polynomial -> exact factorisation into two real quadratics.
//
// The QR iteration above costs ~13 k instructions per 4 x 4 matrix on the device (data-dependent sweeps, ~8 FP64
// divisions per reflector) — 62 % of K1 in the round-1 profile.  For n <= 4 the spectrum is available in closed
// form; what makes the closed form usable at 1e-9 parity is (i) Frobenius scaling so every coefficient is O(1),
// (ii) coefficients from 2 x 2 minors (short sums, no powers of the matrix), (iii) Ferrari's factorisation used
// only as the STARTING point of a Bairstow (Newton) refinement on the unmodified quartic, and (iv) an a-posteriori
// acceptance test: remainder of the division ~ rounding level AND |p'(lambda*)| |lambda*| (the reciprocal
// condition number of the dominant root w.r.t. the coefficients) above a threshold that keeps the estimated
// relative error of rho below ~1e-11.  Anything else falls back to the QR iteration, so the result is never
// worse than before; typical closed loops (separated eigenvalues) take the fast path.
// ---------------------------------------------------------------------------------------------------------------

// max modulus of the roots of x^2 + p x + q, and (re, im >= 0) of the root attaining it
LQ_HD double quad_rho(double p, double q, double* re, double* im, double* sq_abs_disc) {
  const double disc = fma(p, p, -4.0 * q);
  const double sd = sqrt_fast(fabs(disc));
  *sq_abs_disc = sd;
  if (disc < 0.0) {
    *re = -0.5 * p; *im = 0.5 * sd;
    return sqrt_fast(fabs(q));
  }
  const double r = -0.5 * (p + dsign(sd, p));   // larger-magnitude root (no cancellation)
  *re = r; *im = 0.0;
  return fabs(r);
}

// largest real root of z^3 + A z^2 + B z + C (closed form + Newton polish)
LQ_HD double cubic_largest_real_root(double A, double B, double C) {
  const double third = 1.0 / 3.0;
  const double A3 = A * third;
  const double P = fma(-A, A3, B);                                  // B - A^2/3
  const double Qc = fma(A3, fma(2.0 * A3, A3, -B), C);              // 2A^3/27 - AB/3 + C
  const double hq = -0.5 * Qc, tp = P * third;
  const double D = fma(hq, hq, tp * tp * tp);
  double y;
  if (D > 0.0) {
    const double sD = sqrt_fast(D);
    const double u = cbrt(hq + dsign(sD, hq));
    y = (u != 0.0) ? u - tp / u : 0.0;
  } else {
    const double t2 = -tp;                                          // >= 0 here
    const double t = sqrt_fast(t2);
    double arg = (t2 > 0.0) ? hq / (t2 * t) : 0.0;
    arg = dmin(1.0, dmax(-1.0, arg));
    y = 2.0 * t * cos(acos(arg) * third);
  }
  double z = y - A3;
  LQ_UNROLL for (int it = 0; it < 2; ++it) {
    const double g = fma(fma(z + A, z, B), z, C);
    const double dg = fma(fma(3.0, z, 2.0 * A), z, B);
    if (dg > 1e-290) {                  // at the largest real root the slope is >= 0; never step on a flat spot
      const double zn = fma(-g, rcp(dg), z);
      z = (zn == zn) ? zn : z;
    }
  }
  return z;
}

// Roots of x^4 + a x^3 + b x^2 + c x + d with all coefficients O(1) (scaled). Returns true and rho if trusted.
LQ_HD bool quartic_rho(double a, double b, double c, double d, double* rho_out) {
  // depressed quartic t^4 + p t^2 + q t + r, x = t - a/4
  const double a4 = 0.25 * a, a2 = a * a;
  const double p = fma(-0.375, a2, b);
  const double q = fma(a, fma(0.125, a2, -0.5 * b), c);
  const double r = fma(a4, fma(a4, fma(-3.0 * a4, a4, b), -c), d);   // d - ac/4 + a^2 b/16 - 3a^4/256
  // resolvent: z^3 + 2p z^2 + (p^2 - 4r) z - q^2, z = alpha^2 >= 0
  const double B3 = fma(p, p, -4.0 * r);
  double z = cubic_largest_real_root(2.0 * p, B3, -q * q);
  z = dmax(z, 0.0);
  const double alpha = sqrt_fast(z);
  double w;                                                           // w = q / alpha, stable for alpha -> 0 too
  if (z > 1e-6) w = q * rcp(alpha);
  else w = dsign(sqrt_fast(dmax(fma(z, z + 2.0 * p, B3), 0.0)), q);
  const double beta = 0.5 * (p + z - w);
  // first factor in x: x^2 + p1 x + q1
  double p1 = fma(0.5, a, alpha);
  double q1 = fma(a4, a4 + alpha, beta);
  double p2 = 0.0, q2 = 0.0, r1 = 0.0, r0 = 0.0;
  // Bairstow refinement of (p1, q1) on the original quartic; (p2, q2) is the quotient, (r1, r0) the remainder
  LQ_UNROLL for (int it = 0; it < 4; ++it) {
    p2 = a - p1;
    q2 = b - fma(p1, p2, q1);
    r1 = c - fma(p1, q2, q1 * p2);
    r0 = fma(-q1, q2, d);
    if (it == 3) break;
    const double e = p1 - p2;
    const double j11 = fma(-p1, e, q1 - q2), j12 = e, j21 = -q1 * e, j22 = q1 - q2;
    const double det = fma(j11, j22, -j12 * j21);
    if (det != 0.0) {
      const double id = rcp(det);
      const double dp = (fma(j22, r1, -j12 * r0)) * id;
      const double dq = (fma(j11, r0, -j21 * r1)) * id;
      p1 -= dp; q1 -= dq;
    }
  }
  double re1, im1, sd1, re2, im2, sd2;
  const double rho1 = quad_rho(p1, q1, &re1, &im1, &sd1);
  const double rho2 = quad_rho(p2, q2, &re2, &im2, &sd2);
  const bool first = rho1 >= rho2;
  const double rho = first ? rho1 : rho2;
  // |f'(lambda*)| = sqrt|disc_own| * |(p_other - p_own) lambda* + (q_other - q_own)|
  const double dpq = first ? (p2 - p1) : (p1 - p2), dqq = first ? (q2 - q1) : (q1 - q2);
  const double re = first ? re1 : re2, im = first ? im1 : im2, sd = first ? sd1 : sd2;
  const double gr = fma(dpq, re, dqq), gi = dpq * im;
  const double fprime = sd * sqrt_fast(fma(gr, gr, gi * gi));
  *rho_out = rho;
  const bool small_rem = (fabs(r1) + fabs(r0)) <= 2e-14;
  return small_rem && (fprime * rho >= 4e-5) && (rho == rho);
}

// Characteristic polynomial of A / fro, fro = ||A||_F: x^4 + a x^3 + b x^2 + c x + d; for n = 3 it is the cubic times
// x (d = 0), so x^3 + a x^2 + b x + c. The polynomial of A itself has the coefficients a fro, b fro^2, c fro^3, d fro^4.
struct CharPoly {
  double a, b, c, d, fro;
};

// Spectral radius from the characteristic polynomial; *cp receives that polynomial (all zero for the zero matrix).
template <int n>
LQ_HD bool spectral_radius_poly(const double* A, double* rho_out, CharPoly* cp) {
  static_assert(n == 3 || n == 4, "closed-form path is for n = 3, 4");
  double ss = 0.0;
  LQ_UNROLL for (int i = 0; i < n * n; ++i) ss = fma(A[i], A[i], ss);
  if (!(ss > 1e-280 && ss < 1e280)) {
    *rho_out = 0.0;
    cp->a = cp->b = cp->c = cp->d = cp->fro = 0.0;
    return ss == 0.0;                                   // the zero matrix; anything extreme goes to QR
  }
  const double is = rsqrt_pos(ss), fro = ss * is;
  double m[n * n];
  LQ_UNROLL for (int i = 0; i < n * n; ++i) m[i] = A[i] * is;
  double a, b, c, d;
  if (n == 3) {
    const double m01 = fma(m[0], m[4], -m[1] * m[3]);   // principal 2x2 minors
    const double m02 = fma(m[0], m[8], -m[2] * m[6]);
    const double m12 = fma(m[4], m[8], -m[5] * m[7]);
    const double c01_12 = fma(m[1], m[5], -m[2] * m[4]);  // rows 0,1 cols 1,2
    const double c01_02 = fma(m[0], m[5], -m[2] * m[3]);  // rows 0,1 cols 0,2
    const double det = fma(m[6], c01_12, fma(-m[7], c01_02, m[8] * m01));
    a = -(m[0] + m[4] + m[8]);
    b = m01 + m02 + m12;
    c = -det;
    d = 0.0;                                            // p3(x) * x: the extra root 0 never wins the max
  } else {
    // 2x2 minors of rows (0,1) and rows (2,3), column pairs 01 02 03 12 13 23
    const double* r0 = m; const double* r1 = m + n; const double* r2 = m + 2 * n; const double* r3 = m + 3 * n;
    const double u01 = fma(r0[0], r1[1], -r0[1] * r1[0]), u02 = fma(r0[0], r1[2], -r0[2] * r1[0]);
    const double u03 = fma(r0[0], r1[3], -r0[3] * r1[0]), u12 = fma(r0[1], r1[2], -r0[2] * r1[1]);
    const double u13 = fma(r0[1], r1[3], -r0[3] * r1[1]), u23 = fma(r0[2], r1[3], -r0[3] * r1[2]);
    const double v01 = fma(r2[0], r3[1], -r2[1] * r3[0]), v02 = fma(r2[0], r3[2], -r2[2] * r3[0]);
    const double v03 = fma(r2[0], r3[3], -r2[3] * r3[0]), v12 = fma(r2[1], r3[2], -r2[2] * r3[1]);
    const double v13 = fma(r2[1], r3[3], -r2[3] * r3[1]), v23 = fma(r2[2], r3[3], -r2[3] * r3[2]);
    const double det = fma(u01, v23, fma(-u02, v13, fma(u03, v12, fma(u12, v03, fma(-u13, v02, u23 * v01)))));
    const double e2 = u01 + v23 + fma(r0[0], r2[2], -r0[2] * r2[0]) + fma(r0[0], r3[3], -r0[3] * r3[0]) +
                      fma(r1[1], r2[2], -r1[2] * r2[1]) + fma(r1[1], r3[3], -r1[3] * r3[1]);
    const double e3 = fma(r2[0], u12, fma(-r2[1], u02, r2[2] * u01)) +     // {0,1,2}
                      fma(r3[0], u13, fma(-r3[1], u03, r3[3] * u01)) +     // {0,1,3}
                      fma(r0[0], v23, fma(-r0[2], v03, r0[3] * v02)) +     // {0,2,3}
                      fma(r1[1], v23, fma(-r1[2], v13, r1[3] * v12));      // {1,2,3}
    a = -(r0[0] + r1[1] + r2[2] + r3[3]);
    b = e2;
    c = -e3;
    d = det;
  }
  cp->a = a; cp->b = b; cp->c = c; cp->d = d; cp->fro = fro;
  double rho;
  const bool ok = quartic_rho(a, b, c, d, &rho);
  *rho_out = rho * fro;
  return ok;
}

template <int n>
LQ_HD bool spectral_radius_poly(const double* A, double* rho_out) {
  CharPoly cp;
  return spectral_radius_poly<n>(A, rho_out, &cp);
}

template <int n, bool kFast = (n == 3 || n == 4)>
struct RhoFast {
  static LQ_HD bool run(const double*, double*, CharPoly*) { return false; }
  static LQ_HD bool run(const double*, double*) { return false; }
};
template <int n>
struct RhoFast<n, true> {
  static LQ_HD bool run(const double* A, double* rho, CharPoly* cp) { return spectral_radius_poly<n>(A, rho, cp); }
  static LQ_HD bool run(const double* A, double* rho) { return spectral_radius_poly<n>(A, rho); }
};

// Spectral radius of a general real n x n matrix. *ok=false only if the QR fallback did not converge.
// *cp_ok = true when the closed form (n = 3, 4) was accepted; *cp then holds the characteristic polynomial it used.
template <int n>
LQ_HD double spectral_radius(const double* A, bool* ok, CharPoly* cp, bool* cp_ok) {
  double rho;
  *cp_ok = RhoFast<n>::run(A, &rho, cp);
  if (*cp_ok) {
    *ok = true;
    return rho;
  }
  return spectral_radius_qr<n>(A, ok);
}

template <int n>
LQ_HD double spectral_radius(const double* A, bool* ok) {
  CharPoly cp;
  bool cp_ok;
  return spectral_radius<n>(A, ok, &cp, &cp_ok);
}

}  // namespace lq
