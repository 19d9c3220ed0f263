// dyn.cuh — RUN-TIME DIMENSION path: one WARP per sample, every matrix in shared memory (n <= 32, m <= 8).
//
// The thread-per-sample kernels (riccati.cuh, clqr.cuh, bounds.cuh) are templates over a short list of (n, m) pairs with
// every matrix in registers; the reference's classes take ANY (n, m) (utils_class.py:23-46, 293-306). This header is
// the general route: the same algorithms — Riccati gain and closed-loop cost (K1), exact input-box QP by Riccati-
// structured active-set sweeps (K2), DARE + norms + matrix-free Gram spectrum + bound formulas (K3) — written over
// run-time sizes, a warp cooperating on one sample: lanes split the entries of each small product, the sequential
// factorisations distribute rows over lanes, scalars are replicated. It is the correctness route for sizes without a
// register-resident instantiation (slower per sample: its operands come from shared memory, 2 loads per FMA).
//
// Conventions: matrices row-major with an explicit leading dimension; n x n work matrices use ld = n | 1 (odd: column
// walks hit distinct banks). Every routine is called by ALL 32 lanes of the warp and ends with __syncwarp(), so a
// caller may read what it wrote. `lane` = threadIdx.x & 31.
#pragma once
#include "bounds.cuh"

namespace lqd {

using lq::dmax;
using lq::dmin;

struct DynPb {                      // device problem (pointers into one global buffer, see k_dyn.cu: dyn_layout)
  int n, m;
  const double *A, *B, *Q, *R, *Pt, *Pexp, *Qinv, *ulo, *uhi;
  double maxQ, minQ, maxR, minR;
  int has_bounds, qr_scalar;
};

__device__ __forceinline__ double wsum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double wmaxd(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ double wmind(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// C (r x c) = beta C0 + alpha op(A) op(B), op(A) r x kk, op(B) kk x c. C must not alias A or B (C0 may be C).
template <bool TA, bool TB>
__device__ __forceinline__ void wgemm(int lane, int r, int kk, int c, const double* A, int lda, const double* B,
                                      int ldb, double* C, int ldc, double alpha = 1.0, const double* C0 = nullptr,
                                      int ldc0 = 0, double beta = 0.0) {
  for (int e = lane; e < r * c; e += 32) {
    const int i = e / c, j = e - i * c;
    double acc = 0.0;
    for (int k = 0; k < kk; ++k) {
      const double a = TA ? A[k * lda + i] : A[i * lda + k];
      const double b = TB ? B[j * ldb + k] : B[k * ldb + j];
      acc = fma(a, b, acc);
    }
    double v = alpha * acc;
    if (C0) v = fma(beta, C0[i * ldc0 + j], v);
    C[i * ldc + j] = v;
  }
  __syncwarp();
}

__device__ __forceinline__ void wcopy(int lane, int r, int c, const double* A, int lda, double* Bm, int ldb) {
  for (int e = lane; e < r * c; e += 32) {
    const int i = e / c, j = e - i * c;
    Bm[i * ldb + j] = A[i * lda + j];
  }
  __syncwarp();
}

// P <- (P + P') / 2 (n x n)
__device__ __forceinline__ void wsymmetrize(int lane, int n, double* P, int ld) {
  for (int e = lane; e < n * n; e += 32) {
    const int i = e / n, j = e - i * n;
    if (i < j) {
      const double v = 0.5 * (P[i * ld + j] + P[j * ld + i]);
      P[i * ld + j] = v;
      P[j * ld + i] = v;
    }
  }
  __syncwarp();
}

// y (r) = M (r x c) x   [TM: y (c) = M' x with M r x c]
template <bool TM>
__device__ __forceinline__ void wgemv(int lane, int r, int c, const double* M, int ld, const double* x, double* y) {
  const int ro = TM ? c : r, ci = TM ? r : c;
  for (int i = lane; i < ro; i += 32) {
    double acc = 0.0;
    for (int j = 0; j < ci; ++j) acc = fma(TM ? M[j * ld + i] : M[i * ld + j], x[j], acc);
    y[i] = acc;
  }
  __syncwarp();
}

// x' M y (n x n)
__device__ __forceinline__ double wquad(int lane, int n, const double* x, const double* M, int ld, const double* y) {
  double part = 0.0;
  for (int i = lane; i < n; i += 32) {
    double acc = 0.0;
    for (int j = 0; j < n; ++j) acc = fma(M[i * ld + j], y[j], acc);
    part = fma(x[i], acc, part);
  }
  return wsum(part);
}

// In-place G = L D L' of a k x k symmetric matrix (k <= 32; lower triangle read): unit-lower L below the diagonal, the
// pivots on the diagonal, their reciprocals in dinv. Right-looking, lane = row. Returns "every pivot is positive and
// finite" (warp-uniform); a bad pivot is replaced by 1 so that nothing overflows. `v`: k doubles of scratch.
__device__ __forceinline__ bool wldl(int lane, int k, double* G, int ld, double* dinv, double* v) {
  bool ok = true;
  for (int j = 0; j < k; ++j) {
    double d = G[j * ld + j];
    const bool pos = (d > 0.0) && (d < 1.7e308);
    ok = ok && pos;
    d = pos ? d : 1.0;
    const double di = 1.0 / d;
    if (lane > j && lane < k) v[lane] = G[lane * ld + j];
    if (lane == 0) { G[j * ld + j] = d; dinv[j] = di; }
    __syncwarp();
    if (lane > j && lane < k) {
      const double lij = v[lane] * di;
      G[lane * ld + j] = lij;
      for (int c = j + 1; c <= lane; ++c) G[lane * ld + c] = fma(-lij, v[c], G[lane * ld + c]);
    }
    __syncwarp();
  }
  return ok;
}

// W X = Rhs for an n x n matrix (n <= 32) and c right-hand sides, Gaussian elimination with partial pivoting, lane = row.
// Both are overwritten. Returns false on a zero / non-finite pivot (warp-uniform).
__device__ __forceinline__ bool wlu_solve(int lane, int n, double* W, int ldw, double* X, int ldx, int c) {
  bool ok = true;
  for (int k = 0; k < n; ++k) {
    double best = (lane >= k && lane < n) ? fabs(W[lane * ldw + k]) : -1.0;
    int piv = lane;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int op = __shfl_xor_sync(0xffffffffu, piv, o);
      if (ob > best || (ob == best && op < piv)) { best = ob; piv = op; }
    }
    ok = ok && (best > 0.0) && (best < 1.7e308);
    if (piv != k) {
      for (int j = lane; j < n; j += 32) { const double t = W[k * ldw + j]; W[k * ldw + j] = W[piv * ldw + j]; W[piv * ldw + j] = t; }
      for (int j = lane; j < c; j += 32) { const double t = X[k * ldx + j]; X[k * ldx + j] = X[piv * ldx + j]; X[piv * ldx + j] = t; }
    }
    __syncwarp();
    const double pk = W[k * ldw + k];
    const double inv = (pk != 0.0) ? 1.0 / pk : 0.0;
    if (lane > k && lane < n) {
      const double f = W[lane * ldw + k] * inv;
      for (int j = k + 1; j < n; ++j) W[lane * ldw + j] = fma(-f, W[k * ldw + j], W[lane * ldw + j]);
      for (int j = 0; j < c; ++j) X[lane * ldx + j] = fma(-f, X[k * ldx + j], X[lane * ldx + j]);
    }
    __syncwarp();
  }
  for (int j0 = 0; j0 < c; j0 += 32) {                  // back substitution, lane = right-hand side
    const int j = j0 + lane;
    if (j < c)
      for (int i = n - 1; i >= 0; --i) {
        double s = X[i * ldx + j];
        for (int k = i + 1; k < n; ++k) s = fma(-W[i * ldw + k], X[k * ldx + j], s);
        X[i * ldx + j] = s / W[i * ldw + i];
      }
  }
  __syncwarp();
  return ok;
}

// Extreme eigenvalue of a k x k symmetric matrix S (k <= 32) by bisection on the LDL' positivity test of x I - S
// (largest) or S - x I (smallest): the dynamic route's one symmetric-eigenvalue primitive (||M||_2, lambda(Q), ...).
// `T`: k x ldt scratch, `v`: 2k doubles.
__device__ __forceinline__ double wsym_extreme(int lane, int k, const double* S, int ld, bool want_max, double* T,
                                               int ldt, double* v) {
  double glo = HUGE_VAL, ghi = -HUGE_VAL;
  for (int i = lane; i < k; i += 32) {                   // Gershgorin bracket
    double r = 0.0;
    for (int j = 0; j < k; ++j) if (j != i) r += fabs(S[i * ld + j]);
    glo = dmin(glo, S[i * ld + i] - r);
    ghi = dmax(ghi, S[i * ld + i] + r);
  }
  glo = wmind(glo);
  ghi = wmaxd(ghi);
  if (k == 1) return S[0];
  if (!(ghi - glo < 1.7e308)) return want_max ? ghi : glo;          // non-finite data: propagate
  const double span = dmax(fabs(glo), fabs(ghi));
  double lo = glo - 4e-16 * span * k - 1e-300, hi = ghi + 4e-16 * span * k + 1e-300;
  for (int it = 0; it < 120; ++it) {
    const double x = 0.5 * (lo + hi);
    if (!(x > lo) || !(x < hi)) break;
    for (int e = lane; e < k * k; e += 32) {
      const int i = e / k, j = e - i * k;
      if (j <= i) T[i * ldt + j] = want_max ? ((i == j ? x : 0.0) - S[i * ld + j]) : (S[i * ld + j] - (i == j ? x : 0.0));
    }
    __syncwarp();
    const bool pd = wldl(lane, k, T, ldt, v, v + k);
    if (want_max) { if (pd) hi = x; else lo = x; }       // x I - S > 0  <=>  x > lambda_max
    else { if (pd) lo = x; else hi = x; }                // S - x I > 0  <=>  x < lambda_min
    if (hi - lo <= 4.5e-16 * dmax(fabs(lo), fabs(hi))) break;
  }
  return 0.5 * (lo + hi);
}

// ||M||_2 of an r x c matrix (r, c <= 32): sqrt(lambda_max of the smaller Gram matrix). Gm: min(r,c)^2-sized scratch
// with leading dimension ldg, T likewise, v: 64 doubles.
__device__ __forceinline__ double wnorm2(int lane, int r, int c, const double* M, int ld, double* Gm, int ldg, double* T,
                                         double* v) {
  if (r <= c) wgemm<false, true>(lane, r, c, r, M, ld, M, ld, Gm, ldg);
  else wgemm<true, false>(lane, c, r, c, M, ld, M, ld, Gm, ldg);
  const double lm = wsym_extreme(lane, r <= c ? r : c, Gm, ldg, true, T, ldg, v);
  return sqrt(dmax(lm, 0.0));
}

__device__ __forceinline__ double rho_block2(double y, double x, double w) {
  const double p = 0.5 * (y - x);
  const double q = fma(p, p, w);
  const double z = sqrt(fabs(q));
  if (q >= 0.0) {
    const double zz = p + (p >= 0.0 ? z : -z);
    const double r1 = x + zz;
    const double r2 = (zz != 0.0) ? x - w / zz : r1;
    return fmax(fabs(r1), fabs(r2));
  }
  const double re = x + p;
  return sqrt(fma(re, re, z * z));
}

// Warp-synchronous spectral radius of the n x n matrix `a` (shared memory, leading dimension lda, DESTROYED), n <= 32:
// Householder reduction to Hessenberg form, then the Francis double-shift QR iteration with deflation (EISPACK hqr,
// eigenvalues only); lane = row / column of the reflector updates, scalars replicated, deflation and bulge-start
// searches by ballot. `v`: 32 doubles. (Same arithmetic as np.linalg.eigvals + max|.|, utils.py:358.)
__device__ double wspectral_radius(int n, double* a, int lda, double* v, bool* ok) {
  const int lane = threadIdx.x & 31;
#define A_(i, j) a[(i) * lda + (j)]
  *ok = true;
  if (n == 1) return fabs(A_(0, 0));
  for (int k = 0; k < n - 2; ++k) {
    const double xi = (lane > k && lane < n) ? A_(lane, k) : 0.0;
    const double alpha = wsum(xi * xi);
    const double x0 = __shfl_sync(0xffffffffu, xi, k + 1);
    if (alpha - x0 * x0 > 0.0) {
      const double nrm = sqrt(alpha);
      const double beta = (x0 >= 0.0) ? -nrm : nrm;
      const double vi = (lane == k + 1) ? x0 - beta : xi;
      const double tau = 2.0 / wsum(vi * vi);
      v[lane] = vi;
      __syncwarp();
      if (lane < n) {
        double sacc = 0.0;
        for (int i = k + 1; i < n; ++i) sacc = fma(v[i], A_(i, lane), sacc);
        sacc *= tau;
        for (int i = k + 1; i < n; ++i) A_(i, lane) = fma(-sacc, v[i], A_(i, lane));
      }
      __syncwarp();
      if (lane < n) {
        double sacc = 0.0;
        for (int j = k + 1; j < n; ++j) sacc = fma(A_(lane, j), v[j], sacc);
        sacc *= tau;
        for (int j = k + 1; j < n; ++j) A_(lane, j) = fma(-sacc, v[j], A_(lane, j));
      }
      __syncwarp();
      if (lane > k + 1 && lane < n) A_(lane, k) = 0.0;
      __syncwarp();
    }
  }
  double an = 0.0;
  if (lane < n)
    for (int j = (lane > 0 ? lane - 1 : 0); j < n; ++j) an += fabs(A_(lane, j));
  const double anorm = wsum(an);
  double rho = 0.0, t = 0.0;
  int nn = n - 1, its = 0, guard = 0;
  while (nn >= 0 && guard < 150 * n) {
    ++guard;
    int l = 0;
    {
      bool small = false;
      if (lane >= 1 && lane <= nn) {
        double sd = fabs(A_(lane - 1, lane - 1)) + fabs(A_(lane, lane));
        if (sd == 0.0) sd = anorm;
        small = (fabs(A_(lane, lane - 1)) + sd == sd);
      }
      const unsigned bal = __ballot_sync(0xffffffffu, small);
      if (bal) l = 31 - __clz(bal);
    }
    if (l > 0 && lane == 0) A_(l, l - 1) = 0.0;
    __syncwarp();
    double x = A_(nn, nn);
    if (l == nn) { rho = fmax(rho, fabs(x + t)); nn -= 1; its = 0; continue; }
    double y = A_(nn - 1, nn - 1);
    double w = A_(nn, nn - 1) * A_(nn - 1, nn);
    if (l == nn - 1) { rho = fmax(rho, rho_block2(y + t, x + t, w)); nn -= 2; its = 0; continue; }
    if (its >= 120) { *ok = false; break; }
    if (its == 10 || its == 20) {
      t += x;
      __syncwarp();
      if (lane <= nn) A_(lane, lane) -= x;
      __syncwarp();
      const double sd = fabs(A_(nn, nn - 1)) + fabs(A_(nn - 1, nn - 2));
      x = y = 0.75 * sd;
      w = -0.4375 * sd * sd;
    }
    ++its;
    double p = 0.0, q = 0.0, r = 0.0;
    int mst = l;
    {
      bool cand = false;
      if (lane >= l && lane <= nn - 2) {
        const int mm = lane;
        const double z = A_(mm, mm);
        const double rr = x - z, ss = y - z;
        p = (rr * ss - w) / A_(mm + 1, mm) + A_(mm, mm + 1);
        q = A_(mm + 1, mm + 1) - z - rr - ss;
        r = A_(mm + 2, mm + 1);
        const double isc = 1.0 / (fabs(p) + fabs(q) + fabs(r));
        p *= isc; q *= isc; r *= isc;
        cand = (mm == l);
        if (!cand) {
          const double u = fabs(A_(mm, mm - 1)) * (fabs(q) + fabs(r));
          const double vv = fabs(p) * (fabs(A_(mm - 1, mm - 1)) + fabs(z) + fabs(A_(mm + 1, mm + 1)));
          cand = (u + vv == vv);
        }
      }
      const unsigned bal = __ballot_sync(0xffffffffu, cand);
      mst = 31 - __clz(bal);
      p = __shfl_sync(0xffffffffu, p, mst);
      q = __shfl_sync(0xffffffffu, q, mst);
      r = __shfl_sync(0xffffffffu, r, mst);
    }
    __syncwarp();
    if (lane >= mst + 2 && lane <= nn) {
      A_(lane, lane - 2) = 0.0;
      if (lane != mst + 2) A_(lane, lane - 3) = 0.0;
    }
    __syncwarp();
    for (int k = mst; k <= nn - 1; ++k) {
      const bool last = (k == nn - 1);
      double xsc = 0.0;
      if (k != mst) {
        p = A_(k, k - 1);
        q = A_(k + 1, k - 1);
        r = last ? 0.0 : A_(k + 2, k - 1);
        xsc = fabs(p) + fabs(q) + fabs(r);
        if (xsc != 0.0) { const double ix = 1.0 / xsc; p *= ix; q *= ix; r *= ix; }
      }
      const double s2 = fma(p, p, fma(q, q, r * r));
      if (s2 == 0.0) continue;
      const double sn = sqrt(s2);
      const double sg = (p >= 0.0) ? sn : -sn;
      __syncwarp();
      if (lane == 0) {
        if (k == mst) { if (l != mst) A_(k, k - 1) = -A_(k, k - 1); }
        else A_(k, k - 1) = -sg * xsc;
      }
      p += sg;
      const double hx = p / sg, hy = q / sg, hz = r / sg;
      q /= p; r /= p;
      if (lane >= k && lane <= nn) {
        double pp = A_(k, lane) + q * A_(k + 1, lane);
        if (!last) { pp += r * A_(k + 2, lane); A_(k + 2, lane) -= pp * hz; }
        A_(k + 1, lane) -= pp * hy;
        A_(k, lane) -= pp * hx;
      }
      __syncwarp();
      const int imax = (nn < k + 3) ? nn : k + 3;
      if (lane >= l && lane <= imax) {
        double pp = hx * A_(lane, k) + hy * A_(lane, k + 1);
        if (!last) { pp += hz * A_(lane, k + 2); A_(lane, k + 2) -= pp * r; }
        A_(lane, k + 1) -= pp * q;
        A_(lane, k) -= pp;
      }
      __syncwarp();
    }
  }
  if (nn >= 0) *ok = false;
#undef A_
  return rho;
}

// ------------------------------------------------------------------------------------------------ per-warp arena
// nbig n x n work matrices (ld = n | 1) + the small operands every routine needs.
struct Arena {
  int n, m, ld;
  double* big[8];       // n x ld each
  double* Bh;           // n x m
  double* Y;            // n x m
  double* Kt;           // m x n   (gain, row-major m x n)
  double* T_mn;         // m x n   scratch
  double* G;            // m x m
  double* G2;           // m x m
  double* di;           // m
  double* x;            // n
  double* xn;           // n
  double* u;            // m (>= 8)
  double* xa;           // n
  double* xb;           // n
  double* v;            // 64 doubles scratch
  __device__ static int ld_of(int n) { return n | 1; }
  __host__ __device__ static size_t doubles(int n, int m, int nbig) {
    const int ld = n | 1;
    return (size_t)nbig * n * ld + 2 * (size_t)n * m + 2 * (size_t)m * n + 2 * (size_t)m * m + 8 + 4 * (size_t)n + 8 + 64;
  }
  __device__ void carve(double* base, int n_, int m_, int nbig) {
    n = n_; m = m_; ld = n_ | 1;
    double* p = base;
    for (int i = 0; i < 8; ++i) big[i] = nullptr;
    for (int i = 0; i < nbig; ++i) { big[i] = p; p += (size_t)n * ld; }
    Bh = p; p += n * m;
    Y = p; p += n * m;
    Kt = p; p += m * n;
    T_mn = p; p += m * n;
    G = p; p += m * m;
    G2 = p; p += m * m;
    di = p; p += 8;
    x = p; p += n;
    xn = p; p += n;
    u = p; p += 8;
    xa = p; p += n;
    xb = p; p += n;
    v = p; p += 64;
  }
};

// ------------------------------------------------------------------------------------------------ K1 pieces
// One Riccati stage on the estimated model (Ah = big[0], Bh): from the cost-to-go P (big[1]) of horizon k-1
//   Y = P Bh, G = R + Bh'Y = L D L', Z = Y L^-T;   gain K = -L^-T D^-1 Z' Ah (if want_gain, into ar.Kt);
//   P <- Q + Ah' (P - Z D^-1 Z') Ah (if update). big[2], big[3] are scratch. Returns "G positive definite".
__device__ __forceinline__ bool dyn_riccati_stage(int lane, Arena& ar, const double* Qg, const double* Rg,
                                                  bool want_gain, bool update) {
  const int n = ar.n, m = ar.m, ld = ar.ld;
  double* Ah = ar.big[0]; double* P = ar.big[1]; double* T1 = ar.big[2]; double* T2 = ar.big[3];
  wgemm<false, false>(lane, n, n, m, P, ld, ar.Bh, m, ar.Y, m);
  wgemm<true, false>(lane, m, n, m, ar.Bh, m, ar.Y, m, ar.G, m, 1.0, Rg, m, 1.0);
  const bool ok = wldl(lane, m, ar.G, m, ar.di, ar.v);
  for (int i = lane; i < n; i += 32)                       // Z = Y L^-T (unit triangular), lane = row
    for (int j = 1; j < m; ++j) {
      double s = ar.Y[i * m + j];
      for (int k = 0; k < j; ++k) s = fma(-ar.Y[i * m + k], ar.G[j * m + k], s);
      ar.Y[i * m + j] = s;
    }
  __syncwarp();
  if (want_gain) {
    wgemm<true, false>(lane, m, n, n, ar.Y, m, Ah, ld, ar.Kt, n);          // Z' Ah   (m x n)
    for (int c = lane; c < n; c += 32)                      // K = -L^-T D^-1 (.), lane = column
      for (int i = m - 1; i >= 0; --i) {
        double s = ar.Kt[i * n + c] * ar.di[i];
        for (int k = i + 1; k < m; ++k) s = fma(ar.G[k * m + i], ar.Kt[k * n + c], s);   // Kt[k] already holds -K[k]... see below
        ar.Kt[i * n + c] = -s;
      }
    // rows are negated as they are produced: K[i] = -(d_i^-1 t_i - sum_{k>i} L[k][i] K[k]) with K[k] = -stored,
    // i.e. stored_i = -(d_i^-1 t_i + sum_{k>i} L[k][i] stored_k)  — exactly the loop above
    __syncwarp();
  }
  if (update) {
    for (int e = lane; e < n * n; e += 32) {               // T1 = P - Z D^-1 Z'
      const int i = e / n, j = e - i * n;
      double acc = 0.0;
      for (int k = 0; k < m; ++k) acc = fma(ar.Y[i * m + k] * ar.di[k], ar.Y[j * m + k], acc);
      T1[i * ld + j] = P[i * ld + j] - acc;
    }
    __syncwarp();
    wgemm<false, false>(lane, n, n, n, T1, ld, Ah, ld, T2, ld);
    wgemm<true, false>(lane, n, n, n, Ah, ld, T2, ld, P, ld, 1.0, Qg, n, 1.0);
    wsymmetrize(lane, n, P, ld);
  }
  return ok;
}

// Closed-loop figures for the gain in ar.Kt on the TRUE plant: rho(A + B K), J_inf = x0' S x0 (Lyapunov doubling),
// optionally the finite-T cost of utils_class.py:261,282-283. Uses big[4..6] + big[2], big[3] as scratch; x0 in ar.x.
__device__ __forceinline__ void dyn_closed_loop(int lane, Arena& ar, const DynPb& pb, int T, double* J_inf,
                                                double* rho_out, double* J_T, int* flags) {
  const int n = ar.n, m = ar.m, ld = ar.ld;
  double* T1 = ar.big[2]; double* T2 = ar.big[3]; double* Acl = ar.big[4]; double* S = ar.big[5]; double* M = ar.big[6];
  wgemm<false, false>(lane, n, m, n, pb.B, m, ar.Kt, n, Acl, ld, 1.0, pb.A, n, 1.0);
  wgemm<false, false>(lane, m, m, n, pb.R, m, ar.Kt, n, ar.T_mn, n);
  wgemm<true, false>(lane, n, m, n, ar.Kt, n, ar.T_mn, n, S, ld, 1.0, pb.Q, n, 1.0);   // W = Q + K'RK
  wsymmetrize(lane, n, S, ld);
  wcopy(lane, n, n, Acl, ld, T1, ld);
  bool ok;
  const double rho = wspectral_radius(n, T1, ld, ar.v, &ok);
  __syncwarp();
  if (!ok) *flags |= lq::FLAG_EIG_NOCONV;
  *rho_out = rho;
  if (!(rho < 1.0)) {
    *flags |= lq::FLAG_UNSTABLE;
    *J_inf = HUGE_VAL;
  } else {
    wcopy(lane, n, n, Acl, ld, M, ld);
    bool conv = false, bad = false;
    for (int it = 0; it < 64 && !conv && !bad; ++it) {
      wgemm<false, false>(lane, n, n, n, S, ld, M, ld, T1, ld);
      wgemm<true, false>(lane, n, n, n, M, ld, T1, ld, T2, ld);
      double tmax = 0.0, smax = 0.0;
      for (int e = lane; e < n * n; e += 32) {
        const int i = e / n, j = e - i * n;
        if (i <= j) {
          const double inc = 0.5 * (T2[i * ld + j] + T2[j * ld + i]);
          const double val = S[i * ld + j] + inc;
          T1[i * ld + j] = val;                            // staged: S is still being read by other lanes' (j, i)
          tmax = dmax(tmax, fabs(inc));
          smax = dmax(smax, fabs(val));
          if (!(fabs(val) <= 1.7e308)) smax = HUGE_VAL;
        }
      }
      __syncwarp();
      for (int e = lane; e < n * n; e += 32) {
        const int i = e / n, j = e - i * n;
        if (i <= j) { S[i * ld + j] = T1[i * ld + j]; S[j * ld + i] = T1[i * ld + j]; }
      }
      __syncwarp();
      tmax = wmaxd(tmax);
      smax = wmaxd(smax);
      if (!(smax < 1.7e308) || !(tmax == tmax)) { bad = true; break; }
      if (!(tmax > 1e-18 * smax)) { conv = true; break; }
      wgemm<false, false>(lane, n, n, n, M, ld, M, ld, T1, ld);
      wcopy(lane, n, n, T1, ld, M, ld);
    }
    if (!conv) *flags |= lq::FLAG_LYAP_NOCONV;
    const double J = wquad(lane, n, ar.x, S, ld, ar.x);
    if (!(fabs(J) <= 1.79e308)) *flags |= lq::FLAG_NONFINITE;
    *J_inf = J;
  }
  if (T > 0) {                                             // finite-T cost exactly as accumulated upstream
    double* xx = ar.xa;
    double* xn = ar.xb;
    for (int i = lane; i < n; i += 32) xx[i] = ar.x[i];
    __syncwarp();
    double cost = wquad(lane, n, xx, pb.Q, n, xx);
    for (int t = 0; t < T; ++t) {
      wgemv<false>(lane, m, n, ar.Kt, n, xx, ar.u);
      for (int i = lane; i < n; i += 32) {
        double acc = 0.0;
        for (int j = 0; j < n; ++j) acc = fma(pb.A[i * n + j], xx[j], acc);
        for (int j = 0; j < m; ++j) acc = fma(pb.B[i * m + j], ar.u[j], acc);
        xn[i] = acc;
      }
      __syncwarp();
      cost += wquad(lane, n, xn, pb.Q, n, xn);
      cost += wquad(lane, m, ar.u, pb.R, m, ar.u);
      for (int i = lane; i < n; i += 32) xx[i] = xn[i];
      __syncwarp();
    }
    *J_T = cost;
  }
}

// ------------------------------------------------------------------------------------------------ K3 pieces
// Stabilising DARE solution X of (Ah = big[0], Bh) by the structure-preserving doubling algorithm (same iteration as
// lq::dare_sda). Uses big[1..7]; the result is left in big[3] (H). Returns "converged".
__device__ __forceinline__ bool dyn_dare(int lane, Arena& ar, const DynPb& pb) {
  const int n = ar.n, m = ar.m, ld = ar.ld;
  double* Ah = ar.big[0]; double* Ak = ar.big[1]; double* Gm = ar.big[2]; double* H = ar.big[3]; double* W = ar.big[4];
  double* V = ar.big[5]; double* T1 = ar.big[7];
  const int ldv = 2 * n;
  // G = B R^-1 B'
  wcopy(lane, m, m, pb.R, m, ar.G, m);
  wldl(lane, m, ar.G, m, ar.di, ar.v);
  for (int c = lane; c < n; c += 32) {                     // T_mn = R^-1 Bh'  (m x n), lane = column
    for (int i = 0; i < m; ++i) {                          // L y = b
      double sacc = ar.Bh[c * m + i];
      for (int k = 0; k < i; ++k) sacc = fma(-ar.G[i * m + k], ar.T_mn[k * n + c], sacc);
      ar.T_mn[i * n + c] = sacc;
    }
    for (int i = m - 1; i >= 0; --i) {                     // L' x = D^-1 y
      double sacc = ar.T_mn[i * n + c] * ar.di[i];
      for (int k = i + 1; k < m; ++k) sacc = fma(-ar.G[k * m + i], ar.T_mn[k * n + c], sacc);
      ar.T_mn[i * n + c] = sacc;
    }
  }
  __syncwarp();
  wgemm<false, false>(lane, n, m, n, ar.Bh, m, ar.T_mn, n, Gm, ld);
  wsymmetrize(lane, n, Gm, ld);
  wcopy(lane, n, n, Ah, ld, Ak, ld);
  wcopy(lane, n, n, pb.Q, n, H, ld);
  bool conv = false;
  for (int it = 0; it < 60 && !conv; ++it) {
    for (int e = lane; e < n * n; e += 32) {               // W = I + G H ; V = [Ak | G]
      const int i = e / n, j = e - i * n;
      double acc = (i == j) ? 1.0 : 0.0;
      for (int k = 0; k < n; ++k) acc = fma(Gm[i * ld + k], H[k * ld + j], acc);
      W[i * ld + j] = acc;
      V[i * ldv + j] = Ak[i * ld + j];
      V[i * ldv + n + j] = Gm[i * ld + j];
    }
    __syncwarp();
    if (!wlu_solve(lane, n, W, ld, V, ldv, 2 * n)) return false;
    // G+ = G + sym(Ak (W^-1 G) Ak')
    wgemm<false, false>(lane, n, n, n, Ak, ld, V + n, ldv, T1, ld);
    for (int e = lane; e < n * n; e += 32) {
      const int i = e / n, j = e - i * n;
      if (i <= j) {
        double a1 = 0.0, a2 = 0.0;
        for (int k = 0; k < n; ++k) { a1 = fma(T1[i * ld + k], Ak[j * ld + k], a1); a2 = fma(T1[j * ld + k], Ak[i * ld + k], a2); }
        const double val = Gm[i * ld + j] + 0.5 * (a1 + a2);
        Gm[i * ld + j] = val;
        Gm[j * ld + i] = val;
      }
    }
    __syncwarp();
    // H+ = H + sym(Ak' H (W^-1 Ak))
    wgemm<false, false>(lane, n, n, n, H, ld, V, ldv, T1, ld);
    double dmx = 0.0, hmx = 0.0;
    for (int e = lane; e < n * n; e += 32) {
      const int i = e / n, j = e - i * n;
      if (i <= j) {
        double a1 = 0.0, a2 = 0.0;
        for (int k = 0; k < n; ++k) { a1 = fma(Ak[k * ld + i], T1[k * ld + j], a1); a2 = fma(Ak[k * ld + j], T1[k * ld + i], a2); }
        const double inc = 0.5 * (a1 + a2);
        const double val = H[i * ld + j] + inc;
        W[i * ld + j] = val;                               // staged (H is still read by the products of other lanes)
        dmx = dmax(dmx, fabs(inc));
        hmx = dmax(hmx, fabs(val));
        if (!(inc == inc)) dmx = HUGE_VAL;
      }
    }
    __syncwarp();
    dmx = wmaxd(dmx);
    hmx = wmaxd(hmx);
    // A+ = Ak (W^-1 Ak)  (T1 is free again once H has been updated below)
    for (int e = lane; e < n * n; e += 32) {
      const int i = e / n, j = e - i * n;
      if (i <= j) { H[i * ld + j] = W[i * ld + j]; H[j * ld + i] = W[i * ld + j]; }
    }
    __syncwarp();
    wgemm<false, false>(lane, n, n, n, Ak, ld, V, ldv, T1, ld);
    wcopy(lane, n, n, T1, ld, Ak, ld);
    if (!(dmx > 1e-17 * hmx)) conv = (dmx == dmx) && (dmx < 1.7e308);
    if (!(dmx < 1.7e308)) return false;
  }
  return conv;
}

// One elimination stage of the matrix-free Gram spectrum (gramspec.cuh: gs_stage) on P = big[pi]:
// G = Rd + sigma Bh'P Bh, positivity test, P <- Qw + Ah'(P - sigma Z D^-1 Z')Ah unless `last`. Qw = pb.Q or the identity.
__device__ __forceinline__ bool dyn_gs_stage(int lane, Arena& ar, int pi, const double* Qg, bool q_identity,
                                             const double* Rg, double shift, double sigma, bool last) {
  const int n = ar.n, m = ar.m, ld = ar.ld;
  double* Ah = ar.big[0]; double* P = ar.big[pi]; double* T1 = ar.big[3]; double* T2 = ar.big[4];
  wgemm<false, false>(lane, n, n, m, P, ld, ar.Bh, m, ar.Y, m);
  for (int e = lane; e < m * m; e += 32) {
    const int i = e / m, j = e - i * m;
    double acc = 0.0;
    for (int k = 0; k < n; ++k) acc = fma(ar.Bh[k * m + i], ar.Y[k * m + j], acc);
    const double rd = (Rg ? Rg[i * m + j] : 0.0) + ((i == j) ? shift : 0.0);
    ar.G[i * m + j] = fma(sigma, acc, rd);
  }
  __syncwarp();
  const bool ok = wldl(lane, m, ar.G, m, ar.di, ar.v);
  if (last) return ok;
  for (int i = lane; i < n; i += 32)
    for (int j = 1; j < m; ++j) {
      double sacc = ar.Y[i * m + j];
      for (int k = 0; k < j; ++k) sacc = fma(-ar.Y[i * m + k], ar.G[j * m + k], sacc);
      ar.Y[i * m + j] = sacc;
    }
  __syncwarp();
  for (int e = lane; e < n * n; e += 32) {
    const int i = e / n, j = e - i * n;
    double acc = 0.0;
    for (int k = 0; k < m; ++k) acc = fma(ar.Y[i * m + k] * ar.di[k], ar.Y[j * m + k], acc);
    T1[i * ld + j] = fma(-sigma, acc, P[i * ld + j]);
  }
  __syncwarp();
  wgemm<false, false>(lane, n, n, n, T1, ld, Ah, ld, T2, ld);
  for (int e = lane; e < n * n; e += 32) {
    const int i = e / n, j = e - i * n;
    double acc = q_identity ? ((i == j) ? 1.0 : 0.0) : Qg[i * n + j];
    for (int k = 0; k < n; ++k) acc = fma(Ah[k * ld + i], T2[k * ld + j], acc);
    P[i * ld + j] = acc;
  }
  __syncwarp();
  wsymmetrize(lane, n, P, ld);
  return ok;
}

// lambda_max(Gamma'Gamma) and lambda_min(H^) by bisection on the elimination predicates (gramspec.cuh, run-time sizes).
__device__ __forceinline__ void dyn_gram_spectrum(int lane, Arena& ar, const DynPb& pb, int N, double* min_H,
                                                  double* cmax) {
  const int n = ar.n, m = ar.m, ld = ar.ld;
  double* Ah = ar.big[0];
  // brackets (see gramspec.cuh)
  double* Gd = ar.Y; double* Gn = ar.T_mn;                 // n x m each (T_mn is m x n: same size)
  wcopy(lane, n, m, ar.Bh, m, Gd, m);
  double sumF = 0.0, loC = 0.0;
  for (int j = 0; j < m; ++j) ar.u[j] = 0.0;
  __syncwarp();
  for (int d = 0; d < N; ++d) {
    double fro = 0.0;
    for (int e = lane; e < n * m; e += 32) fro = fma(Gd[e], Gd[e], fro);
    fro = wsum(fro);
    sumF += sqrt(fro);
    if (lane < m) {
      double c2 = ar.u[lane];
      for (int r = 0; r < n; ++r) c2 = fma(Gd[r * m + lane], Gd[r * m + lane], c2);
      ar.u[lane] = c2;
    }
    __syncwarp();
    wgemm<false, false>(lane, n, n, m, Ah, ld, Gd, m, Gn, m);
    wcopy(lane, n, m, Gn, m, Gd, m);
  }
  for (int j = 0; j < m; ++j) loC = dmax(loC, ar.u[j]);
  loC *= (1.0 - 1e-14);
  double hiC = sumF * sumF * (1.0 + 1e-14);
  double loH = pb.minR * (1.0 - 1e-15), hiH = HUGE_VAL;
  wgemm<false, false>(lane, n, n, m, pb.Q, n, ar.Bh, m, ar.Y, m);
  for (int j = 0; j < m; ++j) {
    double acc = pb.R[j * m + j];
    for (int k = 0; k < n; ++k) acc = fma(ar.Bh[k * m + j], ar.Y[k * m + j], acc);
    hiH = dmin(hiH, acc);
  }
  hiH *= (1.0 + 1e-14);
  __syncwarp();
  bool liveH = (hiH > loH), liveC = (hiC > loC) && (hiC < 1.7e308);
  if (!(hiC < 1.7e308)) loC = hiC = sumF * sumF;
  for (int pass = 0; pass < 128 && (liveH || liveC); ++pass) {
    if (liveH) {
      const double x = 0.5 * (loH + hiH);
      wcopy(lane, n, n, pb.Q, n, ar.big[1], ld);
      bool ok = true;
      for (int s = 1; s <= N && ok; ++s) ok = dyn_gs_stage(lane, ar, 1, pb.Q, false, pb.R, -x, 1.0, s == N) && ok;
      if (ok) loH = x; else hiH = x;
      const double mid = 0.5 * (loH + hiH);
      liveH = (hiH - loH > lq::kGramSpectrumTol * hiH) && (mid > loH) && (mid < hiH);
    }
    if (liveC) {
      const double x = 0.5 * (loC + hiC);
      for (int e = lane; e < n * n; e += 32) { const int i = e / n, j = e - i * n; ar.big[2][i * ld + j] = (i == j) ? 1.0 : 0.0; }
      __syncwarp();
      bool ok = true;
      for (int s = 1; s <= N && ok; ++s) ok = dyn_gs_stage(lane, ar, 2, nullptr, true, nullptr, x, -1.0, s == N) && ok;
      if (ok) hiC = x; else loC = x;
      const double mid = 0.5 * (loC + hiC);
      liveC = (hiC - loC > lq::kGramSpectrumTol * hiC) && (mid > loC) && (mid < hiC);
    }
  }
  *min_H = 0.5 * (loH + hiH);
  *cmax = 0.5 * (loC + hiC);
}

// Matrix part of the bound computation for the estimated model (big[0] = Ah, Bh) and the gain in ar.Kt (u = +K x);
// x (n doubles, shared memory) is the state energy_bound is evaluated at. Fills `q`; returns flag bits.
__device__ __forceinline__ int dyn_bounds_norms(int lane, Arena& ar, const DynPb& pb, int N, const double* x,
                                                double bar_u, double bar_d_u, lq::BoundsNorms& q) {
  const int n = ar.n, m = ar.m, ld = ar.ld;
  double* Ah = ar.big[0];
  int flags = 0;
  double bu = bar_u, bdu = bar_d_u;
  if (bu < 0.0) { bu = 0.0; for (int j = 0; j < m; ++j) bu += dmax(pb.ulo[j] * pb.ulo[j], pb.uhi[j] * pb.uhi[j]); }
  if (bdu < 0.0) { bdu = 0.0; for (int j = 0; j < m; ++j) bdu += (pb.uhi[j] - pb.ulo[j]) * (pb.uhi[j] - pb.ulo[j]); }
  q.bu = bu; q.bdu = bdu;
  q.fA = wnorm2(lane, n, n, Ah, ld, ar.big[2], ld, ar.big[3], ar.v);
  q.fB = wnorm2(lane, n, m, ar.Bh, m, ar.G, m, ar.G2, ar.v);
  q.nK = wnorm2(lane, m, n, ar.Kt, n, ar.G, m, ar.G2, ar.v);
  double amax = 0.0;
  for (int j = 0; j < m; ++j) {
    const double kq = wquad(lane, n, ar.Kt + j * n, pb.Qinv, n, ar.Kt + j * n);
    if (pb.ulo[j] > -1e300) amax = dmax(amax, kq / (pb.ulo[j] * pb.ulo[j]));
    if (pb.uhi[j] < 1e300) amax = dmax(amax, kq / (pb.uhi[j] * pb.uhi[j]));
  }
  q.eps_K = 1.0 / amax;
  wgemm<false, false>(lane, n, m, n, ar.Bh, m, ar.Kt, n, ar.big[2], ld, 1.0, Ah, ld, 1.0);
  bool eig_ok;
  q.rho_cl = wspectral_radius(n, ar.big[2], ld, ar.v, &eig_ok);
  __syncwarp();
  if (!eig_ok) flags |= lq::FLAG_EIG_NOCONV;
  // ||Phi||_2: lambda_max(sum_{t=0}^{N} (A^t)' A^t)
  {
    double* Mt = ar.big[2]; double* Mn = ar.big[3]; double* acc = ar.big[4];
    for (int e = lane; e < n * n; e += 32) {
      const int i = e / n, j = e - i * n;
      Mt[i * ld + j] = (i == j) ? 1.0 : 0.0;
      acc[i * ld + j] = (i == j) ? 1.0 : 0.0;
    }
    __syncwarp();
    for (int t = 1; t <= N; ++t) {
      wgemm<false, false>(lane, n, n, n, Ah, ld, Mt, ld, Mn, ld);
      wcopy(lane, n, n, Mn, ld, Mt, ld);
      wgemm<true, false>(lane, n, n, n, Mt, ld, Mt, ld, Mn, ld, 1.0, acc, ld, 1.0);
      wcopy(lane, n, n, Mn, ld, acc, ld);
    }
    wsymmetrize(lane, n, acc, ld);
    q.nPhi = sqrt(dmax(wsym_extreme(lane, n, acc, ld, true, ar.big[3], ld, ar.v), 0.0));
  }
  dyn_gram_spectrum(lane, ar, pb, N, &q.min_H, &q.cmax);
  double nx2 = 0.0;
  for (int i = 0; i < n; ++i) nx2 = fma(x[i], x[i], nx2);
  q.nx2 = nx2;
  return flags;
}

// ------------------------------------------------------------------------------------------------ K2 pieces
// Per-warp global scratch of the exact QP (the gains of N stages do not fit shared memory): contiguous per warp.
struct QpWs {
  double *Ku, *Kc, *kc, *z, *zs, *xs;
  __host__ __device__ static size_t doubles(int n, int m, int N) {
    return 2 * (size_t)N * m * n + 3 * (size_t)N * m + (size_t)(N + 1) * n;
  }
  __device__ void carve(double* p, int n, int m, int N) {
    Ku = p; p += (size_t)N * m * n;
    Kc = p; p += (size_t)N * m * n;
    kc = p; p += (size_t)N * m;
    z = p; p += (size_t)N * m;
    zs = p; p += (size_t)N * m;
    xs = p;
  }
};

// Unconstrained Riccati sweep: gains K_k of stages 0..N-1 into ws.Ku, the horizon-N cost-to-go P_0 into big[4].
__device__ __forceinline__ int dyn_plan_prepare(int lane, Arena& ar, const DynPb& pb, int N, const QpWs& ws) {
  const int n = ar.n, m = ar.m, ld = ar.ld;
  wcopy(lane, n, n, pb.Pt, n, ar.big[1], ld);
  int flags = 0;
  for (int k = N - 1; k >= 0; --k) {
    if (!dyn_riccati_stage(lane, ar, pb.Q, pb.R, true, true)) flags |= lq::FLAG_CHOL_FAIL;
    for (int e = lane; e < m * n; e += 32) ws.Ku[(size_t)k * m * n + e] = ar.Kt[e];
    __syncwarp();
  }
  wcopy(lane, n, n, ar.big[1], ld, ar.big[4], ld);
  return flags;
}

__device__ __forceinline__ void dyn_step_model(int lane, int n, int m, const double* A, int lda, const double* B,
                                               const double* x, const double* u, double* xn) {
  for (int i = lane; i < n; i += 32) {
    double acc = 0.0;
    for (int j = 0; j < n; ++j) acc = fma(A[i * lda + j], x[j], acc);
    for (int j = 0; j < m; ++j) acc = fma(B[i * m + j], u[j], acc);
    xn[i] = acc;
  }
  __syncwarp();
}

// Backward affine Riccati sweep for the working set (fixed, athi) — clqr.cuh: clqr_backward with run-time sizes.
// S lives in big[1], uses big[2], big[3], big[5] as scratch; the linear term s in ar.xa.
__device__ __forceinline__ bool dyn_clqr_backward(int lane, Arena& ar, const DynPb& pb, int N, const lq::Mask128& fixed,
                                                  const lq::Mask128& athi, const QpWs& ws, const lq::Refs& rf) {
  const int n = ar.n, m = ar.m, ld = ar.ld;
  double* Ah = ar.big[0]; double* S = ar.big[1]; double* T1 = ar.big[2]; double* T2 = ar.big[3]; double* Acl = ar.big[5];
  double* sv = ar.xa; double* tv = ar.xb;
  wcopy(lane, n, n, pb.Pt, n, S, ld);
  for (int i = lane; i < n; i += 32) {
    double acc = 0.0;
    for (int j = 0; j < n; ++j) acc = fma(-pb.Pt[i * n + j], rf.x(j, N - 1), acc);
    sv[i] = acc;
  }
  __syncwarp();
  bool ok = true;
  for (int k = N - 1; k >= 0; --k) {
    wgemm<false, false>(lane, n, n, m, S, ld, ar.Bh, m, ar.Y, m);                       // S B
    wgemm<true, false>(lane, m, n, m, ar.Bh, m, ar.Y, m, ar.G, m, 1.0, pb.R, m, 1.0);   // G = R + B'SB
    wgemm<true, false>(lane, m, n, n, ar.Y, m, Ah, ld, ar.T_mn, n);                     // Hx = B'S A   (m x n)
    // hs = B's - R u_ref_k  (m), into ar.u; the clamped constants substituted below
    if (lane < m) {
      double acc = 0.0;
      for (int r = 0; r < n; ++r) acc = fma(ar.Bh[r * m + lane], sv[r], acc);
      for (int r = 0; r < m; ++r) acc = fma(-pb.R[lane * m + r], rf.u(r, k), acc);
      ar.u[lane] = acc;
    }
    __syncwarp();
    if (lane == 0) {                                       // clamp: substitute constants for the fixed components
      for (int i = 0; i < m; ++i)
        if (!fixed.test(k * m + i))
          for (int j = 0; j < m; ++j)
            if (fixed.test(k * m + j)) {
              const double uc = athi.test(k * m + j) ? pb.uhi[j] : pb.ulo[j];
              ar.u[i] = fma(ar.G[i * m + j], uc, ar.u[i]);
            }
      for (int i = 0; i < m; ++i)
        for (int j = 0; j < m; ++j)
          if (fixed.test(k * m + i) || fixed.test(k * m + j)) ar.G[i * m + j] = (i == j) ? 1.0 : 0.0;
      for (int i = 0; i < m; ++i)
        if (fixed.test(k * m + i)) {
          const double uc = athi.test(k * m + i) ? pb.uhi[i] : pb.ulo[i];
          for (int j = 0; j < n; ++j) ar.T_mn[i * n + j] = 0.0;
          ar.u[i] = -uc;
        }
    }
    __syncwarp();
    ok = wldl(lane, m, ar.G, m, ar.di, ar.v) && ok;
    // K = -G^-1 Hx (m x n) into Kt, kv = -G^-1 hs into ar.u: forward (unit L), scale, backward, lane = column (n = hs)
    for (int c = lane; c <= n; c += 32) {
      double col[8];
      for (int i = 0; i < m; ++i) {
        double sacc = (c < n) ? ar.T_mn[i * n + c] : ar.u[i];
        for (int kk = 0; kk < i; ++kk) sacc = fma(-ar.G[i * m + kk], col[kk], sacc);
        col[i] = sacc;
      }
      for (int i = m - 1; i >= 0; --i) {
        double sacc = col[i] * ar.di[i];
        for (int kk = i + 1; kk < m; ++kk) sacc = fma(-ar.G[kk * m + i], col[kk], sacc);
        col[i] = sacc;
      }
      for (int i = 0; i < m; ++i) {                        // (column c = n is the offset: only its lane touches ar.u)
        if (c < n) ar.Kt[i * n + c] = -col[i];
        else ar.u[i] = fixed.test(k * m + i) ? (athi.test(k * m + i) ? pb.uhi[i] : pb.ulo[i]) : -col[i];
      }
    }
    __syncwarp();
    for (int e = lane; e < m * n; e += 32) ws.Kc[(size_t)k * m * n + e] = ar.Kt[e];
    if (lane < m) ws.kc[(size_t)k * m + lane] = ar.u[lane];
    __syncwarp();
    if (k > 0) {
      // S_k = Q + K'RK + Acl' S Acl ;  s_k = -Q x_ref_{k-1} + K'R(kv - u_ref_k) + Acl'(S B kv + s)
      wgemm<false, false>(lane, n, m, n, ar.Bh, m, ar.Kt, n, Acl, ld, 1.0, Ah, ld, 1.0);
      for (int i = lane; i < n; i += 32) {                 // t = S (B kv) + s = (S B) kv + s
        double acc = sv[i];
        for (int j = 0; j < m; ++j) acc = fma(ar.Y[i * m + j], ar.u[j], acc);
        tv[i] = acc;
      }
      if (lane < m) {                                      // Rk = R (kv - u_ref_k) into G2[0..m)
        double acc = 0.0;
        for (int j = 0; j < m; ++j) acc = fma(pb.R[lane * m + j], ar.u[j] - rf.u(j, k), acc);
        ar.G2[lane] = acc;
      }
      __syncwarp();
      for (int i = lane; i < n; i += 32) {
        double acc = 0.0;
        for (int r = 0; r < n; ++r) acc = fma(-pb.Q[i * n + r], rf.x(r, k - 1), acc);
        for (int r = 0; r < m; ++r) acc = fma(ar.Kt[r * n + i], ar.G2[r], acc);
        for (int r = 0; r < n; ++r) acc = fma(Acl[r * ld + i], tv[r], acc);
        ar.xn[i] = acc;
      }
      __syncwarp();
      for (int i = lane; i < n; i += 32) sv[i] = ar.xn[i];
      wgemm<false, false>(lane, n, n, n, S, ld, Acl, ld, T1, ld);                        // S Acl
      wgemm<false, false>(lane, m, m, n, pb.R, m, ar.Kt, n, ar.T_mn, n);                 // R K
      wgemm<true, false>(lane, n, m, n, ar.Kt, n, ar.T_mn, n, T2, ld, 1.0, pb.Q, n, 1.0);   // Q + K'RK
      wgemm<true, false>(lane, n, n, n, Acl, ld, T1, ld, S, ld, 1.0, T2, ld, 1.0);
      wsymmetrize(lane, n, S, ld);
    }
  }
  return ok;
}

// Exact constrained solve from the state in ar.x (clqr.cuh: clqr_solve with run-time sizes). Writes u0 (ar.u is
// scratch: the result goes to u0_out[m], shared or global) and *V. Returns flag bits (warp-uniform).
__device__ __forceinline__ int dyn_clqr_solve(int lane, Arena& ar, const DynPb& pb, int N, const double* x0,
                                              const QpWs& ws, double* u0_out, double* V, const lq::Refs& rf) {
  const int n = ar.n, m = ar.m, ld = ar.ld;
  double* Ah = ar.big[0];
  double* x = ar.x; double* xn = ar.xn;                    // rollout state (ar.xa / ar.xb belong to the backward sweep)
  const bool trk = rf.any();
  int flags = 0;
  if (trk && !dyn_clqr_backward(lane, ar, pb, N, lq::Mask128(), lq::Mask128(), ws, rf)) flags |= lq::FLAG_CHOL_FAIL;
  const double* Kst = trk ? ws.Kc : ws.Ku;
  bool feas = true;
  for (int i = lane; i < n; i += 32) x[i] = x0[i];
  __syncwarp();
  double cost_u = wquad(lane, n, x0, pb.Q, n, x0);
  for (int k = 0; k < N; ++k) {
    wgemv<false>(lane, m, n, Kst + (size_t)k * m * n, n, x, ar.u);
    for (int j = 0; j < m; ++j) {                          // replicated scalar work on m <= 8 entries
      double uj = ar.u[j];
      if (trk) uj += ws.kc[(size_t)k * m + j];
      if (uj < pb.ulo[j] || uj > pb.uhi[j]) feas = false;
      if (k == 0 && lane == 0) u0_out[j] = uj;
      __syncwarp();
      if (lane == 0) ar.u[j] = uj;
    }
    __syncwarp();
    if (!feas) break;
    dyn_step_model(lane, n, m, Ah, ld, ar.Bh, x, ar.u, xn);
    if (trk) {
      double part = 0.0;
      for (int j = 0; j < m; ++j) ar.G2[j] = ar.u[j] - rf.u(j, k);
      for (int i = lane; i < n; i += 32) ar.xb[i] = xn[i] - rf.x(i, k);
      __syncwarp();
      part = wquad(lane, m, ar.G2, pb.R, m, ar.G2);
      part += wquad(lane, n, ar.xb, (k == N - 1) ? pb.Pt : pb.Q, n, ar.xb);
      cost_u += part;
    }
    for (int i = lane; i < n; i += 32) x[i] = xn[i];
    __syncwarp();
  }
  if (feas) {
    *V = trk ? cost_u : wquad(lane, n, x0, ar.big[4], ld, x0);
    return flags;
  }
  flags |= lq::FLAG_QP_ACTIVE;
  if (N * m > lq::kMaskBits) {
    if (lane == 0) for (int j = 0; j < m; ++j) u0_out[j] = dmin(dmax(u0_out[j], pb.ulo[j]), pb.uhi[j]);
    __syncwarp();
    *V = NAN;
    return flags | lq::FLAG_QP_MAXITER;
  }
  // ---- feasible start: saturated rollout of the unconstrained law
  lq::Mask128 fixed, athi;
  for (int i = lane; i < n; i += 32) x[i] = x0[i];
  __syncwarp();
  for (int k = 0; k < N; ++k) {
    wgemv<false>(lane, m, n, Kst + (size_t)k * m * n, n, x, ar.u);
    for (int j = 0; j < m; ++j) {
      double uj = ar.u[j];
      if (trk) uj += ws.kc[(size_t)k * m + j];
      const int bit = k * m + j;
      if (uj >= pb.uhi[j]) { uj = pb.uhi[j]; fixed.set(bit); athi.set(bit); }
      else if (uj <= pb.ulo[j]) { uj = pb.ulo[j]; fixed.set(bit); }
      __syncwarp();
      if (lane == 0) { ar.u[j] = uj; ws.z[(size_t)k * m + j] = uj; }
    }
    __syncwarp();
    dyn_step_model(lane, n, m, Ah, ld, ar.Bh, x, ar.u, xn);
    for (int i = lane; i < n; i += 32) x[i] = xn[i];
    __syncwarp();
  }
  // ---- primal active-set iterations
  const int maxit = 8 * N * m + 32;
  bool done = false;
  for (int it = 0; it < maxit && !done; ++it) {
    if (!dyn_clqr_backward(lane, ar, pb, N, fixed, athi, ws, rf)) flags |= lq::FLAG_CHOL_FAIL;
    double alpha = 1.0;
    int block = -1;
    bool block_hi = false;
    for (int i = lane; i < n; i += 32) { x[i] = x0[i]; ws.xs[i] = x0[i]; }
    __syncwarp();
    for (int k = 0; k < N; ++k) {
      wgemv<false>(lane, m, n, ws.Kc + (size_t)k * m * n, n, x, ar.u);
      for (int j = 0; j < m; ++j) {
        double uj = ar.u[j] + ws.kc[(size_t)k * m + j];
        const int bit = k * m + j;
        const bool isfx = fixed.test(bit);
        if (isfx) uj = athi.test(bit) ? pb.uhi[j] : pb.ulo[j];
        if (!isfx) {
          const double zc = ws.z[(size_t)k * m + j];
          if (uj > pb.uhi[j]) {
            const double a = (pb.uhi[j] - zc) / (uj - zc);
            if (a < alpha) { alpha = a; block = bit; block_hi = true; }
          } else if (uj < pb.ulo[j]) {
            const double a = (pb.ulo[j] - zc) / (uj - zc);
            if (a < alpha) { alpha = a; block = bit; block_hi = false; }
          }
        }
        __syncwarp();
        if (lane == 0) { ar.u[j] = uj; ws.zs[(size_t)k * m + j] = uj; }
      }
      __syncwarp();
      dyn_step_model(lane, n, m, Ah, ld, ar.Bh, x, ar.u, xn);
      for (int i = lane; i < n; i += 32) { x[i] = xn[i]; ws.xs[(size_t)(k + 1) * n + i] = xn[i]; }
      __syncwarp();
    }
    if (block >= 0) {
      if (alpha < 0.0) alpha = 0.0;
      for (int e = lane; e < N * m; e += 32) {
        const double zc = ws.z[e];
        ws.z[e] = fma(alpha, ws.zs[e] - zc, zc);
      }
      __syncwarp();
      const int j = block % m;
      if (lane == 0) ws.z[block] = block_hi ? pb.uhi[j] : pb.ulo[j];
      __syncwarp();
      fixed.set(block);
      if (block_hi) athi.set(block); else athi.clear(block);
      continue;
    }
    for (int e = lane; e < N * m; e += 32) ws.z[e] = ws.zs[e];
    __syncwarp();
    // multipliers from the costate sweep: lam in ar.xb
    double* lam = ar.xb; double* tmp = ar.xa;
    for (int i = lane; i < n; i += 32) {
      double acc = 0.0;
      for (int j = 0; j < n; ++j) acc = fma(pb.Pt[i * n + j], ws.xs[(size_t)N * n + j] - rf.x(j, N - 1), acc);
      lam[i] = 2.0 * acc;
    }
    __syncwarp();
    double worst = 0.0;
    int rel = -1;
    for (int k = N - 1; k >= 0; --k) {
      for (int j = 0; j < m; ++j) {
        const int bit = k * m + j;
        if (fixed.test(bit)) {
          double g1 = 0.0, g2 = 0.0;
          for (int r = 0; r < m; ++r) g1 = fma(pb.R[j * m + r], ws.z[(size_t)k * m + r] - rf.u(r, k), g1);
          for (int r = 0; r < n; ++r) g2 = fma(ar.Bh[r * m + j], lam[r], g2);
          const double g = 2.0 * g1 + g2;
          const double tol = 1e-11 * (fabs(2.0 * g1) + fabs(g2)) + 1e-300;
          const double viol = athi.test(bit) ? g : -g;
          if (viol > tol && viol > worst) { worst = viol; rel = bit; }
        }
      }
      if (k > 0) {
        for (int i = lane; i < n; i += 32) {
          double acc = 0.0;
          for (int r = 0; r < n; ++r) acc = fma(pb.Q[i * n + r], ws.xs[(size_t)k * n + r] - rf.x(r, k - 1), acc);
          acc *= 2.0;
          for (int r = 0; r < n; ++r) acc = fma(Ah[r * ld + i], lam[r], acc);
          tmp[i] = acc;
        }
        __syncwarp();
        for (int i = lane; i < n; i += 32) lam[i] = tmp[i];
        __syncwarp();
      }
    }
    if (rel < 0) done = true;
    else fixed.clear(rel);
  }
  if (!done) flags |= lq::FLAG_QP_MAXITER;
  // ---- objective along z
  for (int i = lane; i < n; i += 32) x[i] = x0[i];
  __syncwarp();
  double cost = wquad(lane, n, x0, pb.Q, n, x0);
  for (int k = 0; k < N; ++k) {
    if (lane < m) ar.u[lane] = ws.z[(size_t)k * m + lane];
    __syncwarp();
    if (k == 0 && lane == 0) for (int j = 0; j < m; ++j) u0_out[j] = ar.u[j];
    dyn_step_model(lane, n, m, Ah, ld, ar.Bh, x, ar.u, xn);
    if (lane < m) ar.G2[lane] = ar.u[lane] - rf.u(lane, k);
    for (int i = lane; i < n; i += 32) ar.xb[i] = xn[i] - rf.x(i, k);
    __syncwarp();
    cost += wquad(lane, m, ar.G2, pb.R, m, ar.G2);
    cost += wquad(lane, n, ar.xb, (k == N - 1) ? pb.Pt : pb.Q, n, ar.xb);
    for (int i = lane; i < n; i += 32) x[i] = xn[i];
    __syncwarp();
  }
  *V = cost;
  return flags;
}

// ------------------------------------------------------------------------------------------------ K2c pieces
// Infinite-horizon closed loop (clqr.cuh: certified_closed_loop, run-time sizes).
// Box feasibility certificate of the unconstrained plan (clqr.cuh: plan_prepare's cstar): a copy of P0 (big[4], as
// dyn_plan_prepare leaves it; not modified) is factored as L D L' in big[6], the gains ws.Ku propagate Phi_k (big[2] /
// big[3] / big[5]), and cstar = (1 - 1e-9) min_{k,j} b_j^2 / (g_{k,j} P0^-1 g_{k,j}'), g_k = K_k Phi_k. Returns +inf
// without input bounds, -1 when P0 is not positive definite or the box does not hold the origin in its interior.
// Needs an arena of 7; big[2], big[3], big[5], big[6], ar.xa, ar.xb, ar.Y and ar.T_mn are scratch.
__device__ __forceinline__ double dyn_box_certificate(int lane, Arena& ar, const DynPb& pb, int N, const QpWs& ws) {
  const int n = ar.n, m = ar.m, ld = ar.ld;
  if (!pb.has_bounds) return HUGE_VAL;
  double* Lp = ar.big[6];
  wcopy(lane, n, n, ar.big[4], ld, Lp, ld);
  bool ok = wldl(lane, n, Lp, ld, ar.xa, ar.xb);
  for (int j = 0; j < m; ++j) ok = ok && (dmin(-pb.ulo[j], pb.uhi[j]) > 0.0);
  if (!ok) return -1.0;
  double* Phi = ar.big[2]; double* Acl = ar.big[3]; double* Pn = ar.big[5];
  for (int e = lane; e < n * n; e += 32) { const int i = e / n, j = e - i * n; Phi[i * ld + j] = (i == j) ? 1.0 : 0.0; }
  __syncwarp();
  double cs = HUGE_VAL;
  for (int k = 0; k < N; ++k) {
    const double* K = ws.Ku + (size_t)k * m * n;
    wgemm<false, false>(lane, m, n, n, K, n, Phi, ld, ar.T_mn, n);                     // g = K_k Phi_k (m x n)
    if (lane < m) {                                        // y = L^-1 g_j' (unit L) in column j of ar.Y, q = y' D^-1 y
      const double b = dmin(-pb.ulo[lane], pb.uhi[lane]);
      double q = 0.0;
      for (int i = 0; i < n; ++i) {
        double acc = ar.T_mn[lane * n + i];
        for (int c = 0; c < i; ++c) acc = fma(-Lp[i * ld + c], ar.Y[c * m + lane], acc);
        ar.Y[i * m + lane] = acc;
        q = fma(acc * ar.xa[i], acc, q);
      }
      if (b * b < 1e300 && q > 0.0) cs = dmin(cs, b * b / q);
    }
    __syncwarp();
    if (k + 1 < N) {
      wgemm<false, false>(lane, n, m, n, ar.Bh, m, K, n, Acl, ld, 1.0, ar.big[0], ld, 1.0);   // Ah + Bh K_k
      wgemm<false, false>(lane, n, n, n, Acl, ld, Phi, ld, Pn, ld);
      wcopy(lane, n, n, Pn, ld, Phi, ld);
    }
  }
  cs = wmind(cs);
  return (cs == cs) ? cs * (1.0 - 1e-9) : -1.0;
}

// Level c_S = (1 - 1e-9) cstar / lambda_max(L^-1 P0 L^-T) of the invariant set {x' S x <= c_S} (S = L L'), with P0
// in big[1] and S in big[5]. Copies S to big[6] (kept for the closed loop: dyn_clqr_solve uses big[1..5]) and returns
// NaN when S is not positive definite. With S = L D L' (unit L), the matrix is D^-1/2 L^-1 P0 L^-T D^-1/2; big[2..5]
// are scratch.
__device__ __forceinline__ double dyn_tail_level(int lane, Arena& ar, double cstar) {
  const int n = ar.n, ld = ar.ld;
  double* Ls = ar.big[5]; double* Z = ar.big[2]; double* M = ar.big[3]; const double* P0 = ar.big[1];
  wcopy(lane, n, n, Ls, ld, ar.big[6], ld);
  if (!wldl(lane, n, Ls, ld, ar.xa, ar.xb)) return NAN;
  for (int c = lane; c < n; c += 32)                       // Z = L^-1 P0, lane = column
    for (int i = 0; i < n; ++i) {
      double acc = P0[i * ld + c];
      for (int k = 0; k < i; ++k) acc = fma(-Ls[i * ld + k], Z[k * ld + c], acc);
      Z[i * ld + c] = acc;
    }
  __syncwarp();
  for (int c = lane; c < n; c += 32)                       // M = L^-1 Z', lane = column
    for (int i = 0; i < n; ++i) {
      double acc = Z[c * ld + i];
      for (int k = 0; k < i; ++k) acc = fma(-Ls[i * ld + k], M[k * ld + c], acc);
      M[i * ld + c] = acc;
    }
  __syncwarp();
  for (int e = lane; e < n * n; e += 32) {                 // D^-1/2 (.) D^-1/2, symmetrised, into big[4]
    const int i = e / n, j = e - i * n;
    ar.big[4][i * ld + j] = 0.5 * (M[i * ld + j] + M[j * ld + i]) * sqrt(ar.xa[i] * ar.xa[j]);
  }
  __syncwarp();
  const double lmax = wsym_extreme(lane, n, ar.big[4], ld, true, M, ld, ar.v);
  __syncwarp();
  return (lmax > 0.0 && cstar > 0.0) ? (1.0 - 1e-9) * cstar / lmax : NAN;
}

}  // namespace lqd
