// small_la.cuh — fixed-size dense linear algebra for one system per thread (FP64).
//
// Every routine is a fully unrolled template over compile-time sizes so that, on the device, the operands live
// in registers (no local memory, no dynamic indexing) and FMAs can take the replicated problem constants
// straight from the kernel-parameter constant bank.  The same headers compile with g++ (tests/hostmath) so the
// math can be checked against the oracle in the GPU-less build container; that harness is test-only.
//
// Matrices are row-major: M[i*C + j].
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define LQ_HD __host__ __device__ __forceinline__
#define LQ_HD_NOINLINE static __host__ __device__ __noinline__
#define LQ_HD_NOINLINE_T __host__ __device__ __noinline__
#define LQ_UNROLL _Pragma("unroll")
#else
#define LQ_HD inline
#define LQ_HD_NOINLINE static
#define LQ_HD_NOINLINE_T
#define LQ_UNROLL
#endif

namespace lq {

LQ_HD double dmax(double a, double b) { return a > b ? a : b; }
LQ_HD double dmin(double a, double b) { return a < b ? a : b; }
LQ_HD double dsign(double a, double b) { return b >= 0.0 ? fabs(a) : -fabs(a); }

// Sign-stripped high word of a double: for finite values the order of |v| is the order of this word up to a relative
// 2^-20, and NaN / Inf sort above every finite value. Magnitude tracking for convergence tests runs on it so that it
// costs integer-pipe instructions (LOP + IMNMX) instead of FP64-pipe compares (DSETP + 2 SEL per dmax).
LQ_HD uint32_t abs_hi(double v) {
#if defined(__CUDA_ARCH__)
  return (uint32_t)__double2hiint(v) & 0x7fffffffu;
#else
  uint64_t b;
  memcpy(&b, &v, sizeof(b));
  return (uint32_t)(b >> 32) & 0x7fffffffu;
#endif
}
// "v is a positive NORMAL finite number", decided on the high word (one integer subtract + compare instead of two
// FP64-pipe DSETPs): sign clear and exponent field in [1, 0x7fe]. NaN, Inf, zero, negatives and denormals are false.
LQ_HD bool is_pos_normal(double v) {
#if defined(__CUDA_ARCH__)
  const uint32_t h = (uint32_t)__double2hiint(v);
#else
  uint64_t b;
  memcpy(&b, &v, sizeof(b));
  const uint32_t h = (uint32_t)(b >> 32);
#endif
  return (h - 0x00100000u) < 0x7fe00000u;
}
LQ_HD double from_abs_hi(uint32_t h) {
#if defined(__CUDA_ARCH__)
  return __hiloint2double((int)h, 0);
#else
  const uint64_t b = (uint64_t)h << 32;
  double v;
  memcpy(&v, &b, sizeof(v));
  return v;
#endif
}
LQ_HD uint32_t umax32(uint32_t a, uint32_t b) { return a > b ? a : b; }

// Reciprocal for normal, non-zero x: hardware seed (MUFU.RCP64H, >= 20 good bits) + two Newton steps = 1 MUFU +
// 4 DFMA and <= 1 ulp error, versus ~12 FP64-pipe instructions plus a slow-path call for an IEEE `1.0 / x`.
// Callers guarantee x is finite, non-zero and not subnormal (or guard the result). Host build: plain division.
LQ_HD double rcp(double x) {
#if defined(__CUDA_ARCH__)
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  double e = fma(-x, y, 1.0);
  y = fma(y, e, y);
  e = fma(-x, y, 1.0);
  return fma(y, e, y);
#else
  return 1.0 / x;
#endif
}

// out (R x C) = A (R x K) * B (K x C)
template <int R, int K, int C>
LQ_HD void mm(const double* A, const double* B, double* out) {
  LQ_UNROLL for (int i = 0; i < R; ++i)
    LQ_UNROLL for (int j = 0; j < C; ++j) {
      double acc = A[i * K] * B[j];
      LQ_UNROLL for (int k = 1; k < K; ++k) acc = fma(A[i * K + k], B[k * C + j], acc);
      out[i * C + j] = acc;
    }
}

// out (R x C) = A^T B with A (K x R), B (K x C)
template <int K, int R, int C>
LQ_HD void mtm(const double* A, const double* B, double* out) {
  LQ_UNROLL for (int i = 0; i < R; ++i)
    LQ_UNROLL for (int j = 0; j < C; ++j) {
      double acc = A[i] * B[j];
      LQ_UNROLL for (int k = 1; k < K; ++k) acc = fma(A[k * R + i], B[k * C + j], acc);
      out[i * C + j] = acc;
    }
}

// out (n x n, symmetric) = base + A^T B  where the product is known to be symmetric (A, B are K x n)
template <int K, int n>
LQ_HD void sym_add_mtm(const double* base, const double* A, const double* B, double* out) {
  LQ_UNROLL for (int i = 0; i < n; ++i)
    LQ_UNROLL for (int j = i; j < n; ++j) {
      double acc = base[i * n + j];
      LQ_UNROLL for (int k = 0; k < K; ++k) acc = fma(A[k * n + i], B[k * n + j], acc);
      out[i * n + j] = acc;
      out[j * n + i] = acc;
    }
}

// out (n x n, symmetric) = base - Y Y^T, Y (n x m)
template <int n, int m>
LQ_HD void sym_sub_yyt(const double* base, const double* Y, double* out) {
  LQ_UNROLL for (int i = 0; i < n; ++i)
    LQ_UNROLL for (int j = i; j < n; ++j) {
      double acc = base[i * n + j];
      LQ_UNROLL for (int k = 0; k < m; ++k) acc = fma(-Y[i * m + k], Y[j * m + k], acc);
      out[i * n + j] = acc;
      out[j * n + i] = acc;
    }
}

// x^T M y
template <int n>
LQ_HD double quad(const double* x, const double* M, const double* y) {
  double tot = 0.0;
  LQ_UNROLL for (int i = 0; i < n; ++i) {
    double r = 0.0;
    LQ_UNROLL for (int j = 0; j < n; ++j) r = fma(M[i * n + j], y[j], r);
    tot = fma(x[i], r, tot);
  }
  return tot;
}

// y (R) = M (R x C) x (C)
template <int R, int C>
LQ_HD void mv(const double* M, const double* x, double* y) {
  LQ_UNROLL for (int i = 0; i < R; ++i) {
    double r = 0.0;
    LQ_UNROLL for (int j = 0; j < C; ++j) r = fma(M[i * C + j], x[j], r);
    y[i] = r;
  }
}

// In-place Cholesky G = L L^T (lower triangle of G overwritten by L; strict upper untouched).
// Returns false when a pivot is not positive.
template <int m>
LQ_HD bool chol(double* G) {
  bool ok = true;
  LQ_UNROLL for (int j = 0; j < m; ++j) {
    double d = G[j * m + j];
    LQ_UNROLL for (int k = 0; k < j; ++k) d = fma(-G[j * m + k], G[j * m + k], d);
    ok = ok && (d > 0.0);
    const double l = sqrt(d);
    const double inv = 1.0 / l;
    G[j * m + j] = l;
    LQ_UNROLL for (int i = j + 1; i < m; ++i) {
      double s = G[i * m + j];
      LQ_UNROLL for (int k = 0; k < j; ++k) s = fma(-G[i * m + k], G[j * m + k], s);
      G[i * m + j] = s * inv;
    }
  }
  return ok;
}

// Cholesky that also returns the reciprocals of the diagonal (one rsqrt per column instead of sqrt + division), for the
// triangular solves below that multiply instead of divide — the Riccati step runs 2 of these per horizon step.
// 1 / sqrt(d) for a positive NORMAL d: hardware seed (MUFU.RSQ64H) + two Newton steps in the residual form
// e = 1/2 - (d/2) y^2, y <- y + y e (1 MUFU + 7 FP64 instructions, <= 1 ulp), instead of the library rsqrt() with its
// special-case handling (~11 FP64 instructions and a slow-path branch; 5.7 % of K1's instructions in profile r02).
// Callers test the pivot with is_pos_normal() and flag anything else; the value returned for such a pivot is unspecified.
LQ_HD double rsqrt_pos(double d) {
#if defined(__CUDA_ARCH__)
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
  const double h = 0.5 * d;
  double e = fma(-h * y, y, 0.5);
  y = fma(y, e, y);
  e = fma(-h * y, y, 0.5);
  return fma(y, e, y);
#else
  return 1.0 / sqrt(d);
#endif
}

// sqrt(x) for x >= 0 through the reciprocal square root above (x * rsqrt(x): <= 2 ulp, no slow path); zero and
// denormals return 0. For the closed-form eigenvalue path, whose inputs are scaled to O(1) and whose results pass an
// a-posteriori acceptance test. Host build: plain sqrt.
LQ_HD double sqrt_fast(double x) {
#if defined(__CUDA_ARCH__)
  return is_pos_normal(x) ? x * rsqrt_pos(x) : 0.0;
#else
  return sqrt(x);
#endif
}

template <int m>
LQ_HD bool chol_inv(double* G, double* dinv) {
  bool ok = true;
  LQ_UNROLL for (int j = 0; j < m; ++j) {
    double d = G[j * m + j];
    LQ_UNROLL for (int k = 0; k < j; ++k) d = fma(-G[j * m + k], G[j * m + k], d);
    ok = ok && is_pos_normal(d);
    const double inv = rsqrt_pos(d);
    dinv[j] = inv;
    G[j * m + j] = d * inv;
    LQ_UNROLL for (int i = j + 1; i < m; ++i) {
      double s = G[i * m + j];
      LQ_UNROLL for (int k = 0; k < j; ++k) s = fma(-G[i * m + k], G[j * m + k], s);
      G[i * m + j] = s * inv;
    }
  }
  return ok;
}

template <int r, int m>
LQ_HD void solve_right_lt_inv(const double* L, const double* dinv, double* X) {
  LQ_UNROLL for (int i = 0; i < r; ++i)
    LQ_UNROLL for (int j = 0; j < m; ++j) {
      double s = X[i * m + j];
      LQ_UNROLL for (int k = 0; k < j; ++k) s = fma(-X[i * m + k], L[j * m + k], s);
      X[i * m + j] = s * dinv[j];
    }
}

// Rows of X (r x m) are solved against L^T from the right:  Y L^T = X  (Y overwrites X).
template <int r, int m>
LQ_HD void solve_right_lt(const double* L, double* X) {
  LQ_UNROLL for (int i = 0; i < r; ++i)
    LQ_UNROLL for (int j = 0; j < m; ++j) {
      double s = X[i * m + j];
      LQ_UNROLL for (int k = 0; k < j; ++k) s = fma(-X[i * m + k], L[j * m + k], s);
      X[i * m + j] = s / L[j * m + j];
    }
}

// Solve L Z = X (forward), X is (m x c), overwritten.
template <int m, int c>
LQ_HD void solve_l(const double* L, double* X) {
  LQ_UNROLL for (int j = 0; j < c; ++j)
    LQ_UNROLL for (int i = 0; i < m; ++i) {
      double s = X[i * c + j];
      LQ_UNROLL for (int k = 0; k < i; ++k) s = fma(-L[i * m + k], X[k * c + j], s);
      X[i * c + j] = s / L[i * m + i];
    }
}

// Solve L^T Z = X (backward), X is (m x c), overwritten.
template <int m, int c>
LQ_HD void solve_lt(const double* L, double* X) {
  LQ_UNROLL for (int j = 0; j < c; ++j)
    LQ_UNROLL for (int i = m - 1; i >= 0; --i) {
      double s = X[i * c + j];
      LQ_UNROLL for (int k = i + 1; k < m; ++k) s = fma(-L[k * m + i], X[k * c + j], s);
      X[i * c + j] = s / L[i * m + i];
    }
}

template <int m, int c>
LQ_HD void solve_lt_inv(const double* L, const double* dinv, double* X) {
  LQ_UNROLL for (int j = 0; j < c; ++j)
    LQ_UNROLL for (int i = m - 1; i >= 0; --i) {
      double s = X[i * c + j];
      LQ_UNROLL for (int k = i + 1; k < m; ++k) s = fma(-L[k * m + i], X[k * c + j], s);
      X[i * c + j] = s * dinv[i];
    }
}

// LU with partial pivoting, solves W X = Rhs for n x c right-hand sides (both overwritten). Row swaps are
// predicated selects so that everything stays in registers. Returns false on a zero pivot.
template <int n, int c>
LQ_HD bool lu_solve(double* W, double* X) {
  bool ok = true;
  LQ_UNROLL for (int k = 0; k < n; ++k) {
    // pivot search
    int piv = k;
    double best = fabs(W[k * n + k]);
    LQ_UNROLL for (int i = k + 1; i < n; ++i) {
      const double v = fabs(W[i * n + k]);
      if (v > best) { best = v; piv = i; }
    }
    ok = ok && (best > 0.0);
    LQ_UNROLL for (int i = k + 1; i < n; ++i) {
      const bool sw = (piv == i);
      LQ_UNROLL for (int j = 0; j < n; ++j) {
        const double a = W[k * n + j], b = W[i * n + j];
        W[k * n + j] = sw ? b : a;
        W[i * n + j] = sw ? a : b;
      }
      LQ_UNROLL for (int j = 0; j < c; ++j) {
        const double a = X[k * c + j], b = X[i * c + j];
        X[k * c + j] = sw ? b : a;
        X[i * c + j] = sw ? a : b;
      }
    }
    const double inv = 1.0 / W[k * n + k];
    LQ_UNROLL for (int i = k + 1; i < n; ++i) {
      const double f = W[i * n + k] * inv;
      LQ_UNROLL for (int j = k + 1; j < n; ++j) W[i * n + j] = fma(-f, W[k * n + j], W[i * n + j]);
      LQ_UNROLL for (int j = 0; j < c; ++j) X[i * c + j] = fma(-f, X[k * c + j], X[i * c + j]);
    }
  }
  LQ_UNROLL for (int j = 0; j < c; ++j)
    LQ_UNROLL for (int i = n - 1; i >= 0; --i) {
      double s = X[i * c + j];
      LQ_UNROLL for (int k = i + 1; k < n; ++k) s = fma(-W[i * n + k], X[k * c + j], s);
      X[i * c + j] = s / W[i * n + i];
    }
  return ok;
}

template <int len>
LQ_HD double max_abs(const double* v) {
  double r = 0.0;
  LQ_UNROLL for (int i = 0; i < len; ++i) r = dmax(r, fabs(v[i]));
  return r;
}

// Extremal eigenvalues of a small symmetric matrix by cyclic Jacobi (all indices static -> registers).
// Used for ||M||_2 = sqrt(lambda_max(M^T M)) and lambda_{max,min}(Q), (R).
template <int n>
LQ_HD void sym_eig_minmax(const double* Sin, double* lmin, double* lmax) {
  if (n == 1) { *lmin = *lmax = Sin[0]; return; }
  double a[n * n];
  LQ_UNROLL for (int i = 0; i < n * n; ++i) a[i] = Sin[i];
  for (int sweep = 0; sweep < 30; ++sweep) {
    double off = 0.0, diag = 0.0;
    LQ_UNROLL for (int i = 0; i < n; ++i) {
      diag = dmax(diag, fabs(a[i * n + i]));
      LQ_UNROLL for (int j = i + 1; j < n; ++j) off = dmax(off, fabs(a[i * n + j]));
    }
    if (off <= 1e-300 || off <= 1e-17 * diag) break;
    LQ_UNROLL for (int p = 0; p < n - 1; ++p)
      LQ_UNROLL for (int q = p + 1; q < n; ++q) {
        const double apq = a[p * n + q];
        if (fabs(apq) > 0.0) {
          const double theta = (a[q * n + q] - a[p * n + p]) / (2.0 * apq);
          const double t = dsign(1.0, theta) / (fabs(theta) + sqrt(fma(theta, theta, 1.0)));
          const double c = 1.0 / sqrt(fma(t, t, 1.0));
          const double s = t * c;
          LQ_UNROLL for (int k = 0; k < n; ++k) {   // columns p, q
            const double akp = a[k * n + p], akq = a[k * n + q];
            a[k * n + p] = c * akp - s * akq;
            a[k * n + q] = s * akp + c * akq;
          }
          LQ_UNROLL for (int k = 0; k < n; ++k) {   // rows p, q
            const double apk = a[p * n + k], aqk = a[q * n + k];
            a[p * n + k] = c * apk - s * aqk;
            a[q * n + k] = s * apk + c * aqk;
          }
        }
      }
  }
  double lo = a[0], hi = a[0];
  LQ_UNROLL for (int i = 1; i < n; ++i) { lo = dmin(lo, a[i * n + i]); hi = dmax(hi, a[i * n + i]); }
  *lmin = lo; *lmax = hi;
}

// Full eigen-decomposition S = V diag(w) V' of a small symmetric matrix by the cyclic Jacobi sweeps of
// sym_eig_minmax, with the rotations accumulated into V (row-major, eigenvector j in column j). Returns false when 30
// sweeps end before the off-diagonal tolerance holds.
template <int n>
LQ_HD bool sym_eig_jacobi(const double* Sin, double* w, double* V) {
  double a[n * n];
  LQ_UNROLL for (int i = 0; i < n * n; ++i) a[i] = Sin[i];
  LQ_UNROLL for (int i = 0; i < n; ++i)
    LQ_UNROLL for (int j = 0; j < n; ++j) V[i * n + j] = (i == j) ? 1.0 : 0.0;
  bool conv = n == 1;
  for (int sweep = 0; sweep < 30 && n > 1; ++sweep) {
    double off = 0.0, diag = 0.0;
    LQ_UNROLL for (int i = 0; i < n; ++i) {
      diag = dmax(diag, fabs(a[i * n + i]));
      LQ_UNROLL for (int j = i + 1; j < n; ++j) off = dmax(off, fabs(a[i * n + j]));
    }
    if (off <= 1e-300 || off <= 1e-17 * diag) { conv = true; break; }
    LQ_UNROLL for (int p = 0; p < n - 1; ++p)
      LQ_UNROLL for (int q = p + 1; q < n; ++q) {
        const double apq = a[p * n + q];
        if (fabs(apq) > 0.0) {
          const double theta = (a[q * n + q] - a[p * n + p]) / (2.0 * apq);
          const double t = dsign(1.0, theta) / (fabs(theta) + sqrt(fma(theta, theta, 1.0)));
          const double c = 1.0 / sqrt(fma(t, t, 1.0));
          const double s = t * c;
          LQ_UNROLL for (int k = 0; k < n; ++k) {   // columns p, q of a and of V
            const double akp = a[k * n + p], akq = a[k * n + q];
            a[k * n + p] = c * akp - s * akq;
            a[k * n + q] = s * akp + c * akq;
            const double vkp = V[k * n + p], vkq = V[k * n + q];
            V[k * n + p] = c * vkp - s * vkq;
            V[k * n + q] = s * vkp + c * vkq;
          }
          LQ_UNROLL for (int k = 0; k < n; ++k) {   // rows p, q
            const double apk = a[p * n + k], aqk = a[q * n + k];
            a[p * n + k] = c * apk - s * aqk;
            a[q * n + k] = s * apk + c * aqk;
          }
        }
      }
  }
  LQ_UNROLL for (int i = 0; i < n; ++i) w[i] = a[i * n + i];
  return conv;
}

// Spectral norm of an (r x c) matrix: sqrt(lambda_max of the smaller Gram matrix).
template <int r, int c>
LQ_HD double norm2(const double* M) {
  double lo, hi;
  if (r <= c) {
    double g[r * r];
    LQ_UNROLL for (int i = 0; i < r; ++i)
      LQ_UNROLL for (int j = i; j < r; ++j) {
        double s = 0.0;
        LQ_UNROLL for (int k = 0; k < c; ++k) s = fma(M[i * c + k], M[j * c + k], s);
        g[i * r + j] = s; g[j * r + i] = s;
      }
    sym_eig_minmax<r>(g, &lo, &hi);
  } else {
    double g[c * c];
    LQ_UNROLL for (int i = 0; i < c; ++i)
      LQ_UNROLL for (int j = i; j < c; ++j) {
        double s = 0.0;
        LQ_UNROLL for (int k = 0; k < r; ++k) s = fma(M[k * c + i], M[k * c + j], s);
        g[i * c + j] = s; g[j * c + i] = s;
      }
    sym_eig_minmax<c>(g, &lo, &hi);
  }
  return sqrt(dmax(hi, 0.0));
}

// General inverse of a small matrix (used once per problem for Q^-1, utils.py:560).
template <int n>
LQ_HD bool inverse(const double* M, double* out) {
  double W[n * n];
  LQ_UNROLL for (int i = 0; i < n * n; ++i) W[i] = M[i];
  LQ_UNROLL for (int i = 0; i < n; ++i)
    LQ_UNROLL for (int j = 0; j < n; ++j) out[i * n + j] = (i == j) ? 1.0 : 0.0;
  return lu_solve<n, n>(W, out);
}

}  // namespace lq
