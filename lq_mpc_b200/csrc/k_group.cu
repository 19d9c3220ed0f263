// k_group.cu — K1 for n = 6 and n = 8: one sample per LANE GROUP (sm_100a).
//
// Thread-per-sample K1 stops paying at n >= 6: P, M, MA, A^ alone are 4 n^2 doubles = 512 registers at n = 8, the
// 255-register build spills every product through local memory, and its shifted-QR spectral radius on a 64-entry
// local array dominates the run (FP64 pipe at 0.09 of peak). Here L lanes of one warp share a sample
// (n = 8: 4 lanes x 2 rows, n = 6: 2 lanes x 3 rows):
//   * every n x n iterate (P, M = P - YY', M A^, S, the doubling power) is ROW-DISTRIBUTED: a lane holds R = n / L rows
//     in registers, so an n x n matrix costs 2 R n registers per lane instead of 2 n^2;
//   * the right-hand operand of a product is read from the group's shared-memory arena as 16-byte broadcasts (all L
//     lanes of a group read the same address; the arenas of a warp's groups are staggered by 4 banks). The
//     shared-memory return path moves 128 B per clock per SM whatever the broadcast, i.e. 16 doubles for 64 DFMA
//     lanes: with R rows per lane a loaded double feeds R DFMAs, so R = 2 caps the FP64 pipe near one half and R = 4
//     would lift the cap — but the unrolled R = 4 code overflows the instruction cache (measured, DESIGN.md §4);
//   * A' X products read the left operand column-wise from the arena, so no transposed copy is kept; m x m and m x n
//     quantities (G = R + B^'PB, its Cholesky factor, the gain) are reduced over the group with xor-shuffles and
//     then REPLICATED in every lane, which keeps all control flow group-uniform; the gain and x0 live in the arena;
//   * the spectral radius does NOT run a QR iteration: rho = lim max|Acl^(2^k)|^(1/2^k) by repeated squaring with
//     exact power-of-two rescaling (the products above, FP64-pipe work), accepted early through the traces of two
//     successive powers (dominant real eigenvalue, +- pair or complex pair; see closed_loop_emit) — typically after
//     9-14 squarings — and otherwise by the two-estimate rule of K4a after 40; only a group whose estimates still
//     disagree runs the thread-level Hessenberg + shifted-QR code (eig.cuh) on its lane 0.
// Loops whose trip count depends on the data (squarings, Lyapunov doubling) run to the warp's slowest group with
// finished groups' state frozen, because the groups of a warp share __syncwarp and the shuffles.
// Same evaluation, flags and outputs as riccati.cuh::eval_sample (the reference semantics are cited there).
#include "engine.h"
#include "sampler.cuh"

namespace {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kRhoK1 = 34, kRhoK2 = 40;   // squarings behind the two spectral-radius estimates (as K4a)
constexpr double kRhoEta = 1e-9;           // dominant-pair early acceptance: consistency of successive candidates
constexpr double kRhoMinRoot = 0.02;       //   ... and the smallest root / max|X| ratio a candidate may have

__device__ __forceinline__ double ldg_stream(const double* p) {
  double v;
  asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ void stg_stream(double* p, double v) {
  asm volatile("st.global.L1::no_allocate.f64 [%0], %1;" ::"l"(p), "d"(v));
}

// Reductions over the L lanes of a group. The shuffle mask names the group only, so a branch that is uniform within a
// group but not across the warp (stable / unstable closed loops) may hold one.
template <int L>
__device__ __forceinline__ unsigned group_mask() {
  return ((1u << L) - 1u) << ((threadIdx.x & 31u) & ~(unsigned)(L - 1));
}
template <int L>
__device__ __forceinline__ double g_sum(double v) {
  const unsigned gm = group_mask<L>();
#pragma unroll
  for (int off = L / 2; off >= 1; off >>= 1) v += __shfl_xor_sync(gm, v, off);
  return v;
}
template <int L>
__device__ __forceinline__ uint32_t g_max(uint32_t v) {
  const unsigned gm = group_mask<L>();
#pragma unroll
  for (int off = L / 2; off >= 1; off >>= 1) v = max(v, __shfl_xor_sync(gm, v, off));
  return v;
}
template <int L>
__device__ __forceinline__ double g_fmax(double v) {
  const unsigned gm = group_mask<L>();
#pragma unroll
  for (int off = L / 2; off >= 1; off >>= 1) v = fmax(v, __shfl_xor_sync(gm, v, off));
  return v;
}

// C[r][j] (+)= sum_k X[r][k] Y[k][j], Y (n x c, row-major) in shared memory, own rows r < R
template <int R, int n, int c, bool ACC>
__device__ __forceinline__ void rows_x_smem(const double (&X)[R][n], const double* __restrict__ Y, double (&C)[R][c]) {
  if (!ACC) {
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int j = 0; j < c; ++j) C[r][j] = 0.0;
  }
#pragma unroll
  for (int k = 0; k < n; ++k) {
    if (c % 2 == 0) {
#pragma unroll
      for (int j = 0; j < c; j += 2) {
        const double2 y = *reinterpret_cast<const double2*>(Y + k * c + j);
#pragma unroll
        for (int r = 0; r < R; ++r) {
          C[r][j] = fma(X[r][k], y.x, C[r][j]);
          C[r][j + 1] = fma(X[r][k], y.y, C[r][j + 1]);
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < c; ++j) {
        const double y = Y[k * c + j];
#pragma unroll
        for (int r = 0; r < R; ++r) C[r][j] = fma(X[r][k], y, C[r][j]);
      }
    }
  }
}

// C[r][j] += sum_k M[k][row0 + r] Y[k][j]: own rows of M' Y, both operands (n x n, row-major) in shared memory
template <int R, int n>
__device__ __forceinline__ void colsT_x_smem(const double* __restrict__ M, int row0, const double* __restrict__ Y,
                                             double (&C)[R][n]) {
#pragma unroll
  for (int k = 0; k < n; ++k) {
    double mk[R];
#pragma unroll
    for (int r = 0; r < R; ++r) mk[r] = M[k * n + row0 + r];
#pragma unroll
    for (int j = 0; j < n; j += 2) {
      const double2 y = *reinterpret_cast<const double2*>(Y + k * n + j);
#pragma unroll
      for (int r = 0; r < R; ++r) {
        C[r][j] = fma(mk[r], y.x, C[r][j]);
        C[r][j + 1] = fma(mk[r], y.y, C[r][j + 1]);
      }
    }
  }
}

template <int R, int n>
__device__ __forceinline__ void store_rows(double* __restrict__ dst, int row0, const double (&X)[R][n]) {
#pragma unroll
  for (int r = 0; r < R; ++r)
#pragma unroll
    for (int j = 0; j < n; j += 2)
      *reinterpret_cast<double2*>(dst + (row0 + r) * n + j) = make_double2(X[r][j], X[r][j + 1]);
}

template <int n>
__device__ __noinline__ double spectral_radius_call(const double* A, bool* ok) {
  return lq::spectral_radius<n>(A, ok);
}

template <int n, int m, int L, bool NESTED>
struct GroupLayout {
  static_assert(n % L == 0 && n % 2 == 0 && (n * m) % 2 == 0 && 32 % L == 0, "lane-group K1: n = L R, even sizes");
  static constexpr int R = n / L;
  static constexpr int kThreads = 128;
  static constexpr int kGroups = kThreads / L;
  // per-CTA constants (true plant and weights), then one arena per group
  static constexpr int oA = 0, oB = oA + n * n, oQ = oB + n * m, kConst = oQ + n * n;
  // arena: A^, B^, two n x n work matrices, Y, the gain, x0 and (several horizons per sample) the stashed cost-to-go
  static constexpr int aAh = 0, aBh = aAh + n * n, aM1 = aBh + n * m, aM2 = aM1 + n * n, aY = aM2 + n * n,
                       aK = aY + n * m, aX = aK + m * n, aP = aX + n + (n % 2),
                       kArenaRaw = aP + (NESTED ? n * n : 0);
  // arena stride == 2 (mod 16) doubles: consecutive groups start 4 banks apart, every arena stays 16-byte aligned
  static constexpr int kArena = ((kArenaRaw + 13) / 16) * 16 + 2;
  static constexpr size_t kSmemBytes = sizeof(double) * (size_t)(kConst + kGroups * kArena);
};

// Shared-memory views of one group + the CTA constants
struct GroupMem {
  const double *cA, *cB, *cQ;
  double *Ah, *Bh, *M1, *M2, *Ys, *Ks, *Xs, *Ps;
};

// One Riccati stage from the cost-to-go rows P (horizon k-1): factor, optional gain (into Ks), optional update of P.
template <int n, int m, int L>
__device__ __forceinline__ int riccati_stage(const lq::Problem<n, m>& pb, const GroupMem& g, int row0,
                                              const double (&Bhr)[n / L][m], double (&P)[n / L][n], bool gain,
                                              bool update) {
  constexpr int R = n / L;
  int bad = 0;
  // ---- factor: Y = P B^, G = R + B^' Y = L L', Y <- Y L^-T
  double Y[R][m];
  rows_x_smem<R, n, m, false>(P, g.Bh, Y);
  double Lm[m * m], Li[m];
#pragma unroll
  for (int i = 0; i < m; ++i)
#pragma unroll
    for (int j = 0; j <= i; ++j) {
      double acc = 0.0;
#pragma unroll
      for (int r = 0; r < R; ++r) acc = fma(Bhr[r][i], Y[r][j], acc);
      acc = g_sum<L>(acc) + pb.R[i * m + j];
      Lm[i * m + j] = acc;
      Lm[j * m + i] = acc;
    }
  if (!lq::chol_inv<m>(Lm, Li)) bad = lq::FLAG_CHOL_FAIL;
  lq::solve_right_lt_inv<R, m>(Lm, Li, &Y[0][0]);
#pragma unroll
  for (int r = 0; r < R; ++r)
#pragma unroll
    for (int j = 0; j < m; ++j) g.Ys[(row0 + r) * m + j] = Y[r][j];
  __syncwarp();
  if (gain) {  // K = -L^-T (Y' A^): partial sums over own rows, reduced over the group; lane 0 files it in Ks
    double K[m * n];
#pragma unroll
    for (int i = 0; i < m; ++i)
#pragma unroll
      for (int j = 0; j < n; ++j) {
        double acc = 0.0;
#pragma unroll
        for (int r = 0; r < R; ++r) acc = fma(Y[r][i], g.Ah[(row0 + r) * n + j], acc);
        K[i * n + j] = g_sum<L>(acc);
      }
    lq::solve_lt_inv<m, n>(Lm, Li, K);
    if (row0 == 0) {
#pragma unroll
      for (int e = 0; e < m * n; e += 2) *reinterpret_cast<double2*>(g.Ks + e) = make_double2(-K[e], -K[e + 1]);
    }
  }
  if (update) {  // P+ = Q + A^' (P - Y Y') A^
    double MA[R][n];
    {
      double Mx[R][n];
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int j = 0; j < n; ++j) {
          double acc = P[r][j];
#pragma unroll
          for (int i = 0; i < m; ++i) acc = fma(-Y[r][i], g.Ys[j * m + i], acc);
          Mx[r][j] = acc;
        }
      rows_x_smem<R, n, n, false>(Mx, g.Ah, MA);
    }
    store_rows<R, n>(g.M1, row0, MA);
    __syncwarp();
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int j = 0; j < n; ++j) P[r][j] = g.cQ[(row0 + r) * n + j];
    colsT_x_smem<R, n>(g.Ah, row0, g.M1, P);
  }
  __syncwarp();   // Ys / M1 / Ks are complete (and free for the next writer)
  return bad;
}

template <int R, int n, int m>
__device__ __forceinline__ void closed_loop_rows(const GroupMem& g, int row0, double (&Mr)[R][n]) {
#pragma unroll
  for (int r = 0; r < R; ++r)
#pragma unroll
    for (int j = 0; j < n; ++j) {
      double acl = g.cA[(row0 + r) * n + j];
#pragma unroll
      for (int i = 0; i < m; ++i) acl = fma(g.cB[(row0 + r) * m + i], g.Ks[i * n + j], acl);
      Mr[r][j] = acl;
    }
}

template <int R, int n>
__device__ __forceinline__ double quad_rows(const GroupMem& g, int row0, const double (&P)[R][n]) {
  double acc = 0.0;
#pragma unroll
  for (int r = 0; r < R; ++r) {
    double row = 0.0;
#pragma unroll
    for (int j = 0; j < n; ++j) row = fma(P[r][j], g.Xs[j], row);
    acc = fma(g.Xs[row0 + r], row, acc);
  }
  return acc;
}

// Closed-loop figures of the gain in Ks on the true plant, written to column h of the outputs by the group's lane 0.
template <int n, int m, int L>
__device__ __forceinline__ void closed_loop_emit(const lq::Problem<n, m>& pb, const EvalArgs& a, const GroupMem& g,
                                                 int row0, int gl, bool live, int64_t s, int h, int flags,
                                                 double v_exp, double vn) {
  constexpr int R = n / L;
  // ---- spectral radius: rho = lim max|Acl^(2^k)|^(1/2^k) by kRhoK2 squarings with exact power-of-two rescaling
  //      (log2 rho ~ sum_k 2^-k e_k + 2^-K log2 max|N_K|, N_k the stored rescaled power and e_k its binary exponent);
  //      accepted when the estimates after kRhoK1 and kRhoK2 squarings agree to 5e-10 (the same rule as K4a), else
  //      the group's lane 0 runs the Hessenberg + shifted-QR code on the closed loop.
  double rho = 0.0;
  bool need_qr = false;
  {
    double C[R][n];
    closed_loop_rows<R, n, m>(g, row0, C);
    uint32_t mh = 0;
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int j = 0; j < n; ++j) mh = lq::umax32(mh, lq::abs_hi(C[r][j]));
    mh = g_max<L>(mh);
    double lacc = 0.0, wgt = 1.0, est1 = 0.0, rr_prev = 0.0;
    bool zero = false, fail = false, accepted = false;
    int streak = -1;                                    // -1: no previous candidate
#ifdef LQ_GROUP_STATS
    int kk_acc = 0, kk_end = 0;
#endif
    for (int kk = 0; kk < kRhoK2; ++kk) {
#ifdef LQ_GROUP_STATS
      kk_end = kk;
#endif
      if ((mh >> 20) == 0x7ffu) fail = true;
      if ((mh >> 20) == 0) zero = true;                 // zero (or denormal) power: nilpotent closed loop, rho = 0
      if (__all_sync(kFull, accepted || zero || fail)) break;
      const int e = (zero || fail) ? 0 : (int)(mh >> 20) - 1023;
      const double sc = __hiloint2double((1023 - e) << 20, 0);
      double Nr[R][n];
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int j = 0; j < n; ++j) Nr[r][j] = C[r][j] * sc;
      double* buf = (kk & 1) ? g.M1 : g.M2;             // ping-pong: one __syncwarp per squaring
      store_rows<R, n>(buf, row0, Nr);
      __syncwarp();
      rows_x_smem<R, n, n, false>(Nr, buf, C);
      lacc = fma(wgt, (double)e, lacc);
      // Early acceptance through the two dominant eigenvalues. With X = Acl^p / 2^(p lacc) (p = 2^kk, the rows in Nr)
      // and X^2 (in C): t = tr X = sum lambda_i^p, t' = tr X^2, d = (t^2 - t') / 2 = e_2(lambda^p). When one real
      // eigenvalue, a +- pair or a complex pair dominates, its p-th powers are the roots of z^2 - t z + d up to
      // (|lambda_3| / |lambda_1|)^p, so rho^p = sqrt(d) (complex roots) or the larger root modulus. A candidate is
      // taken only if it is not tiny against max|X| in [1, 2) (an ill-conditioned or defective dominant eigenvalue
      // leaves rounding noise in the traces) and the roots are not nearly double; it is ACCEPTED when two successive
      // squarings reproduce it, r_k 2^(e_k) = r_(k-1)^2 to kRhoEta (the model error then is below kRhoEta in
      // rho^p, i.e. kRhoEta / p in rho, and p is large enough that this is < 2e-10). Everything else runs all
      // kRhoK2 squarings to the norm-based two-estimate test.
      {
        double tau = 0.0, taup = 0.0;
#pragma unroll
        for (int q = 0; q < L; ++q)
          if (gl == q) {
#pragma unroll
            for (int r = 0; r < R; ++r) { tau += Nr[r][q * R + r]; taup += C[r][q * R + r]; }
          }
        tau = g_sum<L>(tau);
        taup = g_sum<L>(taup);
        const double t2 = tau * tau;
        const double d = 0.5 * (t2 - taup), disc = fma(2.0, taup, -t2);
        const double rr = (disc < 0.0) ? sqrt(d) : 0.5 * (fabs(tau) + sqrt(disc));
        const bool cand = (rr > kRhoMinRoot) && (rr < 1e300) && !(fabs(disc) < 1e-4 * t2);
        if (cand) {
          // r_k 2^(e_k) = r_(k-1)^2 up to kRhoEta (relative)
          const double want = rr_prev * rr_prev * __hiloint2double((1023 - e) << 20, 0);
          const bool same = (streak >= 0) && fabs(rr - want) <= kRhoEta * rr;
          if (same && streak >= 1 && kRhoEta * wgt <= 2e-10 && !accepted && !zero && !fail) {
            accepted = true;
#ifdef LQ_GROUP_STATS
            kk_acc = kk + 1;
#endif
            rho = exp(fma(lacc, 0.6931471805599453, wgt * log(rr)));
          }
          streak = same ? streak + 1 : 0;
          rr_prev = rr;
        } else {
          streak = -1;
        }
      }
      wgt *= 0.5;
      mh = 0;
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int j = 0; j < n; ++j) mh = lq::umax32(mh, lq::abs_hi(C[r][j]));
      mh = g_max<L>(mh);
      if (kk + 1 == kRhoK1 || kk + 1 == kRhoK2) {
        double mx = 0.0;
#pragma unroll
        for (int r = 0; r < R; ++r)
#pragma unroll
          for (int j = 0; j < n; ++j) mx = fmax(mx, fabs(C[r][j]));
        mx = g_fmax<L>(mx);
        const double est = fma(lacc, 0.6931471805599453, wgt * log(mx));
        if (kk + 1 == kRhoK1) est1 = est;
        else if (!accepted) {
          rho = exp(est);
          if (!(fabs(rho - exp(est1)) <= 5e-10 * rho)) need_qr = true;
        }
      }
    }
#ifdef LQ_GROUP_STATS
    flags |= (kk_acc << 16) | (kk_end << 24);           // development: squarings to acceptance / to the warp's exit
#endif
    if (accepted) { zero = false; fail = false; need_qr = false; }
    else {
      if ((mh >> 20) == 0x7ffu || (mh >> 20) == 0) { if (!zero) fail = true; }
      if (zero && !fail) { rho = 0.0; need_qr = false; }
      if (fail) need_qr = true;
    }
    __syncwarp();
  }
  double Mr[R][n];
  closed_loop_rows<R, n, m>(g, row0, Mr);
  store_rows<R, n>(g.M1, row0, Mr);                     // the closed loop again (QR fallback, Lyapunov doubling)
  __syncwarp();
  int eig_ok = 1;
  if (__any_sync(kFull, need_qr)) {
    double rq = 0.0;
    if (gl == 0 && need_qr) {
      double Af[n * n];
#pragma unroll
      for (int e = 0; e < n * n; e += 2) {
        const double2 v = *reinterpret_cast<const double2*>(g.M1 + e);
        Af[e] = v.x;
        Af[e + 1] = v.y;
      }
      bool ok;
      rq = spectral_radius_call<n>(Af, &ok);
      eig_ok = ok ? 1 : 0;
    }
    rq = __shfl_sync(kFull, rq, (threadIdx.x & 31) - gl);
    eig_ok = __shfl_sync(kFull, eig_ok, (threadIdx.x & 31) - gl);
    if (need_qr) rho = rq;
  }
  if (!eig_ok) flags |= lq::FLAG_EIG_NOCONV;

  // ---- J_inf = x0' S x0, S = W + Acl' S Acl by squared doubling (S_{j+1} = S_j + M_j' S_j M_j, M_{j+1} = M_j^2)
  double S[R][n];
  {
    double RK[m * n];
#pragma unroll
    for (int i = 0; i < m; ++i)
#pragma unroll
      for (int j = 0; j < n; ++j) {
        double acc = 0.0;
#pragma unroll
        for (int q = 0; q < m; ++q) acc = fma(pb.R[i * m + q], g.Ks[q * n + j], acc);
        RK[i * n + j] = acc;
      }
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int j = 0; j < n; ++j) {
        double w = g.cQ[(row0 + r) * n + j];
#pragma unroll
        for (int i = 0; i < m; ++i) w = fma(g.Ks[i * n + row0 + r], RK[i * n + j], w);
        S[r][j] = w;
      }
  }
  double J = HUGE_VAL;
  const bool stable = rho < 1.0;
  if (!stable) flags |= lq::FLAG_UNSTABLE;
  bool done = !stable, lyap_ok = true;
  for (int it = 0; it < 64; ++it) {
    if (!__any_sync(kFull, !done)) break;
    double T[R][n];
    {
      double SM[R][n];
      rows_x_smem<R, n, n, false>(S, g.M1, SM);
      store_rows<R, n>(g.M2, row0, SM);
    }
    __syncwarp();
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int j = 0; j < n; ++j) T[r][j] = 0.0;
    colsT_x_smem<R, n>(g.M1, row0, g.M2, T);
    uint32_t thi = 0, shi = 0;
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int j = 0; j < n; ++j) {
        thi = lq::umax32(thi, lq::abs_hi(T[r][j]));
        T[r][j] += S[r][j];
        shi = lq::umax32(shi, lq::abs_hi(T[r][j]));
      }
    thi = g_max<L>(thi);
    shi = g_max<L>(shi);
    bool conv = false;
    if (!done) {
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int j = 0; j < n; ++j) S[r][j] = T[r][j];
      if ((thi >> 20) == 0x7ffu || (shi >> 20) == 0x7ffu) { lyap_ok = false; done = true; }
      else if (!(lq::from_abs_hi(thi) > 1e-18 * lq::from_abs_hi(shi))) conv = true;
    }
    done = done || conv;
    if (!__any_sync(kFull, !done)) break;
    double M2r[R][n];
    rows_x_smem<R, n, n, false>(Mr, g.M1, M2r);
    uint32_t mhi = 0;
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int j = 0; j < n; ++j) mhi = lq::umax32(mhi, lq::abs_hi(M2r[r][j]));
    mhi = g_max<L>(mhi);
    __syncwarp();                                     // every read of M1 is done
    if (!done) {
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int j = 0; j < n; ++j) Mr[r][j] = M2r[r][j];
      store_rows<R, n>(g.M1, row0, Mr);
      const double mb = lq::from_abs_hi(mhi) * 1.000002;
      if ((double)(n * n) * mb * mb <= 1e-18) done = true;
    }
    __syncwarp();
  }
  if (!done) lyap_ok = false;
  {
    // (the reduction is a full-mask shuffle: every group runs it, stable or not)
    const double Jq = g_sum<L>(quad_rows<R, n>(g, row0, S));
    if (stable) {
      if (!lyap_ok) flags |= lq::FLAG_LYAP_NOCONV;
      J = Jq;
      if (!(fabs(J) <= 1.79e308)) flags |= lq::FLAG_NONFINITE;
    }
  }
  if (gl == 0) {
    double K[m * n];
#pragma unroll
    for (int e = 0; e < m * n; ++e) K[e] = g.Ks[e];
    double JT = 0.0;
    if (a.T > 0) {  // finite-T cost exactly as accumulated by utils_class.py:261,282-283
      double x[n], xn[n], u[m];
#pragma unroll
      for (int i = 0; i < n; ++i) x[i] = g.Xs[i];
      double cost = lq::quad<n>(x, pb.Q, x);
      for (int t = 0; t < a.T; ++t) {
        lq::mv<m, n>(K, x, u);
#pragma unroll
        for (int i = 0; i < n; ++i) {
          double acc = 0.0;
#pragma unroll
          for (int j = 0; j < n; ++j) acc = fma(pb.A[i * n + j], x[j], acc);
#pragma unroll
          for (int j = 0; j < m; ++j) acc = fma(pb.B[i * m + j], u[j], acc);
          xn[i] = acc;
        }
        cost += lq::quad<n>(xn, pb.Q, xn);
        cost += lq::quad<m>(u, pb.R, u);
#pragma unroll
        for (int i = 0; i < n; ++i) x[i] = xn[i];
      }
      JT = cost;
    }
    if (live) {
      const int64_t o = (int64_t)h * a.ld + s;
      if (a.J) stg_stream(a.J + o, J);
      if (a.rho) stg_stream(a.rho + o, rho);
      if (a.ratio) stg_stream(a.ratio + o, J / v_exp);
      if (a.Vn) stg_stream(a.Vn + o, vn);
      if (a.JT) stg_stream(a.JT + o, JT);
      if (a.flags) a.flags[o] = flags;
      if (a.K0) {
#pragma unroll
        for (int e = 0; e < m * n; ++e) stg_stream(a.K0 + ((int64_t)h * (m * n) + e) * a.ld + s, K[e]);
      }
    }
  }
  __syncwarp();   // M1 / M2 / Ks are free for the next stage
}

// NESTED = false: one horizon per sample and no V_N — the cost-to-go dies before the closed-loop phase;
// NESTED = true: horizons N_min..N_max (or V_N wanted) — it waits in the arena while the closed loop is evaluated.
// lqmpc_eval_seeded on lane groups: the operands are not read but drawn in the kernel (sampler.cuh: seeded_sample — the
// stream is addressed by (global sample index, pair index), so every lane draws exactly its own rows)
struct SeedArgs {
  uint64_t seed;
  int64_t first;
  double e_A, e_B;
};

template <int n, int m, int L, bool NESTED, int MINB, bool SEEDED>
__global__ void __launch_bounds__((GroupLayout<n, m, L, NESTED>::kThreads), MINB)
    group_eval_kernel(const __grid_constant__ lq::Problem<n, m> pb, const __grid_constant__ EvalArgs a,
                      const __grid_constant__ SeedArgs sd) {
  using Lay = GroupLayout<n, m, L, NESTED>;
  constexpr int R = Lay::R;
  extern __shared__ __align__(16) double sm[];
  const int gl = threadIdx.x % L;                       // lane within the group
  const int gi = threadIdx.x / L;                       // group within the CTA
  const int row0 = gl * R;
  const int64_t s_raw = (int64_t)blockIdx.x * Lay::kGroups + gi;
  const bool live = s_raw < a.S;
  const int64_t s = live ? s_raw : a.S - 1;             // tail groups redo the last sample and store nothing

  {
    double* cA = sm + Lay::oA;
    double* cB = sm + Lay::oB;
    double* cQ = sm + Lay::oQ;
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) { cA[e] = pb.A[e]; cQ[e] = pb.Q[e]; }
    for (int e = threadIdx.x; e < n * m; e += blockDim.x) cB[e] = pb.B[e];
  }
  double* ar = sm + Lay::kConst + gi * Lay::kArena;
  GroupMem g;
  g.cA = sm + Lay::oA; g.cB = sm + Lay::oB; g.cQ = sm + Lay::oQ;
  g.Ah = ar + Lay::aAh; g.Bh = ar + Lay::aBh; g.M1 = ar + Lay::aM1; g.M2 = ar + Lay::aM2;
  g.Ys = ar + Lay::aY; g.Ks = ar + Lay::aK; g.Xs = ar + Lay::aX; g.Ps = ar + Lay::aP;
  __syncthreads();

  // ---- operands: every lane fetches its own rows of A^ = A + dA, B^ = B + dB and its entries of x0
  double Bhr[R][m], P[R][n];
  if (SEEDED) {
    static_assert(!SEEDED || ((R * n) % 2 == 0 && (R * m) % 2 == 0 && (n * n) % 2 == 0), "seeded draw: whole pairs per lane");
    const uint32_t k0 = (uint32_t)sd.seed, k1 = (uint32_t)(sd.seed >> 32) ^ lq::kSeededStream;
    const int64_t gs = sd.first + s;
    const uint32_t c0 = (uint32_t)gs, c1 = (uint32_t)((uint64_t)gs >> 32);
    constexpr int nu = n * n + n * m;
#pragma unroll
    for (int q = 0; q < R * n; q += 2) {                 // own rows of dA: elements row0 n + q, + 1
      const int e = row0 * n + q;
      const lq::Philox4 x = lq::philox4x32_10(c0, c1, (uint32_t)(e >> 1), 0u, k0, k1);
      g.Ah[e] = g.cA[e] + sd.e_A * lq::philox_symm(x.v[0], x.v[1]);
      g.Ah[e + 1] = g.cA[e + 1] + sd.e_A * lq::philox_symm(x.v[2], x.v[3]);
    }
#pragma unroll
    for (int q = 0; q < R * m; q += 2) {                 // own rows of dB: elements n n + row0 m + q, + 1
      const int e = row0 * m + q;
      const lq::Philox4 x = lq::philox4x32_10(c0, c1, (uint32_t)((n * n + e) >> 1), 0u, k0, k1);
      const double v0 = g.cB[e] + sd.e_B * lq::philox_symm(x.v[0], x.v[1]);
      const double v1 = g.cB[e + 1] + sd.e_B * lq::philox_symm(x.v[2], x.v[3]);
      Bhr[q / m][q % m] = v0;
      Bhr[(q + 1) / m][(q + 1) % m] = v1;
      g.Bh[e] = v0;
      g.Bh[e + 1] = v1;
    }
    for (int pp = row0 >> 1; pp <= (row0 + R - 1) >> 1; ++pp) {      // own entries of x0 (Box-Muller pairs)
      const lq::Philox4 x = lq::philox4x32_10(c0, c1, (uint32_t)((nu + 1) / 2 + pp), 0u, k0, k1);
      const double u = ((double)(x.v[0] >> 5) * 67108864.0 + (double)(x.v[1] >> 6) + 1.0) * (1.0 / 9007199254740992.0);
      const double v = ((double)(x.v[2] >> 5) * 67108864.0 + (double)(x.v[3] >> 6)) * (1.0 / 9007199254740992.0);
      const double rr = sqrt(-2.0 * log(u)), th = 6.283185307179586476925286766559 * v;
      if (2 * pp >= row0 && 2 * pp < row0 + R) g.Xs[2 * pp] = rr * cos(th);
      if (2 * pp + 1 >= row0 && 2 * pp + 1 < row0 + R) g.Xs[2 * pp + 1] = rr * sin(th);
    }
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int j = 0; j < n; ++j) P[r][j] = pb.Pt[(row0 + r) * n + j];
  } else {
#pragma unroll
    for (int r = 0; r < R; ++r) {
#pragma unroll
      for (int j = 0; j < n; ++j) {
        const int e = (row0 + r) * n + j;
        g.Ah[e] = g.cA[e] + ldg_stream(a.dA + (int64_t)e * a.ld + s);
        P[r][j] = pb.Pt[e];
      }
#pragma unroll
      for (int j = 0; j < m; ++j) {
        const int e = (row0 + r) * m + j;
        const double v = g.cB[e] + ldg_stream(a.dB + (int64_t)e * a.ld + s);
        Bhr[r][j] = v;
        g.Bh[e] = v;
      }
      g.Xs[row0 + r] = ldg_stream(a.x0 + (int64_t)(row0 + r) * a.ld + s);
    }
  }
  __syncwarp();
  double v_exp;
  {
    double x0[n];
#pragma unroll
    for (int e = 0; e < n; ++e) x0[e] = g.Xs[e];
    v_exp = lq::quad<n>(x0, pb.Pexp, x0);
  }

  int sticky = 0;
  if (!NESTED) {
    for (int k = 1; k < a.N_max; ++k) sticky |= riccati_stage<n, m, L>(pb, g, row0, Bhr, P, false, true);
    sticky |= riccati_stage<n, m, L>(pb, g, row0, Bhr, P, true, false);
    closed_loop_emit<n, m, L>(pb, a, g, row0, gl, live, s, 0, sticky, v_exp, 0.0);
  } else {
    const bool want_vn = a.Vn != nullptr;
    for (int k = 1; k <= a.N_max; ++k) {
      const bool emit = (k >= a.N_min);
      sticky |= riccati_stage<n, m, L>(pb, g, row0, Bhr, P, emit, k < a.N_max || want_vn);
      if (!emit) continue;
      const double vn = want_vn ? g_sum<L>(quad_rows<R, n>(g, row0, P)) : 0.0;
      store_rows<R, n>(g.Ps, row0, P);                  // own rows only: no other lane reads them
      closed_loop_emit<n, m, L>(pb, a, g, row0, gl, live, s, k - a.N_min, sticky, v_exp, vn);
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int j = 0; j < n; j += 2) {
          const double2 v = *reinterpret_cast<const double2*>(g.Ps + (row0 + r) * n + j);
          P[r][j] = v.x;
          P[r][j + 1] = v.y;
        }
    }
  }
}

template <int n, int m, int L, bool NESTED, int MINB, bool SEEDED>
int launch_group_t(lqmpc_ctx* ctx, const EvalArgs& a, const SeedArgs& sd, cudaStream_t stream) {
  using Lay = GroupLayout<n, m, L, NESTED>;
  const lq::Problem<n, m>& pb = *reinterpret_cast<const lq::Problem<n, m>*>(ctx->pb);
  const int64_t blocks = (a.S + Lay::kGroups - 1) / Lay::kGroups;
  if (blocks > 0x7fffffffLL) return lq_set_error(ctx, LQMPC_EINVAL, "batch too large for one launch");
  if (a.S <= 0) return 0;
  int rc = lq_check_cuda(ctx, cudaFuncSetAttribute(group_eval_kernel<n, m, L, NESTED, MINB, SEEDED>,
                                                   cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Lay::kSmemBytes),
                         "group_eval_kernel smem attribute");
  if (rc) return rc;
  group_eval_kernel<n, m, L, NESTED, MINB, SEEDED><<<(unsigned)blocks, Lay::kThreads, Lay::kSmemBytes, stream>>>(pb, a, sd);
  ctx->launches++;
  return lq_check_cuda(ctx, cudaGetLastError(), "group_eval_kernel launch");
}

template <int n, int m, int L, int MINB, bool SEEDED = false>
int launch_group(lqmpc_ctx* ctx, const EvalArgs& a, cudaStream_t stream, const SeedArgs& sd = SeedArgs{}) {
  if (a.N_min == a.N_max && a.Vn == nullptr) return launch_group_t<n, m, L, false, MINB, SEEDED>(ctx, a, sd, stream);
  return launch_group_t<n, m, L, true, MINB, SEEDED>(ctx, a, sd, stream);
}

}  // namespace

bool lq_group_supported(int n, int m) { return (n == 8 && m == 2) || (n == 6 && m == 2); }

int lq_launch_eval_group(lqmpc_ctx* ctx, const EvalArgs& a, cudaStream_t stream) {
  // n = 8: 4 lanes x 2 rows at 3 CTAs/SM, the fastest of the lane splits and register budgets measured (DESIGN.md §4)
  if (ctx->n == 8 && ctx->m == 2) return launch_group<8, 2, 4, 3>(ctx, a, stream);
  if (ctx->n == 6 && ctx->m == 2) return launch_group<6, 2, 2, 2>(ctx, a, stream);
  return lq_set_error(ctx, LQMPC_EINVAL, "lane-group K1 is built for 6x2 and 8x2");
}

int lq_launch_eval_group_seeded(lqmpc_ctx* ctx, const EvalArgs& a, uint64_t seed, int64_t first, double e_A, double e_B) {
  const SeedArgs sd{seed, first, e_A, e_B};
  if (ctx->n == 8 && ctx->m == 2) return launch_group<8, 2, 4, 3, true>(ctx, a, ctx->stream, sd);
  if (ctx->n == 6 && ctx->m == 2) return launch_group<6, 2, 2, 2, true>(ctx, a, ctx->stream, sd);
  return lq_set_error(ctx, LQMPC_EINVAL, "lane-group K1 is built for 6x2 and 8x2");
}
