// clqr.cuh — exact solution of the input-box-constrained finite-horizon LQ problem, one sample per thread.
//
// Reference semantics: LQ_MPC_Controller.solve (utils_class.py:48-91) with zero references builds
//     min_{u_0..u_{N-1}}  sum_{k<N} ( x_{k+1}' W_{k+1} x_{k+1} + u_k' R u_k ),  W_k = Q (k<N), W_N = P,
//     x_{k+1} = A^ x_k + B^ u_k,   lo <= u_k <= hi          (F_u u <= 1 with F_u = [diag(1/hi); diag(1/lo)], :81)
// and returns u_0 and V_N = optimum + x0' Q x0 (:91).  The reference hands this to cvxpy; the minimiser of a
// strictly convex QP is unique, so any exact method gives the same u_0 / V_N.
//
// Method (designed for the GPU, not a translation of a dense QP solver): a primal active-set iteration whose
// equality-constrained sub-problems are solved by an *affine Riccati sweep* — clamped inputs are constants, free
// inputs are optimised stage by stage — so one iteration costs O(N n^3) flops on register-resident n x n blocks
// instead of a dense (N m)^3 factorisation, and the KKT multipliers come from a costate sweep over the stored
// trajectory. If the unconstrained plan is feasible it is returned at once (it is the QP minimiser).
//
// Per-thread scratch lives in a strided workspace view (element e at p[e*stride]): coalesced across the warp on
// the device, contiguous on the host test harness.
#pragma once
#include "riccati.cuh"

namespace lq {

struct WsView {
  double* p;
  int64_t stride;
  LQ_HD double& operator[](int64_t e) const { return p[e * stride]; }
};

// Stage loops over the strided workspace are chains of dependent steps whose first instruction waits for a global
// load (ncu, round 2: the first use of a stage's gain held 21 % of the sweep kernels' stall samples at 3 warps per
// scheduler). The addresses do not depend on the data, so the loads of stage k + PF are issued while stage k is
// computed: `fetch(k, v)` fills v[0..W) for stage k, `body(k, v)` consumes it; stages run in order 0..N-1. The
// lookahead is a register ring, hence only for the small dimensions; PF = 0 keeps the plain loop.
#ifndef LQ_K2_PF_SMALL
#define LQ_K2_PF_SMALL 1      // n m <= 2 (the shipped 2-state example)
#endif
#ifndef LQ_K2_PF_MID
#define LQ_K2_PF_MID 1        // n m <= 4
#endif
// Measured on the sweep's two launches (scripts/k2_probe.py, 1e6 samples, N = 5 / 10 / 25 / 50 summed), (n, m) = (2, 1):
// depth 1 at 3 CTAs/SM (160 registers, no spills) 9.99 ms ring solves / 3.05 ms closed loops; no lookahead 13.9 / 3.6-4.0;
// depth 2: 12.0 / 3.45; depth 4: 13.9 / 3.6 at 214 registers, 16.4 / 4.7 held to 168 (the ring spills); 4 or 5 CTAs/SM
// (128 / 96 registers) lose to their spills at every depth.
template <int n, int m>
struct StagePrefetch {
  static constexpr int depth = (n * m <= 2) ? LQ_K2_PF_SMALL : ((n * m <= 4) ? LQ_K2_PF_MID : 0);
};

template <int W, int PF, class Fetch, class Body>
LQ_HD void staged_loop(int N, Fetch fetch, Body body) {
  if (PF == 0) {
    for (int k = 0; k < N; ++k) {
      double v[W];
      fetch(k, v);
      body(k, v);
    }
    return;
  }
  constexpr int D = (PF > 0) ? PF : 1;
  double ring[D][W];
  LQ_UNROLL for (int q = 0; q < D; ++q)
    if (q < N) fetch(q, ring[q]);
  for (int k0 = 0; k0 < N; k0 += D) {
    LQ_UNROLL for (int q = 0; q < D; ++q) {
      const int k = k0 + q;
      if (k < N) {
        double v[W];
        LQ_UNROLL for (int e = 0; e < W; ++e) v[e] = ring[q][e];
        if (k + D < N) fetch(k + D, ring[q]);
        body(k, v);
      }
    }
  }
}

// Shared references of LQ_MPC_Controller.solve (utils_class.py:48-81): x_ref[:, i] is the reference of x_{i+1},
// u_ref[:, i] of u_i (row-major, leading dimension ld >= N; only the first N columns are read). NULL = zeros, which is
// what every caller in the reference passes; non-zero references make the law affine and disable the Riccati fast path.
struct Refs {
  const double* xr = nullptr;
  const double* ur = nullptr;
  int ld = 0;
  LQ_HD bool any() const { return xr != nullptr || ur != nullptr; }
  LQ_HD double x(int i, int k) const { return xr ? xr[i * ld + k] : 0.0; }
  LQ_HD double u(int j, int k) const { return ur ? ur[j * ld + k] : 0.0; }
};

// Working sets of the active-set iterations: one bit per (stage, input component) / (stage, polytope row), 256 bits
// (N m = 240 at BASELINE cfg 5's shape). Word selection is a chain of selects, never a dynamically indexed array,
// so the four words stay in registers.
constexpr int kMaskBits = 256;
struct Mask128 {   // (name kept from the 128-bit first version)
  uint64_t w0 = 0, w1 = 0, w2 = 0, w3 = 0;
  LQ_HD uint64_t word(int b) const { return (b < 128) ? ((b < 64) ? w0 : w1) : ((b < 192) ? w2 : w3); }
  LQ_HD bool test(int b) const { return ((word(b) >> (b & 63)) & 1u) != 0; }
  LQ_HD void put(int b, bool v) {
    const uint64_t bit = (uint64_t)1 << (b & 63);
    uint64_t w = word(b);
    w = v ? (w | bit) : (w & ~bit);
    if (b < 64) w0 = w; else if (b < 128) w1 = w; else if (b < 192) w2 = w; else w3 = w;
  }
  LQ_HD void set(int b) { put(b, true); }
  LQ_HD void clear(int b) { put(b, false); }
  LQ_HD static int top64(uint64_t w) {
#if defined(__CUDA_ARCH__)
    return 63 - __clzll((long long)w);
#else
    return 63 - __builtin_clzll(w);
#endif
  }
  // index of the highest set bit, -1 when empty
  LQ_HD int top_bit() const {
    if (w3) return 192 + top64(w3);
    if (w2) return 128 + top64(w2);
    if (w1) return 64 + top64(w1);
    if (w0) return top64(w0);
    return -1;
  }
};

#ifndef LQ_K2_STORED_P
#define LQ_K2_STORED_P 12
#endif
constexpr int kStoredCostToGo = LQ_K2_STORED_P;
template <int n, int m>
struct ClqrLayout {
  int N, kp;
  int64_t oKu, oKc, okc, oz, ozs, oxs, oP, total;
  static constexpr int np = n * (n + 1) / 2;      // packed upper triangle of a symmetric n x n matrix
  LQ_HD explicit ClqrLayout(int N_) : N(N_) {
    oKu = 0;
    oKc = oKu + (int64_t)N * m * n;
    okc = oKc + (int64_t)N * m * n;
    oz = okc + (int64_t)N * m;
    ozs = oz + (int64_t)N * m;
    oxs = ozs + (int64_t)N * m;
    // unconstrained cost-to-go S_k (packed) of the FIRST kp stages only: a constrained sweep restarts from S_{klast+1},
    // and in the sweeps the inputs saturate during the first steps; a working set reaching a later stage takes the full
    // N-stage sweep instead (exact either way). Storing all N stages was 1.2 of the 4.9 kB written per sample at N = 50.
    kp = (N < kStoredCostToGo) ? N : kStoredCostToGo;
    oP = oxs + (int64_t)(N + 1) * n;
    total = oP + (int64_t)kp * np;
  }
};

template <int n, int m>
LQ_HD int64_t clqr_ws_doubles(int N) {
  return ClqrLayout<n, m>(N).total;
}

// Horizon-range workspace (plan_prepare_range): the layout of an N_max-stage solve with the cost-to-go of EVERY stage
// stored, so that each horizon N <= N_max finds its S_{klast+1} at stage klast + 1 + (N_max - N).
template <int n, int m>
LQ_HD int64_t clqr_range_ws_doubles(int N_max) {
  const ClqrLayout<n, m> L(N_max);
  return L.oP + (int64_t)N_max * L.np;
}

// Per-sample model of the controller (estimated system) + weights, in registers.
template <int n, int m>
struct Plan {
  double Ah[n * n], Bh[n * m];
  double P0[n * n];  // unconstrained horizon-N cost-to-go: V_N = x0' P0 x0 when no bound is active
  // unconstrained first-stage gain: the certificate's fast path reads it every closed-loop step. Register-resident for
  // the small dimensions only (the n >= 6 instantiations already spill; they re-read it from the workspace).
  static constexpr bool kHoldK0 = (n * m <= 8);
  double K0[kHoldK0 ? m * n : 1];
  double cstar;      // feasibility certificate: x0' P0 x0 <= cstar  =>  the whole unconstrained plan stays inside the box
};

// Unconstrained Riccati sweep; stores the gains K_k (u_k = K_k x_k) for k = 0..N-1 in the workspace.
template <int n, int m>
LQ_HD int plan_prepare(const Problem<n, m>& pb, Plan<n, m>& pl, int N, const WsView& ws, bool certificate = true) {
  const ClqrLayout<n, m> L(N);
  double P[n * n];
  LQ_UNROLL for (int i = 0; i < n * n; ++i) P[i] = pb.Pt[i];
  RicStage<n, m> st;
  int flags = 0;
  for (int k = N - 1; k >= 0; --k) {
    riccati_factor<n, m>(P, pl.Bh, pb.R, st);
    if (!st.ok) flags |= FLAG_CHOL_FAIL;
    double K[m * n];
    riccati_gain<n, m>(st, pl.Ah, K);
    LQ_UNROLL for (int e = 0; e < m * n; ++e) ws[L.oKu + (int64_t)k * (m * n) + e] = K[e];
    if (Plan<n, m>::kHoldK0 && k == 0) {
      LQ_UNROLL for (int e = 0; e < m * n; ++e) pl.K0[Plan<n, m>::kHoldK0 ? e : 0] = K[e];
    }
    riccati_update<n, m>(st, pl.Ah, pb.Q, P);
    // S_k: where a constrained sweep may start when every clamped input sits at an earlier stage (clqr_backward)
    if (k < L.kp) {
      int e = 0;
      LQ_UNROLL for (int i = 0; i < n; ++i)
        LQ_UNROLL for (int j = i; j < n; ++j) { ws[L.oP + (int64_t)k * L.np + e] = P[i * n + j]; ++e; }
    }
  }
  LQ_UNROLL for (int i = 0; i < n * n; ++i) pl.P0[i] = P[i];
  // Feasibility certificate of the unconstrained plan. x_k = Phi_k x_0 with Phi_{k+1} = (A^ + B^ K_k) Phi_k, so the
  // planned input is u_k = (K_k Phi_k) x_0 =: g_k x_0 and, by Cauchy-Schwarz in the P0 metric,
  //     |u_{k,j}| <= sqrt(g_{k,j} P0^-1 g_{k,j}') sqrt(x_0' P0 x_0).
  // Hence x_0' P0 x_0 <= cstar := min_{k,j} b_j^2 / (g_{k,j} P0^-1 g_{k,j}'), b_j = min(-lo_j, hi_j), guarantees that no
  // planned input leaves the box: the solve returns the unconstrained answer from ONE quadratic form (which it needs
  // anyway: it is V_N) instead of an N-stage rollout. Sufficient, not necessary — outside the ellipsoid the rollout
  // decides as before, so nothing is approximated. In the closed loops of the sweeps the state enters the ellipsoid
  // after the first few steps. (1 - 1e-9 margin against rounding in cstar itself.)
  // `certificate = false` (the ring solves: a handful of states per sample, chosen OUTSIDE the region where the
  // unconstrained law is feasible) skips the N-stage construction — it costs about 1.7 clipped rollouts — and leaves
  // cstar = -1: every solve then decides feasibility by its rollout, exactly as before the certificate existed.
  pl.cstar = -1.0;
  if (pb.has_bounds && certificate) {
    double Lc[n * n], Lci[n];
    LQ_UNROLL for (int i = 0; i < n * n; ++i) Lc[i] = P[i];
    bool okc = chol_inv<n>(Lc, Lci);
    double bmin2[m];
    LQ_UNROLL for (int j = 0; j < m; ++j) {
      const double b = dmin(-pb.ulo[j], pb.uhi[j]);
      okc = okc && (b > 0.0);
      bmin2[j] = b * b;
    }
    if (okc) {
      double cs = HUGE_VAL;
      double Phi[n * n];
      LQ_UNROLL for (int i = 0; i < n; ++i)
        LQ_UNROLL for (int j = 0; j < n; ++j) Phi[i * n + j] = (i == j) ? 1.0 : 0.0;
      staged_loop<m * n, StagePrefetch<n, m>::depth>(N, [&](int k, double* v) {
        LQ_UNROLL for (int e = 0; e < m * n; ++e) v[e] = ws[L.oKu + (int64_t)k * (m * n) + e];
      }, [&](int k, const double* K) {
        double g[m * n], Acl[n * n], Pn[n * n];
        mm<m, n, n>(K, Phi, g);
        LQ_UNROLL for (int j = 0; j < m; ++j) {             // y = L^-1 g_j' (forward substitution), q = y'y = g_j P0^-1 g_j'
          double y[n], q = 0.0;
          LQ_UNROLL for (int i = 0; i < n; ++i) {
            double acc = g[j * n + i];
            LQ_UNROLL for (int r = 0; r < i; ++r) acc = fma(-Lc[i * n + r], y[r], acc);
            y[i] = acc * Lci[i];
            q = fma(y[i], y[i], q);
          }
          if (bmin2[j] < 1e300 && q > 0.0) cs = dmin(cs, bmin2[j] / q);
        }
        if (k + 1 < N) {
          LQ_UNROLL for (int i = 0; i < n; ++i)
            LQ_UNROLL for (int j = 0; j < n; ++j) {
              double acc = pl.Ah[i * n + j];
              LQ_UNROLL for (int r = 0; r < m; ++r) acc = fma(pl.Bh[i * m + r], K[r * n + j], acc);
              Acl[i * n + j] = acc;
            }
          mm<n, n, n>(Acl, Phi, Pn);
          LQ_UNROLL for (int i = 0; i < n * n; ++i) Phi[i] = Pn[i];
        }
      });
      if (cs == cs) pl.cstar = cs * (1.0 - 1e-9);
    }
  } else if (!pb.has_bounds) {
    pl.cstar = HUGE_VAL;             // no input bounds at all: every plan is feasible
  }
  return flags;
}

// Unconstrained sweep of N_max stages for a whole horizon range. The law of horizon N at stage k is the Riccati iterate
// with N - k stages to go, i.e. stage k + (N_max - N) of this sweep: one sweep holds the gains and cost-to-go of every
// N <= N_max, computed by the same operations in the same order as plan_prepare(N). Stores every gain and every S_k
// (the workspace of clqr_range_ws_doubles) and returns the stages-to-go of the first failed factorisation (N_max + 1:
// none), so that horizon N carries FLAG_CHOL_FAIL iff that number is <= N. No certificate (the ring solves skip it).
template <int n, int m>
LQ_HD int plan_prepare_range(const Problem<n, m>& pb, Plan<n, m>& pl, int N_max, const WsView& ws) {
  const ClqrLayout<n, m> L(N_max);
  double P[n * n];
  LQ_UNROLL for (int i = 0; i < n * n; ++i) P[i] = pb.Pt[i];
  RicStage<n, m> st;
  int first_fail = N_max + 1;
  for (int k = N_max - 1; k >= 0; --k) {
    riccati_factor<n, m>(P, pl.Bh, pb.R, st);
    if (!st.ok && first_fail > N_max) first_fail = N_max - k;
    double K[m * n];
    riccati_gain<n, m>(st, pl.Ah, K);
    LQ_UNROLL for (int e = 0; e < m * n; ++e) ws[L.oKu + (int64_t)k * (m * n) + e] = K[e];
    riccati_update<n, m>(st, pl.Ah, pb.Q, P);
    int e = 0;
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = i; j < n; ++j) { ws[L.oP + (int64_t)k * L.np + e] = P[i * n + j]; ++e; }
  }
  pl.cstar = pb.has_bounds ? -1.0 : HUGE_VAL;
  return first_fail;
}

// Plan of horizon N inside a range sweep of N_max stages (koff = N_max - N): P0 is the stored cost-to-go with N stages
// to go (riccati_update leaves P exactly symmetric, so the packed copy restores it bit for bit), K0 the gain there.
template <int n, int m>
LQ_HD void plan_select_horizon(Plan<n, m>& pl, int N_max, int koff, const WsView& ws) {
  const ClqrLayout<n, m> L(N_max);
  int e = 0;
  LQ_UNROLL for (int i = 0; i < n; ++i)
    LQ_UNROLL for (int j = i; j < n; ++j) {
      const double v = ws[L.oP + (int64_t)koff * L.np + e];
      pl.P0[i * n + j] = v; pl.P0[j * n + i] = v; ++e;
    }
  if (Plan<n, m>::kHoldK0) {
    LQ_UNROLL for (int e2 = 0; e2 < m * n; ++e2)
      pl.K0[Plan<n, m>::kHoldK0 ? e2 : 0] = ws[L.oKu + (int64_t)koff * (m * n) + e2];
  }
}

template <int n, int m>
LQ_HD void step_model(const double* A, const double* B, const double* x, const double* u, double* xn) {
  LQ_UNROLL for (int i = 0; i < n; ++i) {
    double acc = 0.0;
    LQ_UNROLL for (int j = 0; j < n; ++j) acc = fma(A[i * n + j], x[j], acc);
    LQ_UNROLL for (int j = 0; j < m; ++j) acc = fma(B[i * m + j], u[j], acc);
    xn[i] = acc;
  }
}

// Backward affine Riccati sweep for the working set (fixed, athi): stores K_k (m x n) and k_k (m).
// `klast` (regulation only, i.e. no references): the highest stage that holds a clamped input. Stages beyond it are
// unconstrained with a purely quadratic cost-to-go, so their law IS the unconstrained one (ws.Ku, zero offset) and the
// sweep starts at klast from the stored S_{klast+1} — O(klast) stages instead of N per active-set iteration (in the
// sweeps of utils_class.py:802-833 the inputs saturate at the first steps only). Pass N - 1 for a full sweep.
// `koff`: stage offset of the stored unconstrained gains and cost-to-go — horizon N inside a range sweep of N + koff
// stages (plan_prepare_range) reads its stage k at k + koff; 0 for a single-horizon plan.
template <int n, int m>
LQ_HD bool clqr_backward(const Problem<n, m>& pb, const Plan<n, m>& pl, int N, const Mask128& fixed, const Mask128& athi,
                         const WsView& ws, const Refs& rf = Refs(), int klast = -2, int koff = 0) {
  const ClqrLayout<n, m> L(N + koff);
  if (klast < -1 || klast > N - 1) klast = N - 1;
  // cost-to-go INCLUDING the state's own stage term: Phi_k(x) = x'S x + 2 s'x + const; Phi_N = (x - r_{N-1})'P(x - r_{N-1})
  double S[n * n], s[n];
  if (klast == N - 1) {
    LQ_UNROLL for (int i = 0; i < n * n; ++i) S[i] = pb.Pt[i];
    LQ_UNROLL for (int i = 0; i < n; ++i) {
      double acc = 0.0;
      LQ_UNROLL for (int j = 0; j < n; ++j) acc = fma(-pb.Pt[i * n + j], rf.x(j, N - 1), acc);
      s[i] = acc;
    }
  } else {
    int e = 0;
    LQ_UNROLL for (int i = 0; i < n; ++i)
      LQ_UNROLL for (int j = i; j < n; ++j) {
        const double v = ws[L.oP + (int64_t)(klast + 1 + koff) * L.np + e];
        S[i * n + j] = v; S[j * n + i] = v; ++e;
      }
    LQ_UNROLL for (int i = 0; i < n; ++i) s[i] = 0.0;
  }
  bool ok = true;
  for (int k = klast; k >= 0; --k) {
    double SB[n * m], G[m * m], Hx[m * (n + 1)];
    mm<n, n, m>(S, pl.Bh, SB);
    LQ_UNROLL for (int i = 0; i < m; ++i)
      LQ_UNROLL for (int j = 0; j <= i; ++j) {
        double acc = pb.R[i * m + j];
        LQ_UNROLL for (int r = 0; r < n; ++r) acc = fma(pl.Bh[r * m + i], SB[r * m + j], acc);
        G[i * m + j] = acc; G[j * m + i] = acc;
      }
    // Hx = [ B^' S A^ | B^' s ]   (m x (n+1))
    LQ_UNROLL for (int i = 0; i < m; ++i) {
      LQ_UNROLL for (int j = 0; j < n; ++j) {
        double acc = 0.0;
        LQ_UNROLL for (int r = 0; r < n; ++r) acc = fma(SB[r * m + i], pl.Ah[r * n + j], acc);
        Hx[i * (n + 1) + j] = acc;
      }
      double acc = 0.0;
      LQ_UNROLL for (int r = 0; r < n; ++r) acc = fma(pl.Bh[r * m + i], s[r], acc);
      LQ_UNROLL for (int r = 0; r < m; ++r) acc = fma(-pb.R[i * m + r], rf.u(r, k), acc);   // - R u_ref_k
      Hx[i * (n + 1) + n] = acc;
    }
    // clamp: substitute constants for the fixed components
    double uc[m];
    bool fx[m];
    LQ_UNROLL for (int j = 0; j < m; ++j) {
      const int bit = k * m + j;
      fx[j] = fixed.test(bit);
      uc[j] = athi.test(bit) ? pb.uhi[j] : pb.ulo[j];
    }
    LQ_UNROLL for (int i = 0; i < m; ++i) {
      if (!fx[i]) {
        LQ_UNROLL for (int j = 0; j < m; ++j)
          if (fx[j]) Hx[i * (n + 1) + n] = fma(G[i * m + j], uc[j], Hx[i * (n + 1) + n]);
      }
    }
    LQ_UNROLL for (int i = 0; i < m; ++i)
      LQ_UNROLL for (int j = 0; j < m; ++j)
        if (fx[i] || fx[j]) G[i * m + j] = (i == j) ? 1.0 : 0.0;
    LQ_UNROLL for (int i = 0; i < m; ++i)
      if (fx[i]) {
        LQ_UNROLL for (int j = 0; j < n; ++j) Hx[i * (n + 1) + j] = 0.0;
        Hx[i * (n + 1) + n] = -uc[i];
      }
    ok = chol<m>(G) && ok;
    solve_l<m, n + 1>(G, Hx);
    solve_lt<m, n + 1>(G, Hx);
    double K[m * n], kv[m];
    LQ_UNROLL for (int i = 0; i < m; ++i) {
      LQ_UNROLL for (int j = 0; j < n; ++j) K[i * n + j] = -Hx[i * (n + 1) + j];
      kv[i] = fx[i] ? uc[i] : -Hx[i * (n + 1) + n];
    }
    LQ_UNROLL for (int e = 0; e < m * n; ++e) ws[L.oKc + (int64_t)k * (m * n) + e] = K[e];
    LQ_UNROLL for (int e = 0; e < m; ++e) ws[L.okc + (int64_t)k * m + e] = kv[e];
    if (k > 0) {
      // S_k = Q + K'RK + Acl' S Acl ;  s_k = K'R kv + Acl'(S B kv + s)
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
      mv<m, m>(pb.R, kw, Rk);                              // R (k_k - u_ref_k)
      LQ_UNROLL for (int i = 0; i < n; ++i) {
        double acc = 0.0;
        LQ_UNROLL for (int r = 0; r < n; ++r) acc = fma(-pb.Q[i * n + r], rf.x(r, k - 1), acc);   // - Q x_ref_{k-1}
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

// n >= 5: the sweep as a separate, non-inlined function (inlined into the solver the register allocator gives up at
// n = 8: 32 registers and 55 kB of spills per thread).
template <int n, int m>
LQ_HD_NOINLINE_T bool clqr_backward_call(const Problem<n, m>& pb, const Plan<n, m>& pl, int N, const Mask128& fixed,
                                         const Mask128& athi, const WsView& ws, const Refs& rf, int klast,
                                         int koff = 0) {
  return clqr_backward<n, m>(pb, pl, N, fixed, athi, ws, rf, klast, koff);
}

// Exact constrained solve from state x0. Returns flags; writes u0[m] and V (= optimum + x0'Qx0).
// Pass structure (every pass is a sequential N-stage chain on strided scratch, so passes are what the solve costs):
//   one clipped rollout of the unconstrained law (feasible => optimal, done) doubles as the feasible start;
//   per active-set iteration: a backward sweep over the stages up to the last clamped one, ONE forward sweep that
//   also accumulates the objective of its candidate, and a costate sweep over the clamped stages only — the tail
//   beyond them is unconstrained with cost-to-go x'S x, so its costate is 2 S x without a sweep.
// `koff` (see clqr_backward): horizon N of a range sweep reads the stored unconstrained gains / cost-to-go at stage
// k + koff; which working sets restart from a stored S is decided by the stored-stage count of horizon N itself.
template <int n, int m>
LQ_HD int clqr_solve(const Problem<n, m>& pb, const Plan<n, m>& pl, int N, const double* x0, const WsView& ws,
                     double* u0, double* V, const Refs& rf = Refs(), int koff = 0) {
  const ClqrLayout<n, m> L(N + koff);
  const int kp = (N < kStoredCostToGo) ? N : kStoredCostToGo;   // == ClqrLayout(N).kp
  const int64_t oKu = L.oKu + (int64_t)koff * (m * n);
  double x[n], xn[n], u[m];
  const bool trk = rf.any();
  int flags = 0;
  // ---- 1. unconstrained plan, clipped into the box as it is rolled out: no clip => it is the QP minimiser. With
  //         references the plan is affine: gains AND offsets come from the affine sweep with an empty working set.
  if (trk && !((n <= 4) ? clqr_backward<n, m>(pb, pl, N, Mask128(), Mask128(), ws, rf, N - 1, koff)
                        : clqr_backward_call<n, m>(pb, pl, N, Mask128(), Mask128(), ws, rf, N - 1, koff)))
    flags |= FLAG_CHOL_FAIL;
  const int64_t oK = trk ? L.oKc : oKu;
  if (!trk) {
    // ---- 0. regulation: inside the certificate ellipsoid the unconstrained plan is feasible, hence optimal
    const double V0 = quad<n>(x0, pl.P0, x0);
    if (V0 <= pl.cstar) {
      if (Plan<n, m>::kHoldK0) {
        mv<m, n>(pl.K0, x0, u0);
      } else {
        double K[m * n];
        LQ_UNROLL for (int e = 0; e < m * n; ++e) K[e] = ws[oKu + e];
        mv<m, n>(K, x0, u0);
      }
      *V = V0;
      return flags;
    }
  }
  Mask128 fixed, athi;
  bool feas = true;
  LQ_UNROLL for (int i = 0; i < n; ++i) x[i] = x0[i];
  const double c0 = quad<n>(x0, pb.Q, x0);
  double cost_u = c0;
  staged_loop<m * n + m, StagePrefetch<n, m>::depth>(N, [&](int k, double* v) {
    LQ_UNROLL for (int e = 0; e < m * n; ++e) v[e] = ws[oK + (int64_t)k * (m * n) + e];
    LQ_UNROLL for (int j = 0; j < m; ++j) v[m * n + j] = trk ? ws[L.okc + (int64_t)k * m + j] : 0.0;
  }, [&](int k, const double* K) {
    mv<m, n>(K, x, u);
    const bool was_feas = feas;
    LQ_UNROLL for (int j = 0; j < m; ++j) {
      if (trk) u[j] += K[m * n + j];
      if (k == 0) u0[j] = u[j];
      if (u[j] < pb.ulo[j] || u[j] > pb.uhi[j]) feas = false;
      const int bit = k * m + j;
      if (u[j] >= pb.uhi[j]) { u[j] = pb.uhi[j]; fixed.set(bit); athi.set(bit); }
      else if (u[j] <= pb.ulo[j]) { u[j] = pb.ulo[j]; fixed.set(bit); }
    }
    // the plan is only WRITTEN (as the active-set start) once it has left the box: a feasible solve — the closed loop's
    // usual case — stores nothing. The stages before the first violation are replayed (normally there are none).
    if (was_feas && !feas && k > 0) {
      double xr[n], xq[n], ur[m];
      LQ_UNROLL for (int i = 0; i < n; ++i) xr[i] = x0[i];
      for (int kk = 0; kk < k; ++kk) {
        double Kr[m * n];
        LQ_UNROLL for (int e = 0; e < m * n; ++e) Kr[e] = ws[oK + (int64_t)kk * (m * n) + e];
        mv<m, n>(Kr, xr, ur);
        LQ_UNROLL for (int j = 0; j < m; ++j) {
          if (trk) ur[j] += ws[L.okc + (int64_t)kk * m + j];
          ws[L.oz + (int64_t)kk * m + j] = ur[j];
        }
        step_model<n, m>(pl.Ah, pl.Bh, xr, ur, xq);
        LQ_UNROLL for (int i = 0; i < n; ++i) xr[i] = xq[i];
      }
    }
    if (!feas) {
      LQ_UNROLL for (int j = 0; j < m; ++j) ws[L.oz + (int64_t)k * m + j] = u[j];
    }
    step_model<n, m>(pl.Ah, pl.Bh, x, u, xn);
    if (trk && feas) {
      double du[m], dx[n];
      LQ_UNROLL for (int j = 0; j < m; ++j) du[j] = u[j] - rf.u(j, k);
      LQ_UNROLL for (int i = 0; i < n; ++i) dx[i] = xn[i] - rf.x(i, k);
      cost_u += quad<m>(du, pb.R, du);
      cost_u += (k == N - 1) ? quad<n>(dx, pb.Pt, dx) : quad<n>(dx, pb.Q, dx);
    }
    LQ_UNROLL for (int i = 0; i < n; ++i) x[i] = xn[i];
  });
  if (feas) {
    *V = trk ? cost_u : quad<n>(x0, pl.P0, x0);
    return flags;
  }
  flags |= FLAG_QP_ACTIVE;
  if (N * m > kMaskBits) {   // beyond the working-set mask: never approximated — V = NaN, u0 clipped into the box, flagged
    LQ_UNROLL for (int j = 0; j < m; ++j) u0[j] = dmin(dmax(u0[j], pb.ulo[j]), pb.uhi[j]);
    *V = NAN;
    return flags | FLAG_QP_MAXITER;
  }
  // ---- 2. primal active-set iterations from the clipped plan (z in ws[oz..], candidate z* in ws[ozs..]; the two
  //         regions swap roles on a full step instead of being copied)
  int64_t oz = L.oz, ozs = L.ozs;
  const int maxit = 8 * N * m + 32;
  bool done = false;
  double cost = 0.0;
  for (int it = 0; it < maxit && !done; ++it) {
    // regulation: stages beyond the last clamped one keep the unconstrained law — the sweep covers 0..klast only
    const int top = fixed.top_bit();
    int klast = trk ? N - 1 : (top < 0 ? -1 : top / m);
    if (klast + 1 >= kp) klast = N - 1;                    // S_{klast+1} is not stored that far out: full sweep
    if (!((n <= 4) ? clqr_backward<n, m>(pb, pl, N, fixed, athi, ws, rf, klast, koff)
                   : clqr_backward_call<n, m>(pb, pl, N, fixed, athi, ws, rf, klast, koff)))
      flags |= FLAG_CHOL_FAIL;
    // forward sweep: candidate z*, its trajectory (kept up to stage klast + 1: all the costate sweep reads), its
    // objective, and the largest feasible step along z* - z
    double alpha = 1.0;
    int block = -1;
    bool block_hi = false;
    LQ_UNROLL for (int i = 0; i < n; ++i) { x[i] = x0[i]; ws[L.oxs + i] = x0[i]; }
    cost = c0;
    // per stage: the gain, its offset (zero beyond klast: unconstrained law) and the current iterate z_k
    staged_loop<m * n + 2 * m, StagePrefetch<n, m>::depth>(N, [&](int k, double* v) {
      const bool tl = (k > klast);
      const int64_t og = tl ? oKu : L.oKc;
      LQ_UNROLL for (int e = 0; e < m * n; ++e) v[e] = ws[og + (int64_t)k * (m * n) + e];
      LQ_UNROLL for (int j = 0; j < m; ++j) {
        v[m * n + j] = tl ? 0.0 : ws[L.okc + (int64_t)k * m + j];
        v[m * n + m + j] = ws[oz + (int64_t)k * m + j];
      }
    }, [&](int k, const double* K) {
      const bool tail = (k > klast);                       // unconstrained law (zero offset) beyond klast
      mv<m, n>(K, x, u);
      LQ_UNROLL for (int j = 0; j < m; ++j) {
        if (!tail) u[j] += K[m * n + j];
        const int bit = k * m + j;
        const bool isfx = fixed.test(bit);
        if (isfx) u[j] = athi.test(bit) ? pb.uhi[j] : pb.ulo[j];
        ws[ozs + (int64_t)k * m + j] = u[j];
        if (!isfx) {
          const double zc = K[m * n + m + j];
          if (u[j] > pb.uhi[j]) {
            const double a = (pb.uhi[j] - zc) / (u[j] - zc);
            if (a < alpha) { alpha = a; block = k * m + j; block_hi = true; }
          } else if (u[j] < pb.ulo[j]) {
            const double a = (pb.ulo[j] - zc) / (u[j] - zc);
            if (a < alpha) { alpha = a; block = k * m + j; block_hi = false; }
          }
        }
      }
      step_model<n, m>(pl.Ah, pl.Bh, x, u, xn);
      {
        double du[m], dx[n];
        LQ_UNROLL for (int j = 0; j < m; ++j) du[j] = u[j] - rf.u(j, k);
        LQ_UNROLL for (int i = 0; i < n; ++i) dx[i] = xn[i] - rf.x(i, k);
        cost += quad<m>(du, pb.R, du);
        cost += (k == N - 1) ? quad<n>(dx, pb.Pt, dx) : quad<n>(dx, pb.Q, dx);
      }
      LQ_UNROLL for (int i = 0; i < n; ++i) x[i] = xn[i];
      if (k <= klast || k == N - 1) {
        LQ_UNROLL for (int i = 0; i < n; ++i) ws[L.oxs + (int64_t)(k + 1) * n + i] = xn[i];
      }
    });
    if (block >= 0) {
      // partial step to the blocking bound, which joins the working set
      if (alpha < 0.0) alpha = 0.0;
      for (int e = 0; e < N * m; ++e) {
        const double zc = ws[oz + e];
        ws[oz + e] = fma(alpha, ws[ozs + e] - zc, zc);
      }
      const int j = block % m;
      ws[oz + block] = block_hi ? pb.uhi[j] : pb.ulo[j];
      fixed.set(block);
      if (block_hi) athi.set(block); else athi.clear(block);
      continue;
    }
    // full step: z = z* (swap the regions); multipliers of the clamped inputs from the costate sweep
    { const int64_t t = oz; oz = ozs; ozs = t; }
    double lam[n];
    if (klast == N - 1) {
      double xe[n];
      LQ_UNROLL for (int i = 0; i < n; ++i) xe[i] = ws[L.oxs + (int64_t)N * n + i] - rf.x(i, N - 1);
      mv<n, n>(pb.Pt, xe, lam);
      LQ_UNROLL for (int i = 0; i < n; ++i) lam[i] *= 2.0;
    } else {
      // unconstrained tail: cost-to-go x' S_{klast+1} x, hence the costate 2 S x at stage klast + 1
      double Sk[n * n], xe[n];
      int e = 0;
      LQ_UNROLL for (int i = 0; i < n; ++i)
        LQ_UNROLL for (int j = i; j < n; ++j) {
          const double v = ws[L.oP + (int64_t)(klast + 1 + koff) * L.np + e];
          Sk[i * n + j] = v; Sk[j * n + i] = v; ++e;
        }
      LQ_UNROLL for (int i = 0; i < n; ++i) xe[i] = ws[L.oxs + (int64_t)(klast + 1) * n + i];
      mv<n, n>(Sk, xe, lam);
      LQ_UNROLL for (int i = 0; i < n; ++i) lam[i] *= 2.0;
    }
    double worst = 0.0;
    int rel = -1;
    for (int k = klast; k >= 0; --k) {
      double uk[m], g1[m], g2[m];
      LQ_UNROLL for (int j = 0; j < m; ++j) uk[j] = ws[oz + (int64_t)k * m + j] - rf.u(j, k);
      mv<m, m>(pb.R, uk, g1);
      LQ_UNROLL for (int j = 0; j < m; ++j) {
        double acc = 0.0;
        LQ_UNROLL for (int r = 0; r < n; ++r) acc = fma(pl.Bh[r * m + j], lam[r], acc);
        g2[j] = acc;
        const int bit = k * m + j;
        if (fixed.test(bit)) {
          const double g = 2.0 * g1[j] + g2[j];            // dJ/du_{k,j}
          const double tol = 1e-11 * (fabs(2.0 * g1[j]) + fabs(g2[j])) + 1e-300;
          const double viol = athi.test(bit) ? g : -g;     // at hi need g <= 0 ; at lo need g >= 0
          if (viol > tol && viol > worst) { worst = viol; rel = k * m + j; }
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
    else fixed.clear(rel);
  }
  if (done) {                                              // `cost` is the objective of the last candidate = z
    LQ_UNROLL for (int j = 0; j < m; ++j) u0[j] = ws[oz + j];
    *V = cost;
    return flags;
  }
  flags |= FLAG_QP_MAXITER;
  // ---- 3. iteration budget exhausted: objective along the current (feasible, not proven optimal) z
  LQ_UNROLL for (int i = 0; i < n; ++i) x[i] = x0[i];
  cost = c0;
  for (int k = 0; k < N; ++k) {
    LQ_UNROLL for (int j = 0; j < m; ++j) {
      u[j] = ws[oz + (int64_t)k * m + j];
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

// Closed-loop simulation (utils_class.py:245-285): the controller re-solves from the measured state every step,
// the plant is the TRUE model. Optional trajectories X [(T+1)*n], U [T*m] through strided views.
template <int n, int m, class Traj>
LQ_HD int simulate_sample(const Problem<n, m>& pb, const Plan<n, m>& pl, int N, int T, const double* x0,
                          const WsView& ws, double* J_T, int* n_active, Traj& traj, const Refs& rf = Refs()) {
  double x[n], xn[n], u[m];
  LQ_UNROLL for (int i = 0; i < n; ++i) x[i] = x0[i];
  traj.state(0, x);
  double cost = quad<n>(x, pb.Q, x);
  int flags = 0, act = 0;
  for (int t = 0; t < T; ++t) {
    double V;
    const int f = clqr_solve<n, m>(pb, pl, N, x, ws, u, &V, rf);   // the same reference window every step (:269)
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

}  // namespace lq
