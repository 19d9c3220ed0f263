// TEST FIXTURE ONLY — the horizon-range K2a / K3 numerics (clqr.cuh: plan_prepare_range + the stage-offset solve;
// bounds.cuh / gramspec.cuh: bounds_prefix + gram_spectrum_range) next to their single-horizon counterparts,
// compiled with g++ from the engine headers, one sample after another, so that tests/test_horizon_range_host.py can
// compare them on the CPU. Built and loaded by that test only.
#include <stdint.h>
#include <string.h>

#include <vector>

#include "../../lq_mpc_b200/csrc/bounds.cuh"

#define HR_FOR_EACH_DIM(X) X(1, 1) X(2, 1) X(2, 2) X(3, 1) X(3, 2) X(3, 3) X(4, 1) X(4, 2) X(4, 4) X(6, 2) X(8, 2)

namespace {

template <int n, int m>
void fill_problem(lq::Problem<n, m>& pb, const double* A, const double* B, const double* Q, const double* R,
                  const double* P, const double* lo, const double* hi, int N_opc) {
  memset(&pb, 0, sizeof(pb));
  memcpy(pb.A, A, sizeof(pb.A));
  memcpy(pb.B, B, sizeof(pb.B));
  memcpy(pb.Q, Q, sizeof(pb.Q));
  memcpy(pb.R, R, sizeof(pb.R));
  memcpy(pb.Pt, P, sizeof(pb.Pt));
  pb.has_bounds = (lo || hi) ? 1 : 0;
  for (int j = 0; j < m; ++j) {
    pb.ulo[j] = lo ? lo[j] : -HUGE_VAL;
    pb.uhi[j] = hi ? hi[j] : HUGE_VAL;
  }
  lq::prepare_problem<n, m>(pb, N_opc);
}

template <int n, int m>
void load_model(const lq::Problem<n, m>& pb, int64_t S, int64_t s, const double* dA, const double* dB, double* Ah,
                double* Bh) {
  for (int e = 0; e < n * n; ++e) Ah[e] = pb.A[e] + dA[(int64_t)e * S + s];
  for (int e = 0; e < n * m; ++e) Bh[e] = pb.B[e] + dB[(int64_t)e * S + s];
}

// single (Nmin == Nmax == N through plan_prepare) or range (plan_prepare_range + koff) ring solves; outputs
// V [H][P][S], u0 [H][P][m][S], M_V [H][S], flags [H][P][S]
template <int n, int m>
int mpc_t(int range, const double* A, const double* B, const double* Q, const double* R, const double* Pt,
          const double* lo, const double* hi, int64_t S, const double* dA, const double* dB, int Nmin, int Nmax,
          int npts, const double* pts, const double* x0, double* V, double* u0, double* MV, int32_t* flags) {
  lq::Problem<n, m> pb;
  fill_problem<n, m>(pb, A, B, Q, R, Pt, lo, hi, 0);
  const int P = pts ? npts : 1;
  const int H = Nmax - Nmin + 1;
  std::vector<double> wsbuf((size_t)lq::clqr_range_ws_doubles<n, m>(Nmax) + 16);
  const lq::WsView ws{wsbuf.data(), 1};
  for (int64_t s = 0; s < S; ++s) {
    lq::Plan<n, m> pl;
    load_model<n, m>(pb, S, s, dA, dB, pl.Ah, pl.Bh);
    int first_fail = 0;
    if (range) first_fail = lq::plan_prepare_range<n, m>(pb, pl, Nmax, ws);
    for (int h = 0; h < H; ++h) {
      const int N = Nmin + h;
      int pf;
      int koff = 0;
      if (range) {
        koff = Nmax - N;
        lq::plan_select_horizon<n, m>(pl, Nmax, koff, ws);
        pf = (first_fail <= N) ? lq::FLAG_CHOL_FAIL : 0;
      } else {
        pf = lq::plan_prepare<n, m>(pb, pl, N, ws, false);
      }
      double mv = -HUGE_VAL;
      for (int p = 0; p < P; ++p) {
        double xx[n], uu[m], v;
        for (int i = 0; i < n; ++i) xx[i] = pts ? pts[p * n + i] : x0[(int64_t)i * S + s];
        const int f = pf | lq::clqr_solve<n, m>(pb, pl, N, xx, ws, uu, &v, lq::Refs(), koff);
        mv = lq::dmax(mv, v);
        const int64_t hp = (int64_t)h * P + p;
        V[hp * S + s] = v;
        for (int j = 0; j < m; ++j) u0[(hp * m + j) * S + s] = uu[j];
        flags[hp * S + s] = f;
      }
      MV[(int64_t)h * S + s] = mv;
    }
  }
  return 0;
}

template <int n, int m>
lq::BoundsScalars scalars(int64_t S, int64_t s, const double* eA, const double* eB, const double* p3, double Vexp) {
  lq::BoundsScalars sc;
  sc.N = 0;
  sc.e_A = eA[s];
  sc.e_B = eB[s];
  sc.M_V = 0.0;
  sc.p[0] = p3[0]; sc.p[1] = p3[1]; sc.p[2] = p3[2];
  sc.V_expert = Vexp;
  sc.bar_u = -1.0; sc.bar_d_u = -1.0;
  sc.strict_reference = 1;
  (void)S;
  return sc;
}

// bounds of horizons Nmin..Nmax: range (bounds_prefix + gram_spectrum_range) or one bounds_sample per horizon.
// MV [H][S], detail [H][BF_COUNT][S], flags [H][S], stages [S] (range: elimination stages of the range search),
// probes [H][S] (range: bisection passes per horizon)
template <int n, int m>
int bounds_t(int range, const double* A, const double* B, const double* Q, const double* R, const double* Pt,
             const double* lo, const double* hi, int64_t S, const double* dA, const double* dB, int Nmin, int Nmax,
             const double* eA, const double* eB, const double* MV, const double* x, const double* p3, double Vexp,
             double* detail, int32_t* flags, int64_t* stages, int32_t* probes) {
  lq::Problem<n, m> pb;
  fill_problem<n, m>(pb, A, B, Q, R, Pt, lo, hi, 0);
  const int NF = lq::BF_COUNT;
  for (int64_t s = 0; s < S; ++s) {
    double Ah[n * n], Bh[n * m], K[m * n], X[n * n];
    load_model<n, m>(pb, S, s, dA, dB, Ah, Bh);
    int f0 = 0;
    if (!lq::dare_sda<n, m>(Ah, Bh, pb.Q, pb.R, X)) f0 |= lq::FLAG_DARE_NOCONV;
    lq::dlqr_gain<n, m>(Ah, Bh, pb.R, X, K);
    for (int e = 0; e < m * n; ++e) K[e] = -K[e];
    lq::BoundsScalars sc = scalars<n, m>(S, s, eA, eB, p3, Vexp);
    if (range) {
      const lq::BoundsPrefix pr = lq::bounds_prefix<n, m>(pb, Ah, Bh, K, sc);
      lq::PhiGram<n> phi;
      lq::EcRunning ec = lq::ec_running<n>(pr, sc, x);
      stages[s] = lq::gram_spectrum_range<n, m>(Ah, Bh, pb.Q, pb.R, pb.minR, Nmin, Nmax,
                                                [&](int N, const lq::GramSpectrum& gs) {
        const int64_t h = N - Nmin;
        phi.extend_to(Ah, N);
        sc.N = N;
        sc.M_V = MV[h * S + s];
        double out[lq::BF_COUNT];
        for (int i = 0; i < NF; ++i) out[i] = 0.0;
        const lq::EcSums es = ec.at(N);
        flags[h * S + s] = f0 | lq::bounds_horizon<n, m>(pb, pr, phi.norm(), gs.cmax, gs.min_H, x, sc, out, &es);
        for (int i = 0; i < NF; ++i) detail[(h * NF + i) * S + s] = out[i];
        probes[h * S + s] = gs.probes;
      });
    } else {
      const lq::WsView ws{nullptr, 1};
      for (int N = Nmin; N <= Nmax; ++N) {
        const int64_t h = N - Nmin;
        sc.N = N;
        sc.M_V = MV[h * S + s];
        double out[lq::BF_COUNT];
        flags[h * S + s] = f0 | lq::bounds_sample<n, m>(pb, Ah, Bh, K, x, sc, ws, out);
        for (int i = 0; i < NF; ++i) detail[(h * NF + i) * S + s] = out[i];
      }
    }
  }
  return 0;
}

}  // namespace

extern "C" {

int hr_mpc(int range, int n, int m, const double* A, const double* B, const double* Q, const double* R,
           const double* Pt, const double* lo, const double* hi, int64_t S, const double* dA, const double* dB,
           int Nmin, int Nmax, int npts, const double* pts, const double* x0, double* V, double* u0, double* MV,
           int32_t* flags) {
#define X(N_, M_)                                                                                               \
  if (n == N_ && m == M_)                                                                                       \
    return mpc_t<N_, M_>(range, A, B, Q, R, Pt, lo, hi, S, dA, dB, Nmin, Nmax, npts, pts, x0, V, u0, MV, flags);
  HR_FOR_EACH_DIM(X)
#undef X
  return -1;
}

int hr_bounds(int range, int n, int m, const double* A, const double* B, const double* Q, const double* R,
              const double* Pt, const double* lo, const double* hi, int64_t S, const double* dA, const double* dB,
              int Nmin, int Nmax, const double* eA, const double* eB, const double* MV, const double* x,
              const double* p3, double Vexp, double* detail, int32_t* flags, int64_t* stages, int32_t* probes) {
#define X(N_, M_)                                                                                               \
  if (n == N_ && m == M_)                                                                                       \
    return bounds_t<N_, M_>(range, A, B, Q, R, Pt, lo, hi, S, dA, dB, Nmin, Nmax, eA, eB, MV, x, p3, Vexp,     \
                            detail, flags, stages, probes);
  HR_FOR_EACH_DIM(X)
#undef X
  return -1;
}

}  // extern "C"
