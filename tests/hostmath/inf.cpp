// TEST FIXTURE ONLY — the infinite-horizon closed loop of K2c (clqr.cuh: simulate_inf_sample / inf_tail, pclqr.cuh:
// psimulate_inf_sample / poly_certificate) compiled with g++ from the engine headers, one sample after another, so
// that tests/test_simulate_inf_host.py can hold it against a numpy oracle on the CPU. Built and loaded by that test
// (and by the GPU tier's host-vs-device comparison) only.
#include <stdint.h>
#include <string.h>

#include <vector>

#include "../../lq_mpc_b200/csrc/pclqr.cuh"

#define INF_FOR_EACH_DIM(X) X(1, 1) X(2, 1) X(2, 2) X(3, 1) X(3, 2) X(3, 3) X(4, 1) X(4, 2) X(4, 4) X(6, 2) X(8, 2)

namespace {

template <int n, int m>
void fill_problem(lq::Problem<n, m>& pb, const double* A, const double* B, const double* Q, const double* R,
                  const double* P, const double* lo, const double* hi) {
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
  lq::prepare_problem<n, m>(pb, 0);
}

template <int n, int m>
void load_model(const lq::Problem<n, m>& pb, int64_t S, int64_t s, const double* dA, const double* dB,
                lq::Plan<n, m>& pl) {
  for (int e = 0; e < n * n; ++e) pl.Ah[e] = pb.A[e] + dA[(int64_t)e * S + s];
  for (int e = 0; e < n * m; ++e) pl.Bh[e] = pb.B[e] + dB[(int64_t)e * S + s];
}

// J_inf [S], T_cert [S], flags [S] for dA [n*n][S], dB [n*m][S], x0 [n][S]; F (p x m) = NULL: the box
template <int n, int m>
int sim_t(const double* A, const double* B, const double* Q, const double* R, const double* Pt, const double* lo,
          const double* hi, int64_t S, const double* dA, const double* dB, int N, int T_max, const double* x0,
          const double* F, int p, double* J, int32_t* Tc, int32_t* flags) {
  lq::Problem<n, m> pb;
  fill_problem<n, m>(pb, A, B, Q, R, Pt, lo, hi);
  std::vector<double> wsbuf((size_t)lq::clqr_ws_doubles<n, m>(N) + 16);
  const lq::WsView ws{wsbuf.data(), 1};
  for (int64_t s = 0; s < S; ++s) {
    lq::Plan<n, m> pl;
    load_model<n, m>(pb, S, s, dA, dB, pl);
    double xx[n];
    for (int i = 0; i < n; ++i) xx[i] = x0[(int64_t)i * S + s];
    int tc;
    flags[s] = F ? lq::psimulate_inf_sample<n, m>(pb, pl, N, T_max, xx, lq::Poly{F, p}, ws, &J[s], &tc)
                 : lq::simulate_inf_sample<n, m>(pb, pl, N, T_max, xx, ws, &J[s], &tc);
    Tc[s] = tc;
  }
  return 0;
}

// One sample's certificate: S [n*n], c_S, cstar and the unconstrained gains K [N][m*n] of its plan. Returns the flags.
template <int n, int m>
int tail_t(const double* A, const double* B, const double* Q, const double* R, const double* Pt, const double* lo,
           const double* hi, const double* dA, const double* dB, int N, const double* F, int p, double* Sout,
           double* cS, double* cstar, double* K) {
  lq::Problem<n, m> pb;
  fill_problem<n, m>(pb, A, B, Q, R, Pt, lo, hi);
  std::vector<double> wsbuf((size_t)lq::clqr_ws_doubles<n, m>(N) + 16);
  const lq::WsView ws{wsbuf.data(), 1};
  lq::Plan<n, m> pl;
  load_model<n, m>(pb, 1, 0, dA, dB, pl);
  int f = lq::plan_prepare<n, m>(pb, pl, N, ws, F == nullptr);
  *cstar = F ? lq::poly_certificate<n, m>(pl, N, lq::Poly{F, p}, ws) : pl.cstar;
  f |= lq::inf_tail<n, m>(pb, pl, N, *cstar, ws, Sout, cS);
  for (int e = 0; e < N * m * n; ++e) K[e] = wsbuf[e];
  return f;
}

}  // namespace

extern "C" {

int inf_sim(int n, int m, const double* A, const double* B, const double* Q, const double* R, const double* Pt,
            const double* lo, const double* hi, int64_t S, const double* dA, const double* dB, int N, int T_max,
            const double* x0, const double* F, int p, double* J, int32_t* Tc, int32_t* flags) {
#define X(N_, M_) \
  if (n == N_ && m == M_) return sim_t<N_, M_>(A, B, Q, R, Pt, lo, hi, S, dA, dB, N, T_max, x0, F, p, J, Tc, flags);
  INF_FOR_EACH_DIM(X)
#undef X
  return -1;
}

int inf_tail(int n, int m, const double* A, const double* B, const double* Q, const double* R, const double* Pt,
             const double* lo, const double* hi, const double* dA, const double* dB, int N, const double* F, int p,
             double* Sout, double* cS, double* cstar, double* K) {
#define X(N_, M_) \
  if (n == N_ && m == M_) return tail_t<N_, M_>(A, B, Q, R, Pt, lo, hi, dA, dB, N, F, p, Sout, cS, cstar, K);
  INF_FOR_EACH_DIM(X)
#undef X
  return -1;
}

}  // extern "C"
