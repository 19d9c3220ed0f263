// TEST FIXTURE ONLY — the sup-over-x0 mode of worst.cuh (worst_eval / worst_ascent with SUP = true: the ratio
// gamma = lambda_max(S, P_exp), its worst state, eigengap and gradient, and the ascent of gamma) compiled with g++ from
// the engine headers, one sample after another, so that tests/test_ratio_sup_host.py can hold them against scipy and
// a torch autograd oracle on the CPU. Built and loaded by that test (and by the GPU tier's host-vs-device comparison)
// only.
#include <stdint.h>
#include <string.h>

#include <vector>

#include "../../lq_mpc_b200/csrc/worst.cuh"

#define SUP_FOR_EACH_DIM(X) X(1, 1) X(2, 1) X(2, 2) X(3, 1) X(3, 2) X(3, 3) X(4, 1) X(4, 2) X(4, 4) X(6, 2) X(8, 2)

namespace {

template <int n, int m>
void fill_problem(lq::Problem<n, m>& pb, const double* A, const double* B, const double* Q, const double* R,
                  const double* P, int N_opc) {
  memset(&pb, 0, sizeof(pb));
  memcpy(pb.A, A, sizeof(pb.A));
  memcpy(pb.B, B, sizeof(pb.B));
  memcpy(pb.Q, Q, sizeof(pb.Q));
  memcpy(pb.R, R, sizeof(pb.R));
  memcpy(pb.Pt, P, sizeof(pb.Pt));
  for (int j = 0; j < m; ++j) { pb.ulo[j] = -HUGE_VAL; pb.uhi[j] = HUGE_VAL; }
  lq::prepare_problem<n, m>(pb, N_opc);
}

// SoA operands dA [n*n][S], dB [n*m][S]; outputs gamma, gap, rho [S], x_worst [n][S], gA [n*n][S], gB [n*m][S]
// (gA == nullptr: the value-only call)
template <int n, int m>
int ratio_t(const double* A, const double* B, const double* Q, const double* R, const double* Pt, int N_opc, int64_t S,
            const double* dA, const double* dB, int N, double* gamma, double* xw, double* gap, double* rho,
            double* gA, double* gB, int32_t* flags) {
  lq::Problem<n, m> pb;
  fill_problem<n, m>(pb, A, B, Q, R, Pt, N_opc);
  const lq::ExpertFactor<n> ef = lq::expert_factor<n, m>(pb);
  std::vector<double> wsbuf((size_t)lq::worst_ws_doubles<n, m>(N) + 16);
  const lq::WsView ws{wsbuf.data(), 1};
  for (int64_t s = 0; s < S; ++s) {
    double a[n * n], b[n * m], x[n], ga[n * n], gb[n * m];
    for (int e = 0; e < n * n; ++e) a[e] = dA[e * S + s];
    for (int e = 0; e < n * m; ++e) b[e] = dB[e * S + s];
    flags[s] = lq::worst_eval<n, m, true>(pb, a, b, nullptr, N, ws, &gamma[s], &rho[s], gA ? ga : nullptr,
                                          gA ? gb : nullptr, &ef, x, &gap[s]);
    for (int e = 0; e < n; ++e) xw[e * S + s] = x[e];
    if (gA) {
      for (int e = 0; e < n * n; ++e) gA[e * S + s] = ga[e];
      for (int e = 0; e < n * m; ++e) gB[e * S + s] = gb[e];
    }
  }
  return 0;
}

template <int n, int m>
int ascent_t(const double* A, const double* B, const double* Q, const double* R, const double* Pt, int N_opc,
             int64_t S, const double* dA, const double* dB, int N, double eA, double eB, int norm, int max_iter,
             double tol, double* dA_out, double* dB_out, double* gamma, double* xw, double* rho, int32_t* iters,
             int32_t* flags) {
  lq::Problem<n, m> pb;
  fill_problem<n, m>(pb, A, B, Q, R, Pt, N_opc);
  const lq::ExpertFactor<n> ef = lq::expert_factor<n, m>(pb);
  std::vector<double> wsbuf((size_t)lq::worst_ws_doubles<n, m>(N) + 16);
  const lq::WsView ws{wsbuf.data(), 1};
  const lq::AscentSettings as{eA, eB, tol, norm, max_iter};
  for (int64_t s = 0; s < S; ++s) {
    double a[n * n], b[n * m], x[n];
    for (int e = 0; e < n * n; ++e) a[e] = dA[e * S + s];
    for (int e = 0; e < n * m; ++e) b[e] = dB[e * S + s];
    int it;
    flags[s] = lq::worst_ascent<n, m, true>(pb, a, b, nullptr, N, as, ws, &gamma[s], &rho[s], &it, &ef, x);
    iters[s] = it;
    for (int e = 0; e < n; ++e) xw[e * S + s] = x[e];
    for (int e = 0; e < n * n; ++e) dA_out[e * S + s] = a[e];
    for (int e = 0; e < n * m; ++e) dB_out[e * S + s] = b[e];
  }
  return 0;
}

}  // namespace

extern "C" {

int sup_ratio(int n, int m, const double* A, const double* B, const double* Q, const double* R, const double* Pt,
              int N_opc, int64_t S, const double* dA, const double* dB, int N, double* gamma, double* x_worst,
              double* gap, double* rho, double* gA, double* gB, int32_t* flags) {
#define X(N_, M_)                                                                                                     \
  if (n == N_ && m == M_)                                                                                             \
    return ratio_t<N_, M_>(A, B, Q, R, Pt, N_opc, S, dA, dB, N, gamma, x_worst, gap, rho, gA, gB, flags);
  SUP_FOR_EACH_DIM(X)
#undef X
  return -1;
}

int sup_ascent(int n, int m, const double* A, const double* B, const double* Q, const double* R, const double* Pt,
               int N_opc, int64_t S, const double* dA, const double* dB, int N, double eA, double eB, int norm,
               int max_iter, double tol, double* dA_out, double* dB_out, double* gamma, double* x_worst, double* rho,
               int32_t* iters, int32_t* flags) {
#define X(N_, M_)                                                                                                     \
  if (n == N_ && m == M_)                                                                                             \
    return ascent_t<N_, M_>(A, B, Q, R, Pt, N_opc, S, dA, dB, N, eA, eB, norm, max_iter, tol, dA_out, dB_out, gamma, \
                            x_worst, rho, iters, flags);
  SUP_FOR_EACH_DIM(X)
#undef X
  return -1;
}

}  // extern "C"
