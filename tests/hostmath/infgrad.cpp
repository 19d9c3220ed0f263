// TEST FIXTURE ONLY — the gradient of the input-constrained closed loop's certified J_inf and its projected ascent
// (worst_inf.cuh: inf_grad_eval / inf_ascent) compiled with g++ from the engine headers, one sample after another, so
// that tests/test_inf_grad_host.py can hold them against a torch autograd oracle on the CPU. Built and loaded by that
// test (and by the GPU tier's host-vs-device comparison) only.
#include <stdint.h>
#include <string.h>

#include <vector>

#include "../../lq_mpc_b200/csrc/worst_inf.cuh"

#define INFGRAD_FOR_EACH_DIM(X) X(1, 1) X(2, 1) X(2, 2) X(3, 1) X(3, 2) X(3, 3) X(4, 1) X(4, 2) X(4, 4) X(6, 2) X(8, 2)

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
void load(int64_t S, int64_t s, const double* dA, const double* dB, const double* x0, double* a, double* b, double* x) {
  for (int e = 0; e < n * n; ++e) a[e] = dA[e * S + s];
  for (int e = 0; e < n * m; ++e) b[e] = dB[e * S + s];
  for (int e = 0; e < n; ++e) x[e] = x0[e * S + s];
}

// SoA operands dA [n*n][S], dB [n*m][S], x0 [n][S]; outputs [S], gA [n*n][S], gB [n*m][S] (gA NULL: value only)
template <int n, int m>
int grad_t(const double* A, const double* B, const double* Q, const double* R, const double* Pt, const double* lo,
           const double* hi, int64_t S, const double* dA, const double* dB, const double* x0, int N, int T_max,
           double* J, int32_t* Tc, double* rho, double* gA, double* gB, int32_t* flags) {
  lq::Problem<n, m> pb;
  fill_problem<n, m>(pb, A, B, Q, R, Pt, lo, hi);
  std::vector<double> wsbuf((size_t)lq::InfGradLayout<n, m>(N, T_max).total + 16);
  const lq::WsView ws{wsbuf.data(), 1};
  for (int64_t s = 0; s < S; ++s) {
    double a[n * n], b[n * m], x[n], ga[n * n], gb[n * m];
    load<n, m>(S, s, dA, dB, x0, a, b, x);
    int tc;
    flags[s] = lq::inf_grad_eval<n, m>(pb, a, b, x, N, T_max, ws, &J[s], &tc, &rho[s], gA ? ga : nullptr,
                                       gA ? gb : nullptr);
    Tc[s] = tc;
    if (gA) {
      for (int e = 0; e < n * n; ++e) gA[e * S + s] = ga[e];
      for (int e = 0; e < n * m; ++e) gB[e * S + s] = gb[e];
    }
  }
  return 0;
}

template <int n, int m>
int ascent_t(const double* A, const double* B, const double* Q, const double* R, const double* Pt, const double* lo,
             const double* hi, int64_t S, const double* dA, const double* dB, const double* x0, int N, int T_max,
             double eA, double eB, int norm, int max_iter, double tol, double* dA_out, double* dB_out, double* J,
             int32_t* Tc, double* rho, int32_t* iters, int32_t* flags) {
  lq::Problem<n, m> pb;
  fill_problem<n, m>(pb, A, B, Q, R, Pt, lo, hi);
  std::vector<double> wsbuf((size_t)lq::InfGradLayout<n, m>(N, T_max).total + 16);
  const lq::WsView ws{wsbuf.data(), 1};
  const lq::AscentSettings as{eA, eB, tol, norm, max_iter};
  for (int64_t s = 0; s < S; ++s) {
    double a[n * n], b[n * m], x[n];
    load<n, m>(S, s, dA, dB, x0, a, b, x);
    int it, tc;
    flags[s] = lq::inf_ascent<n, m>(pb, a, b, x, N, T_max, as, ws, &J[s], &tc, &rho[s], &it);
    iters[s] = it;
    Tc[s] = tc;
    for (int e = 0; e < n * n; ++e) dA_out[e * S + s] = a[e];
    for (int e = 0; e < n * m; ++e) dB_out[e * S + s] = b[e];
  }
  return 0;
}

}  // namespace

extern "C" {

int infgrad_grad(int n, int m, const double* A, const double* B, const double* Q, const double* R, const double* Pt,
                 const double* lo, const double* hi, int64_t S, const double* dA, const double* dB, const double* x0,
                 int N, int T_max, double* J, int32_t* Tc, double* rho, double* gA, double* gB, int32_t* flags) {
#define X(N_, M_)                                                                                                    \
  if (n == N_ && m == M_)                                                                                            \
    return grad_t<N_, M_>(A, B, Q, R, Pt, lo, hi, S, dA, dB, x0, N, T_max, J, Tc, rho, gA, gB, flags);
  INFGRAD_FOR_EACH_DIM(X)
#undef X
  return -1;
}

int infgrad_ascent(int n, int m, const double* A, const double* B, const double* Q, const double* R, const double* Pt,
                   const double* lo, const double* hi, int64_t S, const double* dA, const double* dB, const double* x0,
                   int N, int T_max, double eA, double eB, int norm, int max_iter, double tol, double* dA_out,
                   double* dB_out, double* J, int32_t* Tc, double* rho, int32_t* iters, int32_t* flags) {
#define X(N_, M_)                                                                                                    \
  if (n == N_ && m == M_)                                                                                            \
    return ascent_t<N_, M_>(A, B, Q, R, Pt, lo, hi, S, dA, dB, x0, N, T_max, eA, eB, norm, max_iter, tol, dA_out,    \
                            dB_out, J, Tc, rho, iters, flags);
  INFGRAD_FOR_EACH_DIM(X)
#undef X
  return -1;
}

}  // extern "C"
