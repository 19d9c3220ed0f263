// TEST FIXTURE ONLY — compiles riccati.cuh's closed-loop cost routines with g++ for
// tests/test_k1_closed_loop_cost.py; nothing in lq_mpc_b200/ links or loads it.
#include <math.h>
#include <stdint.h>

#include "../lq_mpc_b200/csrc/riccati.cuh"

namespace {

// x0' S x0, S = W + Acl' S Acl, by the characteristic-polynomial route (J_poly; accepted = 1 where K1 takes it) and by
// the Lyapunov doubling (J_dbl; its convergence flag in dbl_ok); operands AoS
template <int n>
int lyap_cost_t(int64_t S, const double* Acl, const double* W, const double* x0, double* J_poly, int32_t* accepted,
                double* J_dbl, int32_t* dbl_ok) {
  for (int64_t s = 0; s < S; ++s) {
    const double* A = Acl + s * n * n;
    const double* w = W + s * n * n;
    const double* x = x0 + s * n;
    bool ok, cp_ok;
    lq::CharPoly cp;
    const double rho = lq::spectral_radius<n>(A, &ok, &cp, &cp_ok);
    double J = NAN;
    accepted[s] = (rho < 1.0 && cp_ok && lq::lyapunov_cost_poly<n>(cp, A, w, x, &J)) ? 1 : 0;
    J_poly[s] = J;
    double Sm[n * n];
    dbl_ok[s] = lq::lyapunov_doubling<n>(A, w, Sm) ? 1 : 0;
    J_dbl[s] = lq::quad<n>(x, Sm, x);
  }
  return 0;
}

}  // namespace

extern "C" int k1_closed_loop_cost(int n, int64_t S, const double* Acl, const double* W, const double* x0,
                                   double* J_poly, int32_t* accepted, double* J_dbl, int32_t* dbl_ok) {
  switch (n) {
    case 3: return lyap_cost_t<3>(S, Acl, W, x0, J_poly, accepted, J_dbl, dbl_ok);
    case 4: return lyap_cost_t<4>(S, Acl, W, x0, J_poly, accepted, J_dbl, dbl_ok);
  }
  return -1;
}
