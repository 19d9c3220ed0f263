// k_pclqr.cu — K2 with a GENERAL input polytope F_u u <= 1 (utils_class.py:81; SURVEY 8f.3): instantiates
// k_clqr_impl.cuh with POLY = true (pclqr.cuh). Reached through lq_launch_mpc when lqmpc_set_input_polytope is active.
#include "k_clqr_impl.cuh"

int lq_launch_mpc_poly(lqmpc_ctx* ctx, const MpcArgs& a, bool sim) {
#define X(N_, M_) \
  if (ctx->n == N_ && ctx->m == M_) return launch_mpc_t<N_, M_, true>(ctx, a, sim);
  LQ_FOR_EACH_DIM(X)
#undef X
  return lq_set_error(ctx, LQMPC_EINVAL, "unsupported (n, m); see lqmpc_supported_dims()");
}

int lq_launch_simulate_inf_poly(lqmpc_ctx* ctx, const MpcArgs& a) {
#define X(N_, M_) \
  if (ctx->n == N_ && ctx->m == M_) return launch_simulate_inf_t<N_, M_, true>(ctx, a);
  LQ_FOR_EACH_DIM(X)
#undef X
  return lq_set_error(ctx, LQMPC_EINVAL, "unsupported (n, m); see lqmpc_supported_dims()");
}
