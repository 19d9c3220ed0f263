// k_clqr.cu — K2 with the input BOX (every caller in the reference): instantiates k_clqr_impl.cuh with POLY = false and
// routes to the polytope family (k_pclqr.cu) when lqmpc_set_input_polytope installed a general F_u.
#include "k_clqr_impl.cuh"

int lq_launch_mpc(lqmpc_ctx* ctx, const MpcArgs& a, bool sim) {
  if (ctx->poly_p > 0) return lq_launch_mpc_poly(ctx, a, sim);
#define X(N_, M_) \
  if (ctx->n == N_ && ctx->m == M_) return launch_mpc_t<N_, M_, false>(ctx, a, sim);
  LQ_FOR_EACH_DIM(X)
#undef X
  return lq_set_error(ctx, LQMPC_EINVAL, "unsupported (n, m); see lqmpc_supported_dims()");
}

// Horizon range with the input box and zero references (the caller routes every other case to per-horizon launches).
int lq_launch_mpc_range(lqmpc_ctx* ctx, const MpcArgs& a) {
#define X(N_, M_) \
  if (ctx->n == N_ && ctx->m == M_) return launch_mpc_range_t<N_, M_>(ctx, a);
  LQ_FOR_EACH_DIM(X)
#undef X
  return lq_set_error(ctx, LQMPC_EINVAL, "unsupported (n, m); see lqmpc_supported_dims()");
}
