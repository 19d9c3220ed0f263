// k_worst_inf.cu — exact gradient of the input-constrained closed loop's certified J_inf (K2c) in the model error and
// the projected worst-case ascent on it (worst_inf.cuh), box only, one sample per thread, grid-stride over the batch.
// The per-thread workspace (the solver's scratch, the Riccati stage records, the VJP's plan records and the closed-loop
// states) lives in the context workspace laid out [element][thread], so a warp touches 32 consecutive doubles per
// access; the grid is capped at one wave of resident CTAs (lq_worst_blocks), which keeps it at one wave's worth.
#include "engine.h"
#include "worst_inf.cuh"

namespace {

template <int n, int m>
__device__ __forceinline__ void load_inf_sample(const WorstInfArgs& a, int64_t s, double* dA, double* dB, double* x0) {
#pragma unroll
  for (int e = 0; e < n * n; ++e) dA[e] = a.dA[(int64_t)e * a.S + s];
#pragma unroll
  for (int e = 0; e < n * m; ++e) dB[e] = a.dB[(int64_t)e * a.S + s];
#pragma unroll
  for (int e = 0; e < n; ++e) x0[e] = a.x0_shared ? a.x0_shared[e] : a.x0[(int64_t)e * a.S + s];
}

template <int len>
__device__ __forceinline__ void store_soa(double* out, int64_t S, int64_t s, const double* v) {
  if (out) {
#pragma unroll
    for (int e = 0; e < len; ++e) out[(int64_t)e * S + s] = v[e];
  }
}

// J_inf, T_cert, rho, flags [S]; the gradient gA [n*n][S], gB [n*m][S] only when one of them is requested (a value-only
// call computes K2c's closed loop and rho, and touches the solver's scratch only).
template <int n, int m>
__global__ void __launch_bounds__(128) simulate_inf_grad_kernel(const __grid_constant__ lq::Problem<n, m> pb,
                                                                const __grid_constant__ WorstInfArgs a) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  const lq::WsView ws{a.ws + tid, nthreads};
  const bool grad = a.gA || a.gB;
  for (int64_t s = tid; s < a.S; s += nthreads) {
    double dA[n * n], dB[n * m], x0[n], gA[n * n], gB[n * m], J, rho;
    int tc;
    load_inf_sample<n, m>(a, s, dA, dB, x0);
    const int f = lq::inf_grad_eval<n, m>(pb, dA, dB, x0, a.N, a.T_max, ws, &J, &tc, &rho, grad ? gA : nullptr,
                                          grad ? gB : nullptr);
    if (a.J) a.J[s] = J;
    if (a.T_cert) a.T_cert[s] = tc;
    if (a.rho) a.rho[s] = rho;
    if (a.flags) a.flags[s] = f;
    store_soa<n * n>(a.gA, a.S, s, gA);
    store_soa<n * m>(a.gB, a.S, s, gB);
  }
}

// The ascent; the inputs are read with plain loads: dA_out / dB_out may alias dA / dB (each thread reads its sample
// first).
template <int n, int m>
__global__ void __launch_bounds__(128) worst_case_inf_kernel(const __grid_constant__ lq::Problem<n, m> pb,
                                                             const __grid_constant__ WorstInfArgs a) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  const lq::WsView ws{a.ws + tid, nthreads};
  const lq::AscentSettings as{a.eA, a.eB, a.tol, a.norm, a.max_iter};
  for (int64_t s = tid; s < a.S; s += nthreads) {
    double dA[n * n], dB[n * m], x0[n], J, rho;
    int it, tc;
    load_inf_sample<n, m>(a, s, dA, dB, x0);
    const int f = lq::inf_ascent<n, m>(pb, dA, dB, x0, a.N, a.T_max, as, ws, &J, &tc, &rho, &it);
    store_soa<n * n>(a.dA_out, a.S, s, dA);
    store_soa<n * m>(a.dB_out, a.S, s, dB);
    if (a.J) a.J[s] = J;
    if (a.T_cert) a.T_cert[s] = tc;
    if (a.rho) a.rho[s] = rho;
    if (a.iters) a.iters[s] = it;
    if (a.flags) a.flags[s] = f;
  }
}

template <int n, int m, bool ASCENT>
int launch_inf_t(lqmpc_ctx* ctx, WorstInfArgs a) {
  const lq::Problem<n, m>& pb = *reinterpret_cast<const lq::Problem<n, m>*>(ctx->pb);
  const int threads = 128;
  const auto kernel = ASCENT ? worst_case_inf_kernel<n, m> : simulate_inf_grad_kernel<n, m>;
  const int64_t blocks = lq_worst_blocks(ctx, (const void*)kernel, threads, a.S);
  // the workspace grows with T_max: (T_max + 1) n doubles of closed-loop states per thread
  const int64_t per = (ASCENT || a.gA || a.gB) ? lq::InfGradLayout<n, m>(a.N, a.T_max).total
                                               : lq::clqr_ws_doubles<n, m>(a.N);
  int rc = lq_reserve_ws(ctx, (size_t)(per * blocks * threads) * sizeof(double) + 64);
  if (rc) return rc;
  a.ws = reinterpret_cast<double*>(ctx->ws);
  kernel<<<(unsigned)blocks, threads, 0, ctx->stream>>>(pb, a);
  ctx->launches++;
  return lq_check_cuda(ctx, cudaGetLastError(),
                       ASCENT ? "worst_case_inf_kernel launch" : "simulate_inf_grad_kernel launch");
}

}  // namespace

int lq_launch_simulate_inf_grad(lqmpc_ctx* ctx, const WorstInfArgs& a) {
#define X(N_, M_) \
  if (ctx->n == N_ && ctx->m == M_) return launch_inf_t<N_, M_, false>(ctx, a);
  LQ_FOR_EACH_DIM(X)
#undef X
  return lq_set_error(ctx, LQMPC_EINVAL, "unsupported (n, m); see lqmpc_supported_dims()");
}

int lq_launch_worst_case_inf(lqmpc_ctx* ctx, const WorstInfArgs& a) {
#define X(N_, M_) \
  if (ctx->n == N_ && ctx->m == M_) return launch_inf_t<N_, M_, true>(ctx, a);
  LQ_FOR_EACH_DIM(X)
#undef X
  return lq_set_error(ctx, LQMPC_EINVAL, "unsupported (n, m); see lqmpc_supported_dims()");
}
