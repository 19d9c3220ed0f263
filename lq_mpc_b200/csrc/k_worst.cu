// k_worst.cu — exact gradient of J_inf in the model error and the projected worst-case ascent (worst.cuh), for a given
// x0 and in the sup-over-x0 mode (the ratio gamma = lambda_max(S, P_exp)), one sample per thread, grid-stride over the
// batch. The stage records of the reverse sweep live in the context workspace laid out [element][thread], so a warp
// touches 32 consecutive doubles per access. The grid is capped at one wave of resident CTAs, which keeps the workspace
// at one wave's worth (as K2's launches do).
#include <stdlib.h>

#include "engine.h"
#include "worst.cuh"

namespace {

template <int n, int m>
__device__ __forceinline__ void load_error(const WorstArgs& a, int64_t s, double* dA, double* dB) {
#pragma unroll
  for (int e = 0; e < n * n; ++e) dA[e] = a.dA[(int64_t)e * a.S + s];
#pragma unroll
  for (int e = 0; e < n * m; ++e) dB[e] = a.dB[(int64_t)e * a.S + s];
}

template <int n, int m>
__device__ __forceinline__ void load_sample(const WorstArgs& a, int64_t s, double* dA, double* dB, double* x0) {
  load_error<n, m>(a, s, dA, dB);
#pragma unroll
  for (int e = 0; e < n; ++e) x0[e] = a.x0[(int64_t)e * a.S + s];
}

template <int len>
__device__ __forceinline__ void store_soa(double* out, int64_t S, int64_t s, const double* v) {
  if (out) {
#pragma unroll
    for (int e = 0; e < len; ++e) out[(int64_t)e * S + s] = v[e];
  }
}

template <int n, int m>
__global__ void __launch_bounds__(128) eval_grad_kernel(const __grid_constant__ lq::Problem<n, m> pb,
                                                        const __grid_constant__ WorstArgs a) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  const lq::WsView ws{a.ws + tid, nthreads};
  for (int64_t s = tid; s < a.S; s += nthreads) {
    double dA[n * n], dB[n * m], x0[n], gA[n * n], gB[n * m], J, rho;
    load_sample<n, m>(a, s, dA, dB, x0);
    const int f = lq::worst_eval<n, m>(pb, dA, dB, x0, a.N, ws, &J, &rho, gA, gB);
    if (a.J) a.J[s] = J;
    if (a.rho) a.rho[s] = rho;
    if (a.ratio) a.ratio[s] = J / lq::quad<n>(x0, pb.Pexp, x0);
    if (a.flags) a.flags[s] = f;
    if (a.gA) {
#pragma unroll
      for (int e = 0; e < n * n; ++e) a.gA[(int64_t)e * a.S + s] = gA[e];
    }
    if (a.gB) {
#pragma unroll
      for (int e = 0; e < n * m; ++e) a.gB[(int64_t)e * a.S + s] = gB[e];
    }
  }
}

// The inputs are read with plain loads: dA_out / dB_out may alias dA / dB (each thread reads its sample first).
template <int n, int m>
__global__ void __launch_bounds__(128) worst_case_kernel(const __grid_constant__ lq::Problem<n, m> pb,
                                                         const __grid_constant__ WorstArgs a) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  const lq::WsView ws{a.ws + tid, nthreads};
  const lq::AscentSettings as{a.eA, a.eB, a.tol, a.norm, a.max_iter};
  for (int64_t s = tid; s < a.S; s += nthreads) {
    double dA[n * n], dB[n * m], x0[n], J, rho;
    load_sample<n, m>(a, s, dA, dB, x0);
    int it;
    const int f = lq::worst_ascent<n, m>(pb, dA, dB, x0, a.N, as, ws, &J, &rho, &it);
    if (a.dA_out) {
#pragma unroll
      for (int e = 0; e < n * n; ++e) a.dA_out[(int64_t)e * a.S + s] = dA[e];
    }
    if (a.dB_out) {
#pragma unroll
      for (int e = 0; e < n * m; ++e) a.dB_out[(int64_t)e * a.S + s] = dB[e];
    }
    if (a.J) a.J[s] = J;
    if (a.rho) a.rho[s] = rho;
    if (a.ratio) a.ratio[s] = J / lq::quad<n>(x0, pb.Pexp, x0);
    if (a.iters) a.iters[s] = it;
    if (a.flags) a.flags[s] = f;
  }
}

// Sup over x0 (worst.cuh's SUP mode): gamma -> a.J, x* -> x_worst [n][S], the eigengap -> gap [S]. The gradient is
// computed only when gA or gB is requested; the value-only call gets no workspace (a.ws = nullptr) and touches none.
template <int n, int m>
__global__ void __launch_bounds__(128) ratio_sup_kernel(const __grid_constant__ lq::Problem<n, m> pb,
                                                        const __grid_constant__ WorstArgs a, double* x_worst,
                                                        double* gap) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  const lq::WsView ws{a.ws ? a.ws + tid : nullptr, nthreads};
  const bool grad = a.gA || a.gB;
  const lq::ExpertFactor<n> ef = lq::expert_factor<n, m>(pb);
  for (int64_t s = tid; s < a.S; s += nthreads) {
    double dA[n * n], dB[n * m], gA[n * n], gB[n * m], xs[n], J, rho, g;
    load_error<n, m>(a, s, dA, dB);
    const int f = lq::worst_eval<n, m, true>(pb, dA, dB, nullptr, a.N, ws, &J, &rho, grad ? gA : nullptr,
                                             grad ? gB : nullptr, &ef, xs, &g);
    if (a.J) a.J[s] = J;
    if (a.rho) a.rho[s] = rho;
    if (gap) gap[s] = g;
    if (a.flags) a.flags[s] = f;
    store_soa<n>(x_worst, a.S, s, xs);
    store_soa<n * n>(a.gA, a.S, s, gA);
    store_soa<n * m>(a.gB, a.S, s, gB);
  }
}

// The ascent of gamma; inputs read with plain loads as worst_case_kernel's (dA_out / dB_out may alias dA / dB).
template <int n, int m>
__global__ void __launch_bounds__(128) worst_case_sup_kernel(const __grid_constant__ lq::Problem<n, m> pb,
                                                             const __grid_constant__ WorstArgs a, double* x_worst,
                                                             double*) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  const lq::WsView ws{a.ws + tid, nthreads};
  const lq::AscentSettings as{a.eA, a.eB, a.tol, a.norm, a.max_iter};
  const lq::ExpertFactor<n> ef = lq::expert_factor<n, m>(pb);
  for (int64_t s = tid; s < a.S; s += nthreads) {
    double dA[n * n], dB[n * m], xs[n], J, rho;
    load_error<n, m>(a, s, dA, dB);
    int it;
    const int f = lq::worst_ascent<n, m, true>(pb, dA, dB, nullptr, a.N, as, ws, &J, &rho, &it, &ef, xs);
    store_soa<n * n>(a.dA_out, a.S, s, dA);
    store_soa<n * m>(a.dB_out, a.S, s, dB);
    if (a.J) a.J[s] = J;
    if (a.rho) a.rho[s] = rho;
    if (a.iters) a.iters[s] = it;
    if (a.flags) a.flags[s] = f;
    store_soa<n>(x_worst, a.S, s, xs);
  }
}

template <int n, int m, bool ASCENT>
int launch_worst_t(lqmpc_ctx* ctx, WorstArgs a) {
  const lq::Problem<n, m>& pb = *reinterpret_cast<const lq::Problem<n, m>*>(ctx->pb);
  const int threads = 128;
  const int64_t blocks = ASCENT ? lq_worst_blocks(ctx, (const void*)worst_case_kernel<n, m>, threads, a.S)
                                : lq_worst_blocks(ctx, (const void*)eval_grad_kernel<n, m>, threads, a.S);
  const int64_t nthreads = blocks * threads;
  const int64_t per = lq::worst_ws_doubles<n, m>(a.N);
  int rc = lq_reserve_ws(ctx, (size_t)(per * nthreads) * sizeof(double) + 64);
  if (rc) return rc;
  a.ws = reinterpret_cast<double*>(ctx->ws);
  if (ASCENT)
    worst_case_kernel<n, m><<<(unsigned)blocks, threads, 0, ctx->stream>>>(pb, a);
  else
    eval_grad_kernel<n, m><<<(unsigned)blocks, threads, 0, ctx->stream>>>(pb, a);
  ctx->launches++;
  return lq_check_cuda(ctx, cudaGetLastError(), ASCENT ? "worst_case_kernel launch" : "eval_grad_kernel launch");
}

template <int n, int m, bool ASCENT>
int launch_sup_t(lqmpc_ctx* ctx, WorstArgs a, double* x_worst, double* gap) {
  const lq::Problem<n, m>& pb = *reinterpret_cast<const lq::Problem<n, m>*>(ctx->pb);
  const int threads = 128;
  const auto kernel = ASCENT ? worst_case_sup_kernel<n, m> : ratio_sup_kernel<n, m>;
  const int64_t blocks = lq_worst_blocks(ctx, (const void*)kernel, threads, a.S);
  a.ws = nullptr;
  if (ASCENT || a.gA || a.gB) {
    const int64_t per = lq::worst_ws_doubles<n, m>(a.N);
    int rc = lq_reserve_ws(ctx, (size_t)(per * blocks * threads) * sizeof(double) + 64);
    if (rc) return rc;
    a.ws = reinterpret_cast<double*>(ctx->ws);
  }
  kernel<<<(unsigned)blocks, threads, 0, ctx->stream>>>(pb, a, x_worst, gap);
  ctx->launches++;
  return lq_check_cuda(ctx, cudaGetLastError(), ASCENT ? "worst_case_sup_kernel launch" : "ratio_sup_kernel launch");
}

}  // namespace

// Grid of every worst-case launch: one sample per thread, capped at one wave of resident CTAs of `kernel`.
int64_t lq_worst_blocks(lqmpc_ctx* ctx, const void* kernel, int threads, int64_t S) {
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
  int occ = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, 0);
  if (occ < 1) occ = 1;
  int64_t cap = (int64_t)sms * occ;
  // LQMPC_WORST_CTAS: a smaller grid cap, so that tests can run several samples per thread at small batch sizes
  if (const char* v = getenv("LQMPC_WORST_CTAS")) { if (atoi(v) > 0 && atoi(v) < cap) cap = atoi(v); }
  int64_t blocks = (S + threads - 1) / threads;
  if (blocks > cap) blocks = cap;
  return blocks;
}

int lq_launch_eval_grad(lqmpc_ctx* ctx, const WorstArgs& a) {
#define X(N_, M_) \
  if (ctx->n == N_ && ctx->m == M_) return launch_worst_t<N_, M_, false>(ctx, a);
  LQ_FOR_EACH_DIM(X)
#undef X
  return lq_set_error(ctx, LQMPC_EINVAL, "unsupported (n, m); see lqmpc_supported_dims()");
}

int lq_launch_worst_case(lqmpc_ctx* ctx, const WorstArgs& a) {
#define X(N_, M_) \
  if (ctx->n == N_ && ctx->m == M_) return launch_worst_t<N_, M_, true>(ctx, a);
  LQ_FOR_EACH_DIM(X)
#undef X
  return lq_set_error(ctx, LQMPC_EINVAL, "unsupported (n, m); see lqmpc_supported_dims()");
}

int lq_launch_ratio_sup(lqmpc_ctx* ctx, const WorstArgs& a, double* x_worst, double* gap) {
#define X(N_, M_) \
  if (ctx->n == N_ && ctx->m == M_) return launch_sup_t<N_, M_, false>(ctx, a, x_worst, gap);
  LQ_FOR_EACH_DIM(X)
#undef X
  return lq_set_error(ctx, LQMPC_EINVAL, "unsupported (n, m); see lqmpc_supported_dims()");
}

int lq_launch_worst_case_sup(lqmpc_ctx* ctx, const WorstArgs& a, double* x_worst) {
#define X(N_, M_) \
  if (ctx->n == N_ && ctx->m == M_) return launch_sup_t<N_, M_, true>(ctx, a, x_worst, nullptr);
  LQ_FOR_EACH_DIM(X)
#undef X
  return lq_set_error(ctx, LQMPC_EINVAL, "unsupported (n, m); see lqmpc_supported_dims()");
}
