// k_worst.cu — exact gradient of J_inf in the model error and the projected worst-case ascent (worst.cuh), one sample
// per thread, grid-stride over the batch. The stage records of the reverse sweep live in the context workspace laid out
// [element][thread], so a warp touches 32 consecutive doubles per access. The grid is capped at one wave of resident
// CTAs, which keeps the workspace at one wave's worth (as K2's launches do).
#include <stdlib.h>

#include "engine.h"
#include "worst.cuh"

namespace {

template <int n, int m>
__device__ __forceinline__ void load_sample(const WorstArgs& a, int64_t s, double* dA, double* dB, double* x0) {
#pragma unroll
  for (int e = 0; e < n * n; ++e) dA[e] = a.dA[(int64_t)e * a.S + s];
#pragma unroll
  for (int e = 0; e < n * m; ++e) dB[e] = a.dB[(int64_t)e * a.S + s];
#pragma unroll
  for (int e = 0; e < n; ++e) x0[e] = a.x0[(int64_t)e * a.S + s];
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

template <int n, int m, bool ASCENT>
int launch_worst_t(lqmpc_ctx* ctx, WorstArgs a) {
  const lq::Problem<n, m>& pb = *reinterpret_cast<const lq::Problem<n, m>*>(ctx->pb);
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
  const int threads = 128;
  int occ = 0;
  if (ASCENT) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, worst_case_kernel<n, m>, threads, 0);
  else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, eval_grad_kernel<n, m>, threads, 0);
  if (occ < 1) occ = 1;
  int64_t cap = (int64_t)sms * occ;
  // LQMPC_WORST_CTAS: a smaller grid cap, so that tests can run several samples per thread at small batch sizes
  if (const char* v = getenv("LQMPC_WORST_CTAS")) { if (atoi(v) > 0 && atoi(v) < cap) cap = atoi(v); }
  int64_t blocks = (a.S + threads - 1) / threads;
  if (blocks > cap) blocks = cap;
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

}  // namespace

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
