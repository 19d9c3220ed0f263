// k_clqr_impl.cuh — K2 kernels: batched LQ_MPC_Controller.solve / LQ_MPC_Simulator.simulate with the exact input QP.
// Included by k_clqr.cu (POLY = false: input box, clqr.cuh) and k_pclqr.cu (POLY = true: general input polytope,
// pclqr.cuh) so that the two families compile in parallel and the box kernels keep their register budget.
//
// One sample per thread, grid-stride over the batch; the per-thread scratch of clqr.cuh (gains, plan, trajectory)
// lives in a global workspace laid out [element][thread] so that a warp touches 32 consecutive doubles per access.
#pragma once
#include <stdlib.h>
#include "pclqr.cuh"
#include "engine.h"

namespace {

__device__ __forceinline__ double ld_stream(const double* p) {
  double v;
  asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
}

// CTAs per SM the register allocation of the n m <= 2 instantiations is held to (1 = unconstrained). 3 -> 160 registers
// without spills; measured with the stage lookahead of clqr.cuh (see StagePrefetch).
#ifndef LQ_K2_MINB_SMALL
#define LQ_K2_MINB_SMALL 3
#endif
template <int n, int m>
struct K2Occupancy {
  static constexpr int min_blocks = (n * m <= 2) ? LQ_K2_MINB_SMALL : 1;
};

template <int n, int m>
__device__ __forceinline__ void load_plan(const MpcArgs& a, const lq::Problem<n, m>& pb, int64_t s,
                                          lq::Plan<n, m>& pl) {
#pragma unroll
  for (int e = 0; e < n * n; ++e) pl.Ah[e] = pb.A[e] + (a.dA ? ld_stream(a.dA + (int64_t)e * a.S + s) : 0.0);
#pragma unroll
  for (int e = 0; e < n * m; ++e) pl.Bh[e] = pb.B[e] + (a.dB ? ld_stream(a.dB + (int64_t)e * a.S + s) : 0.0);
}

template <int n, int m, bool POLY>
__global__ void __launch_bounds__(128, K2Occupancy<n, m>::min_blocks) mpc_solve_kernel(const __grid_constant__ lq::Problem<n, m> pb,
                                                        const __grid_constant__ MpcArgs a) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  const lq::WsView ws{a.ws + tid, nthreads};
  lq::Refs rf;
  rf.xr = a.xr; rf.ur = a.ur; rf.ld = a.ref_ld;
  for (int64_t s = tid; s < a.S; s += nthreads) {
    lq::Plan<n, m> pl;
    load_plan<n, m>(a, pb, s, pl);
    const int pf = lq::plan_prepare<n, m>(pb, pl, a.N, ws, /*certificate=*/false);
    const int P = a.pts ? a.npts : 1;
    double mv = -HUGE_VAL;
    for (int p = 0; p < P; ++p) {
      double x0[n], u0[m], V;
#pragma unroll
      for (int i = 0; i < n; ++i) x0[i] = a.pts ? a.pts[p * n + i] : a.x0[(int64_t)i * a.S + s];
      int f = pf;
      if (POLY) f |= lq::pclqr_solve<n, m>(pb, pl, a.N, x0, lq::Poly{a.polyF, a.polyP}, ws, u0, &V, rf);
      else f |= lq::clqr_solve<n, m>(pb, pl, a.N, x0, ws, u0, &V, rf);
      mv = lq::dmax(mv, V);
      if (a.V) a.V[(int64_t)p * a.S + s] = V;
      if (a.u0) {
#pragma unroll
        for (int j = 0; j < m; ++j) a.u0[((int64_t)p * m + j) * a.S + s] = u0[j];
      }
      if (a.flags) a.flags[(int64_t)p * a.S + s] = f;
    }
    if (a.M_V) a.M_V[s] = mv;
  }
}

// Horizon range N_min..N_max (box, zero references): ONE unconstrained sweep of N_max stages per sample
// (plan_prepare_range), then the ring solves of every horizon through the stage-offset view of that sweep. Outputs
// V [H][P][S], u0 [H][P][m][S], M_V [H][S], flags [H][P][S]; bit-identical to H single-horizon launches.
template <int n, int m>
__global__ void __launch_bounds__(128, K2Occupancy<n, m>::min_blocks) mpc_solve_range_kernel(
    const __grid_constant__ lq::Problem<n, m> pb, const __grid_constant__ MpcArgs a) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  const lq::WsView ws{a.ws + tid, nthreads};
  const int P = a.pts ? a.npts : 1;
  for (int64_t s = tid; s < a.S; s += nthreads) {
    lq::Plan<n, m> pl;
    load_plan<n, m>(a, pb, s, pl);
    const int first_fail = lq::plan_prepare_range<n, m>(pb, pl, a.N, ws);
    for (int N = a.N_min; N <= a.N; ++N) {
      const int koff = a.N - N;
      const int64_t h = N - a.N_min;
      lq::plan_select_horizon<n, m>(pl, a.N, koff, ws);
      const int pf = (first_fail <= N) ? lq::FLAG_CHOL_FAIL : 0;   // only the N stages of this horizon count
      double mv = -HUGE_VAL;
      for (int p = 0; p < P; ++p) {
        double x0[n], u0[m], V;
#pragma unroll
        for (int i = 0; i < n; ++i) x0[i] = a.pts ? a.pts[p * n + i] : a.x0[(int64_t)i * a.S + s];
        const int f = pf | lq::clqr_solve<n, m>(pb, pl, N, x0, ws, u0, &V, lq::Refs(), koff);
        mv = lq::dmax(mv, V);
        const int64_t hp = h * P + p;
        if (a.V) a.V[hp * a.S + s] = V;
        if (a.u0) {
#pragma unroll
          for (int j = 0; j < m; ++j) a.u0[(hp * m + j) * a.S + s] = u0[j];
        }
        if (a.flags) a.flags[hp * a.S + s] = f;
      }
      if (a.M_V) a.M_V[h * a.S + s] = mv;
    }
  }
}

template <int n, int m>
struct DevTraj {
  const MpcArgs& a;
  int64_t s;
  __device__ __forceinline__ void state(int t, const double* x) const {
    if (a.X) {
#pragma unroll
      for (int i = 0; i < n; ++i) a.X[((int64_t)t * n + i) * a.S + s] = x[i];
    }
  }
  __device__ __forceinline__ void input(int t, const double* u) const {
    if (a.U) {
#pragma unroll
      for (int j = 0; j < m; ++j) a.U[((int64_t)t * m + j) * a.S + s] = u[j];
    }
  }
};

template <int n, int m, bool POLY>
__global__ void __launch_bounds__(128, K2Occupancy<n, m>::min_blocks) simulate_kernel(const __grid_constant__ lq::Problem<n, m> pb,
                                                       const __grid_constant__ MpcArgs a) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  const lq::WsView ws{a.ws + tid, nthreads};
  lq::Refs rf;
  rf.xr = a.xr; rf.ur = a.ur; rf.ld = a.ref_ld;
  for (int64_t s = tid; s < a.S; s += nthreads) {
    lq::Plan<n, m> pl;
    load_plan<n, m>(a, pb, s, pl);
    const int pf = lq::plan_prepare<n, m>(pb, pl, a.N, ws);
    double x0[n];
#pragma unroll
    for (int i = 0; i < n; ++i) x0[i] = a.pts ? a.pts[i] : a.x0[(int64_t)i * a.S + s];
    DevTraj<n, m> traj{a, s};
    double JT;
    int act;
    int f = pf;
    if (POLY) f |= lq::psimulate_sample<n, m>(pb, pl, a.N, a.T, x0, lq::Poly{a.polyF, a.polyP}, ws, &JT, &act, traj, rf);
    else f |= lq::simulate_sample<n, m>(pb, pl, a.N, a.T, x0, ws, &JT, &act, traj, rf);
    if (a.J_T) a.J_T[s] = JT;
    if (a.flags) a.flags[s] = f;
    if (a.n_active) a.n_active[s] = act;
  }
}

template <int n, int m, bool POLY>
int launch_mpc_t(lqmpc_ctx* ctx, MpcArgs a, bool sim) {
  const lq::Problem<n, m>& pb = *reinterpret_cast<const lq::Problem<n, m>*>(ctx->pb);
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
  const int threads = 128;
  int64_t blocks = (a.S + threads - 1) / threads;
  // Grid-stride beyond `cap` CTAs; the per-thread workspace is sized by the LAUNCHED threads. With one wave of resident
  // CTAs every thread keeps rewriting the same few kB, which the 126 MB L2 partly absorbs (N = 50, 1e6 samples:
  // ring solves 5.22 -> 4.66 ms, closed loops 1.56 -> 1.46); short horizons have little scratch and prefer the
  // finer-grained balance of three waves (measured 1 / 2 / 3 waves and the former 16 CTAs per SM, scripts/k2_probe.py).
  int occ = 0;
  if (sim) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, simulate_kernel<n, m, POLY>, threads, 0);
  else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, mpc_solve_kernel<n, m, POLY>, threads, 0);
  if (occ < 1) occ = 1;
  int waves = (a.N >= 20) ? 1 : 3;
  if (const char* wv = getenv("LQMPC_K2_WAVES")) { if (atoi(wv) > 0) waves = atoi(wv); }   // A/B switch
  const int64_t cap = (int64_t)sms * occ * waves;
  if (blocks > cap) blocks = cap;
  const int64_t nthreads = blocks * threads;
  const int64_t per = lq::clqr_ws_doubles<n, m>(a.N);
  int rc = lq_reserve_ws(ctx, (size_t)(per * nthreads) * sizeof(double));
  if (rc) return rc;
  a.ws = reinterpret_cast<double*>(ctx->ws);
  if (ctx->ref_ld >= a.N) { a.xr = ctx->ref_x; a.ur = ctx->ref_u; a.ref_ld = ctx->ref_ld; }
  else if (ctx->ref_ld > 0) return lq_set_error(ctx, LQMPC_EINVAL, "references hold fewer than N columns");
  if (POLY) { a.polyF = ctx->poly_dev; a.polyP = ctx->poly_p; }
  if (sim)
    simulate_kernel<n, m, POLY><<<(unsigned)blocks, threads, 0, ctx->stream>>>(pb, a);
  else
    mpc_solve_kernel<n, m, POLY><<<(unsigned)blocks, threads, 0, ctx->stream>>>(pb, a);
  ctx->launches++;
  return lq_check_cuda(ctx, cudaGetLastError(), sim ? "simulate_kernel launch" : "mpc_solve_kernel launch");
}

template <int n, int m>
int launch_mpc_range_t(lqmpc_ctx* ctx, MpcArgs a) {
  const lq::Problem<n, m>& pb = *reinterpret_cast<const lq::Problem<n, m>*>(ctx->pb);
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
  const int threads = 128;
  int64_t blocks = (a.S + threads - 1) / threads;
  int occ = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, mpc_solve_range_kernel<n, m>, threads, 0);
  if (occ < 1) occ = 1;
  int waves = (a.N >= 20) ? 1 : 3;                       // the grid cap of launch_mpc_t, at the longest horizon
  if (const char* wv = getenv("LQMPC_K2_WAVES")) { if (atoi(wv) > 0) waves = atoi(wv); }
  const int64_t cap = (int64_t)sms * occ * waves;
  if (blocks > cap) blocks = cap;
  const int64_t nthreads = blocks * threads;
  const int64_t per = lq::clqr_range_ws_doubles<n, m>(a.N);
  int rc = lq_reserve_ws(ctx, (size_t)(per * nthreads) * sizeof(double));
  if (rc) return rc;
  a.ws = reinterpret_cast<double*>(ctx->ws);
  mpc_solve_range_kernel<n, m><<<(unsigned)blocks, threads, 0, ctx->stream>>>(pb, a);
  ctx->launches++;
  return lq_check_cuda(ctx, cudaGetLastError(), "mpc_solve_range_kernel launch");
}

}  // namespace
