// k_bounds.cu — K3: batched bound coefficients (alpha, beta, xi, eta, J_bound) and batched dlqr.
// One sample per thread. The extreme eigenvalues of the (N m) x (N m) Gram operators come from the matrix-free
// bisection of gramspec.cuh (registers only, no scratch); only the literal-kron ordering with non-scalar weights (and
// LQMPC_K3_DENSE=1) takes the dense Householder route with its [element][thread] workspace.
#include "bounds.cuh"
#include <stdlib.h>

#include "engine.h"

namespace {

__device__ __forceinline__ double ld_stream(const double* p) {
  double v;
  asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
}

// CTAs per SM the register allocation of the n m <= 2 instantiation is held to (1 = unconstrained; A/B switch).
// Measured on cfg-sweep-f (bounds phase of 5e7 evals): unconstrained (162 registers, 3 CTAs/SM) 0.314 s,
// 4 (128 registers, 96 B of stack) 0.293 s, 5 (96 registers, 200 B) 0.303 s.
#ifndef LQ_K3_MINB_SMALL
#define LQ_K3_MINB_SMALL 4
#endif
// Per-sample operands of both bound kernels: the estimated model, the terminal gain (given, or -K_dlqr of the model
// with the DARE solution written to P_out) and the state energy_bound is evaluated at. Returns the DARE flag.
template <int n, int m>
__device__ __forceinline__ int load_bounds_operands(const lq::Problem<n, m>& pb, const BoundsArgs& a, int64_t s,
                                                    double* Ah, double* Bh, double* K, double* x) {
#pragma unroll
  for (int e = 0; e < n * n; ++e) Ah[e] = pb.A[e] + (a.dA ? ld_stream(a.dA + (int64_t)e * a.S + s) : 0.0);
#pragma unroll
  for (int e = 0; e < n * m; ++e) Bh[e] = pb.B[e] + (a.dB ? ld_stream(a.dB + (int64_t)e * a.S + s) : 0.0);
  int flags = 0;
  if (a.K_in) {
#pragma unroll
    for (int e = 0; e < m * n; ++e) K[e] = a.K_in[(int64_t)e * a.S + s];
  } else if (a.K_shared) {
#pragma unroll
    for (int e = 0; e < m * n; ++e) K[e] = a.K_shared[e];
  } else {
    double X[n * n];
    if (!lq::dare_sda<n, m>(Ah, Bh, pb.Q, pb.R, X)) flags |= lq::FLAG_DARE_NOCONV;
    lq::dlqr_gain<n, m>(Ah, Bh, pb.R, X, K);
#pragma unroll
    for (int e = 0; e < m * n; ++e) K[e] = -K[e];   // callers pass -K_dlqr (utils_class.py:843-844)
    if (a.P_out) {
#pragma unroll
      for (int e = 0; e < n * n; ++e) a.P_out[(int64_t)e * a.S + s] = X[e];
    }
  }
#pragma unroll
  for (int i = 0; i < n; ++i) x[i] = a.x_shared ? a.x_shared[i] : a.x[(int64_t)i * a.S + s];
  return flags;
}

template <int n, int m>
__device__ __forceinline__ lq::BoundsScalars bounds_scalars(const BoundsArgs& a, int64_t s) {
  lq::BoundsScalars sc;
  sc.N = a.N;
  sc.e_A = a.eA ? a.eA[s] : a.eA_s;
  sc.e_B = a.eB ? a.eB[s] : a.eB_s;
  sc.M_V = a.MV ? a.MV[s] : a.MV_s;
  sc.p[0] = a.p[0]; sc.p[1] = a.p[1]; sc.p[2] = a.p[2];
  sc.V_expert = a.V_expert;
  sc.bar_u = a.bar_u; sc.bar_d_u = a.bar_d_u;
  sc.strict_reference = a.strict;
  sc.polyF = a.polyF; sc.polyP = a.polyP;
  sc.force_dense = a.dense;
  return sc;
}

// outputs of horizon slot h ([h][S] tables, detail [h][BF_COUNT][S]; h = 0 for the single-horizon kernel)
__device__ __forceinline__ void store_bounds(const BoundsArgs& a, int64_t h, int64_t s, const double* out, int flags) {
  const int64_t o = h * a.S + s;
  if (a.alpha) a.alpha[o] = out[lq::BF_ALPHA];
  if (a.beta) a.beta[o] = out[lq::BF_BETA];
  if (a.xi) a.xi[o] = out[lq::BF_XI];
  if (a.eta) a.eta[o] = out[lq::BF_ETA];
  if (a.bound) a.bound[o] = out[lq::BF_BOUND];
  if (a.detail) {
#pragma unroll
    for (int f = 0; f < lq::BF_COUNT; ++f) a.detail[(h * lq::BF_COUNT + f) * a.S + s] = out[f];
  }
  if (a.flags) a.flags[o] = flags;
}

template <int n, int m>
__global__ void __launch_bounds__(128, (n * m <= 2) ? LQ_K3_MINB_SMALL : 1) bounds_kernel(const __grid_constant__ lq::Problem<n, m> pb,
                                                     const __grid_constant__ BoundsArgs a) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  const lq::WsView ws{a.ws + tid, nthreads};
  for (int64_t s = tid; s < a.S; s += nthreads) {
    double Ah[n * n], Bh[n * m], K[m * n], x[n];
    int flags = load_bounds_operands<n, m>(pb, a, s, Ah, Bh, K, x);
    const lq::BoundsScalars sc = bounds_scalars<n, m>(a, s);
    double out[lq::BF_COUNT];
    flags |= lq::bounds_sample<n, m>(pb, Ah, Bh, K, x, sc, ws, out);
    store_bounds(a, 0, s, out, flags);
    if (a.K_out) {
#pragma unroll
      for (int e = 0; e < m * n; ++e) a.K_out[(int64_t)e * a.S + s] = K[e];
    }
  }
}

// Horizon range N_min..N (matrix-free route): the operands, DARE, norms, local_radius and rho_cl once per sample
// (bounds_prefix), ||Phi|| and the error-consistent sums extended by one term per horizon (2 pow calls per horizon
// instead of 2 (N + 1)), both Gram extremes of every horizon from one range search (gram_spectrum_range),
// then the per-horizon formulas. M_V is [H][S]; outputs [H][S] / detail [H][BF_COUNT][S];
// K_out / P_out once.
// Occupancy as bounds_kernel. Measured on cfg-sweep-f's bounds phase with the fused horizons (B200, 1000 W):
// 4 CTAs/SM (128 registers, 684 B of spill stores) 0.169 s, 3 (168 registers) 0.181 s, 2 (240, no spills) 0.177 s.
template <int n, int m>
__global__ void __launch_bounds__(128, (n * m <= 2) ? LQ_K3_MINB_SMALL : 1) bounds_range_kernel(
    const __grid_constant__ lq::Problem<n, m> pb, const __grid_constant__ BoundsArgs a) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  for (int64_t s = tid; s < a.S; s += nthreads) {
    double Ah[n * n], Bh[n * m], K[m * n], x[n];
    const int f0 = load_bounds_operands<n, m>(pb, a, s, Ah, Bh, K, x);
    lq::BoundsScalars sc = bounds_scalars<n, m>(a, s);
    const lq::BoundsPrefix pr = lq::bounds_prefix<n, m>(pb, Ah, Bh, K, sc);
    lq::PhiGram<n> phi;
    lq::EcRunning ec = lq::ec_running<n>(pr, sc, x);
    lq::gram_spectrum_range<n, m>(Ah, Bh, pb.Q, pb.R, pb.minR, a.N_min, a.N, [&](int N, const lq::GramSpectrum& gs) {
      const int64_t h = N - a.N_min;
      phi.extend_to(Ah, N);
      sc.N = N;
      sc.M_V = a.MV ? a.MV[h * a.S + s] : a.MV_s;
      double out[lq::BF_COUNT];
#pragma unroll
      for (int i = 0; i < lq::BF_COUNT; ++i) out[i] = 0.0;
      const lq::EcSums es = ec.at(N);
      const int f = f0 | lq::bounds_horizon<n, m>(pb, pr, phi.norm(), gs.cmax, gs.min_H, x, sc, out, &es);
      store_bounds(a, h, s, out, f);
    });
    if (a.K_out) {
#pragma unroll
      for (int e = 0; e < m * n; ++e) a.K_out[(int64_t)e * a.S + s] = K[e];
    }
  }
}

template <int n, int m>
__global__ void __launch_bounds__(128) dlqr_kernel(const __grid_constant__ lq::Problem<n, m> pb, int64_t S,
                                                   const double* dA, const double* dB, double* K_out, double* P_out,
                                                   int32_t* flags) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  double Ah[n * n], Bh[n * m], K[m * n], X[n * n];
#pragma unroll
  for (int e = 0; e < n * n; ++e) Ah[e] = pb.A[e] + (dA ? ld_stream(dA + (int64_t)e * S + s) : 0.0);
#pragma unroll
  for (int e = 0; e < n * m; ++e) Bh[e] = pb.B[e] + (dB ? ld_stream(dB + (int64_t)e * S + s) : 0.0);
  const bool ok = lq::dare_sda<n, m>(Ah, Bh, pb.Q, pb.R, X);
  lq::dlqr_gain<n, m>(Ah, Bh, pb.R, X, K);
  if (K_out) {
#pragma unroll
    for (int e = 0; e < m * n; ++e) K_out[(int64_t)e * S + s] = K[e];
  }
  if (P_out) {
#pragma unroll
    for (int e = 0; e < n * n; ++e) P_out[(int64_t)e * S + s] = X[e];
  }
  if (flags) flags[s] = ok ? 0 : lq::FLAG_DARE_NOCONV;
}

template <int n, int m>
int launch_bounds_t(lqmpc_ctx* ctx, BoundsArgs a) {
  const lq::Problem<n, m>& pb = *reinterpret_cast<const lq::Problem<n, m>*>(ctx->pb);
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
  const int threads = 128;
  int64_t blocks = (a.S + threads - 1) / threads;
  a.dense = getenv("LQMPC_K3_DENSE") != nullptr ? 1 : 0;
  a.ws = nullptr;
  if (!lq::bounds_matrix_free(pb.qr_scalar, a.strict, a.dense)) {
    // dense route: (N m)^2 doubles of scratch per thread — cap the grid and stride over the batch
    const int64_t cap = (int64_t)sms * 8;
    if (blocks > cap) blocks = cap;
    const int64_t per = lq::bounds_ws_doubles<n, m>(a.N);
    int rc = lq_reserve_ws(ctx, (size_t)(per * blocks * threads) * sizeof(double));
    if (rc) return rc;
    a.ws = reinterpret_cast<double*>(ctx->ws);
  } else if (blocks > 0x7fffffffLL) {
    return lq_set_error(ctx, LQMPC_EINVAL, "batch too large for one launch");
  }
  bounds_kernel<n, m><<<(unsigned)blocks, threads, 0, ctx->stream>>>(pb, a);
  ctx->launches++;
  return lq_check_cuda(ctx, cudaGetLastError(), "bounds_kernel launch");
}

// n <= 6 only. Measured on a B200 (1000 W), bounds of N = 1..50 at scalar weights, fused kernel against the 50
// per-horizon launches: (2, 1) 1e6 samples 0.208 vs 0.217 s, (6, 2) 1e5 samples 0.423 vs 0.524 s, (8, 2) 5e4 samples
// 0.933 vs 0.819 s — at n = 8 the range kernel's per-horizon state spills on top of the search (which runs
// non-inlined, gram_range_next_call) and the per-horizon launches are faster, so n = 8 takes them.
template <int n>
constexpr bool kBoundsRangeFused = (n <= 6);

template <int n, int m>
int launch_bounds_range_t(lqmpc_ctx* ctx, BoundsArgs a) {
  if constexpr (!kBoundsRangeFused<n>) {
    return lq_set_error(ctx, LQMPC_EINVAL, "no fused bounds range kernel for this n (per-horizon route)");
  } else {
  const lq::Problem<n, m>& pb = *reinterpret_cast<const lq::Problem<n, m>*>(ctx->pb);
  const int threads = 128;
  int64_t blocks = (a.S + threads - 1) / threads;
  // one sample per thread; LQMPC_K3_RANGE_WAVES caps the grid at that many waves of resident CTAs (grid-stride tests)
  if (const char* wv = getenv("LQMPC_K3_RANGE_WAVES")) {
    int sms = 148, occ = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, bounds_range_kernel<n, m>, threads, 0);
    const int64_t cap = (int64_t)sms * (occ > 0 ? occ : 1) * (atoi(wv) > 0 ? atoi(wv) : 1);
    if (blocks > cap) blocks = cap;
  }
  if (blocks > 0x7fffffffLL) return lq_set_error(ctx, LQMPC_EINVAL, "batch too large for one launch");
  a.ws = nullptr;
  bounds_range_kernel<n, m><<<(unsigned)blocks, threads, 0, ctx->stream>>>(pb, a);
  ctx->launches++;
  return lq_check_cuda(ctx, cudaGetLastError(), "bounds_range_kernel launch");
  }
}

template <int n, int m>
int launch_dlqr_t(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, double* K, double* P,
                  int32_t* flags) {
  const lq::Problem<n, m>& pb = *reinterpret_cast<const lq::Problem<n, m>*>(ctx->pb);
  const int threads = 128;
  const int64_t blocks = (S + threads - 1) / threads;
  dlqr_kernel<n, m><<<(unsigned)blocks, threads, 0, ctx->stream>>>(pb, S, dA, dB, K, P, flags);
  ctx->launches++;
  return lq_check_cuda(ctx, cudaGetLastError(), "dlqr_kernel launch");
}

}  // namespace

int lq_launch_bounds(lqmpc_ctx* ctx, const BoundsArgs& a) {
#define X(N_, M_) \
  if (ctx->n == N_ && ctx->m == M_) return launch_bounds_t<N_, M_>(ctx, a);
  LQ_FOR_EACH_DIM(X)
#undef X
  return lq_set_error(ctx, LQMPC_EINVAL, "unsupported (n, m); see lqmpc_supported_dims()");
}

// The range kernel covers the matrix-free route of the compiled pairs; the dense route answers per horizon.
bool lq_bounds_range_fused(lqmpc_ctx* ctx, const BoundsArgs& a) {
  if (ctx->dyn) return false;
  bool qr_scalar = false, found = false;
#define X(N_, M_)                                                                                  \
  if (!found && ctx->n == N_ && ctx->m == M_) {                                                   \
    qr_scalar = reinterpret_cast<const lq::Problem<N_, M_>*>(ctx->pb)->qr_scalar != 0;            \
    found = kBoundsRangeFused<N_>;                                                                \
    if (!found) return false;                                                                     \
  }
  LQ_FOR_EACH_DIM(X)
#undef X
  return found && lq::bounds_matrix_free(qr_scalar, a.strict, getenv("LQMPC_K3_DENSE") != nullptr ? 1 : 0);
}

int lq_launch_bounds_range(lqmpc_ctx* ctx, const BoundsArgs& a) {
#define X(N_, M_) \
  if (ctx->n == N_ && ctx->m == M_) return launch_bounds_range_t<N_, M_>(ctx, a);
  LQ_FOR_EACH_DIM(X)
#undef X
  return lq_set_error(ctx, LQMPC_EINVAL, "unsupported (n, m); see lqmpc_supported_dims()");
}

int lq_launch_dlqr(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, double* K, double* P,
                   int32_t* flags) {
#define X(N_, M_) \
  if (ctx->n == N_ && ctx->m == M_) return launch_dlqr_t<N_, M_>(ctx, S, dA, dB, K, P, flags);
  LQ_FOR_EACH_DIM(X)
#undef X
  return lq_set_error(ctx, LQMPC_EINVAL, "unsupported (n, m); see lqmpc_supported_dims()");
}
