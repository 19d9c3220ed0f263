// k_eval.cu — K1: unconstrained certainty-equivalent MPC evaluation, one sample per thread; two per thread for
// one-horizon launches at n <= 4 (sm_100a).
//
// Data movement: SoA operands, element e of sample s at ptr[e*ld + s]; a warp reads 32 consecutive samples of one
// element (256 B, two full 128 B lines) with read-only, no-L1-allocate loads; every output is written the same way.
// The problem constants arrive as a __grid_constant__ kernel parameter, i.e. in the constant bank: FMAs read
// A, B, Q, R, Pexp as uniform constant operands and spend no registers on them.
#include <stdlib.h>

#include "engine.h"
#include "sampler.cuh"

namespace {

__device__ __forceinline__ double ld_stream(const double* p) {
  double v;
  asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ void st_stream(double* p, double v) {
  asm volatile("st.global.L1::no_allocate.f64 [%0], %1;" ::"l"(p), "d"(v));
}

template <int n, int m>
struct DeviceSink {
  const EvalArgs& a;
  int64_t s;
  __device__ __forceinline__ void operator()(int h, double J, double rho, double ratio, double vn, double JT,
                                             int flags, const double* K) const {
    const int64_t o = (int64_t)h * a.ld + s;
    if (a.J) st_stream(a.J + o, J);
    if (a.rho) st_stream(a.rho + o, rho);
    if (a.ratio) st_stream(a.ratio + o, ratio);
    if (a.Vn) st_stream(a.Vn + o, vn);
    if (a.JT) st_stream(a.JT + o, JT);
    if (a.flags) a.flags[o] = flags;
    if (a.K0) {
#pragma unroll
      for (int e = 0; e < m * n; ++e) st_stream(a.K0 + ((int64_t)h * (m * n) + e) * a.ld + s, K[e]);
    }
  }
};

// MINB = minimum resident CTAs per SM the register allocator must allow (occupancy vs. spills; see K1Tune below)
// kLyapPoly: closed-loop cost from the characteristic polynomial where accepted (riccati.cuh, n = 3, 4)
template <int n, int m, int MINB, int THREADS = 128, bool kLyapPoly = true>
__global__ void __launch_bounds__(THREADS, MINB) eval_kernel(const __grid_constant__ lq::Problem<n, m> pb,
                                                         const __grid_constant__ EvalArgs a) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= a.S) return;
  double dA[n * n], dB[n * m], x0[n];
#pragma unroll
  for (int e = 0; e < n * n; ++e) dA[e] = ld_stream(a.dA + (int64_t)e * a.ld + s);
#pragma unroll
  for (int e = 0; e < n * m; ++e) dB[e] = ld_stream(a.dB + (int64_t)e * a.ld + s);
#pragma unroll
  for (int e = 0; e < n; ++e) x0[e] = ld_stream(a.x0 + (int64_t)e * a.ld + s);
  DeviceSink<n, m> sink{a, s};
  lq::eval_sample<n, m, DeviceSink<n, m>, kLyapPoly>(pb, dA, dB, x0, a.N_min, a.N_max, a.T, a.Vn != nullptr, sink);
}

// Same evaluation with the operands DRAWN IN THE KERNEL from the global sample index (sampler.cuh: seeded_sample):
// no operand traffic at all — the fused "generate + evaluate" entry point north_star's Philox design implies.
template <int n, int m, int MINB, bool kLyapPoly = true>
__global__ void __launch_bounds__(128, MINB) eval_seeded_kernel(const __grid_constant__ lq::Problem<n, m> pb,
                                                                const __grid_constant__ EvalArgs a,
                                                                const uint64_t seed, const int64_t first,
                                                                const double e_A, const double e_B) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= a.S) return;
  double dA[n * n], dB[n * m], x0[n];
  lq::seeded_sample<n, m>(seed, first + s, e_A, e_B, dA, dB, x0);
  DeviceSink<n, m> sink{a, s};
  lq::eval_sample<n, m, DeviceSink<n, m>, kLyapPoly>(pb, dA, dB, x0, a.N_min, a.N_max, a.T, a.Vn != nullptr, sink);
}

// ---- two samples per thread (one horizon, n <= 4). One sample per thread leaves the FP64 pipe about a third idle at 8
// warps per SM: each Riccati step is a single dependency chain (PB -> G -> Cholesky -> solve -> P - YY' -> products).
// Here a thread carries two samples through ONE straight-line Riccati loop body, so the scheduler always has a second
// chain to issue from. Each sample runs eval_sample's operation sequence unchanged, so every output is bit-identical
// to eval_kernel's. The closed loop runs once per sample in a loop that is not unrolled, with the sample's K and x0
// picked by selects: one copy of its code (instruction cache) and no dynamically indexed array (local memory).
constexpr int kPairThreads = 128;   // a CTA covers 2 * 128 consecutive samples: s0 = 256 b + t, s1 = s0 + 128

template <int n, int m, bool kLyapPoly>
__device__ __forceinline__ void eval_pair(const lq::Problem<n, m>& pb, const EvalArgs& a, int64_t s0, bool has1,
                                          const double (&Ah)[2][n * n], const double (&Bh)[2][n * m],
                                          const double (&x0)[2][n]) {
  const int N = a.N_max;
  const bool want_vn = a.Vn != nullptr;
  double P[2][n * n], v_exp[2];
  LQ_UNROLL for (int p = 0; p < 2; ++p) {
    LQ_UNROLL for (int i = 0; i < n * n; ++i) P[p][i] = pb.Pt[i];
    v_exp[p] = lq::quad<n>(x0[p], pb.Pexp, x0[p]);
  }
  lq::RicStage<n, m> st[2];
  int sticky[2] = {0, 0};
  for (int k = 1; k < N; ++k) {            // horizons 1..N-1: cost-to-go only
    LQ_UNROLL for (int p = 0; p < 2; ++p) {
      lq::riccati_factor<n, m>(P[p], Bh[p], pb.R, st[p]);
      if (!st[p].ok) sticky[p] |= lq::FLAG_CHOL_FAIL;
      lq::riccati_update<n, m>(st[p], Ah[p], pb.Q, P[p]);
    }
  }
  double K[2][m * n], vn[2];
  LQ_UNROLL for (int p = 0; p < 2; ++p) {  // horizon N: the gain, and the horizon-N cost-to-go only for Vn
    lq::riccati_factor<n, m>(P[p], Bh[p], pb.R, st[p]);
    if (!st[p].ok) sticky[p] |= lq::FLAG_CHOL_FAIL;
    lq::riccati_gain<n, m>(st[p], Ah[p], K[p]);
    if (want_vn) lq::riccati_update<n, m>(st[p], Ah[p], pb.Q, P[p]);
    vn[p] = want_vn ? lq::quad<n>(x0[p], P[p], x0[p]) : 0.0;
  }
#pragma unroll 1
  for (int p = 0; p < 2; ++p) {
    const bool second = p != 0;
    if (second && !has1) break;
    double Kp[m * n], xp[n];
    LQ_UNROLL for (int e = 0; e < m * n; ++e) Kp[e] = second ? K[1][e] : K[0][e];
    LQ_UNROLL for (int i = 0; i < n; ++i) xp[i] = second ? x0[1][i] : x0[0][i];
    int flags = second ? sticky[1] : sticky[0];
    double J, rho, JT = 0.0;
    lq::closed_loop_eval<n, m, kLyapPoly>(pb, Kp, xp, a.T, &J, &rho, &JT, &flags);
    DeviceSink<n, m> sink{a, second ? s0 + kPairThreads : s0};
    sink(0, J, rho, J / (second ? v_exp[1] : v_exp[0]), second ? vn[1] : vn[0], JT, flags, Kp);
  }
}

// Tail: where s1 >= S the second slot runs the Riccati recursion on s0's operands and stores nothing.
template <int n, int m, bool kLyapPoly>
__global__ void __launch_bounds__(kPairThreads, 2) eval_pair_kernel(const __grid_constant__ lq::Problem<n, m> pb,
                                                                    const __grid_constant__ EvalArgs a) {
  const int64_t s0 = (int64_t)blockIdx.x * (2 * kPairThreads) + threadIdx.x;
  if (s0 >= a.S) return;
  const bool has1 = s0 + kPairThreads < a.S;
  const int64_t s1 = has1 ? s0 + kPairThreads : s0;
  double Ah[2][n * n], Bh[2][n * m], x0[2][n];
  LQ_UNROLL for (int p = 0; p < 2; ++p) {
    const int64_t s = p ? s1 : s0;
    LQ_UNROLL for (int e = 0; e < n * n; ++e) Ah[p][e] = pb.A[e] + ld_stream(a.dA + (int64_t)e * a.ld + s);
    LQ_UNROLL for (int e = 0; e < n * m; ++e) Bh[p][e] = pb.B[e] + ld_stream(a.dB + (int64_t)e * a.ld + s);
    LQ_UNROLL for (int e = 0; e < n; ++e) x0[p][e] = ld_stream(a.x0 + (int64_t)e * a.ld + s);
  }
  eval_pair<n, m, kLyapPoly>(pb, a, s0, has1, Ah, Bh, x0);
}

// The seeded entry point with two samples per thread. The draws run in a loop that is not unrolled (one copy of the
// Philox / Box-Muller code); after the first pass both slots hold s0's draw, so a tail thread skips the second. A^ and
// B^ are formed inside the loop, right after the draw: there the compiler fuses e_A u + A into one FMA as it does in
// eval_seeded_kernel, which keeps the two kernels bit-identical (across the loop boundary it could not).
template <int n, int m, bool kLyapPoly>
__global__ void __launch_bounds__(kPairThreads, 2) eval_pair_seeded_kernel(const __grid_constant__ lq::Problem<n, m> pb,
                                                                           const __grid_constant__ EvalArgs a,
                                                                           const uint64_t seed, const int64_t first,
                                                                           const double e_A, const double e_B) {
  const int64_t s0 = (int64_t)blockIdx.x * (2 * kPairThreads) + threadIdx.x;
  if (s0 >= a.S) return;
  const bool has1 = s0 + kPairThreads < a.S;
  double Ah[2][n * n], Bh[2][n * m], x0[2][n];
#pragma unroll 1
  for (int p = 0; p < 2; ++p) {
    if (p != 0 && !has1) break;
    double tA[n * n], tB[n * m], tx[n];
    lq::seeded_sample<n, m>(seed, first + s0 + (p != 0 ? kPairThreads : 0), e_A, e_B, tA, tB, tx);
    LQ_UNROLL for (int e = 0; e < n * n; ++e) {
      const double v = pb.A[e] + tA[e];
      if (p == 0) Ah[0][e] = v;
      Ah[1][e] = v;
    }
    LQ_UNROLL for (int e = 0; e < n * m; ++e) {
      const double v = pb.B[e] + tB[e];
      if (p == 0) Bh[0][e] = v;
      Bh[1][e] = v;
    }
    LQ_UNROLL for (int e = 0; e < n; ++e) { if (p == 0) x0[0][e] = tx[e]; x0[1][e] = tx[e]; }
  }
  eval_pair<n, m, kLyapPoly>(pb, a, s0, has1, Ah, Bh, x0);
}

template <int n, int m>
__global__ void prepare_kernel(lq::Problem<n, m>* pb, int N_opc) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    lq::Problem<n, m> local = *pb;
    lq::prepare_problem<n, m>(local, N_opc);
    *pb = local;
  }
}

// Register budget per (n, m) and mode: 128-thread CTAs, MINB CTAs/SM -> 65536 / (128 MINB) registers per thread.
#ifndef LQ_K1_THREADS_SINGLE
// CTA size / resident CTAs of the one-horizon launch (A/B switches). Registers map to resident warps in steps of four
// (255 -> 8, 168 -> 12, 128 -> 16 warps per SM), so smaller CTAs open no new occupancy point; at 8 warps per SM CTAs of
// 128 / 64 / 32 threads measured 3.425 / 3.416 / 3.409 ms per 1.25e7 evals (within run-to-run noise): 128 stays.
#define LQ_K1_THREADS_SINGLE 128
#endif
#ifndef LQ_K1_MINB_SINGLE
#define LQ_K1_MINB_SINGLE 2
#endif
template <int n, int m>
struct K1Tune {
  // measured on B200 (n=4 m=2, 1.25e7 samples; DESIGN.md §5). From a cold power state
  // every budget ties for one horizon per sample (2 / 3 / 4 / 5 CTAs per SM: 3.50 / 3.61 / 3.55 / 3.51 ms), but the
  // kernel runs into the board's power cap and SUSTAINED the spill-free 255-register build wins clearly
  // (3.49 / 3.73 / 3.89 / 3.97 ms: spill traffic and the extra instructions cost power, i.e. clock). With all horizons
  // 1..10 emitted the order flips (18.0 / 16.4 / 15.9 / 15.6 ms sustained): occupancy hides the per-horizon stores.
  static constexpr int minb_single = LQ_K1_MINB_SINGLE;       // N_min == N_max
  static constexpr int threads_single = LQ_K1_THREADS_SINGLE;
  static constexpr int minb_nested = (n <= 4) ? 4 : 2;  // several horizons per sample
};

// LQMPC_K1_LYAP=doubling (n = 3, 4): the closed-loop cost by Lyapunov doubling for every sample (development A/B)
bool k1_lyap_doubling() {
  const char* v = getenv("LQMPC_K1_LYAP");
  return v && v[0] == 'd';
}

// LQMPC_K1_PAIR=0: one sample per thread for one-horizon launches at n <= 4 too (the reference the tests compare the
// two-sample kernels against, and the A/B)
bool k1_pair() {
  const char* v = getenv("LQMPC_K1_PAIR");
  return !(v && v[0] == '0');
}

template <int n, int m, bool kLyapPoly>
int launch_eval_impl(lqmpc_ctx* ctx, const EvalArgs& a, cudaStream_t stream) {
  const lq::Problem<n, m>& pb = *reinterpret_cast<const lq::Problem<n, m>*>(ctx->pb);
  const int threads = 128;
  const int64_t blocks = (a.S + threads - 1) / threads;
  if (blocks > 0x7fffffffLL) return lq_set_error(ctx, LQMPC_EINVAL, "batch too large for one launch");
  if (a.N_min == a.N_max) {
    if constexpr (n <= 4)
      if (k1_pair()) {
        const int64_t bp = (a.S + 2 * kPairThreads - 1) / (2 * kPairThreads);
        eval_pair_kernel<n, m, kLyapPoly><<<(unsigned)bp, kPairThreads, 0, stream>>>(pb, a);
        ctx->launches++;
        return lq_check_cuda(ctx, cudaGetLastError(), "eval_pair_kernel launch");
      }
    constexpr int ts = (n <= 4) ? K1Tune<n, m>::threads_single : 128, mb = (n <= 4) ? K1Tune<n, m>::minb_single : 2;
    const int64_t bs = (a.S + ts - 1) / ts;
    if (bs > 0x7fffffffLL) return lq_set_error(ctx, LQMPC_EINVAL, "batch too large for one launch");
    eval_kernel<n, m, mb, ts, kLyapPoly><<<(unsigned)bs, ts, 0, stream>>>(pb, a);
  } else
    eval_kernel<n, m, K1Tune<n, m>::minb_nested, 128, kLyapPoly><<<(unsigned)blocks, threads, 0, stream>>>(pb, a);
  ctx->launches++;
  return lq_check_cuda(ctx, cudaGetLastError(), "eval_kernel launch");
}

template <int n, int m>
int launch_eval_t(lqmpc_ctx* ctx, const EvalArgs& a, cudaStream_t stream) {
  if constexpr (n == 3 || n == 4)
    if (k1_lyap_doubling()) return launch_eval_impl<n, m, false>(ctx, a, stream);
  return launch_eval_impl<n, m, true>(ctx, a, stream);
}

template <int n, int m, bool kLyapPoly>
int launch_eval_seeded_impl(lqmpc_ctx* ctx, const EvalArgs& a, uint64_t seed, int64_t first, double e_A,
                            double e_B) {
  const lq::Problem<n, m>& pb = *reinterpret_cast<const lq::Problem<n, m>*>(ctx->pb);
  const int threads = 128;
  const int64_t blocks = (a.S + threads - 1) / threads;
  if (blocks > 0x7fffffffLL) return lq_set_error(ctx, LQMPC_EINVAL, "batch too large for one launch");
  if constexpr (n <= 4)
    if (a.N_min == a.N_max && k1_pair()) {
      const int64_t bp = (a.S + 2 * kPairThreads - 1) / (2 * kPairThreads);
      eval_pair_seeded_kernel<n, m, kLyapPoly><<<(unsigned)bp, kPairThreads, 0, ctx->stream>>>(pb, a, seed, first, e_A, e_B);
      ctx->launches++;
      return lq_check_cuda(ctx, cudaGetLastError(), "eval_pair_seeded_kernel launch");
    }
  if (a.N_min == a.N_max)
    eval_seeded_kernel<n, m, K1Tune<n, m>::minb_single, kLyapPoly><<<(unsigned)blocks, threads, 0, ctx->stream>>>(pb, a, seed, first, e_A, e_B);
  else
    eval_seeded_kernel<n, m, K1Tune<n, m>::minb_nested, kLyapPoly><<<(unsigned)blocks, threads, 0, ctx->stream>>>(pb, a, seed, first, e_A, e_B);
  ctx->launches++;
  return lq_check_cuda(ctx, cudaGetLastError(), "eval_seeded_kernel launch");
}

template <int n, int m>
int launch_eval_seeded_t(lqmpc_ctx* ctx, const EvalArgs& a, uint64_t seed, int64_t first, double e_A, double e_B) {
  if constexpr (n == 3 || n == 4)
    if (k1_lyap_doubling()) return launch_eval_seeded_impl<n, m, false>(ctx, a, seed, first, e_A, e_B);
  return launch_eval_seeded_impl<n, m, true>(ctx, a, seed, first, e_A, e_B);
}

template <int n, int m>
int launch_prepare_t(lqmpc_ctx* ctx) {
  using P = lq::Problem<n, m>;
  if (ctx->pb_dev == nullptr) {
    int rc = lq_check_cuda(ctx, cudaMalloc(&ctx->pb_dev, sizeof(lq::Problem<LQ_MAX_N, LQ_MAX_M>)), "cudaMalloc pb");
    if (rc) return rc;
  }
  int rc = lq_check_cuda(ctx, cudaMemcpyAsync(ctx->pb_dev, ctx->pb, sizeof(P), cudaMemcpyHostToDevice, ctx->stream),
                         "H2D problem");
  if (rc) return rc;
  prepare_kernel<n, m><<<1, 32, 0, ctx->stream>>>(reinterpret_cast<P*>(ctx->pb_dev), ctx->N_opc);
  ctx->launches++;
  rc = lq_check_cuda(ctx, cudaGetLastError(), "prepare_kernel launch");
  if (rc) return rc;
  rc = lq_check_cuda(ctx, cudaMemcpyAsync(ctx->pb, ctx->pb_dev, sizeof(P), cudaMemcpyDeviceToHost, ctx->stream),
                     "D2H problem");
  if (rc) return rc;
  return lq_check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "prepare sync");
}

// ---- FP64 peak: 8 independent DFMA chains per thread
__global__ void __launch_bounds__(256) dfma_kernel(double* out, int iters, double a, double b) {
  double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
  for (int i = 0; i < iters; ++i) {
    x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
    x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
  }
  const double r = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
  if (r == 123.456) out[0] = r;
}

}  // namespace

int lq_launch_eval(lqmpc_ctx* ctx, const EvalArgs& a, cudaStream_t stream) {
  // n = 6, 8: lane-group kernel (k_group.cu) when LQMPC_K1_GROUP is unset; LQMPC_K1_GROUP=0: thread per sample
  if (lq_group_supported(ctx->n, ctx->m)) {
    const char* v = getenv("LQMPC_K1_GROUP");
    if (!(v && v[0] == '0')) return lq_launch_eval_group(ctx, a, stream);
  }
#define X(N_, M_) \
  if (ctx->n == N_ && ctx->m == M_) return launch_eval_t<N_, M_>(ctx, a, stream);
  LQ_FOR_EACH_DIM(X)
#undef X
  return lq_set_error(ctx, LQMPC_EINVAL, "unsupported (n, m); see lqmpc_supported_dims()");
}

int lq_launch_eval_seeded(lqmpc_ctx* ctx, const EvalArgs& a, uint64_t seed, int64_t first, double e_A, double e_B) {
  if (lq_group_supported(ctx->n, ctx->m)) {
    const char* v = getenv("LQMPC_K1_GROUP");
    if (!(v && v[0] == '0')) return lq_launch_eval_group_seeded(ctx, a, seed, first, e_A, e_B);
  }
#define X(N_, M_) \
  if (ctx->n == N_ && ctx->m == M_) return launch_eval_seeded_t<N_, M_>(ctx, a, seed, first, e_A, e_B);
  LQ_FOR_EACH_DIM(X)
#undef X
  return lq_set_error(ctx, LQMPC_EINVAL, "unsupported (n, m); see lqmpc_supported_dims()");
}

int lq_launch_prepare(lqmpc_ctx* ctx) {
#define X(N_, M_) \
  if (ctx->n == N_ && ctx->m == M_) return launch_prepare_t<N_, M_>(ctx);
  LQ_FOR_EACH_DIM(X)
#undef X
  return lq_set_error(ctx, LQMPC_EINVAL, "unsupported (n, m); see lqmpc_supported_dims()");
}

int lq_launch_fp64_peak(lqmpc_ctx* ctx, double* tflops) {
  int rc = lq_reserve_ws(ctx, 64);
  if (rc) return rc;
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
  const int blocks = sms * 8, threads = 256, iters = 1 << 15;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  double best = 0.0;
  for (int rep = 0; rep < 4; ++rep) {
    cudaEventRecord(e0, ctx->stream);
    dfma_kernel<<<blocks, threads, 0, ctx->stream>>>(reinterpret_cast<double*>(ctx->ws), iters, 0.999999, 1e-9);
    ctx->launches++;
    cudaEventRecord(e1, ctx->stream);
    rc = lq_check_cuda(ctx, cudaEventSynchronize(e1), "dfma sync");
    if (rc) break;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    const double fl = 2.0 * 8.0 * (double)iters * (double)blocks * (double)threads;
    const double tf = fl / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *tflops = best;
  return rc;
}
