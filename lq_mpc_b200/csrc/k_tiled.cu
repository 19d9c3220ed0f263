// k_tiled.cu — K4: certainty-equivalent MPC evaluation for LARGER state dimensions (n = 16, 32; BASELINE cfg 5:
// n = 32, m = 8, N = 30), where one system no longer fits one thread's registers.
//
// Same math as K1 (riccati.cuh; reference semantics utils_class.py:48-91, 245-285, stability check utils.py:358),
// different mapping:
//   * k4a `tiled_eval_kernel<n,m>`: ONE CTA (128 threads) PER SAMPLE, persistent over the batch. The sample's
//     (dA, dB, x0) — contiguous in the array-of-matrices layout this path uses — are staged into shared memory by the
//     TMA engine (cp.async.bulk + mbarrier complete_tx); A^, P and the n x n temporaries live in shared memory
//     (leading dimension n+4: the MMA fragment footprints hit the 32 banks with the minimum 2 wavefronts); every
//     matrix product — n x n x n and the skinny n x 8 ones alike — is a set of warp-level FP64 tensor-core MMAs
//     (mma.sync m8n8k4.f64 -> DMMA).
//     The Riccati step is arranged so that the serial 8 x 8 Cholesky chain runs on ONE warp while the other three keep
//     the tensor pipe busy:   P+ = Q + A^'P A^ - W W',  W = Z L^-T,  Z = A^'(P B^),  G = R + B^'P B^ = L L'
//     — only W depends on the factorisation; X = P A^ and T = Q + A^'X (lower blocks, mirrored: P stays exactly
//     symmetric) do not. The Cholesky is replicated in the registers of every lane of the chain warp (no shuffles,
//     no shared-memory round trips on the serial stretch). Lyapunov doubling accumulates M'(S M) straight into S from the GEMM
//     epilogue. The spectral radius comes from the SAME squarings carried on with exact power-of-two rescaling:
//     rho = lim ||A_cl^(2^k)||^(1/2^k). A sample whose dominant eigenvalue is real, a +- pair or a complex pair is
//     accepted after typically 9-14 squarings from the traces of two successive powers (roots of z^2 - t z + d,
//     reproduced by two successive squarings); the others run 40 squarings and are accepted when the k = 34 and
//     k = 40 norm estimates agree to 5e-10 (then the error is ~1e-11 or better); anything else is left to k4b.
//   * k4b `tiled_rho_kernel<n>`: ONE WARP PER PENDING SAMPLE: Householder -> Hessenberg and the Francis double-shift
//     QR iteration run warp-synchronously on a shared-memory copy of A_cl (lane = row or column of the 3-row/3-column
//     reflector updates), scalars replicated across lanes. Only samples k4a did not accept (LQMPC_K4_RHO=qr: all).
#include <stdio.h>
#include <stdlib.h>

#include "engine.h"

namespace {

constexpr int kT = 128;
#ifndef LQ_K4_KUNROLL
#define LQ_K4_KUNROLL 8          // k-steps of a warp tile unrolled together: 1 / 2 / 4 / 8 measured 36.9 / 34.75 / 34.2 / 33.6 ms per 1.25e5 evals at 32 x 8 x 30
#endif
constexpr int kKUnroll = LQ_K4_KUNROLL;

// ------------------------------------------------------------------------------------------------ TMA / mbarrier
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// ------------------------------------------------------------------------------------------------ block helpers
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// all threads get the result; `red` holds >= 2*kT/32 doubles; contains the barriers that order its reuse
__device__ __forceinline__ double block_sum(double v, double* red) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = red[0];
#pragma unroll
  for (int w = 1; w < kT / 32; ++w) t += red[w];
  return t;
}
__device__ __forceinline__ void block_max2(double& a, double& b, double* red) {
  a = warp_max(a);
  b = warp_max(b);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5] = a; red[kT / 32 + (threadIdx.x >> 5)] = b; }
  __syncthreads();
  double ta = red[0], tb = red[kT / 32];
#pragma unroll
  for (int w = 1; w < kT / 32; ++w) { ta = fmax(ta, red[w]); tb = fmax(tb, red[kT / 32 + w]); }
  a = ta; b = tb;
}

// Magnitude reductions on the INTEGER path: for finite doubles the order of |v| is the order of the sign-stripped bit
// pattern, its high word alone fixes the binary exponent (all the rescaling and the convergence tests need), and a NaN
// or Inf sorts above every finite value, so it surfaces in the maximum. One redux.sync per warp, one barrier per block
// — an FP64 fmax/shuffle chain here would queue behind the other CTAs' tensor-core MMAs on the shared FP64 pipe
// (profile r01k4d: 20 % of k4a's stall samples sat in that chain).
__device__ __forceinline__ unsigned hi_abs(double v) { return (unsigned)__double2hiint(v) & 0x7fffffffu; }
__device__ __forceinline__ double from_hi(unsigned h) { return __hiloint2double((int)h, 0); }
__device__ __forceinline__ bool hi_nonfinite(unsigned h) { return (h >> 20) == 0x7ffu; }
// `slot`: 2 * kT/32 unsigned, not touched by a reduction less than one barrier old (callers alternate two groups)
__device__ __forceinline__ void block_max2_u32(unsigned& a, unsigned& b, unsigned* slot) {
  a = __reduce_max_sync(0xffffffffu, a);
  b = __reduce_max_sync(0xffffffffu, b);
  if ((threadIdx.x & 31) == 0) { slot[threadIdx.x >> 5] = a; slot[kT / 32 + (threadIdx.x >> 5)] = b; }
  __syncthreads();
  unsigned ta = slot[0], tb = slot[kT / 32];
#pragma unroll
  for (int w = 1; w < kT / 32; ++w) { ta = max(ta, slot[w]); tb = max(tb, slot[kT / 32 + w]); }
  a = ta; b = tb;
}

// max of `a` and sum of `t` over the block behind ONE barrier (same slot discipline as block_max2_u32)
__device__ __forceinline__ void block_max_u32_sum(unsigned& a, double& t, unsigned* uslot, double* dslot) {
  a = __reduce_max_sync(0xffffffffu, a);
  t = warp_sum(t);
  if ((threadIdx.x & 31) == 0) { uslot[threadIdx.x >> 5] = a; dslot[threadIdx.x >> 5] = t; }
  __syncthreads();
  unsigned ta = uslot[0];
  double tt = dslot[0];
#pragma unroll
  for (int w = 1; w < kT / 32; ++w) { ta = max(ta, uslot[w]); tt += dslot[w]; }
  a = ta; t = tt;
}

// ------------------------------------------------------------------------------------------------ warp-level MMA
// Every matrix product of the Riccati step and of the Lyapunov doubling goes through ONE routine: a warp accumulates an
// (8 MT) x (8 NT) block of C = A B as m8n8k4 FP64 tensor-core MMAs (mma.sync -> DMMA), operands read
// straight from shared memory in fragment order:
//     A fragment: lane (g = lane/4, tg = lane%4) holds A(row g, col tg)     B fragment: B(row tg, col g)
//     C fragment: C(row g, cols 2 tg, 2 tg + 1)
// Leading dimensions are chosen == 4 (mod 16) doubles (n + 4 for the n x n buffers, 12 for the n x 8 ones): the 8 x 4
// and 4 x 8 fragment footprints then map onto the 32 banks with exactly 2 wavefronts per 256-byte fragment, the
// minimum. (Round-1 profile of the first version — 2 x 4 DFMA register tiles, leading dimension n + 2 — showed the
// kernel bound by shared-memory wavefronts: 84 % of the LSU peak, 55 % of them bank conflicts.)
__device__ __forceinline__ void dmma_m8n8k4(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

template <int MT, int NT, class FA, class FB>
__device__ __forceinline__ void warp_mma(int K, int r0, int c0, FA fa, FB fb, double (&c)[MT][NT][2]) {
  const int lane = threadIdx.x & 31, g = lane >> 2, tg = lane & 3;
#pragma unroll
  for (int i = 0; i < MT; ++i)
#pragma unroll
    for (int j = 0; j < NT; ++j) c[i][j][0] = c[i][j][1] = 0.0;
#pragma unroll kKUnroll
  for (int k0 = 0; k0 < K; k0 += 4) {
    double av[MT], bv[NT];
#pragma unroll
    for (int i = 0; i < MT; ++i) av[i] = fa(r0 + 8 * i + g, k0 + tg);
#pragma unroll
    for (int j = 0; j < NT; ++j) bv[j] = fb(k0 + tg, c0 + 8 * j + g);
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
      for (int j = 0; j < NT; ++j) dmma_m8n8k4(c[i][j][0], c[i][j][1], av[i], bv[j]);
  }
}

// visit the C fragment: epi(row, col, value)
template <int MT, int NT, class Epi>
__device__ __forceinline__ void warp_mma_store(int r0, int c0, const double (&c)[MT][NT][2], Epi epi) {
  const int lane = threadIdx.x & 31, g = lane >> 2, tg = lane & 3;
#pragma unroll
  for (int i = 0; i < MT; ++i)
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      epi(r0 + 8 * i + g, c0 + 8 * j + 2 * tg, c[i][j][0]);
      epi(r0 + 8 * i + g, c0 + 8 * j + 2 * tg + 1, c[i][j][1]);
    }
}

// C = opA * B for n x n shared-memory operands (leading dimension LD), 4 warps, warp tile (n/2) x (n/2)
template <int n, bool TA, class Epi>
__device__ __forceinline__ void gemm_nn(const double* __restrict__ A, const double* __restrict__ B, Epi epi) {
  constexpr int LD = n + 4, T = n / 16;
  const int w = threadIdx.x >> 5;
  const int r0 = (w >> 1) * (n / 2), c0 = (w & 1) * (n / 2);
  double c[T][T][2];
  warp_mma<T, T>(n, r0, c0,
                 [&](int i, int k) { return TA ? A[k * LD + i] : A[i * LD + k]; },
                 [&](int k, int j) { return B[k * LD + j]; }, c);
  warp_mma_store<T, T>(r0, c0, c, epi);
}

// ------------------------------------------------------------------------------------------------ k4a
constexpr int kRhoK1 = 34, kRhoK2 = 40;          // squarings behind the two spectral-radius estimates
constexpr double kRhoEta = 1e-9;                  // dominant-pair early acceptance: consistency of successive candidates
constexpr double kRhoMinRoot = 0.02;              //   ... and the smallest root / max|X| ratio a candidate may have
constexpr int kFlagRhoPending = 1 << 30;          // internal: k4b still owes this entry its QR iteration

struct TiledArgs {
  int64_t S;
  const double* dA;      // [S][n*n]  (array of matrices: one sample contiguous)
  const double* dB;      // [S][n*m]
  const double* x0;      // [S][n]
  const double* pb;      // device: A | B | Q | R | Pt | Pexp
  int N_min, N_max;
  double* Jraw;          // [H][S]   scratch: x0' S x0 of the entries left to k4b
  double* vexp;          // [S]
  double* Vn;            // [H][S] or NULL
  int32_t* flags;        // [H][S]
  double* Acl;           // [H][S][n*n]  closed-loop matrices of the entries left to k4b
  double* Pout;          // [n*n] or NULL: final cost-to-go of sample 0 (problem preparation: the expert matrix)
  double* J;             // [H][S] outputs finished here when the squaring estimate is accepted (any may be NULL)
  double* rho;
  double* ratio;
  int rho_qr;            // 1: leave every spectral radius to k4b
  int rho_sub;           // 1: try the dominant-subspace early exit during the squarings (default)
};

template <int n, int m>
struct PbOff {
  static constexpr int A = 0, B = n * n, Q = B + n * m, R = Q + n * n, Pt = R + m * m, Pexp = Pt + n * n;
};

// shared-memory plan (doubles). M8 = 8: the input dimension is padded to one MMA tile (m = 4 -> zero columns).
template <int n, int m>
struct K4Smem {
  static constexpr int LD = n + 4, NN = n * LD, LS = 12, M8 = 8;
  static constexpr int oBh = 0, oPB = oBh + n * LS, oZ = oPB + n * LS, oKg = oZ + n * LS, oRK = oKg + M8 * LD,
                       oG = oRK + M8 * LD, oRs = oG + M8 * LS, oxs = oRs + M8 * LS, ored = oxs + n,
                       obar = ored + 6 * (kT / 32), total = obar + 2;
  static_assert(M8 * LD >= n * m, "dB lands dense in the RK area");
  static_assert((oxs % 2) == 0 && (oRK % 2) == 0 && (oG % 2) == 0, "TMA destinations / 16-byte loads must be aligned");
};

// 1/sqrt(x) for normal x > 0: hardware seed (MUFU.RSQ64H) + two Newton steps, no slow path (callers flag x <= 0).
__device__ __forceinline__ double fast_rsqrt(double x) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  const double h = 0.5 * x;
  double e = fma(-h * y, y, 0.5);
  y = fma(y, e, y);
  e = fma(-h * y, y, 0.5);
  return fma(y, e, y);
}

// named barrier 1: the three worker warps signal "Z is in shared memory", the chain warp waits for it
__device__ __forceinline__ void z_ready_arrive() {
  __threadfence_block();
  asm volatile("bar.arrive 1, %0;" ::"r"(kT) : "memory");
}
__device__ __forceinline__ void z_ready_wait() { asm volatile("bar.sync 1, %0;" ::"r"(kT) : "memory"); }

#ifdef LQ_K4_PROFILE
// development build only: cycles per warp and phase (0 stage, 1 phase A, 2 phase B, 3 phase D, 4 closed loop,
// 5 Lyapunov, 6 squarings, 7 hand-over / finish), accumulated in shared memory and added to a global table at exit
#define K4_PROF(idx) do { if (lane == 0) { const long long t_ = clock64(); sprof[w * 8 + (idx)] += t_ - tlast; tlast = t_; } } while (0)
__device__ unsigned long long g_k4_prof[4 * 8];
#else
#define K4_PROF(idx) do { } while (0)
#endif

// register allocation held to 5 CTAs per SM (<= 102 registers): shared memory fits 5 single-horizon CTAs
template <int n, int m>
__global__ void __launch_bounds__(kT, 5) tiled_eval_kernel(const TiledArgs a, const int nbig) {
  using L = K4Smem<n, m>;
  using O = PbOff<n, m>;
  constexpr int LD = L::LD, NN = L::NN, LS = L::LS, M8 = L::M8, NW = n / 8, T = n / 16, HB = n / 2;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* sm = reinterpret_cast<double*>(smem_raw);
  double* big[5];
  for (int i = 0; i < 5; ++i) big[i] = sm + (i < nbig ? i : nbig - 1) * NN;
  double* sk = sm + nbig * NN;
  double* Bh = sk + L::oBh;             // n x 8 (ld 12), columns >= m are zero
  double* PB = sk + L::oPB;             // n x 8: P B^, later W = Z L^-T
  double* Z = sk + L::oZ;               // n x 8: A^' (P B^)
  double* Kg = sk + L::oKg;             // 8 x n (ld LD), rows >= m are zero
  double* RK = sk + L::oRK;             // 8 x n; also the TMA landing zone of dB
  double* G = sk + L::oG;               // 8 x 8 (ld 12)
  double* Rs = sk + L::oRs;             // 8 x 8 (ld 12): R padded with the identity
  double* xs = sk + L::oxs;             // n
  double* red = sk + L::ored;           // 6 * (kT/32): two slots for block_sum/block_max2, two (as unsigned) + two for the squarings
  uint64_t* bar = reinterpret_cast<uint64_t*>(sk + L::obar);
  int* cflag = reinterpret_cast<int*>(bar + 1);

  const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
#ifdef LQ_K4_PROFILE
  __shared__ unsigned long long sprof[4 * 8];
  if (tid < 32) sprof[tid] = 0;
  long long tlast = clock64();
#endif
  const int cw = blockIdx.x & 3;                       // chain warp of this CTA
  const int widx = (w - cw - 1) & 3;                   // 0..2 for the workers, 3 for the chain warp
  const bool nested = (a.N_min != a.N_max);
  double* Ah = big[0];
  double* P = big[1];
  double* X = big[2];
  double* Mb = nested ? big[3] : big[0];     // single emit (last step): A^ and P are dead, reuse their storage
  double* Sb = nested ? big[4] : big[1];
  const double* gA = a.pb + O::A;
  const double* gB = a.pb + O::B;
  const double* gQ = a.pb + O::Q;
  const double* gR = a.pb + O::R;
  const double* gPt = a.pb + O::Pt;
  const double* gPexp = a.pb + O::Pexp;

  if (tid == 0) {
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int e = tid; e < M8 * LS; e += kT) {
    const int i = e / LS, j = e % LS;
    Rs[e] = (i < m && j < m) ? __ldg(gR + i * m + j) : ((i == j && j < M8) ? 1.0 : 0.0);
  }
  __syncthreads();
  uint32_t parity = 0;

  for (int64_t s = blockIdx.x; s < a.S; s += gridDim.x) {
    // ---- stage this sample's perturbations through the TMA engine (dense), then build A^ = A + dA, B^ = B + dB
    if (tid == 0) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // prior generic-proxy smem writes vs async proxy
      mbar_expect_tx(bar, (uint32_t)((n * n + n * m + n) * sizeof(double)));
      tma_bulk_g2s(X, a.dA + s * (int64_t)(n * n), n * n * sizeof(double), bar);
      tma_bulk_g2s(RK, a.dB + s * (int64_t)(n * m), n * m * sizeof(double), bar);
      tma_bulk_g2s(xs, a.x0 + s * (int64_t)n, n * sizeof(double), bar);
    }
    mbar_wait(bar, parity);
    parity ^= 1;
    for (int e = tid; e < n * n; e += kT) {
      const int i = e / n, j = e % n;
      Ah[i * LD + j] = __ldg(gA + e) + X[e];
      P[i * LD + j] = __ldg(gPt + e);
    }
    for (int e = tid; e < n * M8; e += kT) {
      const int i = e / M8, j = e % M8;
      Bh[i * LS + j] = (j < m) ? __ldg(gB + i * m + j) + RK[i * m + j] : 0.0;
    }
    if (tid == 0) *cflag = 0;
    __syncthreads();
    for (int e = tid; e < M8 * LD; e += kT) { Kg[e] = 0.0; RK[e] = 0.0; }
    // V_expert(x0) = x0' Pexp x0
    double ve = 0.0;
    for (int e = tid; e < n * n; e += kT) ve = fma(xs[e / n] * __ldg(gPexp + e), xs[e % n], ve);
    ve = block_sum(ve, red);
    if (tid == 0 && a.vexp) a.vexp[s] = ve;

    K4_PROF(0);
    for (int k = 1; k <= a.N_max; ++k) {
      const bool emit = (k >= a.N_min);
      const bool advance = (k < a.N_max || a.Vn || a.Pout);       // the cost-to-go of this step is still needed
      // ---- phase A (all warps): P B^ (n x 8; warp w < n/8 owns row tile w) and X = P A^ (quadrants)
      if (w < NW) {
        double c[1][1][2];
        warp_mma<1, 1>(n, 8 * w, 0, [&](int i, int q) { return P[i * LD + q]; },
                       [&](int q, int j) { return Bh[q * LS + j]; }, c);
        warp_mma_store<1, 1>(8 * w, 0, c, [&](int i, int j, double v) { PB[i * LS + j] = v; });
      }
      if (advance) gemm_nn<n, false>(P, Ah, [&](int i, int j, double v) { X[i * LD + j] = v; });
      __syncthreads();
      K4_PROF(1);
      // ---- phase B: the chain warp factorises G while the workers form Z and the part of P+ that does not need it
      if (w == cw) {
        {
          double c[1][1][2];
          warp_mma<1, 1>(n, 0, 0, [&](int i, int q) { return Bh[q * LS + i]; },
                         [&](int q, int j) { return PB[q * LS + j]; }, c);
          warp_mma_store<1, 1>(0, 0, c, [&](int i, int j, double v) { G[i * LS + j] = Rs[i * LS + j] + v; });
        }
        __syncwarp();
        // Cholesky G = L L' replicated in the registers of every lane (broadcast loads; fully unrolled, no shuffles):
        // lo[i][j] holds L(i, j) for i > j, the reciprocal of the diagonal sits in li[].
        double lo[M8][M8], li[M8];
#pragma unroll
        for (int i = 0; i < M8; ++i) {
#pragma unroll
          for (int j = 0; j <= i; j += 2) {
            const double2 v2 = *reinterpret_cast<const double2*>(G + i * LS + j);
            lo[i][j] = v2.x;
            if (j + 1 <= i) lo[i][j + 1] = v2.y;
          }
        }
        bool bad = false;
#pragma unroll
        for (int j = 0; j < M8; ++j) {
          const double d = lo[j][j];
          bad = bad || !(d > 0.0);
          const double inv = fast_rsqrt(d);
          li[j] = inv;
#pragma unroll
          for (int i = j + 1; i < M8; ++i) lo[i][j] *= inv;
#pragma unroll
          for (int i = j + 1; i < M8; ++i)
#pragma unroll
            for (int cc = j + 1; cc <= i; ++cc) lo[i][cc] = fma(-lo[i][j], lo[cc][j], lo[i][cc]);
        }
        if (bad && lane == 0) atomicOr(cflag, (int)lq::FLAG_CHOL_FAIL);
        z_ready_wait();
        // W = Z L^-T, one row per lane; at an emitting step the gain K = -L^-T W' follows, one column per lane
        if (lane < n) {
          double wv[M8];
#pragma unroll
          for (int j = 0; j < M8; j += 2) {
            const double2 v2 = *reinterpret_cast<const double2*>(Z + lane * LS + j);
            wv[j] = v2.x; wv[j + 1] = v2.y;
          }
#pragma unroll
          for (int j = 0; j < M8; ++j) {
            double sacc = wv[j];
#pragma unroll
            for (int cc = 0; cc < j; ++cc) sacc = fma(-wv[cc], lo[j][cc], sacc);
            wv[j] = sacc * li[j];
          }
#pragma unroll
          for (int j = 0; j < M8; j += 2)
            *reinterpret_cast<double2*>(PB + lane * LS + j) = make_double2(wv[j], wv[j + 1]);
          if (emit) {
#pragma unroll
            for (int i = M8 - 1; i >= 0; --i) {
              double sacc = wv[i];
#pragma unroll
              for (int cc = i + 1; cc < M8; ++cc) sacc = fma(-lo[cc][i], wv[cc], sacc);
              wv[i] = sacc * li[i];
              Kg[i * LD + lane] = -wv[i];
            }
          }
        }
      } else {
        // Z = A^' (P B^): row tiles over the workers
        for (int t = widx; t < NW; t += 3) {
          double c[1][1][2];
          warp_mma<1, 1>(n, 8 * t, 0, [&](int i, int q) { return Ah[q * LD + i]; },
                         [&](int q, int j) { return PB[q * LS + j]; }, c);
          warp_mma_store<1, 1>(8 * t, 0, c, [&](int i, int j, double v) { Z[i * LS + j] = v; });
        }
        z_ready_arrive();
        // T = Q + A^' X: the three lower (n/2)-blocks, one per worker, mirrored into the upper triangle
        if (advance) {
          const int bi = (widx + 1) >> 1, bj = widx >> 1;            // (0,0), (1,0), (1,1)
          double c[T][T][2];
          warp_mma<T, T>(n, bi * HB, bj * HB, [&](int i, int q) { return Ah[q * LD + i]; },
                         [&](int q, int j) { return X[q * LD + j]; }, c);
          warp_mma_store<T, T>(bi * HB, bj * HB, c, [&](int i, int j, double v) {
            if (i >= j) {
              const double t = __ldg(gQ + i * n + j) + v;
              P[i * LD + j] = t;
              P[j * LD + i] = t;
            }
          });
        }
      }
      K4_PROF(2);
      __syncthreads();
      // ---- phase D (all warps): P+ = T - W W'
      if (advance) {
        const int r0 = (w >> 1) * HB, c0 = (w & 1) * HB;
        double c[T][T][2];
        warp_mma<T, T>(M8, r0, c0, [&](int i, int q) { return PB[i * LS + q]; },
                       [&](int q, int j) { return PB[j * LS + q]; }, c);
        warp_mma_store<T, T>(r0, c0, c, [&](int i, int j, double v) { P[i * LD + j] -= v; });
        __syncthreads();
        if (a.Pout && s == 0 && k == a.N_max) {            // problem preparation: the horizon-N cost-to-go itself
          for (int e = tid; e < n * n; e += kT) a.Pout[e] = P[(e / n) * LD + e % n];
        }
      }
      K4_PROF(3);
      if (!emit) continue;
      const int h = k - a.N_min;
      const int64_t o = (int64_t)h * a.S + s;
      if (a.Vn) {
        double vn = 0.0;
        for (int e = tid; e < n * n; e += kT) vn = fma(xs[e / n] * P[(e / n) * LD + e % n], xs[e % n], vn);
        vn = block_sum(vn, red);
        if (tid == 0) a.Vn[o] = vn;
      }
      // ---- closed loop on the TRUE plant: R K (8 x n), then A_cl = A + B K -> Mb, W = Q + K' R K -> Sb
      if (w < NW) {
        double c[1][1][2];
        warp_mma<1, 1>(M8, 0, 8 * w, [&](int i, int q) { return Rs[i * LS + q]; },
                       [&](int q, int j) { return Kg[q * LD + j]; }, c);
        warp_mma_store<1, 1>(0, 8 * w, c, [&](int i, int j, double v) { RK[i * LD + j] = v; });
      }
      __syncthreads();
      {
        const int r0 = (w >> 1) * HB, c0 = (w & 1) * HB;
        double c[T][T][2];
        warp_mma<T, T>(M8, r0, c0, [&](int i, int q) { return (q < m) ? __ldg(gB + i * m + q) : 0.0; },
                       [&](int q, int j) { return Kg[q * LD + j]; }, c);
        warp_mma_store<T, T>(r0, c0, c, [&](int i, int j, double v) { Mb[i * LD + j] = __ldg(gA + i * n + j) + v; });
        warp_mma<T, T>(M8, r0, c0, [&](int i, int q) { return Kg[q * LD + i]; },
                       [&](int q, int j) { return RK[q * LD + j]; }, c);
        warp_mma_store<T, T>(r0, c0, c, [&](int i, int j, double v) { Sb[i * LD + j] = __ldg(gQ + i * n + j) + v; });
      }
      __syncthreads();
      K4_PROF(4);
      // ---- Lyapunov squared doubling: S += M' (S M), M <- M^2
      int lflag = lq::FLAG_LYAP_NOCONV, nsq = 64;
      double* Mc = Mb;
      double* Xc = X;
      unsigned* ru = reinterpret_cast<unsigned*>(red + 2 * (kT / 32));     // two groups of 2 * kT/32 unsigned
      int rp = 0;
      for (int it = 0; it < 64; ++it) {
        gemm_nn<n, false>(Sb, Mc, [&](int i, int j, double v) { Xc[i * LD + j] = v; });
        __syncthreads();
        unsigned thi = 0, shi = 0;
        gemm_nn<n, true>(Mc, Xc, [&](int i, int j, double v) {
          const double nv = Sb[i * LD + j] + v;
          Sb[i * LD + j] = nv;
          thi = max(thi, hi_abs(v));
          shi = max(shi, hi_abs(nv));
        });
        block_max2_u32(thi, shi, ru + (rp++ & 1) * (2 * (kT / 32)));     // (its barrier orders the Sb / Xc reuse)
        const double tmax = from_hi(thi), smax = from_hi(shi);            // magnitudes to 2^-20: ample for the tests
        if (hi_nonfinite(thi) || hi_nonfinite(shi)) { lflag = lq::FLAG_NONFINITE; nsq = it; break; }
        if (!(tmax > 1e-18 * smax)) { lflag = 0; nsq = it; break; }
        if (!(smax < 1e300)) { lflag = lq::FLAG_NONFINITE; nsq = it; break; }   // diverging (unstable loop)
        gemm_nn<n, false>(Mc, Mc, [&](int i, int j, double v) { Xc[i * LD + j] = v; });
        __syncthreads();
        double* t = Mc; Mc = Xc; Xc = t;
      }
      double J = 0.0;
      for (int e = tid; e < n * n; e += kT) J = fma(xs[e / n] * Sb[(e / n) * LD + e % n], xs[e % n], J);
      J = block_sum(J, red);
      K4_PROF(5);
      // ---- spectral radius: keep squaring M = A_cl^(2^nsq) with exact power-of-two rescaling,
      //      log2 rho ~ sum_j 2^-j e_j + 2^-k log2 max|N_k|  (N_k the stored, rescaled power; e_j its exponent)
      double rho = 0.0;
      bool accepted = false;
      if (!a.rho_qr && nsq < kRhoK1) {
        // max |N| to full precision (only the two estimates need the mantissa)
        auto absmax = [&](const double* Mm) {
          double mx = 0.0, dummy = 0.0;
          for (int e = tid; e < n * n; e += kT) mx = fmax(mx, fabs(Mm[(e / n) * LD + e % n]));
          block_max2(mx, dummy, red);
          return mx;
        };
        unsigned mh = 0, dm = 0;
        for (int e = tid; e < n * n; e += kT) mh = max(mh, hi_abs(Mc[(e / n) * LD + e % n]));
        block_max2_u32(mh, dm, ru + (rp++ & 1) * (2 * (kT / 32)));
        double lacc = 0.0, wgt = __hiloint2double((1023 - nsq) << 20, 0), est1 = 0.0;
        bool fail = false, zero = false;
        int kk = nsq;
        // Early acceptance through the two dominant eigenvalues (the rule of k_group.cu, where it is derived and
        // its tolerances are explained). With X = 2^-e N_k (max|X| in [1, 2)) and N_(k+1) = X^2: t = tr X, t' = tr X^2,
        // d = (t^2 - t') / 2. When one real eigenvalue, a +- pair or a complex pair dominates, the p-th powers
        // (p = 2^k) of the dominant eigenvalues are the roots of z^2 - t z + d up to (|lambda_3| / |lambda_1|)^p, so
        // rho^p = sqrt(d) (complex roots) or the larger root modulus. A candidate must not be tiny against max|X|
        // (ill-conditioned or defective dominant eigenvalues leave rounding noise in the traces) nor nearly double,
        // and is ACCEPTED when two successive squarings reproduce it, r_k 2^(e_k) = r_(k-1)^2 to kRhoEta; everything
        // else runs on to the norm-based two-estimate test below (and to the QR kernel when that fails too).
        // Replaces round 2's Krylov-vector subspace test, which needed 3 extra mat-vecs per probe and still ran
        // ~30 squarings on most samples; this one costs one trace per squaring and typically stops after 9-14.
        bool sub_ok = false;
        double tr_cur = 0.0, rr_prev = 0.0;
        int streak = -1;
        {
          double tq = 0.0;
          for (int e = tid; e < n; e += kT) tq += Mc[e * LD + e];
          tr_cur = block_sum(tq, red);
        }
        double* dsl = red + 4 * (kT / 32);
        for (; kk < kRhoK2; ++kk) {
          if (hi_nonfinite(mh)) { fail = true; break; }
          if ((mh >> 20) == 0) {                             // a vanishing power: A_cl^(2^kk) = 0 (or subnormal).
            zero = (kk <= 6);                                // Nilpotent (rho = 0) if that early; later it is underflow
            fail = !zero;                                    // of the entries that carry rho (huge Jordan blocks) -> QR
            break;
          }
          if (kk == kRhoK1) est1 = fma(lacc, 0.6931471805599453, wgt * log(absmax(Mc)));
          const int e = (int)(mh >> 20) - 1023;
          if (e < -500 || e > 500) { fail = true; break; }
          // (2^-e N)^2 with the scale applied to the LEFT operand on load: the stored power keeps its full dynamic
          // range (a product of two unnormalised operands would underflow the small entries that carry rho)
          const double s2 = __hiloint2double((1023 - 2 * e) << 20, 0);
          unsigned lh = 0;
          double trn = 0.0;
          {
            const int r0 = (w >> 1) * HB, c0 = (w & 1) * HB;
            double c[T][T][2];
            warp_mma<T, T>(n, r0, c0, [&](int i, int q) { return Mc[i * LD + q] * s2; },
                           [&](int q, int j) { return Mc[q * LD + j]; }, c);
            warp_mma_store<T, T>(r0, c0, c, [&](int i, int j, double v) {
              Xc[i * LD + j] = v;
              lh = max(lh, hi_abs(v));
              if (i == j) trn += v;
            });
          }
          lacc = fma(wgt, (double)e, lacc);
          block_max_u32_sum(lh, trn, ru + (rp & 1) * (2 * (kT / 32)), dsl + (rp & 1) * (kT / 32));
          ++rp;
          if (a.rho_sub) {
            const double sc = __hiloint2double((1023 - e) << 20, 0);
            const double tau = tr_cur * sc, t2 = tau * tau;
            const double d = 0.5 * (t2 - trn), disc = fma(2.0, trn, -t2);
            const double rr = (disc < 0.0) ? sqrt(d) : 0.5 * (fabs(tau) + sqrt(disc));
            if ((rr > kRhoMinRoot) && (rr < 1e300) && !(fabs(disc) < 1e-4 * t2)) {
              const bool same = (streak >= 0) && fabs(rr - rr_prev * rr_prev * sc) <= kRhoEta * rr;
              if (same && streak >= 1 && kRhoEta * wgt <= 2e-10) {
                rho = exp(fma(lacc, 0.6931471805599453, wgt * log(rr)));
                sub_ok = true;
              }
              streak = same ? streak + 1 : 0;
              rr_prev = rr;
            } else {
              streak = -1;
            }
          }
          tr_cur = trn;
          wgt *= 0.5;
          mh = lh;
          double* t = Mc; Mc = Xc; Xc = t;
          if (sub_ok) break;
        }
        if (sub_ok) {
          accepted = true;
        } else if (!fail) {
          if (zero) {
            accepted = true;
          } else if (hi_nonfinite(mh) || (mh >> 20) == 0) {
            fail = true;
          } else {
            const double est2 = fma(lacc, 0.6931471805599453, wgt * log(absmax(Mc)));
            rho = exp(est2);
            accepted = fabs(rho - exp(est1)) <= 5e-10 * rho;
          }
        }
      }
      K4_PROF(6);
      if (accepted) {
        if (tid == 0) {
          int fl = lflag | *cflag;
          double Jo = J;
          if (!(rho < 1.0)) {
            fl = (fl & ~(lq::FLAG_LYAP_NOCONV | lq::FLAG_NONFINITE)) | lq::FLAG_UNSTABLE;
            Jo = HUGE_VAL;
          } else if (!(fabs(Jo) <= 1.79e308)) {
            fl |= lq::FLAG_NONFINITE;
          }
          if (a.J) a.J[o] = Jo;
          if (a.rho) a.rho[o] = rho;
          if (a.ratio) a.ratio[o] = Jo / ve;
          a.flags[o] = fl;
        }
      } else {
        // left to k4b: hand over A_cl = A + B K (rebuilt from the gain, the doubling consumed the shared-memory copy)
        const int r0 = (w >> 1) * HB, c0 = (w & 1) * HB;
        double c[T][T][2];
        warp_mma<T, T>(M8, r0, c0, [&](int i, int q) { return (q < m) ? __ldg(gB + i * m + q) : 0.0; },
                       [&](int q, int j) { return Kg[q * LD + j]; }, c);
        double* gout = a.Acl + o * (int64_t)(n * n);
        warp_mma_store<T, T>(r0, c0, c, [&](int i, int j, double v) { gout[i * n + j] = __ldg(gA + i * n + j) + v; });
        if (tid == 0) {
          a.Jraw[o] = J;
          a.flags[o] = lflag | *cflag | kFlagRhoPending;
        }
      }
      __syncthreads();
      K4_PROF(7);
    }
    __syncthreads();
  }
#ifdef LQ_K4_PROFILE
  __syncthreads();
  if (tid < 32) atomicAdd(&g_k4_prof[tid], sprof[tid]);
#endif
}

// ------------------------------------------------------------------------------------------------ k4b
struct RhoArgs {
  int64_t total;          // H * S matrices
  const double* Acl;      // [total][n*n]
  const double* Jraw;     // [total]
  const double* vexp;     // [S]
  int64_t S;
  double* J;              // [total] or NULL
  double* rho;            // [total] or NULL
  double* ratio;          // [total] or NULL
  int32_t* flags;         // [total] in/out
};

__device__ __forceinline__ double block2_rho_d(double y, double x, double w) {
  const double p = 0.5 * (y - x);
  const double q = fma(p, p, w);
  const double z = sqrt(fabs(q));
  if (q >= 0.0) {
    const double zz = p + (p >= 0.0 ? z : -z);
    const double r1 = x + zz;
    const double r2 = (zz != 0.0) ? x - w / zz : r1;
    return fmax(fabs(r1), fabs(r2));
  }
  const double re = x + p;
  return sqrt(fma(re, re, z * z));
}

// Warp-synchronous spectral radius of the n x n matrix `a` (shared memory, leading dimension n+1, destroyed).
template <int n>
__device__ double warp_spectral_radius(double* a, double* v, bool* ok) {
  constexpr int LDA = n + 1;
  const int lane = threadIdx.x & 31;
#define A_(i, j) a[(i) * LDA + (j)]
  // ---- Householder reduction to upper Hessenberg form
  for (int k = 0; k < n - 2; ++k) {
    const double xi = (lane > k && lane < n) ? A_(lane, k) : 0.0;
    const double alpha = warp_sum(xi * xi);
    const double x0 = __shfl_sync(0xffffffffu, xi, k + 1);
    if (alpha - x0 * x0 > 0.0) {
      const double nrm = sqrt(alpha);
      const double beta = (x0 >= 0.0) ? -nrm : nrm;
      const double vi = (lane == k + 1) ? x0 - beta : xi;
      const double tau = 2.0 / warp_sum(vi * vi);
      v[lane] = vi;
      __syncwarp();
      if (lane < n) {                                   // A <- (I - tau v v') A : lane = column
        double sacc = 0.0;
        for (int i = k + 1; i < n; ++i) sacc = fma(v[i], A_(i, lane), sacc);
        sacc *= tau;
        for (int i = k + 1; i < n; ++i) A_(i, lane) = fma(-sacc, v[i], A_(i, lane));
      }
      __syncwarp();
      if (lane < n) {                                   // A <- A (I - tau v v') : lane = row
        double sacc = 0.0;
        for (int j = k + 1; j < n; ++j) sacc = fma(A_(lane, j), v[j], sacc);
        sacc *= tau;
        for (int j = k + 1; j < n; ++j) A_(lane, j) = fma(-sacc, v[j], A_(lane, j));
      }
      __syncwarp();
      if (lane > k + 1 && lane < n) A_(lane, k) = 0.0;
      __syncwarp();
    }
  }
  double an = 0.0;
  if (lane < n)
    for (int j = (lane > 0 ? lane - 1 : 0); j < n; ++j) an += fabs(A_(lane, j));
  const double anorm = warp_sum(an);
  // ---- Francis double-shift QR with deflation (EISPACK hqr, eigenvalues only); scalars replicated across lanes
  double rho = 0.0, t = 0.0;
  int nn = n - 1, its = 0, guard = 0;
  *ok = true;
  while (nn >= 0 && guard < 150 * n) {
    ++guard;
    // ---- deflation search, one sub-diagonal per lane: l = highest i <= nn with a negligible a(i, i-1)
    int l = 0;
    {
      bool small = false;
      if (lane >= 1 && lane <= nn) {
        double sd = fabs(A_(lane - 1, lane - 1)) + fabs(A_(lane, lane));
        if (sd == 0.0) sd = anorm;
        small = (fabs(A_(lane, lane - 1)) + sd == sd);
      }
      const unsigned bal = __ballot_sync(0xffffffffu, small);
      if (bal) l = 31 - __clz(bal);
    }
    if (l > 0 && lane == 0) A_(l, l - 1) = 0.0;
    __syncwarp();
    double x = A_(nn, nn);
    if (l == nn) { rho = fmax(rho, fabs(x + t)); nn -= 1; its = 0; continue; }
    double y = A_(nn - 1, nn - 1);
    double w = A_(nn, nn - 1) * A_(nn - 1, nn);
    if (l == nn - 1) { rho = fmax(rho, block2_rho_d(y + t, x + t, w)); nn -= 2; its = 0; continue; }
    if (its >= 120) { *ok = false; break; }
    if (its == 10 || its == 20) {                       // exceptional shift
      t += x;
      __syncwarp();
      if (lane <= nn) A_(lane, lane) -= x;
      __syncwarp();
      const double sd = fabs(A_(nn, nn - 1)) + fabs(A_(nn - 1, nn - 2));
      x = y = 0.75 * sd;
      w = -0.4375 * sd * sd;
    }
    ++its;
    // ---- start row of the bulge, one candidate row per lane: the highest mm in [l, nn-2] whose first reflector
    //      column (p, q, r) passes EISPACK's two-small-subdiagonals test (mm = l always qualifies)
    double p = 0.0, q = 0.0, r = 0.0;
    int mst = l;
    {
      bool cand = false;
      if (lane >= l && lane <= nn - 2) {
        const int mm = lane;
        const double z = A_(mm, mm);
        const double rr = x - z, ss = y - z;
        p = (rr * ss - w) / A_(mm + 1, mm) + A_(mm, mm + 1);
        q = A_(mm + 1, mm + 1) - z - rr - ss;
        r = A_(mm + 2, mm + 1);
        const double isc = 1.0 / (fabs(p) + fabs(q) + fabs(r));
        p *= isc; q *= isc; r *= isc;
        cand = (mm == l);
        if (!cand) {
          const double u = fabs(A_(mm, mm - 1)) * (fabs(q) + fabs(r));
          const double vv = fabs(p) * (fabs(A_(mm - 1, mm - 1)) + fabs(z) + fabs(A_(mm + 1, mm + 1)));
          cand = (u + vv == vv);
        }
      }
      const unsigned bal = __ballot_sync(0xffffffffu, cand);
      mst = 31 - __clz(bal);                            // lane l always votes
      p = __shfl_sync(0xffffffffu, p, mst);
      q = __shfl_sync(0xffffffffu, q, mst);
      r = __shfl_sync(0xffffffffu, r, mst);
    }
    __syncwarp();
    if (lane >= mst + 2 && lane <= nn) {
      A_(lane, lane - 2) = 0.0;
      if (lane != mst + 2) A_(lane, lane - 3) = 0.0;
    }
    __syncwarp();
    for (int k = mst; k <= nn - 1; ++k) {
      const bool last = (k == nn - 1);
      double xsc = 0.0;
      if (k != mst) {
        p = A_(k, k - 1);
        q = A_(k + 1, k - 1);
        r = last ? 0.0 : A_(k + 2, k - 1);
        xsc = fabs(p) + fabs(q) + fabs(r);
        if (xsc != 0.0) { const double ix = lq::rcp(xsc); p *= ix; q *= ix; r *= ix; }
      }
      const double s2 = fma(p, p, fma(q, q, r * r));
      if (s2 == 0.0) continue;
      const double isq = rsqrt(s2);                     // |s| = s2 * isq, 1/|s| = isq (p, q, r are scaled to O(1))
      const double sg = (p >= 0.0) ? s2 * isq : -(s2 * isq);
      const double isg = (p >= 0.0) ? isq : -isq;
      __syncwarp();
      if (lane == 0) {
        if (k == mst) { if (l != mst) A_(k, k - 1) = -A_(k, k - 1); }
        else A_(k, k - 1) = -sg * xsc;
      }
      p += sg;                                          // |p + sg| >= |sg| > 0: same signs
      const double ip = lq::rcp(p);
      const double hx = p * isg, hy = q * isg, hz = r * isg;
      q *= ip; r *= ip;
      if (lane >= k && lane <= nn) {                    // row modification: lane = column
        double pp = A_(k, lane) + q * A_(k + 1, lane);
        if (!last) { pp += r * A_(k + 2, lane); A_(k + 2, lane) -= pp * hz; }
        A_(k + 1, lane) -= pp * hy;
        A_(k, lane) -= pp * hx;
      }
      __syncwarp();
      const int imax = (nn < k + 3) ? nn : k + 3;
      if (lane >= l && lane <= imax) {                  // column modification: lane = row
        double pp = hx * A_(lane, k) + hy * A_(lane, k + 1);
        if (!last) { pp += hz * A_(lane, k + 2); A_(lane, k + 2) -= pp * r; }
        A_(lane, k + 1) -= pp * q;
        A_(lane, k) -= pp;
      }
      __syncwarp();
    }
  }
  if (nn >= 0) *ok = false;
#undef A_
  return rho;
}

template <int n>
__global__ void __launch_bounds__(kT) tiled_rho_kernel(const RhoArgs a) {
  constexpr int LDA = n + 1, PER = n * LDA + 32;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* sm = reinterpret_cast<double*>(smem_raw);
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double* am = sm + wib * PER;
  double* v = am + n * LDA;
  const int64_t wid = (int64_t)blockIdx.x * (kT / 32) + wib, nw = (int64_t)gridDim.x * (kT / 32);
  for (int64_t e = wid; e < a.total; e += nw) {
    if (!(a.flags[e] & kFlagRhoPending)) continue;          // k4a finished this entry (warp-uniform)
    const double* src = a.Acl + e * (int64_t)(n * n);
    for (int q = lane; q < n * n; q += 32) am[(q / n) * LDA + q % n] = src[q];
    __syncwarp();
    bool ok;
    const double rho = warp_spectral_radius<n>(am, v, &ok);
    __syncwarp();
    if (lane == 0) {
      int fl = a.flags[e] & ~kFlagRhoPending;
      if (!ok) fl |= lq::FLAG_EIG_NOCONV;
      double J = a.Jraw[e];
      if (!(rho < 1.0)) {
        fl = (fl & ~(lq::FLAG_LYAP_NOCONV | lq::FLAG_NONFINITE)) | lq::FLAG_UNSTABLE;
        J = HUGE_VAL;
      } else if (!(fabs(J) <= 1.79e308)) {
        fl |= lq::FLAG_NONFINITE;
      }
      if (a.J) a.J[e] = J;
      if (a.rho) a.rho[e] = rho;
      if (a.ratio) a.ratio[e] = J / a.vexp[e % a.S];
      a.flags[e] = fl;
    }
  }
}

template <int n, int m>
size_t k4a_smem_bytes(int nbig) {
  return (size_t)(nbig * K4Smem<n, m>::NN + K4Smem<n, m>::total) * sizeof(double) + 16;
}

template <int n, int m>
int launch_tiled_t(lqmpc_ctx* ctx, const TiledEval& t) {
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
  const int H = t.N_max - t.N_min + 1;
  const int nbig = (H > 1) ? 5 : 3;
  const size_t smem = k4a_smem_bytes<n, m>(nbig);
  // spectral radius: repeated squaring inside k4a with the QR kernel as fallback (default), LQMPC_K4_RHO=qr: QR for all
  const char* rhov = getenv("LQMPC_K4_RHO");
  const int rho_qr = (rhov && rhov[0] == 'q') ? 1 : 0;
  const int rho_sub = (rhov && rhov[0] == 's') ? 0 : 1;     // LQMPC_K4_RHO=sq: squarings with the two-estimate test only
  auto r_J = [](const TiledEval& tt, int64_t s0) { return tt.J ? tt.J + s0 : nullptr; };
  auto r_rho = [](const TiledEval& tt, int64_t s0) { return tt.rho ? tt.rho + s0 : nullptr; };
  auto r_ratio = [](const TiledEval& tt, int64_t s0) { return tt.ratio ? tt.ratio + s0 : nullptr; };
  const auto kern = tiled_eval_kernel<n, m>;
  static uint64_t attr_done = 0;                             // function attributes are per DEVICE: one bit each
  if (!((attr_done >> (ctx->device & 63)) & 1)) {
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k4a_smem_bytes<n, m>(5));
    cudaFuncSetAttribute(tiled_rho_kernel<n>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         (int)((kT / 32) * (n * (n + 1) + 32) * sizeof(double)));
    attr_done |= (uint64_t)1 << (ctx->device & 63);
  }
  int per_sm = 1;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kT, smem);
  if (per_sm < 1) per_sm = 1;
  // A_cl scratch: [H][chunk][n*n]; chunk the batch so that the scratch stays below 4 GiB
  int64_t chunk = t.S;
  const int64_t max_mats = ((int64_t)4 << 30) / (int64_t)(n * n * sizeof(double));
  if ((int64_t)H * chunk > max_mats) chunk = max_mats / H;
  if (chunk < 1) chunk = 1;
  const size_t acl_bytes = (size_t)H * chunk * n * n * sizeof(double);
  const size_t need = acl_bytes + (size_t)(H + 1) * chunk * sizeof(double) + (size_t)H * chunk * sizeof(int32_t);
  int rc = lq_reserve_ws(ctx, need);
  if (rc) return rc;
  double* acl = reinterpret_cast<double*>(ctx->ws);
  double* jraw = acl + (size_t)H * chunk * n * n;
  double* vexp = jraw + (size_t)H * chunk;
  int32_t* fscratch = reinterpret_cast<int32_t*>(vexp + chunk);
  if (t.S > chunk && H > 1)
    return lq_set_error(ctx, LQMPC_EINVAL, "tiled path: nested horizons need the batch to fit one chunk (reduce S or H)");
  for (int64_t s0 = 0; s0 < t.S; s0 += chunk) {
    const int64_t cs = (s0 + chunk <= t.S) ? chunk : t.S - s0;
    TiledArgs a;
    a.S = cs;
    a.dA = t.dA + s0 * (int64_t)(n * n); a.dB = t.dB + s0 * (int64_t)(n * m); a.x0 = t.x0 + s0 * (int64_t)n;
    a.pb = reinterpret_cast<const double*>(ctx->tiled_pb);
    a.N_min = t.N_min; a.N_max = t.N_max;
    a.Jraw = jraw; a.vexp = vexp; a.Vn = t.Vn ? t.Vn + s0 : nullptr; a.flags = t.flags ? t.flags + s0 : fscratch; a.Acl = acl;
    a.Pout = t.Pout;
    a.J = r_J(t, s0); a.rho = r_rho(t, s0); a.ratio = r_ratio(t, s0);
    a.rho_qr = rho_qr;
    a.rho_sub = rho_sub;
    int64_t blocks = (int64_t)sms * per_sm;
    if (blocks > cs) blocks = cs;
    kern<<<(unsigned)blocks, kT, smem, ctx->stream>>>(a, nbig);
    RhoArgs r;
    r.total = (int64_t)H * cs; r.Acl = acl; r.Jraw = jraw; r.vexp = vexp; r.S = cs;
    r.J = t.J ? t.J + s0 : nullptr; r.rho = t.rho ? t.rho + s0 : nullptr; r.ratio = t.ratio ? t.ratio + s0 : nullptr;
    r.flags = a.flags;
    const size_t rsmem = (size_t)(kT / 32) * (n * (n + 1) + 32) * sizeof(double);
    int rper = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&rper, tiled_rho_kernel<n>, kT, rsmem);
    if (rper < 1) rper = 1;
    int64_t rblocks = (int64_t)sms * rper;
    const int64_t wantb = (r.total + kT / 32 - 1) / (kT / 32);
    if (rblocks > wantb) rblocks = wantb;
    tiled_rho_kernel<n><<<(unsigned)rblocks, kT, rsmem, ctx->stream>>>(r);
#ifdef LQ_K4_PROFILE
    if (cs > 1000) {
      unsigned long long hp[32];
      cudaStreamSynchronize(ctx->stream);
      cudaMemcpyFromSymbol(hp, g_k4_prof, sizeof(hp));
      unsigned long long z[32] = {0};
      cudaMemcpyToSymbol(g_k4_prof, z, sizeof(z));
      for (int ww = 0; ww < 4; ++ww) {
        fprintf(stderr, "k4prof warp %d (cycles per sample):", ww);
        for (int q = 0; q < 8; ++q) fprintf(stderr, " %9.0f", (double)hp[ww * 8 + q] / (double)cs);
        fprintf(stderr, "\n");
      }
    }
#endif
    ctx->launches += 2;
    rc = lq_check_cuda(ctx, cudaGetLastError(), "tiled kernels launch");
    if (rc) return rc;
  }
  return 0;
}

}  // namespace

// ---- FP64 tensor-core peak: 8 independent m8n8k4 accumulator chains per warp (the K4 roofline denominator)
namespace {
__global__ void __launch_bounds__(256) dmma_peak_kernel(double* out, int iters, double a, double b) {
  double c[8][2];
#pragma unroll
  for (int i = 0; i < 8; ++i) { c[i][0] = threadIdx.x + i; c[i][1] = threadIdx.x - i; }
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 8; ++i) dmma_m8n8k4(c[i][0], c[i][1], a, b);
  }
  double r = 0.0;
#pragma unroll
  for (int i = 0; i < 8; ++i) r += c[i][0] + c[i][1];
  if (r == 123.456) out[0] = r;
}
}  // namespace

int lq_launch_dmma_peak(lqmpc_ctx* ctx, double* tflops) {
  int rc = lq_reserve_ws(ctx, 64);
  if (rc) return rc;
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
  const int blocks = sms * 8, threads = 256, iters = 1 << 13;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  double best = 0.0;
  for (int rep = 0; rep < 4; ++rep) {
    cudaEventRecord(e0, ctx->stream);
    dmma_peak_kernel<<<blocks, threads, 0, ctx->stream>>>(reinterpret_cast<double*>(ctx->ws), iters, 1e-3, 1e-3);
    ctx->launches++;
    cudaEventRecord(e1, ctx->stream);
    rc = lq_check_cuda(ctx, cudaEventSynchronize(e1), "dmma peak sync");
    if (rc) break;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    // one m8n8k4 MMA = 8*8*4 FMAs = 512 flop per warp
    const double fl = 512.0 * 8.0 * (double)iters * (double)blocks * (double)(threads / 32);
    const double tf = fl / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *tflops = best;
  return rc;
}

bool lq_tiled_supported(int n, int m) { return (n == 32 && m == 8) || (n == 16 && m == 4); }

size_t lq_tiled_pb_doubles(int n, int m) { return (size_t)(4 * n * n + n * m + m * m); }

int lq_launch_tiled(lqmpc_ctx* ctx, const TiledEval& t) {
  if (ctx->tn == 32 && ctx->tm == 8) return launch_tiled_t<32, 8>(ctx, t);
  if (ctx->tn == 16 && ctx->tm == 4) return launch_tiled_t<16, 4>(ctx, t);
  return lq_set_error(ctx, LQMPC_EINVAL, "unsupported tiled (n, m): 32x8 and 16x4 are compiled");
}
