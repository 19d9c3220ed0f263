// k_stats.cu — K5: per-column statistics of a result table (max, min, sum, counts, squared deviations).
//
// Replaces the four reductions the reference's plotters draw for every column of every table
// (utils.py:895-898: np.max / np.min / np.mean / np.std over axis 0). The table is column-contiguous
// ([cols][ld], column c = the S results of one error level or horizon), so each block streams a slice of one
// column with coalesced 16-byte loads, reduces in registers -> warp shuffles -> shared memory, and writes one
// partial; a second tiny kernel folds the partials in a fixed order (deterministic, no FP atomics).
// np.std is a two-pass algorithm (mean first, then the mean squared deviation); so is this: pass 2 takes the
// (all-reduced) column means. Non-finite entries (J = +inf of unstable loops, NaN) are counted, not accumulated.
#include "engine.h"

namespace {

struct Part {
  double mx, mn, sum, nfin, nbad;
};

__device__ __forceinline__ void acc_one(double v, Part& p) {
  const bool fin = fabs(v) <= 1.79e308;   // false for NaN and +-inf
  if (fin) {
    p.mx = fmax(p.mx, v);
    p.mn = fmin(p.mn, v);
    p.sum += v;
    p.nfin += 1.0;
  } else {
    p.nbad += 1.0;
  }
}

__device__ __forceinline__ Part warp_fold(Part p) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    p.mx = fmax(p.mx, __shfl_xor_sync(0xffffffffu, p.mx, o));
    p.mn = fmin(p.mn, __shfl_xor_sync(0xffffffffu, p.mn, o));
    p.sum += __shfl_xor_sync(0xffffffffu, p.sum, o);
    p.nfin += __shfl_xor_sync(0xffffffffu, p.nfin, o);
    p.nbad += __shfl_xor_sync(0xffffffffu, p.nbad, o);
  }
  return p;
}

constexpr int kThreads = 256;

// grid = (nblk, cols). partial layout: [cols][nblk][5]
__global__ void __launch_bounds__(kThreads) stats_partial_kernel(const double* __restrict__ table, int64_t S,
                                                                int64_t ld, int nblk, double* __restrict__ part) {
  const int c = blockIdx.y;
  const double* col = table + (int64_t)c * ld;
  Part p{-HUGE_VAL, HUGE_VAL, 0.0, 0.0, 0.0};
  const int64_t per = ((S + nblk - 1) / nblk + 1) & ~(int64_t)1;   // even slice so double2 loads stay aligned
  const int64_t lo = (int64_t)blockIdx.x * per;
  int64_t hi = lo + per;
  if (hi > S) hi = S;
  const bool aligned = ((reinterpret_cast<uintptr_t>(col) & 15) == 0);
  if (aligned) {
    const int64_t npair = (hi > lo) ? (hi - lo) / 2 : 0;
    const double2* c2 = reinterpret_cast<const double2*>(col + lo);
    for (int64_t i = threadIdx.x; i < npair; i += kThreads) {
      const double2 v = __ldg(c2 + i);
      acc_one(v.x, p);
      acc_one(v.y, p);
    }
    if (threadIdx.x == 0 && hi > lo && ((hi - lo) & 1)) acc_one(col[hi - 1], p);
  } else {
    for (int64_t i = lo + threadIdx.x; i < hi; i += kThreads) acc_one(col[i], p);
  }
  p = warp_fold(p);
  __shared__ Part sm[kThreads / 32];
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = p;
  __syncthreads();
  if (threadIdx.x == 0) {
    Part t = sm[0];
    for (int w = 1; w < kThreads / 32; ++w) {
      t.mx = fmax(t.mx, sm[w].mx); t.mn = fmin(t.mn, sm[w].mn);
      t.sum += sm[w].sum; t.nfin += sm[w].nfin; t.nbad += sm[w].nbad;
    }
    double* o = part + ((int64_t)c * nblk + blockIdx.x) * 5;
    o[0] = t.mx; o[1] = t.mn; o[2] = t.sum; o[3] = t.nfin; o[4] = t.nbad;
  }
}

// one thread per column folds the partials in index order -> stats [cols][5]
__global__ void stats_final_kernel(const double* __restrict__ part, int cols, int nblk, double* __restrict__ stats) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  double mx = -HUGE_VAL, mn = HUGE_VAL, sum = 0.0, nf = 0.0, nb = 0.0;
  for (int b = 0; b < nblk; ++b) {
    const double* o = part + ((int64_t)c * nblk + b) * 5;
    mx = fmax(mx, o[0]); mn = fmin(mn, o[1]); sum += o[2]; nf += o[3]; nb += o[4];
  }
  double* s = stats + (int64_t)c * 5;
  s[0] = mx; s[1] = mn; s[2] = sum; s[3] = nf; s[4] = nb;
}

__global__ void __launch_bounds__(kThreads) sqdev_partial_kernel(const double* __restrict__ table, int64_t S,
                                                                int64_t ld, int nblk,
                                                                const double* __restrict__ mean,
                                                                double* __restrict__ part) {
  const int c = blockIdx.y;
  const double* col = table + (int64_t)c * ld;
  const double mu = mean[c];
  const int64_t per = (S + nblk - 1) / nblk;
  const int64_t lo = (int64_t)blockIdx.x * per;
  int64_t hi = lo + per;
  if (hi > S) hi = S;
  double acc = 0.0;
  for (int64_t i = lo + threadIdx.x; i < hi; i += kThreads) {
    const double v = col[i];
    if (fabs(v) <= 1.79e308) { const double d = v - mu; acc = fma(d, d, acc); }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  __shared__ double sm[kThreads / 32];
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = sm[0];
    for (int w = 1; w < kThreads / 32; ++w) t += sm[w];
    part[(int64_t)c * nblk + blockIdx.x] = t;
  }
}

__global__ void sqdev_final_kernel(const double* __restrict__ part, int cols, int nblk, double* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  double t = 0.0;
  for (int b = 0; b < nblk; ++b) t += part[(int64_t)c * nblk + b];
  out[c] = t;
}

// ---- one-pass moments: {max, min, n_finite, n_nonfinite, mean, M2 = sum (x - mean)^2} per column.
// Shifted-data accumulation: s1 = sum (x - k), s2 = sum (x - k)^2 with k = the column's first finite-looking entry
// (any value near the data keeps the cancellation in s2 - s1^2/n harmless); partials add exactly like plain sums, so
// the fold stays a fixed-order tree. Shards/ranks are merged afterwards with Chan's pairwise update
// (lq_mpc_b200/stats.py::merge_moments) — ONE collective instead of three, one pass over the table instead of two.
struct Mom {
  double mx, mn, nfin, nbad, s1, s2;
};

__device__ __forceinline__ void mom_acc(double v, double k, Mom& p) {
  if (fabs(v) <= 1.79e308) {
    p.mx = fmax(p.mx, v);
    p.mn = fmin(p.mn, v);
    p.nfin += 1.0;
    const double d = v - k;
    p.s1 += d;
    p.s2 = fma(d, d, p.s2);
  } else {
    p.nbad += 1.0;
  }
}

__device__ __forceinline__ Mom mom_merge(const Mom& a, const Mom& b) {
  return Mom{fmax(a.mx, b.mx), fmin(a.mn, b.mn), a.nfin + b.nfin, a.nbad + b.nbad, a.s1 + b.s1, a.s2 + b.s2};
}

__device__ __forceinline__ Mom mom_warp_fold(Mom p) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    Mom q;
    q.mx = __shfl_xor_sync(0xffffffffu, p.mx, o); q.mn = __shfl_xor_sync(0xffffffffu, p.mn, o);
    q.nfin = __shfl_xor_sync(0xffffffffu, p.nfin, o); q.nbad = __shfl_xor_sync(0xffffffffu, p.nbad, o);
    q.s1 = __shfl_xor_sync(0xffffffffu, p.s1, o); q.s2 = __shfl_xor_sync(0xffffffffu, p.s2, o);
    p = mom_merge(p, q);   // xor butterfly: every lane ends with the same, order-fixed result
  }
  return p;
}

__device__ __forceinline__ double column_shift(const double* col, int64_t S) {
  const double k = (S > 0) ? col[0] : 0.0;
  return (fabs(k) <= 1.79e308) ? k : 0.0;
}

// grid = (nblk, cols); partial layout [cols][nblk][6]
__global__ void __launch_bounds__(kThreads) moments_partial_kernel(const double* __restrict__ table, int64_t S,
                                                                  int64_t ld, int nblk, double* __restrict__ part) {
  const int c = blockIdx.y;
  const double* col = table + (int64_t)c * ld;
  const double k = column_shift(col, S);
  Mom p{-HUGE_VAL, HUGE_VAL, 0.0, 0.0, 0.0, 0.0};
  const int64_t per = ((S + nblk - 1) / nblk + 1) & ~(int64_t)1;
  const int64_t lo = (int64_t)blockIdx.x * per;
  int64_t hi = lo + per;
  if (hi > S) hi = S;
  if ((reinterpret_cast<uintptr_t>(col) & 15) == 0) {
    const int64_t npair = (hi > lo) ? (hi - lo) / 2 : 0;
    const double2* c2 = reinterpret_cast<const double2*>(col + lo);
    for (int64_t i = threadIdx.x; i < npair; i += kThreads) {
      const double2 v = __ldg(c2 + i);
      mom_acc(v.x, k, p);
      mom_acc(v.y, k, p);
    }
    if (threadIdx.x == 0 && hi > lo && ((hi - lo) & 1)) mom_acc(col[hi - 1], k, p);
  } else {
    for (int64_t i = lo + threadIdx.x; i < hi; i += kThreads) mom_acc(col[i], k, p);
  }
  p = mom_warp_fold(p);
  __shared__ Mom sm[kThreads / 32];
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = p;
  __syncthreads();
  if (threadIdx.x == 0) {
    Mom t = sm[0];
    for (int w = 1; w < kThreads / 32; ++w) t = mom_merge(t, sm[w]);
    double* o = part + ((int64_t)c * nblk + blockIdx.x) * 6;
    o[0] = t.mx; o[1] = t.mn; o[2] = t.nfin; o[3] = t.nbad; o[4] = t.s1; o[5] = t.s2;
  }
}

// one warp per column: lane l folds partials l, l+32, ... in order, then the butterfly -> out [cols][6]
__global__ void __launch_bounds__(32) moments_final_kernel(const double* __restrict__ part,
                                                          const double* __restrict__ table, int64_t S, int64_t ld,
                                                          int nblk, double* __restrict__ out) {
  const int c = blockIdx.x;
  Mom p{-HUGE_VAL, HUGE_VAL, 0.0, 0.0, 0.0, 0.0};
  for (int b = threadIdx.x; b < nblk; b += 32) {
    const double* o = part + ((int64_t)c * nblk + b) * 6;
    p = mom_merge(p, Mom{o[0], o[1], o[2], o[3], o[4], o[5]});
  }
  p = mom_warp_fold(p);
  if (threadIdx.x == 0) {
    const double k = column_shift(table + (int64_t)c * ld, S);
    double* o = out + (int64_t)c * 6;
    const double n = p.nfin;
    const double m1 = (n > 0.0) ? p.s1 / n : 0.0;
    o[0] = p.mx; o[1] = p.mn; o[2] = n; o[3] = p.nbad;
    o[4] = (n > 0.0) ? k + m1 : nan("");
    o[5] = (n > 0.0) ? fmax(p.s2 - p.s1 * m1, 0.0) : nan("");
  }
}

int pick_nblk(lqmpc_ctx* ctx, int cols, int64_t S) {
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
  int64_t want = (S + 8191) / 8192;                 // >= 8192 elements (64 KiB) per block
  int64_t cap = ((int64_t)sms * 8 + cols - 1) / cols;  // ~8 resident blocks per SM over all columns
  if (want > cap) want = cap;
  if (want < 1) want = 1;
  return (int)want;
}

}  // namespace

int lq_launch_stats(lqmpc_ctx* ctx, const double* table, int cols, int64_t S, int64_t ld, double* stats) {
  const int nblk = pick_nblk(ctx, cols, S);
  int rc = lq_reserve_ws(ctx, (size_t)cols * nblk * 5 * sizeof(double));
  if (rc) return rc;
  double* part = reinterpret_cast<double*>(ctx->ws);
  stats_partial_kernel<<<dim3(nblk, cols), kThreads, 0, ctx->stream>>>(table, S, ld, nblk, part);
  stats_final_kernel<<<(cols + 127) / 128, 128, 0, ctx->stream>>>(part, cols, nblk, stats);
  ctx->launches += 2;
  return lq_check_cuda(ctx, cudaGetLastError(), "column stats launch");
}

int lq_launch_moments(lqmpc_ctx* ctx, const double* table, int cols, int64_t S, int64_t ld, double* out) {
  const int nblk = pick_nblk(ctx, cols, S);
  int rc = lq_reserve_ws(ctx, (size_t)cols * nblk * 6 * sizeof(double));
  if (rc) return rc;
  double* part = reinterpret_cast<double*>(ctx->ws);
  moments_partial_kernel<<<dim3(nblk, cols), kThreads, 0, ctx->stream>>>(table, S, ld, nblk, part);
  moments_final_kernel<<<cols, 32, 0, ctx->stream>>>(part, table, S, ld, nblk, out);
  ctx->launches += 2;
  return lq_check_cuda(ctx, cudaGetLastError(), "column moments launch");
}

int lq_launch_sqdev(lqmpc_ctx* ctx, const double* table, int cols, int64_t S, int64_t ld, const double* mean,
                    double* out) {
  const int nblk = pick_nblk(ctx, cols, S);
  int rc = lq_reserve_ws(ctx, (size_t)cols * nblk * sizeof(double));
  if (rc) return rc;
  double* part = reinterpret_cast<double*>(ctx->ws);
  sqdev_partial_kernel<<<dim3(nblk, cols), kThreads, 0, ctx->stream>>>(table, S, ld, nblk, mean, part);
  sqdev_final_kernel<<<(cols + 127) / 128, 128, 0, ctx->stream>>>(part, cols, nblk, out);
  ctx->launches += 2;
  return lq_check_cuda(ctx, cudaGetLastError(), "column sqdev launch");
}

// ---- exact order statistics by radix descent (lqmpc_column_radix_histogram / _select).
// A finite double maps to an order-preserving uint64 key (negatives: all bits flipped; non-negatives: sign bit set),
// so the key of the rank-r finite entry is found one 8-bit digit at a time, most significant first. Pass p counts, for
// every (column, selector), the finite entries whose key agrees with the selector's prefix on the bits above digit p,
// by their digit p. Counts are integers: the histogram is the same whatever the order of the atomics or the CTA count.
namespace {

constexpr int kRadixMaxSel = LQMPC_RADIX_MAX_SEL;   // 32 selectors x 256 bins x 4 B = 32 KB of shared memory

__device__ __forceinline__ unsigned long long radix_key(double v) {
  const unsigned long long b = static_cast<unsigned long long>(__double_as_longlong(v));
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

// grid = (nblk, cols), dynamic shared memory nuniq * 256 * 4 B. Selectors whose prefixes agree on the masked bits
// have the same histogram: it is counted once (slot) and written to each of them.
__global__ void __launch_bounds__(kThreads) radix_hist_kernel(const double* __restrict__ table, int64_t S,
                                                              int64_t ld, int nblk, int nsel, int pass,
                                                              const unsigned long long* __restrict__ prefix,
                                                              unsigned long long* __restrict__ hist) {
  extern __shared__ unsigned int sh[];
  __shared__ unsigned long long pre[kRadixMaxSel];
  __shared__ int slot[kRadixMaxSel];
  __shared__ int nuniq;
  const int c = blockIdx.y;
  const double* col = table + (int64_t)c * ld;
  const unsigned long long mask = pass ? (~0ull << (64 - 8 * pass)) : 0ull;
  const int shift = 56 - 8 * pass;
  if (threadIdx.x == 0) {
    int u = 0;
    for (int k = 0; k < nsel; ++k) {
      const unsigned long long pk = prefix[(int64_t)c * nsel + k] & mask;
      int s = -1;
      for (int j = 0; j < u; ++j)
        if (pre[j] == pk) { s = j; break; }
      if (s < 0) { pre[u] = pk; s = u++; }
      slot[k] = s;
    }
    nuniq = u;
  }
  __syncthreads();
  const int nu = nuniq;
  for (int i = threadIdx.x; i < nu * 256; i += kThreads) sh[i] = 0u;
  __syncthreads();
  auto count = [&](double v) {
    if (!(fabs(v) <= 1.79e308)) return;
    const unsigned long long key = radix_key(v);
    const unsigned int d = (unsigned int)(key >> shift) & 255u;
    for (int u = 0; u < nu; ++u)
      if (((key ^ pre[u]) & mask) == 0ull) atomicAdd(&sh[u * 256 + d], 1u);
  };
  const int64_t per = ((S + nblk - 1) / nblk + 1) & ~(int64_t)1;
  const int64_t lo = (int64_t)blockIdx.x * per;
  int64_t hi = lo + per;
  if (hi > S) hi = S;
  if ((reinterpret_cast<uintptr_t>(col) & 15) == 0) {
    const int64_t npair = (hi > lo) ? (hi - lo) / 2 : 0;
    const double2* c2 = reinterpret_cast<const double2*>(col + lo);
    for (int64_t i = threadIdx.x; i < npair; i += kThreads) {
      const double2 v = __ldg(c2 + i);
      count(v.x);
      count(v.y);
    }
    if (threadIdx.x == 0 && hi > lo && ((hi - lo) & 1)) count(col[hi - 1]);
  } else {
    for (int64_t i = lo + threadIdx.x; i < hi; i += kThreads) count(col[i]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < nsel * 256; i += kThreads) {
    const unsigned int v = sh[slot[i >> 8] * 256 + (i & 255)];
    if (v) atomicAdd(hist + ((int64_t)c * nsel) * 256 + i, (unsigned long long)v);
  }
}

// one thread per (column, selector): the digit whose bucket holds the remaining rank; the counts below it leave the
// rank, the digit joins the prefix. A rank outside the column (no finite entry) leaves both unchanged.
__global__ void radix_select_kernel(const long long* __restrict__ hist, int cols, int nsel, int pass,
                                    long long* __restrict__ rank, unsigned long long* __restrict__ prefix) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)cols * nsel) return;
  const long long* h = hist + t * 256;
  const long long r = rank[t];
  long long below = 0;
  for (int d = 0; d < 256; ++d) {
    const long long cnt = h[d];
    if (r >= below && r < below + cnt) {
      rank[t] = r - below;
      prefix[t] |= (unsigned long long)d << (56 - 8 * pass);
      return;
    }
    below += cnt;
  }
}

// ---- arg-extremes: {max, min} of the finite entries with the lowest index attaining each.
struct Arg {
  double mx, mn;
  long long imx, imn;   // -1: no finite entry yet
};

__device__ __forceinline__ Arg arg_merge(const Arg& a, const Arg& b) {
  Arg r = a;
  if (b.mx > a.mx || (b.mx == a.mx && b.imx >= 0 && (a.imx < 0 || b.imx < a.imx))) { r.mx = b.mx; r.imx = b.imx; }
  if (b.mn < a.mn || (b.mn == a.mn && b.imn >= 0 && (a.imn < 0 || b.imn < a.imn))) { r.mn = b.mn; r.imn = b.imn; }
  return r;
}

__device__ __forceinline__ void arg_acc(double v, long long i, Arg& p) {
  if (fabs(v) <= 1.79e308) {   // entries arrive in increasing index order per thread: strict compares keep the first
    if (v > p.mx) { p.mx = v; p.imx = i; }
    if (v < p.mn) { p.mn = v; p.imn = i; }
  }
}

__device__ __forceinline__ Arg arg_warp_fold(Arg p) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    Arg q;
    q.mx = __shfl_xor_sync(0xffffffffu, p.mx, o); q.mn = __shfl_xor_sync(0xffffffffu, p.mn, o);
    q.imx = __shfl_xor_sync(0xffffffffu, p.imx, o); q.imn = __shfl_xor_sync(0xffffffffu, p.imn, o);
    p = arg_merge(p, q);
  }
  return p;
}

// grid = (nblk, cols); partial layout [cols][nblk] Arg
__global__ void __launch_bounds__(kThreads) argext_partial_kernel(const double* __restrict__ table, int64_t S,
                                                                 int64_t ld, int nblk, Arg* __restrict__ part) {
  const int c = blockIdx.y;
  const double* col = table + (int64_t)c * ld;
  Arg p{-HUGE_VAL, HUGE_VAL, -1, -1};
  const int64_t per = ((S + nblk - 1) / nblk + 1) & ~(int64_t)1;
  const int64_t lo = (int64_t)blockIdx.x * per;
  int64_t hi = lo + per;
  if (hi > S) hi = S;
  if ((reinterpret_cast<uintptr_t>(col) & 15) == 0) {
    const int64_t npair = (hi > lo) ? (hi - lo) / 2 : 0;
    const double2* c2 = reinterpret_cast<const double2*>(col + lo);
    for (int64_t i = threadIdx.x; i < npair; i += kThreads) {
      const double2 v = __ldg(c2 + i);
      arg_acc(v.x, lo + 2 * i, p);
      arg_acc(v.y, lo + 2 * i + 1, p);
    }
    if (threadIdx.x == 0 && hi > lo && ((hi - lo) & 1)) arg_acc(col[hi - 1], hi - 1, p);
  } else {
    for (int64_t i = lo + threadIdx.x; i < hi; i += kThreads) arg_acc(col[i], i, p);
  }
  p = arg_warp_fold(p);
  __shared__ Arg sm[kThreads / 32];
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = p;
  __syncthreads();
  if (threadIdx.x == 0) {
    Arg t = sm[0];
    for (int w = 1; w < kThreads / 32; ++w) t = arg_merge(t, sm[w]);
    part[(int64_t)c * nblk + blockIdx.x] = t;
  }
}

// one warp per column -> val [cols][2] = {max, min}, idx [cols][2] (+ index_base; -1 for an empty column)
__global__ void __launch_bounds__(32) argext_final_kernel(const Arg* __restrict__ part, int nblk, int64_t index_base,
                                                         double* __restrict__ val, long long* __restrict__ idx) {
  const int c = blockIdx.x;
  Arg p{-HUGE_VAL, HUGE_VAL, -1, -1};
  for (int b = threadIdx.x; b < nblk; b += 32) p = arg_merge(p, part[(int64_t)c * nblk + b]);
  p = arg_warp_fold(p);
  if (threadIdx.x == 0) {
    val[2 * c] = p.mx;
    val[2 * c + 1] = p.mn;
    idx[2 * c] = p.imx >= 0 ? p.imx + index_base : -1;
    idx[2 * c + 1] = p.imn >= 0 ? p.imn + index_base : -1;
  }
}

}  // namespace

int lq_launch_radix_hist(lqmpc_ctx* ctx, const double* table, int cols, int64_t S, int64_t ld, int nsel, int pass,
                         const uint64_t* prefix, int64_t* hist) {
  int rc = lq_check_cuda(ctx, cudaMemsetAsync(hist, 0, (size_t)cols * nsel * 256 * sizeof(int64_t), ctx->stream),
                         "radix histogram clear");
  if (rc || S == 0) return rc;
  int nblk = pick_nblk(ctx, cols, S);
  if ((S + nblk - 1) / nblk > ((int64_t)1 << 30)) nblk = (int)((S + ((int64_t)1 << 30) - 1) >> 30);  // uint32 bins
  radix_hist_kernel<<<dim3(nblk, cols), kThreads, (size_t)nsel * 256 * sizeof(unsigned int), ctx->stream>>>(
      table, S, ld, nblk, nsel, pass, reinterpret_cast<const unsigned long long*>(prefix),
      reinterpret_cast<unsigned long long*>(hist));
  ctx->launches += 1;
  return lq_check_cuda(ctx, cudaGetLastError(), "column radix histogram launch");
}

int lq_launch_radix_select(lqmpc_ctx* ctx, const int64_t* hist, int cols, int nsel, int pass, int64_t* rank,
                           uint64_t* prefix) {
  const int64_t n = (int64_t)cols * nsel;
  radix_select_kernel<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(
      reinterpret_cast<const long long*>(hist), cols, nsel, pass, reinterpret_cast<long long*>(rank),
      reinterpret_cast<unsigned long long*>(prefix));
  ctx->launches += 1;
  return lq_check_cuda(ctx, cudaGetLastError(), "column radix select launch");
}

int lq_launch_argext(lqmpc_ctx* ctx, const double* table, int cols, int64_t S, int64_t ld, int64_t index_base,
                     double* val, int64_t* idx) {
  const int nblk = pick_nblk(ctx, cols, S);
  int rc = lq_reserve_ws(ctx, (size_t)cols * nblk * sizeof(Arg));
  if (rc) return rc;
  Arg* part = reinterpret_cast<Arg*>(ctx->ws);
  argext_partial_kernel<<<dim3(nblk, cols), kThreads, 0, ctx->stream>>>(table, S, ld, nblk, part);
  argext_final_kernel<<<cols, 32, 0, ctx->stream>>>(part, nblk, index_base, val, reinterpret_cast<long long*>(idx));
  ctx->launches += 2;
  return lq_check_cuda(ctx, cudaGetLastError(), "column argext launch");
}
