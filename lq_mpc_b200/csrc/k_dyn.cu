// k_dyn.cu — kernels and launchers of the RUN-TIME DIMENSION route (dyn.cuh): one warp per sample, any n <= 32, m <= 8.
// Selected by lqmpc_set_problem for every (n, m) that has no register-resident instantiation (engine.h:
// LQ_FOR_EACH_DIM); the entry points of include/lqmpc_b200.h behave identically on both routes (same operand layouts,
// same outputs and flag bits). Not available on this route: general input polytopes and lqmpc_eval_seeded.
#include "dyn.cuh"
#include "engine.h"

namespace {

using lqd::Arena;
using lqd::DynPb;
using lqd::QpWs;
using namespace lqd;

constexpr int kMaxWarpsPerCta = 4;   // the launcher picks 4, 2 or 1 warps per CTA by the size of the per-warp arena

// device problem buffer (doubles): A | B | Q | R | Pt | Pexp | Qinv | ulo | uhi | maxQ minQ maxR minR has_bounds qr_scalar
struct DynLayout {
  int n, m;
  size_t oA, oB, oQ, oR, oPt, oPexp, oQinv, olo, ohi, osc, total;
  DynLayout(int n_, int m_) : n(n_), m(m_) {
    size_t o = 0;
    oA = o; o += (size_t)n * n;
    oB = o; o += (size_t)n * m;
    oQ = o; o += (size_t)n * n;
    oR = o; o += (size_t)m * m;
    oPt = o; o += (size_t)n * n;
    oPexp = o; o += (size_t)n * n;
    oQinv = o; o += (size_t)n * n;
    olo = o; o += m;
    ohi = o; o += m;
    osc = o; o += 8;
    total = o;
  }
};

DynPb make_pb(const lqmpc_ctx* ctx) {
  const DynLayout L(ctx->n, ctx->m);
  const double* d = reinterpret_cast<const double*>(ctx->dyn_dev);
  const double* h = ctx->dyn_host.data();
  DynPb pb;
  pb.n = ctx->n; pb.m = ctx->m;
  pb.A = d + L.oA; pb.B = d + L.oB; pb.Q = d + L.oQ; pb.R = d + L.oR; pb.Pt = d + L.oPt; pb.Pexp = d + L.oPexp;
  pb.Qinv = d + L.oQinv; pb.ulo = d + L.olo; pb.uhi = d + L.ohi;
  pb.maxQ = h[L.osc + 0]; pb.minQ = h[L.osc + 1]; pb.maxR = h[L.osc + 2]; pb.minR = h[L.osc + 3];
  pb.has_bounds = (int)h[L.osc + 4]; pb.qr_scalar = (int)h[L.osc + 5];
  return pb;
}

__device__ __forceinline__ double* warp_arena(int nbig, int n, int m) {
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  return reinterpret_cast<double*>(dyn_smem) + (size_t)(threadIdx.x >> 5) * Arena::doubles(n, m, nbig);
}

// Ah = A + dA_s, Bh = B + dB_s (SoA operands: element e of sample s at ptr[e * ld + s]; NULL = zero perturbation)
__device__ __forceinline__ void load_model(int lane, Arena& ar, const DynPb& pb, const double* dA, const double* dB,
                                           int64_t ldS, int64_t s) {
  const int n = ar.n, m = ar.m;
  for (int e = lane; e < n * n; e += 32) {
    const int i = e / n, j = e - i * n;
    ar.big[0][i * ar.ld + j] = pb.A[e] + (dA ? dA[(int64_t)e * ldS + s] : 0.0);
  }
  for (int e = lane; e < n * m; e += 32) ar.Bh[e] = pb.B[e] + (dB ? dB[(int64_t)e * ldS + s] : 0.0);
  __syncwarp();
}

// ---------------------------------------------------------------------------------------------------- prepare
__global__ void __launch_bounds__(32) dyn_prepare_kernel(double* buf, int n, int m, int N_opc, size_t oA, size_t oB,
                                                         size_t oQ, size_t oR, size_t oPt, size_t oPexp, size_t oQinv,
                                                         size_t osc) {
  const int lane = threadIdx.x & 31;
  Arena ar;
  ar.carve(warp_arena(5, n, m), n, m, 5);
  const int ld = ar.ld;
  const double* Q = buf + oQ; const double* R = buf + oR;
  // Qinv
  wcopy(lane, n, n, Q, n, ar.big[2], ld);
  for (int e = lane; e < n * n; e += 32) { const int i = e / n, j = e - i * n; ar.big[3][i * ld + j] = (i == j) ? 1.0 : 0.0; }
  __syncwarp();
  lqd::wlu_solve(lane, n, ar.big[2], ld, ar.big[3], ld, n);
  for (int e = lane; e < n * n; e += 32) { const int i = e / n, j = e - i * n; buf[oQinv + e] = ar.big[3][i * ld + j]; }
  // eigenvalue extremes of Q and R, scalar-weights flag
  wcopy(lane, n, n, Q, n, ar.big[2], ld);
  const double maxQ = lqd::wsym_extreme(lane, n, ar.big[2], ld, true, ar.big[3], ld, ar.v);
  const double minQ = lqd::wsym_extreme(lane, n, ar.big[2], ld, false, ar.big[3], ld, ar.v);
  wcopy(lane, m, m, R, m, ar.G, m);
  const double maxR = lqd::wsym_extreme(lane, m, ar.G, m, true, ar.G2, m, ar.v);
  const double minR = lqd::wsym_extreme(lane, m, ar.G, m, false, ar.G2, m, ar.v);
  bool scal = true;
  for (int e = 0; e < n * n; ++e) scal = scal && (Q[e] == (((e / n) == (e % n)) ? Q[0] : 0.0));
  for (int e = 0; e < m * m; ++e) scal = scal && (R[e] == (((e / m) == (e % m)) ? R[0] : 0.0));
  if (lane == 0) {
    buf[osc + 0] = maxQ; buf[osc + 1] = minQ; buf[osc + 2] = maxR; buf[osc + 3] = minR;
    buf[osc + 5] = scal ? 1.0 : 0.0;
  }
  // expert cost matrix: N_opc Riccati steps on the TRUE model from Pt (or to the fixed point when N_opc <= 0)
  wcopy(lane, n, n, buf + oA, n, ar.big[0], ld);
  wcopy(lane, n, m, buf + oB, m, ar.Bh, m);
  wcopy(lane, n, n, buf + oPt, n, ar.big[1], ld);
  const int iters = (N_opc > 0) ? N_opc : 100000;
  for (int k = 0; k < iters; ++k) {
    if (N_opc <= 0) wcopy(lane, n, n, ar.big[1], ld, ar.big[4], ld);
    lqd::dyn_riccati_stage(lane, ar, Q, R, false, true);
    if (N_opc <= 0) {
      double d = 0.0, mx = 0.0;
      for (int e = lane; e < n * n; e += 32) {
        const int i = e / n, j = e - i * n;
        d = lq::dmax(d, fabs(ar.big[1][i * ld + j] - ar.big[4][i * ld + j]));
        mx = lq::dmax(mx, fabs(ar.big[1][i * ld + j]));
      }
      d = lqd::wmaxd(d); mx = lqd::wmaxd(mx);
      if (d <= 1e-16 * mx) break;
    }
  }
  for (int e = lane; e < n * n; e += 32) { const int i = e / n, j = e - i * n; buf[oPexp + e] = ar.big[1][i * ld + j]; }
}

// ---------------------------------------------------------------------------------------------------- K1
__global__ void __launch_bounds__(kMaxWarpsPerCta * 32) dyn_eval_kernel(const DynPb pb, const EvalArgs a) {
  const int lane = threadIdx.x & 31, n = pb.n, m = pb.m;
  Arena ar;
  ar.carve(warp_arena(7, n, m), n, m, 7);
  const int wpc = blockDim.x >> 5;
  const int64_t nw = (int64_t)gridDim.x * wpc;
  for (int64_t s = (int64_t)blockIdx.x * wpc + (threadIdx.x >> 5); s < a.S; s += nw) {
    load_model(lane, ar, pb, a.dA, a.dB, a.ld, s);
    for (int i = lane; i < n; i += 32) ar.x[i] = a.x0[(int64_t)i * a.ld + s];
    lqd::wcopy(lane, n, n, pb.Pt, n, ar.big[1], ar.ld);
    const double v_exp = lqd::wquad(lane, n, ar.x, pb.Pexp, n, ar.x);
    int sticky = 0;
    const bool want_vn = a.Vn != nullptr;
    for (int k = 1; k <= a.N_max; ++k) {
      const bool emit = (k >= a.N_min);
      if (!lqd::dyn_riccati_stage(lane, ar, pb.Q, pb.R, emit, k < a.N_max || want_vn)) sticky |= lq::FLAG_CHOL_FAIL;
      if (!emit) continue;
      int flags = sticky;
      double J, rho, JT = 0.0;
      lqd::dyn_closed_loop(lane, ar, pb, a.T, &J, &rho, &JT, &flags);
      const double vn = want_vn ? lqd::wquad(lane, n, ar.x, ar.big[1], ar.ld, ar.x) : 0.0;
      const int64_t o = (int64_t)(k - a.N_min) * a.ld + s;
      if (lane == 0) {
        if (a.J) a.J[o] = J;
        if (a.rho) a.rho[o] = rho;
        if (a.ratio) a.ratio[o] = J / v_exp;
        if (a.Vn) a.Vn[o] = vn;
        if (a.JT) a.JT[o] = JT;
        if (a.flags) a.flags[o] = flags;
      }
      if (a.K0)
        for (int e = lane; e < m * n; e += 32) a.K0[((int64_t)(k - a.N_min) * (m * n) + e) * a.ld + s] = ar.Kt[e];
      __syncwarp();
    }
  }
}

// ---------------------------------------------------------------------------------------------------- K2
__global__ void __launch_bounds__(kMaxWarpsPerCta * 32) dyn_mpc_kernel(const DynPb pb, const MpcArgs a, const int simulate) {
  const int lane = threadIdx.x & 31, n = pb.n, m = pb.m;
  Arena ar;
  ar.carve(warp_arena(6, n, m), n, m, 6);
  const int wpc = blockDim.x >> 5;
  const int64_t wid = (int64_t)blockIdx.x * wpc + (threadIdx.x >> 5), nw = (int64_t)gridDim.x * wpc;
  QpWs ws;
  ws.carve(a.ws + (size_t)wid * QpWs::doubles(n, m, a.N), n, m, a.N);
  lq::Refs rf;
  rf.xr = a.xr; rf.ur = a.ur; rf.ld = a.ref_ld;
  double* x0 = ar.v + 32;                                  // current / initial state (n <= 32 doubles)
  for (int64_t s = wid; s < a.S; s += nw) {
    load_model(lane, ar, pb, a.dA, a.dB, a.S, s);
    const int pf = lqd::dyn_plan_prepare(lane, ar, pb, a.N, ws);
    if (!simulate) {
      const int P = a.pts ? a.npts : 1;
      double mv = -HUGE_VAL;
      for (int p = 0; p < P; ++p) {
        for (int i = lane; i < n; i += 32) x0[i] = a.pts ? a.pts[p * n + i] : a.x0[(int64_t)i * a.S + s];
        __syncwarp();
        double V;
        double* u0 = ar.v + 8;                             // m <= 8 doubles no routine of the solve touches
        const int f = pf | lqd::dyn_clqr_solve(lane, ar, pb, a.N, x0, ws, u0, &V, rf);
        double u0r[8];
        for (int j = 0; j < m; ++j) u0r[j] = u0[j];
        mv = lq::dmax(mv, V);
        if (lane == 0) {
          if (a.V) a.V[(int64_t)p * a.S + s] = V;
          if (a.u0) for (int j = 0; j < m; ++j) a.u0[((int64_t)p * m + j) * a.S + s] = u0r[j];
          if (a.flags) a.flags[(int64_t)p * a.S + s] = f;
        }
        __syncwarp();
      }
      if (a.M_V && lane == 0) a.M_V[s] = mv;
    } else {
      // closed loop on the TRUE plant (utils_class.py:245-285), the exact QP re-solved from the measured state
      double* u0 = ar.v + 8;
      for (int i = lane; i < n; i += 32) x0[i] = a.pts ? a.pts[i] : a.x0[(int64_t)i * a.S + s];
      __syncwarp();
      if (a.X) for (int i = lane; i < n; i += 32) a.X[(int64_t)i * a.S + s] = x0[i];
      double cost = lqd::wquad(lane, n, x0, pb.Q, n, x0);
      int flags = pf, act = 0;
      for (int t = 0; t < a.T; ++t) {
        double V;
        const int f = lqd::dyn_clqr_solve(lane, ar, pb, a.N, x0, ws, u0, &V, rf);
        flags |= f;
        act += (f & lq::FLAG_QP_ACTIVE) ? 1 : 0;
        if (lane < m) ar.u[lane] = u0[lane];
        __syncwarp();
        lqd::dyn_step_model(lane, n, m, pb.A, n, pb.B, x0, ar.u, ar.xn);
        cost += lqd::wquad(lane, n, ar.xn, pb.Q, n, ar.xn);
        cost += lqd::wquad(lane, m, ar.u, pb.R, m, ar.u);
        if (a.U && lane < m) a.U[((int64_t)t * m + lane) * a.S + s] = ar.u[lane];
        if (a.X) for (int i = lane; i < n; i += 32) a.X[((int64_t)(t + 1) * n + i) * a.S + s] = ar.xn[i];
        for (int i = lane; i < n; i += 32) x0[i] = ar.xn[i];
        __syncwarp();
      }
      if (lane == 0) {
        if (a.J_T) a.J_T[s] = cost;
        if (a.flags) a.flags[s] = flags;
        if (a.n_active) a.n_active[s] = act;
      }
    }
    __syncwarp();
  }
}

// Infinite-horizon closed loop (clqr.cuh: certified_closed_loop): J_inf [S], T_cert [S], flags [S]; a.T = T_max.
// Arena of 7: dyn_clqr_solve works in big[0..5], the tail matrix S stays in big[6].
__global__ void __launch_bounds__(kMaxWarpsPerCta * 32) dyn_simulate_inf_kernel(const DynPb pb, const MpcArgs a) {
  const int lane = threadIdx.x & 31, n = pb.n, m = pb.m;
  Arena ar;
  ar.carve(warp_arena(7, n, m), n, m, 7);
  const int wpc = blockDim.x >> 5;
  const int64_t wid = (int64_t)blockIdx.x * wpc + (threadIdx.x >> 5), nw = (int64_t)gridDim.x * wpc;
  QpWs ws;
  ws.carve(a.ws + (size_t)wid * QpWs::doubles(n, m, a.N), n, m, a.N);
  double* x = ar.v + 32;                                   // closed-loop state (n <= 32 doubles)
  double* u0 = ar.v + 8;                                   // m <= 8 doubles no routine of the solve touches
  for (int64_t s = wid; s < a.S; s += nw) {
    load_model(lane, ar, pb, a.dA, a.dB, a.S, s);
    int flags = lqd::dyn_plan_prepare(lane, ar, pb, a.N, ws);          // K0 in ar.Kt, P0 in big[4]
    const double cstar = lqd::dyn_box_certificate(lane, ar, pb, a.N, ws);
    lqd::wcopy(lane, n, n, ar.big[4], ar.ld, ar.big[1], ar.ld);         // P0 (dyn_closed_loop overwrites big[4])
    for (int i = lane; i < n; i += 32) ar.x[i] = a.pts ? a.pts[i] : a.x0[(int64_t)i * a.S + s];
    __syncwarp();
    double J0, rho, JT;
    lqd::dyn_closed_loop(lane, ar, pb, 0, &J0, &rho, &JT, &flags);     // S in big[5]
    double J = NAN;
    int tc = -1;
    if (flags & lq::FLAG_UNSTABLE) {
      J = HUGE_VAL;
    } else {
      const double cS = (flags & lq::FLAG_LYAP_NOCONV) ? NAN : lqd::dyn_tail_level(lane, ar, cstar);
      for (int i = lane; i < n; i += 32) x[i] = ar.x[i];
      __syncwarp();
      double cost = 0.0;
      for (int t = 0; cS >= 0.0; ++t) {
        const double v = lqd::wquad(lane, n, x, ar.big[6], ar.ld, x);
        if (v <= cS) { J = cost + v; tc = t; break; }
        if (t >= a.T) break;
        double V;
        flags |= lqd::dyn_clqr_solve(lane, ar, pb, a.N, x, ws, u0, &V, lq::Refs());
        if (lane < m) ar.u[lane] = u0[lane];
        __syncwarp();
        cost += lqd::wquad(lane, n, x, pb.Q, n, x);
        cost += lqd::wquad(lane, m, ar.u, pb.R, m, ar.u);
        lqd::dyn_step_model(lane, n, m, pb.A, n, pb.B, x, ar.u, ar.xn);
        for (int i = lane; i < n; i += 32) x[i] = ar.xn[i];
        __syncwarp();
      }
      if (tc < 0) flags |= lq::FLAG_TAIL_UNCERTIFIED;
    }
    if (lane == 0) {
      if (a.J_inf) a.J_inf[s] = J;
      if (a.T_cert) a.T_cert[s] = tc;
      if (a.flags) a.flags[s] = flags;
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------------------- K3 / dlqr
__global__ void __launch_bounds__(kMaxWarpsPerCta * 32) dyn_bounds_kernel(const DynPb pb, const BoundsArgs a,
                                                                       const int dlqr_only, double* K_dlqr,
                                                                       double* P_dlqr, int32_t* f_dlqr, int64_t S) {
  const int lane = threadIdx.x & 31, n = pb.n, m = pb.m;
  Arena ar;
  ar.carve(warp_arena(8, n, m), n, m, 8);
  const int wpc = blockDim.x >> 5;
  const int64_t nw = (int64_t)gridDim.x * wpc;
  for (int64_t s = (int64_t)blockIdx.x * wpc + (threadIdx.x >> 5); s < S; s += nw) {
    load_model(lane, ar, pb, a.dA, a.dB, S, s);
    int flags = 0;
    const bool own_gain = dlqr_only || (!a.K_in && !a.K_shared);
    if (own_gain) {
      if (!lqd::dyn_dare(lane, ar, pb)) flags |= lq::FLAG_DARE_NOCONV;
      double* Pout = dlqr_only ? P_dlqr : a.P_out;
      if (Pout)
        for (int e = lane; e < n * n; e += 32) Pout[(int64_t)e * S + s] = ar.big[3][(e / n) * ar.ld + (e % n)];
      lqd::wcopy(lane, n, n, ar.big[3], ar.ld, ar.big[1], ar.ld);
      lqd::dyn_riccati_stage(lane, ar, pb.Q, pb.R, true, false);      // Kt = -(R + B'XB)^-1 B'XA = -K_dlqr
    } else {
      for (int e = lane; e < m * n; e += 32) ar.Kt[e] = a.K_in ? a.K_in[(int64_t)e * S + s] : a.K_shared[e];
      __syncwarp();
    }
    if (dlqr_only) {
      if (K_dlqr) for (int e = lane; e < m * n; e += 32) K_dlqr[(int64_t)e * S + s] = -ar.Kt[e];   // u = -K x convention
      if (f_dlqr && lane == 0) f_dlqr[s] = flags;
      __syncwarp();
      continue;
    }
    for (int i = lane; i < n; i += 32) ar.x[i] = a.x_shared ? a.x_shared[i] : a.x[(int64_t)i * S + s];
    __syncwarp();
    lq::BoundsNorms q;
    flags |= lqd::dyn_bounds_norms(lane, ar, pb, a.N, ar.x, a.bar_u, a.bar_d_u, q);
    lq::BoundsScalars sc;
    sc.N = a.N;
    sc.e_A = a.eA ? a.eA[s] : a.eA_s;
    sc.e_B = a.eB ? a.eB[s] : a.eB_s;
    sc.M_V = a.MV ? a.MV[s] : a.MV_s;
    sc.p[0] = a.p[0]; sc.p[1] = a.p[1]; sc.p[2] = a.p[2];
    sc.V_expert = a.V_expert; sc.bar_u = a.bar_u; sc.bar_d_u = a.bar_d_u; sc.strict_reference = a.strict;
    double out[lq::BF_COUNT];
    for (int i = 0; i < lq::BF_COUNT; ++i) out[i] = 0.0;
    flags |= lq::bounds_formulas(pb.maxQ, pb.minQ, pb.maxR, pb.minR, sc, q, out);
    for (int i = 0; i < lq::BF_COUNT; ++i)
      if (!(fabs(out[i]) <= 1.79e308)) flags |= lq::FLAG_NONFINITE;
    if (lane == 0) {
      if (a.alpha) a.alpha[s] = out[lq::BF_ALPHA];
      if (a.beta) a.beta[s] = out[lq::BF_BETA];
      if (a.xi) a.xi[s] = out[lq::BF_XI];
      if (a.eta) a.eta[s] = out[lq::BF_ETA];
      if (a.bound) a.bound[s] = out[lq::BF_BOUND];
      if (a.flags) a.flags[s] = flags;
    }
    if (a.detail && lane < lq::BF_COUNT) a.detail[(int64_t)lane * S + s] = out[lane];
    if (a.K_out) for (int e = lane; e < m * n; e += 32) a.K_out[(int64_t)e * S + s] = ar.Kt[e];
    __syncwarp();
  }
}

// CTA shape and grid of a warp-per-sample kernel whose per-warp arena takes `per_warp` bytes of shared memory: the most
// warps per CTA (4, 2, 1) that fit, then as many CTAs as the SMs hold.
int grid_for(lqmpc_ctx* ctx, const void* kern, size_t per_warp, int64_t S, int* blocks_out, int* warps_out) {
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
  int w = kMaxWarpsPerCta;
  while (w > 1 && (size_t)w * per_warp > (size_t)200 * 1024) w >>= 1;
  const size_t smem = (size_t)w * per_warp;
  if (smem > (size_t)220 * 1024)
    return lq_set_error(ctx, LQMPC_EINVAL, "run-time-dimension route: shared memory arena does not fit");
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  int per_sm = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, w * 32, smem);
  if (per_sm < 1) return lq_set_error(ctx, LQMPC_EINVAL, "run-time-dimension route: kernel does not fit an SM");
  int64_t blocks = (int64_t)sms * per_sm;
  const int64_t want = (S + w - 1) / w;
  if (blocks > want) blocks = want;
  if (blocks < 1) blocks = 1;
  *blocks_out = (int)blocks;
  *warps_out = w;
  return LQMPC_OK;
}

}  // namespace

bool lq_dyn_supported(int n, int m) { return n >= 1 && n <= 32 && m >= 1 && m <= 8; }

int lq_dyn_set_problem(lqmpc_ctx* ctx, const double* A, const double* B, const double* Q, const double* R,
                       const double* P, const double* lo, const double* hi) {
  const int n = ctx->n, m = ctx->m;
  const DynLayout L(n, m);
  ctx->dyn_host.assign(L.total, 0.0);
  double* h = ctx->dyn_host.data();
  memcpy(h + L.oA, A, sizeof(double) * n * n);
  memcpy(h + L.oB, B, sizeof(double) * n * m);
  memcpy(h + L.oQ, Q, sizeof(double) * n * n);
  memcpy(h + L.oR, R, sizeof(double) * m * m);
  memcpy(h + L.oPt, P, sizeof(double) * n * n);
  for (int j = 0; j < m; ++j) {
    h[L.olo + j] = lo ? lo[j] : -HUGE_VAL;
    h[L.ohi + j] = hi ? hi[j] : HUGE_VAL;
  }
  h[L.osc + 4] = (lo || hi) ? 1.0 : 0.0;
  if (ctx->dyn_dev) { cudaStreamSynchronize(ctx->stream); cudaFree(ctx->dyn_dev); ctx->dyn_dev = nullptr; }
  int rc = lq_check_cuda(ctx, cudaMalloc(&ctx->dyn_dev, L.total * sizeof(double)), "cudaMalloc dyn problem");
  if (rc) return rc;
  rc = lq_check_cuda(ctx, cudaMemcpyAsync(ctx->dyn_dev, h, L.total * sizeof(double), cudaMemcpyHostToDevice, ctx->stream),
                     "H2D dyn problem");
  if (rc) return rc;
  const size_t smem = Arena::doubles(n, m, 5) * sizeof(double);
  cudaFuncSetAttribute(dyn_prepare_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  dyn_prepare_kernel<<<1, 32, smem, ctx->stream>>>(reinterpret_cast<double*>(ctx->dyn_dev), n, m, ctx->N_opc, L.oA, L.oB,
                                                   L.oQ, L.oR, L.oPt, L.oPexp, L.oQinv, L.osc);
  ctx->launches++;
  rc = lq_check_cuda(ctx, cudaGetLastError(), "dyn_prepare_kernel launch");
  if (rc) return rc;
  rc = lq_check_cuda(ctx, cudaMemcpyAsync(h, ctx->dyn_dev, L.total * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream),
                     "D2H dyn problem");
  if (rc) return rc;
  rc = lq_check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "dyn prepare sync");
  if (rc) return rc;
  h[L.osc + 4] = (lo || hi) ? 1.0 : 0.0;
  return LQMPC_OK;
}

int lq_dyn_get_prepared(lqmpc_ctx* ctx, double* out) {
  const int n = ctx->n;
  const DynLayout L(n, ctx->m);
  const double* h = ctx->dyn_host.data();
  memcpy(out, h + L.oPexp, sizeof(double) * n * n);
  memcpy(out + n * n, h + L.oQinv, sizeof(double) * n * n);
  for (int i = 0; i < 4; ++i) out[2 * n * n + i] = h[L.osc + i];
  return LQMPC_OK;
}

int lq_dyn_eval(lqmpc_ctx* ctx, const EvalArgs& a, cudaStream_t stream) {
  const DynPb pb = make_pb(ctx);
  const size_t per = Arena::doubles(pb.n, pb.m, 7) * sizeof(double);
  int blocks, w;
  int rc = grid_for(ctx, (const void*)dyn_eval_kernel, per, a.S, &blocks, &w);
  if (rc) return rc;
  dyn_eval_kernel<<<blocks, w * 32, w * per, stream>>>(pb, a);
  ctx->launches++;
  return lq_check_cuda(ctx, cudaGetLastError(), "dyn_eval_kernel launch");
}

int lq_dyn_mpc(lqmpc_ctx* ctx, MpcArgs a, bool sim) {
  if (ctx->poly_p > 0)
    return lq_set_error(ctx, LQMPC_EINVAL, "general input polytopes need a compiled (n, m) pair; see lqmpc_supported_dims()");
  const DynPb pb = make_pb(ctx);
  const size_t per_arena = Arena::doubles(pb.n, pb.m, 6) * sizeof(double);
  int blocks, w;
  int rc = grid_for(ctx, (const void*)dyn_mpc_kernel, per_arena, a.S, &blocks, &w);
  if (rc) return rc;
  const size_t per = QpWs::doubles(pb.n, pb.m, a.N);
  rc = lq_reserve_ws(ctx, per * (size_t)blocks * w * sizeof(double));
  if (rc) return rc;
  a.ws = reinterpret_cast<double*>(ctx->ws);
  if (ctx->ref_ld >= a.N) { a.xr = ctx->ref_x; a.ur = ctx->ref_u; a.ref_ld = ctx->ref_ld; }
  else if (ctx->ref_ld > 0) return lq_set_error(ctx, LQMPC_EINVAL, "references hold fewer than N columns");
  dyn_mpc_kernel<<<blocks, w * 32, w * per_arena, ctx->stream>>>(pb, a, sim ? 1 : 0);
  ctx->launches++;
  return lq_check_cuda(ctx, cudaGetLastError(), "dyn_mpc_kernel launch");
}

int lq_dyn_simulate_inf(lqmpc_ctx* ctx, MpcArgs a) {
  if (ctx->poly_p > 0)
    return lq_set_error(ctx, LQMPC_EINVAL, "general input polytopes need a compiled (n, m) pair; see lqmpc_supported_dims()");
  const DynPb pb = make_pb(ctx);
  const size_t per_arena = Arena::doubles(pb.n, pb.m, 7) * sizeof(double);
  int blocks, w;
  int rc = grid_for(ctx, (const void*)dyn_simulate_inf_kernel, per_arena, a.S, &blocks, &w);
  if (rc) return rc;
  const size_t per = QpWs::doubles(pb.n, pb.m, a.N);
  rc = lq_reserve_ws(ctx, per * (size_t)blocks * w * sizeof(double));
  if (rc) return rc;
  a.ws = reinterpret_cast<double*>(ctx->ws);
  dyn_simulate_inf_kernel<<<blocks, w * 32, w * per_arena, ctx->stream>>>(pb, a);
  ctx->launches++;
  return lq_check_cuda(ctx, cudaGetLastError(), "dyn_simulate_inf_kernel launch");
}

int lq_dyn_bounds(lqmpc_ctx* ctx, const BoundsArgs& a) {
  const DynPb pb = make_pb(ctx);
  if (!lq::bounds_matrix_free(pb.qr_scalar, a.strict, 0))
    return lq_set_error(ctx, LQMPC_EINVAL, "literal kron ordering with non-scalar weights needs a compiled (n, m) pair "
                                           "(pass strict_reference = 0 for the time-major weights)");
  if (a.polyP > 0)
    return lq_set_error(ctx, LQMPC_EINVAL, "general input polytopes need a compiled (n, m) pair");
  const size_t per = Arena::doubles(pb.n, pb.m, 8) * sizeof(double);
  int blocks, w;
  int rc = grid_for(ctx, (const void*)dyn_bounds_kernel, per, a.S, &blocks, &w);
  if (rc) return rc;
  dyn_bounds_kernel<<<blocks, w * 32, w * per, ctx->stream>>>(pb, a, 0, nullptr, nullptr, nullptr, a.S);
  ctx->launches++;
  return lq_check_cuda(ctx, cudaGetLastError(), "dyn_bounds_kernel launch");
}

int lq_dyn_dlqr(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, double* K, double* P, int32_t* flags) {
  const DynPb pb = make_pb(ctx);
  BoundsArgs a{};
  a.S = S; a.dA = dA; a.dB = dB;
  const size_t per = Arena::doubles(pb.n, pb.m, 8) * sizeof(double);
  int blocks, w;
  int rc = grid_for(ctx, (const void*)dyn_bounds_kernel, per, S, &blocks, &w);
  if (rc) return rc;
  dyn_bounds_kernel<<<blocks, w * 32, w * per, ctx->stream>>>(pb, a, 1, K, P, flags, S);
  ctx->launches++;
  return lq_check_cuda(ctx, cudaGetLastError(), "dyn_bounds_kernel (dlqr) launch");
}
