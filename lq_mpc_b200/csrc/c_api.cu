// c_api.cu — the extern "C" boundary declared in include/lqmpc_b200.h.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>

#include "../../include/lqmpc_b200.h"
#include "engine.h"
#include "bounds.cuh"
#include "pclqr.cuh"

int lq_set_error(lqmpc_ctx* ctx, int code, const char* what) {
  if (ctx) ctx->err = what ? what : "";
  return code;
}

int lq_check_cuda(lqmpc_ctx* ctx, cudaError_t e, const char* what) {
  if (e == cudaSuccess) return LQMPC_OK;
  if (ctx) {
    ctx->err = std::string(what ? what : "cuda") + ": " + cudaGetErrorString(e);
  }
  return LQMPC_ECUDA;
}

int lq_reserve_ws(lqmpc_ctx* ctx, size_t bytes) {
  if (bytes <= ctx->ws_bytes) return LQMPC_OK;
  if (ctx->ws) {
    cudaStreamSynchronize(ctx->stream);
    cudaFree(ctx->ws);
    ctx->ws = nullptr;
    ctx->ws_bytes = 0;
  }
  size_t want = bytes + bytes / 4;
  int rc = lq_check_cuda(ctx, cudaMalloc(&ctx->ws, want), "cudaMalloc workspace");
  if (rc) return rc;
  ctx->ws_bytes = want;
  return LQMPC_OK;
}

namespace {

// Packs the host problem description into the byte image of lq::Problem<n,m> (field order of riccati.cuh).
template <int n, int m>
void pack_problem(lqmpc_ctx* ctx, const double* A, const double* B, const double* Q, const double* R,
                  const double* P, const double* lo, const double* hi) {
  lq::Problem<n, m> pb;
  memset(&pb, 0, sizeof(pb));
  memcpy(pb.A, A, sizeof(pb.A));
  memcpy(pb.B, B, sizeof(pb.B));
  memcpy(pb.Q, Q, sizeof(pb.Q));
  memcpy(pb.R, R, sizeof(pb.R));
  memcpy(pb.Pt, P, sizeof(pb.Pt));
  pb.has_bounds = (lo != nullptr || hi != nullptr) ? 1 : 0;
  for (int j = 0; j < m; ++j) {
    pb.ulo[j] = lo ? lo[j] : -HUGE_VAL;
    pb.uhi[j] = hi ? hi[j] : HUGE_VAL;
  }
  memcpy(ctx->pb, &pb, sizeof(pb));
}

int ensure_pipe(lqmpc_ctx* ctx, size_t bytes_per_slot) {
  for (int i = 0; i < 2; ++i) {
    if (!ctx->pipe_stream[i]) {
      int rc = lq_check_cuda(ctx, cudaStreamCreateWithFlags(&ctx->pipe_stream[i], cudaStreamNonBlocking),
                             "pipe stream");
      if (rc) return rc;
      rc = lq_check_cuda(ctx, cudaEventCreateWithFlags(&ctx->pipe_done[i], cudaEventDisableTiming), "pipe event");
      if (rc) return rc;
    }
  }
  if (bytes_per_slot > ctx->pipe_bytes) {
    for (int i = 0; i < 2; ++i) {
      if (ctx->pipe_buf[i]) cudaFree(ctx->pipe_buf[i]);
      ctx->pipe_buf[i] = nullptr;
    }
    ctx->pipe_bytes = 0;
    for (int i = 0; i < 2; ++i) {
      int rc = lq_check_cuda(ctx, cudaMalloc(&ctx->pipe_buf[i], bytes_per_slot), "cudaMalloc pipeline slot");
      if (rc) return rc;
    }
    ctx->pipe_bytes = bytes_per_slot;
  }
  return LQMPC_OK;
}

// Error path of the host pipelines: asynchronous copies already enqueued still read from / write to the caller's
// host buffers — drain every stream involved before handing control (and the buffers) back.
int pipe_abort(lqmpc_ctx* ctx, int rc) {
  const std::string keep = ctx->err;
  for (int i = 0; i < 2; ++i)
    if (ctx->pipe_stream[i]) cudaStreamSynchronize(ctx->pipe_stream[i]);
  cudaStreamSynchronize(ctx->stream);
  (void)cudaGetLastError();
  ctx->err = keep;
  return rc;
}

#define LQ_PIPE(call, what)                                   \
  do {                                                        \
    const int rc__ = lq_check_cuda(ctx, (call), (what));      \
    if (rc__) return pipe_abort(ctx, rc__);                   \
  } while (0)

}  // namespace

extern "C" {

int lqmpc_abi_version(void) { return 6; }

const char* lqmpc_supported_dims(void) { return LQ_DIMS_STRING; }

int lqmpc_create(lqmpc_ctx** out, int device, void* cuda_stream) {
  if (!out) return LQMPC_EINVAL;
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count <= 0 || device < 0 || device >= count) return LQMPC_ENODEVICE;
  if (cudaSetDevice(device) != cudaSuccess) return LQMPC_ENODEVICE;
  lqmpc_ctx* ctx = new (std::nothrow) lqmpc_ctx();
  if (!ctx) return LQMPC_EINVAL;
  ctx->device = device;
  // NULL is the legacy default stream (what torch.cuda.current_stream() is unless the caller changed it)
  ctx->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
  ctx->own_stream = false;
  *out = ctx;
  return LQMPC_OK;
}

void lqmpc_destroy(lqmpc_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (ctx->ws) cudaFree(ctx->ws);
  if (ctx->seed_buf) cudaFree(ctx->seed_buf);
  if (ctx->dyn_dev) cudaFree(ctx->dyn_dev);
  if (ctx->pb_dev) cudaFree(ctx->pb_dev);
  if (ctx->ref_x) cudaFree(ctx->ref_x);
  if (ctx->ref_u) cudaFree(ctx->ref_u);
  if (ctx->poly_dev) cudaFree(ctx->poly_dev);
  if (ctx->tiled_pb) cudaFree(ctx->tiled_pb);
  if (ctx->tiled_zero) cudaFree(ctx->tiled_zero);
  for (int i = 0; i < 6; ++i)
    if (ctx->tp_ev[i]) cudaEventDestroy(ctx->tp_ev[i]);
  for (int i = 0; i < 2; ++i) {
    if (ctx->pipe_buf[i]) cudaFree(ctx->pipe_buf[i]);
    if (ctx->pipe_done[i]) cudaEventDestroy(ctx->pipe_done[i]);
    if (ctx->pipe_stream[i]) cudaStreamDestroy(ctx->pipe_stream[i]);
  }
  if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char* lqmpc_last_error(const lqmpc_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int lqmpc_sync(lqmpc_ctx* ctx) {
  if (!ctx) return LQMPC_EINVAL;
  return lq_check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "stream sync");
}

int64_t lqmpc_launch_count(const lqmpc_ctx* ctx) { return ctx ? ctx->launches : 0; }

int lqmpc_set_problem(lqmpc_ctx* ctx, int n, int m, const double* A, const double* B, const double* Q,
                      const double* R, const double* P, const double* lo, const double* hi, int N_opc) {
  if (!ctx) return LQMPC_EINVAL;
  if (!A || !B || !Q || !R || !P) return lq_set_error(ctx, LQMPC_EINVAL, "null problem matrix");
  cudaSetDevice(ctx->device);
  bool found = false;
#define X(N_, M_)                                   \
  if (n == N_ && m == M_) {                         \
    pack_problem<N_, M_>(ctx, A, B, Q, R, P, lo, hi); \
    found = true;                                   \
  }
  LQ_FOR_EACH_DIM(X)
#undef X
  ctx->dyn = false;
  if (found && getenv("LQMPC_FORCE_DYN") != nullptr && lq_dyn_supported(n, m)) found = false;   // A/B measurements
  if (!found) {
    // no register-resident instantiation: the run-time-dimension route (one warp per sample, k_dyn.cu)
    if (!lq_dyn_supported(n, m))
      return lq_set_error(ctx, LQMPC_EINVAL, "unsupported (n, m): n <= 32 and m <= 8 are required");
    ctx->dyn = true;
  }
  if (ctx->ref_x) { cudaStreamSynchronize(ctx->stream); cudaFree(ctx->ref_x); ctx->ref_x = nullptr; }
  if (ctx->ref_u) { cudaStreamSynchronize(ctx->stream); cudaFree(ctx->ref_u); ctx->ref_u = nullptr; }
  ctx->ref_ld = 0;
  if (ctx->poly_dev) { cudaStreamSynchronize(ctx->stream); cudaFree(ctx->poly_dev); ctx->poly_dev = nullptr; }
  ctx->poly_p = 0;
  ctx->n = n;
  ctx->m = m;
  ctx->N_opc = N_opc;
  ctx->has_problem = false;
  int rc = ctx->dyn ? lq_dyn_set_problem(ctx, A, B, Q, R, P, lo, hi) : lq_launch_prepare(ctx);
  if (rc) return rc;
  ctx->has_problem = true;
  return LQMPC_OK;
}

int lqmpc_set_problem_tiled(lqmpc_ctx* ctx, int n, int m, const double* A, const double* B, const double* Q,
                            const double* R, const double* P, int N_opc) {
  if (!ctx) return LQMPC_EINVAL;
  if (!A || !B || !Q || !R || !P) return lq_set_error(ctx, LQMPC_EINVAL, "null problem matrix");
  if (!lq_tiled_supported(n, m)) return lq_set_error(ctx, LQMPC_EINVAL, "unsupported tiled (n, m): 32x8, 16x4");
  cudaSetDevice(ctx->device);
  ctx->has_tiled = false;
  if (ctx->tiled_pb) { cudaStreamSynchronize(ctx->stream); cudaFree(ctx->tiled_pb); ctx->tiled_pb = nullptr; }
  if (ctx->tiled_zero) { cudaFree(ctx->tiled_zero); ctx->tiled_zero = nullptr; }
  const size_t nd = lq_tiled_pb_doubles(n, m);
  const size_t nz = (size_t)(n * n + n * m + n);
  int rc = lq_check_cuda(ctx, cudaMalloc(&ctx->tiled_pb, nd * sizeof(double)), "cudaMalloc tiled problem");
  if (rc) return rc;
  rc = lq_check_cuda(ctx, cudaMalloc(&ctx->tiled_zero, nz * sizeof(double)), "cudaMalloc tiled zeros");
  if (rc) return rc;
  double* d = reinterpret_cast<double*>(ctx->tiled_pb);
  cudaMemsetAsync(ctx->tiled_pb, 0, nd * sizeof(double), ctx->stream);
  cudaMemsetAsync(ctx->tiled_zero, 0, nz * sizeof(double), ctx->stream);
  size_t off = 0;
  const double* src[5] = {A, B, Q, R, P};
  const size_t len[5] = {(size_t)n * n, (size_t)n * m, (size_t)n * n, (size_t)m * m, (size_t)n * n};
  for (int i = 0; i < 5; ++i) {
    rc = lq_check_cuda(ctx, cudaMemcpyAsync(d + off, src[i], len[i] * sizeof(double), cudaMemcpyHostToDevice,
                                            ctx->stream), "H2D tiled problem");
    if (rc) return rc;
    off += len[i];
  }
  ctx->tn = n; ctx->tm = m;
  // expert cost matrix Pexp = N_opc-step Riccati cost-to-go of the TRUE model: the evaluation kernel itself on dA = dB = 0
  TiledEval t;
  const double* z = reinterpret_cast<const double*>(ctx->tiled_zero);
  t.S = 1; t.dA = z; t.dB = z + n * n; t.x0 = z + n * n + n * m;
  t.N_min = t.N_max = (N_opc > 0) ? N_opc : 1000;
  t.J = t.rho = t.ratio = t.Vn = nullptr; t.flags = nullptr;
  t.Pout = d + off;                                  // off == offset of Pexp
  rc = lq_launch_tiled(ctx, t);
  if (rc) return rc;
  rc = lq_check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "tiled prepare sync");
  if (rc) return rc;
  ctx->N_opc = N_opc;
  ctx->has_tiled = true;
  return LQMPC_OK;
}

int lqmpc_get_prepared_tiled(lqmpc_ctx* ctx, double* Pexp_host, int64_t capacity) {
  if (!ctx || !Pexp_host) return LQMPC_EINVAL;
  if (!ctx->has_tiled) return lq_set_error(ctx, LQMPC_ESTATE, "tiled problem not set");
  const int n = ctx->tn, m = ctx->tm;
  if (capacity < (int64_t)n * n) return lq_set_error(ctx, LQMPC_EINVAL, "capacity too small");
  const double* d = reinterpret_cast<const double*>(ctx->tiled_pb) + (3 * n * n + n * m + m * m);
  int rc = lq_check_cuda(ctx, cudaMemcpyAsync(Pexp_host, d, (size_t)n * n * sizeof(double), cudaMemcpyDeviceToHost,
                                              ctx->stream), "D2H Pexp");
  if (rc) return rc;
  return lq_check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "sync");
}

int lqmpc_eval_batch_tiled(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, const double* x0, int N_min,
                           int N_max, double* J, double* rho, double* ratio, double* V_N, int32_t* flags) {
  if (!ctx) return LQMPC_EINVAL;
  if (!ctx->has_tiled) return lq_set_error(ctx, LQMPC_ESTATE, "tiled problem not set");
  if (S < 0 || N_min < 1 || N_max < N_min) return lq_set_error(ctx, LQMPC_EINVAL, "bad S/N_min/N_max");
  if (S == 0) return LQMPC_OK;
  if (!dA || !dB || !x0) return lq_set_error(ctx, LQMPC_EINVAL, "null input");
  if (((uintptr_t)dA | (uintptr_t)dB | (uintptr_t)x0) & 15)
    return lq_set_error(ctx, LQMPC_EINVAL, "tiled inputs must be 16-byte aligned (TMA bulk copies)");
  cudaSetDevice(ctx->device);
  TiledEval t;
  t.S = S; t.dA = dA; t.dB = dB; t.x0 = x0; t.N_min = N_min; t.N_max = N_max;
  t.J = J; t.rho = rho; t.ratio = ratio; t.Vn = V_N; t.flags = flags; t.Pout = nullptr;
  return lq_launch_tiled(ctx, t);
}

int lqmpc_eval_batch_tiled_host(lqmpc_ctx* ctx, int64_t S, const double* dA_h, const double* dB_h, const double* x0_h,
                                int N_min, int N_max, double* J_h, double* rho_h, double* ratio_h, int32_t* flags_h,
                                int64_t chunk) {
  if (!ctx) return LQMPC_EINVAL;
  if (!ctx->has_tiled) return lq_set_error(ctx, LQMPC_ESTATE, "tiled problem not set");
  if (S < 0 || N_min < 1 || N_max < N_min) return lq_set_error(ctx, LQMPC_EINVAL, "bad S/N_min/N_max");
  if (S == 0) return LQMPC_OK;
  if (!dA_h || !dB_h || !x0_h) return lq_set_error(ctx, LQMPC_EINVAL, "null input");
  cudaSetDevice(ctx->device);
  const int n = ctx->tn, m = ctx->tm, H = N_max - N_min + 1;
  if (chunk <= 0) chunk = 16384;
  if (chunk > S) chunk = S;
  chunk = (chunk + 1) & ~(int64_t)1;                       // keeps every slot section 16-byte aligned (TMA sources)
  const int64_t in_d = (int64_t)n * n + (int64_t)n * m + n;
  const size_t slot = (size_t)chunk * 8 * (size_t)(in_d + 3 * H) + (size_t)chunk * 4 * (size_t)H + 64;
  int rc = ensure_pipe(ctx, slot);
  if (rc) return rc;
  for (int i = 0; i < 6; ++i)
    if (!ctx->tp_ev[i]) {
      rc = lq_check_cuda(ctx, cudaEventCreateWithFlags(&ctx->tp_ev[i], cudaEventDisableTiming), "pipeline event");
      if (rc) return rc;
    }
  cudaStream_t s_in = ctx->pipe_stream[0], s_out = ctx->pipe_stream[1], s_cmp = ctx->stream;
  rc = lq_check_cuda(ctx, cudaStreamSynchronize(s_cmp), "pre-pipeline sync");
  if (rc) return rc;
  // three streams: H2D of chunk c+1 and D2H of chunk c-1 overlap the two kernels of chunk c (which share one scratch).
  // The first chunk's H2D is the one copy nothing can hide, so the chunks RAMP: they start at chunk / 8 and grow by 11/8
  // — a chunk's H2D (10.5 kB per sample at 32 x 8 over ~54 GB/s) takes 0.72 of the previous chunk's kernel time at
  // cfg 5, so every later copy stays hidden — until they reach `chunk`. (Fixed chunks of 16 384 left 3.2 ms of the
  // 36.8 ms step exposed: e2e 3.40e6 vs 3.74e6 evals/s device-resident.)
  int64_t cur = chunk / 8;
  if (cur < 512) cur = 512;
  cur = (cur + 1) & ~(int64_t)1;
  if (cur > chunk) cur = chunk;
  int64_t s0 = 0;
  for (int64_t c = 0; s0 < S; ++c) {
    const int b = (int)(c & 1);
    cudaEvent_t ev_in = ctx->tp_ev[b], ev_cmp = ctx->tp_ev[2 + b], ev_out = ctx->tp_ev[4 + b];
    const int64_t cs = (s0 + cur <= S) ? cur : (S - s0);
    double* d_dA = reinterpret_cast<double*>(ctx->pipe_buf[b]);
    double* d_dB = d_dA + (int64_t)n * n * chunk;
    double* d_x0 = d_dB + (int64_t)n * m * chunk;
    double* d_J = d_x0 + (int64_t)n * chunk;
    double* d_rho = d_J + (int64_t)H * chunk;
    double* d_ratio = d_rho + (int64_t)H * chunk;
    int32_t* d_flags = reinterpret_cast<int32_t*>(d_ratio + (int64_t)H * chunk);
    if (c >= 2) LQ_PIPE(cudaStreamWaitEvent(s_in, ctx->tp_ev[2 + b], 0), "wait slot inputs");   // chunk c-2 computed
    LQ_PIPE(cudaMemcpyAsync(d_dA, dA_h + s0 * n * n, (size_t)cs * n * n * 8, cudaMemcpyHostToDevice, s_in), "H2D dA");
    LQ_PIPE(cudaMemcpyAsync(d_dB, dB_h + s0 * n * m, (size_t)cs * n * m * 8, cudaMemcpyHostToDevice, s_in), "H2D dB");
    LQ_PIPE(cudaMemcpyAsync(d_x0, x0_h + s0 * n, (size_t)cs * n * 8, cudaMemcpyHostToDevice, s_in), "H2D x0");
    LQ_PIPE(cudaEventRecord(ev_in, s_in), "record H2D");
    LQ_PIPE(cudaStreamWaitEvent(s_cmp, ev_in, 0), "wait H2D");
    if (c >= 2) LQ_PIPE(cudaStreamWaitEvent(s_cmp, ctx->tp_ev[4 + b], 0), "wait slot outputs");   // chunk c-2 copied back
    TiledEval t;
    t.S = cs; t.dA = d_dA; t.dB = d_dB; t.x0 = d_x0; t.N_min = N_min; t.N_max = N_max;
    t.J = d_J; t.rho = d_rho; t.ratio = d_ratio; t.Vn = nullptr; t.flags = d_flags; t.Pout = nullptr;
    // [H][cs] tables inside the slot: the kernels index outputs with leading dimension S = cs
    rc = lq_launch_tiled(ctx, t);
    if (rc) return pipe_abort(ctx, rc);
    LQ_PIPE(cudaEventRecord(ev_cmp, s_cmp), "record compute");
    LQ_PIPE(cudaStreamWaitEvent(s_out, ev_cmp, 0), "wait compute");
    const size_t w = (size_t)cs * 8, sp = (size_t)S * 8;
    if (J_h) LQ_PIPE(cudaMemcpy2DAsync(J_h + s0, sp, d_J, w, w, (size_t)H, cudaMemcpyDeviceToHost, s_out), "D2H J");
    if (rho_h) LQ_PIPE(cudaMemcpy2DAsync(rho_h + s0, sp, d_rho, w, w, (size_t)H, cudaMemcpyDeviceToHost, s_out), "D2H rho");
    if (ratio_h)
      LQ_PIPE(cudaMemcpy2DAsync(ratio_h + s0, sp, d_ratio, w, w, (size_t)H, cudaMemcpyDeviceToHost, s_out), "D2H ratio");
    if (flags_h)
      LQ_PIPE(cudaMemcpy2DAsync(flags_h + s0, (size_t)S * 4, d_flags, (size_t)cs * 4, (size_t)cs * 4, (size_t)H,
                                cudaMemcpyDeviceToHost, s_out), "D2H flags");
    LQ_PIPE(cudaEventRecord(ev_out, s_out), "record D2H");
    s0 += cs;
    cur = (cur * 11 / 8 + 1) & ~(int64_t)1;
    if (cur > chunk) cur = chunk;
  }
  rc = lq_check_cuda(ctx, cudaStreamSynchronize(s_out), "pipeline sync (D2H)");
  if (rc) return rc;
  rc = lq_check_cuda(ctx, cudaStreamSynchronize(s_cmp), "pipeline sync (compute)");
  if (rc) return rc;
  return lq_check_cuda(ctx, cudaGetLastError(), "tiled host pipeline");
}

int lqmpc_get_prepared(lqmpc_ctx* ctx, double* out, int64_t capacity) {
  if (!ctx || !out) return LQMPC_EINVAL;
  if (!ctx->has_problem) return lq_set_error(ctx, LQMPC_ESTATE, "problem not set");
  const int n = ctx->n;
  if (capacity < 2 * n * n + 4) return lq_set_error(ctx, LQMPC_EINVAL, "capacity too small");
  if (ctx->dyn) return lq_dyn_get_prepared(ctx, out);
  bool done = false;
#define X(N_, M_)                                                                       \
  if (!done && ctx->n == N_ && ctx->m == M_) {                                          \
    const lq::Problem<N_, M_>& pb = *reinterpret_cast<const lq::Problem<N_, M_>*>(ctx->pb); \
    memcpy(out, pb.Pexp, sizeof(pb.Pexp));                                              \
    memcpy(out + N_ * N_, pb.Qinv, sizeof(pb.Qinv));                                    \
    out[2 * N_ * N_ + 0] = pb.maxQ;                                                     \
    out[2 * N_ * N_ + 1] = pb.minQ;                                                     \
    out[2 * N_ * N_ + 2] = pb.maxR;                                                     \
    out[2 * N_ * N_ + 3] = pb.minR;                                                     \
    done = true;                                                                        \
  }
  LQ_FOR_EACH_DIM(X)
#undef X
  return done ? LQMPC_OK : LQMPC_EINVAL;
}

int lqmpc_eval_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, const double* x0, int N_min,
                     int N_max, int T, double* J, double* rho, double* ratio, double* V_N, double* J_T,
                     int32_t* flags, double* K0) {
  if (!ctx) return LQMPC_EINVAL;
  if (!ctx->has_problem) return lq_set_error(ctx, LQMPC_ESTATE, "problem not set");
  if (S < 0 || N_min < 1 || N_max < N_min || T < 0) return lq_set_error(ctx, LQMPC_EINVAL, "bad S/N_min/N_max/T");
  if (S == 0) return LQMPC_OK;
  if (!dA || !dB || !x0) return lq_set_error(ctx, LQMPC_EINVAL, "null input");
  if (J_T && T <= 0) return lq_set_error(ctx, LQMPC_EINVAL, "J_T requested with T <= 0");
  cudaSetDevice(ctx->device);
  EvalArgs a;
  a.S = S; a.ld = S; a.dA = dA; a.dB = dB; a.x0 = x0;
  a.N_min = N_min; a.N_max = N_max; a.T = J_T ? T : 0;
  a.J = J; a.rho = rho; a.ratio = ratio; a.Vn = V_N; a.JT = J_T; a.flags = flags; a.K0 = K0;
  return ctx->dyn ? lq_dyn_eval(ctx, a, ctx->stream) : lq_launch_eval(ctx, a, ctx->stream);
}

int lqmpc_eval_seeded(lqmpc_ctx* ctx, uint64_t seed, int64_t first, int64_t S, double e_A, double e_B, int N_min,
                      int N_max, double* J, double* rho, double* ratio, int32_t* flags, double* moments) {
  if (!ctx) return LQMPC_EINVAL;
  if (!ctx->has_problem) return lq_set_error(ctx, LQMPC_ESTATE, "problem not set");
  if (S < 0 || first < 0 || N_min < 1 || N_max < N_min) return lq_set_error(ctx, LQMPC_EINVAL, "bad S/first/N_min/N_max");
  if (ctx->dyn) return lq_set_error(ctx, LQMPC_EINVAL, "lqmpc_eval_seeded needs a compiled (n, m) pair; see lqmpc_supported_dims()");
  if (S == 0) return LQMPC_OK;
  cudaSetDevice(ctx->device);
  const int H = N_max - N_min + 1;
  double* tab[3] = {J, rho, ratio};
  if (moments) {
    // the moments are taken over ONE contiguous [3 H][S] table (J rows, rho rows, ratio rows): tables the caller did
    // not ask for live in the context's own scratch
    const bool contiguous = J && rho && ratio && rho == J + (int64_t)H * S && ratio == rho + (int64_t)H * S;
    if (!contiguous) {
      if (J || rho || ratio)
        return lq_set_error(ctx, LQMPC_EINVAL, "with moments, pass J/rho/ratio as one contiguous [3H][S] table or all NULL");
      const size_t need = (size_t)3 * H * S * sizeof(double);
      if (need > ctx->seed_bytes) {
        if (ctx->seed_buf) { cudaStreamSynchronize(ctx->stream); cudaFree(ctx->seed_buf); ctx->seed_buf = nullptr; }
        ctx->seed_bytes = 0;
        int rc = lq_check_cuda(ctx, cudaMalloc(&ctx->seed_buf, need), "cudaMalloc seeded tables");
        if (rc) return rc;
        ctx->seed_bytes = need;
      }
      double* b = reinterpret_cast<double*>(ctx->seed_buf);
      tab[0] = b; tab[1] = b + (int64_t)H * S; tab[2] = b + (int64_t)2 * H * S;
    }
  }
  EvalArgs a;
  a.S = S; a.ld = S; a.dA = nullptr; a.dB = nullptr; a.x0 = nullptr;
  a.N_min = N_min; a.N_max = N_max; a.T = 0;
  a.J = tab[0]; a.rho = tab[1]; a.ratio = tab[2]; a.Vn = nullptr; a.JT = nullptr; a.flags = flags; a.K0 = nullptr;
  int rc = lq_launch_eval_seeded(ctx, a, seed, first, e_A, e_B);
  if (rc) return rc;
  if (moments) rc = lq_launch_moments(ctx, tab[0], 3 * H, S, S, moments);
  return rc;
}

int lqmpc_eval_batch_host(lqmpc_ctx* ctx, int64_t S, const double* dA_h, const double* dB_h, const double* x0_h,
                          int N_min, int N_max, int T, double* J_h, double* rho_h, double* ratio_h,
                          int32_t* flags_h, int64_t chunk) {
  if (!ctx) return LQMPC_EINVAL;
  if (!ctx->has_problem) return lq_set_error(ctx, LQMPC_ESTATE, "problem not set");
  if (S < 0 || N_min < 1 || N_max < N_min) return lq_set_error(ctx, LQMPC_EINVAL, "bad S/N_min/N_max");
  if (S == 0) return LQMPC_OK;
  if (!dA_h || !dB_h || !x0_h) return lq_set_error(ctx, LQMPC_EINVAL, "null input");
  (void)T;
  cudaSetDevice(ctx->device);
  const int n = ctx->n, m = ctx->m;
  const int H = N_max - N_min + 1;
  if (chunk <= 0) chunk = 1 << 20;
  if (chunk > S) chunk = S;
  chunk = (chunk + 31) / 32 * 32;
  const int64_t in_rows = (int64_t)n * n + (int64_t)n * m + n;
  const int64_t out_rows = 3 * (int64_t)H;  // J, rho, ratio
  const size_t slot = (size_t)chunk * 8 * (size_t)(in_rows + out_rows) + (size_t)chunk * 4 * (size_t)H;
  int rc = ensure_pipe(ctx, slot);
  if (rc) return rc;
  // the caller's stream must be idle w.r.t. these buffers: order the pipeline after it
  rc = lq_check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "pre-pipeline sync");
  if (rc) return rc;
  int64_t nchunks = (S + chunk - 1) / chunk;
  for (int64_t c = 0; c < nchunks; ++c) {
    const int b = (int)(c & 1);
    cudaStream_t st = ctx->pipe_stream[b];
    const int64_t s0 = c * chunk;
    const int64_t cs = (s0 + chunk <= S) ? chunk : (S - s0);
    double* base = reinterpret_cast<double*>(ctx->pipe_buf[b]);
    double* d_dA = base;
    double* d_dB = d_dA + (int64_t)n * n * chunk;
    double* d_x0 = d_dB + (int64_t)n * m * chunk;
    double* d_J = d_x0 + (int64_t)n * chunk;
    double* d_rho = d_J + (int64_t)H * chunk;
    double* d_ratio = d_rho + (int64_t)H * chunk;
    int32_t* d_flags = reinterpret_cast<int32_t*>(d_ratio + (int64_t)H * chunk);
    const size_t w = (size_t)cs * 8, dp = (size_t)chunk * 8, sp = (size_t)S * 8;
    // stream order makes slot reuse safe: chunk c+2 is enqueued on the same stream after chunk c's D2H
    rc = lq_check_cuda(ctx, cudaMemcpy2DAsync(d_dA, dp, dA_h + s0, sp, w, (size_t)n * n, cudaMemcpyHostToDevice, st),
                       "H2D dA");
    if (rc) return pipe_abort(ctx, rc);
    rc = lq_check_cuda(ctx, cudaMemcpy2DAsync(d_dB, dp, dB_h + s0, sp, w, (size_t)n * m, cudaMemcpyHostToDevice, st),
                       "H2D dB");
    if (rc) return pipe_abort(ctx, rc);
    rc = lq_check_cuda(ctx, cudaMemcpy2DAsync(d_x0, dp, x0_h + s0, sp, w, (size_t)n, cudaMemcpyHostToDevice, st),
                       "H2D x0");
    if (rc) return pipe_abort(ctx, rc);
    EvalArgs a;
    a.S = cs; a.ld = chunk; a.dA = d_dA; a.dB = d_dB; a.x0 = d_x0;
    a.N_min = N_min; a.N_max = N_max; a.T = 0;
    a.J = J_h ? d_J : nullptr; a.rho = rho_h ? d_rho : nullptr; a.ratio = ratio_h ? d_ratio : nullptr;
    a.Vn = nullptr; a.JT = nullptr; a.flags = flags_h ? d_flags : nullptr; a.K0 = nullptr;
    rc = ctx->dyn ? lq_dyn_eval(ctx, a, st) : lq_launch_eval(ctx, a, st);
    if (rc) return pipe_abort(ctx, rc);
    if (J_h) {
      rc = lq_check_cuda(ctx, cudaMemcpy2DAsync(J_h + s0, sp, d_J, dp, w, (size_t)H, cudaMemcpyDeviceToHost, st),
                         "D2H J");
      if (rc) return pipe_abort(ctx, rc);
    }
    if (rho_h) {
      rc = lq_check_cuda(ctx, cudaMemcpy2DAsync(rho_h + s0, sp, d_rho, dp, w, (size_t)H, cudaMemcpyDeviceToHost, st),
                         "D2H rho");
      if (rc) return pipe_abort(ctx, rc);
    }
    if (ratio_h) {
      rc = lq_check_cuda(
          ctx, cudaMemcpy2DAsync(ratio_h + s0, sp, d_ratio, dp, w, (size_t)H, cudaMemcpyDeviceToHost, st), "D2H ratio");
      if (rc) return pipe_abort(ctx, rc);
    }
    if (flags_h) {
      rc = lq_check_cuda(ctx,
                         cudaMemcpy2DAsync(flags_h + s0, (size_t)S * 4, d_flags, (size_t)chunk * 4, (size_t)cs * 4,
                                           (size_t)H, cudaMemcpyDeviceToHost, st),
                         "D2H flags");
      if (rc) return pipe_abort(ctx, rc);
    }
  }
  for (int b = 0; b < 2; ++b) {
    rc = lq_check_cuda(ctx, cudaStreamSynchronize(ctx->pipe_stream[b]), "pipeline sync");
    if (rc) return rc;
  }
  return LQMPC_OK;
}

int lqmpc_set_references(lqmpc_ctx* ctx, int n_cols, const double* x_ref_host, const double* u_ref_host) {
  if (!ctx) return LQMPC_EINVAL;
  if (!ctx->has_problem) return lq_set_error(ctx, LQMPC_ESTATE, "problem not set");
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (ctx->ref_x) { cudaFree(ctx->ref_x); ctx->ref_x = nullptr; }
  if (ctx->ref_u) { cudaFree(ctx->ref_u); ctx->ref_u = nullptr; }
  ctx->ref_ld = 0;
  if (n_cols <= 0 || (!x_ref_host && !u_ref_host)) return LQMPC_OK;     // cleared: zero references
  const int n = ctx->n, m = ctx->m;
  if (x_ref_host) {
    int rc = lq_check_cuda(ctx, cudaMalloc(&ctx->ref_x, (size_t)n * n_cols * sizeof(double)), "cudaMalloc x_ref");
    if (rc) return rc;
    rc = lq_check_cuda(ctx, cudaMemcpy(ctx->ref_x, x_ref_host, (size_t)n * n_cols * sizeof(double),
                                       cudaMemcpyHostToDevice), "H2D x_ref");
    if (rc) return rc;
  }
  if (u_ref_host) {
    int rc = lq_check_cuda(ctx, cudaMalloc(&ctx->ref_u, (size_t)m * n_cols * sizeof(double)), "cudaMalloc u_ref");
    if (rc) return rc;
    rc = lq_check_cuda(ctx, cudaMemcpy(ctx->ref_u, u_ref_host, (size_t)m * n_cols * sizeof(double),
                                       cudaMemcpyHostToDevice), "H2D u_ref");
    if (rc) return rc;
  }
  ctx->ref_ld = n_cols;
  return LQMPC_OK;
}

int lqmpc_set_input_polytope(lqmpc_ctx* ctx, int p, const double* F_host) {
  if (!ctx) return LQMPC_EINVAL;
  if (!ctx->has_problem) return lq_set_error(ctx, LQMPC_ESTATE, "problem not set");
  // validate first: a rejected call leaves the installed polytope (or the box) as it was
  const bool clear = (p <= 0 || !F_host);
  if (!clear) {
    if (ctx->dyn)
      return lq_set_error(ctx, LQMPC_EINVAL, "general input polytopes need a compiled (n, m) pair; see lqmpc_supported_dims()");
    if (p > lq::kPolyMaxRows) return lq_set_error(ctx, LQMPC_EINVAL, "input polytope: at most 12 rows");
    for (int e = 0; e < p * ctx->m; ++e)
      if (!(fabs(F_host[e]) <= 1.79e308)) return lq_set_error(ctx, LQMPC_EINVAL, "input polytope: non-finite entry");
  }
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (ctx->poly_dev) { cudaFree(ctx->poly_dev); ctx->poly_dev = nullptr; }
  ctx->poly_p = 0;
  if (clear) return LQMPC_OK;                                          // cleared: the box of lqmpc_set_problem
  const size_t bytes = (size_t)p * ctx->m * sizeof(double);
  int rc = lq_check_cuda(ctx, cudaMalloc(&ctx->poly_dev, bytes), "cudaMalloc F_u");
  if (rc) return rc;
  rc = lq_check_cuda(ctx, cudaMemcpy(ctx->poly_dev, F_host, bytes, cudaMemcpyHostToDevice), "H2D F_u");
  if (rc) return rc;
  ctx->poly_p = p;
  return LQMPC_OK;
}

int lqmpc_mpc_solve_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, int N, int npts,
                          const double* pts, const double* x0, double* V, double* u0, double* M_V, int32_t* flags) {
  if (!ctx) return LQMPC_EINVAL;
  if (!ctx->has_problem) return lq_set_error(ctx, LQMPC_ESTATE, "problem not set");
  if (S < 0 || N < 1) return lq_set_error(ctx, LQMPC_EINVAL, "bad S/N");
  if (S == 0) return LQMPC_OK;
  if ((pts == nullptr) == (x0 == nullptr)) return lq_set_error(ctx, LQMPC_EINVAL, "give exactly one of pts / x0");
  if (pts && npts < 1) return lq_set_error(ctx, LQMPC_EINVAL, "npts < 1");
  cudaSetDevice(ctx->device);
  MpcArgs a{};
  a.S = S; a.dA = dA; a.dB = dB; a.N = N; a.T = 0; a.npts = npts; a.pts = pts; a.x0 = x0;
  a.V = V; a.u0 = u0; a.M_V = M_V; a.flags = flags;
  return ctx->dyn ? lq_dyn_mpc(ctx, a, false) : lq_launch_mpc(ctx, a, false);
}

int lqmpc_simulate_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, int N, int T,
                         const double* x0_shared, const double* x0, double* J_T, double* X, double* U,
                         int32_t* flags, int32_t* n_active) {
  if (!ctx) return LQMPC_EINVAL;
  if (!ctx->has_problem) return lq_set_error(ctx, LQMPC_ESTATE, "problem not set");
  if (S < 0 || N < 1 || T < 0) return lq_set_error(ctx, LQMPC_EINVAL, "bad S/N/T");
  if (S == 0) return LQMPC_OK;
  if ((x0_shared == nullptr) == (x0 == nullptr))
    return lq_set_error(ctx, LQMPC_EINVAL, "give exactly one of x0_shared / x0");
  cudaSetDevice(ctx->device);
  MpcArgs a{};
  a.S = S; a.dA = dA; a.dB = dB; a.N = N; a.T = T; a.npts = 1; a.pts = x0_shared; a.x0 = x0;
  a.J_T = J_T; a.X = X; a.U = U; a.flags = flags; a.n_active = n_active;
  return ctx->dyn ? lq_dyn_mpc(ctx, a, true) : lq_launch_mpc(ctx, a, true);
}

int lqmpc_simulate_inf_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, int N, int T_max,
                             const double* x0_shared, const double* x0, double* J_inf, int32_t* T_cert,
                             int32_t* flags) {
  if (!ctx) return LQMPC_EINVAL;
  if (!ctx->has_problem) return lq_set_error(ctx, LQMPC_ESTATE, "problem not set");
  if (S < 0 || N < 1 || T_max < 0) return lq_set_error(ctx, LQMPC_EINVAL, "bad S/N/T_max");
  if (S == 0) return LQMPC_OK;
  if ((x0_shared == nullptr) == (x0 == nullptr))
    return lq_set_error(ctx, LQMPC_EINVAL, "give exactly one of x0_shared / x0");
  // with references the state does not converge to the origin and the reference's J_T does not subtract them
  if (ctx->ref_ld > 0) return lq_set_error(ctx, LQMPC_EINVAL, "the infinite-horizon cost is for regulation (no references)");
  cudaSetDevice(ctx->device);
  MpcArgs a{};
  a.S = S; a.dA = dA; a.dB = dB; a.N = N; a.T = T_max; a.npts = 1; a.pts = x0_shared; a.x0 = x0;
  a.J_inf = J_inf; a.T_cert = T_cert; a.flags = flags;
  return ctx->dyn ? lq_dyn_simulate_inf(ctx, a) : lq_launch_simulate_inf(ctx, a);
}

namespace {

// shared checks of the worst-case entry points; the sup-over-x0 ones take no x0 and pass need_x0 = false
int worst_check(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, const double* x0, int N,
                bool need_x0 = true) {
  if (!ctx->has_problem) {
    if (ctx->has_tiled)
      return lq_set_error(ctx, LQMPC_EINVAL, "the worst-case entry points need a compiled (n, m) pair; see "
                                             "lqmpc_supported_dims() (not the tiled route)");
    return lq_set_error(ctx, LQMPC_ESTATE, "problem not set");
  }
  if (ctx->dyn)
    return lq_set_error(ctx, LQMPC_EINVAL, "the worst-case entry points need a compiled (n, m) pair; see "
                                           "lqmpc_supported_dims() (not the run-time-dimension route)");
  if (S < 0 || N < 1) return lq_set_error(ctx, LQMPC_EINVAL, "bad S/N");
  if (S > 0 && (!dA || !dB || (need_x0 && !x0))) return lq_set_error(ctx, LQMPC_EINVAL, "null input");
  return LQMPC_OK;
}

// the ascent's settings, shared by lqmpc_worst_case_batch / lqmpc_worst_case_sup_batch
int ascent_check(lqmpc_ctx* ctx, double e_A, double e_B, int norm_type, int max_iter, double tol) {
  if (!(e_A >= 0.0 && e_A <= 1.79e308) || !(e_B >= 0.0 && e_B <= 1.79e308))
    return lq_set_error(ctx, LQMPC_EINVAL, "e_A / e_B must be finite and >= 0");
  if (norm_type < 0 || norm_type > 2)
    return lq_set_error(ctx, LQMPC_EINVAL, "norm_type: 0 (Frobenius), 1 (spectral) or 2 (entrywise max)");
  if (max_iter < 0) return lq_set_error(ctx, LQMPC_EINVAL, "max_iter < 0");
  if (!(tol > 0.0)) return lq_set_error(ctx, LQMPC_EINVAL, "tol must be > 0");
  return LQMPC_OK;
}

}  // namespace

int lqmpc_eval_grad_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, const double* x0, int N,
                          double* J, double* rho, double* ratio, double* gA, double* gB, int32_t* flags) {
  if (!ctx) return LQMPC_EINVAL;
  int rc = worst_check(ctx, S, dA, dB, x0, N);
  if (rc || S == 0) return rc;
  cudaSetDevice(ctx->device);
  WorstArgs a{};
  a.S = S; a.dA = dA; a.dB = dB; a.x0 = x0; a.N = N;
  a.J = J; a.rho = rho; a.ratio = ratio; a.gA = gA; a.gB = gB; a.flags = flags;
  return lq_launch_eval_grad(ctx, a);
}

int lqmpc_worst_case_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, const double* x0, int N,
                           double e_A, double e_B, int norm_type, int max_iter, double tol, double* dA_out,
                           double* dB_out, double* J, double* rho, double* ratio, int32_t* iters, int32_t* flags) {
  if (!ctx) return LQMPC_EINVAL;
  int rc = worst_check(ctx, S, dA, dB, x0, N);
  if (rc) return rc;
  rc = ascent_check(ctx, e_A, e_B, norm_type, max_iter, tol);
  if (rc || S == 0) return rc;
  cudaSetDevice(ctx->device);
  WorstArgs a{};
  a.S = S; a.dA = dA; a.dB = dB; a.x0 = x0; a.N = N;
  a.eA = e_A; a.eB = e_B; a.norm = norm_type; a.max_iter = max_iter; a.tol = tol;
  a.dA_out = dA_out; a.dB_out = dB_out; a.J = J; a.rho = rho; a.ratio = ratio; a.iters = iters; a.flags = flags;
  return lq_launch_worst_case(ctx, a);
}

int lqmpc_ratio_sup_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, int N, double* gamma,
                          double* x_worst, double* gap, double* rho, double* gA, double* gB, int32_t* flags) {
  if (!ctx) return LQMPC_EINVAL;
  int rc = worst_check(ctx, S, dA, dB, nullptr, N, false);
  if (rc || S == 0) return rc;
  cudaSetDevice(ctx->device);
  WorstArgs a{};
  a.S = S; a.dA = dA; a.dB = dB; a.x0 = nullptr; a.N = N;
  a.J = gamma; a.rho = rho; a.gA = gA; a.gB = gB; a.flags = flags;
  return lq_launch_ratio_sup(ctx, a, x_worst, gap);
}

int lqmpc_worst_case_sup_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, int N, double e_A,
                               double e_B, int norm_type, int max_iter, double tol, double* dA_out, double* dB_out,
                               double* gamma, double* x_worst, double* rho, int32_t* iters, int32_t* flags) {
  if (!ctx) return LQMPC_EINVAL;
  int rc = worst_check(ctx, S, dA, dB, nullptr, N, false);
  if (rc) return rc;
  rc = ascent_check(ctx, e_A, e_B, norm_type, max_iter, tol);
  if (rc || S == 0) return rc;
  cudaSetDevice(ctx->device);
  WorstArgs a{};
  a.S = S; a.dA = dA; a.dB = dB; a.x0 = nullptr; a.N = N;
  a.eA = e_A; a.eB = e_B; a.norm = norm_type; a.max_iter = max_iter; a.tol = tol;
  a.dA_out = dA_out; a.dB_out = dB_out; a.J = gamma; a.rho = rho; a.iters = iters; a.flags = flags;
  return lq_launch_worst_case_sup(ctx, a, x_worst);
}

namespace {

// checks of the constrained worst-case entry points: those of lqmpc_simulate_inf_batch and of the worst-case calls
int worst_inf_check(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, int N, int T_max,
                    const double* x0_shared, const double* x0) {
  int rc = worst_check(ctx, S, dA, dB, nullptr, N, false);
  if (rc) return rc;
  if (T_max < 0) return lq_set_error(ctx, LQMPC_EINVAL, "bad T_max");
  if ((x0_shared == nullptr) == (x0 == nullptr))
    return lq_set_error(ctx, LQMPC_EINVAL, "give exactly one of x0_shared / x0");
  if (ctx->ref_ld > 0) return lq_set_error(ctx, LQMPC_EINVAL, "the infinite-horizon cost is for regulation (no references)");
  if (ctx->poly_p > 0)
    return lq_set_error(ctx, LQMPC_EINVAL, "the constrained worst-case entry points take the input box, not a polytope");
  return LQMPC_OK;
}

}  // namespace

int lqmpc_simulate_inf_grad_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, int N, int T_max,
                                  const double* x0_shared, const double* x0, double* J_inf, int32_t* T_cert,
                                  double* rho, double* gA, double* gB, int32_t* flags) {
  if (!ctx) return LQMPC_EINVAL;
  int rc = worst_inf_check(ctx, S, dA, dB, N, T_max, x0_shared, x0);
  if (rc || S == 0) return rc;
  cudaSetDevice(ctx->device);
  WorstInfArgs a{};
  a.S = S; a.dA = dA; a.dB = dB; a.x0_shared = x0_shared; a.x0 = x0; a.N = N; a.T_max = T_max;
  a.J = J_inf; a.T_cert = T_cert; a.rho = rho; a.gA = gA; a.gB = gB; a.flags = flags;
  return lq_launch_simulate_inf_grad(ctx, a);
}

int lqmpc_worst_case_inf_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, int N, int T_max,
                               const double* x0_shared, const double* x0, double e_A, double e_B, int norm_type,
                               int max_iter, double tol, double* dA_out, double* dB_out, double* J_inf,
                               int32_t* T_cert, double* rho, int32_t* iters, int32_t* flags) {
  if (!ctx) return LQMPC_EINVAL;
  int rc = worst_inf_check(ctx, S, dA, dB, N, T_max, x0_shared, x0);
  if (rc) return rc;
  rc = ascent_check(ctx, e_A, e_B, norm_type, max_iter, tol);
  if (rc || S == 0) return rc;
  cudaSetDevice(ctx->device);
  WorstInfArgs a{};
  a.S = S; a.dA = dA; a.dB = dB; a.x0_shared = x0_shared; a.x0 = x0; a.N = N; a.T_max = T_max;
  a.eA = e_A; a.eB = e_B; a.norm = norm_type; a.max_iter = max_iter; a.tol = tol;
  a.dA_out = dA_out; a.dB_out = dB_out; a.J = J_inf; a.T_cert = T_cert; a.rho = rho; a.iters = iters; a.flags = flags;
  return lq_launch_worst_case_inf(ctx, a);
}

int lqmpc_bounds_fields(void) { return (int)lq::BF_COUNT; }

int lqmpc_bounds_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, int N, const double* e_A,
                       const double* e_B, double e_A_scalar, double e_B_scalar, const double* M_V,
                       double M_V_scalar, const double* x_shared, const double* x, const double* K_in,
                       const double* K_shared, const double* p3_host, double V_expert, double bar_u, double bar_d_u,
                       int strict_reference, double* alpha, double* beta, double* xi, double* eta, double* bound,
                       double* detail, double* K_out, double* P_out, int32_t* flags) {
  if (!ctx) return LQMPC_EINVAL;
  if (!ctx->has_problem) return lq_set_error(ctx, LQMPC_ESTATE, "problem not set");
  if (S < 0 || N < 1) return lq_set_error(ctx, LQMPC_EINVAL, "bad S/N");
  if (S == 0) return LQMPC_OK;
  if ((x_shared == nullptr) == (x == nullptr)) return lq_set_error(ctx, LQMPC_EINVAL, "give exactly one of x_shared / x");
  if (K_in && K_shared) return lq_set_error(ctx, LQMPC_EINVAL, "give at most one of K_in / K_shared");
  if (!p3_host) return lq_set_error(ctx, LQMPC_EINVAL, "null p");
  cudaSetDevice(ctx->device);
  BoundsArgs a{};
  a.S = S; a.dA = dA; a.dB = dB; a.N = N; a.eA = e_A; a.eB = e_B; a.eA_s = e_A_scalar; a.eB_s = e_B_scalar;
  a.MV = M_V; a.MV_s = M_V_scalar; a.x_shared = x_shared; a.x = x; a.K_in = K_in; a.K_shared = K_shared;
  a.p[0] = p3_host[0]; a.p[1] = p3_host[1]; a.p[2] = p3_host[2];
  a.V_expert = V_expert; a.bar_u = bar_u; a.bar_d_u = bar_d_u; a.strict = strict_reference;
  a.alpha = alpha; a.beta = beta; a.xi = xi; a.eta = eta; a.bound = bound; a.detail = detail; a.K_out = K_out;
  a.P_out = P_out; a.flags = flags;
  if (ctx->poly_p > 0) {
    if (bar_u < 0.0 || bar_d_u < 0.0)
      return lq_set_error(ctx, LQMPC_EINVAL, "with an input polytope installed bar_u / bar_d_u must be supplied (>= 0)");
    a.polyF = ctx->poly_dev; a.polyP = ctx->poly_p;
  }
  return ctx->dyn ? lq_dyn_bounds(ctx, a) : lq_launch_bounds(ctx, a);
}

int lqmpc_mpc_solve_range(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, int N_min, int N_max,
                          int npts, const double* pts, const double* x0, double* V, double* u0, double* M_V,
                          int32_t* flags) {
  if (!ctx) return LQMPC_EINVAL;
  if (!ctx->has_problem) return lq_set_error(ctx, LQMPC_ESTATE, "problem not set");
  if (S < 0 || N_min < 1 || N_max < N_min) return lq_set_error(ctx, LQMPC_EINVAL, "bad S/N_min/N_max");
  if (S == 0) return LQMPC_OK;
  if ((pts == nullptr) == (x0 == nullptr)) return lq_set_error(ctx, LQMPC_EINVAL, "give exactly one of pts / x0");
  if (pts && npts < 1) return lq_set_error(ctx, LQMPC_EINVAL, "npts < 1");
  cudaSetDevice(ctx->device);
  if (ctx->dyn || ctx->poly_p > 0 || ctx->ref_ld > 0) {
    // no fused kernel (run-time dimensions, input polytope, references): one single-horizon launch per N
    const int64_t P = pts ? npts : 1;
    for (int N = N_min; N <= N_max; ++N) {
      const int64_t h = N - N_min;
      const int rc = lqmpc_mpc_solve_batch(ctx, S, dA, dB, N, npts, pts, x0, V ? V + h * P * S : nullptr,
                                           u0 ? u0 + h * P * ctx->m * S : nullptr, M_V ? M_V + h * S : nullptr,
                                           flags ? flags + h * P * S : nullptr);
      if (rc) return rc;
    }
    return LQMPC_OK;
  }
  MpcArgs a{};
  a.S = S; a.dA = dA; a.dB = dB; a.N_min = N_min; a.N = N_max; a.T = 0; a.npts = npts; a.pts = pts; a.x0 = x0;
  a.V = V; a.u0 = u0; a.M_V = M_V; a.flags = flags;
  return lq_launch_mpc_range(ctx, a);
}

int lqmpc_bounds_range(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, int N_min, int N_max,
                       const double* e_A, const double* e_B, double e_A_scalar, double e_B_scalar, const double* M_V,
                       double M_V_scalar, const double* x_shared, const double* x, const double* K_in,
                       const double* K_shared, const double* p3_host, double V_expert, double bar_u, double bar_d_u,
                       int strict_reference, double* alpha, double* beta, double* xi, double* eta, double* bound,
                       double* detail, double* K_out, double* P_out, int32_t* flags) {
  if (!ctx) return LQMPC_EINVAL;
  if (!ctx->has_problem) return lq_set_error(ctx, LQMPC_ESTATE, "problem not set");
  if (S < 0 || N_min < 1 || N_max < N_min) return lq_set_error(ctx, LQMPC_EINVAL, "bad S/N_min/N_max");
  if (S == 0) return LQMPC_OK;
  if ((x_shared == nullptr) == (x == nullptr)) return lq_set_error(ctx, LQMPC_EINVAL, "give exactly one of x_shared / x");
  if (K_in && K_shared) return lq_set_error(ctx, LQMPC_EINVAL, "give at most one of K_in / K_shared");
  if (!p3_host) return lq_set_error(ctx, LQMPC_EINVAL, "null p");
  if (ctx->poly_p > 0 && (bar_u < 0.0 || bar_d_u < 0.0))
    return lq_set_error(ctx, LQMPC_EINVAL, "with an input polytope installed bar_u / bar_d_u must be supplied (>= 0)");
  cudaSetDevice(ctx->device);
  BoundsArgs a{};
  a.S = S; a.dA = dA; a.dB = dB; a.N_min = N_min; a.N = N_max; a.eA = e_A; a.eB = e_B; a.eA_s = e_A_scalar;
  a.eB_s = e_B_scalar; a.MV = M_V; a.MV_s = M_V_scalar; a.x_shared = x_shared; a.x = x; a.K_in = K_in;
  a.K_shared = K_shared; a.p[0] = p3_host[0]; a.p[1] = p3_host[1]; a.p[2] = p3_host[2];
  a.V_expert = V_expert; a.bar_u = bar_u; a.bar_d_u = bar_d_u; a.strict = strict_reference;
  a.alpha = alpha; a.beta = beta; a.xi = xi; a.eta = eta; a.bound = bound; a.detail = detail; a.K_out = K_out;
  a.P_out = P_out; a.flags = flags;
  if (ctx->poly_p > 0) { a.polyF = ctx->poly_dev; a.polyP = ctx->poly_p; }
  if (!lq_bounds_range_fused(ctx, a)) {
    // run-time dimensions or the dense route: one single-horizon launch per N (K_out / P_out from the first)
    const int NF = (int)lq::BF_COUNT;
    for (int N = N_min; N <= N_max; ++N) {
      const int64_t h = N - N_min;
      const int rc = lqmpc_bounds_batch(
          ctx, S, dA, dB, N, e_A, e_B, e_A_scalar, e_B_scalar, M_V ? M_V + h * S : nullptr, M_V_scalar, x_shared, x,
          K_in, K_shared, p3_host, V_expert, bar_u, bar_d_u, strict_reference, alpha ? alpha + h * S : nullptr,
          beta ? beta + h * S : nullptr, xi ? xi + h * S : nullptr, eta ? eta + h * S : nullptr,
          bound ? bound + h * S : nullptr, detail ? detail + h * NF * S : nullptr, h == 0 ? K_out : nullptr,
          h == 0 ? P_out : nullptr, flags ? flags + h * S : nullptr);
      if (rc) return rc;
    }
    return LQMPC_OK;
  }
  return lq_launch_bounds_range(ctx, a);
}

int lqmpc_dlqr_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, double* K_out, double* P_out,
                     int32_t* flags) {
  if (!ctx) return LQMPC_EINVAL;
  if (!ctx->has_problem) return lq_set_error(ctx, LQMPC_ESTATE, "problem not set");
  if (S < 0) return lq_set_error(ctx, LQMPC_EINVAL, "bad S");
  if (S == 0) return LQMPC_OK;
  cudaSetDevice(ctx->device);
  return ctx->dyn ? lq_dyn_dlqr(ctx, S, dA, dB, K_out, P_out, flags)
                  : lq_launch_dlqr(ctx, S, dA, dB, K_out, P_out, flags);
}

int lqmpc_column_stats(lqmpc_ctx* ctx, const double* table, int cols, int64_t S, int64_t ld, double* stats) {
  if (!ctx) return LQMPC_EINVAL;
  if (!table || !stats || cols < 1 || S < 0 || ld < S) return lq_set_error(ctx, LQMPC_EINVAL, "bad table/cols/S/ld");
  if (cols > 65535) return lq_set_error(ctx, LQMPC_EINVAL, "too many columns");
  cudaSetDevice(ctx->device);
  return lq_launch_stats(ctx, table, cols, S, ld, stats);
}

int lqmpc_column_sqdev(lqmpc_ctx* ctx, const double* table, int cols, int64_t S, int64_t ld, const double* mean,
                       double* sqdev) {
  if (!ctx) return LQMPC_EINVAL;
  if (!table || !mean || !sqdev || cols < 1 || S < 0 || ld < S)
    return lq_set_error(ctx, LQMPC_EINVAL, "bad table/cols/S/ld");
  if (cols > 65535) return lq_set_error(ctx, LQMPC_EINVAL, "too many columns");
  cudaSetDevice(ctx->device);
  return lq_launch_sqdev(ctx, table, cols, S, ld, mean, sqdev);
}

int lqmpc_column_moments(lqmpc_ctx* ctx, const double* table, int cols, int64_t S, int64_t ld, double* moments) {
  if (!ctx) return LQMPC_EINVAL;
  if (!table || !moments || cols < 1 || S < 0 || ld < S)
    return lq_set_error(ctx, LQMPC_EINVAL, "bad table/cols/S/ld");
  if (cols > 65535) return lq_set_error(ctx, LQMPC_EINVAL, "too many columns");
  cudaSetDevice(ctx->device);
  return lq_launch_moments(ctx, table, cols, S, ld, moments);
}

int lqmpc_column_radix_histogram(lqmpc_ctx* ctx, const double* table, int cols, int64_t S, int64_t ld, int nsel,
                                 int pass, const uint64_t* prefix, int64_t* hist) {
  if (!ctx) return LQMPC_EINVAL;
  if ((!table && S > 0) || !prefix || !hist || cols < 1 || S < 0 || ld < S)
    return lq_set_error(ctx, LQMPC_EINVAL, "bad table/cols/S/ld/prefix/hist");
  if (cols > 65535) return lq_set_error(ctx, LQMPC_EINVAL, "too many columns");
  if (nsel < 1 || nsel > LQMPC_RADIX_MAX_SEL) return lq_set_error(ctx, LQMPC_EINVAL, "nsel outside 1..32");
  if (pass < 0 || pass > 7) return lq_set_error(ctx, LQMPC_EINVAL, "pass outside 0..7");
  cudaSetDevice(ctx->device);
  return lq_launch_radix_hist(ctx, table, cols, S, ld, nsel, pass, prefix, hist);
}

int lqmpc_column_radix_select(lqmpc_ctx* ctx, const int64_t* hist, int cols, int nsel, int pass, int64_t* rank,
                              uint64_t* prefix) {
  if (!ctx) return LQMPC_EINVAL;
  if (!hist || !rank || !prefix || cols < 1) return lq_set_error(ctx, LQMPC_EINVAL, "bad hist/rank/prefix/cols");
  if (nsel < 1 || nsel > LQMPC_RADIX_MAX_SEL) return lq_set_error(ctx, LQMPC_EINVAL, "nsel outside 1..32");
  if (pass < 0 || pass > 7) return lq_set_error(ctx, LQMPC_EINVAL, "pass outside 0..7");
  cudaSetDevice(ctx->device);
  return lq_launch_radix_select(ctx, hist, cols, nsel, pass, rank, prefix);
}

int lqmpc_column_argext(lqmpc_ctx* ctx, const double* table, int cols, int64_t S, int64_t ld, int64_t index_base,
                        double* val, int64_t* idx) {
  if (!ctx) return LQMPC_EINVAL;
  if ((!table && S > 0) || !val || !idx || cols < 1 || S < 0 || ld < S)
    return lq_set_error(ctx, LQMPC_EINVAL, "bad table/cols/S/ld/val/idx");
  if (cols > 65535) return lq_set_error(ctx, LQMPC_EINVAL, "too many columns");
  if (index_base < 0) return lq_set_error(ctx, LQMPC_EINVAL, "negative index_base");
  cudaSetDevice(ctx->device);
  return lq_launch_argext(ctx, table, cols, S, ld, index_base, val, idx);
}

int lqmpc_fp64_tensor_peak(lqmpc_ctx* ctx, double* tflops_out) {
  if (!ctx || !tflops_out) return LQMPC_EINVAL;
  cudaSetDevice(ctx->device);
  return lq_launch_dmma_peak(ctx, tflops_out);
}

int lqmpc_sample_error_grid(lqmpc_ctx* ctx, uint64_t seed, int which, int rows, int cols, int64_t N_sys,
                            int64_t j_first, int n_err, const double* levels_host, int64_t n_boundary, int norm_type,
                            double* out, int64_t* stats_host) {
  if (!ctx) return LQMPC_EINVAL;
  if (!levels_host || !out || rows < 1 || cols < 1 || N_sys < 0 || j_first < 0 || n_err < 1 || n_err > 65535 ||
      which < 0 || which > 15 || (norm_type != 0 && norm_type != 1))
    return lq_set_error(ctx, LQMPC_EINVAL, "bad sampler arguments");
  if (N_sys == 0) return LQMPC_OK;
  cudaSetDevice(ctx->device);
  return lq_launch_sampler(ctx, seed, which, rows, cols, N_sys, j_first, n_err, levels_host, n_boundary, norm_type,
                           out, stats_host);
}

int lqmpc_fp64_peak(lqmpc_ctx* ctx, double* tflops_out) {
  if (!ctx || !tflops_out) return LQMPC_EINVAL;
  cudaSetDevice(ctx->device);
  return lq_launch_fp64_peak(ctx, tflops_out);
}

}  // extern "C"
