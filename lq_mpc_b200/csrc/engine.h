// engine.h — internal (non-ABI) declarations shared by the kernel translation units and c_api.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/lqmpc_b200.h"
#include "riccati.cuh"

// (n, m) pairs every templated kernel is instantiated for. The thread-per-sample register design targets n <= 4;
// n = 6, 8 compile from the same templates (spilling to local memory) and are provided for completeness.
#define LQ_FOR_EACH_DIM(X) X(1, 1) X(2, 1) X(2, 2) X(3, 1) X(3, 2) X(3, 3) X(4, 1) X(4, 2) X(4, 4) X(6, 2) X(8, 2)
#define LQ_DIMS_STRING "1x1,2x1,2x2,3x1,3x2,3x3,4x1,4x2,4x4,6x2,8x2"
#define LQ_MAX_N 8
#define LQ_MAX_M 4

struct lqmpc_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  int n = 0, m = 0;
  bool has_problem = false;
  int N_opc = 0;
  // packed lq::Problem<n,m> (host copy of the device-prepared struct), passed by value to kernels
  alignas(16) unsigned char pb[sizeof(lq::Problem<LQ_MAX_N, LQ_MAX_M>)];
  void* pb_dev = nullptr;
  std::string err;
  int64_t launches = 0;
  // run-time-dimension route (k_dyn.cu): (n, m) without a register-resident instantiation
  bool dyn = false;
  void* dyn_dev = nullptr;              // device problem buffer (layout: k_dyn.cu DynLayout)
  std::vector<double> dyn_host;         // host mirror after the device preparation
  // tiled (large-n) problem: device doubles A | B | Q | R | Pt | Pexp, see k_tiled.cu
  int tn = 0, tm = 0;
  bool has_tiled = false;
  void* tiled_pb = nullptr;
  void* tiled_zero = nullptr;   // n*n + n*m + n zero doubles (problem preparation runs the kernel on dA = dB = 0)
  // shared references of the next mpc_solve / simulate calls (lqmpc_set_references); NULL = zeros
  double* ref_x = nullptr;
  double* ref_u = nullptr;
  int ref_ld = 0;
  // general input polytope F_u u <= 1 (lqmpc_set_input_polytope): device copy of the p x m rows; p = 0 -> the box
  double* poly_dev = nullptr;
  int poly_p = 0;
  // scratch (grown on demand)
  void* ws = nullptr;
  size_t ws_bytes = 0;
  // result tables of lqmpc_eval_seeded when the caller only wants the column moments (grown on demand)
  void* seed_buf = nullptr;
  size_t seed_bytes = 0;
  // host-pipeline resources
  cudaStream_t pipe_stream[2] = {nullptr, nullptr};
  cudaEvent_t pipe_done[2] = {nullptr, nullptr};
  void* pipe_buf[2] = {nullptr, nullptr};
  size_t pipe_bytes = 0;
  cudaEvent_t tp_ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // tiled host pipeline: h2d/comp/d2h x 2 slots
};

struct EvalArgs {
  int64_t S;         // samples in this launch
  int64_t ld;        // leading dimension (stride between consecutive elements) of every SoA operand
  const double* dA;
  const double* dB;
  const double* x0;
  int N_min, N_max, T;
  double* J;
  double* rho;
  double* ratio;
  double* Vn;
  double* JT;
  int32_t* flags;
  double* K0;
};

struct MpcArgs {
  int64_t S;
  const double* dA;   // [n*n][S] or NULL (zero perturbation)
  const double* dB;   // [n*m][S] or NULL
  int N, T;
  int N_min = 0;      // range launch (lq_launch_mpc_range): horizons N_min..N, outputs with a leading [H] axis
  int npts;
  const double* pts;  // shared initial states [npts][n] (device) or NULL
  const double* x0;   // per-sample initial states [n][S] (device), used when pts == NULL
  double* V;          // [P][S]
  double* u0;         // [P][m][S]
  double* M_V;        // [S]
  double* J_T;        // [S]
  double* X;          // [T+1][n][S]
  double* U;          // [T][m][S]
  int32_t* flags;     // solve: [P][S]; simulate: [S]
  int32_t* n_active;  // [S]
  double* ws;         // filled by the launcher
  const double* xr = nullptr;   // shared references (device, row-major [n][ref_ld] / [m][ref_ld]) or NULL = zeros
  const double* ur = nullptr;
  int ref_ld = 0;
  const double* polyF = nullptr;   // filled by the polytope launcher (device, row-major [p][m])
  int polyP = 0;
};

struct BoundsArgs {
  int64_t S;
  const double* dA;
  const double* dB;
  int N;
  int N_min = 0;          // range launch (lq_launch_bounds_range): horizons N_min..N, outputs with a leading [H] axis
  const double* eA;       // [S] or NULL -> eA_s
  const double* eB;
  double eA_s, eB_s;
  const double* MV;       // [S] or NULL -> MV_s
  double MV_s;
  const double* x_shared; // [n] or NULL -> x [n][S]
  const double* x;
  const double* K_in;     // [m*n][S] (u = +Kx) or NULL
  const double* K_shared; // [m*n] or NULL; both NULL -> -K_dlqr of the sample's model
  double p[3];
  double V_expert;
  double bar_u, bar_d_u;
  int strict;
  double *alpha, *beta, *xi, *eta, *bound;  // [S]
  double* detail;         // [BF_COUNT][S]
  double* K_out;          // [m*n][S]
  double* P_out;          // [n*n][S] (DARE solution; only when the gain is computed here)
  int32_t* flags;
  double* ws;
  int dense = 0;                  // force the dense Householder route (LQMPC_K3_DENSE; A/B tests)
  const double* polyF = nullptr;  // general input polytope rows (device, [p][m]) for local_radius, or NULL -> the box
  int polyP = 0;
};

struct TiledEval {
  int64_t S;
  const double* dA;   // [S][n*n] array of matrices
  const double* dB;   // [S][n*m]
  const double* x0;   // [S][n]
  int N_min, N_max;
  double* J;          // [H][S]  (any output may be NULL)
  double* rho;
  double* ratio;
  double* Vn;
  int32_t* flags;
  double* Pout;       // [n*n]: final cost-to-go of sample 0 (problem preparation only)
};

int lq_set_error(lqmpc_ctx* ctx, int code, const char* what);
int lq_check_cuda(lqmpc_ctx* ctx, cudaError_t e, const char* what);
int lq_reserve_ws(lqmpc_ctx* ctx, size_t bytes);

// launchers (one per kernel family; each switches on ctx->n, ctx->m)
int lq_launch_prepare(lqmpc_ctx* ctx);
int lq_launch_eval(lqmpc_ctx* ctx, const EvalArgs& a, cudaStream_t stream);
bool lq_group_supported(int n, int m);
int lq_launch_eval_group(lqmpc_ctx* ctx, const EvalArgs& a, cudaStream_t stream);
int lq_launch_eval_group_seeded(lqmpc_ctx* ctx, const EvalArgs& a, uint64_t seed, int64_t first, double e_A, double e_B);
int lq_launch_eval_seeded(lqmpc_ctx* ctx, const EvalArgs& a, uint64_t seed, int64_t first, double e_A, double e_B);
int lq_launch_fp64_peak(lqmpc_ctx* ctx, double* tflops);
int lq_launch_dmma_peak(lqmpc_ctx* ctx, double* tflops);
int lq_launch_mpc(lqmpc_ctx* ctx, const MpcArgs& a, bool simulate);
int lq_launch_mpc_poly(lqmpc_ctx* ctx, const MpcArgs& a, bool simulate);
int lq_launch_mpc_range(lqmpc_ctx* ctx, const MpcArgs& a);
int lq_launch_bounds(lqmpc_ctx* ctx, const BoundsArgs& a);
bool lq_bounds_range_fused(lqmpc_ctx* ctx, const BoundsArgs& a);
int lq_launch_bounds_range(lqmpc_ctx* ctx, const BoundsArgs& a);
int lq_launch_stats(lqmpc_ctx* ctx, const double* table, int cols, int64_t S, int64_t ld, double* stats);
int lq_launch_moments(lqmpc_ctx* ctx, const double* table, int cols, int64_t S, int64_t ld, double* out);
int lq_launch_sqdev(lqmpc_ctx* ctx, const double* table, int cols, int64_t S, int64_t ld, const double* mean,
                    double* out);
int lq_launch_radix_hist(lqmpc_ctx* ctx, const double* table, int cols, int64_t S, int64_t ld, int nsel, int pass,
                         const uint64_t* prefix, int64_t* hist);
int lq_launch_radix_select(lqmpc_ctx* ctx, const int64_t* hist, int cols, int nsel, int pass, int64_t* rank,
                           uint64_t* prefix);
int lq_launch_argext(lqmpc_ctx* ctx, const double* table, int cols, int64_t S, int64_t ld, int64_t index_base,
                     double* val, int64_t* idx);
bool lq_dyn_supported(int n, int m);
int lq_dyn_set_problem(lqmpc_ctx* ctx, const double* A, const double* B, const double* Q, const double* R,
                       const double* P, const double* lo, const double* hi);
int lq_dyn_get_prepared(lqmpc_ctx* ctx, double* out);
int lq_dyn_eval(lqmpc_ctx* ctx, const EvalArgs& a, cudaStream_t stream);
int lq_dyn_mpc(lqmpc_ctx* ctx, MpcArgs a, bool simulate);
int lq_dyn_bounds(lqmpc_ctx* ctx, const BoundsArgs& a);
int lq_dyn_dlqr(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, double* K, double* P, int32_t* flags);
bool lq_tiled_supported(int n, int m);
size_t lq_tiled_pb_doubles(int n, int m);
int lq_launch_tiled(lqmpc_ctx* ctx, const TiledEval& t);
int lq_launch_sampler(lqmpc_ctx* ctx, uint64_t seed, int which, int rows, int cols, int64_t N_sys, int64_t j_first,
                      int n_err, const double* levels_host, int64_t n_boundary, int norm_type, double* out,
                      int64_t* stats_host);
int lq_launch_dlqr(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, double* K, double* P,
                   int32_t* flags);
