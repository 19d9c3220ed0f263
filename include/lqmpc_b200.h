/* lqmpc_b200.h — C ABI of the B200-native batch engine for the lq_mpc hot path.
 *
 * The reference (lcrekko/lq_mpc) has no FFI/plugin boundary: its boundary is its Python surface
 * (utils_class.py / utils.py).  Each entry point below is the *batched* replacement of the per-sample reference
 * call it cites; `lq_mpc_b200/utils_class.py` and `lq_mpc_b200/utils.py` keep the reference's class and function
 * signatures and bind these symbols through ctypes (see INTEGRATION.md for the stub a maintainer would add).
 *
 * Conventions
 *   - plain C, no torch types; every pointer is a DEVICE pointer to FP64 data unless the name ends in `_host`.
 *   - batched operands are struct-of-arrays: element e of sample s lives at  ptr[e * S + s]  (row-major element
 *     order inside a matrix, e = i*cols + j), so a warp reads 32 consecutive samples of one element: coalesced.
 *   - all work is enqueued on the context's CUDA stream; nothing synchronises unless stated.
 *   - return value: 0 on success, negative LQMPC_E* on error (never throws); lqmpc_last_error() gives the text.
 *   - there is NO CPU path: every function fails with LQMPC_ENODEVICE when no CUDA device is usable.
 *   - a context is not thread-safe; distinct contexts are independent.
 */
#ifndef LQMPC_B200_H
#define LQMPC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LQMPC_OK 0
#define LQMPC_EINVAL (-1)     /* bad argument / unsupported size        */
#define LQMPC_ENODEVICE (-2)  /* no usable CUDA device                  */
#define LQMPC_ECUDA (-3)      /* a CUDA runtime call failed             */
#define LQMPC_ESTATE (-4)     /* problem not set                        */

/* per-eval status bits written to the int32 `flags` outputs */
#define LQMPC_FLAG_UNSTABLE 1
#define LQMPC_FLAG_QP_ACTIVE 2
#define LQMPC_FLAG_QP_MAXITER 4
#define LQMPC_FLAG_DARE_NOCONV 8
#define LQMPC_FLAG_NONFINITE 16
#define LQMPC_FLAG_BOUND_INVALID 32
#define LQMPC_FLAG_LYAP_NOCONV 64
#define LQMPC_FLAG_EIG_NOCONV 128
#define LQMPC_FLAG_CHOL_FAIL 256
#define LQMPC_FLAG_DOMAIN_ERROR 512
#define LQMPC_FLAG_TAIL_UNCERTIFIED 1024
#define LQMPC_FLAG_ASCENT_MAXITER 2048

typedef struct lqmpc_ctx lqmpc_ctx;

/* ABI version (bumped on any signature change) and the list of compiled (n, m) pairs, e.g. "2x1,4x2". */
int lqmpc_abi_version(void);
const char* lqmpc_supported_dims(void);

/* One context per (device, stream). `cuda_stream` is a cudaStream_t (NULL = the legacy default stream). */
int lqmpc_create(lqmpc_ctx** out, int device, void* cuda_stream);
void lqmpc_destroy(lqmpc_ctx* ctx);
const char* lqmpc_last_error(const lqmpc_ctx* ctx);
int lqmpc_sync(lqmpc_ctx* ctx);

/* Problem data shared by every sample (HOST pointers, row-major FP64): the TRUE plant (A n x n, B n x m), the
 * stage weights Q, R, the terminal weight P (every reference caller passes P = Q), the input box u_lo <= u <= u_hi
 * (both NULL: unconstrained) and N_opc, the horizon of the expert open-loop cost V_expert (<=0: DARE limit).
 * Replaces the constructor arguments of LQ_MPC_Controller / LQ_MPC_Simulator / LQ_RDP_Calculator /
 * LQ_RDP_Behavior_Multiple (utils_class.py:23, 218, 293, 691-764). The derived constants (Q^-1, eigenvalue
 * extremes, V_expert's matrix) are computed ON THE DEVICE by a one-thread preparation kernel. */
int lqmpc_set_problem(lqmpc_ctx* ctx, int n, int m, const double* A_true_host, const double* B_true_host,
                      const double* Q_host, const double* R_host, const double* P_term_host,
                      const double* u_lo_host, const double* u_hi_host, int N_opc);

/* Copy the device-prepared constants back: Pexp (n*n), then Qinv (n*n), then maxQ,minQ,maxR,minR. Synchronises. */
int lqmpc_get_prepared(lqmpc_ctx* ctx, double* out_host, int64_t capacity);

/* K1 — unconstrained certainty-equivalent MPC evaluation, nested horizons N_min..N_max (H = N_max-N_min+1 columns).
 * Per (sample s, horizon N): Riccati gain K_0 on (A+dA_s, B+dB_s); closed loop A_cl = A + B K_0 on the true plant;
 * rho(A_cl); J_inf = x0' S x0 (Lyapunov squared doubling; +inf and LQMPC_FLAG_UNSTABLE if rho >= 1);
 * ratio = J_inf / V_expert(x0); optionally J_T (T > 0; the finite sum of utils_class.py:261,282-283), the open-loop
 * value V_N = x0' P_0 x0 (utils_class.py:91) and the gain itself.
 * Replaces, for the unconstrained law, LQ_MPC_Controller.solve (utils_class.py:48-91) +
 * LQ_MPC_Simulator.simulate (utils_class.py:245-285) inside the sweep loops (utils_class.py:802-833, 886-916).
 *   dA [n*n][S], dB [n*m][S], x0 [n][S]            inputs
 *   J, rho, ratio, V_N, J_T : [H][S] (any may be NULL; J_T requires T > 0), flags [H][S] int32 (may be NULL),
 *   K0 [H][m*n][S] (may be NULL) */
int lqmpc_eval_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, const double* x0, int N_min,
                     int N_max, int T, double* J, double* rho, double* ratio, double* V_N, double* J_T,
                     int32_t* flags, double* K0);

/* Same evaluation on SEEDED SYNTHETIC samples drawn inside the kernel (no operand traffic): global sample s in
 * [first, first + S) draws dA, dB entrywise uniform in [-e_A, e_A) / [-e_B, e_B) and x0 ~ N(0, I) from Philox4x32-10
 * keyed by `seed` with the counter (s, pair index) — the stream of BASELINE's synthetic configurations (SURVEY 8d.4:
 * "Philox ... with sample index as counter so every shard size sees identical samples"), restated bit-for-bit
 * (uniforms) in oracle/np_sampler.seeded_samples. Replaces the host-side generation + upload in front of the sweep
 * loops (utils_class.py:802-833 on error_matrix_generator output, utils.py:826-847) for synthetic studies.
 *   J, rho, ratio [H][S], flags [H][S] int32 : device, any may be NULL
 *   moments [3 H][6] device or NULL : the one-pass column moments (see lqmpc_column_moments) of the [3 H][S] table
 *     {J rows, rho rows, ratio rows}; then J/rho/ratio must be that one contiguous table, or all NULL (the tables then
 *     live in the context's scratch and only the moments leave the call). */
int lqmpc_eval_seeded(lqmpc_ctx* ctx, uint64_t seed, int64_t first, int64_t S, double e_A, double e_B, int N_min,
                      int N_max, double* J, double* rho, double* ratio, int32_t* flags, double* moments);

/* Same computation driven from HOST buffers (pinned or pageable): the batch is cut into chunks that are copied
 * H2D, evaluated and copied back D2H on alternating streams so copies overlap compute. All pointers are HOST
 * pointers with the same SoA layout over the full S. Synchronises before returning. This is the call `bench.py`
 * times for the end-to-end figure. */
int lqmpc_eval_batch_host(lqmpc_ctx* ctx, int64_t S, const double* dA_host, const double* dB_host,
                          const double* x0_host, int N_min, int N_max, int T, double* J_host, double* rho_host,
                          double* ratio_host, int32_t* flags_host, int64_t chunk);

/* K4 — the same evaluation for LARGER state dimensions (compiled: n x m = 32 x 8 — BASELINE cfg 5 — and 16 x 4),
 * unconstrained law. One CTA per sample; the sample's operands are staged into shared memory by TMA bulk copies, so
 * this path takes ARRAY-OF-MATRICES operands (one sample contiguous, 16-byte aligned):
 *   dA [S][n*n], dB [S][n*m], x0 [S][n]   inputs (device)
 *   J, rho, ratio, V_N : [H][S] (any may be NULL), flags [H][S] int32 (may be NULL)
 * lqmpc_set_problem_tiled installs (A, B, Q, R, P, N_opc) (host pointers, row-major) and prepares the expert cost
 * matrix on the device with the evaluation kernel itself; lqmpc_get_prepared_tiled copies it back (n*n doubles).
 * Nested horizons (N_min < N_max) need the whole batch to fit one 4 GiB closed-loop scratch chunk. */
int lqmpc_set_problem_tiled(lqmpc_ctx* ctx, int n, int m, const double* A_true_host, const double* B_true_host,
                            const double* Q_host, const double* R_host, const double* P_term_host, int N_opc);
int lqmpc_get_prepared_tiled(lqmpc_ctx* ctx, double* Pexp_host, int64_t capacity);
int lqmpc_eval_batch_tiled(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, const double* x0, int N_min,
                           int N_max, double* J, double* rho, double* ratio, double* V_N, int32_t* flags);

/* Same from HOST buffers (array-of-matrices, ideally pinned; outputs [H][S] on the host): chunks are copied H2D,
 * evaluated and copied back on three streams so that PCIe traffic overlaps the kernels. `chunk` (<= 0: 16 384) is the
 * LARGEST chunk: sizes ramp up from chunk / 8 by 11/8 per chunk so that only a small first copy is exposed. Synchronises. */
int lqmpc_eval_batch_tiled_host(lqmpc_ctx* ctx, int64_t S, const double* dA_host, const double* dB_host,
                                const double* x0_host, int N_min, int N_max, double* J_host, double* rho_host,
                                double* ratio_host, int32_t* flags_host, int64_t chunk);

/* K2a — batched LQ_MPC_Controller.solve (utils_class.py:48-91) with the input box of lqmpc_set_problem, zero
 * references, terminal weight P: for every sample the controller model is (A+dA_s, B+dB_s) (dA/dB NULL = the true
 * model, e.g. for V_expert, utils_class.py:786). The QP is solved EXACTLY (Riccati-structured primal active set).
 * Initial states: either `pts` — npts states shared by all samples, device [npts][n] (the ring of
 * OL_energy_bound, utils_class.py:439-466) — or `x0`, one state per sample, device [n][S] (then P = 1).
 *   V [P][S] open-loop value V_N (incl. x0'Qx0), u0 [P][m][S] first input, M_V [S] = max_p V (utils_class.py:464),
 *   flags [P][S]; any output may be NULL. Needs N*m <= 256 (N*p <= 256 with an input polytope of p rows)
 *   whenever a constraint is active; beyond that the entry is flagged LQMPC_FLAG_QP_MAXITER, never approximated:
 *   its V is NaN and its u0 the unconstrained first input clipped into the input set. */
int lqmpc_mpc_solve_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, int N, int npts,
                          const double* pts, const double* x0, double* V, double* u0, double* M_V, int32_t* flags);

/* Shared references for the following lqmpc_mpc_solve_batch / lqmpc_simulate_batch calls (utils_class.py:48-81:
 * x_ref[:, i] is the reference of x_{i+1}, u_ref[:, i] of u_i; HOST pointers, row-major (n x n_cols), (m x n_cols),
 * n_cols >= N of the calls that follow; either may be NULL = zeros). n_cols <= 0 or both NULL clears them (the state
 * after lqmpc_set_problem). Non-zero references make the law affine: the exact solver then skips the Riccati fast
 * path. The bound kernels (K3) and K1/K4 are regulation-only, as every caller in the reference is. Synchronises. */
int lqmpc_set_references(lqmpc_ctx* ctx, int n_cols, const double* x_ref_host, const double* u_ref_host);

/* General input polytope F_u u <= 1 (utils_class.py:23,81: F_u is an arbitrary p x m matrix; rows with several
 * non-zeros couple the inputs) for the following lqmpc_mpc_solve_batch / lqmpc_simulate_batch / lqmpc_bounds_batch
 * calls: HOST pointer, row-major (p x m), p <= 12, N * p <= 256 per solve. p <= 0 or NULL clears it (back to the box of
 * lqmpc_set_problem, the state after lqmpc_set_problem). The origin must be interior (it is: the right-hand side is 1).
 * With a polytope installed lqmpc_bounds_batch takes local_radius (utils.py:548-564) over these rows and needs bar_u /
 * bar_d_u (utils.py:592-650: maxima of convex functions, attained at vertices) from the caller. A rejected call
 * (too many rows, non-finite entry) leaves the installed constraint set as it was. Synchronises. */
int lqmpc_set_input_polytope(lqmpc_ctx* ctx, int p, const double* F_u_host);

/* K2b — batched LQ_MPC_Simulator.simulate (utils_class.py:245-285): T receding-horizon steps, the controller plans
 * with (A+dA_s, B+dB_s) and horizon N, the plant is the TRUE model; J_T as accumulated at utils_class.py:261,282-283.
 * Initial state: `x0_shared` device [n] (one state for all samples) or `x0` device [n][S].
 *   J_T [S], X [T+1][n][S], U [T][m][S], flags [S], n_active [S] (steps whose QP had an active bound); NULL = skip. */
int lqmpc_simulate_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, int N, int T,
                         const double* x0_shared, const double* x0, double* J_T, double* X, double* U,
                         int32_t* flags, int32_t* n_active);

/* K2c — infinite-horizon cost of the K2b closed loop, J_inf = lim_{T->inf} J_T, exact (no truncation) and certified.
 * Inside the feasibility ellipsoid {x' P0 x <= c*} of the unconstrained N-stage plan the exact QP returns u = K0 x, so
 * from there on the TRUE closed loop A + B K0 has cost matrix S = W + (A + B K0)' S (A + B K0), W = Q + K0' R K0. The
 * level set {x' S x <= c_S}, c_S = (1 - 1e-9) c* / lambda_max(L^-1 P0 L^-T) (S = L L'), is invariant and lies inside
 * the ellipsoid. The closed loop runs with the exact QP (box or installed polytope) until the first step tau <= T_max
 * whose state is in that set: J_inf = sum_{t<tau} (x_t'Q x_t + u_t'R u_t) + x_tau' S x_tau.
 *   J_inf [S], T_cert [S] (= tau), flags [S]: the OR of the plan, every step's solve, the tail and the bits below;
 *   NULL = skip. Initial state as lqmpc_simulate_batch.
 *   rho(A + B K0) >= 1: J_inf = +inf, T_cert = -1, LQMPC_FLAG_UNSTABLE (K1's convention; no simulation).
 *   No certificate within T_max steps, or S not obtained / not positive definite (LQMPC_FLAG_LYAP_NOCONV where the
 *   Lyapunov solve failed): J_inf = NaN, T_cert = -1, LQMPC_FLAG_TAIL_UNCERTIFIED. The certificate is sufficient, not
 *   necessary: "uncertified" is no verdict of instability.
 *   Without input bounds c* = +inf: T_cert = 0 and J_inf = x0' S x0, K1's J for the same horizon.
 * Regulation only: LQMPC_EINVAL with references installed (the state does not converge to the origin), for
 * T_max < 0, and unless exactly one of x0_shared / x0 is given. Not available on the tiled (n = 16 / 32) route. */
int lqmpc_simulate_inf_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, int N, int T_max,
                             const double* x0_shared, const double* x0, double* J_inf, int32_t* T_cert,
                             int32_t* flags);

/* Worst-case model error of the unconstrained law (K1's J_inf at one horizon N). One sample per thread, every compiled
 * (n, m) pair; the input box, an installed polytope and references do not enter (as lqmpc_eval_batch).
 * dA [n*n][S], dB [n*m][S], x0 [n][S] (device, SoA). LQMPC_ESTATE without a problem; LQMPC_EINVAL on the
 * run-time-dimension route, on a tiled-only context and for N < 1; S = 0 returns OK and launches nothing.
 *
 * lqmpc_eval_grad_batch: J, rho, ratio [S] as lqmpc_eval_batch (N_min = N_max = N; here J comes from Lyapunov doubling)
 * and the exact gradient gA = dJ/d(dA) [n*n][S], gB = dJ/d(dB) [n*m][S] by the adjoint of the Riccati recursion and the
 * closed loop (csrc/worst.cuh), O(N n^3) per sample. Unstable (J = +inf, LQMPC_FLAG_UNSTABLE) and failed entries
 * (LQMPC_FLAG_CHOL_FAIL, _LYAP_NOCONV, _EIG_NOCONV, _NONFINITE) have NaN gradients. Any output may be NULL. */
int lqmpc_eval_grad_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, const double* x0, int N,
                          double* J, double* rho, double* ratio, double* gA, double* gB, int32_t* flags);

/* lqmpc_worst_case_batch: projected ascent of J from every sample over {||dA|| <= e_A, ||dB|| <= e_B}, each block
 * separately; norm_type 0 = Frobenius, 1 = spectral, 2 = entrywise max. In u = (dA / e_A, dB / e_B) with gradient
 * g = (e_A dJ/d(dA), e_B dJ/d(dB)): the start is projected onto the set; the ascent stops when the stationarity residual
 * r = ||Proj(u + g/||g||) - u||_2 <= tol (r = 0 when g = 0); trial steps u+ = Proj(u + t g) take t = 0.5 / ||g|| first,
 * then the Barzilai-Borwein step s's / (-s'y) when s'y < 0 and 10 t otherwise, and are accepted when
 * J(u+) >= J(u) + 1e-4 g.(u+ - u), else t <- t / 4. A block with e = 0 stays zero. J never decreases from the projected
 * start's value.
 *   dA_out [n*n][S], dB_out [n*m][S]: the final perturbation (may alias dA / dB); J, rho, ratio [S]; iters [S] (accepted
 *   steps); flags [S]. Any output may be NULL.
 *   An unstable trial lies in the set and destabilises the loop: it is returned, J = +inf, LQMPC_FLAG_UNSTABLE. A trial
 *   with another failure flag is rejected; a start with one is returned as it is. LQMPC_FLAG_ASCENT_MAXITER: max_iter
 *   accepted steps (or a line search that shrank t by 4^60) without r <= tol.
 * LQMPC_EINVAL besides the above: e_A / e_B negative or not finite, unknown norm_type, max_iter < 0, tol <= 0. */
int lqmpc_worst_case_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, const double* x0, int N,
                           double e_A, double e_B, int norm_type, int max_iter, double tol, double* dA_out,
                           double* dB_out, double* J, double* rho, double* ratio, int32_t* iters, int32_t* flags);

/* Worst case over every initial state. For a given model error the performance ratio J_inf(x0) / V_expert(x0) =
 * x0'S x0 / x0'P_exp x0 (S the closed-loop cost matrix S = W + A_cl'S A_cl, P_exp the expert matrix) is a Rayleigh
 * quotient, so its supremum over x0 != 0 is
 *   gamma(dA, dB) = lambda_max(L^-1 S L^-T),  P_exp = L L',
 * attained at x_worst = L^-T w (w the top eigenvector), normalised to x_worst'P_exp x_worst = 1 with its entry of
 * largest magnitude positive (ties to the lowest index). Same scope, operands and validation as the two calls above,
 * without x0: LQMPC_ESTATE without a problem; LQMPC_EINVAL on the run-time-dimension route, on a tiled-only context,
 * for N < 1 and for null inputs; S = 0 returns OK and launches nothing. Every output may be NULL.
 *
 * lqmpc_ratio_sup_batch: gamma, x_worst [n][S], the relative eigengap gap = (lambda_1 - lambda_2) / lambda_1 [S] (1 at
 * n = 1), rho [S], flags [S], and with gA / gB non-NULL the gradient gA = dgamma/d(dA) [n*n][S], gB = dgamma/d(dB)
 * [n*m][S] (x_worst'(dS)x_worst by the adjoint of lqmpc_eval_grad_batch at x0 = x_worst). The gradient is exact
 * where lambda_max is simple; as gap -> 0 gamma has a kink and the gradient is that of one branch. A call without gA
 * and gB computes the value only. Unstable: gamma = +inf, x_worst, gap and the gradient NaN, LQMPC_FLAG_UNSTABLE;
 * LQMPC_FLAG_CHOL_FAIL, _LYAP_NOCONV, _NONFINITE as lqmpc_eval_grad_batch; _EIG_NOCONV also when the Jacobi
 * eigensolver misses its off-diagonal tolerance.
 *
 * lqmpc_worst_case_sup_batch: the projected ascent of lqmpc_worst_case_batch (same e_A, e_B, norm_type, max_iter, tol,
 * checks and stopping rule) with gamma in place of J, i.e. the joint ascent over (dA, dB, x0) of J / V_expert. Outputs
 * dA_out / dB_out (may alias dA / dB), gamma, x_worst, rho, iters, flags at the final point. The result is a stationary
 * point of gamma on the error set (a local maximum in general, or an error that destabilises the loop), not a
 * certified global maximum. */
int lqmpc_ratio_sup_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, int N, double* gamma,
                          double* x_worst, double* gap, double* rho, double* gA, double* gB, int32_t* flags);
int lqmpc_worst_case_sup_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, int N, double e_A,
                               double e_B, int norm_type, int max_iter, double tol, double* dA_out, double* dB_out,
                               double* gamma, double* x_worst, double* rho, int32_t* iters, int32_t* flags);

/* Worst-case model error of the input-constrained closed loop: K2c's certified J_inf (lqmpc_simulate_inf_batch, input
 * box of lqmpc_set_problem, regulation) at one horizon N,
 *   J_inf = sum_{t<tau} (x_t'Q x_t + u_t'R u_t) + x_tau'S x_tau,  u_t = QP_N(x_t; A+dA, B+dB)_0,  x_{t+1} = A x_t + B u_t,
 * with S = W + A_cl'S A_cl, A_cl = A + B K0, K0 the unconstrained horizon-N gain of the model. J_inf is continuous in
 * (dA, dB) and smooth wherever every pre-certificate QP is strictly complementary. One sample per thread, every compiled
 * (n, m) pair. dA [n*n][S], dB [n*m][S] (device, SoA); the initial state as lqmpc_simulate_batch: x0_shared [n] or x0
 * [n][S], exactly one. LQMPC_ESTATE without a problem; LQMPC_EINVAL with references or an input polytope installed, on
 * the run-time-dimension route, on a tiled-only context, for N < 1, T_max < 0 and null dA / dB; S = 0 returns OK and
 * launches nothing. Every output may be NULL. The per-thread workspace grows with T_max: the gradient and the ascent
 * keep the closed-loop states x_0..x_tau, (T_max + 1) n doubles per resident thread, besides O(N (n^2 + n m)) for
 * the solver, the Riccati stage records and the QP plans.
 *
 * lqmpc_simulate_inf_grad_batch: J_inf, T_cert, flags [S] as lqmpc_simulate_inf_batch (the same code computes them),
 * rho [S] = rho(A + B K0), and with gA / gB non-NULL the gradient gA = dJ_inf/d(dA) [n*n][S], gB = dJ_inf/d(dB)
 * [n*m][S] by one reverse pass over the steps t < tau. With lambda_tau = 2 S x_tau and c = 2 R u_t + B'lambda:
 *   a step that took the unconstrained law adds c x_t' to Kbar = dJ/dK0 and sets lambda <- 2 Q x_t + A'lambda + K0'c;
 *   a step with an active bound sets lambda <- 2 Q x_t + A'lambda + Kc0'c (Kc0 the stage-0 gain of the QP's final
 *   working set) and adds the implicit-function vector-Jacobian product of c'u_t in (A+dA, B+dB), from the adjoint LQ
 *   of that working set;
 *   the tail adds 2 (R K0 + B'S A_cl) Lambda, Lambda = x_tau x_tau' + A_cl Lambda A_cl', to Kbar, which the adjoint of
 *   the Riccati recursion (lqmpc_eval_grad_batch's) maps to (gA, gB).
 * The gradient is exact where every pre-certificate solve is strictly complementary; elsewhere it is the gradient for
 * the active sets the solver found. It is NaN where J_inf is +inf or NaN or any of LQMPC_FLAG_CHOL_FAIL, _LYAP_NOCONV,
 * _EIG_NOCONV, _NONFINITE, _QP_MAXITER, _TAIL_UNCERTIFIED is set. A call without gA and gB computes the value only.
 *
 * lqmpc_worst_case_inf_batch: the projected ascent of lqmpc_worst_case_batch (same e_A, e_B, norm_type, max_iter, tol,
 * checks and stopping rule) on this J_inf. A trial with any of the flags above is rejected and a start with one is
 * returned as it is; an unstable trial is the result (J_inf = +inf, T_cert = -1, LQMPC_FLAG_UNSTABLE). Outputs dA_out /
 * dB_out (may alias dA / dB), J_inf, T_cert, rho, iters, flags at the final point. The result is a stationary point of
 * J_inf on the error set (or an error that destabilises the loop), not a certified global maximum. */
int lqmpc_simulate_inf_grad_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, int N, int T_max,
                                  const double* x0_shared, const double* x0, double* J_inf, int32_t* T_cert,
                                  double* rho, double* gA, double* gB, int32_t* flags);
int lqmpc_worst_case_inf_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, int N, int T_max,
                               const double* x0_shared, const double* x0, double e_A, double e_B, int norm_type,
                               int max_iter, double tol, double* dA_out, double* dB_out, double* J_inf,
                               int32_t* T_cert, double* rho, int32_t* iters, int32_t* flags);

/* K3 — batched bound coefficients: LQ_RDP_Calculator.energy_decreasing (utils_class.py:344-373) and
 * .energy_bound (utils_class.py:308-342) with every helper they call (utils.py: local_radius, ex_stability_lq,
 * ex_stability_bounds, fc_omega_eta, fc_ec_h, fc_ec_E, fc_ec_theta, fc_ec_g_*, geo_M, my_eigen, sl_syn_*,
 * bar_u_solve, bar_d_u_solve) and the final J_bound = (alpha V_expert + beta)/(1 - xi - eta)
 * (utils_class.py:858-859), for the estimated model (A+dA_s, B+dB_s) of every sample.
 *   N                      horizon of this launch
 *   e_A, e_B               device [S] (per-sample error level) or NULL -> the scalar arguments
 *   M_V                    device [S] (from lqmpc_mpc_solve_batch) or NULL -> M_V_scalar
 *   x_shared / x           the state energy_bound is evaluated at: device [n] shared, or device [n][S]
 *   K_in / K_shared        terminal gain in the u = +K x convention: device [m*n][S], or device [m*n] shared;
 *                          both NULL: -K_dlqr of the sample's own model (DARE solved in-kernel, utils_class.py:840-844)
 *   p3_host                the three scalars p (HOST), V_expert (utils_class.py:786)
 *   bar_u, bar_d_u         max||u||^2, max||u1-u2||^2 over the input set; negative = derive from the box
 *   strict_reference       keep the literal kron(Q, I) / kron(R, I) ordering of utils.py:317-318 (immaterial when
 *                          Q and R are multiples of the identity)
 * Outputs (device, any may be NULL): alpha, beta, xi, eta, bound [S]; detail [lqmpc_bounds_fields()][S] with every
 * intermediate in the order of `enum BoundField` (bounds.cuh; mirrored in lq_mpc_b200/engine.py); K_out [m*n][S];
 * P_out [n*n][S] (DARE solution, only when the gain is computed in-kernel); flags [S].
 * A reference ValueError (math.log / math.sqrt domain, utils.py:506-507,514) maps to LQMPC_FLAG_DOMAIN_ERROR;
 * 1 - xi - eta <= 0 (void bound, computed silently by the reference) sets LQMPC_FLAG_BOUND_INVALID. */
int lqmpc_bounds_fields(void);
int lqmpc_bounds_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, int N, const double* e_A,
                       const double* e_B, double e_A_scalar, double e_B_scalar, const double* M_V,
                       double M_V_scalar, const double* x_shared, const double* x, const double* K_in,
                       const double* K_shared, const double* p3_host, double V_expert, double bar_u, double bar_d_u,
                       int strict_reference, double* alpha, double* beta, double* xi, double* eta, double* bound,
                       double* detail, double* K_out, double* P_out, int32_t* flags);

/* Horizon-range forms of K2a and K3: the same computation as lqmpc_mpc_solve_batch / lqmpc_bounds_batch for every
 * horizon N_min..N_max (H = N_max - N_min + 1), in one call, results stacked on a leading [H] axis (slot h = N - N_min).
 *   lqmpc_mpc_solve_range: V [H][P][S], u0 [H][P][m][S], M_V [H][S], flags [H][P][S]; any output may be NULL.
 *     Fused for the compiled (n, m) pairs with the input box and zero references: ONE unconstrained Riccati sweep of
 *     N_max stages per sample serves every horizon (the law of horizon N at stage k is the sweep's stage
 *     k + N_max - N), and the results are bit-identical to H single-horizon calls.
 *   lqmpc_bounds_range: the arguments of lqmpc_bounds_batch with N_min, N_max for N; M_V [H][S] (or NULL ->
 *     M_V_scalar); alpha, beta, xi, eta, bound, flags [H][S]; detail [H][lqmpc_bounds_fields()][S] (each horizon's
 *     block has the single-horizon layout); K_out [m*n][S] and P_out [n*n][S] once (they do not depend on N).
 *     Fused for the compiled (n, m) pairs with n <= 6 on the matrix-free route (scalar weights or
 *     strict_reference = 0, with or without an input polytope, K_in / K_shared or the in-kernel DARE): the
 *     horizon-independent part once per sample, the Gram-spectrum bisections of all horizons sharing their probes,
 *     the error-consistent sums extended term by term. ||Gamma||^2 and lambda_min(H^) agree with
 *     lqmpc_bounds_batch to the bisection tolerance 2^-42 of both searches, the fields computed from them to a few
 *     times that; the others are the same formulas, which the compiler may contract into FMAs differently in the two
 *     kernels (last-bit differences). bound = (alpha V_expert + beta) / (1 - xi - eta) magnifies these by
 *     1 / |1 - xi - eta| where that denominator is near 0 (a bound at the edge of validity). Flags, K_out and P_out
 *     are equal.
 * Every other case — the run-time-dimension route, an installed input polytope or references (solve), the dense
 * route of K3 (literal kron with non-scalar weights, LQMPC_K3_DENSE), K3 at n = 8 (measured faster per horizon) — is
 * answered by one single-horizon call per N
 * writing into the [h] slices. */
int lqmpc_mpc_solve_range(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, int N_min, int N_max,
                          int npts, const double* pts, const double* x0, double* V, double* u0, double* M_V,
                          int32_t* flags);
int lqmpc_bounds_range(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, int N_min, int N_max,
                       const double* e_A, const double* e_B, double e_A_scalar, double e_B_scalar, const double* M_V,
                       double M_V_scalar, const double* x_shared, const double* x, const double* K_in,
                       const double* K_shared, const double* p3_host, double V_expert, double bar_u, double bar_d_u,
                       int strict_reference, double* alpha, double* beta, double* xi, double* eta, double* bound,
                       double* detail, double* K_out, double* P_out, int32_t* flags);

/* Batched control.dlqr (utils_class.py:761,840,923): stabilising DARE solution P and K = (R+B'PB)^-1 B'PA
 * (convention u = -Kx) of (A+dA_s, B+dB_s); dA/dB NULL = the true model. K_out [m*n][S], P_out [n*n][S], flags [S]. */
int lqmpc_dlqr_batch(lqmpc_ctx* ctx, int64_t S, const double* dA, const double* dB, double* K_out, double* P_out,
                     int32_t* flags);

/* K5 — per-column statistics of a column-contiguous result table `table[c*ld + s]` (c < cols, s < S): the four
 * reductions the reference's plotters take over axis 0 of every table (utils.py:895-898: max, min, mean, std).
 *   lqmpc_column_stats : stats [cols][5] = { max, min, sum, count_finite, count_nonfinite } over the finite entries
 *   lqmpc_column_sqdev : sqdev [cols]    = sum over finite entries of (x - mean[c])^2   (np.std is two-pass)
 * Both are deterministic (fixed reduction order). Multi-GPU: all-reduce {max, -min} with MAX and
 * {sum, counts} with SUM between the two calls, then all-reduce sqdev with SUM (lq_mpc_b200/stats.py). */
int lqmpc_column_stats(lqmpc_ctx* ctx, const double* table, int cols, int64_t S, int64_t ld, double* stats);
int lqmpc_column_sqdev(lqmpc_ctx* ctx, const double* table, int cols, int64_t S, int64_t ld, const double* mean,
                       double* sqdev);

/* One-pass variant (what lq_mpc_b200/stats.py uses): moments [cols][6] = { max, min, count_finite, count_nonfinite,
 * mean, M2 = sum (x - mean)^2 } over the finite entries of every column (shifted-data accumulation, fixed-order
 * folds: deterministic). Shards are merged with Chan's pairwise update after ONE all-gather of these 6 numbers per
 * column; std = sqrt(M2 / count) as np.std (utils.py:898). Empty column: mean = M2 = NaN, max = -inf, min = +inf. */
int lqmpc_column_moments(lqmpc_ctx* ctx, const double* table, int cols, int64_t S, int64_t ld, double* moments);

/* Order statistics of the same tables, over the population the moments reduce: the entries with |x| <= 1.79e308
 * ("finite" below; NaN, +-inf and the few doubles above 1.79e308 are left out), so the moments' count_finite is the
 * count the ranks refer to.
 * Exact selection by radix descent: a finite double x maps to the order-preserving key
 *   key(x) = bits(x) ^ (x's sign bit set ? 0xFFFFFFFFFFFFFFFF : 0x8000000000000000)
 * and the key of the entry of 0-based rank r among a column's finite entries is found one byte at a time, most
 * significant first (pass 0), in 8 passes of histogram -> select. Multi-GPU: all-reduce `hist` with SUM between the
 * two calls of every pass (lq_mpc_b200/stats.py); counts are integers, so every order of summation agrees.
 *   lqmpc_column_radix_histogram : hist [cols][nsel][256] int64 = counts, by the byte of digit `pass`, of the finite
 *     entries whose key agrees with prefix [cols][nsel] on the bytes above digit `pass`; 1 <= nsel <= 32.
 *   lqmpc_column_radix_select    : for every (column, selector), the digit whose bucket holds rank[c][k]; the counts
 *     of the buckets below it are subtracted from rank (in place) and the digit is written into prefix (in place).
 *     Start with prefix = 0; after pass 7 prefix holds the key. A rank at or past the column's finite count leaves
 *     rank and prefix unchanged.
 *   lqmpc_column_argext : val [cols][2] = {max, min} of the finite entries, idx [cols][2] int64 = index_base + the
 *     lowest position attaining each (index_base >= 0); a column without a finite entry gives -inf / +inf and -1.
 * All pointers are device pointers; S = 0 is allowed (then `table` may be NULL). */
#define LQMPC_RADIX_MAX_SEL 32
int lqmpc_column_radix_histogram(lqmpc_ctx* ctx, const double* table, int cols, int64_t S, int64_t ld, int nsel,
                                 int pass, const uint64_t* prefix, int64_t* hist);
int lqmpc_column_radix_select(lqmpc_ctx* ctx, const int64_t* hist, int cols, int nsel, int pass, int64_t* rank,
                              uint64_t* prefix);
int lqmpc_column_argext(lqmpc_ctx* ctx, const double* table, int cols, int64_t S, int64_t ld, int64_t index_base,
                        double* val, int64_t* idx);

/* K6 — model-error grids generated on the device: the seeded, counter-based restatement of `random_matrix` /
 * `error_matrix_generator` (utils.py:779-847). For every error level i < n_err (bounds levels_host[i]) and perturbation
 * j in [j_first, j_first + N_sys): a rows x cols matrix with entries uniform in [-e, e], accepted when its Frobenius
 * (norm_type 0) or spectral (norm_type 1) norm is <= e; perturbations j < n_boundary are rescaled ONTO the boundary
 * (the reference obtains those by np.isclose rejection). Philox4x32-10 keyed by `seed`, counter = (j, level, attempt):
 * the result does not depend on sharding. `which` (0 for the A grid, 1 for the B grid, ...) separates the streams.
 *   out  device [rows*cols][N_sys*n_err], element (a, b) of pair (j, i) at out[(a*cols + b)*N_sys*n_err + (j-j_first)*n_err + i]
 *        — byte-identical to the reference's error_X.npy array (rows, cols, N_sys, n_err) in C order AND the engine's
 *        SoA operand layout.
 *   stats_host (may be NULL; synchronises): [0] rejected draws, [1] samples projected after 256 rejections. */
int lqmpc_sample_error_grid(lqmpc_ctx* ctx, uint64_t seed, int which, int rows, int cols, int64_t N_sys,
                            int64_t j_first, int n_err, const double* levels_host, int64_t n_boundary, int norm_type,
                            double* out, int64_t* stats_host);

/* DFMA-chain micro-benchmark: achieved FP64 FMA throughput of this device in TFLOP/s (2 flop per FMA), used as the
 * measured denominator of the FP64 roofline (MEASURED_PEAKS.json has none). Synchronises. */
int lqmpc_fp64_peak(lqmpc_ctx* ctx, double* tflops_out);

/* Same for the FP64 tensor cores (mma.sync.m8n8k4.f64 accumulator chains): the roofline denominator of K4. Synchronises. */
int lqmpc_fp64_tensor_peak(lqmpc_ctx* ctx, double* tflops_out);

/* Number of kernels this context has launched since creation (bench.py's `gpu_launches`). */
int64_t lqmpc_launch_count(const lqmpc_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* LQMPC_B200_H */
