/*
 * sgdml_b200 -- C ABI of the B200-native engine for sGDML's two dense hot paths
 * (SURVEY.md section 8).  Plain pointers and sizes only; no torch / C++ types.
 *
 * Conventions
 *  - All arrays are C-order (row-major) float64 / int64, exactly as NumPy hands them over.
 *  - Every data pointer may be a HOST pointer or a DEVICE pointer of the current CUDA
 *    device; the library detects which (cudaPointerGetAttributes) and stages host
 *    buffers through device memory itself (H2D / D2H inside the call).
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Calls
 *    with host outputs synchronise that stream before returning; calls whose outputs
 *    are device pointers are asynchronous on `stream`.
 *  - Return value: 0 = ok; > 0 = LAPACK-style `info` (leading minor of that order is not
 *    positive definite); < 0 = error (-(cudaError_t) for CUDA errors, <= -1000 for
 *    argument errors).  sgdml_b200_last_error() returns a message for the calling thread.
 *  - Notation: N atoms, D = N(N-1)/2 descriptor size, M training points, S permutations.
 *    Pair order d <-> (a,b), a > b, is np.tril_indices(N,-1) (reference desc.py:109-110).
 *
 * Each entry point cites the reference interface it replaces (paths relative to
 * /root/reference/sgdml/).  The reference is pure Python: there is no FFI to bind to,
 * the seam is its `use_torch` engine objects (train.py:1412-1482, predict.py:358-421);
 * INTEGRATION.md shows the ctypes stubs a maintainer would add there.
 */
#ifndef SGDML_B200_H
#define SGDML_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SGDML_B200_ABI_VERSION 1

#define SGDML_B200_OK 0
#define SGDML_B200_ERR_ARG (-1000)
#define SGDML_B200_ERR_UNSUPPORTED (-1001)
#define SGDML_B200_ERR_NO_DEVICE (-1002)

int sgdml_b200_abi_version(void);
/* Frees the persistent device workspaces of the current device (the Cholesky panel workspace, the int8 slice
 * planes): they are kept between calls so that a sigma grid of training runs (cli.py:802-806) pays for them once. */
int sgdml_b200_release_workspaces(void);
const char* sgdml_b200_last_error(void);
/* Number of visible CUDA devices (0 => every compute entry point fails loudly). */
int sgdml_b200_device_count(void);

/* ---------------------------------------------------------------- representation */

/* Desc.perm + tril_perms_lin: utils/desc.py:509-539, train.py:897-904.  Host integer
 * routine, bit-exact.  perms (S,N) int64 -> out (S*D,) int64,
 * out[d*S + p] = d(perms[p][a], perms[p][b]) + p*D for d = d(a,b). */
int sgdml_b200_tril_perms_lin(const int64_t* perms, int64_t n_perms, int64_t n_atoms, int64_t* out);

/* Desc.from_R: utils/desc.py:80-239, 288-365 (no lattice).  R (n_geo, 3N) ->
 * R_desc (n_geo, D), R_d_desc (n_geo, D, 3). */
int sgdml_b200_desc_from_R(const double* R, int64_t n_geo, int64_t n_atoms, double* R_desc,
                           double* R_d_desc, void* stream);

/* Desc.from_R with periodic boundary conditions: utils/desc.py:44-77 (_pbc_diff), 100-108, 200-201.  lattice and
 * lattice_inv are 3 x 3 row-major HOST arrays (lattice vectors as COLUMNS, as task['lattice'] / model['lattice'],
 * train.py:524, 826-827; the inverse as np.linalg.inv gives it, train.py:908-911).  Every pair difference is
 * clamped to the super cell, d -= lattice @ round(lattice_inv @ d), before the distance is taken. */
int sgdml_b200_desc_from_R_pbc(const double* R, int64_t n_geo, int64_t n_atoms, const double* lattice,
                               const double* lattice_inv, double* R_desc, double* R_d_desc, void* stream);

/* Desc.d_desc_dot_vec: utils/desc.py:368-385.  R_d_desc (n_geo, D, 3), vecs (n_geo, 3N)
 * -> out (n_geo, D). */
int sgdml_b200_d_desc_dot_vec(const double* R_d_desc, const double* vecs, int64_t n_geo,
                              int64_t n_atoms, double* out, void* stream);

/* Desc.vec_dot_d_desc: utils/desc.py:388-408.  R_d_desc (n_geo, D, 3), vecs (n_geo, D)
 * -> out (n_geo, 3N). */
int sgdml_b200_vec_dot_d_desc(const double* R_d_desc, const double* vecs, int64_t n_geo,
                              int64_t n_atoms, double* out, void* stream);

/* ---------------------------------------------------------------- predictor (path b) */

typedef struct sgdml_b200_model sgdml_b200_model;

/* GDMLPredict.__init__ / GDMLTorchPredict.__init__: predict.py:249-463,
 * torchtools.py:401-593.  The engine keeps device copies of the (unpermuted) model;
 * permutations are applied to the query inside the kernel, never as an M*S cache
 * (predict.py:426-441 builds that cache on the CPU).
 *   R_desc          (M, D)  -- NOTE: the .npz model stores it transposed (D, M), train.py:807
 *   R_d_desc_alpha  (M, D)
 *   tril_perms_lin  (S*D,)
 *   sig as stored in the model; std, c as GDMLPredict uses them (predict.py:1286-1288). */
int sgdml_b200_model_create(sgdml_b200_model** out, int64_t n_atoms, int64_t n_train,
                            int64_t n_perms, const double* R_desc, const double* R_d_desc_alpha,
                            const int64_t* tril_perms_lin, double sig, double std, double c);
int sgdml_b200_model_destroy(sgdml_b200_model* model);

/* GDMLPredict.predict(R): predict.py:1146-1294 (+ _predict_wkr predict.py:84-245).
 * R (B, 3N) -> E (B,) [may be NULL], F (B, 3N); outputs scaled: F*std, E*std + c. */
int sgdml_b200_predict(sgdml_b200_model* model, const double* R, int64_t n_geo, double* E,
                       double* F, void* stream);

/* Analytic Hessian (an extension: the reference predicts energies and forces only).  R (B, 3N) ->
 * H (B, 3N, 3N) = d^2 E / dR^2, row-major, full and symmetric, in model units (energy / length^2), plus E (B,) and
 * F (B, 3N) as sgdml_b200_predict gives them (E and F may be NULL).  Lattices and alphas_E are honoured.  Every
 * contraction of this call runs in FP64, whatever sgdml_b200_model_set_contraction_slices chose.  Host or device
 * pointers; the call synchronises `stream` before it returns.  Molecules up to ~225 atoms (as the predictor);
 * beyond that SGDML_B200_ERR_UNSUPPORTED.  Derivation: DESIGN.md, "Hessian". */
int sgdml_b200_predict_hessian(sgdml_b200_model* model, const double* R, int64_t n_geo, double* E, double* F,
                               double* H, void* stream);

/* Periodic model (predict.py:332-334: lat_and_inv from model['lattice']): query descriptors of
 * sgdml_b200_predict are built with the minimum-image convention.  Both NULL: back to a free molecule. */
int sgdml_b200_model_set_lattice(sgdml_b200_model* model, const double* lattice, const double* lattice_inv);

/* Energy constraints in the kernel (use_E_cstr models; predict.py:219-229, 443-447, 594-601): alphas_E (M,) or
 * NULL to switch the terms off.  With alphas_E set, every (virtual query row, training point) pair additionally
 * contributes alphas_E[m] * c2 * delta to the descriptor-space force and alphas_E[m] * K_ee to the energy,
 * K_ee = (1 + (n/sig)(1 + n/(3 sig))) exp(-n/sig). */
int sgdml_b200_model_set_alphas_E(sgdml_b200_model* model, const double* alphas_E, void* stream);

/* GDMLPredict.set_R_desc / set_R_d_desc: predict.py:511-549.  Caches the training
 * descriptor Jacobians (M, D, 3) on the device so that set_alphas and the training-point
 * evaluation need no host data. */
int sgdml_b200_model_set_R_d_desc(sgdml_b200_model* model, const double* R_d_desc);

/* GDMLPredict.set_alphas: predict.py:551-601 / torchtools.py:760-875.
 * alphas_F (3NM,) -> R_d_desc_alpha = J_m alpha_m on the device. */
int sgdml_b200_model_set_alphas(sgdml_b200_model* model, const double* alphas_F, void* stream);

/* GDMLPredict.predict() with R=None (training points from the cached descriptors):
 * predict.py:1219-1235; the K.v operator of the iterative solver (iterative.py:183-204)
 * and _recov_int_const (train.py:1136-1147).  Evaluates training points
 * [m_begin, m_end).  scaled != 0: outputs scaled as sgdml_b200_predict; scaled == 0:
 * raw sums (std = 1, c = 0), i.e. F = (K v)[m_begin*3N : m_end*3N] for alphas = v. */
int sgdml_b200_predict_train(sgdml_b200_model* model, int64_t m_begin, int64_t m_end, int scaled,
                             double* E, double* F, void* stream);

/* Large-descriptor models (D > 256: the predictor is four GEMMs around two element-wise kernels): run those GEMMs on
 * the tcgen05 tensor cores through `slices` exact int8 slices per operand (2..7; csrc/ozaki.cu) or in FP64 DMMA (0, the
 * default unless SGDML_B200_OZAKI_PREDICT_SLICES is set when the model is created).  Forces against the FP64 form:
 * 8.8e-9 / 6.5e-11 / 5.4e-13 relative for 4 / 5 / 6 slices.  The iterative solver sets 5 for its K.v products
 * (iterative.py:183-204: tolerance 1e-4).  No effect for D <= 256. */
int sgdml_b200_model_set_contraction_slices(sgdml_b200_model* model, int slices, void* stream);

/* Test / tuning hook: main kernel of the fused predictor (D <= 256).  0 = default (the measured-fastest kernel per
 * descriptor size); 1 = two warp groups running the sweep half a tile apart (72 < D; measured slower); 2 = no split
 * over k in the first contraction: Matern transform on the accumulator fragments, two CTA-wide barriers per tile
 * instead of three (72 < D <= 224); 3 = 2 with C1 / C2 double-buffered and ONE barrier per tile (D <= 224); 4 = the
 * round-1 kernels for every size; 5 = the one-barrier form on 16-point tiles for D <= 40 (two CTAs per SM).  A variant
 * without a kernel for a size runs the default kernel of that size. */
int sgdml_b200_set_predict_variant(int variant);

/* Shape of a model: n_atoms, n_train, n_perms (any pointer may be NULL). */
int sgdml_b200_model_dims(const sgdml_b200_model* model, int64_t* n_atoms, int64_t* n_train, int64_t* n_perms);

/* Reads back R_d_desc_alpha (M, D) -- the `R_d_desc_alpha` key of the model file
 * (train.py:791, 808). */
int sgdml_b200_model_get_R_d_desc_alpha(sgdml_b200_model* model, double* out);

/* ---------------------------------------------------------------- assembly (path a) */

/* GDMLTrain._assemble_kernel_mat / GDMLTorchAssemble.forward: train.py:1260-1535,
 * train.py:97-232, torchtools.py:110-392 (force-force blocks).
 *   K[i*3N + r, c] = scale * K_ref[i*3N + r, col_idxs[c]],  K is (3NM, n_cols), row
 *   stride ldk (>= n_cols).  col_idxs == NULL: all 3NM columns (n_cols must be 3NM);
 *   otherwise a sorted, duplicate-free int64 list (train.py:1341-1345).
 *   scale = -1 gives the matrix the analytic solver factorises (analytic.py:65). */
int sgdml_b200_assemble(const double* R_desc, const double* R_d_desc, const int64_t* tril_perms_lin,
                        int64_t n_atoms, int64_t n_train, int64_t n_perms, double sig,
                        const int64_t* col_idxs, int64_t n_cols, double scale, double* K,
                        int64_t ldk, void* stream);

/* Row-sharded form of sgdml_b200_assemble (SURVEY.md section 8e "explicit K assembly": blocks are
 * independent, each GPU assembles the block rows of its own training points).  Only the row
 * points [m_begin, m_end) are produced: K is ((m_end - m_begin)*3N, n_cols) and
 *   K[(i - m_begin)*3N + r, c] = scale * K_ref[i*3N + r, col_idxs[c]].
 * This is the loop `for i in range(n_train)` of train.py:193-194 cut into ranges. */
int sgdml_b200_assemble_rows(const double* R_desc, const double* R_d_desc,
                             const int64_t* tril_perms_lin, int64_t n_atoms, int64_t n_train,
                             int64_t n_perms, double sig, const int64_t* col_idxs, int64_t n_cols,
                             double scale, int64_t m_begin, int64_t m_end, double* K, int64_t ldk,
                             void* stream);

/* Energy constraints in the kernel (task['use_E_cstr'], train.py:234-300, 1325-1335): fills the M energy rows and
 * columns and the M x M energy-energy block of the (3NM + M)-square matrix K (DEVICE pointer, row stride ldk >= 3NM + M)
 * whose force-force part sgdml_b200_assemble has written with the same `scale`:
 *   K[3NM + i, blk_j] = K[blk_j, 3NM + i] = scale * K_fe(i, j),   K[3NM + j, 3NM + i] = scale * K_ee(i, j). */
int sgdml_b200_assemble_ecstr(const double* R_desc, const double* R_d_desc, const int64_t* tril_perms_lin,
                              int64_t n_atoms, int64_t n_train, int64_t n_perms, double sig, double scale, double* K,
                              int64_t ldk, void* stream);

/* Tuning / test hook: 0 = kernel chosen by molecule size (default), 1 = always the large-molecule
 * kernel (tables in global memory), which molecules above ~50 atoms need; 2 / 3 / 4 = small-molecule kernel with
 * per-permutation phases (k_assemble) / with permutation chunks and resident row tables (k_assemble_v3) / chunks of
 * up to 16 permutations with byte permutation tables and per-kind phases over the kept column atoms (k_assemble_v4);
 * 1000 + r = at most r row
 * points per launch of the small-molecule kernel (default 65535, the grid limit; tests lower it to
 * cover the multi-launch path that row ranges above 65535 training points take). */
int sgdml_b200_set_assemble_variant(int variant);

/* ---------------------------------------------------------------- dense solve (path a) */

/* scipy.linalg.cho_factor (LAPACK dpotrf) as used by analytic.py:94-96 and
 * iterative.py:447-449.  A (n, n) symmetric, row stride lda; only the LOWER triangle
 * (row-major) is read and overwritten with L (A = L L^T).  Returns info > 0 if the
 * leading minor of order info is not positive definite (analytic.py:101 catches the
 * resulting LinAlgError). */
int sgdml_b200_potrf(double* A, int64_t n, int64_t lda, void* stream);

/* scipy.linalg.cho_solve (dpotrs), analytic.py:97-99: solves L L^T X = B in place.
 * L from sgdml_b200_potrf; B (n, nrhs) row-major with row stride ldb. */
int sgdml_b200_potrs(const double* L, int64_t n, int64_t lda, double* B, int64_t nrhs,
                     int64_t ldb, void* stream);

/* Analytic.solve core, analytic.py:65-99: given Kneg = -K_ref (n, n) (device or host;
 * overwritten), adds lam to the diagonal, factorises, and returns
 * alphas = -(Kneg + lam I)^-1 y. */
int sgdml_b200_solve_analytic(double* Kneg, int64_t n, int64_t lda, double lam, const double* y,
                              double* alphas, void* stream);

/* ---------------------------------------------------------------- iterative solver blocks (path a)
 * Nystroem preconditioner of solvers/iterative.py:208-351 on X = K_nm (n_rows x m, row stride ldx),
 * the kernel columns at the inducing columns, resident in HBM (all matrix pointers below must be
 * DEVICE pointers; vectors may be host or device). */

/* K_mm = -X[row_idxs, :] (iterative.py:253); out (m x m), row stride ldo. */
int sgdml_b200_gather_rows_neg(const double* X, int64_t ldx, int64_t m, const int64_t* row_idxs,
                               double* out, int64_t ldo, void* stream);
/* A[i][i] += value (the jitter escalation of _cho_factor_stable, iterative.py:414-471). */
int sgdml_b200_add_diag(double* A, int64_t n, int64_t lda, double value, void* stream);
/* X <- X L^-T for lower-triangular L (m x m): scipy.linalg.solve_triangular(L, X.T, trans='T').T,
 * iterative.py:278-287 and 337-347. */
int sgdml_b200_trsm_right_lt(const double* L, int64_t m, int64_t ldl, double* X, int64_t n_rows,
                             int64_t ldx, void* stream);
/* C = X^T X + lam I, lower triangle (iterative.py:293-295). */
int sgdml_b200_gram_tn(const double* X, int64_t n_rows, int64_t m, int64_t ldx, double lam, double* C,
                       int64_t ldc, void* stream);
/* out[r] = |X[r, :]|^2 -- the leverage scores (iterative.py:107-109). */
int sgdml_b200_row_sqnorms(const double* X, int64_t n_rows, int64_t m, int64_t ldx, double* out,
                           void* stream);
/* out = (X (X^T v) - v) / lam -- the preconditioner P v (iterative.py:136-138). */
int sgdml_b200_nystroem_apply(const double* X, int64_t n_rows, int64_t m, int64_t ldx, double lam,
                              const double* v, double* out, void* stream);

/* The two halves of sgdml_b200_nystroem_apply for a ROW-SHARDED factor (SURVEY.md section 8e
 * "Nystroem factor (m,n): shard n"): each GPU holds the rows X_loc of its own training points,
 *   t_loc = X_loc^T v_loc            (project; the caller all-reduces t over the GPUs)
 *   out_loc = (X_loc t - v_loc)/lam  (expand;  the caller all-gathers out)
 * which together are iterative.py:136-138 on the full factor. */
int sgdml_b200_nystroem_project(const double* X, int64_t n_rows, int64_t m, int64_t ldx,
                                const double* v, double* t, void* stream);
int sgdml_b200_nystroem_expand(const double* X, int64_t n_rows, int64_t m, int64_t ldx, double lam,
                               const double* t, const double* v, double* out, void* stream);

/* ---------------------------------------------------------------- device-resident PCG (path a, large systems)
 * scipy.sparse.linalg.cg as driven by Iterative.solve, iterative.py:740-752, on the operators of
 * iterative.py:183-206 (K v = predict_train(alphas = v), here sgdml_b200_model_set_alphas +
 * sgdml_b200_predict_train on `model`, which must have been given its training Jacobians with
 * sgdml_b200_model_set_R_d_desc) and iterative.py:120-142 (P v = (X (X^T v) - v)/lam with the Nystroem
 * factor X = B^T).  Solves (-K + lam I) x = y; the caller takes alphas = -x (iterative.py:803).
 * All CG vectors stay in HBM (`workspace`, DEVICE memory of at least
 * sgdml_b200_pcg_workspace_doubles(n, n_rows_loc, m_ind, check_every) doubles, n = 3N * n_train); the host sees
 * the residual norms of the last iterations every <= check_every iterations through `progress` (non-zero
 * return = stop: the reference's restart / interrupt logic, iterative.py:726-735), nothing else.
 *   y (n), x (n, in: start vector unless x_is_zero, out: solution): host or device.
 *   tol_abs: stop when |r| <= tol_abs (the reference passes tol * |y|, iterative.py:744).
 * Several GPUs (SURVEY.md 8e): this rank evaluates the K.v rows of training points [m_begin, m_end) and holds
 * the rows X_loc ((m_end - m_begin)*3N x m_ind, row stride ldx) of the factor; `exchange` is called, in stream
 * order, with DEVICE buffers inside `workspace`:
 *   op 0: sum `count` doubles at `buf` over the ranks in place   (X^T v, m_ind doubles)
 *   op 1: all-gather: `buf` is the full vector (count = n), the rows this rank owns are in place
 * and must enqueue the collective on `stream` (torch.distributed / NCCL on the Python host).  exchange == NULL:
 * single rank, m_begin = 0, m_end = n_train.  m_ind = 0: no preconditioner (z = r). */
typedef int (*sgdml_b200_exchange_fn)(void* ctx, int op, double* buf, int64_t count);
typedef int (*sgdml_b200_pcg_progress_fn)(void* ctx, int64_t iters_done, const double* resid_hist, int64_t n_new);
int64_t sgdml_b200_pcg_workspace_doubles(int64_t n, int64_t n_rows_loc, int64_t m_ind, int64_t check_every);
int sgdml_b200_pcg(sgdml_b200_model* model, int64_t m_begin, int64_t m_end, const double* X_loc, int64_t m_ind,
                   int64_t ldx, double lam, const double* y, double* x, int x_is_zero, double tol_abs,
                   int64_t max_iters, int64_t check_every, double* workspace, int64_t workspace_doubles,
                   sgdml_b200_exchange_fn exchange, void* exchange_ctx, sgdml_b200_pcg_progress_fn progress,
                   void* progress_ctx, int64_t* iters_out, double* resid_out, void* stream);

/* C = alpha * A * B^T + beta * C on the FP64 tensor pipe (the building block of potrf's
 * trailing update; exported for tests and benchmarks).  A (m, k) lda, B (n, k) ldb,
 * C (m, n) ldc, all row-major device or host. */
int sgdml_b200_dgemm_nt(int64_t m, int64_t n, int64_t k, double alpha, const double* A,
                        int64_t lda, const double* B, int64_t ldb, double beta, double* C,
                        int64_t ldc, void* stream);

/* EXPERIMENTAL (not yet run on hardware, see csrc/ozaki.cu): the same product through the tcgen05 tensor
 * cores -- A and B are cut into n_slices signed 7-bit slices per row-scaled entry and every slice pair is
 * multiplied exactly by tcgen05.mma kind::i8 (int32 accumulators in tensor memory); C += alpha * A * B^T.
 * n_slices = 7 reproduces the FP64 Cholesky trailing update (analytic.py:94-96) to ~1e-14 relative, 8 would
 * be FP64-equivalent (tools/ozaki_study.py).  tri != 0: m == n, only tiles touching the lower triangle.
 * All pointers must be device pointers; k <= 16384. */
int sgdml_b200_ozaki_gemm_nt(int64_t m, int64_t n, int64_t k, double alpha, const double* A, int64_t lda,
                             const double* B, int64_t ldb, double* C, int64_t ldc, int n_slices, int tri,
                             void* stream);
/* Bring-up aid for the above: also returns the int8 slice planes ([n_slices][rows padded to 128][k padded to
 * 128]), the row exponents and the raw int32 level sums ([n_slices][m][n]); any output may be NULL. */
int sgdml_b200_ozaki_debug(int64_t m, int64_t n, int64_t k, const double* A, int64_t lda, const double* B,
                           int64_t ldb, double* C, int64_t ldc, int n_slices, int8_t* planes_a, int* exps_a,
                           int8_t* planes_b, int* exps_b, int* levels, void* stream);

/* ---------------------------------------------------------------- launch accounting / profiling
 * Kernel families: 0 predictor main kernel, 1 predictor auxiliary kernels, 2 K assembly,
 * 3 DMMA GEMM (Cholesky trailing update), 4 potf2 diagonal tiles, 5 panel TRSM strips,
 * 6 triangular solves, 7 descriptor kernels, 8 misc, 9 the Gram kernel of the analytic Hessian (its other
 * kernels count as 1, its weight GEMMs as 3).
 * `launches` counts kernel launches per family since the last reset (always on).  With
 * profiling enabled, the library brackets each family's launches with CUDA events on the
 * launching stream and accumulates the device time (this synchronises; benchmarks enable it
 * only for the roofline measurement, never inside a throughput-timed region). */
int sgdml_b200_profile_enable(int on);
int sgdml_b200_profile_reset(void);
int sgdml_b200_profile_get(int family, double* total_ms, int64_t* scopes, int64_t* launches);

/* FP64 tensor-pipe peak of the current device, measured live with a register-resident
 * mma.sync.m8n8k4.f64 loop (TFLOP/s); the roofline denominator for the FP64 kernels
 * (MEASURED_PEAKS.json only carries HBM and bf16 numbers). */
int sgdml_b200_fp64_peak_tflops(double* tflops);
/* Same probe held for `seconds` (<= 30); reports the second half: the sustained figure for
 * kernels timed inside a long step (clocks settle under the power cap). */
int sgdml_b200_fp64_peak_tflops_sustained(double seconds, double* tflops);

/* Trailing updates of the Cholesky factorisation: -1 = automatic (default), 0 = FP64 DMMA, 2..7 = that many signed 7-bit
 * slices per operand on the tcgen05 tensor cores (kind::i8, exact int32 accumulation in tensor memory, summed in FP64;
 * csrc/ozaki.cu).  Automatic = the environment variable SGDML_B200_OZAKI_SLICES if set, otherwise 7 slices inside
 * sgdml_b200_solve_analytic for n >= 16384 (BASELINE config 2: residual 3.7e-11, training forces equal to the FP64
 * factorisation's to 2e-11 relative) and FP64 everywhere else (sgdml_b200_potrf, the Nystroem factor). */
int sgdml_b200_set_solve_slices(int n_slices);

/* Test / tuning hook: selects the GEMM kernel used by dgemm_nt and potrf's trailing update.
 * 0 = 128x128 DMMA tiles fed by cp.async, 1 = 128x64 DMMA tiles, 2 = scalar FMA reference kernel,
 * 3 = 128x128 DMMA tiles fed by TMA tensor maps (cp.async.bulk.tensor + mbarrier ring; default). */
int sgdml_b200_set_gemm_variant(int variant);

#ifdef __cplusplus
}
#endif
#endif /* SGDML_B200_H */
