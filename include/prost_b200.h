/*
 * prost_b200.h -- C ABI of the B200-native primal-dual solver core.
 *
 * This is the drop-in boundary for the PDHG/ADMM hot path of tum-vision/prost.  The
 * reference has no C ABI of its own: its boundary is the C++ virtual-class surface in
 * include/prost/ plus the mex string registries (matlab/+prost/private/factory.cpp).
 * Every entry point below names the reference interface it replaces (paths relative
 * to the reference checkout).  The C++ classes in include/prost/ (same names and
 * signatures as the reference's) are thin RAII wrappers over these functions, and
 * INTEGRATION.md shows the mex-side binding a maintainer would add.
 *
 * Conventions
 *  - plain pointers and sizes only; `real` is float (north star), indices size_t,
 *    sparse indices int32_t, permutations int, diagonal offsets int64_t (ssize_t).
 *  - all functions returning int return PB_OK (0) or a negative pb_status; the message
 *    is available from pb_last_error() (thread-local), mirroring the strings the
 *    reference throws as prost::Exception (include/prost/exception.hpp:29-41).
 *  - handles are opaque and reference counted: a problem keeps its blocks/proxes alive,
 *    `*_destroy` only drops the caller's reference.
 *  - pointers named h_* are host memory, d_* are device memory of the context's GPU.
 *  - there is NO CPU fallback: every compute entry point fails with PB_ERR_CUDA when
 *    no CUDA device is usable.
 */
#ifndef PROST_B200_H_
#define PROST_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)   /* the library itself is built with -fvisibility=hidden */
#endif

typedef enum pb_status {
  PB_OK = 0,
  PB_ERR_INVALID = -1,   /* bad argument / inconsistent problem (reference: prost::Exception) */
  PB_ERR_CUDA = -2,      /* CUDA runtime error, no device, launch failure */
  PB_ERR_OOM = -3,       /* "Out of memory" (reference: backend_pdhg.cu:220-225) */
  PB_ERR_UNSUPPORTED = -4
} pb_status;

typedef struct pb_context pb_context;
typedef struct pb_block pb_block;
typedef struct pb_linop pb_linop;
typedef struct pb_prox pb_prox;
typedef struct pb_problem pb_problem;
typedef struct pb_backend pb_backend;
typedef struct pb_comm pb_comm;

/* ---- library / context -------------------------------------------------------------- */

const char* pb_version(void);                 /* reference: get_version(), src/common.cu:28-30 */
const char* pb_last_error(void);              /* last error message of the calling thread */
int pb_device_count(void);                    /* reference: mex "list_gpus", prost.cpp:278-297 */

/* One context per GPU and solve: device + stream + scratch.  `stream` is a cudaStream_t
 * to run on (e.g. torch's current stream) or NULL to let the context create its own.
 * Replaces the global state of the reference (cudaSetDevice in prost.cpp:56,69, static
 * cuBLAS/cuSPARSE handles, BlockDiags::cmem_counter_). */
int pb_context_create(int device, void* stream, pb_context** out);
void pb_context_destroy(pb_context* ctx);
int pb_context_synchronize(pb_context* ctx);
/* Device buffers released by destroyed problems / backends are kept in a per-process cache for the next
 * solve (the reference frees everything in its destructors and, from MATLAB, resets the device before every
 * solve: prost.cpp:69-70).  This returns all cached blocks to the driver.  PB_POOL_MB=0 disables the cache. */
void pb_release_cached_memory(void);
void* pb_context_stream(pb_context* ctx);
int pb_context_device(pb_context* ctx);

/* device memory helpers for callers that hold device vectors (reference: thrust::device_vector) */
int pb_malloc(pb_context* ctx, size_t bytes, void** d_out);
/* Pinned (page-locked) host memory for iterates and results: buffers from here are read / written by ONE DMA, where
 * the reference's std::vector results (solver.cu:152-167) are pageable.  Freed blocks are kept for exact-size
 * reuse (PB_HOST_POOL_MB, default 4096) until pb_release_cached_memory(). */
int pb_host_alloc(size_t bytes, void** h_out);
void pb_host_free(void* h_ptr);
int pb_free(pb_context* ctx, void* d_ptr);
int pb_memcpy_h2d(pb_context* ctx, void* d_dst, const void* h_src, size_t bytes);
int pb_memcpy_d2h(pb_context* ctx, void* h_dst, const void* d_src, size_t bytes);

/* ---- linear-operator blocks --------------------------------------------------------- */
/* Each create replaces the block's constructor + Initialize() (H2D copies). */

/* BlockGradient2D(row,col,nx,ny,L,label_first): include/prost/linop/block_gradient2d.hpp:41-46,
 * kernels src/linop/block_gradient2d.cu:25-139 */
int pb_block_create_gradient2d(pb_context* ctx, size_t row, size_t col, size_t nx, size_t ny,
                               size_t L, int label_first, pb_block** out);
/* BlockGradient3D: include/prost/linop/block_gradient3d.hpp, src/linop/block_gradient3d.cu:25-150 */
int pb_block_create_gradient3d(pb_context* ctx, size_t row, size_t col, size_t nx, size_t ny,
                               size_t L, int label_first, pb_block** out);
/* BlockDiags(row,col,nrows,ncols,ndiags,offsets,factors): include/prost/linop/block_diags.hpp:40-57,
 * src/linop/block_diags.cu:36-119.  No 1024-diagonal constant-memory limit, no ResetConstMem(). */
int pb_block_create_diags(pb_context* ctx, size_t row, size_t col, size_t nrows, size_t ncols,
                          size_t ndiags, const int64_t* h_offsets, const float* h_factors,
                          pb_block** out);
/* BlockSparse::CreateFromCSC(row,col,m,n,nnz,val,ptr,ind): include/prost/linop/block_sparse.hpp:43-51,
 * src/linop/block_sparse.cu:33-68 (CSC input, as MATLAB stores it) */
int pb_block_create_sparse_csc(pb_context* ctx, size_t row, size_t col, int m, int n, int nnz,
                               const float* h_val, const int32_t* h_ptr, const int32_t* h_ind,
                               pb_block** out);
/* BlockDense::CreateFromColFirstData(row,col,nrows,ncols,data): include/prost/linop/block_dense.hpp:42-43 */
int pb_block_create_dense(pb_context* ctx, size_t row, size_t col, size_t nrows, size_t ncols,
                          const float* h_data_colmajor, pb_block** out);
/* BlockDenseKronId::CreateFromColFirstData(diaglength,row,col,nrows,ncols,data): kron(K, I_diaglength), K is
 * nrows x ncols column-major, the block is (nrows*diaglength) x (ncols*diaglength)
 * (include/prost/linop/block_dense_kron_id.hpp:40-46, src/linop/block_dense_kron_id.cu) */
int pb_block_create_dense_kron_id(pb_context* ctx, size_t diaglength, size_t row, size_t col, size_t nrows,
                                  size_t ncols, const float* h_data_colmajor, pb_block** out);
/* BlockIdKronDense::CreateFromColFirstData(...): kron(I_diaglength, K) (block_id_kron_dense.hpp:42-48) */
int pb_block_create_id_kron_dense(pb_context* ctx, size_t diaglength, size_t row, size_t col, size_t nrows,
                                  size_t ncols, const float* h_data_colmajor, pb_block** out);
/* BlockSparseKronId::CreateFromCSC(row,col,diaglength,m,n,nnz,val,ptr,ind): kron(K, I_diaglength) for a sparse m x n
 * factor in CSC with int32 indices (block_sparse_kron_id.hpp:39-48, src/linop/block_sparse_kron_id.cu) */
int pb_block_create_sparse_kron_id(pb_context* ctx, size_t row, size_t col, size_t diaglength, int m, int n, int nnz,
                                   const float* h_val, const int32_t* h_ptr, const int32_t* h_ind, pb_block** out);
/* BlockIdKronSparse::CreateFromCSC(...): kron(I_diaglength, K) (block_id_kron_sparse.hpp:39-48) */
int pb_block_create_id_kron_sparse(pb_context* ctx, size_t row, size_t col, size_t diaglength, int m, int n, int nnz,
                                   const float* h_val, const int32_t* h_ptr, const int32_t* h_ind, pb_block** out);
/* BlockZero(row,col,nrows,ncols): include/prost/linop/block_zero.hpp */
int pb_block_create_zero(pb_context* ctx, size_t row, size_t col, size_t nrows, size_t ncols,
                         pb_block** out);
void pb_block_destroy(pb_block* b);
size_t pb_block_row(const pb_block* b);
size_t pb_block_col(const pb_block* b);
size_t pb_block_nrows(const pb_block* b);
size_t pb_block_ncols(const pb_block* b);
/* Block::row_sum(row,alpha)/col_sum(col,alpha) with block-local indices: block.hpp:63-70 */
float pb_block_row_sum(const pb_block* b, size_t row, float alpha);
float pb_block_col_sum(const pb_block* b, size_t col, float alpha);
size_t pb_block_gpu_mem_amount(const pb_block* b);

/* ---- LinearOperator: include/prost/linop/linearoperator.hpp:36-90 ---------------------- */
int pb_linop_create(pb_context* ctx, pb_linop** out);
void pb_linop_destroy(pb_linop* op);
int pb_linop_add_block(pb_linop* op, pb_block* b);           /* AddBlock */
int pb_linop_initialize(pb_linop* op);                       /* Initialize: sizes + overlap check */
size_t pb_linop_nrows(const pb_linop* op);
size_t pb_linop_ncols(const pb_linop* op);
/* Eval / EvalAdjoint on device vectors: result = beta*result + K rhs (linearoperator.cu:134-170) */
int pb_linop_eval(pb_linop* op, float* d_result, const float* d_rhs, float beta, int transpose);
/* host-vector debug overloads (linearoperator.cu:172-220); *ms_out (may be NULL) = device ms */
int pb_linop_eval_host(pb_linop* op, float* h_result, const float* h_rhs, int transpose,
                       double* ms_out);
float pb_linop_row_sum(const pb_linop* op, size_t row, float alpha);
float pb_linop_col_sum(const pb_linop* op, size_t col, float alpha);
/* all row/col sums at once (what mex EvalLinOp returns, prost.cpp:212-216) */
int pb_linop_row_sums(const pb_linop* op, float alpha, float* h_out);
int pb_linop_col_sums(const pb_linop* op, float alpha, float* h_out);

/* ---- proximal operators ---------------------------------------------------------------- */

/* Function1D family: include/prost/prox/elemop/function_1d.hpp:34-326; ids follow the order
 * of the mex registry (factory.cpp:18-116 "elem_operation:1d:<name>") */
typedef enum pb_function1d {
  PB_FUN_ZERO = 0, PB_FUN_ABS, PB_FUN_SQUARE, PB_FUN_IND_LEQ0, PB_FUN_IND_GEQ0, PB_FUN_IND_EQ0,
  PB_FUN_IND_BOX01, PB_FUN_MAX_POS0, PB_FUN_L0, PB_FUN_HUBER, PB_FUN_LQ, PB_FUN_LQ_PLUS_EPS,
  PB_FUN_TRUNC_QUAD, PB_FUN_TRUNC_LINEAR, PB_FUN_COUNT_
} pb_function1d;
int pb_function1d_from_name(const char* name);   /* "abs","square",... ; -1 if unknown */

/* ProxElemOperation<T,ElemOperation1D<T,FUN>>(index,count,dim,interleaved,diagsteps,coeffs):
 * prox_elem_operation.hpp:66-72, elem_operation_1d.hpp:36-59.  coeffs = 7 arrays a,b,c,d,e,alpha,beta,
 * each of length 1 (scalar) or count (per element), exactly like std::array<vector<T>,7>. */
int pb_prox_create_elem_1d(pb_context* ctx, size_t index, size_t count, size_t dim,
                           int interleaved, int diagsteps, int function,
                           const float* const h_coeffs[7], const size_t coeff_len[7],
                           pb_prox** out);
/* ProxElemOperation<T,ElemOperationNorm2<T,FUN>>: elem_operation_norm2.hpp:39-88 */
int pb_prox_create_elem_norm2(pb_context* ctx, size_t index, size_t count, size_t dim,
                              int interleaved, int diagsteps, int function,
                              const float* const h_coeffs[7], const size_t coeff_len[7],
                              pb_prox** out);
/* ProxElemOperation<T,ElemOperationIndSimplex<T>>: elem_operation_ind_simplex.hpp:47-115 */
int pb_prox_create_ind_simplex(pb_context* ctx, size_t index, size_t count, size_t dim,
                               int interleaved, int diagsteps, pb_prox** out);
/* ProxElemOperation<T,ElemOperationIndSum<T>>: projection of every group onto sum_i x_i = 1
 * (elem_operation_ind_sum.hpp:38-58; mex name "elem_operation:ind_sum", +function/sum_ind_sum.m) */
int pb_prox_create_ind_sum(pb_context* ctx, size_t index, size_t count, size_t dim, int interleaved,
                           int diagsteps, pb_prox** out);
/* ProxIndSum(index,size,count,dim,inds,sum[,count2,dim2,inds2,sum2]) (prox_ind_sum.hpp:37-62, prox_ind_sum.cu:33-145;
 * mex name "ind_sum", +function/sum_ind_sum2.m): groups given as index lists (count*dim entries relative to `index`,
 * group-major) are projected onto sum = `sum` in the metric of the step sizes; all other elements are copied.
 * h_inds2 == NULL: one list.  diagsteps is always true. */
int pb_prox_create_ind_sum_indexed(pb_context* ctx, size_t index, size_t size, size_t count, size_t dim,
                                   const unsigned long long* h_inds, float sum, size_t count2, size_t dim2,
                                   const unsigned long long* h_inds2, float sum2, pb_prox** out);
/* Spectral element operations: ProxElemOperation<T, ElemOperationSingularNx2<T, FUN_2D>> (prox of
 * h(sigma_1) + h(sigma_2) / a Function2D of the singular values of an N x 2 matrix, dim = 2N,
 * elem_operation_singular_nx2.hpp:32-150, function_2d.hpp:28-101) and ElemOperationEigen2x2 / Eigen3x3 / EigenNxN
 * (prox of sum_i h(lambda_i) of the symmetrised matrix, dim = 4 / 9 / n^2 with n <= 32, the reference's N_MAX;
 * elem_operation_eigen_2x2.hpp:94-146, elem_operation_eigen_3x3.hpp:302-377, elem_operation_eigen_nxn.hpp).
 * coeffs = a, b, c, d, e, alpha, beta of c h(a x - b) + d x + (e/2) x^2, 1 or count entries each.
 * function_2d (singular_nx2 only): 0 = sum_1d:<function_1d>, 1 = ind_l1_ball, 2 = moreau:ind_l1_ball. */
typedef enum pb_spectral_kind {
  PB_SPECTRAL_SINGULAR_NX2 = 0, PB_SPECTRAL_EIGEN_2X2 = 1, PB_SPECTRAL_EIGEN_3X3 = 2, PB_SPECTRAL_EIGEN_NXN = 3,
  /* ElemOperationMass4 / Mass5<conjugate> (elem_operation_mass_norm.hpp:17-186; mex names "elem_operation:mass4",
   * "elem_operation:ind_comass4_ball", "...:mass5", "...:ind_comass5_ball"): prox of the mass norm of a 2-vector in
   * R^4 (dim 6) / R^5 (dim 10) resp. projection onto the comass unit ball; coeffs[0] = cost (mass4 only) */
  PB_SPECTRAL_MASS4 = 4, PB_SPECTRAL_COMASS4_BALL = 5, PB_SPECTRAL_MASS5 = 6, PB_SPECTRAL_COMASS5_BALL = 7
} pb_spectral_kind;
int pb_prox_create_spectral(pb_context* ctx, int kind, size_t index, size_t count, size_t dim, int interleaved,
                            int diagsteps, int function_1d, int function_2d, const float* const h_coeffs[7],
                            const size_t coeff_len[7], pb_prox** out);
/* ProxIndRange(index, size, diagsteps) + setA(m, n, nnz, val, ptr, ind) + setAA(n, n, val) (prox_ind_range.hpp:37-50,
 * prox_ind_range.cu:28-300; mex name "ind_range"): projection onto the range of the sparse m x n matrix A (CSC like
 * BlockSparse::CreateFromCSC), x = A (A^T A)^{-1} A^T x0, with the dense column-major AA = A^T A (n <= 4096).
 * m must equal size. */
int pb_prox_create_ind_range(pb_context* ctx, size_t index, size_t size, int diagsteps, int m, int n, int nnz,
                             const float* h_val, const int32_t* h_ptr, const int32_t* h_ind, const float* h_aa,
                             pb_prox** out);
/* ProxIndEpiConjQuad1D (north star: "ProxEpiConjQuadr"; mex name "ind_epi_conjquad_1d"): per (x, y) pair the
 * projection onto the epigraph of the conjugate of rho(u) = a u^2 + b u + c on [alpha, beta], a >= 0.  PARITY
 * UNPINNED: the reference only names the class (cmake/CustomSources.cmake.example:8-14, un-vendored repository
 * preciserelaxation/src/cvpr2016/prost); built on helper.hpp:112-215 and validated against a double-precision
 * brute-force projection.  coeffs = {a, b, c, alpha, beta}, each with 1 or count entries; pairs are planar
 * (x at i, y at count + i) or interleaved. */
int pb_prox_create_ind_epi_conjquad_1d(pb_context* ctx, size_t index, size_t count, int interleaved, int diagsteps,
                                       const float* const h_coeffs[5], const size_t coeff_len[5], pb_prox** out);
/* ProxIndHalfspace(index,count,dim,interleaved,diagsteps,a,b): projection onto <a, x> <= b per group; a has
 * count*dim (planar) or dim entries, b count or 1 (prox_ind_halfspace.hpp:41-52, prox_ind_halfspace.cu:34-137) */
int pb_prox_create_ind_halfspace(pb_context* ctx, size_t index, size_t count, size_t dim, int interleaved,
                                 int diagsteps, const float* h_a, size_t na, const float* h_b, size_t nb,
                                 pb_prox** out);
/* ProxIndSOC(index,count,dim,interleaved,diagsteps,alpha): projection onto |x|_2 <= y, y = last component;
 * alpha must be 1 like in the reference (prox_ind_soc.hpp:39-48, prox_ind_soc.cu:33-120) */
int pb_prox_create_ind_soc(pb_context* ctx, size_t index, size_t count, size_t dim, int interleaved,
                           int diagsteps, float alpha, pb_prox** out);
/* ProxIndEpiQuad(index,count,dim,interleaved,diagsteps,a,b,c): prox_ind_epi_quad.hpp:42-51 */
int pb_prox_create_ind_epi_quad(pb_context* ctx, size_t index, size_t count, size_t dim,
                                int interleaved, int diagsteps, const float* h_a, size_t na,
                                const float* h_b, size_t nb, const float* h_c, size_t nc,
                                pb_prox** out);
/* ProxTransform(shared_ptr<Prox> inner, a, b, c, d, e): prox of c f(a x - b) + <d, x> + (e/2)|x|^2 through the
 * prox of f (prox_transform.hpp:38-44, prox_transform.cu:27-226); every coefficient has 1 or size elements,
 * `a` must not contain zeros (same exception text as the reference) */
int pb_prox_create_transform(pb_context* ctx, pb_prox* inner, const float* const coeffs[5],
                             const size_t coeff_len[5], pb_prox** out);
/* ProxMoreau(shared_ptr<Prox>): prox_moreau.hpp:37, prox_moreau.cu:98-134 */
int pb_prox_create_moreau(pb_context* ctx, pb_prox* conjugate, pb_prox** out);
/* ProxPermute(shared_ptr<Prox>, vector<int>): prox_permute.hpp:37, prox_permute.cu:101-145 */
int pb_prox_create_permute(pb_context* ctx, pb_prox* base, const int* h_perm, size_t n,
                           pb_prox** out);
/* ProxZero(index,size): prox_zero.hpp:34 */
int pb_prox_create_zero(pb_context* ctx, size_t index, size_t size, pb_prox** out);
void pb_prox_destroy(pb_prox* p);
size_t pb_prox_index(const pb_prox* p);
size_t pb_prox_size(const pb_prox* p);
int pb_prox_diagsteps(const pb_prox* p);
size_t pb_prox_gpu_mem_amount(const pb_prox* p);
/* Prox::Eval(result,arg,tau_diag,tau,invert_tau) on full-length device vectors (prox.cu:26-43) */
int pb_prox_eval(pb_prox* p, float* d_result, const float* d_arg, const float* d_tau_diag,
                 float tau, int invert_tau);
/* host-vector overload (prox.cu:45-71); n = length of the three vectors */
int pb_prox_eval_host(pb_prox* p, float* h_result, const float* h_arg, const float* h_tau_diag,
                      size_t n, float tau, int invert_tau, double* ms_out);

/* ---- Problem: include/prost/problem.hpp:64-114, src/problem.cu ---------------------------- */
int pb_problem_create(pb_context* ctx, pb_problem** out);
void pb_problem_destroy(pb_problem* p);
int pb_problem_add_block(pb_problem* p, pb_block* b);
int pb_problem_add_prox_g(pb_problem* p, pb_prox* x);
int pb_problem_add_prox_f(pb_problem* p, pb_prox* x);
int pb_problem_add_prox_gstar(pb_problem* p, pb_prox* x);
int pb_problem_add_prox_fstar(pb_problem* p, pb_prox* x);
int pb_problem_set_dimensions(pb_problem* p, size_t nrows, size_t ncols);
int pb_problem_set_scaling_alpha(pb_problem* p, float alpha);        /* default: alpha = 1 */
int pb_problem_set_scaling_identity(pb_problem* p);
int pb_problem_set_scaling_custom(pb_problem* p, const float* h_left, size_t nleft,
                                  const float* h_right, size_t nright);
int pb_problem_initialize(pb_problem* p);        /* problem.cu:195-323 */
int pb_problem_dualize(pb_problem* p);           /* problem.cu:538-547 */
size_t pb_problem_nrows(const pb_problem* p);
size_t pb_problem_ncols(const pb_problem* p);
size_t pb_problem_gpu_mem_amount(const pb_problem* p);
/* power iteration of problem.cu:428-500.  h_x0 (ncols floats) may be NULL: then the start
 * vector is std::rand()-based like the reference (unseeded there, seeded 0 here). */
int pb_problem_normest(pb_problem* p, float tol, int max_iters, const float* h_x0, float* out);
int pb_problem_get_scaling(const pb_problem* p, float* h_left, float* h_right);

/* ---- Backends: include/prost/backend/backend.hpp:37-95 ---------------------------------- */

/* Solver<T>::Options scalar part (include/prost/solver.hpp:39-70); x0/y0 go to pb_backend_initialize */
typedef struct pb_solver_options {
  float tol_rel_primal, tol_rel_dual, tol_abs_primal, tol_abs_dual;
  int max_iters;
  int num_cback_calls;
  int verbose;
  int solve_dual_problem;
} pb_solver_options;

/* BackendPDHG<T>::Options (include/prost/backend/backend_pdhg.hpp:57-82) */
typedef enum pb_pdhg_stepsize {
  PB_PDHG_ALG1 = 1, PB_PDHG_ALG2 = 2, PB_PDHG_GOLDSTEIN = 3, PB_PDHG_BOYD = 4
} pb_pdhg_stepsize;
typedef struct pb_pdhg_options {
  double tau0, sigma0;
  int residual_iter;
  int scale_steps_operator;
  float alg2_gamma;
  float arg_alpha0, arg_nu, arg_delta;
  float arb_delta, arb_tau;
  int stepsize_variant;       /* pb_pdhg_stepsize */
  /* extensions (not in the reference): */
  int fuse;                   /* 1 (default via pb_pdhg_default_options): fused passes where the
                                 planner can, specialised stencil kernels where the operator is a
                                 planar gradient, and the whole iteration as ONE tiled pass where the
                                 problem has the ROF shape (pb_tile.cu); 3: like 1 without the tiled
                                 pass; 2: generic fused kernels only; 0: reference-shaped unfused
                                 kernels */
  const float* normest_x0;    /* optional ncols-vector start for normest (parity runs); on a slab the rank's
                                 slice of the global start vector (its local ncols floats) */
} pb_pdhg_options;
void pb_solver_default_options(pb_solver_options* o);   /* matlab/+prost/options.m:3-14 */
void pb_pdhg_default_options(pb_pdhg_options* o);       /* matlab/+prost/+backend/pdhg.m:3-14 */

/* BackendADMM<T>::Options (include/prost/backend/backend_admm.hpp:38-63) */
typedef struct pb_admm_options {
  double rho0;
  double alpha;                              /* over-relaxation */
  double cg_tol_pow, cg_tol_min, cg_tol_max;
  int cg_max_iter;
  int residual_iter;
  float arb_delta, arb_tau, arb_gamma;
} pb_admm_options;
void pb_admm_default_options(pb_admm_options* o);       /* matlab/+prost/+backend/admm.m:3-13 */

int pb_pdhg_create(pb_context* ctx, pb_problem* prob, const pb_pdhg_options* opts,
                   const pb_solver_options* sopts, pb_backend** out);
int pb_admm_create(pb_context* ctx, pb_problem* prob, const pb_admm_options* opts,
                   const pb_solver_options* sopts, pb_backend** out);
void pb_backend_destroy(pb_backend* b);
/* Backend::SetOptions(Solver::Options) as called by Solver::Initialize (solver.cu:88-90): the solver's
 * tolerances govern eps_primal / eps_dual and hence the stopping test.  Before pb_backend_initialize. */
int pb_backend_set_solver_options(pb_backend* b, const pb_solver_options* sopts);
/* Backend::Initialize with Solver::Options::x0/y0 (NULL or length 0 => zeros) */
int pb_backend_initialize(pb_backend* b, const float* h_x0, size_t nx0, const float* h_y0,
                          size_t ny0);
/* n x Backend::PerformIteration, enqueued asynchronously on the context's stream.  Residual
 * and step-size semantics at residual_iter boundaries are identical to n single calls. */
int pb_backend_iterate(pb_backend* b, int n_iters);
/* primal_residual, dual_residual, primal_var_norm, dual_var_norm, eps_primal, eps_dual
 * (backend.hpp:58-74) as of the last residual refresh; synchronises the stream. */
int pb_backend_residuals(pb_backend* b, float out[6]);
int pb_backend_stepsizes(pb_backend* b, double out[3]);        /* tau (rho for ADMM), sigma, theta */
size_t pb_backend_iteration(const pb_backend* b);
/* current_solution(x,z,y,w): backend_pdhg.cu:513-563; any pointer may be NULL */
int pb_backend_current_solution(pb_backend* b, float* h_x, float* h_z, float* h_y, float* h_w);
size_t pb_backend_gpu_mem_amount(const pb_backend* b);
/* 1 if the fused-pass planner accepted the problem, 0 if the unfused kernels run */
int pb_backend_is_fused(const pb_backend* b);
/* PDHG: iterations that ran as ONE tiled pass over HBM (pb_tile.cu) since Initialize; 0 for other schedules */
unsigned long long pb_backend_one_pass_iterations(const pb_backend* b);
/* kernels launched by this backend since creation (bench.py "gpu_launches") */
unsigned long long pb_backend_launch_count(const pb_backend* b);
/* Runs n_iters further iterations with CUDA events around every phase and returns the average
 * device milliseconds per iteration of { primal pass, dual pass, residual/step-size finalize }
 * (fused mode) or { primal half, dual half, residuals } (unfused).  Measurement aid for the
 * roofline figures in bench.py; advances the iteration like pb_backend_iterate. */
int pb_backend_profile(pb_backend* b, int n_iters, float out_ms[3]);
/* Same, split by kernel schedule (PDHG, fused mode): out = { primal pass ms, dual pass ms (averages over
 * the iterations that ran as two passes), finalize ms (average over all), whole-iteration tiled kernel
 * ms (average over the tiled iterations that do not refresh the residuals), #two-pass iterations, #such
 * tiled iterations, tiled residual-refresh kernel ms, #tiled residual-refresh iterations } */
int pb_backend_profile_detail(pb_backend* b, int n_iters, float out[8]);
/* device pointers of the current iterates (x: ncols, y: nrows) for zero-copy callers */
/* PB_RING_TRACE=1 (scaling experiments): per launch of the one-pass ring kernel {first CTA start, last CTA end,
 * longest left-edge halo wait, longest right-edge halo wait} in ns of the GPU's global timer; copies up to n
 * launches (4 values each) and returns the number of launches traced so far. */
unsigned pb_ring_trace_read(unsigned long long* h_out, unsigned n);
int pb_backend_device_iterates(pb_backend* b, float** d_x, float** d_y);

/* ---- multi-GPU slab decomposition (no counterpart in the reference, which is single-GPU:
 * SURVEY.md 2a / 8(e)) ----------------------------------------------------------------------
 * One process per GPU.  Every rank builds the Problem of ITS block of image columns
 * (BlockGradient2D/3D with the local nx, prox coefficient arrays sliced to those columns; ranks are
 * ordered left to right along x) and attaches a communicator to the PDHG backend before
 * pb_backend_initialize.  Stencil halos then travel peer-to-peer inside the fused passes (CUDA IPC
 * mapped neighbour memory over NVLink; NCCL send/recv staging when PB_HALO=nccl or IPC is
 * unavailable) and the four residual sums are all-reduced with NCCL at residual_iter boundaries.
 * With a communicator attached, pb_backend_initialize / iterate / residuals / current_solution and
 * pb_solver_solve are COLLECTIVE: every rank must make the same calls.
 * The default options work as on one GPU: on slabs, scale_steps_operator runs the power iteration on the global
 * operator (edge columns exchanged with the neighbours, sums over the ranks; the default start vector is the
 * single-GPU one restricted to the slab); on row shards, alpha scaling gives the preconditioners of the whole
 * operator (pb_problem_get_scaling then returns the global T and this rank's rows of Sigma).
 * pb_problem_normest itself is rank-local on a slab's problem. */
#define PB_COMM_ID_BYTES 128
/* rank 0 creates the id (an ncclUniqueId); the host distributes the 128 bytes to all ranks
 * (torch.distributed broadcast, MPI_Bcast, a file, ...) */
int pb_comm_unique_id(void* h_id_out);
int pb_comm_create(pb_context* ctx, int rank, int world, const void* h_id, pb_comm** out);
void pb_comm_destroy(pb_comm* c);
int pb_comm_rank(const pb_comm* c);
int pb_comm_world(const pb_comm* c);
/* 1: halos stored directly into the neighbour's memory by the kernels; 0: NCCL staging */
int pb_comm_peer_to_peer(const pb_comm* c);
int pb_comm_barrier(pb_comm* c);
/* sum over ranks of n host doubles, in place (host-side reductions of callers, e.g. objectives) */
int pb_comm_allreduce_sum(pb_comm* c, double* h_buf, size_t n);
/* the backend's Problem is the shard of rank pb_comm_rank(c); the comm must outlive the backend.
 * BackendPDHG: a slab of image COLUMNS (stencil halos travel peer to peer inside the kernels).
 * BackendADMM: a block of ROWS of K and of the f-side proxes (SURVEY.md 8(e)); columns and the n-side vectors are
 *   replicated, K^T r is summed over the ranks with one ncclAllReduce of n floats per adjoint apply
 *   (cgls.hpp:290-357, backend_admm.cu:198-272 on one GPU), sums over rows inside the reduction kernels.  With alpha
 *   scaling, pb_backend_initialize replaces the rank-local preconditioners by those of the whole operator (column
 *   sums over all ranks' rows, the empty-row carry across the ranks). */
int pb_backend_set_slab(pb_backend* b, pb_comm* c);

/* ---- Solver loop: Solver<T>::Solve, src/solver.cu:122-209 ------------------------------- */
typedef int (*pb_stopping_cb)(void* user);    /* StoppingCallback, called every iteration */
/* IntermCallback(iteration, primal, dual); returns nonzero to signal convergence */
typedef int (*pb_interm_cb)(void* user, int iteration, const float* h_primal, size_t n_primal,
                            const float* h_dual, size_t n_dual);
typedef enum pb_convergence {
  PB_CONVERGED = 0, PB_STOPPED_MAX_ITERS = 1, PB_STOPPED_USER = 2
} pb_convergence;
/* Runs the reference's loop on an initialised backend.  h_x,h_z,h_y,h_w receive
 * cur_primal_sol / cur_primal_constr_sol / cur_dual_sol / cur_dual_constr_sol (may be NULL).
 * *iters_out = iterations performed. */
int pb_solver_solve(pb_backend* b, const pb_solver_options* sopts, pb_stopping_cb stop,
                    pb_interm_cb interm, void* user, float* h_x, float* h_z, float* h_y,
                    float* h_w, int* result_out, int* iters_out);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* PROST_B200_H_ */
