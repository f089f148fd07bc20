#pragma once
#include "common.cuh"
#include <memory>

namespace gsi {

struct BufDeleter { void operator()(gsi_buf* b) const; };
typedef std::unique_ptr<gsi_buf, BufDeleter> BufPtr;

// an iterate of the algorithm drivers and its distribution over the ranks
struct Iterate {
    BufPtr buf;
    bool sharded = false;     // true: this rank holds rows [row0, row0+mloc) only
};

BufPtr make_buf(gsi_ctx* ctx, int32_t layout, int64_t rows, int64_t cols);
void op_apply(gsi_op* op, int trans, const gsi_buf* X, gsi_buf* Y);
bool op_symmetric(const gsi_op* op);
void resolve_gemm_timing(gsi_ctx* ctx);
BufPtr X_view_for_dense(gsi_op* op, int trans, const gsi_buf* X);
void tsqr_thinQ(gsi_op* op, gsi_buf* Y, bool sharded, double* Rdev);
// local block (mloc x l) -> all m rows on every rank
void gather_rows(gsi_op* op, const gsi_buf* loc, gsi_buf* full);
// an iterate -> the caller's TALL buffer: this rank's mloc rows or all m rows, whichever `out` has; then the deferred
// LU / Jacobi verdicts (synchronises)
void deliver(gsi_op* op, Iterate& res, gsi_buf* out);
void rangefinder_fixed(gsi_op* op, const gsi_buf* Omega, int64_t q, int normaliser, gsi_buf* Q_out);
void randsvd(gsi_op* op, const gsi_buf* Omega, int64_t K, int64_t p, int64_t q, int normaliser, gsi_buf* Z_out,
             double* S_host);

// ---- extras.cu: small dense kernels of eig_nystrom (l <= 256, column-major, ld = l)
__global__ void chol_upper_kernel(double* __restrict__ B, int l, int* __restrict__ flag);
__global__ void triu_inverse_kernel(const double* __restrict__ C, int l, double* __restrict__ Cinv);
__global__ void tall_head_to_cm_kernel(const double* __restrict__ T, int64_t ld, int l, double* __restrict__ M);

// ---- cov_solve.cu: A X = B on a square kernel-covariance operator, preconditioned CG (one recurrence per column)
void kernelcov_solve(gsi_op* op, const gsi_buf* B, const gsi_buf* Omega, double rtol, int64_t maxiter, gsi_buf* X_out,
                     int64_t* iters_out, double* relres_out, double* lambda_out);
// out[c] = sum_i X[i, c] Y[i, c] over rows x cols of TALL blocks (pitch ld) by the solver's fixed-order column
// reduction; part: CS_PARTS_MAX * cols doubles of scratch; nonfinite (optional) is set when an entry of X is not finite
constexpr int CS_PARTS_MAX = 256;
void col_dot(gsi_ctx* ctx, const double* X, const double* Y, int64_t ld, int64_t rows, int64_t cols, double* part,
             double* out, int* nonfinite);

// ---- cov_chol.cu: dense Cholesky factor of a square kernel-covariance operator, solves and kriging variance
// diag: NULL or n host doubles added to the diagonal after the fill; *failed_column: 1-based, 0 unless NOT_POSDEF
gsi_chol* chol_factor(gsi_op* op, const double* diag, int64_t* failed_column);
void chol_destroy(gsi_chol* f);
void chol_download(const gsi_chol* f, double* host, int64_t ldh);
void chol_solve(const gsi_chol* f, int half, const gsi_buf* B, gsi_buf* X);
void chol_variance(const gsi_chol* f, gsi_op* cross, const double* Fs, const double* Ft, int64_t p, double* var_out);
// Z = F_t B + L(T, :) V: conditional (ns > 0) or unconditional (ns = 0) realisations from the factor of the joint matrix
void chol_simulate(const gsi_chol* f, int64_t ns, const double* y, const double* Fs, const double* Ft, int64_t p,
                   const gsi_buf* Xi, gsi_buf* Z);
// Gaussian ML / REML log-likelihood of the operator's parameters (beta by GLS), optionally with its exact gradient
// (grad_out: nstruct (1 + d) + 1 values); factors, evaluates and frees the factor
void chol_loglik(gsi_op* op, const double* y, const double* F, int64_t p, int reml, double* loglik, double* beta_out,
                 double* grad_out, int64_t* failed_column);
// cross-validation of universal kriging on the factor: for each held-out group B (CSR group_ptr / group_idx; group_ptr
// NULL: leave-one-out), err_B = P_BB^-1 (P y)_B, var_B = diag(P_BB^-1) and the log-density of y_B given the other points;
// *failed_group: 1-based, 0 unless a P_BB is not positive definite
void chol_crossval(const gsi_chol* f, const double* y, const double* F, int64_t p, int64_t ngroups,
                   const int64_t* group_ptr, const int64_t* group_idx, double* err_out, double* var_out,
                   double* logpdf_out, int64_t* failed_group);

}  // namespace gsi
