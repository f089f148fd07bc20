// A X = B on a square kernel-covariance operator (the kriging weights w = (C + nugget I)^-1 (y - drift)) by k
// independent preconditioned conjugate-gradient recurrences that share one operator product of width k per
// iteration (not block CG: column j has its own alpha_j, beta_j and stopping test), with the randomized Nystrom
// preconditioner of Frangella, Tropp and Udell, "Randomized Nystrom preconditioning", SIMAX 2023, Alg. 2.1 / eq. 1.3.
//
// Everything around the product (kcov_gemm.cu, unchanged) is here: column-wise reductions over TALL blocks and the
// fused element-wise updates.  Sums are deterministic: every CTA owns a fixed row range and writes one partial per
// column, a second kernel adds the partials in CTA order, no atomics -- a solve is bit-reproducible run to run on a
// given GPU count.  On several ranks the iterates are row-sharded (this rank's rows [row0, row0 + mloc)), the search
// direction is gathered before each product, and the k-length dots and the r x k block U'R are all-reduced.
//
// One iteration (k columns, r-column preconditioner), passes over the mloc x k blocks besides the product:
//   1. p'q partials                                  read P, Q
//   2. X += alpha P, R -= alpha Q, ||r||^2 partials   read X, P, R, Q; write X, R
//   3. W = U'R (dense GEMM, r x k)                   read R
//   4. T = (U diag(d)) W (dense GEMM)                write T
//   5. Z = R + T, r'z partials                       read R, T; write Z
//   6. P = Z + beta P (converged columns: 0)         read Z, P; write P
// Without a preconditioner z = r: passes 1, 2 and 6 (with Z = R) only.  alpha and beta are formed on the device
// from the reduced dots, masked by the converged flags; the host reads two status words per iteration (the number
// of unconverged columns and the breakdown flag) -- the one host synchronisation of an iteration.
#include "common.cuh"
#include "algos.h"
#include <cmath>

namespace gsi {

constexpr int CS_LANES = 32;         // columns of a CTA (one per lane)
constexpr int CS_WARPS = 8;          // row phases of a CTA
constexpr int CS_MAX_PARTS = 256;    // CTAs along the rows, i.e. partials per column
constexpr int CS_MAX_RANK = 256;     // columns of the Nystrom sketch

// Launch shape of the column-wise kernels: CTA (b, y) owns rows [b * chunk, (b + 1) * chunk) and columns
// [32 y, 32 y + 32); warp w of it adds rows b * chunk + w, + 8, ... in order.  The shape depends on rows only.
struct ColLaunch {
    dim3 grid, block;
    int64_t chunk;
    int nparts;
};

static ColLaunch col_launch(int64_t rows, int64_t cols) {
    int64_t np = (rows + 255) / 256;
    if (np < 1) np = 1;
    if (np > CS_MAX_PARTS) np = CS_MAX_PARTS;
    ColLaunch L;
    L.nparts = (int)np;
    L.chunk = (rows + np - 1) / np;
    L.grid = dim3((unsigned)np, (unsigned)((cols + CS_LANES - 1) / CS_LANES));
    L.block = dim3(CS_LANES, CS_WARPS);
    return L;
}

// this CTA's partial of column c: the 8 warp sums added in warp order
__device__ __forceinline__ void cs_store_partial(double acc, int64_t k, double* __restrict__ part) {
    __shared__ double red[CS_WARPS][CS_LANES];
    red[threadIdx.y][threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.y == 0) {
        const int64_t c = (int64_t)blockIdx.y * CS_LANES + threadIdx.x;
        double s = red[0][threadIdx.x];
        for (int w = 1; w < CS_WARPS; ++w) s += red[w][threadIdx.x];
        if (c < k) part[(int64_t)blockIdx.x * k + c] = s;
    }
}

// partials of sum_i X[i, c] Y[i, c]; nonfinite (optional) is set when an entry of X is not finite
__global__ void cov_solve_dot_kernel(const double* __restrict__ X, const double* __restrict__ Y, int64_t ld, int64_t rows,
                                     int64_t k, int64_t chunk, double* __restrict__ part, int* __restrict__ nonfinite) {
    const int64_t c = (int64_t)blockIdx.y * CS_LANES + threadIdx.x;
    const int64_t r0 = (int64_t)blockIdx.x * chunk, r1 = min(rows, r0 + chunk);
    double acc = 0.0;
    bool bad = false;
    if (c < k)
        for (int64_t i = r0 + threadIdx.y; i < r1; i += CS_WARPS) {
            const double x = X[i * ld + c];
            bad |= !isfinite(x);
            acc += x * Y[i * ld + c];
        }
    if (bad && nonfinite) *nonfinite = 1;
    cs_store_partial(acc, k, part);
}

// out[c] = sum of the partials of column c in CTA order
__global__ void cov_solve_reduce_kernel(const double* __restrict__ part, int nparts, int64_t k, double* __restrict__ out) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= k) return;
    double s = 0.0;
    for (int b = 0; b < nparts; ++b) s += part[(int64_t)b * k + c];
    out[c] = s;
}

// alpha_c = rz_c / pq_c on unconverged columns; X += alpha P, R -= alpha Q; partials of ||r_c||^2.  p'Ap <= 0 (or NaN)
// on an unconverged column sets *breakdown.  Converged columns are neither read nor written (partial 0).
__global__ void cov_solve_update_xr_kernel(double* __restrict__ X, double* __restrict__ R, const double* __restrict__ P,
                                           const double* __restrict__ Q, int64_t ld, int64_t rows, int64_t k,
                                           int64_t chunk, const double* __restrict__ rz, const double* __restrict__ pq,
                                           const int* __restrict__ active, double* __restrict__ part,
                                           int* __restrict__ breakdown) {
    const int64_t c = (int64_t)blockIdx.y * CS_LANES + threadIdx.x;
    const int64_t r0 = (int64_t)blockIdx.x * chunk, r1 = min(rows, r0 + chunk);
    double acc = 0.0;
    if (c < k && active[c]) {
        const double d = pq[c];
        if (!(d > 0.0)) {
            if (blockIdx.x == 0 && threadIdx.y == 0) *breakdown = 1;
        } else {
            const double alpha = rz[c] / d;
            for (int64_t i = r0 + threadIdx.y; i < r1; i += CS_WARPS) {
                const int64_t e = i * ld + c;
                X[e] += alpha * P[e];
                const double r = R[e] - alpha * Q[e];
                R[e] = r;
                acc += r * r;
            }
        }
    }
    cs_store_partial(acc, k, part);
}

// Z = R + T on unconverged columns; partials of r'z
__global__ void cov_solve_precond_kernel(double* __restrict__ Z, const double* __restrict__ R, const double* __restrict__ T,
                                         int64_t ld, int64_t rows, int64_t k, int64_t chunk,
                                         const int* __restrict__ active, double* __restrict__ part) {
    const int64_t c = (int64_t)blockIdx.y * CS_LANES + threadIdx.x;
    const int64_t r0 = (int64_t)blockIdx.x * chunk, r1 = min(rows, r0 + chunk);
    double acc = 0.0;
    if (c < k && active[c])
        for (int64_t i = r0 + threadIdx.y; i < r1; i += CS_WARPS) {
            const int64_t e = i * ld + c;
            const double r = R[e], z = r + T[e];
            Z[e] = z;
            acc += r * z;
        }
    cs_store_partial(acc, k, part);
}

// P = Z + beta P with beta_c = rz_new_c / rz_old_c (rz_old == NULL: beta = 0); converged columns: P = 0
__global__ void cov_solve_update_p_kernel(double* __restrict__ P, const double* __restrict__ Z, int64_t ld, int64_t rows,
                                          int64_t k, int64_t chunk, const double* __restrict__ rz_new,
                                          const double* __restrict__ rz_old, const int* __restrict__ active) {
    const int64_t c = (int64_t)blockIdx.y * CS_LANES + threadIdx.x;
    const int64_t r0 = (int64_t)blockIdx.x * chunk, r1 = min(rows, r0 + chunk);
    if (c >= k) return;
    const bool on = active[c] != 0;
    const double beta = (on && rz_old) ? rz_new[c] / rz_old[c] : 0.0;
    for (int64_t i = r0 + threadIdx.y; i < r1; i += CS_WARPS) {
        const int64_t e = i * ld + c;
        P[e] = on ? Z[e] + beta * P[e] : 0.0;
    }
}

// One CTA of round_up(k, 32) threads.  it == 0 starts every column; then column c converges at iteration `it` when
// ||r_c|| <= rtol ||b_c||.  status[0] = number of unconverged columns.
__global__ void cov_solve_converge_kernel(const double* __restrict__ rr, const double* __restrict__ bb, double rtol,
                                          int64_t k, int it, int* __restrict__ active, int* __restrict__ iters,
                                          int* __restrict__ status) {
    const int c = threadIdx.x;
    int a = 0;
    if (c < k) {
        a = it == 0 ? 1 : active[c];
        if (it == 0) iters[c] = 0;
        if (a && sqrt(rr[c]) <= rtol * sqrt(bb[c])) {
            a = 0;
            iters[c] = it;
        }
        active[c] = a;
    }
    const int nact = __syncthreads_count(a);
    if (c == 0) status[0] = nact;
}

// Y += (s ? a * s[0] : a) X on rows x cols of two TALL blocks of pitch ld
__global__ void cov_solve_axpy_kernel(double* __restrict__ Y, const double* __restrict__ X, int64_t ld, int64_t rows,
                                      int64_t cols, double a, const double* __restrict__ s) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * cols) return;
    const int64_t i = idx / cols, c = idx - i * cols;
    const double f = s ? a * s[0] : a;
    Y[i * ld + c] += f * X[i * ld + c];
}

// nu = sqrt(n) 2^-52 ||Y||_F from the column sums of squares (added in column order)
__global__ void cov_solve_nystrom_shift_kernel(const double* __restrict__ colsq, int r, double n, double* __restrict__ nu) {
    double s = 0.0;
    for (int i = 0; i < r; ++i) s += colsq[i];
    nu[0] = sqrt(n) * 0x1p-52 * sqrt(s);
}

// lambda_i = max(0, sigma_i^2 - nu); d_i = (lambda_r + mu) / (lambda_i + mu) - 1; lambda_r + mu <= 0 sets *bad
__global__ void cov_solve_nystrom_eig_kernel(const double* __restrict__ sig, int r, double mu, const double* __restrict__ nu,
                                             double* __restrict__ lam, double* __restrict__ dscale, int* __restrict__ bad) {
    const int i = threadIdx.x;
    if (i >= r) return;
    const double lr = fmax(0.0, sig[r - 1] * sig[r - 1] - nu[0]);
    const double li = fmax(0.0, sig[i] * sig[i] - nu[0]);
    lam[i] = li;
    dscale[i] = (lr + mu) / (li + mu) - 1.0;
    if (i == 0 && !(lr + mu > 0.0)) *bad = 1;
}

// Ud = U diag(d) on rows x r
__global__ void cov_solve_scale_cols_kernel(const double* __restrict__ U, double* __restrict__ Ud, int64_t ld, int64_t rows,
                                            int r, const double* __restrict__ d) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * r) return;
    const int64_t i = idx / r;
    const int c = (int)(idx - i * r);
    Ud[i * ld + c] = U[i * ld + c] * d[c];
}

static unsigned nblk(int64_t n) { return (unsigned)((n + 255) / 256); }

static_assert(CS_PARTS_MAX == CS_MAX_PARTS, "col_dot scratch size");
void col_dot(gsi_ctx* ctx, const double* X, const double* Y, int64_t ld, int64_t rows, int64_t cols, double* part,
             double* out, int* nonfinite) {
    const ColLaunch L = col_launch(rows, cols);
    cov_solve_dot_kernel<<<L.grid, L.block, 0, ctx->stream>>>(X, Y, ld, rows, cols, L.chunk, part, nonfinite);
    GSI_CUDA(cudaGetLastError());
    cov_solve_reduce_kernel<<<nblk(cols), 256, 0, ctx->stream>>>(part, L.nparts, cols, out);
    GSI_CUDA(cudaGetLastError());
    count_launch(ctx, 2);
}

// a TALL row block [row0, row0 + rows) of `b`, not owned
static gsi_buf row_view(const gsi_buf* b, int64_t row0, int64_t rows) {
    gsi_buf v = *b;
    v.owns = false;
    v.d = b->d + row0 * b->ld;
    v.rows = rows;
    return v;
}

// a TALL rows x cols block read as the column-major matrix of its transpose (cols x rows, pitch ld)
static gsi_buf transposed_view(const gsi_buf* b) {
    gsi_buf v;
    v.ctx = b->ctx; v.layout = GSI_LAYOUT_COLMAJOR; v.rows = b->cols; v.cols = b->rows; v.ld = b->ld;
    v.d = b->d; v.owns = false;
    return v;
}

namespace {

struct Solver {
    gsi_op* op;
    gsi_ctx* ctx;
    int64_t n, ml, k;
    bool multi;
    double* part = nullptr;       // [CS_MAX_PARTS * max(k, r)]
    size_t part_bytes = 0;
    int* flags = nullptr;         // [0] unconverged columns, [1] B not finite, [2] breakdown, [3] Cholesky, [4] eig,
                                  // [5] Omega not finite
    int* active = nullptr;        // [k]
    int* iters = nullptr;         // [k]
    size_t int_bytes = 0;

    ~Solver() {
        if (part) pool_free(ctx, part, part_bytes);
        if (flags) pool_free(ctx, flags, int_bytes);
    }

    // out[c] = sum over all rows (all ranks when `reduce`) of X[:, c] Y[:, c]
    void dot(const double* X, const double* Y, int64_t ld, int64_t rows, int64_t cols, double* out, bool reduce,
             int* nonfinite = nullptr) {
        const ColLaunch L = col_launch(rows, cols);
        cov_solve_dot_kernel<<<L.grid, L.block, 0, ctx->stream>>>(X, Y, ld, rows, cols, L.chunk, part, nonfinite);
        finish(L, cols, out, reduce);
    }
    void finish(const ColLaunch& L, int64_t cols, double* out, bool reduce) {
        GSI_CUDA(cudaGetLastError());
        cov_solve_reduce_kernel<<<nblk(cols), 256, 0, ctx->stream>>>(part, L.nparts, cols, out);
        GSI_CUDA(cudaGetLastError());
        count_launch(ctx, 2);
        if (reduce && multi) comm_allreduce_sum(ctx, out, (size_t)cols);
    }
    void axpy(double* Y, const double* X, int64_t ld, int64_t rows, int64_t cols, double a, const double* s) {
        if (rows * cols == 0) return;
        cov_solve_axpy_kernel<<<nblk(rows * cols), 256, 0, ctx->stream>>>(Y, X, ld, rows, cols, a, s);
        GSI_CUDA(cudaGetLastError());
        count_launch(ctx);
    }
    void converge(const double* rr, const double* bb, double rtol, int it) {
        const unsigned threads = (unsigned)((k + 31) / 32 * 32);
        cov_solve_converge_kernel<<<1, threads, 0, ctx->stream>>>(rr, bb, rtol, k, it, active, iters, flags);
        GSI_CUDA(cudaGetLastError());
        count_launch(ctx);
    }
    // the status words (synchronises)
    void read_flags(int* h) {
        GSI_CUDA(cudaMemcpyAsync(h, flags, 6 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        GSI_CUDA(cudaStreamSynchronize(ctx->stream));
    }
};

// The randomized Nystrom preconditioner of A = K + mu I: U (mloc x r, this rank's rows), Ud = U diag(d) and lambda.
struct Nystrom {
    int r = 0;
    BufPtr U, Ud;
    double* small = nullptr;      // Cm | Cinv | R | Us (r x r each) | sig | lam | dscale | colsq (r each) | nu
    size_t small_bytes = 0;
    gsi_ctx* ctx = nullptr;
    ~Nystrom() {
        if (small) pool_free(ctx, small, small_bytes);
    }
    double* lam() const { return small + (size_t)4 * r * r + r; }
    double* dscale() const { return small + (size_t)4 * r * r + 2 * r; }
};

void nystrom_build(Solver& S, const gsi_buf* Omega, Nystrom& N) {
    gsi_op* op = S.op;
    gsi_ctx* ctx = S.ctx;
    cudaStream_t st = ctx->stream;
    const int r = (int)Omega->cols;
    const double mu = op->nugget;
    N.r = r;
    N.ctx = ctx;
    N.small_bytes = ((size_t)4 * r * r + 4 * r + 1) * sizeof(double);
    N.small = static_cast<double*>(pool_alloc(ctx, N.small_bytes));
    double* Cm = N.small;
    double* Cinv = Cm + (size_t)r * r;
    double* Rf = Cm + (size_t)2 * r * r;
    double* Us = Cm + (size_t)3 * r * r;
    double* sig = Cm + (size_t)4 * r * r;
    double* colsq = sig + 3 * r;
    double* nu = colsq + r;
    // 1. Omega <- thin Q of Omega, redundantly on every rank (deterministic QR: the same Q everywhere)
    BufPtr Om = make_buf(ctx, GSI_LAYOUT_TALL, S.n, r);
    tall_copy(ctx, Omega, Om.get());
    qr_thinQ_inplace(ctx, Om.get(), nullptr);
    const gsi_buf Oml = row_view(Om.get(), op->row0, S.ml);
    // 2. Y = A Omega - mu Omega  (this rank's rows)
    BufPtr Y = make_buf(ctx, GSI_LAYOUT_TALL, S.ml, r);
    op_apply(op, 0, Om.get(), Y.get());
    if (mu != 0.0) S.axpy(Y->d, Oml.d, Y->ld, S.ml, r, -mu, nullptr);
    // 3. nu = sqrt(n) eps ||Y||_F ;  4. Y_nu = Y + nu Omega
    S.dot(Y->d, Y->d, Y->ld, S.ml, r, colsq, true);
    cov_solve_nystrom_shift_kernel<<<1, 1, 0, st>>>(colsq, r, (double)S.n, nu);
    GSI_CUDA(cudaGetLastError());
    count_launch(ctx);
    S.axpy(Y->d, Oml.d, Y->ld, S.ml, r, 1.0, nu);
    // 5. G = Omega' Y_nu (r x r, summed over the ranks) ;  6. C = chol(G)
    BufPtr Gt = make_buf(ctx, GSI_LAYOUT_TALL, r, r);
    const gsi_buf Omt = transposed_view(&Oml);
    dense_apply(ctx, &Omt, 0, Y.get(), Gt.get(), 1.0);
    if (S.multi) comm_allreduce_sum(ctx, Gt->d, (size_t)Gt->rows_alloc * Gt->ld);
    tall_head_to_cm_kernel<<<nblk((int64_t)r * r), 256, 0, st>>>(Gt->d, Gt->ld, r, Cm);
    chol_upper_kernel<<<1, 1024, 0, st>>>(Cm, r, S.flags + 3);
    GSI_CUDA(cudaGetLastError());
    count_launch(ctx, 2);
    int h[6];
    S.read_flags(h);
    if (h[3] != 0)
        throw Error(GSI_ERR_NOT_POSDEF, "kernelcov_solve: the Nystrom preconditioner's Cholesky factorisation failed at pivot " +
                                            std::to_string(h[3]) +
                                            " (sketch numerically rank deficient): add a nugget or use a smaller rank r");
    // 7. F = Y_nu C^-1
    triu_inverse_kernel<<<(r + 63) / 64, 64, 0, st>>>(Cm, r, Cinv);
    GSI_CUDA(cudaGetLastError());
    count_launch(ctx);
    BufPtr Ct = make_buf(ctx, GSI_LAYOUT_TALL, r, r);
    small_cm_to_tall(ctx, Cinv, r, r, r, Ct.get());
    BufPtr F = make_buf(ctx, GSI_LAYOUT_TALL, S.ml, r);
    tall_times_small(ctx, Y.get(), Ct.get(), F.get());
    // 8. F = Q_F R, R = U_R Sigma V_R'  =>  U = Q_F U_R, lambda = max(0, Sigma^2 - nu)
    tsqr_thinQ(op, F.get(), S.multi, Rf);
    svd_small(ctx, Rf, r, Us, sig);
    BufPtr Ut = make_buf(ctx, GSI_LAYOUT_TALL, r, r);
    small_cm_to_tall(ctx, Us, r, r, r, Ut.get());
    N.U = make_buf(ctx, GSI_LAYOUT_TALL, S.ml, r);
    tall_times_small(ctx, F.get(), Ut.get(), N.U.get());
    // 9. P^-1 R = R + U diag(d) (U'R), d_i = (lambda_r + mu) / (lambda_i + mu) - 1
    cov_solve_nystrom_eig_kernel<<<1, CS_MAX_RANK, 0, st>>>(sig, r, mu, nu, N.lam(), N.dscale(), S.flags + 4);
    GSI_CUDA(cudaGetLastError());
    count_launch(ctx);
    S.read_flags(h);
    if (h[4] != 0)
        throw Error(GSI_ERR_NOT_POSDEF, "kernelcov_solve: the smallest Nystrom eigenvalue plus the nugget is not positive "
                                        "(no nugget and a numerically rank-deficient sketch): add a nugget or use a smaller rank r");
    N.Ud = make_buf(ctx, GSI_LAYOUT_TALL, S.ml, r);
    if (S.ml > 0) {
        cov_solve_scale_cols_kernel<<<nblk(S.ml * r), 256, 0, st>>>(N.U->d, N.Ud->d, N.U->ld, S.ml, r, N.dscale());
        GSI_CUDA(cudaGetLastError());
        count_launch(ctx);
    }
}

}  // namespace

void kernelcov_solve(gsi_op* op, const gsi_buf* B, const gsi_buf* Omega, double rtol, int64_t maxiter, gsi_buf* X_out,
                     int64_t* iters_out, double* relres_out, double* lambda_out) {
    gsi_ctx* ctx = op->ctx;
    cudaStream_t st = ctx->stream;
    GSI_REQUIRE(op->type == OP_KERNELCOV, GSI_ERR_UNSUPPORTED,
                "kernelcov_solve needs a square kernel-covariance operator (gsi_op_kernelcov, _grid, _model or _model_grid)");
    GSI_REQUIRE(std::isfinite(rtol) && rtol > 0.0, GSI_ERR_INVALID_ARGUMENT, "kernelcov_solve: rtol must be positive and finite");
    GSI_REQUIRE(maxiter >= 0, GSI_ERR_INVALID_ARGUMENT, "kernelcov_solve: maxiter must be >= 0");
    const int64_t n = op->n, ml = op->mloc;
    GSI_REQUIRE(B->layout == GSI_LAYOUT_TALL && B->rows == n, GSI_ERR_DIMENSION_MISMATCH,
                "kernelcov_solve: B must be TALL with all n rows");
    const int64_t k = B->cols;
    // the stopping test runs in one CTA of round_up(k, 32) threads
    GSI_REQUIRE(k >= 1 && k <= kMaxWideCols, GSI_ERR_DIMENSION_MISMATCH, "kernelcov_solve: B must have 1 to 1024 columns");
    GSI_REQUIRE(X_out->layout == GSI_LAYOUT_TALL && X_out->cols == k && (X_out->rows == n || X_out->rows == ml),
                GSI_ERR_DIMENSION_MISMATCH, "kernelcov_solve: X must be TALL with B's columns and n or this rank's mloc rows");
    if (Omega) {
        GSI_REQUIRE(Omega->layout == GSI_LAYOUT_TALL && Omega->rows == n, GSI_ERR_DIMENSION_MISMATCH,
                    "kernelcov_solve: Omega must be TALL with all n rows");
        GSI_REQUIRE(Omega->cols >= 1 && Omega->cols <= CS_MAX_RANK && Omega->cols < n, GSI_ERR_INVALID_ARGUMENT,
                    "kernelcov_solve: the Nystrom rank r = columns of Omega must satisfy 1 <= r <= 256 and r < n");
    }
    const int r = Omega ? (int)Omega->cols : 0;
    lu_reset_flag(ctx);

    Solver S;
    S.op = op; S.ctx = ctx; S.n = n; S.ml = ml; S.k = k; S.multi = ctx->world > 1;
    S.part_bytes = (size_t)CS_MAX_PARTS * (k > r ? k : r) * sizeof(double);
    S.part = static_cast<double*>(pool_alloc(ctx, S.part_bytes));
    S.int_bytes = (size_t)(8 + 2 * k) * sizeof(int);
    S.flags = static_cast<int*>(pool_alloc(ctx, S.int_bytes));
    S.active = S.flags + 8;
    S.iters = S.active + k;
    GSI_CUDA(cudaMemsetAsync(S.flags, 0, S.int_bytes, st));
    const size_t vec_bytes = ((size_t)6 * k + CS_MAX_RANK) * sizeof(double);
    double* vec = static_cast<double*>(pool_alloc(ctx, vec_bytes));
    struct VecGuard { gsi_ctx* c; void* p; size_t b; ~VecGuard() { pool_free(c, p, b); } } vguard{ctx, vec, vec_bytes};
    double* bb = vec;             // ||b_c||^2
    double* rr = vec + k;         // ||r_c||^2
    double* pq = vec + 2 * k;     // p_c' A p_c
    double* rzA = vec + 3 * k;    // r_c' z_c, this and the previous iteration
    double* rzB = vec + 4 * k;
    double* rrt = vec + 5 * k;    // ||b_c - A x_c||^2 of the result
    double* oo = vec + 6 * k;     // ||Omega_c||^2 (finiteness check of the sketch)

    // ||b_c||^2 over all n rows (the same on every rank, so is the finiteness verdict); R = B, X = 0
    // and of Omega (all rows, so the verdict is the same on every rank)
    S.dot(B->d, B->d, B->ld, n, k, bb, false, S.flags + 1);
    if (Omega) S.dot(Omega->d, Omega->d, Omega->ld, n, r, oo, false, S.flags + 5);
    S.converge(bb, bb, rtol, 0);
    int h[6];
    S.read_flags(h);
    GSI_REQUIRE(h[1] == 0, GSI_ERR_INVALID_ARGUMENT, "kernelcov_solve: B has a non-finite entry");
    GSI_REQUIRE(h[5] == 0, GSI_ERR_INVALID_ARGUMENT, "kernelcov_solve: Omega has a non-finite entry");
    int nact = h[0];
    const gsi_buf Bl = row_view(B, op->row0, ml);
    BufPtr X = make_buf(ctx, GSI_LAYOUT_TALL, ml, k);
    BufPtr R = make_buf(ctx, GSI_LAYOUT_TALL, ml, k);
    BufPtr Q = make_buf(ctx, GSI_LAYOUT_TALL, ml, k);
    BufPtr P = make_buf(ctx, GSI_LAYOUT_TALL, ml, k);
    BufPtr Pf = S.multi ? make_buf(ctx, GSI_LAYOUT_TALL, n, k) : BufPtr();
    tall_cols_copy(ctx, Bl.d, Bl.ld, R->d, R->ld, ml, k);
    const int64_t ld = R->ld;

    Nystrom N;
    BufPtr Z, T, W;
    if (Omega) {
        nystrom_build(S, Omega, N);
        Z = make_buf(ctx, GSI_LAYOUT_TALL, ml, k);
        T = make_buf(ctx, GSI_LAYOUT_TALL, ml, k);
        W = make_buf(ctx, GSI_LAYOUT_TALL, r, k);
        if (lambda_out) GSI_CUDA(cudaMemcpyAsync(lambda_out, N.lam(), (size_t)r * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    const ColLaunch L = col_launch(ml, k);
    // rz = r'z with z = P^-1 r (into Z; without a preconditioner z = r and rz = ||r||^2)
    auto precondition = [&](double* rz) -> const double* {
        if (!Omega) {
            GSI_CUDA(cudaMemcpyAsync(rz, rr, (size_t)k * sizeof(double), cudaMemcpyDeviceToDevice, st));
            return R->d;
        }
        const gsi_buf Ut = transposed_view(N.U.get());
        dense_apply(ctx, &Ut, 0, R.get(), W.get(), 1.0);                         // W = U'R
        if (S.multi) comm_allreduce_sum(ctx, W->d, (size_t)W->rows_alloc * W->ld);
        tall_times_small(ctx, N.Ud.get(), W.get(), T.get());                      // T = U diag(d) W
        cov_solve_precond_kernel<<<L.grid, L.block, 0, st>>>(Z->d, R->d, T->d, ld, ml, k, L.chunk, S.active, S.part);
        S.finish(L, k, rz, true);
        return Z->d;
    };
    auto update_p = [&](const double* Zd, const double* rz_new, const double* rz_old) {
        cov_solve_update_p_kernel<<<L.grid, L.block, 0, st>>>(P->d, Zd, ld, ml, k, L.chunk, rz_new, rz_old, S.active);
        GSI_CUDA(cudaGetLastError());
        count_launch(ctx);
    };
    // the operand of a product: this rank's rows of V gathered to all n rows on several ranks
    auto full_rows = [&](gsi_buf* V) -> const gsi_buf* {
        if (!S.multi) return V;
        gather_rows(op, V, Pf.get());
        return Pf.get();
    };

    int64_t it = 0;
    if (nact > 0 && maxiter > 0) {
        GSI_CUDA(cudaMemcpyAsync(rr, bb, (size_t)k * sizeof(double), cudaMemcpyDeviceToDevice, st));
        update_p(precondition(rzA), rzA, nullptr);
    }
    double* rz_old = rzA;
    double* rz_new = rzB;
    while (nact > 0 && it < maxiter) {
        ++it;
        op_apply(op, 0, full_rows(P.get()), Q.get());                                          // Q = A P
        S.dot(P->d, Q->d, ld, ml, k, pq, true);                                                 // p'q
        cov_solve_update_xr_kernel<<<L.grid, L.block, 0, st>>>(X->d, R->d, P->d, Q->d, ld, ml, k, L.chunk, rz_old, pq,
                                                               S.active, S.part, S.flags + 2);
        S.finish(L, k, rr, true);                                                                // ||r||^2
        S.converge(rr, bb, rtol, (int)it);
        S.read_flags(h);
        if (h[2] != 0)
            throw Error(GSI_ERR_NOT_POSDEF, "kernelcov_solve: p'Ap <= 0 at iteration " + std::to_string(it) +
                                                ": the operator is not numerically positive definite (add a nugget)");
        nact = h[0];
        if (nact == 0) break;
        update_p(precondition(rz_new), rz_new, rz_old);
        std::swap(rz_old, rz_new);
    }

    // the true residual b - A x of the returned X, from one more product
    op_apply(op, 0, full_rows(X.get()), Q.get());
    S.axpy(Q->d, Bl.d, ld, ml, k, -1.0, nullptr);
    S.dot(Q->d, Q->d, ld, ml, k, rrt, true);
    std::vector<double> hb(k), ht(k);
    std::vector<int> hi(2 * k);
    GSI_CUDA(cudaMemcpyAsync(hb.data(), bb, (size_t)k * sizeof(double), cudaMemcpyDeviceToHost, st));
    GSI_CUDA(cudaMemcpyAsync(ht.data(), rrt, (size_t)k * sizeof(double), cudaMemcpyDeviceToHost, st));
    GSI_CUDA(cudaMemcpyAsync(hi.data(), S.active, (size_t)2 * k * sizeof(int), cudaMemcpyDeviceToHost, st));
    Iterate res;
    res.buf = std::move(X);
    res.sharded = S.multi;
    deliver(op, res, X_out);                     // synchronises
    for (int64_t c = 0; c < k; ++c) {
        if (iters_out) iters_out[c] = hi[k + c] + (hi[c] ? it : 0);      // unconverged: the iterations run
        if (relres_out) relres_out[c] = hb[c] > 0.0 ? std::sqrt(ht[c]) / std::sqrt(hb[c]) : 0.0;
    }
    if (nact > 0)
        throw Error(GSI_ERR_NO_CONVERGENCE, "kernelcov_solve: " + std::to_string(nact) + " of " + std::to_string(k) +
                                                " columns did not reach rtol in maxiter = " + std::to_string(maxiter) +
                                                " iterations");
}

}  // namespace gsi
