/*
 * gsi_b200.h -- C ABI of the B200-native randomized low-rank factorization path of
 * GeostatInversion.jl (RandMatFact.rangefinder / randsvd + the covariance products
 * feeding pcgalsqr / rga).
 *
 * The reference (pure Julia, /root/reference) has no FFI: its seam is Julia multiple
 * dispatch on a duck-typed operator `A` (size, A*Matrix, A', Adjoint*A;
 * src/RandMatFact.jl:52-55,67,70,85; pattern shown by LowRankCovMatrix,
 * src/lowrank.jl:38-60,115-133).  Each entry point below names the reference
 * statement(s) it replaces; the Julia-side `ccall` shim is in INTEGRATION.md and
 * julia/GeostatInversionB200.jl.
 *
 * Conventions
 *   - Float64 everywhere.  Host matrices are column-major (Julia `Array`) with an
 *     explicit leading dimension; all sizes are int64_t (Julia `Int`).
 *   - Every function returns an int32 status (GSI_OK == 0); nothing throws, exits
 *     or aborts across the ABI.  gsi_last_error_string() gives the message of the
 *     last failure on the calling thread.
 *   - There is NO CPU fallback: context creation fails (GSI_ERR_NO_DEVICE) when no
 *     sm_100 device is present.
 *   - Device buffers are opaque handles owned by the library; host pointers are
 *     only read/written during the call (synchronous upload/download), so Julia
 *     arrays need only `GC.@preserve` for the duration of the `ccall`.
 *   - Random matrices (Omega, omega vectors) are always supplied by the caller, so
 *     host seeding (`Random.seed!`, src/GeostatInversion.jl:24-27) is preserved.
 *   - One context per process and GPU.  Multi-GPU = one process (Julia worker /
 *     torchrun rank) per GPU; ranks share a 128-byte NCCL id
 *     (gsi_comm_unique_id -> broadcast by the host -> gsi_ctx_create).  Iterates
 *     and operators are row-sharded: rank r owns rows [row0, row0 + mloc).
 */
#ifndef GSI_B200_H
#define GSI_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GSI_VERSION 100 /* 0.1.0 */

/* status codes */
#define GSI_OK 0
#define GSI_ERR_INVALID_ARGUMENT 1   /* Julia shim: ErrorException / ArgumentError            */
#define GSI_ERR_DIMENSION_MISMATCH 2 /* Julia shim: DimensionMismatch                          */
#define GSI_ERR_SINGULAR 3           /* exactly-zero LU pivot: LinearAlgebra.SingularException
                                        (lu(...; check=true), src/RandMatFact.jl:60,68,72)     */
#define GSI_ERR_NOT_POSDEF 4         /* eig_nystrom Cholesky: PosDefException (:95)            */
#define GSI_ERR_CUDA 5               /* ErrorException(gsi_last_error_string())                */
#define GSI_ERR_NCCL 6
#define GSI_ERR_NO_DEVICE 7          /* no sm_100 device: the library has no CPU path          */
#define GSI_ERR_UNSUPPORTED 8
#define GSI_ERR_NEGATIVE_ITERATIONS 9 /* q < 0: error("parameter numiterations should be
                                         positive, but numiterations=$q"), src/RandMatFact.jl:63 */
#define GSI_ERR_NO_CONVERGENCE 10

/* device layouts of a buffer */
#define GSI_LAYOUT_TALL 0     /* n x l iterate (l <= 1024): Omega, Y, Q, Z, eta batches ...; wider than 256
                                 columns runs the operator products in 256-column chunks          */
#define GSI_LAYOUT_COLMAJOR 1 /* dense operator storage (A, samples, sketch S, H)              */

/* covariance kernels of the matrix-free operator (NEW: the reference contains no
 * kernel function, SURVEY.md F4).  With u = x ./ ell (scaled once) and
 * r2 = sum_k (u_i[k]-u_j[k])^2:                                                               */
#define GSI_KERNEL_EXPONENTIAL 0 /* sigma2 * exp(-sqrt(r2))                                    */
#define GSI_KERNEL_GAUSSIAN 1    /* sigma2 * exp(-0.5 * r2)                                    */
#define GSI_KERNEL_POWERLAW 2    /* sigma2 * (1 + r2)^(-beta)                                  */
/* Matern nu = 3/2 and 5/2 (Rasmussen-Williams convention, r = sqrt(r2); exponential is nu = 1/2,
 * Gaussian the limit nu -> infinity) and the spherical model (ell is its range; positive definite
 * for d <= 3).  beta is ignored by these kinds.                                                    */
#define GSI_KERNEL_MATERN32 3    /* sigma2 * (1 + sqrt(3) r) * exp(-sqrt(3) r)                 */
#define GSI_KERNEL_MATERN52 4    /* sigma2 * (1 + sqrt(5) r + 5 r2 / 3) * exp(-sqrt(5) r)       */
#define GSI_KERNEL_SPHERICAL 5   /* sigma2 * (1 - 1.5 r + 0.5 r^3) for r < 1, else 0            */

/* normaliser used between power iterations */
#define GSI_NORMALISER_LU_REF 0 /* partial-pivot LU, unit-lower L kept in LAPACK row order
                                   (reference-faithful: src/RandMatFact.jl:60-61,68-69,72-73)  */
#define GSI_NORMALISER_QR 1     /* Householder TSQR (textbook subspace iteration; NOT parity
                                   with the reference when rank(A) > K+p, SURVEY.md F1)        */

typedef struct gsi_ctx gsi_ctx;
typedef struct gsi_buf gsi_buf;
typedef struct gsi_op gsi_op;

/* ---- library ------------------------------------------------------------------- */
int32_t gsi_version(void);
const char* gsi_last_error_string(void);

/* ---- context --------------------------------------------------------------------- */
/* 128-byte NCCL unique id, generated on rank 0 and broadcast by the host.           */
int32_t gsi_comm_unique_id(void* out128);
/* world == 1: unique_id may be NULL.  Fails with GSI_ERR_NO_DEVICE without sm_100.   */
int32_t gsi_ctx_create(int32_t device, int32_t rank, int32_t world, const void* unique_id128,
                       gsi_ctx** out);
int32_t gsi_ctx_destroy(gsi_ctx* ctx);
int32_t gsi_ctx_sync(gsi_ctx* ctx);
/* the CUDA stream all work of this context is issued on (a cudaStream_t)             */
int32_t gsi_ctx_stream(gsi_ctx* ctx, void** stream_out);
/* kernels launched by the library on this context since the last reset               */
int32_t gsi_ctx_launch_count(gsi_ctx* ctx, int64_t* count_out, int32_t reset);
/* CUDA-event timing of the operator-product (GEMM) kernels, for roofline reporting:
 * enable=1 starts accumulating; query returns accumulated ms, launches, flops.       */
int32_t gsi_ctx_gemm_timing(gsi_ctx* ctx, int32_t enable, double* ms_out, int64_t* launches_out,
                            double* flops_out);

/* CUDA-event time per phase while gemm timing is enabled: ms_out8[0] operator products,
 * [1] LU normaliser, [2] QR/TSQR, [3] small SVD, [4] back-multiplication; [5..7] reserved. */
int32_t gsi_ctx_phase_timing(gsi_ctx* ctx, double* ms_out8, int32_t reset);

/* Tuning knobs (no reference counterpart; results do not depend on them beyond rounding-
 * identical reordering of WHEN tiles are read).  Names:
 *   "kcov.sweep_groups"  power of two: CTA b of the matrix-free product kernel starts its
 *                        k sweep (b mod groups) * separation tiles into X
 *   "kcov.sweep_div"     separation = (#k-tiles / div) if div > 0, (-div) tiles if div < 0
 *   "kcov.l2_hint"       1: evict_last cache hint on the X stream
 *   "kcov.window"        > 0: a CTA runs at most this many epochs ahead of the slowest CTA,
 *                        which keeps the shared X stream L2-resident; 0: unthrottled
 *   "kcov.epoch_shift"   epoch = 2^shift k-tiles of 32 points
 *   "svd.fused"          1 (default): the small Jacobi SVD (<= 512 columns) runs all sweeps in
 *                        one thread-block-cluster launch; 0: one launch per round (same rotations)
 *   "lu.panel"           1 (default): one launch per 16-column LU panel, the panel rows resident in
 *                        shared memory -- a single thread-block cluster for short iterates, a
 *                        cooperative grid otherwise; 2: always the cooperative grid; 0: one launch
 *                        pair per column (same pivots and arithmetic in all three, bit-identical L)
 *   "qr.panel"           the same for the Householder QR panels (0 / 1 / 2)
 * The environment variables GSI_SWEEP="groups,div,hint[,window[,epoch_shift]]" and
 * GSI_OPTIONS="name=value,name=value" set the same knobs at context creation.         */
int32_t gsi_ctx_set_option(gsi_ctx* ctx, const char* name, int64_t value);
int32_t gsi_ctx_get_option(gsi_ctx* ctx, const char* name, int64_t* value_out);

/* ---- device buffers (replace Julia `Matrix{Float64}` temporaries) ----------------- */
int32_t gsi_buf_alloc(gsi_ctx* ctx, int32_t layout, int64_t rows, int64_t cols, gsi_buf** out);
int32_t gsi_buf_free(gsi_buf* buf); /* idempotent on NULL, never throws (Julia finalizer) */
int32_t gsi_buf_dims(const gsi_buf* buf, int64_t* rows, int64_t* cols);
/* Page-locked host memory for arrays that are uploaded repeatedly (the batch of forward runs
 * an rga iteration sketches, src/GeostatInversion.jl:102): uploads from such memory are plain
 * DMA; any other (pageable) source is staged through the context's pinned bounce buffers.
 * Julia shim: `unsafe_wrap(Array, Ptr{Float64}(p), dims)`; release with gsi_host_free.  */
int32_t gsi_host_alloc(gsi_ctx* ctx, int64_t bytes, void** out);
int32_t gsi_host_free(gsi_ctx* ctx, void* ptr); /* ptr NULL: no-op; ctx may be NULL */
/* host (column-major, leading dimension ldh) <-> device, synchronous                 */
int32_t gsi_buf_upload(gsi_buf* buf, const double* host, int64_t ldh);
int32_t gsi_buf_download(const gsi_buf* buf, double* host, int64_t ldh);
/* rows [row0, row0+nrows) of a TALL buffer <-> host block (nrows x cols, ld ldh)     */
int32_t gsi_buf_upload_rows(gsi_buf* buf, int64_t row0, int64_t nrows, const double* host,
                            int64_t ldh);
int32_t gsi_buf_download_rows(const gsi_buf* buf, int64_t row0, int64_t nrows, double* host,
                              int64_t ldh);
int32_t gsi_buf_copy(const gsi_buf* src, gsi_buf* dst);
int32_t gsi_buf_zero(gsi_buf* buf);

/* ---- operators: the duck-typed `A` of randsvd / rangefinder ----------------------- */
/* Dense `A::Matrix` (src/GeostatInversion.jl:63).  `A_local` is a COLMAJOR buffer
 * holding rows [row0, row0+mloc) of the m x n matrix (mloc = buffer rows).           */
int32_t gsi_op_dense(gsi_ctx* ctx, gsi_buf* A_local, int64_t row0, int64_t m_global, gsi_op** out);
/* `LowRankCovMatrix(samples)` (src/lowrank.jl:14-30): samples is a COLMAJOR n x N
 * buffer (column i = field i).  remove_mean != 0 subtracts the sample mean on the
 * device (the constructor's lines 17-27).  Products are S (S' B) / (N-1)
 * (src/lowrank.jl:115-133).                                                          */
int32_t gsi_op_lowrankcov(gsi_ctx* ctx, gsi_buf* samples, int32_t remove_mean, gsi_op** out);
/* The same operator row-sharded over the ranks of a multi-GPU context: samples_local holds the rows
 * [row0, row0 + rows) of the n_global x N sample matrix (the sample mean is per row, hence local);
 * a product exchanges one N x l all-reduce.                                          */
int32_t gsi_op_lowrankcov_sharded(gsi_ctx* ctx, gsi_buf* samples_local, int32_t remove_mean, int64_t row0,
                                  int64_t n_global, gsi_op** out);
/* Matrix-free covariance operator (NEW type with LowRankCovMatrix's method set).
 * coords: host, d x n column-major (point j = coords[j*d .. j*d+d)); ell: d length
 * scales.  This rank applies rows [row0, row0+mloc) of C.  d in {1,2,3}.             */
int32_t gsi_op_kernelcov(gsi_ctx* ctx, int32_t kind, int32_t d, int64_t n, const double* coords,
                         const double* ell, double sigma2, double nugget, double beta,
                         int64_t row0, int64_t mloc, gsi_op** out);
/* The same operator for points on a STRUCTURED GRID (dims[0] fastest, Julia linear index;
 * point coordinates idx .* spacing).  A stationary kernel on a lattice takes only
 * prod(dims) distinct values (one per lattice offset), so they are tabulated once (libm on
 * the host, O(n) memory) and the product kernel fetches C(x_i, x_j) by lattice offset --
 * the n x n matrix is still never materialised and the FP64 pipe is left to the tensor
 * MMAs.  Same products and parity contract as gsi_op_kernelcov.                        */
int32_t gsi_op_kernelcov_grid(gsi_ctx* ctx, int32_t kind, int32_t d, const int64_t* dims,
                              const double* spacing, const double* ell, double sigma2, double nugget,
                              double beta, int64_t row0, int64_t mloc, gsi_op** out);
/* Nested covariance models with rotated (geometric) anisotropy: the same operator for a sum of
 * 1 <= nstruct <= GSI_MODEL_MAX_STRUCTURES structures (e.g. nugget + spherical + exponential, as GSLIB,
 * gstools and SGeMS model a fitted variogram).  Structure s has kinds[s] (GSI_KERNEL_*), a sill
 * sills[s] > 0, ranges ranges[s*d .. s*d+d) > 0 along its principal axes, an orthonormal d x d
 * rotation R_s = rotations + s*d*d (column-major; rotations == NULL: every R_s = I) and betas[s]
 * (power law only; betas == NULL: 1).  With pre(kind) the coordinate scaling of gsi_op_kernelcov
 * (1/sqrt(2) Gaussian, sqrt(3) / sqrt(5) Matern, else 1):
 *   u_s,k(x)  = ((sum_j R_s[k,j] x_j) / ranges[s*d+k]) * pre(kinds[s])       (j = 0..d-1 in order)
 *   r2_s(i,j) = sum_k (u_s,k(x_i) - u_s,k(x_j))^2
 *   C[i,j]    = sum_s sills[s] * k_kinds[s](r2_s) + nugget * (i == j)
 * With R_s = I the coordinates are bit-identical to gsi_op_kernelcov's (x / ell) * pre, and one
 * structure gives gsi_op_kernelcov's operator with sigma2 = sills[0].  Invalid nstruct, kinds,
 * sills (<= 0 or not finite), ranges (<= 0) or rotations (not finite, or max |R'R - I| > 1e-12):
 * GSI_ERR_INVALID_ARGUMENT; d outside 1..3: GSI_ERR_UNSUPPORTED.                                */
#define GSI_MODEL_MAX_STRUCTURES 4
int32_t gsi_op_kernelcov_model(gsi_ctx* ctx, int32_t d, int64_t n, const double* coords, int32_t nstruct,
                               const int32_t* kinds, const double* sills, const double* ranges,
                               const double* rotations, const double* betas, double nugget,
                               int64_t row0, int64_t mloc, gsi_op** out);
/* The nested model on a structured grid (dims / spacing as gsi_op_kernelcov_grid): the whole model is
 * tabulated once on the host.  Without rotations (or d = 1) the table is indexed by |lattice offset|;
 * a rotated model is not symmetric in each axis, so its table covers the signed offsets, folded by
 * k(delta) = k(-delta): (2 dims[0] - 1) (2 dims[1] - 1) dims[2] entries in 3-D, (2 dims[0] - 1) dims[1]
 * in 2-D (GSI_ERR_UNSUPPORTED at 2^31 entries or more).                                           */
int32_t gsi_op_kernelcov_model_grid(gsi_ctx* ctx, int32_t d, const int64_t* dims, const double* spacing,
                                    int32_t nstruct, const int32_t* kinds, const double* sills,
                                    const double* ranges, const double* rotations, const double* betas,
                                    double nugget, int64_t row0, int64_t mloc, gsi_op** out);
/* Cross-covariance between two point sets (kriging C(T, S) w, Q H' = C(grid, obs) of point observations):
 * m x n matrix C[i,j] = sum_s sills[s] k_kinds[s](r2_s(t_i, s_j)), t_i = targets[:, i], s_j = sources[:, j] (host,
 * d x m and d x n column-major; model arguments and coordinate scaling exactly as gsi_op_kernelcov_model).  No nugget
 * term: T and S are different sets.  This rank owns target rows [row0, row0 + mloc).  Not symmetric: gsi_op_apply
 * trans = 0 gives this rank's rows of C X (X: all n rows), trans = 1 gives all n rows of C' X summed over ranks (X: all
 * m rows), as for gsi_op_dense; gsi_op_size reports (m, n).  m < 1, n < 1, a bad row block or a missing pointer:
 * GSI_ERR_INVALID_ARGUMENT; d outside 1..3: GSI_ERR_UNSUPPORTED.                                     */
int32_t gsi_op_kernelcov_cross(gsi_ctx* ctx, int32_t d, int64_t m, const double* targets, int64_t n,
                               const double* sources, int32_t nstruct, const int32_t* kinds, const double* sills,
                               const double* ranges, const double* rotations, const double* betas,
                               int64_t row0, int64_t mloc, gsi_op** out);
/* The same for points that are nodes of one structured grid (dims / spacing as gsi_op_kernelcov_grid), given by
 * 0-based linear indices (dims[0] fastest); target_idx == NULL: all prod(dims) nodes in order (m must equal it),
 * likewise source_idx.  Same table as gsi_op_kernelcov_model_grid (signed offsets when a structure is rotated).
 * An index outside 0 .. prod(dims) - 1, or a NULL index list with m (n) != prod(dims): GSI_ERR_INVALID_ARGUMENT;
 * a table of 2^31 entries or more: GSI_ERR_UNSUPPORTED.                                             */
int32_t gsi_op_kernelcov_cross_grid(gsi_ctx* ctx, int32_t d, const int64_t* dims, const double* spacing,
                                    int64_t m, const int64_t* target_idx, int64_t n, const int64_t* source_idx,
                                    int32_t nstruct, const int32_t* kinds, const double* sills, const double* ranges,
                                    const double* rotations, const double* betas, int64_t row0, int64_t mloc,
                                    gsi_op** out);
int32_t gsi_op_free(gsi_op* op);
/* size(A) (src/RandMatFact.jl:52-53, src/lowrank.jl:50-60)                           */
int32_t gsi_op_size(const gsi_op* op, int64_t* m, int64_t* n);
/* `A * X` (trans=0, src/RandMatFact.jl:55,70) or `A' * X` (trans=1, :67; and
 * `(Q' * A)' = A' * Q`, :85).  X: TALL, all n (resp. m) rows.  Y: TALL, this rank's
 * rows of the result (for trans=1 on a row-sharded dense A or cross-covariance the partial
 * products are summed over ranks and every rank receives all n rows).                */
int32_t gsi_op_apply(gsi_op* op, int32_t trans, const gsi_buf* X, gsi_buf* Y);

/* ---- factorisation building blocks (exposed for tests and for the shim) ----------- */
/* `F = lu(Y); Y = F.L` (src/RandMatFact.jl:60-61): in place, unpermuted L.           */
int32_t gsi_lu_L(gsi_ctx* ctx, gsi_buf* Y);
/* thin orthonormal basis of range(Y), replacing `Matrix(qr(Y, Val(true)).Q)`
 * (:57-58,75-76; range-equivalent, SURVEY.md F2).  R_host (l x l col-major) optional. */
int32_t gsi_qr_thinQ(gsi_ctx* ctx, gsi_buf* Y, double* R_host, int64_t ldr);
/* SVD of a small l x l host matrix (col-major) on the device (one-sided Jacobi):
 * U overwrites M, sigma descending.  Used for `svd(B)` (:86) after TSQR(B').         */
int32_t gsi_svd_small(gsi_ctx* ctx, double* M_host, int64_t ldm, int64_t l, double* sigma_host);

/* ---- algorithms -------------------------------------------------------------------- */
/* rangefinder(A, l, q) (src/RandMatFact.jl:50-80).  Omega: TALL n x l (all rows on
 * every rank).  Q_out: TALL, this rank's mloc rows x l.                               */
int32_t gsi_rangefinder_fixed(gsi_op* op, const gsi_buf* Omega, int64_t q, int32_t normaliser,
                              gsi_buf* Q_out);
/* randsvd(A, K, p, q) (src/RandMatFact.jl:83-90).  Omega: TALL n x (K+p).
 * Z_out: TALL, this rank's rows of Z = V * sqrt(diag(S[1:K], 0)) (n x (K+p), last p
 * columns exactly zero).  S_host: K+p singular values of Q'A (may be NULL).           */
int32_t gsi_randsvd(gsi_op* op, const gsi_buf* Omega, int64_t K, int64_t p, int64_t q,
                    int32_t normaliser, gsi_buf* Z_out, double* S_host);
/* rangefinder(A; epsilon, r) (src/RandMatFact.jl:15-48), dense square A, 1 GPU.
 * Omega0: TALL n x r replaces randn(n, r) (:20); omegas: n x maxvec, column t replaces
 * the t-th randn!(omega) (:36).  Q_out: n x maxvec; *j_out = basis size (columns beyond
 * it are zero).  omegas and Q_out may be TALL (maxvec <= 256) or COLMAJOR (any maxvec,
 * e.g. the reference's implicit bound min(m, n)).
 * Returns GSI_ERR_NO_CONVERGENCE if maxvec vectors did not reach epsilon.             */
int32_t gsi_rangefinder_adaptive(gsi_op* op, const gsi_buf* Omega0, const gsi_buf* omegas,
                                 double epsilon, int64_t r, gsi_buf* Q_out, int64_t* j_out);
/* OPT-IN blocked variant of the adaptive range finder (no reference counterpart; NOT the
 * parity mode): the random vectors are consumed `block` (<= 256) at a time, so A is read
 * once per block by a tensor-core GEMM instead of once per vector, the block is projected
 * against the basis (block Gram-Schmidt, twice) and orthonormalised by Householder QR; the
 * reference's stopping estimator (:26) is evaluated on the block's fresh probes.  Same
 * error bound, basis size rounded up to the block, different basis than the reference's.
 * omegas / Q_out as above (TALL or COLMAJOR, n x maxvec).                               */
int32_t gsi_rangefinder_adaptive_blocked(gsi_op* op, const gsi_buf* omegas, double epsilon, int64_t block,
                                         gsi_buf* Q_out, int64_t* j_out);
/* eig_nystrom(A, Q) (src/RandMatFact.jl:92-102): U_out TALL n x l, Sigma_host l.      */
int32_t gsi_eig_nystrom(gsi_op* op, const gsi_buf* Q, gsi_buf* U_out, double* Sigma_host);

/* FFTRF.powerlaw_structuredgrid (src/FFTRF.jl:83-100) for a batch of fields, on the device -- the
 * sampler behind getxis(samplefield, numfields, ...) (src/GeostatInversion.jl:29-38).  dim in {2, 3};
 * Ns[dim] grid sizes (each <= 1024).  phi: COLMAJOR prod(2*Ns) x nfields, column f = the `randn(size(S))`
 * of field f (:75) in Julia's linear order of the (2 Ns[2], 2 Ns[1] [, 2 Ns[3]]) array (:45,52).
 * samples: COLMAJOR prod(Ns) x nfields, column f = vec(field f) (mean k0, corrected std dk) -- ready for
 * gsi_op_lowrankcov without a host round trip.                                                    */
int32_t gsi_fftrf_powerlaw(gsi_ctx* ctx, int32_t dim, const int64_t* Ns, double k0, double dk, double beta,
                           const gsi_buf* phi, gsi_buf* samples);

/* ---- PCGA helpers (src/lsqr.jl:35-63, src/lowrank.jl:83-97, GeostatInversion.jl:101-103) */
/* v = [R xs + E (E' xs) + HX x_end ; HX . xs]  (PCGALowRankMatrix mul!, lowrank.jl:83-97)
 * E: host nobs x K col-major (columns = etas), HX: nobs, Rdiag: nobs (diagonal R) or
 * Rdense nobs x nobs col-major (exactly one non-NULL), x, v: nobs+1.                  */
int32_t gsi_pcga_lowrank_matvec(gsi_ctx* ctx, int64_t nobs, int64_t K, const double* E, int64_t lde,
                                const double* HX, const double* Rdiag, const double* Rdense,
                                int64_t ldr, const double* x, double* v);
/* x = IterativeSolvers.lsqr(PCGALowRankMatrix(etas, HX, R), b) (src/lsqr.jl:53-54),
 * fully on device.  atol/btol/conlim <= 0 select the IterativeSolvers defaults
 * (sqrt(eps), sqrt(eps), 1/sqrt(eps)); maxiter <= 0 selects nobs+1.                   */
int32_t gsi_pcga_lsqr_solve(gsi_ctx* ctx, int64_t nobs, int64_t K, const double* E, int64_t lde,
                            const double* HX, const double* Rdiag, const double* Rdense,
                            int64_t ldr, const double* b, double atol, double btol, double conlim,
                            int64_t maxiter, double* x_out, int64_t* itn_out, int32_t* istop_out);
/* x = pinv([HQH + R, HX; HX', 0]) * b with HQH = sum_i eta_i eta_i' (pcgadirect's dense solve,
 * src/direct.jl:49-58), fully on device: HQH = E E' on the tensor-core GEMM, SVD by one-sided
 * Jacobi, Julia's pinv cut-off (singular values <= eps * (nobs+1) * sigma_max are dropped).
 * Arguments as in gsi_pcga_lsqr_solve; rank_out (optional) = number of singular values kept. */
int32_t gsi_pcga_direct_solve(gsi_ctx* ctx, int64_t nobs, int64_t K, const double* E, int64_t lde,
                              const double* HX, const double* Rdiag, const double* Rdense,
                              int64_t ldr, const double* b, double* x_out, int64_t* rank_out);
/* s = X*beta + sum_i xis[i] * dot(eta_i, xi_bar) (src/lsqr.jl:55-61).
 * Zk: TALL n x K (the xis as columns, device resident).  s_host: n.                   */
int32_t gsi_pcga_update(gsi_ctx* ctx, const gsi_buf* Zk, int64_t K, const double* Xmean,
                        const double* E, int64_t lde, int64_t nobs, const double* x,
                        double* s_host);
/* paramstorun batch (src/lsqr.jl:37-43): P = [s + delta*xi_1 .. s + delta*xi_K,
 * s + delta*X, s + delta*s, s]  as a TALL n x (K+3) buffer.                           */
int32_t gsi_pcga_paramstorun(gsi_ctx* ctx, const gsi_buf* Zk, int64_t K, const double* s,
                             const double* Xmean, double delta, gsi_buf* P_out);
/* out = S * V for the rga sketch (GeostatInversion.jl:102, `x->S*h(x)` batched and
 * `S*y`): S COLMAJOR Nred x nobs, V TALL nobs x c, out TALL Nred x c.                 */
int32_t gsi_sketch_apply(gsi_ctx* ctx, gsi_buf* S, const gsi_buf* V, gsi_buf* out);
/* out = S * diag(Rdiag) * S' (`S*R*S'`, GeostatInversion.jl:102), host Nred x Nred.   */
int32_t gsi_sketch_cov(gsi_ctx* ctx, gsi_buf* S, const double* Rdiag, double* out_host,
                       int64_t ldo);

#ifdef __cplusplus
}
#endif
#endif /* GSI_B200_H */
