// Algorithm drivers: operator application, rangefinder(A, l, q), randsvd(A, K, p, q)
// (reference src/RandMatFact.jl:50-90), TSQR across ranks, eig_nystrom (:92-102) and
// the adaptive range finder (:15-48).  Everything is enqueued on the context stream;
// host synchronisation happens only where a scalar decision is needed (LU singularity
// flag, Jacobi convergence, adaptive stopping test).
#include "common.cuh"
#include "algos.h"
#include <cmath>
#include <memory>

namespace gsi {

BufPtr make_buf(gsi_ctx* ctx, int32_t layout, int64_t rows, int64_t cols) {
    GSI_REQUIRE(rows >= 0 && cols >= 1, GSI_ERR_INVALID_ARGUMENT, "buffer needs rows >= 0 and cols >= 1");
    BufPtr b(new gsi_buf());
    b->ctx = ctx; b->layout = layout; b->rows = rows; b->cols = cols;
    if (layout == GSI_LAYOUT_TALL) {
        GSI_REQUIRE(cols <= kMaxWideCols, GSI_ERR_UNSUPPORTED, "TALL buffers hold at most 1024 columns");
        b->ld = ld_for_cols(cols);
        b->rows_alloc = round_up(rows > 0 ? rows : 1, kRowPad);
    } else if (layout == GSI_LAYOUT_COLMAJOR) {
        b->ld = round_up(rows > 0 ? rows : 1, 2);          // 16-byte column pitch for TMA
        b->rows_alloc = b->ld;
    } else {
        throw Error(GSI_ERR_INVALID_ARGUMENT, "unknown buffer layout");
    }
    b->d = static_cast<double*>(pool_alloc(ctx, b->bytes()));
    ctx_retain(ctx);
    GSI_CUDA(cudaMemsetAsync(b->d, 0, b->bytes(), ctx->stream));
    return b;
}

void BufDeleter::operator()(gsi_buf* b) const {
    if (!b) return;
    gsi_ctx* bctx = b->ctx;
    const bool owned = b->owns && b->d;
    if (owned) pool_free(bctx, b->d, b->bytes());
    delete b;
    if (owned) ctx_release(bctx);
}

// ------------------------------------------------------------------ operator application
void phase_begin(gsi_ctx* ctx) {
    if (!ctx->time_gemm) return;
    if (ctx->ev_used + 2 > ctx->ev_pool.size()) {
        for (int i = 0; i < 64; ++i) {
            cudaEvent_t e;
            GSI_CUDA(cudaEventCreate(&e));
            ctx->ev_pool.push_back(e);
        }
    }
    GSI_CUDA(cudaEventRecord(ctx->ev_pool[ctx->ev_used], ctx->stream));
}
void phase_end(gsi_ctx* ctx, int phase) {
    if (!ctx->time_gemm) return;
    GSI_CUDA(cudaEventRecord(ctx->ev_pool[ctx->ev_used + 1], ctx->stream));
    ctx->ev_used += 2;
    ctx->ev_phase.push_back(phase);
}
static void timed_begin(gsi_ctx* ctx) { phase_begin(ctx); }
static void timed_end(gsi_ctx* ctx, double flops, int nlaunch) {
    if (!ctx->time_gemm) return;
    phase_end(ctx, PH_GEMM);
    ctx->gemm_launches += nlaunch;
    ctx->gemm_flops_accum += flops;
}
// resolve the recorded event pairs into gemm_ms_accum / phase_ms
void resolve_gemm_timing(gsi_ctx* ctx) {
    for (size_t i = 0, j = 0; i + 1 < ctx->ev_used; i += 2, ++j) {
        GSI_CUDA(cudaEventSynchronize(ctx->ev_pool[i + 1]));
        float ms = 0.f;
        GSI_CUDA(cudaEventElapsedTime(&ms, ctx->ev_pool[i], ctx->ev_pool[i + 1]));
        const int ph = ctx->ev_phase[j];
        ctx->phase_ms[ph] += ms;
        if (ph == PH_GEMM) ctx->gemm_ms_accum += ms;
    }
    ctx->ev_used = 0;
    ctx->ev_phase.clear();
}

// Y = op(A) X.   X: all rows of the operand on this rank.  Output distribution:
//   kernelcov / lowrankcov (symmetric): this rank's row block (SHARDED when world > 1)
//   dense and cross-covariance, trans = 0: this rank's row block;  trans = 1: all n rows, summed over ranks
void op_apply(gsi_op* op, int trans, const gsi_buf* X, gsi_buf* Y) {
    gsi_ctx* ctx = op->ctx;
    switch (op->type) {
        case OP_KERNELCOV: {
            timed_begin(ctx);
            kcov_apply(op, 0, X, Y);
            timed_end(ctx, 2.0 * (double)op->mloc * (double)op->n * (double)X->cols, 1);
            break;
        }
        case OP_KERNELCROSS: {
            // trans = 1 on several ranks: this rank's operand rows go to a zero-padded buffer of their own -- in a view
            // into the full operand, the rows past mloc that the last k-tile's padded columns multiply are the next
            // rank's data
            BufPtr xl;
            const gsi_buf* Xk = X;
            if (trans && ctx->world > 1) {
                GSI_REQUIRE(X->rows == op->m, GSI_ERR_DIMENSION_MISMATCH, "cross-covariance C'X: X must hold all m rows");
                xl = make_buf(ctx, GSI_LAYOUT_TALL, op->mloc, X->cols);
                GSI_REQUIRE(xl->ld == X->ld, GSI_ERR_INVALID_ARGUMENT, "cross-covariance C'X: bad pitch");
                GSI_CUDA(cudaMemcpyAsync(xl->d, X->d + op->row0 * X->ld, (size_t)op->mloc * X->ld * 8,
                                         cudaMemcpyDeviceToDevice, ctx->stream));
                Xk = xl.get();
            }
            timed_begin(ctx);
            kcov_apply(op, trans, Xk, Y);
            timed_end(ctx, 2.0 * (double)op->mloc * (double)op->n * (double)X->cols, 1);
            if (trans && ctx->world > 1) comm_allreduce_sum(ctx, Y->d, (size_t)Y->rows_alloc * Y->ld);
            break;
        }
        case OP_DENSE: {
            timed_begin(ctx);
            dense_apply(ctx, op->A, trans, X_view_for_dense(op, trans, X).get(), Y, 1.0);
            timed_end(ctx, 2.0 * (double)op->A->rows * (double)op->A->cols * (double)X->cols, 1);
            if (trans && ctx->world > 1) comm_allreduce_sum(ctx, Y->d, (size_t)Y->rows_alloc * Y->ld);
            break;
        }
        case OP_LOWRANKCOV: {
            // S (S' X) / (N-1)   (reference src/lowrank.jl:115-121 as two skinny GEMMs).  Row-sharded: this rank
            // holds the rows [row0, row0 + mloc) of S; T = sum over ranks of S_g' X_g is one small (N x l)
            // all-reduce, the second product is local.
            const int64_t N = op->A->cols;
            if (!op->tmpT || op->tmpT->cols != X->cols) {
                if (op->tmpT) BufDeleter()(op->tmpT);
                op->tmpT = make_buf(ctx, GSI_LAYOUT_TALL, N, X->cols).release();
            }
            gsi_buf xv = *X;
            xv.owns = false;
            if (ctx->world > 1) {
                GSI_REQUIRE(X->rows == op->n, GSI_ERR_DIMENSION_MISMATCH, "lowrankcov: X must hold all n rows");
                xv.d = X->d + op->row0 * X->ld;
                xv.rows = op->mloc;
            }
            timed_begin(ctx);
            dense_apply(ctx, op->A, 1, &xv, op->tmpT, 1.0);
            if (ctx->world > 1) comm_allreduce_sum(ctx, op->tmpT->d, (size_t)op->tmpT->rows_alloc * op->tmpT->ld);
            dense_apply(ctx, op->A, 0, op->tmpT, Y, op->scale);
            timed_end(ctx, 4.0 * (double)op->A->rows * (double)N * (double)X->cols, 2);
            break;
        }
    }
}

// dense trans=1 on a row-sharded A consumes only this rank's rows of X
BufPtr X_view_for_dense(gsi_op* op, int trans, const gsi_buf* X) {
    BufPtr v(new gsi_buf(*X));
    v->owns = false;
    if (trans && op->ctx->world > 1) {
        GSI_REQUIRE(X->rows == op->m, GSI_ERR_DIMENSION_MISMATCH, "dense A'X: X must hold all m rows");
        v->d = X->d + op->row0 * X->ld;
        v->rows = op->mloc;
    }
    return v;
}

// ------------------------------------------------------------------ distribution helpers
// local block (mloc x l) -> full (m x l) on every rank
void gather_rows(gsi_op* op, const gsi_buf* loc, gsi_buf* full) {
    gsi_ctx* ctx = op->ctx;
    GSI_REQUIRE(loc->ld == full->ld, GSI_ERR_INVALID_ARGUMENT, "gather_rows: pitch mismatch");
    GSI_CUDA(cudaMemcpyAsync(full->d + op->row0 * full->ld, loc->d, (size_t)op->mloc * loc->ld * 8,
                             cudaMemcpyDeviceToDevice, ctx->stream));
    if (ctx->world > 1) {
        std::vector<int64_t> off(ctx->world), cnt(ctx->world);
        for (int r = 0; r < ctx->world; ++r) {
            off[r] = op->part[r] * full->ld;
            cnt[r] = (op->part[r + 1] - op->part[r]) * full->ld;
        }
        comm_allgatherv(ctx, full->d, off.data(), cnt.data());
    }
}

bool op_symmetric(const gsi_op* op) { return op->type != OP_DENSE && op->type != OP_KERNELCROSS; }

// In-place LU normalisation of an iterate all of whose rows are on this device.
static void normalise_lu(gsi_op* op, gsi_buf* Y) {
    gsi_ctx* ctx = op->ctx;
    phase_begin(ctx);
    struct End { gsi_ctx* c; ~End() { try { phase_end(c, PH_LU); } catch (...) {} } } end_{ctx};
    lu_L_inplace(ctx, Y);
}

// TSQR: local Householder QR, all-gather of the R factors, redundant QR of the stack,
// local Q <- Q_local * Qtilde_block.  Rdev (l x l col-major, device) optional.
void tsqr_thinQ(gsi_op* op, gsi_buf* Y, bool sharded, double* Rdev) {
    gsi_ctx* ctx = op->ctx;
    phase_begin(ctx);
    struct End { gsi_ctx* c; ~End() { try { phase_end(c, PH_QR); } catch (...) {} } } end_{ctx};
    const int l = (int)Y->cols;
    if (!(sharded && ctx->world > 1)) {
        qr_thinQ_inplace(ctx, Y, Rdev);
        return;
    }
    const int G = ctx->world;
    // [G][l*l] column-major blocks (+ my own), from the pooled allocator (no cudaMalloc/cudaFree sync)
    const size_t rall_bytes = (size_t)(G + 1) * l * l * sizeof(double);
    double* Rall = static_cast<double*>(pool_alloc(ctx, rall_bytes));
    struct PoolGuard { gsi_ctx* c; void* p; size_t b; ~PoolGuard() { pool_free(c, p, b); } } guard{ctx, Rall, rall_bytes};
    double* Rmine = Rall + (size_t)G * l * l;
    // a rank that owns fewer than l rows factors its block padded with zero rows (same R)
    BufPtr padded;
    gsi_buf* Yl = Y;
    if (Y->rows < l) {
        padded = make_buf(ctx, GSI_LAYOUT_TALL, l, l);
        GSI_CUDA(cudaMemcpyAsync(padded->d, Y->d, (size_t)Y->rows * Y->ld * 8, cudaMemcpyDeviceToDevice, ctx->stream));
        Yl = padded.get();
    }
    qr_thinQ_inplace(ctx, Yl, Rmine);
    comm_allgather(ctx, Rmine, Rall, (size_t)l * l * sizeof(double));
    // stack (G*l x l) as a TALL buffer
    BufPtr stack = make_buf(ctx, GSI_LAYOUT_TALL, (int64_t)G * l, l);
    for (int r = 0; r < G; ++r) {
        gsi_buf view = *stack;
        view.owns = false; view.rows = l; view.rows_alloc = l;
        view.d = stack->d + (size_t)r * l * stack->ld;
        small_cm_to_tall(ctx, Rall + (size_t)r * l * l, l, l, l, &view);
    }
    qr_thinQ_inplace(ctx, stack.get(), Rdev);
    // my block of Qtilde (l x l) as its own TALL buffer (needs zero padded rows)
    BufPtr qt = make_buf(ctx, GSI_LAYOUT_TALL, l, l);
    GSI_CUDA(cudaMemcpyAsync(qt->d, stack->d + (size_t)ctx->rank * l * stack->ld, (size_t)l * stack->ld * 8,
                             cudaMemcpyDeviceToDevice, ctx->stream));
    BufPtr tmp = make_buf(ctx, GSI_LAYOUT_TALL, Yl->rows, l);
    tall_times_small(ctx, Yl, qt.get(), tmp.get());
    GSI_CUDA(cudaMemcpyAsync(Y->d, tmp->d, (size_t)Y->rows * Y->ld * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    // no host synchronisation: the temporaries go back to the stream-ordered pool of this context
}

// Multi-GPU LU normalisation: the next product needs the whole iterate on every rank anyway, so it
// is gathered BEFORE the LU and every rank factors all rows redundantly (deterministic kernels:
// identical factors everywhere, identical to the single-GPU result) -- no per-column pivot
// exchange.  The gathered, normalised iterate is then the next product's operand as it stands.
static void replicate(gsi_op* op, Iterate& it) {
    gsi_ctx* ctx = op->ctx;
    if (!(it.sharded && ctx->world > 1)) return;
    BufPtr full = make_buf(ctx, GSI_LAYOUT_TALL, op->m, it.buf->cols);
    gather_rows(op, it.buf.get(), full.get());
    it.buf = std::move(full);
    it.sharded = false;
}

static void normalise(gsi_op* op, Iterate& it, int normaliser) {
    if (normaliser == GSI_NORMALISER_LU_REF) {
        replicate(op, it);
        normalise_lu(op, it.buf.get());
    } else {
        tsqr_thinQ(op, it.buf.get(), it.sharded, nullptr);
    }
}

// One product step of the iteration.  `cur` holds the current iterate in distribution
// `cur_sharded`; returns the product in `out` and its distribution.
static Iterate apply_step(gsi_op* op, int trans, Iterate& cur, BufPtr& full_scratch) {
    gsi_ctx* ctx = op->ctx;
    const int64_t l = cur.buf->cols;
    const int64_t in_rows = trans ? op->m : op->n;            // rows of the operand
    const gsi_buf* X = cur.buf.get();
    if (cur.sharded && ctx->world > 1) {
        if (!full_scratch || full_scratch->rows != in_rows || full_scratch->cols != l)
            full_scratch = make_buf(ctx, GSI_LAYOUT_TALL, in_rows, l);
        gather_rows(op, cur.buf.get(), full_scratch.get());
        X = full_scratch.get();
    }
    GSI_REQUIRE(X->rows == in_rows, GSI_ERR_DIMENSION_MISMATCH, "operator product: operand rows");
    Iterate out;
    const bool sym = op_symmetric(op);
    if (sym || !trans) {
        out.buf = make_buf(ctx, GSI_LAYOUT_TALL, op->mloc, l);
        out.sharded = ctx->world > 1;
    } else {
        out.buf = make_buf(ctx, GSI_LAYOUT_TALL, op->n, l);   // dense A'X: replicated
        out.sharded = false;
    }
    op_apply(op, sym ? 0 : trans, X, out.buf.get());
    return out;
}

// rangefinder(A, l, q): returns the orthonormal basis as an Iterate (sharded when world > 1)
static Iterate rangefinder_fixed_impl(gsi_op* op, const gsi_buf* Omega, int64_t q, int normaliser) {
    gsi_ctx* ctx = op->ctx;
    if (q < 0)
        throw Error(GSI_ERR_NEGATIVE_ITERATIONS,
                    "parameter numiterations should be positive, but numiterations=" + std::to_string(q));
    GSI_REQUIRE(Omega->layout == GSI_LAYOUT_TALL, GSI_ERR_INVALID_ARGUMENT, "Omega must be a TALL buffer");
    GSI_REQUIRE(Omega->rows == op->n, GSI_ERR_DIMENSION_MISMATCH, "Omega must have size(A, 2) rows");
    const int64_t l = Omega->cols;
    GSI_REQUIRE(l <= op->n && l <= op->m, GSI_ERR_UNSUPPORTED, "l must not exceed min(size(A))");
    BufPtr full_scratch;
    Iterate cur;
    lu_reset_flag(ctx);
    {
        // Y = A * Omega                                         (reference :55)
        Iterate om;
        om.buf.reset(new gsi_buf(*Omega));
        om.buf->owns = false;
        om.sharded = false;
        cur = apply_step(op, 0, om, full_scratch);
    }
    if (q == 0) {                                                // :56-58
        tsqr_thinQ(op, cur.buf.get(), cur.sharded, nullptr);
        return cur;
    }
    normalise(op, cur, normaliser);                              // :60-61
    for (int64_t i = 1; i <= q; ++i) {
        Iterate t = apply_step(op, 1, cur, full_scratch);        // Q = A' * Q     :67
        normalise(op, t, normaliser);                            // :68-69
        cur = apply_step(op, 0, t, full_scratch);                // Q = A * Q      :70
        if (i < q) normalise(op, cur, normaliser);               // :72-73
        else tsqr_thinQ(op, cur.buf.get(), cur.sharded, nullptr);           // :75-76
    }
    (void)ctx;
    return cur;
}

void deliver(gsi_op* op, Iterate& res, gsi_buf* out) {
    gsi_ctx* ctx = op->ctx;
    GSI_REQUIRE(out->layout == GSI_LAYOUT_TALL && out->cols == res.buf->cols, GSI_ERR_DIMENSION_MISMATCH,
                "output buffer: wrong layout or column count");
    if (res.sharded && ctx->world > 1) {
        if (out->rows == op->m) gather_rows(op, res.buf.get(), out);           // full result on every rank
        else if (out->rows == op->mloc) tall_copy(ctx, res.buf.get(), out);    // this rank's block
        else throw Error(GSI_ERR_DIMENSION_MISMATCH, "output buffer: rows match neither the local block nor the full result");
    } else {
        if (out->rows == res.buf->rows) tall_copy(ctx, res.buf.get(), out);
        else if (ctx->world > 1 && out->rows == op->mloc && res.buf->rows == op->m)
            GSI_CUDA(cudaMemcpyAsync(out->d, res.buf->d + op->row0 * res.buf->ld, (size_t)op->mloc * out->ld * 8,
                                     cudaMemcpyDeviceToDevice, ctx->stream));
        else throw Error(GSI_ERR_DIMENSION_MISMATCH, "output buffer: wrong row count");
    }
    lu_check_singular(ctx);          // the one host synchronisation of the algorithm (SingularException of any LU)
    svd_check(ctx);                  // ... and the Jacobi convergence verdict (stream already idle)
}

void rangefinder_fixed(gsi_op* op, const gsi_buf* Omega, int64_t q, int normaliser, gsi_buf* Q_out) {
    Iterate Q = rangefinder_fixed_impl(op, Omega, q, normaliser);
    deliver(op, Q, Q_out);
}

__global__ void scale_cols_kernel(const double* __restrict__ U, const double* __restrict__ sigma, int l, int K,
                                  double* __restrict__ out) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= l * l) return;
    const int c = idx / l;
    out[idx] = (c < K) ? U[idx] * sqrt(sigma[c]) : 0.0;
}

void randsvd(gsi_op* op, const gsi_buf* Omega, int64_t K, int64_t p, int64_t q, int normaliser, gsi_buf* Z_out,
             double* S_host) {
    gsi_ctx* ctx = op->ctx;
    GSI_REQUIRE(K >= 1 && p >= 0, GSI_ERR_INVALID_ARGUMENT, "randsvd: K >= 1 and p >= 0 required");
    GSI_REQUIRE(Omega->cols == K + p, GSI_ERR_DIMENSION_MISMATCH, "randsvd: Omega must have K+p columns");
    const int l = (int)(K + p);
    Iterate Q = rangefinder_fixed_impl(op, Omega, q, normaliser);          // :84
    BufPtr full_scratch;
    Iterate Bt = apply_step(op, 1, Q, full_scratch);                      // B' = A'Q    (:85)
    Q.buf.reset();
    full_scratch.reset();
    // svd(B) (:86): B' = Q_B R_B,  R_B = U_R S V_R'  =>  V = Q_B U_R
    const size_t small_bytes = ((size_t)3 * l * l + l) * sizeof(double);   // R | U | Usc | sigma
    double* small = static_cast<double*>(pool_alloc(ctx, small_bytes));
    struct PoolGuard { gsi_ctx* c; void* p; size_t b; ~PoolGuard() { pool_free(c, p, b); } } guard{ctx, small, small_bytes};
    double* R = small;
    double* U = small + (size_t)l * l;
    double* Usc = small + (size_t)2 * l * l;
    double* sigma = small + (size_t)3 * l * l;
    tsqr_thinQ(op, Bt.buf.get(), Bt.sharded, R);
    phase_begin(ctx);
    svd_small(ctx, R, l, U, sigma, /*defer_check=*/true);
    phase_end(ctx, PH_SVD);
    // Z = V * Diagonal(sqrt.([S[1:K]; zeros(p)]))                        (:87-88)
    scale_cols_kernel<<<(l * l + 255) / 256, 256, 0, ctx->stream>>>(U, sigma, l, (int)K, Usc);
    GSI_CUDA(cudaGetLastError());
    count_launch(ctx);
    BufPtr Mt = make_buf(ctx, GSI_LAYOUT_TALL, l, l);
    small_cm_to_tall(ctx, Usc, l, l, l, Mt.get());
    Iterate Z;
    Z.buf = make_buf(ctx, GSI_LAYOUT_TALL, Bt.buf->rows, l);
    Z.sharded = Bt.sharded;
    phase_begin(ctx);
    tall_times_small(ctx, Bt.buf.get(), Mt.get(), Z.buf.get());
    phase_end(ctx, PH_BACKMUL);
    if (S_host) {
        GSI_CUDA(cudaMemcpyAsync(S_host, sigma, (size_t)l * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    }
    deliver(op, Z, Z_out);
}

}  // namespace gsi
