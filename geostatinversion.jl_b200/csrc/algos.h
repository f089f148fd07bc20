#pragma once
#include "common.cuh"
#include <memory>

namespace gsi {

struct BufDeleter { void operator()(gsi_buf* b) const; };
typedef std::unique_ptr<gsi_buf, BufDeleter> BufPtr;

BufPtr make_buf(gsi_ctx* ctx, int32_t layout, int64_t rows, int64_t cols);
void op_apply(gsi_op* op, int trans, const gsi_buf* X, gsi_buf* Y);
bool op_symmetric(const gsi_op* op);
void resolve_gemm_timing(gsi_ctx* ctx);
BufPtr X_view_for_dense(gsi_op* op, int trans, const gsi_buf* X);
void tsqr_thinQ(gsi_op* op, gsi_buf* Y, bool sharded, double* Rdev);
void rangefinder_fixed(gsi_op* op, const gsi_buf* Omega, int64_t q, int normaliser, gsi_buf* Q_out);
void randsvd(gsi_op* op, const gsi_buf* Omega, int64_t K, int64_t p, int64_t q, int normaliser, gsi_buf* Z_out,
             double* S_host);

}  // namespace gsi
