// Shared host-side declarations of the gsi_b200 library (context, device
// buffers, operators, error plumbing).  Not part of the public ABI: the ABI is
// include/gsi_b200.h.
#pragma once
#include <cuda_runtime.h>
#include <cuda.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>
#include <stdexcept>
#include "../../include/gsi_b200.h"

namespace gsi {

void set_last_error(const std::string& msg);

struct Error : public std::runtime_error {
    int32_t code;
    Error(int32_t c, const std::string& m) : std::runtime_error(m), code(c) {}
};

#define GSI_CUDA(expr)                                                                   \
    do {                                                                                 \
        cudaError_t _e = (expr);                                                         \
        if (_e != cudaSuccess)                                                           \
            throw gsi::Error(GSI_ERR_CUDA, std::string("CUDA error: ") +                 \
                                               cudaGetErrorString(_e) + " at " __FILE__ ":" + \
                                               std::to_string(__LINE__) + " (" #expr ")");   \
    } while (0)

#define GSI_REQUIRE(cond, code, msg)                       \
    do {                                                   \
        if (!(cond)) throw gsi::Error((code), (msg));      \
    } while (0)

inline int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

constexpr int kRowPad = 64;        // tall buffers: allocated rows are a multiple of this
constexpr int kMaxCols = 256;      // widest tall iterate a single GEMM pass handles
constexpr int kMaxWideCols = 1024; // widest tall iterate at all: wider than kMaxCols goes through the products in 256-column chunks
constexpr int kPxchMaxCtas = 256;   // panel kernels: CTAs of one cooperative launch
constexpr int kPxchRec = 40;        // doubles per published record
constexpr size_t kPxchDoubles = (size_t)2 * kPxchMaxCtas * kPxchRec;
constexpr size_t kPbarBytes = (size_t)(1 + 16) * 32 * sizeof(unsigned int);   // barrier counters of the panel kernels (panel_xch.cuh)

// Width bookkeeping of the "tall" layout (row-major, row pitch ld doubles):
//   lp = 8 * NB   (NB = number of 8-column DMMA blocks, from the instantiated list)
//   ld = lp + 4   (pitch = 4 mod 8 doubles -> conflict-free B-fragment LDS.64)
int nb_for_cols(int64_t cols);      // smallest instantiated NB with 8*NB >= cols
inline int64_t ld_for_cols(int64_t cols) {
    return cols <= kMaxCols ? 8 * (int64_t)nb_for_cols(cols) + 4 : 8 * ((cols + 7) / 8) + 4;      // always 4 mod 8 doubles
}

}  // namespace gsi

struct gsi_ctx {
    int device = 0;
    int rank = 0;
    int world = 1;
    int num_sms = 0;
    cudaStream_t stream = nullptr;
    void* nccl_comm = nullptr;           // ncclComm_t (dlopen'ed NCCL), world > 1 only
    // small device scratch reused by the column-step kernels
    double* scratch = nullptr;           // doubles
    size_t scratch_doubles = 0;
    int* dflags = nullptr;               // device int flags [16]
    // buffers / operators alive on this context; gsi_ctx_destroy is deferred until they are gone
    // (Julia finalizers and Python interpreter shutdown run in no particular order)
    int64_t live_objects = 0;
    bool destroy_requested = false;
    // launch counter (kernels launched by this library since last reset)
    int64_t launches = 0;
    // optional event pair around the dominant GEMM kernel (bench roofline)
    double gemm_ms_accum = 0.0;
    int64_t gemm_launches = 0;
    double gemm_flops_accum = 0.0;
    bool time_gemm = false;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // event pairs recorded around operator products while time_gemm is on; resolved
    // (synchronised + summed) only when the host queries them, so timing adds no sync
    std::vector<cudaEvent_t> ev_pool;
    size_t ev_used = 0;
    std::vector<int> ev_phase;           // phase id of each recorded pair
    double phase_ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // 0 gemm, 1 lu, 2 qr, 3 small svd, 4 back-multiply
    // caching device allocator for iterate buffers: cudaMalloc/cudaFree of ~350 MB blocks
    // cost milliseconds and synchronise the device, so freed blocks are kept for reuse
    std::vector<std::pair<size_t, void*>> free_blocks;
    size_t cached_bytes = 0;
    // k-sweep schedule of the matrix-free product kernel (kcov_gemm.cu; gsi_ctx_set_option "kcov.*")
    int kcov_sweep_groups = 64;          // CTAs start their sweep at (b mod groups) * separation tiles
    int kcov_sweep_div = 256;            // separation = nkt / div tiles (div > 0) or -div tiles (div < 0)
    int kcov_l2_hint = 0;                // evict_last cache hint on the X stream
    int kcov_window = 0;                 // epochs a CTA may run ahead of the slowest CTA (0: unthrottled)
    int kcov_epoch_shift = 6;            // epoch = 2^shift k-tiles
    unsigned int* sweep_cnt = nullptr;   // per-epoch arrival counters of one launch
    size_t sweep_cnt_n = 0;
    // small Jacobi SVD: all sweeps in one cluster launch (svd.cu; gsi_ctx_set_option "svd.fused")
    int svd_fused = 1;
    int* jflags = nullptr;               // [60] rotations per sweep, [60] sweeps used
    int svd_last_sweeps = 0;             // sweeps of the last single-launch Jacobi run whose verdict was read (option "svd.last_sweeps", read-only)
    bool svd_pending = false;            // a single-launch Jacobi run whose convergence flag has not been read yet
    // factorisation drivers (lu.cu / qr.cu; gsi_ctx_set_option "lu.panel" / "qr.panel"): 1 = one cooperative
    // launch per 16-column panel with the panel rows resident in shared memory (default), 0 = one or two
    // launches per column (the first round's scheme, kept as the independent implementation to test against)
    // (1: a single thread-block cluster for short iterates, the cooperative grid otherwise; 2: always the grid)
    int lu_panel = 1;
    int qr_panel = 1;
    // pinned bounce buffers for uploads from pageable host memory (tall_ops.cu)
    void* pin[2] = {nullptr, nullptr};
    cudaEvent_t pin_ev[2] = {nullptr, nullptr};
    // exchange area of the panel kernels (used by nothing else): per-CTA records, double-buffered by column parity
    double* pxch = nullptr;              // [kPxchDoubles]
    unsigned int* pbar = nullptr;        // [kPbarBytes]: two-level barrier counters, zeroed before every factorisation
};

struct gsi_buf {
    gsi_ctx* ctx = nullptr;
    int32_t layout = GSI_LAYOUT_TALL;
    int64_t rows = 0, cols = 0;
    int64_t ld = 0;                      // TALL: row pitch; COLMAJOR: column pitch (doubles)
    int64_t rows_alloc = 0;              // TALL: padded row count (zero filled)
    double* d = nullptr;
    bool owns = true;
    size_t bytes() const {
        return layout == GSI_LAYOUT_TALL ? (size_t)rows_alloc * ld * 8 : (size_t)ld * cols * 8;
    }
};

// internal covariance kinds of the matrix-free product kernel (outside the public GSI_KERNEL_* range 0..5)
constexpr int KC_KIND_MODEL = 13;         // nested model: sum of structures, each with its own kind and coordinates
constexpr int KC_KIND_TABLE_SIGNED = 14;  // structured grid, table over signed lattice offsets (rotated anisotropy)
constexpr int KC_KIND_TABLE = 15;         // structured grid, table over |lattice offsets|

enum OpType { OP_DENSE = 0, OP_LOWRANKCOV = 1, OP_KERNELCOV = 2, OP_KERNELCROSS = 3 };

struct gsi_op {
    gsi_ctx* ctx = nullptr;
    OpType type = OP_DENSE;
    int64_t m = 0, n = 0;                // global logical size
    int64_t row0 = 0, mloc = 0;          // locally owned rows [row0, row0 + mloc)
    // dense / lowrankcov
    gsi_buf* A = nullptr;                // COLMAJOR mloc x n (dense) or n x N samples (lowrank)
    double scale = 1.0;
    gsi_buf* tmpT = nullptr;             // lowrankcov: N x l intermediate
    // kernelcov
    int32_t kind = 0, dim = 0;
    double sigma2 = 1.0, nugget = 0.0, beta = 1.0;
    double* ucoords = nullptr;           // [dim][n_pad] scaled coordinates (SoA)
    int64_t n_pad = 0;
    int* lattice = nullptr;              // structured grid: [3][n_pad] lattice indices
    double* table = nullptr;             // structured grid: kernel value per lattice offset
    int grid_nx = 1, grid_ny = 1, grid_nz = 1;
    bool table_signed = false;           // structured grid: the table covers signed offsets (rotated model)
    // nested model generated in the kernel (kind == KC_KIND_MODEL): ucoords is [nstruct][3][n_pad]
    int32_t nstruct = 1;
    int32_t mkinds[GSI_MODEL_MAX_STRUCTURES] = {0, 0, 0, 0};
    double msills[GSI_MODEL_MAX_STRUCTURES] = {0, 0, 0, 0}, mbetas[GSI_MODEL_MAX_STRUCTURES] = {1, 1, 1, 1};
    // cross-covariance C(T, S) (OP_KERNELCROSS): ucoords / lattice hold the n source points, these this rank's mloc
    // target points (compacted, so that bulk copies of them stay 16-byte aligned), same layouts with pitch nt_pad
    double* ucoords_t = nullptr;
    int* lattice_t = nullptr;
    int64_t nt_pad = 0;
    std::vector<int64_t> part;           // row partition over ranks: part[r] .. part[r+1]
};

namespace gsi {

// ---- tall_ops.cu
void tall_zero(gsi_ctx*, gsi_buf*);
void tall_copy(gsi_ctx*, const gsi_buf* src, gsi_buf* dst);
// dst[r, 0:w) = src[r, 0:w) for windows of TALL buffers (pointer to the first column + row pitch)
void tall_cols_copy(gsi_ctx*, const double* src, int64_t lds, double* dst, int64_t ldd, int64_t rows, int64_t w);
void tall_upload(gsi_buf* b, const double* host, int64_t ldh, int64_t row0, int64_t nrows);
void tall_download(const gsi_buf* b, double* host, int64_t ldh, int64_t row0, int64_t nrows);
// out[rows x l2] = Q[rows x l] * M   (M: TALL l x l2 buffer)
void tall_times_small(gsi_ctx*, const gsi_buf* Q, const gsi_buf* Mtall, gsi_buf* out);
// small column-major device matrix -> TALL buffer (zero padded)
void small_cm_to_tall(gsi_ctx*, const double* M, int64_t ldm, int64_t rows, int64_t cols, gsi_buf* T);
void colmajor_upload(gsi_buf* b, const double* host, int64_t ldh);
void colmajor_download(const gsi_buf* b, double* host, int64_t ldh);

// ---- kcov_gemm.cu :  W[local rows] = C[rows, :] * X  (cross-covariance: trans = 1 gives W = C' X, all n rows)
void kcov_apply(gsi_op* op, int trans, const gsi_buf* X, gsi_buf* W);
// ---- dense_gemm.cu : W = A X (trans=0) or A' X (trans=1); alpha scaling
void dense_apply(gsi_ctx*, const gsi_buf* A, int trans, const gsi_buf* X, gsi_buf* W, double alpha);
void tall_window_update(gsi_ctx*, const double* Pd, int64_t ldp, int64_t rows, int64_t kdim, const gsi_buf* X,
                        double* Wd, int64_t ldw, double alpha);
// ---- lu.cu : in place, returns unit-lower-trapezoidal L in LAPACK row order
// (all rows of Y on this device; enqueue only -- the zero-pivot flag is read by lu_check_singular)
void lu_L_inplace(gsi_ctx*, gsi_buf* Y);
void lu_reset_flag(gsi_ctx*);
void lu_check_singular(gsi_ctx*);      // synchronises; throws GSI_ERR_SINGULAR if an LU since the last reset met a zero pivot
// ---- qr.cu : in place thin Q; R (l x l, column-major, device) optional
void qr_thinQ_inplace(gsi_ctx*, gsi_buf* Y, double* Rdev /* l*l or null */);
// ---- svd.cu : one-sided Jacobi on l x l column-major device matrix M (overwritten with U),
//      sigma (device, l) sorted descending, columns of U permuted accordingly
void svd_small(gsi_ctx*, double* M, int l, double* U, double* sigma, bool defer_check = false);
void svd_check(gsi_ctx*);               // verdict of a deferred convergence check (synchronises)
//      the sweeps alone, on the first rows_dot rows of ncols columns (pitch ld); rotations are applied
//      to all rows_all rows (rows below rows_dot accumulate the right singular vectors)
void jacobi_sweeps(gsi_ctx*, double* M, int64_t ld, int rows_dot, int rows_all, int ncols, bool defer_check = false);
// ---- comm.cu
void comm_allgather(gsi_ctx*, const void* send, void* recv, size_t bytes_per_rank);
void comm_allreduce_sum(gsi_ctx*, double* buf, size_t count);
void comm_broadcast(gsi_ctx*, double* buf, size_t count, int root);
// every rank r contributes counts[r] doubles placed at offsets[r] of `full` (in place ok)
void comm_allgatherv(gsi_ctx*, double* full, const int64_t* offsets, const int64_t* counts);
void comm_init(gsi_ctx*, const void* unique_id);
void comm_destroy(gsi_ctx*);
void comm_unique_id(void* out128);

inline void count_launch(gsi_ctx* c, int n = 1) { c->launches += n; }
// ---- algos.cu: event-pair phase timing (active only while time_gemm is on)
enum Phase { PH_GEMM = 0, PH_LU = 1, PH_QR = 2, PH_SVD = 3, PH_BACKMUL = 4 };
void phase_begin(gsi_ctx*);
void phase_end(gsi_ctx*, int phase);
// ---- api.cu: pooled device memory
void* pool_alloc(gsi_ctx*, size_t bytes);
void pool_free(gsi_ctx*, void* p, size_t bytes);
void pool_release(gsi_ctx*);
void ctx_retain(gsi_ctx*);
void ctx_release(gsi_ctx*);      // may destroy the context if gsi_ctx_destroy was already requested

}  // namespace gsi
