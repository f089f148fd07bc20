// extern "C" surface of libgsi_b200.so (declared in include/gsi_b200.h).  Every entry
// point converts C++ exceptions into status codes + a thread-local message; nothing
// throws, exits or aborts across the ABI.
#include "common.cuh"
#include "algos.h"
#include <mutex>
#include <cmath>

#define GSI_API extern "C" __attribute__((visibility("default")))

namespace gsi {
static thread_local std::string g_last_error;
void set_last_error(const std::string& msg) { g_last_error = msg; }

template <typename F>
static int32_t guarded(F&& f) {
    try {
        f();
        return GSI_OK;
    } catch (const Error& e) {
        set_last_error(e.what());
        return e.code;
    } catch (const std::bad_alloc&) {
        set_last_error("out of host memory");
        return GSI_ERR_CUDA;
    } catch (const std::exception& e) {
        set_last_error(e.what());
        return GSI_ERR_INVALID_ARGUMENT;
    } catch (...) {
        set_last_error("unknown error");
        return GSI_ERR_INVALID_ARGUMENT;
    }
}

// Exact-size free list.  Stream-ordered reuse is safe because every consumer of a block
// is enqueued on ctx->stream (a block returned to the pool is only handed out to work that
// is enqueued later on the same stream).
static std::mutex g_pool_mutex;
void* pool_alloc(gsi_ctx* ctx, size_t bytes) {
    {
        std::lock_guard<std::mutex> lock(g_pool_mutex);
        for (size_t i = 0; i < ctx->free_blocks.size(); ++i) {
            if (ctx->free_blocks[i].first == bytes) {
                void* p = ctx->free_blocks[i].second;
                ctx->free_blocks.erase(ctx->free_blocks.begin() + i);
                ctx->cached_bytes -= bytes;
                return p;
            }
        }
    }
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        pool_release(ctx);                      // give cached blocks back and retry once
        GSI_CUDA(cudaMalloc(&p, bytes));
    }
    return p;
}
void pool_free(gsi_ctx* ctx, void* p, size_t bytes) {
    if (!p) return;
    std::lock_guard<std::mutex> lock(g_pool_mutex);
    const size_t kMaxCached = (size_t)24 << 30;
    if (ctx->cached_bytes + bytes > kMaxCached || ctx->free_blocks.size() >= 64) {
        cudaFree(p);
        return;
    }
    ctx->free_blocks.emplace_back(bytes, p);
    ctx->cached_bytes += bytes;
}
void pool_release(gsi_ctx* ctx) {
    std::lock_guard<std::mutex> lock(g_pool_mutex);
    for (auto& b : ctx->free_blocks) cudaFree(b.second);
    ctx->free_blocks.clear();
    ctx->cached_bytes = 0;
}

static void validate_kcov_options(const gsi_ctx* ctx) {
    const int g = ctx->kcov_sweep_groups;
    GSI_REQUIRE(g >= 1 && g <= 1024 && (g & (g - 1)) == 0, GSI_ERR_INVALID_ARGUMENT,
                "kcov.sweep_groups must be a power of two in [1, 1024]");
    GSI_REQUIRE(ctx->kcov_window >= 0 && ctx->kcov_window <= 4096, GSI_ERR_INVALID_ARGUMENT,
                "kcov.window must be in [0, 4096] epochs");
    GSI_REQUIRE(ctx->kcov_epoch_shift >= 2 && ctx->kcov_epoch_shift <= 16, GSI_ERR_INVALID_ARGUMENT,
                "kcov.epoch_shift must be in [2, 16]");
}

static void set_option_impl(gsi_ctx* ctx, const std::string& n, int64_t value) {
    const int v = (int)value;
    const int saved[5] = {ctx->kcov_sweep_groups, ctx->kcov_sweep_div, ctx->kcov_l2_hint, ctx->kcov_window,
                          ctx->kcov_epoch_shift};
    if (n == "kcov.sweep_groups") ctx->kcov_sweep_groups = v;
    else if (n == "kcov.sweep_div") ctx->kcov_sweep_div = v;
    else if (n == "kcov.l2_hint") ctx->kcov_l2_hint = v;
    else if (n == "kcov.window") ctx->kcov_window = v;
    else if (n == "kcov.epoch_shift") ctx->kcov_epoch_shift = v;
    else if (n == "svd.fused") ctx->svd_fused = v < 0 ? 0 : (v > 2 ? 2 : (int)v);
    else if (n == "lu.panel") ctx->lu_panel = v < 0 ? 0 : (v > 2 ? 2 : (int)v);
    else if (n == "qr.panel") ctx->qr_panel = v < 0 ? 0 : (v > 2 ? 2 : (int)v);
    else throw Error(GSI_ERR_INVALID_ARGUMENT, "unknown option '" + n + "'");
    try {
        validate_kcov_options(ctx);
    } catch (...) {
        ctx->kcov_sweep_groups = saved[0]; ctx->kcov_sweep_div = saved[1]; ctx->kcov_l2_hint = saved[2];
        ctx->kcov_window = saved[3]; ctx->kcov_epoch_shift = saved[4];
        throw;
    }
}

// GSI_OPTIONS="name=value,name=value": the gsi_ctx_set_option knobs from the environment
static void options_from_env(gsi_ctx* ctx) {
    const char* e = getenv("GSI_OPTIONS");
    if (!e) return;
    std::string all(e);
    size_t pos = 0;
    while (pos < all.size()) {
        size_t end = all.find(',', pos);
        if (end == std::string::npos) end = all.size();
        const std::string item = all.substr(pos, end - pos);
        pos = end + 1;
        if (item.empty()) continue;
        const size_t eq = item.find('=');
        GSI_REQUIRE(eq != std::string::npos && eq > 0 && eq + 1 < item.size(), GSI_ERR_INVALID_ARGUMENT,
                    "GSI_OPTIONS: expected name=value, got '" + item + "'");
        set_option_impl(ctx, item.substr(0, eq), strtoll(item.c_str() + eq + 1, nullptr, 10));
    }
}

static void use(gsi_ctx* ctx) {
    GSI_REQUIRE(ctx != nullptr, GSI_ERR_INVALID_ARGUMENT, "null context");
    GSI_CUDA(cudaSetDevice(ctx->device));
}
}  // namespace gsi

using namespace gsi;

GSI_API int32_t gsi_version(void) { return GSI_VERSION; }
GSI_API const char* gsi_last_error_string(void) { return g_last_error.c_str(); }

GSI_API int32_t gsi_comm_unique_id(void* out128) {
    return guarded([&] {
        GSI_REQUIRE(out128 != nullptr, GSI_ERR_INVALID_ARGUMENT, "null output");
        comm_unique_id(out128);
    });
}

static void ctx_really_destroy(gsi_ctx* ctx);

GSI_API int32_t gsi_ctx_create(int32_t device, int32_t rank, int32_t world, const void* unique_id128, gsi_ctx** out) {
    return guarded([&] {
        GSI_REQUIRE(out != nullptr, GSI_ERR_INVALID_ARGUMENT, "null output");
        *out = nullptr;
        GSI_REQUIRE(world >= 1 && rank >= 0 && rank < world, GSI_ERR_INVALID_ARGUMENT, "bad rank/world");
        int ndev = 0;
        cudaError_t e = cudaGetDeviceCount(&ndev);
        if (e != cudaSuccess || ndev == 0) {
            cudaGetLastError();
            throw Error(GSI_ERR_NO_DEVICE, "no CUDA device: gsi_b200 has no CPU fallback (needs an sm_100 GPU)");
        }
        GSI_REQUIRE(device >= 0 && device < ndev, GSI_ERR_INVALID_ARGUMENT, "device index out of range");
        cudaDeviceProp prop;
        GSI_CUDA(cudaGetDeviceProperties(&prop, device));
        if (prop.major != 10 || prop.minor != 0)      // sm_100a SASS only: no PTX, not even other 10.x parts can run it
            throw Error(GSI_ERR_NO_DEVICE, std::string("device '") + prop.name + "' is sm_" + std::to_string(prop.major) +
                                               std::to_string(prop.minor) + "; gsi_b200 is built for sm_100a only");
        GSI_CUDA(cudaSetDevice(device));
        // failure paths release whatever was created so far (stream, scratch, events, NCCL communicator)
        std::unique_ptr<gsi_ctx, void (*)(gsi_ctx*)> ctx(new gsi_ctx(), ctx_really_destroy);
        ctx->device = device; ctx->rank = rank; ctx->world = world;
        ctx->num_sms = prop.multiProcessorCount;
        GSI_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        ctx->scratch_doubles = (size_t)1 << 20;
        GSI_CUDA(cudaMalloc(&ctx->scratch, ctx->scratch_doubles * sizeof(double)));
        GSI_CUDA(cudaMalloc(&ctx->dflags, 16 * sizeof(int)));
        GSI_CUDA(cudaMemset(ctx->dflags, 0, 16 * sizeof(int)));
        GSI_CUDA(cudaMalloc(&ctx->jflags, 64 * sizeof(int)));
        GSI_CUDA(cudaMalloc(&ctx->pxch, kPxchDoubles * sizeof(double)));
        GSI_CUDA(cudaMemset(ctx->pxch, 0, kPxchDoubles * sizeof(double)));
        GSI_CUDA(cudaMalloc(&ctx->pbar, kPbarBytes));
        GSI_CUDA(cudaMemset(ctx->pbar, 0, kPbarBytes));
        if (const char* e = getenv("GSI_SVD_FUSED")) ctx->svd_fused = atoi(e) < 0 ? 0 : (atoi(e) > 2 ? 2 : atoi(e));
        GSI_CUDA(cudaEventCreate(&ctx->ev0));
        GSI_CUDA(cudaEventCreate(&ctx->ev1));
        if (const char* e = getenv("GSI_SWEEP"))      // "groups,div,hint[,window[,epoch_shift]]": see gsi_ctx_set_option
            sscanf(e, "%d,%d,%d,%d,%d", &ctx->kcov_sweep_groups, &ctx->kcov_sweep_div, &ctx->kcov_l2_hint,
                   &ctx->kcov_window, &ctx->kcov_epoch_shift);
        validate_kcov_options(ctx.get());
        options_from_env(ctx.get());
        if (world > 1) comm_init(ctx.get(), unique_id128);
        *out = ctx.release();
    });
}

static void ctx_really_destroy(gsi_ctx* ctx) {
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    comm_destroy(ctx);
    pool_release(ctx);
    if (ctx->scratch) cudaFree(ctx->scratch);
    if (ctx->dflags) cudaFree(ctx->dflags);
    if (ctx->sweep_cnt) cudaFree(ctx->sweep_cnt);
    if (ctx->jflags) cudaFree(ctx->jflags);
    if (ctx->pxch) cudaFree(ctx->pxch);
    if (ctx->pbar) cudaFree(ctx->pbar);
    for (int i = 0; i < 2; ++i) {
        if (ctx->pin[i]) cudaFreeHost(ctx->pin[i]);
        if (ctx->pin_ev[i]) cudaEventDestroy(ctx->pin_ev[i]);
    }
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    for (cudaEvent_t e : ctx->ev_pool) cudaEventDestroy(e);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

namespace gsi {
static std::mutex g_ctx_mutex;
void ctx_retain(gsi_ctx* ctx) {
    std::lock_guard<std::mutex> lock(g_ctx_mutex);
    ++ctx->live_objects;
}
void ctx_release(gsi_ctx* ctx) {
    bool kill = false;
    {
        std::lock_guard<std::mutex> lock(g_ctx_mutex);
        --ctx->live_objects;
        kill = ctx->destroy_requested && ctx->live_objects <= 0;
    }
    if (kill) ctx_really_destroy(ctx);
}
}  // namespace gsi

GSI_API int32_t gsi_ctx_destroy(gsi_ctx* ctx) {
    return guarded([&] {
        if (!ctx) return;
        bool now = false;
        {
            std::lock_guard<std::mutex> lock(g_ctx_mutex);
            ctx->destroy_requested = true;
            now = ctx->live_objects <= 0;
        }
        if (now) ctx_really_destroy(ctx);      // otherwise the last buffer / operator release does it
    });
}

GSI_API int32_t gsi_ctx_set_option(gsi_ctx* ctx, const char* name, int64_t value) {
    return guarded([&] {
        use(ctx);
        GSI_REQUIRE(name != nullptr, GSI_ERR_INVALID_ARGUMENT, "null option name");
        set_option_impl(ctx, name, value);
    });
}

GSI_API int32_t gsi_ctx_get_option(gsi_ctx* ctx, const char* name, int64_t* value_out) {
    return guarded([&] {
        use(ctx);
        GSI_REQUIRE(name != nullptr && value_out != nullptr, GSI_ERR_INVALID_ARGUMENT, "null argument");
        const std::string n(name);
        if (n == "kcov.sweep_groups") *value_out = ctx->kcov_sweep_groups;
        else if (n == "kcov.sweep_div") *value_out = ctx->kcov_sweep_div;
        else if (n == "kcov.l2_hint") *value_out = ctx->kcov_l2_hint;
        else if (n == "kcov.window") *value_out = ctx->kcov_window;
        else if (n == "kcov.epoch_shift") *value_out = ctx->kcov_epoch_shift;
        else if (n == "svd.fused") *value_out = ctx->svd_fused;
        else if (n == "svd.last_sweeps") *value_out = ctx->svd_last_sweeps;
        else if (n == "lu.panel") *value_out = ctx->lu_panel;
        else if (n == "qr.panel") *value_out = ctx->qr_panel;
        else throw Error(GSI_ERR_INVALID_ARGUMENT, "unknown option '" + n + "'");
    });
}

GSI_API int32_t gsi_ctx_sync(gsi_ctx* ctx) {
    return guarded([&] { use(ctx); GSI_CUDA(cudaStreamSynchronize(ctx->stream)); });
}

GSI_API int32_t gsi_ctx_stream(gsi_ctx* ctx, void** stream_out) {
    return guarded([&] { use(ctx); *stream_out = (void*)ctx->stream; });
}

GSI_API int32_t gsi_ctx_launch_count(gsi_ctx* ctx, int64_t* count_out, int32_t reset) {
    return guarded([&] {
        use(ctx);
        if (count_out) *count_out = ctx->launches;
        if (reset) ctx->launches = 0;
    });
}

GSI_API int32_t gsi_ctx_gemm_timing(gsi_ctx* ctx, int32_t enable, double* ms_out, int64_t* launches_out,
                                    double* flops_out) {
    return guarded([&] {
        use(ctx);
        resolve_gemm_timing(ctx);
        if (ms_out) *ms_out = ctx->gemm_ms_accum;
        if (launches_out) *launches_out = ctx->gemm_launches;
        if (flops_out) *flops_out = ctx->gemm_flops_accum;
        if (enable >= 0) {
            ctx->time_gemm = enable != 0;
            ctx->gemm_ms_accum = 0.0; ctx->gemm_launches = 0; ctx->gemm_flops_accum = 0.0;
        }
    });
}

GSI_API int32_t gsi_ctx_phase_timing(gsi_ctx* ctx, double* ms_out8, int32_t reset) {
    return guarded([&] {
        use(ctx);
        resolve_gemm_timing(ctx);
        if (ms_out8) for (int i = 0; i < 8; ++i) ms_out8[i] = ctx->phase_ms[i];
        if (reset) for (int i = 0; i < 8; ++i) ctx->phase_ms[i] = 0.0;
    });
}

// ---- buffers
GSI_API int32_t gsi_buf_alloc(gsi_ctx* ctx, int32_t layout, int64_t rows, int64_t cols, gsi_buf** out) {
    return guarded([&] {
        use(ctx);
        GSI_REQUIRE(out != nullptr, GSI_ERR_INVALID_ARGUMENT, "null output");
        *out = make_buf(ctx, layout, rows, cols).release();
    });
}

GSI_API int32_t gsi_buf_free(gsi_buf* buf) {
    if (!buf) return GSI_OK;
    return guarded([&] {
        cudaSetDevice(buf->ctx->device);
        BufDeleter()(buf);
    });
}

// Page-locked host memory (cudaHostAlloc) for host arrays that are uploaded again and again, e.g. the
// batch of forward runs an rga iteration sketches: a source in such memory is copied by DMA directly
// instead of through the context's bounce buffers.
GSI_API int32_t gsi_host_alloc(gsi_ctx* ctx, int64_t bytes, void** out) {
    return guarded([&] {
        use(ctx);
        GSI_REQUIRE(out != nullptr && bytes >= 0, GSI_ERR_INVALID_ARGUMENT, "gsi_host_alloc: bad argument");
        *out = nullptr;
        if (bytes == 0) return;
        void* q = nullptr;
        const cudaError_t e = cudaHostAlloc(&q, (size_t)bytes, cudaHostAllocDefault);
        if (e != cudaSuccess) {
            cudaGetLastError();
            throw Error(GSI_ERR_CUDA, std::string("gsi_host_alloc: ") + cudaGetErrorString(e));
        }
        *out = q;
    });
}

GSI_API int32_t gsi_host_free(gsi_ctx* ctx, void* ptr) {
    if (!ptr) return GSI_OK;
    return guarded([&] {
        if (ctx) GSI_CUDA(cudaSetDevice(ctx->device));      // ctx may be NULL (context already destroyed)
        GSI_CUDA(cudaFreeHost(ptr));
    });
}

GSI_API int32_t gsi_buf_dims(const gsi_buf* buf, int64_t* rows, int64_t* cols) {
    return guarded([&] {
        GSI_REQUIRE(buf != nullptr, GSI_ERR_INVALID_ARGUMENT, "null buffer");
        if (rows) *rows = buf->rows;
        if (cols) *cols = buf->cols;
    });
}

GSI_API int32_t gsi_buf_upload(gsi_buf* buf, const double* host, int64_t ldh) {
    return guarded([&] {
        GSI_REQUIRE(buf && host, GSI_ERR_INVALID_ARGUMENT, "null argument");
        use(buf->ctx);
        if (buf->layout == GSI_LAYOUT_TALL) tall_upload(buf, host, ldh, 0, buf->rows);
        else colmajor_upload(buf, host, ldh);
    });
}

GSI_API int32_t gsi_buf_download(const gsi_buf* buf, double* host, int64_t ldh) {
    return guarded([&] {
        GSI_REQUIRE(buf && host, GSI_ERR_INVALID_ARGUMENT, "null argument");
        use(buf->ctx);
        if (buf->layout == GSI_LAYOUT_TALL) tall_download(buf, host, ldh, 0, buf->rows);
        else colmajor_download(buf, host, ldh);
    });
}

GSI_API int32_t gsi_buf_upload_rows(gsi_buf* buf, int64_t row0, int64_t nrows, const double* host, int64_t ldh) {
    return guarded([&] {
        GSI_REQUIRE(buf && host, GSI_ERR_INVALID_ARGUMENT, "null argument");
        use(buf->ctx);
        tall_upload(buf, host, ldh, row0, nrows);
    });
}

GSI_API int32_t gsi_buf_download_rows(const gsi_buf* buf, int64_t row0, int64_t nrows, double* host, int64_t ldh) {
    return guarded([&] {
        GSI_REQUIRE(buf && host, GSI_ERR_INVALID_ARGUMENT, "null argument");
        use(buf->ctx);
        tall_download(buf, host, ldh, row0, nrows);
    });
}

GSI_API int32_t gsi_buf_copy(const gsi_buf* src, gsi_buf* dst) {
    return guarded([&] {
        GSI_REQUIRE(src && dst, GSI_ERR_INVALID_ARGUMENT, "null argument");
        use(src->ctx);
        tall_copy(src->ctx, src, dst);
        GSI_CUDA(cudaStreamSynchronize(src->ctx->stream));
    });
}

GSI_API int32_t gsi_buf_zero(gsi_buf* buf) {
    return guarded([&] {
        GSI_REQUIRE(buf != nullptr, GSI_ERR_INVALID_ARGUMENT, "null buffer");
        use(buf->ctx);
        tall_zero(buf->ctx, buf);
    });
}

// ---- operators
static void set_partition(gsi_op* op) {
    gsi_ctx* ctx = op->ctx;
    op->part.assign(ctx->world + 1, 0);
    if (ctx->world == 1) {
        GSI_REQUIRE(op->row0 == 0 && op->mloc == op->m, GSI_ERR_INVALID_ARGUMENT,
                    "single-rank operator must own all rows (row0 = 0, mloc = m)");
        op->part[1] = op->m;
        return;
    }
    int64_t* dev = reinterpret_cast<int64_t*>(ctx->scratch);
    int64_t mine = op->row0;
    GSI_CUDA(cudaMemcpyAsync(dev + ctx->world, &mine, sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
    comm_allgather(ctx, dev + ctx->world, dev, sizeof(int64_t));
    GSI_CUDA(cudaMemcpyAsync(op->part.data(), dev, ctx->world * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    GSI_CUDA(cudaStreamSynchronize(ctx->stream));
    op->part[ctx->world] = op->m;
    for (int r = 0; r < ctx->world; ++r)
        GSI_REQUIRE(op->part[r] <= op->part[r + 1], GSI_ERR_INVALID_ARGUMENT, "row partition must be ordered by rank");
    GSI_REQUIRE(op->part[0] == 0 && op->part[ctx->rank + 1] - op->part[ctx->rank] == op->mloc, GSI_ERR_INVALID_ARGUMENT,
                "row partition must be contiguous and cover all rows");
}

// failure paths of the operator constructors: device arrays of a half-built operator are released
struct OpAbort {
    void operator()(gsi_op* op) const {
        if (!op) return;
        if (op->ucoords) cudaFree(op->ucoords);
        if (op->table) cudaFree(op->table);
        if (op->lattice) cudaFree(op->lattice);
        if (op->ucoords_t) cudaFree(op->ucoords_t);
        if (op->lattice_t) cudaFree(op->lattice_t);
        delete op;
    }
};

GSI_API int32_t gsi_op_dense(gsi_ctx* ctx, gsi_buf* A_local, int64_t row0, int64_t m_global, gsi_op** out) {
    return guarded([&] {
        use(ctx);
        GSI_REQUIRE(A_local && out, GSI_ERR_INVALID_ARGUMENT, "null argument");
        GSI_REQUIRE(A_local->layout == GSI_LAYOUT_COLMAJOR, GSI_ERR_INVALID_ARGUMENT, "dense operator needs a COLMAJOR buffer");
        std::unique_ptr<gsi_op> op(new gsi_op());
        op->ctx = ctx; op->type = OP_DENSE; op->A = A_local;
        op->m = m_global; op->n = A_local->cols; op->row0 = row0; op->mloc = A_local->rows;
        set_partition(op.get());
        ctx_retain(ctx);
        *out = op.release();
    });
}

__global__ void remove_mean_kernel(double* __restrict__ S, int64_t ld, int64_t n, int64_t N) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double mean = 0.0;
    for (int64_t c = 0; c < N; ++c) mean += S[c * ld + i];      // same order as src/lowrank.jl:19-23
    mean = mean / (double)N;
    for (int64_t c = 0; c < N; ++c) S[c * ld + i] -= mean;
}

static void make_lowrankcov(gsi_ctx* ctx, gsi_buf* samples, int32_t remove_mean, int64_t row0, int64_t n_global, gsi_op** out) {
    use(ctx);
    GSI_REQUIRE(samples && out, GSI_ERR_INVALID_ARGUMENT, "null argument");
    GSI_REQUIRE(samples->layout == GSI_LAYOUT_COLMAJOR, GSI_ERR_INVALID_ARGUMENT, "samples must be a COLMAJOR buffer");
    GSI_REQUIRE(samples->cols >= 2, GSI_ERR_INVALID_ARGUMENT, "LowRankCovMatrix needs at least 2 samples");
    GSI_REQUIRE(row0 >= 0 && row0 + samples->rows <= n_global, GSI_ERR_INVALID_ARGUMENT, "lowrankcov: bad row block");
    std::unique_ptr<gsi_op> op(new gsi_op());
    op->ctx = ctx; op->type = OP_LOWRANKCOV; op->A = samples;
    op->m = op->n = n_global; op->row0 = row0; op->mloc = samples->rows;
    op->scale = 1.0 / (double)(samples->cols - 1);
    if (remove_mean && samples->rows > 0) {        // the mean is over the samples, row by row: local to the row block
        remove_mean_kernel<<<(unsigned)((samples->rows + 255) / 256), 256, 0, ctx->stream>>>(samples->d, samples->ld,
                                                                                             samples->rows, samples->cols);
        GSI_CUDA(cudaGetLastError());
        count_launch(ctx);
    }
    set_partition(op.get());
    ctx_retain(ctx);
    *out = op.release();
}

GSI_API int32_t gsi_op_lowrankcov(gsi_ctx* ctx, gsi_buf* samples, int32_t remove_mean, gsi_op** out) {
    return guarded([&] {
        GSI_REQUIRE(samples != nullptr, GSI_ERR_INVALID_ARGUMENT, "null argument");
        make_lowrankcov(ctx, samples, remove_mean, 0, samples->rows, out);
    });
}

GSI_API int32_t gsi_op_lowrankcov_sharded(gsi_ctx* ctx, gsi_buf* samples_local, int32_t remove_mean, int64_t row0,
                                          int64_t n_global, gsi_op** out) {
    return guarded([&] { make_lowrankcov(ctx, samples_local, remove_mean, row0, n_global, out); });
}

namespace gsi {
// A covariance model: nstruct structures, each a kind, a sill, d ranges, an optional rotation (column-major d x d,
// u = R x) and a power-law exponent.  gsi_op_kernelcov / _grid are the one-structure, unrotated case.
struct CovModel {
    int d = 1, nstruct = 1;
    int kinds[GSI_MODEL_MAX_STRUCTURES] = {};
    double sills[GSI_MODEL_MAX_STRUCTURES] = {}, betas[GSI_MODEL_MAX_STRUCTURES] = {};
    double ranges[GSI_MODEL_MAX_STRUCTURES][3] = {};
    double rot[GSI_MODEL_MAX_STRUCTURES][9] = {};
    bool rotated[GSI_MODEL_MAX_STRUCTURES] = {};
    bool any_rotated() const {
        for (int s = 0; s < nstruct; ++s)
            if (rotated[s]) return true;
        return false;
    }
};

static CovModel single_structure(int32_t kind, int32_t d, const double* ell, double sigma2, double beta) {
    CovModel m;
    m.d = d; m.nstruct = 1; m.kinds[0] = kind; m.sills[0] = sigma2; m.betas[0] = beta;
    for (int k = 0; k < d; ++k) m.ranges[0][k] = ell[k];
    return m;
}

// the public model arguments, checked (d was checked by the caller)
static CovModel model_from_args(int32_t d, int32_t nstruct, const int32_t* kinds, const double* sills,
                                const double* ranges, const double* rotations, const double* betas) {
    GSI_REQUIRE(nstruct >= 1 && nstruct <= GSI_MODEL_MAX_STRUCTURES, GSI_ERR_INVALID_ARGUMENT,
                "kernelcov_model: nstruct must be in 1..GSI_MODEL_MAX_STRUCTURES");
    CovModel m;
    m.d = d; m.nstruct = nstruct;
    for (int s = 0; s < nstruct; ++s) {
        GSI_REQUIRE(kinds[s] >= GSI_KERNEL_EXPONENTIAL && kinds[s] <= GSI_KERNEL_SPHERICAL, GSI_ERR_INVALID_ARGUMENT,
                    "kernelcov_model: unknown kernel kind");
        GSI_REQUIRE(std::isfinite(sills[s]) && sills[s] > 0.0, GSI_ERR_INVALID_ARGUMENT,
                    "kernelcov_model: sills must be positive and finite");
        m.kinds[s] = kinds[s]; m.sills[s] = sills[s]; m.betas[s] = betas ? betas[s] : 1.0;
        for (int k = 0; k < d; ++k) {
            GSI_REQUIRE(ranges[s * d + k] > 0.0, GSI_ERR_INVALID_ARGUMENT, "kernelcov_model: ranges must be positive");
            m.ranges[s][k] = ranges[s * d + k];
        }
        if (!rotations) continue;
        const double* R = rotations + (size_t)s * d * d;
        double dev = 0.0;
        for (int a = 0; a < d; ++a)
            for (int b = 0; b < d; ++b) {
                GSI_REQUIRE(std::isfinite(R[a + d * b]), GSI_ERR_INVALID_ARGUMENT, "kernelcov_model: rotation not finite");
                double rr = 0.0;                                   // (R'R)[a, b]
                for (int k = 0; k < d; ++k) rr += R[k + d * a] * R[k + d * b];
                dev = std::fmax(dev, std::fabs(rr - (a == b ? 1.0 : 0.0)));
            }
        GSI_REQUIRE(dev <= 1e-12, GSI_ERR_INVALID_ARGUMENT, "kernelcov_model: rotation is not orthonormal");
        for (int q = 0; q < d * d; ++q) m.rot[s][q] = R[q];
        m.rotated[s] = true;
    }
    return m;
}

// coordinate scaling of the kinds: Gaussian: an extra 1/sqrt(2) folds the factor 1/2 of exp(-r2/2) into r2; Matern
// nu = 3/2 / 5/2: an extra sqrt(3) / sqrt(5), so the kernel's sqrt(r2) is the argument sqrt(2 nu) r of exp and of the
// polynomial
static double kind_pre(int kind) {
    return kind == GSI_KERNEL_GAUSSIAN   ? 0.70710678118654752440
           : kind == GSI_KERNEL_MATERN32 ? 1.73205080756887729353
           : kind == GSI_KERNEL_MATERN52 ? 2.23606797749978969641
                                         : 1.0;
}

// u[k] = ((sum_j R[k,j] x_j) / range[k]) * pre of structure s; without a rotation (x[k] / range[k]) * pre
static void structure_coords(const CovModel& m, int s, const double* x, double pre, double* u) {
    for (int k = 0; k < m.d; ++k) {
        double y = x[k];
        if (m.rotated[s]) {
            y = 0.0;
            for (int j = 0; j < m.d; ++j) y += m.rot[s][k + m.d * j] * x[j];
        }
        u[k] = (y / m.ranges[s][k]) * pre;
    }
}

// k(r2) with libm, r2 in unscaled coordinates (x / range): the value of every lattice-table entry
static double kern_host(int kind, double r2, double beta) {
    if (kind == GSI_KERNEL_EXPONENTIAL) return std::exp(-std::sqrt(r2));
    if (kind == GSI_KERNEL_GAUSSIAN) return std::exp(-0.5 * r2);
    if (kind == GSI_KERNEL_MATERN32) {
        const double s = std::sqrt(3.0 * r2);
        return (1.0 + s) * std::exp(-s);
    }
    if (kind == GSI_KERNEL_MATERN52) {
        const double s = std::sqrt(5.0 * r2);
        return (1.0 + s + s * s / 3.0) * std::exp(-s);
    }
    if (kind == GSI_KERNEL_SPHERICAL) {
        const double r = std::sqrt(r2);
        return r < 1.0 ? 0.5 * (1.0 - r) * (1.0 - r) * (2.0 + r) : 0.0;   // = 1 - 1.5 r + 0.5 r^3, no cancellation
    }
    return std::exp(-beta * std::log1p(r2));
}

// the table value of the offset x (one structure: k, scaled by sigma2 = its sill in the epilogue; several: the sum)
static double model_host(const CovModel& m, const double* x) {
    double v = 0.0;
    for (int s = 0; s < m.nstruct; ++s) {
        double u[3];
        structure_coords(m, s, x, 1.0, u);
        double r2 = u[0] * u[0];
        if (m.d > 1) r2 += u[1] * u[1];
        if (m.d > 2) r2 += u[2] * u[2];
        const double k = kern_host(m.kinds[s], r2, m.betas[s]);
        if (m.nstruct == 1) return k;
        v += m.sills[s] * k;
    }
    return v;
}

// the operator's model parameters: one structure is the specialised KIND kernel with sigma2 = its sill; several are
// KC_KIND_MODEL (arithmetic) or a table of the sum (grid), both with sigma2 = 1
static void set_model(gsi_op* op, const CovModel& m, double nugget, bool generated) {
    op->type = OP_KERNELCOV; op->dim = m.d; op->nugget = nugget;
    op->kind = m.kinds[0]; op->sigma2 = m.sills[0]; op->beta = m.betas[0];
    for (int s = 0; s < m.nstruct; ++s)
        for (int k = 0; k < m.d; ++k) op->mranges[s][k] = m.ranges[s][k];
    if (m.nstruct == 1) return;
    op->sigma2 = 1.0; op->beta = 1.0;
    if (!generated) return;
    op->kind = KC_KIND_MODEL;
    op->nstruct = m.nstruct;
    for (int s = 0; s < m.nstruct; ++s) {
        op->mkinds[s] = m.kinds[s]; op->msills[s] = m.sills[s]; op->mbetas[s] = m.betas[s];
    }
}

// scaled SoA coordinates u[s][k][j] of every structure (one structure: u[k][j]) of `count` points (point j at
// coords + j * d) -> device array dst with pitch pad = round_up(count, kRowPad); the padding repeats the last point
static void upload_coords(gsi_ctx* ctx, const CovModel& m, int64_t count, const double* coords, double*& dst,
                          int64_t& pad) {
    const int d = m.d;
    pad = round_up(count, kRowPad);
    if (count == 0) return;
    std::vector<double> u((size_t)m.nstruct * 3 * pad, 0.0);
    for (int s = 0; s < m.nstruct; ++s) {
        const double pre = kind_pre(m.kinds[s]);
        double* us = u.data() + (size_t)s * 3 * pad;
        for (int64_t j = 0; j < count; ++j) {
            double uj[3];
            structure_coords(m, s, coords + j * d, pre, uj);
            for (int k = 0; k < d; ++k) us[(size_t)k * pad + j] = uj[k];
        }
        for (int k = 0; k < d; ++k)
            for (int64_t j = count; j < pad; ++j) us[(size_t)k * pad + j] = us[(size_t)k * pad + count - 1];
    }
    GSI_CUDA(cudaMalloc(&dst, u.size() * sizeof(double)));
    GSI_CUDA(cudaMemcpyAsync(dst, u.data(), u.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    GSI_CUDA(cudaStreamSynchronize(ctx->stream));
}

static void make_kernelcov(gsi_ctx* ctx, int64_t n, const double* coords, const CovModel& m, double nugget, int64_t row0,
                           int64_t mloc, gsi_op** out) {
    GSI_REQUIRE(n >= 1 && row0 >= 0 && mloc >= 0 && row0 + mloc <= n, GSI_ERR_INVALID_ARGUMENT, "kernelcov: bad row block");
    std::unique_ptr<gsi_op, OpAbort> op(new gsi_op());
    op->ctx = ctx;
    set_model(op.get(), m, nugget, true);
    op->m = op->n = n; op->row0 = row0; op->mloc = mloc;
    upload_coords(ctx, m, n, coords, op->ucoords, op->n_pad);
    set_partition(op.get());
    ctx_retain(ctx);
    *out = op.release();
}

// a structured grid (dims / spacing of the public calls) and the size of the model's lattice table over it
struct GridSpec {
    int64_t nd[3] = {1, 1, 1};
    double h[3] = {1, 1, 1};
    int64_t n = 1;          // nodes
    bool sgn = false;       // the table covers signed offsets
    int64_t ex = 1, ey = 1, tsize = 1;
};

static GridSpec grid_spec(const int64_t* dims, const double* spacing, const CovModel& m) {
    const int d = m.d;
    GridSpec g;
    for (int k = 0; k < d; ++k) {
        GSI_REQUIRE(dims[k] >= 1, GSI_ERR_INVALID_ARGUMENT, "kernelcov_grid: bad dims / length scales");
        g.nd[k] = dims[k]; g.h[k] = spacing[k];
        g.n *= dims[k];
    }
    GSI_REQUIRE(g.n < ((int64_t)1 << 31), GSI_ERR_UNSUPPORTED, "kernelcov_grid: more than 2^31 points");
    // a rotated model is not symmetric in each axis: its table covers signed offsets, folded by k(delta) = k(-delta)
    // (the last axis as |delta|, the others from -(n - 1) to n - 1).  d = 1 is symmetric whatever the rotation (+-1)
    g.sgn = m.any_rotated() && d >= 2;
    g.ex = g.sgn ? 2 * g.nd[0] - 1 : g.nd[0];
    g.ey = g.sgn && d == 3 ? 2 * g.nd[1] - 1 : g.nd[1];
    g.tsize = g.ex * g.ey * g.nd[2];
    return g;
}

static void check_table_size(const GridSpec& g) {
    GSI_REQUIRE(g.tsize < ((int64_t)1 << 31), GSI_ERR_UNSUPPORTED, "kernelcov_grid: lattice table of 2^31 entries or more");
}

// the grid parameters of the operator and its lattice table: the model value of every lattice offset (libm, same
// formula as the dense definition)
static void upload_table(gsi_ctx* ctx, gsi_op* op, const CovModel& m, const GridSpec& g) {
    op->grid_nx = (int)g.nd[0]; op->grid_ny = (int)g.nd[1]; op->grid_nz = (int)g.nd[2];
    op->table_signed = g.sgn;
    const int64_t ox = g.sgn ? g.nd[0] - 1 : 0, oy = g.sgn && m.d == 3 ? g.nd[1] - 1 : 0;
    std::vector<double> tab((size_t)g.tsize);
    for (int64_t iz = 0; iz < g.nd[2]; ++iz)
        for (int64_t iy = 0; iy < g.ey; ++iy)
            for (int64_t ix = 0; ix < g.ex; ++ix) {
                const double x[3] = {(double)(ix - ox) * g.h[0], (double)(iy - oy) * g.h[1], (double)iz * g.h[2]};
                tab[(size_t)(ix + g.ex * (iy + g.ey * iz))] = model_host(m, x);
            }
    GSI_CUDA(cudaMalloc(&op->table, tab.size() * sizeof(double)));
    GSI_CUDA(cudaMemcpyAsync(op->table, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    GSI_CUDA(cudaStreamSynchronize(ctx->stream));
}

// lattice indices [3][pad] (SoA, pad = round_up(count, kRowPad)) of `count` grid nodes, node j at the linear index
// idx[j] (idx == NULL: j), dims[0] fastest; the padding repeats the last node
static void upload_lattice(gsi_ctx* ctx, const GridSpec& g, int64_t count, const int64_t* idx, int*& dst, int64_t& pad) {
    pad = round_up(count, kRowPad);
    if (count == 0) return;
    std::vector<int> lat((size_t)3 * pad, 0);
    for (int64_t j = 0; j < pad; ++j) {
        const int64_t jc = j < count ? j : count - 1;
        const int64_t jj = idx ? idx[jc] : jc;
        lat[(size_t)0 * pad + j] = (int)(jj % g.nd[0]);
        lat[(size_t)1 * pad + j] = (int)((jj / g.nd[0]) % g.nd[1]);
        lat[(size_t)2 * pad + j] = (int)(jj / (g.nd[0] * g.nd[1]));
    }
    GSI_CUDA(cudaMalloc(&dst, lat.size() * sizeof(int)));
    GSI_CUDA(cudaMemcpyAsync(dst, lat.data(), lat.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    GSI_CUDA(cudaStreamSynchronize(ctx->stream));
}

static void make_kernelcov_grid(gsi_ctx* ctx, const int64_t* dims, const double* spacing, const CovModel& m, double nugget,
                                int64_t row0, int64_t mloc, gsi_op** out) {
    const GridSpec g = grid_spec(dims, spacing, m);
    const int64_t n = g.n;
    GSI_REQUIRE(row0 >= 0 && mloc >= 0 && row0 + mloc <= n, GSI_ERR_INVALID_ARGUMENT, "kernelcov_grid: bad row block");
    check_table_size(g);
    std::unique_ptr<gsi_op, OpAbort> op(new gsi_op());
    op->ctx = ctx;
    set_model(op.get(), m, nugget, false);
    op->m = op->n = n; op->row0 = row0; op->mloc = mloc;
    upload_table(ctx, op.get(), m, g);
    upload_lattice(ctx, g, n, nullptr, op->lattice, op->n_pad);
    set_partition(op.get());
    ctx_retain(ctx);
    *out = op.release();
}

// Cross-covariance C(T, S): m targets (this rank: [row0, row0 + mloc), compacted), n sources, no nugget
static void check_cross_rows(int64_t m, int64_t n, int64_t row0, int64_t mloc) {
    GSI_REQUIRE(m >= 1 && n >= 1, GSI_ERR_INVALID_ARGUMENT, "kernelcov_cross: m and n must be at least 1");
    GSI_REQUIRE(row0 >= 0 && mloc >= 0 && row0 + mloc <= m, GSI_ERR_INVALID_ARGUMENT, "kernelcov_cross: bad row block");
}

static void make_kernelcross(gsi_ctx* ctx, int64_t m, const double* targets, int64_t n, const double* sources,
                             const CovModel& model, int64_t row0, int64_t mloc, gsi_op** out) {
    check_cross_rows(m, n, row0, mloc);
    std::unique_ptr<gsi_op, OpAbort> op(new gsi_op());
    op->ctx = ctx;
    set_model(op.get(), model, 0.0, true);
    op->type = OP_KERNELCROSS;
    op->m = m; op->n = n; op->row0 = row0; op->mloc = mloc;
    upload_coords(ctx, model, n, sources, op->ucoords, op->n_pad);
    upload_coords(ctx, model, mloc, targets + row0 * model.d, op->ucoords_t, op->nt_pad);
    set_partition(op.get());
    ctx_retain(ctx);
    *out = op.release();
}

static void make_kernelcross_grid(gsi_ctx* ctx, const int64_t* dims, const double* spacing, int64_t m,
                                  const int64_t* target_idx, int64_t n, const int64_t* source_idx,
                                  const CovModel& model, int64_t row0, int64_t mloc, gsi_op** out) {
    const GridSpec g = grid_spec(dims, spacing, model);
    check_cross_rows(m, n, row0, mloc);
    GSI_REQUIRE(target_idx || m == g.n, GSI_ERR_INVALID_ARGUMENT,
                "kernelcov_cross_grid: without target indices m must be the number of grid nodes");
    GSI_REQUIRE(source_idx || n == g.n, GSI_ERR_INVALID_ARGUMENT,
                "kernelcov_cross_grid: without source indices n must be the number of grid nodes");
    for (int64_t i = 0; target_idx && i < m; ++i)
        GSI_REQUIRE(target_idx[i] >= 0 && target_idx[i] < g.n, GSI_ERR_INVALID_ARGUMENT,
                    "kernelcov_cross_grid: target index outside the grid");
    for (int64_t j = 0; source_idx && j < n; ++j)
        GSI_REQUIRE(source_idx[j] >= 0 && source_idx[j] < g.n, GSI_ERR_INVALID_ARGUMENT,
                    "kernelcov_cross_grid: source index outside the grid");
    check_table_size(g);
    std::unique_ptr<gsi_op, OpAbort> op(new gsi_op());
    op->ctx = ctx;
    set_model(op.get(), model, 0.0, false);
    op->type = OP_KERNELCROSS;
    op->m = m; op->n = n; op->row0 = row0; op->mloc = mloc;
    upload_table(ctx, op.get(), model, g);
    upload_lattice(ctx, g, n, source_idx, op->lattice, op->n_pad);
    if (target_idx) {
        upload_lattice(ctx, g, mloc, target_idx + row0, op->lattice_t, op->nt_pad);
    } else {
        std::vector<int64_t> rows((size_t)mloc);
        for (int64_t i = 0; i < mloc; ++i) rows[(size_t)i] = row0 + i;
        upload_lattice(ctx, g, mloc, rows.data(), op->lattice_t, op->nt_pad);
    }
    set_partition(op.get());
    ctx_retain(ctx);
    *out = op.release();
}
}  // namespace gsi

GSI_API int32_t gsi_op_kernelcov(gsi_ctx* ctx, int32_t kind, int32_t d, int64_t n, const double* coords,
                                 const double* ell, double sigma2, double nugget, double beta, int64_t row0,
                                 int64_t mloc, gsi_op** out) {
    return guarded([&] {
        use(ctx);
        GSI_REQUIRE(coords && ell && out, GSI_ERR_INVALID_ARGUMENT, "null argument");
        GSI_REQUIRE(d >= 1 && d <= 3, GSI_ERR_UNSUPPORTED, "kernelcov: d must be 1, 2 or 3");
        GSI_REQUIRE(kind >= GSI_KERNEL_EXPONENTIAL && kind <= GSI_KERNEL_SPHERICAL, GSI_ERR_INVALID_ARGUMENT,
                    "kernelcov: unknown kernel kind");
        GSI_REQUIRE(n >= 1 && row0 >= 0 && mloc >= 0 && row0 + mloc <= n, GSI_ERR_INVALID_ARGUMENT, "kernelcov: bad row block");
        for (int k = 0; k < d; ++k) GSI_REQUIRE(ell[k] > 0.0, GSI_ERR_INVALID_ARGUMENT, "kernelcov: length scales must be positive");
        make_kernelcov(ctx, n, coords, single_structure(kind, d, ell, sigma2, beta), nugget, row0, mloc, out);
    });
}

GSI_API int32_t gsi_op_kernelcov_grid(gsi_ctx* ctx, int32_t kind, int32_t d, const int64_t* dims, const double* spacing,
                                      const double* ell, double sigma2, double nugget, double beta, int64_t row0,
                                      int64_t mloc, gsi_op** out) {
    return guarded([&] {
        use(ctx);
        GSI_REQUIRE(dims && spacing && ell && out, GSI_ERR_INVALID_ARGUMENT, "null argument");
        GSI_REQUIRE(d >= 1 && d <= 3, GSI_ERR_UNSUPPORTED, "kernelcov_grid: d must be 1, 2 or 3");
        GSI_REQUIRE(kind >= GSI_KERNEL_EXPONENTIAL && kind <= GSI_KERNEL_SPHERICAL, GSI_ERR_INVALID_ARGUMENT,
                    "kernelcov_grid: unknown kernel kind");
        for (int k = 0; k < d; ++k)
            GSI_REQUIRE(dims[k] >= 1 && ell[k] > 0.0, GSI_ERR_INVALID_ARGUMENT, "kernelcov_grid: bad dims / length scales");
        make_kernelcov_grid(ctx, dims, spacing, single_structure(kind, d, ell, sigma2, beta), nugget, row0, mloc, out);
    });
}

GSI_API int32_t gsi_op_kernelcov_model(gsi_ctx* ctx, int32_t d, int64_t n, const double* coords, int32_t nstruct,
                                       const int32_t* kinds, const double* sills, const double* ranges,
                                       const double* rotations, const double* betas, double nugget, int64_t row0,
                                       int64_t mloc, gsi_op** out) {
    return guarded([&] {
        use(ctx);
        GSI_REQUIRE(coords && kinds && sills && ranges && out, GSI_ERR_INVALID_ARGUMENT, "null argument");
        GSI_REQUIRE(d >= 1 && d <= 3, GSI_ERR_UNSUPPORTED, "kernelcov_model: d must be 1, 2 or 3");
        const CovModel m = model_from_args(d, nstruct, kinds, sills, ranges, rotations, betas);
        make_kernelcov(ctx, n, coords, m, nugget, row0, mloc, out);
    });
}

GSI_API int32_t gsi_op_kernelcov_model_grid(gsi_ctx* ctx, int32_t d, const int64_t* dims, const double* spacing,
                                            int32_t nstruct, const int32_t* kinds, const double* sills,
                                            const double* ranges, const double* rotations, const double* betas,
                                            double nugget, int64_t row0, int64_t mloc, gsi_op** out) {
    return guarded([&] {
        use(ctx);
        GSI_REQUIRE(dims && spacing && kinds && sills && ranges && out, GSI_ERR_INVALID_ARGUMENT, "null argument");
        GSI_REQUIRE(d >= 1 && d <= 3, GSI_ERR_UNSUPPORTED, "kernelcov_model_grid: d must be 1, 2 or 3");
        const CovModel m = model_from_args(d, nstruct, kinds, sills, ranges, rotations, betas);
        make_kernelcov_grid(ctx, dims, spacing, m, nugget, row0, mloc, out);
    });
}

GSI_API int32_t gsi_op_kernelcov_cross(gsi_ctx* ctx, int32_t d, int64_t m, const double* targets, int64_t n,
                                       const double* sources, int32_t nstruct, const int32_t* kinds, const double* sills,
                                       const double* ranges, const double* rotations, const double* betas, int64_t row0,
                                       int64_t mloc, gsi_op** out) {
    return guarded([&] {
        use(ctx);
        GSI_REQUIRE(targets && sources && kinds && sills && ranges && out, GSI_ERR_INVALID_ARGUMENT, "null argument");
        GSI_REQUIRE(d >= 1 && d <= 3, GSI_ERR_UNSUPPORTED, "kernelcov_cross: d must be 1, 2 or 3");
        const CovModel model = model_from_args(d, nstruct, kinds, sills, ranges, rotations, betas);
        make_kernelcross(ctx, m, targets, n, sources, model, row0, mloc, out);
    });
}

GSI_API int32_t gsi_op_kernelcov_cross_grid(gsi_ctx* ctx, int32_t d, const int64_t* dims, const double* spacing,
                                            int64_t m, const int64_t* target_idx, int64_t n, const int64_t* source_idx,
                                            int32_t nstruct, const int32_t* kinds, const double* sills,
                                            const double* ranges, const double* rotations, const double* betas,
                                            int64_t row0, int64_t mloc, gsi_op** out) {
    return guarded([&] {
        use(ctx);
        GSI_REQUIRE(dims && spacing && kinds && sills && ranges && out, GSI_ERR_INVALID_ARGUMENT, "null argument");
        GSI_REQUIRE(d >= 1 && d <= 3, GSI_ERR_UNSUPPORTED, "kernelcov_cross_grid: d must be 1, 2 or 3");
        const CovModel model = model_from_args(d, nstruct, kinds, sills, ranges, rotations, betas);
        make_kernelcross_grid(ctx, dims, spacing, m, target_idx, n, source_idx, model, row0, mloc, out);
    });
}

GSI_API int32_t gsi_op_free(gsi_op* op) {
    if (!op) return GSI_OK;
    return guarded([&] {
        cudaSetDevice(op->ctx->device);
        if (op->ucoords) cudaFree(op->ucoords);
        if (op->table) cudaFree(op->table);
        if (op->lattice) cudaFree(op->lattice);
        if (op->ucoords_t) cudaFree(op->ucoords_t);
        if (op->lattice_t) cudaFree(op->lattice_t);
        if (op->tmpT) BufDeleter()(op->tmpT);
        gsi_ctx* octx = op->ctx;
        delete op;
        ctx_release(octx);
    });
}

GSI_API int32_t gsi_op_size(const gsi_op* op, int64_t* m, int64_t* n) {
    return guarded([&] {
        GSI_REQUIRE(op != nullptr, GSI_ERR_INVALID_ARGUMENT, "null operator");
        if (m) *m = op->m;
        if (n) *n = op->n;
    });
}

GSI_API int32_t gsi_op_apply(gsi_op* op, int32_t trans, const gsi_buf* X, gsi_buf* Y) {
    return guarded([&] {
        GSI_REQUIRE(op && X && Y, GSI_ERR_INVALID_ARGUMENT, "null argument");
        use(op->ctx);
        op_apply(op, op_symmetric(op) ? 0 : trans, X, Y);
        GSI_CUDA(cudaStreamSynchronize(op->ctx->stream));
    });
}

// ---- building blocks
GSI_API int32_t gsi_lu_L(gsi_ctx* ctx, gsi_buf* Y) {
    return guarded([&] {
        use(ctx);
        GSI_REQUIRE(Y != nullptr, GSI_ERR_INVALID_ARGUMENT, "null buffer");
        lu_reset_flag(ctx);
        lu_L_inplace(ctx, Y);
        lu_check_singular(ctx);
    });
}

GSI_API int32_t gsi_qr_thinQ(gsi_ctx* ctx, gsi_buf* Y, double* R_host, int64_t ldr) {
    return guarded([&] {
        use(ctx);
        GSI_REQUIRE(Y != nullptr, GSI_ERR_INVALID_ARGUMENT, "null buffer");
        const int l = (int)Y->cols;
        double* Rdev = nullptr;
        if (R_host) {
            GSI_REQUIRE(ldr >= l, GSI_ERR_INVALID_ARGUMENT, "qr: ldr < l");
            GSI_CUDA(cudaMalloc(&Rdev, (size_t)l * l * sizeof(double)));
        }
        std::unique_ptr<double, void (*)(double*)> guard(Rdev, [](double* p) { if (p) cudaFree(p); });
        lu_reset_flag(ctx);
        qr_thinQ_inplace(ctx, Y, Rdev);
        if (R_host)
            GSI_CUDA(cudaMemcpy2DAsync(R_host, ldr * 8, Rdev, (size_t)l * 8, (size_t)l * 8, l, cudaMemcpyDeviceToHost, ctx->stream));
        lu_check_singular(ctx);              // synchronises; reports a panel-exchange time-out
    });
}

GSI_API int32_t gsi_svd_small(gsi_ctx* ctx, double* M_host, int64_t ldm, int64_t l, double* sigma_host) {
    return guarded([&] {
        use(ctx);
        GSI_REQUIRE(M_host && sigma_host, GSI_ERR_INVALID_ARGUMENT, "null argument");
        GSI_REQUIRE(l >= 1 && l <= kMaxWideCols && ldm >= l, GSI_ERR_INVALID_ARGUMENT, "svd_small: bad size");
        double* dev = nullptr;
        GSI_CUDA(cudaMalloc(&dev, ((size_t)2 * l * l + l) * sizeof(double)));
        std::unique_ptr<double, void (*)(double*)> guard(dev, [](double* p) { cudaFree(p); });
        double* U = dev + (size_t)l * l;
        double* sig = dev + (size_t)2 * l * l;
        GSI_CUDA(cudaMemcpy2DAsync(dev, (size_t)l * 8, M_host, ldm * 8, (size_t)l * 8, l, cudaMemcpyHostToDevice, ctx->stream));
        svd_small(ctx, dev, (int)l, U, sig);
        GSI_CUDA(cudaMemcpy2DAsync(M_host, ldm * 8, U, (size_t)l * 8, (size_t)l * 8, l, cudaMemcpyDeviceToHost, ctx->stream));
        GSI_CUDA(cudaMemcpyAsync(sigma_host, sig, (size_t)l * 8, cudaMemcpyDeviceToHost, ctx->stream));
        GSI_CUDA(cudaStreamSynchronize(ctx->stream));
    });
}

// ---- algorithms
GSI_API int32_t gsi_rangefinder_fixed(gsi_op* op, const gsi_buf* Omega, int64_t q, int32_t normaliser, gsi_buf* Q_out) {
    return guarded([&] {
        GSI_REQUIRE(op && Omega && Q_out, GSI_ERR_INVALID_ARGUMENT, "null argument");
        use(op->ctx);
        rangefinder_fixed(op, Omega, q, normaliser, Q_out);
    });
}

GSI_API int32_t gsi_randsvd(gsi_op* op, const gsi_buf* Omega, int64_t K, int64_t p, int64_t q, int32_t normaliser,
                            gsi_buf* Z_out, double* S_host) {
    return guarded([&] {
        GSI_REQUIRE(op && Omega && Z_out, GSI_ERR_INVALID_ARGUMENT, "null argument");
        use(op->ctx);
        if (q < 0)
            throw Error(GSI_ERR_NEGATIVE_ITERATIONS,
                        "parameter numiterations should be positive, but numiterations=" + std::to_string(q));
        randsvd(op, Omega, K, p, q, normaliser, Z_out, S_host);
    });
}

GSI_API int32_t gsi_kernelcov_solve(gsi_op* op, const gsi_buf* B, const gsi_buf* Omega, double rtol, int64_t maxiter,
                                    gsi_buf* X, int64_t* iters_out, double* relres_out, double* lambda_out) {
    return guarded([&] {
        GSI_REQUIRE(op && B && X && iters_out && relres_out, GSI_ERR_INVALID_ARGUMENT, "null argument");
        use(op->ctx);
        kernelcov_solve(op, B, Omega, rtol, maxiter, X, iters_out, relres_out, lambda_out);
    });
}

GSI_API int32_t gsi_op_kernelcov_block(gsi_op* op, int64_t row0, int64_t col0, gsi_buf* out) {
    return guarded([&] {
        GSI_REQUIRE(op && out, GSI_ERR_INVALID_ARGUMENT, "null argument");
        use(op->ctx);
        GSI_REQUIRE(op->type == OP_KERNELCOV || op->type == OP_KERNELCROSS, GSI_ERR_UNSUPPORTED,
                    "kernelcov_block needs a kernel-covariance operator");
        GSI_REQUIRE(out->layout == GSI_LAYOUT_COLMAJOR, GSI_ERR_DIMENSION_MISMATCH, "kernelcov_block: out must be COLMAJOR");
        const bool cross = op->type == OP_KERNELCROSS;
        const int64_t nrows = cross ? op->mloc : op->n;
        GSI_REQUIRE(row0 >= 0 && col0 >= 0 && row0 + out->rows <= nrows && col0 + out->cols <= op->n,
                    GSI_ERR_DIMENSION_MISMATCH, "kernelcov_block: the block lies outside the operator");
        KcovBlock b;
        b.r0 = row0; b.rows = out->rows; b.c0 = col0; b.cols = out->cols;
        b.nr_valid = nrows; b.nc_valid = op->n; b.nugget_diag = cross ? 0 : 1; b.lower = 0;
        b.out = out->d; b.rs = 1; b.cs = out->ld;
        kcov_block(op, cross ? KB_CROSS : KB_SQUARE, b);
        GSI_CUDA(cudaStreamSynchronize(op->ctx->stream));
    });
}

GSI_API int32_t gsi_kernelcov_chol(gsi_op* op, gsi_chol** out, int64_t* failed_column_out) {
    if (failed_column_out) *failed_column_out = 0;
    return guarded([&] {
        GSI_REQUIRE(op && out, GSI_ERR_INVALID_ARGUMENT, "null argument");
        use(op->ctx);
        *out = nullptr;
        gsi_chol* f = chol_factor(op, nullptr, failed_column_out);
        ctx_retain(op->ctx);
        *out = f;
    });
}

GSI_API int32_t gsi_kernelcov_chol_diag(gsi_op* op, const double* diag, gsi_chol** out, int64_t* failed_column_out) {
    if (failed_column_out) *failed_column_out = 0;
    return guarded([&] {
        GSI_REQUIRE(op && out, GSI_ERR_INVALID_ARGUMENT, "null argument");
        use(op->ctx);
        *out = nullptr;
        gsi_chol* f = chol_factor(op, diag, failed_column_out);
        ctx_retain(op->ctx);
        *out = f;
    });
}

GSI_API int32_t gsi_chol_free(gsi_chol* f) {
    if (!f) return GSI_OK;
    return guarded([&] {
        gsi_ctx* c = f->ctx;
        chol_destroy(f);
        ctx_release(c);
    });
}

GSI_API int32_t gsi_chol_size(const gsi_chol* f, int64_t* n_out) {
    return guarded([&] {
        GSI_REQUIRE(f && n_out, GSI_ERR_INVALID_ARGUMENT, "null argument");
        *n_out = f->n;
    });
}

GSI_API int32_t gsi_chol_logdet(const gsi_chol* f, double* logdet_out) {
    return guarded([&] {
        GSI_REQUIRE(f && logdet_out, GSI_ERR_INVALID_ARGUMENT, "null argument");
        *logdet_out = f->logdet;
    });
}

GSI_API int32_t gsi_chol_download(const gsi_chol* f, double* L_host, int64_t ldh) {
    return guarded([&] {
        GSI_REQUIRE(f, GSI_ERR_INVALID_ARGUMENT, "null factor");
        use(f->ctx);
        chol_download(f, L_host, ldh);
    });
}

GSI_API int32_t gsi_chol_solve(gsi_chol* f, int32_t half, const gsi_buf* B, gsi_buf* X) {
    return guarded([&] {
        GSI_REQUIRE(f && B && X, GSI_ERR_INVALID_ARGUMENT, "null argument");
        use(f->ctx);
        chol_solve(f, half, B, X);
    });
}

GSI_API int32_t gsi_chol_krige_variance(gsi_chol* f, gsi_op* cross, const double* F_s, const double* F_t, int64_t p,
                                        double* var_out) {
    return guarded([&] {
        GSI_REQUIRE(f && cross && var_out, GSI_ERR_INVALID_ARGUMENT, "null argument");
        use(f->ctx);
        chol_variance(f, cross, F_s, F_t, p, var_out);
    });
}

GSI_API int32_t gsi_chol_simulate(gsi_chol* f, int64_t ns, const double* y, const double* F_s, const double* F_t,
                                  int64_t p, const gsi_buf* Xi, gsi_buf* Z) {
    return guarded([&] {
        GSI_REQUIRE(f && Xi && Z, GSI_ERR_INVALID_ARGUMENT, "null argument");
        use(f->ctx);
        chol_simulate(f, ns, y, F_s, F_t, p, Xi, Z);
    });
}

GSI_API int32_t gsi_kernelcov_loglik(gsi_op* op, const double* y, const double* F, int64_t p, int32_t reml,
                                     double* loglik_out, double* beta_out, double* grad_out, int64_t* failed_column_out) {
    if (failed_column_out) *failed_column_out = 0;
    return guarded([&] {
        GSI_REQUIRE(op && y && loglik_out, GSI_ERR_INVALID_ARGUMENT, "null argument");
        use(op->ctx);
        chol_loglik(op, y, F, p, reml, loglik_out, beta_out, grad_out, failed_column_out);
    });
}

GSI_API int32_t gsi_chol_crossval(gsi_chol* f, const double* y, const double* F, int64_t p, int64_t ngroups,
                                  const int64_t* group_ptr, const int64_t* group_idx, double* err_out, double* var_out,
                                  double* logpdf_out, int64_t* failed_group_out) {
    if (failed_group_out) *failed_group_out = 0;
    return guarded([&] {
        GSI_REQUIRE(f && y && err_out && var_out, GSI_ERR_INVALID_ARGUMENT, "null argument");
        use(f->ctx);
        chol_crossval(f, y, F, p, ngroups, group_ptr, group_idx, err_out, var_out, logpdf_out, failed_group_out);
    });
}
