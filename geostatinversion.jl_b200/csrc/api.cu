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
        std::unique_ptr<gsi_op, OpAbort> op(new gsi_op());
        op->ctx = ctx; op->type = OP_KERNELCOV; op->kind = kind; op->dim = d;
        op->m = op->n = n; op->row0 = row0; op->mloc = mloc;
        op->sigma2 = sigma2; op->nugget = nugget; op->beta = beta;
        op->n_pad = round_up(n, kRowPad);
        // scaled SoA coordinates u[k][j] = x_j[k] / ell[k]; padding repeats the last point.
        // Gaussian: an extra 1/sqrt(2) folds the factor 1/2 of exp(-r2/2) into r2; Matern nu = 3/2 / 5/2: an extra
        // sqrt(3) / sqrt(5), so the kernel's sqrt(r2) is the argument sqrt(2 nu) r of exp and of the polynomial.
        const double pre = kind == GSI_KERNEL_GAUSSIAN   ? 0.70710678118654752440
                           : kind == GSI_KERNEL_MATERN32 ? 1.73205080756887729353
                           : kind == GSI_KERNEL_MATERN52 ? 2.23606797749978969641
                                                         : 1.0;
        std::vector<double> u((size_t)3 * op->n_pad, 0.0);
        for (int k = 0; k < d; ++k) {
            double* uk = u.data() + (size_t)k * op->n_pad;
            for (int64_t j = 0; j < n; ++j) uk[j] = (coords[j * d + k] / ell[k]) * pre;
            for (int64_t j = n; j < op->n_pad; ++j) uk[j] = uk[n - 1];
        }
        GSI_CUDA(cudaMalloc(&op->ucoords, u.size() * sizeof(double)));
        GSI_CUDA(cudaMemcpyAsync(op->ucoords, u.data(), u.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        GSI_CUDA(cudaStreamSynchronize(ctx->stream));
        set_partition(op.get());
        ctx_retain(ctx);
        *out = op.release();
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
        int64_t nd[3] = {1, 1, 1};
        double h[3] = {1, 1, 1}, el[3] = {1, 1, 1};
        int64_t n = 1;
        for (int k = 0; k < d; ++k) {
            GSI_REQUIRE(dims[k] >= 1 && ell[k] > 0.0, GSI_ERR_INVALID_ARGUMENT, "kernelcov_grid: bad dims / length scales");
            nd[k] = dims[k]; h[k] = spacing[k]; el[k] = ell[k];
            n *= dims[k];
        }
        GSI_REQUIRE(n < ((int64_t)1 << 31), GSI_ERR_UNSUPPORTED, "kernelcov_grid: more than 2^31 points");
        GSI_REQUIRE(row0 >= 0 && mloc >= 0 && row0 + mloc <= n, GSI_ERR_INVALID_ARGUMENT, "kernelcov_grid: bad row block");
        std::unique_ptr<gsi_op, OpAbort> op(new gsi_op());
        op->ctx = ctx; op->type = OP_KERNELCOV; op->kind = kind; op->dim = d;
        op->m = op->n = n; op->row0 = row0; op->mloc = mloc;
        op->sigma2 = sigma2; op->nugget = nugget; op->beta = beta;
        op->n_pad = round_up(n, kRowPad);
        op->grid_nx = (int)nd[0]; op->grid_ny = (int)nd[1]; op->grid_nz = (int)nd[2];
        // kernel value of every lattice offset (libm, same formula as the dense definition)
        std::vector<double> tab((size_t)n);
        for (int64_t dz = 0; dz < nd[2]; ++dz)
            for (int64_t dy = 0; dy < nd[1]; ++dy)
                for (int64_t dx = 0; dx < nd[0]; ++dx) {
                    const double ux = (dx * h[0]) / el[0], uy = (dy * h[1]) / el[1], uz = (dz * h[2]) / el[2];
                    double r2 = ux * ux;
                    if (d > 1) r2 += uy * uy;
                    if (d > 2) r2 += uz * uz;
                    double v;
                    if (kind == GSI_KERNEL_EXPONENTIAL) v = std::exp(-std::sqrt(r2));
                    else if (kind == GSI_KERNEL_GAUSSIAN) v = std::exp(-0.5 * r2);
                    else if (kind == GSI_KERNEL_MATERN32) {
                        const double s = std::sqrt(3.0 * r2);
                        v = (1.0 + s) * std::exp(-s);
                    } else if (kind == GSI_KERNEL_MATERN52) {
                        const double s = std::sqrt(5.0 * r2);
                        v = (1.0 + s + s * s / 3.0) * std::exp(-s);
                    } else if (kind == GSI_KERNEL_SPHERICAL) {
                        const double r = std::sqrt(r2);
                        v = r < 1.0 ? 0.5 * (1.0 - r) * (1.0 - r) * (2.0 + r) : 0.0;   // = 1 - 1.5 r + 0.5 r^3, no cancellation
                    } else v = std::exp(-beta * std::log1p(r2));
                    tab[(size_t)(dx + nd[0] * (dy + nd[1] * dz))] = v;
                }
        // lattice indices of every point (SoA, padding repeats the last point)
        std::vector<int> lat((size_t)3 * op->n_pad, 0);
        for (int64_t j = 0; j < op->n_pad; ++j) {
            const int64_t jj = j < n ? j : n - 1;
            lat[(size_t)0 * op->n_pad + j] = (int)(jj % nd[0]);
            lat[(size_t)1 * op->n_pad + j] = (int)((jj / nd[0]) % nd[1]);
            lat[(size_t)2 * op->n_pad + j] = (int)(jj / (nd[0] * nd[1]));
        }
        GSI_CUDA(cudaMalloc(&op->table, tab.size() * sizeof(double)));
        GSI_CUDA(cudaMalloc(&op->lattice, lat.size() * sizeof(int)));
        GSI_CUDA(cudaMemcpyAsync(op->table, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        GSI_CUDA(cudaMemcpyAsync(op->lattice, lat.data(), lat.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
        GSI_CUDA(cudaStreamSynchronize(ctx->stream));
        set_partition(op.get());
        ctx_retain(ctx);
        *out = op.release();
    });
}

GSI_API int32_t gsi_op_free(gsi_op* op) {
    if (!op) return GSI_OK;
    return guarded([&] {
        cudaSetDevice(op->ctx->device);
        if (op->ucoords) cudaFree(op->ucoords);
        if (op->table) cudaFree(op->table);
        if (op->lattice) cudaFree(op->lattice);
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
        const bool sym = op->type != OP_DENSE;
        op_apply(op, sym ? 0 : trans, X, Y);
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
