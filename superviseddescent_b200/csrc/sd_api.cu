// Context, error handling and memory helpers of libsd_b200.so (C ABI: include/sd_b200.h).
#include "sd_internal.cuh"

#include <cstring>

int sd_fail(sd_ctx* ctx, int code, const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf;
    return code;
}

int sd_check_cuda(sd_ctx* ctx, cudaError_t e, const char* what)
{
    if (e == cudaSuccess) return SD_OK;
    return sd_fail(ctx, SD_ERR_CUDA, "CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
}

void* sd_workspace(sd_ctx* ctx, int slot, size_t bytes)
{
    if (bytes == 0) bytes = 256;
    if (ctx->ws_bytes[slot] >= bytes) return ctx->ws[slot];
    if (ctx->ws[slot]) {
        // wait for in-flight users before the buffer goes away
        cudaStreamSynchronize(ctx->stream);
        cudaFree(ctx->ws[slot]);
        ctx->ws[slot] = nullptr;
        ctx->ws_bytes[slot] = 0;
    }
    size_t want = bytes + bytes / 8;   // grow-only with slack
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
        want = bytes;
        e = cudaMalloc(&p, want);
    }
    if (e != cudaSuccess) {
        sd_check_cuda(ctx, e, "cudaMalloc(workspace)");
        return nullptr;
    }
    ctx->ws[slot] = p;
    ctx->ws_bytes[slot] = want;
    return p;
}

int sd_eyes_to_dev(sd_ctx* ctx, const sd_normalisation* n, int num_landmarks, sd_eyes_dev* out)
{
    memset(out, 0, sizeof(*out));
    if (!n || n->kind == 0) { out->kind = 0; return SD_OK; }
    if (n->kind != 1) return sd_fail(ctx, SD_ERR_INVALID, "unknown normalisation kind %d", n->kind);
    if (n->n_right < 1 || n->n_right > SD_MAX_EYES || n->n_left < 1 || n->n_left > SD_MAX_EYES)
        return sd_fail(ctx, SD_ERR_INVALID, "eye identifier counts must be in [1,%d]", SD_MAX_EYES);
    out->kind = 1;
    out->n_right = n->n_right;
    out->n_left = n->n_left;
    for (int i = 0; i < n->n_right; ++i) {
        if (n->right_idx[i] < 0 || n->right_idx[i] >= num_landmarks)
            return sd_fail(ctx, SD_ERR_MISSING_ID, "one of given rightEyeIdentifiers ids not present in lms");
        out->right_idx[i] = n->right_idx[i];
    }
    for (int i = 0; i < n->n_left; ++i) {
        if (n->left_idx[i] < 0 || n->left_idx[i] >= num_landmarks)
            return sd_fail(ctx, SD_ERR_MISSING_ID, "one of given leftEyeIdentifiers ids not present in lms");
        out->left_idx[i] = n->left_idx[i];
    }
    return SD_OK;
}

// The projection kernels raise bits in their own status word (d_scratch[1]); every synchronising entry point that consumed
// HOG output reports and clears them, so an error belongs to the call (or the sd_sync) that follows the launch.
int sd_check_hog_status(sd_ctx* ctx, const char* what)
{
    int* h = reinterpret_cast<int*>(ctx->h_scratch) + 1;
    int* d = reinterpret_cast<int*>(ctx->d_scratch) + 1;
    SD_CUDA(ctx, cudaMemcpyAsync(h, d, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    SD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const int st = *h;
    if (st) {
        SD_CUDA(ctx, cudaMemsetAsync(d, 0, sizeof(int), ctx->stream));
        if (st & 2) return sd_fail(ctx, SD_ERR_INVALID, "%s: image index out of range", what);
        if (st & 1) return sd_fail(ctx, SD_ERR_INVALID, "%s: empty HOG patch (inter-eye distance too small)", what);
    }
    return SD_OK;
}

extern "C" {

const char* sd_version(void) { return "superviseddescent_b200 0.1 (sm_100a)"; }

int sd_ctx_create(int device, void* stream, sd_ctx** out)
{
    if (!out) return SD_ERR_INVALID;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0 || device < 0 || device >= count) {
        // no CPU fallback: the product path needs a GPU
        return SD_ERR_CUDA;
    }
    if (cudaSetDevice(device) != cudaSuccess) return SD_ERR_CUDA;
    sd_ctx* ctx = new sd_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->sm_count = prop.multiProcessorCount;
    if (stream == SD_STREAM_OWN) {
        if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return SD_ERR_CUDA; }
        ctx->own_stream = true;
    } else {
        ctx->stream = (cudaStream_t)stream;   // NULL = the CUDA default stream (what torch calls its default stream)
        ctx->own_stream = false;
    }
    // the staging stream outranks the compute stream: its (short) gather / copy work must slip in between
    // the waves of the HOG kernels instead of queueing behind them
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    bool ok = cudaStreamCreateWithPriority(&ctx->copy_stream, cudaStreamNonBlocking, prio_hi) == cudaSuccess;
    for (int i = 0; i < 6 && ok; ++i) ok = cudaEventCreate(&ctx->ev[i]) == cudaSuccess;
    for (int i = 0; i < 2 && ok; ++i) {
        ok = cudaEventCreateWithFlags(&ctx->stage_ev[i], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&ctx->stage_done[i], cudaEventDisableTiming) == cudaSuccess;
    }
    ok = ok && cudaMallocHost(&ctx->h_scratch, 4096) == cudaSuccess && cudaMalloc(&ctx->d_scratch, 4096) == cudaSuccess &&
         cudaMemset(ctx->d_scratch, 0, 4096) == cudaSuccess;
    if (!ok) { sd_ctx_destroy(ctx); return SD_ERR_CUDA; }
    *out = ctx;
    return SD_OK;
}

void sd_ctx_destroy(sd_ctx* ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    for (int i = 0; i < SD_WS_COUNT; ++i) if (ctx->ws[i]) cudaFree(ctx->ws[i]);
    for (int i = 0; i <= SD_MAX_BINS; ++i) if (ctx->hog_lut[i]) cudaFree(ctx->hog_lut[i]);
    for (int i = 0; i < 2; ++i) {
        if (ctx->d_stage[i]) cudaFree(ctx->d_stage[i]);
        if (ctx->stage_ev[i]) cudaEventDestroy(ctx->stage_ev[i]);
        if (ctx->stage_done[i]) cudaEventDestroy(ctx->stage_done[i]);
    }
    for (int i = 0; i < 6; ++i) if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    for (int i = 0; i < 8; ++i) if (ctx->cg_ev[i]) cudaEventDestroy(ctx->cg_ev[i]);
    if (ctx->h_scratch) cudaFreeHost(ctx->h_scratch);
    if (ctx->d_scratch) cudaFree(ctx->d_scratch);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->chain_stream) { cudaStreamSynchronize(ctx->chain_stream); cudaStreamDestroy(ctx->chain_stream); }
    for (int i = 0; i < 2; ++i) if (ctx->chain_ev[i]) cudaEventDestroy(ctx->chain_ev[i]);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char* sd_last_error(const sd_ctx* ctx) { return ctx ? ctx->err.c_str() : "no context (is a CUDA device present?)"; }

int sd_sync(sd_ctx* ctx)
{
    if (!ctx) return SD_ERR_INVALID;
    return sd_check_hog_status(ctx, "sync");                  // synchronises the stream; reports flags raised by sd_hog_batch
}

int64_t sd_launch_count(const sd_ctx* ctx) { return ctx ? ctx->launches : 0; }
int64_t sd_roi_fallback_count(const sd_ctx* ctx) { return ctx ? ctx->roi_fallbacks : 0; }

int sd_malloc(sd_ctx* ctx, size_t bytes, void** d_ptr)
{
    if (!ctx || !d_ptr) return SD_ERR_INVALID;
    SD_CUDA(ctx, cudaSetDevice(ctx->device));
    SD_CUDA(ctx, cudaMalloc(d_ptr, bytes ? bytes : 1));
    return SD_OK;
}

int sd_free(sd_ctx* ctx, void* d_ptr)
{
    if (!ctx) return SD_ERR_INVALID;
    if (d_ptr) { cudaStreamSynchronize(ctx->stream); SD_CUDA(ctx, cudaFree(d_ptr)); }
    return SD_OK;
}

int sd_host_alloc(sd_ctx* ctx, size_t bytes, void** h_ptr)
{
    if (!ctx || !h_ptr) return SD_ERR_INVALID;
    SD_CUDA(ctx, cudaMallocHost(h_ptr, bytes ? bytes : 1));
    return SD_OK;
}

int sd_host_free(sd_ctx* ctx, void* h_ptr)
{
    if (!ctx) return SD_ERR_INVALID;
    if (h_ptr) SD_CUDA(ctx, cudaFreeHost(h_ptr));
    return SD_OK;
}

int sd_memcpy_h2d(sd_ctx* ctx, void* d_dst, const void* h_src, size_t bytes)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_CUDA(ctx, cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return SD_OK;
}

int sd_memcpy_d2h(sd_ctx* ctx, void* h_dst, const void* d_src, size_t bytes)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_CUDA(ctx, cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return SD_OK;
}

int sd_memcpy2d_h2d(sd_ctx* ctx, void* d_dst, size_t dst_pitch, const void* h_src, size_t src_pitch, size_t row_bytes, size_t rows)
{
    if (!ctx) return SD_ERR_INVALID;
    if (rows == 0 || row_bytes == 0) return SD_OK;
    SD_CUDA(ctx, cudaMemcpy2DAsync(d_dst, dst_pitch, h_src, src_pitch, row_bytes, rows, cudaMemcpyHostToDevice, ctx->stream));
    return SD_OK;
}

int sd_memcpy2d_d2h(sd_ctx* ctx, void* h_dst, size_t dst_pitch, const void* d_src, size_t src_pitch, size_t row_bytes, size_t rows)
{
    if (!ctx) return SD_ERR_INVALID;
    if (rows == 0 || row_bytes == 0) return SD_OK;
    SD_CUDA(ctx, cudaMemcpy2DAsync(h_dst, dst_pitch, d_src, src_pitch, row_bytes, rows, cudaMemcpyDeviceToHost, ctx->stream));
    return SD_OK;
}

int sd_memcpy2d_d2d(sd_ctx* ctx, void* d_dst, size_t dst_pitch, const void* d_src, size_t src_pitch, size_t row_bytes, size_t rows)
{
    if (!ctx) return SD_ERR_INVALID;
    if (rows == 0 || row_bytes == 0) return SD_OK;
    SD_CUDA(ctx, cudaMemcpy2DAsync(d_dst, dst_pitch, d_src, src_pitch, row_bytes, rows, cudaMemcpyDeviceToDevice, ctx->stream));
    return SD_OK;
}

int sd_memset(sd_ctx* ctx, void* d_dst, int value, size_t bytes)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_CUDA(ctx, cudaMemsetAsync(d_dst, value, bytes, ctx->stream));
    return SD_OK;
}

int sd_set_gram_mode(sd_ctx* ctx, int mode)
{
    if (!ctx || mode < 0 || mode > 3) return SD_ERR_INVALID;
    ctx->gram_mode = mode;
    return SD_OK;
}

int sd_set_solver(sd_ctx* ctx, int mode)
{
    if (!ctx || mode < 0 || mode > 1) return SD_ERR_INVALID;
    ctx->solver_mode = mode;
    return SD_OK;
}

int sd_solver_iterations(const sd_ctx* ctx) { return ctx ? ctx->cg_iterations : 0; }

int sd_solver_timings(sd_ctx* ctx, float ms_out[4])
{
    if (!ctx || !ms_out) return SD_ERR_INVALID;
    // [0] "At * A", [1] "AtA + Reg", [2] "Decomposition", [3] "solve()"  (verbose_solver.hpp:66-103)
    cudaStreamSynchronize(ctx->stream);
    for (int i = 0; i < 4; ++i) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ctx->ev[i], ctx->ev[i + 1]) != cudaSuccess) { ms = 0.f; cudaGetLastError(); }
        ms_out[i] = ms;
    }
    return SD_OK;
}

}  // extern "C"
