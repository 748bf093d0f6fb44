// Internal definitions shared by the .cu translation units of libsd_b200.so.
// Nothing here is part of the C ABI (include/sd_b200.h).
#pragma once

#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "sd_b200.h"

#define SD_MAX_EYES 4
#define SD_MAX_BINS 16   // undirected orientations K supported by the HOG kernel

enum { SD_WS_GRAM_EXT = 0, SD_WS_FEATURES, SD_WS_SCRATCH, SD_WS_DIAGINV,
       SD_WS_PARTIAL, SD_WS_GEOM, SD_WS_GEMM_PARTIAL, SD_WS_DIAGINV2, SD_WS_PANEL, SD_WS_BIAS, SD_WS_CG, SD_WS_CGMAT, SD_WS_COUNT };

// Block-row ownership of a distributed factorisation: global row r of the matrix belongs to rank (r / block) % nranks.
// first_row = global row of the first row of the C sub-matrix a kernel is launched on.
struct sd_row_filter {
    int block;
    int nranks, rank;
    int64_t first_row;
};

struct sd_comm;   // sd_comm.cu

struct sd_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaStream_t copy_stream = nullptr;   // host<->device staging for sd_detect_batch_host
    cudaStream_t chain_stream = nullptr;  // Cholesky look-ahead: next panel's diagonal blocks while the trailing update runs
    cudaEvent_t chain_ev[2] = {nullptr, nullptr};
    int syrk_sm_reserve = 0;              // SMs the persistent SYRK leaves free (1 while a look-ahead chain runs beside it)
    std::string err;
    std::vector<int2> tile_scratch;       // host side of the tensor-core tile lists
    int64_t launches = 0;
    int sm_count = 148;
    int gram_mode = 0;
    int solver_mode = 0;           // systems with D > 256: 0 = blocked Cholesky, 1 = conjugate gradients (Cholesky if they stall)
    int cg_iterations = 0;         // of the last solve (0: the factorisation ran)
    cudaEvent_t cg_ev[8] = {};     // convergence read-backs of the CG loop (the host runs a few iterations ahead of them)
    int64_t roi_fallbacks = 0;     // faces repeated from the full frame because a patch left its ROI
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    void* hog_lut[SD_MAX_BINS + 1] = {};   // per K: (gx,gy) -> orientation bin table (sd_hog.cu)
    void* ws[SD_WS_COUNT] = {};
    size_t ws_bytes[SD_WS_COUNT] = {};
    // pinned scratch for small device->host results (lambda, residual, status flags)
    void* h_scratch = nullptr;
    void* d_scratch = nullptr;   // 4 KB
    // staging buffers of sd_detect_batch_host
    void* d_stage[2] = {nullptr, nullptr};
    size_t stage_bytes[2] = {0, 0};
    cudaEvent_t stage_ev[2] = {nullptr, nullptr};
    cudaEvent_t stage_done[2] = {nullptr, nullptr};
};

int sd_fail(sd_ctx* ctx, int code, const char* fmt, ...);
int sd_check_cuda(sd_ctx* ctx, cudaError_t e, const char* what);
// grow-only workspace; returns nullptr (and sets the error) on failure
void* sd_workspace(sd_ctx* ctx, int slot, size_t bytes);

#define SD_CUDA(ctx, call)                                                        \
    do {                                                                          \
        cudaError_t _e = (call);                                                  \
        if (_e != cudaSuccess) return sd_check_cuda((ctx), _e, #call);            \
    } while (0)

#define SD_LAUNCH_CHECK(ctx, name)                                                \
    do {                                                                          \
        (ctx)->launches++;                                                        \
        cudaError_t _e = cudaGetLastError();                                      \
        if (_e != cudaSuccess) return sd_check_cuda((ctx), _e, name);             \
    } while (0)

#define SD_REQUIRE(ctx, cond, msg)                                                \
    do {                                                                          \
        if (!(cond)) return sd_fail((ctx), SD_ERR_INVALID, "%s: %s", __func__, msg); \
    } while (0)

static inline int sd_div_up(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// ---- internal entry points shared between translation units ---------------------------------

// C[i,j] = beta*C[i,j] + alpha * sum_{k<K} S[k,i] * S[k,j]   for i < MI, j < NJ, restricted to the
// tiles that intersect j >= i (upper triangle).  S: K x NJ row-major (lds), C: MI x NJ (ldc).
// Used for the Gram matrix [A^T A | A^T B] and for the Cholesky trailing update.
// path: 0 = choose by size, 1 = tensor cores whenever the operands allow it, 2 = fp32 SIMT.  A factorisation step
// passes the same choice for every piece of one rank-k update (mixing the two kernels inside one update was measured
// to double the error of the solved weights).  unbiased_split: round the hi operand (gram mode 3) for this call.
int sd_syrk_update(sd_ctx* ctx, const float* d_S, int64_t lds, int K, int MI, int NJ,
                   float* d_C, int64_t ldc, float alpha, float beta, int path = 0, bool unbiased_split = false,
                   const sd_row_filter* rows = nullptr);
int sd_syrk_simt(sd_ctx* ctx, const float* d_S, int64_t lds, int K, int MI, int NJ,
                 float* d_C, int64_t ldc, float alpha, float beta);
int sd_syrk_tc(sd_ctx* ctx, const float* d_S, int64_t lds, int K, int MI, int NJ,
               float* d_C, int64_t ldc, float alpha, float beta, int passes, bool unbiased_split = false,
               const sd_row_filter* rows = nullptr);
// C = beta*C + alpha * SA^T SB on the tensor cores (SA: K x MI, SB: K x NJ, row-major); see sd_gram_tc.cu
int sd_gemm_tn_tc(sd_ctx* ctx, const float* d_SA, int64_t lda, const float* d_SB, int64_t ldb, int K, int MI, int NJ,
                  float* d_C, int64_t ldc, float alpha, float beta, int passes, bool unbiased_split, bool upper_only,
                  const sd_row_filter* rows = nullptr, int ksplit = 1);
bool sd_syrk_tc_supported(const float* d_S, int64_t lds, int K, int MI, int NJ, const float* d_C, int64_t ldc);

int sd_check_hog_status(sd_ctx* ctx, const char* what);   // sd_api.cu: synchronises, reports and clears the projection's flags

// one B,G,R frame -> 8UC1 conversion of a bgr2gray_kernel launch (sd_hog.cu); offsets in bytes from the launch's base pointers
struct sd_bgr2gray_job {
    int64_t src_offset, dst_offset;
    int32_t width, height;
    int64_t src_row_stride, dst_row_stride;
};
// cv::cvtColor(BGR2GRAY) of `count` frames in one launch on `stream`: jobs[j] (d_jobs, device) or, with d_jobs == NULL, `uniform`
// moved by j image strides.  max_groups: the most 4-pixel groups (height x ceil(width / 4)) of any one frame.
int sd_bgr2gray_launch(sd_ctx* ctx, cudaStream_t stream, const uint8_t* d_bgr, uint8_t* d_gray, const sd_bgr2gray_job& uniform,
                       int64_t bgr_image_stride, int64_t gray_image_stride, const sd_bgr2gray_job* d_jobs, int count,
                       int64_t max_groups);

// numerical rank of the symmetric matrix whose upper triangle is in d_G (pivoted Cholesky, sd_rank.cu); rank -1: not computed
int sd_gram_rank(sd_ctx* ctx, const float* d_G, int64_t ldg, int D, int* rank_out, float* first_pivot, float* last_pivot);

// prepared launches of the tensor-core TN-GEMM (sd_gram_tc.cu): plan_storage = SD_TC_PLAN_BYTES bytes, 64-byte aligned
#define SD_TC_PLAN_BYTES 640
int sd_gemm_tn_tc_prepare(sd_ctx* ctx, const float* d_SA, int64_t lda, const float* d_SB, int64_t ldb, int K, int MI, int NJ,
                          float* d_C, int64_t ldc, float alpha, float beta, int passes, bool unbiased_split, bool upper_only,
                          const sd_row_filter* rows, int ksplit, void* d_tiles_buf, void* plan_storage, bool* empty,
                          bool narrow = false /* a single tile column of <= 192 columns may use the narrow-N kernel variants */,
                          int a_strip_rows = 0 /* > 0: operand A strip-major, see sd_gram_tc.cu */);
int sd_gemm_tn_tc_launch(sd_ctx* ctx, const void* plan_storage);

// multi-GPU helpers (sd_comm.cu); a null communicator is a single rank
int sd_comm_rank_of(const sd_comm* c);
int sd_comm_size_of(const sd_comm* c);
int sd_comm_bcast(sd_ctx* ctx, sd_comm* c, float* d_buf, size_t count, int root, cudaStream_t stream);
int sd_comm_group_start(sd_ctx* ctx);
int sd_comm_group_end(sd_ctx* ctx);
int sd_comm_allreduce_f64(sd_ctx* ctx, sd_comm* c, double* d_buf, size_t count, cudaStream_t stream);
int sd_comm_allreduce_f32(sd_ctx* ctx, sd_comm* c, float* d_buf, size_t count, cudaStream_t stream);
// conjugate gradients on the tensor cores (sd_cg.cu); SD_ERR_NUMERIC = did not converge, use the factorisation
int sd_cg_solve(sd_ctx* ctx, sd_comm* comm, float* G, int64_t ldg, int n, int col0, int M, float** W_out, int* ldw_out, int* iters);
// rows [k0, k1) of the n x n system whose part of the product S P rank `me` computes in the shared CG route (multiples of 16 rows)
inline void sd_cg_slab(int n, int nranks, int me, int* k0, int* k1)
{
    *k0 = 0; *k1 = n;
    if (nranks > 1) {
        const int per = ((n + nranks - 1) / nranks + 15) / 16 * 16;
        *k0 = me * per < n ? me * per : n;
        *k1 = (me + 1) * per < n ? (me + 1) * per : n;
    }
}
// true when sd_reduce_scatter_gram leaves the rows block-row-cyclic (large, 16-byte aligned systems); smaller ones are all-reduced
bool sd_gram_is_scattered(int D, int64_t ldg, const float* d_G);

// device-side normalisation factors, shared by the HOG and cascade kernels
struct sd_eyes_dev {
    int kind;
    int n_right, n_left;
    int right_idx[SD_MAX_EYES];
    int left_idx[SD_MAX_EYES];
};
int sd_eyes_to_dev(sd_ctx* ctx, const sd_normalisation* n, int num_landmarks, sd_eyes_dev* out);

#ifdef __CUDACC__
// cv::cvtColor(BGR2GRAY) of one 8-bit pixel, OpenCV >= 3 fixed point (15-bit coefficients; SURVEY.md 8c, pinned against cv2)
__device__ __forceinline__ uint32_t sd_bgr2gray_px(uint32_t b, uint32_t g, uint32_t r)
{
    return (3735u * b + 19235u * g + 9798u * r + (1u << 14)) >> 15;
}

// Inter-eye distance exactly as helpers.hpp:136-160 evaluates it: eye centres are float sums
// scaled by the float reciprocal of the count (cv::Vec /= float), the difference is taken in float,
// squares are accumulated in double (cv::norm NORM_L2) and the root is a double sqrt.
__device__ __forceinline__ double sd_device_ied(const float* __restrict__ row, int L, const sd_eyes_dev& e)
{
    float rx = 0.f, ry = 0.f, lx = 0.f, ly = 0.f;
    for (int i = 0; i < e.n_right; ++i) {
        rx = __fadd_rn(rx, row[e.right_idx[i]]);
        ry = __fadd_rn(ry, row[e.right_idx[i] + L]);
    }
    const float ir = __fdiv_rn(1.0f, (float)e.n_right);
    rx = __fmul_rn(rx, ir);
    ry = __fmul_rn(ry, ir);
    for (int i = 0; i < e.n_left; ++i) {
        lx = __fadd_rn(lx, row[e.left_idx[i]]);
        ly = __fadd_rn(ly, row[e.left_idx[i] + L]);
    }
    const float il = __fdiv_rn(1.0f, (float)e.n_left);
    lx = __fmul_rn(lx, il);
    ly = __fmul_rn(ly, il);
    const double dx = (double)__fsub_rn(rx, lx);
    const double dy = (double)__fsub_rn(ry, ly);
    return sqrt(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
}
#endif
