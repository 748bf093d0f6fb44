// LinearRegressor / Solver / cascade-step kernels of libsd_b200.so.
//
//   sd_gram            [A^T A | A^T B]                         regressors.hpp:208,225 (verbose_solver.hpp:67,94)
//   sd_solve_gram      lambda rule + diagonal + factorise/solve regressors.hpp:126-148,215-225
//   sd_learn           = sd_gram + sd_solve_gram                regressors.hpp:345-350
//   sd_predict         values * x                               regressors.hpp:377-381
//   sd_test_residual   ||pred - labels|| / ||labels||           regressors.hpp:361-369
//   sd_cascade_targets b = (x - x_gt) (.) norm(x)               superviseddescent.hpp:199-205
//   sd_cascade_update  x <- x - (A X) (.) 1/norm(x)             superviseddescent.hpp:209-215,296-301,336-339
//
// Factorisation: the reference calls Eigen::PartialPivLU on A^T A + Lambda.  That matrix is symmetric
// positive definite whenever lambda > 0 with an all-ones bias column (SURVEY 7, hard part 2), so for
// D > kLuMaxDim a blocked right-looking Cholesky (G = U^T U) is used, whose trailing update is the same
// "Gram-like" product as A^T A and runs on the tensor-core SYRK (sd_gram_tc.cu).  For D <= kLuMaxDim a
// single-CTA LU with partial pivoting restates the reference's solver operation by operation (this is
// the path the reference's unit tests exercise, including lambda = 0).
#include "sd_internal.cuh"

#include <cmath>
#include <cstring>

namespace {

constexpr int kLuMaxDim = 256;   // D up to which the faithful partial-pivot LU is used
constexpr int kCholNb = 128;     // Cholesky block size

// =================================================================================================
// SIMT SYRK-like update: C[i,j] = beta*C[i,j] + alpha * sum_k S[k,i]*S[k,j]  (upper-triangle tiles)
// =================================================================================================
constexpr int ST = 64;    // tile edge
constexpr int SK = 16;    // k chunk

__global__ void __launch_bounds__(256) syrk_simt_kernel(const float* __restrict__ S, long long lds, int K, int MI, int NJ,
                                                        float* __restrict__ C, long long ldc, float alpha, float beta,
                                                        float* __restrict__ partial, int k_per_split)
{
    const int tj = blockIdx.x, ti = blockIdx.y;
    if (tj * ST + ST - 1 < ti * ST) return;               // tile entirely below the diagonal
    __shared__ __align__(16) float As[SK][ST + 4];
    __shared__ __align__(16) float Bs[SK][ST + 4];
    const int tid = threadIdx.x;
    const int ty = tid >> 4, tx = tid & 15;
    const int i0 = ti * ST, j0 = tj * ST;
    const int kbeg = blockIdx.z * k_per_split;
    const int kend = min(K, kbeg + k_per_split);
    float acc[4][4] = {};
    const int lk = tid >> 4;          // 0..15 : row of the k chunk
    const int lc = (tid & 15) * 4;    // 0..60 : column inside the tile
    for (int k0 = kbeg; k0 < kend; k0 += SK) {
        const int k = k0 + lk;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int ia = i0 + lc + e, jb = j0 + lc + e;
            As[lk][lc + e] = (k < kend && ia < MI) ? S[(long long)k * lds + ia] : 0.f;
            Bs[lk][lc + e] = (k < kend && jb < NJ) ? S[(long long)k * lds + jb] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < SK; ++kk) {
            const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[r][c] = fmaf(av[r], bv[c], acc[r][c]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int i = i0 + ty * 4 + r;
        if (i >= MI) continue;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int j = j0 + tx * 4 + c;
            if (j >= NJ) continue;
            if (partial) {
                partial[((long long)blockIdx.z * MI + i) * NJ + j] = acc[r][c];
            } else {
                float* p = C + (long long)i * ldc + j;
                *p = (beta == 0.f) ? alpha * acc[r][c] : fmaf(alpha, acc[r][c], beta * (*p));
            }
        }
    }
}

__global__ void syrk_reduce_kernel(const float* __restrict__ partial, int splits, int MI, int NJ,
                                   float* __restrict__ C, long long ldc, float alpha, float beta)
{
    const long long total = (long long)MI * NJ;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(idx / NJ), j = (int)(idx - (long long)i * NJ);
        if ((j / ST) * ST + ST - 1 < (i / ST) * ST) continue;      // tile not computed
        float s = 0.f;
        for (int z = 0; z < splits; ++z) s += partial[(long long)z * total + idx];   // fixed order
        float* p = C + (long long)i * ldc + j;
        *p = (beta == 0.f) ? alpha * s : fmaf(alpha, s, beta * (*p));
    }
}

// =================================================================================================
// GEMM NN: C[N x M] = beta*C + alpha * A[N x D] * B[D x M], with the cascade-update epilogue
// =================================================================================================
constexpr int GT = 64, GK = 16;

struct GemmEpilogue {
    int mode;                 // 0: plain store, 1: x_next = x - acc * (1/norm(x))
    const float* x;           // mode 1: current landmarks [N x M]
    float* x_next;
    sd_eyes_dev eyes;
};

// blockIdx.z = split along D; with gridDim.z > 1 every split writes its partial sums (double) to
// `partial` [split][N][M] and gemm_finalize_kernel reduces them in a fixed order.
__global__ void __launch_bounds__(256) gemm_nn_kernel(const float* __restrict__ A, long long lda, int N, int D,
                                                      const float* __restrict__ B, long long ldb, int M,
                                                      float* __restrict__ C, long long ldc, float alpha, float beta,
                                                      const GemmEpilogue ep, double* __restrict__ partial, int k_per_split)
{
    __shared__ __align__(16) float As[GK][GT + 4];     // transposed: As[k][row]
    __shared__ __align__(16) float Bs[GK][GT + 4];
    __shared__ float s_scale[GT];
    const int tid = threadIdx.x;
    const int ty = tid >> 4, tx = tid & 15;
    const int r0 = blockIdx.y * GT, c0 = blockIdx.x * GT;
    const int kbeg = blockIdx.z * k_per_split;
    const int kend = min(D, kbeg + k_per_split);
    if (ep.mode == 1 && !partial && tid < GT) {
        const int r = r0 + tid;
        float inv_n = 1.0f;
        if (r < N && ep.eyes.kind == 1) {
            const double ied = sd_device_ied(ep.x + (long long)r * M, M / 2, ep.eyes);
            const float n = (float)__ddiv_rn(1.0, ied);      // ones / ied           (model.hpp:97)
            inv_n = __fdiv_rn(1.0f, n);                      // 1 / normalisation    (superviseddescent.hpp:213)
        }
        s_scale[tid] = inv_n;
    }
    // cv::gemm accumulates float products in double (the reference's predict, regressors.hpp:379).
    // Here: fp32 FMA inside a 16-deep k chunk, chunk sums added into double accumulators.
    double acc[4][4] = {};
    const int la_r = tid >> 2;           // 0..63 row
    const int la_k = (tid & 3) * 4;      // 0..12 k offset
    const int lb_k = tid >> 4;           // 0..15
    const int lb_c = (tid & 15) * 4;     // 0..60
    const bool a_vec = (lda % 4 == 0) && ((reinterpret_cast<uintptr_t>(A) & 15) == 0) && (kbeg % 4 == 0);
    const bool b_vec = (ldb % 4 == 0) && ((reinterpret_cast<uintptr_t>(B) & 15) == 0);
    for (int k0 = kbeg; k0 < kend; k0 += GK) {
        {
            const int r = r0 + la_r, k = k0 + la_k;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r < N) {
                const float* src = A + (long long)r * lda + k;
                if (a_vec && k + 3 < kend) v = *reinterpret_cast<const float4*>(src);
                else {
                    if (k < kend) v.x = src[0];
                    if (k + 1 < kend) v.y = src[1];
                    if (k + 2 < kend) v.z = src[2];
                    if (k + 3 < kend) v.w = src[3];
                }
            }
            As[la_k][la_r] = v.x; As[la_k + 1][la_r] = v.y; As[la_k + 2][la_r] = v.z; As[la_k + 3][la_r] = v.w;
            const int kb = k0 + lb_k, c = c0 + lb_c;
            float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
            if (kb < kend) {
                const float* src = B + (long long)kb * ldb + c;
                if (b_vec && c + 3 < M) w = *reinterpret_cast<const float4*>(src);
                else {
                    if (c < M) w.x = src[0];
                    if (c + 1 < M) w.y = src[1];
                    if (c + 2 < M) w.z = src[2];
                    if (c + 3 < M) w.w = src[3];
                }
            }
            *reinterpret_cast<float4*>(&Bs[lb_k][lb_c]) = w;
        }
        __syncthreads();
        float part[4][4] = {};
#pragma unroll
        for (int kk = 0; kk < GK; ++kk) {
            const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < 4; ++c) part[r][c] = fmaf(av[r], bv[c], part[r][c]);
        }
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[r][c] += (double)part[r][c];
        __syncthreads();
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int i = r0 + ty * 4 + r;
        if (i >= N) continue;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int j = c0 + tx * 4 + c;
            if (j >= M) continue;
            if (partial) {
                partial[((long long)blockIdx.z * N + i) * M + j] = acc[r][c];
                continue;
            }
            const float accf = (float)acc[r][c];
            if (ep.mode == 1) {
                const float upd = __fmul_rn(accf, s_scale[ty * 4 + r]);
                ep.x_next[(long long)i * M + j] = __fsub_rn(ep.x[(long long)i * M + j], upd);
            } else {
                float* p = C + (long long)i * ldc + j;
                *p = (beta == 0.f) ? alpha * accf : fmaf(alpha, accf, beta * (*p));
            }
        }
    }
}


// ---- skinny-output GEMM of the cascade (LinearRegressor::predict, regressors.hpp:377-381: values * x with 2L output columns) ----
// One THREAD per sample row: it streams its own feature row from HBM (128-bit loads, each 128-byte line is consumed by the
// same thread over 8 loads) and keeps up to 48 output columns in registers; the weight chunk [32 x 48] sits in shared memory
// and every read of it is a broadcast (all lanes the same address: one wavefront), so the inner loop is FFMA-bound: 48 FFMA
// per 12 LDS.128 + 0.25 LDG.128.  (The 64 x 64 smem-tiled kernel below spends its time on shared-memory traffic when only 44
// of its 64 tile columns exist.)  Split over D across blockIdx.y; products are summed in fp32 inside a 32-deep chunk and the
// chunk sums in double -- cv::gemm accumulates float products in double -- then gemm_finalize_kernel adds the splits in a
// fixed order.  blockIdx.z walks column groups of 48 (2L = 136 for the 68-point model).
constexpr int PR_ROWS = 256, PR_KC = 32, PR_COLS = 48;

__global__ void __launch_bounds__(PR_ROWS, 1) predict_rows_kernel(const float* __restrict__ A, long long lda, int N, int D,
                                                                  const float* __restrict__ X, long long ldb, int M,
                                                                  double* __restrict__ partial, int k_per_split)
{
    __shared__ __align__(16) float Xs[PR_KC][PR_COLS];
    const int tid = threadIdx.x;
    const int row = blockIdx.x * PR_ROWS + tid;
    const int c0 = blockIdx.z * PR_COLS;
    const int kbeg = blockIdx.y * k_per_split;
    const int kend = min(D, kbeg + k_per_split);
    const bool live = row < N;
    const float* __restrict__ arow = A + (long long)(live ? row : 0) * lda;
    double dacc[PR_COLS];
#pragma unroll
    for (int c = 0; c < PR_COLS; ++c) dacc[c] = 0.0;
    for (int k0 = kbeg; k0 < kend; k0 += PR_KC) {
        // this thread's 32 feature values of the chunk (columns at or beyond kend may hold anything: masked to zero)
        float4 av[PR_KC / 4];
#pragma unroll
        for (int q = 0; q < PR_KC / 4; ++q) {
            const int k = k0 + 4 * q;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (live && k < kend) {
                v = __ldg(reinterpret_cast<const float4*>(arow + k));       // lda and kbeg are multiples of 4, the base is 16-byte aligned
                if (k + 1 >= kend) v.y = 0.f;
                if (k + 2 >= kend) v.z = 0.f;
                if (k + 3 >= kend) v.w = 0.f;
            }
            av[q] = v;
        }
        __syncthreads();                                                    // the previous chunk's weights are no longer read
        for (int i = tid; i < PR_KC * PR_COLS; i += PR_ROWS) {
            const int kk = i / PR_COLS, c = i - kk * PR_COLS;
            const int k = k0 + kk;
            Xs[kk][c] = (k < kend && c0 + c < M) ? __ldg(X + (long long)k * ldb + c0 + c) : 0.f;
        }
        __syncthreads();
        float acc[PR_COLS];
#pragma unroll
        for (int c = 0; c < PR_COLS; ++c) acc[c] = 0.f;
#pragma unroll
        for (int q = 0; q < PR_KC / 4; ++q) {
            const float a4[4] = {av[q].x, av[q].y, av[q].z, av[q].w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float a = a4[e];
#pragma unroll
                for (int c = 0; c < PR_COLS; c += 4) {
                    const float4 w = *reinterpret_cast<const float4*>(&Xs[4 * q + e][c]);
                    acc[c] = fmaf(a, w.x, acc[c]); acc[c + 1] = fmaf(a, w.y, acc[c + 1]);
                    acc[c + 2] = fmaf(a, w.z, acc[c + 2]); acc[c + 3] = fmaf(a, w.w, acc[c + 3]);
                }
            }
        }
#pragma unroll
        for (int c = 0; c < PR_COLS; ++c) dacc[c] += (double)acc[c];
    }
    if (live) {
        double* out = partial + ((long long)blockIdx.y * N + row) * M + c0;
#pragma unroll
        for (int c = 0; c < PR_COLS; ++c)
            if (c0 + c < M) out[c] = dacc[c];
    }
}

// sums the split partials in a fixed order (double) and applies the epilogue
__global__ void gemm_finalize_kernel(const double* __restrict__ partial, int splits, int N, int M,
                                     float* __restrict__ C, long long ldc, float alpha, float beta, const GemmEpilogue ep)
{
    const int i = blockIdx.x * blockDim.y + threadIdx.y;
    if (i >= N) return;
    float inv_n = 1.0f;
    if (ep.mode == 1 && ep.eyes.kind == 1) {
        const double ied = sd_device_ied(ep.x + (long long)i * M, M / 2, ep.eyes);
        inv_n = __fdiv_rn(1.0f, (float)__ddiv_rn(1.0, ied));
    }
    for (int j = threadIdx.x; j < M; j += blockDim.x) {
        double s = 0.0;
        for (int z = 0; z < splits; ++z) s += partial[((long long)z * N + i) * M + j];
        const float accf = (float)s;
        if (ep.mode == 1) {
            ep.x_next[(long long)i * M + j] = __fsub_rn(ep.x[(long long)i * M + j], __fmul_rn(accf, inv_n));
        } else {
            float* p = C + (long long)i * ldc + j;
            *p = (beta == 0.f) ? alpha * accf : fmaf(alpha, accf, beta * (*p));
        }
    }
}

int launch_gemm_nn(sd_ctx* ctx, const float* A, int64_t lda, int N, int D, const float* B, int64_t ldb, int M,
                   float* C, int64_t ldc, float alpha, float beta, const GemmEpilogue& ep)
{
    if (N <= 0 || M <= 0) return SD_OK;
    // the cascade's shape -- a long contraction, 2L output columns -- goes to the row-per-thread kernel for ANY number of rows: its
    // chunk boundaries are global multiples of 32, so a row's result does not depend on the batch it is computed in
    if (D >= 1024 && M <= 4 * PR_COLS && (lda % 4) == 0 && (reinterpret_cast<uintptr_t>(A) & 15) == 0) {
        const int row_blocks = sd_div_up(N, PR_ROWS), col_groups = sd_div_up(M, PR_COLS);
        int splits = (int)(2LL * ctx->sm_count / ((long long)row_blocks * col_groups));     // two CTAs' worth of work per SM, whole waves
        if (N < PR_ROWS) splits = splits * N / PR_ROWS + 1;                                 // few rows: few threads per CTA are live anyway
        const int maxs = sd_div_up(D, 4 * PR_KC);
        if (splits > maxs) splits = maxs;
        if (splits < 1) splits = 1;
        const int kps = sd_div_up(sd_div_up(D, splits), PR_KC) * PR_KC;
        splits = sd_div_up(D, kps);
        double* partial = (double*)sd_workspace(ctx, SD_WS_GEMM_PARTIAL, (size_t)splits * N * M * sizeof(double));
        if (!partial) return SD_ERR_CUDA;
        const dim3 pgrid(row_blocks, splits, col_groups);
        predict_rows_kernel<<<pgrid, PR_ROWS, 0, ctx->stream>>>(A, lda, N, D, B, ldb, M, partial, kps);
        SD_LAUNCH_CHECK(ctx, "predict_rows_kernel");
        dim3 fblock(32, 8);
        gemm_finalize_kernel<<<sd_div_up(N, 8), fblock, 0, ctx->stream>>>(partial, splits, N, M, C, ldc, alpha, beta, ep);
        SD_LAUNCH_CHECK(ctx, "gemm_finalize_kernel");
        return SD_OK;
    }
    dim3 grid(sd_div_up(M, GT), sd_div_up(N, GT), 1);
    SD_REQUIRE(ctx, grid.y <= 65535, "too many rows for one GEMM launch");
    // skinny outputs (M = 2L columns) leave most SMs idle: split the contraction dimension
    const long long tiles = (long long)grid.x * grid.y;
    int splits = 1;
    if (tiles < 3LL * ctx->sm_count && D >= 1024) {
        splits = (int)((4LL * ctx->sm_count + tiles - 1) / tiles);
        const int maxs = D / 512;
        if (splits > maxs) splits = maxs;
        if (splits > 32) splits = 32;
        if (splits < 1) splits = 1;
    }
    if (splits == 1) {
        gemm_nn_kernel<<<grid, 256, 0, ctx->stream>>>(A, lda, N, D, B, ldb, M, C, ldc, alpha, beta, ep, nullptr, D);
        SD_LAUNCH_CHECK(ctx, "gemm_nn_kernel");
        return SD_OK;
    }
    const int kps = sd_div_up(sd_div_up(D, splits), GK) * GK;
    grid.z = sd_div_up(D, kps);
    double* partial = (double*)sd_workspace(ctx, SD_WS_GEMM_PARTIAL, (size_t)grid.z * N * M * sizeof(double));
    if (!partial) return SD_ERR_CUDA;
    gemm_nn_kernel<<<grid, 256, 0, ctx->stream>>>(A, lda, N, D, B, ldb, M, C, ldc, alpha, beta, ep, partial, kps);
    SD_LAUNCH_CHECK(ctx, "gemm_nn_kernel(split)");
    dim3 fblock(32, 8);
    gemm_finalize_kernel<<<sd_div_up(N, 8), fblock, 0, ctx->stream>>>(partial, (int)grid.z, N, M, C, ldc, alpha, beta, ep);
    SD_LAUNCH_CHECK(ctx, "gemm_finalize_kernel");
    return SD_OK;
}

// =================================================================================================
// small element-wise kernels
// =================================================================================================
__global__ void pack_ext_kernel(const float* __restrict__ A, long long lda, const float* __restrict__ B, long long ldb,
                                int N, int D, int M, float* __restrict__ E, long long lde)
{
    const long long total = (long long)N * lde;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long n = idx / lde;
        const int c = (int)(idx - n * lde);
        float v = 0.f;
        if (c < D) v = A[n * lda + c];
        else if (c < D + M) v = B[n * ldb + (c - D)];
        E[idx] = v;
    }
}

__global__ void targets_kernel(const float* __restrict__ x, const float* __restrict__ x_gt, int N, int P,
                               const sd_eyes_dev eyes, float* __restrict__ B, long long ldb)
{
    const int i = blockIdx.x * blockDim.y + threadIdx.y;
    if (i >= N) return;
    float n = 1.0f;
    if (eyes.kind == 1) n = (float)__ddiv_rn(1.0, sd_device_ied(x + (long long)i * P, P / 2, eyes));
    for (int j = threadIdx.x; j < P; j += blockDim.x)
        B[(long long)i * ldb + j] = __fmul_rn(__fsub_rn(x[(long long)i * P + j], x_gt[(long long)i * P + j]), n);
}

__global__ void subtract_kernel(float* __restrict__ A, long long lda, const float* __restrict__ T, long long ldt, int N, int D)
{
    const long long total = (long long)N * D;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long n = idx / D;
        const int c = (int)(idx - n * D);
        A[n * lda + c] = __fsub_rn(A[n * lda + c], T[n * ldt + c]);
    }
}


// ---- centred features -----------------------------------------------------------------------------------------------------
// HOG features are non-negative with means of the size of their spread, so every entry of A^T A is dominated by N mu_i mu_j and
// the part that decides the weights -- the covariance -- sits several digits down: a Gram matrix that is accurate to 2e-7 still
// loses those digits when the bias column is eliminated (measured: weights 2.9e-4 from the float64 solve, the reference's own
// float32 arithmetic 2.0e-3).  Subtracting a per-column shift mu (the column mean) BEFORE the Gram removes the problem at the
// source.  It is the same least-squares problem:  A w + c 1 = (A - 1 mu^T) w + (c + mu.w) 1,  so the solve runs on the centred
// rows and the bias is shifted back at the end (bias = c' - mu.w); the MatrixNorm lambda still needs ||A^T A||_F of the
// UNcentred matrix, which follows from the centred Gram, its bias column s' and mu (frob_upper_kernel below).
// Column sums in double: blockIdx.y splits the rows, partials [splits][D] are folded in a fixed order.
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ A, long long lda, int N, int D, double* __restrict__ part)
{
    const int c = blockIdx.x * 32 + (threadIdx.x & 31);
    const int rl = threadIdx.x >> 5;                      // 8 row lanes
    const int rows_per = (N + gridDim.y - 1) / gridDim.y;
    const int r0 = blockIdx.y * rows_per, r1 = min(N, r0 + rows_per);
    double acc = 0.0, sq = 0.0;
    if (c < D)
        for (int r = r0 + rl; r < r1; r += 8) {
            const double v = (double)A[(long long)r * lda + c];
            acc += v;
            if (c == D - 1) sq += v * v;
        }
    __shared__ double red[8][33], red2[8][33];
    red[rl][threadIdx.x & 31] = acc;
    red2[rl][threadIdx.x & 31] = sq;
    __syncthreads();
    if (rl == 0 && c < D) {
        double s = 0.0, q = 0.0;
#pragma unroll
        for (int k = 0; k < 8; ++k) { s += red[k][threadIdx.x & 31]; q += red2[k][threadIdx.x & 31]; }
        part[(long long)blockIdx.y * (D + 1) + c] = s;
        if (c == D - 1) part[(long long)blockIdx.y * (D + 1) + D] = q;     // sum of squares of the last column
    }
}

__global__ void colsum_finish_kernel(double* __restrict__ part, int splits, int D)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c > D) return;
    double s = 0.0;
    for (int k = 0; k < splits; ++k) s += part[(long long)k * (D + 1) + c];
    part[c] = s;
}

// mu[c] = (float)(sum[c] / n) for the feature columns, 0 for the last (bias) column.  The shift is only a reformulation of the
// same problem when the last column is exactly all ones (sum == n and sum of squares == n) and carries no penalty; otherwise
// mu = 0 and the rows stay as they are.
__global__ void colmean_kernel(const double* __restrict__ sums, int D, int n_global, int enabled, float* __restrict__ mu)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const bool ones = enabled && sums[D - 1] == (double)n_global && sums[D] == (double)n_global;
    if (c < D) mu[c] = (ones && c < D - 1) ? (float)(sums[c] / (double)n_global) : 0.f;
}

__global__ void __launch_bounds__(256) centre_kernel(float* __restrict__ A, long long lda, int N, int D, const float* __restrict__ mu)
{
    const long long total = (long long)N * (D - 1);
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long r = idx / (D - 1);
        const int c = (int)(idx - r * (D - 1));
        A[r * lda + c] = __fsub_rn(A[r * lda + c], __ldg(mu + c));
    }
}

// ---- regulariser (regressors.hpp:126-148) ---------------------------------------------------------
// sum of squares of the full symmetric D x D matrix from its upper triangle, in double (cv::norm)
// Rows are dealt round-robin to the blocks (balanced triangle), a block's 1024 threads stride along the row with
// four independent loads in flight each; fixed grid and fixed order, so the sum is reproducible.
// own_block/nranks/rank: only the rows of this rank's block rows are summed (distributed solve; the partial sums are then
// all-reduced).
// Centred features (mu != NULL): G is the Gram of the rows shifted by mu (bias column unshifted, so G[:, D-1] = s' = A_c^T 1);
// the norm is taken of the uncentred matrix it stands for,  G[i][j] + s'_i mu_j + mu_i s'_j + n mu_i mu_j  (bias column:
// G[i][D-1] + n mu_i), entry by entry in double.  sv = s' (bias_extract_kernel), n = global sample count.
__global__ void __launch_bounds__(1024) frob_upper_centred_kernel(const float* __restrict__ G, long long ldg, int D, double* __restrict__ out,
                                                                  int own_block, int nranks, int rank, const float* __restrict__ mu,
                                                                  const double* __restrict__ sv, double n)
{
    double s0 = 0.0;
    for (int i = blockIdx.x; i < D; i += gridDim.x) {
        if (nranks > 1 && (i / own_block) % nranks != rank) continue;
        const float* row = G + (long long)i * ldg;
        const double mi = (double)mu[i], si = i < D - 1 ? sv[i] : 0.0;
        for (int j = i + threadIdx.x; j < D; j += 1024) {
            double v = (double)row[j];
            if (j == D - 1) v += (i == D - 1) ? 0.0 : n * mi;
            else v += si * (double)mu[j] + mi * sv[j] + n * mi * (double)mu[j];
            s0 += (j == i) ? 0.5 * v * v : v * v;                 // the diagonal counts once, everything is doubled below
        }
    }
    __shared__ double red[1024];
    red[threadIdx.x] = 2.0 * s0;
    __syncthreads();
    for (int o = 512; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[blockIdx.x] = red[0];
}

__global__ void __launch_bounds__(1024) frob_upper_kernel(const float* __restrict__ G, long long ldg, int D, double* __restrict__ out,
                                                          int own_block, int nranks, int rank)
{
    double s0 = 0.0, s1 = 0.0;
    for (int i = blockIdx.x; i < D; i += gridDim.x) {
        if (nranks > 1 && (i / own_block) % nranks != rank) continue;
        const float* row = G + (long long)i * ldg;
        if (threadIdx.x == 0) { const double v = (double)row[i]; s0 -= 0.5 * v * v; }  // the diagonal counts once, everything is doubled below
        int j = i + threadIdx.x;
        for (; j + 3 * 1024 < D; j += 4 * 1024) {
            const float a = row[j], b = row[j + 1024], c = row[j + 2048], d = row[j + 3072];
            s0 += (double)a * a; s1 += (double)b * b; s0 += (double)c * c; s1 += (double)d * d;
        }
        for (; j < D; j += 1024) { const float a = row[j]; s0 += (double)a * a; }
    }
    __shared__ double red[1024];
    red[threadIdx.x] = 2.0 * (s0 + s1);
    __syncthreads();
    for (int o = 512; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[blockIdx.x] = red[0];
}

// partial[0] <- sum of the partials (one double per rank travels through the all-reduce of the distributed solve)
__global__ void sum_partials_kernel(double* __restrict__ partial, int nparts)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double s = 0.0;
        for (int i = 0; i < nparts; ++i) s += partial[i];
        partial[0] = s;
    }
}

// scal[0] <- lambda ; then the diagonal gets lambda (0 for the bias row if !regularise_last_row)
__global__ void lambda_kernel(const double* __restrict__ partial, int nparts, int type, float param, int n_train, float* __restrict__ scal)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        float lambda = param;
        if (type == 1) {
            double s = 0.0;
            for (int i = 0; i < nparts; ++i) s += partial[i];
            // lambda * (float)cv::norm(AtA) / (float)num_training_elements  (regressors.hpp:135)
            lambda = __fdiv_rn(__fmul_rn(param, (float)sqrt(s)), (float)n_train);
        }
        scal[0] = lambda;
    }
}

__global__ void add_diag_kernel(float* __restrict__ G, long long ldg, int D, const float* __restrict__ scal, int regularise_last_row)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= D) return;
    const float lambda = (i == D - 1 && !regularise_last_row) ? 0.0f : scal[0];
    G[(long long)i * ldg + i] = __fadd_rn(G[(long long)i * ldg + i], lambda);
}


// ---- last column first --------------------------------------------------------------------------------------------------
// The last column of the RCR feature matrix is the bias (all ones, adaptive_vlhog.hpp:182-183) and by default gets no lambda
// (regressors.hpp:143-146).  Eliminated LAST -- where it sits -- its pivot is N - s^T (G_ww + lambda I)^-1 s: a difference of
// two nearly equal numbers that costs fp32 three digits (the system's condition number is ~7e4 on real HOG features; the
// reference's own float LU is 2e-3 off the float64 weights there, tests/test_gpu_train.py).  Eliminated FIRST its pivot is
// the exact integer N, and what remains, G_ww - s s^T / N + lambda I, is the Gram matrix of the CENTRED features: condition
// number ~4.  Same linear system, same solution, a better pivot order -- symmetric pivoting on the largest diagonal entry
// would pick that column first as well.
//   sv[0..D-2] = s (the bias column above the diagonal), sv[D-1] = pivot, sv[D..D+M) = the bias row of the right-hand sides
__global__ void bias_extract_kernel(const float* __restrict__ G, long long ldg, int D, int M, double* __restrict__ sv,
                                    int own_block, int nranks, int rank)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= D + M) return;
    const int row = i < D ? i : D - 1;
    const bool mine = nranks <= 1 || (row / own_block) % nranks == rank;       // others contribute zero to the all-reduce
    double v = 0.0;
    if (mine) v = (double)(i < D ? G[(long long)i * ldg + (D - 1)] : G[(long long)(D - 1) * ldg + i]);
    sv[i] = v;
}

// rows i < D-1 (owned ones): G[i][j] -= s_i * t_j / pivot for j in [i, D-1) (t = s) and j in [D, D+M) (t = bias row of the
// right-hand sides); column D-1 keeps s: it rides through the factorisation as one more right-hand side.
// part (shared CG route, where a rank only ever reads what its slab [k0, k1) of the product touches): 0 = everything,
// 1 = the slab's rows, the slab's columns above them and the right-hand sides, 2 = the rest (before a fall-back to the factorisation).
__global__ void __launch_bounds__(256) bias_downdate_kernel(float* __restrict__ G, long long ldg, int D, int M,
                                                            const double* __restrict__ sv, int own_block, int nranks, int rank,
                                                            int part, int k0, int k1)
{
    const double inv_p = 1.0 / sv[D - 1];
    for (int i = blockIdx.x; i < D - 1; i += gridDim.x) {
        if (nranks > 1 && (i / own_block) % nranks != rank) continue;
        const double f = sv[i] * inv_p;
        float* row = G + (long long)i * ldg;
        const bool slab_row = i >= k0 && i < k1;
        // up to three column ranges [a, b) of this row
        int ra[3], rb[3], nr = 0;
        if (part == 0 || (part == 1 && slab_row)) { ra[0] = i; rb[0] = D + M; nr = 1; }
        else if (part == 1) {
            if (i < k0) { ra[nr] = k0; rb[nr] = k1; ++nr; }
            ra[nr] = D; rb[nr] = D + M; ++nr;
        } else if (!slab_row) {                                           // part 2: what part 1 left out of [i, D)
            if (i < k0) { ra[nr] = i; rb[nr] = k0; ++nr; ra[nr] = k1; rb[nr] = D; ++nr; }
            else { ra[nr] = i; rb[nr] = D; ++nr; }
        }
        for (int q = 0; q < nr; ++q)
            for (int j = ra[q] + threadIdx.x; j < rb[q]; j += 256) {
                if (j == D - 1) continue;
                row[j] = (float)((double)row[j] - f * sv[j]);
            }
    }
}

// X[0..D-2] = w = columns [wcol0, wcol0 + M) of Xp (pitch ldw; after the factorisation column 0 is the solve of the carried bias
// column), X[D-1] = (rb - s^T w) / pivot
// Centred features: mu shifts the bias back (bias = c' - mu.w); Xc (optional) receives the weights that go with the CENTRED rows
// (same w, bias c'), which is what the cascade update multiplies the centred feature buffer with.
__global__ void __launch_bounds__(256) bias_finish_kernel(const float* __restrict__ Xp, int ldw, int wcol0, int D, int M,
                                                          const double* __restrict__ sv, float* __restrict__ X,
                                                          const float* __restrict__ mu, float* __restrict__ Xc)
{
    const int c = blockIdx.x;
    if (c < M) {
        double acc = 0.0, shift = 0.0;
        for (int i = threadIdx.x; i < D - 1; i += 256) {
            const double w = (double)Xp[(long long)i * ldw + wcol0 + c];
            acc += sv[i] * w;
            if (mu) shift += (double)mu[i] * w;
        }
        __shared__ double red[256], red2[256];
        red[threadIdx.x] = acc;
        red2[threadIdx.x] = shift;
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
            if ((int)threadIdx.x < o) { red[threadIdx.x] += red[threadIdx.x + o]; red2[threadIdx.x] += red2[threadIdx.x + o]; }
            __syncthreads();
        }
        if (threadIdx.x == 0) {
            const double cprime = (sv[D + c] - red[0]) / sv[D - 1];
            X[(long long)(D - 1) * M + c] = (float)(cprime - red2[0]);
            if (Xc) Xc[(long long)(D - 1) * M + c] = (float)cprime;
        }
    } else {
        const long long total = (long long)(D - 1) * M;
        for (long long idx = (long long)(blockIdx.x - M) * 256 + threadIdx.x; idx < total; idx += (long long)(gridDim.x - M) * 256) {
            const long long r = idx / M;
            const int cc = (int)(idx - r * M);
            const float w = Xp[r * ldw + wcol0 + cc];
            X[idx] = w;
            if (Xc) Xc[idx] = w;
        }
    }
}

// ---- LU with partial pivoting, single CTA (regressors.hpp:224-225 for small systems) ---------------
// G: D x W row-major (W = D + M: matrix and right-hand sides side by side).  On exit the RHS columns hold X.
__global__ void __launch_bounds__(1024) lu_small_kernel(float* __restrict__ G, long long ldg, int D, int M, int* __restrict__ status)
{
    __shared__ float s_val[32];
    __shared__ int s_idx[32];
    __shared__ int s_piv;
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int W = D + M;
    // mirror the upper triangle into the lower one (the SYRK only wrote tiles with j >= i)
    for (int idx = tid; idx < D * D; idx += nthr) {
        const int i = idx / D, j = idx - i * D;
        if (j < i) G[(long long)i * ldg + j] = G[(long long)j * ldg + i];
    }
    __syncthreads();
    for (int k = 0; k < D; ++k) {
        // pivot search: largest |G[i][k]|, first occurrence wins (ascending i), as the oracle
        float best = -1.f;
        int bi = k;
        for (int i = k + tid; i < D; i += nthr) {
            const float v = fabsf(G[(long long)i * ldg + k]);
            if (v > best) { best = v; bi = i; }
        }
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_down_sync(0xffffffffu, best, o);
            const int oi = __shfl_down_sync(0xffffffffu, bi, o);
            if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
        }
        if ((tid & 31) == 0) { s_val[tid >> 5] = best; s_idx[tid >> 5] = bi; }
        __syncthreads();
        if (tid < 32) {
            best = tid < (nthr >> 5) ? s_val[tid] : -1.f;
            bi = tid < (nthr >> 5) ? s_idx[tid] : 0x7fffffff;
            for (int o = 16; o > 0; o >>= 1) {
                const float ov = __shfl_down_sync(0xffffffffu, best, o);
                const int oi = __shfl_down_sync(0xffffffffu, bi, o);
                if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
            }
            if (tid == 0) {
                s_piv = bi;
                if (!(best > 0.f)) atomicOr(status, 4);    // singular: the reference would return inf/nan
            }
        }
        __syncthreads();
        const int piv = s_piv;
        if (piv != k) {
            for (int j = tid; j < W; j += nthr) {
                const float t = G[(long long)k * ldg + j];
                G[(long long)k * ldg + j] = G[(long long)piv * ldg + j];
                G[(long long)piv * ldg + j] = t;
            }
        }
        __syncthreads();
        const float pv = G[(long long)k * ldg + k];
        // multipliers
        for (int i = k + 1 + tid; i < D; i += nthr) G[(long long)i * ldg + k] = __fdiv_rn(G[(long long)i * ldg + k], pv);
        __syncthreads();
        // trailing update incl. right-hand sides (un-fused mul/sub: the oracle's x86 arithmetic)
        const int rows = D - k - 1, cols = W - k - 1;
        for (int idx = tid; idx < rows * cols; idx += nthr) {
            const int i = k + 1 + idx / cols, j = k + 1 + idx % cols;
            const float l = G[(long long)i * ldg + k];
            if (l != 0.f) G[(long long)i * ldg + j] = __fsub_rn(G[(long long)i * ldg + j], __fmul_rn(l, G[(long long)k * ldg + j]));
        }
        __syncthreads();
    }
    // back substitution, one thread per right-hand side column
    for (int c = tid; c < M; c += nthr) {
        for (int i = D - 1; i >= 0; --i) {
            float r = G[(long long)i * ldg + D + c];
            for (int k = i + 1; k < D; ++k) r = __fsub_rn(r, __fmul_rn(G[(long long)i * ldg + k], G[(long long)k * ldg + D + c]));
            G[(long long)i * ldg + D + c] = __fdiv_rn(r, G[(long long)i * ldg + i]);
        }
    }
}

__global__ void copy_block_kernel(const float* __restrict__ src, long long lds, int rows, int cols, float* __restrict__ dst, long long ldd)
{
    const long long total = (long long)rows * cols;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long r = idx / cols;
        const int c = (int)(idx - r * cols);
        dst[r * ldd + c] = src[r * lds + c];
    }
}

// ---- blocked Cholesky G = U^T U (upper), right-looking ---------------------------------------------
// One CTA factors a 128 x 128 diagonal block and inverts the factor.  Inner blocking by 32: the 32 x 32
// diagonal sub-block is factored AND inverted in the same 32 right-looking steps on [A | I] (potrf32_block), the
// row panel and the trailing update inside the block are small register-tiled GEMMs by all 8 warps.  Outputs:
// U (in place in G), W = U^-1 and W^T (workspace) -- so that the panel solve U12 = U11^-T G12 and the back
// substitution X_j = U_jj^-1 Y_j become plain GEMMs.  Blocks narrower than 128 are padded with the identity.
// Phase timings (clock64, -DSD_PROFILE_POTRF + tools/potrf_prof.py): 369k cycles before the restructuring
// (4 x 65k in the single-warp phases), ~120k now (load 5k, 4 x 14.6k potrf32, panels 8k, trailing 10k, W 28k, store 7k;
// the fused rank-128 update of the look-ahead path adds ~30k).
constexpr int PB = 128, PS = 32, PLD = PB + 1;
#ifdef SD_PROFILE_POTRF
__device__ long long sd_dbg_clk[64];
#define SD_CLK(i) do { __syncthreads(); if (threadIdx.x == 0) sd_dbg_clk[i] = clock64(); } while (0)
#else
#define SD_CLK(i) do {} while (0)
#endif

// cp.async staging: all of a CTA's global->shared copies are put in flight at once (the block kernels of the
// factorisation are latency-bound: measured 37 us per back-substitution step with plain load/store loops).
// valid == false zero-fills the destination (src-size 0; the source pointer is then only required to be mapped).
__device__ __forceinline__ void cp_async16(float* dst_smem, const float* src, bool valid)
{
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst_smem);
    const int n = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(src), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async4(float* dst_smem, const float* src, bool valid)
{
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst_smem);
    const int n = valid ? 4 : 0;
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(d), "l"(src), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all()
{
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}

// Factor and invert the 32 x 32 diagonal sub-block at (k0, k0) of sA.  History (clock64 per sub-block): single warp,
// right-looking + separate back substitution 65k cycles; single warp, left-looking with the inverse carried along 21k;
// whole CTA, right-looking on the augmented block (below) 14.6k.  A fully unrolled register/shuffle version was no
// faster than the first one: ~50 KB of straight-line code thrashes the instruction cache of a lone warp.
//
// Whole CTA, right-looking on the augmented block M = [A | I]
// (32 x 64, work copy in sM): per pivot k every thread reads the pivot row, rows k+1.. get their rank-1 update
// (4 rows x 64 columns per pass), the scaled pivot row goes straight to its destination (U -> sA, U^-T -> sT as T).
// One __syncthreads per pivot; ~190 cycles per pivot instead of ~660 for the single-warp left-looking version.
constexpr int MLD = 2 * PS + 1;
constexpr int ULD = PB + 4;          // row pitch of the panel rows staged for the fused update (float4-aligned)
__device__ __forceinline__ void potrf32_block(float* sA, float* sT, float* sM, int k0, int tid, bool& bad)
{
    const int c = tid & 63, g = tid >> 6;
    for (int idx = tid; idx < PS * 2 * PS; idx += 256) {
        const int r = idx >> 6, cc = idx & 63;
        sM[r * MLD + cc] = (cc < PS) ? sA[(k0 + r) * PLD + k0 + cc] : ((cc - PS == r) ? 1.f : 0.f);
    }
    __syncthreads();
    for (int k = 0; k < PS; ++k) {
        const float pk = sM[k * MLD + k];
        if (!(pk > 0.f)) bad = true;
        const float pks = pk > 0.f ? pk : 1.f;
        float rinv = rsqrtf(pks);
        rinv = rinv * fmaf(-0.5f * pks * rinv, rinv, 1.5f);        // one Newton step
        const float pr = sM[k * MLD + c];
        const float ps = pr * rinv;                                // scaled pivot row = row k of [U | U^-T]
        if (g == 0) {
            if (c < PS) { if (c >= k) sA[(k0 + k) * PLD + k0 + c] = (c == k) ? pks * rinv : ps; }
            else sT[(c - PS) * (PS + 1) + k] = (c - PS <= k) ? ps : 0.f;      // T[e][k] = U^-T[k][e]
        }
        // up to 8 rows per thread: all loads first, then the stores (a rolled loop serialises on possible aliasing)
        float f[8], o[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int i = k + 1 + g + 4 * u;
            const bool ok = i < PS;
            f[u] = ok ? sM[k * MLD + i] : 0.f;
            o[u] = ok ? sM[i * MLD + c] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int i = k + 1 + g + 4 * u;
            if (i < PS) sM[i * MLD + c] = fmaf(-(f[u] * rinv), ps, o[u]);      // f * rinv = U[k][i]
        }
        __syncthreads();
    }
}

// Optional fused update (look-ahead path): the block is first reduced by A^T A, A = nk x nb rows of the panel that
// was just solved (the part of the trailing update this diagonal block still misses).
__global__ void __launch_bounds__(256) potrf_inv_kernel(float* __restrict__ G, long long ldg, int nb,
                                                        float* __restrict__ W, float* __restrict__ Wt, int* __restrict__ status,
                                                        const float* __restrict__ A, long long lda, int nk)
{
    extern __shared__ float sm[];
    float* sA = sm;                    // PB x PLD : the block, becomes U
    float* sW = sm + PB * PLD;         // PB x PLD : U^-1
    float* sT = sW + PB * PLD;         // PS x (PS+1) scratch (inverse of the current diagonal sub-block / partial sums)
    float* sM = sT + PS * (PS + 1);    // PS x MLD work copy of [A | I] for potrf32_block
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    SD_CLK(0);
    // the block (upper triangle, identity padding outside nb) and, for the fused update, the panel rows A go to shared
    // memory as one batch of asynchronous copies; W's area doubles as the staging buffer for A
    for (int idx = tid; idx < PB * PB; idx += 256) {
        const int i = idx >> 7, j = idx & (PB - 1);
        const bool ok = i < nb && j < nb && j >= i;
        if (ok) cp_async4(sA + i * PLD + j, G + (long long)i * ldg + j, true);
        else sA[i * PLD + j] = (i == j && i >= nb) ? 1.f : 0.f;
        if (A) {
            const bool oka = i < nk && j < nb;                      // here i = panel row q, j = column of the block
            cp_async4(sW + i * ULD + j, oka ? A + (long long)i * lda + j : A, oka);   // 16-byte aligned rows (spills into sT/sM)
        } else {
            sW[i * PLD + j] = 0.f;
        }
    }
    cp_async_wait_all();
    if (A) {
        __syncthreads();
        const int tx = tid & 15, ty = tid >> 4;                   // rows ty*8 + m, columns tx*4 + n and 64 + tx*4 + n
        float acc[8][8];
#pragma unroll
        for (int m = 0; m < 8; ++m)
#pragma unroll
            for (int n = 0; n < 8; ++n) acc[m][n] = 0.f;
#pragma unroll 4
        for (int q = 0; q < PB; ++q) {
            const float4 r0 = *reinterpret_cast<const float4*>(sW + q * ULD + ty * 8);
            const float4 r1 = *reinterpret_cast<const float4*>(sW + q * ULD + ty * 8 + 4);
            const float4 c0 = *reinterpret_cast<const float4*>(sW + q * ULD + tx * 4);
            const float4 c1 = *reinterpret_cast<const float4*>(sW + q * ULD + 64 + tx * 4);
            const float ar[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
            const float ac[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
#pragma unroll
            for (int m = 0; m < 8; ++m)
#pragma unroll
                for (int n = 0; n < 8; ++n) acc[m][n] = fmaf(ar[m], ac[n], acc[m][n]);
        }
#pragma unroll
        for (int m = 0; m < 8; ++m)
#pragma unroll
            for (int n = 0; n < 8; ++n) {
                const int i = ty * 8 + m, j = (n < 4 ? 0 : 60) + tx * 4 + n;
                if (j >= i && j < nb) sA[i * PLD + j] -= acc[m][n];
            }
        __syncthreads();
        for (int idx = tid; idx < PB * PLD; idx += 256) sW[idx] = 0.f;
    }
    __syncthreads();
    SD_CLK(1);
    for (int kb = 0; kb < PB / PS; ++kb) {
        const int k0 = kb * PS;
        {
            bool bad = false;
            potrf32_block(sA, sT, sM, k0, tid, bad);
            if (bad && tid == 0) atomicOr(status, 8);                   // not positive definite
            for (int idx = tid; idx < PS * PS; idx += 256) {
                const int i = idx >> 5, jj = idx & 31;
                sW[(k0 + i) * PLD + k0 + jj] = sT[i * (PS + 1) + jj];
            }
        }
        __syncthreads();
        SD_CLK(2 + kb * 3);
        const int ncols = PB - k0 - PS;                                  // columns right of the diagonal sub-block
        if (ncols > 0) {
            // row panel: U12 = T^T * A12   (T = inverse of the diagonal sub-block)
            float out[3][4];
#pragma unroll
            for (int cc = 0; cc < 3; ++cc)
#pragma unroll
                for (int m = 0; m < 4; ++m) out[cc][m] = 0.f;
            const int ncc = ncols >> 5;
#pragma unroll 4
            for (int q = 0; q < PS; ++q) {                        // T[q][r] = 0 for q > r, so the full range is exact
                float t[4], av[3];
#pragma unroll
                for (int m = 0; m < 4; ++m) t[m] = sT[q * (PS + 1) + warp + 8 * m];
#pragma unroll
                for (int cc = 0; cc < 3; ++cc) av[cc] = (cc < ncc) ? sA[(k0 + q) * PLD + k0 + PS + cc * 32 + lane] : 0.f;
#pragma unroll
                for (int cc = 0; cc < 3; ++cc)
#pragma unroll
                    for (int m = 0; m < 4; ++m) out[cc][m] = fmaf(t[m], av[cc], out[cc][m]);
            }
            __syncthreads();
#pragma unroll
            for (int cc = 0; cc < 3; ++cc)
                if (cc * 32 < ncols) {
                    const int c = k0 + PS + cc * 32 + lane;
#pragma unroll
                    for (int m = 0; m < 4; ++m) sA[(k0 + warp + 8 * m) * PLD + c] = out[cc][m];
                }
            __syncthreads();
            SD_CLK(3 + kb * 3);
            // trailing update inside the block: A22 -= U12^T U12 (upper part)
            // work unit = 8 rows x 32 columns of one 32 x 32 tile (ti <= tj); 9 shared loads per 8 FMAs
            const int nt = ncols >> 5, npairs = nt * (nt + 1) / 2;
            for (int u = warp; u < npairs * 4; u += 8) {
                int p = u >> 2, ti = 0;
                while (p >= nt - ti) { p -= nt - ti; ++ti; }
                const int tj = ti + p;
                const int i0 = k0 + PS + ti * 32 + (u & 3) * 8, j = k0 + PS + tj * 32 + lane;
                float acc[8];
#pragma unroll
                for (int m = 0; m < 8; ++m) acc[m] = 0.f;
#pragma unroll 4
                for (int q = 0; q < PS; ++q) {
                    const float uj = sA[(k0 + q) * PLD + j];
#pragma unroll
                    for (int m = 0; m < 8; ++m) acc[m] = fmaf(sA[(k0 + q) * PLD + i0 + m], uj, acc[m]);
                }
#pragma unroll
                for (int m = 0; m < 8; ++m)
                    if (j >= i0 + m) sA[(i0 + m) * PLD + j] -= acc[m];
            }
            __syncthreads();
            SD_CLK(4 + kb * 3);
        }
    }
    SD_CLK(14);
    // off-diagonal blocks of W = U^-1:  W_ij = -T_i * sum_{k=i+1..j} U_ik W_kj   (block column by block column)
    for (int jb = 1; jb < PB / PS; ++jb) {
        for (int ib = jb - 1; ib >= 0; --ib) {
            float part[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
            for (int kq = (ib + 1) * PS; kq < (jb + 1) * PS; ++kq) {         // 5 shared loads per 4 FMAs
                const float w = sW[kq * PLD + jb * PS + lane];
#pragma unroll
                for (int m = 0; m < 4; ++m) part[m] = fmaf(sA[(ib * PS + warp + 8 * m) * PLD + kq], w, part[m]);
            }
#pragma unroll
            for (int m = 0; m < 4; ++m) sT[(warp + 8 * m) * (PS + 1) + lane] = part[m];
            __syncthreads();
#pragma unroll
            for (int m = 0; m < 4; ++m) {
                const int r = warp + 8 * m;
                float acc = 0.f;
#pragma unroll 8
                for (int q = r; q < PS; ++q) acc = fmaf(sW[(ib * PS + r) * PLD + ib * PS + q], sT[q * (PS + 1) + lane], acc);   // T_i is upper
                part[m] = -acc;
            }
            __syncthreads();
#pragma unroll
            for (int m = 0; m < 4; ++m) sW[(ib * PS + warp + 8 * m) * PLD + jb * PS + lane] = part[m];
            __syncthreads();
        }
    }
    SD_CLK(15);
    for (int idx = tid; idx < PB * PB; idx += 256) {
        const int i = idx >> 7, j = idx & (PB - 1);
        if (i < nb && j < nb && j >= i) G[(long long)i * ldg + j] = sA[i * PLD + j];
        W[idx] = sW[i * PLD + j];
        Wt[idx] = sW[j * PLD + i];
    }
    SD_CLK(16);
}
#ifdef SD_PROFILE_POTRF
extern "C" __attribute__((visibility("default"))) void sd_debug_read_clk(long long* out) { cudaMemcpyFromSymbol(out, sd_dbg_clk, sizeof(long long) * 64); }
#endif

// Block-row solve as a GEMM with the explicit inverse, in place:
//     B <- W^T (B - A^T P)            B: nb x cols block row of G,  W = U_jj^-1 (PB x PB, identity padded)
// The optional A^T P term (A = nk x nb, P = nk x cols) is the rank-nk update the block row still misses (second
// block row of a 256-row panel).  One CTA owns 64 columns over all rows, so the update is safe in place; thread
// tile 8 x 4 with 3 shared 128-bit loads per 32 FMAs.
constexpr int TA_COLS = 64;
struct TrsmArgs {
    float* B; long long ldb; int nb; int cols;
    const float* W;
    const float* A; long long lda; int nk;
    const float* P; long long ldp;
};

__global__ void __launch_bounds__(256) trsm_apply_kernel(const TrsmArgs a)
{
    extern __shared__ __align__(16) float sm_ta[];
    float* sW = sm_ta;                       // [PB][PB]      W[k][i]
    float* sT = sW + PB * PB;                // [PB][TA_COLS] B tile, then T = B - A^T P
    float* sA = sT + PB * TA_COLS;           // fused only: [PB][PB] A[q][k]
    float* sP = sA + PB * PB;                // fused only: [PB][TA_COLS]
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int c0 = blockIdx.x * TA_COLS;
    for (int idx = tid; idx < PB * PB / 4; idx += 256) cp_async16(sW + idx * 4, a.W + idx * 4, true);
    const bool full = c0 + TA_COLS <= a.cols;
    if (full && (a.ldb & 3) == 0 && ((reinterpret_cast<uintptr_t>(a.B) & 15) == 0)) {
        for (int idx = tid; idx < PB * TA_COLS / 4; idx += 256) {
            const int k = idx >> 4, c = (idx & 15) * 4;
            cp_async16(sT + idx * 4, a.B + (long long)(k < a.nb ? k : 0) * a.ldb + c0 + c, k < a.nb);
        }
    } else {
        for (int idx = tid; idx < PB * TA_COLS; idx += 256) {
            const int k = idx >> 6, c = idx & (TA_COLS - 1);
            const bool ok = k < a.nb && c0 + c < a.cols;
            cp_async4(sT + idx, ok ? a.B + (long long)k * a.ldb + c0 + c : a.B, ok);
        }
    }
    if (a.A) {
        if ((a.lda & 3) == 0 && ((reinterpret_cast<uintptr_t>(a.A) & 15) == 0) && (a.nb & 3) == 0) {
            for (int idx = tid; idx < PB * PB / 4; idx += 256) {
                const int q = idx >> 5, k = (idx & 31) * 4;
                const bool ok = q < a.nk && k < a.nb;
                cp_async16(sA + idx * 4, ok ? a.A + (long long)q * a.lda + k : a.A, ok);
            }
        } else {
            for (int idx = tid; idx < PB * PB; idx += 256) {
                const int q = idx >> 7, k = idx & (PB - 1);
                const bool ok = q < a.nk && k < a.nb;
                cp_async4(sA + idx, ok ? a.A + (long long)q * a.lda + k : a.A, ok);
            }
        }
        if (full && (a.ldp & 3) == 0 && ((reinterpret_cast<uintptr_t>(a.P) & 15) == 0)) {
            for (int idx = tid; idx < PB * TA_COLS / 4; idx += 256) {
                const int q = idx >> 4, c = (idx & 15) * 4;
                cp_async16(sP + idx * 4, a.P + (long long)(q < a.nk ? q : 0) * a.ldp + c0 + c, q < a.nk);
            }
        } else {
            for (int idx = tid; idx < PB * TA_COLS; idx += 256) {
                const int q = idx >> 6, c = idx & (TA_COLS - 1);
                const bool ok = q < a.nk && c0 + c < a.cols;
                cp_async4(sP + idx, ok ? a.P + (long long)q * a.ldp + c0 + c : a.P, ok);
            }
        }
    }
    cp_async_wait_all();
    __syncthreads();
    float acc[8][4];
    if (a.A) {
#pragma unroll
        for (int m = 0; m < 8; ++m) { acc[m][0] = acc[m][1] = acc[m][2] = acc[m][3] = 0.f; }
#pragma unroll 4
        for (int q = 0; q < PB; ++q) {
            const float4 a0 = *reinterpret_cast<const float4*>(sA + q * PB + ty * 8);
            const float4 a1 = *reinterpret_cast<const float4*>(sA + q * PB + ty * 8 + 4);
            const float4 pv = *reinterpret_cast<const float4*>(sP + q * TA_COLS + tx * 4);
            const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
            for (int m = 0; m < 8; ++m) {
                acc[m][0] = fmaf(av[m], pv.x, acc[m][0]); acc[m][1] = fmaf(av[m], pv.y, acc[m][1]);
                acc[m][2] = fmaf(av[m], pv.z, acc[m][2]); acc[m][3] = fmaf(av[m], pv.w, acc[m][3]);
            }
        }
#pragma unroll
        for (int m = 0; m < 8; ++m) {                               // every thread updates only its own entries of T
            float4* t = reinterpret_cast<float4*>(sT + (ty * 8 + m) * TA_COLS + tx * 4);
            float4 v = *t;
            v.x -= acc[m][0]; v.y -= acc[m][1]; v.z -= acc[m][2]; v.w -= acc[m][3];
            *t = v;
        }
        __syncthreads();
    }
#pragma unroll
    for (int m = 0; m < 8; ++m) { acc[m][0] = acc[m][1] = acc[m][2] = acc[m][3] = 0.f; }
#pragma unroll 4
    for (int k = 0; k < PB; ++k) {
        const float4 w0 = *reinterpret_cast<const float4*>(sW + k * PB + ty * 8);
        const float4 w1 = *reinterpret_cast<const float4*>(sW + k * PB + ty * 8 + 4);
        const float4 tv = *reinterpret_cast<const float4*>(sT + k * TA_COLS + tx * 4);
        const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
        for (int m = 0; m < 8; ++m) {
            acc[m][0] = fmaf(wv[m], tv.x, acc[m][0]); acc[m][1] = fmaf(wv[m], tv.y, acc[m][1]);
            acc[m][2] = fmaf(wv[m], tv.z, acc[m][2]); acc[m][3] = fmaf(wv[m], tv.w, acc[m][3]);
        }
    }
#pragma unroll
    for (int m = 0; m < 8; ++m) {
        const int i = ty * 8 + m;
        if (i >= a.nb) continue;
        float* row = a.B + (long long)i * a.ldb + c0 + tx * 4;
#pragma unroll
        for (int n = 0; n < 4; ++n)
            if (c0 + tx * 4 + n < a.cols) row[n] = acc[m][n];
    }
}

// One step of the back substitution U X = Y (right-looking over block columns, from the last):
//     X_j = U_jj^-1 Y_j            (every CTA, redundantly: 128 x 128 x 64 -- cheaper than a second dependent launch)
//     Y[rows of chunk r] -= U[chunk r, block j] X_j
// grid.x = 128-row chunks above block j (at least 1; CTA 0 also stores X_j), grid.y = 64-column tiles of the right-hand sides.
constexpr int BS_COLS = 64, BS_ULD = PB + 4;      // 16-byte aligned rows for cp.async
struct BackArgs {
    float* G; long long ldg; int D; int M; int j; int nb; int nchunks;
    int cg_first, cg_step;  // column groups of BS_COLS right-hand sides handled by this launch: cg_first + blockIdx.y * cg_step
    const float* Wt;        // (U_jj^-1)^T, PB x PB row-major, identity padded
    float* X;               // D x M
};

__global__ void __launch_bounds__(256) backsub_step_kernel(const BackArgs a)
{
    extern __shared__ __align__(16) float sm_bs[];
    float* sWt = sm_bs;                      // [PB][PB]        Wt[k][i] = W[i][k]
    float* sY = sWt + PB * PB;               // [PB][BS_COLS]   Y_j tile
    float* sX = sY + PB * BS_COLS;           // [PB][BS_COLS]   X_j tile
    float* sU = sX + PB * BS_COLS;           // [PB][BS_ULD]    U[chunk rows][block columns]
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int c0 = (a.cg_first + (int)blockIdx.y * a.cg_step) * BS_COLS;
    const int r0 = blockIdx.x * PB;
    const bool update = (int)blockIdx.x < a.nchunks;
    for (int idx = tid; idx < PB * PB / 4; idx += 256) cp_async16(sWt + idx * 4, a.Wt + idx * 4, true);
    for (int idx = tid; idx < PB * BS_COLS; idx += 256) {
        const int k = idx >> 6, c = idx & (BS_COLS - 1);
        const bool ok = k < a.nb && c0 + c < a.M;
        cp_async4(sY + idx, ok ? a.G + (long long)(a.j + k) * a.ldg + a.D + c0 + c : a.G, ok);
    }
    if (update) {
        const float* Ub = a.G + (long long)r0 * a.ldg + a.j;
        if ((a.ldg & 3) == 0 && (reinterpret_cast<uintptr_t>(Ub) & 15) == 0 && (a.nb & 3) == 0) {
            for (int idx = tid; idx < PB * PB / 4; idx += 256) {
                const int i = idx >> 5, k = (idx & 31) * 4;
                cp_async16(sU + i * BS_ULD + k, Ub + (long long)i * a.ldg + k, k < a.nb);
            }
        } else {
            for (int idx = tid; idx < PB * PB; idx += 256) {
                const int i = idx >> 7, k = idx & (PB - 1);
                cp_async4(sU + i * BS_ULD + k, Ub + (long long)i * a.ldg + k, k < a.nb);
            }
        }
    }
    cp_async_wait_all();
    __syncthreads();
    float acc[8][4];
#pragma unroll
    for (int m = 0; m < 8; ++m) { acc[m][0] = acc[m][1] = acc[m][2] = acc[m][3] = 0.f; }
#pragma unroll 4
    for (int k = 0; k < PB; ++k) {
        const float4 w0 = *reinterpret_cast<const float4*>(sWt + k * PB + ty * 8);
        const float4 w1 = *reinterpret_cast<const float4*>(sWt + k * PB + ty * 8 + 4);
        const float4 yv = *reinterpret_cast<const float4*>(sY + k * BS_COLS + tx * 4);
        const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
        for (int m = 0; m < 8; ++m) {
            acc[m][0] = fmaf(wv[m], yv.x, acc[m][0]); acc[m][1] = fmaf(wv[m], yv.y, acc[m][1]);
            acc[m][2] = fmaf(wv[m], yv.z, acc[m][2]); acc[m][3] = fmaf(wv[m], yv.w, acc[m][3]);
        }
    }
#pragma unroll
    for (int m = 0; m < 8; ++m) {
        const int i = ty * 8 + m;
        *reinterpret_cast<float4*>(sX + i * BS_COLS + tx * 4) = make_float4(acc[m][0], acc[m][1], acc[m][2], acc[m][3]);
        if (blockIdx.x == 0 && i < a.nb) {
#pragma unroll
            for (int n = 0; n < 4; ++n)
                if (c0 + tx * 4 + n < a.M) a.X[(long long)(a.j + i) * a.M + c0 + tx * 4 + n] = acc[m][n];
        }
    }
    if (!update) return;
    __syncthreads();
#pragma unroll
    for (int m = 0; m < 8; ++m) { acc[m][0] = acc[m][1] = acc[m][2] = acc[m][3] = 0.f; }
#pragma unroll 4
    for (int k = 0; k < PB; ++k) {
        const float4 xv = *reinterpret_cast<const float4*>(sX + k * BS_COLS + tx * 4);
#pragma unroll
        for (int m = 0; m < 8; ++m) {
            const float u = sU[(ty * 8 + m) * BS_ULD + k];
            acc[m][0] = fmaf(u, xv.x, acc[m][0]); acc[m][1] = fmaf(u, xv.y, acc[m][1]);
            acc[m][2] = fmaf(u, xv.z, acc[m][2]); acc[m][3] = fmaf(u, xv.w, acc[m][3]);
        }
    }
#pragma unroll
    for (int m = 0; m < 8; ++m) {
        float* row = a.G + (long long)(r0 + ty * 8 + m) * a.ldg + a.D + c0 + tx * 4;
#pragma unroll
        for (int n = 0; n < 4; ++n)
            if (c0 + tx * 4 + n < a.M) row[n] -= acc[m][n];
    }
}

int launch_trsm_apply(sd_ctx* ctx, cudaStream_t stream, float* B, int64_t ldb, int nb, int cols, const float* W,
                      const float* A, int64_t lda, int nk, const float* P, int64_t ldp)
{
    if (nb <= 0 || cols <= 0) return SD_OK;
    TrsmArgs a;
    a.B = B; a.ldb = ldb; a.nb = nb; a.cols = cols; a.W = W; a.A = A; a.lda = lda; a.nk = nk; a.P = P; a.ldp = ldp;
    const size_t smem = (size_t)(PB * PB + PB * TA_COLS) * sizeof(float) * (A ? 2 : 1);
    trsm_apply_kernel<<<sd_div_up(cols, TA_COLS), 256, smem, stream>>>(a);
    SD_LAUNCH_CHECK(ctx, "trsm_apply_kernel");
    return SD_OK;
}

bool sd_syrk_is_big(int K, int64_t MI, int64_t NJ)
{
    return MI * NJ >= 256 * 256 && K >= 64;
}

// comm (optional, more than one rank): DISTRIBUTED factorisation.  Block-row-cyclic ownership in units of one 256-row panel
// (rank = panel % nranks): on entry every rank holds the summed rows of its own panels (sd_reduce_scatter_gram), the other rows
// are undefined.  The owner factors its panel (chain + block-row solve), broadcasts the finished panel rows [P1;P2] (and the
// inverses of the two diagonal blocks) over NVLink, and every rank applies the rank-256 update to the block rows it owns.  The
// look-ahead is kept: the owner of panel p+1 updates that panel first and factors its diagonal blocks on the second stream while
// its share of the trailing update runs.  At the end every rank holds all of U and Y, so the (cheap) back substitution runs
// replicated and every rank ends up with the same X bit for bit.
int cholesky_solve(sd_ctx* ctx, float* G, int64_t ldg, int D, int M, float* X, sd_comm* comm = nullptr)
{
    const int nranks = sd_comm_size_of(comm), me = sd_comm_rank_of(comm);
    const bool dist = nranks > 1;
    int* status = reinterpret_cast<int*>(ctx->d_scratch);
    const int W_ = D + M;
    const int nblocks = sd_div_up(D, kCholNb);
    const size_t smem_potrf = (size_t)(2 * PB * PLD + PS * (PS + 1) + PS * MLD) * sizeof(float);
    SD_CUDA(ctx, cudaFuncSetAttribute(potrf_inv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_potrf));
    SD_CUDA(ctx, cudaFuncSetAttribute(trsm_apply_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)((PB * PB + PB * TA_COLS) * sizeof(float) * 2)));
    // per block: W = U_jj^-1 and its transpose (row-major 128 x 128 each)
    float* inv = (float*)sd_workspace(ctx, SD_WS_DIAGINV2, (size_t)nblocks * 2 * PB * PB * sizeof(float));
    if (!inv) return SD_ERR_CUDA;
    if (!ctx->chain_stream) {
        int prio_lo = 0, prio_hi = 0;
        SD_CUDA(ctx, cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        SD_CUDA(ctx, cudaStreamCreateWithPriority(&ctx->chain_stream, cudaStreamNonBlocking, prio_hi));
        for (int i = 0; i < 2; ++i) SD_CUDA(ctx, cudaEventCreateWithFlags(&ctx->chain_ev[i], cudaEventDisableTiming));
    }
    cudaStream_t main_s = ctx->stream, chain_s = ctx->chain_stream;
    cudaEvent_t ev_head = ctx->chain_ev[0], ev_chain = ctx->chain_ev[1];
    GemmEpilogue ep;
    memset(&ep, 0, sizeof(ep));
    // ---- factorisation G = U^T U in 256-row panels (two 128-blocks), carrying the right-hand sides along (Y = U^-T R) ----
    //   chain(p)  [one SM]  : A11 = U11^T U11 ; P1a = U11^-T A12 ; A22 - P1a^T P1a = U22^T U22           (diagonal blocks)
    //   bulk(p)             : P1 = U11^-T [rest of block row 1] ; P2 = U22^-T ([rest of block row 2] - P1a^T P1)
    //   head(p)             : rows of panel p+1      -= [P1;P2]^T [P1;P2]     (K = 256, tensor cores)
    //   tail(p)             : everything below them  -= [P1;P2]^T [P1;P2]
    // Look-ahead: chain(p+1) only needs head(p), so it runs on a second stream on the one SM that tail(p) leaves free;
    // the 134 dependent single-CTA factorisations are hidden behind the trailing updates while those are long enough.
    // Every element still receives its updates in panel order (events), so the result does not depend on timing.
    auto panel_dims = [&](int b, int& j, int& nb1, int& nb2) {
        j = b * kCholNb;
        nb1 = (D - j < kCholNb) ? D - j : kCholNb;
        nb2 = (b + 1 < nblocks) ? ((D - j - nb1 < kCholNb) ? D - j - nb1 : kCholNb) : 0;
    };
    auto launch_chain = [&](int b) -> int {
        int j, nb1, nb2;
        panel_dims(b, j, nb1, nb2);
        float* G11 = G + (int64_t)j * ldg + j;
        float* W1 = inv + (size_t)b * 2 * PB * PB;
        potrf_inv_kernel<<<1, 256, smem_potrf, chain_s>>>(G11, ldg, nb1, W1, W1 + PB * PB, status, nullptr, 0, 0);
        SD_LAUNCH_CHECK(ctx, "potrf_inv_kernel");
        if (nb2 > 0) {
            int rc = launch_trsm_apply(ctx, chain_s, G11 + nb1, ldg, nb1, nb2, W1, nullptr, 0, 0, nullptr, 0);   // P1a
            if (rc) return rc;
            float* G22 = G + (int64_t)(j + nb1) * ldg + (j + nb1);
            float* W2 = inv + (size_t)(b + 1) * 2 * PB * PB;
            potrf_inv_kernel<<<1, 256, smem_potrf, chain_s>>>(G22, ldg, nb2, W2, W2 + PB * PB, status, G11 + nb1, ldg, nb1);
            SD_LAUNCH_CHECK(ctx, "potrf_inv_kernel");
        }
        return SD_OK;
    };
    int rc = SD_OK;
    SD_CUDA(ctx, cudaEventRecord(ev_head, main_s));                   // G is ready (regulariser applied) for chain(0)
    if (me == 0) {
        SD_CUDA(ctx, cudaStreamWaitEvent(chain_s, ev_head, 0));
        rc = launch_chain(0);
        if (rc) return rc;
        SD_CUDA(ctx, cudaEventRecord(ev_chain, chain_s));
    }
    for (int b = 0; b < nblocks; b += 2) {
        int j, nb1, nb2;
        panel_dims(b, j, nb1, nb2);
        const int owner = dist ? (b / 2) % nranks : me;
        const int next_owner = dist ? (b / 2 + 1) % nranks : me;
        const int j3 = j + nb1 + nb2;                                 // first column right of the panel
        const int cols3 = W_ - j3;
        float* W1 = inv + (size_t)b * 2 * PB * PB;
        float* row1 = G + (int64_t)j * ldg + j3;
        if (me == owner) {
            SD_CUDA(ctx, cudaStreamWaitEvent(main_s, ev_chain, 0));   // chain(p) done
            if (cols3 > 0) {
                rc = launch_trsm_apply(ctx, main_s, row1, ldg, nb1, cols3, W1, nullptr, 0, 0, nullptr, 0);             // P1
                if (rc) return rc;
                if (nb2 > 0) {
                    float* W2 = inv + (size_t)(b + 1) * 2 * PB * PB;
                    float* row2 = G + (int64_t)(j + nb1) * ldg + j3;
                    const float* P1a = G + (int64_t)j * ldg + (j + nb1);
                    rc = launch_trsm_apply(ctx, main_s, row2, ldg, nb2, cols3, W2, P1a, ldg, nb1, row1, ldg);           // P2
                    if (rc) return rc;
                }
            }
        }
        if (dist) {
            // the finished panel rows, from the diagonal column of the first row to the end of the last row (one contiguous
            // range of G), and U_jj^-1 / U_jj^-T of its diagonal blocks for the back substitution
            rc = sd_comm_group_start(ctx);
            if (rc) return rc;
            rc = sd_comm_bcast(ctx, comm, G + (int64_t)j * ldg + j, (size_t)(nb1 + nb2) * ldg - j, owner, main_s);
            if (!rc) rc = sd_comm_bcast(ctx, comm, W1, (size_t)(nb2 > 0 ? 2 : 1) * 2 * PB * PB, owner, main_s);
            const int rc2 = sd_comm_group_end(ctx);
            if (rc || rc2) return rc ? rc : rc2;
        }
        if (cols3 <= 0) continue;
        const int rest = D - j3;                                      // rows (= diagonal columns) below the panel
        if (rest <= 0) continue;
        const int kp = nb1 + nb2;                                     // rows of [P1;P2], contiguous in G
        const int head = rest < 2 * kCholNb ? rest : 2 * kCholNb;
        float* C3 = G + (int64_t)j3 * ldg + j3;
        // one kernel family per rank-kp update, chosen from the size of the whole trailing matrix; the updates use the
        // unbiased hi/lo split: a truncated hi leaves a one-signed lo*lo term behind, which is harmless in the Gram (it
        // scales [AtA|Atb] almost uniformly) but is amplified by the cancellation inside Schur complements
        const int path = sd_syrk_is_big(kp, rest, cols3) ? 1 : 2;
        if (me == next_owner) {
            rc = sd_syrk_update(ctx, row1, ldg, kp, head, cols3, C3, ldg, -1.0f, 1.0f, path, true);
            if (rc) return rc;
            SD_CUDA(ctx, cudaEventRecord(ev_head, main_s));
            SD_CUDA(ctx, cudaStreamWaitEvent(chain_s, ev_head, 0));
            rc = launch_chain(b + 2);
            if (rc) return rc;
            SD_CUDA(ctx, cudaEventRecord(ev_chain, chain_s));
        }
        if (rest > head) {
            sd_row_filter own;
            own.block = 2 * kCholNb; own.nranks = nranks; own.rank = me; own.first_row = j3 + head;
            ctx->syrk_sm_reserve = (me == next_owner) ? 1 : 0;   // leave one SM to the chain running beside it
            rc = sd_syrk_update(ctx, row1 + head, ldg, kp, rest - head, cols3 - head, C3 + (int64_t)head * ldg + head, ldg, -1.0f, 1.0f, path,
                                true, dist ? &own : nullptr);
            ctx->syrk_sm_reserve = 0;
            if (rc) return rc;
        }
    }
    SD_CUDA(ctx, cudaStreamWaitEvent(main_s, ev_chain, 0));
    SD_CUDA(ctx, cudaEventRecord(ctx->ev[3], ctx->stream));   // end of "Decomposition"
    // ---- back substitution U X = Y, right-looking over block columns from the last: one launch per block ----
    const size_t smem_bs = (size_t)(PB * PB + 2 * PB * BS_COLS + PB * BS_ULD) * sizeof(float);
    SD_CUDA(ctx, cudaFuncSetAttribute(backsub_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bs));
    // distributed: the column groups of the right-hand sides are independent, so rank r substitutes groups r, r + G, ... and one
    // all-reduce of X (every entry has exactly one non-zero contributor) hands everybody the whole solution
    const int ngroups = sd_div_up(M, BS_COLS);
    const int my_groups = dist ? (ngroups > me ? (ngroups - me + nranks - 1) / nranks : 0) : ngroups;
    if (dist) SD_CUDA(ctx, cudaMemsetAsync(X, 0, (size_t)D * M * sizeof(float), main_s));
    for (int b = nblocks - 1; b >= 0 && my_groups > 0; --b) {
        BackArgs ba;
        ba.G = G; ba.ldg = ldg; ba.D = D; ba.M = M; ba.j = b * kCholNb;
        ba.nb = (D - ba.j < kCholNb) ? D - ba.j : kCholNb;
        ba.nchunks = b;                                              // full 128-row chunks above block b
        ba.cg_first = dist ? me : 0;
        ba.cg_step = dist ? nranks : 1;
        ba.Wt = inv + (size_t)b * 2 * PB * PB + PB * PB;
        ba.X = X;
        const dim3 grid(b > 0 ? b : 1, my_groups);
        backsub_step_kernel<<<grid, 256, smem_bs, main_s>>>(ba);
        SD_LAUNCH_CHECK(ctx, "backsub_step_kernel");
    }
    if (dist) {
        rc = sd_comm_allreduce_f32(ctx, comm, X, (size_t)D * M, main_s);
        if (rc) return rc;
    }
    return SD_OK;
}

int check_status(sd_ctx* ctx, const char* what)
{
    int* h = reinterpret_cast<int*>(ctx->h_scratch);
    SD_CUDA(ctx, cudaMemcpyAsync(h, ctx->d_scratch, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    SD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const int st = h[0];
    if (st) {
        SD_CUDA(ctx, cudaMemsetAsync(ctx->d_scratch, 0, sizeof(int), ctx->stream));
        if (st & 8) return sd_fail(ctx, SD_ERR_NUMERIC, "%s: regularised AtA is not positive definite (increase lambda)", what);
        if (st & 4) return sd_fail(ctx, SD_ERR_NUMERIC, "%s: singular system (zero pivot)", what);
    }
    return SD_OK;
}

}  // namespace

// =================================================================================================
// internal dispatch
// =================================================================================================
int sd_syrk_simt(sd_ctx* ctx, const float* d_S, int64_t lds, int K, int MI, int NJ, float* d_C, int64_t ldc,
                 float alpha, float beta)
{
    if (MI <= 0 || NJ <= 0) return SD_OK;
    dim3 grid(sd_div_up(NJ, ST), sd_div_up(MI, ST), 1);
    SD_REQUIRE(ctx, grid.y <= 65535, "matrix too large for the SIMT SYRK");
    const long long tiles = (long long)grid.x * grid.y;
    int splits = 1;
    if (tiles < 2LL * ctx->sm_count && K > 2048) {
        splits = (int)((4LL * ctx->sm_count + tiles - 1) / tiles);
        const int maxs = sd_div_up(K, 512);
        if (splits > maxs) splits = maxs;
        if (splits > 64) splits = 64;
        if (splits < 1) splits = 1;
    }
    if (splits == 1) {
        syrk_simt_kernel<<<grid, 256, 0, ctx->stream>>>(d_S, lds, K, MI, NJ, d_C, ldc, alpha, beta, nullptr, K);
        SD_LAUNCH_CHECK(ctx, "syrk_simt_kernel");
    } else {
        float* partial = (float*)sd_workspace(ctx, SD_WS_PARTIAL, (size_t)splits * MI * NJ * sizeof(float));
        if (!partial) return SD_ERR_CUDA;
        const int kps = sd_div_up(sd_div_up(K, splits), SK) * SK;
        grid.z = sd_div_up(K, kps);
        syrk_simt_kernel<<<grid, 256, 0, ctx->stream>>>(d_S, lds, K, MI, NJ, d_C, ldc, alpha, beta, partial, kps);
        SD_LAUNCH_CHECK(ctx, "syrk_simt_kernel(split)");
        const int blocks = sd_div_up((int64_t)MI * NJ, 256) > 2048 ? 2048 : sd_div_up((int64_t)MI * NJ, 256);
        syrk_reduce_kernel<<<blocks, 256, 0, ctx->stream>>>(partial, (int)grid.z, MI, NJ, d_C, ldc, alpha, beta);
        SD_LAUNCH_CHECK(ctx, "syrk_reduce_kernel");
    }
    return SD_OK;
}

int sd_syrk_update(sd_ctx* ctx, const float* d_S, int64_t lds, int K, int MI, int NJ, float* d_C, int64_t ldc,
                   float alpha, float beta, int path, bool unbiased_split, const sd_row_filter* rows)
{
    const bool want_tc = path == 1 || (path == 0 && sd_syrk_is_big(K, MI, NJ));
    if (ctx->gram_mode != 2 && path != 2 && want_tc && sd_syrk_tc_supported(d_S, lds, K, MI, NJ, d_C, ldc))
        return sd_syrk_tc(ctx, d_S, lds, K, MI, NJ, d_C, ldc, alpha, beta, ctx->gram_mode == 1 ? 1 : 3, unbiased_split, rows);
    // the SIMT kernel updates every row: rows of other ranks are never read before their owner's broadcast overwrites them
    return sd_syrk_simt(ctx, d_S, lds, K, MI, NJ, d_C, ldc, alpha, beta);
}

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

int sd_gram(sd_ctx* ctx, const float* d_A, int64_t lda, const float* d_B, int64_t ldb, int N, int D, int M,
            float* d_G, int64_t ldg)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_REQUIRE(ctx, d_A && d_G && N >= 1 && D >= 1 && M >= 0, "bad argument");
    SD_REQUIRE(ctx, lda >= D && ldg >= D + M && (M == 0 || (d_B && ldb >= M)), "bad leading dimension");
    const float* S = d_A;
    int64_t lds = lda;
    if (M > 0 && !(d_B == d_A + D && ldb == lda)) {
        // A and B live apart: pack [A | B] (zero padded to a multiple of 4 columns) into the workspace
        lds = ((int64_t)(D + M) + 3) / 4 * 4;
        float* E = (float*)sd_workspace(ctx, SD_WS_GRAM_EXT, (size_t)N * lds * sizeof(float));
        if (!E) return SD_ERR_CUDA;
        const int blocks = sd_div_up((int64_t)N * lds, 256) > 4096 ? 4096 : sd_div_up((int64_t)N * lds, 256);
        pack_ext_kernel<<<blocks, 256, 0, ctx->stream>>>(d_A, lda, d_B, ldb, N, D, M, E, lds);
        SD_LAUNCH_CHECK(ctx, "pack_ext_kernel");
        S = E;
    }
    return sd_syrk_update(ctx, S, lds, N, D, D + M, d_G, ldg, 1.0f, 0.0f);
}

// route: 0 = every rank holds the summed G (one GPU, or after sd_allreduce_gram) and solves it alone;
//        1 = G is reduce-scattered over comm: distributed blocked Cholesky;
//        2 = every rank holds the summed G and the ranks share the CG iterations (contraction sharded, one small all-reduce each)
static int solve_gram_impl(sd_ctx* ctx, sd_comm* comm, float* d_G, int64_t ldg, int D, int M, const sd_regulariser* reg,
                           int n_train_global, float* d_X, float* lambda_out, int* rank_out = nullptr, int route = 0,
                           const float* d_mu = nullptr, float* d_Xc = nullptr)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_REQUIRE(ctx, d_G && d_X && reg && D >= 1 && M >= 1 && ldg >= D + M, "bad argument");
    SD_REQUIRE(ctx, reg->type == 0 || reg->type == 1, "unknown regularisation type");
    SD_REQUIRE(ctx, n_train_global >= 1, "n_train_global must be >= 1");
    // the distributed factorisation needs whole panels per rank; small systems were all-reduced and are solved replicated
    const int nranks = sd_comm_size_of(comm);
    const bool dist = route == 1 && nranks > 1 && sd_gram_is_scattered(D, ldg, d_G);
    float* scal = reinterpret_cast<float*>(ctx->d_scratch) + 16;
    double* partial = reinterpret_cast<double*>(reinterpret_cast<char*>(ctx->d_scratch) + 1024);   // up to 384 doubles
    // errors belong to the call that caused them: HOG status bits raised earlier were reported by their own entry points
    SD_CUDA(ctx, cudaMemsetAsync(ctx->d_scratch, 0, sizeof(int), ctx->stream));
    SD_CUDA(ctx, cudaEventRecord(ctx->ev[1], ctx->stream));
    int nparts = 0;
    // the norm is a sum over rows: the ranks of the distributed routes take the row blocks they own (in route 2 every rank holds the
    // whole matrix, but reading an eighth of it and all-reducing one double is cheaper than reading all of it)
    const bool share_norm = dist || (route == 2 && nranks > 1 && D > kLuMaxDim);
    SD_REQUIRE(ctx, !d_mu || D > kLuMaxDim, "centred features are for the factorisation route (D > 256)");
    if (reg->type == 1) {
        nparts = D < 296 ? D : 296;                                   // 2 x 148 SMs; at most 384 partials fit the scratch
        if (d_mu) {
            // s' = bias column of the centred Gram, needed entry by entry for the norm of the uncentred matrix
            double* sv0 = (double*)sd_workspace(ctx, SD_WS_BIAS, (size_t)(D + M) * sizeof(double) + (size_t)(D - 1) * (M + 1) * sizeof(float));
            if (!sv0) return SD_ERR_CUDA;
            bias_extract_kernel<<<sd_div_up(D + M, 256), 256, 0, ctx->stream>>>(d_G, ldg, D, M, sv0, 2 * kCholNb, dist ? nranks : 1, sd_comm_rank_of(comm));
            SD_LAUNCH_CHECK(ctx, "bias_extract_kernel");
            if (dist) {
                int rc0 = sd_comm_allreduce_f64(ctx, comm, sv0, (size_t)(D + M), ctx->stream);
                if (rc0) return rc0;
            }
            frob_upper_centred_kernel<<<nparts, 1024, 0, ctx->stream>>>(d_G, ldg, D, partial, 2 * kCholNb, share_norm ? nranks : 1, sd_comm_rank_of(comm),
                                                                        d_mu, sv0, (double)n_train_global);
            SD_LAUNCH_CHECK(ctx, "frob_upper_centred_kernel");
        } else {
            frob_upper_kernel<<<nparts, 1024, 0, ctx->stream>>>(d_G, ldg, D, partial, 2 * kCholNb, share_norm ? nranks : 1, sd_comm_rank_of(comm));
            SD_LAUNCH_CHECK(ctx, "frob_upper_kernel");
        }
        if (share_norm) {
            sum_partials_kernel<<<1, 32, 0, ctx->stream>>>(partial, nparts);
            SD_LAUNCH_CHECK(ctx, "sum_partials_kernel");
            int rc = sd_comm_allreduce_f64(ctx, comm, partial, 1, ctx->stream);
            if (rc) return rc;
            nparts = 1;
        }
    }
    lambda_kernel<<<1, 32, 0, ctx->stream>>>(partial, nparts, reg->type, reg->param, n_train_global, scal);
    SD_LAUNCH_CHECK(ctx, "lambda_kernel");
    add_diag_kernel<<<sd_div_up(D, 256), 256, 0, ctx->stream>>>(d_G, ldg, D, scal, reg->regularise_last_row);
    SD_LAUNCH_CHECK(ctx, "add_diag_kernel");
    SD_CUDA(ctx, cudaEventRecord(ctx->ev[2], ctx->stream));
    int rc = SD_OK;
    int rank = -1;
    if (rank_out) {                                                   // ColPivHouseholderQRSolver's diagnostic (regressors.hpp:288-293)
        rc = sd_gram_rank(ctx, d_G, ldg, D, &rank, nullptr, nullptr);
        if (rc) return rc;
        *rank_out = rank;
    }
    if (D <= kLuMaxDim) {
        lu_small_kernel<<<1, 1024, 0, ctx->stream>>>(d_G, ldg, D, M, reinterpret_cast<int*>(ctx->d_scratch));
        SD_LAUNCH_CHECK(ctx, "lu_small_kernel");
        SD_CUDA(ctx, cudaEventRecord(ctx->ev[3], ctx->stream));
        const int blocks = sd_div_up((int64_t)D * M, 256);
        copy_block_kernel<<<blocks, 256, 0, ctx->stream>>>(d_G + D, ldg, D, M, d_X, M);
        SD_LAUNCH_CHECK(ctx, "copy_block_kernel");
    } else {
        // last column first (see bias_extract_kernel), then the blocked Cholesky of the remaining (D-1) x (D-1) system with the
        // bias column riding along as right-hand side 0
        const int me = sd_comm_rank_of(comm), nr = dist ? nranks : 1;
        double* sv = (double*)sd_workspace(ctx, SD_WS_BIAS, (size_t)(D + M) * sizeof(double) + (size_t)(D - 1) * (M + 1) * sizeof(float));
        if (!sv) return SD_ERR_CUDA;
        float* Xp = reinterpret_cast<float*>(sv + D + M);
        bias_extract_kernel<<<sd_div_up(D + M, 256), 256, 0, ctx->stream>>>(d_G, ldg, D, M, sv, 2 * kCholNb, nr, me);
        SD_LAUNCH_CHECK(ctx, "bias_extract_kernel");
        if (dist) {
            rc = sd_comm_allreduce_f64(ctx, comm, sv, (size_t)(D + M), ctx->stream);
            if (rc) return rc;
        }
        const bool try_cg = !dist && (ctx->solver_mode == 1 || route == 2) && M <= 192;
        // shared CG: this rank reads only its slab's rows and columns of the matrix; the rest is downdated if the factorisation
        // has to take over
        int k0 = 0, k1 = D - 1;
        const bool partial_downdate = try_cg && route == 2 && nranks > 1;
        if (partial_downdate) sd_cg_slab(D - 1, nranks, me, &k0, &k1);
        bias_downdate_kernel<<<4 * ctx->sm_count, 256, 0, ctx->stream>>>(d_G, ldg, D, M, sv, 2 * kCholNb, nr, me, partial_downdate ? 1 : 0, k0, k1);
        SD_LAUNCH_CHECK(ctx, "bias_downdate_kernel");
        bool solved = false;
        ctx->cg_iterations = 0;
        if (try_cg) {
            // conjugate gradients on the (well conditioned) centred system; falls back to the factorisation when it stalls
            float* W = nullptr;
            int ldw = 0, its = 0;
            rc = sd_cg_solve(ctx, route == 2 ? comm : nullptr, d_G, ldg, D - 1, D, M, &W, &ldw, &its);
            ctx->cg_iterations = its;
            if (rc == SD_OK) {
                SD_CUDA(ctx, cudaEventRecord(ctx->ev[3], ctx->stream));
                bias_finish_kernel<<<M + 2 * ctx->sm_count, 256, 0, ctx->stream>>>(W, ldw, 0, D, M, sv, d_X, d_mu, d_Xc);
                SD_LAUNCH_CHECK(ctx, "bias_finish_kernel");
                solved = true;
            } else if (rc != SD_ERR_NUMERIC) {
                return rc;
            }
        }
        if (!solved) {
            if (partial_downdate) {
                bias_downdate_kernel<<<4 * ctx->sm_count, 256, 0, ctx->stream>>>(d_G, ldg, D, M, sv, 2 * kCholNb, nr, me, 2, k0, k1);
                SD_LAUNCH_CHECK(ctx, "bias_downdate_kernel");
            }
            rc = cholesky_solve(ctx, d_G, ldg, D - 1, M + 1, Xp, dist ? comm : nullptr);
            if (rc) return rc;
            bias_finish_kernel<<<M + 2 * ctx->sm_count, 256, 0, ctx->stream>>>(Xp, M + 1, 1, D, M, sv, d_X, d_mu, d_Xc);
            SD_LAUNCH_CHECK(ctx, "bias_finish_kernel");
        }
    }
    SD_CUDA(ctx, cudaEventRecord(ctx->ev[4], ctx->stream));
    if (lambda_out) {
        float* h = reinterpret_cast<float*>(ctx->h_scratch) + 16;
        SD_CUDA(ctx, cudaMemcpyAsync(h, scal, sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
        SD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        *lambda_out = *h;
    }
    rc = check_status(ctx, "solve");
    if (rc && rank >= 0 && rank < D)
        return sd_fail(ctx, rc, "The regularised AtA is not invertible. (The rank is %d, full rank would be %d). Increase lambda.", rank, D);
    return rc;
}

int sd_solve_gram(sd_ctx* ctx, float* d_G, int64_t ldg, int D, int M, const sd_regulariser* reg, int n_train_global,
                  float* d_X, float* lambda_out)
{
    return solve_gram_impl(ctx, nullptr, d_G, ldg, D, M, reg, n_train_global, d_X, lambda_out);
}

int sd_solve_gram_dist(sd_ctx* ctx, sd_comm* comm, float* d_G, int64_t ldg, int D, int M, const sd_regulariser* reg,
                       int n_train_global, float* d_X, float* lambda_out)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_REQUIRE(ctx, comm != nullptr, "no communicator");
    return solve_gram_impl(ctx, comm, d_G, ldg, D, M, reg, n_train_global, d_X, lambda_out, nullptr, 1);
}

int sd_learn_dist(sd_ctx* ctx, sd_comm* comm, const float* d_A, int64_t lda, const float* d_B, int64_t ldb, int N_local, int D, int M,
                  const sd_regulariser* reg, int n_train_global, int distributed_solve, float* d_X, float* lambda_out)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_REQUIRE(ctx, comm != nullptr && M >= 1 && N_local >= 0, "bad argument");
    const int64_t ldg = ((int64_t)(D + M) + 3) / 4 * 4;
    float* G = (float*)sd_workspace(ctx, SD_WS_SCRATCH, (size_t)D * ldg * sizeof(float));
    if (!G) return SD_ERR_CUDA;
    SD_CUDA(ctx, cudaEventRecord(ctx->ev[0], ctx->stream));
    int rc;
    if (N_local > 0) rc = sd_gram(ctx, d_A, lda, d_B, ldb, N_local, D, M, G, ldg);
    else rc = sd_check_cuda(ctx, cudaMemsetAsync(G, 0, (size_t)D * ldg * sizeof(float), ctx->stream), "memset(G)");
    if (rc) return rc;
    if (distributed_solve == 1) {
        rc = sd_reduce_scatter_gram(ctx, comm, G, ldg, D, M);
        if (rc) return rc;
        return sd_solve_gram_dist(ctx, comm, G, ldg, D, M, reg, n_train_global, d_X, lambda_out);
    }
    rc = sd_allreduce_gram(ctx, comm, G, ldg, D, M);
    if (rc) return rc;
    // 2: the ranks share the CG iterations; 0: every rank solves alone (factorisation, or CG if sd_set_solver chose it)
    return solve_gram_impl(ctx, comm, G, ldg, D, M, reg, n_train_global, d_X, lambda_out, nullptr, distributed_solve == 2 ? 2 : 0);
}

int sd_centre_features(sd_ctx* ctx, sd_comm* comm, float* d_A, int64_t lda, int N_local, int D, int n_global,
                       const sd_regulariser* reg, float* d_mu)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_REQUIRE(ctx, d_mu && reg && D >= 1 && N_local >= 0 && n_global >= 1 && (N_local == 0 || (d_A && lda >= D)), "bad argument");
    if (D <= kLuMaxDim || reg->regularise_last_row) {       // a penalised last column cannot absorb the shift                                   // the small systems keep the reference-order LU on the rows as they are
        SD_CUDA(ctx, cudaMemsetAsync(d_mu, 0, (size_t)D * sizeof(float), ctx->stream));
        return SD_OK;
    }
    int splits = N_local / 512;
    splits = splits < 1 ? 1 : (splits > 16 ? 16 : splits);
    double* part = (double*)sd_workspace(ctx, SD_WS_PARTIAL, (size_t)splits * (D + 1) * sizeof(double));
    if (!part) return SD_ERR_CUDA;
    if (N_local > 0) {
        const dim3 grid(sd_div_up(D, 32), splits);
        colsum_kernel<<<grid, 256, 0, ctx->stream>>>(d_A, lda, N_local, D, part);
        SD_LAUNCH_CHECK(ctx, "colsum_kernel");
        colsum_finish_kernel<<<sd_div_up(D + 1, 256), 256, 0, ctx->stream>>>(part, splits, D);
        SD_LAUNCH_CHECK(ctx, "colsum_finish_kernel");
    } else {
        SD_CUDA(ctx, cudaMemsetAsync(part, 0, (size_t)(D + 1) * sizeof(double), ctx->stream));
    }
    int rc = sd_comm_allreduce_f64(ctx, comm, part, (size_t)D + 1, ctx->stream);     // no-op without a communicator
    if (rc) return rc;
    colmean_kernel<<<sd_div_up(D, 256), 256, 0, ctx->stream>>>(part, D, n_global, 1, d_mu);
    SD_LAUNCH_CHECK(ctx, "colmean_kernel");
    if (N_local > 0) {
        const long long total = (long long)N_local * (D - 1);
        const int blocks = (int)(sd_div_up(total, 256) < 32LL * ctx->sm_count ? sd_div_up(total, 256) : 32LL * ctx->sm_count);
        centre_kernel<<<blocks, 256, 0, ctx->stream>>>(d_A, lda, N_local, D, d_mu);
        SD_LAUNCH_CHECK(ctx, "centre_kernel");
    }
    return SD_OK;
}

int sd_learn_centred(sd_ctx* ctx, sd_comm* comm, const float* d_Ac, int64_t lda, const float* d_B, int64_t ldb, int N_local, int D, int M,
                     const sd_regulariser* reg, int n_train_global, int route, const float* d_mu, float* d_X, float* d_Xc, float* lambda_out)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_REQUIRE(ctx, M >= 1 && N_local >= 0 && d_mu && d_X, "bad argument");
    const int64_t ldg = ((int64_t)(D + M) + 3) / 4 * 4;
    float* G = (float*)sd_workspace(ctx, SD_WS_SCRATCH, (size_t)D * ldg * sizeof(float));
    if (!G) return SD_ERR_CUDA;
    SD_CUDA(ctx, cudaEventRecord(ctx->ev[0], ctx->stream));
    int rc;
    if (N_local > 0) rc = sd_gram(ctx, d_Ac, lda, d_B, ldb, N_local, D, M, G, ldg);
    else rc = sd_check_cuda(ctx, cudaMemsetAsync(G, 0, (size_t)D * ldg * sizeof(float), ctx->stream), "memset(G)");
    if (rc) return rc;
    const bool multi = sd_comm_size_of(comm) > 1;
    if (multi) {
        rc = route == 1 ? sd_reduce_scatter_gram(ctx, comm, G, ldg, D, M) : sd_allreduce_gram(ctx, comm, G, ldg, D, M);
        if (rc) return rc;
    }
    const float* mu = D > kLuMaxDim ? d_mu : nullptr;       // sd_centre_features leaves the small systems alone
    rc = solve_gram_impl(ctx, multi ? comm : nullptr, G, ldg, D, M, reg, n_train_global, d_X, lambda_out, nullptr, multi ? route : 0, mu, d_Xc);
    if (rc) return rc;
    if (!mu && d_Xc && d_Xc != d_X) SD_CUDA(ctx, cudaMemcpyAsync(d_Xc, d_X, (size_t)D * M * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
    return SD_OK;
}

int sd_learn_rank_revealing(sd_ctx* ctx, const float* d_A, int64_t lda, const float* d_B, int64_t ldb, int N, int D, int M,
                            const sd_regulariser* reg, float* d_X, float* lambda_out, int* rank_out)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_REQUIRE(ctx, M >= 1 && rank_out, "bad argument");
    const int64_t ldg = ((int64_t)(D + M) + 3) / 4 * 4;
    float* G = (float*)sd_workspace(ctx, SD_WS_SCRATCH, (size_t)D * ldg * sizeof(float));
    if (!G) return SD_ERR_CUDA;
    SD_CUDA(ctx, cudaEventRecord(ctx->ev[0], ctx->stream));
    int rc = sd_gram(ctx, d_A, lda, d_B, ldb, N, D, M, G, ldg);
    if (rc) return rc;
    return solve_gram_impl(ctx, nullptr, G, ldg, D, M, reg, N, d_X, lambda_out, rank_out);
}

int sd_learn(sd_ctx* ctx, const float* d_A, int64_t lda, const float* d_B, int64_t ldb, int N, int D, int M,
             const sd_regulariser* reg, float* d_X, float* lambda_out)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_REQUIRE(ctx, M >= 1, "labels must have at least one column");
    const int64_t ldg = ((int64_t)(D + M) + 3) / 4 * 4;
    float* G = (float*)sd_workspace(ctx, SD_WS_SCRATCH, (size_t)D * ldg * sizeof(float));
    if (!G) return SD_ERR_CUDA;
    SD_CUDA(ctx, cudaEventRecord(ctx->ev[0], ctx->stream));
    int rc = sd_gram(ctx, d_A, lda, d_B, ldb, N, D, M, G, ldg);
    if (rc) return rc;
    return sd_solve_gram(ctx, G, ldg, D, M, reg, N, d_X, lambda_out);
}

int sd_predict(sd_ctx* ctx, const float* d_values, int64_t ldv, int N, int D, const float* d_X, int M,
               float* d_out, int64_t ldo)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_REQUIRE(ctx, d_values && d_X && d_out && N >= 0 && D >= 1 && M >= 1 && ldv >= D && ldo >= M, "bad argument");
    GemmEpilogue ep;
    memset(&ep, 0, sizeof(ep));
    return launch_gemm_nn(ctx, d_values, ldv, N, D, d_X, M, M, d_out, ldo, 1.0f, 0.0f, ep);
}

__global__ void residual_kernel(const float* __restrict__ pred, const float* __restrict__ labels, long long ldl, int N, int M,
                                double* __restrict__ out /* [2] */)
{
    double num = 0.0, den = 0.0;
    const long long total = (long long)N * M;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long n = idx / M;
        const int c = (int)(idx - n * M);
        const float l = labels[n * ldl + c];
        const double d = (double)__fsub_rn(pred[idx], l);
        num += d * d;
        den += (double)l * (double)l;
    }
    __shared__ double rn[256], rd[256];
    rn[threadIdx.x] = num; rd[threadIdx.x] = den;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) { rn[threadIdx.x] += rn[threadIdx.x + o]; rd[threadIdx.x] += rd[threadIdx.x + o]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { atomicAdd(&out[0], rn[0]); atomicAdd(&out[1], rd[0]); }
}

int sd_test_residual(sd_ctx* ctx, const float* d_values, int64_t ldv, const float* d_labels, int64_t ldl, int N, int D,
                     const float* d_X, int M, double* residual_out)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_REQUIRE(ctx, d_values && d_labels && d_X && residual_out && N >= 1, "bad argument");
    float* pred = (float*)sd_workspace(ctx, SD_WS_PARTIAL, (size_t)N * M * sizeof(float));
    if (!pred) return SD_ERR_CUDA;
    int rc = sd_predict(ctx, d_values, ldv, N, D, d_X, M, pred, M);
    if (rc) return rc;
    double* acc = reinterpret_cast<double*>(reinterpret_cast<char*>(ctx->d_scratch) + 512);
    SD_CUDA(ctx, cudaMemsetAsync(acc, 0, 2 * sizeof(double), ctx->stream));
    const int blocks = sd_div_up((int64_t)N * M, 256) > 512 ? 512 : sd_div_up((int64_t)N * M, 256);
    residual_kernel<<<blocks, 256, 0, ctx->stream>>>(pred, d_labels, ldl, N, M, acc);
    SD_LAUNCH_CHECK(ctx, "residual_kernel");
    double* h = reinterpret_cast<double*>(reinterpret_cast<char*>(ctx->h_scratch) + 512);
    SD_CUDA(ctx, cudaMemcpyAsync(h, acc, 2 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    SD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *residual_out = sqrt(h[0]) / sqrt(h[1]);
    return SD_OK;
}

int sd_cascade_targets(sd_ctx* ctx, const float* d_x, const float* d_x_gt, int N, int P, const sd_normalisation* norm,
                       float* d_B, int64_t ldb)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_REQUIRE(ctx, d_x && d_x_gt && d_B && N >= 0 && P >= 1 && ldb >= P, "bad argument");
    if (N == 0) return SD_OK;
    sd_eyes_dev eyes;
    int rc = sd_eyes_to_dev(ctx, norm, P / 2, &eyes);
    if (rc) return rc;
    dim3 block(32, 8);
    targets_kernel<<<sd_div_up(N, 8), block, 0, ctx->stream>>>(d_x, d_x_gt, N, P, eyes, d_B, ldb);
    SD_LAUNCH_CHECK(ctx, "targets_kernel");
    return SD_OK;
}

int sd_cascade_update(sd_ctx* ctx, const float* d_A, int64_t lda, int N, int D, const float* d_X, int P,
                      const float* d_x, const sd_normalisation* norm, float* d_x_next)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_REQUIRE(ctx, d_A && d_X && d_x && d_x_next && N >= 0 && D >= 1 && P >= 1 && lda >= D, "bad argument");
    GemmEpilogue ep;
    memset(&ep, 0, sizeof(ep));
    ep.mode = 1;
    ep.x = d_x;
    ep.x_next = d_x_next;
    int rc = sd_eyes_to_dev(ctx, norm, P / 2, &ep.eyes);
    if (rc) return rc;
    SD_REQUIRE(ctx, d_x != d_x_next, "x_next must not alias x");
    return launch_gemm_nn(ctx, d_A, lda, N, D, d_X, P, P, nullptr, 0, 1.0f, 0.0f, ep);
}

int sd_subtract_templates(sd_ctx* ctx, float* d_A, int64_t lda, const float* d_T, int64_t ldt, int N, int D)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_REQUIRE(ctx, d_A && d_T && lda >= D && ldt >= D, "bad argument");
    if (N <= 0) return SD_OK;
    const int blocks = sd_div_up((int64_t)N * D, 256) > 4096 ? 4096 : sd_div_up((int64_t)N * D, 256);
    subtract_kernel<<<blocks, 256, 0, ctx->stream>>>(d_A, lda, d_T, ldt, N, D);
    SD_LAUNCH_CHECK(ctx, "subtract_kernel");
    return SD_OK;
}

}  // extern "C"
