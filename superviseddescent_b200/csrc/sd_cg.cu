// Conjugate-gradient solve of the regularised normal equations on the tensor cores (optional route of sd_solve_gram).
//
// After the bias column has been eliminated first (sd_linalg.cu, bias_extract_kernel) the system matrix is the Gram matrix of
// the CENTRED features plus lambda I.  With the reference's MatrixNorm rule lambda = 1.5 ||A^T A||_F / N is of the size of the
// largest eigenvalues, so the matrix is very well conditioned: measured condition number 3.5 at N = 900 samples, 10.5 at 3,600
// (it grows like N: ~30 for config 4, a few hundred for config 5).  CG then needs a few dozen iterations of
//     Q = S P   (one skinny product with the D x D matrix: 2 D^2 2L flops, the tcgen05 TN-GEMM of sd_gram_tc.cu in its narrow
//                variant: S is the 128-row operand, P the 64-column one, so the product is bound by the single read of S)
// instead of the D^3/3 factorisation whose chain of D dependent pivots does not parallelise -- and the product shards over
// GPUs by rows of S with one small all-reduce (2L x D floats) per iteration, which the factorisation cannot.
//
// All 2L right-hand sides advance in lockstep (independent CG recurrences sharing the product).  Reductions are two-stage with a
// fixed order, so the result is reproducible.  If the recurrence breaks down (p^T S p <= 0: not positive definite) or does not
// reach the tolerance, the caller falls back to the blocked Cholesky: the upper triangle of S and the right-hand sides are never
// modified here (only the unused lower triangle is filled with the mirror image).
#include "sd_internal.cuh"

#include <cmath>

namespace {

constexpr int CG_BX = 64, CG_BY = 4;           // block: 64 column lanes x 4 row lanes
constexpr int CG_G = 3;                        // column groups per thread: up to 192 right-hand sides (2L = 136 for 68 landmarks)
constexpr int CG_MAXCOLS = CG_BX * CG_G;

// The product streams the symmetric matrix once per iteration, so it gets a copy laid out for that: strip-major,
//     T[s][k - k0][c] = S[k][128 s + c],   k in [k0, k0 + kp) (this rank's slab of the contraction, zero rows beyond k1), c < 128
// -- the 128 columns of one CTA's tile are contiguous, a CTA reads its strip front to back (row-major S would give it 512-byte
// pieces 68 KB apart: measured 2.1 TB/s).  Built from the upper triangle only (S[k][j] = S[j][k] below the diagonal, transposed
// through shared memory); G itself is not modified.  One block per 32 x 32 tile of (k, j).
__global__ void __launch_bounds__(256) cg_pack_kernel(const float* __restrict__ G, long long ldg, int n, int k0, int k1, int kp, float* __restrict__ T)
{
    __shared__ float tile[32][33];
    const int tk = k0 + blockIdx.y * 32;                // rows k of the output tile (k0 is a multiple of 16, tiles may straddle)
    const int tj = blockIdx.x * 32;                     // columns j of the output tile
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const bool upper = tj >= tk + 31, lower = tj + 31 < tk;      // entirely on or above / strictly below the diagonal
    if (upper || !lower) {
        // direct part: S[k][j] for j >= k
        for (int r = ty; r < 32; r += 8) {
            const int k = tk + r, j = tj + tx;
            tile[r][tx] = (k < k1 && k < n && j < n && j >= k) ? G[(long long)k * ldg + j] : 0.f;
        }
    }
    float low[4] = {0.f, 0.f, 0.f, 0.f};
    if (!upper) {
        // mirrored part: S[k][j] = G[j][k] for j < k, read along k (coalesced) and transposed through shared memory
        __shared__ float tr[32][33];
        for (int r = ty; r < 32; r += 8) {
            const int j = tj + r, k = tk + tx;
            tr[r][tx] = (k < k1 && k < n && j < k) ? G[(long long)j * ldg + k] : 0.f;
        }
        __syncthreads();
        for (int q = 0; q < 4; ++q) low[q] = tr[tx][ty + 8 * q];
    }
    __syncthreads();
    for (int q = 0; q < 4; ++q) {
        const int r = ty + 8 * q, k = tk + r, j = tj + tx;
        if (k - k0 >= kp) continue;
        float v = 0.f;
        if (k < k1 && k < n && j < n) v = (j >= k) ? ((upper || !lower) ? tile[r][tx] : 0.f) : low[q];
        T[((long long)(j >> 7) * kp + (k - k0)) * 128 + (j & 127)] = v;
    }
}

struct CgBuf {
    float *X, *R, *P, *Q;
    double *part;          // [2][nblk][CG_MAXCOLS]: partial sums of p.q and of r.r, one row per 32-row tile
    float *rs;             // [2][CG_MAXCOLS] ping-pong r.r
    float *bb;             // [CG_MAXCOLS]   b.b
    float *ab;             // [2][CG_MAXCOLS] alpha, beta of the current iteration
    float *conv;           // [0] max_c sqrt(rs / bb) of the latest iteration; [1] breakdown flag
    int nblk;              // number of 32-row tiles
};

constexpr int CG_TR = 32;                      // rows per tile of the vector kernels

// folds the 4 row lanes of a tile and stores the tile's partial sums
__device__ __forceinline__ void cg_store_partials(const double (&acc)[CG_G], double* __restrict__ dst)
{
    __shared__ double red[4][CG_MAXCOLS];
    const int cx = threadIdx.x & 63, ry = threadIdx.x >> 6;
#pragma unroll
    for (int g = 0; g < CG_G; ++g) red[ry][cx + g * CG_BX] = acc[g];
    __syncthreads();
    if (ry == 0)
#pragma unroll
        for (int g = 0; g < CG_G; ++g) {
            const int c = cx + g * CG_BX;
            dst[c] = red[0][c] + red[1][c] + red[2][c] + red[3][c];
        }
}


// Sum of the tiles' partial sums for every column, by ONE block of 1024 threads: 16 threads per column add interleaved subsets,
// then the 16 sub-sums are folded in a fixed order (reproducible).  out[c] valid for c < CG_MAXCOLS after the call (all threads).
__device__ __forceinline__ void cg_sum_partials(const double* __restrict__ part, int nblk, int M, double* s_out /* [CG_MAXCOLS] shared */)
{
    __shared__ double s_sub[16][CG_BX];
    const int cx = threadIdx.x & 63, sub = threadIdx.x >> 6;          // 64 x 16
    for (int g = 0; g < CG_G; ++g) {
        const int c = cx + g * CG_BX;
        double acc = 0.0;
        if (c < M)
            for (int k = sub; k < nblk; k += 16) acc += part[(long long)k * CG_MAXCOLS + c];
        s_sub[sub][cx] = acc;
        __syncthreads();
        if (sub == 0) {
            double t = 0.0;
#pragma unroll
            for (int q = 0; q < 16; ++q) t += s_sub[q][cx];
            s_out[c] = t;
        }
        __syncthreads();
    }
}

// R = P = B (the right-hand-side columns of G), X = 0, partial sums of b.b; one 32-row tile per block
__global__ void __launch_bounds__(256) cg_init_kernel(const float* __restrict__ G, long long ldg, int n, int col0, int M, int Mp, CgBuf b)
{
    const int cx = threadIdx.x & 63, ry = threadIdx.x >> 6, i0 = blockIdx.x * CG_TR;
    double acc[CG_G] = {};
    for (int r = ry; r < CG_TR; r += 4) {
        const int i = i0 + r;
        if (i >= n) break;
#pragma unroll
        for (int g = 0; g < CG_G; ++g) {
            const int c = cx + g * CG_BX;
            if (c < Mp) {
                const float v = c < M ? G[(long long)i * ldg + col0 + c] : 0.f;
                b.R[(long long)i * Mp + c] = v;
                b.P[(long long)i * Mp + c] = v;
                b.X[(long long)i * Mp + c] = 0.f;
                acc[g] += (double)v * (double)v;
            }
        }
    }
    cg_store_partials(acc, b.part + (long long)blockIdx.x * CG_MAXCOLS);
}

// one block: rs[0] = bb = sum of the tiles' partials
__global__ void __launch_bounds__(1024) cg_init_finish_kernel(CgBuf b, int M)
{
    __shared__ double s_sum[CG_MAXCOLS];
    cg_sum_partials(b.part, b.nblk, M, s_sum);
    const int c = threadIdx.x;
    if (c >= CG_MAXCOLS) return;
    b.rs[c] = c < M ? (float)s_sum[c] : 0.f;
    b.bb[c] = c < M ? (float)s_sum[c] : 0.f;
    if (c == 0) { b.conv[0] = 1.f; b.conv[1] = 0.f; }
}

// partial[tile][c] = sum over the tile's rows of P[i][c] * Q[i][c]
__global__ void __launch_bounds__(256) cg_dot_kernel(CgBuf b, int n, int M, int Mp)
{
    const int cx = threadIdx.x & 63, ry = threadIdx.x >> 6, i0 = blockIdx.x * CG_TR;
    double acc[CG_G] = {};
    for (int r = ry; r < CG_TR && i0 + r < n; r += 4)
#pragma unroll
        for (int g = 0; g < CG_G; ++g) {
            const int c = cx + g * CG_BX;
            if (c < M) {
                const long long o = (long long)(i0 + r) * Mp + c;
                acc[g] += (double)b.P[o] * (double)b.Q[o];
            }
        }
    cg_store_partials(acc, b.part + (long long)blockIdx.x * CG_MAXCOLS);
}

// one block: alpha = rs / (p.q), partials added in a fixed order
__global__ void __launch_bounds__(1024) cg_alpha_kernel(CgBuf b, int M, int parity)
{
    __shared__ double s_sum[CG_MAXCOLS];
    cg_sum_partials(b.part, b.nblk, M, s_sum);
    const int c = threadIdx.x;
    if (c >= CG_MAXCOLS) return;
    float alpha = 0.f;
    if (c < M) {
        const double pq = s_sum[c];
        const float rs = b.rs[parity * CG_MAXCOLS + c];
        if (rs > 0.f) {
            if (pq > 0.0) alpha = (float)((double)rs / pq);
            else b.conv[1] = 1.f;                                       // p^T S p <= 0: the matrix is not positive definite
        }
    }
    b.ab[c] = alpha;
}

// X += alpha P; R -= alpha Q; partials of r.r
__global__ void __launch_bounds__(256) cg_update_xr_kernel(CgBuf b, int n, int M, int Mp)
{
    const int cx = threadIdx.x & 63, ry = threadIdx.x >> 6, i0 = blockIdx.x * CG_TR;
    double acc[CG_G] = {};
    for (int r = ry; r < CG_TR && i0 + r < n; r += 4)
#pragma unroll
        for (int g = 0; g < CG_G; ++g) {
            const int c = cx + g * CG_BX;
            if (c < M) {
                const float alpha = b.ab[c];
                const long long o = (long long)(i0 + r) * Mp + c;
                b.X[o] = fmaf(alpha, b.P[o], b.X[o]);
                const float rr = fmaf(-alpha, b.Q[o], b.R[o]);
                b.R[o] = rr;
                acc[g] += (double)rr * (double)rr;
            }
        }
    cg_store_partials(acc, b.part + ((long long)b.nblk + blockIdx.x) * CG_MAXCOLS);
}

// one block: beta = rs_new / rs, rs_new, the convergence measure
__global__ void __launch_bounds__(1024) cg_beta_kernel(CgBuf b, int M, int parity)
{
    __shared__ double s_sum[CG_MAXCOLS];
    __shared__ float s_rel[CG_MAXCOLS];
    cg_sum_partials(b.part + (long long)b.nblk * CG_MAXCOLS, b.nblk, M, s_sum);
    const int c = threadIdx.x;
    if (c < CG_MAXCOLS) {
        const double rn = c < M ? s_sum[c] : 0.0;
        const float rs = b.rs[parity * CG_MAXCOLS + c];
        b.ab[CG_MAXCOLS + c] = (c < M && rs > 0.f) ? (float)(rn / (double)rs) : 0.f;
        const float bbv = b.bb[c];
        s_rel[c] = (c < M && bbv > 0.f) ? sqrtf((float)rn / bbv) : 0.f;
        b.rs[(parity ^ 1) * CG_MAXCOLS + c] = c < M ? (float)rn : 0.f;
    }
    __syncthreads();
    if (c == 0) {
        float m = 0.f;
        for (int k = 0; k < CG_MAXCOLS; ++k) m = fmaxf(m, s_rel[k]);
        b.conv[0] = m;
    }
}

// P = R + beta P
__global__ void __launch_bounds__(256) cg_update_p_kernel(CgBuf b, int n, int Mp)
{
    const long long total = (long long)n * Mp;
    for (long long idx = blockIdx.x * 256LL + threadIdx.x; idx < total; idx += (long long)gridDim.x * 256) {
        const int c = (int)(idx % Mp);
        b.P[idx] = fmaf(b.ab[CG_MAXCOLS + c], b.P[idx], b.R[idx]);
    }
}

}  // namespace

// Solves S W = B for the n x n symmetric matrix whose upper triangle sits in G (pitch ldg) and whose M right-hand sides are the
// columns [col0, col0 + M) of the same rows.  W: n x Mp row-major (Mp = M rounded up to 4) in *W_out (workspace owned by ctx).
// Returns SD_OK when converged (iterations in *iters), SD_ERR_NUMERIC when the caller should fall back to the factorisation.
int sd_cg_solve(sd_ctx* ctx, sd_comm* comm, float* G, int64_t ldg, int n, int col0, int M, float** W_out, int* ldw_out, int* iters)
{
    SD_REQUIRE(ctx, M >= 1 && M <= CG_MAXCOLS && n >= 1, "CG route: 1..192 right-hand sides");
    const int Mp = (M + 3) / 4 * 4;
    const int nranks = sd_comm_size_of(comm), me = sd_comm_rank_of(comm);
    CgBuf b;
    b.nblk = sd_div_up(n, CG_TR);
    const size_t vec = (size_t)n * Mp;
    const size_t tile_cap = ((size_t)sd_div_up(n, 128) + 1) * 2 * 2;                                      // int2 entries, as floats
    const size_t floats = 4 * vec + 6 * CG_MAXCOLS + 64 + tile_cap + 8;
    const size_t bytes = floats * sizeof(float) + (size_t)2 * b.nblk * CG_MAXCOLS * sizeof(double) + 256;
    char* ws = (char*)sd_workspace(ctx, SD_WS_CG, bytes);
    if (!ws) return SD_ERR_CUDA;
    b.part = reinterpret_cast<double*>(ws);
    float* f = reinterpret_cast<float*>(ws + (size_t)2 * b.nblk * CG_MAXCOLS * sizeof(double));
    b.X = f; b.R = f + vec; b.P = f + 2 * vec; b.Q = f + 3 * vec;
    float* tail = b.Q + vec;
    tail = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(tail) + 15) & ~(uintptr_t)15);
    b.rs = tail; b.bb = tail + 2 * CG_MAXCOLS; b.ab = tail + 3 * CG_MAXCOLS; b.conv = tail + 5 * CG_MAXCOLS;
    void* d_tile_buf = tail + 5 * CG_MAXCOLS + 16;

    // this rank's slab of the contraction (rows of S), multiples of 16 rows
    int k0 = 0, k1 = n;
    sd_cg_slab(n, nranks, me, &k0, &k1);
    const int nstrips = sd_div_up(n, 128);
    const int kp = (k1 - k0 + 15) / 16 * 16;
    float* T = nullptr;
    if (k1 > k0) {
        T = (float*)sd_workspace(ctx, SD_WS_CGMAT, (size_t)nstrips * kp * 128 * sizeof(float));
        if (!T) return SD_ERR_CUDA;
        const dim3 pg(nstrips * 4, sd_div_up(kp, 32));
        cg_pack_kernel<<<pg, 256, 0, ctx->stream>>>(G, ldg, n, k0, k1, kp, T);
        SD_LAUNCH_CHECK(ctx, "cg_pack_kernel");
    }
    cg_init_kernel<<<b.nblk, 256, 0, ctx->stream>>>(G, ldg, n, col0, M, Mp, b);
    SD_LAUNCH_CHECK(ctx, "cg_init_kernel");
    cg_init_finish_kernel<<<1, 1024, 0, ctx->stream>>>(b, M);
    SD_LAUNCH_CHECK(ctx, "cg_init_finish_kernel");

    constexpr float tol = 2e-6f;
    constexpr int max_iter = 600;
    // The product is the same launch every iteration: Q[n x M] = S[k0:k1, :]^T P[k0:k1, :]  ( = S P summed over the ranks' slabs of
    // the contraction: S is symmetric ); prepared once (tensor maps, tile list).  S is the 128-row operand: n / 128 tiles keep the
    // SMs busy at any slab size, P is the narrow operand.  Pad columns of Q and the rows of a rank without slab stay zero.
    SD_CUDA(ctx, cudaMemsetAsync(b.Q, 0, vec * sizeof(float), ctx->stream));
    alignas(64) unsigned char plan[SD_TC_PLAN_BYTES];
    bool no_tiles = true;
    int rc = SD_OK;
    if (k1 > k0) {
        rc = sd_gemm_tn_tc_prepare(ctx, T, 128, b.P + (size_t)k0 * Mp, Mp, k1 - k0, n, M, b.Q, Mp, 1.0f, 0.0f, 3, true, false,
                                   nullptr, 1, d_tile_buf, plan, &no_tiles, true, kp);
        if (rc) return rc;
    }
    // convergence read-backs: slot it % 8 holds {max relative residual, breakdown flag} after iteration it; the host looks at the
    // slot of LAG iterations ago, so the GPU never waits for the host
    constexpr int LAG = 3;
    float* h_conv = reinterpret_cast<float*>(reinterpret_cast<char*>(ctx->h_scratch) + 2048);
    for (int i = 0; i < 8; ++i)
        if (!ctx->cg_ev[i]) SD_CUDA(ctx, cudaEventCreateWithFlags(&ctx->cg_ev[i], cudaEventDisableTiming));
    int it = 0, prev_it = 0;
    float prev_conv = 0.f;
    bool converged = false, failed = false;
    for (; it < max_iter && !converged && !failed; ++it) {
        const int parity = it & 1;
        if (!no_tiles) {
            rc = sd_gemm_tn_tc_launch(ctx, plan);
            if (rc) return rc;
        } else {
            // a rank without slab (more ranks than 16-row groups) contributes zeros; Q holds last iteration's sum by now
            SD_CUDA(ctx, cudaMemsetAsync(b.Q, 0, vec * sizeof(float), ctx->stream));
        }
        if (nranks > 1) {
            rc = sd_comm_allreduce_f32(ctx, comm, b.Q, vec, ctx->stream);
            if (rc) return rc;
        }
        cg_dot_kernel<<<b.nblk, 256, 0, ctx->stream>>>(b, n, M, Mp);
        SD_LAUNCH_CHECK(ctx, "cg_dot_kernel");
        cg_alpha_kernel<<<1, 1024, 0, ctx->stream>>>(b, M, parity);
        SD_LAUNCH_CHECK(ctx, "cg_alpha_kernel");
        cg_update_xr_kernel<<<b.nblk, 256, 0, ctx->stream>>>(b, n, M, Mp);
        SD_LAUNCH_CHECK(ctx, "cg_update_xr_kernel");
        cg_beta_kernel<<<1, 1024, 0, ctx->stream>>>(b, M, parity);
        SD_LAUNCH_CHECK(ctx, "cg_beta_kernel");
        cg_update_p_kernel<<<2 * ctx->sm_count, 256, 0, ctx->stream>>>(b, n, Mp);
        SD_LAUNCH_CHECK(ctx, "cg_update_p_kernel");
        SD_CUDA(ctx, cudaMemcpyAsync(h_conv + 2 * (it & 7), b.conv, 2 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
        SD_CUDA(ctx, cudaEventRecord(ctx->cg_ev[it & 7], ctx->stream));
        const int look = it - LAG;
        if (look >= 4) {
            SD_CUDA(ctx, cudaEventSynchronize(ctx->cg_ev[look & 7]));
            const float cv = h_conv[2 * (look & 7)], bad = h_conv[2 * (look & 7) + 1];
            if (bad != 0.f || !(cv == cv)) { failed = true; break; }
            if (cv <= tol) converged = true;
            else if (look >= 30 && prev_conv > 0.f && look > prev_it) {
                // a system that would need more than max_iter iterations at the observed rate is the factorisation's job
                const double rate = pow((double)cv / (double)prev_conv, 1.0 / (double)(look - prev_it));
                if (rate >= 1.0 || (double)look + log((double)tol / (double)cv) / log(rate) > (double)max_iter) { failed = true; break; }
            }
            if ((look % 8) == 0) { prev_conv = cv; prev_it = look; }
        }
    }
    if (!converged && !failed) {
        // drain: the last LAG iterations have not been looked at yet
        SD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        for (int look = it - LAG < 0 ? 0 : it - LAG; look < it; ++look) {
            const float cv = h_conv[2 * (look & 7)], bad = h_conv[2 * (look & 7) + 1];
            if (bad != 0.f || !(cv == cv)) failed = true;
            else if (cv <= tol) converged = true;
        }
    }
    if (iters) *iters = it;
    if (!converged) return SD_ERR_NUMERIC;
    *W_out = b.X;
    *ldw_out = Mp;
    return SD_OK;
}
