/*
 * sd_b200.h -- C ABI of the B200-native cascaded-regression engine.
 *
 * This is the drop-in boundary for the hot path of patrikhuber/superviseddescent
 * (HOG projection -> LinearRegressor::learn -> predict/detect cascade).  Plain C:
 * opaque handles, raw pointers, explicit sizes, int status codes.  No C++ / torch
 * types cross this boundary.  The C++14 header shells in
 * superviseddescent_b200/include/ (same class names and call signatures as the
 * reference) and the ctypes binding in superviseddescent_b200/ sit on top of it.
 *
 * Conventions (reference: SURVEY.md 8b)
 *   - matrices are row-major float32, one sample per row (cv::Mat CV_32FC1 as the
 *     reference uses it, regressors.hpp:202-206); `ld` = row stride in floats.
 *   - landmark rows are [x_0..x_{L-1}, y_0..y_{L-1}] (adaptive_vlhog.hpp:96-97).
 *   - images are 8-bit single channel (adaptive_vlhog.hpp:115-120 grey path); the host-frame detect calls also take
 *     8-bit B,G,R frames and convert them as cv::cvtColor(BGR2GRAY) does.
 *   - pointers named d_* are DEVICE pointers, h_* are HOST pointers.
 *   - every call is asynchronous on the context's stream unless it returns host
 *     data; sd_sync() waits.  Functions are re-entrant on distinct contexts.
 *   - return value 0 = SD_OK; otherwise an sd_status and sd_last_error(ctx) holds
 *     a message.  There is NO CPU fallback: without a usable GPU every compute
 *     entry point fails with SD_ERR_CUDA.
 *
 * Citations are file:line under the reference tree (/root/reference).
 */
#ifndef SD_B200_H
#define SD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define SD_API __attribute__((visibility("default")))
#else
#define SD_API
#endif

typedef enum {
    SD_OK = 0,
    SD_ERR_INVALID = 1,    /* bad argument / shape (the reference asserts) */
    SD_ERR_CUDA = 2,       /* CUDA runtime / driver failure, or no GPU */
    SD_ERR_IO = 3,         /* model file could not be opened/parsed (model.hpp:199 throws) */
    SD_ERR_MISSING_ID = 4, /* eye identifier not among the landmarks (helpers.hpp:144,153 throws) */
    SD_ERR_NUMERIC = 5,    /* non-finite result / non-positive pivot */
    SD_ERR_UNSUPPORTED = 6
} sd_status;

typedef struct sd_ctx sd_ctx;       /* one per host thread / stream */
typedef struct sd_model sd_model;   /* rcr::detection_model resident on the device */
typedef struct sd_comm sd_comm;     /* multi-GPU communicator (see "multi-GPU training" below) */

/* rcr::HoGParam (adaptive_vlhog.hpp:41-60); same field order as its cereal archive */
typedef struct {
    int32_t variant;             /* 0 = VlHogVariantDalalTriggs, 1 = VlHogVariantUoctti (hog.h:70) */
    int32_t num_cells;
    int32_t cell_size;
    int32_t num_bins;            /* undirected orientations K */
    float relative_patch_size;   /* patch width as a fraction of the inter-eye distance */
} sd_hog_param;

/* superviseddescent::Regulariser (regressors.hpp:87-169) */
typedef struct {
    int32_t type;                /* 0 = Manual, 1 = MatrixNorm (regressors.hpp:93-97) */
    float param;                 /* lambda, or the factor applied to ||AtA||_F / N */
    int32_t regularise_last_row; /* 0: the bias row gets no lambda (regressors.hpp:143-146) */
} sd_regulariser;

/* NormalisationStrategy of the optimiser: NoNormalisation (superviseddescent.hpp:60-74)
 * or rcr::InterEyeDistanceNormalisation (model.hpp:84-116).  Eye landmarks are given as
 * row indices into the landmark list (the host shells resolve the string ids). */
typedef struct {
    int32_t kind;                /* 0 = none, 1 = inter-eye distance */
    int32_t n_right, n_left;     /* 1..4 each */
    int32_t right_idx[4];
    int32_t left_idx[4];
} sd_normalisation;

/* Region of interest of one frame that is resident on the device (see sd_image_batch.d_roi). */
typedef struct {
    int32_t x, y, w, h;          /* in frame coordinates */
    int32_t row_stride;          /* bytes between ROI rows in the packed buffer (multiple of 4) */
    int32_t reserved;
    int64_t offset;              /* byte offset of the ROI's first pixel from d_data */
} sd_roi;

/* One frame of a batch whose frames differ in size (the reference's HogTransform takes a std::vector<cv::Mat> of arbitrary
 * sizes: rcr-train and examples/landmark_detection.cpp train on photographs of different resolutions). */
typedef struct {
    int32_t width, height;       /* defines where the zero padding of a patch starts for THIS frame */
    int32_t row_stride;          /* bytes */
    int32_t reserved;
    int64_t offset;              /* byte offset of the frame's first pixel from d_data */
} sd_frame;

/* A batch of 8UC1 images resident on the device: equally sized (width/height/strides below), or -- d_frames != NULL -- one
 * descriptor per frame. */
typedef struct {
    const uint8_t* d_data;
    int32_t width, height;       /* frame size: defines where the zero padding of a patch starts */
    int32_t row_stride;          /* bytes */
    int64_t image_stride;        /* bytes between consecutive images */
    int32_t count;
    /* Optional (NULL = whole frames are resident): only a region of interest of every frame was uploaded.
     * d_roi[i] locates it inside d_data; a patch that needs frame pixels outside its ROI sets d_roi_miss[i]
     * (sd_detect_batch_host then repeats that face from the full frame). */
    const sd_roi* d_roi;
    uint8_t* d_roi_miss;
    /* Optional (NULL = equally sized frames): per-frame size / pitch / position; width, height, row_stride and image_stride
     * above are then ignored.  With d_roi, d_frames[i] gives only the size of the frame that d_roi[i] was cut from (its
     * row_stride and offset are unused). */
    const sd_frame* d_frames;
} sd_image_batch;

/* One frame in host memory for sd_detect_faces_host / sd_detect_faces_host_init; frames need not be contiguous or equally
 * sized.  channels: 0 or 1 = 8UC1, 3 = 8UC3 interleaved B,G,R (cv::imread / cv::VideoCapture output; converted as
 * cv::cvtColor(BGR2GRAY), adaptive_vlhog.hpp:114-120, bit for bit like sd_bgr2gray).  The frame is `height` rows of
 * `row_stride` bytes (at least channels x width) from h_data; its last row needs only channels x width readable bytes. */
typedef struct {
    const uint8_t* h_data;
    int32_t width, height, row_stride;
    int32_t channels;
} sd_host_frame;

/* ---- context --------------------------------------------------------------------------- */
/* stream: a cudaStream_t owned by the caller (e.g. torch's current stream); NULL is the CUDA default
 * stream (which is also torch's default stream); SD_STREAM_OWN lets the context create and own a
 * non-blocking stream. */
#define SD_STREAM_OWN ((void*)(intptr_t)-1)
SD_API int sd_ctx_create(int device, void* stream, sd_ctx** out);
SD_API void sd_ctx_destroy(sd_ctx* ctx);
SD_API const char* sd_last_error(const sd_ctx* ctx);
SD_API int sd_sync(sd_ctx* ctx);
SD_API const char* sd_version(void);
/* number of kernels of THIS library launched on ctx since creation (bench.py's gpu_launches) */
SD_API int64_t sd_launch_count(const sd_ctx* ctx);
/* faces that sd_detect_batch_host / sd_detect_faces_host had to repeat from their full frame (a patch left the uploaded ROI) */
SD_API int64_t sd_roi_fallback_count(const sd_ctx* ctx);

/* device / pinned-host memory for hosts that do not bring their own allocator */
SD_API int sd_malloc(sd_ctx* ctx, size_t bytes, void** d_ptr);
SD_API int sd_free(sd_ctx* ctx, void* d_ptr);
SD_API int sd_host_alloc(sd_ctx* ctx, size_t bytes, void** h_ptr);   /* pinned */
SD_API int sd_host_free(sd_ctx* ctx, void* h_ptr);
SD_API int sd_memcpy_h2d(sd_ctx* ctx, void* d_dst, const void* h_src, size_t bytes);  /* async */
SD_API int sd_memcpy_d2h(sd_ctx* ctx, void* h_dst, const void* d_src, size_t bytes);  /* async */
SD_API int sd_memset(sd_ctx* ctx, void* d_dst, int value, size_t bytes);
/* strided rows in one call (cv::Mat rows with a step, or [A | B] side by side on the device): `rows` rows of `row_bytes`
 * bytes, pitches in bytes; async on the context's stream */
SD_API int sd_memcpy2d_h2d(sd_ctx* ctx, void* d_dst, size_t dst_pitch, const void* h_src, size_t src_pitch, size_t row_bytes, size_t rows);
SD_API int sd_memcpy2d_d2h(sd_ctx* ctx, void* h_dst, size_t dst_pitch, const void* d_src, size_t src_pitch, size_t row_bytes, size_t rows);
SD_API int sd_memcpy2d_d2d(sd_ctx* ctx, void* d_dst, size_t dst_pitch, const void* d_src, size_t src_pitch, size_t row_bytes, size_t rows);

/* ---- projection h: rcr::HogTransform::operator() batched (adaptive_vlhog.hpp:109-185) -- */
/* D = L * num_cells^2 * (3K+4 | 4K) + 1 */
SD_API int sd_hog_feature_length(int num_landmarks, const sd_hog_param* p);
/* Asynchronous.  A degenerate sample (inter-eye distance too small for a patch: the reference's cv::resize would throw) or an
 * image index out of range raises a flag on the device that the NEXT synchronising call on the context reports as
 * SD_ERR_INVALID: sd_sync, sd_hog_debug, sd_detect_batch_device / _host.
 * For sample i: image = images[d_image_index ? d_image_index[i] : i], landmarks = d_x[i, 0:2L].
 * Writes the reference's feature row (per landmark [dim][cell col][cell row], then bias 1)
 * to d_A[i*ld .. i*ld + D).  Columns [D, ld) are left untouched.  hog.c:174-204,595-728,857-1062
 * run fused with the crop / zero-pad / cv::resize glue of adaptive_vlhog.hpp:123-176.
 * eyes == NULL (or eyes->kind == 0) selects the NON-adaptive HogTransform of the hello-world example
 * (examples/landmark_detection.cpp:195-261): patch half-size = num_cells * (cell_size / 2), no resize,
 * relative_patch_size ignored; cell_size must be even.  That functor has no bias column: use the first D - 1 columns. */
SD_API int sd_hog_batch(sd_ctx* ctx, const sd_image_batch* images, const int32_t* d_image_index,
                        const float* d_x, int64_t ldx, int num_samples, int num_landmarks,
                        const sd_normalisation* eyes, const sd_hog_param* p,
                        float* d_A, int64_t ld);
/* parity taps (integer results that must match the reference exactly): per (sample, landmark)
 * patch centre/half size, and optionally the resized u8 patches and per-pixel orientation bins. */
SD_API int sd_hog_debug(sd_ctx* ctx, const sd_image_batch* images, const int32_t* d_image_index,
                        const float* d_x, int64_t ldx, int num_samples, int num_landmarks,
                        const sd_normalisation* eyes, const sd_hog_param* p,
                        int32_t* d_geometry /* N*L*3: cx, cy, half */,
                        uint8_t* d_patches /* N*L*fs*fs or NULL */,
                        int8_t* d_bins /* N*L*fs*fs or NULL, -1 on border / zero gradient */);

/* Colour frames: HogTransform::operator() converts 3-channel images with cv::cvtColor(BGR2GRAY) before anything else
 * (adaptive_vlhog.hpp:114-120).  Same conversion on the device, once per frame instead of once per call:
 *   gray = (3735 B + 19235 G + 9798 R + 2^14) >> 15      (OpenCV >= 3 fixed point; SURVEY.md 8c, pinned against cv2)
 * d_bgr: count frames of height x width interleaved B,G,R bytes; strides in bytes. */
SD_API int sd_bgr2gray(sd_ctx* ctx, const uint8_t* d_bgr, int width, int height, int64_t bgr_row_stride,
                       int64_t bgr_image_stride, int count, uint8_t* d_gray, int64_t gray_row_stride,
                       int64_t gray_image_stride);

/* ---- regressor: LinearRegressor<Solver> (regressors.hpp:318-400) ------------------------ */
/* Solver::solve (regressors.hpp:199-234 == verbose_solver.hpp:53-111):
 *   X = (A^T A + Lambda)^-1 A^T B ;  A: N x D, B: N x M, X: D x M (ldx_out = M).
 * lambda_out (host, may be NULL) receives the lambda actually applied (regressors.hpp:126-148).
 * n_train_global: the N used in the MatrixNorm rule (== N on one GPU; the global sample count
 * when the Gram was summed over ranks).  Phase timings (ms) of the last call, named as the
 * reference's VerbosePartialPivLUSolver prints them, are available from sd_solver_timings. */
SD_API int sd_learn(sd_ctx* ctx, const float* d_A, int64_t lda, const float* d_B, int64_t ldb,
                    int N, int D, int M, const sd_regulariser* reg, float* d_X, float* lambda_out);
/* The training path on CENTRED feature rows (what the shells' and the Python mirror's train() use for D > 256).
 * HOG features are non-negative, so A^T A is dominated by n mu mu^T and the covariance that decides the weights sits several
 * digits down; a float32 Gram matrix -- the reference's as much as this one -- then loses three digits of the weights (the
 * reference's own arithmetic is 2e-3 away from the float64 solution on RCR features).  Subtracting the column means before the
 * Gram is the same least-squares problem (A w + c 1 = (A - 1 mu^T) w + (c + mu.w) 1) without that loss:
 *   sd_centre_features : d_mu[c] = mean of column c over ALL ranks' rows (0 for the last = bias column); d_A[:, c] -= d_mu[c]
 *                        in place.  The shift is only the same problem when the last column is exactly all ones and is not
 *                        regularised (regressors.hpp:143-146): otherwise -- and for D <= 256 (reference-order LU) -- the rows are
 *                        left untouched and d_mu = 0, with which sd_learn_centred is sd_learn / sd_learn_dist.
 *   sd_learn_centred   : Gram of the centred rows, exchange (comm may be NULL; route as in sd_learn_dist), lambda from the norm
 *                        of the UNcentred A^T A (regressors.hpp:135: reconstructed from the centred Gram and mu), solve.
 *                        d_X  : D x M weights for uncentred features -- the model (bias shifted back: c' - mu.w);
 *                        d_Xc : (optional) the weights that go with the centred buffer, for sd_cascade_update on it. */
SD_API int sd_centre_features(sd_ctx* ctx, sd_comm* comm, float* d_A, int64_t lda, int N_local, int D, int n_global,
                              const sd_regulariser* reg, float* d_mu);
SD_API int sd_learn_centred(sd_ctx* ctx, sd_comm* comm, const float* d_Ac, int64_t lda, const float* d_B, int64_t ldb,
                            int N_local, int D, int M, const sd_regulariser* reg, int n_train_global, int route,
                            const float* d_mu, float* d_X, float* d_Xc, float* lambda_out);

/* ColPivHouseholderQRSolver::solve (regressors.hpp:264-305): the same system, plus the one diagnostic that solver exists for --
 * the numerical rank of the regularised A^T A (regressors.hpp:288-293 prints it and asks for a larger lambda).  A^T A + Lambda is
 * symmetric positive semi-definite, so the rank comes from a diagonally pivoted Cholesky (threshold eps * D relative to the
 * largest pivot, Eigen's default rule), D <= 4096; beyond that *rank_out = -1 (not computed).  Like the reference the call goes
 * on to solve when the matrix is rank deficient; if the solve itself then breaks down the status is SD_ERR_NUMERIC and
 * sd_last_error carries the reference's message with the rank. */
SD_API int sd_learn_rank_revealing(sd_ctx* ctx, const float* d_A, int64_t lda, const float* d_B, int64_t ldb,
                                   int N, int D, int M, const sd_regulariser* reg, float* d_X, float* lambda_out, int* rank_out);
/* The same, split at the multi-GPU exchange point (superviseddescent.hpp:207 / SURVEY 8e):
 *   1. sd_gram      : d_G[Dx(D+M)] = [A^T A | A^T B] of the local rows (upper triangle of the
 *                     D x D part is valid; row stride ldg >= D+M)
 *   2. (caller)     : allreduce d_G over ranks
 *   3. sd_solve_gram: regularise with n_train_global and solve, replicated on every rank */
SD_API int sd_gram(sd_ctx* ctx, const float* d_A, int64_t lda, const float* d_B, int64_t ldb,
                   int N, int D, int M, float* d_G, int64_t ldg);
SD_API int sd_solve_gram(sd_ctx* ctx, float* d_G, int64_t ldg, int D, int M,
                         const sd_regulariser* reg, int n_train_global, float* d_X, float* lambda_out);
/* LinearRegressor::predict (regressors.hpp:377-381): out[N x M] = values[N x D] * X[D x M] */
SD_API int sd_predict(sd_ctx* ctx, const float* d_values, int64_t ldv, int N, int D,
                      const float* d_X, int M, float* d_out, int64_t ldo);
/* LinearRegressor::test (regressors.hpp:361-369): ||values X - labels||_2 / ||labels||_2 */
SD_API int sd_test_residual(sd_ctx* ctx, const float* d_values, int64_t ldv, const float* d_labels,
                            int64_t ldl, int N, int D, const float* d_X, int M, double* residual_out);
/* timings of the last sd_learn / sd_solve_gram: [0] "At * A", [1] "AtA + Reg", [2] "Decomposition",
 * [3] "solve()" in milliseconds (verbose_solver.hpp:66-103) */
SD_API int sd_solver_timings(sd_ctx* ctx, float ms_out[4]);
/* precision of the tensor-core Gram: 0 = 3xTF32 split on the truncated operand (default: Gram ~2e-7),
 * 3 = 3xTF32 split with the hi part rounded in shared memory (unbiased: Gram ~7e-8, ~15 % slower),
 * 1 = single TF32 pass (~7e-5), 2 = force the fp32 SIMT kernel (~3e-7) */
SD_API int sd_set_gram_mode(sd_ctx* ctx, int mode);

/* ---- multi-GPU training: the exchange at superviseddescent.hpp:207 (SURVEY 8e) ----------------------------------------
 * One process per GPU, samples (rows of A) sharded over the ranks.  [A^T A | A^T b] is a sum over the shards, so per cascade
 * level there is ONE collective on it; lambda uses the global sample count.  The collectives are NCCL (bound at run time:
 * libnccl.so.2 must be loadable when nranks > 1).  Three routes:
 *   replicated : sd_gram -> sd_allreduce_gram -> sd_solve_gram on every rank (small systems; the solve does not scale)
 *   shared CG  : sd_gram -> sd_allreduce_gram -> conjugate gradients whose product S P is split over the ranks by slabs of the
 *                contraction, one all-reduce of 2L x D floats per iteration (sd_learn_dist / sd_learn_centred with
 *                distributed_solve = 2); falls back to the replicated factorisation when CG does not converge
 *   distributed: sd_gram -> sd_reduce_scatter_gram -> sd_solve_gram_dist: the 256-row panels of [AtA|Atb] are owned
 *                block-row-cyclically (panel p by rank p % nranks); the owner factors its panel, broadcasts it, every rank
 *                updates the block rows it owns (blocked right-looking Cholesky, same kernels as on one GPU); every rank
 *                ends with the same X.  sd_learn_dist runs any of the routes from the local rows.
 * Determinism: for a fixed nranks the result is reproducible bit for bit; it differs from the one-GPU result only by the
 * summation order of the partial Gram matrices (~1e-7 relative). */
#define SD_COMM_ID_BYTES 128
/* rank 0 obtains an id and hands it to the other ranks by any means the host has (MPI, torch.distributed, a file) */
SD_API int sd_comm_get_unique_id(uint8_t* id_out /* SD_COMM_ID_BYTES */);
SD_API int sd_comm_create(sd_ctx* ctx, const uint8_t* id, int rank, int nranks, sd_comm** out);   /* collective */
/* adopt a ncclComm_t the host already owns (it is not destroyed by sd_comm_destroy) */
SD_API int sd_comm_adopt(sd_ctx* ctx, void* nccl_comm, int rank, int nranks, sd_comm** out);
SD_API void sd_comm_destroy(sd_comm* comm);
SD_API int sd_comm_rank(const sd_comm* comm);
SD_API int sd_comm_size(const sd_comm* comm);
/* sum of one host integer over the ranks (the N of the MatrixNorm rule, regressors.hpp:135) */
SD_API int sd_comm_sum_int64(sd_ctx* ctx, sd_comm* comm, int64_t* h_value);
/* d_recv[r * bytes_per_rank ..] = rank r's d_send (current landmarks for a training callback, superviseddescent.hpp:217) */
SD_API int sd_comm_allgather(sd_ctx* ctx, sd_comm* comm, const void* d_send, size_t bytes_per_rank, void* d_recv);
/* in place on d_G (D x ldg, as written by sd_gram): sums over the ranks the part the solve reads -- every 256-row band from
 * its diagonal column to the end of its rows (the upper triangle and the right-hand sides; about half of the buffer) */
SD_API int sd_allreduce_gram(sd_ctx* ctx, sd_comm* comm, float* d_G, int64_t ldg, int D, int M);
/* the same sums, but band p is only delivered to rank p % nranks (what sd_solve_gram_dist expects) */
SD_API int sd_reduce_scatter_gram(sd_ctx* ctx, sd_comm* comm, float* d_G, int64_t ldg, int D, int M);
/* sd_solve_gram on a reduce-scattered d_G; collective, every rank receives X (and the same lambda) */
SD_API int sd_solve_gram_dist(sd_ctx* ctx, sd_comm* comm, float* d_G, int64_t ldg, int D, int M,
                              const sd_regulariser* reg, int n_train_global, float* d_X, float* lambda_out);
/* LinearRegressor::learn on sharded rows: local Gram, exchange, solve.  distributed_solve: 0 = all-reduce, every rank solves
 * alone; 1 = reduce to the panel owners + distributed factorisation; 2 = all-reduce + conjugate gradients shared by the ranks
 * (see sd_set_solver).  N_local may be 0. */
SD_API int sd_learn_dist(sd_ctx* ctx, sd_comm* comm, const float* d_A, int64_t lda, const float* d_B, int64_t ldb,
                         int N_local, int D, int M, const sd_regulariser* reg, int n_train_global, int distributed_solve,
                         float* d_X, float* lambda_out);

/* Solver of the systems with D > 256 (smaller ones always take the reference-order partial-pivot LU):
 *   0 = blocked Cholesky (default): the direct solve that stands in for Eigen::PartialPivLU (regressors.hpp:224-225);
 *   1 = conjugate gradients on the tensor cores: after the bias column has been eliminated the regularised Gram matrix of the
 *       centred features is very well conditioned under the MatrixNorm rule (condition number ~ N / 350 for RCR features), so a
 *       few dozen products with the D x D matrix replace the D^3 / 3 factorisation; it stops at a relative residual of 2e-6 and
 *       falls back to the Cholesky if the recurrence breaks down or stalls (ill-conditioned systems, tiny lambda).
 * sd_learn_dist: distributed_solve 2 = the ranks share the CG iterations (rows of the matrix sharded, one all-reduce of
 * 2L x D floats per iteration).  sd_solver_iterations: CG iterations of the last solve (0 = the factorisation ran). */
SD_API int sd_set_solver(sd_ctx* ctx, int mode);
SD_API int sd_solver_iterations(const sd_ctx* ctx);

/* ---- cascade steps: SupervisedDescentOptimiser (superviseddescent.hpp:165-344) ---------- */
/* b_i = (x_i - x_gt_i) (.) norm(x_i)     (superviseddescent.hpp:199-205) */
SD_API int sd_cascade_targets(sd_ctx* ctx, const float* d_x, const float* d_x_gt, int N, int P,
                              const sd_normalisation* norm, float* d_B, int64_t ldb);
/* x_next_i = x_i - (A_i X) (.) (1 / norm(x_i))   (superviseddescent.hpp:209-215, 296-301, 336-339)
 * d_x_next must not alias d_x. */
SD_API int sd_cascade_update(sd_ctx* ctx, const float* d_A, int64_t lda, int N, int D,
                             const float* d_X, int P, const float* d_x, const sd_normalisation* norm,
                             float* d_x_next);
/* observed = features - templates (superviseddescent.hpp:191-197), in place on A */
SD_API int sd_subtract_templates(sd_ctx* ctx, float* d_A, int64_t lda, const float* d_T, int64_t ldt,
                                 int N, int D);

/* ---- rcr::detection_model (model.hpp:122-219) -------------------------------------------- */
/* load_detection_model / save_detection_model (model.hpp:192-219): cereal binary, byte compatible */
SD_API int sd_model_load(sd_ctx* ctx, const char* path, sd_model** out);
SD_API int sd_model_save(sd_ctx* ctx, const sd_model* m, const char* path);
/* build a model from trained parts (detection_model ctor, model.hpp:128-129); weights are host
 * pointers, one D_s x 2L matrix per level; ids are NUL-terminated strings. */
SD_API int sd_model_create(sd_ctx* ctx, int num_levels, int num_landmarks,
                           const float* const* h_weights, const sd_regulariser* regs,
                           const sd_hog_param* hog_params, const float* h_mean,
                           const char* const* landmark_ids,
                           const char* const* right_eye_ids, int n_right,
                           const char* const* left_eye_ids, int n_left, sd_model** out);
SD_API void sd_model_destroy(sd_model* m);
SD_API int sd_model_num_levels(const sd_model* m);
SD_API int sd_model_num_landmarks(const sd_model* m);
SD_API int sd_model_hog_param(const sd_model* m, int level, sd_hog_param* out);
SD_API int sd_model_regulariser(const sd_model* m, int level, sd_regulariser* out);
SD_API int sd_model_normalisation(const sd_model* m, sd_normalisation* out);
SD_API int sd_model_get_mean(const sd_model* m, float* h_mean /* 2L */);            /* get_mean, model.hpp:159 */
SD_API int sd_model_get_weights(const sd_model* m, int level, float* h_w /* D x 2L */, int* rows, int* cols);
SD_API const char* sd_model_landmark_id(const sd_model* m, int i);
/* rcr::align_mean (model.hpp:64-76); host-side, a few flops */
SD_API int sd_align_mean(const float* h_mean, int num_landmarks, int box_x, int box_y, int box_w, int box_h,
                         float scaling_x, float scaling_y, float translation_x, float translation_y,
                         float* h_out);
/* Training front end of apps/rcr/rcr-train.cpp.
 * perturb (:130-146): translate a face box by fractions of its size and scale it about its centre (float arithmetic,
 * truncation toward zero like cv::Rect(int)); host-side, a few flops. */
SD_API int sd_perturb_box(int box_x, int box_y, int box_w, int box_h, float translation_x, float translation_y,
                          float scaling, int32_t out_box[4]);
/* calculate_normalised_landmark_errors (:149-212): d_err[r, i] = || pred[r, i] - gt[r, i] ||_2 / IED(pred[r]) for N rows of
 * 2L landmarks each ([x.., y..]); d_err: N x L, row pitch lde. */
SD_API int sd_normalised_landmark_errors(sd_ctx* ctx, const float* d_pred, int64_t ldp, const float* d_gt, int64_t ldgt,
                                         int N, int num_landmarks, const sd_normalisation* eyes, float* d_err, int64_t lde);
/* detection_model::detect(image, initialisation) batched, everything on the device
 * (model.hpp:147-157 -> superviseddescent.hpp:323-344).  d_x0: B x 2L initial landmarks. */
SD_API int sd_detect_batch_device(sd_ctx* ctx, const sd_model* m, const sd_image_batch* images,
                                  const float* d_x0, int count, float* d_landmarks);
/* detection_model::detect(image, facebox) batched with HOST buffers (model.hpp:132-144): aligns the
 * mean to each box, copies the frames host->device in chunks overlapped with compute, runs the cascade
 * and copies the B x 2L landmarks back.  h_images: count x height x row_stride bytes (8UC1; pinned
 * memory makes the copies asynchronous); h_boxes: count x 4 (x, y, w, h). */
SD_API int sd_detect_batch_host(sd_ctx* ctx, const sd_model* m, const uint8_t* h_images, int count,
                                int width, int height, int row_stride, const int32_t* h_boxes,
                                float* h_landmarks);

/* ---- several faces per frame, frames of any size ---------------------------------------------------------------------
 * A face detector returns a list of boxes per frame (cv::CascadeClassifier::detectMultiScale); these calls take every face of
 * a batch of frames in one call, each face carrying the index of its frame.  Results are bit-identical to detecting each face
 * on its own frame with the calls above. */
/* align_mean(mean, box) (model.hpp:64-76) for count boxes on the device: d_boxes is count x 4 (x, y, w, h) int32, row i of
 * d_x0 (row stride ldx floats) receives the 2L initial landmarks, bit-identical to sd_align_mean(.., 1, 1, 0, 0).  Async. */
SD_API int sd_model_align_boxes(sd_ctx* ctx, const sd_model* m, const int32_t* d_boxes, int count,
                                float* d_x0, int64_t ldx);
/* detect(image, initialisation) for count faces, everything on the device: face i starts from d_x0[i*2L ..] and reads frame
 * d_frame_index[i] of `frames` (equally sized frames, or one d_frames descriptor each; d_roi is not accepted).  An index out
 * of range is reported as SD_ERR_INVALID through the projection's status flag (the call synchronises). */
SD_API int sd_detect_faces_device(sd_ctx* ctx, const sd_model* m, const sd_image_batch* frames,
                                  const int32_t* d_frame_index, const float* d_x0, int count, float* d_landmarks);
/* detect(image, facebox) for count faces in num_frames host frames: face i has box h_boxes[4i ..] in frame
 * h_frames[h_frame_index[i]]; h_landmarks receives count x 2L.  Every index and every referenced frame (size, pitch,
 * channels) is checked before any work is queued (SD_ERR_INVALID); frames without faces are never read.  count == 0
 * returns SD_OK.  Gray and colour frames may be mixed.
 * Route: when every referenced frame is pinned and device-mapped with 16-byte aligned base and pitch, the neighbourhoods of
 * the faces are gathered from host memory (ROIs of one frame that intersect are gathered once, as one region; a colour ROI
 * is converted to gray as it is gathered, so only the neighbourhood is read and converted); otherwise every referenced frame
 * is copied to the device once, whatever its number of faces (colour frames as B,G,R, converted there). */
SD_API int sd_detect_faces_host(sd_ctx* ctx, const sd_model* m, const sd_host_frame* h_frames, int num_frames,
                                const int32_t* h_frame_index, const int32_t* h_boxes, int count, float* h_landmarks);
/* detect(image, initialisation) (model.hpp:147-157, e.g. the landmarks of the previous frame of a video) for count faces in
 * host frames: face i starts from h_x0[i * ldx .. + 2L] (ldx >= 2L floats).  Checks, routes and results as
 * sd_detect_faces_host, which is this call with the mean aligned to each box. */
SD_API int sd_detect_faces_host_init(sd_ctx* ctx, const sd_model* m, const sd_host_frame* h_frames, int num_frames,
                                     const int32_t* h_frame_index, const float* h_x0, int64_t ldx, int count,
                                     float* h_landmarks);

#ifdef __cplusplus
}
#endif
#endif /* SD_B200_H */
