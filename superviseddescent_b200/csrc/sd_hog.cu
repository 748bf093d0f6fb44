// Batched per-landmark HOG projection: the CUDA restatement of rcr::HogTransform::operator()
// (reference include/rcr/adaptive_vlhog.hpp:109-185) fused with VLFeat's vl_hog_put_image /
// vl_hog_extract (reference include/rcr/hog.c:595-728, :857-1062).
//
// One CTA walks the patches of up to kHogGroup consecutive landmarks of one sample.  Everything between the 8-bit source
// image in HBM and the feature row in HBM lives in shared memory:
//   geometry (IED -> half patch size, cvRound centre)            adaptive_vlhog.hpp:123,132-133
//   zero-padded crop: ONE TMA tile load per patch (3-D tensor map over the frame batch; out-of-frame
//     bytes are zero-filled by the TMA = copyMakeBorder(BORDER_CONSTANT 0))   adaptive_vlhog.hpp:135-151
//   cv::resize INTER_LINEAR (fixed point), tables precomputed once per face   adaptive_vlhog.hpp:154-155
//   gradient, orientation arg-max from a device-generated table (integer result, bit exact), modulus   hog.c:631-672
//   bilinear spatial vote as two separable passes (rows x cell columns, then cell rows; no atomics)      hog.c:697-724
//   cell energy, 2x2-block normalisation in double, clamp 0.2, for two patches at once    hog.c:875-1053
//   per-dimension transpose + landmark concatenation + bias      adaptive_vlhog.hpp:166-183
//
// Arithmetic that decides an INTEGER result (crop centre, half size, resize taps, orientation bin)
// is written with explicit round-to-nearest intrinsics so that no FMA contraction can change it;
// the reference is built for baseline x86-64 (mul then add).  The only deviation from the
// reference's value stream is the summation ORDER of the float votes inside a cell histogram
// (fixed, deterministic tree here; raster order there): ~1e-7 relative.
#include "sd_internal.cuh"

#include <cuda.h>

#include <cmath>

namespace {

constexpr int kHogThreads = 256;
constexpr int kHogWarps = kHogThreads / 32;
constexpr int kLutDim = 511;                       // gx, gy in [-255, 255]
constexpr int kHogGroup = 11;                      // landmarks per CTA (at most; profiles/r05_hog_face.md)

struct HogArgs {
    const uint8_t* images;
    int width, height, row_stride;
    long long image_stride;
    int image_count;
    const int* image_index;
    const sd_roi* roi;          // optional: only a region of every frame is resident
    const sd_frame* frames;     // optional: frames of different sizes
    uint8_t* roi_miss;
    const float* x;
    long long ldx;
    int N, L;
    int groups, gsz;            // a CTA walks gsz consecutive landmarks of one sample (the last group of a sample may be shorter)
    int pair;                   // 1: S4-S8 run once per pair of consecutive patches (two tail slots in shared memory)
    int variant, nc, cs, K, fs, dd;
    const int* half;            // per sample: half patch size (hog_geometry_kernel)
    const int8_t* lut;          // (gy+255)*511 + (gx+255) -> directed orientation bin, -1 for a zero gradient
    const int* rtab;            // per sample: resize tables [5][fs] (hog_geometry_kernel)
    const float* btab;          // per launch: spatial binning weights [nc][fs], then lo[nc], hi[nc] (hog_bintab_kernel)
    int tma_count;              // number of usable tensor-map size classes (0: the window is staged by load loops)
    float* A;
    long long ld;
    int* geometry;
    uint8_t* patches;
    int8_t* bins;
    int* status;
};

// ---- per-sample geometry: IED -> half patch size (adaptive_vlhog.hpp:123) and the interpolation tables of cv::resize
//      (INTER_LINEAR, 8U, 11-bit fixed point) for a P x P -> fs x fs resize, once per sample instead of once per thread of
//      every one of its L patches.  One CTA per sample.  rtab[sample][0..4][fs]: x source index, x weights (2 x int16),
//      y source index 0 / 1 (clamped), y weights. -------------------------------------------------------------------------
__device__ __forceinline__ int clip_index(int x, int a, int b) { return x >= a ? (x < b ? x : b - 1) : a; }
__device__ __forceinline__ short sat_short(int v) { return (short)(v > 32767 ? 32767 : (v < -32768 ? -32768 : v)); }

__global__ void hog_geometry_kernel(const float* __restrict__ x, long long ldx, int N, int L, const sd_eyes_dev eyes, float rel,
                                    int fixed_half, int fs, int* __restrict__ half_out, int* __restrict__ rtab, int* __restrict__ status)
{
    const int i = blockIdx.x;
    if (i >= N) return;
    __shared__ int s_half;
    if (threadIdx.x == 0) {
        int half = fixed_half;       // > 0: non-adaptive HogTransform of examples/landmark_detection.cpp:213
        if (fixed_half <= 0) {
            const double ied = sd_device_ied(x + (long long)i * ldx, L, eyes);
            half = (int)round(__dmul_rn(__dmul_rn((double)rel, ied), 0.5));   // std::round(float rel * double ied / 2)
            if (half < 1) {          // cv::resize would throw on the empty ROI; flag it and keep going
                half = 1;
                atomicOr(status, 1);
            }
        }
        half_out[i] = half;
        s_half = half;
    }
    __syncthreads();
    const int P = 2 * s_half;
    int* rt = rtab + (long long)i * 5 * fs;
    for (int t = threadIdx.x; t < fs; t += blockDim.x) {
        const double inv_scale = __ddiv_rn((double)fs, (double)P);
        const double scale = __ddiv_rn(1.0, inv_scale);
        float f = (float)__dadd_rn(__dmul_rn((double)t + 0.5, scale), -0.5);
        const int s = (int)floorf(f);
        f = __fsub_rn(f, (float)s);
        int sx = s;
        float fx = f;
        if (sx < 0) { fx = 0.f; sx = 0; }
        if (sx >= P - 1) { fx = 0.f; sx = P - 1; }
        const short2 xa = make_short2(sat_short(__float2int_rn(__fmul_rn(__fsub_rn(1.f, fx), 2048.f))),
                                      sat_short(__float2int_rn(__fmul_rn(fx, 2048.f))));
        const short2 yb = make_short2(sat_short(__float2int_rn(__fmul_rn(__fsub_rn(1.f, f), 2048.f))),
                                      sat_short(__float2int_rn(__fmul_rn(f, 2048.f))));
        rt[t] = sx;
        rt[fs + t] = *reinterpret_cast<const int*>(&xa);
        rt[2 * fs + t] = clip_index(s, 0, P);
        rt[3 * fs + t] = clip_index(s + 1, 0, P);
        rt[4 * fs + t] = *reinterpret_cast<const int*>(&yb);
    }
}

// ---- spatial binning tables of vl_hog_put_image (hog.c:697-709), once per launch: btab[c * fs + t] = weight with which pixel
//      coordinate t votes into cell index c (w1 for its own bin, w2 for the next one, 0 otherwise); then, as ints, the first and
//      last interior coordinate that votes into cell c (same tables for rows and columns: square patch, square cells) ---------
__global__ void hog_bintab_kernel(int fs, int nc, int cs, float* __restrict__ btab)
{
    __shared__ int s_sbin[256];
    for (int t = threadIdx.x; t < fs; t += blockDim.x) {
        const float h = (float)__dadd_rn(__ddiv_rn((double)t + 0.5, (double)cs), -0.5);
        int b = (int)h;                                   // vl_floor_f, hog.h:52-58
        if (!(h >= 0.f || (float)b == h)) b -= 1;
        const float w2 = __fsub_rn(h, (float)b);
        const float w1 = (float)__dadd_rn(1.0, -(double)w2);
        s_sbin[t] = b;
        for (int c = 0; c < nc; ++c) btab[c * fs + t] = (b == c) ? w1 : ((b == c - 1) ? w2 : 0.f);
    }
    __syncthreads();
    int* lohi = reinterpret_cast<int*>(btab + nc * fs);
    for (int c = threadIdx.x; c < nc; c += blockDim.x) {
        int lo = fs, hi = -1;
        for (int t = 1; t <= fs - 2; ++t) {
            const int b = s_sbin[t];
            if (b == c || b == c - 1) { if (t < lo) lo = t; hi = t; }
        }
        lohi[c] = lo;
        lohi[nc + c] = hi;
    }
}

// ---- (gx, gy) -> orientation bin table, generated ON THE DEVICE with the reference's float expression
//      (hog.c:645-672): gradients of an 8-bit patch are integers in [-255, 255], so the arg-max is a pure
//      function of the pair and can be tabulated exactly. ---------------------------------------------
struct LutArgs {
    int K;
    float ox[SD_MAX_BINS], oy[SD_MAX_BINS];
};

__global__ void hog_lut_kernel(const LutArgs t, int8_t* __restrict__ lut)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= kLutDim * kLutDim) return;
    const float gx = (float)(idx % kLutDim - 255), gy = (float)(idx / kLutDim - 255);
    const float g2 = __fadd_rn(__fmul_rn(gx, gx), __fmul_rn(gy, gy));
    int bin = -1;
    if (g2 > 0.f) {
        const float g = __fsqrt_rn(g2);
        // (float)((double)gx / max((double)g, 1e-10)) == gx / g in float: double rounding is innocuous for
        // division when the wide format has >= 2p+2 bits (53 >= 50).
        const float ux = __fdiv_rn(gx, g);
        const float uy = __fdiv_rn(gy, g);
        float best = 0.f;
        for (int k = 0; k < t.K; ++k) {
            float s = __fadd_rn(__fmul_rn(ux, t.ox[k]), __fmul_rn(uy, t.oy[k]));
            int b = k;
            if (s < 0.f) { s = -s; b += t.K; }
            if (s > best) { best = s; bin = b; }   // strict >, ascending k
        }
    }
    lut[idx] = (int8_t)bin;
}

// shared-memory carve-up (same function on host and device)
struct HogSmem {
    int patch, bin, r1, xofs, yofs0, yofs1, xa, yb, wcell, lo, hi, hist, energy, fac, vote, feat, mbar, total;
    int tpad;      // tasks of the horizontal vote pass, padded to a multiple of 32
};

__host__ __device__ inline int align_up(int v, int a) { return (v + a - 1) / a * a; }

// The feature slice is sized for the larger of the two variants' dimension counts (UoCTTI 3K + 4, Dalal-Triggs 4K), so the
// layout is a function of (fs, nc, K) and the number of tail slots (1, or 2 when S4-S8 run for pairs of patches) alone: a
// compile-time constant in the baked schedules.
__host__ __device__ inline HogSmem hog_smem_layout(int fs, int nc, int K, int slots)
{
    HogSmem s;
    const int cells = nc * nc;
    const int dd = 3 * K + 4 > 4 * K ? 3 * K + 4 : 4 * K;
    int o = 0;
    s.patch = o;  o = align_up(o + fs * fs, 128);
    s.bin = o;    o = align_up(o + fs * fs, 16);            // [bin | r1] doubles as the staging area of the source window (128-byte
    s.r1 = o;     o = align_up(o + fs * fs * 4, 16);        //  aligned: TMA destination); r1 = gradient modulus
    s.xofs = o;   o += fs * 4;
    s.yofs0 = o;  o += fs * 4;
    s.yofs1 = o;  o += fs * 4;
    s.xa = o;     o += fs * 4;                              // 2 x int16
    s.yb = o;     o += fs * 4;
    s.wcell = o;  o += nc * fs * 4;                         // weight of pixel t for cell index c (0 if it does not vote)
    s.lo = o;     o += nc * 4;
    s.hi = o;     o += nc * 4;
    s.hist = o;   o += slots * cells * 2 * K * 4;           // hist, energy, fac, feat: one slot per patch of a pair
    s.energy = o; o = align_up(o + slots * cells * 4, 16);
    s.fac = o;    o += slots * cells * 4 * 8;
    s.tpad = align_up((fs - 2) * nc, 32);
    o = align_up(o, 16);
    s.vote = o;   o += 2 * K * s.tpad * 4;                  // horizontal pass of the vote: T[bin][(cell column, row)]
    s.feat = o;   o += slots * cells * dd * 4;
    s.mbar = align_up(o, 8); o = s.mbar + 8;
    s.total = align_up(o, 16);
    return s;
}

// KT / NCT / CST > 0 bake the bin count, cells per side and cell size into the kernel (the schedules the
// reference ships: 5x5 cells of 11/10/8/6 px, K = 4 or 9), which lets the compiler strength-reduce every
// index computation; 0 = taken from the arguments at run time (any other configuration).
// tensor maps of the frame batch (u8, dims {W, H, count}), one per square box size: a patch uses the smallest box that covers
// its P x P source window
constexpr int kTmaClasses = 8;
__host__ __device__ constexpr int hog_tma_box(int c) { return c == 0 ? 32 : c == 1 ? 48 : c == 2 ? 64 : c == 3 ? 80 : c == 4 ? 96 : c == 5 ? 112 : c == 6 ? 128 : 160; }
struct HogMaps { CUtensorMap m[kTmaClasses]; };

// The baked schedules must keep five CTAs resident per SM (<= 51 registers a thread): four measured 21 % slower.  The run-time
// schedules keep the four (<= 64 registers) they had before.
template <int KT, int NCT, int CST>
__global__ void __launch_bounds__(kHogThreads, NCT > 0 ? 5 : 4) hog_patch_kernel(const HogArgs a, const __grid_constant__ HogMaps maps)
{
    extern __shared__ __align__(128) unsigned char smem[];
    const int K = KT > 0 ? KT : a.K;
    const int nc = NCT > 0 ? NCT : a.nc;
    const int fs = (NCT > 0 && CST > 0) ? NCT * CST : a.fs;
    const int dd = a.dd;
    const int cells = nc * nc;
    // both layouts are compile-time constants in the baked schedules
    const HogSmem lay = a.pair ? hog_smem_layout(fs, nc, K, 2) : hog_smem_layout(fs, nc, K, 1);
    uint8_t* s_patch = smem + lay.patch;
    int8_t* s_bin = reinterpret_cast<int8_t*>(smem + lay.bin);
    float* s_gmag = reinterpret_cast<float*>(smem + lay.r1);
    int* s_xofs = reinterpret_cast<int*>(smem + lay.xofs);
    int* s_yofs0 = reinterpret_cast<int*>(smem + lay.yofs0);
    int* s_yofs1 = reinterpret_cast<int*>(smem + lay.yofs1);
    short2* s_xa = reinterpret_cast<short2*>(smem + lay.xa);
    short2* s_yb = reinterpret_cast<short2*>(smem + lay.yb);
    float* s_wcell = reinterpret_cast<float*>(smem + lay.wcell);
    int* s_lo = reinterpret_cast<int*>(smem + lay.lo);
    int* s_hi = reinterpret_cast<int*>(smem + lay.hi);
    float* s_hist = reinterpret_cast<float*>(smem + lay.hist);
    float* s_energy = reinterpret_cast<float*>(smem + lay.energy);
    double* s_fac = reinterpret_cast<double*>(smem + lay.fac);
    float* s_T = reinterpret_cast<float*>(smem + lay.vote);
    float* s_feat = reinterpret_cast<float*>(smem + lay.feat);
    uint64_t* s_mbar = reinterpret_cast<uint64_t*>(smem + lay.mbar);

    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    // this CTA's patches: landmarks [lm_begin, lm_end) of one sample
    const int sample = (int)blockIdx.x / a.groups;
    const int lm_begin = ((int)blockIdx.x - sample * a.groups) * a.gsz;
    const int lm_end = min(lm_begin + a.gsz, a.L);

    // ---- S0: per-sample state, once per CTA: half size from the per-sample pre-pass (adaptive_vlhog.hpp:123), the frame
    //      and the region of it that is resident (the whole frame, or the ROI that sd_detect_batch_host uploaded)
    const float* __restrict__ row = a.x + (long long)sample * a.ldx;
    const int half = __ldg(a.half + sample);
    const int P = 2 * half;
    int img_idx = a.image_index ? a.image_index[sample] : sample;
    if (img_idx < 0 || img_idx >= a.image_count) {
        img_idx = 0;
        if (tid == 0 && a.status) atomicOr(a.status, 2);
    }
    int W = a.width, H = a.height, rs = a.row_stride;
    const uint8_t* __restrict__ img = a.images + (long long)img_idx * a.image_stride;
    if (a.frames) {
        const sd_frame f = a.frames[img_idx];
        W = f.width; H = f.height; rs = f.row_stride;
        img = a.images + f.offset;
    }
    int rx = 0, ry = 0, rw = W, rh = H;
    if (a.roi) {
        const sd_roi r = a.roi[img_idx];
        rx = r.x; ry = r.y; rw = r.w; rh = r.h; rs = r.row_stride;
        img = a.images + r.offset;
    }
    const uint32_t bar = (uint32_t)__cvta_generic_to_shared(s_mbar);
    if (tid == 0 && a.tma_count > 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // tables shared by every patch of the CTA: cv::resize taps of this sample (hog_geometry_kernel), spatial binning weights
    // of this launch (hog_bintab_kernel).  They are visible after the first patch's staging barrier.
    {
        const int* __restrict__ rt = a.rtab + (long long)sample * 5 * fs;
        for (int t = tid; t < fs; t += kHogThreads) {
            s_xofs[t] = __ldg(rt + t);
            const int xa = __ldg(rt + fs + t), yb = __ldg(rt + 4 * fs + t);
            s_xa[t] = *reinterpret_cast<const short2*>(&xa);
            s_yofs0[t] = __ldg(rt + 2 * fs + t);
            s_yofs1[t] = __ldg(rt + 3 * fs + t);
            s_yb[t] = *reinterpret_cast<const short2*>(&yb);
        }
        for (int i = tid; i < nc * fs; i += kHogThreads) s_wcell[i] = __ldg(a.btab + i);
        const int* __restrict__ lohi = reinterpret_cast<const int*>(a.btab + nc * fs);
        if (tid < nc) { s_lo[tid] = __ldg(lohi + tid); s_hi[tid] = __ldg(lohi + nc + tid); }
    }
    uint8_t* s_stage = smem + lay.bin;                                 // [bin | r1]: dead between S8 and the next S2
    const int stage_cap = lay.xofs - lay.bin;
    uint32_t tma_phase = 0;                                            // parity of the mbarrier phase the next TMA completes

    // Shared-memory regions live in each phase of one patch (the loop's barriers separate consecutive patches):
    //   S1  stage = [bin | r1] (window), patch (written), tables, T (zeroed)
    //   S2  patch (read), bin + gmag (r1) written
    //   S3  bin, gmag, tables, T -> hist
    //   S4-S7  hist, energy, fac, feat (once per pair of patches)
    //   S8  feat
    for (int lm = lm_begin; lm < lm_end; ++lm) {
        const int slot = a.pair ? (lm - lm_begin) & 1 : 0;             // hist / feat slot of this patch in its pair
        const int patch_id = sample * a.L + lm;                        // < 2^31: launch_hog checks N * L
        const int cx = __float2int_rn(row[lm]);                        // centre = cvRound (adaptive_vlhog.hpp:132-133)
        const int cy = __float2int_rn(row[lm + a.L]);
        if (tid == 0 && a.geometry) {
            a.geometry[patch_id * 3 + 0] = cx;
            a.geometry[patch_id * 3 + 1] = cy;
            a.geometry[patch_id * 3 + 2] = half;
        }

        // ---- S1: zero-padded crop + fixed-point bilinear resize.  The P x P source window is staged in shared memory with
        //      its zero padding materialised, then resampled from there: one output row per warp pass, lanes along x.
        const int x0 = cx - half, y0 = cy - half;
        // TMA route: whole frames resident and describable by a tensor map; the smallest box class that covers the window and
        // fits the staging area
        int tma_box = 0;
        // The TMA wants the box to start on a 16-byte boundary of the innermost dimension (an unaligned start faults with
        // "illegal instruction"): the box starts at x0 rounded down to a multiple of 16 and the window sits tma_shift bytes
        // into its rows.
        const int tma_shift = x0 & 15;
#pragma unroll
        for (int c = kTmaClasses - 1; c >= 0; --c)
            if (c < a.tma_count && hog_tma_box(c) >= P + tma_shift && hog_tma_box(c) * hog_tma_box(c) <= stage_cap) tma_box = hog_tma_box(c);
        if (tma_box > 0 && tid == 0) {
            // one elected thread: the box lands densely (pitch = box width); bytes outside the frame are zero-filled by the
            // TMA, which is exactly copyMakeBorder(..., BORDER_CONSTANT, 0) (adaptive_vlhog.hpp:136-147).  The previous
            // patch's generic-proxy writes to the staging area were fenced before the barrier that ended it.
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(tma_box * tma_box) : "memory");
            int cls = 0;
#pragma unroll
            for (int c = 0; c < kTmaClasses; ++c) if (hog_tma_box(c) == tma_box) cls = c;
            asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                         ::"r"((uint32_t)__cvta_generic_to_shared(s_stage)), "l"(&maps.m[cls]), "r"(bar), "r"(x0 - tma_shift), "r"(y0), "r"(img_idx)
                         : "memory");
        }
        {
            float4* T4 = reinterpret_cast<float4*>(s_T);
            for (int i = tid; i < K * lay.tpad / 2; i += kHogThreads) T4[i] = make_float4(0.f, 0.f, 0.f, 0.f);     // 2K * tpad floats
        }
        {
            const bool resident = x0 >= rx && y0 >= ry && x0 + P <= rx + rw && y0 + P <= ry + rh && x0 >= 0 && y0 >= 0 && x0 + P <= W && y0 + P <= H;
            const uintptr_t align_bits = reinterpret_cast<uintptr_t>(img) | (uintptr_t)rs;
            const bool vec16 = !tma_box && resident && (align_bits & 15) == 0;      // rows can be fetched as aligned 16-byte vectors
            const bool words = !tma_box && resident && (align_bits & 3) == 0;
            // column c of the staged window sits at byte shiftb + c of its row
            const int shiftb = tma_box ? tma_shift : (vec16 ? ((x0 - rx) & 15) : (words ? ((x0 - rx) & 3) : 0));
            const int pitch = tma_box ? tma_box : ((P + 15 + 15) & ~15);
            const bool staged = pitch * P <= stage_cap;
            bool miss = false;
            if (staged) {
                if (tma_box) {
                    // nothing to do: the tile is in flight
                } else if (vec16) {
                    // 8 / 16 / 32 lanes per source row, one aligned uint4 each: ~P * nvec / 32 warp loads in total
                    const int nvec = (shiftb + P + 15) >> 4;
                    const int gs = nvec <= 8 ? 3 : (nvec <= 16 ? 4 : 5);
                    const int lv = lane & ((1 << gs) - 1), lr = lane >> gs, rows_per_pass = 32 >> gs;
                    const uint8_t* wrow = img + (long long)(y0 - ry) * rs + (x0 - rx - shiftb);
                    for (int r = warp * rows_per_pass + lr; r < P; r += kHogWarps * rows_per_pass)
                        for (int v = lv; v < nvec; v += (1 << gs))
                            reinterpret_cast<uint4*>(s_stage + r * pitch)[v] = __ldg(reinterpret_cast<const uint4*>(wrow + (long long)r * rs) + v);
                } else if (words) {
                    const int nwords = (shiftb + P + 3) >> 2;
                    const uint8_t* wrow = img + (long long)(y0 - ry) * rs + (x0 - rx - shiftb);
                    for (int r = warp; r < P; r += kHogWarps) {
                        const uint32_t* src = reinterpret_cast<const uint32_t*>(wrow + (long long)r * rs);
                        uint32_t* dst = reinterpret_cast<uint32_t*>(s_stage + r * pitch);
                        for (int w = lane; w < nwords; w += 32) dst[w] = __ldg(src + w);
                    }
                } else {
                    for (int r = warp; r < P; r += kHogWarps) {
                        const int iy = y0 + r;
                        const bool rowin = (unsigned)iy < (unsigned)H;
                        const bool rowres = iy >= ry && iy < ry + rh;
                        for (int c = lane; c < P; c += 32) {
                            const int ix = x0 + c;
                            int v = 0;
                            if (rowin && (unsigned)ix < (unsigned)W) {
                                if (rowres && ix >= rx && ix < rx + rw) v = __ldg(img + (long long)(iy - ry) * rs + (ix - rx));
                                else miss = true;                      // a frame pixel that was not uploaded
                            }
                            s_stage[r * pitch + c] = (uint8_t)v;
                        }
                    }
                }
                __syncthreads();                                       // tables (and the load loops' stores) visible
                if (tma_box) {
                    uint32_t ok = 0;
                    const long long t0 = clock64();
                    while (!ok) {                                      // bounded: a protocol bug must trap, never hang the GPU
                        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                                     : "=r"(ok) : "r"(bar), "r"(tma_phase) : "memory");
                        if (!ok && clock64() - t0 > 4000000000LL) __trap();
                    }
                    tma_phase ^= 1;
                }
                if (fs <= 64) {
                    // a thread keeps ONE output column (its two source taps and weights stay in registers) and walks down the rows
                    const int dx = tid & 63, g = tid >> 6;
                    if (dx < fs) {
                        const int sx = s_xofs[dx];
                        const int sx1 = min(sx + 1, P - 1);            // clamped tap has zero weight
                        const int ax = s_xa[dx].x, bx = s_xa[dx].y;
                        const uint8_t* base = s_stage + shiftb;
#pragma unroll 4
                        for (int dy = g; dy < fs; dy += kHogThreads / 64) {
                            const short2 yb = s_yb[dy];
                            const uint8_t* r0 = base + s_yofs0[dy] * pitch;
                            const uint8_t* r1 = base + s_yofs1[dy] * pitch;
                            const int t0 = (int)r0[sx] * ax + (int)r0[sx1] * bx;
                            const int t1 = (int)r1[sx] * ax + (int)r1[sx1] * bx;
                            const int v = ((((int)yb.x * (t0 >> 4)) >> 16) + (((int)yb.y * (t1 >> 4)) >> 16) + 2) >> 2;
                            s_patch[dy * fs + dx] = (uint8_t)v;        // s_patch precedes the staging area: no overlap
                        }
                    }
                } else {
                    for (int dy = warp; dy < fs; dy += kHogWarps) {
                        const short2 yb = s_yb[dy];
                        const uint8_t* r0 = s_stage + s_yofs0[dy] * pitch + shiftb;
                        const uint8_t* r1 = s_stage + s_yofs1[dy] * pitch + shiftb;
                        for (int dx = lane; dx < fs; dx += 32) {
                            const int sx = s_xofs[dx];
                            const int sx1 = min(sx + 1, P - 1);
                            const short2 xa = s_xa[dx];
                            const int t0 = (int)r0[sx] * xa.x + (int)r0[sx1] * xa.y;
                            const int t1 = (int)r1[sx] * xa.x + (int)r1[sx1] * xa.y;
                            const int v = ((((int)yb.x * (t0 >> 4)) >> 16) + (((int)yb.y * (t1 >> 4)) >> 16) + 2) >> 2;
                            s_patch[dy * fs + dx] = (uint8_t)v;
                        }
                    }
                }
            } else {
                // window too large for the staging area: sample straight from global memory with full checks
                __syncthreads();                                       // tables visible
                for (int dy = warp; dy < fs; dy += kHogWarps) {
                    const short2 yb = s_yb[dy];
                    const int iy0 = y0 + s_yofs0[dy], iy1 = y0 + s_yofs1[dy];
                    for (int dx = lane; dx < fs; dx += 32) {
                        const int sx = s_xofs[dx];
                        const short2 xa = s_xa[dx];
                        int p[4];
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int ix = x0 + sx + (q & 1), iy = (q & 2) ? iy1 : iy0;
                            int v = 0;
                            if ((q & 1) && xa.y == 0) { p[q] = 0; continue; }
                            if ((unsigned)ix < (unsigned)W && (unsigned)iy < (unsigned)H) {
                                if (ix >= rx && ix < rx + rw && iy >= ry && iy < ry + rh) v = __ldg(img + (long long)(iy - ry) * rs + (ix - rx));
                                else miss = true;
                            }
                            p[q] = v;
                        }
                        const int t0 = p[0] * xa.x + p[1] * xa.y;
                        const int t1 = p[2] * xa.x + p[3] * xa.y;
                        const int v = ((((int)yb.x * (t0 >> 4)) >> 16) + (((int)yb.y * (t1 >> 4)) >> 16) + 2) >> 2;
                        s_patch[dy * fs + dx] = (uint8_t)v;
                    }
                }
            }
            if (miss && a.roi_miss) a.roi_miss[img_idx] = 1;
            if (a.patches) {
                __syncthreads();
                for (int i = tid; i < fs * fs; i += kHogThreads) a.patches[(long long)patch_id * fs * fs + i] = s_patch[i];
            }
        }
        __syncthreads();

        // ---- S2: gradient + orientation arg-max per interior pixel (hog.c:631-672): the arg-max comes from the
        //      device-generated table (the gradient of an 8-bit patch is a pair of integers in [-255, 255]); the modulus is
        //      sqrtf of the exactly representable integer gx*gx + gy*gy (hog.c:645), computed in registers
        {
            // linear index over the interior pixels (all lanes busy); four pixels per thread in flight so that the four table
            // look-ups overlap (the phase was bound by their latency: profiles/r02_summary.md)
            const int iw = fs - 2, npix = iw * iw;
            for (int i0 = tid; i0 < npix; i0 += 4 * kHogThreads) {
                int idx[4], gxs[4], gys[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int i = i0 + k * kHogThreads;
                    const int y = i / iw, x = i - y * iw;
                    idx[k] = (y + 1) * fs + (x + 1);
                    if (i < npix) {
                        gxs[k] = (int)s_patch[idx[k] + 1] - (int)s_patch[idx[k] - 1];
                        gys[k] = (int)s_patch[idx[k] + fs] - (int)s_patch[idx[k] - fs];
                    } else { gxs[k] = 0; gys[k] = 0; }
                }
                int8_t bn[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) bn[k] = __ldg(a.lut + (gys[k] + 255) * kLutDim + (gxs[k] + 255));
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (i0 + k * kHogThreads < npix) {
                        s_bin[idx[k]] = bn[k];
                        s_gmag[idx[k]] = __fsqrt_rn((float)(gxs[k] * gxs[k] + gys[k] * gys[k]));
                    }
            }
        }
        if (a.bins) {
            __syncthreads();
            for (int idx = tid; idx < fs * fs; idx += kHogThreads) {
                const int y = idx / fs, x = idx - y * fs;
                const bool interior = x >= 1 && x <= fs - 2 && y >= 1 && y <= fs - 2;
                a.bins[(long long)patch_id * fs * fs + idx] = interior ? s_bin[idx] : (int8_t)-1;
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // bin / gmag writes before the next patch's TMA
        __syncthreads();

        // ---- S3: bilinear spatial vote (hog.c:697-724), separable:  hist[b][cj][ci] = sum_y wy[cj][y] * ( sum_x wx[ci][x] * g[y][x] * [bin[y][x] == b] ).
        //      Pass 1: one thread per (cell column ci, interior row y) walks the <= 2*cs pixels of that row that vote into ci and adds
        //      g * wx into ITS OWN column of T[bin][task] (bank == task mod 32: conflict free, no atomics, fixed order).
        //      Pass 2: one thread per (bin, cell) folds the rows with wy.  The reference adds (g * wx) * wy per pixel in raster
        //      order; this is the same sum associated differently (~1e-7 relative), deterministic.
        {
            const int nrow = fs - 2, ntask = nrow * nc, tpad = lay.tpad;
            for (int task = tid; task < ntask; task += kHogThreads) {
                const int ci = task / nrow, y = 1 + task - ci * nrow;
                const int xlo = s_lo[ci], xhi = s_hi[ci];
                const int8_t* bp = s_bin + y * fs + xlo;
                const float* gp = s_gmag + y * fs + xlo;
                const float* wp = s_wcell + ci * fs + xlo;
                float* T = s_T + task;
#pragma unroll 2
                for (int x = xlo; x <= xhi; ++x) {
                    const int b = max((int)*bp++, 0);                     // zero gradient: bin -1, modulus 0 -> adds +0 to bin 0
                    float* q = T + b * tpad;
                    *q = __fadd_rn(*q, __fmul_rn(*gp++, *wp++));
                }
            }
            __syncthreads();
            for (int i = tid; i < 2 * K * cells; i += kHogThreads) {
                const int b = i / cells, c = i - b * cells;
                const int cj = c / nc, ci = c - cj * nc;                  // cell row (y), cell column (x)
                const int ylo = s_lo[cj], yhi = s_hi[cj];
                const float* Tp = s_T + b * tpad + ci * nrow + (ylo - 1);
                const float* wy = s_wcell + cj * fs + ylo;
                float acc = 0.f;
                for (int y = ylo; y <= yhi; ++y) acc = __fadd_rn(acc, __fmul_rn(*Tp++, *wy++));
                s_hist[slot * 2 * K * cells + b * cells + c] = acc;
            }
        }
        __syncthreads();

        // ---- S4-S8 run once per pair of consecutive patches (or for the last patch alone): twice the threads per phase, half
        //      the barriers per patch.  Slot p of the pair is patch lm_first + p.
        if (slot == 1 || lm + 1 == lm_end || !a.pair) {
            const int npair = slot + 1, lm_first = lm - slot;

            // ---- S4: undirected cell energy (hog.c:875-890) -------------------------------------------
            for (int i = tid; i < npair * cells; i += kHogThreads) {
                const int p = i >= cells ? 1 : 0, c = i - p * cells;
                const float* hist = s_hist + p * 2 * K * cells;
                float e = 0.f;
                for (int k = 0; k < K; ++k) {
                    const float h = __fadd_rn(hist[k * cells + c], hist[(k + K) * cells + c]);
                    e = __fadd_rn(e, __fmul_rn(h, h));
                }
                s_energy[i] = e;
            }
            __syncthreads();

            // ---- S5: the four block factors of each cell, in double (hog.c:930-982) ------------------
            for (int i = tid; i < npair * cells * 4; i += kHogThreads) {
                const int p = i >= cells * 4 ? 1 : 0, ii = i - p * cells * 4;
                const int c = ii >> 2, f = ii & 3;
                const int y = c / nc, x = c - y * nc;
                const int xm = max(x - 1, 0), xp = min(x + 1, nc - 1);
                const int ym = max(y - 1, 0), yp = min(y + 1, nc - 1);
                // factor1: n1+n2+n4+n5, factor2: n2+n3+n5+n6, factor3: n4+n5+n7+n8, factor4: n5+n6+n8+n9
                const int xa = (f & 1) ? x : xm, xb = (f & 1) ? xp : x;
                const int ya = (f & 2) ? y : ym, yb = (f & 2) ? yp : y;
                const float* energy = s_energy + p * cells;
                double e = (double)energy[xa + ya * nc];
                e = __dadd_rn(e, (double)energy[xb + ya * nc]);
                e = __dadd_rn(e, (double)energy[xa + yb * nc]);
                e = __dadd_rn(e, (double)energy[xb + yb * nc]);
                e = __dadd_rn(e, 1e-4);
                s_fac[i] = __ddiv_rn(1.0, sqrt(e));
            }
            __syncthreads();

            // ---- S6: normalise, clamp at 0.2, project (hog.c:985-1044) ------------------------------
            for (int i = tid; i < npair * cells * K; i += kHogThreads) {
                const int p = i >= cells * K ? 1 : 0, ii = i - p * cells * K;
                const int k = ii / cells, c = ii - k * cells;
                const int cj = c / nc, ci = c - cj * nc;
                const int oc = ci * nc + cj;                        // per-dimension transpose, adaptive_vlhog.hpp:168-174
                const float* hist = s_hist + p * 2 * K * cells;
                const double* fac4 = s_fac + p * cells * 4 + c * 4;
                float* feat = s_feat + p * cells * dd;
                const double ha = (double)hist[k * cells + c];
                const double hb = (double)hist[(k + K) * cells + c];
                double sa = 0.0, sb = 0.0, sc = 0.0;
                double hcv[4];
#pragma unroll
                for (int f = 0; f < 4; ++f) {
                    const double fac = fac4[f];
                    double haf = __dmul_rn(fac, ha);
                    double hbf = __dmul_rn(fac, hb);
                    double hcf = __dadd_rn(haf, hbf);
                    haf = (0.2 < haf) ? 0.2 : haf;
                    hbf = (0.2 < hbf) ? 0.2 : hbf;
                    hcf = (0.2 < hcf) ? 0.2 : hcf;
                    hcv[f] = hcf;
                    sa = (f == 0) ? haf : __dadd_rn(sa, haf);
                    sb = (f == 0) ? hbf : __dadd_rn(sb, hbf);
                    sc = (f == 0) ? hcf : __dadd_rn(sc, hcf);
                }
                if (a.variant == 1) {                               // UoCTTI
                    feat[k * cells + oc] = (float)__dmul_rn(0.5, sa);
                    feat[(k + K) * cells + oc] = (float)__dmul_rn(0.5, sb);
                    feat[(k + 2 * K) * cells + oc] = (float)__dmul_rn(0.5, sc);
                } else {                                            // Dalal-Triggs
#pragma unroll
                    for (int f = 0; f < 4; ++f) feat[(k + f * K) * cells + oc] = (float)hcv[f];
                }
            }

            // ---- S7: texture dims = 1/sqrt(18) * sum_k hc_f, summed in ascending k (hog.c:1046-1053).  A thread recomputes the
            //      clamped hc_f of its cell from hist and fac with S6's operations (same bits), so S7 needs no barrier after S6.
            if (a.variant == 1) {
                for (int i = tid; i < npair * cells * 4; i += kHogThreads) {
                    const int p = i >= cells * 4 ? 1 : 0, ii = i - p * cells * 4;
                    const int c = ii >> 2, f = ii & 3;
                    const int cj = c / nc, ci = c - cj * nc;
                    const float* hist = s_hist + p * 2 * K * cells;
                    const double fac = s_fac[i];
                    double t = 0.0;
                    for (int k = 0; k < K; ++k) {
                        const double hcf = __dadd_rn(__dmul_rn(fac, (double)hist[k * cells + c]), __dmul_rn(fac, (double)hist[(k + K) * cells + c]));
                        t = __dadd_rn(t, (0.2 < hcf) ? 0.2 : hcf);
                    }
                    const float c18 = __fdiv_rn(1.0f, __fsqrt_rn(18.0f));
                    s_feat[p * cells * dd + (3 * K + f) * cells + ci * nc + cj] = (float)__dmul_rn((double)c18, t);
                }
            }
            __syncthreads();

            // ---- S8: coalesced write of the pair's slices of the feature row (consecutive landmarks are adjacent) ----------
            if (a.A) {
                const int per_lm = cells * dd;
                float* __restrict__ out = a.A + (long long)sample * a.ld + (long long)lm_first * per_lm;
                for (int i = tid; i < npair * per_lm; i += kHogThreads) out[i] = s_feat[i];
                if (lm_first == 0 && tid == 0) a.A[(long long)sample * a.ld + (long long)a.L * per_lm] = 1.0f;   // bias, :182-183
            }
        }
    }
}

typedef CUresult (*PFN_hogEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                       const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                       CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_hogEncodeTiled hog_encode_fn()
{
    static PFN_hogEncodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_hogEncodeTiled>(p);
    }
    return fn;
}

int launch_hog(sd_ctx* ctx, const sd_image_batch* images, const int32_t* d_image_index, const float* d_x,
               int64_t ldx, int N, int L, const sd_normalisation* eyes, const sd_hog_param* p, float* d_A,
               int64_t ld, int32_t* d_geometry, uint8_t* d_patches, int8_t* d_bins)
{
    SD_REQUIRE(ctx, images && images->d_data && d_x && p, "null argument");
    SD_REQUIRE(ctx, N >= 0 && L >= 1, "bad sample / landmark count");
    SD_REQUIRE(ctx, p->variant == 0 || p->variant == 1, "unknown HOG variant");
    SD_REQUIRE(ctx, p->num_bins >= 1 && p->num_bins <= SD_MAX_BINS, "num_bins must be in [1,16]");
    SD_REQUIRE(ctx, p->num_cells >= 1 && p->cell_size >= 1, "bad cell configuration");
    const int fs = p->num_cells * p->cell_size;
    SD_REQUIRE(ctx, fs > 3 && fs <= 256, "resized patch must be 4..256 px (hog.c:545-546 asserts > 3)");
    SD_REQUIRE(ctx, (fs + p->cell_size / 2) / p->cell_size == p->num_cells, "hogWidth != num_cells");
    SD_REQUIRE(ctx, ldx >= 2 * L, "ldx < 2L");
    if (N == 0) return SD_OK;
    // eyes == NULL (or kind 0): the fixed-patch HogTransform of the hello-world example (examples/landmark_detection.cpp:
    // 195-261): half = num_cells * (cell_size / 2), no resize.  The kernel's resize stage is the identity when the patch is
    // already num_cells * cell_size wide, which holds for even cell sizes; an odd cell size would change the HOG grid of
    // the un-resized patch and is rejected.
    const bool fixed = !eyes || eyes->kind == 0;
    int fixed_half = 0;
    if (fixed) {
        fixed_half = p->num_cells * (p->cell_size / 2);
        SD_REQUIRE(ctx, 2 * fixed_half == fs, "the fixed-patch HogTransform needs an even cell_size (patch == num_cells * cell_size)");
    } else if (eyes->kind != 1) {
        return sd_fail(ctx, SD_ERR_INVALID, "unknown normalisation kind");
    }

    HogArgs a;
    sd_eyes_dev eyes_dev;
    memset(&eyes_dev, 0, sizeof(eyes_dev));
    int rc = fixed ? SD_OK : sd_eyes_to_dev(ctx, eyes, L, &eyes_dev);
    if (rc) return rc;
    a.images = images->d_data;
    a.width = images->width; a.height = images->height; a.row_stride = images->row_stride;
    a.image_stride = images->image_stride; a.image_count = images->count;
    a.image_index = d_image_index;
    a.roi = images->d_roi;
    a.roi_miss = images->d_roi_miss;
    a.frames = images->d_frames;
    if (!d_image_index) SD_REQUIRE(ctx, images->count >= N, "fewer images than samples and no image index");
    a.x = d_x; a.ldx = ldx; a.N = N; a.L = L;
    a.variant = p->variant; a.nc = p->num_cells; a.cs = p->cell_size; a.K = p->num_bins; a.fs = fs;
    a.dd = p->variant == 1 ? 3 * p->num_bins + 4 : 4 * p->num_bins;
    a.A = d_A; a.ld = ld;
    if (d_A) SD_REQUIRE(ctx, ld >= (int64_t)L * a.nc * a.nc * a.dd + 1, "ld < feature length");
    a.geometry = d_geometry; a.patches = d_patches; a.bins = d_bins;
    a.status = reinterpret_cast<int*>(ctx->d_scratch) + 1;   // the projection's own status word: bit 0 empty patch, bit 1 bad image index

    // orientation table for this K, built once per context (hog.c:195-204: host libm cos/sin, as the reference)
    if (!ctx->hog_lut[a.K]) {
        LutArgs t;
        t.K = a.K;
        for (int k = 0; k < SD_MAX_BINS; ++k) { t.ox[k] = 0.f; t.oy[k] = 0.f; }
        for (int k = 0; k < a.K; ++k) {
            const double angle = k * 3.141592653589793 / a.K;
            t.ox[k] = (float)cos(angle);
            t.oy[k] = (float)sin(angle);
        }
        void* lut = nullptr;
        SD_CUDA(ctx, cudaMalloc(&lut, (size_t)kLutDim * kLutDim));
        hog_lut_kernel<<<sd_div_up(kLutDim * kLutDim, 256), 256, 0, ctx->stream>>>(t, (int8_t*)lut);
        SD_LAUNCH_CHECK(ctx, "hog_lut_kernel");
        ctx->hog_lut[a.K] = lut;
    }
    a.lut = (const int8_t*)ctx->hog_lut[a.K];

    // per-sample tables (half size, cv::resize taps) and the per-launch spatial binning table
    const size_t geom_bytes = (size_t)N * sizeof(int) + (size_t)N * 5 * fs * sizeof(int) + (size_t)(a.nc * fs + 2 * a.nc) * sizeof(float);
    int* d_half = (int*)sd_workspace(ctx, SD_WS_GEOM, geom_bytes);
    if (!d_half) return SD_ERR_CUDA;
    int* d_rtab = d_half + N;
    float* d_btab = reinterpret_cast<float*>(d_rtab + (size_t)N * 5 * fs);
    hog_geometry_kernel<<<N, 64, 0, ctx->stream>>>(d_x, ldx, N, L, eyes_dev, p->relative_patch_size, fixed_half, fs, d_half, d_rtab, a.status);
    SD_LAUNCH_CHECK(ctx, "hog_geometry_kernel");
    hog_bintab_kernel<<<1, 256, 0, ctx->stream>>>(fs, a.nc, a.cs, d_btab);
    SD_LAUNCH_CHECK(ctx, "hog_bintab_kernel");
    a.half = d_half;
    a.rtab = d_rtab;
    a.btab = d_btab;

    // tensor maps of the frame batch for the TMA staging route: whole frames resident, 16-byte aligned base and pitches
    HogMaps maps;
    memset(&maps, 0, sizeof(maps));
    a.tma_count = 0;
    if (!images->d_roi && !images->d_frames && (reinterpret_cast<uintptr_t>(images->d_data) & 15) == 0 && (images->row_stride % 16) == 0 &&
        (images->image_stride % 16) == 0 && (images->count == 1 || images->image_stride > 0)) {
        PFN_hogEncodeTiled enc = hog_encode_fn();
        if (enc) {
            bool ok = true;
            for (int c = 0; c < kTmaClasses && ok; ++c) {
                if (hog_tma_box(c) > 256) break;
                cuuint64_t gdim[3] = {(cuuint64_t)images->width, (cuuint64_t)images->height, (cuuint64_t)images->count};
                cuuint64_t gstride[2] = {(cuuint64_t)images->row_stride, (cuuint64_t)(images->count > 1 ? images->image_stride : (int64_t)images->row_stride * images->height)};
                if (gstride[1] % 16) gstride[1] = (gstride[1] + 15) / 16 * 16;
                cuuint32_t box[3] = {(cuuint32_t)hog_tma_box(c), (cuuint32_t)hog_tma_box(c), 1};
                cuuint32_t estr[3] = {1, 1, 1};
                ok = enc(&maps.m[c], CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<uint8_t*>(images->d_data), gdim, gstride, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
                if (ok) a.tma_count = c + 1;               // classes are usable up to the first one the driver refuses
            }
        }
    }

    const HogSmem lay1 = hog_smem_layout(fs, a.nc, a.K, 1), lay2 = hog_smem_layout(fs, a.nc, a.K, 2);
    SD_REQUIRE(ctx, lay1.total <= 227 * 1024, "HOG configuration needs more than 227 KB of shared memory");
    SD_REQUIRE(ctx, (long long)N * L < 2147483647LL, "too many patches for one launch");
    // A CTA walks the patches of kHogGroup consecutive landmarks of one sample and pays the per-sample work (image and ROI
    // look-up, resize taps, binning weights, mbarrier set-up) once for all of them.  The landmarks of a sample are split
    // into groups of equal size up to one.
    a.groups = sd_div_up(L, kHogGroup);
    a.gsz = sd_div_up(L, a.groups);
    const long long blocks = (long long)N * a.groups;
    auto kern = hog_patch_kernel<0, 0, 0>;
    if (a.K == 4) kern = hog_patch_kernel<4, 0, 0>;
    else if (a.K == 9) kern = hog_patch_kernel<9, 0, 0>;
    if (a.nc == 5 && (a.K == 4 || a.K == 9)) {
#define SD_HOG_PICK(KK, CC) if (a.K == KK && a.cs == CC) kern = hog_patch_kernel<KK, 5, CC>;
        SD_HOG_PICK(4, 11) SD_HOG_PICK(4, 10) SD_HOG_PICK(4, 8) SD_HOG_PICK(4, 6)
        SD_HOG_PICK(9, 11) SD_HOG_PICK(9, 10) SD_HOG_PICK(9, 8) SD_HOG_PICK(9, 6)
#undef SD_HOG_PICK
    }
    // Pairs of patches share the tail unless the second slot costs resident CTAs (with K = 9 at cs = 10 it would take the
    // kernel from five to four CTAs per SM).
    a.pair = 0;
    if (lay2.total <= 227 * 1024) {
        int occ1 = 0, occ2 = 0;
        SD_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, lay2.total));
        SD_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ1, kern, kHogThreads, lay1.total));
        SD_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ2, kern, kHogThreads, lay2.total));
        a.pair = occ2 >= occ1 ? 1 : 0;
    }
    const HogSmem lay = a.pair ? lay2 : lay1;
    SD_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, lay.total));
    // (Measured, profiles/r02_summary.md: forcing six resident CTAs per SM with the whole shared-memory carve-out is SLOWER than
    // five with the default split -- the orientation table lives in L1, which the larger carve-out takes away.)
    kern<<<(unsigned)blocks, kHogThreads, lay.total, ctx->stream>>>(a, maps);
    SD_LAUNCH_CHECK(ctx, "hog_patch_kernel");
    return SD_OK;
}

}  // namespace

namespace {
// cv::cvtColor(BGR2GRAY), 8-bit, OpenCV >= 3 fixed point (15-bit coefficients): HBM-bound, 3 bytes read + 1 written per
// pixel.  A thread converts four pixels: three aligned 32-bit loads, one 32-bit store (scalar path for the row tail or
// unaligned rows).  Frame j of the launch is jobs[j] (frames of any sizes, e.g. the colour frames of one staging chunk), or
// with jobs == NULL `uniform` shifted by j image strides.  blockIdx.y strides over the frames, blockIdx.x over one frame.
__global__ void bgr2gray_kernel(const uint8_t* __restrict__ bgr, uint8_t* __restrict__ gray, sd_bgr2gray_job uniform,
                                long long simg, long long dimg, const sd_bgr2gray_job* __restrict__ jobs, int count)
{
    for (int j = blockIdx.y; j < count; j += gridDim.y) {
        const sd_bgr2gray_job job = jobs ? jobs[j] : uniform;
        const uint8_t* sbase = bgr + job.src_offset + (jobs ? 0 : j * simg);
        uint8_t* dbase = gray + job.dst_offset + (jobs ? 0 : j * dimg);
        const int width = job.width;
        const long long srow = job.src_row_stride, drow = job.dst_row_stride;
        const bool vec_ok = ((reinterpret_cast<uintptr_t>(sbase) | reinterpret_cast<uintptr_t>(dbase) | (uintptr_t)srow | (uintptr_t)drow) & 3) == 0;
        const int groups = (width + 3) >> 2;
        const long long total = (long long)job.height * groups;
        for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
            const int g = (int)(t % groups);
            const int y = (int)(t / groups);
            const uint8_t* s = sbase + (long long)y * srow + 12 * g;
            uint8_t* d = dbase + (long long)y * drow + 4 * g;
            const int x0 = 4 * g;
            if (vec_ok && x0 + 4 <= width) {
                const uint32_t w0 = *reinterpret_cast<const uint32_t*>(s), w1 = *reinterpret_cast<const uint32_t*>(s + 4),
                               w2 = *reinterpret_cast<const uint32_t*>(s + 8);
                // bytes: w0 = B0 G0 R0 B1 | w1 = G1 R1 B2 G2 | w2 = R2 B3 G3 R3   (little endian)
                *reinterpret_cast<uint32_t*>(d) = sd_bgr2gray_px(w0 & 255, (w0 >> 8) & 255, (w0 >> 16) & 255) |
                                                  (sd_bgr2gray_px(w0 >> 24, w1 & 255, (w1 >> 8) & 255) << 8) |
                                                  (sd_bgr2gray_px((w1 >> 16) & 255, w1 >> 24, w2 & 255) << 16) |
                                                  (sd_bgr2gray_px((w2 >> 8) & 255, (w2 >> 16) & 255, w2 >> 24) << 24);
            } else {
                for (int k = 0; k < 4 && x0 + k < width; ++k) d[k] = (uint8_t)sd_bgr2gray_px(s[3 * k], s[3 * k + 1], s[3 * k + 2]);
            }
        }
    }
}
}  // namespace

int sd_bgr2gray_launch(sd_ctx* ctx, cudaStream_t stream, const uint8_t* d_bgr, uint8_t* d_gray, const sd_bgr2gray_job& uniform,
                       int64_t bgr_image_stride, int64_t gray_image_stride, const sd_bgr2gray_job* d_jobs, int count,
                       int64_t max_groups)
{
    if (count <= 0) return SD_OK;
    // about 16 CTAs per SM in all: one row of the grid per frame while there are fewer frames than that
    const int64_t want = 16LL * ctx->sm_count;
    const int gy = (int)(count < 65535 ? count : 65535);
    int64_t gx = sd_div_up(max_groups, 256);
    const int64_t share = sd_div_up(want, gy);
    gx = gx < share ? gx : share;
    gx = gx < 1 ? 1 : gx;
    bgr2gray_kernel<<<dim3((unsigned)gx, (unsigned)gy), 256, 0, stream>>>(d_bgr, d_gray, uniform, bgr_image_stride, gray_image_stride,
                                                                          d_jobs, count);
    SD_LAUNCH_CHECK(ctx, "bgr2gray_kernel");
    return SD_OK;
}

extern "C" {

int sd_hog_feature_length(int num_landmarks, const sd_hog_param* p)
{
    if (!p) return -1;
    const int dd = p->variant == 1 ? 3 * p->num_bins + 4 : 4 * p->num_bins;
    return num_landmarks * p->num_cells * p->num_cells * dd + 1;
}

int sd_hog_batch(sd_ctx* ctx, const sd_image_batch* images, const int32_t* d_image_index, const float* d_x,
                 int64_t ldx, int num_samples, int num_landmarks, const sd_normalisation* eyes,
                 const sd_hog_param* p, float* d_A, int64_t ld)
{
    if (!ctx) return SD_ERR_INVALID;
    if (num_samples == 0) return SD_OK;
    SD_REQUIRE(ctx, d_A, "null output");
    return launch_hog(ctx, images, d_image_index, d_x, ldx, num_samples, num_landmarks, eyes, p, d_A, ld,
                      nullptr, nullptr, nullptr);
}

int sd_hog_debug(sd_ctx* ctx, const sd_image_batch* images, const int32_t* d_image_index, const float* d_x,
                 int64_t ldx, int num_samples, int num_landmarks, const sd_normalisation* eyes,
                 const sd_hog_param* p, int32_t* d_geometry, uint8_t* d_patches, int8_t* d_bins)
{
    if (!ctx) return SD_ERR_INVALID;
    return launch_hog(ctx, images, d_image_index, d_x, ldx, num_samples, num_landmarks, eyes, p, nullptr, 0,
                      d_geometry, d_patches, d_bins);
}

int sd_bgr2gray(sd_ctx* ctx, const uint8_t* d_bgr, int width, int height, int64_t bgr_row_stride, int64_t bgr_image_stride,
                int count, uint8_t* d_gray, int64_t gray_row_stride, int64_t gray_image_stride)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_REQUIRE(ctx, count >= 0 && width > 0 && height > 0, "bad argument");
    if (count == 0) return SD_OK;
    SD_REQUIRE(ctx, d_bgr && d_gray && bgr_row_stride >= 3LL * width && gray_row_stride >= width, "bad argument");
    const sd_bgr2gray_job uniform{0, 0, width, height, bgr_row_stride, gray_row_stride};
    return sd_bgr2gray_launch(ctx, ctx->stream, d_bgr, d_gray, uniform, bgr_image_stride, gray_image_stride, nullptr, count,
                              (int64_t)height * ((width + 3) >> 2));
}

}  // extern "C"
