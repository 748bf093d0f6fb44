// rcr::detection_model on the device: load / save (cereal binary, byte compatible with the reference's
// face_landmarks_model_rcr_*.bin), align_mean, and the batched detect cascade.
//
//   file format    model.hpp:178-182 -> superviseddescent.hpp:356-360 -> regressors.hpp:395-399,164-168
//                  -> utils/mat_cerealisation.hpp:42-99 ; model.hpp:111-115 ; adaptive_vlhog.hpp:55-59
//   detect         model.hpp:132-157 -> superviseddescent.hpp:323-344 (predict: sequential over levels)
#include "sd_internal.cuh"

#include <cmath>
#include <cstring>
#include <exception>
#include <fstream>
#include <string>
#include <vector>

struct sd_model {
    int device = 0;
    int num_levels = 0;
    int num_landmarks = 0;
    std::vector<int> rows, cols;
    std::vector<std::vector<float>> weights;      // host copies (for save / getters)
    std::vector<float*> d_weights;                // device copies
    std::vector<sd_regulariser> regs;
    std::vector<sd_hog_param> hog;
    std::vector<float> mean;
    float* d_mean = nullptr;                      // device copy for sd_model_align_boxes
    std::vector<std::string> ids, right_ids, left_ids;
    sd_normalisation norm{};
};

namespace {

// ---- little-endian byte cursor over the whole file -------------------------------------------------
struct Cursor {
    const std::vector<unsigned char>& buf;
    size_t pos = 0;
    bool good = true;
    explicit Cursor(const std::vector<unsigned char>& b) : buf(b) {}
    template <class T> T get()
    {
        T v{};
        if (pos + sizeof(T) > buf.size()) { good = false; return v; }
        memcpy(&v, buf.data() + pos, sizeof(T));
        pos += sizeof(T);
        return v;
    }
    bool bytes(void* dst, size_t n)
    {
        if (pos + n > buf.size()) { good = false; return false; }
        memcpy(dst, buf.data() + pos, n);
        pos += n;
        return true;
    }
    std::vector<std::string> strings()
    {
        std::vector<std::string> out;
        const uint64_t n = get<uint64_t>();                 // cereal size_type
        if (!good || n > buf.size()) { good = false; return out; }
        for (uint64_t i = 0; i < n && good; ++i) {
            const uint64_t len = get<uint64_t>();
            if (!good || len > buf.size() - pos) { good = false; break; }
            out.emplace_back(reinterpret_cast<const char*>(buf.data() + pos), (size_t)len);
            pos += (size_t)len;
        }
        return out;
    }
    bool matrix(std::vector<float>& data, int& r, int& c)
    {
        r = get<int32_t>();
        c = get<int32_t>();
        const int32_t type = get<int32_t>();
        (void)get<uint8_t>();                               // isContinuous: same bytes either way for a packed Mat
        if (!good || type != 5 /* CV_32FC1 */ || r < 0 || c < 0) { good = false; return false; }
        if ((uint64_t)r * (uint64_t)c > (buf.size() - pos) / sizeof(float)) { good = false; return false; }   // corrupt header: do not allocate
        data.resize((size_t)r * c);
        return bytes(data.data(), data.size() * sizeof(float));
    }
};

struct Writer {
    std::vector<unsigned char> out;
    template <class T> void put(T v)
    {
        const unsigned char* p = reinterpret_cast<const unsigned char*>(&v);
        out.insert(out.end(), p, p + sizeof(T));
    }
    void strings(const std::vector<std::string>& v)
    {
        put<uint64_t>(v.size());
        for (const auto& s : v) { put<uint64_t>(s.size()); out.insert(out.end(), s.begin(), s.end()); }
    }
    void matrix(const std::vector<float>& d, int r, int c)
    {
        put<int32_t>(r); put<int32_t>(c); put<int32_t>(5); put<uint8_t>(1);
        const unsigned char* p = reinterpret_cast<const unsigned char*>(d.data());
        out.insert(out.end(), p, p + d.size() * sizeof(float));
    }
};

int resolve_eyes(sd_ctx* ctx, sd_model* m)
{
    auto find = [&](const std::string& s) {
        for (size_t i = 0; i < m->ids.size(); ++i) if (m->ids[i] == s) return (int)i;
        return -1;
    };
    if (m->right_ids.empty() || m->left_ids.empty() || m->right_ids.size() > SD_MAX_EYES || m->left_ids.size() > SD_MAX_EYES)
        return sd_fail(ctx, SD_ERR_INVALID, "a model needs 1..%d eye identifiers per eye", SD_MAX_EYES);
    m->norm.kind = 1;
    m->norm.n_right = (int)m->right_ids.size();
    m->norm.n_left = (int)m->left_ids.size();
    for (int i = 0; i < m->norm.n_right; ++i) {
        m->norm.right_idx[i] = find(m->right_ids[i]);
        if (m->norm.right_idx[i] < 0) return sd_fail(ctx, SD_ERR_MISSING_ID, "one of given rightEyeIdentifiers ids not present in lms");
    }
    for (int i = 0; i < m->norm.n_left; ++i) {
        m->norm.left_idx[i] = find(m->left_ids[i]);
        if (m->norm.left_idx[i] < 0) return sd_fail(ctx, SD_ERR_MISSING_ID, "one of given leftEyeIdentifiers ids not present in lms");
    }
    return SD_OK;
}

int validate_and_upload(sd_ctx* ctx, sd_model* m)
{
    const int L = m->num_landmarks;
    if (L < 1 || (int)m->mean.size() != 2 * L) return sd_fail(ctx, SD_ERR_INVALID, "mean must have 2L entries");
    for (int s = 0; s < m->num_levels; ++s) {
        const int D = sd_hog_feature_length(L, &m->hog[s]);
        if (m->rows[s] != D || m->cols[s] != 2 * L)
            return sd_fail(ctx, SD_ERR_INVALID, "level %d: regressor is %dx%d but the HOG parameters give %dx%d", s, m->rows[s], m->cols[s], D, 2 * L);
    }
    int rc = resolve_eyes(ctx, m);
    if (rc) return rc;
    m->device = ctx->device;
    m->d_weights.assign(m->num_levels, nullptr);
    for (int s = 0; s < m->num_levels; ++s) {
        const size_t bytes = m->weights[s].size() * sizeof(float);
        SD_CUDA(ctx, cudaMalloc(&m->d_weights[s], bytes));
        SD_CUDA(ctx, cudaMemcpyAsync(m->d_weights[s], m->weights[s].data(), bytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    SD_CUDA(ctx, cudaMalloc(&m->d_mean, m->mean.size() * sizeof(float)));
    SD_CUDA(ctx, cudaMemcpyAsync(m->d_mean, m->mean.data(), m->mean.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    SD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SD_OK;
}

// d_image_index: frame of each face (NULL: face i reads frame i)
int detect_device(sd_ctx* ctx, const sd_model* m, const sd_image_batch* images, const int32_t* d_image_index, const float* d_x0,
                  int count, float* d_landmarks)
{
    const int L = m->num_landmarks, P = 2 * L;
    if (count <= 0) return SD_OK;
    // ping-pong landmark buffers
    float* xa = (float*)sd_workspace(ctx, SD_WS_SCRATCH, (size_t)2 * count * P * sizeof(float));
    if (!xa) return SD_ERR_CUDA;
    float* xb = xa + (size_t)count * P;
    SD_CUDA(ctx, cudaMemcpyAsync(xa, d_x0, (size_t)count * P * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
    int maxD = 0;
    for (int s = 0; s < m->num_levels; ++s) maxD = m->rows[s] > maxD ? m->rows[s] : maxD;
    const int64_t ld = ((int64_t)maxD + 3) / 4 * 4;
    float* A = (float*)sd_workspace(ctx, SD_WS_FEATURES, (size_t)count * ld * sizeof(float));
    if (!A) return SD_ERR_CUDA;
    float* cur = xa;
    float* nxt = xb;
    for (int s = 0; s < m->num_levels; ++s) {               // superviseddescent.hpp:326-342
        int rc = sd_hog_batch(ctx, images, d_image_index, cur, P, count, L, &m->norm, &m->hog[s], A, ld);
        if (rc) return rc;
        rc = sd_cascade_update(ctx, A, ld, count, m->rows[s], m->d_weights[s], P, cur, &m->norm, nxt);
        if (rc) return rc;
        float* t = cur; cur = nxt; nxt = t;
    }
    SD_CUDA(ctx, cudaMemcpyAsync(d_landmarks, cur, (size_t)count * P * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
    return SD_OK;
}


// ---- region-of-interest upload (sd_detect_batch_host, sd_detect_faces_host) --------------------------------
// The cascade only ever reads a neighbourhood of the face, so instead of copying whole frames over PCIe a small kernel pulls
// the rows of every ROI straight out of the caller's PINNED host frames (zero-copy loads through the unified address space,
// 16-byte vectors) into a packed device buffer.  If a patch later needs a frame pixel outside its ROI the HOG kernel raises
// d_roi_miss[roi] and the faces of that ROI are repeated from their full frame, so the result never depends on the ROI
// heuristic.

// where ROI i is read from: the device-mapped address of its frame's first pixel, the frame's pitch in bytes and its channel
// count (1: 8UC1, 3: 8UC3 B,G,R)
struct RoiSource {
    const uint8_t* frame;
    long long row_stride;
    int channels;
};

// one 16-byte vector of gray pixels from 48 bytes of interleaved B,G,R (16 pixels), cv::cvtColor(BGR2GRAY) bit for bit
__device__ __forceinline__ uint4 bgr48_to_gray16(const uint4& a, const uint4& b, const uint4& c)
{
    const uint32_t w[12] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w};
    uint32_t g[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        uint32_t v = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int p = 3 * (4 * q + k);                // byte of the pixel's B in the 48 bytes
            const uint32_t bb = (w[p >> 2] >> (8 * (p & 3))) & 255;
            const uint32_t gg = (w[(p + 1) >> 2] >> (8 * ((p + 1) & 3))) & 255;
            const uint32_t rr = (w[(p + 2) >> 2] >> (8 * ((p + 2) & 3))) & 255;
            v |= sd_bgr2gray_px(bb, gg, rr) << (8 * k);
        }
        g[q] = v;
    }
    return make_uint4(g[0], g[1], g[2], g[3]);
}

// One CTA per ROI (grid-stride over the ROIs); the instance for CH channels gathers the ROIs of CH-channel frames and skips the
// others.  A colour ROI is converted to gray as it is gathered: three 16-byte loads (16 B,G,R pixels) per stored 16-byte gray
// vector, so the packed buffer holds gray ROIs only.  Two instances rather than a branch on the channel count: the colour loop
// keeps twelve 16-byte loads and their conversion live (80 registers a thread, the gray loop 48), and one kernel holding both
// loops took 116, a footprint the gray gather would then carry beside the HOG kernels it overlaps.
template <int CH>
__global__ void __launch_bounds__(256) roi_gather_kernel(const RoiSource* __restrict__ srcs, const sd_roi* __restrict__ roi, int first,
                                                         int n, uint8_t* __restrict__ dst)
{
    for (int f = blockIdx.x; f < n; f += gridDim.x) {
        const RoiSource s = srcs[first + f];
        if (s.channels != CH) continue;
        const sd_roi r = roi[first + f];
        const long long row_stride = s.row_stride;
        uint8_t* d = dst + r.offset;
        const int vec_per_row = r.row_stride >> 4;
        const int total = vec_per_row * r.h;
        if (CH == 3) {
            // x is a multiple of 16 pixels = 48 bytes: with a 16-byte aligned base and pitch every load is aligned
            const uint8_t* src = s.frame + (long long)r.y * row_stride + 3LL * r.x;
            // four vectors (twelve 16-byte reads) in flight per thread before the stores: PCIe read latency is ~1 us
            for (int i0 = threadIdx.x; i0 < total; i0 += 4 * blockDim.x) {
                uint4 v[4][3];
                int row[4], col[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int i = i0 + u * blockDim.x;
                    row[u] = i / vec_per_row;
                    col[u] = i - row[u] * vec_per_row;
                    if (i < total) {
                        const uint4* p = reinterpret_cast<const uint4*>(src + (long long)row[u] * row_stride) + 3 * col[u];
                        v[u][0] = p[0]; v[u][1] = p[1]; v[u][2] = p[2];
                    }
                }
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (i0 + u * blockDim.x < total)
                        reinterpret_cast<uint4*>(d + (long long)row[u] * r.row_stride)[col[u]] = bgr48_to_gray16(v[u][0], v[u][1], v[u][2]);
            }
            continue;
        }
        const uint8_t* src = s.frame + (long long)r.y * row_stride + r.x;
        // four independent 16-byte reads in flight per thread before the stores: PCIe read latency is ~1 us
        for (int i0 = threadIdx.x; i0 < total; i0 += 4 * blockDim.x) {
            uint4 v[4];
            int row[4], col[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = i0 + u * blockDim.x;
                row[u] = i / vec_per_row;
                col[u] = i - row[u] * vec_per_row;
                if (i < total) v[u] = reinterpret_cast<const uint4*>(src + (long long)row[u] * row_stride)[col[u]];
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (i0 + u * blockDim.x < total) reinterpret_cast<uint4*>(d + (long long)row[u] * r.row_stride)[col[u]] = v[u];
        }
    }
}

// sd_align_mean(mean, box, 1, 1, 0, 0) for every coordinate of every box, bit for bit: the scale and offset are formed in
// double and rounded to float as the host does, and the product and sum are separately rounded (no FMA contraction)
__global__ void align_boxes_kernel(const float* __restrict__ mean, int L, const int32_t* __restrict__ boxes, int count,
                                   float* __restrict__ x0, long long ldx)
{
    const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const int P = 2 * L;
    if (t >= (long long)count * P) return;
    const int i = (int)(t / P), j = (int)(t - (long long)i * P);
    const bool is_y = j >= L;
    const int origin = boxes[4 * i + (is_y ? 1 : 0)], size = boxes[4 * i + (is_y ? 3 : 2)];
    const float a = __double2float_rn(__dmul_rn(1.0, (double)size));
    const float b = __double2float_rn(__dadd_rn(__dmul_rn(__dadd_rn(0.5, 0.0), (double)size), (double)origin));
    x0[(long long)i * ldx + j] = __fadd_rn(__fmul_rn(mean[j], a), b);
}

// conservative ROI of one face: landmark bounding box of the initialisation, grown by the largest patch
// half size of the schedule plus a drift allowance, clipped to the frame, x aligned to 16 pixels; row_pixels = the frame's pitch
// in pixels (row_stride / channels): rows are never read past it
sd_roi face_roi(const sd_model* m, const float* x0, int width, int height, int row_pixels)
{
    const int L = m->num_landmarks;
    float minx = x0[0], maxx = x0[0], miny = x0[L], maxy = x0[L];
    for (int i = 1; i < L; ++i) {
        minx = x0[i] < minx ? x0[i] : minx; maxx = x0[i] > maxx ? x0[i] : maxx;
        miny = x0[i + L] < miny ? x0[i + L] : miny; maxy = x0[i + L] > maxy ? x0[i + L] : maxy;
    }
    float rxs = 0, rys = 0, lxs = 0, lys = 0;
    for (int i = 0; i < m->norm.n_right; ++i) { rxs += x0[m->norm.right_idx[i]]; rys += x0[m->norm.right_idx[i] + L]; }
    for (int i = 0; i < m->norm.n_left; ++i) { lxs += x0[m->norm.left_idx[i]]; lys += x0[m->norm.left_idx[i] + L]; }
    rxs /= m->norm.n_right; rys /= m->norm.n_right; lxs /= m->norm.n_left; lys /= m->norm.n_left;
    const float ied = std::sqrt((rxs - lxs) * (rxs - lxs) + (rys - lys) * (rys - lys));
    // per level: half patch (the IED may grow a little) + how far the landmarks may have drifted by then (none at level 0)
    float grow = 0.f;
    for (size_t l = 0; l < m->hog.size(); ++l) {
        const float g = 0.5f * m->hog[l].relative_patch_size * ied * 1.1f + (l > 0 ? 0.2f * ied : 0.f);
        grow = g > grow ? g : grow;
    }
    grow += 4.f;
    int xa = (int)std::floor(minx - grow), xb = (int)std::ceil(maxx + grow);
    int ya = (int)std::floor(miny - grow), yb = (int)std::ceil(maxy + grow);
    xa = xa < 0 ? 0 : xa; ya = ya < 0 ? 0 : ya;
    xb = xb > width ? width : xb; yb = yb > height ? height : yb;
    sd_roi r{};
    if (xb <= xa || yb <= ya) { xa = 0; ya = 0; xb = 16 < width ? 16 : width; yb = 1; }   // face entirely outside the frame
    r.x = xa & ~15;
    int w = ((xb - r.x) + 15) & ~15;
    const int maxw = (row_pixels - r.x) & ~15;
    if (w > maxw) w = maxw;
    r.w = w; r.y = ya; r.h = yb - ya; r.row_stride = w; r.reserved = 0; r.offset = 0;
    return r;
}

}  // namespace

namespace {
// apps/rcr/rcr-train.cpp:149-212: one warp per row; cv::norm's float differences / double sum / double sqrt, the result
// stored as float (:169) and multiplied by the float factor (float)(1.0f / IED(prediction)).
__global__ void landmark_error_kernel(const float* __restrict__ pred, long long ldp, const float* __restrict__ gt, long long ldgt, int N,
                                      int L, const sd_eyes_dev eyes, float* __restrict__ err, long long lde)
{
    const int r = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (r >= N) return;
    const float* p = pred + (long long)r * ldp;
    const float* g = gt + (long long)r * ldgt;
    const double ied = sd_device_ied(p, L, eyes);
    const float f = (float)(1.0 / ied);
    for (int i = lane; i < L; i += 32) {
        const float dx = __fsub_rn(p[i], g[i]), dy = __fsub_rn(p[i + L], g[i + L]);
        const float n = (float)sqrt(__dadd_rn(__dmul_rn((double)dx, (double)dx), __dmul_rn((double)dy, (double)dy)));
        err[(long long)r * lde + i] = __fmul_rn(n, f);
    }
}
}  // namespace

extern "C" {

int sd_align_mean(const float* h_mean, int L, int box_x, int box_y, int box_w, int box_h, float sx, float sy,
                  float tx, float ty, float* h_out)
{
    if (!h_mean || !h_out || L < 1) return SD_ERR_INVALID;
    // model.hpp:72-73.  OpenCV folds (m*s + 0.5f + t) * w + x into one scaled conversion
    // m * (float)(s*w) + (float)((0.5 + t)*w + x), evaluated in float (mul, then add).
    const float ax = (float)((double)sx * (double)box_w);
    const float bx = (float)(((double)0.5f + (double)tx) * (double)box_w + (double)box_x);
    const float ay = (float)((double)sy * (double)box_h);
    const float by = (float)(((double)0.5f + (double)ty) * (double)box_h + (double)box_y);
    for (int i = 0; i < L; ++i) {
        volatile float px = h_mean[i] * ax;        // volatile: keep mul and add un-fused on any host compiler
        h_out[i] = px + bx;
        volatile float py = h_mean[i + L] * ay;
        h_out[i + L] = py + by;
    }
    return SD_OK;
}

int sd_perturb_box(int box_x, int box_y, int box_w, int box_h, float tx, float ty, float scaling, int32_t out_box[4])
{
    if (!out_box) return SD_ERR_INVALID;
    // rcr-train.cpp:133-143, float arithmetic; volatile keeps every product / sum a separately rounded float
    volatile float tx_pixel = tx * (float)box_w;
    volatile float ty_pixel = ty * (float)box_h;
    volatile float pw = (float)box_w * scaling;
    volatile float ph = (float)box_h * scaling;
    volatile float hx = ((float)box_w - pw) / 2.0f, hy = ((float)box_h - ph) / 2.0f;
    volatile float x = (float)box_x + hx, y = (float)box_y + hy;
    out_box[0] = (int32_t)(x + tx_pixel);
    out_box[1] = (int32_t)(y + ty_pixel);
    out_box[2] = (int32_t)pw;
    out_box[3] = (int32_t)ph;
    return SD_OK;
}

int sd_normalised_landmark_errors(sd_ctx* ctx, const float* d_pred, int64_t ldp, const float* d_gt, int64_t ldgt, int N, int L,
                                  const sd_normalisation* eyes, float* d_err, int64_t lde)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_REQUIRE(ctx, d_pred && d_gt && d_err && N >= 0 && L >= 1 && ldp >= 2 * L && ldgt >= 2 * L && lde >= L, "bad argument");
    SD_REQUIRE(ctx, eyes && eyes->kind == 1, "the normalised error needs the eye landmark indices");
    if (N == 0) return SD_OK;
    sd_eyes_dev eyes_dev;
    int rc = sd_eyes_to_dev(ctx, eyes, L, &eyes_dev);
    if (rc) return rc;
    landmark_error_kernel<<<sd_div_up(N, 4), 128, 0, ctx->stream>>>(d_pred, ldp, d_gt, ldgt, N, L, eyes_dev, d_err, lde);
    SD_LAUNCH_CHECK(ctx, "landmark_error_kernel");
    return SD_OK;
}

static int model_load_impl(sd_ctx* ctx, const char* path, sd_model** out)
{
    std::ifstream f(path, std::ios::binary);
    if (!f) return sd_fail(ctx, SD_ERR_IO, "The given model file could not be opened: %s", path);   // model.hpp:199
    std::vector<unsigned char> buf((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
    Cursor c(buf);
    sd_model* m = new sd_model();
    auto bail = [&](const char* why) { delete m; return sd_fail(ctx, SD_ERR_IO, "%s: %s", why, path); };

    const uint64_t nreg = c.get<uint64_t>();                 // vector<LinearRegressor>
    if (!c.good || nreg == 0 || nreg > 256) return bail("not a detection_model archive (regressor count)");
    m->num_levels = (int)nreg;
    m->rows.resize(nreg); m->cols.resize(nreg); m->weights.resize(nreg); m->regs.resize(nreg);
    for (uint64_t i = 0; i < nreg; ++i) {
        if (!c.matrix(m->weights[i], m->rows[i], m->cols[i])) return bail("truncated regressor matrix");
        m->regs[i].type = c.get<int32_t>();                  // Regulariser: type, lambda, regularise_last_row
        m->regs[i].param = c.get<float>();
        m->regs[i].regularise_last_row = c.get<uint8_t>();
    }
    const auto n_ids = c.strings();                          // InterEyeDistanceNormalisation's own copies
    const auto n_right = c.strings();
    const auto n_left = c.strings();
    int mr = 0, mc = 0;
    if (!c.matrix(m->mean, mr, mc)) return bail("truncated mean");
    m->ids = c.strings();
    const uint64_t nhog = c.get<uint64_t>();
    if (!c.good || nhog != nreg) return bail("hog_params count differs from the regressor count");
    m->hog.resize(nhog);
    for (uint64_t i = 0; i < nhog; ++i) {
        m->hog[i].variant = c.get<int32_t>();
        m->hog[i].num_cells = c.get<int32_t>();
        m->hog[i].cell_size = c.get<int32_t>();
        m->hog[i].num_bins = c.get<int32_t>();
        m->hog[i].relative_patch_size = c.get<float>();
    }
    m->right_ids = c.strings();
    m->left_ids = c.strings();
    if (!c.good || c.pos != buf.size()) return bail("truncated archive or trailing bytes");
    if (mr != 1 || n_ids != m->ids || n_right != m->right_ids || n_left != m->left_ids)
        return bail("inconsistent archive (normaliser ids differ from the model's)");
    m->num_landmarks = (int)m->ids.size();
    int rc = validate_and_upload(ctx, m);
    if (rc) { sd_model_destroy(m); return rc; }
    *out = m;
    return SD_OK;
}

int sd_model_load(sd_ctx* ctx, const char* path, sd_model** out)
{
    if (!ctx || !path || !out) return SD_ERR_INVALID;
    *out = nullptr;
    try {                                                     // nothing may unwind through the C boundary
        return model_load_impl(ctx, path, out);
    } catch (const std::exception& e) {
        return sd_fail(ctx, SD_ERR_IO, "could not read %s: %s", path, e.what());
    } catch (...) {
        return sd_fail(ctx, SD_ERR_IO, "could not read %s", path);
    }
}

int sd_model_save(sd_ctx* ctx, const sd_model* m, const char* path)
{
    if (!ctx || !m || !path) return SD_ERR_INVALID;
    Writer w;
    w.put<uint64_t>((uint64_t)m->num_levels);
    for (int i = 0; i < m->num_levels; ++i) {
        w.matrix(m->weights[i], m->rows[i], m->cols[i]);
        w.put<int32_t>(m->regs[i].type);
        w.put<float>(m->regs[i].param);
        w.put<uint8_t>(m->regs[i].regularise_last_row ? 1 : 0);
    }
    w.strings(m->ids); w.strings(m->right_ids); w.strings(m->left_ids);
    w.matrix(m->mean, 1, 2 * m->num_landmarks);
    w.strings(m->ids);
    w.put<uint64_t>((uint64_t)m->num_levels);
    for (int i = 0; i < m->num_levels; ++i) {
        w.put<int32_t>(m->hog[i].variant); w.put<int32_t>(m->hog[i].num_cells); w.put<int32_t>(m->hog[i].cell_size);
        w.put<int32_t>(m->hog[i].num_bins); w.put<float>(m->hog[i].relative_patch_size);
    }
    w.strings(m->right_ids); w.strings(m->left_ids);
    std::ofstream f(path, std::ios::binary);
    if (!f) return sd_fail(ctx, SD_ERR_IO, "could not open %s for writing", path);
    f.write(reinterpret_cast<const char*>(w.out.data()), (std::streamsize)w.out.size());
    return f.good() ? SD_OK : sd_fail(ctx, SD_ERR_IO, "short write to %s", path);
}

int sd_model_create(sd_ctx* ctx, int num_levels, int num_landmarks, const float* const* h_weights,
                    const sd_regulariser* regs, const sd_hog_param* hog_params, const float* h_mean,
                    const char* const* landmark_ids, const char* const* right_eye_ids, int n_right,
                    const char* const* left_eye_ids, int n_left, sd_model** out)
{
    if (!ctx || !out) return SD_ERR_INVALID;
    *out = nullptr;
    SD_REQUIRE(ctx, num_levels >= 1 && num_landmarks >= 1 && h_weights && regs && hog_params && h_mean && landmark_ids &&
                        right_eye_ids && left_eye_ids, "null / empty argument");
    sd_model* m = new sd_model();
    m->num_levels = num_levels;
    m->num_landmarks = num_landmarks;
    for (int i = 0; i < num_landmarks; ++i) m->ids.emplace_back(landmark_ids[i]);
    for (int i = 0; i < n_right; ++i) m->right_ids.emplace_back(right_eye_ids[i]);
    for (int i = 0; i < n_left; ++i) m->left_ids.emplace_back(left_eye_ids[i]);
    m->mean.assign(h_mean, h_mean + 2 * num_landmarks);
    m->rows.resize(num_levels); m->cols.resize(num_levels); m->weights.resize(num_levels);
    m->regs.assign(regs, regs + num_levels);
    m->hog.assign(hog_params, hog_params + num_levels);
    for (int s = 0; s < num_levels; ++s) {
        m->rows[s] = sd_hog_feature_length(num_landmarks, &hog_params[s]);
        m->cols[s] = 2 * num_landmarks;
        m->weights[s].assign(h_weights[s], h_weights[s] + (size_t)m->rows[s] * m->cols[s]);
    }
    int rc = validate_and_upload(ctx, m);
    if (rc) { sd_model_destroy(m); return rc; }
    *out = m;
    return SD_OK;
}

void sd_model_destroy(sd_model* m)
{
    if (!m) return;
    cudaSetDevice(m->device);
    for (float* p : m->d_weights) if (p) cudaFree(p);
    if (m->d_mean) cudaFree(m->d_mean);
    delete m;
}

int sd_model_num_levels(const sd_model* m) { return m ? m->num_levels : -1; }
int sd_model_num_landmarks(const sd_model* m) { return m ? m->num_landmarks : -1; }
int sd_model_hog_param(const sd_model* m, int level, sd_hog_param* out)
{
    if (!m || !out || level < 0 || level >= m->num_levels) return SD_ERR_INVALID;
    *out = m->hog[level];
    return SD_OK;
}
int sd_model_regulariser(const sd_model* m, int level, sd_regulariser* out)
{
    if (!m || !out || level < 0 || level >= m->num_levels) return SD_ERR_INVALID;
    *out = m->regs[level];
    return SD_OK;
}
int sd_model_normalisation(const sd_model* m, sd_normalisation* out)
{
    if (!m || !out) return SD_ERR_INVALID;
    *out = m->norm;
    return SD_OK;
}
int sd_model_get_mean(const sd_model* m, float* h_mean)
{
    if (!m || !h_mean) return SD_ERR_INVALID;
    memcpy(h_mean, m->mean.data(), m->mean.size() * sizeof(float));
    return SD_OK;
}
int sd_model_get_weights(const sd_model* m, int level, float* h_w, int* rows, int* cols)
{
    if (!m || level < 0 || level >= m->num_levels) return SD_ERR_INVALID;
    if (rows) *rows = m->rows[level];
    if (cols) *cols = m->cols[level];
    if (h_w) memcpy(h_w, m->weights[level].data(), m->weights[level].size() * sizeof(float));
    return SD_OK;
}
const char* sd_model_landmark_id(const sd_model* m, int i)
{
    if (!m || i < 0 || i >= m->num_landmarks) return nullptr;
    return m->ids[i].c_str();
}

int sd_detect_batch_device(sd_ctx* ctx, const sd_model* m, const sd_image_batch* images, const float* d_x0, int count,
                           float* d_landmarks)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_REQUIRE(ctx, m && images && d_x0 && d_landmarks && count >= 0, "bad argument");
    SD_REQUIRE(ctx, images->count >= count, "fewer images than faces");
    const int rc = detect_device(ctx, m, images, nullptr, d_x0, count, d_landmarks);
    if (rc) return rc;
    // a degenerate face (inter-eye distance too small for a patch) or a bad frame index is an error here, as it is in the
    // reference (cv::resize on an empty ROI throws); reading the flag synchronises the stream
    return sd_check_hog_status(ctx, "detect");
}

}  // extern "C"

namespace {

// one frame in host memory (channels 1: 8UC1, 3: 8UC3 B,G,R); d_alias: its device-mapped address when it is pinned with 16-byte
// aligned base and pitch
struct HostFrame {
    const uint8_t* h;
    const uint8_t* d_alias;
    int width, height, row_stride;
    int channels;
};

int ensure_staging(sd_ctx* ctx, size_t bytes)
{
    for (int b = 0; b < 2; ++b) {
        if (ctx->stage_bytes[b] < bytes) {
            if (ctx->d_stage[b]) { SD_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); SD_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream)); SD_CUDA(ctx, cudaFree(ctx->d_stage[b])); ctx->d_stage[b] = nullptr; }
            SD_CUDA(ctx, cudaMalloc(&ctx->d_stage[b], bytes));
            ctx->stage_bytes[b] = bytes;
        }
    }
    return SD_OK;
}

// Whole-frame route.  Faces [0, count) with frame[k] = frames[fidx[k]], fidx non-decreasing; h_x0 / h_out in that order.
// Every referenced frame is uploaded once into the double-buffered staging, in chunks of whole frames (~128 MB, or a single
// frame larger than that) together with all of their faces.  A chunk of equally sized frames is staged as a uniform batch (the
// HOG kernel's TMA route applies), any other chunk is described by sd_frame records.  A colour frame goes up as B,G,R into the
// chunk's buffer behind its gray frames (the 128 MB count both) and one conversion launch per chunk, on the copy stream before
// the chunk's stage event, writes its gray frame with a 16-byte aligned pitch.
int detect_host_full(sd_ctx* ctx, const sd_model* m, const HostFrame* frames, const int* fidx, const float* h_x0, int count, float* h_out)
{
    const int P = 2 * m->num_landmarks;
    const size_t cap = (size_t)128 << 20;
    // distinct referenced frames (in face order) and the chunks they are staged in
    std::vector<int> uf;                       // unique frame -> frames[]
    std::vector<int> face_u(count);            // face -> unique frame
    for (int k = 0; k < count; ++k) {
        if (k == 0 || fidx[k] != fidx[k - 1]) uf.push_back(fidx[k]);
        face_u[k] = (int)uf.size() - 1;
    }
    // gray pitch in the staging buffer: a gray frame keeps its own, a colour frame is converted into 16-byte aligned rows
    auto gray_pitch = [](const HostFrame& f) { return f.channels == 3 ? (f.width + 15) & ~15 : f.row_stride; };
    struct Chunk { int u0, u1, f0, f1; bool uniform; size_t bgr_bytes; };
    std::vector<Chunk> chunks;
    std::vector<sd_frame> rec(uf.size());
    std::vector<size_t> src_off(uf.size());    // where the frame's host bytes go in the staging buffer (gray: rec offset)
    size_t used = 0, bgr_used = 0, stage_need = 0;
    for (int u = 0; u < (int)uf.size(); ++u) {
        const HostFrame& f = frames[uf[u]];
        const size_t padded = ((size_t)f.height * gray_pitch(f) + 15) & ~(size_t)15;
        const size_t bgr = f.channels == 3 ? (size_t)f.height * f.row_stride : 0;
        if (chunks.empty() || used + bgr_used + padded + bgr > cap) { chunks.push_back({u, u, 0, 0, true, 0}); used = 0; bgr_used = 0; }
        rec[u] = sd_frame{f.width, f.height, gray_pitch(f), 0, (int64_t)used};
        src_off[u] = bgr_used;                 // relative to the chunk's B,G,R region until the chunk is complete
        used += padded;
        bgr_used += bgr;
        chunks.back().u1 = u + 1;
        chunks.back().bgr_bytes = bgr_used;
    }
    std::vector<sd_bgr2gray_job> jobs;
    std::vector<int> chunk_job0;               // first conversion job of every chunk
    for (Chunk& c : chunks) {
        const HostFrame& f0 = frames[uf[c.u0]];
        for (int u = c.u0; u < c.u1; ++u) {
            const HostFrame& f = frames[uf[u]];
            c.uniform = c.uniform && f.width == f0.width && f.height == f0.height && gray_pitch(f) == gray_pitch(f0);
        }
        const size_t fb = (size_t)f0.height * gray_pitch(f0);
        if (c.uniform)                          // packed back to back, like one (n, height, row_stride) array
            for (int u = c.u0; u < c.u1; ++u) rec[u].offset = (int64_t)((u - c.u0) * fb);
        const HostFrame& fl = frames[uf[c.u1 - 1]];
        const size_t gray_bytes = (size_t)(rec[c.u1 - 1].offset) + (size_t)fl.height * gray_pitch(fl);
        const size_t bgr0 = (gray_bytes + 15) & ~(size_t)15;
        chunk_job0.push_back((int)jobs.size());
        for (int u = c.u0; u < c.u1; ++u) {
            const HostFrame& f = frames[uf[u]];
            if (f.channels != 3) { src_off[u] = (size_t)rec[u].offset; continue; }
            src_off[u] += bgr0;
            jobs.push_back(sd_bgr2gray_job{(int64_t)src_off[u], rec[u].offset, f.width, f.height, f.row_stride, rec[u].row_stride});
        }
        const size_t bytes = c.bgr_bytes ? bgr0 + c.bgr_bytes : gray_bytes;
        stage_need = bytes > stage_need ? bytes : stage_need;
    }
    chunk_job0.push_back((int)jobs.size());
    for (size_t c = 0, k = 0; c < chunks.size(); ++c) {
        chunks[c].f0 = (int)k;
        while (k < (size_t)count && face_u[k] < chunks[c].u1) ++k;
        chunks[c].f1 = (int)k;
    }
    int rc = ensure_staging(ctx, stage_need);
    if (rc) return rc;
    // device tables: landmarks (in, out), frame of every face relative to its chunk, frame records, conversion jobs
    std::vector<int32_t> local(count);
    bool identity = true;                       // one face per frame: no index needed
    for (const Chunk& c : chunks)
        for (int k = c.f0; k < c.f1; ++k) { local[k] = face_u[k] - c.u0; identity = identity && local[k] == k - c.f0; }
    const size_t xbytes = (size_t)count * P * sizeof(float);
    const size_t ibytes = ((size_t)count * sizeof(int32_t) + 15) & ~(size_t)15;
    const size_t rbytes = rec.size() * sizeof(sd_frame);
    unsigned char* tab = (unsigned char*)sd_workspace(ctx, SD_WS_PARTIAL, 2 * xbytes + ibytes + rbytes + jobs.size() * sizeof(sd_bgr2gray_job));
    if (!tab) return SD_ERR_CUDA;
    float* d_x = (float*)tab;
    float* d_out = (float*)(tab + xbytes);
    int32_t* d_idx = (int32_t*)(tab + 2 * xbytes);
    sd_frame* d_rec = (sd_frame*)(tab + 2 * xbytes + ibytes);
    sd_bgr2gray_job* d_jobs = (sd_bgr2gray_job*)(tab + 2 * xbytes + ibytes + rbytes);
    SD_CUDA(ctx, cudaMemcpyAsync(d_x, h_x0, xbytes, cudaMemcpyHostToDevice, ctx->stream));
    if (!identity) SD_CUDA(ctx, cudaMemcpyAsync(d_idx, local.data(), (size_t)count * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    bool any_mixed = false;
    for (const Chunk& c : chunks) any_mixed = any_mixed || !c.uniform;
    if (any_mixed) SD_CUDA(ctx, cudaMemcpyAsync(d_rec, rec.data(), rbytes, cudaMemcpyHostToDevice, ctx->stream));
    if (!jobs.empty()) SD_CUDA(ctx, cudaMemcpyAsync(d_jobs, jobs.data(), jobs.size() * sizeof(sd_bgr2gray_job), cudaMemcpyHostToDevice, ctx->stream));
    // the copy stream must not run ahead of work already queued on the compute stream that still reads the staging buffers
    // (the stage_done events also order the table uploads above before the first conversion)
    SD_CUDA(ctx, cudaEventRecord(ctx->stage_done[0], ctx->stream));
    SD_CUDA(ctx, cudaEventRecord(ctx->stage_done[1], ctx->stream));
    int buf = 0;
    for (size_t c = 0; c < chunks.size(); ++c, buf ^= 1) {
        const Chunk& ch = chunks[c];
        uint8_t* stage = (uint8_t*)ctx->d_stage[buf];
        SD_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->stage_done[buf], 0));
        // one copy per run of frames that lie back to back both in host memory and in the staging buffer; the last row of a run
        // is copied up to its width only (the caller's buffer may end there)
        for (int u = ch.u0; u < ch.u1;) {
            const HostFrame& f = frames[uf[u]];
            const size_t fb = (size_t)f.height * f.row_stride;
            int v = u + 1;
            while (v < ch.u1 && frames[uf[v]].h == f.h + (v - u) * fb && src_off[v] == src_off[u] + (v - u) * fb &&
                   frames[uf[v]].row_stride == f.row_stride && frames[uf[v]].height == f.height && frames[uf[v]].width == f.width &&
                   frames[uf[v]].channels == f.channels)
                ++v;
            const size_t bytes = (size_t)(v - u - 1) * fb + (size_t)(f.height - 1) * f.row_stride + (size_t)f.channels * f.width;
            SD_CUDA(ctx, cudaMemcpyAsync(stage + src_off[u], f.h, bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
            u = v;
        }
        const int j0 = chunk_job0[c], nj = chunk_job0[c + 1] - j0;
        if (nj > 0) {
            int64_t max_groups = 0;
            for (int j = j0; j < j0 + nj; ++j) {
                const int64_t g = (int64_t)jobs[j].height * ((jobs[j].width + 3) >> 2);
                max_groups = g > max_groups ? g : max_groups;
            }
            rc = sd_bgr2gray_launch(ctx, ctx->copy_stream, stage, stage, sd_bgr2gray_job{}, 0, 0, d_jobs + j0, nj, max_groups);
            if (rc) return rc;
        }
        SD_CUDA(ctx, cudaEventRecord(ctx->stage_ev[buf], ctx->copy_stream));
        SD_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->stage_ev[buf], 0));
        sd_image_batch ib{};
        ib.d_data = stage;
        ib.count = ch.u1 - ch.u0;
        if (ch.uniform) {
            const HostFrame& f = frames[uf[ch.u0]];
            ib.width = f.width; ib.height = f.height; ib.row_stride = gray_pitch(f); ib.image_stride = (int64_t)f.height * gray_pitch(f);
        } else {
            ib.d_frames = d_rec + ch.u0;
        }
        const int n = ch.f1 - ch.f0;
        rc = detect_device(ctx, m, &ib, identity ? nullptr : d_idx + ch.f0, d_x + (size_t)ch.f0 * P, n, d_out + (size_t)ch.f0 * P);
        if (rc) return rc;
        SD_CUDA(ctx, cudaEventRecord(ctx->stage_done[buf], ctx->stream));
    }
    SD_CUDA(ctx, cudaMemcpyAsync(h_out, d_out, xbytes, cudaMemcpyDeviceToHost, ctx->stream));
    return sd_check_hog_status(ctx, "detect");                // synchronises
}

bool roi_intersect(const sd_roi& a, const sd_roi& b)
{
    return a.x < b.x + b.w && b.x < a.x + a.w && a.y < b.y + b.h && b.y < a.y + a.h;
}

// ROI route: every referenced frame pinned and device-mapped (HostFrame::d_alias).  Same face order and arguments as
// detect_host_full.  The ROIs of the faces of one frame that intersect are merged into one ROI group, gathered once; face ->
// group is the image index of the HOG launch, and d_roi / d_roi_miss / the gather's source table are indexed by group.
int detect_host_roi(sd_ctx* ctx, const sd_model* m, const HostFrame* frames, const int* fidx, const float* h_x0, int count, float* h_out)
{
    const int P = 2 * m->num_landmarks;
    const size_t chunk_cap = (size_t)48 << 20;            // packed ROI bytes per staging buffer
    // ROI groups, frame by frame: merge until no two groups of the frame intersect
    std::vector<sd_roi> groups;
    std::vector<int> group_frame;
    std::vector<int> face_group(count);
    for (int k0 = 0; k0 < count;) {
        int k1 = k0;
        while (k1 < count && fidx[k1] == fidx[k0]) ++k1;
        const HostFrame& f = frames[fidx[k0]];
        const int g0 = (int)groups.size();
        for (int k = k0; k < k1; ++k) {
            sd_roi r = face_roi(m, h_x0 + (size_t)k * P, f.width, f.height, f.row_stride / f.channels);
            int g = -1;
            for (int j = g0; j < (int)groups.size() && g < 0; ++j) if (roi_intersect(groups[j], r)) g = j;
            if (g < 0) { groups.push_back(r); group_frame.push_back(fidx[k0]); face_group[k] = (int)groups.size() - 1; continue; }
            face_group[k] = g;
            for (bool grown = true; grown;) {              // the union may now reach other groups of this frame: absorb them
                sd_roi& u = groups[g];
                const int xa = u.x < r.x ? u.x : r.x, ya = u.y < r.y ? u.y : r.y;
                const int xb = u.x + u.w > r.x + r.w ? u.x + u.w : r.x + r.w, yb = u.y + u.h > r.y + r.h ? u.y + u.h : r.y + r.h;
                u.x = xa; u.y = ya; u.w = xb - xa; u.h = yb - ya; u.row_stride = u.w;   // x and w stay multiples of 16
                grown = false;
                for (int j = g0; j < (int)groups.size(); ++j) {
                    if (j == g || !roi_intersect(groups[j], groups[g])) continue;
                    r = groups[j];
                    const int ng = j < g ? g - 1 : g;      // index of group g once j is erased
                    for (int q = k0; q < k; ++q) face_group[q] = face_group[q] == j ? ng : (face_group[q] > j ? face_group[q] - 1 : face_group[q]);
                    groups.erase(groups.begin() + j);
                    group_frame.erase(group_frame.begin() + j);
                    g = ng;
                    face_group[k] = g;
                    grown = true;
                    break;
                }
            }
        }
        k0 = k1;
    }
    const int G = (int)groups.size();
    // faces ordered by group (stable): the faces of a group are contiguous, so chunks of whole groups are ranges of faces
    std::vector<int> pos(count);                           // group order -> position in the caller's order
    {
        std::vector<int> start(G + 1, 0);
        for (int k = 0; k < count; ++k) start[face_group[k] + 1]++;
        for (int g = 0; g < G; ++g) start[g + 1] += start[g];
        for (int k = 0; k < count; ++k) pos[start[face_group[k]]++] = k;
    }
    bool identity = G == count;                            // one face per group, groups in face order
    for (int k = 0; k < count && identity; ++k) identity = pos[k] == k && face_group[k] == k;
    std::vector<float> gx0, gout;
    const float* x0 = h_x0;
    float* out = h_out;
    if (!identity) {
        gx0.resize((size_t)count * P); gout.resize((size_t)count * P);
        for (int k = 0; k < count; ++k) memcpy(&gx0[(size_t)k * P], h_x0 + (size_t)pos[k] * P, P * sizeof(float));
        x0 = gx0.data(); out = gout.data();
    }
    std::vector<int> gface0(G + 1, 0);                     // first face (group order) of every group
    for (int k = 0; k < count; ++k) gface0[face_group[pos[k]] + 1]++;
    for (int g = 0; g < G; ++g) gface0[g + 1] += gface0[g];
    std::vector<int32_t> local(count);                     // face -> group, relative to the chunk's first group
    std::vector<int> chunk_first;                          // groups
    std::vector<char> chunk_gray, chunk_colour;            // the chunk holds ROIs of gray / colour frames
    std::vector<RoiSource> srcs(G);
    bool same_size = true;
    size_t used = 0;
    for (int g = 0; g < G; ++g) {
        const HostFrame& f = frames[group_frame[g]];
        same_size = same_size && f.width == frames[group_frame[0]].width && f.height == frames[group_frame[0]].height;
        const size_t bytes = (size_t)groups[g].row_stride * groups[g].h;
        if (bytes > chunk_cap)                                // a face window larger than a staging buffer: whole-frame route
            return detect_host_full(ctx, m, frames, fidx, h_x0, count, h_out);
        if (chunk_first.empty() || used + bytes > chunk_cap) { chunk_first.push_back(g); chunk_gray.push_back(0); chunk_colour.push_back(0); used = 0; }
        groups[g].offset = (int64_t)used;
        used += bytes;
        srcs[g] = RoiSource{f.d_alias, (long long)f.row_stride, f.channels};
        (f.channels == 3 ? chunk_colour : chunk_gray).back() = 1;
        for (int k = gface0[g]; k < gface0[g + 1]; ++k) local[k] = g - chunk_first.back();
    }
    chunk_first.push_back(G);
    int rc = ensure_staging(ctx, chunk_cap + (1u << 20));
    if (rc) return rc;
    // frames of different sizes: the size of every group's frame (where the zero padding of a patch starts)
    std::vector<sd_frame> gframes;
    if (!same_size)
        for (int g = 0; g < G; ++g) gframes.push_back(sd_frame{frames[group_frame[g]].width, frames[group_frame[g]].height, 0, 0, 0});
    // device tables: landmarks (in, out), ROI records, gather sources, face -> group, frame sizes, miss flags
    const size_t xbytes = (size_t)count * P * sizeof(float);
    const size_t rbytes = (size_t)G * sizeof(sd_roi);
    const size_t sbytes = (size_t)G * sizeof(RoiSource);
    const size_t ibytes = ((size_t)count * sizeof(int32_t) + 15) & ~(size_t)15;
    const size_t fbytes = gframes.size() * sizeof(sd_frame);
    unsigned char* tab = (unsigned char*)sd_workspace(ctx, SD_WS_PARTIAL, 2 * xbytes + rbytes + sbytes + ibytes + fbytes + G + 64);
    if (!tab) return SD_ERR_CUDA;
    float* d_x = (float*)tab;
    float* d_out = (float*)(tab + xbytes);
    sd_roi* d_roi = (sd_roi*)(tab + 2 * xbytes);
    RoiSource* d_src = (RoiSource*)(tab + 2 * xbytes + rbytes);
    int32_t* d_idx = (int32_t*)(tab + 2 * xbytes + rbytes + sbytes);
    sd_frame* d_gframes = (sd_frame*)(tab + 2 * xbytes + rbytes + sbytes + ibytes);
    uint8_t* d_miss = tab + 2 * xbytes + rbytes + sbytes + ibytes + fbytes;
    SD_CUDA(ctx, cudaMemcpyAsync(d_x, x0, xbytes, cudaMemcpyHostToDevice, ctx->stream));
    SD_CUDA(ctx, cudaMemcpyAsync(d_roi, groups.data(), rbytes, cudaMemcpyHostToDevice, ctx->stream));
    SD_CUDA(ctx, cudaMemcpyAsync(d_src, srcs.data(), sbytes, cudaMemcpyHostToDevice, ctx->stream));
    if (!identity) SD_CUDA(ctx, cudaMemcpyAsync(d_idx, local.data(), (size_t)count * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    if (fbytes) SD_CUDA(ctx, cudaMemcpyAsync(d_gframes, gframes.data(), fbytes, cudaMemcpyHostToDevice, ctx->stream));
    SD_CUDA(ctx, cudaMemsetAsync(d_miss, 0, G, ctx->stream));
    SD_CUDA(ctx, cudaEventRecord(ctx->stage_done[0], ctx->stream));
    SD_CUDA(ctx, cudaEventRecord(ctx->stage_done[1], ctx->stream));
    const HostFrame& f0 = frames[group_frame[0]];
    int buf = 0;
    for (size_t c = 0; c + 1 < chunk_first.size(); ++c, buf ^= 1) {
        const int first = chunk_first[c], n = chunk_first[c + 1] - first;
        SD_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->stage_done[buf], 0));   // also orders the table uploads before the first gather
        const int blocks = n < 8 * ctx->sm_count ? n : 8 * ctx->sm_count;
        if (chunk_gray[c]) {
            roi_gather_kernel<1><<<blocks, 256, 0, ctx->copy_stream>>>(d_src, d_roi, first, n, (uint8_t*)ctx->d_stage[buf]);
            SD_LAUNCH_CHECK(ctx, "roi_gather_kernel");
        }
        if (chunk_colour[c]) {
            roi_gather_kernel<3><<<blocks, 256, 0, ctx->copy_stream>>>(d_src, d_roi, first, n, (uint8_t*)ctx->d_stage[buf]);
            SD_LAUNCH_CHECK(ctx, "roi_gather_kernel");
        }
        SD_CUDA(ctx, cudaEventRecord(ctx->stage_ev[buf], ctx->copy_stream));
        SD_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->stage_ev[buf], 0));
        sd_image_batch ib{};
        ib.d_data = (const uint8_t*)ctx->d_stage[buf];
        ib.width = f0.width; ib.height = f0.height; ib.row_stride = f0.row_stride; ib.image_stride = 0; ib.count = n;
        ib.d_roi = d_roi + first;
        ib.d_roi_miss = d_miss + first;
        if (fbytes) ib.d_frames = d_gframes + first;
        const int k0 = gface0[first], nf = gface0[first + n] - k0;
        rc = detect_device(ctx, m, &ib, identity ? nullptr : d_idx + k0, d_x + (size_t)k0 * P, nf, d_out + (size_t)k0 * P);
        if (rc) return rc;
        SD_CUDA(ctx, cudaEventRecord(ctx->stage_done[buf], ctx->stream));
    }
    std::vector<uint8_t> miss(G);
    SD_CUDA(ctx, cudaMemcpyAsync(out, d_out, xbytes, cudaMemcpyDeviceToHost, ctx->stream));
    SD_CUDA(ctx, cudaMemcpyAsync(miss.data(), d_miss, G, cudaMemcpyDeviceToHost, ctx->stream));
    rc = sd_check_hog_status(ctx, "detect");             // synchronises
    if (rc) return rc;
    // groups whose cascade wandered outside the uploaded region: repeat their faces from the full frame, uploaded once
    for (int g = 0; g < G; ++g) {
        if (!miss[g]) continue;
        const int k0 = gface0[g], nf = gface0[g + 1] - k0;
        ctx->roi_fallbacks += nf;
        const std::vector<int> zero(nf, 0);
        rc = detect_host_full(ctx, m, &frames[group_frame[g]], zero.data(), x0 + (size_t)k0 * P, nf, out + (size_t)k0 * P);
        if (rc) return rc;
    }
    if (!identity)
        for (int k = 0; k < count; ++k) memcpy(h_out + (size_t)pos[k] * P, &gout[(size_t)k * P], P * sizeof(float));
    return SD_OK;
}

// detect(image, facebox) (h_boxes) or detect(image, initialisation) (h_x0, row stride ldx floats) for count faces; face i in
// frames[frame_index ? frame_index[i] : i] (indices already validated).  Faces are taken frame by frame (stable), their
// initial landmarks aligned on the host (model.hpp:135) or copied.
int detect_host(sd_ctx* ctx, const sd_model* m, const std::vector<HostFrame>& frames, const int32_t* frame_index, const int32_t* h_boxes,
                const float* h_x0, int64_t ldx, int count, float* h_landmarks, bool roi)
{
    const int L = m->num_landmarks, P = 2 * L;
    const int F = (int)frames.size();
    std::vector<int> order(count), fidx(count);
    if (frame_index) {
        std::vector<int> start(F + 1, 0);
        for (int i = 0; i < count; ++i) start[frame_index[i] + 1]++;
        for (int f = 0; f < F; ++f) start[f + 1] += start[f];
        for (int i = 0; i < count; ++i) order[start[frame_index[i]]++] = i;
        for (int k = 0; k < count; ++k) fidx[k] = frame_index[order[k]];
    } else {
        for (int i = 0; i < count; ++i) order[i] = fidx[i] = i;
    }
    bool identity = true;
    for (int k = 0; k < count && identity; ++k) identity = order[k] == k;
    std::vector<float> x0((size_t)count * P), sorted_out;
    for (int k = 0; k < count; ++k) {
        if (h_boxes) {
            const int32_t* b = h_boxes + 4 * (size_t)order[k];
            sd_align_mean(m->mean.data(), L, b[0], b[1], b[2], b[3], 1.f, 1.f, 0.f, 0.f, &x0[(size_t)k * P]);
        } else {
            memcpy(&x0[(size_t)k * P], h_x0 + (size_t)order[k] * ldx, P * sizeof(float));
        }
    }
    float* out = h_landmarks;
    if (!identity) { sorted_out.resize((size_t)count * P); out = sorted_out.data(); }
    const int rc = roi ? detect_host_roi(ctx, m, frames.data(), fidx.data(), x0.data(), count, out)
                       : detect_host_full(ctx, m, frames.data(), fidx.data(), x0.data(), count, out);
    if (rc) return rc;
    if (!identity)
        for (int k = 0; k < count; ++k) memcpy(h_landmarks + (size_t)order[k] * P, &sorted_out[(size_t)k * P], P * sizeof(float));
    return SD_OK;
}

// device-mapped address of a pinned host buffer, or null (pageable memory: not an error)
const uint8_t* mapped_alias(const void* h)
{
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, h) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return attr.type == cudaMemoryTypeHost ? (const uint8_t*)attr.devicePointer : nullptr;
}

// the frames of an sd_detect_faces_host(_init) call, checked: every frame index, and the size, pitch and channel count of every
// referenced frame (frames without faces are never read).  roi: every referenced frame is pinned, device-mapped and aligned.
int host_frames(sd_ctx* ctx, const char* fn, const sd_host_frame* h_frames, int num_frames, const int32_t* h_frame_index, int count,
                std::vector<HostFrame>& frames, bool& roi)
{
    std::vector<char> used(num_frames, 0);
    for (int i = 0; i < count; ++i) {
        if (h_frame_index[i] < 0 || h_frame_index[i] >= num_frames)
            return sd_fail(ctx, SD_ERR_INVALID, "%s: face %d: frame index %d is not in [0, %d)", fn, i, h_frame_index[i], num_frames);
        used[h_frame_index[i]] = 1;
    }
    frames.assign(num_frames, HostFrame{nullptr, nullptr, 0, 0, 0, 1});
    for (int f = 0; f < num_frames; ++f) {
        if (!used[f]) continue;
        const sd_host_frame& hf = h_frames[f];
        const int channels = hf.channels == 0 ? 1 : hf.channels;
        if (channels != 1 && channels != 3)
            return sd_fail(ctx, SD_ERR_INVALID, "%s: frame %d: %d channels (1 = gray or 3 = B,G,R)", fn, f, hf.channels);
        if (!hf.h_data || hf.width <= 0 || hf.height <= 0 || (int64_t)hf.row_stride < (int64_t)channels * hf.width)
            return sd_fail(ctx, SD_ERR_INVALID, "%s: frame %d: bad data pointer or size", fn, f);
        frames[f] = HostFrame{hf.h_data, nullptr, hf.width, hf.height, hf.row_stride, channels};
    }
    // ROI route when the frames are in pinned, device-mapped host memory with 16-byte aligned rows
    roi = true;
    for (int f = 0; f < num_frames && roi; ++f) {
        if (!used[f]) continue;
        const uint8_t* alias = mapped_alias(frames[f].h);
        roi = alias && ((reinterpret_cast<uintptr_t>(alias) | (uintptr_t)frames[f].row_stride) & 15) == 0;
        frames[f].d_alias = alias;
    }
    return SD_OK;
}

}  // namespace

extern "C" {

int sd_detect_batch_host(sd_ctx* ctx, const sd_model* m, const uint8_t* h_images, int count, int width, int height,
                         int row_stride, const int32_t* h_boxes, float* h_landmarks)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_REQUIRE(ctx, m && h_images && h_boxes && h_landmarks && count >= 0 && width > 0 && height > 0 && row_stride >= width, "bad argument");
    if (count == 0) return SD_OK;
    // ROI route when the frames are in pinned, device-mapped host memory with 16-byte aligned rows
    const size_t frame_bytes = (size_t)height * row_stride;
    const uint8_t* alias = mapped_alias(h_images);
    const bool aligned = alias && ((reinterpret_cast<uintptr_t>(alias) | (uintptr_t)row_stride | (uintptr_t)frame_bytes) & 15) == 0;
    std::vector<HostFrame> frames(count);
    for (int i = 0; i < count; ++i)
        frames[i] = HostFrame{h_images + i * frame_bytes, aligned ? alias + i * frame_bytes : nullptr, width, height, row_stride, 1};
    return detect_host(ctx, m, frames, nullptr, h_boxes, nullptr, 0, count, h_landmarks, aligned);
}

int sd_model_align_boxes(sd_ctx* ctx, const sd_model* m, const int32_t* d_boxes, int count, float* d_x0, int64_t ldx)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_REQUIRE(ctx, m && count >= 0 && ldx >= 2 * (int64_t)m->num_landmarks, "bad argument");
    if (count == 0) return SD_OK;
    SD_REQUIRE(ctx, d_boxes && d_x0, "null argument");
    const int L = m->num_landmarks;
    const long long total = (long long)count * 2 * L;
    align_boxes_kernel<<<sd_div_up(total, 256), 256, 0, ctx->stream>>>(m->d_mean, L, d_boxes, count, d_x0, ldx);
    SD_LAUNCH_CHECK(ctx, "align_boxes_kernel");
    return SD_OK;
}

int sd_detect_faces_device(sd_ctx* ctx, const sd_model* m, const sd_image_batch* frames, const int32_t* d_frame_index, const float* d_x0,
                           int count, float* d_landmarks)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_REQUIRE(ctx, m && frames && count >= 0, "bad argument");
    if (count == 0) return SD_OK;
    SD_REQUIRE(ctx, d_frame_index && d_x0 && d_landmarks && frames->count >= 1, "bad argument");
    SD_REQUIRE(ctx, !frames->d_roi, "d_roi is not supported here");
    const int rc = detect_device(ctx, m, frames, d_frame_index, d_x0, count, d_landmarks);
    if (rc) return rc;
    return sd_check_hog_status(ctx, "detect");               // a frame index out of range is reported here
}

int sd_detect_faces_host(sd_ctx* ctx, const sd_model* m, const sd_host_frame* h_frames, int num_frames, const int32_t* h_frame_index,
                         const int32_t* h_boxes, int count, float* h_landmarks)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_REQUIRE(ctx, m && count >= 0 && num_frames >= 0, "bad argument");
    if (count == 0) return SD_OK;
    SD_REQUIRE(ctx, h_frames && h_frame_index && h_boxes && h_landmarks && num_frames >= 1, "bad argument");
    std::vector<HostFrame> frames;
    bool roi = false;
    const int rc = host_frames(ctx, __func__, h_frames, num_frames, h_frame_index, count, frames, roi);
    if (rc) return rc;
    return detect_host(ctx, m, frames, h_frame_index, h_boxes, nullptr, 0, count, h_landmarks, roi);
}

int sd_detect_faces_host_init(sd_ctx* ctx, const sd_model* m, const sd_host_frame* h_frames, int num_frames, const int32_t* h_frame_index,
                              const float* h_x0, int64_t ldx, int count, float* h_landmarks)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_REQUIRE(ctx, m && count >= 0 && num_frames >= 0, "bad argument");
    if (count == 0) return SD_OK;
    SD_REQUIRE(ctx, h_frames && h_frame_index && h_x0 && h_landmarks && num_frames >= 1 && ldx >= 2 * (int64_t)m->num_landmarks,
               "bad argument");
    std::vector<HostFrame> frames;
    bool roi = false;
    const int rc = host_frames(ctx, __func__, h_frames, num_frames, h_frame_index, count, frames, roi);
    if (rc) return rc;
    return detect_host(ctx, m, frames, h_frame_index, nullptr, h_x0, ldx, count, h_landmarks, roi);
}

}  // extern "C"
