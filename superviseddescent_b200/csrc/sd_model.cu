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
    SD_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SD_OK;
}

int detect_device(sd_ctx* ctx, const sd_model* m, const sd_image_batch* images, const float* d_x0, int count,
                  float* d_landmarks)
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
        int rc = sd_hog_batch(ctx, images, nullptr, cur, P, count, L, &m->norm, &m->hog[s], A, ld);
        if (rc) return rc;
        rc = sd_cascade_update(ctx, A, ld, count, m->rows[s], m->d_weights[s], P, cur, &m->norm, nxt);
        if (rc) return rc;
        float* t = cur; cur = nxt; nxt = t;
    }
    SD_CUDA(ctx, cudaMemcpyAsync(d_landmarks, cur, (size_t)count * P * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
    return SD_OK;
}


// ---- region-of-interest upload (sd_detect_batch_host) ------------------------------------------------
// The cascade only ever reads a neighbourhood of the face, so instead of copying whole 640x480 frames over
// PCIe a small kernel pulls the ROI rows of every face straight out of the caller's PINNED host buffer
// (zero-copy loads through the unified address space, 16-byte vectors) into a packed device buffer.  If a
// patch later needs a frame pixel outside its ROI the HOG kernel raises d_roi_miss[face] and that face is
// repeated from its full frame, so the result never depends on the ROI heuristic.
__global__ void __launch_bounds__(256) roi_gather_kernel(const uint8_t* __restrict__ h_frames, long long frame_bytes, int row_stride,
                                                         const sd_roi* __restrict__ roi, int first, int n, uint8_t* __restrict__ dst)
{
    for (int f = blockIdx.x; f < n; f += gridDim.x) {
        const sd_roi r = roi[first + f];
        const uint8_t* src = h_frames + (long long)(first + f) * frame_bytes + (long long)r.y * row_stride + r.x;
        uint8_t* d = dst + r.offset;
        const int vec_per_row = r.row_stride >> 4;
        const int total = vec_per_row * r.h;
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

// conservative ROI of one face: landmark bounding box of the initialisation, grown by the largest patch
// half size of the schedule plus a drift allowance, clipped to the frame, x aligned to 16 bytes
sd_roi face_roi(const sd_model* m, const float* x0, int width, int height, int row_stride)
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
    const int maxw = (row_stride - r.x) & ~15;
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
    const int rc = detect_device(ctx, m, images, d_x0, count, d_landmarks);
    if (rc) return rc;
    // a degenerate face (inter-eye distance too small for a patch) or a bad frame index is an error here, as it is in the
    // reference (cv::resize on an empty ROI throws); reading the flag synchronises the stream
    return sd_check_hog_status(ctx, "detect");
}

static int detect_host_full(sd_ctx* ctx, const sd_model* m, const uint8_t* h_images, int count, int width, int height,
                            int row_stride, const int32_t* h_boxes, float* h_landmarks)
{
    const int L = m->num_landmarks, P = 2 * L;
    const size_t frame_bytes = (size_t)height * row_stride;
    // chunking: ~128 MB of frames per staging buffer, at least 1 face
    int chunk = (int)((size_t)(128u << 20) / frame_bytes);
    if (chunk < 1) chunk = 1;
    if (chunk > count) chunk = count;
    for (int b = 0; b < 2; ++b) {
        if (ctx->stage_bytes[b] < (size_t)chunk * frame_bytes) {
            if (ctx->d_stage[b]) { SD_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); SD_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream)); SD_CUDA(ctx, cudaFree(ctx->d_stage[b])); ctx->d_stage[b] = nullptr; }
            SD_CUDA(ctx, cudaMalloc(&ctx->d_stage[b], (size_t)chunk * frame_bytes));
            ctx->stage_bytes[b] = (size_t)chunk * frame_bytes;
        }
    }
    // initial landmarks for every face: align_mean on the host (model.hpp:135), one small upload
    std::vector<float> x0((size_t)count * P);
    for (int i = 0; i < count; ++i)
        sd_align_mean(m->mean.data(), L, h_boxes[4 * i], h_boxes[4 * i + 1], h_boxes[4 * i + 2], h_boxes[4 * i + 3], 1.f, 1.f, 0.f, 0.f, &x0[(size_t)i * P]);
    float* d_x = (float*)sd_workspace(ctx, SD_WS_PARTIAL, (size_t)2 * count * P * sizeof(float));
    if (!d_x) return SD_ERR_CUDA;
    float* d_out = d_x + (size_t)count * P;
    SD_CUDA(ctx, cudaMemcpyAsync(d_x, x0.data(), x0.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    // the copy stream must not run ahead of work already queued on the compute stream that still reads the staging buffers
    SD_CUDA(ctx, cudaEventRecord(ctx->stage_done[0], ctx->stream));
    SD_CUDA(ctx, cudaEventRecord(ctx->stage_done[1], ctx->stream));
    int buf = 0;
    for (int first = 0; first < count; first += chunk, buf ^= 1) {
        const int n = (count - first < chunk) ? count - first : chunk;
        SD_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->stage_done[buf], 0));
        SD_CUDA(ctx, cudaMemcpyAsync(ctx->d_stage[buf], h_images + (size_t)first * frame_bytes, (size_t)n * frame_bytes,
                                     cudaMemcpyHostToDevice, ctx->copy_stream));
        SD_CUDA(ctx, cudaEventRecord(ctx->stage_ev[buf], ctx->copy_stream));
        SD_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->stage_ev[buf], 0));
        sd_image_batch ib{};
        ib.d_data = (const uint8_t*)ctx->d_stage[buf];
        ib.width = width; ib.height = height; ib.row_stride = row_stride; ib.image_stride = (int64_t)frame_bytes; ib.count = n;
        int rc = detect_device(ctx, m, &ib, d_x + (size_t)first * P, n, d_out + (size_t)first * P);
        if (rc) return rc;
        SD_CUDA(ctx, cudaEventRecord(ctx->stage_done[buf], ctx->stream));
    }
    SD_CUDA(ctx, cudaMemcpyAsync(h_landmarks, d_out, (size_t)count * P * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    return sd_check_hog_status(ctx, "detect");                // synchronises
}

// ROI route: needs the caller's frames in pinned (device-mapped) host memory
static int detect_host_roi(sd_ctx* ctx, const sd_model* m, const uint8_t* h_images, const uint8_t* d_alias, int count, int width,
                           int height, int row_stride, const int32_t* h_boxes, float* h_landmarks)
{
    const int L = m->num_landmarks, P = 2 * L;
    const size_t frame_bytes = (size_t)height * row_stride;
    const size_t chunk_cap = (size_t)48 << 20;            // packed ROI bytes per staging buffer
    // initial landmarks and the ROI of every face; faces are grouped into chunks that fit one staging buffer
    std::vector<float> x0((size_t)count * P);
    std::vector<sd_roi> rois(count);
    std::vector<int> chunk_first;
    size_t used = 0;
    for (int i = 0; i < count; ++i) {
        sd_align_mean(m->mean.data(), L, h_boxes[4 * i], h_boxes[4 * i + 1], h_boxes[4 * i + 2], h_boxes[4 * i + 3], 1.f, 1.f, 0.f, 0.f, &x0[(size_t)i * P]);
        sd_roi r = face_roi(m, &x0[(size_t)i * P], width, height, row_stride);
        const size_t bytes = (size_t)r.row_stride * r.h;
        if (bytes > chunk_cap)                                // a face window larger than a staging buffer: whole-frame route
            return detect_host_full(ctx, m, h_images, count, width, height, row_stride, h_boxes, h_landmarks);
        if (chunk_first.empty() || used + bytes > chunk_cap) { chunk_first.push_back(i); used = 0; }
        r.offset = (int64_t)used;
        used += bytes;
        rois[i] = r;
    }
    chunk_first.push_back(count);
    for (int b = 0; b < 2; ++b) {
        if (ctx->stage_bytes[b] < chunk_cap + (1u << 20)) {
            if (ctx->d_stage[b]) { SD_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); SD_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream)); SD_CUDA(ctx, cudaFree(ctx->d_stage[b])); ctx->d_stage[b] = nullptr; }
            SD_CUDA(ctx, cudaMalloc(&ctx->d_stage[b], chunk_cap + (1u << 20)));
            ctx->stage_bytes[b] = chunk_cap + (1u << 20);
        }
    }
    // device tables: landmarks (in, out), ROI records, miss flags
    const size_t xbytes = (size_t)count * P * sizeof(float);
    const size_t rbytes = (size_t)count * sizeof(sd_roi);
    unsigned char* tab = (unsigned char*)sd_workspace(ctx, SD_WS_PARTIAL, 2 * xbytes + rbytes + count + 64);
    if (!tab) return SD_ERR_CUDA;
    float* d_x = (float*)tab;
    float* d_out = (float*)(tab + xbytes);
    sd_roi* d_roi = (sd_roi*)(tab + 2 * xbytes);
    uint8_t* d_miss = tab + 2 * xbytes + rbytes;
    SD_CUDA(ctx, cudaMemcpyAsync(d_x, x0.data(), xbytes, cudaMemcpyHostToDevice, ctx->stream));
    SD_CUDA(ctx, cudaMemcpyAsync(d_roi, rois.data(), rbytes, cudaMemcpyHostToDevice, ctx->stream));
    SD_CUDA(ctx, cudaMemsetAsync(d_miss, 0, count, ctx->stream));
    SD_CUDA(ctx, cudaEventRecord(ctx->stage_done[0], ctx->stream));
    SD_CUDA(ctx, cudaEventRecord(ctx->stage_done[1], ctx->stream));
    int buf = 0;
    for (size_t c = 0; c + 1 < chunk_first.size(); ++c, buf ^= 1) {
        const int first = chunk_first[c], n = chunk_first[c + 1] - first;
        SD_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->stage_done[buf], 0));   // also orders the table uploads before the first gather
        const int blocks = n < 8 * ctx->sm_count ? n : 8 * ctx->sm_count;
        roi_gather_kernel<<<blocks, 256, 0, ctx->copy_stream>>>(d_alias, (long long)frame_bytes, row_stride, d_roi, first, n, (uint8_t*)ctx->d_stage[buf]);
        SD_LAUNCH_CHECK(ctx, "roi_gather_kernel");
        SD_CUDA(ctx, cudaEventRecord(ctx->stage_ev[buf], ctx->copy_stream));
        SD_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->stage_ev[buf], 0));
        sd_image_batch ib{};
        ib.d_data = (const uint8_t*)ctx->d_stage[buf];
        ib.width = width; ib.height = height; ib.row_stride = row_stride; ib.image_stride = 0; ib.count = n;
        ib.d_roi = d_roi + first;
        ib.d_roi_miss = d_miss + first;
        int rc = detect_device(ctx, m, &ib, d_x + (size_t)first * P, n, d_out + (size_t)first * P);
        if (rc) return rc;
        SD_CUDA(ctx, cudaEventRecord(ctx->stage_done[buf], ctx->stream));
    }
    std::vector<uint8_t> miss(count);
    SD_CUDA(ctx, cudaMemcpyAsync(h_landmarks, d_out, xbytes, cudaMemcpyDeviceToHost, ctx->stream));
    SD_CUDA(ctx, cudaMemcpyAsync(miss.data(), d_miss, count, cudaMemcpyDeviceToHost, ctx->stream));
    {
        const int rc = sd_check_hog_status(ctx, "detect");    // synchronises
        if (rc) return rc;
    }
    // faces whose cascade wandered outside the uploaded region: repeat them from their full frames
    for (int i = 0; i < count; ++i) {
        if (!miss[i]) continue;
        ctx->roi_fallbacks++;
        int rc = detect_host_full(ctx, m, h_images + (size_t)i * frame_bytes, 1, width, height, row_stride, h_boxes + 4 * i, h_landmarks + (size_t)i * P);
        if (rc) return rc;
    }
    return SD_OK;
}

int sd_detect_batch_host(sd_ctx* ctx, const sd_model* m, const uint8_t* h_images, int count, int width, int height,
                         int row_stride, const int32_t* h_boxes, float* h_landmarks)
{
    if (!ctx) return SD_ERR_INVALID;
    SD_REQUIRE(ctx, m && h_images && h_boxes && h_landmarks && count >= 0 && width > 0 && height > 0 && row_stride >= width, "bad argument");
    if (count == 0) return SD_OK;
    // ROI route when the frames are in pinned, device-mapped host memory with 16-byte aligned rows
    const size_t frame_bytes = (size_t)height * row_stride;
    cudaPointerAttributes attr;
    const bool pinned = cudaPointerGetAttributes(&attr, h_images) == cudaSuccess && attr.type == cudaMemoryTypeHost && attr.devicePointer;
    if (!pinned) cudaGetLastError();
    const bool aligned = pinned && ((reinterpret_cast<uintptr_t>(attr.devicePointer) | (uintptr_t)row_stride | (uintptr_t)frame_bytes) & 15) == 0;
    if (aligned)
        return detect_host_roi(ctx, m, h_images, (const uint8_t*)attr.devicePointer, count, width, height, row_stride, h_boxes, h_landmarks);
    return detect_host_full(ctx, m, h_images, count, width, height, row_stride, h_boxes, h_landmarks);
}

}  // extern "C"
