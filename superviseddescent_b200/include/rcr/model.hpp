// B200 drop-in for include/rcr/model.hpp: align_mean (:64-76), InterEyeDistanceNormalisation (:84-116),
// detection_model (:122-183) and load/save_detection_model (:192-219).  detect() runs the whole cascade
// on the GPU through sd_detect_batch_host; the file format is byte compatible with the reference's
// cereal archives (face_landmarks_model_rcr_22.bin loads unchanged).
#pragma once

#include <string>
#include <vector>

#include "rcr/adaptive_vlhog.hpp"
#include "rcr/helpers.hpp"
#include "superviseddescent/superviseddescent.hpp"
#include "superviseddescent/verbose_solver.hpp"

namespace rcr {

inline cv::Mat align_mean(cv::Mat mean, cv::Rect facebox, float scaling_x = 1.0f, float scaling_y = 1.0f, float translation_x = 0.0f, float translation_y = 0.0f)
{
    cv::Mat aligned(1, mean.cols, CV_32FC1);
    const int rc = sd_align_mean(mean.ptr<float>(0), mean.cols / 2, facebox.x, facebox.y, facebox.width, facebox.height, scaling_x, scaling_y,
                                 translation_x, translation_y, aligned.ptr<float>(0));
    if (rc != SD_OK) throw std::runtime_error("align_mean: bad arguments");
    return aligned;
}

class InterEyeDistanceNormalisation {
public:
    InterEyeDistanceNormalisation() = default;
    InterEyeDistanceNormalisation(std::vector<std::string> modelLandmarksList, std::vector<std::string> rightEyeIdentifiers, std::vector<std::string> leftEyeIdentifiers)
        : modelLandmarksList(modelLandmarksList), rightEyeIdentifiers(rightEyeIdentifiers), leftEyeIdentifiers(leftEyeIdentifiers) {}

    // 1 / IED of the given landmark row, replicated (model.hpp:94-98)
    inline cv::Mat operator()(cv::Mat params)
    {
        const double ied = get_ied(to_landmark_collection(params, modelLandmarksList), rightEyeIdentifiers, leftEyeIdentifiers);
        const float n = static_cast<float>(1.0 / ied);
        cv::Mat out(1, params.cols, CV_32FC1);
        for (int i = 0; i < params.cols; ++i) out.at<float>(0, i) = n;
        return out;
    }

    sd_normalisation c_normalisation() const
    {
        sd_normalisation nrm{};
        nrm.kind = 1;
        const auto r = eye_indices(modelLandmarksList, rightEyeIdentifiers, "right");
        const auto l = eye_indices(modelLandmarksList, leftEyeIdentifiers, "left");
        nrm.n_right = static_cast<int>(r.size());
        nrm.n_left = static_cast<int>(l.size());
        for (size_t i = 0; i < r.size() && i < 4; ++i) nrm.right_idx[i] = r[i];
        for (size_t i = 0; i < l.size() && i < 4; ++i) nrm.left_idx[i] = l[i];
        return nrm;
    }

private:
    std::vector<std::string> modelLandmarksList, rightEyeIdentifiers, leftEyeIdentifiers;
};

class detection_model {
public:
    using model_type = superviseddescent::SupervisedDescentOptimiser<superviseddescent::LinearRegressor<superviseddescent::VerbosePartialPivLUSolver>, InterEyeDistanceNormalisation>;

    detection_model() = default;

    // model.hpp:128-129: a model assembled from a trained optimiser
    detection_model(model_type optimised_model, cv::Mat mean, std::vector<std::string> landmark_ids, std::vector<rcr::HoGParam> hog_params,
                    std::vector<std::string> right_eye_ids, std::vector<std::string> left_eye_ids)
        : landmark_ids(landmark_ids)
    {
        auto& regs = optimised_model.get_regressors();
        std::vector<const float*> w;
        std::vector<sd_regulariser> r;
        std::vector<sd_hog_param> hp;
        std::vector<cv::Mat> keep;
        for (size_t i = 0; i < regs.size(); ++i) {
            keep.push_back(regs[i].x.isContinuous() ? regs[i].x : regs[i].x.clone());
            w.push_back(keep.back().ptr<float>(0));
            r.push_back(regs[i].get_regulariser().c());
            hp.push_back(hog_params[i].c());
        }
        std::vector<const char*> ids, rid, lid;
        for (auto& s : landmark_ids) ids.push_back(s.c_str());
        for (auto& s : right_eye_ids) rid.push_back(s.c_str());
        for (auto& s : left_eye_ids) lid.push_back(s.c_str());
        sd_ctx* ctx = sd_b200::context();
        sd_model* m = nullptr;
        sd_b200::check(ctx, sd_model_create(ctx, static_cast<int>(regs.size()), static_cast<int>(landmark_ids.size()), w.data(), r.data(), hp.data(),
                                            mean.ptr<float>(0), ids.data(), rid.data(), static_cast<int>(rid.size()), lid.data(), static_cast<int>(lid.size()), &m),
                       "sd_model_create");
        handle.reset(m, sd_model_destroy);
    }

    // Run the model from a face box: init with the aligned mean, then optimise (model.hpp:132-144)
    LandmarkCollection<cv::Vec2f> detect(cv::Mat image, cv::Rect facebox)
    {
        std::vector<cv::Mat> out = detect(std::vector<cv::Mat>{image}, std::vector<cv::Rect>{facebox});
        return to_landmark_collection(out[0], landmark_ids);
    }

    // Run the model from a landmark initialisation, e.g. the previous frame (model.hpp:147-157)
    LandmarkCollection<cv::Vec2f> detect(cv::Mat image, cv::Mat initialisation)
    {
        sd_ctx* ctx = sd_b200::context();
        const cv::Mat& gray = image;               // size only; colour frames are converted on the device
        const size_t frame = static_cast<size_t>(gray.cols) * gray.rows;
        sd_b200::DeviceBuffer dimg(frame), dx, dout(static_cast<size_t>(initialisation.cols) * sizeof(float)), bgr;
        upload_gray(ctx, image, dimg.as<unsigned char>(), bgr);
        sd_b200::upload(initialisation, dx, initialisation.cols);
        sd_image_batch ib{};
        ib.d_data = dimg.as<unsigned char>(); ib.width = gray.cols; ib.height = gray.rows; ib.row_stride = gray.cols; ib.image_stride = static_cast<int64_t>(frame); ib.count = 1;
        sd_b200::check(ctx, sd_detect_batch_device(ctx, handle.get(), &ib, dx.as<float>(), 1, dout.as<float>()), "sd_detect_batch_device");
        return to_landmark_collection(sd_b200::download(dout.as<float>(), 1, initialisation.cols, initialisation.cols), landmark_ids);
    }

    // Batched detect: equally sized frames, one face box each; returns one 1 x 2L row per frame.
    std::vector<cv::Mat> detect(const std::vector<cv::Mat>& images, const std::vector<cv::Rect>& faceboxes)
    {
        if (images.empty() || images.size() != faceboxes.size()) throw std::runtime_error("detect: images / faceboxes size mismatch");
        sd_ctx* ctx = sd_b200::context();
        const int n = static_cast<int>(images.size());
        const int w = images[0].cols, h = images[0].rows;
        const int P = 2 * sd_model_num_landmarks(handle.get());
        bool colour = false;
        for (int i = 0; i < n; ++i) {
            if (images[i].cols != w || images[i].rows != h) throw std::runtime_error("detect: the batched path needs equally sized images");
            colour = colour || images[i].channels() == 3;
        }
        if (colour) {
            // colour frames: upload B,G,R, convert on the device (sd_bgr2gray), start from the aligned mean, stay on the device
            const size_t frame = static_cast<size_t>(w) * h;
            sd_b200::DeviceBuffer dimg(frame * n), dx(static_cast<size_t>(n) * P * sizeof(float)), dout(static_cast<size_t>(n) * P * sizeof(float)), bgr;
            std::vector<float> x0(static_cast<size_t>(n) * P);
            const cv::Mat mean = get_mean();
            for (int i = 0; i < n; ++i) {
                upload_gray(ctx, images[i], dimg.as<unsigned char>() + i * frame, bgr);
                sd_b200::check(ctx, sd_align_mean(mean.ptr<float>(0), P / 2, faceboxes[i].x, faceboxes[i].y, faceboxes[i].width, faceboxes[i].height,
                                                  1.f, 1.f, 0.f, 0.f, &x0[static_cast<size_t>(i) * P]), "sd_align_mean");
            }
            sd_b200::check(ctx, sd_memcpy_h2d(ctx, dx.as<float>(), x0.data(), x0.size() * sizeof(float)), "detect");
            sd_image_batch ib{};
            ib.d_data = dimg.as<unsigned char>(); ib.width = w; ib.height = h; ib.row_stride = w; ib.image_stride = static_cast<int64_t>(frame); ib.count = n;
            sd_b200::check(ctx, sd_detect_batch_device(ctx, handle.get(), &ib, dx.as<float>(), n, dout.as<float>()), "sd_detect_batch_device");
            const cv::Mat all = sd_b200::download(dout.as<float>(), n, P, P);
            std::vector<cv::Mat> rows;
            for (int i = 0; i < n; ++i) rows.push_back(all.row(i).clone());
            return rows;
        }
        std::vector<unsigned char> frames(static_cast<size_t>(n) * w * h);
        std::vector<int32_t> boxes(static_cast<size_t>(n) * 4);
        for (int i = 0; i < n; ++i) {
            const cv::Mat& g = images[i];
            for (int y = 0; y < h; ++y) std::memcpy(&frames[(static_cast<size_t>(i) * h + y) * w], g.ptr<unsigned char>(y), w);
            boxes[4 * i] = faceboxes[i].x; boxes[4 * i + 1] = faceboxes[i].y; boxes[4 * i + 2] = faceboxes[i].width; boxes[4 * i + 3] = faceboxes[i].height;
        }
        std::vector<float> lms(static_cast<size_t>(n) * P);
        sd_b200::check(ctx, sd_detect_batch_host(ctx, handle.get(), frames.data(), n, w, h, w, boxes.data(), lms.data()), "sd_detect_batch_host");
        std::vector<cv::Mat> out;
        for (int i = 0; i < n; ++i) {
            cv::Mat row(1, P, CV_32FC1);
            std::memcpy(row.ptr<float>(0), &lms[static_cast<size_t>(i) * P], sizeof(float) * P);
            out.push_back(row);
        }
        return out;
    }

    // Several faces per frame, frames of any sizes (the box list a face detector such as detectMultiScale returns for each
    // frame): result[i][j] holds the landmarks of faceboxes[i][j] in images[i].  Gray frames are read in place through their
    // own row pointers (sd_detect_faces_host); if any frame with faces is colour, the frames go to the device, are converted
    // there (sd_bgr2gray) and the boxes are aligned there (sd_model_align_boxes, sd_detect_faces_device).
    std::vector<std::vector<LandmarkCollection<cv::Vec2f>>> detect(const std::vector<cv::Mat>& images, const std::vector<std::vector<cv::Rect>>& faceboxes)
    {
        if (images.size() != faceboxes.size()) throw std::runtime_error("detect: images / faceboxes size mismatch");
        sd_ctx* ctx = sd_b200::context();
        const int P = 2 * sd_model_num_landmarks(handle.get());
        std::vector<int32_t> index, boxes;
        bool colour = false;
        for (size_t i = 0; i < images.size(); ++i) {
            if (faceboxes[i].empty()) continue;
            if (images[i].empty()) throw std::runtime_error("detect: empty image with face boxes");
            colour = colour || images[i].channels() == 3;
            for (const cv::Rect& b : faceboxes[i]) {
                index.push_back(static_cast<int32_t>(i));
                boxes.push_back(b.x); boxes.push_back(b.y); boxes.push_back(b.width); boxes.push_back(b.height);
            }
        }
        const int count = static_cast<int>(index.size());
        std::vector<float> lms(static_cast<size_t>(count) * P);
        if (count > 0 && !colour) {
            std::vector<sd_host_frame> frames(images.size());
            for (size_t i = 0; i < images.size(); ++i)
                if (!faceboxes[i].empty())
                    frames[i] = sd_host_frame{images[i].ptr<unsigned char>(0), images[i].cols, images[i].rows, static_cast<int32_t>(images[i].step()), 0};
            sd_b200::check(ctx, sd_detect_faces_host(ctx, handle.get(), frames.data(), static_cast<int>(frames.size()), index.data(), boxes.data(), count,
                                                     lms.data()), "sd_detect_faces_host");
        } else if (count > 0) {
            // the frames with faces, packed on the device as 8UC1 with 16-byte aligned rows, one sd_frame record each
            std::vector<sd_frame> rec;
            std::vector<int32_t> local(images.size(), -1);
            int64_t off = 0;
            for (size_t i = 0; i < images.size(); ++i) {
                if (faceboxes[i].empty()) continue;
                const int w = images[i].cols, h = images[i].rows, stride = (w + 15) / 16 * 16;
                local[i] = static_cast<int32_t>(rec.size());
                rec.push_back(sd_frame{w, h, stride, 0, off});
                off += static_cast<int64_t>(h) * stride;
            }
            for (int32_t& f : index) f = local[f];
            sd_b200::DeviceBuffer dimg(static_cast<size_t>(off)), drec(rec.size() * sizeof(sd_frame)), didx(index.size() * sizeof(int32_t)),
                dboxes(boxes.size() * sizeof(int32_t)), dx(lms.size() * sizeof(float)), dout(lms.size() * sizeof(float)), bgr;
            for (size_t i = 0; i < images.size(); ++i)
                if (local[i] >= 0) upload_gray(ctx, images[i], dimg.as<unsigned char>() + rec[local[i]].offset, bgr, rec[local[i]].row_stride);
            sd_b200::check(ctx, sd_memcpy_h2d(ctx, drec.as<sd_frame>(), rec.data(), rec.size() * sizeof(sd_frame)), "detect");
            sd_b200::check(ctx, sd_memcpy_h2d(ctx, didx.as<int32_t>(), index.data(), index.size() * sizeof(int32_t)), "detect");
            sd_b200::check(ctx, sd_memcpy_h2d(ctx, dboxes.as<int32_t>(), boxes.data(), boxes.size() * sizeof(int32_t)), "detect");
            sd_b200::check(ctx, sd_model_align_boxes(ctx, handle.get(), dboxes.as<int32_t>(), count, dx.as<float>(), P), "sd_model_align_boxes");
            sd_image_batch ib{};
            ib.d_data = dimg.as<unsigned char>(); ib.count = static_cast<int32_t>(rec.size()); ib.d_frames = drec.as<sd_frame>();
            sd_b200::check(ctx, sd_detect_faces_device(ctx, handle.get(), &ib, didx.as<int32_t>(), dx.as<float>(), count, dout.as<float>()),
                           "sd_detect_faces_device");
            const cv::Mat all = sd_b200::download(dout.as<float>(), count, P, P);
            std::memcpy(lms.data(), all.ptr<float>(0), lms.size() * sizeof(float));
        }
        std::vector<std::vector<LandmarkCollection<cv::Vec2f>>> out(images.size());
        size_t k = 0;
        for (size_t i = 0; i < images.size(); ++i)
            for (size_t j = 0; j < faceboxes[i].size(); ++j, ++k) {
                cv::Mat row(1, P, CV_32FC1);
                std::memcpy(row.ptr<float>(0), &lms[k * P], sizeof(float) * P);
                out[i].push_back(to_landmark_collection(row, landmark_ids));
            }
        return out;
    }

    cv::Mat get_mean()
    {
        cv::Mat mean(1, 2 * sd_model_num_landmarks(handle.get()), CV_32FC1);
        sd_model_get_mean(handle.get(), mean.ptr<float>(0));
        return mean;
    }

    sd_model* native() const { return handle.get(); }

private:
    friend detection_model load_detection_model(std::string filename);
    // frame -> device as 8UC1 with rows dst_stride bytes apart (0: packed); colour frames go up as B,G,R and are converted
    // there (cv::cvtColor BGR2GRAY of adaptive_vlhog.hpp:115-117 == sd_bgr2gray)
    static void upload_gray(sd_ctx* ctx, const cv::Mat& image, unsigned char* d_dst, sd_b200::DeviceBuffer& bgr, int dst_stride = 0)
    {
        const int w = image.cols, h = image.rows;
        const size_t frame = static_cast<size_t>(w) * h;
        const size_t ds = dst_stride > 0 ? static_cast<size_t>(dst_stride) : static_cast<size_t>(w);
        if (image.channels() == 3) {
            bgr.allocate(3 * frame);
            for (int y = 0; y < h; ++y)
                sd_b200::check(ctx, sd_memcpy_h2d(ctx, bgr.as<unsigned char>() + static_cast<size_t>(y) * 3 * w, image.ptr<unsigned char>(y), 3 * static_cast<size_t>(w)), "detect upload");
            sd_b200::check(ctx, sd_bgr2gray(ctx, bgr.as<unsigned char>(), w, h, 3 * static_cast<int64_t>(w), 3 * static_cast<int64_t>(frame), 1, d_dst,
                                            static_cast<int64_t>(ds), static_cast<int64_t>(ds * h)), "sd_bgr2gray");
        } else {
            for (int y = 0; y < h; ++y)
                sd_b200::check(ctx, sd_memcpy_h2d(ctx, d_dst + static_cast<size_t>(y) * ds, image.ptr<unsigned char>(y), w), "detect upload");
        }
    }

    std::shared_ptr<sd_model> handle;
    std::vector<std::string> landmark_ids;
};

// model.hpp:192-205
inline detection_model load_detection_model(std::string filename)
{
    sd_ctx* ctx = sd_b200::context();
    sd_model* m = nullptr;
    const int rc = sd_model_load(ctx, filename.c_str(), &m);
    if (rc != SD_OK) throw std::runtime_error(sd_last_error(ctx));   // "The given model file could not be opened: ..." (model.hpp:199)
    detection_model model;
    model.handle.reset(m, sd_model_destroy);
    for (int i = 0; i < sd_model_num_landmarks(m); ++i) model.landmark_ids.emplace_back(sd_model_landmark_id(m, i));
    return model;
}

// model.hpp:214-219
inline void save_detection_model(detection_model model, std::string filename)
{
    sd_ctx* ctx = sd_b200::context();
    sd_b200::check(ctx, sd_model_save(ctx, model.native(), filename.c_str()), "save_detection_model");
}

}  // namespace rcr
