// B200 drop-in for include/rcr/model.hpp: align_mean (:64-76), InterEyeDistanceNormalisation (:84-116),
// detection_model (:122-183) and load/save_detection_model (:192-219).  detect() runs the whole cascade
// on the GPU through sd_detect_batch_host / sd_detect_faces_host(_init), reading host frames in place (8UC1, or 8UC3 B,G,R
// converted on the device); the file format is byte compatible with the reference's
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
        const cv::Mat x0 = initialisation.isContinuous() ? initialisation : initialisation.clone();
        if (x0.rows * x0.cols != 2 * sd_model_num_landmarks(handle.get())) throw std::runtime_error("detect: the initialisation needs 2L values");
        const std::vector<float> lms = detect_host(std::vector<cv::Mat>{image}, std::vector<int32_t>{0}, nullptr, x0.ptr<float>(0));
        cv::Mat row(1, static_cast<int>(lms.size()), CV_32FC1);
        std::memcpy(row.ptr<float>(0), lms.data(), sizeof(float) * lms.size());
        return to_landmark_collection(row, landmark_ids);
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
        std::vector<int32_t> boxes(static_cast<size_t>(n) * 4);
        for (int i = 0; i < n; ++i) {
            if (images[i].cols != w || images[i].rows != h) throw std::runtime_error("detect: the batched path needs equally sized images");
            colour = colour || images[i].channels() == 3;
            boxes[4 * i] = faceboxes[i].x; boxes[4 * i + 1] = faceboxes[i].y; boxes[4 * i + 2] = faceboxes[i].width; boxes[4 * i + 3] = faceboxes[i].height;
        }
        std::vector<float> lms;
        if (colour) {
            // colour frames (8UC3 B,G,R) are read in place and converted to gray on the device (sd_detect_faces_host)
            std::vector<int32_t> index(n);
            for (int i = 0; i < n; ++i) index[i] = i;
            lms = detect_host(images, index, boxes.data(), nullptr);
        } else {
            std::vector<unsigned char> frames(static_cast<size_t>(n) * w * h);
            for (int i = 0; i < n; ++i) {
                const cv::Mat& g = images[i];
                for (int y = 0; y < h; ++y) std::memcpy(&frames[(static_cast<size_t>(i) * h + y) * w], g.ptr<unsigned char>(y), w);
            }
            lms.resize(static_cast<size_t>(n) * P);
            sd_b200::check(ctx, sd_detect_batch_host(ctx, handle.get(), frames.data(), n, w, h, w, boxes.data(), lms.data()), "sd_detect_batch_host");
        }
        std::vector<cv::Mat> out;
        for (int i = 0; i < n; ++i) {
            cv::Mat row(1, P, CV_32FC1);
            std::memcpy(row.ptr<float>(0), &lms[static_cast<size_t>(i) * P], sizeof(float) * P);
            out.push_back(row);
        }
        return out;
    }

    // Several faces per frame, frames of any sizes (the box list a face detector such as detectMultiScale returns for each
    // frame): result[i][j] holds the landmarks of faceboxes[i][j] in images[i].  Frames, gray or colour (8UC3 B,G,R), are read
    // in place through their own row pointers (sd_detect_faces_host).
    std::vector<std::vector<LandmarkCollection<cv::Vec2f>>> detect(const std::vector<cv::Mat>& images, const std::vector<std::vector<cv::Rect>>& faceboxes)
    {
        if (images.size() != faceboxes.size()) throw std::runtime_error("detect: images / faceboxes size mismatch");
        std::vector<int32_t> index, boxes;
        for (size_t i = 0; i < images.size(); ++i)
            for (const cv::Rect& b : faceboxes[i]) {
                index.push_back(static_cast<int32_t>(i));
                boxes.push_back(b.x); boxes.push_back(b.y); boxes.push_back(b.width); boxes.push_back(b.height);
            }
        return per_frame(images.size(), faceboxes, detect_host(images, index, boxes.data(), nullptr));
    }

    // Several tracked faces per frame (detect(image, initialisation) for each): result[i][j] holds the landmarks of the face
    // that starts from initialisations[i][j] (1 x 2L, e.g. its landmarks in the previous frame) in images[i].
    std::vector<std::vector<LandmarkCollection<cv::Vec2f>>> detect(const std::vector<cv::Mat>& images, const std::vector<std::vector<cv::Mat>>& initialisations)
    {
        if (images.size() != initialisations.size()) throw std::runtime_error("detect: images / initialisations size mismatch");
        const size_t P = 2 * static_cast<size_t>(sd_model_num_landmarks(handle.get()));
        std::vector<int32_t> index;
        std::vector<float> x0;
        for (size_t i = 0; i < images.size(); ++i)
            for (const cv::Mat& init : initialisations[i]) {
                if (static_cast<size_t>(init.rows) * init.cols != P) throw std::runtime_error("detect: an initialisation needs 2L values");
                const cv::Mat row = init.isContinuous() ? init : init.clone();
                index.push_back(static_cast<int32_t>(i));
                x0.insert(x0.end(), row.ptr<float>(0), row.ptr<float>(0) + P);
            }
        return per_frame(images.size(), initialisations, detect_host(images, index, nullptr, x0.data()));
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
    // Every face of `index` (the frame of each face) through sd_detect_faces_host (boxes: 4 per face) or sd_detect_faces_host_init
    // (x0: 2L per face); returns count x 2L.  Frames are read in place through their own pointer and pitch; colour frames (8UC3
    // B,G,R) are converted on the device as cv::cvtColor(BGR2GRAY) of adaptive_vlhog.hpp:115-117 would.
    std::vector<float> detect_host(const std::vector<cv::Mat>& images, const std::vector<int32_t>& index, const int32_t* boxes, const float* x0)
    {
        sd_ctx* ctx = sd_b200::context();
        const int P = 2 * sd_model_num_landmarks(handle.get());
        const int count = static_cast<int>(index.size());
        std::vector<float> lms(static_cast<size_t>(count) * P);
        if (count == 0) return lms;
        std::vector<sd_host_frame> frames(images.size(), sd_host_frame{nullptr, 0, 0, 0, 0});
        for (int32_t i : index) {
            const cv::Mat& im = images[i];
            if (im.empty()) throw std::runtime_error("detect: empty image with faces");
            frames[i] = sd_host_frame{im.ptr<unsigned char>(0), im.cols, im.rows, static_cast<int32_t>(im.step()), im.channels()};
        }
        if (boxes)
            sd_b200::check(ctx, sd_detect_faces_host(ctx, handle.get(), frames.data(), static_cast<int>(frames.size()), index.data(), boxes, count,
                                                     lms.data()), "sd_detect_faces_host");
        else
            sd_b200::check(ctx, sd_detect_faces_host_init(ctx, handle.get(), frames.data(), static_cast<int>(frames.size()), index.data(), x0, P,
                                                          count, lms.data()), "sd_detect_faces_host_init");
        return lms;
    }

    // count x 2L landmark rows, faces in frame order -> one list of landmark collections per frame
    template <class PerFrame>
    std::vector<std::vector<LandmarkCollection<cv::Vec2f>>> per_frame(size_t num_frames, const std::vector<PerFrame>& faces, const std::vector<float>& lms)
    {
        const size_t P = 2 * static_cast<size_t>(sd_model_num_landmarks(handle.get()));
        std::vector<std::vector<LandmarkCollection<cv::Vec2f>>> out(num_frames);
        size_t k = 0;
        for (size_t i = 0; i < num_frames; ++i)
            for (size_t j = 0; j < faces[i].size(); ++j, ++k) {
                cv::Mat row(1, static_cast<int>(P), CV_32FC1);
                std::memcpy(row.ptr<float>(0), &lms[k * P], sizeof(float) * P);
                out[i].push_back(to_landmark_collection(row, landmark_ids));
            }
        return out;
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
