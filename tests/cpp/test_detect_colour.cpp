// rcr::detection_model::detect on colour (8UC3 B,G,R) cv::Mats through the C++14 shell.  Every overload must give the landmarks
// it gives on the gray frames (cv::cvtColor(BGR2GRAY) of the colour ones) bit for bit: detect(image, facebox),
// detect(image, initialisation), detect(images, faceboxes) with one box per frame and with a box list per frame, and
// detect(images, initialisations) with several tracked faces per frame.  Colour frames are read in place by
// sd_detect_faces_host / sd_detect_faces_host_init and converted on the device.
//
//   test_detect_colour MODEL A.bgr A.gray WA HA B.bgr B.gray WB HB  X Y W H  X Y W H  X Y W H
//     two boxes on frame A, one on frame B (raw B,G,R and 8UC1 files)
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <vector>

#include "rcr/model.hpp"

static int failures = 0;

static bool same(const rcr::LandmarkCollection<cv::Vec2f>& a, const rcr::LandmarkCollection<cv::Vec2f>& b)
{
    if (a.size() != b.size()) return false;
    for (size_t i = 0; i < a.size(); ++i)
        if (std::memcmp(&a[i].coordinates[0], &b[i].coordinates[0], sizeof(float)) != 0 ||
            std::memcmp(&a[i].coordinates[1], &b[i].coordinates[1], sizeof(float)) != 0 || a[i].name != b[i].name)
            return false;
    return true;
}

static bool same_rows(const cv::Mat& a, const cv::Mat& b)
{
    return a.cols == b.cols && std::memcmp(a.ptr<float>(0), b.ptr<float>(0), sizeof(float) * a.cols) == 0;
}

static void expect(bool ok, const char* what)
{
    if (!ok) { std::printf("FAIL %s\n", what); ++failures; }
}

static std::vector<unsigned char> read_raw(const char* path, size_t bytes)
{
    std::vector<unsigned char> v(bytes);
    std::ifstream f(path, std::ios::binary);
    f.read(reinterpret_cast<char*>(v.data()), static_cast<std::streamsize>(bytes));
    if (!f) throw std::runtime_error(std::string("cannot read ") + path);
    return v;
}

// a landmark row from a collection (x..., y...), the layout detect(image, initialisation) takes
static cv::Mat start_from(const rcr::LandmarkCollection<cv::Vec2f>& lms)
{
    const int L = static_cast<int>(lms.size());
    cv::Mat row(1, 2 * L, CV_32FC1);
    for (int i = 0; i < L; ++i) {
        row.at<float>(0, i) = lms[i].coordinates[0] + 1.25f;           // moved off the converged landmarks: a real start
        row.at<float>(0, i + L) = lms[i].coordinates[1] - 0.75f;
    }
    return row;
}

int main(int argc, char** argv)
{
    try {
        // fails loudly (std::runtime_error from the context) when there is no GPU
        rcr::detection_model m = rcr::load_detection_model(argc >= 2 ? argv[1] : "face_landmarks_model_rcr_22.bin");
        if (argc < 22) { std::printf("usage: test_detect_colour MODEL A.bgr A.gray WA HA B.bgr B.gray WB HB (X Y W H) x 3\n"); return 2; }
        std::vector<std::vector<unsigned char>> bgr_raw, gray_raw;
        std::vector<cv::Mat> gray, colour;
        for (int k = 0; k < 2; ++k) {
            const int w = std::atoi(argv[4 + 4 * k]), h = std::atoi(argv[5 + 4 * k]);
            bgr_raw.push_back(read_raw(argv[2 + 4 * k], static_cast<size_t>(w) * h * 3));
            gray_raw.push_back(read_raw(argv[3 + 4 * k], static_cast<size_t>(w) * h));
        }
        for (int k = 0; k < 2; ++k) {
            const int w = std::atoi(argv[4 + 4 * k]), h = std::atoi(argv[5 + 4 * k]);
            colour.emplace_back(h, w, CV_8UC3, bgr_raw[k].data());
            gray.emplace_back(h, w, CV_8UC1, gray_raw[k].data());
        }
        std::vector<cv::Rect> b;
        for (int j = 0; j < 3; ++j) b.emplace_back(std::atoi(argv[10 + 4 * j]), std::atoi(argv[11 + 4 * j]), std::atoi(argv[12 + 4 * j]), std::atoi(argv[13 + 4 * j]));

        // detect(image, facebox)
        const auto g0 = m.detect(gray[0], b[0]), g1 = m.detect(gray[0], b[1]), g2 = m.detect(gray[1], b[2]);
        expect(same(m.detect(colour[0], b[0]), g0), "detect(colour, facebox) frame A");
        expect(same(m.detect(colour[1], b[2]), g2), "detect(colour, facebox) frame B");
        // detect(images, faceboxes), one box per equally sized frame
        const auto batch_gray = m.detect(std::vector<cv::Mat>{gray[0], gray[0]}, std::vector<cv::Rect>{b[0], b[1]});
        const auto batch_colour = m.detect(std::vector<cv::Mat>{colour[0], colour[0]}, std::vector<cv::Rect>{b[0], b[1]});
        expect(batch_colour.size() == 2 && same_rows(batch_colour[0], batch_gray[0]) && same_rows(batch_colour[1], batch_gray[1]),
               "detect(colour images, faceboxes)");
        // detect(images, box list per image), colour frames and one gray and one colour frame in one call
        const std::vector<std::vector<cv::Rect>> boxes{{b[0], b[1]}, {b[2]}};
        for (const auto& frames : {colour, std::vector<cv::Mat>{gray[0], colour[1]}}) {
            const auto got = m.detect(frames, boxes);
            const bool shape = got.size() == 2 && got[0].size() == 2 && got[1].size() == 1;
            expect(shape, "detect(images, box lists) shape");
            if (shape) expect(same(got[0][0], g0) && same(got[0][1], g1) && same(got[1][0], g2), "detect(images, box lists)");
        }
        // detect(image, initialisation): the tracking call
        const cv::Mat i0 = start_from(g0), i1 = start_from(g1), i2 = start_from(g2);
        const auto t0 = m.detect(gray[0], i0), t1 = m.detect(gray[0], i1), t2 = m.detect(gray[1], i2);
        expect(same(m.detect(colour[0], i0), t0), "detect(colour, initialisation)");
        // detect(images, initialisations): several tracked faces per frame
        const std::vector<std::vector<cv::Mat>> inits{{i0, i1}, {i2}};
        for (const auto* frames : {&gray, &colour}) {
            const auto got = m.detect(*frames, inits);
            const bool shape = got.size() == 2 && got[0].size() == 2 && got[1].size() == 1;
            expect(shape, "detect(images, initialisations) shape");
            if (shape) expect(same(got[0][0], t0) && same(got[0][1], t1) && same(got[1][0], t2),
                              frames == &gray ? "detect(gray images, initialisations)" : "detect(colour images, initialisations)");
        }
        const auto none = m.detect(colour, std::vector<std::vector<cv::Mat>>(2));
        expect(none.size() == 2 && none[0].empty() && none[1].empty(), "no initialisations");
        std::printf("LANDMARKS %s %.6f %.6f\n", t0[0].name.c_str(), t0[0].coordinates[0], t0[0].coordinates[1]);
    } catch (const std::exception& e) {
        std::printf("exception: %s\n", e.what());
        return 1;
    }
    if (failures) { std::printf("%d failure(s)\n", failures); return 1; }
    std::printf("ALL OK\n");
    return 0;
}
