// rcr::detection_model::detect(images, list of face boxes per image) through the C++14 shell: several faces per frame, frames
// of different sizes.  Every face must equal the single-face detect(image, facebox) bit for bit, on the gray route (frames read
// in place by sd_detect_faces_host) and on the colour route (sd_bgr2gray + sd_model_align_boxes + sd_detect_faces_device).
//
//   test_detect_faces MODEL A.raw WA HA B.raw WB HB  X Y W H  X Y W H  X Y W H
//     two boxes on frame A, one on frame B (8UC1 raw files)
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

static void expect(bool ok, const char* what)
{
    if (!ok) { std::printf("FAIL %s\n", what); ++failures; }
}

int main(int argc, char** argv)
{
    try {
        // fails loudly (std::runtime_error from the context) when there is no GPU
        rcr::detection_model m = rcr::load_detection_model(argc >= 2 ? argv[1] : "face_landmarks_model_rcr_22.bin");
        if (argc < 20) { std::printf("usage: test_detect_faces MODEL A.raw WA HA B.raw WB HB (X Y W H) x 3\n"); return 2; }
        std::vector<std::vector<unsigned char>> raw(2);
        std::vector<cv::Mat> gray, colour;
        std::vector<std::vector<unsigned char>> bgr(2);
        for (int k = 0; k < 2; ++k) {
            const int w = std::atoi(argv[3 + 3 * k]), h = std::atoi(argv[4 + 3 * k]);
            raw[k].resize(static_cast<size_t>(w) * h);
            std::ifstream f(argv[2 + 3 * k], std::ios::binary);
            f.read(reinterpret_cast<char*>(raw[k].data()), static_cast<std::streamsize>(raw[k].size()));
            gray.emplace_back(h, w, CV_8UC1, raw[k].data());
            // B = G = R: cvtColor(BGR2GRAY) gives the gray frame back exactly
            bgr[k].resize(raw[k].size() * 3);
            for (size_t i = 0; i < raw[k].size(); ++i) bgr[k][3 * i] = bgr[k][3 * i + 1] = bgr[k][3 * i + 2] = raw[k][i];
            colour.emplace_back(h, w, CV_8UC3, bgr[k].data());
        }
        std::vector<cv::Rect> b;
        for (int j = 0; j < 3; ++j) b.emplace_back(std::atoi(argv[8 + 4 * j]), std::atoi(argv[9 + 4 * j]), std::atoi(argv[10 + 4 * j]), std::atoi(argv[11 + 4 * j]));
        const std::vector<std::vector<cv::Rect>> boxes{{b[0], b[1]}, {b[2]}};
        const auto single0 = m.detect(gray[0], b[0]), single1 = m.detect(gray[0], b[1]), single2 = m.detect(gray[1], b[2]);
        for (const auto* frames : {&gray, &colour}) {
            const auto got = m.detect(*frames, boxes);
            expect(got.size() == 2 && got[0].size() == 2 && got[1].size() == 1, "result shape");
            if (got.size() == 2 && got[0].size() == 2 && got[1].size() == 1) {
                expect(same(got[0][0], single0), frames == &gray ? "gray frame A face 0" : "colour frame A face 0");
                expect(same(got[0][1], single1), frames == &gray ? "gray frame A face 1" : "colour frame A face 1");
                expect(same(got[1][0], single2), frames == &gray ? "gray frame B face 0" : "colour frame B face 0");
            }
        }
        // a frame without boxes is skipped, an empty call returns empty lists
        const auto none = m.detect(gray, std::vector<std::vector<cv::Rect>>(2));
        expect(none.size() == 2 && none[0].empty() && none[1].empty(), "no boxes");
        std::printf("LANDMARKS %s %.6f %.6f\n", single0[0].name.c_str(), single0[0].coordinates[0], single0[0].coordinates[1]);
    } catch (const std::exception& e) {
        std::printf("exception: %s\n", e.what());
        return 1;
    }
    if (failures) { std::printf("%d failure(s)\n", failures); return 1; }
    std::printf("ALL OK\n");
    return 0;
}
