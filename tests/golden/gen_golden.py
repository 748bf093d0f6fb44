"""Generates the committed golden fixtures under tests/golden/.

Run in the BUILD container only (needs /root/reference, cv2 4.13 and oracle/_ref):

    python tests/golden/gen_golden.py

Outputs (all small, committed):
  face_landmarks_model_rcr_22.bin   the reference's shipped model (DATA fixture named by BASELINE.json config 3;
                                    byte-for-byte copy of /root/reference/apps/rcr/data/..., not source code)
  examples.npz                      the 5 annotated example frames of the reference as 8-bit grey (cv2 BGR2GRAY),
                                    a BGR crop + its grey conversion, their ibug .pts landmarks (0-based), and the
                                    Viola-Jones face boxes (cv2's haarcascade_frontalface_alt2, SURVEY 8c)
  mean_ibug_lfpw_68.npy             the 68-point mean shape (x then y)
  resize_cv2.npz                    cv2.resize INTER_LINEAR 8UC1 input/output pairs (pins oracle.resize_linear_u8)
  hog_ref.npz                       outputs of the reference's own hog.c (oracle/_ref) on seeded inputs
                                    (pins oracle.hog_core when /root/reference is absent, i.e. on the GPU box)
  detect_ref.npz                    oracle detect() on the example frames with hog.c as the HOG core
  hog_live_ref.npz                  the reference's hog.c on the inputs of tests/test_oracle.py's comparisons with
                                    oracle/_ref (seeded images through the HOG core, and one frame through the
                                    fixed-patch transform), stored with those inputs
"""
import os
import shutil
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import oracle as O  # noqa: E402

REF = "/root/reference"
BOXES = [[91, 157, 209, 209], [46, 116, 170, 170], [79, 99, 150, 150], [178, 197, 283, 283], [242, 219, 317, 317]]


def read_pts(path):
    lines = [l.strip() for l in open(path)]
    s, e = lines.index("{"), lines.index("}")
    # include/rcr/landmarks_io.hpp:43-85: ibug files are 1-based, the reader subtracts 1
    return np.array([[float(v) for v in l.split()] for l in lines[s + 1:e]], dtype=np.float32) - 1.0


def main():
    O.build()
    shutil.copyfile(f"{REF}/apps/rcr/data/face_landmarks_model_rcr_22.bin", f"{HERE}/face_landmarks_model_rcr_22.bin")
    mean68 = np.array([float(v) for v in open(f"{REF}/apps/rcr/data/mean_ibug_lfpw_68.txt").read().replace("\n", "").split(",") if v.strip()],
                      dtype=np.float32)
    assert mean68.size == 136
    np.save(f"{HERE}/mean_ibug_lfpw_68.npy", mean68)

    # ---- example frames ----
    ex = {}
    cascade = cv2.CascadeClassifier(os.path.join(cv2.data.haarcascades, "haarcascade_frontalface_alt2.xml"))
    for i in range(5):
        bgr = cv2.imread(f"{REF}/examples/data/ibug_lfpw_trainset/image_000{i + 1}.png")
        gray = cv2.cvtColor(bgr, cv2.COLOR_BGR2GRAY)
        ex[f"gray{i}"] = gray
        ex[f"pts{i}"] = read_pts(f"{REF}/examples/data/ibug_lfpw_trainset/image_000{i + 1}.pts")
        det = cascade.detectMultiScale(bgr)
        print("image", i, gray.shape, "V&J boxes:", [list(map(int, d)) for d in det], "-> using", BOXES[i])
        if i == 0:
            crop = bgr[100:164, 120:216].copy()
            ex["bgr_crop"] = crop
            ex["bgr_crop_gray"] = cv2.cvtColor(crop, cv2.COLOR_BGR2GRAY)
    ex["boxes"] = np.array(BOXES, dtype=np.int32)
    np.savez_compressed(f"{HERE}/examples.npz", **ex)

    # ---- cv2.resize goldens ----
    rng = np.random.default_rng(20240923)
    rs = {}
    cases = [(90, 55), (64, 50), (36, 40), (22, 30), (110, 55), (55, 55), (7, 30), (200, 55), (33, 50), (100, 50), (41, 40), (58, 30)]
    for n, (P, fs) in enumerate(cases):
        src = rng.integers(0, 256, (P, P), dtype=np.uint8)
        if n % 3 == 1:
            src = cv2.GaussianBlur(src, (0, 0), 1.5)
        rs[f"src{n}"] = src
        rs[f"dst{n}"] = cv2.resize(src, (fs, fs))
        assert np.array_equal(rs[f"dst{n}"], O.resize_linear_u8(src, fs, fs)), (P, fs)
    np.savez_compressed(f"{HERE}/resize_cv2.npz", **rs)

    # ---- reference hog.c goldens ----
    hg = {}
    n = 0
    for K in (4, 9):
        for fs, cs in ((55, 11), (50, 10), (40, 8), (30, 6)):
            for variant in (1, 0):
                img = rng.integers(0, 256, (fs, fs)).astype(np.float32)
                if n % 2:
                    img = np.round(cv2.GaussianBlur(img, (0, 0), 2.0))
                out = O.hog_core(img, cs, K, variant, use_ref=True)
                assert np.array_equal(out.view(np.uint32), O.hog_core(img, cs, K, variant).view(np.uint32))
                hg[f"img{n}"] = img.astype(np.uint8)
                hg[f"out{n}"] = out
                hg[f"cfg{n}"] = np.array([K, cs, variant], dtype=np.int32)
                n += 1
    np.savez_compressed(f"{HERE}/hog_ref.npz", **hg)

    # ---- end-to-end detect goldens (oracle glue + the reference's hog.c) ----
    m = O.Model(f"{HERE}/face_landmarks_model_rcr_22.bin")
    dt = {}
    for i in range(5):
        lm = m.detect(ex[f"gray{i}"], BOXES[i], use_ref=True)
        assert np.array_equal(lm, m.detect(ex[f"gray{i}"], BOXES[i], use_ref=False))
        dt[f"landmarks{i}"] = lm
        feats = O.hog_transform(ex[f"gray{i}"], O.align_mean(m.mean, BOXES[i]), m.hog_params[0], m.right_idx, m.left_idx, use_ref=True)
        dt[f"features_l0_{i}"] = feats
    np.savez_compressed(f"{HERE}/detect_ref.npz", **dt)
    live_reference_goldens()
    for f in sorted(os.listdir(HERE)):
        print(f, os.path.getsize(os.path.join(HERE, f)))


def live_reference_goldens():
    """hog_live_ref.npz: the inputs are built exactly as test_hog_core_matches_live_reference and
    test_fixed_patch_transform_equals_adaptive_one_at_matching_size build them."""
    sys.path.insert(0, os.path.dirname(HERE))
    import synth
    O.build()
    assert O.ref_available(), "oracle/_ref is not built"
    g = {}
    rng = np.random.default_rng(7)
    n = 0
    for K in (4, 9, 6):
        for fs, cs in ((55, 11), (30, 6), (48, 8)):
            img = rng.integers(0, 256, (fs, fs)).astype(np.float32)
            g[f"core_img{n}"] = img.astype(np.uint8)
            g[f"core_out{n}"] = O.hog_core(img, cs, K, 1, use_ref=True)
            g[f"core_cfg{n}"] = np.array([K, cs], dtype=np.int32)
            n += 1
    img = synth.smooth_images(1, 120, 160, seed=3)[0]
    nc, cs, K, L = 3, 12, 4, 6
    rng = np.random.default_rng(2)
    x = np.concatenate([rng.uniform(10, 150, L), rng.uniform(10, 110, L)]).astype(np.float32)
    x[0], x[L] = 40.0, 60.0
    x[1], x[L + 1] = 40.0 + nc * cs, 60.0
    x[2], x[L + 2] = 2.0, 118.0
    g["fixed_img"], g["fixed_x"] = img, x
    for variant in (0, 1):
        g[f"fixed_out{variant}"] = O.hog_transform_fixed(img, x, O.HogParam(variant, nc, cs, K, 1.0), use_ref=True)
    np.savez_compressed(f"{HERE}/hog_live_ref.npz", **g)


if __name__ == "__main__":
    main()
