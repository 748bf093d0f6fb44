"""Pins the CPU oracle (oracle/sd_oracle.c) against the reference's own golden data (no GPU needed).

  - cv2 4.13 resize / BGR2GRAY outputs                      (tests/golden/resize_cv2.npz, examples.npz)
  - the reference's hog.c outputs                            (tests/golden/hog_ref.npz, hog_live_ref.npz, and live vs oracle/_ref when built)
  - the shipped model file + the 5 annotated example frames  (byte round-trip, landmark error)
  - every literal of the reference's gtest suite             (tests/known_answers.py)
"""
import ctypes as C
import os

import numpy as np
import pytest

import known_answers as K
from conftest import rel_err


def test_resize_matches_cv2_goldens(oracle, golden):
    n = len([k for k in golden.resize.files if k.startswith("src")])
    assert n >= 10
    for i in range(n):
        src, dst = golden.resize[f"src{i}"], golden.resize[f"dst{i}"]
        got = oracle.resize_linear_u8(src, dst.shape[1], dst.shape[0])
        assert np.array_equal(got, dst), f"case {i}: {src.shape}->{dst.shape}"


def test_bgr2gray_matches_cv2_golden(oracle, golden):
    assert np.array_equal(oracle.bgr2gray_u8(golden.examples["bgr_crop"]), golden.examples["bgr_crop_gray"])


def test_hog_core_matches_reference_goldens_bit_exact(oracle, golden):
    n = len([k for k in golden.hog.files if k.startswith("img")])
    assert n == 16
    for i in range(n):
        K_, cs, variant = [int(v) for v in golden.hog[f"cfg{i}"]]
        got = oracle.hog_core(golden.hog[f"img{i}"].astype(np.float32), cs, K_, variant)
        assert np.array_equal(got.view(np.uint32), golden.hog[f"out{i}"].view(np.uint32)), f"case {i} K={K_} cs={cs} v={variant}"


def test_hog_core_matches_live_reference(oracle, golden):
    """Against the reference's hog.c outputs stored in hog_live_ref.npz, and against oracle/_ref itself where it is built."""
    ref = np.load(os.path.join(golden.dir, "hog_live_ref.npz"))
    n = len([k for k in ref.files if k.startswith("core_img")])
    assert n == 9
    for i in range(n):
        K_, cs = [int(v) for v in ref[f"core_cfg{i}"]]
        img = ref[f"core_img{i}"].astype(np.float32)
        a = oracle.hog_core(img, cs, K_, 1)
        assert np.array_equal(a.view(np.uint32), ref[f"core_out{i}"].view(np.uint32)), f"case {i} K={K_} cs={cs}"
        if oracle.ref_available():
            b = oracle.hog_core(img, cs, K_, 1, use_ref=True)
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


def test_orientation_ties_are_resolved_like_the_reference(oracle):
    """Integer-valued gradients make exact ties common (hog.c:656-672 strict '>', ascending k)."""
    img = np.zeros((8, 8), dtype=np.float32)
    img[:, 4:] = 100.0                       # pure +x gradient -> bin 0
    img2 = img.T.copy()                      # pure +y gradient -> k = K/2 for even K
    b = oracle.hog_orientation_bins(img, 4)
    assert b[3, 3] == 0 and b[3, 4] == 0 and b[0, 0] == -1
    b2 = oracle.hog_orientation_bins(img2, 4)
    assert b2[3, 3] == 2
    d = np.zeros((8, 8), dtype=np.float32)   # 45 degrees: exact tie between k=0 (0 deg) and k=1 (45 deg)? no: 45 deg is bin 1
    for y in range(8):
        for x in range(8):
            d[y, x] = 10.0 * (x + y)
    assert oracle.hog_orientation_bins(d, 4)[3, 3] == 1
    assert oracle.hog_orientation_bins(-d, 4)[3, 3] == 5


def test_model_file_parses_and_round_trips(oracle, golden, tmp_path):
    m = oracle.Model(golden.model_path)
    assert m.num_levels == 4 and m.num_landmarks == 22
    assert [w.shape for w in m.weights] == [(8801, 44)] * 4
    assert m.regularisers == [(1, 1.5, 0)] * 4                       # MatrixNorm 1.5, bias unregularised
    assert [(p.variant, p.num_cells, p.cell_size, p.num_bins) for p in m.hog_params] == [(1, 5, 11, 4), (1, 5, 10, 4), (1, 5, 8, 4), (1, 5, 6, 4)]
    assert np.allclose([p.relative_patch_size for p in m.hog_params], [1.0, 0.7, 0.4, 0.25])
    assert m.right_ids == ["37", "40"] and m.left_ids == ["43", "46"]
    assert m.right_idx == [4, 7] and m.left_idx == [10, 13]
    out = tmp_path / "rt.bin"
    m.save(str(out))
    assert out.read_bytes() == open(golden.model_path, "rb").read()


def test_model_errors(oracle, tmp_path):
    with pytest.raises(RuntimeError):
        oracle.Model(str(tmp_path / "does_not_exist.bin"))
    bad = tmp_path / "bad.bin"
    bad.write_bytes(b"\x04\x00\x00\x00\x00\x00\x00\x00garbage")
    with pytest.raises(RuntimeError):
        oracle.Model(str(bad))


def _gt_row(pts, ids):
    gt = np.array([pts[int(s) - 1] for s in ids], dtype=np.float32)
    return np.concatenate([gt[:, 0], gt[:, 1]])


def test_detect_on_reference_example_frames(oracle, golden):
    m = oracle.Model(golden.model_path)
    for i in range(5):
        gray, box = golden.examples[f"gray{i}"], golden.examples["boxes"][i]
        lm = m.detect(gray, box)
        assert np.array_equal(lm, golden.detect[f"landmarks{i}"]), "oracle drifted from the committed reference-HOG detect"
        gt = _gt_row(golden.examples[f"pts{i}"], m.landmark_ids)
        ied = oracle.get_ied(gt, m.right_idx, m.left_idx)
        err0 = np.mean(np.hypot(*(oracle.align_mean(m.mean, box) - gt).reshape(2, -1))) / ied
        err = np.mean(np.hypot(*(lm - gt).reshape(2, -1))) / ied
        assert 0.05 < err0 < 0.1 and err < 0.0125, (i, err0, err)     # SURVEY 8c: 0.062-0.084 -> 0.0062-0.0104
        feats = oracle.hog_transform(gray, oracle.align_mean(m.mean, box), m.hog_params[0], m.right_idx, m.left_idx)
        assert np.array_equal(feats.view(np.uint32), golden.detect[f"features_l0_{i}"].view(np.uint32))
        assert feats[-1] == 1.0 and feats.size == 8801


def test_patch_geometry_rounding_rules(oracle):
    assert [oracle.cv_round(v) for v in (0.5, 1.5, 2.5, -0.5, -1.5, 2.4999, 2.5001)] == [0, 2, 2, 0, -2, 2, 3]   # cvRound: half to even
    lib = oracle.lib()
    lib.orc_patch_half.restype = C.c_int
    assert lib.orc_patch_half(C.c_float(1.0), C.c_double(5.0)) == 3      # std::round: half away from zero
    assert lib.orc_patch_half(C.c_float(1.0), C.c_double(3.0)) == 2
    assert lib.orc_patch_half(C.c_float(0.25), C.c_double(90.0)) == 11


def test_crop_zero_pads_outside_the_frame(oracle):
    img = (np.arange(100, dtype=np.uint8).reshape(10, 10) + 1)
    p = oracle.crop_patch_u8(img, 0, 0, 3)
    assert p.shape == (6, 6) and np.all(p[:3, :] == 0) and np.all(p[:, :3] == 0) and np.array_equal(p[3:, 3:], img[:3, :3])
    p = oracle.crop_patch_u8(img, 9, 9, 2)
    assert np.array_equal(p[:3, :3], img[7:10, 7:10]) and np.all(p[3:, :] == 0) and np.all(p[:, 3:] == 0)
    assert np.all(oracle.crop_patch_u8(img, 40, 40, 2) == 0)


# ---- regressor known answers (reference gtest literals) ---------------------------------------------
class OracleBackend:
    def __init__(self, O, precision):
        self.O, self.precision = O, precision

    def learn(self, data, labels, reg):
        r = self.O.Regulariser(int(reg[0]), float(reg[1]), int(reg[2]))
        X, lam = self.O.solve(np.asarray(data, np.float32), np.asarray(labels, np.float32), r, self.precision)
        return X

    def predict(self, values, X):
        return self.O.predict(np.asarray(values, np.float32), X)

    def residual(self, data, labels, X):
        return self.O.test_residual(np.asarray(data, np.float32), np.asarray(labels, np.float32), X)

    def train(self, x_gt, x0, y, h, n_reg, callback=None):
        regs = [self.O.Regulariser(0, 0.0, 1) for _ in range(n_reg)]
        D = np.atleast_1d(h(x0[0], 0, 0)).size
        w, xf, rc = self.O.cascade_train(x_gt, x0, y, regs, [D] * n_reg, h, None, self.precision, callback)
        return w, xf

    def test(self, weights, x0, y, h):
        return self.O.cascade_apply(x0, y, weights, h, None)


def run_lr_cases(backend):
    report = []
    for name, data, labels, x in K.LR1D_LEARN:
        X = backend.learn(data, labels, (0, 0.0, True))
        assert abs(float(X[0, 0]) - x) <= K.REL_TOL * abs(x), name
    X = backend.learn(K.LR1D_PREDICT["data"], K.LR1D_PREDICT["labels"], (0, 0.0, True))
    for v, exp in K.LR1D_PREDICT["tests"]:
        assert abs(float(backend.predict([[v]], X)[0, 0]) - exp) <= 1e-6
    for case in K.LR1D_RESIDUAL:
        r = backend.residual(case["test"], case["gt"], X)
        assert abs(r - case["residual"]) <= K.REL_TOL * max(case["residual"], 1e-3)
    for case in K.ND_CASES:
        X = backend.learn(case["data"], case["labels"], case["reg"])
        exp = np.array(case["x"], dtype=np.float64)
        e = rel_err(X, exp)
        report.append((case["name"], e))
        if "x_abs_tol" in case:
            assert np.max(np.abs(X - exp)) <= case["x_abs_tol"] + K.REL_TOL * np.max(np.abs(exp)), case["name"]
        else:
            assert e <= K.REL_TOL, (case["name"], e)
        if "predict" in case:
            v, p = case["predict"]
            assert rel_err(backend.predict(v, X), p) <= K.REL_TOL
        if "test" in case:
            r = backend.residual(case["test"], case["gt"], X)
            assert r <= case["residual_le"] * 2.0, (case["name"], r)     # groundtruth literals carry 4 decimals
    return report


def run_sdo_cases(backend):
    report = []
    for name, fname, train, test, n_reg, tr_res, ts_res, line in K.SDO_CASES:
        h, y_tr, x_tr, x0, y_ts, x_ts, x0_ts = K.sdo_case_data(fname, train, test)
        seen = []
        w, xf = backend.train(x_tr, x0, y_tr, h, n_reg, callback=lambda cur, lvl=None: seen.append(K.nlsr(cur, x_tr)))
        assert len(seen) == n_reg                                  # the epoch callback fires once per level (:217)
        pred = backend.test(w, x0, y_tr, h)
        r_tr = K.nlsr(pred, x_tr)
        assert abs(seen[-1] - r_tr) <= 1e-6 * max(r_tr, 1e-3)
        r_ts = K.nlsr(backend.test(w, x0_ts, y_ts, h), x_ts)
        report.append((name, abs(r_tr - tr_res) / tr_res, abs(r_ts - ts_res) / ts_res))
        assert abs(r_tr - tr_res) <= K.REL_TOL * tr_res, (name, r_tr, tr_res)
        # XCubeConvergence's own tolerance is 2e-5 absolute (:192)
        assert abs(r_ts - ts_res) <= max(K.REL_TOL * ts_res, 2.5e-5 if name == "XCubeConvergence" else 0), (name, r_ts, ts_res)
    h, y_tr, x_tr, x0, y_ts, x_ts, x0_ts = K.sdo_multi_data()
    w, xf = backend.train(x_tr, x0, y_tr, h, K.SDO_MULTI["n_regressors"])
    r_tr = K.nlsr(backend.test(w, x0, y_tr, h), x_tr)
    r_ts = K.nlsr(backend.test(w, x0_ts, y_ts, h), x_ts)
    report.append(("SinErfConvergenceCascadeMultiY", r_tr, r_ts))
    # a 10-deep cascade of nearly singular 2x2 systems: the reference's literal carries 4 digits (:496,:520)
    assert abs(r_tr - K.SDO_MULTI["train_residual"]) <= 25 * K.SDO_MULTI["train_tol"] + 0.05 * K.SDO_MULTI["train_residual"]
    assert abs(r_ts - K.SDO_MULTI["test_residual"]) <= 25 * K.SDO_MULTI["test_tol"] + 0.05 * K.SDO_MULTI["test_residual"]
    return report


@pytest.mark.parametrize("precision", [0, 1])
def test_linear_regressor_known_answers(oracle, precision):
    rep = run_lr_cases(OracleBackend(oracle, precision))
    print("oracle precision", precision, [(n, f"{e:.2e}") for n, e in rep])


@pytest.mark.parametrize("precision", [0, 1])
def test_optimiser_known_answers(oracle, precision):
    rep = run_sdo_cases(OracleBackend(oracle, precision))
    print("oracle precision", precision, [(r[0], f"{r[1]:.2e}", f"{r[2]:.2e}") for r in rep])


def test_matrixnorm_lambda_rule(oracle):
    """regressors.hpp:133-136: lambda = param * ||AtA||_F / N, bias row optionally excluded."""
    rng = np.random.default_rng(3)
    A = rng.random((50, 6)).astype(np.float32)
    A[:, -1] = 1.0
    B = rng.random((50, 2)).astype(np.float32)
    reg = oracle.Regulariser(1, 0.5, 0)
    X, lam = oracle.solve(A, B, reg, 0)
    G = A.astype(np.float64).T @ A.astype(np.float64)
    assert abs(lam - 0.5 * np.linalg.norm(G) / 50) <= 1e-5 * lam
    Lam = np.eye(6) * lam
    Lam[-1, -1] = 0
    Xd = np.linalg.solve(G + Lam, A.astype(np.float64).T @ B.astype(np.float64))
    assert rel_err(X, Xd) < 1e-4


def test_pose_estimation_example_config2(oracle):
    """BASELINE config 2: examples/pose_estimation.cpp -- 500 samples x 20 features -> 6 pose parameters, three
    regressors with MatrixNorm 2.0, known-template training (y = projected landmarks)."""
    import pose_example as P
    x_tr, y_tr, x0 = P.training_set()
    regs = [oracle.Regulariser(1, 2.0, 1) for _ in range(3)]
    residuals = []
    w, xf, rc = oracle.cascade_train(x_tr, x0, y_tr, regs, [20] * 3, P.projection, None, 0,
                                     lambda cur, lvl: residuals.append(K.nlsr(cur, x_tr)))
    assert rc == 0 and len(residuals) == 3 and residuals[0] > residuals[1] > residuals[2] and residuals[2] < 0.01
    pred = oracle.cascade_apply(P.TEST_INIT, P.TEST_LANDMARKS, w, P.projection, None)[0]
    print("oracle pose residuals", residuals, "predicted pitch/yaw/roll", pred[:3])
    assert np.all(np.abs(pred[:3] - np.array([11.0, -25.0, -10.0])) < 6.0)      # example's ground truth (:334)


def test_fixed_patch_transform_equals_adaptive_one_at_matching_size(oracle, golden):
    """examples/landmark_detection.cpp:195-261 (fixed patch, no resize, no bias) against adaptive_vlhog.hpp:109-185: when
    the inter-eye distance makes the adaptive patch exactly num_cells * cell_size wide, cv::resize is the identity and the
    two functors must agree value for value (the adaptive one appends its bias)."""
    import synth
    img = synth.smooth_images(1, 120, 160, seed=3)[0]
    nc, cs, K = 3, 12, 4
    L = 6
    rng = np.random.default_rng(2)
    x = np.concatenate([rng.uniform(10, 150, L), rng.uniform(10, 110, L)]).astype(np.float32)
    x[0], x[L] = 40.0, 60.0                       # right eye
    x[1], x[L + 1] = 40.0 + nc * cs, 60.0         # left eye: IED = 36 -> half = round(1.0 * 36 / 2) = 18 = nc * (cs / 2)
    x[2], x[L + 2] = 2.0, 118.0                   # near a corner: zero padding on two sides
    ref = np.load(os.path.join(golden.dir, "hog_live_ref.npz"))   # the same frame and landmarks through the reference's hog.c
    for variant in (0, 1):
        hp = oracle.HogParam(variant, nc, cs, K, 1.0)
        adaptive = oracle.hog_transform(img, x, hp, [0], [1])
        fixed = oracle.hog_transform_fixed(img, x, hp)
        assert fixed.size == adaptive.size - 1 and adaptive[-1] == 1.0
        assert np.array_equal(fixed, adaptive[:-1])
        assert np.array_equal(oracle.hog_transform_fixed(ref["fixed_img"], ref["fixed_x"], hp), ref[f"fixed_out{variant}"])
        if oracle.ref_available():
            assert np.array_equal(oracle.hog_transform_fixed(img, x, hp, use_ref=True), fixed)


def test_perturb_box_rcr_train_semantics(oracle):
    """perturb() of apps/rcr/rcr-train.cpp:130-146: float arithmetic, truncation toward zero in cv::Rect(int)."""
    assert oracle.perturb_box((100, 50, 200, 100), 0.0, 0.0, 1.0) == (100, 50, 200, 100)
    assert oracle.perturb_box((100, 50, 200, 100), 0.1, -0.1, 1.0) == (120, 40, 200, 100)
    # scaling keeps the centre: width 200 -> 220, x moves by -10; 0.95 -> 190 wide, x + 5
    assert oracle.perturb_box((100, 50, 200, 100), 0.0, 0.0, 1.1) == (90, 45, 220, 110)
    assert oracle.perturb_box((100, 50, 200, 100), 0.0, 0.0, 0.95) == (105, 52, 190, 95)
    # truncation toward zero (not floor) for negative coordinates: -0.5 -> 0
    assert oracle.perturb_box((0, 0, 10, 10), -0.05, -0.05, 1.0) == (0, 0, 10, 10)
    assert oracle.perturb_box((0, 0, 10, 10), -0.15, -0.25, 1.0) == (-1, -2, 10, 10)


def test_normalised_landmark_errors_match_a_float64_restatement(oracle):
    rng = np.random.default_rng(4)
    L = 22
    gt = rng.uniform(50, 300, size=(9, 2 * L)).astype(np.float32)
    pred = (gt + rng.normal(0, 3, size=gt.shape)).astype(np.float32)
    r, l = [4, 7], [10, 13]
    got = oracle.normalised_landmark_errors(pred, gt, r, l)
    re = np.stack([pred[:, r].mean(1), pred[:, [i + L for i in r]].mean(1)], 1).astype(np.float64)
    le = np.stack([pred[:, l].mean(1), pred[:, [i + L for i in l]].mean(1)], 1).astype(np.float64)
    ied = np.linalg.norm(re - le, axis=1)
    d = np.hypot(pred[:, :L].astype(np.float64) - gt[:, :L], pred[:, L:].astype(np.float64) - gt[:, L:])
    assert np.allclose(got, d / ied[:, None], rtol=1e-6, atol=0)


def test_hog_transform_properties(oracle):
    """Size-independent properties of the projection (adaptive_vlhog.hpp:109-185) that any restatement must keep:
    a constant image gives the zero descriptor (plus the bias); shifting the frame and the landmarks by the same integer
    offset leaves interior descriptors unchanged; cv::resize to the same size is the identity."""
    import synth
    rng = np.random.default_rng(21)
    hp = oracle.HogParam(1, 5, 10, 4, 1.0)
    L = 6
    x = np.concatenate([rng.uniform(70, 130, L), rng.uniform(70, 110, L)]).astype(np.float32)
    x[0], x[L], x[1], x[L + 1] = 80.0, 90.0, 130.0, 90.0          # IED = 50 -> half = 25, patch 50 = num_cells * cell_size
    flat = np.full((200, 220), 97, np.uint8)
    f = oracle.hog_transform(flat, x, hp, [0], [1])
    assert f[-1] == 1.0 and not np.any(f[:-1])
    img = synth.smooth_images(1, 200, 220, seed=8)[0]
    base = oracle.hog_transform(img, x, hp, [0], [1])
    dx, dy = 7, 11
    shifted = np.zeros_like(img)
    shifted[dy:, dx:] = img[:-dy, :-dx]
    xs = x.copy()
    xs[:L] += dx
    xs[L:] += dy
    assert np.array_equal(oracle.hog_transform(shifted, xs, hp, [0], [1]), base)
    patch = rng.integers(0, 256, size=(37, 37), dtype=np.uint8)
    assert np.array_equal(oracle.resize_linear_u8(patch, 37, 37), patch)
