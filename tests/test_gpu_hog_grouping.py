"""The HOG kernel walks several landmarks of one face per CTA.  A face's descriptors must not depend on which other faces share
the launch, on the order of the faces, on the number of landmarks (remainder groups), or on the route that stages each source
window (TMA tile, 16-byte / word / byte load loops, unstaged windows too large for shared memory, ROI buffers, frames of
different sizes).  Every comparison between launches is bitwise; the oracle check uses the 1e-4 tolerance of test_gpu_hog."""
import numpy as np
import pytest
import torch

import synth
from conftest import rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-4


def _landmarks(m, L):
    """L landmark names that contain one right-eye and one left-eye name, and the column of the model's 22 landmarks each one
    takes its position from (names past the 22nd repeat earlier landmarks with an offset)."""
    r, l = m.right_ids[0], m.left_ids[0]
    others = [i for i in m.landmark_ids if i not in (r, l)]
    names = [r, l] + others
    src = [m.landmark_ids.index(n) for n in names]
    while len(names) < L:
        k = len(names)
        names.append(f"extra{k}")
        src.append(src[k % 22])
    return names[:L], src[:L], [r], [l]


def _params(oracle, m, boxes, src, jitter):
    x22 = np.stack([oracle.align_mean(m.mean, b) for b in boxes])
    L = len(src)
    x = np.concatenate([x22[:, src], x22[:, [22 + s for s in src]]], axis=1).astype(np.float32)
    x[:, 22:L] += jitter
    x[:, L + 22:] -= jitter
    return x


def _check_grouping(ht, x, idx, seed):
    """full launch == one face per launch == permuted faces == faces repeated (image index with repeats)"""
    full = ht(x, 0, idx).cpu().numpy()
    for i in range(x.shape[0]):
        assert np.array_equal(ht(x[i:i + 1], 0, idx[i:i + 1]).cpu().numpy()[0], full[i]), f"face {i} alone"
    rng = np.random.default_rng(seed)
    perm = rng.permutation(x.shape[0])
    assert np.array_equal(ht(x[perm], 0, idx[perm]).cpu().numpy(), full[perm]), "permuted faces"
    rep = np.concatenate([perm[:3], perm[:3], perm])
    assert np.array_equal(ht(x[rep], 0, idx[rep]).cpu().numpy(), full[rep]), "repeated faces"
    return full


def _frames_for_route(route):
    """frames whose HOG launch stages windows by the given route, and face boxes in them"""
    if route == "tma":          # uniform frames, 16-byte pitch: tensor maps
        return synth.smooth_images(5, 120, 160, seed=21), synth.face_boxes(5, 120, 160, seed=21, border_fraction=0.5)
    if route == "words":        # 4-byte but not 16-byte pitch: word load loop
        return synth.smooth_images(5, 120, 156, seed=22), synth.face_boxes(5, 120, 156, seed=22, border_fraction=0.5)
    if route == "bytes":        # odd pitch: byte load loop
        return synth.smooth_images(5, 121, 151, seed=23), synth.face_boxes(5, 121, 151, seed=23, border_fraction=0.5)
    if route == "mixed":        # frames of different sizes (packed, 16-byte rows): 16-byte load loop
        sizes = [(120, 160), (97, 131), (200, 150), (64, 64), (150, 90)]
        frames = [synth.smooth_images(1, h, w, seed=30 + i)[0] for i, (h, w) in enumerate(sizes)]
        boxes = np.array([synth.face_boxes(1, h, w, seed=30 + i, border_fraction=0.5)[0] for i, (h, w) in enumerate(sizes)])
        return frames, boxes
    assert route == "large"     # windows larger than the staging area: sampled straight from global memory
    boxes = np.array([(20, 10, 440, 440), (-100, -60, 400, 400), (200, 150, 320, 320), (50, 40, 90, 90), (300, 20, 460, 460)])
    return synth.smooth_images(5, 480, 640, seed=24), boxes


CASES = [(22, 4, 1, "tma"), (22, 9, 1, "tma"), (22, 4, 0, "tma"), (22, 9, 0, "large"), (1, 4, 1, "tma"), (3, 9, 1, "words"),
         (3, 4, 0, "bytes"), (29, 4, 1, "mixed"), (29, 9, 0, "tma"), (22, 4, 1, "large"), (29, 9, 1, "bytes"), (22, 4, 1, "mixed")]


@pytest.mark.parametrize("L,K,variant,route", CASES)
def test_hog_descriptors_do_not_depend_on_grouping(sd, oracle, golden, L, K, variant, route):
    m = oracle.Model(golden.model_path)
    frames, boxes = _frames_for_route(route)
    n = len(boxes)
    names, src, right, left = _landmarks(m, max(L, 2))
    if L == 1:                  # the adaptive transform needs both eyes: one landmark goes through the fixed-patch transform
        ht = sd.FixedHogTransform(np.stack(frames), variant, 5, 6, K)
        x = _params(oracle, m, boxes, src[:1], 0.0)
        full = _check_grouping(ht, x, np.arange(n, dtype=np.int32)[::-1].copy(), L)
        hp = oracle.HogParam(variant, 5, 6, K, 0.0)
        want = np.stack([oracle.hog_transform_fixed(frames[n - 1 - i], x[i], hp) for i in range(n)])
        assert rel_err(full, want) <= TOL
        return
    x = _params(oracle, m, boxes, src, 3.0)
    idx = np.arange(n, dtype=np.int32)[::-1].copy()
    x = x[idx]                  # face i lies in frame idx[i]
    for cs, rel in ((11, 1.0), (6, 0.25)):
        hp = sd.HoGParam(variant, 5, cs, K, rel)
        ht = sd.HogTransform(list(frames) if route == "mixed" else np.stack(frames), [hp], names, right, left)
        full = _check_grouping(ht, x, idx, L + cs)
        ohp = oracle.HogParam(variant, 5, cs, K, rel)
        ridx, lidx = [names.index(r) for r in right], [names.index(s) for s in left]
        for i in range(n):
            ref = oracle.hog_transform(frames[idx[i]], x[i], ohp, ridx, lidx)
            assert rel_err(full[i], ref) <= TOL, (i, cs)


def test_detect_faces_roi_route_does_not_depend_on_grouping(sd, golden):
    """Pinned host frames of mixed sizes take the ROI route (faces of a frame share one uploaded region): every face must
    equal its detection alone and in a permuted batch."""
    m = sd.load_detection_model(golden.model_path)
    sizes = [(480, 640), (240, 320), (300, 200)]
    frames = [synth.smooth_images(1, h, w, seed=50 + i)[0] for i, (h, w) in enumerate(sizes)]
    pinned = []
    for f in frames:
        h, w = f.shape
        stride = (w + 15) // 16 * 16
        buf = torch.zeros((h, stride), dtype=torch.uint8).pin_memory()
        buf[:, :w].copy_(torch.from_numpy(f))
        pinned.append(buf[:, :w])
    index = np.array([0, 0, 0, 1, 1, 2, 0, 2], dtype=np.int32)
    boxes = np.concatenate([synth.face_boxes(1, *sizes[i], seed=60 + k, border_fraction=0.25) for k, i in enumerate(index)])
    full = m.detect_faces(pinned, boxes, index)
    for i in range(len(index)):
        assert np.array_equal(m.detect_faces(pinned, boxes[i:i + 1], index[i:i + 1])[0], full[i]), f"face {i} alone"
    perm = np.random.default_rng(7).permutation(len(index))
    assert np.array_equal(m.detect_faces(pinned, boxes[perm], index[perm]), full[perm])
    assert np.array_equal(m.detect_faces(list(frames), boxes, index), full)          # pageable frames: device route
