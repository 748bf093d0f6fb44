"""Several faces per frame, frames of any size: detection_model.detect_faces / detect_faces_device / align_boxes
(sd_detect_faces_host, sd_detect_faces_device, sd_model_align_boxes).  Every face must come out bit-identical to detecting it
alone on its own frame."""
import numpy as np
import pytest
import torch

import synth
from superviseddescent_b200._capi import SdError

pytestmark = pytest.mark.gpu


def _pinned_frames(frames, pad=False):
    """One pinned CPU tensor per frame; pad=True gives rows a 16-byte aligned pitch (a view into a wider buffer)."""
    out = []
    for f in frames:
        h, w = f.shape
        stride = (w + 15) // 16 * 16 if pad else w
        buf = torch.zeros((h, stride), dtype=torch.uint8).pin_memory()
        buf[:, :w].copy_(torch.from_numpy(np.ascontiguousarray(f)))
        out.append(buf[:, :w])
    return out


def test_align_boxes_equals_host_align_mean(sd, golden):
    m = sd.load_detection_model(golden.model_path)
    rng = np.random.default_rng(2024)
    n = 1000
    boxes = np.stack([rng.integers(-500, 1500, n), rng.integers(-500, 1500, n), rng.integers(1, 2001, n), rng.integers(1, 2001, n)],
                     axis=1).astype(np.int32)
    got = m.align_boxes(boxes).cpu().numpy()
    mean = m.get_mean()
    ref = np.stack([sd.align_mean(mean, b) for b in boxes])
    assert np.array_equal(got, ref)


def _several_faces_per_frame():
    H, W = 480, 640
    frames = synth.smooth_images(8, H, W, seed=4321)
    rng = np.random.default_rng(4321)
    per_frame = rng.integers(0, 7, 8)
    per_frame[0], per_frame[3] = 0, 6                        # a frame without faces, a frame with six
    total = int(per_frame.sum())
    boxes = synth.face_boxes(total, H, W, seed=4321, border_fraction=0.25)
    index = np.repeat(np.arange(8), per_frame).astype(np.int32)
    # overlapping faces: the second face of a frame is moved next to the first
    k = 0
    for f in range(8):
        if per_frame[f] >= 2:
            boxes[k + 1, 0] = boxes[k, 0] + boxes[k, 2] // 5
            boxes[k + 1, 1] = boxes[k, 1] + boxes[k, 3] // 7
        k += per_frame[f]
    perm = rng.permutation(total)                              # faces in any order
    return frames, boxes[perm], index[perm]


def test_several_faces_per_frame_equal_duplicated_frames(sd, golden):
    m = sd.load_detection_model(golden.model_path)
    frames, boxes, index = _several_faces_per_frame()
    ref = m.detect_batch(np.ascontiguousarray(frames[index]), boxes)
    pageable = m.detect_faces(list(frames), boxes, index)
    assert np.array_equal(pageable, ref)
    assert np.array_equal(m.detect_faces(frames, boxes, index), ref)            # one (n, H, W) array
    fb0 = m.ctx.roi_fallbacks()
    pinned = m.detect_faces(_pinned_frames(frames), boxes, index)
    print("ROI route: fallbacks", m.ctx.roi_fallbacks() - fb0, "of", len(boxes))
    assert np.array_equal(pinned, ref)
    assert np.array_equal(m.detect_faces(torch.from_numpy(frames).pin_memory(), boxes, index), ref)
    dev_frames = torch.from_numpy(frames).cuda()
    device = m.detect_faces_device(dev_frames, index, m.align_boxes(boxes)).cpu().numpy()
    assert np.array_equal(device, ref)
    # determinism
    assert np.array_equal(m.detect_faces(list(frames), boxes, index), pageable)
    assert np.array_equal(m.detect_faces(_pinned_frames(frames), boxes, index), pinned)


def test_mixed_sizes_against_the_reference(sd, golden):
    m = sd.load_detection_model(golden.model_path)
    grays = [np.ascontiguousarray(golden.examples[f"gray{i}"]) for i in range(5)]
    assert len({g.shape for g in grays}) == 5
    rng = np.random.default_rng(5)
    order = list(rng.permutation(5)) + [3, 0]                  # shuffled, two frames listed twice
    frames = [grays[i] for i in order]
    index = np.array(list(rng.permutation(len(frames))), dtype=np.int32)
    boxes = np.stack([golden.examples["boxes"][order[f]] for f in index]).astype(np.int32)
    single = [m.detect(grays[i], golden.examples["boxes"][i]) for i in range(5)]
    routes = {
        "pageable": m.detect_faces(frames, boxes, index),
        "pinned": m.detect_faces(_pinned_frames(frames), boxes, index),
        "pinned, aligned pitch": m.detect_faces(_pinned_frames(frames, pad=True), boxes, index),
        "colour": m.detect_faces([np.repeat(f[:, :, None], 3, axis=2) for f in frames], boxes, index),
        "device": m.detect_faces_device([torch.from_numpy(f).cuda() for f in frames], index, m.align_boxes(boxes)).cpu().numpy(),
    }
    for name, got in routes.items():
        for k, f in enumerate(index):
            i = order[f]
            ref = golden.detect[f"landmarks{i}"]
            assert np.max(np.abs(got[k] - ref)) <= 1e-4 * np.max(np.abs(ref)), (name, k)
            assert np.array_equal(got[k], single[i]), (name, k)


def test_errors_and_empty_calls(sd, golden):
    m = sd.load_detection_model(golden.model_path)
    frames = synth.smooth_images(3, 240, 320, seed=9)
    boxes = synth.face_boxes(2, 240, 320, seed=9)
    launches = m.ctx.launches()
    for bad in (-1, 3):
        with pytest.raises(SdError) as e:
            m.detect_faces(list(frames), boxes, np.array([0, bad], dtype=np.int32))
        assert e.value.code == 1
    # the C entry point itself checks the indices before queueing anything
    import ctypes as C
    from superviseddescent_b200 import _capi
    hf = (_capi.HostFrameC * 3)(*[_capi.HostFrameC(f.ctypes.data, 320, 240, 320, 0) for f in frames])
    out = np.empty((2, 2 * m.num_landmarks), dtype=np.float32)
    for bad in (-1, 3):
        idx = np.array([1, bad], dtype=np.int32)
        rc = _capi.lib().sd_detect_faces_host(m.ctx.h, m._m, hf, 3, idx.ctypes.data_as(C.c_void_p), boxes.ctypes.data_as(C.c_void_p), 2,
                                              out.ctypes.data_as(C.c_void_p))
        assert rc == 1
    assert m.ctx.launches() == launches
    # device route: reported through the projection's status flag
    with pytest.raises(SdError) as e:
        m.detect_faces_device(torch.from_numpy(frames).cuda(), np.array([0, 3], dtype=np.int32), m.align_boxes(boxes))
    assert e.value.code == 1
    # the context stays usable, and count == 0 is an empty result
    assert np.array_equal(m.detect_faces(list(frames), boxes, np.array([2, 2], dtype=np.int32)),
                          m.detect_batch(np.ascontiguousarray(frames[[2, 2]]), boxes))
    empty = m.detect_faces(list(frames), np.zeros((0, 4), dtype=np.int32), np.zeros(0, dtype=np.int32))
    assert empty.shape == (0, 2 * m.num_landmarks)
