"""Colour (8UC3 B,G,R) host frames through detection_model.detect_faces / detect_faces_from / detect_batch / detect
(sd_detect_faces_host, sd_detect_faces_host_init).  B,G,R -> gray is per pixel, so every face must come out bit-identical to
detecting it on the gray frame, on every route: the region-of-interest gather that converts as it reads, and the whole-frame
upload that converts on the device."""
import ctypes as C

import numpy as np
import pytest
import torch

import colour_examples
import synth
from superviseddescent_b200 import _capi

pytestmark = pytest.mark.gpu


def _pinned(frame, pitch=None):
    """A pinned CPU tensor view of an (H, W) or (H, W, 3) frame whose rows lie `pitch` bytes apart (default: packed)."""
    h, w = frame.shape[:2]
    c = frame.shape[2] if frame.ndim == 3 else 1
    pitch = pitch or w * c
    buf = torch.zeros(h * pitch + 16, dtype=torch.uint8).pin_memory()
    view = buf.as_strided((h, w, c), (pitch, c, 1))
    view.copy_(torch.from_numpy(np.ascontiguousarray(frame)).reshape(h, w, c))
    return view if c == 3 else view[:, :, 0]


def _inputs(frames):
    """The same frames as pageable arrays and as pinned tensors with a packed, a 16-byte aligned and an odd row pitch."""
    def row_bytes(f):
        return f.shape[1] * (f.shape[2] if f.ndim == 3 else 1)
    return {
        "pageable": list(frames),
        "pinned": [_pinned(f) for f in frames],
        "pinned, 16-byte pitch": [_pinned(f, (row_bytes(f) + 15) // 16 * 16) for f in frames],
        "pinned, odd pitch": [_pinned(f, (row_bytes(f) + 1) | 1) for f in frames],
    }


@pytest.fixture(scope="module")
def bgr_examples(golden):
    return colour_examples.load(golden.dir)


def test_colour_photographs_equal_gray_detect_and_the_reference(sd, golden, bgr_examples):
    m = sd.load_detection_model(golden.model_path)
    grays = [np.ascontiguousarray(golden.examples[f"gray{i}"]) for i in range(5)]
    rng = np.random.default_rng(11)
    order = list(rng.permutation(5)) + [3, 0]                  # shuffled, two frames listed twice
    frames = [bgr_examples[i] for i in order]
    index = list(rng.permutation(len(frames)))
    boxes = [golden.examples["boxes"][order[f]] for f in index]
    # two more faces on the frame listed first: its own box again and an overlapping shifted one (one merged ROI)
    b = golden.examples["boxes"][order[0]]
    shifted = np.array([b[0] + b[2] // 6, b[1] - b[3] // 8, b[2], b[3]], dtype=np.int32)
    index += [0, 0]
    boxes += [b, shifted]
    index = np.array(index, dtype=np.int32)
    boxes = np.stack(boxes).astype(np.int32)
    single = [m.detect(grays[order[f]], boxes[k]) for k, f in enumerate(index)]
    for name, inp in _inputs(frames).items():
        got = m.detect_faces(inp, boxes, index)
        for k, f in enumerate(index):
            assert np.array_equal(got[k], single[k]), (name, k)
            if k <= len(frames):                                 # the faces with the photograph's own box
                ref = golden.detect[f"landmarks{order[f]}"]
                assert np.max(np.abs(got[k] - ref)) <= 1e-4 * np.max(np.abs(ref)), (name, k)
    # one face per frame through detect_batch, and detect(image, facebox), on colour input
    for i in (1, 3):
        assert np.array_equal(m.detect(bgr_examples[i], golden.examples["boxes"][i]), m.detect(grays[i], golden.examples["boxes"][i]))
    two = np.stack([bgr_examples[2], bgr_examples[2]])
    b2 = np.stack([golden.examples["boxes"][2], golden.examples["boxes"][2] + np.array([5, -3, 0, 0])]).astype(np.int32)
    assert np.array_equal(m.detect_batch(two, b2), m.detect_batch(np.stack([grays[2], grays[2]]), b2))
    assert np.array_equal(m.detect_batch(torch.from_numpy(two).pin_memory(), b2), m.detect_batch(np.stack([grays[2], grays[2]]), b2))


def _colour_frame(h, w, seed):
    """Independent smooth B, G and R planes, so the conversion weights all matter."""
    planes = [synth.smooth_images(1, h, w, seed=seed + c)[0] for c in range(3)]
    return np.ascontiguousarray(np.stack(planes, axis=2))


def _mixed_call():
    sizes = [(480, 640), (360, 500), (600, 800), (240, 333), (480, 640), (300, 417)]
    frames = []
    for k, (h, w) in enumerate(sizes):
        f = _colour_frame(h, w, seed=100 + 10 * k)
        frames.append(f if k % 3 != 1 else np.ascontiguousarray(f[:, :, 1]))     # frames 1 and 4 gray
    rng = np.random.default_rng(77)
    per_frame = [3, 2, 0, 1, 4, 2]                                                  # frame 2 has no faces
    index, boxes = [], []
    for f, n in enumerate(per_frame):
        if n == 0:
            continue
        h, w = sizes[f]
        bs = synth.face_boxes(n, h, w, seed=200 + f, border_fraction=0.25)
        if n >= 2:                                                                   # overlapping faces: one merged ROI
            bs[1, 0], bs[1, 1] = bs[0, 0] + bs[0, 2] // 5, bs[0, 1] + bs[0, 3] // 7
        index += [f] * n
        boxes.append(bs)
    boxes = np.concatenate(boxes).astype(np.int32)
    perm = rng.permutation(len(index))
    return frames, boxes[perm], np.array(index, dtype=np.int32)[perm]


def test_mixed_gray_and_colour_frames_of_mixed_sizes(sd, golden):
    m = sd.load_detection_model(golden.model_path)
    frames, boxes, index = _mixed_call()
    converted = [sd.bgr2gray(f[None], m.ctx)[0].cpu().numpy() if f.ndim == 3 else f for f in frames]
    ref = m.detect_faces(converted, boxes, index)
    device = m.detect_faces_device([torch.from_numpy(f).cuda() for f in frames], index, m.align_boxes(boxes)).cpu().numpy()
    assert np.array_equal(device, ref)
    fb0 = m.ctx.roi_fallbacks()
    for name, inp in _inputs(frames).items():
        assert np.array_equal(m.detect_faces(inp, boxes, index), ref), name
    print("ROI route: fallbacks", m.ctx.roi_fallbacks() - fb0)
    # a batch of equally sized colour frames, one (n, H, W, 3) array, pageable and pinned
    batch = np.stack([_colour_frame(240, 320, seed=300 + k) for k in range(4)])
    bidx = np.array([0, 1, 1, 3, 3, 3], dtype=np.int32)
    bboxes = synth.face_boxes(6, 240, 320, seed=5, border_fraction=0.2)
    bref = m.detect_faces(list(sd.bgr2gray(batch, m.ctx).cpu().numpy()), bboxes, bidx)
    assert np.array_equal(m.detect_faces(batch, bboxes, bidx), bref)
    assert np.array_equal(m.detect_faces(torch.from_numpy(batch).pin_memory(), bboxes, bidx), bref)


def test_detect_from_initialisations(sd, golden, bgr_examples):
    m = sd.load_detection_model(golden.model_path)
    frames, boxes, index = _mixed_call()
    x0 = m.align_boxes(boxes).cpu().numpy()
    x0 += np.float32(3.0) * np.sin(np.arange(x0.size, dtype=np.float32)).reshape(x0.shape)   # not the aligned mean
    ref = m.detect_faces_device([torch.from_numpy(f).cuda() for f in frames], index, torch.from_numpy(x0).cuda()).cpu().numpy()
    for name, inp in _inputs(frames).items():
        assert np.array_equal(m.detect_faces_from(inp, x0, index), ref), name
    gray_only = [f if f.ndim == 2 else np.ascontiguousarray(f[:, :, 0]) for f in frames]
    gref = m.detect_faces_device([torch.from_numpy(f).cuda() for f in gray_only], index, torch.from_numpy(x0).cuda()).cpu().numpy()
    assert np.array_equal(m.detect_faces_from(gray_only, x0, index), gref)
    assert np.array_equal(m.detect_faces_from([_pinned(f) for f in gray_only], x0, index), gref)
    # the tracking call on one colour photograph: detect(colour, initialisation) == detect(gray, initialisation)
    gray = np.ascontiguousarray(golden.examples["gray1"])
    init = m.detect(gray, golden.examples["boxes"][1]) + np.float32(1.5)
    got = m.detect(bgr_examples[1], init)
    assert np.array_equal(got, m.detect(gray, init))
    assert np.array_equal(got, m.detect_faces_device(torch.from_numpy(gray).cuda()[None], np.zeros(1, np.int32), init[None]).cpu().numpy()[0])
    assert np.array_equal(m.detect(_pinned(bgr_examples[1]), init), got)


def test_errors_and_empty_calls(sd, golden):
    m = sd.load_detection_model(golden.model_path)
    frame = _colour_frame(120, 160, seed=9)
    boxes = synth.face_boxes(2, 120, 160, seed=9)
    idx = np.array([0, 0], dtype=np.int32)
    x0 = np.ascontiguousarray(m.align_boxes(boxes).cpu().numpy())
    out = np.empty((2, 2 * m.num_landmarks), dtype=np.float32)
    lib = _capi.lib()

    def call(hf, count=2, init=False):
        if init:
            return lib.sd_detect_faces_host_init(m.ctx.h, m._m, C.byref(hf), 1, idx.ctypes.data_as(C.c_void_p), x0.ctypes.data_as(C.c_void_p),
                                                 C.c_int64(2 * m.num_landmarks), count, out.ctypes.data_as(C.c_void_p))
        return lib.sd_detect_faces_host(m.ctx.h, m._m, C.byref(hf), 1, idx.ctypes.data_as(C.c_void_p), boxes.ctypes.data_as(C.c_void_p), count,
                                        out.ctypes.data_as(C.c_void_p))
    launches = m.ctx.launches()
    for init in (False, True):
        for channels in (2, 4, -1):
            assert call(_capi.HostFrameC(frame.ctypes.data, 160, 120, 480, channels), init=init) == 1
        assert call(_capi.HostFrameC(frame.ctypes.data, 160, 120, 479, 3), init=init) == 1          # pitch below 3 x width
        assert call(_capi.HostFrameC(frame.ctypes.data, 160, 120, 480, 4), count=0, init=init) == 0   # nothing to do
    assert lib.sd_detect_faces_host_init(m.ctx.h, m._m, C.byref(_capi.HostFrameC(frame.ctypes.data, 160, 120, 480, 3)), 1,
                                         idx.ctypes.data_as(C.c_void_p), x0.ctypes.data_as(C.c_void_p), C.c_int64(2 * m.num_landmarks - 1), 2,
                                         out.ctypes.data_as(C.c_void_p)) == 1                          # ldx below 2L
    assert m.ctx.launches() == launches
    # the context stays usable; a good colour record works, and empty Python calls return empty results
    assert call(_capi.HostFrameC(frame.ctypes.data, 160, 120, 480, 3)) == 0
    assert np.array_equal(out, m.detect_faces([frame], boxes, idx))
    assert m.detect_faces([frame], np.zeros((0, 4), np.int32), np.zeros(0, np.int32)).shape == (0, 2 * m.num_landmarks)
    assert m.detect_faces_from([frame], np.zeros((0, 2 * m.num_landmarks), np.float32), np.zeros(0, np.int32)).shape == (0, 2 * m.num_landmarks)
