"""Faces/s of detection with several faces per frame (detection_model.detect_faces / detect_faces_device) against the same faces
through the one-face-per-frame calls on frames duplicated once per face.

    python tools/bench_faces.py [--frames 1024] [--reps 5] [--cases a,b,c,d] [--out DIR]

(a) device-resident 640x480 frames with 1, 4 and 16 faces each: detect_faces_device vs detect_batch_device on duplicated frames
(b) the same from pinned and from pageable host frames: detect_faces vs detect_batch (sd_detect_batch_host) on duplicated frames
(c) frames of mixed sizes vs equally sized 640x480 frames with the same number of faces, on each route
(d) colour 640x480 B,G,R host frames (independent B, G and R planes) with 1, 4 and 16 faces each, pinned and pageable:
    detect_faces, which converts only each face's neighbourhood (pinned) or each frame once on the device (pageable), against
    the route without it, built from public calls: bgr2gray of the whole host batch + align_boxes + detect_faces_device

Prints the card's name and power limit first, then one JSON line per measurement; with --out also writes them to DIR/bench_faces.json.
Every pair of rates is checked to give bit-identical landmarks.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
MODEL = os.path.join(ROOT, "tests", "golden", "face_landmarks_model_rcr_22.bin")
MIXED_SIZES = [(480, 640), (600, 800), (768, 1024), (360, 480), (720, 1280), (412, 600)]   # (H, W)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def smooth_frame(h, w, gen, dev):
    """Low-pass filtered uniform noise (sigma = 3 px) stretched to 0..255, 8UC1, generated on the GPU."""
    sigma, r = 3.0, 9
    k = torch.exp(-0.5 * (torch.arange(-r, r + 1, device=dev, dtype=torch.float32) / sigma) ** 2)
    k = k / k.sum()
    x = torch.rand((1, 1, h + 2 * r, w + 2 * r), generator=gen, device=dev)
    x = F.conv2d(F.conv2d(x, k.view(1, 1, -1, 1)), k.view(1, 1, 1, -1))[0, 0]
    x = (x - x.min()) / (x.max() - x.min())
    return torch.round(x * 255).to(torch.uint8)


def grid_boxes(h, w, k, rng):
    """k square faces on a ceil(sqrt(k))-wide grid of the frame, each 60-75 % of its cell, jittered inside it."""
    g = int(np.ceil(np.sqrt(k)))
    cw, ch = w // g, h // g
    out = []
    for j in range(k):
        cx, cy = (j % g) * cw, (j // g) * ch
        s = int(min(cw, ch) * rng.uniform(0.6, 0.75))
        out.append((cx + int(rng.integers(0, cw - s + 1)), cy + int(rng.integers(0, ch - s + 1)), s, s))
    return out


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--faces", default="1,4,16")
    ap.add_argument("--cases", default="a,b,c,d")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_faces needs a CUDA device")
    from superviseddescent_b200 import api as sd
    dev = torch.device("cuda", 0)
    m = sd.load_detection_model(MODEL)
    gen = torch.Generator(device=dev)
    gen.manual_seed(7)
    rng = np.random.default_rng(7)
    results = [{"card": card(), "frames": args.frames, "reps": args.reps}]
    print(json.dumps(results[0]), flush=True)

    def report(**kw):
        results.append(kw)
        print(json.dumps(kw), flush=True)

    n = args.frames
    cases = set(args.cases.split(","))
    if "d" in cases:
        colour_case(m, sd, n, args, gen, rng, dev, report)
    if not cases & {"a", "b", "c"}:
        return finish(args, results)
    frames = torch.stack([smooth_frame(480, 640, gen, dev) for _ in range(n)])
    frames_pinned = frames.cpu().pin_memory()
    frames_np = frames.cpu().numpy()
    for k in [int(v) for v in args.faces.split(",")] if cases & {"a", "b"} else []:
        boxes = np.array([b for _ in range(n) for b in grid_boxes(480, 640, k, rng)], dtype=np.int32)
        index = np.repeat(np.arange(n, dtype=np.int32), k)
        faces = len(boxes)
        # (a) device-resident
        idx_dev = torch.from_numpy(index).to(dev)
        x0 = m.align_boxes(boxes)
        dup = frames[idx_dev.long()]
        t_new, got = timed(lambda: m.detect_faces_device(frames, idx_dev, x0), args.reps)
        t_dup, ref = timed(lambda: m.detect_batch_device(dup, x0), args.reps)
        assert torch.equal(got, ref)
        ref = ref.cpu().numpy()
        report(case="a", route="device", faces_per_frame=k, faces=faces, faces_per_s=faces / t_new, duplicated_faces_per_s=faces / t_dup)
        del dup
        # (b) host frames: pinned (region-of-interest gather) and pageable (each frame uploaded once)
        dup_pinned = frames_pinned[torch.from_numpy(index).long()].pin_memory()
        t_new, got = timed(lambda: m.detect_faces(frames_pinned, boxes, index), args.reps)
        assert np.array_equal(got, ref)
        fb = m.ctx.roi_fallbacks()
        t_dup, got = timed(lambda: m.detect_batch(dup_pinned.numpy(), boxes), args.reps)
        assert np.array_equal(got, ref)
        report(case="b", route="pinned", faces_per_frame=k, faces=faces, faces_per_s=faces / t_new, duplicated_faces_per_s=faces / t_dup,
               roi_fallbacks_per_call=(m.ctx.roi_fallbacks() - fb) / (args.reps + 1))
        del dup_pinned
        dup_np = frames_np[index]
        t_new, got = timed(lambda: m.detect_faces(frames_np, boxes, index), args.reps)
        assert np.array_equal(got, ref)
        t_dup, got = timed(lambda: m.detect_batch(dup_np, boxes), args.reps)
        assert np.array_equal(got, ref)
        report(case="b", route="pageable", faces_per_frame=k, faces=faces, faces_per_s=faces / t_new, duplicated_faces_per_s=faces / t_dup)
        del dup_np

    if "c" not in cases:
        return finish(args, results)
    # (c) mixed sizes against equally sized frames, 4 faces per frame
    k = 4
    sizes = [MIXED_SIZES[i % len(MIXED_SIZES)] for i in range(n)]
    mixed = [smooth_frame(h, w, gen, dev) for h, w in sizes]
    mboxes = np.array([b for (h, w) in sizes for b in grid_boxes(h, w, k, rng)], dtype=np.int32)
    uboxes = np.array([b for _ in range(n) for b in grid_boxes(480, 640, k, rng)], dtype=np.int32)
    index = np.repeat(np.arange(n, dtype=np.int32), k)
    idx_dev = torch.from_numpy(index).to(dev)
    mx0, ux0 = m.align_boxes(mboxes), m.align_boxes(uboxes)

    def pinned_aligned(fs):
        out = []
        for f in fs:
            h, w = f.shape
            buf = torch.zeros((h, (w + 15) // 16 * 16), dtype=torch.uint8).pin_memory()
            buf[:, :w].copy_(f)
            out.append(buf[:, :w])
        return out
    # the mixed frames packed on the device once (pack_frames), called through the C ABI so that packing is not timed
    import ctypes as C
    from superviseddescent_b200 import _capi
    data, table = sd.pack_frames(mixed, m.ctx)
    ib = sd.ImageBatchC(C.c_void_p(data.data_ptr()), 0, 0, 0, 0, n, None, None, C.c_void_p(table.data_ptr()))

    def mixed_device():
        out = torch.empty((len(mboxes), 2 * m.num_landmarks), dtype=torch.float32, device=dev)
        rc = _capi.lib().sd_detect_faces_device(m.ctx.h, m._m, C.byref(ib), _capi.ptr(idx_dev), _capi.ptr(mx0), len(mboxes), _capi.ptr(out))
        assert rc == 0
        return out
    routes = {
        "device": (mixed_device, lambda: m.detect_faces_device(frames, idx_dev, ux0)),
        "pinned": (lambda fs=pinned_aligned(mixed): m.detect_faces(fs, mboxes, index), lambda: m.detect_faces(frames_pinned, uboxes, index)),
        "pageable": (lambda fs=[f.cpu().numpy() for f in mixed]: m.detect_faces(fs, mboxes, index), lambda: m.detect_faces(frames_np, uboxes, index)),
    }
    ref = None
    for route, (fm, fu) in routes.items():
        t_m, got = timed(fm, args.reps)
        got = got.cpu().numpy() if isinstance(got, torch.Tensor) else got
        if ref is None:
            ref = got
        assert np.array_equal(got, ref)
        t_u, _ = timed(fu, args.reps)
        report(case="c", route=route, faces_per_frame=k, faces=len(mboxes), mixed_faces_per_s=len(mboxes) / t_m, uniform_faces_per_s=len(uboxes) / t_u,
               mixed_sizes=sorted({f"{w}x{h}" for h, w in sizes}))
    finish(args, results)


def colour_case(m, sd, n, args, gen, rng, dev, report):
    """(d): colour host frames through detect_faces against bgr2gray of the whole batch + align_boxes + detect_faces_device."""
    frames = torch.stack([torch.stack([smooth_frame(480, 640, gen, dev) for _ in range(3)], dim=2) for _ in range(n)])
    frames_pinned = frames.cpu().pin_memory()
    frames_np = frames.cpu().numpy()
    del frames
    for k in [int(v) for v in args.faces.split(",")]:
        boxes = np.array([b for _ in range(n) for b in grid_boxes(480, 640, k, rng)], dtype=np.int32)
        index = np.repeat(np.arange(n, dtype=np.int32), k)
        for route, host in (("pinned", frames_pinned), ("pageable", frames_np)):
            fb = m.ctx.roi_fallbacks()
            t_new, got = timed(lambda: m.detect_faces(host, boxes, index), args.reps)
            fallbacks = (m.ctx.roi_fallbacks() - fb) / (args.reps + 1)
            t_old, ref = timed(lambda: m.detect_faces_device(sd.bgr2gray(host, m.ctx), index, m.align_boxes(boxes)).cpu().numpy(), args.reps)
            assert np.array_equal(got, ref)
            report(case="d", route=route, faces_per_frame=k, faces=len(boxes), faces_per_s=len(boxes) / t_new,
                   whole_frame_bgr2gray_faces_per_s=len(boxes) / t_old, roi_fallbacks_per_call=fallbacks)


def finish(args, results):
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_faces.json"), "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
