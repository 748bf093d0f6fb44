"""The five example photographs of the reference as 8UC3 B,G,R frames, rebuilt from their gray frames (examples.npz) and the
4 x 4 block colour differences in examples_bgr.npz (tests/golden/gen_examples_bgr.py).  cv::cvtColor(BGR2GRAY) of every
rebuilt frame is its gray frame, pixel for pixel."""
import os

import numpy as np


def rebuild(gray, cb, cr):
    """(H, W, 3) uint8 B,G,R from an (H, W) gray frame and the block differences B - gray (cb) and R - gray (cr).  G is the
    smallest value with (3735 B + 19235 G + 9798 R + 2^14) >> 15 == gray; where none exists the pixel is B = G = R = gray."""
    y = gray.astype(np.int64)
    h, w = y.shape

    def up(d):
        return np.repeat(np.repeat(d.astype(np.int64), 4, axis=0), 4, axis=1)[:h, :w]
    b = np.clip(y + up(cb), 0, 255)
    r = np.clip(y + up(cr), 0, 255)
    # one more G raises the weighted sum by 19235 < 2^15, so the output takes every value between its ends: the smallest G
    # that reaches gray gives exactly gray
    g = np.clip(-(-((y << 15) - (1 << 14) - 3735 * b - 9798 * r) // 19235), 0, 255)
    ok = ((3735 * b + 19235 * g + 9798 * r + (1 << 14)) >> 15) == y
    return np.stack([np.where(ok, c, y) for c in (b, g, r)], axis=2).astype(np.uint8)


def load(golden_dir):
    """[bgr_0 .. bgr_4], the frames of examples.npz's gray0 .. gray4 in colour."""
    gray = np.load(os.path.join(golden_dir, "examples.npz"))
    d = np.load(os.path.join(golden_dir, "examples_bgr.npz"))
    return [rebuild(gray[f"gray{i}"], d[f"cb{i}"], d[f"cr{i}"]) for i in range(5)]
