"""Generates tests/golden/examples_bgr.npz: the colour of the five annotated example frames of the reference, read exactly as
gen_golden.py reads them (cv2.imread, B,G,R) before converting them to the gray frames of examples.npz.

Run in the BUILD container only (needs /root/reference and cv2):

    python tests/golden/gen_examples_bgr.py

The raw B,G,R photographs would take 3.3 MB.  The fixture stores instead, per frame, the B - gray and R - gray differences
averaged over 4 x 4 pixel blocks (cb_i, cr_i: int8, 108 KB for the five).  tests/colour_examples.py rebuilds full-resolution
B,G,R frames from them and the gray frames of examples.npz, choosing G per pixel so that cv::cvtColor(BGR2GRAY) gives the gray
frame back exactly; each channel ends up within about one level of the photograph on average (printed below).
"""
import os
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import colour_examples  # noqa: E402

REF = "/root/reference"


def main():
    gray = np.load(os.path.join(HERE, "examples.npz"))
    out = {}
    for i in range(5):
        bgr = cv2.imread(f"{REF}/examples/data/ibug_lfpw_trainset/image_000{i + 1}.png")
        y = gray[f"gray{i}"]
        assert np.array_equal(cv2.cvtColor(bgr, cv2.COLOR_BGR2GRAY), y), i
        h, w = y.shape
        hb, wb = -(-h // 4) * 4, -(-w // 4) * 4

        def blocks(channel):
            d = np.pad(channel.astype(np.int64) - y, ((0, hb - h), (0, wb - w)), mode="edge").astype(np.float64)
            return np.clip(np.round(d.reshape(hb // 4, 4, wb // 4, 4).mean(axis=(1, 3))), -128, 127).astype(np.int8)
        out[f"cb{i}"], out[f"cr{i}"] = blocks(bgr[:, :, 0]), blocks(bgr[:, :, 2])
        rebuilt = colour_examples.rebuild(y, out[f"cb{i}"], out[f"cr{i}"])
        assert np.array_equal(cv2.cvtColor(rebuilt, cv2.COLOR_BGR2GRAY), y), i
        print("frame", i, "mean |rebuilt - photograph| per B,G,R channel:", np.abs(rebuilt.astype(int) - bgr).mean(axis=(0, 1)).round(2))
    np.savez_compressed(os.path.join(HERE, "examples_bgr.npz"), **out)
    print("examples_bgr.npz", os.path.getsize(os.path.join(HERE, "examples_bgr.npz")))


if __name__ == "__main__":
    main()
