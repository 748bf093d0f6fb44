"""Probes variants of the host-frame route of sd_detect_batch_host.  Development helper, not part of the product."""
import os, sys, time, numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from superviseddescent_b200 import api as sd
ctx = sd.Context(0)
m = sd.load_detection_model(bench.MODEL, ctx)
B = int(os.environ.get("B", "4096"))
frames = bench.synth_frames_torch(B, 1234, torch.device("cuda", 0))
boxes = bench.synth_boxes(B, 1234)
h = torch.empty((B, bench.H_IMG, bench.W_IMG), dtype=torch.uint8).pin_memory(); h.copy_(frames); torch.cuda.synchronize()
hn = h.numpy()
pageable = np.array(hn, copy=True)
def t(fn, n=5):
    for _ in range(2): fn()
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(n): r = fn()
    torch.cuda.synchronize(); return (time.perf_counter() - t0) / n * 1e3, r
f0 = ctx.roi_fallbacks()
ms, a = t(lambda: m.detect_batch(hn, boxes))
print("pinned (ROI route): %.2f ms/step -> %.0f faces/s, fallbacks %d" % (ms, B / ms * 1e3, ctx.roi_fallbacks() - f0))
ms2, b = t(lambda: m.detect_batch(pageable, boxes))
print("pageable (full frames): %.2f ms/step -> %.0f faces/s" % (ms2, B / ms2 * 1e3))
print("identical:", np.array_equal(a, b))
x0 = np.stack([sd.align_mean(m.get_mean(), bb) for bb in boxes]); x0d = torch.from_numpy(x0).cuda()
ms3, c = t(lambda: m.detect_batch_device(frames, x0d))
print("device resident: %.2f ms/step -> %.0f faces/s" % (ms3, B / ms3 * 1e3), np.array_equal(c.cpu().numpy(), a))
