"""Times the HOG launch of every cascade level and the whole device-resident detect step (development helper for comparing
two builds of the library): python tools/hog_ab.py [batch] [--dump DIR]

--dump DIR also writes each level's descriptors as DIR/hog_level<i>.npy, so that two builds can be compared bit for bit."""
import ctypes as C, os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
from superviseddescent_b200 import api as sd, _capi
args = sys.argv[1:]
DUMP = None
if "--dump" in args:
    i = args.index("--dump")
    DUMP = args[i + 1]
    del args[i:i + 2]
    os.makedirs(DUMP, exist_ok=True)
B = int(args[0]) if args else 4096
dev = torch.device("cuda", 0)
ctx = sd.Context(0)
model = sd.load_detection_model(bench.MODEL, ctx)
L = model.num_landmarks
frames = bench.synth_frames_torch(B, 1234, dev)
boxes = bench.synth_boxes(B, 1234)
x0 = torch.from_numpy(np.stack([sd.align_mean(model.get_mean(), b) for b in boxes])).to(dev)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
out = []
for level in range(model.num_levels):
    hp = model.hog_param(level)
    D = _capi.lib().sd_hog_feature_length(L, C.byref(hp))
    ld = (D + 3) // 4 * 4
    A = torch.empty((B, ld), dtype=torch.float32, device=dev)
    norm = sd.NormalisationC()
    _capi.lib().sd_model_normalisation(model._m, C.byref(norm))
    ib = sd.ImageBatchC(C.c_void_p(frames.data_ptr()), bench.W_IMG, bench.H_IMG, frames.stride(1), frames.stride(0), B)
    def hog():
        assert _capi.lib().sd_hog_batch(ctx.h, C.byref(ib), None, _capi.ptr(x0), C.c_int64(2 * L), B, L, C.byref(norm), C.byref(hp), _capi.ptr(A), C.c_int64(ld)) == 0
    for _ in range(3): hog()
    torch.cuda.synchronize(); e0.record()
    for _ in range(10): hog()
    e1.record(); torch.cuda.synchronize()
    out.append(round(e0.elapsed_time(e1) / 10, 4))
    if DUMP:
        np.save(os.path.join(DUMP, f"hog_level{level}.npy"), A[:, :D].cpu().numpy())
for _ in range(3): model.detect_batch_device(frames, x0)
torch.cuda.synchronize(); e0.record()
for _ in range(5): model.detect_batch_device(frames, x0)
e1.record(); torch.cuda.synchronize()
print(f"hog ms per level {out} sum {sum(out):.3f}; detect step {e0.elapsed_time(e1) / 5:.3f} ms ({B * 5 / e0.elapsed_time(e1) * 1e3:.0f} faces/s)", flush=True)
