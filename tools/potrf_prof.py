"""Prints the clock64 phase timings of potrf_inv_kernel from the instrumented library (tools/build_prof.sh).
Development helper, not part of the product."""
import ctypes as C, os, sys, numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from superviseddescent_b200 import _capi
_capi.LIB_PATH = os.path.join(ROOT, "superviseddescent_b200", "lib_prof", "libsd_b200.so")
from superviseddescent_b200 import api as sd
rng = np.random.default_rng(0)
n, d = 2000, 1500
A = rng.random((n, d)).astype(np.float32); A[:, -1] = 1
B = rng.standard_normal((n, 8)).astype(np.float32)
lr = sd.LinearRegressor(sd.Regulariser(sd.RegularisationType.MatrixNorm, 1.0, False))
for _ in range(2): lr.learn(A, B)
torch.cuda.synchronize()
out = (C.c_longlong * 64)()
_capi.lib().sd_debug_read_clk(out)
v = [out[i] for i in range(17)]
names = ["load"] + sum([[f"potrf32[{k}]", f"panel[{k}]", f"trail[{k}]"] for k in range(4)], []) + ["(loop end)", "W assembly", "store"]
prev = v[0]
for i in range(1, 17):
    if v[i] == 0: continue
    print(f"{names[i-1]:14s} {v[i]-prev:8d} cycles"); prev = v[i]
print("total", v[16] - v[0])
