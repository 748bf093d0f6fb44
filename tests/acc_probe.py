"""Accuracy probe (test infrastructure: it uses the CPU oracle): weights of a few systems vs float64 truth, per gram mode.
   python tests/acc_probe.py   on a GPU box"""
import sys, os, numpy as np
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE)); sys.path.insert(0, HERE)
from oracle import oracle as O
from superviseddescent_b200 import api as sd
ctx = sd.default_context()
def rel(a, b): return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))
def probe(name, A, B, lam):
    Xo, _ = O.solve(A, B, O.Regulariser(1, lam, 0), 1)
    Xf, _ = O.solve(A, B, O.Regulariser(1, lam, 0), 0)
    out = [f"f32-oracle {rel(Xf, Xo):.2e}"]
    for mode in (0, 3, 2):
        ctx.set_gram_mode(mode)
        lr = sd.LinearRegressor(sd.Regulariser(sd.RegularisationType.MatrixNorm, lam, False))
        lr.learn(A, B)
        X = lr.x.cpu().numpy()
        out.append(f"mode{mode} X {rel(X, Xo):.2e} pred {rel(A @ X, A @ Xo):.2e}")
    ctx.set_gram_mode(0)
    print(name, " | ".join(out), flush=True)
rng = np.random.default_rng(0)
A = rng.random((400, 300)).astype(np.float32); A[:, -1] = 1.0
B = rng.standard_normal((400, 8)).astype(np.float32)
probe("smoke 400x300 uniform", A, B, 1.0)
A = rng.random((3000, 1200)).astype(np.float32); A[:, -1] = 1.0
B = rng.standard_normal((3000, 44)).astype(np.float32)
probe("3000x1200 uniform", A, B, 1.5)
import test_gpu_regressor as T
A = T._features_like(np.random.default_rng(123), 1500, 700)
B = (0.05 * np.random.default_rng(5).standard_normal((1500, 44))).astype(np.float32)
probe("1500x700 hog-like", A, B, 1.5)
A = T._features_like(np.random.default_rng(7), 6000, 3000)
B = (0.05 * np.random.default_rng(8).standard_normal((6000, 44))).astype(np.float32)
probe("6000x3000 hog-like", A, B, 1.5)
