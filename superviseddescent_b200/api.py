"""Host-side mirror of the reference's public interface for the hot path, on top of the C ABI.

Class and method names follow patrikhuber/superviseddescent:
  Regulariser, LinearRegressor                  include/superviseddescent/regressors.hpp:87-169, 318-400
  SupervisedDescentOptimiser, NoNormalisation    include/superviseddescent/superviseddescent.hpp:60-74, 85-361
  HoGParam, HogTransform                         include/rcr/adaptive_vlhog.hpp:41-60, 70-195
  InterEyeDistanceNormalisation, align_mean,
  detection_model, load/save_detection_model     include/rcr/model.hpp:64-219

The C++14 header shells (superviseddescent_b200/include/) are the drop-in for C++ callers; this module
is the same surface for Python callers, the tests and bench.py.  Matrices are row-major float32, one
sample per row; on the device they are torch CUDA tensors (torch = allocator + stream + distributed
plumbing only -- every computation below is a kernel of libsd_b200.so).
"""
from __future__ import annotations

import ctypes as C
import enum
from typing import Callable, List, Optional, Sequence

import numpy as np
import torch

from . import _capi
from ._capi import HogParam as HoGParam  # same field names as rcr::HoGParam
from ._capi import ImageBatchC, NormalisationC, RegulariserC, SdError, ptr


def _check(ctx, rc: int) -> None:
    if rc != 0:
        msg = _capi.lib().sd_last_error(ctx).decode() if ctx else "no context"
        raise SdError(rc, msg)


class Context:
    """One sd_ctx bound to a device and to torch's current stream on it."""

    def __init__(self, device: int = 0):
        if not torch.cuda.is_available():
            raise SdError(2, "no CUDA device: the B200 engine has no CPU fallback")
        self.device = int(device)
        torch.cuda.set_device(self.device)
        self.stream = torch.cuda.current_stream(self.device)
        self._h = C.c_void_p()
        rc = _capi.lib().sd_ctx_create(self.device, C.c_void_p(self.stream.cuda_stream), C.byref(self._h))
        if rc != 0:
            raise SdError(rc, "sd_ctx_create failed (is a CUDA device visible?)")

    @property
    def h(self):
        return self._h

    def sync(self):
        _check(self._h, _capi.lib().sd_sync(self._h))

    def launches(self) -> int:
        return int(_capi.lib().sd_launch_count(self._h))

    def roi_fallbacks(self) -> int:
        return int(_capi.lib().sd_roi_fallback_count(self._h))

    def set_gram_mode(self, mode: int):
        """0 = 3xTF32 tensor-core Gram (default), 3 = unbiased 3xTF32, 1 = single-pass TF32, 2 = fp32 SIMT."""
        _check(self._h, _capi.lib().sd_set_gram_mode(self._h, int(mode)))

    def set_solver(self, mode) -> None:
        """Solver of systems with D > 256: 0 / "cholesky" = blocked Cholesky (default), 1 / "cg" = conjugate gradients on the
        tensor cores (falls back to the Cholesky if they stall)."""
        m = {"cholesky": 0, "cg": 1}.get(mode, mode)
        _check(self._h, _capi.lib().sd_set_solver(self._h, int(m)))

    def solver_iterations(self) -> int:
        """CG iterations of the last solve (0: the factorisation ran)."""
        return int(_capi.lib().sd_solver_iterations(self._h))

    def solver_timings(self):
        out = (C.c_float * 4)()
        _check(self._h, _capi.lib().sd_solver_timings(self._h, out))
        return {"At * A": out[0], "AtA + Reg": out[1], "Decomposition": out[2], "solve()": out[3]}

    def close(self):
        if self._h:
            _capi.lib().sd_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_ctx: Optional[Context] = None


def default_context() -> Context:
    global _default_ctx
    if _default_ctx is None:
        dev = torch.cuda.current_device() if torch.cuda.is_available() else 0
        _default_ctx = Context(dev)
    return _default_ctx


def _dev(a, ctx: Context, dtype=torch.float32) -> torch.Tensor:
    if isinstance(a, torch.Tensor):
        t = a.to(device=f"cuda:{ctx.device}", dtype=dtype)
    else:
        t = torch.from_numpy(np.ascontiguousarray(a)).to(device=f"cuda:{ctx.device}", dtype=dtype)
    return t.contiguous()


# ------------------------------------------------------------------------------------------------
# regressors.hpp
# ------------------------------------------------------------------------------------------------
class RegularisationType(enum.IntEnum):
    Manual = 0
    MatrixNorm = 1


class Regulariser:
    """superviseddescent::Regulariser (regressors.hpp:87-169)."""

    RegularisationType = RegularisationType

    def __init__(self, regularisation_type: RegularisationType = RegularisationType.Manual, param: float = 0.0,
                 regularise_last_row: bool = True):
        self.regularisation_type = RegularisationType(regularisation_type)
        self.param = float(param)
        self.regularise_last_row = bool(regularise_last_row)

    def c(self) -> RegulariserC:
        return RegulariserC(int(self.regularisation_type), self.param, int(self.regularise_last_row))


class PartialPivLUSolver:
    """regressors.hpp:180-235 (also VerbosePartialPivLUSolver): the default Solver."""
    rank_revealing = False


class ColPivHouseholderQRSolver:
    """regressors.hpp:245-306: the Solver that checks invertibility.  Same solve, plus the numerical rank of the regularised
    AtA (diagonally pivoted Cholesky on the device); a deficient rank prints the reference's message (:290-293)."""
    rank_revealing = True


class LinearRegressor:
    """superviseddescent::LinearRegressor<Solver> (regressors.hpp:318-400); `solver` plays the template parameter."""

    def __init__(self, regulariser: Optional[Regulariser] = None, ctx: Optional[Context] = None, solver=None):
        self.regulariser = regulariser or Regulariser()
        self.ctx = ctx
        self.solver = solver or PartialPivLUSolver()
        self.x: Optional[torch.Tensor] = None   # D x M, device
        self.last_lambda: Optional[float] = None
        self.last_rank: Optional[int] = None    # ColPivHouseholderQRSolver only

    def _ctx(self) -> Context:
        if self.ctx is None:
            self.ctx = default_context()
        return self.ctx

    def learn(self, data, labels) -> bool:
        """regressors.hpp:345-350 -> Solver::solve (:199-234).  Always returns True, like the reference."""
        ctx = self._ctx()
        A = _dev(data, ctx)
        B = _dev(labels, ctx)
        N, D = A.shape
        M = B.shape[1]
        X = torch.empty((D, M), dtype=torch.float32, device=A.device)
        lam = C.c_float(0)
        reg = self.regulariser.c()
        if D > 256 and not getattr(self.solver, "rank_revealing", False):
            # the factorisation route works on centred rows (include/sd_b200.h, sd_centre_features): on a private copy
            if isinstance(data, torch.Tensor) and A.data_ptr() == data.data_ptr():
                A = A.clone()
            mu = torch.empty(D, dtype=torch.float32, device=A.device)
            _check(ctx.h, _capi.lib().sd_centre_features(ctx.h, None, ptr(A), C.c_int64(A.stride(0)), N, D, N, C.byref(reg), ptr(mu)))
            _check(ctx.h, _capi.lib().sd_learn_centred(ctx.h, None, ptr(A), C.c_int64(A.stride(0)), ptr(B), C.c_int64(B.stride(0)), N, D, M,
                                                       C.byref(reg), N, 0, ptr(mu), ptr(X), None, C.byref(lam)))
            self.x = X
            self.last_lambda = lam.value
            return True
        if getattr(self.solver, "rank_revealing", False):
            rank = C.c_int(-1)
            rc = _capi.lib().sd_learn_rank_revealing(ctx.h, ptr(A), C.c_int64(A.stride(0)), ptr(B), C.c_int64(B.stride(0)),
                                                     N, D, M, C.byref(reg), ptr(X), C.byref(lam), C.byref(rank))
            self.last_rank = rank.value
            if 0 <= rank.value < D:
                print("The regularised AtA is not invertible. We continued learning, but Eigen may return garbage (their docu is not "
                      f"very specific). (The rank is {rank.value}, full rank would be {D}). Increase lambda.")
                if rc == 5:                       # SD_ERR_NUMERIC: the factorisation of the singular matrix stopped; the reference returns garbage here
                    X.fill_(float("nan"))
                    rc = 0
            _check(ctx.h, rc)
        else:
            _check(ctx.h, _capi.lib().sd_learn(ctx.h, ptr(A), C.c_int64(A.stride(0)), ptr(B), C.c_int64(B.stride(0)),
                                               N, D, M, C.byref(reg), ptr(X), C.byref(lam)))
        self.x = X
        self.last_lambda = lam.value
        return True

    def predict(self, values) -> torch.Tensor:
        """regressors.hpp:377-381: values * x."""
        ctx = self._ctx()
        V = _dev(values, ctx)
        if V.dim() == 1:
            V = V.reshape(1, -1)
        N, D = V.shape
        M = self.x.shape[1]
        out = torch.empty((N, M), dtype=torch.float32, device=V.device)
        _check(ctx.h, _capi.lib().sd_predict(ctx.h, ptr(V), C.c_int64(V.stride(0)), N, D, ptr(self.x), M, ptr(out), C.c_int64(M)))
        return out

    def test(self, data, labels) -> float:
        """regressors.hpp:361-369: normalised least-squares residual."""
        ctx = self._ctx()
        V = _dev(data, ctx)
        Lb = _dev(labels, ctx)
        res = C.c_double(0)
        _check(ctx.h, _capi.lib().sd_test_residual(ctx.h, ptr(V), C.c_int64(V.stride(0)), ptr(Lb), C.c_int64(Lb.stride(0)),
                                                   V.shape[0], V.shape[1], ptr(self.x), self.x.shape[1], C.byref(res)))
        return res.value


# ------------------------------------------------------------------------------------------------
# normalisation strategies
# ------------------------------------------------------------------------------------------------
class NoNormalisation:
    """superviseddescent.hpp:60-74."""

    def c(self, num_landmarks: int) -> NormalisationC:
        return NormalisationC(0, 0, 0, (C.c_int32 * 4)(), (C.c_int32 * 4)())


class InterEyeDistanceNormalisation:
    """rcr::InterEyeDistanceNormalisation (model.hpp:84-116): normaliser = 1 / IED(params)."""

    def __init__(self, model_landmarks_list: Sequence[str], right_eye_identifiers: Sequence[str],
                 left_eye_identifiers: Sequence[str]):
        self.model_landmarks_list = [str(s) for s in model_landmarks_list]
        self.right_eye_identifiers = [str(s) for s in right_eye_identifiers]
        self.left_eye_identifiers = [str(s) for s in left_eye_identifiers]

    def _idx(self, ids, which):
        out = []
        for s in ids:
            if s not in self.model_landmarks_list:
                # helpers.hpp:144,153 throw std::runtime_error with this text
                raise RuntimeError(f"one of given {which}EyeIdentifiers ids not present in lms")
            out.append(self.model_landmarks_list.index(s))
        return out

    def c(self, num_landmarks: int = 0) -> NormalisationC:
        r = self._idx(self.right_eye_identifiers, "right")
        l = self._idx(self.left_eye_identifiers, "left")
        if not (1 <= len(r) <= 4 and 1 <= len(l) <= 4):
            raise ValueError("1..4 eye identifiers per eye are supported")
        return NormalisationC(1, len(r), len(l), (C.c_int32 * 4)(*(r + [0] * (4 - len(r)))), (C.c_int32 * 4)(*(l + [0] * (4 - len(l)))))


# ------------------------------------------------------------------------------------------------
# rcr::HogTransform (adaptive_vlhog.hpp:70-195), batched
# ------------------------------------------------------------------------------------------------
class FixedHogTransform:
    """The non-adaptive projection functor of the reference's hello-world (examples/landmark_detection.cpp:127-272):
    HogTransform(images, vlhog_variant, num_cells, cell_size, num_bins) -- a fixed patch of half-size
    num_cells * (cell_size / 2) around every landmark, no resize, no bias column.  Batched like HogTransform."""

    def __init__(self, images, vlhog_variant: int, num_cells: int, cell_size: int, num_bins: int, ctx: Optional["Context"] = None):
        self.ctx = ctx or default_context()
        imgs = images if isinstance(images, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(images))
        if imgs.dim() == 2:
            imgs = imgs.unsqueeze(0)
        if imgs.dtype == torch.uint8 and imgs.dim() == 4 and imgs.shape[3] == 3:
            imgs = bgr2gray(imgs, self.ctx)                      # :201-206
        if imgs.dtype != torch.uint8 or imgs.dim() != 3:
            raise ValueError("images must be (count, H, W) uint8 or (count, H, W, 3) uint8")
        self.images = imgs.to(f"cuda:{self.ctx.device}").contiguous()
        self.param = HoGParam(int(vlhog_variant), num_cells, cell_size, num_bins, 0.0)

    def feature_length(self, num_landmarks: int) -> int:
        return _capi.lib().sd_hog_feature_length(num_landmarks, C.byref(self.param)) - 1     # no bias column

    def __call__(self, parameters, regressor_level: int = 0, training_index=None) -> torch.Tensor:
        ctx = self.ctx
        x = _dev(parameters, ctx)
        single = x.dim() == 1
        if single:
            x = x.unsqueeze(0)
        n, L = x.shape[0], x.shape[1] // 2
        idx = None
        if training_index is not None:
            idx = torch.as_tensor(np.atleast_1d(np.asarray(training_index)), dtype=torch.int32).to(x.device)
        D = self.feature_length(L) + 1
        out = torch.empty((n, D), dtype=torch.float32, device=x.device)
        self.into(x, out, idx)
        feats = out[:, :D - 1]
        return feats[0] if single else feats

    def into(self, parameters: torch.Tensor, out: torch.Tensor, image_index: Optional[torch.Tensor] = None):
        """Writes the feature rows into out[:, :D]; column D receives the kernel's bias 1 (not part of this functor's
        output: callers overwrite or ignore it)."""
        ctx = self.ctx
        n, L = parameters.shape[0], parameters.shape[1] // 2
        h, w = self.images.shape[1], self.images.shape[2]
        ib = ImageBatchC(C.c_void_p(self.images.data_ptr()), w, h, self.images.stride(1), self.images.stride(0), self.images.shape[0])
        _check(ctx.h, _capi.lib().sd_hog_batch(ctx.h, C.byref(ib), ptr(image_index) if image_index is not None else C.c_void_p(0),
                                               ptr(parameters), C.c_int64(parameters.stride(0)), n, L, None, C.byref(self.param),
                                               ptr(out), C.c_int64(out.stride(0))))


def bgr2gray(images, ctx: Optional["Context"] = None) -> torch.Tensor:
    """cv::cvtColor(BGR2GRAY) on the device (adaptive_vlhog.hpp:114-120): (count, H, W, 3) uint8 -> (count, H, W) uint8.
    Host arrays are uploaded first; the result stays in HBM."""
    ctx = ctx or default_context()
    t = images if isinstance(images, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(images))
    if t.dim() == 3:
        t = t.unsqueeze(0)
    if t.dtype != torch.uint8 or t.dim() != 4 or t.shape[3] != 3:
        raise ValueError("images must be (count, H, W, 3) uint8 (interleaved B, G, R)")
    t = t.to(f"cuda:{ctx.device}").contiguous()
    n, h, w, _ = t.shape
    out = torch.empty((n, h, w), dtype=torch.uint8, device=t.device)
    _check(ctx.h, _capi.lib().sd_bgr2gray(ctx.h, ptr(t), w, h, C.c_int64(t.stride(1)), C.c_int64(t.stride(0)), n,
                                          ptr(out), C.c_int64(out.stride(1)), C.c_int64(out.stride(0))))
    return out


_FRAME_DTYPE = np.dtype([("w", "<i4"), ("h", "<i4"), ("s", "<i4"), ("r", "<i4"), ("o", "<i8")])   # sd_frame


def _gray_frame(im, ctx: "Context"):
    """One frame as a 2-D uint8 array / tensor; (H, W, 3) B,G,R frames are converted on the device (sd_bgr2gray)."""
    t = im if isinstance(im, torch.Tensor) else np.ascontiguousarray(im, dtype=np.uint8)
    if t.ndim == 3 and t.shape[2] == 3:
        t = bgr2gray(t[None], ctx)[0]
    if t.ndim != 2 or t.dtype not in (np.uint8, torch.uint8):
        raise ValueError("every frame must be (H, W) uint8 or (H, W, 3) uint8")
    return t


def pack_frames(images, ctx: Optional["Context"] = None):
    """Frames of any sizes ((H, W) uint8 or (H, W, 3) uint8 B,G,R; host arrays or tensors) packed back to back on the device,
    each row padded with zeros to a multiple of 16 bytes.  Returns (data, table): the uint8 device buffer and one sd_frame
    record per frame (as a uint8 device tensor), the d_data / d_frames pair of an sd_image_batch."""
    ctx = ctx or default_context()
    dev = f"cuda:{ctx.device}"
    grays = [_gray_frame(im, ctx) for im in images]
    recs, off = [], 0
    for g in grays:
        h, w = g.shape
        stride = (w + 15) // 16 * 16
        recs.append((w, h, stride, 0, off))
        off += h * stride
    data = torch.zeros(max(off, 1), dtype=torch.uint8, device=dev)
    for g, (w, h, stride, _, o) in zip(grays, recs):
        src = g if isinstance(g, torch.Tensor) else torch.from_numpy(g)
        data[o:o + h * stride].view(h, stride)[:, :w].copy_(src)
    table = np.array(recs, dtype=_FRAME_DTYPE)
    return data, torch.from_numpy(table.view(np.uint8).copy()).to(dev)


class HogTransform:
    """Projection functor h.  images: (count, H, W) uint8 (8UC1) or (count, H, W, 3) uint8 (8UC3, B G R: converted
    once on the device as adaptive_vlhog.hpp:114-120 does per call), on host or device.

    __call__(parameters, regressor_level, training_index) keeps the reference's meaning
    (adaptive_vlhog.hpp:109) but takes ALL rows at once: parameters is (N, 2L) and training_index an
    optional (N,) int array (default: row i uses image i, as train()/test() do).  A single (2L,) row
    with an int training_index is accepted too (predict()'s call shape, superviseddescent.hpp:332).
    """

    def __init__(self, images, hog_params: Sequence[HoGParam], model_landmarks_list: Sequence[str],
                 right_eye_identifiers: Sequence[str], left_eye_identifiers: Sequence[str], ctx: Optional[Context] = None):
        self.ctx = ctx or default_context()
        self.frames = None
        if isinstance(images, (list, tuple)) and len({np.asarray(im).shape for im in images}) > 1:
            # frames of different sizes (the reference takes a std::vector<cv::Mat>)
            self.images, self.frames = pack_frames(images, self.ctx)
            self.frame_count = len(images)
        else:
            if isinstance(images, (list, tuple)):
                images = np.stack([np.asarray(im) for im in images])
            imgs = images if isinstance(images, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(images))
            if imgs.dim() == 2:
                imgs = imgs.unsqueeze(0)
            if imgs.dtype == torch.uint8 and imgs.dim() == 4 and imgs.shape[3] == 3:
                imgs = bgr2gray(imgs, self.ctx)
            if imgs.dtype != torch.uint8 or imgs.dim() != 3:
                raise ValueError("images must be (count, H, W) uint8, (count, H, W, 3) uint8, or a list of such frames of any sizes")
            self.images = imgs.to(f"cuda:{self.ctx.device}").contiguous()
        self.hog_params = list(hog_params)
        self.norm = InterEyeDistanceNormalisation(model_landmarks_list, right_eye_identifiers, left_eye_identifiers)
        self.num_landmarks = len(self.norm.model_landmarks_list)

    def batch(self) -> ImageBatchC:
        if self.frames is not None:
            return ImageBatchC(C.c_void_p(self.images.data_ptr()), 0, 0, 0, 0, self.frame_count, None, None, C.c_void_p(self.frames.data_ptr()))
        n, h, w = self.images.shape
        return ImageBatchC(C.c_void_p(self.images.data_ptr()), w, h, self.images.stride(1), self.images.stride(0), n)

    def feature_length(self, level: int) -> int:
        return _capi.lib().sd_hog_feature_length(self.num_landmarks, C.byref(self.hog_params[level]))

    def into(self, parameters: torch.Tensor, level: int, out: torch.Tensor, image_index: Optional[torch.Tensor] = None):
        """Writes the feature rows into out[:, :D] (out may be wider: extended [A | b] operand)."""
        ctx = self.ctx
        n = parameters.shape[0]
        eyes = self.norm.c()
        ib = self.batch()
        idx_ptr = ptr(image_index) if image_index is not None else C.c_void_p(0)
        _check(ctx.h, _capi.lib().sd_hog_batch(ctx.h, C.byref(ib), idx_ptr, ptr(parameters), C.c_int64(parameters.stride(0)),
                                               n, self.num_landmarks, C.byref(eyes), C.byref(self.hog_params[level]),
                                               ptr(out), C.c_int64(out.stride(0))))

    def __call__(self, parameters, regressor_level: int, training_index=None) -> torch.Tensor:
        ctx = self.ctx
        x = _dev(parameters, ctx)
        single = x.dim() == 1
        if single:
            x = x.reshape(1, -1)
        idx = None
        if training_index is not None:
            if np.isscalar(training_index):
                training_index = [int(training_index)] * x.shape[0]
            idx = _dev(np.asarray(training_index, dtype=np.int32), ctx, dtype=torch.int32)
        elif single:
            idx = torch.zeros(1, dtype=torch.int32, device=x.device)
        D = self.feature_length(regressor_level)
        out = torch.empty((x.shape[0], D), dtype=torch.float32, device=x.device)
        self.into(x, regressor_level, out, idx)
        return out[0] if single else out

    def debug(self, parameters, level: int, training_index=None):
        """Integer parity taps: (geometry [N,L,3] = cx,cy,half ; patches [N,L,fs,fs] u8 ; bins [N,L,fs,fs] i8)."""
        ctx = self.ctx
        x = _dev(parameters, ctx)
        n = x.shape[0]
        p = self.hog_params[level]
        fs = p.num_cells * p.cell_size
        L = self.num_landmarks
        geo = torch.empty((n, L, 3), dtype=torch.int32, device=x.device)
        patches = torch.empty((n, L, fs, fs), dtype=torch.uint8, device=x.device)
        bins = torch.empty((n, L, fs, fs), dtype=torch.int8, device=x.device)
        idx = None
        if training_index is not None:
            idx = _dev(np.asarray(training_index, dtype=np.int32), ctx, dtype=torch.int32)
        eyes = self.norm.c()
        ib = self.batch()
        _check(ctx.h, _capi.lib().sd_hog_debug(ctx.h, C.byref(ib), ptr(idx), ptr(x), C.c_int64(x.stride(0)), n, L,
                                               C.byref(eyes), C.byref(p), ptr(geo), ptr(patches), ptr(bins)))
        return geo, patches, bins


# ------------------------------------------------------------------------------------------------
# superviseddescent.hpp: the cascade
# ------------------------------------------------------------------------------------------------
class SupervisedDescentOptimiser:
    """superviseddescent::SupervisedDescentOptimiser<LinearRegressor, Normalisation> (superviseddescent.hpp:85-361).

    projection: either a HogTransform (stays on the device) or any callable
    h(x_row: np.ndarray, regressor_level: int, sample_index: int) -> row / float, evaluated on the host
    exactly as the reference evaluates user functors (superviseddescent.hpp:178-189).
    """

    def __init__(self, regressors: List[LinearRegressor], normalisation=None, ctx: Optional[Context] = None):
        self.regressors = list(regressors)
        self.normalisation_strategy = normalisation or NoNormalisation()
        self.ctx = ctx

    def _ctx(self) -> Context:
        if self.ctx is None:
            self.ctx = default_context()
        for r in self.regressors:
            if r.ctx is None:
                r.ctx = self.ctx
        return self.ctx

    # -- projection of all rows into an (N, ld) buffer with `extra` spare columns on the right
    def _project(self, h, x: torch.Tensor, level: int, extra: int) -> (torch.Tensor, int):
        ctx = self._ctx()
        n = x.shape[0]
        if isinstance(h, HogTransform):
            D = h.feature_length(level)
            ld = (D + extra + 3) // 4 * 4
            buf = torch.empty((n, ld), dtype=torch.float32, device=x.device)
            h.into(x, level, buf)
            return buf, D
        if isinstance(h, FixedHogTransform):
            D = h.feature_length(x.shape[1] // 2)
            ld = (D + max(extra, 1) + 3) // 4 * 4                 # the kernel's bias lands in the first spare column
            buf = torch.empty((n, ld), dtype=torch.float32, device=x.device)
            h.into(x, buf)
            return buf, D
        xs = x.cpu().numpy()
        rows = [np.atleast_1d(np.asarray(h(xs[i].copy(), level, i), dtype=np.float32)).ravel() for i in range(n)]
        D = rows[0].size
        ld = (D + extra + 3) // 4 * 4
        host = np.zeros((n, ld), dtype=np.float32)
        host[:, :D] = np.stack(rows)
        return _dev(host, ctx), D

    def train(self, parameters, initialisations, templates, projection, on_training_epoch_callback=None, group=None, comm=None,
              distributed_solve=None):
        """superviseddescent.hpp:165-219.  Multi-GPU: pass `comm` (a parallel.Communicator) or a torch.distributed `group`
        (a communicator is then made from it) -- each rank passes its own shard of rows; per level the C ABI does ONE exchange of
        [AtA | Atb] and the solve (SURVEY 8e).  distributed_solve: None = by size (shared CG below parallel.DIST_SOLVE_MIN_D features,
        the distributed factorisation from there), True = reduce-scatter +
        distributed blocked Cholesky, False = all-reduce + replicated solve, "cg" = all-reduce + conjugate gradients shared by the
        ranks."""
        from . import parallel
        ctx = self._ctx()
        lib = _capi.lib()
        x_gt = _dev(parameters, ctx)
        cur = _dev(initialisations, ctx).clone()
        n, P = cur.shape
        tmpl = _dev(templates, ctx) if templates is not None and np.size(templates) > 0 else None
        own_comm = False
        if comm is None and group is not None:
            comm, own_comm = parallel.Communicator(ctx, group), True
        distributed = comm is not None and comm.size > 1
        n_global = comm.sum_int(n) if distributed else n
        for level, reg in enumerate(self.regressors):
            norm = self.normalisation_strategy.c(P // 2)
            A, D = self._project(projection, cur, level, extra=P)             # 1) features (:173-189)
            if tmpl is not None:                                             #    observed = features - templates (:191-197)
                _check(ctx.h, lib.sd_subtract_templates(ctx.h, ptr(A), C.c_int64(A.stride(0)), ptr(tmpl), C.c_int64(tmpl.stride(0)), n, D))
            Bv = A[:, D:D + P]                                               # 2) b = (x - x_gt) .* norm(x)  (:199-205)
            _check(ctx.h, lib.sd_cascade_targets(ctx.h, ptr(cur), ptr(x_gt), n, P, C.byref(norm), ptr(Bv), C.c_int64(A.stride(0))))
            X = torch.empty((D, P), dtype=torch.float32, device=cur.device)  # 3) learn (:207), on centred rows (sd_centre_features)
            Xc = torch.empty((D, P), dtype=torch.float32, device=cur.device)
            mu = torch.empty(D, dtype=torch.float32, device=cur.device)
            lam = C.c_float(0)
            rc_ = reg.regulariser.c()
            ds = 0
            if distributed:
                if distributed_solve is None:
                    ds = 1 if D >= parallel.DIST_SOLVE_MIN_D else 2     # big systems: distributed factorisation; else shared CG
                else:
                    ds = 2 if distributed_solve == "cg" else int(bool(distributed_solve))
            ch = comm.h if distributed else None
            _check(ctx.h, lib.sd_centre_features(ctx.h, ch, ptr(A), C.c_int64(A.stride(0)), n, D, n_global, C.byref(rc_), ptr(mu)))
            _check(ctx.h, lib.sd_learn_centred(ctx.h, ch, ptr(A), C.c_int64(A.stride(0)), ptr(Bv), C.c_int64(A.stride(0)), n, D, P,
                                               C.byref(rc_), n_global, int(ds), ptr(mu), ptr(X), ptr(Xc), C.byref(lam)))
            reg.x, reg.last_lambda = X, lam.value                            #    X: the model (for uncentred features)
            nxt = torch.empty_like(cur)                                      # 4) x <- x - (A X) .* 1/norm(x) (:209-215); A is centred now: Xc
            _check(ctx.h, lib.sd_cascade_update(ctx.h, ptr(A), C.c_int64(A.stride(0)), n, D, ptr(Xc), P, ptr(cur), C.byref(norm), ptr(nxt)))
            cur = nxt
            del A, Bv
            if on_training_epoch_callback is not None:                       # 5) callback (:217)
                on_training_epoch_callback(comm.allgather_rows(cur) if distributed else cur)
        ctx.sync()                                                           # surfaces flags raised by the projection kernels
        if own_comm:
            comm.close()
        return cur

    def test(self, initialisations, templates, projection, on_regressor_iteration_callback=None):
        """superviseddescent.hpp:262-306."""
        ctx = self._ctx()
        lib = _capi.lib()
        cur = _dev(initialisations, ctx).clone()
        if cur.dim() == 1:
            cur = cur.reshape(1, -1)
        n, P = cur.shape
        tmpl = _dev(templates, ctx) if templates is not None and np.size(templates) > 0 else None
        for level, reg in enumerate(self.regressors):
            norm = self.normalisation_strategy.c(P // 2)
            A, D = self._project(projection, cur, level, extra=0)
            if tmpl is not None:
                _check(ctx.h, lib.sd_subtract_templates(ctx.h, ptr(A), C.c_int64(A.stride(0)), ptr(tmpl), C.c_int64(tmpl.stride(0)), n, D))
            nxt = torch.empty_like(cur)
            _check(ctx.h, lib.sd_cascade_update(ctx.h, ptr(A), C.c_int64(A.stride(0)), n, D, ptr(reg.x), P, ptr(cur), C.byref(norm), ptr(nxt)))
            cur = nxt
            if on_regressor_iteration_callback is not None:
                on_regressor_iteration_callback(cur)
        return cur

    def predict(self, initialisations, templates, projection):
        """superviseddescent.hpp:323-344 (same arithmetic as test(), no callback)."""
        return self.test(initialisations, templates, projection)


# ------------------------------------------------------------------------------------------------
# rcr/model.hpp
# ------------------------------------------------------------------------------------------------
def align_mean(mean, facebox, scaling_x=1.0, scaling_y=1.0, translation_x=0.0, translation_y=0.0) -> np.ndarray:
    """rcr::align_mean (model.hpp:64-76); facebox = (x, y, width, height)."""
    mean = np.ascontiguousarray(mean, dtype=np.float32).ravel()
    out = np.empty_like(mean)
    rc = _capi.lib().sd_align_mean(mean.ctypes.data_as(C.c_void_p), mean.size // 2, int(facebox[0]), int(facebox[1]),
                                   int(facebox[2]), int(facebox[3]), C.c_float(scaling_x), C.c_float(scaling_y),
                                   C.c_float(translation_x), C.c_float(translation_y), out.ctypes.data_as(C.c_void_p))
    if rc:
        raise SdError(rc, "sd_align_mean")
    return out


def perturb(facebox, translation_x: float, translation_y: float, scaling: float = 1.0):
    """perturb() of apps/rcr/rcr-train.cpp:130-146: (x, y, w, h) -> perturbed (x, y, w, h)."""
    out = (C.c_int32 * 4)()
    rc = _capi.lib().sd_perturb_box(int(facebox[0]), int(facebox[1]), int(facebox[2]), int(facebox[3]), C.c_float(translation_x),
                                    C.c_float(translation_y), C.c_float(scaling), out)
    if rc != 0:
        raise SdError(rc, "sd_perturb_box")
    return tuple(int(v) for v in out)


def calculate_normalised_landmark_errors(predictions, groundtruth, model_landmarks: Sequence[str], right_eye_identifiers: Sequence[str],
                                         left_eye_identifiers: Sequence[str], ctx: Optional[Context] = None) -> torch.Tensor:
    """calculate_normalised_landmark_errors() of apps/rcr/rcr-train.cpp:200-212: (N, L) per-landmark L2 errors divided by
    the inter-eye distance of the prediction; the mean over everything is the figure rcr-train prints (:520-524)."""
    ctx = ctx or default_context()
    p = _dev(predictions, ctx)
    g = _dev(groundtruth, ctx)
    n, L = p.shape[0], p.shape[1] // 2
    eyes = InterEyeDistanceNormalisation(model_landmarks, right_eye_identifiers, left_eye_identifiers).c(L)
    out = torch.empty((n, L), dtype=torch.float32, device=p.device)
    _check(ctx.h, _capi.lib().sd_normalised_landmark_errors(ctx.h, ptr(p), C.c_int64(p.stride(0)), ptr(g), C.c_int64(g.stride(0)), n, L,
                                                            C.byref(eyes), ptr(out), C.c_int64(out.stride(0))))
    return out


_HOST_FRAME_DTYPE = np.dtype([("p", "<u8"), ("w", "<i4"), ("h", "<i4"), ("s", "<i4"), ("channels", "<i4")])   # sd_host_frame


def _host_frame_table(frames):
    """sd_host_frame records of host frames read in place: an (n, H, W) or (n, H, W, 3) uint8 array / CPU tensor, or a list of
    (H, W) / (H, W, 3) ones (3 channels: interleaved B, G, R).  Returns (table, objects that must stay alive during the call)."""
    def plain(f, colour):   # rows of contiguous pixels: in place where they already are
        if isinstance(f, torch.Tensor):
            if f.is_cuda or f.dtype != torch.uint8:
                raise ValueError("host frames must be uint8 CPU tensors or arrays")
            return f if f.stride(-1) == 1 and (not colour or f.stride(-2) == 3) else f.contiguous()
        ok = f.dtype == np.uint8 and f.strides[-1] == 1 and (not colour or f.strides[-2] == 3)
        return f if ok else np.ascontiguousarray(f, dtype=np.uint8)

    def geometry(f, colour):   # base address, (H, W), row pitch in bytes
        r = -3 if colour else -2
        if isinstance(f, torch.Tensor):
            return f.data_ptr(), (f.shape[r], f.shape[r + 1]), f.stride(r)
        return f.ctypes.data, (f.shape[r], f.shape[r + 1]), f.strides[r]

    if isinstance(frames, (np.ndarray, torch.Tensor)):            # one batch: records computed, not looped over
        colour = frames.ndim == 4
        if frames.ndim not in (3, 4) or (colour and frames.shape[3] != 3):
            raise ValueError("a batch of host frames must be (n, H, W) uint8 or (n, H, W, 3) uint8")
        f = plain(frames, colour)
        base, (h, w), pitch = geometry(f, colour)
        step = f.stride(0) if isinstance(f, torch.Tensor) else f.strides[0]
        table = np.zeros(f.shape[0], dtype=_HOST_FRAME_DTYPE)
        table["p"] = base + step * np.arange(f.shape[0], dtype=np.uint64)
        table["w"], table["h"], table["s"], table["channels"] = w, h, pitch, 3 if colour else 1
        return table, f
    keep = []
    table = np.zeros(len(frames), dtype=_HOST_FRAME_DTYPE)
    for k, f in enumerate(frames):
        f = f if isinstance(f, torch.Tensor) else np.asarray(f)
        colour = f.ndim == 3 and f.shape[2] == 3
        if f.ndim != 2 and not colour:
            raise ValueError("every host frame must be (H, W) uint8 or (H, W, 3) uint8")
        keep.append(plain(f, colour))
        base, (h, w), pitch = geometry(keep[-1], colour)
        table[k] = (base, w, h, pitch, 3 if colour else 1)
    return table, keep


def _on_device(frames) -> bool:
    if isinstance(frames, torch.Tensor):
        return frames.is_cuda
    return isinstance(frames, (list, tuple)) and any(isinstance(f, torch.Tensor) and f.is_cuda for f in frames)


class detection_model:
    """rcr::detection_model (model.hpp:122-183) resident on the GPU."""

    def __init__(self, handle, ctx: Context):
        self._m = handle
        self.ctx = ctx
        lib = _capi.lib()
        self.num_levels = lib.sd_model_num_levels(handle)
        self.num_landmarks = lib.sd_model_num_landmarks(handle)
        self.landmark_ids = [lib.sd_model_landmark_id(handle, i).decode() for i in range(self.num_landmarks)]

    @classmethod
    def from_parts(cls, optimised_model: SupervisedDescentOptimiser, mean, landmark_ids, hog_params, right_eye_ids,
                   left_eye_ids, ctx: Optional[Context] = None) -> "detection_model":
        """detection_model(optimised_model, mean, landmark_ids, hog_params, right_eye_ids, left_eye_ids) (model.hpp:128)."""
        ctx = ctx or default_context()
        S = len(optimised_model.regressors)
        ws = [np.ascontiguousarray(r.x.cpu().numpy(), dtype=np.float32) for r in optimised_model.regressors]
        wp = (C.c_void_p * S)(*[w.ctypes.data_as(C.c_void_p) for w in ws])
        regs = (RegulariserC * S)(*[r.regulariser.c() for r in optimised_model.regressors])
        hps = (HoGParam * S)(*hog_params)
        mean = np.ascontiguousarray(mean, dtype=np.float32).ravel()
        ids = (C.c_char_p * len(landmark_ids))(*[str(s).encode() for s in landmark_ids])
        rid = (C.c_char_p * len(right_eye_ids))(*[str(s).encode() for s in right_eye_ids])
        lid = (C.c_char_p * len(left_eye_ids))(*[str(s).encode() for s in left_eye_ids])
        h = C.c_void_p()
        _check(ctx.h, _capi.lib().sd_model_create(ctx.h, S, len(landmark_ids), wp, regs, hps, mean.ctypes.data_as(C.c_void_p),
                                                  ids, rid, len(right_eye_ids), lid, len(left_eye_ids), C.byref(h)))
        return cls(h, ctx)

    def get_mean(self) -> np.ndarray:
        out = np.empty(2 * self.num_landmarks, dtype=np.float32)
        _capi.lib().sd_model_get_mean(self._m, out.ctypes.data_as(C.c_void_p))
        return out

    def hog_param(self, level: int) -> HoGParam:
        p = HoGParam()
        _capi.lib().sd_model_hog_param(self._m, level, C.byref(p))
        return p

    def weights(self, level: int) -> np.ndarray:
        r, c = C.c_int(0), C.c_int(0)
        _capi.lib().sd_model_get_weights(self._m, level, None, C.byref(r), C.byref(c))
        out = np.empty((r.value, c.value), dtype=np.float32)
        _capi.lib().sd_model_get_weights(self._m, level, out.ctypes.data_as(C.c_void_p), None, None)
        return out

    def detect(self, image, facebox_or_initialisation) -> np.ndarray:
        """detect(image, facebox) / detect(image, initialisation) (model.hpp:132-157): one frame, (H, W) or (H, W, 3) B,G,R
        uint8, returns the 2L row."""
        arg = np.asarray(facebox_or_initialisation)
        if not isinstance(image, torch.Tensor):
            image = np.ascontiguousarray(image, dtype=np.uint8)
        if arg.size == 4:
            return self.detect_batch(image[None], np.asarray(arg, dtype=np.int32)[None])[0]
        return self.detect_faces_from([image], arg.reshape(1, -1), np.zeros(1, dtype=np.int32))[0]

    def detect_batch(self, images: np.ndarray, boxes: np.ndarray) -> np.ndarray:
        """Batched detect(image, facebox) with HOST buffers (copies are part of the call), one face per frame.  Colour frames
        (count, H, W, 3), B,G,R as cv::imread gives them, are converted to gray on the device as they are read
        (model.hpp:134-145 calls cvtColor through HogTransform)."""
        if isinstance(images, torch.Tensor):
            images_np = images.numpy()
        else:
            images_np = np.ascontiguousarray(images, dtype=np.uint8)
        if images_np.ndim == 4:
            n = images_np.shape[0]
            return self.detect_faces(images_np, np.asarray(boxes, dtype=np.int32).reshape(n, 4), np.arange(n, dtype=np.int32))
        n, h, w = images_np.shape
        boxes = np.ascontiguousarray(boxes, dtype=np.int32).reshape(n, 4)
        out = np.empty((n, 2 * self.num_landmarks), dtype=np.float32)
        _check(self.ctx.h, _capi.lib().sd_detect_batch_host(self.ctx.h, self._m, images_np.ctypes.data_as(C.c_void_p), n, w, h,
                                                            images_np.strides[1], boxes.ctypes.data_as(C.c_void_p),
                                                            out.ctypes.data_as(C.c_void_p)))
        return out

    def detect_batch_device(self, images: torch.Tensor, x0: torch.Tensor) -> torch.Tensor:
        """Batched detect(image, initialisation), frames and landmarks already resident in HBM."""
        n, h, w = images.shape
        ib = ImageBatchC(C.c_void_p(images.data_ptr()), w, h, images.stride(1), images.stride(0), n)
        out = torch.empty((n, 2 * self.num_landmarks), dtype=torch.float32, device=images.device)
        _check(self.ctx.h, _capi.lib().sd_detect_batch_device(self.ctx.h, self._m, C.byref(ib), ptr(x0), n, ptr(out)))
        return out

    def align_boxes(self, boxes) -> torch.Tensor:
        """align_mean(mean, box) (model.hpp:64-76) for every (x, y, w, h) row of `boxes`, on the device: (count, 2L) float32,
        bit-identical to align_mean() on the host."""
        b = _dev(np.asarray(boxes, dtype=np.int32).reshape(-1, 4) if not isinstance(boxes, torch.Tensor) else boxes.reshape(-1, 4),
                 self.ctx, dtype=torch.int32)
        out = torch.empty((b.shape[0], 2 * self.num_landmarks), dtype=torch.float32, device=b.device)
        _check(self.ctx.h, _capi.lib().sd_model_align_boxes(self.ctx.h, self._m, ptr(b), b.shape[0], ptr(out), C.c_int64(out.stride(0))))
        return out

    def _device_frames(self, frames):
        """(sd_image_batch, tensors to keep alive) for frames on the device: an (n, H, W) / (n, H, W, 3) uint8 tensor or array,
        or a list of frames of any sizes (packed with pack_frames)."""
        if isinstance(frames, (list, tuple)):
            data, table = pack_frames(frames, self.ctx)
            return ImageBatchC(C.c_void_p(data.data_ptr()), 0, 0, 0, 0, len(frames), None, None, C.c_void_p(table.data_ptr())), (data, table)
        t = frames if isinstance(frames, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(frames, dtype=np.uint8))
        if t.dim() == 2:
            t = t.unsqueeze(0)
        if t.dim() == 4 and t.shape[3] == 3:
            t = bgr2gray(t, self.ctx)
        if t.dtype != torch.uint8 or t.dim() != 3:
            raise ValueError("frames must be (n, H, W) uint8, (n, H, W, 3) uint8 or a list of frames")
        t = t.to(f"cuda:{self.ctx.device}").contiguous()
        n, h, w = t.shape
        return ImageBatchC(C.c_void_p(t.data_ptr()), w, h, t.stride(1), t.stride(0), n), (t,)

    def detect_faces_device(self, frames, frame_index, x0) -> torch.Tensor:
        """detect(image, initialisation) for several faces per frame on the device: face i starts from x0[i] (count, 2L) and
        reads frames[frame_index[i]].  frames: an (n, H, W) uint8 tensor, or a list of frames of any sizes.  An index out of
        range raises SdError with code 1 (SD_ERR_INVALID)."""
        ib, keep = self._device_frames(frames)
        idx = _dev(np.asarray(frame_index, dtype=np.int32).ravel() if not isinstance(frame_index, torch.Tensor) else frame_index.reshape(-1),
                   self.ctx, dtype=torch.int32)
        x = _dev(x0, self.ctx).reshape(-1, 2 * self.num_landmarks)
        if x.shape[0] != idx.shape[0]:
            raise ValueError("one frame index per initialisation")
        out = torch.empty((x.shape[0], 2 * self.num_landmarks), dtype=torch.float32, device=x.device)
        _check(self.ctx.h, _capi.lib().sd_detect_faces_device(self.ctx.h, self._m, C.byref(ib), ptr(idx), ptr(x), x.shape[0], ptr(out)))
        del keep
        return out

    def _frames_and_index(self, frames, frame_index, count: int, what: str):
        """(frames, int32 index, batch?) of a detect_faces / detect_faces_from call; an index out of range raises SdError 1."""
        idx = np.ascontiguousarray(frame_index, dtype=np.int32).ravel()
        if idx.shape[0] != count:
            raise ValueError(f"one frame index per {what}")
        batch = isinstance(frames, (np.ndarray, torch.Tensor))
        if batch and frames.ndim != 3 and frames.ndim != 4:
            raise ValueError("frames must be an (n, H, W) / (n, H, W, 3) array or a list of frames")
        if not batch:
            frames = [f if isinstance(f, (np.ndarray, torch.Tensor)) else np.asarray(f) for f in frames]
        bad = (idx < 0) | (idx >= len(frames))
        if count and bad.any():
            i = int(np.argmax(bad))
            raise SdError(1, f"detect_faces: face {i}: frame index {int(idx[i])} is not in [0, {len(frames)})")
        return frames, idx

    def detect_faces(self, frames, boxes, frame_index) -> np.ndarray:
        """detect(image, facebox) for every face of a batch of frames of any sizes: face i has box boxes[i] = (x, y, w, h) in
        frames[frame_index[i]]; returns (count, 2L).  frames: a list of (H, W) / (H, W, 3) uint8 frames (3 channels: B,G,R),
        or an (n, H, W) / (n, H, W, 3) array.  Host frames, gray or colour, are read in place (each referenced frame is uploaded
        once; pinned torch tensors take the region-of-interest route, which converts colour neighbourhoods to gray as it
        gathers them); frames already on the device take the device route.  A frame index out of range raises SdError with
        code 1 before any work is queued."""
        b = np.ascontiguousarray(boxes, dtype=np.int32).reshape(-1, 4)
        count, P = b.shape[0], 2 * self.num_landmarks
        frames, idx = self._frames_and_index(frames, frame_index, count, "box")
        out = np.empty((count, P), dtype=np.float32)
        if count == 0:
            return out
        if _on_device(frames):
            return self.detect_faces_device(frames, idx, self.align_boxes(b)).cpu().numpy()
        table, keep = _host_frame_table(frames)
        _check(self.ctx.h, _capi.lib().sd_detect_faces_host(self.ctx.h, self._m, table.ctypes.data_as(C.c_void_p), len(table),
                                                            idx.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p), count,
                                                            out.ctypes.data_as(C.c_void_p)))
        del keep
        return out

    def detect_faces_from(self, frames, initialisations, frame_index) -> np.ndarray:
        """detect(image, initialisation) (model.hpp:147-157, e.g. the landmarks of the previous video frame) for every face of a
        batch of frames: face i starts from initialisations[i] (count, 2L) in frames[frame_index[i]]; returns (count, 2L).
        Frames and routes as in detect_faces."""
        P = 2 * self.num_landmarks
        x0 = np.ascontiguousarray(initialisations.cpu().numpy() if isinstance(initialisations, torch.Tensor) else initialisations,
                                  dtype=np.float32).reshape(-1, P)
        count = x0.shape[0]
        frames, idx = self._frames_and_index(frames, frame_index, count, "initialisation")
        out = np.empty((count, P), dtype=np.float32)
        if count == 0:
            return out
        if _on_device(frames):
            return self.detect_faces_device(frames, idx, x0).cpu().numpy()
        table, keep = _host_frame_table(frames)
        _check(self.ctx.h, _capi.lib().sd_detect_faces_host_init(self.ctx.h, self._m, table.ctypes.data_as(C.c_void_p), len(table),
                                                                 idx.ctypes.data_as(C.c_void_p), x0.ctypes.data_as(C.c_void_p),
                                                                 C.c_int64(P), count, out.ctypes.data_as(C.c_void_p)))
        del keep
        return out

    def save(self, filename: str) -> None:
        _check(self.ctx.h, _capi.lib().sd_model_save(self.ctx.h, self._m, filename.encode()))

    def __del__(self):
        try:
            if self._m:
                _capi.lib().sd_model_destroy(self._m)
                self._m = None
        except Exception:
            pass


def load_detection_model(filename: str, ctx: Optional[Context] = None) -> detection_model:
    """rcr::load_detection_model (model.hpp:192-205)."""
    ctx = ctx or default_context()
    h = C.c_void_p()
    _check(ctx.h, _capi.lib().sd_model_load(ctx.h, filename.encode(), C.byref(h)))
    return detection_model(h, ctx)


def save_detection_model(model: detection_model, filename: str) -> None:
    """rcr::save_detection_model (model.hpp:214-219)."""
    model.save(filename)
