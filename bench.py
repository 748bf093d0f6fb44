#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 cascaded-regression engine.

Metric (BASELINE.json): faces/sec, RCR 22-landmark detect with the reference's pre-trained
face_landmarks_model_rcr_22.bin on 640x480 synthetic 8UC1 frames, batched, one face box per frame
(config 3, "configs[2]").  A "step" = one pass of the detect cascade (4 levels: HOG -> feature x weight
GEMM -> IED-scaled update) over one batch of B frames.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl ours|reference] [--dump-outputs DIR]

  value        whole-job faces/s with frames + initial landmarks already resident in HBM
  e2e          the same through the reference-facing call detection_model::detect(image, facebox)
               batched with HOST (pinned) buffers: H2D of the frames and D2H of the landmarks are inside
               the timed region
  roofline     the dominant kernel (HOG, cascade level 0) against measured HBM bandwidth
  cpu_baseline the reference's own hog.c (oracle/_ref) inside the restated HogTransform/predict glue,
               timed on this box's host cores on a bounded sample
  train        (N=1 only, extra) regressor-train seconds of a reduced RCR training config

--impl reference times the CPU path alone (rank 0), same metric/config.

--dump-outputs DIR writes what the last timed step returned (rank 0's share) as DIR/<name>.npy in float32: the landmarks
of the detect workload; the weights of every level and the final landmarks of the train workloads.  The inputs depend on
the arguments only, so two builds run with the same arguments can be compared array for array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
MODEL = os.path.join(ROOT, "tests", "golden", "face_landmarks_model_rcr_22.bin")
W_IMG, H_IMG = 640, 480


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_BYTES = 60 * 10 ** 6      # data of all dumped arrays; leaves room for the .npy headers under 64 MB


def dump_outputs(dirname, arrays):
    """Writes each array as dirname/<name>.npy in float32.  When together they exceed DUMP_BYTES, every array larger than an
    even share of it is cut to a fixed, seeded sample of its rows (in row order, the same rows on every run)."""
    os.makedirs(dirname, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    over = sum(a.nbytes for a in arrays.values()) > DUMP_BYTES
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float32)
        if over and a.nbytes > share:
            keep = max(1, share // (a.nbytes // a.shape[0]))
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(dirname, name + ".npy"), a)


def synth_boxes(count, seed):
    """SURVEY 8d: one square face box per frame, w=h in U{200..280}, fully inside the 640x480 frame."""
    rng = np.random.Generator(np.random.PCG64(seed))
    s = rng.integers(200, 281, size=count)
    x = (rng.random(count) * (W_IMG - s - 40) + 20).astype(np.int64)
    y = (rng.random(count) * (H_IMG - s - 40) + 20).astype(np.int64)
    return np.stack([x, y, s, s], axis=1).astype(np.int32)


def synth_frames_torch(count, seed, device):
    """Low-pass filtered uniform noise (sigma = 3 px) stretched to 0..255, 8UC1, generated on the GPU."""
    import torch
    import torch.nn.functional as F
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    sigma, r = 3.0, 9
    k = torch.exp(-0.5 * (torch.arange(-r, r + 1, device=device, dtype=torch.float32) / sigma) ** 2)
    k = k / k.sum()
    out = torch.empty((count, H_IMG, W_IMG), dtype=torch.uint8, device=device)
    for i0 in range(0, count, 128):
        n = min(128, count - i0)
        x = torch.rand((n, 1, H_IMG + 2 * r, W_IMG + 2 * r), generator=g, device=device)
        x = F.conv2d(x, k.view(1, 1, -1, 1))
        x = F.conv2d(x, k.view(1, 1, 1, -1))
        lo = x.amin(dim=(2, 3), keepdim=True)
        hi = x.amax(dim=(2, 3), keepdim=True)
        out[i0:i0 + n] = ((x - lo) / (hi - lo) * 255.0).round().clamp(0, 255).to(torch.uint8)[:, 0]
    return out


def synth_frames_numpy(count, seed):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import synth
    return synth.smooth_images(count, H_IMG, W_IMG, seed)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


def cpu_detect_rate(n_faces, threads, seed):
    """Reference CPU path: oracle glue + the reference's hog.c when oracle/_ref is built."""
    from oracle import oracle as O
    om = O.Model(MODEL)
    use_ref = O.ref_available()
    frames = synth_frames_numpy(min(n_faces, 64), seed)
    reps = (n_faces + frames.shape[0] - 1) // frames.shape[0]
    frames = np.concatenate([frames] * reps)[:n_faces]
    boxes = synth_boxes(n_faces, seed)
    om.detect_batch(frames[:threads], boxes[:threads], use_ref=use_ref, threads=threads)   # warm-up
    t0 = time.perf_counter()
    om.detect_batch(frames, boxes, use_ref=use_ref, threads=threads)
    dt = time.perf_counter() - t0
    return n_faces / dt, ("reference" if use_ref else "port"), dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_cores()
    if args.workload != "detect":
        # regressor-train seconds of the reference's CPU path: one level on a bounded sample, scaled (see cpu_train_level_seconds)
        cfg = TRAIN_CFGS[args.workload]
        n_cpu = min(cfg["n"], 10000) if cfg["landmarks"] == 22 else 1500
        lvl = cpu_train_level_seconds(n_cpu, cores, cfg)
        S = len(cfg["cell_sizes"])
        value = lvl["total_extrapolated_s"] * S
        sample_txt = (f"ONE level (level 0) on {n_cpu} of the {cfg['n']} samples: HOG {lvl['hog_s']:.2f} s, Gram {lvl['gram_s']:.2f} s, LU+solve {lvl['lu_solve_s']:.2f} s, "
                      f"update {lvl['update_s']:.2f} s, scaled to the full level and x{S} levels (extrapolated); {lvl['kind']}")
        print(json.dumps({"impl": "reference", "metric": "regressor train sec (RCR, all cascade levels)", "value": value, "unit": "s", "n_gpus": args.gpus,
                          "steps": 1, "warmup": 0, "ms_per_step": value * 1e3, "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
                          "data": "synthetic", "config": {"workload": cfg["name"]},
                          "cpu_baseline": {"value": value, "unit": "s", "cores": cores, "kind": "port", "sample": sample_txt},
                          "e2e": {"value": value, "unit": "s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))
        return
    sample = max(cores * 8, 256)
    rates = []
    kind = "port"
    for s in range(args.warmup + args.steps):
        r, kind, dt = cpu_detect_rate(sample, cores, 1234 + s)
        if s >= args.warmup:
            rates.append((sample, dt))
    faces = sum(a for a, _ in rates)
    secs = sum(b for _, b in rates)
    value = faces / secs
    r1, _, _ = cpu_detect_rate(64, 1, 99)
    line = {
        "impl": "reference", "metric": "faces/sec RCR 22-landmark detect", "value": value, "unit": "faces/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / max(len(rates), 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[2]: RCR 22-landmark detect, face_landmarks_model_rcr_22.bin, 640x480 8UC1 synthetic frames, "
                               f"{sample} faces per step on host cores", "frames_per_step": sample},
        "cpu_baseline": {"value": value, "unit": "faces/s", "cores": cores, "kind": kind,
                         "sample": f"{sample} faces/step x {args.steps} steps, one face per thread; single-thread (reference-faithful sequential predict): {r1:.1f} faces/s",
                         "single_thread_value": r1},
        "e2e": {"value": value, "unit": "faces/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# static profile facts about the level-0 HOG kernel: NOT measured in the bench run, quoted from the committed ncu summary
HOG_STATIC_PROFILE = {"source": "profiles/r02_summary.md section 2 (one `ncu --set full` capture of hog_patch_kernel<4,5,11>, 2048 faces)",
                      "dram_bytes_per_face": (170.898432e6 + 52.981504e6) / 2048, "issue_slots_busy_pct": 61.5,
                      "warp_instructions_per_patch": 16166, "shared_wavefronts_pct_of_lsu_path": 76}

TRAIN_CFGS = {
    # SURVEY 8d config 4 / BASELINE configs[3]
    "train": {"name": "configs[3]: RCR training, 10k synthetic 128x128 crops, 22 landmarks, 31-bin HOG (K=9), 5 cascade levels",
              "n": 10000, "size": 128, "landmarks": 22, "num_bins": 9, "cells": 5, "cell_sizes": [11, 10, 8, 6, 6],
              "rel": [1.0, 0.7, 0.4, 0.25, 0.25], "lambda_factor": 1.5, "seed": 2024},
    # SURVEY 8d config 5 / BASELINE configs[4]
    "train5": {"name": "configs[4]: RCR training, 100k synthetic 256x256 crops, 68 landmarks, 31-bin HOG (K=9), 6 cascade levels",
               "n": 100000, "size": 256, "landmarks": 68, "num_bins": 9, "cells": 5, "cell_sizes": [11, 10, 8, 6, 6, 6],
               "rel": [1.0, 0.7, 0.4, 0.25, 0.25, 0.25], "lambda_factor": 1.5, "seed": 2025},
}
TRAIN_CFG = TRAIN_CFGS["train"]
GEN_CHUNK = 256      # synthetic samples are generated in global chunks of this many, seeded by the chunk index


def train_shape_model(cfg, model):
    """(mean, landmark ids, right eye ids, left eye ids) of a training config: the rcr_22 model's for 22 landmarks, the
    reference's 68-point mean (examples/data/mean_ibug_lfpw_68.txt, committed as tests/golden/mean_ibug_lfpw_68.npy) otherwise."""
    if cfg["landmarks"] == 22:
        import ctypes as C
        from superviseddescent_b200 import _capi
        from superviseddescent_b200 import api as sd
        ids = model.landmark_ids
        norm_c = sd.NormalisationC()
        _capi.lib().sd_model_normalisation(model._m, C.byref(norm_c))
        return (model.get_mean(), ids, [ids[norm_c.right_idx[i]] for i in range(norm_c.n_right)],
                [ids[norm_c.left_idx[i]] for i in range(norm_c.n_left)])
    mean = np.load(os.path.join(ROOT, "tests", "golden", "mean_ibug_lfpw_68.npy")).astype(np.float32).reshape(-1)
    return mean, [str(i) for i in range(1, 69)], ["37", "40"], ["43", "46"]


def synth_train_images(cfg, b, e, dev):
    """Crops [b, e) of the GLOBAL synthetic training set (low-pass filtered noise, 8UC1): every chunk of GEN_CHUNK samples has
    its own seed, so the set is the same whatever the number of ranks it is sharded over."""
    import torch
    import torch.nn.functional as F
    size = cfg["size"]
    sigma, r = 3.0, 9
    k = torch.exp(-0.5 * (torch.arange(-r, r + 1, device=dev, dtype=torch.float32) / sigma) ** 2)
    k = k / k.sum()
    imgs = torch.empty((e - b, size, size), dtype=torch.uint8, device=dev)
    g = torch.Generator(device=dev)
    for c in range(b // GEN_CHUNK, (e + GEN_CHUNK - 1) // GEN_CHUNK):
        g.manual_seed(cfg["seed"] * 1000003 + c)
        x = torch.rand((GEN_CHUNK, 1, size + 2 * r, size + 2 * r), generator=g, device=dev)
        x = F.conv2d(F.conv2d(x, k.view(1, 1, -1, 1)), k.view(1, 1, 1, -1))
        lo, hi = x.amin(dim=(2, 3), keepdim=True), x.amax(dim=(2, 3), keepdim=True)
        x = ((x - lo) / (hi - lo) * 255.0).round().clamp(0, 255).to(torch.uint8)[:, 0]
        g0, g1 = max(b, c * GEN_CHUNK), min(e, (c + 1) * GEN_CHUNK)
        imgs[g0 - b:g1 - b] = x[g0 - c * GEN_CHUNK:g1 - c * GEN_CHUNK]
    return imgs


def synth_train_landmarks(sd, mean, cfg, b, e):
    """SURVEY 8d: box = crop shrunk by 10 %, ground truth = mean shape in a box jittered N(0, 0.04) in translation and
    N(1, 0.04) in scale (rcr-train.cpp:387-395), x0 = mean in the unjittered box; rows [b, e) of the global set."""
    size = cfg["size"]
    rng = np.random.Generator(np.random.PCG64(cfg["seed"]))
    jit = rng.normal(0.0, 0.04, size=(cfg["n"], 4))[b:e]
    m = int(round(size * 0.05))
    box = (m, m, size - 2 * m, size - 2 * m)
    x0 = np.tile(sd.align_mean(mean, box), (e - b, 1)).astype(np.float32)
    x_gt = np.stack([sd.align_mean(mean, box, 1.0 + j[0], 1.0 + j[1], j[2], j[3]) for j in jit]).astype(np.float32)
    return x0, x_gt


def syrk_executed_flops(n, D, M, passes=3):
    """MMA flops the Gram kernel executes: every 128 x 256 tile that touches the upper triangle of [AtA | Atb], three TF32 passes."""
    TI, TJ = (D + 127) // 128, (D + M + 255) // 256
    tiles = sum(1 for ti in range(TI) for tj in range(TJ) if tj * 256 + 255 >= ti * 128)
    return passes * 2.0 * n * tiles * 128 * 256


def run_train(sd, ctx, model, world, rank, dev, barrier, max_over_ranks, comm, cfg=None, steps=1, warmup=1, e2e=False, distributed_solve=None,
              solver="cholesky", outputs=None):
    """Regressor-train seconds (all S levels: HOG + targets + Gram + exchange + solve + update), strong scaling: the SAME global
    training set for every number of ranks (samples are generated by global index).  A dict passed as outputs receives what
    the last timed step returned: the weights of every level and this rank's final landmarks."""
    import torch
    from superviseddescent_b200 import parallel
    cfg = cfg or TRAIN_CFG
    ctx.set_solver(solver)
    mean, ids, right, left = train_shape_model(cfg, model)
    L = cfg["landmarks"]
    b, e = parallel.shard_range(cfg["n"], world, rank)
    imgs = synth_train_images(cfg, b, e, dev)
    x0, x_gt = synth_train_landmarks(sd, mean, cfg, b, e)
    hps = [sd.HoGParam(1, cfg["cells"], cs, cfg["num_bins"], rel) for cs, rel in zip(cfg["cell_sizes"], cfg["rel"])]
    ht = sd.HogTransform(imgs, hps, ids, right, left, ctx)
    D = ht.feature_length(0)
    S = len(hps)
    ds = ((True if D >= parallel.DIST_SOLVE_MIN_D else "cg") if distributed_solve is None else distributed_solve) if world > 1 else None
    gram_ms = []

    def one_run(levels=None):
        use = hps if levels is None else hps[:levels]
        regs = [sd.LinearRegressor(sd.Regulariser(sd.RegularisationType.MatrixNorm, cfg["lambda_factor"], False), ctx) for _ in use]
        sdo = sd.SupervisedDescentOptimiser(regs, sd.InterEyeDistanceNormalisation(ids, right, left), ctx)
        xf = sdo.train(x_gt, x0, None, ht, None, comm=comm, distributed_solve=ds)
        return sdo, xf

    for _ in range(max(warmup, 1)):
        one_run(1 if cfg["n"] > 20000 else None)     # warm-up (workspaces, tensor maps, NCCL channels); one level of the big config
    barrier()
    l0 = ctx.launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        sdo, xf = one_run()
    e1.record()
    barrier()
    secs = max_over_ranks(e0.elapsed_time(e1)) * 1e-3 / steps
    launches = int(ctx.launches() - l0) // steps
    if outputs is not None:
        outputs.update({f"weights_level{i}": r.x.cpu().numpy() for i, r in enumerate(sdo.regressors)})
        outputs["landmarks"] = xf.cpu().numpy()
    solver_ms = ctx.solver_timings()
    g = torch.from_numpy(x_gt).to(dev)
    num = torch.stack([torch.sum((torch.from_numpy(x0).to(dev) - g) ** 2), torch.sum((xf - g) ** 2), torch.sum(g ** 2)]).double()
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(num)
    res0, res1 = float(torch.sqrt(num[0] / num[2])), float(torch.sqrt(num[1] / num[2]))
    # the trained model's fingerprint: identical data for every N, so these agree across N up to summation order
    checksum = [float(r.x.double().abs().sum()) for r in sdo.regressors]
    out = {"metric": "regressor train sec (RCR, all cascade levels)", "value": secs, "unit": "s", "higher_is_better": False, "scaling": "strong",
           "n_gpus": world, "steps": steps, "warmup": max(warmup, 1), "ms_per_step": secs * 1e3, "dtype": "f32", "data": "synthetic", "vs_baseline": None,
           "config": {"workload": cfg["name"], "samples_global": cfg["n"], "samples_this_rank": e - b, "feature_dim": D, "levels": S,
                      "landmarks": L, "l2": f"per-level operands ({(e - b) * D * 4 / 1e9:.2f} GB of features, {D * (D + 2 * L) * 4 / 1e9:.2f} GB Gram) exceed the 126 MB L2",
                      "parallelism": (f"samples sharded over {world} GPU(s); per level one exchange of the upper row bands of [AtA|Atb] "
                                      f"({parallel.band_offsets(D, (D + 2 * L + 3) // 4 * 4)[-1] * 4 / 1e9:.2f} of {D * (D + 2 * L) * 4 / 1e9:.2f} GB): "
                                      + ("all-reduce + conjugate gradients shared by the ranks (one all-reduce of 2L x D floats per iteration)" if ds == "cg"
                                         else "reduce to the block-row-cyclic owners + distributed blocked Cholesky (panel broadcast)" if ds
                                         else "all-reduce + replicated solve" if world > 1 else "single GPU")),
                      "solver": ("conjugate gradients (tcgen05 3xTF32 products)" if (ds == "cg" or solver == "cg") else "blocked Cholesky"),
                      "solver_iterations_last_level": ctx.solver_iterations()},
           "gpu_launches": launches,
           "train_residual": {"before": res0, "after": res1},
           "weights_checksum_abs_sum_per_level": checksum,
           "last_level_solver_ms": solver_ms}
    # roofline of the dominant kernel: the tensor-core Gram SYRK of the last level, timed by CUDA events inside the library on
    # the launching stream ("At * A" of the reference's VerbosePartialPivLUSolver)
    n_loc = e - b
    alg = n_loc * D * (D + 1.0) + 2.0 * n_loc * D * 2 * L
    t = solver_ms["At * A"] * 1e-3
    if t > 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("bf16_tflops_sustained", 0) or 0) or 1500.0
        out["roofline"] = {"kernel": "syrk_tc2_kernel ([AtA|Atb] of the last level, tcgen05 3xTF32)", "bound": "tensor", "achieved": alg / t / 1e12, "peak": peak,
                           "unit": "TFLOP/s", "frac": alg / t / 1e12 / peak,
                           # DRAM bytes of this launch from the committed ncu capture: only valid for the shape it was taken on
                           "traffic": 8569163000 + 584547000 if (world == 1 and cfg is TRAIN_CFGS["train"]) else None,
                           "traffic_source": "profiles/r02_summary.md section 3 (ncu --set full capture of this launch shape on one GPU), not this run",
                           "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (dense bf16; the kernel runs kind::tf32 at half that rate, three passes)" if peaks else "fallback 1500 (B200_PROFILING.md)",
                           "ms_per_launch": solver_ms["At * A"], "algorithmic_flops_per_launch": alg,
                           "executed_tf32_tflops": syrk_executed_flops(n_loc, D, 2 * L) / t / 1e12,
                           "static_profile": {"source": "profiles/r02_summary.md section 3 (ncu --set full capture of the config-4 Gram launch on one GPU: tensor-pipe activity and the DRAM bytes reported as traffic)",
                                              "tensor_pipe_active_pct": 84.15}}
    out["algorithmic_tflop"] = {"gram_syrk": S * (cfg["n"] * D * (D + 1.0) + 2.0 * cfg["n"] * D * 2 * L) / 1e12, "cholesky_and_solve": S * (D ** 3 / 3.0 + 2.0 * D * D * 2 * L) / 1e12}
    if e2e:
        # the same run from HOST buffers: crops and landmark rows in pinned memory, uploads inside the timed region, the trained
        # weights read back to the host
        h_imgs = torch.empty(imgs.shape, dtype=torch.uint8).pin_memory()
        h_imgs.copy_(imgs)
        del ht, imgs
        torch.cuda.synchronize()
        barrier()
        e0.record()
        for _ in range(steps):
            d_imgs = h_imgs.to(dev, non_blocking=True)
            ht2 = sd.HogTransform(d_imgs, hps, ids, right, left, ctx)
            regs = [sd.LinearRegressor(sd.Regulariser(sd.RegularisationType.MatrixNorm, cfg["lambda_factor"], False), ctx) for _ in hps]
            sdo = sd.SupervisedDescentOptimiser(regs, sd.InterEyeDistanceNormalisation(ids, right, left), ctx)
            sdo.train(x_gt, x0, None, ht2, None, comm=comm, distributed_solve=ds)
            w_host = [r.x.cpu() for r in regs]
            del ht2, d_imgs
        e1.record()
        barrier()
        secs2 = max_over_ranks(e0.elapsed_time(e1)) * 1e-3 / steps
        out["e2e"] = {"value": secs2, "unit": "s", "h2d_bytes_per_step": int(h_imgs.numel() + x0.nbytes + x_gt.nbytes),
                      "d2h_bytes_per_step": int(sum(w.numel() * 4 for w in w_host)),
                      "api": "SupervisedDescentOptimiser.train with HogTransform over crops uploaded from pinned host memory; trained weights copied back"}
    ctx.set_solver("cholesky")
    return out


def cpu_train_level_seconds(n_samples, threads, cfg=None):
    """Reference CPU path for ONE training level (level 0: the most expensive one), all host threads: the reference's hog.c
    inside the restated HogTransform glue (one sample per thread, as the thread pool of superviseddescent.hpp:173-189), then
    BLAS/LAPACK (numpy/scipy sgemm, sgetrf, sgetrs) standing in for Eigen's A^T A and PartialPivLU (regressors.hpp:199-234) --
    BASELINE.md section 3.  n_samples may be a bounded sample of the config's N; total_extrapolated_s scales the parts."""
    import scipy.linalg
    from oracle import oracle as O
    cfg = cfg or TRAIN_CFG
    om = O.Model(MODEL)
    use_ref = O.ref_available()
    size = cfg["size"]
    L = cfg["landmarks"]
    if L == 22:
        mean, right_idx, left_idx = om.mean, om.right_idx, om.left_idx
    else:
        mean = np.load(os.path.join(ROOT, "tests", "golden", "mean_ibug_lfpw_68.npy")).astype(np.float32).reshape(-1)
        right_idx, left_idx = [36, 39], [42, 45]          # ids "37","40" / "43","46" of the 1-based 68-point list
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import synth
    base = synth.smooth_images(64, size, size, cfg["seed"])
    imgs = np.concatenate([base] * ((n_samples + 63) // 64))[:n_samples]
    m = int(round(size * 0.05))
    box = (m, m, size - 2 * m, size - 2 * m)
    rng = np.random.Generator(np.random.PCG64(cfg["seed"]))
    x0 = np.tile(O.align_mean(mean, box), (n_samples, 1)).astype(np.float32)
    x_gt = np.stack([O.align_mean(mean, box, 1.0 + rng.normal(0, 0.04), 1.0 + rng.normal(0, 0.04), rng.normal(0, 0.04), rng.normal(0, 0.04))
                     for _ in range(n_samples)]).astype(np.float32)
    hp = O.HogParam(1, cfg["cells"], cfg["cell_sizes"][0], cfg["num_bins"], cfg["rel"][0])
    t0 = time.perf_counter()
    A = O.hog_transform_batch(imgs, x0, hp, right_idx, left_idx, use_ref=use_ref, threads=threads)
    t_hog = time.perf_counter() - t0
    D_full = A.shape[1]
    if D_full > 20000:                                   # bounded sample: a 52,701-column LU does not fit a bench run
        keep = np.r_[0:17050, D_full - 1]
        A = np.ascontiguousarray(A[:, keep])
    D = A.shape[1]
    ied = np.array([O.get_ied(x0[i], right_idx, left_idx) for i in range(n_samples)])
    b = ((x0 - x_gt) / ied[:, None]).astype(np.float32)
    t0 = time.perf_counter()
    G = A.T @ A
    lam = 1.5 * np.linalg.norm(G) / n_samples
    G[np.diag_indices_from(G)] += lam
    G[-1, -1] -= lam
    t_gram = time.perf_counter() - t0
    t0 = time.perf_counter()
    lu = scipy.linalg.lu_factor(G, overwrite_a=True, check_finite=False)
    X = scipy.linalg.lu_solve(lu, A.T @ b, check_finite=False)
    t_lu = time.perf_counter() - t0
    t0 = time.perf_counter()
    _ = x0 - (A @ X) * ied[:, None]
    t_upd = time.perf_counter() - t0
    fn = cfg["n"] / n_samples
    fd = D_full / D
    total_x = t_hog * fn + t_gram * fn * fd * fd + t_lu * fd ** 3 + t_upd * fn * fd
    return {"hog_s": t_hog, "gram_s": t_gram, "lu_solve_s": t_lu, "update_s": t_upd, "total_s": t_hog + t_gram + t_lu + t_upd,
            "total_extrapolated_s": total_x, "D": D, "D_full": D_full,
            "kind": "reference hog.c + BLAS/LAPACK for Eigen" if use_ref else "port + BLAS/LAPACK"}


def run_train_workload(args, sd, ctx, model, world, rank, local, dev, barrier, max_over_ranks, comm):
    """--workload train / train5: the regressor-train metric of BASELINE.json as the line itself."""
    cfg = TRAIN_CFGS[args.workload]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ds = {"auto": None, "replicated": False, "distributed": True, "cg": "cg"}[args.solve]
    outputs = {} if args.dump_outputs else None
    line = run_train(sd, ctx, model, world, rank, dev, barrier, max_over_ranks, comm, cfg, steps=args.steps, warmup=args.warmup, e2e=True,
                     distributed_solve=ds, solver="cg" if args.solve == "cg" else "cholesky", outputs=outputs)
    clocks = sampler.stop() if rank == 0 else None
    if rank != 0:
        return
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    line["clocks"] = clocks
    if world == 1 and not args.no_cpu:
        try:
            cores = host_cores()
            n_cpu = min(cfg["n"], 10000) if cfg["landmarks"] == 22 else 1500
            lvl = cpu_train_level_seconds(n_cpu, cores, cfg)
            S = len(cfg["cell_sizes"])
            line["cpu_baseline"] = {"value": lvl["total_extrapolated_s"] * S, "unit": "s", "cores": cores, "kind": "port",
                                    "sample": f"ONE level (level 0) on {n_cpu} of the {cfg['n']} samples on the host: HOG {lvl['hog_s']:.2f} s, "
                                              f"Gram {lvl['gram_s']:.2f} s, LU+solve {lvl['lu_solve_s']:.2f} s, update {lvl['update_s']:.2f} s; "
                                              f"HOG/Gram/update scaled linearly to {cfg['n']} samples"
                                              + (", LU at the sample's D" if lvl["D"] == lvl["D_full"] else f", LU scaled by (D/{lvl['D']})^3 to D={lvl['D_full']}")
                                              + f"; x{S} levels (extrapolated); {lvl['kind']}"}
        except Exception as ex:
            line["cpu_baseline"] = {"error": repr(ex)[:200]}
    print(json.dumps(line))


def run_ours(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        group = dist.group.WORLD
    from superviseddescent_b200 import api as sd
    from superviseddescent_b200 import parallel
    ctx = sd.Context(local)
    model = sd.load_detection_model(MODEL, ctx)
    comm = parallel.Communicator(ctx, group) if world > 1 else None   # the C ABI's NCCL communicator (training exchange)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world > 1:
            t = torch.tensor([v], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return v

    if args.workload != "detect":
        run_train_workload(args, sd, ctx, model, world, rank, local, dev, barrier, max_over_ranks, comm)
        if comm is not None:
            comm.close()
        if world > 1:
            dist.destroy_process_group()
        return

    B = args.batch
    L = model.num_landmarks

    frames = synth_frames_torch(B, 1234 + rank, dev)
    boxes = synth_boxes(B, 1234 + rank)
    mean = model.get_mean()
    x0 = np.stack([sd.align_mean(mean, b) for b in boxes])
    x0_dev = torch.from_numpy(x0).to(dev)
    h_frames = torch.empty((B, H_IMG, W_IMG), dtype=torch.uint8).pin_memory()
    h_frames.copy_(frames)
    torch.cuda.synchronize()
    h_np = h_frames.numpy()

    # ---------------- device-resident throughput ----------------
    for _ in range(args.warmup):
        out = model.detect_batch_device(frames, x0_dev)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = ctx.launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = model.detect_batch_device(frames, x0_dev)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    launches = ctx.launches() - l0
    value = world * B * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"landmarks": out.cpu().numpy()})

    # ---------------- end to end through the host-buffer call ----------------
    for _ in range(min(args.warmup, 2)):
        lm = model.detect_batch(h_np, boxes)
    barrier()
    e0.record()
    for _ in range(args.steps):
        lm = model.detect_batch(h_np, boxes)
    e1.record()
    barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if rank == 0 else None      # sampled across both timed regions (device-resident and e2e)
    e2e = world * B * args.steps / (ms_e2e * 1e-3)
    assert np.array_equal(lm, out.cpu().numpy()), "host and device paths disagree"

    # ---------------- roofline of the dominant kernel: HOG, cascade level 0 ----------------
    import ctypes as C
    from superviseddescent_b200 import _capi
    hp0 = model.hog_param(0)
    D0 = _capi.lib().sd_hog_feature_length(L, C.byref(hp0))
    ld = (D0 + 3) // 4 * 4
    A = torch.empty((B, ld), dtype=torch.float32, device=dev)
    norm = sd.NormalisationC()
    _capi.lib().sd_model_normalisation(model._m, C.byref(norm))
    ib = sd.ImageBatchC(C.c_void_p(frames.data_ptr()), W_IMG, H_IMG, frames.stride(1), frames.stride(0), B)

    def hog0():
        rc = _capi.lib().sd_hog_batch(ctx.h, C.byref(ib), None, _capi.ptr(x0_dev), C.c_int64(2 * L), B, L, C.byref(norm), C.byref(hp0), _capi.ptr(A), C.c_int64(ld))
        assert rc == 0
    for _ in range(3):
        hog0()
    torch.cuda.synchronize()
    reps = max(5, args.steps)
    e0.record()
    for _ in range(reps):
        hog0()
    e1.record()
    torch.cuda.synchronize()
    hog_ms = e0.elapsed_time(e1) / reps
    # algorithmic bytes (SURVEY 8d): unique source pixels read once + the descriptor row written once
    ri = [norm.right_idx[i] for i in range(norm.n_right)]
    li = [norm.left_idx[i] for i in range(norm.n_left)]
    ied = np.hypot(x0[:, ri].mean(1) - x0[:, li].mean(1), x0[:, [i + L for i in ri]].mean(1) - x0[:, [i + L for i in li]].mean(1))
    P = 2 * np.round(hp0.relative_patch_size * ied / 2)
    alg_bytes = float(np.sum(np.minimum(L * P * P, W_IMG * H_IMG)) + B * D0 * 4)
    fs0 = hp0.num_cells * hp0.cell_size
    alg_flops = float(B * L * fs0 * fs0 * (24 + 4 * hp0.num_bins))
    peak, peak_src = measured_peaks()
    achieved = alg_bytes / (hog_ms * 1e-3) / 1e9
    fp32_peak = 148 * 128 * 2 * 1.965e9 / 1e12      # 148 SMs x 128 FMA lanes x 2 flop x boost clock (B200_PROFILING.md)
    roofline = {"kernel": f"hog_patch_kernel<{hp0.num_bins}> (cascade level 0, fs={fs0})",
                "bound": "issue", "bound_note": "instruction-issue / fp32-ALU + shared-memory bound (~40 flop per algorithmic byte, SURVEY 8d), not HBM; "
                                                 "achieved/peak/frac are the HBM figures the contract asks for, frac_binding is the fp32 one",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src, "ms_per_launch": hog_ms,
                # DRAM bytes per launch from the committed `ncu --set full` capture (2048 faces), scaled per face: a capture, not this run
                "traffic": HOG_STATIC_PROFILE["dram_bytes_per_face"] * B, "traffic_source": HOG_STATIC_PROFILE["source"],
                "algorithmic_bytes_per_launch": alg_bytes,
                "achieved_fp32_tflops": alg_flops / (hog_ms * 1e-3) / 1e12, "fp32_peak_tflops": fp32_peak,
                "frac_binding": alg_flops / (hog_ms * 1e-3) / 1e12 / fp32_peak,
                "static_profile": dict(HOG_STATIC_PROFILE, dram_bytes_this_batch=HOG_STATIC_PROFILE["dram_bytes_per_face"] * B,
                                       note="quoted from a committed ncu capture, not measured in this run")}

    train = None
    if not args.no_train:
        try:
            train = run_train(sd, ctx, model, world, rank, dev, barrier, max_over_ranks, comm)
        except Exception as ex:   # the headline line must still be printed
            train = {"error": repr(ex)[:300]}
    if comm is not None:
        comm.close()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    line = {
        "metric": "faces/sec RCR 22-landmark detect", "value": value, "unit": "faces/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[2]: RCR 22-landmark detect, pre-trained face_landmarks_model_rcr_22.bin, 640x480 8UC1 synthetic frames, batched",
                   "frames_per_gpu": B, "global_batch": world * B, "cascade_levels": model.num_levels, "landmarks": L,
                   "parallelism": f"face-batch sharded over {world} GPU(s), no collective",
                   "l2": f"inputs ({B * W_IMG * H_IMG / 1e6:.0f} MB of frames per GPU) exceed the 126 MB L2"},
        "e2e": {"value": e2e, "unit": "faces/s", "h2d_bytes_per_step": int(B * W_IMG * H_IMG + B * 2 * L * 4), "d2h_bytes_per_step": int(B * 2 * L * 4),
                "ms_per_step": ms_e2e / args.steps, "api": "detection_model.detect_batch (sd_detect_batch_host), pinned host frames",
                "note": "h2d_bytes_per_step counts the host frames handed to the call; the engine's region-of-interest route reads only "
                        "each face's window (~1/4 of a frame) over PCIe inside the timed region (DESIGN.md 4.5)"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
    }
    if train is not None:
        line["train"] = train
    if world == 1 and not args.no_cpu and train is not None and "value" in train:
        try:
            cores = host_cores()
            lvl = cpu_train_level_seconds(TRAIN_CFG["n"], cores, TRAIN_CFG)
            train["cpu_baseline"] = {"value": lvl["total_s"] * len(TRAIN_CFG["cell_sizes"]), "unit": "s", "cores": cores, "kind": "port",
                                     "sample": f"ONE full level (level 0, all {TRAIN_CFG['n']} samples) timed on the host: HOG {lvl['hog_s']:.2f} s, "
                                               f"Gram {lvl['gram_s']:.2f} s, LU+solve {lvl['lu_solve_s']:.2f} s, update {lvl['update_s']:.2f} s; "
                                               f"x{len(TRAIN_CFG['cell_sizes'])} levels (extrapolated); {lvl['kind']}"}
        except Exception as ex:
            train["cpu_baseline"] = {"error": repr(ex)[:200]}
    if world == 1 and not args.no_cpu:
        cores = host_cores()
        n = max(256, cores * 32)
        r, kind, dt = cpu_detect_rate(n, cores, 4321)
        r1, _, _ = cpu_detect_rate(48, 1, 4322)
        line["cpu_baseline"] = {"value": r, "unit": "faces/s", "cores": cores, "kind": kind,
                                "sample": f"{n} faces of the same workload, one face per thread ({dt:.1f} s); single-thread reference-faithful predict: {r1:.1f} faces/s",
                                "single_thread_value": r1}
    if world > 1:
        dist.destroy_process_group()
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--workload", default="detect", choices=["detect", "train", "train5"],
                    help="detect = configs[2] (the default headline line); train = configs[3] and train5 = configs[4]: regressor-train "
                         "seconds as a first-class line (strong scaling over --gpus)")
    ap.add_argument("--solve", default="auto", choices=["auto", "replicated", "distributed", "cg"],
                    help="solve route of the train workloads: replicated / distributed blocked Cholesky, or conjugate gradients (cg)")
    ap.add_argument("--batch", type=int, default=4096, help="frames per GPU per step")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-train", action="store_true", help="skip the extra regressor-train measurement")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (float32, at most 64 MB; a seeded sample of rows when larger)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = {"detect": 10, "train": 3, "train5": 1}[args.workload]
    if args.warmup is None:
        args.warmup = {"detect": 3, "train": 1, "train5": 1}[args.workload]
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
