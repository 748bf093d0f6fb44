"""The C++14 shell's detect overloads on colour (8UC3 B,G,R) frames, compiled against libsd_b200.so.

CPU: the translation unit compiles as C++14 and the binary fails loudly without a GPU.  GPU: two example photographs (two
sizes) in colour give the gray-frame landmarks bit for bit through every detect overload, the tracking ones included."""
import os
import subprocess

import numpy as np
import pytest

import colour_examples

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def colour_binary(tmp_path_factory):
    from superviseddescent_b200 import build
    lib = build.build()
    out = str(tmp_path_factory.mktemp("cpp") / "test_detect_colour")
    cmd = ["g++", "-std=c++14", "-O1", "-Wall", "-Werror=return-type", "-I", os.path.join(ROOT, "include"),
           "-I", os.path.join(ROOT, "superviseddescent_b200", "include"), os.path.join(ROOT, "tests", "cpp", "test_detect_colour.cpp"),
           "-L", os.path.dirname(lib), "-lsd_b200", f"-Wl,-rpath,{os.path.dirname(lib)}", "-lpthread", "-o", out]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-4000:]
    return out


def test_detect_colour_shell_compiles_as_cxx14(colour_binary):
    assert os.path.exists(colour_binary)


def test_detect_colour_shell_fails_loudly_without_gpu(colour_binary, golden):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = subprocess.run([colour_binary, golden.model_path], capture_output=True, text=True)
    assert r.returncode != 0 and "no usable CUDA device" in r.stdout


@pytest.mark.gpu
def test_detect_colour_shell_equals_gray_frames(colour_binary, golden, tmp_path):
    bgr = colour_examples.load(golden.dir)
    args = [colour_binary, golden.model_path]
    for i in (1, 3):
        gray = np.ascontiguousarray(golden.examples[f"gray{i}"])
        (tmp_path / f"frame{i}.bgr").write_bytes(bgr[i].tobytes())
        (tmp_path / f"frame{i}.gray").write_bytes(gray.tobytes())
        args += [str(tmp_path / f"frame{i}.bgr"), str(tmp_path / f"frame{i}.gray"), str(gray.shape[1]), str(gray.shape[0])]
    b1, b3 = golden.examples["boxes"][1], golden.examples["boxes"][3]
    shifted = (int(b1[0]) + int(b1[2]) // 6, int(b1[1]) - int(b1[3]) // 8, int(b1[2]), int(b1[3]))   # overlaps the first box
    for box in (b1, shifted, b3):
        args += [str(int(v)) for v in box]
    r = subprocess.run(args, capture_output=True, text=True, timeout=300)
    print(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "ALL OK" in r.stdout
