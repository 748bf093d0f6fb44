"""The C++14 shell's detect(images, list of face boxes per image), compiled against libsd_b200.so.

CPU: the translation unit compiles as C++14 and the binary fails loudly without a GPU.  GPU: two boxes on one example frame and
one on another (two sizes) equal the single-face detect(image, facebox), on the gray and the colour route."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def faces_binary(tmp_path_factory):
    from superviseddescent_b200 import build
    lib = build.build()
    out = str(tmp_path_factory.mktemp("cpp") / "test_detect_faces")
    cmd = ["g++", "-std=c++14", "-O1", "-Wall", "-Werror=return-type", "-I", os.path.join(ROOT, "include"),
           "-I", os.path.join(ROOT, "superviseddescent_b200", "include"), os.path.join(ROOT, "tests", "cpp", "test_detect_faces.cpp"),
           "-L", os.path.dirname(lib), "-lsd_b200", f"-Wl,-rpath,{os.path.dirname(lib)}", "-lpthread", "-o", out]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-4000:]
    return out


def test_detect_faces_shell_compiles_as_cxx14(faces_binary):
    assert os.path.exists(faces_binary)


def test_detect_faces_shell_fails_loudly_without_gpu(faces_binary, golden):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = subprocess.run([faces_binary, golden.model_path], capture_output=True, text=True)
    assert r.returncode != 0 and "no usable CUDA device" in r.stdout


@pytest.mark.gpu
def test_detect_faces_shell_equals_single_face_detect(faces_binary, golden, tmp_path):
    args = [faces_binary, golden.model_path]
    for i in (1, 3):
        gray = np.ascontiguousarray(golden.examples[f"gray{i}"])
        raw = tmp_path / f"frame{i}.raw"
        raw.write_bytes(gray.tobytes())
        args += [str(raw), str(gray.shape[1]), str(gray.shape[0])]
    b1, b3 = golden.examples["boxes"][1], golden.examples["boxes"][3]
    shifted = (int(b1[0]) + int(b1[2]) // 6, int(b1[1]) - int(b1[3]) // 8, int(b1[2]), int(b1[3]))   # overlaps the first box
    for box in (b1, shifted, b3):
        args += [str(int(v)) for v in box]
    r = subprocess.run(args, capture_output=True, text=True, timeout=300)
    print(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "ALL OK" in r.stdout
