"""bench.py --dump-outputs: what it writes (the pixels, the fixed sample of a large frame, the size bound) without a GPU, and on
the GPU that the dump is the frame the last timed step upscaled, bit for bit."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import fsr1_b200 as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("fsr1_bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_dump_writes_every_pixel_of_a_small_frame(tmp_path):
    b = _bench()
    img = torch.from_numpy(F.to_half(F.uniform(5, 3, 7)))
    b.dump_output(str(tmp_path), "output", img, max_pixels=15)
    got = np.load(tmp_path / "output.npy")
    assert got.dtype == np.float32 and np.array_equal(got, img.float().numpy().reshape(15, 4))


def test_dump_of_a_large_frame_is_the_same_seeded_sample_every_time(tmp_path):
    b = _bench()
    img = torch.from_numpy(F.uniform(40, 30, 8))
    for name in ("a", "b"):
        b.dump_output(str(tmp_path), name, img, max_pixels=100)
    a = np.load(tmp_path / "a.npy")
    assert a.shape == (100, 4) and np.array_equal(a, np.load(tmp_path / "b.npy"))
    idx = np.sort(np.random.default_rng(0).choice(40 * 30, 100, replace=False))
    assert np.array_equal(a, img.numpy().reshape(-1, 4)[idx])
    assert b.DUMP_PIXELS * 4 * 4 <= 64 << 20


def test_dump_needs_the_gpu_path():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", "x"],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode != 0 and "--dump-outputs" in r.stderr


@pytest.mark.gpu
def test_dump_is_the_frame_of_the_last_timed_step(tmp_path):
    b = _bench()
    steps = 3
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "0",
                        "--no-cpu", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["gpu_launches"] == 2 * steps            # the timed region ran `steps` frames of one EASU + one RCAS launch each
    iw, ih, ow, oh = b.WORKLOADS["1080p-4k-fp16"][:4]
    frame = torch.from_numpy(F.uniform(iw, ih, 12345 + (steps - 1) % b.RING).astype(np.float16)).cuda()
    tmp = torch.empty((oh, ow, 4), dtype=torch.float16, device="cuda")
    want = torch.empty_like(tmp)
    F.api.upscale(frame, tmp, want, F.api.easu_con(iw, ih, iw, ih, ow, oh), F.api.rcas_con(b.SHARPNESS))
    torch.cuda.synchronize()
    idx = np.sort(np.random.default_rng(0).choice(ow * oh, b.DUMP_PIXELS, replace=False))
    got = np.load(tmp_path / "output.npy")
    assert got.dtype == np.float32 and got.shape == (b.DUMP_PIXELS, 4)
    assert np.array_equal(got, want.float().cpu().numpy().reshape(-1, 4)[idx])
