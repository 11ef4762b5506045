"""Host side of the feature buffers, without a GPU: the PFM writer the CLI's -a option uses, and the CLI's refusal of
-a together with several GPUs (checked while parsing, before any CUDA work)."""
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def read_pfm(path):
    """a plain Portable FloatMap reader: header "PF"/"Pf", "<w> <h>", scale (< 0: little-endian), rows bottom to top"""
    with open(path, "rb") as f:
        data = f.read()
    head, size, scale, body = data.split(b"\n", 3)
    w, h = map(int, size.split())
    comp = {b"PF": 3, b"Pf": 1}[head]
    dtype = "<f4" if float(scale) < 0 else ">f4"
    img = np.frombuffer(body, dtype, count=w * h * comp).reshape(h, w, comp)[::-1]
    return head, float(scale), (img if comp == 3 else img[..., 0])


def test_pfm_writer_round_trip(api, tmp_path):
    _, host = api.load()
    rng = np.random.default_rng(3)
    rgb = rng.normal(size=(7, 5, 3)).astype(np.float32)
    rgb[0, 0] = (np.inf, -0.0, 1e-45)  # non-finite, signed zero and a denormal survive bit for bit
    grey = rng.uniform(0, 100, (4, 9)).astype(np.float32)
    p = tmp_path / "rgb.pfm"
    assert host.rt_write_pfm(str(p).encode(), 5, 7, 3, rgb.ctypes.data) == 1
    head, scale, back = read_pfm(p)
    assert head == b"PF" and scale == -1.0
    assert np.array_equal(back.view(np.uint32), rgb.view(np.uint32))
    raw = p.read_bytes()
    assert raw.startswith(b"PF\n5 7\n-1.0\n")
    # the first stored row is the BOTTOM row of the image (row 6), little-endian
    assert raw[len(b"PF\n5 7\n-1.0\n"):][:12] == rgb[6, 0].astype("<f4").tobytes()
    p = tmp_path / "grey.pfm"
    assert host.rt_write_pfm(str(p).encode(), 9, 4, 1, grey.ctypes.data) == 1
    head, scale, back = read_pfm(p)
    assert head == b"Pf" and scale == -1.0 and np.array_equal(back, grey)
    assert host.rt_write_pfm(b"/nonexistent-dir/x.pfm", 9, 4, 1, grey.ctypes.data) == 0
    assert host.rt_write_pfm(str(tmp_path / "y.pfm").encode(), 9, 4, 2, grey.ctypes.data) == 0


def test_cli_rejects_feature_buffers_on_several_gpus(tmp_path):
    exe = os.path.join(ROOT, "raytracer.c_b200", "bin", "raytracer")
    r = subprocess.run([exe, "-w", "64", "-h", "36", "-s", "1", "-o", str(tmp_path / "x.png"), "-G", "2", "-a",
                        str(tmp_path / "aov")], capture_output=True, text=True)
    assert r.returncode != 0
    assert "-a" in r.stderr and "-G 2" in r.stderr and "Usage:" in r.stderr
    assert os.listdir(tmp_path) == [], "nothing is rendered or written"
