#!/usr/bin/env python
"""Hold a `bench.py --dump-outputs DIR` directory against the oracle: "faster, not different" at the size bench timed.

    python tools/check_bench_dump.py DIR --workload cN [--scale F] [--gpus N] [--pixels K]

The oracle (tests/oracle_lib.pixel_paths: brute force, every sample of each pixel) replays K of the dumped pixels --
a seeded choice among pixel_index.npy where bench cut the frame, else among the whole frame, plus its corners -- with
bench.py's scene, frame, depth, seed and sample count (the named spp times --scale, the whole job over --gpus):

  accum.npy        every checked sum within the float bound of the pixel's oracle vertices (render_bound, counted
                   with 64 planes, the most the library cuts a frame into), one GPU only
  framebuffer.npy  every checked byte within one level of oracle_tonemap of the oracle's sums (all a dump of
                   several GPUs holds)

Prints the largest error-to-bound ratio; exits 1 when a value is out of bounds.  Cost: about 0.6 s of 8 CPU threads
per C3 pixel, far less on the sphere workloads.
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench  # noqa: E402
import oracle_lib as ol  # noqa: E402
from test_gpu_bench_frames import oracle_pixels  # noqa: E402

MAX_PLANES = 64  # rtb_plane_split's cap without a pinned plane count


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("dir")
    ap.add_argument("--workload", required=True, choices=sorted(bench.WORKLOADS))
    ap.add_argument("--scale", type=float, default=1.0, help="bench.py's --scale")
    ap.add_argument("--gpus", type=int, default=1, help="bench.py's --gpus (strong scaling: the same whole job)")
    ap.add_argument("--pixels", type=int, default=32, help="pixels to replay (plus the frame's corners where dumped)")
    args = ap.parse_args()

    W, H, spp, depth, _ = bench.WORKLOADS[args.workload]
    spp = max(1, int(round(spp * args.scale)))
    fb = np.load(os.path.join(args.dir, "framebuffer.npy"))
    acc_path = os.path.join(args.dir, "accum.npy")
    acc = np.load(acc_path) if os.path.exists(acc_path) else None
    if args.gpus == 1 and acc is None:
        raise SystemExit(f"{acc_path} missing: a one-GPU dump holds the sums")
    idx_path = os.path.join(args.dir, "pixel_index.npy")
    if os.path.exists(idx_path):
        dumped = np.load(idx_path).astype(np.int64)  # rows of the cut frames
    else:
        dumped = np.arange(W * H)
    fb = fb.reshape(len(dumped), 3)
    acc = acc.reshape(len(dumped), 3) if acc is not None else None

    rng = np.random.default_rng(bench.SEED)
    rows = rng.choice(len(dumped), min(args.pixels, len(dumped)), replace=False)
    corners = np.flatnonzero(np.isin(dumped, [0, W - 1, (H - 1) * W, H * W - 1]))
    rows = np.unique(np.concatenate([rows, corners]))
    pixels = dumped[rows]

    api = ol.pkg.api
    source, *_ = bench.build_host_scene(api, args.workload, W, H)
    cam = api.init_camera(W, H)
    want, bound, _ = oracle_pixels(ol, ol.abi, source, cam, W, H, pixels, spp, depth, MAX_PLANES)

    ok = True
    fb_want = ol.tonemap(want.reshape(1, -1, 3), spp).reshape(-1, 3).astype(int)
    level = np.abs(fb[rows].astype(int) - fb_want)
    print(f"{args.workload}: {W}x{H} {spp} spp, {len(pixels)} pixels; framebuffer: largest difference {level.max()} level(s)")
    if level.max() > 1:
        ok = False
        k = int(np.argmax(level.max(axis=1)))
        print(f"  FAIL framebuffer at pixel {pixels[k]}: {fb[rows][k]} vs oracle {fb_want[k]}")
    if acc is not None:
        got = acc[rows].astype(np.float64)
        err = np.abs(got - want)
        ratio = err / np.maximum(bound, 1e-300)
        print(f"  accum: largest error / bound = {ratio.max():.3f}")
        if (err > bound).any():
            ok = False
            k = int(np.argmax(ratio.max(axis=1)))
            print(f"  FAIL accum at pixel {pixels[k]}: {got[k]} vs oracle {want[k]} (bound {bound[k]})")
    print("OK" if ok else "FAILED")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
