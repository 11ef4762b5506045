"""Cost of the built-in denoiser (rtb_denoise) and of a denoised render (rtb_render_denoised) against the plain render
(rtb_render_mean).

    python tools/denoise_bench.py [--out profiles/denoise_bench.json] [--reps 7] [--spp 4,16,64]

C3 (1 002 528-triangle height-field room) at 1920x1080:
  1. rtb_denoise alone, default passes, on C3's own accum and feature sums (16 spp): CUDA events on one stream,
     median of `reps`, with a 512 MB memset between timed steps (L2 overwritten, not timed).
  2. rtb_render_denoised against rtb_render_mean at each sample count, both returning the 8-bit framebuffer only
     (host buffers out, so each call ends in a device synchronise): host clock, median of `reps`, the two alternating.
The card's name and power limit are read in the same run (a query only).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry  # noqa: E402

SEED = 1666943821


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = ""
    return out or "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--spp", default="4,16,64")
    args = ap.parse_args()
    import torch

    api = entry.load_package().api
    api.load()
    dev = torch.device("cuda:0")
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    W, H = 1920, 1080
    n_px = W * H
    src = api.mesh_room(api.heightfield_mesh(708, 20 * W / H * 0.98), W, H)
    cam = api.init_camera(W, H)
    result = {"tool": "tools/denoise_bench.py", "card": card(), "reps": args.reps, "scene": "c3", "width": W,
              "height": H, "denoise_defaults": "iterations 5, sigma_luminance 48, sigma_normal 128, sigma_depth 0.1, "
                                                "albedo_epsilon 1e-3"}
    f32 = dict(dtype=torch.float32, device=dev)
    b = dict(accum=torch.empty(3 * n_px, **f32), albedo=torch.empty(3 * n_px, **f32),
             normal=torch.empty(3 * n_px, **f32), depth=torch.empty(n_px, **f32),
             hits=torch.empty(n_px, dtype=torch.int32, device=dev), object=torch.empty(n_px, dtype=torch.int32, device=dev),
             out=torch.empty(3 * n_px, **f32))
    ptrs = [b[k].data_ptr() for k in ("accum", "albedo", "normal", "depth", "hits", "object", "out")]
    with api.Scene(src) as sc:
        spp = 16
        desc = api.make_desc(W, H, 0, spp, max_depth=5, seed=SEED, profile=0)
        sc.render_accum(cam, desc, b["accum"].data_ptr(), stream=stream)
        sc.render_aov_accum(cam, desc, *ptrs[1:6], stream=stream)
        api.denoise(W, H, spp, *ptrs, stream=stream)  # warm-up
        times = []
        for i in range(args.reps):
            flush.fill_(i & 0xFF)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            api.denoise(W, H, spp, *ptrs, stream=stream)
            e1.record()
            e1.synchronize()
            times.append(e0.elapsed_time(e1))
        out = b["out"].cpu().numpy()
        assert np.isfinite(out).all() and (out >= 0).all()
        result["denoise"] = {"spp_of_inputs": spp, "timing": "CUDA events, median of reps, 512 MB memset between steps",
                             "ms": float(np.median(times)), "ms_all": times,
                             "mpixels_s": n_px / (float(np.median(times)) * 1e-3) / 1e6}
        print(json.dumps({k: v for k, v in result["denoise"].items() if k != "ms_all"}), flush=True)

        rows = []
        for spp in [int(s) for s in args.spp.split(",")]:
            desc = api.make_desc(W, H, 0, spp, max_depth=5, seed=SEED, profile=0)
            plain = lambda: sc.render(cam, desc)  # noqa: E731  (rtb_render = rtb_render_mean, total = spp)
            dn = lambda: sc.render_denoised(cam, desc, want_denoised=False)  # noqa: E731  (framebuffer only, as plain)
            plain()
            dn()
            t = {"render_mean": [], "render_denoised": []}
            for _ in range(args.reps):
                for which, fn in (("render_mean", plain), ("render_denoised", dn)):
                    t0 = time.perf_counter()
                    fn()
                    t[which].append((time.perf_counter() - t0) * 1e3)
            r, d = float(np.median(t["render_mean"])), float(np.median(t["render_denoised"]))
            row = {"spp": spp, "render_mean_ms": r, "render_denoised_ms": d, "extra_ms": d - r, "ratio": d / r,
                   "render_mean_ms_all": t["render_mean"], "render_denoised_ms_all": t["render_denoised"]}
            rows.append(row)
            print(json.dumps({k: v for k, v in row.items() if not k.endswith("_all")}), flush=True)
        result["render_vs_render_denoised"] = {
            "timing": "host clock around calls that end in a device synchronise (framebuffer only, host buffer), "
                      "median of reps, alternating", "rows": rows}
    print(json.dumps({"card": result["card"]}))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
