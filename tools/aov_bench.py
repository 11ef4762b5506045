"""Cost of the first-hit feature-buffer pass (rtb_render_aov) next to the render it accompanies (rtb_render_accum).

    python tools/aov_bench.py [--out FILE.json] [--reps 5] [--spp 1,16,128]

For C3 (1 002 528-triangle height-field room, 1920x1080) and C1 (the reference scene, 320x180): after a warm-up,
the AOV pass (all five outputs) and the render (trace_path, depth 5, the default wavefront kernels) are timed with
CUDA events, alternating, `reps` times each per sample count, with a 512 MB memset between timed steps (L2 flushed).
Reported per sample count: median ms of both, the AOV pass's primary rays per second, the render's rays per second
(its own ray counter), the ratio AOV / render, and the primary rays' share of the render's rays -- the cost a fused
bounce-0 write would have instead.  The card's name and power limit are recorded with the numbers (a query only).
"""
import argparse
import json
import os
import subprocess
import sys

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


def scenes(api):
    W, H = 1920, 1080
    c3 = api.mesh_room(api.heightfield_mesh(708, 20 * W / H * 0.98), W, H)
    return [("c3", c3, W, H), ("c1", api.scene_default(320, 180), 320, 180)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--spp", default="1,16,128")
    args = ap.parse_args()
    import torch

    api = entry.load_package().api
    api.load()
    dev = torch.device("cuda:0")
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    result = {"tool": "tools/aov_bench.py", "card": card(), "reps": args.reps,
              "timing": "CUDA events on one stream, median of reps; 512 MB memset between timed steps (not timed)",
              "render": "rtb_render_accum, trace_path, max_depth 5, kernel 0 (wavefront), planes auto",
              "aov": "rtb_render_aov, all five outputs, planes auto", "configs": []}
    for name, src, W, H in scenes(api):
        cam = api.init_camera(W, H)
        n_px = W * H
        accum = torch.empty(n_px * 3, dtype=torch.float32, device=dev)
        bufs = [torch.empty(n_px * 3, dtype=torch.float32, device=dev), torch.empty(n_px * 3, dtype=torch.float32, device=dev),
                torch.empty(n_px, dtype=torch.float32, device=dev), torch.empty(n_px, dtype=torch.int32, device=dev),
                torch.empty(n_px, dtype=torch.int32, device=dev)]
        ptrs = [b.data_ptr() for b in bufs]
        with api.Scene(src) as sc:
            for spp in [int(s) for s in args.spp.split(",")]:
                desc = api.make_desc(W, H, 0, spp, max_depth=5, seed=SEED, profile=0)
                render = lambda: sc.render_accum(cam, desc, accum.data_ptr(), stream=stream)  # noqa: E731
                aov = lambda: sc.render_aov_accum(cam, desc, *ptrs, stream=stream)  # noqa: E731
                r_ctr = sc.render_accum(cam, desc, accum.data_ptr(), stream=stream, want_counters=True)  # warm-up + counts
                a_ctr = sc.render_aov_accum(cam, desc, *ptrs, stream=stream, want_counters=True)
                times = {"render": [], "aov": []}
                for i in range(args.reps):
                    for which, fn in (("render", render), ("aov", aov)):
                        flush.fill_(i & 0xFF)
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        fn()
                        e1.record()
                        e1.synchronize()
                        times[which].append(e0.elapsed_time(e1))
                r_ms, a_ms = float(np.median(times["render"])), float(np.median(times["aov"]))
                primary = n_px * spp
                row = {"scene": name, "width": W, "height": H, "spp": spp,
                       "render_ms": r_ms, "render_ms_all": times["render"], "render_rays": int(r_ctr.rays),
                       "render_grays_s": r_ctr.rays / (r_ms * 1e-3) / 1e9,
                       "aov_ms": a_ms, "aov_ms_all": times["aov"], "aov_primary_rays": int(a_ctr.rays),
                       "aov_mrays_s": primary / (a_ms * 1e-3) / 1e6, "aov_prim_tests": int(a_ctr.prim_tests),
                       "aov_over_render": a_ms / r_ms, "primary_share_of_render_rays": primary / r_ctr.rays}
                assert a_ctr.rays == primary
                result["configs"].append(row)
                print(json.dumps({k: v for k, v in row.items() if not k.endswith("_all")}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
