"""Cost and gain of next-event estimation (RTB_INTEGRATOR_PATH_NEE) against trace_path (RTB_INTEGRATOR_PATH).

    python tools/nee_bench.py [--out profiles/nee_bench.json] [--reps 5]

1. Time per sample: C1 (the reference scene, 320x180) and C3 (1 002 528-triangle height-field room, 1920x1080), depth 5,
   the default wavefront kernels, rtb_render_accum timed with CUDA events, PATH and NEE alternating, `reps` times each,
   a 512 MB memset between timed steps (L2 overwritten, not timed).
2. Equal time on C1 320x180: for PATH budgets of 4, 16 and 64 spp, NEE gets the samples that fit in the same measured
   time; both frames are scored against the reference's converged frame (tests/golden/c1_converged_320x180.npz), raw
   and denoised (rtb_render_denoised, default settings), as PSNR of the 8-bit frames.
The card's name and power limit are recorded with the numbers (a query only).
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import __graft_entry__ as entry  # noqa: E402

SEED = 1666943821
PATH, NEE = 0, 2


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = ""
    return out or "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "nee_bench.json"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch
    import oracle_lib as ol
    from denoise_ref import psnr_vs

    api = entry.load_package().api
    api.load()
    dev = torch.device("cuda:0")
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    result = {"tool": "tools/nee_bench.py", "card": card(), "reps": args.reps,
              "timing": "CUDA events on one stream, median of reps, PATH and NEE alternating; 512 MB memset between "
                        "timed steps (not timed)",
              "render": "rtb_render_accum, max_depth 5, kernel 0 (wavefront), planes auto, stochastic dielectric",
              "time_per_spp": [], "equal_time_c1": []}

    W3, H3 = 1920, 1080
    c3 = api.mesh_room(api.heightfield_mesh(708, 20 * W3 / H3 * 0.98), W3, H3)
    ms_per_spp = {}
    for name, src, W, H, spp in (("c1", api.scene_default(320, 180), 320, 180, 64), ("c3", c3, W3, H3, 16)):
        cam = api.init_camera(W, H)
        accum = torch.empty(W * H * 3, dtype=torch.float32, device=dev)
        with api.Scene(src) as sc:
            descs = {k: api.make_desc(W, H, 0, spp, max_depth=5, seed=SEED, profile=0, integrator=k) for k in (PATH, NEE)}
            ctrs = {k: sc.render_accum(cam, descs[k], accum.data_ptr(), stream=stream, want_counters=True) for k in descs}
            times = {PATH: [], NEE: []}
            for i in range(args.reps):
                for k in (PATH, NEE):
                    flush.fill_(i & 0xFF)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    sc.render_accum(cam, descs[k], accum.data_ptr(), stream=stream)
                    e1.record()
                    e1.synchronize()
                    times[k].append(e0.elapsed_time(e1))
        med = {k: float(np.median(v)) for k, v in times.items()}
        ms_per_spp[name] = {k: med[k] / spp for k in med}
        row = {"scene": name, "width": W, "height": H, "spp": spp,
               "path_ms_per_spp": med[PATH] / spp, "nee_ms_per_spp": med[NEE] / spp, "nee_over_path": med[NEE] / med[PATH],
               "path_ms_all": times[PATH], "nee_ms_all": times[NEE], "rays": int(ctrs[PATH].rays),
               "nee_rays": int(ctrs[NEE].rays), "shadow_rays": int(ctrs[NEE].shadow_rays),
               "shadow_hits": int(ctrs[NEE].shadow_hits)}
        assert row["rays"] == row["nee_rays"]
        result["time_per_spp"].append(row)
        print(json.dumps({k: v for k, v in row.items() if not k.endswith("_all")}), flush=True)

    W, H = 320, 180
    golden = np.load(os.path.join(ROOT, "tests", "golden", "c1_converged_320x180.npz"))["mean"].astype(np.float64)
    cam = api.init_camera(W, H)
    ratio = ms_per_spp["c1"][PATH] / ms_per_spp["c1"][NEE]
    with api.Scene(api.scene_default(W, H)) as sc:
        for path_spp in (4, 16, 64):
            nee_spp = max(1, int(path_spp * ratio))
            row = {"path_spp": path_spp, "nee_spp": nee_spp}
            for tag, k, spp in (("path", PATH, path_spp), ("nee", NEE, nee_spp)):
                desc = api.make_desc(W, H, 0, spp, max_depth=5, seed=SEED, profile=0, integrator=k)
                _, acc, _ = sc.render(cam, desc, want_accum=True)
                _, den, _, _ = sc.render_denoised(cam, desc)
                row[f"{tag}_psnr_raw"] = psnr_vs(acc.astype(np.float64) / spp, golden, ol)
                row[f"{tag}_psnr_denoised"] = psnr_vs(den.astype(np.float64), golden, ol)
            row["gain_raw_db"] = row["nee_psnr_raw"] - row["path_psnr_raw"]
            row["gain_denoised_db"] = row["nee_psnr_denoised"] - row["path_psnr_denoised"]
            result["equal_time_c1"].append(row)
            print(json.dumps(row), flush=True)

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
