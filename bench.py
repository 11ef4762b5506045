#!/usr/bin/env python
"""bench.py -- throughput of the render() hot path on N B200s (one process per GPU).

    python bench.py --gpus N --steps K --warmup W [--workload c1|c2|c3|c4|c5] [--scale F] [--dump-outputs DIR]
    python bench.py --impl reference ...        # the reference's CPU algorithm on host cores

--dump-outputs DIR writes what the last timed step computed (see dump_outputs) so that two builds can be
compared output for output: the inputs are seeded, identical from run to run for the same arguments.

A "step" is one pass of the hot path over one frame of synthetic input: the workload's frame at its
named samples per pixel.  With N GPUs the job is FIXED (--scaling strong, the default: C3 is "1080p,
128 spp", C4 "4096 spp sharded across 8"): rank r renders its 1/N of the global sample indices, the
per-GPU float sums are reduced to rank 0 by ONE ncclReduce, and rank 0 runs the gamma/quantise kernel --
all behind the C ABI (rtb_comm_render); torch.distributed only carries the 128-byte NCCL id, the
barrier and the max-over-ranks of the timings.  --scaling weak renders the named spp PER GPU.
`value` is whole-job Mrays/s with the scene and BVH already resident in HBM (ray = one trace_path
invocation, the reference's ray_count, raytracer.c:484).  `e2e` is the same metric through the
reference-facing call with HOST (pageable) buffers: scene upload + BVH build + render + framebuffer
read-back inside the timed region, every step (N > 1: rtb_render_multi, the upload sharded over the
GPUs' PCIe links and all-gathered over NVLink).

Workloads (BASELINE.json configs / SURVEY.md 8d):
  c1  reference main.c default scene, 320x180, 50 spp, depth 5
  c2  10k random spheres + walls, 1920x1080, 256 spp, depth 8
  c3  ~1M-triangle height-field mesh room, 1920x1080, 128 spp, depth 5   (default: the
      configuration the target ">= 1 Grays/s on 1 B200 for the 1080p mesh scene" is quoted on)
  c4  dielectric/metal-heavy 10k spheres, 3840x2160, 4096 spp, depth 8
  c5  all-dielectric deep-bounce stress, 512x512, 64 spp, depth 64
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry  # noqa: E402

WORKLOADS = {
    #      W     H    spp depth  description
    "c1": (320, 180, 50, 5, "reference main.c default scene (38 spheres), 320x180, 50 spp, depth 5"),
    "c2": (1920, 1080, 256, 8, "10k random spheres + 6 walls + 2 lights, 1920x1080, 256 spp, depth 8"),
    "c3": (1920, 1080, 128, 5, "1,002,528-triangle height-field mesh + 12 spheres, 1920x1080, 128 spp, depth 5"),
    "c4": (3840, 2160, 4096, 8, "10k spheres 40% dielectric / 40% mirror, 3840x2160, 4096 spp (sharded over the GPUs), depth 8"),
    "c5": (512, 512, 64, 64, "2k all-dielectric spheres deep-bounce stress, 512x512, 64 spp, depth 64"),
}
SEED = 1666943821  # main.c:182


def build_host_scene(api, name, W, H, pinned=False):
    """-> (source for api.Scene, n_bvh_levels L, bytes per primitive S, flops per test P, h2d bytes)"""
    if name == "c1":
        objs = api.scene_default(W, H)
        return objs, None, 16, 20, objs.nbytes
    if name in ("c2", "c4", "c5"):
        mix = {"c2": (0.5, 0.2, 0.2), "c4": (0.2, 0.4, 0.4), "c5": (0.1, 0.9, 0.0)}[name]
        count = 2000 if name == "c5" else 10000
        objs = api.scene_sphere_field(count, W, H, mix=mix, seed=SEED)
        return objs, len(objs), 16, 20, objs.nbytes
    if name == "c3":
        verts = api.heightfield_mesh(708, 20 * W / H * 0.98)
        if pinned:
            import torch
            buf = torch.empty(verts.nbytes, dtype=torch.uint8).pin_memory()
            pinned_np = buf.numpy().view(verts.dtype)
            pinned_np[:] = verts
            holder = api.mesh_room(pinned_np, W, H)
            holder._keep.append(buf)
        else:
            holder = api.mesh_room(verts, W, H)
        return holder, len(verts) // 3 + 12, 48, 51, verts.nbytes + 12 * 96
    raise SystemExit(f"unknown workload {name}")


def workload_config(name, total_spp, world, strong=True):
    W, H, _, depth, text = WORKLOADS[name]
    return {"workload": f"{name}: {text}", "width": W, "height": H, "spp_total": total_spp,
            "spp_per_gpu": total_spp / world, "max_depth": depth, "seed": SEED,
            "l2": "512 MB memset between timed steps (L2 flushed)",
            "parallelism": f"samples sharded x{world} ({'fixed job' if strong else 'fixed work per GPU'}), one ncclReduce of the float sums"
                           + (", scene upload sharded + all-gathered" if world > 1 else ""),
            "kernel": "wavefront (k_wf_generate / k_wf_trace / k_wf_shade), compressed BVH4"}


def algorithmic_cost(name, n_prims, S, P):
    """SURVEY.md 8(d): per INTERSECTED ray.  flops = 2*L*22 + 4*P + 60, bytes = L*64 + 4*S,
    L = ceil(log2(N/4)); C1 is the brute-force case 38*20+60 flop, 38*16 B."""
    if name == "c1":
        return 38 * 20 + 60, 38 * 16
    L = max(1, math.ceil(math.log2(max(n_prims, 8) / 4.0)))
    return 2 * L * 22 + 4 * P + 60, L * 64 + 4 * S


DUMP_LIMIT_BYTES = 60 * 10 ** 6  # under 64 MB in all, .npy headers included


def dump_outputs(out_dir, frames):
    """frames: {name: (H, W, 3) host array}, written as out_dir/<name>.npy in float32.  When the whole frames
    would exceed DUMP_LIMIT_BYTES, every frame is cut to the same fixed, seeded sample of pixels (rows of
    (n, 3)), and pixel_index.npy (float64) holds their flat indices y * W + x."""
    os.makedirs(out_dir, exist_ok=True)
    frames = {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in frames.items()}
    h, w, c = next(iter(frames.values())).shape
    n_pix = h * w
    per_pixel = len(frames) * c * 4
    if n_pix * per_pixel > DUMP_LIMIT_BYTES:
        keep = DUMP_LIMIT_BYTES // (per_pixel + 8)
        idx = np.sort(np.random.default_rng(SEED).choice(n_pix, keep, replace=False))
        frames = {k: v.reshape(n_pix, c)[idx] for k, v in frames.items()}
        frames["pixel_index"] = idx.astype(np.float64)
    for k, v in frames.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)"""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for k, nme in enumerate(names):
                if len(r) > 4 + k and r[4 + k].lower().startswith("active"):
                    reasons.add(nme)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d.get("hbm_gbs", 6650.0)), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(workload):
    """DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) of the k_wf_trace launches PER INTERSECTED RAY, from
    the committed ncu launch list of the same command (profiles/ncu_traffic.json), if any"""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        if d.get("kernel") == "k_wf_trace":
            return d.get(workload + "_bytes_per_intersected_ray")
    return None


# ---- CPU arm -------------------------------------------------------------------------------

def cpu_sample(name, W, H, depth):
    """a bounded sample of the same workload for the host cores: same scene, reduced frame"""
    # sized for roughly 10-20 s of host work per pass (the brute-force loop visits every primitive)
    return {"c1": (320, 180, 2000), "c2": (960, 540, 1), "c3": (64, 36, 1), "c4": (960, 540, 1), "c5": (512, 512, 8)}[name]


def run_cpu_step(api, ol, name, source, depth, step, threads):
    """one pass of the reference algorithm over the bounded sample -> (rays, seconds, kind).
    The oracle port (oracle/oracle.c: the reference's brute-force intersect() and trace_path()
    restated, bit-identical to the reference for sphere scenes) with OpenMP over rows and the
    keyed RNG.  The unmodified reference cannot run these workloads: it has no live mesh path
    (c3), its dielectric split is 2^depth (c5) and its OpenMP build serialises on rand()
    (SURVEY.md section 6)."""
    w, h, spp = cpu_sample(name, 0, 0, depth)
    cam = api.init_camera(w, h)
    t0 = time.perf_counter()
    _, (rays, _) = ol.render_sum(source, cam, w, h, spp, rng="philox", dielectric="stochastic", max_depth=depth,
                                 seed=SEED, sample_offset=step * spp, threads=threads)
    return rays, time.perf_counter() - t0, "port", f"{w}x{h}x{spp}spp of the same scene, oracle port, {threads} OpenMP threads"


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    pkg = entry.load_package()
    api = pkg.api
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as ol
    W, H, spp, depth, text = WORKLOADS[args.workload]
    spp = max(1, int(round(spp * args.scale)))
    strong = args.scaling == "strong"
    total_spp = spp if strong else spp * args.gpus
    threads = os.cpu_count() or 1
    exe = os.path.join(ROOT, "oracle", "_ref", "ref_main_cpu")
    if args.workload == "c1" and os.path.exists(exe):
        # the one config the UNMODIFIED reference program can run: /root/reference/main.c + raytracer.c as
        # shipped (Makefile:2 flags, default OpenMP threads), a bounded sample per step
        import re
        import tempfile
        w, h, s_ = 320, 180, 8
        sample = f"{w}x{h}x{s_}spp of C1 per step, the unmodified reference program as shipped (oracle/_ref/ref_main_cpu), {threads} OpenMP threads"
        kind = "reference"

        def one():
            with tempfile.TemporaryDirectory() as d:
                t0 = time.perf_counter()
                r = subprocess.run([exe, "-w", str(w), "-h", str(h), "-s", str(s_), "-o", os.path.join(d, "o.png")],
                                   capture_output=True, text=True, cwd=d, timeout=1800)
                dt = time.perf_counter() - t0
            return int(re.search(r"cast (\d+) rays", r.stdout).group(1)), dt
    else:
        # the bounded sample keeps the FULL scene (brute force over all primitives, like the reference)
        source, _, _, _, _ = build_host_scene(api, args.workload, W, H)
        kind = "port"
        sample = None
        step_no = [0]

        def one():
            nonlocal sample
            rays, dt, _, sample = run_cpu_step(api, ol, args.workload, source, depth, step_no[0], threads)
            step_no[0] += 1
            return rays, dt
    for _ in range(args.warmup):
        one()
    rays_total, t_total = 0, 0.0
    for _ in range(args.steps):
        rays, dt = one()
        rays_total += rays
        t_total += dt
    value = rays_total / t_total / 1e6
    line = {
        "impl": "reference", "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / max(1, args.steps),
        "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": dict(workload_config(args.workload, total_spp, args.gpus, strong), integrator=args.integrator, sample=sample,
                       note="the reference arm runs the bounded sample named in `sample` of this workload, on the host cores of rank 0"),
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ---- GPU arm -------------------------------------------------------------------------------

def reference_as_shipped(name):
    """BASELINE.md section 3 on C1, the one config the unmodified reference can run: oracle/_ref/ref_main_cpu is
    /root/reference/main.c + raytracer.c built with the reference's own flags (Makefile:2).
      (i)  as shipped: default OpenMP threads (they serialise on glibc's rand() lock, raytracer.c:227);
      (ii) one single-thread process per core, throughput summed.
    Rays are the reference's own ray_count (`cast N rays`, main.c:436).  A bounded sample: 320x180 at 8 spp."""
    exe = os.path.join(ROOT, "oracle", "_ref", "ref_main_cpu")
    if name != "c1" or not os.path.exists(exe):
        return None
    import re
    import tempfile
    cores = os.cpu_count() or 1
    W, H, S = 320, 180, 8
    out = {"sample": f"{W}x{H}x{S}spp of C1, the unmodified reference program (oracle/_ref/ref_main_cpu)", "cores": cores}

    def run(env_threads, tag):
        env = dict(os.environ)
        if env_threads:
            env["OMP_NUM_THREADS"] = str(env_threads)
        else:
            env.pop("OMP_NUM_THREADS", None)
        with tempfile.TemporaryDirectory() as d:
            return subprocess.Popen([exe, "-w", str(W), "-h", str(H), "-s", str(S), "-o", os.path.join(d, f"{tag}.png")],
                                    stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, env=env, cwd=d), d

    def rays_of(p):
        text = p.communicate(timeout=600)[0]
        m = re.search(r"cast (\d+) rays", text)
        return int(m.group(1)) if m else 0

    t0 = time.perf_counter()
    p, _ = run(None, "shipped")
    rays = rays_of(p)
    dt = time.perf_counter() - t0
    out["as_shipped"] = {"value": rays / dt / 1e6, "unit": "Mrays/s", "threads": cores, "seconds": dt}
    t0 = time.perf_counter()
    procs = [run(1, f"p{k}")[0] for k in range(cores)]
    rays = sum(rays_of(p) for p in procs)
    dt = time.perf_counter() - t0
    out["single_thread_processes"] = {"value": rays / dt / 1e6, "unit": "Mrays/s", "processes": cores, "seconds": dt}
    return out


def main_gpu(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    pkg = entry.load_package()
    api, abi = pkg.api, pkg.abi
    W, H, spp_named, depth, text = WORKLOADS[args.workload]
    spp_named = max(1, int(round(spp_named * args.scale)))
    # strong scaling (default): the named job, its samples split over the GPUs; weak: the named spp PER GPU
    strong = args.scaling == "strong"
    total_spp = spp_named if strong else spp_named * world
    integrator = 1 if args.integrator == "whitted" else 0
    source, n_prims, S, P, h2d_bytes = build_host_scene(api, args.workload, W, H, pinned=False)
    cam = api.init_camera(W, H)

    # ---- the group: behind the C ABI (rtb_comm_*); torch.distributed only carries the 128-byte id ------
    comm = None
    if world > 1:
        idt = torch.zeros(api.UNIQUE_ID_BYTES, dtype=torch.uint8, device=dev)
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(api.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, src=0)
        comm = api.Comm.rank(bytes(idt.cpu().numpy().tobytes()), rank, world, local)
        scene = comm.scene(source)          # sharded upload + all-gather + BVH build on every GPU
    else:
        scene = api.Scene(source, device=local)

    fb = torch.zeros((H, W, 3), dtype=torch.uint8, device=dev)
    accum = torch.zeros((H, W, 3), dtype=torch.float32, device=dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    stream = torch.cuda.current_stream(dev)
    # the WHOLE job; profile=0: no per-kernel events, so the wavefront pipeline runs as it does in production (two streams)
    desc = api.make_desc(W, H, 0, total_spp, max_depth=depth, seed=SEED, integrator=integrator, profile=0)

    def step(want_counters=False):
        """device-resident: accumulate (this rank's samples) -> one ncclReduce -> tonemap on rank 0"""
        if comm is not None:
            return scene.render(cam, desc, fb.data_ptr() if rank == 0 else None, want_counters=want_counters)
        c = scene.render_accum(cam, desc, accum.data_ptr(), stream=stream.cuda_stream, want_counters=want_counters)
        api.tonemap(accum.data_ptr(), W, H, total_spp, fb.data_ptr(), device=local, stream=stream.cuda_stream)
        return c

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # warm-up; the first pass, with counters, gives the (deterministic) whole-job ray count of a step
    ctr = step(want_counters=True)
    rays_step, hits_step = float(ctr.rays), float(ctr.rays_intersected)
    prim_tests = float(ctr.prim_tests)
    node_visits_rank, hits_prof = 0.0, 1.0  # node visits are counted by the profiling pass below (rank 0's share)
    launches_per_step = int(ctr.launches) + (1 if world == 1 else 0)  # whole job (+ the tonemap launch)
    for _ in range(max(3, args.warmup)):
        step()
    sync_all()

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    sync_all()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for i in range(args.steps):
        flush.fill_(i & 0xFF)  # evict L2 between timed steps (not timed)
        if world > 1:
            dist.barrier()
        ev[i][0].record(stream)
        step()
        ev[i][1].record(stream)
    sync_all()
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        # the last timed step's results, before the e2e and kernel-timing passes below reuse the buffers;
        # a group keeps the per-rank sums inside the library and hands rank 0 the framebuffer only
        frames = {"framebuffer": fb.cpu().numpy()}
        if comm is None:
            frames["accum"] = accum.cpu().numpy()
        dump_outputs(args.dump_outputs, frames)
    ms_local = sum(a.elapsed_time(b) for a, b in ev)
    t = torch.tensor([ms_local], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = t[0].item() / args.steps
    value = rays_step / ms_per_step / 1e3  # Mrays/s, whole job
    paths_per_s = W * H * total_spp / ms_per_step * 1e3

    # ---- e2e: the reference-facing call with HOST buffers, every step ------------------------
    # upload of the caller's (pageable, malloc'ed) scene + BVH build + render + framebuffer read-back
    e2e_steps = max(1, min(args.steps, 3))
    import ctypes as C
    _, host = pkg.load()
    opt = abi.Options()
    opt.width, opt.height, opt.samples = W, H, total_spp
    rp = abi.RenderParams()
    host.render_params_default(rp)
    rp.max_depth, rp.seed, rp.device, rp.integrator, rp.num_gpus = depth, SEED, local, integrator, 1
    fb_host = np.zeros((H, W, 3), dtype=np.uint8)

    def e2e_step(src):
        if world == 1:
            # the drop-in: render()/render_scene() of the C99 host library (raytracer.h:156)
            if isinstance(src, abi.SceneHolder):
                host.render_scene(fb_host.ctypes.data, C.addressof(src.objects), src.n, C.byref(cam), C.byref(opt), C.byref(rp))
            else:
                host.render_ex(fb_host.ctypes.data, src.ctypes.data, len(src), C.byref(cam), C.byref(opt), C.byref(rp))
        else:
            comm.render_host(src, cam, desc, want_counters=False, fb=fb_host)  # rtb_render_multi, collective

    def time_e2e(src):
        e2e_step(src)  # warm
        sync_all()
        calls = []
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            tc = time.perf_counter()
            e2e_step(src)
            calls.append((time.perf_counter() - tc) * 1e3)
        sync_all()
        te = torch.tensor([(time.perf_counter() - t0) * 1e3 / e2e_steps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        return te[0].item(), calls

    e2e_ms, e2e_calls = time_e2e(source)
    e2e_value = rays_step / e2e_ms / 1e3
    e2e_pinned = None
    if world == 1 and args.workload == "c3":
        # the same call with the scene in page-locked host memory (what a caller that registers its buffers gets)
        pinned_source, _, _, _, _ = build_host_scene(api, args.workload, W, H, pinned=True)
        pms, _ = time_e2e(pinned_source)
        e2e_pinned = {"value": rays_step / pms / 1e3, "ms_per_step": pms}

    # ---- roofline of the dominant kernel (k_wf_trace), rank 0's GPU --------------------------
    # its launches of one step (one per bounce and wave) are timed live with CUDA events on the launching
    # stream (rtb_counters.trace_ms); L2 flushed before each pass like the timed steps
    trace_ms_list, step_ms_list, trace_launches, hit_rank = [], [], 0, hits_step / world
    if integrator == 0:
        s0, s1 = api.shard_samples(0, total_spp, rank, world)
        rdesc = api.make_desc(W, H, s0, s1, max_depth=depth, seed=SEED)
        one = scene._handles[0] if comm is not None else None
        for i in range(min(args.steps, 3)):
            flush.fill_(i & 0xFF)
            if comm is not None:
                cc = abi.RtbCounters()
                api._check(api.load()[0].rtb_render_accum(one, cam.as_array().ctypes.data_as(C.POINTER(C.c_double)), C.byref(rdesc),
                                                          C.c_void_p(accum.data_ptr()), None, C.byref(cc)), "rtb_render_accum")
            else:
                cc = scene.render_accum(cam, rdesc, accum.data_ptr(), stream=stream.cuda_stream, want_counters=True)
            trace_ms_list.append(cc.trace_ms)
            step_ms_list.append(cc.gpu_ms)
            trace_launches = int(cc.trace_launches)
            hit_rank = float(cc.rays_intersected)
            node_visits_rank, hits_prof = float(cc.node_visits), max(1.0, float(cc.rays_intersected))
    trace_ms = sum(trace_ms_list) / max(1, len(trace_ms_list))
    trace_share = trace_ms / (sum(step_ms_list) / len(step_ms_list)) if step_ms_list else None
    flops_ray, bytes_ray = algorithmic_cost(args.workload, n_prims or 38, S, P)
    hbm_peak, hbm_src = measured_peaks()
    l2_peak = api.probe_l2_bandwidth(32 << 20, 50, device=local) if rank == 0 else 0.0  # measured now, GB/s
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    fp32_nominal = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12
    fp32_peak = api.probe_fp32_tflops(4096, device=local) if rank == 0 else fp32_nominal  # measured now
    HBM_BYTES_RAY = 64 + 16  # queue entry read once (o, d as doubles + the seeded hit record) + the hit record written back

    line = None
    if rank == 0:
        cpu_baseline, cpu_reference = None, None
        if world == 1 and not args.no_cpu_baseline:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import oracle_lib as ol
            threads = os.cpu_count() or 1
            # the bounded sample keeps the full scene (brute force over every primitive)
            rays, dt, kind, sample = run_cpu_step(api, ol, args.workload, source, depth, 0, threads)
            cpu_baseline = {"value": rays / dt / 1e6, "unit": "Mrays/s", "cores": threads, "kind": kind,
                            "sample": sample, "seconds": dt}
            cpu_reference = reference_as_shipped(args.workload)
        roofline = None
        if trace_ms > 0:
            sec = trace_ms * 1e-3
            l2_gbs = hit_rank * bytes_ray / sec / 1e9
            hbm_gbs = hit_rank * HBM_BYTES_RAY / sec / 1e9
            tflops = hit_rank * flops_ray / sec / 1e12
            per_launch = 1.0 / max(1, trace_launches)
            traffic_ray = ncu_traffic(args.workload)  # DRAM bytes per intersected ray (ncu)
            traffic = traffic_ray * hit_rank if traffic_ray else None  # per step
            traffic_launch = traffic * per_launch if traffic else None
            roofline = {
                # what bounds the kernel is neither HBM nor the tensor cores (north_star: not a dense contraction):
                # its algorithmic bytes are BVH-node and primitive fetches served by L1/L2, so the denominator is L2
                "bound": "l2", "kernel": "k_wf_trace", "achieved": l2_gbs, "peak": l2_peak, "unit": "GB/s",
                "frac": l2_gbs / l2_peak if l2_peak else None,
                "peak_source": "measured in this run: rtb_probe_l2_bandwidth, 32 MB L2-resident buffer, ld.global.cg.v4 from all SMs",
                "traffic": traffic_launch,
                "traffic_def": "DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) of the average launch: ncu's bytes per intersected ray over all k_wf_trace launches of this command (profiles/ncu_traffic.json, profiles/r2_launches_c3.csv) x the rays of the average launch",
                "bytes_per_launch": hit_rank * bytes_ray * per_launch, "avg_launch_ms": trace_ms * per_launch,
                "launches_per_step": trace_launches, "kernel_ms_per_step": trace_ms, "share_of_step": trace_share,
                "bytes_per_intersected_ray": bytes_ray, "intersected_rays_per_step": hit_rank,
                "achieved_def": "SURVEY 8(d) bytes per intersected ray (L*64 + 4*S: node + primitive fetches, L1/L2-served) x rays of one launch / average launch duration (CUDA events around every k_wf_trace launch)",
                "hbm": {"bound": "hbm", "achieved": hbm_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_gbs / hbm_peak,
                        "peak_source": hbm_src, "bytes_per_intersected_ray": HBM_BYTES_RAY,
                        "achieved_def": "HBM-algorithmic bytes only: each queue entry read once (64 B) + the hit record written (16 B)",
                        "traffic_over_algorithmic": (traffic / (hit_rank * HBM_BYTES_RAY)) if traffic else None},
                "fp32": {"bound": "fp32", "achieved": tflops, "peak": fp32_peak, "unit": "TFLOP/s", "frac": tflops / fp32_peak,
                         "flops_per_intersected_ray": flops_ray,
                         "peak_source": "measured in this run: rtb_probe_fp32_tflops (8 independent FFMA chains per thread, all SMs)",
                         "nominal": fp32_nominal, "nominal_def": f"148 SM x 128 lanes x 2 x {sm_mhz:.0f} MHz (median clock under load)"},
                "limiter": "issue slots and latency with 17 of 32 lanes active per instruction (profiles/r2_wf_trace_ncu.md): no memory level or pipe is saturated",
            }
        line = {
            "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong" if strong else "weak",
            "vs_baseline": None, "dtype": "f64 geometry / f32 colour", "data": "synthetic",
            "config": dict(workload_config(args.workload, total_spp, world, strong), integrator=args.integrator),
            "paths_per_s": paths_per_s, "rays_per_step": rays_step, "rays_per_path": rays_step / (W * H * total_spp),
            "node_visits_per_ray": node_visits_rank / hits_prof, "prim_tests_per_ray": prim_tests / max(1.0, hits_step),
            "e2e": {"value": e2e_value, "unit": "Mrays/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": int(h2d_bytes),
                    "d2h_bytes_per_step": int(W * H * 3), "ms_per_call": [round(x, 2) for x in e2e_calls],
                    "host_memory": "pageable (malloc'ed by the caller, like the reference's main.c); h2d_bytes_per_step counts the caller's "
                                   "buffers -- the library's staging threads narrow float-representable vertices to 60 B per triangle, "
                                   "so about half of the mesh bytes cross the link",
                    "pinned": e2e_pinned,
                    "api": "render_scene()/render_ex() of libraytracer_b200.so" if world == 1
                    else "rtb_render_multi(): sharded upload + all-gather + BVH build + render + ncclReduce + tonemap + D2H, all behind the C ABI"},
            "gpu_launches": launches_per_step * args.steps,
            "roofline": roofline,
            "clocks": clocks, "cpu_baseline": cpu_baseline, "cpu_reference_as_shipped": cpu_reference,
        }
        if comm is None:
            info = scene.info
            line["scene"] = {"objects": int(info.n_objects), "spheres": int(info.n_spheres), "triangles": int(info.n_triangles),
                             "bvh_nodes": int(info.n_bvh_nodes), "bvh_depth": int(info.bvh_depth), "big_prims": int(info.n_big_prims),
                             "device_bytes": int(info.device_bytes), "build_ms": float(info.build_ms)}
        print(json.dumps(line), flush=True)
    scene.close()
    if comm is not None:
        dist.barrier()
        comm.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--scale", type=float, default=1.0, help="scale spp (debug only; 1.0 = the named config)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong (default): the named job, samples split over the GPUs; weak: the named spp per GPU")
    ap.add_argument("--integrator", default="path", choices=["path", "whitted"],
                    help="path = trace_path (raytracer.c:482-554, the upstream default); whitted = cast_ray (raytracer.c:556-641)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's framebuffer and per-pixel sums as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to the GPU arm (--impl b200)")
        return main_reference(args)
    return main_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
