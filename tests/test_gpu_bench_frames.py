"""The frames bench.py times, at their full frame size and sample count, against the oracle.

Every other oracle comparison renders small frames with a few samples: one or two waves, a handful of planes.  The
benchmark's configurations cut their samples into up to 64 planes (rtb_plane_split) that run several waves in two
plane groups on two streams, with guided trace batches over queues of millions of rays.  Here each workload is
rendered as bench.py's timed step renders it -- scene, frame, depth and seed from bench.py, planes = 0, profile = 0,
rtb_render_accum into a torch buffer on a torch stream, then rtb_tonemap on the same stream -- and checked:

  sampled pixels  the oracle replays every sample of a seeded sample of pixels plus the four corners
                  (oracle_lib.pixel_paths): each sum within the float bound of its vertices (render_bound), each
                  8-bit value within one level of oracle_tonemap of the oracle's sums
  C1 in full      the whole frame against oracle_render_sum, path and Whitted integrators
  scheduler       the two-stream frame equals, bit for bit, the one-stream frame (profile = 1) and the megakernel
                  (kernel 4) at the plane count the library chose; ray, hit and path counts are equal.  This sees a
                  single dropped or doubled ray anywhere in the frame.
  tonemap, e2e    the framebuffer is oracle_tonemap of the GPU's own sums on every pixel, and so are sums at every
                  8-bit level edge at the workload's sample count; the reference-facing call bench.py times
                  (render_ex / render_scene) returns the same framebuffer

C4 runs 512 of its 4096 samples (17 planes of 31 samples, the last of 16; about 7 s per render on one B200 at a
1000 W power limit).
rtb_comm_render, the device-resident call bench.py times with several GPUs, is checked on two or more GPUs.
"""
import ctypes as C
import time

import numpy as np
import pytest

import bench
from test_gpu_wavefront_paths import _crafted_sums, materials, render_bound, slot_sums

pytestmark = pytest.mark.gpu

SPP = {"c1": 50, "c2": 256, "c3": 128, "c4": 512, "c5": 64}
# sampled pixels (plus the four corners), sized by the oracle's brute-force cost per ray: about 1.6 ms over C3's
# million triangles and 0.02 ms over 10k spheres with 8 threads
PIXELS = {"c1": 512, "c2": 192, "c3": 32, "c4": 192, "c5": 512}


def sample_pixels(W, H, n):
    """n pixels drawn with bench.dump_outputs' generator, and the four corners -> sorted flat indices"""
    idx = np.random.default_rng(bench.SEED).choice(W * H, n, replace=False)
    return np.unique(np.concatenate([idx, [0, W - 1, (H - 1) * W, H * W - 1]]))


def oracle_pixels(ol, abi, source, cam, W, H, pixels, spp, depth, planes, sample_offset=0):
    """the oracle on `pixels` -> (sums [n, 3] float64, float bound [n, 3], rays)"""
    log = ol.pixel_paths(source, cam, W, H, pixels, spp, max_depth=depth, seed=bench.SEED, sample_offset=sample_offset)
    slot = np.searchsorted(pixels, log["pixel"])
    flags, emission = materials(source)
    want = slot_sums(slot, len(pixels), log["contrib"])
    return want, render_bound(abi, log, flags, emission, slot, len(pixels), planes), int(log["rays"].sum())


def bench_step(api, sc, cam, desc, stream):
    """bench.py's timed step on one GPU: rtb_render_accum into a torch buffer, rtb_tonemap after it on the same
    torch stream, one synchronise at the end -> (sums [H, W, 3] f32, framebuffer [H, W, 3] u8)"""
    import torch
    W, H = desc.width, desc.height
    accum = torch.full((H, W, 3), float("nan"), dtype=torch.float32, device="cuda:0")  # every pixel must be written
    fb = torch.full((H, W, 3), 77, dtype=torch.uint8, device="cuda:0")
    stream.wait_stream(torch.cuda.current_stream())
    sc.render_accum(cam, desc, accum.data_ptr(), stream=stream.cuda_stream)
    api.tonemap(accum.data_ptr(), W, H, desc.sample_end - desc.sample_begin, fb.data_ptr(), device=0,
                stream=stream.cuda_stream)
    stream.synchronize()
    return accum.cpu().numpy(), fb.cpu().numpy()


def tonemap_level_edges(api, ol, spp, stream):
    """rtb_tonemap on the bench's stream at the workload's sample count, on sums within 4 ulps of every 8-bit level
    edge (k/255)^5 * spp and the special values of test_tonemap_byte_for_byte: a frame's own sums rarely sit that
    close to an edge, so the division by the sample count is pinned here"""
    import torch
    v = _crafted_sums(spp)
    d_acc = torch.from_numpy(v).to("cuda:0")
    d_fb = torch.empty(len(v), dtype=torch.uint8, device="cuda:0")
    stream.wait_stream(torch.cuda.current_stream())
    api.tonemap(d_acc.data_ptr(), len(v) // 3, 1, spp, d_fb.data_ptr(), device=0, stream=stream.cuda_stream)
    stream.synchronize()
    got = d_fb.cpu().numpy()
    want = ol.tonemap(v.astype(np.float64).reshape(1, -1, 3), spp).reshape(-1)
    bad = np.flatnonzero(got != want)
    assert len(bad) == 0, f"{spp} spp: {len(bad)} bytes differ, e.g. sums {v[bad[:5]]}: {got[bad[:5]]} vs {want[bad[:5]]}"


def render_sums(sc, cam, desc):
    """rtb_render_accum with counters (synchronous) -> (sums [H, W, 3] f32, counters)"""
    import torch
    accum = torch.full((desc.height, desc.width, 3), float("nan"), dtype=torch.float32, device="cuda:0")
    torch.cuda.synchronize()
    ctr = sc.render_accum(cam, desc, accum.data_ptr(), want_counters=True)
    return accum.cpu().numpy(), ctr


def e2e_frame(pkg, source, cam, W, H, spp, depth, integrator):
    """the reference-facing call as bench.py's e2e arm makes it: render_scene / render_ex with host buffers"""
    abi = pkg.abi
    _, host = pkg.load()
    opt = abi.Options()
    opt.width, opt.height, opt.samples = W, H, spp
    rp = abi.RenderParams()
    host.render_params_default(rp)
    rp.max_depth, rp.seed, rp.device, rp.integrator, rp.num_gpus = depth, bench.SEED, 0, integrator, 1
    fb = np.zeros((H, W, 3), dtype=np.uint8)
    if isinstance(source, abi.SceneHolder):
        host.render_scene(fb.ctypes.data, C.addressof(source.objects), source.n, C.byref(cam), C.byref(opt), C.byref(rp))
    else:
        host.render_ex(fb.ctypes.data, source.ctypes.data, len(source), C.byref(cam), C.byref(opt), C.byref(rp))
    return fb


def same_bits(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint32), np.ascontiguousarray(b).view(np.uint32))


@pytest.mark.parametrize("name", ["c1", "c2", "c3", "c4", "c5"])
def test_bench_frame_against_the_oracle(gpu_api, abi, pkg, ol, name):
    import torch
    t0 = time.perf_counter()
    W, H, _, depth, _ = bench.WORKLOADS[name]
    spp = SPP[name]
    source, *_ = bench.build_host_scene(gpu_api, name, W, H)
    cam = gpu_api.init_camera(W, H)
    desc = gpu_api.make_desc(W, H, 0, spp, max_depth=depth, seed=bench.SEED, integrator=0, profile=0)
    stream = torch.cuda.Stream(device=0)
    with gpu_api.Scene(source, device=0) as sc:
        acc, fb = bench_step(gpu_api, sc, cam, desc, stream)
        # the same desc with counters (bench.py's first pass), and the one-stream schedule of per-kernel timing
        acc0, c0 = render_sums(sc, cam, desc)
        acc1, c1 = render_sums(sc, cam, gpu_api.make_desc(W, H, 0, spp, max_depth=depth, seed=bench.SEED, profile=1))
    assert np.isfinite(acc).all() and (acc >= 0).all()
    assert same_bits(acc0, acc), "the step with counters differs from the asynchronous step"

    # the plane count the library chose: profile = 1 runs one plane group, one trace launch per wave and bounce
    waves = c1.trace_launches // (depth + 1)
    assert waves >= 1 and c1.trace_launches == waves * (depth + 1), c1.trace_launches
    planes = -(-spp // waves)
    assert gpu_api.wf_planes(gpu_api.make_desc(W, H, 0, spp, planes=planes)) == (planes, waves)

    # the scheduler: two streams == one stream == the megakernel at that plane count, bit for bit
    assert same_bits(acc1, acc), "the two-stream frame differs from the one-stream frame"
    with gpu_api.Scene(source, device=0, all_trees=True) as sc:
        acc_m, c_m = render_sums(sc, cam, gpu_api.make_desc(W, H, 0, spp, max_depth=depth, seed=bench.SEED, kernel=4,
                                                            planes=planes))
    assert same_bits(acc_m, acc), f"the wavefront frame differs from the megakernel's in {np.count_nonzero(acc_m != acc)} values"
    for k in ("rays", "rays_intersected", "paths"):
        assert getattr(c0, k) == getattr(c1, k) == getattr(c_m, k), (k, getattr(c0, k), getattr(c1, k), getattr(c_m, k))
    assert c0.paths == W * H * spp

    # tonemap on every pixel, and the e2e call
    assert np.array_equal(fb, ol.tonemap(acc.astype(np.float64), spp)), "framebuffer != oracle_tonemap(the GPU's sums)"
    tonemap_level_edges(gpu_api, ol, spp, stream)
    fb_e2e = e2e_frame(pkg, source, cam, W, H, spp, depth, 0)
    assert np.array_equal(fb_e2e, fb), f"the e2e frame differs in {np.count_nonzero(fb_e2e != fb)} bytes"
    t_gpu = time.perf_counter() - t0

    # the oracle on sampled pixels
    pixels = sample_pixels(W, H, PIXELS[name])
    want, bound, _ = oracle_pixels(ol, abi, source, cam, W, H, pixels, spp, depth, planes)
    got = acc.reshape(-1, 3)[pixels].astype(np.float64)
    err = np.abs(got - want)
    ratio = float(np.max(err / np.maximum(bound, 1e-300)))
    print(f"{name}: {W}x{H} {spp} spp, {planes} planes x {waves} waves, {c0.rays} rays; {len(pixels)} pixels: "
          f"largest error / bound = {ratio:.3f}; GPU side {t_gpu:.1f} s, oracle {time.perf_counter() - t0 - t_gpu:.1f} s")
    bad = np.argwhere(err > bound)
    assert len(bad) == 0, (f"{len(bad)} values beyond the float bound, e.g. pixel {pixels[bad[0][0]]}: "
                           f"{got[bad[0][0]]} vs {want[bad[0][0]]} (bound {bound[bad[0][0]]})")
    fb_want = ol.tonemap(want.reshape(1, -1, 3), spp).reshape(-1, 3)
    assert np.abs(fb.reshape(-1, 3)[pixels].astype(int) - fb_want.astype(int)).max() <= 1

    if name == "c1":
        # the whole frame (the bar of test_gpu_configs._compare)
        full, (rays, _) = ol.render_sum(source, cam, W, H, spp, max_depth=depth, seed=bench.SEED)
        assert c0.rays == rays
        np.testing.assert_allclose(acc, full, rtol=1e-3, atol=1e-4)


def test_c1_whitted_bench_frame(gpu_api, abi, pkg, ol):
    """bench.py --workload c1 --integrator whitted: the whole frame against the oracle's cast_ray (the bar of
    test_gpu_whitted), the framebuffer against oracle_tonemap of the GPU's sums, and the e2e call"""
    import torch
    W, H, spp, depth, _ = bench.WORKLOADS["c1"]
    source, *_ = bench.build_host_scene(gpu_api, "c1", W, H)
    cam = gpu_api.init_camera(W, H)
    desc = gpu_api.make_desc(W, H, 0, spp, max_depth=depth, seed=bench.SEED, integrator=1, profile=0)
    with gpu_api.Scene(source, device=0) as sc:
        acc, fb = bench_step(gpu_api, sc, cam, desc, torch.cuda.Stream(device=0))
        acc0, c0 = render_sums(sc, cam, desc)
    assert same_bits(acc0, acc)
    want, (rays, _) = ol.render_sum(source, cam, W, H, spp, max_depth=depth, seed=bench.SEED, integrator="whitted")
    assert c0.rays == rays and c0.paths == W * H * spp
    np.testing.assert_allclose(acc, want, rtol=2e-7, atol=1e-7)
    assert np.array_equal(fb, ol.tonemap(acc.astype(np.float64), spp))
    assert np.array_equal(e2e_frame(pkg, source, cam, W, H, spp, depth, 1), fb)


# ---- rtb_comm_render: the device-resident call of bench.py --gpus N ----------------------------------------------

@pytest.mark.parametrize("name,W,H,spp", [("c2", 480, 270, 8), ("c3", 480, 270, 4), ("c2", 480, 270, 1)],
                         ids=["c2-8spp", "c3-4spp", "c2-1spp-empty-root-share"])
def test_comm_render_frame(gpu_api, abi, ol, name, W, H, spp):
    """a local group over every visible GPU (at most 8), the framebuffer in a torch buffer on GPU 0: within one
    level of the one-GPU frame of the same desc and of the oracle's sums on sampled pixels; whole-job counters.
    At 1 spp rank 0, the root of the reduction, renders no sample."""
    n = min(gpu_api.device_count(), 8)
    if n < 2:
        pytest.skip("needs 2 GPUs")
    import torch
    depth = bench.WORKLOADS[name][3]
    source, *_ = bench.build_host_scene(gpu_api, name, W, H)
    cam = gpu_api.init_camera(W, H)
    desc = gpu_api.make_desc(W, H, 0, spp, max_depth=depth, seed=bench.SEED, profile=0)
    if spp == 1:
        assert gpu_api.shard_samples(0, spp, 0, n) == (0, 0)
    fb = torch.full((H, W, 3), 77, dtype=torch.uint8, device="cuda:0")
    torch.cuda.synchronize()
    with gpu_api.Comm.local(n) as comm:
        with comm.scene(source) as ms:
            ctr = ms.render(cam, desc, fb.data_ptr(), want_counters=True)
    for d in range(n):
        torch.cuda.synchronize(d)
    got = fb.cpu().numpy()
    with gpu_api.Scene(source, device=0) as sc:
        fb1, acc1, c1 = sc.render(cam, desc, want_accum=True)
    assert ctr.rays == c1.rays and ctr.paths == W * H * spp
    assert np.abs(got.astype(int) - fb1.astype(int)).max() <= 1
    pixels = sample_pixels(W, H, 64 if name == "c3" else 256)
    want, _, _ = oracle_pixels(ol, abi, source, cam, W, H, pixels, spp, depth, 1)
    fb_want = ol.tonemap(want.reshape(1, -1, 3), spp).reshape(-1, 3)
    assert np.abs(got.reshape(-1, 3)[pixels].astype(int) - fb_want.astype(int)).max() <= 1
