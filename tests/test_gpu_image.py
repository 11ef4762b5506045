"""GPU image-level parity: check 3 of the north star.

"The converged image must match the reference's own high-spp render at PSNR >= 40 dB, or at
the Monte Carlo noise floor, whichever is lower."  The reference renders are the committed
golden means (tests/golden/*_converged_*.npz: the UNMODIFIED reference's trace_path under
libc rand(), double precision, dielectrics SPLIT as upstream).  PSNR is taken on the 8-bit
frames after the reference's own transfer (mean, gamma 5.0, truncation; raytracer.c:215-220).

The reference renders are 32 768 spp (C1) and 16 384 spp (dielectric scene): 8 independent
srand() seeds, one single-threaded reference process each (tests/golden/make_converged.py).
The noise floor is measured, not assumed: the golden file also holds an independent
reference render (other seeds) at a quarter of the samples; PSNR(ref_quarter, ref_full) is
what the reference achieves against itself.  The GPU frame, rendered with 4x the full
sample count, must do at least as well as that (+1 dB: it carries less noise than the
quarter render) or reach 40 dB.
"""
import os

import numpy as np
import pytest

from conftest import psnr_u8, random_rays_in_room

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _gate(gpu_api, ol, objs, W, H, gold_file, gpu_spp, max_depth=5):
    g = np.load(os.path.join(GOLD, gold_file))
    ref_full = g["mean"].astype(np.float64)
    ref_quarter = g["mean_quarter"].astype(np.float64)
    cam = gpu_api.init_camera(W, H)
    with gpu_api.Scene(objs) as sc:
        _, acc, ctr = sc.render(cam, gpu_api.make_desc(W, H, 0, gpu_spp, max_depth=max_depth), want_accum=True)
    gpu_mean = acc.astype(np.float64) / gpu_spp
    fb_ref, fb_q, fb_gpu = ol.tonemap(ref_full, 1), ol.tonemap(ref_quarter, 1), ol.tonemap(gpu_mean, 1)
    floor = psnr_u8(fb_q, fb_ref)
    got = psnr_u8(fb_gpu, fb_ref)
    bias = (gpu_mean.mean() - ref_full.mean()) / ref_full.mean()
    print(f"{gold_file}: PSNR(gpu {gpu_spp} spp, ref {int(g['spp'][0])} spp) = {got:.2f} dB; reference noise floor "
          f"PSNR(ref {int(g['spp'][1])} spp, ref {int(g['spp'][0])} spp) = {floor:.2f} dB; mean bias {bias:+.4f}")
    return got, floor, bias


def test_psnr_default_scene(gpu_api, ol):
    W, H = 96, 54
    objs = gpu_api.scene_default(W, H)
    got, floor, bias = _gate(gpu_api, ol, objs, W, H, "c1_converged_96x54.npz", gpu_spp=131072)
    assert got >= min(40.0, floor + 1.0), (got, floor)
    assert abs(bias) < 0.01, "frame-average radiance must agree to 1% (unbiased estimator)"


def test_psnr_dielectric_scene_stochastic_vs_split(gpu_api, ol):
    """the GPU picks ONE child at a dielectric vertex, the reference traces both: same
    expectation, so the converged frames agree at the noise floor"""
    W, H = 64, 36
    objs = gpu_api.scene_sphere_field(60, W, H, mix=(0.3, 0.4, 0.2))
    got, floor, bias = _gate(gpu_api, ol, objs, W, H, "dielectric_converged_64x36.npz", gpu_spp=65536)
    assert got >= min(40.0, floor + 1.0), (got, floor)
    assert abs(bias) < 0.01


def test_golden_hits_on_device(gpu_api):
    """nearest hit against the reference's own intersect() output (golden, bit-level)"""
    g = np.load(os.path.join(GOLD, "c1_hits.npz"))
    objs = gpu_api.scene_default(320, 180)
    rays = random_rays_in_room(np.random.default_rng(105), 3000)
    with gpu_api.Scene(objs, all_trees=True) as sc:
        for mode in (1, 2, 3, 4, 5, 0):  # BVH, BVH + FP32 pre-test, while-while, BVH4, compressed BVH4, brute force
            got = sc.trace_rays(rays, use_bvh=mode)
            assert np.array_equal(got["ids"], g["ids"]), mode
            # same double arithmetic without contraction on both sides: bit-identical
            assert np.array_equal(got["points"], g["points"]), mode
            assert np.array_equal(got["normals"], g["normals"]), mode
            np.testing.assert_allclose(got["uvs"], g["uvs"], rtol=0, atol=1e-15)  # atan2: libm vs CUDA


def _checkered_scene(gpu_api, abi, W, H):
    """scene_mesh_room with checkered surfaces of every material (mesh, walls, mirror and glass balls) and a mesh
    whose texture coordinates are genuine doubles, unrelated to position: the scene keeps them as doubles, and a
    texture coordinate read from the wrong triangle or rounded to float changes the checker at M = 100 000"""
    verts = gpu_api.heightfield_mesh(40, 20 * W / H * 0.98)
    verts["tex"] = np.random.default_rng(8).uniform(0.0, 1.0, (len(verts), 2))
    holder = gpu_api.mesh_room(verts, W, H)
    for k in (1, 2, 6, 11, 12):
        holder.objects[k].material.flags |= abi.M_CHECKERED
    return holder


@pytest.mark.parametrize("kernel,scene", [(k, "field") for k in range(1, 7)] + [(k, "checkered") for k in range(1, 7)],
                         ids=[str(k) for k in range(1, 7)] + [f"{k}-checkered" for k in range(1, 7)])
def test_kernel_variants_agree(gpu_api, abi, kernel, scene):
    """megakernel, warp-scheduled state machine, the FP32 pre-test variants and the wavefront
    kernels compute the same per-pixel sums (same Philox streams, same exact tests, same
    order of additions) -- on a sphere field and on a scene with checkered surfaces"""
    W, H, SPP = 96, 54, 8
    if scene == "field":
        objs = gpu_api.scene_sphere_field(400, W, H, mix=(0.3, 0.3, 0.3))
    else:
        objs = _checkered_scene(gpu_api, abi, W, H)
    cam = gpu_api.init_camera(W, H)
    with gpu_api.Scene(objs, all_trees=True) as sc:
        info = sc.info
        _, base, c0 = sc.render(cam, gpu_api.make_desc(W, H, 0, SPP, max_depth=8, kernel=0), want_accum=True)
        _, acc, c1 = sc.render(cam, gpu_api.make_desc(W, H, 0, SPP, max_depth=8, kernel=kernel), want_accum=True)
    assert np.array_equal(acc, base)
    assert c0.rays == c1.rays and c0.paths == c1.paths
    assert info.double_texcoords == (scene == "checkered")


@pytest.mark.parametrize("spp,planes,checkered", [(7, 3, False), (6, 1, False), (5, 5, False), (9, 2, False),
                                                  (7, 3, True), (5, 5, True)],
                         ids=["7-3", "6-1", "5-5", "9-2", "7-3-checkered", "5-5-checkered"])
def test_wavefront_equals_megakernel_on_a_mesh(gpu_api, abi, spp, planes, checkered):
    """wavefront (ray queues + persistent trace kernel) vs megakernel on a mesh + spheres scene,
    including ragged plane/wave combinations: bit-identical sums and equal counters; also with
    checkered surfaces and double texture coordinates"""
    W, H = 80, 46  # not a multiple of the 8x4 tile
    if checkered:
        holder = _checkered_scene(gpu_api, abi, W, H)
    else:
        verts = gpu_api.heightfield_mesh(40, 20 * W / H * 0.98)
        holder = gpu_api.mesh_room(verts, W, H)
    cam = gpu_api.init_camera(W, H)
    with gpu_api.Scene(holder, all_trees=True) as sc:
        _, base, c0 = sc.render(cam, gpu_api.make_desc(W, H, 3, 3 + spp, max_depth=6, kernel=4, planes=planes), want_accum=True)
        _, acc, c1 = sc.render(cam, gpu_api.make_desc(W, H, 3, 3 + spp, max_depth=6, kernel=6, planes=planes), want_accum=True)
        _, acc2, c2 = sc.render(cam, gpu_api.make_desc(W, H, 3, 3 + spp, max_depth=6, kernel=6, planes=planes, tune=(2 << 16) | (16 << 8) | 1), want_accum=True)  # BVH2 walk, refill at 1 idle lane
        wide = (10 << 16) | (16 << 8)  # BVH4 walk
        _, acc3, c3 = sc.render(cam, gpu_api.make_desc(W, H, 3, 3 + spp, max_depth=6, kernel=6, planes=planes, tune=wide), want_accum=True)
        wideq = (22 << 16) | (16 << 8)  # compressed BVH4 walk
        _, acc5, c5 = sc.render(cam, gpu_api.make_desc(W, H, 3, 3 + spp, max_depth=6, kernel=6, planes=planes, tune=wideq), want_accum=True)
        assert np.array_equal(acc5, base) and c5.rays == c0.rays
        # round 2: byte conversions split between the conversion and ALU/FMA pipes (32, 64), two-entry pops (128)
        for v in (54, 86, 150, 182, 214, 1024):
            _, accv, cv = sc.render(cam, gpu_api.make_desc(W, H, 3, 3 + spp, max_depth=6, kernel=6, planes=planes, tune=(v << 16) | (16 << 8)), want_accum=True)
            assert np.array_equal(accv, base) and cv.rays == c0.rays and cv.prim_tests == c5.prim_tests, v
        _, acc4, c4 = sc.render(cam, gpu_api.make_desc(W, H, 3, 3 + spp, max_depth=6, kernel=6, planes=planes, tune2=3), want_accum=True)
    assert np.array_equal(acc, base) and np.array_equal(acc2, base)
    assert np.array_equal(acc3, base) and c3.rays == c0.rays and c3.node_visits < c0.node_visits
    assert np.array_equal(acc4, base) and c4.rays == c0.rays  # sorted queues: same sums
    assert c0.rays == c1.rays == c2.rays and c0.paths == c1.paths == W * H * spp
    assert c0.rays_intersected == c1.rays_intersected
    assert c2.node_visits == c0.node_visits and c2.prim_tests == c0.prim_tests  # same BVH2, same order


def test_guided_ray_batches_change_nothing_but_the_schedule(gpu_api, monkeypatch):
    """k_wf_trace sizes its ray batches by the rays left in the queue (guided self-scheduling; only launches with
    more than 32 rays per warp and batch, hence a 720p frame): sums, ray counts and primitive-test counts equal
    those of fixed batches, bit for bit"""
    W, H = 1280, 720
    holder = gpu_api.mesh_room(gpu_api.heightfield_mesh(96, 20 * W / H * 0.98), W, H)
    cam = gpu_api.init_camera(W, H)
    desc = gpu_api.make_desc(W, H, 0, 2, max_depth=5, profile=1)
    out = {}
    with gpu_api.Scene(holder) as sc:
        for g in ("0", "1", "34"):  # fixed; the default rule; rays left / (2 warps) with a 2 048 cap
            monkeypatch.setenv("RTB_WF_GUIDED", g)
            _, acc, ctr = sc.render(cam, desc, want_accum=True)
            out[g] = (acc.copy(), ctr.rays, ctr.prim_tests, ctr.node_visits, ctr.rays_intersected)
    monkeypatch.delenv("RTB_WF_GUIDED")
    for g in ("1", "34"):
        assert np.array_equal(out[g][0], out["0"][0]), g
        assert out[g][1:] == out["0"][1:], g


def test_counters_without_profiling(gpu_api):
    """rtb_render_desc.profile = 0 (what the drop-in render() uses): same sums, same ray and
    primitive-test counts, no node-visit count, no per-kernel times"""
    W, H = 64, 36
    objs = gpu_api.scene_sphere_field(200, W, H, mix=(0.3, 0.3, 0.3))
    cam = gpu_api.init_camera(W, H)
    with gpu_api.Scene(objs) as sc:
        _, a1, c1 = sc.render(cam, gpu_api.make_desc(W, H, 0, 4, max_depth=6, profile=1), want_accum=True)
        _, a0, c0 = sc.render(cam, gpu_api.make_desc(W, H, 0, 4, max_depth=6, profile=0), want_accum=True)
    assert np.array_equal(a0, a1)
    assert c0.rays == c1.rays and c0.prim_tests == c1.prim_tests and c0.paths == c1.paths
    assert c1.node_visits > 0 and c1.trace_ms > 0 and c1.trace_launches == 7
    assert c0.node_visits == 0 and c0.trace_ms == 0


def test_workspace_is_reused_across_scenes(gpu_api):
    """render() creates and destroys a scene per call: the ray-queue workspace is parked per
    device and taken over by the next scene (no growth of used device memory)"""
    import torch
    W, H = 128, 72
    objs = gpu_api.scene_default(W, H)
    cam = gpu_api.init_camera(W, H)
    used = []
    for _ in range(4):
        with gpu_api.Scene(objs) as sc:
            sc.render(cam, gpu_api.make_desc(W, H, 0, 8))
        torch.cuda.synchronize()
        free, total = torch.cuda.mem_get_info()
        used.append(total - free)
    assert max(used[1:]) - min(used[1:]) < (64 << 20), used


def test_wave_shrinks_when_memory_is_short(gpu_api):
    """the ray queues want up to 23.4 GB; with little free memory the render must still succeed
    (smaller waves), and give the same image up to float summation order"""
    import torch
    W, H, SPP = 1920, 1080, 32
    objs = gpu_api.scene_default(W, H)
    cam = gpu_api.init_camera(W, H)
    with gpu_api.Scene(objs) as sc:
        _, ref, c0 = sc.render(cam, gpu_api.make_desc(W, H, 0, SPP), want_accum=True)
    gpu_api.release_workspace(0)
    torch.cuda.synchronize()
    free, total = torch.cuda.mem_get_info()
    hog = torch.empty(max(0, free - (5 << 30)), dtype=torch.uint8, device="cuda")  # leave ~5 GB
    try:
        with gpu_api.Scene(objs) as sc:
            _, acc, c1 = sc.render(cam, gpu_api.make_desc(W, H, 0, SPP), want_accum=True)
    finally:
        del hog
        torch.cuda.empty_cache()
        gpu_api.release_workspace(0)
    assert c1.rays == c0.rays and c1.paths == c0.paths
    np.testing.assert_allclose(acc, ref, rtol=1e-5, atol=1e-5)


def test_wavefront_depth_zero_and_empty(gpu_api):
    """max_depth 0 (one vertex per path) and an empty sample range"""
    W, H = 64, 36
    objs = gpu_api.scene_default(W, H)
    cam = gpu_api.init_camera(W, H)
    with gpu_api.Scene(objs, all_trees=True) as sc:
        _, a0, c0 = sc.render(cam, gpu_api.make_desc(W, H, 0, 4, max_depth=0, kernel=4), want_accum=True)
        _, a1, c1 = sc.render(cam, gpu_api.make_desc(W, H, 0, 4, max_depth=0, kernel=6), want_accum=True)
        _, e, ce = sc.render(cam, gpu_api.make_desc(W, H, 5, 5, kernel=6), want_accum=True)
    assert np.array_equal(a0, a1) and c0.rays == c1.rays
    assert not e.any() and ce.rays == 0


def test_full_size_properties(gpu_api):
    """size-independent properties at BASELINE.json's full frame size (1080p, mesh scene):
    sums are finite and non-negative, sample sharding is additive, rays/path in range"""
    W, H = 1920, 1080
    verts = gpu_api.heightfield_mesh(708, 20 * W / H * 0.98)
    holder = gpu_api.mesh_room(verts, W, H)
    cam = gpu_api.init_camera(W, H)
    with gpu_api.Scene(holder, all_trees=True) as sc:
        info = sc.info
        assert info.n_triangles == 1002528 and info.n_bvh_prims + info.n_big_prims == 1002528 + 12
        _, a, ca = sc.render(cam, gpu_api.make_desc(W, H, 0, 2), want_accum=True)
        _, b, cb = sc.render(cam, gpu_api.make_desc(W, H, 2, 4), want_accum=True)
        _, ab, cab = sc.render(cam, gpu_api.make_desc(W, H, 0, 4), want_accum=True)
        # 4k random rays: BVH == brute force over 1M triangles
        rays = random_rays_in_room(np.random.default_rng(9), 4096)
        bvh, brute = sc.trace_rays(rays, use_bvh=1), sc.trace_rays(rays, use_bvh=0)
        bvh4 = sc.trace_rays(rays, use_bvh=4)
        bvh4q = sc.trace_rays(rays, use_bvh=5)
    # (a path that Russian roulette stops on a non-emissive surface contributes exactly 0)
    assert np.isfinite(ab).all() and (ab >= 0).all() and (ab.reshape(-1, 3).sum(axis=1) > 0).mean() > 0.3
    np.testing.assert_allclose(a + b, ab, rtol=1e-5, atol=1e-6)
    assert ca.rays + cb.rays == cab.rays and cab.paths == W * H * 4
    assert 2.0 < cab.rays / cab.paths < 7.0
    for k in ("ids", "prims", "t", "points", "normals"):
        assert np.array_equal(bvh[k], brute[k]), k
        assert np.array_equal(bvh4[k], brute[k]), k
        assert np.array_equal(bvh4q[k], brute[k]), k
