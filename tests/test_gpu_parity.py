"""GPU parity tests: the CUDA path, called through the C ABI, against the oracle.

The three-way check BASELINE.json asks for:
  1. primary-ray hit object ids bit-exact (shared jitter: both sides derive it from the
     same Philox words);
  2. 1-bounce normals and depth within 1e-4 relative (depth = |point - origin|, not the
     reference's Hit.t, quirk Q9);
  3. converged image PSNR against the reference's own high-spp render (test_gpu_image.py).
Tolerances are written next to each assert.  Integer/index results are exact.
"""
import os

import numpy as np
import pytest

from conftest import random_rays_in_room

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

REL_1E4 = 1e-4  # north_star: "1-bounce normals and depth must match within 1e-4 relative"


def _assert_hits_equal(got, want, what, n_obj=None):
    assert np.array_equal(got["ids"], want["ids"]), f"{what}: hit ids differ at {np.flatnonzero(got['ids'] != want['ids'])[:10]}"
    hit = want["ids"] >= 0
    if "prims" in want and "prims" in got:
        assert np.array_equal(got["prims"][hit], want["prims"][hit]), f"{what}: primitive (tie-break) ids differ"
    # exact double tests on both sides: expect ~1e-15, demand 1e-9 (far inside the 1e-4 budget)
    np.testing.assert_allclose(got["points"][hit], want["points"][hit], rtol=1e-9, atol=1e-9, err_msg=what)
    np.testing.assert_allclose(got["normals"][hit], want["normals"][hit], rtol=1e-9, atol=1e-9, err_msg=what)
    if "t" in want and "t" in got:
        np.testing.assert_allclose(got["t"][hit], want["t"][hit], rtol=1e-12, atol=0, err_msg=what)


def test_philox_kat_on_device(gpu_api):
    """Random123 known-answer vectors for philox4x32-10 (kat_vectors)"""
    ctr = np.array([[0, 0, 0, 0], [0xFFFFFFFF] * 4, [0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344]], dtype=np.uint32)
    key = np.array([[0, 0], [0xFFFFFFFF] * 2, [0xA4093822, 0x299F31D0]], dtype=np.uint32)
    want = np.array([[0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8],
                     [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD],
                     [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]], dtype=np.uint32)
    assert np.array_equal(gpu_api.philox(ctr, key), want)


def test_philox_matches_oracle_bulk(gpu_api, ol):
    rng = np.random.default_rng(7)
    ctr = rng.integers(0, 2 ** 32, size=(512, 4), dtype=np.uint64).astype(np.uint32)
    key = rng.integers(0, 2 ** 32, size=(512, 2), dtype=np.uint64).astype(np.uint32)
    assert np.array_equal(gpu_api.philox(ctr, key), ol.philox(ctr, key))


def test_default_scene_structure(gpu_api):
    objs = gpu_api.scene_default(320, 180)
    with gpu_api.Scene(objs) as sc:
        info = sc.info
        assert info.n_objects == 38 and info.n_spheres == 38 and info.n_triangles == 0
        assert info.n_big_prims == 6, "the six r=10000 walls go to the brute list"
        assert info.n_bvh_prims == 32


@pytest.mark.parametrize("use_bvh", [True, False])
def test_nearest_hit_default_scene(gpu_api, ol, use_bvh):
    """intersect() (raytracer.c:393-464) on the reference scene: camera rays through pixel
    centres plus random rays from inside the room"""
    W, H = 320, 180
    objs = gpu_api.scene_default(W, H)
    cam = gpu_api.init_camera(W, H)
    ys, xs = np.mgrid[0:H:3, 0:W:3]
    rays = np.stack([ol.camera_ray(cam, (x + 0.5) / (W - 1.0), (y + 0.5) / (H - 1.0))
                     for x, y in zip(xs.ravel(), ys.ravel())])
    rays = np.concatenate([rays, random_rays_in_room(np.random.default_rng(1), 20000)])
    want = ol.intersect_rays(objs, rays)
    with gpu_api.Scene(objs) as sc:
        got = sc.trace_rays(rays, use_bvh=use_bvh)
    _assert_hits_equal(got, want, f"default scene use_bvh={use_bvh}")
    assert (want["ids"] >= 0).all(), "the room is closed: every ray hits something"


def test_nearest_hit_vs_reference_binary(gpu_api, ref_or_skip):
    """same check directly against the unmodified reference's static intersect()"""
    ol = ref_or_skip
    W, H = 320, 180
    objs = gpu_api.scene_default(W, H)
    rays = random_rays_in_room(np.random.default_rng(2), 20000)
    want = ol.ref_intersect_rays(objs, rays)
    with gpu_api.Scene(objs) as sc:
        got = sc.trace_rays(rays)
    assert np.array_equal(got["ids"], want["ids"])
    np.testing.assert_allclose(got["points"], want["points"], rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(got["normals"], want["normals"], rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(got["uvs"], want["uvs"], rtol=1e-9, atol=1e-9)


def test_nearest_hit_vs_reference_golden(gpu_api):
    """the same check against the unmodified reference's intersect() outputs stored in
    tests/golden/c1_hits.npz (make_golden.py): runs without the reference build"""
    g = np.load(os.path.join(GOLD, "c1_hits.npz"))
    rays = random_rays_in_room(np.random.default_rng(105), 3000)
    with gpu_api.Scene(gpu_api.scene_default(320, 180)) as sc:
        got = sc.trace_rays(rays)
    assert np.array_equal(got["ids"], g["ids"])
    hit = g["ids"] >= 0
    assert hit.sum() > 1000
    for k in ("points", "normals", "uvs"):
        np.testing.assert_allclose(got[k][hit], g[k][hit], rtol=1e-9, atol=1e-9, err_msg=k)


def test_bvh_equals_bruteforce_10k_spheres(gpu_api, ol):
    """north_star (3): the BVH returns the same nearest hit as the brute-force loop"""
    W, H = 192, 108
    objs = gpu_api.scene_sphere_field(10000, W, H)
    rays = random_rays_in_room(np.random.default_rng(3), 200000)
    with gpu_api.Scene(objs) as sc:
        info = sc.info
        assert info.n_big_prims == 6 and info.n_bvh_prims == len(objs) - 6
        bvh = sc.trace_rays(rays, use_bvh=True)
        brute = sc.trace_rays(rays, use_bvh=False)
    for k in ("ids", "prims", "t", "points", "normals"):
        assert np.array_equal(bvh[k], brute[k]), f"BVH and brute force disagree on {k}"
    # and a slice of it against the CPU oracle
    want = ol.intersect_rays(objs, rays[:3000])
    _assert_hits_equal({k: v[:3000] for k, v in bvh.items()}, want, "10k spheres")


def test_tie_break_lowest_index_wins(gpu_api, ol):
    """strict `<` in loop order (raytracer.c:404): duplicates of a sphere are hit at equal t,
    the lowest object index must win -- inside the BVH and in the big list"""
    rng = np.random.default_rng(4)
    base = gpu_api.scene_sphere_field(500, 192, 108)
    dup = np.concatenate([base, base[6:206][::-1], base[:6]])  # reversed duplicates + duplicate walls
    rays = random_rays_in_room(rng, 50000)
    want = ol.intersect_rays(dup, rays)
    with gpu_api.Scene(dup) as sc:
        got = sc.trace_rays(rays)
        brute = sc.trace_rays(rays, use_bvh=False)
    assert want["ids"].max() < len(base), "a duplicate (higher index) won a tie in the oracle?"
    _assert_hits_equal(got, want, "ties (bvh)")
    _assert_hits_equal(brute, want, "ties (brute)")


def test_mesh_nearest_hit(gpu_api, ol):
    """Moeller-Trumbore + flat normal (raytracer.c:120-174, :42-45) on a height-field mesh
    mixed with spheres; object id = the mesh's object index"""
    W, H = 192, 108
    verts = gpu_api.heightfield_mesh(24, 20 * W / H * 0.98)
    holder = gpu_api.mesh_room(verts, W, H)
    rng = np.random.default_rng(5)
    rays = random_rays_in_room(rng, 6000)
    want = ol.intersect_rays(holder, rays)
    with gpu_api.Scene(holder) as sc:
        info = sc.info
        assert info.n_triangles == 2 * 24 * 24
        got = sc.trace_rays(rays)
        brute = sc.trace_rays(rays, use_bvh=False)
    _assert_hits_equal(got, want, "mesh room (bvh)")
    _assert_hits_equal(brute, want, "mesh room (brute)")
    assert (want["ids"] == 6).sum() > 500, "the mesh (object 6) must be hit by a good share of rays"
    # interpolated texcoords of the nearest triangle
    m = want["ids"] == 6
    np.testing.assert_allclose(got["uvs"][m], want["uvs"][m], rtol=1e-9, atol=1e-12)


def test_primary_ids_and_one_bounce(gpu_api, ol):
    """checks 1 and 2 of the north star on the reference scene at its default resolution"""
    W, H = 320, 180
    objs = gpu_api.scene_default(W, H)
    cam = gpu_api.init_camera(W, H)
    desc = gpu_api.make_desc(W, H, 0, 1, max_depth=5)
    with gpu_api.Scene(objs) as sc:
        for sample in (0, 3):
            got = sc.path_records(cam, desc, sample, n_vertices=2)
            want = ol.path_records(objs, cam, W, H, sample, n_vertices=2)
            # 1. primary-ray hit ids: bit-exact
            assert np.array_equal(got["ids"][:, 0], want["ids"][:, 0])
            # 2. 1-bounce ids, normals, depth
            assert np.array_equal(got["ids"][:, 1], want["ids"][:, 1])
            for v in (0, 1):
                hit = want["ids"][:, v] >= 0
                np.testing.assert_allclose(got["normals"][hit, v], want["normals"][hit, v], rtol=REL_1E4, atol=REL_1E4)
                np.testing.assert_allclose(got["dists"][hit, v], want["dists"][hit, v], rtol=REL_1E4)
                # in fact both sides run the same double arithmetic:
                np.testing.assert_allclose(got["dists"][hit, v], want["dists"][hit, v], rtol=1e-11)
            # per-sample radiance: FP32 colour arithmetic vs double
            np.testing.assert_allclose(got["radiance"], want["radiance"], rtol=2e-5, atol=1e-6)


def test_primary_ids_vs_reference_camera(gpu_api, ref_or_skip):
    """primary hit ids against the UNMODIFIED reference: its get_camera_ray fed with the
    jitter the GPU derives from Philox, then its intersect()"""
    ol = ref_or_skip
    W, H = 320, 180
    objs = gpu_api.scene_default(W, H)
    cam = gpu_api.init_camera(W, H)
    desc = gpu_api.make_desc(W, H, 0, 1)
    rays = np.zeros((W * H, 6))
    for pix in range(0, W * H, 7):
        j = ol.keyed_jitter(desc.seed, pix, 0)
        x, y = pix % W, pix // W
        rays[pix] = ol.ref_camera_ray(cam, (x + j[0]) / (W - 1.0), (y + j[1]) / (H - 1.0))
    sel = np.arange(0, W * H, 7)
    want = ol.ref_intersect_rays(objs, rays[sel])
    with gpu_api.Scene(objs) as sc:
        got = sc.path_records(cam, desc, 0, n_vertices=1)
    assert np.array_equal(got["ids"][sel, 0], want["ids"])
    np.testing.assert_allclose(got["normals"][sel, 0], want["normals"], rtol=1e-9, atol=1e-9)


@pytest.mark.parametrize("max_depth", [0, 1, 5, 8])
def test_accumulation_matches_oracle(gpu_api, ol, max_depth):
    """the whole integrator: per-pixel sums over 4 samples, same Philox streams on both
    sides.  Tolerance 1e-3 relative (+1e-4 absolute): FP32 colour math and FP32 summation
    against the oracle's double."""
    W, H, SPP = 96, 54, 4
    objs = gpu_api.scene_default(W, H)
    cam = gpu_api.init_camera(W, H)
    desc = gpu_api.make_desc(W, H, 0, SPP, max_depth=max_depth)
    with gpu_api.Scene(objs) as sc:
        fb, acc, ctr = sc.render(cam, desc, want_accum=True)
    want, (rays, tests) = ol.render_sum(objs, cam, W, H, SPP, rng="philox", dielectric="stochastic", max_depth=max_depth)
    np.testing.assert_allclose(acc, want, rtol=1e-3, atol=1e-4)
    assert ctr.rays == rays, "ray_count (trace_path invocations) must match the oracle exactly"
    assert ctr.paths == W * H * SPP
    # 8-bit output: identical up to truncation boundaries
    want_fb = ol.tonemap(want, SPP)
    assert np.abs(fb.astype(int) - want_fb.astype(int)).max() <= 1


def test_dielectric_and_mirror_scene(gpu_api, ol):
    """C4/C5-style material mix (40% refraction, 40% reflection), deeper paths"""
    W, H, SPP = 64, 36, 4
    objs = gpu_api.scene_sphere_field(300, W, H, mix=(0.2, 0.4, 0.4))
    cam = gpu_api.init_camera(W, H)
    desc = gpu_api.make_desc(W, H, 0, SPP, max_depth=16)
    with gpu_api.Scene(objs) as sc:
        fb, acc, ctr = sc.render(cam, desc, want_accum=True)
    want, (rays, _) = ol.render_sum(objs, cam, W, H, SPP, rng="philox", dielectric="stochastic", max_depth=16)
    np.testing.assert_allclose(acc, want, rtol=2e-3, atol=2e-4)
    assert ctr.rays == rays


def test_mesh_scene_accumulation(gpu_api, ol):
    W, H, SPP = 48, 27, 2
    verts = gpu_api.heightfield_mesh(16, 20 * W / H * 0.98)
    holder = gpu_api.mesh_room(verts, W, H)
    cam = gpu_api.init_camera(W, H)
    desc = gpu_api.make_desc(W, H, 0, SPP, max_depth=5)
    with gpu_api.Scene(holder) as sc:
        fb, acc, ctr = sc.render(cam, desc, want_accum=True)
    want, (rays, _) = ol.render_sum(holder, cam, W, H, SPP, rng="philox", dielectric="stochastic", max_depth=5)
    np.testing.assert_allclose(acc, want, rtol=1e-3, atol=1e-4)
    assert ctr.rays == rays


def test_sample_sharding_is_the_same_estimator(gpu_api):
    """multi-GPU contract (SURVEY 8e): samples [0,8) == samples [0,4) + [4,8)"""
    W, H = 64, 36
    objs = gpu_api.scene_default(W, H)
    cam = gpu_api.init_camera(W, H)
    with gpu_api.Scene(objs) as sc:
        _, whole, c0 = sc.render(cam, gpu_api.make_desc(W, H, 0, 8), want_accum=True)
        _, a, c1 = sc.render(cam, gpu_api.make_desc(W, H, 0, 4), want_accum=True)
        _, b, c2 = sc.render(cam, gpu_api.make_desc(W, H, 4, 8), want_accum=True)
    np.testing.assert_allclose(a + b, whole, rtol=1e-5, atol=1e-6)
    assert c1.rays + c2.rays == c0.rays


def test_render_is_deterministic(gpu_api):
    W, H = 64, 36
    objs = gpu_api.scene_default(W, H)
    cam = gpu_api.init_camera(W, H)
    desc = gpu_api.make_desc(W, H, 0, 6)
    with gpu_api.Scene(objs) as sc:
        fb1, acc1, _ = sc.render(cam, desc, want_accum=True)
        fb2, acc2, _ = sc.render(cam, desc, want_accum=True)
    assert np.array_equal(acc1, acc2) and np.array_equal(fb1, fb2)


def test_edge_cases(gpu_api, abi):
    W, H = 16, 8
    cam = gpu_api.init_camera(W, H)
    # empty scene: every path misses -> BACKGROUND (10/255) per sample (raytracer.c:487-490)
    empty = np.zeros(0, dtype=abi.OBJECT_DTYPE)
    with gpu_api.Scene(empty) as sc:
        fb, acc, ctr = sc.render(cam, gpu_api.make_desc(W, H, 0, 3), want_accum=True)
        np.testing.assert_allclose(acc, 3 * 10.0 / 255.0, rtol=1e-6)
        assert ctr.rays == W * H * 3
        assert (fb == int(255 * (10 / 255.0) ** 0.2)).all()
        # zero samples: all-zero sums
        _, acc0, _ = sc.render(cam, gpu_api.make_desc(W, H, 0, 0), want_accum=True)
        assert (acc0 == 0).all()
        # width/height of 1 divide by zero upstream (quirk Q11): rejected
        with pytest.raises(gpu_api.RtbError):
            sc.render(cam, gpu_api.make_desc(1, H, 0, 1))
    # a single sphere, a single emissive pixel column
    one = np.zeros(1, dtype=abi.OBJECT_DTYPE)
    one["flags"], one["radius"], one["center"] = abi.M_DEFAULT, 20.0, (0, 0, 0)
    one["color"], one["emission"] = (0, 0, 0), (1, 2, 3)
    with gpu_api.Scene(one) as sc:
        _, acc, _ = sc.render(cam, gpu_api.make_desc(W, H, 0, 1), want_accum=True)
        centre = acc[H // 2, W // 2]
        np.testing.assert_allclose(centre, (1, 2, 3), rtol=1e-6)  # colour 0 -> RR always stops: emission only
        np.testing.assert_allclose(acc[0, 0], 10.0 / 255.0, rtol=1e-6)


def test_dropin_render_entry(gpu_api):
    """the reference signature render(fb, Object*, n, Camera*, Options*) through the C99 host
    library gives the same frame as the C ABI with default parameters"""
    W, H, SPP = 64, 36, 5
    objs = gpu_api.scene_default(W, H)
    cam = gpu_api.init_camera(W, H)
    fb_host = gpu_api.render(objs, cam, W, H, SPP)
    with gpu_api.Scene(objs) as sc:
        fb_abi, _, _ = sc.render(cam, gpu_api.make_desc(W, H, 0, SPP, max_depth=5))
    assert np.array_equal(fb_host, fb_abi)


def test_deep_unbalanced_tree(gpu_api, abi):
    """spheres spaced geometrically along a line give a chain-like LBVH; if it is too deep for the
    BVH4 walk's stack the scene falls back to the BVH2 walk -- either way the nearest hit equals
    the brute-force loop and the wavefront sums equal the megakernel's"""
    n = 58
    objs = np.zeros(n, dtype=abi.OBJECT_DTYPE)
    for k in range(n):
        x = 30.0 * 0.62 ** k
        objs[k]["flags"] = 2 if k % 3 else 4
        objs[k]["radius"] = x * 0.2
        objs[k]["center"] = (x, 0.3 * x, -5.0 + 0.1 * x)
        objs[k]["color"] = (0.7, 0.6, 0.5)
        objs[k]["emission"] = (0.5, 0.5, 0.5) if k % 5 == 0 else (0.0, 0.0, 0.0)
    rng = np.random.default_rng(77)
    o = rng.uniform(-2, 32, (4000, 3)) * np.array([1.0, 0.3, 0.05]) + np.array([0, 0, 10.0])
    pick = rng.integers(0, n, 4000)
    t = objs["center"][pick] + rng.normal(0.0, 0.6, (4000, 3)) * objs["radius"][pick][:, None]
    d = t - o
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays = np.concatenate([o, d], axis=1)
    W, H = 64, 36
    cam = gpu_api.init_camera(W, H)
    with gpu_api.Scene(objs, all_trees=True) as sc:
        info = sc.info
        brute = sc.trace_rays(rays, use_bvh=0)
        for mode in (1, 3, 4, 5):
            got = sc.trace_rays(rays, use_bvh=mode)
            for k in ("ids", "prims", "t", "points", "normals"):
                assert np.array_equal(got[k], brute[k]), (mode, k)
        _, a4, c4 = sc.render(cam, gpu_api.make_desc(W, H, 0, 4, kernel=4, planes=2), want_accum=True)
        _, a6, c6 = sc.render(cam, gpu_api.make_desc(W, H, 0, 4, kernel=6, planes=2), want_accum=True)
    print("bvh depth", info.bvh_depth, "hit fraction", (brute["ids"] >= 0).mean())
    assert (brute["ids"] >= 0).mean() > 0.5 and info.bvh_depth >= 12
    assert np.array_equal(a4, a6) and c4.rays == c6.rays


def test_tree_walks_on_adversarial_rays(gpu_api):
    """rays aimed exactly at mesh vertices and edge midpoints (ties between neighbouring
    triangles, hits on box faces), axis-aligned rays (zero direction components) and rays that
    start far outside the scene: BVH2, while-while, BVH4 and compressed BVH4 walks all return
    the brute-force loop's nearest hit, bit for bit"""
    W, H = 96, 54
    verts = gpu_api.heightfield_mesh(100, 20 * W / H * 0.98)  # 20 000 triangles
    holder = gpu_api.mesh_room(verts, W, H)
    pos = verts["pos"].reshape(-1, 3, 3)
    rng = np.random.default_rng(2024)
    pick = rng.integers(0, len(pos), 6000)
    targets = np.concatenate([
        pos[pick[:2000], rng.integers(0, 3, 2000)],                       # vertices
        0.5 * (pos[pick[2000:4000], 0] + pos[pick[2000:4000], 1]),         # edge midpoints
        pos[pick[4000:]].mean(axis=1),                                     # centroids
    ])
    origins = np.concatenate([
        rng.uniform(-25, 25, (3000, 3)) * np.array([1.0, 0.3, 1.0]) + np.array([0.0, 8.0, 0.0]),  # inside the room
        rng.normal(size=(3000, 3)) * 400.0 + np.array([0.0, 600.0, 0.0]),                           # far outside
    ])
    d = targets - origins
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays = [np.concatenate([origins, d], axis=1)]
    # axis-aligned rays straight down / sideways through vertices: direction components exactly 0
    t2 = pos[rng.integers(0, len(pos), 1500), 0]
    for axis, sign in ((1, -1.0), (0, 1.0), (2, -1.0)):
        dd = np.zeros((500, 3))
        dd[:, axis] = sign
        oo = t2[500 * (axis % 3):500 * (axis % 3) + 500] - dd * 30.0
        rays.append(np.concatenate([oo, dd], axis=1))
    rays = np.concatenate(rays)
    with gpu_api.Scene(holder, all_trees=True) as sc:
        brute = sc.trace_rays(rays, use_bvh=0)
        for mode in (1, 3, 4, 5):
            got = sc.trace_rays(rays, use_bvh=mode)
            for k in ("ids", "prims", "t", "points", "normals"):
                assert np.array_equal(got[k], brute[k]), (mode, k)
    assert (brute["ids"] >= 0).mean() > 0.9


def test_many_oversized_spheres(gpu_api):
    """more oversized spheres than the every-ray list holds (32): the rest go into the tree, whose Morton
    grid they stretch -- slower, but the nearest hit must still be the brute-force one, ties included"""
    rng = np.random.default_rng(17)
    W, H = 64, 36
    small = gpu_api.scene_sphere_field(500, W, H)
    room = small[:6].copy()                       # the six r = 10 000 walls
    extra = np.repeat(room, 7, axis=0)            # 42 more oversized spheres, slightly displaced
    extra["center"] += rng.uniform(-3.0, 3.0, size=extra["center"].shape)
    extra["radius"] *= rng.uniform(0.999, 1.001, size=len(extra))
    objs = np.concatenate([small, extra])
    rays = random_rays_in_room(rng, 4000)
    with gpu_api.Scene(objs) as sc:
        assert sc.info.n_big_prims == 32
        bvh, brute = sc.trace_rays(rays, use_bvh=1), sc.trace_rays(rays, use_bvh=0)
        cam = gpu_api.init_camera(W, H)
        _, acc, ctr = sc.render(cam, gpu_api.make_desc(W, H, 0, 2), want_accum=True)
    _assert_hits_equal(bvh, brute, "48 oversized spheres")
    assert np.isfinite(acc).all() and ctr.rays > 0


def test_counters_are_deterministic_when_many_rays_skip_the_walk(gpu_api):
    """ADVICE r1: a lane refilled with a ray that needs no walk (it misses the guard box of a small tree inside a
    big-list room) used to fetch a duplicate ray in the same refill; the image was unaffected, the primitive-test
    counter was double-counted and depended on scheduling.  Equal counters run to run, and equal to the ray-pool
    kernel's (same tree, same tests, different scheduling)."""
    W, H = 160, 90
    objs = gpu_api.scene_default(W, H)[:12].copy()          # the six walls + a few spheres: most rays miss the tree
    objs["radius"][6:] *= 0.25
    cam = gpu_api.init_camera(W, H)
    with gpu_api.Scene(objs) as sc:
        runs = [sc.render(cam, gpu_api.make_desc(W, H, 0, 8, max_depth=5), want_accum=True) for _ in range(3)]
        pool = sc.render(cam, gpu_api.make_desc(W, H, 0, 8, max_depth=5, tune=(1024 << 16) | (16 << 8)), want_accum=True)
    for fb, acc, c in runs[1:] + [pool]:
        assert c.prim_tests == runs[0][2].prim_tests and c.rays == runs[0][2].rays
        assert np.array_equal(acc, runs[0][1])


@pytest.mark.parametrize("doubles", [False, True])
def test_degenerate_and_duplicate_triangles(gpu_api, ol, abi, doubles):
    """a mesh with exact duplicates of some triangles (equal t: the lower loop index must win, raytracer.c:404),
    zero-area triangles (three equal vertices, collinear vertices: |det| < EPSILON, raytracer.c:134), a triangle
    spanning the whole room and triangles 1e-5 across -- as floats and as genuine doubles (the tri64 path):
    every walk returns the oracle's brute-force hit, primitive index included, and the accumulated frame
    matches the oracle's"""
    W, H = 96, 54
    base = gpu_api.heightfield_mesh(30, 20 * W / H * 0.98)
    pos = base["pos"].reshape(-1, 3, 3).copy()
    rng = np.random.default_rng(99)
    dup = pos[rng.integers(0, len(pos), 300)]                      # appended later: higher loop index
    point = np.repeat(pos[rng.integers(0, len(pos), 50), :1], 3, axis=1)                    # v0 = v1 = v2
    a, b = pos[rng.integers(0, len(pos), 50), 0], pos[rng.integers(0, len(pos), 50), 1]
    collinear = np.stack([a, 0.5 * (a + b), b], axis=1)
    huge = np.array([[[-60.0, 16.0, -40.0], [60.0, 16.0, -40.0], [0.0, 16.5, 45.0]]])      # above the ray origins
    c = rng.uniform(-15, 15, (200, 1, 3)) * np.array([1.0, 0.2, 1.0]) + np.array([0.0, 2.0, 0.0])
    tiny = c + rng.normal(size=(200, 3, 3)) * 1e-5
    tris = np.concatenate([pos, dup, point, collinear, huge, tiny])
    if doubles:
        tris = tris * (1.0 + 2.0 ** -40) + 2.0 ** -30                                        # not float-representable
    else:
        tris = tris.astype(np.float32).astype(np.float64)
    verts = np.zeros(3 * len(tris), dtype=abi.VERTEX_DTYPE)
    verts["pos"] = tris.reshape(-1, 3)
    verts["tex"] = rng.uniform(0, 1, (3 * len(tris), 2))
    holder = gpu_api.mesh_room(verts, W, H)
    # rays: random ones, and rays aimed at the duplicated, degenerate and tiny triangles
    aim = np.concatenate([dup.mean(axis=1), dup[:, 0], point[:, 0], collinear[:, 1], tiny.mean(axis=1)])
    o = rng.uniform(-20, 20, (len(aim), 3)) * np.array([1.0, 0.1, 1.0]) + np.array([0.0, 12.0, 0.0])
    d = aim - o
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays = np.concatenate([random_rays_in_room(rng, 4000), np.concatenate([o, d], axis=1)])
    want = ol.intersect_rays(holder, rays)
    with gpu_api.Scene(holder, all_trees=True) as sc:
        assert bool(sc.info.double_triangles) == doubles
        for mode in (0, 1, 3, 4, 5):
            _assert_hits_equal(sc.trace_rays(rays, use_bvh=mode), want, f"degenerate mesh, walk {mode}")
        cam = gpu_api.init_camera(W, H)
        _, acc, ctr = sc.render(cam, gpu_api.make_desc(W, H, 0, 4, max_depth=5), want_accum=True)
    n_base = len(pos)
    first = want["prims"][want["ids"] == 6] - 6          # triangle index inside the mesh (6 walls precede it)
    assert ((first >= n_base) & (first < n_base + 300)).sum() == 0, "a duplicate (higher index) won a tie"
    assert (first == n_base + 400).sum() > 100, "the room-spanning triangle must be hit"
    ref_sum, (ref_rays, _) = ol.render_sum(holder, cam, W, H, 4, rng="philox", dielectric="stochastic", max_depth=5)
    assert ctr.rays == ref_rays
    np.testing.assert_allclose(acc, ref_sum, rtol=1e-3, atol=1e-4)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_overlapping_nested_and_extreme_spheres(gpu_api, ol, abi, seed):
    """the generators only make disjoint spheres; here they overlap, nest, span radii 1e-3 .. 3e2 and many rays
    START INSIDE spheres (quirk Q10: tca < 0 misses even then, the far root counts when t0 < 0) or ON a sphere's
    surface (EPSILON self-hit guard, raytracer.c:109): nearest hit == the oracle's brute-force loop in every walk"""
    rng = np.random.default_rng(seed)
    n = 400
    objs = np.zeros(n, dtype=abi.OBJECT_DTYPE)
    objs["flags"] = rng.choice([2, 4, 8, 18], n)
    objs["radius"] = 10.0 ** rng.uniform(-3, 2.5, n)
    objs["center"] = rng.normal(size=(n, 3)) * 20.0
    objs["center"][0:399:7] = objs["center"][1:399:7]                           # concentric pairs (nested shells)
    objs["color"] = rng.uniform(0, 1, (n, 3))
    objs["emission"] = rng.uniform(0, 1, (n, 3)) * (rng.uniform(size=(n, 1)) < 0.3)
    k = rng.integers(0, n, 6000)
    inside = objs["center"][k[:2000]] + rng.normal(size=(2000, 3)) * 0.3 * objs["radius"][k[:2000], None]
    u = rng.normal(size=(2000, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    on_surface = objs["center"][k[2000:4000]] + u * objs["radius"][k[2000:4000], None]
    outside = rng.normal(size=(2000, 3)) * 60.0
    o = np.concatenate([inside, on_surface, outside])
    d = rng.normal(size=(6000, 3))
    d[4000:] = objs["center"][k[4000:]] - outside + rng.normal(size=(2000, 3)) * objs["radius"][k[4000:], None]
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays = np.concatenate([o, d], axis=1)
    want = ol.intersect_rays(objs, rays)
    with gpu_api.Scene(objs, all_trees=True) as sc:
        for mode in (0, 1, 3, 4, 5):
            _assert_hits_equal(sc.trace_rays(rays, use_bvh=mode), want, f"nested spheres, walk {mode}")
        W, H = 64, 36
        cam = gpu_api.init_camera(W, H)
        _, acc, ctr = sc.render(cam, gpu_api.make_desc(W, H, 0, 3, max_depth=6), want_accum=True)
    ref_sum, (ref_rays, _) = ol.render_sum(objs, cam, W, H, 3, rng="philox", dielectric="stochastic", max_depth=6)
    assert ctr.rays == ref_rays
    np.testing.assert_allclose(acc, ref_sum, rtol=1e-3, atol=1e-4)
    assert (want["ids"] >= 0).mean() > 0.5
