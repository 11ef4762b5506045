"""The wavefront renderer's trace kernel (k_wf_trace, k_wf_trace_pool) against the oracle, ray for ray.

rtb_trace_rays_wf queues caller rays exactly as the renderer queues its own (hit record seeded from the oversized
list by the producer), runs ONE launch of the trace kernel the tuning word selects -- through the same dispatch as
wf_render -- and reads the hit records back with rtb_trace_rays' read-out.  So a wrong tie-break, a stale seed, a
skipped ray or a ray fetched twice shows up as a wrong id, primitive or t of a named ray, where a render sum cannot
show it.

The bar is the oracle's brute-force loop (oracle_lib.intersect_rays), or the GPU brute force (rtb_trace_rays
use_bvh = 0, bit-identical to the oracle on every scene of test_gpu_parity.py) where the CPU would take too long,
with a slice against the oracle.  Ids, primitives, t, points, normals and mesh texture coordinates must be
bit-identical: both sides run the same IEEE double arithmetic without FMA contraction (DESIGN.md, a5-a7).  Sphere
texture coordinates go through atan2, whose libm and CUDA forms may differ in the last bit: 1e-15.
"""
import numpy as np
import pytest

from conftest import random_rays_in_room

pytestmark = pytest.mark.gpu

FIELDS = ("ids", "prims", "t", "points", "normals")
TUNE_POOL = 1024 << 16
COMPRESSED = (22, 54, 86, 150, 182, 214)  # compressed-BVH4 variants of k_wf_trace (bit 16)
BVH2 = (0, 2, 6)


def tune_word(variant, node_exit=0, refill=0):
    """rtb_render_desc.reserved: bits 0-7 refill threshold, 8-15 node-phase exit (0xFF = none), 16-27 variant"""
    return (variant << 16) | (node_exit << 8) | refill


def assert_same_records(got, want, what):
    """GPU against GPU: every field of every ray bit-identical, misses included"""
    for k in FIELDS + ("uvs",):
        diff = got[k] != want[k]
        bad = np.flatnonzero(diff.any(axis=tuple(range(1, diff.ndim))) if diff.ndim > 1 else diff)
        assert len(bad) == 0, f"{what}: {k} differs on {len(bad)} rays, e.g. ray {bad[:5]}: {got[k][bad[:3]]} vs {want[k][bad[:3]]}"


def assert_oracle_records(got, want, what, mesh_ids=()):
    """against the oracle: ids exact on every ray; prims, t, points, normals and mesh uvs bit-identical on hits;
    sphere uvs within 1e-15 (atan2 of libm and of CUDA)"""
    bad = np.flatnonzero(got["ids"] != want["ids"])
    assert len(bad) == 0, f"{what}: ids differ on {len(bad)} rays, e.g. ray {bad[:5]}: {got['ids'][bad[:5]]} vs {want['ids'][bad[:5]]}"
    hit = want["ids"] >= 0
    for k in ("prims", "t", "points", "normals"):
        g, w = got[k][hit].reshape(hit.sum(), -1), want[k][hit].reshape(hit.sum(), -1)
        bad = np.flatnonzero(hit)[(g != w).any(axis=1)]
        assert len(bad) == 0, f"{what}: {k} differs on {len(bad)} rays, e.g. ray {bad[:5]}"
    mesh = hit & np.isin(want["ids"], list(mesh_ids))
    bad = np.flatnonzero(mesh)[(got["uvs"][mesh] != want["uvs"][mesh]).any(axis=1)]
    assert len(bad) == 0, f"{what}: mesh uvs differ on {len(bad)} rays, e.g. ray {bad[:5]}"
    sphere = hit & ~mesh
    np.testing.assert_allclose(got["uvs"][sphere], want["uvs"][sphere], rtol=0, atol=1e-15, err_msg=what)


def wf(sc, rays, tune=0, perm=None):
    return sc.trace_rays_wf(rays, tune=tune, perm=perm)[0]


def unit(v):
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def aimed(origins, targets):
    return np.concatenate([origins, unit(targets - origins)], axis=1)


# ---- scenes ---------------------------------------------------------------------------------------------------

def mesh_room(gpu_api, grid=100, W=96, H=54):
    """scene_mesh_room with a height-field mesh (2 * grid^2 triangles, object 6) -> (holder, triangles [T, 3, 3])"""
    verts = gpu_api.heightfield_mesh(grid, 20 * W / H * 0.98)
    return gpu_api.mesh_room(verts, W, H), verts["pos"].reshape(-1, 3, 3).copy()


def mesh_targets(pos, rng, n):
    """vertices, edge midpoints and centroids of random triangles (ties between neighbours, hits on box faces)"""
    pick = rng.integers(0, len(pos), n)
    k = n // 3
    return np.concatenate([pos[pick[:k], rng.integers(0, 3, k)],
                           0.5 * (pos[pick[k:2 * k], 0] + pos[pick[k:2 * k], 1]),
                           pos[pick[2 * k:]].mean(axis=1)])


def degenerate_mesh(gpu_api, abi, doubles, rng, W=96, H=54):
    """exact duplicates (the lower loop index must win), zero-area, tiny and room-spanning triangles"""
    pos = gpu_api.heightfield_mesh(30, 20 * W / H * 0.98)["pos"].reshape(-1, 3, 3)
    dup = pos[rng.integers(0, len(pos), 300)]
    point = np.repeat(pos[rng.integers(0, len(pos), 50), :1], 3, axis=1)
    a, b = pos[rng.integers(0, len(pos), 50), 0], pos[rng.integers(0, len(pos), 50), 1]
    collinear = np.stack([a, 0.5 * (a + b), b], axis=1)
    huge = np.array([[[-60.0, 16.0, -40.0], [60.0, 16.0, -40.0], [0.0, 16.5, 45.0]]])
    tiny = rng.uniform(-15, 15, (200, 1, 3)) * np.array([1.0, 0.2, 1.0]) + np.array([0.0, 2.0, 0.0])
    tiny = tiny + rng.normal(size=(200, 3, 3)) * 1e-5
    tris = np.concatenate([pos, dup, point, collinear, huge, tiny])
    tris = tris * (1.0 + 2.0 ** -40) + 2.0 ** -30 if doubles else tris.astype(np.float32).astype(np.float64)
    verts = np.zeros(3 * len(tris), dtype=abi.VERTEX_DTYPE)
    verts["pos"] = tris.reshape(-1, 3)
    verts["tex"] = rng.uniform(0, 1, (3 * len(tris), 2))
    aim = np.concatenate([dup.mean(axis=1), dup[:, 0], point[:, 0], collinear[:, 1], tiny.mean(axis=1)])
    o = rng.uniform(-20, 20, (len(aim), 3)) * np.array([1.0, 0.1, 1.0]) + np.array([0.0, 12.0, 0.0])
    rays = np.concatenate([random_rays_in_room(rng, 4000), aimed(o, aim)])
    return gpu_api.mesh_room(verts, W, H), rays


def nested_spheres(abi, rng, n=400):
    """overlapping, nested (concentric pairs) spheres of radii 1e-3 .. 3e2; rays from inside, from the surface and
    from outside"""
    objs = np.zeros(n, dtype=abi.OBJECT_DTYPE)
    objs["flags"] = rng.choice([2, 4, 8, 18], n)
    objs["radius"] = 10.0 ** rng.uniform(-3, 2.5, n)
    objs["center"] = rng.normal(size=(n, 3)) * 20.0
    objs["center"][0:399:7] = objs["center"][1:399:7]
    objs["color"] = rng.uniform(0, 1, (n, 3))
    k = rng.integers(0, n, 6000)
    inside = objs["center"][k[:2000]] + rng.normal(size=(2000, 3)) * 0.3 * objs["radius"][k[:2000], None]
    on_surface = objs["center"][k[2000:4000]] + unit(rng.normal(size=(2000, 3))) * objs["radius"][k[2000:4000], None]
    outside = rng.normal(size=(2000, 3)) * 60.0
    d = rng.normal(size=(6000, 3))
    d[4000:] = objs["center"][k[4000:]] - outside + rng.normal(size=(2000, 3)) * objs["radius"][k[4000:], None]
    return objs, np.concatenate([np.concatenate([inside, on_surface, outside]), unit(d)], axis=1)


def deep_chain_spheres(abi):
    """spheres spaced geometrically along a line (test_gpu_parity.py::test_deep_unbalanced_tree): a chain-like tree
    (the trees at the stack bound, with and without the BVH4 fallback, are section D)"""
    n = 58
    objs = np.zeros(n, dtype=abi.OBJECT_DTYPE)
    x = 30.0 * 0.62 ** np.arange(n)
    objs["flags"] = np.where(np.arange(n) % 3 != 0, 2, 4)
    objs["radius"] = x * 0.2
    objs["center"] = np.stack([x, 0.3 * x, -5.0 + 0.1 * x], axis=1)
    objs["color"] = (0.7, 0.6, 0.5)
    rng = np.random.default_rng(77)
    o = rng.uniform(-2, 32, (4000, 3)) * np.array([1.0, 0.3, 0.05]) + np.array([0, 0, 10.0])
    pick = rng.integers(0, n, 4000)
    t = objs["center"][pick] + rng.normal(0.0, 0.6, (4000, 3)) * objs["radius"][pick][:, None]
    return objs, aimed(o, t)


# ---- A. oracle parity of the renderer's default trace kernel -------------------------------------------------

def test_default_scene_and_reference_golden(gpu_api, ol):
    """C1: camera rays through every third pixel and random rays from inside the room; and the unmodified
    reference's intersect() outputs stored in tests/golden/c1_hits.npz"""
    import os
    W, H = 320, 180
    objs = gpu_api.scene_default(W, H)
    cam = gpu_api.init_camera(W, H)
    ys, xs = np.mgrid[0:H:3, 0:W:3]
    rays = np.stack([ol.camera_ray(cam, (x + 0.5) / (W - 1.0), (y + 0.5) / (H - 1.0)) for x, y in zip(xs.ravel(), ys.ravel())])
    rays = np.concatenate([rays, random_rays_in_room(np.random.default_rng(1), 4000)])
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "c1_hits.npz"))
    golden_rays = random_rays_in_room(np.random.default_rng(105), 3000)
    with gpu_api.Scene(objs) as sc:
        got = wf(sc, rays)
        gold = wf(sc, golden_rays)
    assert_oracle_records(got, ol.intersect_rays(objs, rays), "C1")
    assert np.array_equal(gold["ids"], g["ids"])
    hit = g["ids"] >= 0
    # records of the unmodified reference build (tests/golden/make_golden.py), at the tolerance
    # test_gpu_parity.py::test_nearest_hit_vs_reference_golden holds them to
    for k in ("points", "normals", "uvs"):
        np.testing.assert_allclose(gold[k][hit], g[k][hit], rtol=1e-9, atol=1e-9, err_msg=k)


def test_ten_thousand_spheres(gpu_api, ol):
    objs = gpu_api.scene_sphere_field(10000, 192, 108)
    rays = random_rays_in_room(np.random.default_rng(3), 200000)
    with gpu_api.Scene(objs) as sc:
        got = wf(sc, rays)
        brute = sc.trace_rays(rays, use_bvh=0)
    assert_same_records(got, brute, "10k spheres vs GPU brute force")
    assert_oracle_records({k: v[:10000] for k, v in got.items()}, ol.intersect_rays(objs, rays[:10000]), "10k spheres")


def test_duplicate_spheres_and_walls(gpu_api, ol):
    """equal t between duplicates in the tree and in the oversized list: the lowest index wins"""
    base = gpu_api.scene_sphere_field(500, 192, 108)
    dup = np.concatenate([base, base[6:206][::-1], base[:6]])
    rays = random_rays_in_room(np.random.default_rng(4), 20000)
    want = ol.intersect_rays(dup, rays)
    with gpu_api.Scene(dup) as sc:
        got = wf(sc, rays)
    assert want["ids"].max() < len(base)
    assert_oracle_records(got, want, "duplicates")


def test_mesh_vertices_edges_and_centroids(gpu_api, ol):
    """20 000 triangles; rays aimed at vertices, edge midpoints and centroids from inside the room and from far
    outside, and axis-aligned rays through vertices"""
    holder, pos = mesh_room(gpu_api)
    rng = np.random.default_rng(2024)
    targets = mesh_targets(pos, rng, 6000)
    origins = np.concatenate([rng.uniform(-25, 25, (3000, 3)) * np.array([1.0, 0.3, 1.0]) + np.array([0.0, 8.0, 0.0]),
                              rng.normal(size=(3000, 3)) * 400.0 + np.array([0.0, 600.0, 0.0])])
    rays = [aimed(origins, targets)]
    v = pos[rng.integers(0, len(pos), 1500), 0]
    for k, (axis, sign) in enumerate(((1, -1.0), (0, 1.0), (2, -1.0))):
        d = np.zeros((500, 3))
        d[:, axis] = sign
        rays.append(np.concatenate([v[500 * k:500 * k + 500] - 30.0 * d, d], axis=1))
    rays = np.concatenate(rays)
    want = ol.intersect_rays(holder, rays)
    with gpu_api.Scene(holder) as sc:
        got = wf(sc, rays)
    assert_oracle_records(got, want, "mesh", mesh_ids=(6,))
    assert (want["ids"] == 6).mean() > 0.5


@pytest.mark.parametrize("doubles", [False, True], ids=["float", "double"])
def test_degenerate_duplicate_tiny_and_spanning_triangles(gpu_api, ol, abi, doubles):
    """as floats and as doubles: the double mesh runs the T64 instantiation of the trace kernel"""
    rng = np.random.default_rng(99)
    holder, rays = degenerate_mesh(gpu_api, abi, doubles, rng)
    want = ol.intersect_rays(holder, rays)
    with gpu_api.Scene(holder) as sc:
        assert bool(sc.info.double_triangles) == doubles
        got = wf(sc, rays)
        pool = wf(sc, rays, TUNE_POOL)
    assert_oracle_records(got, want, "degenerate mesh", mesh_ids=(6,))
    assert_oracle_records(pool, want, "degenerate mesh, ray pool", mesh_ids=(6,))


def test_double_texcoords(gpu_api, ol):
    """a mesh whose texture coordinates are not float-representable (tex64): uvs bit-identical"""
    holder_verts = gpu_api.heightfield_mesh(40, 20 * 96 / 54 * 0.98)
    rng = np.random.default_rng(8)
    holder_verts["tex"] = rng.uniform(-1000.0, 1000.0, (len(holder_verts), 2))
    holder = gpu_api.mesh_room(holder_verts, 96, 54)
    pos = holder_verts["pos"].reshape(-1, 3, 3)
    w = rng.dirichlet((1.0, 1.0, 1.0), 8000)
    target = np.einsum("nk,nka->na", w, pos[rng.integers(0, len(pos), 8000)])
    o = rng.uniform(-20, 20, (8000, 3)) * np.array([1.0, 0.2, 1.0]) + np.array([0.0, 10.0, 0.0])
    rays = aimed(o, target)
    want = ol.intersect_rays(holder, rays)
    with gpu_api.Scene(holder) as sc:
        assert sc.info.double_texcoords == 1
        got = wf(sc, rays)
    assert_oracle_records(got, want, "tex64 mesh", mesh_ids=(6,))
    assert (want["ids"] == 6).mean() > 0.6


@pytest.mark.parametrize("seed", [1, 2])
def test_nested_and_extreme_spheres(gpu_api, ol, abi, seed):
    objs, rays = nested_spheres(abi, np.random.default_rng(seed))
    want = ol.intersect_rays(objs, rays)
    with gpu_api.Scene(objs) as sc:
        got = wf(sc, rays)
    assert_oracle_records(got, want, "nested spheres")
    assert (want["ids"] >= 0).mean() > 0.5


def test_many_oversized_spheres(gpu_api, ol):
    """48 oversized spheres: 32 in the oversized list (the producer's seed), the rest in the tree"""
    rng = np.random.default_rng(17)
    small = gpu_api.scene_sphere_field(500, 64, 36)
    extra = np.repeat(small[:6].copy(), 7, axis=0)
    extra["center"] += rng.uniform(-3.0, 3.0, size=extra["center"].shape)
    extra["radius"] *= rng.uniform(0.999, 1.001, size=len(extra))
    objs = np.concatenate([small, extra])
    rays = random_rays_in_room(rng, 6000)
    want = ol.intersect_rays(objs, rays)
    with gpu_api.Scene(objs) as sc:
        assert sc.info.n_big_prims == 32
        got = wf(sc, rays)
    assert_oracle_records(got, want, "48 oversized spheres")


def test_everything_in_the_oversized_list_and_empty_scene(gpu_api, ol, abi, monkeypatch):
    """no tree at all: the producer's seed is the answer (RTB_BIG_RATIO=0 sends every sphere to the oversized list)"""
    rays = random_rays_in_room(np.random.default_rng(6), 5000)
    objs = gpu_api.scene_default(320, 180)[:20].copy()
    monkeypatch.setenv("RTB_BIG_RATIO", "0")
    with gpu_api.Scene(objs) as sc:
        assert sc.info.n_big_prims == 20 and sc.info.n_bvh_prims == 0
        got, ctr = sc.trace_rays_wf(rays)
    assert_oracle_records(got, ol.intersect_rays(objs, rays), "oversized list only")
    assert ctr.node_visits == 0
    monkeypatch.delenv("RTB_BIG_RATIO")
    with gpu_api.Scene(np.zeros(0, dtype=abi.OBJECT_DTYPE)) as sc:
        got, ctr = sc.trace_rays_wf(rays)
    assert (got["ids"] == -1).all() and ctr.prim_tests == 0 and ctr.node_visits == 0


def test_deep_unbalanced_tree(gpu_api, ol, abi):
    objs, rays = deep_chain_spheres(abi)
    want = ol.intersect_rays(objs, rays)
    with gpu_api.Scene(objs) as sc:
        got = wf(sc, rays)
        pool = wf(sc, rays, TUNE_POOL)
    assert_oracle_records(got, want, "deep chain")
    assert_same_records(pool, got, "deep chain, ray pool")
    assert (want["ids"] >= 0).mean() > 0.5


# ---- A'. new ray shapes ---------------------------------------------------------------------------------------

TINY = (0.0, -0.0, 1e-300, -1e-300, 1e-40, -1e-40, 1e-30, -1e-30)


def test_direction_components_zero_or_below_float_range(gpu_api, ol):
    """direction components exactly +-0, or non-zero doubles that round to 0 (1e-300) or to a subnormal (1e-40,
    1e-30 -> its reciprocal overflows) as floats, along each axis, through mesh vertices"""
    holder, pos = mesh_room(gpu_api, grid=60)
    rng = np.random.default_rng(31)
    rays = []
    for axis, sign, dist in ((1, -1.0, 30.0), (0, 1.0, 40.0), (2, -1.0, 40.0), (1, 1.0, 8.0)):
        others = [a for a in range(3) if a != axis]
        for e1 in TINY:
            for e2 in TINY:
                v = pos[rng.integers(0, len(pos), 24), rng.integers(0, 3, 24)]
                d = np.zeros((24, 3))
                d[:, axis], d[:, others[0]], d[:, others[1]] = sign, e1, e2
                rays.append(np.concatenate([v - dist * d, d], axis=1))
    rays = np.concatenate(rays)
    want = ol.intersect_rays(holder, rays)
    with gpu_api.Scene(holder, all_trees=True) as sc:
        for tune in (0, tune_word(10), TUNE_POOL):
            assert_oracle_records(wf(sc, rays, tune), want, f"tiny direction components, tune {tune:#x}", mesh_ids=(6,))
    assert (want["ids"] == 6).mean() > 0.5


def _round_down(x):
    f = x.astype(np.float32)
    return np.where(f.astype(np.float64) > x, np.nextafter(f, np.float32(-np.inf)), f)


def _round_up(x):
    f = x.astype(np.float32)
    return np.where(f.astype(np.float64) < x, np.nextafter(f, np.float32(np.inf)), f)


def guard_box(objs):
    """the guard box k_build_params derives from the BVH spheres' boxes: scene box grown by its diagonal, as floats"""
    c, r = objs["center"], np.abs(objs["radius"])[:, None]
    lo, hi = _round_down(c - r).min(axis=0), _round_up(c + r).max(axis=0)
    diag = np.sqrt(((hi.astype(np.float64) - lo.astype(np.float64)) ** 2).sum())
    return (lo.astype(np.float64) - diag).astype(np.float32), (hi.astype(np.float64) + diag).astype(np.float32)


def test_origins_on_the_guard_box_faces(gpu_api, ol):
    """origins exactly on a face of the guard box (and one float step either side), where rayf_walk_setup switches
    between re-basing the ray and walking it from its own origin"""
    objs = gpu_api.scene_sphere_field(500, 96, 54)[6:].copy()  # no walls: every sphere is in the tree
    rng = np.random.default_rng(12)
    g_lo, g_hi = guard_box(objs)
    rays = []
    for axis in range(3):
        for face in (g_lo[axis], g_hi[axis]):
            for f in (np.nextafter(face, np.float32(-np.inf)), face, np.nextafter(face, np.float32(np.inf))):
                o = rng.uniform(g_lo, g_hi, (400, 3)).astype(np.float64)
                o[:, axis] = float(f)
                tgt = objs["center"][rng.integers(0, len(objs), 400)]
                rays.append(aimed(o[:300], tgt[:300]))
                rays.append(aimed(o[300:], 2.0 * o[300:] - tgt[300:]))  # pointing away from the scene
    rays = np.concatenate(rays)
    want = ol.intersect_rays(objs, rays)
    with gpu_api.Scene(objs, all_trees=True) as sc:
        assert sc.info.n_big_prims == 0
        for tune in (0, tune_word(6), TUNE_POOL):
            assert_oracle_records(wf(sc, rays, tune), want, f"guard-box faces, tune {tune:#x}")
    assert (want["ids"] >= 0).mean() > 0.3


def test_origins_far_outside_the_scene(gpu_api, ol, abi):
    """origins 1e2 .. 1e12 scene diagonals away, aimed at mesh vertices, edges and centroids and at spheres.  Up to
    SceneView::far_t outside the guard box (here about 260 diagonals) the FP32 walk re-bases the ray and must stay
    conservative; beyond it the walk enters every box.  Before that rule, origins from about 1e4 diagonals on lost
    nearer hits: the re-based origin left the envelope the box padding covers, and the reference's sphere test
    (d2 = L.L - tca^2) accepts rays that pass outside the padded box of a small sphere.  Every walk of the probes
    shares the set-up and is held to the same records."""
    verts = gpu_api.heightfield_mesh(100, 34.0)
    spheres = gpu_api.scene_sphere_field(200, 96, 54)[6:]
    items = [("mesh", verts, abi.M_DEFAULT, (0.6, 0.6, 0.6), (0.0, 0.0, 0.0))] + [("sphere", s) for s in spheres]
    holder = abi.SceneHolder.build(items)
    pos = verts["pos"].reshape(-1, 3, 3)
    rng = np.random.default_rng(5)
    lo = np.minimum(pos.reshape(-1, 3).min(axis=0), (spheres["center"] - spheres["radius"][:, None]).min(axis=0))
    hi = np.maximum(pos.reshape(-1, 3).max(axis=0), (spheres["center"] + spheres["radius"][:, None]).max(axis=0))
    diag = np.linalg.norm(hi - lo)
    n = 9000
    targets = np.concatenate([mesh_targets(pos, rng, 6000),
                              spheres["center"][rng.integers(0, len(spheres), 3000)] +
                              rng.normal(size=(3000, 3)) * 0.5 * spheres["radius"][rng.integers(0, len(spheres), 3000), None]])
    dist = diag * 10.0 ** rng.uniform(2.0, 12.0, n)
    u = unit(rng.normal(size=(n, 3)))
    u[:, 1] = np.abs(u[:, 1])  # from above the height field
    rays = aimed(0.5 * (lo + hi) + u * dist[:, None], targets)
    want = ol.intersect_rays(holder, rays)
    with gpu_api.Scene(holder, all_trees=True) as sc:
        for tune in (0, tune_word(6), TUNE_POOL):
            assert_oracle_records(wf(sc, rays, tune), want, f"far origins, tune {tune:#x}", mesh_ids=(0,))
        for mode in (1, 2, 3, 4, 5):
            assert_oracle_records(sc.trace_rays(rays, use_bvh=mode), want, f"far origins, walk {mode}", mesh_ids=(0,))
    assert (want["ids"] >= 0).mean() > 0.7


# ---- B. every trace kernel the renderer can run ---------------------------------------------------------------

@pytest.fixture(scope="module")
def knob_scene(gpu_api):
    """all_trees mesh-plus-spheres scene, rays from inside the room and aimed at the mesh, and the brute force"""
    holder, pos = mesh_room(gpu_api, grid=60)
    rng = np.random.default_rng(41)
    o = rng.uniform(-25, 25, (10000, 3)) * np.array([1.0, 0.3, 1.0]) + np.array([0.0, 8.0, 0.0])
    rays = np.concatenate([random_rays_in_room(rng, 10000), aimed(o, mesh_targets(pos, rng, 10000))])
    sc = gpu_api.Scene(holder, all_trees=True)
    brute = sc.trace_rays(rays, use_bvh=0)
    yield sc, rays, brute
    sc.close()


def _knob_runs(sc, rays, monkeypatch):
    """(label, tune, guided, perm) -> (records, counters) over every knob of the issue's list"""
    n = len(rays)
    perms = {"none": None, "reversed": np.arange(n)[::-1].copy(), "random": np.random.default_rng(9).permutation(n)}
    runs = {}
    for v in BVH2 + (10,) + COMPRESSED:
        runs[(f"variant {v}", tune_word(v, 16, 8), "1", "none")] = None
    runs[("pool", TUNE_POOL, "1", "none")] = None
    for base, label in ((22, "variant 22"), (1024, "pool")):
        for ne in (0xFF, 1, 16, 31):
            for refill in (1, 8, 32):
                runs[(f"{label} node_exit {ne} refill {refill}", tune_word(base, ne, refill), "1", "none")] = None
    for g in ("0", "1", "34"):
        for p in perms:
            runs[(f"default guided {g} perm {p}", 0, g, p)] = None
            runs[(f"pool guided {g} perm {p}", TUNE_POOL, g, p)] = None
    for key in runs:
        _, tune, g, p = key
        monkeypatch.setenv("RTB_WF_GUIDED", g)
        runs[key] = sc.trace_rays_wf(rays, tune=tune, perm=perms[p])
    return runs


def test_every_kernel_and_knob_equals_brute_force(knob_scene, monkeypatch):
    """variants 0 2 6 10 22 54 86 150 182 214 and the pool; node_exit x refill for 22 and the pool; guided batch
    words 0 1 34; fetch order none / reversed / random.  Hits bit-equal to brute force; per-walk counters equal
    across every scheduling knob (they depend only on the rays and the tree walked)"""
    sc, rays, brute = knob_scene
    runs = _knob_runs(sc, rays, monkeypatch)
    for (label, *_), (got, _) in runs.items():
        assert_same_records(got, brute, label)
    assert (brute["ids"] == 6).sum() > 5000
    groups = {"compressed BVH4": lambda lab: not lab.startswith("variant ") or int(lab.split()[1]) in COMPRESSED,
              "BVH2": lambda lab: lab.startswith("variant ") and int(lab.split()[1]) in BVH2}
    for name, member in groups.items():
        ctrs = {lab: (c.prim_tests, c.node_visits) for (lab, *_), (_, c) in runs.items() if member(lab)}
        assert len(set(ctrs.values())) == 1, f"{name}: counters depend on scheduling: {ctrs}"
        assert next(iter(ctrs.values()))[1] > 0


@pytest.mark.parametrize("tune", [0, TUNE_POOL, tune_word(6), tune_word(10, 0xFF, 1)], ids=["default", "pool", "bvh2", "bvh4"])
def test_counters_are_additive(knob_scene, tune):
    """T(rays) = T(rays[:k]) + T(rays[k:]): a ray fetched twice or skipped breaks it"""
    sc, rays, _ = knob_scene
    whole = sc.trace_rays_wf(rays, tune=tune)[1]
    for k in (1, 12345, len(rays) - 33):
        a, b = sc.trace_rays_wf(rays[:k], tune=tune)[1], sc.trace_rays_wf(rays[k:], tune=tune)[1]
        assert (a.prim_tests + b.prim_tests, a.node_visits + b.node_visits) == (whole.prim_tests, whole.node_visits), k


@pytest.mark.parametrize("variant", [2, 6, 10])
def test_variants_without_their_tree_are_rejected(gpu_api, variant):
    """the BVH2 and the uncompressed BVH4 exist only with RTB_SCENE_ALL_TREES: a tuning word that selects a walk
    over them on a product scene is an error (it used to read through a NULL node array), in the probe and in the
    renderer; the default kernel and the pool still run"""
    objs = gpu_api.scene_sphere_field(300, 64, 36)
    rays = random_rays_in_room(np.random.default_rng(2), 1000)
    cam = gpu_api.init_camera(64, 36)
    with gpu_api.Scene(objs) as sc:
        with pytest.raises(gpu_api.RtbError, match="RTB_SCENE_ALL_TREES"):
            sc.trace_rays_wf(rays, tune=tune_word(variant))
        with pytest.raises(gpu_api.RtbError, match="RTB_SCENE_ALL_TREES"):
            sc.render(cam, gpu_api.make_desc(64, 36, 0, 1, kernel=6, tune=tune_word(variant)))
        brute = sc.trace_rays(rays, use_bvh=0)
        for tune in (0, TUNE_POOL):
            assert_same_records(wf(sc, rays, tune), brute, f"tune {tune:#x} after a rejected word")


def test_perm_must_be_a_permutation(knob_scene, gpu_api):
    sc, rays, _ = knob_scene
    n = 100
    for bad in (np.full(n, 3), np.r_[np.arange(n - 1), n], np.r_[np.arange(n - 1), 2 ** 31]):
        with pytest.raises(gpu_api.RtbError, match="permutation"):
            sc.trace_rays_wf(rays[:n], perm=bad)


# ---- C. queue lengths where the scheduler changes behaviour ---------------------------------------------------

def _n_warps():
    """resident warps of the default trace kernel: SMs x 8 blocks x 4 warps (4 736 on 148 SMs)"""
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count * 8 * 4


QUEUE_SIZES = ["0", "1", "31", "32", "33", "511", "512", "513", "32w-1", "32w+1", "128w-1", "128w+1", "2000017"]
PATTERNS = {"alternating": lambda i: i % 2 == 1, "none": lambda i: np.zeros(len(i), bool),
            "all": lambda i: np.ones(len(i), bool)}
for _run in (1, 7, 31, 32, 33, 100):
    PATTERNS[f"runs of {_run}"] = (lambda L: lambda i: (i // L) % 2 == 1)(_run)


@pytest.fixture(scope="module")
def queue_scene(gpu_api):
    """a sphere field without walls (no oversized list: every seed is a miss) and two ray pools: rays from inside
    the scene box aimed at a sphere (each has a tree hit, nearer than its seed) and rays from outside the guard box
    pointing away (no walk at all; the seeded miss is final)"""
    objs = gpu_api.scene_sphere_field(600, 96, 54)[6:].copy()
    g_lo, g_hi = guard_box(objs)
    m = 2000017
    rng = np.random.default_rng(23)
    lo, hi = objs["center"].min(axis=0), objs["center"].max(axis=0)
    o = rng.uniform(lo, hi, (m, 3))
    walk = aimed(o, objs["center"][rng.integers(0, len(objs), m)])
    u = unit(rng.normal(size=(m, 3)))
    centre = 0.5 * (g_lo.astype(np.float64) + g_hi.astype(np.float64))
    far = centre + u * 2.0 * np.linalg.norm(g_hi.astype(np.float64) - g_lo.astype(np.float64))
    away = np.concatenate([far, u], axis=1)
    sc = gpu_api.Scene(objs)
    assert sc.info.n_big_prims == 0
    want_walk, want_away = sc.trace_rays(walk, use_bvh=0), sc.trace_rays(away, use_bvh=0)
    assert (want_walk["ids"] >= 0).all() and (want_away["ids"] == -1).all()
    yield sc, objs, walk, away, want_walk, want_away
    sc.close()


@pytest.mark.parametrize("size", QUEUE_SIZES)
def test_queue_lengths_and_rays_without_a_walk(queue_scene, ol, monkeypatch, size):
    """every queue length where batch sizes, warp counts or guided batches change, with rays that need no walk
    mixed in (alternating, in runs of 1 7 31 32 33 100, all, none): every ray gets its own nearest hit"""
    sc, objs, walk, away, want_walk, want_away = queue_scene
    nw = _n_warps()
    n = {"32w-1": 32 * nw - 1, "32w+1": 32 * nw + 1, "128w-1": 128 * nw - 1, "128w+1": 128 * nw + 1}.get(size)
    n = int(size) if n is None else n
    guided = ("0", "1", "34") if n > 256 * nw else ("1",)
    i = np.arange(n)
    for name, pattern in PATTERNS.items():
        skip = pattern(i)
        rays = np.where(skip[:, None], away[:n], walk[:n])
        want = {k: np.where(skip.reshape((-1,) + (1,) * (want_walk[k].ndim - 1)), want_away[k][:n], want_walk[k][:n])
                for k in want_walk}
        ctrs = set()
        for g in guided:
            monkeypatch.setenv("RTB_WF_GUIDED", g)
            for tune in (0, TUNE_POOL):
                got, c = sc.trace_rays_wf(rays, tune=tune)
                assert_same_records(got, want, f"n={n} {name} tune={tune:#x} guided={g}")
                ctrs.add((c.prim_tests, c.node_visits))
        assert len(ctrs) == 1, f"n={n} {name}: counters depend on the kernel or batch sizes: {ctrs}"
        if name == "alternating" and n > 0:
            a = sc.trace_rays_wf(rays[skip])[1]
            b = sc.trace_rays_wf(rays[~skip])[1]
            assert (a.prim_tests + b.prim_tests, a.node_visits + b.node_visits) == ctrs.pop()
            assert a.node_visits == 0, "rays from outside the guard box pointing away must not walk"
    k = min(n, 2000)
    if k:
        assert_oracle_records({f: v[:k] for f, v in got.items()}, ol.intersect_rays(objs, rays[:k]), f"n={n} vs oracle")


# ---- D. trees at the traversal-stack bound --------------------------------------------------------------------

def chain_objects(abi, depth):
    """small spheres (radius 0.5 on a unit grid, none oversized) whose Morton codes make a Karras chain of BVH2
    depth `depth`.

    k_morton quantises box centres to 21 bits per axis, normalised by the largest extent; code bit 3j+2 is bit j of
    x, 3j+1 of y, 3j of z.  A set of codes c_0 = 0 < c_1 < ... in which c_k's highest set bit is k-1 gives a chain:
    every split peels off the largest code.  Here c_k is the grid point
        highest bit 3j:   (2^j - 1, 2^j - 1, 2^j)
        highest bit 3j+1: (2^j - 1, 2^j, 2^j)
        highest bit 3j+2: (2^j, 2^j, 2^j)
    all within one cell of the main diagonal, for highest bits 0 .. depth - 2, plus the far corner (2^21 - 2)^3 (bit
    62): the root's split.  Centres sit at grid + 0.5, so the quantised value is the grid point; the far corner's box
    ends at 2^21 - 1, so the normalisation is exact."""
    pts = [(0, 0, 0)]
    for b in range(depth - 1):
        j, a = divmod(b, 3)
        p = 1 << j
        pts.append(((p - 1, p - 1, p), (p - 1, p, p), (p, p, p))[a])
    pts.append((2 ** 21 - 2,) * 3)
    objs = np.zeros(len(pts), dtype=abi.OBJECT_DTYPE)
    objs["flags"] = abi.M_DEFAULT
    objs["radius"] = 0.5
    objs["center"] = np.array(pts, dtype=np.float64) + 0.5
    objs["color"] = (0.5, 0.5, 0.5)
    return objs


def chain_rays(objs, rng):
    """rays along the diagonal line (t - 0.5, t - 0.25, t), which passes through every sphere's box: from below the
    origin corner outward (every node's near child is the inner one, so every level pushes its leaf and the stack
    reaches its worst case before the first leaf test), inward from beyond the far corner, and rays aimed at each
    sphere from the origin side"""
    d = unit(np.ones((1, 3)))
    starts = np.array([[-3.5, -3.25, -3.0], [-1e3 - 0.5, -1e3 - 0.25, -1e3]])
    rays = [np.concatenate([starts, np.repeat(d, 2, axis=0)], axis=1),
            np.concatenate([np.array([[2.0 ** 22 - 0.5, 2.0 ** 22 - 0.25, 2.0 ** 22]]), -d], axis=1)]
    o = np.array([-3.5, -3.25, -3.0]) + rng.normal(size=(len(objs) * 8, 3)) * 0.2
    rays.append(aimed(o, np.repeat(objs["center"], 8, axis=0) + rng.normal(size=(len(objs) * 8, 3)) * 0.2))
    return np.concatenate(rays)


@pytest.mark.parametrize("depth,bvh4_depth", [(60, 20), (61, 0), (62, 0)],
                         ids=["deepest-walked-bvh4", "shallowest-bvh4-fallback", "bvh2-at-the-bound"])
def test_trees_at_the_traversal_stack_bound(gpu_api, ol, abi, depth, bvh4_depth):
    """Worst-case stack use of every walk, RTB_STACK_SIZE = 64 entries (k_wf_trace: 8 in shared memory + 56 in
    local memory; probes: 64 in local memory; k_wf_trace_pool: one cached top + 64 in global memory per slot):
      - BVH2 walks (rtb_trace_rays use_bvh 1..3, k_wf_trace variants 0 2 6): a node step pushes at most one entry,
        the far child, and an entry lives until popped, so the stack holds at most one entry per inner node on the
        path from the root: bvh_depth <= 62 entries.  POP2 (bit 128) only READS the two top entries (sp - 1, sp - 2
        when sp > 1) and never pushes.
      - BVH4 walks (use_bvh 4, 5, variants 10 22 54 86 150 182 214, the pool): at most three pushes per level,
        3 * bvh4_depth <= 62 entries (the build walks the BVH4 only then); the pool keeps the newest of them in
        shared memory, so its global stack holds at most 61.
    So the build's bounds (bvh_depth <= 62, 3 * bvh4_depth <= 62) keep every walk within 64 entries; this test
    reaches them: a BVH2 of depth exactly 62, the deepest BVH4 still walked (20 levels, 60 entries) and the
    shallowest one that falls back to the BVH2 (21 levels)."""
    objs = chain_objects(abi, depth)
    rays = chain_rays(objs, np.random.default_rng(depth))
    want = ol.intersect_rays(objs, rays)
    with gpu_api.Scene(objs, all_trees=True) as sc:
        info = sc.info
        assert (info.bvh_depth, info.bvh4_depth, info.n_big_prims) == (depth, bvh4_depth, 0)
        brute = sc.trace_rays(rays, use_bvh=0)
        assert_oracle_records(brute, want, f"chain {depth}, brute force")
        for mode in (1, 2, 3, 4, 5):
            assert_same_records(sc.trace_rays(rays, use_bvh=mode), brute, f"chain {depth}, walk {mode}")
        for tune in (0, TUNE_POOL, tune_word(6, 0xFF, 1), tune_word(150, 0xFF, 1), tune_word(214, 16, 8)):
            assert_same_records(wf(sc, rays, tune), brute, f"chain {depth}, tune {tune:#x}")
    assert (want["ids"][:3] >= 0).all(), "the diagonal rays hit the chain"


def test_tree_one_level_too_deep_is_rejected(gpu_api, abi):
    """a BVH2 of depth 63 could overflow the BVH2 walks' stack: scene creation fails, nothing is walked"""
    with pytest.raises(gpu_api.RtbError, match="deeper than the traversal stack"):
        gpu_api.Scene(chain_objects(abi, 63))
    with gpu_api.Scene(chain_objects(abi, 62)) as sc:  # the build still works afterwards
        assert sc.info.bvh_depth == 62
