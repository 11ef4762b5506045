"""Texture coordinates and the checker pattern on the GPU against the oracle.

M_CHECKERED (raytracer.c:386-391) scales a surface's albedo by 0.3 or 0.7 depending on fmod(u * M, 1) and
fmod(v * M, 1), with M = 100 000 in trace_path and M = 10 in cast_ray.  At M = 100 000 a change in the 9th digit of
a texture coordinate flips the factor, a 2.3x change of the path's radiance.  So the tests here hold the device's
(u, v) to the oracle's bit for bit on meshes (both sides interpolate the caller's doubles in the same order,
rtb_device.cuh surface_at against oracle.c:291), and to 1e-15 on spheres (atan2 of libm and of CUDA may differ in
the last bit).

Texture coordinate kinds of the meshes:
  float   float-representable, in [0, 1] (OBJ files, the C3 generator): the scene keeps float texcoords;
  double  uniform random doubles in [0, 1], unrelated to position (a mix-up of triangles cannot hide);
  wide    doubles in [-1000, 1000]: the negative fmod branch, and one float ulp (6e-5) would randomise the checker.
The last two make the scene keep the caller's doubles (rtb_scene_info.double_texcoords).
"""
import numpy as np
import pytest

from conftest import random_rays_in_room

pytestmark = pytest.mark.gpu

M_PATH, M_WHITTED = 100000.0, 10.0
KINDS = ("float", "double", "wide")
WALKS = (0, 1, 3, 4, 5)  # brute force, BVH2, while-while, BVH4, compressed BVH4
MESH = 6                 # object index of the mesh in scene_mesh_room


def checker_on(uv, M):
    """the checker's choice (raytracer.c:386-391) in numpy: True = factor 0.7"""
    return (np.fmod(uv[:, 0] * M, 1.0) > 0.5) ^ (np.fmod(uv[:, 1] * M, 1.0) < 0.5)


def near_cell_edge(uv, M, eps=1e-9):
    """u * M or v * M within eps of a multiple of 0.5, where the checker changes"""
    x = 2.0 * uv * M
    return (np.abs(x - np.round(x)) < 2.0 * eps).any(axis=1)


def texcoords(kind, n, rng):
    if kind == "float":
        return rng.uniform(0.0, 1.0, (n, 2)).astype(np.float32).astype(np.float64)
    t = rng.uniform(0.0, 1.0, (n, 2)) if kind == "double" else rng.uniform(-1000.0, 1000.0, (n, 2))
    assert not np.array_equal(t, t.astype(np.float32).astype(np.float64))
    return t


def checkered_room(gpu_api, abi, grid, kind, W, H, seed=0):
    """scene_mesh_room with a height-field mesh of `kind` texcoords -> (holder, vertices)"""
    verts = gpu_api.heightfield_mesh(grid, 20 * W / H * 0.98)
    verts["tex"] = texcoords(kind, len(verts), np.random.default_rng(seed))
    return checkered(abi, gpu_api.mesh_room(verts, W, H)), verts


def checkered(abi, holder):
    """checker the mesh, the mirror ball, the glass ball and the back and left walls of a scene_mesh_room: M_CHECKERED
    together with M_DEFAULT, M_REFLECTION and M_REFRACTION (the factor scales the albedo whatever the material)"""
    kinds = [holder.objects[k].material.flags for k in range(holder.n)]
    assert kinds[MESH] == abi.M_DEFAULT and kinds[11] == abi.M_REFLECTION and kinds[12] == abi.M_REFRACTION
    for k in (1, 2, MESH, 11, 12):
        holder.objects[k].material.flags |= abi.M_CHECKERED
    return holder


def checkered_field(gpu_api, abi, W, H, count=400):
    """a packed sphere field (diffuse, mirror, glass, emissive) with every other sphere checkered"""
    objs = gpu_api.scene_sphere_field(count, W, H, mix=(0.3, 0.3, 0.3))
    objs["flags"][::2] |= abi.M_CHECKERED
    return objs


def mesh_rays(verts, rng, n):
    """rays from inside the room aimed at random triangles of the mesh"""
    pos = verts["pos"].reshape(-1, 3, 3)
    pick = rng.integers(0, len(pos), n)
    w = rng.dirichlet((1.0, 1.0, 1.0), n)
    target = np.einsum("nk,nka->na", w, pos[pick])
    o = rng.uniform(-20, 20, (n, 3)) * np.array([1.0, 0.2, 1.0]) + np.array([0.0, 10.0, 0.0])
    d = target - o
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return np.concatenate([o, d], axis=1)


def assert_uvs_match(got, want, what, is_mesh_hit):
    """ids exact; mesh uvs bit-identical; sphere uvs within 1e-15; the checker choice equal on every hit at both
    M, except sphere hits on a cell edge (returned: how many there were)"""
    assert np.array_equal(got["ids"], want["ids"]), f"{what}: ids differ"
    hit = want["ids"] >= 0
    assert np.array_equal(got["prims"][hit], want["prims"][hit]), f"{what}: primitives differ"
    mesh = hit & is_mesh_hit(want)
    sphere = hit & ~mesh
    bad = np.flatnonzero(mesh)[~(got["uvs"][mesh] == want["uvs"][mesh]).all(axis=1)]
    assert len(bad) == 0, f"{what}: {len(bad)} mesh uvs differ, e.g. {got['uvs'][bad[:3]]} vs {want['uvs'][bad[:3]]}"
    np.testing.assert_allclose(got["uvs"][sphere], want["uvs"][sphere], rtol=0, atol=1e-15, err_msg=what)
    edges = 0
    for M in (M_PATH, M_WHITTED):
        flip = hit & (checker_on(got["uvs"], M) != checker_on(want["uvs"], M))
        edge = sphere & near_cell_edge(want["uvs"], M)
        assert not (flip & ~edge).any(), f"{what}: checker differs at M={M} on {np.flatnonzero(flip & ~edge)[:10]}"
        edges += int(edge.sum())
    return edges


def mesh_hit(want):
    return want["ids"] == MESH


# ---- 1. uv parity, ray by ray --------------------------------------------------------------------------------

@pytest.mark.parametrize("kind", KINDS)
def test_mesh_uvs_bit_identical_in_every_walk(gpu_api, ol, abi, kind):
    """a checkered mesh (3 200 triangles) with checkered spheres around it: every walk returns the oracle's
    texture coordinates bit for bit, and the checker makes the same choice on every hit"""
    W, H = 96, 54
    holder, verts = checkered_room(gpu_api, abi, 40, kind, W, H, seed=11)
    rng = np.random.default_rng(12)
    rays = np.concatenate([random_rays_in_room(rng, 8000), mesh_rays(verts, rng, 8000)])
    want = ol.intersect_rays(holder, rays)
    assert (want["ids"] == MESH).sum() > 6000
    with gpu_api.Scene(holder, all_trees=True) as sc:
        edges = [assert_uvs_match(sc.trace_rays(rays, use_bvh=mode), want, f"{kind} mesh, walk {mode}", mesh_hit)
                 for mode in WALKS]
        assert sc.info.double_texcoords == (kind != "float")
        assert sc.info.double_triangles == 0
    print(f"{kind}: sphere hits within 1e-9 of a cell edge: {edges}")
    if kind == "wide":
        assert (want["uvs"][want["ids"] == MESH] < 0).any(), "negative texture coordinates must be hit"


def test_sphere_uvs_in_every_walk(gpu_api, ol, abi):
    """a checkered sphere field: uvs within 1e-15 (atan2: libm vs CUDA), same checker choice on every hit"""
    W, H = 96, 54
    objs = checkered_field(gpu_api, abi, W, H)
    rays = random_rays_in_room(np.random.default_rng(13), 20000)
    want = ol.intersect_rays(objs, rays)
    with gpu_api.Scene(objs, all_trees=True) as sc:
        assert sc.info.double_texcoords == 0
        edges = [assert_uvs_match(sc.trace_rays(rays, use_bvh=mode), want, f"sphere field, walk {mode}",
                                  lambda w: np.zeros(len(w["ids"]), bool)) for mode in WALKS]
    print(f"sphere hits within 1e-9 of a cell edge: {edges}")


# ---- 2. sphere seam, poles and cell edges ----------------------------------------------------------------------

def test_sphere_seam_poles_and_cell_edges(gpu_api, ol, abi):
    """rays in the plane x = c.x onto the back of a sphere (n.x = +0 or -0: atan2 gives u = 1 or 0), rays along
    +-y through the centre (n.x = n.z = 0) and rays aimed so that u * M lands on a cell edge (k + 0.5): the same
    bar as ray by ray; every checker difference must sit within 1e-9 of an edge"""
    rng = np.random.default_rng(21)
    centres = np.array([[0.0, 0.0, 0.0], [0.0, 3.25, -7.5], [7.123456789, -2.2, 1.0 / 3.0], [-11.0, 5.5, -3.0]])
    radii = np.array([2.0, 1.7, 3.1, 0.9])
    objs = np.zeros(len(centres), dtype=abi.OBJECT_DTYPE)
    objs["flags"] = abi.M_DEFAULT | abi.M_CHECKERED
    objs["center"], objs["radius"] = centres, radii
    objs["color"] = 0.8
    rays, seam = [], []
    for c, r in zip(centres, radii):
        # seam: d.x = 0 and o.x = c.x; for c.x = 0 also o.x = d.x = -0.0, so that p.x - c.x = -0 and u ~ 0, not ~ 1
        for sx in (0.0, -0.0):
            for dy in np.linspace(-0.8, 0.8, 9):
                o = np.array([sx if c[0] == 0.0 else c[0], c[1] + dy * r, c[2] - 4.0 * r])
                d = np.array([sx, 0.0, 1.0])
                seam.append(len(rays))
                rays.append(np.concatenate([o, d]))
        # poles, from above and below
        rays.append(np.array([c[0], c[1] + 4.0 * r, c[2], 0.0, -1.0, 0.0]))
        rays.append(np.array([c[0], c[1] - 4.0 * r, c[2], 0.0, 1.0, 0.0]))
        # cell edges of u at both M: phi from u = atan2(n.x, n.z) / (2 pi') + 0.5, pi' = 3.14159265359 (raytracer.h:22)
        for M in (M_PATH, M_WHITTED):
            k = rng.integers(0, int(M), 200)
            u = (k + 0.5) / M
            phi = (u - 0.5) * 2.0 * 3.14159265359
            ny = rng.uniform(-0.9, 0.9, 200)
            s = np.sqrt(1.0 - ny * ny)
            n = np.stack([s * np.sin(phi), ny, s * np.cos(phi)], axis=1)
            o = c + 3.0 * r * n
            rays += list(np.concatenate([o, -n], axis=1))
    rays = np.array(rays)
    want = ol.intersect_rays(objs, rays)
    assert (want["ids"] >= 0).all()
    u_seam = want["uvs"][seam, 0]
    assert (np.abs(u_seam - np.round(u_seam)) < 1e-9).all(), "the seam rays must land on u ~ 0 or 1"
    assert (u_seam < 0.5).sum() == 2 * 9, "-0 on both spheres centred at x = 0"
    with gpu_api.Scene(objs, all_trees=True) as sc:
        edges = [assert_uvs_match(sc.trace_rays(rays, use_bvh=mode), want, f"seam/pole/edge rays, walk {mode}",
                                  lambda w: np.zeros(len(w["ids"]), bool)) for mode in WALKS]
    print(f"seam / pole / cell-edge rays: {len(rays)}, hits within 1e-9 of a cell edge per walk: {edges}")
    assert edges[0] > 0, "the cell-edge rays must land near edges"


# ---- 3. path tracer, sample by sample, and whole frames ------------------------------------------------------

def _path_sources(gpu_api, abi, W, H):
    return {
        "field": lambda: checkered_field(gpu_api, abi, W, H, count=300),
        "mesh-float": lambda: checkered_room(gpu_api, abi, 24, "float", W, H, seed=31)[0],
        "mesh-double": lambda: checkered_room(gpu_api, abi, 24, "double", W, H, seed=32)[0],
    }


@pytest.mark.parametrize("scene", ["field", "mesh-float", "mesh-double"])
def test_path_records_with_checkered_surfaces(gpu_api, ol, abi, scene):
    """trace_path (M = 100 000) path by path: vertex ids exact, radiance at the bar of the north-star check
    (FP32 colour arithmetic against double); a flipped checker factor would be a 2.3x error"""
    W, H = 96, 54
    src = _path_sources(gpu_api, abi, W, H)[scene]()
    cam = gpu_api.init_camera(W, H)
    desc = gpu_api.make_desc(W, H, 0, 1, max_depth=5)
    with gpu_api.Scene(src) as sc:
        for sample in (0, 3):
            got = sc.path_records(cam, desc, sample, n_vertices=3)
            want = ol.path_records(src, cam, W, H, sample, n_vertices=3)
            assert np.array_equal(got["ids"], want["ids"]), (scene, sample)
            np.testing.assert_allclose(got["radiance"], want["radiance"], rtol=2e-5, atol=1e-6,
                                       err_msg=f"{scene} sample {sample}")
    if scene != "field":
        assert (want["ids"] == MESH).sum() > W * H // 4


@pytest.mark.parametrize("scene", ["field", "mesh-float", "mesh-double"])
@pytest.mark.parametrize("mode", ["stochastic", "split", "offset"])
def test_render_with_checkered_surfaces(gpu_api, ol, abi, scene, mode):
    """render() against the oracle's render_sum: sums to 1e-3, ray_count exact -- the stochastic dielectric
    estimator, the reference's split (depth 5), and a sample range that does not start at 0"""
    W, H, SPP = 64, 36, 3
    src = _path_sources(gpu_api, abi, W, H)[scene]()
    cam = gpu_api.init_camera(W, H)
    begin = 5 if mode == "offset" else 0
    dielectric = 1 if mode == "split" else 0
    with gpu_api.Scene(src) as sc:
        _, acc, ctr = sc.render(cam, gpu_api.make_desc(W, H, begin, begin + SPP, max_depth=5, dielectric=dielectric),
                                want_accum=True)
    want, (rays, _) = ol.render_sum(src, cam, W, H, SPP, rng="philox", max_depth=5, sample_offset=begin,
                                    dielectric="split" if dielectric else "stochastic")
    assert ctr.rays == rays
    np.testing.assert_allclose(acc, want, rtol=1e-3, atol=1e-4)


# ---- 5. Whitted: the checker at M = 10 -------------------------------------------------------------------------

def close(a, b, rtol=1e-12):
    return np.abs(a - b).max() <= rtol * max(1.0, np.abs(b).max())


@pytest.mark.parametrize("depth", [0, 1, 5, 12])
@pytest.mark.parametrize("scene", ["field", "mesh-float", "mesh-double", "mesh-wide"])
def test_cast_rays_with_checkered_surfaces(gpu_api, ol, abi, scene, depth):
    """cast_ray (raytracer.c:556-641) ray by ray: calls exact, colours within 1e-12 (test_gpu_whitted.py's bar)"""
    W, H = 96, 54
    if scene == "field":
        src = checkered_field(gpu_api, abi, W, H)
        rays = random_rays_in_room(np.random.default_rng(41 + depth), 4000)
    else:
        src, verts = checkered_room(gpu_api, abi, 24, scene.split("-")[1], W, H, seed=42)
        rng = np.random.default_rng(43 + depth)
        rays = np.concatenate([random_rays_in_room(rng, 2000), mesh_rays(verts, rng, 2000)])
    with gpu_api.Scene(src) as sc:
        rgb, calls = sc.cast_rays(rays, max_depth=depth)
    ref_rgb, ref_calls = ol.cast_rays(src, rays, max_depth=depth)
    assert np.array_equal(calls.astype(np.int64), ref_calls)
    assert close(rgb, ref_rgb)


def test_cast_rays_on_checkered_spheres_vs_reference(gpu_api, ref_or_skip, abi):
    """the same against the unmodified reference's cast_ray"""
    ol = ref_or_skip
    objs = checkered_field(gpu_api, abi, 96, 54)
    rays = random_rays_in_room(np.random.default_rng(45), 3000)
    with gpu_api.Scene(objs) as sc:
        for depth in (0, 5):
            rgb, calls = sc.cast_rays(rays, max_depth=depth)
            ref_rgb, ref_calls = ol.ref_cast_rays(objs, rays, max_depth=depth)
            assert np.array_equal(calls.astype(np.int64), ref_calls)
            assert close(rgb, ref_rgb)


# ---- 6. every upload path keeps double texture coordinates ------------------------------------------------------

def _uv_probe(gpu_api, holder, rays):
    with gpu_api.Scene(holder) as sc:
        info = sc.info
        got = sc.trace_rays(rays)
    return got, info


def _assert_mesh_uvs(got, want, what, meshes):
    assert np.array_equal(got["ids"], want["ids"]), what
    m = np.isin(want["ids"], meshes)
    assert m.sum() > 1000, what
    assert np.array_equal(got["uvs"][m], want["uvs"][m]), what


def test_double_texcoords_survive_every_upload_path(gpu_api, ol, abi, monkeypatch):
    """a mesh above the narrowing threshold (10 368 triangles) with double texcoords goes up raw, with the raw
    upload forced, and with positions moved in double (tri64 and tex64 together): uvs bit-identical to the oracle
    and to each other; the same mesh with float texcoords keeps the narrowed float records"""
    from test_gpu_configs import _transformed_mesh
    W, H = 96, 54
    rng = np.random.default_rng(51)
    verts = gpu_api.heightfield_mesh(72, 20 * W / H * 0.9)
    verts["tex"] = texcoords("double", len(verts), rng)
    holder = checkered(abi, gpu_api.mesh_room(verts, W, H))
    rays = np.concatenate([random_rays_in_room(rng, 4000), mesh_rays(verts, rng, 4000)])
    want = ol.intersect_rays(holder, rays)
    got, info = _uv_probe(gpu_api, holder, rays)
    _assert_mesh_uvs(got, want, "pageable upload", [MESH])
    assert (info.double_texcoords, info.double_triangles) == (1, 0)
    monkeypatch.setenv("RTB_UPLOAD_NARROW", "0")
    raw, info = _uv_probe(gpu_api, holder, rays)
    monkeypatch.delenv("RTB_UPLOAD_NARROW")
    for k in ("ids", "prims", "points", "normals", "uvs"):
        assert np.array_equal(raw[k], got[k]), k
    assert info.double_texcoords == 1

    moved = _transformed_mesh(gpu_api, 72, W, H)
    moved["tex"] = texcoords("wide", len(moved), rng)
    holder_m = checkered(abi, gpu_api.mesh_room(moved, W, H))
    rays_m = np.concatenate([random_rays_in_room(rng, 4000), mesh_rays(moved, rng, 4000)])
    want_m = ol.intersect_rays(holder_m, rays_m)
    got_m, info = _uv_probe(gpu_api, holder_m, rays_m)
    _assert_mesh_uvs(got_m, want_m, "moved mesh", [MESH])
    hit = want_m["ids"] >= 0
    assert np.array_equal(got_m["points"][hit], want_m["points"][hit])
    assert (info.double_texcoords, info.double_triangles) == (1, 1)

    exact = verts.copy()
    exact["tex"] = exact["tex"].astype(np.float32).astype(np.float64)
    holder_f = checkered(abi, gpu_api.mesh_room(exact, W, H))
    want_f = ol.intersect_rays(holder_f, rays)
    got_f, info = _uv_probe(gpu_api, holder_f, rays)
    assert (info.double_texcoords, info.double_triangles) == (0, 0)
    _assert_mesh_uvs(got_f, want_f, "float texcoords", [MESH])


def test_float_and_double_texcoord_meshes_in_one_scene(gpu_api, ol, abi):
    """one mesh with float texcoords (uploaded narrowed, its doubles are its floats widened) and one with double
    texcoords (uploaded raw), in both orders: uvs of both meshes bit-identical to the oracle"""
    from test_gpu_configs import _with_second_mesh
    W, H = 96, 54
    rng = np.random.default_rng(61)
    exact = gpu_api.heightfield_mesh(72, 20 * W / H * 0.9)
    assert np.array_equal(exact["tex"], exact["tex"].astype(np.float32).astype(np.float64))
    doubles = gpu_api.heightfield_mesh(72, 12.0, half_d=10.0, y0=-4.0)  # a smaller patch above the first mesh
    doubles["tex"] = texcoords("double", len(doubles), rng)
    for first, second in ((exact, doubles), (doubles, exact)):
        holder = _with_second_mesh(abi, checkered(abi, gpu_api.mesh_room(first, W, H)), second)  # both checkered
        rays = np.concatenate([random_rays_in_room(rng, 3000), mesh_rays(first, rng, 3000),
                               mesh_rays(second, rng, 3000)])
        want = ol.intersect_rays(holder, rays)
        got, info = _uv_probe(gpu_api, holder, rays)
        for k in (MESH, holder.n - 1):
            _assert_mesh_uvs(got, want, f"mesh {k}", [k])
        assert (info.double_texcoords, info.double_triangles) == (1, 0)


def test_obj_loaded_mesh_keeps_float_texcoords(gpu_api, ol, abi, tmp_path):
    """an OBJ file stores floats (tinyobj parses `float`): whatever texcoords the writer was given, the loaded
    mesh keeps the compact float records and its uvs equal the oracle's"""
    W, H = 96, 54
    verts = gpu_api.heightfield_mesh(24, 20 * W / H * 0.98)
    verts["tex"] = texcoords("double", len(verts), np.random.default_rng(71))
    path = str(tmp_path / "mesh.obj")
    gpu_api.write_obj(path, verts)
    loaded = gpu_api.load_obj(path)
    holder = checkered(abi, gpu_api.mesh_room(loaded, W, H))
    rng = np.random.default_rng(72)
    rays = np.concatenate([random_rays_in_room(rng, 2000), mesh_rays(loaded, rng, 2000)])
    want = ol.intersect_rays(holder, rays)
    got, info = _uv_probe(gpu_api, holder, rays)
    assert (info.double_texcoords, info.double_triangles) == (0, 0)
    _assert_mesh_uvs(got, want, "OBJ mesh", [MESH])


def test_sharded_upload_of_double_texcoords(gpu_api, ol, abi):
    """the sharded upload (every rank marshals its share, the flags are max-reduced, tex64 all-gathered): the
    two-GPU frame of a checkered double-texcoord mesh equals the one-GPU frame and the oracle's"""
    if gpu_api.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    W, H, SPP = 96, 54, 2
    holder, _ = checkered_room(gpu_api, abi, 96, "double", W, H, seed=81)  # 18 432 triangles > 2 x 4096
    cam = gpu_api.init_camera(W, H)
    desc = gpu_api.make_desc(W, H, 0, SPP, max_depth=5)
    with gpu_api.Scene(holder) as sc:
        assert sc.info.double_texcoords == 1
        _, acc0, c0 = sc.render(cam, desc, want_accum=True)
    with gpu_api.Comm.local(2) as comm:
        _, acc1, c1 = comm.render_host(holder, cam, desc, want_accum=True)
    assert c1.rays == c0.rays and c1.prim_tests == c0.prim_tests
    np.testing.assert_allclose(acc1, acc0, rtol=2e-5, atol=1e-5)
    want, (rays, _) = ol.render_sum(holder, cam, W, H, SPP, rng="philox", dielectric="stochastic", max_depth=5)
    assert c0.rays == rays
    np.testing.assert_allclose(acc0, want, rtol=1e-3, atol=1e-4)


def test_render_of_a_double_texcoord_mesh(gpu_api, ol, abi):
    """the visible symptom: a checkered mesh with double texcoords, rendered, against the oracle at 1e-3"""
    W, H, SPP = 96, 54, 4
    holder, _ = checkered_room(gpu_api, abi, 40, "double", W, H, seed=91)
    cam = gpu_api.init_camera(W, H)
    with gpu_api.Scene(holder) as sc:
        info = sc.info
        _, acc, ctr = sc.render(cam, gpu_api.make_desc(W, H, 0, SPP, max_depth=5), want_accum=True)
    want, (rays, _) = ol.render_sum(holder, cam, W, H, SPP, rng="philox", dielectric="stochastic", max_depth=5)
    assert ctr.rays == rays
    np.testing.assert_allclose(acc, want, rtol=1e-3, atol=1e-4)
    assert info.double_texcoords == 1
