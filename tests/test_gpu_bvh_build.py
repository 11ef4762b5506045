"""The scene build (csrc/rtb_scene.cu) read back through rtb_scene_tree and checked primitive by primitive.

Rays sample a tree thinly: a triangle missing from every leaf, a leaf range off by one, a tri64 row reordered with
the wrong index or a quantised box one cell short shows up as a rare wrong hit.  Here every dump goes through
bvh_check.check (records, oversized list, topology, boxes with pad / 2 to spare, build parameters) on reference-size
scenes, upload paths, degenerate geometry, tiny trees, oversized-list edges, trees at the stack bound and every leaf
size; builds are compared in canonical form (BVH4 node indices come from atomics).
"""
import os

import numpy as np
import pytest

import bvh_check as bc
from conftest import random_rays_in_room
from test_gpu_wavefront_hits import (assert_same_records, chain_objects, degenerate_mesh, mesh_room,
                                     nested_spheres)

pytestmark = pytest.mark.gpu

C3_W, C3_H = 1920, 1080


def built(gpu_api, source, all_trees=False, ratio=32.0):
    """build, dump, check; -> (tree, scene info)"""
    with gpu_api.Scene(source, all_trees=all_trees) as sc:
        tree, info = sc.tree(), sc.info
    bc.check(tree, bc.geometry(source), info, ratio)
    return tree, info


def spheres(abi, centers, radii):
    objs = np.zeros(len(radii), dtype=abi.OBJECT_DTYPE)
    objs["flags"] = abi.M_DEFAULT
    objs["center"] = centers
    objs["radius"] = radii
    objs["color"] = (0.5, 0.5, 0.5)
    return objs


def mesh_holder(abi, tri, uv=None):
    tri = np.asarray(tri, np.float64).reshape(-1, 9)
    verts = np.zeros(3 * len(tri), dtype=abi.VERTEX_DTYPE)
    verts["pos"] = tri.reshape(-1, 3)
    if uv is not None:
        verts["tex"] = np.asarray(uv).reshape(-1, 2)
    return abi.SceneHolder.build([("mesh", verts, abi.M_DEFAULT, (0.5, 0.5, 0.5), (0.0, 0.0, 0.0))])


def c3_verts(gpu_api):
    return gpu_api.heightfield_mesh(708, 20 * C3_W / C3_H * 0.98)


MATRIX = np.array([[0.93 * np.cos(0.12), 0, np.sin(0.12), 0.3], [0, 1.1, 0, 0.7], [-np.sin(0.12), 0, np.cos(0.12), -1.3],
                   [0, 0, 0, 1]])


# ---- reference-size scenes -------------------------------------------------------------------------------------

def test_c1_with_its_oversized_walls(gpu_api):
    tree, info = built(gpu_api, gpu_api.scene_default(320, 180), all_trees=True)
    assert info.n_big_prims == 6 and tree["info"].walks_bvh4


@pytest.mark.parametrize("n", [2000, 10000])
def test_sphere_fields(gpu_api, n):
    built(gpu_api, gpu_api.scene_sphere_field(n, 192, 108), all_trees=n == 2000)


@pytest.mark.parametrize("variant", ["plain", "apply_matrix", "double_texcoords"])
def test_c3_mesh_room(gpu_api, variant):
    verts = c3_verts(gpu_api)
    if variant == "apply_matrix":
        gpu_api.apply_matrix(verts, MATRIX)
    elif variant == "double_texcoords":
        verts["tex"] = verts["tex"] * (1.0 + 2.0 ** -33) + 1e-9
    tree, info = built(gpu_api, gpu_api.mesh_room(verts, C3_W, C3_H), all_trees=variant == "plain")
    assert info.n_triangles == 1002528
    assert (tree["tri64"] is not None, tree["tex64"] is not None) == (variant == "apply_matrix", variant == "double_texcoords")


def test_mesh_across_the_staging_chunk(gpu_api, abi, monkeypatch):
    """2 101 250 triangles: two 2^21-triangle upload pieces; one coordinate of the second is not a float, so the first
    goes up narrowed and is widened into tri64 (k_widen_tri64), the second raw"""
    verts = gpu_api.heightfield_mesh(1025, 34.0)
    verts["pos"][3 * ((1 << 21) + 777) + 1, 1] += 2.0 ** -30
    monkeypatch.setenv("RTB_UPLOAD_NARROW", "1")
    holder = abi.SceneHolder.build([("mesh", verts, abi.M_DEFAULT, (0.5, 0.5, 0.5), (0.0, 0.0, 0.0))])
    tree, info = built(gpu_api, holder)
    assert info.n_triangles == 2101250 and info.double_triangles == 1 and tree["tri64"] is not None


# ---- degenerate geometry ---------------------------------------------------------------------------------------

def test_degenerate_and_nested(gpu_api, abi):
    rng = np.random.default_rng(8)
    for doubles in (False, True):
        holder, _ = degenerate_mesh(gpu_api, abi, doubles, rng)
        built(gpu_api, holder, all_trees=True)
    built(gpu_api, nested_spheres(abi, rng)[0], all_trees=True)
    built(gpu_api, spheres(abi, np.tile([1.0, 2.0, 3.0], (1000, 1)), np.full(1000, 0.5)), all_trees=True)


@pytest.mark.parametrize("shape", ["flat", "collinear", "offset 1e6", "scale 1e-3", "scale 1e3"])
def test_flat_collinear_offset_and_scaled(gpu_api, abi, shape):
    rng = np.random.default_rng(9)
    c = rng.uniform(-20, 20, (3000, 3))
    r = rng.uniform(0.05, 0.5, 3000)
    if shape == "collinear":
        c = np.outer(rng.uniform(-20, 20, 3000), [1.0, 0.5, -0.25])
    if shape == "flat":  # triangles in the plane y = 1: zero extent on one axis
        tri = rng.uniform(-20, 20, (3000, 3, 3))
        tri[:, :, 1] = 1.0
        built(gpu_api, mesh_holder(abi, tri), all_trees=True)
        c[:, 1], r[:] = 1.0, 0.0
    scale, off = {"offset 1e6": (1.0, 1e6), "scale 1e-3": (1e-3, 0.0), "scale 1e3": (1e3, 0.0)}.get(shape, (1.0, 0.0))
    built(gpu_api, spheres(abi, c * scale + off, r * scale), all_trees=True)


# ---- tiny trees ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 9])
def test_tiny_trees(gpu_api, abi, n):
    rng = np.random.default_rng(n)
    tree, info = built(gpu_api, spheres(abi, rng.uniform(-5, 5, (n, 3)), np.full(n, 0.3)), all_trees=True)
    assert tree["info"].n_prims == n and (n > 1) == (tree["info"].root_ref == 0)  # spheres: one per leaf
    tri = rng.uniform(-5, 5, (n, 3, 3))
    tree, info = built(gpu_api, mesh_holder(abi, tri), all_trees=True)
    assert (n > 2) == (tree["info"].root_ref == 0)  # meshes: two per leaf; N <= 2 is a root leaf and no nodes
    assert (len(tree["nodes4q"]) == 0) == (n <= 2)


def test_empty_tree(gpu_api, monkeypatch):
    monkeypatch.setenv("RTB_BIG_RATIO", "0")
    objs = gpu_api.scene_default(320, 180)[:20].copy()
    tree, info = built(gpu_api, objs, ratio=0.0)
    assert tree["info"].n_prims == 0 and info.n_big_prims == 20 and tree["info"].root_ref == bc.REF_NONE


# ---- the oversized list ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("n_big", [31, 32, 33, 48])
@pytest.mark.parametrize("radii", ["distinct", "equal", "negative"])
def test_oversized_candidates(gpu_api, abi, n_big, radii):
    rng = np.random.default_rng(n_big)
    c = rng.uniform(-30, 30, (500, 3))
    r = np.full(500, 0.5)
    pick = rng.choice(500, n_big, replace=False)
    r[pick] = {"distinct": rng.uniform(100, 1000, n_big), "equal": np.full(n_big, 200.0),
               "negative": -rng.uniform(100, 1000, n_big)}[radii]
    tree, info = built(gpu_api, spheres(abi, c, r))
    assert info.n_big_prims == min(n_big, 32)


def test_oversized_median_decided_by_a_mesh(gpu_api, abi):
    """4 spheres and 20 000 triangles: the median is a mesh sample (every 9th triangle, each counted 9 times)"""
    rng = np.random.default_rng(10)
    tri = rng.uniform(-20, 20, (20000, 1, 3)) + rng.uniform(-0.05, 0.05, (20000, 3, 3))
    verts = np.zeros(60000, dtype=abi.VERTEX_DTYPE)
    verts["pos"] = tri.reshape(-1, 3)
    items = [("sphere", s) for s in spheres(abi, rng.uniform(-5, 5, (4, 3)), [0.5, 1.2, 1.4, 30.0])]
    holder = abi.SceneHolder.build(items + [("mesh", verts, abi.M_DEFAULT, (0.5,) * 3, (0.0,) * 3)])
    want = bc.choose_big(bc.geometry(holder))
    assert 0 < len(want) < 4
    built(gpu_api, holder)


# ---- trees at the traversal-stack bound ------------------------------------------------------------------------

@pytest.mark.parametrize("depth,walks_bvh4", [(60, 1), (61, 0), (62, 0)])
def test_chains_at_the_stack_bound(gpu_api, abi, depth, walks_bvh4):
    for all_trees in (False, True):
        tree, info = built(gpu_api, chain_objects(abi, depth), all_trees=all_trees)
        assert tree["info"].walks_bvh4 == walks_bvh4 and info.bvh_depth == depth
        # the node count is the walked tree's: the BVH2 of a chain has one node per level
        assert info.n_bvh_nodes == (len(tree["nodes4q"]) if walks_bvh4 else depth)


# ---- every leaf size -------------------------------------------------------------------------------------------

@pytest.mark.parametrize("leaf_max", [1, 3, 5, 8])
def test_leaf_sizes(gpu_api, abi, monkeypatch, leaf_max):
    """RTB_LEAF_MAX 1..8 (the top of the 3-bit count field): the trees check out and the trace kernel on them equals
    the GPU brute force"""
    monkeypatch.setenv("RTB_LEAF_MAX", str(leaf_max))
    rng = np.random.default_rng(leaf_max)
    holder, _ = mesh_room(gpu_api, grid=60)
    for source in (holder, gpu_api.scene_sphere_field(3000, 96, 54)):
        rays = random_rays_in_room(rng, 20000)
        with gpu_api.Scene(source, all_trees=True) as sc:
            tree, info = sc.tree(), sc.info
            got = sc.trace_rays_wf(rays)[0]
            brute = sc.trace_rays(rays, use_bvh=0)
        bc.check(tree, bc.geometry(source), info)
        assert tree["info"].leaf_max == leaf_max
        refs = tree["nodes4q"][:, 4:8].view(np.int32).astype(np.int64)
        count = bc.leaf_decode(refs[refs < 0])[1]
        assert count.max() <= leaf_max and (leaf_max < 5 or count.max() >= 5)
        assert_same_records(got, brute, f"leaf_max {leaf_max}")


# ---- determinism -----------------------------------------------------------------------------------------------

def canonical(gpu_api, source, all_trees=False):
    with gpu_api.Scene(source, all_trees=all_trees) as sc:
        return bc.canonical(sc.tree())


def test_builds_are_reproducible(gpu_api, abi, monkeypatch):
    """two builds of one scene, the narrowed and the raw upload of a float mesh, and Object and SceneObject records
    of one sphere scene give the same canonical dump"""
    holder, _ = mesh_room(gpu_api, grid=120)
    a, b = canonical(gpu_api, holder, True), canonical(gpu_api, holder, True)
    assert not bc.same_canonical(a, b)
    monkeypatch.setenv("RTB_UPLOAD_NARROW", "0")
    raw = canonical(gpu_api, holder, True)
    monkeypatch.setenv("RTB_UPLOAD_NARROW", "1")
    narrowed = canonical(gpu_api, holder, True)
    assert not bc.same_canonical(raw, a) and not bc.same_canonical(narrowed, a)
    objs = gpu_api.scene_sphere_field(2000, 96, 54)
    assert not bc.same_canonical(canonical(gpu_api, objs), canonical(gpu_api, abi.SceneHolder.from_objects(objs)))


def test_sharded_build_equals_one_gpu(gpu_api):
    """with two GPUs: each rank's build from the sharded upload + all-gather equals the one-GPU dump"""
    if gpu_api.device_count() < 2:
        pytest.skip("needs two GPUs")
    verts = c3_verts(gpu_api)
    gpu_api.apply_matrix(verts, MATRIX)
    holder = gpu_api.mesh_room(verts, C3_W, C3_H)
    want = canonical(gpu_api, holder)
    with gpu_api.Comm.local(2) as comm, comm.scene(holder) as ms:
        for k in range(2):
            sc = gpu_api.Scene.__new__(gpu_api.Scene)
            sc._cu, sc._h, sc.device = comm._cu, gpu_api.C.c_void_p(ms._handles[k]), k
            got = bc.canonical(sc.tree())
            sc._h = gpu_api.C.c_void_p()  # the handle belongs to the MultiScene
            assert not bc.same_canonical(got, want), f"rank {k}"


# ---- the checker on real dumps ---------------------------------------------------------------------------------

@pytest.mark.parametrize("kind", ["qhi lowered by one cell", "leaf slot emptied", "leaf range duplicated",
                                  "prims records swapped", "tri64 bit flipped", "wrong oversized pick"])
def test_checker_reports_faults_in_a_real_dump(gpu_api, abi, kind):
    import test_bvh_check as hand
    verts = gpu_api.heightfield_mesh(40, 30.0)
    gpu_api.apply_matrix(verts, MATRIX)
    holder = gpu_api.mesh_room(verts, 96, 54)
    with gpu_api.Scene(holder) as sc:
        tree, info = sc.tree(), sc.info
    geom = bc.geometry(holder)
    bc.check(tree, geom, info)
    if kind == "prims records swapped":
        tree["prims"][[0, tree["info"].n_prims - 1]] = tree["prims"][[tree["info"].n_prims - 1, 0]]
    else:
        hand.mutate(kind, tree, geom)
    with pytest.raises(bc.BuildError):
        bc.check(tree, geom, info)


# ---- non-finite geometry ---------------------------------------------------------------------------------------

def _nan_sources(gpu_api, abi, where, value):
    objs = gpu_api.scene_sphere_field(300, 64, 36)
    if where == "sphere centre":
        objs["center"][100, 1] = value
    elif where == "sphere radius":
        objs["radius"][100] = value
    if where.startswith("sphere"):
        return {"Object": objs, "SceneObject": abi.SceneHolder.from_objects(objs)}
    verts = gpu_api.heightfield_mesh(100, 20.0)
    verts["pos"][3 * 5000 + 2, 1] = value
    return {"narrowed": verts, "raw": verts}


@pytest.mark.parametrize("where", ["sphere centre", "sphere radius", "triangle vertex"])
def test_nan_geometry_is_rejected(gpu_api, abi, monkeypatch, where):
    """NaN anywhere in the geometry is "non-finite geometry" (fminf / fmaxf of the box reduction used to drop it, and
    a NaN radius reached choose_big's sort), through both ways a primitive arrives"""
    for path, src in _nan_sources(gpu_api, abi, where, np.nan).items():
        if where == "triangle vertex":
            monkeypatch.setenv("RTB_UPLOAD_NARROW", "1" if path == "narrowed" else "0")
            src = abi.SceneHolder.build([("mesh", src, abi.M_DEFAULT, (0.5,) * 3, (0.0,) * 3)])
        with pytest.raises(gpu_api.RtbError, match="non-finite geometry"):
            gpu_api.Scene(src)
    with gpu_api.Scene(gpu_api.scene_sphere_field(300, 64, 36)) as sc:  # the device is fine afterwards
        assert sc.info.n_bvh_prims > 0


@pytest.mark.parametrize("value", [np.inf, -np.inf, 1e39, -1e39])
def test_infinite_and_out_of_float_range_geometry(gpu_api, abi, value):
    """pinned: a tree primitive whose float box reaches +-inf (a coordinate +-inf or beyond FLT_MAX) is rejected; a
    sphere whose radius is +-inf or beyond FLT_MAX is oversized and goes to the every-ray list, which has no box"""
    for where in ("sphere centre", "triangle vertex"):
        for src in _nan_sources(gpu_api, abi, where, value).values():
            if where == "triangle vertex":
                src = abi.SceneHolder.build([("mesh", src, abi.M_DEFAULT, (0.5,) * 3, (0.0,) * 3)])
            with pytest.raises(gpu_api.RtbError, match="non-finite geometry"):
                gpu_api.Scene(src)
    objs = _nan_sources(gpu_api, abi, "sphere radius", value)["Object"]
    tree, info = built(gpu_api, objs)
    assert 100 in tree["big"][:, 9]
