"""The BVH checker (bvh_check.py) on a hand-built tree: the tree passes, and each kind of fault is reported.

The tree is encoded here the way the build encodes it (k_marshal_*, k_build_params, k_emit4, build_scene's far_t),
over 12 spheres and a mesh of 6 triangles with double vertices and texture coordinates (so tri64, tex and tex64 exist),
two of the spheres oversized; leaf_max 2, three BVH4 levels.  test_gpu_bvh_build.py runs the same mutations on real
dumps.
"""
import numpy as np
import pytest

import bvh_check as bc

def geometry():
    """prim k (k = 0..15) sits at x = 3k; even k a sphere of radius 1, odd k a small triangle; two walls of radius 1e4
    first in object order"""
    parts = [("sphere", 0, (0.0, 0.0, -1e4 - 50.0, 1e4)), ("sphere", 1, (0.0, 1e4 + 50.0, 0.0, 1e4))]
    tris, uvs = [], []
    for k in range(16):
        x = 3.0 * k
        if k % 2 == 0 and len(parts) < 10:
            parts.append(("sphere", len(parts), (x, 0.5, -0.25, 1.0)))
        else:
            base = np.array([[x, 0.0, 0.0], [x + 0.7, 0.1, 0.3], [x + 0.2, 0.9, -0.4]]) * (1.0 + 2.0 ** -40)
            tris.append(base.reshape(9))
            uvs.append(np.array([0.1, 0.2, 0.3, 0.4, 0.5, 0.6]) * (1.0 + 2.0 ** -35))
    parts.append(("mesh", len(parts), np.array(tris), np.array(uvs)))
    return bc.Geometry.concat(parts)


def _leaf_ref(first, count):
    return ~((first << 3) | (count - 1))


def encode_node(lo, hi, refs, dummy):
    """k_emit4's compressed node from padded float slot boxes lo / hi [4, 3] (unused rows ignored)"""
    used = [r is not None for r in refs]
    w = np.zeros(16, np.uint32)
    org = np.array([min(lo[k][a] for k in range(4) if used[k]) for a in range(3)], np.float32)
    nhi = np.array([max(hi[k][a] for k in range(4) if used[k]) for a in range(3)], np.float32)
    cells = []
    for a in range(3):
        ext = float(nhi[a]) - float(org[a])
        e = int(np.frexp(ext / 255.0)[1]) if ext > 0 else -126
        e = max(-126, min(127, e))
        while 2.0 ** e * 255.0 < ext and e < 127:
            e += 1
        cells.append(np.float32(2.0 ** e))
    w[0:3] = org.view(np.uint32)
    w[3] = np.float32(cells[0]).view(np.uint32)
    w[14], w[15] = np.float32(cells[1]).view(np.uint32), np.float32(cells[2]).view(np.uint32)
    w[4:8] = np.array([r if r is not None else dummy for r in refs], np.int32).view(np.uint32)
    for a in range(3):
        ql = qh = 0
        for k in range(4):
            l, h = 255, 0
            if used[k]:
                c = float(cells[a])
                l = int(min(max(np.floor((float(lo[k][a]) - float(org[a])) / c), 0), 255))
                h = int(min(max(np.ceil((float(hi[k][a]) - float(org[a])) / c), 0), 255))
            ql |= l << (8 * k)
            qh |= h << (8 * k)
        w[8 + a], w[11 + a] = ql, qh
    return w


def build(geom):
    """-> (tree dict as api.Scene.tree() returns it, scene info stand-in)"""
    big = bc.choose_big(geom)
    keep = np.setdiff1d(np.arange(len(geom.is_sphere)), big)
    x = np.where(geom.is_sphere[keep], geom.sph[keep, 0], geom.tri[keep, 0])
    gid = keep[np.argsort(x, kind="stable")]  # BVH order: along x
    N = len(gid)
    sph = geom.is_sphere[gid]
    prims = np.zeros((N + 1, 12), np.uint32)
    prims[:N, :8] = np.where(sph[:, None], bc._sphere_words(geom.sph[gid]), 0)
    prims[~np.r_[sph, True], :9] = geom.tri[gid[~sph]].astype(np.float32).view(np.uint32)
    prims[:N, 9] = gid
    prims[:N, 10] = geom.obj[gid].astype(np.uint32) | np.where(sph, np.uint32(bc.SPHERE_BIT), np.uint32(0))
    c, r = geom.sph[gid, :3], np.abs(geom.sph[gid, 3:4])
    p = geom.tri[gid].reshape(-1, 3, 3)
    blo = np.where(sph[:, None], bc.round_down(c - r), bc.round_down(p).min(axis=1)).astype(np.float32)
    bhi = np.where(sph[:, None], bc.round_up(c + r), bc.round_up(p).max(axis=1)).astype(np.float32)
    lo, hi = blo.min(axis=0), bhi.max(axis=0)
    d = hi.astype(np.float64) - lo.astype(np.float64)
    diag = float(np.sqrt((d * d).sum()))
    g_lo, g_hi = (lo - diag).astype(np.float32), (hi + diag).astype(np.float32)
    pad = np.float32((float(np.abs(np.r_[g_lo, g_hi]).astype(np.float64).max()) + 3.0 * diag * 1.7320508) / 1048576.0)
    # leaves of two along BVH order: root = 3 leaves + node 1, node 1 = 3 leaves + node 2, node 2 = 2 leaves
    dummy = _leaf_ref(N, 1)
    layout = [[(0, 2), (2, 2), (4, 2), 1], [(6, 2), (8, 2), (10, 2), 2], [(12, 2), (14, 2), None, None]]
    span = {0: (0, 16), 1: (6, 16), 2: (12, 16)}
    nodes = []
    for slots in layout:
        slo, shi, refs = [], [], []
        for s in slots:
            if s is None:
                slo.append(np.zeros(3, np.float32)), shi.append(np.zeros(3, np.float32)), refs.append(None)
                continue
            a, b = (s[0], s[0] + s[1]) if isinstance(s, tuple) else span[s]
            slo.append(blo[a:b].min(axis=0) - pad)
            shi.append(bhi[a:b].max(axis=0) + pad)
            refs.append(_leaf_ref(*s) if isinstance(s, tuple) else s)
        nodes.append(encode_node(slo, shi, refs, dummy))
    tri64 = np.zeros((N + 1, 9))
    tri64[:N][~sph] = geom.tri[gid[~sph]]
    tex64 = np.where(sph[:, None], 0.0, geom.uv[gid])
    info = type("Info", (), {})()
    for k, v in dict(n_prims=N, n_big=len(big), n_nodes4q=3, n_nodes4=0, n_nodes2=0, root_ref=0, leaf_max=2, depth4=3,
                     walks_bvh4=1, has_tex=1, has_tri64=1, has_tex64=1, scene_lo=lo, scene_hi=hi, guard_lo=g_lo,
                     guard_hi=g_hi, pad=pad).items():
        setattr(info, k, v)
    gd = 0.0
    for k in range(3):
        e = float(g_hi[k]) - float(g_lo[k])
        gd += e * e
    gd = float(np.sqrt(gd))
    far = min(300.0 * gd, float(np.sqrt(2.0 * float(r[sph].min()) * float(pad) * 9007199254740992.0 / 16.0)) - gd)
    info.far_t = np.float32(max(far, 0.0))
    bigrec = np.zeros((len(big), 12), np.uint32)
    bigrec[:, :8] = bc._sphere_words(geom.sph[big])
    bigrec[:, 9] = big
    bigrec[:, 10] = geom.obj[big].astype(np.uint32) | np.uint32(bc.SPHERE_BIT)
    cp = np.zeros((len(big), 8), np.float32)
    cp[:, :4] = geom.sph[big].astype(np.float32)
    cp[:, 4] = np.abs(cp[:, :4]).sum(axis=1) * np.float32(1.0000005)
    tree = dict(info=info, nodes4q=np.array(nodes), nodes4=np.zeros((0, 32), np.uint32),
                nodes=np.zeros((0, 16), np.uint32), prims=prims, big=bigrec, big_fp32=cp, tri64=tri64,
                tex=tex64.astype(np.float32), tex64=tex64)
    scene_info = type("SceneInfo", (), dict(n_bvh_prims=N, n_big_prims=len(big), n_bvh_nodes=3, bvh4_depth=3,
                                            bvh_depth=8))()
    return tree, scene_info


def copy(tree):
    return {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in tree.items()}


def test_hand_built_tree_passes():
    geom = geometry()
    tree, si = build(geom)
    assert tree["info"].n_big == 2 and tree["info"].n_prims == 16
    bc.check(tree, geom, si)
    assert not bc.same_canonical(bc.canonical(tree), bc.canonical(copy(tree)))


def lower_qhi_uncovering(tree, geom):
    """lower one qhi by one cell where that uncovers a primitive of the slot; -> (node, slot, axis)"""
    plo, phi = bc.prim_bounds(tree, geom)
    org, cell, refs, qlo, qhi = bc.decode4q(tree["nodes4q"])
    pad = float(tree["info"].pad)
    for n in range(len(refs)):
        for s in range(4):
            if refs[n, s] >= 0 or qhi[n, s, 0] == 0:
                continue
            first, count = bc.leaf_decode(refs[n, s])
            if first >= tree["info"].n_prims:
                continue
            for a in range(3):
                new = float(org[n, a]) + (qhi[n, s, a] - 1) * float(cell[n, a])
                if new < phi[first:first + count, a].max() + pad / 2:
                    word = 11 + a
                    tree["nodes4q"][n, word] -= np.uint32(1 << (8 * s))
                    return n, s, a
    raise AssertionError("no qhi whose lowering uncovers a primitive")


def mutate(kind, tree, geom):
    q, prims = tree["nodes4q"], tree["prims"]
    if kind == "qhi lowered by one cell":
        lower_qhi_uncovering(tree, geom)
    elif kind == "leaf slot emptied":
        N = tree["info"].n_prims
        q[0, 5] = np.array([_leaf_ref(N, 1)], np.int32).view(np.uint32)[0]
        for a in range(3):
            q[0, 8 + a] |= np.uint32(0xFF << 8)
            q[0, 11 + a] &= np.uint32(~(0xFF << 8) & 0xFFFFFFFF)
    elif kind == "leaf range duplicated":
        q[0, 5] = q[0, 4]
    elif kind == "prims records swapped":
        prims[[0, 15]] = prims[[15, 0]]
    elif kind == "tri64 bit flipped":
        row = int(np.flatnonzero((prims[:-1, 10] & bc.SPHERE_BIT) == 0)[2])
        tree["tri64"][row:row + 1].view(np.uint64)[0, 4] ^= np.uint64(1 << 17)
    elif kind == "wrong oversized pick":
        tree["big"][1] = prims[3]
        tree["big_fp32"][1, :4] = bc.f32(prims[3, :8]).view(np.float64).astype(np.float32)
    else:
        raise ValueError(kind)


MUTATIONS = ["qhi lowered by one cell", "leaf slot emptied", "leaf range duplicated", "prims records swapped",
             "tri64 bit flipped", "wrong oversized pick"]


@pytest.mark.parametrize("kind", MUTATIONS)
def test_checker_reports_each_fault(kind):
    geom = geometry()
    tree, si = build(geom)
    mutate(kind, tree, geom)
    with pytest.raises(bc.BuildError):
        bc.check(tree, geom, si)


def test_choose_big_rules():
    """threshold 32 x median, at most 32, largest first with ties to the lower index, negative radii by |r|, and the
    median taken over mesh samples too"""
    def spheres(r):
        return bc.Geometry.concat([("sphere", i, (0.0, 0.0, 0.0, v)) for i, v in enumerate(r)])
    r = np.ones(100)
    r[[5, 7, 9]] = [33.0, 32.0, -40.0]
    assert list(bc.choose_big(spheres(r))) == [5, 9]
    r = np.ones(200)
    r[10:60] = 100.0  # 50 equal candidates, median 1: the first 32 by index
    assert list(bc.choose_big(spheres(r))) == list(range(10, 42))
    r[70] = -1000.0  # the largest |r| goes first
    assert list(bc.choose_big(spheres(r))) == list(range(10, 41)) + [70]
    # 3 spheres of radius 10 and a mesh of 4096 triangles of half-extent 0.1: step 2, each sample counted twice
    tri = np.zeros((4096, 9))
    tri[:, 3] = 0.2
    g = bc.Geometry.concat([("sphere", 0, (0, 0, 0, 10.0)), ("sphere", 1, (0, 0, 0, 3.3)),
                            ("sphere", 2, (0, 0, 0, 3.1)), ("mesh", 3, tri, np.zeros((4096, 6)))])
    assert list(bc.choose_big(g)) == [0, 1]
    assert list(bc.choose_big(g, ratio=0.0)) == [0, 1, 2]
