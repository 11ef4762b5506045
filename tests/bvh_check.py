"""Exact checks of a built scene (rtb_scene_tree, include/rtb200.h) against the caller's geometry, in numpy.

check(tree, geom) raises BuildError naming the node, slot or primitive at fault.  It holds the build to:
  - records: prims[0..N) is a permutation of the primitives outside the oversized list, each record equal to its
    primitive (sphere doubles bit for bit, triangle floats rounded to nearest, tri64 / tex64 rows the caller's doubles,
    tex the rounded floats), record N and tri64 row N all zero; the oversized list equal to choose_big() below, and
    each FP32 copy's bound A_c at least |cx| + |cy| + |cz| + |r|, exactly;
  - topology of every tree present: each node reached from the root exactly once, leaf ranges of 1..leaf_max
    primitives that partition [0, N), a node's slot ranges disjoint with a contiguous union; for the BVH4 also empty
    slots (qlo 255, qhi 0, the dummy leaf (N, 1)), no inner slot in a node with fewer than four used slots, and a
    breadth-first node order (a node's inner children consecutive and after it, levels as index blocks);
  - boxes: per compressed node and axis a power-of-two cell in the normal float range; every used slot's box (decoded
    org + q * cell for the compressed BVH4, the floats of the uncompressed BVH4 and BVH2) contains each primitive of
    its range with pad / 2 to spare on every side, and a compressed slot contains the uncompressed slot of the same
    node.  The decoded bounds are exact in float64: org is a float and org + q * cell spans under 40 bits;
  - build parameters: the scene box bit for bit; guard box and pad to 1e-6 (the device may contract them into FMA);
    far_t by the host formula of build_scene.

What does NOT hold, and is not asserted: decoded boxes do not nest (a child's quantised slot may overshoot its parent's
by a cell), BVH4 node indices are not reproducible (atomics; compare canonical() forms), slot order is not range
order, and a BVH2-fallback scene's BVH4 is incomplete (only the walked tree is held to the node count and depth).
"""
import ctypes as C
from fractions import Fraction

import numpy as np

REF_NONE = 0x7FFFFFFF
SPHERE_BIT = 0x80000000
STACK_SIZE = 64


class BuildError(AssertionError):
    pass


def _fail(msg):
    raise BuildError(msg)


# ---- the caller's geometry ----------------------------------------------------------------------------------------

class Geometry:
    """The caller's primitives in the reference's loop order (object order, then triangle order): gid = row.
    is_sphere [P] bool, obj [P], sph [P, 4] (cx, cy, cz, r), tri [P, 9], uv [P, 6] (float64, zero where unused),
    meshes: (first gid, triangles) per mesh object with triangles, in object order."""

    def __init__(self, is_sphere, obj, sph, tri, uv, meshes):
        self.is_sphere, self.obj, self.sph, self.tri, self.uv = is_sphere, obj, sph, tri, uv
        self.meshes = list(meshes)

    @staticmethod
    def concat(parts):
        """parts: ("sphere", obj, (cx, cy, cz, r)) or ("mesh", obj, tri [T, 9], uv [T, 6]), in object order"""
        rows, meshes, gid = [], [], 0
        for p in parts:
            if p[0] == "sphere":
                rows.append((True, p[1], np.asarray(p[2], np.float64)[None], np.zeros((1, 9)), np.zeros((1, 6))))
                gid += 1
            elif len(p[2]):
                t = len(p[2])
                rows.append((False, p[1], np.zeros((t, 4)), np.asarray(p[2], np.float64).reshape(t, 9),
                             np.asarray(p[3], np.float64).reshape(t, 6)))
                meshes.append((gid, t))
                gid += t
        if not rows:
            return Geometry(np.zeros(0, bool), np.zeros(0, np.int64), np.zeros((0, 4)), np.zeros((0, 9)),
                            np.zeros((0, 6)), [])
        n = [len(r[2]) for r in rows]
        return Geometry(np.repeat([r[0] for r in rows], n), np.repeat([r[1] for r in rows], n).astype(np.int64),
                        np.concatenate([r[2] for r in rows]), np.concatenate([r[3] for r in rows]),
                        np.concatenate([r[4] for r in rows]), meshes)


def geometry(source):
    """Geometry of a structured Object array or of an abi.SceneHolder (its SceneObject records read back)"""
    if not hasattr(source, "objects"):
        return _object_array(source)
    parts = []
    for i in range(source.n):
        so = source.objects[i]
        if so.type == 0:
            s = so.geometry.sphere.contents
            parts.append(("sphere", i, (s.center.x, s.center.y, s.center.z, s.radius)))
        else:
            m = so.geometry.mesh.contents
            t = int(m.num_triangles)
            addr = C.cast(m.vertices, C.c_void_p).value
            v = np.frombuffer((C.c_double * (15 * t)).from_address(addr), np.float64).reshape(t, 3, 5) if t else \
                np.zeros((0, 3, 5))
            parts.append(("mesh", i, v[:, :, :3].reshape(t, 9), v[:, :, 3:].reshape(t, 6)))
    return Geometry.concat(parts)


def _object_array(objs):
    n = len(objs)
    return Geometry(np.ones(n, bool), np.arange(n, dtype=np.int64),
                    np.concatenate([objs["center"], objs["radius"][:, None]], axis=1).astype(np.float64),
                    np.zeros((n, 9)), np.zeros((n, 6)), [])


def choose_big(geom, ratio=32.0):
    """gids of the oversized spheres, in index order: choose_big of rtb_scene.cu restated.  Sizes: |r| of every
    sphere, then per mesh every step-th triangle (step = max(1, T / 2048)) with half its largest axis extent, counted
    min(step, 64) times; the median is element (n - 1) / 2 of the sorted sizes (nth_element); candidates have
    |r| > ratio * median or a non-finite r; the 32 largest |r| win, ties to the lower index."""
    sph = np.flatnonzero(geom.is_sphere)
    r = geom.sph[sph, 3]
    sizes = [np.abs(r)]
    for first, t in geom.meshes:
        step = max(1, t // 2048)
        p = geom.tri[first + np.arange(0, t, step)].reshape(-1, 3, 3)
        ext = np.maximum((p.max(axis=1) - p.min(axis=1)).max(axis=1), 0.0)
        sizes.append(np.repeat(0.5 * ext, min(step, 64)))
    sizes = np.concatenate(sizes)
    if len(sizes) < 2:
        return np.zeros(0, np.int64)
    median = np.sort(sizes)[(len(sizes) - 1) // 2]
    cand = np.flatnonzero((np.abs(r) > ratio * median) | ~np.isfinite(r))
    pick = cand[np.lexsort((cand, -np.abs(r[cand])))][:32]
    return sph[np.sort(pick)]


# ---- float helpers ------------------------------------------------------------------------------------------------

def round_down(x):
    f = np.asarray(x, np.float64).astype(np.float32)
    return np.where(f.astype(np.float64) > x, np.nextafter(f, np.float32(-np.inf)), f)


def round_up(x):
    f = np.asarray(x, np.float64).astype(np.float32)
    return np.where(f.astype(np.float64) < x, np.nextafter(f, np.float32(np.inf)), f)


def f32(u32):
    return np.ascontiguousarray(u32, np.uint32).view(np.float32)


def leaf_decode(ref):
    v = ~np.asarray(ref, np.int64)
    return v >> 3, (v & 7) + 1


# ---- records ------------------------------------------------------------------------------------------------------

def _sphere_words(sph):
    return np.ascontiguousarray(sph, np.float64).view(np.uint32).reshape(-1, 8)


def check_records(tree, geom, ratio=32.0):
    info, prims = tree["info"], tree["prims"]
    N, P = info.n_prims, len(geom.is_sphere)
    big = choose_big(geom, ratio)
    want_n = P - len(big)
    if N != want_n:
        _fail(f"{N} primitives in the tree, want {want_n} ({P} minus {len(big)} oversized)")
    if N == 0:
        if len(prims):
            _fail("records dumped for an empty tree")
    else:
        if prims.shape != (N + 1, 12):
            _fail(f"prims has shape {prims.shape}, want {(N + 1, 12)}")
        if prims[N].any():
            _fail(f"record N = {N} (the empty slots' dummy) is not all zero: {prims[N]}")
        gid = prims[:N, 9].astype(np.int64)
        if ((gid < 0) | (gid >= P)).any():
            k = int(np.flatnonzero((gid < 0) | (gid >= P))[0])
            _fail(f"prims[{k}] has gid {gid[k]} outside [0, {P})")
        count = np.bincount(gid, minlength=P)
        want = np.ones(P, np.int64)
        want[big] = 0
        bad = np.flatnonzero(count != want)
        if len(bad):
            g = int(bad[0])
            _fail(f"gid {g} sits in {count[g]} records (positions {np.flatnonzero(gid == g)[:4]}), want {want[g]}"
                  f" ({len(bad)} gids wrong)")
        sph = geom.is_sphere[gid]
        flag = prims[:N, 10]
        want_flag = geom.obj[gid].astype(np.uint32) | np.where(sph, np.uint32(SPHERE_BIT), np.uint32(0))
        _first_diff(flag != want_flag, "object / sphere word", gid)
        _first_diff(prims[:N, 11] != 0, "word c.w", gid)
        s = np.flatnonzero(sph)
        _first_diff((prims[s, :8] != _sphere_words(geom.sph[gid[s]])).any(axis=1) | (prims[s, 8] != 0),
                    "sphere record", gid[s], s)
        t = np.flatnonzero(~sph)
        _first_diff((prims[t, :9] != geom.tri[gid[t]].astype(np.float32).view(np.uint32)).any(axis=1),
                    "triangle floats", gid[t], t)
        tri_exact = (geom.tri[gid[t]].astype(np.float32).astype(np.float64) == geom.tri[gid[t]]).all()
        uv_exact = (geom.uv[gid[t]].astype(np.float32).astype(np.float64) == geom.uv[gid[t]]).all()
        if bool(info.has_tri64) != (not tri_exact):
            _fail(f"has_tri64 = {info.has_tri64}, but the positions are {'' if tri_exact else 'not '}all floats")
        if bool(info.has_tex64) != (not uv_exact):
            _fail(f"has_tex64 = {info.has_tex64}, but the texture coordinates are {'' if uv_exact else 'not '}all floats")
        if bool(info.has_tex) != (len(t) > 0):
            _fail(f"has_tex = {info.has_tex} with {len(t)} triangles")
        if tree["tri64"] is not None:
            tri64 = tree["tri64"]
            if tri64[N].view(np.uint64).any():
                _fail("tri64 row N (the dummy) is not all zero")
            _first_diff((tri64[t].view(np.uint64) != geom.tri[gid[t]].view(np.uint64)).any(axis=1), "tri64 row",
                        gid[t], t)
        if tree["tex"] is not None:
            want_tex = np.where(sph[:, None], 0.0, geom.uv[gid]).astype(np.float32)
            _first_diff((tree["tex"].view(np.uint32) != want_tex.view(np.uint32)).any(axis=1), "tex row", gid)
        if tree["tex64"] is not None:
            want64 = np.where(sph[:, None], 0.0, geom.uv[gid])
            _first_diff((tree["tex64"].view(np.uint64) != want64.view(np.uint64)).any(axis=1), "tex64 row", gid)
    # the oversized list
    rec, cp = tree["big"], tree["big_fp32"]
    if info.n_big != len(big) or len(rec) != len(big):
        _fail(f"{info.n_big} oversized spheres, want {len(big)} (gids {big[:8]})")
    want_rec = np.zeros((len(big), 12), np.uint32)
    want_rec[:, :8] = _sphere_words(geom.sph[big])
    want_rec[:, 9] = big.astype(np.uint32)
    want_rec[:, 10] = geom.obj[big].astype(np.uint32) | np.uint32(SPHERE_BIT)
    bad = np.flatnonzero((rec != want_rec).any(axis=1))
    if len(bad):
        k = int(bad[0])
        _fail(f"oversized record {k} is gid {rec[k, 9]}, want gid {big[k]} (choose_big order: {big[:8]})")
    for k, g in enumerate(big):
        c = geom.sph[g]
        with np.errstate(over="ignore"):
            c32 = c.astype(np.float32)  # beyond FLT_MAX: +-inf
        if not (cp[k, :4] == c32).all():
            _fail(f"oversized FP32 copy {k} (gid {g}): {cp[k, :4]} is not {c32}")
        a = float(cp[k, 4])
        if a == np.inf:  # bounds everything, also an infinite centre or radius
            continue
        need = sum(abs(Fraction(float(v))) for v in c) if np.isfinite(c).all() else None
        if need is None or not np.isfinite(a) or Fraction(a) < need:
            _fail(f"oversized FP32 copy {k} (gid {g}): A_c = {a!r} < |cx|+|cy|+|cz|+|r| = "
                  f"{np.abs(c).sum()!r}")


def _first_diff(bad, what, gid, pos=None):
    idx = np.flatnonzero(bad)
    if len(idx):
        k = int(idx[0])
        p = k if pos is None else int(pos[k])
        _fail(f"{what} of prims[{p}] (gid {gid[k]}) differs from the caller's primitive ({len(idx)} records)")


def prim_bounds(tree, geom):
    """[N, 3] lo and hi of every BVH-ordered primitive, as the exact tests read it: c -+ |r| in double for a sphere;
    for a triangle the min / max of its tri64 doubles if the scene has them, else of its floats"""
    N, prims = tree["info"].n_prims, tree["prims"]
    sph = (prims[:N, 10] & SPHERE_BIT) != 0
    c = np.ascontiguousarray(prims[:N, :8]).view(np.float64)
    v = tree["tri64"][:N] if tree["tri64"] is not None else f32(prims[:N, :9]).astype(np.float64)
    v = np.where(sph[:, None], 0.0, v).reshape(N, 3, 3)  # sphere rows hold no triangle
    r = np.abs(c[:, 3:4])
    lo = np.where(sph[:, None], c[:, :3] - r, v.min(axis=1))
    hi = np.where(sph[:, None], c[:, :3] + r, v.max(axis=1))
    return lo, hi


def check_params(tree, geom, ratio=32.0):
    info = tree["info"]
    if info.n_prims == 0:
        return
    gid = tree["prims"][:info.n_prims, 9].astype(np.int64)
    sph = geom.is_sphere[gid]
    c, r = geom.sph[gid, :3], np.abs(geom.sph[gid, 3:4])
    p = geom.tri[gid].reshape(-1, 3, 3)
    lo = np.where(sph[:, None], round_down(c - r), round_down(p).min(axis=1))
    hi = np.where(sph[:, None], round_up(c + r), round_up(p).max(axis=1))
    lo, hi = lo.astype(np.float32).min(axis=0), hi.astype(np.float32).max(axis=0)
    got_lo, got_hi = np.array(info.scene_lo, np.float32), np.array(info.scene_hi, np.float32)
    if not (np.array_equal(got_lo.view(np.uint32), lo.view(np.uint32))
            and np.array_equal(got_hi.view(np.uint32), hi.view(np.uint32))):
        _fail(f"scene box {got_lo} {got_hi}, want {lo} {hi}")
    d = hi.astype(np.float64) - lo.astype(np.float64)
    diag = float(np.sqrt((d * d).sum()))
    if not diag > 0:
        diag = 1e-3
    g_lo, g_hi = (lo - diag).astype(np.float32), (hi + diag).astype(np.float32)
    max_abs = float(np.abs(np.concatenate([g_lo, g_hi]).astype(np.float64)).max())
    pad = (max_abs + 3.0 * diag * 1.7320508) * (1.0 / 1048576.0)
    for name, got, want, scale in (("guard_lo", info.guard_lo, g_lo, diag), ("guard_hi", info.guard_hi, g_hi, diag),
                                   ("pad", [info.pad], [pad], pad)):
        got, want = np.array(got, np.float64), np.array(want, np.float64)
        if (np.abs(got - want) > 1e-6 * (np.abs(want) + scale)).any():
            _fail(f"{name} = {got}, want {want} (k_build_params)")
    gd = 0.0
    for k in range(3):
        e = float(info.guard_hi[k]) - float(info.guard_lo[k])
        gd += e * e
    gd = float(np.sqrt(gd))
    far = 300.0 * gd
    if sph.any():
        r_min = float(r[sph].min())
        far = min(far, float(np.sqrt(2.0 * r_min * float(info.pad) * 9007199254740992.0 / 16.0)) - gd)
    if np.float32(info.far_t) != np.float32(max(far, 0.0)):
        _fail(f"far_t = {info.far_t!r}, want {np.float32(max(far, 0.0))!r} (build_scene)")


# ---- trees --------------------------------------------------------------------------------------------------------

def _slot_ranges(refs, N, node_first, node_end):
    """per slot [first, end) and used mask: leaves decoded, inner slots from their node's range"""
    first, count = leaf_decode(refs)
    inner = refs >= 0
    lo = np.where(inner, node_first[np.where(inner, refs, 0)], first)
    hi = np.where(inner, node_end[np.where(inner, refs, 0)], first + count)
    return lo, hi


def _walk(refs, N, leaf_max, used, what, root_ref):
    """common topology of a tree given per-node child refs [M, S] and used-slot mask: reachability, leaf partition,
    per-node contiguity.  Returns (levels: list of node index arrays in breadth-first slot order, node_first,
    node_end, leaf slots (node, slot) sorted by first)"""
    M = len(refs)
    if N == 0:
        if root_ref != REF_NONE:
            _fail(f"{what}: empty tree with root_ref {root_ref:#x}")
        return [], None, None, None
    if root_ref < 0:
        f, c = leaf_decode(root_ref)
        if (f, c) != (0, N) or N > leaf_max:
            _fail(f"{what}: root leaf ({f}, {c}) for N = {N}, leaf_max {leaf_max}")
        return [], None, None, None
    if root_ref != 0 or M == 0:
        _fail(f"{what}: root_ref {root_ref} with {M} nodes")
    inner = used & (refs >= 0)
    if (refs[inner] >= M).any():
        n, s = np.argwhere(inner & (refs >= M))[0]
        _fail(f"{what}: node {n} slot {s} refers to node {refs[n, s]} of {M}")
    seen = np.zeros(M, np.int64)
    levels, frontier = [], np.array([0])
    seen[0] = 1
    while len(frontier):
        levels.append(frontier)
        if len(levels) > STACK_SIZE + 2:
            _fail(f"{what}: more than {STACK_SIZE + 2} levels (a cycle?)")
        r = refs[frontier]
        nxt = r[inner[frontier]]
        np.add.at(seen, nxt, 1)
        twice = np.flatnonzero(seen > 1)
        if len(twice):
            _fail(f"{what}: node {twice[0]} is reached {seen[twice[0]]} times from the root")
        frontier = nxt
    if (seen == 0).any():
        _fail(f"{what}: node {np.flatnonzero(seen == 0)[0]} is not reached from the root "
              f"({int((seen == 0).sum())} of {M})")
    # leaves
    leaf = used & (refs < 0)
    ln, ls = np.nonzero(leaf)
    first, count = leaf_decode(refs[ln, ls])
    bad = np.flatnonzero((count < 1) | (count > leaf_max) | (first < 0) | (first + count > N))
    if len(bad):
        k = bad[0]
        _fail(f"{what}: node {ln[k]} slot {ls[k]}: leaf ({first[k]}, {count[k]}) outside [0, {N}) or count > {leaf_max}")
    order = np.lexsort((count, first))
    first, count, ln, ls = first[order], count[order], ln[order], ls[order]
    end = first + count
    if first[0] != 0:
        _fail(f"{what}: primitives [0, {first[0]}) are in no leaf")
    gap = np.flatnonzero(first[1:] != end[:-1])
    if len(gap):
        k = gap[0]
        kind = "overlap" if first[k + 1] < end[k] else "leave a gap"
        _fail(f"{what}: leaves node {ln[k]} slot {ls[k]} [{first[k]}, {end[k]}) and node {ln[k + 1]} slot {ls[k + 1]} "
              f"[{first[k + 1]}, {end[k + 1]}) {kind}")
    if end[-1] != N:
        _fail(f"{what}: primitives [{end[-1]}, {N}) are in no leaf")
    # per node: slot ranges disjoint, union contiguous (bottom-up)
    node_first, node_end = np.zeros(M, np.int64), np.zeros(M, np.int64)
    for lev in reversed(levels):
        lo, hi = _slot_ranges(refs[lev], N, node_first, node_end)
        u = used[lev]
        lo_s = np.where(u, lo, np.iinfo(np.int64).max)
        o = np.argsort(lo_s, axis=1, kind="stable")
        lo_o, hi_o, u_o = (np.take_along_axis(a, o, axis=1) for a in (lo, hi, u))
        chain = (lo_o[:, 1:] == hi_o[:, :-1]) | ~u_o[:, 1:]
        bad = np.flatnonzero(~chain.all(axis=1))
        if len(bad):
            n = lev[bad[0]]
            _fail(f"{what}: node {n}: slot ranges {list(zip(lo[bad[0]][u[bad[0]]], hi[bad[0]][u[bad[0]]]))} are not "
                  f"disjoint with a contiguous union")
        node_first[lev] = lo_o[:, 0]
        node_end[lev] = np.where(u, hi, -1).max(axis=1)
    return levels, node_first, node_end, (ln, ls)


def _slot_prim_bounds(levels, refs, used, N, leaves, plo, phi):
    """[M, S, 3] lo / hi of the primitives under every used slot (exact: min / max over the slot's range)"""
    M, S = refs.shape
    ln, ls = leaves
    first, _ = leaf_decode(refs[ln, ls])
    slo, shi = np.full((M, S, 3), np.inf), np.full((M, S, 3), -np.inf)
    slo[ln, ls] = np.minimum.reduceat(plo, first, axis=0)
    shi[ln, ls] = np.maximum.reduceat(phi, first, axis=0)
    nlo, nhi = np.full((M, 3), np.inf), np.full((M, 3), -np.inf)
    for lev in reversed(levels):
        r = refs[lev]
        inner = used[lev] & (r >= 0)
        a, b = np.nonzero(inner)
        slo[lev[a], b] = nlo[r[a, b]]
        shi[lev[a], b] = nhi[r[a, b]]
        nlo[lev] = np.where(used[lev][..., None], slo[lev], np.inf).min(axis=1)
        nhi[lev] = np.where(used[lev][..., None], shi[lev], -np.inf).max(axis=1)
    return slo, shi


def _contain(what, blo, bhi, slo, shi, used, margin):
    short = used[..., None] & ((blo > slo - margin) | (bhi < shi + margin))
    if short.any():
        n, s, a = np.argwhere(short)[0]
        _fail(f"{what}: node {n} slot {s} axis {'xyz'[a]}: box [{blo[n, s, a]!r}, {bhi[n, s, a]!r}] does not hold its "
              f"primitives [{slo[n, s, a]!r}, {shi[n, s, a]!r}] with pad/2 = {margin!r} to spare")


def decode4q(q):
    """compressed BVH4 words [M, 16] -> org [M, 3], cell [M, 3] (float32), refs [M, 4], qlo / qhi [M, 4 slots, 3]"""
    org = f32(q[:, 0:3])
    cell = f32(q[:, [3, 14, 15]])
    refs = q[:, 4:8].view(np.int32).astype(np.int64)
    k = np.arange(4) * 8
    qlo = ((q[:, 8:11, None] >> k) & 0xFF).transpose(0, 2, 1).astype(np.int64)
    qhi = ((q[:, 11:14, None] >> k) & 0xFF).transpose(0, 2, 1).astype(np.int64)
    return org, cell, refs, qlo, qhi


def check_bvh4(tree, scene_info, plo, phi):
    info = tree["info"]
    N, leaf_max, pad = info.n_prims, info.leaf_max, float(info.pad)
    q = tree["nodes4q"]
    M = len(q)
    if N <= leaf_max:
        if M:
            _fail(f"{M} BVH4 nodes for a tree of {N} <= leaf_max primitives")
        return _walk(np.zeros((0, 4), np.int64), N, leaf_max, np.zeros((0, 4), bool), "BVH4", info.root_ref)
    if not info.walks_bvh4:  # BVH2 fallback: the BVH4 stopped after (STACK_SIZE - 2) / 3 + 2 levels, unchecked
        if scene_info is not None and scene_info.bvh4_depth != 0:
            _fail(f"bvh4_depth = {scene_info.bvh4_depth} on a scene that walks the BVH2")
        if 3 * info.depth4 <= STACK_SIZE - 2:
            _fail(f"the BVH2 is walked although the BVH4's {info.depth4} levels fit the walk's stack")
        return None
    org, cell, refs, qlo, qhi = decode4q(q)
    dummy = ~((N << 3) | 0)
    used = refs != dummy
    empty = ~used
    inv = (qlo != 255) | (qhi != 0)
    bad = np.argwhere(empty & inv.any(axis=2))
    if len(bad):
        n, s = bad[0]
        _fail(f"BVH4 node {n} slot {s}: empty slot with qlo {qlo[n, s]} qhi {qhi[n, s]} (want 255 / 0)")
    few = np.flatnonzero((used.sum(axis=1) < 4) & (used & (refs >= 0)).any(axis=1))
    if len(few):
        _fail(f"BVH4 node {few[0]}: {used[few[0]].sum()} used slots, one of them inner (the collapse fills four first)")
    levels, nf, ne, leaves = _walk(refs, N, leaf_max, used, "BVH4", info.root_ref)
    # breadth-first: inner children consecutive, after the parent; levels are index blocks
    start = 0
    for d, lev in enumerate(levels):
        if not np.array_equal(np.sort(lev), np.arange(start, start + len(lev))):
            _fail(f"BVH4 level {d} is not the index block [{start}, {start + len(lev)})")
        start += len(lev)
    inner = used & (refs >= 0)
    rank = np.cumsum(inner, axis=1) - 1
    first_child = np.where(inner, refs, np.iinfo(np.int64).max).min(axis=1)
    bad = np.flatnonzero((inner & (refs != first_child[:, None] + rank)).any(axis=1)
                         | (inner.any(axis=1) & (first_child <= np.arange(M))))
    if len(bad):
        n = bad[0]
        _fail(f"BVH4 node {n}: inner children {refs[n][inner[n]]} are not consecutive indices after it")
    depth = len(levels)
    if scene_info is not None and (scene_info.bvh4_depth != depth or scene_info.n_bvh_nodes != M):
        _fail(f"BVH4 of {depth} levels, {M} nodes; scene info says {scene_info.bvh4_depth} levels, "
              f"{scene_info.n_bvh_nodes} nodes")
    if info.depth4 != depth or 3 * depth > STACK_SIZE - 2:
        _fail(f"BVH4 of {depth} levels: depth4 = {info.depth4}, walk stack needs 3 * {depth} <= {STACK_SIZE - 2}")
    # cells
    bits = cell.view(np.uint32)
    e = (bits >> 23) & 0xFF
    bad = np.argwhere(((bits & 0x807FFFFF) != 0) | (e < 1) | (e > 254))
    if len(bad):
        n, a = bad[0]
        _fail(f"BVH4 node {n} axis {'xyz'[a]}: cell {cell[n, a]!r} is not a normal power of two")
    slo, shi = _slot_prim_bounds(levels, refs, used, N, leaves, plo, phi)
    ext = np.where(used[..., None], shi, -np.inf).max(axis=1) - np.where(used[..., None], slo, np.inf).min(axis=1)
    bad = np.argwhere(255.0 * cell.astype(np.float64) < ext)
    if len(bad):
        n, a = bad[0]
        _fail(f"BVH4 node {n} axis {'xyz'[a]}: 255 cells of {cell[n, a]!r} do not span the primitives' {ext[n, a]!r}")
    o, c = org.astype(np.float64)[:, None, :], cell.astype(np.float64)[:, None, :]
    dlo, dhi = o + qlo * c, o + qhi * c
    _contain("compressed BVH4", dlo, dhi, slo, shi, used, pad / 2)
    if len(tree["nodes4"]):
        u = tree["nodes4"]
        if len(u) != M:
            _fail(f"{len(u)} uncompressed BVH4 nodes, {M} compressed")
        ulo = np.stack([f32(u[:, 0:4]), f32(u[:, 8:12]), f32(u[:, 16:20])], axis=2).astype(np.float64)
        uhi = np.stack([f32(u[:, 4:8]), f32(u[:, 12:16]), f32(u[:, 20:24])], axis=2).astype(np.float64)
        urefs = u[:, 24:28].view(np.int32).astype(np.int64)
        want = np.where(used, refs, REF_NONE)
        bad = np.argwhere(urefs != want)
        if len(bad):
            n, s = bad[0]
            _fail(f"BVH4 node {n} slot {s}: uncompressed ref {urefs[n, s]}, compressed {refs[n, s]}")
        short = used[..., None] & ((dlo > ulo) | (dhi < uhi))
        if short.any():
            n, s, a = np.argwhere(short)[0]
            _fail(f"BVH4 node {n} slot {s} axis {'xyz'[a]}: compressed [{dlo[n, s, a]!r}, {dhi[n, s, a]!r}] does "
                  f"not contain uncompressed [{ulo[n, s, a]!r}, {uhi[n, s, a]!r}]")
        _contain("uncompressed BVH4", ulo, uhi, slo, shi, used, pad / 2)
    return levels, nf, ne, leaves


def check_bvh2(tree, scene_info, plo, phi):
    info = tree["info"]
    N, leaf_max, pad = info.n_prims, info.leaf_max, float(info.pad)
    w = tree["nodes"]
    if len(w) == 0:
        if not info.walks_bvh4 and N > leaf_max:
            _fail("the BVH2 is walked but was not dumped")
        return
    if len(w) != N - 1:
        _fail(f"{len(w)} BVH2 slots for N = {N}")
    refs = w[:, 12:14].view(np.int32).astype(np.int64)
    used = np.ones_like(refs, bool)
    # only emitted slots are reachable: walk from node 0 over the refs of reached nodes
    reached = np.zeros(len(w), bool)
    frontier = np.array([0])
    while len(frontier):
        reached[frontier] = True
        r = refs[frontier]
        frontier = r[r >= 0]
        if (frontier >= len(w)).any():
            _fail(f"BVH2 ref {frontier.max()} outside the {len(w)} slots")
        if reached[frontier].any():
            _fail(f"BVH2 node {frontier[reached[frontier]][0]} is reached twice")
    idx = np.flatnonzero(reached)
    sub = np.full(len(w), -1, np.int64)
    sub[idx] = np.arange(len(idx))
    rr = np.where(refs[idx] >= 0, sub[np.maximum(refs[idx], 0)], refs[idx])
    levels, nf, ne, leaves = _walk(rr, N, leaf_max, used[idx], "BVH2", 0)
    if w[~reached].any():
        _fail(f"BVH2 slot {np.flatnonzero(~reached & w.any(axis=1))[0]} is written but not reached")
    depth = len(levels)
    if scene_info is not None:
        if not (scene_info.bvh_depth - (leaf_max - 1) <= depth <= scene_info.bvh_depth):
            _fail(f"BVH2 of {depth} levels; bvh_depth {scene_info.bvh_depth} with leaf_max {leaf_max}")
        if not info.walks_bvh4 and scene_info.n_bvh_nodes != len(idx):
            _fail(f"the walked BVH2 has {len(idx)} nodes, scene info says {scene_info.n_bvh_nodes}")
    f = f32(w[idx])
    blo = np.stack([np.stack([f[:, 0], f[:, 2], f[:, 8]], 1), np.stack([f[:, 4], f[:, 6], f[:, 10]], 1)], 1)
    bhi = np.stack([np.stack([f[:, 1], f[:, 3], f[:, 9]], 1), np.stack([f[:, 5], f[:, 7], f[:, 11]], 1)], 1)
    slo, shi = _slot_prim_bounds(levels, rr, used[idx], N, leaves, plo, phi)
    _contain("BVH2", blo.astype(np.float64), bhi.astype(np.float64), slo, shi, used[idx], pad / 2)


def check(tree, geom, scene_info=None, ratio=32.0):
    """every check of the module docstring; scene_info: the scene's abi.RtbSceneInfo (node count and depths)"""
    check_records(tree, geom, ratio)
    check_params(tree, geom, ratio)
    info = tree["info"]
    if scene_info is not None and (scene_info.n_bvh_prims != info.n_prims or scene_info.n_big_prims != info.n_big):
        _fail("scene info and tree disagree on the primitive counts")
    if info.n_prims:
        plo, phi = prim_bounds(tree, geom)
    else:
        plo = phi = np.zeros((0, 3))
    check_bvh4(tree, scene_info, plo, phi)
    check_bvh2(tree, scene_info, plo, phi)


def canonical(tree):
    """the dump with BVH4 node indices replaced by their position in a breadth-first walk from the root in slot order
    (k_emit4 takes indices from an atomicAdd; everything else of the build is deterministic)"""
    info = tree["info"]
    q = tree["nodes4q"]
    out = {k: (None if v is None else np.array(v)) for k, v in tree.items() if k != "info"}
    names = [f for f, _ in getattr(type(info), "_fields_", [])] or sorted(vars(info))
    out["info"] = repr([(f, np.asarray(getattr(info, f)).tolist()) for f in names])
    if len(q) and info.root_ref == 0:
        refs = q[:, 4:8].view(np.int32).astype(np.int64)
        order, frontier = [], np.array([0])
        while len(frontier):
            order.append(frontier)
            r = refs[frontier]
            frontier = r[r >= 0]
        perm = np.concatenate(order)
        pos = np.full(len(q), -1, np.int64)
        pos[perm] = np.arange(len(perm))
        cq = q[perm].copy()
        r = refs[perm]
        cq[:, 4:8] = np.where(r >= 0, pos[np.maximum(r, 0)], r).astype(np.int32).view(np.uint32)
        out["nodes4q"] = cq
        if len(tree["nodes4"]):
            cu = tree["nodes4"][perm].copy()
            u = cu[:, 24:28].view(np.int32).astype(np.int64)
            cu[:, 24:28] = np.where((u >= 0) & (u != REF_NONE), pos[np.clip(u, 0, len(q) - 1)], u).astype(np.int32).view(np.uint32)
            out["nodes4"] = cu
    return out


def same_canonical(a, b):
    """-> list of the keys where two canonical dumps differ"""
    diff = []
    for k in sorted(set(a) | set(b)):
        x, y = a.get(k), b.get(k)
        if isinstance(x, str) or isinstance(y, str):
            if x != y:
                diff.append(k)
        elif (x is None) != (y is None) or (x is not None and not np.array_equal(np.asarray(x), np.asarray(y))):
            diff.append(k)
    return diff
