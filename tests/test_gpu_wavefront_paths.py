"""The wavefront renderer's generate and shade kernels (k_wf_generate, k_wf_shade) against the oracle, ray for ray,
at every bounce, in both dielectric estimators.

rtb_wf_generate runs one wave of the camera-ray kernel and rtb_wf_bounce one bounce -- queue fill, one launch of
the renderer's trace kernel, one launch of k_wf_shade -- with wf_render's own arguments, plane groups and grids.
Feeding each bounce's output queue back in walks every path (the whole tree for the split estimator) through the
product kernels, and every bounce is compared with the forward oracle (oracle_path_vertex, the same vertex as
trace(): tests/test_oracle_path_log.py pins the two together):

  exact    the keys (path slot, branch) and the origin and direction bits of every queued ray against the oracle's
           path log; hit ids, primitives and t; the ray-counter increments (which count the depth cuts)
  bounded  outgoing throughputs, computed by the oracle in double from the GPU's incoming float throughput, and the
           per-slot contributions of the bounce (planes zeroed before the launch) -- see `throughput_units` and
           `contribution_bound` for the float operations the bounds count

The closure tests carry the planes across bounces instead and must land on rtb_render_accum's sums: bit for bit
for the stochastic estimator, within the reassociation bound of the atomic adds for the split one.  That is what
shows the probes run the renderer's own launches.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

U = 2.0 ** -24             # unit roundoff of float
BG = 10.0 / 255.0          # BACKGROUND (raytracer.h), returned on a miss and on a depth cut
# double-precision slack on either side (the directions and t are bit-identical; fresnel's x*x*x against
# pow(x, 3) and the oracle's double products differ by a few units of 2^-53): far below one float rounding
SLACK = 2.0 ** -40


# ---- scenes ---------------------------------------------------------------------------------------------------

def _mesh(api, W, H, grid=24):
    return api.heightfield_mesh(grid, 20 * W / H * 0.98)


def _tri64(api, W, H):
    a = np.radians(7.0)
    m = np.array([[0.93 * np.cos(a), 0, np.sin(a), 0.3], [0, 1.1, 0, 0.7], [-np.sin(a), 0, np.cos(a), -1.3], [0, 0, 0, 1]])
    return api.mesh_room(api.apply_matrix(_mesh(api, W, H), m), W, H)


def _checkered_field(api, abi, W, H):
    objs = api.scene_sphere_field(300, W, H, mix=(0.3, 0.3, 0.3))
    objs["flags"][::2] |= abi.M_CHECKERED
    return objs


def _tex64_room(api, abi, W, H):
    verts = _mesh(api, W, H)
    verts["tex"] = np.random.default_rng(5).uniform(0.0, 1.0, (len(verts), 2))
    holder = api.mesh_room(verts, W, H)
    for k in (1, 2, 6, 11, 12):  # back and left walls, the mesh, the mirror ball, the glass ball
        holder.objects[k].material.flags |= abi.M_CHECKERED
    return holder


def _material_sweep(api, abi, W, H):
    """every material edge of path_shade on the spheres of a small field: colour 0 (never survives), max channel
    exactly 1 (always survives), a colour above 1 (prob > 1), prob exactly 0.5, one zero channel, reflection and
    refraction together (refraction wins), emission only"""
    objs = api.scene_sphere_field(90, W, H, mix=(0.4, 0.3, 0.3))
    sweep = [(abi.M_DEFAULT, (0.0, 0.0, 0.0), (0.0, 0.0, 0.0)),
             (abi.M_DEFAULT, (1.0, 0.5, 0.25), (0.0, 0.0, 0.0)),
             (abi.M_DEFAULT, (1.5, 0.7, 0.2), (0.0, 0.0, 0.0)),
             (abi.M_DEFAULT, (0.5, 0.25, 0.5), (0.0, 0.0, 0.0)),
             (abi.M_DEFAULT, (0.8, 0.0, 0.6), (0.0, 0.0, 0.0)),
             (abi.M_REFLECTION | abi.M_REFRACTION, (0.9, 0.8, 0.9), (0.0, 0.0, 0.0)),
             (abi.M_DEFAULT, (0.0, 0.0, 0.0), (4.0, 3.0, 2.0)),
             (abi.M_REFRACTION, (1.0, 1.0, 1.0), (0.0, 0.0, 0.0)),
             (abi.M_REFLECTION, (0.5, 0.5, 0.5), (0.0, 0.0, 0.0))]
    small = np.flatnonzero(objs["radius"] < 100.0)
    for j, k in enumerate(small):
        flags, color, emission = sweep[j % len(sweep)]
        objs["flags"][k], objs["color"][k], objs["emission"][k] = flags, color, emission
    return objs


SCENES = {
    "c1": lambda api, abi, W, H: api.scene_default(W, H),  # r = 10 000 walls: the oversized list (slot < 0)
    "field300": lambda api, abi, W, H: api.scene_sphere_field(300, W, H, mix=(0.4, 0.3, 0.3)),
    "c5": lambda api, abi, W, H: api.scene_sphere_field(2000, W, H, mix=(0.1, 0.9, 0.0)),
    "c4": lambda api, abi, W, H: api.scene_sphere_field(10000, W, H, mix=(0.2, 0.4, 0.4)),
    "mesh-float": lambda api, abi, W, H: api.mesh_room(_mesh(api, W, H), W, H),
    "mesh-tri64": lambda api, abi, W, H: _tri64(api, W, H),
    "checkered-field": _checkered_field,
    "checkered-tex64": _tex64_room,
    "materials": _material_sweep,
}


def materials(src):
    """(flags [n] u32, emission [n, 3] f64) per object of an Object array or an abi.SceneHolder"""
    if isinstance(src, np.ndarray):
        return np.array(src["flags"], np.uint32), np.array(src["emission"], np.float64)
    objs = [src.objects[k].material for k in range(src.n)]
    return (np.array([m.flags for m in objs], np.uint32),
            np.array([[m.emission.x, m.emission.y, m.emission.z] for m in objs], np.float64))


# ---- the bounds -----------------------------------------------------------------------------------------------

def throughput_units(abi, flags):
    """float roundings between a vertex's incoming float throughput and a child's (path_shade), per parent object:
      (float)(colour * (1 / prob))            1   (the scene's albedo / prob, rounded once at upload)
      tp *= albedo / prob                     1
      M_CHECKERED: (float)checker, tp *= c    2
      dielectric: (float)(kr / p), (float)(kr / (1 - p)) or the split's (float)kr / (float)kt, tp *= w   2
      diffuse: (float)cos, tp *= cos          2
      mirror: no weight                       0
    The double factors (directions, cos, kr, kt, p) are the oracle's up to a few units of 2^-53 (SLACK)."""
    flags = np.asarray(flags, np.uint32)
    mirror = ((flags & abi.M_REFLECTION) != 0) & ((flags & abi.M_REFRACTION) == 0)
    return 2 + 2 * ((flags & abi.M_CHECKERED) != 0) + 2 * ~mirror


def vertex_terms(abi, ref, flags, emission):
    """the float terms a vertex adds to its path slot -> (magnitude [n, 3] summed over the vertex's terms, magnitude
    weighted by each term's roundings [n, 3], number of terms [n]).  Each term is a float product of a throughput
    and a colour rounded to float (emission, or RT_BACKGROUND = 10.0f / 255.0f): 2 roundings, plus the child's
    throughput roundings for the background of a child cut at depth > max_depth."""
    hit = ref["id"] >= 0
    ids = np.where(hit, ref["id"], 0)
    colour = np.where(hit[:, None], emission[ids], BG)
    mag = np.abs(ref["tp"] * colour)
    weighted = 2 * mag
    count = np.ones(len(ref), np.int64)
    k_child = np.where(hit, throughput_units(abi, flags[ids]), 0)
    for k in range(2):
        cut = (ref["cut"][:, k] != 0)[:, None]
        m = np.where(cut, np.abs(ref["child_tp"][:, k]) * BG, 0.0)
        mag += m
        weighted += m * (k_child + 2)[:, None]
        count += cut[:, 0]
    return mag, weighted, count


def slot_sums(pid, n_slots, values):
    out = np.zeros((n_slots,) + values.shape[1:], values.dtype)
    np.add.at(out, pid, values)
    return out


def contribution_bound(pid, n_slots, mag, weighted, count):
    """|planes - sum of the oracle's terms| per slot after one bounce on zeroed planes: each term carries its own
    roundings (weighted), and adding n terms in any order (the split estimator's atomics) adds at most (n - 1)
    roundings of the sum of their magnitudes"""
    m, w = slot_sums(pid, n_slots, mag), slot_sums(pid, n_slots, weighted)
    n = slot_sums(pid, n_slots, count)
    return U * (w + np.maximum(n - 1, 0)[:, None] * m) * (1 + 1e-6) + SLACK * m


# ---- the walk -------------------------------------------------------------------------------------------------

def _bits(rays):
    return np.ascontiguousarray(rays, np.float64).view(np.uint64).reshape(-1, 6)


def _rows_differ(got, want):
    d = np.asarray(got != want)
    return np.flatnonzero(d.reshape(d.shape[0], int(np.prod(d.shape[1:]))).any(axis=1))


def _sorted(pixel, sample, branch, rays, *extra):
    """rows ordered by (pixel, sample, branch, ray bits)"""
    b = _bits(rays)
    order = np.lexsort([b[:, k] for k in range(5, -1, -1)] + [branch, sample, pixel])
    return [np.asarray(a)[order] for a in (pixel, sample, branch, b) + extra]


class Walk:
    def __init__(self, api, abi, ol, name, W, H, spp, s_begin, planes, max_depth, dielectric, tune=0):
        self.api, self.abi, self.ol = api, abi, ol
        self.src = SCENES[name](api, abi, W, H)
        self.W, self.H, self.max_depth, self.dielectric = W, H, max_depth, dielectric
        self.cam = api.init_camera(W, H)
        self.desc = api.make_desc(W, H, s_begin, s_begin + spp, max_depth=max_depth, planes=planes, tune=tune,
                                  dielectric=1 if dielectric == "split" else 0)
        self.splits, self.chunk = api.wf_planes(self.desc)
        self.n_px = W * H
        self.flags, self.emission = materials(self.src)
        self.stats = dict(vertices=0, tries3=0, flipped=0, rays=0, bounces=0, max_branch=0)

    def sample_of(self, pid, wave):
        return (self.desc.sample_begin + (pid // self.n_px) * self.chunk + wave).astype(np.uint32)

    def run(self, sc, carry=False, check=True):
        """every bounce of every wave; check: compare each with the oracle (planes zeroed per bounce); carry: keep
        the planes across bounces and waves, as the renderer does -> (planes, rays counted by the kernels)"""
        planes = np.zeros((self.splits, self.n_px, 4), np.float32)
        log = self.ol.path_log(self.src, self.cam, self.W, self.H, self.desc.sample_end - self.desc.sample_begin,
                               dielectric=self.dielectric, max_depth=self.max_depth,
                               sample_offset=self.desc.sample_begin) if check else None
        rays = 0
        for wave in range(self.chunk):
            q = sc.wf_generate(self.cam, self.desc, wave)
            if check:
                self.check_camera(q, wave)
            depth = 0
            while len(q["pid"]):
                assert depth <= self.max_depth, "a ray was queued beyond max_depth"
                if not carry:
                    planes[:] = 0
                out, hits, ctr = sc.wf_bounce(self.cam, self.desc, wave, depth, q, planes)
                rays += ctr.rays
                if check:
                    self.check_bounce(log, wave, depth, q, out, hits, ctr, planes)
                q = out
                depth += 1
        return planes, rays

    def check_camera(self, q, wave):
        """queue 0: one camera ray per valid (plane, pixel), throughput exactly 1, branch 1"""
        last_len = (self.desc.sample_end - self.desc.sample_begin) - (self.splits - 1) * self.chunk
        valid = self.splits - 1 if wave >= last_len else self.splits
        assert len(q["pid"]) == valid * self.n_px
        assert np.array_equal(np.sort(q["pid"]), np.arange(valid * self.n_px, dtype=np.uint32))
        assert np.all(q["throughput"] == 1.0) and np.all(q["branch"] == 1)

    def check_bounce(self, log, wave, depth, q, out, hits, ctr, planes):
        abi, n_px = self.abi, self.n_px
        pid = q["pid"].astype(np.int64)
        pixel, sample = (pid % n_px).astype(np.uint32), self.sample_of(pid, wave)
        what = f"wave {wave} bounce {depth}"
        # the queue is the oracle's: keys and ray bits of every vertex at this depth
        sel = (log["depth"] == depth) & np.isin(log["sample"], np.unique(self.sample_of(np.arange(self.splits * n_px), wave)))
        want = _sorted(log["pixel"][sel], log["sample"][sel], log["branch"][sel], log["ray"][sel])
        got = _sorted(pixel, sample, q["branch"], q["rays"])
        assert len(got[0]) == len(want[0]), f"{what}: {len(got[0])} queued rays, the oracle has {len(want[0])}"
        for g, w, name in zip(got, want, ("pixel", "sample", "branch", "ray bits")):
            bad = _rows_differ(g, w)
            assert len(bad) == 0, f"{what}: {name} differs on {len(bad)} rays, e.g. {g[bad[:3]]} vs {w[bad[:3]]}"
        # the oracle's vertex from the GPU's own incoming ray and float throughput
        ref = self.ol.path_vertex(self.src, q["rays"], depth, q["branch"], pixel, sample,
                                  q["throughput"].astype(np.float64), dielectric=self.dielectric,
                                  max_depth=self.max_depth, seed=self.desc.seed)
        bad = np.flatnonzero(hits["ids"] != ref["id"])
        assert len(bad) == 0, f"{what}: hit ids differ on {len(bad)} rays, e.g. {hits['ids'][bad[:5]]} vs {ref['id'][bad[:5]]}"
        hit = ref["id"] >= 0
        assert np.array_equal(hits["prims"][hit], ref["prim"][hit]), f"{what}: primitives differ"
        assert np.array_equal(hits["t"][hit].view(np.uint64), ref["t"][hit].view(np.uint64)), f"{what}: t differs"
        assert ctr.rays == int(ref["rays"].sum()), f"{what}: {ctr.rays} rays counted, the oracle {ref['rays'].sum()}"
        assert ctr.rays_intersected == len(pid)
        # children: the same set, bit for bit, with bounded throughputs
        k_par, k_child = np.nonzero((np.arange(2)[None, :] < ref["n_children"][:, None]) & (ref["cut"] == 0))
        w_pid = q["pid"][k_par].astype(np.int64)
        want = _sorted((w_pid % n_px).astype(np.uint32), self.sample_of(w_pid, wave), ref["child_branch"][k_par, k_child],
                       ref["child_ray"][k_par, k_child], ref["child_tp"][k_par, k_child],
                       throughput_units(abi, self.flags[ref["id"][k_par]]))
        o_pid = out["pid"].astype(np.int64)
        got = _sorted((o_pid % n_px).astype(np.uint32), self.sample_of(o_pid, wave), out["branch"], out["rays"],
                      out["throughput"].astype(np.float64))
        assert len(got[0]) == len(want[0]), f"{what}: {len(got[0])} children queued, the oracle has {len(want[0])}"
        for g, w, name in zip(got[:4], want[:4], ("pixel", "sample", "branch", "ray bits")):
            bad = _rows_differ(g, w)
            assert len(bad) == 0, f"{what}: child {name} differs on {len(bad)} rays, e.g. {g[bad[:3]]} vs {w[bad[:3]]}"
        tp_gpu, tp_ref, units = got[4], want[4], want[5]
        err = np.abs(tp_gpu - tp_ref)
        bound = (units[:, None] * U * (1 + 1e-6) + SLACK) * np.abs(tp_ref)
        bad = np.flatnonzero((err > bound).any(axis=1))
        assert len(bad) == 0, (f"{what}: child throughput beyond its bound on {len(bad)} rays, e.g. {tp_gpu[bad[:3]]} vs "
                               f"{tp_ref[bad[:3]]} ({units[bad[:3]]} units)")
        # contributions of the bounce, per path slot
        n_slots = self.splits * n_px
        mag, weighted, count = vertex_terms(abi, ref, self.flags, self.emission)
        want_c = slot_sums(pid, n_slots, ref["contrib"])
        bound = contribution_bound(pid, n_slots, mag, weighted, count)
        got_c = planes.reshape(n_slots, 4)[:, :3].astype(np.float64)
        err = np.abs(got_c - want_c)
        bad = np.flatnonzero((err > bound).any(axis=1))
        assert len(bad) == 0, (f"{what}: contribution beyond its bound in {len(bad)} slots, e.g. slot {bad[:3]}: "
                               f"{got_c[bad[:3]]} vs {want_c[bad[:3]]} (bound {bound[bad[:3]]})")
        assert np.all(planes.reshape(n_slots, 4)[:, 3] == 0.0)
        s = self.stats
        s["vertices"] += len(pid)
        s["tries3"] += int(np.count_nonzero(ref["tries"] >= 3))
        s["flipped"] += int(np.count_nonzero(ref["flipped"]))
        s["bounces"] += 1
        s["max_branch"] = max(s["max_branch"], int(q["branch"].max()) if len(q["branch"]) else 0)


# ---- 1. camera rays -------------------------------------------------------------------------------------------

@pytest.mark.parametrize("W,H", [(80, 46), (33, 17)])
@pytest.mark.parametrize("dielectric", ["stochastic", "split"])
def test_camera_rays(gpu_api, abi, ol, W, H, dielectric):
    """queue 0 of every wave: frames that are not a multiple of the 8x4 tile, sample_begin 3, 7 samples over 3
    planes (3 + 3 + 1: the last plane runs out after the first wave); the rays must be the oracle's camera rays with
    the keyed jitter, bit for bit"""
    wk = Walk(gpu_api, abi, ol, "c1", W, H, spp=7, s_begin=3, planes=3, max_depth=0, dielectric=dielectric)
    log = ol.path_log(wk.src, wk.cam, W, H, 7, dielectric=dielectric, max_depth=0, sample_offset=3)
    with gpu_api.Scene(wk.src) as sc:
        for wave in range(wk.chunk):
            q = sc.wf_generate(wk.cam, wk.desc, wave)
            wk.check_camera(q, wave)
            pid = q["pid"].astype(np.int64)
            sample = wk.sample_of(pid, wave)
            sel = np.isin(log["sample"], np.unique(sample))
            got = _sorted((pid % wk.n_px).astype(np.uint32), sample, q["branch"], q["rays"])
            want = _sorted(log["pixel"][sel], log["sample"][sel], log["branch"][sel], log["ray"][sel])
            for g, w in zip(got, want):
                assert np.array_equal(g, w), f"wave {wave}: queue 0 differs from the oracle's camera rays"


# ---- 2. every vertex of every path ----------------------------------------------------------------------------

PATH_CASES = [
    # scene, W, H, spp, s_begin, planes, max_depth, dielectric
    ("c1", 40, 23, 3, 1, 2, 5, "stochastic"),
    ("c1", 40, 23, 3, 1, 2, 5, "split"),
    ("field300", 48, 27, 3, 0, 2, 5, "stochastic"),
    ("field300", 48, 27, 3, 0, 2, 3, "split"),
    ("field300", 48, 27, 2, 0, 2, 5, "split"),
    ("c5", 32, 32, 2, 0, 1, 63, "stochastic"),
    ("c5", 32, 32, 2, 0, 1, 64, "stochastic"),
    ("c5", 32, 32, 2, 0, 1, 65, "stochastic"),
    ("c5", 24, 24, 1, 0, 1, 5, "split"),
    ("field300", 24, 14, 1, 0, 1, 16, "split"),  # split trees of 2^17 branch ids: bits above 2^24 of the bounce word
    ("mesh-float", 40, 23, 2, 2, 2, 5, "stochastic"),
    ("mesh-float", 40, 23, 2, 2, 2, 5, "split"),
    ("mesh-tri64", 40, 23, 2, 0, 2, 5, "stochastic"),
    ("checkered-field", 40, 23, 2, 0, 2, 5, "stochastic"),
    ("checkered-field", 40, 23, 2, 0, 2, 3, "split"),
    ("checkered-tex64", 40, 23, 2, 0, 2, 5, "stochastic"),
    ("materials", 48, 27, 3, 0, 3, 5, "stochastic"),
    ("materials", 48, 27, 2, 0, 2, 5, "split"),
]


@pytest.mark.parametrize("case", PATH_CASES, ids=["-".join(map(str, (c[0], c[7], f"d{c[6]}"))) + f"-{i}"
                                                   for i, c in enumerate(PATH_CASES)])
def test_every_vertex_of_every_path(gpu_api, abi, ol, case):
    name, W, H, spp, s_begin, planes, max_depth, dielectric = case
    wk = Walk(gpu_api, abi, ol, name, W, H, spp, s_begin, planes, max_depth, dielectric)
    with gpu_api.Scene(wk.src) as sc:
        if name == "mesh-tri64":
            assert sc.info.double_triangles == 1
        if name == "checkered-tex64":
            assert sc.info.double_texcoords == 1
        wk.run(sc)
    s = wk.stats
    print(f"{name} {dielectric} depth {max_depth}: {s['vertices']} vertices in {s['bounces']} bounces, "
          f"{s['tries3']} hemisphere samples of >= 3 Philox blocks, {s['flipped']} flipped, largest branch id {s['max_branch']}")
    assert s["vertices"] > 0
    if name not in ("c5",):  # C5 has no diffuse spheres, only its walls are
        assert s["tries3"] > 0 and s["flipped"] > 0
    if dielectric == "split" and max_depth == 16:
        assert s["max_branch"] >= 1 << 16, "no branch id above 2^16 reached the bounce word"


def test_coverage_over_all_paths_includes_deep_rejection_and_flips(gpu_api, abi, ol):
    """the hemisphere sampler's later Philox blocks and its flip branch, on the C1 walls"""
    wk = Walk(gpu_api, abi, ol, "c1", 64, 36, 2, 0, 1, 3, "stochastic")
    with gpu_api.Scene(wk.src) as sc:
        wk.run(sc)
    print(f"c1: {wk.stats}")
    assert wk.stats["tries3"] > 0 and wk.stats["flipped"] > 0


# ---- 3. closure with the renderer -----------------------------------------------------------------------------

CLOSURE_CASES = [("c1", "stochastic", 5), ("field300", "stochastic", 5), ("mesh-float", "stochastic", 5),
                 ("c5", "stochastic", 64), ("materials", "stochastic", 5), ("c1", "split", 5), ("field300", "split", 5),
                 ("checkered-tex64", "split", 3)]


def _plane_sum(planes):
    acc = np.zeros(planes.shape[1:2] + (3,), np.float32)
    for k in range(planes.shape[0]):
        acc = acc + planes[k, :, :3]  # float32 adds in plane order, as k_wf_sum_planes
    return acc


@pytest.mark.parametrize("name,dielectric,max_depth", CLOSURE_CASES)
def test_probe_walk_lands_on_the_render(gpu_api, abi, ol, name, dielectric, max_depth):
    """the planes carried across every bounce and wave, summed in plane order, against rtb_render's sums; the frame
    against oracle_tonemap of those sums"""
    W, H, spp, s_begin, planes = 37, 21, 7, 2, 3
    wk = Walk(gpu_api, abi, ol, name, W, H, spp, s_begin, planes, max_depth, dielectric)
    with gpu_api.Scene(wk.src) as sc:
        got_planes, rays = wk.run(sc, carry=True, check=False)
        fb, acc, ctr = sc.render(wk.cam, wk.desc, want_accum=True)
    got = _plane_sum(got_planes).reshape(H, W, 3)
    assert rays == ctr.rays
    assert np.array_equal(fb, ol.tonemap(acc.astype(np.float64), spp)), "frame != oracle_tonemap(the render's sums)"
    if dielectric == "stochastic":
        bad = np.argwhere(got.view(np.uint32) != acc.view(np.uint32))
        assert len(bad) == 0, f"{len(bad)} sums differ from the render, e.g. {bad[:3]}: {got[tuple(bad[0])]} vs {acc[tuple(bad[0])]}"
    else:
        # the atomics of a slot may add in another order: per pixel, within (n - 1) roundings of the magnitude of its
        # float terms (taken from the oracle's log, 1 % margin for the GPU's own rounding of them), twice (both sides)
        log = ol.path_log(wk.src, wk.cam, W, H, spp, dielectric=dielectric, max_depth=max_depth, sample_offset=s_begin)
        mag, _, count = vertex_terms(abi, log, wk.flags, wk.emission)
        m = slot_sums(log["pixel"].astype(np.int64), W * H, mag).reshape(H, W, 3)
        n = slot_sums(log["pixel"].astype(np.int64), W * H, count).reshape(H, W, 1)
        bound = 2 * U * (n + planes) * m * 1.01
        err = np.abs(got.astype(np.float64) - acc)
        bad = np.argwhere(err > bound)
        assert len(bad) == 0, f"{len(bad)} sums beyond the reassociation bound, e.g. {bad[:3]}"


# ---- 4. per-pixel bound on whole renders ----------------------------------------------------------------------

@pytest.mark.parametrize("name,max_depth", [("c1", 5), ("c4", 8), ("c5", 64)])
@pytest.mark.parametrize("dielectric", ["stochastic", "split"])
def test_render_within_the_float_bound_of_the_oracle(gpu_api, abi, ol, name, max_depth, dielectric):
    """|gpu - oracle| <= K_pixel 2^-24 per pixel and channel, K_pixel from the pixel's vertices in the oracle log:
    a term of a vertex at depth d is a float product of a throughput that went through d + 1 vertices of at most 6
    roundings each (throughput_units) and a colour (2 roundings); the pixel's n terms are added in float, first per
    plane, then the planes in order (n + planes roundings of the magnitude)"""
    if dielectric == "split":
        max_depth = min(max_depth, 5)
    W, H, spp, planes = 32, 18, 4, 2
    wk = Walk(gpu_api, abi, ol, name, W, H, spp, 0, planes, max_depth, dielectric)
    with gpu_api.Scene(wk.src) as sc:
        _, acc, _ = sc.render(wk.cam, wk.desc, want_accum=True)
    log = ol.path_log(wk.src, wk.cam, W, H, spp, dielectric=dielectric, max_depth=max_depth)
    want, _ = ol.render_sum(wk.src, wk.cam, W, H, spp, dielectric=dielectric, max_depth=max_depth)
    mag, _, count = vertex_terms(abi, log, wk.flags, wk.emission)
    pix = log["pixel"].astype(np.int64)
    k_term = 6 * (log["depth"] + 1) + 2
    weighted = slot_sums(pix, W * H, mag * k_term[:, None]).reshape(H, W, 3)
    m = slot_sums(pix, W * H, mag).reshape(H, W, 3)
    n = slot_sums(pix, W * H, count).reshape(H, W, 1)
    bound = U * (weighted + (n + planes) * m) * (1 + 1e-6) + SLACK * m
    err = np.abs(acc.astype(np.float64) - want)
    print(f"{name} {dielectric}: largest error / bound = {np.max(err / np.maximum(bound, 1e-300)):.3f}")
    bad = np.argwhere(err > bound)
    assert len(bad) == 0, f"{len(bad)} values beyond the bound, e.g. {bad[:3]}: {acc[tuple(bad[0])]} vs {want[tuple(bad[0])]}"


# ---- 5. tonemap byte for byte ---------------------------------------------------------------------------------

def _crafted_sums(spp):
    k = np.arange(1, 256, dtype=np.float64)
    centre = ((k / 255.0) ** 5 * spp).astype(np.float32)
    near = [centre]
    for step in range(1, 5):
        up, down = centre.copy(), centre.copy()
        for _ in range(step):
            up = np.nextafter(up, np.float32(np.inf))
            down = np.nextafter(down, np.float32(0))
        near += [up, down]
    tiny = np.float32(np.finfo(np.float32).smallest_subnormal)
    special = np.array([0.0, -0.0, tiny, tiny * 7, np.finfo(np.float32).tiny * np.float32(0.5), spp, spp * 1.5, spp * 1e6,
                        np.inf, -np.inf, np.nan, -1.0, -tiny, np.float32(spp) * np.float32(1 - 2 ** -24),
                        np.nextafter(np.float32(spp), np.float32(np.inf))], np.float32)
    v = np.concatenate(near + [special])
    return np.concatenate([v, np.zeros((-len(v)) % 3, np.float32)])


@pytest.mark.parametrize("spp", [1, 49, 98, 103, 107])
def test_tonemap_byte_for_byte(gpu_api, ol, spp):
    """rtb_tonemap against oracle_tonemap on sums around every (k/255)^5 threshold (+-4 ulps), at sum = spp (for 49,
    98, 103 and 107, x * (1/x) rounds to 1 - 2^-53), 0, -0, subnormals, values above 1, inf, NaN and negatives"""
    import torch
    v = _crafted_sums(spp)
    w = len(v) // 3
    d_acc = torch.from_numpy(v).to("cuda:0")
    d_fb = torch.empty(len(v), dtype=torch.uint8, device="cuda:0")
    gpu_api.tonemap(d_acc.data_ptr(), w, 1, spp, d_fb.data_ptr())
    torch.cuda.synchronize()
    got = d_fb.cpu().numpy()
    want = ol.tonemap(v.astype(np.float64).reshape(1, w, 3), spp).reshape(-1)
    bad = np.flatnonzero(got != want)
    assert len(bad) == 0, f"{len(bad)} bytes differ, e.g. sums {v[bad[:5]]}: {got[bad[:5]]} vs {want[bad[:5]]}"
