"""First-hit feature buffers (rtb_render_aov: albedo, normal, depth, hit count, object id) against the oracle.

The expected sums are built from the oracle alone: for every pixel and sample the render's own camera ray (the
Philox jitter of oracle_keyed_jitter, then oracle_camera_ray), its brute-force nearest hit (oracle_intersect_rays),
the albedo from the scene's colours and the checker in numpy.  They are summed in the library's order: samples in
float64, sequentially, per plane, rounded to float32 once, then the planes in float32 in plane order.  So sums, hits
and object ids must be bit-identical (np.array_equal).  The one exception is the checker on spheres: the sphere's u
goes through atan2, whose libm and CUDA forms may differ in the last bit (DESIGN.md section 2), so pixels where a
checkered sphere's u * M or v * M lies within 1e-9 of a cell edge are left out of the albedo comparison.
"""
import os
import subprocess

import numpy as np
import pytest

from test_gpu_texture import checkered_field, checkered_room, near_cell_edge
from test_gpu_wavefront_hits import chain_objects

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W, H = 64, 36
N_SAMPLES = 10                     # oracle records are made for samples 0..9 of every pixel
M_OF = {0: 100000.0, 1: 10.0}      # checker M of trace_path (raytracer.c:508) and cast_ray (raytracer.c:584)
MEGAKERNEL_THREADS = 148 * 2048 * 2
# (sample_begin, sample_end, planes): one plane, an uneven split (7 over 3: 3 + 3 + 1), an offset start, auto planes
RANGES = [(0, 4, 1), (0, 7, 3), (3, 10, 3), (5, 8, 0)]
OUTS = ("albedo", "normal", "depth", "hits", "object")


def plane_split(n_px, planes, spp, want_threads=MEGAKERNEL_THREADS):
    """rtb_plane_split: -> (splits, chunk)"""
    splits = min(max(1, (want_threads + n_px - 1) // n_px), 64)
    if planes > 0:
        splits = min(planes, 1024)
    splits = max(1, min(splits, spp))
    chunk = (spp + splits - 1) // splits if spp > 0 else 0
    if chunk > 0:
        splits = (spp + chunk - 1) // chunk
    return splits, chunk


def materials(src):
    """(colors [n, 3] float64, flags [n] uint32) of an Object array or an abi.SceneHolder"""
    if isinstance(src, np.ndarray):
        return np.array(src["color"], np.float64), np.array(src["flags"], np.uint32)
    objs = [src.objects[k] for k in range(src.n)]
    return (np.array([[o.material.color.x, o.material.color.y, o.material.color.z] for o in objs]),
            np.array([o.material.flags for o in objs], np.uint32))


def camera_rays(ol, cam, seed, w, h, samples, pixels=None):
    """the render's camera rays: [len(samples), n_pixels, 6]"""
    pixels = np.arange(w * h) if pixels is None else pixels
    rays = np.zeros((len(samples), len(pixels), 6))
    for i, s in enumerate(samples):
        for k, pix in enumerate(pixels):
            j = ol.keyed_jitter(seed, int(pix), int(s))
            x, y = pix % w, pix // w
            rays[i, k] = ol.camera_ray(cam, (x + j[0]) / (w - 1.0), (y + j[1]) / (h - 1.0))
    return rays


class OracleHits:
    """oracle hit records of samples 0..n-1 of every pixel: ids, t, normals, uvs as [n, n_px, ...]"""

    def __init__(self, ol, src, cam, seed, w, h, n=N_SAMPLES, pixels=None):
        rays = camera_rays(ol, cam, seed, w, h, range(n), pixels)
        rec = ol.intersect_rays(src, rays.reshape(-1, 6))
        shape = rays.shape[:2]
        self.ids = rec["ids"].reshape(shape)
        self.t = rec["t"].reshape(shape)
        self.normals = rec["normals"].reshape(shape + (3,))
        self.uvs = rec["uvs"].reshape(shape + (2,))
        self.colors, self.flags = materials(src)
        self.is_sphere = self.sphere_mask(src)

    @staticmethod
    def sphere_mask(src):
        if isinstance(src, np.ndarray):
            return np.ones(len(src), bool)
        return np.array([src.objects[k].type == 0 for k in range(src.n)])

    def per_sample(self, M):
        """per-sample values (float64) and the checkered-sphere cell-edge mask"""
        hit = self.ids >= 0
        obj = np.where(hit, self.ids, 0)
        checkered = hit & ((self.flags[obj] & 16) != 0)
        on = (np.fmod(self.uvs[..., 0] * M, 1.0) > 0.5) ^ (np.fmod(self.uvs[..., 1] * M, 1.0) < 0.5)
        k = np.where(on, 0.7, 0.3)  # 0.3 * (1 - on) + 0.7 * on in double is exactly 0.3 or 0.7
        albedo = np.where(hit[..., None], self.colors[obj], 0.0)
        albedo = np.where(checkered[..., None], albedo * k[..., None], albedo)
        normal = np.where(hit[..., None], self.normals, 0.0)
        depth = np.where(hit, self.t, 0.0)
        edge = checkered & self.is_sphere[obj] & near_cell_edge(self.uvs.reshape(-1, 2), M).reshape(hit.shape)
        return dict(albedo=albedo, normal=normal, depth=depth), hit, edge

    def sums(self, begin, end, planes, M):
        """expected outputs of rtb_render_aov for [begin, end), in the library's summation order"""
        vals, hit, edge = self.per_sample(M)
        n_px = self.ids.shape[1]
        splits, chunk = plane_split(n_px, planes, end - begin)
        out = {}
        for name, v in vals.items():
            total = np.zeros(v.shape[1:], np.float32)
            for p in range(splits):
                acc = np.zeros(v.shape[1:], np.float64)
                for s in range(begin + p * chunk, min(end, begin + (p + 1) * chunk)):
                    acc = acc + v[s]  # sequential, as the kernel: np.sum would be pairwise
                total = total + acc.astype(np.float32)
            out[name] = total
        out["hits"] = hit[begin:end].sum(axis=0).astype(np.uint32)
        out["object"] = (self.ids[begin] if end > begin else np.full(n_px, -1)).astype(np.int32)
        return out, edge[begin:end].any(axis=0)


def flat(got):
    """render_aov's [H, W, ...] arrays as [n_px, ...]"""
    return {k: v.reshape(W * H, -1).squeeze(-1) if v.ndim == 2 else v.reshape(W * H, 3) for k, v in got.items()}


def assert_aov_equal(got, want, edge, what, allow_edges=False):
    got = flat(got)
    for k in OUTS:
        g, w = got[k], want[k]
        if k == "albedo" and allow_edges:
            g, w = g[~edge], w[~edge]
        bad = np.flatnonzero((g != w).reshape(len(g), -1).any(axis=1))
        assert len(bad) == 0, f"{what}: {k} differs on {len(bad)} pixels, e.g. {bad[:5]}: {g[bad[:3]]} vs {w[bad[:3]]}"


# ---- scenes ---------------------------------------------------------------------------------------------------

def _mesh_matrix(gpu_api, abi):
    """the mesh room with its mesh placed by apply_matrix (main.c:140-147): positions no longer float-representable"""
    verts = gpu_api.heightfield_mesh(24, 20 * W / H * 0.98)
    a = np.radians(7.0)
    m = np.array([[0.93 * np.cos(a), 0, np.sin(a), 0.3], [0, 1.1, 0, 0.7], [-np.sin(a), 0, np.cos(a), -1.3], [0, 0, 0, 1]])
    return gpu_api.mesh_room(gpu_api.apply_matrix(verts, m), W, H)


SCENES = {
    "c1": lambda api, abi: (api.scene_default(W, H), None),
    "sphere-field": lambda api, abi: (api.scene_sphere_field(300, W, H), None),
    "mesh-room": lambda api, abi: (api.mesh_room(api.heightfield_mesh(24, 20 * W / H * 0.98), W, H), None),
    "mesh-matrix": lambda api, abi: (_mesh_matrix(api, abi), None),
    "checker-spheres": lambda api, abi: (checkered_field(api, abi, W, H, count=300), None),
    "checker-mesh": lambda api, abi: (checkered_room(api, abi, 24, "double", W, H, seed=41)[0], None),
    "bvh2-fallback": lambda api, abi: (chain_objects(abi, 61), ((-6.0, -5.0, -4.0), (6.0, 6.5, 7.0))),
}


def _camera(api, view):
    return api.init_camera(W, H) if view is None else api.init_camera(W, H, pos=view[0], target=view[1])


# ---- 1. bit-identical sums, hits and ids against the oracle ----------------------------------------------------

@pytest.mark.parametrize("scene", list(SCENES))
def test_sums_hits_and_ids_bit_identical_to_the_oracle(gpu_api, ol, abi, scene):
    """both integrators (checker M = 100 000 and 10), one plane, an uneven split (7 samples over 3 planes), a sample
    range not starting at 0 and the automatic plane count"""
    src, view = SCENES[scene](gpu_api, abi)
    cam = _camera(gpu_api, view)
    seed = abi.SCENE_SEED
    want_hits = OracleHits(ol, src, cam, seed, W, H)
    assert (want_hits.ids >= 0).any() and (scene != "bvh2-fallback" or (want_hits.ids < 0).any())
    edges = 0
    with gpu_api.Scene(src) as sc:
        info = sc.info
        if scene == "mesh-matrix":
            assert info.double_triangles == 1
        if scene == "checker-mesh":
            assert info.double_texcoords == 1
        if scene == "bvh2-fallback":
            assert info.bvh4_depth == 0 and info.bvh_depth == 61
        for integrator in (0, 1):
            for begin, end, planes in RANGES:
                desc = gpu_api.make_desc(W, H, begin, end, planes=planes, integrator=integrator, seed=seed)
                got = sc.render_aov(cam, desc)
                want, edge = want_hits.sums(begin, end, planes, M_OF[integrator])
                what = f"{scene}, integrator {integrator}, samples [{begin}, {end}), planes {planes}"
                assert_aov_equal(got, want, edge, what, allow_edges=scene.startswith("checker"))
                edges += int(edge.sum())
    # sphere u differs from libm's only in the last bit: the excluded pixels are a small fraction
    assert edges <= 0.01 * W * H * len(RANGES) * 2, edges
    if scene.startswith("checker"):
        hit_obj = want_hits.ids[want_hits.ids >= 0]
        assert ((want_hits.flags[hit_obj] & abi.M_CHECKERED) != 0).mean() > 0.2, "the checker must be exercised"


# ---- 2. the same rays as the render ----------------------------------------------------------------------------

@pytest.mark.parametrize("scene", ["c1", "checker-mesh"])
def test_one_sample_equals_vertex_zero_of_the_path_records(gpu_api, abi, scene):
    """a 1-spp call at sample_begin = s hits what vertex 0 of rtb_path_records(sample = s) hits: same object, same
    normal (the render's primary ray, for every s)"""
    src, view = SCENES[scene](gpu_api, abi)
    cam = _camera(gpu_api, view)
    with gpu_api.Scene(src) as sc:
        for s in (0, 1, 5, 17):
            got = flat(sc.render_aov(cam, gpu_api.make_desc(W, H, s, s + 1)))
            rec = sc.path_records(cam, gpu_api.make_desc(W, H, 0, 1), s, n_vertices=1)
            assert np.array_equal(got["object"], rec["ids"][:, 0]), (scene, s)
            assert np.array_equal(got["normal"], rec["normals"][:, 0].astype(np.float32)), (scene, s)
            assert np.array_equal(got["hits"], (rec["ids"][:, 0] >= 0).astype(np.uint32)), (scene, s)


# ---- 3. the render is untouched --------------------------------------------------------------------------------

def test_render_sums_unchanged_by_aov_calls(gpu_api, abi):
    """rtb_render_accum on a scene gives the same bits before and after feature-buffer calls on that scene"""
    src, _ = SCENES["checker-mesh"](gpu_api, abi)
    cam = gpu_api.init_camera(W, H)
    descs = [gpu_api.make_desc(W, H, 0, 6), gpu_api.make_desc(W, H, 0, 6, planes=3, integrator=1),
             gpu_api.make_desc(W, H, 2, 9, planes=2)]
    with gpu_api.Scene(src) as sc:
        before = [sc.render(cam, d, want_accum=True)[1] for d in descs]
        for d in descs:
            sc.render_aov(cam, d)
            sc.render_aov(cam, gpu_api.make_desc(W, H, 0, 40, planes=40))
        after = [sc.render(cam, d, want_accum=True)[1] for d in descs]
    for k, (a, b) in enumerate(zip(before, after)):
        assert np.array_equal(a, b), k


def _render_scene(gpu_api, abi, holder, cam, spp, params):
    _, host = gpu_api.load()
    import ctypes as C
    fb = np.zeros((H, W, 3), np.uint8)
    opt = abi.Options()
    opt.width, opt.height, opt.samples = W, H, spp
    host.render_scene(fb.ctypes.data, C.addressof(holder.objects), holder.n, C.byref(cam), C.byref(opt), C.byref(params))
    return fb


@pytest.mark.parametrize("integrator", [0, 1])
def test_render_scene_aov_frame_and_means(gpu_api, abi, integrator):
    """render_scene_aov: the framebuffer and accum_out of render_scene with the same parameters, and the means of
    rtb_render_aov's sums in float (albedo, normal / spp; depth / hits, 0 where nothing was hit)"""
    import ctypes as C
    src, _ = SCENES["checker-mesh"](gpu_api, abi)
    cam = gpu_api.init_camera(W, H)
    spp, offset = 5, 3
    _, host = gpu_api.load()

    def params(acc):
        p = abi.RenderParams()
        host.render_params_default(C.byref(p))
        p.sample_offset, p.integrator, p.num_gpus = offset, integrator, 1
        p.accum_out = acc.ctypes.data_as(C.POINTER(C.c_float))
        return p

    acc0, acc1 = np.zeros((H, W, 3), np.float32), np.zeros((H, W, 3), np.float32)
    fb0 = _render_scene(gpu_api, abi, src, cam, spp, params(acc0))
    fb1, means = gpu_api.render_scene_aov(src, cam, W, H, spp, params(acc1))
    assert np.array_equal(fb0, fb1) and np.array_equal(acc0, acc1)
    with gpu_api.Scene(src) as sc:
        sums = sc.render_aov(cam, gpu_api.make_desc(W, H, offset, offset + spp, integrator=integrator))
    n = np.float32(spp)
    assert np.array_equal(means["albedo"], sums["albedo"] / n)
    assert np.array_equal(means["normal"], sums["normal"] / n)
    hits = sums["hits"]
    depth = np.where(hits > 0, sums["depth"] / np.maximum(hits, 1).astype(np.float32), np.float32(0))
    assert np.array_equal(means["depth"], depth)
    assert np.array_equal(means["object"], sums["object"])
    assert hits.max() == spp and (means["object"] >= 0).any()


# ---- 4. the device API -----------------------------------------------------------------------------------------

def test_device_api_streams_null_outputs_errors_and_additivity(gpu_api, abi):
    import torch
    src, _ = SCENES["c1"](gpu_api, abi)
    cam = gpu_api.init_camera(W, H)
    desc = gpu_api.make_desc(W, H, 0, 8, planes=3)
    dev = torch.device("cuda:0")
    shapes = dict(albedo=((H, W, 3), torch.float32), normal=((H, W, 3), torch.float32), depth=((H, W), torch.float32),
                  hits=((H, W), torch.int32), object=((H, W), torch.int32))
    with gpu_api.Scene(src) as sc:
        want = sc.render_aov(cam, desc)
        assert np.array_equal(sc.render_aov(cam, desc)["albedo"], want["albedo"]), "two calls differ"
        stream = torch.cuda.Stream(device=dev)
        for subset in (OUTS, ("albedo",), ("normal", "object"), ("depth", "hits"), ("hits",), ("object",)):
            bufs = {k: torch.full(shapes[k][0], 7, dtype=shapes[k][1], device=dev) for k in subset}
            torch.cuda.synchronize()
            ctr = sc.render_aov_accum(cam, desc, *(bufs[k].data_ptr() if k in bufs else 0 for k in OUTS),
                                      stream=stream.cuda_stream, want_counters=(subset == OUTS))
            stream.synchronize()
            for k, t in bufs.items():
                got = t.cpu().numpy()
                got = got.view(np.uint32) if k == "hits" else got
                assert np.array_equal(got, want[k]), (subset, k)
            if ctr is not None:
                assert ctr.rays == ctr.paths == W * H * 8 and ctr.prim_tests > 0 and ctr.launches == 4 and ctr.gpu_ms > 0
        with pytest.raises(gpu_api.RtbError, match=r"\(-1\)"):
            sc.render_aov_accum(cam, desc, 0, 0, 0, 0, 0)
        for bad in (gpu_api.make_desc(1, H, 0, 4), gpu_api.make_desc(W, H, 4, 2), gpu_api.make_desc(W, H, 0, 4, integrator=2)):
            with pytest.raises(gpu_api.RtbError, match=r"\(-1\)"):
                sc.render_aov(cam, bad)
        # sums over [0, 4) + [4, 8): hits exactly, the float sums to rounding
        a = sc.render_aov(cam, gpu_api.make_desc(W, H, 0, 4))
        b = sc.render_aov(cam, gpu_api.make_desc(W, H, 4, 8))
        whole = sc.render_aov(cam, gpu_api.make_desc(W, H, 0, 8))
        assert np.array_equal(a["hits"] + b["hits"], whole["hits"])
        for k in ("albedo", "normal", "depth"):
            np.testing.assert_allclose(a[k] + b[k], whole[k], rtol=1e-6, atol=1e-6, err_msg=k)
        # no samples: zeros and object -1
        empty = sc.render_aov(cam, gpu_api.make_desc(W, H, 3, 3))
        assert all((empty[k] == 0).all() for k in ("albedo", "normal", "depth", "hits")) and (empty["object"] == -1).all()


# ---- 5. full size ----------------------------------------------------------------------------------------------

def test_c3_full_size_against_brute_force(gpu_api, ol):
    """C3 (1 002 528 triangles) at 1920x1080, 1 spp: 64 seeded pixels against the oracle's brute force"""
    FW, FH = 1920, 1080
    verts = gpu_api.heightfield_mesh(708, 20 * FW / FH * 0.98)
    holder = gpu_api.mesh_room(verts, FW, FH)
    cam = gpu_api.init_camera(FW, FH)
    pixels = np.sort(np.random.default_rng(5).choice(FW * FH, 64, replace=False))
    rays = camera_rays(ol, cam, 1666943821, FW, FH, [0], pixels)[0]
    rec = ol.intersect_rays(holder, rays)
    colors, _ = materials(holder)
    with gpu_api.Scene(holder) as sc:
        got = sc.render_aov(cam, gpu_api.make_desc(FW, FH, 0, 1))
    g = {k: v.reshape(FW * FH, -1)[pixels] for k, v in got.items()}
    hit = rec["ids"] >= 0
    assert (rec["ids"] == 6).sum() >= 8, "the camera sees the mesh"
    assert np.array_equal(g["object"][:, 0], rec["ids"])
    assert np.array_equal(g["hits"][:, 0], hit.astype(np.uint32))
    albedo = np.where(hit[:, None], colors[np.maximum(rec["ids"], 0)], 0.0)  # no checkered object in C3
    assert np.array_equal(g["albedo"], albedo.astype(np.float32))
    assert np.array_equal(g["normal"], rec["normals"].astype(np.float32))
    assert np.array_equal(g["depth"][:, 0], rec["t"].astype(np.float32))


# ---- 6. CLI ----------------------------------------------------------------------------------------------------

def read_pfm(path):
    with open(path, "rb") as f:
        data = f.read()
    head, rest = data.split(b"\n", 1)
    size, rest = rest.split(b"\n", 1)
    scale, body = rest.split(b"\n", 1)
    w, h = map(int, size.split())
    comp = 3 if head == b"PF" else 1
    assert head in (b"PF", b"Pf") and float(scale) < 0
    img = np.frombuffer(body, "<f4").reshape(h, w, comp)[::-1]  # stored bottom row first
    return img if comp == 3 else img[..., 0]


def test_cli_writes_the_feature_buffers(gpu_api, tmp_path):
    """bin/raytracer -a <prefix>: three PFMs equal to the host API's means; the PNG is byte-identical to a run
    without -a"""
    exe = os.path.join(ROOT, "raytracer.c_b200", "bin", "raytracer")
    cw, ch, spp = 96, 54, 4
    base = [exe, "-w", str(cw), "-h", str(ch), "-s", str(spp)]
    r = subprocess.run(base + ["-o", str(tmp_path / "plain.png")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run(base + ["-o", str(tmp_path / "aov.png"), "-a", str(tmp_path / "x")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert (tmp_path / "plain.png").read_bytes() == (tmp_path / "aov.png").read_bytes()
    objs = gpu_api.scene_default(cw, ch)
    cam = gpu_api.init_camera(cw, ch)
    with gpu_api.Scene(objs) as sc:
        sums = sc.render_aov(cam, gpu_api.make_desc(cw, ch, 0, spp))
    n = np.float32(spp)
    assert np.array_equal(read_pfm(tmp_path / "x_albedo.pfm"), sums["albedo"] / n)
    assert np.array_equal(read_pfm(tmp_path / "x_normal.pfm"), sums["normal"] / n)
    hits = sums["hits"]
    depth = np.where(hits > 0, sums["depth"] / np.maximum(hits, 1).astype(np.float32), np.float32(0))
    assert np.array_equal(read_pfm(tmp_path / "x_depth.pfm"), depth)
