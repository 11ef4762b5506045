"""Python bindings of the product libraries (ctypes; no compute happens in Python).

  librtb200.so          the CUDA kernels behind the C ABI of include/rtb200.h
  libraytracer_b200.so  the C99 host side with the reference's raytracer.h entry points

Loading fails loudly if either library is missing -- there is no CPU fallback.  The
oracle under oracle/ is never imported from here.
"""
import ctypes as C
import os

import numpy as np

from . import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_CUDA = os.environ.get("RTB200_LIB_OVERRIDE") or os.path.join(_HERE, "librtb200.so")  # override: dev A/B builds only
LIB_HOST = os.path.join(_HERE, "libraytracer_b200.so")

# every symbol include/rtb200.h declares
RTB_SYMBOLS = [
    "rtb_last_error", "rtb_version", "rtb_device_count", "rtb_scene_create_objects", "rtb_scene_create",
    "rtb_scene_create_objects_flags", "rtb_scene_create_flags",
    "rtb_scene_info_get", "rtb_scene_destroy", "rtb_release_workspace", "rtb_render_accum", "rtb_tonemap", "rtb_render",
    "rtb_trace_rays", "rtb_trace_rays_wf", "rtb_path_records", "rtb_philox4x32_10", "rtb_probe_l2_bandwidth", "rtb_cast_rays",
    "rtb_probe_fp32_tflops", "rtb_render_mean", "rtb_comm_unique_id", "rtb_comm_create_rank", "rtb_comm_create_local", "rtb_comm_size",
    "rtb_warm_up", "rtb_comm_local_ranks", "rtb_comm_destroy", "rtb_comm_shard_samples", "rtb_comm_scene_create", "rtb_comm_render", "rtb_render_multi",
]
# the reference's exported surface (raytracer.h:135-164) plus the documented extensions
HOST_SYMBOLS = [
    "random_double", "random_range", "point_at", "calculate_surface_normal", "intersect_sphere",
    "intersect_triangle", "print_v", "print_m", "clamp", "init_camera", "render", "load_obj",
    "ray_count", "intersection_test_count",
    "render_params_default", "render_scene", "render_ex", "free_mesh", "apply_matrix", "load_obj_ex", "render_warm_up",
    "scene_default", "scene_room_walls", "scene_random_spheres", "scene_sphere_field",
    "scene_heightfield_mesh", "scene_write_obj", "scene_mesh_room", "scene_from_objects", "rt_write_png",
]


class RtbError(RuntimeError):
    pass


_libs = None


def load():
    """dlopen both libraries (RTLD_GLOBAL so the host lib resolves rtb_* symbols)"""
    global _libs
    if _libs is not None:
        return _libs
    for p in (LIB_CUDA, LIB_HOST):
        if not os.path.exists(p):
            raise RtbError(f"{p} is missing: build it with `make -C {_HERE}` "
                           "(python -c 'import __graft_entry__ as g; g.build()'). There is no CPU fallback.")
    cu = C.CDLL(LIB_CUDA, mode=C.RTLD_GLOBAL)
    host = C.CDLL(LIB_HOST, mode=C.RTLD_GLOBAL)
    _bind(cu, host)
    _libs = (cu, host)
    return _libs


def _bind(cu, host):
    dp = C.POINTER(C.c_double)
    cu.rtb_last_error.restype = C.c_char_p
    cu.rtb_version.restype = C.c_char_p
    cu.rtb_device_count.restype = C.c_int
    cu.rtb_scene_create_objects.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.POINTER(C.c_void_p)]
    cu.rtb_scene_create.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.POINTER(C.c_void_p)]
    cu.rtb_scene_create_objects_flags.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_uint, C.POINTER(C.c_void_p)]
    cu.rtb_scene_create_flags.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_uint, C.POINTER(C.c_void_p)]
    cu.rtb_scene_info_get.argtypes = [C.c_void_p, C.POINTER(abi.RtbSceneInfo)]
    cu.rtb_scene_destroy.argtypes = [C.c_void_p]
    cu.rtb_scene_destroy.restype = None
    cu.rtb_render_accum.argtypes = [C.c_void_p, dp, C.POINTER(abi.RtbRenderDesc), C.c_void_p, C.c_void_p,
                                    C.POINTER(abi.RtbCounters)]
    cu.rtb_tonemap.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    cu.rtb_render.argtypes = [C.c_void_p, dp, C.POINTER(abi.RtbRenderDesc), C.c_void_p, C.c_void_p,
                              C.POINTER(abi.RtbCounters)]
    cu.rtb_trace_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int] + [C.c_void_p] * 6
    cu.rtb_trace_rays_wf.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int] + [C.c_void_p] * 7 + [
        C.POINTER(abi.RtbCounters)]
    cu.rtb_path_records.argtypes = [C.c_void_p, dp, C.POINTER(abi.RtbRenderDesc), C.c_int, C.c_int] + [C.c_void_p] * 5
    cu.rtb_philox4x32_10.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int]
    cu.rtb_cast_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_void_p]
    cu.rtb_probe_l2_bandwidth.argtypes = [C.c_size_t, C.c_int, C.c_int, C.POINTER(C.c_float)]
    cu.rtb_render_mean.argtypes = [C.c_void_p, dp, C.POINTER(abi.RtbRenderDesc), C.c_int, C.c_void_p, C.c_void_p,
                                   C.POINTER(abi.RtbCounters)]
    cu.rtb_comm_unique_id.argtypes = [C.c_void_p]
    cu.rtb_comm_create_rank.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
    cu.rtb_comm_create_local.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]
    cu.rtb_comm_size.argtypes = [C.c_void_p]
    cu.rtb_comm_local_ranks.argtypes = [C.c_void_p]
    cu.rtb_comm_destroy.argtypes = [C.c_void_p]
    cu.rtb_comm_destroy.restype = None
    cu.rtb_comm_scene_create.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_uint, C.POINTER(C.c_void_p)]
    cu.rtb_comm_render.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), dp, C.POINTER(abi.RtbRenderDesc), C.c_void_p,
                                   C.POINTER(abi.RtbCounters)]
    cu.rtb_render_multi.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, dp, C.POINTER(abi.RtbRenderDesc),
                                    C.c_void_p, C.c_void_p, C.POINTER(abi.RtbCounters)]

    host.init_camera.argtypes = [C.POINTER(abi.Camera), abi.Vec3, abi.Vec3, C.POINTER(abi.Options)]
    host.init_camera.restype = None
    host.render.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(abi.Camera), C.POINTER(abi.Options)]
    host.render.restype = None
    host.render_ex.argtypes = host.render.argtypes + [C.POINTER(abi.RenderParams)]
    host.render_ex.restype = None
    host.render_scene.argtypes = host.render_ex.argtypes
    host.render_scene.restype = None
    host.render_params_default.argtypes = [C.POINTER(abi.RenderParams)]
    host.render_params_default.restype = None
    host.load_obj.argtypes = [C.c_char_p, C.POINTER(abi.TriangleMesh)]
    host.load_obj.restype = C.c_bool
    host.load_obj_ex.argtypes = [C.c_char_p, C.POINTER(abi.TriangleMesh), C.c_int, C.c_size_t]
    host.load_obj_ex.restype = C.c_bool
    host.free_mesh.argtypes = [C.POINTER(abi.TriangleMesh)]
    host.free_mesh.restype = None
    host.apply_matrix.argtypes = [C.POINTER(abi.TriangleMesh), C.POINTER(C.c_double)]
    host.apply_matrix.restype = None
    host.calculate_surface_normal.argtypes = [abi.Vec3, abi.Vec3, abi.Vec3]
    host.calculate_surface_normal.restype = abi.Vec3
    host.scene_default.argtypes = [C.c_void_p, C.c_int, C.c_int]
    host.scene_default.restype = C.c_size_t
    host.scene_sphere_field.argtypes = [C.POINTER(C.c_void_p), C.c_size_t, C.c_int, C.c_int, abi.SceneMix, C.c_uint64]
    host.scene_sphere_field.restype = C.c_size_t
    host.scene_heightfield_mesh.argtypes = [C.POINTER(abi.TriangleMesh), C.c_int, C.c_double, C.c_double,
                                            C.c_double, C.c_double]
    host.scene_heightfield_mesh.restype = None
    host.scene_mesh_room.argtypes = [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(abi.TriangleMesh),
                                     C.c_int, C.c_int]
    host.scene_mesh_room.restype = C.c_size_t
    host.scene_write_obj.argtypes = [C.c_char_p, C.POINTER(abi.TriangleMesh)]
    host.scene_write_obj.restype = C.c_bool
    host.rt_write_png.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]
    host.rt_write_png.restype = C.c_int


def _check(rc, what):
    if rc != 0:
        cu, _ = load()
        raise RtbError(f"{what} failed ({rc}): {cu.rtb_last_error().decode()}")


def device_count():
    cu, _ = load()
    return cu.rtb_device_count()


# ---- host-side helpers (C99 code in libraytracer_b200.so) ---------------------------------

def init_camera(width, height, pos=(0.0, 0.0, 50.0), target=(0.0, 0.0, 0.0)):
    """raytracer.c:47-75; the defaults are main.c:424-425"""
    _, host = load()
    cam = abi.Camera()
    opt = abi.Options()
    opt.width, opt.height = width, height
    host.init_camera(C.byref(cam), abi.Vec3(*pos), abi.Vec3(*target), C.byref(opt))
    return cam


def scene_default(width=320, height=180):
    """C1: the reference default scene (main.c:244-397) as a structured Object array"""
    _, host = load()
    objs = (abi.Object * 38)()
    n = host.scene_default(objs, width, height)
    return abi.objects_to_numpy(objs, n)


def scene_sphere_field(count, width, height, mix=(0.5, 0.2, 0.2), seed=abi.SCENE_SEED):
    """C2/C4/C5: walls + `count` packed spheres + lights (generate_random_spheres semantics)"""
    _, host = load()
    libc = C.CDLL(None)
    libc.free.argtypes = [C.c_void_p]
    p = C.c_void_p()
    n = host.scene_sphere_field(C.byref(p), count, width, height, abi.SceneMix(*mix), seed)
    arr = np.frombuffer(C.string_at(p.value, 88 * n), dtype=abi.OBJECT_DTYPE).copy()
    libc.free(p)
    return arr


def heightfield_mesh(grid, half_w, half_d=29.0, y0=-12.0, amplitude=5.0):
    """C3 geometry: 2*grid*grid triangles as a VERTEX_DTYPE array"""
    _, host = load()
    libc = C.CDLL(None)
    libc.free.argtypes = [C.c_void_p]
    mesh = abi.TriangleMesh()
    host.scene_heightfield_mesh(C.byref(mesh), grid, half_w, half_d, y0, amplitude)
    n = mesh.num_triangles * 3
    arr = np.frombuffer(C.string_at(C.cast(mesh.vertices, C.c_void_p).value, 40 * n), dtype=abi.VERTEX_DTYPE).copy()
    libc.free(C.cast(mesh.vertices, C.c_void_p))
    return arr


def mesh_room(verts, width, height):
    """C3 scene from scene_mesh_room (host/scenes.c): 6 walls, the mesh, then lights, a
    mirror and a dielectric ball.  Returns an abi.SceneHolder that owns everything."""
    _, host = load()
    libc = C.CDLL(None)
    libc.free.argtypes = [C.c_void_p]
    verts = np.ascontiguousarray(verts, dtype=abi.VERTEX_DTYPE)
    mesh = abi.TriangleMesh()
    mesh.num_triangles = len(verts) // 3
    mesh.vertices = C.cast(verts.ctypes.data, C.POINTER(abi.Vertex))
    p_obj, p_sph = C.c_void_p(), C.c_void_p()
    n = host.scene_mesh_room(C.byref(p_obj), C.byref(p_sph), C.byref(mesh), width, height)
    h = abi.SceneHolder()
    h.n = n
    h.objects = (abi.SceneObject * n).from_address(p_obj.value)
    h._keep += [verts, mesh]
    h._free = [(libc, p_obj), (libc, p_sph)]
    return h


def apply_matrix(verts, matrix):
    """apply_matrix (main.c:140-147): every position through mat4_vector_mult, in double, in place"""
    _, host = load()
    assert verts.dtype == abi.VERTEX_DTYPE and verts.flags["C_CONTIGUOUS"]
    m = np.ascontiguousarray(matrix, dtype=np.float64).reshape(16)
    mesh = abi.TriangleMesh()
    mesh.num_triangles = len(verts) // 3
    mesh.vertices = C.cast(verts.ctypes.data, C.POINTER(abi.Vertex))
    host.apply_matrix(C.byref(mesh), m.ctypes.data_as(C.POINTER(C.c_double)))
    return verts


def load_obj(path, threads=None, min_chunk_bytes=0):
    """load_obj (raytracer.h:158); with `threads` given, load_obj_ex (same result for any chunking)"""
    _, host = load()
    mesh = abi.TriangleMesh()
    if threads is None:
        ok = host.load_obj(os.fsencode(path), C.byref(mesh))
    else:
        ok = host.load_obj_ex(os.fsencode(path), C.byref(mesh), int(threads), C.c_size_t(min_chunk_bytes))
    if not ok:
        raise RtbError(f"load_obj({path!r}) failed")
    n = mesh.num_triangles * 3
    arr = np.frombuffer(C.string_at(C.cast(mesh.vertices, C.c_void_p).value, 40 * n), dtype=abi.VERTEX_DTYPE).copy()
    host.free_mesh(C.byref(mesh))
    return arr


def write_obj(path, verts):
    _, host = load()
    verts = np.ascontiguousarray(verts, dtype=abi.VERTEX_DTYPE)
    mesh = abi.TriangleMesh()
    mesh.num_triangles = len(verts) // 3
    mesh.vertices = C.cast(verts.ctypes.data, C.POINTER(abi.Vertex))
    if not host.scene_write_obj(os.fsencode(path), C.byref(mesh)):
        raise RtbError(f"scene_write_obj({path!r}) failed")


def render(objects, camera, width, height, samples):
    """The drop-in call: the reference's render() signature (raytracer.h:156)."""
    _, host = load()
    arr = np.ascontiguousarray(objects, dtype=abi.OBJECT_DTYPE)
    fb = np.zeros((height, width, 3), dtype=np.uint8)
    opt = abi.Options()
    opt.width, opt.height, opt.samples = width, height, samples
    host.render(fb.ctypes.data, arr.ctypes.data, len(arr), C.byref(camera), C.byref(opt))
    return fb


# ---- the C ABI ----------------------------------------------------------------------------

def make_desc(width, height, sample_begin, sample_end, max_depth=5, seed=abi.SCENE_SEED, kernel=0, tune=0, planes=0, tune2=0, integrator=0, profile=1,
              dielectric=0):
    d = abi.RtbRenderDesc()
    d.width, d.height = width, height
    d.sample_begin, d.sample_end = sample_begin, sample_end
    d.max_depth = max_depth
    d.dielectric_mode = dielectric  # 0 stochastic (one child per dielectric vertex), 1 the reference's two-way split
    d.seed = seed
    d.kernel = kernel
    d.reserved = tune
    d.planes = planes
    d.reserved2 = tune2
    d.integrator = integrator
    d.profile = profile
    return d


class Scene:
    """Device-resident scene (SoA geometry + BVH).  `source` is a structured Object array
    (spheres) or an abi.SceneHolder (spheres and meshes)."""

    def __init__(self, source, device=0, all_trees=False):
        """all_trees: also build the BVH2 and the uncompressed BVH4 (RTB_SCENE_ALL_TREES) that the
        parity probes (trace_rays use_bvh 2..4) and the megakernel variants (kernel 1..5) walk"""
        cu, _ = load()
        self._cu = cu
        self._h = C.c_void_p()
        self.device = device
        flags = 1 if all_trees else 0
        if isinstance(source, abi.SceneHolder):
            self._src = source
            _check(cu.rtb_scene_create_flags(C.addressof(source.objects), source.n, device, flags, C.byref(self._h)),
                   "rtb_scene_create")
        else:
            arr = np.ascontiguousarray(source, dtype=abi.OBJECT_DTYPE)
            self._src = arr
            _check(cu.rtb_scene_create_objects_flags(arr.ctypes.data, len(arr), device, flags, C.byref(self._h)),
                   "rtb_scene_create_objects")

    def close(self):
        if self._h:
            self._cu.rtb_scene_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def info(self):
        i = abi.RtbSceneInfo()
        _check(self._cu.rtb_scene_info_get(self._h, C.byref(i)), "rtb_scene_info_get")
        return i

    def render_accum(self, camera, desc, d_accum_ptr, stream=None, want_counters=False):
        """device float[H*W*3] sum; asynchronous on `stream` unless counters are wanted"""
        cam = camera.as_array()
        ctr = abi.RtbCounters() if want_counters else None
        _check(self._cu.rtb_render_accum(self._h, cam.ctypes.data_as(C.POINTER(C.c_double)), C.byref(desc),
                                         C.c_void_p(d_accum_ptr), C.c_void_p(stream or 0),
                                         C.byref(ctr) if ctr is not None else None), "rtb_render_accum")
        return ctr

    def render(self, camera, desc, want_accum=False):
        """host u8 framebuffer (+ host float sums) through rtb_render"""
        cam = camera.as_array()
        fb = np.zeros((desc.height, desc.width, 3), dtype=np.uint8)
        acc = np.zeros((desc.height, desc.width, 3), dtype=np.float32) if want_accum else None
        ctr = abi.RtbCounters()
        _check(self._cu.rtb_render(self._h, cam.ctypes.data_as(C.POINTER(C.c_double)), C.byref(desc),
                                   fb.ctypes.data, acc.ctypes.data if want_accum else None, C.byref(ctr)),
               "rtb_render")
        return fb, acc, ctr

    def trace_rays(self, rays, use_bvh=True):
        rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
        n = len(rays)
        out = dict(ids=np.zeros(n, np.int32), prims=np.zeros(n, np.int64), t=np.zeros(n, np.float64),
                   points=np.zeros((n, 3), np.float64), normals=np.zeros((n, 3), np.float64),
                   uvs=np.zeros((n, 2), np.float64))
        _check(self._cu.rtb_trace_rays(self._h, rays.ctypes.data, n, int(use_bvh), out["ids"].ctypes.data,
                                       out["prims"].ctypes.data, out["t"].ctypes.data, out["points"].ctypes.data,
                                       out["normals"].ctypes.data, out["uvs"].ctypes.data), "rtb_trace_rays")
        return out

    def trace_rays_wf(self, rays, tune=0, perm=None):
        """the same records as trace_rays, from the wavefront renderer's trace kernel (rtb_trace_rays_wf): `tune` is
        a rtb_render_desc.reserved word (0 = the renderer's default kernel), `perm` the order the kernel fetches
        the rays in -> (records, abi.RtbCounters with prim_tests and node_visits)"""
        rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
        n = len(rays)
        out = dict(ids=np.zeros(n, np.int32), prims=np.zeros(n, np.int64), t=np.zeros(n, np.float64),
                   points=np.zeros((n, 3), np.float64), normals=np.zeros((n, 3), np.float64),
                   uvs=np.zeros((n, 2), np.float64))
        p = None if perm is None else np.ascontiguousarray(perm, dtype=np.uint32)
        if p is not None and p.shape != (n,):
            raise ValueError(f"perm must have {n} entries")
        ctr = abi.RtbCounters()
        _check(self._cu.rtb_trace_rays_wf(self._h, rays.ctypes.data, n, int(tune), p.ctypes.data if p is not None else None,
                                          out["ids"].ctypes.data, out["prims"].ctypes.data, out["t"].ctypes.data,
                                          out["points"].ctypes.data, out["normals"].ctypes.data, out["uvs"].ctypes.data,
                                          C.byref(ctr)), "rtb_trace_rays_wf")
        return out, ctr

    def cast_rays(self, rays, max_depth=5):
        """cast_ray() of the Whitted integrator (raytracer.c:556-641) for arbitrary rays ->
        (rgb float64 [n, 3], cast_ray invocations per ray)"""
        rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
        n = len(rays)
        rgb = np.zeros((n, 3), np.float64)
        counts = np.zeros(n, np.uint64)
        _check(self._cu.rtb_cast_rays(self._h, rays.ctypes.data, n, int(max_depth), rgb.ctypes.data,
                                      counts.ctypes.data), "rtb_cast_rays")
        return rgb, counts

    def path_records(self, camera, desc, sample, n_vertices=2):
        cam = camera.as_array()
        n = desc.width * desc.height
        out = dict(ids=np.zeros((n, n_vertices), np.int32), points=np.zeros((n, n_vertices, 3), np.float64),
                   normals=np.zeros((n, n_vertices, 3), np.float64), dists=np.zeros((n, n_vertices), np.float64),
                   radiance=np.zeros((n, 3), np.float32))
        _check(self._cu.rtb_path_records(self._h, cam.ctypes.data_as(C.POINTER(C.c_double)), C.byref(desc), sample,
                                         n_vertices, out["ids"].ctypes.data, out["points"].ctypes.data,
                                         out["normals"].ctypes.data, out["dists"].ctypes.data,
                                         out["radiance"].ctypes.data), "rtb_path_records")
        return out


# ---- all the GPUs of one box (rtb_comm_*, include/rtb200.h) ---------------------------------------

UNIQUE_ID_BYTES = 128


_nccl_preloaded = False


def _prefer_bundled_nccl():
    """librtb200.so binds libnccl.so.2 with dlopen on first use (a copy already in the process wins).  In a
    Python process PyTorch may be imported LATER and needs its own, newer NCCL under the same soname: load
    that copy first, so both sides share it whatever the import order.  A C caller gets the system's."""
    global _nccl_preloaded
    if _nccl_preloaded or os.environ.get("RTB_NCCL_LIB"):
        return
    _nccl_preloaded = True
    try:
        import importlib.util
        spec = importlib.util.find_spec("nvidia")
        for base in (spec.submodule_search_locations if spec else []):
            cand = os.path.join(base, "nccl", "lib", "libnccl.so.2")
            if os.path.exists(cand):
                C.CDLL(cand, mode=C.RTLD_GLOBAL)
                return
    except (ImportError, OSError, AttributeError):
        pass


def comm_unique_id():
    """rank 0 of a one-process-per-GPU job: the 128-byte id the other ranks need (send it through the
    launcher's own channel, e.g. torch.distributed.broadcast)"""
    cu, _ = load()
    _prefer_bundled_nccl()
    buf = (C.c_ubyte * UNIQUE_ID_BYTES)()
    _check(cu.rtb_comm_unique_id(buf), "rtb_comm_unique_id")
    return bytes(buf)


def shard_samples(sample_begin, sample_end, rank, n_ranks):
    """the sample range rank `rank` renders (rtb_comm_shard_samples; host arithmetic only)"""
    cu, _ = load()
    a, b = C.c_int(), C.c_int()
    _check(cu.rtb_comm_shard_samples(sample_begin, sample_end, rank, n_ranks, C.byref(a), C.byref(b)),
           "rtb_comm_shard_samples")
    return a.value, b.value


def _source_records(source):
    """-> (pointer, count, record bytes, keep-alive) for a structured Object array or an abi.SceneHolder"""
    if isinstance(source, abi.SceneHolder):
        return C.addressof(source.objects), source.n, 96, source
    arr = np.ascontiguousarray(source, dtype=abi.OBJECT_DTYPE)
    return arr.ctypes.data, len(arr), 88, arr


class Comm:
    """A group of GPUs, one rank each.  Comm.rank(...) = this process is one rank (torchrun);
    Comm.local(n) = this process drives n GPUs (what render() does for RenderParams.num_gpus > 1)."""

    def __init__(self, handle):
        cu, _ = load()
        self._cu, self._h = cu, handle
        self.size = cu.rtb_comm_size(handle)
        self.local_ranks = cu.rtb_comm_local_ranks(handle)

    @classmethod
    def rank(cls, unique_id, rank, n_ranks, device):
        cu, _ = load()
        _prefer_bundled_nccl()
        h = C.c_void_p()
        buf = (C.c_ubyte * UNIQUE_ID_BYTES).from_buffer_copy(unique_id)
        _check(cu.rtb_comm_create_rank(buf, rank, n_ranks, device, C.byref(h)), "rtb_comm_create_rank")
        return cls(h)

    @classmethod
    def local(cls, n_devices, devices=None):
        cu, _ = load()
        _prefer_bundled_nccl()
        h = C.c_void_p()
        arr = (C.c_int * n_devices)(*devices) if devices is not None else None
        _check(cu.rtb_comm_create_local(arr, n_devices, C.byref(h)), "rtb_comm_create_local")
        return cls(h)

    def close(self):
        if self._h:
            self._cu.rtb_comm_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def scene(self, source, all_trees=False):
        """collective: sharded upload + all-gather + per-GPU BVH build -> MultiScene"""
        ptr, n, kind, keep = _source_records(source)
        handles = (C.c_void_p * self.local_ranks)()
        _check(self._cu.rtb_comm_scene_create(self._h, ptr, n, kind, 1 if all_trees else 0, handles),
               "rtb_comm_scene_create")
        return MultiScene(self, handles, keep)

    def render_host(self, source, camera, desc, want_accum=False, want_counters=True, fb=None):
        """collective: the whole render() with host buffers on all GPUs (rtb_render_multi).
        The framebuffer (and sums) are valid on the process that holds rank 0.  `fb`: the caller's own
        (H, W, 3) uint8 buffer, like the framebuffer main.c allocates once (main.c:413)."""
        ptr, n, kind, keep = _source_records(source)
        cam = camera.as_array()
        if fb is None:
            fb = np.zeros((desc.height, desc.width, 3), dtype=np.uint8)
        acc = np.zeros((desc.height, desc.width, 3), dtype=np.float32) if want_accum else None
        ctr = abi.RtbCounters() if want_counters else None
        _check(self._cu.rtb_render_multi(self._h, ptr, n, kind, cam.ctypes.data_as(C.POINTER(C.c_double)), C.byref(desc),
                                         fb.ctypes.data, acc.ctypes.data if want_accum else None,
                                         C.byref(ctr) if ctr is not None else None), "rtb_render_multi")
        return fb, acc, ctr


class MultiScene:
    def __init__(self, comm, handles, keep):
        self._comm, self._handles, self._keep = comm, handles, keep

    def render(self, camera, desc, d_fb_root_ptr=None, want_counters=False):
        """collective, device-resident: accumulate (sample-sharded) -> ncclReduce -> tonemap on rank 0"""
        cam = camera.as_array()
        ctr = abi.RtbCounters() if want_counters else None
        _check(self._comm._cu.rtb_comm_render(self._comm._h, self._handles, cam.ctypes.data_as(C.POINTER(C.c_double)),
                                              C.byref(desc), C.c_void_p(d_fb_root_ptr or 0),
                                              C.byref(ctr) if ctr is not None else None), "rtb_comm_render")
        return ctr

    def close(self):
        for k in range(len(self._handles)):
            if self._handles[k]:
                self._comm._cu.rtb_scene_destroy(self._handles[k])
                self._handles[k] = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


def tonemap(d_accum_ptr, width, height, total_samples, d_fb_ptr, device=0, stream=None):
    cu, _ = load()
    _check(cu.rtb_tonemap(C.c_void_p(d_accum_ptr), width, height, total_samples, C.c_void_p(d_fb_ptr), device,
                          C.c_void_p(stream or 0)), "rtb_tonemap")


def release_workspace(device=0):
    """give the per-device cache of parked buffers (ray queues, scene arrays) back to the driver"""
    cu, _ = load()
    cu.rtb_release_workspace.restype = None
    cu.rtb_release_workspace(C.c_int(device))


def probe_l2_bandwidth(nbytes=32 << 20, iters=50, device=0):
    """read bandwidth (GB/s) of an L2-resident buffer: the denominator for the walk's algorithmic bytes"""
    cu, _ = load()
    out = C.c_float(0.0)
    _check(cu.rtb_probe_l2_bandwidth(nbytes, iters, device, C.byref(out)), "rtb_probe_l2_bandwidth")
    return float(out.value)


def probe_fp32_tflops(iters=4096, device=0):
    """FP32 FMA throughput (TFLOP/s) measured on the device: the denominator for the walk's algorithmic flops"""
    cu, _ = load()
    out = C.c_float(0.0)
    cu.rtb_probe_fp32_tflops.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_float)]
    _check(cu.rtb_probe_fp32_tflops(iters, device, C.byref(out)), "rtb_probe_fp32_tflops")
    return float(out.value)


def philox(ctr, key, device=0):
    cu, _ = load()
    ctr = np.ascontiguousarray(ctr, dtype=np.uint32).reshape(-1, 4)
    key = np.ascontiguousarray(key, dtype=np.uint32).reshape(-1, 2)
    out = np.zeros_like(ctr)
    _check(cu.rtb_philox4x32_10(ctr.ctypes.data, key.ctypes.data, len(ctr), out.ctypes.data, device),
           "rtb_philox4x32_10")
    return out
