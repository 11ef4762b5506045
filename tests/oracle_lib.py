"""TEST INFRASTRUCTURE: ctypes bindings of the two checkers.

  oracle/liboracle.so     the CPU restatement (oracle/oracle.c)
  oracle/_ref/libref.so   the unmodified reference compiled where it lies (oracle/ref_harness.c)

Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs import this module.
The product package never does.
"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry  # noqa: E402

pkg = entry.load_package()
abi = pkg.abi

ORACLE_SO = os.path.join(ROOT, "oracle", "liboracle.so")
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libref.so")

RNG = {"libc": 0, "stream": 1, "philox": 2}
DIELECTRIC = {"stochastic": 0, "split": 1}
INTEGRATOR = {"path": 0, "whitted": 1}


class OracleParams(C.Structure):
    _fields_ = [("max_depth", C.c_int), ("rng_mode", C.c_int), ("dielectric_mode", C.c_int),
                ("sample_offset", C.c_int), ("seed", C.c_uint64), ("threads", C.c_int), ("integrator", C.c_int)]


_oracle = None
_ref = None


def oracle():
    global _oracle
    if _oracle is None:
        if not os.path.exists(ORACLE_SO):
            raise RuntimeError(f"{ORACLE_SO} missing: run `make -C oracle`")
        lib = C.CDLL(ORACLE_SO)
        lib.oracle_trace_path_stream.restype = C.c_longlong
        lib.oracle_intersect_sphere.restype = C.c_int
        lib.oracle_intersect_triangle.restype = C.c_int
        lib.oracle_intersect_sphere.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_void_p]
        lib.oracle_checkered.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_void_p]
        lib.oracle_refract.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_void_p]
        lib.oracle_camera_ray.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_void_p]
        lib.oracle_keyed_jitter.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p]
        _oracle = lib
    return _oracle


def have_ref():
    return os.path.exists(REF_SO)


def ref():
    global _ref
    if _ref is None:
        if not have_ref():
            raise RuntimeError(f"{REF_SO} missing: run `make -C oracle ref` where /root/reference exists")
        lib = C.CDLL(REF_SO)
        lib.ref_sizeof.restype = C.c_size_t
        lib.ref_ray_count.restype = C.c_longlong
        lib.ref_intersection_test_count.restype = C.c_longlong
        lib.ref_trace_path_stream.restype = C.c_longlong
        lib.ref_intersect_sphere.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_void_p]
        lib.ref_checkered.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_void_p]
        lib.ref_refract.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_void_p]
        lib.ref_camera_ray.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_void_p]
        lib.ref_random_double_from.restype = C.c_double
        lib.ref_random_double_from.argtypes = [C.c_int32]
        _ref = lib
    return _ref


def params(rng="libc", dielectric="split", max_depth=5, seed=abi.SCENE_SEED, sample_offset=0, threads=None,
           integrator="path"):
    p = OracleParams()
    p.max_depth = max_depth
    p.rng_mode = RNG[rng]
    p.dielectric_mode = DIELECTRIC[dielectric]
    p.sample_offset = sample_offset
    p.seed = seed
    p.threads = threads if threads is not None else (os.cpu_count() or 1)
    p.integrator = INTEGRATOR[integrator]
    return p


def _holder(scene):
    if isinstance(scene, abi.SceneHolder):
        return scene
    return abi.SceneHolder.from_objects(scene)


def _dptr(a):
    return a.ctypes.data_as(C.c_void_p)


# ---- oracle (restatement) ----------------------------------------------------------------

def init_camera(width, height, pos=(0.0, 0.0, 50.0), target=(0.0, 0.0, 0.0)):
    cam = abi.Camera()
    p = np.array(pos, dtype=np.float64)
    t = np.array(target, dtype=np.float64)
    oracle().oracle_init_camera(C.byref(cam), _dptr(p), _dptr(t), width, height)
    return cam


def camera_ray(cam, u, v):
    out = np.zeros(6)
    oracle().oracle_camera_ray(C.byref(cam), float(u), float(v), _dptr(out))
    return out


def render_sum(scene, cam, width, height, samples, rng="philox", dielectric="stochastic", max_depth=5,
               seed=abi.SCENE_SEED, sample_offset=0, threads=None, integrator="path"):
    """per-pixel SUM over samples, float64 [H,W,3]; returns (sum, (rays, prim_tests))"""
    h = _holder(scene)
    out = np.zeros((height, width, 3), dtype=np.float64)
    ctr = (C.c_longlong * 2)()
    p = params(rng, dielectric, max_depth, seed, sample_offset, threads, integrator)
    oracle().oracle_render_sum(_dptr(out), h.objects, C.c_size_t(h.n), C.byref(cam), width, height, samples,
                               C.byref(p), ctr)
    return out, (ctr[0], ctr[1])


def tonemap(sum_rgb, total_samples):
    sum_rgb = np.ascontiguousarray(sum_rgb, dtype=np.float64)
    hh, ww, _ = sum_rgb.shape
    fb = np.zeros((hh, ww, 3), dtype=np.uint8)
    oracle().oracle_tonemap(_dptr(fb), _dptr(sum_rgb), ww, hh, total_samples)
    return fb


def render(scene, cam, width, height, samples, **kw):
    s, ctr = render_sum(scene, cam, width, height, samples, **kw)
    return tonemap(s, samples), ctr


def intersect_rays(scene, rays, threads=None):
    h = _holder(scene)
    rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
    n = len(rays)
    out = dict(ids=np.zeros(n, np.int32), prims=np.zeros(n, np.int64), t=np.zeros(n), points=np.zeros((n, 3)),
               normals=np.zeros((n, 3)), uvs=np.zeros((n, 2)))
    oracle().oracle_intersect_rays(h.objects, C.c_size_t(h.n), _dptr(rays), C.c_longlong(n), _dptr(out["ids"]),
                                   _dptr(out["prims"]), _dptr(out["t"]), _dptr(out["points"]),
                                   _dptr(out["normals"]), _dptr(out["uvs"]),
                                   threads if threads is not None else (os.cpu_count() or 1))
    return out


def cast_rays(scene, rays, max_depth=5, threads=None):
    """the restated cast_ray (raytracer.c:556-641) -> (rgb [n,3], cast_ray calls per ray)"""
    h = _holder(scene)
    rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
    n = len(rays)
    rgb = np.zeros((n, 3))
    counts = np.zeros(n, np.int64)
    oracle().oracle_cast_rays(h.objects, C.c_size_t(h.n), _dptr(rays), C.c_longlong(n), int(max_depth), _dptr(rgb),
                              _dptr(counts), threads if threads is not None else (os.cpu_count() or 1))
    return rgb, counts


def trace_path_stream(scene, ray6, stream, depth=0, dielectric="split", max_depth=5):
    h = _holder(scene)
    ray6 = np.ascontiguousarray(ray6, dtype=np.float64)
    stream = np.ascontiguousarray(stream, dtype=np.int32)
    rad = np.zeros(3)
    p = params("stream", dielectric, max_depth)
    used = oracle().oracle_trace_path_stream(h.objects, C.c_size_t(h.n), _dptr(ray6), depth, C.byref(p),
                                             _dptr(stream), C.c_longlong(len(stream)), _dptr(rad))
    return rad, used


def path_records(scene, cam, width, height, sample, n_vertices=2, dielectric="stochastic", max_depth=5,
                 seed=abi.SCENE_SEED, threads=None):
    h = _holder(scene)
    n = width * height
    out = dict(ids=np.zeros((n, n_vertices), np.int32), points=np.zeros((n, n_vertices, 3)),
               normals=np.zeros((n, n_vertices, 3)), dists=np.zeros((n, n_vertices)), radiance=np.zeros((n, 3)))
    p = params("philox", dielectric, max_depth, seed, 0, threads)
    oracle().oracle_path_records(h.objects, C.c_size_t(h.n), C.byref(cam), width, height, sample, n_vertices,
                                 C.byref(p), _dptr(out["ids"]), _dptr(out["points"]), _dptr(out["normals"]),
                                 _dptr(out["dists"]), _dptr(out["radiance"]))
    return out


# oracle.h OracleVertex: one vertex of trace_path in forward form
VERTEX_DTYPE = np.dtype([("ray", "f8", 6), ("tp", "f8", 3), ("contrib", "f8", 3), ("t", "f8"), ("child_ray", "f8", (2, 6)),
                         ("child_tp", "f8", (2, 3)), ("prim", "i8"), ("pixel", "u4"), ("sample", "u4"), ("branch", "u4"),
                         ("child_branch", "u4", 2), ("depth", "i4"), ("id", "i4"), ("survived", "i4"), ("rays", "i4"),
                         ("n_children", "i4"), ("cut", "i4", 2), ("tries", "i4"), ("flipped", "i4")], align=True)
assert VERTEX_DTYPE.itemsize == 312


def path_vertex(scene, rays, depth, branch, pixel, sample, tp, dielectric="stochastic", max_depth=5,
                seed=abi.SCENE_SEED, threads=None):
    """one forward vertex of trace_path per ray (oracle_path_vertex), keyed by (pixel, sample, depth | branch << 8),
    from the incoming throughput `tp` [n, 3] -> VERTEX_DTYPE [n]"""
    h = _holder(scene)
    rays = np.ascontiguousarray(rays, np.float64).reshape(-1, 6)
    n = len(rays)
    cols = [np.ascontiguousarray(np.broadcast_to(v, (n,)), dt) for v, dt in
            ((depth, np.int32), (branch, np.uint32), (pixel, np.uint32), (sample, np.uint32))]
    tp = np.ascontiguousarray(tp, np.float64).reshape(n, 3)
    out = np.zeros(n, VERTEX_DTYPE)
    p = params("philox", dielectric, max_depth, seed, 0, threads)
    oracle().oracle_path_vertex(h.objects, C.c_size_t(h.n), C.byref(p), _dptr(rays), *(_dptr(c) for c in cols), _dptr(tp),
                                C.c_longlong(n), _dptr(out))
    return out


def path_log(scene, cam, width, height, samples, dielectric="stochastic", max_depth=5, seed=abi.SCENE_SEED,
             sample_offset=0, threads=None):
    """every vertex of every path of samples [sample_offset, sample_offset + samples) (oracle_path_log) ->
    VERTEX_DTYPE [n], rows in order"""
    h = _holder(scene)
    p = params("philox", dielectric, max_depth, seed, sample_offset, threads)
    lib = oracle()
    lib.oracle_path_log.restype = C.c_longlong
    cap = width * height * samples * 4
    while True:
        out = np.zeros(cap, VERTEX_DTYPE)
        n = lib.oracle_path_log(h.objects, C.c_size_t(h.n), C.byref(cam), width, height, samples, C.byref(p),
                                _dptr(out), C.c_longlong(cap))
        if n <= cap:
            return out[:n]
        cap = n


def philox(ctr, key):
    ctr = np.ascontiguousarray(ctr, dtype=np.uint32).reshape(-1, 4)
    key = np.ascontiguousarray(key, dtype=np.uint32).reshape(-1, 2)
    out = np.zeros_like(ctr)
    for i in range(len(ctr)):
        oracle().oracle_philox4x32_10(_dptr(ctr[i:i + 1]), _dptr(key[i:i + 1]), _dptr(out[i:i + 1]))
    return out


def keyed_jitter(seed, pixel, sample):
    out = np.zeros(2)
    oracle().oracle_keyed_jitter(C.c_uint64(seed), C.c_uint32(pixel), C.c_uint32(sample), _dptr(out))
    return out


# ---- the unmodified reference ----------------------------------------------------------------

def ref_init_camera(width, height, pos=(0.0, 0.0, 50.0), target=(0.0, 0.0, 0.0)):
    cam = abi.Camera()
    p = np.array(pos, dtype=np.float64)
    t = np.array(target, dtype=np.float64)
    ref().ref_init_camera(C.byref(cam), _dptr(p), _dptr(t), width, height)
    return cam


def ref_camera_ray(cam, u, v):
    out = np.zeros(6)
    ref().ref_camera_ray(C.byref(cam), float(u), float(v), _dptr(out))
    return out


def ref_render(objs, cam, width, height, samples, seed=abi.SCENE_SEED, max_depth=5, threads=1):
    arr = np.ascontiguousarray(objs, dtype=abi.OBJECT_DTYPE)
    fb = np.zeros((height, width, 3), dtype=np.uint8)
    ref().ref_reset_counters()
    ref().ref_render(_dptr(fb), _dptr(arr), C.c_size_t(len(arr)), C.byref(cam), width, height, samples,
                     C.c_uint(seed), max_depth, threads)
    return fb, (ref().ref_ray_count(), ref().ref_intersection_test_count())


def ref_render_mean(objs, cam, width, height, samples, seed=abi.SCENE_SEED, max_depth=5):
    arr = np.ascontiguousarray(objs, dtype=abi.OBJECT_DTYPE)
    out = np.zeros((height, width, 3), dtype=np.float64)
    ref().ref_reset_counters()
    ref().ref_render_mean(_dptr(out), _dptr(arr), C.c_size_t(len(arr)), C.byref(cam), width, height, samples,
                          C.c_uint(seed), max_depth)
    return out, (ref().ref_ray_count(), ref().ref_intersection_test_count())


def ref_intersect_rays(objs, rays):
    arr = np.ascontiguousarray(objs, dtype=abi.OBJECT_DTYPE)
    rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
    n = len(rays)
    out = dict(ids=np.zeros(n, np.int32), points=np.zeros((n, 3)), normals=np.zeros((n, 3)),
               uvs=np.zeros((n, 2)), last_t=np.zeros(n))
    ref().ref_intersect_rays(_dptr(arr), C.c_size_t(len(arr)), _dptr(rays), C.c_longlong(n), _dptr(out["ids"]),
                             _dptr(out["points"]), _dptr(out["normals"]), _dptr(out["uvs"]), _dptr(out["last_t"]))
    return out


def ref_cast_rays(objs, rays, max_depth=5):
    """the reference's own cast_ray for arbitrary rays -> (rgb [n,3], cast_ray calls per ray)"""
    arr = np.ascontiguousarray(objs, dtype=abi.OBJECT_DTYPE)
    rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
    n = len(rays)
    rgb = np.zeros((n, 3))
    counts = np.zeros(n, np.int64)
    ref().ref_cast_rays(_dptr(arr), C.c_size_t(len(arr)), _dptr(rays), C.c_longlong(n), int(max_depth), _dptr(rgb),
                        _dptr(counts))
    return rgb, counts


def ref_trace_path_stream(objs, ray6, stream, depth=0, max_depth=5):
    arr = np.ascontiguousarray(objs, dtype=abi.OBJECT_DTYPE)
    ray6 = np.ascontiguousarray(ray6, dtype=np.float64)
    stream = np.ascontiguousarray(stream, dtype=np.int32)
    rad = np.zeros(3)
    used = ref().ref_trace_path_stream(_dptr(arr), C.c_size_t(len(arr)), _dptr(ray6), depth, max_depth,
                                       _dptr(stream), C.c_longlong(len(stream)), _dptr(rad))
    return rad, used
