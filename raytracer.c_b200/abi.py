"""ctypes mirrors of the reference's C records (raytracer.h:60-131) and of rtb200.h.

Shared by the product bindings (api.py) and by the tests' oracle bindings, so both sides
describe a scene with the very same bytes.  Sizes are asserted against the values
measured on the reference with gcc 13.3 x86-64 (SURVEY.md 8a): Vertex 40, Ray 48,
Material 80, Sphere 32, TriangleMesh 16, Object 88, Hit 80, Camera 96, Options 56.
"""
import ctypes as C

import numpy as np

M_DEFAULT = 1 << 1
M_REFLECTION = 1 << 2
M_REFRACTION = 1 << 3
M_CHECKERED = 1 << 4

GEOMETRY_SPHERE = 0
GEOMETRY_MESH = 1

SCENE_SEED = 1666943821  # main.c:182


class Vec2(C.Structure):
    _fields_ = [("x", C.c_double), ("y", C.c_double)]


class Vec3(C.Structure):
    _fields_ = [("x", C.c_double), ("y", C.c_double), ("z", C.c_double)]

    def tolist(self):
        return [self.x, self.y, self.z]


class Vertex(C.Structure):
    _fields_ = [("pos", Vec3), ("tex", Vec2)]


class Material(C.Structure):
    _fields_ = [("flags", C.c_uint32), ("color", Vec3), ("emission", Vec3),
                ("ka", C.c_double), ("ks", C.c_double), ("kd", C.c_double)]


class Sphere(C.Structure):
    _fields_ = [("center", Vec3), ("radius", C.c_double)]


class TriangleMesh(C.Structure):
    _fields_ = [("num_triangles", C.c_size_t), ("vertices", C.POINTER(Vertex))]


class Object(C.Structure):
    """flat sphere record, raytracer.h:104-111"""
    _fields_ = [("flags", C.c_uint32), ("radius", C.c_double), ("center", Vec3),
                ("color", Vec3), ("emission", Vec3)]


class Geometry(C.Union):
    _fields_ = [("mesh", C.POINTER(TriangleMesh)), ("sphere", C.POINTER(Sphere))]


class SceneObject(C.Structure):
    """the record commented out at raytracer.h:95-102, resurrected for meshes"""
    _fields_ = [("type", C.c_int), ("material", Material), ("geometry", Geometry)]


class Camera(C.Structure):
    _fields_ = [("position", Vec3), ("horizontal", Vec3), ("vertical", Vec3),
                ("lower_left_corner", Vec3)]

    def as_array(self):
        return np.frombuffer(bytes(self), dtype=np.float64).copy()


class Options(C.Structure):
    _fields_ = [("background", Vec3), ("result", C.c_char_p), ("obj", C.c_char_p),
                ("width", C.c_int), ("height", C.c_int), ("samples", C.c_int)]


class RenderParams(C.Structure):
    _fields_ = [("max_depth", C.c_int), ("seed", C.c_uint64), ("sample_offset", C.c_int),
                ("total_samples", C.c_int), ("dielectric_mode", C.c_int), ("device", C.c_int),
                ("accum_out", C.POINTER(C.c_float)), ("integrator", C.c_int), ("num_gpus", C.c_int)]


class SceneMix(C.Structure):
    _fields_ = [("emissive", C.c_double), ("refraction", C.c_double), ("reflection", C.c_double)]


class RtbRenderDesc(C.Structure):
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("sample_begin", C.c_int),
                ("sample_end", C.c_int), ("max_depth", C.c_int), ("dielectric_mode", C.c_int),
                ("seed", C.c_uint64), ("kernel", C.c_int), ("reserved", C.c_int),
                ("planes", C.c_int), ("reserved2", C.c_int), ("integrator", C.c_int), ("profile", C.c_int)]


class RtbCounters(C.Structure):
    _fields_ = [("rays", C.c_ulonglong), ("rays_intersected", C.c_ulonglong),
                ("prim_tests", C.c_ulonglong), ("node_visits", C.c_ulonglong),
                ("paths", C.c_ulonglong), ("launches", C.c_ulonglong),
                ("gpu_ms", C.c_float), ("build_ms", C.c_float),
                ("trace_ms", C.c_float), ("shade_ms", C.c_float), ("trace_launches", C.c_ulonglong)]


class RtbSceneInfo(C.Structure):
    _fields_ = [("n_objects", C.c_size_t), ("n_spheres", C.c_size_t), ("n_triangles", C.c_size_t),
                ("n_bvh_prims", C.c_size_t), ("n_bvh_nodes", C.c_size_t), ("n_big_prims", C.c_size_t),
                ("device_bytes", C.c_size_t), ("build_ms", C.c_float), ("bvh_depth", C.c_int),
                ("device", C.c_int), ("double_triangles", C.c_int), ("double_texcoords", C.c_int),
                ("bvh4_depth", C.c_int)]


EXPECTED_SIZES = {Vertex: 40, Material: 80, Sphere: 32, TriangleMesh: 16, Object: 88,
                  SceneObject: 96, Camera: 96, Options: 56}
for _t, _n in EXPECTED_SIZES.items():
    assert C.sizeof(_t) == _n, (_t.__name__, C.sizeof(_t), _n)


# ---- numpy <-> record helpers --------------------------------------------------------

OBJECT_DTYPE = np.dtype({
    "names": ["flags", "radius", "center", "color", "emission"],
    "formats": [np.uint32, np.float64, (np.float64, 3), (np.float64, 3), (np.float64, 3)],
    "offsets": [0, 8, 16, 40, 64],
    "itemsize": 88,
})
VERTEX_DTYPE = np.dtype([("pos", np.float64, 3), ("tex", np.float64, 2)])
assert VERTEX_DTYPE.itemsize == 40


def objects_to_numpy(objs, n):
    """view an Object[n] ctypes array as a structured numpy array (copy)"""
    buf = C.string_at(C.addressof(objs), 88 * n)
    return np.frombuffer(buf, dtype=OBJECT_DTYPE).copy()


def objects_from_numpy(arr):
    arr = np.ascontiguousarray(arr, dtype=OBJECT_DTYPE)
    out = (Object * len(arr))()
    C.memmove(out, arr.ctypes.data, 88 * len(arr))
    return out


class SceneHolder:
    """A SceneObject[] plus everything it points to, kept alive together."""

    def __init__(self):
        self.objects = None
        self.n = 0
        self._keep = []
        self._free = []  # (libc, pointer) pairs malloc'ed by the C scene builders

    def __del__(self):
        for libc, ptr in getattr(self, "_free", []):
            try:
                libc.free(ptr)
            except Exception:
                pass
        self._free = []

    @staticmethod
    def from_objects(obj_array):
        """wrap a structured Object array (spheres only)"""
        arr = np.ascontiguousarray(obj_array, dtype=OBJECT_DTYPE)
        h = SceneHolder()
        h.n = len(arr)
        h.objects = (SceneObject * max(1, h.n))()
        spheres = (Sphere * max(1, h.n))()
        h._keep.append(spheres)
        for i in range(h.n):
            h._fill_sphere(i, spheres, i, arr[i])
        return h

    def _fill_sphere(self, i, spheres, si, rec):
        spheres[si].center = Vec3(*[float(v) for v in rec["center"]])
        spheres[si].radius = float(rec["radius"])
        so = self.objects[i]
        so.type = GEOMETRY_SPHERE
        so.material.flags = int(rec["flags"])
        so.material.color = Vec3(*[float(v) for v in rec["color"]])
        so.material.emission = Vec3(*[float(v) for v in rec["emission"]])
        so.geometry.sphere = C.pointer(spheres[si])

    @staticmethod
    def build(items):
        """items: list of ("sphere", rec) with rec an OBJECT_DTYPE scalar/dict, or
        ("mesh", vertices[VERTEX_DTYPE, 3*T], flags, color, emission)"""
        h = SceneHolder()
        h.n = len(items)
        h.objects = (SceneObject * max(1, h.n))()
        n_sph = sum(1 for it in items if it[0] == "sphere")
        spheres = (Sphere * max(1, n_sph))()
        h._keep.append(spheres)
        si = 0
        for i, it in enumerate(items):
            if it[0] == "sphere":
                h._fill_sphere(i, spheres, si, it[1])
                si += 1
            else:
                _, verts, flags, color, emission = it
                verts = np.ascontiguousarray(verts, dtype=VERTEX_DTYPE)
                assert len(verts) % 3 == 0
                mesh = TriangleMesh()
                mesh.num_triangles = len(verts) // 3
                mesh.vertices = C.cast(verts.ctypes.data, C.POINTER(Vertex))
                h._keep += [verts, mesh]
                so = h.objects[i]
                so.type = GEOMETRY_MESH
                so.material.flags = int(flags)
                so.material.color = Vec3(*[float(v) for v in color])
                so.material.emission = Vec3(*[float(v) for v in emission])
                so.geometry.mesh = C.pointer(mesh)
        return h
