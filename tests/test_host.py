"""CPU-only tests of the host side: the C-ABI libraries load and export every declared
symbol (no compute call is made -- there is no GPU here), the scene builders, load_obj, the
PNG writer, the CLI's argument handling, and the multi-GPU sample sharding over gloo."""
import ctypes as C
import os
import re
import struct
import subprocess
import sys
import zlib

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- the boundary ------------------------------------------------------------------------------

def test_libraries_load_and_export_declared_symbols(api):
    cu, host = api.load()
    for name in api.RTB_SYMBOLS:
        assert hasattr(cu, name), f"librtb200.so does not export {name}"
    for name in api.HOST_SYMBOLS:
        assert hasattr(host, name), f"libraraytracer_b200.so does not export {name}"
    assert cu.rtb_version().decode().startswith("rtb200")


def test_header_declarations_match_binding_list(api):
    """every function include/rtb200.h declares is in RTB_SYMBOLS (and the other way round)"""
    text = open(os.path.join(ROOT, "include", "rtb200.h")).read()
    declared = set(re.findall(r"\b(rtb_[a-z0-9_]+)\s*\(", text))
    assert declared == set(api.RTB_SYMBOLS), declared ^ set(api.RTB_SYMBOLS)
    text = open(os.path.join(ROOT, "include", "raytracer.h")).read()
    for name in ("render", "init_camera", "load_obj", "intersect_sphere", "intersect_triangle",
                 "calculate_surface_normal", "point_at", "random_double", "random_range", "print_v", "print_m",
                 "render_scene", "render_ex"):
        assert re.search(r"\b%s\s*\(" % name, text), name


def test_cuda_library_contains_sm100a_code():
    """the shipped kernels are compiled for sm_100a (no PTX-only fallback)"""
    so = os.path.join(ROOT, "raytracer.c_b200", "librtb200.so")
    out = subprocess.run(["cuobjdump", "-lelf", so], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump not available")
    assert "sm_100a" in out.stdout, out.stdout


def test_no_gpu_means_loud_failure_not_fallback(api, abi):
    """without a CUDA device the compute entry points fail with an error -- never a CPU path"""
    if api.device_count() > 0:
        pytest.skip("a GPU is present")
    objs = api.scene_default(64, 36)
    with pytest.raises(api.RtbError):
        api.Scene(objs)


def test_product_never_imports_the_oracle():
    """the package and bench's GPU arm must not reference oracle/ (checker only)"""
    pkg_dir = os.path.join(ROOT, "raytracer.c_b200")
    for dirpath, _, files in os.walk(pkg_dir):
        for f in files:
            if f.endswith((".py", ".c", ".h", ".cu", ".cuh")) or f == "Makefile":
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "oracle_lib" not in text and "liboracle" not in text and "libref" not in text, os.path.join(dirpath, f)


# ---- scenes -------------------------------------------------------------------------------------

def test_default_scene_is_the_reference_scene(api, abi):
    """main.c:244-397: 6 walls + 30 packed spheres + 2 lights; wall x-positions follow the aspect ratio (Q15)"""
    objs = api.scene_default(320, 180)
    assert len(objs) == 38
    assert (objs["radius"][:6] == 10000).all()
    room_w = 20 * 320 / 180
    assert objs["center"][2][0] == -10000 - room_w and objs["center"][3][0] == 10000 + room_w
    assert objs["center"][0][1] == -10020 and objs["center"][5][2] == 10060
    assert tuple(objs["center"][36]) == (0, 33.5, 0) and objs["radius"][36] == 15
    np.testing.assert_allclose(objs["emission"][36], (0, 750 / 255, 2400 / 255))
    assert tuple(objs["center"][37]) == (2, -17, 12)
    n_mirror = int((objs["flags"][6:36] == abi.M_REFLECTION).sum())
    assert n_mirror == 13 and int((objs["flags"][6:36] == abi.M_DEFAULT).sum()) == 17
    sq = api.scene_default(512, 512)
    assert sq["center"][3][0] == 10020


def test_sphere_field_generator(api, abi):
    """generate_random_spheres semantics (main.c:65-138): no overlaps, inside the box, mix"""
    a = api.scene_sphere_field(2000, 1920, 1080, seed=5)
    b = api.scene_sphere_field(2000, 1920, 1080, seed=5)
    c = api.scene_sphere_field(2000, 1920, 1080, seed=6)
    same = lambda p, q: all(np.array_equal(p[f], q[f]) for f in p.dtype.names)  # noqa: E731  (padding bytes excluded)
    assert same(a, b) and not same(a, c)
    assert len(a) == 2008
    s = a[6:2006]
    ctr, r = s["center"], s["radius"]
    half = np.array([20 * 1920 / 1080, 20, 30])
    assert (np.abs(ctr) + r[:, None] <= half + 1e-9).all()
    d = np.linalg.norm(ctr[:, None, :] - ctr[None, :, :], axis=2) + np.eye(len(s)) * 1e9
    assert (d >= r[:, None] + r[None, :]).all(), "spheres overlap"
    emissive = (s["emission"].sum(axis=1) > 0).mean()
    assert 0.45 < emissive < 0.55
    assert 0.15 < (s["flags"] == abi.M_REFRACTION).mean() < 0.25
    assert 0.15 < (s["flags"] == abi.M_REFLECTION).mean() < 0.25


def test_heightfield_mesh(api, ol):
    verts = api.heightfield_mesh(8, 30.0)
    assert len(verts) == 3 * 2 * 8 * 8
    pos = verts["pos"]
    assert np.array_equal(pos, pos.astype(np.float32).astype(np.float64)), "OBJ-style float positions"
    # winding: calculate_surface_normal (raytracer.c:42-45) must point up
    n = np.zeros(3)
    for t in range(0, len(verts) // 3, 7):
        v9 = np.ascontiguousarray(pos[3 * t:3 * t + 3].reshape(-1))
        ol.oracle().oracle_surface_normal(v9.ctypes.data_as(C.c_void_p), n.ctypes.data_as(C.c_void_p))
        assert n[1] > 0.3


# ---- load_obj -----------------------------------------------------------------------------------

CUBE_OBJ = """# cube in the style of the reference's assets/cube.obj: quads, v//vn corners, no vt
mtllib cube.mtl
o Cube
v 1.000000 -1.000000 -1.000000
v 1.000000 -1.000000 1.000000
v -1.000000 -1.000000 1.000000
v -1.000000 -1.000000 -1.000000
v 1.000000 1.000000 -0.999999
v 0.999999 1.000000 1.000001
v -1.000000 1.000000 1.000000
v -1.000000 1.000000 -1.000000
vn 0.0000 -1.0000 0.0000
vn 0.0000 1.0000 0.0000
usemtl CubeMaterial
s off
f 1//1 2//1 3//1 4//1
f 5//2 8//2 7//2 6//2
f 1//1 5//1 6//1 2//1
f 2//1 6//1 7//1 3//1
f 3//1 7//1 8//1 4//1
f 5//2 1//2 4//2 8//2"""


def test_load_obj_cube(api, tmp_path):
    """8 vertices, 6 quads -> 12 triangles by fan triangulation (i0, i[k-1], i[k]),
    positions narrowed to float, missing texcoords -> (0,0); no trailing newline needed"""
    p = tmp_path / "cube.obj"
    p.write_text(CUBE_OBJ)  # deliberately no final newline (cube.obj:30-31 works around a tinyobj bug)
    v = api.load_obj(str(p))
    assert len(v) == 36
    assert (v["tex"] == 0).all()
    f32 = lambda x: float(np.float32(x))  # noqa: E731
    assert np.array_equal(v["pos"][0], (1, -1, -1)) and np.array_equal(v["pos"][1], (1, -1, 1))
    assert np.array_equal(v["pos"][2], (-1, -1, 1))
    # second triangle of the first quad: (v1, v3, v4)
    assert np.array_equal(v["pos"][3], (1, -1, -1)) and np.array_equal(v["pos"][4], (-1, -1, 1))
    assert np.array_equal(v["pos"][5], (-1, -1, -1))
    assert v["pos"][6][2] == f32(-0.999999) and v["pos"][6][2] != -0.999999


def test_load_obj_features(api, tmp_path):
    text = "v 0 0 0\nv 1 0 0\nv 0 1 0\nv 0 0 1\nvt 0.25 0.5\nvt 0.75 1\nvt 0 0\n" \
           "f 1/1 2/2 3/3\nf -3/-2 -2/-1 -1\n# comment\nf 1 2 3 4 1\n"
    p = tmp_path / "t.obj"
    p.write_text(text)
    v = api.load_obj(str(p))
    assert len(v) == 3 * (1 + 1 + 3)
    assert np.array_equal(v["tex"][0], (0.25, 0.5)) and np.array_equal(v["tex"][1], (0.75, 1))
    # negative indices are relative to the end
    assert np.array_equal(v["pos"][3], (1, 0, 0)) and np.array_equal(v["tex"][3], (0.75, 1))
    assert np.array_equal(v["pos"][5], (0, 0, 1)) and np.array_equal(v["tex"][5], (0, 0))
    with pytest.raises(api.RtbError):
        api.load_obj(str(tmp_path / "missing.obj"))
    bad = tmp_path / "bad.obj"
    bad.write_text("v 0 0 0\nf 1 2 3\n")
    with pytest.raises(api.RtbError):
        api.load_obj(str(bad))


def test_obj_round_trip(api, tmp_path):
    verts = api.heightfield_mesh(6, 10.0)
    p = tmp_path / "hf.obj"
    api.write_obj(str(p), verts)
    back = api.load_obj(str(p))
    assert np.array_equal(back["pos"], verts["pos"])
    assert np.array_equal(back["tex"], verts["tex"])


# ---- PNG + CLI --------------------------------------------------------------------------------------

def _read_png(path):
    data = open(path, "rb").read()
    assert data[:8] == b"\x89PNG\r\n\x1a\n"
    pos, chunks = 8, []
    while pos < len(data):
        n, = struct.unpack(">I", data[pos:pos + 4])
        typ = data[pos + 4:pos + 8]
        body = data[pos + 8:pos + 8 + n]
        crc, = struct.unpack(">I", data[pos + 8 + n:pos + 12 + n])
        assert crc == (zlib.crc32(typ + body) & 0xFFFFFFFF)
        chunks.append((typ, body))
        pos += 12 + n
    w, h, depth, ctype = struct.unpack(">IIBB", chunks[0][1][:10])
    raw = zlib.decompress(b"".join(b for t, b in chunks if t == b"IDAT"))
    rows = np.frombuffer(raw, np.uint8).reshape(h, 1 + w * 3)
    assert (rows[:, 0] == 0).all()
    return rows[:, 1:].reshape(h, w, 3)


def test_png_writer(api, tmp_path):
    _, host = api.load()
    rng = np.random.default_rng(0)
    img = rng.integers(0, 256, size=(37, 211, 3), dtype=np.uint8)  # > 65535 bytes: several stored blocks
    big = rng.integers(0, 256, size=(200, 300, 3), dtype=np.uint8)
    white = np.full((1080, 1920, 3), 255, np.uint8)  # worst case for the deferred Adler-32 modulo; the bench frame size
    tiny = rng.integers(0, 256, size=(1, 1, 3), dtype=np.uint8)  # shorter than one 8-byte CRC step
    odd = rng.integers(0, 256, size=(5, 3, 3), dtype=np.uint8)
    for k, im in enumerate((img, big, white, tiny, odd)):
        p = tmp_path / f"o{k}.png"
        assert host.rt_write_png(str(p).encode(), im.shape[1], im.shape[0], 3, im.ctypes.data, im.shape[1] * 3) != 0
        assert np.array_equal(_read_png(str(p)), im)
    assert host.rt_write_png(b"/nonexistent-dir/x.png", 4, 4, 3, img.ctypes.data, 12) == 0


def test_cli_usage_and_errors():
    exe = os.path.join(ROOT, "raytracer.c_b200", "bin", "raytracer")
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode != 0 and "Usage:" in r.stderr and "-w <width>" in r.stderr  # main.c:189-193
    r = subprocess.run([exe, "-w", "64", "-h"], capture_output=True, text=True)
    assert r.returncode != 0
    r = subprocess.run([exe, "-w", "1", "-h", "64", "-s", "1", "-o", "x.png"], capture_output=True, text=True)
    assert r.returncode != 0


# ---- multi-GPU host logic (gloo, world_size 2) ---------------------------------------------------------
# The multi-GPU data path lives behind the C ABI (rtb_comm_*, csrc/rtb_multi.cu): sample ranges per rank,
# ncclReduce, tonemap on rank 0.  What can run without a GPU is its host logic: the shard arithmetic
# (rtb_comm_shard_samples) and the launcher-side plumbing bench.py uses -- rank 0's 128-byte id reaches
# every rank through torch.distributed, every rank derives its own sample range from the same job.

def test_shard_ranges(pkg):
    api = pkg.api
    assert api.shard_samples(0, 4096, 0, 8) == (0, 512) and api.shard_samples(0, 4096, 7, 8) == (3584, 4096)
    got = [api.shard_samples(0, 128, r, 3) for r in range(3)]
    assert got[0][0] == 0 and got[-1][1] == 128 and all(a[1] == b[0] for a, b in zip(got, got[1:]))
    assert sorted(e - b for b, e in got) == [42, 43, 43]
    for world in (1, 2, 3, 4, 8):
        for begin, end in ((0, 4096), (7, 7 + 128), (5, 5), (0, 3)):  # also fewer samples than ranks
            cover = []
            for r in range(world):
                b, e = api.shard_samples(begin, end, r, world)
                cover += list(range(b, e))
            assert cover == list(range(begin, end))
    with pytest.raises(api.RtbError):
        api.shard_samples(0, 4, 2, 2)
    with pytest.raises(api.RtbError):
        api.shard_samples(4, 0, 0, 2)


_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import numpy as np, torch, torch.distributed as dist
import __graft_entry__ as entry
pkg = entry.load_package()
api = pkg.api
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", rank=rank, world_size=world)
# 1. the id travels from rank 0 to everybody (bench.py does this with the real rtb_comm_unique_id)
idt = torch.zeros(api.UNIQUE_ID_BYTES, dtype=torch.uint8)
if rank == 0:
    idt.copy_(torch.frombuffer(bytearray(bytes(range(128))), dtype=torch.uint8))
dist.broadcast(idt, src=0)
assert bytes(idt.numpy().tobytes()) == bytes(range(128))
# 2. every rank derives its share of the SAME job through the C ABI
W, H, begin, end = 16, 8, 3, 3 + 9
b, e = api.shard_samples(begin, end, rank, world)
# stand-in for the per-GPU float sums: sample s contributes (s+1) to every pixel
accum = torch.full((H, W, 3), float(sum(s + 1 for s in range(b, e))), dtype=torch.float32)
dist.reduce(accum, dst=0, op=dist.ReduceOp.SUM)   # gloo standing in for the ncclReduce of rtb_comm_render
if rank == 0:
    want = float(sum(s + 1 for s in range(begin, end)))
    assert torch.all(accum == want), (accum[0, 0], want)
    print("OK", e - b, want)
dist.barrier()
dist.destroy_process_group()
"""


def test_two_rank_job_over_gloo(tmp_path):
    """the N>1 host logic: id broadcast, disjoint covering sample ranges per rank, one SUM reduce to rank 0"""
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT))
    port = 29500 + (os.getpid() % 2000)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", str(port), str(script)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "OK 4 72.0" in r.stdout


def test_render_params_carry_num_gpus(pkg):
    """RenderParams.num_gpus defaults to 1, or to $RTB_NUM_GPUS (how the unchanged main.c gets the whole box)"""
    import ctypes as C
    _, host = pkg.load()
    rp = pkg.abi.RenderParams()
    old = os.environ.pop("RTB_NUM_GPUS", None)
    try:
        host.render_params_default(C.byref(rp))
        assert rp.num_gpus == 1 and rp.total_samples == 0 and rp.max_depth == 5
        os.environ["RTB_NUM_GPUS"] = "8"
        host.render_params_default(C.byref(rp))
        assert rp.num_gpus == 8
    finally:
        os.environ.pop("RTB_NUM_GPUS", None)
        if old is not None:
            os.environ["RTB_NUM_GPUS"] = old


# ---- narrowed mesh upload: the host-side conversion (csrc/rtb_narrow.cpp) --------------------------------

def _narrow_fns(api):
    import ctypes as C
    cu, _ = api.load()
    fns = []
    for name in ("rtb_narrow_vertices", "rtb_narrow_vertices_scalar"):
        f = getattr(cu, name)
        f.restype = C.c_bool
        f.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        fns.append(f)
    return fns


def test_narrow_vertices_equals_numpy_and_flags_every_inexact_lane(api):
    """15 doubles -> 15 floats per triangle: round-to-nearest like numpy, vector form == scalar form, and the
    `exact` result is false exactly when some lane -- a position or a texture coordinate -- loses bits, overflows
    or is NaN"""
    fns = _narrow_fns(api)
    rng = np.random.default_rng(5)
    for n in (0, 1, 3, 4, 5, 12, 13, 1000, 4099):
        src = rng.uniform(-50, 50, (n, 5)).astype(np.float32).astype(np.float64)
        src[:, 3:] = rng.uniform(0, 1, (n, 2)).astype(np.float32)  # texture coordinates: floats, like an OBJ file's
        for f in fns:
            dst = np.full((n, 5), -1.0, np.float32)
            assert f(src.ctypes.data, dst.ctypes.data, n) is True
            assert np.array_equal(dst, src.astype(np.float32))
        if n == 0:
            continue
        for bad in (1.0 + 2.0 ** -40, 1e300, -1e300, float("nan"), 2.0 ** -160):
            for v in sorted({0, n // 2, n - 1}):
                for a in range(5):
                    s2 = src.copy()
                    s2[v, a] = bad
                    for f in fns:
                        dst = np.zeros((n, 5), np.float32)
                        exact = f(s2.ctypes.data, dst.ctypes.data, n)
                        assert exact is False, (n, v, a, bad)
                        with np.errstate(over="ignore"):
                            assert np.array_equal(dst, s2.astype(np.float32), equal_nan=True)


def test_narrow_vertices_flags_an_inexact_texcoord_in_every_lane(api):
    """only a texture coordinate is not float-representable (a caller's double texcoords): both forms report
    "inexact" wherever it sits -- every texcoord slot of a four-vertex group, i.e. each of the five 256-bit vectors
    of the AVX2 form and every lane position a texcoord takes there, and the scalar tail -- and still convert like
    numpy; positions alone that are floats stay exact"""
    fns = _narrow_fns(api)
    rng = np.random.default_rng(6)
    for n in (4, 8, 11):
        src = rng.uniform(-50, 50, (n, 5)).astype(np.float32).astype(np.float64)
        src[:, 3:] = rng.uniform(0, 1, (n, 2)).astype(np.float32)
        slots = set()
        for v in range(n):
            for a in (3, 4):
                k = 5 * (v % 4) + a  # double index inside the vertex's group of four
                if v < 4 * (n // 4):
                    slots.add((k // 4, k % 4))  # (vector, lane) of the AVX2 form
                for bad in (src[v, a] + 2.0 ** -40, -700.123456789, 1e300, float("nan")):
                    s2 = src.copy()
                    s2[v, a] = bad
                    for f in fns:
                        dst = np.zeros((n, 5), np.float32)
                        assert f(s2.ctypes.data, dst.ctypes.data, n) is False, (n, v, a, bad)
                        with np.errstate(over="ignore"):
                            assert np.array_equal(dst, s2.astype(np.float32), equal_nan=True)
        assert {vec for vec, _ in slots} == {0, 1, 2, 3, 4}
        assert len(slots) == 8  # texcoords are doubles 3, 4, 8, 9, 13, 14, 18, 19 of a group


def test_apply_matrix_is_the_same_for_any_thread_count(api, monkeypatch):
    """apply_matrix (main.c:140-147) runs over the host cores for large meshes: vertex by vertex the result is the
    scalar mat4_vector_mult of the reference, bit for bit"""
    verts = api.heightfield_mesh(120, 10.0)  # 28 800 triangles: above the parallel threshold
    assert len(verts) > 65536
    m = np.array([[0.7, 0.1, 0.0, 0.123456789], [0.0, 1.3, -0.2, 1.0 / 3.0], [0.3, 0.0, 0.9, -2.0 / 7.0], [0, 0, 0, 1.0]])
    want = verts["pos"].copy()
    # mat4_vector_mult (vector.h:63-74): row . (x, y, z, 1), left to right
    x, y, z = want[:, 0].copy(), want[:, 1].copy(), want[:, 2].copy()
    for r in range(3):
        want[:, r] = ((m[r, 0] * x + m[r, 1] * y) + m[r, 2] * z) + m[r, 3] * 1.0
    got = api.apply_matrix(verts.copy(), m)
    assert np.array_equal(got["pos"], want)
    assert np.array_equal(got["tex"], verts["tex"])


def test_render_warm_up_returns_at_once_and_never_fails(api):
    """render_warm_up() only starts a thread; without a GPU the thread's error is dropped (the render call reports it)"""
    _, host = api.load()
    host.render_warm_up(None)
    host.render_warm_up(None)  # joins the first, starts another; the library joins at exit


# ---- bench.py: the two arms of the measurement contract ----------------------------------------------------

def _run_bench(*args, timeout=300):
    import json as _json
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         timeout=timeout, cwd=ROOT)
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    return out, (_json.loads(lines[-1]) if lines else None)


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` times the reference's CPU implementation (C1: the unmodified program of
    oracle/_ref, else the oracle port) and prints ONE JSON line with the keys the driver reads"""
    out, line = _run_bench("--impl", "reference", "--workload", "c1", "--steps", "1", "--warmup", "0")
    assert out.returncode == 0, out.stderr[-2000:]
    assert line is not None, out.stdout[-2000:]
    assert line["impl"] == "reference" and line["metric"] == "Mrays/s" and line["unit"] == "Mrays/s"
    assert line["higher_is_better"] is True and line["n_gpus"] == 1 and line["steps"] == 1
    assert line["value"] > 0 and line["ms_per_step"] > 0
    assert line["e2e"] == {"value": line["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert "c1" in line["config"]["workload"]


def test_bench_gpu_arm_fails_loudly_without_a_gpu(api):
    """no CUDA device -> the product arm refuses to run (there is no CPU fallback to time by mistake)"""
    if api.device_count() > 0:
        pytest.skip("a GPU is present")
    out, line = _run_bench("--steps", "1", "--warmup", "1", timeout=120)
    assert out.returncode != 0 and line is None
    assert "CUDA device" in (out.stderr + out.stdout)
