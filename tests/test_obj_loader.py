"""load_obj (host/obj_loader.c, raytracer.h:158) against the reference's own vendored OBJ parser.

The reference declares load_obj and vendors tinyobjloader-c (lib/tinyobj_loader.h:118-144, compiled into
raytracer.c:4-5) but never defines the function.  oracle/ref_harness.c holds the loader a maintainer would
write on that parser (tinyobj_parse_obj + TINYOBJ_FLAG_TRIANGULATE, SURVEY.md 8f N1); it lives in
oracle/_ref/libref.so together with the unmodified reference.  The product's loader does not use tinyobj;
these tests check that both give the same Vertex array, bit for bit.
"""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib as ol

needs_tinyobj = pytest.mark.skipif(not ol.have_ref(), reason="oracle/_ref/libref.so not built")

REF_CUBE = "/root/reference/assets/cube.obj"  # only where the reference tree exists (this container)


def tinyobj_load(path):
    lib = ol.ref()
    lib.ref_tinyobj_load.restype = C.c_longlong
    lib.ref_tinyobj_load.argtypes = [C.c_char_p, C.c_void_p, C.c_longlong]
    n = lib.ref_tinyobj_load(os.fsencode(path), None, 0)
    assert n >= 0, f"tinyobj_parse_obj failed on {path}"
    out = np.zeros((3 * n, 5), np.float64)
    got = lib.ref_tinyobj_load(os.fsencode(path), out.ctypes.data, n)
    assert got == n
    return out


def ours(api, path):
    v = api.load_obj(path)
    return np.concatenate([v["pos"].reshape(-1, 3), v["tex"].reshape(-1, 2)], axis=1)


@pytest.fixture(scope="module")
def api():
    import __graft_entry__ as entry
    return entry.load_package().api


@needs_tinyobj
@pytest.mark.skipif(not os.path.exists(REF_CUBE), reason="reference tree absent")
def test_reference_cube_asset(api):
    """assets/cube.obj:1-31: 8 vertices, 6 quads with v//vn corners -> 12 triangles, no texcoords"""
    want = tinyobj_load(REF_CUBE)
    got = ours(api, REF_CUBE)
    assert want.shape == (36, 5)
    assert np.array_equal(got, want)


@needs_tinyobj
def test_heightfield_obj_round_trip(api, tmp_path):
    """the C3 generator written out as OBJ (scene_write_obj) and read back by both parsers"""
    verts = api.heightfield_mesh(24, 10.0)
    p = str(tmp_path / "hf.obj")
    api.write_obj(p, verts)
    want = tinyobj_load(p)
    got = ours(api, p)
    assert len(want) == len(verts) == 3 * 2 * 24 * 24
    assert np.array_equal(got, want)
    # and the file reproduces the generator's (float-representable) positions exactly
    assert np.array_equal(got[:, :3], verts["pos"].reshape(-1, 3))


TRICKY = """# corners in every syntax, polygons, relative indices, numbers in every notation
v 0 0 0
v 1.5 0 0
v 1.5 2.25e0 0
v 0 2.25 -.5
v -3.125E-1 +4 1
vt 0 0
vt 1 0
vt 1 1
vt 0.25 0.75
vn 0 0 1
f 1 2 3
f 1/1 2/2 3/3
f 1//1 2//1 3//1 4//1
f 1/1/1 2/2/1 3/3/1 4/4/1 5/1/1
f -5 -4 -3
f -1/-1 -2/-2 -3/-3 -4/-4
v 9 9 9
f 6 1 2
"""


@needs_tinyobj
def test_tricky_syntax(api, tmp_path):
    p = str(tmp_path / "tricky.obj")
    with open(p, "w") as f:
        f.write(TRICKY)
    want = tinyobj_load(p)
    got = ours(api, p)
    assert len(want) == 3 * (1 + 1 + 2 + 3 + 1 + 2 + 1)
    assert np.array_equal(got, want)


@needs_tinyobj
def test_decimal_parsing_matches_tinyobj(api, tmp_path):
    """tinyobj parses reals with its own routine (tinyobj_loader.h:272-468) and narrows to float
    (:470-481); ours uses strtod and narrows.  2000 random decimal strings must give the same floats."""
    rng = np.random.default_rng(7)
    vals = np.concatenate([rng.uniform(-100, 100, 3000), rng.uniform(-1e-3, 1e-3, 1500), rng.uniform(-1e6, 1e6, 1500)])
    lines = []
    for k in range(0, len(vals), 3):
        a, b, c = vals[k:k + 3]
        lines.append(f"v {a:.6f} {b:.9g} {c:.7e}")
    n = len(lines)
    lines += [f"f {k + 1} {k + 2} {k + 3}" for k in range(0, n - 2, 3)]
    p = str(tmp_path / "dec.obj")
    with open(p, "w") as f:
        f.write("\n".join(lines) + "\n")
    want = tinyobj_load(p)
    got = ours(api, p)
    assert np.array_equal(got, want)


def test_slash_at_end_of_corner_does_not_eat_the_next_one(api, tmp_path):
    """ADVICE r1: `f 1// 2// 3//` used to lose corners because strtol() skips blanks and newlines"""
    p = str(tmp_path / "slash.obj")
    with open(p, "w") as f:
        f.write("v 0 0 0\nv 1 0 0\nv 0 1 0\nv 0 0 1\nf 1// 2// 3//\nf 1/ 2/ 4/\nf 2 3 4")  # no trailing newline
    got = ours(api, p)
    assert got.shape == (9, 5)
    assert np.array_equal(got[:, :3], np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 0], [1, 0, 0], [0, 0, 1],
                                                [1, 0, 0], [0, 1, 0], [0, 0, 1]], float))


def _rows(v):
    return np.concatenate([v["pos"].reshape(-1, 3), v["tex"].reshape(-1, 2)], axis=1)


@pytest.mark.parametrize("threads,chunk", [(1, 1 << 30), (1, 64), (3, 64), (8, 200), (4, 4096), (16, 1)])
def test_chunked_parallel_parse_is_the_serial_parse(api, tmp_path, threads, chunk):
    """load_obj_ex cuts the file into line-aligned chunks parsed by several threads; whatever the chunking --
    a chunk per line, chunks that hold only `v` lines or only faces, relative indices that reach back across
    chunks, CRLF line ends, no trailing newline -- the triangles are the one-chunk result, and the tinyobj
    path's"""
    rng = np.random.default_rng(11)
    lines = ["# interleaved vertices, texcoords and faces"]
    n_v = n_t = 0
    for k in range(400):
        for _ in range(rng.integers(1, 6)):
            x, y, z = rng.uniform(-50, 50, 3)
            lines.append(f"v {x:.7f} {y:.5g} {z:.3e}")
            n_v += 1
        for _ in range(rng.integers(0, 3)):
            lines.append(f"vt {rng.uniform():.6f} {rng.uniform():.6f}")
            n_t += 1
        if n_v >= 5:
            n = int(rng.integers(3, 6))
            if rng.uniform() < 0.5:  # absolute indices anywhere before this line
                c = [f"{rng.integers(1, n_v + 1)}" + (f"/{rng.integers(1, n_t + 1)}" if n_t else "") for _ in range(n)]
            else:                    # relative ones, some far back
                c = [f"-{rng.integers(1, n_v + 1)}" + (f"/-{rng.integers(1, n_t + 1)}" if n_t else "//") for _ in range(n)]
            lines.append("f " + " ".join(c))
    text = "\r\n".join(lines[:300]) + "\r\n" + "\n".join(lines[300:])  # first part CRLF, no newline at the end
    p = str(tmp_path / "mixed.obj")
    with open(p, "w", newline="") as f:
        f.write(text)
    serial = _rows(api.load_obj(p, threads=1, min_chunk_bytes=1 << 30))
    got = _rows(api.load_obj(p, threads=threads, min_chunk_bytes=chunk))
    assert len(serial) > 1500 and np.array_equal(got, serial)
    assert np.array_equal(_rows(api.load_obj(p)), serial)
    if ol.have_ref():
        assert np.array_equal(serial, tinyobj_load(p))


def test_chunked_parse_of_a_segregated_file(api, tmp_path):
    """the usual layout -- every `v`, then every `vt`, then every `f` (scene_write_obj) -- in 1 KB chunks"""
    verts = api.heightfield_mesh(16, 10.0)
    p = str(tmp_path / "hf.obj")
    api.write_obj(p, verts)
    got = api.load_obj(p, threads=5, min_chunk_bytes=1024)
    assert np.array_equal(got["pos"], verts["pos"]) and np.array_equal(got["tex"], verts["tex"])


@pytest.mark.parametrize("chunk", [1 << 30, 16])
def test_parse_failures_do_not_depend_on_the_chunking(api, tmp_path, chunk):
    """a face may only use vertices defined before it; a `v` line needs three numbers: the load fails as a whole"""
    for name, text in (("forward.obj", "v 0 0 0\nv 1 0 0\nf 1 2 3\nv 0 1 0\n"),
                       ("range.obj", "v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 -4\n"),
                       ("short.obj", "v 0 0 0\nv 1 0\nv 0 1 0\nf 1 2 3\n")):
        p = str(tmp_path / name)
        with open(p, "w") as f:
            f.write(text)
        with pytest.raises(api.RtbError):
            api.load_obj(p, threads=4, min_chunk_bytes=chunk)
    empty = str(tmp_path / "empty.obj")
    open(empty, "w").close()
    assert len(api.load_obj(empty, threads=4, min_chunk_bytes=chunk)) == 0
