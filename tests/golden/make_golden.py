"""Generates the golden vectors in this directory FROM THE UNMODIFIED REFERENCE
(oracle/_ref/libref.so, built from /root/reference by oracle/Makefile).  Run it in the
container that has /root/reference:

    make -C oracle && python tests/golden/make_golden.py

The vectors are small on purpose (they are committed).  Random inputs are regenerated from
the recorded numpy seeds, so only outputs are stored.
"""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import oracle_lib as ol  # noqa: E402
from conftest import random_rays_in_room  # noqa: E402

api = ol.pkg.api


def sphere_cases(seed=101, n=600):
    rng = np.random.default_rng(seed)
    rays, cs, rs = [], [], []
    for i in range(n):
        o = rng.uniform(-30, 30, 3)
        d = rng.normal(size=3)
        d /= np.linalg.norm(d)
        c = rng.uniform(-30, 30, 3)
        r = [rng.uniform(0.1, 12), 10000.0][i % 7 == 0]
        if i % 5 == 0:
            o = c + rng.uniform(-0.5, 0.5, 3) * r
        rays.append(np.concatenate([o, d]))
        cs.append(c)
        rs.append(r)
    return np.array(rays), np.array(cs), np.array(rs)


def triangle_cases(seed=102, n=600):
    rng = np.random.default_rng(seed)
    rays, verts = [], []
    for i in range(n):
        v = np.zeros((3, 5))
        v[:, :3] = rng.uniform(-5, 5, (3, 3))
        v[:, 3:] = rng.uniform(0, 1, (3, 2))
        target = v[:, :3].T @ rng.dirichlet((1, 1, 1)) if i % 2 == 0 else rng.uniform(-6, 6, 3)
        o = rng.uniform(-15, 15, 3)
        d = target - o
        d /= np.linalg.norm(d)
        rays.append(np.concatenate([o, d]))
        verts.append(v)
    return np.array(rays), np.array(verts)


def path_cases(seed=103, n=200):
    rng = np.random.default_rng(seed)
    cam = ol.ref_init_camera(320, 180)
    rays = np.array([ol.ref_camera_ray(cam, rng.uniform(0, 1), rng.uniform(0, 1)) for _ in range(n)])
    streams = rng.integers(0, 2 ** 31, size=(n, 2048), dtype=np.int64).astype(np.int32)
    return rays, streams


def whitted_golden():
    """cast_ray (raytracer.c:556-641) of the unmodified reference on fixed rays: the default scene
    (diffuse and mirror spheres; no checkered object) and a packed sphere field with mixed materials
    (tests/test_gpu_texture.py checks checkered spheres against the reference's cast_ray)"""
    out = {}
    rays = random_rays_in_room(np.random.default_rng(106), 3000)
    objs = api.scene_default(320, 180)
    out["c1_rgb"], out["c1_calls"] = ol.ref_cast_rays(objs, rays, max_depth=5)
    field = api.scene_sphere_field(400, 96, 54, mix=(0.3, 0.3, 0.3))
    out["field_rgb"], out["field_calls"] = ol.ref_cast_rays(field, rays, max_depth=8)
    np.savez_compressed(os.path.join(HERE, "whitted.npz"), **out)


def main():
    if len(sys.argv) > 1 and sys.argv[1] == "whitted":
        whitted_golden()
        return
    whitted_golden()
    ref = ol.ref()
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731

    # leaf primitives (raytracer.c:77-174)
    rays, cs, rs = sphere_cases()
    hit, t = np.zeros(len(rays), np.int8), np.zeros(len(rays))
    for i in range(len(rays)):
        tt = C.c_double()
        hit[i] = ref.ref_intersect_sphere(p(rays[i]), p(cs[i]), float(rs[i]), C.byref(tt))
        t[i] = tt.value if hit[i] else 0.0
    rays_t, verts = triangle_cases()
    hit_t, tuv = np.zeros(len(rays_t), np.int8), np.zeros((len(rays_t), 3))
    for i in range(len(rays_t)):
        out = np.zeros(3)
        hit_t[i] = ref.ref_intersect_triangle(p(rays_t[i]), p(verts[i]), p(out))
        tuv[i] = out if hit_t[i] else 0.0
    np.savez_compressed(os.path.join(HERE, "prims.npz"), sphere_hit=hit, sphere_t=t, tri_hit=hit_t, tri_tuv=tuv)

    # camera (raytracer.c:47-75, 375-384)
    cams = {f"{w}x{h}": ol.ref_init_camera(w, h).as_array() for w, h in ((320, 180), (1920, 1080), (512, 512))}
    cam = ol.ref_init_camera(320, 180)
    uv = np.random.default_rng(104).uniform(0, 1, (64, 2))
    cam_rays = np.array([ol.ref_camera_ray(cam, u, v) for u, v in uv])
    np.savez_compressed(os.path.join(HERE, "camera.npz"), cam_rays=cam_rays, **cams)

    # nearest hit on the default scene (raytracer.c:393-464)
    objs = api.scene_default(320, 180)
    rays = random_rays_in_room(np.random.default_rng(105), 3000)
    h = ol.ref_intersect_rays(objs, rays)
    np.savez_compressed(os.path.join(HERE, "c1_hits.npz"), ids=h["ids"], points=h["points"], normals=h["normals"], uvs=h["uvs"])

    # single paths, random draws replayed from a stream (raytracer.c:482-554)
    prays, streams = path_cases()
    rad, used = np.zeros((len(prays), 3)), np.zeros(len(prays), np.int64)
    for i in range(len(prays)):
        rad[i], used[i] = ol.ref_trace_path_stream(objs, prays[i], streams[i], max_depth=5)
    np.savez_compressed(os.path.join(HERE, "c1_paths.npz"), radiance=rad, used=used)

    # whole frames under srand(seed) (raytracer.c:176-223)
    frames = {}
    for (W, H, S, depth) in ((64, 36, 6, 5), (48, 27, 4, 8)):
        o = api.scene_default(W, H)
        c = ol.ref_init_camera(W, H)
        fb, ctr = ol.ref_render(o, c, W, H, S, max_depth=depth)
        mean, _ = ol.ref_render_mean(o, c, W, H, S, max_depth=depth)
        frames[f"fb_{W}x{H}_s{S}_d{depth}"] = fb
        frames[f"mean_{W}x{H}_s{S}_d{depth}"] = mean
        frames[f"ctr_{W}x{H}_s{S}_d{depth}"] = np.array(ctr, dtype=np.int64)
    np.savez_compressed(os.path.join(HERE, "c1_frames.npz"), **frames)

    # the converged reference renders for the PSNR gate are made by make_converged.py (one process per seed)
    for f in sorted(os.listdir(HERE)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(HERE, f)))


if __name__ == "__main__":
    main()
