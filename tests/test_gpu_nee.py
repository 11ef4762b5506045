"""Next-event estimation on the GPU (RTB_INTEGRATOR_PATH_NEE: k_wf_shade_nee, the shadow-ray trace, k_wf_shadow_resolve)
against the oracle's NEE estimator (tests/test_oracle_nee.py holds that one to the reference's converged frames).

Every light sample is a decision in correctly rounded double arithmetic on both sides, so the ray, shadow-ray and
shadow-hit counts must be the oracle's exactly; the sums differ only by the GPU's float accumulation.
"""
import os

import numpy as np
import pytest

import oracle_nee_lib as onl
import test_gpu_wavefront_paths as wp
from test_oracle_nee import GOLDEN, block_test

pytestmark = pytest.mark.gpu
NEE = 2


def _scene(api, abi, name, W, H):
    return wp.SCENES[name](api, abi, W, H)


def _render(api, src, cam, desc):
    with api.Scene(src, device=0) as sc:
        _, acc, ctr = sc.render(cam, desc, want_accum=True)
    return acc.astype(np.float64), ctr


def _close(acc, want):
    """the float sums of the same samples: 1e-3 relative, as smoke() holds trace_path"""
    return np.max(np.abs(acc - want) / (np.abs(want) + 1e-3))


CASES = [("c1", 96, 54, 8, "stochastic"), ("c1", 96, 54, 8, "split"), ("field300", 64, 36, 8, "stochastic"),
         ("checkered-field", 64, 36, 8, "stochastic"), ("mesh-tri64", 40, 23, 4, "stochastic")]


@pytest.mark.parametrize("name,W,H,spp,dielectric", CASES)
def test_against_oracle(gpu_api, abi, ol, name, W, H, spp, dielectric):
    src = _scene(gpu_api, abi, name, W, H)
    cam = gpu_api.init_camera(W, H)
    d = 1 if dielectric == "split" else 0
    acc, ctr = _render(gpu_api, src, cam, gpu_api.make_desc(W, H, 0, spp, integrator=NEE, dielectric=d))
    want, (rays, _, shadow, hits) = onl.render_sum(src, ol.init_camera(W, H), W, H, spp, dielectric=dielectric)
    assert (ctr.rays, ctr.shadow_rays, ctr.shadow_hits) == (rays, shadow, hits)
    assert shadow > 0
    assert _close(acc, want) < 1e-3


@pytest.mark.parametrize("dielectric", [0, 1])
def test_no_emissive_sphere_is_path(gpu_api, dielectric):
    W, H = 64, 36
    objs = gpu_api.scene_default(W, H)
    objs["emission"][:] = 0.0
    cam = gpu_api.init_camera(W, H)
    a, c = _render(gpu_api, objs, cam, gpu_api.make_desc(W, H, 0, 8, planes=3, dielectric=dielectric))
    b, n = _render(gpu_api, objs, cam, gpu_api.make_desc(W, H, 0, 8, planes=3, dielectric=dielectric, integrator=NEE))
    assert np.array_equal(a, b)
    assert (n.shadow_rays, n.shadow_hits, c.shadow_rays) == (0, 0, 0)


def test_path_rays_are_paths(gpu_api):
    W, H = 96, 54
    objs = gpu_api.scene_default(W, H)
    cam = gpu_api.init_camera(W, H)
    _, c = _render(gpu_api, objs, cam, gpu_api.make_desc(W, H, 0, 16))
    _, n = _render(gpu_api, objs, cam, gpu_api.make_desc(W, H, 0, 16, integrator=NEE))
    assert (n.rays, n.rays_intersected, n.paths) == (c.rays, c.rays_intersected, c.paths)
    assert n.shadow_rays > n.shadow_hits > 0


def test_reproducible_and_sharded(gpu_api):
    W, H, S, K = 96, 54, 12, 5
    objs = gpu_api.scene_default(W, H)
    cam = gpu_api.init_camera(W, H)
    a, _ = _render(gpu_api, objs, cam, gpu_api.make_desc(W, H, 0, S, planes=4, integrator=NEE))
    b, _ = _render(gpu_api, objs, cam, gpu_api.make_desc(W, H, 0, S, planes=4, integrator=NEE))
    assert np.array_equal(a, b)
    lo, _ = _render(gpu_api, objs, cam, gpu_api.make_desc(W, H, 0, K, integrator=NEE))
    hi, _ = _render(gpu_api, objs, cam, gpu_api.make_desc(W, H, K, S, integrator=NEE))
    assert np.max(np.abs(lo + hi - a) / (np.abs(a) + 1e-3)) < 1e-4


def test_unbiased_c1_320(gpu_api):
    """the device's NEE converges to the reference's own converged frame (the oracle test's block test)"""
    W, H, SPP, B = 320, 180, 64, 32
    objs = gpu_api.scene_default(W, H)
    cam = gpu_api.init_camera(W, H)
    with gpu_api.Scene(objs, device=0) as sc:
        def batch(k):
            _, acc, _ = sc.render(cam, gpu_api.make_desc(W, H, k * SPP, (k + 1) * SPP, integrator=NEE), want_accum=True)
            return acc.astype(np.float64) / SPP

        rel, z = block_test(batch, os.path.join(GOLDEN, "c1_converged_320x180.npz"), B)
    assert rel < 0.005, rel
    assert z.max() < 5.0, z.max()


@pytest.mark.parametrize("workload", ["c1", "c2", "c3", "c4", "c5"])
def test_bench_workloads(gpu_api, workload):
    """every benchmark scene renders with NEE at a small sample count (C5 at its depth 64: mostly dielectric, so few
    diffuse vertices), path rays equal to trace_path's"""
    import bench
    W, H, _, depth, _ = bench.WORKLOADS[workload]
    W, H = W // 4, H // 4
    src = bench.build_host_scene(gpu_api, workload, W, H)[0]
    cam = gpu_api.init_camera(W, H)
    with gpu_api.Scene(src, device=0) as sc:
        _, _, c = sc.render(cam, gpu_api.make_desc(W, H, 0, 2, max_depth=depth, seed=bench.SEED))
        _, acc_n, n = sc.render(cam, gpu_api.make_desc(W, H, 0, 2, max_depth=depth, seed=bench.SEED, integrator=NEE),
                                want_accum=True)
    assert n.rays == c.rays and n.paths == c.paths
    assert np.isfinite(acc_n).all() and acc_n.min() >= 0.0
    assert n.shadow_rays > 0


def test_denoised_nee(gpu_api):
    """rtb_render_denoised of an NEE render: the raw sums are the NEE render's; rtb_render_aov itself still takes the
    PATH / Whitted integrators only"""
    W, H = 64, 36
    objs = gpu_api.scene_default(W, H)
    cam = gpu_api.init_camera(W, H)
    with gpu_api.Scene(objs, device=0) as sc:
        with pytest.raises(gpu_api.RtbError):
            sc.render_aov(cam, gpu_api.make_desc(W, H, 0, 4, integrator=NEE))
        _, out, acc, ctr = sc.render_denoised(cam, gpu_api.make_desc(W, H, 0, 4, integrator=NEE), want_accum=True)
        _, plain, _ = sc.render(cam, gpu_api.make_desc(W, H, 0, 4, integrator=NEE), want_accum=True)
    assert np.array_equal(acc, plain)
    assert ctr.shadow_rays > 0 and np.isfinite(out).all()


def test_denoised_aov_is_path_features(gpu_api, abi):
    """render_denoised_aov of an NEE render hands back rtb_render_aov's feature sums for RTB_INTEGRATOR_PATH, bit for
    bit"""
    import ctypes as C
    W, H = 64, 36
    objs = gpu_api.scene_default(W, H)
    objs["flags"][::3] |= abi.M_CHECKERED
    cam = gpu_api.init_camera(W, H)
    with gpu_api.Scene(objs, device=0) as sc:
        want = sc.render_aov(cam, gpu_api.make_desc(W, H, 0, 4))
        got = dict(albedo=np.zeros((H, W, 3), np.float32), normal=np.zeros((H, W, 3), np.float32),
                   depth=np.zeros((H, W), np.float32), hits=np.zeros((H, W), np.uint32), object=np.zeros((H, W), np.int32))
        fb = np.zeros((H, W, 3), np.uint8)
        desc = gpu_api.make_desc(W, H, 0, 4, integrator=NEE)
        cu, _ = gpu_api.load()
        cam12 = cam.as_array()
        ptr = lambda a: C.c_void_p(a.ctypes.data)  # noqa: E731
        rc = cu.rtb_render_denoised_aov(sc._h, cam12.ctypes.data_as(C.POINTER(C.c_double)),
                                        C.byref(desc), C.c_int(4), None, ptr(fb), None, None,
                                        *(ptr(got[k]) for k in ("albedo", "normal", "depth", "hits", "object")), None)
        assert rc == 0, cu.rtb_last_error().decode()
    for k, v in got.items():
        assert np.array_equal(want[k], v), k


@pytest.mark.parametrize("kernel", [1, 2, 3, 4, 5])
def test_megakernels_reject_nee(gpu_api, kernel):
    W, H = 32, 18
    with gpu_api.Scene(gpu_api.scene_default(W, H), device=0, all_trees=True) as sc:
        with pytest.raises(gpu_api.RtbError):
            sc.render(gpu_api.init_camera(W, H), gpu_api.make_desc(W, H, 0, 1, kernel=kernel, integrator=NEE))


def test_multi_gpu_is_sum_of_shards(gpu_api):
    n_gpus = gpu_api.device_count()
    if n_gpus < 2:
        pytest.skip("needs 2 GPUs")
    W, H, S = 96, 54, 12
    objs = gpu_api.scene_default(W, H)
    cam = gpu_api.init_camera(W, H)
    desc = gpu_api.make_desc(W, H, 0, S, integrator=NEE)
    with gpu_api.Comm.local(2) as comm:
        _, acc, ctr = comm.render_host(objs, cam, desc, want_accum=True)
    parts, shadow = [], 0
    for r in range(2):
        b, e = gpu_api.shard_samples(0, S, r, 2)
        a, c = _render(gpu_api, objs, cam, gpu_api.make_desc(W, H, b, e, integrator=NEE))
        parts.append(a)
        shadow += c.shadow_rays
    total = parts[0] + parts[1]
    assert np.max(np.abs(acc - total) / (np.abs(total) + 1e-3)) < 1e-4
    assert ctr.shadow_rays == shadow
