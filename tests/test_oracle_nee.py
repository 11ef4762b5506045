"""Next-event estimation (RTB_INTEGRATOR_PATH_NEE, DESIGN.md section 4.7) in the oracle: the estimator the GPU is held to.

  no light      without an emissive sphere NEE is trace_path itself: the same sums bit for bit, no shadow ray
  same paths    the path rays are trace_path's, one for one (the light samples draw from their own Philox block)
  unbiased      NEE converges to the REFERENCE's converged frames (tests/golden/*_converged_*.npz, rendered by the
                unmodified reference under libc rand): frame mean within 0.5 %, every 8x6 block within 5 standard errors
  less noise    at 4 / 16 / 64 spp NEE beats trace_path's PSNR against the converged frame by the committed margins
Philox is keyed, so every number here is fixed: the tests cannot be flaky.
"""
import os

import numpy as np
import pytest

import oracle_lib as ol
import oracle_nee_lib as onl
from denoise_ref import psnr_vs

api = ol.pkg.api
abi = ol.abi
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# PSNR (dB, 8-bit frames) against c1_converged_320x180.npz, oracle Philox renders of C1 at 320x180, seed
# abi.SCENE_SEED, max depth 5, stochastic dielectric (measured with this file's render):
#   spp   PATH    NEE     gain
#     4    9.09   11.78   2.69
#    16   14.25   20.26   6.01
#    64   21.85   27.37   5.53
# The floors sit just below the measured gains.
GAIN_FLOOR_DB = {4: 2.5, 16: 5.8, 64: 5.3}


def _no_sphere_light(objs):
    objs = objs.copy()
    objs["emission"][:] = 0.0
    return objs


def _mesh_light_room(W, H):
    """the C3 room with its light spheres dark and the mesh emissive: a light NEE cannot sample"""
    h = api.mesh_room(api.heightfield_mesh(8, 20 * W / H * 0.98), W, H)
    for k in range(h.n):
        m = h.objects[k].material
        if h.objects[k].type == 0:
            m.emission.x = m.emission.y = m.emission.z = 0.0
        else:
            m.emission.x, m.emission.y, m.emission.z = 0.6, 0.5, 0.4
    return h


@pytest.mark.parametrize("scene", ["walls", "mesh-light"])
@pytest.mark.parametrize("dielectric", ["stochastic", "split"])
def test_no_emissive_sphere_is_path(scene, dielectric):
    W, H, SPP = 48, 27, 8
    src = _no_sphere_light(api.scene_default(W, H)) if scene == "walls" else _mesh_light_room(W, H)
    cam = ol.init_camera(W, H)
    path, (rays, tests) = ol.render_sum(src, cam, W, H, SPP, dielectric=dielectric)
    nee, (rays_n, tests_n, shadow, shadow_hits) = onl.render_sum(src, cam, W, H, SPP, dielectric=dielectric)
    assert shadow == 0 and shadow_hits == 0
    assert (rays_n, tests_n) == (rays, tests)
    assert np.array_equal(nee, path)
    if scene == "mesh-light":
        assert path.max() > 0.1  # the mesh does light the room


@pytest.mark.parametrize("dielectric", ["stochastic", "split"])
def test_same_path_rays(dielectric):
    W, H, SPP = 96, 54, 8
    objs = api.scene_default(W, H)
    cam = ol.init_camera(W, H)
    _, (rays, _) = ol.render_sum(objs, cam, W, H, SPP, dielectric=dielectric)
    _, (rays_n, _, shadow, shadow_hits) = onl.render_sum(objs, cam, W, H, SPP, dielectric=dielectric)
    assert rays_n == rays
    assert 0 < shadow_hits < shadow < rays


def block_test(render_batch, golden, batches, bw=8, bh=6):
    """`batches` independent NEE renders (mean radiance each) against the converged golden frame: the standard error of
    a block is the spread of its batch means plus the golden frame's own noise (from its disjoint quarter render).
    Enough batches (32) that the spread is a good estimate: with few, its Student-t tails over thousands of blocks
    would put some block beyond 5 standard errors by chance."""
    g = np.load(golden)
    full, quarter = g["mean"].astype(np.float64), g["mean_quarter"].astype(np.float64)
    n_full, n_quarter = (int(v) for v in g["spp"])
    H, W, _ = full.shape

    def blocks(img):
        return img[:H // bh * bh, :W // bw * bw].reshape(H // bh, bh, W // bw, bw, 3).mean(axis=(1, 3))

    means = np.array([render_batch(k) for k in range(batches)])
    est = means.mean(axis=0)
    b = np.array([blocks(m) for m in means])
    se_est = b.std(axis=0, ddof=1) / np.sqrt(batches)
    # full - quarter has variance s2 (1/n_full + 1/n_quarter); the full frame's share is s2 / n_full
    d = blocks(full) - blocks(quarter)
    se_gold = np.sqrt(np.mean(d ** 2, axis=(0, 1)) * (1.0 / n_full) / (1.0 / n_full + 1.0 / n_quarter))
    z = np.abs(blocks(est) - blocks(full)) / np.sqrt(se_est ** 2 + se_gold ** 2 + 1e-30)
    rel = abs(est.mean() - full.mean()) / full.mean()
    return rel, z


def test_unbiased_c1():
    W, H, SPP, B = 96, 54, 32, 32
    objs = api.scene_default(W, H)
    cam = ol.init_camera(W, H)

    def batch(k):
        s, _ = onl.render_sum(objs, cam, W, H, SPP, sample_offset=k * SPP)
        return s / SPP

    rel, z = block_test(batch, os.path.join(GOLDEN, "c1_converged_96x54.npz"), B)
    assert rel < 0.005, rel
    assert z.max() < 5.0, (z.max(), np.unravel_index(z.argmax(), z.shape))


@pytest.mark.parametrize("dielectric", ["stochastic", "split"])
def test_unbiased_dielectric(dielectric):
    """the dielectric golden scene (tests/golden/make_converged.py): a sphere field with glass, mirrors and lights"""
    W, H, SPP, B = 64, 36, 32, 32
    objs = api.scene_sphere_field(60, W, H, mix=(0.3, 0.4, 0.2))
    cam = ol.init_camera(W, H)

    def batch(k):
        s, _ = onl.render_sum(objs, cam, W, H, SPP, dielectric=dielectric, sample_offset=k * SPP)
        return s / SPP

    rel, z = block_test(batch, os.path.join(GOLDEN, "dielectric_converged_64x36.npz"), B)
    assert rel < 0.005, rel
    assert z.max() < 5.0, (z.max(), np.unravel_index(z.argmax(), z.shape))


@pytest.mark.parametrize("spp", [4, 16, 64])
def test_less_noise_c1(spp):
    W, H = 320, 180
    objs = api.scene_default(W, H)
    cam = ol.init_camera(W, H)
    golden = np.load(os.path.join(GOLDEN, "c1_converged_320x180.npz"))["mean"].astype(np.float64)
    path, _ = ol.render_sum(objs, cam, W, H, spp)
    nee, _ = onl.render_sum(objs, cam, W, H, spp)
    gain = psnr_vs(nee / spp, golden, ol) - psnr_vs(path / spp, golden, ol)
    assert gain > GAIN_FLOOR_DB[spp], gain
