"""The denoiser's restatement (tests/denoise_ref.py) on the CPU: the calibration that fixes rtb_denoise's defaults,
and the properties the GPU kernel must share with it.

Calibration: the oracle's Philox renders (the GPU's own sample streams) with the oracle's feature sums, denoised with
the defaults, scored by PSNR on 8-bit frames against converged references.  The floors are the gains measured when
the defaults were chosen, minus a margin (DESIGN.md section 4.6); tests/test_gpu_denoise.py holds the GPU's frames
to the same C1 floors.
"""
import os

import numpy as np
import pytest

import denoise_ref as dr

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ROOM_W, ROOM_H, ROOM_REF_SPP = 64, 36, 2048
# checkered mesh room (below): PSNR floors of the denoised frame against the oracle's 2048-spp render
ROOM_PSNR_FLOOR = {4: 14.0, 16: 16.5, 64: 20.0}


def _c1_raw_and_denoised(ol, api, spp):
    W, H = dr.C1_W, dr.C1_H
    objs = api.scene_default(W, H)
    cam = api.init_camera(W, H)
    s, _ = ol.render_sum(objs, cam, W, H, spp, rng="philox", dielectric="stochastic")
    f = dr.oracle_feature_sums(ol, objs, cam, W, H, spp)
    acc = s.astype(np.float32)
    return acc / np.float32(spp), dr.denoise(acc, f["albedo"], f["normal"], f["depth"], f["hits"], f["object"], spp)


@pytest.mark.parametrize("spp", dr.C1_SPP)
def test_calibration_c1_against_the_converged_golden(ol, api, spp):
    ref = np.load(os.path.join(GOLD, "c1_converged_320x180.npz"))["mean"]
    raw, den = _c1_raw_and_denoised(ol, api, spp)
    p_raw, p_den = dr.psnr_vs(raw, ref, ol), dr.psnr_vs(den, ref, ol)
    print(f"C1 {spp} spp: raw {p_raw:.2f} dB, denoised {p_den:.2f} dB")
    assert p_den >= dr.C1_PSNR_FLOOR[spp], (spp, p_raw, p_den)
    assert p_den >= p_raw + dr.C1_GAIN_FLOOR[spp], (spp, p_raw, p_den)
    assert abs(den.mean() / raw.mean() - 1.0) < dr.C1_MEAN_BOUND, (den.mean(), raw.mean())


def test_calibration_checkered_mesh_room(ol, api, abi):
    """a mesh room whose mesh, balls and two walls carry the checker (texture the demodulation must keep sharp),
    against the oracle's own render at 2048 spp with other Philox keys"""
    from test_gpu_texture import checkered_room
    W, H = ROOM_W, ROOM_H
    src, _ = checkered_room(api, abi, 12, "float", W, H, seed=3)
    cam = api.init_camera(W, H)
    ref, _ = ol.render_sum(src, cam, W, H, ROOM_REF_SPP, rng="philox", dielectric="stochastic", seed=12345)
    ref = ref / ROOM_REF_SPP
    for spp in (4, 16, 64):
        s, _ = ol.render_sum(src, cam, W, H, spp, rng="philox", dielectric="stochastic")
        f = dr.oracle_feature_sums(ol, src, cam, W, H, spp)
        acc = s.astype(np.float32)
        den = dr.denoise(acc, f["albedo"], f["normal"], f["depth"], f["hits"], f["object"], spp)
        p_raw, p_den = dr.psnr_vs(acc / np.float32(spp), ref, ol), dr.psnr_vs(den, ref, ol)
        print(f"checkered room {spp} spp: raw {p_raw:.2f} dB, denoised {p_den:.2f} dB")
        assert p_den >= ROOM_PSNR_FLOOR[spp], (spp, p_raw, p_den)


def test_vectorised_camera_rays_are_the_oracles(ol, api):
    W, H = 40, 23
    cam = api.init_camera(W, H)
    for s in (0, 5):
        rays = dr.camera_rays(cam, ol.abi.SCENE_SEED, W, H, s)
        for pix in (0, 17, 411, W * H - 1):
            j = ol.keyed_jitter(ol.abi.SCENE_SEED, pix, s)
            want = ol.camera_ray(cam, (pix % W + j[0]) / (W - 1.0), (pix // W + j[1]) / (H - 1.0))
            assert np.array_equal(rays[pix], want), (s, pix)


# ---- properties ---------------------------------------------------------------------------------------------------

def _random_inputs(rng, H=24, W=37, spp=4, n_obj=3):
    obj = rng.integers(-1, n_obj, (H, W)).astype(np.int32)
    obj[:, : W // 2] = np.where(obj[:, : W // 2] == -1, 0, obj[:, : W // 2])
    hits = np.where(obj >= 0, rng.integers(1, spp + 1, (H, W)), 0).astype(np.uint32)
    accum = rng.exponential(1.0, (H, W, 3)).astype(np.float32) * spp
    albedo = (rng.uniform(0.0, 1.0, (H, W, 3)) * hits[..., None]).astype(np.float32)
    n = rng.normal(size=(H, W, 3))
    n /= np.linalg.norm(n, axis=-1, keepdims=True)
    normal = (n * hits[..., None]).astype(np.float32)
    depth = (rng.uniform(5.0, 60.0, (H, W)) * hits).astype(np.float32)
    return accum, albedo, normal, depth, hits, obj, spp


def test_no_iterations_is_the_plain_mean():
    accum, albedo, normal, depth, hits, obj, spp = _random_inputs(np.random.default_rng(1), spp=7)
    out = dr.denoise(accum, albedo, normal, depth, hits, obj, spp, iterations=-1)
    assert out.dtype == np.float32 and np.array_equal(out, accum / np.float32(7))


def test_constant_frame_of_one_object_stays_constant():
    H, W, spp = 40, 50, 16
    accum = np.full((H, W, 3), 0.37 * spp, np.float32)
    albedo = np.full((H, W, 3), 0.6 * spp, np.float32)
    normal = np.zeros((H, W, 3), np.float32)
    normal[..., 2] = spp
    depth = np.full((H, W), 31.0 * spp, np.float32)
    hits = np.full((H, W), spp, np.uint32)
    obj = np.full((H, W), 4, np.int32)
    out = dr.denoise(accum, albedo, normal, depth, hits, obj, spp)
    want = accum[0, 0] / np.float32(spp)
    assert np.allclose(out, want, rtol=16 * np.finfo(np.float32).eps, atol=0), np.abs(out - want).max()


@pytest.mark.parametrize("victim", [1, -1])
def test_object_isolation_is_exact(victim):
    rng = np.random.default_rng(2)
    accum, albedo, normal, depth, hits, obj, spp = _random_inputs(rng)
    a = dr.denoise(accum, albedo, normal, depth, hits, obj, spp)
    accum2 = accum.copy()
    accum2[obj == victim] *= np.float32(37.0)
    b = dr.denoise(accum2, albedo, normal, depth, hits, obj, spp)
    keep = obj != victim
    assert (obj == victim).any() and np.array_equal(a[keep], b[keep])
    assert not np.array_equal(a[~keep], b[~keep])
    assert np.isfinite(a).all() and (a >= 0).all()


def test_cli_refuses_the_denoiser_on_several_gpus(tmp_path):
    import subprocess
    exe = os.path.join(os.path.dirname(GOLD), os.pardir, "raytracer.c_b200", "bin", "raytracer")
    r = subprocess.run([exe, "-w", "64", "-h", "36", "-s", "1", "-o", str(tmp_path / "x.png"), "-G", "2", "-n", "5"],
                       capture_output=True, text=True)
    assert r.returncode != 0
    assert "-n" in r.stderr and "-G 2" in r.stderr and "-n <passes>" in r.stderr
    assert os.listdir(tmp_path) == [], "nothing is rendered or written"
