"""The denoiser on the GPU (rtb_denoise, rtb_render_denoised) against its numpy restatement (tests/denoise_ref.py).

The kernels and the restatement take the same float32 steps in the same order; they differ by the device's fused
multiply-adds and by expf / powf against numpy's, a few float32 ulps per weight.  So the denoised means agree within
REL_BOUND of the frame's largest value, and the 8-bit frames (the reference's transfer) agree except for +-1 level
on at most LEVEL_FRACTION of the values.  What must hold bit for bit does: no filtering is accum / float32(spp), no
value of one object reaches another, and the render's own sums do not change.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import denoise_ref as dr
from test_gpu_aov import SCENES, W, H, _camera, _render_scene

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
REL_BOUND = 1e-4        # |kernel - restatement| <= REL_BOUND * max |restatement|
LEVEL_FRACTION = 0.002  # 8-bit values that may differ by one level
SPP = 8


def _inputs(sc, cam, desc):
    """the GPU's own sums: accum (rtb_render) and the feature buffers (rtb_render_aov)"""
    _, acc, _ = sc.render(cam, desc, want_accum=True)
    f = sc.render_aov(cam, desc)
    return dict(accum=acc, albedo=f["albedo"], normal=f["normal"], depth=f["depth"], hits=f["hits"], object=f["object"])


def _to_dev(a):
    import torch
    a = np.ascontiguousarray(a)
    if a.dtype == np.uint32:
        a = a.view(np.int32)
    return torch.from_numpy(a).cuda()


def gpu_denoise(api, inp, spp, dn=None, stream=None):
    """rtb_denoise on device copies of `inp` -> the denoised mean [H, W, 3]"""
    import torch
    h, w = inp["hits"].shape
    dev = {k: _to_dev(v) for k, v in inp.items()}
    out = torch.full((h, w, 3), -7.0, dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    api.denoise(w, h, spp, *(dev[k].data_ptr() for k in ("accum", "albedo", "normal", "depth", "hits", "object")),
                out.data_ptr(), dn=dn, stream=stream)
    torch.cuda.synchronize()
    return out.cpu().numpy()


def ref_denoise(inp, spp, **kw):
    return dr.denoise(inp["accum"], inp["albedo"], inp["normal"], inp["depth"], inp["hits"], inp["object"], spp, **kw)


def assert_close_to_restatement(ol, got, want, what, nonneg=True):
    """nonneg: the sums are >= 0 (the Whitted integrator's cast_ray can return negative radiance, and a weighted mean
    of negative values stays negative)"""
    assert np.isfinite(got).all() and (not nonneg or (got >= 0).all()), what
    err = np.abs(got.astype(np.float64) - want) / np.abs(want).max()
    print(f"{what}: max |kernel - restatement| / max = {err.max():.2e}")
    assert err.max() <= REL_BOUND, (what, err.max())
    fg, fw = ol.tonemap(got.astype(np.float64), 1), ol.tonemap(want.astype(np.float64), 1)
    diff = np.abs(fg.astype(int) - fw.astype(int))
    assert diff.max() <= 1 and (diff > 0).mean() <= LEVEL_FRACTION, (what, diff.max(), (diff > 0).mean())


# ---- 1. the kernel equals the restatement -------------------------------------------------------------------------

FRAMES = {  # scene of test_gpu_aov, integrator
    "c1": ("c1", 0), "sphere-field": ("sphere-field", 0), "checker-mesh-tex64": ("checker-mesh", 0),
    "mesh-matrix-tri64": ("mesh-matrix", 0), "whitted-checker-spheres": ("checker-spheres", 1),
}


@pytest.mark.parametrize("frame", list(FRAMES))
def test_kernel_equals_the_restatement(gpu_api, ol, abi, frame):
    scene, integrator = FRAMES[frame]
    src, view = SCENES[scene](gpu_api, abi)
    cam = _camera(gpu_api, view)
    with gpu_api.Scene(src) as sc:
        info = sc.info
        assert scene != "checker-mesh" or info.double_texcoords == 1
        assert scene != "mesh-matrix" or info.double_triangles == 1
        inp = _inputs(sc, cam, gpu_api.make_desc(W, H, 0, SPP, integrator=integrator))
    nonneg = bool((inp["accum"] >= 0).all())
    assert nonneg or integrator == 1
    assert_close_to_restatement(ol, gpu_denoise(gpu_api, inp, SPP), ref_denoise(inp, SPP), frame, nonneg)
    dn = gpu_api.denoise_params(iterations=3, sigma_luminance=2.5, sigma_normal=64.0, sigma_depth=0.3,
                                albedo_epsilon=0.02)
    assert_close_to_restatement(ol, gpu_denoise(gpu_api, inp, SPP, dn=dn),
                                ref_denoise(inp, SPP, iterations=3, sigma_luminance=2.5, sigma_normal=64.0,
                                            sigma_depth=0.3, albedo_epsilon=0.02), frame + " (own parameters)", nonneg)


# ---- 2. exact structure -------------------------------------------------------------------------------------------

def test_no_filtering_is_the_plain_mean_bit_for_bit(gpu_api, abi):
    src, _ = SCENES["c1"](gpu_api, abi)
    cam = gpu_api.init_camera(W, H)
    with gpu_api.Scene(src) as sc:
        inp = _inputs(sc, cam, gpu_api.make_desc(W, H, 0, 7))
        fb, out, acc, _ = sc.render_denoised(cam, gpu_api.make_desc(W, H, 0, 7), dn=gpu_api.denoise_params(-1),
                                             want_accum=True)
    got = gpu_denoise(gpu_api, inp, 7, dn=gpu_api.denoise_params(iterations=-1))
    assert np.array_equal(got, inp["accum"] / np.float32(7))
    assert np.array_equal(out, acc / np.float32(7))


@pytest.mark.parametrize("scene", ["checker-mesh", "bvh2-fallback"])
def test_object_isolation_is_exact(gpu_api, abi, scene):
    """change the accum of every pixel of object B (and of the pixels that hit nothing, id -1): no pixel of any other
    object changes by a single bit"""
    src, view = SCENES[scene](gpu_api, abi)
    cam = _camera(gpu_api, view)
    with gpu_api.Scene(src) as sc:
        inp = _inputs(sc, cam, gpu_api.make_desc(W, H, 0, SPP))
    base = gpu_denoise(gpu_api, inp, SPP)
    assert np.isfinite(base).all() and (base >= 0).all()
    ids, counts = np.unique(inp["object"], return_counts=True)
    victims = [int(ids[np.argmax(np.where(ids >= 0, counts, 0))])] + ([-1] if (ids == -1).any() else [])
    assert scene != "bvh2-fallback" or -1 in victims
    for b in victims:
        changed = dict(inp)
        changed["accum"] = inp["accum"].copy()
        changed["accum"][inp["object"] == b] *= np.float32(41.0)
        got = gpu_denoise(gpu_api, changed, SPP)
        keep = inp["object"] != b
        assert np.array_equal(got[keep], base[keep]), (scene, b)
        assert not np.array_equal(got[~keep], base[~keep]), (scene, b)


# ---- 3. the render is untouched -----------------------------------------------------------------------------------

def test_render_sums_are_untouched(gpu_api, abi):
    src, _ = SCENES["checker-mesh"](gpu_api, abi)
    cam = gpu_api.init_camera(W, H)
    descs = [gpu_api.make_desc(W, H, 0, 6), gpu_api.make_desc(W, H, 2, 9, planes=2, integrator=1)]
    with gpu_api.Scene(src) as sc:
        before = [sc.render(cam, d, want_accum=True)[1] for d in descs]
        for d in descs:
            _, _, acc, _ = sc.render_denoised(cam, d, want_accum=True)
            assert np.array_equal(acc, sc.render(cam, d, want_accum=True)[1])
            gpu_denoise(gpu_api, _inputs(sc, cam, d), d.sample_end - d.sample_begin)
        after = [sc.render(cam, d, want_accum=True)[1] for d in descs]
    for a, b in zip(before, after):
        assert np.array_equal(a, b)


def test_render_scene_denoised_keeps_accum_out(gpu_api, abi, ol):
    src, _ = SCENES["checker-mesh"](gpu_api, abi)
    cam = gpu_api.init_camera(W, H)
    _, host = gpu_api.load()
    spp = 5

    def params(acc):
        p = abi.RenderParams()
        host.render_params_default(C.byref(p))
        p.num_gpus = 1
        p.accum_out = acc.ctypes.data_as(C.POINTER(C.c_float))
        return p

    acc0, acc1 = np.zeros((H, W, 3), np.float32), np.zeros((H, W, 3), np.float32)
    fb0 = _render_scene(gpu_api, abi, src, cam, spp, params(acc0))
    fb1 = gpu_api.render_scene_denoised(src, cam, W, H, spp, params(acc1))
    assert np.array_equal(acc0, acc1) and not np.array_equal(fb0, fb1)
    with gpu_api.Scene(src) as sc:
        fb2, out, _, _ = sc.render_denoised(cam, gpu_api.make_desc(W, H, 0, spp))
    assert np.array_equal(fb1, fb2)


def test_render_scene_denoised_with_feature_buffers(gpu_api, abi):
    """render_scene_denoised with a RenderAov: the same frame as without it, and the feature means render_scene_aov
    returns (taken from the denoiser's own feature pass)"""
    src, _ = SCENES["checker-mesh"](gpu_api, abi)
    cam = gpu_api.init_camera(W, H)
    _, host = gpu_api.load()
    p = abi.RenderParams()
    host.render_params_default(C.byref(p))
    p.num_gpus, p.sample_offset, p.integrator = 1, 3, 1
    fb_dn = gpu_api.render_scene_denoised(src, cam, W, H, 6, p)
    fb_both, means = gpu_api.render_scene_denoised(src, cam, W, H, 6, p, want_aov=True)
    _, want = gpu_api.render_scene_aov(src, cam, W, H, 6, p)
    assert np.array_equal(fb_dn, fb_both)
    for k in ("albedo", "normal", "depth", "object"):
        assert np.array_equal(means[k], want[k]), k


# ---- 4. quality ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("spp", dr.C1_SPP)
def test_quality_c1_against_the_converged_golden(gpu_api, ol, spp):
    ref = np.load(os.path.join(GOLD, "c1_converged_320x180.npz"))["mean"]
    w, h = dr.C1_W, dr.C1_H
    objs = gpu_api.scene_default(w, h)
    cam = gpu_api.init_camera(w, h)
    desc = gpu_api.make_desc(w, h, 0, spp)
    with gpu_api.Scene(objs) as sc:
        fb, out, acc, _ = sc.render_denoised(cam, desc, want_accum=True)
        f = sc.render_aov(cam, desc)
    raw = acc / np.float32(spp)
    want = dr.denoise(acc, f["albedo"], f["normal"], f["depth"], f["hits"], f["object"], spp)
    p_raw, p_gpu, p_ref = dr.psnr_vs(raw, ref, ol), dr.psnr_vs(out, ref, ol), dr.psnr_vs(want, ref, ol)
    print(f"C1 {spp} spp on the GPU: raw {p_raw:.2f} dB, denoised {p_gpu:.2f} dB, restatement {p_ref:.2f} dB")
    assert p_gpu >= dr.C1_PSNR_FLOOR[spp], (spp, p_gpu)
    assert abs(p_gpu - p_ref) <= 0.3, (p_gpu, p_ref)
    assert abs(out.mean() / raw.mean() - 1.0) < dr.C1_MEAN_BOUND, (out.mean(), raw.mean())
    from conftest import psnr_u8
    assert psnr_u8(fb, ol.tonemap(ref.astype(np.float64), 1)) >= dr.C1_PSNR_FLOOR[spp]


# ---- 5. API -------------------------------------------------------------------------------------------------------

def test_device_pointers_on_a_torch_stream_match_the_host_call(gpu_api, abi):
    import torch
    src, _ = SCENES["c1"](gpu_api, abi)
    cam = gpu_api.init_camera(W, H)
    desc = gpu_api.make_desc(W, H, 0, SPP, planes=3)
    n_px = W * H
    with gpu_api.Scene(src) as sc:
        _, want, _, _ = sc.render_denoised(cam, desc)
        stream = torch.cuda.Stream()
        b = dict(accum=torch.zeros(3 * n_px), albedo=torch.zeros(3 * n_px), normal=torch.zeros(3 * n_px),
                 depth=torch.zeros(n_px), hits=torch.zeros(n_px, dtype=torch.int32),
                 object=torch.zeros(n_px, dtype=torch.int32), out=torch.zeros(3 * n_px))
        b = {k: v.cuda() for k, v in b.items()}
        torch.cuda.synchronize()
        sc.render_accum(cam, desc, b["accum"].data_ptr(), stream=stream.cuda_stream)
        sc.render_aov_accum(cam, desc, *(b[k].data_ptr() for k in ("albedo", "normal", "depth", "hits", "object")),
                            stream=stream.cuda_stream)
        gpu_api.denoise(W, H, SPP, *(b[k].data_ptr() for k in ("accum", "albedo", "normal", "depth", "hits", "object",
                                                                 "out")), stream=stream.cuda_stream)
        stream.synchronize()
    assert np.array_equal(b["out"].cpu().numpy().reshape(H, W, 3), want)


def test_invalid_arguments(gpu_api, abi):
    import torch
    n_px = W * H
    bufs = [torch.zeros(3 * n_px, device="cuda") for _ in range(3)] + [torch.zeros(n_px, device="cuda")] + [
        torch.zeros(n_px, dtype=torch.int32, device="cuda") for _ in range(2)] + [torch.zeros(3 * n_px, device="cuda")]
    ptrs = [t.data_ptr() for t in bufs]
    ok = dict(width=W, height=H, total_samples=4)
    gpu_api.denoise(W, H, 4, *ptrs)
    bad_calls = [
        (dict(ok), [0] + ptrs[1:], None),                                # NULL accum
        (dict(ok), ptrs[:5] + [0, ptrs[6]], None),                         # NULL object
        (dict(ok), ptrs[:6] + [0], None),                                  # NULL output
        (dict(ok, total_samples=0), ptrs, None),
        (dict(ok, width=1), ptrs, None),
        (dict(ok, height=1), ptrs, None),
        (dict(ok), ptrs, gpu_api.denoise_params(iterations=7)),            # step 64 >= 36
        (dict(ok), ptrs, gpu_api.denoise_params(sigma_luminance=-1.0)),
        (dict(ok), ptrs, gpu_api.denoise_params(sigma_depth=float("nan"))),
    ]
    for kw, p, dn in bad_calls:
        with pytest.raises(gpu_api.RtbError, match=r"\(-1\)"):
            gpu_api.denoise(kw["width"], kw["height"], kw["total_samples"], *p, dn=dn)
    gpu_api.denoise(W, H, 4, *ptrs, dn=gpu_api.denoise_params(iterations=6))  # step 32 < 36: allowed
    src, _ = SCENES["c1"](gpu_api, abi)
    cam = gpu_api.init_camera(W, H)
    with gpu_api.Scene(src) as sc:
        for total, dn in ((0, None), (4, gpu_api.denoise_params(iterations=7))):
            with pytest.raises(gpu_api.RtbError, match=r"\(-1\)"):
                sc.render_denoised(cam, gpu_api.make_desc(W, H, 0, 4), total_samples=total, dn=dn)


def _crop_check(ol, inp, got, spp, y0, x0, size, what):
    """the restatement on a crop; pixels farther than the filter's reach (1 + 2 * (1 + 2 + 4 + 8 + 16) = 63) from a
    crop edge that is not a frame edge depend on nothing outside the crop"""
    fh, fw = inp["hits"].shape
    crop = {k: v[y0:y0 + size, x0:x0 + size] for k, v in inp.items()}
    want = ref_denoise(crop, spp)
    m = 64
    ya, yb = (0 if y0 == 0 else m), (size if y0 + size == fh else size - m)
    xa, xb = (0 if x0 == 0 else m), (size if x0 + size == fw else size - m)
    assert_close_to_restatement(ol, got[y0:y0 + size, x0:x0 + size][ya:yb, xa:xb], want[ya:yb, xa:xb], what)


def test_4k_frame_and_a_frame_off_the_block_tile(gpu_api, ol):
    """3840x2160 (C4's size): crops at a corner and inside; 83x45 (not a multiple of the 16x8 tile): whole frame"""
    for (fw, fh, count, spp) in ((3840, 2160, 2000, 2), (83, 45, 300, 6)):
        objs = gpu_api.scene_sphere_field(count, fw, fh)
        cam = gpu_api.init_camera(fw, fh)
        desc = gpu_api.make_desc(fw, fh, 0, spp)
        with gpu_api.Scene(objs) as sc:
            fb, out, acc, _ = sc.render_denoised(cam, desc, want_accum=True)
            inp = _inputs(sc, cam, desc)
        assert np.array_equal(acc, inp["accum"])
        assert np.isfinite(out).all() and (out >= 0).all()
        if fw == 83:
            assert_close_to_restatement(ol, out, ref_denoise(inp, spp), "83x45")
        else:
            for y0, x0 in ((0, 0), (1000, 1700), (2160 - 256, 3840 - 256)):
                _crop_check(ol, inp, out, spp, y0, x0, 256, f"4K crop at ({y0}, {x0})")


# ---- 6. CLI -------------------------------------------------------------------------------------------------------

def _png_of(gpu_api, fb, path):
    _, host = gpu_api.load()
    h, w, _ = fb.shape
    assert host.rt_write_png(os.fsencode(str(path)), w, h, 3, np.ascontiguousarray(fb).ctypes.data, w * 3) != 0
    return path.read_bytes()


def test_cli_writes_the_denoised_png(gpu_api, abi, tmp_path):
    """bin/raytracer -n 5: the PNG of render_scene_denoised's frame; without -n, the PNG of render_scene's frame"""
    exe = os.path.join(ROOT, "raytracer.c_b200", "bin", "raytracer")
    cw, ch, spp, grid = 96, 54, 4, 24
    base = [exe, "-w", str(cw), "-h", str(ch), "-s", str(spp), "-c", f"mesh:{grid}"]
    env = dict(os.environ, RTB_NUM_GPUS="1")
    r = subprocess.run(base + ["-o", str(tmp_path / "dn.png"), "-n", "5", "-a", str(tmp_path / "x")],
                       capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    r = subprocess.run(base + ["-o", str(tmp_path / "plain.png")], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    holder = gpu_api.mesh_room(gpu_api.heightfield_mesh(grid, 20 * cw / ch * 0.98), cw, ch)
    cam = gpu_api.init_camera(cw, ch)
    fb_dn = gpu_api.render_scene_denoised(holder, cam, cw, ch, spp)
    fb_plain = _render_scene_fb(gpu_api, abi, holder, cam, cw, ch, spp)
    assert (tmp_path / "dn.png").read_bytes() == _png_of(gpu_api, fb_dn, tmp_path / "api_dn.png")
    assert (tmp_path / "plain.png").read_bytes() == _png_of(gpu_api, fb_plain, tmp_path / "api_plain.png")
    # the feature buffers written next to the denoised frame are the plain -a run's (one feature pass serves both)
    from test_gpu_aov import read_pfm
    _, means = gpu_api.render_scene_aov(holder, cam, cw, ch, spp)
    for k in ("albedo", "normal", "depth"):
        assert np.array_equal(read_pfm(tmp_path / f"x_{k}.pfm"), means[k]), k


def _render_scene_fb(gpu_api, abi, holder, cam, w, h, spp):
    _, host = gpu_api.load()
    fb = np.zeros((h, w, 3), np.uint8)
    opt = abi.Options()
    opt.width, opt.height, opt.samples = w, h, spp
    p = abi.RenderParams()
    host.render_params_default(C.byref(p))
    p.num_gpus = 1
    host.render_scene(fb.ctypes.data, C.addressof(holder.objects), holder.n, C.byref(cam), C.byref(opt), C.byref(p))
    return fb
