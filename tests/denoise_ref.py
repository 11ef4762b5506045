"""Restatement of the denoiser (rtb_denoise, csrc/rtb_denoise.cu) in numpy, step by step in float32, and the oracle
inputs its calibration uses.

The filter (DESIGN.md section 4.6): per-pixel means from the sums (colour, albedo and normal / spp, depth / hits);
the colour divided by max(albedo, eps) per channel where some sample hit (demodulation); the luminance variance of the
demodulated colour over the 3x3 neighbours of the same object id; then K a-trous passes of the 5x5 B3-spline at step
2^i, each tap weighted by the normal, depth, object-id and luminance terms, with the variance carried as
sum(w^2 var) / sum(w)^2; the albedo multiplied back at the end.  Taps are visited row by row (dy outer, dx inner)
and summed in that order, as the kernel sums them.

Imported by tests/test_denoise_ref.py (CPU) and tests/test_gpu_denoise.py (GPU).
"""
import numpy as np

F32 = np.float32

# defaults of rtb_denoise (RTB_DENOISE_DEFAULT_* in include/rtb200.h), fixed by the calibration in DESIGN.md 4.6
DEFAULTS = dict(iterations=5, sigma_luminance=48.0, sigma_normal=128.0, sigma_depth=0.1, albedo_epsilon=1e-3)
TINY = F32(1e-6)                  # keeps the depth and luminance denominators above 0
LUMA = (F32(0.2126), F32(0.7152), F32(0.0722))
SPLINE = (F32(1 / 16), F32(1 / 4), F32(3 / 8), F32(1 / 4), F32(1 / 16))

# C1 at 320x180 (oracle Philox render, oracle feature sums) against tests/golden/c1_converged_320x180.npz:
# PSNR of the denoised frame must reach these (measured gain minus a margin, DESIGN.md 4.6)
C1_SPP = (4, 16, 64)
C1_PSNR_FLOOR = {4: 22.5, 16: 25.5, 64: 28.5}
# ... and raise it over the raw frame's by at least these (measured: 14.4 / 12.3 / 7.6 dB)
C1_GAIN_FLOOR = {4: 13.0, 16: 11.0, 64: 6.5}
C1_W, C1_H = 320, 180
# |frame mean of the denoised frame / frame mean of the raw frame - 1| stays below this at every spp (measured with
# the defaults on C1: 1.3 / 0.7 / 0.6 % at 4 / 16 / 64 spp)
C1_MEAN_BOUND = 0.02


def _shift(a, dy, dx):
    """a[y + dy, x + dx] with zeros outside the frame, and the in-frame mask"""
    h, w = a.shape[:2]
    out = np.zeros_like(a)
    inside = np.zeros((h, w), bool)
    if abs(dy) >= h or abs(dx) >= w:
        return out, inside
    ys, yd = slice(max(0, dy), h + min(0, dy)), slice(max(0, -dy), h + min(0, -dy))
    xs, xd = slice(max(0, dx), w + min(0, dx)), slice(max(0, -dx), w + min(0, -dx))
    out[yd, xd] = a[ys, xs]
    inside[yd, xd] = True
    return out, inside


def luminance(c):
    return c[..., 0] * LUMA[0] + c[..., 1] * LUMA[1] + c[..., 2] * LUMA[2]


def features(albedo, normal, depth, hits, spp, eps):
    """(demodulation factor [H, W, 3], mean normal [H, W, 3], mean depth [H, W]) as the kernel forms them"""
    n = F32(spp)
    hit = hits > 0
    a = np.where(hit[..., None], np.maximum(albedo / n, F32(eps)), F32(1))
    z = np.where(hit, depth / np.maximum(hits, 1).astype(F32), F32(0))
    return a.astype(F32), (normal / n).astype(F32), z.astype(F32)


def initial_variance(c, obj):
    """luminance variance of the demodulated colour over the 3x3 neighbours with the pixel's object id"""
    lum = luminance(c)
    s1 = np.zeros(lum.shape, F32)
    s2 = np.zeros(lum.shape, F32)
    cnt = np.zeros(lum.shape, F32)
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            lq, inside = _shift(lum, dy, dx)
            oq, _ = _shift(obj, dy, dx)
            m = inside & (oq == obj)
            s1 = np.where(m, s1 + lq, s1)
            s2 = np.where(m, s2 + lq * lq, s2)
            cnt = np.where(m, cnt + F32(1), cnt)
    mean = s1 / cnt
    return np.maximum(F32(0), s2 / cnt - mean * mean)


def atrous_pass(c, var, nrm, z, obj, step, sigma_l, sigma_n, sigma_z):
    lum = luminance(c)
    denom_l = F32(sigma_l) * np.sqrt(var) + TINY
    sum_w = np.zeros(lum.shape, F32)
    sum_c = np.zeros(c.shape, F32)
    sum_v = np.zeros(lum.shape, F32)
    for ky in range(-2, 3):
        for kx in range(-2, 3):
            h = SPLINE[ky + 2] * SPLINE[kx + 2]
            if ky == 0 and kx == 0:
                w = np.full(lum.shape, h, F32)
                cq, vq = c, var
            else:
                dy, dx = ky * step, kx * step
                cq, inside = _shift(c, dy, dx)
                vq, _ = _shift(var, dy, dx)
                nq, _ = _shift(nrm, dy, dx)
                zq, _ = _shift(z, dy, dx)
                oq, _ = _shift(obj, dy, dx)
                dist = F32(step) * np.sqrt(F32(ky * ky + kx * kx))
                dot = nrm[..., 0] * nq[..., 0] + nrm[..., 1] * nq[..., 1] + nrm[..., 2] * nq[..., 2]
                wn = np.power(np.maximum(F32(0), dot), F32(sigma_n))
                wz = np.exp(-np.abs(z - zq) / (F32(sigma_z) * z * dist + TINY))
                wl = np.exp(-np.abs(lum - luminance(cq)) / denom_l)
                w = h * wn * wz * wl
                w = w * (oq == obj).astype(F32)  # the object-id term: exactly 0 across objects
                w = np.where(inside, w, F32(0))   # taps outside the frame are skipped
            sum_w = sum_w + w
            sum_c = sum_c + w[..., None] * cq
            sum_v = sum_v + (w * w) * vq
    return (sum_c / sum_w[..., None]).astype(F32), (sum_v / (sum_w * sum_w)).astype(F32)


def denoise(accum, albedo, normal, depth, hits, obj, spp, iterations=None, sigma_luminance=None, sigma_normal=None,
            sigma_depth=None, albedo_epsilon=None):
    """the denoised MEAN [H, W, 3] float32 of the sums rtb_render_accum / rtb_render_aov return; None = default,
    iterations < 0 = no filtering (accum / float32(spp))"""
    p = dict(DEFAULTS)
    for k, v in dict(iterations=iterations, sigma_luminance=sigma_luminance, sigma_normal=sigma_normal,
                     sigma_depth=sigma_depth, albedo_epsilon=albedo_epsilon).items():
        if v is not None:
            p[k] = v
    accum = np.asarray(accum, F32)
    colour = accum / F32(spp)
    if p["iterations"] < 0:
        return colour
    obj = np.asarray(obj, np.int32)
    a, nrm, z = features(np.asarray(albedo, F32), np.asarray(normal, F32), np.asarray(depth, F32),
                         np.asarray(hits, np.uint32), spp, p["albedo_epsilon"])
    c = colour / a
    var = initial_variance(c, obj)
    for i in range(p["iterations"]):
        c, var = atrous_pass(c, var, nrm, z, obj, 1 << i, p["sigma_luminance"], p["sigma_normal"], p["sigma_depth"])
    return c * a


# ---- oracle inputs ----------------------------------------------------------------------------------------------

_PHILOX_M0, _PHILOX_M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)


def keyed_jitter(seed, pixels, sample):
    """oracle_keyed_jitter for many pixels of one sample: Philox4x32-10 of (pixel, sample, 0xFFFFFFFF, 0)"""
    c0 = pixels.astype(np.uint32)
    c1 = np.full_like(c0, sample)
    c2 = np.full_like(c0, 0xFFFFFFFF)
    c3 = np.zeros_like(c0)
    k0, k1 = seed & 0xFFFFFFFF, seed >> 32
    for _ in range(10):
        p0 = _PHILOX_M0 * c0.astype(np.uint64)
        p1 = _PHILOX_M1 * c2.astype(np.uint64)
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)).astype(np.uint32) ^ c1 ^ np.uint32(k0), p1.astype(np.uint32),
                          (p0 >> np.uint64(32)).astype(np.uint32) ^ c3 ^ np.uint32(k1), p0.astype(np.uint32))
        k0, k1 = (k0 + 0x9E3779B9) & 0xFFFFFFFF, (k1 + 0xBB67AE85) & 0xFFFFFFFF
    return (c0 >> np.uint32(1)).astype(np.float64) / 2147483648.0, (c1 >> np.uint32(1)).astype(np.float64) / 2147483648.0


def camera_rays(cam, seed, w, h, sample, pixels=None):
    """the render's camera rays of one sample for every pixel (or the flat pixel indices `pixels`), [n, 6]
    (oracle_camera_ray, vectorised)"""
    pix = np.arange(w * h) if pixels is None else np.asarray(pixels, np.int64)
    j1, j2 = keyed_jitter(seed, pix, sample)
    u = ((pix % w) + j1) / (w - 1.0)
    v = ((pix // w) + j2) / (h - 1.0)
    pos = np.array(cam.position.tolist())
    hor, ver, llc = (np.array(getattr(cam, k).tolist()) for k in ("horizontal", "vertical", "lower_left_corner"))
    on_plane = llc + (hor * u[:, None] + ver * v[:, None])
    d = pos - on_plane
    length = np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2])
    d = d * (1.0 / length)[:, None]
    return np.concatenate([np.broadcast_to(pos, d.shape), d], axis=1)


def oracle_feature_sums(ol, src, cam, w, h, spp, integrator=0, seed=None):
    """rtb_render_aov's sums of samples [0, spp) from the oracle (brute-force nearest hits of the render's own camera
    rays), summed in the library's order by test_gpu_aov.OracleHits -> dict of [H, W, ...] arrays"""
    from test_gpu_aov import M_OF, OracleHits, materials
    seed = ol.abi.SCENE_SEED if seed is None else seed
    rays = np.stack([camera_rays(cam, seed, w, h, s) for s in range(spp)])
    rec = ol.intersect_rays(src, rays.reshape(-1, 6))
    oh = OracleHits.__new__(OracleHits)
    shape = rays.shape[:2]
    oh.ids, oh.t = rec["ids"].reshape(shape), rec["t"].reshape(shape)
    oh.normals, oh.uvs = rec["normals"].reshape(shape + (3,)), rec["uvs"].reshape(shape + (2,))
    oh.colors, oh.flags = materials(src)
    oh.is_sphere = OracleHits.sphere_mask(src)
    sums, _ = oh.sums(0, spp, 0, M_OF[integrator])
    return {k: (v.reshape(h, w, 3) if v.ndim == 2 else v.reshape(h, w)) for k, v in sums.items()}


def psnr_vs(mean, ref_mean, ol):
    """PSNR of two mean-radiance frames on their 8-bit frames (the reference's transfer, raytracer.c:215-220)"""
    from conftest import psnr_u8
    return psnr_u8(ol.tonemap(np.asarray(mean, np.float64), 1), ol.tonemap(np.asarray(ref_mean, np.float64), 1))
