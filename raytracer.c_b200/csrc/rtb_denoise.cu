/*
 * rtb_denoise.cu -- edge-avoiding a-trous denoiser of a rendered frame, guided by the first-hit feature buffers of
 * rtb_render_aov (Dammertz et al. 2010; the variance-guided weights of SVGF, Schied et al. 2017, spatial part only).
 *
 * Inputs are the SUMS rtb_render_accum and rtb_render_aov return, and the sample count; the kernels form the means:
 *   colour = accum / spp, albedo = albedo / spp, normal = normal / spp, depth = depth / hits (0 where hits = 0).
 * Steps (DESIGN.md section 4.6; tests/denoise_ref.py restates them in numpy):
 *   1. k_dn_demod     demodulated colour c = colour / max(albedo, eps) per channel where some sample hit (else the
 *                     factor is 1), so that texture is not blurred; the features (normal, depth) and the factor.
 *   2. k_dn_variance  luminance variance of c over the 3x3 neighbours with the pixel's object id.
 *   3. k_dn_atrous    K passes of the 5x5 B3-spline (1/16, 1/4, 3/8, 1/4, 1/16)^2 at offsets 2^i (dx, dy).  The weight
 *                     of tap q for pixel p is the spline weight times
 *                       max(0, n_p . n_q)^sigma_n
 *                       exp(-|z_p - z_q| / (sigma_z z_p |offset| + tiny))
 *                       [id_p == id_q]
 *                       exp(-|l_p - l_q| / (sigma_l sqrt(var_p) + tiny));
 *                     the centre tap's weight is its spline weight.  Taps outside the frame are skipped, the weights
 *                     renormalised; the variance is carried as sum(w^2 var) / (sum w)^2.  Taps are summed row by row
 *                     (dy outer, dx inner).  The last pass multiplies the albedo factor back and writes the mean.
 * A tap of another object has weight exactly 0: the kernel skips it before it reads anything of that pixel, which
 * adds what 0 * its value would add without any chance of 0 * inf.  So no value of one object can reach the output of
 * another, bit for bit.  Arithmetic is float32.
 *
 * Buffers of one call (demodulated colour + variance twice for the ping-pong, features, albedo factor: 64 B per pixel)
 * come from the stream-ordered pool; the render's scene and its scratch are not touched.
 */
#include "rtb_internal.h"

#define RTB_DN_BX 16 /* block tile of the 2D kernels: 16 x 8 pixels */
#define RTB_DN_BY 8
#define RTB_DN_TINY 1e-6f

__device__ __forceinline__ float dn_luminance(float4 c) { return c.x * 0.2126f + c.y * 0.7152f + c.z * 0.0722f; }

/* iterations < 0: the plain mean */
__global__ void k_dn_mean(const float *__restrict__ accum, size_t n, float spp, float *__restrict__ out)
{
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n)
    out[i] = accum[i] / spp;
}

/* per-pixel means; col = (demodulated colour, 0), feat = (mean normal, mean depth), alb = (factor, 0) */
__global__ void k_dn_demod(const float *__restrict__ accum, const float *__restrict__ albedo,
                           const float *__restrict__ normal, const float *__restrict__ depth,
                           const uint32_t *__restrict__ hits, size_t n_px, float spp, float eps,
                           float4 *__restrict__ col, float4 *__restrict__ feat, float4 *__restrict__ alb)
{
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_px)
    return;
  const uint32_t h = hits[i];
  float a[3], c[3], nm[3];
  for (int k = 0; k < 3; k++)
  {
    a[k] = h ? fmaxf(albedo[3 * i + k] / spp, eps) : 1.0f;
    c[k] = (accum[3 * i + k] / spp) / a[k];
    nm[k] = normal[3 * i + k] / spp;
  }
  col[i] = make_float4(c[0], c[1], c[2], 0.0f);
  feat[i] = make_float4(nm[0], nm[1], nm[2], h ? depth[i] / (float)h : 0.0f);
  alb[i] = make_float4(a[0], a[1], a[2], 0.0f);
}

/* out = (colour of in, luminance variance over the 3x3 neighbours of the same object) */
__global__ void k_dn_variance(const float4 *__restrict__ in, const int32_t *__restrict__ object, int width, int height,
                              float4 *__restrict__ out)
{
  const int x = blockIdx.x * RTB_DN_BX + threadIdx.x, y = blockIdx.y * RTB_DN_BY + threadIdx.y;
  if (x >= width || y >= height)
    return;
  const size_t p = (size_t)y * width + x;
  const int id = object[p];
  float s1 = 0.0f, s2 = 0.0f, cnt = 0.0f;
#pragma unroll
  for (int dy = -1; dy <= 1; dy++)
#pragma unroll
    for (int dx = -1; dx <= 1; dx++)
    {
      const int qx = x + dx, qy = y + dy;
      if (qx < 0 || qx >= width || qy < 0 || qy >= height)
        continue;
      const size_t q = (size_t)qy * width + qx;
      if (object[q] != id)
        continue;
      const float l = dn_luminance(in[q]);
      s1 += l;
      s2 += l * l;
      cnt += 1.0f;
    }
  const float mean = s1 / cnt;
  const float4 c = in[p];
  out[p] = make_float4(c.x, c.y, c.z, fmaxf(0.0f, s2 / cnt - mean * mean));
}

struct DnPass
{
  const float4 *in, *feat, *alb;
  const int32_t *object;
  float4 *out;  /* not the last pass: next (colour, variance) */
  float *out3;  /* last pass: the denoised mean, H*W*3 */
  int width, height, step;
  float sigma_l, sigma_n, sigma_z;
};

template <bool LAST>
__global__ void __launch_bounds__(RTB_DN_BX *RTB_DN_BY) k_dn_atrous(const __grid_constant__ DnPass P)
{
  const int x = blockIdx.x * RTB_DN_BX + threadIdx.x, y = blockIdx.y * RTB_DN_BY + threadIdx.y;
  if (x >= P.width || y >= P.height)
    return;
  const size_t p = (size_t)y * P.width + x;
  const float4 cp = P.in[p], fp = P.feat[p];
  const int id = P.object[p];
  const float lp = dn_luminance(cp);
  const float den_l = P.sigma_l * sqrtf(cp.w) + RTB_DN_TINY;
  const float spline[5] = { 1.0f / 16, 1.0f / 4, 3.0f / 8, 1.0f / 4, 1.0f / 16 };
  float sw = 0.0f, sr = 0.0f, sg = 0.0f, sb = 0.0f, sv = 0.0f;
#pragma unroll
  for (int ky = -2; ky <= 2; ky++)
  {
    const int qy = y + ky * P.step;
    if (qy < 0 || qy >= P.height)
      continue;
#pragma unroll
    for (int kx = -2; kx <= 2; kx++)
    {
      const float h = spline[ky + 2] * spline[kx + 2];
      float w;
      float4 cq;
      if (ky == 0 && kx == 0)
      {
        w = h;
        cq = cp;
      }
      else
      {
        const int qx = x + kx * P.step;
        if (qx < 0 || qx >= P.width)
          continue;
        const size_t q = (size_t)qy * P.width + qx;
        if (P.object[q] != id)
          continue; /* the object-id term: exactly 0 */
        const float4 fq = P.feat[q];
        cq = P.in[q];
        const float dist = (float)P.step * sqrtf((float)(ky * ky + kx * kx));
        const float dot = fp.x * fq.x + fp.y * fq.y + fp.z * fq.z;
        const float wn = powf(fmaxf(0.0f, dot), P.sigma_n);
        const float wz = expf(-fabsf(fp.w - fq.w) / (P.sigma_z * fp.w * dist + RTB_DN_TINY));
        const float wl = expf(-fabsf(lp - dn_luminance(cq)) / den_l);
        w = h * wn * wz * wl;
      }
      sw += w;
      sr += w * cq.x;
      sg += w * cq.y;
      sb += w * cq.z;
      sv += (w * w) * cq.w;
    }
  }
  if (LAST)
  {
    const float4 a = P.alb[p];
    P.out3[3 * p + 0] = (sr / sw) * a.x;
    P.out3[3 * p + 1] = (sg / sw) * a.y;
    P.out3[3 * p + 2] = (sb / sw) * a.z;
  }
  else
    P.out[p] = make_float4(sr / sw, sg / sw, sb / sw, sv / (sw * sw));
}

/* 0 = default: the parameters of one call */
static int dn_resolve(const rtb_denoise_desc *dn, int width, int height, rtb_denoise_desc *out)
{
  rtb_denoise_desc d = {};
  if (dn)
    d = *dn;
  if (!(d.sigma_luminance >= 0.0f) || !(d.sigma_normal >= 0.0f) || !(d.sigma_depth >= 0.0f) ||
      !(d.albedo_epsilon >= 0.0f) || !isfinite(d.sigma_luminance) || !isfinite(d.sigma_normal) ||
      !isfinite(d.sigma_depth) || !isfinite(d.albedo_epsilon))
  {
    rtb_set_error("rtb_denoise: sigmas and albedo_epsilon must be finite and >= 0 (0 = default)");
    return RTB_EINVAL;
  }
  if (d.iterations == 0)
    d.iterations = RTB_DENOISE_DEFAULT_ITERATIONS;
  if (d.sigma_luminance == 0.0f)
    d.sigma_luminance = RTB_DENOISE_DEFAULT_SIGMA_LUMINANCE;
  if (d.sigma_normal == 0.0f)
    d.sigma_normal = RTB_DENOISE_DEFAULT_SIGMA_NORMAL;
  if (d.sigma_depth == 0.0f)
    d.sigma_depth = RTB_DENOISE_DEFAULT_SIGMA_DEPTH;
  if (d.albedo_epsilon == 0.0f)
    d.albedo_epsilon = RTB_DENOISE_DEFAULT_ALBEDO_EPSILON;
  /* the last pass's step 2^(K-1) must stay inside the frame */
  if (d.iterations > 0 && (d.iterations > 30 || (1 << (d.iterations - 1)) >= (width < height ? width : height)))
  {
    rtb_set_error("rtb_denoise: " + std::to_string(d.iterations) + " passes: the step of the last one (2^" +
                  std::to_string(d.iterations - 1) + ") must be below the frame's smaller side (" +
                  std::to_string(width < height ? width : height) + ")");
    return RTB_EINVAL;
  }
  *out = d;
  return RTB_OK;
}

extern "C" int rtb_denoise(const rtb_denoise_desc *dn, int width, int height, int total_samples, const float *d_accum3,
                           const float *d_albedo3, const float *d_normal3, const float *d_depth, const uint32_t *d_hits,
                           const int32_t *d_object, float *d_out3, int device, void *stream_)
{
  if (!d_accum3 || !d_albedo3 || !d_normal3 || !d_depth || !d_hits || !d_object || !d_out3)
  {
    rtb_set_error("rtb_denoise: NULL buffer");
    return RTB_EINVAL;
  }
  if (width < 2 || height < 2 || (long long)width * height >= (1ll << 30) || total_samples <= 0)
  {
    rtb_set_error("rtb_denoise: need width, height >= 2 (fewer than 2^30 pixels) and total_samples > 0");
    return RTB_EINVAL;
  }
  rtb_denoise_desc d;
  int rc = dn_resolve(dn, width, height, &d);
  if (rc != RTB_OK)
    return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  RTB_CUDA(cudaSetDevice(device));
  const size_t n_px = (size_t)width * height;
  const float spp = (float)total_samples;
  if (d.iterations < 0)
  {
    k_dn_mean<<<(unsigned)((3 * n_px + 255) / 256), 256, 0, stream>>>(d_accum3, 3 * n_px, spp, d_out3);
    RTB_CUDA(cudaGetLastError());
    return RTB_OK;
  }

  PoolBufs pool;
  pool.stream = stream;
  float4 *col[2], *feat, *alb;
  for (float4 **b : { &col[0], &col[1], &feat, &alb })
    RTB_CUDA(pool.alloc(reinterpret_cast<void **>(b), sizeof(float4) * n_px));
  k_dn_demod<<<(unsigned)((n_px + 255) / 256), 256, 0, stream>>>(d_accum3, d_albedo3, d_normal3, d_depth, d_hits, n_px,
                                                                  spp, d.albedo_epsilon, col[0], feat, alb);
  RTB_CUDA(cudaGetLastError());
  const dim3 block(RTB_DN_BX, RTB_DN_BY), grid((width + RTB_DN_BX - 1) / RTB_DN_BX, (height + RTB_DN_BY - 1) / RTB_DN_BY);
  k_dn_variance<<<grid, block, 0, stream>>>(col[0], d_object, width, height, col[1]);
  RTB_CUDA(cudaGetLastError());
  DnPass P;
  P.feat = feat;
  P.alb = alb;
  P.object = d_object;
  P.out3 = d_out3;
  P.width = width;
  P.height = height;
  P.sigma_l = d.sigma_luminance;
  P.sigma_n = d.sigma_normal;
  P.sigma_z = d.sigma_depth;
  for (int i = 0; i < d.iterations; i++)
  {
    P.in = col[(i + 1) & 1];
    P.out = col[i & 1];
    P.step = 1 << i;
    if (i + 1 == d.iterations)
      k_dn_atrous<true><<<grid, block, 0, stream>>>(P);
    else
      k_dn_atrous<false><<<grid, block, 0, stream>>>(P);
    RTB_CUDA(cudaGetLastError());
  }
  return RTB_OK;
}

extern "C" int rtb_render_denoised_aov(rtb_scene *scene, const double *camera12, const rtb_render_desc *desc,
                                       int total_samples, const rtb_denoise_desc *dn_or_null, uint8_t *framebuffer,
                                       float *denoised3_or_null, float *accum_or_null, float *albedo3_or_null,
                                       float *normal3_or_null, float *depth_or_null, uint32_t *hits_or_null,
                                       int32_t *object_or_null, rtb_counters *counters)
{
  if (!scene || !camera12 || !framebuffer || total_samples <= 0)
  {
    rtb_set_error("rtb_render_denoised: NULL scene, camera or framebuffer, or total_samples <= 0");
    return RTB_EINVAL;
  }
  int rc = rtb_check_desc(desc);
  if (rc != RTB_OK)
    return rc;
  rtb_denoise_desc d;
  rc = dn_resolve(dn_or_null, desc->width, desc->height, &d); /* before any work */
  if (rc != RTB_OK)
    return rc;
  RTB_CUDA(cudaSetDevice(scene->device));
  const size_t n_px = (size_t)desc->width * desc->height;
  PoolBufs pool; /* the legacy default stream, like rtb_render */
  float *d_accum, *d_albedo, *d_normal, *d_depth, *d_out;
  uint32_t *d_hits;
  int32_t *d_object;
  uint8_t *d_fb;
  RTB_CUDA(pool.alloc(reinterpret_cast<void **>(&d_accum), sizeof(float) * 3 * n_px));
  RTB_CUDA(pool.alloc(reinterpret_cast<void **>(&d_albedo), sizeof(float) * 3 * n_px));
  RTB_CUDA(pool.alloc(reinterpret_cast<void **>(&d_normal), sizeof(float) * 3 * n_px));
  RTB_CUDA(pool.alloc(reinterpret_cast<void **>(&d_depth), sizeof(float) * n_px));
  RTB_CUDA(pool.alloc(reinterpret_cast<void **>(&d_hits), sizeof(uint32_t) * n_px));
  RTB_CUDA(pool.alloc(reinterpret_cast<void **>(&d_object), sizeof(int32_t) * n_px));
  RTB_CUDA(pool.alloc(reinterpret_cast<void **>(&d_out), sizeof(float) * 3 * n_px));
  RTB_CUDA(pool.alloc(reinterpret_cast<void **>(&d_fb), 3 * n_px));
  rc = rtb_render_accum(scene, camera12, desc, d_accum, nullptr, counters);
  /* the features of a next-event-estimation render are the first hits of trace_path's own camera samples */
  rtb_render_desc feat = *desc;
  if (feat.integrator == RTB_INTEGRATOR_PATH_NEE)
    feat.integrator = RTB_INTEGRATOR_PATH;
  if (rc == RTB_OK)
    rc = rtb_render_aov(scene, camera12, &feat, d_albedo, d_normal, d_depth, d_hits, d_object, nullptr, nullptr);
  if (rc == RTB_OK)
    rc = rtb_denoise(&d, desc->width, desc->height, total_samples, d_accum, d_albedo, d_normal, d_depth, d_hits,
                     d_object, d_out, scene->device, nullptr);
  if (rc == RTB_OK)
    rc = rtb_tonemap(d_out, desc->width, desc->height, 1, d_fb, scene->device, nullptr);
  if (rc != RTB_OK)
    return rc;
  RTB_CUDA(cudaMemcpy(framebuffer, d_fb, 3 * n_px, cudaMemcpyDeviceToHost));
  if (denoised3_or_null)
    RTB_CUDA(cudaMemcpy(denoised3_or_null, d_out, sizeof(float) * 3 * n_px, cudaMemcpyDeviceToHost));
  if (accum_or_null)
    RTB_CUDA(cudaMemcpy(accum_or_null, d_accum, sizeof(float) * 3 * n_px, cudaMemcpyDeviceToHost));
  /* the feature sums the filter used: a caller that also wants them does not pay for a second feature pass */
  const struct { void *host; const void *dev; size_t bytes; } feats[5] = {
    { albedo3_or_null, d_albedo, sizeof(float) * 3 * n_px }, { normal3_or_null, d_normal, sizeof(float) * 3 * n_px },
    { depth_or_null, d_depth, sizeof(float) * n_px }, { hits_or_null, d_hits, sizeof(uint32_t) * n_px },
    { object_or_null, d_object, sizeof(int32_t) * n_px } };
  for (const auto &f : feats)
    if (f.host)
      RTB_CUDA(cudaMemcpy(f.host, f.dev, f.bytes, cudaMemcpyDeviceToHost));
  return RTB_OK;
}

extern "C" int rtb_render_denoised(rtb_scene *scene, const double *camera12, const rtb_render_desc *desc,
                                   int total_samples, const rtb_denoise_desc *dn_or_null, uint8_t *framebuffer,
                                   float *denoised3_or_null, float *accum_or_null, rtb_counters *counters)
{
  return rtb_render_denoised_aov(scene, camera12, desc, total_samples, dn_or_null, framebuffer, denoised3_or_null,
                                 accum_or_null, nullptr, nullptr, nullptr, nullptr, nullptr, counters);
}
