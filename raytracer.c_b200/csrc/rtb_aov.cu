/*
 * rtb_aov.cu -- first-hit feature buffers ("AOVs") of the render's own camera samples: albedo, normal, depth, hit
 * count and object id per pixel.  A denoiser (OIDN, OptiX) wants albedo and normal buffers with the pixel footprint of
 * the image; compositing wants depth and an object mask.
 *
 * For every pixel and every sample s of [sample_begin, sample_end) the camera ray is path_begin's, with the render's
 * own Philox jitter words, so it is the primary ray of that sample in both integrators.  Its exact nearest hit
 * (nearest_hit: the compressed BVH4, or the BVH2 when the scene has none) and surface_at give, all in double:
 *   albedo  colors[obj], times the checker factor (0.3 or 0.7) for an M_CHECKERED object at the integrator's M:
 *           100 000 for trace_path (raytracer.c:508), 10 for cast_ray (raytracer.c:584)
 *   normal  surface_at's normal (outward on spheres, cross(v2 - v0, v1 - v0) on triangles; not flipped to the camera)
 *   depth   t of the hit (the camera direction is unit length)
 *   hits    1
 * and 0 on a miss.  The object id (-1 on a miss) is the one of the call's first sample.
 *
 * Summation order, the same as the megakernel / Whitted renders': the samples are cut into planes (rtb_plane_split),
 * one thread per (plane, pixel) sums its plane's samples in double in sample order and rounds to float once, and the
 * planes are summed in float in plane order (rtb_sum_planes).  Hits are an exact integer count.  The outputs are SUMS,
 * like the render's, so that a caller may shard the sample range.
 *
 * The pass is separate from the render kernels, which it leaves untouched: it traces the primary rays a second time.
 */
#include <cstring>

#include "rtb_path.cuh"

struct AovArgs
{
  float *albedo, *normal, *depth; /* [plane][H*W*3], [plane][H*W*3], [plane][H*W]; any may be NULL */
  unsigned *hits;                 /* [H*W], zeroed by the caller, or NULL */
  int *object;                    /* [H*W] or NULL */
  double checker_M;
  unsigned long long *counters;   /* [0] rays, [1] prim tests, [2] node visits (STATS only) */
};

/* one thread per (plane, pixel); a warp covers an 8 x 4 pixel tile (as k_wf_generate), so its rays are coherent */
template <bool STATS>
__global__ void __launch_bounds__(128, 1) k_render_aov(const __grid_constant__ RenderArgs A, const __grid_constant__ AovArgs O)
{
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int tile = (int)(warp % A.n_tiles);
  const int plane = (int)(warp / A.n_tiles);
  const int x = (tile % A.tiles_x) * 8 + (lane & 7);
  const int y = (tile / A.tiles_x) * 4 + (lane >> 3);
  const bool valid = x < A.width && y < A.height && plane < A.splits;
  const int s0 = A.s_begin + plane * A.chunk;
  const int s1 = valid ? min(A.s_end, s0 + A.chunk) : s0;
  const unsigned pix = valid ? (unsigned)(y * A.width + x) : 0u;

  d3 albedo = d3_make(0, 0, 0), normal = d3_make(0, 0, 0);
  double depth = 0.0;
  unsigned hits = 0;
  int first_object = -1;
  TraceStats ts = { 0u, 0u };
  for (int s = s0; s < s1; s++)
  {
    PathState st;
    path_begin(A, st, x, y, pix, (unsigned)s);
    HitRec best;
    if (!nearest_hit<STATS>(A.sv, st.o, st.d, best, ts))
      continue; /* a miss adds 0 everywhere */
    int obj;
    {
      const float4 *rec = best.slot >= 0 ? A.sv.prims + 3 * best.slot : A.sv.big + 3 * (~best.slot);
      obj = (int)(__float_as_uint(__ldg(rec + 2).z) & 0x7FFFFFFFu);
    }
    const bool checkered = (__float_as_uint(__ldg(A.sv.mats + 2 * obj + 1).w) & RT_M_CHECKERED) != 0;
    const Surface sf = surface_at(A.sv, st.o, st.d, best, checkered);
    d3 c = d3_make(A.sv.colors[3 * obj + 0], A.sv.colors[3 * obj + 1], A.sv.colors[3 * obj + 2]);
    if (checkered)
      c = checker_color(c, sf.u, sf.v, O.checker_M);
    albedo = d3_add(albedo, c);
    normal = d3_add(normal, sf.normal);
    depth = __dadd_rn(depth, best.t);
    hits++;
    if (s == A.s_begin)
      first_object = sf.object;
  }

  if (valid)
  {
    const size_t n_px = (size_t)A.width * A.height;
    if (O.albedo)
    {
      float *p = O.albedo + (size_t)plane * 3 * n_px + 3 * (size_t)pix;
      p[0] = (float)albedo.x; p[1] = (float)albedo.y; p[2] = (float)albedo.z;
    }
    if (O.normal)
    {
      float *p = O.normal + (size_t)plane * 3 * n_px + 3 * (size_t)pix;
      p[0] = (float)normal.x; p[1] = (float)normal.y; p[2] = (float)normal.z;
    }
    if (O.depth)
      O.depth[(size_t)plane * n_px + pix] = (float)depth;
    if (O.hits && hits)
      atomicAdd(O.hits + pix, hits);
    if (O.object && plane == 0)
      O.object[pix] = first_object;
  }
  if (STATS)
  {
    unsigned long long rays = (unsigned long long)(s1 - s0), tests = ts.prim_tests, nodes = ts.node_visits;
    for (int off = 16; off > 0; off >>= 1)
    {
      rays += __shfl_xor_sync(0xFFFFFFFFu, rays, off);
      tests += __shfl_xor_sync(0xFFFFFFFFu, tests, off);
      nodes += __shfl_xor_sync(0xFFFFFFFFu, nodes, off);
    }
    if (lane == 0)
    {
      atomicAdd(&O.counters[0], rays);
      atomicAdd(&O.counters[1], tests);
      atomicAdd(&O.counters[2], nodes);
    }
  }
}

extern "C" int rtb_render_aov(rtb_scene *scene, const double *camera12, const rtb_render_desc *desc, float *d_albedo3,
                              float *d_normal3, float *d_depth, uint32_t *d_hits, int32_t *d_object, void *stream_,
                              rtb_counters *counters)
{
  if (!scene || !camera12)
  {
    rtb_set_error("rtb_render_aov: NULL scene or camera");
    return RTB_EINVAL;
  }
  if (!d_albedo3 && !d_normal3 && !d_depth && !d_hits && !d_object)
  {
    rtb_set_error("rtb_render_aov: every output is NULL");
    return RTB_EINVAL;
  }
  int rc = rtb_check_desc(desc);
  if (rc != RTB_OK)
    return rc;
  if (desc->integrator == RTB_INTEGRATOR_PATH_NEE)
  {
    /* integrator only selects the checker's M here; an NEE render's features are RTB_INTEGRATOR_PATH's */
    rtb_set_error("rtb_render_aov: integrator RTB_INTEGRATOR_PATH or RTB_INTEGRATOR_WHITTED");
    return RTB_EINVAL;
  }
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  RTB_CUDA(cudaSetDevice(scene->device));

  RenderArgs A;
  fill_args(A, scene, camera12, desc);
  const int spp = desc->sample_end - desc->sample_begin;
  const size_t n_px = (size_t)desc->width * desc->height;
  int chunk = 0;
  const int splits = rtb_plane_split(RTB_MEGAKERNEL_THREADS, n_px, desc->planes, spp, &chunk);
  A.chunk = chunk;
  A.splits = splits;
  A.out = nullptr;

  PoolBufs pool;
  pool.stream = stream;
  Events ev;
  unsigned long long *d_ctr = nullptr;
  if (counters)
  {
    RTB_CUDA(cudaEventCreate(&ev.a));
    RTB_CUDA(cudaEventCreate(&ev.b));
    RTB_CUDA(pool.alloc(reinterpret_cast<void **>(&d_ctr), sizeof(unsigned long long) * 3));
    RTB_CUDA(cudaMemsetAsync(d_ctr, 0, sizeof(unsigned long long) * 3, stream));
    RTB_CUDA(cudaEventRecord(ev.a, stream));
  }

  unsigned long long launches = 0;
  if (d_hits)
    RTB_CUDA(cudaMemsetAsync(d_hits, 0, sizeof(uint32_t) * n_px, stream));
  if (spp == 0)
  {
    if (d_albedo3) RTB_CUDA(cudaMemsetAsync(d_albedo3, 0, sizeof(float) * 3 * n_px, stream));
    if (d_normal3) RTB_CUDA(cudaMemsetAsync(d_normal3, 0, sizeof(float) * 3 * n_px, stream));
    if (d_depth) RTB_CUDA(cudaMemsetAsync(d_depth, 0, sizeof(float) * n_px, stream));
    if (d_object) RTB_CUDA(cudaMemsetAsync(d_object, 0xFF, sizeof(int32_t) * n_px, stream)); /* -1 */
  }
  else
  {
    AovArgs O;
    O.albedo = d_albedo3;
    O.normal = d_normal3;
    O.depth = d_depth;
    O.hits = d_hits;
    O.object = d_object;
    O.checker_M = desc->integrator == RTB_INTEGRATOR_WHITTED ? 10.0 : 100000.0;
    O.counters = d_ctr;
    if (splits > 1)
    {
      /* one plane buffer per float output, summed into the caller's buffer after the kernel */
      if (d_albedo3) RTB_CUDA(pool.alloc(reinterpret_cast<void **>(&O.albedo), sizeof(float) * 3 * n_px * splits));
      if (d_normal3) RTB_CUDA(pool.alloc(reinterpret_cast<void **>(&O.normal), sizeof(float) * 3 * n_px * splits));
      if (d_depth) RTB_CUDA(pool.alloc(reinterpret_cast<void **>(&O.depth), sizeof(float) * n_px * splits));
    }
    const long long threads = (long long)A.n_tiles * splits * 32;
    const unsigned blocks = (unsigned)((threads + 127) / 128);
    if (counters)
      k_render_aov<true><<<blocks, 128, 0, stream>>>(A, O);
    else
      k_render_aov<false><<<blocks, 128, 0, stream>>>(A, O);
    RTB_CUDA(cudaGetLastError());
    launches++;
    if (splits > 1)
    {
      const struct { const float *planes; float *out; size_t n; } sums[3] = {
        { O.albedo, d_albedo3, 3 * n_px }, { O.normal, d_normal3, 3 * n_px }, { O.depth, d_depth, n_px } };
      for (const auto &s : sums)
        if (s.out)
        {
          rc = rtb_sum_planes(s.planes, splits, s.n, s.out, stream);
          if (rc != RTB_OK)
            return rc;
          launches++;
        }
    }
  }

  if (counters)
  {
    RTB_CUDA(cudaEventRecord(ev.b, stream));
    RTB_CUDA(cudaEventSynchronize(ev.b));
    unsigned long long h[3];
    RTB_CUDA(cudaMemcpy(h, d_ctr, sizeof(h), cudaMemcpyDeviceToHost));
    memset(counters, 0, sizeof(*counters));
    counters->rays = h[0];
    counters->rays_intersected = h[0];
    counters->paths = h[0];
    counters->prim_tests = h[1];
    counters->node_visits = h[2];
    counters->launches = launches;
    RTB_CUDA(cudaEventElapsedTime(&counters->gpu_ms, ev.a, ev.b));
    counters->build_ms = scene->info.build_ms;
  }
  return RTB_OK;
}

extern "C" int rtb_render_aov_host(rtb_scene *scene, const double *camera12, const rtb_render_desc *desc, float *albedo3,
                                   float *normal3, float *depth, uint32_t *hits, int32_t *object, rtb_counters *counters)
{
  if (!scene || !desc)
  {
    rtb_set_error("rtb_render_aov_host: NULL scene or desc");
    return RTB_EINVAL;
  }
  int rc = rtb_check_desc(desc);
  if (rc != RTB_OK)
    return rc;
  RTB_CUDA(cudaSetDevice(scene->device));
  const size_t n_px = (size_t)desc->width * desc->height;
  struct Out { void *host; size_t bytes; void *dev; } outs[5] = {
    { albedo3, sizeof(float) * 3 * n_px, nullptr }, { normal3, sizeof(float) * 3 * n_px, nullptr },
    { depth, sizeof(float) * n_px, nullptr }, { hits, sizeof(uint32_t) * n_px, nullptr },
    { object, sizeof(int32_t) * n_px, nullptr } };
  PoolBufs pool; /* the legacy default stream, like rtb_render */
  for (Out &o : outs)
    if (o.host)
      RTB_CUDA(pool.alloc(&o.dev, o.bytes));
  rc = rtb_render_aov(scene, camera12, desc, static_cast<float *>(outs[0].dev), static_cast<float *>(outs[1].dev),
                      static_cast<float *>(outs[2].dev), static_cast<uint32_t *>(outs[3].dev),
                      static_cast<int32_t *>(outs[4].dev), nullptr, counters);
  if (rc != RTB_OK)
    return rc;
  for (Out &o : outs)
    if (o.host)
      RTB_CUDA(cudaMemcpy(o.host, o.dev, o.bytes, cudaMemcpyDeviceToHost));
  return RTB_OK;
}
