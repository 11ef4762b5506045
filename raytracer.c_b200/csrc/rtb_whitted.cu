/*
 * rtb_whitted.cu -- the reference's second integrator, cast_ray (raytracer.c:556-641): Whitted
 * style ray tracing with one point light, Phong shading, a shadow ray, mirror reflection and
 * "refraction".  Upstream it is compiled out (`#if 1` at raytracer.c:207 selects trace_path);
 * here it is a run-time choice (rtb_render_desc.integrator = RTB_INTEGRATOR_WHITTED).
 *
 * cast_ray draws no random numbers, so apart from the pixel jitter the result is a pure function
 * of the ray.  Everything is IEEE double in the reference's operation order without FMA
 * contraction (the __d*_rn intrinsics), and the recursion is evaluated post-order with an
 * explicit frame stack, so a colour is built by the same sequence of operations as upstream:
 * GPU and reference agree to the last bit except where libm and the CUDA math library differ
 * in pow()/atan2()/fmod() (a few ulp).
 *
 * Quirks kept (SURVEY.md 8.1 and 8f N4):
 *   - the shadow test is intersect(&light_ray, ..., NULL): ANY sphere along the unbounded ray
 *     towards the light, also beyond it (raytracer.c:571) -- inside the closed room of the
 *     default scene everything is "in shadow";
 *   - refract(d, n, 1.0) returns d (quirk Q3): the refracted ray continues straight on;
 *   - a depth cut and a miss both return BACKGROUND (raytracer.c:561-564);
 *   - with both M_REFLECTION and M_REFRACTION set, kr of the reflection is overwritten by the
 *     Fresnel term (raytracer.c:611,622);
 *   - the checker uses M = 10 here (raytracer.c:584), not 100000.
 */
#include "rtb_path.cuh"

#define WH_MAX_DEPTH 15 /* frames of the explicit recursion stack: depth 0 .. max_depth + 1 */

struct WhFrame
{
  d3 surface, refl;
  d3 point, dir_in, normal;
  double kr, kt;
  unsigned flags;
  int stage; /* 0: before the reflection child, 1: before the refraction child, 2: refraction child running */
};

__device__ __forceinline__ d3 d3_mul(const d3 &a, const d3 &b)
{
  return d3_make(__dmul_rn(a.x, b.x), __dmul_rn(a.y, b.y), __dmul_rn(a.z, b.z));
}

/* cast_ray(ray, objects, nobj, 0); `rays` counts the calls (ray_count++, raytracer.c:558) */
__device__ d3 whitted_cast(const SceneView &sv, const d3 &o0, const d3 &d0, int max_depth, unsigned long long &rays)
{
  const double bg = 10 / 255.0; /* RGB(10, 10, 10), raytracer.h:46 */
  const d3 BACKGROUND = d3_make(bg, bg, bg);
  const d3 ZERO = d3_make(0 / 255.0, 0 / 255.0, 0 / 255.0);
  WhFrame frames[WH_MAX_DEPTH + 2];
  int sp = 0;        /* frames in use = depth of the pending call */
  d3 o = o0, d = d0; /* arguments of the pending call */
  d3 ret = ZERO;     /* value returned by the call that just finished */
  enum { PH_CALL, PH_RETURN, PH_ADVANCE };
  int phase = PH_CALL;

  while (true)
  {
    if (phase == PH_CALL)
    {
      /* ---- cast_ray(&{o, d}, ..., depth = sp) up to the recursive calls ---- */
      rays++;
      HitRec best;
      if (sp > max_depth || !nearest_hit(sv, o, d, best))
      {
        ret = BACKGROUND;
        phase = PH_RETURN;
        continue;
      }
      int slot_obj;
      {
        const float4 *rec = best.slot >= 0 ? sv.prims + 3 * best.slot : sv.big + 3 * (~best.slot);
        slot_obj = (int)(__float_as_uint(__ldg(rec + 2).z) & 0x7FFFFFFFu);
      }
      const unsigned flags = __float_as_uint(__ldg(sv.mats + 2 * slot_obj + 1).w);
      Surface s = surface_at(sv, o, d, best, (flags & RT_M_CHECKERED) != 0);

      const d3 light_pos = d3_make(2, 7, 2);
      const d3 light_color = d3_make(1, 1, 1);
      const d3 light_dir = d3_normalize(d3_sub(light_pos, s.point));
      HitRec shadow;
      const bool in_shadow = nearest_hit(sv, s.point, light_dir, shadow);

      d3 object_color = d3_make(sv.colors[3 * slot_obj + 0], sv.colors[3 * slot_obj + 1], sv.colors[3 * slot_obj + 2]);
      const double ka = 0.25, kd = 0.5, ks = 0.8, alpha = 10.0;
      if (flags & RT_M_CHECKERED)
        object_color = checker_color(object_color, s.u, s.v, 10);

      const d3 ambient = d3_scale(light_color, ka);
      const double ndl = d3_dot(s.normal, light_dir);
      const d3 diffuse = d3_scale(light_color, __dmul_rn(kd, (0.0 > ndl) ? 0.0 : ndl)); /* MAX(0.0, x) */
      const d3 reflected = reflect_dir(light_dir, s.normal);
      const d3 view_dir = d3_normalize(d3_sub(s.point, o));
      const double vdr = d3_dot(view_dir, reflected);
      const d3 specular = d3_scale(light_color, __dmul_rn(ks, pow((vdr > 0.0) ? vdr : 0.0, alpha))); /* MAX(x, 0.0) */
      const d3 lit = d3_scale(d3_add(specular, diffuse), in_shadow ? 0.0 : 1.0);
      WhFrame &f = frames[sp];
      f.surface = d3_mul(d3_add(ambient, lit), object_color);
      f.refl = ZERO;
      f.point = s.point;
      f.dir_in = d;
      f.normal = s.normal;
      f.kr = 0;
      f.kt = 0;
      f.flags = flags;
      f.stage = 0;
      sp++;
      phase = PH_ADVANCE;
      continue;
    }
    if (phase == PH_RETURN)
    {
      /* ---- a call returned `ret` to the frame on top, or to the caller ---- */
      if (sp == 0)
        return ret;
      WhFrame &f = frames[sp - 1];
      if (f.stage == 1)
      {
        f.refl = ret; /* reflection = cast_ray(...) */
        phase = PH_ADVANCE;
        continue;
      }
      /* stage 2: refraction = cast_ray(...); combine (raytracer.c:630-640) */
      d3 out = d3_add(ZERO, f.surface);
      out = d3_add(out, d3_add(d3_scale(f.refl, f.kr), d3_scale(ret, f.kt)));
      ret = out;
      sp--;
      continue; /* still PH_RETURN */
    }
    /* ---- PH_ADVANCE: the rest of cast_ray for the frame on top ---- */
    WhFrame &f = frames[sp - 1];
    if (f.stage == 0)
    {
      f.stage = 1;
      if (f.flags & RT_M_REFLECTION)
      {
        f.kr = 1.0;
        o = f.point;
        d = d3_normalize(reflect_dir(f.dir_in, f.normal));
        phase = PH_CALL;
        continue;
      }
    }
    /* stage 1 */
    f.stage = 2;
    if (f.flags & RT_M_REFRACTION)
    {
      const double transparency = 0.5;
      const double facing = -d3_dot(f.dir_in, f.normal);
      const double fresnel = __dadd_rn(__dmul_rn(1.0, 0.1), __dmul_rn(pow(__dsub_rn(1.0, facing), 3.0), __dsub_rn(1.0, 0.1)));
      f.kr = fresnel;
      f.kt = __dmul_rn(__dsub_rn(1.0, fresnel), transparency);
      /* refract(d, n, 1.0): cosi == 1, eta == 1, k == 1 -> In*1 + (-N)*(1*1 - sqrtf(1)) */
      const d3 nn = d3_scale(f.normal, -1.0);
      const double w = __dsub_rn(__dmul_rn(1.0, 1.0), (double)sqrtf(1.0f));
      o = f.point;
      d = d3_normalize(d3_add(d3_scale(f.dir_in, 1.0), d3_scale(nn, w)));
      phase = PH_CALL;
      continue;
    }
    /* no refraction child: refraction = ZERO_VECTOR, kt = 0 */
    d3 out = d3_add(ZERO, f.surface);
    out = d3_add(out, d3_add(d3_scale(f.refl, f.kr), d3_scale(ZERO, f.kt)));
    ret = out;
    sp--;
    phase = PH_RETURN;
  }
}

/* one thread per (plane, pixel): sum over the plane's samples, jitter as in path_begin (same Philox words, so the
 * primary rays are those of the path tracer).  Planes = contiguous sample sub-ranges, summed in order by the
 * caller (k_sum_planes): small frames still fill the GPU (C1 is 57 600 pixels, a B200 holds 300 000 threads). */
__global__ void __launch_bounds__(64) k_whitted_render(const __grid_constant__ RenderArgs A)
{
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int n_px = A.width * A.height;
  const int plane = (int)(tid / n_px);
  const int pix = (int)(tid - (long long)plane * n_px);
  unsigned long long rays = 0, paths = 0;
  if (plane < A.splits)
  {
    const int x = pix % A.width, y = pix / A.width;
    const int s0 = A.s_begin + plane * A.chunk, s1 = min(A.s_end, s0 + A.chunk);
    d3 sum = d3_make(0, 0, 0);
    for (int s = s0; s < s1; s++)
    {
      PathState st;
      path_begin(A, st, x, y, (unsigned)pix, (unsigned)s);
      const d3 c = whitted_cast(A.sv, st.o, st.d, A.max_depth, rays);
      sum = d3_add(sum, c);
      paths++;
    }
    float *out = A.out + (size_t)plane * 3 * n_px;
    out[3 * (size_t)pix + 0] = (float)sum.x;
    out[3 * (size_t)pix + 1] = (float)sum.y;
    out[3 * (size_t)pix + 2] = (float)sum.z;
  }
  const int lane = threadIdx.x & 31;
  for (int off = 16; off > 0; off >>= 1)
  {
    rays += __shfl_xor_sync(0xFFFFFFFFu, rays, off);
    paths += __shfl_xor_sync(0xFFFFFFFFu, paths, off);
  }
  if (lane == 0)
  {
    atomicAdd(&A.counters[0], rays);
    atomicAdd(&A.counters[4], paths);
  }
}

__global__ void __launch_bounds__(64) k_cast_rays(const __grid_constant__ SceneView sv, const double *__restrict__ rays6,
                                                  size_t n, int max_depth, double *__restrict__ rgb,
                                                  unsigned long long *__restrict__ ray_counts)
{
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n)
    return;
  const d3 o = d3_make(rays6[6 * i + 0], rays6[6 * i + 1], rays6[6 * i + 2]);
  const d3 d = d3_make(rays6[6 * i + 3], rays6[6 * i + 4], rays6[6 * i + 5]);
  unsigned long long rays = 0;
  const d3 c = whitted_cast(sv, o, d, max_depth, rays);
  rgb[3 * i + 0] = c.x; rgb[3 * i + 1] = c.y; rgb[3 * i + 2] = c.z;
  if (ray_counts)
    ray_counts[i] = rays;
}

int whitted_render(rtb_scene *scene, RenderArgs &A, cudaStream_t stream, unsigned long long &launches)
{
  if (A.max_depth > WH_MAX_DEPTH)
  {
    rtb_set_error("Whitted integrator: max_depth must be <= 15");
    return RTB_EINVAL;
  }
  const size_t n_threads = (size_t)A.width * A.height * (size_t)A.splits;
  k_whitted_render<<<(unsigned)((n_threads + 63) / 64), 64, 0, stream>>>(A);
  RTB_CUDA(cudaGetLastError());
  (void)launches; /* counted by the caller together with the plane sum */
  (void)scene;
  return RTB_OK;
}

template <typename T>
struct WhDev
{
  T *p = nullptr;
  ~WhDev() { if (p) cudaFree(p); }
};

extern "C" int rtb_cast_rays(rtb_scene *scene, const double *rays6, size_t n_rays, int max_depth, double *rgb,
                             unsigned long long *ray_counts)
{
  if (!scene || (n_rays && (!rays6 || !rgb)) || max_depth < 0 || max_depth > WH_MAX_DEPTH)
  {
    rtb_set_error("rtb_cast_rays: bad argument (max_depth 0..15)");
    return RTB_EINVAL;
  }
  if (n_rays == 0)
    return RTB_OK;
  RTB_CUDA(cudaSetDevice(scene->device));
  WhDev<double> d_rays, d_rgb;
  WhDev<unsigned long long> d_cnt;
  RTB_CUDA(cudaMalloc(&d_rays.p, sizeof(double) * 6 * n_rays));
  RTB_CUDA(cudaMalloc(&d_rgb.p, sizeof(double) * 3 * n_rays));
  RTB_CUDA(cudaMalloc(&d_cnt.p, sizeof(unsigned long long) * n_rays));
  RTB_CUDA(cudaMemcpy(d_rays.p, rays6, sizeof(double) * 6 * n_rays, cudaMemcpyHostToDevice));
  k_cast_rays<<<(unsigned)((n_rays + 63) / 64), 64>>>(scene->view, d_rays.p, n_rays, max_depth, d_rgb.p, d_cnt.p);
  RTB_CUDA(cudaGetLastError());
  RTB_CUDA(cudaDeviceSynchronize());
  RTB_CUDA(cudaMemcpy(rgb, d_rgb.p, sizeof(double) * 3 * n_rays, cudaMemcpyDeviceToHost));
  if (ray_counts)
    RTB_CUDA(cudaMemcpy(ray_counts, d_cnt.p, sizeof(unsigned long long) * n_rays, cudaMemcpyDeviceToHost));
  return RTB_OK;
}
