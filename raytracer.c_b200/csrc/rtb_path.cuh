/*
 * rtb_path.cuh -- one vertex of trace_path (raytracer.c:482-554) and the camera sample that
 * starts a path (raytracer.c:203-209, :375-384), shared by the megakernels (rtb_render.cu)
 * and the wavefront kernels (rtb_wavefront.cu).  Every kernel variant calls the very same
 * path_begin / path_shade, which is what makes their sums bit-identical.
 */
#ifndef RTB_PATH_CUH
#define RTB_PATH_CUH

#include "rtb_device.cuh"
struct RenderArgs
{
  SceneView sv;
  CameraView cam;
  int width, height, tiles_x, n_tiles;
  int s_begin, s_end, chunk, splits;
  int max_depth, dielectric_mode;
  int suspend_lanes; /* k_render_pw: suspend the walk when fewer lanes than this are walking */
  int plane_base;    /* wavefront: first plane of the group this launch works on (two groups run on two streams) */
  uint2 key;
  float *out; /* [splits][height*width*3] */
  unsigned long long *counters;
};

struct PathState
{
  d3 o, d;
  float tr, tg, tb; /* throughput */
  int depth;
  bool alive;
  unsigned branch; /* 1 on the camera ray; a dielectric vertex of the SPLIT estimator gives its children 2b and 2b+1 */
};

struct PathCounters
{
  unsigned rays, rays_hit;
};

#ifndef RTB_SMEM_STACK
#define RTB_SMEM_STACK 8 /* stack entries per thread kept in shared memory (default kernel) */
#endif

#define RT_BACKGROUND (10.0f / 255.0f) /* raytracer.h:46, also returned on a depth cut (quirk Q2) */

/* ---- next-event estimation (RTB_INTEGRATOR_PATH_NEE, DESIGN.md section 4.7) ------------------------------------------
 * Light list: every sphere object with nonzero emission, in object order, built on the first NEE render of a scene
 * (rtb_wavefront.cu, nee_lights).  Light j is chosen with probability P_j = cdf[j] - cdf[j-1], cdf the normalised
 * running sum of (|e.r| + |e.g| + |e.b|) r^2 in double (e the float emission the shade kernel adds).  Every decision
 * is made in correctly rounded double arithmetic without transcendental functions, so the oracle (oracle/oracle_nee.c)
 * reproduces each light sample bit for bit. */
struct NeeLight /* 64 bytes */
{
  double cx, cy, cz, r; /* the sphere, exactly as the caller gave it */
  double P, cdf;        /* selection probability and the running sum it is drawn with */
  float er, eg, eb;     /* emission */
  int obj;              /* object index */
};

struct NeeView
{
  const NeeLight *lights;
  const int *light_of; /* object index -> light index, -1 for objects that are not sampled */
  int n_lights;
};

/* what one vertex of the NEE estimator takes in and gives out besides PathState */
struct NeeIO
{
  bool from_diffuse; /* in: the incoming ray left a diffuse vertex (its emission gets the BSDF-side MIS weight) */
  bool diffuse_out;  /* out: the continuation ray leaves a diffuse vertex */
  bool shadow;       /* out: a shadow ray towards light `light` along `sd` from the vertex */
  int light;
  d3 sd;
  float pr, pg, pb; /* its payload: tp' * cos / (1 + 2 pi P_j p_j); the emission is applied when it reaches the light */
};

#define NEE_PHILOX_BLOCK 0x80000000u /* light samples: block 0x80000000 + k of the vertex (hemisphere tries use 1..98) */
#define NEE_DISK_TRIES 64

/* 1 - cos(theta_max) of light L seen from x, or 0 when x is inside or on the sphere (no light sample there).
 * 2 pi P p = P / (1 - cos theta_max): the cone pdf is 1 / (2 pi (1 - cos theta_max)). */
__device__ __forceinline__ double nee_one_minus_cos(const NeeLight &L, const d3 &x, d3 *axis)
{
  const d3 v = d3_make(__dsub_rn(L.cx, x.x), __dsub_rn(L.cy, x.y), __dsub_rn(L.cz, x.z));
  const double d2 = d3_dot(v, v);
  const double r2 = __dmul_rn(L.r, L.r);
  if (!(d2 > r2))
    return 0.0;
  const double s2 = __ddiv_rn(r2, d2);                    /* sin^2 theta_max */
  const double cmax = __dsqrt_rn(__dsub_rn(1.0, s2));
  if (axis)
    *axis = d3_normalize(v);
  return __ddiv_rn(s2, __dadd_rn(1.0, cmax)); /* 1 - cos theta_max without cancellation */
}

/* weight of emission reached by a hemisphere ray from x_prev on light L: 1 / (1 + 2 pi P p(x_prev)) */
__device__ __forceinline__ float nee_bsdf_weight(const NeeLight &L, const d3 &x_prev)
{
  const double omc = nee_one_minus_cos(L, x_prev, nullptr);
  if (!(omc > 0.0))
    return 1.0f;
  return (float)__ddiv_rn(1.0, __dadd_rn(1.0, __ddiv_rn(L.P, omc)));
}

/* the light sample of a diffuse vertex at x with normal n: light choice, uniform direction in its cone; false when
 * there is none (x inside or on the sphere, or the direction below the surface).  *g = cos / (1 + P / (1 - cos max)). */
__device__ __forceinline__ bool nee_sample(const NeeView &nv, const uint2 key, unsigned pixel, unsigned sample,
                                           unsigned bounce_word, const d3 &x, const d3 &n, int &j, d3 &dir, double &g)
{
  const uint4 w = philox4x32_10(make_uint4(pixel, sample, bounce_word, NEE_PHILOX_BLOCK), key);
  const double u = uniform31(w.x);
  int lo = 0, hi = nv.n_lights - 1;
  while (lo < hi)
  {
    const int mid = (lo + hi) >> 1;
    if (u < __ldg(&nv.lights[mid].cdf))
      hi = mid;
    else
      lo = mid + 1;
  }
  j = lo;
  const NeeLight &L = nv.lights[j];
  d3 axis;
  const double omc = nee_one_minus_cos(L, x, &axis);
  if (!(omc > 0.0))
    return false;
  /* cos theta uniform in [cos theta_max, 1]: 1 - cos theta = xi (1 - cos theta_max) */
  const double um = __dmul_rn(uniform31(w.y), omc);
  const double cos_t = __dsub_rn(1.0, um);
  const double sin_t = __dsqrt_rn(__dmul_rn(um, __dsub_rn(2.0, um)));
  /* (cos phi, sin phi): a point of the unit disk by rejection, normalised */
  double a = __dsub_rn(__dmul_rn(uniform31(w.z), 2.0), 1.0), b = __dsub_rn(__dmul_rn(uniform31(w.w), 2.0), 1.0);
  double q = __dadd_rn(__dmul_rn(a, a), __dmul_rn(b, b));
  for (unsigned k = 1; !(q <= 1.0 && q > 0.0); k++)
  {
    if (k >= NEE_DISK_TRIES)
    {
      a = 1.0; b = 0.0; q = 1.0;
      break;
    }
    const uint4 r = philox4x32_10(make_uint4(pixel, sample, bounce_word, NEE_PHILOX_BLOCK + k), key);
    a = __dsub_rn(__dmul_rn(uniform31(r.x), 2.0), 1.0);
    b = __dsub_rn(__dmul_rn(uniform31(r.y), 2.0), 1.0);
    q = __dadd_rn(__dmul_rn(a, a), __dmul_rn(b, b));
  }
  const double inv = __ddiv_rn(1.0, __dsqrt_rn(q));
  const double cphi = __dmul_rn(a, inv), sphi = __dmul_rn(b, inv);
  /* orthonormal frame around the axis (Duff et al. 2017) */
  const double sg = axis.z >= 0.0 ? 1.0 : -1.0;
  const double fa = __ddiv_rn(-1.0, __dadd_rn(sg, axis.z));
  const double fb = __dmul_rn(__dmul_rn(axis.x, axis.y), fa);
  const d3 t1 = d3_make(__dadd_rn(1.0, __dmul_rn(__dmul_rn(__dmul_rn(sg, axis.x), axis.x), fa)), __dmul_rn(sg, fb),
                        -__dmul_rn(sg, axis.x));
  const d3 t2 = d3_make(fb, __dadd_rn(sg, __dmul_rn(__dmul_rn(axis.y, axis.y), fa)), -axis.y);
  const d3 v = d3_add(d3_add(d3_scale(t1, __dmul_rn(sin_t, cphi)), d3_scale(t2, __dmul_rn(sin_t, sphi))),
                      d3_scale(axis, cos_t));
  dir = d3_normalize(v);
  const double c = d3_dot(dir, n);
  if (!(c > 0.0))
    return false;
  g = __ddiv_rn(c, __dadd_rn(1.0, __ddiv_rn(L.P, omc)));
  return true;
}

__device__ __forceinline__ void path_begin(const RenderArgs &A, PathState &st, int x, int y, unsigned pixel, unsigned sample)
{
  /* jitter: u = (x + xi1)/(W-1), v = (y + xi2)/(H-1), raytracer.c:203-204 */
  uint4 w = philox4x32_10(make_uint4(pixel, sample, 0xFFFFFFFFu, 0u), A.key);
  double u = __ddiv_rn(__dadd_rn((double)x, uniform31(w.x)), __dsub_rn((double)A.width, 1.0));
  double v = __ddiv_rn(__dadd_rn((double)y, uniform31(w.y)), __dsub_rn((double)A.height, 1.0));
  camera_ray(A.cam, u, v, st.o, st.d);
  st.tr = st.tg = st.tb = 1.0f;
  st.depth = 0;
  st.alive = true;
  st.branch = 1u;
}

/* One vertex of the path: the body of trace_path after the scene query.
 * `sum` accumulates throughput * (emission | background).
 * SPLIT: the reference's own dielectric estimator (raytracer.c:522-529): BOTH children are traced, the
 * retro-"refraction" ray with weight kt and the reflection with weight kr.  `st` continues as the first
 * (refraction, evaluated first upstream), `*second` as the other; second->alive says whether it exists. */
/* NEE: the next-event-estimation form (RTB_INTEGRATOR_PATH_NEE): the same path rays and draws; emission reached from a
 * diffuse vertex is MIS-weighted, and a diffuse vertex that is not depth-cut emits one shadow ray (*io). */
template <bool SPLIT = false, bool NEE = false>
__device__ __forceinline__ void path_shade(const RenderArgs &A, PathState &st, const HitRec &best, unsigned pixel,
                                           unsigned sample, float &sr, float &sg, float &sb, PathCounters &pc,
                                           Surface *surf_out, PathState *second = nullptr, const NeeView *nv = nullptr,
                                           NeeIO *io = nullptr)
{
  if constexpr (NEE)
  {
    io->diffuse_out = false;
    io->shadow = false;
  }
  if (SPLIT)
    second->alive = false;
  if (best.t >= 1e300)
  {
    sr += st.tr * RT_BACKGROUND; sg += st.tg * RT_BACKGROUND; sb += st.tb * RT_BACKGROUND;
    st.alive = false;
    return;
  }
  /* material first: uv is only needed for checkered objects */
  int slot_obj;
  {
    const float4 *rec = best.slot >= 0 ? A.sv.prims + 3 * best.slot : A.sv.big + 3 * (~best.slot);
    slot_obj = (int)(__float_as_uint(__ldg(rec + 2).z) & 0x7FFFFFFFu);
  }
  const float4 m0 = __ldg(A.sv.mats + 2 * slot_obj + 0);
  const float4 m1 = __ldg(A.sv.mats + 2 * slot_obj + 1);
  const unsigned flags = __float_as_uint(m1.w);
  Surface s = surface_at(A.sv, st.o, st.d, best, (flags & RT_M_CHECKERED) != 0);
  if (surf_out)
    *surf_out = s;

  /* emission is added whether or not the path survives (raytracer.c:502,553) */
  if constexpr (NEE)
  {
    /* the hemisphere side of the balance heuristic; weight 1 (the very same sum) for everything NEE cannot sample */
    float ew = 1.0f;
    if (io->from_diffuse)
    {
      const int j = __ldg(nv->light_of + slot_obj);
      if (j >= 0)
        ew = nee_bsdf_weight(nv->lights[j], st.o);
    }
    sr += (st.tr * ew) * m1.x; sg += (st.tg * ew) * m1.y; sb += (st.tb * ew) * m1.z;
  }
  else
  {
    sr += st.tr * m1.x; sg += st.tg * m1.y; sb += st.tb * m1.z;
  }

  /* Russian roulette, one draw per vertex (raytracer.c:497-502) */
  const unsigned bounce_word = (unsigned)st.depth | (st.branch << 8);
  uint4 w = philox4x32_10(make_uint4(pixel, sample, bounce_word, 0u), A.key);
  if ((w.x >> 1) >= __float_as_uint(m0.w))
  {
    st.alive = false;
    return;
  }
  st.tr *= m0.x; st.tg *= m0.y; st.tb *= m0.z; /* albedo / prob */
  if (flags & RT_M_CHECKERED)
  {
    float c = checker_factor(s.u, s.v, 100000.0); /* raytracer.c:508 */
    st.tr *= c; st.tg *= c; st.tb *= c;
  }

  if (flags & RT_M_REFRACTION)
  {
    /* raytracer.c:514-529.  refract(-d, n, 1.0) returns -d (quirk Q3), so the "refracted"
     * ray is the retro-ray normalize(-d); the reflected one is normalize(reflect(d, n)).
     * The reference traces both; here one is chosen with p = clamp(kr, .05, .95) and
     * weighted kr/p or kt/(1-p) -- the same expectation. */
    double facing = -d3_dot(st.d, s.normal);
    /* mix(pow(1 - facing, 3), 1, 0.1) (raytracer.c:518); x*x*x differs from libm pow(x, 3) by
     * at most 1 ulp, and only scales a colour weight (never geometry) */
    double omf = __dsub_rn(1.0, facing);
    double cube = __dmul_rn(__dmul_rn(omf, omf), omf);
    double fresnel = __dadd_rn(__dmul_rn(1.0, 0.1), __dmul_rn(cube, __dsub_rn(1.0, 0.1)));
    double kr = fresnel;
    double kt = __dmul_rn(__dsub_rn(1.0, fresnel), 1.0);
    double p = kr < 0.05 ? 0.05 : (kr > 0.95 ? 0.95 : kr);
    float wgt;
    if (SPLIT)
    {
      const d3 dir_in = st.d;
      *second = st;
      second->d = d3_normalize(reflect_dir(d3_scale(dir_in, 1.0), s.normal));
      const float wr = (float)kr;
      second->tr *= wr; second->tg *= wr; second->tb *= wr;
      second->branch = (st.branch << 1) | 1u;
      second->alive = true;
      st.d = d3_normalize(d3_scale(dir_in, -1.0));
      st.branch = st.branch << 1;
      wgt = (float)kt;
    }
    else if (uniform31(w.y) < p)
    {
      st.d = d3_normalize(reflect_dir(d3_scale(st.d, 1.0), s.normal));
      wgt = (float)__ddiv_rn(kr, p);
    }
    else
    {
      st.d = d3_normalize(d3_scale(st.d, -1.0));
      wgt = (float)__ddiv_rn(kt, __dsub_rn(1.0, p));
    }
    st.tr *= wgt; st.tg *= wgt; st.tb *= wgt;
  }
  else if (flags & RT_M_REFLECTION)
  {
    st.d = reflect_dir(st.d, s.normal); /* not renormalised (quirk Q8) */
  }
  else
  {
    /* uniform direction by cube rejection, flipped into the normal's hemisphere; weight
     * cos(theta), no pdf (raytracer.c:231-253,545-551; quirk Q5) */
    d3 p;
    unsigned k = 0;
    uint4 r = w;
    double px = uniform31(r.y), py = uniform31(r.z), pz = uniform31(r.w);
    while (true)
    {
      p = d3_make(__dadd_rn(__dmul_rn(px, 2.0), -1.0), __dadd_rn(__dmul_rn(py, 2.0), -1.0),
                  __dadd_rn(__dmul_rn(pz, 2.0), -1.0));
      /* vec3_length(p) > 1.0 (raytracer.c:236) without the square root, exactly: for the
       * correctly rounded sqrt, sqrt(x) > 1 <=> x > 1 + 2^-52 (sqrt(1 + 2^-52) = 1 + 2^-53 - ...
       * rounds to 1; sqrt(1 + 2^-51) = 1 + 2^-52 - ... rounds to 1 + 2^-52) */
      if (!(d3_dot(p, p) > 1.0000000000000002) || k >= 98u)
        break;
      k++;
      r = philox4x32_10(make_uint4(pixel, sample, bounce_word, k), A.key);
      px = uniform31(r.x); py = uniform31(r.y); pz = uniform31(r.z);
    }
    d3 dir = d3_normalize(p);
    if (d3_dot(dir, s.normal) < 0)
      dir = d3_scale(dir, -1.0);
    if constexpr (NEE)
    {
      if (nv->n_lights > 0 && st.depth + 1 <= A.max_depth)
      {
        double g;
        io->shadow = nee_sample(*nv, A.key, pixel, sample, bounce_word, s.point, s.normal, io->light, io->sd, g);
        if (io->shadow)
        {
          const float gf = (float)g;
          io->pr = st.tr * gf; io->pg = st.tg * gf; io->pb = st.tb * gf;
        }
      }
      io->diffuse_out = true;
    }
    float c = (float)d3_dot(dir, s.normal);
    st.d = dir;
    st.tr *= c; st.tg *= c; st.tb *= c;
  }
  st.o = s.point;
  st.depth++;
  if (SPLIT && second->alive)
  {
    second->o = s.point;
    second->depth = st.depth;
  }
  if (st.depth > A.max_depth)
  {
    /* the next trace_path call returns BACKGROUND without intersecting (raytracer.c:487) */
    pc.rays++;
    sr += st.tr * RT_BACKGROUND; sg += st.tg * RT_BACKGROUND; sb += st.tb * RT_BACKGROUND;
    st.alive = false;
    if (SPLIT && second->alive)
    {
      pc.rays++;
      sr += second->tr * RT_BACKGROUND; sg += second->tg * RT_BACKGROUND; sb += second->tb * RT_BACKGROUND;
      second->alive = false;
    }
  }
}

/* rtb_render.cu: the camera, frame, sample range, key and scene of a call (chunk, splits and out are the caller's) */
void fill_args(RenderArgs &A, const rtb_scene *scene, const double *camera12, const rtb_render_desc *desc);

/* rtb_wavefront.cu: render [A.s_begin, A.s_end) with the wavefront kernels into d_accum
 * (A.splits planes of A.chunk samples each must be set) */
int wf_render(rtb_scene *scene, RenderArgs &A, const rtb_render_desc *desc, float *d_accum, cudaStream_t stream,
              bool stats, unsigned long long &launches, float *phase_ms);

/* rtb_whitted.cu: the cast_ray integrator, one launch; writes A.splits planes to A.out (summed by the caller) */
int whitted_render(rtb_scene *scene, RenderArgs &A, cudaStream_t stream, unsigned long long &launches);

#endif /* RTB_PATH_CUH */
