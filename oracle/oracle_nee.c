/*
 * oracle_nee.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * The CPU restatement of RTB_INTEGRATOR_PATH_NEE (next-event estimation, DESIGN.md section 4.7), the checker of the
 * GPU's NEE kernels.  It is built as its own library (liboracle_nee.so, __graft_entry__.build()) from oracle.c itself,
 * included below unchanged, so trace() and everything NEE shares with it -- nearest hit, hemisphere sampling, the
 * Philox layout, the camera -- are the restatement's own code, and the pinned oracle stays exactly as it is.
 * Same build flags as oracle.c (-std=c99 -O3 -ffp-contract=off): bit-exactness depends on them.
 */
#include "oracle.c"

/* ---- next-event estimation (RTB_INTEGRATOR_PATH_NEE, DESIGN.md section 4.7) ----------------------------------------
 * trace() with one light sample per diffuse vertex, combined with the hemisphere ray by the balance heuristic.  The
 * light list, the selection CDF, the cone and disk sampling and the MIS weights are those of the GPU
 * (raytracer.c_b200/csrc/rtb_path.cuh), operation for operation, so every light sample -- its light, its direction, and
 * whether it is taken -- is the GPU's bit for bit.  Light samples use Philox block 0x80000000 + k of the vertex. */

typedef struct
{
  double cx, cy, cz, r;
  double P, cdf;
  vec3 emission;
  int obj;
} NeeLight;

typedef struct
{
  NeeLight *l;
  int n;
  int *light_of; /* object -> light, -1 */
} NeeList;

typedef struct /* one thread's light list and shadow-ray counts */
{
  const NeeList *N;
  long long shadow_rays, shadow_hits;
} NeeCtx;

#define NEE_PHILOX_BLOCK 0x80000000u
#define NEE_DISK_TRIES 64

/* every sphere object whose (float) emission is nonzero, in object order; P_j from the running sum of
 * (|e.r| + |e.g| + |e.b|) r^2 of the float emission, as the GPU's light list is built */
static void nee_build(NeeList *N, const SceneObject *objects, size_t n)
{
  N->l = (NeeLight *)calloc(n > 0 ? n : 1, sizeof(NeeLight));
  N->light_of = (int *)malloc(sizeof(int) * (n > 0 ? n : 1));
  if (!N->l || !N->light_of)
  {
    fprintf(stderr, "oracle: out of memory\n");
    exit(EXIT_FAILURE);
  }
  N->n = 0;
  double total = 0.0;
  for (size_t i = 0; i < n; i++)
  {
    N->light_of[i] = -1;
    if (objects[i].type != GEOMETRY_SPHERE)
      continue;
    const vec3 e = objects[i].material.emission;
    const float ex = (float)e.x, ey = (float)e.y, ez = (float)e.z;
    if (ex == 0.0f && ey == 0.0f && ez == 0.0f)
      continue;
    const Sphere *sp = objects[i].geometry.sphere;
    NeeLight *L = &N->l[N->n];
    L->cx = sp->center.x; L->cy = sp->center.y; L->cz = sp->center.z; L->r = sp->radius;
    L->emission = e;
    L->obj = (int)i;
    const double w = ((double)fabsf(ex) + (double)fabsf(ey) + (double)fabsf(ez)) * L->r * L->r;
    total += w;
    L->cdf = total;
    N->light_of[i] = N->n++;
  }
  double prev = 0.0;
  for (int k = 0; k < N->n; k++)
  {
    N->l[k].cdf = N->l[k].cdf / total;
    N->l[k].P = N->l[k].cdf - prev;
    prev = N->l[k].cdf;
  }
}

static void nee_free(NeeList *N)
{
  free(N->l);
  free(N->light_of);
}

/* 1 - cos(theta_max) of L seen from x, 0 when x is inside or on the sphere */
static double nee_one_minus_cos(const NeeLight *L, vec3 x, vec3 *axis)
{
  vec3 v = { L->cx - x.x, L->cy - x.y, L->cz - x.z };
  double d2 = vec3_dot(v, v);
  double r2 = L->r * L->r;
  if (!(d2 > r2))
    return 0.0;
  double s2 = r2 / d2;
  double cmax = sqrt(1.0 - s2);
  if (axis)
    *axis = vec3_normalize(v);
  return s2 / (1.0 + cmax);
}

static double nee_bsdf_weight(const NeeLight *L, vec3 x_prev)
{
  double omc = nee_one_minus_cos(L, x_prev, NULL);
  if (!(omc > 0.0))
    return 1.0;
  return 1.0 / (1.0 + L->P / omc);
}

static bool nee_sample(const NeeList *N, const Rng *g, uint32_t bounce_word, vec3 x, vec3 normal, int *j_out,
                       vec3 *dir_out, double *g_out)
{
  uint32_t w[4];
  keyed_block(g, bounce_word, NEE_PHILOX_BLOCK, w);
  double u = uniform_from_word(w[0]);
  int lo = 0, hi = N->n - 1;
  while (lo < hi)
  {
    int mid = (lo + hi) >> 1;
    if (u < N->l[mid].cdf)
      hi = mid;
    else
      lo = mid + 1;
  }
  *j_out = lo;
  const NeeLight *L = &N->l[lo];
  vec3 axis;
  double omc = nee_one_minus_cos(L, x, &axis);
  if (!(omc > 0.0))
    return false;
  double um = uniform_from_word(w[1]) * omc;
  double cos_t = 1.0 - um;
  double sin_t = sqrt(um * (2.0 - um));
  double a = uniform_from_word(w[2]) * 2.0 - 1.0, b = uniform_from_word(w[3]) * 2.0 - 1.0;
  double q = a * a + b * b;
  for (uint32_t k = 1; !(q <= 1.0 && q > 0.0); k++)
  {
    if (k >= NEE_DISK_TRIES)
    {
      a = 1.0; b = 0.0; q = 1.0;
      break;
    }
    uint32_t r[4];
    keyed_block(g, bounce_word, NEE_PHILOX_BLOCK + k, r);
    a = uniform_from_word(r[0]) * 2.0 - 1.0;
    b = uniform_from_word(r[1]) * 2.0 - 1.0;
    q = a * a + b * b;
  }
  double inv = 1.0 / sqrt(q);
  double cphi = a * inv, sphi = b * inv;
  double sg = axis.z >= 0.0 ? 1.0 : -1.0;
  double fa = -1.0 / (sg + axis.z);
  double fb = axis.x * axis.y * fa;
  vec3 t1 = { 1.0 + sg * axis.x * axis.x * fa, sg * fb, -(sg * axis.x) };
  vec3 t2 = { fb, sg + axis.y * axis.y * fa, -axis.y };
  vec3 v = vec3_add(vec3_add(vec3_scalar_mult(t1, sin_t * cphi), vec3_scalar_mult(t2, sin_t * sphi)),
                    vec3_scalar_mult(axis, cos_t));
  vec3 dir = vec3_normalize(v);
  double c = vec3_dot(dir, normal);
  if (!(c > 0.0))
    return false;
  *dir_out = dir;
  *g_out = c / (1.0 + L->P / omc);
  return true;
}

/* trace() with next-event estimation; from_diffuse: `ray` left a diffuse vertex (its emission gets the hemisphere
 * side's MIS weight when it reaches a sampled light) */
static vec3 trace_nee(NeeCtx *C, Tracer *T, Rng *g, const Ray *ray, int depth, uint32_t branch, int from_diffuse)
{
  const NeeList *N = C->N;
  g->rays++;
  const vec3 background = BACKGROUND;
  if (depth > T->max_depth)
    return background;
  Nearest hit = nearest_hit(ray, T->objects, T->n, &g->tests);
  if (!hit.found)
    return background;

  const Material *m = &T->objects[hit.object_id].material;
  vec3 albedo = m->color;
  vec3 emission = m->emission;
  if (from_diffuse && N->light_of[hit.object_id] >= 0)
    emission = vec3_scalar_mult(emission, nee_bsdf_weight(&N->l[N->light_of[hit.object_id]], ray->origin));

  VertexRng vr;
  memset(&vr, 0, sizeof(vr));
  double prob = MAX(albedo.x, MAX(albedo.y, albedo.z));
  if (rng_rr(g, &vr, depth, branch) < prob)
    albedo = vec3_scalar_mult(albedo, 1 / prob);
  else
    return emission;

  uint flags = m->flags;
  if (flags & M_CHECKERED)
    albedo = checker(albedo, hit.u, hit.v, 100000);

  Ray R;
  R.origin = hit.point;
  vec3 radiance;

  if (flags & M_REFRACTION)
  {
    double transparency = 1.0;
    double facing = -vec3_dot(ray->direction, hit.normal);
    double fresnel = mix(pow(1 - facing, 3), 1, 0.1);
    double kr = fresnel;
    double kt = (1 - fresnel) * transparency;
    vec3 dir_t = vec3_normalize(refract_dir(vec3_scalar_mult(ray->direction, -1), hit.normal, 1.0));
    vec3 dir_r = vec3_normalize(reflect_dir(vec3_scalar_mult(ray->direction, 1), hit.normal));
    if (T->dielectric_mode == ORACLE_DIELECTRIC_SPLIT)
    {
      R.direction = dir_t;
      vec3 refraction = trace_nee(C, T, g, &R, depth + 1, (branch << 1) | 0u, 0);
      R.direction = dir_r;
      vec3 reflection = trace_nee(C, T, g, &R, depth + 1, (branch << 1) | 1u, 0);
      radiance = vec3_add(vec3_scalar_mult(refraction, kt), vec3_scalar_mult(reflection, kr));
    }
    else
    {
      double p = kr < 0.05 ? 0.05 : (kr > 0.95 ? 0.95 : kr);
      if (rng_choice(g, &vr) < p)
      {
        R.direction = dir_r;
        radiance = vec3_scalar_mult(trace_nee(C, T, g, &R, depth + 1, branch, 0), kr / p);
      }
      else
      {
        R.direction = dir_t;
        radiance = vec3_scalar_mult(trace_nee(C, T, g, &R, depth + 1, branch, 0), kt / (1 - p));
      }
    }
  }
  else if (flags & M_REFLECTION)
  {
    R.direction = reflect_dir(ray->direction, hit.normal);
    radiance = trace_nee(C, T, g, &R, depth + 1, branch, 0);
  }
  else
  {
    R.direction = hemisphere_dir(g, &vr, hit.normal);
    vec3 direct = { 0, 0, 0 };
    int j;
    vec3 sdir;
    double gw;
    /* no light sample where the continuation is depth-cut: the reference returns background there, not the light */
    if (N->n > 0 && depth + 1 <= T->max_depth && nee_sample(N, g, vr.bounce_word, hit.point, hit.normal, &j, &sdir, &gw))
    {
      C->shadow_rays++;
      Ray S = { hit.point, sdir };
      Nearest sh = nearest_hit(&S, T->objects, T->n, &g->tests);
      if (sh.found && (int)sh.object_id == N->l[j].obj)
      {
        C->shadow_hits++;
        direct = vec3_scalar_mult(N->l[j].emission, gw);
      }
    }
    double cos_theta = vec3_dot(R.direction, hit.normal);
    radiance = vec3_add(direct, vec3_scalar_mult(trace_nee(C, T, g, &R, depth + 1, branch, 1), cos_theta));
  }
  return vec3_add(emission, vec3_mult(albedo, radiance));
}

/* oracle_render_sum with the NEE estimator: per-pixel sums over samples [sample_offset, sample_offset + samples) in
 * double, keyed Philox (p->rng_mode is not consulted), p->integrator ignored.  counters: [0] rays (trace_path
 * invocations), [1] primitive tests, [2] shadow rays, [3] shadow rays whose nearest hit was their light. */
void oracle_render_sum_nee(double *sum_rgb, const SceneObject *objects, size_t n, const Camera *camera, int width,
                           int height, int samples, const OracleParams *p, long long *counters)
{
  OracleParams q = *p;
  q.rng_mode = ORACLE_RNG_PHILOX;
  long long rays = 0, tests = 0, shadow_rays = 0, shadow_hits = 0;
  int threads = q.threads > 0 ? q.threads : 1;
  NeeList nee;
  nee_build(&nee, objects, n);

#pragma omp parallel for num_threads(threads) schedule(dynamic, 1) reduction(+ : rays, tests, shadow_rays, shadow_hits)
  for (int y = 0; y < height; y++)
  {
    Rng g;
    rng_setup(&g, &q);
    Tracer T;
    tracer_setup(&T, objects, n, &q);
    NeeCtx C = { &nee, 0, 0 };
    for (int x = 0; x < width; x++)
    {
      vec3 pixel = { 0, 0, 0 };
      for (int s = 0; s < samples; s++)
      {
        g.pixel = (uint32_t)(y * width + x);
        g.sample = (uint32_t)(q.sample_offset + s);
        double j1, j2;
        rng_jitter(&g, &j1, &j2);
        double u = (double)(x + j1) / ((double)width - 1.0);
        double v = (double)(y + j2) / ((double)height - 1.0);
        Ray ray = camera_ray(camera, u, v);
        pixel = vec3_add(pixel, trace_nee(&C, &T, &g, &ray, 0, 1u, 0));
      }
      double *o = sum_rgb + 3 * ((size_t)y * width + x);
      o[0] = pixel.x; o[1] = pixel.y; o[2] = pixel.z;
    }
    rays += g.rays;
    tests += g.tests;
    shadow_rays += C.shadow_rays;
    shadow_hits += C.shadow_hits;
  }
  if (counters)
  {
    counters[0] = rays;
    counters[1] = tests;
    counters[2] = shadow_rays;
    counters[3] = shadow_hits;
  }
  nee_free(&nee);
}
