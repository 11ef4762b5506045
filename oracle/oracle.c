/*
 * oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * A plain-C, IEEE-double CPU restatement of the reference path tracer's hot path
 * (/root/reference/raytracer.c:42-118,120-223,227-259,349-391,393-464,482-554), used as
 * the checker for the CUDA path.  Only tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline / --impl reference legs may load liboracle.so; the product must never
 * route through it.
 *
 * PARITY PINNED: with rng_mode=ORACLE_RNG_LIBC and dielectric_mode=SPLIT this file
 * reproduces the unmodified reference (oracle/_ref/libref.so, built from the reference
 * sources where they lie) BIT FOR BIT -- whole 8-bit frames under srand(seed), double
 * per-pixel means, per-ray hit records and single paths replayed from a shared random
 * stream.  tests/test_oracle_vs_ref.py holds those checks and tests/golden/ the vectors
 * generated from the reference (the reference's own tests pin nothing on this path,
 * SURVEY.md section 4).
 *
 * On top of the reference behaviour it restates, for the GPU comparison:
 *   - a mesh-aware nearest hit (the reference's mesh branch is commented out,
 *     raytracer.c:414-434; this follows it plus the live intersect_triangle and
 *     calculate_surface_normal).  Deviation, documented in DESIGN.md: u,v of a mesh hit
 *     are the interpolated texcoords of the NEAREST triangle (the dead block would leak
 *     the last successful triangle test's u,v);
 *   - run-time MAX_DEPTH;
 *   - Philox4x32-10 keyed by (pixel, sample, bounce, block) in place of rand();
 *   - the stochastic dielectric estimator (one child per vertex) next to the
 *     reference's deterministic 2-way split.
 *
 * Every expression keeps the reference's evaluation order, and the file must be built
 * with -std=c99 -O3 -ffp-contract=off (no FMA contraction), like the reference build
 * (Makefile:2), or bit-exactness is lost.
 */
#include "raytracer.h" /* repo include/: ABI structs only */
#include "oracle.h"

#include <omp.h>

/* ---- Philox4x32-10 (Salmon et al., SC'11; Random123 v1.09 philox.h) ------- */

#define PHILOX_M0 0xD2511F53u
#define PHILOX_M1 0xCD9E8D57u
#define PHILOX_W0 0x9E3779B9u
#define PHILOX_W1 0xBB67AE85u

void oracle_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4])
{
  uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3];
  uint32_t k0 = key[0], k1 = key[1];
  for (int round = 0; round < 10; round++)
  {
    uint64_t p0 = (uint64_t)PHILOX_M0 * c0;
    uint64_t p1 = (uint64_t)PHILOX_M1 * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    uint32_t n1 = (uint32_t)p1;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    uint32_t n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += PHILOX_W0;
    k1 += PHILOX_W1;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

/* ---- random source ---------------------------------------------------------
 * The integrator asks for draws by ROLE, so the same code serves the reference's
 * sequential rand() order and the GPU's counter-based layout:
 *   jitter      2 draws  (raytracer.c:203-204, u first)
 *   rr          1 draw   (raytracer.c:499)
 *   choice      1 draw   (stochastic dielectric only; no reference counterpart)
 *   try k       3 draws  (raytracer.c:239, x then y then z)
 * Keyed layout: counter = (pixel, sample, bounce | branch<<8, block), key = seed.
 *   jitter: bounce word = 0xFFFFFFFF, block 0, words 0,1
 *   block 0 of a bounce: word 0 = rr, words 1..3 = try 0 (word 1 doubles as `choice`;
 *   a vertex is either dielectric or diffuse, never both)
 *   block k>=1: words 0..2 = try k
 * A 32-bit word w becomes the uniform (w >> 1) / 2^31, the reference's 31-bit
 * resolution (raytracer.c:227 with RAND_MAX = 2^31-1). */

typedef struct
{
  int mode;
  /* stream replay */
  const int32_t *stream;
  long long stream_len, stream_pos, overrun;
  /* keyed */
  uint32_t key[2];
  uint32_t pixel, sample;
  /* stats */
  long long rays, tests;
} Rng;

static inline double uniform_from_r31(int32_t r31)
{
  return (double)r31 / ((double)2147483647 + 1); /* raytracer.c:227 */
}

static inline double seq_next(Rng *g)
{
  if (g->mode == ORACLE_RNG_LIBC)
    return uniform_from_r31(rand());
  if (g->stream_pos >= g->stream_len)
  {
    g->overrun++;
    return 0.0;
  }
  return uniform_from_r31(g->stream[g->stream_pos++]);
}

static inline void keyed_block(const Rng *g, uint32_t bounce_word, uint32_t block, uint32_t out[4])
{
  uint32_t ctr[4] = { g->pixel, g->sample, bounce_word, block };
  oracle_philox4x32_10(ctr, g->key, out);
}

static inline double uniform_from_word(uint32_t w) { return uniform_from_r31((int32_t)(w >> 1)); }

static void rng_jitter(Rng *g, double *j1, double *j2)
{
  if (g->mode == ORACLE_RNG_PHILOX)
  {
    uint32_t w[4];
    keyed_block(g, 0xFFFFFFFFu, 0, w);
    *j1 = uniform_from_word(w[0]);
    *j2 = uniform_from_word(w[1]);
  }
  else
  {
    *j1 = seq_next(g);
    *j2 = seq_next(g);
  }
}

/* per-vertex draws */
typedef struct
{
  uint32_t bounce_word;
  uint32_t block0[4];
  int tries;   /* hemisphere_dir: cube-rejection tries, i.e. Philox blocks of the keyed layout */
  int flipped; /* hemisphere_dir: the direction was flipped into the normal's hemisphere */
} VertexRng;

static double rng_rr(Rng *g, VertexRng *v, int depth, uint32_t branch)
{
  if (g->mode == ORACLE_RNG_PHILOX)
  {
    v->bounce_word = (uint32_t)depth | (branch << 8);
    keyed_block(g, v->bounce_word, 0, v->block0);
    return uniform_from_word(v->block0[0]);
  }
  return seq_next(g);
}

static double rng_choice(Rng *g, VertexRng *v)
{
  if (g->mode == ORACLE_RNG_PHILOX)
    return uniform_from_word(v->block0[1]);
  return seq_next(g);
}

static void rng_try(Rng *g, VertexRng *v, int k, double xyz[3])
{
  v->tries = k + 1;
  if (g->mode == ORACLE_RNG_PHILOX)
  {
    if (k == 0)
    {
      xyz[0] = uniform_from_word(v->block0[1]);
      xyz[1] = uniform_from_word(v->block0[2]);
      xyz[2] = uniform_from_word(v->block0[3]);
    }
    else
    {
      uint32_t w[4];
      keyed_block(g, v->bounce_word, (uint32_t)k, w);
      xyz[0] = uniform_from_word(w[0]);
      xyz[1] = uniform_from_word(w[1]);
      xyz[2] = uniform_from_word(w[2]);
    }
  }
  else
  {
    xyz[0] = seq_next(g);
    xyz[1] = seq_next(g);
    xyz[2] = seq_next(g);
  }
}

/* ---- camera (raytracer.c:47-75, 375-384) ---------------------------------- */

void oracle_init_camera(Camera *camera, const double *pos, const double *target, int width, int height)
{
  double theta = 60.0 * (PI / 180);
  double half = tan(theta / 2);
  double vp_h = 2.0 * half;
  double aspect = (double)width / (double)height;
  double vp_w = aspect * vp_h;

  vec3 position = { pos[0], pos[1], pos[2] };
  vec3 tgt = { target[0], target[1], target[2] };
  vec3 world_up = { 0, 1, 0 };

  vec3 forward = vec3_normalize(vec3_sub(tgt, position));
  vec3 right = vec3_normalize(vec3_cross(world_up, forward));
  vec3 up = vec3_normalize(vec3_cross(forward, right));

  camera->position = position;
  camera->vertical = vec3_scalar_mult(up, vp_h);
  camera->horizontal = vec3_scalar_mult(right, vp_w);

  vec3 half_v = vec3_scalar_div(camera->vertical, 2);
  vec3 half_h = vec3_scalar_div(camera->horizontal, 2);

  /* the image plane sits one unit BEHIND the eye: pos - H/2 - (V/2 - (-forward)) */
  camera->lower_left_corner =
      vec3_sub(vec3_sub(camera->position, half_h), vec3_sub(half_v, vec3_scalar_mult(forward, -1)));
}

static Ray camera_ray(const Camera *c, double u, double v)
{
  vec3 on_plane = vec3_add(c->lower_left_corner,
                           vec3_add(vec3_scalar_mult(c->horizontal, u), vec3_scalar_mult(c->vertical, v)));
  Ray r;
  r.origin = c->position;
  r.direction = vec3_normalize(vec3_sub(c->position, on_plane));
  return r;
}

void oracle_camera_ray(const Camera *camera, double u, double v, double *ray6)
{
  Ray r = camera_ray(camera, u, v);
  ray6[0] = r.origin.x; ray6[1] = r.origin.y; ray6[2] = r.origin.z;
  ray6[3] = r.direction.x; ray6[4] = r.direction.y; ray6[5] = r.direction.z;
}

/* ---- primitives ----------------------------------------------------------- */

/* geometric ray/sphere test, raytracer.c:77-118.  Assumes |direction| = 1. */
static bool sphere_test(const Ray *ray, vec3 center, double radius, double *t_out)
{
  vec3 L = vec3_sub(center, ray->origin);
  double tca = vec3_dot(L, ray->direction);
  if (tca < 0)
    return false; /* also when the origin is inside the sphere (quirk Q10) */
  double d2 = vec3_dot(L, L) - tca * tca;
  double r2 = radius * radius;
  if (d2 > r2)
    return false;
  double thc = sqrt(r2 - d2);
  double t0 = tca - thc;
  double t1 = tca + thc;
  if (t0 > t1)
  {
    double swap = t0;
    t0 = t1;
    t1 = swap;
  }
  if (t0 < 0)
  {
    t0 = t1;
    if (t0 < 0)
      return false;
  }
  if (t0 > EPSILON)
  {
    *t_out = t0;
    return true;
  }
  return false;
}

/* Moeller-Trumbore, raytracer.c:120-174.  No backface culling. */
static bool triangle_test(const Ray *ray, const Vertex *a, const Vertex *b, const Vertex *c,
                          double *t_out, double *tex_u, double *tex_v)
{
  vec3 e1 = vec3_sub(b->pos, a->pos);
  vec3 e2 = vec3_sub(c->pos, a->pos);
  vec3 h = vec3_cross(ray->direction, e2);
  double det = vec3_dot(e1, h);
  if (det > -EPSILON && det < EPSILON)
    return false;
  double f = 1.0 / det;
  vec3 s = vec3_sub(ray->origin, a->pos);
  double u = f * vec3_dot(s, h);
  if (u < 0.0 || u > 1.0)
    return false;
  vec3 q = vec3_cross(s, e1);
  double v = f * vec3_dot(ray->direction, q);
  if (v < 0.0 || u + v > 1.0)
    return false;
  double t = f * vec3_dot(e2, q);
  if (t > EPSILON)
  {
    *t_out = t;
    vec2 tex = vec2_add(vec2_add(vec2_scalar_mult(a->tex, 1 - u - v), vec2_scalar_mult(b->tex, u)),
                        vec2_scalar_mult(c->tex, v));
    *tex_u = tex.x;
    *tex_v = tex.y;
    return true;
  }
  return false;
}

/* raytracer.c:42-45: cross(v2-v0, v1-v0), i.e. the NEGATED counter-clockwise normal */
static vec3 surface_normal(vec3 v0, vec3 v1, vec3 v2)
{
  return vec3_normalize(vec3_cross(vec3_sub(v2, v0), vec3_sub(v1, v0)));
}

int oracle_intersect_sphere(const double *ray6, const double *center, double radius, double *t)
{
  Ray ray = { { ray6[0], ray6[1], ray6[2] }, { ray6[3], ray6[4], ray6[5] } };
  vec3 c = { center[0], center[1], center[2] };
  double tt = DBL_MAX;
  bool ok = sphere_test(&ray, c, radius, &tt);
  *t = tt;
  return ok;
}

int oracle_intersect_triangle(const double *ray6, const double *verts, double *tuv)
{
  Ray ray = { { ray6[0], ray6[1], ray6[2] }, { ray6[3], ray6[4], ray6[5] } };
  Vertex v[3];
  for (int k = 0; k < 3; k++)
  {
    v[k].pos = (vec3){ verts[5 * k], verts[5 * k + 1], verts[5 * k + 2] };
    v[k].tex = (vec2){ verts[5 * k + 3], verts[5 * k + 4] };
  }
  tuv[0] = DBL_MAX; tuv[1] = 0; tuv[2] = 0;
  return triangle_test(&ray, &v[0], &v[1], &v[2], &tuv[0], &tuv[1], &tuv[2]);
}

void oracle_surface_normal(const double *v9, double *n3)
{
  vec3 n = surface_normal((vec3){ v9[0], v9[1], v9[2] }, (vec3){ v9[3], v9[4], v9[5] },
                          (vec3){ v9[6], v9[7], v9[8] });
  n3[0] = n.x; n3[1] = n.y; n3[2] = n.z;
}

/* ---- nearest hit (raytracer.c:393-464, mesh branch after :414-434) -------- */

typedef struct
{
  bool found;
  double t;      /* nearest t (the reference's Hit.t is the LAST tested hit, quirk Q9) */
  double u, v;
  vec3 point, normal;
  uint object_id;
  long long prim; /* global primitive index in loop order (tie-break key) */
} Nearest;

static Nearest nearest_hit(const Ray *ray, const SceneObject *objects, size_t n, long long *tests)
{
  Nearest best;
  memset(&best, 0, sizeof(best));
  double min_t = DBL_MAX;
  long long prim = 0;
  for (size_t i = 0; i < n; i++)
  {
    const SceneObject *ob = &objects[i];
    if (ob->type == GEOMETRY_SPHERE)
    {
      const Sphere *sp = ob->geometry.sphere;
      double t;
      (*tests)++;
      if (sphere_test(ray, sp->center, sp->radius, &t) && t < min_t) /* strict <: lowest index wins ties */
      {
        min_t = t;
        best.found = true;
        best.t = t;
        best.object_id = (uint)i;
        best.prim = prim;
        best.point = vec3_add(ray->origin, vec3_scalar_mult(ray->direction, t));
        best.normal = vec3_normalize(vec3_sub(best.point, sp->center));
        best.u = atan2(best.normal.x, best.normal.z) / (2 * PI) + 0.5;
        best.v = best.normal.y * 0.5 + 0.5;
      }
      prim++;
    }
    else
    {
      const TriangleMesh *mesh = ob->geometry.mesh;
      for (size_t ti = 0; ti < mesh->num_triangles; ti++, prim++)
      {
        const Vertex *a = &mesh->vertices[3 * ti + 0];
        const Vertex *b = &mesh->vertices[3 * ti + 1];
        const Vertex *c = &mesh->vertices[3 * ti + 2];
        double t, tu, tv;
        (*tests)++;
        if (triangle_test(ray, a, b, c, &t, &tu, &tv) && t < min_t)
        {
          min_t = t;
          best.found = true;
          best.t = t;
          best.object_id = (uint)i;
          best.prim = prim;
          best.point = vec3_add(ray->origin, vec3_scalar_mult(ray->direction, t));
          best.normal = surface_normal(a->pos, b->pos, c->pos);
          best.u = tu;
          best.v = tv;
        }
      }
    }
  }
  return best;
}

/* ---- scatter helpers ------------------------------------------------------ */

static vec3 reflect_dir(vec3 in, vec3 n) /* raytracer.c:349-352 */
{
  return vec3_sub(in, vec3_scalar_mult(n, 2 * vec3_dot(in, n)));
}

/* raytracer.c:354-373 with the CLAMP_BETWEEN bug (quirk Q3): cosi is the constant 1, so
 * the `else` arm always runs.  Kept operation for operation; for iot = 1 it returns
 * `in` (up to the sign of zeros). */
static vec3 refract_dir(vec3 in, vec3 N, double iot)
{
  double cosi = CLAMP_BETWEEN(0, -1, 1);
  double etai = 1, etat = iot;
  vec3 n = N;
  if (cosi < 0)
    cosi = -cosi;
  else
  {
    double swap = etai;
    etai = etat;
    etat = swap;
    n = vec3_scalar_mult(N, -1);
  }
  double eta = etai / etat;
  double k = 1 - eta * eta * (1 - cosi * cosi);
  if (k < 0)
    return (vec3){ 0, 0, 0 };
  return vec3_add(vec3_scalar_mult(in, eta), vec3_scalar_mult(n, eta * cosi - sqrtf(k)));
}

static vec3 checker(vec3 color, double u, double v, double M) /* raytracer.c:386-391 */
{
  double on = (fmod(u * M, 1.0) > 0.5) ^ (fmod(v * M, 1.0) < 0.5);
  double c = 0.3 * (1 - on) + 0.7 * on;
  return vec3_scalar_mult(color, c);
}

static double mix(double a, double b, double m) { return b * m + a * (1 - m); } /* raytracer.c:255 */

/* cube rejection then normalise, flipped to the normal's side (raytracer.c:231-253) */
static vec3 hemisphere_dir(Rng *g, VertexRng *vr, vec3 normal)
{
  vec3 p;
  int k = 0;
  do
  {
    assert(k < 99);
    double r[3];
    rng_try(g, vr, k++, r);
    /* random_range(-1,1) = r*(1-(-1)) + (-1), raytracer.c:229 */
    p = (vec3){ r[0] * (1.0 - -1.0) + -1.0, r[1] * (1.0 - -1.0) + -1.0, r[2] * (1.0 - -1.0) + -1.0 };
  } while (vec3_length(p) > 1);
  vec3 d = vec3_normalize(p);
  vr->flipped = vec3_dot(d, normal) < 0;
  if (vec3_dot(d, normal) < 0)
    return vec3_scalar_mult(d, -1);
  return d;
}

void oracle_reflect(const double *in3, const double *n3, double *out3)
{
  vec3 r = reflect_dir((vec3){ in3[0], in3[1], in3[2] }, (vec3){ n3[0], n3[1], n3[2] });
  out3[0] = r.x; out3[1] = r.y; out3[2] = r.z;
}

void oracle_refract(const double *in3, const double *n3, double iot, double *out3)
{
  vec3 r = refract_dir((vec3){ in3[0], in3[1], in3[2] }, (vec3){ n3[0], n3[1], n3[2] }, iot);
  out3[0] = r.x; out3[1] = r.y; out3[2] = r.z;
}

void oracle_checkered(const double *color3, double u, double v, double M, double *out3)
{
  vec3 r = checker((vec3){ color3[0], color3[1], color3[2] }, u, v, M);
  out3[0] = r.x; out3[1] = r.y; out3[2] = r.z;
}

/* ---- the integrator (raytracer.c:482-554) --------------------------------- */

typedef struct
{
  const SceneObject *objects;
  size_t n;
  int max_depth;
  int dielectric_mode;
  /* optional vertex recorder: first `rec_cap` vertices of the (non-split) path */
  int rec_cap, rec_n;
  int32_t *rec_id;
  double *rec_point, *rec_normal, *rec_dist;
} Tracer;

static vec3 trace(Tracer *T, Rng *g, const Ray *ray, int depth, uint32_t branch)
{
  g->rays++;
  const vec3 background = BACKGROUND;
  if (depth > T->max_depth)
    return background;
  Nearest hit = nearest_hit(ray, T->objects, T->n, &g->tests);
  if (T->rec_n < T->rec_cap)
  {
    int k = T->rec_n++;
    T->rec_id[k] = hit.found ? (int32_t)hit.object_id : -1;
    vec3 d = vec3_sub(hit.point, ray->origin);
    T->rec_dist[k] = hit.found ? vec3_length(d) : 0.0;
    for (int c = 0; c < 3; c++)
    {
      T->rec_point[3 * k + c] = hit.found ? ((double *)&hit.point)[c] : 0.0;
      T->rec_normal[3 * k + c] = hit.found ? ((double *)&hit.normal)[c] : 0.0;
    }
  }
  if (!hit.found)
    return background;

  const Material *m = &T->objects[hit.object_id].material;
  vec3 albedo = m->color;
  vec3 emission = m->emission;

  /* Russian roulette at every vertex, one draw always consumed (quirk Q6) */
  VertexRng vr;
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
    /* "refraction" = retro-ray along -d (quirks Q3,Q4); reflection uses +d */
    vec3 dir_t = vec3_normalize(refract_dir(vec3_scalar_mult(ray->direction, -1), hit.normal, 1.0));
    vec3 dir_r = vec3_normalize(reflect_dir(vec3_scalar_mult(ray->direction, 1), hit.normal));
    if (T->dielectric_mode == ORACLE_DIELECTRIC_SPLIT)
    {
      R.direction = dir_t;
      vec3 refraction = trace(T, g, &R, depth + 1, (branch << 1) | 0u);
      R.direction = dir_r;
      vec3 reflection = trace(T, g, &R, depth + 1, (branch << 1) | 1u);
      radiance = vec3_add(vec3_scalar_mult(refraction, kt), vec3_scalar_mult(reflection, kr));
    }
    else
    {
      /* one child: reflection with probability p = clamp(kr, .05, .95), weights kr/p and
       * kt/(1-p); same expectation as the split for any kr (also kr > 1, kt < 0) */
      double p = kr < 0.05 ? 0.05 : (kr > 0.95 ? 0.95 : kr);
      if (rng_choice(g, &vr) < p)
      {
        R.direction = dir_r;
        radiance = vec3_scalar_mult(trace(T, g, &R, depth + 1, branch), kr / p);
      }
      else
      {
        R.direction = dir_t;
        radiance = vec3_scalar_mult(trace(T, g, &R, depth + 1, branch), kt / (1 - p));
      }
    }
  }
  else if (flags & M_REFLECTION)
  {
    R.direction = reflect_dir(ray->direction, hit.normal); /* not renormalised (quirk Q8) */
    radiance = trace(T, g, &R, depth + 1, branch);
  }
  else
  {
    /* uniform hemisphere, weight albedo*cos, no pdf factor (quirk Q5) */
    R.direction = hemisphere_dir(g, &vr, hit.normal);
    double cos_theta = vec3_dot(R.direction, hit.normal);
    radiance = vec3_scalar_mult(trace(T, g, &R, depth + 1, branch), cos_theta);
  }
  return vec3_add(emission, vec3_mult(albedo, radiance));
}

/* ---- drivers -------------------------------------------------------------- */

/* ---- Whitted integrator: cast_ray (raytracer.c:556-641), operation for operation -----------
 * Differences from upstream, both forced by the mesh-capable scene: the nearest hit is
 * nearest_hit() above (mesh-aware), and the material is SceneObject.material instead of the
 * flat Object's colour/flags.  For sphere-only scenes this function is bit-identical to the
 * reference's cast_ray (tests/test_oracle_vs_ref.py::test_cast_ray_bit_exact). */
static vec3 cast(const Tracer *T, long long *rays, long long *tests, const Ray *ray, int depth)
{
  (*rays)++;
  const vec3 background = BACKGROUND;
  if (depth > T->max_depth)
    return background;
  Nearest hit = nearest_hit(ray, T->objects, T->n, tests);
  if (!hit.found)
    return background;

  vec3 out_color = ZERO_VECTOR;
  vec3 light_pos = { 2, 7, 2 };
  vec3 light_color = { 1, 1, 1 };

  Ray light_ray = { hit.point, vec3_normalize(vec3_sub(light_pos, hit.point)) };
  /* intersect(&light_ray, ..., NULL): any primitive along the unbounded ray (raytracer.c:571) */
  bool in_shadow = nearest_hit(&light_ray, T->objects, T->n, tests).found;

  const Material *m = &T->objects[hit.object_id].material;
  vec3 object_color = m->color;
  uint flags = m->flags;

  double ka = 0.25;
  double kd = 0.5;
  double ks = 0.8;
  double alpha = 10.0;

  if (flags & M_CHECKERED)
    object_color = checker(object_color, hit.u, hit.v, 10);

  vec3 ambient = vec3_scalar_mult(light_color, ka);
  vec3 diffuse = vec3_scalar_mult(light_color, kd * MAX(0.0, vec3_dot(hit.normal, light_ray.direction)));
  vec3 reflected = reflect_dir(light_ray.direction, hit.normal);
  vec3 view_dir = vec3_normalize(vec3_sub(hit.point, ray->origin));
  vec3 specular = vec3_scalar_mult(light_color, ks * pow(MAX(vec3_dot(view_dir, reflected), 0.0), alpha));

  vec3 surface = vec3_mult(vec3_add(ambient, vec3_scalar_mult(vec3_add(specular, diffuse), in_shadow ? 0 : 1)),
                           object_color);

  vec3 reflection = ZERO_VECTOR, refraction = ZERO_VECTOR;
  double kr = 0, kt = 0;

  if (flags & M_REFLECTION)
  {
    kr = 1.0;
    Ray r = { hit.point, vec3_normalize(reflect_dir(ray->direction, hit.normal)) };
    reflection = cast(T, rays, tests, &r, depth + 1);
  }
  if (flags & M_REFRACTION)
  {
    double transparency = 0.5;
    double facingratio = -vec3_dot(ray->direction, hit.normal);
    double fresnel = mix(pow(1 - facingratio, 3), 1, 0.1);
    kr = fresnel;
    kt = (1 - fresnel) * transparency;
    Ray r = { hit.point, vec3_normalize(refract_dir(ray->direction, hit.normal, 1.0)) };
    refraction = cast(T, rays, tests, &r, depth + 1);
  }

  out_color = vec3_add(out_color, surface);
  out_color = vec3_add(out_color, vec3_add(vec3_scalar_mult(reflection, kr), vec3_scalar_mult(refraction, kt)));
  return out_color;
}

void oracle_params_default(OracleParams *p)
{
  memset(p, 0, sizeof(*p));
  p->max_depth = MAX_DEPTH;
  p->rng_mode = ORACLE_RNG_LIBC;
  p->dielectric_mode = ORACLE_DIELECTRIC_SPLIT;
  p->seed = 1666943821u; /* main.c:182 */
  p->threads = 1;
}

static void rng_setup(Rng *g, const OracleParams *p)
{
  memset(g, 0, sizeof(*g));
  g->mode = p->rng_mode;
  g->key[0] = (uint32_t)(p->seed & 0xFFFFFFFFu);
  g->key[1] = (uint32_t)(p->seed >> 32);
}

static void tracer_setup(Tracer *T, const SceneObject *objects, size_t n, const OracleParams *p)
{
  memset(T, 0, sizeof(*T));
  T->objects = objects;
  T->n = n;
  T->max_depth = p->max_depth;
  T->dielectric_mode = p->dielectric_mode;
}

/* ---- trace() in forward form, one vertex at a time ------------------------------------------
 * The same helpers and draws as trace(), but the throughput is carried forward: the vertex adds
 * tp * emission (tp * background on a miss) and hands each child tp * albedo * weight.  A child at
 * depth > max_depth is not traced: it adds its throughput * background and one ray (raytracer.c:487).
 * Summed over a path (its whole tree for the split estimator), the contributions are trace()'s value
 * up to the association of the products. */
static void path_vertex(const Tracer *T, Rng *g, const Ray *ray, int depth, uint32_t branch, const double tp[3],
                        OracleVertex *o)
{
  memset(o, 0, sizeof(*o));
  memcpy(o->ray, &ray->origin, 3 * sizeof(double));
  memcpy(o->ray + 3, &ray->direction, 3 * sizeof(double));
  memcpy(o->tp, tp, 3 * sizeof(double));
  o->pixel = g->pixel;
  o->sample = g->sample;
  o->branch = branch;
  o->depth = depth;
  o->id = -1;
  o->prim = -1;
  o->rays = 1;
  const vec3 background = BACKGROUND;
  const vec3 t = { tp[0], tp[1], tp[2] };
  vec3 contrib;
  Nearest hit;
  if (depth > T->max_depth || !(hit = nearest_hit(ray, T->objects, T->n, &g->tests)).found)
  {
    contrib = vec3_mult(t, background);
    memcpy(o->contrib, &contrib, sizeof(contrib));
    return;
  }
  o->id = (int32_t)hit.object_id;
  o->prim = hit.prim;
  o->t = hit.t;
  const Material *m = &T->objects[hit.object_id].material;
  vec3 albedo = m->color;
  contrib = vec3_mult(t, m->emission);

  VertexRng vr;
  memset(&vr, 0, sizeof(vr));
  double prob = MAX(albedo.x, MAX(albedo.y, albedo.z));
  if (rng_rr(g, &vr, depth, branch) < prob)
    albedo = vec3_scalar_mult(albedo, 1 / prob);
  else
  {
    memcpy(o->contrib, &contrib, sizeof(contrib));
    return;
  }
  o->survived = 1;
  uint flags = m->flags;
  if (flags & M_CHECKERED)
    albedo = checker(albedo, hit.u, hit.v, 100000);

  vec3 dir[2];
  double weight[2];
  uint32_t child_branch[2] = { branch, branch };
  int n_children = 1;
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
      n_children = 2;
      dir[0] = dir_t; weight[0] = kt; child_branch[0] = branch << 1;
      dir[1] = dir_r; weight[1] = kr; child_branch[1] = (branch << 1) | 1u;
    }
    else
    {
      double p = kr < 0.05 ? 0.05 : (kr > 0.95 ? 0.95 : kr);
      if (rng_choice(g, &vr) < p)
      {
        dir[0] = dir_r; weight[0] = kr / p;
      }
      else
      {
        dir[0] = dir_t; weight[0] = kt / (1 - p);
      }
    }
  }
  else if (flags & M_REFLECTION)
  {
    dir[0] = reflect_dir(ray->direction, hit.normal); /* not renormalised (quirk Q8) */
    weight[0] = 1.0;
  }
  else
  {
    dir[0] = hemisphere_dir(g, &vr, hit.normal);
    weight[0] = vec3_dot(dir[0], hit.normal);
    o->tries = vr.tries;
    o->flipped = vr.flipped;
  }
  o->n_children = n_children;
  for (int k = 0; k < n_children; k++)
  {
    vec3 ct = vec3_scalar_mult(vec3_mult(t, albedo), weight[k]);
    memcpy(o->child_ray[k], &hit.point, sizeof(vec3));
    memcpy(o->child_ray[k] + 3, &dir[k], sizeof(vec3));
    memcpy(o->child_tp[k], &ct, sizeof(vec3));
    o->child_branch[k] = child_branch[k];
    if (depth + 1 > T->max_depth)
    {
      o->cut[k] = 1;
      o->rays++;
      contrib = vec3_add(contrib, vec3_mult(ct, background));
    }
  }
  memcpy(o->contrib, &contrib, sizeof(contrib));
}

void oracle_path_vertex(const SceneObject *objects, size_t n, const OracleParams *p, const double *rays6,
                        const int32_t *depth, const uint32_t *branch, const uint32_t *pixel, const uint32_t *sample,
                        const double *tp3, long long count, OracleVertex *out)
{
  int threads = p->threads > 0 ? p->threads : 1;
#pragma omp parallel for num_threads(threads) schedule(dynamic, 256)
  for (long long i = 0; i < count; i++)
  {
    OracleParams q = *p;
    q.rng_mode = ORACLE_RNG_PHILOX;
    Rng g;
    rng_setup(&g, &q);
    g.pixel = pixel[i];
    g.sample = sample[i];
    Tracer T;
    tracer_setup(&T, objects, n, &q);
    Ray ray = { { rays6[6 * i], rays6[6 * i + 1], rays6[6 * i + 2] }, { rays6[6 * i + 3], rays6[6 * i + 4], rays6[6 * i + 5] } };
    path_vertex(&T, &g, &ray, depth[i], branch[i], tp3 + 3 * i, &out[i]);
  }
}

typedef struct
{
  OracleVertex *v;
  long long n, cap;
} VertexList;

static void vertex_push(VertexList *l, const OracleVertex *v)
{
  if (l->n == l->cap)
  {
    l->cap = l->cap ? 2 * l->cap : 1024;
    l->v = (OracleVertex *)realloc(l->v, sizeof(OracleVertex) * (size_t)l->cap);
    if (!l->v)
    {
      fprintf(stderr, "oracle: out of memory\n");
      exit(EXIT_FAILURE);
    }
  }
  l->v[l->n++] = *v;
}

long long oracle_path_log(const SceneObject *objects, size_t n, const Camera *camera, int width, int height,
                          int samples, const OracleParams *p, OracleVertex *out, long long cap)
{
  int threads = p->threads > 0 ? p->threads : 1;
  VertexList *rows = (VertexList *)calloc((size_t)height, sizeof(VertexList));
  if (!rows)
  {
    fprintf(stderr, "oracle: out of memory\n");
    exit(EXIT_FAILURE);
  }
#pragma omp parallel for num_threads(threads) schedule(dynamic, 1)
  for (int y = 0; y < height; y++)
  {
    OracleParams q = *p;
    q.rng_mode = ORACLE_RNG_PHILOX;
    Rng g;
    rng_setup(&g, &q);
    Tracer T;
    tracer_setup(&T, objects, n, &q);
    /* pending rays of one path: at most one per depth and branch bit, so depth + 2 per level suffices */
    int stack_cap = 2 * (q.max_depth + 2) + 2;
    OracleVertex *stack = (OracleVertex *)malloc(sizeof(OracleVertex) * (size_t)stack_cap);
    for (int x = 0; x < width; x++)
      for (int s = 0; s < samples; s++)
      {
        g.pixel = (uint32_t)(y * width + x);
        g.sample = (uint32_t)(p->sample_offset + s);
        double j1, j2;
        rng_jitter(&g, &j1, &j2);
        double u = (double)(x + j1) / ((double)width - 1.0);
        double v = (double)(y + j2) / ((double)height - 1.0);
        Ray ray = camera_ray(camera, u, v);
        /* stack entries use ray[], tp[], depth and branch only */
        int top = 0;
        memcpy(stack[0].ray, &ray.origin, 3 * sizeof(double));
        memcpy(stack[0].ray + 3, &ray.direction, 3 * sizeof(double));
        stack[0].tp[0] = stack[0].tp[1] = stack[0].tp[2] = 1.0;
        stack[0].depth = 0;
        stack[0].branch = 1u;
        top = 1;
        while (top > 0)
        {
          OracleVertex e = stack[--top], o;
          Ray r = { { e.ray[0], e.ray[1], e.ray[2] }, { e.ray[3], e.ray[4], e.ray[5] } };
          path_vertex(&T, &g, &r, e.depth, e.branch, e.tp, &o);
          vertex_push(&rows[y], &o);
          for (int k = o.n_children - 1; k >= 0; k--) /* child 0 first, as trace() recurses */
            if (!o.cut[k])
            {
              OracleVertex *c = &stack[top++];
              memcpy(c->ray, o.child_ray[k], sizeof(c->ray));
              memcpy(c->tp, o.child_tp[k], sizeof(c->tp));
              c->depth = o.depth + 1;
              c->branch = o.child_branch[k];
            }
        }
      }
    free(stack);
  }
  long long total = 0;
  for (int y = 0; y < height; y++)
    total += rows[y].n;
  if (total <= cap)
  {
    long long at = 0;
    for (int y = 0; y < height; y++)
    {
      if (rows[y].n)
        memcpy(out + at, rows[y].v, sizeof(OracleVertex) * (size_t)rows[y].n);
      at += rows[y].n;
    }
  }
  for (int y = 0; y < height; y++)
    free(rows[y].v);
  free(rows);
  return total;
}

/* sum over samples [sample_offset, sample_offset+samples) per pixel, in double.
 * The loop nest is raytracer.c:184-213. */
void oracle_render_sum(double *sum_rgb, const SceneObject *objects, size_t n, const Camera *camera,
                       int width, int height, int samples, const OracleParams *p, long long *counters)
{
  long long rays = 0, tests = 0;
  if (p->rng_mode == ORACLE_RNG_LIBC)
    srand((unsigned)p->seed);
  int threads = (p->rng_mode == ORACLE_RNG_PHILOX && p->threads > 0) ? p->threads : 1;

#pragma omp parallel for num_threads(threads) schedule(dynamic, 1) reduction(+ : rays, tests)
  for (int y = 0; y < height; y++)
  {
    Rng g;
    rng_setup(&g, p);
    Tracer T;
    tracer_setup(&T, objects, n, p);
    for (int x = 0; x < width; x++)
    {
      vec3 pixel = { 0, 0, 0 };
      for (int s = 0; s < samples; s++)
      {
        g.pixel = (uint32_t)(y * width + x);
        g.sample = (uint32_t)(p->sample_offset + s);
        double j1, j2;
        rng_jitter(&g, &j1, &j2);
        double u = (double)(x + j1) / ((double)width - 1.0);
        double v = (double)(y + j2) / ((double)height - 1.0);
        Ray ray = camera_ray(camera, u, v);
        vec3 sample = p->integrator == ORACLE_INTEGRATOR_WHITTED ? cast(&T, &g.rays, &g.tests, &ray, 0)
                                                                 : trace(&T, &g, &ray, 0, 1u);
        pixel = vec3_add(pixel, sample);
      }
      double *o = sum_rgb + 3 * ((size_t)y * width + x);
      o[0] = pixel.x; o[1] = pixel.y; o[2] = pixel.z;
    }
    rays += g.rays;
    tests += g.tests;
  }
  if (counters)
  {
    counters[0] = rays;
    counters[1] = tests;
  }
}

/* mean, gamma 5.0, truncation to 8 bits (raytracer.c:215-220; NaN -> 255 via CLAMP) */
void oracle_tonemap(uint8_t *fb, const double *sum_rgb, int width, int height, int total_samples)
{
  const double gamma = 5.0;
  for (size_t i = 0; i < (size_t)width * height; i++)
  {
    vec3 pixel = { sum_rgb[3 * i], sum_rgb[3 * i + 1], sum_rgb[3 * i + 2] };
    pixel = vec3_scalar_mult(pixel, 1.0 / (double)total_samples);
    fb[3 * i + 0] = (uint8_t)(255.0 * CLAMP(pow(pixel.x, 1 / gamma)));
    fb[3 * i + 1] = (uint8_t)(255.0 * CLAMP(pow(pixel.y, 1 / gamma)));
    fb[3 * i + 2] = (uint8_t)(255.0 * CLAMP(pow(pixel.z, 1 / gamma)));
  }
}

void oracle_render(uint8_t *fb, const SceneObject *objects, size_t n, const Camera *camera, int width,
                   int height, int samples, const OracleParams *p, long long *counters)
{
  double *sum = (double *)malloc(sizeof(double) * 3 * (size_t)width * height);
  if (!sum)
  {
    fprintf(stderr, "oracle: out of memory\n");
    exit(EXIT_FAILURE);
  }
  oracle_render_sum(sum, objects, n, camera, width, height, samples, p, counters);
  oracle_tonemap(fb, sum, width, height, samples);
  free(sum);
}

/* nearest hit of arbitrary rays: id (-1 miss), prim, t, point, normal, uv */
void oracle_intersect_rays(const SceneObject *objects, size_t n_obj, const double *rays, long long n_rays,
                           int32_t *ids, int64_t *prims, double *ts, double *points, double *normals,
                           double *uvs, int threads)
{
#pragma omp parallel for num_threads(threads > 0 ? threads : 1) schedule(static)
  for (long long i = 0; i < n_rays; i++)
  {
    const double *r = rays + 6 * i;
    Ray ray = { { r[0], r[1], r[2] }, { r[3], r[4], r[5] } };
    long long tests = 0;
    Nearest h = nearest_hit(&ray, objects, n_obj, &tests);
    ids[i] = h.found ? (int32_t)h.object_id : -1;
    if (prims) prims[i] = h.found ? h.prim : -1;
    if (ts) ts[i] = h.found ? h.t : 0.0;
    if (points)  { points[3 * i] = h.point.x; points[3 * i + 1] = h.point.y; points[3 * i + 2] = h.point.z; }
    if (normals) { normals[3 * i] = h.normal.x; normals[3 * i + 1] = h.normal.y; normals[3 * i + 2] = h.normal.z; }
    if (uvs)     { uvs[2 * i] = h.u; uvs[2 * i + 1] = h.v; }
  }
}

/* One path, random draws replayed from a stream (for the draw-for-draw comparison with
 * the reference's trace_path).  Returns draws consumed, -1 on overrun. */
long long oracle_trace_path_stream(const SceneObject *objects, size_t n_obj, const double *ray6, int depth,
                                   const OracleParams *p, const int32_t *stream, long long stream_len,
                                   double *radiance3)
{
  OracleParams q = *p;
  q.rng_mode = ORACLE_RNG_STREAM;
  Rng g;
  rng_setup(&g, &q);
  g.stream = stream;
  g.stream_len = stream_len;
  Tracer T;
  tracer_setup(&T, objects, n_obj, &q);
  Ray ray = { { ray6[0], ray6[1], ray6[2] }, { ray6[3], ray6[4], ray6[5] } };
  vec3 c = trace(&T, &g, &ray, depth, 1u);
  radiance3[0] = c.x; radiance3[1] = c.y; radiance3[2] = c.z;
  return g.overrun ? -1 : g.stream_pos;
}

/* Per-pixel path records for ONE sample index (keyed RNG): the first `n_vertices`
 * vertices of each pixel's path -- object id, point, normal, |point - origin| -- and the
 * sample's radiance.  Vertex 0 is the primary hit, vertex 1 the 1-bounce hit. */
void oracle_path_records(const SceneObject *objects, size_t n, const Camera *camera, int width, int height,
                         int sample, int n_vertices, const OracleParams *p, int32_t *ids, double *points,
                         double *normals, double *dists, double *radiance)
{
  int threads = p->threads > 0 ? p->threads : 1;
#pragma omp parallel for num_threads(threads) schedule(dynamic, 1)
  for (int y = 0; y < height; y++)
  {
    OracleParams q = *p;
    q.rng_mode = ORACLE_RNG_PHILOX;
    Rng g;
    rng_setup(&g, &q);
    for (int x = 0; x < width; x++)
    {
      size_t pix = (size_t)y * width + x;
      Tracer T;
      tracer_setup(&T, objects, n, &q);
      T.rec_cap = n_vertices;
      T.rec_id = ids + pix * n_vertices;
      T.rec_point = points + 3 * pix * n_vertices;
      T.rec_normal = normals + 3 * pix * n_vertices;
      T.rec_dist = dists + pix * n_vertices;
      for (int k = 0; k < n_vertices; k++)
      {
        T.rec_id[k] = -2; /* path ended before this vertex */
        T.rec_dist[k] = 0;
        for (int c = 0; c < 3; c++)
          T.rec_point[3 * k + c] = T.rec_normal[3 * k + c] = 0;
      }
      g.pixel = (uint32_t)pix;
      g.sample = (uint32_t)sample;
      double j1, j2;
      rng_jitter(&g, &j1, &j2);
      double u = (double)(x + j1) / ((double)width - 1.0);
      double v = (double)(y + j2) / ((double)height - 1.0);
      Ray ray = camera_ray(camera, u, v);
      vec3 c = trace(&T, &g, &ray, 0, 1u);
      if (radiance)
      {
        radiance[3 * pix] = c.x; radiance[3 * pix + 1] = c.y; radiance[3 * pix + 2] = c.z;
      }
    }
  }
}

/* jitter of (pixel, sample) under the keyed layout, for feeding the reference's
 * get_camera_ray with the very same (u,v) the GPU uses */
/* cast_ray() for arbitrary rays: rgb[3*i..] and (optionally) the number of cast_ray calls per ray */
void oracle_cast_rays(const SceneObject *objects, size_t n_obj, const double *rays, long long n_rays,
                      int max_depth, double *rgb, long long *ray_counts, int threads)
{
  OracleParams p;
  oracle_params_default(&p);
  p.max_depth = max_depth;
  if (threads < 1)
    threads = 1;
#pragma omp parallel for num_threads(threads) schedule(dynamic, 64)
  for (long long i = 0; i < n_rays; i++)
  {
    Tracer T;
    tracer_setup(&T, objects, n_obj, &p);
    Ray ray = { { rays[6 * i + 0], rays[6 * i + 1], rays[6 * i + 2] }, { rays[6 * i + 3], rays[6 * i + 4], rays[6 * i + 5] } };
    long long nrays = 0, tests = 0;
    vec3 c = cast(&T, &nrays, &tests, &ray, 0);
    rgb[3 * i + 0] = c.x; rgb[3 * i + 1] = c.y; rgb[3 * i + 2] = c.z;
    if (ray_counts)
      ray_counts[i] = nrays;
  }
}

void oracle_keyed_jitter(uint64_t seed, uint32_t pixel, uint32_t sample, double *j2)
{
  OracleParams p;
  oracle_params_default(&p);
  p.seed = seed;
  p.rng_mode = ORACLE_RNG_PHILOX;
  Rng g;
  rng_setup(&g, &p);
  g.pixel = pixel;
  g.sample = sample;
  rng_jitter(&g, &j2[0], &j2[1]);
}
