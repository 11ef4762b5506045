/*
 * raytracer_host.c -- C99 host side of the B200 path tracer: the reference's
 * raytracer.h entry points (raytracer.h:135-164), re-implemented on top of the C ABI in
 * rtb200.h.  render() is the drop-in for /root/reference/raytracer.c:176-223; all the
 * pixel work happens in librtb200.so on the GPU.  There is no CPU rendering path here:
 * if CUDA is unavailable render() reports the error and exits, following the
 * reference's error convention (main.c:42,192,418).
 *
 * The small scalar helpers the reference also exports (intersect_sphere,
 * intersect_triangle, calculate_surface_normal, point_at, ...) are kept because
 * unchanged callers link against them (test.c uses calculate_surface_normal); they are
 * conveniences for host code, not a rendering fallback.
 */
#include <time.h>
#include <stdlib.h>
#include <pthread.h>

#include "raytracer.h"
#include "rtb200.h"

long long ray_count = 0;
long long intersection_test_count = 0;

/* ---- small exported helpers ------------------------------------------------------- */

double random_double(void) { return (double)rand() / ((double)RAND_MAX + 1); } /* raytracer.c:227 */

double random_range(double lo, double hi) { return random_double() * (hi - lo) + lo; }

vec3 point_at(const Ray *ray, double t) { return vec3_add(ray->origin, vec3_scalar_mult(ray->direction, t)); }

vec3 clamp(const vec3 v) { return (vec3){ CLAMP(v.x), CLAMP(v.y), CLAMP(v.z) }; }

/* raytracer.c:42-45 -- note the operand order: this is the negated CCW normal */
vec3 calculate_surface_normal(vec3 v0, vec3 v1, vec3 v2)
{
  vec3 a = vec3_sub(v2, v0);
  vec3 b = vec3_sub(v1, v0);
  return vec3_normalize(vec3_cross(a, b));
}

void print_v(const char *msg, const vec3 v) { printf("%s: (vec3) { %f, %f, %f }\n", msg, v.x, v.y, v.z); }

void print_m(const mat4 m)
{
  for (int row = 0; row < 4; row++)
  {
    for (int col = 0; col < 4; col++)
      printf(" %6.1f, ", m[row * 4 + col]);
    printf("\n");
  }
}

/* host scalar versions of the two primitive tests (raytracer.c:77-174) */
bool intersect_sphere(const Ray *ray, vec3 center, double radius, Hit *hit)
{
  intersection_test_count++;
  vec3 to_center = vec3_sub(center, ray->origin);
  double along = vec3_dot(to_center, ray->direction);
  if (along < 0)
    return false;
  double perp2 = vec3_dot(to_center, to_center) - along * along;
  double r2 = radius * radius;
  if (perp2 > r2)
    return false;
  double half_chord = sqrt(r2 - perp2);
  double near_t = along - half_chord, far_t = along + half_chord;
  if (near_t > far_t)
  {
    double tmp = near_t;
    near_t = far_t;
    far_t = tmp;
  }
  if (near_t < 0)
  {
    near_t = far_t;
    if (near_t < 0)
      return false;
  }
  if (!(near_t > EPSILON))
    return false;
  hit->t = near_t;
  return true;
}

bool intersect_triangle(const Ray *ray, Vertex vertex0, Vertex vertex1, Vertex vertex2, Hit *hit)
{
  intersection_test_count++;
  vec3 e1 = vec3_sub(vertex1.pos, vertex0.pos);
  vec3 e2 = vec3_sub(vertex2.pos, vertex0.pos);
  vec3 pvec = vec3_cross(ray->direction, e2);
  double det = vec3_dot(e1, pvec);
  if (det > -EPSILON && det < EPSILON)
    return false;
  double inv_det = 1.0 / det;
  vec3 tvec = vec3_sub(ray->origin, vertex0.pos);
  double bu = inv_det * vec3_dot(tvec, pvec);
  if (bu < 0.0 || bu > 1.0)
    return false;
  vec3 qvec = vec3_cross(tvec, e1);
  double bv = inv_det * vec3_dot(ray->direction, qvec);
  if (bv < 0.0 || bu + bv > 1.0)
    return false;
  double t = inv_det * vec3_dot(e2, qvec);
  if (!(t > EPSILON))
    return false;
  hit->t = t;
  vec2 tex = vec2_add(vec2_add(vec2_scalar_mult(vertex0.tex, 1 - bu - bv), vec2_scalar_mult(vertex1.tex, bu)),
                      vec2_scalar_mult(vertex2.tex, bv));
  hit->u = tex.x;
  hit->v = tex.y;
  return true;
}

/* ---- camera (raytracer.c:47-75) ----------------------------------------------------- */

void init_camera(Camera *camera, vec3 position, vec3 target, Options *options)
{
  const double fov = 60.0 * (PI / 180);
  const double view_h = 2.0 * tan(fov / 2);
  const double view_w = ((double)options->width / (double)options->height) * view_h;

  vec3 forward = vec3_normalize(vec3_sub(target, position));
  vec3 right = vec3_normalize(vec3_cross((vec3){ 0, 1, 0 }, forward));
  vec3 up = vec3_normalize(vec3_cross(forward, right));

  camera->position = position;
  camera->vertical = vec3_scalar_mult(up, view_h);
  camera->horizontal = vec3_scalar_mult(right, view_w);

  vec3 half_v = vec3_scalar_div(camera->vertical, 2);
  vec3 half_h = vec3_scalar_div(camera->horizontal, 2);
  /* image plane one unit behind the eye: pos - H/2 - (V/2 - (-forward)) */
  vec3 behind = vec3_scalar_mult(forward, -1);
  camera->lower_left_corner = vec3_sub(vec3_sub(camera->position, half_h), vec3_sub(half_v, behind));
}

/* ---- render -------------------------------------------------------------------------- */

void render_params_default(RenderParams *p)
{
  memset(p, 0, sizeof(*p));
  p->max_depth = MAX_DEPTH;
  p->seed = 1666943821u; /* main.c:182 */
  p->sample_offset = 0;
  p->total_samples = 0;
  p->dielectric_mode = RT_DIELECTRIC_STOCHASTIC;
  p->device = 0;
  p->accum_out = NULL;
  p->integrator = RT_INTEGRATOR_PATH;
  /* the unchanged main.c calls render() without parameters: RTB_NUM_GPUS lets it use the whole box */
  const char *env = getenv("RTB_NUM_GPUS");
  p->num_gpus = env ? atoi(env) : 1;
  if (p->num_gpus < 1)
    p->num_gpus = 1;
}

static void die(const char *where)
{
  fprintf(stderr, "%s: %s\n", where, rtb_last_error());
  exit(EXIT_FAILURE);
}

/* mesh placement helper of the reference's driver (main.c:140-147): every vertex position through
 * mat4_vector_mult (vector.h:63-74), in double.  The transformed positions are in general no longer
 * float-representable; the scene upload keeps them in double for the exact triangle test. */
void apply_matrix(TriangleMesh *mesh, mat4 matrix)
{
  const long long n = (long long)mesh->num_triangles * 3;
  /* every vertex on its own: the same doubles whatever the thread count */
#pragma omp parallel for schedule(static) if (n > 65536)
  for (long long i = 0; i < n; i++)
    mesh->vertices[i].pos = mat4_vector_mult(matrix, mesh->vertices[i].pos);
}

/* render_warm_up: CUDA contexts created on a background thread while the caller loads its scene */
static pthread_t g_warm_thread;
static int g_warm_running = 0;
static int g_warm_first = 0, g_warm_count = 0;

static void *warm_up_main(void *arg)
{
  (void)arg;
  for (int d = g_warm_first; d < g_warm_first + g_warm_count; d++)
    rtb_warm_up(d); /* an error shows up again, with its message, in the render call */
  return NULL;
}

static void warm_up_join(void)
{
  if (g_warm_running)
  {
    pthread_join(g_warm_thread, NULL);
    g_warm_running = 0;
  }
}

void render_warm_up(const RenderParams *params)
{
  RenderParams p;
  if (params)
    p = *params;
  else
    render_params_default(&p);
  warm_up_join();
  g_warm_first = p.num_gpus > 1 ? 0 : p.device;
  g_warm_count = p.num_gpus > 1 ? p.num_gpus : 1;
  static int at_exit_set = 0;
  if (!at_exit_set)
  {
    atexit(warm_up_join); /* a driver that gives up before it renders must not exit under a starting context */
    at_exit_set = 1;
  }
  g_warm_running = pthread_create(&g_warm_thread, NULL, warm_up_main, NULL) == 0;
}

static void fill_desc(rtb_render_desc *desc, const Options *options, const RenderParams *p)
{
  memset(desc, 0, sizeof(*desc));
  desc->width = options->width;
  desc->height = options->height;
  desc->sample_begin = p->sample_offset;
  desc->sample_end = p->sample_offset + options->samples;
  desc->max_depth = p->max_depth;
  desc->dielectric_mode = p->dielectric_mode == RT_DIELECTRIC_SPLIT ? RTB_DIELECTRIC_SPLIT : RTB_DIELECTRIC_STOCHASTIC;
  desc->seed = p->seed;
  desc->integrator = p->integrator == RT_INTEGRATOR_WHITTED    ? RTB_INTEGRATOR_WHITTED
                     : p->integrator == RT_INTEGRATOR_PATH_NEE ? RTB_INTEGRATOR_PATH_NEE
                                                               : RTB_INTEGRATOR_PATH;
}

/* One comm per process and GPU count, made on first use (NCCL communicator set-up costs ~0.1-1 s) and
 * kept: render() is called once per frame by the reference's driver, a viewer would call it per frame. */
static rtb_comm *g_comm = NULL;
static int g_comm_gpus = 0;

static void drop_comm(void)
{
  if (g_comm)
    rtb_comm_destroy(g_comm);
  g_comm = NULL;
}

static rtb_comm *local_comm(int num_gpus)
{
  if (g_comm && g_comm_gpus == num_gpus)
    return g_comm;
  static int registered = 0;
  drop_comm();
  if (rtb_comm_create_local(NULL, num_gpus, &g_comm) != RTB_OK)
    die("render: multi-GPU set-up");
  g_comm_gpus = num_gpus;
  if (!registered)
  {
    atexit(drop_comm);
    registered = 1;
  }
  return g_comm;
}

/* the frame on one scene (denoised when `dn` is given) and, with `aov`, the means of its feature buffers in float.
 * The denoiser runs the feature pass itself and hands its sums back, so that pass runs once either way. */
static int render_on_scene(rtb_scene *scene, const double *cam, const rtb_render_desc *desc, int divisor,
                           const DenoiseParams *dn, const RenderAov *aov, uint8_t *framebuffer, float *accum_out,
                           rtb_counters *counters)
{
  const size_t n_px = (size_t)desc->width * desc->height;
  const int spp = desc->sample_end - desc->sample_begin;
  uint32_t *hits = aov && aov->depth ? (uint32_t *)malloc(sizeof(uint32_t) * n_px) : NULL;
  if (aov && aov->depth && !hits)
  {
    fprintf(stderr, "render: out of host memory for the hit counts\n");
    return RTB_ENOMEM;
  }
  int rc;
  if (dn)
  {
    const rtb_denoise_desc d = { dn->iterations, dn->sigma_luminance, dn->sigma_normal, dn->sigma_depth,
                                 dn->albedo_epsilon };
    rc = rtb_render_denoised_aov(scene, cam, desc, divisor, &d, framebuffer, NULL, accum_out,
                                 aov ? aov->albedo : NULL, aov ? aov->normal : NULL, aov ? aov->depth : NULL, hits,
                                 aov ? aov->object : NULL, counters);
  }
  else
  {
    rc = rtb_render_mean(scene, cam, desc, divisor, framebuffer, accum_out, counters);
    /* the features of a next-event-estimation render are the first hits of trace_path's own camera samples */
    rtb_render_desc feat = *desc;
    if (feat.integrator == RTB_INTEGRATOR_PATH_NEE)
      feat.integrator = RTB_INTEGRATOR_PATH;
    if (rc == RTB_OK && aov)
      rc = rtb_render_aov_host(scene, cam, &feat, aov->albedo, aov->normal, aov->depth, hits, aov->object, NULL);
  }
  if (rc == RTB_OK && aov)
  {
    const float n_samples = spp > 0 ? (float)spp : 1.0f; /* spp == 0: the sums are 0 */
    for (size_t i = 0; i < 3 * n_px; i++)
    {
      if (aov->albedo)
        aov->albedo[i] = aov->albedo[i] / n_samples;
      if (aov->normal)
        aov->normal[i] = aov->normal[i] / n_samples;
    }
    if (aov->depth)
      for (size_t i = 0; i < n_px; i++)
        aov->depth[i] = hits[i] ? aov->depth[i] / (float)hits[i] : 0.0f;
  }
  free(hits);
  return rc;
}

/* the body of render(): objects are Object (88-byte) or SceneObject (96-byte) records */
static void render_records(uint8_t *framebuffer, const void *objects, size_t n_objects, int record_bytes,
                           Camera *camera, Options *options, const RenderParams *params, const RenderAov *aov,
                           const DenoiseParams *dn)
{
  RenderParams p;
  if (params)
    p = *params;
  else
    render_params_default(&p);
  if (p.max_depth < 0)
    p.max_depth = MAX_DEPTH;
  if (p.num_gpus < 1)
    p.num_gpus = 1;
  warm_up_join(); /* a render_warm_up() still creating contexts */

  rtb_render_desc desc;
  fill_desc(&desc, options, &p);
  const double *cam = (const double *)camera; /* 12 doubles, raytracer.h:121-124 */
  const int divisor = p.total_samples > 0 ? p.total_samples : options->samples;
  rtb_counters counters;
  if (aov && !aov->albedo && !aov->normal && !aov->depth && !aov->object)
    aov = NULL;

  if (p.num_gpus > 1)
  {
    if (aov)
    {
      fprintf(stderr, "render: feature buffers (RenderAov) are single-GPU; render them with num_gpus = 1\n");
      exit(EXIT_FAILURE);
    }
    if (dn)
    {
      fprintf(stderr, "render: the denoiser is single-GPU; denoise with num_gpus = 1\n");
      exit(EXIT_FAILURE);
    }
    /* all GPUs of the box: spp-sharded, one ncclReduce of the float sums (rtb200.h) */
    if (p.total_samples > 0 && p.total_samples != options->samples)
    {
      fprintf(stderr, "render: total_samples is for a caller that shards samples itself; with num_gpus > 1 the library does\n");
      exit(EXIT_FAILURE);
    }
    if (rtb_render_multi(local_comm(p.num_gpus), objects, n_objects, record_bytes, cam, &desc, framebuffer, p.accum_out,
                         &counters) != RTB_OK)
      die("render");
  }
  else
  {
    rtb_scene *scene = NULL;
    const int timing = getenv("RTB_TIMING") != NULL; /* development aid: where an end-to-end call spends its time */
    struct timespec t0, t1, t2;
    clock_gettime(CLOCK_MONOTONIC, &t0);
    int rc = record_bytes == 96 ? rtb_scene_create(objects, n_objects, p.device, &scene)
                                : rtb_scene_create_objects(objects, n_objects, p.device, &scene);
    if (rc != RTB_OK)
      die("render: scene upload");
    clock_gettime(CLOCK_MONOTONIC, &t1);
    if (render_on_scene(scene, cam, &desc, divisor, dn, aov, framebuffer, p.accum_out, &counters) != RTB_OK)
    {
      rtb_scene_destroy(scene);
      die("render");
    }
    clock_gettime(CLOCK_MONOTONIC, &t2);
    rtb_scene_destroy(scene);
    if (timing)
      fprintf(stderr, "render: create %.1f ms, render %.1f ms\n",
              1e3 * (double)(t1.tv_sec - t0.tv_sec) + 1e-6 * (double)(t1.tv_nsec - t0.tv_nsec),
              1e3 * (double)(t2.tv_sec - t1.tv_sec) + 1e-6 * (double)(t2.tv_nsec - t1.tv_nsec));
  }
  /* same meaning as the reference's globals (raytracer.c:36-37) */
  ray_count += (long long)counters.rays;
  intersection_test_count += (long long)counters.prim_tests;
}

void render_ex(uint8_t *framebuffer, Object *objects, size_t n_objects, Camera *camera, Options *options,
               const RenderParams *params)
{
  render_records(framebuffer, objects, n_objects, 88, camera, options, params, NULL, NULL);
}

void render_ex_aov(uint8_t *framebuffer, Object *objects, size_t n_objects, Camera *camera, Options *options,
                   const RenderParams *params, const RenderAov *aov)
{
  render_records(framebuffer, objects, n_objects, 88, camera, options, params, aov, NULL);
}

void render(uint8_t *framebuffer, Object *objects, size_t n_objects, Camera *camera, Options *options)
{
  render_ex(framebuffer, objects, n_objects, camera, options, NULL);
}

void render_scene(uint8_t *framebuffer, SceneObject *objects, size_t n_objects, Camera *camera,
                  Options *options, const RenderParams *params)
{
  render_records(framebuffer, objects, n_objects, 96, camera, options, params, NULL, NULL);
}

void render_scene_aov(uint8_t *framebuffer, SceneObject *objects, size_t n_objects, Camera *camera, Options *options,
                      const RenderParams *params, const RenderAov *aov)
{
  render_records(framebuffer, objects, n_objects, 96, camera, options, params, aov, NULL);
}

void denoise_params_default(DenoiseParams *p)
{
  p->iterations = RTB_DENOISE_DEFAULT_ITERATIONS;
  p->sigma_luminance = RTB_DENOISE_DEFAULT_SIGMA_LUMINANCE;
  p->sigma_normal = RTB_DENOISE_DEFAULT_SIGMA_NORMAL;
  p->sigma_depth = RTB_DENOISE_DEFAULT_SIGMA_DEPTH;
  p->albedo_epsilon = RTB_DENOISE_DEFAULT_ALBEDO_EPSILON;
}

void render_ex_denoised(uint8_t *framebuffer, Object *objects, size_t n_objects, Camera *camera, Options *options,
                        const RenderParams *params, const RenderAov *aov, const DenoiseParams *dn)
{
  DenoiseParams d;
  if (!dn)
    denoise_params_default(&d);
  render_records(framebuffer, objects, n_objects, 88, camera, options, params, aov, dn ? dn : &d);
}

void render_scene_denoised(uint8_t *framebuffer, SceneObject *objects, size_t n_objects, Camera *camera,
                           Options *options, const RenderParams *params, const RenderAov *aov, const DenoiseParams *dn)
{
  DenoiseParams d;
  if (!dn)
    denoise_params_default(&d);
  render_records(framebuffer, objects, n_objects, 96, camera, options, params, aov, dn ? dn : &d);
}
