/*
 * raytracer.h -- host-side surface of the B200 path tracer.
 *
 * Drop-in for the reference's public header (/root/reference/raytracer.h:21-164): the
 * same struct layouts, macro names, function names and argument meanings, so an
 * unchanged caller (reference main.c / test.c) compiles and links against
 * libraytracer_b200.so.  `render()` no longer runs an OpenMP loop on the host: it
 * marshals the scene to SoA, builds a BVH on the GPU and launches the sm_100a kernels
 * declared in rtb200.h.  There is no CPU fallback: without a CUDA device `render()`
 * prints the CUDA error and exits with EXIT_FAILURE, the reference's own error
 * convention (main.c:42,192,418).
 *
 * Struct sizes (checked by static asserts below, measured on the reference with gcc
 * 13.3 x86-64): Vertex 40, Ray 48, Material 80, Sphere 32, TriangleMesh 16, Object 88,
 * Hit 80, Camera 96, Options 56.
 *
 * Section "extensions" at the end is additive (SURVEY.md 8(b)): a mesh-capable scene
 * object, run-time depth / seed / device count, and a float accumulation output.
 */
#ifndef RAYTRACER_H
#define RAYTRACER_H

#include <stdio.h>
#include <stdlib.h>
#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>
#include <string.h>
#include <float.h>
#include <math.h>
#include <assert.h>

#include "vector.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---- constants (raytracer.h:21-31) ---------------------------------------- */

#ifndef PI
#define PI 3.14159265359 /* truncated on purpose: feeds the camera FOV and sphere u,v */
#endif
#define EPSILON 1e-8  /* self-hit guard of both primitive tests */
#define MAX_DEPTH 5   /* default bounce limit; run-time value lives in RenderParams */
#define MONTE_CARLO_SAMPLES 1

#define MAX(a, b) ((a) > (b) ? (a) : (b))
#define MIN(a, b) ((a) < (b) ? (a) : (b))
#define CLAMP(x) (MAX(0, MIN(x, 1)))
/* Kept bug-for-bug (quirk Q3): the first argument is ignored, the value is always 1. */
#define CLAMP_BETWEEN(x, min_v, max_v) (MAX(min_v, MIN(max_v, 1)))
#define ABS(x) ((x < 0) ? (-x) : (x))
#define EQ(a, b) (ABS((a) - (b)) < EPSILON)

#define VECTOR(x, y, z) ((vec3){ (x), (y), (z) })
#define RGB(r, g, b) (VECTOR((r) / 255.0, (g) / 255.0, (b) / 255.0))
#define RAY(o, d) ((Ray){ .origin = o, .direction = d })

#define RED RGB(255, 0, 0)
#define GREEN RGB(0, 192, 48)
#define BLUE RGB(0, 0, 255)
#define WHITE RGB(255, 255, 255)
#define BLACK RGB(0, 0, 0)
#define BACKGROUND RGB(10, 10, 10) /* returned on a miss AND on a depth cut (quirk Q2) */
#define ZERO_VECTOR RGB(0, 0, 0)
#define ONE_VECTOR (VECTOR(1.0, 1.0, 1.0))
#define RANDOM_COLOR \
  (vec3) { random_double(), random_double(), random_double() }

/* material flag bits (raytracer.h:53-56); priority REFRACTION > REFLECTION > diffuse */
#define M_DEFAULT ((uint)1 << 1)
#define M_REFLECTION ((uint)1 << 2)
#define M_REFRACTION ((uint)1 << 3)
#define M_CHECKERED ((uint)1 << 4)

/* ---- types (raytracer.h:60-131) ------------------------------------------- */

typedef uint32_t uint;

typedef struct { vec3 pos; vec2 tex; } Vertex;
typedef struct { vec3 origin, direction; } Ray;

typedef struct
{
  uint flags;
  vec3 color, emission;
  double ka, ks, kd;
} Material;

typedef struct
{
  vec3 center;
  double radius;
} Sphere;

typedef struct
{
  size_t num_triangles;
  Vertex *vertices; /* 3 * num_triangles, triangle t = vertices[3t .. 3t+2] */
} TriangleMesh;

typedef union
{
  TriangleMesh *mesh;
  Sphere *sphere;
} Geometry;

typedef enum
{
  GEOMETRY_SPHERE,
  GEOMETRY_MESH,
} GeometryType;

/* The flat sphere record of the reference at HEAD (raytracer.h:104-111). */
typedef struct
{
  uint flags;
  double radius;
  vec3 center;
  vec3 color;
  vec3 emission;
} Object;

typedef struct
{
  double t, u, v;
  vec3 point;
  vec3 normal;
  uint object_id;
} Hit;

typedef struct
{
  vec3 position, horizontal, vertical, lower_left_corner;
} Camera;

typedef struct
{
  vec3 background; /* never read, like the reference */
  char *result, *obj;
  int width, height, samples;
} Options;

/* ---- reference entry points (raytracer.h:135-164) ------------------------- */

double random_double(void);
double random_range(double, double);

vec3 point_at(const Ray *ray, double t);
vec3 calculate_surface_normal(vec3 v0, vec3 v1, vec3 v2);

bool intersect_sphere(const Ray *ray, vec3 center, double radius, Hit *hit);
bool intersect_triangle(const Ray *ray, Vertex vertex0, Vertex vertex1, Vertex vertex2, Hit *hit);

void print_v(const char *msg, const vec3 v);
void print_m(const mat4 m);
vec3 clamp(const vec3 v);

void init_camera(Camera *camera, vec3 position, vec3 target, Options *options);

/* Fills framebuffer[H][W][3] (RGB8, row 0 = top).  GPU path; see rtb200.h. */
void render(uint8_t *framebuffer, Object *objects, size_t n_objects, Camera *camera, Options *options);

/* Declared but never defined upstream (raytracer.h:158); defined here. */
bool load_obj(const char *filename, TriangleMesh *mesh);

extern long long ray_count;
extern long long intersection_test_count;

/* ---- extensions (not in the reference) ------------------------------------ */

/* The polymorphic scene record the reference has commented out (raytracer.h:95-102),
 * resurrected so a scene can hold meshes.  Only material.flags/color/emission are read
 * by the path tracer, like the flat Object. */
typedef struct
{
  GeometryType type;
  Material material;
  Geometry geometry;
} SceneObject;

/* integrator: the reference compiles trace_path in and cast_ray out (raytracer.c:207-211) */
enum
{
  RT_INTEGRATOR_PATH = 0,    /* trace_path, raytracer.c:482-554 */
  RT_INTEGRATOR_WHITTED = 1, /* cast_ray, raytracer.c:556-641 */
  RT_INTEGRATOR_PATH_NEE = 2 /* trace_path's estimator with next-event estimation (RTB_INTEGRATOR_PATH_NEE of rtb200.h):
                                the same image in expectation, less noise */
};

/* dielectric estimator */
enum
{
  RT_DIELECTRIC_STOCHASTIC = 0, /* one child per vertex, chosen with p = clamp(kr) */
  RT_DIELECTRIC_SPLIT = 1       /* the reference's 2-way split (raytracer.c:522-529) */
};

typedef struct
{
  int max_depth;       /* run-time MAX_DEPTH; <0 means the default 5 */
  uint64_t seed;       /* Philox key */
  int sample_offset;   /* global index of this call's first sample (spp sharding) */
  int total_samples;   /* divisor of the mean; <=0 means options->samples */
  int dielectric_mode; /* RT_DIELECTRIC_* */
  int device;          /* CUDA device ordinal */
  float *accum_out;    /* optional HOST float[H*W*3] sum of samples (not the mean) */
  int integrator;      /* RT_INTEGRATOR_*: upstream picks at compile time (`#if 1`, raytracer.c:207) */
  int num_gpus;        /* GPUs 0..num_gpus-1 of the box render disjoint sample ranges and one ncclReduce sums the
                          float buffers on GPU 0 (rtb200.h); default 1, or $RTB_NUM_GPUS so that the unchanged
                          main.c -- which calls render() without parameters -- can use the whole box */
} RenderParams;

void render_params_default(RenderParams *p);

/* Mesh-capable render.  `params` may be NULL (defaults). */
void render_scene(uint8_t *framebuffer, SceneObject *objects, size_t n_objects, Camera *camera,
                  Options *options, const RenderParams *params);

/* Same as render() with explicit parameters. */
void render_ex(uint8_t *framebuffer, Object *objects, size_t n_objects, Camera *camera,
               Options *options, const RenderParams *params);

/* First-hit feature buffers of a render (rtb_render_aov in rtb200.h), the inputs a denoiser (OIDN, OptiX) or a
 * compositor wants next to the frame.  HOST arrays of H*W pixels, row 0 = top; any may be NULL:
 *   albedo  float[H*W*3]  mean over the samples of the first hit's colour (times the checker factor), 0 on a miss
 *   normal  float[H*W*3]  mean of the first hit's outward surface normal, 0 on a miss
 *   depth   float[H*W]    mean distance to the first hit over the samples that hit, 0 where none did
 *   object  int32[H*W]    object index hit by the first sample (params->sample_offset), -1 on a miss
 * The frame itself is rendered exactly as without them.  Single GPU only (num_gpus == 1). */
typedef struct
{
  float *albedo, *normal, *depth;
  int32_t *object;
} RenderAov;

/* render_ex / render_scene that also fill `aov` (NULL = render_ex / render_scene) */
void render_ex_aov(uint8_t *framebuffer, Object *objects, size_t n_objects, Camera *camera, Options *options,
                   const RenderParams *params, const RenderAov *aov);
void render_scene_aov(uint8_t *framebuffer, SceneObject *objects, size_t n_objects, Camera *camera, Options *options,
                      const RenderParams *params, const RenderAov *aov);

/* Built-in denoiser (rtb_denoise in rtb200.h, DESIGN.md section 4.6): an edge-avoiding a-trous filter guided by the
 * frame's first-hit feature buffers.  A field 0 takes the library's default; iterations < 0 turns the filter off. */
typedef struct
{
  int iterations;        /* a-trous passes, default 5 */
  float sigma_luminance; /* default 48 */
  float sigma_normal;    /* default 128 */
  float sigma_depth;     /* default 0.1 */
  float albedo_epsilon;  /* default 1e-3 */
} DenoiseParams;

/* fills the library's defaults */
void denoise_params_default(DenoiseParams *p);

/* render_ex_aov / render_scene_aov whose framebuffer gets the DENOISED frame (the denoised mean through the
 * reference's transfer); params->accum_out still gets the raw sums, the same bits as without denoising, and `aov`
 * (may be NULL) the feature means.  `dn` NULL = defaults.  Single GPU only (num_gpus == 1). */
void render_ex_denoised(uint8_t *framebuffer, Object *objects, size_t n_objects, Camera *camera, Options *options,
                        const RenderParams *params, const RenderAov *aov, const DenoiseParams *dn);
void render_scene_denoised(uint8_t *framebuffer, SceneObject *objects, size_t n_objects, Camera *camera,
                           Options *options, const RenderParams *params, const RenderAov *aov, const DenoiseParams *dn);

/* Optional: starts creating the CUDA context(s) a later render*() with these parameters will use (NULL = defaults)
 * on a background thread and returns at once.  A driver calls it first and then reads its scene -- the reference's
 * main.c:413-429 builds the scene between allocating the frame and calling render() -- so that driver start-up
 * (0.4-2 s per process) and scene loading overlap.  The next render*() joins the thread. */
void render_warm_up(const RenderParams *params);

void free_mesh(TriangleMesh *mesh);

/* load_obj() with explicit parallelism (extension): the file is cut into line-aligned chunks of about
 * `min_chunk_bytes` (0 = 4 MB) that `threads` threads (0 = the OpenMP default, at most 32) parse; the result
 * does not depend on either argument.  load_obj(f, m) == load_obj_ex(f, m, 0, 0). */
bool load_obj_ex(const char *filename, TriangleMesh *mesh, int threads, size_t min_chunk_bytes);

/* mesh placement helper of the reference's driver (main.c:140-147) */
void apply_matrix(TriangleMesh *mesh, mat4 matrix);

#ifdef __cplusplus
}
#endif

/* layout guards: the GPU marshalling code and the ctypes mirrors depend on these */
#if defined(__STDC_VERSION__) && __STDC_VERSION__ >= 201112L
_Static_assert(sizeof(Vertex) == 40, "Vertex layout");
_Static_assert(sizeof(Ray) == 48, "Ray layout");
_Static_assert(sizeof(Material) == 80, "Material layout");
_Static_assert(sizeof(Object) == 88, "Object layout");
_Static_assert(sizeof(Hit) == 80, "Hit layout");
_Static_assert(sizeof(Camera) == 96, "Camera layout");
_Static_assert(sizeof(Options) == 56, "Options layout");
_Static_assert(sizeof(SceneObject) == 96, "SceneObject layout");
#endif

#endif /* RAYTRACER_H */
