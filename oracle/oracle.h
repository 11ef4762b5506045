/*
 * oracle.h -- TEST INFRASTRUCTURE.  Interface of the CPU restatement in oracle.c.
 * See the header of oracle.c for what it follows in the reference and how it is pinned.
 * Scene structs come from the repo's include/raytracer.h (ABI-identical to the
 * reference's raytracer.h:60-131).
 */
#ifndef RTB200_ORACLE_H
#define RTB200_ORACLE_H

#include <stdint.h>
#include <stddef.h>

enum { ORACLE_RNG_LIBC = 0, ORACLE_RNG_STREAM = 1, ORACLE_RNG_PHILOX = 2 };
enum { ORACLE_DIELECTRIC_STOCHASTIC = 0, ORACLE_DIELECTRIC_SPLIT = 1 };
enum { ORACLE_INTEGRATOR_PATH = 0, ORACLE_INTEGRATOR_WHITTED = 1 };

typedef struct
{
  int max_depth;       /* run-time MAX_DEPTH (raytracer.h:25) */
  int rng_mode;        /* ORACLE_RNG_* */
  int dielectric_mode; /* ORACLE_DIELECTRIC_* */
  int sample_offset;   /* keyed RNG: global index of the first sample */
  uint64_t seed;       /* srand() seed (LIBC) or Philox key (PHILOX) */
  int threads;         /* OpenMP threads (keyed RNG only; LIBC is sequential) */
  int integrator;      /* ORACLE_INTEGRATOR_*: trace_path (raytracer.c:482) or cast_ray (raytracer.c:556) */
} OracleParams;

void oracle_params_default(OracleParams *p);

void oracle_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);
void oracle_keyed_jitter(uint64_t seed, uint32_t pixel, uint32_t sample, double *j2);

void oracle_init_camera(Camera *camera, const double *pos, const double *target, int width, int height);
void oracle_camera_ray(const Camera *camera, double u, double v, double *ray6);

int oracle_intersect_sphere(const double *ray6, const double *center, double radius, double *t);
int oracle_intersect_triangle(const double *ray6, const double *verts15, double *tuv);
void oracle_surface_normal(const double *v9, double *n3);
void oracle_reflect(const double *in3, const double *n3, double *out3);
void oracle_refract(const double *in3, const double *n3, double iot, double *out3);
void oracle_checkered(const double *color3, double u, double v, double M, double *out3);

void oracle_render_sum(double *sum_rgb, const SceneObject *objects, size_t n, const Camera *camera,
                       int width, int height, int samples, const OracleParams *p, long long *counters);
void oracle_tonemap(uint8_t *fb, const double *sum_rgb, int width, int height, int total_samples);
void oracle_render(uint8_t *fb, const SceneObject *objects, size_t n, const Camera *camera, int width,
                   int height, int samples, const OracleParams *p, long long *counters);

void oracle_intersect_rays(const SceneObject *objects, size_t n_obj, const double *rays, long long n_rays,
                           int32_t *ids, int64_t *prims, double *ts, double *points, double *normals,
                           double *uvs, int threads);
long long oracle_trace_path_stream(const SceneObject *objects, size_t n_obj, const double *ray6, int depth,
                                   const OracleParams *p, const int32_t *stream, long long stream_len,
                                   double *radiance3);
void oracle_path_records(const SceneObject *objects, size_t n, const Camera *camera, int width, int height,
                         int sample, int n_vertices, const OracleParams *p, int32_t *ids, double *points,
                         double *normals, double *dists, double *radiance);

/* One vertex of trace_path in forward form (oracle.c, path_vertex).  Field order is ABI: tests/oracle_lib.py. */
typedef struct
{
  double ray[6];          /* the incoming ray: origin, direction */
  double tp[3];           /* incoming throughput */
  double contrib[3];      /* tp * emission (tp * background on a miss) + child tp * background per cut child */
  double t;               /* nearest hit distance (0 on a miss) */
  double child_ray[2][6]; /* origin (the hit point) and direction of each child */
  double child_tp[2][3];  /* tp * albedo / prob [* checker] * weight */
  int64_t prim;           /* primitive hit in loop order, -1 on a miss */
  uint32_t pixel, sample, branch, child_branch[2];
  int32_t depth, id;      /* id: object hit, -1 on a miss */
  int32_t survived;       /* Russian roulette let the path go on (0 on a miss) */
  int32_t rays;           /* ray-counter increment: this ray plus every cut child */
  int32_t n_children;     /* 0, 1 or 2 (split dielectric), cut children included */
  int32_t cut[2];         /* child k has depth > max_depth: it adds background and a ray, and is not traced */
  int32_t tries;          /* cube-rejection tries (Philox blocks) of a diffuse vertex, else 0 */
  int32_t flipped;        /* the hemisphere sample was flipped into the normal's side */
} OracleVertex;

/* vertex i of `count`: rays6[6i..], depth[i], branch[i], keyed by (pixel[i], sample[i]), incoming throughput tp3[3i..] */
void oracle_path_vertex(const SceneObject *objects, size_t n, const OracleParams *p, const double *rays6,
                        const int32_t *depth, const uint32_t *branch, const uint32_t *pixel, const uint32_t *sample,
                        const double *tp3, long long count, OracleVertex *out);
/* every vertex of every path (the whole tree for the split estimator) of samples [sample_offset, +samples) of the
 * frame, rows in order; returns the number of vertices and writes them only when it is <= cap */
long long oracle_path_log(const SceneObject *objects, size_t n, const Camera *camera, int width, int height,
                          int samples, const OracleParams *p, OracleVertex *out, long long cap);

void oracle_cast_rays(const SceneObject *objects, size_t n_obj, const double *rays, long long n_rays,
                      int max_depth, double *rgb, long long *ray_counts, int threads);

#endif
