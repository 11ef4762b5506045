/*
 * rtb200.h -- C ABI of librtb200.so, the sm_100a CUDA implementation of the reference's
 * render() hot path.  Plain pointers and sizes only; no C++ or torch types.
 *
 * What each entry point replaces in the reference (/root/reference):
 *   rtb_scene_create*      the implicit "scene" = the Object[] the caller hands to
 *                          render() (raytracer.h:156, main.c:256-397, main.c:429); here it
 *                          is uploaded once (a pageable Vertex array is narrowed to floats on the way up when
 *                          every coordinate is float-representable), converted AoS-double -> SoA on the device and
 *                          a BVH is built over it (replaces the O(n) loop of intersect(),
 *                          raytracer.c:393-464)
 *   rtb_render_accum       the loop nest of render() up to the per-pixel sum
 *                          (raytracer.c:184-213): camera rays (raytracer.c:375-384),
 *                          trace_path (raytracer.c:482-554), RNG (raytracer.c:227)
 *   rtb_tonemap            mean, gamma 5.0, 8-bit truncation (raytracer.c:215-220)
 *   rtb_render             the whole of render() (raytracer.c:176-223), host buffers in/out
 *   rtb_render_aov         no reference counterpart: first-hit feature buffers (albedo, normal, depth, hit count,
 *                          object id) of the render's own camera samples, the inputs of a denoiser or a compositor
 *   rtb_denoise            no reference counterpart: edge-avoiding a-trous denoiser of a frame's sums, guided by the
 *                          feature buffers of rtb_render_aov
 *   rtb_render_denoised    render() + feature pass + denoiser + tonemap of the denoised mean, host buffers out
 *                          (rtb_render_denoised_aov: also the feature sums)
 *   rtb_trace_rays         intersect() for arbitrary rays (raytracer.c:393-464): parity probe
 *   rtb_trace_rays_wf      the same records from the wavefront renderer's trace kernel: parity probe
 *   rtb_wf_generate, rtb_wf_bounce   the wavefront renderer's camera-ray and shade kernels, one launch at a time
 *                          (trace_path's vertices, raytracer.c:482-554): parity probes
 *   rtb_path_records       per-path vertex records: parity probe for the 1-bounce check
 *   rtb_cast_rays          cast_ray() for arbitrary rays (raytracer.c:556-641): parity probe of the
 *                          Whitted integrator (rtb_render_desc.integrator = RTB_INTEGRATOR_WHITTED)
 *   rtb_philox4x32_10      random_double()'s replacement (raytracer.c:227): KAT probe
 *   rtb_warm_up            no reference counterpart: creates the CUDA context early (a driver calls it on a second
 *                          thread while it reads its scene, main.c:413-429)
 *   rtb_probe_l2_bandwidth, rtb_probe_fp32_tflops   no reference counterpart: measure the L2 and FP32 roofline denominators
 *   rtb_comm_*, rtb_render_multi   render() on all GPUs of the box: spp-sharded, ONE ncclReduce of the
 *                          float sums, sharded scene upload + all-gather (no reference counterpart:
 *                          upstream is `#pragma omp parallel for` over rows, raytracer.c:184)
 *
 * Array arguments named `objects` are arrays of the reference's own records:
 *   - flat sphere record `Object`, 88 bytes (raytracer.h:104-111):
 *       u32 flags @0, f64 radius @8, f64 center[3] @16, f64 color[3] @40, f64 emission[3] @64
 *   - `SceneObject`, 96 bytes (the record commented out at raytracer.h:95-102):
 *       i32 type @0 (0 sphere, 1 mesh), Material @8 {u32 flags @8, f64 color[3] @16,
 *       f64 emission[3] @40, f64 ka,ks,kd @64}, pointer @88 to Sphere{f64 center[3], f64 radius}
 *       or TriangleMesh{size_t num_triangles, Vertex* vertices}, Vertex = {f64 pos[3], f64 tex[2]}
 * `camera` is the reference Camera (raytracer.h:121-124) viewed as 12 doubles:
 *   position, horizontal, vertical, lower_left_corner.
 *
 * All functions return 0 on success or a negative RTB_E* code; rtb_last_error() gives the
 * text (CUDA error string included).  There is no CPU fallback: without a usable CUDA
 * device every compute entry point fails with RTB_ECUDA.
 *
 * Threading: a scene may be rendered from one host thread at a time.  Device pointers
 * (`d_` prefix) belong to the scene's device; `stream` is a cudaStream_t (NULL = the
 * legacy default stream).
 */
#ifndef RTB200_H
#define RTB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTB_OK 0
#define RTB_EINVAL (-1)
#define RTB_ECUDA (-2)
#define RTB_ENOMEM (-3)

#define RTB_DIELECTRIC_STOCHASTIC 0
#define RTB_DIELECTRIC_SPLIT 1

#define RTB_INTEGRATOR_PATH 0
#define RTB_INTEGRATOR_WHITTED 1
/* trace_path's estimator with next-event estimation: at every diffuse vertex one shadow ray towards an emissive
 * sphere, combined with the hemisphere ray by the balance heuristic (DESIGN.md section 4.7).  Same expectation as
 * RTB_INTEGRATOR_PATH, less noise.  Wavefront kernel only (kernel 0 or 6), both dielectric estimators.  The path rays
 * are RTB_INTEGRATOR_PATH's, one for one (rays, rays_intersected and paths are equal); light samples draw from their
 * own Philox block.  Emissive spheres are sampled; emissive MESHES are not, they keep contributing through the
 * hemisphere ray at full weight (unbiased, just not variance-reduced). */
#define RTB_INTEGRATOR_PATH_NEE 2

typedef struct rtb_scene rtb_scene; /* opaque: device-resident SoA geometry, materials, BVH */

typedef struct
{
  int width, height;
  int sample_begin, sample_end; /* global sample indices [begin, end) rendered by this call */
  int max_depth;                /* run-time MAX_DEPTH (raytracer.h:25); path dies at depth > max_depth */
  int dielectric_mode;          /* RTB_DIELECTRIC_* */
  uint64_t seed;                /* Philox key */
  int kernel;                   /* 0 = auto; 1 megakernel (if-if walk); 2 warp-scheduled state machine;
                                   3 megakernel + FP32 sphere pre-test; 4 while-while walk; 5 suspendable walk;
                                   6 wavefront (ray queues in HBM, persistent trace kernel that refills idle lanes) */
  int reserved;                 /* tuning: kernel 5 suspend threshold in lanes; kernel 6 refill threshold in idle
                                   lanes (0 = default) */
  int planes;                   /* sample sub-ranges accumulated separately and summed in order (fixes the
                                   floating-point summation order); 0 = auto */
  int reserved2;                /* kernel 6 tuning: ray sorting mode (0 = off) */
  int integrator;               /* RTB_INTEGRATOR_PATH: trace_path (raytracer.c:482-554, the upstream default);
                                   RTB_INTEGRATOR_WHITTED: cast_ray (raytracer.c:556-641), max_depth <= 15;
                                   RTB_INTEGRATOR_PATH_NEE: trace_path with next-event estimation (kernel 0 or 6) */
  int profile;                  /* with `counters`: 1 = also count BVH node visits and time the wavefront kernels
                                   with CUDA events (trace_ms, shade_ms); 0 = rays, primitive tests and paths only */
} rtb_render_desc;

typedef struct
{
  unsigned long long rays;            /* trace_path invocations (the reference's ray_count, raytracer.c:484) */
  unsigned long long rays_intersected; /* of those, the ones that ran the scene query */
  unsigned long long prim_tests;      /* exact primitive tests (intersection_test_count, raytracer.c:79,122) */
  unsigned long long node_visits;     /* BVH nodes fetched */
  unsigned long long paths;           /* camera samples */
  unsigned long long launches;        /* kernels launched by the call */
  float gpu_ms;                       /* CUDA-event time of the call's kernels on `stream` */
  float build_ms;                     /* scene create only: upload + marshal + BVH build */
  float trace_ms;                     /* wavefront kernels: CUDA-event time summed over the k_wf_trace launches */
  float shade_ms;                     /* wavefront kernels: same for k_wf_generate + k_wf_shade */
  unsigned long long trace_launches;  /* number of k_wf_trace launches */
  unsigned long long shadow_rays;     /* RTB_INTEGRATOR_PATH_NEE: shadow rays traced (never counted in `rays`); else 0 */
  unsigned long long shadow_hits;     /* of those, the ones whose nearest hit was their light */
} rtb_counters;

typedef struct
{
  size_t n_objects, n_spheres, n_triangles;
  size_t n_bvh_prims, n_bvh_nodes, n_big_prims;
  size_t device_bytes;
  float build_ms;
  int bvh_depth;
  int device;
  int double_triangles; /* 1: some mesh coordinate is not float-representable, the scene keeps the caller's doubles
                           (72 B per triangle) for the exact triangle test; 0: the float records are exact */
  int double_texcoords; /* 1: some texture coordinate is not float-representable, the scene keeps the caller's doubles
                           (48 B per triangle) for the checker pattern; 0: the float texture coordinates are exact */
  int bvh4_depth;       /* levels of the compressed BVH4 the product path walks; 0 when it walks the BVH2 instead (a
                           tree too deep for the BVH4 walk's stack) or there is no tree */
} rtb_scene_info;

const char *rtb_last_error(void);
const char *rtb_version(void);
int rtb_device_count(void);
/* Creates the CUDA context of `device` and loads the library's kernels, so that the first scene does not pay for it
 * (0.4-2 s on a box without a persistence daemon).  Thread-safe and optional: a driver calls it from a second thread
 * while it still reads its scene from disk (render_warm_up() of raytracer.h; the reference's main.c:413-429 has the
 * same order: allocate, build the scene, then render). */
int rtb_warm_up(int device);

/* scene: upload + marshal + BVH build (blocking).  The product path builds and walks ONE tree, the
 * compressed BVH4.  RTB_SCENE_ALL_TREES also keeps the BVH2 and the uncompressed BVH4 the parity
 * probes and the megakernel variants walk (rtb_trace_rays use_bvh 1..4, rtb_render_desc.kernel 1..5). */
#define RTB_SCENE_ALL_TREES 1u
int rtb_scene_create_objects(const void *objects88, size_t n_objects, int device, rtb_scene **out);
int rtb_scene_create(const void *scene_objects96, size_t n_objects, int device, rtb_scene **out);
int rtb_scene_create_objects_flags(const void *objects88, size_t n_objects, int device, unsigned flags, rtb_scene **out);
int rtb_scene_create_flags(const void *scene_objects96, size_t n_objects, int device, unsigned flags, rtb_scene **out);
int rtb_scene_info_get(const rtb_scene *scene, rtb_scene_info *info);
void rtb_scene_destroy(rtb_scene *scene);

/* What the build made, for a checker to hold against the caller's geometry (tests/bvh_check.py). */
typedef struct
{
  size_t n_prims;   /* N: primitives in the tree */
  size_t n_big;     /* oversized spheres, tested for every ray */
  size_t n_nodes4q; /* compressed BVH4 nodes written */
  size_t n_nodes4;  /* uncompressed BVH4 nodes (RTB_SCENE_ALL_TREES), else 0 */
  size_t n_nodes2;  /* BVH2 node slots (N - 1, indexed like the build's binary hierarchy) when the BVH2 exists, else 0 */
  int root_ref;     /* 0 = node 0; < 0 a leaf, ~ref = (first << 3) | (count - 1); 0x7FFFFFFF when N = 0 */
  int leaf_max;     /* most primitives per leaf */
  int depth4;       /* levels of the BVH4 the build emitted */
  int walks_bvh4;   /* 1: the product path walks the compressed BVH4; 0: the BVH2 (or there is no tree) */
  int has_tex, has_tri64, has_tex64; /* which of the optional arrays exist */
  float scene_lo[3], scene_hi[3]; /* min / max of the primitives' float boxes */
  float guard_lo[3], guard_hi[3], pad, far_t;
} rtb_scene_tree_info;
/* Read-out probe (blocking copies to HOST buffers): *info, and those of the arrays below that are not NULL, in the
 * device layouts of csrc/rtb_internal.h.  Sizes:
 *   nodes4q 64 B x n_nodes4q; nodes4 128 B x n_nodes4; nodes 64 B x n_nodes2;
 *   prims 48 B x (N + 1) (BVH order, then the all-zero record empty BVH4 slots refer to; nothing when N = 0);
 *   big 80 B x n_big (the n_big 48-byte records, then their 32-byte FP32 copies);
 *   tri64 72 B x (N + 1), tex 24 B x N, tex64 48 B x N, each only when it exists (has_*). */
int rtb_scene_tree(const rtb_scene *scene, rtb_scene_tree_info *info, void *nodes4q, void *nodes4, void *nodes,
                   void *prims, void *big, void *tri64, void *tex, void *tex64);

/* A destroyed scene parks its device buffers (scene arrays and the wavefront kernels' ray queues, up
 * to 23.4 GB) in a per-device cache and the next scene reuses them, so that render() -- one scene per
 * call -- allocates nothing in steady state.  This returns everything cached for `device` to the driver. */
void rtb_release_workspace(int device);

/* d_accum: DEVICE float[height*width*3], OVERWRITTEN with the sum over the call's samples.
 * Asynchronous on `stream` unless `counters` is non-NULL (then it synchronises to read them). */
int rtb_render_accum(rtb_scene *scene, const double *camera12, const rtb_render_desc *desc,
                     float *d_accum, void *stream, rtb_counters *counters);

/* d_fb: DEVICE u8[height*width*3] = trunc(255*clamp((accum/total_samples)^(1/5))) */
int rtb_tonemap(const float *d_accum, int width, int height, int total_samples, uint8_t *d_fb,
                int device, void *stream);

/* whole render() with HOST buffers: framebuffer out, optional host float accum out */
int rtb_render(rtb_scene *scene, const double *camera12, const rtb_render_desc *desc,
               uint8_t *framebuffer, float *accum_or_null, rtb_counters *counters);

/* same, with an explicit divisor of the mean: a caller that shards the sample range over several calls
 * (sample_begin/end = its share) passes the job's total sample count */
int rtb_render_mean(rtb_scene *scene, const double *camera12, const rtb_render_desc *desc, int total_samples,
                    uint8_t *framebuffer, float *accum_or_null, rtb_counters *counters);

/* first-hit feature buffers of the call's primary rays (the render's own camera samples): SUMS over
 * [sample_begin, sample_end); any output may be NULL, not all; desc->kernel/dielectric_mode/max_depth unused,
 * desc->integrator selects the checker's M.  Asynchronous on `stream` unless `counters` is non-NULL.
 * Per sample, in double, on a hit (0 on a miss): d_albedo3 += the object's colour, times the checker factor 0.3 or 0.7
 * for an M_CHECKERED object at the integrator's M (100000 trace_path, raytracer.c:508; 10 cast_ray, :584); d_normal3
 * += the outward surface normal (cross(v2-v0, v1-v0) normalised on triangles, raytracer.c:44; not flipped towards the
 * camera); d_depth += t; d_hits += 1.  d_object: the object index hit by the first sample, -1 on a miss.
 * Summation: samples in double per plane (desc->planes, else automatic), rounded to float once, planes summed in
 * float in plane order, as the megakernel and Whitted renders sum; hits are an exact count.  Every buffer is
 * [height*width] (times 3 for albedo and normal) of the scene's device; counters: rays = paths = primary rays, prim_tests,
 * node_visits, launches, gpu_ms. */
int rtb_render_aov(rtb_scene *scene, const double *camera12, const rtb_render_desc *desc,
                   float *d_albedo3, float *d_normal3, float *d_depth, uint32_t *d_hits, int32_t *d_object,
                   void *stream, rtb_counters *counters);
/* the same with HOST buffers (blocking) */
int rtb_render_aov_host(rtb_scene *scene, const double *camera12, const rtb_render_desc *desc,
                        float *albedo3, float *normal3, float *depth, uint32_t *hits, int32_t *object,
                        rtb_counters *counters);

/* Denoiser: edge-avoiding a-trous filter (Dammertz et al. 2010) with SVGF's variance-guided weights (Schied et al.
 * 2017, spatial part only), DESIGN.md section 4.6.  A field 0 (or a NULL desc) takes the default below. */
typedef struct
{
  int iterations;        /* a-trous passes (steps 1, 2, 4, ...); < 0: no filtering, the output is accum / total_samples;
                            2^(iterations - 1) must be below the frame's smaller side */
  float sigma_luminance; /* luminance term exp(-|l_p - l_q| / (sigma_luminance sqrt(var_p) + tiny)) */
  float sigma_normal;    /* normal term max(0, n_p . n_q)^sigma_normal */
  float sigma_depth;     /* depth term exp(-|z_p - z_q| / (sigma_depth z_p |offset| + tiny)) */
  float albedo_epsilon;  /* the colour is filtered as colour / max(albedo, albedo_epsilon) and multiplied back */
} rtb_denoise_desc;
#define RTB_DENOISE_DEFAULT_ITERATIONS 5
#define RTB_DENOISE_DEFAULT_SIGMA_LUMINANCE 48.0f
#define RTB_DENOISE_DEFAULT_SIGMA_NORMAL 128.0f
#define RTB_DENOISE_DEFAULT_SIGMA_DEPTH 0.1f
#define RTB_DENOISE_DEFAULT_ALBEDO_EPSILON 1e-3f
/* d_out3: DEVICE float[height*width*3], the denoised MEAN radiance of a frame, from the SUMS of rtb_render_accum
 * (d_accum3) and rtb_render_aov (the other inputs) over total_samples samples; the means (colour, albedo, normal /
 * total_samples, depth / hits) are formed on the device.  d_out3 must not overlap an input.  Pixels of different
 * object ids never contribute to each other.  Asynchronous on `stream`; scratch (64 B per pixel) comes from the
 * stream-ordered pool.  RTB_EINVAL: a NULL buffer, width or height < 2, total_samples <= 0, a negative or non-finite
 * sigma, or more passes than the frame can use. */
int rtb_denoise(const rtb_denoise_desc *dn, int width, int height, int total_samples, const float *d_accum3,
                const float *d_albedo3, const float *d_normal3, const float *d_depth, const uint32_t *d_hits,
                const int32_t *d_object, float *d_out3, int device, void *stream);
/* render (rtb_render_accum) + feature pass (rtb_render_aov) + rtb_denoise + rtb_tonemap of the denoised mean (total
 * samples 1), all on the device; HOST buffers out (blocking): framebuffer u8[H*W*3]; denoised3_or_null the denoised
 * mean; accum_or_null the raw sums, the very bits rtb_render_mean returns.  counters: the render's.  dn_or_null: NULL
 * = defaults. */
int rtb_render_denoised(rtb_scene *scene, const double *camera12, const rtb_render_desc *desc, int total_samples,
                        const rtb_denoise_desc *dn_or_null, uint8_t *framebuffer, float *denoised3_or_null,
                        float *accum_or_null, rtb_counters *counters);
/* the same, and the feature sums the filter used (rtb_render_aov's for desc, HOST buffers, each may be NULL), so that
 * a caller who wants the frame's feature buffers too does not run the feature pass twice */
int rtb_render_denoised_aov(rtb_scene *scene, const double *camera12, const rtb_render_desc *desc, int total_samples,
                            const rtb_denoise_desc *dn_or_null, uint8_t *framebuffer, float *denoised3_or_null,
                            float *accum_or_null, float *albedo3_or_null, float *normal3_or_null, float *depth_or_null,
                            uint32_t *hits_or_null, int32_t *object_or_null, rtb_counters *counters);

/* parity probes (host buffers) */
int rtb_trace_rays(rtb_scene *scene, const double *rays6, size_t n_rays, int use_bvh, int32_t *ids,
                   int64_t *prims, double *ts, double *points, double *normals, double *uvs);
/* same records as rtb_trace_rays, computed by the wavefront renderer's own trace kernel: the rays are queued with
 * their hit records seeded from the oversized list, as the renderer queues them, and one launch of the trace kernel
 * that `tune` selects (rtb_render_desc.reserved encoding, 0 = the renderer's default) finds the nearest hits.
 * perm_or_null: the order the kernel fetches queue entries in (a permutation of [0, n_rays), else RTB_EINVAL).
 * counters_or_null: prim_tests (oversized list + leaves) and node_visits of the call. */
int rtb_trace_rays_wf(rtb_scene *scene, const double *rays6, size_t n_rays, int tune,
                      const uint32_t *perm_or_null, int32_t *ids, int64_t *prims, double *ts,
                      double *points, double *normals, double *uvs, rtb_counters *counters_or_null);
/* The wavefront renderer's generate and shade kernels, one launch at a time, on the renderer's own arguments, plane
 * groups, trace kernel (desc->reserved) and shade grid.  desc must fix the plane count (desc->planes > 0): path slot
 * pid = plane * width * height + pixel carries sample sample_begin + plane * chunk + wave, chunk = ceil(spp / planes).
 * Rays are 6 doubles (origin, direction), throughputs 3 floats, branch ids 1 on the camera ray (children 2b, 2b+1 of a
 * split dielectric vertex).  Queue order is the kernels' (atomics).  Host buffers, blocking.
 * rtb_wf_generate: camera rays of sample number `wave` of every plane (k_wf_generate): queue 0 of that wave; the
 * arrays hold `cap` >= planes * width * height entries, *n_out gets the queue length. */
int rtb_wf_generate(rtb_scene *scene, const double *camera12, const rtb_render_desc *desc, int wave, size_t cap,
                    double *rays6, uint32_t *pid, float *throughput3, uint32_t *branch, size_t *n_out);
/* rtb_wf_bounce: bounce `depth` of wave `wave` for n_rays queued rays (branch_or_null: NULL = 1 each; the split
 * estimator needs them): the rays are queued as the renderer queues them, one trace launch finds their hits and one
 * k_wf_shade launch shades them into planes4 (float[planes][height*width][4], read and written: planes_len floats) and
 * appends the survivors to the output queue (cap_out >= 2 * n_rays entries; *n_out its length).  ids/prims/ts
 * (optional): the hit record of every input ray (rtb_trace_rays' read-out).  counters_or_null: rays (the renderer's
 * ray count of this bounce), rays_intersected, prim_tests (oversized-list tests of the outgoing rays).
 * RTB_EINVAL on a path slot beyond the planes, a branch id 0 (or not 1 without split), depth outside [0, max_depth]. */
int rtb_wf_bounce(rtb_scene *scene, const double *camera12, const rtb_render_desc *desc, int wave, int depth,
                  size_t n_rays, const double *rays6, const uint32_t *pid, const float *throughput3,
                  const uint32_t *branch_or_null, float *planes4, size_t planes_len, int32_t *ids_or_null,
                  int64_t *prims_or_null, double *ts_or_null, size_t cap_out, double *rays6_out, uint32_t *pid_out,
                  float *throughput3_out, uint32_t *branch_out, size_t *n_out, rtb_counters *counters_or_null);
int rtb_path_records(rtb_scene *scene, const double *camera12, const rtb_render_desc *desc, int sample,
                     int n_vertices, int32_t *ids, double *points, double *normals, double *dists,
                     float *radiance);
int rtb_philox4x32_10(const uint32_t *ctr4, const uint32_t *key2, size_t n, uint32_t *out4, int device);

/* cast_ray() for arbitrary rays (raytracer.c:556-641): parity probe of the Whitted integrator.
 * rgb: HOST double[3*n]; ray_counts (optional): cast_ray invocations per ray (ray_count, raytracer.c:558) */
int rtb_cast_rays(rtb_scene *scene, const double *rays6, size_t n_rays, int max_depth, double *rgb,
                  unsigned long long *ray_counts);

/* ---- all the GPUs of one box ------------------------------------------------------------------------
 * Replaces nothing upstream (the reference is single-node CPU + OpenMP, raytracer.c:184); it is how
 * render() (raytracer.h:156, call site main.c:429) uses more than one GPU.  The per-pixel sum of
 * raytracer.c:199-213 is sharded over SAMPLES: rank r of G renders its share of the global sample
 * range, the per-GPU float sums meet in one ncclReduce(sum) on rank 0 (NVLink / NVSwitch), rank 0 runs
 * the gamma + quantise kernel.  The scene upload is sharded too: each rank sends 1/G of the triangles
 * over its PCIe link and the marshalled records are all-gathered over NVLink.
 *
 * A comm is a group of ranks, one per GPU:
 *   rtb_comm_create_rank    this process is ONE rank (one process per GPU: torchrun, mpirun); id128 comes
 *                           from rtb_comm_unique_id on rank 0 and travels through the launcher's channel
 *   rtb_comm_create_local   this process drives ALL ranks (devices[k] = CUDA ordinal of rank k, NULL = 0..n-1)
 * Calls that take a comm are collective: every rank makes them with the same arguments; a local comm
 * makes the per-rank calls itself, one host thread per GPU.  `scenes` / `scenes_out` are arrays of
 * rtb_comm_local_ranks(comm) handles (1 or n).  `record_bytes` = 88 (Object) or 96 (SceneObject).
 * desc->sample_begin/end is the WHOLE job's sample range. */
typedef struct rtb_comm rtb_comm;
#define RTB_UNIQUE_ID_BYTES 128
int rtb_comm_unique_id(void *id128);
int rtb_comm_create_rank(const void *id128, int rank, int n_ranks, int device, rtb_comm **out);
int rtb_comm_create_local(const int *devices_or_null, int n_devices, rtb_comm **out);
int rtb_comm_size(const rtb_comm *comm);
int rtb_comm_local_ranks(const rtb_comm *comm);
void rtb_comm_destroy(rtb_comm *comm);
/* which global sample indices rank `rank` of `n_ranks` renders of [sample_begin, sample_end): contiguous,
 * disjoint, covering, sizes differ by at most one (pure host arithmetic, no GPU needed) */
int rtb_comm_shard_samples(int sample_begin, int sample_end, int rank, int n_ranks, int *begin_out, int *end_out);

/* sharded upload + NVLink all-gather + per-GPU BVH build (blocking) */
int rtb_comm_scene_create(rtb_comm *comm, const void *objects, size_t n_objects, int record_bytes, unsigned flags,
                          rtb_scene **scenes_out);
/* device-resident frame: accumulate (sharded) -> ncclReduce -> tonemap on rank 0 into d_fb_root (DEVICE
 * u8[H*W*3] on rank 0's GPU, may be NULL: an internal buffer is used).  Asynchronous on each GPU's legacy
 * default stream unless `counters` is given; counters are whole-job (sums over ranks, times = slowest rank) */
int rtb_comm_render(rtb_comm *comm, rtb_scene *const *scenes, const double *camera12, const rtb_render_desc *desc,
                    uint8_t *d_fb_root, rtb_counters *counters);
/* whole render() with HOST buffers on all GPUs: scene in, framebuffer (+ optional float sums) out on rank 0 */
int rtb_render_multi(rtb_comm *comm, const void *objects, size_t n_objects, int record_bytes, const double *camera12,
                     const rtb_render_desc *desc, uint8_t *framebuffer, float *accum_or_null, rtb_counters *counters);

/* measurement probe: read bandwidth of an L2-resident buffer of `bytes` (128-bit ld.global.cg from every SM,
 * `iters` passes), in GB/s -- the denominator bench.py uses for the walk's L1/L2-served algorithmic bytes */
int rtb_probe_l2_bandwidth(size_t bytes, int iters, int device, float *gb_per_s);
/* measurement probe: FP32 FMA throughput (8 independent chains per thread, every SM full), in TFLOP/s -- the
 * denominator bench.py uses for the walk's algorithmic flops */
int rtb_probe_fp32_tflops(int iters, int device, float *tflops);

#ifdef __cplusplus
}
#endif
#endif /* RTB200_H */
