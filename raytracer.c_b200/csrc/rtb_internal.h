/*
 * rtb_internal.h -- structures shared by the translation units of librtb200.so.
 * Not part of the C ABI (that is include/rtb200.h).
 */
#ifndef RTB_INTERNAL_H
#define RTB_INTERNAL_H

#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <string>
#include <utility>
#include <vector>

#include "rtb200.h"

/* ---- byte layouts of the reference records (raytracer.h:60-131) ------------ */

struct RefVec3 { double x, y, z; };
struct RefVertex { RefVec3 pos; double tex[2]; };                                     /* 40 B */
struct RefObject { uint32_t flags; uint32_t pad; double radius; RefVec3 center, color, emission; }; /* 88 B */
struct RefMaterial { uint32_t flags; uint32_t pad; RefVec3 color, emission; double ka, ks, kd; };   /* 80 B */
struct RefSphere { RefVec3 center; double radius; };                                  /* 32 B */
struct RefMesh { size_t num_triangles; const RefVertex *vertices; };                  /* 16 B */
struct RefSceneObject { int32_t type; int32_t pad; RefMaterial material; const void *geometry; }; /* 96 B */

static_assert(sizeof(RefVertex) == 40, "Vertex");
static_assert(sizeof(RefObject) == 88, "Object");
static_assert(sizeof(RefMaterial) == 80, "Material");
static_assert(sizeof(RefSphere) == 32, "Sphere");
static_assert(sizeof(RefMesh) == 16, "TriangleMesh");
static_assert(sizeof(RefSceneObject) == 96, "SceneObject");

/* rtb_narrow.cpp: n_vertices Vertex records (five doubles) -> five floats each, on the host (AVX2 where the CPU has
 * it); true when every double -- positions and texture coordinates -- is float-representable */
extern "C" bool rtb_narrow_vertices(const double *src, float *dst, size_t n_vertices);
extern "C" bool rtb_narrow_vertices_scalar(const double *src, float *dst, size_t n_vertices);

#define RT_M_REFLECTION (1u << 2)
#define RT_M_REFRACTION (1u << 3)
#define RT_M_CHECKERED (1u << 4)

/* ---- device geometry --------------------------------------------------------
 * One 48-byte record per primitive, three 16-byte loads (SoA of float4 triples):
 *   sphere:   a = {cx, cy} as two doubles, b = {cz, r} as two doubles, c = {-, gid, obj|SPHERE, -}
 *   triangle: a = {v0x, v0y, v0z, v1x}, b = {v1y, v1z, v2x, v2y}, c = {v2z, gid, obj, -}
 * gid = index of the primitive in the reference's loop order (object order, then
 * triangle order inside a mesh): the tie-break key of the nearest-hit query.
 * Sphere centres and radii stay IEEE double (the exact test needs them); triangle
 * vertices are float (OBJ positions are parsed as float upstream). */
struct PrimRec { float4 a, b, c; };
#define RTB_PRIM_SPHERE_BIT 0x80000000u

/* BVH2 node, 64 bytes: both children's boxes + child references.
 *   n0 = {c0.lo.x, c0.hi.x, c0.lo.y, c0.hi.y}
 *   n1 = {c1.lo.x, c1.hi.x, c1.lo.y, c1.hi.y}
 *   n2 = {c0.lo.z, c0.hi.z, c1.lo.z, c1.hi.z}
 *   n3 = {ref0, ref1, -, -} as int bits
 * ref >= 0: inner node index; ref < 0: leaf, ~ref = (first << 3) | (count - 1), `first`
 * indexing the BVH-ordered primitive array. */
struct BvhNode { float4 n0, n1, n2, n3; };

/* BVH4 node, 128 bytes (four 256-bit loads): the BVH2 collapsed greedily by surface area
 * (k_emit4).  Half the dependent fetches per ray.
 *   q0 = lo.x of children 0..3, q1 = hi.x, q2 = lo.y, q3 = hi.y, q4 = lo.z, q5 = hi.z
 *   q6 = child references as int bits (same encoding as BvhNode; RTB_REF_NONE = empty slot)
 *   q7 = unused
 * Dense, breadth-first; node 0 is the root. */
struct Bvh4Node { float4 q[8]; };

/* Compressed BVH4 node, 64 bytes (two 256-bit loads): child boxes quantised to 8 bits per
 * coordinate on a per-node grid (origin + q * 2^e per axis, after Ylitie et al. 2017); lo is
 * rounded down and hi up, so a decoded box always contains the padded float box.
 *   w0 = {origin.x, origin.y, origin.z, ex | ey << 8 | ez << 16}   e = IEEE-754 exponent byte of the cell size
 *   w1 = child references (int bits, RTB_REF_NONE = empty slot)
 *   w2 = {qlo.x[0..3], qlo.y[0..3], qlo.z[0..3], qhi.x[0..3]}      one byte per child
 *   w3 = {qhi.y[0..3], qhi.z[0..3], -, -}
 * The L1 data pipe is the bound of the walk (one wavefront per 32-byte sector a lane touches):
 * this node costs 2 wavefronts per visit instead of 4 (Bvh4Node) or 2 x 2 (two BvhNode). */
struct Bvh4QNode { float4 w[4]; };
#define RTB_LEAF_MAX 4
#define RTB_STACK_SIZE 64
#define RTB_WF_MAX_GROUPS 4
#define RTB_REF_NONE 0x7FFFFFFF

struct SceneView
{
  const float4 *nodes; /* 4 float4 per node */
  const float4 *nodes4; /* 8 float4 per BVH4 node */
  const float4 *nodes4q; /* 4 float4 per compressed BVH4 node */
  const float4 *prims; /* 3 float4 per BVH primitive, BVH order */
  const float4 *big;   /* 3 float4 per oversized primitive (tested for every ray) */
  const float4 *mats;  /* 2 float4 per object */
  const float2 *tex;   /* 3 float2 per BVH primitive (BVH order) or NULL */
  const double *colors; /* 3 doubles per object: the unscaled material colour (Whitted integrator) */
  const double *tri64;  /* 9 doubles per BVH primitive slot: triangle vertices exactly as the caller gave them, or
                           NULL when every mesh coordinate is float-representable (the floats of PrimRec are exact) */
  int n_prims, n_big, root_ref, n_objects;
  float guard_lo[3], guard_hi[3]; /* box rays are re-based into before FP32 traversal */
  /* last, so that the fields the trace kernels read keep their parameter offsets */
  const double *tex64;  /* 6 doubles per BVH primitive slot: texture coordinates exactly as the caller gave them, or
                           NULL when every texture coordinate is float-representable (the floats of `tex` are exact) */
  float far_t; /* origins farther than this outside the guard box are walked without culling (rayf_walk_setup) */
};

struct rtb_scene
{
  int device = 0;
  SceneView view{};
  /* owned device allocations */
  float4 *d_nodes4 = nullptr, *d_nodes4q = nullptr;
  float4 *d_nodes = nullptr, *d_prims = nullptr, *d_big = nullptr, *d_mats = nullptr;
  float2 *d_tex = nullptr;
  double *d_colors = nullptr;
  double *d_tri64 = nullptr;
  double *d_tex64 = nullptr;
  float *d_scratch = nullptr; /* split planes */
  size_t scratch_bytes = 0;
  void *d_wf = nullptr;       /* wavefront kernels: ray queues + accumulation planes (rtb_wavefront.cu) */
  cudaStream_t wf_streams[RTB_WF_MAX_GROUPS] = {}; /* extra streams of the wavefront pipeline: one per plane group in flight ([0] unused: the caller's stream) */
  cudaEvent_t wf_fork = nullptr, wf_joins[RTB_WF_MAX_GROUPS] = {};
  size_t wf_bytes = 0;
  unsigned long long *d_counters = nullptr;
  rtb_scene_info info{};
  std::vector<std::pair<void *, size_t>> owned; /* every device buffer of the scene arrays, with its size */
};

/* Per-device cache of device buffers.  render() creates and destroys a scene per call; sending
 * ~13 buffers (0.1 GB of scene arrays, up to 23.4 GB of ray queues) through the CUDA memory pool
 * on every call made the call time erratic: the pool re-grows whenever its free blocks get carved
 * up differently, and a fresh allocation costs 0.1-1.5 s on this platform (measured:
 * scene create 4 ms typically, 20-1500 ms on every third call).  A destroyed scene parks its
 * buffers here; the next scene takes any parked buffer that fits (same shape -> exact matches,
 * no allocation at all).  rtb_release_workspace() empties the cache. */
void *rtb_cache_take(int device, size_t need, size_t *bytes); /* NULL if nothing parked fits */
void rtb_cache_park(int device, void *p, size_t bytes);       /* the device must be done with p */

/* ---- multi-GPU (rtb_multi.cu) -------------------------------------------------------------------
 * One rank per GPU.  `nccl` is an ncclComm_t (kept opaque here so that only rtb_multi.cu needs nccl.h). */
struct rtb_scene_shard
{
  int rank, n_ranks;
  void *nccl;
};
/* in-place all-gather (chunk `rank` of each array is this rank's) of the marshalled triangle records,
 * their boxes and (optionally) texture coordinates, on the legacy default stream of the current device;
 * d_flags_max_or_null: int[2] max-reduced over the ranks ("needs double positions", "needs double texcoords") */
int rtb_shard_allgather(const rtb_scene_shard *shard, void *prims, size_t prim_chunk_bytes, void *box_lo, void *box_hi,
                        size_t box_chunk_bytes, void *tex_or_null, size_t tex_chunk_bytes, int *d_flags_max_or_null);
int rtb_shard_allgather_bytes(const rtb_scene_shard *shard, void *base, size_t chunk_bytes);
int rtb_scene_create_sharded(const void *objects, size_t n_objects, int kind, int device, unsigned flags,
                             const rtb_scene_shard *shard, rtb_scene **out);

/* a plain cudaMalloc'd buffer of the probes, freed on every return path */
template <typename T>
struct Dev
{
  T *p = nullptr;
  ~Dev() { if (p) cudaFree(p); }
};

/* error plumbing */
void rtb_set_error(const std::string &msg);
#define RTB_CUDA(call)                                                                         \
  do                                                                                           \
  {                                                                                            \
    cudaError_t e_ = (call);                                                                   \
    if (e_ != cudaSuccess)                                                                     \
    {                                                                                          \
      rtb_set_error(std::string(#call) + ": " + cudaGetErrorString(e_));                       \
      return RTB_ECUDA;                                                                        \
    }                                                                                          \
  } while (0)

#endif
