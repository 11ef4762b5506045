/*
 * rtb_scene.cu -- scene upload, AoS-double -> SoA marshalling and the GPU BVH build.
 *
 * Replaces the implicit scene of the reference (the Object[] handed to render(),
 * raytracer.h:156) and the O(n) loop of intersect() (raytracer.c:393-464) with a
 * device-resident structure:
 *   1. the host walks the caller's records once (pointers only), uploads sphere records
 *      and the raw 40-byte Vertex arrays, and kernels convert them to 48-byte PrimRecs;
 *   2. LBVH: 63-bit Morton codes of primitive centroids, radix sort (CUB), Karras 2012
 *      hierarchy, bottom-up box fit, subtrees of <= RTB_LEAF_MAX primitives collapsed to
 *      leaves, nodes emitted in the 64-byte two-child-box layout the walk wants;
 *   3. primitives that are far larger than the rest (the r=10000 wall spheres of
 *      main.c:258-299) are kept out of the tree in a short list tested for every ray:
 *      their centroids would otherwise stretch the Morton grid until all real geometry
 *      collapses into a handful of cells.
 * Boxes are padded so the FP32 walk is conservative w.r.t. the exact double tests (see
 * rtb_device.cuh and DESIGN.md "Precision").
 */
#include "rtb_internal.h"

#include <cub/device/device_radix_sort.cuh>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cmath>
#include <cfloat>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

/* ---- error text ------------------------------------------------------------- */

static thread_local std::string g_last_error;
void rtb_set_error(const std::string &msg) { g_last_error = msg; }
extern "C" const char *rtb_last_error(void) { return g_last_error.c_str(); }
extern "C" const char *rtb_version(void) { return "rtb200 0.1 (sm_100a)"; }

extern "C" int rtb_device_count(void)
{
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess)
  {
    rtb_set_error(std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e));
    return 0;
  }
  return n;
}

/* ---- marshalling kernels ------------------------------------------------------ */

struct SphereIn
{
  double cx, cy, cz, r;
  int obj, gid;
};

__device__ __forceinline__ float4 pack_double2(double a, double b)
{
  return make_float4(__int_as_float(__double2loint(a)), __int_as_float(__double2hiint(a)),
                     __int_as_float(__double2loint(b)), __int_as_float(__double2hiint(b)));
}

__global__ void k_marshal_spheres(const SphereIn *__restrict__ in, int n, PrimRec *__restrict__ out,
                                  float4 *__restrict__ box_lo, float4 *__restrict__ box_hi,
                                  float4 *__restrict__ fp32_copy)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n)
    return;
  SphereIn s = in[i];
  if (fp32_copy)
  {
    /* FP32 view for the conservative pre-test of the oversized list (rtb_device.cuh):
     * {cx, cy, cz, r} and A_c = |c|_1 + r, rounded up */
    float cx = (float)s.cx, cy = (float)s.cy, cz = (float)s.cz, r = (float)s.r;
    fp32_copy[2 * i + 0] = make_float4(cx, cy, cz, r);
    fp32_copy[2 * i + 1] = make_float4((fabsf(cx) + fabsf(cy) + fabsf(cz) + fabsf(r)) * 1.0000005f, 0.0f, 0.0f, 0.0f);
  }
  PrimRec r;
  r.a = pack_double2(s.cx, s.cy);
  r.b = pack_double2(s.cz, s.r);
  r.c = make_float4(0.0f, __int_as_float(s.gid), __uint_as_float((unsigned)s.obj | RTB_PRIM_SPHERE_BIT), 0.0f);
  out[i] = r;
  if (box_lo)
  {
    double rr = fabs(s.r);
    box_lo[i] = make_float4(__double2float_rd(s.cx - rr), __double2float_rd(s.cy - rr), __double2float_rd(s.cz - rr), 0.0f);
    box_hi[i] = make_float4(__double2float_ru(s.cx + rr), __double2float_ru(s.cy + rr), __double2float_ru(s.cz + rr), 0.0f);
  }
}

/* tri64 (9 doubles per triangle) keeps the positions exactly as given; inexact[0] is raised when a position
 * is not float-representable -- only then does the scene keep tri64 for the exact test (the reference's
 * arithmetic is all-double, vector.h:7; OBJ-loaded meshes are float, tinyobj_loader.h:470-481).  tex64 (6 doubles
 * per triangle) and inexact[1] do the same for the texture coordinates the checker pattern reads. */
__global__ void k_marshal_tris(const RefVertex *__restrict__ verts, int n_tris, int obj, int gid_first,
                               PrimRec *__restrict__ out, float4 *__restrict__ box_lo,
                               float4 *__restrict__ box_hi, float2 *__restrict__ tex, double *__restrict__ tri64,
                               double *__restrict__ tex64, int *__restrict__ inexact)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_tris)
    return;
  const double *p = reinterpret_cast<const double *>(verts + 3 * (size_t)i);
  /* 3 vertices x 5 doubles, contiguous */
  float v[3][3], t[3][2];
  float lo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, hi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
  bool exact = true, tex_exact = true, nan = false;
#pragma unroll
  for (int k = 0; k < 3; k++)
  {
#pragma unroll
    for (int a = 0; a < 3; a++)
    {
      const double x = p[5 * k + a];
      v[k][a] = __double2float_rn(x);
      exact = exact && ((double)v[k][a] == x);
      nan = nan || isnan(x);
      lo[a] = fminf(lo[a], __double2float_rd(x)); /* the box contains the double triangle */
      hi[a] = fmaxf(hi[a], __double2float_ru(x));
      if (tri64)
        tri64[9 * (size_t)i + 3 * k + a] = x;
    }
#pragma unroll
    for (int a = 0; a < 2; a++)
    {
      const double x = p[5 * k + 3 + a];
      t[k][a] = __double2float_rn(x);
      tex_exact = tex_exact && ((double)t[k][a] == x);
      if (tex64)
        tex64[6 * (size_t)i + 2 * k + a] = x;
    }
  }
  /* benign races: every writer stores the same value */
  if (!exact && inexact)
    inexact[0] = 1;
  if (!tex_exact && inexact)
    inexact[1] = 1;
  if (nan) /* fminf above drops a NaN: put it back into the box, where k_bounds reports it */
    lo[0] = __int_as_float(0x7FC00000);
  PrimRec r;
  r.a = make_float4(v[0][0], v[0][1], v[0][2], v[1][0]);
  r.b = make_float4(v[1][1], v[1][2], v[2][0], v[2][1]);
  r.c = make_float4(v[2][2], __int_as_float(gid_first + i), __uint_as_float((unsigned)obj), 0.0f);
  out[i] = r;
  box_lo[i] = make_float4(lo[0], lo[1], lo[2], 0.0f);
  box_hi[i] = make_float4(hi[0], hi[1], hi[2], 0.0f);
  if (tex)
  {
    tex[3 * (size_t)i + 0] = make_float2(t[0][0], t[0][1]);
    tex[3 * (size_t)i + 1] = make_float2(t[1][0], t[1][1]);
    tex[3 * (size_t)i + 2] = make_float2(t[2][0], t[2][1]);
  }
}

/* The same records from the narrowed upload (upload_narrowed: 15 floats per triangle, converted by the host's
 * staging threads, every position float-representable): no double copy is written, the box of a triangle is the
 * box of its floats. */
__global__ void k_marshal_tris_f32(const float *__restrict__ verts, int n_tris, int obj, int gid_first,
                                   PrimRec *__restrict__ out, float4 *__restrict__ box_lo,
                                   float4 *__restrict__ box_hi, float2 *__restrict__ tex)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_tris)
    return;
  const float *p = verts + 15 * (size_t)i;
  float v[3][3], t[3][2];
  float lo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, hi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
#pragma unroll
  for (int k = 0; k < 3; k++)
  {
#pragma unroll
    for (int a = 0; a < 3; a++)
    {
      v[k][a] = p[5 * k + a];
      lo[a] = fminf(lo[a], v[k][a]);
      hi[a] = fmaxf(hi[a], v[k][a]);
    }
    t[k][0] = p[5 * k + 3];
    t[k][1] = p[5 * k + 4];
  }
  PrimRec r;
  r.a = make_float4(v[0][0], v[0][1], v[0][2], v[1][0]);
  r.b = make_float4(v[1][1], v[1][2], v[2][0], v[2][1]);
  r.c = make_float4(v[2][2], __int_as_float(gid_first + i), __uint_as_float((unsigned)obj), 0.0f);
  out[i] = r;
  box_lo[i] = make_float4(lo[0], lo[1], lo[2], 0.0f);
  box_hi[i] = make_float4(hi[0], hi[1], hi[2], 0.0f);
  if (tex)
  {
    tex[3 * (size_t)i + 0] = make_float2(t[0][0], t[0][1]);
    tex[3 * (size_t)i + 1] = make_float2(t[1][0], t[1][1]);
    tex[3 * (size_t)i + 2] = make_float2(t[2][0], t[2][1]);
  }
}

/* A scene that needs double vertices after all (another mesh, or another rank's share, is not
 * float-representable): the double copy of a narrowed piece is its floats, widened */
__global__ void k_widen_tri64(const PrimRec *__restrict__ recs, int n_tris, double *__restrict__ tri64)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_tris)
    return;
  const PrimRec r = recs[i];
  double *o = tri64 + 9 * (size_t)i;
  o[0] = (double)r.a.x; o[1] = (double)r.a.y; o[2] = (double)r.a.z;
  o[3] = (double)r.a.w; o[4] = (double)r.b.x; o[5] = (double)r.b.y;
  o[6] = (double)r.b.z; o[7] = (double)r.b.w; o[8] = (double)r.c.x;
}

/* the same for texture coordinates: the double copy of a piece whose texture coordinates are exact is its floats */
__global__ void k_widen_tex64(const float2 *__restrict__ tex, int n_tris, double *__restrict__ tex64)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_tris)
    return;
  for (int k = 0; k < 3; k++)
  {
    const float2 t = tex[3 * (size_t)i + k];
    tex64[6 * (size_t)i + 2 * k + 0] = (double)t.x;
    tex64[6 * (size_t)i + 2 * k + 1] = (double)t.y;
  }
}

/* ---- bounds ------------------------------------------------------------------- */

__device__ __forceinline__ unsigned float_to_ordered(float f)
{
  unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

/* bounds[0..2] = min of box_lo, bounds[3..5] = max of box_hi (ordered-uint encoded).  fminf / fmaxf drop NaN, so a
 * NaN in any box is reported separately: bounds[3] becomes +inf, which k_build_params rejects as non-finite. */
__global__ void k_bounds(const float4 *__restrict__ box_lo, const float4 *__restrict__ box_hi, int n,
                         unsigned *__restrict__ bounds)
{
  float lo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, hi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
  bool nan = false;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
  {
    float4 a = box_lo[i], b = box_hi[i];
    lo[0] = fminf(lo[0], a.x); lo[1] = fminf(lo[1], a.y); lo[2] = fminf(lo[2], a.z);
    hi[0] = fmaxf(hi[0], b.x); hi[1] = fmaxf(hi[1], b.y); hi[2] = fmaxf(hi[2], b.z);
    nan = nan || isnan(a.x) || isnan(a.y) || isnan(a.z) || isnan(b.x) || isnan(b.y) || isnan(b.z);
  }
  nan = __any_sync(0xFFFFFFFFu, nan);
#pragma unroll
  for (int k = 0; k < 3; k++)
  {
    for (int off = 16; off > 0; off >>= 1)
    {
      lo[k] = fminf(lo[k], __shfl_xor_sync(0xFFFFFFFFu, lo[k], off));
      hi[k] = fmaxf(hi[k], __shfl_xor_sync(0xFFFFFFFFu, hi[k], off));
    }
  }
  if ((threadIdx.x & 31) == 0)
  {
#pragma unroll
    for (int k = 0; k < 3; k++)
    {
      atomicMin(&bounds[k], float_to_ordered(lo[k]));
      atomicMax(&bounds[3 + k], float_to_ordered(hi[k]));
    }
    if (nan)
      atomicMax(&bounds[3], float_to_ordered(INFINITY));
  }
}

/* ---- Morton codes --------------------------------------------------------------- */

__device__ __forceinline__ unsigned long long spread21(unsigned v)
{
  unsigned long long x = v & 0x1FFFFFull;
  x = (x | x << 32) & 0x1F00000000FFFFull;
  x = (x | x << 16) & 0x1F0000FF0000FFull;
  x = (x | x << 8) & 0x100F00F00F00F00Full;
  x = (x | x << 4) & 0x10C30C30C30C30C3ull;
  x = (x | x << 2) & 0x1249249249249249ull;
  return x;
}

/* Derived on the device from the scene box so the build needs no mid-way host round trip:
 *   guard box  = scene box grown by its diagonal on every side (rays starting outside it are
 *                re-based before the FP32 walk);
 *   pad        = 2^-20 * (largest |coordinate| in the guard box + longest parametric distance
 *                inside it): covers float rounding of the re-based ray and of the slab
 *                arithmetic (DESIGN.md "Precision");
 *   Morton grid = cubic cells over the scene box. */
struct BuildParams
{
  float lo[3], hi[3];
  float guard_lo[3], guard_hi[3];
  float pad, inv_extent;
  int finite;
};

__device__ __forceinline__ float ordered_to_float_dev(unsigned u)
{
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u);
}

__global__ void k_build_params(const unsigned *__restrict__ bounds, BuildParams *__restrict__ bp)
{
  if (threadIdx.x != 0 || blockIdx.x != 0)
    return;
  BuildParams p;
  bool finite = true;
  for (int k = 0; k < 3; k++)
  {
    p.lo[k] = ordered_to_float_dev(bounds[k]);
    p.hi[k] = ordered_to_float_dev(bounds[3 + k]);
    finite = finite && isfinite(p.lo[k]) && isfinite(p.hi[k]);
  }
  double dx = (double)p.hi[0] - p.lo[0], dy = (double)p.hi[1] - p.lo[1], dz = (double)p.hi[2] - p.lo[2];
  double diag = sqrt(dx * dx + dy * dy + dz * dz);
  if (!(diag > 0.0))
    diag = 1e-3;
  double max_abs = 0.0;
  for (int k = 0; k < 3; k++)
  {
    p.guard_lo[k] = (float)(p.lo[k] - diag);
    p.guard_hi[k] = (float)(p.hi[k] + diag);
    max_abs = fmax(max_abs, fmax(fabs((double)p.guard_lo[k]), fabs((double)p.guard_hi[k])));
  }
  p.pad = (float)((max_abs + 3.0 * diag * 1.7320508) * (1.0 / 1048576.0));
  float ext = fmaxf(p.hi[0] - p.lo[0], fmaxf(p.hi[1] - p.lo[1], p.hi[2] - p.lo[2]));
  p.inv_extent = ext > 0.0f ? 1.0f / ext : 0.0f;
  p.finite = finite ? 1 : 0;
  *bp = p;
}

__global__ void k_morton(const float4 *__restrict__ box_lo, const float4 *__restrict__ box_hi, int n,
                         const BuildParams *__restrict__ bp, unsigned long long *__restrict__ keys,
                         unsigned *__restrict__ vals)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n)
    return;
  const float3 origin = make_float3(bp->lo[0], bp->lo[1], bp->lo[2]);
  const float inv = bp->inv_extent;
  const float3 inv_extent = make_float3(inv, inv, inv);
  float4 a = box_lo[i], b = box_hi[i];
  float cx = (0.5f * (a.x + b.x) - origin.x) * inv_extent.x;
  float cy = (0.5f * (a.y + b.y) - origin.y) * inv_extent.y;
  float cz = (0.5f * (a.z + b.z) - origin.z) * inv_extent.z;
  const float scale = 2097151.0f; /* 2^21 - 1 */
  unsigned qx = (unsigned)fminf(fmaxf(cx * scale, 0.0f), scale);
  unsigned qy = (unsigned)fminf(fmaxf(cy * scale, 0.0f), scale);
  unsigned qz = (unsigned)fminf(fmaxf(cz * scale, 0.0f), scale);
  keys[i] = (spread21(qx) << 2) | (spread21(qy) << 1) | spread21(qz);
  vals[i] = (unsigned)i;
}

/* ---- Karras 2012 hierarchy ------------------------------------------------------ */

__device__ __forceinline__ int delta(const unsigned long long *__restrict__ keys, int n, int i, int j)
{
  if (j < 0 || j >= n)
    return -1;
  unsigned long long x = keys[i] ^ keys[j];
  if (x == 0ull)
    return 64 + __clz((unsigned)i ^ (unsigned)j);
  return __clzll((long long)x);
}

/* child encoding inside the build: >= 0 inner node, < 0 leaf at sorted position ~c */
__global__ void k_karras(const unsigned long long *__restrict__ keys, int n, int2 *__restrict__ children,
                         int *__restrict__ parent_inner, int *__restrict__ parent_leaf,
                         int *__restrict__ range_first)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n - 1)
    return;
  int d = (delta(keys, n, i, i + 1) - delta(keys, n, i, i - 1)) >= 0 ? 1 : -1;
  int dmin = delta(keys, n, i, i - d);
  int lmax = 2;
  while (delta(keys, n, i, i + lmax * d) > dmin)
    lmax <<= 1;
  int l = 0;
  for (int t = lmax >> 1; t >= 1; t >>= 1)
    if (delta(keys, n, i, i + (l + t) * d) > dmin)
      l += t;
  int j = i + l * d;
  int dnode = delta(keys, n, i, j);
  int s = 0;
  int t = l;
  do
  {
    t = (t + 1) >> 1;
    if (delta(keys, n, i, i + (s + t) * d) > dnode)
      s += t;
  } while (t > 1);
  int gamma = i + s * d + min(d, 0);
  int lo = min(i, j), hi = max(i, j);
  int left = (lo == gamma) ? ~gamma : gamma;
  int right = (hi == gamma + 1) ? ~(gamma + 1) : (gamma + 1);
  children[i] = make_int2(left, right);
  range_first[i] = lo;
  if (left >= 0) parent_inner[left] = i; else parent_leaf[~left] = i;
  if (right >= 0) parent_inner[right] = i; else parent_leaf[~right] = i;
  if (i == 0)
    parent_inner[0] = -1;
}

/* bottom-up: the second thread to reach a node computes its box and primitive count */
__global__ void k_fit(const unsigned *__restrict__ vals, const float4 *__restrict__ box_lo,
                      const float4 *__restrict__ box_hi, int n, const int2 *__restrict__ children,
                      const int *__restrict__ parent_inner, const int *__restrict__ parent_leaf,
                      float4 *__restrict__ node_lo, float4 *__restrict__ node_hi, int *__restrict__ flags,
                      int *__restrict__ max_depth)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n)
    return;
  int node = parent_leaf[i];
  while (node >= 0)
  {
    __threadfence();
    if (atomicAdd(&flags[node], 1) == 0)
      return;
    __threadfence();
    int2 ch = children[node];
    float4 alo, ahi, blo, bhi;
    int acount, bcount;
    if (ch.x < 0) { unsigned p = vals[~ch.x]; alo = box_lo[p]; ahi = box_hi[p]; acount = 1; }
    else { alo = __ldcg(&node_lo[ch.x]); ahi = __ldcg(&node_hi[ch.x]); acount = __float_as_int(alo.w); }
    if (ch.y < 0) { unsigned p = vals[~ch.y]; blo = box_lo[p]; bhi = box_hi[p]; bcount = 1; }
    else { blo = __ldcg(&node_lo[ch.y]); bhi = __ldcg(&node_hi[ch.y]); bcount = __float_as_int(blo.w); }
    float4 lo = make_float4(fminf(alo.x, blo.x), fminf(alo.y, blo.y), fminf(alo.z, blo.z), __int_as_float(acount + bcount));
    float4 hi = make_float4(fmaxf(ahi.x, bhi.x), fmaxf(ahi.y, bhi.y), fmaxf(ahi.z, bhi.z), 0.0f);
    __stcg(&node_lo[node], lo);
    __stcg(&node_hi[node], hi);
    node = parent_inner[node];
  }
  (void)max_depth;
}

__global__ void k_depth(int n, const int *__restrict__ parent_inner, const int *__restrict__ parent_leaf,
                        int *__restrict__ max_depth)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  int depth = 0; /* lanes past the end stay in the warp: the shuffle below names every lane */
  if (i < n)
    for (int node = parent_leaf[i]; node >= 0; node = parent_inner[node])
      depth++;
  for (int off = 16; off > 0; off >>= 1)
    depth = max(depth, __shfl_xor_sync(0xFFFFFFFFu, depth, off));
  if ((threadIdx.x & 31) == 0)
    atomicMax(max_depth, depth);
}

__host__ __device__ __forceinline__ int leaf_ref(int first, int count) { return ~((first << 3) | (count - 1)); }

/* one traversal node per inner node whose subtree holds more than RTB_LEAF_MAX primitives */
__global__ void k_emit(const unsigned *__restrict__ vals, const float4 *__restrict__ box_lo,
                       const float4 *__restrict__ box_hi, int n, const int2 *__restrict__ children,
                       const int *__restrict__ range_first, const float4 *__restrict__ node_lo,
                       const float4 *__restrict__ node_hi, const BuildParams *__restrict__ bp,
                       float4 *__restrict__ out_nodes, int *__restrict__ emitted, int leaf_max)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n - 1)
    return;
  const float pad = bp->pad;
  int count = __float_as_int(node_lo[i].w);
  if (count <= leaf_max)
    return;
  int2 ch = children[i];
  float4 lo[2], hi[2];
  int ref[2];
  int c[2] = { ch.x, ch.y };
#pragma unroll
  for (int k = 0; k < 2; k++)
  {
    if (c[k] < 0)
    {
      unsigned p = vals[~c[k]];
      lo[k] = box_lo[p];
      hi[k] = box_hi[p];
      ref[k] = leaf_ref(~c[k], 1);
    }
    else
    {
      lo[k] = node_lo[c[k]];
      hi[k] = node_hi[c[k]];
      int cc = __float_as_int(lo[k].w);
      ref[k] = (cc <= leaf_max) ? leaf_ref(range_first[c[k]], cc) : c[k];
    }
  }
  out_nodes[4 * (size_t)i + 0] = make_float4(lo[0].x - pad, hi[0].x + pad, lo[0].y - pad, hi[0].y + pad);
  out_nodes[4 * (size_t)i + 1] = make_float4(lo[1].x - pad, hi[1].x + pad, lo[1].y - pad, hi[1].y + pad);
  out_nodes[4 * (size_t)i + 2] = make_float4(lo[0].z - pad, hi[0].z + pad, lo[1].z - pad, hi[1].z + pad);
  out_nodes[4 * (size_t)i + 3] = make_float4(__int_as_float(ref[0]), __int_as_float(ref[1]), 0.0f, 0.0f);
  atomicAdd(emitted, 1);
}

/* BVH4 by greedy collapse of the BVH2, one launch per BVH4 level.
 * A work item is {BVH2 node that becomes a BVH4 node, index of that BVH4 node}.  The item starts
 * with the node's two children and, while it has fewer than four, replaces the INNER child with
 * the largest surface area by that child's two children (Wald et al. 2008).  Inner children get
 * consecutive BVH4 indices from one atomicAdd (siblings are adjacent) and go to the next level's
 * queue, so the node arrays are dense and in breadth-first order: the top of the tree is one
 * contiguous block. */
struct Emit4Queues
{
  int2 *items[2]; /* {bvh2 node, bvh4 index} */
  int *counts;    /* [64 + 1] items per level */
  int *n_nodes;   /* BVH4 nodes allocated so far */
};

__global__ void k_emit4_seed(Emit4Queues q)
{
  q.items[0][0] = make_int2(0, 0);
  q.counts[0] = 1;
  *q.n_nodes = 1;
}

__global__ void k_emit4(const unsigned *__restrict__ vals, const float4 *__restrict__ box_lo,
                        const float4 *__restrict__ box_hi, int n, const int2 *__restrict__ children,
                        const int *__restrict__ range_first, const float4 *__restrict__ node_lo,
                        const float4 *__restrict__ node_hi, const BuildParams *__restrict__ bp,
                        float4 *__restrict__ out_nodes, float4 *__restrict__ out_nodes_q, Emit4Queues q, int level,
                        int leaf_max, int dummy_ref)
{
  const int item = blockIdx.x * blockDim.x + threadIdx.x;
  if (item >= q.counts[level])
    return;
  const int2 work = q.items[level & 1][item];
  const int i = work.y; /* index of the BVH4 node written here */

  /* candidate children as BVH2 references: < 0 single primitive, >= 0 BVH2 inner node */
  int cand[4];
  int m = 2;
  {
    const int2 ch = children[work.x];
    cand[0] = ch.x;
    cand[1] = ch.y;
  }
  auto is_inner = [&](int c) { return c >= 0 && __float_as_int(node_lo[c].w) > leaf_max; };
  auto area = [&](int c) {
    const float4 a = node_lo[c], b = node_hi[c];
    const float dx = b.x - a.x, dy = b.y - a.y, dz = b.z - a.z;
    return dx * dy + dy * dz + dz * dx;
  };
  while (m < 4)
  {
    int pick = -1;
    float best = -1.0f;
    for (int k = 0; k < m; k++)
      if (is_inner(cand[k]))
      {
        const float ar = area(cand[k]);
        if (ar > best)
        {
          best = ar;
          pick = k;
        }
      }
    if (pick < 0)
      break;
    const int2 g = children[cand[pick]];
    cand[pick] = g.x;
    cand[m++] = g.y;
  }
  int n_inner = 0;
  for (int k = 0; k < m; k++)
    n_inner += is_inner(cand[k]) ? 1 : 0;
  int child_index = 0, slot = 0;
  if (n_inner > 0)
  {
    child_index = atomicAdd(q.n_nodes, n_inner);
    slot = atomicAdd(&q.counts[level + 1], n_inner);
  }

  const float pad = bp->pad;
  float lo[4][3], hi[4][3];
  int ref[4];
  for (int k = 0; k < m; k++)
  {
    const int c = cand[k];
    float4 a, b;
    int r;
    if (c < 0)
    {
      unsigned p = vals[~c];
      a = box_lo[p]; b = box_hi[p];
      r = leaf_ref(~c, 1);
    }
    else
    {
      a = node_lo[c]; b = node_hi[c];
      int cc = __float_as_int(a.w);
      if (cc <= leaf_max)
        r = leaf_ref(range_first[c], cc);
      else
      {
        r = child_index;
        q.items[(level + 1) & 1][slot] = make_int2(c, child_index);
        child_index++;
        slot++;
      }
    }
    lo[k][0] = a.x - pad; lo[k][1] = a.y - pad; lo[k][2] = a.z - pad;
    hi[k][0] = b.x + pad; hi[k][1] = b.y + pad; hi[k][2] = b.z + pad;
    ref[k] = r;
  }
  for (; m < 4; m++)
  {
    for (int a = 0; a < 3; a++) { lo[m][a] = 0.0f; hi[m][a] = 0.0f; }
    ref[m] = RTB_REF_NONE;
  }
  if (out_nodes) /* the uncompressed BVH4 is a parity probe (RTB_SCENE_ALL_TREES) */
  {
    float4 *o = out_nodes + 8 * (size_t)i;
    o[0] = make_float4(lo[0][0], lo[1][0], lo[2][0], lo[3][0]);
    o[1] = make_float4(hi[0][0], hi[1][0], hi[2][0], hi[3][0]);
    o[2] = make_float4(lo[0][1], lo[1][1], lo[2][1], lo[3][1]);
    o[3] = make_float4(hi[0][1], hi[1][1], hi[2][1], hi[3][1]);
    o[4] = make_float4(lo[0][2], lo[1][2], lo[2][2], lo[3][2]);
    o[5] = make_float4(hi[0][2], hi[1][2], hi[2][2], hi[3][2]);
    o[6] = make_float4(__int_as_float(ref[0]), __int_as_float(ref[1]), __int_as_float(ref[2]), __int_as_float(ref[3]));
    o[7] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  }

  /* compressed copy: per-node grid origin + q * 2^e, lo rounded down, hi rounded up */
  float org[3], cellf[3];
  unsigned qlo[3] = { 0u, 0u, 0u }, qhi[3] = { 0u, 0u, 0u };
  for (int a = 0; a < 3; a++)
  {
    float nlo = 3.0e38f, nhi = -3.0e38f;
    for (int k = 0; k < 4; k++)
      if (ref[k] != RTB_REF_NONE)
      {
        nlo = fminf(nlo, lo[k][a]);
        nhi = fmaxf(nhi, hi[k][a]);
      }
    org[a] = nlo;
    /* smallest power of two s with 255 * s >= extent (computed in double, then checked) */
    const double ext = (double)nhi - (double)nlo;
    int e = 0;
    frexp(ext / 255.0, &e); /* ext/255 = m * 2^e, m in [0.5, 1) -> 2^e >= ext/255 */
    if (!(ext > 0.0))
      e = -126;
    e = max(-126, min(127, e));
    double cell = ldexp(1.0, e);
    while (cell * 255.0 < ext && e < 127) { e++; cell = ldexp(1.0, e); }
    cellf[a] = (float)cell; /* a power of two in the normal range: exact */
    for (int k = 0; k < 4; k++)
    {
      unsigned ql = 255u, qh = 0u; /* empty slot: inverted box, never entered before it is left */
      if (ref[k] != RTB_REF_NONE)
      {
        double l = floor(((double)lo[k][a] - (double)nlo) / cell);
        double h = ceil(((double)hi[k][a] - (double)nlo) / cell);
        ql = (unsigned)fmin(fmax(l, 0.0), 255.0);
        qh = (unsigned)fmin(fmax(h, 0.0), 255.0);
      }
      qlo[a] |= ql << (8 * k);
      qhi[a] |= qh << (8 * k);
    }
  }
  /* an empty slot refers to the degenerate triangle stored behind the last primitive */
  for (int k = 0; k < 4; k++)
    if (ref[k] == RTB_REF_NONE)
      ref[k] = dummy_ref;
  float4 *oq = out_nodes_q + 4 * (size_t)i;
  oq[0] = make_float4(org[0], org[1], org[2], cellf[0]);
  oq[1] = make_float4(__int_as_float(ref[0]), __int_as_float(ref[1]), __int_as_float(ref[2]), __int_as_float(ref[3]));
  oq[2] = make_float4(__uint_as_float(qlo[0]), __uint_as_float(qlo[1]), __uint_as_float(qlo[2]), __uint_as_float(qhi[0]));
  oq[3] = make_float4(__uint_as_float(qhi[1]), __uint_as_float(qhi[2]), cellf[1], cellf[2]);
}

__global__ void k_reorder(const unsigned *__restrict__ vals, int n, const PrimRec *__restrict__ in,
                          PrimRec *__restrict__ out, const float2 *__restrict__ tex_in, float2 *__restrict__ tex_out)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n)
    return;
  unsigned p = vals[i];
  out[i] = in[p];
  if (tex_in)
  {
    tex_out[3 * (size_t)i + 0] = tex_in[3 * (size_t)p + 0];
    tex_out[3 * (size_t)i + 1] = tex_in[3 * (size_t)p + 1];
    tex_out[3 * (size_t)i + 2] = tex_in[3 * (size_t)p + 2];
  }
}

/* W doubles per primitive: 9 (tri64) or 6 (tex64) */
template <int W>
__global__ void k_reorder64(const unsigned *__restrict__ vals, int n, const double *__restrict__ in, double *__restrict__ out)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n)
    return;
  const unsigned p = vals ? vals[i] : (unsigned)i;
  for (int k = 0; k < W; k++)
    out[W * (size_t)i + k] = in[W * (size_t)p + k];
}

/* ---- host side ------------------------------------------------------------------- */

namespace
{
struct MeshRange
{
  const RefVertex *verts;
  size_t n_tris;
  int obj;
  long long gid_first;
  bool checkered;
};

struct HostScene
{
  std::vector<SphereIn> spheres;
  std::vector<MeshRange> meshes;
  std::vector<float4> mats; /* 2 per object */
  std::vector<double> colors; /* 3 per object, unscaled (cast_ray reads objects[i].color, raytracer.c:575) */
  size_t n_objects = 0;
  long long n_prims = 0;
};

/* Stream-ordered, pooled device memory.  cudaMalloc/cudaFree cost 1-100+ ms each on this
 * platform (measured: scene create 126..1145 ms for 0.6 ms of kernels), so every buffer --
 * temporaries and the scene's own arrays -- comes from the device's default memory pool with
 * an unlimited release threshold: after the first scene, create/destroy recycle pool memory. */
static cudaError_t pool_setup(int device)
{
  static std::atomic<bool> done[64]; /* zero-initialised */
  if (device < 64 && done[device].load())
    return cudaSuccess;
  cudaMemPool_t pool;
  cudaError_t e = cudaDeviceGetDefaultMemPool(&pool, device);
  if (e != cudaSuccess)
    return e;
  unsigned long long threshold = ~0ull;
  e = cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &threshold);
  if (e == cudaSuccess && device < 64)
    done[device].store(true);
  return e;
}

/* ---- host -> device upload of a caller's pageable array ------------------------------------------
 * The reference's driver malloc()s its scene (main.c:413), so the 120 MB of Vertex records of C3 arrive in
 * pageable memory: one cudaMemcpy of it runs at the speed of the driver's single staging thread (~10 GB/s,
 * 12 ms), a quarter of the PCIe link.  Here a few host threads copy interleaved 4 MB chunks into their own
 * page-locked double buffers and DMA them from there, each on its own stream.  The streams are ordinary
 * (blocking) streams: work on the legacy default stream -- the marshalling kernel -- orders itself after them. */
namespace
{
const size_t kStageChunk = 4u << 20;
const int kStageMaxThreads = 16;
struct StageLane
{
  char *pinned[2] = { nullptr, nullptr };
  cudaStream_t stream = nullptr;
  cudaEvent_t done[2] = { nullptr, nullptr };
};
struct StagePool
{
  std::mutex mutex; /* one upload at a time per device */
  StageLane lanes[kStageMaxThreads];
  int ready = 0;
};
StagePool g_stage[64];

cudaError_t stage_lane_init(StageLane &l)
{
  for (int k = 0; k < 2; k++)
  {
    cudaError_t e = cudaHostAlloc(reinterpret_cast<void **>(&l.pinned[k]), kStageChunk, cudaHostAllocDefault);
    if (e != cudaSuccess) return e;
    e = cudaEventCreateWithFlags(&l.done[k], cudaEventDisableTiming);
    if (e != cudaSuccess) return e;
  }
  return cudaStreamCreate(&l.stream);
}

cudaError_t upload_pageable(int device, void *dst, const void *src, size_t bytes, int threads)
{
  cudaPointerAttributes attr;
  const bool host_pinned = cudaPointerGetAttributes(&attr, src) == cudaSuccess && attr.type == cudaMemoryTypeHost;
  cudaGetLastError(); /* an unregistered pointer is not an error */
  threads = std::max(1, std::min(threads, kStageMaxThreads));
  if (host_pinned || bytes < 2 * kStageChunk || threads < 2 || device < 0 || device >= 64)
    return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, 0);
  StagePool &pool = g_stage[device];
  std::lock_guard<std::mutex> lock(pool.mutex);
  for (; pool.ready < threads; pool.ready++)
  {
    cudaError_t e = stage_lane_init(pool.lanes[pool.ready]);
    if (e != cudaSuccess)
      return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, 0); /* no page-locked memory left: plain copy */
  }
  const size_t n_chunks = (bytes + kStageChunk - 1) / kStageChunk;
  std::vector<cudaError_t> err((size_t)threads, cudaSuccess);
  std::vector<std::thread> workers;
  for (int t = 0; t < threads; t++)
    workers.emplace_back([&, t]() {
      cudaError_t e = cudaSetDevice(device);
      StageLane &l = pool.lanes[t];
      int turn = 0;
      for (size_t c = (size_t)t; c < n_chunks && e == cudaSuccess; c += (size_t)threads, turn++)
      {
        const int slot = turn & 1;
        if (turn >= 2)
          e = cudaEventSynchronize(l.done[slot]); /* the DMA that last read this buffer */
        const size_t off = c * kStageChunk, len = std::min(kStageChunk, bytes - off);
        memcpy(l.pinned[slot], static_cast<const char *>(src) + off, len);
        if (e == cudaSuccess)
          e = cudaMemcpyAsync(static_cast<char *>(dst) + off, l.pinned[slot], len, cudaMemcpyHostToDevice, l.stream);
        if (e == cudaSuccess)
          e = cudaEventRecord(l.done[slot], l.stream);
      }
      /* the buffers may be refilled by the next upload only after their DMAs: wait here, the copies of the
       * other lanes keep the link busy meanwhile */
      if (e == cudaSuccess)
        e = cudaStreamSynchronize(l.stream);
      err[(size_t)t] = e;
    });
  for (std::thread &w : workers)
    w.join();
  for (cudaError_t e : err)
    if (e != cudaSuccess)
      return e;
  return cudaSuccess;
}

/* The narrowed form of upload_pageable for Vertex records (rtb_narrow.cpp): the staging threads convert the five
 * doubles of a vertex to five floats while they copy, so the host writes and the link carries 60 B per triangle
 * instead of 120 B.  *exact = false when some coordinate is not float-representable: the device buffer then holds
 * garbage and the caller uploads the piece as raw doubles (upload_pageable).  Returns cudaErrorNotSupported when
 * the piece is not worth it or no page-locked memory is left (same fallback). */
cudaError_t upload_narrowed(int device, float *dst, const RefVertex *src, size_t n_vertices, int threads, bool *exact)
{
  *exact = true;
  cudaPointerAttributes attr;
  const bool host_pinned = cudaPointerGetAttributes(&attr, src) == cudaSuccess && attr.type == cudaMemoryTypeHost;
  cudaGetLastError();
  threads = std::max(1, std::min(threads, kStageMaxThreads));
  /* whole triangles and whole groups of four vertices per chunk; small uploads get small chunks so that the
   * first DMA starts early */
  const size_t max_chunk = (kStageChunk / (5 * sizeof(float))) / 12 * 12;
  size_t chunk = std::min(max_chunk, std::max<size_t>(12288, n_vertices / ((size_t)threads * 4) / 12 * 12));
  if (host_pinned || n_vertices < 24576 || device < 0 || device >= 64)
    return cudaErrorNotSupported;
  StagePool &pool = g_stage[device];
  std::lock_guard<std::mutex> lock(pool.mutex);
  for (; pool.ready < threads; pool.ready++)
    if (stage_lane_init(pool.lanes[pool.ready]) != cudaSuccess)
    {
      cudaGetLastError();
      return cudaErrorNotSupported;
    }
  const size_t n_chunks = (n_vertices + chunk - 1) / chunk;
  std::vector<cudaError_t> err((size_t)threads, cudaSuccess);
  std::atomic<bool> inexact(false);
  std::vector<std::thread> workers;
  for (int t = 0; t < threads; t++)
    workers.emplace_back([&, t]() {
      cudaError_t e = cudaSetDevice(device);
      StageLane &l = pool.lanes[t];
      int turn = 0;
      for (size_t c = (size_t)t; c < n_chunks && e == cudaSuccess && !inexact.load(std::memory_order_relaxed);
           c += (size_t)threads, turn++)
      {
        const int slot = turn & 1;
        if (turn >= 2)
          e = cudaEventSynchronize(l.done[slot]); /* the DMA that last read this buffer */
        const size_t first = c * chunk, cnt = std::min(chunk, n_vertices - first);
        if (!rtb_narrow_vertices(reinterpret_cast<const double *>(src + first), reinterpret_cast<float *>(l.pinned[slot]), cnt))
          inexact.store(true, std::memory_order_relaxed);
        if (e == cudaSuccess)
          e = cudaMemcpyAsync(dst + 5 * first, l.pinned[slot], 5 * sizeof(float) * cnt, cudaMemcpyHostToDevice, l.stream);
        if (e == cudaSuccess)
          e = cudaEventRecord(l.done[slot], l.stream);
      }
      if (e == cudaSuccess)
        e = cudaStreamSynchronize(l.stream);
      err[(size_t)t] = e;
    });
  for (std::thread &w : workers)
    w.join();
  for (cudaError_t e : err)
    if (e != cudaSuccess)
      return e;
  *exact = !inexact.load();
  return cudaSuccess;
}
} // namespace

/* The build reads a few words back (scene box, tree depth, node count, flags).  Into pageable memory every such
 * copy is a host wait in the middle of the build; into a page-locked block they are asynchronous, and the whole
 * build -- ~90 launches -- is enqueued behind the upload without the GPU ever waiting for the host. */
struct BuildReadback
{
  BuildParams bp;
  int levels[RTB_STACK_SIZE + 2];
  int misc[2];
  int nodes4;
  int inexact[2]; /* some position / some texture coordinate is not float-representable */
};

namespace
{
std::mutex g_readback_mutex;
std::vector<BuildReadback *> g_readback_free;

struct ReadbackLease
{
  BuildReadback *p = nullptr;
  ReadbackLease()
  {
    {
      std::lock_guard<std::mutex> lock(g_readback_mutex);
      if (!g_readback_free.empty())
      {
        p = g_readback_free.back();
        g_readback_free.pop_back();
      }
    }
    if (!p && cudaHostAlloc(reinterpret_cast<void **>(&p), sizeof(BuildReadback), cudaHostAllocPortable) != cudaSuccess)
    {
      cudaGetLastError();
      p = nullptr;
    }
    if (p)
      memset(p, 0, sizeof(*p));
  }
  ~ReadbackLease()
  {
    if (p)
    {
      std::lock_guard<std::mutex> lock(g_readback_mutex);
      g_readback_free.push_back(p);
    }
  }
};
} // namespace

template <typename T>
struct DevBuf
{
  T *p = nullptr;
  ~DevBuf() { if (p) cudaFreeAsync(p, 0); }
  cudaError_t alloc(size_t n) { return cudaMallocAsync(reinterpret_cast<void **>(&p), sizeof(T) * (n ? n : 1), 0); }
  T *release() { T *q = p; p = nullptr; return q; }
};

template <typename T>
static cudaError_t pool_alloc(T **p, size_t n)
{
  return cudaMallocAsync(reinterpret_cast<void **>(p), sizeof(T) * (n ? n : 1), 0);
}

/* a buffer that lives as long as the scene: from the per-device cache if one fits, else from the pool */
template <typename T>
static cudaError_t scene_alloc(rtb_scene *sc, T **p, size_t n)
{
  const size_t need = sizeof(T) * (n ? n : 1);
  size_t got = 0;
  if (void *q = rtb_cache_take(sc->device, need, &got))
  {
    *p = static_cast<T *>(q);
    sc->owned.emplace_back(q, got);
    return cudaSuccess;
  }
  cudaError_t e = pool_alloc(p, n);
  if (e == cudaSuccess)
    sc->owned.emplace_back(static_cast<void *>(*p), need);
  return e;
}

void push_material(HostScene &hs, uint32_t flags, const RefVec3 &color, const RefVec3 &emission)
{
  /* Russian roulette (raytracer.c:497-502): survive iff u < prob with u = r31 / 2^31, i.e.
   * iff r31 < ceil(prob * 2^31) -- an integer threshold, so the decision is exact.  The
   * surviving albedo albedo * (1/prob) is computed in double, then rounded once. */
  double prob = std::max(color.x, std::max(color.y, color.z)); /* MAX(a.x, MAX(a.y, a.z)) */
  uint32_t threshold;
  if (!(prob > 0.0)) threshold = 0u; /* also NaN: `u < NaN` is false upstream */
  else if (prob >= 1.0) threshold = 0x80000000u;
  else threshold = (uint32_t)std::ceil(prob * 2147483648.0);
  double inv = 1 / prob;
  float ax = (float)(color.x * inv), ay = (float)(color.y * inv), az = (float)(color.z * inv);
  if (threshold == 0u) ax = ay = az = 0.0f;
  float4 m0, m1;
  m0.x = ax; m0.y = ay; m0.z = az;
  memcpy(&m0.w, &threshold, 4);
  m1.x = (float)emission.x; m1.y = (float)emission.y; m1.z = (float)emission.z;
  memcpy(&m1.w, &flags, 4);
  hs.mats.push_back(m0);
  hs.mats.push_back(m1);
  hs.colors.push_back(color.x);
  hs.colors.push_back(color.y);
  hs.colors.push_back(color.z);
}

int gather_scene_objects(const RefSceneObject *objs, size_t n, HostScene &hs)
{
  hs.n_objects = n;
  long long gid = 0;
  for (size_t i = 0; i < n; i++)
  {
    const RefSceneObject &o = objs[i];
    push_material(hs, o.material.flags, o.material.color, o.material.emission);
    if (o.type == 0)
    {
      const RefSphere *s = static_cast<const RefSphere *>(o.geometry);
      if (!s) { rtb_set_error("sphere object with NULL geometry"); return RTB_EINVAL; }
      hs.spheres.push_back(SphereIn{ s->center.x, s->center.y, s->center.z, s->radius, (int)i, (int)gid });
      gid += 1;
    }
    else if (o.type == 1)
    {
      const RefMesh *m = static_cast<const RefMesh *>(o.geometry);
      if (!m) { rtb_set_error("mesh object with NULL geometry"); return RTB_EINVAL; }
      if (m->num_triangles > 0)
      {
        if (!m->vertices) { rtb_set_error("mesh with NULL vertices"); return RTB_EINVAL; }
        hs.meshes.push_back(MeshRange{ m->vertices, m->num_triangles, (int)i, gid,
                                       (o.material.flags & RT_M_CHECKERED) != 0 });
        gid += (long long)m->num_triangles;
      }
    }
    else
    {
      rtb_set_error("unknown geometry type"); /* raytracer.c:449-453 exits here */
      return RTB_EINVAL;
    }
  }
  hs.n_prims = gid;
  if (gid >= (1ll << 27) || n >= (1ull << 30))
  {
    rtb_set_error("scene too large (>= 2^27 primitives)");
    return RTB_EINVAL;
  }
  return RTB_OK;
}

/* pick the oversized spheres (see file header): radius > 32 x the median primitive size,
 * at most 32 of them, largest first */
std::vector<char> choose_big(const HostScene &hs)
{
  std::vector<char> big(hs.spheres.size(), 0);
  std::vector<double> sizes;
  for (const SphereIn &s : hs.spheres)
    sizes.push_back(std::fabs(s.r));
  for (const MeshRange &m : hs.meshes)
  {
    size_t step = std::max<size_t>(1, m.n_tris / 2048);
    for (size_t t = 0; t < m.n_tris; t += step)
    {
      const RefVertex *v = m.verts + 3 * t;
      double ext = 0;
      for (int a = 0; a < 3; a++)
      {
        const double *p0 = &v[0].pos.x, *p1 = &v[1].pos.x, *p2 = &v[2].pos.x;
        double lo = std::min(p0[a], std::min(p1[a], p2[a])), hi = std::max(p0[a], std::max(p1[a], p2[a]));
        ext = std::max(ext, hi - lo);
      }
      /* weight a sampled triangle by the triangles it stands for */
      for (size_t r = 0; r < std::min<size_t>(step, 64); r++)
        sizes.push_back(0.5 * ext);
    }
  }
  if (sizes.size() < 2)
    return big;
  std::vector<double> sorted = sizes;
  std::nth_element(sorted.begin(), sorted.begin() + (sorted.size() - 1) / 2, sorted.end());
  double median = sorted[(sorted.size() - 1) / 2];
  double ratio = 32.0;
  if (const char *e = getenv("RTB_BIG_RATIO"))
    ratio = atof(e);
  double threshold = ratio * median;
  std::vector<std::pair<double, size_t>> cand;
  for (size_t i = 0; i < hs.spheres.size(); i++)
    if (std::fabs(hs.spheres[i].r) > threshold || !std::isfinite(hs.spheres[i].r))
      cand.push_back({ std::fabs(hs.spheres[i].r), i });
  std::sort(cand.begin(), cand.end(), [](const std::pair<double, size_t> &a, const std::pair<double, size_t> &b) {
    return a.first > b.first || (a.first == b.first && a.second < b.second);
  });
  /* at most 32: big_list_select_test keeps its candidates in a 32-bit mask.  Further oversized spheres
   * stay in the tree: correct, only slower (tests/test_gpu_parity.py::test_many_oversized_spheres) */
  for (size_t k = 0; k < cand.size() && k < 32; k++)
    big[cand[k].second] = 1;
  return big;
}

int build_scene(HostScene &hs, int device, unsigned flags, const rtb_scene_shard *shard, rtb_scene **out)
{
  const bool all_trees = (flags & RTB_SCENE_ALL_TREES) != 0;
  int ndev = 0;
  RTB_CUDA(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev)
  {
    rtb_set_error("invalid CUDA device ordinal");
    return RTB_EINVAL;
  }
  RTB_CUDA(cudaSetDevice(device));
  RTB_CUDA(pool_setup(device));

  struct EventPair /* destroyed on every return path */
  {
    cudaEvent_t a = nullptr, b = nullptr;
    ~EventPair()
    {
      if (a) cudaEventDestroy(a);
      if (b) cudaEventDestroy(b);
    }
  } evp;
  cudaEvent_t &ev0 = evp.a, &ev1 = evp.b;
  RTB_CUDA(cudaEventCreate(&ev0));
  RTB_CUDA(cudaEventCreate(&ev1));
  RTB_CUDA(cudaEventRecord(ev0, 0));
  /* development aid ($RTB_TIMING): where the build spends its time; the marks synchronise, so the sum is longer
   * than an unobserved build */
  const bool timing = getenv("RTB_TIMING") != nullptr;
  std::vector<std::pair<const char *, double>> marks;
  auto mark = [&](const char *what) {
    if (!timing)
      return;
    cudaStreamSynchronize(0);
    marks.emplace_back(what, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count());
  };
  mark("start");

  /* development knobs (documented in DESIGN.md): leaf size and oversized-primitive ratio */
  /* measured on B200 (profiles/r1_tuning.md): sphere scenes are fastest with one sphere per
   * leaf (the exact test is cheap to skip, a leaf visit is not), meshes with two triangles */
  int leaf_max = hs.meshes.empty() ? 1 : 2;
  if (const char *e = getenv("RTB_LEAF_MAX"))
    leaf_max = std::max(1, std::min(8, atoi(e)));
  /* NaN would break choose_big's ordering (a NaN radius is a candidate); triangles are checked on the device */
  for (const SphereIn &s : hs.spheres)
    if (std::isnan(s.cx) || std::isnan(s.cy) || std::isnan(s.cz) || std::isnan(s.r))
    {
      rtb_set_error("non-finite geometry");
      return RTB_EINVAL;
    }
  std::vector<char> big = choose_big(hs);
  std::vector<SphereIn> big_spheres, bvh_spheres;
  for (size_t i = 0; i < hs.spheres.size(); i++)
    (big[i] ? big_spheres : bvh_spheres).push_back(hs.spheres[i]);
  size_t n_tris = 0;
  for (const MeshRange &m : hs.meshes)
    n_tris += m.n_tris;
  /* texcoords ride along with every mesh (24 B/triangle, only read for M_CHECKERED) */
  const bool want_tex = n_tris > 0;
  const size_t n_bs = bvh_spheres.size();
  const size_t N = n_bs + n_tris; /* primitives in the tree */

  struct SceneDeleter { void operator()(rtb_scene *s) const { rtb_scene_destroy(s); } };
  std::unique_ptr<rtb_scene, SceneDeleter> sc(new rtb_scene());
  sc->device = device;
  size_t dev_bytes = 0;

  /* materials, counters, big list */
  RTB_CUDA(scene_alloc(sc.get(), &sc->d_mats, std::max<size_t>(2, hs.mats.size())));
  if (!hs.mats.empty())
    RTB_CUDA(cudaMemcpyAsync(sc->d_mats, hs.mats.data(), sizeof(float4) * hs.mats.size(), cudaMemcpyHostToDevice, 0));
  dev_bytes += sizeof(float4) * hs.mats.size();
  RTB_CUDA(scene_alloc(sc.get(), &sc->d_colors, std::max<size_t>(3, hs.colors.size())));
  if (!hs.colors.empty())
    RTB_CUDA(cudaMemcpyAsync(sc->d_colors, hs.colors.data(), sizeof(double) * hs.colors.size(), cudaMemcpyHostToDevice, 0));
  dev_bytes += sizeof(double) * hs.colors.size();
  RTB_CUDA(scene_alloc(sc.get(), &sc->d_counters, 8));
  /* 3 float4 per record, followed by 2 float4 per FP32 copy */
  RTB_CUDA(scene_alloc(sc.get(), &sc->d_big, 5 * std::max<size_t>(1, big_spheres.size())));
  DevBuf<SphereIn> d_big_in, d_bvh_in;
  if (!big_spheres.empty())
  {
    RTB_CUDA(d_big_in.alloc(big_spheres.size()));
    RTB_CUDA(cudaMemcpyAsync(d_big_in.p, big_spheres.data(), sizeof(SphereIn) * big_spheres.size(), cudaMemcpyHostToDevice, 0));
    k_marshal_spheres<<<1, 32>>>(d_big_in.p, (int)big_spheres.size(), reinterpret_cast<PrimRec *>(sc->d_big), nullptr, nullptr,
                                 sc->d_big + 3 * big_spheres.size());
    RTB_CUDA(cudaGetLastError());
  }
  dev_bytes += sizeof(PrimRec) * big_spheres.size();

  SceneView &view = sc->view;
  view.n_big = (int)big_spheres.size();
  view.n_objects = (int)hs.n_objects;
  view.n_prims = (int)N;
  view.root_ref = RTB_REF_NONE;
  view.tex = nullptr;
  for (int k = 0; k < 3; k++)
  {
    view.guard_lo[k] = -FLT_MAX;
    view.guard_hi[k] = FLT_MAX;
  }
  view.far_t = FLT_MAX;
  int bvh_depth = 0;
  size_t n_nodes = 0;

  /* every temporary lives until the end of this function; frees are stream-ordered */
  DevBuf<PrimRec> d_unsorted;
  DevBuf<float4> d_lo, d_hi, d_node_lo, d_node_hi;
  DevBuf<float2> d_tex_unsorted;
  DevBuf<double> d_tri64_unsorted; /* triangle vertices as given; kept only if some are not float-representable */
  DevBuf<double> d_tex64_unsorted; /* texture coordinates as given; the same */
  DevBuf<int> d_inexact;           /* [0] positions, [1] texture coordinates */
  ReadbackLease lease; /* page-locked: the read-backs below never make the host wait */
  if (!lease.p)
  {
    rtb_set_error("no page-locked memory for the build's read-back block");
    return RTB_ENOMEM;
  }
  BuildReadback &rb = *lease.p;
  int &h_inexact = rb.inexact[0];
  int &h_tex_inexact = rb.inexact[1];
  DevBuf<RefVertex> d_stage;
  std::vector<std::pair<size_t, size_t>> narrowed; /* (first slot, triangles) of the pieces uploaded as floats */
  DevBuf<unsigned> d_bounds, d_vals, d_vals_sorted;
  DevBuf<BuildParams> d_bp;
  DevBuf<unsigned long long> d_keys, d_keys_sorted;
  DevBuf<unsigned char> d_temp;
  DevBuf<int2> d_children;
  DevBuf<int> d_parent_inner, d_parent_leaf, d_first, d_flags, d_misc, d_misc4, d_level_counts;
  DevBuf<int2> d_items_a, d_items_b;
  int *const h_levels = rb.levels;
  BuildParams &h_bp = rb.bp;
  int *const h_misc = rb.misc;
  int &h_nodes4 = rb.nodes4;
  bool bvh4_ok = true;
  int depth4 = 0; /* levels of the BVH4 */
  int emitted_levels = 0; /* BVH4 levels k_emit4 ran for */

  if (N > 0)
  {
    const int T = 256;
    const int blocks = (int)((N + T - 1) / T);
    /* Sharded upload (rtb_multi.cu): with G ranks on one box every rank uploads and marshals only its
     * 1/G of the triangles (120 B each over PCIe) and the marshalled records (104 B each) are
     * all-gathered over NVLink, instead of every GPU pulling the whole mesh through its own PCIe link.
     * The arrays are padded to G equal chunks so the gather can run in place. */
    const bool sharded = shard != nullptr && shard->n_ranks > 1 && n_tris >= (size_t)shard->n_ranks * 4096;
    const size_t G = sharded ? (size_t)shard->n_ranks : 1;
    const size_t tri_chunk = (n_tris + G - 1) / G;
    const size_t N_alloc = n_bs + tri_chunk * G;
    RTB_CUDA(d_unsorted.alloc(N_alloc));
    RTB_CUDA(d_lo.alloc(N_alloc));
    RTB_CUDA(d_hi.alloc(N_alloc));
    if (n_tris)
    {
      RTB_CUDA(d_tri64_unsorted.alloc(9 * N_alloc));
      RTB_CUDA(d_tex64_unsorted.alloc(6 * N_alloc));
      RTB_CUDA(d_inexact.alloc(2));
      RTB_CUDA(cudaMemsetAsync(d_inexact.p, 0, sizeof(int) * 2, 0));
    }
    if (want_tex)
    {
      RTB_CUDA(d_tex_unsorted.alloc(3 * N_alloc));
      if (n_bs)
        RTB_CUDA(cudaMemsetAsync(d_tex_unsorted.p, 0, sizeof(float2) * 3 * n_bs, 0));
    }
    if (n_bs)
    {
      RTB_CUDA(d_bvh_in.alloc(n_bs));
      RTB_CUDA(cudaMemcpyAsync(d_bvh_in.p, bvh_spheres.data(), sizeof(SphereIn) * n_bs, cudaMemcpyHostToDevice, 0));
      k_marshal_spheres<<<(int)((n_bs + T - 1) / T), T>>>(d_bvh_in.p, (int)n_bs, d_unsorted.p, d_lo.p, d_hi.p, nullptr);
      RTB_CUDA(cudaGetLastError());
    }
    {
      /* raw Vertex arrays go up as they are (120 B per triangle) and are converted on the
       * device; staging is bounded so huge meshes do not double their footprint */
      const size_t chunk_tris = 1u << 21;
      /* host threads staging the pageable vertex array (see upload_pageable); ranks of one box share the host */
      const int host_cores = std::max(1, (int)std::thread::hardware_concurrency());
      int upload_threads = std::max(2, std::min(8, host_cores / (int)G));
      if (const char *e = getenv("RTB_UPLOAD_THREADS"))
        upload_threads = atoi(e);
      /* narrowing pays when enough threads on the box share the conversion (measured on the B200 box, C3's 120 MB:
       * 8 threads 5.3 -> 4.4 ms, under the 4.5 ms of a page-locked source; 2 ranks x 2 threads lose 15 % to a plain
       * copy: one thread converts more slowly than it copies, many threads are bound by the host's memory system,
       * where the narrowed form moves a third less).  Development knob: RTB_UPLOAD_NARROW=0 / 1 */
      bool narrow_upload = upload_threads * (int)G >= 6;
      if (const char *e = getenv("RTB_UPLOAD_NARROW"))
        narrow_upload = atoi(e) != 0;
      /* this rank's share of the concatenated triangle list: everything, or chunk `rank` of G */
      const size_t my_first = sharded ? std::min(n_tris, tri_chunk * (size_t)shard->rank) : 0;
      const size_t my_end = sharded ? std::min(n_tris, my_first + tri_chunk) : n_tris;
      size_t max_chunk = 0, tri_first = 0;
      for (const MeshRange &m : hs.meshes)
      {
        const size_t lo = std::max(tri_first, my_first), hi = std::min(tri_first + m.n_tris, my_end);
        if (hi > lo)
          max_chunk = std::max(max_chunk, std::min(chunk_tris, hi - lo));
        tri_first += m.n_tris;
      }
      if (max_chunk)
        RTB_CUDA(d_stage.alloc(3 * max_chunk));
      tri_first = 0;
      for (const MeshRange &m : hs.meshes)
      {
        const size_t lo = std::max(tri_first, my_first), hi = std::min(tri_first + m.n_tris, my_end);
        for (size_t g0 = lo; g0 < hi; g0 += chunk_tris)
        {
          const size_t cnt = std::min(chunk_tris, hi - g0);
          const size_t t0 = g0 - tri_first;    /* first triangle of the piece inside its mesh */
          const size_t offset = n_bs + g0;     /* its slot in the (unsorted) primitive arrays */
          /* narrowed (60 B per triangle, converted by the staging threads) when every coordinate of the piece is
           * float-representable, else as raw doubles (120 B) */
          bool exact = false;
          cudaError_t ne = narrow_upload ? upload_narrowed(device, reinterpret_cast<float *>(d_stage.p), m.verts + 3 * t0,
                                                           3 * cnt, upload_threads, &exact)
                                         : cudaErrorNotSupported;
          if (ne != cudaSuccess && ne != cudaErrorNotSupported)
            RTB_CUDA(ne);
          if (ne == cudaSuccess && exact)
          {
            k_marshal_tris_f32<<<(int)((cnt + T - 1) / T), T>>>(reinterpret_cast<const float *>(d_stage.p), (int)cnt, m.obj,
                                                                (int)(m.gid_first + (long long)t0), d_unsorted.p + offset,
                                                                d_lo.p + offset, d_hi.p + offset,
                                                                want_tex ? d_tex_unsorted.p + 3 * offset : nullptr);
            RTB_CUDA(cudaGetLastError());
            narrowed.emplace_back(offset, cnt);
            continue;
          }
          RTB_CUDA(upload_pageable(device, d_stage.p, m.verts + 3 * t0, sizeof(RefVertex) * 3 * cnt, upload_threads));
          k_marshal_tris<<<(int)((cnt + T - 1) / T), T>>>(d_stage.p, (int)cnt, m.obj, (int)(m.gid_first + (long long)t0),
                                                          d_unsorted.p + offset, d_lo.p + offset, d_hi.p + offset,
                                                          want_tex ? d_tex_unsorted.p + 3 * offset : nullptr,
                                                          d_tri64_unsorted.p + 9 * offset, d_tex64_unsorted.p + 6 * offset,
                                                          d_inexact.p);
          RTB_CUDA(cudaGetLastError());
        }
        tri_first += m.n_tris;
      }
      mark("upload + marshal");
      if (sharded)
      {
        /* one NCCL group: the four gathers and the max of the two "needs doubles" flags; no host wait */
        int grc = rtb_shard_allgather(shard, d_unsorted.p + n_bs, sizeof(PrimRec) * tri_chunk, d_lo.p + n_bs, d_hi.p + n_bs,
                                      sizeof(float4) * tri_chunk, want_tex ? d_tex_unsorted.p + 3 * n_bs : nullptr,
                                      sizeof(float2) * 3 * tri_chunk, d_inexact.p);
        if (grc != RTB_OK)
          return grc;
      }
      if (n_tris)
        RTB_CUDA(cudaMemcpyAsync(rb.inexact, d_inexact.p, sizeof(int) * 2, cudaMemcpyDeviceToHost, 0));
      mark("all-gather");
    }

    /* scene box -> guard box, padding, Morton grid (all on the device) */
    RTB_CUDA(d_bounds.alloc(6));
    RTB_CUDA(d_bp.alloc(1));
    static const unsigned init_bounds[6] = { 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0u, 0u, 0u };
    RTB_CUDA(cudaMemcpyAsync(d_bounds.p, init_bounds, sizeof(init_bounds), cudaMemcpyHostToDevice, 0));
    k_bounds<<<std::min(blocks, 1184), T>>>(d_lo.p, d_hi.p, (int)N, d_bounds.p);
    RTB_CUDA(cudaGetLastError());
    k_build_params<<<1, 32>>>(d_bounds.p, d_bp.p);
    RTB_CUDA(cudaGetLastError());
    RTB_CUDA(cudaMemcpyAsync(&h_bp, d_bp.p, sizeof(h_bp), cudaMemcpyDeviceToHost, 0));

    /* one record more than primitives: the degenerate triangle empty BVH4 slots refer to */
    RTB_CUDA(scene_alloc(sc.get(), &sc->d_prims, 3 * (N + 1)));
    RTB_CUDA(cudaMemsetAsync(sc->d_prims + 3 * N, 0, sizeof(PrimRec), 0)); /* all-zero triangle: det = 0, never hit */
    if (want_tex)
      RTB_CUDA(scene_alloc(sc.get(), &sc->d_tex, 3 * N));

    if ((int)N <= leaf_max)
    {
      /* a single leaf; order = insertion order */
      RTB_CUDA(cudaMemcpyAsync(sc->d_prims, d_unsorted.p, sizeof(PrimRec) * N, cudaMemcpyDeviceToDevice, 0));
      if (want_tex)
        RTB_CUDA(cudaMemcpyAsync(sc->d_tex, d_tex_unsorted.p, sizeof(float2) * 3 * N, cudaMemcpyDeviceToDevice, 0));
      RTB_CUDA(scene_alloc(sc.get(), &sc->d_nodes, 4));
      view.root_ref = ~(((0) << 3) | ((int)N - 1));
    }
    else
    {
      RTB_CUDA(d_keys.alloc(N));
      RTB_CUDA(d_keys_sorted.alloc(N));
      RTB_CUDA(d_vals.alloc(N));
      RTB_CUDA(d_vals_sorted.alloc(N));
      k_morton<<<blocks, T>>>(d_lo.p, d_hi.p, (int)N, d_bp.p, d_keys.p, d_vals.p);
      RTB_CUDA(cudaGetLastError());
      size_t temp_bytes = 0;
      RTB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, d_keys.p, d_keys_sorted.p, d_vals.p,
                                               d_vals_sorted.p, (int)N, 0, 63, 0));
      RTB_CUDA(d_temp.alloc(temp_bytes));
      RTB_CUDA(cub::DeviceRadixSort::SortPairs(d_temp.p, temp_bytes, d_keys.p, d_keys_sorted.p, d_vals.p,
                                               d_vals_sorted.p, (int)N, 0, 63, 0));

      RTB_CUDA(d_children.alloc(N - 1));
      RTB_CUDA(d_parent_inner.alloc(N - 1));
      RTB_CUDA(d_parent_leaf.alloc(N));
      RTB_CUDA(d_first.alloc(N - 1));
      RTB_CUDA(d_flags.alloc(N - 1));
      RTB_CUDA(d_misc.alloc(2));
      RTB_CUDA(d_misc4.alloc(1));
      RTB_CUDA(cudaMemsetAsync(d_misc4.p, 0, sizeof(int), 0));
      RTB_CUDA(d_items_a.alloc(N));
      RTB_CUDA(d_items_b.alloc(N));
      RTB_CUDA(d_level_counts.alloc(RTB_STACK_SIZE + 2));
      RTB_CUDA(cudaMemsetAsync(d_level_counts.p, 0, sizeof(int) * (RTB_STACK_SIZE + 2), 0));
      RTB_CUDA(d_node_lo.alloc(N - 1));
      RTB_CUDA(d_node_hi.alloc(N - 1));
      RTB_CUDA(cudaMemsetAsync(d_flags.p, 0, sizeof(int) * (N - 1), 0));
      RTB_CUDA(cudaMemsetAsync(d_misc.p, 0, sizeof(int) * 2, 0));
      k_karras<<<blocks, T>>>(d_keys_sorted.p, (int)N, d_children.p, d_parent_inner.p, d_parent_leaf.p, d_first.p);
      RTB_CUDA(cudaGetLastError());
      k_fit<<<blocks, T>>>(d_vals_sorted.p, d_lo.p, d_hi.p, (int)N, d_children.p, d_parent_inner.p,
                           d_parent_leaf.p, d_node_lo.p, d_node_hi.p, d_flags.p, d_misc.p);
      RTB_CUDA(cudaGetLastError());
      k_depth<<<blocks, T>>>((int)N, d_parent_inner.p, d_parent_leaf.p, d_misc.p);
      RTB_CUDA(cudaGetLastError());

      /* the product path walks the compressed BVH4 only; the BVH2 and the uncompressed BVH4 are
       * parity probes (RTB_SCENE_ALL_TREES) -- or the fallback for a tree too deep for the BVH4 stack */
      if (all_trees)
      {
        RTB_CUDA(scene_alloc(sc.get(), &sc->d_nodes, 4 * (N - 1)));
        RTB_CUDA(cudaMemsetAsync(sc->d_nodes, 0, sizeof(BvhNode) * (N - 1), 0));
        k_emit<<<blocks, T>>>(d_vals_sorted.p, d_lo.p, d_hi.p, (int)N, d_children.p, d_first.p, d_node_lo.p,
                              d_node_hi.p, d_bp.p, sc->d_nodes, d_misc.p + 1, leaf_max);
        RTB_CUDA(cudaGetLastError());
        RTB_CUDA(scene_alloc(sc.get(), &sc->d_nodes4, 8 * (N - 1)));
      }
      RTB_CUDA(scene_alloc(sc.get(), &sc->d_nodes4q, 4 * (N - 1)));
      {
        Emit4Queues eq;
        eq.items[0] = d_items_a.p;
        eq.items[1] = d_items_b.p;
        eq.counts = d_level_counts.p;
        eq.n_nodes = d_misc4.p;
        k_emit4_seed<<<1, 1>>>(eq);
        /* a BVH4 level consumes at least one BVH2 level; an empty level costs an empty launch */
        const int half_blocks = (int)((N / 2 + T) / T);
        /* (a tree over N primitives has fewer than N levels: small scenes skip the empty launches; a BVH4 deeper
         * than (RTB_STACK_SIZE - 2) / 3 levels is not walked anyway -- see bvh4_ok below -- so it is not finished) */
        const int max_levels = (int)std::min<size_t>((RTB_STACK_SIZE - 2) / 3 + 2, N);
        emitted_levels = max_levels;
        for (int level = 0; level < max_levels; level++)
          k_emit4<<<half_blocks, T>>>(d_vals_sorted.p, d_lo.p, d_hi.p, (int)N, d_children.p, d_first.p, d_node_lo.p,
                                      d_node_hi.p, d_bp.p, sc->d_nodes4, sc->d_nodes4q, eq, level, leaf_max,
                                      leaf_ref((int)N, 1));
        RTB_CUDA(cudaGetLastError());
        RTB_CUDA(cudaMemcpyAsync(h_levels, d_level_counts.p, sizeof(int) * (RTB_STACK_SIZE + 1), cudaMemcpyDeviceToHost, 0));
      }
      k_reorder<<<blocks, T>>>(d_vals_sorted.p, (int)N, d_unsorted.p, reinterpret_cast<PrimRec *>(sc->d_prims),
                               want_tex ? d_tex_unsorted.p : nullptr, sc->d_tex);
      RTB_CUDA(cudaGetLastError());
      RTB_CUDA(cudaMemcpyAsync(h_misc, d_misc.p, sizeof(h_misc), cudaMemcpyDeviceToHost, 0));
      RTB_CUDA(cudaMemcpyAsync(&h_nodes4, d_misc4.p, sizeof(int), cudaMemcpyDeviceToHost, 0));
      view.root_ref = 0;
      dev_bytes += ((all_trees ? sizeof(BvhNode) + sizeof(Bvh4Node) : 0) + sizeof(Bvh4QNode)) * (N - 1);
    }
    dev_bytes += sizeof(PrimRec) * N + (want_tex ? sizeof(float2) * 3 * N : 0);
  }
  else
  {
    RTB_CUDA(scene_alloc(sc.get(), &sc->d_prims, 3));
    RTB_CUDA(scene_alloc(sc.get(), &sc->d_nodes, 4));
  }
  RTB_CUDA(cudaEventRecord(ev1, 0));
  RTB_CUDA(cudaEventSynchronize(ev1)); /* the only host wait of the build */
  mark("sort + hierarchy + BVH4");
  if (timing)
  {
    std::string line = "rtb_scene_create";
    if (shard) line += " rank " + std::to_string(shard->rank);
    for (size_t k = 1; k < marks.size(); k++)
    {
      char buf[96];
      snprintf(buf, sizeof(buf), "%s %s %.2f ms", k == 1 ? ":" : ",", marks[k].first, marks[k].second - marks[k - 1].second);
      line += buf;
    }
    fprintf(stderr, "%s\n", line.c_str());
  }
  float ms = 0;
  RTB_CUDA(cudaEventElapsedTime(&ms, ev0, ev1));

  if (N > 0 && h_inexact)
  {
    /* some mesh coordinate is not float-representable (a mesh transformed in double, main.c:140-147): keep the
     * caller's doubles, in BVH order, for the exact triangle test and the surface normal */
    for (const std::pair<size_t, size_t> &piece : narrowed)
    {
      k_widen_tri64<<<(int)((piece.second + 255) / 256), 256>>>(d_unsorted.p + piece.first, (int)piece.second,
                                                                 d_tri64_unsorted.p + 9 * piece.first);
      RTB_CUDA(cudaGetLastError());
    }
    if (shard != nullptr && shard->n_ranks > 1 && n_tris >= (size_t)shard->n_ranks * 4096)
    {
      /* sharded upload: every rank holds the doubles of its own triangles only (the flag is the max over the ranks,
       * so all of them are here) */
      const size_t chunk = (n_tris + (size_t)shard->n_ranks - 1) / (size_t)shard->n_ranks;
      int grc = rtb_shard_allgather_bytes(shard, d_tri64_unsorted.p + 9 * n_bs, sizeof(double) * 9 * chunk);
      if (grc != RTB_OK)
        return grc;
    }
    RTB_CUDA(scene_alloc(sc.get(), &sc->d_tri64, 9 * (N + 1)));
    RTB_CUDA(cudaMemsetAsync(sc->d_tri64 + 9 * N, 0, sizeof(double) * 9, 0)); /* the degenerate triangle of empty slots */
    k_reorder64<9><<<(int)((N + 255) / 256), 256>>>(d_vals_sorted.p, (int)N, d_tri64_unsorted.p, sc->d_tri64);
    RTB_CUDA(cudaGetLastError());
    RTB_CUDA(cudaStreamSynchronize(0));
    dev_bytes += sizeof(double) * 9 * N;
  }
  if (N > 0 && h_tex_inexact)
  {
    /* some texture coordinate is not float-representable: keep the caller's doubles, in BVH order, for the checker
     * pattern (raytracer.c:386-391 reads u * 100000); the same steps as for tri64 above */
    if (n_bs)
      RTB_CUDA(cudaMemsetAsync(d_tex64_unsorted.p, 0, sizeof(double) * 6 * n_bs, 0)); /* sphere slots: never read */
    for (const std::pair<size_t, size_t> &piece : narrowed)
    {
      k_widen_tex64<<<(int)((piece.second + 255) / 256), 256>>>(d_tex_unsorted.p + 3 * piece.first, (int)piece.second,
                                                                 d_tex64_unsorted.p + 6 * piece.first);
      RTB_CUDA(cudaGetLastError());
    }
    if (shard != nullptr && shard->n_ranks > 1 && n_tris >= (size_t)shard->n_ranks * 4096)
    {
      const size_t chunk = (n_tris + (size_t)shard->n_ranks - 1) / (size_t)shard->n_ranks;
      int grc = rtb_shard_allgather_bytes(shard, d_tex64_unsorted.p + 6 * n_bs, sizeof(double) * 6 * chunk);
      if (grc != RTB_OK)
        return grc;
    }
    RTB_CUDA(scene_alloc(sc.get(), &sc->d_tex64, 6 * N));
    k_reorder64<6><<<(int)((N + 255) / 256), 256>>>(d_vals_sorted.p, (int)N, d_tex64_unsorted.p, sc->d_tex64);
    RTB_CUDA(cudaGetLastError());
    RTB_CUDA(cudaStreamSynchronize(0));
    dev_bytes += sizeof(double) * 6 * N;
  }
  if (N > 0)
  {
    if (!h_bp.finite)
    {
      rtb_set_error("non-finite geometry");
      return RTB_EINVAL;
    }
    for (int k = 0; k < 3; k++)
    {
      view.guard_lo[k] = h_bp.guard_lo[k];
      view.guard_hi[k] = h_bp.guard_hi[k];
    }
    /* How far outside the guard box an origin may lie for the culling FP32 walk to stay conservative (beyond it,
     * rayf_walk_setup walks every box: the nearest hit is then the brute-force one by construction):
     *  - the walk re-bases such a ray to 0.001 t_in before the guard box; within 300 guard diagonals that point
     *    stays within one guard diagonal of it, inside the envelope the box padding was sized for (k_build_params);
     *  - the exact sphere test (raytracer.c:77-118) computes d2 = L.L - tca^2 with an error of at most
     *    16 |L|^2 2^-53; a box cull is safe while that stays below 2 r pad (a ray that passes the padded box
     *    of a sphere of radius r cannot then be accepted by the exact test), which bounds |L| for the smallest
     *    sphere in the tree. */
    {
      double gd = 0.0;
      for (int k = 0; k < 3; k++)
        gd += ((double)h_bp.guard_hi[k] - h_bp.guard_lo[k]) * ((double)h_bp.guard_hi[k] - h_bp.guard_lo[k]);
      gd = sqrt(gd);
      double far = 300.0 * gd;
      double r_min = HUGE_VAL;
      for (const SphereIn &s : bvh_spheres)
        r_min = std::min(r_min, std::fabs(s.r));
      if (r_min < HUGE_VAL)
        far = std::min(far, sqrt(2.0 * r_min * (double)h_bp.pad * 9007199254740992.0 / 16.0) - gd);
      view.far_t = (float)std::max(far, 0.0);
    }
    bvh_depth = h_misc[0];
    while (depth4 < RTB_STACK_SIZE && h_levels[depth4] > 0)
      depth4++;
    /* the BVH2 walk pushes at most one entry per level, the BVH4 walk at most three */
    if (bvh_depth > RTB_STACK_SIZE - 2)
    {
      rtb_set_error("BVH deeper than the traversal stack");
      return RTB_EINVAL;
    }
    /* a very unbalanced tree can be too deep for the BVH4 walk's stack while the BVH2 walk still
     * fits: such a scene is rendered with the BVH2 walk (same results, see SceneView::nodes4q) */
    bvh4_ok = 3 * depth4 <= RTB_STACK_SIZE - 2;
    if (!bvh4_ok && !all_trees)
      return build_scene(hs, device, flags | RTB_SCENE_ALL_TREES, shard, out); /* rare: build the BVH2 as well */
    n_nodes = (size_t)(bvh4_ok ? h_nodes4 : h_misc[1]); /* nodes of the tree the default path walks */
  }
  size_t nodes4_written = 0; /* a fallback scene's BVH4 stops after emitted_levels levels */
  for (int l = 0; l < emitted_levels; l++)
    nodes4_written += (size_t)h_levels[l];

  view.nodes = sc->d_nodes;
  view.nodes4 = bvh4_ok ? sc->d_nodes4 : nullptr;
  view.nodes4q = bvh4_ok ? sc->d_nodes4q : nullptr;
  view.prims = sc->d_prims;
  view.big = sc->d_big;
  view.mats = sc->d_mats;
  view.colors = sc->d_colors;
  view.tex = sc->d_tex;
  view.tri64 = sc->d_tri64;
  view.tex64 = sc->d_tex64;

  sc->info.n_objects = hs.n_objects;
  sc->info.n_spheres = hs.spheres.size();
  sc->info.n_triangles = n_tris;
  sc->info.n_bvh_prims = N;
  sc->info.n_bvh_nodes = n_nodes;
  sc->info.n_big_prims = big_spheres.size();
  sc->info.device_bytes = dev_bytes;
  sc->info.build_ms = ms;
  sc->info.bvh_depth = bvh_depth;
  sc->info.device = device;
  sc->info.double_triangles = h_inexact ? 1 : 0;
  sc->info.double_texcoords = h_tex_inexact ? 1 : 0;
  sc->info.bvh4_depth = view.nodes4q != nullptr ? depth4 : 0;

  rtb_scene_tree_info &t = sc->tree;
  t.n_prims = N;
  t.n_big = big_spheres.size();
  t.n_nodes4q = nodes4_written;
  t.n_nodes4 = sc->d_nodes4 ? nodes4_written : 0;
  t.n_nodes2 = all_trees && (int)N > leaf_max ? N - 1 : 0;
  t.root_ref = view.root_ref;
  t.leaf_max = leaf_max;
  t.depth4 = depth4;
  t.walks_bvh4 = view.nodes4q != nullptr ? 1 : 0;
  t.has_tex = sc->d_tex != nullptr;
  t.has_tri64 = sc->d_tri64 != nullptr;
  t.has_tex64 = sc->d_tex64 != nullptr;
  for (int k = 0; k < 3; k++)
  {
    t.scene_lo[k] = N > 0 ? h_bp.lo[k] : 0.0f;
    t.scene_hi[k] = N > 0 ? h_bp.hi[k] : 0.0f;
    t.guard_lo[k] = view.guard_lo[k];
    t.guard_hi[k] = view.guard_hi[k];
  }
  t.pad = N > 0 ? h_bp.pad : 0.0f;
  t.far_t = view.far_t;
  *out = sc.release();
  return RTB_OK;
}
} // namespace

extern "C" int rtb_scene_create(const void *scene_objects96, size_t n_objects, int device, rtb_scene **out)
{
  return rtb_scene_create_flags(scene_objects96, n_objects, device, 0u, out);
}

extern "C" int rtb_scene_create_objects(const void *objects88, size_t n_objects, int device, rtb_scene **out)
{
  return rtb_scene_create_objects_flags(objects88, n_objects, device, 0u, out);
}

extern "C" int rtb_scene_create_flags(const void *scene_objects96, size_t n_objects, int device, unsigned flags,
                                      rtb_scene **out)
{
  if (!out || (n_objects && !scene_objects96))
  {
    rtb_set_error("rtb_scene_create: NULL argument");
    return RTB_EINVAL;
  }
  *out = nullptr;
  HostScene hs;
  int rc = gather_scene_objects(static_cast<const RefSceneObject *>(scene_objects96), n_objects, hs);
  if (rc != RTB_OK)
    return rc;
  return build_scene(hs, device, flags, nullptr, out);
}

extern "C" int rtb_scene_create_objects_flags(const void *objects88, size_t n_objects, int device, unsigned flags,
                                              rtb_scene **out)
{
  if (!out || (n_objects && !objects88))
  {
    rtb_set_error("rtb_scene_create_objects: NULL argument");
    return RTB_EINVAL;
  }
  *out = nullptr;
  if (n_objects >= (1ull << 27))
  {
    rtb_set_error("scene too large (>= 2^27 primitives)");
    return RTB_EINVAL;
  }
  const RefObject *objs = static_cast<const RefObject *>(objects88);
  HostScene hs;
  hs.n_objects = n_objects;
  hs.n_prims = (long long)n_objects;
  for (size_t i = 0; i < n_objects; i++)
  {
    push_material(hs, objs[i].flags, objs[i].color, objs[i].emission);
    hs.spheres.push_back(SphereIn{ objs[i].center.x, objs[i].center.y, objs[i].center.z, objs[i].radius, (int)i, (int)i });
  }
  return build_scene(hs, device, flags, nullptr, out);
}

/* rtb_multi.cu: the collective form of rtb_scene_create*; kind = 88 (Object) or 96 (SceneObject) */
int rtb_scene_create_sharded(const void *objects, size_t n_objects, int kind, int device, unsigned flags,
                             const rtb_scene_shard *shard, rtb_scene **out)
{
  if (!out || (n_objects && !objects) || (kind != 88 && kind != 96))
  {
    rtb_set_error("rtb_scene_create_sharded: bad argument");
    return RTB_EINVAL;
  }
  *out = nullptr;
  HostScene hs;
  if (kind == 96)
  {
    int rc = gather_scene_objects(static_cast<const RefSceneObject *>(objects), n_objects, hs);
    if (rc != RTB_OK)
      return rc;
  }
  else
  {
    if (n_objects >= (1ull << 27))
    {
      rtb_set_error("scene too large (>= 2^27 primitives)");
      return RTB_EINVAL;
    }
    const RefObject *objs = static_cast<const RefObject *>(objects);
    hs.n_objects = n_objects;
    hs.n_prims = (long long)n_objects;
    for (size_t i = 0; i < n_objects; i++)
    {
      push_material(hs, objs[i].flags, objs[i].color, objs[i].emission);
      hs.spheres.push_back(SphereIn{ objs[i].center.x, objs[i].center.y, objs[i].center.z, objs[i].radius, (int)i, (int)i });
    }
  }
  return build_scene(hs, device, flags, shard, out);
}

extern "C" int rtb_scene_info_get(const rtb_scene *scene, rtb_scene_info *info)
{
  if (!scene || !info)
  {
    rtb_set_error("rtb_scene_info_get: NULL argument");
    return RTB_EINVAL;
  }
  *info = scene->info;
  return RTB_OK;
}

extern "C" int rtb_scene_tree(const rtb_scene *scene, rtb_scene_tree_info *info, void *nodes4q, void *nodes4, void *nodes,
                              void *prims, void *big, void *tri64, void *tex, void *tex64)
{
  if (!scene || !info)
  {
    rtb_set_error("rtb_scene_tree: NULL argument");
    return RTB_EINVAL;
  }
  const rtb_scene_tree_info &t = scene->tree;
  *info = t;
  const size_t N = t.n_prims;
  const struct { void *dst; const void *src; size_t bytes; } copies[] = {
    { nodes4q, scene->d_nodes4q, sizeof(Bvh4QNode) * t.n_nodes4q },
    { nodes4, scene->d_nodes4, sizeof(Bvh4Node) * t.n_nodes4 },
    { nodes, scene->d_nodes, sizeof(BvhNode) * t.n_nodes2 },
    { prims, scene->d_prims, N ? sizeof(PrimRec) * (N + 1) : 0 },
    { big, scene->d_big, (sizeof(PrimRec) + 2 * sizeof(float4)) * t.n_big },
    { tri64, scene->d_tri64, t.has_tri64 ? sizeof(double) * 9 * (N + 1) : 0 },
    { tex, scene->d_tex, t.has_tex ? sizeof(float2) * 3 * N : 0 },
    { tex64, scene->d_tex64, t.has_tex64 ? sizeof(double) * 6 * N : 0 },
  };
  RTB_CUDA(cudaSetDevice(scene->device));
  for (const auto &c : copies)
    if (c.dst && c.bytes)
      RTB_CUDA(cudaMemcpy(c.dst, c.src, c.bytes, cudaMemcpyDeviceToHost));
  return RTB_OK;
}

namespace
{
struct ParkedBuffer { void *p; size_t bytes; };
const size_t kCacheEntries = 24;
std::mutex g_cache_mutex;
std::vector<ParkedBuffer> g_cache[64];
}

void *rtb_cache_take(int device, size_t need, size_t *bytes)
{
  if (device < 0 || device >= 64)
    return nullptr;
  std::lock_guard<std::mutex> lock(g_cache_mutex);
  std::vector<ParkedBuffer> &c = g_cache[device];
  int pick = -1;
  for (size_t k = 0; k < c.size(); k++)
    if (c[k].bytes >= need && c[k].bytes <= need + need / 4 + 65536 && (pick < 0 || c[k].bytes < c[(size_t)pick].bytes))
      pick = (int)k;
  if (pick < 0)
    return nullptr;
  void *p = c[(size_t)pick].p;
  *bytes = c[(size_t)pick].bytes;
  c.erase(c.begin() + pick);
  return p;
}

void rtb_cache_park(int device, void *p, size_t bytes)
{
  if (!p)
    return;
  std::vector<void *> drop;
  if (device >= 0 && device < 64)
  {
    /* keep at most kCacheEntries buffers and an eighth of the device memory; oldest go first */
    static size_t total_mem[64] = { 0 }; /* cudaMemGetInfo costs milliseconds: asked once per device */
    std::lock_guard<std::mutex> lock(g_cache_mutex);
    if (total_mem[device] == 0)
    {
      size_t free_b = 0, total_b = 0;
      cudaMemGetInfo(&free_b, &total_b);
      total_mem[device] = total_b ? total_b : 1;
    }
    const size_t cap = std::max<size_t>(total_mem[device] / 8, bytes);
    std::vector<ParkedBuffer> &c = g_cache[device];
    c.push_back(ParkedBuffer{ p, bytes });
    size_t held = 0;
    for (const ParkedBuffer &b : c)
      held += b.bytes;
    while (c.size() > 1 && (c.size() > kCacheEntries || held > cap))
    {
      held -= c.front().bytes;
      drop.push_back(c.front().p);
      c.erase(c.begin());
    }
  }
  else
    drop.push_back(p);
  for (void *d : drop)
    cudaFree(d);
}

extern "C" void rtb_release_workspace(int device)
{
  if (device < 0 || device >= 64)
    return;
  cudaSetDevice(device);
  std::vector<ParkedBuffer> drop;
  {
    std::lock_guard<std::mutex> lock(g_cache_mutex);
    drop.swap(g_cache[device]);
  }
  for (const ParkedBuffer &b : drop)
    cudaFree(b.p);
}

extern "C" void rtb_scene_destroy(rtb_scene *scene)
{
  if (!scene)
    return;
  cudaSetDevice(scene->device);
  /* nothing may still be using the buffers when the next scene takes them over */
  cudaDeviceSynchronize();
  for (const std::pair<void *, size_t> &b : scene->owned)
    rtb_cache_park(scene->device, b.first, b.second);
  if (scene->d_wf)
    rtb_cache_park(scene->device, scene->d_wf, scene->wf_bytes);
  for (int g = 0; g < RTB_WF_MAX_GROUPS; g++)
  {
    if (scene->wf_joins[g]) cudaEventDestroy(scene->wf_joins[g]);
  }
  if (scene->wf_fork) cudaEventDestroy(scene->wf_fork);
  if (scene->d_nee) cudaFree(scene->d_nee);
  if (scene->d_scratch)
    rtb_cache_park(scene->device, scene->d_scratch, scene->scratch_bytes);
  delete scene;
}

extern "C" int rtb_warm_up(int device)
{
  RTB_CUDA(cudaSetDevice(device));
  RTB_CUDA(cudaFree(nullptr)); /* creates the primary context */
  RTB_CUDA(pool_setup(device));
  return RTB_OK;
}
