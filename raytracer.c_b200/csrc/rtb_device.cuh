/*
 * rtb_device.cuh -- device-side building blocks of the path tracer (sm_100a).
 *
 * Numerics contract (DESIGN.md "Precision"):
 *   - everything that decides WHICH primitive is hit, and where, is IEEE double with the
 *     reference's operation order and NO fused multiply-add (the reference is built with
 *     ISO-C gcc on x86-64: no contraction).  The __d*_rn intrinsics are never contracted
 *     by nvcc, so t, the hit point and the normal are bit-identical to the reference's
 *     for the same ray;
 *   - the BVH is walked in FP32 with conservatively padded boxes: it only PROPOSES
 *     candidates, the double test disposes;
 *   - colour arithmetic (throughput, emission) is FP32.
 */
#ifndef RTB_DEVICE_CUH
#define RTB_DEVICE_CUH

#include "rtb_internal.h"
#include <float.h>

/* ---- double3 without contraction (vector.h:16-61 operation order) ---------- */

struct d3 { double x, y, z; };

__device__ __forceinline__ d3 d3_make(double x, double y, double z) { d3 r; r.x = x; r.y = y; r.z = z; return r; }
__device__ __forceinline__ d3 d3_add(d3 a, d3 b) { return d3_make(__dadd_rn(a.x, b.x), __dadd_rn(a.y, b.y), __dadd_rn(a.z, b.z)); }
__device__ __forceinline__ d3 d3_sub(d3 a, d3 b) { return d3_make(__dsub_rn(a.x, b.x), __dsub_rn(a.y, b.y), __dsub_rn(a.z, b.z)); }
__device__ __forceinline__ d3 d3_scale(d3 v, double s) { return d3_make(__dmul_rn(v.x, s), __dmul_rn(v.y, s), __dmul_rn(v.z, s)); }
__device__ __forceinline__ double d3_dot(d3 a, d3 b)
{
  return __dadd_rn(__dadd_rn(__dmul_rn(a.x, b.x), __dmul_rn(a.y, b.y)), __dmul_rn(a.z, b.z));
}
__device__ __forceinline__ d3 d3_cross(d3 a, d3 b)
{
  return d3_make(__dsub_rn(__dmul_rn(a.y, b.z), __dmul_rn(a.z, b.y)),
                 __dsub_rn(__dmul_rn(a.z, b.x), __dmul_rn(a.x, b.z)),
                 __dsub_rn(__dmul_rn(a.x, b.y), __dmul_rn(a.y, b.x)));
}
__device__ __forceinline__ double d3_length(d3 v) { return __dsqrt_rn(d3_dot(v, v)); }
/* vec3_normalize: multiply by the reciprocal of the length (vector.h:56-61) */
__device__ __forceinline__ d3 d3_normalize(d3 v) { return d3_scale(v, __ddiv_rn(1.0, d3_length(v))); }
__device__ __forceinline__ d3 d3_neg(d3 v) { return d3_make(-v.x, -v.y, -v.z); }

/* ---- Philox4x32-10 (replaces random_double, raytracer.c:227) --------------- */

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k)
{
#pragma unroll
  for (int round = 0; round < 10; round++)
  {
    const unsigned M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
    unsigned hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
    unsigned hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}

/* 32-bit word -> the reference's 31-bit uniform in [0,1): (w>>1) / 2^31, exact */
__device__ __forceinline__ double uniform31(unsigned w) { return (double)(w >> 1) * (1.0 / 2147483648.0); }

/* ---- exact primitive tests -------------------------------------------------- */

#define RT_EPSILON 1e-8 /* raytracer.h:24 */

/* raytracer.c:77-118, operation for operation */
__device__ __forceinline__ bool sphere_exact(const d3 &o, const d3 &d, double cx, double cy, double cz,
                                             double radius, double &t_out)
{
  d3 L = d3_make(__dsub_rn(cx, o.x), __dsub_rn(cy, o.y), __dsub_rn(cz, o.z));
  double tca = d3_dot(L, d);
  if (tca < 0)
    return false;
  double d2 = __dsub_rn(d3_dot(L, L), __dmul_rn(tca, tca));
  double r2 = __dmul_rn(radius, radius);
  if (d2 > r2)
    return false;
  double thc = __dsqrt_rn(__dsub_rn(r2, d2));
  double t0 = __dsub_rn(tca, thc);
  double t1 = __dadd_rn(tca, thc);
  if (t0 > t1)
  {
    double s = t0;
    t0 = t1;
    t1 = s;
  }
  if (t0 < 0)
  {
    t0 = t1;
    if (t0 < 0)
      return false;
  }
  if (t0 > RT_EPSILON)
  {
    t_out = t0;
    return true;
  }
  return false;
}

/* raytracer.c:120-174 (Moeller-Trumbore), operation for operation; bu,bv = barycentrics */
__device__ __forceinline__ bool triangle_exact(const d3 &o, const d3 &d, const d3 &v0, const d3 &v1,
                                               const d3 &v2, double &t_out, double &bu, double &bv)
{
  d3 e1 = d3_sub(v1, v0);
  d3 e2 = d3_sub(v2, v0);
  d3 h = d3_cross(d, e2);
  double det = d3_dot(e1, h);
  if (det > -RT_EPSILON && det < RT_EPSILON)
    return false;
  double f = __ddiv_rn(1.0, det);
  d3 s = d3_sub(o, v0);
  double u = __dmul_rn(f, d3_dot(s, h));
  if (u < 0.0 || u > 1.0)
    return false;
  d3 q = d3_cross(s, e1);
  double v = __dmul_rn(f, d3_dot(d, q));
  if (v < 0.0 || __dadd_rn(u, v) > 1.0)
    return false;
  double t = __dmul_rn(f, d3_dot(e2, q));
  if (t > RT_EPSILON)
  {
    t_out = t;
    bu = u;
    bv = v;
    return true;
  }
  return false;
}

/* ---- primitive records ------------------------------------------------------ */

__device__ __forceinline__ double rec_double(float lo, float hi)
{
  return __hiloint2double(__float_as_int(hi), __float_as_int(lo));
}

struct PrimView
{
  float4 a, b, c;
  __device__ __forceinline__ bool is_sphere() const { return (__float_as_uint(c.z) & RTB_PRIM_SPHERE_BIT) != 0; }
  __device__ __forceinline__ int gid() const { return __float_as_int(c.y); }
  __device__ __forceinline__ int object() const { return (int)(__float_as_uint(c.z) & 0x7FFFFFFFu); }
  __device__ __forceinline__ double cx() const { return rec_double(a.x, a.y); }
  __device__ __forceinline__ double cy() const { return rec_double(a.z, a.w); }
  __device__ __forceinline__ double cz() const { return rec_double(b.x, b.y); }
  __device__ __forceinline__ double radius() const { return rec_double(b.z, b.w); }
  __device__ __forceinline__ d3 v0() const { return d3_make((double)a.x, (double)a.y, (double)a.z); }
  __device__ __forceinline__ d3 v1() const { return d3_make((double)a.w, (double)b.x, (double)b.y); }
  __device__ __forceinline__ d3 v2() const { return d3_make((double)b.z, (double)b.w, (double)c.x); }
};

__device__ __forceinline__ PrimView load_prim(const float4 *__restrict__ base, int index)
{
  PrimView p;
  p.a = __ldg(base + 3 * index + 0);
  p.b = __ldg(base + 3 * index + 1);
  p.c = __ldg(base + 3 * index + 2);
  return p;
}

/* nearest-hit bookkeeping: strict `<` in index order == lowest gid wins equal t
 * (raytracer.c:404) */
struct HitRec
{
  double t;
  int gid;
  int slot; /* >= 0: index into the BVH-ordered array; < 0: ~index into the big list */
};

/* vertices of the triangle in BVH slot `slot` as the caller's own doubles (SceneView::tri64): only scenes
 * whose mesh vertices are not float-representable carry them (apply_matrix, main.c:140-147) */
__device__ __forceinline__ void load_tri64(const double *__restrict__ tri64, int slot, d3 &v0, d3 &v1, d3 &v2)
{
  const double *p = tri64 + 9 * (size_t)slot; /* 72-byte records: 8-byte aligned only */
  v0 = d3_make(__ldg(p + 0), __ldg(p + 1), __ldg(p + 2));
  v1 = d3_make(__ldg(p + 3), __ldg(p + 4), __ldg(p + 5));
  v2 = d3_make(__ldg(p + 6), __ldg(p + 7), __ldg(p + 8));
}

/* tri64: NULL = triangle vertices are the record's floats (exact for OBJ-loaded meshes) */
__device__ __forceinline__ void test_prim(const PrimView &p, int slot, const d3 &o, const d3 &d, HitRec &best,
                                          const double *__restrict__ tri64 = nullptr)
{
  double t, bu, bv;
  bool hit;
  if (p.is_sphere())
    hit = sphere_exact(o, d, p.cx(), p.cy(), p.cz(), p.radius(), t);
  else if (tri64 != nullptr && slot >= 0)
  {
    d3 v0, v1, v2;
    load_tri64(tri64, slot, v0, v1, v2);
    hit = triangle_exact(o, d, v0, v1, v2, t, bu, bv);
  }
  else
    hit = triangle_exact(o, d, p.v0(), p.v1(), p.v2(), t, bu, bv);
  if (hit)
  {
    int gid = p.gid();
    if (t < best.t || (t == best.t && gid < best.gid))
    {
      best.t = t;
      best.gid = gid;
      best.slot = slot;
    }
  }
}

/* ---- conservative FP32 sphere pre-test -----------------------------------------
 * Decides, in FP32 with explicit error bounds, that the exact double test cannot produce a
 * hit that beats `best`: either the reference's test certainly returns false (tca < 0 or
 * d2 > r2, raytracer.c:84-89) or even a lower bound of its t exceeds best.t.  Never rejects
 * a primitive the exact test would accept as the new nearest hit (ties included), so the
 * result of the query is unchanged; it only saves FP64 work.
 * Error model: every coordinate entering the test is rounded to float (relative 2^-24);
 * A = |c|_1 + r + |o|_1 bounds every intermediate magnitude, linear quantities (L, tca) are
 * off by at most e = A*2^-20, quadratic ones (d2, r2-d2) by at most eq = 10*A*A*2^-20. */
/* returns false if the reference's test certainly misses; otherwise t_lo = a lower bound of
 * the t it would report */
__device__ __forceinline__ bool sphere_lower_bound(const PrimView &p, float ofx, float ofy, float ofz, float dfx,
                                                   float dfy, float dfz, float o_abs1, float &t_lo)
{
  float cx = (float)p.cx(), cy = (float)p.cy(), cz = (float)p.cz(), r = (float)p.radius();
  float A = (fabsf(cx) + fabsf(cy) + fabsf(cz) + fabsf(r) + o_abs1) * 1.0000005f;
  float e = A * 9.5367431640625e-07f;            /* 2^-20 */
  float eq = 10.0f * A * e;
  float Lx = cx - ofx, Ly = cy - ofy, Lz = cz - ofz;
  float tca = fmaf(Lz, dfz, fmaf(Ly, dfy, Lx * dfx));
  if (tca < -e)
    return false;
  float d2 = fmaf(Lz, Lz, fmaf(Ly, Ly, Lx * Lx)) - tca * tca;
  float disc = fmaf(r, r, -d2);
  if (disc < -eq)
    return false;
  float thc_hi = sqrtf(fmaxf(disc + eq, 0.0f)) * 1.000001f;
  t_lo = tca - e - thc_hi;                       /* lower bound of the near root */
  return true;
}

__device__ __forceinline__ bool sphere_may_win(const PrimView &p, float ofx, float ofy, float ofz, float dfx,
                                               float dfy, float dfz, float o_abs1, float best_t_up)
{
  float t_lo;
  if (!sphere_lower_bound(p, ofx, ofy, ofz, dfx, dfy, dfz, o_abs1, t_lo))
    return false;
  return !(t_lo > best_t_up);
}

template <bool FILTER>
__device__ __forceinline__ void test_prim_filtered(const PrimView &p, int slot, const d3 &o, const d3 &d,
                                                   float ofx, float ofy, float ofz, float dfx, float dfy, float dfz,
                                                   float o_abs1, HitRec &best, unsigned &exact_tests,
                                                   const double *__restrict__ tri64 = nullptr)
{
  if (FILTER && p.is_sphere())
  {
    float best_up = best.t >= 1e30 ? 3.0e38f : __double2float_ru(best.t) * 1.0000005f;
    if (!sphere_may_win(p, ofx, ofy, ofz, dfx, dfy, dfz, o_abs1, best_up))
      return;
  }
  exact_tests++;
  test_prim(p, slot, o, d, best, tri64);
}

/* ---- nearest hit: big list + FP32 BVH walk with exact leaf tests ------------
 * The pieces below are shared by the simple per-ray loop (closest_hit, used by the probes)
 * and by the warp-scheduled state machine of k_render. */

struct TraceStats
{
  unsigned prim_tests, node_visits;
};

/* the FP32 view of a ray used by the walk */
struct RayF
{
  float dfx, dfy, dfz;    /* direction rounded to float (for the sphere pre-test) */
  float ofx, ofy, ofz;    /* ORIGINAL origin rounded to float (sphere pre-test) */
  float idx, idy, idz;    /* 1/direction, zero components replaced by +-tiny */
  float oodx, oody, oodz; /* (re-based origin) * idir */
  float o_abs1;           /* |o|_1 of the original origin */
  float tmax;             /* walk bound in the re-based frame */
  float t_base;           /* parametric offset of the re-based origin */
};

#define RTB_WIDEN 1.0000005f /* > (1+2^-23)^4: slab arithmetic rounding */

__device__ __forceinline__ void rayf_basic(const d3 &o, const d3 &d, RayF &rf)
{
  rf.ofx = (float)o.x; rf.ofy = (float)o.y; rf.ofz = (float)o.z;
  rf.dfx = (float)d.x; rf.dfy = (float)d.y; rf.dfz = (float)d.z;
  rf.o_abs1 = fabsf(rf.ofx) + fabsf(rf.ofy) + fabsf(rf.ofz);
}

/* Prepares the walk.  Returns false if the ray cannot touch the tree (no primitives, or it
 * misses the guard box).  If the origin lies outside the guard box the ray is first
 * advanced (in double) to just before its entry point so that float rounding of the origin
 * stays within the padding the boxes were built with. */
__device__ __forceinline__ bool rayf_walk_setup(const SceneView &sv, const d3 &o, const d3 &d, const HitRec &best, RayF &rf)
{
  if (sv.n_prims == 0)
    return false;
  float ofx = rf.ofx, ofy = rf.ofy, ofz = rf.ofz;
  float dfx = rf.dfx, dfy = rf.dfy, dfz = rf.dfz;
  const float tiny = 1e-24f;
  if (fabsf(dfx) < tiny) dfx = copysignf(tiny, dfx);
  if (fabsf(dfy) < tiny) dfy = copysignf(tiny, dfy);
  if (fabsf(dfz) < tiny) dfz = copysignf(tiny, dfz);
  rf.idx = __frcp_rn(dfx); rf.idy = __frcp_rn(dfy); rf.idz = __frcp_rn(dfz);
  rf.t_base = 0.0f;
  bool outside = ofx < sv.guard_lo[0] || ofx > sv.guard_hi[0] || ofy < sv.guard_lo[1] ||
                 ofy > sv.guard_hi[1] || ofz < sv.guard_lo[2] || ofz > sv.guard_hi[2];
  if (outside)
  {
    /* an origin too far away for the culling walk to be conservative (SceneView::far_t, set by the build): every
     * box is entered at distance 0 and no stack entry is culled, so every leaf gets its exact test */
    const float dist = fmaxf(fmaxf(fmaxf(sv.guard_lo[0] - ofx, ofx - sv.guard_hi[0]), fmaxf(sv.guard_lo[1] - ofy, ofy - sv.guard_hi[1])),
                             fmaxf(sv.guard_lo[2] - ofz, ofz - sv.guard_hi[2]));
    if (dist > sv.far_t)
    {
      rf.idx = rf.idy = rf.idz = 0.0f;
      rf.oodx = rf.oody = rf.oodz = 0.0f;
      rf.tmax = 3.0e38f;
      return true;
    }
    float ax = (sv.guard_lo[0] - ofx) * rf.idx, bx = (sv.guard_hi[0] - ofx) * rf.idx;
    float ay = (sv.guard_lo[1] - ofy) * rf.idy, by = (sv.guard_hi[1] - ofy) * rf.idy;
    float az = (sv.guard_lo[2] - ofz) * rf.idz, bz = (sv.guard_hi[2] - ofz) * rf.idz;
    float t_in = fmaxf(fmaxf(fminf(ax, bx), fminf(ay, by)), fminf(az, bz));
    float t_out = fminf(fminf(fmaxf(ax, bx), fmaxf(ay, by)), fmaxf(az, bz));
    /* the guard box is far larger than the padded scene box, so this rough FP32 test
     * cannot reject a ray that touches the scene box */
    if (t_out < 0.0f || t_in > t_out * 1.001f + 1e-3f)
      return false;
    if (t_in > 0.0f)
    {
      rf.t_base = t_in * 0.999f;
      ofx = (float)fma(d.x, (double)rf.t_base, o.x);
      ofy = (float)fma(d.y, (double)rf.t_base, o.y);
      ofz = (float)fma(d.z, (double)rf.t_base, o.z);
    }
  }
  rf.oodx = ofx * rf.idx; rf.oody = ofy * rf.idy; rf.oodz = ofz * rf.idz;
  rf.tmax = (best.t >= 1e30) ? 3.0e38f : __double2float_ru(best.t - (double)rf.t_base) * RTB_WIDEN;
  return true;
}

__device__ __forceinline__ void rayf_update_tmax(RayF &rf, const HitRec &best)
{
  if (best.t < 1e30)
    rf.tmax = __double2float_ru(best.t - (double)rf.t_base) * RTB_WIDEN;
}

/* Traversal stack.  The first SD entries of every thread live in shared memory, laid out
 * [entry][thread] (conflict-free), the rest in local memory.  SD = 0 keeps everything in
 * local memory.  Entry = {reference, entry distance as float bits}.
 * (Keeping the most recent entry in two registers so that a pop never waits for memory was
 * measured 5 % slower: register pressure.) */
template <int SD>
struct WalkStack
{
  int2 *smem;  /* this thread's column: entry k at smem[k * stride]; unused when SD == 0 */
  int2 *local; /* RTB_STACK_SIZE - SD entries */
  int stride;
  int sp;      /* entries in memory */
  __device__ __forceinline__ void put(int at, int2 e) const
  {
    if (SD > 0 && at < SD) smem[at * stride] = e;
    else local[at - SD] = e;
  }
  __device__ __forceinline__ int2 get(int at) const
  {
    if (SD > 0 && at < SD) return smem[at * stride];
    return local[at - SD];
  }
  __device__ __forceinline__ void reset() { sp = 0; }
  __device__ __forceinline__ void push(int2 e)
  {
    put(sp, e);
    sp++;
  }
  /* the next subtree that can still contain a nearer hit; RTB_REF_NONE when done */
  __device__ __forceinline__ int pop(const RayF &rf)
  {
    while (sp > 0)
    {
      sp--;
      const int2 e = get(sp);
      if (__int_as_float(e.y) <= rf.tmax)
        return e.x;
    }
    return RTB_REF_NONE;
  }
  /* same result, but the top TWO entries are read together: one round trip to local memory per
   * two culled entries (the dependent load of the pop loop was 12.5 % of the walk's stall samples
   * at 3 active lanes, profiles/r1_wf_trace_ncu.md) */
  __device__ __forceinline__ int pop2(const RayF &rf)
  {
    while (sp > 0)
    {
      const int2 e0 = get(sp - 1);
      const int2 e1 = get(sp > 1 ? sp - 2 : sp - 1);
      if (__int_as_float(e0.y) <= rf.tmax)
      {
        sp -= 1;
        return e0.x;
      }
      if (sp > 1 && __int_as_float(e1.y) <= rf.tmax)
      {
        sp -= 2;
        return e1.x;
      }
      sp = sp > 1 ? sp - 2 : 0;
    }
    return RTB_REF_NONE;
  }
};

/* 256-bit read-only global load (pointer must be 32-byte aligned) */
__device__ __forceinline__ void ld256_nc(const float4 *p, float4 &a, float4 &b)
{
  asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
               : "l"(p));
}

/* One inner node: tests both children, returns the reference to continue with
 * (RTB_REF_NONE if neither is hit) and pushes the farther one. */
template <class STK>
__device__ __forceinline__ int node_step(const SceneView &sv, const RayF &rf, int cur, STK &stack)
{
  /* 64-byte node = two 256-bit loads (LDG.E.256, new on sm_100): half the L1 wavefronts of
   * four 128-bit loads -- the L1 data pipe was 60 % busy with node fetches
   * (profiles/r1_wf_trace_ncu.md) */
  float4 n0, n1, n2, n3;
  ld256_nc(sv.nodes + 4 * cur, n0, n1);
  ld256_nc(sv.nodes + 4 * cur + 2, n2, n3);

  float c0lx = fmaf(n0.x, rf.idx, -rf.oodx), c0hx = fmaf(n0.y, rf.idx, -rf.oodx);
  float c0ly = fmaf(n0.z, rf.idy, -rf.oody), c0hy = fmaf(n0.w, rf.idy, -rf.oody);
  float c0lz = fmaf(n2.x, rf.idz, -rf.oodz), c0hz = fmaf(n2.y, rf.idz, -rf.oodz);
  float c1lx = fmaf(n1.x, rf.idx, -rf.oodx), c1hx = fmaf(n1.y, rf.idx, -rf.oodx);
  float c1ly = fmaf(n1.z, rf.idy, -rf.oody), c1hy = fmaf(n1.w, rf.idy, -rf.oody);
  float c1lz = fmaf(n2.z, rf.idz, -rf.oodz), c1hz = fmaf(n2.w, rf.idz, -rf.oodz);

  float c0min = fmaxf(fmaxf(fminf(c0lx, c0hx), fminf(c0ly, c0hy)), fmaxf(fminf(c0lz, c0hz), 0.0f));
  float c0max = fminf(fminf(fmaxf(c0lx, c0hx), fmaxf(c0ly, c0hy)), fminf(fmaxf(c0lz, c0hz), rf.tmax));
  float c1min = fmaxf(fmaxf(fminf(c1lx, c1hx), fminf(c1ly, c1hy)), fmaxf(fminf(c1lz, c1hz), 0.0f));
  float c1max = fminf(fminf(fmaxf(c1lx, c1hx), fmaxf(c1ly, c1hy)), fminf(fmaxf(c1lz, c1hz), rf.tmax));

  bool h0 = c0min <= c0max * RTB_WIDEN;
  bool h1 = c1min <= c1max * RTB_WIDEN;
  int r0 = __float_as_int(n3.x), r1 = __float_as_int(n3.y);
  if (h0 && h1)
  {
    bool swap = c1min < c0min;
    stack.push(make_int2(swap ? r0 : r1, __float_as_int(swap ? c0min : c1min)));
    return swap ? r1 : r0;
  }
  if (h0) return r0;
  if (h1) return r1;
  return RTB_REF_NONE;
}

/* One BVH4 node: tests up to four children, continues with the nearest one hit and pushes the
 * others far-to-near (so the nearer is popped first). */
__device__ __forceinline__ void cswap(float &da, int &ra, float &db, int &rb)
{
  const bool s = db < da;
  const float dt = s ? db : da, du = s ? da : db;
  const int rt = s ? rb : ra, ru = s ? ra : rb;
  da = dt; db = du; ra = rt; rb = ru;
}

template <class STK>
__device__ __forceinline__ int node_step4(const SceneView &sv, const RayF &rf, int cur, STK &stack)
{
  const float4 *np = sv.nodes4 + 8 * (size_t)cur;
  float4 lox, hix, loy, hiy, loz, hiz, rr, spare;
  ld256_nc(np + 0, lox, hix);
  ld256_nc(np + 2, loy, hiy);
  ld256_nc(np + 4, loz, hiz);
  ld256_nc(np + 6, rr, spare);
  const float INF = 3.0e38f;
  float dist[4];
  int ref[4] = { __float_as_int(rr.x), __float_as_int(rr.y), __float_as_int(rr.z), __float_as_int(rr.w) };
  const float lx[4] = { lox.x, lox.y, lox.z, lox.w }, hx[4] = { hix.x, hix.y, hix.z, hix.w };
  const float ly[4] = { loy.x, loy.y, loy.z, loy.w }, hy[4] = { hiy.x, hiy.y, hiy.z, hiy.w };
  const float lz[4] = { loz.x, loz.y, loz.z, loz.w }, hz[4] = { hiz.x, hiz.y, hiz.z, hiz.w };
#pragma unroll
  for (int k = 0; k < 4; k++)
  {
    const float ax = fmaf(lx[k], rf.idx, -rf.oodx), bx = fmaf(hx[k], rf.idx, -rf.oodx);
    const float ay = fmaf(ly[k], rf.idy, -rf.oody), by = fmaf(hy[k], rf.idy, -rf.oody);
    const float az = fmaf(lz[k], rf.idz, -rf.oodz), bz = fmaf(hz[k], rf.idz, -rf.oodz);
    const float tmin = fmaxf(fmaxf(fminf(ax, bx), fminf(ay, by)), fmaxf(fminf(az, bz), 0.0f));
    const float tmax = fminf(fminf(fmaxf(ax, bx), fmaxf(ay, by)), fminf(fmaxf(az, bz), rf.tmax));
    const bool hit = (tmin <= tmax * RTB_WIDEN) && ref[k] != RTB_REF_NONE;
    dist[k] = hit ? tmin : INF;
  }
  /* sorting network for 4 keys */
  cswap(dist[0], ref[0], dist[1], ref[1]);
  cswap(dist[2], ref[2], dist[3], ref[3]);
  cswap(dist[0], ref[0], dist[2], ref[2]);
  cswap(dist[1], ref[1], dist[3], ref[3]);
  cswap(dist[1], ref[1], dist[2], ref[2]);
  if (dist[0] >= INF)
    return RTB_REF_NONE;
  if (dist[3] < INF) stack.push(make_int2(ref[3], __float_as_int(dist[3])));
  if (dist[2] < INF) stack.push(make_int2(ref[2], __float_as_int(dist[2])));
  if (dist[1] < INF) stack.push(make_int2(ref[1], __float_as_int(dist[1])));
  return ref[0];
}

/* One compressed BVH4 node (Bvh4QNode, rtb_internal.h): slab distances straight from the
 * quantised planes, t = q * (2^e / d) + (origin - o) / d.
 *
 * Instruction budget (profiles/r2_wf_trace_ncu.md): the round-1 form of this function was 148
 * SASS instructions per visit, 100 of them on the ALU pipe (2 cycles per warp instruction) and 24
 * I2F.U8 on the conversion pipe -- both pipes as busy as the issue slots.  This form
 *   - picks the near/far plane word per AXIS from the sign of the ray direction (6 SEL per node)
 *     instead of min/max-ing both planes per child (44 -> 16 FMNMX/FMNMX3);
 *   - needs no validity test per child: an empty slot is an inverted box (qlo 255, qhi 0) whose
 *     reference is a degenerate triangle at the end of the primitive array, so even a rounding
 *     coincidence cannot send the walk to a bad address;
 *   - reads the per-axis cell size as a ready float (no exponent-byte extraction);
 *   - converts CONV_ALU of the 24 plane bytes on the ALU + FMA pipes (PRMT into the mantissa of
 *     2^23, FADD -2^23) instead of the conversion pipe, to balance the three pipes. */
__device__ __forceinline__ float qbyte(unsigned w, int k) { return (float)((w >> (8 * k)) & 0xFFu); }
/* byte k of w as a float without the conversion pipe: 0x4B0000bb = 2^23 + bb exactly */
__device__ __forceinline__ float qbyte_alu(unsigned w, int k)
{
  return __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7650u + (unsigned)k)) - 8388608.0f;
}

template <int CONV_ALU, class STK>
__device__ __forceinline__ int node_step4q(const SceneView &sv, const RayF &rf, int cur, STK &stack)
{
  const float4 *np = sv.nodes4q + 4 * (size_t)cur;
  float4 w0, w1, w2, w3;
  ld256_nc(np + 0, w0, w1);
  ld256_nc(np + 2, w2, w3);
  const float sx = w0.w * rf.idx, sy = w3.z * rf.idy, sz = w3.w * rf.idz;
  const float bx = fmaf(w0.x, rf.idx, -rf.oodx), by = fmaf(w0.y, rf.idy, -rf.oody), bz = fmaf(w0.z, rf.idz, -rf.oodz);
  const unsigned qlx = __float_as_uint(w2.x), qly = __float_as_uint(w2.y), qlz = __float_as_uint(w2.z);
  const unsigned qhx = __float_as_uint(w2.w), qhy = __float_as_uint(w3.x), qhz = __float_as_uint(w3.y);
  /* entry plane = lo for a positive direction component, hi for a negative one */
  const bool nx = rf.idx < 0.0f, ny = rf.idy < 0.0f, nz = rf.idz < 0.0f;
  const unsigned nrx = nx ? qhx : qlx, frx = nx ? qlx : qhx;
  const unsigned nry = ny ? qhy : qly, fry = ny ? qly : qhy;
  const unsigned nrz = nz ? qhz : qlz, frz = nz ? qlz : qhz;
  const float INF = 3.0e38f;
  float dist[4];
  int ref[4] = { __float_as_int(w1.x), __float_as_int(w1.y), __float_as_int(w1.z), __float_as_int(w1.w) };
#pragma unroll
  for (int k = 0; k < 4; k++)
  {
    /* the first CONV_ALU far-plane conversions of the node go through PRMT + FADD */
    const float ax = fmaf(qbyte(nrx, k), sx, bx);
    const float ay = fmaf(qbyte(nry, k), sy, by);
    const float az = fmaf(qbyte(nrz, k), sz, bz);
    const float cx = fmaf((3 * k + 0 < CONV_ALU) ? qbyte_alu(frx, k) : qbyte(frx, k), sx, bx);
    const float cy = fmaf((3 * k + 1 < CONV_ALU) ? qbyte_alu(fry, k) : qbyte(fry, k), sy, by);
    const float cz = fmaf((3 * k + 2 < CONV_ALU) ? qbyte_alu(frz, k) : qbyte(frz, k), sz, bz);
    const float tmin = fmaxf(fmaxf(ax, ay), fmaxf(az, 0.0f));
    const float tmax = fminf(fminf(cx, cy), fminf(cz, rf.tmax));
    dist[k] = (tmin <= tmax * RTB_WIDEN) ? tmin : INF;
  }
  cswap(dist[0], ref[0], dist[1], ref[1]);
  cswap(dist[2], ref[2], dist[3], ref[3]);
  cswap(dist[0], ref[0], dist[2], ref[2]);
  cswap(dist[1], ref[1], dist[3], ref[3]);
  cswap(dist[1], ref[1], dist[2], ref[2]);
  if (dist[0] >= INF)
    return RTB_REF_NONE;
  if (dist[3] < INF) stack.push(make_int2(ref[3], __float_as_int(dist[3])));
  if (dist[2] < INF) stack.push(make_int2(ref[2], __float_as_int(dist[2])));
  if (dist[1] < INF) stack.push(make_int2(ref[1], __float_as_int(dist[1])));
  return ref[0];
}

/* WIDE: 0 = BvhNode (two children, 64 B), 1 = Bvh4Node (128 B), 2 = Bvh4QNode (compressed, 64 B);
 * 3, 4 = Bvh4QNode with 6 / 12 of the 24 byte conversions on the ALU + FMA pipes */
template <int WIDE, class STK>
__device__ __forceinline__ int node_step_w(const SceneView &sv, const RayF &rf, int cur, STK &stack)
{
  if (WIDE >= 2)
    return node_step4q<(WIDE - 2) * 6>(sv, rf, cur, stack);
  if (WIDE == 1)
    return node_step4(sv, rf, cur, stack);
  return node_step(sv, rf, cur, stack);
}

template <bool STATS, bool FILTER>
__device__ __forceinline__ void closest_hit(const SceneView &sv, const d3 &o, const d3 &d, HitRec &best,
                                            TraceStats &st)
{
  best.t = DBL_MAX;
  best.gid = 0x7FFFFFFF;
  best.slot = 0;
  RayF rf;
  rayf_basic(o, d, rf);
  unsigned exact = 0;

  /* oversized primitives (the r=10000 wall spheres): candidates for every ray */
  for (int k = 0; k < sv.n_big; k++)
    test_prim_filtered<FILTER>(load_prim(sv.big, k), ~k, o, d, rf.ofx, rf.ofy, rf.ofz, rf.dfx, rf.dfy, rf.dfz, rf.o_abs1, best, exact);

  if (rayf_walk_setup(sv, o, d, best, rf))
  {
    int2 stack_mem[RTB_STACK_SIZE];
    WalkStack<0> stack = { nullptr, stack_mem, 0 };
    stack.reset();
    int cur = sv.root_ref;
    while (cur != RTB_REF_NONE)
    {
      if (cur >= 0)
      {
        if (STATS) st.node_visits++;
        cur = node_step(sv, rf, cur, stack);
        if (cur != RTB_REF_NONE)
          continue;
      }
      else
      {
        int code = ~cur;
        int first = code >> 3, count = (code & 7) + 1;
        for (int k = 0; k < count; k++)
          test_prim_filtered<FILTER>(load_prim(sv.prims, first + k), first + k, o, d, rf.ofx, rf.ofy, rf.ofz, rf.dfx,
                             rf.dfy, rf.dfz, rf.o_abs1, best, exact, sv.tri64);
        rayf_update_tmax(rf, best);
      }
      cur = stack.pop(rf);
    }
  }
  if (STATS) st.prim_tests += exact;
}

/* same bound from the FP32 copy of an oversized sphere ({cx,cy,cz,r}, A_c): no FP64->FP32
 * conversions in the per-ray loop */
__device__ __forceinline__ bool sphere_lower_bound_f(const float4 c, float Ac, float ofx, float ofy, float ofz,
                                                     float dfx, float dfy, float dfz, float o_abs1, float &t_lo)
{
  float A = (Ac + o_abs1) * 1.0000005f;
  float e = A * 9.5367431640625e-07f; /* 2^-20 */
  float eq = 10.0f * A * e;
  float Lx = c.x - ofx, Ly = c.y - ofy, Lz = c.z - ofz;
  float tca = fmaf(Lz, dfz, fmaf(Ly, dfy, Lx * dfx));
  if (tca < -e)
    return false;
  float d2 = fmaf(Lz, Lz, fmaf(Ly, Ly, Lx * Lx)) - tca * tca;
  float disc = fmaf(c.w, c.w, -d2);
  if (disc < -eq)
    return false;
  float thc_hi = sqrtf(fmaxf(disc + eq, 0.0f)) * 1.000001f;
  t_lo = tca - e - thc_hi;
  return true;
}

/* oversized list, "select, then test": an FP32 lower bound per sphere picks the most
 * promising one, which all lanes test exactly at once; the few others whose bound still
 * beats the result follow */
__device__ __forceinline__ void big_list_select_test(const SceneView &sv, const d3 &o, const d3 &d, const RayF &rf,
                                                     HitRec &best, unsigned &exact)
{
  if (sv.n_big <= 0)
    return;
  const float4 *fcopy = sv.big + 3 * sv.n_big;
  float tlo_min = 3.0e38f, tlo_second = 3.0e38f;
  int kmin = -1;
  unsigned mask = 0u;
  for (int k = 0; k < sv.n_big; k++)
  {
    float tlo;
    const float4 c = __ldg(fcopy + 2 * k);
    const float Ac = __ldg(fcopy + 2 * k + 1).x;
    if (sphere_lower_bound_f(c, Ac, rf.ofx, rf.ofy, rf.ofz, rf.dfx, rf.dfy, rf.dfz, rf.o_abs1, tlo))
    {
      mask |= 1u << k;
      if (tlo < tlo_min)
      {
        tlo_second = tlo_min;
        tlo_min = tlo;
        kmin = k;
      }
      else
        tlo_second = fminf(tlo_second, tlo);
    }
  }
  if (kmin < 0)
    return;
  test_prim(load_prim(sv.big, kmin), ~kmin, o, d, best);
  exact++;
  mask &= ~(1u << kmin);
  /* nobody else can win if even the second-smallest lower bound exceeds the result */
  float best_up = best.t >= 1e30 ? 3.0e38f : __double2float_ru(best.t) * 1.0000005f;
  if (tlo_second > best_up)
    return;
  while (mask)
  {
    int k = __ffs(mask) - 1;
    mask &= mask - 1u;
    test_prim_filtered<true>(load_prim(sv.big, k), ~k, o, d, rf.ofx, rf.ofy, rf.ofz, rf.dfx, rf.dfy, rf.dfz,
                             rf.o_abs1, best, exact);
  }
}

/* "while-while" variant (Aila & Laine 2009): all lanes first walk inner nodes until each has
 * reached a leaf, then the leaf tests run together.  The exact FP64 tests -- the expensive
 * part -- are executed with most lanes active instead of one or two
 * (profiles/r1_c3_megakernel_ncu.md).  The oversized list is handled "select, then test":
 * an FP32 lower bound per sphere picks the most promising one, which is tested exactly by
 * all lanes at once; the few others whose bound still beats the result follow. */
template <bool STATS, int SD, int WIDE = 0>
__device__ __forceinline__ void closest_hit_ww(const SceneView &sv, const d3 &o, const d3 &d, HitRec &best,
                                               TraceStats &st, int2 *smem_column, int smem_stride)
{
  best.t = DBL_MAX;
  best.gid = 0x7FFFFFFF;
  best.slot = 0;
  RayF rf;
  rayf_basic(o, d, rf);
  unsigned exact = 0;

  big_list_select_test(sv, o, d, rf, best, exact);

  if (rayf_walk_setup(sv, o, d, best, rf))
  {
    int2 stack_mem[RTB_STACK_SIZE - SD];
    WalkStack<SD> stack = { smem_column, stack_mem, smem_stride };
    stack.reset();
    int cur = sv.root_ref;
    while (cur != RTB_REF_NONE)
    {
      while (cur >= 0 && cur != RTB_REF_NONE)
      {
        if (STATS) st.node_visits++;
        int nxt = node_step_w<WIDE>(sv, rf, cur, stack);
        cur = (nxt != RTB_REF_NONE) ? nxt : stack.pop(rf);
      }
      if (cur == RTB_REF_NONE)
        break;
      int code = ~cur;
      int first = code >> 3, count = (code & 7) + 1;
      for (int k = 0; k < count; k++)
        test_prim_filtered<false>(load_prim(sv.prims, first + k), first + k, o, d, rf.ofx, rf.ofy, rf.ofz, rf.dfx,
                                  rf.dfy, rf.dfz, rf.o_abs1, best, exact, sv.tri64);
      rayf_update_tmax(rf, best);
      cur = stack.pop(rf);
    }
  }
  if (STATS) st.prim_tests += exact;
}

/* brute force over every primitive: the reference's own O(n) loop (raytracer.c:401-456),
 * kept as a debug path for the BVH == brute-force parity test */
__device__ __forceinline__ void closest_hit_bruteforce(const SceneView &sv, const d3 &o, const d3 &d, HitRec &best)
{
  best.t = DBL_MAX;
  best.gid = 0x7FFFFFFF;
  best.slot = 0;
  for (int k = 0; k < sv.n_big; k++)
    test_prim(load_prim(sv.big, k), ~k, o, d, best);
  for (int k = 0; k < sv.n_prims; k++)
    test_prim(load_prim(sv.prims, k), k, o, d, best, sv.tri64);
}

/* ---- surface at the nearest hit (raytracer.c:406-411, :428-431) ------------- */

struct Surface
{
  d3 point, normal;
  int object;
  double u, v; /* only filled when want_uv */
};

__device__ __forceinline__ Surface surface_at(const SceneView &sv, const d3 &o, const d3 &d, const HitRec &best,
                                              bool want_uv)
{
  Surface s;
  PrimView p = best.slot >= 0 ? load_prim(sv.prims, best.slot) : load_prim(sv.big, ~best.slot);
  s.object = p.object();
  s.point = d3_add(o, d3_scale(d, best.t)); /* point_at, raytracer.c:257 */
  s.u = 0.0;
  s.v = 0.0;
  if (p.is_sphere())
  {
    d3 c = d3_make(p.cx(), p.cy(), p.cz());
    s.normal = d3_normalize(d3_sub(s.point, c));
    if (want_uv)
    {
      const double RT_PI = 3.14159265359; /* raytracer.h:22 */
      s.u = __dadd_rn(__ddiv_rn(atan2(s.normal.x, s.normal.z), __dmul_rn(2.0, RT_PI)), 0.5);
      s.v = __dadd_rn(__dmul_rn(s.normal.y, 0.5), 0.5);
    }
  }
  else
  {
    d3 v0 = p.v0(), v1 = p.v1(), v2 = p.v2();
    if (sv.tri64 != nullptr && best.slot >= 0)
      load_tri64(sv.tri64, best.slot, v0, v1, v2);
    s.normal = d3_normalize(d3_cross(d3_sub(v2, v0), d3_sub(v1, v0))); /* raytracer.c:44 */
    if (want_uv && sv.tex != nullptr && best.slot >= 0)
    {
      double t, bu, bv;
      if (triangle_exact(o, d, v0, v1, v2, t, bu, bv))
      {
        double t0x, t0y, t1x, t1y, t2x, t2y;
        if (sv.tex64 != nullptr)
        {
          const double *q = sv.tex64 + 6 * (size_t)best.slot; /* 48-byte records: 16-byte aligned */
          const double2 a = __ldg(reinterpret_cast<const double2 *>(q) + 0);
          const double2 b = __ldg(reinterpret_cast<const double2 *>(q) + 1);
          const double2 c = __ldg(reinterpret_cast<const double2 *>(q) + 2);
          t0x = a.x; t0y = a.y; t1x = b.x; t1y = b.y; t2x = c.x; t2y = c.y;
        }
        else
        {
          const float2 a = __ldg(sv.tex + 3 * best.slot + 0);
          const float2 b = __ldg(sv.tex + 3 * best.slot + 1);
          const float2 c = __ldg(sv.tex + 3 * best.slot + 2);
          t0x = a.x; t0y = a.y; t1x = b.x; t1y = b.y; t2x = c.x; t2y = c.y;
        }
        double w0 = __dsub_rn(__dsub_rn(1.0, bu), bv); /* 1 - u - v, raytracer.c:160 */
        s.u = __dadd_rn(__dadd_rn(__dmul_rn(t0x, w0), __dmul_rn(t1x, bu)), __dmul_rn(t2x, bv));
        s.v = __dadd_rn(__dadd_rn(__dmul_rn(t0y, w0), __dmul_rn(t1y, bu)), __dmul_rn(t2y, bv));
      }
    }
  }
  return s;
}

/* record i of the nearest-hit probes (rtb_trace_rays, rtb_trace_rays_wf): object id (-1 = miss), primitive gid, t,
 * point, normal and texture coordinates at the hit; any output pointer but ids may be NULL */
__device__ __forceinline__ void store_hit_record(const SceneView &sv, const d3 &o, const d3 &d, const HitRec &best, size_t i,
                                                 int *__restrict__ ids, long long *__restrict__ prims,
                                                 double *__restrict__ ts, double *__restrict__ points,
                                                 double *__restrict__ normals, double *__restrict__ uvs)
{
  bool hit = best.t < 1e300;
  Surface s;
  if (hit)
    s = surface_at(sv, o, d, best, true);
  ids[i] = hit ? s.object : -1;
  if (prims) prims[i] = hit ? (long long)best.gid : -1ll;
  if (ts) ts[i] = hit ? best.t : 0.0;
  if (points)  { points[3 * i] = hit ? s.point.x : 0; points[3 * i + 1] = hit ? s.point.y : 0; points[3 * i + 2] = hit ? s.point.z : 0; }
  if (normals) { normals[3 * i] = hit ? s.normal.x : 0; normals[3 * i + 1] = hit ? s.normal.y : 0; normals[3 * i + 2] = hit ? s.normal.z : 0; }
  if (uvs)     { uvs[2 * i] = hit ? s.u : 0; uvs[2 * i + 1] = hit ? s.v : 0; }
}

/* ---- camera (raytracer.c:375-384) ------------------------------------------- */

struct CameraView
{
  double pos[3], horizontal[3], vertical[3], llc[3];
};

__device__ __forceinline__ void camera_ray(const CameraView &c, double u, double v, d3 &o, d3 &d)
{
  d3 pos = d3_make(c.pos[0], c.pos[1], c.pos[2]);
  d3 H = d3_make(c.horizontal[0], c.horizontal[1], c.horizontal[2]);
  d3 V = d3_make(c.vertical[0], c.vertical[1], c.vertical[2]);
  d3 llc = d3_make(c.llc[0], c.llc[1], c.llc[2]);
  d3 on_plane = d3_add(llc, d3_add(d3_scale(H, u), d3_scale(V, v)));
  o = pos;
  d = d3_normalize(d3_sub(pos, on_plane));
}

/* ---- scatter helpers ---------------------------------------------------------- */

/* raytracer.c:349-352 */
__device__ __forceinline__ d3 reflect_dir(const d3 &in, const d3 &n)
{
  return d3_sub(in, d3_scale(n, __dmul_rn(2.0, d3_dot(in, n))));
}

/* raytracer.c:386-391: factor 0.3 or 0.7 */
__device__ __forceinline__ float checker_factor(double u, double v, double M)
{
  bool a = fmod(__dmul_rn(u, M), 1.0) > 0.5;
  bool b = fmod(__dmul_rn(v, M), 1.0) < 0.5;
  double on = (a ^ b) ? 1.0 : 0.0;
  return (float)__dadd_rn(__dmul_rn(0.3, __dsub_rn(1.0, on)), __dmul_rn(0.7, on));
}

#endif /* RTB_DEVICE_CUH */
