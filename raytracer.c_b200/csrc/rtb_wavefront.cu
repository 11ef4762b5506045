/*
 * rtb_wavefront.cu -- the wavefront form of render() (raytracer.c:176-223).
 *
 * Why it exists (profiles/r1_c3_default_ncu.md): in the megakernel a warp's 32 lanes each own
 * one path; after the first bounce the rays are incoherent and traversal lengths have a long
 * tail, so the warp waits for its slowest ray at every bounce -- 4 of 32 lanes were walking
 * on average.  Here a bounce is split in two kernels that exchange rays through queues in HBM:
 *
 *   k_wf_generate  camera samples (raytracer.c:203-209)                    -> queue[0]
 *   k_wf_trace     nearest hit for every queued ray.  PERSISTENT: a lane that finishes its
 *                  ray does not wait for its neighbours -- as soon as enough lanes are idle
 *                  the warp refills them from the queue (Aila & Laine's "replace terminated
 *                  rays", made cheap because a ray is one 64-byte read, not a shading pass)
 *   k_wf_shade     the body of trace_path after the scene query (raytracer.c:492-553) with all
 *                  lanes busy; survivors are appended to the next queue by warp-aggregated
 *                  atomics (ballot + one atomicAdd per warp)
 *
 * Queue entry = 80 bytes in five 16-byte SoA arrays (coalesced): origin and direction as
 * doubles, {path id, throughput}, and the hit record {t, gid, slot}.  The oversized-sphere
 * list is tested by the producer (all lanes busy), so the hit record arrives pre-seeded.
 *
 * Determinism: a path slot (plane, pixel) carries exactly one path per wave, so its float4
 * accumulator is read-modify-written by one thread at a time in vertex order -- the same
 * sequence of additions the megakernel performs in registers.  Queue ORDER depends on atomics,
 * results do not.  Sums are bit-identical to the megakernel's for the same number of planes.
 */
#include "rtb_path.cuh"

#include <algorithm>
#include <cstring>
#include <mutex>
#include <vector>
#include <cub/cub.cuh>

#define WF_FULL 0xFFFFFFFFu
#define WF_MAX_GROUPS RTB_WF_MAX_GROUPS /* plane groups in flight, one stream each */
#ifndef WF_SMEM_STACK
#define WF_SMEM_STACK 8
#endif
#ifndef WF_SHADE_BLOCKS
#define WF_SHADE_BLOCKS 8
#endif
#ifndef WF_TRACE_BLOCKS_PER_SM
#define WF_TRACE_BLOCKS_PER_SM 8
#endif

struct WfQueue
{
  double2 *o_xy;  /* origin.x, origin.y */
  double2 *oz_dx; /* origin.z, direction.x */
  double2 *d_yz;  /* direction.y, direction.z */
  uint4 *path;    /* path slot id, throughput r, g, b (float bits) */
  uint4 *hit;     /* best.t (two words), gid, slot */
  unsigned *branch; /* SPLIT dielectric estimator only (else NULL): branch id of the ray (PathState::branch) */
  unsigned cap;     /* entries the arrays hold; only the SPLIT estimator can run into it */
};


__device__ __forceinline__ uint4 pack_hit(const HitRec &h)
{
  return make_uint4((unsigned)__double2loint(h.t), (unsigned)__double2hiint(h.t), (unsigned)h.gid, (unsigned)h.slot);
}

__device__ __forceinline__ HitRec unpack_hit(const uint4 v)
{
  HitRec h;
  h.t = __hiloint2double((int)v.y, (int)v.x);
  h.gid = (int)v.z;
  h.slot = (int)v.w;
  return h;
}

/* the part of the scene query that does not walk the tree: oversized primitives */
__device__ __forceinline__ void ray_seed_hit(const SceneView &sv, const d3 &o, const d3 &d, HitRec &best, unsigned &exact)
{
  best.t = DBL_MAX;
  best.gid = 0x7FFFFFFF;
  best.slot = 0;
  RayF rf;
  rayf_basic(o, d, rf);
  big_list_select_test(sv, o, d, rf, best, exact);
}

/* ---- ray reordering key ---------------------------------------------------------------------
 * Secondary rays are incoherent; sorting a queue by a key built from the quantised origin and
 * direction puts rays that walk the same part of the tree into the same warp.
 * 18 origin bits (6 per axis, Morton order, relative to the guard box) and 6 direction bits
 * (octahedral map, 8x8 cells); `mode` picks how they are interleaved. */
__device__ __forceinline__ unsigned spread3(unsigned v) /* 6 bits -> every third bit */
{
  unsigned r = 0;
#pragma unroll
  for (int k = 0; k < 6; k++)
    r |= ((v >> k) & 1u) << (3 * k);
  return r;
}

__device__ __forceinline__ unsigned ray_sort_key(const SceneView &sv, const d3 &o, const d3 &d, int mode)
{
  unsigned q[3];
  const float of[3] = { (float)o.x, (float)o.y, (float)o.z };
#pragma unroll
  for (int k = 0; k < 3; k++)
  {
    const float ext = sv.guard_hi[k] - sv.guard_lo[k];
    /* the scene box is the middle third of the guard box: zoom into it */
    float u = (ext > 0.0f && ext < 1e30f) ? ((of[k] - sv.guard_lo[k]) / ext * 3.0f - 1.0f) : 0.0f;
    u = fminf(fmaxf(u, 0.0f), 0.999999f);
    q[k] = (unsigned)(u * 64.0f);
  }
  const unsigned morton = spread3(q[0]) | (spread3(q[1]) << 1) | (spread3(q[2]) << 2); /* 18 bits */
  /* octahedral direction -> 3 + 3 bits */
  float dx = (float)d.x, dy = (float)d.y, dz = (float)d.z;
  const float inv = 1.0f / (fabsf(dx) + fabsf(dy) + fabsf(dz) + 1e-30f);
  float px = dx * inv, py = dy * inv;
  if (dz < 0.0f)
  {
    const float ox_ = (1.0f - fabsf(py)) * (px >= 0.0f ? 1.0f : -1.0f);
    const float oy_ = (1.0f - fabsf(px)) * (py >= 0.0f ? 1.0f : -1.0f);
    px = ox_; py = oy_;
  }
  const unsigned du = (unsigned)fminf(fmaxf((px * 0.5f + 0.5f) * 8.0f, 0.0f), 7.0f);
  const unsigned dv = (unsigned)fminf(fmaxf((py * 0.5f + 0.5f) * 8.0f, 0.0f), 7.0f);
  const unsigned dir = (du << 3) | dv; /* 6 bits */
  const unsigned octant = (dx < 0.0f ? 1u : 0u) | (dy < 0.0f ? 2u : 0u) | (dz < 0.0f ? 4u : 0u);
  switch (mode)
  {
  case 1: return ((morton >> 6) << 12) | (dir << 6) | (morton & 63u);  /* origin hi | dir | origin lo */
  case 2: return (dir << 18) | morton;                                  /* direction major */
  case 3: return (morton << 6) | dir;                                   /* origin major */
  case 4: return (octant << 18) | morton;                               /* octant, then origin */
  case 5: return ((morton >> 9) << 15) | (dir << 9) | (morton & 511u); /* origin 3 bits/axis | dir | rest */
  default: return morton << 6;
  }
}

/* warp-aggregated append: every lane of the warp must call this */
__device__ __forceinline__ void wf_enqueue(const WfQueue &q, unsigned *count, bool want, int lane, const d3 &o, const d3 &d,
                                           unsigned pid, float tr, float tg, float tb, const HitRec &seed,
                                           unsigned *keys = nullptr, unsigned key = 0u, unsigned branch = 1u,
                                           unsigned *overflow = nullptr)
{
  const unsigned m = __ballot_sync(WF_FULL, want);
  if (m == 0u)
    return;
  const int leader = __ffs(m) - 1;
  unsigned base = 0;
  if (lane == leader)
    base = atomicAdd(count, (unsigned)__popc(m));
  base = __shfl_sync(WF_FULL, base, leader);
  if (want)
  {
    const unsigned i = base + (unsigned)__popc(m & ((1u << lane) - 1u));
    if (overflow != nullptr && i >= q.cap)
    {
      *overflow = 1u; /* the split tree outgrew the queue: the host retries with fewer paths per wave */
      return;
    }
    if (q.branch)
      __stcs(q.branch + i, branch);
    /* queue traffic is streamed once: evict-first, so it does not push the BVH out of L2 */
    __stcs(q.o_xy + i, make_double2(o.x, o.y));
    __stcs(q.oz_dx + i, make_double2(o.z, d.x));
    __stcs(q.d_yz + i, make_double2(d.y, d.z));
    __stcs(q.path + i, make_uint4(pid, __float_as_uint(tr), __float_as_uint(tg), __float_as_uint(tb)));
    __stcs(q.hit + i, pack_hit(seed));
    if (keys)
      __stcs(keys + i, key);
  }
}

__device__ __forceinline__ void wf_add_counters(unsigned long long *totals, int lane, unsigned long long c0,
                                                unsigned long long c1, unsigned long long c2, unsigned long long c3,
                                                unsigned long long c4)
{
  for (int off = 16; off > 0; off >>= 1)
  {
    c0 += __shfl_xor_sync(WF_FULL, c0, off);
    c1 += __shfl_xor_sync(WF_FULL, c1, off);
    c2 += __shfl_xor_sync(WF_FULL, c2, off);
    c3 += __shfl_xor_sync(WF_FULL, c3, off);
    c4 += __shfl_xor_sync(WF_FULL, c4, off);
  }
  if (lane == 0)
  {
    if (c0) atomicAdd(&totals[0], c0);
    if (c1) atomicAdd(&totals[1], c1);
    if (c2) atomicAdd(&totals[2], c2);
    if (c3) atomicAdd(&totals[3], c3);
    if (c4) atomicAdd(&totals[4], c4);
  }
}

/* ---- camera samples of one wave ------------------------------------------------------------
 * One thread per path slot; warps map to 8x4 pixel tiles of one plane so that the primary
 * rays a trace warp later fetches together are coherent.  The planes that still have a sample
 * in this wave are a prefix [0, n_valid_planes), so the queue position of a ray is computed,
 * not allocated: no atomics (one same-address atomic per warp made this kernel atomic-bound,
 * 8 % of a step). */
__global__ void __launch_bounds__(256, 4) k_wf_generate(const __grid_constant__ RenderArgs A, int wave, int n_valid_planes,
                                                     WfQueue q, unsigned *count)
{
  __shared__ unsigned s_exact;
  if (threadIdx.x == 0)
    s_exact = 0u;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int tile = (int)(warp % A.n_tiles);
  const int plane = (int)(warp / A.n_tiles); /* within this launch's group of planes (A.plane_base is its first) */
  const int x = (tile % A.tiles_x) * 8 + (lane & 7);
  const int y = (tile / A.tiles_x) * 4 + (lane >> 3);
  const int s = A.s_begin + (A.plane_base + plane) * A.chunk + wave;
  const bool valid = x < A.width && y < A.height && plane < n_valid_planes;
  const unsigned n_px = (unsigned)(A.width * A.height);
  const unsigned pixel = (unsigned)(y * A.width + x);
  const bool tiled = (A.width % 8) == 0 && (A.height % 4) == 0; /* every lane of every tile is a pixel */

  unsigned exact = 0;
  if (valid)
  {
    PathState st;
    HitRec seed;
    path_begin(A, st, x, y, pixel, (unsigned)s);
    ray_seed_hit(A.sv, st.o, st.d, seed, exact);
    const unsigned pid = (unsigned)(A.plane_base + plane) * n_px + pixel;
    const unsigned i = (unsigned)plane * n_px + (tiled ? (unsigned)tile * 32u + (unsigned)lane : pixel);
    __stcs(q.o_xy + i, make_double2(st.o.x, st.o.y));
    __stcs(q.oz_dx + i, make_double2(st.o.z, st.d.x));
    __stcs(q.d_yz + i, make_double2(st.d.y, st.d.z));
    __stcs(q.path + i, make_uint4(pid, __float_as_uint(st.tr), __float_as_uint(st.tg), __float_as_uint(st.tb)));
    __stcs(q.hit + i, pack_hit(seed));
    if (q.branch)
      __stcs(q.branch + i, 1u);
  }
  for (int off = 16; off > 0; off >>= 1)
    exact += __shfl_xor_sync(WF_FULL, exact, off);
  if (lane == 0 && exact)
    atomicAdd(&s_exact, exact);
  __syncthreads();
  if (threadIdx.x == 0)
  {
    if (s_exact)
      atomicAdd(&A.counters[2], (unsigned long long)s_exact);
    if (blockIdx.x == 0)
    {
      const unsigned n = (unsigned)n_valid_planes * n_px;
      *count = n;
      atomicAdd(&A.counters[4], (unsigned long long)n);
    }
  }
}

/* ---- nearest hit for a whole queue -----------------------------------------------------------
 * Persistent warps.  Each warp grabs batches of consecutive rays (one atomic per batch) and
 * keeps its lanes supplied from the batch: whenever `refill_idle` or more lanes have no ray,
 * the walk is interrupted and the idle lanes load the next rays.  The walk itself is the
 * while-while loop of closest_hit_ww (inner nodes until every lane has reached a leaf, then
 * the exact FP64 leaf tests together).
 * V (variant bits): 1 = the double-precision ray is NOT kept in registers during the walk but
 * re-read from the queue at every leaf (fewer registers -> more warps per SM);
 * 2 = streaming (evict-first) loads/stores for queue data; 4 = whole traversal stack in local
 * memory (no shared-memory top); 8 = BVH4 (128-byte nodes, rtb_internal.h); 16 = compressed BVH4 (64-byte nodes);
 * 32 / 64 = with 16: 6 / 12 of the 24 plane-byte conversions of a node on the ALU + FMA pipes instead of
 * the conversion pipe; 128 = pops read the top two stack entries at once.
 * (Measured and removed in round 2, profiles/r2_wf_tuning.md: prefetching the next rays of the batch into
 * L1 / L2 after every refill; reading the FP32 walk set-up from the queue, written by the producer;
 * prefetching a leaf's primitives when the walk reaches it; dropping the whole stack at once when a hit
 * ends before the nearest entry ever pushed.) */
template <int V> struct WfTraceCfg { static constexpr int blocks = (V & 1) ? 10 : 8; static constexpr int sd = (V & 4) ? 0 : WF_SMEM_STACK; };

__device__ __forceinline__ double2 wf_ld(const double2 *p, bool stream)
{
  return stream ? __ldcs(p) : *p;
}
__device__ __forceinline__ uint4 wf_ld(const uint4 *p, bool stream)
{
  return stream ? __ldcs(p) : *p;
}

/* T64: the scene carries double-precision triangle vertices (SceneView::tri64); a separate instantiation so
 * that the common case -- float-representable meshes -- has no extra branch in the leaf loop */
template <bool STATS, int V, bool T64 = false>
__global__ void __launch_bounds__(128, WfTraceCfg<V>::blocks)
k_wf_trace(const __grid_constant__ SceneView sv, WfQueue q, const unsigned *__restrict__ n_ptr, unsigned *fetch_ctr,
           unsigned long long *totals, int refill_idle_word, int node_exit, const unsigned *__restrict__ perm)
{
  const int refill_idle = refill_idle_word & 0xFF;
  const unsigned guided = (unsigned)(refill_idle_word >> 8); /* != 0: batches shrink with the rays left in the queue */
  constexpr bool RELOAD = (V & 1) != 0, STREAM = (V & 2) != 0;
  constexpr int WIDE = (V & 16) ? (2 + ((V >> 5) & 3)) : ((V & 8) ? 1 : 0);
  constexpr bool POP2 = (V & 128) != 0;
  constexpr int SD = WfTraceCfg<V>::sd;
  __shared__ int2 s_stack[SD > 0 ? SD : 1][128];
  const int lane = threadIdx.x & 31;
  const unsigned n = min(*n_ptr, q.cap);
  const unsigned n_warps = (gridDim.x * blockDim.x) >> 5;
  /* batch: large enough to make the atomic rare, small enough that every warp gets work */
  unsigned batch = (n / (n_warps * 4u)) & ~31u;
  batch = batch < 32u ? 32u : (batch > 512u ? 512u : batch);

  unsigned next = 0, end = 0; /* the warp's current batch, warp-uniform */
  bool pool_empty = n == 0u;

  bool active = false;
  unsigned ray = 0;
  d3 o = d3_make(0, 0, 0), d = d3_make(0, 0, 1);
  RayF rf;
  rf.idx = rf.idy = rf.idz = rf.oodx = rf.oody = rf.oodz = rf.tmax = rf.t_base = 0.0f;
  HitRec best;
  best.t = DBL_MAX; best.gid = 0x7FFFFFFF; best.slot = 0;
  int2 stack_mem[RTB_STACK_SIZE - SD];
  WalkStack<SD> stack = { &s_stack[0][threadIdx.x], stack_mem, 128 };
  stack.reset();
  int cur = RTB_REF_NONE;
  unsigned node_visits = 0, prim_tests = 0;

  while (true)
  {
    /* ---- refill idle lanes ---- */
    unsigned bidle = __ballot_sync(WF_FULL, !active);
    while (bidle != 0u && !pool_empty)
    {
      if (next >= end)
      {
        unsigned base = 0, take = batch;
        if (lane == 0)
        {
          if (guided != 0u && batch > 32u)
          {
            /* guided self-scheduling: a batch is this warp's share of what is left (a stale read of the
             * cursor only changes the size, never the ownership, of a batch), so the last batches are short
             * and the kernel's tail is one short batch, not one of 512 rays */
            const unsigned cur_ = *reinterpret_cast<volatile unsigned *>(fetch_ctr);
            const unsigned left = cur_ < n ? n - cur_ : 0u;
            const unsigned cap_ = 512u << (guided >> 4);
            take = (left / (n_warps * (guided & 15u))) & ~31u;
            take = take < 32u ? 32u : (take > cap_ ? cap_ : take);
          }
          base = atomicAdd(fetch_ctr, take);
        }
        base = __shfl_sync(WF_FULL, base, 0);
        take = __shfl_sync(WF_FULL, take, 0);
        if (base >= n)
        {
          pool_empty = true;
          break;
        }
        next = base;
        end = min(base + take, n);
      }
      const unsigned mine = next + (unsigned)__popc(bidle & ((1u << lane) - 1u));
      /* only the lanes counted in bidle take a ray: a lane served earlier in this refill whose ray
       * needed no walk is idle too, but it is not in bidle and must not fetch a duplicate */
      const bool take = ((bidle >> lane) & 1u) != 0u && mine < end;
      if (take)
      {
        ray = perm ? __ldcs(perm + mine) : mine;
        const double2 a = wf_ld(q.o_xy + ray, STREAM), b = wf_ld(q.oz_dx + ray, STREAM), c = wf_ld(q.d_yz + ray, STREAM);
        d3 o_ = d3_make(a.x, a.y, b.x), d_ = d3_make(b.y, c.x, c.y);
        best = unpack_hit(wf_ld(q.hit + ray, STREAM));
        rayf_basic(o_, d_, rf);
        if (rayf_walk_setup(sv, o_, d_, best, rf))
        {
          stack.reset();
          cur = sv.root_ref;
          active = cur != RTB_REF_NONE;
        }
        if (!RELOAD)
        {
          o = o_;
          d = d_;
        }
        /* else: the seeded hit record is already final, the lane stays idle */
      }
      next = min(next + (unsigned)__popc(bidle), end);
      /* lanes the batch could not serve try the next batch; a lane whose ray needed no walk
       * (the seeded hit record is final) is refilled on the next trip of the outer loop */
      bidle = __ballot_sync(WF_FULL, ((bidle >> lane) & 1u) != 0u && mine >= end);
    }
    if (__all_sync(WF_FULL, !active))
    {
      if (pool_empty)
        break;
      continue;
    }

    /* ---- walk until enough lanes are idle again ---- */
    while (true)
    {
      if (node_exit <= 0)
      {
        while (cur >= 0 && cur != RTB_REF_NONE)
        {
          if (STATS) node_visits++;
          int nxt = node_step_w<WIDE>(sv, rf, cur, stack);
          cur = (nxt != RTB_REF_NONE) ? nxt : (POP2 ? stack.pop2(rf) : stack.pop(rf));
        }
      }
      else
      {
        /* leave the node phase as soon as fewer than node_exit lanes are still at inner nodes */
        while (true)
        {
          const bool at_node = cur >= 0 && cur != RTB_REF_NONE;
          const unsigned bnode = __ballot_sync(WF_FULL, at_node);
          if (bnode == 0u)
            break;
          if (at_node)
          {
            if (STATS) node_visits++;
            int nxt = node_step_w<WIDE>(sv, rf, cur, stack);
            cur = (nxt != RTB_REF_NONE) ? nxt : (POP2 ? stack.pop2(rf) : stack.pop(rf));
          }
          if (__popc(bnode) < node_exit)
            break;
        }
      }
      if (cur < 0)
      {
        if (RELOAD)
        {
          const double2 a = q.o_xy[ray], b = q.oz_dx[ray], c = q.d_yz[ray];
          o = d3_make(a.x, a.y, b.x);
          d = d3_make(b.y, c.x, c.y);
        }
        const int code = ~cur;
        const int first = code >> 3, count = (code & 7) + 1;
        for (int k = 0; k < count; k++)
          test_prim(load_prim(sv.prims, first + k), first + k, o, d, best, T64 ? sv.tri64 : nullptr);
        prim_tests += (unsigned)count;
        rayf_update_tmax(rf, best);
        cur = POP2 ? stack.pop2(rf) : stack.pop(rf);
      }
      if (active && cur == RTB_REF_NONE)
      {
        if (STREAM)
          __stcs(q.hit + ray, pack_hit(best));
        else
          q.hit[ray] = pack_hit(best);
        active = false;
      }
      const unsigned bact = __ballot_sync(WF_FULL, active);
      if (bact == 0u)
        break;
      if (!pool_empty && 32 - __popc(bact) >= refill_idle)
        break;
    }
  }

  wf_add_counters(totals, lane, 0ull, 0ull, prim_tests, STATS ? node_visits : 0u, 0ull);
}

template <int V>
static void launch_trace(bool stats, int sm_count, cudaStream_t stream, const SceneView &sv,
                         const WfQueue &q, const unsigned *n_ptr, unsigned *fetch, unsigned long long *totals,
                         int refill_idle, int node_exit, const unsigned *perm)
{
  const int blocks = sm_count * WfTraceCfg<V>::blocks;
  if (sv.tri64 != nullptr)
  {
    if (stats)
      k_wf_trace<true, V, true><<<blocks, 128, 0, stream>>>(sv, q, n_ptr, fetch, totals, refill_idle, node_exit, perm);
    else
      k_wf_trace<false, V, true><<<blocks, 128, 0, stream>>>(sv, q, n_ptr, fetch, totals, refill_idle, node_exit, perm);
  }
  else if (stats)
    k_wf_trace<true, V><<<blocks, 128, 0, stream>>>(sv, q, n_ptr, fetch, totals, refill_idle, node_exit, perm);
  else
    k_wf_trace<false, V><<<blocks, 128, 0, stream>>>(sv, q, n_ptr, fetch, totals, refill_idle, node_exit, perm);
}


/* ---- nearest hit for a whole queue, "ray pool" form --------------------------------------------------
 * k_wf_trace ties a ray to a lane: whatever phase most lanes are in runs, the others idle -- 16.9 of 32
 * lanes per issued instruction (profiles/r2_wf_trace_ncu.md: node step 20 lanes, leaf tests 8-12, refill
 * 12-16, pop loops 4-7).  Here a warp owns a POOL of WF_POOL_RAYS rays whose walk state lives in shared
 * memory and whose traversal stacks live in global memory, indexed by pool slot, so ANY lane can advance
 * ANY ray.  Three lists (slots waiting for a node step, for a leaf test, free slots) are kept by
 * warp-aggregated appends; every turn the warp takes up to 32 slots from ONE list and runs that phase with
 * (nearly) all lanes.  Same node step, same exact tests, same acceptance rule: the hit records are
 * bit-identical to k_wf_trace's. */
#ifndef WF_POOL_RAYS
#define WF_POOL_RAYS 64
#endif

/* The WalkStack interface for a pool slot.  Entry k of the slot's stack lives in global memory at
 * base[k * WF_POOL_RAYS] (L1 does not allocate on a store, so a pop of it is an L2 round trip); the TOP entry
 * is therefore kept in shared memory (loaded into top_ref / top_dist for the duration of a step): the pop
 * that follows a node without hit children -- the common one -- never leaves the SM.  Deeper pops read four
 * entries at once. */
struct PoolStack
{
  int2 *base;
  int sp;         /* entries in global memory (the cached top not counted) */
  int top_ref;    /* RTB_REF_NONE: no cached top */
  float top_dist;
  __device__ __forceinline__ void push(int2 e)
  {
    if (top_ref != RTB_REF_NONE)
    {
      base[(size_t)sp * WF_POOL_RAYS] = make_int2(top_ref, __float_as_int(top_dist));
      sp++;
    }
    top_ref = e.x;
    top_dist = __int_as_float(e.y);
  }
  __device__ __forceinline__ int pop(const RayF &rf)
  {
    if (top_ref != RTB_REF_NONE)
    {
      const int r = top_ref;
      top_ref = RTB_REF_NONE;
      if (top_dist <= rf.tmax)
        return r;
    }
    while (sp > 0)
    {
      int2 e[4];
#pragma unroll
      for (int k = 0; k < 4; k++)
        e[k] = base[(size_t)max(sp - 1 - k, 0) * WF_POOL_RAYS];
#pragma unroll
      for (int k = 0; k < 4; k++)
        if (sp - 1 - k >= 0 && __int_as_float(e[k].y) <= rf.tmax)
        {
          sp = sp - 1 - k;
          return e[k].x;
        }
      sp = max(sp - 4, 0);
    }
    return RTB_REF_NONE;
  }
};

struct PoolShared /* one per warp */
{
  int cur[WF_POOL_RAYS], sp[WF_POOL_RAYS];
  float idx[WF_POOL_RAYS], idy[WF_POOL_RAYS], idz[WF_POOL_RAYS];
  float oodx[WF_POOL_RAYS], oody[WF_POOL_RAYS], oodz[WF_POOL_RAYS];
  float tmax[WF_POOL_RAYS], tbase[WF_POOL_RAYS];
  int t_lo[WF_POOL_RAYS], t_hi[WF_POOL_RAYS], gid[WF_POOL_RAYS], slot[WF_POOL_RAYS];
  int top_ref[WF_POOL_RAYS];
  float top_dist[WF_POOL_RAYS];
  unsigned ray[WF_POOL_RAYS];
  unsigned char node_list[WF_POOL_RAYS], leaf_list[WF_POOL_RAYS], free_list[WF_POOL_RAYS];
};

/* every lane of the warp calls this: lanes with `want` append `value` to list[0 .. n) */
__device__ __forceinline__ void pool_append(unsigned char *list, int &n, bool want, unsigned value, int lane)
{
  const unsigned m = __ballot_sync(WF_FULL, want);
  if (want)
    list[n + __popc(m & ((1u << lane) - 1u))] = (unsigned char)value;
  n += __popc(m);
}

template <bool STATS, bool T64>
__global__ void __launch_bounds__(128, 8)
k_wf_trace_pool(const __grid_constant__ SceneView sv, WfQueue q, const unsigned *__restrict__ n_ptr, unsigned *fetch_ctr,
                unsigned long long *totals, int2 *__restrict__ stacks, int leaf_min)
{
  __shared__ PoolShared s_pool[4];
  const int lane = threadIdx.x & 31;
  PoolShared &P = s_pool[threadIdx.x >> 5];
  const unsigned gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int2 *const my_stacks = stacks + (size_t)gwarp * RTB_STACK_SIZE * WF_POOL_RAYS;
  const unsigned n = min(*n_ptr, q.cap);
  const unsigned n_warps = (gridDim.x * blockDim.x) >> 5;
  unsigned batch = (n / (n_warps * 4u)) & ~31u;
  batch = batch < 32u ? 32u : (batch > 512u ? 512u : batch);
  unsigned next = 0, end = 0; /* the warp's current batch */
  bool pool_empty = n == 0u;

  int n_node = 0, n_leaf = 0, n_free = WF_POOL_RAYS;
  for (int k = lane; k < WF_POOL_RAYS; k += 32)
    P.free_list[k] = (unsigned char)k;
  __syncwarp();
  unsigned node_visits = 0, prim_tests = 0;

  while (true)
  {
    /* ---- which phase runs this turn: one that can fill the warp, else the fullest list ---- */
    enum { PH_NODE, PH_LEAF, PH_FILL, PH_NONE };
    const int can_fill = pool_empty ? 0 : n_free;
    int phase;
    if (can_fill >= 32) phase = PH_FILL;
    else if (n_node >= 32) phase = PH_NODE;
    else if (n_leaf >= leaf_min) phase = PH_LEAF;
    else if (can_fill > 0 && can_fill >= n_node) phase = PH_FILL;
    else if (n_node > 0) phase = PH_NODE;
    else if (n_leaf > 0) phase = PH_LEAF;
    else if (can_fill > 0) phase = PH_FILL;
    else break;

    int s = -1;                /* the pool slot this lane works on */
    int nxt = RTB_REF_NONE;    /* where its ray stands afterwards */
    bool worked = false;

    if (phase == PH_FILL)
    {
      if (next >= end)
      {
        unsigned base = 0;
        if (lane == 0)
          base = atomicAdd(fetch_ctr, batch);
        base = __shfl_sync(WF_FULL, base, 0);
        if (base >= n)
        {
          pool_empty = true;
          continue;
        }
        next = base;
        end = min(base + batch, n);
      }
      const int k = min(min(32, n_free), (int)(end - next));
      if (lane < k)
      {
        s = P.free_list[n_free - k + lane];
        const unsigned ray = next + (unsigned)lane;
        const double2 a = __ldcs(q.o_xy + ray), b = __ldcs(q.oz_dx + ray), c = __ldcs(q.d_yz + ray);
        const d3 o = d3_make(a.x, a.y, b.x), d = d3_make(b.y, c.x, c.y);
        const uint4 hv = __ldcs(q.hit + ray);
        const HitRec best = unpack_hit(hv);
        RayF rf;
        rayf_basic(o, d, rf);
        rf.idx = rf.idy = rf.idz = rf.oodx = rf.oody = rf.oodz = rf.tmax = rf.t_base = 0.0f;
        worked = true;
        if (rayf_walk_setup(sv, o, d, best, rf))
        {
          nxt = sv.root_ref;
          P.sp[s] = 0;
          P.top_ref[s] = RTB_REF_NONE;
          P.idx[s] = rf.idx; P.idy[s] = rf.idy; P.idz[s] = rf.idz;
          P.oodx[s] = rf.oodx; P.oody[s] = rf.oody; P.oodz[s] = rf.oodz;
          P.tmax[s] = rf.tmax; P.tbase[s] = rf.t_base;
          P.t_lo[s] = (int)hv.x; P.t_hi[s] = (int)hv.y; P.gid[s] = (int)hv.z; P.slot[s] = (int)hv.w;
          P.ray[s] = ray;
          P.cur[s] = nxt;
        }
        /* else: the seeded hit record in the queue is already final; the slot stays free */
      }
      n_free -= k;
      next += (unsigned)k;
    }
    else if (phase == PH_NODE)
    {
      const int k = min(32, n_node);
      if (lane < k)
      {
        s = P.node_list[n_node - k + lane];
        RayF rf;
        rf.idx = P.idx[s]; rf.idy = P.idy[s]; rf.idz = P.idz[s];
        rf.oodx = P.oodx[s]; rf.oody = P.oody[s]; rf.oodz = P.oodz[s];
        rf.tmax = P.tmax[s];
        PoolStack stack = { my_stacks + s, P.sp[s], P.top_ref[s], P.top_dist[s] };
        if (STATS) node_visits++;
        nxt = node_step4q<0>(sv, rf, P.cur[s], stack);
        if (nxt == RTB_REF_NONE)
          nxt = stack.pop(rf);
        P.sp[s] = stack.sp;
        P.top_ref[s] = stack.top_ref;
        P.top_dist[s] = stack.top_dist;
        P.cur[s] = nxt;
        worked = true;
      }
      n_node -= k;
    }
    else /* PH_LEAF */
    {
      const int k = min(32, n_leaf);
      if (lane < k)
      {
        s = P.leaf_list[n_leaf - k + lane];
        const unsigned ray = P.ray[s];
        const double2 a = __ldcg(q.o_xy + ray), b = __ldcg(q.oz_dx + ray), c = __ldcg(q.d_yz + ray);
        const d3 o = d3_make(a.x, a.y, b.x), d = d3_make(b.y, c.x, c.y);
        HitRec best;
        best.t = __hiloint2double(P.t_hi[s], P.t_lo[s]);
        best.gid = P.gid[s];
        best.slot = P.slot[s];
        const int code = ~P.cur[s];
        const int first = code >> 3, count = (code & 7) + 1;
        const double t_before = best.t;
        const int gid_before = best.gid;
        for (int j = 0; j < count; j++)
          test_prim(load_prim(sv.prims, first + j), first + j, o, d, best, T64 ? sv.tri64 : nullptr);
        prim_tests += (unsigned)count;
        RayF rf;
        rf.tmax = P.tmax[s];
        rf.t_base = P.tbase[s];
        if (best.t != t_before || best.gid != gid_before)
        {
          rayf_update_tmax(rf, best);
          P.tmax[s] = rf.tmax;
          P.t_lo[s] = __double2loint(best.t); P.t_hi[s] = __double2hiint(best.t);
          P.gid[s] = best.gid; P.slot[s] = best.slot;
        }
        PoolStack stack = { my_stacks + s, P.sp[s], P.top_ref[s], P.top_dist[s] };
        nxt = stack.pop(rf);
        P.sp[s] = stack.sp;
        P.top_ref[s] = stack.top_ref;
        P.cur[s] = nxt;
        worked = true;
      }
      n_leaf -= k;
    }

    /* ---- where every worked-on ray goes next ---- */
    const bool to_node = worked && nxt >= 0 && nxt != RTB_REF_NONE;
    const bool to_leaf = worked && nxt < 0;
    const bool finished = worked && nxt == RTB_REF_NONE;
    if (finished && phase != PH_FILL)
    {
      /* the walk of this ray is over: its hit record goes back to the queue */
      const HitRec best = { __hiloint2double(P.t_hi[s], P.t_lo[s]), P.gid[s], P.slot[s] };
      __stcs(q.hit + P.ray[s], pack_hit(best));
    }
    __syncwarp();
    pool_append(P.node_list, n_node, to_node, (unsigned)s, lane);
    pool_append(P.leaf_list, n_leaf, to_leaf, (unsigned)s, lane);
    pool_append(P.free_list, n_free, finished, (unsigned)s, lane);
    __syncwarp();
  }
  wf_add_counters(totals, lane, 0ull, 0ull, prim_tests, STATS ? node_visits : 0u, 0ull);
}

static void launch_trace_pool(bool stats, int sm_count, cudaStream_t stream, const SceneView &sv, const WfQueue &q,
                              const unsigned *n_ptr, unsigned *fetch, unsigned long long *totals, int2 *stacks, int leaf_min)
{
  const int blocks = sm_count * 8;
  const bool t64 = sv.tri64 != nullptr;
  if (stats)
  {
    if (t64) k_wf_trace_pool<true, true><<<blocks, 128, 0, stream>>>(sv, q, n_ptr, fetch, totals, stacks, leaf_min);
    else k_wf_trace_pool<true, false><<<blocks, 128, 0, stream>>>(sv, q, n_ptr, fetch, totals, stacks, leaf_min);
  }
  else
  {
    if (t64) k_wf_trace_pool<false, true><<<blocks, 128, 0, stream>>>(sv, q, n_ptr, fetch, totals, stacks, leaf_min);
    else k_wf_trace_pool<false, false><<<blocks, 128, 0, stream>>>(sv, q, n_ptr, fetch, totals, stacks, leaf_min);
  }
}

/* ---- shading of a whole queue ------------------------------------------------------------------
 * Thread i handles ray i: the body of trace_path after intersect() (path_shade), then, if the
 * path goes on, the oversized-list test of the NEXT ray and a warp-aggregated append. */
/* SPLIT: the reference's deterministic two-way split at dielectrics (raytracer.c:522-529): a vertex may append
 * two rays, several rays of one path slot are in flight at once (so the accumulator is updated with atomics
 * and the sums are no longer bit-reproducible), and the queue can overflow (flag -> host retries smaller). */
template <bool SPLIT>
__global__ void __launch_bounds__(128, WF_SHADE_BLOCKS) k_wf_shade(const __grid_constant__ RenderArgs A, int wave, int depth, WfQueue qin,
                                                  const unsigned *__restrict__ n_in, WfQueue qout, unsigned *n_out,
                                                  float4 *__restrict__ planes, unsigned *keys_out, int sort_mode,
                                                  unsigned *overflow)
{
  const int lane = threadIdx.x & 31;
  const unsigned n = min(*n_in, qin.cap);
  const unsigned gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const unsigned n_warps = (gridDim.x * blockDim.x) >> 5;
  const unsigned n_px = (unsigned)(A.width * A.height);
  PathCounters pc = { 0u, 0u };
  unsigned exact = 0;

  for (unsigned base = gwarp * 32u; base < n; base += n_warps * 32u)
  {
    const unsigned i = base + (unsigned)lane;
    PathState st;
    st.o = d3_make(0, 0, 0);
    st.d = d3_make(0, 0, 1);
    st.tr = st.tg = st.tb = 0.0f;
    st.depth = depth;
    st.alive = false;
    st.branch = 1u;
    PathState second;
    second.alive = false;
    unsigned pid = 0;
    HitRec seed, seed2;
    seed.t = DBL_MAX; seed.gid = 0x7FFFFFFF; seed.slot = 0;
    seed2 = seed;
    if (i < n)
    {
      const uint4 p = __ldcs(qin.path + i);
      const double2 a = __ldcs(qin.o_xy + i), b = __ldcs(qin.oz_dx + i), c = __ldcs(qin.d_yz + i);
      const HitRec best = unpack_hit(__ldcs(qin.hit + i));
      pid = p.x;
      st.o = d3_make(a.x, a.y, b.x);
      st.d = d3_make(b.y, c.x, c.y);
      st.tr = __uint_as_float(p.y); st.tg = __uint_as_float(p.z); st.tb = __uint_as_float(p.w);
      st.alive = true;
      const unsigned plane = pid / n_px;
      const unsigned pixel = pid - plane * n_px;
      const unsigned sample = (unsigned)(A.s_begin + (int)plane * A.chunk + wave);
      pc.rays++;
      pc.rays_hit++;
      if (SPLIT)
      {
        st.branch = __ldcs(qin.branch + i);
        float r = 0.0f, g = 0.0f, b2 = 0.0f;
        path_shade<true>(A, st, best, pixel, sample, r, g, b2, pc, nullptr, &second);
        float *acc = reinterpret_cast<float *>(planes + pid);
        if (r != 0.0f) atomicAdd(acc + 0, r);
        if (g != 0.0f) atomicAdd(acc + 1, g);
        if (b2 != 0.0f) atomicAdd(acc + 2, b2);
        if (second.alive)
          ray_seed_hit(A.sv, second.o, second.d, seed2, exact);
      }
      else
      {
        float4 acc = __ldcs(planes + pid);
        const float4 before = acc;
        path_shade<false>(A, st, best, pixel, sample, acc.x, acc.y, acc.z, pc, nullptr);
        if (__float_as_uint(acc.x) != __float_as_uint(before.x) || __float_as_uint(acc.y) != __float_as_uint(before.y) ||
            __float_as_uint(acc.z) != __float_as_uint(before.z))
          __stcs(planes + pid, acc);
      }
      if (st.alive)
        ray_seed_hit(A.sv, st.o, st.d, seed, exact);
    }
    wf_enqueue(qout, n_out, st.alive, lane, st.o, st.d, pid, st.tr, st.tg, st.tb, seed, keys_out,
               (keys_out && st.alive) ? ray_sort_key(A.sv, st.o, st.d, sort_mode) : 0u, st.branch, SPLIT ? overflow : nullptr);
    if (SPLIT)
      wf_enqueue(qout, n_out, second.alive, lane, second.o, second.d, pid, second.tr, second.tg, second.tb, seed2, nullptr, 0u,
                 second.branch, overflow);
  }
  wf_add_counters(A.counters, lane, pc.rays, pc.rays_hit, exact, 0ull, 0ull);
}

/* out[pixel][c] = sum over planes, in plane order (deterministic; same order as k_sum_planes) */
__global__ void k_wf_sum_planes(const float4 *__restrict__ planes, int n_planes, unsigned n_px, float *__restrict__ out)
{
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_px)
    return;
  float r = 0.0f, g = 0.0f, b = 0.0f;
  for (int k = 0; k < n_planes; k++)
  {
    const float4 v = planes[(size_t)k * n_px + i];
    r += v.x; g += v.y; b += v.z;
  }
  out[3 * (size_t)i + 0] = r;
  out[3 * (size_t)i + 1] = g;
  out[3 * (size_t)i + 2] = b;
}

/* ---- host ---------------------------------------------------------------------------------- */

__global__ void k_wf_iota(unsigned *v, unsigned n)
{
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n)
    v[i] = i;
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

/* the trace kernel a tuning word selects (rtb_render_desc.reserved): bits 0-7 refill threshold, 8-15 node-phase
 * exit threshold, 16-27 trace kernel variant; 0 = the measured defaults */
struct WfTraceTune
{
  int variant;     /* template argument of k_wf_trace */
  bool pool;       /* k_wf_trace_pool instead */
  int refill_word; /* refill threshold | guided batch word << 8 */
  int node_exit;   /* 0 = pure while-while */
  int leaf_min;    /* k_wf_trace_pool: leaf-phase threshold */
};

static int wf_trace_tune(const SceneView &sv, int tune, WfTraceTune &t)
{
  int refill_idle = ((tune & 0xFF) > 0 && (tune & 0xFF) <= 32) ? (tune & 0xFF) : 8;
  /* bits 8-15 of the word handed to k_wf_trace: guided self-scheduling of the ray batches -- a batch is
   * min(512 << (g >> 4), rays left / (warps * (g & 15))), at least 32.  Measured default g = 1
   * (profiles/r2_wf_tuning.md section 2i); development knob RTB_WF_GUIDED (0: fixed batches) */
  {
    const char *e = getenv("RTB_WF_GUIDED");
    refill_idle |= (e ? (atoi(e) & 0xFF) : 1) << 8;
  }
  t.refill_word = refill_idle;
  t.node_exit = (tune >> 8) & 0xFF;
  t.variant = (tune >> 16) & 0xFFF;
  if (tune == 0)
  {
    /* measured defaults (profiles/r1_wf_tuning.md) */
    t.node_exit = 16;
    t.variant = 22; /* compressed BVH4 + local stack + streaming queue loads */
  }
  if (t.node_exit == 0xFF)
    t.node_exit = 0; /* pure while-while */
  if ((t.variant & (8 | 16)) != 0 && sv.nodes4q == nullptr && sv.root_ref >= 0 && sv.root_ref != RTB_REF_NONE)
    t.variant = 6; /* the scene has no BVH4 (tree too deep for its stack): BVH2 walk */
  t.pool = t.variant == 1024 && sv.nodes4q != nullptr; /* the ray-pool form of the trace kernel */
  t.leaf_min = (tune & 0xFF00) ? std::min(std::max(t.node_exit, 1), 32) : 32;
  /* the BVH2 and the uncompressed BVH4 exist only in RTB_SCENE_ALL_TREES scenes (or as the fallback above) */
  const bool walks = sv.root_ref >= 0 && sv.root_ref != RTB_REF_NONE;
  const bool bvh2 = !t.pool && (t.variant & (8 | 16)) == 0, bvh4 = !t.pool && (t.variant & (8 | 16)) == 8;
  if (walks && ((bvh2 && sv.nodes == nullptr) || (bvh4 && sv.nodes4 == nullptr)))
  {
    rtb_set_error("wavefront trace variant " + std::to_string(t.variant) +
                  " walks the BVH2 / uncompressed BVH4: create the scene with RTB_SCENE_ALL_TREES");
    return RTB_EINVAL;
  }
  return RTB_OK;
}

/* device bytes of the ray pool's traversal stacks (0 unless the tuning word selects the pool) */
static size_t wf_pool_stack_bytes(const WfTraceTune &t, int sm_count)
{
  return t.pool ? align_up((size_t)sm_count * 8 * 4 * RTB_STACK_SIZE * WF_POOL_RAYS * sizeof(int2), 256) : 0;
}

/* one launch of the trace kernel `t` selects over queue q (the ray pool reads the queue in order: no perm) */
static void wf_launch_trace(const WfTraceTune &t, bool stats, int sm_count, cudaStream_t st, const SceneView &sv,
                            const WfQueue &q, const unsigned *n_ptr, unsigned *fetch, unsigned long long *totals,
                            int2 *pool_stacks, const unsigned *perm)
{
  const int ri = t.refill_word, ne = t.node_exit;
  if (t.pool)
  {
    launch_trace_pool(stats, sm_count, st, sv, q, n_ptr, fetch, totals, pool_stacks, t.leaf_min);
    return;
  }
  switch (t.variant)
  {
  case 2: launch_trace<2>(stats, sm_count, st, sv, q, n_ptr, fetch, totals, ri, ne, perm); break;
  case 22: launch_trace<22>(stats, sm_count, st, sv, q, n_ptr, fetch, totals, ri, ne, perm); break;
  case 54: launch_trace<54>(stats, sm_count, st, sv, q, n_ptr, fetch, totals, ri, ne, perm); break;
  case 86: launch_trace<86>(stats, sm_count, st, sv, q, n_ptr, fetch, totals, ri, ne, perm); break;
  case 150: launch_trace<150>(stats, sm_count, st, sv, q, n_ptr, fetch, totals, ri, ne, perm); break;
  case 182: launch_trace<182>(stats, sm_count, st, sv, q, n_ptr, fetch, totals, ri, ne, perm); break;
  case 214: launch_trace<214>(stats, sm_count, st, sv, q, n_ptr, fetch, totals, ri, ne, perm); break;
  case 10: launch_trace<10>(stats, sm_count, st, sv, q, n_ptr, fetch, totals, ri, ne, perm); break;
  case 6: launch_trace<6>(stats, sm_count, st, sv, q, n_ptr, fetch, totals, ri, ne, perm); break;
  default: launch_trace<0>(stats, sm_count, st, sv, q, n_ptr, fetch, totals, ri, ne, perm); break;
  }
}

/* blocks of the grid-stride shade kernel */
static int wf_shade_blocks(int sm_count)
{
  if (const char *e = getenv("RTB_WF_SHADE_BLOCKS")) /* development knob: blocks per SM */
    return sm_count * std::max(1, atoi(e));
  return sm_count * 16;
}

/* Two groups of planes, each with its own queues and its own stream: the persistent kernels of one group
 * drain (their last warps finishing the longest rays) while the other group's next kernel fills the SMs that
 * become free.  A path slot belongs to one group, so the order of additions per slot -- and the result, bit
 * for bit -- is that of the one-stream schedule.  Not with per-kernel timing, the split estimator, ray sorting
 * or the ray-pool kernel (one set of their buffers). */
static int wf_group_count(const RenderArgs &A, bool timed, bool split, bool sorted, bool pool)
{
  const bool may = !timed && !split && !sorted && !pool;
  int n_groups = may ? 2 : 1;
  if (const char *e = getenv("RTB_WF_STREAMS"))
    n_groups = may ? atoi(e) : 1;
  return std::max(1, std::min(std::min(n_groups, WF_MAX_GROUPS), A.splits));
}

/* one group of planes: planes [A.plane_base, A.plane_base + planes), its slices of the two queues, its queue
 * lengths and trace fetch cursors (the stream is the caller's) */
struct WfGroup
{
  cudaStream_t stream;
  RenderArgs A;
  WfQueue q[2];
  unsigned *counts, *fetch;
  int planes, gen_blocks;
  bool has_last;
};

/* the groups of wf_render: queues q[] hold `cap` entries; group g's counters start at ctr_base + g * ctr_one */
static void wf_groups(const RenderArgs &A, int n_groups, const WfQueue q[2], size_t cap, char *ctr_base, size_t ctr_one,
                      int n_bounces, WfGroup *G)
{
  const size_t n_px = (size_t)A.width * A.height;
  for (int g = 0; g < n_groups; g++)
  {
    WfGroup &R = G[g];
    R.stream = nullptr;
    R.A = A;
    R.A.plane_base = (int)((long long)A.splits * g / n_groups);
    R.planes = (int)((long long)A.splits * (g + 1) / n_groups) - R.A.plane_base;
    R.has_last = g == n_groups - 1;
    const size_t first_slot = (size_t)R.A.plane_base * n_px;
    for (int k = 0; k < 2; k++)
    {
      R.q[k] = q[k];
      R.q[k].o_xy += first_slot; R.q[k].oz_dx += first_slot; R.q[k].d_yz += first_slot;
      R.q[k].path += first_slot; R.q[k].hit += first_slot;
      if (R.q[k].branch) R.q[k].branch += first_slot;
      R.q[k].cap = n_groups == 1 ? (unsigned)cap : (unsigned)((size_t)R.planes * n_px);
    }
    R.counts = reinterpret_cast<unsigned *>(ctr_base + (size_t)g * ctr_one);
    R.fetch = R.counts + (n_bounces + 2);
    R.gen_blocks = (int)(((long long)A.n_tiles * R.planes * 32 + 255) / 256);
  }
}

/* planes of group R whose sub-range still has a sample number `wave`: all, or all but the (shorter) last */
static int wf_valid_planes(const WfGroup &R, const RenderArgs &A, int wave)
{
  const int last_len = (A.s_end - A.s_begin) - (A.splits - 1) * A.chunk;
  return (R.has_last && wave >= last_len) ? R.planes - 1 : R.planes;
}

int wf_render(rtb_scene *scene, RenderArgs &A, const rtb_render_desc *desc, float *d_accum, cudaStream_t stream,
              bool stats, unsigned long long &launches, float *phase_ms)
{
  const size_t n_px = (size_t)A.width * A.height;
  const size_t slots = n_px * (size_t)A.splits;
  if (slots >= (1ull << 31))
  {
    rtb_set_error("wavefront: width*height*planes must stay below 2^31");
    return RTB_EINVAL;
  }
  const int n_bounces = A.max_depth + 1;
  /* SPLIT dielectric estimator: a path becomes a tree of up to 2^(depth+1) rays; the queues hold `split_factor`
   * entries per path slot (exact worst case up to max_depth 5, the reference's MAX_DEPTH; beyond that the
   * overflow flag reports a scene that needs more) */
  const bool split = A.dielectric_mode == RTB_DIELECTRIC_SPLIT;
  const size_t split_factor = split ? ((size_t)1 << std::min(A.max_depth + 1, 6)) : 1;
  const size_t cap = slots * split_factor;
  if (cap >= (1ull << 31))
  {
    rtb_set_error("wavefront: width*height*planes*split factor must stay below 2^31");
    return RTB_EINVAL;
  }

  /* tuning word (desc->reserved): the trace kernel, wf_trace_tune; desc->reserved2: ray sorting mode (0 = off) */
  WfTraceTune tune;
  const int tune_rc = wf_trace_tune(A.sv, desc->reserved, tune);
  if (tune_rc != RTB_OK)
    return tune_rc;
  const int sort_mode = split ? 0 : (desc->reserved2 & 0xFF);
  const int sort_from = 1;                                           /* primary rays are coherent already */
  const int sort_until = (desc->reserved2 >> 8) & 0xFF ? (desc->reserved2 >> 8) & 0xFF : 255;

  /* one allocation: 2 queues x 5 arrays of 16 B, the planes, sort buffers, the per-wave counters */
  const size_t arr = align_up(cap * 16, 256);
  const size_t arr_planes = align_up(slots * 16, 256);
  const size_t arr4 = align_up(cap * 4, 256);
  const size_t ctr_one = align_up(sizeof(unsigned) * (2 * (size_t)(n_bounces + 2) + 1), 256);
  const size_t ctr_bytes = WF_MAX_GROUPS * ctr_one; /* per plane group (stream) */
  size_t sort_tmp_bytes = 0;
  if (sort_mode)
  {
    unsigned *nul = nullptr;
    cub::DeviceRadixSort::SortPairs(nullptr, sort_tmp_bytes, nul, nul, nul, nul, (int)slots, 0, 24, stream);
    sort_tmp_bytes = align_up(sort_tmp_bytes, 256);
  }
  int sm_count = 148;
  cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, scene->device);
  const bool pool = tune.pool;
  const size_t pool_bytes = wf_pool_stack_bytes(tune, sm_count);
  const size_t need = arr * 10 + arr_planes + ctr_bytes + (sort_mode ? arr4 * 4 + sort_tmp_bytes : 0) + (split ? arr4 * 2 : 0) + pool_bytes;
  if (scene->wf_bytes < need)
  {
    if (scene->d_wf)
    {
      RTB_CUDA(cudaStreamSynchronize(stream)); /* an earlier call on this scene may still use it */
      RTB_CUDA(cudaFree(scene->d_wf));
    }
    scene->d_wf = nullptr;
    scene->wf_bytes = 0;
    size_t got = 0;
    if (void *parked = rtb_cache_take(scene->device, need, &got))
    {
      scene->d_wf = parked;
      scene->wf_bytes = got;
    }
    else
    {
      if (cudaMalloc(&scene->d_wf, need) != cudaSuccess)
      {
        cudaGetLastError(); /* not sticky: the caller retries with fewer planes */
        scene->d_wf = nullptr;
        rtb_set_error("wavefront: not enough device memory for the ray queues");
        return RTB_ENOMEM;
      }
      scene->wf_bytes = need;
    }
  }
  char *p = static_cast<char *>(scene->d_wf);
  WfQueue q[2];
  for (int k = 0; k < 2; k++)
  {
    q[k].o_xy = reinterpret_cast<double2 *>(p); p += arr;
    q[k].oz_dx = reinterpret_cast<double2 *>(p); p += arr;
    q[k].d_yz = reinterpret_cast<double2 *>(p); p += arr;
    q[k].path = reinterpret_cast<uint4 *>(p); p += arr;
    q[k].hit = reinterpret_cast<uint4 *>(p); p += arr;
    q[k].branch = nullptr;
    q[k].cap = (unsigned)cap;
  }
  float4 *planes = reinterpret_cast<float4 *>(p); p += arr_planes;
  unsigned *counts = reinterpret_cast<unsigned *>(p);            /* [n_bounces + 2] queue lengths */
  unsigned *fetch = counts + (n_bounces + 2);                    /* [n_bounces + 2] trace fetch cursors */
  unsigned *overflow = fetch + (n_bounces + 2);                  /* SPLIT: a queue ran out of entries */
  char *const ctr_base = p; /* group g: its counts and fetch cursors at ctr_base + g * ctr_one */
  p += ctr_bytes;
  if (split)
  {
    q[0].branch = reinterpret_cast<unsigned *>(p); p += arr4;
    q[1].branch = reinterpret_cast<unsigned *>(p); p += arr4;
    RTB_CUDA(cudaMemsetAsync(overflow, 0, sizeof(unsigned), stream));
  }
  int2 *pool_stacks = nullptr;
  if (pool)
  {
    pool_stacks = reinterpret_cast<int2 *>(p);
    p += pool_bytes;
  }
  unsigned *keys = nullptr, *keys_sorted = nullptr, *iota = nullptr, *perm = nullptr;
  void *sort_tmp = nullptr;
  if (sort_mode)
  {
    keys = reinterpret_cast<unsigned *>(p); p += arr4;
    keys_sorted = reinterpret_cast<unsigned *>(p); p += arr4;
    iota = reinterpret_cast<unsigned *>(p); p += arr4;
    perm = reinterpret_cast<unsigned *>(p); p += arr4;
    sort_tmp = p;
    k_wf_iota<<<(unsigned)((slots + 255) / 256), 256, 0, stream>>>(iota, (unsigned)slots);
    launches++;
  }

  RTB_CUDA(cudaMemsetAsync(planes, 0, slots * 16, stream));

  const int shade_blocks = wf_shade_blocks(sm_count);

  /* per-kernel timing (only with counters): events around every trace launch */
  struct EventList : std::vector<cudaEvent_t> /* destroyed on every return path */
  {
    ~EventList()
    {
      for (cudaEvent_t e : *this)
        cudaEventDestroy(e);
    }
  } ev;
  auto mark = [&]() {
    if (!phase_ms)
      return;
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, stream);
    ev.push_back(e);
  };
  const int n_groups = wf_group_count(A, phase_ms != nullptr, split, sort_mode != 0, pool);
  for (int g = 1; g < n_groups; g++)
    if (!scene->wf_streams[g])
    {
      /* the streams are made once per device and kept (render() makes a new scene per call); the events are the scene's */
      static std::mutex stream_mutex;
      static cudaStream_t device_streams[64][WF_MAX_GROUPS] = {};
      const int dev = scene->device & 63;
      {
        std::lock_guard<std::mutex> lock(stream_mutex);
        if (!device_streams[dev][g])
          RTB_CUDA(cudaStreamCreateWithFlags(&device_streams[dev][g], cudaStreamNonBlocking));
        scene->wf_streams[g] = device_streams[dev][g];
      }
      RTB_CUDA(cudaEventCreateWithFlags(&scene->wf_joins[g], cudaEventDisableTiming));
      if (!scene->wf_fork)
        RTB_CUDA(cudaEventCreateWithFlags(&scene->wf_fork, cudaEventDisableTiming));
    }
  WfGroup G[WF_MAX_GROUPS];
  wf_groups(A, n_groups, q, cap, ctr_base, ctr_one, n_bounces, G);
  for (int g = 0; g < n_groups; g++)
    G[g].stream = g == 0 ? stream : scene->wf_streams[g];
  if (n_groups > 1)
  {
    RTB_CUDA(cudaEventRecord(scene->wf_fork, stream)); /* the planes are zeroed, the scene is built */
    for (int g = 1; g < n_groups; g++)
      RTB_CUDA(cudaStreamWaitEvent(scene->wf_streams[g], scene->wf_fork, 0));
  }
  for (int wave = 0; wave < A.chunk; wave++)
  {
    for (int g = 0; g < n_groups; g++)
    {
      WfGroup &R = G[g];
      RTB_CUDA(cudaMemsetAsync(R.counts, 0, sizeof(unsigned) * 2 * (size_t)(n_bounces + 2), R.stream));
      k_wf_generate<<<R.gen_blocks, 256, 0, R.stream>>>(R.A, wave, wf_valid_planes(R, A, wave), R.q[0], &R.counts[0]);
      launches++;
    }
    for (int b = 0; b < n_bounces; b++)
      for (int g = 0; g < n_groups; g++)
      {
        WfGroup &R = G[g];
        cudaStream_t st = R.stream;
        unsigned *cnt = R.counts, *fch = R.fetch;
        const WfQueue &qi = R.q[b & 1], &qo = R.q[(b + 1) & 1];
        const bool sorted_in = sort_mode && b >= sort_from && b <= sort_until;        /* queue b was sorted */
        const bool sort_out = sort_mode && b + 1 >= sort_from && b + 1 <= sort_until && b + 1 < n_bounces;
        const unsigned *use_perm = sorted_in ? perm : nullptr;
        mark();
        wf_launch_trace(tune, stats, sm_count, st, A.sv, qi, &cnt[b], &fch[b], A.counters, pool_stacks, use_perm);
        mark();
        if (sort_out) /* slots beyond the queue's end keep the largest key and sort to the back */
          RTB_CUDA(cudaMemsetAsync(keys, 0xFF, slots * 4, st));
        if (split)
          k_wf_shade<true><<<shade_blocks, 128, 0, st>>>(R.A, wave, b, qi, &cnt[b], qo, &cnt[b + 1], planes, nullptr, 0, overflow);
        else
          k_wf_shade<false><<<shade_blocks, 128, 0, st>>>(R.A, wave, b, qi, &cnt[b], qo, &cnt[b + 1], planes,
                                                          sort_out ? keys : nullptr, sort_mode, nullptr);
        launches += 2;
        if (sort_out)
        {
          size_t tmp = sort_tmp_bytes;
          cub::DeviceRadixSort::SortPairs(sort_tmp, tmp, keys, keys_sorted, iota, perm, (int)slots, 0, 24, st);
          launches += 4;
        }
      }
    RTB_CUDA(cudaGetLastError());
  }
  for (int g = 1; g < n_groups; g++)
  {
    RTB_CUDA(cudaEventRecord(scene->wf_joins[g], scene->wf_streams[g]));
    RTB_CUDA(cudaStreamWaitEvent(stream, scene->wf_joins[g], 0));
  }
  k_wf_sum_planes<<<(unsigned)((n_px + 255) / 256), 256, 0, stream>>>(planes, A.splits, (unsigned)n_px, d_accum);
  RTB_CUDA(cudaGetLastError());
  launches++;
  if (split)
  {
    unsigned h_overflow = 0;
    RTB_CUDA(cudaMemcpyAsync(&h_overflow, overflow, sizeof(unsigned), cudaMemcpyDeviceToHost, stream));
    RTB_CUDA(cudaStreamSynchronize(stream));
    if (h_overflow)
    {
      rtb_set_error("RTB_DIELECTRIC_SPLIT: the split tree of some path outgrew the ray queue (max_depth > 5 with many "
                    "dielectric surfaces); use RTB_DIELECTRIC_STOCHASTIC, the same estimator in expectation");
      return RTB_EINVAL;
    }
  }
  if (phase_ms)
  {
    /* ev = [t0 trace t1] shade/generate [t2 trace t3] ...: odd gaps are trace launches */
    mark();
    RTB_CUDA(cudaEventSynchronize(ev.back()));
    float trace = 0.0f, total = 0.0f;
    for (size_t k = 0; k + 1 < ev.size(); k += 2)
    {
      float ms = 0.0f;
      cudaEventElapsedTime(&ms, ev[k], ev[k + 1]);
      trace += ms;
    }
    cudaEventElapsedTime(&total, ev.front(), ev.back());
    phase_ms[0] = trace;
    phase_ms[1] = total - trace; /* generate of later waves + shade + sum (the first generate is before ev[0]) */
    phase_ms[2] = (float)(ev.size() / 2);
  }
  return RTB_OK;
}

/* ---- parity probe: the product trace kernel on caller rays -------------------------------------- */

/* queue entry i = ray i with its hit record seeded from the oversized list, exactly as k_wf_generate / k_wf_shade
 * write it, and path slot pid[i] (else i), throughput tp3[3i..] (else 0) and branch[i] (else 1); the big-list exact
 * tests go to totals[2] */
__global__ void k_wf_fill(const __grid_constant__ SceneView sv, const double *__restrict__ rays,
                          const unsigned *__restrict__ pid, const float *__restrict__ tp3, const unsigned *__restrict__ branch,
                          unsigned n, WfQueue q, unsigned long long *totals)
{
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  unsigned exact = 0;
  if (i < n)
  {
    const d3 o = d3_make(rays[6 * (size_t)i + 0], rays[6 * (size_t)i + 1], rays[6 * (size_t)i + 2]);
    const d3 d = d3_make(rays[6 * (size_t)i + 3], rays[6 * (size_t)i + 4], rays[6 * (size_t)i + 5]);
    HitRec seed;
    ray_seed_hit(sv, o, d, seed, exact);
    q.o_xy[i] = make_double2(o.x, o.y);
    q.oz_dx[i] = make_double2(o.z, d.x);
    q.d_yz[i] = make_double2(d.y, d.z);
    const float r = tp3 ? tp3[3 * (size_t)i + 0] : 0.0f, g = tp3 ? tp3[3 * (size_t)i + 1] : 0.0f,
                b = tp3 ? tp3[3 * (size_t)i + 2] : 0.0f;
    q.path[i] = make_uint4(pid ? pid[i] : i, __float_as_uint(r), __float_as_uint(g), __float_as_uint(b));
    q.hit[i] = pack_hit(seed);
    if (q.branch)
      q.branch[i] = branch ? branch[i] : 1u;
  }
  wf_add_counters(totals, lane, 0ull, 0ull, exact, 0ull, 0ull);
}

/* hit record of queue entry i -> the probe's output arrays (the same read-out as rtb_trace_rays) */
__global__ void k_wf_read_hits(const __grid_constant__ SceneView sv, WfQueue q, unsigned n, int *__restrict__ ids,
                               long long *__restrict__ prims, double *__restrict__ ts, double *__restrict__ points,
                               double *__restrict__ normals, double *__restrict__ uvs)
{
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n)
    return;
  const double2 a = q.o_xy[i], b = q.oz_dx[i], c = q.d_yz[i];
  const d3 o = d3_make(a.x, a.y, b.x), d = d3_make(b.y, c.x, c.y);
  store_hit_record(sv, o, d, unpack_hit(q.hit[i]), i, ids, prims, ts, points, normals, uvs);
}

extern "C" int rtb_trace_rays_wf(rtb_scene *scene, const double *rays6, size_t n_rays, int tune,
                                 const uint32_t *perm_or_null, int32_t *ids, int64_t *prims, double *ts, double *points,
                                 double *normals, double *uvs, rtb_counters *counters_or_null)
{
  if (!scene || (n_rays && (!rays6 || !ids)))
  {
    rtb_set_error("rtb_trace_rays_wf: NULL argument");
    return RTB_EINVAL;
  }
  if (n_rays >= (1ull << 31))
  {
    rtb_set_error("rtb_trace_rays_wf: n_rays must stay below 2^31");
    return RTB_EINVAL;
  }
  if (perm_or_null)
  {
    /* the kernel reads queue entry perm[k]: anything but a permutation would read outside the queue */
    std::vector<char> seen(n_rays, 0);
    for (size_t k = 0; k < n_rays; k++)
    {
      if (perm_or_null[k] >= n_rays || seen[perm_or_null[k]])
      {
        rtb_set_error("rtb_trace_rays_wf: perm is not a permutation of [0, n_rays)");
        return RTB_EINVAL;
      }
      seen[perm_or_null[k]] = 1;
    }
  }
  const SceneView &sv = scene->view;
  WfTraceTune t;
  const int tune_rc = wf_trace_tune(sv, tune, t);
  if (tune_rc != RTB_OK)
    return tune_rc;
  RTB_CUDA(cudaSetDevice(scene->device));
  int sm_count = 148;
  cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, scene->device);
  const unsigned n = (unsigned)n_rays;
  const size_t m = n_rays > 0 ? n_rays : 1; /* no zero-byte allocations */

  Dev<double> d_rays, d_ts, d_points, d_normals, d_uvs;
  Dev<double2> d_oxy, d_ozdx, d_dyz;
  Dev<uint4> d_path, d_hit;
  Dev<unsigned> d_ctl, d_perm; /* d_ctl: queue length, fetch cursor */
  Dev<unsigned long long> d_totals;
  Dev<int2> d_stacks;
  Dev<int> d_ids;
  Dev<long long> d_prims;
  RTB_CUDA(cudaMalloc(&d_rays.p, sizeof(double) * 6 * m));
  RTB_CUDA(cudaMalloc(&d_oxy.p, sizeof(double2) * m));
  RTB_CUDA(cudaMalloc(&d_ozdx.p, sizeof(double2) * m));
  RTB_CUDA(cudaMalloc(&d_dyz.p, sizeof(double2) * m));
  RTB_CUDA(cudaMalloc(&d_path.p, sizeof(uint4) * m));
  RTB_CUDA(cudaMalloc(&d_hit.p, sizeof(uint4) * m));
  RTB_CUDA(cudaMalloc(&d_ctl.p, sizeof(unsigned) * 2));
  RTB_CUDA(cudaMalloc(&d_totals.p, sizeof(unsigned long long) * 5));
  if (perm_or_null)
    RTB_CUDA(cudaMalloc(&d_perm.p, sizeof(unsigned) * m));
  if (t.pool)
    RTB_CUDA(cudaMalloc(&d_stacks.p, wf_pool_stack_bytes(t, sm_count)));
  RTB_CUDA(cudaMalloc(&d_ids.p, sizeof(int) * m));
  RTB_CUDA(cudaMalloc(&d_prims.p, sizeof(long long) * m));
  RTB_CUDA(cudaMalloc(&d_ts.p, sizeof(double) * m));
  RTB_CUDA(cudaMalloc(&d_points.p, sizeof(double) * 3 * m));
  RTB_CUDA(cudaMalloc(&d_normals.p, sizeof(double) * 3 * m));
  RTB_CUDA(cudaMalloc(&d_uvs.p, sizeof(double) * 2 * m));
  if (n_rays)
    RTB_CUDA(cudaMemcpy(d_rays.p, rays6, sizeof(double) * 6 * n_rays, cudaMemcpyHostToDevice));
  if (perm_or_null && n_rays)
    RTB_CUDA(cudaMemcpy(d_perm.p, perm_or_null, sizeof(unsigned) * n_rays, cudaMemcpyHostToDevice));
  const unsigned ctl[2] = { n, 0u };
  RTB_CUDA(cudaMemcpy(d_ctl.p, ctl, sizeof(ctl), cudaMemcpyHostToDevice));
  RTB_CUDA(cudaMemset(d_totals.p, 0, sizeof(unsigned long long) * 5));

  WfQueue q;
  q.o_xy = d_oxy.p;
  q.oz_dx = d_ozdx.p;
  q.d_yz = d_dyz.p;
  q.path = d_path.p;
  q.hit = d_hit.p;
  q.branch = nullptr;
  q.cap = n;
  const unsigned blocks = (unsigned)((m + 127) / 128);
  k_wf_fill<<<blocks, 128>>>(sv, d_rays.p, nullptr, nullptr, nullptr, n, q, d_totals.p);
  RTB_CUDA(cudaGetLastError());
  wf_launch_trace(t, true, sm_count, 0, sv, q, d_ctl.p, d_ctl.p + 1, d_totals.p, d_stacks.p, d_perm.p);
  RTB_CUDA(cudaGetLastError());
  k_wf_read_hits<<<blocks, 128>>>(sv, q, n, d_ids.p, d_prims.p, d_ts.p, d_points.p, d_normals.p, d_uvs.p);
  RTB_CUDA(cudaGetLastError());
  RTB_CUDA(cudaDeviceSynchronize());
  if (n_rays)
  {
    RTB_CUDA(cudaMemcpy(ids, d_ids.p, sizeof(int) * n_rays, cudaMemcpyDeviceToHost));
    if (prims) RTB_CUDA(cudaMemcpy(prims, d_prims.p, sizeof(long long) * n_rays, cudaMemcpyDeviceToHost));
    if (ts) RTB_CUDA(cudaMemcpy(ts, d_ts.p, sizeof(double) * n_rays, cudaMemcpyDeviceToHost));
    if (points) RTB_CUDA(cudaMemcpy(points, d_points.p, sizeof(double) * 3 * n_rays, cudaMemcpyDeviceToHost));
    if (normals) RTB_CUDA(cudaMemcpy(normals, d_normals.p, sizeof(double) * 3 * n_rays, cudaMemcpyDeviceToHost));
    if (uvs) RTB_CUDA(cudaMemcpy(uvs, d_uvs.p, sizeof(double) * 2 * n_rays, cudaMemcpyDeviceToHost));
  }
  if (counters_or_null)
  {
    unsigned long long h[5];
    RTB_CUDA(cudaMemcpy(h, d_totals.p, sizeof(h), cudaMemcpyDeviceToHost));
    memset(counters_or_null, 0, sizeof(*counters_or_null));
    counters_or_null->rays = n_rays;
    counters_or_null->prim_tests = h[2];
    counters_or_null->node_visits = h[3];
    counters_or_null->launches = 3;
    counters_or_null->trace_launches = 1;
  }
  return RTB_OK;
}

/* ---- parity probes: the product generate and shade kernels, one launch at a time ------------------------------
 * They run what wf_render runs -- the same RenderArgs (fill_args, rtb_plane_split), plane groups (wf_groups), trace
 * dispatch (wf_trace_tune, wf_launch_trace) and shade grid -- on queues they own, so that a test can compare every
 * ray of every bounce with the oracle.  The plane count must be fixed (desc->planes > 0): it decides which sample
 * a path slot carries.  Queue ORDER is the kernels' (atomics); the caller sorts. */

/* the device arrays of one probe queue of `cap` entries; branch ids only for the split estimator */
struct WfProbeQueue
{
  Dev<double2> oxy, ozdx, dyz;
  Dev<uint4> path, hit;
  Dev<unsigned> branch;
  WfQueue q;
  int alloc(size_t cap, bool split)
  {
    const size_t m = cap > 0 ? cap : 1;
    RTB_CUDA(cudaMalloc(&oxy.p, sizeof(double2) * m));
    RTB_CUDA(cudaMalloc(&ozdx.p, sizeof(double2) * m));
    RTB_CUDA(cudaMalloc(&dyz.p, sizeof(double2) * m));
    RTB_CUDA(cudaMalloc(&path.p, sizeof(uint4) * m));
    RTB_CUDA(cudaMalloc(&hit.p, sizeof(uint4) * m));
    if (split)
      RTB_CUDA(cudaMalloc(&branch.p, sizeof(unsigned) * m));
    q.o_xy = oxy.p; q.oz_dx = ozdx.p; q.d_yz = dyz.p; q.path = path.p; q.hit = hit.p; q.branch = branch.p;
    q.cap = (unsigned)cap;
    return RTB_OK;
  }
};

/* entries [first, first + n) of q -> host rays (origin, direction), path slot, throughput, branch (1 without ids) */
static int wf_probe_read(const WfQueue &q, size_t first, size_t n, double *rays6, uint32_t *pid, float *tp3, uint32_t *branch)
{
  if (n == 0)
    return RTB_OK;
  std::vector<double2> a(n), b(n), c(n);
  std::vector<uint4> p(n);
  std::vector<unsigned> br(n, 1u);
  RTB_CUDA(cudaMemcpy(a.data(), q.o_xy + first, sizeof(double2) * n, cudaMemcpyDeviceToHost));
  RTB_CUDA(cudaMemcpy(b.data(), q.oz_dx + first, sizeof(double2) * n, cudaMemcpyDeviceToHost));
  RTB_CUDA(cudaMemcpy(c.data(), q.d_yz + first, sizeof(double2) * n, cudaMemcpyDeviceToHost));
  RTB_CUDA(cudaMemcpy(p.data(), q.path + first, sizeof(uint4) * n, cudaMemcpyDeviceToHost));
  if (q.branch)
    RTB_CUDA(cudaMemcpy(br.data(), q.branch + first, sizeof(unsigned) * n, cudaMemcpyDeviceToHost));
  for (size_t i = 0; i < n; i++)
  {
    const double r[6] = { a[i].x, a[i].y, b[i].x, b[i].y, c[i].x, c[i].y };
    memcpy(rays6 + 6 * i, r, sizeof(r));
    pid[i] = p[i].x;
    memcpy(tp3 + 3 * i, &p[i].y, 3 * sizeof(float));
    branch[i] = br[i];
  }
  return RTB_OK;
}

/* the RenderArgs and trace kernel of a probe call, with wf_render's chunk and splits */
static int wf_probe_args(const char *who, rtb_scene *scene, const double *camera12, const rtb_render_desc *desc, int wave,
                         RenderArgs &A, WfTraceTune &tune, int &sm_count)
{
  const std::string name(who);
  if (!scene || !camera12 || !desc)
  {
    rtb_set_error(name + ": NULL argument");
    return RTB_EINVAL;
  }
  int rc = rtb_check_desc(desc);
  if (rc != RTB_OK)
    return rc;
  if (desc->integrator != RTB_INTEGRATOR_PATH || (desc->kernel != 0 && desc->kernel != 6))
  {
    rtb_set_error(name + ": the wavefront path tracer only (integrator RTB_INTEGRATOR_PATH, kernel 0 or 6)");
    return RTB_EINVAL;
  }
  const int spp = desc->sample_end - desc->sample_begin;
  if (desc->planes <= 0 || spp <= 0)
  {
    rtb_set_error(name + ": need desc->planes > 0 (it fixes the sample of every path slot) and at least one sample");
    return RTB_EINVAL;
  }
  fill_args(A, scene, camera12, desc);
  const size_t n_px = (size_t)A.width * A.height;
  int chunk = 0;
  A.splits = rtb_plane_split((long long)n_px, n_px, desc->planes, spp, &chunk);
  A.chunk = chunk;
  if (n_px * (size_t)A.splits >= (1ull << 31))
  {
    rtb_set_error(name + ": width*height*planes must stay below 2^31");
    return RTB_EINVAL;
  }
  if (wave < 0 || wave >= A.chunk)
  {
    rtb_set_error(name + ": wave must lie in [0, samples per plane)");
    return RTB_EINVAL;
  }
  rc = wf_trace_tune(A.sv, desc->reserved, tune);
  if (rc != RTB_OK)
    return rc;
  RTB_CUDA(cudaSetDevice(scene->device));
  sm_count = 148;
  cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, scene->device);
  return RTB_OK;
}

extern "C" int rtb_wf_generate(rtb_scene *scene, const double *camera12, const rtb_render_desc *desc, int wave,
                               size_t cap, double *rays6, uint32_t *pid, float *throughput3, uint32_t *branch,
                               size_t *n_out)
{
  RenderArgs A;
  WfTraceTune tune;
  int sm_count = 0;
  int rc = wf_probe_args("rtb_wf_generate", scene, camera12, desc, wave, A, tune, sm_count);
  if (rc != RTB_OK)
    return rc;
  const size_t n_px = (size_t)A.width * A.height, slots = n_px * (size_t)A.splits;
  if (!rays6 || !pid || !throughput3 || !branch || !n_out || cap < slots)
  {
    rtb_set_error("rtb_wf_generate: NULL output, or cap below planes*width*height");
    return RTB_EINVAL;
  }
  const bool split = A.dielectric_mode == RTB_DIELECTRIC_SPLIT;
  const int sort_mode = split ? 0 : (desc->reserved2 & 0xFF);
  const int n_groups = wf_group_count(A, false, split, sort_mode != 0, tune.pool);
  const int n_bounces = A.max_depth + 1;
  const size_t ctr_one = align_up(sizeof(unsigned) * (2 * (size_t)(n_bounces + 2) + 1), 256);
  WfProbeQueue pq;
  rc = pq.alloc(slots, split);
  if (rc != RTB_OK)
    return rc;
  Dev<char> d_ctr;
  Dev<unsigned long long> d_totals;
  RTB_CUDA(cudaMalloc(&d_ctr.p, ctr_one * WF_MAX_GROUPS));
  RTB_CUDA(cudaMalloc(&d_totals.p, sizeof(unsigned long long) * 8));
  RTB_CUDA(cudaMemset(d_ctr.p, 0, ctr_one * WF_MAX_GROUPS));
  RTB_CUDA(cudaMemset(d_totals.p, 0, sizeof(unsigned long long) * 8));
  A.counters = d_totals.p;
  const WfQueue q[2] = { pq.q, pq.q };
  WfGroup G[WF_MAX_GROUPS];
  wf_groups(A, n_groups, q, slots, d_ctr.p, ctr_one, n_bounces, G);
  for (int g = 0; g < n_groups; g++)
    k_wf_generate<<<G[g].gen_blocks, 256>>>(G[g].A, wave, wf_valid_planes(G[g], A, wave), G[g].q[0], &G[g].counts[0]);
  RTB_CUDA(cudaGetLastError());
  RTB_CUDA(cudaDeviceSynchronize());
  size_t n = 0;
  for (int g = 0; g < n_groups; g++)
  {
    unsigned len = 0;
    RTB_CUDA(cudaMemcpy(&len, G[g].counts, sizeof(unsigned), cudaMemcpyDeviceToHost));
    rc = wf_probe_read(pq.q, (size_t)G[g].A.plane_base * n_px, len, rays6 + 6 * n, pid + n, throughput3 + 3 * n, branch + n);
    if (rc != RTB_OK)
      return rc;
    n += len;
  }
  *n_out = n;
  return RTB_OK;
}

extern "C" int rtb_wf_bounce(rtb_scene *scene, const double *camera12, const rtb_render_desc *desc, int wave, int depth,
                             size_t n_rays, const double *rays6, const uint32_t *pid, const float *throughput3,
                             const uint32_t *branch_or_null, float *planes4, size_t planes_len, int32_t *ids_or_null,
                             int64_t *prims_or_null, double *ts_or_null, size_t cap_out, double *rays6_out,
                             uint32_t *pid_out, float *throughput3_out, uint32_t *branch_out, size_t *n_out,
                             rtb_counters *counters_or_null)
{
  RenderArgs A;
  WfTraceTune tune;
  int sm_count = 0;
  int rc = wf_probe_args("rtb_wf_bounce", scene, camera12, desc, wave, A, tune, sm_count);
  if (rc != RTB_OK)
    return rc;
  const size_t n_px = (size_t)A.width * A.height, slots = n_px * (size_t)A.splits;
  const bool split = A.dielectric_mode == RTB_DIELECTRIC_SPLIT;
  auto bad = [](const char *why) {
    rtb_set_error(std::string("rtb_wf_bounce: ") + why);
    return RTB_EINVAL;
  };
  if (n_rays >= (1ull << 31))
    return bad("n_rays must stay below 2^31");
  if ((n_rays && (!rays6 || !pid || !throughput3)) || !planes4 || !rays6_out || !pid_out || !throughput3_out ||
      !branch_out || !n_out)
    return bad("NULL argument");
  if (depth < 0 || depth > A.max_depth)
    return bad("depth must lie in [0, max_depth]");
  if (planes_len != 4 * slots)
    return bad("planes must hold 4 floats per path slot (planes * width * height slots)");
  if (cap_out < 2 * n_rays)
    return bad("the output queue must hold two children per ray");
  if (split && n_rays && !branch_or_null)
    return bad("the split estimator needs the branch id of every ray");
  for (size_t i = 0; i < n_rays; i++)
  {
    if (pid[i] >= slots)
      return bad("path slot id beyond planes * width * height");
    if (branch_or_null && (branch_or_null[i] == 0u || (!split && branch_or_null[i] != 1u)))
      return bad("branch ids start at 1, and the stochastic estimator carries no other");
  }
  const unsigned n = (unsigned)n_rays;
  const size_t m = n_rays > 0 ? n_rays : 1;
  WfProbeQueue qin, qout;
  if ((rc = qin.alloc(n_rays, split)) != RTB_OK || (rc = qout.alloc(2 * n_rays, split)) != RTB_OK)
    return rc;
  Dev<double> d_rays, d_ts;
  Dev<unsigned> d_pid, d_branch, d_ctl; /* d_ctl: queue length in, trace fetch cursor, queue length out, overflow */
  Dev<float> d_tp;
  Dev<float4> d_planes;
  Dev<unsigned long long> d_totals, d_trace_totals;
  Dev<int2> d_stacks;
  Dev<int> d_ids;
  Dev<long long> d_prims;
  RTB_CUDA(cudaMalloc(&d_rays.p, sizeof(double) * 6 * m));
  RTB_CUDA(cudaMalloc(&d_pid.p, sizeof(unsigned) * m));
  RTB_CUDA(cudaMalloc(&d_tp.p, sizeof(float) * 3 * m));
  RTB_CUDA(cudaMalloc(&d_ctl.p, sizeof(unsigned) * 4));
  RTB_CUDA(cudaMalloc(&d_planes.p, sizeof(float4) * slots));
  RTB_CUDA(cudaMalloc(&d_totals.p, sizeof(unsigned long long) * 8));
  RTB_CUDA(cudaMalloc(&d_trace_totals.p, sizeof(unsigned long long) * 5));
  RTB_CUDA(cudaMalloc(&d_ids.p, sizeof(int) * m));
  RTB_CUDA(cudaMalloc(&d_prims.p, sizeof(long long) * m));
  RTB_CUDA(cudaMalloc(&d_ts.p, sizeof(double) * m));
  if (branch_or_null)
    RTB_CUDA(cudaMalloc(&d_branch.p, sizeof(unsigned) * m));
  if (tune.pool)
    RTB_CUDA(cudaMalloc(&d_stacks.p, wf_pool_stack_bytes(tune, sm_count)));
  if (n_rays)
  {
    RTB_CUDA(cudaMemcpy(d_rays.p, rays6, sizeof(double) * 6 * n_rays, cudaMemcpyHostToDevice));
    RTB_CUDA(cudaMemcpy(d_pid.p, pid, sizeof(unsigned) * n_rays, cudaMemcpyHostToDevice));
    RTB_CUDA(cudaMemcpy(d_tp.p, throughput3, sizeof(float) * 3 * n_rays, cudaMemcpyHostToDevice));
    if (branch_or_null)
      RTB_CUDA(cudaMemcpy(d_branch.p, branch_or_null, sizeof(unsigned) * n_rays, cudaMemcpyHostToDevice));
  }
  RTB_CUDA(cudaMemcpy(d_planes.p, planes4, sizeof(float4) * slots, cudaMemcpyHostToDevice));
  const unsigned ctl[4] = { n, 0u, 0u, 0u };
  RTB_CUDA(cudaMemcpy(d_ctl.p, ctl, sizeof(ctl), cudaMemcpyHostToDevice));
  RTB_CUDA(cudaMemset(d_totals.p, 0, sizeof(unsigned long long) * 8));
  RTB_CUDA(cudaMemset(d_trace_totals.p, 0, sizeof(unsigned long long) * 5));
  A.counters = d_totals.p;

  const unsigned blocks = (unsigned)((m + 127) / 128);
  k_wf_fill<<<blocks, 128>>>(A.sv, d_rays.p, d_pid.p, d_tp.p, d_branch.p, n, qin.q, d_trace_totals.p);
  wf_launch_trace(tune, false, sm_count, 0, A.sv, qin.q, d_ctl.p, d_ctl.p + 1, d_trace_totals.p, d_stacks.p, nullptr);
  if (split)
    k_wf_shade<true><<<wf_shade_blocks(sm_count), 128>>>(A, wave, depth, qin.q, d_ctl.p, qout.q, d_ctl.p + 2, d_planes.p,
                                                         nullptr, 0, d_ctl.p + 3);
  else
    k_wf_shade<false><<<wf_shade_blocks(sm_count), 128>>>(A, wave, depth, qin.q, d_ctl.p, qout.q, d_ctl.p + 2, d_planes.p,
                                                          nullptr, 0, nullptr);
  if (ids_or_null)
    k_wf_read_hits<<<blocks, 128>>>(A.sv, qin.q, n, d_ids.p, d_prims.p, d_ts.p, nullptr, nullptr, nullptr);
  RTB_CUDA(cudaGetLastError());
  RTB_CUDA(cudaDeviceSynchronize());

  unsigned got[4];
  RTB_CUDA(cudaMemcpy(got, d_ctl.p, sizeof(got), cudaMemcpyDeviceToHost));
  if (got[3] || got[2] > 2 * n)
  {
    rtb_set_error("rtb_wf_bounce: the output queue overflowed");
    return RTB_ECUDA;
  }
  rc = wf_probe_read(qout.q, 0, got[2], rays6_out, pid_out, throughput3_out, branch_out);
  if (rc != RTB_OK)
    return rc;
  *n_out = got[2];
  RTB_CUDA(cudaMemcpy(planes4, d_planes.p, sizeof(float4) * slots, cudaMemcpyDeviceToHost));
  if (ids_or_null && n_rays)
  {
    RTB_CUDA(cudaMemcpy(ids_or_null, d_ids.p, sizeof(int) * n_rays, cudaMemcpyDeviceToHost));
    if (prims_or_null) RTB_CUDA(cudaMemcpy(prims_or_null, d_prims.p, sizeof(long long) * n_rays, cudaMemcpyDeviceToHost));
    if (ts_or_null) RTB_CUDA(cudaMemcpy(ts_or_null, d_ts.p, sizeof(double) * n_rays, cudaMemcpyDeviceToHost));
  }
  if (counters_or_null)
  {
    unsigned long long h[8];
    RTB_CUDA(cudaMemcpy(h, d_totals.p, sizeof(h), cudaMemcpyDeviceToHost));
    memset(counters_or_null, 0, sizeof(*counters_or_null));
    counters_or_null->rays = h[0];
    counters_or_null->rays_intersected = h[1];
    counters_or_null->prim_tests = h[2];
    counters_or_null->launches = ids_or_null ? 4 : 3;
    counters_or_null->trace_launches = 1;
  }
  return RTB_OK;
}
