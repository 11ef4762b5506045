/*
 * rtb_render.cu -- the path-tracing kernels and the render / probe entry points.
 *
 * k_render is a "megakernel with path regeneration": one thread owns one pixel and a
 * contiguous range of that pixel's samples.  Every loop iteration is one trace_path
 * invocation of the reference (raytracer.c:482-554): nearest hit, Russian roulette,
 * scatter.  When a path ends the lane starts the pixel's next sample in the same
 * iteration slot, so lanes stay busy until their whole sample range is done; the warp
 * re-converges once per iteration at the __all_sync at the top of the loop.
 * Warps map to 8x4 pixel tiles so primary rays are coherent.
 *
 * Random numbers: Philox4x32-10, counter = (pixel, sample, bounce | 0x100, block),
 * key = seed (see rtb_device.cuh and oracle/oracle.c for the layout; both sides must
 * agree word for word).
 */
#include "rtb_path.cuh"

#include <atomic>

#include <algorithm>
#include <vector>
#include <cstring>


/* WALK: 0 = if-if loop, 1 = if-if + FP32 sphere pre-test, 2 = while-while + select-then-test */
template <bool STATS, int WALK>
__global__ void __launch_bounds__(128, WALK == 2 ? 8 : 4) k_render(const __grid_constant__ RenderArgs A)
{
  /* top of the traversal stack in shared memory (WALK == 2): keeps the hottest local-memory
   * traffic out of L1/L2 (profiles/r1_c3_default_ncu.md: 27 GB of local write-back per launch) */
  __shared__ int2 s_stack[WALK == 2 ? RTB_SMEM_STACK : 1][128];
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int tile = warp % A.n_tiles;
  const int split = warp / A.n_tiles;
  const int x = (tile % A.tiles_x) * 8 + (lane & 7);
  const int y = (tile / A.tiles_x) * 4 + (lane >> 3);
  const bool valid = x < A.width && y < A.height && split < A.splits;
  const unsigned pixel = (unsigned)(y * A.width + x);

  int s = A.s_begin + split * A.chunk;
  const int s_end = valid ? min(A.s_end, s + A.chunk) : s;

  PathState st;
  st.alive = false;
  st.depth = 0;
  st.tr = st.tg = st.tb = 0.0f;
  st.o = d3_make(0, 0, 0);
  st.d = d3_make(0, 0, 1);
  float sr = 0.0f, sg = 0.0f, sb = 0.0f;
  PathCounters pc = { 0u, 0u };
  TraceStats ts = { 0u, 0u };
  unsigned paths = 0;

  while (true)
  {
    if (!st.alive && s < s_end)
    {
      path_begin(A, st, x, y, pixel, (unsigned)s);
      paths++;
    }
    if (__all_sync(0xFFFFFFFFu, !st.alive))
      break;
    if (st.alive)
    {
      HitRec best;
      pc.rays++;
      pc.rays_hit++;
      if (WALK == 2)
        closest_hit_ww<STATS, RTB_SMEM_STACK>(A.sv, st.o, st.d, best, ts, &s_stack[0][threadIdx.x], 128);
      else
        closest_hit<STATS, WALK == 1>(A.sv, st.o, st.d, best, ts);
      path_shade(A, st, best, pixel, (unsigned)s, sr, sg, sb, pc, nullptr);
      if (!st.alive)
        s++;
    }
  }

  if (valid)
  {
    float *o = A.out + ((size_t)split * A.width * A.height + pixel) * 3;
    o[0] = sr; o[1] = sg; o[2] = sb;
  }

  /* counters: warp reduce, one atomic per warp and counter */
  unsigned long long c0 = pc.rays, c1 = pc.rays_hit, c2 = ts.prim_tests, c3 = ts.node_visits, c4 = paths;
  for (int off = 16; off > 0; off >>= 1)
  {
    c0 += __shfl_xor_sync(0xFFFFFFFFu, c0, off);
    c1 += __shfl_xor_sync(0xFFFFFFFFu, c1, off);
    c4 += __shfl_xor_sync(0xFFFFFFFFu, c4, off);
    if (STATS)
    {
      c2 += __shfl_xor_sync(0xFFFFFFFFu, c2, off);
      c3 += __shfl_xor_sync(0xFFFFFFFFu, c3, off);
    }
  }
  if (lane == 0)
  {
    atomicAdd(&A.counters[0], c0);
    atomicAdd(&A.counters[1], c1);
    atomicAdd(&A.counters[4], c4);
    if (STATS)
    {
      atomicAdd(&A.counters[2], c2);
      atomicAdd(&A.counters[3], c3);
    }
  }
}

/* ---- the production kernel: warp-scheduled state machine ---------------------------------
 * Same per-lane work as k_render, different control flow.  Profiling k_render on the
 * 1M-triangle scene (profiles/r1_c3_megakernel.md) showed 4.95 active lanes per issued
 * instruction: lanes sat idle while a few neighbours ran the long FP64 leaf tests or the
 * shading code.  Here every lane is in one of three states and each loop iteration the WARP
 * picks, by ballot, the state most lanes are in and executes only that block:
 *   NODE   walk inner BVH nodes (FP32 slab tests), a short burst per turn
 *   PRIM   one candidate primitive: FP32 pre-test, then the exact FP64 test
 *   SHADE  path_shade (Russian roulette, scatter), next sample, next ray set-up
 * Lanes in the other states wait for their turn, so the expensive blocks run with many
 * lanes active instead of one or two.  Progress is guaranteed: the chosen class is never
 * empty and every step of a class moves its lanes towards SHADE/IDLE. */
#ifndef RTB_NODE_BURST
#define RTB_NODE_BURST 3
#endif

enum { MODE_NODE = 0, MODE_PRIM = 1, MODE_SHADE = 2, MODE_IDLE = 3 };

template <bool STATS>
__global__ void __launch_bounds__(128, 8) k_render_sm(const __grid_constant__ RenderArgs A)
{
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int tile = warp % A.n_tiles;
  const int split = warp / A.n_tiles;
  const int x = (tile % A.tiles_x) * 8 + (lane & 7);
  const int y = (tile / A.tiles_x) * 4 + (lane >> 3);
  const bool valid = x < A.width && y < A.height && split < A.splits;
  const unsigned pixel = (unsigned)(y * A.width + x);

  int s = A.s_begin + split * A.chunk;
  const int s_end = valid ? min(A.s_end, s + A.chunk) : s;

  PathState st;
  st.alive = false;
  st.depth = 0;
  st.tr = st.tg = st.tb = 0.0f;
  st.o = d3_make(0, 0, 0);
  st.d = d3_make(0, 0, 1);
  float sr = 0.0f, sg = 0.0f, sb = 0.0f;
  PathCounters pc = { 0u, 0u };
  TraceStats ts = { 0u, 0u };
  unsigned paths = 0;

  HitRec best;
  best.t = DBL_MAX; best.gid = 0x7FFFFFFF; best.slot = 0;
  RayF rf;
  int2 stack_mem[RTB_STACK_SIZE];
  WalkStack<0> stack = { nullptr, stack_mem, 0 };
  stack.reset();
  int cur = 0, prim_i = 0, prim_end = 0;
  bool big_phase = false;
  int mode = (s < s_end) ? MODE_SHADE : MODE_IDLE;

  auto set_cur = [&](int ref) {
    if (ref == RTB_REF_NONE)
      mode = MODE_SHADE;
    else if (ref >= 0)
    {
      cur = ref;
      mode = MODE_NODE;
    }
    else
    {
      int code = ~ref;
      prim_i = code >> 3;
      prim_end = prim_i + (code & 7) + 1;
      mode = MODE_PRIM;
    }
  };
  auto begin_walk = [&]() {
    big_phase = false;
    if (!rayf_walk_setup(A.sv, st.o, st.d, best, rf))
    {
      mode = MODE_SHADE;
      return;
    }
    stack.reset();
    set_cur(A.sv.root_ref);
  };
  auto begin_ray = [&]() {
    best.t = DBL_MAX; best.gid = 0x7FFFFFFF; best.slot = 0;
    rayf_basic(st.o, st.d, rf);
    pc.rays++;
    pc.rays_hit++;
    if (A.sv.n_big > 0)
    {
      big_phase = true;
      prim_i = 0;
      prim_end = A.sv.n_big;
      mode = MODE_PRIM;
    }
    else
      begin_walk();
  };

  while (true)
  {
    const unsigned bn = __ballot_sync(0xFFFFFFFFu, mode == MODE_NODE);
    const unsigned bp = __ballot_sync(0xFFFFFFFFu, mode == MODE_PRIM);
    const unsigned bs = __ballot_sync(0xFFFFFFFFu, mode == MODE_SHADE);
    if ((bn | bp | bs) == 0u)
      break;
    const int cn = __popc(bn), cp = __popc(bp), cs = __popc(bs);
    if (cn >= cp && cn >= cs)
    {
      if (mode == MODE_NODE)
      {
#pragma unroll 1
        for (int it = 0; it < RTB_NODE_BURST && mode == MODE_NODE; it++)
        {
          if (STATS) ts.node_visits++;
          int nxt = node_step(A.sv, rf, cur, stack);
          if (nxt == RTB_REF_NONE)
            nxt = stack.pop(rf);
          set_cur(nxt);
        }
      }
    }
    else if (cp >= cs)
    {
      if (mode == MODE_PRIM)
      {
        PrimView p = load_prim(big_phase ? A.sv.big : A.sv.prims, prim_i);
        test_prim_filtered<true>(p, big_phase ? ~prim_i : prim_i, st.o, st.d, rf.ofx, rf.ofy, rf.ofz, rf.dfx, rf.dfy,
                           rf.dfz, rf.o_abs1, best, ts.prim_tests, big_phase ? nullptr : A.sv.tri64);
        prim_i++;
        if (prim_i == prim_end)
        {
          if (big_phase)
            begin_walk();
          else
          {
            rayf_update_tmax(rf, best);
            set_cur(stack.pop(rf));
          }
        }
      }
    }
    else
    {
      if (mode == MODE_SHADE)
      {
        if (st.alive)
        {
          path_shade(A, st, best, pixel, (unsigned)s, sr, sg, sb, pc, nullptr);
          if (!st.alive)
            s++;
        }
        if (!st.alive && s < s_end)
        {
          path_begin(A, st, x, y, pixel, (unsigned)s);
          paths++;
        }
        if (st.alive)
          begin_ray();
        else
          mode = MODE_IDLE;
      }
    }
  }

  if (valid)
  {
    float *o = A.out + ((size_t)split * A.width * A.height + pixel) * 3;
    o[0] = sr; o[1] = sg; o[2] = sb;
  }

  unsigned long long c0 = pc.rays, c1 = pc.rays_hit, c2 = ts.prim_tests, c3 = ts.node_visits, c4 = paths;
  for (int off = 16; off > 0; off >>= 1)
  {
    c0 += __shfl_xor_sync(0xFFFFFFFFu, c0, off);
    c1 += __shfl_xor_sync(0xFFFFFFFFu, c1, off);
    c4 += __shfl_xor_sync(0xFFFFFFFFu, c4, off);
    if (STATS)
    {
      c2 += __shfl_xor_sync(0xFFFFFFFFu, c2, off);
      c3 += __shfl_xor_sync(0xFFFFFFFFu, c3, off);
    }
  }
  if (lane == 0)
  {
    atomicAdd(&A.counters[0], c0);
    atomicAdd(&A.counters[1], c1);
    atomicAdd(&A.counters[4], c4);
    if (STATS)
    {
      atomicAdd(&A.counters[2], c2);
      atomicAdd(&A.counters[3], c3);
    }
  }
}

/* ---- megakernel with a SUSPENDABLE walk -------------------------------------------------------
 * profiles/r1_c3_k4_ncu.md: with the while-while walk only ~4 of 32 lanes are walking on
 * average -- traversal lengths have a long tail and a warp waits for its slowest ray at every
 * bounce.  Here a lane's walk state (current node, stack, best hit) survives across loop
 * trips: as soon as fewer than RTB_SUSPEND_LANES lanes are still walking AND some lanes are
 * waiting with a finished query, the walkers are suspended, the waiting lanes are shaded and
 * given their next ray (next bounce, or the pixel's next sample), and everybody resumes
 * walking together.  This is the persistent-threads "replace finished rays" idea (Aila &
 * Laine) inside the megakernel: no ray queues in memory, state stays in registers. */
#ifndef RTB_SUSPEND_LANES
#define RTB_SUSPEND_LANES 20
#endif

template <bool STATS>
__global__ void __launch_bounds__(128, 8) k_render_pw(const __grid_constant__ RenderArgs A)
{
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int tile = warp % A.n_tiles;
  const int split = warp / A.n_tiles;
  const int x = (tile % A.tiles_x) * 8 + (lane & 7);
  const int y = (tile / A.tiles_x) * 4 + (lane >> 3);
  const bool valid = x < A.width && y < A.height && split < A.splits;
  const unsigned pixel = (unsigned)(y * A.width + x);

  int s = A.s_begin + split * A.chunk;
  const int s_end = valid ? min(A.s_end, s + A.chunk) : s;

  PathState st;
  st.alive = false;
  st.depth = 0;
  st.tr = st.tg = st.tb = 0.0f;
  st.o = d3_make(0, 0, 0);
  st.d = d3_make(0, 0, 1);
  float sr = 0.0f, sg = 0.0f, sb = 0.0f;
  PathCounters pc = { 0u, 0u };
  TraceStats ts = { 0u, 0u };
  unsigned paths = 0;

  HitRec best;
  best.t = DBL_MAX; best.gid = 0x7FFFFFFF; best.slot = 0;
  RayF rf;
  rf.idx = rf.idy = rf.idz = rf.oodx = rf.oody = rf.oodz = rf.tmax = rf.t_base = 0.0f;
  int2 stack_mem[RTB_STACK_SIZE];
  WalkStack<0> stack = { nullptr, stack_mem, 0 };
  stack.reset();
  int cur = RTB_REF_NONE;
  bool walking = false;

  while (true)
  {
    if (!walking)
    {
      if (st.alive)
      {
        path_shade(A, st, best, pixel, (unsigned)s, sr, sg, sb, pc, nullptr);
        if (!st.alive)
          s++;
      }
      if (!st.alive && s < s_end)
      {
        path_begin(A, st, x, y, pixel, (unsigned)s);
        paths++;
      }
      if (st.alive)
      {
        pc.rays++;
        pc.rays_hit++;
        best.t = DBL_MAX; best.gid = 0x7FFFFFFF; best.slot = 0;
        rayf_basic(st.o, st.d, rf);
        big_list_select_test(A.sv, st.o, st.d, rf, best, ts.prim_tests);
        if (rayf_walk_setup(A.sv, st.o, st.d, best, rf))
        {
          stack.reset();
          cur = A.sv.root_ref;
          walking = cur != RTB_REF_NONE;
        }
      }
    }
    if (__all_sync(0xFFFFFFFFu, !st.alive))
      break;

    while (true)
    {
      const unsigned bw = __ballot_sync(0xFFFFFFFFu, walking);
      if (bw == 0u)
        break;
      const unsigned bwait = __ballot_sync(0xFFFFFFFFu, st.alive && !walking);
      if (bwait != 0u && __popc(bw) < A.suspend_lanes)
        break;
      /* node phase: inner nodes only; ends as soon as fewer than half of the walkers are
       * still at inner nodes (the others wait with a leaf or a finished query) */
      const int n_walk = __popc(bw);
      while (true)
      {
        const bool at_node = walking && cur >= 0 && cur != RTB_REF_NONE;
        const unsigned bnode = __ballot_sync(0xFFFFFFFFu, at_node);
        if (bnode == 0u || 2 * __popc(bnode) < n_walk)
          break;
        if (at_node)
        {
          if (STATS) ts.node_visits++;
          int nxt = node_step(A.sv, rf, cur, stack);
          cur = (nxt != RTB_REF_NONE) ? nxt : stack.pop(rf);
          if (cur == RTB_REF_NONE)
            walking = false;
        }
      }
      /* leaf phase */
      if (walking && cur < 0)
      {
        int code = ~cur;
        int first = code >> 3, count = (code & 7) + 1;
        for (int k = 0; k < count; k++)
        {
          test_prim(load_prim(A.sv.prims, first + k), first + k, st.o, st.d, best, A.sv.tri64);
          if (STATS) ts.prim_tests++;
        }
        rayf_update_tmax(rf, best);
        cur = stack.pop(rf);
        if (cur == RTB_REF_NONE)
          walking = false;
      }
    }
  }

  if (valid)
  {
    float *o = A.out + ((size_t)split * A.width * A.height + pixel) * 3;
    o[0] = sr; o[1] = sg; o[2] = sb;
  }

  unsigned long long c0 = pc.rays, c1 = pc.rays_hit, c2 = ts.prim_tests, c3 = ts.node_visits, c4 = paths;
  for (int off = 16; off > 0; off >>= 1)
  {
    c0 += __shfl_xor_sync(0xFFFFFFFFu, c0, off);
    c1 += __shfl_xor_sync(0xFFFFFFFFu, c1, off);
    c4 += __shfl_xor_sync(0xFFFFFFFFu, c4, off);
    if (STATS)
    {
      c2 += __shfl_xor_sync(0xFFFFFFFFu, c2, off);
      c3 += __shfl_xor_sync(0xFFFFFFFFu, c3, off);
    }
  }
  if (lane == 0)
  {
    atomicAdd(&A.counters[0], c0);
    atomicAdd(&A.counters[1], c1);
    atomicAdd(&A.counters[4], c4);
    if (STATS)
    {
      atomicAdd(&A.counters[2], c2);
      atomicAdd(&A.counters[3], c3);
    }
  }
}

/* sum of the split planes, in plane order (deterministic) */
__global__ void k_sum_planes(const float *__restrict__ planes, int splits, size_t n, float *__restrict__ out)
{
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n)
    return;
  float acc = 0.0f;
  for (int k = 0; k < splits; k++)
    acc += planes[(size_t)k * n + i];
  out[i] = acc;
}

/* raytracer.c:215-220: mean, pow(c, 1/5.0), clamp, truncate.  NaN -> 255 (CLAMP macro). */
__global__ void k_tonemap(const float *__restrict__ accum, size_t n, double inv_samples, uint8_t *__restrict__ fb)
{
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n)
    return;
  double c = __dmul_rn((double)accum[i], inv_samples);
  double g = pow(c, __ddiv_rn(1.0, 5.0));
  double clamped = (g < 1.0) ? g : 1.0; /* MIN(x, 1): NaN -> 1 */
  clamped = (0.0 > clamped) ? 0.0 : clamped; /* MAX(0, .) */
  fb[i] = (uint8_t)(__dmul_rn(255.0, clamped));
}

/* ---- probes ------------------------------------------------------------------------ */

__global__ void k_trace_rays(const __grid_constant__ SceneView sv, const double *__restrict__ rays, size_t n,
                             int use_bvh, int *__restrict__ ids, long long *__restrict__ prims,
                             double *__restrict__ ts, double *__restrict__ points, double *__restrict__ normals,
                             double *__restrict__ uvs)
{
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n)
    return;
  d3 o = d3_make(rays[6 * i + 0], rays[6 * i + 1], rays[6 * i + 2]);
  d3 d = d3_make(rays[6 * i + 3], rays[6 * i + 4], rays[6 * i + 5]);
  HitRec best;
  TraceStats st = { 0u, 0u };
  if ((use_bvh == 5 || sv.nodes == nullptr) && use_bvh != 0 && sv.nodes4q != nullptr)
    closest_hit_ww<false, 0, 2>(sv, o, d, best, st, nullptr, 0);
  else if (use_bvh == 4 && sv.nodes4 != nullptr)
    closest_hit_ww<false, 0, 1>(sv, o, d, best, st, nullptr, 0);
  else if (use_bvh >= 3)
    closest_hit_ww<false, 0>(sv, o, d, best, st, nullptr, 0);
  else if (use_bvh == 2)
    closest_hit<false, true>(sv, o, d, best, st);
  else if (use_bvh)
    closest_hit<false, false>(sv, o, d, best, st);
  else
    closest_hit_bruteforce(sv, o, d, best);
  store_hit_record(sv, o, d, best, i, ids, prims, ts, points, normals, uvs);
}

/* the first n_vertices vertices of sample `sample` of every pixel, through the very same
 * path_begin / closest_hit / path_shade as k_render */
__global__ void k_path_records(const __grid_constant__ RenderArgs A, int sample, int n_vertices,
                               int *__restrict__ ids, double *__restrict__ points, double *__restrict__ normals,
                               double *__restrict__ dists, float *__restrict__ radiance)
{
  int pix = blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= A.width * A.height)
    return;
  int x = pix % A.width, y = pix / A.width;
  for (int k = 0; k < n_vertices; k++)
  {
    ids[(size_t)pix * n_vertices + k] = -2;
    dists[(size_t)pix * n_vertices + k] = 0.0;
    for (int c = 0; c < 3; c++)
    {
      points[((size_t)pix * n_vertices + k) * 3 + c] = 0.0;
      normals[((size_t)pix * n_vertices + k) * 3 + c] = 0.0;
    }
  }
  PathState st;
  path_begin(A, st, x, y, (unsigned)pix, (unsigned)sample);
  float sr = 0, sg = 0, sb = 0;
  PathCounters pc = { 0u, 0u };
  TraceStats ts = { 0u, 0u };
  int vertex = 0;
  while (st.alive)
  {
    HitRec best;
    if (A.sv.nodes4q != nullptr)
      closest_hit_ww<false, 0, 2>(A.sv, st.o, st.d, best, ts, nullptr, 0);
    else
      closest_hit<false, false>(A.sv, st.o, st.d, best, ts);
    d3 origin = st.o;
    Surface s;
    bool hit = best.t < 1e300;
    path_shade(A, st, best, (unsigned)pix, (unsigned)sample, sr, sg, sb, pc, &s);
    if (vertex < n_vertices)
    {
      size_t r = (size_t)pix * n_vertices + vertex;
      ids[r] = hit ? s.object : -1;
      if (hit)
      {
        dists[r] = d3_length(d3_sub(s.point, origin));
        points[3 * r] = s.point.x; points[3 * r + 1] = s.point.y; points[3 * r + 2] = s.point.z;
        normals[3 * r] = s.normal.x; normals[3 * r + 1] = s.normal.y; normals[3 * r + 2] = s.normal.z;
      }
    }
    vertex++;
  }
  if (radiance)
  {
    radiance[3 * (size_t)pix] = sr; radiance[3 * (size_t)pix + 1] = sg; radiance[3 * (size_t)pix + 2] = sb;
  }
}

__global__ void k_philox(const uint4 *__restrict__ ctr, const uint2 *__restrict__ key, size_t n, uint4 *__restrict__ out)
{
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n)
    out[i] = philox4x32_10(ctr[i], key[i]);
}

/* ---- host entry points ---------------------------------------------------------------- */

static int check_desc(const rtb_render_desc *d)
{
  if (!d || d->width < 2 || d->height < 2 || d->sample_end < d->sample_begin || d->max_depth < 0 ||
      d->max_depth > 255 || (long long)d->width * d->height >= (1ll << 30))
  {
    /* width/height 1 divide by zero upstream (quirk Q11) */
    rtb_set_error("rtb_render_desc: need width,height >= 2, sample_end >= sample_begin, 0 <= max_depth <= 255");
    return RTB_EINVAL;
  }
  if (d->kernel < 0 || d->kernel > 6)
  {
    rtb_set_error("rtb_render_desc.kernel: 0 auto, 1..5 megakernel variants, 6 wavefront");
    return RTB_EINVAL;
  }
  if (d->integrator != RTB_INTEGRATOR_PATH && d->integrator != RTB_INTEGRATOR_WHITTED)
  {
    rtb_set_error("rtb_render_desc.integrator: RTB_INTEGRATOR_PATH or RTB_INTEGRATOR_WHITTED");
    return RTB_EINVAL;
  }
  if (d->dielectric_mode != RTB_DIELECTRIC_STOCHASTIC && d->dielectric_mode != RTB_DIELECTRIC_SPLIT)
  {
    rtb_set_error("dielectric_mode: RTB_DIELECTRIC_STOCHASTIC or RTB_DIELECTRIC_SPLIT");
    return RTB_EINVAL;
  }
  if (d->dielectric_mode == RTB_DIELECTRIC_SPLIT &&
      (d->max_depth > 16 || (d->kernel != 0 && d->kernel != 6) || d->integrator != RTB_INTEGRATOR_PATH))
  {
    /* 2^(depth+1) rays per path: the reference's estimator is tractable for shallow paths only (its MAX_DEPTH is 5) */
    rtb_set_error("RTB_DIELECTRIC_SPLIT: wavefront path tracer only (kernel 0 or 6), max_depth <= 16");
    return RTB_EINVAL;
  }
  return RTB_OK;
}

static void fill_args(RenderArgs &A, const rtb_scene *scene, const double *camera12, const rtb_render_desc *desc)
{
  A.sv = scene->view;
  for (int k = 0; k < 3; k++)
  {
    A.cam.pos[k] = camera12[k];
    A.cam.horizontal[k] = camera12[3 + k];
    A.cam.vertical[k] = camera12[6 + k];
    A.cam.llc[k] = camera12[9 + k];
  }
  A.width = desc->width;
  A.height = desc->height;
  A.tiles_x = (desc->width + 7) / 8;
  A.n_tiles = A.tiles_x * ((desc->height + 3) / 4);
  A.s_begin = desc->sample_begin;
  A.s_end = desc->sample_end;
  A.max_depth = desc->max_depth;
  A.dielectric_mode = desc->dielectric_mode;
  A.suspend_lanes = (desc->reserved > 0 && desc->reserved <= 32) ? desc->reserved : RTB_SUSPEND_LANES;
  A.plane_base = 0;
  A.key = make_uint2((unsigned)(desc->seed & 0xFFFFFFFFull), (unsigned)(desc->seed >> 32));
  A.counters = scene->d_counters;
}

namespace
{
struct EventPair /* two CUDA events, destroyed on every return path */
{
  cudaEvent_t a = nullptr, b = nullptr;
  ~EventPair()
  {
    if (a) cudaEventDestroy(a);
    if (b) cudaEventDestroy(b);
  }
};
} // namespace

extern "C" int rtb_render_accum(rtb_scene *scene, const double *camera12, const rtb_render_desc *desc,
                                float *d_accum, void *stream_, rtb_counters *counters)
{
  if (!scene || !camera12 || !d_accum)
  {
    rtb_set_error("rtb_render_accum: NULL argument");
    return RTB_EINVAL;
  }
  int rc = check_desc(desc);
  if (rc != RTB_OK)
    return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  RTB_CUDA(cudaSetDevice(scene->device));

  RenderArgs A;
  fill_args(A, scene, camera12, desc);
  const int spp = desc->sample_end - desc->sample_begin;
  const size_t n_px = (size_t)desc->width * desc->height;
  /* Planes: the call's samples are cut into `splits` contiguous sub-ranges that are accumulated
   * separately and summed in order -- this fixes the floating-point summation order, so every
   * kernel variant gives the same bits for the same number of planes.
   * Megakernels: enough threads to fill 148 SMs a few times over even for small frames.
   * Wavefront: up to 128 M paths in flight, in two plane groups of 64 M on two streams (23.4 GB of queues
   * out of 180 GB): the deep bounces then still have enough rays to fill 148 SMs and the tail of one
   * group's persistent kernel is covered by the other group's next kernel (measured C3, round 2: 32 M
   * 4.19, 64 M 4.29, 128 M 4.35 Grays/s); never more than a quarter of the free device memory. */
  const bool whitted = desc->integrator == RTB_INTEGRATOR_WHITTED;
  const bool wavefront = (desc->kernel == 6 || desc->kernel == 0) && !whitted;
  if (!wavefront && desc->integrator == RTB_INTEGRATOR_PATH && scene->view.nodes == nullptr && scene->view.root_ref >= 0 &&
      scene->view.root_ref != RTB_REF_NONE)
  {
    rtb_set_error("rtb_render_desc.kernel 1..5 walk the BVH2: create the scene with RTB_SCENE_ALL_TREES");
    return RTB_EINVAL;
  }
  long long want_threads = 148ll * 2048 * 2;
  if (wavefront)
  {
    /* the free memory is read once per device (cudaMemGetInfo costs milliseconds, render() makes a
     * new scene per call); it also keeps the plane count -- and with it the summation order --
     * the same from call to call */
    long long wave_paths = 128ll << 20; /* path slots in flight (both plane groups together): 23.4 GB of queues */
    if (const char *e = getenv("RTB_WF_PATHS_M"))
      wave_paths = std::max(1ll, atoll(e)) << 20;
    static std::atomic<long long> path_cap[64]; /* zero-initialised; scenes on several devices render from several host threads */
    const int dev = scene->device;
    if (dev < 0 || dev >= 64 || path_cap[dev].load() == 0)
    {
      size_t free_b = 0, total_b = 0;
      RTB_CUDA(cudaMemGetInfo(&free_b, &total_b));
      const long long cap = std::max<long long>(1ll << 20, (long long)((free_b + scene->wf_bytes) / 4 / 192));
      if (dev >= 0 && dev < 64)
        path_cap[dev].store(cap);
      want_threads = std::min<long long>(wave_paths, cap);
    }
    else
      want_threads = std::min<long long>(wave_paths, path_cap[dev].load());
    if (desc->dielectric_mode == RTB_DIELECTRIC_SPLIT) /* the queues hold up to 64 entries per path slot */
      want_threads >>= std::min(desc->max_depth + 1, 6);
    want_threads = std::max<long long>(want_threads, (long long)n_px);
  }
  int splits = (int)std::min<long long>(std::max<long long>(1, (want_threads + (long long)n_px - 1) / (long long)n_px), 64);
  if (desc->planes > 0)
    splits = std::min(desc->planes, 1024);
  splits = std::max(1, std::min(splits, spp));
  int chunk = spp > 0 ? (spp + splits - 1) / splits : 0;
  if (chunk > 0)
    splits = (spp + chunk - 1) / chunk;
  A.chunk = chunk;
  A.splits = splits;

  unsigned long long launches = 0;
  float phase_ms[3] = { 0.0f, 0.0f, 0.0f };
  EventPair evp;
  cudaEvent_t &ev0 = evp.a, &ev1 = evp.b;
  if (counters)
  {
    RTB_CUDA(cudaEventCreate(&ev0));
    RTB_CUDA(cudaEventCreate(&ev1));
    RTB_CUDA(cudaMemsetAsync(scene->d_counters, 0, sizeof(unsigned long long) * 8, stream));
    RTB_CUDA(cudaEventRecord(ev0, stream));
  }

  if (spp == 0)
  {
    RTB_CUDA(cudaMemsetAsync(d_accum, 0, sizeof(float) * 3 * n_px, stream));
  }
  else
  {
    if (wavefront)
    {
      int wrc = wf_render(scene, A, desc, d_accum, stream, counters != nullptr && desc->profile != 0, launches,
                          (counters && desc->profile != 0) ? phase_ms : nullptr);
      /* the free memory was sampled once per device: if the queues no longer fit, halve the wave
       * (only when the caller did not pin the plane count, which fixes the summation order) */
      while (wrc == RTB_ENOMEM && desc->planes == 0 && A.splits > 1)
      {
        A.splits = (A.splits + 1) / 2;
        A.chunk = (spp + A.splits - 1) / A.splits;
        A.splits = (spp + A.chunk - 1) / A.chunk;
        launches = 0;
        wrc = wf_render(scene, A, desc, d_accum, stream, counters != nullptr && desc->profile != 0, launches,
                        (counters && desc->profile != 0) ? phase_ms : nullptr);
      }
      if (wrc != RTB_OK)
        return wrc;
    }
    else
    {
    if (splits > 1)
    {
      size_t need = sizeof(float) * 3 * n_px * splits;
      if (scene->scratch_bytes < need)
      {
        if (scene->d_scratch)
          RTB_CUDA(cudaFreeAsync(scene->d_scratch, stream));
        scene->d_scratch = nullptr;
        scene->scratch_bytes = 0;
        RTB_CUDA(cudaMallocAsync(reinterpret_cast<void **>(&scene->d_scratch), need, stream));
        scene->scratch_bytes = need;
      }
      A.out = scene->d_scratch;
    }
    else
      A.out = d_accum;
    const int threads = 128;
    const long long warps = (long long)A.n_tiles * splits;
    const int blocks = (int)((warps * 32 + threads - 1) / threads);
    if (whitted)
    {
      /* cast_ray: one thread per (plane, pixel), like the megakernels */
      int wrc = whitted_render(scene, A, stream, launches);
      if (wrc != RTB_OK)
        return wrc;
    }
    else
    /* desc->kernel: 0/1 megakernel (default), 2 warp-scheduled state machine (+FP32 sphere
     * pre-test), 3 megakernel + FP32 sphere pre-test.  See DESIGN.md "Kernel choice". */
    switch (desc->kernel)
    {
    case 1: /* the first megakernel: if-if walk, 16 warps/SM (kept as the measured baseline) */
      if (counters) k_render<true, 0><<<blocks, threads, 0, stream>>>(A);
      else k_render<false, 0><<<blocks, threads, 0, stream>>>(A);
      break;
    case 2:
      if (counters) k_render_sm<true><<<blocks, threads, 0, stream>>>(A);
      else k_render_sm<false><<<blocks, threads, 0, stream>>>(A);
      break;
    case 3:
      if (counters) k_render<true, 1><<<blocks, threads, 0, stream>>>(A);
      else k_render<false, 1><<<blocks, threads, 0, stream>>>(A);
      break;
    case 5:
      if (counters) k_render_pw<true><<<blocks, threads, 0, stream>>>(A);
      else k_render_pw<false><<<blocks, threads, 0, stream>>>(A);
      break;
    default: /* 4: while-while walk + select-then-test, 64 registers -> 32 warps/SM */
      if (counters) k_render<true, 2><<<blocks, threads, 0, stream>>>(A);
      else k_render<false, 2><<<blocks, threads, 0, stream>>>(A);
      break;
    }
    RTB_CUDA(cudaGetLastError());
    launches++;
    if (splits > 1)
    {
      size_t n = 3 * n_px;
      k_sum_planes<<<(int)((n + 255) / 256), 256, 0, stream>>>(scene->d_scratch, splits, n, d_accum);
      RTB_CUDA(cudaGetLastError());
      launches++;
    }
    }
  }

  if (counters)
  {
    RTB_CUDA(cudaEventRecord(ev1, stream));
    RTB_CUDA(cudaEventSynchronize(ev1));
    unsigned long long h[8];
    RTB_CUDA(cudaMemcpy(h, scene->d_counters, sizeof(h), cudaMemcpyDeviceToHost));
    memset(counters, 0, sizeof(*counters));
    counters->rays = h[0];
    counters->rays_intersected = h[1];
    counters->prim_tests = h[2];
    counters->node_visits = h[3];
    counters->paths = h[4];
    counters->launches = launches;
    RTB_CUDA(cudaEventElapsedTime(&counters->gpu_ms, ev0, ev1));
    counters->build_ms = scene->info.build_ms;
    counters->trace_ms = phase_ms[0];
    counters->shade_ms = phase_ms[1];
    counters->trace_launches = (unsigned long long)phase_ms[2];
  }
  return RTB_OK;
}

extern "C" int rtb_tonemap(const float *d_accum, int width, int height, int total_samples, uint8_t *d_fb,
                           int device, void *stream_)
{
  if (!d_accum || !d_fb || width <= 0 || height <= 0 || total_samples <= 0)
  {
    rtb_set_error("rtb_tonemap: bad argument");
    return RTB_EINVAL;
  }
  RTB_CUDA(cudaSetDevice(device));
  size_t n = (size_t)3 * width * height;
  k_tonemap<<<(int)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream_)>>>(d_accum, n, 1.0 / (double)total_samples, d_fb);
  RTB_CUDA(cudaGetLastError());
  return RTB_OK;
}

extern "C" int rtb_render(rtb_scene *scene, const double *camera12, const rtb_render_desc *desc,
                          uint8_t *framebuffer, float *accum_or_null, rtb_counters *counters)
{
  const int spp = desc ? desc->sample_end - desc->sample_begin : 0;
  return rtb_render_mean(scene, camera12, desc, spp > 0 ? spp : 1, framebuffer, accum_or_null, counters);
}

extern "C" int rtb_render_mean(rtb_scene *scene, const double *camera12, const rtb_render_desc *desc, int total_samples,
                               uint8_t *framebuffer, float *accum_or_null, rtb_counters *counters)
{
  if (!scene || !framebuffer || total_samples <= 0)
  {
    rtb_set_error("rtb_render: NULL argument or total_samples <= 0");
    return RTB_EINVAL;
  }
  int rc = check_desc(desc);
  if (rc != RTB_OK)
    return rc;
  RTB_CUDA(cudaSetDevice(scene->device));
  size_t n = (size_t)3 * desc->width * desc->height;
  float *d_accum = nullptr;
  uint8_t *d_fb = nullptr;
  /* pooled, stream-ordered (see rtb_scene.cu: cudaMalloc/cudaFree are the dominant host cost) */
  RTB_CUDA(cudaMallocAsync(reinterpret_cast<void **>(&d_accum), sizeof(float) * n, 0));
  if (cudaMallocAsync(reinterpret_cast<void **>(&d_fb), n, 0) != cudaSuccess)
  {
    cudaFreeAsync(d_accum, 0);
    rtb_set_error("rtb_render: framebuffer allocation failed");
    return RTB_ECUDA;
  }
  rc = rtb_render_accum(scene, camera12, desc, d_accum, nullptr, counters);
  if (rc == RTB_OK)
    rc = rtb_tonemap(d_accum, desc->width, desc->height, total_samples, d_fb, scene->device, nullptr);
  if (rc == RTB_OK)
  {
    cudaError_t e = cudaMemcpy(framebuffer, d_fb, n, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && accum_or_null)
      e = cudaMemcpy(accum_or_null, d_accum, sizeof(float) * n, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess)
    {
      rtb_set_error(std::string("rtb_render: ") + cudaGetErrorString(e));
      rc = RTB_ECUDA;
    }
    if (counters)
      counters->launches += 1;
  }
  cudaFreeAsync(d_accum, 0);
  cudaFreeAsync(d_fb, 0);
  return rc;
}

extern "C" int rtb_trace_rays(rtb_scene *scene, const double *rays6, size_t n_rays, int use_bvh, int32_t *ids,
                              int64_t *prims, double *ts, double *points, double *normals, double *uvs)
{
  if (!scene || (n_rays && (!rays6 || !ids)))
  {
    rtb_set_error("rtb_trace_rays: NULL argument");
    return RTB_EINVAL;
  }
  if (n_rays == 0)
    return RTB_OK;
  if (use_bvh >= 2 && use_bvh <= 4 && scene->view.nodes == nullptr && scene->view.root_ref >= 0 &&
      scene->view.root_ref != RTB_REF_NONE)
  {
    rtb_set_error("rtb_trace_rays: use_bvh 2..4 walk the BVH2 / uncompressed BVH4: create the scene with RTB_SCENE_ALL_TREES");
    return RTB_EINVAL;
  }
  RTB_CUDA(cudaSetDevice(scene->device));
  Dev<double> d_rays, d_ts, d_points, d_normals, d_uvs;
  Dev<int> d_ids;
  Dev<long long> d_prims;
  RTB_CUDA(cudaMalloc(&d_rays.p, sizeof(double) * 6 * n_rays));
  RTB_CUDA(cudaMalloc(&d_ids.p, sizeof(int) * n_rays));
  RTB_CUDA(cudaMalloc(&d_prims.p, sizeof(long long) * n_rays));
  RTB_CUDA(cudaMalloc(&d_ts.p, sizeof(double) * n_rays));
  RTB_CUDA(cudaMalloc(&d_points.p, sizeof(double) * 3 * n_rays));
  RTB_CUDA(cudaMalloc(&d_normals.p, sizeof(double) * 3 * n_rays));
  RTB_CUDA(cudaMalloc(&d_uvs.p, sizeof(double) * 2 * n_rays));
  RTB_CUDA(cudaMemcpy(d_rays.p, rays6, sizeof(double) * 6 * n_rays, cudaMemcpyHostToDevice));
  k_trace_rays<<<(int)((n_rays + 127) / 128), 128>>>(scene->view, d_rays.p, n_rays, use_bvh, d_ids.p, d_prims.p,
                                                     d_ts.p, d_points.p, d_normals.p, d_uvs.p);
  RTB_CUDA(cudaGetLastError());
  RTB_CUDA(cudaDeviceSynchronize());
  RTB_CUDA(cudaMemcpy(ids, d_ids.p, sizeof(int) * n_rays, cudaMemcpyDeviceToHost));
  if (prims) RTB_CUDA(cudaMemcpy(prims, d_prims.p, sizeof(long long) * n_rays, cudaMemcpyDeviceToHost));
  if (ts) RTB_CUDA(cudaMemcpy(ts, d_ts.p, sizeof(double) * n_rays, cudaMemcpyDeviceToHost));
  if (points) RTB_CUDA(cudaMemcpy(points, d_points.p, sizeof(double) * 3 * n_rays, cudaMemcpyDeviceToHost));
  if (normals) RTB_CUDA(cudaMemcpy(normals, d_normals.p, sizeof(double) * 3 * n_rays, cudaMemcpyDeviceToHost));
  if (uvs) RTB_CUDA(cudaMemcpy(uvs, d_uvs.p, sizeof(double) * 2 * n_rays, cudaMemcpyDeviceToHost));
  return RTB_OK;
}

extern "C" int rtb_path_records(rtb_scene *scene, const double *camera12, const rtb_render_desc *desc, int sample,
                                int n_vertices, int32_t *ids, double *points, double *normals, double *dists,
                                float *radiance)
{
  if (!scene || !camera12 || !ids || !points || !normals || !dists || n_vertices < 1)
  {
    rtb_set_error("rtb_path_records: bad argument");
    return RTB_EINVAL;
  }
  int rc = check_desc(desc);
  if (rc != RTB_OK)
    return rc;
  RTB_CUDA(cudaSetDevice(scene->device));
  RenderArgs A;
  fill_args(A, scene, camera12, desc);
  A.chunk = 1;
  A.splits = 1;
  A.out = nullptr;
  size_t n_px = (size_t)desc->width * desc->height, nr = n_px * n_vertices;
  Dev<int> d_ids;
  Dev<double> d_points, d_normals, d_dists;
  Dev<float> d_rad;
  RTB_CUDA(cudaMalloc(&d_ids.p, sizeof(int) * nr));
  RTB_CUDA(cudaMalloc(&d_points.p, sizeof(double) * 3 * nr));
  RTB_CUDA(cudaMalloc(&d_normals.p, sizeof(double) * 3 * nr));
  RTB_CUDA(cudaMalloc(&d_dists.p, sizeof(double) * nr));
  RTB_CUDA(cudaMalloc(&d_rad.p, sizeof(float) * 3 * n_px));
  k_path_records<<<(int)((n_px + 127) / 128), 128>>>(A, sample, n_vertices, d_ids.p, d_points.p, d_normals.p,
                                                     d_dists.p, d_rad.p);
  RTB_CUDA(cudaGetLastError());
  RTB_CUDA(cudaDeviceSynchronize());
  RTB_CUDA(cudaMemcpy(ids, d_ids.p, sizeof(int) * nr, cudaMemcpyDeviceToHost));
  RTB_CUDA(cudaMemcpy(points, d_points.p, sizeof(double) * 3 * nr, cudaMemcpyDeviceToHost));
  RTB_CUDA(cudaMemcpy(normals, d_normals.p, sizeof(double) * 3 * nr, cudaMemcpyDeviceToHost));
  RTB_CUDA(cudaMemcpy(dists, d_dists.p, sizeof(double) * nr, cudaMemcpyDeviceToHost));
  if (radiance)
    RTB_CUDA(cudaMemcpy(radiance, d_rad.p, sizeof(float) * 3 * n_px, cudaMemcpyDeviceToHost));
  return RTB_OK;
}

/* ---- L2 read-bandwidth probe: the denominator for the walk's algorithmic bytes (SURVEY 8d asks for
 * a measured L2 peak; MEASURED_PEAKS.json only holds HBM and BF16) -------------------------------- */
__global__ void __launch_bounds__(256) k_probe_l2(const uint4 *__restrict__ buf, size_t n_vec, int iters, unsigned *sink)
{
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  uint4 acc = make_uint4(0u, 0u, 0u, 0u);
  for (int it = 0; it < iters; it++)
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += stride)
    {
      const uint4 v = __ldcg(buf + i); /* cached in L2 only */
      acc.x ^= v.x; acc.y ^= v.y; acc.z ^= v.z; acc.w ^= v.w;
    }
  if ((acc.x ^ acc.y ^ acc.z ^ acc.w) == 0x9E3779B9u)
    *sink = 1u;
}

extern "C" int rtb_probe_l2_bandwidth(size_t bytes, int iters, int device, float *gb_per_s)
{
  if (!gb_per_s || bytes < 4096 || iters < 1)
  {
    rtb_set_error("rtb_probe_l2_bandwidth: bad argument");
    return RTB_EINVAL;
  }
  RTB_CUDA(cudaSetDevice(device));
  Dev<uint4> d_buf;
  Dev<unsigned> d_sink;
  const size_t n_vec = bytes / sizeof(uint4);
  RTB_CUDA(cudaMalloc(&d_buf.p, n_vec * sizeof(uint4)));
  RTB_CUDA(cudaMalloc(&d_sink.p, sizeof(unsigned)));
  RTB_CUDA(cudaMemset(d_buf.p, 1, n_vec * sizeof(uint4)));
  int sm_count = 148;
  cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, device);
  EventPair ev;
  cudaEvent_t &e0 = ev.a, &e1 = ev.b;
  RTB_CUDA(cudaEventCreate(&e0));
  RTB_CUDA(cudaEventCreate(&e1));
  k_probe_l2<<<sm_count * 8, 256>>>(d_buf.p, n_vec, 2, d_sink.p); /* warm: pull the buffer into L2 */
  RTB_CUDA(cudaEventRecord(e0));
  k_probe_l2<<<sm_count * 8, 256>>>(d_buf.p, n_vec, iters, d_sink.p);
  RTB_CUDA(cudaEventRecord(e1));
  RTB_CUDA(cudaEventSynchronize(e1));
  float ms = 0.0f;
  RTB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
  *gb_per_s = (float)((double)n_vec * sizeof(uint4) * iters / (ms * 1e-3) / 1e9);
  return RTB_OK;
}

/* ---- FP32 FMA throughput probe: the denominator of the walk's algorithmic flops (SURVEY 8d asks for a measured
 * FP32 peak as well) ------------------------------------------------------------------------------------------ */
__global__ void __launch_bounds__(256) k_probe_fp32(int iters, float seed, float *sink)
{
  /* 8 independent FMA chains per thread: enough ILP to keep the FMA pipe fed at 8 warps per scheduler */
  float a0 = seed + threadIdx.x, a1 = a0 + 1.0f, a2 = a0 + 2.0f, a3 = a0 + 3.0f, a4 = a0 + 4.0f, a5 = a0 + 5.0f, a6 = a0 + 6.0f,
        a7 = a0 + 7.0f;
  const float m = 0.999999f, c = 1e-7f;
  for (int it = 0; it < iters; it++)
  {
#pragma unroll
    for (int u = 0; u < 16; u++)
    {
      a0 = fmaf(a0, m, c); a1 = fmaf(a1, m, c); a2 = fmaf(a2, m, c); a3 = fmaf(a3, m, c);
      a4 = fmaf(a4, m, c); a5 = fmaf(a5, m, c); a6 = fmaf(a6, m, c); a7 = fmaf(a7, m, c);
    }
  }
  const float r = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
  if (r == 123456.789f)
    *sink = r;
}

extern "C" int rtb_probe_fp32_tflops(int iters, int device, float *tflops)
{
  if (!tflops || iters < 1)
  {
    rtb_set_error("rtb_probe_fp32_tflops: bad argument");
    return RTB_EINVAL;
  }
  RTB_CUDA(cudaSetDevice(device));
  Dev<float> d_sink;
  RTB_CUDA(cudaMalloc(&d_sink.p, sizeof(float)));
  int sm_count = 148;
  cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, device);
  const int blocks = sm_count * 8, threads = 256;
  EventPair ev;
  cudaEvent_t &e0 = ev.a, &e1 = ev.b;
  RTB_CUDA(cudaEventCreate(&e0));
  RTB_CUDA(cudaEventCreate(&e1));
  k_probe_fp32<<<blocks, threads>>>(iters / 8 + 1, 1.0f, d_sink.p); /* warm */
  RTB_CUDA(cudaEventRecord(e0));
  k_probe_fp32<<<blocks, threads>>>(iters, 1.0f, d_sink.p);
  RTB_CUDA(cudaEventRecord(e1));
  RTB_CUDA(cudaEventSynchronize(e1));
  float ms = 0.0f;
  RTB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
  const double flops = 2.0 * 8.0 * 16.0 * (double)iters * (double)blocks * threads;
  *tflops = (float)(flops / (ms * 1e-3) / 1e12);
  return RTB_OK;
}

extern "C" int rtb_philox4x32_10(const uint32_t *ctr4, const uint32_t *key2, size_t n, uint32_t *out4, int device)
{
  if (!ctr4 || !key2 || !out4)
  {
    rtb_set_error("rtb_philox4x32_10: NULL argument");
    return RTB_EINVAL;
  }
  if (n == 0)
    return RTB_OK;
  RTB_CUDA(cudaSetDevice(device));
  Dev<uint4> d_ctr, d_out;
  Dev<uint2> d_key;
  RTB_CUDA(cudaMalloc(&d_ctr.p, sizeof(uint4) * n));
  RTB_CUDA(cudaMalloc(&d_out.p, sizeof(uint4) * n));
  RTB_CUDA(cudaMalloc(&d_key.p, sizeof(uint2) * n));
  RTB_CUDA(cudaMemcpy(d_ctr.p, ctr4, sizeof(uint4) * n, cudaMemcpyHostToDevice));
  RTB_CUDA(cudaMemcpy(d_key.p, key2, sizeof(uint2) * n, cudaMemcpyHostToDevice));
  k_philox<<<(int)((n + 127) / 128), 128>>>(d_ctr.p, d_key.p, n, d_out.p);
  RTB_CUDA(cudaGetLastError());
  RTB_CUDA(cudaDeviceSynchronize());
  RTB_CUDA(cudaMemcpy(out4, d_out.p, sizeof(uint4) * n, cudaMemcpyDeviceToHost));
  return RTB_OK;
}
