/*
 * rtb_multi.cu -- render() on all the GPUs of one box, behind the C ABI.
 *
 * The path shards over samples (SURVEY.md 8e): the per-pixel sum of raytracer.c:199-213 is a sum of
 * independent samples, so rank r of G renders the global sample indices
 * [begin + r*spp/G, begin + (r+1)*spp/G) -- the Philox counter carries the GLOBAL index, the G-GPU image
 * is the same estimator as the 1-GPU one -- into its own float accumulation buffer, and the buffers are
 * summed by ONE ncclReduce(sum, float32) to rank 0 over NVLink / NVSwitch before the gamma + quantise
 * kernel (raytracer.c:215-220) runs there.  The second exchange step is the scene: with G GPUs every rank
 * uploads and marshals 1/G of the triangles over its own PCIe link (120 B each) and the marshalled records
 * (104 B each) are all-gathered over NVLink (rtb_scene.cu); every rank then builds its own BVH (1 ms).
 *
 * Two ways to form the group:
 *   rtb_comm_create_rank   one process per GPU (torchrun / mpirun): the 128-byte id from rtb_comm_unique_id
 *                          on rank 0 is passed to the others by whatever the launcher offers;
 *   rtb_comm_create_local  one process drives all GPUs (the unchanged main.c: render() is called from
 *                          one thread, main.c:429): ncclCommInitAll, one host thread per GPU inside the
 *                          collective calls below.
 * Every entry point taking a comm is COLLECTIVE: all ranks of the group call it with the same arguments
 * (a local group makes the per-rank calls itself).
 */
#include "rtb_internal.h"

#include <nccl.h> /* types and prototypes only: the library is bound at run time, see nccl_api() */

#include <dlfcn.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <thread>
#include <vector>

static_assert(RTB_UNIQUE_ID_BYTES == sizeof(ncclUniqueId), "rtb200.h: RTB_UNIQUE_ID_BYTES must be sizeof(ncclUniqueId)");

/* NCCL is bound with dlopen on first use, not at link time, for two reasons: single-GPU callers need no
 * NCCL at all, and a process may already hold a libnccl.so.2 (PyTorch bundles its own, newer than the
 * system's): a link-time dependency would pull the system copy in first and break the later
 * `import torch` (same soname, missing symbols).  Order: $RTB_NCCL_LIB, a copy already loaded in the
 * process, then the system's libnccl.so.2.  Only entry points that exist since NCCL 2.4 are used. */
namespace
{
struct NcclApi
{
  decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
  decltype(&ncclCommInitRank) CommInitRank = nullptr;
  decltype(&ncclCommInitAll) CommInitAll = nullptr;
  decltype(&ncclCommDestroy) CommDestroy = nullptr;
  decltype(&ncclAllGather) AllGather = nullptr;
  decltype(&ncclAllReduce) AllReduce = nullptr;
  decltype(&ncclReduce) Reduce = nullptr;
  decltype(&ncclGroupStart) GroupStart = nullptr;
  decltype(&ncclGroupEnd) GroupEnd = nullptr;
  decltype(&ncclGetErrorString) GetErrorString = nullptr;
  bool ok = false;
  std::string error;
};

const NcclApi &nccl_api()
{
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, []() {
    void *h = nullptr;
    if (const char *path = getenv("RTB_NCCL_LIB"))
      h = dlopen(path, RTLD_NOW | RTLD_GLOBAL);
    if (!h)
      h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL | RTLD_NOLOAD);
    if (!h)
      h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h)
    {
      api.error = std::string("libnccl.so.2 not found: ") + dlerror();
      return;
    }
    bool all = true;
    auto bind = [&](auto &fn, const char *name) {
      fn = reinterpret_cast<std::remove_reference_t<decltype(fn)>>(dlsym(h, name));
      if (!fn)
      {
        all = false;
        api.error = std::string("libnccl.so.2 lacks ") + name;
      }
    };
    bind(api.GetUniqueId, "ncclGetUniqueId");
    bind(api.CommInitRank, "ncclCommInitRank");
    bind(api.CommInitAll, "ncclCommInitAll");
    bind(api.CommDestroy, "ncclCommDestroy");
    bind(api.AllGather, "ncclAllGather");
    bind(api.AllReduce, "ncclAllReduce");
    bind(api.Reduce, "ncclReduce");
    bind(api.GroupStart, "ncclGroupStart");
    bind(api.GroupEnd, "ncclGroupEnd");
    bind(api.GetErrorString, "ncclGetErrorString");
    api.ok = all;
  });
  return api;
}
} // namespace

#define RTB_NEED_NCCL()                                                                        \
  do                                                                                           \
  {                                                                                            \
    if (!nccl_api().ok)                                                                        \
    {                                                                                          \
      rtb_set_error("multi-GPU entry points need NCCL: " + nccl_api().error);                  \
      return RTB_ECUDA;                                                                        \
    }                                                                                          \
  } while (0)

#define RTB_NCCL(call)                                                                         \
  do                                                                                           \
  {                                                                                            \
    ncclResult_t r_ = (call);                                                                  \
    if (r_ != ncclSuccess)                                                                     \
    {                                                                                          \
      rtb_set_error(std::string(#call) + ": " + nccl_api().GetErrorString(r_));                       \
      return RTB_ECUDA;                                                                        \
    }                                                                                          \
  } while (0)

struct RankCtx
{
  int rank = 0, device = 0;
  ncclComm_t nccl = nullptr;
  float *d_accum = nullptr;          /* [H*W*3] this rank's sum */
  uint8_t *d_fb = nullptr;           /* [H*W*3] rank 0 only */
  unsigned long long *d_ctr = nullptr; /* 8 counters and 4 times (10 words) for the whole-job reduction */
  size_t accum_elems = 0;
};

struct rtb_comm
{
  int n_ranks = 0;
  std::vector<RankCtx> local; /* the ranks this process drives: 1 (one process per GPU) or all of them */
};

extern "C" int rtb_comm_unique_id(void *id128)
{
  if (!id128)
  {
    rtb_set_error("rtb_comm_unique_id: NULL argument");
    return RTB_EINVAL;
  }
  RTB_NEED_NCCL();
  ncclUniqueId id;
  RTB_NCCL(nccl_api().GetUniqueId(&id));
  memcpy(id128, &id, sizeof(id));
  return RTB_OK;
}

extern "C" int rtb_comm_create_rank(const void *id128, int rank, int n_ranks, int device, rtb_comm **out)
{
  if (!id128 || !out || n_ranks < 1 || rank < 0 || rank >= n_ranks)
  {
    rtb_set_error("rtb_comm_create_rank: bad argument");
    return RTB_EINVAL;
  }
  *out = nullptr;
  RTB_NEED_NCCL();
  RTB_CUDA(cudaSetDevice(device));
  ncclUniqueId id;
  memcpy(&id, id128, sizeof(id));
  RankCtx r;
  r.rank = rank;
  r.device = device;
  RTB_NCCL(nccl_api().CommInitRank(&r.nccl, n_ranks, id, rank));
  rtb_comm *c = new rtb_comm();
  c->n_ranks = n_ranks;
  c->local.push_back(r);
  *out = c;
  return RTB_OK;
}

extern "C" int rtb_comm_create_local(const int *devices_or_null, int n_devices, rtb_comm **out)
{
  if (!out || n_devices < 1)
  {
    rtb_set_error("rtb_comm_create_local: bad argument");
    return RTB_EINVAL;
  }
  *out = nullptr;
  int have = 0;
  RTB_CUDA(cudaGetDeviceCount(&have));
  if (n_devices > 1)
    RTB_NEED_NCCL();
  std::vector<int> devs(n_devices);
  for (int k = 0; k < n_devices; k++)
  {
    devs[k] = devices_or_null ? devices_or_null[k] : k;
    if (devs[k] < 0 || devs[k] >= have)
    {
      rtb_set_error("rtb_comm_create_local: device ordinal out of range (" + std::to_string(have) + " visible)");
      return RTB_EINVAL;
    }
  }
  std::vector<ncclComm_t> comms(n_devices, nullptr);
  if (n_devices > 1) /* a group of one needs no communicator: every collective below is skipped for it */
    RTB_NCCL(nccl_api().CommInitAll(comms.data(), n_devices, devs.data()));
  rtb_comm *c = new rtb_comm();
  c->n_ranks = n_devices;
  for (int k = 0; k < n_devices; k++)
  {
    RankCtx r;
    r.rank = k;
    r.device = devs[k];
    r.nccl = comms[k];
    c->local.push_back(r);
  }
  *out = c;
  return RTB_OK;
}

extern "C" int rtb_comm_size(const rtb_comm *comm) { return comm ? comm->n_ranks : 0; }
extern "C" int rtb_comm_local_ranks(const rtb_comm *comm) { return comm ? (int)comm->local.size() : 0; }

extern "C" void rtb_comm_destroy(rtb_comm *comm)
{
  if (!comm)
    return;
  for (RankCtx &r : comm->local)
  {
    cudaSetDevice(r.device);
    cudaDeviceSynchronize();
    if (r.d_accum) cudaFree(r.d_accum);
    if (r.d_fb) cudaFree(r.d_fb);
    if (r.d_ctr) cudaFree(r.d_ctr);
    if (r.nccl && nccl_api().ok) nccl_api().CommDestroy(r.nccl);
  }
  delete comm;
}

/* rtb_scene.cu calls this in the middle of a sharded build */
int rtb_shard_allgather(const rtb_scene_shard *shard, void *prims, size_t prim_chunk_bytes, void *box_lo, void *box_hi,
                        size_t box_chunk_bytes, void *tex_or_null, size_t tex_chunk_bytes, int *d_flags_max_or_null)
{
  ncclComm_t comm = static_cast<ncclComm_t>(shard->nccl);
  const size_t r = (size_t)shard->rank;
  auto mine = [&](void *base, size_t chunk) { return static_cast<char *>(base) + r * chunk; };
  RTB_NCCL(nccl_api().GroupStart());
  RTB_NCCL(nccl_api().AllGather(mine(prims, prim_chunk_bytes), prims, prim_chunk_bytes, ncclChar, comm, 0));
  RTB_NCCL(nccl_api().AllGather(mine(box_lo, box_chunk_bytes), box_lo, box_chunk_bytes, ncclChar, comm, 0));
  RTB_NCCL(nccl_api().AllGather(mine(box_hi, box_chunk_bytes), box_hi, box_chunk_bytes, ncclChar, comm, 0));
  if (tex_or_null)
    RTB_NCCL(nccl_api().AllGather(mine(tex_or_null, tex_chunk_bytes), tex_or_null, tex_chunk_bytes, ncclChar, comm, 0));
  if (d_flags_max_or_null)
    RTB_NCCL(nccl_api().AllReduce(d_flags_max_or_null, d_flags_max_or_null, 2, ncclInt32, ncclMax, comm, 0));
  RTB_NCCL(nccl_api().GroupEnd());
  return RTB_OK;
}

int rtb_shard_allgather_bytes(const rtb_scene_shard *shard, void *base, size_t chunk_bytes)
{
  ncclComm_t comm = static_cast<ncclComm_t>(shard->nccl);
  RTB_NCCL(nccl_api().AllGather(static_cast<char *>(base) + (size_t)shard->rank * chunk_bytes, base, chunk_bytes, ncclChar, comm, 0));
  return RTB_OK;
}

static void shard_samples(int begin, int end, int rank, int n_ranks, int &s0, int &s1)
{
  const long long spp = (long long)end - begin;
  s0 = begin + (int)(spp * rank / n_ranks);
  s1 = begin + (int)(spp * (rank + 1) / n_ranks);
}

/* pure host arithmetic, exported so that launchers and tests can see which samples a rank renders */
extern "C" int rtb_comm_shard_samples(int sample_begin, int sample_end, int rank, int n_ranks, int *begin_out, int *end_out)
{
  if (!begin_out || !end_out || n_ranks < 1 || rank < 0 || rank >= n_ranks || sample_end < sample_begin)
  {
    rtb_set_error("rtb_comm_shard_samples: bad argument");
    return RTB_EINVAL;
  }
  shard_samples(sample_begin, sample_end, rank, n_ranks, *begin_out, *end_out);
  return RTB_OK;
}

static int ensure_buffers(RankCtx &R, size_t elems)
{
  if (R.accum_elems < elems)
  {
    if (R.d_accum) RTB_CUDA(cudaFree(R.d_accum));
    if (R.d_fb) RTB_CUDA(cudaFree(R.d_fb));
    R.d_accum = nullptr;
    R.d_fb = nullptr;
    R.accum_elems = 0;
    RTB_CUDA(cudaMalloc(reinterpret_cast<void **>(&R.d_accum), sizeof(float) * elems));
    if (R.rank == 0)
      RTB_CUDA(cudaMalloc(reinterpret_cast<void **>(&R.d_fb), elems));
    R.accum_elems = elems;
  }
  if (!R.d_ctr)
    RTB_CUDA(cudaMalloc(reinterpret_cast<void **>(&R.d_ctr), sizeof(unsigned long long) * 10));
  return RTB_OK;
}

/* ---- one rank's part of the collectives ------------------------------------------------------ */

static int rank_scene_create(RankCtx &R, int n_ranks, const void *objects, size_t n_objects, int kind, unsigned flags,
                             rtb_scene **out)
{
  RTB_CUDA(cudaSetDevice(R.device));
  rtb_scene_shard sh = { R.rank, n_ranks, R.nccl };
  return rtb_scene_create_sharded(objects, n_objects, kind, R.device, flags, &sh, out);
}

/* accumulate this rank's share of [desc->sample_begin, desc->sample_end), reduce to rank 0, tonemap there.
 * Device-resident: rank 0's d_fb_out / d_accum_out (optional) receive the frame.  Asynchronous on the
 * legacy default stream unless `counters` is given. */
static int rank_render_reduce(RankCtx &R, int n_ranks, rtb_scene *scene, const double *camera12,
                              const rtb_render_desc *desc, uint8_t *d_fb_out, rtb_counters *counters)
{
  RTB_CUDA(cudaSetDevice(R.device));
  const size_t elems = (size_t)3 * desc->width * desc->height;
  int rc = ensure_buffers(R, elems);
  if (rc != RTB_OK)
    return rc;
  rtb_render_desc d = *desc;
  shard_samples(desc->sample_begin, desc->sample_end, R.rank, n_ranks, d.sample_begin, d.sample_end);
  rtb_counters mine;
  rc = rtb_render_accum(scene, camera12, &d, R.d_accum, nullptr, counters ? &mine : nullptr);
  if (rc != RTB_OK)
    return rc;
  /* the ONE collective of the data path: per-GPU float sums -> rank 0 */
  if (n_ranks > 1)
    RTB_NCCL(nccl_api().Reduce(R.d_accum, R.d_accum, elems, ncclFloat32, ncclSum, 0, R.nccl, 0));
  const int total = desc->sample_end - desc->sample_begin;
  if (R.rank == 0)
  {
    rc = rtb_tonemap(R.d_accum, desc->width, desc->height, total > 0 ? total : 1, d_fb_out ? d_fb_out : R.d_fb, R.device, nullptr);
    if (rc != RTB_OK)
      return rc;
  }
  if (counters)
  {
    /* whole-job counters: sums over ranks (times: the slowest rank) */
    unsigned long long h[8] = { mine.rays, mine.rays_intersected, mine.prim_tests, mine.node_visits, mine.paths,
                                mine.launches + (R.rank == 0 ? 1ull : 0ull), mine.shadow_rays, mine.shadow_hits };
    float t[4] = { mine.gpu_ms, mine.trace_ms, mine.shade_ms, mine.build_ms };
    if (n_ranks > 1)
    {
      float *d_t = reinterpret_cast<float *>(R.d_ctr + 8);
      RTB_CUDA(cudaMemcpyAsync(R.d_ctr, h, sizeof(unsigned long long) * 8, cudaMemcpyHostToDevice, 0));
      RTB_CUDA(cudaMemcpyAsync(d_t, t, sizeof(t), cudaMemcpyHostToDevice, 0));
      RTB_NCCL(nccl_api().GroupStart());
      RTB_NCCL(nccl_api().AllReduce(R.d_ctr, R.d_ctr, 8, ncclUint64, ncclSum, R.nccl, 0));
      RTB_NCCL(nccl_api().AllReduce(d_t, d_t, 4, ncclFloat32, ncclMax, R.nccl, 0));
      RTB_NCCL(nccl_api().GroupEnd());
      RTB_CUDA(cudaMemcpyAsync(h, R.d_ctr, sizeof(unsigned long long) * 8, cudaMemcpyDeviceToHost, 0));
      RTB_CUDA(cudaMemcpyAsync(t, d_t, sizeof(t), cudaMemcpyDeviceToHost, 0));
      RTB_CUDA(cudaStreamSynchronize(0));
    }
    memset(counters, 0, sizeof(*counters));
    counters->rays = h[0];
    counters->rays_intersected = h[1];
    counters->prim_tests = h[2];
    counters->node_visits = h[3];
    counters->paths = h[4];
    counters->launches = h[5];
    counters->gpu_ms = t[0];
    counters->trace_ms = t[1];
    counters->shade_ms = t[2];
    counters->build_ms = t[3];
    counters->trace_launches = mine.trace_launches;
    counters->shadow_rays = h[6];
    counters->shadow_hits = h[7];
  }
  return RTB_OK;
}

/* whole render() with host buffers on one rank */
static int rank_render_host(RankCtx &R, int n_ranks, const void *objects, size_t n_objects, int kind,
                            const double *camera12, const rtb_render_desc *desc, uint8_t *framebuffer,
                            float *accum_or_null, rtb_counters *counters)
{
  rtb_scene *scene = nullptr;
  const bool timing = getenv("RTB_TIMING") != nullptr; /* development aid: where an end-to-end call spends its time */
  auto now = []() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t0 = now();
  int rc = rank_scene_create(R, n_ranks, objects, n_objects, kind, 0u, &scene);
  if (rc != RTB_OK)
    return rc;
  const double t1 = now();
  rc = rank_render_reduce(R, n_ranks, scene, camera12, desc, nullptr, counters);
  const double t2 = now();
  if (rc == RTB_OK)
  {
    const size_t elems = (size_t)3 * desc->width * desc->height;
    cudaError_t e = cudaSuccess;
    if (R.rank == 0)
    {
      e = cudaMemcpy(framebuffer, R.d_fb, elems, cudaMemcpyDeviceToHost);
      if (e == cudaSuccess && accum_or_null)
        e = cudaMemcpy(accum_or_null, R.d_accum, sizeof(float) * elems, cudaMemcpyDeviceToHost);
    }
    else
      e = cudaStreamSynchronize(0);
    if (e != cudaSuccess)
    {
      rtb_set_error(std::string("rtb_render_multi: ") + cudaGetErrorString(e));
      rc = RTB_ECUDA;
    }
  }
  const double t3 = now();
  rtb_scene_destroy(scene);
  if (timing)
    fprintf(stderr, "rtb_render_multi rank %d: scene %.2f ms, launch %.2f ms, wait + read-back %.2f ms, destroy %.2f ms\n", R.rank,
            t1 - t0, t2 - t1, t3 - t2, now() - t3);
  return rc;
}

/* run f(rank ctx) for every local rank: inline for one, one host thread per GPU otherwise (the
 * collectives inside need all ranks in flight at once) */
template <class F>
static int for_local_ranks(rtb_comm *comm, F f)
{
  if (comm->local.size() == 1)
    return f(comm->local[0], 0);
  std::vector<int> rc(comm->local.size(), RTB_OK);
  std::vector<std::string> err(comm->local.size());
  std::vector<std::thread> th;
  for (size_t k = 0; k < comm->local.size(); k++)
    th.emplace_back([&, k]() {
      rc[k] = f(comm->local[k], (int)k);
      if (rc[k] != RTB_OK)
        err[k] = rtb_last_error(); /* thread-local: carry it to the caller's thread */
    });
  for (std::thread &t : th)
    t.join();
  for (size_t k = 0; k < rc.size(); k++)
    if (rc[k] != RTB_OK)
    {
      rtb_set_error("rank " + std::to_string(comm->local[k].rank) + ": " + err[k]);
      return rc[k];
    }
  return RTB_OK;
}

/* ---- C ABI ------------------------------------------------------------------------------------ */

static int check_multi(rtb_comm *comm, const rtb_render_desc *desc, const char *who)
{
  if (!comm || !desc)
  {
    rtb_set_error(std::string(who) + ": NULL argument");
    return RTB_EINVAL;
  }
  return RTB_OK;
}

extern "C" int rtb_comm_scene_create(rtb_comm *comm, const void *objects, size_t n_objects, int record_bytes,
                                     unsigned flags, rtb_scene **scenes_out)
{
  if (!comm || !scenes_out)
  {
    rtb_set_error("rtb_comm_scene_create: NULL argument");
    return RTB_EINVAL;
  }
  for (size_t k = 0; k < comm->local.size(); k++)
    scenes_out[k] = nullptr;
  int rc = for_local_ranks(comm, [&](RankCtx &R, int k) {
    return rank_scene_create(R, comm->n_ranks, objects, n_objects, record_bytes, flags, &scenes_out[k]);
  });
  if (rc != RTB_OK)
    for (size_t k = 0; k < comm->local.size(); k++)
    {
      rtb_scene_destroy(scenes_out[k]);
      scenes_out[k] = nullptr;
    }
  return rc;
}

extern "C" int rtb_comm_render(rtb_comm *comm, rtb_scene *const *scenes, const double *camera12,
                               const rtb_render_desc *desc, uint8_t *d_fb_root, rtb_counters *counters)
{
  int rc = check_multi(comm, desc, "rtb_comm_render");
  if (rc != RTB_OK)
    return rc;
  if (!scenes || !camera12)
  {
    rtb_set_error("rtb_comm_render: NULL argument");
    return RTB_EINVAL;
  }
  std::vector<rtb_counters> per(comm->local.size());
  rc = for_local_ranks(comm, [&](RankCtx &R, int k) {
    return rank_render_reduce(R, comm->n_ranks, scenes[k], camera12, desc, R.rank == 0 ? d_fb_root : nullptr,
                              counters ? &per[k] : nullptr);
  });
  if (rc == RTB_OK && counters)
    *counters = per[0]; /* already whole-job on every rank */
  return rc;
}

extern "C" int rtb_render_multi(rtb_comm *comm, const void *objects, size_t n_objects, int record_bytes,
                                const double *camera12, const rtb_render_desc *desc, uint8_t *framebuffer,
                                float *accum_or_null, rtb_counters *counters)
{
  int rc = check_multi(comm, desc, "rtb_render_multi");
  if (rc != RTB_OK)
    return rc;
  if (!camera12 || (n_objects && !objects))
  {
    rtb_set_error("rtb_render_multi: NULL argument");
    return RTB_EINVAL;
  }
  bool has_root = false;
  for (const RankCtx &r : comm->local)
    has_root = has_root || r.rank == 0;
  if (has_root && !framebuffer)
  {
    rtb_set_error("rtb_render_multi: rank 0 needs a framebuffer");
    return RTB_EINVAL;
  }
  std::vector<rtb_counters> per(comm->local.size());
  rc = for_local_ranks(comm, [&](RankCtx &R, int k) {
    return rank_render_host(R, comm->n_ranks, objects, n_objects, record_bytes, camera12, desc, framebuffer,
                            accum_or_null, counters ? &per[k] : nullptr);
  });
  if (rc == RTB_OK && counters)
    *counters = per[0];
  return rc;
}
