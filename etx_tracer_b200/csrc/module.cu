// module.cu — C ABI (include/etx_b200.h) over the wavefront kernels: context, scene upload, iteration driver.
// Host-side counterpart of CPUVCMImpl (sources/etx/rt/integrators/vcm_cpu.cxx:30-241) and of
// Raytracing::commit_changes (sources/etx/rt/rt.cxx:58-88).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <mutex>
#include <thread>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <deque>
#include <string>
#include <vector>

#include <dlfcn.h>
#include <nccl.h>

#include "bvh_build.h"
#include "kernels.cuh"
#include "kernels_pt.cuh"

using namespace etxb;

#if defined(ETXB_PARITY) && ETXB_PARITY
static const char* kFlavor = "parity";
#else
static const char* kFlavor = "fast";
#endif

namespace {

enum KernelId : uint32_t {
  K_LIGHT_BEGIN,
  K_TRACE_LIGHT,
  K_LIGHT_BOUNCE,
  K_LV_SCAN,
  K_LV_REORDER,
  K_GRID_BBOX,
  K_GRID_KEYS,
  K_GRID_SORT,
  K_GRID_BUILD,
  K_CAMERA_BEGIN,
  K_TRACE_CAMERA,
  K_CAMERA_SHADE,
  K_CAMERA_CONNECT,
  K_SHADOW_TRACE,
  K_QUEUE_SORT,
  K_CAMERA_MERGE_SORT,
  K_CAMERA_MERGE,
  K_CAMERA_MERGE_SERIAL,
  K_CAMERA_CONTINUE,
  K_FILM_COMMIT,
  K_COMM_LIGHT_IMAGE,
  K_COMM_PHOTONS,
  K_PT_BEGIN,
  K_PT_SHADE,
  K_PT_ACCUMULATE,
  K_FILM_NOISE,
  K_COUNT
};
const char* kKernelNames[K_COUNT] = {"light_begin", "trace_closest(light)", "light_bounce", "lv_scan", "lv_reorder", "grid_bbox", "grid_keys", "grid_sort", "grid_build",
  "camera_begin", "trace_closest(camera)", "camera_shade", "camera_connect", "shadow_trace", "queue_sort", "camera_merge_sort", "camera_merge", "camera_merge_generic", "camera_continue", "film_commit_light", "nccl_allreduce_light_image", "nccl_allgather_photons",
  "pt_begin", "pt_shade", "pt_accumulate", "film_noise_levels"};

template <class T>
struct DevBuf {
  T* ptr = nullptr;
  size_t count = 0;
  cudaError_t alloc(size_t n) {
    release();
    count = n;
    if (n == 0) return cudaSuccess;
    return cudaMalloc(&ptr, n * sizeof(T));
  }
  void release() {
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    count = 0;
  }
  size_t bytes() const { return count * sizeof(T); }
};

struct TimedLaunch {
  uint32_t kernel;
  cudaEvent_t start, stop;
};

}  // namespace

struct etxb_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  std::string error;
  bool scene_ready = false;
  bool spectral = false;
  bool profile = false;
  bool has_stochastic_merge = false;  // some material that can be merged at is not Lambert (needs the serial gather)
  bool plain_scene = false;           // set at upload: no media / Boundary surfaces / subsurface, so the bounce kernels take their specialised instantiation
  bool opaque_scene = false;          // set at upload: no alpha test can reject a hit (every opacity 1, no alpha images), no Boundary surfaces / media

  // scene in HBM
  DevBuf<DVertex> vertices;
  DevBuf<DTriangle> triangles;
  DevBuf<uint32_t> tri_emitter;
  DevBuf<etxb_material> materials;
  DevBuf<etxb_emitter_profile> profiles;
  DevBuf<etxb_emitter> emitters;
  DevBuf<DSpectrum> spectra;
  DevBuf<DImage> images;
  DevBuf<DMedium> mediums;
  std::vector<DevBuf<float>> medium_density;
  std::vector<DevBuf<uint8_t>> image_pixels, image_dists;
  DevBuf<etxb_distribution_entry> emitter_dist;
  DevBuf<BvhNode> bvh_nodes;
  DevBuf<WideNode> wide_nodes;
  bool debug_trace_wide = false;      // etxb_debug_select_tree: etxb_debug_trace walks the 4-wide tree when the scene has one
  DevBuf<float4> bvh_tris;
  DevBuf<float> xyz_table, rgb_response_table;
  DevBuf<uint8_t> bn_sobol, bn_scrambling, bn_ranking;
  float y_integral = 0.0f;
  DeviceScene dscene = {};
  double bvh_build_seconds = 0.0;

  // per-path state + queues
  uint32_t width = 0, height = 0, path_count = 0;
  DevBuf<float4> ray_o, ray_d, thr, mis, hit, gathered, merged, camera_value, bs_weight_pdf, bs_wo_eta;
  DevBuf<uint4> misc;
  DevBuf<uint2> bs_props;
  DevBuf<float> wavelength;
  DevBuf<uint32_t> queue_sorted, queue_keys, queue_keys_sorted;  // path queue grouped by hit material (scenes with stochastic BSDFs)
  DevBuf<uint2> conn_list_sorted;
  DevBuf<uint32_t> lv_count, lp_offset, queue_a, queue_b, queue_counts, sampler_end_light, sampler_end_camera, merge_key, conn_seed, conn_count;
  DevBuf<uint2> conn_list, shadow_span;
  DevBuf<float4> shadow_p0, shadow_p1, shadow_value;
  DevBuf<uint32_t> shadow_result, shadow_count, trace_cursor;
  // light vertices + grid
  uint32_t lv_capacity = 0, max_light_vertices_cfg = 0;
  DevBuf<LightVertexRec> lv_tmp, lv_final;
  DevBuf<uint32_t> lv_tmp_count, overflow, grid_bbox, keys_in, keys_out, vals_in, vals_out;
  DevBuf<uint2> cell_range;
  DevBuf<float4> g_pos, g_nrm, g_win, g_thr;
  DevBuf<uint8_t> cub_temp;
  DevBuf<DeviceCounters> counters;
  // film
  DevBuf<float4> film_camera, film_light, film_light_iteration, film_out;

  // unidirectional path tracer (SURVEY 8(f) N3): the same context renders with CPUPathTracing's algorithm once etxb_set_integrator selects it
  uint32_t integrator = ETXB_INTEGRATOR_VCM;
  etxb_pt_options pt_options = {1u, 1u, 1u, 1u};
  DevBuf<float4> film_normals, film_albedo, film_adaptive;  // Film's Normals / Albedo / CameraAdaptive layers (allocated with the first PT run)
  DevBuf<uint32_t> film_ldr;                                 // the tone-mapped RGBA8 frame of etxb_read_film_ldr
  DevBuf<uint32_t> pt_info, pt_info_next, pt_stats;          // InternalData (sample count, converged, tmp); [converged this pass, error sum bits]
  DevBuf<float> pt_error;
  uint32_t pixel_sampler_image = 0xffffffffu;
  float pixel_sampler_radius = 1.0f, noise_threshold = 0.0f, radiance_clamp = 0.0f;
  uint32_t scene_samples = 0;
  uint32_t pt_pixels_processed = 0, pt_active_pixels = 0;  // active pixels of the last iteration; Film::active_pixel_count
  float pt_noise_level = 0.0f;                             // Film::noise_level

  etxb_vcm_options options = {};
  uint32_t iteration = 0;            // absolute iteration index (VCMIteration::iteration)
  uint32_t iteration_stride = 1;     // etxb_set_iteration_stride: this context renders iterations first, first + stride, ...
  uint32_t completed = 0;            // iterations finished since etxb_begin
  uint32_t rank = 0, world = 1;
  bool light_full = false;           // camera-split iterations (etxb_group replicas): the partition applies to the camera pass only, the light pass traces every path
  uint32_t last_light_vertices = 0;
  uint32_t overflow_flag = 0;
  double last_iteration_time = 0.0, total_time = 0.0;
  uint64_t kernel_launches = 0;
  GridData grid = {};
  bool light_pass_done = false, grid_done = false;

  // pixel-tile sharding across processes (one per GPU): NCCL communicator over NVLink, created by etxb_comm_init
  ncclComm_t comm = nullptr;
  cudaStream_t comm_stream = nullptr;  // highest priority: a collective's few CTAs start as soon as ANY slot frees up instead of queueing behind the
                                       // tens of thousands of blocks of another lane's kernel (measured, 2 GPUs x 4 lanes: 43 ms per all-reduce waiting otherwise)
  cudaEvent_t comm_ev_in = nullptr, comm_ev_out = nullptr;
  DevBuf<uint32_t> comm_counts;   // [world] stored light vertices per rank (all-gathered every iteration)
  DevBuf<float4> film_reduced;    // rank 0: sum of every rank's camera tiles (etxb_comm_reduce_film)
  double comm_ms = 0.0;           // device time of the collectives of the iterations since etxb_begin

  // etxb_enqueue_iteration is asynchronous (CPUVCM::update returns at once, vcm_cpu.cxx:264-276): the iteration's host loop — it reads queue
  // sizes back between bounces — runs on this context's own worker thread; etxb_poll never blocks, etxb_wait drains
  std::thread worker;
  std::mutex worker_m;
  std::condition_variable worker_cv, worker_idle;
  uint32_t worker_queued = 0;
  bool worker_busy = false, worker_quit = false;
  int worker_error = ETXB_OK;

  cudaEvent_t ev_iter_start = nullptr, ev_iter_stop = nullptr;
  std::vector<TimedLaunch> timed;
  std::vector<cudaEvent_t> event_pool;
  size_t event_cursor = 0;
  float kernel_ms[K_COUNT] = {};
  uint32_t kernel_count[K_COUNT] = {};
};

namespace {

// NCCL is bound at run time: a single-GPU host needs no libnccl, and a torch host that already loaded its bundled libnccl.so.2 shares it.
struct NcclApi {
  void* handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Reduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
NcclApi* nccl_api() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return;
    bool ok = true;
    auto bind = [&](auto& fn, const char* name) {
      fn = reinterpret_cast<std::remove_reference_t<decltype(fn)>>(dlsym(h, name));
      ok = ok && (fn != nullptr);
    };
    bind(api.GetUniqueId, "ncclGetUniqueId");
    bind(api.CommInitRank, "ncclCommInitRank");
    bind(api.CommDestroy, "ncclCommDestroy");
    bind(api.AllReduce, "ncclAllReduce");
    bind(api.AllGather, "ncclAllGather");
    bind(api.Reduce, "ncclReduce");
    bind(api.Broadcast, "ncclBroadcast");
    bind(api.GroupStart, "ncclGroupStart");
    bind(api.GroupEnd, "ncclGroupEnd");
    bind(api.GetErrorString, "ncclGetErrorString");
    if (ok) api.handle = h;
  });
  return api.handle ? &api : nullptr;
}

int ctx_drain_impl(etxb_ctx* ctx);

int fail(etxb_ctx* ctx, int code, const char* fmt, ...) {
  char buf[1024];
  va_list args;
  va_start(args, fmt);
  vsnprintf(buf, sizeof(buf), fmt, args);
  va_end(args);
  if (ctx) ctx->error = buf;
  return code;
}

#define CUDA_OK(ctx, call)                                                                                   \
  do {                                                                                                       \
    cudaError_t err__ = (call);                                                                              \
    if (err__ != cudaSuccess) {                                                                              \
      return fail(ctx, (err__ == cudaErrorMemoryAllocation) ? ETXB_ERR_OUT_OF_MEMORY : ETXB_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(err__), \
        __FILE__, __LINE__);                                                                                 \
    }                                                                                                        \
  } while (0)

#define NCCL_OK(ctx, call)                                                                                                 \
  do {                                                                                                                     \
    ncclResult_t res__ = (call);                                                                                           \
    if (res__ != ncclSuccess) return fail(ctx, ETXB_ERR_CUDA, "%s failed: %s (%s:%d)", #call, nccl_api()->GetErrorString(res__), __FILE__, __LINE__); \
  } while (0)

template <class T>
int upload(etxb_ctx* ctx, DevBuf<T>& buf, const T* host, size_t n) {
  CUDA_OK(ctx, buf.alloc(std::max<size_t>(n, 1)));
  if (n) CUDA_OK(ctx, cudaMemcpyAsync(buf.ptr, host, n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
  return ETXB_OK;
}

cudaEvent_t next_event(etxb_ctx* ctx) {
  if (ctx->event_cursor == ctx->event_pool.size()) {
    cudaEvent_t e;
    cudaEventCreate(&e);
    ctx->event_pool.push_back(e);
  }
  return ctx->event_pool[ctx->event_cursor++];
}

struct LaunchTimer {
  etxb_ctx* ctx;
  TimedLaunch t;
  LaunchTimer(etxb_ctx* c, uint32_t kernel) : ctx(c) {
    ctx->kernel_launches += 1;
    ctx->kernel_count[kernel] += 1;
    if (ctx->profile) {
      t.kernel = kernel;
      t.start = next_event(ctx);
      t.stop = next_event(ctx);
      cudaEventRecord(t.start, ctx->stream);
    }
  }
  ~LaunchTimer() {
    if (ctx->profile) {
      cudaEventRecord(t.stop, ctx->stream);
      ctx->timed.push_back(t);
    }
  }
};

bool material_class_supported_host(uint32_t cls) { return cls <= ETXB_MAT_VOID; }

// A Distribution over `size` items holds size + 1 entries (DistributionBuilder allocates the closing {0, 0, 1} entry, distribution_builder.hxx:8-14,
// 52) while `values.count` says `size` (the reference's loader) or size + 1 (hosts that count the closing entry): both are accepted, and the
// device always gets the size + 1 entries.
bool distribution_covers(uint64_t count, uint64_t size) { return (count == size) || (count == size + 1u); }

uint32_t next_pow2(uint64_t v) {
  // next_power_of_two (math.hxx:1001-1010)
  v--;
  v |= v >> 1;
  v |= v >> 2;
  v |= v >> 4;
  v |= v >> 8;
  v |= v >> 16;
  v |= v >> 32;
  v++;
  return uint32_t(v);
}

LaunchParams make_params(etxb_ctx* ctx) {
  LaunchParams p = {};
  p.scene = ctx->dscene;
  p.paths = {ctx->ray_o.ptr, ctx->ray_d.ptr, ctx->thr.ptr, ctx->mis.ptr, ctx->misc.ptr, ctx->hit.ptr, ctx->gathered.ptr, ctx->merged.ptr, ctx->wavelength.ptr,
    ctx->lv_count.ptr, ctx->bs_weight_pdf.ptr, ctx->bs_wo_eta.ptr, ctx->bs_props.ptr, ctx->merge_key.ptr, ctx->conn_seed.ptr};
  p.film = {ctx->film_camera.ptr, ctx->film_light.ptr, ctx->film_light_iteration.ptr, ctx->width, ctx->height};
  p.grid = ctx->grid;
  p.lv_tmp = ctx->lv_tmp.ptr;
  p.lv_final = ctx->lv_final.ptr;
  p.lv_tmp_count = ctx->lv_tmp_count.ptr;
  p.lv_capacity = ctx->lv_capacity;
  p.lp_offset = ctx->lp_offset.ptr;
  p.overflow = ctx->overflow.ptr;
  p.counters = ctx->counters.ptr;
  p.sampler_end_light = ctx->sampler_end_light.ptr;
  p.sampler_end_camera = ctx->sampler_end_camera.ptr;
  p.camera_value = ctx->camera_value.ptr;
  p.path_count = ctx->path_count;
  p.rank = ctx->rank;
  p.world = ctx->world;
  p.light_world = ctx->light_full ? 1u : ctx->world;
  p.camera_sample_index = ctx->completed;
  p.conn_list = ctx->conn_list.ptr;
  p.conn_count = ctx->conn_count.ptr;
  p.conn_capacity = ctx->lv_capacity;
  p.conn_key = (ctx->has_stochastic_merge && ctx->conn_list_sorted.count) ? ctx->keys_in.ptr : nullptr;  // keys_in / vals_in are free after the grid build
  p.paths.shadow_span = ctx->shadow_span.ptr;
  p.shadow_p0 = ctx->shadow_p0.ptr;
  p.shadow_p1 = ctx->shadow_p1.ptr;
  p.shadow_value = ctx->shadow_value.ptr;
  p.shadow_result = ctx->shadow_result.ptr;
  p.shadow_count = ctx->shadow_count.ptr;
  p.shadow_capacity = uint32_t(ctx->shadow_p0.count);
  p.shadow_stage = (ctx->dscene.deferred_shadow_rays && ctx->shadow_p0.count) ? 1u : 0u;
#if defined(ETXB_PARITY) && ETXB_PARITY
  p.shadow_atomic = 0;
#else
  p.shadow_atomic = (!p.shadow_stage && ctx->opaque_scene && ctx->plain_scene && ctx->has_stochastic_merge && ctx->shadow_p0.count) ? 1u : 0u;
#endif
  p.merge_material_major = ctx->has_stochastic_merge ? 1u : 0u;
#if defined(ETXB_PARITY) && ETXB_PARITY
  p.connect_stage = 0;
#else
  p.connect_stage = ctx->has_stochastic_merge ? 1u : 0u;
#endif
  // start_next_iteration (vcm_cpu.cxx:95-113)
  VcmParams& v = p.vcm;
  v.options = ctx->options.options;
  v.kernel = ctx->options.kernel;
  v.blue_noise = (ctx->options.blue_noise != 0) && ctx->dscene.has_blue_noise;
  v.iteration = ctx->iteration;
  float used_radius = ctx->options.initial_radius;
  if (used_radius == 0.0f) {
    uint32_t max_dim = std::max(ctx->width, ctx->height);
    used_radius = 5.0f * ctx->dscene.bounding_sphere_radius / float(max_dim);
  }
  float radius_scale = 1.0f / (1.0f + float(ctx->iteration) / float(ctx->options.radius_decay));
  v.current_radius = used_radius * radius_scale;
  float eta_vcm = kPi * (v.current_radius * v.current_radius) * float(ctx->path_count);
  v.vc_weight = 1.0f / eta_vcm;
  v.vm_weight = (ctx->options.options & ETXB_VCM_ENABLE_MERGING) ? eta_vcm : 0.0f;
  v.vm_normalization = 1.0f / eta_vcm;
  return p;
}

uint32_t blocks_for(uint32_t n, uint32_t block) { return (n + block - 1u) / block; }
constexpr uint32_t kMergeSortMinQueries = 16384u;  // below this the merge queries are not sorted
constexpr uint32_t kMergeMinWarps = 148u * 32u;    // the merge wants at least this many warps in flight (148 SMs)

int read_u32(etxb_ctx* ctx, const uint32_t* dptr, uint32_t& out) {
  CUDA_OK(ctx, cudaMemcpyAsync(&out, dptr, 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  return ETXB_OK;
}

// Size of the next bounce's queue.  A long queue is read back every bounce (the grids are sized by it).  In the tail of a pass the
// queue only shrinks and every kernel guards on the device-side count, so the previous size stays a valid upper bound for the launch
// grids: the host then enqueues several bounces back to back and reads the count only every kTailBatch bounces.
constexpr uint32_t kTailQueue = 8192u;
constexpr uint32_t kTailBatch = 4u;
int next_queue_size(etxb_ctx* ctx, const uint32_t* dptr, uint32_t& active, uint32_t& unsynced) {
  if ((active < kTailQueue) && (unsynced + 1u < kTailBatch)) {
    unsynced += 1u;
    return ETXB_OK;
  }
  unsynced = 0;
  return read_u32(ctx, dptr, active);
}

// Scenes with stochastic BSDFs: the bounce kernels spend their time in the BSDF class of the surface that was hit, and a warp that holds
// several classes runs them one after the other.  k_trace_closest leaves one key per queue slot (material index; 0xff = miss; 0x100 = slot
// past the device-side count); a stable 9-bit radix sort groups the queue, slots past the count stay at the end.  Returns the queue the
// rest of the bounce must use.  Short queues (the tail of a pass) are latency bound and skip it.
constexpr uint32_t kSortQueueMin = 1024u;
inline bool sorts_queue(const etxb_ctx* ctx, uint32_t active) { return ctx->has_stochastic_merge && (active >= kSortQueueMin) && ctx->queue_sorted.count; }
int sort_queue_by_material(etxb_ctx* ctx, const uint32_t* queue, uint32_t active, const uint32_t** sorted) {
  size_t temp_bytes = ctx->cub_temp.bytes();
  CUDA_OK(ctx, cub::DeviceRadixSort::SortPairs(ctx->cub_temp.ptr, temp_bytes, ctx->queue_keys.ptr, ctx->queue_keys_sorted.ptr, queue, ctx->queue_sorted.ptr, int(active), 0, 9,
                 ctx->stream));
  *sorted = ctx->queue_sorted.ptr;
  return ETXB_OK;
}

// closest hits of a queue, one ray per thread.  The persistent, nodelet-staged, lane-refilled walk that the shadow segments take (2-3x as many
// rays, from one list) lost here on the B200 (C3, round 2: 27.1 against 22.9 ms per iteration): one ray per path leaves little to refill from.
void launch_trace_closest(etxb_ctx* ctx, const LaunchParams& p, const uint32_t* queue, const uint32_t* count, uint32_t* keys, uint32_t active) {
  if (p.scene.wide_nodes != nullptr) {
    k_trace_closest_wide<<<blocks_for(active, 256), 256, 0, ctx->stream>>>(p, queue, count, keys, active);
  } else {
    k_trace_closest<<<blocks_for(active, 256), 256, 0, ctx->stream>>>(p, queue, count, keys, active);
  }
}
// the bounce's shadow segments (ShadowBatch, atomic mode): traced and added to their targets
int launch_shadow_resolve(etxb_ctx* ctx, const LaunchParams& p, uint32_t active) {
  CUDA_OK(ctx, cudaMemsetAsync(ctx->trace_cursor.ptr, 0, 4, ctx->stream));
  const uint32_t blocks = std::min<uint32_t>(blocks_for(std::min<uint64_t>(uint64_t(active) * 4ull, 0x7fffffffull), kTraversalBlock), 148u);
  if (p.scene.wide_nodes != nullptr) {
    k_shadow_resolve<true><<<blocks, kTraversalBlock, 0, ctx->stream>>>(p, ctx->trace_cursor.ptr);
  } else {
    k_shadow_resolve<false><<<blocks, kTraversalBlock, 0, ctx->stream>>>(p, ctx->trace_cursor.ptr);
  }
  return ETXB_OK;
}

template <bool SP>
int run_light_pass(etxb_ctx* ctx) {
  LaunchParams p = make_params(ctx);
  uint32_t* counts = ctx->queue_counts.ptr;  // [0] = current, [1] = next
  CUDA_OK(ctx, cudaMemsetAsync(counts, 0, 8, ctx->stream));
  CUDA_OK(ctx, cudaMemsetAsync(ctx->lv_tmp_count.ptr, 0, 4, ctx->stream));
  uint32_t* qin = ctx->queue_a.ptr;
  uint32_t* qout = ctx->queue_b.ptr;
  {
    LaunchTimer t(ctx, K_LIGHT_BEGIN);
    k_light_begin<SP><<<blocks_for(ctx->path_count, 128), 128, 0, ctx->stream>>>(p, qin, counts + 0);
  }
  uint32_t active = 0;
  if (int rc = read_u32(ctx, counts + 0, active)) return rc;
  uint32_t cur = 0, unsynced = 0;
  while (active > 0) {
    const bool sorted = sorts_queue(ctx, active);
    const uint32_t* q = qin;
    {
      LaunchTimer t(ctx, K_TRACE_LIGHT);
      launch_trace_closest(ctx, p, qin, counts + cur, sorted ? ctx->queue_keys.ptr : nullptr, active);
    }
    if (sorted) {
      LaunchTimer t(ctx, K_QUEUE_SORT);
      if (int rc = sort_queue_by_material(ctx, qin, active, &q)) return rc;
    }
    CUDA_OK(ctx, cudaMemsetAsync(counts + (cur ^ 1u), 0, 4, ctx->stream));
    if (p.shadow_atomic) CUDA_OK(ctx, cudaMemsetAsync(ctx->shadow_count.ptr, 0, 8, ctx->stream));
    {
      LaunchTimer t(ctx, K_LIGHT_BOUNCE);
      if (ctx->plain_scene) {
        k_light_bounce<SP, true><<<blocks_for(active, 128), 128, 0, ctx->stream>>>(p, q, counts + cur, qout, counts + (cur ^ 1u));
      } else {
        k_light_bounce<SP, false><<<blocks_for(active, 128), 128, 0, ctx->stream>>>(p, q, counts + cur, qout, counts + (cur ^ 1u));
      }
    }
    if (p.shadow_atomic) {
      // the light-to-camera connections of this bounce: segments -> splats (light image)
      LaunchTimer t(ctx, K_SHADOW_TRACE);
      if (int rc = launch_shadow_resolve(ctx, p, active)) return rc;
    }
    cur ^= 1u;
    std::swap(qin, qout);
    if (int rc = next_queue_size(ctx, counts + cur, active, unsynced)) return rc;
  }
  CUDA_OK(ctx, cudaGetLastError());

  // path-major vertex pool: offsets = exclusive scan of per-path counts (VCMLightPath::index)
  uint32_t total = 0;
  if (int rc = read_u32(ctx, ctx->lv_tmp_count.ptr, total)) return rc;
  uint32_t ovf = 0;
  if (int rc = read_u32(ctx, ctx->overflow.ptr, ovf)) return rc;
  ctx->overflow_flag |= ovf;
  total = std::min(total, ctx->lv_capacity);
  {
    LaunchTimer t(ctx, K_LV_SCAN);
    size_t temp_bytes = ctx->cub_temp.bytes();
    CUDA_OK(ctx, cub::DeviceScan::ExclusiveSum(ctx->cub_temp.ptr, temp_bytes, ctx->lv_count.ptr, ctx->lp_offset.ptr, int(ctx->path_count), ctx->stream));
  }
  if (total > 0) {
    LaunchTimer t(ctx, K_LV_REORDER);
    k_lv_reorder<<<blocks_for(total, 256), 256, 0, ctx->stream>>>(p, total);
  }
  ctx->last_light_vertices = total;
  CUDA_OK(ctx, cudaGetLastError());
  ctx->light_pass_done = true;
  return ETXB_OK;
}

template <bool SP>
int run_grid_build(etxb_ctx* ctx, const LightVertexRec* records, uint32_t count) {
  ctx->grid = {};
  ctx->grid_done = true;
  LaunchParams p = make_params(ctx);
  {
    // complete_light_vertices -> Film::commit_light_iteration(iteration) (vcm_cpu.cxx:209-211); in a multi-GPU run the
    // host has all-reduced ETXB_BUF_FILM_LIGHT_ITERATION across ranks before this call
    LaunchTimer t(ctx, K_FILM_COMMIT);
    // the running mean counts the iterations THIS context has accumulated since etxb_begin (= the absolute index in the reference's flow,
    // which always starts at 0; after etxb_begin(ctx, k != 0) or with interleaved iterations the absolute index would scale the first
    // commit by 1/(k+1) against a cleared film)
    k_film_commit_light<<<blocks_for(ctx->path_count, 256), 256, 0, ctx->stream>>>(p.film, ctx->completed);
  }
  bool merging = (ctx->options.options & ETXB_VCM_ENABLE_MERGING) && (ctx->options.options & ETXB_VCM_MERGE_VERTICES);
  if (!merging || (count == 0)) return ETXB_OK;
  p.lv_final = const_cast<LightVertexRec*>(records);
  float radius = p.vcm.current_radius;
  uint32_t init[6];
  for (int k = 0; k < 3; ++k) {
    init[k] = 0xffffffffu;
    init[3 + k] = 0u;
  }
  CUDA_OK(ctx, cudaMemcpyAsync(ctx->grid_bbox.ptr, init, sizeof(init), cudaMemcpyHostToDevice, ctx->stream));
  {
    LaunchTimer t(ctx, K_GRID_BBOX);
    k_grid_bbox<<<std::min<uint32_t>(blocks_for(count, 256), 148u * 8u), 256, 0, ctx->stream>>>(records, count, ctx->grid_bbox.ptr);
  }
  uint32_t table_size = next_pow2(count);
  uint32_t mask = table_size - 1u;
  float cell_size = 2.0f * radius;
  {
    LaunchTimer t(ctx, K_GRID_KEYS);
    k_grid_keys<<<blocks_for(count, 256), 256, 0, ctx->stream>>>(records, count, ctx->grid_bbox.ptr, cell_size, mask, ctx->keys_in.ptr, ctx->vals_in.ptr);
  }
  {
    LaunchTimer t(ctx, K_GRID_SORT);
    size_t temp_bytes = ctx->cub_temp.bytes();
    int end_bit = 1;
    while ((1ull << end_bit) < table_size) end_bit++;
    if (ctx->dscene.medium_count) end_bit = 32;  // medium vertices carry the key 0xffffffff and must sort behind every cell
    CUDA_OK(ctx, cub::DeviceRadixSort::SortPairs(ctx->cub_temp.ptr, temp_bytes, ctx->keys_in.ptr, ctx->keys_out.ptr, ctx->vals_in.ptr, ctx->vals_out.ptr, int(count), 0,
                   end_bit, ctx->stream));
  }
  CUDA_OK(ctx, cudaMemsetAsync(ctx->cell_range.ptr, 0, size_t(table_size) * sizeof(uint2), ctx->stream));
  {
    LaunchTimer t(ctx, K_GRID_BUILD);
    k_grid_build<SP><<<blocks_for(count, 256), 256, 0, ctx->stream>>>(p, ctx->keys_out.ptr, ctx->vals_out.ptr, count, ctx->cell_range.ptr, ctx->g_pos.ptr, ctx->g_nrm.ptr,
      ctx->g_win.ptr, ctx->g_thr.ptr);
  }
  uint32_t bbox[6];
  CUDA_OK(ctx, cudaMemcpyAsync(bbox, ctx->grid_bbox.ptr, sizeof(bbox), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  GridData& g = ctx->grid;
  g.cell_range = ctx->cell_range.ptr;
  g.pos_dvcm = ctx->g_pos.ptr;
  g.nrm_dvm = ctx->g_nrm.ptr;
  g.win_len = ctx->g_win.ptr;
  g.thr_rgb = ctx->g_thr.ptr;
  g.bbox_min = {ordered_to_float(bbox[0]), ordered_to_float(bbox[1]), ordered_to_float(bbox[2])};
  g.bbox_max = {ordered_to_float(bbox[3]), ordered_to_float(bbox[4]), ordered_to_float(bbox[5])};
  g.hash_table_mask = mask;
  g.photon_count = count;
  g.cell_size = cell_size;
  g.radius_squared = radius * radius;
  g.inv_radius_squared = (g.radius_squared > 0.0f) ? 1.0f / g.radius_squared : 0.0f;
  CUDA_OK(ctx, cudaGetLastError());
  return ETXB_OK;
}

template <bool SP>
int run_camera_pass(etxb_ctx* ctx) {
  LaunchParams p = make_params(ctx);
  uint32_t* counts = ctx->queue_counts.ptr;
  CUDA_OK(ctx, cudaMemsetAsync(counts, 0, 8, ctx->stream));
  uint32_t* qin = ctx->queue_a.ptr;
  uint32_t* qout = ctx->queue_b.ptr;
  {
    LaunchTimer t(ctx, K_CAMERA_BEGIN);
    k_camera_begin<SP><<<blocks_for(ctx->path_count, 128), 128, 0, ctx->stream>>>(p, qin, counts + 0);
  }
  uint32_t active = 0;
  if (int rc = read_u32(ctx, counts + 0, active)) return rc;
  uint32_t cur = 0, unsynced = 0;
  const bool merging = (ctx->options.options & ETXB_VCM_ENABLE_MERGING) && (ctx->options.options & ETXB_VCM_MERGE_VERTICES);
  while (active > 0) {
    const bool sorted = sorts_queue(ctx, active);
    const uint32_t* q = qin;  // the queue every stage of this bounce reads
    {
      LaunchTimer t(ctx, K_TRACE_CAMERA);
      launch_trace_closest(ctx, p, qin, counts + cur, sorted ? ctx->queue_keys.ptr : nullptr, active);
    }
    if (sorted) {
      LaunchTimer t(ctx, K_QUEUE_SORT);
      if (int rc = sort_queue_by_material(ctx, qin, active, &q)) return rc;
    }
    CUDA_OK(ctx, cudaMemsetAsync(counts + (cur ^ 1u), 0, 4, ctx->stream));
    if (p.connect_stage) CUDA_OK(ctx, cudaMemsetAsync(ctx->conn_count.ptr, 0, 4, ctx->stream));
    if (p.shadow_stage || p.shadow_atomic) CUDA_OK(ctx, cudaMemsetAsync(ctx->shadow_count.ptr, 0, 8, ctx->stream));
    {
      LaunchTimer t(ctx, K_CAMERA_SHADE);
      if (ctx->plain_scene) {
        k_camera_shade<SP, true><<<blocks_for(active, 128), 128, 0, ctx->stream>>>(p, q, counts + cur);
      } else {
        k_camera_shade<SP, false><<<blocks_for(active, 128), 128, 0, ctx->stream>>>(p, q, counts + cur);
      }
    }
    if (p.shadow_stage && (ctx->options.options & ETXB_VCM_CONNECT_VERTICES)) {
      // one thread per (camera vertex, light vertex) pair of the bounce, grid-stride over the reserved shadow slots (count on the device)
      LaunchTimer t(ctx, K_CAMERA_CONNECT);
      uint32_t blocks = std::min<uint32_t>(148u * 16u, blocks_for(std::min<uint64_t>(uint64_t(active) * 8ull, 0x7fffffffull), 128));
      k_camera_connect_deferred<SP><<<blocks, 128, 0, ctx->stream>>>(p);
    }
    if (p.shadow_stage) {
      // persistent warps over the bounce's deferred shadow rays (the number of rays stays on the device)
      LaunchTimer t(ctx, K_SHADOW_TRACE);
      uint32_t blocks = std::min<uint32_t>(148u * 8u, blocks_for(std::min<uint64_t>(uint64_t(active) * 32ull, 0x7fffffffull), 256));
      k_shadow_trace<<<blocks, 256, 0, ctx->stream>>>(p);
    }
    if (p.connect_stage && (ctx->options.options & ETXB_VCM_CONNECT_VERTICES)) {
      if (active < kTailQueue) {
        // tail of the pass: the pair count stays on the device (k_camera_connect is grid-stride), no host round trip per bounce
        LaunchTimer t(ctx, K_CAMERA_CONNECT);
        const uint32_t blocks = std::min<uint32_t>(148u * 4u, blocks_for(active * 4u, 128));
        if (ctx->plain_scene) {
          k_camera_connect<SP, true><<<blocks, 128, 0, ctx->stream>>>(p, ctx->conn_list.ptr);
        } else {
          k_camera_connect<SP, false><<<blocks, 128, 0, ctx->stream>>>(p, ctx->conn_list.ptr);
        }
      } else {
        uint32_t pending = 0;
        if (int rc = read_u32(ctx, ctx->conn_count.ptr, pending)) return rc;
        pending = std::min(pending, ctx->lv_capacity);
        if (pending) {
          const uint2* list = ctx->conn_list.ptr;
          if (p.conn_key && (pending >= kSortQueueMin)) {
            // connections grouped by (camera vertex material, light vertex material): one pair of BSDF classes per warp
            LaunchTimer t(ctx, K_QUEUE_SORT);
            size_t temp_bytes = ctx->cub_temp.bytes();
            CUDA_OK(ctx, cub::DeviceRadixSort::SortPairs(ctx->cub_temp.ptr, temp_bytes, ctx->keys_in.ptr, ctx->vals_in.ptr, reinterpret_cast<const unsigned long long*>(ctx->conn_list.ptr),
                           reinterpret_cast<unsigned long long*>(ctx->conn_list_sorted.ptr), int(pending), 0, 16, ctx->stream));
            list = ctx->conn_list_sorted.ptr;
          }
          LaunchTimer t(ctx, K_CAMERA_CONNECT);
          if (ctx->plain_scene) {
            k_camera_connect<SP, true><<<blocks_for(pending, 128), 128, 0, ctx->stream>>>(p, list);
          } else {
            k_camera_connect<SP, false><<<blocks_for(pending, 128), 128, 0, ctx->stream>>>(p, list);
          }
        }
      }
    }
    if (p.shadow_atomic) {
      // emitter-sample and vertex-connection segments of this bounce: traced, the unoccluded ones added to their paths' gathered sums
      LaunchTimer t(ctx, K_SHADOW_TRACE);
      if (int rc = launch_shadow_resolve(ctx, p, active)) return rc;
    }
#if defined(ETXB_PARITY) && ETXB_PARITY
    if (merging) {
      LaunchTimer t(ctx, K_CAMERA_MERGE_SERIAL);
      k_camera_merge_serial<SP><<<blocks_for(active, 128), 128, 0, ctx->stream>>>(p, q, counts + cur);
    }
#else
    if (merging && ctx->grid.photon_count) {
      const uint32_t* ids = q;
      const uint32_t* keys = ctx->merge_key.ptr;
      if (active >= kMergeSortMinQueries) {
        // queries sorted by the Morton code of their base cell: neighbours in the queue read the same photon cells.  A short queue
        // (the tail of the pass) is latency bound, not bandwidth bound: it goes in queue order and saves the sort launches.
        LaunchTimer t(ctx, K_CAMERA_MERGE_SORT);
        size_t temp_bytes = ctx->cub_temp.bytes();
        CUDA_OK(ctx, cub::DeviceRadixSort::SortPairs(ctx->cub_temp.ptr, temp_bytes, ctx->merge_key.ptr, ctx->keys_out.ptr, q, ctx->vals_out.ptr, int(active), 0, 32,
                       ctx->stream));
        ids = ctx->vals_out.ptr;
        keys = ctx->keys_out.ptr;
      }
      // queries per warp: 32 while that still fills the machine, fewer for short queues (a warp serialises its queries)
      uint32_t qpw = 32u;
      while ((qpw > 1u) && (active / qpw < kMergeMinWarps)) qpw >>= 1;
      const uint32_t merge_blocks = blocks_for(blocks_for(active, qpw), kMergeWarpsPerBlock);
      {
        LaunchTimer t(ctx, K_CAMERA_MERGE);
        k_camera_merge_coop<SP><<<merge_blocks, kMergeWarpsPerBlock * 32, 0, ctx->stream>>>(p, ids, keys, counts + cur, qpw);
      }
      if (ctx->has_stochastic_merge) {
        LaunchTimer t(ctx, K_CAMERA_MERGE_SERIAL);
        const uint32_t closure_blocks = blocks_for(blocks_for(active, qpw), kClosureWarpsPerBlock);
        k_camera_merge_closure<SP><<<closure_blocks, kClosureWarpsPerBlock * 32, 0, ctx->stream>>>(p, ids, keys, counts + cur, qpw);
      }
    }
#endif
    {
      LaunchTimer t(ctx, K_CAMERA_CONTINUE);
      k_camera_continue<SP><<<blocks_for(active, 128), 128, 0, ctx->stream>>>(p, q, counts + cur, qout, counts + (cur ^ 1u));
    }
    cur ^= 1u;
    std::swap(qin, qout);
    if (int rc = next_queue_size(ctx, counts + cur, active, unsynced)) return rc;
  }
  CUDA_OK(ctx, cudaGetLastError());
  return ETXB_OK;
}

// Pixel-tile sharding (SURVEY 8(e), north star): between the light pass and the grid build of an iteration the ranks exchange what is global —
//   (a) the light-tracing splats land on ANY pixel (vcm_cpu.cxx:147-154): all-reduce(sum) of the per-iteration light image, after which every
//       rank commits the same running mean (film.cxx:332-343);
//   (b) merging queries the photon map of ALL light paths (vcm_cpu.cxx:219-221): all-gather of the path-major vertex records (96 B each, block
//       sizes differ per rank: counts first, then one broadcast per owner inside a group call = an uneven all-gather), into the allocation-order
//       pool, which is free once the path-major pool exists; every rank then builds the same grid.
// Camera tiles are disjoint: they meet only when a frame is wanted (etxb_comm_reduce_film).
int comm_exchange(etxb_ctx* ctx, const void** records, uint64_t* count) {
  NcclApi* n = nccl_api();
  *records = nullptr;
  *count = 0;
  // the collectives run on the context's high-priority stream, fenced against its work stream by events on both sides
  cudaStream_t cs = ctx->comm_stream;
  auto fence_out = [&]() -> cudaError_t {
    cudaError_t e = cudaEventRecord(ctx->comm_ev_out, cs);
    return (e == cudaSuccess) ? cudaStreamWaitEvent(ctx->stream, ctx->comm_ev_out, 0) : e;
  };
  {
    LaunchTimer t(ctx, K_COMM_LIGHT_IMAGE);
    CUDA_OK(ctx, cudaEventRecord(ctx->comm_ev_in, ctx->stream));
    CUDA_OK(ctx, cudaStreamWaitEvent(cs, ctx->comm_ev_in, 0));
    NCCL_OK(ctx, n->AllReduce(ctx->film_light_iteration.ptr, ctx->film_light_iteration.ptr, size_t(ctx->path_count) * 4u, ncclFloat, ncclSum, ctx->comm, cs));
    CUDA_OK(ctx, fence_out());
  }
  const bool merging = (ctx->options.options & ETXB_VCM_ENABLE_MERGING) && (ctx->options.options & ETXB_VCM_MERGE_VERTICES);
  if (!merging) return ETXB_OK;
  const uint32_t world = ctx->world, rank = ctx->rank;
  std::vector<uint32_t> counts(world, 0u);
  {
    LaunchTimer t(ctx, K_COMM_PHOTONS);
    uint32_t mine = ctx->last_light_vertices;
    CUDA_OK(ctx, cudaMemcpyAsync(ctx->comm_counts.ptr + rank, &mine, 4, cudaMemcpyHostToDevice, cs));
    NCCL_OK(ctx, n->AllGather(ctx->comm_counts.ptr + rank, ctx->comm_counts.ptr, 1, ncclUint32, ctx->comm, cs));
    CUDA_OK(ctx, cudaMemcpyAsync(counts.data(), ctx->comm_counts.ptr, size_t(world) * 4u, cudaMemcpyDeviceToHost, cs));
    CUDA_OK(ctx, cudaStreamSynchronize(cs));
    uint64_t total = 0;
    std::vector<uint64_t> offsets(world, 0u);
    for (uint32_t r = 0; r < world; ++r) {
      offsets[r] = total;
      total += counts[r];
    }
    if (total > ctx->lv_capacity) return fail(ctx, ETXB_ERR_OVERFLOW, "gathered photon count %llu exceeds the pool capacity %u", (unsigned long long)total, ctx->lv_capacity);
    constexpr size_t kRecordFloats = sizeof(LightVertexRec) / 4u;
    NCCL_OK(ctx, n->GroupStart());
    for (uint32_t r = 0; r < world; ++r) {
      if (counts[r] == 0u) continue;
      ncclResult_t res = n->Broadcast(ctx->lv_final.ptr, ctx->lv_tmp.ptr + offsets[r], size_t(counts[r]) * kRecordFloats, ncclFloat, int(r), ctx->comm, cs);
      if (res != ncclSuccess) {
        n->GroupEnd();
        return fail(ctx, ETXB_ERR_CUDA, "ncclBroadcast failed: %s", n->GetErrorString(res));
      }
    }
    NCCL_OK(ctx, n->GroupEnd());
    CUDA_OK(ctx, fence_out());
    *records = ctx->lv_tmp.ptr;
    *count = total;
  }
  return ETXB_OK;
}

void resolve_timers(etxb_ctx* ctx) {
  for (auto& t : ctx->timed) {
    float ms = 0.0f;
    if (cudaEventElapsedTime(&ms, t.start, t.stop) == cudaSuccess) ctx->kernel_ms[t.kernel] += ms;
  }
  ctx->timed.clear();
  ctx->event_cursor = 0;
}

int finish_iteration(etxb_ctx* ctx) {
  CUDA_OK(ctx, cudaEventRecord(ctx->ev_iter_stop, ctx->stream));
  CUDA_OK(ctx, cudaEventSynchronize(ctx->ev_iter_stop));
  float ms = 0.0f;
  CUDA_OK(ctx, cudaEventElapsedTime(&ms, ctx->ev_iter_start, ctx->ev_iter_stop));
  ctx->last_iteration_time = double(ms) * 1e-3;
  ctx->total_time += ctx->last_iteration_time;
  resolve_timers(ctx);
  ctx->completed += 1;
  ctx->iteration += ctx->iteration_stride;
  ctx->light_pass_done = false;
  ctx->grid_done = false;
  return ETXB_OK;
}

// ---- unidirectional path tracer (SURVEY 8(f) N3) -----------------------------------------------------------------------------------------
// The film layers and the per-pixel history only CPUPathTracing touches (film.cxx:14-40, 104-121), allocated with the first run.
int pt_ensure_film(etxb_ctx* ctx) {
  const size_t n = ctx->path_count;
  if (ctx->film_normals.count == n) return ETXB_OK;
  DevBuf<float4>* f4[] = {&ctx->film_normals, &ctx->film_albedo, &ctx->film_adaptive};
  for (auto* b : f4) {
    CUDA_OK(ctx, b->alloc(n));
    CUDA_OK(ctx, cudaMemsetAsync(b->ptr, 0, n * 16, ctx->stream));
  }
  CUDA_OK(ctx, ctx->pt_info.alloc(n));
  CUDA_OK(ctx, ctx->pt_info_next.alloc(n));
  CUDA_OK(ctx, ctx->pt_error.alloc(n));
  CUDA_OK(ctx, ctx->pt_stats.alloc(2));
  CUDA_OK(ctx, cudaMemsetAsync(ctx->pt_info.ptr, 0, n * 4, ctx->stream));
  CUDA_OK(ctx, cudaMemsetAsync(ctx->pt_error.ptr, 0, n * 4, ctx->stream));
  return ETXB_OK;
}

PtFilm make_pt_film(etxb_ctx* ctx) { return {ctx->film_normals.ptr, ctx->film_albedo.ptr, ctx->film_adaptive.ptr, ctx->pt_info.ptr, ctx->pt_error.ptr, ctx->pt_info_next.ptr}; }

// Film::estimate_noise_levels (film.cxx:233-330) after iteration `sample_index`
constexpr uint32_t kFilmMinSamples = 32u;
int pt_estimate_noise_levels(etxb_ctx* ctx, uint32_t sample_index) {
  const float threshold = ctx->noise_threshold;
  if ((threshold == 0.0f) || (sample_index < kFilmMinSamples) || ((sample_index % 2u) != 0u)) return ETXB_OK;
  LaunchTimer t(ctx, K_FILM_NOISE);
  const uint32_t n = ctx->path_count;
  FilmBuffers film = {ctx->film_camera.ptr, ctx->film_light.ptr, ctx->film_light_iteration.ptr, ctx->width, ctx->height};
  PtFilm pf = make_pt_film(ctx);
  CUDA_OK(ctx, cudaMemsetAsync(ctx->pt_stats.ptr, 0, 8, ctx->stream));
  k_film_noise_level<<<blocks_for(n, 256), 256, 0, ctx->stream>>>(film, pf, threshold, ctx->pt_stats.ptr);
  k_film_noise_rows<<<blocks_for(n, 256), 256, 0, ctx->stream>>>(film, ctx->pt_info.ptr, ctx->pt_info_next.ptr);
  k_film_noise_columns<<<blocks_for(n, 256), 256, 0, ctx->stream>>>(film, ctx->pt_info_next.ptr, ctx->pt_info.ptr);
  ctx->kernel_launches += 2;
  uint32_t stats[2] = {0u, 0u};
  CUDA_OK(ctx, cudaMemcpyAsync(stats, ctx->pt_stats.ptr, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  float total = 0.0f;
  memcpy(&total, &stats[1], 4);
  ctx->pt_active_pixels = stats[0];
  ctx->pt_noise_level = (stats[0] > 0u) ? (total / float(stats[0])) : total;
  return ETXB_OK;
}

// One CPUPathTracingImpl task (path_tracing.cxx:50-83) followed by update()'s bookkeeping (:85-110): every active pixel's path, the film update,
// the noise estimate.
template <bool SP>
int run_pt_iteration(etxb_ctx* ctx) {
  CUDA_OK(ctx, cudaEventRecord(ctx->ev_iter_start, ctx->stream));
  if (int rc = pt_ensure_film(ctx)) return rc;
  LaunchParams p = make_params(ctx);
  p.connect_stage = 0;
  p.shadow_stage = 0;  // the slot-ordered deferred shadow rays belong to the VCM camera step; the path tracer uses the atomic list or traces inline
  PtParams pt = {};
  pt.nee = ctx->pt_options.nee;
  pt.direct = ctx->pt_options.direct;
  pt.mis = ctx->pt_options.mis;
  pt.blue_noise = (ctx->pt_options.blue_noise != 0u) && ctx->dscene.has_blue_noise;
  pt.iteration = ctx->iteration;
  pt.pixel_sampler_image = ctx->pixel_sampler_image;
  pt.pixel_sampler_radius = ctx->pixel_sampler_radius;
  pt.radiance_clamp = ctx->radiance_clamp;
  PtFilm pf = make_pt_film(ctx);
  const bool plain = ctx->plain_scene;
  uint32_t* counts = ctx->queue_counts.ptr;
  CUDA_OK(ctx, cudaMemsetAsync(counts, 0, 8, ctx->stream));
  uint32_t* qin = ctx->queue_a.ptr;
  uint32_t* qout = ctx->queue_b.ptr;
  {
    LaunchTimer t(ctx, K_PT_BEGIN);
    k_pt_begin<SP><<<blocks_for(ctx->path_count, 128), 128, 0, ctx->stream>>>(p, pt, pf, qin, counts + 0);
  }
  uint32_t active = 0;
  if (int rc = read_u32(ctx, counts + 0, active)) return rc;
  ctx->pt_pixels_processed = active;
  uint32_t cur = 0, unsynced = 0;
  while (active > 0) {
    const bool sorted = sorts_queue(ctx, active);
    const uint32_t* q = qin;
    {
      LaunchTimer t(ctx, K_TRACE_CAMERA);
      launch_trace_closest(ctx, p, qin, counts + cur, sorted ? ctx->queue_keys.ptr : nullptr, active);
    }
    if (sorted) {
      LaunchTimer t(ctx, K_QUEUE_SORT);
      if (int rc = sort_queue_by_material(ctx, qin, active, &q)) return rc;
    }
    CUDA_OK(ctx, cudaMemsetAsync(counts + (cur ^ 1u), 0, 4, ctx->stream));
    if (p.shadow_atomic) CUDA_OK(ctx, cudaMemsetAsync(ctx->shadow_count.ptr, 0, 8, ctx->stream));
    {
      LaunchTimer t(ctx, K_PT_SHADE);
      if (plain) {
        k_pt_shade<SP, true><<<blocks_for(active, 128), 128, 0, ctx->stream>>>(p, pt, q, counts + cur, qout, counts + (cur ^ 1u));
      } else {
        k_pt_shade<SP, false><<<blocks_for(active, 128), 128, 0, ctx->stream>>>(p, pt, q, counts + cur, qout, counts + (cur ^ 1u));
      }
    }
    if (p.shadow_atomic) {
      LaunchTimer t(ctx, K_SHADOW_TRACE);
      if (int rc = launch_shadow_resolve(ctx, p, active)) return rc;
    }
    cur ^= 1u;
    std::swap(qin, qout);
    if (int rc = next_queue_size(ctx, counts + cur, active, unsynced)) return rc;
  }
  {
    LaunchTimer t(ctx, K_PT_ACCUMULATE);
    k_pt_accumulate<SP><<<blocks_for(ctx->path_count, 256), 256, 0, ctx->stream>>>(p, pt, pf);
  }
  if (int rc = pt_estimate_noise_levels(ctx, ctx->iteration)) return rc;
  CUDA_OK(ctx, cudaGetLastError());
  return finish_iteration(ctx);
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------------
extern "C" {

const char* etxb_build_flavor(void) { return kFlavor; }

int etxb_device_count(void) {
  int n = 0;
  cudaError_t err = cudaGetDeviceCount(&n);
  if (err != cudaSuccess) return ETXB_ERR_NO_DEVICE;
  return n;
}

int etxb_create(etxb_ctx** out_ctx, const etxb_device_config* cfg) {
  if (!out_ctx) return ETXB_ERR_INVALID_ARGUMENT;
  *out_ctx = nullptr;
  int n = etxb_device_count();
  if (n <= 0) return ETXB_ERR_NO_DEVICE;
  int device = cfg ? cfg->device_index : 0;
  if (device < 0 || device >= n) return ETXB_ERR_INVALID_ARGUMENT;
  if (cudaSetDevice(device) != cudaSuccess) return ETXB_ERR_CUDA;
  auto* ctx = new etxb_ctx();
  ctx->device = device;
  ctx->max_light_vertices_cfg = cfg ? cfg->max_light_vertices : 0;
  ctx->profile = cfg ? (cfg->flags & 1u) != 0 : false;
  if (ctx->profile) {
    // the per-launch timing events of an iteration (two per launch, a few thousand per iteration) exist from the start: a lane that renders its first
    // iteration inside a timed region (the camera-split lane of the replica mode) must not pay for creating them there
    ctx->event_pool.reserve(8192);
    for (uint32_t k = 0; k < 6144u; ++k) {
      cudaEvent_t e = nullptr;
      if (cudaEventCreate(&e) != cudaSuccess) break;
      ctx->event_pool.push_back(e);
    }
  }
  if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete ctx;
    return ETXB_ERR_CUDA;
  }
  cudaEventCreate(&ctx->ev_iter_start);
  cudaEventCreate(&ctx->ev_iter_stop);
  etxb_options_default(&ctx->options);
  *out_ctx = ctx;
  return ETXB_OK;
}

void etxb_destroy(etxb_ctx* ctx) {
  if (!ctx) return;
  if (ctx->worker.joinable()) {
    {
      std::lock_guard<std::mutex> lock(ctx->worker_m);
      ctx->worker_queued = 0;
      ctx->worker_quit = true;
    }
    ctx->worker_cv.notify_all();
    ctx->worker.join();
  }
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (ctx->comm != nullptr) {
    if (NcclApi* n = nccl_api()) n->CommDestroy(ctx->comm);
    ctx->comm = nullptr;
  }
  ctx->comm_counts.release();
  ctx->film_reduced.release();
  if (ctx->comm_stream) cudaStreamDestroy(ctx->comm_stream);
  if (ctx->comm_ev_in) cudaEventDestroy(ctx->comm_ev_in);
  if (ctx->comm_ev_out) cudaEventDestroy(ctx->comm_ev_out);
  for (auto e : ctx->event_pool) cudaEventDestroy(e);
  cudaEventDestroy(ctx->ev_iter_start);
  cudaEventDestroy(ctx->ev_iter_stop);
  DevBuf<float4>* f4[] = {&ctx->ray_o, &ctx->ray_d, &ctx->thr, &ctx->mis, &ctx->hit, &ctx->gathered, &ctx->merged, &ctx->camera_value, &ctx->bvh_tris, &ctx->g_pos, &ctx->g_nrm,
    &ctx->g_win, &ctx->g_thr, &ctx->film_camera, &ctx->film_light, &ctx->film_light_iteration, &ctx->film_out};
  for (auto* b : f4) b->release();
  DevBuf<uint32_t>* u32[] = {&ctx->tri_emitter, &ctx->lv_count, &ctx->lp_offset, &ctx->queue_a, &ctx->queue_b, &ctx->queue_counts, &ctx->sampler_end_light,
    &ctx->sampler_end_camera, &ctx->merge_key, &ctx->conn_seed, &ctx->conn_count, &ctx->lv_tmp_count, &ctx->overflow, &ctx->grid_bbox, &ctx->keys_in, &ctx->keys_out, &ctx->vals_in, &ctx->vals_out};
  for (auto* b : u32) b->release();
  ctx->vertices.release();
  ctx->triangles.release();
  ctx->materials.release();
  ctx->profiles.release();
  ctx->emitters.release();
  ctx->spectra.release();
  ctx->images.release();
  ctx->mediums.release();
  for (auto& b : ctx->medium_density) b.release();
  for (auto& b : ctx->image_pixels) b.release();
  for (auto& b : ctx->image_dists) b.release();
  ctx->emitter_dist.release();
  ctx->bvh_nodes.release();
  ctx->wide_nodes.release();
  ctx->xyz_table.release();
  ctx->rgb_response_table.release();
  ctx->bn_sobol.release();
  ctx->bn_scrambling.release();
  ctx->bn_ranking.release();
  ctx->misc.release();
  ctx->wavelength.release();
  ctx->lv_tmp.release();
  ctx->lv_final.release();
  ctx->cell_range.release();
  ctx->conn_list.release();
  ctx->conn_list_sorted.release();
  ctx->queue_sorted.release();
  ctx->queue_keys.release();
  ctx->queue_keys_sorted.release();
  ctx->shadow_span.release();
  ctx->shadow_p0.release();
  ctx->shadow_p1.release();
  ctx->shadow_value.release();
  ctx->shadow_result.release();
  ctx->shadow_count.release();
  ctx->trace_cursor.release();
  ctx->bs_props.release();
  ctx->bs_weight_pdf.release();
  ctx->bs_wo_eta.release();
  ctx->film_ldr.release();
  ctx->film_normals.release();
  ctx->film_albedo.release();
  ctx->film_adaptive.release();
  ctx->pt_info.release();
  ctx->pt_info_next.release();
  ctx->pt_stats.release();
  ctx->pt_error.release();
  ctx->cub_temp.release();
  ctx->counters.release();
  cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char* etxb_last_error(const etxb_ctx* ctx) { return ctx ? ctx->error.c_str() : "null context"; }

int etxb_upload_color_tables(etxb_ctx* ctx, const float* xyz_441x3, const float* rgb_response_391x3) {
  if (!ctx || !xyz_441x3 || !rgb_response_391x3) return ETXB_ERR_INVALID_ARGUMENT;
  cudaSetDevice(ctx->device);
  if (int rc = upload(ctx, ctx->xyz_table, xyz_441x3, 441 * 3)) return rc;
  if (int rc = upload(ctx, ctx->rgb_response_table, rgb_response_391x3, 391 * 3)) return rc;
  float sum = 0.0f;  // spectrum::kYIntegral (spectrum.hxx:187-193): float sum in table order
  for (int i = 0; i < 441; ++i) sum += xyz_441x3[i * 3 + 1];
  ctx->y_integral = sum;
  ctx->dscene.xyz_table = ctx->xyz_table.ptr;
  ctx->dscene.rgb_response_table = ctx->rgb_response_table.ptr;
  ctx->dscene.y_scale = 1.0f / sum;
  CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  return ETXB_OK;
}

int etxb_upload_blue_noise(etxb_ctx* ctx, const uint8_t* sobol_256x256, const uint8_t* scrambling, const uint8_t* ranking) {
  if (!ctx || !sobol_256x256 || !scrambling || !ranking) return ETXB_ERR_INVALID_ARGUMENT;
  cudaSetDevice(ctx->device);
  if (int rc = upload(ctx, ctx->bn_sobol, sobol_256x256, 256 * 256)) return rc;
  if (int rc = upload(ctx, ctx->bn_scrambling, scrambling, 128 * 128 * 8)) return rc;
  if (int rc = upload(ctx, ctx->bn_ranking, ranking, 128 * 128 * 8)) return rc;
  ctx->dscene.bn_sobol = ctx->bn_sobol.ptr;
  ctx->dscene.bn_scrambling = ctx->bn_scrambling.ptr;
  ctx->dscene.bn_ranking = ctx->bn_ranking.ptr;
  ctx->dscene.has_blue_noise = 1;
  CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  return ETXB_OK;
}

int etxb_upload_scene(etxb_ctx* ctx, const void* scene_blob, uint64_t scene_bytes, const void* camera_blob, uint64_t camera_bytes) {
  if (!ctx || !scene_blob || !camera_blob) return ETXB_ERR_INVALID_ARGUMENT;
  if (scene_bytes != sizeof(etxb_scene) || camera_bytes != sizeof(etxb_camera))
    return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "scene/camera size mismatch: got %llu/%llu, expected %zu/%zu", (unsigned long long)scene_bytes,
      (unsigned long long)camera_bytes, sizeof(etxb_scene), sizeof(etxb_camera));
  if (!ctx->xyz_table.ptr) return fail(ctx, ETXB_ERR_NOT_READY, "etxb_upload_color_tables must be called before etxb_upload_scene");
  ctx_drain_impl(ctx);
  cudaSetDevice(ctx->device);
  ctx->scene_ready = false;
  const etxb_scene& s = *static_cast<const etxb_scene*>(scene_blob);
  const etxb_camera& cam = *static_cast<const etxb_camera*>(camera_blob);

  // ---- what the device path does not cover yet fails loudly (no CPU fallback) --------------------------------------
  if (cam.cls > 1u) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "unknown camera class %u", cam.cls);
  if (cam.lens_image != ETXB_INVALID_INDEX) {
    if (cam.lens_image >= s.images.count) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "camera lens image index out of range");
    const auto& lens = static_cast<const etxb_image*>(s.images.a)[cam.lens_image];
    if (!distribution_covers(lens.y_distribution.values.count, lens.isize[1])) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "camera lens image has no sampling table");
  }
  const auto* mats = static_cast<const etxb_material*>(s.materials.a);
  for (uint64_t i = 0; i < s.materials.count; ++i) {
    const etxb_material& m = mats[i];
    if (!material_class_supported_host(m.cls)) return fail(ctx, ETXB_ERR_UNSUPPORTED, "material %llu: class %u is not supported on the device yet", (unsigned long long)i, m.cls);
    if (m.diffuse_variation > 2u) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "material %llu: unknown diffuse_variation %u", (unsigned long long)i, m.diffuse_variation);
    if (m.subsurface.cls > 2u) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "material %llu: unknown subsurface class %u", (unsigned long long)i, m.subsurface.cls);
    if (m.subsurface.cls != 0) {
      if (s.subsurface_exit_material >= s.materials.count) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "material %llu uses subsurface scattering but scene.subsurface_exit_material is not set", (unsigned long long)i);
      if ((m.subsurface.image_index != ETXB_INVALID_INDEX) && (m.subsurface.image_index >= s.images.count))
        return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "material %llu: subsurface image index out of range", (unsigned long long)i);
    }
    uint32_t imgs[] = {m.reflectance.image_index, m.scattering.image_index, m.emission.image_index, m.roughness.image_index, m.normal_image_index, m.thinfilm.thickness_image};
    for (uint32_t im : imgs)
      if ((im != ETXB_INVALID_INDEX) && (im >= s.images.count)) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "material %llu: image index %u out of range", (unsigned long long)i, im);
    if (((m.int_medium != ETXB_INVALID_INDEX) && (m.int_medium >= s.mediums.count)) || ((m.ext_medium != ETXB_INVALID_INDEX) && (m.ext_medium >= s.mediums.count)))
      return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "material %llu: medium index out of range", (unsigned long long)i);
  }
  ctx->has_stochastic_merge = false;
  for (uint64_t i = 0; i < s.materials.count; ++i) {
    const etxb_material& m = mats[i];
    bool lambert = (m.cls == ETXB_MAT_DIFFUSE) && (m.diffuse_variation == 0);
    bool smooth = (std::max(m.roughness.value[0], m.roughness.value[1]) <= 1.0e-4f) && (m.roughness.image_index == ETXB_INVALID_INDEX);
    bool always_delta = (((m.cls == ETXB_MAT_DIELECTRIC) || (m.cls == ETXB_MAT_CONDUCTOR)) && smooth) || (m.cls == ETXB_MAT_THINFILM) || (m.cls == ETXB_MAT_MIRROR) ||
                        (m.cls == ETXB_MAT_VOID);
    if (!lambert && !always_delta) ctx->has_stochastic_merge = true;
  }
  const auto* emitters = static_cast<const etxb_emitter*>(s.emitter_instances.a);
  for (uint64_t i = 0; i < s.emitter_instances.count; ++i) {
    if (emitters[i].cls > 2u) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "emitter %llu: unknown class %u", (unsigned long long)i, emitters[i].cls);
    if (emitters[i].cls == 1u) {
      const auto& prof = static_cast<const etxb_emitter_profile*>(s.emitter_profiles.a)[emitters[i].profile];
      if (prof.emission.image_index >= s.images.count) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "environment emitter %llu has no image", (unsigned long long)i);
      const auto& img = static_cast<const etxb_image*>(s.images.a)[prof.emission.image_index];
      if (!distribution_covers(img.y_distribution.values.count, img.isize[1])) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "environment emitter %llu: image has no sampling table", (unsigned long long)i);
    }
  }
  // ---- media (medium.hxx:8-47): dense density grids go to HBM as they are -------------------------------------------------------
  {
    const auto* meds = static_cast<const etxb_medium*>(s.mediums.a);
    std::vector<DMedium> dmeds(s.mediums.count);
    for (auto& b : ctx->medium_density) b.release();
    ctx->medium_density.assign(s.mediums.count, {});
    for (uint64_t i = 0; i < s.mediums.count; ++i) {
      const etxb_medium& md = meds[i];
      DMedium& d = dmeds[i];
      d = {};
      d.bounds_min = {md.bounds_min[0], md.bounds_min[1], md.bounds_min[2]};
      d.bounds_max = {md.bounds_max[0], md.bounds_max[1], md.bounds_max[2]};
      d.cls = md.cls;
      d.enable_explicit_connections = md.enable_explicit_connections;
      d.absorption_index = md.absorption_index;
      d.scattering_index = md.scattering_index;
      d.phase_function_g = md.phase_function_g;
      d.max_sigma = md.max_sigma;
      d.dim_x = md.dimensions[0];
      d.dim_y = md.dimensions[1];
      d.dim_z = md.dimensions[2];
      if (md.cls == 1u) {
        size_t n = size_t(d.dim_x) * d.dim_y * d.dim_z;
        if ((n == 0) || (md.density.count != n)) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "medium %llu: density grid does not match its dimensions", (unsigned long long)i);
        CUDA_OK(ctx, ctx->medium_density[i].alloc(n));
        CUDA_OK(ctx, cudaMemcpyAsync(ctx->medium_density[i].ptr, md.density.a, n * 4, cudaMemcpyHostToDevice, ctx->stream));
        d.density = ctx->medium_density[i].ptr;
      } else if (md.cls != 0u) {
        return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "medium %llu: unknown class %u", (unsigned long long)i, md.cls);
      }
    }
    if (int rc = upload(ctx, ctx->mediums, dmeds.data(), dmeds.size())) return rc;
    ctx->dscene.mediums = ctx->mediums.ptr;
    ctx->dscene.medium_count = uint32_t(dmeds.size());
    ctx->dscene.has_boundaries = 0;
    ctx->dscene.has_subsurface = 0;
    ctx->dscene.subsurface_exit_material = s.subsurface_exit_material;
    for (uint64_t i = 0; i < s.materials.count; ++i) {
      if (mats[i].cls == ETXB_MAT_BOUNDARY) ctx->dscene.has_boundaries = 1;
      if (mats[i].subsurface.cls != 0) ctx->dscene.has_subsurface = 1;
    }
    if ((cam.medium_index != ETXB_INVALID_INDEX) && (cam.medium_index >= s.mediums.count)) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "camera medium index out of range");
    // deferred shadow rays (ShadowBatch, dvcm.cuh) need: no alpha test that can reject, no Boundary surfaces / media (transmittance is 0 or 1),
    // no BSDF whose evaluation draws from the sampler, no subsurface exits
    bool deferred = !ctx->has_stochastic_merge && !ctx->dscene.has_boundaries && !ctx->dscene.has_subsurface && (s.mediums.count == 0) && (cam.medium_index == ETXB_INVALID_INDEX);
    const auto* all_images = static_cast<const etxb_image*>(s.images.a);
    for (uint64_t i = 0; deferred && (i < s.materials.count); ++i) {
      if (mats[i].opacity != 1.0f) deferred = false;
      uint32_t im = mats[i].scattering.image_index;
      if ((im != ETXB_INVALID_INDEX) && (all_images[im].options & kImageHasAlpha)) deferred = false;
    }
    ctx->dscene.deferred_shadow_rays = deferred ? 1u : 0u;
    {
      bool opaque = !ctx->dscene.has_boundaries && !ctx->dscene.has_subsurface && (s.mediums.count == 0) && (cam.medium_index == ETXB_INVALID_INDEX);
      for (uint64_t i = 0; opaque && (i < s.materials.count); ++i) {
        if (mats[i].opacity != 1.0f) opaque = false;
        uint32_t im = mats[i].scattering.image_index;
        if ((im != ETXB_INVALID_INDEX) && (all_images[im].options & kImageHasAlpha)) opaque = false;
      }
      ctx->opaque_scene = opaque;
    }
    ctx->plain_scene = !ctx->dscene.has_boundaries && !ctx->dscene.has_subsurface && (s.mediums.count == 0) && (cam.medium_index == ETXB_INVALID_INDEX);
  }
  // ---- images: pixels + flattened row/column CDFs (image.hxx:8-50) ---------------------------------------------------------------
  {
    const auto* imgs = static_cast<const etxb_image*>(s.images.a);
    std::vector<DImage> dimgs(s.images.count);
    for (auto& b : ctx->image_pixels) b.release();
    for (auto& b : ctx->image_dists) b.release();
    ctx->image_pixels.assign(s.images.count, {});
    ctx->image_dists.assign(s.images.count * 2, {});
    for (uint64_t i = 0; i < s.images.count; ++i) {
      const etxb_image& im = imgs[i];
      DImage& d = dimgs[i];
      d = {};
      if ((im.format != 1u) && (im.format != 2u)) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "image %llu: unknown pixel format %u", (unsigned long long)i, im.format);
      size_t px = size_t(im.isize[0]) * im.isize[1];
      if (px == 0) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "image %llu is empty", (unsigned long long)i);
      size_t bytes = px * (im.format == 1u ? 16 : 4);
      CUDA_OK(ctx, ctx->image_pixels[i].alloc(bytes));
      CUDA_OK(ctx, cudaMemcpyAsync(ctx->image_pixels[i].ptr, im.pixels.a, bytes, cudaMemcpyHostToDevice, ctx->stream));
      d.pixels_f32 = (im.format == 1u) ? reinterpret_cast<const float4*>(ctx->image_pixels[i].ptr) : nullptr;
      d.pixels_u8 = (im.format == 2u) ? reinterpret_cast<const uchar4*>(ctx->image_pixels[i].ptr) : nullptr;
      d.fsize_x = im.fsize[0]; d.fsize_y = im.fsize[1];
      d.offset_x = im.offset[0]; d.offset_y = im.offset[1];
      d.scale_x = im.scale[0]; d.scale_y = im.scale[1];
      d.isize_x = im.isize[0]; d.isize_y = im.isize[1];
      d.normalization = im.normalization;
      d.options = im.options;
      d.format = im.format;
      if ((im.y_distribution.values.a != nullptr) && distribution_covers(im.y_distribution.values.count, im.isize[1]) && (im.x_distributions.count == im.isize[1])) {
        size_t nx = size_t(im.isize[0]) + 1u, ny = size_t(im.isize[1]) + 1u;
        std::vector<etxb_distribution_entry> flat(nx * im.isize[1]);
        const auto* rows = static_cast<const etxb_distribution*>(im.x_distributions.a);
        for (uint32_t y = 0; y < im.isize[1]; ++y) {
          if (!distribution_covers(rows[y].values.count, im.isize[0])) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "image %llu: row %u distribution has %llu entries", (unsigned long long)i, y, (unsigned long long)rows[y].values.count);
          memcpy(flat.data() + size_t(y) * nx, rows[y].values.a, nx * sizeof(etxb_distribution_entry));
        }
        CUDA_OK(ctx, ctx->image_dists[i * 2].alloc(flat.size() * sizeof(etxb_distribution_entry)));
        CUDA_OK(ctx, cudaMemcpy(ctx->image_dists[i * 2].ptr, flat.data(), flat.size() * sizeof(etxb_distribution_entry), cudaMemcpyHostToDevice));
        CUDA_OK(ctx, ctx->image_dists[i * 2 + 1].alloc(ny * sizeof(etxb_distribution_entry)));
        CUDA_OK(ctx, cudaMemcpy(ctx->image_dists[i * 2 + 1].ptr, im.y_distribution.values.a, ny * sizeof(etxb_distribution_entry), cudaMemcpyHostToDevice));
        d.x_dist = reinterpret_cast<const etxb_distribution_entry*>(ctx->image_dists[i * 2].ptr);
        d.y_dist = reinterpret_cast<const etxb_distribution_entry*>(ctx->image_dists[i * 2 + 1].ptr);
        d.has_distribution = 1;
      }
    }
    if (int rc = upload(ctx, ctx->images, dimgs.data(), dimgs.size())) return rc;
    ctx->dscene.images = ctx->images.ptr;
    ctx->dscene.image_count = uint32_t(dimgs.size());
  }
  if (s.emitter_instances.count == 0) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "scene has no emitters");
  const auto* spectra = static_cast<const etxb_spectrum*>(s.spectrums.a);
  std::vector<DSpectrum> dspec(s.spectrums.count);
  for (uint64_t i = 0; i < s.spectrums.count; ++i) {
    const etxb_spectrum& sp = spectra[i];
    if (sp.entry_count != 441) return fail(ctx, ETXB_ERR_UNSUPPORTED, "spectrum %llu has %u entries; the loader's 441-entry 390..830 nm grid is required", (unsigned long long)i, sp.entry_count);
    for (uint32_t k = 0; k < 441; ++k) {
      if (sp.entries[k].wavelength != float(390 + k)) return fail(ctx, ETXB_ERR_UNSUPPORTED, "spectrum %llu is not on the integer 390..830 nm grid", (unsigned long long)i);
      dspec[i].power[k] = sp.entries[k].power;
    }
    memcpy(dspec[i].rgb, sp.integrated, 12);
  }

  // ---- geometry ------------------------------------------------------------------------------------------------------
  // every index the host builder and the kernels follow is checked here: a malformed scene is an error, not an out-of-bounds read
  {
    const auto* tris = static_cast<const etxb_triangle*>(s.triangles.a);
    for (uint64_t i = 0; i < s.triangles.count; ++i) {
      const etxb_triangle& t = tris[i];
      if ((t.i[0] >= s.vertices.count) || (t.i[1] >= s.vertices.count) || (t.i[2] >= s.vertices.count))
        return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "triangle %llu: vertex index out of range", (unsigned long long)i);
      if (t.material_index >= s.materials.count) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "triangle %llu: material index %u out of range", (unsigned long long)i, t.material_index);
    }
    if (s.triangle_to_emitter.count != s.triangles.count)
      return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "triangle_to_emitter has %llu entries for %llu triangles", (unsigned long long)s.triangle_to_emitter.count, (unsigned long long)s.triangles.count);
    const auto* t2e = static_cast<const uint32_t*>(s.triangle_to_emitter.a);
    for (uint64_t i = 0; i < s.triangle_to_emitter.count; ++i)
      if ((t2e[i] != ETXB_INVALID_INDEX) && (t2e[i] >= s.emitter_instances.count)) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "triangle %llu: emitter index out of range", (unsigned long long)i);
    for (uint64_t i = 0; i < s.emitter_instances.count; ++i) {
      if (emitters[i].profile >= s.emitter_profiles.count) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "emitter %llu: profile index out of range", (unsigned long long)i);
      if ((emitters[i].cls == 0u) && (emitters[i].triangle_index >= s.triangles.count)) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "area emitter %llu: triangle index out of range", (unsigned long long)i);
    }
    if (!distribution_covers(s.emitters_distribution.values.count, s.emitter_instances.count))
      return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "emitter distribution has %llu entries for %llu emitters", (unsigned long long)s.emitters_distribution.values.count, (unsigned long long)s.emitter_instances.count);
  }
  const auto* verts = static_cast<const etxb_vertex*>(s.vertices.a);
  std::vector<DVertex> dverts(s.vertices.count);
  for (uint64_t i = 0; i < s.vertices.count; ++i) {
    const etxb_vertex& v = verts[i];
    dverts[i].pos_u = make_float4(v.pos[0], v.pos[1], v.pos[2], v.tex[0]);
    dverts[i].nrm_v = make_float4(v.nrm[0], v.nrm[1], v.nrm[2], v.tex[1]);
    dverts[i].tan = make_float4(v.tan[0], v.tan[1], v.tan[2], 0.0f);
    dverts[i].btn = make_float4(v.btn[0], v.btn[1], v.btn[2], 0.0f);
  }
  static_assert(sizeof(DTriangle) == sizeof(etxb_triangle), "triangle layout");
  Bvh bvh;
  {
    cudaEvent_t dummy;
    (void)dummy;
    auto t0 = std::clock();
    build_bvh(reinterpret_cast<const float*>(s.vertices.a), sizeof(etxb_vertex), reinterpret_cast<const uint32_t*>(s.triangles.a), sizeof(etxb_triangle),
      uint32_t(s.triangles.count), bvh);
    ctx->bvh_build_seconds = double(std::clock() - t0) / CLOCKS_PER_SEC;
  }
  if (bvh.max_depth >= uint32_t(kBvhStackSize)) return fail(ctx, ETXB_ERR_UNSUPPORTED, "BVH depth %u exceeds the traversal stack (%d)", bvh.max_depth, kBvhStackSize);
  if (int rc = upload(ctx, ctx->vertices, dverts.data(), dverts.size())) return rc;
  if (int rc = upload(ctx, ctx->triangles, reinterpret_cast<const DTriangle*>(s.triangles.a), size_t(s.triangles.count))) return rc;
  if (int rc = upload(ctx, ctx->tri_emitter, static_cast<const uint32_t*>(s.triangle_to_emitter.a), size_t(s.triangle_to_emitter.count))) return rc;
  if (int rc = upload(ctx, ctx->materials, mats, size_t(s.materials.count))) return rc;
  if (int rc = upload(ctx, ctx->profiles, static_cast<const etxb_emitter_profile*>(s.emitter_profiles.a), size_t(s.emitter_profiles.count))) return rc;
  if (int rc = upload(ctx, ctx->emitters, emitters, size_t(s.emitter_instances.count))) return rc;
  if (int rc = upload(ctx, ctx->spectra, dspec.data(), dspec.size())) return rc;
  if (int rc = upload(ctx, ctx->emitter_dist, static_cast<const etxb_distribution_entry*>(s.emitters_distribution.values.a), size_t(s.emitter_instances.count) + 1u))
    return rc;
  if (int rc = upload(ctx, ctx->bvh_nodes, bvh.nodes.data(), bvh.nodes.size())) return rc;
  if (int rc = upload(ctx, ctx->bvh_tris, reinterpret_cast<const float4*>(bvh.tri_pos.data()), bvh.tri_pos.size())) return rc;

  DeviceScene& d = ctx->dscene;
  d.vertices = ctx->vertices.ptr;
  d.triangles = ctx->triangles.ptr;
  d.tri_emitter = ctx->tri_emitter.ptr;
  d.materials = ctx->materials.ptr;
  d.emitter_profiles = ctx->profiles.ptr;
  d.emitters = ctx->emitters.ptr;
  d.spectra = ctx->spectra.ptr;
  d.emitter_dist = ctx->emitter_dist.ptr;
  d.bvh_nodes = ctx->bvh_nodes.ptr;
  d.bvh_tris = ctx->bvh_tris.ptr;
  d.bvh_node_count = uint32_t(bvh.nodes.size());
  d.wide_nodes = nullptr;
  d.wide_node_count = 0;
#if !(defined(ETXB_PARITY) && ETXB_PARITY)
  if (ctx->has_stochastic_merge) {
    // the sampler streams of such a scene's stochastic stages are the product build's own already: its traversal kernels may meet candidates in
    // another order, so they walk the 4-wide quantised form of the tree (dwide.cuh); Lambert / delta scenes keep the oracle's candidate order
    WideBvh wide;
    build_wide_bvh(bvh, wide);
    if (wide.max_stack < uint32_t(kWideStackSize)) {
      if (int rc = upload(ctx, ctx->wide_nodes, wide.nodes.data(), wide.nodes.size())) return rc;
      d.wide_nodes = ctx->wide_nodes.ptr;
      d.wide_node_count = uint32_t(wide.nodes.size());
    }
  }
#endif
  d.emitter_count = uint32_t(s.emitter_instances.count);
  d.triangle_count = uint32_t(s.triangles.count);
  d.emitter_total_weight = s.emitters_distribution.total_weight;
  memcpy(d.env_emitters, s.environment_emitters, sizeof(d.env_emitters));
  d.env_emitter_count = s.environment_emitter_count;
  d.bounding_sphere_center = {s.bounding_sphere_center[0], s.bounding_sphere_center[1], s.bounding_sphere_center[2]};
  d.bounding_sphere_radius = s.bounding_sphere_radius;
  d.min_path_length = s.min_path_length;
  d.max_path_length = s.max_path_length;
  d.samples = s.samples;
  d.random_path_termination = s.random_path_termination;
  d.spectral = (s.flags & ETXB_SCENE_SPECTRAL) ? 1u : 0u;
  d.spectrum_count = uint32_t(s.spectrums.count);
  d.default_dielectric_eta = s.default_dielectric_eta;
  d.default_conductor_eta = s.default_conductor_eta;
  d.default_conductor_k = s.default_conductor_k;
  d.camera = cam;
  ctx->spectral = d.spectral != 0;
  if ((s.pixel_sampler_image != 0xffffffffu) && (s.pixel_sampler_image >= s.images.count)) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "pixel sampler image out of range");
  ctx->pixel_sampler_image = s.pixel_sampler_image;
  ctx->pixel_sampler_radius = s.pixel_sampler_radius;
  ctx->noise_threshold = s.noise_threshold;
  ctx->radiance_clamp = s.radiance_clamp;
  ctx->scene_samples = s.samples;
  ctx->film_normals.release();  // sized by the film: re-allocated by the next path-tracer run

  // ---- film + queues (Film::allocate, film.cxx) ----------------------------------------------------------------------
  ctx->width = cam.film_size[0];
  ctx->height = cam.film_size[1];
  ctx->path_count = ctx->width * ctx->height;
  size_t n = ctx->path_count;
  if (n == 0) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "empty film");
  DevBuf<float4>* per_path_f4[] = {&ctx->ray_o, &ctx->ray_d, &ctx->thr, &ctx->mis, &ctx->hit, &ctx->gathered, &ctx->merged, &ctx->camera_value, &ctx->film_camera,
    &ctx->film_light, &ctx->film_light_iteration, &ctx->film_out, &ctx->bs_weight_pdf, &ctx->bs_wo_eta};
  for (auto* b : per_path_f4) CUDA_OK(ctx, b->alloc(n));
  CUDA_OK(ctx, ctx->bs_props.alloc(n));
  CUDA_OK(ctx, ctx->misc.alloc(n));
  CUDA_OK(ctx, ctx->wavelength.alloc(n));
  DevBuf<uint32_t>* per_path_u32[] = {&ctx->lv_count, &ctx->lp_offset, &ctx->queue_a, &ctx->queue_b, &ctx->sampler_end_light, &ctx->sampler_end_camera, &ctx->merge_key, &ctx->conn_seed};
  for (auto* b : per_path_u32) CUDA_OK(ctx, b->alloc(n));
  CUDA_OK(ctx, ctx->conn_count.alloc(1));
  CUDA_OK(ctx, ctx->queue_counts.alloc(4));
  CUDA_OK(ctx, ctx->lv_tmp_count.alloc(1));
  CUDA_OK(ctx, ctx->overflow.alloc(1));
  CUDA_OK(ctx, ctx->grid_bbox.alloc(8));
  CUDA_OK(ctx, ctx->counters.alloc(1));
  uint64_t cap = ctx->max_light_vertices_cfg ? ctx->max_light_vertices_cfg : uint64_t(n) * 16ull;
  cap = std::min<uint64_t>(cap, 0x7fffffffull);
  ctx->lv_capacity = uint32_t(cap);
  CUDA_OK(ctx, ctx->lv_tmp.alloc(cap));
  CUDA_OK(ctx, ctx->lv_final.alloc(cap));
  CUDA_OK(ctx, ctx->conn_list.alloc(cap));
  if (ctx->has_stochastic_merge) {
    CUDA_OK(ctx, ctx->conn_list_sorted.alloc(cap));
    CUDA_OK(ctx, ctx->queue_sorted.alloc(n));
    CUDA_OK(ctx, ctx->queue_keys.alloc(n));
    CUDA_OK(ctx, ctx->queue_keys_sorted.alloc(n));
  } else {
    ctx->conn_list_sorted.release();
    ctx->queue_sorted.release();
    ctx->queue_keys.release();
    ctx->queue_keys_sorted.release();
  }
  CUDA_OK(ctx, ctx->trace_cursor.alloc(1));
  const bool atomic_candidate = ctx->opaque_scene && ctx->plain_scene && ctx->has_stochastic_merge;
  if (ctx->dscene.deferred_shadow_rays || atomic_candidate) {
    // atomic mode: a camera bounce queues its vertex connections (<= cap, the pair list's capacity) plus one emitter segment per path
    const uint64_t shadow_cap = std::min<uint64_t>(cap + (atomic_candidate ? n : 0), 0x7fffffffull);
    CUDA_OK(ctx, ctx->shadow_span.alloc(n));
    CUDA_OK(ctx, ctx->shadow_p0.alloc(shadow_cap));
    CUDA_OK(ctx, ctx->shadow_p1.alloc(shadow_cap));
    CUDA_OK(ctx, ctx->shadow_value.alloc(shadow_cap));
    CUDA_OK(ctx, ctx->shadow_result.alloc(shadow_cap));
    CUDA_OK(ctx, ctx->shadow_count.alloc(2));
  } else {
    ctx->shadow_span.release();
    ctx->shadow_p0.release();
    ctx->shadow_p1.release();
    ctx->shadow_value.release();
    ctx->shadow_result.release();
  }
  // the sort buffers also hold the gather queue and the path queues (up to one entry per path), whatever the configured pool capacity
  const uint64_t sort_cap = std::max<uint64_t>(cap, n);
  DevBuf<uint32_t>* per_vertex_u32[] = {&ctx->keys_in, &ctx->keys_out, &ctx->vals_in, &ctx->vals_out};
  for (auto* b : per_vertex_u32) CUDA_OK(ctx, b->alloc(sort_cap));
  DevBuf<float4>* per_vertex_f4[] = {&ctx->g_pos, &ctx->g_nrm, &ctx->g_win, &ctx->g_thr};
  for (auto* b : per_vertex_f4) CUDA_OK(ctx, b->alloc(cap));
  CUDA_OK(ctx, ctx->cell_range.alloc(next_pow2(cap)));
  // one scratch buffer for every CUB call of an iteration: the 32-bit pair sorts (photon grid, gather queue, path queues), the pair-list
  // sort with its 64-bit (path, light vertex) values, and the scan over the per-path vertex counts
  size_t temp_sort = 0, temp_sort64 = 0, temp_scan = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, temp_sort, (uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr, int(sort_cap));
  cub::DeviceRadixSort::SortPairs(nullptr, temp_sort64, (uint32_t*)nullptr, (uint32_t*)nullptr, (unsigned long long*)nullptr, (unsigned long long*)nullptr, int(sort_cap), 0, 16);
  cub::DeviceScan::ExclusiveSum(nullptr, temp_scan, (uint32_t*)nullptr, (uint32_t*)nullptr, int(n));
  CUDA_OK(ctx, ctx->cub_temp.alloc(std::max(std::max(temp_sort, temp_sort64), temp_scan) + 256));
  CUDA_OK(ctx, cudaMemsetAsync(ctx->overflow.ptr, 0, 4, ctx->stream));
  CUDA_OK(ctx, cudaMemsetAsync(ctx->counters.ptr, 0, sizeof(DeviceCounters), ctx->stream));
  CUDA_OK(ctx, cudaMemsetAsync(ctx->sampler_end_light.ptr, 0, n * 4, ctx->stream));
  CUDA_OK(ctx, cudaMemsetAsync(ctx->sampler_end_camera.ptr, 0, n * 4, ctx->stream));
  CUDA_OK(ctx, cudaMemsetAsync(ctx->lv_count.ptr, 0, n * 4, ctx->stream));
  CUDA_OK(ctx, cudaMemsetAsync(ctx->lp_offset.ptr, 0, n * 4, ctx->stream));
  CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->scene_ready = true;
  return etxb_begin(ctx, 0);
}

void etxb_options_default(etxb_vcm_options* opt) {
  if (!opt) return;
  opt->options = ETXB_VCM_FULL;
  opt->radius_decay = 256u;
  opt->kernel = 1u;
  opt->initial_radius = 0.0f;
  opt->blue_noise = 1u;
}

int etxb_options_set_key(etxb_vcm_options* opt, const char* key, double value) {
  if (!opt || !key) return ETXB_ERR_INVALID_ARGUMENT;
  auto set_bit = [&](uint32_t bit) { opt->options = (value != 0.0) ? (opt->options | bit) : (opt->options & ~bit); };
  std::string k = key;
  if (k == "vcm-initial_radius") opt->initial_radius = float(value);
  else if (k == "vcm-radius_decay") opt->radius_decay = uint32_t(value);
  else if (k == "vcm-blue_noise") opt->blue_noise = value != 0.0;
  else if (k == "vcm-kernel") opt->kernel = uint32_t(value);
  else if (k == "vcm-direct_hit") set_bit(ETXB_VCM_DIRECT_HIT);
  else if (k == "vcm-connect_to_light") set_bit(ETXB_VCM_CONNECT_TO_LIGHT);
  else if (k == "vcm-connect_to_camera") set_bit(ETXB_VCM_CONNECT_TO_CAMERA);
  else if (k == "vcm-connect_vertices") set_bit(ETXB_VCM_CONNECT_VERTICES);
  else if (k == "vcm-merge_vertices") set_bit(ETXB_VCM_MERGE_VERTICES);
  else if (k == "vcm-mis") set_bit(ETXB_VCM_ENABLE_MIS);
  else if (k == "vcm-merging") set_bit(ETXB_VCM_ENABLE_MERGING);
  else return ETXB_ERR_INVALID_ARGUMENT;
  return ETXB_OK;
}

int etxb_set_options(etxb_ctx* ctx, const etxb_vcm_options* opt) {
  if (!ctx || !opt) return ETXB_ERR_INVALID_ARGUMENT;
  if (opt->radius_decay == 0) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "radius_decay must be >= 1");
  ctx->options = *opt;
  return ETXB_OK;
}

int etxb_set_partition(etxb_ctx* ctx, uint32_t rank, uint32_t world) {
  if (!ctx || world == 0 || rank >= world) return ETXB_ERR_INVALID_ARGUMENT;
  ctx->rank = rank;
  ctx->world = world;
  return ETXB_OK;
}

int etxb_set_iteration_stride(etxb_ctx* ctx, uint32_t stride) {
  if (!ctx || (stride == 0u)) return ETXB_ERR_INVALID_ARGUMENT;
  ctx->iteration_stride = stride;
  return ETXB_OK;
}

int etxb_set_next_iteration(etxb_ctx* ctx, uint32_t iteration) {
  if (!ctx) return ETXB_ERR_INVALID_ARGUMENT;
  ctx->iteration = iteration;
  ctx->iteration_stride = 0;  // externally driven: no auto-advance, the film mean counts this context's own iterations
  return ETXB_OK;
}

int etxb_begin(etxb_ctx* ctx, uint32_t first_iteration) {
  if (!ctx) return ETXB_ERR_INVALID_ARGUMENT;
  if (!ctx->scene_ready) return fail(ctx, ETXB_ERR_NOT_READY, "no scene uploaded");
  ctx_drain_impl(ctx);  // Integrator::run first stops what is running (vcm_cpu.cxx:255-262)
  cudaSetDevice(ctx->device);
  size_t n = ctx->path_count;
  CUDA_OK(ctx, cudaMemsetAsync(ctx->film_camera.ptr, 0, n * 16, ctx->stream));
  CUDA_OK(ctx, cudaMemsetAsync(ctx->film_light.ptr, 0, n * 16, ctx->stream));
  CUDA_OK(ctx, cudaMemsetAsync(ctx->film_light_iteration.ptr, 0, n * 16, ctx->stream));
  CUDA_OK(ctx, cudaMemsetAsync(ctx->counters.ptr, 0, sizeof(DeviceCounters), ctx->stream));
  CUDA_OK(ctx, cudaMemsetAsync(ctx->overflow.ptr, 0, 4, ctx->stream));
  if (ctx->pt_info.count == n) {
    // Film::clear(ClearCameraData) (film.cxx:345-368): the per-pixel history starts over
    CUDA_OK(ctx, cudaMemsetAsync(ctx->pt_info.ptr, 0, n * 4, ctx->stream));
    CUDA_OK(ctx, cudaMemsetAsync(ctx->pt_error.ptr, 0, n * 4, ctx->stream));
    DevBuf<float4>* layers[] = {&ctx->film_normals, &ctx->film_albedo, &ctx->film_adaptive};
    for (auto* b : layers) CUDA_OK(ctx, cudaMemsetAsync(b->ptr, 0, n * 16, ctx->stream));
  }
  ctx->pt_pixels_processed = 0;
  ctx->pt_active_pixels = ctx->path_count;
  ctx->pt_noise_level = 0.0f;
  CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->iteration = first_iteration;
  ctx->completed = 0;
  ctx->total_time = 0.0;
  ctx->last_iteration_time = 0.0;
  ctx->overflow_flag = 0;
  ctx->kernel_launches = 0;
  ctx->light_pass_done = ctx->grid_done = false;
  memset(ctx->kernel_ms, 0, sizeof(ctx->kernel_ms));
  memset(ctx->kernel_count, 0, sizeof(ctx->kernel_count));
  return ETXB_OK;
}

int etxb_enqueue_light_pass(etxb_ctx* ctx) {
  if (!ctx) return ETXB_ERR_INVALID_ARGUMENT;
  if (!ctx->scene_ready) return fail(ctx, ETXB_ERR_NOT_READY, "no scene uploaded");
  cudaSetDevice(ctx->device);
  CUDA_OK(ctx, cudaEventRecord(ctx->ev_iter_start, ctx->stream));
  return ctx->spectral ? run_light_pass<true>(ctx) : run_light_pass<false>(ctx);
}

int etxb_enqueue_grid_build(etxb_ctx* ctx, const void* device_photon_records, uint64_t photon_count) {
  if (!ctx) return ETXB_ERR_INVALID_ARGUMENT;
  if (!ctx->light_pass_done) return fail(ctx, ETXB_ERR_NOT_READY, "light pass has not run");
  cudaSetDevice(ctx->device);
  const LightVertexRec* records = ctx->lv_final.ptr;
  uint32_t count = ctx->last_light_vertices;
  if (device_photon_records != nullptr) {
    // multi-GPU: the caller all-gathered every rank's path-major records (ETXB_BUF_PHOTON_RECORDS, 96 B each) into one device buffer
    if (photon_count > ctx->lv_capacity) return fail(ctx, ETXB_ERR_OVERFLOW, "gathered photon count %llu exceeds capacity %u", (unsigned long long)photon_count, ctx->lv_capacity);
    records = static_cast<const LightVertexRec*>(device_photon_records);
    count = uint32_t(photon_count);
  }
  return ctx->spectral ? run_grid_build<true>(ctx, records, count) : run_grid_build<false>(ctx, records, count);
}

int etxb_enqueue_camera_pass(etxb_ctx* ctx) {
  if (!ctx) return ETXB_ERR_INVALID_ARGUMENT;
  if (!ctx->light_pass_done || !ctx->grid_done) return fail(ctx, ETXB_ERR_NOT_READY, "light pass / grid build have not run");
  cudaSetDevice(ctx->device);
  int rc = ctx->spectral ? run_camera_pass<true>(ctx) : run_camera_pass<false>(ctx);
  if (rc) return rc;
  return finish_iteration(ctx);
}

// one whole iteration on the calling thread; returns when it has finished (the bounce loops read queue sizes back)
static int run_iteration_blocking(etxb_ctx* ctx) {
  if (ctx->integrator == ETXB_INTEGRATOR_PT) {
    cudaSetDevice(ctx->device);
    return ctx->spectral ? run_pt_iteration<true>(ctx) : run_pt_iteration<false>(ctx);
  }
  if (int rc = etxb_enqueue_light_pass(ctx)) return rc;
  const void* records = nullptr;
  uint64_t count = 0;
  if (ctx->comm != nullptr) {  // pixel tiles over several GPUs: light image + photon records are exchanged here (comm_exchange)
    if (int rc = comm_exchange(ctx, &records, &count)) return rc;
  }
  if (int rc = etxb_enqueue_grid_build(ctx, records, count)) return rc;
  return etxb_enqueue_camera_pass(ctx);
}

static void ctx_worker(etxb_ctx* ctx) {
  std::unique_lock<std::mutex> lock(ctx->worker_m);
  for (;;) {
    ctx->worker_cv.wait(lock, [&] { return ctx->worker_quit || (ctx->worker_queued > 0); });
    if (ctx->worker_quit) return;
    ctx->worker_queued -= 1;
    ctx->worker_busy = true;
    lock.unlock();
    int rc = run_iteration_blocking(ctx);
    lock.lock();
    ctx->worker_busy = false;
    if ((rc != ETXB_OK) && (ctx->worker_error == ETXB_OK)) {
      ctx->worker_error = rc;
      ctx->worker_queued = 0;
    }
    if (ctx->worker_queued == 0) ctx->worker_idle.notify_all();
  }
}

// blocks until every queued iteration has finished; returns (and clears) the first error one of them hit
static int ctx_drain(etxb_ctx* ctx) { return ctx_drain_impl(ctx); }
extern "C++" {
namespace {
int ctx_drain_impl(etxb_ctx* ctx) {
  std::unique_lock<std::mutex> lock(ctx->worker_m);
  ctx->worker_idle.wait(lock, [&] { return (ctx->worker_queued == 0) && !ctx->worker_busy; });
  int rc = ctx->worker_error;
  ctx->worker_error = ETXB_OK;
  return rc;
}
}  // namespace
}  // extern "C++"

int etxb_enqueue_iteration(etxb_ctx* ctx) {
  if (!ctx) return ETXB_ERR_INVALID_ARGUMENT;
  if (!ctx->scene_ready) return fail(ctx, ETXB_ERR_NOT_READY, "no scene uploaded");
  std::lock_guard<std::mutex> lock(ctx->worker_m);
  if (ctx->worker_error != ETXB_OK) {
    int rc = ctx->worker_error;
    ctx->worker_error = ETXB_OK;
    return rc;
  }
  if (!ctx->worker.joinable()) ctx->worker = std::thread(ctx_worker, ctx);
  ctx->worker_queued += 1;
  ctx->worker_cv.notify_one();
  return ETXB_OK;
}


// ---- unidirectional path tracer (CPUPathTracing, rt/integrators/path_tracing.cxx) ---------------------------------------------------------
void etxb_pt_options_default(etxb_pt_options* opt) {
  if (!opt) return;
  opt->nee = opt->direct = opt->mis = opt->blue_noise = 1u;  // PTOptions (path_tracing_shared.hxx:8-14)
}

// the reference's option ids (path_tracing.cxx:36-39, 112-119)
int etxb_pt_options_set_key(etxb_pt_options* opt, const char* key, double value) {
  if (!opt || !key) return ETXB_ERR_INVALID_ARGUMENT;
  const uint32_t v = (value != 0.0) ? 1u : 0u;
  if (!strcmp(key, "direct")) opt->direct = v;
  else if (!strcmp(key, "nee")) opt->nee = v;
  else if (!strcmp(key, "mis")) opt->mis = v;
  else if (!strcmp(key, "bn")) opt->blue_noise = v;
  else return ETXB_ERR_INVALID_ARGUMENT;
  return ETXB_OK;
}

int etxb_pt_set_options(etxb_ctx* ctx, const etxb_pt_options* opt) {
  if (!ctx || !opt) return ETXB_ERR_INVALID_ARGUMENT;
  if (int rc = ctx_drain_impl(ctx)) return rc;
  ctx->pt_options = *opt;
  return ETXB_OK;
}

int etxb_set_integrator(etxb_ctx* ctx, uint32_t integrator) {
  if (!ctx || (integrator > ETXB_INTEGRATOR_PT)) return ETXB_ERR_INVALID_ARGUMENT;
  if (int rc = ctx_drain_impl(ctx)) return rc;
  if ((integrator == ETXB_INTEGRATOR_PT) && (ctx->world > 1u)) return fail(ctx, ETXB_ERR_UNSUPPORTED, "the path tracer runs on one GPU per context");
  ctx->integrator = integrator;
  return ETXB_OK;
}

int etxb_pt_get_status(etxb_ctx* ctx, etxb_pt_status* out) {
  if (!ctx || !out) return ETXB_ERR_INVALID_ARGUMENT;
  memset(out, 0, sizeof(*out));
  out->pixels_processed = ctx->pt_pixels_processed;
  out->active_pixels = ctx->pt_active_pixels;
  out->noise_level = ctx->pt_noise_level;
  out->max_sample_count = ctx->scene_samples;
  return ETXB_OK;
}

// Scene::noise_threshold / radiance_clamp / samples are scene settings the application edits between runs (ui.cxx) without a new upload
int etxb_set_scene_settings(etxb_ctx* ctx, float noise_threshold, float radiance_clamp) {
  if (!ctx || !(noise_threshold >= 0.0f) || !(radiance_clamp >= 0.0f)) return ETXB_ERR_INVALID_ARGUMENT;
  if (int rc = ctx_drain_impl(ctx)) return rc;
  ctx->noise_threshold = noise_threshold;
  ctx->radiance_clamp = radiance_clamp;
  return ETXB_OK;
}

// ---- pixel-tile sharding over NCCL -------------------------------------------------------------------------------------------------------
int etxb_comm_unique_id(void* out_id, uint64_t bytes) {
  if (!out_id || (bytes < sizeof(ncclUniqueId))) return ETXB_ERR_INVALID_ARGUMENT;
  NcclApi* n = nccl_api();
  if (!n) return ETXB_ERR_NOT_READY;
  ncclUniqueId id;
  if (n->GetUniqueId(&id) != ncclSuccess) return ETXB_ERR_CUDA;
  memcpy(out_id, &id, sizeof(id));
  return ETXB_OK;
}

int etxb_comm_init(etxb_ctx* ctx, uint32_t world, uint32_t rank, const void* id, uint64_t bytes) {
  if (!ctx || !id || (bytes < sizeof(ncclUniqueId)) || (world == 0u) || (rank >= world)) return ETXB_ERR_INVALID_ARGUMENT;
  NcclApi* n = nccl_api();
  if (!n) return fail(ctx, ETXB_ERR_NOT_READY, "libnccl.so.2 could not be loaded");
  if (ctx->comm != nullptr) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "the context already has a communicator");
  cudaSetDevice(ctx->device);
  ncclUniqueId uid;
  memcpy(&uid, id, sizeof(uid));
  NCCL_OK(ctx, n->CommInitRank(&ctx->comm, int(world), uid, int(rank)));
  ctx->rank = rank;
  ctx->world = world;
  CUDA_OK(ctx, ctx->comm_counts.alloc(world));
  int prio_low = 0, prio_high = 0;
  CUDA_OK(ctx, cudaDeviceGetStreamPriorityRange(&prio_low, &prio_high));
  CUDA_OK(ctx, cudaStreamCreateWithPriority(&ctx->comm_stream, cudaStreamNonBlocking, prio_high));
  CUDA_OK(ctx, cudaEventCreateWithFlags(&ctx->comm_ev_in, cudaEventDisableTiming));
  CUDA_OK(ctx, cudaEventCreateWithFlags(&ctx->comm_ev_out, cudaEventDisableTiming));
  return ETXB_OK;
}

int etxb_comm_world(const etxb_ctx* ctx, uint32_t* world, uint32_t* rank) {
  if (!ctx || !world || !rank) return ETXB_ERR_INVALID_ARGUMENT;
  *world = (ctx->comm != nullptr) ? ctx->world : 1u;
  *rank = (ctx->comm != nullptr) ? ctx->rank : 0u;
  return ETXB_OK;
}

// Collective: every rank calls it.  The disjoint camera tiles are summed on rank 0 (ncclReduce of the float4 film); the light layer is already
// complete on every rank.  On rank 0 `dst_rgba` (may be null elsewhere) receives the layer like etxb_read_film.
int etxb_comm_reduce_film(etxb_ctx* ctx, uint32_t layer, float* dst_rgba, uint64_t dst_bytes) {
  if (!ctx || (layer > ETXB_FILM_LIGHT)) return ETXB_ERR_INVALID_ARGUMENT;
  if (!ctx->scene_ready) return fail(ctx, ETXB_ERR_NOT_READY, "no scene uploaded");
  if (ctx->comm == nullptr) return etxb_read_film(ctx, layer, dst_rgba, dst_bytes);
  if (int rc = ctx_drain_impl(ctx)) return rc;
  NcclApi* n = nccl_api();
  cudaSetDevice(ctx->device);
  const size_t px = ctx->path_count;
  if (ctx->film_reduced.count < px) CUDA_OK(ctx, ctx->film_reduced.alloc(px));
  if (layer != ETXB_FILM_LIGHT)
    NCCL_OK(ctx, n->Reduce(ctx->film_camera.ptr, ctx->film_reduced.ptr, px * 4u, ncclFloat, ncclSum, 0, ctx->comm, ctx->stream));
  if (ctx->rank != 0u) {
    CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    return ETXB_OK;
  }
  if (!dst_rgba || (dst_bytes < px * 16u)) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "film buffer too small");
  const float4* src = ctx->film_light.ptr;
  if (layer == ETXB_FILM_CAMERA) src = ctx->film_reduced.ptr;
  if (layer == ETXB_FILM_RESULT) {
    FilmBuffers film = {ctx->film_reduced.ptr, ctx->film_light.ptr, ctx->film_light_iteration.ptr, ctx->width, ctx->height};
    k_film_resolve<<<blocks_for(ctx->path_count, 256), 256, 0, ctx->stream>>>(film, ctx->film_out.ptr);
    ctx->kernel_launches += 1;
    src = ctx->film_out.ptr;
  }
  CUDA_OK(ctx, cudaMemcpyAsync(dst_rgba, src, px * 16u, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  return ETXB_OK;
}

int etxb_poll(etxb_ctx* ctx, etxb_status* status) {
  if (!ctx || !status) return ETXB_ERR_INVALID_ARGUMENT;
  memset(status, 0, sizeof(*status));
  status->last_iteration_time = ctx->last_iteration_time;
  status->total_time = ctx->total_time;
  status->completed_iterations = ctx->completed;
  status->current_iteration = ctx->iteration;
  {
    std::lock_guard<std::mutex> lock(ctx->worker_m);
    status->iteration_in_flight = ((ctx->worker_queued > 0) || ctx->worker_busy) ? 1u : 0u;
  }
  status->light_vertices = ctx->last_light_vertices;
  status->overflow = ctx->overflow_flag;
  return ETXB_OK;
}

int etxb_wait(etxb_ctx* ctx) {
  if (!ctx) return ETXB_ERR_INVALID_ARGUMENT;
  if (int rc = ctx_drain(ctx)) return rc;
  cudaSetDevice(ctx->device);
  CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  return ETXB_OK;
}

// CPUVCM::stop (vcm_cpu.cxx:278-288): Immediate drops the queued iterations (the one in flight still completes: its film update is atomic per
// iteration), WaitForCompletion lets everything queued finish
int etxb_stop(etxb_ctx* ctx, int wait_for_iteration) {
  if (!ctx) return ETXB_ERR_INVALID_ARGUMENT;
  if (!wait_for_iteration) {
    std::lock_guard<std::mutex> lock(ctx->worker_m);
    ctx->worker_queued = 0;
  }
  return etxb_wait(ctx);
}

int etxb_film_size(const etxb_ctx* ctx, uint32_t* width, uint32_t* height) {
  if (!ctx || !width || !height) return ETXB_ERR_INVALID_ARGUMENT;
  *width = ctx->width;
  *height = ctx->height;
  return ETXB_OK;
}

// Film::layer (film.cxx:381-418): the device buffer that holds `layer` as float4 (computed into film_out where the layer is derived)
static int film_layer_source(etxb_ctx* ctx, uint32_t layer, const float4** out_src) {
  if (!ctx->scene_ready) return fail(ctx, ETXB_ERR_NOT_READY, "no scene uploaded");
  cudaSetDevice(ctx->device);
  const float4* src = nullptr;
  switch (layer) {
    case ETXB_FILM_RESULT: {
      FilmBuffers film = {ctx->film_camera.ptr, ctx->film_light.ptr, ctx->film_light_iteration.ptr, ctx->width, ctx->height};
      k_film_resolve<<<blocks_for(ctx->path_count, 256), 256, 0, ctx->stream>>>(film, ctx->film_out.ptr);
      ctx->kernel_launches += 1;
      src = ctx->film_out.ptr;
      break;
    }
    case ETXB_FILM_CAMERA:
      src = ctx->film_camera.ptr;
      break;
    case ETXB_FILM_LIGHT:
      src = ctx->film_light.ptr;
      break;
    case ETXB_FILM_LIGHT_ITERATION:
      src = ctx->film_light_iteration.ptr;
      break;
    case ETXB_FILM_NORMALS:
    case ETXB_FILM_ALBEDO:
    case ETXB_FILM_CAMERA_ADAPTIVE: {
      if (int rc = pt_ensure_film(ctx)) return rc;
      if (layer == ETXB_FILM_NORMALS) {
        k_film_layer_normals<<<blocks_for(ctx->path_count, 256), 256, 0, ctx->stream>>>(ctx->film_normals.ptr, ctx->film_out.ptr, ctx->path_count);
        ctx->kernel_launches += 1;
        src = ctx->film_out.ptr;
      } else {
        src = (layer == ETXB_FILM_ALBEDO) ? ctx->film_albedo.ptr : ctx->film_adaptive.ptr;
      }
      break;
    }
    default:
      return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "unknown film layer %u", layer);
  }
  *out_src = src;
  return ETXB_OK;
}

int etxb_read_film(etxb_ctx* ctx, uint32_t layer, float* dst_rgba, uint64_t dst_bytes) {
  if (!ctx || !dst_rgba) return ETXB_ERR_INVALID_ARGUMENT;
  size_t n = ctx->path_count;
  if (ctx->scene_ready && (dst_bytes < n * 16)) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "film buffer too small");
  const float4* src = nullptr;
  if (int rc = film_layer_source(ctx, layer, &src)) return rc;
  CUDA_OK(ctx, cudaMemcpyAsync(dst_rgba, src, n * 16, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  return ETXB_OK;
}

// The tone-mapped 8-bit frame the application shows and exports (app.cxx:268-282): computed on the device, 4 bytes per pixel cross the bus.
int etxb_read_film_ldr(etxb_ctx* ctx, uint32_t layer, float exposure, uint8_t* dst_rgba8, uint64_t dst_bytes) {
  if (!ctx || !dst_rgba8) return ETXB_ERR_INVALID_ARGUMENT;
  size_t n = ctx->path_count;
  if (ctx->scene_ready && (dst_bytes < n * 4)) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "film buffer too small");
  const float4* src = nullptr;
  if (int rc = film_layer_source(ctx, layer, &src)) return rc;
  // a buffer of its own: a preview may be taken while an iteration is in flight on this stream, whose scratch buffers must stay untouched
  if (ctx->film_ldr.count != n) CUDA_OK(ctx, ctx->film_ldr.alloc(n));
  uint32_t* packed = ctx->film_ldr.ptr;
  k_film_tonemap<<<blocks_for(ctx->path_count, 256), 256, 0, ctx->stream>>>(src, packed, ctx->path_count, exposure);
  ctx->kernel_launches += 1;
  CUDA_OK(ctx, cudaMemcpyAsync(dst_rgba8, packed, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  return ETXB_OK;
}

// RTApplication::on_save_image_selected (app.cxx:261-295): mode 0 = the float layer as OpenEXR, mode 1 = the tone-mapped layer as PNG
int etxb_save_film(etxb_ctx* ctx, uint32_t layer, const char* file_name, uint32_t mode, float exposure) {
  if (!ctx || !file_name || (mode > ETXB_SAVE_PNG_TONEMAPPED)) return ETXB_ERR_INVALID_ARGUMENT;
  if (!ctx->scene_ready) return fail(ctx, ETXB_ERR_NOT_READY, "no scene uploaded");
  if (int rc = ctx_drain_impl(ctx)) return rc;
  const size_t n = ctx->path_count;
  int rc = ETXB_OK;
  if (mode == ETXB_SAVE_EXR) {
    std::vector<float> pixels(n * 4u);
    if ((rc = etxb_read_film(ctx, layer, pixels.data(), pixels.size() * 4u)) != ETXB_OK) return rc;
    rc = etxb_write_exr(file_name, pixels.data(), ctx->width, ctx->height);
  } else {
    std::vector<uint8_t> pixels(n * 4u);
    if ((rc = etxb_read_film_ldr(ctx, layer, exposure, pixels.data(), pixels.size())) != ETXB_OK) return rc;
    rc = etxb_write_png(file_name, pixels.data(), ctx->width, ctx->height);
  }
  return (rc == ETXB_OK) ? ETXB_OK : fail(ctx, rc, "could not write %s", file_name);
}

int etxb_get_counters(etxb_ctx* ctx, etxb_counters* out) {
  if (!ctx || !out) return ETXB_ERR_INVALID_ARGUMENT;
  cudaSetDevice(ctx->device);
  DeviceCounters c;
  CUDA_OK(ctx, cudaMemcpyAsync(&c, ctx->counters.ptr, sizeof(c), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  out->rays_closest = c.rays_closest;
  out->rays_shadow = c.rays_shadow;
  out->nodes_visited = c.nodes;
  out->tris_tested = c.tris;
  out->bounces_light = c.bounces_light;
  out->bounces_camera = c.bounces_camera;
  out->light_vertices = c.light_vertices;
  out->connections = c.connections;
  out->merge_queries = c.merge_queries;
  out->merge_candidates = c.merge_candidates;
  out->merge_accepts = c.merge_accepts;
  out->splats = c.splats;
  out->kernel_launches = ctx->kernel_launches;
  out->nodes_closest = c.nodes_closest;
  out->tris_closest = c.tris_closest;
  return ETXB_OK;
}

int etxb_get_kernel_times(etxb_ctx* ctx, const char** names, float* ms, uint32_t* launches, uint32_t capacity) {
  if (!ctx) return ETXB_ERR_INVALID_ARGUMENT;
  uint32_t n = std::min<uint32_t>(capacity, K_COUNT);
  for (uint32_t i = 0; i < n; ++i) {
    if (names) names[i] = kKernelNames[i];
    if (ms) ms[i] = ctx->kernel_ms[i];
    if (launches) launches[i] = ctx->kernel_count[i];
  }
  return int(K_COUNT);
}

int etxb_device_pointer(etxb_ctx* ctx, uint32_t buffer_id, void** out_ptr, uint64_t* out_bytes) {
  if (!ctx || !out_ptr || !out_bytes) return ETXB_ERR_INVALID_ARGUMENT;
  size_t n = ctx->path_count;
  switch (buffer_id) {
    case ETXB_BUF_LIGHT_PATH_COUNT: *out_ptr = ctx->lv_count.ptr; *out_bytes = n * 4; break;
    case ETXB_BUF_LIGHT_PATH_OFFSET: *out_ptr = ctx->lp_offset.ptr; *out_bytes = n * 4; break;
    case ETXB_BUF_LIGHT_PATH_WAVELENGTH: *out_ptr = ctx->wavelength.ptr; *out_bytes = n * 4; break;
    case ETXB_BUF_LIGHT_SAMPLER: *out_ptr = ctx->sampler_end_light.ptr; *out_bytes = n * 4; break;
    case ETXB_BUF_CAMERA_SAMPLER: *out_ptr = ctx->sampler_end_camera.ptr; *out_bytes = n * 4; break;
    case ETXB_BUF_FILM_LIGHT_ITERATION: *out_ptr = ctx->film_light_iteration.ptr; *out_bytes = n * 16; break;
    case ETXB_BUF_FILM_CAMERA: *out_ptr = ctx->film_camera.ptr; *out_bytes = n * 16; break;
    case ETXB_BUF_FILM_LIGHT: *out_ptr = ctx->film_light.ptr; *out_bytes = n * 16; break;
    case ETXB_BUF_PHOTON_RECORDS: *out_ptr = ctx->lv_final.ptr; *out_bytes = size_t(ctx->last_light_vertices) * sizeof(LightVertexRec); break;
    case ETXB_BUF_CAMERA_GATHERED: *out_ptr = ctx->camera_value.ptr; *out_bytes = n * 16; break;
    case ETXB_BUF_PIXEL_INFO:
      if (ctx->pt_info.count != n) return fail(ctx, ETXB_ERR_NOT_READY, "the path tracer has not run on this film");
      *out_ptr = ctx->pt_info.ptr; *out_bytes = n * 4; break;
    case ETXB_BUF_PIXEL_ERROR:
      if (ctx->pt_error.count != n) return fail(ctx, ETXB_ERR_NOT_READY, "the path tracer has not run on this film");
      *out_ptr = ctx->pt_error.ptr; *out_bytes = n * 4; break;
    default: return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "buffer %u has no direct device pointer", buffer_id);
  }
  return ETXB_OK;
}

int etxb_read_buffer(etxb_ctx* ctx, uint32_t buffer_id, void* dst, uint64_t dst_bytes, uint64_t* out_bytes) {
  if (!ctx) return ETXB_ERR_INVALID_ARGUMENT;
  if (int rc = ctx_drain_impl(ctx)) return rc;
  cudaSetDevice(ctx->device);
  size_t lv = ctx->last_light_vertices;
  if (buffer_id == ETXB_BUF_LV_POS || buffer_id == ETXB_BUF_LV_THROUGHPUT || buffer_id == ETXB_BUF_LV_MIS) {
    uint64_t need = lv * 12;
    if (out_bytes) *out_bytes = need;
    if (!dst) return ETXB_OK;
    if (dst_bytes < need) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "buffer too small");
    std::vector<LightVertexRec> host(lv);
    if (lv) CUDA_OK(ctx, cudaMemcpy(host.data(), ctx->lv_final.ptr, lv * sizeof(LightVertexRec), cudaMemcpyDeviceToHost));
    float* out = static_cast<float*>(dst);
    for (size_t i = 0; i < lv; ++i) {
      const LightVertexRec& r = host[i];
      if (buffer_id == ETXB_BUF_LV_POS) {
        out[i * 3 + 0] = r.pos_tri.x; out[i * 3 + 1] = r.pos_tri.y; out[i * 3 + 2] = r.pos_tri.z;
      } else if (buffer_id == ETXB_BUF_LV_THROUGHPUT) {
        out[i * 3 + 0] = r.thr_dvcm.x; out[i * 3 + 1] = r.thr_dvcm.y; out[i * 3 + 2] = r.thr_dvcm.z;
      } else {
        out[i * 3 + 0] = r.thr_dvcm.w; out[i * 3 + 1] = r.wi_dvc.w; out[i * 3 + 2] = r.bc_dvm.w;
      }
    }
    return ETXB_OK;
  }
  void* ptr = nullptr;
  uint64_t bytes = 0;
  if (int rc = etxb_device_pointer(ctx, buffer_id, &ptr, &bytes)) return rc;
  if (buffer_id == ETXB_BUF_CAMERA_GATHERED) {
    uint64_t need = uint64_t(ctx->path_count) * 12;
    if (out_bytes) *out_bytes = need;
    if (!dst) return ETXB_OK;
    if (dst_bytes < need) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "buffer too small");
    std::vector<float4> host(ctx->path_count);
    CUDA_OK(ctx, cudaMemcpy(host.data(), ptr, bytes, cudaMemcpyDeviceToHost));
    float* out = static_cast<float*>(dst);
    for (size_t i = 0; i < host.size(); ++i) {
      out[i * 3 + 0] = host[i].x; out[i * 3 + 1] = host[i].y; out[i * 3 + 2] = host[i].z;
    }
    return ETXB_OK;
  }
  if (out_bytes) *out_bytes = bytes;
  if (!dst) return ETXB_OK;
  if (dst_bytes < bytes) return fail(ctx, ETXB_ERR_INVALID_ARGUMENT, "buffer too small");
  if (bytes) CUDA_OK(ctx, cudaMemcpy(dst, ptr, bytes, cudaMemcpyDeviceToHost));
  return ETXB_OK;
}

void* etxb_stream(etxb_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int etxb_debug_trace(etxb_ctx* ctx, const float* rays, uint32_t* seeds, uint32_t count, float* hits_uv_t, uint32_t* hits_tri) {
  if (!ctx || !rays || !seeds || !hits_uv_t || !hits_tri) return ETXB_ERR_INVALID_ARGUMENT;
  if (!ctx->scene_ready) return fail(ctx, ETXB_ERR_NOT_READY, "no scene uploaded");
  cudaSetDevice(ctx->device);
  DevBuf<float> d_rays, d_uvt;
  DevBuf<uint32_t> d_seeds, d_tri;
  CUDA_OK(ctx, d_rays.alloc(size_t(count) * 8));
  CUDA_OK(ctx, d_uvt.alloc(size_t(count) * 3));
  CUDA_OK(ctx, d_seeds.alloc(count));
  CUDA_OK(ctx, d_tri.alloc(count));
  CUDA_OK(ctx, cudaMemcpy(d_rays.ptr, rays, d_rays.bytes(), cudaMemcpyHostToDevice));
  CUDA_OK(ctx, cudaMemcpy(d_seeds.ptr, seeds, d_seeds.bytes(), cudaMemcpyHostToDevice));
  if (ctx->debug_trace_wide && (ctx->dscene.wide_nodes != nullptr)) {
    k_debug_trace_wide<<<blocks_for(count, 128), 128, 0, ctx->stream>>>(ctx->dscene, d_rays.ptr, d_seeds.ptr, count, d_uvt.ptr, d_tri.ptr);
  } else {
    k_debug_trace<<<blocks_for(count, 128), 128, 0, ctx->stream>>>(ctx->dscene, d_rays.ptr, d_seeds.ptr, count, d_uvt.ptr, d_tri.ptr);
  }
  ctx->kernel_launches += 1;
  CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  CUDA_OK(ctx, cudaMemcpy(seeds, d_seeds.ptr, d_seeds.bytes(), cudaMemcpyDeviceToHost));
  CUDA_OK(ctx, cudaMemcpy(hits_uv_t, d_uvt.ptr, d_uvt.bytes(), cudaMemcpyDeviceToHost));
  CUDA_OK(ctx, cudaMemcpy(hits_tri, d_tri.ptr, d_tri.bytes(), cudaMemcpyDeviceToHost));
  d_rays.release();
  d_uvt.release();
  d_seeds.release();
  d_tri.release();
  return ETXB_OK;
}

// Test hook: which tree etxb_debug_trace walks (0: the BVH2 shared with the oracle; 1: the 4-wide quantised tree of the product build).  Returns 1
// when the requested tree exists for the uploaded scene.
int etxb_debug_select_tree(etxb_ctx* ctx, int wide) {
  if (!ctx) return ETXB_ERR_INVALID_ARGUMENT;
  ctx->debug_trace_wide = wide != 0;
  return (!wide || (ctx->dscene.wide_nodes != nullptr)) ? 1 : 0;
}

int etxb_debug_sampler(etxb_ctx* ctx, const uint32_t* a, const uint32_t* b, uint32_t count, uint32_t draws, uint32_t* out_seed, float* out_values) {
  if (!ctx || !a || !b || !out_seed || !out_values) return ETXB_ERR_INVALID_ARGUMENT;
  cudaSetDevice(ctx->device);
  DevBuf<uint32_t> da, db, ds;
  DevBuf<float> dv;
  CUDA_OK(ctx, da.alloc(count));
  CUDA_OK(ctx, db.alloc(count));
  CUDA_OK(ctx, ds.alloc(size_t(count) * (draws + 1)));
  CUDA_OK(ctx, dv.alloc(size_t(count) * std::max(draws, 1u)));
  CUDA_OK(ctx, cudaMemcpy(da.ptr, a, da.bytes(), cudaMemcpyHostToDevice));
  CUDA_OK(ctx, cudaMemcpy(db.ptr, b, db.bytes(), cudaMemcpyHostToDevice));
  k_debug_sampler<<<blocks_for(count, 128), 128, 0, ctx->stream>>>(da.ptr, db.ptr, count, draws, ds.ptr, dv.ptr);
  ctx->kernel_launches += 1;
  CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  CUDA_OK(ctx, cudaMemcpy(out_seed, ds.ptr, ds.bytes(), cudaMemcpyDeviceToHost));
  if (draws) CUDA_OK(ctx, cudaMemcpy(out_values, dv.ptr, size_t(count) * draws * 4, cudaMemcpyDeviceToHost));
  da.release();
  db.release();
  ds.release();
  dv.release();
  return ETXB_OK;
}

int etxb_debug_math(etxb_ctx* ctx, uint32_t fn, const float* x, const float* y, uint32_t count, float* out) {
  if (!ctx || !x || !out) return ETXB_ERR_INVALID_ARGUMENT;
  cudaSetDevice(ctx->device);
  DevBuf<float> dx, dy, dout;
  CUDA_OK(ctx, dx.alloc(count));
  CUDA_OK(ctx, dout.alloc(count));
  CUDA_OK(ctx, cudaMemcpy(dx.ptr, x, dx.bytes(), cudaMemcpyHostToDevice));
  if (y) {
    CUDA_OK(ctx, dy.alloc(count));
    CUDA_OK(ctx, cudaMemcpy(dy.ptr, y, dy.bytes(), cudaMemcpyHostToDevice));
  }
  k_debug_math<<<blocks_for(count, 128), 128, 0, ctx->stream>>>(ctx->dscene, fn, dx.ptr, y ? dy.ptr : nullptr, count, dout.ptr);
  ctx->kernel_launches += 1;
  CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
  CUDA_OK(ctx, cudaMemcpy(out, dout.ptr, dout.bytes(), cudaMemcpyDeviceToHost));
  dx.release();
  dy.release();
  dout.release();
  return ETXB_OK;
}


// ---------------------------------------------------------------------------------------------------------------------
// Iterations in flight (etxb_group): L contexts on one device, one host thread each, pulling iteration indices from a shared
// counter.  VCM iterations are independent (vcm_cpu.cxx:95-113: the index only sets the merge radius and the sampler seeds), and
// the bounce loop of one iteration ends in a long latency-bound tail (a few thousand paths, ~50 bounces); with several iterations in
// flight that tail overlaps the full-width head of another iteration.  The film is the mean of the lanes' films weighted by the
// iterations each lane finished — the same set of iterations, hence the same estimate, as one context running them in sequence.
// ---------------------------------------------------------------------------------------------------------------------
constexpr uint32_t kMaxLanes = 9;  // 8 whole-iteration lanes + the camera-split lane of the replica mode
struct FilmLanes {
  const float4* camera[kMaxLanes];
  const float4* light[kMaxLanes];
  float weight[kMaxLanes];        // camera layer
  float weight_light[kMaxLanes];  // light layer (differs from `weight` only for a camera-split lane that is not part 0)
  float weight_count[kMaxLanes];  // raw mode: what the lane adds to .w
  uint32_t lanes, layer, pixels;
  uint32_t raw;  // 1: no clamp, alpha = sum of the weights (a partial sum that another stage finishes)
};
__global__ void __launch_bounds__(256) k_film_combine(FilmLanes f, float4* out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= f.pixels) return;
  float x = 0.0f, y = 0.0f, z = 0.0f;
  for (uint32_t l = 0; l < f.lanes; ++l) {
    float4 c = (f.layer != ETXB_FILM_LIGHT) ? f.camera[l][i] : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    float4 g = (f.layer != ETXB_FILM_CAMERA) ? f.light[l][i] : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    x += f.weight[l] * c.x + f.weight_light[l] * g.x;
    y += f.weight[l] * c.y + f.weight_light[l] * g.y;
    z += f.weight[l] * c.z + f.weight_light[l] * g.z;
  }
  if (f.raw) {
    float w = 0.0f;
    for (uint32_t l = 0; l < f.lanes; ++l) w += f.weight_count[l];
    out[i] = make_float4(x, y, z, w);
    return;
  }
  if (f.layer == ETXB_FILM_RESULT) {  // Film::layer(Result): max(0, camera + light) (film.cxx:381-418)
    x = fmaxf(0.0f, x);
    y = fmaxf(0.0f, y);
    z = fmaxf(0.0f, z);
  }
  out[i] = make_float4(x, y, z, 1.0f);
}
// rank 0 of a replica run: the reduced sum of (iterations x mean film) over the ranks -> the mean over all iterations (.w carries the count)
__global__ void __launch_bounds__(256) k_film_finish_mean(const float4* sum, float4* out, uint32_t pixels, uint32_t clamp) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= pixels) return;
  float4 v = sum[i];
  float inv = (v.w > 0.0f) ? 1.0f / v.w : 0.0f;
  float x = v.x * inv, y = v.y * inv, z = v.z * inv;
  if (clamp) {
    x = fmaxf(0.0f, x);
    y = fmaxf(0.0f, y);
    z = fmaxf(0.0f, z);
  }
  out[i] = make_float4(x, y, z, 1.0f);
}

struct etxb_group {
  std::vector<etxb_ctx*> lanes;
  std::vector<std::thread> workers;
  std::mutex m;
  std::condition_variable cv_work, cv_idle;
  uint32_t first_iteration = 0, stride = 1, taken = 0;  // the k-th iteration handed out renders index first + k * stride
  uint32_t pending = 0, in_flight = 0;
  bool quit = false;
  int error = ETXB_OK;
  std::string error_text;
  std::chrono::steady_clock::time_point busy_since;
  double busy_seconds = 0.0;   // wall time with at least one iteration queued or in flight
  double last_iteration_seconds = 0.0;
  DevBuf<float4> combined;
  int device = 0;
  // pixel-tile sharding over several processes (etxb_group_comm_init): every lane has its own communicator, and the k-th iteration of lane l is
  // the ordinal l + k * lanes on EVERY rank (the shared counter of the single-GPU mode would pair different iterations across ranks)
  bool sharded = false;
  struct ReplicaItem {
    uint32_t index;        // ordinal of the iteration within the job
    uint32_t part, parts;  // parts == 1: the whole frame; else the camera pass of part `part` (tile % parts == part), light pass in full
  };
  std::deque<ReplicaItem> whole_queue, split_queue;
  uint32_t split_lane = 0xffffffffu;  // replicas: the lane reserved for camera-split iterations (etxb_group_reserve_split_lane), or none
  uint32_t split_part = 0, split_parts = 0;  // the (part, parts) that lane's film is made of; 0 parts = not used yet
  bool replicas = false;             // etxb_group_comm_init_replicas: whole-frame iterations dealt to the ranks (global index j -> rank j % world), one film reduce
  uint32_t job_enqueued = 0;         // replicas: iterations enqueued for the whole job
  uint32_t world = 1, rank = 0;
  uint32_t enqueued_total = 0;
  std::vector<uint32_t> lane_next;
  ncclComm_t reduce_comm = nullptr;  // the frame reduce has its own communicator: the lanes' ones are busy with iterations in flight
  cudaStream_t stream = nullptr;
  DevBuf<float4> combined_light, reduced;
};

// What one rank takes of `iterations` more iterations of a replica-mode job (ordinals base .. base + iterations - 1).  Whole frames are dealt
// round-robin (ordinal j on rank j % world).  What is left when the count is not a multiple of the ranks would leave some ranks a whole iteration
// behind the others (20 iterations on 8 ranks: 3, 3, 3, 3, 2, 2, 2, 2): with a split lane those R iterations are split instead, each over
// P = world / R ranks by camera tile — every part traces the whole light pass itself (same photon map, no exchange) and the camera pass of its
// tiles; the parts meet in the frame reduce.  A split lane's film is made of ONE (part, parts) geometry: a later round that would need another
// one is dealt as whole frames.  Returns the parts of this round's split (0: none).
static uint32_t replica_plan(uint32_t world, uint32_t rank, uint32_t base, uint32_t iterations, bool split_lane, uint32_t have_part, uint32_t have_parts,
                             std::vector<etxb_group::ReplicaItem>& out) {
  uint32_t whole = iterations, rest = 0, parts = 1;
  if ((iterations >= world) && split_lane) {
    rest = iterations % world;
    parts = rest ? (world / rest) : 1u;
    if ((parts >= 2u) && ((have_parts == 0u) || (have_parts == parts))) {
      whole = iterations - rest;
    } else {
      rest = 0;
    }
  }
  for (uint32_t j = base; j < base + whole; ++j)
    if ((j % world) == rank) out.push_back({j, 0u, 1u});
  for (uint32_t r = 0; r < rest; ++r) {
    if ((rank / parts) != r) continue;
    const uint32_t part = rank % parts;
    if ((have_parts != 0u) && (have_part != part)) continue;  // cannot happen while `parts` stays the same: a rank's part is rank % parts
    out.push_back({base + whole + r, part, parts});
  }
  return rest ? parts : 0u;
}

static bool group_has_work(const etxb_group* grp, uint32_t lane) {
  if (grp->replicas) return (lane == grp->split_lane) ? !grp->split_queue.empty() : !grp->whole_queue.empty();
  if (lane == grp->split_lane) return false;
  return grp->sharded ? (grp->lane_next[lane] < grp->enqueued_total) : (grp->pending > 0);
}
static bool group_idle(const etxb_group* grp) {
  if (grp->in_flight > 0) return false;
  if (grp->replicas) return grp->whole_queue.empty() && grp->split_queue.empty();
  if (!grp->sharded) return grp->pending == 0;
  for (uint32_t next : grp->lane_next)
    if (next < grp->enqueued_total) return false;
  return true;
}

static void group_worker(etxb_group* grp, uint32_t lane) {
  cudaSetDevice(grp->device);
  etxb_ctx* ctx = grp->lanes[lane];
  std::unique_lock<std::mutex> lock(grp->m);
  for (;;) {
    grp->cv_work.wait(lock, [&] { return grp->quit || group_has_work(grp, lane); });
    if (grp->quit) return;
    uint32_t ordinal = 0;
    etxb_group::ReplicaItem item = {0u, 0u, 1u};
    if (grp->replicas) {
      auto& queue = (lane == grp->split_lane) ? grp->split_queue : grp->whole_queue;
      item = queue.front();
      queue.pop_front();
      ordinal = item.index;
      grp->taken = std::max(grp->taken, ordinal + 1u);
    } else if (grp->sharded) {
      ordinal = grp->lane_next[lane];
      grp->lane_next[lane] += uint32_t(grp->lanes.size());
      grp->taken = std::max(grp->taken, ordinal + 1u);
    } else {
      ordinal = grp->taken++;
      grp->pending -= 1;
    }
    uint32_t iteration = grp->first_iteration + ordinal * grp->stride;
    grp->in_flight += 1;
    lock.unlock();
    if (grp->replicas && (lane == grp->split_lane)) {
      // this lane renders the camera pass of its part only; the light pass (and so the photon map) in full
      ctx->rank = item.part;
      ctx->world = item.parts;
      ctx->light_full = true;
    }
    int rc = etxb_set_next_iteration(ctx, iteration);
    if (rc == ETXB_OK) rc = run_iteration_blocking(ctx);  // returns when the iteration has finished (the bounce loops read queue sizes back)
    lock.lock();
    grp->in_flight -= 1;
    grp->last_iteration_seconds = ctx->last_iteration_time;
    if ((rc != ETXB_OK) && (grp->error == ETXB_OK)) {
      grp->error = rc;
      grp->error_text = etxb_last_error(ctx);
      grp->pending = 0;
      grp->whole_queue.clear();
      grp->split_queue.clear();
      for (auto& next : grp->lane_next) next = 0xffffffffu;
    }
    if (group_idle(grp)) {
      grp->busy_seconds += std::chrono::duration<double>(std::chrono::steady_clock::now() - grp->busy_since).count();
      grp->cv_idle.notify_all();
    }
  }
}

int etxb_group_create(etxb_group** out, const etxb_device_config* cfg, uint32_t lanes) {
  if (!out || (lanes == 0) || (lanes > kMaxLanes)) return ETXB_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  auto* grp = new etxb_group();
  grp->device = cfg ? cfg->device_index : 0;
  for (uint32_t l = 0; l < lanes; ++l) {
    etxb_ctx* ctx = nullptr;
    int rc = etxb_create(&ctx, cfg);
    if (rc != ETXB_OK) {
      for (auto* c : grp->lanes) etxb_destroy(c);
      delete grp;
      return rc;
    }
    grp->lanes.push_back(ctx);
  }
  grp->lane_next.assign(lanes, 0u);
  cudaSetDevice(grp->device);
  {
    // the frame combine / reduce must not queue behind the lanes' kernels: highest priority
    int prio_low = 0, prio_high = 0;
    cudaDeviceGetStreamPriorityRange(&prio_low, &prio_high);
    cudaStreamCreateWithPriority(&grp->stream, cudaStreamNonBlocking, prio_high);
  }
  for (uint32_t l = 0; l < lanes; ++l) grp->workers.emplace_back(group_worker, grp, l);
  *out = grp;
  return ETXB_OK;
}

void etxb_group_destroy(etxb_group* grp) {
  if (!grp) return;
  {
    std::lock_guard<std::mutex> lock(grp->m);
    grp->quit = true;
    grp->pending = 0;
  }
  grp->cv_work.notify_all();
  for (auto& w : grp->workers) w.join();
  cudaSetDevice(grp->device);
  grp->combined.release();
  grp->combined_light.release();
  grp->reduced.release();
  if (grp->reduce_comm != nullptr) {
    if (NcclApi* n = nccl_api()) n->CommDestroy(grp->reduce_comm);
  }
  if (grp->stream) cudaStreamDestroy(grp->stream);
  for (auto* c : grp->lanes) etxb_destroy(c);
  delete grp;
}

uint32_t etxb_group_lanes(const etxb_group* grp) { return grp ? uint32_t(grp->lanes.size()) : 0u; }
etxb_ctx* etxb_group_lane(etxb_group* grp, uint32_t lane) { return (grp && (lane < grp->lanes.size())) ? grp->lanes[lane] : nullptr; }
const char* etxb_group_last_error(const etxb_group* grp) { return grp ? grp->error_text.c_str() : "null group"; }

int etxb_group_wait(etxb_group* grp) {
  if (!grp) return ETXB_ERR_INVALID_ARGUMENT;
  std::unique_lock<std::mutex> lock(grp->m);
  grp->cv_idle.wait(lock, [&] { return group_idle(grp); });
  return grp->error;
}

int etxb_group_begin(etxb_group* grp, uint32_t first_iteration) {
  if (!grp) return ETXB_ERR_INVALID_ARGUMENT;
  if (int rc = etxb_group_wait(grp)) return rc;
  for (auto* c : grp->lanes)
    if (int rc = etxb_begin(c, first_iteration)) return rc;
  std::lock_guard<std::mutex> lock(grp->m);
  grp->first_iteration = first_iteration;
  grp->taken = 0;
  grp->enqueued_total = 0;
  grp->job_enqueued = 0;
  grp->whole_queue.clear();
  grp->split_queue.clear();
  grp->split_part = grp->split_parts = 0;
  for (uint32_t l = 0; l < grp->lane_next.size(); ++l) grp->lane_next[l] = l;
  grp->busy_seconds = 0.0;
  grp->error = ETXB_OK;
  grp->error_text.clear();
  return ETXB_OK;
}

int etxb_group_set_stride(etxb_group* grp, uint32_t stride) {
  if (!grp || (stride == 0u)) return ETXB_ERR_INVALID_ARGUMENT;
  std::lock_guard<std::mutex> lock(grp->m);
  grp->stride = stride;
  return ETXB_OK;
}

int etxb_group_enqueue(etxb_group* grp, uint32_t iterations) {
  if (!grp) return ETXB_ERR_INVALID_ARGUMENT;
  {
    std::lock_guard<std::mutex> lock(grp->m);
    if (grp->error != ETXB_OK) return grp->error;
    if (iterations == 0) return ETXB_OK;
    if (group_idle(grp)) grp->busy_since = std::chrono::steady_clock::now();
    if (grp->sharded) {
      grp->enqueued_total += iterations;
    } else if (grp->replicas) {
      // `iterations` more of the JOB's iterations.  Whole frames are dealt round-robin (the job's j-th iteration on rank j % world).  What is left
      // when the count is not a multiple of the ranks would leave some ranks a whole iteration behind the others (20 iterations on 8 ranks: 3, 3, 3, 3,
      // 2, 2, 2, 2): those R iterations are split instead, each over P = world / R ranks by camera tile — every part traces the whole light pass itself
      // (same photon map, no exchange) and the camera pass of its tiles; the parts meet in the frame reduce.
      std::vector<etxb_group::ReplicaItem> items;
      uint32_t parts_used = replica_plan(grp->world, grp->rank, grp->job_enqueued, iterations, grp->split_lane != 0xffffffffu, grp->split_part, grp->split_parts, items);
      for (const auto& it : items) {
        if (it.parts == 1u) {
          grp->whole_queue.push_back(it);
        } else {
          grp->split_part = it.part;
          grp->split_queue.push_back(it);
        }
      }
      if (parts_used) grp->split_parts = parts_used;  // every rank records the split geometry, also those that got no part of this round
      grp->job_enqueued += iterations;
    } else {
      grp->pending += iterations;
    }
  }
  grp->cv_work.notify_all();
  return ETXB_OK;
}

int etxb_group_poll(etxb_group* grp, etxb_status* status) {
  if (!grp || !status) return ETXB_ERR_INVALID_ARGUMENT;
  memset(status, 0, sizeof(*status));
  std::lock_guard<std::mutex> lock(grp->m);
  for (size_t l = 0; l < grp->lanes.size(); ++l) {
    etxb_ctx* c = grp->lanes[l];
    // a camera-split iteration is finished by several ranks: it counts where part 0 ran
    if (!((l == grp->split_lane) && (grp->split_part != 0u))) status->completed_iterations += c->completed;
    status->light_vertices = std::max(status->light_vertices, c->last_light_vertices);
    status->overflow |= c->overflow_flag;
  }
  status->current_iteration = grp->first_iteration + grp->taken * grp->stride;
  status->iteration_in_flight = group_idle(grp) ? 0u : 1u;
  status->last_iteration_time = grp->last_iteration_seconds;
  status->total_time = grp->busy_seconds;
  if (status->iteration_in_flight) status->total_time += std::chrono::duration<double>(std::chrono::steady_clock::now() - grp->busy_since).count();
  return ETXB_OK;
}

static int group_combine_into(etxb_group* grp, uint32_t layer, DevBuf<float4>& target, uint32_t* completed, bool raw = false) {
  etxb_ctx* first = grp->lanes[0];
  if (!first->scene_ready) return fail(first, ETXB_ERR_NOT_READY, "no scene uploaded");
  size_t n = first->path_count;
  cudaSetDevice(grp->device);
  if (target.count < n) {
    target.release();
    CUDA_OK(first, target.alloc(n));
  }
  FilmLanes f = {};
  f.lanes = uint32_t(grp->lanes.size());
  f.layer = layer;
  f.pixels = uint32_t(n);
  uint32_t total = 0;
  for (auto* c : grp->lanes) total += c->completed;
  for (uint32_t l = 0; l < f.lanes; ++l) {
    f.camera[l] = grp->lanes[l]->film_camera.ptr;
    f.light[l] = grp->lanes[l]->film_light.ptr;
    f.weight[l] = raw ? float(grp->lanes[l]->completed) : (total ? float(double(grp->lanes[l]->completed) / double(total)) : 0.0f);
    f.weight_light[l] = f.weight[l];
    f.weight_count[l] = f.weight[l];
    if (raw && (l == grp->split_lane) && (grp->split_part != 0u)) {
      // a camera-split lane that is not part 0: its camera tiles count, its (complete, redundant) light image and its iteration count do not
      f.weight_light[l] = 0.0f;
      f.weight_count[l] = 0.0f;
    }
  }
  f.raw = raw ? 1u : 0u;
  // lanes that are still rendering keep updating their films (a preview, like reading the reference's film while it runs); after
  // etxb_group_wait every lane has synchronised its stream and the result is exact
  k_film_combine<<<blocks_for(f.pixels, 256), 256, 0, grp->stream>>>(f, target.ptr);
  CUDA_OK(first, cudaStreamSynchronize(grp->stream));
  if (completed) *completed = total;
  return ETXB_OK;
}

int etxb_group_combine(etxb_group* grp, uint32_t layer, void** device_ptr, uint64_t* bytes, uint32_t* completed) {
  if (!grp || (layer > ETXB_FILM_LIGHT)) return ETXB_ERR_INVALID_ARGUMENT;
  if (int rc = group_combine_into(grp, layer, grp->combined, completed)) return rc;
  if (device_ptr) *device_ptr = grp->combined.ptr;
  if (bytes) *bytes = uint64_t(grp->lanes[0]->path_count) * 16u;
  return ETXB_OK;
}

// Pixel tiles over several processes, `lanes` iterations in flight on each: ids = (lanes + 1) NCCL unique ids of 128 bytes, the same on every
// rank (lane l of every rank forms communicator l; the last one carries the frame reduce).  Collective.
int etxb_group_comm_init(etxb_group* grp, uint32_t world, uint32_t rank, const void* ids, uint32_t id_count) {
  if (!grp || !ids || (world == 0u) || (rank >= world) || (id_count != grp->lanes.size() + 1u)) return ETXB_ERR_INVALID_ARGUMENT;
  if (int rc = etxb_group_wait(grp)) return rc;
  NcclApi* n = nccl_api();
  etxb_ctx* first = grp->lanes[0];
  if (!n) return fail(first, ETXB_ERR_NOT_READY, "libnccl.so.2 could not be loaded");
  const uint8_t* bytes = static_cast<const uint8_t*>(ids);
  for (size_t l = 0; l < grp->lanes.size(); ++l) {
    if (int rc = etxb_comm_init(grp->lanes[l], world, rank, bytes + l * sizeof(ncclUniqueId), sizeof(ncclUniqueId))) {
      grp->error_text = etxb_last_error(grp->lanes[l]);
      return rc;
    }
  }
  cudaSetDevice(grp->device);
  ncclUniqueId uid;
  memcpy(&uid, bytes + grp->lanes.size() * sizeof(ncclUniqueId), sizeof(uid));
  NCCL_OK(first, n->CommInitRank(&grp->reduce_comm, int(world), uid, int(rank)));
  std::lock_guard<std::mutex> lock(grp->m);
  grp->sharded = world > 1u;
  grp->world = world;
  grp->rank = rank;
  for (uint32_t l = 0; l < grp->lane_next.size(); ++l) grp->lane_next[l] = l;
  grp->enqueued_total = 0;
  return ETXB_OK;
}

// Test hook (no device needed): what rank `rank` of `world` takes of an etxb_group_enqueue(iterations) in replica mode — triples (ordinal, part,
// parts) into out; returns their number.
int etxb_debug_replica_plan(uint32_t world, uint32_t rank, uint32_t base, uint32_t iterations, int split_lane, uint32_t* out_triples, uint32_t capacity) {
  if ((world == 0u) || (rank >= world) || !out_triples) return ETXB_ERR_INVALID_ARGUMENT;
  std::vector<etxb_group::ReplicaItem> items;
  replica_plan(world, rank, base, iterations, split_lane != 0, 0u, 0u, items);
  uint32_t n = 0;
  for (const auto& it : items) {
    if (n >= capacity) break;
    out_triples[n * 3u + 0u] = it.index;
    out_triples[n * 3u + 1u] = it.part;
    out_triples[n * 3u + 2u] = it.parts;
    n += 1u;
  }
  return int(n);
}

// Replica mode: reserves the group's LAST lane for camera-split iterations (see etxb_group_enqueue); it takes no whole-frame iterations.  Call
// before etxb_group_comm_init_replicas; needs at least two lanes.
int etxb_group_reserve_split_lane(etxb_group* grp) {
  if (!grp || (grp->lanes.size() < 2u)) return ETXB_ERR_INVALID_ARGUMENT;
  if (int rc = etxb_group_wait(grp)) return rc;
  std::lock_guard<std::mutex> lock(grp->m);
  grp->split_lane = uint32_t(grp->lanes.size()) - 1u;
  return ETXB_OK;
}

// The other way to split a K-iteration render over the ranks: whole-frame iterations, the job's j-th iteration on rank j % world (each rank's
// lanes take that rank's share in order).  No collective inside an iteration; one ncclReduce of the (count-weighted) films per frame.  id = one
// NCCL unique id.  Collective.
int etxb_group_comm_init_replicas(etxb_group* grp, uint32_t world, uint32_t rank, const void* id, uint64_t bytes) {
  if (!grp || !id || (bytes < sizeof(ncclUniqueId)) || (world == 0u) || (rank >= world)) return ETXB_ERR_INVALID_ARGUMENT;
  if (int rc = etxb_group_wait(grp)) return rc;
  NcclApi* n = nccl_api();
  etxb_ctx* first = grp->lanes[0];
  if (!n) return fail(first, ETXB_ERR_NOT_READY, "libnccl.so.2 could not be loaded");
  cudaSetDevice(grp->device);
  ncclUniqueId uid;
  memcpy(&uid, id, sizeof(uid));
  NCCL_OK(first, n->CommInitRank(&grp->reduce_comm, int(world), uid, int(rank)));
  std::lock_guard<std::mutex> lock(grp->m);
  grp->replicas = world > 1u;
  grp->world = world;
  grp->rank = rank;
  grp->job_enqueued = 0;
  return ETXB_OK;
}

// Collective over the ranks of a sharded group: the lanes' films are combined locally (mean weighted by the iterations each lane finished —
// the same weights on every rank, the lane -> iteration map is fixed), the camera tiles are summed on rank 0, Result = max(0, camera + light).
int etxb_group_comm_reduce_film(etxb_group* grp, uint32_t layer, float* dst_rgba, uint64_t dst_bytes) {
  if (!grp || (layer > ETXB_FILM_LIGHT)) return ETXB_ERR_INVALID_ARGUMENT;
  if (!grp->sharded && !grp->replicas) return etxb_group_read_film(grp, layer, dst_rgba, dst_bytes);
  NcclApi* n = nccl_api();
  etxb_ctx* first = grp->lanes[0];
  const size_t px = first->path_count;
  cudaSetDevice(grp->device);
  if (grp->replicas) {
    // every rank: sum over its lanes of (iterations finished x mean film), .w = iterations; rank 0 divides the reduced sum by the reduced count
    if (int rc = group_combine_into(grp, layer, grp->combined, nullptr, true)) return rc;
    if (grp->reduced.count < px) CUDA_OK(first, grp->reduced.alloc(px));
    NCCL_OK(first, n->Reduce(grp->combined.ptr, grp->reduced.ptr, px * 4u, ncclFloat, ncclSum, 0, grp->reduce_comm, grp->stream));
    if (grp->rank != 0u) {
      CUDA_OK(first, cudaStreamSynchronize(grp->stream));
      return ETXB_OK;
    }
    if (!dst_rgba || (dst_bytes < px * 16u)) return fail(first, ETXB_ERR_INVALID_ARGUMENT, "film buffer too small");
    k_film_finish_mean<<<blocks_for(uint32_t(px), 256), 256, 0, grp->stream>>>(grp->reduced.ptr, grp->combined.ptr, uint32_t(px), (layer == ETXB_FILM_RESULT) ? 1u : 0u);
    CUDA_OK(first, cudaMemcpyAsync(dst_rgba, grp->combined.ptr, px * 16u, cudaMemcpyDeviceToHost, grp->stream));
    CUDA_OK(first, cudaStreamSynchronize(grp->stream));
    return ETXB_OK;
  }
  if (layer != ETXB_FILM_LIGHT) {
    if (int rc = group_combine_into(grp, ETXB_FILM_CAMERA, grp->combined, nullptr)) return rc;
    if (grp->reduced.count < px) CUDA_OK(first, grp->reduced.alloc(px));
    NCCL_OK(first, n->Reduce(grp->combined.ptr, grp->reduced.ptr, px * 4u, ncclFloat, ncclSum, 0, grp->reduce_comm, grp->stream));
  }
  if (grp->rank != 0u) {
    CUDA_OK(first, cudaStreamSynchronize(grp->stream));
    return ETXB_OK;
  }
  if (!dst_rgba || (dst_bytes < px * 16u)) return fail(first, ETXB_ERR_INVALID_ARGUMENT, "film buffer too small");
  const float4* src = grp->reduced.ptr;
  if (layer != ETXB_FILM_CAMERA) {
    if (int rc = group_combine_into(grp, ETXB_FILM_LIGHT, grp->combined_light, nullptr)) return rc;
    src = grp->combined_light.ptr;
  }
  if (layer == ETXB_FILM_RESULT) {
    FilmBuffers film = {grp->reduced.ptr, grp->combined_light.ptr, nullptr, first->width, first->height};
    k_film_resolve<<<blocks_for(uint32_t(px), 256), 256, 0, grp->stream>>>(film, grp->combined.ptr);
    src = grp->combined.ptr;
  }
  CUDA_OK(first, cudaMemcpyAsync(dst_rgba, src, px * 16u, cudaMemcpyDeviceToHost, grp->stream));
  CUDA_OK(first, cudaStreamSynchronize(grp->stream));
  return ETXB_OK;
}

int etxb_group_read_film(etxb_group* grp, uint32_t layer, float* dst_rgba, uint64_t dst_bytes) {
  if (!grp || !dst_rgba) return ETXB_ERR_INVALID_ARGUMENT;
  void* src = nullptr;
  uint64_t bytes = 0;
  if (int rc = etxb_group_combine(grp, layer, &src, &bytes, nullptr)) return rc;
  etxb_ctx* first = grp->lanes[0];
  if (dst_bytes < bytes) return fail(first, ETXB_ERR_INVALID_ARGUMENT, "film buffer too small");
  CUDA_OK(first, cudaMemcpy(dst_rgba, src, bytes, cudaMemcpyDeviceToHost));
  return ETXB_OK;
}

}  // extern "C"
