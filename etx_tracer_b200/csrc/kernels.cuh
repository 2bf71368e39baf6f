// kernels.cuh — the wavefront kernels of one VCM iteration (included once, by module.cu).
//
// Stage list (reference decomposition: bin/optix/vcm/*.cu + vcm_cpu.cxx:95-241, redesigned for sm_100a):
//   light pass : k_light_begin -> { k_trace_closest -> k_light_bounce }*          (queues of path ids, ping-pong)
//   vertices   : scan(counts) -> k_lv_reorder (path-major pool, = the oracle's vertex order)
//   photon map : k_grid_bbox -> k_grid_keys -> radix sort (stable) -> k_grid_build
//   camera pass: k_camera_begin -> { k_trace_closest -> k_camera_shade -> k_camera_merge -> k_camera_continue }*
//   film       : k_film_commit_light, k_film_resolve
// Kernel parameters are `const __grid_constant__`: the out-of-line BSDF / traversal routines take the scene by reference, and without it every
// thread first copies the whole parameter block to its local-memory stack frame (ncu, round 2: 1.6 KB written per thread of k_camera_connect).
// Path state lives in HBM as SoA float4/uint4 columns indexed by path id (128-bit coalesced loads/stores);
// queues are compacted with warp ballot + one atomic per warp.
#pragma once
#include "dvcm.cuh"
#include "dsss.cuh"
#include "dclosure.cuh"
#include "dtrav.cuh"
#include "dwide.cuh"

// resident blocks per SM the bounce / connection kernels are compiled for (128 threads each: 4 blocks = 128 registers per thread).
// Measured on the B200 (bench.py --lanes 1): 1|1 -> 4|4 gives C2 11.04 -> 11.36 and C3 5.55 -> 5.79 Msamples/s; 2 and 3 change nothing.
namespace etxb {

constexpr int kBounceMinBlocks = 4;
constexpr int kConnectMinBlocks = 4;

struct PathBuffers {
  float4* ray_o;     // o.xyz, min_t
  float4* ray_d;     // d.xyz, max_t
  float4* thr;       // throughput (x[,y,z]), path_distance
  float4* mis;       // d_vcm, d_vc, d_vm, eta
  uint4* misc;       // sampler seed, total_path_depth, medium_index, flags
  float4* hit;       // u, v, t, triangle index (bits)
  float4* gathered;  // camera: gathered.xyz
  float4* merged;    // camera: merged.xyz
  float* wavelength;
  uint32_t* lv_count;  // light: vertices stored by the path (VCMLightPath::count)
  float4* bs_weight_pdf;  // camera: pending BSDF sample between the shade and continue stages: weight, pdf
  float4* bs_wo_eta;      //         w_o, eta
  uint2* bs_props;        //         properties, medium index
  uint32_t* merge_key;    // camera: per queue slot, Morton code of the merge query's base grid cell (0xffffffff = no merge)
  uint32_t* conn_seed;    // camera (product build): sampler state the vertex-connection stage derives its per-connection streams from
  uint2* shadow_span;     // camera: (first deferred shadow ray, path connections | NEE << 16) of the vertex shaded this bounce
};

struct DeviceCounters {
  unsigned long long rays_closest, rays_shadow, nodes, tris, bounces_light, bounces_camera, light_vertices, connections, merge_queries, merge_candidates, merge_accepts,
    splats, nodes_closest, tris_closest;
};

struct FilmBuffers {
  float4* camera;           // running mean over iterations (y-flipped storage like film.cxx:189)
  float4* light;            // running mean
  float4* light_iteration;  // per-iteration splats
  uint32_t width, height;
};

struct LaunchParams {
  DeviceScene scene;
  VcmParams vcm;
  PathBuffers paths;
  FilmBuffers film;
  GridData grid;
  LightVertexRec* lv_tmp;    // allocation order
  LightVertexRec* lv_final;  // path-major order
  uint32_t* lv_tmp_count;
  uint32_t lv_capacity;
  const uint32_t* lp_offset;  // VCMLightPath::index
  uint32_t* overflow;
  DeviceCounters* counters;
  uint32_t* sampler_end_light;   // debug taps (ETXB_BUF_LIGHT_SAMPLER / CAMERA_SAMPLER)
  uint32_t* sampler_end_camera;
  float4* camera_value;          // ETXB_BUF_CAMERA_GATHERED
  uint32_t path_count;           // N = W*H
  uint32_t rank, world;          // pixel-tile partition
  uint32_t light_world;          // the light pass's partition: `world` (tiles over NCCL: every rank traces its own pixels' light paths) or 1 (a camera-split
                                 //    iteration: every part traces ALL light paths itself — the same photon map everywhere, nothing to exchange)
  uint32_t camera_sample_index;  // Film sample_count of every pixel before this iteration
  uint2* conn_list;              // product build: (path id, light-vertex ordinal) of every pending vertex connection of this bounce
  uint32_t* conn_count;
  uint32_t conn_capacity;
  uint32_t* conn_key;            // per conn_list entry: (camera vertex material << 8) | light vertex material, or null — the host sorts the list by
                                 // it so that a warp of k_camera_connect evaluates one pair of BSDF classes instead of up to 32
  uint32_t connect_stage;        // 1: vertex connections run in k_camera_connect (product build, scenes with stochastic BSDFs)
  // deferred shadow rays of the camera step (ShadowBatch, dvcm.cuh): segment end points, unoccluded contribution, result (1 = occluded)
  float4* shadow_p0;
  float4* shadow_p1;
  float4* shadow_value;
  uint32_t* shadow_result;
  uint32_t* shadow_count;        // [0] rays reserved this bounce, [1] work cursor of k_shadow_trace
  uint32_t shadow_capacity;
  uint32_t shadow_stage;         // 1: the scene qualifies (DeviceScene::deferred_shadow_rays) and the buffers exist
  uint32_t shadow_atomic;        // 1 (product build, opaque scenes with stochastic BSDFs): the shadow segments of NEE, vertex connections and
                                 //    light-to-camera connections go to the shadow list with their target address; k_shadow_resolve adds the unoccluded ones
  uint32_t merge_material_major; // 1 (scenes with stochastic BSDFs): the gather queue is ordered by (material, Morton code) instead of the Morton code alone
};

#ifdef ETXB_COUNT_TRAVERSAL
#define STATS_DECL TraverseStats stats_obj; TraverseStats* stats = &stats_obj
#define STATS_NODES stats_obj.nodes
#define STATS_TRIS stats_obj.tris
#else
#define STATS_DECL TraverseStats* stats = nullptr
#define STATS_NODES 0u
#define STATS_TRIS 0u
#endif

// PLAIN (template parameter of the bounce kernels): compile-time promise that the scene has no media, Boundary surfaces or subsurface
// materials — what C1-C3-class scenes otherwise pay for in registers, stack and instruction footprint (measured +4 % C2, +6 % on C3's bounce
// kernels).  The host picks the instantiation from the DeviceScene flags.
template <bool PLAIN = false>
DEV bool scene_has_subsurface(const DeviceScene& sc) {
  if constexpr (PLAIN) return false;
  return sc.has_subsurface != 0u;
}

DEV void counter_add(unsigned long long* dst, uint32_t v) {
  uint32_t total = __reduce_add_sync(__activemask(), v);
  uint32_t leader = __ffs(__activemask()) - 1;
  if ((threadIdx.x & 31u) == leader && total) atomicAdd(dst, (unsigned long long)total);
}

// warp-aggregated append of `id` to a queue when `alive`
DEV void queue_push(uint32_t* queue, uint32_t* queue_count, bool alive, uint32_t id) {
  uint32_t mask = __activemask();
  uint32_t ballot = __ballot_sync(mask, alive);
  if (ballot == 0) return;
  uint32_t lane = threadIdx.x & 31u;
  uint32_t leader = __ffs(ballot) - 1;
  uint32_t base = 0;
  if (lane == leader) base = atomicAdd(queue_count, __popc(ballot));
  base = __shfl_sync(mask, base, leader);
  if (alive) queue[base + __popc(ballot & ((1u << lane) - 1u))] = id;
}

DEV bool pixel_owned(const LaunchParams& p, uint32_t index, bool light_pass = false) {
  const uint32_t world = light_pass ? p.light_world : p.world;
  if (world <= 1u) return true;
  uint32_t x = index % p.film.width, y = index / p.film.width;
  uint32_t tiles_x = (p.film.width + 31u) / 32u;
  uint32_t tile = (y / 32u) * tiles_x + (x / 32u);
  return (tile % world) == p.rank;
}

template <bool SP>
DEV void store_state(const PathBuffers& b, uint32_t i, const PathState<SP>& s) {
  V3 t = s.throughput.as_v3();
  b.ray_o[i] = make_float4(s.ray_o.x, s.ray_o.y, s.ray_o.z, s.ray_min_t);
  b.ray_d[i] = make_float4(s.ray_d.x, s.ray_d.y, s.ray_d.z, s.ray_max_t);
  b.thr[i] = make_float4(t.x, t.y, t.z, s.path_distance);
  b.mis[i] = make_float4(s.d_vcm, s.d_vc, s.d_vm, s.eta);
  b.misc[i] = make_uint4(s.sampler.seed, s.total_path_depth, s.medium_index, s.flags);
}
template <bool SP>
DEV PathState<SP> load_state(const PathBuffers& b, uint32_t i) {
  PathState<SP> s;
  float4 o = b.ray_o[i], d = b.ray_d[i], t = b.thr[i], m = b.mis[i];
  uint4 u = b.misc[i];
  s.ray_o = {o.x, o.y, o.z};
  s.ray_min_t = o.w;
  s.ray_d = {d.x, d.y, d.z};
  s.ray_max_t = d.w;
  s.throughput = Spec<SP>::make3({t.x, t.y, t.z});
  s.path_distance = t.w;
  s.d_vcm = m.x;
  s.d_vc = m.y;
  s.d_vm = m.z;
  s.eta = m.w;
  s.sampler.seed = u.x;
  s.sampler.fixed_u = s.sampler.fixed_v = s.sampler.fixed_w = 0.0f;
  s.total_path_depth = u.y;
  s.medium_index = u.z;
  s.flags = u.w;
  s.wavelength = b.wavelength[i];
  s.gathered = Spec<SP>::make(0.0f);
  s.merged = {0.0f, 0.0f, 0.0f};
  s.lv_count = 0;
  return s;
}

// ---------------------------------------------------------------------------------------------------------------------
// light pass
// ---------------------------------------------------------------------------------------------------------------------
template <bool SP>
__global__ void __launch_bounds__(128) k_light_begin(const __grid_constant__ LaunchParams p, uint32_t* queue, uint32_t* queue_count) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  bool alive = false;
  if (i < p.path_count) {
    bool owned = pixel_owned(p, i, true);
    PathState<SP> s = generate_emitter_state<SP>(p.scene, p.vcm, i);
    p.paths.wavelength[i] = s.wavelength;
    p.paths.lv_count[i] = 0;
    alive = owned && ((s.flags & kPathValid) == kPathValid);
    if (alive) {
      store_state<SP>(p.paths, i, s);
    } else {
      p.sampler_end_light[i] = s.sampler.seed;
    }
  }
  queue_push(queue, queue_count, alive, i);
}

// Sort key of a queue slot after its closest-hit query: the hit material (0xff = miss; 0x100 = slot past the device-side count, sorts last)
constexpr uint32_t kQueueKeyPastCount = 0x100u;
DEV uint32_t queue_sort_key(const LaunchParams& p, uint32_t tri) { return (tri == kInvalidIndex) ? 0xffu : umin(load_triangle_material(p.scene, tri), 0xfeu); }

// closest-hit traversal for every queued path (Raytracing::trace, rt.cxx:428): SoA ray in, hit record out,
// sampler advanced by one draw per candidate
__global__ void __launch_bounds__(256) k_trace_closest(const __grid_constant__ LaunchParams p, const uint32_t* queue, const uint32_t* queue_count, uint32_t* material_keys, uint32_t key_limit) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= *queue_count) {
    // the host sorts `key_limit` (its upper bound of the queue size) slots by material: slots past the device-side count sort last
    if ((material_keys != nullptr) && (q < key_limit)) material_keys[q] = kQueueKeyPastCount;
    return;
  }
  uint32_t i = queue[q];
  float4 o = p.paths.ray_o[i], d = p.paths.ray_d[i];
  uint4 misc = p.paths.misc[i];
  Smp smp;
  smp.seed = misc.x;
  smp.fixed_u = smp.fixed_v = smp.fixed_w = 0.0f;
  STATS_DECL;
  HitRec h = trace_closest(p.scene, {o.x, o.y, o.z}, {d.x, d.y, d.z}, o.w, d.w, smp, stats);
  p.paths.hit[i] = make_float4(h.u, h.v, h.t, __uint_as_float(h.tri));
  p.paths.misc[i].x = smp.seed;
  // the bounce kernels' cost is the BSDF class of the surface that was hit: paths are grouped by material before they are shaded
  if (material_keys != nullptr) material_keys[q] = queue_sort_key(p, h.tri);
  counter_add(&p.counters->rays_closest, 1u);
  counter_add(&p.counters->nodes, STATS_NODES);
  counter_add(&p.counters->tris, STATS_TRIS);
#ifdef ETXB_COUNT_TRAVERSAL
  counter_add(&p.counters->nodes_closest, STATS_NODES);
  counter_add(&p.counters->tris_closest, STATS_TRIS);
#endif
}

// Film::atomic_add_light_iteration (film.cxx:147-171) of one light-tracing contribution (vcm_cpu.cxx:147-154), in two halves: value -> RGB and
// pixel (false: below the driver's cut or off the film), then the three float atomics
template <bool SP>
DEV bool splat_prepare(const LaunchParams& p, Spec<SP> value, V2 uv, float wavelength, V3& rgb, uint32_t& pixel, uint32_t& counted) {
  rgb = spec_to_rgb<SP>(p.scene, value, wavelength) / sampling_pdf<SP>(wavelength);
  if (!(dot(rgb, rgb) > kEpsilon)) return false;
  counted = 1u;
  V2 uv01 = uv * 0.5f + 0.5f;
  uint32_t x = static_cast<uint32_t>(uv01.x * float(p.film.width));
  uint32_t y = static_cast<uint32_t>(uv01.y * float(p.film.height));
  if ((x >= p.film.width) || (y >= p.film.height)) return false;
  pixel = x + (p.film.height - 1u - y) * p.film.width;
  return true;
}
DEV void splat_add(const LaunchParams& p, uint32_t pixel, V3 rgb) {
  float* dst = reinterpret_cast<float*>(p.film.light_iteration + pixel);
  atomicAdd(dst + 0, rgb.x);
  atomicAdd(dst + 1, rgb.y);
  atomicAdd(dst + 2, rgb.z);
}
template <bool SP>
DEV uint32_t splat_light(const LaunchParams& p, Spec<SP> value, V2 uv, float wavelength) {
  V3 rgb;
  uint32_t pixel = 0, counted = 0;
  if (splat_prepare<SP>(p, value, uv, wavelength, rgb, pixel, counted)) splat_add(p, pixel, rgb);
  return counted;
}

// store one light vertex in allocation order (k_lv_reorder makes the pool path-major)
DEV bool store_light_vertex(const LaunchParams& p, const LightVertexRec& rec) {
  uint32_t slot = atomicAdd(p.lv_tmp_count, 1u);
  if (slot >= p.lv_capacity) {
    *p.overflow = 1u;
    return false;
  }
  float4* dst = reinterpret_cast<float4*>(p.lv_tmp + slot);
  dst[0] = rec.thr_dvcm;
  dst[1] = rec.wi_dvc;
  dst[2] = rec.bc_dvm;
  dst[3] = rec.pos_tri;
  dst[4] = rec.nrm_mat;
  reinterpret_cast<uint4*>(dst)[5] = rec.ids;
  return true;
}

// vcm_light_step after the trace (vcm_shared.hxx:1090-1260): medium events, boundary crossings, surface events
// which endpoints of the current vertex run explicit connections
enum : uint32_t { kEpNone = 0u, kEpMedium = 1u, kEpSurface = 2u, kEpSubsurface = 3u };

// vcm_light_step (vcm_shared.hxx:1086-1259).  Three phases so that every heavy routine has ONE call site: (A) the event at the end of
// the segment (medium scattering, boundary crossing, surface hit incl. the subsurface walk), (B) camera connections from the
// endpoint(s) it produced — one, or every gathered subsurface exit (:1207-1222), (C) the continuation.
template <bool SP, bool PLAIN>
__global__ void __launch_bounds__(128, kBounceMinBlocks) k_light_bounce(const __grid_constant__ LaunchParams p, const uint32_t* queue_in, const uint32_t* count_in, uint32_t* queue_out, uint32_t* count_out) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  bool alive = false;
  uint32_t i = 0;
  uint32_t shadow_rays = 0, splats = 0, stored = 0;
  STATS_DECL;
  if (q < *count_in) {
    i = queue_in[q];
    const DeviceScene& sc = p.scene;
    PathState<SP> state = load_state<SP>(p.paths, i);
    state.lv_count = p.paths.lv_count[i];
    float4 hit = p.paths.hit[i];
    uint32_t tri_index = __float_as_uint(hit.w);
    const bool found = tri_index != kInvalidIndex;
    uint32_t ep_mode = kEpNone;
    bool at_medium = false, at_surface = false, ss_path = false, ss_sampled = false;
    V2 rnd_bsdf = {0.0f, 0.0f}, rnd_connection = {0.0f, 0.0f}, rnd_support = {0.0f, 0.0f};
    V3 medium_pos = {0.0f, 0.0f, 0.0f};
    Isect isect{};
    BSample<SP> bs;
    SSGather<SP> ssg;
    ssg.count = 0;
    // ---- (A) ----
    MediumSample<SP> medium_sample = vcm_try_sampling_medium<SP, PLAIN>(sc, state, found ? hit.z : kMaxFloat);
    if (medium_sample.sampled_medium()) {
      // :1097-1170
      at_medium = true;
      medium_pos = medium_sample.pos;
      rnd_bsdf = state.sampler.next_2d();
      rnd_connection = state.sampler.next_2d();
      rnd_support = state.sampler.next_2d();
      float seg = state.path_distance + medium_sample.sampled_medium_t;
      state.d_vcm *= sqr(seg);
      state.path_distance = 0.0f;
      const DMedium& med = sc.mediums[state.medium_index];
      if (p.vcm.connect_vertices() && (state.total_path_depth + 1 <= sc.max_path_length)) {
        if (store_light_vertex(p, make_medium_light_vertex<SP>(state, medium_pos, i))) {
          state.lv_count += 1;
          stored = 1;
        }
      }
      if (p.vcm.connect_to_camera() && med.enable_explicit_connections && (state.total_path_depth + 1 <= sc.max_path_length)) ep_mode = kEpMedium;
    } else if (found) {
      isect = make_intersection(sc, state.ray_d, tri_index, hit.x, hit.y, hit.z);
      if (vcm_handle_boundary<SP, PLAIN>(sc, isect, state)) {
        alive = true;
      } else {
        at_surface = true;
        const etxb_material& mat = sc.materials[isect.material_index];
        BData bsdf_data = make_bdata(isect, isect.w_i, state.wavelength, state.medium_index, kPathLight);
        rnd_bsdf = state.sampler.next_2d();
        rnd_connection = state.sampler.next_2d();
        rnd_support = state.sampler.next_2d();
        state.sampler.push_fixed(rnd_bsdf.x, rnd_bsdf.y, rnd_support.x);
        bs = bsdf_sample<SP>(sc, bsdf_data, mat, state.sampler);
        bool is_connectible = (bs.properties & kBsdfDelta) == 0;
        state.sampler.pop_fixed();
        // vcm_update_light_vcm (:451-461)
        if ((state.total_path_depth > 0) || (state.flags & kPathLocalEmitter)) {
          state.d_vcm *= sqr(state.path_distance + isect.t);
        }
        float cos_to_prev = fabsf(dot(isect.nrm, -state.ray_d));
        state.d_vcm /= cos_to_prev;
        state.d_vc /= cos_to_prev;
        state.d_vm /= cos_to_prev;
        state.path_distance = 0.0f;
        ss_path = scene_has_subsurface<PLAIN>(sc) && (bs.properties & kBsdfDiffuse) && (mat.subsurface.cls != 0u);
        if (ss_path) ss_sampled = ss_gather<SP>(sc, state.wavelength, isect, state.sampler, ssg, stats, shadow_rays);
        if (is_connectible) {
          if (store_light_vertex(p, make_light_vertex<SP>(state, isect, i))) {  // the vertex stays at the entry point (:1204)
            state.lv_count += 1;
            stored = 1;
          }
          if (p.vcm.connect_to_camera() && (state.total_path_depth + 1 <= sc.max_path_length)) ep_mode = ss_sampled ? kEpSubsurface : kEpSurface;
        }
      }
    }
    // ---- (B) ----
    if (ep_mode != kEpNone) {
      uint32_t n = (ep_mode == kEpSubsurface) ? ssg.count : 1u;
      Isect ep_isect = isect;
#pragma unroll 1
      for (uint32_t k = 0; k < n; ++k) {
        Spec<SP> w = Spec<SP>::make(1.0f);
        if (ep_mode == kEpSubsurface) {
          ep_isect = ss_exit_intersection<SP>(sc, ssg, k, sc.subsurface_exit_material);
          w = ssg.weights[k];
        }
        Endpoint ep{ep_mode == kEpMedium, &ep_isect, medium_pos};  // one object behind the pointer: it stays in registers
        state.sampler.push_fixed(rnd_connection.x, rnd_connection.y, rnd_support.y);
        Spec<SP> value;
        V2 uv;
        V3 segment[2];
        const bool defer = PLAIN && (p.shadow_atomic != 0u);
        bool ok = vcm_connect_to_camera<SP, PLAIN>(sc, p.vcm, ep, state, value, uv, stats, shadow_rays, defer ? segment : nullptr);
        state.sampler.pop_fixed();
        if (ok && (value.maximum() > kEpsilon)) {
          if (defer) {
            // the segment goes to the bounce's shadow list with the pixel it lands on; k_shadow_resolve splats it if nothing is in between
            V3 rgb;
            uint32_t pixel = 0, counted = 0;
            if (splat_prepare<SP>(p, value, uv, state.wavelength, rgb, pixel, counted)) {
              ShadowBatch batch = {p.shadow_p0, p.shadow_p1, p.shadow_value, 0u, 0u, p.shadow_count, p.shadow_capacity, pixel | kShadowTargetPixel};
              batch.push_rgb(segment[0], segment[1], rgb);
            }
          } else {
            splats += splat_light<SP>(p, (ep_mode == kEpSubsurface) ? (w * value) : value, uv, state.wavelength);
          }
        }
      }
    }
    // ---- (C) ----
    if (at_medium) {
      const DMedium& med = sc.mediums[state.medium_index];
      V3 w_i = state.ray_d;
      V3 w_o_smp = sample_phase_function(w_i, med.phase_function_g, rnd_bsdf);
      float pdf_fwd = phase_function(w_i, w_o_smp, med.phase_function_g);
      float pdf_rev = phase_function(w_o_smp, w_i, med.phase_function_g);
      state.d_vc = (1.0f / pdf_fwd) * (state.d_vc * pdf_rev + state.d_vcm);
      state.d_vm = (1.0f / pdf_fwd) * (state.d_vm * pdf_rev + 0.0f);
      state.d_vcm = 1.0f / pdf_fwd;
      state.ray_o = medium_pos;
      state.ray_d = w_o_smp;
      state.ray_max_t = kMaxFloat;
      state.ray_min_t = kRayEpsilon;
      state.total_path_depth += 1;
      alive = (state.total_path_depth + 1 <= sc.max_path_length) &&
              random_continue<SP>(state.total_path_depth, sc.random_path_termination, state.eta, state.sampler, state.throughput);
    } else if (at_surface && !(ss_path && !ss_sampled)) {
      if (ss_sampled) {
        // :1237-1249 — continue from the selected exit with a cosine lobe; the light step keeps the hit's own material
        state.throughput *= ssg.weights[ssg.selected] * ssg.selected_sample_weight;
        isect = ss_exit_intersection<SP>(sc, ssg, ssg.selected, isect.material_index);
        bs.w_o = sample_cosine_around(state.sampler.next_2d(), isect.nrm, 1.0f);
        bs.pdf = fabsf(dot(bs.w_o, isect.nrm)) / kPi;
        bs.eta = 1.0f;
      }
      BData bsdf_data = make_bdata(isect, isect.w_i, state.wavelength, state.medium_index, kPathLight);
      if (vcm_next_ray<SP>(sc, true, state, p.vcm, isect, bsdf_data, bs, ss_sampled)) {
        alive = state.total_path_depth + 1u < sc.max_path_length;
      }
    }
    p.paths.lv_count[i] = state.lv_count;
    if (alive) {
      store_state<SP>(p.paths, i, state);
    } else {
      p.sampler_end_light[i] = state.sampler.seed;
    }
  }
  queue_push(queue_out, count_out, alive, i);
  counter_add(&p.counters->bounces_light, (q < *count_in) ? 1u : 0u);
  counter_add(&p.counters->rays_shadow, shadow_rays);
  counter_add(&p.counters->splats, splats);
  counter_add(&p.counters->light_vertices, stored);
  counter_add(&p.counters->nodes, STATS_NODES);
  counter_add(&p.counters->tris, STATS_TRIS);
}

// pool in allocation order -> path-major order: dst = VCMLightPath::index + ordinal (vcm_cpu.cxx:155-171)
__global__ void __launch_bounds__(256) k_lv_reorder(const __grid_constant__ LaunchParams p, uint32_t count) {
  uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= count) return;
  const float4* src = reinterpret_cast<const float4*>(p.lv_tmp + s);
  float4 r0 = src[0], r1 = src[1], r2 = src[2], r3 = src[3], r4 = src[4];
  uint4 ids = reinterpret_cast<const uint4*>(src)[5];
  uint32_t dst_index = p.lp_offset[ids.z] + ids.w;
  float4* dst = reinterpret_cast<float4*>(p.lv_final + dst_index);
  dst[0] = r0;
  dst[1] = r1;
  dst[2] = r2;
  dst[3] = r3;
  dst[4] = r4;
  reinterpret_cast<uint4*>(dst)[5] = ids;
}

// ---------------------------------------------------------------------------------------------------------------------
// photon hash grid (VCMSpatialGrid::construct, vcm_shared.cxx:49-152)
// ---------------------------------------------------------------------------------------------------------------------
DEV uint32_t float_to_ordered(float f) {
  uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ inline float ordered_to_float(uint32_t o) {
  uint32_t u = (o & 0x80000000u) ? (o & 0x7fffffffu) : ~o;
  union { uint32_t u; float f; } c;
  c.u = u;
  return c.f;
}

// bbox[0..2] = min (ordered uint), bbox[3..5] = max
__global__ void __launch_bounds__(256) k_grid_bbox(const LightVertexRec* pool, uint32_t count, uint32_t* bbox) {
  // grid-stride over the pool, then warp -> block -> 6 atomics per block (min / max are order independent: same box as any other order)
  __shared__ float s_mn[8][3], s_mx[8][3];
  float mn[3] = {kMaxFloat, kMaxFloat, kMaxFloat}, mx[3] = {-kMaxFloat, -kMaxFloat, -kMaxFloat};
  for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s < count; s += gridDim.x * blockDim.x) {
    float4 pt = reinterpret_cast<const float4*>(pool + s)[3];
    if (__float_as_uint(pt.w) != kInvalidIndex) {  // medium vertices are never merged (vcm_shared.cxx:70)
      mn[0] = fminf(mn[0], pt.x);
      mx[0] = fmaxf(mx[0], pt.x);
      mn[1] = fminf(mn[1], pt.y);
      mx[1] = fmaxf(mx[1], pt.y);
      mn[2] = fminf(mn[2], pt.z);
      mx[2] = fmaxf(mx[2], pt.z);
    }
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    for (int o = 16; o > 0; o >>= 1) {
      mn[k] = fminf(mn[k], __shfl_xor_sync(0xffffffffu, mn[k], o));
      mx[k] = fmaxf(mx[k], __shfl_xor_sync(0xffffffffu, mx[k], o));
    }
  }
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      s_mn[warp][k] = mn[k];
      s_mx[warp][k] = mx[k];
    }
  }
  __syncthreads();
  if (threadIdx.x < 3u) {
    float a = s_mn[0][threadIdx.x], b = s_mx[0][threadIdx.x];
    for (uint32_t w = 1; w < (blockDim.x >> 5); ++w) {
      a = fminf(a, s_mn[w][threadIdx.x]);
      b = fmaxf(b, s_mx[w][threadIdx.x]);
    }
    atomicMin(&bbox[threadIdx.x], float_to_ordered(a));
    atomicMax(&bbox[3 + threadIdx.x], float_to_ordered(b));
  }
}

__global__ void __launch_bounds__(256) k_grid_keys(const LightVertexRec* pool, uint32_t count, const uint32_t* bbox, float cell_size, uint32_t mask, uint32_t* keys,
  uint32_t* values) {
  uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= count) return;
  V3 bmin = {ordered_to_float(bbox[0]), ordered_to_float(bbox[1]), ordered_to_float(bbox[2])};
  float4 pt = reinterpret_cast<const float4*>(pool + s)[3];
  keys[s] = (__float_as_uint(pt.w) == kInvalidIndex) ? 0xffffffffu : grid_position_to_index({pt.x, pt.y, pt.z}, bmin, cell_size, mask);
  values[s] = s;
}

// after the stable sort by cell: gather photon SoA (60 B -> 4 x 16 B) and mark [begin,end) per cell
template <bool SP>
__global__ void __launch_bounds__(256) k_grid_build(const __grid_constant__ LaunchParams p, const uint32_t* sorted_keys, const uint32_t* sorted_values, uint32_t count, uint2* cell_range,
  float4* pos_dvcm, float4* nrm_dvm, float4* win_len, float4* thr_rgb) {
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= count) return;
  uint32_t key = sorted_keys[j];
  if (key == 0xffffffffu) return;  // medium vertices sort to the end and stay out of the grid
  if ((j == 0) || (sorted_keys[j - 1] != key)) cell_range[key].x = j;
  if ((j + 1 == count) || (sorted_keys[j + 1] != key)) cell_range[key].y = j + 1;
  const float4* src = reinterpret_cast<const float4*>(p.lv_final + sorted_values[j]);
  float4 r0 = src[0], r1 = src[1], r2 = src[2], r3 = src[3], r4 = src[4];
  uint4 ids = reinterpret_cast<const uint4*>(src)[5];
  pos_dvcm[j] = make_float4(r3.x, r3.y, r3.z, r0.w);
  nrm_dvm[j] = make_float4(r4.x, r4.y, r4.z, r2.w);
  win_len[j] = make_float4(r1.x, r1.y, r1.z, __uint_as_float(ids.y));
  // (s.throughput / s.throughput.sampling_pdf()).to_rgb() (vcm_shared.cxx:141); the path's wavelength travels with it
  float wavelength = p.paths.wavelength[ids.z];
  Spec<SP> t = Spec<SP>::make3({r0.x, r0.y, r0.z}) / sampling_pdf<SP>(wavelength);
  V3 rgb = spec_to_rgb<SP>(p.scene, t, wavelength);
  thr_rgb[j] = make_float4(rgb.x, rgb.y, rgb.z, 0.0f);
}

// ---------------------------------------------------------------------------------------------------------------------
// camera pass
// ---------------------------------------------------------------------------------------------------------------------
template <bool SP>
__global__ void __launch_bounds__(128) k_camera_begin(const __grid_constant__ LaunchParams p, uint32_t* queue, uint32_t* queue_count) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  bool alive = false;
  if (i < p.path_count) {
    alive = pixel_owned(p, i);
    if (alive) {
      uint32_t px = i % p.film.width, py = i / p.film.width;
      PathState<SP> s = generate_camera_state<SP>(p.scene, p.vcm, px, py, i, p.paths.wavelength[i]);
      p.paths.wavelength[i] = s.wavelength;
      store_state<SP>(p.paths, i, s);
      p.paths.gathered[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      p.paths.merged[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    }
  }
  queue_push(queue, queue_count, alive, i);
}

// Sort key of a merge query: Morton code of its base grid cell, so that queries which read the same photon cells are
// processed back to back (L1/L2 reuse instead of ~19 KB of DRAM traffic per incoherent query).
DEV uint32_t morton_part(uint32_t v) {
  v = (v | (v << 16)) & 0x030000FFu;
  v = (v | (v << 8)) & 0x0300F00Fu;
  v = (v | (v << 4)) & 0x030C30C3u;
  v = (v | (v << 2)) & 0x09249249u;
  return v;
}
DEV uint32_t merge_query_key(const GridData& g, V3 pos) {
  if (!((pos.x >= g.bbox_min.x) && (pos.y >= g.bbox_min.y) && (pos.z >= g.bbox_min.z) && (pos.x <= g.bbox_max.x) && (pos.y <= g.bbox_max.y) && (pos.z <= g.bbox_max.z)))
    return 0xffffffffu;
  V3 m = vfloor((pos - g.bbox_min) / g.cell_size);
  uint32_t x = umin(uint32_t(m.x), 1023u), y = umin(uint32_t(m.y), 1023u), z = umin(uint32_t(m.z), 1023u);
  return morton_part(x) | (morton_part(y) << 1) | (morton_part(z) << 2);
}

// vcm_camera_step after the trace (vcm_shared.hxx:927-1079), split into the wavefront stages
//   shade    : intersection, 6 pre-drawn randoms (+ blue noise), BSDF sample, MIS update, direct hit, vertex connections, NEE
//   merge    : hash-grid photon gather (VCMSpatialGridData::gather, :886-924) — warp-cooperative in the product build
//   continue : vcm_next_ray (RR, recurrences, next ray) or, when the path ends, the epilogue of gather_camera_vertices
//              (vcm_cpu.cxx:195-198) + Film::accumulate_camera_image
// The pending BSDF sample travels between stages in `bs_*` (40 B per path).
// bs_props.x markers for bounces that do not end in a pending BSDF sample (medium scattering, boundary crossing)
constexpr uint32_t kBounceResolvedAlive = 0x80000001u;
constexpr uint32_t kBounceResolvedDead = 0x80000000u;

// bs_props.x flag: the pending sample leaves from a subsurface exit point — the hit record holds the exit, ray_d holds its w_i, and the
// vertex uses the scene's exit material (vcm_shared.hxx:1062-1064)
constexpr uint32_t kBounceSubsurfaceExit = 0x40000000u;

// the camera vertex the merge / continue stages work on, rebuilt from the path's hit record
template <bool SP>
DEV Isect stage_intersection(const LaunchParams& p, const PathState<SP>& state, uint32_t i, float4 hit) {
  Isect isect = make_intersection(p.scene, state.ray_d, __float_as_uint(hit.w), hit.x, hit.y, hit.z);
  if (scene_has_subsurface(p.scene) && (p.paths.bs_props[i].x & kBounceSubsurfaceExit)) isect.material_index = p.scene.subsurface_exit_material;
  return isect;
}

// Scenes with stochastic BSDFs (product build): the camera-vertex x light-vertex connections (vcm_shared.hxx:765-803) become their
// own wavefront stage, one thread per connection (k_camera_connect); the shade stage only emits the work list.
template <bool SP>
DEV void camera_emit_connections(const LaunchParams& p, uint32_t i, uint32_t camera_material, PathState<SP>& state, uint32_t& connections) {
  const DeviceScene& sc = p.scene;
  if (p.vcm.connect_vertices() == false) return;
  uint32_t lp_count = p.paths.lv_count[i];
  uint32_t d2 = state.total_path_depth + 2u;  // target_path_length = depth + k + 2 must lie in [min_path_length, max_path_length]
  uint32_t k_begin = (sc.min_path_length > d2) ? (sc.min_path_length - d2) : 0u;
  uint32_t k_end = (sc.max_path_length >= d2) ? umin(lp_count, sc.max_path_length - d2 + 1u) : 0u;
  if (k_end > k_begin) {
    uint32_t cnt = k_end - k_begin;
    uint32_t base = atomicAdd(p.conn_count, cnt);
    if (base + cnt <= p.conn_capacity) {
      for (uint32_t k = 0; k < cnt; ++k) p.conn_list[base + k] = make_uint2(i, k_begin + k);
      if (p.conn_key != nullptr) {
        uint32_t cam_mat = umin(camera_material, 0xffu) << 8;
        const LightVertexRec* lvs = p.lv_final + p.lp_offset[i] + k_begin;
        for (uint32_t k = 0; k < cnt; ++k) p.conn_key[base + k] = cam_mat | umin(__float_as_uint(__ldg(&lvs[k].nrm_mat.w)), 0xffu);
      }
    } else {
      *p.overflow = 1u;
    }
    p.paths.conn_seed[i] = state.sampler.seed;
    state.sampler.next();  // the path's own stream moves on by one draw for the whole stage
    connections += cnt;
  }
}

// vcm_camera_step (vcm_shared.hxx:921-1080) up to the merge: same three phases as k_light_bounce — (A) the event, (B) connections to
// the paired light path and to a sampled emitter from the endpoint(s) the event produced (one, or every gathered subsurface exit,
// :1037-1053), (C) the MIS update / pending continuation sample handed to the merge and continue stages.
template <bool SP, bool PLAIN>
__global__ void __launch_bounds__(128, kBounceMinBlocks) k_camera_shade(const __grid_constant__ LaunchParams p, const uint32_t* queue_in, const uint32_t* count_in) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t shadow_rays = 0, connections = 0;
  uint32_t merge_key = 0xffffffffu;
  STATS_DECL;
  if (q < *count_in) {
    uint32_t i = queue_in[q];
    const DeviceScene& sc = p.scene;
    PathState<SP> state = load_state<SP>(p.paths, i);
    float4 g = p.paths.gathered[i];
    state.gathered = Spec<SP>::make3({g.x, g.y, g.z});
    float4 hit = p.paths.hit[i];
    uint32_t tri_index = __float_as_uint(hit.w);
    const bool found = tri_index != kInvalidIndex;
    uint2 resolved = make_uint2(kBounceResolvedDead, kInvalidIndex);
    bool pending_sample = false;
    uint32_t ep_mode = kEpNone;
    bool at_medium = false, at_surface = false, is_connectible = false, ss_path = false, ss_sampled = false;
    V2 rnd_bsdf = {0.0f, 0.0f}, rnd_connection = {0.0f, 0.0f}, rnd_support = {0.0f, 0.0f};
    V3 medium_pos = {0.0f, 0.0f, 0.0f};
    Isect isect{};
    BSample<SP> bs;
    SSGather<SP> ssg;
    ssg.count = 0;
    // ---- (A) ----
    MediumSample<SP> medium_sample = vcm_try_sampling_medium<SP, PLAIN>(sc, state, found ? hit.z : kMaxFloat);
    if (medium_sample.sampled_medium() || found) {
      if (medium_sample.sampled_medium()) {
        at_medium = true;
        medium_pos = medium_sample.pos;
      } else {
        isect = make_intersection(sc, state.ray_d, tri_index, hit.x, hit.y, hit.z);
        if (vcm_handle_boundary<SP, PLAIN>(sc, isect, state)) {
          resolved.x = kBounceResolvedAlive;  // :1002-1007
        } else {
          at_surface = true;
        }
      }
      if (at_medium || at_surface) {
        rnd_bsdf = state.sampler.next_2d();
        rnd_connection = state.sampler.next_2d();
        rnd_support = state.sampler.next_2d();
        if (p.vcm.blue_noise && (state.total_path_depth == 1) && (p.vcm.iteration < 256u)) {
          uint32_t px = i % p.film.width, py = i / p.film.width;
          rnd_bsdf = sample_blue_noise(sc, px, py, p.vcm.iteration, 0);
          rnd_connection = sample_blue_noise(sc, px, py, p.vcm.iteration, 2);
          rnd_support = sample_blue_noise(sc, px, py, p.vcm.iteration, 4);
        }
      }
      if (at_medium) {
        // :934-970
        float seg = state.path_distance + medium_sample.sampled_medium_t;
        state.d_vcm *= sqr(seg);
        state.path_distance = 0.0f;
        const DMedium& med = sc.mediums[state.medium_index];
        if (med.enable_explicit_connections && (state.total_path_depth + 1 <= sc.max_path_length)) ep_mode = kEpMedium;
      } else if (at_surface) {
        const etxb_material& mat = sc.materials[isect.material_index];
        BData bsdf_data = make_bdata(isect, isect.w_i, state.wavelength, state.medium_index, kPathCamera);
        state.sampler.push_fixed(rnd_bsdf.x, rnd_bsdf.y, rnd_support.x);
        bs = bsdf_sample<SP>(sc, bsdf_data, mat, state.sampler);
        is_connectible = (bs.properties & kBsdfDelta) == 0;
        state.sampler.pop_fixed();
        // vcm_update_camera_vcm (:589-595)
        float cos_to_prev = fabsf(dot(isect.nrm, -state.ray_d));
        state.d_vcm *= sqr(state.path_distance + isect.t) / cos_to_prev;
        state.d_vc /= cos_to_prev;
        state.d_vm /= cos_to_prev;
        state.path_distance = 0.0f;
        vcm_handle_direct_hit<SP>(sc, p.vcm, isect, state);
        ss_path = scene_has_subsurface<PLAIN>(sc) && (bs.properties & kBsdfDiffuse) && (mat.subsurface.cls != 0u);
        if (ss_path) ss_sampled = ss_gather<SP>(sc, state.wavelength, isect, state.sampler, ssg, stats, shadow_rays);
        if (is_connectible) ep_mode = ss_sampled ? kEpSubsurface : kEpSurface;
      }
    } else {
      vcm_cam_handle_miss<SP>(sc, p.vcm, state.ray_d, state.d_vcm, state.d_vc, state.path_distance, state.total_path_depth, state.wavelength, state.throughput, state.gathered);
    }
    // ---- (B) ----
    uint2 shadow_span = make_uint2(0u, 0u);
    if (ep_mode != kEpNone) {
      uint32_t n = (ep_mode == kEpSubsurface) ? ssg.count : 1u;
      Isect ep_isect = isect;
      // deferred shadow rays: reserve one slot per possible segment of this vertex (its light path + the emitter sample)
      ShadowBatch batch = {p.shadow_p0, p.shadow_p1, p.shadow_value, 0u, 0u};
      ShadowBatch* deferred = nullptr;
      uint32_t reserved = 0;
      if (p.shadow_stage && (ep_mode == kEpSurface) && !p.connect_stage) {
        reserved = p.paths.lv_count[i] + 1u;
        batch.base = atomicAdd(p.shadow_count, reserved);
        if (batch.base + reserved <= p.shadow_capacity) deferred = &batch;  // otherwise this vertex traces inline (same result)
      } else if (PLAIN && p.shadow_atomic && (ep_mode == kEpSurface)) {
        // product build, opaque scene: the emitter-sample segment joins the bounce's shadow list; its contribution is added to this path's
        // `gathered` by k_shadow_resolve
        batch.atomic_cursor = p.shadow_count;
        batch.capacity = p.shadow_capacity;
        batch.target = i;
        deferred = &batch;
      }
#pragma unroll 1
      for (uint32_t k = 0; k < n; ++k) {
        Spec<SP> w = Spec<SP>::make(1.0f);
        if (ep_mode == kEpSubsurface) {
          ep_isect = ss_exit_intersection<SP>(sc, ssg, k, sc.subsurface_exit_material);
          w = ssg.weights[k];
        }
        Endpoint ep{ep_mode == kEpMedium, &ep_isect, medium_pos};  // one object behind the pointer: it stays in registers
        // a surface vertex connects to the light path first and to the emitter second; a medium vertex the other way round (:961-970)
#pragma unroll 1
        for (uint32_t step = 0; step < 2u; ++step) {
          Spec<SP> c;
          if ((step == 0u) == (ep_mode == kEpMedium)) {
            state.sampler.push_fixed(rnd_connection.x, rnd_connection.y, rnd_support.y);
            c = vcm_connect_to_light<SP, PLAIN>(sc, p.vcm, ep, state, stats, shadow_rays, deferred);
            state.sampler.pop_fixed();
          } else if (p.connect_stage && (ep_mode == kEpSurface)) {
            camera_emit_connections<SP>(p, i, isect.material_index, state, connections);
            continue;
          } else if (deferred) {
            // one slot per connection of this vertex, in the reference's order (vcm_shared.hxx:765-803); k_camera_connect_deferred
            // evaluates each pair in its own thread and fills (or voids) the slot — no BSDF of such a scene draws from the sampler
            if (p.vcm.connect_vertices()) {
              uint32_t lp_count = p.paths.lv_count[i];
              uint32_t d2 = state.total_path_depth + 2u;  // target_path_length = depth + k + 2 must lie in [min_path_length, max_path_length]
              uint32_t k_begin = (sc.min_path_length > d2) ? (sc.min_path_length - d2) : 0u;
              uint32_t k_end = (sc.max_path_length >= d2) ? umin(lp_count, sc.max_path_length - d2 + 1u) : 0u;
              for (uint32_t k = k_begin; k < k_end; ++k) p.conn_list[batch.base + batch.count++] = make_uint2(i, k);
              connections += batch.count;
            }
            shadow_span.y = batch.count;
            continue;
          } else {
            // reference order: serial over the paired path's vertices with the path's own sampler
            c = vcm_connect_to_light_path<SP, PLAIN>(sc, p.vcm, p.lv_final, p.lp_offset[i], p.paths.lv_count[i], ep, state, stats, shadow_rays, connections);
          }
          state.gathered += (ep_mode == kEpSubsurface) ? (w * c) : c;
        }
      }
      if (reserved) {
        if (deferred) {
          shadow_span.x = batch.base;
          shadow_span.y |= (batch.count - shadow_span.y) << 16;
        }
        // reserved slots that were not used (failed connections, or a reservation that ran past the capacity) are marked empty
        for (uint32_t k = batch.base + batch.count; (k < batch.base + reserved) && (k < p.shadow_capacity); ++k) p.shadow_p0[k].w = -1.0f;
        // slots that are no vertex connection (the emitter segment, unused ones) carry no pair
        for (uint32_t k = batch.base + (shadow_span.y & 0xffffu); (k < batch.base + reserved) && (k < p.shadow_capacity); ++k) p.conn_list[k].x = kInvalidIndex;
      }
    }
    if (p.shadow_stage) p.paths.shadow_span[i] = shadow_span;
    // ---- (C) ----
    if (at_medium) {
      // :974-995
      const DMedium& med = sc.mediums[state.medium_index];
      V3 w_o_smp = sample_phase_function(state.ray_d, med.phase_function_g, rnd_bsdf);
      float pdf_fwd = phase_function(state.ray_d, w_o_smp, med.phase_function_g);
      float pdf_rev = phase_function(w_o_smp, state.ray_d, med.phase_function_g);
      state.d_vc = (1.0f / pdf_fwd) * (state.d_vc * pdf_rev + state.d_vcm);
      state.d_vm = (1.0f / pdf_fwd) * (state.d_vm * pdf_rev + 0.0f);
      state.d_vcm = 1.0f / pdf_fwd;
      state.ray_o = medium_pos;
      state.ray_d = w_o_smp;
      state.ray_max_t = kMaxFloat;
      state.ray_min_t = kRayEpsilon;
      state.total_path_depth += 1;
      bool cont = !(state.total_path_depth + 1 > sc.max_path_length) &&
                  random_continue<SP>(state.total_path_depth, sc.random_path_termination, state.eta, state.sampler, state.throughput);
      resolved.x = cont ? kBounceResolvedAlive : kBounceResolvedDead;
    } else if (at_surface) {
      uint32_t ss_flag = 0u;
      if (ss_sampled) {
        // :1056-1067 — the vertex moves to the selected exit: the hit record, w_i (kept in ray_d) and the pending cosine-lobe sample are
        // rewritten for the merge and continue stages
        state.throughput *= ssg.weights[ssg.selected] * ssg.selected_sample_weight;
        isect = ss_exit_intersection<SP>(sc, ssg, ssg.selected, sc.subsurface_exit_material);
        bs.w_o = sample_cosine_around(state.sampler.next_2d(), isect.nrm, 1.0f);
        bs.pdf = fabsf(dot(bs.w_o, isect.nrm)) / kPi;
        bs.eta = 1.0f;
        HitRec h = ssg.hits[ssg.selected];
        p.paths.hit[i] = make_float4(h.u, h.v, h.t, __uint_as_float(h.tri));
        state.ray_d = ssg.w_i[ssg.selected];
        ss_flag = kBounceSubsurfaceExit;
      }
      if (is_connectible && p.vcm.merge_vertices() && (state.total_path_depth + 1 <= sc.max_path_length) && (p.grid.photon_count != 0u)) {
        merge_key = merge_query_key(p.grid, isect.pos);
        // material-major order of the gather queue, so that the warps in flight evaluate ONE BSDF class at a time (the generic gather waited on
        // instruction fetch, profiles/r1b_c3_k_*.raw.csv; measured on the B200, round 2: C3 generic gather 60.6 -> 46.1 ms per iteration)
        if (p.merge_material_major && (merge_key != 0xffffffffu)) merge_key = (umin(isect.material_index, 0x7eu) << 24) | (merge_key >> 6);
      }
      V3 w = bs.weight.as_v3();
      p.paths.bs_weight_pdf[i] = make_float4(w.x, w.y, w.z, bs.pdf);
      p.paths.bs_wo_eta[i] = make_float4(bs.w_o.x, bs.w_o.y, bs.w_o.z, bs.eta);
      p.paths.bs_props[i] = make_uint2(bs.properties | ss_flag, bs.medium_index);
      pending_sample = !(ss_path && !ss_sampled);  // a failed walk ends the path after the merge (:1072-1074)
    }
    if (!pending_sample) p.paths.bs_props[i] = resolved;
    store_state<SP>(p.paths, i, state);
    V3 gv = state.gathered.as_v3();
    p.paths.gathered[i] = make_float4(gv.x, gv.y, gv.z, 0.0f);
    p.paths.merge_key[q] = merge_key;
  }
  counter_add(&p.counters->bounces_camera, (q < *count_in) ? 1u : 0u);
  counter_add(&p.counters->rays_shadow, shadow_rays);
  counter_add(&p.counters->connections, connections);
  counter_add(&p.counters->nodes, STATS_NODES);
  counter_add(&p.counters->tris, STATS_TRIS);
}

// vcm_connect_to_light_vertex (vcm_shared.hxx:673-763) on vertex closures: both end points are prepared once and each closure_evaluate returns
// value, pdf and reverse pdf together (the generic routine re-derives IORs / thin film / tints from the Material record in each of its four
// evaluate / reverse_pdf calls).  Surface camera vertices only; the light vertex may be a medium vertex.
template <bool SP>
DEV bool vcm_connect_to_light_vertex_closure(const DeviceScene& sc, const VcmParams& it, PathState<SP>& state, const LightVertexRec& lv, const Isect& cam, V3& target_position,
  Spec<SP>& value) {
  const uint32_t lv_tri = __float_as_uint(lv.pos_tri.w);
  const bool lv_is_medium = lv_tri == kInvalidIndex;
  const V3 lv_wi = {lv.wi_dvc.x, lv.wi_dvc.y, lv.wi_dvc.z};
  Isect light_v = {};
  TriRec light_tri = {};
  if (lv_is_medium == false) {
    light_tri = load_triangle(sc, lv_tri);
    V3 bc = {lv.bc_dvm.x, lv.bc_dvm.y, lv.bc_dvm.z};
    lerp_vertex(sc, light_tri, bc, light_v.pos, light_v.nrm, light_v.tan, light_v.btn, light_v.tex);
  }
  target_position = lv_is_medium ? V3{lv.pos_tri.x, lv.pos_tri.y, lv.pos_tri.z} : light_v.pos;
  V3 w_o = target_position - cam.pos;
  float distance_squared = dot(w_o, w_o);
  if (distance_squared <= kEpsilon) return false;
  w_o /= sqrtf(distance_squared);
  float w_dot_l = 1.0f;
  if (lv_is_medium == false) w_dot_l = -dot(light_v.nrm, w_o);

  BData camera_data = make_bdata(cam, cam.w_i, state.wavelength, state.medium_index, kPathCamera);
  Closure<SP> cc = make_closure<SP>(sc, camera_data, cam.material_index, state.sampler);
  CEval<SP> ce = closure_evaluate<SP>(sc, cc, w_o, state.sampler);
  if (ce.valid() == false) return false;
  const float camera_area_pdf = ce.pdf * fabsf(w_dot_l) / distance_squared;

  float light_area_pdf = 0.0f, light_rev_pdf = 0.0f;
  Spec<SP> light_scatter = Spec<SP>::make(0.0f);
  if (lv_is_medium) {
    float pf = medium_phase(sc, lv.ids.x, lv_wi, -w_o);
    if (pf <= 0.0f) return false;
    light_area_pdf = pf * fabsf(dot(cam.nrm, w_o)) / distance_squared;
    light_rev_pdf = medium_phase(sc, lv.ids.x, -w_o, lv_wi);
    light_scatter = Spec<SP>::make(pf);
  } else {
    BData light_data = {light_v.pos, light_v.nrm, light_v.tan, light_v.btn, light_v.tex, lv_wi, state.wavelength, kPathLight, state.medium_index};
    Closure<SP> lc = make_closure<SP>(sc, light_data, __float_as_uint(lv.nrm_mat.w), state.sampler);
    CEval<SP> le = closure_evaluate<SP>(sc, lc, -w_o, state.sampler);
    if (le.valid() == false) return false;
    light_area_pdf = le.pdf * fabsf(dot(cam.nrm, w_o)) / distance_squared;
    light_rev_pdf = le.rev_pdf;
    light_scatter = le.bsdf * fix_shading_normal(light_tri.geo_n, light_data.nrm, light_data.w_i, -w_o);
  }
  float vmW_pair = lv_is_medium ? 0.0f : it.vm_weight;
  float w_light = camera_area_pdf * (vmW_pair + lv.thr_dvcm.w + lv.wi_dvc.w * light_rev_pdf);
  float w_camera = light_area_pdf * (vmW_pair + state.d_vcm + state.d_vc * ce.rev_pdf);
  float weight = it.enable_mis() ? 1.0f / (1.0f + w_light + w_camera) : 1.0f;
  Spec<SP> lv_throughput = Spec<SP>::make3({lv.thr_dvcm.x, lv.thr_dvcm.y, lv.thr_dvcm.z});
  value = (ce.bsdf * state.throughput) * (light_scatter * lv_throughput) * (weight / distance_squared);
  return true;
}

// Product build: one thread per (camera vertex, light vertex) connection — vcm_connect_to_light_vertex + the shadow ray of
// vcm_connect_to_light_path (vcm_shared.hxx:673-803).  Each connection draws from its own stream derived from the path's sampler
// (the reference shares one stream across the serial loop; the parity build keeps that order inside k_camera_shade).
template <bool SP, bool PLAIN>
__global__ void __launch_bounds__(128, kConnectMinBlocks) k_camera_connect(const __grid_constant__ LaunchParams p, const uint2* conn_list) {
  uint32_t shadow_rays = 0;
  STATS_DECL;
  const DeviceScene& sc = p.scene;
  // grid-stride over the device-side pair count: the host sizes the grid by the count when it has read it (long queues) and by the
  // queue size when it has not (the tail of a pass runs without a host round trip per bounce)
  const uint32_t total = umin(*p.conn_count, p.conn_capacity);
  for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += gridDim.x * blockDim.x) {
    uint2 entry = conn_list[t];
    uint32_t i = entry.x;
    PathState<SP> state = load_state<SP>(p.paths, i);
    float4 hit = p.paths.hit[i];
    Isect isect = make_intersection(sc, state.ray_d, __float_as_uint(hit.w), hit.x, hit.y, hit.z);
    state.sampler.seed = p.paths.conn_seed[i] ^ ((entry.y + 1u) * 0x9E3779B1u);
    state.sampler.next();
    LightVertexRec lv = load_light_vertex(p.lv_final + p.lp_offset[i] + entry.y);
    Endpoint ep{false, &isect, {0.0f, 0.0f, 0.0f}};
    V3 target_position;
    Spec<SP> value;
#if defined(ETXB_PARITY) && ETXB_PARITY
    const bool connected = vcm_connect_to_light_vertex<SP>(sc, p.vcm, state, lv, ep, target_position, value);
#else
    const bool connected = vcm_connect_to_light_vertex_closure<SP>(sc, p.vcm, state, lv, isect, target_position, value);
#endif
    if (connected && PLAIN && p.shadow_atomic) {
      shadow_rays += 1;
      V3 p0 = shading_pos(sc, load_triangle(sc, isect.triangle_index), isect.barycentric, normalize(target_position - isect.pos));
      ShadowBatch batch = {p.shadow_p0, p.shadow_p1, p.shadow_value, 0u, 0u, p.shadow_count, p.shadow_capacity, i};
      batch.push<SP>(p0, target_position, value);
    } else if (connected) {
      shadow_rays += 1;
      Spec<SP> tr = vcm_connection_transmittance<SP, PLAIN>(sc, ep, lv, target_position, state, stats);
      if (tr.is_zero() == false) {
        V3 v = (tr * value).as_v3();
        float* dst = reinterpret_cast<float*>(p.paths.gathered + i);
        atomicAdd(dst + 0, v.x);
        if (!SP) {
          atomicAdd(dst + 1, v.y);
          atomicAdd(dst + 2, v.z);
        }
      }
    }
  }
  counter_add(&p.counters->rays_shadow, shadow_rays);
  counter_add(&p.counters->nodes, STATS_NODES);
  counter_add(&p.counters->tris, STATS_TRIS);
}

// Scenes with deferred shadow rays (no stochastic BSDF, no media): the connections of vcm_connect_to_light_path (vcm_shared.hxx:765-803)
// one per thread.  Shadow slot `t` of the bounce was reserved by the shade stage; conn_list[t] names its (path, light vertex) pair.  A
// connection that succeeds writes the slot's segment and unoccluded contribution (k_shadow_trace resolves it, k_camera_continue adds the
// visible ones in slot order = reference order); one that fails voids the slot.  Same values, same order as the serial loop.
template <bool SP>
__global__ void __launch_bounds__(128, kConnectMinBlocks) k_camera_connect_deferred(const __grid_constant__ LaunchParams p) {
  const uint32_t total = umin(p.shadow_count[0], p.shadow_capacity);
  const DeviceScene& sc = p.scene;
  uint32_t shadow_rays = 0;
  for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += gridDim.x * blockDim.x) {
    uint2 entry = p.conn_list[t];
    if (entry.x == kInvalidIndex) continue;
    uint32_t i = entry.x;
    PathState<SP> state = load_state<SP>(p.paths, i);
    float4 hit = p.paths.hit[i];
    Isect isect = make_intersection(sc, state.ray_d, __float_as_uint(hit.w), hit.x, hit.y, hit.z);
    LightVertexRec lv = load_light_vertex(p.lv_final + p.lp_offset[i] + entry.y);
    Endpoint ep{false, &isect, {0.0f, 0.0f, 0.0f}};
    V3 target_position;
    Spec<SP> value;
    if (vcm_connect_to_light_vertex<SP>(sc, p.vcm, state, lv, ep, target_position, value)) {
      V3 p0 = shading_pos(sc, load_triangle(sc, isect.triangle_index), isect.barycentric, normalize(target_position - isect.pos));
      V3 c = value.as_v3();
      p.shadow_p0[t] = make_float4(p0.x, p0.y, p0.z, 0.0f);
      p.shadow_p1[t] = make_float4(target_position.x, target_position.y, target_position.z, 0.0f);
      p.shadow_value[t] = make_float4(c.x, c.y, c.z, 0.0f);
      shadow_rays += 1;
    } else {
      p.shadow_p0[t].w = -1.0f;  // not traced; "visible" with a zero contribution
      p.shadow_value[t] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      p.shadow_result[t] = 0u;
    }
  }
  counter_add(&p.counters->rays_shadow, shadow_rays);
}

// Lambert surfaces (Diffuse, variation 0: bsdf_various.hxx:36-133) evaluate without touching the sampler and their BSDF value does
// not depend on the photon direction, so the product build gathers them with the whole warp: one query at a time is broadcast,
// the 32 lanes test 32 photons of a cell per step (coalesced 16-B position loads), accepted lanes finish the MIS weight, and the
// partial sums are reduced with shuffles.  Any other material class (stochastic evaluate) and the parity build take the serial,
// reference-ordered path.
DEV bool merge_is_lambert(const etxb_material& m) { return (m.cls == ETXB_MAT_DIFFUSE) && (m.diffuse_variation == 0u); }

// Serial, reference-ordered gather (VCMSpatialGridData::gather): every merging vertex in the parity build, the non-Lambert
// ones (stochastic evaluate consuming the path's sampler) in the product build.
template <bool SP>
__global__ void __launch_bounds__(128) k_camera_merge_serial(const __grid_constant__ LaunchParams p, const uint32_t* queue_in, const uint32_t* count_in) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  const DeviceScene& sc = p.scene;
  uint32_t merge_queries = 0, candidates = 0, accepts = 0;
  if ((q < *count_in) && (p.paths.merge_key[q] != 0xffffffffu)) {
    uint32_t i = queue_in[q];
    float4 hit = p.paths.hit[i];
    uint32_t tri_index = __float_as_uint(hit.w);
    PathState<SP> state = load_state<SP>(p.paths, i);
    Isect isect = stage_intersection<SP>(p, state, i, hit);
#if defined(ETXB_PARITY) && ETXB_PARITY
    const bool mine = true;
#else
    const bool mine = !merge_is_lambert(sc.materials[isect.material_index]);
#endif
    if (mine) {
      merge_queries = 1;
      V3 m = grid_gather<SP>(sc, p.grid, p.vcm, isect, state, candidates, accepts);
      float4 mg = p.paths.merged[i];
      p.paths.merged[i] = make_float4(mg.x + m.x, mg.y + m.y, mg.z + m.z, 0.0f);
      p.paths.misc[i].x = state.sampler.seed;
    }
  }
  counter_add(&p.counters->merge_queries, merge_queries);
  counter_add(&p.counters->merge_candidates, candidates);
  counter_add(&p.counters->merge_accepts, accepts);
}

// Warp-cooperative Lambert gather (product build).  Input: the queue sorted by merge_query_key.  One query at a time is
// broadcast to the warp; the eight cell ranges are concatenated into one virtual range that the 32 lanes sweep with coalesced
// 16-B position loads; photons inside the radius are compacted (ballot + prefix) into a per-warp shared list and finished 32 at
// a time with all lanes busy (normal / path-length / cosine tests, MIS weight, kernel); partial sums meet in a shuffle reduction.
constexpr uint32_t kMergeWarpsPerBlock = 8;
constexpr uint32_t kMergeListSize = 64;

// Lambert camera vertices only (BSDF value independent of the photon direction, no sampler use); k_camera_merge_closure gathers the others.
template <bool SP>
__global__ void __launch_bounds__(kMergeWarpsPerBlock * 32) k_camera_merge_coop(const __grid_constant__ LaunchParams p, const uint32_t* sorted_ids, const uint32_t* sorted_keys, const uint32_t* count_in,
                                                                                uint32_t queries_per_warp) {
  __shared__ uint32_t s_idx[kMergeWarpsPerBlock][kMergeListSize];
  __shared__ float s_d2[kMergeWarpsPerBlock][kMergeListSize];
  __shared__ float s_dvcm[kMergeWarpsPerBlock][kMergeListSize];
  const DeviceScene& sc = p.scene;
  const GridData& g = p.grid;
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t lane_lt = (1u << lane) - 1u;
  // A warp works through its queries one after the other, so a query's latency is paid `queries_per_warp` times per warp: 32 when the
  // queue is long (every lane brings one query), fewer when it is short (the tail of the pass), so that the queries spread over more warps.
  uint32_t q = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * queries_per_warp + lane;
  uint32_t merge_queries = 0, candidates = 0, accepts = 0;
  bool coop_active = (lane < queries_per_warp) && (q < *count_in) && (sorted_keys[q] != 0xffffffffu);
  uint32_t i = 0;
  V3 qpos = {0, 0, 0}, qnrm = {0, 0, 0}, qfn = {0, 0, 0}, qc = {0, 0, 0};
  float q_wcam_base = 0.0f, q_dvm = 0.0f, q_rev_cos = 0.0f;
  uint32_t q_depth = 0;
  if (coop_active) {
    i = sorted_ids[q];
    float4 hit = p.paths.hit[i];
    PathState<SP> state = load_state<SP>(p.paths, i);
    Isect isect = stage_intersection<SP>(p, state, i, hit);
    const etxb_material& mat = sc.materials[isect.material_index];
    coop_active = merge_is_lambert(mat);
    if (coop_active) {
      merge_queries = 1;
      qpos = isect.pos;
      qnrm = isect.nrm;
      q_wcam_base = state.d_vcm * p.vcm.vc_weight;
      q_dvm = state.d_vm;
      q_depth = state.total_path_depth;
      Spec<SP> t_camera = state.throughput / sampling_pdf<SP>(state.wavelength);
      bool entering = dot(isect.nrm, isect.w_i) < 0.0f;
      qfn = entering ? isect.nrm : -isect.nrm;  // frame normal of the camera vertex
      Spec<SP> diffuse = apply_image<SP>(sc, mat.scattering, isect.tex, state.wavelength);
      qc = spec_to_rgb<SP>(sc, (diffuse / kPi) * t_camera, state.wavelength);  // camera_bsdf.func * t_camera: direction independent
      q_rev_cos = dot(isect.nrm, -isect.w_i);  // reverse pdf = cos between -w_i(camera) and the normal facing the photon (bsdf_various.hxx:113-121)
    }
  }
  uint32_t pending = __ballot_sync(0xffffffffu, coop_active);
  V3 my_sum = {0.0f, 0.0f, 0.0f};
  const bool use_mis = p.vcm.enable_mis();
  const bool use_epan = (p.vcm.kernel == 1u);
  const float vc_weight = p.vcm.vc_weight;
  while (pending) {
    uint32_t src = __ffs(pending) - 1u;
    pending &= pending - 1u;
    V3 bpos = {__shfl_sync(0xffffffffu, qpos.x, src), __shfl_sync(0xffffffffu, qpos.y, src), __shfl_sync(0xffffffffu, qpos.z, src)};
    V3 bnrm = {__shfl_sync(0xffffffffu, qnrm.x, src), __shfl_sync(0xffffffffu, qnrm.y, src), __shfl_sync(0xffffffffu, qnrm.z, src)};
    V3 bfn = {__shfl_sync(0xffffffffu, qfn.x, src), __shfl_sync(0xffffffffu, qfn.y, src), __shfl_sync(0xffffffffu, qfn.z, src)};
    V3 bqc = {__shfl_sync(0xffffffffu, qc.x, src), __shfl_sync(0xffffffffu, qc.y, src), __shfl_sync(0xffffffffu, qc.z, src)};
    float b_wcam_base = __shfl_sync(0xffffffffu, q_wcam_base, src);
    float b_dvm = __shfl_sync(0xffffffffu, q_dvm, src);
    float b_rev_cos = __shfl_sync(0xffffffffu, q_rev_cos, src);
    uint32_t b_depth = __shfl_sync(0xffffffffu, q_depth, src);
    // the eight cells (vcm_shared.hxx:895-916): lanes 0..7 fetch their ranges, then an 8-wide exclusive scan of the counts
    // (prefetching the next query's ranges and the next 32 candidate positions was measured: no gain, the sweep is L2-bandwidth bound)
    uint32_t my_begin = 0, my_cnt = 0;
    if (lane < 8u) {
      V3 m = (bpos - g.bbox_min) / g.cell_size;
      V3 mf = vfloor(m);
      V3 md = m - mf;
      int32_t acx = static_cast<int32_t>(mf.x), acy = static_cast<int32_t>(mf.y), acz = static_cast<int32_t>(mf.z);
      int32_t cx = (lane & 1u) ? acx + ((md.x < 0.5f) ? -1 : +1) : acx;
      int32_t cy = (lane & 2u) ? acy + ((md.y < 0.5f) ? -1 : +1) : acy;
      int32_t cz = (lane & 4u) ? acz + ((md.z < 0.5f) ? -1 : +1) : acz;
      uint2 r = __ldg(&g.cell_range[grid_cell_index(g.hash_table_mask, cx, cy, cz)]);
      my_begin = r.x;
      my_cnt = r.y - r.x;
    }
    uint32_t incl = my_cnt;
#pragma unroll
    for (uint32_t o = 1; o < 8u; o <<= 1) {
      uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    uint32_t my_excl = incl - my_cnt;
    const uint32_t total = __shfl_sync(0xffffffffu, incl, 7);
    uint32_t e1 = __shfl_sync(0xffffffffu, my_excl, 1), e2 = __shfl_sync(0xffffffffu, my_excl, 2), e3 = __shfl_sync(0xffffffffu, my_excl, 3),
             e4 = __shfl_sync(0xffffffffu, my_excl, 4), e5 = __shfl_sync(0xffffffffu, my_excl, 5), e6 = __shfl_sync(0xffffffffu, my_excl, 6),
             e7 = __shfl_sync(0xffffffffu, my_excl, 7);
    float wx = 0.0f, wy = 0.0f, wz = 0.0f;  // per-lane partial sums
    uint32_t n_list = 0;                    // warp-uniform fill of the shared list

    auto finish = [&](uint32_t n) {
      // lanes < n take one photon that passed the radius test
      if (lane < n) {
        uint32_t j = s_idx[warp][lane];
        float distance_squared = s_d2[warp][lane];
        float dvcm = s_dvcm[warp][lane];
        float4 wl = __ldg(&g.win_len[j]);
        float4 nd = __ldg(&g.nrm_dvm[j]);
        float4 lt = __ldg(&g.thr_rgb[j]);
        bool ok = !(__float_as_uint(wl.w) + b_depth + 1 > sc.max_path_length);
        ok = ok && !(dot(bnrm, V3{nd.x, nd.y, nd.z}) <= kEpsilon);
        float cos_o = -(bfn.x * wl.x + bfn.y * wl.y + bfn.z * wl.z);  // local_w_o.z of DiffuseBSDF::evaluate(-w_in)
        ok = ok && (cos_o > kEpsilon);
        float bsdf_pdf_v = kInvPi * cos_o;
        float facing = (dot(bnrm, V3{wl.x, wl.y, wl.z}) < 0.0f) ? b_rev_cos : -b_rev_cos;
        float rev_pdf = (facing <= kEpsilon) ? 0.0f : kInvPi * facing;
        if (ok) {
          float w_light = dvcm * vc_weight + nd.w * bsdf_pdf_v;
          float w_camera = b_wcam_base + b_dvm * rev_pdf;
          float weight = use_mis ? (1.0f / (1.0f + w_light + w_camera)) : 1.0f;
          float kernel_weight = use_epan ? fmaxf(2.0f * (1.0f - distance_squared * g.inv_radius_squared), 0.0f) : 1.0f;
          float kw = kernel_weight * weight;
          wx += lt.x * kw;
          wy += lt.y * kw;
          wz += lt.z * kw;
          accepts += 1;
        }
      }
    };

    for (uint32_t base = 0; base < total; base += 32u) {
      uint32_t k = base + lane;
      bool valid = k < total;
      uint32_t c = uint32_t(k >= e1) + uint32_t(k >= e2) + uint32_t(k >= e3) + uint32_t(k >= e4) + uint32_t(k >= e5) + uint32_t(k >= e6) + uint32_t(k >= e7);
      uint32_t cb = __shfl_sync(0xffffffffu, my_begin, c);
      uint32_t ce = __shfl_sync(0xffffffffu, my_excl, c);
      uint32_t j = cb + (k - ce);
      bool inside = false;
      float distance_squared = 0.0f, dvcm = 0.0f;
      if (valid) {
        float4 pd = __ldg(&g.pos_dvcm[j]);
        V3 d = V3{pd.x, pd.y, pd.z} - bpos;
        distance_squared = dot(d, d);
        dvcm = pd.w;
        inside = !(distance_squared > g.radius_squared);
        candidates += 1;
      }
      uint32_t bal = __ballot_sync(0xffffffffu, inside);
      if (inside) {
        uint32_t slot = n_list + __popc(bal & lane_lt);
        s_idx[warp][slot] = j;
        s_d2[warp][slot] = distance_squared;
        s_dvcm[warp][slot] = dvcm;
      }
      n_list += __popc(bal);
      __syncwarp();
      if (n_list >= 32u) {
        finish(32u);
        __syncwarp();
        uint32_t rest = n_list - 32u;  // < 32: move the tail to the front
        uint32_t tj = 0;
        float td = 0.0f, tv = 0.0f;
        if (lane < rest) {
          tj = s_idx[warp][32u + lane];
          td = s_d2[warp][32u + lane];
          tv = s_dvcm[warp][32u + lane];
        }
        __syncwarp();
        if (lane < rest) {
          s_idx[warp][lane] = tj;
          s_d2[warp][lane] = td;
          s_dvcm[warp][lane] = tv;
        }
        n_list = rest;
        __syncwarp();
      }
    }
    if (n_list) finish(n_list);
    __syncwarp();
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      wx += __shfl_xor_sync(0xffffffffu, wx, o);
      wy += __shfl_xor_sync(0xffffffffu, wy, o);
      wz += __shfl_xor_sync(0xffffffffu, wz, o);
    }
    if (lane == src) {
      V3 l = {wx, wy, wz};
      if (SP) l *= V3{0.817660332f, 1.05418909f, 1.09945524f};  // kRGBLuminanceScale (:876-878)
      my_sum = qc * l;
    }
  }
  if (merge_queries) {
    float4 mg = p.paths.merged[i];
    p.paths.merged[i] = make_float4(mg.x + my_sum.x, mg.y + my_sum.y, mg.z + my_sum.z, 0.0f);
  }
  counter_add(&p.counters->merge_queries, merge_queries);
  counter_add(&p.counters->merge_candidates, candidates);
  counter_add(&p.counters->merge_accepts, accepts);
}

// Product build, scenes with stochastic BSDFs: the generic gather on vertex closures (dclosure.cuh).  The evaluations are batched ACROSS
// the queries of a warp: the (query, photon) pairs of all its queries go through one shared list, 32 pairs per step whatever query they
// belong to, and the contributions meet in per-query shared accumulators.  The camera vertex of a query is PREPARED once (material record ->
// evaluated IORs, thin film, roughness, tints: a Closure in shared memory) instead of being re-derived from the Material inside every
// evaluate / pdf call of every pair, and one closure_evaluate returns value, pdf and reverse pdf together.  Each in-radius photon is
// evaluated with a lane-local sampler derived from (path seed, photon index) and the path's sampler advances by one draw per query —
// statistically equivalent to the reference's serial order (which the parity build keeps), 32x more parallel.
constexpr uint32_t kClosureWarpsPerBlock = 4;
constexpr int kClosureMinBlocks = 4;
struct MergeQueryAux {
  float qc[3];  // t_camera = throughput / pdf(lambda)
  float wcam_base, dvm;
  uint32_t depth, seed;
};
template <bool SP>
__global__ void __launch_bounds__(kClosureWarpsPerBlock * 32, kClosureMinBlocks) k_camera_merge_closure(const __grid_constant__ LaunchParams p, const uint32_t* sorted_ids, const uint32_t* sorted_keys, const uint32_t* count_in,
                                                                                     uint32_t queries_per_warp) {
  __shared__ Closure<SP> s_cl[kClosureWarpsPerBlock][32];
  __shared__ MergeQueryAux s_aux[kClosureWarpsPerBlock][32];
  __shared__ uint32_t s_idx[kClosureWarpsPerBlock][kMergeListSize];
  __shared__ float s_d2[kClosureWarpsPerBlock][kMergeListSize];
  __shared__ float s_dvcm[kClosureWarpsPerBlock][kMergeListSize];
  __shared__ uint32_t s_src[kClosureWarpsPerBlock][kMergeListSize];
  __shared__ float s_sum[kClosureWarpsPerBlock][32][3];
  constexpr uint32_t kFull = 0xffffffffu;
  const DeviceScene& sc = p.scene;
  const GridData& g = p.grid;
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t lane_lt = (1u << lane) - 1u;
  uint32_t q = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * queries_per_warp + lane;
  uint32_t merge_queries = 0, candidates = 0, accepts = 0;
  bool active = (lane < queries_per_warp) && (q < *count_in) && (sorted_keys[q] != 0xffffffffu);
  uint32_t i = 0;
  V3 qpos = {0, 0, 0};
  if (active) {
    i = sorted_ids[q];
    float4 hit = p.paths.hit[i];
    PathState<SP> state = load_state<SP>(p.paths, i);
    Isect isect = stage_intersection<SP>(p, state, i, hit);
    active = !merge_is_lambert(sc.materials[isect.material_index]);
    if (active) {
      merge_queries = 1;
      qpos = isect.pos;
      MergeQueryAux aux;
      V3 t_camera = (state.throughput / sampling_pdf<SP>(state.wavelength)).as_v3();
      aux.qc[0] = t_camera.x;
      aux.qc[1] = t_camera.y;
      aux.qc[2] = t_camera.z;
      aux.wcam_base = state.d_vcm * p.vcm.vc_weight;
      aux.dvm = state.d_vm;
      aux.depth = state.total_path_depth;
      aux.seed = state.sampler.seed;
      state.sampler.next();  // the path's own stream moves on by one draw per query
      p.paths.misc[i].x = state.sampler.seed;
      Smp prep;  // the closure's own stream (RGB thin-film wavelength jitter)
      prep.seed = aux.seed ^ 0x85ebca6bu;
      prep.fixed_u = prep.fixed_v = prep.fixed_w = 0.0f;
      prep.next();
      BData cam = make_bdata(isect, isect.w_i, state.wavelength, state.medium_index, kPathCamera);
      s_cl[warp][lane] = make_closure<SP>(sc, cam, isect.material_index, prep);
      s_aux[warp][lane] = aux;
    }
  }
  s_sum[warp][lane][0] = 0.0f;
  s_sum[warp][lane][1] = 0.0f;
  s_sum[warp][lane][2] = 0.0f;
  __syncwarp();
  uint32_t pending = __ballot_sync(kFull, active);
  const bool use_mis = p.vcm.enable_mis();
  const bool use_epan = (p.vcm.kernel == 1u);
  const float vc_weight = p.vcm.vc_weight;
  uint32_t n_list = 0;  // warp-uniform fill of the shared pair list

  auto finish = [&](uint32_t n) {
    if (lane < n) {
      const uint32_t j = s_idx[warp][lane], s = s_src[warp][lane];
      const float distance_squared = s_d2[warp][lane], dvcm = s_dvcm[warp][lane];
      const Closure<SP>& c = s_cl[warp][s];
      const MergeQueryAux& aux = s_aux[warp][s];
      float4 wl = __ldg(&g.win_len[j]);
      float4 nd = __ldg(&g.nrm_dvm[j]);
      bool ok = !(__float_as_uint(wl.w) + aux.depth + 1 > sc.max_path_length);
      ok = ok && !(dot(c.nrm, V3{nd.x, nd.y, nd.z}) <= kEpsilon);
      if (ok) {
        Smp lane_smp;
        lane_smp.seed = aux.seed ^ ((j + 1u) * 0x9E3779B1u);
        lane_smp.fixed_u = lane_smp.fixed_v = lane_smp.fixed_w = 0.0f;
        lane_smp.next();
        CEval<SP> e = closure_evaluate<SP>(sc, c, V3{-wl.x, -wl.y, -wl.z}, lane_smp);
        if (e.valid()) {
          float4 lt = __ldg(&g.thr_rgb[j]);
          V3 c_value = spec_to_rgb<SP>(sc, e.func * Spec<SP>::make3(V3{aux.qc[0], aux.qc[1], aux.qc[2]}), c.wavelength);
          float w_light = dvcm * vc_weight + nd.w * e.pdf;
          float w_camera = aux.wcam_base + aux.dvm * e.rev_pdf;
          float weight = use_mis ? (1.0f / (1.0f + w_light + w_camera)) : 1.0f;
          float kernel_weight = use_epan ? fmaxf(2.0f * (1.0f - distance_squared * g.inv_radius_squared), 0.0f) : 1.0f;
          float kw = kernel_weight * weight;
          atomicAdd(&s_sum[warp][s][0], c_value.x * lt.x * kw);
          atomicAdd(&s_sum[warp][s][1], c_value.y * lt.y * kw);
          atomicAdd(&s_sum[warp][s][2], c_value.z * lt.z * kw);
          accepts += 1;
        }
      }
    }
  };

  while (pending) {
    uint32_t src = __ffs(pending) - 1u;
    pending &= pending - 1u;
    V3 bpos = {__shfl_sync(kFull, qpos.x, src), __shfl_sync(kFull, qpos.y, src), __shfl_sync(kFull, qpos.z, src)};
    // the eight cells (vcm_shared.hxx:895-916): lanes 0..7 fetch their ranges, then an 8-wide exclusive scan of the counts
    uint32_t my_begin = 0, my_cnt = 0;
    if (lane < 8u) {
      V3 m = (bpos - g.bbox_min) / g.cell_size;
      V3 mf = vfloor(m);
      V3 md = m - mf;
      int32_t acx = static_cast<int32_t>(mf.x), acy = static_cast<int32_t>(mf.y), acz = static_cast<int32_t>(mf.z);
      int32_t cx = (lane & 1u) ? acx + ((md.x < 0.5f) ? -1 : +1) : acx;
      int32_t cy = (lane & 2u) ? acy + ((md.y < 0.5f) ? -1 : +1) : acy;
      int32_t cz = (lane & 4u) ? acz + ((md.z < 0.5f) ? -1 : +1) : acz;
      uint2 r = __ldg(&g.cell_range[grid_cell_index(g.hash_table_mask, cx, cy, cz)]);
      my_begin = r.x;
      my_cnt = r.y - r.x;
    }
    uint32_t incl = my_cnt;
#pragma unroll
    for (uint32_t o = 1; o < 8u; o <<= 1) {
      uint32_t v = __shfl_up_sync(kFull, incl, o);
      if (lane >= o) incl += v;
    }
    uint32_t my_excl = incl - my_cnt;
    const uint32_t total = __shfl_sync(kFull, incl, 7);
    uint32_t e1 = __shfl_sync(kFull, my_excl, 1), e2 = __shfl_sync(kFull, my_excl, 2), e3 = __shfl_sync(kFull, my_excl, 3), e4 = __shfl_sync(kFull, my_excl, 4),
             e5 = __shfl_sync(kFull, my_excl, 5), e6 = __shfl_sync(kFull, my_excl, 6), e7 = __shfl_sync(kFull, my_excl, 7);
    for (uint32_t base = 0; base < total; base += 32u) {
      uint32_t k = base + lane;
      bool valid = k < total;
      uint32_t c = uint32_t(k >= e1) + uint32_t(k >= e2) + uint32_t(k >= e3) + uint32_t(k >= e4) + uint32_t(k >= e5) + uint32_t(k >= e6) + uint32_t(k >= e7);
      uint32_t cb = __shfl_sync(kFull, my_begin, c);
      uint32_t ce = __shfl_sync(kFull, my_excl, c);
      uint32_t j = cb + (k - ce);
      bool inside = false;
      float distance_squared = 0.0f, dvcm = 0.0f;
      if (valid) {
        float4 pd = __ldg(&g.pos_dvcm[j]);
        V3 d = V3{pd.x, pd.y, pd.z} - bpos;
        distance_squared = dot(d, d);
        dvcm = pd.w;
        inside = !(distance_squared > g.radius_squared);
        candidates += 1;
      }
      uint32_t bal = __ballot_sync(kFull, inside);
      if (inside) {
        uint32_t slot = n_list + __popc(bal & lane_lt);
        s_idx[warp][slot] = j;
        s_d2[warp][slot] = distance_squared;
        s_dvcm[warp][slot] = dvcm;
        s_src[warp][slot] = src;
      }
      n_list += __popc(bal);
      __syncwarp();
      if (n_list >= 32u) {
        finish(32u);
        __syncwarp();
        uint32_t rest = n_list - 32u;  // < 32: move the tail to the front
        uint32_t tj = 0, ts = 0;
        float td = 0.0f, tv = 0.0f;
        if (lane < rest) {
          tj = s_idx[warp][32u + lane];
          td = s_d2[warp][32u + lane];
          tv = s_dvcm[warp][32u + lane];
          ts = s_src[warp][32u + lane];
        }
        __syncwarp();
        if (lane < rest) {
          s_idx[warp][lane] = tj;
          s_d2[warp][lane] = td;
          s_dvcm[warp][lane] = tv;
          s_src[warp][lane] = ts;
        }
        n_list = rest;
        __syncwarp();
      }
    }
  }
  if (n_list) finish(n_list);
  __syncwarp();
  if (merge_queries) {
    V3 l = {s_sum[warp][lane][0], s_sum[warp][lane][1], s_sum[warp][lane][2]};
    if (SP) l *= V3{0.817660332f, 1.05418909f, 1.09945524f};  // kRGBLuminanceScale (:876-878)
    float4 mg = p.paths.merged[i];
    p.paths.merged[i] = make_float4(mg.x + l.x, mg.y + l.y, mg.z + l.z, 0.0f);
  }
  counter_add(&p.counters->merge_queries, merge_queries);
  counter_add(&p.counters->merge_candidates, candidates);
  counter_add(&p.counters->merge_accepts, accepts);
}

// Candidate test of the closest-hit walk (Raytracing::trace, rt.cxx:428-466): Void surfaces and alpha-rejected hits are skipped, any other
// candidate becomes the closest hit so far.
struct ClosestHitVisitor {
  const DeviceScene& sc;
  Smp* smp;
  HitRec* best;
  DEV int operator()(uint32_t triangle_index, float u, float v, float t) {
    const etxb_material& mat = sc.materials[load_triangle_material(sc, triangle_index)];
    if (mat.cls == ETXB_MAT_VOID) return kCandIgnore;
    if (alpha_test_rejects(sc, mat, triangle_index, u, v, *smp)) return kCandIgnore;
    *best = {u, v, t, triangle_index};
    return kCandAccept;
  }
};

// Closest hit through the 4-wide quantised tree (dwide.cuh), one ray per thread: the product build's kernel for scenes with stochastic BSDFs.
__global__ void __launch_bounds__(256) k_trace_closest_wide(const __grid_constant__ LaunchParams p, const uint32_t* queue, const uint32_t* queue_count, uint32_t* material_keys,
                                                            uint32_t key_limit) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= *queue_count) {
    if ((material_keys != nullptr) && (q < key_limit)) material_keys[q] = kQueueKeyPastCount;
    return;
  }
  uint32_t i = queue[q];
  float4 o = p.paths.ray_o[i], d = p.paths.ray_d[i];
  Smp smp;
  smp.seed = p.paths.misc[i].x;
  smp.fixed_u = smp.fixed_v = smp.fixed_w = 0.0f;
  HitRec best = {0.0f, 0.0f, 0.0f, kInvalidIndex};
  ClosestHitVisitor visit{p.scene, &smp, &best};
  const WideNodes nodes{nullptr, p.scene.wide_nodes, 0u};
  WideWalk walk;
  WideHit stack[kWideStackSize];
  uint32_t n_nodes = 0, n_tris = 0;
  wide_begin(walk, {o.x, o.y, o.z}, {d.x, d.y, d.z}, o.w, d.w);
  while (!wide_step(walk, stack, nodes, p.scene.bvh_tris, visit, n_nodes, n_tris)) {
  }
  p.paths.hit[i] = make_float4(best.u, best.v, best.t, __uint_as_float(best.tri));
  p.paths.misc[i].x = smp.seed;
  if (material_keys != nullptr) material_keys[q] = queue_sort_key(p, best.tri);
  counter_add(&p.counters->rays_closest, 1u);
#ifdef ETXB_COUNT_TRAVERSAL
  counter_add(&p.counters->nodes, n_nodes);
  counter_add(&p.counters->tris, n_tris);
  counter_add(&p.counters->nodes_closest, n_nodes);
  counter_add(&p.counters->tris_closest, n_tris);
#endif
}

// One CTA of kTraversalBlock threads per SM: the staged nodelet then costs 32 KB of the SM's shared memory / L1 once (four 256-thread CTAs each
// staging their own copy took 128 KB away from the L1 that caches the rest of the tree: ncu, L1 hit rate 64 % -> 46 %, and the kernel got slower).
constexpr uint32_t kTraversalBlock = 1024u;

// The shadow segments of one bounce (ShadowBatch, atomic mode): any-hit on a persistent, nodelet-staged, lane-refilled walk (dtrav.cuh); a segment
// that reaches its end adds its contribution to its target (a path's gathered sum, or a pixel of the light image).  Opaque scenes only: any
// non-Void surface on the segment occludes (rt.cxx:468-579 without Boundary crossings).
template <bool WIDE>
__global__ void __launch_bounds__(kTraversalBlock) k_shadow_resolve(const __grid_constant__ LaunchParams p, uint32_t* cursor) {
  // 32 KB of shared memory: the top kNodeletNodes nodes of the tree this instantiation walks (both node types are 64 bytes)
  __shared__ __align__(128) BvhNode s_nodes[kNodeletNodes];
  __shared__ __align__(8) uint64_t s_bar;
  static_assert(sizeof(WideNode) == sizeof(BvhNode), "one staging buffer serves both trees");
  const uint32_t staged = WIDE ? nodelet_stage(s_nodes, &s_bar, reinterpret_cast<const BvhNode*>(p.scene.wide_nodes), p.scene.wide_node_count)
                               : nodelet_stage(s_nodes, &s_bar, p.scene.bvh_nodes, p.scene.bvh_node_count);
  const StagedNodes nodes{s_nodes, p.scene.bvh_nodes, staged};
  const WideNodes wide_nodes{reinterpret_cast<const WideNode*>(s_nodes), p.scene.wide_nodes, staged};
  const uint32_t total = umin(p.shadow_count[0], p.shadow_capacity);
  bool active = false, exhausted = false;
  uint32_t k = 0, n_nodes = 0, n_tris = 0, splats = 0;
  RayWalk walk;
  WideWalk wide_walk;
  int32_t stack[WIDE ? 1 : kBvhStackSize];
  WideHit wide_stack[WIDE ? kWideStackSize : 1];
  OcclusionVisitor visit{p.scene, false};
  auto contribute = [&](uint32_t slot, uint32_t target) {
    float4 v = p.shadow_value[slot];
    if (target & kShadowTargetPixel) {
      splat_add(p, target & ~kShadowTargetPixel, V3{v.x, v.y, v.z});
      splats += 1u;
    } else {
      float* dst = reinterpret_cast<float*>(p.paths.gathered + target);
      atomicAdd(dst + 0, v.x);
      if (p.scene.spectral == 0u) {
        atomicAdd(dst + 1, v.y);
        atomicAdd(dst + 2, v.z);
      }
    }
  };
  uint32_t target = 0;
  for (;;) {
    uint32_t next = 0;
    if (warp_refill(!active, cursor, total, next, exhausted)) {
      k = next;
      float4 a = p.shadow_p0[k], b = p.shadow_p1[k];
      target = reinterpret_cast<const uint32_t*>(p.shadow_p1 + k)[3];  // raw bits (see ShadowBatch::push_rgb)
      V3 direction = V3{b.x, b.y, b.z} - V3{a.x, a.y, a.z};
      float t_max = dot(direction, direction);
      if (t_max <= kRayEpsilon) {
        contribute(k, target);  // a degenerate segment is unoccluded (rt.cxx:474-477)
      } else {
        t_max = sqrtf(t_max);
        direction /= t_max;
        t_max -= fmaxf(kRayEpsilon, t_max * kRayEpsilon);
        if constexpr (WIDE) {
          wide_begin(wide_walk, {a.x, a.y, a.z}, direction, kRayEpsilon, t_max);
        } else {
          walk.begin({a.x, a.y, a.z}, direction, kRayEpsilon, t_max);
        }
        visit.occluded = false;
        active = true;
      }
    }
    if (!__any_sync(0xffffffffu, active)) {
      if (exhausted) break;
      continue;
    }
    while (active) {
      bool done;
      if constexpr (WIDE) {
        done = wide_step(wide_walk, wide_stack, wide_nodes, p.scene.bvh_tris, visit, n_nodes, n_tris);
      } else {
        done = walk_step(walk, stack, nodes, p.scene.bvh_tris, visit, n_nodes, n_tris);
      }
      if (done) {
        if (!visit.occluded) contribute(k, target);
        active = false;
      } else if (!exhausted && (__popc(__activemask()) < kRefillLanes)) {
        break;
      }
    }
  }
  counter_add(&p.counters->splats, splats);
#ifdef ETXB_COUNT_TRAVERSAL
  counter_add(&p.counters->nodes, n_nodes);
  counter_add(&p.counters->tris, n_tris);
#endif
}

// The deferred shadow rays of one camera bounce (ShadowBatch, dvcm.cuh): a traversal-only kernel — persistent warps take 32 segments at a
// time from a shared cursor, every lane answers "is anything but a Void surface on this segment?".
__global__ void __launch_bounds__(256) k_shadow_trace(const __grid_constant__ LaunchParams p) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t total = umin(p.shadow_count[0], p.shadow_capacity);
  for (;;) {
    uint32_t base = 0;
    if (lane == 0) base = atomicAdd(p.shadow_count + 1, 32u);
    base = __shfl_sync(0xffffffffu, base, 0);
    if (base >= total) break;
    uint32_t k = base + lane;
    if (k < total) {
      float4 a = p.shadow_p0[k];
      if (a.w >= 0.0f) {
        float4 b = p.shadow_p1[k];
        p.shadow_result[k] = trace_occluded(p.scene, V3{a.x, a.y, a.z}, V3{b.x, b.y, b.z}) ? 1u : 0u;
      }
    }
  }
}

template <bool SP>
__global__ void __launch_bounds__(128) k_camera_continue(const __grid_constant__ LaunchParams p, const uint32_t* queue_in, const uint32_t* count_in, uint32_t* queue_out, uint32_t* count_out) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  bool alive = false;
  uint32_t i = 0;
  if (q < *count_in) {
    i = queue_in[q];
    const DeviceScene& sc = p.scene;
    PathState<SP> state = load_state<SP>(p.paths, i);
    float4 hit = p.paths.hit[i];
    uint32_t tri_index = __float_as_uint(hit.w);
    uint2 bp = p.paths.bs_props[i];
    if (p.shadow_stage) {
      // resolve the vertex's deferred shadow rays: visible contributions are added in the reference's order (the sum over the light path
      // first, vcm_shared.hxx:765-803, then the emitter sample), and the sampler moves on by one draw per occluded segment
      uint2 span = p.paths.shadow_span[i];
      uint32_t n_path = span.y & 0xffffu, n_total = n_path + (span.y >> 16);
      if (n_total) {
        float4 g = p.paths.gathered[i];
        Spec<SP> gathered = Spec<SP>::make3({g.x, g.y, g.z});
        Spec<SP> path_sum = Spec<SP>::make(0.0f);
        for (uint32_t k = 0; k < n_total; ++k) {
          if (k == n_path) gathered += path_sum;
          if (p.shadow_result[span.x + k]) {
            state.sampler.next();
          } else {
            float4 v = p.shadow_value[span.x + k];
            Spec<SP> c = Spec<SP>::make3({v.x, v.y, v.z});
            if (k < n_path) {
              path_sum += c;
            } else {
              gathered += c;
            }
          }
        }
        if (n_total == n_path) gathered += path_sum;
        V3 gv = gathered.as_v3();
        p.paths.gathered[i] = make_float4(gv.x, gv.y, gv.z, 0.0f);
      }
    }
    if (bp.x & 0x80000000u) {
      alive = bp.x == kBounceResolvedAlive;  // medium scattering / boundary crossing / miss: the shade stage already advanced the path
    } else if (tri_index != kInvalidIndex) {
      Isect isect = stage_intersection<SP>(p, state, i, hit);
      BData bsdf_data = make_bdata(isect, isect.w_i, state.wavelength, state.medium_index, kPathCamera);
      float4 bw = p.paths.bs_weight_pdf[i], bd = p.paths.bs_wo_eta[i];
      BSample<SP> bs;
      bs.weight = Spec<SP>::make3({bw.x, bw.y, bw.z});
      bs.pdf = bw.w;
      bs.w_o = {bd.x, bd.y, bd.z};
      bs.eta = bd.w;
      bs.properties = bp.x & ~kBounceSubsurfaceExit;
      bs.medium_index = bp.y;
      alive = vcm_next_ray<SP>(sc, false, state, p.vcm, isect, bsdf_data, bs, (bp.x & kBounceSubsurfaceExit) != 0u);
    }
    if (alive) {
      store_state<SP>(p.paths, i, state);
    } else {
      // vcm_cpu.cxx:195-198 + Film::accumulate_camera_image (film.cxx:173-230, camera layer)
      float4 g = p.paths.gathered[i], mg = p.paths.merged[i];
      V3 merged = {mg.x, mg.y, mg.z};
      merged *= p.vcm.vm_normalization;
      merged += spec_to_rgb<SP>(sc, Spec<SP>::make3({g.x, g.y, g.z}) / sampling_pdf<SP>(state.wavelength), state.wavelength);
      uint32_t px = i % p.film.width, py = i / p.film.width;
      uint32_t fi = px + (p.film.height - 1u - py) * p.film.width;
      float4 old = p.film.camera[fi];
      V3 result = merged;
      if (p.camera_sample_index != 0u) {
        double ds = double(p.camera_sample_index);
        float t = float(ds / (ds + 1.0));
        result = {lerpf(merged.x, old.x, t), lerpf(merged.y, old.y, t), lerpf(merged.z, old.z, t)};
      }
      p.film.camera[fi] = make_float4(result.x, result.y, result.z, 1.0f);
      p.sampler_end_camera[i] = state.sampler.seed;
      p.camera_value[i] = make_float4(merged.x, merged.y, merged.z, 0.0f);
    }
  }
  queue_push(queue_out, count_out, alive, i);
}

// ---------------------------------------------------------------------------------------------------------------------
// film (film.cxx:332-343, 381-418)
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_film_commit_light(const __grid_constant__ FilmBuffers film, uint32_t iteration_index) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= film.width * film.height) return;
  float t = float(double(iteration_index) / double(iteration_index + 1u));
  float4 s = film.light_iteration[i], d = film.light[i];
  V3 sv = {s.x, s.y, s.z}, dv = {d.x, d.y, d.z};
  V3 r = (t == 0.0f) ? sv : lerp3(sv, dv, t);
  film.light[i] = make_float4(r.x, r.y, r.z, 1.0f);
  film.light_iteration[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
}

__global__ void __launch_bounds__(256) k_film_resolve(const __grid_constant__ FilmBuffers film, float4* out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= film.width * film.height) return;
  float4 c = film.camera[i], l = film.light[i];
  out[i] = make_float4(fmaxf(0.0f, c.x + l.x), fmaxf(0.0f, c.y + l.y), fmaxf(0.0f, c.z + l.z), 1.0f);
}

// ---------------------------------------------------------------------------------------------------------------------
// debug / known-answer kernels
// ---------------------------------------------------------------------------------------------------------------------
__global__ void k_debug_trace(const __grid_constant__ DeviceScene sc, const float* rays, uint32_t* seeds, uint32_t count, float* hits_uv_t, uint32_t* hits_tri) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const float* r = rays + size_t(i) * 8;
  Smp smp;
  smp.seed = seeds[i];
  smp.fixed_u = smp.fixed_v = smp.fixed_w = 0.0f;
  HitRec h = trace_closest(sc, {r[0], r[1], r[2]}, {r[4], r[5], r[6]}, r[3], r[7], smp, nullptr);
  seeds[i] = smp.seed;
  hits_tri[i] = h.tri;
  bool hit = h.tri != kInvalidIndex;
  hits_uv_t[size_t(i) * 3 + 0] = hit ? h.u : 0.0f;
  hits_uv_t[size_t(i) * 3 + 1] = hit ? h.v : 0.0f;
  hits_uv_t[size_t(i) * 3 + 2] = hit ? h.t : 0.0f;
}

// the same query through the 4-wide quantised tree (product build, scenes that have one)
__global__ void k_debug_trace_wide(const __grid_constant__ DeviceScene sc, const float* rays, uint32_t* seeds, uint32_t count, float* hits_uv_t, uint32_t* hits_tri) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const float* r = rays + size_t(i) * 8;
  Smp smp;
  smp.seed = seeds[i];
  smp.fixed_u = smp.fixed_v = smp.fixed_w = 0.0f;
  HitRec h = {0.0f, 0.0f, 0.0f, kInvalidIndex};
  ClosestHitVisitor visit{sc, &smp, &h};
  const WideNodes nodes{nullptr, sc.wide_nodes, 0u};
  WideWalk walk;
  WideHit stack[kWideStackSize];
  uint32_t n_nodes = 0, n_tris = 0;
  wide_begin(walk, {r[0], r[1], r[2]}, {r[4], r[5], r[6]}, r[3], r[7]);
  while (!wide_step(walk, stack, nodes, sc.bvh_tris, visit, n_nodes, n_tris)) {
  }
  seeds[i] = smp.seed;
  hits_tri[i] = h.tri;
  bool hit = h.tri != kInvalidIndex;
  hits_uv_t[size_t(i) * 3 + 0] = hit ? h.u : 0.0f;
  hits_uv_t[size_t(i) * 3 + 1] = hit ? h.v : 0.0f;
  hits_uv_t[size_t(i) * 3 + 2] = hit ? h.t : 0.0f;
}

__global__ void k_debug_sampler(const uint32_t* a, const uint32_t* b, uint32_t count, uint32_t draws, uint32_t* out_seed, float* out_values) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  Smp s;
  s.init(a[i], b[i]);
  out_seed[size_t(i) * (draws + 1u)] = s.seed;
  for (uint32_t d = 0; d < draws; ++d) {
    out_values[size_t(i) * draws + d] = s.next();
    out_seed[size_t(i) * (draws + 1u) + d + 1u] = s.seed;
  }
}

__global__ void k_debug_math(const __grid_constant__ DeviceScene sc, uint32_t fn, const float* x, const float* y, uint32_t count, float* out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  float a = x[i], b = y ? y[i] : 0.0f, r = 0.0f;
  switch (fn) {
    case 0: r = m_sin(a); break;
    case 1: r = m_cos(a); break;
    case 2: r = m_exp(a); break;
    case 3: r = m_log(a); break;
    case 4: r = m_pow(a, b); break;
    case 5: r = m_acos(a); break;
    case 6: r = m_atan2(a, b); break;
    case 7: r = spectral_sample_wavelength(a); break;
    case 8: r = spectral_sampling_pdf(a); break;
    case 9: r = spec_to_rgb<true>(sc, Spec<true>{1.0f}, a).x; break;
    case 10: r = spec_to_rgb<true>(sc, Spec<true>{1.0f}, a).y; break;
    case 11: r = spec_to_rgb<true>(sc, Spec<true>{1.0f}, a).z; break;
    case 12: r = m_atan(a); break;
    case 13: r = m_asin(a); break;
    case 14: r = sample_blue_noise(sc, uint32_t(a) & 127u, uint32_t(a) >> 7, uint32_t(b), 0).x; break;
    case 15: r = sample_blue_noise(sc, uint32_t(a) & 127u, uint32_t(a) >> 7, uint32_t(b), 4).y; break;
    default: break;
  }
  out[i] = r;
}

}  // namespace etxb
