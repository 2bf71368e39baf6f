// kernels_pt.cuh — wavefront kernels of the unidirectional path tracer (SURVEY §8(f) N3; included once, by module.cu, after kernels.cuh).
//
// Reference: CPUPathTracingImpl::execute_range (sources/etx/rt/integrators/path_tracing.cxx:50-83), run_path_iteration
// (rt/shared/path_tracing_shared.hxx:485-510), Film::accumulate_camera_image with the normal / albedo layers and the adaptive-sampling history
// (render/host/film.cxx:173-230), Film::active_pixel (:434-461), Film::estimate_noise_levels (:233-330).
//
// Stage list of one iteration:
//   k_pt_begin -> { k_trace_closest* -> [sort by material] -> k_pt_shade [-> k_shadow_resolve] }* -> k_pt_accumulate -> [k_film_noise_level -> _rows -> _columns]
// The payload lives in the VCM camera path's SoA columns (one PathBuffers allocation serves both integrators): thr.w = sampled_bsdf_pdf,
// mis.x = eta, misc = (seed, path_length, medium, mis_weight), gathered = accumulated, bs_weight_pdf = view_albedo, bs_wo_eta = view_normal.
#pragma once
#include "dpt.cuh"

namespace etxb {

// the film layers only the path tracer writes (film.cxx:14-40) — storage is y-flipped like the camera layer
struct PtFilm {
  float4* normals;
  float4* albedo;
  float4* adaptive;      // StorageCameraAdaptive: the mean over every other sample
  uint32_t* info;        // InternalData: sample_count (bits 0-29), converged (bit 30), tmp (bit 31)
  float* error_level;
  uint32_t* info_next;   // ping-pong partner of `info` for the two dilation passes
};
constexpr uint32_t kPtConverged = 1u << 30u;
constexpr uint32_t kPtTmp = 1u << 31u;
constexpr uint32_t kPtCountMask = kPtConverged - 1u;

template <bool SP>
DEV void pt_store(const PathBuffers& b, uint32_t i, const PtState<SP>& s) {
  V3 t = s.throughput.as_v3(), a = s.accumulated.as_v3();
  b.ray_o[i] = make_float4(s.ray_o.x, s.ray_o.y, s.ray_o.z, s.ray_min_t);
  b.ray_d[i] = make_float4(s.ray_d.x, s.ray_d.y, s.ray_d.z, s.ray_max_t);
  b.thr[i] = make_float4(t.x, t.y, t.z, s.sampled_bsdf_pdf);
  b.mis[i] = make_float4(s.eta, 0.0f, 0.0f, 0.0f);
  b.misc[i] = make_uint4(s.smp.seed, s.path_length, s.medium, s.mis_weight ? 1u : 0u);
  b.gathered[i] = make_float4(a.x, a.y, a.z, 0.0f);
}
template <bool SP>
DEV PtState<SP> pt_load(const PathBuffers& b, uint32_t i) {
  PtState<SP> s;
  float4 o = b.ray_o[i], d = b.ray_d[i], t = b.thr[i], a = b.gathered[i];
  uint4 u = b.misc[i];
  s.ray_o = {o.x, o.y, o.z};
  s.ray_min_t = o.w;
  s.ray_d = {d.x, d.y, d.z};
  s.ray_max_t = d.w;
  s.throughput = Spec<SP>::make3({t.x, t.y, t.z});
  s.sampled_bsdf_pdf = t.w;
  s.accumulated = Spec<SP>::make3({a.x, a.y, a.z});
  s.eta = b.mis[i].x;
  s.smp.seed = u.x;
  s.smp.fixed_u = s.smp.fixed_v = s.smp.fixed_w = 0.0f;
  s.path_length = u.y;
  s.medium = u.z;
  s.mis_weight = (u.w & 1u) != 0u;
  s.wavelength = b.wavelength[i];
  s.view_albedo = Spec<SP>::make(0.0f);
  s.view_normal = {0.0f, 0.0f, 0.0f};
  return s;
}

DEV uint32_t pt_film_index(const FilmBuffers& film, uint32_t i) {
  uint32_t px = i % film.width, py = i / film.width;
  return px + (film.height - 1u - py) * film.width;
}

// make_ray_payload for every active pixel (path_tracing.cxx:57-62; Film::active_pixel with pixel_size == 1: a converged pixel is skipped)
template <bool SP>
__global__ void __launch_bounds__(128) k_pt_begin(const __grid_constant__ LaunchParams p, const __grid_constant__ PtParams pt, const __grid_constant__ PtFilm pf, uint32_t* queue,
                                                  uint32_t* queue_count) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  bool alive = false;
  if (i < p.path_count) {
    alive = pixel_owned(p, i) && ((pf.info[pt_film_index(p.film, i)] & kPtConverged) == 0u);
    if (alive) {
      PtState<SP> s = pt_make_payload<SP>(p.scene, pt, i % p.film.width, i / p.film.width, i);
      p.paths.wavelength[i] = s.wavelength;
      pt_store<SP>(p.paths, i, s);
      p.paths.bs_weight_pdf[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      p.paths.bs_wo_eta[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      // run_path_iteration's first test (:486): a path longer than the limit is not traced at all
      alive = s.path_length <= p.scene.max_path_length;
      if (!alive) p.sampler_end_camera[i] = s.smp.seed;
    } else {
      // a pixel that is skipped (converged, or another rank's tile) has no path in this iteration: its debug taps read zero, like the oracle's
      p.sampler_end_camera[i] = 0u;
      p.camera_value[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    }
  }
  queue_push(queue, queue_count, alive, i);
}

// run_path_iteration after the trace (:485-510): medium event, surface hit or miss.  A path that goes on is queued for the next bounce; one that
// ends leaves its sums in the path columns for k_pt_accumulate.
template <bool SP, bool PLAIN>
__global__ void __launch_bounds__(128, kBounceMinBlocks) k_pt_shade(const __grid_constant__ LaunchParams p, const __grid_constant__ PtParams pt, const uint32_t* queue_in,
                                                                           const uint32_t* count_in, uint32_t* queue_out, uint32_t* count_out) {
  uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t shadow_rays = 0, i = 0;
  bool alive = false;
  STATS_DECL;
  if (q < *count_in) {
    i = queue_in[q];
    const DeviceScene& sc = p.scene;
    PtState<SP> s = pt_load<SP>(p.paths, i);
    float4 hit = p.paths.hit[i];
    const uint32_t tri_index = __float_as_uint(hit.w);
    const bool found = tri_index != kInvalidIndex;
    MediumSample<SP> ms;
    ms.weight = Spec<SP>::make(0.0f);
    ms.pos = {0.0f, 0.0f, 0.0f};
    ms.sampled_medium_t = 0.0f;
    if constexpr (!PLAIN) {
      if (s.medium != kInvalidIndex) {  // try_sampling_medium (:259-268)
        ms = sample_medium<SP>(sc, sc.mediums[s.medium], s.wavelength, s.throughput, s.smp, s.ray_o, s.ray_d, found ? hit.z : kMaxFloat);
        s.throughput *= ms.weight;
      }
    }
    if (ms.sampled_medium()) {
      if constexpr (!PLAIN) {
        pt_handle_sampled_medium<SP, PLAIN>(sc, pt, ms, s, stats, shadow_rays);
        alive = random_continue<SP>(s.path_length, sc.random_path_termination, s.eta, s.smp, s.throughput);
      }
    } else if (found) {
      Isect isect = make_intersection(sc, s.ray_d, tri_index, hit.x, hit.y, hit.z);
      ShadowBatch batch = {p.shadow_p0, p.shadow_p1, p.shadow_value, 0u, 0u};
      ShadowBatch* deferred = nullptr;
      if (PLAIN && p.shadow_atomic) {
        batch.atomic_cursor = p.shadow_count;
        batch.capacity = p.shadow_capacity;
        batch.target = i;
        deferred = &batch;
      }
      const bool first = s.path_length == 1u;
      alive = pt_handle_hit_ray<SP, PLAIN>(sc, pt, isect, i % p.film.width, i / p.film.width, s, stats, shadow_rays, deferred);
      if (first) {
        V3 a = s.view_albedo.as_v3();
        p.paths.bs_weight_pdf[i] = make_float4(a.x, a.y, a.z, 0.0f);
        p.paths.bs_wo_eta[i] = make_float4(s.view_normal.x, s.view_normal.y, s.view_normal.z, 0.0f);
      }
    } else if (pt.direct) {
      pt_handle_missed_ray<SP>(sc, s);
    }
    // the next run_path_iteration call starts with the length test (:486)
    alive = alive && (s.path_length <= sc.max_path_length);
    pt_store<SP>(p.paths, i, s);
    if (!alive) p.sampler_end_camera[i] = s.smp.seed;
  }
  queue_push(queue_out, count_out, alive, i);
  counter_add(&p.counters->bounces_camera, (q < *count_in) ? 1u : 0u);
  counter_add(&p.counters->rays_shadow, shadow_rays);
  counter_add(&p.counters->nodes, STATS_NODES);
  counter_add(&p.counters->tris, STATS_TRIS);
}

// The end of execute_range's loop body (path_tracing.cxx:68-81) + Film::accumulate_camera_image (film.cxx:173-230) for every pixel that was
// active in this iteration: colour, normal and albedo running means, the every-other-sample mean the noise estimate compares against, the
// per-pixel sample counter.
template <bool SP>
__global__ void __launch_bounds__(256) k_pt_accumulate(const __grid_constant__ LaunchParams p, const __grid_constant__ PtParams pt, const __grid_constant__ PtFilm pf) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.path_count) return;
  const uint32_t fi = pt_film_index(p.film, i);
  const uint32_t info = pf.info[fi];
  if (!pixel_owned(p, i) || (info & kPtConverged)) return;
  const float wavelength = p.paths.wavelength[i];
  float4 acc = p.paths.gathered[i], alb = p.paths.bs_weight_pdf[i], nrm = p.paths.bs_wo_eta[i];
  const float pdf = sampling_pdf<SP>(wavelength);
  V3 normal = {nrm.x, nrm.y, nrm.z};
  V3 albedo = spec_to_rgb<SP>(p.scene, Spec<SP>::make3({alb.x, alb.y, alb.z}) / pdf, wavelength);
  V3 color = spec_to_rgb<SP>(p.scene, Spec<SP>::make3({acc.x, acc.y, acc.z}) / pdf, wavelength);
  if ((pt.radiance_clamp > 0.0f) && (p.paths.misc[i].y > 1u)) {
    float lum = luminance(color);
    if (lum > pt.radiance_clamp) color *= pt.radiance_clamp / lum;
  }
  const uint32_t sample_index = info & kPtCountMask;
  float4 c_old = p.film.camera[fi], n_old = pf.normals[fi], a_old = pf.albedo[fi], v_old = pf.adaptive[fi];
  V3 c = color, n = normal, a = albedo, v = color;
  if (sample_index != 0u) {
    double ds = double(sample_index);
    float t = float(ds / (ds + 1.0));
    c = {lerpf(color.x, c_old.x, t), lerpf(color.y, c_old.y, t), lerpf(color.z, c_old.z, t)};
    n = {lerpf(normal.x, n_old.x, t), lerpf(normal.y, n_old.y, t), lerpf(normal.z, n_old.z, t)};
    a = {lerpf(albedo.x, a_old.x, t), lerpf(albedo.y, a_old.y, t), lerpf(albedo.z, a_old.z, t)};
    v = {v_old.x, v_old.y, v_old.z};
    if ((sample_index % 2u) == 0u) {
      t = float(ds / (ds + 2.0));
      v = {lerpf(color.x, v_old.x, t), lerpf(color.y, v_old.y, t), lerpf(color.z, v_old.z, t)};
    }
  }
  p.film.camera[fi] = make_float4(c.x, c.y, c.z, 1.0f);
  pf.normals[fi] = make_float4(n.x, n.y, n.z, 1.0f);
  pf.albedo[fi] = make_float4(a.x, a.y, a.z, 1.0f);
  pf.adaptive[fi] = make_float4(v.x, v.y, v.z, 1.0f);
  pf.info[fi] = (info & ~kPtCountMask) | ((sample_index + 1u) & kPtCountMask);
  p.camera_value[i] = make_float4(color.x, color.y, color.z, 0.0f);
}

// Film::estimate_noise_levels (film.cxx:233-330), first pass: error level of every pixel that has not converged, the convergence decision, and
// the two sums noise_level() is made of.  stats[0] = pixels that converged in this pass (the reference's `active_pixels`), stats[1] = bits of the
// float sum of error levels (atomic adds: the summation order is not the reference's, which is itself thread-order dependent).
__global__ void __launch_bounds__(256) k_film_noise_level(const __grid_constant__ FilmBuffers film, const __grid_constant__ PtFilm pf, float threshold, uint32_t* stats) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  float error_level = 0.0f;
  uint32_t converged = 0u;
  if (i < film.width * film.height) {
    uint32_t info = pf.info[i];
    if ((info & kPtConverged) == 0u) {
      float4 c = film.camera[i], a = pf.adaptive[i];
      float error_diff = fabsf(c.x - a.x) + fabsf(c.y - a.y) + fabsf(c.z - a.z);
      float error_norm = fabsf(c.x) + fabsf(c.y) + fabsf(c.z);
      error_level = error_diff / (((error_norm < 1.0f) ? sqrtf(error_norm) : error_norm) + kEpsilon);
      converged = (error_level < threshold) ? 1u : 0u;
      pf.error_level[i] = error_level;
      pf.info[i] = (info & kPtCountMask) | (converged ? (kPtConverged | kPtTmp) : 0u);
    }
  }
  uint32_t n = __reduce_add_sync(0xffffffffu, converged);
  float sum = error_level;
  for (uint32_t o = 16u; o > 0u; o >>= 1u) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  if ((threadIdx.x & 31u) == 0u) {
    if (n) atomicAdd(stats + 0, n);
    if (sum != 0.0f) atomicAdd(reinterpret_cast<float*>(stats + 1), sum);
  }
}

// second pass (:283-298): every pixel that has not converged clears `tmp` of the pixels x - 5 .. x + 4 of its row — as a gather: pixel p loses
// `tmp` when a pixel x in [p - 4, p + 5] of its row has not converged
constexpr int32_t kNoiseBlock = 5;
__global__ void __launch_bounds__(256) k_film_noise_rows(const __grid_constant__ FilmBuffers film, const uint32_t* info_in, uint32_t* info_out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= film.width * film.height) return;
  const int32_t w = int32_t(film.width), x = int32_t(i % film.width), row = int32_t(i / film.width) * w;
  uint32_t info = info_in[i];
  if (info & kPtTmp) {
    for (int32_t q = max(0, x - (kNoiseBlock - 1)); q <= min(w - 1, x + kNoiseBlock); ++q) {
      if ((info_in[row + q] & kPtConverged) == 0u) {
        info &= ~kPtTmp;
        break;
      }
    }
  }
  info_out[i] = info;
}

// third pass (:304-320): every pixel without `tmp` clears `converged` of the pixels y - 5 .. y + 4 of its column
__global__ void __launch_bounds__(256) k_film_noise_columns(const __grid_constant__ FilmBuffers film, const uint32_t* info_in, uint32_t* info_out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= film.width * film.height) return;
  const int32_t w = int32_t(film.width), h = int32_t(film.height), x = int32_t(i % film.width), y = int32_t(i / film.width);
  uint32_t info = info_in[i];
  if (info & kPtConverged) {
    for (int32_t q = max(0, y - (kNoiseBlock - 1)); q <= min(h - 1, y + kNoiseBlock); ++q) {
      if ((info_in[x + q * w] & kPtTmp) == 0u) {
        info &= ~kPtConverged;
        break;
      }
    }
  }
  info_out[i] = info;
}

// Film::layer for the layers the VCM integrator leaves empty (film.cxx:406-414): normals are shown as n * 0.5 + 0.5
__global__ void __launch_bounds__(256) k_film_layer_normals(const float4* normals, float4* out, uint32_t count) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  float4 n = normals[i];
  out[i] = make_float4(n.x * 0.5f + 0.5f, n.y * 0.5f + 0.5f, n.z * 0.5f + 0.5f, 1.0f);
}

// The tone map of the application's LDR export and viewer (app.cxx:268-282, render.cxx:307-320) on the device: 1 - exp(-exposure * c), sRGB
// transfer curve, 8 bits, alpha 255 — a preview frame leaves the GPU as 4 bytes per pixel instead of 16.
__global__ void __launch_bounds__(256) k_film_tonemap(const float4* layer, uint32_t* out_rgba8, uint32_t count, float exposure) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  float4 v = layer[i];
  float c[3] = {v.x, v.y, v.z};
  uint32_t packed = 0xff000000u;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    float tm = 1.0f - expf(-exposure * c[k]);
    float g = (tm <= 0.0031308f) ? (12.92f * tm) : (1.055f * powf(tm, 1.0f / 2.4f) - 0.055f);
    g = (g > 0.0f) ? fminf(g, 1.0f) : 0.0f;
    packed |= uint32_t(255.0f * g) << (8 * k);
  }
  out_rgba8[i] = packed;
}

}  // namespace etxb
