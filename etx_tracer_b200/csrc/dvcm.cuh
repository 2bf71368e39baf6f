// dvcm.cuh — per-path VCM logic: emitter / camera sampling, MIS recurrences, connections, merging.
// Restates sources/etx/rt/shared/vcm_shared.hxx (line refs inline), render/shared/scene_emitters.hxx and
// scene_camera.hxx for the device.  One sampler per path; every consumer draws in the oracle's order.
#pragma once
#include "dbsdf.cuh"
#include "dclosure.cuh"
#include "dtrace.cuh"

namespace etxb {

// VCMOptions bits (vcm_shared.hxx:24-37)
struct VcmParams {
  uint32_t options;
  uint32_t kernel;  // 1 = Epanechnikov
  uint32_t blue_noise;
  uint32_t iteration;
  float current_radius, vm_weight, vc_weight, vm_normalization;
  DEV bool connect_to_camera() const { return options & ETXB_VCM_CONNECT_TO_CAMERA; }
  DEV bool direct_hit() const { return options & ETXB_VCM_DIRECT_HIT; }
  DEV bool connect_to_light() const { return options & ETXB_VCM_CONNECT_TO_LIGHT; }
  DEV bool connect_vertices() const { return options & ETXB_VCM_CONNECT_VERTICES; }
  DEV bool enable_mis() const { return options & ETXB_VCM_ENABLE_MIS; }
  DEV bool enable_merging() const { return options & ETXB_VCM_ENABLE_MERGING; }
  DEV bool merge_vertices() const { return enable_merging() && (options & ETXB_VCM_MERGE_VERTICES); }
};

enum : uint32_t {  // VCMPathState flags (vcm_shared.hxx:92-98)
  kPathDeltaEmitter = 1u << 0u,
  kPathLocalEmitter = 1u << 3u,
  kPathValid = 1u << 4u,
};

// VCMPathState (vcm_shared.hxx:91-150) held in registers between the SoA load and store of a kernel
template <bool SP>
struct PathState {
  Spec<SP> throughput;
  Spec<SP> gathered;
  V3 merged;
  V3 ray_o, ray_d;
  float ray_min_t, ray_max_t;
  Smp sampler;
  float wavelength;
  float path_distance;
  float d_vcm, d_vc, d_vm, eta;
  uint32_t total_path_depth;
  uint32_t medium_index;
  uint32_t flags;
  uint32_t lv_count;  // light vertices stored so far by this path
};

// ---- emitters (scene_emitters.hxx) ---------------------------------------------------------------------------
DEV float collimation_to_exponent(float normalized) {  // scene.hxx:67-71
  float t = saturatef(normalized);
  float denom = sqr(sqr(1.0f - t));
  return 1.0f / fmaxf(kEpsilon, denom);
}
// Distribution::sample (distribution.hxx:16-35)
DEV uint32_t distribution_sample(const etxb_distribution_entry* values, uint32_t count, float rnd) {
  uint32_t b = 0, e = count;
  do {
    uint32_t m = b + (e - b) / 2;
    if (__ldg(&values[m].cdf) >= rnd) {
      e = m;
    } else {
      b = m;
    }
  } while ((e - b) > 1);
  return b;
}
DEV float emitter_discrete_pdf(const DeviceScene& sc, const etxb_emitter& e) { return (e.spectrum_weight * e.additional_weight) / sc.emitter_total_weight; }

template <bool SP>
struct EmitterSample {
  Spec<SP> value;
  V3 barycentric, origin, normal, direction;
  float pdf_sample, pdf_area, pdf_dir, pdf_dir_out;
  uint32_t emitter_index, triangle_index, medium_index;
  bool is_delta, is_distant;
};

// math.hxx:809-823, 952-999, 1023-1034
DEV float distance_to_sphere(V3 r_origin, V3 r_direction, V3 center, float radius) {
  V3 e = r_origin - center;
  float b = dot(r_direction, e);
  float d = (b * b) - dot(e, e) + (radius * radius);
  if (d < 0.0f) return 0.0f;
  d = sqrtf(d);
  float a0 = -b - d;
  float a1 = -b + d;
  return (a0 < 0.0f) ? ((a1 < 0.0f) ? 0.0f : a1) : a0;
}
DEV V2 disk_uv(V3 normal, V3 in_dir, float sz, float csz) {
  V2 pc = {0.0f, 0.0f};
  if (sz != 0.0f) {
    Basis basis = orthonormal_basis(normal);
    pc.x = dot(basis.u, in_dir) / (0.5f * sz * csz);
    pc.y = dot(basis.v, in_dir) / (0.5f * sz * csz);
  }
  return {saturatef(pc.x * 0.5f + 0.5f), saturatef(pc.y * 0.5f + 0.5f)};
}
DEV V3 from_spherical(float phi, float theta) {
  float cos_p = m_cos(phi), sin_p = m_sin(phi), cos_t = m_cos(theta), sin_t = m_sin(theta);
  return {1.0f * cos_p * cos_t, 1.0f * sin_t, 1.0f * sin_p * cos_t};
}
DEV V3 uv_to_direction(V2 uv, float offset_x, float u_scale) {
  float u = uv.x;
  if (u_scale < 0.0f) u = 1.0f - u;
  u = u - offset_x;
  u = u - floorf(u);
  float phi = (u * 2.0f - 1.0f) * kPi;
  float theta = (0.5f - uv.y) * kPi;
  return from_spherical(phi, theta);
}
DEV V2 direction_to_uv(V3 dir, float offset_x, float u_scale) {
  float r = length(dir);
  float phi = m_atan2(dir.z, dir.x);
  float theta = m_asin(dir.y / r);
  float u = (phi / kPi + 1.0f) / 2.0f;
  if (u_scale < 0.0f) u = 1.0f - u;
  u = u + offset_x;
  u = u - floorf(u);
  float v = 0.5f - theta / kPi;
  return {u, v};
}

enum : uint32_t { kEmitterArea = 0u, kEmitterEnvironment = 1u, kEmitterDirectional = 2u };  // EmitterProfile::Class (emitter.hxx:8-13)

// emitter_get_radiance (scene_emitters.hxx:40-112)
template <bool SP>
DEV Spec<SP> emitter_get_radiance(const DeviceScene& sc, const etxb_emitter& em_inst, float wavelength, V3 source_position, V3 target_position, V3 direction, V2 uv,
  bool directly_visible, float& pdf_area, float& pdf_dir, float& pdf_dir_out) {
  pdf_dir = 0.0f;
  pdf_area = 0.0f;
  pdf_dir_out = 0.0f;
  const etxb_emitter_profile& em = sc.emitter_profiles[em_inst.profile];
  if (em_inst.cls == kEmitterDirectional) {
    V3 em_dir = {em.direction[0], em.direction[1], em.direction[2]};
    if ((directly_visible == false) || (em.angular_size <= 0.0f) || (dot(direction, em_dir) < em.angular_size_cosine)) return Spec<SP>::make(0.0f);
    pdf_dir = 1.0f;
    pdf_area = 1.0f / (kPi * sc.bounding_sphere_radius * sc.bounding_sphere_radius);
    pdf_dir_out = pdf_dir * pdf_area;
    V2 duv = disk_uv(em_dir, direction, em.equivalent_disk_size, em.angular_size_cosine);
    Spec<SP> direct_scale = 1.0f / (spectrum_query<SP>(sc, em.emission.spectrum_index, wavelength) * kDoublePi * (1.0f - em.angular_size_cosine));
    return apply_image<SP>(sc, em.emission, duv, wavelength) * direct_scale;
  }
  if (em_inst.cls == kEmitterEnvironment) {
    const DImage& img = sc.images[em.emission.image_index];
    V2 euv = direction_to_uv(direction, img.offset_x, img.scale_x);
    float sin_t = fmaxf(kEpsilon, m_sin(euv.y * kPi));
    float image_pdf = 0.0f;
    Spec<SP> eval = apply_image<SP>(sc, em.emission, euv, wavelength, &image_pdf);
    pdf_area = 1.0f / (kPi * sc.bounding_sphere_radius * sc.bounding_sphere_radius);
    pdf_dir = image_pdf / (2.0f * kPi * kPi * sin_t);
    pdf_dir_out = pdf_area * pdf_dir;
    return eval;
  }
  TriRec tri = load_triangle(sc, em_inst.triangle_index);
  const etxb_material& material = sc.materials[tri.material_index];
  if (dot(tri.geo_n, target_position - source_position) >= 0.0f) return Spec<SP>::make(0.0f);
  pdf_area = 1.0f / em_inst.triangle_area;
  V3 dp = source_position - target_position;
  float distance_squared = dot(dp, dp);
  if (distance_squared > 0.0f) {
    float cos_t = fabsf(dot(dp, tri.geo_n)) / sqrtf(distance_squared);
    float exponent = collimation_to_exponent(material.emission_collimation);
    float cos_tx = directly_visible ? cos_t : m_pow(cos_t, exponent);
    if (cos_tx > kEpsilon) {
      pdf_dir = pdf_area * distance_squared / cos_tx;
      pdf_dir_out = pdf_area * cos_tx * kInvPi;
    }
  }
  return apply_image<SP>(sc, em.emission, uv, wavelength);
}

// sample_emission (scene_emitters.hxx:226-305)
template <bool SP>
DEV EmitterSample<SP> sample_emission(const DeviceScene& sc, float wavelength, Smp& smp) {
  EmitterSample<SP> r;
  r.value = Spec<SP>::make(0.0f);
  r.pdf_area = r.pdf_dir = r.pdf_dir_out = 0.0f;
  r.barycentric = {0.0f, 0.0f, 0.0f};
  r.emitter_index = distribution_sample(sc.emitter_dist, sc.emitter_count + 1u, smp.next());
  r.pdf_sample = __ldg(&sc.emitter_dist[r.emitter_index].pdf);
  const etxb_emitter& em_inst = sc.emitters[r.emitter_index];
  const etxb_emitter_profile& em = sc.emitter_profiles[em_inst.profile];
  r.medium_index = kInvalidIndex;
  if (em_inst.cls == kEmitterArea) {
    TriRec tri = load_triangle(sc, em_inst.triangle_index);
    const etxb_material& material = sc.materials[tri.material_index];
    r.barycentric = random_barycentric(smp.next_2d());
    V3 pos, nrm, tan, btn;
    V2 tex;
    lerp_vertex(sc, tri, r.barycentric, pos, nrm, tan, btn, tex);
    r.origin = pos;
    r.normal = nrm;
    r.direction = sample_cosine_frame(smp.next_2d(), nrm, tan, btn, collimation_to_exponent(material.emission_collimation));
    // emitter_evaluate_out_local (:22-38)
    r.pdf_dir = tmax(0.0f, dot(r.normal, r.direction)) * kInvPi;
    if (r.pdf_dir > 0.0f) {
      r.pdf_area = 1.0f / em_inst.triangle_area;
      r.pdf_dir_out = r.pdf_dir * r.pdf_area;
      r.value = apply_image<SP>(sc, em.emission, tex, wavelength);
    }
    r.medium_index = material.ext_medium;
  } else if (em_inst.cls == kEmitterDirectional) {
    V3 direction_to_scene = V3{em.direction[0], em.direction[1], em.direction[2]} * (-1.0f);
    Basis basis = orthonormal_basis(direction_to_scene);
    V2 pos_sample = sample_disk(smp.next_2d());
    V2 dir_sample = sample_disk(smp.next_2d());
    r.direction = normalize(direction_to_scene + basis.u * dir_sample.x * (0.5f * em.equivalent_disk_size) + basis.v * dir_sample.y * (0.5f * em.equivalent_disk_size));
    r.pdf_dir = 1.0f;
    r.pdf_area = 1.0f / (kPi * sc.bounding_sphere_radius * sc.bounding_sphere_radius);
    r.pdf_dir_out = r.pdf_dir * r.pdf_area;
    r.normal = direction_to_scene;
    r.origin = sc.bounding_sphere_center + sc.bounding_sphere_radius * (pos_sample.x * basis.u + pos_sample.y * basis.v - direction_to_scene);
    r.origin += r.direction * distance_to_sphere(r.origin, r.direction, sc.bounding_sphere_center, sc.bounding_sphere_radius);
    r.value = apply_image<SP>(sc, em.emission, dir_sample * 0.5f + 0.5f, wavelength);
  } else {
    const DImage& img = sc.images[em.emission.image_index];
    float pdf_image = 0.0f;
    F4v image_value;
    V2 uv = image_sample(img, smp.next_2d(), pdf_image, image_value);
    if (pdf_image == 0.0f) {
      r.pdf_dir = 0.0f;
      r.triangle_index = kInvalidIndex;
      r.is_delta = false;
      r.is_distant = true;
      r.origin = r.normal = r.direction = {0.0f, 0.0f, 0.0f};
      return r;
    }
    float sin_t = fmaxf(kEpsilon, m_sin(uv.y * kPi));
    V3 d = -uv_to_direction(uv, img.offset_x, img.scale_x);
    Basis basis = orthonormal_basis(d);
    V2 disk_sample = sample_disk(smp.next_2d());
    r.direction = d;
    r.normal = r.direction;
    r.origin = sc.bounding_sphere_center + sc.bounding_sphere_radius * (disk_sample.x * basis.u + disk_sample.y * basis.v - r.direction);
    r.origin += r.direction * distance_to_sphere(r.origin, r.direction, sc.bounding_sphere_center, sc.bounding_sphere_radius);
    r.value = apply_rgb<SP>(sc, wavelength, spectrum_query<SP>(sc, em.emission.spectrum_index, wavelength), image_value);
    r.pdf_area = 1.0f / (kPi * sc.bounding_sphere_radius * sc.bounding_sphere_radius);
    r.pdf_dir = pdf_image / (2.0f * kPi * kPi * sin_t);
    r.pdf_dir_out = r.pdf_area * r.pdf_dir;
  }
  r.triangle_index = em_inst.triangle_index;
  r.is_delta = em_inst.cls == kEmitterDirectional;
  r.is_distant = em_inst.cls != kEmitterArea;
  return r;
}

// sample_emitter (scene_emitters.hxx:216-224) -> emitter_sample_in (:139-203)
template <bool SP>
DEV EmitterSample<SP> sample_emitter(const DeviceScene& sc, float wavelength, uint32_t emitter_index, V2 rnd, V3 from_point) {
  EmitterSample<SP> r;
  r.barycentric = {0.0f, 0.0f, 0.0f};
  r.medium_index = kInvalidIndex;
  const etxb_emitter& em_inst = sc.emitters[emitter_index];
  const etxb_emitter_profile& em = sc.emitter_profiles[em_inst.profile];
  if (em_inst.cls == kEmitterArea) {
    TriRec tri = load_triangle(sc, em_inst.triangle_index);
    r.barycentric = random_barycentric(rnd);
    r.origin = lerp_pos(sc, tri, r.barycentric);
    r.normal = lerp_normal(sc, tri, r.barycentric);
    r.direction = normalize(r.origin - from_point);
    r.value = emitter_get_radiance<SP>(sc, em_inst, wavelength, from_point, r.origin, {0.0f, 0.0f, 0.0f}, lerp_uv(sc, tri, r.barycentric), false, r.pdf_area, r.pdf_dir,
      r.pdf_dir_out);
    r.medium_index = sc.materials[tri.material_index].ext_medium;
  } else if (em_inst.cls == kEmitterDirectional) {
    V3 em_dir = {em.direction[0], em.direction[1], em.direction[2]};
    V2 disk_sample = {0.0f, 0.0f};
    if (em.angular_size > 0.0f) {
      Basis basis = orthonormal_basis(em_dir);
      disk_sample = sample_disk(rnd);
      r.direction = normalize(em_dir + basis.u * disk_sample.x * (0.5f * em.equivalent_disk_size) + basis.v * disk_sample.y * (0.5f * em.equivalent_disk_size));
    } else {
      r.direction = em_dir;
    }
    r.pdf_area = 1.0f / (kPi * sc.bounding_sphere_radius * sc.bounding_sphere_radius);
    r.pdf_dir = 1.0f;
    r.pdf_dir_out = r.pdf_dir * r.pdf_area;
    r.origin = from_point + r.direction * distance_to_sphere(from_point, r.direction, sc.bounding_sphere_center, sc.bounding_sphere_radius);
    r.normal = em_dir * (-1.0f);
    r.value = apply_image<SP>(sc, em.emission, disk_sample * 0.5f + 0.5f, wavelength);
  } else {
    const DImage& img = sc.images[em.emission.image_index];
    float pdf_image = 0.0f;
    F4v image_value;
    V2 uv = image_sample(img, rnd, pdf_image, image_value);
    float sin_t = fmaxf(kEpsilon, m_sin(uv.y * kPi));
    r.direction = uv_to_direction(uv, img.offset_x, img.scale_x);
    r.normal = -r.direction;
    r.origin = from_point + r.direction * distance_to_sphere(from_point, r.direction, sc.bounding_sphere_center, sc.bounding_sphere_radius);
    r.pdf_dir = pdf_image / (2.0f * kPi * kPi * sin_t);
    r.pdf_area = 1.0f / (kPi * sc.bounding_sphere_radius * sc.bounding_sphere_radius);
    r.pdf_dir_out = r.pdf_area * r.pdf_dir;
    r.value = apply_rgb<SP>(sc, wavelength, spectrum_query<SP>(sc, em.emission.spectrum_index, wavelength), image_value);
  }
  r.pdf_sample = emitter_discrete_pdf(sc, em_inst);
  r.emitter_index = emitter_index;
  r.triangle_index = em_inst.triangle_index;
  r.is_delta = em_inst.cls == kEmitterDirectional;
  r.is_distant = em_inst.cls != kEmitterArea;
  return r;
}

// vcm_cam_handle_miss (vcm_shared.hxx:537-587)
template <bool SP>
DEV void vcm_cam_handle_miss(const DeviceScene& sc, const VcmParams& it, V3 ray_d, float& d_vcm, float d_vc, float& path_distance, uint32_t total_path_depth, float wavelength,
  Spec<SP> throughput, Spec<SP>& gathered) {
  if (it.direct_hit() == false) return;
  if (path_distance > 0.0f) {
    d_vcm *= sqr(path_distance);
    path_distance = 0.0f;
  }
  Spec<SP> accumulated_value = Spec<SP>::make(0.0f);
  float sum_pdf_dir_out = 0.0f, sum_pdf_dir = 0.0f;
  for (uint32_t ie = 0; ie < sc.env_emitter_count; ++ie) {
    const etxb_emitter& emitter_instance = sc.emitters[sc.env_emitters[ie]];
    float pdf_area = 0.0f, pdf_dir = 0.0f, pdf_dir_out = 0.0f;
    Spec<SP> value = emitter_get_radiance<SP>(sc, emitter_instance, wavelength, {0.0f, 0.0f, 0.0f}, {0.0f, 0.0f, 0.0f}, ray_d, {0.0f, 0.0f}, total_path_depth <= 1, pdf_area, pdf_dir,
      pdf_dir_out);
    if (pdf_dir > kEpsilon) {
      float pdf_discrete = emitter_discrete_pdf(sc, emitter_instance);
      sum_pdf_dir_out += pdf_dir_out * pdf_discrete;
      sum_pdf_dir += pdf_dir * pdf_discrete;
      accumulated_value += value;
    }
  }
  if (accumulated_value.maximum() > kEpsilon) {
    float inv_count = (sc.env_emitter_count > 0u) ? (1.0f / float(sc.env_emitter_count)) : 0.0f;
    sum_pdf_dir *= inv_count;
    sum_pdf_dir_out *= inv_count;
    float w_camera_sum = d_vcm * sum_pdf_dir + d_vc * sum_pdf_dir_out;
    float weight = it.enable_mis() && (total_path_depth > 1) ? (1.0f / (1.0f + w_camera_sum)) : 1.0f;
    Spec<SP> add = throughput * accumulated_value * weight;
    gathered += add;
  }
}

// ---- camera (scene_camera.hxx) ---------------------------------------------------------------------------------
DEV V3 cam3(const float* p) { return {p[0], p[1], p[2]}; }
DEV bool camera_has_lens(const etxb_camera& c) { return (c.lens_radius > kEpsilon) && (c.focal_distance > kEpsilon); }

// point on the lens in [-1, 1]^2: the unit disk, or the camera's aperture image sampled by its luminance table (:44-48, 73-81)
DEV V2 sample_lens(const DeviceScene& sc, const etxb_camera& camera, V2 rnd) {
  if (camera.lens_image == kInvalidIndex) return sample_disk(rnd);
  float pdf = 0.0f;
  F4v value;
  V2 uv = image_sample(sc.images[camera.lens_image], rnd, pdf, value);
  return uv * 2.0f - 1.0f;
}

// generate_ray (:26-62)
DEV void generate_ray(const DeviceScene& sc, const etxb_camera& camera, V2 uv, V2 sensor_rnd, V3& origin, V3& w_o, float& t_near, float& t_far) {
  origin = cam3(camera.position);
  if (camera.cls == 1u) {  // Camera::Class::Equirectangular (:29-31)
    w_o = from_spherical(uv.x * kPi, uv.y * kHalfPi);
    t_near = kRayEpsilon;
    t_far = kMaxFloat;
    return;
  }
  V3 direction = cam3(camera.direction);
  V3 s = uv.x * cam3(camera.side);
  V3 u = uv.y * cam3(camera.up) / camera.aspect;
  w_o = normalize(camera.tan_half_fov * (s + u) + direction);
  if (camera_has_lens(camera)) {
    V2 sensor_sample = sample_lens(sc, camera, sensor_rnd);
    sensor_sample = sensor_sample * camera.lens_radius;
    origin = origin + cam3(camera.side) * sensor_sample.x + cam3(camera.up) * sensor_sample.y;
    float focal_plane_distance = camera.focal_distance / dot(w_o, direction);
    V3 p = cam3(camera.position) + focal_plane_distance * w_o;
    w_o = normalize(p - origin);
  }
  float cos_t = dot(w_o, direction);
  float tn = camera.clip_near > 0.0f ? camera.clip_near / cos_t : kRayEpsilon;
  t_far = camera.clip_far > 0.0f ? camera.clip_far / cos_t : kMaxFloat;
  t_near = fmaxf(tn, kRayEpsilon);
}

struct CameraSample {
  V3 position, direction;
  V2 uv;
  float weight, pdf_dir, pdf_dir_out;
};
// sample_film (:64-118)
DEV CameraSample sample_film(Smp& smp, const DeviceScene& sc, const etxb_camera& camera, V3 from_point) {
  CameraSample r = {};
  if (camera.cls == 1u) return r;  // the reference has no film sampling for the equirectangular camera (:65-68): light paths never connect to it
  V2 sensor_sample = {0.0f, 0.0f};
  if (camera_has_lens(camera)) {
    sensor_sample = sample_lens(sc, camera, smp.next_2d());
    sensor_sample = sensor_sample * camera.lens_radius;
  }
  r.position = cam3(camera.position) + sensor_sample.x * cam3(camera.side) + sensor_sample.y * cam3(camera.up);
  r.direction = r.position - from_point;
  V3 normal = cam3(camera.direction);
  float cos_t = -dot(r.direction, normal);
  if (cos_t < 0.0f) return CameraSample{};
  float distance_squared = dot(r.direction, r.direction);
  float distance = sqrtf(distance_squared);
  r.direction /= distance;
  cos_t /= distance;
  float focal_plane_distance = camera_has_lens(camera) ? camera.focal_distance : 1.0f;
  V3 focus_point = r.position - r.direction * (focal_plane_distance / cos_t);
  const float* m = camera.view_proj;
  float px = m[0] * focus_point.x + m[4] * focus_point.y + m[8] * focus_point.z + m[12] * 1.0f;
  float py = m[1] * focus_point.x + m[5] * focus_point.y + m[9] * focus_point.z + m[13] * 1.0f;
  float pw = m[3] * focus_point.x + m[7] * focus_point.y + m[11] * focus_point.z + m[15] * 1.0f;
  r.uv = {px / pw, py / pw};
  if ((pw <= 0.0f) || (r.uv.x < -1.0f) || (r.uv.y < -1.0f) || (r.uv.x > 1.0f) || (r.uv.y > 1.0f)) return CameraSample{};
  float lens_area = (camera.lens_radius > kEpsilon) ? kPi * sqr(camera.lens_radius) : 1.0f;
  float pdf_area = 1.0f / lens_area;
  r.pdf_dir = pdf_area * distance_squared / cos_t;
  r.pdf_dir_out = 1.0f / (camera.area * lens_area * cos_t * cos_t * cos_t);
  float importance = r.pdf_dir_out / cos_t;
  r.weight = importance / r.pdf_dir;
  return r;
}

// ---- path start ----------------------------------------------------------------------------------------------------
// vcm_generate_emitter_state (vcm_shared.hxx:310-349)
template <bool SP>
DEV PathState<SP> generate_emitter_state(const DeviceScene& sc, const VcmParams& it, uint32_t index) {
  PathState<SP> s = {};
  s.throughput = Spec<SP>::make(0.0f);
  s.gathered = Spec<SP>::make(0.0f);
  s.eta = 1.0f;
  s.medium_index = kInvalidIndex;
  s.ray_min_t = kRayEpsilon;
  s.ray_max_t = kMaxFloat;
  s.sampler.init(index, it.iteration);
  s.wavelength = SP ? spectral_sample_wavelength(s.sampler.next()) : -1.0f;
  EmitterSample<SP> es = sample_emission<SP>(sc, s.wavelength, s.sampler);
  if (es.pdf_dir <= 0.0f) return s;
  float cos_t = dot(es.direction, es.normal);
  s.throughput = es.value * (cos_t / (es.pdf_dir * es.pdf_area * es.pdf_sample));
  s.ray_o = es.origin;
  s.ray_d = es.direction;
  if (es.triangle_index != kInvalidIndex) {
    s.ray_o = shading_pos(sc, load_triangle(sc, es.triangle_index), es.barycentric, s.ray_d);
  }
  s.d_vcm = es.is_distant ? 1.0f / es.pdf_area : 1.0f / es.pdf_dir;
  if (es.is_delta == false) {
    s.d_vc = (es.is_distant ? 1.0f : cos_t) / (es.pdf_dir * es.pdf_area * es.pdf_sample);
  }
  s.d_vm = s.d_vc * it.vc_weight;
  s.eta = 1.0f;
  s.medium_index = es.medium_index;
  s.flags = (es.is_delta ? kPathDeltaEmitter : 0u) | (es.is_distant ? 0u : kPathLocalEmitter) | kPathValid;
  return s;
}

// vcm_generate_camera_state (vcm_shared.hxx:351-377)
template <bool SP>
DEV PathState<SP> generate_camera_state(const DeviceScene& sc, const VcmParams& it, uint32_t px, uint32_t py, uint32_t index, float light_wavelength) {
  PathState<SP> s = {};
  s.sampler.init(index, it.iteration);
  if constexpr (SP) {
    float sampled = spectral_sample_wavelength(s.sampler.next());
    s.wavelength = (light_wavelength == 0.0f) ? sampled : light_wavelength;
  } else {
    s.wavelength = light_wavelength;  // kUndefinedWavelength (-1)
  }
  const etxb_camera& camera = sc.camera;
  // get_jittered_uv (scene_camera.hxx:12-18)
  float sample_radius = 0.5f;
  V2 uv;
  uv.x = (float(px) + 0.5f + sample_radius * (s.sampler.next() * 2.0f - 1.0f)) / float(camera.film_size[0]) * 2.0f - 1.0f;
  uv.y = (float(py) + 0.5f + sample_radius * (s.sampler.next() * 2.0f - 1.0f)) / float(camera.film_size[1]) * 2.0f - 1.0f;
  generate_ray(sc, camera, uv, s.sampler.next_2d(), s.ray_o, s.ray_d, s.ray_min_t, s.ray_max_t);
  s.throughput = Spec<SP>::make(1.0f);
  s.gathered = Spec<SP>::make(0.0f);
  s.merged = {0.0f, 0.0f, 0.0f};
  // film_evaluate_out (scene_camera.hxx:120-126)
  float cos_t = dot(s.ray_d, cam3(camera.direction));
  float pdf_dir = (camera.cls == 1u) ? 1.0f : 1.0f / (camera.area * cos_t * cos_t * cos_t);
  s.d_vcm = 1.0f / pdf_dir;
  s.d_vc = 0.0f;
  s.d_vm = 0.0f;
  s.medium_index = camera.medium_index;
  s.eta = 1.0f;
  s.path_distance = 0.0f;
  s.total_path_depth = 1;
  return s;
}

// ---- light vertex record (VCMLightVertex, vcm_shared.hxx:154-197): 6 x 16 B in HBM ------------------------------------
struct LightVertexRec {
  float4 thr_dvcm;  // throughput (x only in spectral mode), d_vcm
  float4 wi_dvc;    // w_i, d_vc
  float4 bc_dvm;    // barycentric, d_vm
  float4 pos_tri;   // pos, triangle index (bits)
  float4 nrm_mat;   // nrm, material index (bits)
  uint4 ids;        // medium index, path_length, path_index, ordinal within the path
};
static_assert(sizeof(LightVertexRec) == 96, "light vertex record is 96 bytes");

template <bool SP>
DEV LightVertexRec make_light_vertex(const PathState<SP>& s, const Isect& i, uint32_t path_index) {
  LightVertexRec r;
  V3 t = s.throughput.as_v3();
  r.thr_dvcm = make_float4(t.x, t.y, t.z, s.d_vcm);
  r.wi_dvc = make_float4(s.ray_d.x, s.ray_d.y, s.ray_d.z, s.d_vc);
  r.bc_dvm = make_float4(i.barycentric.x, i.barycentric.y, i.barycentric.z, s.d_vm);
  r.pos_tri = make_float4(i.pos.x, i.pos.y, i.pos.z, __uint_as_float(i.triangle_index));
  r.nrm_mat = make_float4(i.nrm.x, i.nrm.y, i.nrm.z, __uint_as_float(i.material_index));
  r.ids = make_uint4(s.medium_index, s.total_path_depth, path_index, s.lv_count);
  return r;
}

// medium light vertex (vcm_shared.hxx:1110-1127): no triangle / material, position = the sampled medium point
template <bool SP>
DEV LightVertexRec make_medium_light_vertex(const PathState<SP>& s, V3 pos, uint32_t path_index) {
  LightVertexRec r;
  V3 t = s.throughput.as_v3();
  r.thr_dvcm = make_float4(t.x, t.y, t.z, s.d_vcm);
  r.wi_dvc = make_float4(s.ray_d.x, s.ray_d.y, s.ray_d.z, s.d_vc);
  r.bc_dvm = make_float4(0.0f, 0.0f, 0.0f, s.d_vm);
  r.pos_tri = make_float4(pos.x, pos.y, pos.z, __uint_as_float(kInvalidIndex));
  r.nrm_mat = make_float4(0.0f, 0.0f, 0.0f, __uint_as_float(kInvalidIndex));
  r.ids = make_uint4(s.medium_index, s.total_path_depth, path_index, s.lv_count);
  return r;
}

// ---- shared step pieces ------------------------------------------------------------------------------------------------
// vcm_next_ray (vcm_shared.hxx:218-283)
template <bool SP>
DEV bool vcm_next_ray(const DeviceScene& sc, bool light_path, PathState<SP>& state, const VcmParams& it, const Isect& isect, const BData& bsdf_data, const BSample<SP>& bs,
                      bool subsurface_sample = false) {
  if (state.total_path_depth + 1 > sc.max_path_length) return false;
  if (bs.valid() == false) return false;
  TriRec tri = load_triangle(sc, isect.triangle_index);
  const etxb_material& mat = sc.materials[isect.material_index];
  state.throughput *= bs.weight;
  if (light_path) {
    state.throughput *= fix_shading_normal(tri.geo_n, isect.nrm, isect.w_i, bs.w_o);
  }
  if (state.throughput.is_zero()) return false;
  if (random_continue<SP>(state.total_path_depth, sc.random_path_termination, state.eta, state.sampler, state.throughput) == false) return false;
  if (bs.properties & kBsdfMediumChanged) {
    state.medium_index = bs.medium_index;
  }
  float cos_theta_bsdf = fabsf(dot(isect.nrm, bs.w_o));
  if (bs.is_delta()) {
    state.d_vc *= cos_theta_bsdf;
    state.d_vm *= cos_theta_bsdf;
    state.d_vcm = 0.0f;
  } else {
    float rev_sample_pdf = subsurface_sample ? fabsf(dot(bsdf_data.w_i, isect.nrm)) / kPi : bsdf_reverse_pdf<SP>(sc, bsdf_data, bs.w_o, mat, state.sampler);
    state.d_vc = (cos_theta_bsdf / bs.pdf) * (state.d_vc * rev_sample_pdf + state.d_vcm + it.vm_weight);
    state.d_vm = (cos_theta_bsdf / bs.pdf) * (state.d_vm * rev_sample_pdf + state.d_vcm * it.vc_weight + 1.0f);
    state.d_vcm = 1.0f / bs.pdf;
  }
  state.ray_d = bs.w_o;
  state.ray_o = shading_pos(sc, tri, isect.barycentric, bs.w_o);
  state.ray_max_t = kMaxFloat;
  state.ray_min_t = kRayEpsilon;
  state.eta *= bs.eta;
  state.total_path_depth += 1u;
  return true;
}

// A connection endpoint on the eye/light subpath: a surface point (isect) or a medium scattering point (pos only).
struct Endpoint {
  bool at_medium;
  const Isect* isect;
  V3 medium_pos;
  DEV V3 pos() const { return at_medium ? medium_pos : isect->pos; }
};
DEV float medium_phase(const DeviceScene& sc, uint32_t medium_index, V3 w_i, V3 w_o) { return phase_function(w_i, w_o, sc.mediums[medium_index].phase_function_g); }

// vcm_try_sampling_medium (vcm_shared.hxx:379-388)
template <bool SP, bool PLAIN = false>
DEV MediumSample<SP> vcm_try_sampling_medium(const DeviceScene& sc, PathState<SP>& state, float max_t) {
  MediumSample<SP> r;
  r.weight = Spec<SP>::make(0.0f);
  r.pos = {0.0f, 0.0f, 0.0f};
  r.sampled_medium_t = 0.0f;
  if constexpr (PLAIN) return r;  // no media in the scene
  if (state.medium_index == kInvalidIndex) return r;
  r = sample_medium<SP>(sc, sc.mediums[state.medium_index], state.wavelength, state.throughput, state.sampler, state.ray_o, state.ray_d, max_t);
  state.throughput *= r.weight;
  return r;
}

// vcm_handle_boundary_bsdf (vcm_shared.hxx:436-449)
template <bool SP, bool PLAIN = false>
DEV bool vcm_handle_boundary(const DeviceScene& sc, const Isect& isect, PathState<SP>& state) {
  if constexpr (PLAIN) return false;  // no Boundary surfaces in the scene
  const etxb_material& mat = sc.materials[isect.material_index];
  if (mat.cls != ETXB_MAT_BOUNDARY) return false;
  TriRec tri = load_triangle(sc, isect.triangle_index);
  uint32_t new_medium = (dot(tri.geo_n, state.ray_d) < 0.0f) ? mat.int_medium : mat.ext_medium;
  state.path_distance += isect.t;
  state.medium_index = new_medium;
  state.ray_o = shading_pos(sc, tri, isect.barycentric, state.ray_d);
  state.ray_max_t = kMaxFloat;
  state.ray_min_t = kRayEpsilon;
  return true;
}

// vcm_connect_to_camera (vcm_shared.hxx:463-535)
template <bool SP, bool PLAIN = false>
DEV bool vcm_connect_to_camera(const DeviceScene& sc, const VcmParams& it, const Endpoint& ep, PathState<SP>& state, Spec<SP>& out_value, V2& uv, TraverseStats* stats,
  uint32_t& shadow_rays, V3* deferred_segment = nullptr) {
  if ((it.connect_to_camera() == false) || (state.total_path_depth + 2 > sc.max_path_length) || (state.total_path_depth + 2 < sc.min_path_length)) return false;
  const etxb_camera& camera = sc.camera;
  V3 sample_pos = ep.pos();
  CameraSample cs = sample_film(state.sampler, sc, camera, sample_pos);
  if (cs.pdf_dir <= 0.0f) return false;
  V3 direction = cs.position - sample_pos;
  float dist2 = dot(direction, direction);
  if (dist2 <= kEpsilon) return false;
  V3 w_o = normalize(direction);
  Spec<SP> scatter = Spec<SP>::make(0.0f);
  float reverse_pdf = 0.0f;
  V3 origin = sample_pos;
  if (ep.at_medium == false) {
    const Isect& isect = *ep.isect;
    const etxb_material& mat = sc.materials[isect.material_index];
    BData data = make_bdata(isect, isect.w_i, state.wavelength, state.medium_index, kPathLight);
#if defined(ETXB_PARITY) && ETXB_PARITY
    BEval<SP> eval = bsdf_evaluate<SP>(sc, data, w_o, mat, state.sampler);
    if (eval.valid() == false) return false;
    scatter = eval.bsdf;
    reverse_pdf = bsdf_reverse_pdf<SP>(sc, data, w_o, mat, state.sampler);
#else
    if ((mat.cls == ETXB_MAT_DIFFUSE) && (mat.diffuse_variation == 0u)) {
      BEval<SP> eval = bsdf_evaluate<SP>(sc, data, w_o, mat, state.sampler);
      if (eval.valid() == false) return false;
      scatter = eval.bsdf;
      reverse_pdf = bsdf_reverse_pdf<SP>(sc, data, w_o, mat, state.sampler);
    } else {  // product build: value and reverse pdf from one prepared closure (dclosure.cuh)
      Closure<SP> cl = make_closure<SP>(sc, data, isect.material_index, state.sampler);
      CEval<SP> ce = closure_evaluate<SP>(sc, cl, w_o, state.sampler);
      if (ce.valid() == false) return false;
      scatter = ce.bsdf;
      reverse_pdf = ce.rev_pdf;
    }
#endif
    origin = shading_pos(sc, load_triangle(sc, isect.triangle_index), isect.barycentric, w_o);
  } else {
    float p = medium_phase(sc, state.medium_index, state.ray_d, w_o);
    if (p <= 0.0f) return false;
    scatter = Spec<SP>::make(p);
    reverse_pdf = medium_phase(sc, state.medium_index, w_o, state.ray_d);
  }
  float len = length(cs.position - origin);
  float cos_t = fabsf(dot(cs.direction, cam3(camera.direction)));
  V3 clip_pos = origin + cs.direction * fmaxf(0.0f, len - camera.clip_near / cos_t);
  shadow_rays += 1;
  Spec<SP> tr = Spec<SP>::make(1.0f);
  if (deferred_segment != nullptr) {  // the caller queues the segment (ShadowBatch, atomic mode); out_value is the unoccluded contribution
    deferred_segment[0] = origin;
    deferred_segment[1] = clip_pos;
  } else {
    tr = trace_transmittance<SP, PLAIN>(sc, state.wavelength, origin, clip_pos, state.medium_index, state.sampler, stats);
    if (tr.is_zero()) return false;
  }
  uv = cs.uv;
  float camera_pdf = cs.pdf_dir_out * (ep.at_medium ? 1.0f : fabsf(dot(ep.isect->nrm, w_o))) / dist2;
  float vmW_cam = ep.at_medium ? 0.0f : it.vm_weight;
  float w_light = camera_pdf * (vmW_cam + state.d_vcm + state.d_vc * reverse_pdf);
  float weight = it.enable_mis() ? (1.0f / (1.0f + w_light)) : 1.0f;
  if (ep.at_medium == false) {
    const Isect& isect = *ep.isect;
    weight *= fix_shading_normal(load_triangle(sc, isect.triangle_index).geo_n, isect.nrm, isect.w_i, w_o);
  }
  out_value = tr * scatter * state.throughput * cs.weight * weight;
  return true;
}

// vcm_get_radiance + vcm_handle_direct_hit (vcm_shared.hxx:285-308, 597-606)
template <bool SP>
DEV void vcm_handle_direct_hit(const DeviceScene& sc, const VcmParams& it, const Isect& isect, PathState<SP>& state) {
  if ((it.direct_hit() == false) || (isect.emitter_index == kInvalidIndex)) return;
  if ((state.total_path_depth > sc.max_path_length) || (state.total_path_depth < sc.min_path_length)) return;
  const etxb_emitter& emitter = sc.emitters[isect.emitter_index];
  float pdf_emitter_area, pdf_emitter_dir, pdf_emitter_dir_out;
  Spec<SP> radiance = emitter_get_radiance<SP>(sc, emitter, state.wavelength, state.ray_o, isect.pos, state.ray_d, isect.tex, state.total_path_depth == 1, pdf_emitter_area,
    pdf_emitter_dir, pdf_emitter_dir_out);
  if (pdf_emitter_dir <= kEpsilon) return;
  float emitter_sample_pdf = emitter_discrete_pdf(sc, emitter);
  float w_camera = state.d_vcm * pdf_emitter_area * emitter_sample_pdf + state.d_vc * (pdf_emitter_dir_out * emitter_sample_pdf);
  float weight = (it.enable_mis() && (state.total_path_depth > 1)) ? (1.0f / (1.0f + w_camera)) : 1.0f;
  state.gathered += weight * (state.throughput * radiance);
}

// Deferred shadow rays.  In a scene where every surface is opaque (no alpha test can reject), without Boundary materials, media
// or stochastic BSDFs, a shadow ray of the camera step does exactly two things (rt.cxx:468-579): it decides visible / occluded, and it
// draws ONE value from the path's sampler if it is occluded (the alpha test of the hit that blocks it), none if it is visible.  Neither
// depends on the order candidates are met, and nothing else draws between a vertex's connections and its continuation.  So the
// connection routines only WRITE the segment and the unoccluded contribution here; k_shadow_trace resolves all segments of the bounce in
// a traversal-only kernel, and k_camera_continue adds the visible contributions in the reference's order and advances the sampler by the
// number of occluded ones — bit-identical to tracing inline.
struct ShadowBatch {
  float4* p0;
  float4* p1;
  float4* value;
  uint32_t base, count;
  // Product build, opaque scenes with stochastic BSDFs (no slot order to keep: those stages already run on derived sampler streams): segments
  // from every producer of a bounce go to ONE list through an atomic cursor, each carrying the address its contribution is added to when the
  // segment turns out unoccluded (k_shadow_resolve): a path's `gathered` sum, or a pixel of the light image (bit 31 set).
  uint32_t* atomic_cursor = nullptr;
  uint32_t capacity = 0;
  uint32_t target = 0;
  template <bool SP>
  DEV void push(V3 a, V3 b, Spec<SP> v) {
    push_rgb(a, b, v.as_v3());
  }
  DEV void push_rgb(V3 a, V3 b, V3 c) {
    uint32_t k = (atomic_cursor != nullptr) ? atomicAdd(atomic_cursor, 1u) : (base + count);
    count += 1u;
    if ((atomic_cursor != nullptr) && (k >= capacity)) return;  // the host sized the list for every segment a bounce can produce; the resolver clamps
    p0[k] = make_float4(a.x, a.y, a.z, 0.0f);
    // the target travels as raw bits in p1.w.  It is stored through an integer lane: small integers are denormal bit patterns, and a float
    // select on them is flushed to zero by the product build's -ftz (measured: every contribution landed on path 0 / pixel 0)
    p1[k] = make_float4(b.x, b.y, b.z, 0.0f);
    if (atomic_cursor != nullptr) reinterpret_cast<uint32_t*>(p1 + k)[3] = target;
    value[k] = make_float4(c.x, c.y, c.z, 0.0f);
  }
};
constexpr uint32_t kShadowTargetPixel = 0x80000000u;

// vcm_connect_to_light (vcm_shared.hxx:608-671)
template <bool SP, bool PLAIN = false>
DEV Spec<SP> vcm_connect_to_light(const DeviceScene& sc, const VcmParams& it, const Endpoint& ep, PathState<SP>& state, TraverseStats* stats, uint32_t& shadow_rays,
                                  ShadowBatch* batch = nullptr) {
  Spec<SP> zero = Spec<SP>::make(0.0f);
  if ((it.connect_to_light() == false) || (state.total_path_depth + 1 > sc.max_path_length) || (state.total_path_depth + 1 < sc.min_path_length)) return zero;
  V3 sample_pos = ep.pos();
  uint32_t emitter_index = distribution_sample(sc.emitter_dist, sc.emitter_count + 1u, state.sampler.fixed_w);
  EmitterSample<SP> es = sample_emitter<SP>(sc, state.wavelength, emitter_index, {state.sampler.fixed_u, state.sampler.fixed_v}, sample_pos);
  if (es.pdf_dir <= 0.0f) return zero;
  V3 w_o = es.direction;
  Spec<SP> scatter = zero;
  float reverse_pdf = 0.0f;
  V3 origin = sample_pos;
  float camera_factor = 1.0f;
  float closure_pdf = -1.0f;  // product build: the forward pdf that came with the evaluation (the reference asks bsdf::pdf again, :650-653)
  if (ep.at_medium) {
    float p = medium_phase(sc, state.medium_index, state.ray_d, w_o);
    if (p <= 0.0f) return zero;
    scatter = Spec<SP>::make(p);
    reverse_pdf = medium_phase(sc, state.medium_index, w_o, state.ray_d);
  } else {
    const Isect& isect = *ep.isect;
    const etxb_material& mat = sc.materials[isect.material_index];
    BData data = make_bdata(isect, isect.w_i, state.wavelength, state.medium_index, kPathCamera);
#if defined(ETXB_PARITY) && ETXB_PARITY
    BEval<SP> eval = bsdf_evaluate<SP>(sc, data, w_o, mat, state.sampler);
    if (eval.valid() == false) return zero;
    scatter = eval.bsdf;
    reverse_pdf = bsdf_reverse_pdf<SP>(sc, data, w_o, mat, state.sampler);
#else
    if ((mat.cls == ETXB_MAT_DIFFUSE) && (mat.diffuse_variation == 0u)) {
      BEval<SP> eval = bsdf_evaluate<SP>(sc, data, w_o, mat, state.sampler);
      if (eval.valid() == false) return zero;
      scatter = eval.bsdf;
      reverse_pdf = bsdf_reverse_pdf<SP>(sc, data, w_o, mat, state.sampler);
      closure_pdf = eval.pdf;
    } else {  // product build: value, pdf and reverse pdf from one prepared closure (dclosure.cuh)
      Closure<SP> cl = make_closure<SP>(sc, data, isect.material_index, state.sampler);
      CEval<SP> ce = closure_evaluate<SP>(sc, cl, w_o, state.sampler);
      if (ce.valid() == false) return zero;
      scatter = ce.bsdf;
      reverse_pdf = ce.rev_pdf;
      closure_pdf = (cl.kind == kClGeneric) ? -1.0f : ce.pdf;  // classes without a closure form answer bsdf::pdf themselves
    }
#endif
    TriRec tri = load_triangle(sc, isect.triangle_index);
    origin = shading_pos(sc, tri, isect.barycentric, normalize(es.origin - isect.pos));
    camera_factor = fabsf(dot(w_o, tri.geo_n));
  }
  shadow_rays += 1;
  Spec<SP> tr = Spec<SP>::make(1.0f);
  if (batch == nullptr) {
    tr = trace_transmittance<SP, PLAIN>(sc, state.wavelength, origin, es.origin, state.medium_index, state.sampler, stats);
    if (tr.is_zero()) return zero;
  }
  float l_dot_e = fabsf(dot(es.direction, es.normal));
  float w_light = 0.0f;
  if (es.is_delta == false) {
    if (ep.at_medium) {
      w_light = scatter.component(0) / (es.pdf_dir * es.pdf_sample);  // SpectralResponse{spect, p}.value
    } else {
      const Isect& isect = *ep.isect;
      BData data = make_bdata(isect, isect.w_i, state.wavelength, state.medium_index, kPathCamera);
      float conn_pdf = (closure_pdf >= 0.0f) ? closure_pdf : bsdf_pdf<SP>(sc, data, w_o, sc.materials[isect.material_index], state.sampler);
      w_light = conn_pdf / (es.pdf_dir * es.pdf_sample);
    }
  }
  float vmW_nee = ep.at_medium ? 0.0f : it.vm_weight;
  float w_camera = (es.pdf_dir_out * camera_factor) / (es.pdf_dir * l_dot_e) * (vmW_nee + state.d_vcm + state.d_vc * reverse_pdf);
  float weight = it.enable_mis() ? 1.0f / (1.0f + w_light + w_camera) : 1.0f;
  Spec<SP> result = tr * state.throughput * scatter * es.value * (weight / (es.pdf_dir * es.pdf_sample));
  if (batch != nullptr) {
    batch->push<SP>(origin, es.origin, result);  // tr == 1 here: the product above is the unoccluded contribution, bit for bit
    return zero;
  }
  return result;
}

// vcm_connect_to_light_vertex (vcm_shared.hxx:673-763)
template <bool SP>
DEV bool vcm_connect_to_light_vertex(const DeviceScene& sc, const VcmParams& it, PathState<SP>& state, const LightVertexRec& lv, const Endpoint& ep, V3& target_position,
  Spec<SP>& value) {
  const uint32_t lv_tri = __float_as_uint(lv.pos_tri.w);
  const bool lv_is_medium = lv_tri == kInvalidIndex;
  const V3 lv_wi = {lv.wi_dvc.x, lv.wi_dvc.y, lv.wi_dvc.z};
  Isect light_v = {};  // VCMLightVertex::vertex(): lerp_vertex from (triangle, barycentric)
  TriRec light_tri = {};
  if (lv_is_medium == false) {
    light_tri = load_triangle(sc, lv_tri);
    V3 bc = {lv.bc_dvm.x, lv.bc_dvm.y, lv.bc_dvm.z};
    lerp_vertex(sc, light_tri, bc, light_v.pos, light_v.nrm, light_v.tan, light_v.btn, light_v.tex);
  }
  target_position = lv_is_medium ? V3{lv.pos_tri.x, lv.pos_tri.y, lv.pos_tri.z} : light_v.pos;
  V3 w_o = target_position - ep.pos();
  float distance_squared = dot(w_o, w_o);
  if (distance_squared <= kEpsilon) return false;
  w_o /= sqrtf(distance_squared);
  float w_dot_l = 1.0f;
  if (lv_is_medium == false) w_dot_l = -dot(light_v.nrm, w_o);

  float camera_area_pdf = 0.0f, camera_rev_pdf = 0.0f;
  Spec<SP> camera_scatter = Spec<SP>::make(0.0f);
  const uint32_t state_medium = state.medium_index;
  if (ep.at_medium) {
    float p = medium_phase(sc, state_medium, state.ray_d, w_o);
    if (p <= 0.0f) return false;
    float p_rev = medium_phase(sc, state_medium, w_o, state.ray_d);
    camera_area_pdf = p * fabsf(w_dot_l) / distance_squared;
    camera_rev_pdf = p_rev;
    camera_scatter = Spec<SP>::make(p);
  } else {
    const Isect& cam = *ep.isect;
    const etxb_material& mat = sc.materials[cam.material_index];
    BData camera_data = make_bdata(cam, cam.w_i, state.wavelength, state_medium, kPathCamera);
    BEval<SP> camera_bsdf = bsdf_evaluate<SP>(sc, camera_data, w_o, mat, state.sampler);
    if (camera_bsdf.valid() == false) return false;
    camera_area_pdf = camera_bsdf.pdf * fabsf(w_dot_l) / distance_squared;
    camera_rev_pdf = bsdf_reverse_pdf<SP>(sc, camera_data, w_o, mat, state.sampler);
    camera_scatter = camera_bsdf.bsdf;
  }

  float light_area_pdf = 0.0f, light_rev_pdf = 0.0f;
  Spec<SP> light_scatter = Spec<SP>::make(0.0f);
  if (lv_is_medium) {
    float p = medium_phase(sc, lv.ids.x, lv_wi, -w_o);
    if (p <= 0.0f) return false;
    float p_rev = medium_phase(sc, lv.ids.x, -w_o, lv_wi);
    light_area_pdf = p * (ep.at_medium ? 1.0f : fabsf(dot(ep.isect->nrm, w_o))) / distance_squared;
    light_rev_pdf = p_rev;
    light_scatter = Spec<SP>::make(p);
  } else {
    const etxb_material& light_mat = sc.materials[__float_as_uint(lv.nrm_mat.w)];
    BData light_data = {light_v.pos, light_v.nrm, light_v.tan, light_v.btn, light_v.tex, lv_wi, state.wavelength, kPathLight, ep.at_medium ? lv.ids.x : state_medium};
    BEval<SP> light_bsdf = bsdf_evaluate<SP>(sc, light_data, -w_o, light_mat, state.sampler);
    if (light_bsdf.valid() == false) return false;
    if (ep.at_medium) {
      light_area_pdf = light_bsdf.pdf / distance_squared;
    } else {
      float w_dot_c = dot(ep.isect->nrm, w_o);
      light_area_pdf = light_bsdf.pdf * fabsf(w_dot_c) / distance_squared;
    }
    light_rev_pdf = bsdf_reverse_pdf<SP>(sc, light_data, -w_o, light_mat, state.sampler);
    light_scatter = light_bsdf.bsdf * fix_shading_normal(light_tri.geo_n, light_data.nrm, light_data.w_i, -w_o);
  }

  float vmW_pair = (ep.at_medium || lv_is_medium) ? 0.0f : it.vm_weight;
  float w_light = camera_area_pdf * (vmW_pair + lv.thr_dvcm.w + lv.wi_dvc.w * light_rev_pdf);
  float w_camera = light_area_pdf * (vmW_pair + state.d_vcm + state.d_vc * camera_rev_pdf);
  float weight = it.enable_mis() ? 1.0f / (1.0f + w_light + w_camera) : 1.0f;
  Spec<SP> lv_throughput = Spec<SP>::make3({lv.thr_dvcm.x, lv.thr_dvcm.y, lv.thr_dvcm.z});
  value = (camera_scatter * state.throughput) * (light_scatter * lv_throughput) * (weight / distance_squared);
  return true;
}

DEV LightVertexRec load_light_vertex(const LightVertexRec* p_rec) {
  const float4* p = reinterpret_cast<const float4*>(p_rec);
  LightVertexRec lv;
  lv.thr_dvcm = __ldg(p + 0);
  lv.wi_dvc = __ldg(p + 1);
  lv.bc_dvm = __ldg(p + 2);
  lv.pos_tri = __ldg(p + 3);
  lv.nrm_mat = __ldg(p + 4);
  lv.ids = __ldg(reinterpret_cast<const uint4*>(p) + 5);
  return lv;
}

// the shadow segment of one vertex connection (vcm_shared.hxx:784-799)
template <bool SP, bool PLAIN = false>
DEV Spec<SP> vcm_connection_transmittance(const DeviceScene& sc, const Endpoint& ep, const LightVertexRec& lv, V3 target_position, PathState<SP>& state, TraverseStats* stats) {
  if (ep.at_medium) {
    return trace_transmittance<SP, PLAIN>(sc, state.wavelength, ep.medium_pos, {lv.pos_tri.x, lv.pos_tri.y, lv.pos_tri.z}, state.medium_index, state.sampler, stats);
  }
  const Isect& isect = *ep.isect;
  V3 p0 = shading_pos(sc, load_triangle(sc, isect.triangle_index), isect.barycentric, normalize(target_position - isect.pos));
  return trace_transmittance<SP, PLAIN>(sc, state.wavelength, p0, target_position, state.medium_index, state.sampler, stats);
}

// vcm_connect_to_light_path (vcm_shared.hxx:765-803): serial over the paired path's vertices (shared sampler)
template <bool SP, bool PLAIN = false>
DEV Spec<SP> vcm_connect_to_light_path(const DeviceScene& sc, const VcmParams& it, const LightVertexRec* pool, uint32_t lp_index, uint32_t lp_count, const Endpoint& ep,
  PathState<SP>& state, TraverseStats* stats, uint32_t& shadow_rays, uint32_t& connections) {
  Spec<SP> result = Spec<SP>::make(0.0f);
  if (it.connect_vertices() == false) return result;
  for (uint32_t i = 0; i < lp_count; ++i) {
    const uint64_t target_path_length = uint64_t(state.total_path_depth) + i + 2u;
    if (target_path_length < sc.min_path_length) continue;
    if (target_path_length > sc.max_path_length) break;
    LightVertexRec lv = load_light_vertex(pool + lp_index + i);
    connections += 1;
    V3 target_position;
    Spec<SP> value;
    if (vcm_connect_to_light_vertex<SP>(sc, it, state, lv, ep, target_position, value)) {
      shadow_rays += 1;
      Spec<SP> tr = vcm_connection_transmittance<SP, PLAIN>(sc, ep, lv, target_position, state, stats);
      if (tr.is_zero() == false) {
        result += tr * value;
      }
    }
  }
  return result;
}

// ---- photon hash grid (VCMSpatialGridData, vcm_shared.hxx:805-925) ------------------------------------------------------
struct GridData {
  const uint2* cell_range;  // [begin, end) per hash cell
  const float4* pos_dvcm;   // position, d_vcm
  const float4* nrm_dvm;    // normal, d_vm
  const float4* win_len;    // w_in, path_length (bits)
  const float4* thr_rgb;    // throughput.to_rgb() / pdf_lambda
  V3 bbox_min, bbox_max;
  uint32_t hash_table_mask;
  uint32_t photon_count;
  float cell_size, radius_squared, inv_radius_squared;
};
DEV uint32_t grid_cell_index(uint32_t mask, int32_t x, int32_t y, int32_t z) {
  return ((uint32_t(x) * 73856093u) ^ (uint32_t(y) * 19349663u) ^ (uint32_t(z) * 83492791u)) & mask;
}
DEV uint32_t grid_position_to_index(V3 pos, V3 bbox_min, float cell_size, uint32_t mask) {
  V3 m = vfloor((pos - bbox_min) / cell_size);
  return grid_cell_index(mask, static_cast<int32_t>(m.x), static_cast<int32_t>(m.y), static_cast<int32_t>(m.z));
}

template <bool SP>
DEV V3 grid_gather(const DeviceScene& sc, const GridData& g, const VcmParams& it, const Isect& isect, PathState<SP>& state, uint32_t& candidates, uint32_t& accepts) {
  V3 merged = {0.0f, 0.0f, 0.0f};
  if (g.photon_count == 0) return merged;
  V3 pos = isect.pos;
  if (!((pos.x >= g.bbox_min.x) && (pos.y >= g.bbox_min.y) && (pos.z >= g.bbox_min.z) && (pos.x <= g.bbox_max.x) && (pos.y <= g.bbox_max.y) && (pos.z <= g.bbox_max.z)))
    return merged;
  V3 m = (pos - g.bbox_min) / g.cell_size;
  V3 mf = vfloor(m);
  V3 md = m - mf;
  int32_t acx = static_cast<int32_t>(mf.x), acy = static_cast<int32_t>(mf.y), acz = static_cast<int32_t>(mf.z);
  int32_t bcx = acx + ((md.x < 0.5f) ? -1 : +1);
  int32_t bcy = acy + ((md.y < 0.5f) ? -1 : +1);
  int32_t bcz = acz + ((md.z < 0.5f) ? -1 : +1);

  const etxb_material& mat = sc.materials[isect.material_index];
  BData camera_data = make_bdata(isect, isect.w_i, state.wavelength, state.medium_index, kPathCamera);
  const float w_camera_base = state.d_vcm * it.vc_weight;
  const bool use_mis = it.enable_mis();
  const bool use_epan = (it.kernel == 1u);

#pragma unroll 1
  for (uint32_t c = 0; c < 8; ++c) {
    uint32_t cell = grid_cell_index(g.hash_table_mask, (c & 1u) ? bcx : acx, (c & 2u) ? bcy : acy, (c & 4u) ? bcz : acz);
    uint2 range = __ldg(&g.cell_range[cell]);
    V3 cell_merged = {0.0f, 0.0f, 0.0f};
    for (uint32_t j = range.x; j < range.y; ++j) {
      float4 pd = __ldg(&g.pos_dvcm[j]);
      candidates += 1;
      V3 d = V3{pd.x, pd.y, pd.z} - pos;
      float distance_squared = dot(d, d);
      float4 wl = __ldg(&g.win_len[j]);
      if ((distance_squared > g.radius_squared) || (__float_as_uint(wl.w) + state.total_path_depth + 1 > sc.max_path_length)) continue;
      float4 nd = __ldg(&g.nrm_dvm[j]);
      if (dot(isect.nrm, V3{nd.x, nd.y, nd.z}) <= kEpsilon) continue;
      const V3 wi = {wl.x, wl.y, wl.z};
      BEval<SP> camera_bsdf = bsdf_evaluate<SP>(sc, camera_data, -wi, mat, state.sampler);
      if (camera_bsdf.valid() == false) continue;
      float camera_rev_pdf = bsdf_reverse_pdf<SP>(sc, camera_data, -wi, mat, state.sampler);
      accepts += 1;
      float w_light = pd.w * it.vc_weight + nd.w * camera_bsdf.pdf;
      float w_camera = w_camera_base + state.d_vm * camera_rev_pdf;
      float weight = use_mis ? (1.0f / (1.0f + w_light + w_camera)) : 1.0f;
      float kernel_weight = 1.0f;
      float u2 = distance_squared * g.inv_radius_squared;
      if (use_epan) {
        float one_minus = 1.0f - u2;
        kernel_weight = fmaxf(2.0f * one_minus, 0.0f);
      }
      Spec<SP> t_camera = state.throughput / sampling_pdf<SP>(state.wavelength);
      V3 c_value = spec_to_rgb<SP>(sc, camera_bsdf.func * t_camera, state.wavelength);
      float4 lt = __ldg(&g.thr_rgb[j]);
      V3 l_value = {lt.x, lt.y, lt.z};
      if (SP) {
        l_value *= V3{0.817660332f, 1.05418909f, 1.09945524f};
      }
      cell_merged += (c_value * l_value) * (kernel_weight * weight);
    }
    merged += cell_merged;
  }
  return merged;
}

}  // namespace etxb
