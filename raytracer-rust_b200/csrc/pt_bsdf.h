// pt_bsdf.h — Material::emitted / Material::scatter of every material, driven by explicit uniforms.
//   Lambertian, Metal, Dielectric, EmissiveLight, NullMaterial   src/material.rs:29-252
//   PlasticMaterial, CheckerTexture, RoughConductor (+helpers)   src/tungsten/materials.rs:12-377
// The weights returned are exactly what the reference's `scatter` returns (energy-losing quirks included).
//
// Uniform order per scatter (one Philox block, pt_philox.h):
//   Lambertian / checker : u0,u1 -> direction on S^2
//   Metal (fuzz > 0)      : u0,u1 -> direction, u2 -> radius^(1/3)        (uniform point in the unit ball)
//   Dielectric            : u0 -> reflect-vs-refract, only when not totally reflecting (material.rs:145)
//   Plastic               : u0 -> specular-vs-diffuse, then u1,u2 -> direction
//   RoughConductor        : u0,u1 -> half vector (sample_ggx / sample_beckmann)
// The reference draws its sphere points by rejection from a cube (src/vec3.rs:54-61); the direct map used here
// has the same distribution (uniform in the ball, uniform on the sphere once normalised).
#pragma once
#include "pt_math.h"
#include "pt_types.h"

namespace pt {

struct USeq {
  const float *u;
  int i;
  PT_HD float next() { return u[(i++) & 3]; }
};

PT_HD V3 sphere_point(float u0, float u1) {
  const float z = 1.0f - 2.0f * u0;
  const float r = sqrtf(fmaxf(0.0f, 1.0f - z * z));
  const float phi = 2.0f * kPi * u1;
  float s, c;
#if defined(__CUDA_ARCH__)
  sincosf(phi, &s, &c);
#else
  s = sinf(phi);
  c = cosf(phi);
#endif
  return v3(r * c, r * s, z);
}
// Vec3::random_in_unit_sphere(rng).normalized()
PT_HD V3 random_unit_vector(USeq &q) {
  const float u0 = q.next(), u1 = q.next();
  return normalized(sphere_point(u0, u1));
}
// Vec3::random_in_unit_sphere(rng)
PT_HD V3 random_in_unit_ball(USeq &q) {
  const float u0 = q.next(), u1 = q.next(), u2 = q.next();
  return sphere_point(u0, u1) * cbrtf(u2);
}

// material.rs:194-206 and tungsten/materials.rs:292-304
PT_HD V3 reflect_checked(V3 v, V3 n) {
  if (has_nan(v) || has_nan(n) || is_zero(n)) return v3(NAN, NAN, NAN);
  return v - n * 2.0f * dot(v, n);
}
PT_HD float powi5(float x) {  // f32::powi(5)
  const float x2 = x * x;
  const float x4 = x2 * x2;
  return x * x4;
}
PT_HD float schlick_reflectance(float cosine, float ref_idx_ratio) {  // material.rs:221-227
  float r0 = (1.0f - ref_idx_ratio) / (1.0f + ref_idx_ratio);
  r0 = r0 * r0;
  return r0 + (1.0f - r0) * powi5(1.0f - cosine);
}
PT_HD bool refract(V3 uv, V3 n, float etai_over_etat, V3 &out) {  // material.rs:208-219
  const float cos_theta = fminf(dot(-uv, n), 1.0f);
  const V3 perp = (uv + n * cos_theta) * etai_over_etat;
  const float par2 = 1.0f - length_squared(perp);
  if (par2 < 0.0f) return false;
  out = perp + n * (-sqrtf(par2));
  return true;
}
PT_HD int32_t f32_as_i32_sat(float f) {  // Rust `as i32`: saturating, NaN -> 0
  if (isnan_f(f)) return 0;
  if (f >= 2147483648.0f) return INT32_MAX;
  if (f <= -2147483648.0f) return INT32_MIN;
  return (int32_t)f;
}
PT_HD V3 checker_value(const DMaterial &m, V3 p) {  // tungsten/materials.rs:89-99
  const int32_t xc = f32_as_i32_sat(floorf(p.x * m.inv_scale));
  const int32_t yc = f32_as_i32_sat(floorf(p.y * m.inv_scale));
  const int32_t zc = f32_as_i32_sat(floorf(p.z * m.inv_scale));
  const int32_t s = (int32_t)((uint32_t)xc + (uint32_t)yc + (uint32_t)zc);
  if (s % 2 == 0) return v3(m.albedo[0], m.albedo[1], m.albedo[2]);  // Rust %: -1 % 2 == -1 -> "off"
  return v3(m.off_color[0], m.off_color[1], m.off_color[2]);
}
PT_HD V3 fresnel_conductor(float cos_theta, V3 eta, V3 k) {  // tungsten/materials.rs:184-202 (t4 = t2 as written)
  cos_theta = cos_theta < 0.0f ? 0.0f : (cos_theta > 1.0f ? 1.0f : cos_theta);
  const V3 cos2 = splat(cos_theta * cos_theta);
  const V3 sin2 = splat(1.0f) - cos2;
  const V3 eta2 = eta * eta;
  const V3 k2 = k * k;
  const V3 t0 = eta2 - k2 - sin2;
  const V3 a2plusb2 = sqrt3(t0 * t0 + splat(4.0f) * eta2 * k2);
  const V3 t1 = a2plusb2 + cos2;
  const V3 a = sqrt3((a2plusb2 + t0) * splat(0.5f));
  const V3 t2 = splat(2.0f * cos_theta) * a;
  const V3 rs = (t1 - t2) / (t1 + t2);
  const V3 t3 = cos2 * a2plusb2 + sin2 * sin2;
  const V3 t4 = t2;
  const V3 rp = rs * ((t3 - t4) / (t3 + t4));
  return (rs + rp) * splat(0.5f);
}
PT_HD float ggx_g1(float n_dot_x, float roughness) {  // tungsten/materials.rs:205-216
  if (n_dot_x <= 0.0f) return 0.0f;
  const float a = roughness * roughness;
  const float k = a / 2.0f;
  const float denom = n_dot_x * (1.0f - k) + k;
  if (denom < kEps) return 1.0f;
  return n_dot_x / denom;
}
PT_HD float beckmann_lambda(float a, float x) {  // tungsten/materials.rs:225-232
  const float t = 1.0f / (a * x);
  if (t < 1.6f) return (1.0f - 1.259f * t + 0.396f * t * t) / (3.535f * t + 2.181f * t * t);
  return 0.0f;
}
PT_HD V3 sample_half_vector(V3 n, float roughness, int distribution, USeq &q) {  // tungsten/materials.rs:236-290
  if (has_nan(n) || is_zero(n)) return v3(NAN, NAN, NAN);
  const float u1 = fmaxf(q.next(), 1e-6f);
  const float u2 = q.next();
  float theta_arg;
  if (distribution == 0) {  // Ggx
    const float a = roughness * roughness;
    theta_arg = a * a * (-logf(u1)) / (1.0f - u1);
  } else {  // Beckmann
    theta_arg = -(roughness * roughness * logf(u1));
  }
  if (isnan_f(theta_arg) || isinf_f(theta_arg) || theta_arg < 0.0f) return to_world(v3(0, 0, 1), n);
  const float theta = atanf(sqrtf(theta_arg));
  const float phi = 2.0f * kPi * u2;
  const float st = sinf(theta), ct = cosf(theta);
  const V3 h_local = v3(st * cosf(phi), st * sinf(phi), ct);
  if (has_nan(h_local)) return to_world(v3(0, 0, 1), n);
  return to_world(h_local, n);
}

PT_HD V3 mat_emitted(const DMaterial &m) {  // material.rs:18-20,188-190
  if (m.type == 4) return v3(m.albedo[0], m.albedo[1], m.albedo[2]);
  return v3(0, 0, 0);
}

// Returns true and fills (scattered ray, attenuation) like Some((ray, color)); false = None.
PT_HD bool mat_scatter(const DMaterial &m, V3 ray_d, V3 pos, V3 n, bool front_face, const float *u4, Ray &scattered,
                       V3 &attenuation) {
  USeq q{u4, 0};
  switch (m.type) {
    case 0:    // Lambertian solid      material.rs:48-70
    case 1: {  // Lambertian checker
      V3 dir = n + random_unit_vector(q);
      if (near_zero(dir)) dir = n;
      scattered = ray_new(pos + n * kEps, normalized(dir));
      attenuation = m.type == 0 ? v3(m.albedo[0], m.albedo[1], m.albedo[2]) : checker_value(m, pos);
      return true;
    }
    case 2: {  // Metal                 material.rs:88-109
      const V3 reflected = reflect_checked(normalized(ray_d), n);
      const V3 fuzzed = m.fuzz > 0.0f ? reflected + random_in_unit_ball(q) * m.fuzz : reflected;
      if (dot(fuzzed, n) > 0.0f) {
        scattered = ray_new(pos + n * kEps, normalized(fuzzed));
        attenuation = v3(m.albedo[0], m.albedo[1], m.albedo[2]);
        return true;
      }
      return false;
    }
    case 3: {  // Dielectric            material.rs:123-162
      const float ratio = front_face ? 1.0f / m.ior : m.ior / 1.0f;
      const V3 unit = normalized(ray_d);
      const float cos_theta = fminf(dot(-unit, n), 1.0f);
      const float sin2 = 1.0f - cos_theta * cos_theta;
      const bool cannot_refract = ratio * ratio * sin2 > 1.0f;
      const float reflectance = schlick_reflectance(cos_theta, 1.0f / ratio);
      V3 dir;
      if (cannot_refract || reflectance > q.next()) {
        dir = reflect_checked(unit, n);
      } else {
        V3 r;
        dir = refract(unit, n, ratio, r) ? r : reflect_checked(unit, n);
      }
      const V3 origin = dot(dir, n) > 0.0f ? pos + n * kEps : pos - n * kEps;
      scattered = ray_new(origin, normalized(dir));
      attenuation = v3(1, 1, 1);
      return true;
    }
    case 5: {  // PlasticMaterial       tungsten/materials.rs:30-65
      const float dn = dot(ray_d, n);
      const float cosine = dn > 0.0f ? m.ior * dn / length(ray_d) : -dn / length(ray_d);
      float r0 = (1.0f - m.ior) / (1.0f + m.ior);
      const float r0_sq = r0 * r0;
      const float reflect_prob = r0_sq + (1.0f - r0_sq) * powi5(1.0f - cosine);
      if (q.next() < reflect_prob) {
        scattered = ray_new(pos + n * kEps, normalized(reflect_plain(ray_d, n)));
        attenuation = v3(0.9f, 0.9f, 0.9f);
      } else {
        V3 dir = n + random_unit_vector(q);
        if (near_zero(dir)) dir = n;
        scattered = ray_new(pos + n * kEps, normalized(dir));
        attenuation = v3(m.albedo[0], m.albedo[1], m.albedo[2]);
      }
      return true;
    }
    case 6: {  // RoughConductor        tungsten/materials.rs:307-376
      if (has_nan(ray_d)) return false;
      if (has_nan(n) || is_zero(n)) return false;
      const V3 v = -normalized(ray_d);
      if (has_nan(v)) return false;
      const float rough = m.roughness;
      const V3 hv = sample_half_vector(n, rough, m.distribution, q);
      if (has_nan(hv)) return false;
      const V3 l = reflect_checked(-v, hv);
      if (has_nan(l)) return false;
      if (dot(l, n) <= 0.0f) return false;
      const float n_dot_l = fmaxf(dot(n, l), 0.0f);
      const float n_dot_v = fmaxf(dot(n, v), 0.0f);
      const float n_dot_h = fmaxf(dot(n, hv), 0.0f);
      const float v_dot_h = fmaxf(dot(v, hv), 0.0f);
      const float g = m.distribution == 0
                          ? ggx_g1(n_dot_v, rough) * ggx_g1(n_dot_l, rough)
                          : 1.0f / (1.0f + beckmann_lambda(rough, n_dot_v) + beckmann_lambda(rough, n_dot_l));
      const V3 fr = fresnel_conductor(v_dot_h, v3(m.eta[0], m.eta[1], m.eta[2]), v3(m.k[0], m.k[1], m.k[2]));
      const V3 num = fr * g * v_dot_h;
      const float den = n_dot_v * n_dot_h + kEps;
      attenuation = den > kEps ? v3(m.albedo[0], m.albedo[1], m.albedo[2]) * (num / den) : v3(0, 0, 0);
      scattered = ray_new(pos + n * kEps, normalized(l));
      return true;
    }
    default:  // EmissiveLight (4), NullMaterial (7): scatter -> None
      return false;
  }
}


// ---- next-event estimation (PTC_FLAG_NEE; no counterpart in the reference, whose integrator finds emitters by BSDF
// sampling alone, renderer.rs:19-65).  Everything below is derived FROM the reference's scatter(): the "BSDF" is the one
// its estimator implies, weight(wi) * pdf(wi), so that light sampling + MIS converges to the very image the reference's
// integrator converges to.
//
// Solid-angle density of the half vector sample_half_vector() draws, as a function of cos(theta_h) = n.h.
//   Beckmann : tan^2 = -alpha^2 ln u           ->  exp(-tan^2 / alpha^2) / (pi alpha^2 cos^3)       (= D cos)
//   "Ggx"    : tan^2 = a^2 g(u), a = alpha^2,  g(u) = -ln u / (1 - u), u in [1e-6, 1)  (tungsten/materials.rs:247-262; not the
//              GGX distribution: tan^2 never falls below a^2).  g is inverted by bisection; |g'| has a removable
//              singularity at u = 1, hence the series.
PT_HD float half_vector_pdf(float cos_h, float roughness, int distribution) {
  if (!(cos_h > 1e-6f)) return 0.0f;
  const float c2 = cos_h * cos_h;
  const float tan2 = fmaxf(1.0f - c2, 0.0f) / c2;
  const float c3 = c2 * cos_h;
  if (distribution != 0) {
    const float al2 = roughness * roughness;
    if (tan2 > 13.8155f * al2) return 0.0f;  // u1 is clamped to >= 1e-6
    return expf(-tan2 / al2) / (kPi * al2 * c3);
  }
  const float a2 = roughness * roughness * roughness * roughness;
  const float y = tan2 / a2;
  if (!(y > 1.0f) || y >= 13.8155f) return 0.0f;
  float lo = 1e-6f, hi = 1.0f;
  for (int it = 0; it < 26; it++) {
    const float mid = 0.5f * (lo + hi), w = 1.0f - mid;
    const float g = w < 0.05f ? 1.0f + w * (0.5f + w * (1.0f / 3.0f + w * 0.25f)) : -logf(mid) / w;
    if (g > y) lo = mid;  // g decreases
    else hi = mid;
  }
  const float u = 0.5f * (lo + hi), w = 1.0f - u;
  const float gp = w < 0.1f ? (0.5f + w * (1.0f / 6.0f + w * (1.0f / 12.0f))) / u : (w + u * logf(u)) / (u * w * w);
  return 1.0f / (kPi * a2 * c3 * gp);
}

PT_HD float plastic_reflect_prob(const DMaterial &m, V3 ray_d, V3 n) {  // tungsten/materials.rs:33-45, as in mat_scatter
  const float dn = dot(ray_d, n);
  const float cosine = dn > 0.0f ? m.ior * dn / length(ray_d) : -dn / length(ray_d);
  const float r0 = (1.0f - m.ior) / (1.0f + m.ior);
  const float r0_sq = r0 * r0;
  return r0_sq + (1.0f - r0_sq) * powi5(1.0f - cosine);
}

// f * cos of the continuous lobe scatter() samples at this hit, towards wi, and the solid-angle pdf with which scatter()
// itself generates wi.  false: the material has no lobe light sampling can use (mirror, glass, fuzzed metal, emitters).
PT_HD bool mat_eval_pdf(const DMaterial &m, V3 ray_d, V3 pos, V3 n, V3 wi, V3 &fcos, float &pdf) {
  fcos = v3(0, 0, 0);
  pdf = 0.0f;
  const float c = dot(n, wi);
  switch (m.type) {
    case 0:
    case 1: {  // cosine-weighted hemisphere (n + unit vector), weight = albedo
      if (!(c > 0.0f)) return true;
      pdf = c * (1.0f / kPi);
      fcos = (m.type == 0 ? v3(m.albedo[0], m.albedo[1], m.albedo[2]) : checker_value(m, pos)) * pdf;
      return true;
    }
    case 5: {  // diffuse branch, taken with probability 1 - reflect_prob, weight = albedo
      if (!(c > 0.0f)) return true;
      pdf = (1.0f - plastic_reflect_prob(m, ray_d, n)) * c * (1.0f / kPi);
      fcos = v3(m.albedo[0], m.albedo[1], m.albedo[2]) * pdf;
      return true;
    }
    case 6: {  // weight = albedo F G (v.h) / (n.v n.h + 1e-4), l = reflect(-v, h), pdf(l) = p_h / (4 v.h)
      if (!(c > 0.0f)) return true;
      const V3 v = -normalized(ray_d);
      const V3 hv = normalized(v + wi);
      const float n_dot_v = fmaxf(dot(n, v), 0.0f), n_dot_h = fmaxf(dot(n, hv), 0.0f), v_dot_h = fmaxf(dot(v, hv), 0.0f);
      if (!(v_dot_h > 1e-6f)) return true;
      const float ph = half_vector_pdf(n_dot_h, m.roughness, m.distribution);
      if (!(ph > 0.0f)) return true;
      pdf = ph / (4.0f * v_dot_h);
      const float g = m.distribution == 0
                          ? ggx_g1(n_dot_v, m.roughness) * ggx_g1(c, m.roughness)
                          : 1.0f / (1.0f + beckmann_lambda(m.roughness, n_dot_v) + beckmann_lambda(m.roughness, c));
      const V3 fr = fresnel_conductor(v_dot_h, v3(m.eta[0], m.eta[1], m.eta[2]), v3(m.k[0], m.k[1], m.k[2]));
      const float den = n_dot_v * n_dot_h + kEps;
      if (den > kEps) fcos = v3(m.albedo[0], m.albedo[1], m.albedo[2]) * fr * (g * v_dot_h / den * pdf);
      return true;
    }
    default:
      return false;
  }
}
// pdf of the direction scatter() just produced with uniforms u4, or -1 when it came from a delta / unsupported lobe
PT_HD float mat_sampled_pdf(const DMaterial &m, V3 ray_d, V3 pos, V3 n, const float *u4, V3 wi) {
  if (m.type == 5 && u4[0] < plastic_reflect_prob(m, ray_d, n)) return -1.0f;  // the mirror branch
  V3 fcos;
  float pdf;
  if (!mat_eval_pdf(m, ray_d, pos, n, wi, fcos, pdf)) return -1.0f;
  return pdf;
}

// A point on light L seen from x: direction, distance and solid-angle pdf (uniform over the light's area; the emitters are
// two-sided, material.rs:188-190).
PT_HD bool light_sample(const DLight &L, V3 x, float u0, float u1, V3 &wi, float &dist, float &pdf) {
  V3 y, nl;
  if (L.type == OBJ_SPHERE) {
    nl = sphere_point(u0, u1);
    y = v3(L.f[0], L.f[1], L.f[2]) + nl * L.f[3];
  } else {
    y = v3(L.f[0], L.f[1], L.f[2]) + v3(L.f[3], L.f[4], L.f[5]) * u0 + v3(L.f[6], L.f[7], L.f[8]) * u1;
    nl = v3(L.f[9], L.f[10], L.f[11]);
  }
  const V3 d = y - x;
  const float d2 = length_squared(d);
  if (!(d2 > 1e-12f)) return false;
  dist = sqrtf(d2);
  wi = d * (1.0f / dist);
  const float cos_l = fabsf(dot(nl, wi));
  if (!(cos_l > 1e-6f)) return false;
  pdf = d2 / (cos_l * L.area);
  return true;
}
// the same density for a point of L that a BSDF-sampled ray hit at distance `dist` under |cos| = cos_l
PT_HD float light_pdf(const DLight &L, float dist, float cos_l) { return cos_l > 1e-6f ? dist * dist / (cos_l * L.area) : 0.0f; }

// Sky / background for a ray that missed everything (renderer.rs:38-63)
PT_HD uint32_t f32_as_u32_sat(float f) {  // Rust `as u32`
  if (!(f > 0.0f)) return 0u;
  if (f >= 4294967296.0f) return 0xffffffffu;
  return (uint32_t)f;
}
// the texel of the HDR sky a direction looks up (renderer.rs:40-54); shared by sky_color and the sky light's pdf
PT_HD void sky_texel(const DScene &sc, V3 ray_d, uint32_t &xp, uint32_t &yp) {
  const V3 dir = normalized(ray_d);
  const float theta = acosf(dir.y);
  const float phi = atan2f(dir.z, dir.x) + kPi;
  const float u = phi / (2.0f * kPi);
  const float v = theta / kPi;
  xp = f32_as_u32_sat(fmaxf(u * (float)(sc.sky_w - 1), 0.0f));
  yp = f32_as_u32_sat(fmaxf(v * (float)(sc.sky_h - 1), 0.0f));
  if (xp > (uint32_t)(sc.sky_w - 1)) xp = (uint32_t)(sc.sky_w - 1);
  if (yp > (uint32_t)(sc.sky_h - 1)) yp = (uint32_t)(sc.sky_h - 1);
}
PT_HD V3 sky_color(const DScene &sc, V3 ray_d) {
  if (sc.sky != nullptr) {
    uint32_t xp, yp;
    sky_texel(sc, ray_d, xp, yp);
    const float *px = sc.sky + ((size_t)yp * sc.sky_w + xp) * 3;
    return v3(px[0], px[1], px[2]);
  }
  return v3(0.5f, 0.5f, 0.5f);  // Color::GRAY
}

// The HDR sky as a light (PTC_FLAG_NEE_SKY; layout and cell mapping: pt_types.h, SkyDist).  Needs sc.sky_dist != nullptr.
// P(cell) is a product of differences of the stored CDF entries the sampler searches, so sampler and pdf agree.
PT_HD float sky_cell_prob(const SkyDist &d, uint32_t x, uint32_t y) {
  const float *row = d.cond + (size_t)y * (uint32_t)(d.wc + 1);
  return (d.marg[y + 1] - d.marg[y]) * (row[x + 1] - row[x]);
}
// solid-angle density of direction ray_d (0 in the last texel column / row, which the lookup reaches on a null set only)
PT_HD float sky_pdf(const DScene &sc, V3 ray_d) {
  const SkyDist d = sky_dist_view(sc.sky_dist, sc.sky_w, sc.sky_h);
  uint32_t x, y;
  sky_texel(sc, ray_d, x, y);
  if (x >= (uint32_t)d.wc || y >= (uint32_t)d.hc) return 0.0f;
  return sky_cell_prob(d, x, y) * d.inv_sa[y];
}
// first i in [0, n) with cdf[i + 1] > u, for cdf[0] = 0 <= u < cdf[n] = 1: never an interval of width 0
PT_HD uint32_t cdf_search(const float *cdf, uint32_t n, float u) {
  uint32_t lo = 0, hi = n - 1;
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (cdf[mid + 1] > u) hi = mid;
    else lo = mid + 1;
  }
  return lo;
}
// a direction with density sky_pdf from four uniforms: row, column, then uniform in phi and cos(theta) inside the cell
// (uniform in solid angle), mapped back through the lookup's angles: atan2(z, x) = phi - pi, y = cos(theta)
PT_HD V3 sky_sample(const DScene &sc, const float *u4, float &pdf) {
  const SkyDist d = sky_dist_view(sc.sky_dist, sc.sky_w, sc.sky_h);
  const uint32_t y = cdf_search(d.marg, (uint32_t)d.hc, u4[0]);
  const uint32_t x = cdf_search(d.cond + (size_t)y * (uint32_t)(d.wc + 1), (uint32_t)d.wc, u4[1]);
  pdf = sky_cell_prob(d, x, y) * d.inv_sa[y];
  const float ct = d.cos[y] + u4[3] * (d.cos[y + 1] - d.cos[y]);
  const float st = sqrtf(fmaxf(0.0f, 1.0f - ct * ct));
  const float a = (2.0f * kPi) * (((float)x + u4[2]) / (float)d.wc) - kPi;
  float s, c;
#if defined(__CUDA_ARCH__)
  sincosf(a, &s, &c);
#else
  s = sinf(a);
  c = cosf(a);
#endif
  return v3(st * c, ct, st * s);
}

// Camera::get_ray (src/camera.rs:33-42)
struct DCamera {
  float position[3], forward[3], right[3], true_up[3];
  float half_width, half_height;
};
PT_HD Ray camera_get_ray(const DCamera &c, float u, float v) {
  const float ndc_x = 2.0f * u - 1.0f;
  const float ndc_y = 1.0f - 2.0f * v;
  const V3 right = v3(c.right[0], c.right[1], c.right[2]), up = v3(c.true_up[0], c.true_up[1], c.true_up[2]);
  const V3 fwd = v3(c.forward[0], c.forward[1], c.forward[2]);
  const V3 offset = right * (ndc_x * c.half_width) + up * (ndc_y * c.half_height);
  const V3 dir = normalized(fwd + offset);
  return ray_new(v3(c.position[0], c.position[1], c.position[2]), dir);
}

// renderer.rs:112-120 + color.rs:87-93: sqrt "gamma", clamp, *255, truncate, 0x00RRGGBB
PT_HD uint32_t resolve_channel(float c) {
  float r = sqrtf(c);
  if (r < 0.0f) r = 0.0f;  // f32::clamp keeps NaN; `as u32` then maps NaN to 0
  if (r > 1.0f) r = 1.0f;
  const float v = r * 255.0f;
  if (!(v > 0.0f)) return 0u;
  return (uint32_t)v;
}
PT_HD uint32_t resolve_pixel(float r, float g, float b) {
  return (resolve_channel(r) << 16) | (resolve_channel(g) << 8) | resolve_channel(b);
}

}  // namespace pt
