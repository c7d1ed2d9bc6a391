// tests/hostsim/hostsim.cpp — TEST INFRASTRUCTURE.  Compiles the device math headers
// (pypbr_b200/csrc/pbr_math.cuh, pbr_shade.cuh) as plain C++ so the CPU suite can replay the golden
// vectors through the very expressions the CUDA kernels execute (only MUFU pow differs: powf here).
// Build: g++ -O2 -ffp-contract=off -shared -fPIC   (tests/conftest.py does it).
// Never loaded by the product package.
#include <cstdint>
#include <cstring>
#include <type_traits>
#include <vector>

#include "pbr_shade.cuh"

using namespace pbr;

namespace {

struct Dims {
  int B, H, W, L;
};

// sums in double: [L][3] w.r.t. light position / unit direction, then [3] w.r.t. the unit view direction (or the camera
// position)
struct HostGeomSink {
  static constexpr bool kOn = true;
  double* d_geo;
  int L;
  void light(int l, const float (&g)[3]) const { for (int c = 0; c < 3; ++c) d_geo[3 * l + c] += g[c]; }
  void view(const float (&g)[3]) const { for (int c = 0; c < 3; ++c) d_geo[3 * L + c] += g[c]; }
};

template <class V>
struct HostSavedOut {
  bool on;
  V out[3];
  bool have() const { return on; }
  void operator()(V (&o)[3][1]) const { for (int c = 0; c < 3; ++c) o[c][0] = out[c]; }
};

// kLightPointCached: what the kernels' prologue does per texel pair, with a private cache
template <int LIGHT, class V>
GeomCache<V> fill_cache(const CtStage& S, int L, V x, float y, V* store) {
  GeomCache<V> gc{store, 1, 1};
  if (is_cached(LIGHT))
    for (int l = 0; l < L; ++l) {
      LightGeomT<V> g;
      point_light_geom(S.light[l].p[0], S.light[l].p[1], S.light[l].p[2], x, y, S.vx, S.vy, S.vz, g);
      geom_cache_store<geom_fields(LIGHT), V>(gc, l, 0, g);
    }
  return gc;
}

// The view of one call's lane-values: the staged direction (OrthoView), or with CAM a camera at the position `cam`, what
// the kernels' cam_* entry points compute per texel (LaneViews from camera_view).
template <bool CAM, class V>
using ViewT = typename std::conditional<CAM, LaneViews<V, 1>, OrthoView>::type;
template <class V>
void fill_views(const float*, V, float, OrthoView&) {}
template <class V>
void fill_views(const float* cam, V x, float y, LaneViews<V, 1>& v) { camera_view(cam, x, y, v.x[0], v.y[0], v.z[0], v.len[0]); }

// per texel, as the kernels' grid_coords: the views, then the geometry of a hoisted point light
template <int LIGHT, bool CAM, class V>
void texel_views(const CtStage& S, const float* cam, V x, float y, ViewT<CAM, V>& views, LightGeomT<V>& hg) {
  fill_views(cam, x, y, views);
  if (LIGHT == kLightPointHoisted)
    point_light_geom(S.light[0].p[0], S.light[0].p[1], S.light[0].p[2], x, y, view_x(S, views, 0), view_y(S, views, 0),
                     view_z(S, views, 0), hg);
}

// One call shades Lanes<V>::n horizontally adjacent texels (V = float: 1, V = f2: 2, the packing the
// CUDA kernels use); at a ragged right edge the second lane repeats the last column and is dropped.
template <int WF, bool HASN, int LIGHT, class V, bool CAM = false>
void fwd_impl(const Dims& d, const CtStage& S, const CtFlags& F, const float* albedo, const float* normal,
              const float* rough, const float* metspec, float* out, const float* cam = nullptr) {
  constexpr int NL = Lanes<V>::n;
  const int mc = WF == 0 ? 1 : 3;  // WF 2: metallic with 3 channels
  const int64_t HW = (int64_t)d.H * d.W;
  for (int b = 0; b < d.B; ++b)
    for (int yy = 0; yy < d.H; ++yy)
      for (int xx = 0; xx < d.W; xx += NL) {
        int64_t o[2];
        for (int k = 0; k < NL; ++k) o[k] = (int64_t)yy * d.W + (xx + k < d.W ? xx + k : d.W - 1);
        const int live = (xx + NL <= d.W) ? NL : d.W - xx;
        V a[3][1], n[3][1], r[1], m[3][1], x[1];
        for (int k = 0; k < NL; ++k) {
          for (int c = 0; c < 3; ++c) lane_set(a[c][0], k, albedo[(b * 3 + c) * HW + o[k]]);
          for (int c = 0; c < 3; ++c) lane_set(n[c][0], k, HASN ? normal[(b * 3 + c) * HW + o[k]] : (c == 2 ? 1.0f : 0.0f));
          lane_set(r[0], k, rough[b * HW + o[k]]);
          for (int c = 0; c < 3; ++c) lane_set(m[c][0], k, c < mc ? metspec[(b * mc + c) * HW + o[k]] : 0.0f);
          lane_set(x[0], k, linspace_at(S.lsx, xx + k < d.W ? xx + k : d.W - 1));
        }
        float y = linspace_at(S.lsy, yy);
        auto emit = [&](int l, const V(&v)[3][1]) {
          for (int k = 0; k < live; ++k)
            for (int c = 0; c < 3; ++c) {
              int64_t idx = F.per_light ? (((int64_t)b * d.L + l) * 3 + c) * HW + o[k] : ((int64_t)b * 3 + c) * HW + o[k];
              out[idx] = lane_get(v[c][0], k);
            }
        };
        ViewT<CAM, V> views;
        LightGeomT<V> hg[1];
        texel_views<LIGHT, CAM>(S, cam, x[0], y, views, hg[0]);
        V store[PBR_MAX_LIGHTS * 8];
        ct_forward_group<WF, LIGHT, V, 1>(S, F, a, n, r, m, x, y, hg, emit, fill_cache<LIGHT, V>(S, d.L, x[0], y, store),
                                          views);
      }
}

template <int WF, bool HASN, int LIGHT, class V, bool CAM = false>
void bwd_impl(const Dims& d, const CtStage& S, const CtFlags& F, const float* albedo, const float* normal,
              const float* rough, const float* metspec, const float* grad_out, const float* target,
              float loss_scale, double* loss_sum, float* d_albedo, float* d_normal, float* d_rough, float* d_met,
              double* d_int, double* d_geo = nullptr, bool use_saved_out = false, const float* cam = nullptr) {
  constexpr int NL = Lanes<V>::n;
  const int mc = WF == 0 ? 1 : 3;  // WF 2: metallic with 3 channels
  const int64_t HW = (int64_t)d.H * d.W;
  for (int b = 0; b < d.B; ++b)
    for (int yy = 0; yy < d.H; ++yy)
      for (int xx = 0; xx < d.W; xx += NL) {
        int64_t o[2];
        for (int k = 0; k < NL; ++k) o[k] = (int64_t)yy * d.W + (xx + k < d.W ? xx + k : d.W - 1);
        const int live = (xx + NL <= d.W) ? NL : d.W - xx;
        V a[3][1], n[3][1], r[1], m[3][1], x[1];
        for (int k = 0; k < NL; ++k) {
          for (int c = 0; c < 3; ++c) lane_set(a[c][0], k, albedo[(b * 3 + c) * HW + o[k]]);
          for (int c = 0; c < 3; ++c) lane_set(n[c][0], k, HASN ? normal[(b * 3 + c) * HW + o[k]] : (c == 2 ? 1.0f : 0.0f));
          lane_set(r[0], k, rough[b * HW + o[k]]);
          for (int c = 0; c < 3; ++c) lane_set(m[c][0], k, c < mc ? metspec[(b * mc + c) * HW + o[k]] : 0.0f);
          lane_set(x[0], k, linspace_at(S.lsx, xx + k < d.W ? xx + k : d.W - 1));
        }
        float y = linspace_at(S.lsy, yy);
        auto gout = [&](int l, const V(&outv)[3][1], V(&g)[3][1]) {
          for (int c = 0; c < 3; ++c)
            for (int k = 0; k < NL; ++k) {
              if (k >= live) {  // dropped lane: contributes nothing (the kernels zero it the same way)
                lane_set(g[c][0], k, 0.0f);
                continue;
              }
              int64_t idx = F.per_light ? (((int64_t)b * d.L + l) * 3 + c) * HW + o[k] : ((int64_t)b * 3 + c) * HW + o[k];
              if (target) {
                float diff = lane_get(outv[c][0], k) - target[idx];
                *loss_sum += (double)diff * diff;
                lane_set(g[c][0], k, 2.0f * loss_scale * diff);
              } else {
                lane_set(g[c][0], k, grad_out[idx]);
              }
            }
        };
        auto sink = [&](int l, const float(&gi)[3]) {
          if (d_int)
            for (int c = 0; c < 3; ++c) d_int[3 * l + c] += gi[c];
        };
        V da[3][1], dn[3][1], dr[1], dm[3][1];
        ViewT<CAM, V> views;
        LightGeomT<V> hg[1];
        texel_views<LIGHT, CAM>(S, cam, x[0], y, views, hg[0]);
        V store[PBR_MAX_LIGHTS * 8];
        // accumulate mode, L > 1, "saved forward output" flavour: what the forward launch wrote for these texels
        HostSavedOut<V> saved{false, {}};
        if (use_saved_out && !F.per_light && d.L > 1) {
          auto keep = [&](int, const V(&v)[3][1]) { for (int c = 0; c < 3; ++c) saved.out[c] = v[c][0]; };
          ct_forward_group<WF, LIGHT, V, 1>(S, F, a, n, r, m, x, y, hg, keep, fill_cache<LIGHT, V>(S, d.L, x[0], y, store));
          saved.on = true;
        }
        bool done = false;
        if constexpr (LIGHT == kLightDirectional || LIGHT == kLightPoint || (CAM && LIGHT == kLightPointHoisted)) {
          if (d_geo) {   // gradients of the light positions / directions and of the view direction (camera position)
            ct_backward_group<WF, LIGHT, V, 1>(S, F, a, n, r, m, x, y, hg, gout, sink, da, dn, dr, dm, NoFetch(),
                                               GeomCache<V>(), HostGeomSink{d_geo, d.L}, saved, true, views);
            done = true;
          }
        }
        if (!done)
          ct_backward_group<WF, LIGHT, V, 1>(S, F, a, n, r, m, x, y, hg, gout, sink, da, dn, dr, dm, NoFetch(),
                                             fill_cache<LIGHT, V>(S, d.L, x[0], y, store), NoGeomSink(), saved, true, views);
        for (int k = 0; k < live; ++k) {
          for (int c = 0; c < 3; ++c) d_albedo[(b * 3 + c) * HW + o[k]] = lane_get(da[c][0], k);
          if (HASN && d_normal)
            for (int c = 0; c < 3; ++c) d_normal[(b * 3 + c) * HW + o[k]] = lane_get(dn[c][0], k);
          d_rough[b * HW + o[k]] = lane_get(dr[0], k);
          for (int c = 0; c < mc; ++c) d_met[(b * mc + c) * HW + o[k]] = lane_get(dm[c][0], k);
        }
      }
}

void make_stage(const Dims& d, int light_type, float light_size, const float* view, const float* lights,
                const float* inten, CtStage& S) {
  stage_view(view, S.vx, S.vy, S.vz);
  float s = light_size > 0.0f ? light_size : 1.0f;
  S.lsx = make_linspace(-s / 2, s / 2, d.W);
  S.lsy = make_linspace(-s / 2, s / 2, d.H);
  for (int l = 0; l < d.L; ++l) stage_light(l, lights, inten, light_type == 1, S.vx, S.vy, S.vz, S.light[l]);
}

// light mode: directional / point / point-hoisted (the kernels pick the hoisted variant for L == 1) / point-cached
// (the kernels pick it for L > 1 when a thread walks over several materials).
// `force_generic` bit 0: generic light mode; bit 1: V = f2 (two texels per call, the packing of the CUDA kernels);
// bit 2: point lights with L > 1 go through the geometry cache (kLightPointCached); bits 2+3: kLightPointCachedAll.
// CAM: the camera at a finite position, whose kernels have no cached mode: with force_generic 0 the same formula picks their
// directional / per-texel point / hoisted modes, and the cached cases compile nothing of their own.
#define DISPATCH_LM(fn, WF, HN, V, CAM, ...)                             \
  switch (lm) {                                                           \
    case 0: fn<WF, HN, 0, V, CAM>(__VA_ARGS__); break;                    \
    case 1: fn<WF, HN, 1, V, CAM>(__VA_ARGS__); break;                    \
    case 2: fn<WF, HN, 2, V, CAM>(__VA_ARGS__); break;                    \
    case 3: fn<WF, HN, (CAM ? 1 : 3), V, CAM>(__VA_ARGS__); break;        \
    default: fn<WF, HN, (CAM ? 1 : 4), V, CAM>(__VA_ARGS__); break;       \
  }
#define DISPATCH_V(fn, V, CAM, ...)                                                                       \
  do {                                                                                                     \
    int lm = light_type == 1 ? ((L == 1 && !(force_generic & 1)) ? 2 : ((L > 1 && (force_generic & 4)) ? ((force_generic & 8) ? 4 : 3) : 1)) : 0; \
    switch (workflow * 2 + (normal != nullptr)) {                                                          \
      case 0: DISPATCH_LM(fn, 0, false, V, CAM, __VA_ARGS__) break;                                        \
      case 1: DISPATCH_LM(fn, 0, true, V, CAM, __VA_ARGS__) break;                                         \
      case 2: DISPATCH_LM(fn, 1, false, V, CAM, __VA_ARGS__) break;                                        \
      case 3: DISPATCH_LM(fn, 1, true, V, CAM, __VA_ARGS__) break;                                         \
      case 4: DISPATCH_LM(fn, 2, false, V, CAM, __VA_ARGS__) break;                                        \
      case 5: DISPATCH_LM(fn, 2, true, V, CAM, __VA_ARGS__) break;                                         \
    }                                                                                                      \
  } while (0)
#define DISPATCH(fn, ...)                                                                   \
  do {                                                                                      \
    if (force_generic & 2) DISPATCH_V(fn, f2, false, __VA_ARGS__);                          \
    else DISPATCH_V(fn, float, false, __VA_ARGS__);                                         \
  } while (0)

// the kernels' flush of the geometry gradients: the Jacobians of F.normalize(dir) / F.normalize(view) applied once to the
// sums (`view` null: the sum is already w.r.t. the camera position)
void flush_geom(const std::vector<double>& geo, int L, int light_type, const float* lights, const float* view,
                double* d_lights, double* d_view) {
  for (int l = 0; l <= L; ++l) {
    const float g[3] = {(float)geo[3 * l], (float)geo[3 * l + 1], (float)geo[3 * l + 2]};
    float o[3] = {g[0], g[1], g[2]};
    if (l == L && view) normalize_bwd(view, g, o);
    else if (l < L && light_type != 1) normalize_bwd(lights + 3 * l, g, o);
    double* dst = l == L ? d_view : d_lights + 3 * l;
    for (int c = 0; c < 3; ++c) dst[c] = o[c];
  }
}

}  // namespace

extern "C" {

int hs_ct_forward(int B, int H, int W, int L, int workflow, int light_type, int albedo_is_srgb, int specular_is_srgb,
                  int return_srgb, int per_light, float light_size, const float* albedo, const float* normal,
                  const float* rough, const float* metspec, const float* view, const float* lights,
                  const float* inten, float* out, int force_generic) {
  if (L > PBR_MAX_LIGHTS) return -4;
  Dims d{B, H, W, L};
  static CtStage S;
  make_stage(d, light_type, light_size, view, lights, inten, S);
  CtFlags F{L, light_type == 1, albedo_is_srgb != 0, specular_is_srgb != 0, return_srgb != 0, per_light != 0};
  DISPATCH(fwd_impl, d, S, F, albedo, normal, rough, metspec, out);
  return 0;
}

int hs_ct_backward(int B, int H, int W, int L, int workflow, int light_type, int albedo_is_srgb, int specular_is_srgb,
                   int return_srgb, int per_light, float light_size, const float* albedo, const float* normal,
                   const float* rough, const float* metspec, const float* view, const float* lights,
                   const float* inten, const float* grad_out, const float* target, float loss_scale,
                   double* loss_sum, float* d_albedo, float* d_normal, float* d_rough, float* d_met, double* d_int,
                   int force_generic) {
  if (L > PBR_MAX_LIGHTS) return -4;
  Dims d{B, H, W, L};
  static CtStage S;
  make_stage(d, light_type, light_size, view, lights, inten, S);
  CtFlags F{L, light_type == 1, albedo_is_srgb != 0, specular_is_srgb != 0, return_srgb != 0, per_light != 0};
  // bit 4 of force_generic: accumulate-mode backward in one pass from the saved forward output (PbrCtGrads.fwd_out)
  DISPATCH(bwd_impl, d, S, F, albedo, normal, rough, metspec, grad_out, target, loss_scale, loss_sum, d_albedo,
           d_normal, d_rough, d_met, d_int, nullptr, (force_generic & 16) != 0);
  return 0;
}

// As hs_ct_backward, plus d_lights (L*3) and d_view (3): gradients w.r.t. the light positions / raw directions and the raw
// view direction.  Always the uncached per-texel light modes (what the kernels pick when these are requested).
int hs_ct_backward_geom(int B, int H, int W, int L, int workflow, int light_type, int albedo_is_srgb, int specular_is_srgb,
                        int return_srgb, int per_light, float light_size, const float* albedo, const float* normal,
                        const float* rough, const float* metspec, const float* view, const float* lights,
                        const float* inten, const float* grad_out, const float* target, float loss_scale,
                        double* loss_sum, float* d_albedo, float* d_normal, float* d_rough, float* d_met, double* d_int,
                        double* d_lights, double* d_view, int force_generic) {
  if (L > PBR_MAX_LIGHTS) return -4;
  Dims d{B, H, W, L};
  static CtStage S;
  make_stage(d, light_type, light_size, view, lights, inten, S);
  CtFlags F{L, light_type == 1, albedo_is_srgb != 0, specular_is_srgb != 0, return_srgb != 0, per_light != 0};
  std::vector<double> geo(3 * L + 3, 0.0);
  force_generic = (force_generic & 2) | 1;
  DISPATCH(bwd_impl, d, S, F, albedo, normal, rough, metspec, grad_out, target, loss_scale, loss_sum, d_albedo,
           d_normal, d_rough, d_met, d_int, geo.data());
  flush_geom(geo, L, light_type, lights, view, d_lights, d_view);
  return 0;
}

// A camera at a finite position (view_type="point"): `cam` is its position, the texels are shaded as the kernels' kCam
// instantiations shade them (V = f2, per-texel views, directional / per-texel point / hoisted lights).  d_int, d_lights
// [L][3] and d_cam [3] are sums in double; d_int is accumulated into.
int hs_ct_forward_camera(int B, int H, int W, int L, int workflow, int light_type, float light_size, int albedo_is_srgb,
                         int specular_is_srgb, int return_srgb, int per_light, const float* cam, const float* lights,
                         const float* inten, const float* albedo, const float* normal, const float* rough,
                         const float* metspec, float* out) {
  if (L > PBR_MAX_LIGHTS) return -4;
  Dims d{B, H, W, L};
  static CtStage S;
  make_stage(d, light_type, light_size, cam, lights, inten, S);
  CtFlags F{L, light_type == 1, albedo_is_srgb != 0, specular_is_srgb != 0, return_srgb != 0, per_light != 0};
  const int force_generic = 0;
  DISPATCH_V(fwd_impl, f2, true, d, S, F, albedo, normal, rough, metspec, out, cam);
  return 0;
}

int hs_ct_backward_camera(int B, int H, int W, int L, int workflow, int light_type, float light_size, int albedo_is_srgb,
                          int specular_is_srgb, int return_srgb, int per_light, const float* cam, const float* lights,
                          const float* inten, const float* albedo, const float* normal, const float* rough,
                          const float* metspec, const float* grad_out, float* d_albedo, float* d_normal, float* d_rough,
                          float* d_met, double* d_int, double* d_lights, double* d_cam) {
  if (L > PBR_MAX_LIGHTS) return -4;
  Dims d{B, H, W, L};
  static CtStage S;
  make_stage(d, light_type, light_size, cam, lights, inten, S);
  CtFlags F{L, light_type == 1, albedo_is_srgb != 0, specular_is_srgb != 0, return_srgb != 0, per_light != 0};
  std::vector<double> geo(3 * L + 3, 0.0);
  const int force_generic = 0;
  DISPATCH_V(bwd_impl, f2, true, d, S, F, albedo, normal, rough, metspec, grad_out, nullptr, 0.0f, nullptr, d_albedo,
             d_normal, d_rough, d_met, d_int, geo.data(), false, cam);
  flush_geom(geo, L, light_type, lights, nullptr, d_lights, d_cam);
  return 0;
}

void hs_convert_m2s(int64_t n_texels, int albedo_is_srgb, const float* albedo, const float* met, float* diffuse,
                    float* specular) {
  // single material (3, n_texels) planar
  for (int64_t i = 0; i < n_texels; ++i) {
    float a[3] = {albedo[i], albedo[n_texels + i], albedo[2 * n_texels + i]}, dd[3], ss[3];
    const float m3[3] = {met[i], met[i], met[i]};
    convert_m2s(a, m3, albedo_is_srgb != 0, dd, ss);
    for (int c = 0; c < 3; ++c) {
      diffuse[c * n_texels + i] = dd[c];
      specular[c * n_texels + i] = ss[c];
    }
  }
}

void hs_convert_s2m(int64_t n, int albedo_is_srgb, const float* diffuse, const float* specular, float* basecolor,
                    float* metallic) {
  for (int64_t i = 0; i < n; ++i) convert_s2m(diffuse[i], specular[i], albedo_is_srgb != 0, &basecolor[i], &metallic[i]);
}

void hs_blend(int64_t n_texels, int channels, int is_normal, const float* mask, const float* a, const float* b,
              float* out) {
  for (int64_t i = 0; i < n_texels; ++i) {
    if (is_normal) {
      float aa[3] = {a[i], a[n_texels + i], a[2 * n_texels + i]};
      float bb[3] = {b[i], b[n_texels + i], b[2 * n_texels + i]};
      float o[3];
      blend_normal(mask[i], aa, bb, o);
      for (int c = 0; c < 3; ++c) out[c * n_texels + i] = o[c];
    } else {
      for (int c = 0; c < channels; ++c) out[c * n_texels + i] = blend_lerp(mask[i], a[c * n_texels + i], b[c * n_texels + i]);
    }
  }
}

void hs_sigmoid_mask(int64_t n, const float* p1, const float* p2, float shift, int apply_shift, float blend_width,
                     float* out) {
  float w = blend_width + 1e-6f;
  for (int64_t i = 0; i < n; ++i) out[i] = sigmoid_mask(p1[i], p2[i], shift, apply_shift != 0, w);
}

void hs_linspace(float start, float end, int n, float* out) {
  Linspace ls = make_linspace(start, end, n);
  for (int i = 0; i < n; ++i) out[i] = linspace_at(ls, i);
}

void hs_srgb(int64_t n, int to_linear, const float* in, float* out) {
  for (int64_t i = 0; i < n; ++i)
    out[i] = to_linear ? srgb_decode<false, float>(in[i], nullptr) : srgb_encode<false, float>(in[i], nullptr);
}

void hs_ingest_normal(int64_t n_texels, int channels, const float* in, float* out) {
  for (int64_t i = 0; i < n_texels; ++i) {
    float o[3];
    if (channels == 3) {
      float v[3] = {in[i], in[n_texels + i], in[2 * n_texels + i]};
      ingest_normal3(v, o);
    } else {
      float v[2] = {in[i], in[n_texels + i]};
      ingest_normal2(v, o);
    }
    for (int c = 0; c < 3; ++c) out[c * n_texels + i] = o[c];
  }
}

// ---- adjoints of the streaming kernels (pbr_grad_kernels.cuh runs these per texel)
void hs_convert_m2s_bwd(int64_t n, int albedo_is_srgb, int met_channels, const float* albedo, const float* met, const float* g0,
                        const float* g1, float* d_albedo, float* d_met) {
  for (int64_t i = 0; i < n; ++i) {
    const float a[3] = {albedo[i], albedo[n + i], albedo[2 * n + i]};
    const float m3[3] = {met[i], met_channels == 3 ? met[n + i] : met[i], met_channels == 3 ? met[2 * n + i] : met[i]};
    const float gd[3] = {g0[i], g0[n + i], g0[2 * n + i]}, gs[3] = {g1[i], g1[n + i], g1[2 * n + i]};
    float da[3], dm[3];
    convert_m2s_bwd(a, m3, albedo_is_srgb != 0, gd, gs, da, dm);
    for (int c = 0; c < 3; ++c) d_albedo[c * n + i] = da[c];
    if (met_channels == 3) for (int c = 0; c < 3; ++c) d_met[c * n + i] = dm[c];
    else d_met[i] = (dm[0] + dm[1]) + dm[2];
  }
}

void hs_convert_s2m_bwd(int64_t n, int albedo_is_srgb, const float* diffuse, const float* specular, const float* g_b, const float* g_m,
                        float* d_albedo, float* d_spec) {
  for (int64_t i = 0; i < n; ++i) convert_s2m_bwd(diffuse[i], specular[i], albedo_is_srgb != 0, g_b[i], g_m[i], &d_albedo[i], &d_spec[i]);
}

// one map of a blend: d_a, d_b, and dmask += this map's contribution
void hs_blend_bwd(int64_t n, int channels, int is_normal, const float* mask, const float* a, const float* b, const float* g,
                  float* d_a, float* d_b, float* dmask) {
  for (int64_t i = 0; i < n; ++i) {
    if (is_normal) {
      const float aa[3] = {a[i], a[n + i], a[2 * n + i]}, bb[3] = {b[i], b[n + i], b[2 * n + i]}, gg[3] = {g[i], g[n + i], g[2 * n + i]};
      float da[3], db[3];
      dmask[i] += blend_normal_bwd(mask[i], aa, bb, gg, da, db);
      for (int c = 0; c < 3; ++c) { d_a[c * n + i] = da[c]; d_b[c * n + i] = db[c]; }
    } else {
      for (int c = 0; c < channels; ++c) {
        const float go = g[c * n + i];
        dmask[i] += go * (a[c * n + i] - b[c * n + i]);
        d_a[c * n + i] = mask[i] * go;
        d_b[c * n + i] = (1.0f - mask[i]) * go;
      }
    }
  }
}

void hs_ingest_normal_bwd(int64_t n, int channels, const float* in, const float* g, float* d_in) {
  for (int64_t i = 0; i < n; ++i) {
    const float gg[3] = {g[i], g[n + i], g[2 * n + i]};
    if (channels == 3) {
      const float v[3] = {in[i], in[n + i], in[2 * n + i]};
      float d[3];
      ingest_normal3_bwd(v, gg, d);
      for (int c = 0; c < 3; ++c) d_in[c * n + i] = d[c];
    } else {
      const float v[2] = {in[i], in[n + i]};
      float d[2];
      ingest_normal2_bwd(v, gg, d);
      d_in[i] = d[0]; d_in[n + i] = d[1];
    }
  }
}

// Markstein division with a correctly rounded reciprocal vs IEEE division: returns mismatches.
int64_t hs_div_check(int64_t n, const float* a, const float* b) {
  int64_t bad = 0;
  for (int64_t i = 0; i < n; ++i) {
    float q = xdiv_r(a[i], b[i], xrcp(b[i]));
    float e = a[i] / b[i];
    if (memcmp(&q, &e, 4) != 0) ++bad;
  }
  return bad;
}

}  // extern "C"

extern "C" {
// seeded sqrt / reciprocal recurrences vs IEEE: mismatch counts (sqrt, reciprocal-of-sqrt-based division)
void hs_seeded_check(int64_t n, const float* ss, const float* num, int64_t* bad_sqrt, int64_t* bad_div) {
  *bad_sqrt = 0;
  *bad_div = 0;
  for (int64_t i = 0; i < n; ++i) {
    float seed;
    float len = sqrt_seeded(ss[i], &seed);
    float ref = sqrtf(ss[i]);
    if (memcmp(&len, &ref, 4) != 0) ++*bad_sqrt;
    float r = refine_rcp(ref, seed);
    float q = xdiv_r(num[i], ref, r);
    float e = num[i] / ref;
    if (memcmp(&q, &e, 4) != 0) ++*bad_div;
  }
}
}
