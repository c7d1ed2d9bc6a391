// tests/hostsim/camsim.cpp — TEST INFRASTRUCTURE.  The device math headers compiled as plain C++ (like hostsim.cpp)
// with the camera view type: each texel pair is shaded the way the cam_* kernels shade it (V = f2, LaneViews from
// camera_view, the kernels' light modes), so the CPU suite checks the camera path's arithmetic against the oracle
// without a GPU.  Build: g++ -O2 -ffp-contract=off -shared -fPIC (tests/test_camera_host.py does it).
#include <cstdint>

#include "pbr_shade.cuh"

using namespace pbr;

namespace {

typedef f2 V;

struct Dims {
  int B, H, W, L, wf;   // wf: 0 metallic (1-channel map), 1 specular, 2 metallic with a 3-channel map
};

// sums in double: [L][3] w.r.t. light position / unit direction, then [3] w.r.t. the camera position
struct HostGeomSink {
  static constexpr bool kOn = true;
  double* d_geo;
  int L;
  void light(int l, const float (&g)[3]) const { for (int c = 0; c < 3; ++c) d_geo[3 * l + c] += g[c]; }
  void view(const float (&g)[3]) const { for (int c = 0; c < 3; ++c) d_geo[3 * L + c] += g[c]; }
};

// one texel pair of material b at row yy, columns xx, xx + 1 (the second lane repeats the last column at a ragged edge)
struct Pair {
  int64_t o[2];
  int live;
  V a[3][1], n[3][1], r[1], m[3][1], x[1];
  float y;
  LaneViews<V, 1> cv;
  LightGeomT<V> hg[1];
};

template <int WF, int LIGHT>
void load_pair(const Dims& d, const CtStage& S, const float* cam, int b, int yy, int xx, const float* albedo,
               const float* normal, const float* rough, const float* metspec, Pair& p) {
  const int mc = WF == 0 ? 1 : 3;
  const int64_t HW = (int64_t)d.H * d.W;
  for (int k = 0; k < 2; ++k) p.o[k] = (int64_t)yy * d.W + (xx + k < d.W ? xx + k : d.W - 1);
  p.live = (xx + 2 <= d.W) ? 2 : d.W - xx;
  for (int k = 0; k < 2; ++k) {
    for (int c = 0; c < 3; ++c) lane_set(p.a[c][0], k, albedo[(b * 3 + c) * HW + p.o[k]]);
    for (int c = 0; c < 3; ++c) lane_set(p.n[c][0], k, normal ? normal[(b * 3 + c) * HW + p.o[k]] : (c == 2 ? 1.0f : 0.0f));
    lane_set(p.r[0], k, rough[b * HW + p.o[k]]);
    for (int c = 0; c < 3; ++c) lane_set(p.m[c][0], k, c < mc ? metspec[(b * mc + c) * HW + p.o[k]] : 0.0f);
    lane_set(p.x[0], k, linspace_at(S.lsx, xx + k < d.W ? xx + k : d.W - 1));
  }
  p.y = linspace_at(S.lsy, yy);
  camera_view(cam, p.x[0], p.y, p.cv.x[0], p.cv.y[0], p.cv.z[0], p.cv.len[0]);
  if (LIGHT == kLightPointHoisted)
    point_light_geom(S.light[0].p[0], S.light[0].p[1], S.light[0].p[2], p.x[0], p.y, p.cv.x[0], p.cv.y[0], p.cv.z[0], p.hg[0]);
}

template <int WF, int LIGHT>
void fwd_impl(const Dims& d, const CtStage& S, const CtFlags& F, const float* cam, const float* albedo, const float* normal,
              const float* rough, const float* metspec, float* out) {
  const int64_t HW = (int64_t)d.H * d.W;
  for (int b = 0; b < d.B; ++b)
    for (int yy = 0; yy < d.H; ++yy)
      for (int xx = 0; xx < d.W; xx += 2) {
        Pair p;
        load_pair<WF, LIGHT>(d, S, cam, b, yy, xx, albedo, normal, rough, metspec, p);
        auto emit = [&](int l, const V(&v)[3][1]) {
          for (int k = 0; k < p.live; ++k)
            for (int c = 0; c < 3; ++c)
              out[(F.per_light ? (((int64_t)b * d.L + l) * 3 + c) : ((int64_t)b * 3 + c)) * HW + p.o[k]] = lane_get(v[c][0], k);
        };
        ct_forward_group<WF, LIGHT, V, 1, decltype(emit), kFwdUnroll, LaneViews<V, 1>>(S, F, p.a, p.n, p.r, p.m, p.x, p.y, p.hg,
                                                                                     emit, GeomCache<V>(), p.cv);
      }
}

template <int WF, int LIGHT>
void bwd_impl(const Dims& d, const CtStage& S, const CtFlags& F, const float* cam, const float* albedo, const float* normal,
              const float* rough, const float* metspec, const float* grad_out, float* d_albedo, float* d_normal,
              float* d_rough, float* d_met, double* d_int, double* d_geo) {
  const int mc = WF == 0 ? 1 : 3;
  const int64_t HW = (int64_t)d.H * d.W;
  for (int b = 0; b < d.B; ++b)
    for (int yy = 0; yy < d.H; ++yy)
      for (int xx = 0; xx < d.W; xx += 2) {
        Pair p;
        load_pair<WF, LIGHT>(d, S, cam, b, yy, xx, albedo, normal, rough, metspec, p);
        auto gout = [&](int l, const V(&)[3][1], V(&g)[3][1]) {
          for (int c = 0; c < 3; ++c)
            for (int k = 0; k < 2; ++k) {
              const int64_t idx = (F.per_light ? (((int64_t)b * d.L + l) * 3 + c) : ((int64_t)b * 3 + c)) * HW + p.o[k];
              lane_set(g[c][0], k, k < p.live ? grad_out[idx] : 0.0f);   // a dropped lane contributes nothing
            }
        };
        auto sink = [&](int l, const float(&gi)[3]) {
          for (int c = 0; c < 3; ++c) d_int[3 * l + c] += gi[c];
        };
        V da[3][1], dn[3][1], dr[1], dm[3][1];
        ct_backward_group<WF, LIGHT, V, 1, decltype(gout), decltype(sink), NoFetch, HostGeomSink, NoSavedOut, kBwdUnroll,
                          LaneViews<V, 1>>(S, F, p.a, p.n, p.r, p.m, p.x, p.y, p.hg, gout, sink, da, dn, dr, dm, NoFetch(),
                                           GeomCache<V>(), HostGeomSink{d_geo, d.L}, NoSavedOut(), true, p.cv);
        for (int k = 0; k < p.live; ++k) {
          for (int c = 0; c < 3; ++c) d_albedo[(b * 3 + c) * HW + p.o[k]] = lane_get(da[c][0], k);
          if (normal)
            for (int c = 0; c < 3; ++c) d_normal[(b * 3 + c) * HW + p.o[k]] = lane_get(dn[c][0], k);
          d_rough[b * HW + p.o[k]] = lane_get(dr[0], k);
          for (int c = 0; c < mc; ++c) d_met[(b * mc + c) * HW + p.o[k]] = lane_get(dm[c][0], k);
        }
      }
}

void setup(const Dims& d, int point, float light_size, int albedo_is_srgb, int specular_is_srgb, int return_srgb,
           int per_light, const float* cam, const float* lights, const float* inten, CtStage& S, CtFlags& F) {
  stage_view(cam, S.vx, S.vy, S.vz);   // (unused by the camera path: the stage keeps the kernels' layout)
  const float s = light_size > 0.0f ? light_size : 1.0f;
  S.lsx = make_linspace(-s / 2, s / 2, d.W);
  S.lsy = make_linspace(-s / 2, s / 2, d.H);
  for (int l = 0; l < d.L; ++l) stage_light(l, lights, inten, point != 0, S.vx, S.vy, S.vz, S.light[l]);
  F.L = d.L;
  F.point = point != 0;
  F.albedo_is_srgb = albedo_is_srgb != 0;
  F.specular_is_srgb = specular_is_srgb != 0;
  F.return_srgb = return_srgb != 0;
  F.per_light = per_light != 0;
}

// the cam_* kernels' light modes
#define CAM_DISPATCH(fn, ...)                                                                   \
  do {                                                                                          \
    const int lm = !point ? kLightDirectional : (d.L == 1 ? kLightPointHoisted : kLightPoint);  \
    switch (d.wf * 3 + lm) {                                                                    \
      case 0: fn<0, 0>(__VA_ARGS__); break;                                                     \
      case 1: fn<0, 1>(__VA_ARGS__); break;                                                     \
      case 2: fn<0, 2>(__VA_ARGS__); break;                                                     \
      case 3: fn<1, 0>(__VA_ARGS__); break;                                                     \
      case 4: fn<1, 1>(__VA_ARGS__); break;                                                     \
      case 5: fn<1, 2>(__VA_ARGS__); break;                                                     \
      case 6: fn<2, 0>(__VA_ARGS__); break;                                                     \
      case 7: fn<2, 1>(__VA_ARGS__); break;                                                     \
      default: fn<2, 2>(__VA_ARGS__); break;                                                    \
    }                                                                                           \
  } while (0)

}  // namespace

extern "C" {

int cs_forward(int B, int H, int W, int L, int wf, int point, float light_size, int albedo_is_srgb, int specular_is_srgb,
               int return_srgb, int per_light, const float* cam, const float* lights, const float* inten,
               const float* albedo, const float* normal, const float* rough, const float* metspec, float* out) {
  if (L < 1 || L > PBR_MAX_LIGHTS || wf < 0 || wf > 2) return 1;
  const Dims d{B, H, W, L, wf};
  static CtStage S;
  CtFlags F;
  setup(d, point, light_size, albedo_is_srgb, specular_is_srgb, return_srgb, per_light, cam, lights, inten, S, F);
  CAM_DISPATCH(fwd_impl, d, S, F, cam, albedo, normal, rough, metspec, out);
  return 0;
}

// d_int [L][3], d_lights [L][3] (w.r.t. the positions, or the raw directions), d_cam [3]: sums in double
int cs_backward(int B, int H, int W, int L, int wf, int point, float light_size, int albedo_is_srgb, int specular_is_srgb,
                int return_srgb, int per_light, const float* cam, const float* lights, const float* inten,
                const float* albedo, const float* normal, const float* rough, const float* metspec, const float* grad_out,
                float* d_albedo, float* d_normal, float* d_rough, float* d_met, double* d_int, double* d_lights,
                double* d_cam) {
  if (L < 1 || L > PBR_MAX_LIGHTS || wf < 0 || wf > 2) return 1;
  const Dims d{B, H, W, L, wf};
  static CtStage S;
  CtFlags F;
  setup(d, point, light_size, albedo_is_srgb, specular_is_srgb, return_srgb, per_light, cam, lights, inten, S, F);
  double geo[(PBR_MAX_LIGHTS + 1) * 3] = {};
  for (int i = 0; i < 3 * L; ++i) d_int[i] = 0.0;
  CAM_DISPATCH(bwd_impl, d, S, F, cam, albedo, normal, rough, metspec, grad_out, d_albedo, d_normal, d_rough, d_met, d_int, geo);
  for (int l = 0; l < L; ++l) {
    float g[3] = {(float)geo[3 * l], (float)geo[3 * l + 1], (float)geo[3 * l + 2]}, o[3] = {g[0], g[1], g[2]};
    if (!point) normalize_bwd(lights + 3 * l, g, o);   // as the kernels' flush: the unit direction's Jacobian, once
    for (int c = 0; c < 3; ++c) d_lights[3 * l + c] = o[c];
  }
  for (int c = 0; c < 3; ++c) d_cam[c] = geo[3 * L + c];
  return 0;
}

}  // extern "C"
