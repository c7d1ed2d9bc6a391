// pbr_shade.cuh — staging of the view / light parameters and the per-thread drivers that shade a
// group of N lane-values V (consecutive columns of one row) over L lights, forward and backward.
// V = f2 (two adjacent texels, packed FP32 math) in the CUDA kernels, V = float or f2 in the host
// build of the CPU test-suite.  CtStage lives in shared memory on the device.
#pragma once

#include "pbr_math.cuh"

namespace pbr {
// light-loop unrolling (independent chains for the scheduler), tuned on the GPU: the forward evaluation, pass 1 of the
// two-pass backward, and the main light loop of the backward
constexpr int kFwdUnroll = 1, kP1Unroll = 2, kBwdUnroll = 1;
}
#ifndef PBR_MAX_LIGHTS
#define PBR_MAX_LIGHTS 64
#endif

namespace pbr {

struct CtLight {
  float p[3];      // point: position; directional: raw direction
  float inten[3];
  LightGeom geom;  // directional lights: complete geometry (constant over the image)
};

// What the kernel prologue stages in shared memory.
struct CtStage {
  float vx, vy, vz;  // F.normalize(view_dir), cooktorrance.py:95
  Linspace lsx, lsy; // the plane grid of cooktorrance.py:132-133
  CtLight light[PBR_MAX_LIGHTS];
};

struct CtFlags {
  int L;
  bool point;             // light_type == point
  bool albedo_is_srgb, specular_is_srgb, return_srgb, per_light;
};

PBR_HD void stage_view(const float* view, float& vx, float& vy, float& vz) {
  float dn = fmaxf(xnorm3(view[0], view[1], view[2]), kNormEps);
  vx = xdiv(view[0], dn);
  vy = xdiv(view[1], dn);
  vz = xdiv(view[2], dn);
}

PBR_HD void stage_light(int l, const float* lights, const float* inten, bool point, float vx, float vy, float vz,
                        CtLight& out) {
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    out.p[c] = lights[3 * l + c];
    out.inten[c] = inten[3 * l + c];
  }
  if (!point) dir_light_geom(out.p[0], out.p[1], out.p[2], vx, vy, vz, out.geom);
}

// torch.linspace(-s/2, s/2, n) parameters, computed once on the host.
inline Linspace make_linspace(float start, float end, int n) {
  Linspace ls;
  ls.start = start;
  ls.end = end;
  ls.n = n;
  if (n <= 1) {  // aten fills [start]
    ls.step = 0.0f;
    ls.half = 1;
  } else {
    ls.step = (end - start) / (float)(n - 1);
    ls.half = n / 2;
  }
  return ls;
}

// How the per-texel light geometry is obtained.
enum LightMode {
  kLightDirectional = 0,  // constant over the image: read from the stage
  kLightPoint = 1,        // computed per texel and per light
  kLightPointHoisted = 2, // point light, L == 1: computed once per texel by the caller and reused for
                          // every material of the batch the thread walks over (geometry does not
                          // depend on the material)
  kLightPointCached = 3,  // point lights, L > 1: the caller computes the geometry of every light once per
                          // texel, parks it in its own shared-memory slots (GeomCache) and the light loops
                          // of all the materials it walks over read it back.  Caches l and h (6 fields).
  kLightPointCachedAll = 4,  // same with all 8 fields cached: for few lights, where the cache does not cost occupancy
  kLightPointCachedAllBig = 5   // all 8 fields, backward with the full register budget: 4 < L <= 8, where 2 CTAs per SM still fit
                                // (loss kernel at L = 8: 2.73 -> 2.68 ms per 32 x 1024^2, profiles/r2_tune_*.json)
};
// (Tried and dropped: caching h only - 3 fields - for the forward of many lights, so that the cache leaves room for 4 CTAs per
// SM instead of 2: l and the attenuation recomputed per light cost more than the occupancy gave back, 0.824 -> 0.912 ms at
// L = 16: that kernel is bound by the FP32 pipe, not by latency.)
PBR_HDC bool is_cached(int light_mode) { return light_mode >= kLightPointCached && light_mode <= kLightPointCachedAllBig; }
// Fields: l (3), h (3) [, p5, att].  The fields that are not cached are recomputed from the plane position
// (they live in the tolerant zone; l and h feed N.L / N.H and stay bit-exact).
PBR_HDC int geom_fields(int light_mode) { return (light_mode == kLightPointCachedAll || light_mode == kLightPointCachedAllBig) ? 8 : 6; }

// Per-thread geometry cache (kLightPointCached).  Field f of light l of lane-value i lives at
// base[(l * kGeomFields + f) * fstride + i * stride]; `base` already points at the calling thread's slot,
// `stride` is the thread count and `fstride` = lane-values per thread * stride, so a warp-level access touches
// consecutive 8-byte words (conflict-free LDS.64).
// A thread only ever reads what it wrote itself: no synchronisation.
template <class V>
struct GeomCache {
  V* base;
  int stride, fstride;
};

template <class V>
PBR_HD V p5_from_half(V hx, V hy, V hz, float vx, float vy, float vz) {
  V c = xdot3_sat(hx, hy, hz, splat<V>(vx), splat<V>(vy), splat<V>(vz));
  V omc = 1.0f - c;
  V o2 = omc * omc;
  return o2 * o2 * omc;
}

template <int kGeomFields, class V>
PBR_HD void geom_cache_store(const GeomCache<V>& gc, int l, int i, const LightGeomT<V>& g) {
  const int fs = gc.fstride;
  V* q = gc.base + (l * kGeomFields) * fs + i * gc.stride;
  q[0] = g.lx; q[fs] = g.ly; q[2 * fs] = g.lz;
  q[3 * fs] = g.hx; q[4 * fs] = g.hy; q[5 * fs] = g.hz;
  if (kGeomFields >= 7) q[6 * fs] = g.p5;
  if (kGeomFields >= 8) q[7 * fs] = g.att;
}

template <int kGeomFields, class V>
PBR_HD void geom_cache_load(const GeomCache<V>& gc, int l, int i, const float p[3], V x, float y, float vx, float vy,
                            float vz, LightGeomT<V>& g) {
  const int fs = gc.fstride;
  const V* q = gc.base + (l * kGeomFields) * fs + i * gc.stride;
  g.lx = q[0]; g.ly = q[fs]; g.lz = q[2 * fs];
  g.hx = q[3 * fs]; g.hy = q[4 * fs]; g.hz = q[5 * fs];
  if (kGeomFields >= 7) g.p5 = q[6 * fs];
  else g.p5 = p5_from_half(g.hx, g.hy, g.hz, vx, vy, vz);
  if (kGeomFields >= 8) {
    g.att = q[7 * fs];
  } else {
    // 1/(d^2 + 1e-7), cooktorrance.py:140: tolerant zone (scales the colour linearly)
    const float ly = p[1] + y;
    const float yz = ly * ly + p[2] * p[2];
    V Lx = splat<V>(p[0]) - x;
    g.att = fast_rcp(Lx * Lx + (yz + kEps7));
  }
}

// The view direction the group functions below shade with (template parameter View):
//   OrthoView : the CTA-uniform unit vector staged in CtStage (S.vx, S.vy, S.vz), the orthographic camera of the
//               reference - every ct_* kernel;
//   LaneViews : a camera at a finite position - the unit view vector of every lane-value and |c - P| for its adjoint
//               (camera_view in pbr_math.cuh), computed once per texel by the cam_* kernels.
struct OrthoView {};
template <class V, int N>
struct LaneViews {
  V x[N], y[N], z[N], len[N];
};
PBR_HD float view_x(const CtStage& S, const OrthoView&, int) { return S.vx; }
PBR_HD float view_y(const CtStage& S, const OrthoView&, int) { return S.vy; }
PBR_HD float view_z(const CtStage& S, const OrthoView&, int) { return S.vz; }
template <class V, int N> PBR_HD V view_x(const CtStage&, const LaneViews<V, N>& v, int i) { return v.x[i]; }
template <class V, int N> PBR_HD V view_y(const CtStage&, const LaneViews<V, N>& v, int i) { return v.y[i]; }
template <class V, int N> PBR_HD V view_z(const CtStage&, const LaneViews<V, N>& v, int i) { return v.z[i]; }
// directional light: l is image-constant, but with a per-texel view the half vector and (1 - h.v)^5 are per texel too
template <class V> PBR_HD void dir_view_geom(const OrthoView&, int, LightGeomT<V>&) {}
template <class V, int N> PBR_HD void dir_view_geom(const LaneViews<V, N>& v, int i, LightGeomT<V>& g) {
  half_vector(v.x[i], v.y[i], v.z[i], g);
}
// d/d unit view vector of lane-value i -> d/d camera position (in place); the orthographic view's Jacobian is applied
// once per CTA by the caller instead (it is image-constant)
template <class V> PBR_HD void view_bwd(const OrthoView&, int, V*) {}
template <class V, int N> PBR_HD void view_bwd(const LaneViews<V, N>& v, int i, V* g) {
  camera_view_bwd(v.x[i], v.y[i], v.z[i], v.len[i], g);
}

template <int kLight, class V, int N, class View = OrthoView>
PBR_HD void light_geom(const CtStage& S, int l, const V (&x)[N], float y, const LightGeomT<V> (&hoisted)[N], int i,
                       const GeomCache<V>& gc, LightGeomT<V>& g, const View& view = View()) {
  if (is_cached(kLight)) {   // (orthographic view only)
    geom_cache_load<geom_fields(kLight), V>(gc, l, i, S.light[l].p, x[i], y, S.vx, S.vy, S.vz, g);
  } else if (kLight == kLightPoint) {
    point_light_geom(S.light[l].p[0], S.light[l].p[1], S.light[l].p[2], x[i], y, view_x(S, view, i), view_y(S, view, i),
                     view_z(S, view, i), g);
  } else if (kLight == kLightPointHoisted) {
    g = hoisted[i];
  } else {
    g = splat_geom<V>(S.light[l].geom);
    dir_view_geom(view, i, g);
  }
}

// Saved forward outputs from which the gate / slope of encode(clamp(sum)) cannot be read off reliably:
//   out >= top : a sum of exactly 1, above 1, or within an ulp or two below 1 all encode to `top` (torch.clamp's gate is
//                inclusive at 1);
//   out within 5e-7 of the knee's image (sRGB only): the two branches of linear_to_srgb do not meet exactly at 0.0031308 -
//                the power branch starts 7e-8 BELOW 12.92 * knee - so a sum just above the knee encodes to a value the
//                linear branch also produces, and their slopes differ by 1.8 % (seen once in 12.6 M texels at the C3 shape).
// Those texels recompute the sum; everything else reads the slope off the output.
constexpr float kKneeImage = 12.92f * kSrgbEncKnee;   // 0.040449936
PBR_HD bool at_boundary(float v, float top, bool srgb) { return v >= top || (srgb && fabsf(v - kKneeImage) < 5e-7f); }
PBR_HD bool at_boundary(f2 v, float top, bool srgb) { return at_boundary(v.x, top, srgb) || at_boundary(v.y, top, srgb); }

// c is a colour the caller has just clamped to [0, 1]
template <class V>
PBR_HD V encode_out(V c, bool return_srgb) { return return_srgb ? srgb_encode01<false>(c, (V*)nullptr) : c; }
template <class V>
PBR_HD V encode_out_d(V c, bool return_srgb, V* d) {
  if (return_srgb) return srgb_encode01<true>(c, d);
  *d = splat<V>(1.0f);
  return c;
}

// ------------------------------------------------------------------------------------------------
// forward: N lane-values of one row.  emit(l, out[3][N]) receives the encoded colour of light l
// (per-light mode) or, once, of the accumulated image (l = 0).
// ------------------------------------------------------------------------------------------------
template <int kWorkflow, int kLight, class V, int N, class Emit, int kUnroll = kFwdUnroll, class View = OrthoView>
PBR_HD void ct_forward_group(const CtStage& S, const CtFlags& F, const V (&araw)[3][N], const V (&nraw)[3][N],
                             const V (&rough)[N], const V (&mraw)[3][N], const V (&x)[N], float y,
                             const LightGeomT<V> (&hoisted)[N], Emit emit, GeomCache<V> gc = GeomCache<V>(),
                             const View& view = View()) {
  Texel<kWorkflow, V> t[N];
#pragma unroll
  for (int i = 0; i < N; ++i) {
    const V a3[3] = {araw[0][i], araw[1][i], araw[2][i]};
    const V n3[3] = {nraw[0][i], nraw[1][i], nraw[2][i]};
    const V m3[3] = {mraw[0][i], mraw[1][i], mraw[2][i]};
    texel_setup<kWorkflow, false>(a3, n3, rough[i], m3, F.albedo_is_srgb, F.specular_is_srgb, view_x(S, view, i),
                                  view_y(S, view, i), view_z(S, view, i), t[i]);
  }
  V acc[3][N];
#pragma unroll
  for (int c = 0; c < 3; ++c)
#pragma unroll
    for (int i = 0; i < N; ++i) acc[c][i] = splat<V>(0.0f);

  const int L = (kLight == kLightPointHoisted) ? 1 : F.L;
#pragma unroll kUnroll
  for (int l = 0; l < L; ++l) {
    V outv[3][N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
      LightGeomT<V> g;
      light_geom<kLight, V, N>(S, l, x, y, hoisted, i, gc, g, view);
      LightFwd<V> f;
      V col[3];
      shade_light_fwd<kWorkflow, false>(t[i], g, S.light[l].inten, f, col);
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        if (F.per_light) outv[c][i] = encode_out(col[c], F.return_srgb);
        else acc[c][i] = xadd(acc[c][i], col[c]);
      }
    }
    if (F.per_light) emit(l, outv);
  }
  if (!F.per_light) {
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
      for (int i = 0; i < N; ++i) acc[c][i] = encode_out(clamp01(acc[c][i]), F.return_srgb);
    emit(0, acc);
  }
}

// ------------------------------------------------------------------------------------------------
// backward: N lane-values of one row.
//   gout(l, out[3][N], g[3][N]) : given the encoded output of light l (or of the accumulated image,
//        l = 0) fills g = dLoss/d out.  The plain backward ignores `out` and loads grad_out; the fused
//        loss kernel computes 2*scale*(out - target) and accumulates the loss.
//   fetch(-1)                   : called once after the light loop (the per-light registers are dead from here on);
//   fetch(l)                    : software prefetch hook of the generic kernels: "what was fetched last becomes
//        current, start loading the grad_out / target of light l" (l == L: rotate only).  gout(l) then reads the
//        current buffer, which was requested one whole light iteration earlier.
//   int_sink(l, g_int[3])       : per-light intensity gradient summed over the texels of the group (only called when
//        `want_int`, the last argument, is set).
//   gc                          : kLightPointCached only, the calling thread's geometry cache.
// Results: d_albedo/d_normal/d_met [3][N], d_rough[N].
// ------------------------------------------------------------------------------------------------
struct NoFetch {
  PBR_HD void operator()(int) const {}
};
//   geom_sink.light(l, g[3])    : (GeomSink != NoGeomSink only) gradient w.r.t. the position of point light l, or
//        w.r.t. the UNIT direction of directional light l, summed over the texels of the group;
//   geom_sink.view(g[3])        : gradient w.r.t. the UNIT view direction (OrthoView) or w.r.t. the camera position
//        (LaneViews), summed over the group's texels and lights.
struct NoGeomSink {
  static constexpr bool kOn = false;
  PBR_HD void light(int, const float (&)[3]) const {}
  PBR_HD void view(const float (&)[3]) const {}
};

//   saved_out                   : accumulate mode with L > 1 only.  saved_out.have() (uniform over the kernel): the
//        encoded output of the FORWARD launch is at hand (what autograd keeps anyway) and saved_out(out[3][N]) loads it;
//        the gate of clamp(sum) and the slope of the encode are then derived from it and pass 1 - a complete second
//        forward evaluation of every light - is skipped.
struct NoSavedOut {
  PBR_HD bool have() const { return false; }
  template <class V, int N>
  PBR_HD void operator()(V (&)[3][N]) const {}
};

// d encode(clamp(acc)) / d acc from out = encode(clamp(acc)) (utils/functions.py:50-66 inverted on its upper branch:
// t^(1/2.4 - 1) = u^-1.4 with u = (out + 0.055)/1.055).  out >= encode(1) - which is 0.99999994, not 1, in fp32:
// 1.055 - 0.055 rounds down, in the reference too - is read as "the sum was clamped" here; the caller recomputes the sum
// for exactly those texels (at_boundary), because a sum of exactly 1 (torch.clamp's gate is inclusive) and the one
// or two fp32 sums just below it encode to the same number.
template <class V>
PBR_HD V encode_slope_from_out(V out, bool return_srgb) {
  V slope = splat<V>(1.0f);
  float top = 1.0f;   // what the forward wrote wherever the sum reached 1
  if (return_srgb) {
    V u = out * kInv1_055 + (0.055f * kInv1_055);
    slope = vsel(vle(out, 12.92f * kSrgbEncKnee), 12.92f, (1.055f * 0.416666657f) * pow_pos(u, -1.4f));
    top = srgb_encode<false, float>(1.0f, nullptr);
  }
  return vsel(vge(out, top), 0.0f, slope);
}

template <int kWorkflow, int kLight, class V, int N, class Gout, class IntSink, class Fetch = NoFetch,
          class GeomSink = NoGeomSink, class SavedOut = NoSavedOut, int kUnroll = kBwdUnroll, class View = OrthoView>
PBR_HD void ct_backward_group(const CtStage& S, const CtFlags& F, const V (&araw)[3][N], const V (&nraw)[3][N],
                              const V (&rough)[N], const V (&mraw)[3][N], const V (&x)[N], float y,
                              const LightGeomT<V> (&hoisted)[N], Gout gout, IntSink int_sink, V (&d_albedo)[3][N],
                              V (&d_normal)[3][N], V (&d_rough)[N], V (&d_met)[3][N], Fetch fetch = Fetch(),
                              GeomCache<V> gc = GeomCache<V>(), GeomSink geom_sink = GeomSink(),
                              SavedOut saved_out = SavedOut(), bool want_int = true, const View& view = View()) {
  constexpr bool kGeom = GeomSink::kOn;
  static_assert(!kGeom || kLight == kLightDirectional || kLight == kLightPoint || kLight == kLightPointHoisted ||
                    kLight == kLightPointCached,
                "geometry gradients: directional, per-texel or hoisted point lights, or the 6-field geometry cache");
  V g_view[kGeom ? N : 1][3];
  if (kGeom) {
#pragma unroll
    for (int i = 0; i < N; ++i) g_view[i][0] = g_view[i][1] = g_view[i][2] = splat<V>(0.0f);
  }
  Texel<kWorkflow, V> t[N];
  TexelGrad<V> tg[N];
#pragma unroll
  for (int i = 0; i < N; ++i) {
    const V a3[3] = {araw[0][i], araw[1][i], araw[2][i]};
    const V n3[3] = {nraw[0][i], nraw[1][i], nraw[2][i]};
    const V m3[3] = {mraw[0][i], mraw[1][i], mraw[2][i]};
    texel_setup<kWorkflow, true>(a3, n3, rough[i], m3, F.albedo_is_srgb, F.specular_is_srgb, view_x(S, view, i),
                                 view_y(S, view, i), view_z(S, view, i), t[i]);
    texel_grad_zero(tg[i]);
  }

  const int L = (kLight == kLightPointHoisted) ? 1 : F.L;
  const bool two_pass = (!F.per_light) && L > 1;
  V g_tot[3][N];  // two-pass only: gradient w.r.t. every per-light colour
  fetch(0);
  if (two_pass) {
    // The gate of clamp(sum) and the slope of the encode.  With the forward launch's output at hand both are read off it
    // (single pass) - except where that output does not determine them (at_boundary: the clamp's upper end, the knee of
    // the sRGB curve): those texels - and only those - recompute the summed image like the two-pass path.
    V outv[3][N], slope[3][N];
    bool recompute = true;
    if (saved_out.have()) {
      saved_out(outv);
      recompute = false;
      const float top = F.return_srgb ? srgb_encode<false, float>(1.0f, nullptr) : 1.0f;
#pragma unroll
      for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int i = 0; i < N; ++i) {
          slope[c][i] = encode_slope_from_out(outv[c][i], F.return_srgb);
          recompute = recompute || at_boundary(outv[c][i], top, F.return_srgb);
        }
    }
    if (recompute) {
      // pass 1: the accumulated image, to know where clamp(sum) gates and the slope of the encode
      V acc[3][N];
#pragma unroll
      for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int i = 0; i < N; ++i) acc[c][i] = splat<V>(0.0f);
#pragma unroll kP1Unroll
      for (int l = 0; l < L; ++l) {
#pragma unroll
        for (int i = 0; i < N; ++i) {
          LightGeomT<V> g;
          light_geom<kLight, V, N>(S, l, x, y, hoisted, i, gc, g, view);
          LightFwd<V> f;
          V col[3];
          shade_light_fwd<kWorkflow, false>(t[i], g, S.light[l].inten, f, col);
#pragma unroll
          for (int c = 0; c < 3; ++c) acc[c][i] = xadd(acc[c][i], col[c]);
        }
      }
#pragma unroll
      for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int i = 0; i < N; ++i) {
          const V cl = clamp01(acc[c][i]);
          V sl;
          const V o = encode_out_d(cl, F.return_srgb, &sl);
          if (!saved_out.have()) outv[c][i] = o;
          slope[c][i] = gated(sl, acc[c][i], cl);
        }
    }
    fetch(L);   // rotate: the buffer requested before pass 1 becomes current
    gout(0, outv, g_tot);
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
      for (int i = 0; i < N; ++i) g_tot[c][i] *= slope[c][i];
  }

#pragma unroll kUnroll
  for (int l = 0; l < L; ++l) {
    if (!two_pass) fetch(l + 1);   // light l becomes current, light l + 1 is requested
    LightGeomT<V> g[N];
    LightFwd<V> f[N];
    V outv[3][N], slope[3][N], gl[3][N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
      light_geom<kLight, V, N>(S, l, x, y, hoisted, i, gc, g[i], view);
      V col[3];
      shade_light_fwd<kWorkflow>(t[i], g[i], S.light[l].inten, f[i], col);
      if (!two_pass) {
#pragma unroll
        for (int c = 0; c < 3; ++c) outv[c][i] = encode_out_d(col[c], F.return_srgb, &slope[c][i]);
      }
    }
    if (!two_pass) {
      gout(l, outv, gl);
#pragma unroll
      for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int i = 0; i < N; ++i) gl[c][i] *= slope[c][i];
    }
    float gi_sum[3] = {0.0f, 0.0f, 0.0f};
    float glt_sum[3] = {0.0f, 0.0f, 0.0f};
#pragma unroll
    for (int i = 0; i < N; ++i) {
      const V gcol[3] = {two_pass ? g_tot[0][i] : gl[0][i], two_pass ? g_tot[1][i] : gl[1][i],
                         two_pass ? g_tot[2][i] : gl[2][i]};
      V gi[3];
      GeomGrad<V> gg;
      shade_light_bwd<kWorkflow, kGeom>(t[i], g[i], S.light[l].inten, f[i], gcol, tg[i], gi, &gg);
      if (want_int) {   // (uniform over the launch: the intensity gradient's arithmetic is skipped when nobody asked for it)
#pragma unroll
        for (int c = 0; c < 3; ++c) gi_sum[c] += lane_sum(gi[c]);
      }
      if (kGeom) {
        V glt[3];
        light_geom_bwd<kLight != kLightDirectional>(g[i], gg, S.light[l].p, x[i], y, view_x(S, view, i), view_y(S, view, i),
                                                    view_z(S, view, i), glt, g_view[i]);
#pragma unroll
        for (int c = 0; c < 3; ++c) glt_sum[c] += lane_sum(glt[c]);
      }
    }
    if (want_int) int_sink(l, gi_sum);
    if (kGeom) geom_sink.light(l, glt_sum);
  }
  fetch(-1);   // the light loop is over and its registers are free: the caller may start loading whatever comes next

#pragma unroll
  for (int i = 0; i < N; ++i) {
    V da[3], dn[3], dm[3], dr, g_ndv;
    texel_finish_grad<kWorkflow>(t[i], tg[i], rough[i], view_x(S, view, i), view_y(S, view, i), view_z(S, view, i), da, dn,
                                 &dr, dm, kGeom ? &g_ndv : nullptr);
    if (kGeom) {
      g_view[i][0] += g_ndv * t[i].nx; g_view[i][1] += g_ndv * t[i].ny; g_view[i][2] += g_ndv * t[i].nz;
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      d_albedo[c][i] = da[c];
      d_normal[c][i] = dn[c];
      d_met[c][i] = dm[c];
    }
    d_rough[i] = dr;
  }
  if (kGeom) {
    float gv[3] = {0.0f, 0.0f, 0.0f};
#pragma unroll
    for (int i = 0; i < N; ++i) {
      view_bwd(view, i, g_view[i]);
#pragma unroll
      for (int c = 0; c < 3; ++c) gv[c] += lane_sum(g_view[i][c]);
    }
    geom_sink.view(gv);
  }
}

}  // namespace pbr
