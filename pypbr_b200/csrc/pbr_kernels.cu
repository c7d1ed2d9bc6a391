// pbr_kernels.cu — sm_100a kernels and the C ABI of libpbrcuda.so (include/pbrcuda.h).
//
// Thread mapping shared by every kernel: one thread owns kTexels consecutive texels of one row
// (128-bit LDG/STG per plane when the layout allows it), a CTA covers blockDim.y rows x
// blockDim.x*kTexels columns, blockIdx.z is the material of the batch.  All maps are channel-planar,
// so every warp-level load is a run of 512 contiguous bytes of one plane.
//
// The view / light parameters are staged once per CTA in shared memory by the prologue
// (normalised view vector, per-light position + intensity, and for directional lights the complete,
// image-constant light geometry), then broadcast-read inside the light loop.
#include <cuda_runtime.h>

#include <atomic>
#include <climits>
#include <cstdlib>

#include "../../include/pbrcuda.h"
#include "pbr_shade.cuh"

// Build-time split (__graft_entry__.build_cuda): the Cook-Torrance kernels are instantiated per workflow (WF = 0 metallic,
// 1 specular, 2 metallic with a 3-channel map), a third of the compile time each.  -DPBR_PART=k compiles only the
// instantiations of workflow k and their launcher (pbr::launch_wf<k>); part 0 also holds the streaming kernels, the
// dispatch and the C ABI.  Without PBR_PART everything lands in one translation unit (same code, three times the wait).
#ifndef PBR_PART
#define PBR_PART (-1)
#endif
#define PBR_MAIN_PART (PBR_PART <= 0)
#define PBR_HAS_WF(k) (PBR_PART < 0 || PBR_PART == (k))

namespace pbr {

#ifndef PBR_THREADS
#define PBR_THREADS 256
#endif
#ifndef PBR_FWD_MIN_CTAS
#define PBR_FWD_MIN_CTAS 4   // __launch_bounds__ minBlocksPerSM hints (register caps), tuned on the GPU (profiles/)
#endif
#ifndef PBR_BWD_MIN_CTAS
#define PBR_BWD_MIN_CTAS 3
#endif
#ifndef PBR_HOIST_MATS
#define PBR_HOIST_MATS 16    // materials a thread walks over when the light geometry is hoisted
#endif
#ifndef PBR_TEXELS
#define PBR_TEXELS 4         // texels per thread: 4 (float4 per plane), 2 (float2) or 1 (scalar, coalesced per warp)
#endif
constexpr int kTexels = PBR_TEXELS;     // texels per thread
constexpr int kThreads = PBR_THREADS;   // threads per CTA of the streaming kernels (conversions, blend, colour, normals)
#ifndef PBR_CT_THREADS
#define PBR_CT_THREADS 128   // threads per CTA of the generic Cook-Torrance kernels (168 registers x 3 CTAs per SM in the backward)
#endif
constexpr int kCtThreads = PBR_CT_THREADS;

static std::atomic<uint64_t> g_launches{0};

// ------------------------------------------------------------------------------------------------
// row-segment load / store (streaming: every byte is touched once -> evict-first cache hints)
// ------------------------------------------------------------------------------------------------
template <int N>
__device__ __forceinline__ void load_seg(const float* __restrict__ p, bool vec, int valid, float (&dst)[N]) {
  if (N == 4 && vec) {
    float4 v = __ldcs(reinterpret_cast<const float4*>(p));
    dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; dst[3] = v.w;
  } else if (N == 2 && vec) {
    float2 v = __ldcs(reinterpret_cast<const float2*>(p));
    dst[0] = v.x; dst[1] = v.y;
  } else {
#pragma unroll
    for (int i = 0; i < N; ++i) dst[i] = __ldcs(p + (i < valid ? i : (valid > 0 ? valid - 1 : 0)));  // N == 1 lands here
  }
}

template <int N>
__device__ __forceinline__ void store_seg(float* __restrict__ p, bool vec, int valid, const float (&src)[N]) {
  if (N == 4 && vec) {
    __stcs(reinterpret_cast<float4*>(p), make_float4(src[0], src[1], src[2], src[3]));
  } else if (N == 2 && vec) {
    __stcs(reinterpret_cast<float2*>(p), make_float2(src[0], src[1]));
  } else {
#pragma unroll
    for (int i = 0; i < N; ++i)
      if (i < valid) __stcs(p + i, src[i]);
  }
}

__device__ __forceinline__ int64_t plane_off(const PbrPlane& pl, int b, int c, int row, int col) {
  return (int64_t)b * pl.sb + (int64_t)c * pl.sc + (int64_t)row * pl.sh + col;
}

// position of this thread's texel group; out-of-range threads are clamped onto the last valid group
// (so warp-wide reductions stay convergent) and flagged inactive.
struct Where {
  int b, row, col0, valid;
  bool active, vec;
};
template <int N>
__device__ __forceinline__ Where locate_n(int H, int W, bool vec_ok) {
  Where w;
  w.b = blockIdx.z;
  int row = blockIdx.y * blockDim.y + threadIdx.y;
  int col0 = (blockIdx.x * blockDim.x + threadIdx.x) * N;
  w.active = row < H && col0 < W;
  w.row = row < H ? row : H - 1;
  w.col0 = col0 < W ? col0 : ((W - 1) / N) * N;
  int rem = W - w.col0;
  w.valid = rem < N ? rem : N;
  w.vec = vec_ok && w.valid == N;
  return w;
}
__device__ __forceinline__ Where locate(int H, int W, bool vec_ok) { return locate_n<kTexels>(H, W, vec_ok); }

// ------------------------------------------------------------------------------------------------
// Cook-Torrance kernels
// ------------------------------------------------------------------------------------------------
// A thread of the generic kernels owns kCtTexels consecutive texels of one row, shaded as kSlots = kCtTexels/2
// packed pairs (V = f2: FFMA2/FMUL2/FADD2).  One pair per thread keeps the adjoint's working set in registers.
#ifndef PBR_CT_TEXELS
#define PBR_CT_TEXELS 2
#endif
constexpr int kCtTexels = PBR_CT_TEXELS;
// -DPBR_SCALAR_LANES builds the one-texel-per-lane flavour (V = float) for A/B accuracy and speed checks.
#if defined(PBR_SCALAR_LANES)
typedef float V;
#else
typedef f2 V;
#endif
constexpr int kLanes = Lanes<V>::n;
static_assert(kCtTexels % kLanes == 0, "texels per thread must be a multiple of the lane count");
constexpr int kSlots = kCtTexels / kLanes;
#ifndef PBR_FWD_GROUP
#define PBR_FWD_GROUP 1   // pairs shaded together (ILP) by the generic forward kernel
#endif
#ifndef PBR_BWD_GROUP
#define PBR_BWD_GROUP 1   // ... by the generic backward kernel (register pressure)
#endif

// torch.optim.Adam (single-tensor path): m = lerp(m, g, 1-b1); v = v*b2 + (1-b2)*g*g;
// p -= (lr / (1-b1^t)) * m / (sqrt(v)/sqrt(1-b2^t) + eps).  Shared by adam_kernel and the fused fit epilogue.
struct AdamCoef {
  float step_size, one_minus_beta1, beta2, one_minus_beta2, bias2_sqrt, eps;
};
__device__ __forceinline__ float adam_update(float p, float g, float& m, float& v, const AdamCoef& d) {
  m = m + (g - m) * d.one_minus_beta1;
  v = v * d.beta2 + d.one_minus_beta2 * g * g;
  const float denom = xdiv(xsqrt(v), d.bias2_sqrt) + d.eps;
  return p - d.step_size * xdiv(m, denom);
}

// The same update for the epilogue of the fused fit step, on lane-values (packed FP32) and with the MUFU reciprocal /
// reciprocal square root (relative error ~2e-7 on a step that is lr-sized): the IEEE division and square root of
// adam_update cost ~50 instructions per element, a quarter of the whole fit kernel at 8 lights.
template <class VV>
__device__ __forceinline__ VV adam_update_fast(VV p, VV g, VV& m, VV& v, const AdamCoef& d, float inv_bias2_sqrt) {
  m = m + (g - m) * d.one_minus_beta1;
  v = v * d.beta2 + (g * g) * d.one_minus_beta2;
  const VV sv = v * seed_rsqrt(vmax(v, 1e-36f));   // sqrt(v); 0 for v == 0
  const VV denom = sv * inv_bias2_sqrt + d.eps;
  return p - (m * d.step_size) * fast_rcp(denom);
}

struct CtKParams {
  int B, H, W;
  int mats_per_cta;      // materials a thread walks over (blockIdx.z selects the chunk)
  CtFlags flags;
  int vec_ok;
  int vec_fast;          // host: the kVec = true flavour of the generic kernels applies (see locate_ct)
  int is_loss;           // backward: grad_out is derived from (render - target)
  int force_generic;     // PbrCtDesc.force_generic
  PbrPlane albedo, normal, roughness, metspec, out;
  int64_t out_sl;
  // backward: `gsrc` is grad_out, or the target image when is_loss
  PbrPlane gsrc;
  int64_t gsrc_sl;
  PbrPlane fout;         // backward, accumulate mode, L > 1: the forward launch's output (optional: single-pass backward)
  PbrPlane d_albedo, d_normal, d_roughness, d_metspec;
  float* d_intensity;
  float* d_lights;       // L*3: d/d light position (point) or raw direction (directional); geometry-gradient kernels
  float* d_view;         // 3:   d/d raw view direction
  float loss_scale;
  float* loss_sum;
  // fused fit step (pbr_ct_fit_step): the epilogue applies Adam + projection to the maps in place instead of
  // writing the gradients.  Moments in the order albedo, normal, roughness, metspec.
  int adam_on, adam_project;
  int adam_smem_off;     // byte offset of the Adam staging area in the dynamic shared memory (after the geometry cache)
  int part_on;           // shared-parameter gradients are accumulated in per-thread shared-memory slots (see ct_backward_kernel)
  int part_smem_off;     // ... at this byte offset of the dynamic shared memory
  AdamCoef adam;
  PbrPlane adam_m[4], adam_v[4];
  // staging sources
  Linspace lsx, lsy;
  const float* view_dev;    // non-null: parameters live in device memory
  const float* lights_dev;
  const float* inten_dev;
  float view[3];
  float lights[PBR_MAX_LIGHTS * 3];
  float inten[PBR_MAX_LIGHTS * 3];
};

__device__ __forceinline__ void stage_params(const CtKParams& p, CtStage& S) {
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  const int nth = blockDim.x * blockDim.y;
  const float* view = p.view_dev ? p.view_dev : p.view;
  const float* lights = p.lights_dev ? p.lights_dev : p.lights;
  const float* inten = p.inten_dev ? p.inten_dev : p.inten;
  if (tid < p.flags.L || tid == 0) {
    float vx, vy, vz;
    stage_view(view, vx, vy, vz);
    if (tid == 0) {
      S.vx = vx; S.vy = vy; S.vz = vz;
      S.lsx = p.lsx; S.lsy = p.lsy;
    }
    for (int l = tid; l < p.flags.L; l += nth) stage_light(l, lights, inten, p.flags.point, vx, vy, vz, S.light[l]);
  }
  __syncthreads();
}

// Generic Cook-Torrance kernels come in two flavours (template parameter kVec):
//   kVec = true : the fast flavour.  The host has checked that every plane is 8-byte aligned with even strides, that W is a
//                 multiple of the texels per thread (no thread has a ragged segment) and that every in-plane offset fits
//                 32 bits.  Loads / stores / cp.async are 64-bit with no fallback code in the instruction stream, and an
//                 address is a uniform 64-bit base (plane pointer + batch and channel strides: the same for the whole
//                 CTA) plus ONE 32-bit per-thread offset - the predicated-off scalar copies and the 64-bit per-thread
//                 address arithmetic were a fifth of the fused fit kernel's instructions (profiles/r1_ncu_summary.md).
//   kVec = false: any alignment, ragged widths, planes beyond 2^31 elements: element accesses, 64-bit offsets; only the
//                 uncached light modes are instantiated for it (light_mode()).
template <bool kVec>
__device__ __forceinline__ Where locate_ct(const CtKParams& p) {
  Where w = locate_n<kCtTexels>(p.H, p.W, p.vec_ok != 0);
  if (kVec) {
    w.vec = true;
    w.valid = kCtTexels;
  } else {
    w.vec = p.vec_ok != 0 && (p.W % kCtTexels) == 0;
  }
  return w;
}

template <bool kVec> struct OffT { typedef int64_t type; };
template <> struct OffT<true> { typedef int type; };
// element (b, c, w.row, w.col0 + dcol) of a plane: uniform base + per-thread offset
template <bool kVec>
__device__ __forceinline__ float* at(const PbrPlane& pl, int b, int c, const Where& w, int dcol = 0) {
  typedef typename OffT<kVec>::type T;
  float* base = pl.ptr + ((int64_t)b * pl.sb + (int64_t)c * pl.sc);
  return base + ((T)w.row * (T)pl.sh + (T)(w.col0 + dcol));
}

template <int WF, bool kVec>
__device__ __forceinline__ void load_material(const CtKParams& p, const Where& w, int b, float (&araw)[3][kCtTexels],
                                              float (&nraw)[3][kCtTexels], float (&rough)[kCtTexels],
                                              float (&mraw)[3][kCtTexels], bool has_normal) {
#pragma unroll
  for (int c = 0; c < 3; ++c) load_seg<kCtTexels>(at<kVec>(p.albedo, b, c, w), w.vec, w.valid, araw[c]);
  if (has_normal) {
#pragma unroll
    for (int c = 0; c < 3; ++c) load_seg<kCtTexels>(at<kVec>(p.normal, b, c, w), w.vec, w.valid, nraw[c]);
  } else {
#pragma unroll
    for (int i = 0; i < kCtTexels; ++i) { nraw[0][i] = 0.0f; nraw[1][i] = 0.0f; nraw[2][i] = 1.0f; }
  }
  load_seg<kCtTexels>(at<kVec>(p.roughness, b, 0, w), w.vec, w.valid, rough);
  constexpr int mc = WF == 0 ? 1 : 3;  // WF: 0 metallic (1 ch), 1 specular, 2 metallic (3 ch)
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    if (c < mc) {
      load_seg<kCtTexels>(at<kVec>(p.metspec, b, c, w), w.vec, w.valid, mraw[c]);
    } else {
#pragma unroll
      for (int i = 0; i < kCtTexels; ++i) mraw[c][i] = 0.0f;
    }
  }
}

// The maps of the NEXT material of the walk are pulled into L2 while the current one is shaded (one request per 128-byte
// line: a warp's row segment of a plane is 256 bytes), so the loads at the top of the next iteration hit L2 instead of
// waiting for HBM.  No registers, no shared memory (the multi-light kernels have neither to spare).
#ifndef PBR_BWD_LATE_PREFETCH
#define PBR_BWD_LATE_PREFETCH 0   // measured: +1.6 % on C3, -3 % on the C5 fit kernel (same instantiation, per-light mode) -> off
#endif
constexpr bool kBwdLatePrefetch = PBR_BWD_LATE_PREFETCH != 0;
#ifndef PBR_FWD_REG_PREFETCH
#define PBR_FWD_REG_PREFETCH 1
#endif
constexpr bool kFwdRegPrefetch = PBR_FWD_REG_PREFETCH != 0;
#ifndef PBR_PREFETCH_NEXT
#define PBR_PREFETCH_NEXT 1
#endif
__device__ __forceinline__ void prefetch_l2(const float* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

template <int WF, bool kVec>
__device__ __forceinline__ void prefetch_material(const CtKParams& p, const Where& w, int b, bool has_normal) {
  if (!PBR_PREFETCH_NEXT || ((threadIdx.x * kCtTexels) & 31) != 0) return;   // first thread of every 128-byte line
#pragma unroll
  for (int c = 0; c < 3; ++c) prefetch_l2(at<kVec>(p.albedo, b, c, w));
  if (has_normal) {
#pragma unroll
    for (int c = 0; c < 3; ++c) prefetch_l2(at<kVec>(p.normal, b, c, w));
  }
  prefetch_l2(at<kVec>(p.roughness, b, 0, w));
#pragma unroll
  for (int c = 0; c < (WF == 0 ? 1 : 3); ++c) prefetch_l2(at<kVec>(p.metspec, b, c, w));
}

// texels [kLanes*s0, kLanes*(s0+G)) of a thread's row segment as G lane-values
template <int G, int N>
__device__ __forceinline__ void pairs_of(const float (&src)[N], int s0, V (&dst)[G]) {
#pragma unroll
  for (int i = 0; i < G; ++i)
#pragma unroll
    for (int k = 0; k < kLanes; ++k) lane_set(dst[i], k, src[kLanes * (s0 + i) + k]);
}
template <int G, int N>
__device__ __forceinline__ void pairs_of3(const float (&src)[3][N], int s0, V (&dst)[3][G]) {
#pragma unroll
  for (int c = 0; c < 3; ++c) pairs_of<G, N>(src[c], s0, dst[c]);
}
template <int G, int N>
__device__ __forceinline__ void unpair_to(const V (&src)[G], int s0, float (&dst)[N]) {
#pragma unroll
  for (int i = 0; i < G; ++i)
#pragma unroll
    for (int k = 0; k < kLanes; ++k) dst[kLanes * (s0 + i) + k] = lane_get(src[i], k);
}

// dynamic shared memory of the kLightPointCached* kernels: the geometry cache, L * geom_fields * kSlots * kCtThreads V's
extern __shared__ __align__(16) unsigned char s_dyn[];

template <int kLight>
__device__ __forceinline__ void grid_coords(const CtStage& S, const Where& w, int L, V (&x)[kSlots], float& y,
                                            LightGeomT<V> (&hg)[kSlots], GeomCache<V>& gc) {
  gc.base = reinterpret_cast<V*>(s_dyn) + (threadIdx.y * blockDim.x + threadIdx.x);
  gc.stride = kCtThreads;
  gc.fstride = kSlots * kCtThreads;
  (void)L;
#pragma unroll
  for (int i = 0; i < kSlots; ++i)
#pragma unroll
    for (int k = 0; k < kLanes; ++k) {
      const int col = w.col0 + kLanes * i + k;
      lane_set(x[i], k, linspace_at(S.lsx, col < S.lsx.n ? col : S.lsx.n - 1));
    }
  y = linspace_at(S.lsy, w.row);
  if (kLight == kLightPointHoisted) {
#pragma unroll
    for (int i = 0; i < kSlots; ++i)
      point_light_geom(S.light[0].p[0], S.light[0].p[1], S.light[0].p[2], x[i], y, S.vx, S.vy, S.vz, hg[i]);
  }
  if (is_cached(kLight)) {
    // every light's geometry once per texel pair, reused by all the materials this thread walks over
    for (int l = 0; l < L; ++l) {
#pragma unroll
      for (int i = 0; i < kSlots; ++i) {
        LightGeomT<V> g;
        point_light_geom(S.light[l].p[0], S.light[l].p[1], S.light[l].p[2], x[i], y, S.vx, S.vy, S.vz, g);
        geom_cache_store<geom_fields(kLight), V>(gc, l, i, g);
      }
    }
  }
}

// Register budget of the generic forward: the cached multi-light flavours take the full budget (2 CTAs per SM): registers buy
// them more than occupancy does (tools/tune.py, 16 x 1024^2: L = 16 0.810 -> 0.771 ms, L = 8 0.403 -> 0.390, L = 4 0.227 -> 0.222;
// unrolling the light loop on top of it is slower again), the memory-bound single-light / uncached flavours keep 4 CTAs.
#ifndef PBR_FWD_CACHED_MIN_CTAS
#define PBR_FWD_CACHED_MIN_CTAS 2
#endif
constexpr int fwd_min_ctas(int light_mode) { return is_cached(light_mode) ? PBR_FWD_CACHED_MIN_CTAS : PBR_FWD_MIN_CTAS; }

// Plain-case flavours of the generic kernels (template parameter kFM, round 2): like kFast of the streamed kernels, the host picks
// them when the launch is what the reference's defaults produce - sRGB albedo and output, a normal map, 64-bit accesses - and
//   kFmAccum: lights accumulated into one image (forward; backward from the saved forward output, map gradients only).
// The switches that are warp-uniform at run time in the general flavour are constants here, so the light loop carries no
// flag tests (8 BRA + UISETP + LDCU triples per texel-pair-light in the general code) and is one basic block to schedule:
// static size of the backward's light loop 410 -> 190 instructions (executed: 259 -> 190), forward 147 -> 86.
// Measured on C3 (16 x 2048^2, 16 lights): forward 3.07 -> 2.85 ms, backward 7.67 -> 6.17 ms, step 10.74 -> 9.02 ms.
// (The same treatment of the fused fit step - per-light targets, loss, Adam epilogue as constants - was built and measured:
// 286 instead of ~300 instructions per texel-pair-light, 255 registers with a small spill, C5 12.347 -> 12.317 ms.  That
// kernel waits on the per-light encode / slope chains (MUFU) at 8 warps per SM, not on instruction issue: not kept.)

enum { kFmGeneric = 0, kFmAccum = 1 };
#ifndef PBR_GENERIC_FAST
#define PBR_GENERIC_FAST 1
#endif
constexpr bool kGenericFast = PBR_GENERIC_FAST != 0;
#ifndef PBR_PLAIN_UNROLL
#define PBR_PLAIN_UNROLL 2   // light-loop unrolling of the plain-case flavours
#endif
constexpr int kPlainUnroll = PBR_PLAIN_UNROLL;
template <int kFM>
__device__ __forceinline__ CtFlags plain_flags(const CtFlags& f) {
  CtFlags F = f;
  if (kFM != kFmGeneric) {
    F.albedo_is_srgb = true; F.specular_is_srgb = true; F.return_srgb = true;
    F.per_light = false;
    if (kFM == kFmAccum && F.L < 2) F.L = 2;   // (never taken: the host only picks kFmAccum for L > 1; tells the compiler so)
  }
  return F;
}

template <int WF, int kLight, bool kVec = true, int kFM = kFmGeneric>
__global__ void __launch_bounds__(kCtThreads, fwd_min_ctas(kLight)) ct_forward_kernel(const __grid_constant__ CtKParams p) {
  constexpr int G = PBR_FWD_GROUP;
  __shared__ CtStage S;
  stage_params(p, S);
  const Where w = locate_ct<kVec>(p);
  if (!w.active) return;
  const CtFlags F = plain_flags<kFM>(p.flags);
  const bool has_normal = kFM != kFmGeneric || p.normal.ptr != nullptr;

  V x[kSlots];
  float y;
  LightGeomT<V> hg[kSlots];
  GeomCache<V> gc;
  grid_coords<kLight>(S, w, p.flags.L, x, y, hg, gc);

  const int b0 = blockIdx.z * p.mats_per_cta;
  const int b1 = min(b0 + p.mats_per_cta, p.B);
  // The forward has registers to spare (96 of the 128 its occupancy allows), so the maps of the next material of the walk
  // are loaded into a second register set while the current one is shaded (the backward, at 235 registers, prefetches
  // into L2 instead).
  float nx_a[3][kCtTexels], nx_n[3][kCtTexels], nx_r[kCtTexels], nx_m[3][kCtTexels];
  if (kFwdRegPrefetch) load_material<WF, kVec>(p, w, b0, nx_a, nx_n, nx_r, nx_m, has_normal);
  for (int b = b0; b < b1; ++b) {
    float araw[3][kCtTexels], nraw[3][kCtTexels], rough[kCtTexels], mraw[3][kCtTexels];
    if (kFwdRegPrefetch) {
#pragma unroll
      for (int i = 0; i < kCtTexels; ++i) {
#pragma unroll
        for (int c = 0; c < 3; ++c) { araw[c][i] = nx_a[c][i]; nraw[c][i] = nx_n[c][i]; mraw[c][i] = nx_m[c][i]; }
        rough[i] = nx_r[i];
      }
      if (b + 1 < b1) load_material<WF, kVec>(p, w, b + 1, nx_a, nx_n, nx_r, nx_m, has_normal);
    } else {
      load_material<WF, kVec>(p, w, b, araw, nraw, rough, mraw, has_normal);
      if (b + 1 < b1) prefetch_material<WF, kVec>(p, w, b + 1, has_normal);
    }
    float outv[3][kCtTexels];
#pragma unroll
    for (int s = 0; s < kSlots; s += G) {
      V a[3][G], n[3][G], r[G], m[3][G], xs[G];
      LightGeomT<V> hgs[G];
      pairs_of3<G>(araw, s, a); pairs_of3<G>(nraw, s, n); pairs_of3<G>(mraw, s, m); pairs_of<G>(rough, s, r);
#pragma unroll
      for (int i = 0; i < G; ++i) { xs[i] = x[s + i]; hgs[i] = hg[s + i]; }
      auto emit = [&](int l, const V(&v)[3][G]) {
        if (F.per_light) {
          // one image per light: store this sub-group directly (64/128-bit when the group allows)
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            float tv[kLanes * G];
            unpair_to<G>(v[c], 0, tv);
            int vs = w.valid - kLanes * s;
            store_seg<kLanes * G>(at<kVec>(p.out, b, c, w, kLanes * s) + (int64_t)l * p.out_sl,
                                  w.vec, vs < 0 ? 0 : vs, tv);
          }
        } else {
#pragma unroll
          for (int c = 0; c < 3; ++c) unpair_to<G>(v[c], s, outv[c]);
        }
      };
      GeomCache<V> gcs = gc;   // lane-value i of the group is lane-value s + i of the thread
      gcs.base += s * gc.stride;
      // plain-case flavour: the light loop is one basic block, two lights interleave (L = 16: 0.717 -> 0.696 ms per 16 x 1024^2)
      ct_forward_group<WF, kLight, V, G, decltype(emit), (kFM != kFmGeneric ? kPlainUnroll : kFwdUnroll)>(S, F, a, n, r, m, xs, y, hgs, emit, gcs);
    }
    if (!F.per_light) {
#pragma unroll
      for (int c = 0; c < 3; ++c)
        store_seg<kCtTexels>(at<kVec>(p.out, b, c, w), w.vec, w.valid, outv[c]);
    }
  }
}

#ifndef PBR_COLD_UNROLL
#define PBR_COLD_UNROLL 4   // measured: branching over the cold path (1) is not faster than predicating it
#endif
#ifndef PBR_PACKED_LOSS
#define PBR_PACKED_LOSS 1
#endif
constexpr int kColdUnroll = PBR_COLD_UNROLL;
constexpr bool kPackedLoss = PBR_PACKED_LOSS != 0;

// per-thread asynchronous copies global -> shared (LDGSTS) for the backward kernel's grad_out / target ring
constexpr int kRing = 4;
__device__ __forceinline__ void cp_async8(float* dst_smem, const float* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async4(float* dst_smem, const float* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Backward / fused loss.  Runtime (warp-uniform) switches:
//   p.is_loss     : gsrc is the target image; grad_out = 2*loss_scale*(render - target) and the squared
//                   error is reduced warp-shuffle -> shared -> ONE atomic per CTA.
//   p.d_intensity : per-light intensity gradients, reduced the same way.
// CTAs per SM the backward's register budget is sized for.  With the 6-field cache the shared memory already caps
// the SM at 2-3 CTAs and the light loop is long: the full 255-register budget (no spills) beats a third CTA
// (tools/tune.py, L = 8: 3.29 vs 3.80 ms; L = 16: 2.53 vs 2.99 ms).
#ifndef PBR_BWD_CACHED_MIN_CTAS
#define PBR_BWD_CACHED_MIN_CTAS 2
#endif
constexpr int bwd_min_ctas(int light_mode) {
  return (light_mode == kLightPointCached || light_mode == kLightPointCachedAllBig) ? PBR_BWD_CACHED_MIN_CTAS : PBR_BWD_MIN_CTAS;
}
// Light-loop unrolling of the general backward: by two where the full register budget is available (per-light loss kernel,
// 32 x 1024^2: L = 8 2.654 -> 2.571 ms, L = 16 2.470 -> 2.393 ms; the 168-register flavours spill over it: L = 4 1.624 -> 1.794 ms).
#ifndef PBR_BWD_BIG_UNROLL
#define PBR_BWD_BIG_UNROLL 2
#endif
PBR_HDC int bwd_unroll(int light_mode) {
  return (light_mode == kLightPointCached || light_mode == kLightPointCachedAllBig) ? PBR_BWD_BIG_UNROLL : kBwdUnroll;
}

// The saved forward output of the row segment being back-propagated (PbrCtGrads.fwd_out).  It travels through slot 1 of
// the thread's cp.async ring (accumulate mode keeps only slot 0 busy, with grad_out), requested together with grad_out
// before the per-texel setup, so its latency is hidden like grad_out's.
struct CtaSavedOut {
  const float* slot1;   // this thread's column of ring slot 1: [channel][thread][NT]
  bool on;
  __device__ __forceinline__ bool have() const { return on; }
  template <int G>
  __device__ __forceinline__ void operator()(V (&o)[3][G]) const {
    cp_async_wait<0>();
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float tv[kLanes * G];
#pragma unroll
      for (int i = 0; i < kLanes * G; ++i) tv[i] = slot1[c * (kCtThreads * kLanes * G) + i];
      pairs_of<G>(tv, 0, o[c]);
    }
  }
};

// Sink of the geometry gradients (kGeom kernels).  Per light: into the calling thread's own shared-memory slots (`part`, see
// ct_backward_kernel) when the launch has them, else warp shuffle -> shared atomics; the view gradient (once per material and
// texel pair) always takes the shuffle.  Flushed once per CTA.
struct CtaGeomSink {
  static constexpr bool kOn = true;
  float* s_geo;   // [L][3] lights, then [3] view
  int L, tid;
  float live;
  float* part;    // this thread's column of the partial-sum slots, or nullptr
  __device__ __forceinline__ void add(int slot, const float (&g)[3]) const {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float sum = warp_sum(g[c] * live);
      if ((tid & 31) == 0) atomicAdd(&s_geo[3 * slot + c], sum);
    }
  }
  __device__ __forceinline__ void light(int l, const float (&g)[3]) const {
    if (part) {
#pragma unroll
      for (int c = 0; c < 3; ++c) part[(l * 6 + 3 + c) * kCtThreads] += g[c] * live;
    } else {
      add(l, g);
    }
  }
  __device__ __forceinline__ void view(const float (&g)[3]) const { add(L, g); }
};

// kGeom: also d/d(light position | direction) and d/d(view direction) (PbrCtGrads.d_lights / d_view), which the
// reference delivers through plain autograd (cooktorrance.py:95,125-140).  Uncached per-texel light modes only.
template <int WF, int kLight, bool kGeom = false, bool kVec = true, int kFM = kFmGeneric>
__global__ void __launch_bounds__(kCtThreads, kGeom ? 2 : bwd_min_ctas(kLight)) ct_backward_kernel(const __grid_constant__ CtKParams p) {
  static_assert(kFM == kFmGeneric || (!kGeom && kVec), "plain-case flavours: map gradients, 64-bit accesses");
  constexpr int G = PBR_BWD_GROUP;
  __shared__ CtStage S;
  __shared__ float s_int[PBR_MAX_LIGHTS * 3];
  __shared__ float s_geo[kGeom ? (PBR_MAX_LIGHTS + 1) * 3 : 1];
  __shared__ float s_loss[kCtThreads / 32];
  __shared__ __align__(16) float s_ring[kRing * 3 * kCtThreads * kLanes * PBR_BWD_GROUP];
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  const CtFlags F = plain_flags<kFM>(p.flags);
  const bool int_grad = kFM != kFmGeneric ? false : p.d_intensity != nullptr;
  const bool is_loss = kFM != kFmGeneric ? false : p.is_loss != 0;
  const bool adam_on = kFM != kFmGeneric ? false : p.adam_on != 0;
  const bool has_normal = kFM != kFmGeneric || p.normal.ptr != nullptr;
  const bool part_on = kFM != kFmGeneric ? false : p.part_on != 0;
  if (int_grad) {
    for (int i = tid; i < p.flags.L * 3; i += kCtThreads) s_int[i] = 0.0f;
  }
  if (kGeom) {
    for (int i = tid; i < (p.flags.L + 1) * 3; i += kCtThreads) s_geo[i] = 0.0f;
  }
  // Shared-parameter gradients (d_intensity; kGeom: + d_lights) are sums over every texel, light by light.  A warp shuffle
  // reduction + shared atomic per light and value - 30 SHFL per texel-pair-light with kGeom - made the fit with unknown
  // lighting 2.4x slower than the plain loss kernel (24.9 vs 10.4 ms on C5).  Each thread therefore adds into its OWN
  // shared-memory slots, [value][thread] (one LDS + FADD + STS, no synchronisation), over all the lights and all the
  // materials it walks over, and the CTA reduces the slots once at the end.  K values per light: 3 (intensity) or 6 (kGeom).
  constexpr int K = kGeom ? 6 : 3;
  float* const s_part = part_on ? reinterpret_cast<float*>(s_dyn + p.part_smem_off) + tid : nullptr;
  if (s_part) {
    for (int i = 0; i < p.flags.L * K; ++i) s_part[i * kCtThreads] = 0.0f;
  }
  stage_params(p, S);  // ends with __syncthreads()
  const Where w = locate_ct<kVec>(p);
  const float live = w.active ? 1.0f : 0.0f;
  if (!w.active && !int_grad && !is_loss && !kGeom) return;  // nothing to reduce: edge threads may leave

  V x[kSlots];
  float y;
  LightGeomT<V> hg[kSlots];
  GeomCache<V> gc;
  grid_coords<kLight>(S, w, p.flags.L, x, y, hg, gc);
  // Adam staging of the fused fit step: [channel slot][p | m | v][thread][texel], this thread's column
  float* const s_adam = reinterpret_cast<float*>(s_dyn + p.adam_smem_off) + tid * kCtTexels;

  float loss_local = 0.0f;
  V loss_v = splat<V>(0.0f);   // squared error of the vector path, one partial sum per lane
  const int b0 = blockIdx.z * p.mats_per_cta;
  const int b1 = min(b0 + p.mats_per_cta, p.B);
  // The maps of material b + 1 are requested when the light loop of material b is over - its ~70 registers are free by
  // then - and land (from L2, where prefetch_material sent them) while the gradients of b are finished and stored.
  // Only where it was measured to pay: the 255-register flavour in accumulate mode (L = 16: 2.49 -> 2.45 ms per
  // 16 x 1024^2); the 168-register flavours spill over it (L = 4: 0.83 -> 1.02 ms), the per-light loss kernel is neutral.
  const bool late_prefetch = kBwdLatePrefetch && kLight == kLightPointCached && !F.per_light;
  float nx_a[3][kCtTexels], nx_n[3][kCtTexels], nx_r[kCtTexels], nx_m[3][kCtTexels];
  for (int b = b0; b < b1; ++b) {
    float araw[3][kCtTexels], nraw[3][kCtTexels], rough[kCtTexels], mraw[3][kCtTexels];
    if (late_prefetch && b > b0) {
#pragma unroll
      for (int i = 0; i < kCtTexels; ++i) {
#pragma unroll
        for (int c = 0; c < 3; ++c) { araw[c][i] = nx_a[c][i]; nraw[c][i] = nx_n[c][i]; mraw[c][i] = nx_m[c][i]; }
        rough[i] = nx_r[i];
      }
    } else {
      load_material<WF, kVec>(p, w, b, araw, nraw, rough, mraw, has_normal);
    }
    if (b + 1 < b1) prefetch_material<WF, kVec>(p, w, b + 1, has_normal);
    if (adam_on) {
      // Fused fit step: what the Adam epilogue of THIS material needs (parameters and both moments of every channel)
      // starts travelling now, as per-thread cp.async copies into shared memory, and lands while the light loop runs.
      // A dependent load -> update -> store chain per channel in the epilogue would expose 8 DRAM round trips per
      // material (measured: 25.1 instead of 13.3 + 4.6 ms on C5).  The group is older than the target ring's groups,
      // so the ring's first wait also covers it.
      int ch = 0;
      auto send = [&](const PbrPlane& P, int q, int c) {
        const float* src[3] = {at<kVec>(P, b, c, w), at<kVec>(p.adam_m[q], b, c, w),
                               at<kVec>(p.adam_v[q], b, c, w)};
#pragma unroll
        for (int j = 0; j < 3; ++j) {
          float* dst = s_adam + ((3 * ch + j) * kCtThreads) * kCtTexels;
          if (kCtTexels == 2 && (kVec || w.vec)) {
            cp_async8(dst, src[j]);
          } else {
#pragma unroll kColdUnroll   // cold path, branched over
            for (int i = 0; i < kCtTexels; ++i) cp_async4(dst + i, src[j] + (i < w.valid ? i : (w.valid > 0 ? w.valid - 1 : 0)));
          }
        }
        ++ch;
      };
#pragma unroll
      for (int c = 0; c < 3; ++c) send(p.albedo, 0, c);
      if (has_normal) {
#pragma unroll
        for (int c = 0; c < 3; ++c) send(p.normal, 1, c);
      } else {
        ch += 3;
      }
      send(p.roughness, 2, 0);
#pragma unroll
      for (int c = 0; c < (WF == 0 ? 1 : 3); ++c) send(p.metspec, 3, c);
      cp_async_commit();
    }
    float d_albedo[3][kCtTexels], d_normal[3][kCtTexels], d_rough[kCtTexels], d_met[3][kCtTexels];
#pragma unroll
    for (int s = 0; s < kSlots; s += G) {
      V a[3][G], n[3][G], r[G], m[3][G], xs[G];
      LightGeomT<V> hgs[G];
      pairs_of3<G>(araw, s, a); pairs_of3<G>(nraw, s, n); pairs_of3<G>(mraw, s, m); pairs_of<G>(rough, s, r);
#pragma unroll
      for (int i = 0; i < G; ++i) { xs[i] = x[s + i]; hgs[i] = hg[s + i]; }
      const int vs = (w.valid - kLanes * s) < 0 ? 0 : (w.valid - kLanes * s);   // live texels of this sub-group
      // grad_out / target of the light being shaded.  The per-light images are the only global loads inside
      // the light loop; at 12 warps per SM a plain load (even one light ahead in registers) leaves ~1.3 MB in
      // flight chip-wide, i.e. ~1.2 TB/s - the fused fit step then waits for them a quarter of its time
      // (profiles/).  So every thread runs its own cp.async (LDGSTS) ring in shared memory, kRing - 1 lights
      // ahead: no registers, no cross-thread synchronisation (a thread only ever reads what it copied).
      constexpr int NT = kLanes * G;
      float* ring = s_ring + tid * NT;   // [slot][channel][thread][NT]
      const int nl_src = F.per_light ? F.L : 1;
      const float* const gbase = at<kVec>(p.gsrc, b, 0, w, kLanes * s);   // once per material
      const bool have_fout = kFM == kFmAccum ? true : p.fout.ptr != nullptr;   // accumulate mode only (nl_src == 1): slot 1 carries the saved forward output
      const float* const fbase = have_fout ? at<kVec>(p.fout, b, 0, w, kLanes * s) : nullptr;
      auto issue = [&](int l) {
        const bool saved = have_fout && l == 1;
        if (l < nl_src || saved) {
          const float* const gl = saved ? fbase : gbase + (int64_t)l * p.gsrc_sl;
          const int64_t csc = saved ? p.fout.sc : p.gsrc.sc;
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            const float* src = gl + (int64_t)c * csc;
            float* dst = ring + ((l % kRing) * 3 + c) * (kCtThreads * NT);
            if (NT == 2 && (kVec || w.vec)) {
              cp_async8(dst, src);
            } else {
#pragma unroll kColdUnroll   // cold path (ragged or unaligned rows): a real loop is branched over instead of predicated
              for (int i = 0; i < NT; ++i) cp_async4(dst + i, src + (i < vs ? i : (vs > 0 ? vs - 1 : 0)));
            }
          }
        }
        cp_async_commit();   // always: keeps the group count uniform
      };
      auto fetch = [&](int l) {
        if (l < 0) {   // after the light loop
          if (late_prefetch && s + G >= kSlots && b + 1 < b1) load_material<WF, kVec>(p, w, b + 1, nx_a, nx_n, nx_r, nx_m, has_normal);
          return;
        }
        if (l == 0) {
#pragma unroll
          for (int q = 0; q < kRing - 1; ++q) issue(q);
        } else {
          issue(l + kRing - 2);
        }
      };
      float t_cur[3][NT];
      auto take = [&](int l) {   // light l has landed once at most kRing - 1 younger groups are pending
        cp_async_wait<kRing - 1>();
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
          for (int i = 0; i < NT; ++i) t_cur[c][i] = ring[((l % kRing) * 3 + c) * (kCtThreads * NT) + i];
      };
      auto gout = [&](int l, const V(&outv)[3][G], V(&g)[3][G]) {
        take(l);
        if (kPackedLoss && (kVec || w.vec)) {   // every lane is a live texel (uniform over the grid): packed arithmetic, no masks
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            V t[G];
            pairs_of<G>(t_cur[c], 0, t);
#pragma unroll
            for (int i = 0; i < G; ++i) {
              if (is_loss) {
                const V diff = outv[c][i] - t[i];
                loss_v += diff * diff;
                g[c][i] = diff * (2.0f * p.loss_scale);
              } else {
                g[c][i] = t[i];
              }
            }
          }
          return;
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          float ov[kLanes * G], gv[kLanes * G];
          unpair_to<G>(outv[c], 0, ov);
#pragma unroll
          for (int i = 0; i < kLanes * G; ++i) {
            if (is_loss) {
              float diff = (i < vs) ? ov[i] - t_cur[c][i] : 0.0f;
              loss_local += diff * diff;
              gv[i] = 2.0f * p.loss_scale * diff;
            } else {
              gv[i] = (i < vs) ? t_cur[c][i] : 0.0f;
            }
          }
          pairs_of<G>(gv, 0, g[c]);
        }
      };
      auto int_sink = [&](int l, const float(&gi)[3]) {
        if (int_grad) {
          if (s_part) {   // (the same test as CtaGeomSink's: one uniform branch per light for both)
#pragma unroll
            for (int c = 0; c < 3; ++c) s_part[(l * K + c) * kCtThreads] += gi[c] * live;
          } else {
#pragma unroll
            for (int c = 0; c < 3; ++c) {
              float sum = warp_sum(gi[c] * live);
              if ((tid & 31) == 0) atomicAdd(&s_int[3 * l + c], sum);
            }
          }
        }
      };
      V da[3][G], dn[3][G], dr[G], dm[3][G];
      GeomCache<V> gcs = gc;
      gcs.base += s * gc.stride;
      if constexpr (kGeom) {
        ct_backward_group<WF, kLight, V, G>(S, F, a, n, r, m, xs, y, hgs, gout, int_sink, da, dn, dr, dm, fetch, gcs,
                                            CtaGeomSink{s_geo, p.flags.L, tid, live, s_part}, CtaSavedOut{ring + 3 * (kCtThreads * NT), have_fout}, int_grad);
      } else {
        // (plain-case flavour, light loop unrolled by two: L = 16 1.570 -> 1.549 ms, L = 8 0.916 -> 0.886 ms per 16 x 1024^2)
        ct_backward_group<WF, kLight, V, G, decltype(gout), decltype(int_sink), decltype(fetch), NoGeomSink, CtaSavedOut,
                          (kFM != kFmGeneric ? kPlainUnroll : bwd_unroll(kLight))>(S, F, a, n, r, m, xs, y, hgs, gout, int_sink, da, dn, dr, dm, fetch,
                                                                          gcs, NoGeomSink(), CtaSavedOut{ring + 3 * (kCtThreads * NT), have_fout}, int_grad);
      }
#pragma unroll
      for (int c = 0; c < 3; ++c) { unpair_to<G>(da[c], s, d_albedo[c]); unpair_to<G>(dn[c], s, d_normal[c]); unpair_to<G>(dm[c], s, d_met[c]); }
      unpair_to<G>(dr, s, d_rough);
    }
    if (!w.active && adam_on) cp_async_wait<0>();
    if (w.active && adam_on) {
      // fused fit step: the gradients never reach HBM; parameters and moments were prefetched into shared memory
      constexpr int mc = WF == 0 ? 1 : 3;
      const bool proj = p.adam_project != 0;
      cp_async_wait<0>();
      int ch = 0;   // same channel order as the prefetch above
      const float inv_b2 = 1.0f / p.adam.bias2_sqrt;
      auto channel = [&](const PbrPlane&, int q, int c, const float(&g)[kCtTexels], float(&pn)[kCtTexels]) {
        float pv[kCtTexels], m[kCtTexels], v[kCtTexels];
        const float* st = s_adam + (3 * ch * kCtThreads) * kCtTexels;
#pragma unroll
        for (int i = 0; i < kCtTexels; ++i) {
          pv[i] = st[i]; m[i] = st[kCtThreads * kCtTexels + i]; v[i] = st[2 * kCtThreads * kCtTexels + i];
        }
        ++ch;
        V pp[kSlots], gp[kSlots], mp[kSlots], vp[kSlots];
        pairs_of<kSlots>(pv, 0, pp); pairs_of<kSlots>(g, 0, gp); pairs_of<kSlots>(m, 0, mp); pairs_of<kSlots>(v, 0, vp);
#pragma unroll
        for (int i = 0; i < kSlots; ++i) pp[i] = adam_update_fast(pp[i], gp[i], mp[i], vp[i], p.adam, inv_b2);
        unpair_to<kSlots>(pp, 0, pn); unpair_to<kSlots>(mp, 0, m); unpair_to<kSlots>(vp, 0, v);
        store_seg<kCtTexels>(at<kVec>(p.adam_m[q], b, c, w), w.vec, w.valid, m);
        store_seg<kCtTexels>(at<kVec>(p.adam_v[q], b, c, w), w.vec, w.valid, v);
      };
      auto put = [&](const PbrPlane& P, int c, float(&pn)[kCtTexels], bool clamp) {
        if (clamp) {
#pragma unroll
          for (int i = 0; i < kCtTexels; ++i) pn[i] = fminf(fmaxf(pn[i], 0.0f), 1.0f);
        }
        store_seg<kCtTexels>(at<kVec>(P, b, c, w), w.vec, w.valid, pn);
      };
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        float pn[kCtTexels];
        channel(p.albedo, 0, c, d_albedo[c], pn);
        put(p.albedo, c, pn, proj);
      }
      if (!has_normal) ch += 3;
      if (has_normal) {
        float pn[3][kCtTexels];
#pragma unroll
        for (int c = 0; c < 3; ++c) channel(p.normal, 1, c, d_normal[c], pn[c]);
        if (proj) {
#pragma unroll
          for (int i = 0; i < kCtTexels; ++i) {
            float o3[3];
            normalize3(pn[0][i], pn[1][i], pn[2][i], o3);   // F.normalize(dim=channel), eps 1e-12
            pn[0][i] = o3[0]; pn[1][i] = o3[1]; pn[2][i] = o3[2];
          }
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) put(p.normal, c, pn[c], false);
      }
      {
        float pn[kCtTexels];
        channel(p.roughness, 2, 0, d_rough, pn);
        put(p.roughness, 0, pn, proj);
      }
#pragma unroll
      for (int c = 0; c < mc; ++c) {
        float pn[kCtTexels];
        channel(p.metspec, 3, c, d_met[c], pn);
        put(p.metspec, c, pn, proj);
      }
    } else if (w.active) {
      constexpr bool kAll = kFM == kFmAccum;   // every gradient plane was requested
      if (kAll || p.d_albedo.ptr) {
#pragma unroll
        for (int c = 0; c < 3; ++c) store_seg<kCtTexels>(at<kVec>(p.d_albedo, b, c, w), w.vec, w.valid, d_albedo[c]);
      }
      if (kAll || (has_normal && p.d_normal.ptr)) {
#pragma unroll
        for (int c = 0; c < 3; ++c) store_seg<kCtTexels>(at<kVec>(p.d_normal, b, c, w), w.vec, w.valid, d_normal[c]);
      }
      if (kAll || p.d_roughness.ptr) store_seg<kCtTexels>(at<kVec>(p.d_roughness, b, 0, w), w.vec, w.valid, d_rough);
      if (kAll || p.d_metspec.ptr) {
        constexpr int mc = WF == 0 ? 1 : 3;
#pragma unroll
        for (int c = 0; c < mc; ++c) store_seg<kCtTexels>(at<kVec>(p.d_metspec, b, c, w), w.vec, w.valid, d_met[c]);
      }
    }
  }

  if (is_loss) {
    loss_local += lane_sum(loss_v);
    float sum = warp_sum(loss_local * live);
    if ((tid & 31) == 0) s_loss[tid >> 5] = sum;
  }
  if (part_on) {
    // the per-thread slots -> the CTA's sums: warp w reduces values w, w + 4, ... (128 slots each: 4 per lane, then a shuffle)
    __syncthreads();
    const float* base = reinterpret_cast<const float*>(s_dyn + p.part_smem_off);
    const int lane = tid & 31;
    for (int v = tid >> 5; v < p.flags.L * K; v += kCtThreads / 32) {
      float sum = 0.0f;
#pragma unroll
      for (int j = 0; j < kCtThreads / 32; ++j) sum += base[v * kCtThreads + lane + 32 * j];
      sum = warp_sum(sum);
      if (lane == 0) {
        const int l = v / K, j = v - l * K;
        if (j < 3) {
          if (int_grad) s_int[3 * l + j] += sum;          // one writer per value
        } else if (kGeom) {
          s_geo[3 * l + (j - 3)] += sum;
        }
      }
    }
  }
  if (is_loss || int_grad || kGeom) __syncthreads();
  if (kGeom) {
    // one thread per light (and one for the view) turns the CTA's partial sums into gradients of the RAW parameters:
    // the Jacobians of F.normalize(dir) / F.normalize(view) are constant over the image, hence applied here, once
    const float* view = p.view_dev ? p.view_dev : p.view;
    const float* lights = p.lights_dev ? p.lights_dev : p.lights;
    if (tid <= p.flags.L) {
      const float g[3] = {s_geo[3 * tid], s_geo[3 * tid + 1], s_geo[3 * tid + 2]};
      float o[3] = {g[0], g[1], g[2]};
      float* dst = nullptr;
      if (tid == p.flags.L) {
        normalize_bwd(view, g, o);
        dst = p.d_view;
      } else {
        if (!p.flags.point) normalize_bwd(lights + 3 * tid, g, o);
        dst = p.d_lights ? p.d_lights + 3 * tid : nullptr;
      }
      if (dst) {
#pragma unroll
        for (int c = 0; c < 3; ++c) atomicAdd(dst + c, o[c]);
      }
    }
  }
  if (is_loss && tid == 0) {
    float sum = 0.0f;
    const int nw = (blockDim.x * blockDim.y + 31) >> 5;
    for (int i = 0; i < nw; ++i) sum += s_loss[i];
    atomicAdd(p.loss_sum, sum);
  }
  if (int_grad) {
    for (int i = tid; i < p.flags.L * 3; i += kCtThreads) atomicAdd(&p.d_intensity[i], s_int[i]);
  }
}

// ------------------------------------------------------------------------------------------------
// Camera at a finite position (pbr_ct_*_camera): the view vector of a texel is F.normalize(c - P) with c = PbrCtDesc.view
// and P = (x, -y, 0) its plane position, instead of the one CTA-uniform direction of the ct_* kernels.
// The design of the generic kernels: V = f2, kCtThreads threads, a walk over up to kHoistMats materials, element-access
// loads and stores (any alignment and width).  The view vectors - and, for one point light, its geometry - are computed
// once per texel and reused by every material of the walk (they do not depend on the material).  Light modes:
// kLightDirectional (l is image-constant, h and (1 - h.v)^5 per texel), kLightPointHoisted (L == 1) and kLightPoint.
// The backward always computes the geometry adjoints (the camera gradient runs through h, N.V and the Fresnel term).
// ------------------------------------------------------------------------------------------------
template <int kLight>
__device__ __forceinline__ void cam_setup(const CtKParams& p, const CtStage& S, const Where& w, V (&x)[kSlots], float& y,
                                          LaneViews<V, kSlots>& cv, LightGeomT<V> (&hg)[kSlots]) {
  GeomCache<V> gc;
  grid_coords<kLightPoint>(S, w, p.flags.L, x, y, hg, gc);   // the plane coordinates only
  const float* cam = p.view_dev ? p.view_dev : p.view;
  const float c[3] = {cam[0], cam[1], cam[2]};
#pragma unroll
  for (int i = 0; i < kSlots; ++i) {
    camera_view(c, x[i], y, cv.x[i], cv.y[i], cv.z[i], cv.len[i]);
    if (kLight == kLightPointHoisted)
      point_light_geom(S.light[0].p[0], S.light[0].p[1], S.light[0].p[2], x[i], y, cv.x[i], cv.y[i], cv.z[i], hg[i]);
  }
}

template <int WF, int kLight>
__global__ void __launch_bounds__(kCtThreads, PBR_FWD_MIN_CTAS) cam_forward_kernel(const __grid_constant__ CtKParams p) {
  __shared__ CtStage S;
  stage_params(p, S);
  const Where w = locate_ct<false>(p);
  if (!w.active) return;
  const CtFlags& F = p.flags;
  const bool has_normal = p.normal.ptr != nullptr;
  V x[kSlots];
  float y;
  LaneViews<V, kSlots> cv;
  LightGeomT<V> hg[kSlots];
  cam_setup<kLight>(p, S, w, x, y, cv, hg);

  const int b0 = blockIdx.z * p.mats_per_cta;
  const int b1 = min(b0 + p.mats_per_cta, p.B);
  for (int b = b0; b < b1; ++b) {
    float araw[3][kCtTexels], nraw[3][kCtTexels], rough[kCtTexels], mraw[3][kCtTexels];
    load_material<WF, false>(p, w, b, araw, nraw, rough, mraw, has_normal);
    if (b + 1 < b1) prefetch_material<WF, false>(p, w, b + 1, has_normal);
    V a[3][kSlots], n[3][kSlots], r[kSlots], m[3][kSlots];
    pairs_of3<kSlots>(araw, 0, a); pairs_of3<kSlots>(nraw, 0, n); pairs_of3<kSlots>(mraw, 0, m); pairs_of<kSlots>(rough, 0, r);
    auto emit = [&](int l, const V(&v)[3][kSlots]) {   // light l (per-light mode) or the accumulated image (l = 0)
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        float tv[kCtTexels];
        unpair_to<kSlots>(v[c], 0, tv);
        store_seg<kCtTexels>(at<false>(p.out, b, c, w) + (F.per_light ? (int64_t)l * p.out_sl : 0), w.vec, w.valid, tv);
      }
    };
    ct_forward_group<WF, kLight, V, kSlots, decltype(emit), kFwdUnroll, LaneViews<V, kSlots>>(S, F, a, n, r, m, x, y, hg, emit,
                                                                                                GeomCache<V>(), cv);
  }
}

// Backward / fused loss (p.is_loss), with d_intensity, d_lights and d_view (= d camera position) when their pointers are
// set.  Accumulate mode with L > 1 runs the two-pass backward (the summed image is recomputed).  The shared-parameter
// gradients go warp shuffle -> shared atomics per light, and one global atomic per CTA and value.
template <int WF, int kLight>
__global__ void __launch_bounds__(kCtThreads, 2) cam_backward_kernel(const __grid_constant__ CtKParams p) {
  __shared__ CtStage S;
  __shared__ float s_int[PBR_MAX_LIGHTS * 3];
  __shared__ float s_geo[(PBR_MAX_LIGHTS + 1) * 3];
  __shared__ float s_loss[kCtThreads / 32];
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  const CtFlags& F = p.flags;
  const bool int_grad = p.d_intensity != nullptr;
  const bool is_loss = p.is_loss != 0;
  const bool has_normal = p.normal.ptr != nullptr;
  for (int i = tid; i < F.L * 3; i += kCtThreads) s_int[i] = 0.0f;
  for (int i = tid; i < (F.L + 1) * 3; i += kCtThreads) s_geo[i] = 0.0f;
  stage_params(p, S);  // ends with __syncthreads()
  const Where w = locate_ct<false>(p);
  const float live = w.active ? 1.0f : 0.0f;   // edge threads stay for the warp-wide reductions

  V x[kSlots];
  float y;
  LaneViews<V, kSlots> cv;
  LightGeomT<V> hg[kSlots];
  cam_setup<kLight>(p, S, w, x, y, cv, hg);

  float loss_local = 0.0f;
  const int b0 = blockIdx.z * p.mats_per_cta;
  const int b1 = min(b0 + p.mats_per_cta, p.B);
  for (int b = b0; b < b1; ++b) {
    float araw[3][kCtTexels], nraw[3][kCtTexels], rough[kCtTexels], mraw[3][kCtTexels];
    load_material<WF, false>(p, w, b, araw, nraw, rough, mraw, has_normal);
    if (b + 1 < b1) prefetch_material<WF, false>(p, w, b + 1, has_normal);
    V a[3][kSlots], n[3][kSlots], r[kSlots], m[3][kSlots];
    pairs_of3<kSlots>(araw, 0, a); pairs_of3<kSlots>(nraw, 0, n); pairs_of3<kSlots>(mraw, 0, m); pairs_of<kSlots>(rough, 0, r);
    // dLoss/d out of light l (per-light mode) or of the accumulated image: grad_out, or 2 * loss_scale * (out - target)
    auto gout = [&](int l, const V(&outv)[3][kSlots], V(&g)[3][kSlots]) {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        float src[kCtTexels], ov[kCtTexels], gv[kCtTexels];
        load_seg<kCtTexels>(at<false>(p.gsrc, b, c, w) + (F.per_light ? (int64_t)l * p.gsrc_sl : 0), w.vec, w.valid, src);
        unpair_to<kSlots>(outv[c], 0, ov);
#pragma unroll
        for (int i = 0; i < kCtTexels; ++i) {
          if (is_loss) {
            const float diff = (i < w.valid) ? ov[i] - src[i] : 0.0f;
            loss_local += diff * diff;
            gv[i] = 2.0f * p.loss_scale * diff;
          } else {
            gv[i] = (i < w.valid) ? src[i] : 0.0f;
          }
        }
        pairs_of<kSlots>(gv, 0, g[c]);
      }
    };
    auto int_sink = [&](int l, const float(&gi)[3]) {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float sum = warp_sum(gi[c] * live);
        if ((tid & 31) == 0) atomicAdd(&s_int[3 * l + c], sum);
      }
    };
    V da[3][kSlots], dn[3][kSlots], dr[kSlots], dm[3][kSlots];
    ct_backward_group<WF, kLight, V, kSlots, decltype(gout), decltype(int_sink), NoFetch, CtaGeomSink, NoSavedOut, kBwdUnroll,
                      LaneViews<V, kSlots>>(S, F, a, n, r, m, x, y, hg, gout, int_sink, da, dn, dr, dm, NoFetch(), GeomCache<V>(),
                                            CtaGeomSink{s_geo, F.L, tid, live, nullptr}, NoSavedOut(), int_grad, cv);
    if (w.active) {
      float d_albedo[3][kCtTexels], d_normal[3][kCtTexels], d_rough[kCtTexels], d_met[3][kCtTexels];
#pragma unroll
      for (int c = 0; c < 3; ++c) { unpair_to<kSlots>(da[c], 0, d_albedo[c]); unpair_to<kSlots>(dn[c], 0, d_normal[c]); unpair_to<kSlots>(dm[c], 0, d_met[c]); }
      unpair_to<kSlots>(dr, 0, d_rough);
      if (p.d_albedo.ptr) {
#pragma unroll
        for (int c = 0; c < 3; ++c) store_seg<kCtTexels>(at<false>(p.d_albedo, b, c, w), w.vec, w.valid, d_albedo[c]);
      }
      if (has_normal && p.d_normal.ptr) {
#pragma unroll
        for (int c = 0; c < 3; ++c) store_seg<kCtTexels>(at<false>(p.d_normal, b, c, w), w.vec, w.valid, d_normal[c]);
      }
      if (p.d_roughness.ptr) store_seg<kCtTexels>(at<false>(p.d_roughness, b, 0, w), w.vec, w.valid, d_rough);
      if (p.d_metspec.ptr) {
#pragma unroll
        for (int c = 0; c < (WF == 0 ? 1 : 3); ++c) store_seg<kCtTexels>(at<false>(p.d_metspec, b, c, w), w.vec, w.valid, d_met[c]);
      }
    }
  }

  if (is_loss) {
    const float sum = warp_sum(loss_local * live);
    if ((tid & 31) == 0) s_loss[tid >> 5] = sum;
  }
  __syncthreads();
  if (tid <= F.L) {
    // the camera sum is already d/d c (camera_view_bwd per texel); a directional light's sum is w.r.t. its UNIT
    // direction, whose Jacobian is image-constant and applied here, once
    const float g[3] = {s_geo[3 * tid], s_geo[3 * tid + 1], s_geo[3 * tid + 2]};
    float o[3] = {g[0], g[1], g[2]};
    float* dst = p.d_view;
    if (tid < F.L) {
      const float* lights = p.lights_dev ? p.lights_dev : p.lights;
      if (!F.point) normalize_bwd(lights + 3 * tid, g, o);
      dst = p.d_lights ? p.d_lights + 3 * tid : nullptr;
    }
    if (dst) {
#pragma unroll
      for (int c = 0; c < 3; ++c) atomicAdd(dst + c, o[c]);
    }
  }
  if (is_loss && tid == 0) {
    float sum = 0.0f;
    for (int i = 0; i < kCtThreads / 32; ++i) sum += s_loss[i];
    atomicAdd(p.loss_sum, sum);
  }
  if (int_grad) {
    for (int i = tid; i < F.L * 3; i += kCtThreads) atomicAdd(&p.d_intensity[i], s_int[i]);
  }
}

}  // namespace pbr

#include "pbr_ct_stream.cuh"

#if PBR_MAIN_PART

namespace pbr {

// ------------------------------------------------------------------------------------------------
// streaming kernels: workflow conversions, blend, colour space, normal ingestion
// ------------------------------------------------------------------------------------------------
struct ConvKParams {
  int B, H, W, vec_ok, albedo_is_srgb;
  int met_channels;   // m2s: 1 or 3
  PbrPlane albedo, metspec, out0, out1;
  PbrPlane g0, g1, d_albedo, d_metspec;   // backward
};

template <bool kM2S>
__global__ void __launch_bounds__(kThreads) convert_kernel(const __grid_constant__ ConvKParams p) {
  const Where w = locate(p.H, p.W, p.vec_ok != 0);
  if (!w.active) return;
  float a[3][kTexels], m[3][kTexels], o0[3][kTexels], o1[3][kTexels];
#pragma unroll
  for (int c = 0; c < 3; ++c) load_seg<kTexels>(p.albedo.ptr + plane_off(p.albedo, w.b, c, w.row, w.col0), w.vec, w.valid, a[c]);
  const int mc = kM2S ? p.met_channels : 3;
#pragma unroll
  for (int c = 0; c < 3; ++c)
    if (c < mc) load_seg<kTexels>(p.metspec.ptr + plane_off(p.metspec, w.b, c, w.row, w.col0), w.vec, w.valid, m[c]);
#pragma unroll
  for (int i = 0; i < kTexels; ++i) {
    if (kM2S) {
      const float a3[3] = {a[0][i], a[1][i], a[2][i]};
      const float m3[3] = {m[0][i], mc == 3 ? m[1][i] : m[0][i], mc == 3 ? m[2][i] : m[0][i]};
      float d3[3], s3[3];
      convert_m2s(a3, m3, p.albedo_is_srgb != 0, d3, s3);
#pragma unroll
      for (int c = 0; c < 3; ++c) { o0[c][i] = d3[c]; o1[c][i] = s3[c]; }
    } else {
#pragma unroll
      for (int c = 0; c < 3; ++c) convert_s2m(a[c][i], m[c][i], p.albedo_is_srgb != 0, &o0[c][i], &o1[c][i]);
    }
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    store_seg<kTexels>(p.out0.ptr + plane_off(p.out0, w.b, c, w.row, w.col0), w.vec, w.valid, o0[c]);
    store_seg<kTexels>(p.out1.ptr + plane_off(p.out1, w.b, c, w.row, w.col0), w.vec, w.valid, o1[c]);
  }
}

__device__ __forceinline__ void atomic_min_float(float* addr, float v) {
  if (v >= 0.0f) atomicMin(reinterpret_cast<int*>(addr), __float_as_int(v));
  else atomicMax(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// CTA-wide minimum -> ONE atomic per CTA (a per-warp atomic on a single address serialises ~10^5 operations per
// launch at 4096^2).  Every thread of the CTA must call it.
__device__ __forceinline__ void cta_min_atomic(float v, float* dst) {
  __shared__ float s_min[kThreads / 32];
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  v = warp_min(v);
  if ((tid & 31) == 0) s_min[tid >> 5] = v;
  __syncthreads();
  if (tid == 0) {
    float m = s_min[0];
    for (int i = 1; i < kThreads / 32; ++i) m = fminf(m, s_min[i]);
    if (m != INFINITY) atomic_min_float(dst, m);
  }
}

struct BlendKParams {
  PbrBlendDesc d;
  int vec_ok;
  float width_eps;     // blend_width + 1e-6 (fp32)
  Linspace grad;       // gradient modes: linspace(0, 1, W or H)
};

__global__ void __launch_bounds__(kThreads) blend_kernel(const __grid_constant__ BlendKParams p) {
  const PbrBlendDesc& d = p.d;
  const Where w = locate(d.H, d.W, p.vec_ok != 0);
  float mask[kTexels];
  if (d.mask_mode == PBR_MASK_GIVEN) {
    load_seg<kTexels>(d.mask.ptr + plane_off(d.mask, w.b, 0, w.row, w.col0), w.vec, w.valid, mask);
  } else if (d.mask_mode == PBR_MASK_SIGMOID) {
    float p1[kTexels], p2[kTexels];
    load_seg<kTexels>(d.prop1.ptr + plane_off(d.prop1, w.b, 0, w.row, w.col0), w.vec, w.valid, p1);
    load_seg<kTexels>(d.prop2.ptr + plane_off(d.prop2, w.b, 0, w.row, w.col0), w.vec, w.valid, p2);
#pragma unroll
    for (int i = 0; i < kTexels; ++i) mask[i] = sigmoid_mask(p1[i], p2[i], d.shift, d.apply_shift != 0, p.width_eps);
  } else if (d.mask_mode == PBR_MASK_GRADIENT_H) {
#pragma unroll
    for (int i = 0; i < kTexels; ++i) {
      int col = w.col0 + i;
      mask[i] = linspace_at(p.grad, col < d.W ? col : d.W - 1);
    }
  } else {
    float v = linspace_at(p.grad, w.row);
#pragma unroll
    for (int i = 0; i < kTexels; ++i) mask[i] = v;
  }
  if (d.mask_mode != PBR_MASK_GIVEN && d.mask_out.ptr && w.active)
    store_seg<kTexels>(d.mask_out.ptr + plane_off(d.mask_out, w.b, 0, w.row, w.col0), w.vec, w.valid, mask);

  float nmin = INFINITY;
  for (int m = 0; m < d.n_maps; ++m) {
    const PbrBlendMap& bm = d.maps[m];
    if (bm.is_normal) {
      float a[3][kTexels], b[3][kTexels], o[3][kTexels];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        load_seg<kTexels>(bm.a.ptr + plane_off(bm.a, w.b, c, w.row, w.col0), w.vec, w.valid, a[c]);
        load_seg<kTexels>(bm.b.ptr + plane_off(bm.b, w.b, c, w.row, w.col0), w.vec, w.valid, b[c]);
      }
#pragma unroll
      for (int i = 0; i < kTexels; ++i) {
        const float a3[3] = {a[0][i], a[1][i], a[2][i]};
        const float b3[3] = {b[0][i], b[1][i], b[2][i]};
        float o3[3];
        blend_normal(mask[i], a3, b3, o3);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          o[c][i] = o3[c];
          if (i < w.valid) nmin = fminf(nmin, o3[c]);
        }
      }
      if (w.active) {
#pragma unroll
        for (int c = 0; c < 3; ++c) store_seg<kTexels>(bm.out.ptr + plane_off(bm.out, w.b, c, w.row, w.col0), w.vec, w.valid, o[c]);
      }
    } else {
      for (int c = 0; c < bm.channels; ++c) {
        float a[kTexels], b[kTexels], o[kTexels];
        load_seg<kTexels>(bm.a.ptr + plane_off(bm.a, w.b, c, w.row, w.col0), w.vec, w.valid, a);
        load_seg<kTexels>(bm.b.ptr + plane_off(bm.b, w.b, c, w.row, w.col0), w.vec, w.valid, b);
#pragma unroll
        for (int i = 0; i < kTexels; ++i) o[i] = blend_lerp(mask[i], a[i], b[i]);
        if (w.active) store_seg<kTexels>(bm.out.ptr + plane_off(bm.out, w.b, c, w.row, w.col0), w.vec, w.valid, o);
      }
    }
  }
  if (d.normal_min) cta_min_atomic(w.active ? nmin : INFINITY, d.normal_min);
}

struct ColorKParams {
  int B, C, H, W, vec_ok, to_linear;
  PbrPlane in, out;
};

__global__ void __launch_bounds__(kThreads) color_kernel(const __grid_constant__ ColorKParams p) {
  const Where w = locate(p.H, p.W, p.vec_ok != 0);
  if (!w.active) return;
  for (int c = 0; c < p.C; ++c) {
    float v[kTexels];
    load_seg<kTexels>(p.in.ptr + plane_off(p.in, w.b, c, w.row, w.col0), w.vec, w.valid, v);
#pragma unroll
    for (int i = 0; i < kTexels; ++i) v[i] = p.to_linear ? srgb_decode<false, float>(v[i], nullptr) : srgb_encode<false, float>(v[i], nullptr);
    store_seg<kTexels>(p.out.ptr + plane_off(p.out, w.b, c, w.row, w.col0), w.vec, w.valid, v);
  }
}

struct NormalKParams {
  int B, H, W, vec_ok, channels;
  PbrPlane in, out;
  float* result;
  const float* cond_min;   // ingest: skip the launch's work when *cond_min < 0 (PbrNormalDesc.cond_min)
  PbrPlane g_out, d_in;    // backward
};

__global__ void __launch_bounds__(kThreads) normal_min_kernel(const __grid_constant__ NormalKParams p) {
  const Where w = locate(p.H, p.W, p.vec_ok != 0);
  float mn = INFINITY;
  for (int c = 0; c < p.channels; ++c) {
    float v[kTexels];
    load_seg<kTexels>(p.in.ptr + plane_off(p.in, w.b, c, w.row, w.col0), w.vec, w.valid, v);
#pragma unroll
    for (int i = 0; i < kTexels; ++i)
      if (i < w.valid) mn = fminf(mn, v[i]);
  }
  cta_min_atomic(w.active ? mn : INFINITY, p.result);
}

__global__ void __launch_bounds__(kThreads) normal_ingest_kernel(const __grid_constant__ NormalKParams p) {
  const Where w = locate(p.H, p.W, p.vec_ok != 0);
  if (!w.active) return;
  if (p.cond_min && __ldg(p.cond_min) < 0.0f) return;   // base.py:212: a map with a negative component is kept as it is
  float v[3][kTexels], o[3][kTexels];
  for (int c = 0; c < p.channels; ++c) load_seg<kTexels>(p.in.ptr + plane_off(p.in, w.b, c, w.row, w.col0), w.vec, w.valid, v[c]);
#pragma unroll
  for (int i = 0; i < kTexels; ++i) {
    float o3[3];
    if (p.channels == 3) {
      const float v3[3] = {v[0][i], v[1][i], v[2][i]};
      ingest_normal3(v3, o3);
    } else {
      const float v2[2] = {v[0][i], v[1][i]};
      ingest_normal2(v2, o3);
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) o[c][i] = o3[c];
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) store_seg<kTexels>(p.out.ptr + plane_off(p.out, w.b, c, w.row, w.col0), w.vec, w.valid, o[c]);
}

}  // namespace pbr

#include "pbr_aux_kernels.cuh"
#include "pbr_grad_kernels.cuh"
#endif   // PBR_MAIN_PART


namespace pbr {

// ------------------------------------------------------------------------------------------------
// host side of the C ABI
// ------------------------------------------------------------------------------------------------
// vector access of kTexels floats is legal when the base pointer and every stride keep that alignment
static bool plane_vec_ok(const PbrPlane& pl) {
  if (!pl.ptr || kTexels == 1) return true;
  return (reinterpret_cast<uintptr_t>(pl.ptr) % (4 * kTexels) == 0) && (pl.sb % kTexels == 0) && (pl.sc % kTexels == 0) &&
         (pl.sh % kTexels == 0);
}

// A CTA of `threads` threads covers a strip of up to 256 texels of blockDim.y consecutive rows.
static void launch_shape(int B, int H, int W, dim3& grid, dim3& block, int threads = kThreads, int texels = kTexels) {
  const int max_bx = 256 / texels < threads ? 256 / texels : threads;
  int groups = (W + texels - 1) / texels;
  int bx = 1;
  while (bx < groups && bx < max_bx) bx <<= 1;
  int by = threads / bx;
  block = dim3(bx, by, 1);
  grid = dim3((groups + bx - 1) / bx, (H + by - 1) / by, B);
}
// smallest blockDim.y any kernel is launched with
constexpr int kMinBy = 1;

static int check_dims(int B, int H, int W) {
  if (B < 1 || H < 1 || W < 1 || B > 65535 || H > 65535 * kMinBy) return PBR_E_SHAPE;  // grid.z = ceil(B / mats), grid.y = ceil(H / blockDim.y), blockDim.y >= kMinBy
  return PBR_OK;
}

static int fill_ct_params(const PbrCtDesc* d, CtKParams& k) {
  if (!d) return PBR_E_NULL;
  if (int rc = check_dims(d->B, d->H, d->W)) return rc;
  if (d->L < 1) return PBR_E_SHAPE;
  if (d->L > PBR_MAX_LIGHTS) return PBR_E_TOO_MANY;
  if (d->workflow != PBR_WORKFLOW_METALLIC && d->workflow != PBR_WORKFLOW_SPECULAR) return PBR_E_ENUM;
  if (d->metallic_channels != 0 && d->metallic_channels != 1 && d->metallic_channels != 3) return PBR_E_CHANNELS;
  if (d->light_type != PBR_LIGHT_DIRECTIONAL && d->light_type != PBR_LIGHT_POINT) return PBR_E_ENUM;
  if (!d->albedo.ptr || !d->roughness.ptr || !d->metspec.ptr || !d->view || !d->lights || !d->intensity) return PBR_E_NULL;
  k.B = d->B; k.H = d->H; k.W = d->W;
  k.force_generic = d->force_generic;
  k.flags.L = d->L;
  k.flags.point = d->light_type == PBR_LIGHT_POINT;
  k.flags.albedo_is_srgb = d->albedo_is_srgb != 0;
  k.flags.specular_is_srgb = d->specular_is_srgb != 0;
  k.flags.return_srgb = d->return_srgb != 0;
  k.flags.per_light = d->per_light != 0;
  k.albedo = d->albedo; k.normal = d->normal; k.roughness = d->roughness; k.metspec = d->metspec;
  k.out = d->out; k.out_sl = d->out_sl;
  k.vec_ok = plane_vec_ok(d->albedo) && plane_vec_ok(d->normal) && plane_vec_ok(d->roughness) && plane_vec_ok(d->metspec);
  const float s = d->light_size > 0.0f ? d->light_size : 1.0f;  // `light_size or 1.0`, cooktorrance.py:130
  k.lsx = make_linspace(-s / 2, s / 2, d->W);
  k.lsy = make_linspace(-s / 2, s / 2, d->H);
  if (d->params_on_device) {
    k.view_dev = d->view; k.lights_dev = d->lights; k.inten_dev = d->intensity;
  } else {
    k.view_dev = nullptr; k.lights_dev = nullptr; k.inten_dev = nullptr;
    for (int i = 0; i < 3; ++i) k.view[i] = d->view[i];
    for (int i = 0; i < 3 * d->L; ++i) { k.lights[i] = d->lights[i]; k.inten[i] = d->intensity[i]; }
  }
  return PBR_OK;
}

static int launch_result() {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaGetLastError();   // this launch's own status: read AND cleared, so a failure is reported once, here
  return e == cudaSuccess ? PBR_OK : (int)e;
}

// Point light with L == 1: the light geometry of a texel is shared by every material of the batch,
// so a thread walks over up to kHoistMats materials and computes it once.
constexpr int kHoistMats = PBR_HOIST_MATS;

// Point lights with L > 1: the geometry of every light is computed once per texel pair, parked in shared memory
// (GeomCache, pbr_shade.cuh) and reused by every material of the walk - it is ~55 % of the forward arithmetic of a
// texel-light.  Worth it from two materials on, and while the cache leaves room for enough CTAs per SM.
#ifndef PBR_GC_MAX_BYTES
#define PBR_GC_MAX_BYTES (100 * 1024)   // L <= 16 with the 6-field cache: at least 2 CTAs per SM
#endif
#ifndef PBR_GC_ALL_MAX_LIGHTS
#define PBR_GC_ALL_MAX_LIGHTS 4   // up to here all 8 geometry fields are cached and the backward keeps 3 CTAs per SM
#endif
static size_t geom_cache_bytes(int L, int light_mode) { return (size_t)L * geom_fields(light_mode) * kSlots * kCtThreads * sizeof(V); }
static bool vec_fast_disabled() {   // A/B and test switch: run the element-access flavour on shapes the fast one would take
  static const bool off = [] { const char* e = getenv("PBR_DISABLE_VEC_FAST"); return e && e[0] && e[0] != '0'; }();
  return off;
}
static bool geom_cache_disabled() {
  static const bool off = [] { const char* e = getenv("PBR_DISABLE_GEOM_CACHE"); return e && e[0] && e[0] != '0'; }();
  return off;
}

#ifndef PBR_GC_BIG_MAX_LIGHTS
#define PBR_GC_BIG_MAX_LIGHTS 8   // backward, 4 < L <= 8: all 8 fields cached, full register budget (2 CTAs per SM by registers anyway)
#endif
static int light_mode(const CtKParams& k, bool backward) {
  if (!k.flags.point) return kLightDirectional;
  if (!k.vec_fast) return kLightPoint;              // the element-access flavour only exists for the uncached light modes
  if (k.d_lights || k.d_view) {
    // geometry gradients (shared parameters of a fit with unknown lighting): the 6-field cache when a walk over several
    // materials pays for it, else the per-texel geometry
    if (backward && k.flags.L > 1 && k.B >= 2 && !geom_cache_disabled() &&
        geom_cache_bytes(k.flags.L, kLightPointCached) <= (size_t)PBR_GC_MAX_BYTES) return kLightPointCached;
    return kLightPoint;
  }
  if (k.flags.L == 1) return kLightPointHoisted;
  if (k.B >= 2 && !geom_cache_disabled()) {
    if (k.flags.L <= PBR_GC_ALL_MAX_LIGHTS) return kLightPointCachedAll;
    // (not under the Adam epilogue: with its 30 KB of staging the two CTAs would leave the SM almost no L1, 12.21 -> 12.35 ms on C5)
    if (backward && !k.adam_on && k.flags.L <= PBR_GC_BIG_MAX_LIGHTS) return kLightPointCachedAllBig;
    if (geom_cache_bytes(k.flags.L, kLightPointCached) <= (size_t)PBR_GC_MAX_BYTES) return kLightPointCached;
  }
  return kLightPoint;
}

static void ct_launch_shape(CtKParams& k, dim3& grid, dim3& block, bool backward) {
  launch_shape(k.B, k.H, k.W, grid, block, kCtThreads, kCtTexels);
  const int lm = light_mode(k, backward);
  k.mats_per_cta = (lm == kLightPointHoisted || is_cached(lm)) ? (k.B < kHoistMats ? k.B : kHoistMats) : 1;
  grid.z = (k.B + k.mats_per_cta - 1) / k.mats_per_cta;
}

// most dynamic shared memory a generic kernel is ever launched with: geometry cache + Adam staging (or the partial-sum slots)
constexpr size_t kMaxDynSmem = (size_t)PBR_GC_MAX_BYTES + 30 * kCtThreads * kCtTexels * 4;
// launch with `smem` bytes of dynamic shared memory (opt-in above 48 KB, once per kernel instantiation and device)
template <void (*Kern)(CtKParams)>
static void launch_dyn(const CtKParams& k, dim3 grid, dim3 block, size_t smem, cudaStream_t st) {
  static std::atomic<uint64_t> configured{0};
  int dev = 0;
  cudaGetDevice(&dev);
  const uint64_t bit = 1ull << (dev & 63);
  if (!(configured.load(std::memory_order_acquire) & bit)) {   // static + dynamic may exceed 48 KB before dynamic alone does
    cudaFuncSetAttribute(Kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxDynSmem);
    configured.fetch_or(bit, std::memory_order_release);
  }
  Kern<<<grid, block, smem, st>>>(k);
}

// kernel workflow index: 0 metallic (1-channel map), 1 specular, 2 metallic with a 3-channel map
static int kernel_workflow(const PbrCtDesc* d) {
  if (d->workflow == PBR_WORKFLOW_SPECULAR) return 1;
  return d->metallic_channels == 3 ? 2 : 0;
}

// what the plain-case flavour (kFmAccum) assumes besides its own mode: the reference's default colour handling and a
// normal map, on the 64-bit-access flavour
static bool generic_fast_disabled() {   // A/B and test switch: run the general flavour where a plain-case one would be picked
  static const bool off = [] { const char* e = getenv("PBR_DISABLE_GENERIC_FAST"); return e && e[0] && e[0] != '0'; }();
  return off;
}
template <int WF>
static bool plain_case(const CtKParams& k) {
  return kGenericFast && !generic_fast_disabled() && k.vec_fast && k.flags.albedo_is_srgb && k.flags.return_srgb && (WF != 1 || k.flags.specular_is_srgb) &&
         k.normal.ptr != nullptr;
}

template <int WF>
static void launch_fwd(const CtKParams& k, dim3 grid, dim3 block, cudaStream_t st) {
  const int lm = light_mode(k, false);
  if (!k.vec_fast) {   // any alignment / ragged width: element accesses, uncached light modes
    if (lm == kLightDirectional) ct_forward_kernel<WF, kLightDirectional, false><<<grid, block, 0, st>>>(k);
    else ct_forward_kernel<WF, kLightPoint, false><<<grid, block, 0, st>>>(k);
    return;
  }
  const bool accum = plain_case<WF>(k) && !k.flags.per_light;   // the kFmAccum flavour applies
  switch (lm) {
    case kLightDirectional: ct_forward_kernel<WF, kLightDirectional><<<grid, block, 0, st>>>(k); break;
    case kLightPoint:
      if (accum && k.flags.L > 1) ct_forward_kernel<WF, kLightPoint, true, kFmAccum><<<grid, block, 0, st>>>(k);
      else ct_forward_kernel<WF, kLightPoint><<<grid, block, 0, st>>>(k);
      break;
    case kLightPointCached:
      if (accum) launch_dyn<ct_forward_kernel<WF, kLightPointCached, true, kFmAccum>>(k, grid, block, geom_cache_bytes(k.flags.L, kLightPointCached), st);
      else launch_dyn<ct_forward_kernel<WF, kLightPointCached>>(k, grid, block, geom_cache_bytes(k.flags.L, kLightPointCached), st);
      break;
    case kLightPointCachedAll:
      if (accum) launch_dyn<ct_forward_kernel<WF, kLightPointCachedAll, true, kFmAccum>>(k, grid, block, geom_cache_bytes(k.flags.L, kLightPointCachedAll), st);
      else launch_dyn<ct_forward_kernel<WF, kLightPointCachedAll>>(k, grid, block, geom_cache_bytes(k.flags.L, kLightPointCachedAll), st);
      break;
    default: ct_forward_kernel<WF, kLightPointHoisted><<<grid, block, 0, st>>>(k); break;
  }
}

// Adam staging of the fused fit step: parameter + two moments of up to 10 channels per texel (pbr_ct_fit_step)
constexpr size_t kAdamSmemBytes = (size_t)30 * kCtThreads * kCtTexels * sizeof(float);

template <int WF>
static void launch_bwd(const CtKParams& k_in, dim3 grid, dim3 block, cudaStream_t st) {
  CtKParams k = k_in;
  const int lm = light_mode(k, true);
  const size_t cache = is_cached(lm) ? geom_cache_bytes(k.flags.L, lm) : 0;
  k.adam_smem_off = (int)cache;
  size_t smem = cache + (k.adam_on ? kAdamSmemBytes : 0);
  // per-thread slots of the shared-parameter gradients, when they fit next to the cache (else: warp-shuffle reduction per light)
  k.part_on = 0;
  if (k.d_intensity || k.d_lights || k.d_view) {
    const size_t part = (size_t)k.flags.L * ((k.d_lights || k.d_view) ? 6 : 3) * kCtThreads * sizeof(float);
    if (part <= 48 * 1024 && smem + part <= kMaxDynSmem) {
      k.part_on = 1;
      k.part_smem_off = (int)smem;
      smem += part;
    }
  }
  if (k.d_lights || k.d_view) {   // geometry gradients: the uncached per-texel light modes
    if (k.vec_fast) {
      if (lm == kLightPointCached) launch_dyn<ct_backward_kernel<WF, kLightPointCached, true>>(k, grid, block, smem, st);
      else if (k.flags.point) launch_dyn<ct_backward_kernel<WF, kLightPoint, true>>(k, grid, block, smem, st);
      else launch_dyn<ct_backward_kernel<WF, kLightDirectional, true>>(k, grid, block, smem, st);
    } else {
      if (k.flags.point) launch_dyn<ct_backward_kernel<WF, kLightPoint, true, false>>(k, grid, block, smem, st);
      else launch_dyn<ct_backward_kernel<WF, kLightDirectional, true, false>>(k, grid, block, smem, st);
    }
    return;
  }
  if (!k.vec_fast) {
    if (lm == kLightDirectional) launch_dyn<ct_backward_kernel<WF, kLightDirectional, false, false>>(k, grid, block, smem, st);
    else launch_dyn<ct_backward_kernel<WF, kLightPoint, false, false>>(k, grid, block, smem, st);
    return;
  }
  // the kFmAccum flavour: what autograd asks for after an accumulated render (every map gradient, the saved output handed in)
  const bool accum = plain_case<WF>(k) && !k.flags.per_light && k.flags.L > 1 && !k.is_loss && !k.adam_on && !k.d_intensity &&
                     k.fout.ptr && k.d_albedo.ptr && k.d_normal.ptr && k.d_roughness.ptr && k.d_metspec.ptr;
  switch (lm) {
    case kLightDirectional: launch_dyn<ct_backward_kernel<WF, kLightDirectional>>(k, grid, block, smem, st); break;
    case kLightPoint:
      if (accum) launch_dyn<ct_backward_kernel<WF, kLightPoint, false, true, kFmAccum>>(k, grid, block, smem, st);
      else launch_dyn<ct_backward_kernel<WF, kLightPoint>>(k, grid, block, smem, st);
      break;
    case kLightPointCached:
      if (accum) launch_dyn<ct_backward_kernel<WF, kLightPointCached, false, true, kFmAccum>>(k, grid, block, smem, st);
      else launch_dyn<ct_backward_kernel<WF, kLightPointCached>>(k, grid, block, smem, st);
      break;
    case kLightPointCachedAll:
      if (accum) launch_dyn<ct_backward_kernel<WF, kLightPointCachedAll, false, true, kFmAccum>>(k, grid, block, smem, st);
      else launch_dyn<ct_backward_kernel<WF, kLightPointCachedAll>>(k, grid, block, smem, st);
      break;
    case kLightPointCachedAllBig:
      if (accum) launch_dyn<ct_backward_kernel<WF, kLightPointCachedAllBig, false, true, kFmAccum>>(k, grid, block, smem, st);
      else launch_dyn<ct_backward_kernel<WF, kLightPointCachedAllBig>>(k, grid, block, smem, st);
      break;
    default: launch_dyn<ct_backward_kernel<WF, kLightPointHoisted>>(k, grid, block, smem, st); break;
  }
}

static int fill_grads(const PbrCtGrads* g, CtKParams& k) {
  if (!g) return PBR_E_NULL;
  k.d_albedo = g->d_albedo; k.d_normal = g->d_normal; k.d_roughness = g->d_roughness; k.d_metspec = g->d_metspec;
  k.d_intensity = g->d_intensity;
  k.d_lights = g->d_lights; k.d_view = g->d_view;
  if (k.d_lights || k.d_view) k.force_generic = 1;
  k.vec_ok = k.vec_ok && plane_vec_ok(g->d_albedo) && plane_vec_ok(g->d_normal) && plane_vec_ok(g->d_roughness) &&
             plane_vec_ok(g->d_metspec);
  return PBR_OK;
}

// ------------------------------------------------------------------------------------------------
// streamed (TMA-fed) fast path: one light, 16-byte aligned planes, W % 4 == 0 (pbr_ct_stream.cuh)
// ------------------------------------------------------------------------------------------------
static bool stream_disabled() {
  static const bool off = [] { const char* e = getenv("PBR_DISABLE_STREAM"); return e && e[0] && e[0] != '0'; }();
  return off;
}

static bool fits_i32(const PbrPlane& pl, int H, int W) {
  return !pl.ptr || ((int64_t)(H - 1) * pl.sh + W) < (int64_t)INT32_MAX;
}

static bool stream_shape(const CtKParams& k, dim3& grid, dim3& block, int& mats, bool per_warp) {
  if (stream_disabled() || k.force_generic || k.flags.L != 1 || !k.vec_ok || (k.W % 4) != 0) return false;
  static const int min_bx = [] { const char* e = getenv("PBR_STREAM_MIN_BX"); int v = e ? atoi(e) : 1; return v < 1 ? 1 : v; }();
  int groups = k.W / kST, bx = min_bx < 4 / kST ? 4 / kST : min_bx;   // a row segment is a multiple of 16 bytes
  if (per_warp) {   // per-warp copy pipelines: a warp must sit inside one tile row
    if (groups < 32) return false;   // narrower than one warp segment: the generic kernels take it
    if (bx < 32) bx = 32;
  }
  while (bx < groups && bx < kStreamThreads) bx <<= 1;
  int by = kStreamThreads / bx;
  int64_t gy = ((int64_t)k.H + by - 1) / by;
  if (gy > 65535) return false;
  mats = k.B < kHoistMats ? k.B : kHoistMats;
  block = dim3(bx, by, 1);
  grid = dim3((groups + bx - 1) / bx, (unsigned)gy, (k.B + mats - 1) / mats);
  return true;
}

template <void (*Kern)(CtKParams)>
static void stream_launch(const CtKParams& k, dim3 grid, dim3 block, int planes, cudaStream_t st) {
  static std::atomic<uint64_t> configured{0};   // per kernel instantiation: bit d = opted in on device d
  int dev = 0;
  cudaGetDevice(&dev);
  const uint64_t bit = 1ull << (dev & 63);
  if (!(configured.load(std::memory_order_acquire) & bit)) {
    cudaFuncSetAttribute(Kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSrcPlanes * kTileFloats * 4 * kStages);
    configured.fetch_or(bit, std::memory_order_release);
  }
  size_t smem = (size_t)planes * kTileFloats * 4 * kStages;
  Kern<<<grid, block, smem, st>>>(k);
}

template <int WF>
static void launch_fwd_stream(const CtKParams& k, dim3 grid, dim3 block, cudaStream_t st) {
  const int planes = k.normal.ptr ? Slots<WF, false>::count : Slots<WF, false>::count_no_normal;
  const bool fast = kStreamFast && block.x == (unsigned)kStreamThreads && block.y == 1 && (k.W % kTileFloats) == 0 && k.normal.ptr &&
                    k.flags.albedo_is_srgb && k.flags.return_srgb && (WF != 1 || k.flags.specular_is_srgb);
  if (fast) {
    if (k.flags.point) stream_launch<ct_forward_stream<WF, kLightPointHoisted, true>>(k, grid, block, planes, st);
    else stream_launch<ct_forward_stream<WF, kLightDirectional, true>>(k, grid, block, planes, st);
    return;
  }
  if (k.flags.point) stream_launch<ct_forward_stream<WF, kLightPointHoisted>>(k, grid, block, planes, st);
  else stream_launch<ct_forward_stream<WF, kLightDirectional>>(k, grid, block, planes, st);
}

template <int WF, int kMode>
static void launch_bwd_stream_m(const CtKParams& k, dim3 grid, dim3 block, cudaStream_t st) {
  const int planes = k.normal.ptr ? Slots<WF, true>::count : Slots<WF, true>::count_no_normal;
  // the plain case (full tiles of one row, a normal map, every gradient requested) runs the kFast flavour (pbr_ct_stream.cuh)
  const bool fast = kStreamFast && block.x == (unsigned)kStreamThreads && block.y == 1 && (k.W % kTileFloats) == 0 && k.normal.ptr &&
                    k.flags.albedo_is_srgb && k.flags.return_srgb && (WF != 1 || k.flags.specular_is_srgb) &&
                    k.d_albedo.ptr && k.d_normal.ptr && k.d_roughness.ptr && k.d_metspec.ptr;
  if (fast) {
    if (k.flags.point) stream_launch<ct_backward_stream<WF, kLightPointHoisted, kMode, true>>(k, grid, block, planes, st);
    else stream_launch<ct_backward_stream<WF, kLightDirectional, kMode, true>>(k, grid, block, planes, st);
    return;
  }
  if (k.flags.point) stream_launch<ct_backward_stream<WF, kLightPointHoisted, kMode>>(k, grid, block, planes, st);
  else stream_launch<ct_backward_stream<WF, kLightDirectional, kMode>>(k, grid, block, planes, st);
}

template <int WF>
static void launch_bwd_stream(const CtKParams& k, dim3 grid, dim3 block, cudaStream_t st) {
  const int mode = (k.is_loss ? kModeLoss : 0) | (k.d_intensity ? kModeIntGrad : 0);
  switch (mode) {
    case 0: launch_bwd_stream_m<WF, 0>(k, grid, block, st); break;
    case 1: launch_bwd_stream_m<WF, 1>(k, grid, block, st); break;
    case 2: launch_bwd_stream_m<WF, 2>(k, grid, block, st); break;
    default: launch_bwd_stream_m<WF, 3>(k, grid, block, st); break;
  }
}

// every Cook-Torrance kernel of one workflow behind one plain function (see PBR_PART at the top of this file)
template <int WF>
static void launch_wf(CtKParams& k, dim3 grid, dim3 block, bool stream, bool backward, cudaStream_t st) {
  if (stream) {
    if (backward) launch_bwd_stream<WF>(k, grid, block, st);
    else launch_fwd_stream<WF>(k, grid, block, st);
  } else {
    if (backward) launch_bwd<WF>(k, grid, block, st);
    else launch_fwd<WF>(k, grid, block, st);
  }
}
void launch_wf0(CtKParams& k, dim3 grid, dim3 block, bool stream, bool backward, cudaStream_t st);
void launch_wf1(CtKParams& k, dim3 grid, dim3 block, bool stream, bool backward, cudaStream_t st);
void launch_wf2(CtKParams& k, dim3 grid, dim3 block, bool stream, bool backward, cudaStream_t st);
#if PBR_HAS_WF(0)
void launch_wf0(CtKParams& k, dim3 grid, dim3 block, bool stream, bool backward, cudaStream_t st) { launch_wf<0>(k, grid, block, stream, backward, st); }
#endif
#if PBR_HAS_WF(1)
void launch_wf1(CtKParams& k, dim3 grid, dim3 block, bool stream, bool backward, cudaStream_t st) { launch_wf<1>(k, grid, block, stream, backward, st); }
#endif
#if PBR_HAS_WF(2)
void launch_wf2(CtKParams& k, dim3 grid, dim3 block, bool stream, bool backward, cudaStream_t st) { launch_wf<2>(k, grid, block, stream, backward, st); }
#endif

// the camera kernels of one workflow (pbr_ct_*_camera): directional lights, one point light (hoisted), several point lights
template <int WF>
static void launch_cam(const CtKParams& k, dim3 grid, dim3 block, bool backward, cudaStream_t st) {
  const int lm = !k.flags.point ? kLightDirectional : (k.flags.L == 1 ? kLightPointHoisted : kLightPoint);
  switch (lm) {
    case kLightDirectional:
      if (backward) cam_backward_kernel<WF, kLightDirectional><<<grid, block, 0, st>>>(k);
      else cam_forward_kernel<WF, kLightDirectional><<<grid, block, 0, st>>>(k);
      break;
    case kLightPointHoisted:
      if (backward) cam_backward_kernel<WF, kLightPointHoisted><<<grid, block, 0, st>>>(k);
      else cam_forward_kernel<WF, kLightPointHoisted><<<grid, block, 0, st>>>(k);
      break;
    default:
      if (backward) cam_backward_kernel<WF, kLightPoint><<<grid, block, 0, st>>>(k);
      else cam_forward_kernel<WF, kLightPoint><<<grid, block, 0, st>>>(k);
      break;
  }
}
void launch_cam_wf0(const CtKParams& k, dim3 grid, dim3 block, bool backward, cudaStream_t st);
void launch_cam_wf1(const CtKParams& k, dim3 grid, dim3 block, bool backward, cudaStream_t st);
void launch_cam_wf2(const CtKParams& k, dim3 grid, dim3 block, bool backward, cudaStream_t st);
#if PBR_HAS_WF(0)
void launch_cam_wf0(const CtKParams& k, dim3 grid, dim3 block, bool backward, cudaStream_t st) { launch_cam<0>(k, grid, block, backward, st); }
#endif
#if PBR_HAS_WF(1)
void launch_cam_wf1(const CtKParams& k, dim3 grid, dim3 block, bool backward, cudaStream_t st) { launch_cam<1>(k, grid, block, backward, st); }
#endif
#if PBR_HAS_WF(2)
void launch_cam_wf2(const CtKParams& k, dim3 grid, dim3 block, bool backward, cudaStream_t st) { launch_cam<2>(k, grid, block, backward, st); }
#endif

#if PBR_MAIN_PART
// shared tail of the three Cook-Torrance entry points
// every in-plane offset (row * sh + col) of a plane fits 32 bits
static bool planes_fit_i32(const CtKParams& k) {
  const PbrPlane* all[] = {&k.albedo, &k.normal, &k.roughness, &k.metspec, &k.out, &k.gsrc, &k.fout, &k.d_albedo, &k.d_normal,
                           &k.d_roughness, &k.d_metspec, &k.adam_m[0], &k.adam_m[1], &k.adam_m[2], &k.adam_m[3],
                           &k.adam_v[0], &k.adam_v[1], &k.adam_v[2], &k.adam_v[3]};
  for (const PbrPlane* pl : all)
    if (pl->ptr && (pl->sh < 0 || (int64_t)(k.H - 1) * pl->sh + k.W >= (int64_t)INT32_MAX)) return false;
  return true;
}

static int ct_dispatch(CtKParams& k, int wf, bool backward, cudaStream_t st) {
  dim3 grid, block;
  int mats = 1;
  k.vec_fast = k.vec_ok && (k.W % kCtTexels) == 0 && planes_fit_i32(k) && !vec_fast_disabled();
  bool stream = stream_shape(k, grid, block, mats, backward ? kPerWarpBwd : kPerWarpFwd);
  if (stream) {
    if (backward) stream = fits_i32(k.d_albedo, k.H, k.W) && fits_i32(k.d_normal, k.H, k.W) && fits_i32(k.d_roughness, k.H, k.W) && fits_i32(k.d_metspec, k.H, k.W);
    else stream = fits_i32(k.out, k.H, k.W);
  }
  if (stream) k.mats_per_cta = mats;
  else ct_launch_shape(k, grid, block, backward);
  switch (wf) {
    case 0: launch_wf0(k, grid, block, stream, backward, st); break;
    case 1: launch_wf1(k, grid, block, stream, backward, st); break;
    default: launch_wf2(k, grid, block, stream, backward, st); break;
  }
  return launch_result();
}

// the same for the camera kernels: every material walk spans up to kHoistMats materials (the views are per texel)
static int cam_dispatch(CtKParams& k, int wf, bool backward, cudaStream_t st) {
  dim3 grid, block;
  launch_shape(k.B, k.H, k.W, grid, block, kCtThreads, kCtTexels);
  k.mats_per_cta = k.B < kHoistMats ? k.B : kHoistMats;
  grid.z = (k.B + k.mats_per_cta - 1) / k.mats_per_cta;
  switch (wf) {
    case 0: launch_cam_wf0(k, grid, block, backward, st); break;
    case 1: launch_cam_wf1(k, grid, block, backward, st); break;
    default: launch_cam_wf2(k, grid, block, backward, st); break;
  }
  return launch_result();
}

static int dispatch(CtKParams& k, int wf, bool backward, bool camera, cudaStream_t st) {
  return camera ? cam_dispatch(k, wf, backward, st) : ct_dispatch(k, wf, backward, st);
}
#endif   // PBR_MAIN_PART

}  // namespace pbr

#if PBR_MAIN_PART
using namespace pbr;

extern "C" {

int pbr_abi_version(void) { return PBR_ABI_VERSION; }

const char* pbr_strerror(int code) {
  switch (code) {
    case PBR_OK: return "ok";
    case PBR_E_NULL: return "required pointer is NULL";
    case PBR_E_SHAPE: return "B/H/W/L out of range";
    case PBR_E_ENUM: return "workflow / light_type / mode out of range";
    case PBR_E_TOO_MANY: return "too many lights or maps for one launch";
    case PBR_E_CHANNELS: return "unsupported channel count";
    default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown pbr error";
  }
}

uint64_t pbr_sizeof(int which) {
  switch (which) {
    case 0: return sizeof(PbrPlane);
    case 1: return sizeof(PbrCtDesc);
    case 2: return sizeof(PbrCtGrads);
    case 3: return sizeof(PbrCtLoss);
    case 4: return sizeof(PbrConvDesc);
    case 5: return sizeof(PbrBlendMap);
    case 6: return sizeof(PbrBlendDesc);
    case 7: return sizeof(PbrColorDesc);
    case 8: return sizeof(PbrNormalDesc);
    case 9: return sizeof(PbrIngestDesc);
    case 10: return sizeof(PbrIndexMap);
    case 11: return sizeof(PbrIndexDesc);
    case 12: return sizeof(PbrAdamMap);
    case 13: return sizeof(PbrAdamDesc);
    case 14: return sizeof(PbrCtAdam);
    case 15: return sizeof(PbrNormalOpDesc);
    case 16: return sizeof(PbrConvGrads);
    case 17: return sizeof(PbrBlendGradMap);
    case 18: return sizeof(PbrBlendGrads);
    case 19: return sizeof(PbrNormalGrads);
    default: return 0;
  }
}

uint64_t pbr_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

// camera: desc->view is the camera position (cam_* kernels) instead of the view direction (ct_* kernels)
static int ct_forward(const PbrCtDesc* desc, bool camera, pbr_stream_t stream) {
  CtKParams k{};
  if (int rc = fill_ct_params(desc, k)) return rc;
  if (!desc->out.ptr) return PBR_E_NULL;
  k.vec_ok = k.vec_ok && plane_vec_ok(desc->out) && (desc->out_sl % kTexels == 0);
  return dispatch(k, kernel_workflow(desc), false, camera, (cudaStream_t)stream);
}

static int ct_backward(const PbrCtDesc* desc, const PbrCtGrads* grads, bool camera, pbr_stream_t stream) {
  CtKParams k{};
  if (int rc = fill_ct_params(desc, k)) return rc;
  if (int rc = fill_grads(grads, k)) return rc;
  if (!grads->grad_out.ptr) return PBR_E_NULL;
  k.gsrc = grads->grad_out; k.gsrc_sl = grads->grad_out_sl;
  k.is_loss = 0;
  k.vec_ok = k.vec_ok && plane_vec_ok(grads->grad_out) && (grads->grad_out_sl % kTexels == 0);
  if (!camera && !desc->per_light && desc->L > 1) {   // only the accumulate-mode backward of several lights has a use for it
    k.fout = grads->fwd_out;
    k.vec_ok = k.vec_ok && plane_vec_ok(grads->fwd_out);
  }
  return dispatch(k, kernel_workflow(desc), true, camera, (cudaStream_t)stream);
}

static int ct_loss_fwd_bwd(const PbrCtDesc* desc, const PbrCtLoss* loss, const PbrCtGrads* grads, bool camera,
                           pbr_stream_t stream) {
  CtKParams k{};
  if (int rc = fill_ct_params(desc, k)) return rc;
  if (int rc = fill_grads(grads, k)) return rc;
  if (!loss || !loss->target.ptr || !loss->loss_sum) return PBR_E_NULL;
  k.gsrc = loss->target; k.gsrc_sl = loss->target_sl;
  k.is_loss = 1;
  k.loss_scale = loss->loss_scale; k.loss_sum = loss->loss_sum;
  k.vec_ok = k.vec_ok && plane_vec_ok(loss->target) && (loss->target_sl % kTexels == 0);
  return dispatch(k, kernel_workflow(desc), true, camera, (cudaStream_t)stream);
}

int pbr_ct_forward(const PbrCtDesc* desc, pbr_stream_t stream) { return ct_forward(desc, false, stream); }
int pbr_ct_backward(const PbrCtDesc* desc, const PbrCtGrads* grads, pbr_stream_t stream) { return ct_backward(desc, grads, false, stream); }
int pbr_ct_loss_fwd_bwd(const PbrCtDesc* desc, const PbrCtLoss* loss, const PbrCtGrads* grads, pbr_stream_t stream) {
  return ct_loss_fwd_bwd(desc, loss, grads, false, stream);
}
int pbr_ct_forward_camera(const PbrCtDesc* desc, pbr_stream_t stream) { return ct_forward(desc, true, stream); }
int pbr_ct_backward_camera(const PbrCtDesc* desc, const PbrCtGrads* grads, pbr_stream_t stream) {
  return ct_backward(desc, grads, true, stream);
}
int pbr_ct_loss_fwd_bwd_camera(const PbrCtDesc* desc, const PbrCtLoss* loss, const PbrCtGrads* grads, pbr_stream_t stream) {
  return ct_loss_fwd_bwd(desc, loss, grads, true, stream);
}

int pbr_ct_fit_step(const PbrCtDesc* desc, const PbrCtLoss* loss, const PbrCtAdam* adam, float* d_intensity,
                    pbr_stream_t stream) {
  CtKParams k{};
  if (int rc = fill_ct_params(desc, k)) return rc;
  if (!loss || !loss->target.ptr || !loss->loss_sum || !adam) return PBR_E_NULL;
  // the maps are updated in place: a batch-broadcast map (sb == 0) would be written by every material
  if (desc->B > 1 && (desc->albedo.sb == 0 || desc->roughness.sb == 0 || desc->metspec.sb == 0 || (desc->normal.ptr && desc->normal.sb == 0)))
    return PBR_E_SHAPE;
  const PbrPlane* mom[8] = {&adam->m_albedo, &adam->v_albedo, &adam->m_normal, &adam->v_normal,
                            &adam->m_roughness, &adam->v_roughness, &adam->m_metspec, &adam->v_metspec};
  for (int q = 0; q < 4; ++q) {
    const bool need = q != 1 || desc->normal.ptr != nullptr;
    if (need && (!mom[2 * q]->ptr || !mom[2 * q + 1]->ptr)) return PBR_E_NULL;
    k.adam_m[q] = *mom[2 * q]; k.adam_v[q] = *mom[2 * q + 1];
    k.vec_ok = k.vec_ok && plane_vec_ok(k.adam_m[q]) && plane_vec_ok(k.adam_v[q]);
  }
  k.d_intensity = d_intensity;
  k.gsrc = loss->target; k.gsrc_sl = loss->target_sl;
  k.is_loss = 1;
  k.loss_scale = loss->loss_scale; k.loss_sum = loss->loss_sum;
  k.vec_ok = k.vec_ok && plane_vec_ok(loss->target) && (loss->target_sl % kTexels == 0);
  k.adam_on = 1;
  k.adam_project = adam->project;
  k.adam = AdamCoef{adam->step_size, adam->one_minus_beta1, adam->beta2, adam->one_minus_beta2, adam->bias2_sqrt, adam->eps};
  k.force_generic = 1;   // the Adam epilogue lives in the generic kernels (any L)
  return ct_dispatch(k, kernel_workflow(desc), true, (cudaStream_t)stream);
}

static int run_convert(const PbrConvDesc* d, bool m2s, pbr_stream_t stream) {
  if (!d) return PBR_E_NULL;
  if (int rc = check_dims(d->B, d->H, d->W)) return rc;
  if (!d->albedo.ptr || !d->metspec.ptr || !d->out0.ptr || !d->out1.ptr) return PBR_E_NULL;
  if (m2s && d->metallic_channels != 0 && d->metallic_channels != 1 && d->metallic_channels != 3) return PBR_E_CHANNELS;
  ConvKParams k{};
  k.B = d->B; k.H = d->H; k.W = d->W; k.albedo_is_srgb = d->albedo_is_srgb;
  k.met_channels = d->metallic_channels == 3 ? 3 : 1;
  k.albedo = d->albedo; k.metspec = d->metspec; k.out0 = d->out0; k.out1 = d->out1;
  k.vec_ok = plane_vec_ok(d->albedo) && plane_vec_ok(d->metspec) && plane_vec_ok(d->out0) && plane_vec_ok(d->out1);
  dim3 grid, block;
  launch_shape(k.B, k.H, k.W, grid, block);
  if (m2s) convert_kernel<true><<<grid, block, 0, (cudaStream_t)stream>>>(k);
  else convert_kernel<false><<<grid, block, 0, (cudaStream_t)stream>>>(k);
  return launch_result();
}

static int run_convert_backward(const PbrConvDesc* d, const PbrConvGrads* g, bool m2s, pbr_stream_t stream) {
  if (!d || !g) return PBR_E_NULL;
  if (int rc = check_dims(d->B, d->H, d->W)) return rc;
  if (!d->albedo.ptr || !d->metspec.ptr) return PBR_E_NULL;
  if (m2s && d->metallic_channels != 0 && d->metallic_channels != 1 && d->metallic_channels != 3) return PBR_E_CHANNELS;
  ConvKParams k{};
  k.B = d->B; k.H = d->H; k.W = d->W; k.albedo_is_srgb = d->albedo_is_srgb;
  k.met_channels = d->metallic_channels == 3 ? 3 : 1;
  k.albedo = d->albedo; k.metspec = d->metspec;
  k.g0 = g->g_out0; k.g1 = g->g_out1; k.d_albedo = g->d_albedo; k.d_metspec = g->d_metspec;
  k.vec_ok = plane_vec_ok(d->albedo) && plane_vec_ok(d->metspec) && plane_vec_ok(g->g_out0) && plane_vec_ok(g->g_out1) &&
             plane_vec_ok(g->d_albedo) && plane_vec_ok(g->d_metspec);
  dim3 grid, block;
  launch_shape(k.B, k.H, k.W, grid, block);
  if (m2s) convert_bwd_kernel<true><<<grid, block, 0, (cudaStream_t)stream>>>(k);
  else convert_bwd_kernel<false><<<grid, block, 0, (cudaStream_t)stream>>>(k);
  return launch_result();
}

int pbr_convert_m2s(const PbrConvDesc* desc, pbr_stream_t stream) { return run_convert(desc, true, stream); }
int pbr_convert_s2m(const PbrConvDesc* desc, pbr_stream_t stream) { return run_convert(desc, false, stream); }
int pbr_convert_m2s_backward(const PbrConvDesc* desc, const PbrConvGrads* grads, pbr_stream_t stream) { return run_convert_backward(desc, grads, true, stream); }
int pbr_convert_s2m_backward(const PbrConvDesc* desc, const PbrConvGrads* grads, pbr_stream_t stream) { return run_convert_backward(desc, grads, false, stream); }

int pbr_blend(const PbrBlendDesc* d, pbr_stream_t stream) {
  if (!d) return PBR_E_NULL;
  if (int rc = check_dims(d->B, d->H, d->W)) return rc;
  if (d->n_maps < 0) return PBR_E_SHAPE;
  if (d->n_maps > PBR_MAX_BLEND_MAPS) return PBR_E_TOO_MANY;
  if (d->mask_mode < PBR_MASK_GIVEN || d->mask_mode > PBR_MASK_GRADIENT_V) return PBR_E_ENUM;
  if (d->mask_mode == PBR_MASK_GIVEN && !d->mask.ptr) return PBR_E_NULL;
  if (d->mask_mode == PBR_MASK_SIGMOID && (!d->prop1.ptr || !d->prop2.ptr)) return PBR_E_NULL;
  BlendKParams k{};
  k.d = *d;
  bool vec = plane_vec_ok(d->mask) && plane_vec_ok(d->prop1) && plane_vec_ok(d->prop2) && plane_vec_ok(d->mask_out);
  if (d->mask_mode != PBR_MASK_GIVEN) k.d.mask.ptr = nullptr;
  for (int m = 0; m < d->n_maps; ++m) {
    const PbrBlendMap& bm = d->maps[m];
    if (!bm.a.ptr || !bm.b.ptr || !bm.out.ptr) return PBR_E_NULL;
    if (bm.channels < 1 || bm.channels > 4 || (bm.is_normal && bm.channels != 3)) return PBR_E_CHANNELS;
    vec = vec && plane_vec_ok(bm.a) && plane_vec_ok(bm.b) && plane_vec_ok(bm.out);
  }
  k.vec_ok = vec;
  k.width_eps = d->blend_width + 1e-6f;
  if (d->mask_mode == PBR_MASK_GRADIENT_H) k.grad = make_linspace(0.0f, 1.0f, d->W);
  if (d->mask_mode == PBR_MASK_GRADIENT_V) k.grad = make_linspace(0.0f, 1.0f, d->H);
  dim3 grid, block;
  launch_shape(d->B, d->H, d->W, grid, block);
  blend_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(k);
  return launch_result();
}

int pbr_blend_backward(const PbrBlendDesc* d, const PbrBlendGrads* g, pbr_stream_t stream) {
  if (!d || !g) return PBR_E_NULL;
  if (int rc = check_dims(d->B, d->H, d->W)) return rc;
  if (d->n_maps < 0) return PBR_E_SHAPE;
  if (d->n_maps > PBR_MAX_BLEND_MAPS) return PBR_E_TOO_MANY;
  if (d->mask_mode < PBR_MASK_GIVEN || d->mask_mode > PBR_MASK_GRADIENT_V) return PBR_E_ENUM;
  if (!g->mask.ptr) return PBR_E_NULL;
  BlendBwdKParams k{};
  k.d = *d;
  k.g = *g;
  bool vec = plane_vec_ok(g->mask) && plane_vec_ok(g->g_mask_out) && plane_vec_ok(g->d_mask) && plane_vec_ok(g->d_prop1) && plane_vec_ok(g->d_prop2);
  for (int m = 0; m < d->n_maps; ++m) {
    const PbrBlendMap& bm = d->maps[m];
    if (!bm.a.ptr || !bm.b.ptr) return PBR_E_NULL;
    if (bm.channels < 1 || bm.channels > 4 || (bm.is_normal && bm.channels != 3)) return PBR_E_CHANNELS;
    vec = vec && plane_vec_ok(bm.a) && plane_vec_ok(bm.b) && plane_vec_ok(g->maps[m].g_out) && plane_vec_ok(g->maps[m].d_a) && plane_vec_ok(g->maps[m].d_b);
  }
  k.vec_ok = vec;
  k.width_eps = d->blend_width + 1e-6f;
  k.need_dmask = (d->mask_mode == PBR_MASK_GIVEN && g->d_mask.ptr) || (d->mask_mode == PBR_MASK_SIGMOID && (g->d_prop1.ptr || g->d_prop2.ptr));
  dim3 grid, block;
  launch_shape(d->B, d->H, d->W, grid, block);
  blend_bwd_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(k);
  return launch_result();
}

int pbr_color_convert(const PbrColorDesc* d, pbr_stream_t stream) {
  if (!d) return PBR_E_NULL;
  if (int rc = check_dims(d->B, d->H, d->W)) return rc;
  if (d->C < 1) return PBR_E_CHANNELS;
  if (!d->in.ptr || !d->out.ptr) return PBR_E_NULL;
  ColorKParams k{};
  k.B = d->B; k.C = d->C; k.H = d->H; k.W = d->W; k.to_linear = d->to_linear;
  k.in = d->in; k.out = d->out;
  k.vec_ok = plane_vec_ok(d->in) && plane_vec_ok(d->out);
  dim3 grid, block;
  launch_shape(k.B, k.H, k.W, grid, block);
  color_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(k);
  return launch_result();
}

static int fill_normal(const PbrNormalDesc* d, NormalKParams& k, bool need_out) {
  if (!d) return PBR_E_NULL;
  if (int rc = check_dims(d->B, d->H, d->W)) return rc;
  if (d->channels != 2 && d->channels != 3) return PBR_E_CHANNELS;
  if (!d->in.ptr || (need_out && !d->out.ptr)) return PBR_E_NULL;
  k.B = d->B; k.H = d->H; k.W = d->W; k.channels = d->channels;
  k.in = d->in; k.out = d->out;
  k.vec_ok = plane_vec_ok(d->in) && (!need_out || plane_vec_ok(d->out));
  return PBR_OK;
}

int pbr_normal_min(const PbrNormalDesc* d, float* result, pbr_stream_t stream) {
  NormalKParams k{};
  if (int rc = fill_normal(d, k, false)) return rc;
  if (!result) return PBR_E_NULL;
  k.result = result;
  dim3 grid, block;
  launch_shape(k.B, k.H, k.W, grid, block);
  normal_min_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(k);
  return launch_result();
}

int pbr_normal_ingest(const PbrNormalDesc* d, pbr_stream_t stream) {
  NormalKParams k{};
  if (int rc = fill_normal(d, k, true)) return rc;
  if (d->channels == 2 && d->in.ptr == d->out.ptr) return PBR_E_NULL;   // 2 -> 3 channels cannot run in place
  k.cond_min = d->cond_min;
  dim3 grid, block;
  launch_shape(k.B, k.H, k.W, grid, block);
  normal_ingest_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(k);
  return launch_result();
}

int pbr_normal_ingest_backward(const PbrNormalDesc* d, const PbrNormalGrads* g, pbr_stream_t stream) {
  NormalKParams k{};
  if (int rc = fill_normal(d, k, false)) return rc;
  if (!g || !g->g_out.ptr || !g->d_in.ptr) return PBR_E_NULL;
  k.g_out = g->g_out; k.d_in = g->d_in;
  k.vec_ok = k.vec_ok && plane_vec_ok(g->g_out) && plane_vec_ok(g->d_in);
  dim3 grid, block;
  launch_shape(k.B, k.H, k.W, grid, block);
  normal_ingest_bwd_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(k);
  return launch_result();
}

int pbr_ingest_image(const PbrIngestDesc* d, pbr_stream_t stream) {
  if (!d) return PBR_E_NULL;
  if (int rc = check_dims(d->B, d->H, d->W)) return rc;
  if (d->bits != 8 && d->bits != 16) return PBR_E_ENUM;
  if (d->mode < PBR_INGEST_PLAIN || d->mode > PBR_INGEST_NORMAL2) return PBR_E_ENUM;
  if (d->src_channels < 1 || d->src_channels > 4) return PBR_E_CHANNELS;
  const int need = d->mode == PBR_INGEST_NORMAL3 ? 3 : (d->mode == PBR_INGEST_NORMAL2 ? 2 : d->channels);
  if (need < 1 || need > d->src_channels) return PBR_E_CHANNELS;
  if (!d->src || !d->out.ptr) return PBR_E_NULL;
  IngestKParams k{};
  k.d = *d;
  k.vec_ok = plane_vec_ok(d->out);
  k.src_words_ok = (reinterpret_cast<uintptr_t>(d->src) % 4 == 0) && (d->src_row_stride % 4 == 0) && (d->src_batch_stride % 4 == 0);
  dim3 grid, block;
  launch_shape(d->B, d->H, d->W, grid, block);
  cudaStream_t st = (cudaStream_t)stream;
  switch (d->src_channels * 2 + (d->bits == 16)) {
    case 2: ingest_kernel<1, 8><<<grid, block, 0, st>>>(k); break;
    case 3: ingest_kernel<1, 16><<<grid, block, 0, st>>>(k); break;
    case 4: ingest_kernel<2, 8><<<grid, block, 0, st>>>(k); break;
    case 5: ingest_kernel<2, 16><<<grid, block, 0, st>>>(k); break;
    case 6: ingest_kernel<3, 8><<<grid, block, 0, st>>>(k); break;
    case 7: ingest_kernel<3, 16><<<grid, block, 0, st>>>(k); break;
    case 8: ingest_kernel<4, 8><<<grid, block, 0, st>>>(k); break;
    default: ingest_kernel<4, 16><<<grid, block, 0, st>>>(k); break;
  }
  return launch_result();
}

int pbr_index_transform(const PbrIndexDesc* d, pbr_stream_t stream) {
  if (!d) return PBR_E_NULL;
  if (int rc = check_dims(d->B, d->H_out, d->W_out)) return rc;
  if (d->H_in < 1 || d->W_in < 1) return PBR_E_SHAPE;
  if ((d->step_y != 1 && d->step_y != -1) || (d->step_x != 1 && d->step_x != -1)) return PBR_E_ENUM;
  if (d->n_maps < 0) return PBR_E_SHAPE;
  if (d->n_maps > PBR_MAX_INDEX_MAPS) return PBR_E_TOO_MANY;
  if (d->reduce_y < 0 || d->reduce_x < 0 || d->reduce_y > 4096 || d->reduce_x > 4096) return PBR_E_SHAPE;
  IndexKParams k{};
  k.d = *d;
  bool vec = true;
  for (int m = 0; m < d->n_maps; ++m) {
    const PbrIndexMap& im = d->maps[m];
    if (!im.in.ptr || !im.out.ptr) return PBR_E_NULL;
    if (im.channels < 1 || im.channels > 4) return PBR_E_CHANNELS;
    vec = vec && plane_vec_ok(im.out);
  }
  k.vec_ok = vec;
  dim3 grid, block;
  launch_shape(d->B, d->H_out, d->W_out, grid, block);
  index_transform_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(k);
  return launch_result();
}

int pbr_adam_step(const PbrAdamDesc* d, pbr_stream_t stream) {
  if (!d) return PBR_E_NULL;
  if (int rc = check_dims(d->B, d->H, d->W)) return rc;
  if (d->n_maps < 0) return PBR_E_SHAPE;
  if (d->n_maps > PBR_MAX_ADAM_MAPS) return PBR_E_TOO_MANY;
  AdamKParams k{};
  k.d = *d;
  bool vec = true;
  for (int m = 0; m < d->n_maps; ++m) {
    const PbrAdamMap& am = d->maps[m];
    if (!am.param.ptr || !am.grad.ptr || !am.exp_avg.ptr || !am.exp_avg_sq.ptr) return PBR_E_NULL;
    if (am.channels < 1 || am.channels > 4) return PBR_E_CHANNELS;
    if (am.project < PBR_PROJECT_NONE || am.project > PBR_PROJECT_NORMALIZE) return PBR_E_ENUM;
    if (am.project == PBR_PROJECT_NORMALIZE && am.channels != 3) return PBR_E_CHANNELS;
    vec = vec && plane_vec_ok(am.param) && plane_vec_ok(am.grad) && plane_vec_ok(am.exp_avg) && plane_vec_ok(am.exp_avg_sq);
  }
  k.vec_ok = vec;
  dim3 grid, block;
  launch_shape(d->B, d->H, d->W, grid, block);
  adam_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(k);
  return launch_result();
}

int pbr_normal_op(const PbrNormalOpDesc* d, pbr_stream_t stream) {
  if (!d) return PBR_E_NULL;
  if (int rc = check_dims(d->B, d->H, d->W)) return rc;
  if (d->op < PBR_NORMAL_OP_ROTATE || d->op > PBR_NORMAL_OP_DIVERGENCE_BWD) return PBR_E_ENUM;
  if (!d->in.ptr || !d->out.ptr) return PBR_E_NULL;
  const bool adjoint = d->op == PBR_NORMAL_OP_FROM_HEIGHT_BWD || d->op == PBR_NORMAL_OP_ROTATE_BWD || d->op == PBR_NORMAL_OP_DIVERGENCE_BWD;
  if (adjoint && (!d->aux.ptr || d->aux.ptr == d->out.ptr)) return PBR_E_NULL;
  if (d->op != PBR_NORMAL_OP_ROTATE && d->in.ptr == d->out.ptr) return PBR_E_NULL;   // a stencil / an adjoint cannot run in place
  NormalOpKParams k{};
  k.d = *d;
  const bool row_loads = d->op == PBR_NORMAL_OP_ROTATE || d->op == PBR_NORMAL_OP_ROTATE_BWD || d->op == PBR_NORMAL_OP_DIVERGENCE_BWD;
  k.vec_ok = plane_vec_ok(d->out) && (!row_loads || plane_vec_ok(d->in)) && (d->op != PBR_NORMAL_OP_ROTATE_BWD || plane_vec_ok(d->aux));
  dim3 grid, block;
  launch_shape(d->B, d->H, d->W, grid, block);
  normal_op_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(k);
  return launch_result();
}

}  // extern "C"
#endif   // PBR_MAIN_PART
