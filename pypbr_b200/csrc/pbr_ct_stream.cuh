// pbr_ct_stream.cuh — the streamed (TMA-fed) Cook-Torrance kernels: the fast path of
// pbr_ct_forward / pbr_ct_backward / pbr_ct_loss_fwd_bwd for ONE light (L == 1) on 16-byte aligned,
// W % 4 == 0 maps.  Included by pbr_kernels.cu after the generic kernels.
//
// Why: the shading math costs a few hundred instructions per texel, so a thread that issues its own
// global loads and then computes keeps too few bytes in flight at the occupancy the register budget
// allows (ncu: 24 % warps active, 64 % issue-slot use, 55 % of HBM peak for the generic backward).
// Here the copy engine does the loading:
//
//   tile    = blockDim.y rows x (blockDim.x * kST) texels of ONE material: every input plane of the tile
//             (albedo x3, roughness, metallic | specular, normal x3, and grad_out | target x3 for the
//             backward) is kTileFloats contiguous floats of shared memory per stage, in image order;
//   producer= every warp for itself (per-warp pipelines): a warp owns 32 x kST contiguous texels
//             of the tile row, i.e. one cp.async.bulk of 512 B per plane and stage, completion counted in bytes on the
//             warp's own mbarrier (pbr_async.cuh); right after it has read a stage into registers one lane per plane
//             re-arms the barrier and issues the copies of the tile kStages ahead.  No cross-warp synchronisation at all.
//   consumer= all threads.  A thread owns kSSlots lane-values (texel pairs) of one tile row, INTERLEAVED
//             with the other threads of the row: slot j of thread tx covers the texels
//             j*(bx*kLanes) + tx*kLanes ... + kLanes-1 of the row.  So one warp-level LDS.64 / STG.64
//             touches 256 contiguous bytes: no shared-memory bank conflicts, full 32-byte sectors on
//             the way out.  The forward kernel shades all of a thread's slots together (ILP); the
//             backward takes them one at a time - inputs come out of the stage right before they are
//             used and the gradients leave right after, so only one pair's working set is live in
//             registers (the adjoint needs ~170 of them).  No CTA-wide barrier in the loop.
//
// A CTA walks over `mats_per_cta` materials at a fixed image position, so for a point light the
// per-texel light geometry (material independent) is computed once and reused - as in the generic
// kernels - and the pipeline stays full for the whole walk.
//
// Measured floor of this data-movement design with the shading math compiled out (a debug build, DESIGN §3.1):
// 6.4-6.6 TB/s forward and backward, i.e. 98-100 % of the measured copy peak;
// whatever the real kernels lose against that is instruction issue, not memory.  With the kFast flavour (below) they
// lose almost nothing: forward 0.446-0.451 ms (100 %), backward 0.783-0.807 ms (96-99 %) at 64 x 1024^2.
#pragma once

#include "pbr_async.cuh"

namespace pbr {

constexpr int kStages = 2;
constexpr int kStreamThreads = 128;
constexpr int kST = 4;   // texels per thread: two packed pairs
constexpr int kStreamFwdMinCtas = 4;   // 128 registers
constexpr int kStreamBwdMinCtas = 3;   // 168 registers
static_assert(kST % kLanes == 0, "stream kernels: whole lane-values per thread");
constexpr int kSSlots = kST / kLanes;               // lane-values per thread
constexpr int kTileFloats = kStreamThreads * kST;   // floats of one plane in one stage (2 KB at 128 threads x 4 texels)
// Per-warp pipelines: every warp runs its OWN copy pipeline over its own 32 x kST texels of a tile row (plane stride
// inside a stage = one warp segment) instead of warp 0 feeding the whole CTA: a warp refills a stage right after its own
// last read of it, without waiting for the other warps or for its own arithmetic.
// Measured (C2 shape, bare C ABI): forward 0.499 -> 0.474 ms (95 % of the HBM copy peak).  The backward used to be
// 1.5 % slower that way (0.944 -> 0.959 ms): the per-warp issue of 11 small copies per tile cost what the decoupling gave.
// With the kFast flavour (below) the balance flips - CTA-level 0.852 ms, per-warp 0.807 ms at 64 x 1024^2
// (profiles/r2_tune_c2_kfast_variants.json) - so both kernels run per-warp pipelines.  Deeper pipelines (3, 4 stages) are
// slower in both, and so were a backward that refills after the whole tile instead of after its last read (0.808 ms) and
// a CTA-level backward in which the warp that reads a stage last refills it (0.860 ms; DESIGN §3.1).
constexpr int kWarpSeg = 32 * kST;                  // floats of one plane a warp owns per tile row = floats between two planes of a stage
constexpr int kPipes = kStreamThreads / 32;         // independent copy pipelines per CTA
constexpr int kMaxSrcPlanes = 13;                   // albedo 3 + roughness 1 + metallic|specular 3 + normal 3 + grad_out|target 3

// backward flavours (compile-time, so the plain backward carries no reduction code)
constexpr int kModeLoss = 1;      // gsrc is the target image: grad_out = 2*scale*(render - target), loss reduced
constexpr int kModeIntGrad = 2;   // reduce d loss / d light intensity

struct StreamSrc {
  const float* base;   // plane pointer at (b = 0, channel, first row of the tile, first column of the tile)
  int64_t sb, sh;      // batch and row strides in elements
  int slot;            // plane slot inside a stage buffer
  int pad;
};

struct StreamShared {
  uint64_t full[kStages * kPipes];   // producer -> consumers: the copies of the stage have landed (transaction bytes)
  StreamSrc src[kMaxSrcPlanes];
  int n_src;
};

// plane slots of a stage: fixed at compile time so that the consumer's LDS use immediate offsets
template <int WF, bool kBwd>
struct Slots {
  static constexpr int mc = WF == 0 ? 1 : 3;
  static constexpr int albedo = 0, rough = 3, met = 4;
  static constexpr int gsrc = 4 + mc;                       // backward only
  static constexpr int normal = kBwd ? 7 + mc : 4 + mc;     // last, so a missing normal map shortens the stage
  static constexpr int count_no_normal = normal;
  static constexpr int count = normal + 3;
};

template <int WF, bool kBwd>
__device__ __forceinline__ void stream_build_table(const CtKParams& p, int row0, int col0, StreamShared& sh) {
  using SL = Slots<WF, kBwd>;
  int n = 0;
  auto add = [&](const PbrPlane& pl, int c, int slot) {
    sh.src[n].base = pl.ptr + (int64_t)c * pl.sc + (int64_t)row0 * pl.sh + col0;
    sh.src[n].sb = pl.sb;
    sh.src[n].sh = pl.sh;
    sh.src[n].slot = slot;
    ++n;
  };
  for (int c = 0; c < 3; ++c) add(p.albedo, c, SL::albedo + c);
  add(p.roughness, 0, SL::rough);
  for (int c = 0; c < SL::mc; ++c) add(p.metspec, c, SL::met + c);
  if (kBwd)
    for (int c = 0; c < 3; ++c) add(p.gsrc, c, SL::gsrc + c);
  if (p.normal.ptr)
    for (int c = 0; c < 3; ++c) add(p.normal, c, SL::normal + c);
  sh.n_src = n;
}

// per-warp pipeline: the calling warp enqueues ITS segment (32 x kST texels of its row) of every plane of material `b`
__device__ __forceinline__ void warp_issue(const StreamShared& sh, uint64_t* bar, float* stage, int b, int64_t row_in_tile,
                                           int col_in_tile, int seg_bytes, uint64_t policy) {
  const int lane = threadIdx.x & 31;
  if (lane == 0) mbar_arrive_expect_tx(bar, (uint32_t)(sh.n_src * seg_bytes));
  __syncwarp();
  if (lane < sh.n_src) {
    const StreamSrc& s = sh.src[lane];
    bulk_g2s(stage + s.slot * kWarpSeg, s.base + (int64_t)b * s.sb + row_in_tile * s.sh + col_in_tile, (uint32_t)seg_bytes, bar,
             policy);
  }
}
// orders this thread's earlier shared-memory reads before copies the async proxy performs later
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// one lane-value (kLanes consecutive floats) from shared memory / to global memory
__device__ __forceinline__ V lds_v(const float* p) {
  const float2 v = *reinterpret_cast<const float2*>(p);
  return V{v.x, v.y};
}
__device__ __forceinline__ void stg_v(float* p, V v) { __stcs(reinterpret_cast<float2*>(p), make_float2(v.x, v.y)); }

// Geometry of the tile this CTA owns and of the thread inside it.
struct StreamWhere {
  int row0, col0;       // tile origin
  int row, col;         // this thread's row and the first texel of its slot 0
  int slot_stride;      // texels between a thread's consecutive slots (= 32 * kLanes)
  int toff;             // offset of slot 0 inside the warp's segment of a plane (floats)
  int seg_bytes;        // bytes of the warp's segment of one plane row (0: the warp has nothing to copy or shade)
  int wcol;             // offset of the warp's segment inside the tile row
  bool row_ok;
};
// blockDim.x is a multiple of 32: a warp sits inside one tile row and owns kWarpSeg contiguous texels of it
__device__ __forceinline__ StreamWhere stream_locate(int H, int W) {
  StreamWhere w;
  const int lane = threadIdx.x & 31;
  w.row0 = blockIdx.y * blockDim.y;
  w.col0 = blockIdx.x * (blockDim.x * kST);
  w.row = w.row0 + threadIdx.y;
  w.row_ok = w.row < H;
  w.wcol = (threadIdx.x >> 5) * kWarpSeg;           // first texel of the warp's segment inside the tile row
  w.slot_stride = 32 * kLanes;
  w.col = w.col0 + w.wcol + lane * kLanes;
  w.toff = lane * kLanes;
  const int left = W - (w.col0 + w.wcol);
  w.seg_bytes = (w.row_ok && left > 0) ? min(kWarpSeg, left) * 4 : 0;
  return w;
}
// kFast flavour of the streamed kernels (round 2).  The host picks it when the launch is the plain case: blockDim = (kStreamThreads, 1),
// every tile full (W % (kStreamThreads * kST) == 0), a normal map, the reference's default colour handling (sRGB albedo /
// specular in, sRGB out: compile-time flags, forward tile loop 644 -> 500 instructions) and - in the backward - all four
// gradient planes requested.
// Then the tile geometry is compile-time (immediate LDS / STG offsets), no slot or output is ever inactive, and the loop
// carries no null checks: ncu had ~215 of the backward's 1172 instructions per tile and warp on index rematerialisation
// (S2R, LDC, IMAD), predicates on the output pointers and 64-bit address rebuilds; a lean loop needs ~65.
// Measured at 64 x 1024^2 (bare C ABI): backward 0.923 -> 0.852 ms (586 M -> 519 M warp-instructions), with per-warp
// pipelines 0.807 ms = 96 % of the measured copy peak (floor with the math compiled out: 0.775 ms); forward
// 0.461 -> 0.446 ms = the copy peak.
__device__ __forceinline__ StreamWhere stream_locate_fast() {
  StreamWhere w;
  const int lane = threadIdx.x & 31;
  w.row0 = blockIdx.y;
  w.col0 = blockIdx.x * kTileFloats;
  w.row = w.row0;
  w.row_ok = true;
  w.wcol = (threadIdx.x >> 5) * kWarpSeg;
  w.slot_stride = 32 * kLanes;
  w.col = w.col0 + w.wcol + lane * kLanes;
  w.toff = lane * kLanes;
  w.seg_bytes = kWarpSeg * 4;
  return w;
}
// kFast also fixes the colour handling to the reference's defaults (sRGB albedo / specular in, sRGB out), which the host checks
template <bool kFast>
__device__ __forceinline__ CtFlags stream_flags(const CtFlags& f) {
  CtFlags F = f;
  if (kFast) { F.albedo_is_srgb = true; F.specular_is_srgb = true; F.return_srgb = true; F.per_light = false; F.L = 1; }
  return F;
}
// W % 4 == 0 (and kLanes <= 2): a slot's texels are all inside or all outside the image
__device__ __forceinline__ bool slot_active(const StreamWhere& w, int j, int W) { return w.row_ok && w.col + j * w.slot_stride < W; }

template <int kLight>
__device__ __forceinline__ void stream_coords(const CtStage& S, const StreamWhere& w, int W, V (&x)[kSSlots], float& y,
                                              LightGeomT<V> (&hg)[kSSlots]) {
  const int row = w.row_ok ? w.row : 0;
#pragma unroll
  for (int j = 0; j < kSSlots; ++j)
#pragma unroll
    for (int k = 0; k < kLanes; ++k) {
      const int col = w.col + j * w.slot_stride + k;
      lane_set(x[j], k, linspace_at(S.lsx, col < W ? col : W - 1));
    }
  y = linspace_at(S.lsy, row);
  if (kLight == kLightPointHoisted) {
#pragma unroll
    for (int j = 0; j < kSSlots; ++j)
      point_light_geom(S.light[0].p[0], S.light[0].p[1], S.light[0].p[2], x[j], y, S.vx, S.vy, S.vz, hg[j]);
  }
}

// ------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------
template <int WF, int kLight, bool kFast = false>
__global__ void __launch_bounds__(kStreamThreads, kStreamFwdMinCtas) ct_forward_stream(const __grid_constant__ CtKParams p) {
  using SL = Slots<WF, false>;
  constexpr int G = kSSlots;   // all of the thread's pairs are shaded together
  extern __shared__ __align__(128) float stream_smem[];
  __shared__ CtStage S;
  __shared__ StreamShared sh;
  const int tid = kFast ? threadIdx.x : threadIdx.y * blockDim.x + threadIdx.x;
  const StreamWhere w = kFast ? stream_locate_fast() : stream_locate(p.H, p.W);
  const int row_in_tile = kFast ? 0 : threadIdx.y;
  if (tid == 0) {
    stream_build_table<WF, false>(p, w.row0, w.col0, sh);
#pragma unroll
    for (int s = 0; s < kStages * kPipes; ++s) mbar_init(&sh.full[s], 1);
    mbar_init_fence();
  }
  stage_params<false>(p, S);  // ends with __syncthreads()  (never shades per-material parameters)

  const int b0 = blockIdx.z * p.mats_per_cta;
  const int ntiles = min(b0 + p.mats_per_cta, p.B) - b0;
  const int stage_floats = ((kFast || p.normal.ptr) ? SL::count : SL::count_no_normal) * kTileFloats;
  // this warp's barriers and stage buffers (planes x kWarpSeg floats per stage)
  const int pipe = tid >> 5;
  uint64_t* const full = sh.full + pipe * kStages;
  float* const my_stages = stream_smem + pipe * kStages * (stage_floats / (kTileFloats / kWarpSeg));
  const int my_stage_floats = stage_floats / (kTileFloats / kWarpSeg);
  const uint64_t policy = l2_evict_first_policy();
  if (w.seg_bytes > 0)
    for (int k = 0; k < kStages && k < ntiles; ++k)
      warp_issue(sh, &full[k], my_stages + k * my_stage_floats, b0 + k, row_in_tile, w.wcol, w.seg_bytes, policy);

  V x[kSSlots];
  float y;
  LightGeomT<V> hg[kSSlots];
  stream_coords<kLight>(S, w, p.W, x, y, hg);
  const bool has_normal = kFast || p.normal.ptr != nullptr;
  bool act[kSSlots];
  bool any = false;
#pragma unroll
  for (int j = 0; j < kSSlots; ++j) { act[j] = kFast || slot_active(w, j, p.W); any = any || act[j]; }
  // output pointer of material b0 at slot 0; advanced by one batch stride per tile (strides sit in the
  // __grid_constant__ parameter block, i.e. the constant bank)
  float* o = p.out.ptr + ((int64_t)b0 * p.out.sb + (int64_t)w.row * p.out.sh + w.col);

  for (int k = 0; k < ntiles; ++k) {
    const int s = k % kStages;
    const float* st = my_stages + s * my_stage_floats + w.toff;
    if (w.seg_bytes > 0) mbar_wait(&full[s], (k / kStages) & 1);
    V a[3][G], n[3][G], r[G], m[3][G];
#pragma unroll
    for (int j = 0; j < G; ++j) {
      const float* sj = st + j * w.slot_stride;
#pragma unroll
      for (int c = 0; c < 3; ++c) a[c][j] = lds_v(sj + (SL::albedo + c) * kWarpSeg);
      r[j] = lds_v(sj + SL::rough * kWarpSeg);
#pragma unroll
      for (int c = 0; c < 3; ++c) m[c][j] = c < SL::mc ? lds_v(sj + (SL::met + c) * kWarpSeg) : splat<V>(0.0f);
#pragma unroll
      for (int c = 0; c < 3; ++c) n[c][j] = has_normal ? lds_v(sj + (SL::normal + c) * kWarpSeg) : splat<V>(c == 2 ? 1.0f : 0.0f);
    }
    // this warp holds its texels in registers: refill its own stage (no CTA-wide barrier - warps drift freely)
    __syncwarp();
    if (w.seg_bytes > 0 && k + kStages < ntiles) {
      fence_proxy_async();
      warp_issue(sh, &full[s], my_stages + s * my_stage_floats, b0 + k + kStages, row_in_tile, w.wcol, w.seg_bytes, policy);
    }
    if (any) {
      V outv[3][G];
      auto emit = [&](int, const V(&v)[3][G]) {
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
          for (int j = 0; j < G; ++j) outv[c][j] = v[c][j];
      };
      ct_forward_group<WF, kLight, V, G>(S, stream_flags<kFast>(p.flags), a, n, r, m, x, y, hg, emit);
#pragma unroll
      for (int j = 0; j < G; ++j)
        if (act[j]) {
#pragma unroll
          for (int c = 0; c < 3; ++c) stg_v(o + c * p.out.sc + j * w.slot_stride, outv[c][j]);
        }
    }
    o += p.out.sb;
  }
}

// ------------------------------------------------------------------------------------------------
// backward / fused loss
// ------------------------------------------------------------------------------------------------
template <int WF, int kLight, int kMode, bool kFast = false>
__global__ void __launch_bounds__(kStreamThreads, kStreamBwdMinCtas) ct_backward_stream(const __grid_constant__ CtKParams p) {
  using SL = Slots<WF, true>;
  constexpr bool kLoss = (kMode & kModeLoss) != 0;
  constexpr bool kIntGrad = (kMode & kModeIntGrad) != 0;
  extern __shared__ __align__(128) float stream_smem[];
  __shared__ CtStage S;
  __shared__ StreamShared sh;
  __shared__ float s_red[kStreamThreads / 32][4];
  const int tid = kFast ? threadIdx.x : threadIdx.y * blockDim.x + threadIdx.x;
  const StreamWhere w = kFast ? stream_locate_fast() : stream_locate(p.H, p.W);
  if (tid == 0) {
    stream_build_table<WF, true>(p, w.row0, w.col0, sh);
#pragma unroll
    for (int s = 0; s < kStages * kPipes; ++s) mbar_init(&sh.full[s], 1);
    mbar_init_fence();
  }
  stage_params<false>(p, S);  // ends with __syncthreads()  (never shades per-material parameters)

  const int b0 = blockIdx.z * p.mats_per_cta;
  const int ntiles = min(b0 + p.mats_per_cta, p.B) - b0;
  const int stage_floats = ((kFast || p.normal.ptr) ? SL::count : SL::count_no_normal) * kTileFloats;
  // this warp's barriers and stage buffers (planes x kWarpSeg floats per stage)
  const int pipe = tid >> 5;
  uint64_t* const full = sh.full + pipe * kStages;
  float* const my_stages = stream_smem + pipe * kStages * (stage_floats / (kTileFloats / kWarpSeg));
  const int my_stage_floats = stage_floats / (kTileFloats / kWarpSeg);
  const int row_in_tile = kFast ? 0 : threadIdx.y;
  const uint64_t policy = l2_evict_first_policy();
  if (w.seg_bytes > 0)
    for (int k = 0; k < kStages && k < ntiles; ++k)
      warp_issue(sh, &full[k], my_stages + k * my_stage_floats, b0 + k, row_in_tile, w.wcol, w.seg_bytes, policy);

  V x[kSSlots];
  float y;
  LightGeomT<V> hg[kSSlots];
  stream_coords<kLight>(S, w, p.W, x, y, hg);
  const bool has_normal = kFast || p.normal.ptr != nullptr;
  // gradient pointers of material b0 at slot 0; advanced by one batch stride per tile
  float* o_a = (kFast || p.d_albedo.ptr) ? p.d_albedo.ptr + ((int64_t)b0 * p.d_albedo.sb + (int64_t)w.row * p.d_albedo.sh + w.col) : nullptr;
  float* o_n = (kFast || (has_normal && p.d_normal.ptr)) ? p.d_normal.ptr + ((int64_t)b0 * p.d_normal.sb + (int64_t)w.row * p.d_normal.sh + w.col) : nullptr;
  float* o_r = (kFast || p.d_roughness.ptr) ? p.d_roughness.ptr + ((int64_t)b0 * p.d_roughness.sb + (int64_t)w.row * p.d_roughness.sh + w.col) : nullptr;
  float* o_m = (kFast || p.d_metspec.ptr) ? p.d_metspec.ptr + ((int64_t)b0 * p.d_metspec.sb + (int64_t)w.row * p.d_metspec.sh + w.col) : nullptr;
  V loss_pair = splat<V>(0.0f);
  float gi_local[3] = {0.0f, 0.0f, 0.0f};

  for (int k = 0; k < ntiles; ++k) {
    const int s = k % kStages;
    const float* st = my_stages + s * my_stage_floats + w.toff;
    if (w.seg_bytes > 0) mbar_wait(&full[s], (k / kStages) & 1);
#pragma unroll
    for (int j = 0; j < kSSlots; ++j) {
      const float* sj = st + j * w.slot_stride;
      V a[3][1], n[3][1], r[1], m[3][1], gs[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) a[c][0] = lds_v(sj + (SL::albedo + c) * kWarpSeg);
      r[0] = lds_v(sj + SL::rough * kWarpSeg);
#pragma unroll
      for (int c = 0; c < 3; ++c) m[c][0] = c < SL::mc ? lds_v(sj + (SL::met + c) * kWarpSeg) : splat<V>(0.0f);
#pragma unroll
      for (int c = 0; c < 3; ++c) gs[c] = lds_v(sj + (SL::gsrc + c) * kWarpSeg);   // grad_out, or the target image in loss mode
#pragma unroll
      for (int c = 0; c < 3; ++c) n[c][0] = has_normal ? lds_v(sj + (SL::normal + c) * kWarpSeg) : splat<V>(c == 2 ? 1.0f : 0.0f);
      if (j == kSSlots - 1) {
        // last read of the stage by this warp: refill it (no CTA-wide barrier - warps drift freely)
        __syncwarp();
        if (w.seg_bytes > 0 && k + kStages < ntiles) {
          fence_proxy_async();
          warp_issue(sh, &full[s], my_stages + s * my_stage_floats, b0 + k + kStages, row_in_tile, w.wcol, w.seg_bytes, policy);
        }
      }
      if (kFast || slot_active(w, j, p.W)) {
        const V xs[1] = {x[j]};
        const LightGeomT<V> hgs[1] = {hg[j]};
        auto gout = [&](int, const V(&outv)[3][1], V(&g)[3][1]) {
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            if (kLoss) {
              const V diff = outv[c][0] - gs[c];
              loss_pair = loss_pair + diff * diff;
              g[c][0] = (2.0f * p.loss_scale) * diff;
            } else {
              g[c][0] = gs[c];
            }
          }
        };
        auto int_sink = [&](int, const float(&gi)[3]) {
          if (kIntGrad) {
#pragma unroll
            for (int c = 0; c < 3; ++c) gi_local[c] += gi[c];
          }
        };
        V da[3][1], dn[3][1], dr[1], dm[3][1];
        ct_backward_group<WF, kLight, V, 1>(S, stream_flags<kFast>(p.flags), a, n, r, m, xs, y, hgs, gout, int_sink, da, dn, dr, dm, NoFetch(), GeomCache<V>(),
                                            NoGeomSink(), NoSavedOut(), kIntGrad);
        const int jo = j * w.slot_stride;
        if (kFast || o_a) {
#pragma unroll
          for (int c = 0; c < 3; ++c) stg_v(o_a + c * p.d_albedo.sc + jo, da[c][0]);
        }
        if (kFast || o_n) {
#pragma unroll
          for (int c = 0; c < 3; ++c) stg_v(o_n + c * p.d_normal.sc + jo, dn[c][0]);
        }
        if (kFast || o_r) stg_v(o_r + jo, dr[0]);
        if (kFast || o_m) {
#pragma unroll
          for (int c = 0; c < SL::mc; ++c) stg_v(o_m + c * p.d_metspec.sc + jo, dm[c][0]);
        }
      }
    }
    if (kFast || o_a) o_a += p.d_albedo.sb;
    if (kFast || o_n) o_n += p.d_normal.sb;
    if (kFast || o_r) o_r += p.d_roughness.sb;
    if (kFast || o_m) o_m += p.d_metspec.sb;
  }

  // CTA-level reductions: warp shuffle -> shared -> ONE atomic per CTA and value
  if (kLoss || kIntGrad) {
    float v[4] = {kLoss ? lane_sum(loss_pair) : 0.0f, gi_local[0], gi_local[1], gi_local[2]};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if ((j == 0 && !kLoss) || (j > 0 && !kIntGrad)) continue;
      float sum = warp_sum(v[j]);
      if ((tid & 31) == 0) s_red[tid >> 5][j] = sum;
    }
    __syncthreads();
    if (tid < 4 && ((tid == 0 && kLoss) || (tid > 0 && kIntGrad))) {
      float sum = 0.0f;
#pragma unroll
      for (int i = 0; i < kStreamThreads / 32; ++i) sum += s_red[i][tid];
      if (tid == 0) atomicAdd(p.loss_sum, sum);
      else atomicAdd(&p.d_intensity[tid - 1], sum);
    }
  }
}

}  // namespace pbr
