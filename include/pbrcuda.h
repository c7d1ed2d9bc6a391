/*
 * pbrcuda.h — C ABI of libpbrcuda.so: the B200 (sm_100a) per-texel shading hot path of PyPBR.
 *
 * The reference (giuvecchio/PyPBR, pure Python) has no FFI layer: its boundary for this path is the
 * Python API.  Every entry point below replaces the ATen eager-op sequence inside one reference
 * function; the Python host layer (pypbr_b200/) keeps the reference's names and signatures and calls
 * these through ctypes (INTEGRATION.md shows the stub a PyPBR maintainer would add).
 *
 * Conventions
 *   - every function returns int: 0 = OK, negative = PBR_E_* (argument errors, detected on the host
 *     before any launch), positive = cudaError_t of the launch.  Nothing throws, nothing allocates
 *     device memory, nothing synchronises: work is enqueued on `stream` of the CURRENT device.
 *   - all maps are float32, channel-planar, with unit stride along W; batch / channel / row strides
 *     are given in ELEMENTS (so crops and batched (B,C,H,W) or unbatched (C,H,W) tensors are passed
 *     without a copy).  128-bit vector access is used when every pointer is 16-byte aligned and every
 *     stride is a multiple of 4; otherwise the same kernels run their scalar path.
 *   - the caller owns every buffer and keeps it alive until the stream has passed the launch.
 *   - the library keeps no mutable global state except an atomic launch counter; it is re-entrant
 *     and thread-safe.
 */
#ifndef PBRCUDA_H_
#define PBRCUDA_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PBR_ABI_VERSION 5
#define PBR_MAX_LIGHTS 64      /* lights per launch (parameters are staged in shared memory) */
#define PBR_MAX_BLEND_MAPS 12  /* maps blended by one pbr_blend launch */
#define PBR_MAX_INDEX_MAPS 12  /* maps moved by one pbr_index_transform launch */
#define PBR_MAX_ADAM_MAPS 8    /* parameter maps updated by one pbr_adam_step launch */

/* error codes (negative) */
#define PBR_OK 0
#define PBR_E_NULL (-1)        /* required pointer is NULL */
#define PBR_E_SHAPE (-2)       /* B/H/W/L out of range */
#define PBR_E_ENUM (-3)        /* workflow / light_type / mode out of range */
#define PBR_E_TOO_MANY (-4)    /* L > PBR_MAX_LIGHTS or n_maps > PBR_MAX_BLEND_MAPS */
#define PBR_E_CHANNELS (-5)    /* unsupported channel count */

typedef void* pbr_stream_t;    /* cudaStream_t */

/* One channel-planar map: element (b, c, y, x) lives at ptr[b*sb + c*sc + y*sh + x]. */
typedef struct PbrPlane {
  float* ptr;
  int64_t sb, sc, sh;
} PbrPlane;

enum { PBR_WORKFLOW_METALLIC = 0, PBR_WORKFLOW_SPECULAR = 1 };
enum { PBR_LIGHT_DIRECTIONAL = 0, PBR_LIGHT_POINT = 1 };

/*
 * Cook-Torrance shading descriptor.
 * Replaces CookTorranceBRDF.forward, pypbr/models/cooktorrance.py:68-182 (with fresnel_schlick
 * :184-196, normal_distribution_ggx :198-218, geometry_schlick_ggx :220-235, geometry_smith :237-260),
 * MaterialBase.linear_albedo pypbr/materials/base.py:262-277, DiffuseSpecularMaterial.linear_specular
 * pypbr/materials/diffuse.py:76-91, srgb_to_linear / linear_to_srgb pypbr/utils/functions.py:31-66.
 */
typedef struct PbrCtDesc {
  int32_t B, H, W, L;
  int32_t workflow;         /* PBR_WORKFLOW_*  (cooktorrance.py:103-118) */
  int32_t light_type;       /* PBR_LIGHT_*     (cooktorrance.py:125-142) */
  int32_t albedo_is_srgb;   /* base.py:272 */
  int32_t specular_is_srgb; /* diffuse.py:86 */
  int32_t return_srgb;      /* cooktorrance.py:179 */
  int32_t per_light;        /* 0: accumulate L lights into (B,3,H,W); 1: write (B,L,3,H,W) */
  int32_t params_on_device; /* 0: view/lights/intensity are HOST arrays (copied into the launch); 1: device arrays */
  float light_size;         /* physical plane size for point lights; <= 0 means 1.0 (cooktorrance.py:130) */
  PbrPlane albedo;          /* 3 ch */
  PbrPlane normal;          /* 3 ch, already in [-1,1]; ptr == NULL -> (0,0,1) (cooktorrance.py:143-151) */
  PbrPlane roughness;       /* 1 ch */
  PbrPlane metspec;         /* metallic: 1 ch (or 3, see metallic_channels); specular: 3 ch */
  int32_t metallic_channels;/* metallic workflow: 1 (usual) or 3 (the per-channel metallic that
                               to_basecolor_metallic_material produces, diffuse.py:150-156); 0 means 1 */
  const float* view;        /* 3 floats, not normalised */
  const float* lights;      /* L*3: direction (directional) or position (point) */
  const float* intensity;   /* L*3 */
  PbrPlane out;             /* 3 ch; per_light: sb is the stride of b, `out_sl` the stride of l */
  int64_t out_sl;
  int32_t force_generic;    /* 0: pick the kernel automatically (streamed TMA-fed kernels for L == 1 on 16-byte aligned,
                               W % 4 == 0 maps; generic kernels otherwise); 1: always the generic kernels (A/B tests) */
} PbrCtDesc;

/* Gradient buffers for pbr_ct_backward.  Any d_* with ptr == NULL is not computed. */
typedef struct PbrCtGrads {
  PbrPlane grad_out;        /* same logical shape as PbrCtDesc.out */
  int64_t grad_out_sl;
  PbrPlane d_albedo;        /* 3 ch */
  PbrPlane d_normal;        /* 3 ch */
  PbrPlane d_roughness;     /* 1 ch */
  PbrPlane d_metspec;       /* 1 or 3 ch */
  float* d_intensity;       /* device, L*3, ACCUMULATED with atomics: caller zero-fills; may be NULL */
  /* Gradients of the shared geometry parameters, which the reference delivers through plain autograd
     (cooktorrance.py:95 view_dir, :125-140 light direction / position).  Device, ACCUMULATED with atomics (caller
     zero-fills), may be NULL.  Requesting either selects the generic kernels with per-texel light geometry. */
  float* d_lights;          /* L*3: w.r.t. PbrCtDesc.lights as passed (raw direction or position) */
  float* d_view;            /* 3:   w.r.t. PbrCtDesc.view as passed (not normalised) */
  /* Optional (ptr may be NULL): the output pbr_ct_forward wrote for the same descriptor.  Used in accumulate mode with
     L > 1 only: the gate of clamp(sum over lights) and the slope of the sRGB encode are derived from it, which saves the
     backward a complete second forward evaluation of every light (otherwise it recomputes the sum first: two passes). */
  PbrPlane fwd_out;
} PbrCtGrads;

/*
 * Fused rendering-loss step (docs/source/tutorials/06_advanced.rst:73-107 scaled to a batch):
 *   loss_sum += sum((render(desc) - target)^2)   over every element this launch covers,
 *   d_* = d(loss_scale * that sum)/d(map), where the caller passes loss_scale = 1/numel for MSE.
 * The colour image is never written.  Per-tile warp-shuffle reduction, one atomic per CTA.
 */
typedef struct PbrCtLoss {
  PbrPlane target;          /* same logical shape as the render (desc.out is ignored) */
  int64_t target_sl;
  float loss_scale;
  float* loss_sum;          /* device scalar, ACCUMULATED: caller zero-fills */
} PbrCtLoss;

/*
 * Workflow conversions.
 * m2s replaces BasecolorMetallicMaterial.to_diffuse_specular_material arithmetic, pypbr/materials/metallic.py:90-109.
 * s2m replaces DiffuseSpecularMaterial.to_basecolor_metallic_material arithmetic, pypbr/materials/diffuse.py:112-147.
 */
typedef struct PbrConvDesc {
  int32_t B, H, W;
  int32_t albedo_is_srgb;
  PbrPlane albedo;          /* in, 3 ch */
  PbrPlane metspec;         /* in: metallic 1 ch or 3 ch (m2s, see metallic_channels) / raw specular 3 ch (s2m) */
  PbrPlane out0;            /* out 3 ch: diffuse (m2s) / basecolor (s2m) */
  PbrPlane out1;            /* out 3 ch: specular (m2s) / metallic, 3 channels (s2m) */
  int32_t metallic_channels;/* m2s: 1 (usual; 0 means 1) or 3 - the per-channel metallic s2m produces (diffuse.py:150-156);
                               the reference broadcasts either against the 3-channel albedo (metallic.py:103-106) */
} PbrConvDesc;

/*
 * Adjoints of the two conversions (the reference's are plain differentiable torch ops, metallic.py:103-109 and
 * diffuse.py:129-147, so a fit that goes through a conversion back-propagates through it): recompute the forward
 * per texel, follow autograd's conventions (inclusive clamp gates, torch.where routes, the sRGB decode slope).
 *   m2s: d_albedo = (g0 (1-m) + g1 m) decode'(albedo);  d_metallic = sum_c [-g0_c a_c + g1_c (a_c - 0.04)]
 *        (per channel for a 3-channel metallic);  s2m: through clamp / where / the two divisions (see the kernel).
 * `desc` is the forward's descriptor (out0 / out1 are ignored).  g_out*.ptr == NULL means a zero gradient; d_*.ptr ==
 * NULL means not required.
 */
typedef struct PbrConvGrads {
  PbrPlane g_out0, g_out1;  /* 3 ch each: gradients w.r.t. the forward's two outputs */
  PbrPlane d_albedo;        /* 3 ch */
  PbrPlane d_metspec;       /* m2s: 1 or 3 ch (metallic_channels); s2m: 3 ch (raw specular) */
} PbrConvGrads;

/*
 * Blending.  Replaces blend_with_mask / _blend_normals / blend_on_height / blend_on_properties /
 * blend_with_gradient arithmetic, pypbr/blending/functional.py:64-286: mask construction, the per-map
 * lerp `mask*m1 + (1-mask)*m2`, and the normalise-lerp-normalise of normal maps, all maps in one pass.
 */
enum { PBR_MASK_GIVEN = 0, PBR_MASK_SIGMOID = 1, PBR_MASK_GRADIENT_H = 2, PBR_MASK_GRADIENT_V = 3 };

typedef struct PbrBlendMap {
  PbrPlane a, b, out;
  int32_t channels;         /* 1..4 */
  int32_t is_normal;        /* 1: _blend_normals (functional.py:119-145), requires channels == 3 */
} PbrBlendMap;

typedef struct PbrBlendDesc {
  int32_t B, H, W;
  int32_t n_maps;
  int32_t mask_mode;        /* PBR_MASK_* */
  float blend_width;        /* sigmoid: mask = sigmoid(((p1 + shift) - p2) / (blend_width + 1e-6)) */
  float shift;
  int32_t apply_shift;      /* blend_on_height adds `shift` (functional.py:188); blend_on_properties has no such op */
  PbrPlane mask;            /* GIVEN: input (1 ch; sb may be 0 to broadcast over the batch) */
  PbrPlane prop1, prop2;    /* SIGMOID: the two 1-ch property / height maps */
  PbrPlane mask_out;        /* non-GIVEN modes: the mask is returned to the caller, so it is written (1 ch); may be NULL */
  float* normal_min;        /* optional device scalar (caller sets +inf): min over the blended normal, the
                               `normal_map.min() < 0` probe of MaterialBase._process_normal_map base.py:212 */
  PbrBlendMap maps[PBR_MAX_BLEND_MAPS];
} PbrBlendDesc;

/*
 * Adjoint of pbr_blend (functional.py:104-108 and :134-143 are plain differentiable torch ops in the reference).
 * `desc` is the forward's descriptor (maps[i].out, mask_out and normal_min are ignored); `mask` is the mask the forward
 * used: the given one, or the mask_out it wrote.  Per map i: d_a = mask g, d_b = (1-mask) g, through the three
 * normalisations for a normal map; d_mask = g_mask_out + sum over maps and channels of g (a - b);
 * SIGMOID: d_prop1 = d_mask mask (1 - mask) / (blend_width + 1e-6), d_prop2 = -d_prop1 (GRADIENT modes have no mask input).
 * NULL pointers: g_out -> zero gradient, d_* -> not required.
 */
typedef struct PbrBlendGradMap {
  PbrPlane g_out, d_a, d_b; /* same channel count as desc->maps[i] */
} PbrBlendGradMap;
typedef struct PbrBlendGrads {
  PbrPlane mask;            /* 1 ch, required */
  PbrPlane g_mask_out;      /* 1 ch: gradient flowing into the returned mask; may be NULL */
  PbrPlane d_mask;          /* GIVEN: 1 ch; may be NULL */
  PbrPlane d_prop1, d_prop2;/* SIGMOID: 1 ch each; may be NULL */
  PbrBlendGradMap maps[PBR_MAX_BLEND_MAPS];
} PbrBlendGrads;

/* sRGB <-> linear on an arbitrary C-channel map (pypbr/utils/functions.py:31-66). to_linear: 1 = decode, 0 = encode. */
typedef struct PbrColorDesc {
  int32_t B, C, H, W;
  int32_t to_linear;
  PbrPlane in, out;
} PbrColorDesc;

/*
 * Normal-map ingestion (MaterialBase._process_normal_map, pypbr/materials/base.py:191-242).
 * pbr_normal_min: *result = min(*result, min over all elements)  (the `min() < 0` probe, base.py:212).
 * pbr_normal_ingest: channels == 3: normalize(n*2-1) (base.py:215-217);
 *                    channels == 2: xy*2-1, z = sqrt(clamp(1-x^2-y^2, 1e-6)), normalise (base.py:223-242).
 */
typedef struct PbrNormalDesc {
  int32_t B, H, W;
  int32_t channels;         /* of `in`: 2 or 3; `out` always has 3 */
  PbrPlane in, out;         /* channels == 3: in == out is allowed (each thread reads its texels before it writes them) */
  const float* cond_min;    /* pbr_normal_ingest only, optional DEVICE scalar: the launch does nothing when *cond_min < 0.
                               It carries base.py:212's decision `normal_map.min() < 0 -> keep as is` for a probe result that
                               is still on the device (pbr_blend's normal_min), so the host never reads it back */
} PbrNormalDesc;

/* Adjoint of pbr_normal_ingest (base.py:215-217 / :235-242 are differentiable torch ops): `desc->in` is the forward's
   input (desc->out is ignored), g_out the gradient w.r.t. its 3-channel output, d_in receives `channels` channels. */
typedef struct PbrNormalGrads {
  PbrPlane g_out, d_in;
} PbrNormalGrads;

/*
 * Image ingestion - the step before the shading path (SURVEY.md 8f rank 2).  Replaces
 * MaterialBase._to_tensor for 8/16-bit images (pypbr/materials/base.py:122-168: TF.to_tensor divides by 255,
 * 16-bit by 65535) fused with MaterialBase._process_normal_map (base.py:191-242) for normal maps, so a material
 * travels host -> device as 8 (or 16) bit texels instead of float32.
 *   src: DEVICE pointer to an interleaved image (H, W, src_channels) of uint8 (bits = 8) or uint16 (bits = 16);
 *        strides in BYTES; out receives the first `channels` channels (PLAIN) or 3 channels (NORMAL2/3).
 */
enum { PBR_INGEST_PLAIN = 0, PBR_INGEST_NORMAL3 = 1, PBR_INGEST_NORMAL2 = 2 };
typedef struct PbrIngestDesc {
  int32_t B, H, W;
  int32_t bits;             /* 8 or 16 */
  int32_t src_channels;     /* interleaved channels per pixel in src (1..4) */
  int32_t channels;         /* PLAIN: channels to extract (1..4, <= src_channels) */
  int32_t mode;             /* PBR_INGEST_* */
  const void* src;
  int64_t src_batch_stride, src_row_stride;   /* bytes */
  PbrPlane out;
} PbrIngestDesc;

/*
 * Index transforms of every map of a material in one pass (SURVEY.md 8f rank 1).  Replaces the per-map
 * tensor.flip / torch.roll / tensor.repeat / TF.crop calls of MaterialBase.flip_horizontal, flip_vertical, roll,
 * tile and crop (pypbr/materials/base.py:490-537, 605-655), including the sign flip of the normal's x / y.
 *   out[c, y, x] = sign_c * in[c, origin_y + step_y*y, origin_x + step_x*x]; indices are wrapped modulo the input
 *   size when `wrap`, otherwise texels that fall outside the input are 0 (TF.crop zero-pads).  Pure data movement:
 *   results are bit-identical to the reference's torch calls.
 */
typedef struct PbrIndexMap {
  PbrPlane in, out;
  int32_t channels;         /* 1..4 */
  int32_t negate_mask;      /* bit c set: channel c changes sign (normal x for a horizontal flip, y for a vertical one) */
} PbrIndexMap;
typedef struct PbrIndexDesc {
  int32_t B, H_in, W_in, H_out, W_out;
  int32_t origin_y, step_y, origin_x, step_x;
  int32_t wrap;
  int32_t n_maps;
  /* Adjoint of a tile (tensor.repeat): out[y, x] = sum over i < reduce_y, j < reduce_x of the formula above evaluated at
     (y + i*H_out, x + j*W_out).  0 or 1 = plain gather.  The adjoints of flip and roll are gathers themselves. */
  int32_t reduce_y, reduce_x;
  PbrIndexMap maps[PBR_MAX_INDEX_MAPS];
} PbrIndexDesc;

/*
 * Adam step + projection of every parameter map of the inverse-rendering fit in one pass - the step after the
 * shading path (SURVEY.md 8f rank 3).  No reference code exists (docs/source/tutorials/06_advanced.rst:136-137
 * leaves the optimiser to the reader); the update is torch.optim.Adam's:
 *   m = m + (1-beta1)(g - m); v = beta2 v + (1-beta2) g^2; p -= step_size * m / (sqrt(v)/bias2_sqrt + eps)
 * with g = grad * grad_scale, step_size = lr / (1 - beta1^t), bias2_sqrt = sqrt(1 - beta2^t) computed by the caller.
 * Projection keeps the maps valid: CLAMP to [lo, hi] (albedo, roughness, metallic, specular), NORMALIZE the 3-vector
 * (normal).  param / exp_avg / exp_avg_sq are updated in place.
 */
enum { PBR_PROJECT_NONE = 0, PBR_PROJECT_CLAMP = 1, PBR_PROJECT_NORMALIZE = 2 };
typedef struct PbrAdamMap {
  PbrPlane param, grad, exp_avg, exp_avg_sq;
  int32_t channels;         /* 1..4; NORMALIZE requires 3 */
  int32_t project;          /* PBR_PROJECT_* */
  float lo, hi;
} PbrAdamMap;
typedef struct PbrAdamDesc {
  int32_t B, H, W;
  int32_t n_maps;
  float step_size, one_minus_beta1, beta2, one_minus_beta2, bias2_sqrt, eps, grad_scale;
  PbrAdamMap maps[PBR_MAX_ADAM_MAPS];
} PbrAdamDesc;

/*
 * Per-texel normal utilities of an augmentation pipeline (SURVEY.md 8f rank 4).
 *   ROTATE     : rotate_normals, pypbr/utils/functions.py:69-108 (the vector part of MaterialBase.rotate,
 *                base.py:598-600): (x, y) @ R(angle)^T with cos_a / sin_a computed by the caller in double and
 *                rounded to float as torch.tensor(...) does, then F.normalize over the 3 channels.  `in` has 3 channels;
 *                in == out is allowed (the reference rotates in place).
 *   FROM_HEIGHT: compute_normal_from_height, pypbr/utils/functions.py:123-177: grad_x = h[x-1] - h[x+1],
 *                grad_y = h[y-1] - h[y+1] with zeros outside the image, normal = normalize(-gx*scale, -gy*scale, 1)
 *                (flip_y = 0, OpenGL convention) or (-gx*scale, +gy*scale, 1) (flip_y = 1, DirectX).  `in` has 1 channel;
 *                in and out must not overlap.
 *   DIVERGENCE : the per-texel half of compute_height_from_normal, pypbr/utils/functions.py:211-283: the gradient field
 *                g = (-Nx, -Ny | +Ny) / (Nz + 1e-8) * scale (flip_y as above) and its forward-difference divergence with
 *                replicate padding.  `in` has 3 channels, `out` ONE channel; in and out must not overlap.  The Poisson
 *                solve that follows (utils/functions.py:286-323) is two FFT library calls and stays with the caller.
 *   FROM_HEIGHT_BWD: the adjoint of FROM_HEIGHT (the reference's op sequence is differentiable, so a height map can be fitted
 *                through the normals it induces): `in` = the height map (1 ch), `aux` = the gradient w.r.t. the 3-channel normal
 *                map, `out` = the gradient w.r.t. the height map (1 ch):
 *                d_h[y,x] = scale * (a[y,x+1] - a[y,x-1] + b[y+1,x] - b[y-1,x]) with a = -g_u.x, b = -+g_u.y of the neighbour texel,
 *                g_u the gradient pushed through that texel's normalisation (recomputed), zero outside the image.
 *   ROTATE_BWD : the adjoint of ROTATE (the reference's rotation is a matmul + F.normalize on a tensor autograd tracks; with
 *                cos_a = strength, sin_a = 0 it is the adjoint of MaterialBase.adjust_normal_strength, base.py:689-706):
 *                `in` = the normal map BEFORE the rotation (3 ch), `aux` = the gradient w.r.t. the rotated map (3 ch),
 *                `out` = the gradient w.r.t. `in` (3 ch); in, aux and out must not overlap.
 *   DIVERGENCE_BWD: the adjoint of DIVERGENCE: `in` = the normal map (3 ch), `aux` = the gradient w.r.t. the divergence (1 ch),
 *                `out` = the gradient w.r.t. the normal map (3 ch).  (The Poisson solve and the [0,1] normalisation around it
 *                are differentiable library calls on the caller's side.)
 */
enum { PBR_NORMAL_OP_ROTATE = 0, PBR_NORMAL_OP_FROM_HEIGHT = 1, PBR_NORMAL_OP_DIVERGENCE = 2, PBR_NORMAL_OP_FROM_HEIGHT_BWD = 3,
       PBR_NORMAL_OP_ROTATE_BWD = 4, PBR_NORMAL_OP_DIVERGENCE_BWD = 5 };
typedef struct PbrNormalOpDesc {
  int32_t B, H, W;
  int32_t op;               /* PBR_NORMAL_OP_* */
  float cos_a, sin_a;       /* ROTATE, ROTATE_BWD */
  float scale;              /* FROM_HEIGHT, DIVERGENCE and their adjoints */
  int32_t flip_y;           /* FROM_HEIGHT, DIVERGENCE and their adjoints: 1 = NormalConvention.DIRECTX */
  PbrPlane in, out;         /* out: 3 ch (DIVERGENCE, FROM_HEIGHT_BWD: 1 ch) */
  PbrPlane aux;             /* the adjoints: the incoming gradient (FROM_HEIGHT_BWD, ROTATE_BWD: 3 ch; DIVERGENCE_BWD: 1 ch); otherwise unused */
} PbrNormalOpDesc;

/*
 * Fused fit step (SURVEY.md 8f rank 3, "Adam ... fused into K3's epilogue"): pbr_ct_loss_fwd_bwd whose epilogue
 * applies the Adam update + projection of pbr_adam_step to the maps IN PLACE (desc->albedo / normal / roughness /
 * metspec are written) instead of storing the gradients: per texel the 32 B of gradients are neither written nor
 * read back, and the optimiser's pass over parameters and moments rides along a kernel that is FP32-bound.
 * Gradients are d(loss_scale * sum((render - target)^2))/d(map), so loss_scale must already be 1/(global numel);
 * the loss all-reduce of a sharded fit is only needed for reporting and stays off the critical path.
 * project != 0: clamp albedo / roughness / metallic | specular to [0,1], renormalise the normal (eps 1e-12).
 * m_normal / v_normal are ignored when desc->normal.ptr is NULL.
 */
typedef struct PbrCtAdam {
  PbrPlane m_albedo, v_albedo;        /* exp_avg, exp_avg_sq: same shapes as the maps, updated in place */
  PbrPlane m_normal, v_normal;
  PbrPlane m_roughness, v_roughness;
  PbrPlane m_metspec, v_metspec;
  float step_size, one_minus_beta1, beta2, one_minus_beta2, bias2_sqrt, eps;   /* as in PbrAdamDesc */
  int32_t project;
} PbrCtAdam;

int pbr_abi_version(void);
const char* pbr_strerror(int code);

int pbr_ct_forward(const PbrCtDesc* desc, pbr_stream_t stream);
int pbr_ct_backward(const PbrCtDesc* desc, const PbrCtGrads* grads, pbr_stream_t stream);
int pbr_ct_loss_fwd_bwd(const PbrCtDesc* desc, const PbrCtLoss* loss, const PbrCtGrads* grads, pbr_stream_t stream);
/* d_intensity: device, L*3, accumulated with atomics (caller zero-fills); may be NULL */
int pbr_ct_fit_step(const PbrCtDesc* desc, const PbrCtLoss* loss, const PbrCtAdam* adam, float* d_intensity,
                    pbr_stream_t stream);
/* Camera at a finite position: the same three calls with desc->view read as the camera POSITION c (same frame as a
 * point light's position; host or device memory according to params_on_device) instead of the view direction.  Texel
 * (i, j) sits at P = (x_j, -y_i, 0) on the plane of side s = light_size (> 0, else 1) - for both light types - and is
 * shaded with the view vector F.normalize(c - P).  grads->d_view receives the gradient w.r.t. c.  force_generic and
 * fwd_out are ignored; the argument checks and error codes are those of pbr_ct_forward / _backward / _loss_fwd_bwd. */
int pbr_ct_forward_camera(const PbrCtDesc* desc, pbr_stream_t stream);
int pbr_ct_backward_camera(const PbrCtDesc* desc, const PbrCtGrads* grads, pbr_stream_t stream);
int pbr_ct_loss_fwd_bwd_camera(const PbrCtDesc* desc, const PbrCtLoss* loss, const PbrCtGrads* grads, pbr_stream_t stream);

/*
 * Per-material parameters of a batch: material b is shaded with its own view (or camera position), lights and intensities
 * at desc->view + b*view_sb, desc->lights + b*lights_sb and desc->intensity + b*intensity_sb (strides in floats).  A stride
 * of 0 shares that parameter across the batch, as the calls above do; each of the three is shared or per material on its
 * own.  The gradient buffers grads->d_view / d_lights / d_intensity (and the fit step's d_intensity) take the same
 * strides: a per-material parameter receives its own material's sums, a shared one the sum over the batch.  Results are
 * those of B calls with B = 1, one per material.  camera = 1 reads desc->view as the camera position (pbr_ct_*_camera).
 * Argument errors, before any launch: pb == NULL -> PBR_E_NULL; camera not 0 / 1, or a non-zero stride with
 * params_on_device = 0 -> PBR_E_ENUM; a non-zero stride below 3 (view) or 3L (lights, intensity) -> PBR_E_SHAPE;
 * camera = 1 on the fit step -> PBR_E_ENUM.  Otherwise the checks and codes of the calls without _pb.
 */
typedef struct PbrCtParamBatch {
  int32_t camera;           /* 0: desc->view is the view direction; 1: the camera position */
  int32_t pad;
  int64_t view_sb, lights_sb, intensity_sb;
} PbrCtParamBatch;

int pbr_ct_forward_pb(const PbrCtDesc* desc, const PbrCtParamBatch* pb, pbr_stream_t stream);
int pbr_ct_backward_pb(const PbrCtDesc* desc, const PbrCtParamBatch* pb, const PbrCtGrads* grads, pbr_stream_t stream);
int pbr_ct_loss_fwd_bwd_pb(const PbrCtDesc* desc, const PbrCtParamBatch* pb, const PbrCtLoss* loss, const PbrCtGrads* grads,
                           pbr_stream_t stream);
int pbr_ct_fit_step_pb(const PbrCtDesc* desc, const PbrCtParamBatch* pb, const PbrCtLoss* loss, const PbrCtAdam* adam,
                       float* d_intensity, pbr_stream_t stream);

int pbr_convert_m2s(const PbrConvDesc* desc, pbr_stream_t stream);
int pbr_convert_s2m(const PbrConvDesc* desc, pbr_stream_t stream);
int pbr_convert_m2s_backward(const PbrConvDesc* desc, const PbrConvGrads* grads, pbr_stream_t stream);
int pbr_convert_s2m_backward(const PbrConvDesc* desc, const PbrConvGrads* grads, pbr_stream_t stream);
int pbr_blend(const PbrBlendDesc* desc, pbr_stream_t stream);
int pbr_blend_backward(const PbrBlendDesc* desc, const PbrBlendGrads* grads, pbr_stream_t stream);
int pbr_color_convert(const PbrColorDesc* desc, pbr_stream_t stream);
int pbr_normal_min(const PbrNormalDesc* desc, float* result, pbr_stream_t stream);
int pbr_normal_ingest(const PbrNormalDesc* desc, pbr_stream_t stream);
int pbr_normal_ingest_backward(const PbrNormalDesc* desc, const PbrNormalGrads* grads, pbr_stream_t stream);
int pbr_ingest_image(const PbrIngestDesc* desc, pbr_stream_t stream);
int pbr_index_transform(const PbrIndexDesc* desc, pbr_stream_t stream);
int pbr_adam_step(const PbrAdamDesc* desc, pbr_stream_t stream);
int pbr_normal_op(const PbrNormalOpDesc* desc, pbr_stream_t stream);

/* sizeof() of the descriptor structs as THIS library was compiled (binding self-check):
   which = 0 PbrPlane, 1 PbrCtDesc, 2 PbrCtGrads, 3 PbrCtLoss, 4 PbrConvDesc, 5 PbrBlendMap, 6 PbrBlendDesc,
   7 PbrColorDesc, 8 PbrNormalDesc, 9 PbrIngestDesc, 10 PbrIndexMap, 11 PbrIndexDesc, 12 PbrAdamMap, 13 PbrAdamDesc, 14 PbrCtAdam, 15 PbrNormalOpDesc,
   16 PbrConvGrads, 17 PbrBlendGradMap, 18 PbrBlendGrads, 19 PbrNormalGrads, 20 PbrCtParamBatch;
   anything else returns 0. */
uint64_t pbr_sizeof(int which);

/* Number of kernel launches this process has enqueued through the library (for bench accounting). */
uint64_t pbr_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* PBRCUDA_H_ */
