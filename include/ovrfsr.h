/*
 * ovrfsr.h -- C ABI of the B200-native FSR1 / NIS eye-texture post-process.
 *
 * This is the drop-in boundary for ONE path of fholger/openvr_fsr: the per-eye pass that
 * vr::PostProcessor::Apply runs from the IVRCompositor::Submit hook
 * (src/postprocess/PostProcessor.cpp:123-164, called from src/postprocess/VrHooks.cpp:53,71,84).
 * Everything D3D11 did on that path (compute-shader dispatch of fsr_easu / fsr_rcas /
 * NIS_Upscale / NIS_Sharpen, constant buffers, intermediate textures) is behind these calls
 * as hand-written sm_100a CUDA kernels.  Plain pointers and sizes only; no C++ or torch
 * types cross this boundary.  All citations are relative to /root/reference/.
 *
 * The C++ class a maintainer links instead of the D3D11 one is
 * openvr_fsr_b200/csrc/postprocessor.h (same Apply/Reset surface); INTEGRATION.md shows
 * the binding.  There is NO CPU fallback: every entry point that launches work returns
 * OVRFSR_ERR_CUDA if no sm_100 device / driver is usable.
 */
#ifndef OVRFSR_H
#define OVRFSR_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define OVRFSR_API __declspec(dllexport)
#else
#define OVRFSR_API __attribute__((visibility("default")))
#endif

#define OVRFSR_VERSION 0x00010000u

/* status codes.  The reference's error convention is "log, disable, pass the frame through"
 * (PostProcessor.cpp:23-28,145-152); the C++ wrapper maps any non-zero status to that. */
typedef enum ovrfsr_status {
  OVRFSR_OK = 0,
  OVRFSR_ERR_INVALID = 1,     /* null / malformed argument */
  OVRFSR_ERR_UNSUPPORTED = 2, /* format or scale the path does not handle */
  OVRFSR_ERR_CUDA = 3,        /* CUDA runtime / driver failure, or no device */
  OVRFSR_ERR_NOMEM = 4,
  OVRFSR_PASSTHROUGH = 5      /* fsr_enabled == 0: nothing done, caller submits its own texture */
} ovrfsr_status;

/* pixel formats: the DXGI formats the path binds (PostProcessor.cpp:30-74) */
typedef enum ovrfsr_format {
  OVRFSR_FORMAT_RGBA8 = 0,   /* DXGI_FORMAT_R8G8B8A8_UNORM (sRGB variants are viewed as UNORM, :50-61) */
  OVRFSR_FORMAT_BGRA8 = 1,   /* DXGI_FORMAT_B8G8R8A8_UNORM */
  OVRFSR_FORMAT_RGBA16F = 2, /* DXGI_FORMAT_R16G16B16A16_FLOAT */
  OVRFSR_FORMAT_RGBA32F = 3, /* DXGI_FORMAT_R32G32B32A32_FLOAT (input: PostProcessor.cpp:32-33; as an output it
                                exposes the pre-quantisation result) */
  OVRFSR_FORMAT_RGB10A2 = 4, /* DXGI_FORMAT_R10G10B10A2_UNORM: one little-endian u32 per texel, R bits 0-9, G 10-19,
                                B 20-29, A 30-31.  As an output it is only produced from an RGB10A2 source -- the case
                                DetermineOutputFormat() exists for (:63-74) */
  OVRFSR_FORMAT_BGRX8 = 5,   /* DXGI_FORMAT_B8G8R8X8_UNORM (:54-55): source only; the X byte reads as alpha 1 */
  OVRFSR_FORMAT_RGB32F = 6,  /* DXGI_FORMAT_R32G32B32_FLOAT (:34-35): source only, 12 bytes per texel, alpha reads as 1;
                                ovrfsr_apply expands it to RGBA32F first (ovrfsr_expand_rgb32f), the stateless dispatches
                                return OVRFSR_ERR_UNSUPPORTED for it */
  OVRFSR_FORMAT_AUTO = -1    /* output only: DetermineOutputFormat(), :63-74 -> RGB10A2 for an RGB10A2 source, else RGBA8 */
} ovrfsr_format;

/* DXGI variant tags, OR-ed into ovrfsr_image::format of a SOURCE image.  The kernels view _SRGB and _TYPELESS textures as
 * plain UNORM (MakeSrgbFormatsTypeless / TranslateTypelessFormats, PostProcessor.cpp:30-61: no sRGB decode happens on this
 * path), so the tags change no pixel; they exist so that vr::PostProcessor can reproduce the colour-space tag the
 * reference hands to the real Submit (inputIsSrgb, :504 with IsConsideredSrgbByOpenVR, :76-92). */
#define OVRFSR_FORMAT_LAYOUT_MASK 0xff
#define OVRFSR_FORMAT_SRGB_BIT 0x100     /* DXGI_FORMAT_*_UNORM_SRGB */
#define OVRFSR_FORMAT_TYPELESS_BIT 0x200 /* DXGI_FORMAT_*_TYPELESS */

/* arithmetic mode of the kernels */
typedef enum ovrfsr_math {
  OVRFSR_MATH_FAST = 0,  /* FMA contraction + regrouped taps: each pass is <= 1 LSB (RGBA8) from the reference lines
                            on identical inputs.  Note that EASU -> RGBA8 -> RCAS amplifies a 1-LSB intermediate
                            difference in dark regions (RCAS divides by the ring maximum), as it does between any two
                            D3D11 GPUs; use STRICT when the composed result must match to the bit.  Measured on the
                            C2-sized test images: max 3 LSB, < 6e-6 of the channel values beyond 1 LSB (asserted <= 4
                            LSB / 1e-4 in tests/test_gpu_fsr_parity.py). */
  OVRFSR_MATH_STRICT = 1 /* the reference's operation order, no contraction: bit-identical to the reference lines,
                            end to end.  The default of ovrfsr_config_default. */
} ovrfsr_math;

/* Device-resident image: the CUDA analogue of the ID3D11Texture2D* that Texture_t::handle
 * carries (headers/openvr.h:177-182).  data is a device pointer unless stated otherwise. */
typedef struct ovrfsr_image {
  void *data;
  uint32_t width;
  uint32_t height;
  uint32_t pitch;       /* bytes per row; rows need not be tightly packed */
  int32_t format;       /* ovrfsr_format */
  uint32_t array_slices;/* >1: right eye lives in slice 1 (PostProcessor.cpp:254-268); 0 is treated as 1 */
  uint32_t slice_pitch; /* bytes between slices when array_slices > 1 */
  uint32_t sample_count;/* >1: multisampled source (D3D11_TEXTURE2D_DESC::SampleDesc.Count): the samples of one texel
                           are consecutive, row = width*sample_count texel-sized entries; ovrfsr_apply resolves it
                           first like GetInputView's ResolveSubresource (PostProcessor.cpp:219-226).  0 = 1. */
} ovrfsr_image;

/* The Config fields that steer the path (src/postprocess/Config.h:11-17) plus what the
 * reference pulls from the live runtime (projection centres, PostProcessor.cpp:104-121). */
typedef struct ovrfsr_config {
  uint32_t struct_size;   /* sizeof(ovrfsr_config) */
  int32_t fsr_enabled;    /* Config::fsrEnabled */
  int32_t use_nis;        /* Config::useNis */
  float render_scale;     /* Config::renderScale */
  float sharpness;        /* Config::sharpness */
  float radius;           /* Config::radius */
  int32_t debug_mode;     /* Config::debugMode: tints the outside-radius region, enables timing */
  float proj_centre[4];   /* {leftX,leftY,rightX,rightY}; 0.5 each for a symmetric HMD */
  int32_t device;         /* CUDA device ordinal, -1 = current device */
  int32_t output_format;  /* ovrfsr_format, AUTO = reference behaviour */
  int32_t math_mode;      /* ovrfsr_math */
  int32_t flags;          /* OVRFSR_FLAG_* bits; 0 = defaults */
  int32_t reserved[4];
} ovrfsr_config;

/* ovrfsr_config::flags */
/* Run EASU -> RCAS as ONE fused kernel that keeps the upscaled image in shared memory (same output bits, 79.7 -> 35.0 MB
 * of traffic per C2 eye, one launch) whenever both passes run on the FSR path and the intermediate is UNORM (RGBA8 /
 * RGB10A2).  Off by default: on B200 the pass is instruction-issue-bound, not traffic-bound, and the fused kernel's
 * recomputed ring and lower occupancy make it 10-15 % SLOWER than the two dispatches (DESIGN.md section 5 has the
 * measurements at radius 2.0, 0.5 and 0).  Default (bit clear): the reference's two dispatches (PostProcessor.cpp:586-594),
 * with the outside-radius pixels written straight to the final image by the first one. */
#define OVRFSR_FLAG_FUSED_FSR 1

typedef struct ovrfsr_ctx ovrfsr_ctx;

/* ---- lifetime ------------------------------------------------------------------------- */
/* Fills cfg with the reference defaults (Config.h:11-17: enabled=false, renderScale=1,
 * sharpness=0.75, radius=0.5) and proj centres 0.5. */
OVRFSR_API void ovrfsr_config_default(ovrfsr_config *cfg);
/* Replaces the `PostProcessor postProcessor;` global (VrHooks.cpp:19).  No GPU work happens here. */
OVRFSR_API int ovrfsr_create(ovrfsr_ctx **out, const ovrfsr_config *cfg);
OVRFSR_API void ovrfsr_destroy(ovrfsr_ctx *ctx);
/* PostProcessor::Reset (PostProcessor.cpp:166-194): drops every cached resource, re-enables. */
OVRFSR_API int ovrfsr_reset(ovrfsr_ctx *ctx);
/* What the hotkeys do (PostProcessor.cpp:670-704): mutate Config, then Reset. */
OVRFSR_API int ovrfsr_set_config(ovrfsr_ctx *ctx, const ovrfsr_config *cfg);
OVRFSR_API int ovrfsr_get_config(const ovrfsr_ctx *ctx, ovrfsr_config *cfg);

/* ---- the hot path --------------------------------------------------------------------- */
/* PostProcessor::Apply minus the OpenVR types (PostProcessor.cpp:123-164,563-638).
 *   eye           EVREye (0 left, 1 right)
 *   src           borrowed, read-only
 *   only_one_eye  |uMax-uMin| > .5 of the submit bounds (:146); 0 = both eyes side by side in src
 *   out           receives the ctx-owned output image (upscaled+sharpened); valid until the next
 *                 apply for the same eye, reset or destroy.  One output per eye (the reference
 *                 shares one between both eyes, PostProcessor.h:43,58).
 *   stream        cudaStream_t; work is enqueued asynchronously, nothing is synchronised.  The ctx reuses its per-eye
 *                 intermediates and outputs on every call, so successive calls for the SAME eye of one ctx must be
 *                 ordered (same stream, or the caller's own events); the two eyes may run on different streams, and
 *                 frames in flight beyond that take one ctx each.
 * Lazy-initialises on first call and re-initialises when src dimensions change (:136-143).
 * Pass selection: upscale iff renderScale != 1; sharpen iff !useNis || renderScale == 1 (:586-594). */
OVRFSR_API int ovrfsr_apply(ovrfsr_ctx *ctx, int eye, const ovrfsr_image *src, int only_one_eye,
                            ovrfsr_image *out, void *stream);
/* Same pass with HOST images: copies src host->device, runs ovrfsr_apply, copies the result to
 * dst_host (which must be outW x outH of the ctx output format), all on `stream`.  Pinned host
 * memory makes the copies asynchronous.  This is the end-to-end entry bench.py times. */
OVRFSR_API int ovrfsr_apply_host(ovrfsr_ctx *ctx, int eye, const ovrfsr_image *src_host, int only_one_eye,
                                 const ovrfsr_image *dst_host, void *stream);

/* Both eyes of one frame in one call, for hosts that hold both textures when they submit (the reference's hook sees them
 * one Submit at a time, VrHooks.cpp:50-66; its D3D11 context is free to overlap the two eyes' dispatches, which have no
 * hazard between them -- a single CUDA stream is not).  Same result and same per-eye state as
 *   ovrfsr_apply(ctx, 0, src_left, only_one_eye, &out[0], stream); ovrfsr_apply(ctx, 1, src_right, only_one_eye, &out[1], stream);
 * but the right eye's passes run on a ctx-owned stream forked from `stream` before the left eye is queued and joined
 * back into it before the call returns, so the tail of one eye's launches overlaps the other eye's (C2, one caller
 * stream: see DESIGN.md section 7).  Everything queued on `stream` afterwards sees both outputs; capturable into a CUDA
 * graph.  With only_one_eye == 0 (one texture holding both eyes) it is exactly the two calls above. */
OVRFSR_API int ovrfsr_apply_pair(ovrfsr_ctx *ctx, const ovrfsr_image *src_left, const ovrfsr_image *src_right,
                                 int only_one_eye, ovrfsr_image out[2], void *stream);

/* VRTextureBounds_t (headers/openvr.h:609-613): the part of an eye texture that holds the image, in [0, 1] texture
 * coordinates.  {0, 0, 1, 1} is the whole texture. */
typedef struct ovrfsr_bounds {
  float u_min, v_min, u_max, v_max;
} ovrfsr_bounds;
/* a rectangle of texels: x, y = its top-left texel */
typedef struct ovrfsr_rect {
  uint32_t x, y, width, height;
} ovrfsr_rect;

/* Extension: ovrfsr_apply for an eye submitted with texture bounds (dynamic resolution, both eyes side by side in one
 * texture).  The eye is processed exactly as if its rectangle had been cut out as a texture of its own and given to
 * ovrfsr_apply with only_one_eye = 1, and the result is written at the matching rectangle of the usual full-size
 * output, so the compositor's bounds still address the output unchanged:
 *   - rectangles (single-precision host arithmetic): u0 = clamp(min(u_min, u_max), 0, 1), u1 = clamp(max(u_min, u_max),
 *     0, 1), likewise v (flipped bounds give the same rectangle; the flip stays with the compositor);
 *     source x0 = (uint32_t)(u0 * (float)W + 0.5f), x1 = (uint32_t)(u1 * (float)W + 0.5f), likewise y with H, in the
 *     eye's texture (its slice for an array texture) of W x H texels; the output rectangle is the same formula on the
 *     ctx output size ovrfsr_output_size(W, H, renderScale).  ovrfsr_bounds_rects computes both.
 *   - constants: ovrfsr_make_upscale_constants / _sharpen_constants / ovrfsr_make_nis_config for the eye with the
 *     rectangle sizes and only_one_eye = 1 -- the foveation centre and radius follow the view;
 *   - at the rectangle's edges EASU, NVScaler and NVSharpen clamp to the edge and RCAS reads zero, as at a texture's
 *     edge; texels outside the source rectangle never influence the result, pixels outside the output rectangle are
 *     not written.
 * Each call processes its eye (no "shared texture processed once" rule: a side-by-side texture is two rectangles).  A
 * rectangle change is not a size change: it resets, reallocates and synchronises nothing; a texture size or format
 * change resets as in ovrfsr_apply.  ovrfsr_apply and ovrfsr_apply_bounds may be mixed on one ctx.  The opt-in fused
 * kernel (OVRFSR_FLAG_FUSED_FSR) runs only for full bounds; other rectangles take the two dispatches (same bits).
 *   bounds    NULL = {0, 0, 1, 1}; an empty rectangle (either dimension) is OVRFSR_ERR_INVALID
 *   out       the full ctx-owned output image, as ovrfsr_apply returns it
 *   out_rect  nullable: receives the output rectangle */
OVRFSR_API int ovrfsr_apply_bounds(ovrfsr_ctx *ctx, int eye, const ovrfsr_image *src, const ovrfsr_bounds *bounds,
                                   ovrfsr_image *out, ovrfsr_rect *out_rect, void *stream);
/* The two rectangles of ovrfsr_apply_bounds for a W x H eye texture and an out_w x out_h output (pure CPU).  bounds NULL
 * = {0, 0, 1, 1}.  OVRFSR_ERR_INVALID for an empty rectangle or NaN bounds; either output pointer may be NULL. */
OVRFSR_API int ovrfsr_bounds_rects(uint32_t w, uint32_t h, uint32_t out_w, uint32_t out_h, const ovrfsr_bounds *bounds,
                                   ovrfsr_rect *src_rect, ovrfsr_rect *dst_rect);

/* ---- individual dispatches (ApplyUpscaling / ApplySharpening, PostProcessor.cpp:385-401,483-496) --
 * Stateless: explicit constant blocks, caller-owned destination.  math_mode as ovrfsr_math. */
/* g_FSRUpscaleShader: consts = UpscaleConstants, 24 x u32 (PostProcessor.cpp:276-283) */
OVRFSR_API int ovrfsr_dispatch_fsr_easu(const ovrfsr_image *src, const ovrfsr_image *dst, const uint32_t consts[24],
                                        int math_mode, void *stream);
/* g_FSRSharpenShader: consts = SharpenConstants, 12 x u32 (PostProcessor.cpp:403-407) */
OVRFSR_API int ovrfsr_dispatch_fsr_rcas(const ovrfsr_image *src, const ovrfsr_image *dst, const uint32_t consts[12],
                                        int math_mode, void *stream);
/* g_FSRUpscaleShader followed by g_FSRSharpenShader (ApplyPostProcess, PostProcessor.cpp:586-594) as ONE kernel: the
 * upscaled image is quantised to dst->format (RGBA8, or RGB10A2 for an RGB10A2 source) exactly as the first dispatch
 * stores it, but never leaves shared memory.  Bit-identical to the two dispatches above run back to back.  The two
 * constant blocks must carry the same centres / radius words (they do when built by ovrfsr_make_*_constants for one
 * eye); OVRFSR_ERR_UNSUPPORTED if this pair cannot be fused (formats, out->in scale above ~1.05). */
OVRFSR_API int ovrfsr_dispatch_fsr_fused(const ovrfsr_image *src, const ovrfsr_image *dst, const uint32_t upscale_consts[24],
                                         const uint32_t sharpen_consts[12], int math_mode, void *stream);
/* g_NISUpscaleShader / g_NISSharpenShader: cfg = NISConfig, 256 bytes (NIS_Config.h:37-77 + the
 * mod's centre/radius at byte 112, PostProcessor.cpp:310) */
OVRFSR_API int ovrfsr_dispatch_nis_scaler(const ovrfsr_image *src, const ovrfsr_image *dst, const void *cfg256,
                                          int math_mode, void *stream);
OVRFSR_API int ovrfsr_dispatch_nis_sharpen(const ovrfsr_image *src, const ovrfsr_image *dst, const void *cfg256,
                                           int math_mode, void *stream);

/* ---- host-side constant setup (pure CPU; usable without a GPU) -------------------------- */
/* PrepareResources, PostProcessor.cpp:509-518 */
OVRFSR_API void ovrfsr_output_size(uint32_t in_w, uint32_t in_h, float render_scale, uint32_t *out_w,
                                   uint32_t *out_h);
/* FsrEasuCon, ffx_fsr1.h:156-202 */
OVRFSR_API void ovrfsr_fsr_easu_con(uint32_t con[16], float in_vp_w, float in_vp_h, float in_w, float in_h,
                                    float out_w, float out_h);
/* FsrRcasCon, ffx_fsr1.h:662-672 (argument in stops) */
OVRFSR_API void ovrfsr_fsr_rcas_con(uint32_t con[4], float sharpness_stops);
/* UpscaleConstants for one eye, PostProcessor.cpp:293-305,331-337 */
OVRFSR_API void ovrfsr_make_upscale_constants(uint32_t consts[24], const ovrfsr_config *cfg, int eye,
                                              int only_one_eye, uint32_t in_w, uint32_t in_h, uint32_t out_w,
                                              uint32_t out_h);
/* SharpenConstants for one eye, PostProcessor.cpp:416-430,453-459 */
OVRFSR_API void ovrfsr_make_sharpen_constants(uint32_t consts[12], const ovrfsr_config *cfg, int eye,
                                              int only_one_eye, uint32_t out_w, uint32_t out_h);
/* NISConfig for one eye: NVScalerUpdateConfig (sharpen_only=0, PostProcessor.cpp:307-310) or
 * NVSharpenUpdateConfig (sharpen_only=1, :432-435).  Returns the bool the mod ignores (1 = scale in range). */
OVRFSR_API int ovrfsr_make_nis_config(void *cfg256, const ovrfsr_config *cfg, int sharpen_only, int eye,
                                      int only_one_eye, uint32_t in_w, uint32_t in_h, uint32_t out_w,
                                      uint32_t out_h);
/* coef_scale / coef_usm, NIS_Config.h:261-393: 64 phases x 8 floats */
OVRFSR_API const float *ovrfsr_nis_coef_scale(void);
OVRFSR_API const float *ovrfsr_nis_coef_usm(void);

/* ---- introspection -------------------------------------------------------------------- */
/* constant blocks the ctx built for `eye` (valid after the first apply) */
OVRFSR_API int ovrfsr_get_upscale_constants(const ovrfsr_ctx *ctx, int eye, uint32_t consts[24]);
OVRFSR_API int ovrfsr_get_sharpen_constants(const ovrfsr_ctx *ctx, int eye, uint32_t consts[12]);
/* Device self-test: strict-math RCAS replaces rcp.rn by MUFU.RCP + one Newton step when the source is UNORM8 (its
 * reciprocal operands then come from a set of 512 values); this runs both over the whole set on the current device.
 * *mismatches must come back 0. */
OVRFSR_API int ovrfsr_selftest_rcp(uint32_t *mismatches, uint32_t *checked);
/* Device self-test: strict-math NVScaler / NVSharpen with a UNORM source evaluate GetEdgeMap's and CalcLTI's quotients
 * (NIS_Scaler.h:244-247,373) with the in-range form of IEEE division (no exponent-range fallback); this compares it
 * with div.rn on ~19 M pseudo-random operand pairs of that range on the current device.  *mismatches must be 0. */
OVRFSR_API int ovrfsr_selftest_div(uint32_t *mismatches, uint32_t *checked);
/* kernels launched by this library in this process since load (bench.py's gpu_launches) */
OVRFSR_API uint64_t ovrfsr_kernel_launches(void);
/* debugMode profiling (PostProcessor.cpp:547-557,601-628): mean GPU ms per apply over the samples
 * collected so far (cudaEvent pairs read back a few frames late); returns samples used, 0 if none. */
OVRFSR_API int ovrfsr_get_gpu_time_ms(ovrfsr_ctx *ctx, float *mean_ms);
OVRFSR_API const char *ovrfsr_last_error(const ovrfsr_ctx *ctx);
OVRFSR_API const char *ovrfsr_status_string(int status);
OVRFSR_API uint32_t ovrfsr_version(void);
/* device image helpers (cudaMalloc with a 256-byte-aligned pitch, cudaFree) */
OVRFSR_API int ovrfsr_image_alloc(ovrfsr_image *img, uint32_t width, uint32_t height, int32_t format);
OVRFSR_API void ovrfsr_image_free(ovrfsr_image *img);


/* ---- the callers either side of the path (SURVEY.md 8f rows 2-4) -------------------------- */
/* R32G32B32_FLOAT source (PostProcessor.cpp:34-35) -> RGBA32F with alpha 1, what a shader reads from such a view.
 * src->format RGB32F (12-byte texels), dst->format RGBA32F, same size.  Asynchronous on `stream`. */
OVRFSR_API int ovrfsr_expand_rgb32f(const ovrfsr_image *src, const ovrfsr_image *dst, void *stream);
/* IsConsideredSrgbByOpenVR (PostProcessor.cpp:76-92) on a tagged ovrfsr_format: 1 for the _SRGB variants of RGBA8 /
 * BGRA8 / BGRX8 and for the _TYPELESS variants of RGBA8 / BGRA8 / BGRX8 / RGB10A2 */
OVRFSR_API int ovrfsr_format_considered_srgb(int32_t tagged_format);
/* GetInputView's MSAA branch (PostProcessor.cpp:219-226, ResolveSubresource): dst[x,y] = mean of the
 * sample_count samples of texel (x,y), same format in and out; src_samples laid out as ovrfsr_image::sample_count
 * describes (its width is the texel width).  Asynchronous on `stream`. */
OVRFSR_API int ovrfsr_resolve_msaa(const ovrfsr_image *src_samples, const ovrfsr_image *dst, void *stream);
/* IVRSystem_GetRecommendedRenderTargetSize detour (VrHooks.cpp:37-48): in/out the runtime's recommendation; scaled
 * by renderScale when fsr_enabled and renderScale < 1 (u32 *= float, truncating). */
OVRFSR_API void ovrfsr_recommended_render_size(const ovrfsr_config *cfg, uint32_t *width, uint32_t *height);
/* the MIP LOD bias handed to the sampler hook: -log2(outputWidth / (float)inputWidth), PostProcessor.cpp:537-538 */
OVRFSR_API float ovrfsr_mip_lod_bias(uint32_t input_width, uint32_t output_width);
/* D3D11Context_PSSetSamplers' rule (VrHooks.cpp:123-128): the bias a replacement sampler gets -- added only to
 * samplers without a bias of their own that filter anisotropically. */
OVRFSR_API float ovrfsr_sampler_lod_bias(float sampler_mip_lod_bias, uint32_t sampler_max_anisotropy, float mip_lod_bias);

/* The legacy CAS shaders the reference keeps under src/cas but never dispatches (src/CMakeLists.txt builds only fsr/
 * and nis/): CasSetup (src/cas/ffx_cas.h:375-397; consts = const0[4], const1[4]) and one CasFilter per output pixel,
 * alpha 1 (src/cas/cas.compute.h:25-47).  sharpen_only = cas.sharpen.hlsl (CAS_BETTER_DIAGONALS; dst size == src
 * size), else cas.upscale.hlsl (dst at least as large as src).  No radius mask exists on this path. */
OVRFSR_API void ovrfsr_cas_setup(uint32_t consts[8], float sharpness, float max_color_delta, float in_w, float in_h,
                                 float out_w, float out_h);
OVRFSR_API int ovrfsr_dispatch_cas(const ovrfsr_image *src, const ovrfsr_image *dst, const uint32_t consts[8],
                                   int sharpen_only, int math_mode, void *stream);

/* F7 capture (PostProcessor.cpp:630-657): the next apply for the LEFT eye writes its output image to
 * <directory>/capture_<YYYYmmdd_HHMMSS>_<fsr|nis>_s<sharpness*100>_r<radius*100>.dds and clears the request.
 * That apply synchronises the stream (the reference's SaveDDSTextureToFile maps a staging copy). */
OVRFSR_API int ovrfsr_request_capture(ovrfsr_ctx *ctx, const char *directory);
OVRFSR_API const char *ovrfsr_last_capture_path(const ovrfsr_ctx *ctx);
/* file name part of SaveTextureToFile (:641-652) for a given local time (seconds since the epoch) */
OVRFSR_API int ovrfsr_capture_filename(const ovrfsr_config *cfg, int64_t unix_time, char *buf, uint32_t buf_size);
/* DDS container exactly as ScreenGrab11's SaveDDSTextureToFile lays it out (ScreenGrab11.cpp:815-935): RGBA8 with
 * the legacy A8B8G8R8 masks, BGRA8 with A8R8G8B8, RGBA16F / RGBA32F as D3DFMT FourCC 113 / 116, RGB10A2 through the
 * 'DX10' extension header (dxgiFormat 24); one mip, tight rows.
 * host_image->data is HOST memory.  ovrfsr_dds_read allocates host_image->data (release with ovrfsr_host_free), so
 * a capture taken on a real D3D11 box can be diffed against this library's output. */
OVRFSR_API int ovrfsr_dds_write(const char *path, const ovrfsr_image *host_image);
OVRFSR_API int ovrfsr_dds_read(const char *path, ovrfsr_image *host_image);
OVRFSR_API void ovrfsr_host_free(void *p);

#ifdef __cplusplus
}
#endif
#endif /* OVRFSR_H */
