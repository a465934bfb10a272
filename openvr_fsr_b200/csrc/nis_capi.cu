// nis_capi.cu -- NIS half of include/ovrfsr.h: NISConfig setup, filter banks, NVScaler / NVSharpen dispatch.
#include <cstring>
#include <mutex>

#include "kernels.h"
#include "nis_host.h"
#include "nis_coef_table.inc"

using namespace ovrfsr;

namespace {
float g_coefScale[64][8], g_coefUsm[64][8]; // reference layout: 64 phases x kFilterSize(8), 6 used
std::once_flag g_coefOnce;
void expand_coef() {
  for (int p = 0; p < 64; ++p)
    for (int t = 0; t < 8; ++t) {
      g_coefScale[p][t] = t < 6 ? (float)(kNisCoefScale1e4[p][t] / 10000.0) : 0.0f;
      g_coefUsm[p][t] = t < 6 ? (float)(kNisCoefUsm1e4[p][t] / 10000.0) : 0.0f;
    }
}
} // namespace

extern "C" {

int ovrfsr_make_nis_config(void *cfg256, const ovrfsr_config *cfg, int sharpen_only, int eye, int only_one_eye,
                           uint32_t in_w, uint32_t in_h, uint32_t out_w, uint32_t out_h) {
  if (!cfg256 || !cfg) return 0;
  host::NisConfig c;
  const bool ok = host::make_nis_config(c, *cfg, sharpen_only != 0, eye, only_one_eye != 0, in_w, in_h, out_w, out_h);
  std::memcpy(cfg256, &c, sizeof(c));
  return ok ? 1 : 0;
}

const float *ovrfsr_nis_coef_scale(void) { std::call_once(g_coefOnce, expand_coef); return &g_coefScale[0][0]; }
const float *ovrfsr_nis_coef_usm(void) { std::call_once(g_coefOnce, expand_coef); return &g_coefUsm[0][0]; }

} // extern "C"

// ---- dispatches (ApplyUpscaling / ApplySharpening with useNis, PostProcessor.cpp:385-401,483-496) ------------
namespace {
inline uint32_t bpp(int fmt) { return fmt == OVRFSR_FORMAT_RGBA32F ? 16u : (fmt == OVRFSR_FORMAT_RGBA16F ? 8u : 4u); }
int check(const ovrfsr_image *im, bool isDst) {
  if (!im || !im->data || im->width == 0 || im->height == 0) return OVRFSR_ERR_INVALID;
  if (im->format < OVRFSR_FORMAT_RGBA8 || im->format > OVRFSR_FORMAT_BGRX8) return OVRFSR_ERR_UNSUPPORTED; /* RGB32F: expand first */
  if ((isDst && (im->format == OVRFSR_FORMAT_BGRA8 || im->format == OVRFSR_FORMAT_BGRX8)) || im->sample_count > 1) return OVRFSR_ERR_UNSUPPORTED;
  if (im->pitch < im->width * bpp(im->format) || im->pitch % bpp(im->format) ||
      reinterpret_cast<uintptr_t>(im->data) % bpp(im->format)) return OVRFSR_ERR_INVALID;
  return OVRFSR_OK;
}
PassImage pass(const ovrfsr_image &im) { return PassImage{im.data, im.pitch, (int)im.width, (int)im.height, im.format}; }
int status_of(cudaError_t e) {
  if (e == cudaSuccess) return OVRFSR_OK;
  return (e == cudaErrorInvalidConfiguration || e == cudaErrorInvalidValue) ? OVRFSR_ERR_UNSUPPORTED : OVRFSR_ERR_CUDA;
}
} // namespace

cudaError_t ovrfsr::launch_nis(bool sharpen, const PassImage &src, const PassImage &dst, const void *cfg256, int math_mode,
                               cudaStream_t s) {
  static float both[2][64 * 8];
  static std::once_flag once;
  std::call_once(once, [&] { std::memcpy(both[0], ovrfsr_nis_coef_scale(), sizeof(both[0])); std::memcpy(both[1], ovrfsr_nis_coef_usm(), sizeof(both[1])); });
  const bool strict = math_mode == OVRFSR_MATH_STRICT;
  if (sharpen) return strict ? launch_nis_sharpen_strict(src, dst, cfg256, nullptr, s) : launch_nis_sharpen_fast(src, dst, cfg256, nullptr, s);
  return strict ? launch_nis_scaler_strict(src, dst, cfg256, &both[0][0], s) : launch_nis_scaler_fast(src, dst, cfg256, &both[0][0], s);
}

extern "C" {

int ovrfsr_dispatch_nis_scaler(const ovrfsr_image *src, const ovrfsr_image *dst, const void *cfg256, int math_mode,
                               void *stream) {
  ovrfsr_image src_untagged_{};
  if (src) { src_untagged_ = *src; if (src_untagged_.format >= 0) src_untagged_.format &= OVRFSR_FORMAT_LAYOUT_MASK; src = &src_untagged_; }
  if (!cfg256) return OVRFSR_ERR_INVALID;
  int rc = check(src, false);
  if (rc != OVRFSR_OK || (rc = check(dst, true)) != OVRFSR_OK) return rc;
  return status_of(launch_nis(false, pass(*src), pass(*dst), cfg256, math_mode, static_cast<cudaStream_t>(stream)));
}

int ovrfsr_dispatch_nis_sharpen(const ovrfsr_image *src, const ovrfsr_image *dst, const void *cfg256, int math_mode,
                                void *stream) {
  ovrfsr_image src_untagged_{};
  if (src) { src_untagged_ = *src; if (src_untagged_.format >= 0) src_untagged_.format &= OVRFSR_FORMAT_LAYOUT_MASK; src = &src_untagged_; }
  if (!cfg256) return OVRFSR_ERR_INVALID;
  int rc = check(src, false);
  if (rc != OVRFSR_OK || (rc = check(dst, true)) != OVRFSR_OK) return rc;
  if (src->width != dst->width || src->height != dst->height) return OVRFSR_ERR_INVALID;
  return status_of(launch_nis(true, pass(*src), pass(*dst), cfg256, math_mode, static_cast<cudaStream_t>(stream)));
}

} // extern "C"
