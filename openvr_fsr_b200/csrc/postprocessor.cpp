// postprocessor.cpp -- see postprocessor.h.  Mirrors the control flow of
// /root/reference/src/postprocess/PostProcessor.cpp:123-194: guard, lazy init from the Config singleton,
// "log once, disable, pass through" on failure, handle/colour-space swap on success.
#include "postprocessor.h"

#include <cmath>
#include <cstdio>
#include <iostream>

Config &Config::Instance() {
  static Config instance;
  return instance;
}

static std::ostream *g_log = nullptr;
std::ostream &Log() { return g_log ? *g_log : std::clog; }
void SetLogStream(std::ostream *os) { g_log = os; }

namespace vr {

static ovrfsr_config config_from_singleton() {
  const Config &c = Config::Instance();
  ovrfsr_config k;
  ovrfsr_config_default(&k);
  k.fsr_enabled = c.fsrEnabled;
  k.use_nis = c.useNis;
  k.render_scale = c.renderScale;
  k.sharpness = c.sharpness;
  k.radius = c.radius;
  k.debug_mode = c.debugMode;
  for (int i = 0; i < 4; ++i) k.proj_centre[i] = c.projCentre[i];
  k.device = c.cudaDevice;
  k.math_mode = c.strictMath ? OVRFSR_MATH_STRICT : OVRFSR_MATH_FAST;
  k.flags = c.fusedFsr ? OVRFSR_FLAG_FUSED_FSR : 0;
  return k;
}

PostProcessor::~PostProcessor() {
  if (ctx) ovrfsr_destroy(ctx);
}

void PostProcessor::Apply(EVREye eEye, const Texture_t *pTexture, const VRTextureBounds_t *pBounds,
                          EVRSubmitFlags /*nSubmitFlags*/) {
  if (!enabled || pTexture == nullptr || pTexture->eType != TextureType_OvrFsrCuda || pTexture->handle == nullptr) {
    return;
  }
  static VRTextureBounds_t defaultBounds{0, 0, 1, 1};
  if (pBounds == nullptr) {
    pBounds = &defaultBounds;
  }
  if (!Config::Instance().fsrEnabled) {
    return;
  }
  const ovrfsr_image *texture = static_cast<const ovrfsr_image *>(pTexture->handle);

  if (!initialized) {
    // the reference re-reads the Config singleton whenever it (re)creates resources
    const ovrfsr_config k = config_from_singleton();
    int rc = ctx ? ovrfsr_set_config(ctx, &k) : ovrfsr_create(&ctx, &k);
    if (rc != OVRFSR_OK) {
      Log() << "Resource creation failed, disabling (" << ovrfsr_status_string(rc) << ")\n";
      enabled = false;
      return;
    }
    // PostProcessor.cpp:504: Gamma, or Auto on a format OpenVR treats as sRGB (the _SRGB / _TYPELESS DXGI variants,
    // carried as tag bits of ovrfsr_image::format)
    inputIsSrgb = pTexture->eColorSpace == ColorSpace_Gamma ||
                  (pTexture->eColorSpace == ColorSpace_Auto && ovrfsr_format_considered_srgb(texture->format));
    Log() << "Creating post-processing resources\n";
    Log() << "Using " << (k.use_nis ? "NVIDIA Image Scaling" : "AMD FidelityFX SuperResolution") << "\n";
    initialized = true;
  }

  if (takeCapture) {
    takeCapture = false;
    ovrfsr_request_capture(ctx, captureDir);
  }
  const int onlyOneEye = std::abs(pBounds->uMax - pBounds->uMin) > .5f;
  const int eye = eEye == Eye_Right ? 1 : 0;
  ovrfsr_image out{};
  int rc;
  if (Config::Instance().honourTextureBounds) {
    // the bounds go on to the real Submit untouched: the output rectangle sits where they point
    const ovrfsr_bounds b{pBounds->uMin, pBounds->vMin, pBounds->uMax, pBounds->vMax};
    rc = ovrfsr_apply_bounds(ctx, eye, texture, &b, &out, nullptr, stream);
  } else {
    rc = ovrfsr_apply(ctx, eye, texture, onlyOneEye, &out, stream);
  }
  if (rc == OVRFSR_PASSTHROUGH) {
    return;
  }
  if (rc != OVRFSR_OK) {
    Log() << "Post-processing failed, disabling: " << ovrfsr_last_error(ctx) << "\n";
    enabled = false;
    return;
  }
  outputImage[eye] = out;
  const_cast<Texture_t *>(pTexture)->handle = &outputImage[eye];
  const_cast<Texture_t *>(pTexture)->eColorSpace = inputIsSrgb ? ColorSpace_Gamma : ColorSpace_Auto;
}

void PostProcessor::Reset() {
  enabled = true;
  initialized = false;
  if (ctx) ovrfsr_reset(ctx);
  outputImage[0] = outputImage[1] = ovrfsr_image{};
}

void PostProcessor::TakeCapture(const char *directory) {
  std::snprintf(captureDir, sizeof(captureDir), "%s", directory ? directory : "");
  takeCapture = true;
}

bool PostProcessor::GetAverageGpuTimeMs(float *ms) { return ctx && ovrfsr_get_gpu_time_ms(ctx, ms) > 0; }

} // namespace vr
