// config.h -- the process-wide Config singleton the hook layer reads
// (/root/reference/src/postprocess/Config.h:10-28,65-68), reduced to the fields that steer this path.
// Loading openvr_mod.cfg (jsoncpp, Win32 paths) stays with the mod; whoever owns the file fills this in.
#pragma once

#include "../../include/ovrfsr.h"

struct Config {
  bool fsrEnabled = false;
  bool applyMIPBias = true; // consumed by the D3D11 sampler hook (VrHooks.cpp:94-136), not by this path
  float renderScale = 1.f;
  float sharpness = 0.75f;
  float radius = 0.5f;
  bool debugMode = false;
  bool useNis = false;
  // not in the reference's Config: what it queries from the live runtime / picks implicitly
  float projCentre[4] = {0.5f, 0.5f, 0.5f, 0.5f}; // CalculateProjectionCenter, PostProcessor.cpp:104-121
  int cudaDevice = -1;
  bool strictMath = true;   // bit-identical to the reference lines (the library default); false = FMA-contracted kernels, <= 1 LSB per pass
  bool fusedFsr = false;    // OVRFSR_FLAG_FUSED_FSR: one fused EASU->RCAS kernel instead of the two dispatches
  // extension: post-process only the submitted VRTextureBounds_t rectangle of each eye (ovrfsr_apply_bounds) -- for
  // dynamic resolution and side-by-side eyes.  false = the reference, which filters the whole texture.
  bool honourTextureBounds = false;

  // ONE instance per process, owned by libovrfsr.so (an inline function-local static would be duplicated in every
  // module that includes this header when the library is built with hidden visibility)
  OVRFSR_API static Config &Instance();
};
