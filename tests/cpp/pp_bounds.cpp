// pp_bounds.cpp -- drives the C++ drop-in with Config::honourTextureBounds set: each eye is submitted with texture
// bounds, as a title with dynamic resolution or side-by-side eyes does, and the whole output image is written out.
// usage: pp_bounds <in.rgba> <w> <h> <renderScale> <sharpness> <radius> <useNis> <uMin> <vMin> <uMax> <vMax> <out.rgba>
// The right eye is submitted with the same bounds flipped vertically (vMin > vMax, OpenGL style), which selects the
// same rectangle.  Built and run by tests/test_gpu_cpp_bounds.py (nvcc, links the in-tree libovrfsr.so).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <sstream>
#include <vector>

#include <cuda_runtime.h>

#include "postprocessor.h"

static int fail(const char *what) { std::fprintf(stderr, "pp_bounds: %s\n", what); return 1; }

int main(int argc, char **argv) {
  if (argc != 13) return fail("bad arguments");
  const int w = std::atoi(argv[2]), h = std::atoi(argv[3]);
  std::vector<unsigned char> host((size_t)w * h * 4);
  FILE *f = std::fopen(argv[1], "rb");
  if (!f || std::fread(host.data(), 1, host.size(), f) != host.size()) return fail("cannot read input");
  std::fclose(f);

  std::ostringstream log;
  SetLogStream(&log);
  Config &cfg = Config::Instance();
  cfg.fsrEnabled = true;
  cfg.renderScale = (float)std::atof(argv[4]);
  cfg.sharpness = (float)std::atof(argv[5]);
  cfg.radius = (float)std::atof(argv[6]);
  cfg.useNis = std::atoi(argv[7]) != 0;
  cfg.strictMath = true;
  cfg.honourTextureBounds = true;
  const vr::VRTextureBounds_t bounds[2] = {
      {(float)std::atof(argv[8]), (float)std::atof(argv[9]), (float)std::atof(argv[10]), (float)std::atof(argv[11])},
      {(float)std::atof(argv[8]), (float)std::atof(argv[11]), (float)std::atof(argv[10]), (float)std::atof(argv[9])}};

  ovrfsr_image tex;
  if (ovrfsr_image_alloc(&tex, w, h, OVRFSR_FORMAT_RGBA8) != OVRFSR_OK) return fail("image alloc (no GPU?)");
  if (cudaMemcpy2D(tex.data, tex.pitch, host.data(), (size_t)w * 4, (size_t)w * 4, h, cudaMemcpyHostToDevice) != cudaSuccess)
    return fail("upload");

  vr::PostProcessor postProcessor;
  std::vector<unsigned char> res[2];
  for (int e = 0; e < 2; ++e) {
    vr::Texture_t t{&tex, vr::TextureType_OvrFsrCuda, vr::ColorSpace_Gamma};
    vr::VRTextureBounds_t b = bounds[e];
    postProcessor.Apply(e ? vr::Eye_Right : vr::Eye_Left, &t, &b, vr::Submit_Default);
    if (t.handle == &tex) { std::fputs(log.str().c_str(), stderr); return fail("Apply did not swap the handle"); }
    if (std::memcmp(&b, &bounds[e], sizeof(b)) != 0) return fail("Apply changed the bounds the real Submit gets");
    const ovrfsr_image *out = static_cast<const ovrfsr_image *>(t.handle);
    res[e].resize((size_t)out->width * out->height * 4);
    if (cudaMemcpy2D(res[e].data(), (size_t)out->width * 4, out->data, out->pitch, (size_t)out->width * 4, out->height,
                     cudaMemcpyDeviceToHost) != cudaSuccess)
      return fail("download");
    std::printf("eye %d: %ux%u\n", e, out->width, out->height);
  }
  FILE *o = std::fopen(argv[12], "wb");
  if (!o || std::fwrite(res[0].data(), 1, res[0].size(), o) != res[0].size() ||
      std::fwrite(res[1].data(), 1, res[1].size(), o) != res[1].size())
    return fail("cannot write output");
  std::fclose(o);
  ovrfsr_image_free(&tex);
  return 0;
}
