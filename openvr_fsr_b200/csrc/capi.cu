// capi.cu -- implementation of include/ovrfsr.h: the state machine of vr::PostProcessor
// (src/postprocess/PostProcessor.cpp:123-194,498-638 in /root/reference) over CUDA resources,
// plus the stateless per-dispatch entry points.  No CPU fallback exists: if CUDA is unusable the
// calls fail with OVRFSR_ERR_CUDA.
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <new>
#include <ctime>
#include <string>
#include <vector>

#include "host_constants.h"
#include "kernels.h"

namespace ovrfsr {
static std::atomic<uint64_t> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
} // namespace ovrfsr

using namespace ovrfsr;

namespace {

constexpr int kQueryCount = 6; // QUERY_COUNT, PostProcessor.h:78

inline uint32_t bytes_per_pixel(int fmt) {
  return fmt == OVRFSR_FORMAT_RGBA32F ? 16u : (fmt == OVRFSR_FORMAT_RGB32F ? 12u : (fmt == OVRFSR_FORMAT_RGBA16F ? 8u : 4u));
}
inline bool valid_format(int fmt) { return fmt >= OVRFSR_FORMAT_RGBA8 && fmt <= OVRFSR_FORMAT_RGB32F; }
// the DXGI variant tags (_SRGB / _TYPELESS) change no pixel on this path: strip them at the boundary
inline ovrfsr_image untagged(const ovrfsr_image *im) {
  ovrfsr_image r = *im;
  if (r.format >= 0) r.format &= OVRFSR_FORMAT_LAYOUT_MASK;
  return r;
}
inline uint32_t align_up(uint32_t v, uint32_t a) { return (v + a - 1) / a * a; }

struct DeviceImage {
  ovrfsr_image img{};
  bool alloc(uint32_t w, uint32_t h, int fmt) {
    release();
    img.width = w; img.height = h; img.format = fmt; img.array_slices = 1; img.slice_pitch = 0;
    img.pitch = align_up(w * bytes_per_pixel(fmt), 256u);
    return cudaMalloc(&img.data, (size_t)img.pitch * h) == cudaSuccess;
  }
  void release() {
    if (img.data) cudaFree(img.data);
    img = ovrfsr_image{};
  }
};

// linear device scratch for the host entry: PCIe copies are issued as ONE contiguous cudaMemcpyAsync each way
// (2-D pitched copies in opposite directions were measured not to overlap on B200: 795 pairs/s vs 1100) and a
// small kernel moves rows between the tight host layout and the 256-byte-pitched device images.
struct DeviceBuffer {
  void *ptr = nullptr;
  size_t bytes = 0;
  bool ensure(size_t n) {
    if (n <= bytes) return true;
    release();
    if (cudaMalloc(&ptr, n) != cudaSuccess) { ptr = nullptr; return false; }
    bytes = n;
    return true;
  }
  void release() {
    if (ptr) cudaFree(ptr);
    ptr = nullptr; bytes = 0;
  }
};

// rows of `rowWords` 32-bit words from pitch `spitch` to pitch `dpitch` (bytes, multiples of 4); HBM-bound, ~10 us/eye
__global__ void __launch_bounds__(256) repitch_rows_kernel(uint8_t *__restrict__ dst, size_t dpitch, const uint8_t *__restrict__ src,
                                                           size_t spitch, uint32_t rowWords, uint32_t rows) {
  for (uint32_t y = blockIdx.y; y < rows; y += gridDim.y) {
    const uint32_t *s = reinterpret_cast<const uint32_t *>(src + (size_t)y * spitch);
    uint32_t *d = reinterpret_cast<uint32_t *>(dst + (size_t)y * dpitch);
    for (uint32_t x = blockIdx.x * blockDim.x + threadIdx.x; x < rowWords; x += gridDim.x * blockDim.x) d[x] = s[x];
  }
}

cudaError_t repitch_rows(void *dst, size_t dpitch, const void *src, size_t spitch, size_t rowBytes, uint32_t rows, cudaStream_t s) {
  const uint32_t rowWords = (uint32_t)(rowBytes / 4);
  dim3 grid((rowWords + 1023) / 1024, rows < 4096 ? rows : 4096);
  repitch_rows_kernel<<<grid, 256, 0, s>>>(static_cast<uint8_t *>(dst), dpitch, static_cast<const uint8_t *>(src), spitch, rowWords, rows);
  count_launch();
  return cudaGetLastError();
}

// R32G32B32_FLOAT -> RGBA32F, alpha 1 (a three-component view reads 1 in .w)
__global__ void __launch_bounds__(256) expand_rgb32f_kernel(float4 *__restrict__ dst, size_t dpitch, const float *__restrict__ src, size_t spitch,
                                                            uint32_t w, uint32_t h) {
  const uint32_t x = blockIdx.x * 256 + threadIdx.x, y = blockIdx.y;
  if (x >= w || y >= h) return;
  const float *s = reinterpret_cast<const float *>(reinterpret_cast<const uint8_t *>(src) + (size_t)y * spitch) + 3 * (size_t)x;
  reinterpret_cast<float4 *>(reinterpret_cast<uint8_t *>(dst) + (size_t)y * dpitch)[x] = make_float4(s[0], s[1], s[2], 1.0f);
}
cudaError_t expand_rgb32f(const ovrfsr_image &src, const ovrfsr_image &dst, cudaStream_t s) {
  const dim3 grid((src.width + 255) / 256, src.height);
  expand_rgb32f_kernel<<<grid, 256, 0, s>>>(static_cast<float4 *>(dst.data), dst.pitch, static_cast<const float *>(src.data), src.pitch,
                                              src.width, src.height);
  count_launch();
  return cudaGetLastError();
}

PassImage pass_image(const ovrfsr_image &im, int slice = 0) {
  PassImage p;
  p.ptr = static_cast<uint8_t *>(im.data) + (size_t)slice * im.slice_pitch;
  p.pitch = im.pitch; p.w = (int)im.width; p.h = (int)im.height; p.format = im.format;
  return p;
}
// the rectangle r of the whole image t (nullptr: all of it)
PassImage crop(const PassImage &t, const ovrfsr_rect *r) {
  if (!r) return t;
  PassImage p = t;
  p.ptr = static_cast<uint8_t *>(t.ptr) + (size_t)r->y * t.pitch + (size_t)r->x * bytes_per_pixel(t.format);
  p.w = (int)r->width; p.h = (int)r->height;
  p.x0 = (int)r->x; p.y0 = (int)r->y; p.texW = t.w; p.texH = t.h;
  return p;
}
inline bool same_rect(const ovrfsr_rect &a, const ovrfsr_rect &b) {
  return a.x == b.x && a.y == b.y && a.width == b.width && a.height == b.height;
}

// the constant blocks one apply runs with
struct EyeConsts {
  const uint32_t *upscale, *sharpen;
  const uint8_t *nisScaler, *nisSharpen;
};

} // namespace

struct ovrfsr_ctx {
  ovrfsr_config cfg{};
  // PostProcessor.h:16-24
  bool enabled = true;
  bool initialized = false;
  uint32_t inputWidth = 0, inputHeight = 0, outputWidth = 0, outputHeight = 0;
  bool textureContainsOnlyOneEye = true;
  int outFormat = OVRFSR_FORMAT_RGBA8;
  int inFormat = OVRFSR_FORMAT_RGBA8;
  // per-eye constant blocks (upscaleConstantsBuffer[2] / sharpenConstantsBuffer[2], PostProcessor.h:41,56)
  uint32_t upscaleConstants[2][24]{};
  uint32_t sharpenConstants[2][12]{};
  alignas(16) uint8_t nisScalerConfig[2][256]{};
  alignas(16) uint8_t nisSharpenConfig[2][256]{};
  // ovrfsr_apply_bounds: per eye, the last rectangles and the constant blocks built for them (beside the full-texture
  // ones above, so that ovrfsr_apply and ovrfsr_apply_bounds can be mixed on one ctx)
  struct BoundsEye {
    bool valid = false;
    ovrfsr_rect src{}, dst{};
    uint32_t upscale[24]{}, sharpen[12]{};
    alignas(16) uint8_t nisScaler[256]{}, nisSharpen[256]{};
  } bounds[2];
  // one set of intermediates/outputs PER EYE (the reference shares one; see ovrfsr.h)
  DeviceImage upscaled[2], sharpened[2];
  DeviceImage hostStage[2]; // device staging of host-submitted eyes (ovrfsr_apply_host)
  DeviceBuffer hostLinearIn[2], hostLinearOut[2];
  DeviceImage resolved[2];  // copiedTexture (PostProcessor.h:29): the resolved copy of a multisampled source
  DeviceImage expanded[2];  // RGBA32F copy of an R32G32B32_FLOAT source
  // F7 capture (takeCapture, PostProcessor.h:88 / PostProcessor.cpp:630-637)
  bool takeCapture = false;
  std::string captureDir, lastCapturePath;
  const void *lastSubmittedTexture = nullptr;
  ovrfsr_image lastOutput{};
  int eyeCount = 0;
  // debugMode profiling ring (PostProcessor.h:72-82)
  cudaEvent_t evStart[kQueryCount]{}, evEnd[kQueryCount]{};
  bool evPending[kQueryCount]{};
  bool evCreated = false;
  int currentQuery = 0;
  float summedGpuTime = 0.f;
  int countedQueries = 0;
  // ovrfsr_apply_pair: the right eye's chain runs on this stream between a fork and a join event
  cudaStream_t pairStream = nullptr;
  cudaEvent_t pairFork = nullptr, pairJoin = nullptr;
  std::string lastError;
};

namespace {

int fail(ovrfsr_ctx *ctx, int status, const char *what, cudaError_t e = cudaSuccess) {
  if (ctx) {
    ctx->lastError = what;
    if (e != cudaSuccess) { ctx->lastError += ": "; ctx->lastError += cudaGetErrorString(e); }
  }
  return status;
}

void release_resources(ovrfsr_ctx *c) {
  for (int e = 0; e < 2; ++e) { c->upscaled[e].release(); c->sharpened[e].release(); c->hostStage[e].release(); c->hostLinearIn[e].release(); c->hostLinearOut[e].release(); c->resolved[e].release(); c->expanded[e].release(); }
  if (c->evCreated) {
    for (int i = 0; i < kQueryCount; ++i) { cudaEventDestroy(c->evStart[i]); cudaEventDestroy(c->evEnd[i]); c->evPending[i] = false; }
    c->evCreated = false;
  }
}

int select_device(ovrfsr_ctx *c) {
  if (c->cfg.device >= 0) {
    cudaError_t e = cudaSetDevice(c->cfg.device);
    if (e != cudaSuccess) return fail(c, OVRFSR_ERR_CUDA, "cudaSetDevice", e);
  }
  return OVRFSR_OK;
}

bool upscale_pass(const ovrfsr_config &cfg) { return cfg.render_scale != 1.f; }                    // PostProcessor.cpp:586
bool sharpen_pass(const ovrfsr_config &cfg) { return !cfg.use_nis || cfg.render_scale == 1.f; }    // PostProcessor.cpp:591
// both FSR passes run and the caller opted into the fused kernel (the intermediate is then never materialised)
bool fused_pass(const ovrfsr_config &cfg) {
  return !cfg.use_nis && upscale_pass(cfg) && sharpen_pass(cfg) && (cfg.flags & OVRFSR_FLAG_FUSED_FSR);
}

// PostProcessor::PrepareResources, PostProcessor.cpp:498-561
int prepare_resources(ovrfsr_ctx *c, const ovrfsr_image *src) {
  c->inputWidth = src->width;
  c->inputHeight = src->height;
  c->inFormat = src->format;
  host::output_size(src->width, src->height, c->cfg.render_scale, &c->outputWidth, &c->outputHeight);
  if (c->outputWidth == 0 || c->outputHeight == 0) return fail(c, OVRFSR_ERR_INVALID, "output size is zero");
  // DetermineOutputFormat (PostProcessor.cpp:63-74): 10-bit sources keep a 10-bit target, everything else gets
  // RGBA8, unless the caller asks for a float output (extension)
  const bool tenBit = src->format == OVRFSR_FORMAT_RGB10A2;
  c->outFormat = c->cfg.output_format == OVRFSR_FORMAT_AUTO ? (tenBit ? OVRFSR_FORMAT_RGB10A2 : OVRFSR_FORMAT_RGBA8) : c->cfg.output_format;
  if (c->outFormat != OVRFSR_FORMAT_RGBA16F && c->outFormat != OVRFSR_FORMAT_RGBA32F &&
      c->outFormat != (tenBit ? OVRFSR_FORMAT_RGB10A2 : OVRFSR_FORMAT_RGBA8))
    return fail(c, OVRFSR_ERR_UNSUPPORTED, tenBit ? "output format for an RGB10A2 source must be RGB10A2, RGBA16F or RGBA32F"
                                                  : "output format must be RGBA8, RGBA16F or RGBA32F");
  const bool one = c->textureContainsOnlyOneEye;
  const int neyes = one ? 2 : 1;
  for (int e = 0; e < neyes; ++e) {
    host::make_upscale_constants(c->upscaleConstants[e], c->cfg, e, one, c->inputWidth, c->inputHeight, c->outputWidth,
                                 c->outputHeight);
    host::make_sharpen_constants(c->sharpenConstants[e], c->cfg, e, one, c->outputWidth, c->outputHeight);
    ovrfsr_make_nis_config(c->nisScalerConfig[e], &c->cfg, 0, e, one, c->inputWidth, c->inputHeight, c->outputWidth,
                           c->outputHeight);
    ovrfsr_make_nis_config(c->nisSharpenConfig[e], &c->cfg, 1, e, one, c->inputWidth, c->inputHeight, c->outputWidth,
                           c->outputHeight);
    // the upscaled image only exists when the two dispatches run (the fused kernel keeps it in shared memory; if a
    // shape turns out not to be fusable it is allocated on first use)
    const bool wantMid = upscale_pass(c->cfg) && !(fused_pass(c->cfg) && (c->outFormat == OVRFSR_FORMAT_RGBA8 || c->outFormat == OVRFSR_FORMAT_RGB10A2));
    if (wantMid && !c->upscaled[e].alloc(c->outputWidth, c->outputHeight, c->outFormat))
      return fail(c, OVRFSR_ERR_NOMEM, "allocating upscaled texture", cudaGetLastError());
    if (sharpen_pass(c->cfg) && !c->sharpened[e].alloc(c->outputWidth, c->outputHeight, c->outFormat))
      return fail(c, OVRFSR_ERR_NOMEM, "allocating sharpened texture", cudaGetLastError());
  }
  if (c->cfg.debug_mode) {
    for (int i = 0; i < kQueryCount; ++i) {
      if (cudaEventCreate(&c->evStart[i]) != cudaSuccess || cudaEventCreate(&c->evEnd[i]) != cudaSuccess)
        return fail(c, OVRFSR_ERR_CUDA, "creating profiling events", cudaGetLastError());
      c->evPending[i] = false;
    }
    c->evCreated = true;
  }
  c->initialized = true;
  return OVRFSR_OK;
}

// harvest finished profiling samples (the GetData loop of PostProcessor.cpp:601-628, non-blocking)
void harvest_queries(ovrfsr_ctx *c) {
  if (!c->evCreated) return;
  for (int i = 0; i < kQueryCount; ++i) {
    if (!c->evPending[i] || cudaEventQuery(c->evEnd[i]) != cudaSuccess) continue;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, c->evStart[i], c->evEnd[i]) == cudaSuccess) { c->summedGpuTime += ms; ++c->countedQueries; }
    c->evPending[i] = false;
  }
}

// EASU followed by RCAS in one apply with a UNORM target: EASU writes the outside-radius groups straight to the final
// image and RCAS only visits what is inside the radius (kernels.h)
bool paired_passes(const ovrfsr_ctx *c) {
  static const bool off = getenv("OVRFSR_NO_PAIR") != nullptr; // dev A/B switch
  return !off && !c->cfg.use_nis && upscale_pass(c->cfg) && sharpen_pass(c->cfg) &&
         (c->outFormat == OVRFSR_FORMAT_RGBA8 || c->outFormat == OVRFSR_FORMAT_RGB10A2);
}

int nis_status(cudaError_t e) {
  if (e == cudaSuccess) return OVRFSR_OK;
  return (e == cudaErrorInvalidConfiguration || e == cudaErrorInvalidValue) ? OVRFSR_ERR_UNSUPPORTED : OVRFSR_ERR_CUDA;
}

// `fin` = the final image (the output rectangle of the sharpened texture): the paired EASU writes its outside-radius
// groups there
int run_upscale(ovrfsr_ctx *c, const EyeConsts &k, const PassImage &in, const PassImage &out, const PassImage &fin, cudaStream_t s) {
  const bool strict = c->cfg.math_mode == OVRFSR_MATH_STRICT;
  cudaError_t e;
  if (c->cfg.use_nis) {
    int rc = nis_status(launch_nis(false, in, out, k.nisScaler, c->cfg.math_mode, s));
    return rc == OVRFSR_OK ? rc : fail(c, rc, "NIS scaler dispatch");
  }
  const PassImage *direct = paired_passes(c) ? &fin : nullptr;
  const float tint = 1.0f - (float)k.sharpen[3] * 0.3f;
  e = strict ? launch_easu_strict(in, out, k.upscale, s, direct, tint) : launch_easu_fast(in, out, k.upscale, s, direct, tint);
  return e == cudaSuccess ? OVRFSR_OK : fail(c, OVRFSR_ERR_CUDA, "EASU launch", e);
}

int run_sharpen(ovrfsr_ctx *c, const EyeConsts &k, const PassImage &in, const PassImage &out, cudaStream_t s) {
  const bool strict = c->cfg.math_mode == OVRFSR_MATH_STRICT;
  if (c->cfg.use_nis) {
    int rc = nis_status(launch_nis(true, in, out, k.nisSharpen, c->cfg.math_mode, s));
    return rc == OVRFSR_OK ? rc : fail(c, rc, "NIS sharpen dispatch");
  }
  const bool skip = paired_passes(c);
  cudaError_t e = strict ? launch_rcas_strict(in, out, k.sharpen, s, skip) : launch_rcas_fast(in, out, k.sharpen, s, skip);
  return e == cudaSuccess ? OVRFSR_OK : fail(c, OVRFSR_ERR_CUDA, "RCAS launch", e);
}

// PostProcessor::SaveTextureToFile, PostProcessor.cpp:640-657: staging copy, then the DDS writer (capture.cpp)
int save_capture(ovrfsr_ctx *c, const ovrfsr_image &img, cudaStream_t s) {
  const size_t rowBytes = (size_t)img.width * bytes_per_pixel(img.format);
  std::vector<uint8_t> host(rowBytes * img.height);
  cudaError_t e = cudaMemcpy2DAsync(host.data(), rowBytes, img.data, img.pitch, rowBytes, img.height, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) return fail(c, OVRFSR_ERR_CUDA, "capture read-back", e);
  char name[96];
  if (ovrfsr_capture_filename(&c->cfg, (int64_t)std::time(nullptr), name, sizeof(name)) != OVRFSR_OK)
    return fail(c, OVRFSR_ERR_INVALID, "capture file name");
  c->lastCapturePath = c->captureDir.empty() ? std::string(name) : c->captureDir + "/" + name;
  const ovrfsr_image h{host.data(), img.width, img.height, (uint32_t)rowBytes, img.format, 1, 0, 0};
  int rc = ovrfsr_dds_write(c->lastCapturePath.c_str(), &h);
  if (rc != OVRFSR_OK) { c->lastCapturePath.clear(); return fail(c, rc, "Error taking screen capture"); }
  return OVRFSR_OK;
}

// PostProcessor::ApplyPostProcess, PostProcessor.cpp:563-638 (the D3D11 binding save/restore and the Win32 hotkey
// polling stay in the caller; the F7 capture is served through ovrfsr_request_capture).
// srcRect / dstRect (ovrfsr_apply_bounds, nullptr = the whole images): the passes read the source rectangle of the
// (resolved / expanded / sliced) eye texture and write the output rectangle of the ctx images; `k` holds the constants
// built for those sizes.
int apply_post_process(ovrfsr_ctx *c, int eye, const ovrfsr_image *src, ovrfsr_image *out, cudaStream_t s, const EyeConsts &k,
                       const ovrfsr_rect *srcRect = nullptr, const ovrfsr_rect *dstRect = nullptr) {
  // GetInputView: array textures keep the right eye in slice 1 (PostProcessor.cpp:254-268)
  const int slice = (src->array_slices > 1 && eye == 1) ? 1 : 0;
  PassImage in = pass_image(*src, slice);
  ovrfsr_image result = *src;
  if (src->sample_count > 1) { // GetInputView: multisampled sources are resolved into copiedTexture first (:219-226)
    DeviceImage &r = c->resolved[eye];
    if ((!r.img.data || r.img.width != src->width || r.img.height != src->height || r.img.format != src->format) &&
        !r.alloc(src->width, src->height, src->format))
      return fail(c, OVRFSR_ERR_NOMEM, "allocating the MSAA resolve target", cudaGetLastError());
    cudaError_t e = launch_resolve_msaa(in, (int)src->sample_count, pass_image(r.img), s);
    if (e != cudaSuccess) return fail(c, OVRFSR_ERR_CUDA, "MSAA resolve launch", e);
    in = pass_image(r.img);
    result = r.img;
  }
  if (src->format == OVRFSR_FORMAT_RGB32F) { // three-component float source: the kernels read it through an RGBA32F copy
    if (src->sample_count > 1) return fail(c, OVRFSR_ERR_UNSUPPORTED, "multisampled R32G32B32_FLOAT source");
    DeviceImage &x = c->expanded[eye];
    if ((!x.img.data || x.img.width != src->width || x.img.height != src->height) && !x.alloc(src->width, src->height, OVRFSR_FORMAT_RGBA32F))
      return fail(c, OVRFSR_ERR_NOMEM, "allocating the RGBA32F copy of an RGB32F source", cudaGetLastError());
    ovrfsr_image sl = *src;
    sl.data = static_cast<uint8_t *>(src->data) + (size_t)slice * src->slice_pitch;
    cudaError_t e = expand_rgb32f(sl, x.img, s);
    if (e != cudaSuccess) return fail(c, OVRFSR_ERR_CUDA, "RGB32F expansion launch", e);
    in = pass_image(x.img);
    result = x.img;
  }
  in = crop(in, srcRect);
  int q = -1;
  if (c->evCreated) {
    harvest_queries(c);
    q = c->currentQuery;
    c->currentQuery = (c->currentQuery + 1) % kQueryCount;
    if (c->evPending[q]) q = -1; // oldest sample still in flight: skip this frame rather than block
    else cudaEventRecord(c->evStart[q], s);
  }
  bool fused = false;
  if (fused_pass(c->cfg) && (c->outFormat == OVRFSR_FORMAT_RGBA8 || c->outFormat == OVRFSR_FORMAT_RGB10A2)) {
    // ApplyUpscaling + ApplySharpening (PostProcessor.cpp:586-594) as one kernel; shapes it does not cover take the
    // two dispatches below
    const bool strict = c->cfg.math_mode == OVRFSR_MATH_STRICT;
    const PassImage out2 = crop(pass_image(c->sharpened[eye].img), dstRect);
    const cudaError_t e = strict ? launch_fsr_fused_strict(in, out2, k.upscale, k.sharpen, s) : launch_fsr_fused_fast(in, out2, k.upscale, k.sharpen, s);
    if (e == cudaSuccess) { fused = true; result = c->sharpened[eye].img; }
    else if (e != cudaErrorInvalidValue && e != cudaErrorInvalidConfiguration) return fail(c, OVRFSR_ERR_CUDA, "fused EASU+RCAS launch", e);
  }
  if (!fused && upscale_pass(c->cfg)) {
    if (!c->upscaled[eye].img.data && !c->upscaled[eye].alloc(c->outputWidth, c->outputHeight, c->outFormat))
      return fail(c, OVRFSR_ERR_NOMEM, "allocating upscaled texture", cudaGetLastError());
    const PassImage mid = crop(pass_image(c->upscaled[eye].img), dstRect);
    int rc = run_upscale(c, k, in, mid, crop(pass_image(c->sharpened[eye].img), dstRect), s);
    if (rc != OVRFSR_OK) return rc;
    in = mid;
    result = c->upscaled[eye].img;
  }
  if (!fused && sharpen_pass(c->cfg)) {
    int rc = run_sharpen(c, k, in, crop(pass_image(c->sharpened[eye].img), dstRect), s);
    if (rc != OVRFSR_OK) return rc;
    result = c->sharpened[eye].img;
  }
  if (q >= 0) { cudaEventRecord(c->evEnd[q], s); c->evPending[q] = true; }
  *out = result;
  if (c->takeCapture && eye == 0) { // PostProcessor.cpp:634-637
    c->takeCapture = false;
    int rc = save_capture(c, result, s);
    if (rc != OVRFSR_OK) return rc;
  }
  return OVRFSR_OK;
}

int validate_image(const ovrfsr_image *im) {
  if (!im || !im->data || im->width == 0 || im->height == 0) return OVRFSR_ERR_INVALID;
  if (!valid_format(im->format)) return OVRFSR_ERR_UNSUPPORTED;
  const uint64_t rowEntries = (uint64_t)im->width * (im->sample_count > 1 ? im->sample_count : 1u);
  // rows and the base are aligned to the texel (to its 4-byte components for the 12-byte R32G32B32_FLOAT texel)
  const uint32_t align = im->format == OVRFSR_FORMAT_RGB32F ? 4u : bytes_per_pixel(im->format);
  if (im->sample_count > 32 || im->pitch < rowEntries * bytes_per_pixel(im->format) || (im->pitch % align) != 0) return OVRFSR_ERR_INVALID;
  if ((reinterpret_cast<uintptr_t>(im->data) % align) != 0) return OVRFSR_ERR_INVALID;
  return OVRFSR_OK;
}

} // namespace

extern "C" {

void ovrfsr_config_default(ovrfsr_config *cfg) {
  if (!cfg) return;
  std::memset(cfg, 0, sizeof(*cfg));
  cfg->struct_size = sizeof(ovrfsr_config);
  cfg->fsr_enabled = 0;   // Config.h:11
  cfg->use_nis = 0;       // Config.h:17
  cfg->render_scale = 1.f;
  cfg->sharpness = 0.75f;
  cfg->radius = 0.5f;
  cfg->debug_mode = 0;
  cfg->proj_centre[0] = cfg->proj_centre[1] = cfg->proj_centre[2] = cfg->proj_centre[3] = 0.5f;
  cfg->device = -1;
  cfg->output_format = OVRFSR_FORMAT_AUTO;
  cfg->math_mode = OVRFSR_MATH_STRICT; // parity first: bit-identical to the reference lines end to end
}

int ovrfsr_create(ovrfsr_ctx **out, const ovrfsr_config *cfg) {
  if (!out || !cfg || cfg->struct_size != sizeof(ovrfsr_config)) return OVRFSR_ERR_INVALID;
  if (!(cfg->render_scale > 0.f)) return OVRFSR_ERR_INVALID;
  ovrfsr_ctx *c = new (std::nothrow) ovrfsr_ctx();
  if (!c) return OVRFSR_ERR_NOMEM;
  c->cfg = *cfg;
  *out = c;
  return OVRFSR_OK;
}

void ovrfsr_destroy(ovrfsr_ctx *ctx) {
  if (ctx && ctx->pairStream) {
    cudaStreamSynchronize(ctx->pairStream);
    cudaEventDestroy(ctx->pairFork);
    cudaEventDestroy(ctx->pairJoin);
    cudaStreamDestroy(ctx->pairStream);
  }
  if (!ctx) return;
  if (ctx->initialized || ctx->hostStage[0].img.data || ctx->hostStage[1].img.data) {
    if (ctx->cfg.device >= 0) cudaSetDevice(ctx->cfg.device);
    release_resources(ctx);
  }
  delete ctx;
}

int ovrfsr_reset(ovrfsr_ctx *ctx) {
  if (!ctx) return OVRFSR_ERR_INVALID;
  if (ctx->initialized) {
    if (ctx->cfg.device >= 0) cudaSetDevice(ctx->cfg.device);
    cudaDeviceSynchronize(); // outputs may still be in flight on the caller's stream
    release_resources(ctx);
  }
  ctx->enabled = true;
  ctx->initialized = false;
  ctx->bounds[0].valid = ctx->bounds[1].valid = false;
  ctx->lastSubmittedTexture = nullptr;
  ctx->lastOutput = ovrfsr_image{};
  ctx->eyeCount = 0;
  ctx->currentQuery = 0;
  ctx->summedGpuTime = 0.f;
  ctx->countedQueries = 0;
  return OVRFSR_OK;
}

int ovrfsr_set_config(ovrfsr_ctx *ctx, const ovrfsr_config *cfg) {
  if (!ctx || !cfg || cfg->struct_size != sizeof(ovrfsr_config) || !(cfg->render_scale > 0.f)) return OVRFSR_ERR_INVALID;
  int rc = ovrfsr_reset(ctx);
  ctx->cfg = *cfg;
  return rc;
}

int ovrfsr_get_config(const ovrfsr_ctx *ctx, ovrfsr_config *cfg) {
  if (!ctx || !cfg) return OVRFSR_ERR_INVALID;
  *cfg = ctx->cfg;
  return OVRFSR_OK;
}

int ovrfsr_apply(ovrfsr_ctx *ctx, int eye, const ovrfsr_image *src_tagged, int only_one_eye, ovrfsr_image *out, void *stream) {
  if (!ctx || !out || (eye != 0 && eye != 1)) return OVRFSR_ERR_INVALID;
  ovrfsr_image src_untagged{};
  if (src_tagged) src_untagged = untagged(src_tagged);
  const ovrfsr_image *src = src_tagged ? &src_untagged : nullptr;
  // PostProcessor.cpp:124: disabled or unusable texture -> the frame passes through untouched
  if (!ctx->enabled || !ctx->cfg.fsr_enabled) return OVRFSR_PASSTHROUGH;
  int rc = validate_image(src);
  if (rc != OVRFSR_OK) return fail(ctx, rc, "invalid source image");
  if ((rc = select_device(ctx)) != OVRFSR_OK) return rc;
  if (ctx->initialized && (src->width != ctx->inputWidth || src->height != ctx->inputHeight || src->format != ctx->inFormat)) {
    ovrfsr_reset(ctx); // "Texture size changed, recreating resources", PostProcessor.cpp:139-142
  }
  if (!ctx->initialized) {
    ctx->textureContainsOnlyOneEye = only_one_eye != 0; // PostProcessor.cpp:146
    rc = prepare_resources(ctx, src);
    if (rc != OVRFSR_OK) { // PostProcessor.cpp:148-152: "Resource creation failed, disabling"
      release_resources(ctx);
      ctx->enabled = false;
      return rc;
    }
  }
  // a single shared texture for both eyes is processed on the first Submit only (PostProcessor.cpp:155-160)
  if (ctx->eyeCount == 0 || ctx->textureContainsOnlyOneEye || src->data != ctx->lastSubmittedTexture) {
    const int e = ctx->textureContainsOnlyOneEye ? eye : 0;
    const EyeConsts k{ctx->upscaleConstants[e], ctx->sharpenConstants[e], ctx->nisScalerConfig[e], ctx->nisSharpenConfig[e]};
    rc = apply_post_process(ctx, e, src, &ctx->lastOutput, static_cast<cudaStream_t>(stream), k);
    if (rc != OVRFSR_OK) return rc;
  }
  ctx->lastSubmittedTexture = src->data;
  ctx->eyeCount = (ctx->eyeCount + 1) % 2;
  *out = ctx->lastOutput;
  return OVRFSR_OK;
}

int ovrfsr_bounds_rects(uint32_t w, uint32_t h, uint32_t out_w, uint32_t out_h, const ovrfsr_bounds *bounds,
                        ovrfsr_rect *src_rect, ovrfsr_rect *dst_rect) {
  const ovrfsr_bounds whole{0.f, 0.f, 1.f, 1.f};
  const ovrfsr_bounds &b = bounds ? *bounds : whole;
  if (std::isnan(b.u_min) || std::isnan(b.v_min) || std::isnan(b.u_max) || std::isnan(b.v_max)) return OVRFSR_ERR_INVALID;
  const auto unit = [](float t) { return t < 0.f ? 0.f : (t > 1.f ? 1.f : t); };
  const float u0 = unit(std::fmin(b.u_min, b.u_max)), u1 = unit(std::fmax(b.u_min, b.u_max));
  const float v0 = unit(std::fmin(b.v_min, b.v_max)), v1 = unit(std::fmax(b.v_min, b.v_max));
  const auto edge = [](float t, uint32_t n) {
    const float p = t * (float)n;
    return (uint32_t)(p + 0.5f);
  };
  const ovrfsr_rect s{edge(u0, w), edge(v0, h), edge(u1, w) - edge(u0, w), edge(v1, h) - edge(v0, h)};
  const ovrfsr_rect d{edge(u0, out_w), edge(v0, out_h), edge(u1, out_w) - edge(u0, out_w), edge(v1, out_h) - edge(v0, out_h)};
  if (s.width == 0 || s.height == 0 || d.width == 0 || d.height == 0) return OVRFSR_ERR_INVALID;
  if (src_rect) *src_rect = s;
  if (dst_rect) *dst_rect = d;
  return OVRFSR_OK;
}

int ovrfsr_apply_bounds(ovrfsr_ctx *ctx, int eye, const ovrfsr_image *src_tagged, const ovrfsr_bounds *bounds, ovrfsr_image *out,
                        ovrfsr_rect *out_rect, void *stream) {
  if (!ctx || !out || (eye != 0 && eye != 1)) return OVRFSR_ERR_INVALID;
  ovrfsr_image src_untagged{};
  if (src_tagged) src_untagged = untagged(src_tagged);
  const ovrfsr_image *src = src_tagged ? &src_untagged : nullptr;
  if (!ctx->enabled || !ctx->cfg.fsr_enabled) return OVRFSR_PASSTHROUGH;
  int rc = validate_image(src);
  if (rc != OVRFSR_OK) return fail(ctx, rc, "invalid source image");
  if ((rc = select_device(ctx)) != OVRFSR_OK) return rc;
  if (ctx->initialized && (src->width != ctx->inputWidth || src->height != ctx->inputHeight || src->format != ctx->inFormat))
    ovrfsr_reset(ctx); // a texture size or format change, as in ovrfsr_apply (a rectangle change is not one)
  if (!ctx->initialized) {
    ctx->textureContainsOnlyOneEye = true;
    rc = prepare_resources(ctx, src);
    if (rc != OVRFSR_OK) {
      release_resources(ctx);
      ctx->enabled = false;
      return rc;
    }
  }
  ovrfsr_rect sr, dr;
  if ((rc = ovrfsr_bounds_rects(src->width, src->height, ctx->outputWidth, ctx->outputHeight, bounds, &sr, &dr)) != OVRFSR_OK)
    return fail(ctx, rc, "texture bounds select an empty rectangle");
  ovrfsr_ctx::BoundsEye &b = ctx->bounds[eye];
  if (!b.valid || !same_rect(b.src, sr) || !same_rect(b.dst, dr)) {
    host::make_upscale_constants(b.upscale, ctx->cfg, eye, true, sr.width, sr.height, dr.width, dr.height);
    host::make_sharpen_constants(b.sharpen, ctx->cfg, eye, true, dr.width, dr.height);
    ovrfsr_make_nis_config(b.nisScaler, &ctx->cfg, 0, eye, 1, sr.width, sr.height, dr.width, dr.height);
    ovrfsr_make_nis_config(b.nisSharpen, &ctx->cfg, 1, eye, 1, sr.width, sr.height, dr.width, dr.height);
    b.src = sr; b.dst = dr; b.valid = true;
  }
  // a ctx that ovrfsr_apply set up for one texture holding both eyes has no right-eye output yet
  if (sharpen_pass(ctx->cfg) && !ctx->sharpened[eye].img.data &&
      !ctx->sharpened[eye].alloc(ctx->outputWidth, ctx->outputHeight, ctx->outFormat))
    return fail(ctx, OVRFSR_ERR_NOMEM, "allocating sharpened texture", cudaGetLastError());
  const EyeConsts k{b.upscale, b.sharpen, b.nisScaler, b.nisSharpen};
  ovrfsr_image result{};
  rc = apply_post_process(ctx, eye, src, &result, static_cast<cudaStream_t>(stream), k, &sr, &dr);
  if (rc != OVRFSR_OK) return rc;
  *out = result;
  if (out_rect) *out_rect = dr;
  return OVRFSR_OK;
}

int ovrfsr_apply_pair(ovrfsr_ctx *ctx, const ovrfsr_image *src_left, const ovrfsr_image *src_right, int only_one_eye,
                      ovrfsr_image out[2], void *stream) {
  if (!ctx || !src_left || !src_right || !out) return OVRFSR_ERR_INVALID;
  if (!ctx->enabled || !ctx->cfg.fsr_enabled) return OVRFSR_PASSTHROUGH;
  int rc = select_device(ctx);
  if (rc != OVRFSR_OK) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  // one texture holding both eyes is processed once (PostProcessor.cpp:155-160): nothing to run side by side
  if (!only_one_eye) {
    if ((rc = ovrfsr_apply(ctx, 0, src_left, 0, &out[0], stream)) != OVRFSR_OK) return rc;
    return ovrfsr_apply(ctx, 1, src_right, 0, &out[1], stream);
  }
  if (!ctx->pairStream) {
    cudaError_t e = cudaStreamCreateWithFlags(&ctx->pairStream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->pairFork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->pairJoin, cudaEventDisableTiming);
    if (e != cudaSuccess) return fail(ctx, OVRFSR_ERR_CUDA, "creating the pair stream", e);
  }
  // fork BEFORE the left eye is queued (the right eye must not wait for it), but queue the left eye first: it is the
  // call that (re)creates the resources when the source size changed
  cudaError_t e = cudaEventRecord(ctx->pairFork, s);
  if (e != cudaSuccess) return fail(ctx, OVRFSR_ERR_CUDA, "forking the pair stream", e);
  rc = ovrfsr_apply(ctx, 0, src_left, 1, &out[0], stream);
  if (rc != OVRFSR_OK) return rc;
  e = cudaStreamWaitEvent(ctx->pairStream, ctx->pairFork, 0);
  if (e != cudaSuccess) return fail(ctx, OVRFSR_ERR_CUDA, "forking the pair stream", e);
  rc = ovrfsr_apply(ctx, 1, src_right, 1, &out[1], ctx->pairStream);
  e = cudaEventRecord(ctx->pairJoin, ctx->pairStream);
  if (e == cudaSuccess) e = cudaStreamWaitEvent(s, ctx->pairJoin, 0);
  if (e != cudaSuccess) return fail(ctx, OVRFSR_ERR_CUDA, "joining the pair stream", e);
  return rc;
}

int ovrfsr_apply_host(ovrfsr_ctx *ctx, int eye, const ovrfsr_image *src_tagged, int only_one_eye,
                      const ovrfsr_image *dst_host, void *stream) {
  if (!ctx || (eye != 0 && eye != 1)) return OVRFSR_ERR_INVALID;
  ovrfsr_image src_untagged{};
  if (src_tagged) src_untagged = untagged(src_tagged);
  const ovrfsr_image *src_host = src_tagged ? &src_untagged : nullptr;
  if (!ctx->enabled || !ctx->cfg.fsr_enabled) return OVRFSR_PASSTHROUGH;
  int rc = validate_image(src_host);
  if (rc != OVRFSR_OK) return fail(ctx, rc, "invalid host source image");
  if ((rc = validate_image(dst_host)) != OVRFSR_OK) return fail(ctx, rc, "invalid host destination image");
  if (src_host->sample_count > 1 || dst_host->sample_count > 1) return fail(ctx, OVRFSR_ERR_UNSUPPORTED, "multisampled host images");
  if ((rc = select_device(ctx)) != OVRFSR_OK) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  // "Texture size changed, recreating resources" (PostProcessor.cpp:139-142) must happen BEFORE this eye is staged:
  // the reset releases every ctx-owned image, the staging images included
  if (ctx->initialized && (src_host->width != ctx->inputWidth || src_host->height != ctx->inputHeight || src_host->format != ctx->inFormat))
    ovrfsr_reset(ctx);
  DeviceImage &st = ctx->hostStage[eye];
  if (!st.img.data || st.img.width != src_host->width || st.img.height != src_host->height || st.img.format != src_host->format) {
    if (!st.alloc(src_host->width, src_host->height, src_host->format))
      return fail(ctx, OVRFSR_ERR_NOMEM, "allocating host staging image", cudaGetLastError());
  }
  const size_t rowBytes = (size_t)src_host->width * bytes_per_pixel(src_host->format);
  cudaError_t e;
  if (src_host->pitch == rowBytes) { // tight host rows: one contiguous PCIe copy, re-pitched on the device
    DeviceBuffer &lin = ctx->hostLinearIn[eye];
    if (!lin.ensure(rowBytes * src_host->height)) return fail(ctx, OVRFSR_ERR_NOMEM, "allocating linear upload buffer", cudaGetLastError());
    e = cudaMemcpyAsync(lin.ptr, src_host->data, rowBytes * src_host->height, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = repitch_rows(st.img.data, st.img.pitch, lin.ptr, rowBytes, rowBytes, src_host->height, s);
  } else {
    e = cudaMemcpy2DAsync(st.img.data, st.img.pitch, src_host->data, src_host->pitch, rowBytes, src_host->height,
                          cudaMemcpyHostToDevice, s);
  }
  if (e != cudaSuccess) return fail(ctx, OVRFSR_ERR_CUDA, "host->device copy", e);
  ovrfsr_image out{};
  rc = ovrfsr_apply(ctx, eye, &st.img, only_one_eye, &out, stream);
  if (rc != OVRFSR_OK) return rc;
  if (dst_host->width != out.width || dst_host->height != out.height || dst_host->format != out.format)
    return fail(ctx, OVRFSR_ERR_INVALID, "host destination does not match the output size/format");
  const size_t outRowBytes = (size_t)out.width * bytes_per_pixel(out.format);
  if (dst_host->pitch == outRowBytes && out.pitch != outRowBytes) {
    DeviceBuffer &lin = ctx->hostLinearOut[eye];
    if (!lin.ensure(outRowBytes * out.height)) return fail(ctx, OVRFSR_ERR_NOMEM, "allocating linear download buffer", cudaGetLastError());
    e = repitch_rows(lin.ptr, outRowBytes, out.data, out.pitch, outRowBytes, out.height, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dst_host->data, lin.ptr, outRowBytes * out.height, cudaMemcpyDeviceToHost, s);
  } else {
    e = cudaMemcpy2DAsync(dst_host->data, dst_host->pitch, out.data, out.pitch, outRowBytes, out.height, cudaMemcpyDeviceToHost, s);
  }
  return e == cudaSuccess ? OVRFSR_OK : fail(ctx, OVRFSR_ERR_CUDA, "device->host copy", e);
}

int ovrfsr_request_capture(ovrfsr_ctx *ctx, const char *directory) {
  if (!ctx) return OVRFSR_ERR_INVALID;
  ctx->captureDir = directory ? directory : "";
  ctx->takeCapture = true; // the hotkey sets the flag, the next left-eye frame is saved (PostProcessor.cpp:699-702,634)
  return OVRFSR_OK;
}

const char *ovrfsr_last_capture_path(const ovrfsr_ctx *ctx) { return ctx ? ctx->lastCapturePath.c_str() : ""; }

int ovrfsr_resolve_msaa(const ovrfsr_image *src, const ovrfsr_image *dst, void *stream) {
  ovrfsr_image src_untagged_{};
  if (src) { src_untagged_ = untagged(src); src = &src_untagged_; }
  int rc = validate_image(src);
  if (rc != OVRFSR_OK || (rc = validate_image(dst)) != OVRFSR_OK) return rc;
  if (src->sample_count < 2 || dst->sample_count > 1 || src->format != dst->format || src->width != dst->width || src->height != dst->height)
    return OVRFSR_ERR_INVALID;
  cudaError_t e = launch_resolve_msaa(pass_image(*src), (int)src->sample_count, pass_image(*dst), static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? OVRFSR_OK : (e == cudaErrorInvalidValue ? OVRFSR_ERR_UNSUPPORTED : OVRFSR_ERR_CUDA);
}

int ovrfsr_expand_rgb32f(const ovrfsr_image *src, const ovrfsr_image *dst, void *stream) {
  ovrfsr_image src_untagged_{};
  if (src) { src_untagged_ = untagged(src); src = &src_untagged_; }
  int rc = validate_image(src);
  if (rc != OVRFSR_OK || (rc = validate_image(dst)) != OVRFSR_OK) return rc;
  if (src->format != OVRFSR_FORMAT_RGB32F || dst->format != OVRFSR_FORMAT_RGBA32F || src->width != dst->width || src->height != dst->height ||
      src->sample_count > 1 || dst->sample_count > 1)
    return OVRFSR_ERR_INVALID;
  return expand_rgb32f(*src, *dst, static_cast<cudaStream_t>(stream)) == cudaSuccess ? OVRFSR_OK : OVRFSR_ERR_CUDA;
}

int ovrfsr_format_considered_srgb(int32_t f) {
  if (f < 0) return 0;
  const int layout = f & OVRFSR_FORMAT_LAYOUT_MASK;
  const bool eightBit = layout == OVRFSR_FORMAT_RGBA8 || layout == OVRFSR_FORMAT_BGRA8 || layout == OVRFSR_FORMAT_BGRX8;
  if ((f & OVRFSR_FORMAT_SRGB_BIT) && eightBit) return 1;                                            // PostProcessor.cpp:78-81
  if ((f & OVRFSR_FORMAT_TYPELESS_BIT) && (eightBit || layout == OVRFSR_FORMAT_RGB10A2)) return 1;  // :82-87
  return 0;
}

// ---- stateless dispatches ---------------------------------------------------------------------
static int check_pair(const ovrfsr_image *src, const ovrfsr_image *dst) {
  int rc = validate_image(src);
  if (rc != OVRFSR_OK) return rc;
  if ((rc = validate_image(dst)) != OVRFSR_OK) return rc;
  if (src->format == OVRFSR_FORMAT_RGB32F) return OVRFSR_ERR_UNSUPPORTED;                                   /* expand first (ovrfsr_expand_rgb32f / ovrfsr_apply) */
  if (dst->format == OVRFSR_FORMAT_BGRX8 || dst->format == OVRFSR_FORMAT_RGB32F) return OVRFSR_ERR_UNSUPPORTED; /* source-only formats */
  if (src->sample_count > 1 || dst->sample_count > 1) return OVRFSR_ERR_UNSUPPORTED; /* resolve first (ovrfsr_resolve_msaa / ovrfsr_apply) */
  if (dst->format == OVRFSR_FORMAT_BGRA8) return OVRFSR_ERR_UNSUPPORTED; /* outputs are RGBA8 / RGB10A2 (reference) or float */
  if ((dst->format == OVRFSR_FORMAT_RGB10A2) != (src->format == OVRFSR_FORMAT_RGB10A2) && dst->format != OVRFSR_FORMAT_RGBA16F &&
      dst->format != OVRFSR_FORMAT_RGBA32F)
    return OVRFSR_ERR_UNSUPPORTED; /* UNORM targets follow DetermineOutputFormat: 10-bit in <-> 10-bit out */
  return OVRFSR_OK;
}

int ovrfsr_dispatch_fsr_easu(const ovrfsr_image *src, const ovrfsr_image *dst, const uint32_t consts[24], int math_mode,
                             void *stream) {
  ovrfsr_image src_untagged_{};
  if (src) { src_untagged_ = untagged(src); src = &src_untagged_; }
  if (!consts) return OVRFSR_ERR_INVALID;
  int rc = check_pair(src, dst);
  if (rc != OVRFSR_OK) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  cudaError_t e = math_mode == OVRFSR_MATH_STRICT ? launch_easu_strict(pass_image(*src), pass_image(*dst), consts, s)
                                                  : launch_easu_fast(pass_image(*src), pass_image(*dst), consts, s);
  if (e == cudaErrorInvalidConfiguration || e == cudaErrorInvalidValue) return OVRFSR_ERR_UNSUPPORTED;
  return e == cudaSuccess ? OVRFSR_OK : OVRFSR_ERR_CUDA;
}

int ovrfsr_dispatch_fsr_fused(const ovrfsr_image *src, const ovrfsr_image *dst, const uint32_t upscale_consts[24],
                              const uint32_t sharpen_consts[12], int math_mode, void *stream) {
  ovrfsr_image src_untagged_{};
  if (src) { src_untagged_ = untagged(src); src = &src_untagged_; }
  if (!upscale_consts || !sharpen_consts) return OVRFSR_ERR_INVALID;
  int rc = check_pair(src, dst);
  if (rc != OVRFSR_OK) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  cudaError_t e = math_mode == OVRFSR_MATH_STRICT
                      ? launch_fsr_fused_strict(pass_image(*src), pass_image(*dst), upscale_consts, sharpen_consts, s)
                      : launch_fsr_fused_fast(pass_image(*src), pass_image(*dst), upscale_consts, sharpen_consts, s);
  if (e == cudaErrorInvalidConfiguration || e == cudaErrorInvalidValue) return OVRFSR_ERR_UNSUPPORTED;
  return e == cudaSuccess ? OVRFSR_OK : OVRFSR_ERR_CUDA;
}

int ovrfsr_dispatch_fsr_rcas(const ovrfsr_image *src, const ovrfsr_image *dst, const uint32_t consts[12], int math_mode,
                             void *stream) {
  ovrfsr_image src_untagged_{};
  if (src) { src_untagged_ = untagged(src); src = &src_untagged_; }
  if (!consts) return OVRFSR_ERR_INVALID;
  int rc = check_pair(src, dst);
  if (rc != OVRFSR_OK) return rc;
  if (src->width != dst->width || src->height != dst->height) return OVRFSR_ERR_INVALID;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  cudaError_t e = math_mode == OVRFSR_MATH_STRICT ? launch_rcas_strict(pass_image(*src), pass_image(*dst), consts, s)
                                                  : launch_rcas_fast(pass_image(*src), pass_image(*dst), consts, s);
  if (e == cudaErrorInvalidValue) return OVRFSR_ERR_UNSUPPORTED;
  return e == cudaSuccess ? OVRFSR_OK : OVRFSR_ERR_CUDA;
}

// ---- host constants -----------------------------------------------------------------------------
void ovrfsr_output_size(uint32_t in_w, uint32_t in_h, float render_scale, uint32_t *out_w, uint32_t *out_h) {
  uint32_t w = 0, h = 0;
  host::output_size(in_w, in_h, render_scale, &w, &h);
  if (out_w) *out_w = w;
  if (out_h) *out_h = h;
}
void ovrfsr_fsr_easu_con(uint32_t con[16], float vw, float vh, float iw, float ih, float ow, float oh) {
  host::fsr_easu_con(con, vw, vh, iw, ih, ow, oh);
}
void ovrfsr_fsr_rcas_con(uint32_t con[4], float stops) { host::fsr_rcas_con(con, stops); }
void ovrfsr_make_upscale_constants(uint32_t consts[24], const ovrfsr_config *cfg, int eye, int only_one_eye, uint32_t in_w,
                                   uint32_t in_h, uint32_t out_w, uint32_t out_h) {
  host::make_upscale_constants(consts, *cfg, eye, only_one_eye != 0, in_w, in_h, out_w, out_h);
}
void ovrfsr_make_sharpen_constants(uint32_t consts[12], const ovrfsr_config *cfg, int eye, int only_one_eye, uint32_t out_w,
                                   uint32_t out_h) {
  host::make_sharpen_constants(consts, *cfg, eye, only_one_eye != 0, out_w, out_h);
}

// ---- introspection ------------------------------------------------------------------------------
int ovrfsr_get_upscale_constants(const ovrfsr_ctx *ctx, int eye, uint32_t consts[24]) {
  if (!ctx || !consts || (eye != 0 && eye != 1) || !ctx->initialized) return OVRFSR_ERR_INVALID;
  std::memcpy(consts, ctx->upscaleConstants[ctx->textureContainsOnlyOneEye ? eye : 0], 96);
  return OVRFSR_OK;
}
int ovrfsr_get_sharpen_constants(const ovrfsr_ctx *ctx, int eye, uint32_t consts[12]) {
  if (!ctx || !consts || (eye != 0 && eye != 1) || !ctx->initialized) return OVRFSR_ERR_INVALID;
  std::memcpy(consts, ctx->sharpenConstants[ctx->textureContainsOnlyOneEye ? eye : 0], 48);
  return OVRFSR_OK;
}
void ovrfsr_cas_setup(uint32_t consts[8], float sharpness, float max_color_delta, float in_w, float in_h, float out_w, float out_h) {
  if (consts) host::cas_setup(consts, sharpness, max_color_delta, in_w, in_h, out_w, out_h);
}

int ovrfsr_dispatch_cas(const ovrfsr_image *src, const ovrfsr_image *dst, const uint32_t consts[8], int sharpen_only, int math_mode,
                        void *stream) {
  ovrfsr_image src_untagged_{};
  if (src) { src_untagged_ = untagged(src); src = &src_untagged_; }
  if (!consts) return OVRFSR_ERR_INVALID;
  int rc = check_pair(src, dst);
  if (rc != OVRFSR_OK) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  cudaError_t e = math_mode == OVRFSR_MATH_STRICT ? launch_cas_strict(pass_image(*src), pass_image(*dst), consts, sharpen_only, s)
                                                  : launch_cas_fast(pass_image(*src), pass_image(*dst), consts, sharpen_only, s);
  if (e == cudaErrorInvalidValue) return OVRFSR_ERR_UNSUPPORTED;
  return e == cudaSuccess ? OVRFSR_OK : OVRFSR_ERR_CUDA;
}

int ovrfsr_selftest_rcp(uint32_t *mismatches, uint32_t *checked) {
  uint32_t r[2] = {0, 0};
  if (selftest_rcas_rcp(r, nullptr) != cudaSuccess) return OVRFSR_ERR_CUDA;
  if (mismatches) *mismatches = r[0];
  if (checked) *checked = r[1];
  return OVRFSR_OK;
}
int ovrfsr_selftest_div(uint32_t *mismatches, uint32_t *checked) {
  uint32_t r[2] = {0, 0};
  if (selftest_nis_div(r, nullptr) != cudaSuccess) return OVRFSR_ERR_CUDA;
  if (mismatches) *mismatches = r[0];
  if (checked) *checked = r[1];
  return OVRFSR_OK;
}
uint64_t ovrfsr_kernel_launches(void) { return ovrfsr::g_launches.load(std::memory_order_relaxed); }

int ovrfsr_get_gpu_time_ms(ovrfsr_ctx *ctx, float *mean_ms) {
  if (!ctx || !mean_ms) return 0;
  harvest_queries(ctx);
  if (ctx->countedQueries == 0) return 0;
  // "Average GPU processing time for upscale", x2 when each texture holds one eye (PostProcessor.cpp:619-626)
  float avg = ctx->summedGpuTime / (float)ctx->countedQueries;
  if (ctx->textureContainsOnlyOneEye) avg *= 2;
  *mean_ms = avg;
  return ctx->countedQueries;
}

const char *ovrfsr_last_error(const ovrfsr_ctx *ctx) { return ctx ? ctx->lastError.c_str() : "null context"; }

const char *ovrfsr_status_string(int status) {
  switch (status) {
    case OVRFSR_OK: return "ok";
    case OVRFSR_ERR_INVALID: return "invalid argument";
    case OVRFSR_ERR_UNSUPPORTED: return "unsupported format or scale";
    case OVRFSR_ERR_CUDA: return "CUDA failure or no device";
    case OVRFSR_ERR_NOMEM: return "out of memory";
    case OVRFSR_PASSTHROUGH: return "post-processing disabled: pass-through";
    default: return "unknown status";
  }
}
uint32_t ovrfsr_version(void) { return OVRFSR_VERSION; }

int ovrfsr_image_alloc(ovrfsr_image *img, uint32_t width, uint32_t height, int32_t format) {
  if (!img || width == 0 || height == 0 || !valid_format(format)) return OVRFSR_ERR_INVALID;
  DeviceImage d;
  if (!d.alloc(width, height, format)) return OVRFSR_ERR_NOMEM;
  *img = d.img;
  return OVRFSR_OK;
}
void ovrfsr_image_free(ovrfsr_image *img) {
  if (img && img->data) cudaFree(img->data);
  if (img) *img = ovrfsr_image{};
}

} // extern "C"
