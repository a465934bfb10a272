// kernels.h -- host-visible launchers of the sm_100a kernels, one set per math mode.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/ovrfsr.h"

namespace ovrfsr {

// ptr/pitch/w/h: the image a pass reads or writes.  It may be a rectangle of a larger texture (ovrfsr_apply_bounds):
// ptr then points at the rectangle's texel (x0, y0) of a texture texW x texH texels large.  texW == 0: the image is
// the whole texture.  The kernels treat the rectangle's edge as the texture's edge; TMA descriptors stay keyed by
// the whole texture, so a rectangle that changes every frame keeps hitting the descriptor cache.
struct PassImage {
  void *ptr; uint32_t pitch; int w, h; int format;
  int x0 = 0, y0 = 0, texW = 0, texH = 0;
  bool is_crop() const { return texW != 0 && (x0 != 0 || y0 != 0 || w != texW || h != texH); }
};

// FSR (fsr_kernels.cuh).  consts are the reference's constant-buffer layouts.
// `direct` (EASU) / `skipOutside` (RCAS) are the ctx path's pairing of the two passes: when RCAS follows EASU in the same
// apply, EASU writes the outside-radius groups -- which RCAS would only copy (x the debug tint `tintGB`) -- straight
// to the final image `direct`, and RCAS visits only tiles / groups inside the radius.  Same output bits as two plain
// dispatches; a stateless dispatch passes nullptr / false.
cudaError_t launch_easu_fast(const PassImage &src, const PassImage &dst, const uint32_t consts[24], cudaStream_t s,
                             const PassImage *direct = nullptr, float tintGB = 1.0f);
cudaError_t launch_easu_strict(const PassImage &src, const PassImage &dst, const uint32_t consts[24], cudaStream_t s,
                               const PassImage *direct = nullptr, float tintGB = 1.0f);
cudaError_t launch_rcas_fast(const PassImage &src, const PassImage &dst, const uint32_t consts[12], cudaStream_t s,
                             bool skipOutside = false);
cudaError_t launch_rcas_strict(const PassImage &src, const PassImage &dst, const uint32_t consts[12], cudaStream_t s,
                               bool skipOutside = false);

// EASU -> RCAS in one kernel (fsr_fused.cuh): ku = UpscaleConstants, ks = SharpenConstants; dst.format (RGBA8, or RGB10A2
// for an RGB10A2 source) is also the format the intermediate is quantised to.  cudaErrorInvalidValue /
// cudaErrorInvalidConfiguration = this pair of passes cannot be fused (the caller runs the two dispatches instead).
cudaError_t launch_fsr_fused_fast(const PassImage &src, const PassImage &dst, const uint32_t ku[24], const uint32_t ks[12], cudaStream_t s);
cudaError_t launch_fsr_fused_strict(const PassImage &src, const PassImage &dst, const uint32_t ku[24], const uint32_t ks[12], cudaStream_t s);

// NIS (nis_kernels.cuh).  cfg = the 256-byte NISConfig block; coef = [2][64][8] floats (scale, usm) on the host.
cudaError_t launch_nis_scaler_fast(const PassImage &src, const PassImage &dst, const void *cfg256, const float *coef, cudaStream_t s);
cudaError_t launch_nis_scaler_strict(const PassImage &src, const PassImage &dst, const void *cfg256, const float *coef, cudaStream_t s);
cudaError_t launch_nis_sharpen_fast(const PassImage &src, const PassImage &dst, const void *cfg256, const float *coef, cudaStream_t s);
cudaError_t launch_nis_sharpen_strict(const PassImage &src, const PassImage &dst, const void *cfg256, const float *coef, cudaStream_t s);

// NVScaler (sharpen == false) or NVSharpen in the given math mode: what ovrfsr_dispatch_nis_scaler / _sharpen run on
// their checked images, and the ctx path's NIS passes (nis_capi.cu)
cudaError_t launch_nis(bool sharpen, const PassImage &src, const PassImage &dst, const void *cfg256, int math_mode, cudaStream_t s);

// legacy CAS (cas_kernels.cuh).  consts = const0, const1 of src/cas/cas.compute.h:1-4 as CasSetup fills them.
cudaError_t launch_cas_fast(const PassImage &src, const PassImage &dst, const uint32_t consts[8], int sharpenOnly, cudaStream_t s);
cudaError_t launch_cas_strict(const PassImage &src, const PassImage &dst, const uint32_t consts[8], int sharpenOnly, cudaStream_t s);

// exhaustive device check of strict RCAS's UNORM8 reciprocal: result = {mismatches, operands checked}
cudaError_t selftest_rcas_rcp(uint32_t result[2], cudaStream_t s);
// strict NIS's in-range IEEE quotient (div_rn_inrange) against div.rn on ~19 M operand pairs: {mismatches, checked}
cudaError_t selftest_nis_div(uint32_t result[2], cudaStream_t s);

// MSAA resolve front-end (GetInputView's ResolveSubresource, PostProcessor.cpp:219-226): dst = mean over the
// `samples` consecutive samples of each texel; same format both sides.  One arithmetic (strict) for both math modes.
cudaError_t launch_resolve_msaa(const PassImage &srcSamples, int samples, const PassImage &dst, cudaStream_t s);

// bumped once per kernel launch by every launcher (ovrfsr_kernel_launches)
void count_launch();

} // namespace ovrfsr
