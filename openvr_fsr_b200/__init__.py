"""openvr_fsr_b200 -- B200-native (sm_100a) FSR1 EASU+RCAS / NIS eye-texture post-process.

Only the one hot path of fholger/openvr_fsr lives here (SURVEY.md section 8): csrc/ holds the CUDA kernels,
the C ABI (include/ovrfsr.h) and the C++ vr::PostProcessor drop-in; api.py mirrors that surface for Python.
"""
from ._lib import (ERR_CUDA, ERR_INVALID, ERR_NOMEM, ERR_UNSUPPORTED, FORMAT_AUTO, FORMAT_BGRA8, FORMAT_RGBA8,  # noqa
                   FORMAT_RGBA16F, FORMAT_RGBA32F, FORMAT_RGB10A2, FORMAT_BGRX8, FORMAT_RGB32F, FORMAT_SRGB_BIT,
                   FORMAT_TYPELESS_BIT, MATH_FAST, MATH_STRICT, OK, PASSTHROUGH, OvrFsrError)
from .api import (EYE_LEFT, EYE_RIGHT, Config, PostProcessor, TextureBounds, alloc_image, fsr_easu, fsr_fused, fsr_rcas, image_of,  # noqa
                  kernel_launches, make_nis_config, make_sharpen_constants, make_upscale_constants, nis_scaler,
                  nis_sharpen, output_size, to_image, resolve_msaa, expand_rgb32f, format_considered_srgb, recommended_render_size, mip_lod_bias,
                  sampler_lod_bias, capture_filename, save_dds, load_dds, cas, cas_setup, bounds_rects)
