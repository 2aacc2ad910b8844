// datum_b200 — launch interface of the equirect -> cube stage (internal to libdatum_ibl_cuda).
#pragma once

#include "ibl_math.cuh"

#include <cuda_runtime.h>
#include <cstdint>

namespace ibl
{
  // Texel format of the level 0 these stages write (include/datum_ibl_cuda.h: DATUM_IBL_FORMAT_*): kFormatRgbe
  // stores rgbe() words like the reference; kFloatFormatF32 / kFloatFormatF16 (prefilter_f.h) store the texel
  // of a float chain instead (F32: the fp32 rgb; F16: min(x, 65504) rounded to nearest-even; alpha 1.0).
  constexpr int kFormatRgbe = 0;

  struct ResampleParams
  {
    float4 const *image;   // HDRImage::bits, imgw*imgh RGBA fp32 (tools/hdr.h:24)
    int imgw, imgh;
    int width, height;     // cube face size
    float area_x, area_y;  // tools/hdr.cpp:345
    Quatf quats[6];        // tools/hdr.cpp:335-343 (same table as tools/ibl.cpp:253-261)
    void *dst;             // 6*width*height texels of the format the launch is given
  };

  // tools/hdr.cpp:347-356: box-filtered equirect lookup per cube texel, packed with rgbe() or stored in `format`.
  // The float formats keep the arithmetic up to sum / totalweight and replace only rgbe().
  cudaError_t launch_equirect_resample(ResampleParams const &p, int format, cudaStream_t stream);

  // tools/assetbuilder.cpp:443-462: six ARGB32 face images -> level 0 of the payload.  Per pixel
  // rgbe(srgba(pixel)) (color.h:125-128: c/255 then pow 2.2, table `lut` of the 256 possible values),
  // or the linear rgb stored in `format`; rows mirrored vertically (QImage::mirrored), faces in argument
  // order.  `argb` = 6*width*height pixels.
  cudaError_t launch_ingest_argb32(uint32_t const *argb, float const *lut, int width, int height, int format, void *dst, int sm_count, cudaStream_t stream);

  // tools/hdr.cpp:173-318 on one level: the twelve 0.3/0.4/0.3 edge blends, in the reference's order.  Each
  // loop reads the texels of `format` as stored (halves widened) and stores its results in `format`.
  cudaError_t launch_blend_edges(void *level, int format, int width, int height, cudaStream_t stream);
}
