// datum_b200 host shim — the reference's tools/ibl.h:9-15, unchanged signatures.
#pragma once

#include "hdr.h"

void image_buildmips_cube_ibl(int width, int height, int levels, void *bits);

void image_pack_cube_ibl(HDRImage const &image, int width, int height, int levels, void *bits);

void image_pack_envbrdf(int width, int height, void *bits);

void image_pack_watercolor(lml::Color3 const &deepcolor, lml::Color3 const &shallowcolor, float depthscale, lml::Color3 const &fresnelcolor, float fresnelbias, float fresnelpower, int width, int height, void *bits);

// Extensions with no counterpart in the reference's tools (SURVEY.md §8b): the SH9
// projection of data/project.comp as an offline step, `sh` = float[9][3] like
// Irradiance::L (src/renderer/envmap.h:112-115); and the sample count of the bake
// (tools/ibl.cpp:162 hard-codes 1024, which stays the default).
void image_project_sh9_cube(int width, int height, void const *level0_rgbe, float *sh);

// On-disk form of the probe irradiance (SURVEY.md 8 f4; the reference has none — its runtime gets
// `Irradiance` from data/project.comp only).  Both are ordinary IMAG payloads for write_imag_asset
// (tools/assetpacker.h:26), so a pack needs no new chunk type:
//   SH9 ............. width 3, height 9, layers 1, levels 1, PackImageHeader::f32 (src/assetpack.h:89):
//                     27 floats, byte for byte `Irradiance::L[9][3]` (src/renderer/envmap.h:112-115); a loader
//                     memcpy's the 108-byte payload into the struct it hands to LightList::push_probe
//                     (src/renderer/lightlist.cpp:102-112).  image_pack_irradiance_sh9 fills it from level 0
//                     of a baked (or just ingested) rgbe cube payload.
//   irradiance cube . width w, height h, layers 6, levels 1, PackImageHeader::rgbe: E(n) of
//                     data/lighting.inc:351-371 at the texel directions of tools/ibl.cpp:269, the face order
//                     of every other cube payload; loads through the existing EnvMap path.
void image_pack_irradiance_sh9(int width, int height, void const *level0_rgbe, void *bits);
void image_pack_irradiance_cube(void const *sh9_bits, int width, int height, void *bits);

// The body of write_skybox_asset(fout, id, paths) between image loading and
// write_imag_asset (tools/assetbuilder.cpp:443-465) as one call: `argb` points at six
// width*height blocks of QImage::Format_ARGB32 pixels (image.bits() after
// convertToFormat, :445) in the caller's face order; per pixel rgbe(srgba(pixel)),
// vertical mirror, then the prefilter chain.  `bits` = the whole payload.
void image_pack_cube_faces_ibl(unsigned int const *argb, int width, int height, int levels, void *bits);

// The .hdr flow of write_skybox_asset (tools/assetbuilder.cpp:473-491) producing a float probe: the resample
// and edge blend of image_pack_cube_ibl with level 0 stored as RGBA32F or RGBA16F texels (`format` =
// DATUM_IBL_FORMAT_F32 or DATUM_IBL_FORMAT_F16) instead of rgbe, then the float prefilter chain
// (datum_ibl_pack_cube_float_ibl).  `chain` = the whole chain, 16 or 8 bytes per texel, levels of the payload.
void image_pack_cube_float_ibl(HDRImage const &image, int width, int height, int levels, int format, void *chain);
void image_set_ibl_samples(int samples);

// `count` image_buildmips_cube_ibl calls as one: payloads of the same width/height/levels, their
// uploads, kernels and downloads overlapped (datum_ibl_bake_probes).  `sh` (may be null)
// receives count x float[9][3], the SH9 projection of every level 0.
void image_buildmips_cube_ibl_batch(int count, int width, int height, int levels, void *const *bits, float *sh);
